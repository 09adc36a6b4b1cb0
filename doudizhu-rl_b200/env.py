"""Batched, GPU-resident Doudizhu env with the reference's Python env API.

Mirrors reference envi.py:16-217 (classes Env / EnvComplicated / EnvCooperation / EnvCooperationSimplify):
same verbs (reset, prepare, face, valid_actions, step_manual, step_random, step_auto), same tensor layouts
(face float32 [C,15,4], actions float32 [N,15,4] thermometer one-hot), over a leading batch of B envs.
`BatchedEnv*` are the batched classes; `Env*` are B=1 views with the exact single-env signatures so the
reference's game.py / dqn.py / net.py loop runs on them unchanged.

All arithmetic happens in hand-written sm_100a kernels behind the C-ABI of include/ddz_b200.h; PyTorch only
owns the buffers and the stream.  There is no CPU fallback.
"""
from collections import namedtuple

import numpy as np
import torch

from . import _native as N
from .deals import DEAL_SEED0, default_deals, random_deals, adversarial_pairs, ADVERSARIAL_POOL  # noqa: F401  (re-exported)

VARIANT_CHANNELS = (4, 7, 9, 6)
DEFAULT_REWARDS = (50, 100, 50)          # role 0 up, 1 lord, 2 down  (reference game.py:13-14)
_SHIFTS = None


def _shifts(device):
    return (torch.arange(15, device=device, dtype=torch.int64) * 4)


def pack_counts(counts):
    """int [...,15] per-rank counts -> int64 packed nibbles (the library's uint64 move/hand format)."""
    c = torch.as_tensor(counts)
    return (c.to(torch.int64) << _shifts(c.device)).sum(-1)


def unpack_counts(packed):
    """int64 packed nibbles [...] -> int64 [...,15] per-rank counts."""
    p = torch.as_tensor(packed)
    return (p.unsqueeze(-1) >> _shifts(p.device)) & 15


def _align(x, a):
    return (x + a - 1) // a * a


class StepResults:
    """Outputs of one step in ONE contiguous buffer (a single D2H copy fetches them): r int8[B] | done uint8[B] |
    cat int8[B] | pad | reward float32[B,3]."""

    def __init__(self, B, device, pin=False, buf=None):
        self.B = B
        self.off_reward = _align(3 * B, 16)
        self.nbytes = self.off_reward + 12 * B
        self.buf = buf if buf is not None else torch.zeros(self.nbytes, dtype=torch.uint8, device=device)
        if pin:
            self.buf = self.buf.pin_memory()
        self.r = self.buf[0:B].view(torch.int8)
        self.done = self.buf[B:2 * B]
        self.cat = self.buf[2 * B:3 * B].view(torch.int8)
        self.reward = self.buf[self.off_reward:].view(torch.float32).view(B, 3)
        if pin:   # host copies: numpy views of the same pinned memory, for cheap per-step reads
            self.r_np, self.done_np, self.cat_np, self.reward_np = (t.numpy() for t in (self.r, self.done, self.cat, self.reward))


class Trajectory:
    """Output buffers of a multi-step call (BatchedEnv.rollout_steps): slice s of every tensor is the observation
    and the step results after step s -- offsets int32 [K,B+1], actions_u64 int64 [K,cap], actions_f32 [K,cap,15,4],
    face [K,B,C,15,4], r / done / cat [K,B], reward [K,B,3]."""

    def __init__(self, env, nsteps, want_reward=True):
        K, B, dev = int(nsteps), env.B, env.device
        if K < 1:
            raise ValueError("nsteps must be positive")
        self.K, self.B, self.C = K, B, env.C
        self.cap = env.cap
        self.offsets = torch.zeros((K, B + 1), dtype=torch.int32, device=dev)
        self.actions_u64 = torch.zeros((K, self.cap), dtype=torch.int64, device=dev)
        self.actions_f32 = N.row_tensor((K, self.cap, 15, 4), dev)
        self.face = N.row_tensor((K, B, env.C, 15, 4), dev)
        self.r = torch.zeros((K, B), dtype=torch.int8, device=dev)
        self.done = torch.zeros((K, B), dtype=torch.uint8, device=dev)
        self.cat = torch.zeros((K, B), dtype=torch.int8, device=dev)
        self.reward = torch.zeros((K, B, 3), dtype=torch.float32, device=dev) if want_reward else None

    def valid_actions(self, s):
        """(float32 [N_s,15,4], int32 [B+1]) of slice s (synchronises to read the total)"""
        n = int(self.offsets[s, self.B].item())
        return self.actions_f32[s, :min(n, self.cap)], self.offsets[s]


class BatchedEnv:
    """B independent Doudizhu games on one GPU.  Reference: envi.py:16-157 (class Env, C=4 face)."""

    VARIANT = N.FACE_FIRST

    def __init__(self, num_envs=1, debug=False, seed=None, device=None, max_actions_per_env=None,
                 rewards=DEFAULT_REWARDS, env0=0, stats=None):
        if not torch.cuda.is_available():
            raise N.DdzError("BatchedEnv needs a CUDA device: the env runs as sm_100a kernels, there is no CPU path")
        self.B = int(num_envs)
        if self.B <= 0:
            raise ValueError("num_envs must be positive")
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.debug = debug
        self.seed = int(seed) if seed else 0          # `if seed:` like envi.py:18 (seed=0 == unseeded)
        self.env0 = int(env0)                          # global id of env 0 (multi-GPU sharding)
        self.C = VARIANT_CHANNELS[self.VARIANT]
        per_env = int(max_actions_per_env) if max_actions_per_env else N.MAX_LEGAL
        self.cap = self.B * per_env
        dev, B = self.device, self.B
        with torch.cuda.device(dev):
            self._state = torch.zeros(N.lib.ddz_state_bytes(B) // 4, dtype=torch.int32, device=dev)
            self._ws = torch.zeros(max(1, N.lib.ddz_workspace_bytes(B) // 4), dtype=torch.int32, device=dev)
            self._offsets = [torch.zeros(B + 1, dtype=torch.int32, device=dev) for _ in range(2)]
            self._actions_u64 = [torch.zeros(self.cap, dtype=torch.int64, device=dev) for _ in range(2)]
            self._actions_f32 = N.row_tensor((self.cap, 15, 4), dev)      # compressible memory where the GPU has it
            self._face = N.row_tensor((B, self.C, 15, 4), dev)
            self._results = [StepResults(B, dev) for _ in range(2)]   # two sets: a D2H read of one may overlap the next step
            self._res = 0
            # int64 [16] counters the kernels add to atomically; several envs (the groups of a GroupedEnv) may share one
            self.stats = stats if stats is not None else torch.zeros(16, dtype=torch.int64, device=dev)
            self._rewards = torch.tensor(list(rewards), dtype=torch.int32, device="cpu")
        self._buf_gen = 0        # bumped when the list buffers are reallocated (cached pointers / captured graphs are stale)
        self._cur = 0            # which ping-pong list describes the current state
        self._fresh = False      # lists/face valid for the current state?
        self._n_total = None
        self._stepno = 0
        self._games_dealt = 0
        self._perm_dev = None
        self._lord_dev = None
        self.reset()

    # results of the most recent step (device tensors; views into one contiguous buffer)
    @property
    def r(self):
        return self._results[self._res].r

    @property
    def done(self):
        return self._results[self._res].done

    @property
    def cat(self):
        return self._results[self._res].cat

    @property
    def reward(self):
        return self._results[self._res].reward

    # ------------------------------------------------------------------ plumbing
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    @staticmethod
    def _p(t):
        return None if t is None else t.data_ptr()

    def _fields(self):
        """int64 view [9,B] (hand[3], hist[3], recent[3]) and int32 meta [B] of the state buffer."""
        B = self.B
        f = self._state[: 18 * B].view(torch.int64).view(9, B)
        meta = self._state[18 * B: 19 * B]
        return f, meta

    def _to_dev(self, a, dtype):
        if a is None:
            return None
        t = torch.as_tensor(a)
        if t.dtype != dtype:
            t = t.to(dtype)
        return t.to(self.device, non_blocking=True).contiguous()

    # ------------------------------------------------------------------ reference API
    def reset(self):
        """envi.py:30-36 + CEnv.reset: clear the table (hands are empty until prepare())."""
        self._state.zero_()
        f, meta = self._fields()
        meta.fill_(1)            # lord to move, not done, no deals consumed
        self._ws.zero_()         # tile ticket / look-back words / device step counter
        self._fresh = False
        self._stepno = 0

    def prepare(self, perm=None, lord_pile=None, only_done=False, pool_games=1):
        """CEnv.prepare (game.py:171): deal.  perm int8 [pool_games*B,54] host or device, lord_pile int8 [pool_games*B].
        Without perm the documented default stream is used (default_deals)."""
        B = self.B
        if perm is None:
            perm, lord_pile = default_deals(self._games_dealt, B)
            pool_games = 1
        perm_d = self._to_dev(perm, torch.int8)
        if perm_d.numel() != pool_games * B * 54:
            raise ValueError("perm must have shape [pool_games*B, 54]")
        lord_d = self._to_dev(lord_pile, torch.int8)
        if lord_d is not None and lord_d.numel() != pool_games * B:
            raise ValueError("lord_pile must have shape [pool_games*B]")
        self._perm_dev, self._lord_dev = perm_d, lord_d      # keep alive while the launch is in flight
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_reset(self._p(self._state), self._p(perm_d), self._p(lord_d), int(pool_games),
                                    int(bool(only_done)), self._p(self.stats), B, self._stream()), "ddz_reset")
        self._games_dealt += B
        self._fresh = False
        self._check_errors("prepare")

    def observe(self):
        """Run legal-move generation + encoders for the current state (the work behind env.face and
        env.valid_actions(), envi.py:87-116)."""
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_observe(self._p(self._state), self._p(self._ws), self.VARIANT,
                                      self._p(self._offsets[self._cur]), self._p(self._actions_u64[self._cur]),
                                      self._p(self._actions_f32), self.cap, self._p(self._face),
                                      self._p(self.stats), self.B, self._stream()), "ddz_observe")
        self._fresh, self._n_total = True, None
        return self

    def _ensure(self):
        if not self._fresh:
            self.observe()

    @property
    def offsets(self):
        self._ensure()
        return self._offsets[self._cur]

    @property
    def num_actions(self):
        """total number of legal moves over the batch (host int; synchronises).  If the lists did not fit the action buffer
        (max_actions_per_env below the worst case; the launch said so in stats[7]) the buffers are grown to what the
        offsets ask for and the state is observed once more: the caller always gets complete lists."""
        self._ensure()
        if self._n_total is None:
            n = int(self._offsets[self._cur][self.B].item())
            if n > self.cap:
                self._grow(n)
                self.observe()
                n = int(self._offsets[self._cur][self.B].item())
                if n > self.cap:
                    raise N.DdzError("legal-move lists overflowed the action buffer (%d > cap %d)" % (n, self.cap))
            self._n_total = n
        return self._n_total

    def _grow(self, need):
        """reallocate the list buffers for at least `need` moves (+25 %); the packed lists of the other ping-pong set are kept"""
        cap = min(self.B * N.MAX_LEGAL, max(int(need) + int(need) // 4, self.cap + 1))
        dev = self.device
        with torch.cuda.device(dev):
            for i in range(2):
                new = torch.zeros(cap, dtype=torch.int64, device=dev)
                new[: self.cap] = self._actions_u64[i]
                self._actions_u64[i] = new
            self._actions_f32 = N.row_tensor((cap, 15, 4), dev)
        self.cap = cap
        self._buf_gen += 1

    @property
    def face(self):
        """float32 [B,C,15,4] on the GPU (envi.py:87-96)."""
        self._ensure()
        return self._face

    @property
    def actions_packed(self):
        n = self.num_actions              # first: it may grow (replace) the list buffers
        return self._actions_u64[self._cur][:n]

    def valid_actions(self, tensor=True):
        """tensor=True: (float32 [sumN,15,4], int32 offsets [B+1]); False: per-env lists of 15-int lists (envi.py:98-116)."""
        self._ensure()
        n = self.num_actions
        if tensor:
            return self._actions_f32[:n], self._offsets[self._cur]
        counts = unpack_counts(self._actions_u64[self._cur][:n]).cpu().numpy()
        off = self._offsets[self._cur].cpu().numpy()
        return [[[int(x) for x in row] for row in counts[off[b]:off[b + 1]]] for b in range(self.B)]

    def legal_counts(self):
        """int32 [B]: number of legal moves of the player to move in every env, in closed form (ddz_legal_count) -- no
        lists are built or needed (e.g. to size buffers, or to draw a uniformly random move index for ddz_kth_moves)."""
        counts = torch.empty(self.B, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_legal_count(self._p(self._state), counts.data_ptr(), self.B, self._stream()), "ddz_legal_count")
        return counts

    def state_actions(self, env_mask=None):
        """The Q-network's input for every legal move, written in place (net.py:81-90 without `face.repeat` and
        `torch.cat`): float32 [n, C+1, 15, 4], row i = [face of the move's env | the move's one-hot].  env_mask bool [B]:
        only the moves of those envs, packed in env order.  Returns (x, rows) with rows = indices of the encoded moves in
        the CSR action list (None when every move is encoded)."""
        self._ensure()
        off = self._offsets[self._cur]
        if env_mask is None:
            n, dst, rows, mask8 = self.num_actions, None, None, None
        else:
            mask = env_mask.to(self.device, torch.bool)
            cnt = (off[1:] - off[:-1]) * mask
            dst = torch.zeros(self.B + 1, dtype=torch.int32, device=self.device)
            dst[1:] = torch.cumsum(cnt, 0)
            n = int(dst[-1].item())
            owner_mask = torch.repeat_interleave(mask, (off[1:] - off[:-1]).to(torch.int64), output_size=self.num_actions)
            rows = owner_mask.nonzero(as_tuple=True)[0]
            mask8 = mask.to(torch.uint8)
        x = torch.empty((n, self.C + 1, 15, 4), dtype=torch.float32, device=self.device)
        if n:
            with torch.cuda.device(self.device):
                N.check(N.lib.ddz_encode_state_actions(self._p(self._state), self.VARIANT, self._p(off),
                                                       self._p(self._actions_u64[self._cur]), self._p(mask8), self._p(dst),
                                                       x.data_ptr(), self.B, self._stream()), "ddz_encode_state_actions")
        return x, rows

    def _step(self, choice, mode):
        self._ensure()
        if self.cap < self.B * N.MAX_LEGAL:
            # ddz_step reads the lists without knowing their capacity: with a reduced max_actions_per_env make sure the
            # observation was complete (num_actions raises on an overflow) before any index is resolved against it
            self.num_actions
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_step(self._p(self._state), self._p(self._offsets[self._cur]),
                                   self._p(self._actions_u64[self._cur]), self._p(choice), mode,
                                   self.seed, self.env0, self._stepno, self._rewards.data_ptr(),
                                   self._p(self.r), self._p(self.done), self._p(self.cat), self._p(self.reward),
                                   self._p(self.stats), self.B, self._stream()), "ddz_step")
        self._fresh = False
        self._stepno += 1
        self._check_errors("step")
        return self.r, self.done, self.cat

    def step(self, choice):
        """apply legal move number choice[b] of every env (the index stream of the parity contract)."""
        return self._step(self._to_dev(choice, torch.int32), N.CHOICE_INDEX)

    def legal_ids(self):
        """int32 [sumN]: the action id (move_ids) of every legal move, in CSR order parallel to valid_actions() -- the ids
        of one env's list strictly increase."""
        return move_ids(self.actions_packed, self.device)

    def legal_mask(self, layout="bool"):
        """One row per env over the 13 551 action ids (ddz_legal_mask; the counterpart of the reference's
        get_mask_onehot60): "bool" -> bool [B, 13551]; "bits" -> int32 [B, 424], bit id & 31 of word id >> 5.  A finished
        env has an all-zero row.  The lists are complete (the buffers grow as num_actions does)."""
        lay = {"bool": N.MASK_BYTES, "bits": N.MASK_BITS}.get(layout)
        if lay is None:
            raise ValueError("layout must be 'bool' or 'bits', not %r" % (layout,))
        self.num_actions
        shape, dtype = ((self.B, N.NUM_ACTION_IDS), torch.bool) if lay == N.MASK_BYTES else ((self.B, N.MASK_WORDS), torch.int32)
        out = torch.empty(shape, dtype=dtype, device=self.device)
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_legal_mask(self._p(self._offsets[self._cur]), self._p(self._actions_u64[self._cur]), self.cap,
                                         lay, out.data_ptr(), self._p(self.stats), self.B, self._stream()), "ddz_legal_mask")
        return out

    def step_ids(self, ids):
        """apply the move with action id ids[b] in every env (moves_of_ids, then the DDZ_CHOICE_MOVE step).  An id that is
        not legal in its env, or outside [0, 13551), is an illegal choice: the env is left as it is, its sticky error bit
        is set, stats[7] counts it, and debug=True raises."""
        return self._step(moves_of_ids(self._to_dev(ids, torch.int32), self.device), N.CHOICE_MOVE)

    def step_manual(self, onehot_cards):
        """envi.py:63-70: onehot float/int [B,15,4] (a row of valid_actions per env) -> (r, done, cat)."""
        oh = torch.as_tensor(onehot_cards, device=self.device)
        moves = pack_counts(oh.reshape(self.B, 15, 4).sum(-1).round().to(torch.int64)).contiguous()
        return self._step(moves, N.CHOICE_MOVE)

    def step_random(self, entropy=None):
        """envi.py:79-85: uniform random legal move.  entropy uint32/int32 [B] -> index = entropy % N (host-supplied
        stream); None -> device Philox4x32-10 keyed (seed, env0+b, step number)."""
        if entropy is None:
            return self._step(None, N.CHOICE_PHILOX)
        return self._step(self._to_dev(np.asarray(entropy).view(np.int32) if isinstance(entropy, np.ndarray)
                                       else entropy, torch.int32), N.CHOICE_MOD)

    def step_auto(self):
        """envi.py:72-77: RHCP heuristic opponent -- out of scope for this build (SURVEY.md 2.1)."""
        raise NotImplementedError("step_auto (RHCP rule AI of the absent native env) is not part of the hot path")

    def rollout_step(self, choice=None, mode=N.CHOICE_PHILOX, perm=None, lord_pile=None, pool_games=1, auto_step=False):
        """One fused env-step in ONE launch (ddz_rollout_step): apply the chosen move, re-deal finished envs from perm
        (device int8 [pool*B,54]) when given, and produce face + legal lists of the new state.  auto_step: the Philox
        step number comes from the device-side counter instead of the host (CUDA-graph replay, see GraphedRollout)."""
        self._ensure()
        nxt = 1 - self._cur
        self._res = nxt               # result set follows the ping-pong, so a graph replay leaves it consistent
        if choice is not None:
            choice = self._to_dev(choice, torch.int64 if mode == N.CHOICE_MOVE else torch.int32)
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_rollout_step(
                self._p(self._state), self._p(self._ws), self.VARIANT,
                self._p(self._offsets[self._cur]), self._p(self._actions_u64[self._cur]),
                self._p(choice), mode, self.seed, self.env0, N.STEPNO_AUTO if auto_step else self._stepno,
                self._rewards.data_ptr(), self._p(perm), self._p(lord_pile), int(pool_games),
                self._p(self.r), self._p(self.done), self._p(self.cat), self._p(self.reward),
                self._p(self._offsets[nxt]), self._p(self._actions_u64[nxt]), self._p(self._actions_f32), self.cap,
                self._p(self._face), self._p(self.stats), self.B, self._stream()), "ddz_rollout_step")
        self._cur, self._fresh, self._n_total = nxt, True, None
        self._stepno += 1
        return self.r, self.done, self.cat

    def rollout_steps(self, traj, entropy=None, perm=None, lord_pile=None, pool_games=1, auto_step=False):
        """traj.K fused env-steps enqueued by ONE native call (ddz_rollout_steps), every step's observation and results
        kept in `traj`: the random rollout (envi.py:79-85 for all three seats, game.py:259-275) needs no host decision
        between steps.  Moves: Philox stream of the env (entropy None) or host-made entropy int32 [K,B]
        (index = entropy % N).  Equal to traj.K calls of rollout_step; the env's own lists are stale afterwards
        (the next .face / .valid_actions() re-observes)."""
        self._ensure()
        K = traj.K
        if traj.cap != self.cap:
            raise ValueError("the trajectory must have the env's list capacity (max_actions_per_env)")
        mode = N.CHOICE_PHILOX if entropy is None else N.CHOICE_MOD
        if entropy is not None:
            entropy = self._to_dev(entropy, torch.int32)
            if entropy.numel() != K * self.B:
                raise ValueError("entropy must be [K,B]")
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_rollout_steps(
                self._p(self._state), self._p(self._ws), self.VARIANT, K,
                self._p(self._offsets[self._cur]), self._p(self._actions_u64[self._cur]), self._p(entropy), mode,
                self.seed, self.env0, N.STEPNO_AUTO if auto_step else self._stepno, self._rewards.data_ptr(),
                self._p(perm), self._p(lord_pile), int(pool_games), self._p(traj.r), self._p(traj.done),
                self._p(traj.cat), self._p(traj.reward), self._p(traj.offsets), self._p(traj.actions_u64),
                self._p(traj.actions_f32), traj.cap, self._p(traj.face), self._p(self.stats), self.B, self._stream()),
                "ddz_rollout_steps")
        self._fresh, self._n_total = False, None
        self._stepno += K
        return traj

    def playout(self, max_steps=256, policy="uniform"):
        """Random playout of every env (MCTS default policy, server/mcts/default_policy.py:4-10): up to max_steps random
        legal moves per env or to the end of its game, Philox stream continued from the env's step counter.  One launch,
        no lists / features written.  Returns int32 [B] decisions played; winners are in `winner`, counters in `stats`.
        policy "uniform": every legal move is equally likely (step_random, envi.py:79-85); "search": the draw is from the
        search bot's own pruned move list (server/mcts/get_moves.py:36-69), as the reference's playouts do."""
        if policy not in ("uniform", "search"):
            raise ValueError("policy must be 'uniform' or 'search'")
        fn = N.lib.ddz_playout if policy == "uniform" else N.lib.ddz_playout_pruned
        steps = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            N.check(fn(self._p(self._state), int(max_steps), self.seed, self.env0, self._stepno,
                       self._rewards.data_ptr(), steps.data_ptr(), self._p(self.stats), self.B,
                       self._stream()), "ddz_playout")
        self._fresh = False
        self._stepno += int(max_steps)
        return steps

    def _sync_auto_step(self):
        """write the host's step number into the device-side Philox step counter (workspace header, uint32 at byte 12).
        Only the fused launches keep that counter up to date; step() / step_random() / playout() advance the step number
        on the host alone, so a graph replay (stepno = DDZ_STEPNO_AUTO) after one of them re-arms the counter first."""
        self._ws[3:4].fill_(int(self._stepno) & 0x7FFFFFFF)

    def _check_errors(self, what):
        if self.debug:
            err = int(self.stats[7].item())
            if err:
                raise N.DdzError("%s: %d env(s) flagged an error (illegal choice, bad permutation or list overflow)" % (what, err))

    # ------------------------------------------------------------------ getters (native env getters, App. A)
    def get_role_ID(self):
        """1 = up, 2 = lord, 3 = down (envi.py:64) -> int64 [B]"""
        return (self._fields()[1] & 3).to(torch.int64) + 1

    def _role(self):
        return (self._fields()[1] & 3).to(torch.int64)

    def hands(self):
        """int64 [B,3,15] counts of every role's hand."""
        return unpack_counts(self._fields()[0][0:3].t().contiguous())

    def get_curr_handcards(self):
        """counts int64 [B,15] of the player to move (the reference returns card values 3..17; see Env view)."""
        h = self.hands()
        return h[torch.arange(self.B, device=self.device), self._role()]

    def get_last_two_cards(self):
        """int64 [B,2,15]: [previous player's hand-out, the one before]; zeros = pass (envi.py:103)."""
        rec = self._recent_t()
        s = self._role()
        ar = torch.arange(self.B, device=self.device)
        return torch.stack([rec[ar, (s + 2) % 3], rec[ar, (s + 1) % 3]], 1)

    @property
    def left(self):
        """cards left per role int64 [B,3] (envi.py:23,39)."""
        return self.hands().sum(-1)

    def _history_t(self):
        return unpack_counts(self._fields()[0][3:6].t().contiguous())

    def _recent_t(self):
        return unpack_counts(self._fields()[0][6:9].t().contiguous())

    @property
    def history(self):
        """int64 [B,3,15] (envi.py:25,41)."""
        return self._history_t()

    @property
    def taken(self):
        """int64 [B,15] (envi.py:22,40)."""
        return self._history_t().sum(1)

    @property
    def recent_handout(self):
        """int64 [B,3,15] (envi.py:26,42-43)."""
        return self._recent_t()

    def get_state_prob(self):
        """native get_state_prob (envi.py:94): float32 [B,120] = the two probability planes of the face, flattened."""
        return BatchedEnv.face.fget(self)[:, self.C - 2:].reshape(self.B, 120)

    @classmethod
    def get_state_prob_manual(cls, known60, size1, size2, device=None):
        """native get_state_prob_manual (server/core.py:26-33): known60 = thermometer one-hot [.., 60] of (played cards +
        own hand), size1 / size2 = cards left of the next / next-next player.  float32 [.., 120] (SURVEY App. A form A)."""
        k = torch.as_tensor(known60, device=device).reshape(-1, 15, 4)
        if N.lib.ddz_prob_form() == 1:     # form B build: deck60 - known60, element by element (DESIGN.md 2: the one layout nothing in the reference pins)
            deck = torch.ones(15, 4, device=k.device)
            deck[13:, 1:] = 0
            thermo = (deck - (k != 0).to(torch.float32)).clamp_(min=0).reshape(-1, 60)
        else:                              # form A: thermometer of the number of unknown cards per rank
            known = (k != 0).sum(-1)
            total = torch.tensor([4] * 13 + [1, 1], device=k.device)
            unknown = (total - known).clamp_(min=0)
            thermo = (torch.arange(4, device=k.device)[None, None, :] < unknown[:, :, None]).to(torch.float32).reshape(-1, 60)
        s1 = torch.as_tensor(size1, device=k.device, dtype=torch.float32).reshape(-1, 1)
        s2 = torch.as_tensor(size2, device=k.device, dtype=torch.float32).reshape(-1, 1)
        tot = s1 + s2
        p1 = torch.where(tot > 0, s1 / tot, torch.zeros_like(tot))
        p2 = torch.where(tot > 0, s2 / tot, torch.zeros_like(tot))
        out = torch.cat([thermo * p1, thermo * p2], -1)
        return out if out.shape[0] > 1 else out[0]

    @property
    def is_done(self):
        return ((self._fields()[1] >> 2) & 1).to(torch.bool)

    @property
    def winner(self):
        return ((self._fields()[1] >> 3) & 3).to(torch.int64)

    def state_dict(self):
        """Exact-resume checkpoint of the env (the reference never checkpoints env state, SURVEY.md 5)."""
        return {"state": self._state.clone(), "stepno": self._stepno, "games_dealt": self._games_dealt,
                "stats": self.stats.clone()}      # the device-side step counter is re-derived from stepno on load

    def load_state_dict(self, sd):
        self._state.copy_(sd["state"])
        self.stats.copy_(sd["stats"])
        self._stepno, self._games_dealt = int(sd["stepno"]), int(sd["games_dealt"])
        self._sync_auto_step()
        self._fresh = False

    # ------------------------------------------------------------------ converters (envi.py:118-157)
    @classmethod
    def arr2cards(cls, arr):
        """counts[15] -> card values 3..17, ascending (envi.py:119-130)"""
        arr = np.asarray(arr).astype(np.int64).reshape(15)
        return np.repeat(np.arange(3, 18), arr)

    @classmethod
    def cards2arr(cls, cards):
        """card values 3..17 -> counts[15] (envi.py:133-137)"""
        cards = np.asarray(cards, dtype=np.int64).reshape(-1)
        return np.bincount(cards - 3, minlength=15).astype(np.int64) if cards.size else np.zeros(15, np.int64)

    @classmethod
    def batch_arr2onehot(cls, batch_arr):
        """counts [n,15] -> thermometer one-hot int [n,15,4]: res[i][rank][:count] = 1 (envi.py:140-146)"""
        a = np.asarray(batch_arr).astype(np.int64).reshape(-1, 15)
        return (np.arange(4)[None, None, :] < a[:, :, None]).astype(np.int64)

    @classmethod
    def onehot2arr(cls, onehot_cards):
        """one-hot [15,4] -> counts[15] (row sums, envi.py:149-157)"""
        if torch.is_tensor(onehot_cards):
            onehot_cards = onehot_cards.detach().cpu().numpy()
        return np.asarray(onehot_cards).reshape(15, 4).sum(-1).round().astype(np.int64)

    @staticmethod
    def encode_actions(packed):
        """packed moves int64 [n] on the GPU -> float32 [n,15,4] (envi.py:113)."""
        packed = packed.contiguous()
        out = torch.empty((packed.numel(), 15, 4), dtype=torch.float32, device=packed.device)
        with torch.cuda.device(packed.device):
            N.check(N.lib.ddz_encode_actions(packed.data_ptr(), packed.numel(), out.data_ptr(),
                                             torch.cuda.current_stream(packed.device).cuda_stream), "ddz_encode_actions")
        return out


class GraphedRollout:
    """CUDA-graph replay of the fused env-step: the two launches of a ping-pong pair are captured once and replayed,
    which removes the per-step host cost (argument marshalling + launch) from a rollout loop.  Moves are chosen on
    the device (Philox stream, or host-refreshed entropy in `entropy`); finished envs re-deal from `perm`."""

    def __init__(self, env, perm=None, lord_pile=None, pool_games=1, entropy=None):
        self.env = env
        env._ensure()
        torch.cuda.synchronize(env.device)
        mode = N.CHOICE_PHILOX if entropy is None else N.CHOICE_MOD
        kw = dict(choice=entropy, mode=mode, perm=perm, lord_pile=lord_pile, pool_games=pool_games, auto_step=True)
        self._keep = (perm, lord_pile, entropy)
        self.graph = torch.cuda.CUDAGraph()
        stepno = env._stepno
        env._sync_auto_step()
        torch.cuda.synchronize(env.device)
        with torch.cuda.graph(self.graph):
            env.rollout_step(**kw)
            env.rollout_step(**kw)
        env._stepno = stepno          # capture launched nothing; the device counter still holds `stepno`
        self._next = stepno
        self._cur0 = env._cur         # the ping-pong set the graph's first launch reads
        self._gen = env._buf_gen

    def replay(self):
        """two env-steps"""
        env = self.env
        if env._buf_gen != self._gen:
            raise N.DdzError("the list buffers were reallocated after the capture: capture again")
        if env._cur != self._cur0:                # an odd number of eager fused steps in between: the graph reads the other set
            env._cur, env._fresh = self._cur0, False
        env._ensure()                             # e.g. after step() / step_random(): lists of the CURRENT state, in that set
        if env._stepno != self._next:             # stepped by other means since the last replay
            env._sync_auto_step()
        self.graph.replay()
        self.env._stepno += 2
        self._next = self.env._stepno
        self.env._n_total = None


class GroupedEnv:
    """The envs of one GPU as several independent groups, each with its own stream, state and CSR outputs.

    The step kernel has a load-only prologue (no stores for the first ~8 us) and a tail; a single chain of launches
    pays both every step.  With two (or more) unsynchronised chains one group's prologue and tail overlap another
    group's store phase (+17 % env-steps/s at 131 072 envs with two groups, +27 % with four once the row buffers are
    compressible; profiles/r1_two_stream_experiment.json, r1u_group_sweep.json) -- the classic
    double-buffered actor: while group A's observations are consumed, group B steps.  Global env ids (Philox stream,
    deal rows) are those of one big batch, so every env's trajectory is independent of the grouping.
    """

    def __init__(self, env_cls, num_envs, groups=2, seed=None, device=None, env0=0, **kw):
        if num_envs % groups:
            raise ValueError("num_envs must be divisible by groups")
        self.B, self.G, self.Bg = int(num_envs), int(groups), int(num_envs) // int(groups)
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.streams = [torch.cuda.Stream(self.device) for _ in range(self.G)]
        # ONE statistics vector for all groups: every kernel adds to it atomically, so reading the rank's counters (and
        # the multi-GPU all-reduce, sharding.allreduce_stats) needs no reduction over the groups
        self._stats = torch.zeros(16, dtype=torch.int64, device=self.device)
        self.envs = []
        for g in range(self.G):
            with torch.cuda.stream(self.streams[g]):
                self.envs.append(env_cls(self.Bg, seed=seed, device=self.device, env0=env0 + g * self.Bg,
                                         stats=self._stats, **kw))
        self.graphs = None
        self._pool = None

    def _fork(self):
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        for s in self.streams:
            s.wait_event(ev)

    def join(self):
        """make the current stream wait for every group's stream"""
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            ev = torch.cuda.Event()
            ev.record(s)
            cur.wait_event(ev)

    def prepare(self, perm, lord_pile, pool_games=1):
        """perm int8 [pool_games*B,54], lord_pile int8 [pool_games*B] for the whole batch (host or device); each group
        keeps its slice as its device-resident deal pool."""
        P = int(pool_games)
        perm_t = torch.as_tensor(perm).reshape(P, self.B, 54)
        lord_t = torch.as_tensor(lord_pile).reshape(P, self.B)
        self._pool = []
        self._fork()
        for g, env in enumerate(self.envs):
            with torch.cuda.stream(self.streams[g]):
                pg = perm_t[:, g * self.Bg:(g + 1) * self.Bg].to(self.device).contiguous()
                lg = lord_t[:, g * self.Bg:(g + 1) * self.Bg].to(self.device).contiguous()
                self._pool.append((pg, lg, P))
                env.prepare(pg, lg, pool_games=P)
                env.observe()
        self.join()

    def rollout_step(self, **kw):
        """one fused env-step of every group, each on its own stream (Philox moves, re-deal from the group's pool)"""
        for g, env in enumerate(self.envs):
            with torch.cuda.stream(self.streams[g]):
                pg, lg, P = self._pool[g]
                env.rollout_step(perm=pg, lord_pile=lg, pool_games=P, **kw)

    def capture(self, steps_per_graph=8):
        """one CUDA graph per group with `steps_per_graph` (even) fused env-steps; replay() launches all of them"""
        if steps_per_graph % 2:
            raise ValueError("steps_per_graph must be even (ping-pong buffers)")
        torch.cuda.synchronize(self.device)
        self.graphs, self.steps_per_graph = [], int(steps_per_graph)
        for g, env in enumerate(self.envs):
            pg, lg, P = self._pool[g]
            env._ensure()
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            stepno = env._stepno
            with torch.cuda.stream(self.streams[g]):
                env._sync_auto_step()
            torch.cuda.synchronize(self.device)
            with torch.cuda.graph(graph, stream=self.streams[g]):
                for _ in range(self.steps_per_graph):
                    env.rollout_step(perm=pg, lord_pile=lg, pool_games=P, auto_step=True)
            env._stepno = stepno
            env._graph_next, env._graph_cur0, env._graph_gen = stepno, env._cur, env._buf_gen
            self.graphs.append(graph)
        torch.cuda.synchronize(self.device)

    def replay(self):
        for g, graph in enumerate(self.graphs):
            env = self.envs[g]
            if env._buf_gen != env._graph_gen:
                raise N.DdzError("the list buffers were reallocated after the capture: capture again")
            with torch.cuda.stream(self.streams[g]):
                if env._cur != env._graph_cur0:        # an odd number of eager / host-pipe steps in between
                    env._cur, env._fresh = env._graph_cur0, False
                env._ensure()
                if env._stepno != env._graph_next:     # stepped by other means (eager step, host pipe) since the last replay
                    env._sync_auto_step()
                graph.replay()
            env._stepno += self.steps_per_graph
            env._graph_next = env._stepno
            env._n_total = None

    @property
    def stats(self):
        """int64 [16], shared by all groups (call join() / synchronize before reading it)"""
        return self._stats


class HostRollout:
    """Rollout driven from HOST buffers: the call a host-side user makes per env-step.

    Every step the caller hands over a pinned host array of entropy (uint32/int32 [B]: move index = entropy % N, the
    batched form of envi.py:83 random.choice) and gets the step's results (r, done, cat, reward) back in pinned host
    memory.  Deck permutations are host-supplied too: `refill(slot, perm, lord_pile)` uploads one slot of the
    device-resident deal pool (each env consumes one deal per game, so one slot per ~game length keeps it fresh).
    The per-step sequencing lives in the library (ddz_pipe_step): H2D and D2H run on the pipe's own copy streams, so
    the H2D of step t+1 and the D2H of step t-1 overlap the kernel of step t, and a step costs one native call.
    """

    def __init__(self, env, perm, lord_pile, pool_games, fetch_reward=False):
        """fetch_reward: also read the float32 [B,3] reward block back every step (12 of the 15 result bytes per env).
        The reference's step returns only (r, done, cat) and derives rewards on the host (game.py:109-118), so by
        default only r | done | cat travel over PCIe; the rewards stay available on the device (env.reward)."""
        self.env, self.G = env, int(pool_games)
        dev, B = env.device, env.B
        self.perm_d = env._to_dev(perm, torch.int8).reshape(self.G, B, 54).contiguous()
        self.lord_d = env._to_dev(lord_pile, torch.int8).reshape(self.G, B).contiguous()
        self.entropy_d = [torch.zeros(B, dtype=torch.int32, device=dev) for _ in range(2)]
        self.results_h = [StepResults(B, "cpu", pin=True) for _ in range(N.PIPE_DEPTH)]   # ring: read up to 3 steps late
        self.d2h_bytes = self.results_h[0].nbytes if fetch_reward else _align(3 * B, 16)
        self._stage = None
        with torch.cuda.device(dev):
            self._pipe = N.lib.ddz_pipe_create()
        if not self._pipe:
            raise N.DdzError("ddz_pipe_create failed: %s" % N.lib.ddz_last_error().decode())
        self.i = 0
        self._argv = None
        self._main = torch.cuda.current_stream(dev)      # every step is issued on the stream current at construction
        env._ensure()

    def __del__(self):
        pipe, self._pipe = getattr(self, "_pipe", None), None
        if pipe and N is not None and getattr(N, "lib", None) is not None:   # module globals may be gone at interpreter exit
            N.lib.ddz_pipe_destroy(pipe)

    def refill(self, slot, perm, lord_pile, now=False):
        """upload one slot of the deal pool: perm int8 [B,54], lord_pile int8 [B], pinned host memory.  The upload
        lands in a staging buffer on its own copy stream (overlapping the kernels); the slot itself is replaced by a
        device-to-device copy ordered between two steps -- no kernel ever reads a half-written permutation -- issued by
        the first step() that finds the upload complete, so no step waits for it.  now=True (or flush()) makes the
        replacement take effect before the next step, at the price of that step waiting for the upload."""
        env, B = self.env, self.env.B
        if self._stage is None:
            self._stage = (torch.empty((B, 54), dtype=torch.int8, device=env.device),
                           torch.empty(B, dtype=torch.int8, device=env.device))
        perm, lord_pile = torch.as_tensor(perm), torch.as_tensor(lord_pile)
        self._keep = (perm, lord_pile)
        with torch.cuda.device(env.device):
            N.check(N.lib.ddz_pipe_refill(self._pipe, self.perm_d[slot].data_ptr(), self.lord_d[slot].data_ptr(),
                                          perm.data_ptr(), lord_pile.data_ptr(), self._stage[0].data_ptr(),
                                          self._stage[1].data_ptr(), B, self._main.cuda_stream), "ddz_pipe_refill")
        if now:
            self.flush()

    def flush(self):
        """commit a staged refill now: the next step sees the new deals (the stream waits for the upload)"""
        with torch.cuda.device(self.env.device):
            N.check(N.lib.ddz_pipe_flush(self._pipe, self._main.cuda_stream), "ddz_pipe_flush")

    def _build_args(self):
        """Everything ddz_pipe_step needs is constant per (list parity, step index % PIPE_DEPTH): marshal it once."""
        import ctypes as C
        env = self.env
        vp = lambda t: C.c_void_p(None if t is None else t.data_ptr())
        self._argv = {}
        for cur in (0, 1):
            nxt = 1 - cur
            for k in range(N.PIPE_DEPTH):
                self._argv[(cur, k)] = [
                    C.c_void_p(self._pipe), vp(env._state), vp(env._ws), C.c_int(env.VARIANT),
                    vp(env._offsets[cur]), vp(env._actions_u64[cur]),
                    None, vp(self.entropy_d[k & 1]), C.c_uint64(env.seed), C.c_uint64(env.env0), None,
                    vp(env._rewards), vp(self.perm_d), vp(self.lord_d), C.c_int(self.G),
                    vp(env._results[nxt].buf), vp(self.results_h[k].buf), C.c_size_t(self.d2h_bytes),
                    vp(env._offsets[nxt]), vp(env._actions_u64[nxt]), vp(env._actions_f32), C.c_int64(env.cap),
                    vp(env._face), vp(env.stats), C.c_int(env.B), C.c_void_p(self._main.cuda_stream)]
        self._same_device = torch.cuda.current_device() == (env.device.index or 0)
        self._gen = env._buf_gen

    def step(self, entropy_h):
        """entropy_h: pinned int32 [B].  Returns the StepResults (pinned host views) this step will fill; they are
        valid after `wait(results)` (or any later synchronisation) and are reused PIPE_DEPTH steps later."""
        env, k = self.env, self.i % N.PIPE_DEPTH
        if self._argv is None or self._gen != env._buf_gen:
            self._build_args()
        cur = env._cur
        argv = self._argv[(cur, k)]
        argv[6] = entropy_h.data_ptr()
        argv[10] = env._stepno
        if self._same_device:
            rc = N.lib.ddz_pipe_step(*argv)
        else:
            with torch.cuda.device(env.device):
                rc = N.lib.ddz_pipe_step(*argv)
        if rc:
            N.check(rc, "ddz_pipe_step")
        nxt = 1 - cur
        env._cur, env._res, env._fresh, env._n_total = nxt, nxt, True, None
        env._stepno += 1
        res_h = self.results_h[k]
        res_h._slot, res_h._pipe = k, self._pipe
        self.i += 1
        return res_h

    @staticmethod
    def wait(results):
        N.check(N.lib.ddz_pipe_wait(results._pipe, results._slot), "ddz_pipe_wait")
        return results


class GroupStepResults:
    """Host view of one step's results of all groups (pinned): r | done | cat per group, group-major."""

    def __init__(self, sizes, pin=True):
        self.sizes = list(sizes)
        self.nbytes = 3 * sum(self.sizes)
        self.buf = torch.zeros(self.nbytes, dtype=torch.uint8)
        if pin:
            self.buf = self.buf.pin_memory()
        self.r, self.done, self.cat = [], [], []
        off = 0
        for B in self.sizes:
            self.r.append(self.buf[off:off + B].view(torch.int8).numpy())
            self.done.append(self.buf[off + B:off + 2 * B].numpy())
            self.cat.append(self.buf[off + 2 * B:off + 3 * B].view(torch.int8).numpy())
            off += 3 * B


class HostRolloutGroups:
    """HostRollout for a GroupedEnv: ONE native call per env-step of all groups (ddz_mpipe_step) -- one H2D of the step's
    entropy (pinned int32 [B], global env order) on a copy stream, one launch per group on its stream, one D2H of every
    group's r | done | cat into a ring of PIPE_DEPTH pinned buffers; device buffers rotate through the same ring, so no
    stream waits for an older step.  4 G + 4 CUDA calls per step instead of 12 G.
    refill(slot, perm [B,54], lord [B]) uploads one slot of every group's deal pool."""

    def __init__(self, ge):
        import ctypes as C
        self.ge, self.G, dev = ge, ge.G, ge.device
        if ge._pool is None:
            raise ValueError("prepare() the GroupedEnv first (it owns the device-resident deal pools)")
        self.P = ge._pool[0][2]
        self.sizes = [e.B for e in ge.envs]
        B = sum(self.sizes)
        self.entropy_d = [torch.zeros(B, dtype=torch.int32, device=dev) for _ in range(N.PIPE_DEPTH)]
        self.results_d = [torch.zeros(3 * B, dtype=torch.uint8, device=dev) for _ in range(N.PIPE_DEPTH)]
        self.results_h = [GroupStepResults(self.sizes) for _ in range(N.PIPE_DEPTH)]
        self.h2d_bytes, self.d2h_bytes = 4 * B, 3 * B
        # staging buffers of the deal-pool uploads: allocated here, not by the first refill (an allocation synchronises)
        self._stage = (torch.empty((B, 54), dtype=torch.int8, device=dev), torch.empty(B, dtype=torch.int8, device=dev))
        self._slot_ptrs = {}
        with torch.cuda.device(dev):
            self._pipe = N.lib.ddz_mpipe_create(self.G)
        if not self._pipe:
            raise N.DdzError("ddz_mpipe_create failed: %s" % N.lib.ddz_last_error().decode())
        self.i = 0
        for e in ge.envs:
            e._ensure()
        # the group descriptors are constant per list parity: marshal them once
        self._gs = {}
        for cur in (0, 1):
            arr = (N.GroupStep * self.G)()
            for g, e in enumerate(ge.envs):
                nxt = 1 - cur
                pg, lg, _ = ge._pool[g]
                q = arr[g]
                q.state, q.workspace = e._state.data_ptr(), e._ws.data_ptr()
                q.prev_offsets, q.prev_actions_u64 = e._offsets[cur].data_ptr(), e._actions_u64[cur].data_ptr()
                q.out_offsets, q.out_actions_u64 = e._offsets[nxt].data_ptr(), e._actions_u64[nxt].data_ptr()
                q.out_actions_f32, q.face = e._actions_f32.data_ptr(), e._face.data_ptr()
                q.perm, q.lord_pile = pg.data_ptr(), lg.data_ptr()
                q.reward = e._results[nxt].reward.data_ptr()
                q.cap, q.env0, q.B, q.stream = e.cap, e.env0, e.B, ge.streams[g].cuda_stream
            self._gs[cur] = arr
        self._gens = [e._buf_gen for e in ge.envs]
        e0 = ge.envs[0]
        self._const = (C.c_int(e0.VARIANT), C.c_uint64(e0.seed), C.c_void_p(e0._rewards.data_ptr()), C.c_int(self.P),
                       C.c_void_p(ge.stats.data_ptr()))
        self._same_device = torch.cuda.current_device() == (dev.index or 0)

    def __del__(self):
        pipe, self._pipe = getattr(self, "_pipe", None), None
        if pipe and N is not None and getattr(N, "lib", None) is not None:
            N.lib.ddz_mpipe_destroy(pipe)

    def step(self, entropy_h):
        """entropy_h: pinned int32 [B] (global env order).  Returns the GroupStepResults this step fills; valid after
        wait(results), reused PIPE_DEPTH steps later."""
        ge, k = self.ge, self.i % N.PIPE_DEPTH
        if [e._buf_gen for e in ge.envs] != self._gens:
            raise N.DdzError("an env's list buffers were reallocated: build a new HostRolloutGroups")
        for g, e in enumerate(ge.envs):
            if not e._fresh or e._cur != ge.envs[0]._cur:      # stepped eagerly in between: lists of the current state first
                with torch.cuda.stream(ge.streams[g]):
                    e._cur, e._fresh = ge.envs[0]._cur, e._fresh and e._cur == ge.envs[0]._cur
                    e._ensure()
        cur = ge.envs[0]._cur
        variant, seed, rewards, P, stats = self._const
        args = (self._pipe, self._gs[cur], variant, entropy_h.data_ptr(), self.entropy_d[k].data_ptr(), seed,
                ge.envs[0]._stepno, rewards, P, self.results_d[k].data_ptr(), self.results_h[k].buf.data_ptr(), stats)
        if self._same_device:
            rc = N.lib.ddz_mpipe_step(*args)
        else:
            with torch.cuda.device(ge.device):
                rc = N.lib.ddz_mpipe_step(*args)
        if rc:
            N.check(rc, "ddz_mpipe_step")
        nxt = 1 - cur
        for e in ge.envs:
            e._cur, e._res, e._fresh, e._n_total = nxt, nxt, True, None
            e._stepno += 1
        res = self.results_h[k]
        res._slot, res._pipe = k, self._pipe
        self.i += 1
        return res

    @staticmethod
    def wait(results):
        N.check(N.lib.ddz_mpipe_wait(results._pipe, results._slot), "ddz_mpipe_wait")
        return results

    def refill(self, slot, perm, lord_pile, now=False):
        """upload one slot of every group's deal pool from pinned host arrays perm int8 [B,54], lord_pile int8 [B]
        (global env order); committed between two steps by the first step() that finds the upload complete"""
        import ctypes as C
        ge = self.ge
        perm, lord_pile = torch.as_tensor(perm), torch.as_tensor(lord_pile)
        self._keep = (perm, lord_pile)
        if slot not in self._slot_ptrs:
            self._slot_ptrs[slot] = ((C.c_void_p * self.G)(*[ge._pool[g][0][slot].data_ptr() for g in range(self.G)]),
                                     (C.c_void_p * self.G)(*[ge._pool[g][1][slot].data_ptr() for g in range(self.G)]))
        pp, ll = self._slot_ptrs[slot]
        with torch.cuda.device(ge.device):
            N.check(N.lib.ddz_mpipe_refill(self._pipe, self._gs[0], pp, ll, perm.data_ptr(), lord_pile.data_ptr(),
                                           self._stage[0].data_ptr(), self._stage[1].data_ptr()), "ddz_mpipe_refill")
        if now:
            self.flush()

    def flush(self):
        with torch.cuda.device(self.ge.device):
            N.check(N.lib.ddz_mpipe_flush(self._pipe, self._gs[0]), "ddz_mpipe_flush")

    def join(self, stream=None):
        """make `stream` (default: the current one) wait for the device-to-host copy of the latest step's results"""
        st = stream if stream is not None else torch.cuda.current_stream(self.ge.device)
        with torch.cuda.device(self.ge.device):
            N.check(N.lib.ddz_mpipe_join(self._pipe, st.cuda_stream), "ddz_mpipe_join")


class BatchedEnvComplicated(BatchedEnv):
    """envi.py:160-178, C=7"""
    VARIANT = N.FACE_COMPLICATED


class BatchedEnvCooperation(BatchedEnv):
    """envi.py:181-198, C=9"""
    VARIANT = N.FACE_COOPERATION


class BatchedEnvCooperationSimplify(BatchedEnv):
    """envi.py:201-217, C=6"""
    VARIANT = N.FACE_SIMPLIFY


class MoveGenerator:
    """Batched r.get_moves (envi.py:111) with preallocated buffers: n independent (hand, last) pairs per call."""

    def __init__(self, n, device=None, max_moves_per_hand=N.MAX_LEGAL):
        if not torch.cuda.is_available():
            raise N.DdzError("MoveGenerator needs a CUDA device")
        self.n = int(n)
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        self.cap = self.n * int(max_moves_per_hand)
        self._ws = torch.zeros(max(1, N.lib.ddz_workspace_bytes(self.n) // 4 + 1), dtype=torch.int32, device=self.device)
        self.offsets = torch.zeros(self.n + 1, dtype=torch.int32, device=self.device)
        self.actions = torch.zeros(self.cap, dtype=torch.int64, device=self.device)
        self.stats = torch.zeros(16, dtype=torch.int64, device=self.device)

    def generate(self, hands_packed, lasts_packed):
        """packed int64 [n] device tensors -> (actions int64 [cap] (first offsets[n] valid), offsets int32 [n+1]); async."""
        with torch.cuda.device(self.device):
            N.check(N.lib.ddz_legal_moves(hands_packed.data_ptr(), lasts_packed.data_ptr(), self._ws.data_ptr(),
                                          self.offsets.data_ptr(), self.actions.data_ptr(), self.cap,
                                          self.stats.data_ptr(), self.n,
                                          torch.cuda.current_stream(self.device).cuda_stream), "ddz_legal_moves")
        return self.actions, self.offsets


def kth_moves(hands, lasts, idx, device=None):
    """idx[i]-th move of r.get_moves(hands[i], lasts[i]) without building the lists: (packed int64 [n], counts int32 [n])."""
    if not torch.cuda.is_available():
        raise N.DdzError("kth_moves needs a CUDA device")
    dev = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
    h = pack_counts(torch.as_tensor(np.asarray(hands)).reshape(-1, 15).to(dev)).contiguous()
    l = pack_counts(torch.as_tensor(np.asarray(lasts)).reshape(-1, 15).to(dev)).contiguous()
    k = torch.as_tensor(np.asarray(idx), dtype=torch.int32).to(dev).contiguous()
    out = torch.zeros(h.numel(), dtype=torch.int64, device=dev)
    cnt = torch.zeros(h.numel(), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_kth_moves(h.data_ptr(), l.data_ptr(), k.data_ptr(), out.data_ptr(), cnt.data_ptr(), h.numel(),
                                    torch.cuda.current_stream(dev).cuda_stream), "ddz_kth_moves")
    return out, cnt


def mcts_moves(hands, lasts, device=None):
    """Batched mcts.get_moves.get_moves (server/mcts/get_moves.py:36-69): the search bot's move list -- r.get_moves, pruned
    to its lowest- and highest-valued thirds when it has more than 10 entries, in the reference's order.
    hands/lasts int [n,15] -> (packed int64 [n, 344], counts int32 [n]) on the device."""
    if not torch.cuda.is_available():
        raise N.DdzError("mcts_moves needs a CUDA device")
    dev = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
    h = pack_counts(torch.as_tensor(np.asarray(hands)).reshape(-1, 15).to(dev)).contiguous()
    l = pack_counts(torch.as_tensor(np.asarray(lasts)).reshape(-1, 15).to(dev)).contiguous()
    out = torch.zeros((h.numel(), N.MCTS_MAX_MOVES), dtype=torch.int64, device=dev)
    cnt = torch.zeros(h.numel(), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_mcts_moves(h.data_ptr(), l.data_ptr(), out.data_ptr(), cnt.data_ptr(), h.numel(),
                                     torch.cuda.current_stream(dev).cuda_stream), "ddz_mcts_moves")
    return out, cnt


def get_moves(hands, lasts, device=None):
    """Batched r.get_moves(hand15, last15) (envi.py:111): hands/lasts int [n,15] -> (packed int64 [sumN], offsets int32 [n+1])."""
    if not torch.cuda.is_available():
        raise N.DdzError("get_moves needs a CUDA device")
    dev = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
    h = pack_counts(torch.as_tensor(np.asarray(hands)).reshape(-1, 15).to(dev)).contiguous()
    l = pack_counts(torch.as_tensor(np.asarray(lasts)).reshape(-1, 15).to(dev)).contiguous()
    n = h.numel()
    ws = torch.zeros(max(1, N.lib.ddz_workspace_bytes(n) // 4), dtype=torch.int32, device=dev)
    offsets = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    cap = n * N.MAX_LEGAL
    out = torch.zeros(cap, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_legal_moves(h.data_ptr(), l.data_ptr(), ws.data_ptr(), offsets.data_ptr(), out.data_ptr(),
                                      cap, None, n, torch.cuda.current_stream(dev).cuda_stream), "ddz_legal_moves")
    return out[: int(offsets[n].item())], offsets


# ---------------------------------------------------------------------- action ids (a fixed index per move)
ActionSpace = namedtuple("ActionSpace", "moves card_py_index id_of_card_py")


def _id_device(device):
    if not torch.cuda.is_available():
        raise N.DdzError("action ids are computed on a CUDA device")
    return torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())


def _as_int_tensor(x, dtype, dev):
    if isinstance(x, np.ndarray) and x.dtype == np.uint64:
        x = x.view(np.int64)
    t = torch.as_tensor(x)
    if t.dtype == torch.uint64:
        t = t.view(torch.int64)
    return t.to(device=dev, dtype=dtype).contiguous()


def move_ids(packed, device=None):
    """Action id of every packed move (include/ddz_b200.h, ddz_move_ids): its index in the universe of 13 551 moves -- the
    reference's action space (card.py) plus the 24 rocket-kicker moves of r.get_moves, id 0 = pass --, or -1 for a value
    that is not a move.  packed int64 / uint64 [...] -> int32 [...] on the device."""
    dev = _id_device(device)
    p = _as_int_tensor(packed, torch.int64, dev)
    out = torch.empty(p.shape, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_move_ids(p.data_ptr(), p.numel(), out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                "ddz_move_ids")
    return out


def moves_of_ids(ids, device=None):
    """The packed move of every action id (ddz_moves_of_ids): int [...] -> int64 [...] on the device; an id outside
    [0, 13551) gives MOVE_INVALID (all bits set, never a legal move)."""
    dev = _id_device(device)
    i = _as_int_tensor(ids, torch.int32, dev)
    out = torch.empty(i.shape, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_moves_of_ids(i.data_ptr(), i.numel(), out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream),
                "ddz_moves_of_ids")
    return out


def action_space(device=None):
    """The whole universe of action ids: moves int64 [13551] (moves[id] = packed move), card_py_index int64 [13551] (the
    move's index in card.py's 13 527-move action space, -1 for the 24 rocket-kicker moves card.py leaves out) and
    id_of_card_py int64 [13527] (the inverse map)."""
    dev = _id_device(device)
    moves = moves_of_ids(torch.arange(N.NUM_ACTION_IDS, dtype=torch.int32, device=dev), dev)
    c = unpack_counts(moves)
    # the rocket-kicker extras are the only moves with both jokers among 6 (4+1+1) or 8 (two-trio 3+1 plane) cards
    extra = (c[:, 13] == 1) & (c[:, 14] == 1) & ((c.sum(-1) == 6) | (c.sum(-1) == 8))
    keep = ~extra
    card_py = torch.where(keep, torch.cumsum(keep.to(torch.int64), 0) - 1, torch.full_like(moves, -1))
    return ActionSpace(moves, card_py, keep.nonzero(as_tuple=True)[0])


# ---------------------------------------------------------------------- B = 1 views (exact reference signatures)
class _RoleDict:
    """history / recent_handout of the reference are dicts role -> float array[15] (envi.py:25-26)."""

    def __init__(self, fn):
        self._fn = fn

    def __getitem__(self, role):
        return np.asarray(self._fn()[int(role)], dtype=np.float64)


class Env(BatchedEnv):
    """Single-env drop-in for reference envi.Env: same attribute names, shapes and return types."""

    _NIBBLE_SHIFTS = (4 * np.arange(15, dtype=np.uint64))[None, :]
    CARD_NAMES = dict(zip(range(3, 18), [str(i) for i in range(3, 11)] + ["J", "Q", "K", "A", "2", "小", "大"]))   # config.py:16-18

    def __init__(self, debug=False, seed=None, device=None):
        self.old_cards = dict()                      # role -> hand before its latest move (envi.py:27, 65)
        self._snap_key, self._snap_val, self._raw = None, None, None
        self._last_results = (0, False, -1)
        self._face_copy = self._acts_copy = None
        self.verbose = bool(debug)                   # envi.py:44-61 narrates every move when debug=True
        super().__init__(1, debug=debug, seed=seed, device=device)
        # Everything the single-env loop of game.py asks for after a decision lives in ONE 160-byte device block -- the
        # state (19 words), both result sets (r | done | cat | reward) and both offset pairs -- mirrored to pinned host
        # memory by one async copy: ONE synchronisation per decision instead of one per getter.
        dev = self.device
        self._blob = torch.zeros(40, dtype=torch.int32, device=dev)
        self._state = self._blob[0:19]
        self._results = [StepResults(1, dev, buf=self._blob[20 + 8 * i:27 + 8 * i].view(torch.uint8)) for i in range(2)]
        self._offsets = [self._blob[36:38], self._blob[38:40]]
        self._mirror = torch.zeros(40, dtype=torch.int32).pin_memory()
        self._mirror_np = self._mirror.numpy()
        self._choice_h = torch.zeros(2, dtype=torch.int32).pin_memory()
        self._choice_d = torch.zeros(2, dtype=torch.int32, device=dev)
        self.reset()

    def reset(self):
        self.old_cards = dict()
        self._snap_val = self._face_copy = self._acts_copy = None
        return super().reset()

    @classmethod
    def cards2str(cls, cards):
        """envi.py:159-161"""
        return [cls.CARD_NAMES[int(i)] for i in cards]

    def _note_move(self, role, before):
        """the bookkeeping of envi.py:38-61 that is visible from outside: old_cards, and the narration of debug mode
        (without the reference's blocking input() prompts)"""
        self.old_cards[role] = before
        if self.verbose:
            name, char = (("上家", "$"), ("地主", "#"), ("下家", "$"))[role]
            played = self.arr2cards(self._snap()["recent"][role])
            print("\n%s %s手牌: %s" % (char, name, self.cards2str(before)))
            print("%s %s出牌： %s，分别剩余： %s" % (char, name, self.cards2str(played), self.left))

    # The reference returns NEW tensors from face / valid_actions (envi.py:96,113): game.py keeps them across later steps
    # (s0, a0 of a transition, game.py:95-127).  The batched buffers are overwritten by the next observation, so the view
    # hands out copies (one per state).
    @property
    def face(self):
        if self._face_copy is None or self._face_copy[0] != self._key():
            f = BatchedEnv.face.fget(self)[0].clone()
            self._face_copy = (self._key(), f)
        return self._face_copy[1]

    def valid_actions(self, tensor=True):
        if not tensor:
            return super().valid_actions(False)[0]
        if self._acts_copy is None or self._acts_copy[0] != self._key():
            a = super().valid_actions(True)[0].clone()
            self._acts_copy = (self._key(), a)
        return self._acts_copy[1]

    def _key(self):
        return (self._stepno, self._games_dealt, self._cur, self._fresh)

    def _refresh_mirror(self, with_results=False):
        """state, results of the latest step and the length of the fresh lists -> host: one copy, one synchronisation"""
        self._mirror.copy_(self._blob, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        host = self._mirror_np
        self._raw = host[:19].copy()
        self._snap_val = None
        self._snap_key = self._key()
        if with_results:
            b = host[20 + 8 * self._res:21 + 8 * self._res].view(np.int8)
            self._last_results = (int(b[0]), bool(b[1]), int(b[2]))
        if self._fresh:
            self._n_total = int(host[37 + 2 * self._cur])

    # One small D2H per state serves every getter of the reference API (role, hands, hand-outs, history, left): the
    # single-env loop of game.py asks for several of them per decision, and each would otherwise be its own sync.
    def _snap(self):
        if self._snap_key != self._key() or self._raw is None:
            self._refresh_mirror()
        if self._snap_val is None:
            cnt = ((self._raw[:18].view(np.uint64)[:, None] >> self._NIBBLE_SHIFTS) & 15).astype(np.int64)
            meta = int(self._raw[18]) & 0xFFFFFFFF
            self._snap_val = {"hand": cnt[0:3], "hist": cnt[3:6], "recent": cnt[6:9], "role": meta & 3,
                              "done": bool((meta >> 2) & 1), "winner": (meta >> 3) & 3, "error": bool((meta >> 5) & 1)}
        return self._snap_val

    def observe(self):
        super().observe()
        self._refresh_mirror()
        return self

    def _decide(self, value, mode):
        """One decision of the single-env loop = ONE launch (apply the move, legal moves + face of the new state:
        ddz_rollout_step without re-deal) and ONE synchronisation.  value: python int (index / entropy / packed move)."""
        self._ensure()
        sn = self._snap()
        role, before = sn["role"], self.arr2cards(sn["hand"][sn["role"]])
        choice = None
        if mode != N.CHOICE_PHILOX:
            self._choice_h.view(torch.int64)[0] = int(value)
            self._choice_d.copy_(self._choice_h, non_blocking=True)
            choice = self._choice_d.view(torch.int64) if mode == N.CHOICE_MOVE else self._choice_d[0:1]
        BatchedEnv.rollout_step(self, choice, mode=mode)
        self._refresh_mirror(with_results=True)
        if self.debug and self._snap()["error"]:
            raise N.DdzError("step: the env flagged an error (illegal choice)")
        self._note_move(role, before)
        return self._last_results

    def step_manual(self, onehot_cards):
        """envi.py:63-70.  A row of valid_actions() (what dqn.py returns) is recognised by its address: no conversion."""
        oh = onehot_cards
        if (torch.is_tensor(oh) and oh.is_cuda and oh.dtype == torch.float32 and oh.numel() == 60 and oh.is_contiguous()
                and self._acts_copy is not None and self._acts_copy[0] == self._key()):
            off = oh.data_ptr() - self._acts_copy[1].data_ptr()
            if 0 <= off < 240 * self._acts_copy[1].shape[0] and off % 240 == 0:
                return self._decide(off // 240, N.CHOICE_INDEX)
        if torch.is_tensor(oh):
            oh = oh.detach().cpu().numpy()
        counts = np.asarray(oh).reshape(15, 4).sum(-1).round().astype(np.int64)
        packed = int((counts.astype(np.uint64) << (4 * np.arange(15, dtype=np.uint64))).sum())
        return self._decide(packed, N.CHOICE_MOVE)

    def step_random(self, entropy=None):
        if entropy is None:
            return self._decide(0, N.CHOICE_PHILOX)
        return self._decide(int(entropy) & 0xFFFFFFFF, N.CHOICE_MOD)

    def prepare(self, *args, **kw):
        self._raw = None
        return super().prepare(*args, **kw)

    def load_state_dict(self, sd):
        self._raw = None
        return super().load_state_dict(sd)

    def get_state_prob(self):
        """native get_state_prob (envi.py:94): float32 [120]"""
        return super().get_state_prob()[0].clone()

    def get_role_ID(self):
        return self._snap()["role"] + 1

    def get_curr_handcards(self):
        sn = self._snap()
        return self.arr2cards(sn["hand"][sn["role"]])

    def get_last_two_cards(self):
        sn = self._snap()
        s = sn["role"]
        return [list(self.arr2cards(sn["recent"][(s + 2) % 3])), list(self.arr2cards(sn["recent"][(s + 1) % 3]))]

    @property
    def left(self):
        return self._snap()["hand"].sum(-1)

    @property
    def taken(self):
        return self._snap()["hist"].sum(0).astype(np.float64)

    @property
    def history(self):
        return _RoleDict(lambda: self._snap()["hist"])

    @property
    def recent_handout(self):
        return _RoleDict(lambda: self._snap()["recent"])


class EnvComplicated(Env):
    VARIANT = N.FACE_COMPLICATED


class EnvCooperation(Env):
    VARIANT = N.FACE_COOPERATION


class EnvCooperationSimplify(Env):
    VARIANT = N.FACE_SIMPLIFY
