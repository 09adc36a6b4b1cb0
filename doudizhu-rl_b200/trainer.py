"""Batched rollout / trainer driver pieces (SURVEY.md 8f rank 2).

Reference: Game.play / Game.step / Game.feedback (game.py:90-181) assemble one transition (s0, a0, r, s1, a1, done) per
decision of a learning role with a DELAYED feedback rule, and DQNFirst.perceive (dqn.py:21-48) pushes it into a
`deque(maxlen=20000)` and does one TD step on a random minibatch.  Here the same assembly runs for all envs at once on
the device, the replay buffer is a ring of GPU tensors, and the TD step is the reference's arithmetic.

The delayed-feedback rule for a learning role R (game.py:128-168):
  * at R's turn it observes s0 = face and plays a0;
  * the NEXT time it is R's turn (nobody finished in between) the pending (s0, a0) is closed with r = 0,
    s1 = the face R sees now, a1 = the greedy action at s1, done = 0;
  * when the game ends first, the pending (s0, a0) is closed with r = +reward if R's side won else -reward,
    s1 = the face after the terminal move (still queried, game.py:121-122), a1 = zeros, done = 1.

Packed replay: a face is a function of the env's 76-byte packed state and an action row of one packed move, so
`PackedReplayBuffer` keeps s0 / s1 as library states and a0 / a1 as packed moves (176 B a transition instead of
2 * 240 * (C + 1) + 8 B) and rebuilds the float rows of a sampled minibatch on the device (ddz_encode_face_gather);
`TransitionCollector(packed=True)` emits transitions in that form.
"""
import torch

from . import _native as N


class ReplayBuffer:
    """Ring buffer of transitions on the GPU (dqn.py:14 deque(maxlen=REPLAY_SIZE), :22-29 sample)."""

    def __init__(self, capacity, face_channels, device):
        self.capacity, self.size, self.head = int(capacity), 0, 0
        dev = torch.device(device)
        self.s0 = torch.zeros((capacity, face_channels, 15, 4), dtype=torch.float32, device=dev)
        self.s1 = torch.zeros_like(self.s0)
        self.a0 = torch.zeros((capacity, 15, 4), dtype=torch.float32, device=dev)
        self.a1 = torch.zeros_like(self.a0)
        self.r = torch.zeros((capacity, 1), dtype=torch.float32, device=dev)
        self.done = torch.zeros((capacity, 1), dtype=torch.float32, device=dev)

    def __len__(self):
        return self.size

    def append(self, s0, a0, r, s1, a1, done):
        """append n transitions (oldest are overwritten, like a bounded deque)"""
        n = s0.shape[0]
        if n == 0:
            return
        if n > self.capacity:
            s0, a0, r, s1, a1, done = (x[-self.capacity:] for x in (s0, a0, r, s1, a1, done))
            n = self.capacity
        idx = (self.head + torch.arange(n, device=self.s0.device)) % self.capacity
        self.s0[idx], self.a0[idx], self.s1[idx], self.a1[idx] = s0, a0, s1, a1
        self.r[idx] = r.reshape(n, 1).to(torch.float32)
        self.done[idx] = done.reshape(n, 1).to(torch.float32)
        self.head = (self.head + n) % self.capacity
        self.size = min(self.capacity, self.size + n)

    def sample(self, batch_size, generator=None):
        idx = torch.randint(0, self.size, (batch_size,), device=self.s0.device, generator=generator)
        return self.s0[idx], self.a0[idx], self.r[idx], self.s1[idx], self.a1[idx], self.done[idx]


def state_fields(state, B):
    """int64 [9, B] (hand[3], hist[3], recent[3]) and int32 meta [B] views of a library state (int32 [19 B], the layout of
    include/ddz_b200.h)"""
    return state[: 18 * B].view(torch.int64).view(9, B), state[18 * B: 19 * B]


def _gather(f, meta, idx):
    n = idx.numel()
    out = torch.empty(N.STATE_WORDS * n, dtype=torch.int32, device=meta.device)
    of, om = state_fields(out, n)
    of.copy_(f[:, idx])
    om.copy_(meta[idx])
    return out


def gather_states(env, idx):
    """library state (int32 [19 n]) of the envs idx of a batched env: their SoA columns and meta, copied"""
    return _gather(*env._fields(), idx)


def decode_rows(state, variant, rows, moves=None, concat=False):
    """ddz_encode_face_gather: the float rows of envs `rows` (int64 [n], any order, duplicates allowed; a row outside [0, B)
    gives zero rows) of a library state of B envs (int32 [19 B]) and of their packed moves (int64 [B], or None).
    concat=False: (face [n, C, 15, 4] = ddz_encode_face's rows, move one-hots [n, 15, 4] or None);
    concat=True: [n, C+1, 15, 4] = the Q-network input of net.py:88-90 (needs moves)."""
    dev = state.device
    if dev.type != "cuda":
        raise N.DdzError("decoding packed states needs a CUDA device: the rows are built by an sm_100a kernel")
    C = N.lib.ddz_face_channels(int(variant))
    if C < 0:
        raise ValueError("unknown face variant %r" % (variant,))
    B = state.numel() // N.STATE_WORDS
    rows = rows.to(device=dev, dtype=torch.int64).contiguous()
    n = rows.numel()
    face = torch.empty((n, C + 1 if concat else C, 15, 4), dtype=torch.float32, device=dev)
    mv = torch.empty((n, 15, 4), dtype=torch.float32, device=dev) if moves is not None and not concat else None
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_encode_face_gather(state.data_ptr(), int(variant), rows.data_ptr(), n,
                                             None if moves is None else moves.data_ptr(), face.data_ptr(),
                                             None if mv is None else mv.data_ptr(),
                                             N.ROWS_CONCAT if concat else N.ROWS_SPLIT, B,
                                             torch.cuda.current_stream(dev).cuda_stream), "ddz_encode_face_gather")
    return face if concat else (face, mv)


class PackedReplayBuffer:
    """ReplayBuffer's ring with every transition kept packed: s0 / s1 as library states, a0 / a1 as packed moves, r and done
    as floats.  sample() draws the same indices as ReplayBuffer.sample and returns the same float 6-tuple, rebuilt on the
    device for the sampled rows only (one ddz_encode_face_gather launch), so td_step is unchanged."""

    bytes_per_transition = 2 * 4 * N.STATE_WORDS + 2 * 8 + 4 + 4      # 176 B (the float ring: 2 * 240 * (C + 1) + 8 B)

    def __init__(self, capacity, variant, device):
        self.capacity, self.size, self.head = int(capacity), 0, 0
        self.variant = int(variant)
        self.face_channels = N.lib.ddz_face_channels(self.variant)
        if self.face_channels < 0:
            raise ValueError("unknown face variant %r" % (variant,))
        cap, dev = self.capacity, torch.device(device)
        # ONE library state of 2 cap envs, so the kernel reads it directly: s0 of slot i is env i, s1 is env cap + i
        self.state = torch.zeros(N.STATE_WORDS * 2 * cap, dtype=torch.int32, device=dev)
        self.moves = torch.zeros(2 * cap, dtype=torch.int64, device=dev)      # a0 of slot i at i, a1 at cap + i
        self.r = torch.zeros((cap, 1), dtype=torch.float32, device=dev)
        self.done = torch.zeros((cap, 1), dtype=torch.float32, device=dev)
        self._f, self._meta = state_fields(self.state, 2 * cap)

    def __len__(self):
        return self.size

    def append(self, s0, a0, r, s1, a1, done):
        """append n transitions as TransitionCollector(packed=True) emits them: s0 / s1 library states of n envs (int32
        [19 n]), a0 / a1 packed moves (int64 [n]), r / done [n] (oldest are overwritten, like ReplayBuffer)"""
        n = a0.shape[0]
        if n == 0:
            return
        f0, m0 = state_fields(s0, n)
        f1, m1 = state_fields(s1, n)
        cap = self.capacity
        if n > cap:
            f0, m0, f1, m1 = f0[:, n - cap:], m0[n - cap:], f1[:, n - cap:], m1[n - cap:]
            a0, r, a1, done = (x[-cap:] for x in (a0, r, a1, done))
            n = cap
        idx = (self.head + torch.arange(n, device=self.state.device)) % cap
        self._f[:, idx], self._meta[idx] = f0, m0
        self._f[:, idx + cap], self._meta[idx + cap] = f1, m1
        self.moves[idx], self.moves[idx + cap] = a0, a1
        self.r[idx] = r.reshape(n, 1).to(torch.float32)
        self.done[idx] = done.reshape(n, 1).to(torch.float32)
        self.head = (self.head + n) % cap
        self.size = min(cap, self.size + n)

    def decode(self, idx):
        """the float transitions (s0, a0, r, s1, a1, done) of slots idx, as ReplayBuffer holds them"""
        idx = idx.to(self.state.device, torch.int64)
        m = idx.numel()
        face, rows = decode_rows(self.state, self.variant, torch.cat((idx, idx + self.capacity)), self.moves)
        return face[:m], rows[:m], self.r[idx], face[m:], rows[m:], self.done[idx]

    def sample(self, batch_size, generator=None):
        idx = torch.randint(0, self.size, (batch_size,), device=self.state.device, generator=generator)
        return self.decode(idx)


def td_step(policy_net, target_net, optimizer, batch, gamma):
    """one minibatch update with the reference's arithmetic (dqn.py:39-47): y = r + (1 - done) * gamma * Q_target(s1, a1),
    MSE against Q_policy(s0, a0)."""
    s0, a0, r, s1, a1, done = batch
    with torch.no_grad():
        y_true = r + (1 - done) * gamma * target_net(s1, a1)
    loss = torch.nn.functional.mse_loss(policy_net(s0, a0), y_true)
    optimizer.zero_grad()
    loss.backward()
    optimizer.step()
    return loss.detach()


class TransitionCollector:
    """Delayed-feedback transition assembly for one learning role over a batched env (game.py:109-168)."""

    def __init__(self, env, role=1, reward=100.0, packed=False):
        """packed=True: the pending s0 is kept as the env's packed state and a0 as a packed move; on_turn takes packed moves
        int64 [B] and both calls return (s0_states, a0_u64, r, s1_states, a1_u64, done, env_index) with library states of
        n envs (int32 [19 n]), the input of PackedReplayBuffer.append."""
        self.env, self.role, self.reward = env, int(role), float(reward)
        self.packed = bool(packed)
        B, C, dev = env.B, env.C, env.device
        if self.packed:
            self.s0 = torch.zeros(N.STATE_WORDS * B, dtype=torch.int32, device=dev)     # a library state of B envs
            self.a0 = torch.zeros(B, dtype=torch.int64, device=dev)
        else:
            self.s0 = torch.zeros((B, C, 15, 4), dtype=torch.float32, device=dev)
            self.a0 = torch.zeros((B, 15, 4), dtype=torch.float32, device=dev)
        self.pending = torch.zeros(B, dtype=torch.bool, device=dev)

    def on_turn(self, a0, a1):
        """Call BEFORE stepping, with the env observed.  a0 [B,15,4]: the action each env is about to play (used where it is
        the role's turn); a1 [B,15,4]: the greedy action at the current state (the reference evaluates it separately,
        game.py:125).  Returns the transitions closed by this turn: (s0, a0, r, s1, a1, done, env_index)."""
        if self.packed:
            return self._on_turn_packed(a0, a1)
        env = self.env
        mine = ((env.get_role_ID() - 1) == self.role) & ~env.is_done
        close = mine & self.pending
        idx = close.nonzero(as_tuple=True)[0]
        face = env.face
        out = (self.s0[idx].clone(), self.a0[idx].clone(), torch.zeros(idx.numel(), device=face.device),
               face[idx].clone(), a1[idx].clone(), torch.zeros(idx.numel(), device=face.device), idx)
        m = mine.nonzero(as_tuple=True)[0]
        self.s0[m], self.a0[m] = face[m], a0[m]
        self.pending |= mine
        return out

    def _on_turn_packed(self, a0, a1):
        env = self.env
        mine = ((env.get_role_ID() - 1) == self.role) & ~env.is_done
        close = mine & self.pending
        idx = close.nonzero(as_tuple=True)[0]
        f0, m0 = state_fields(self.s0, env.B)
        f, meta = env._fields()
        zeros = torch.zeros(idx.numel(), device=meta.device)
        out = (_gather(f0, m0, idx), self.a0[idx], zeros, _gather(f, meta, idx), a1[idx], zeros.clone(), idx)
        m = mine.nonzero(as_tuple=True)[0]
        f0[:, m], m0[m], self.a0[m] = f[:, m], meta[m], a0[m]
        self.pending |= mine
        return out

    def on_step_done(self, done_now):
        """Call AFTER stepping WITHOUT re-deal and after env.observe(): done_now bool [B] = envs that finished with this
        step.  Closes their pending transition with the terminal reward; env.face is the face after the terminal move."""
        env = self.env
        close = done_now & self.pending
        idx = close.nonzero(as_tuple=True)[0]
        winner = env.winner[idx]
        won = (winner == 1) if self.role == 1 else (winner != 1)
        r = torch.where(won, torch.full_like(won, self.reward, dtype=torch.float32),
                        torch.full_like(won, -self.reward, dtype=torch.float32))
        if self.packed:
            n, dev = idx.numel(), r.device
            out = (_gather(*state_fields(self.s0, env.B), idx), self.a0[idx], r, gather_states(env, idx),
                   torch.zeros(n, dtype=torch.int64, device=dev), torch.ones(n, device=dev), idx)
            self.pending &= ~done_now
            return out
        face = env.face
        out = (self.s0[idx].clone(), self.a0[idx].clone(), r, face[idx].clone(),
               torch.zeros((idx.numel(), 15, 4), device=face.device), torch.ones(idx.numel(), device=face.device), idx)
        self.pending &= ~done_now
        return out
