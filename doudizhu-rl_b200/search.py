"""UCT search on the batched env (SURVEY.md 8f rank 4): the reference's search bot, `mcts(payload)`
(server/mcts/interface.py:15-45), with the device doing what costs time.

The reference algorithm, kept as it is:
  * `computation_budget` iterations of  tree policy -> default policy -> back-up  (interface.py:37-41);
  * tree policy (tree_policy.py:4-13): walk down while the node is fully expanded, choosing the child with the highest
    UCB value when the node's player is the searching player and the LOWEST otherwise (get_bestchild.py:4-33,
    value = reward/visit + 0.7 * sqrt(2 ln(parent visits) / visit)); at the first node with an untried move, expand ONE
    untried move chosen at random (tree.py:28-52) and stop there;
  * default policy (default_policy.py:4-10): uniformly random legal moves until somebody is out of cards; the reward is 1
    when the searching player's side has won (tree.py:71-81);
  * back-up (backup.py:1-5): visit += 1, reward += reward on the path to the root;
  * answer: the root child with the best reward / visit (get_bestchild_.py:35-42).

  * both the tree and the default policy take their moves from the bot's OWN move list, mcts.get_moves.get_moves
    (get_moves.py:36-69; tree.py:33,86): a list of more than 10 moves loses its rocket-kicker moves, is ranked by
    cards_value - 0.1 * cards left (evaluator.py:17-57) and keeps its lowest- and highest-valued thirds.  `prune=True`
    (the default) does the same; `prune=False` searches and plays over the full r.get_moves lists.

What runs where: a node's move list comes from ddz_mcts_moves (ddz_legal_moves without pruning), the default policy is
ddz_playout_pruned (ddz_playout) -- `width` random playouts of the expanded node in one launch (Philox stream keyed by the
iteration), backed up as `width` visits; width = 1 is the reference's sequential search.  The tree itself (a few thousand
nodes, pointer chasing) stays on the host.
Exact ties are broken at random among the tied candidates, as the reference does with np.random.choice
(get_bestchild.py:8,17,37 -- with one visit per child most of a young node's children tie), and the untried move to
expand is drawn at random (tree.py:42); both draws come from ONE seeded numpy generator, so with the same seed the search
is reproducible, and the same algorithm written over the CPU restatement of the env (tests/uct_reference_algorithm.py)
picks the same move.
"""
import math

import numpy as np
import torch

from . import _native as N
from .deals import pack_counts_np
from .env import BatchedEnv, MoveGenerator

UCB_C = 0.7                      # get_bestchild.py:4
_LN = {}                         # device -> ln table (float64, grown on demand)
_WS = {}                         # (device, stream) -> search workspace (grown on demand, kept until release_workspaces())


class _Node:
    __slots__ = ("parent", "children", "reward", "visit", "hands", "recent", "cur", "winner", "action", "untried", "nmoves")

    def __init__(self, parent, hands, recent, cur, winner, action):
        self.parent, self.children, self.reward, self.visit = parent, [], 0.0, 0
        self.hands, self.recent, self.cur, self.winner, self.action = hands, recent, cur, winner, action
        self.untried, self.nmoves = None, None


def _trick(recent, cur):
    """the hand-out to beat: previous player's, else the one before (envi.py:103-110)"""
    p = recent[(cur + 2) % 3]
    return p if p.any() else recent[(cur + 1) % 3]


class UctSearch:
    def __init__(self, role, hands, last_taken, width=1, c=UCB_C, seed=1, device=None, prune=True):
        if not torch.cuda.is_available():
            raise N.DdzError("UctSearch needs a CUDA device")
        self.me = int(role)
        self.width, self.c, self.seed, self.prune = int(width), float(c), int(seed), bool(prune)
        self.rng = np.random.Generator(np.random.PCG64(self.seed))
        self.env = BatchedEnv(self.width, seed=self.seed if self.seed else None, device=device)
        self.env.seed = self.seed
        self.dev = self.env.device
        self.gen = MoveGenerator(1, device=self.dev)
        self._pair = torch.zeros(2, dtype=torch.int64).pin_memory()
        self._pair_d = torch.zeros(2, dtype=torch.int64, device=self.dev)
        self._list_d = torch.zeros(N.MCTS_MAX_MOVES + 1, dtype=torch.int64, device=self.dev)     # pruned list | its length
        self._list_h = torch.zeros(N.MCTS_MAX_MOVES + 1, dtype=torch.int64).pin_memory()
        self._state_h = torch.zeros(10, dtype=torch.int64).pin_memory()
        self._state_d = torch.zeros(10, dtype=torch.int64, device=self.dev)
        hands = np.asarray(hands, np.int64).reshape(3, 15).copy()
        recent = np.asarray(last_taken, np.int64).reshape(3, 15).copy()
        self.root = _Node(None, hands, recent, self.me, -1, None)
        self.iterations = 0
        self.playouts = 0

    # ------------------------------------------------------------------ device work
    def _legal_moves(self, node):
        """int64 [n,15]: the move list of the player to move against the trick to beat -- the bot's pruned list in the
        reference's order, or r.get_moves in canonical order"""
        self._pair[0] = int(pack_counts_np(node.hands[node.cur]).astype(np.int64))
        self._pair[1] = int(pack_counts_np(_trick(node.recent, node.cur)).astype(np.int64))
        self._pair_d.copy_(self._pair, non_blocking=True)
        if self.prune:
            count = self._list_d[N.MCTS_MAX_MOVES:].view(torch.int32)
            with torch.cuda.device(self.dev):
                N.check(N.lib.ddz_mcts_moves(self._pair_d[0:1].data_ptr(), self._pair_d[1:2].data_ptr(),
                                             self._list_d.data_ptr(), count.data_ptr(), 1,
                                             torch.cuda.current_stream(self.dev).cuda_stream), "ddz_mcts_moves")
            self._list_h.copy_(self._list_d, non_blocking=True)
            torch.cuda.current_stream(self.dev).synchronize()
            n = int(self._list_h[N.MCTS_MAX_MOVES:].view(torch.int32)[0])
            packed = self._list_h[:n].numpy().view(np.uint64).copy()
        else:
            acts, offs = self.gen.generate(self._pair_d[0:1], self._pair_d[1:2])
            n = int(offs[1].item())
            packed = acts[:n].cpu().numpy().view(np.uint64)
        return ((packed[:, None] >> (np.arange(15, dtype=np.uint64) * np.uint64(4))) & np.uint64(15)).astype(np.int64)

    def _default_policy(self, node, it):
        """`width` random playouts of `node` in one launch; returns the number the searching side won"""
        if node.winner >= 0:
            return float(self.width) * self._won(node.winner)
        env, W = self.env, self.width
        self._state_h[0:3] = torch.as_tensor(pack_counts_np(node.hands).astype(np.int64))
        self._state_h[3:6] = 0
        self._state_h[6:9] = torch.as_tensor(pack_counts_np(node.recent).astype(np.int64))
        self._state_h[9] = node.cur
        self._state_d.copy_(self._state_h, non_blocking=True)
        f, meta = env._fields()
        f.copy_(self._state_d[0:9, None].expand(9, W))
        meta.copy_(self._state_d[9:10].expand(W).to(torch.int32))
        env._fresh = False
        env.env0, env._stepno = it * W, 0            # Philox counters of this iteration's playouts
        env.playout(max_steps=400, policy="search" if self.prune else "uniform")
        winner = (env._fields()[1] >> 3) & 3
        lord_won = int((winner == 1).sum().item())
        self.playouts += W
        return float(lord_won if self.me == 1 else W - lord_won)

    def _won(self, winner):
        return 1.0 if (winner == 1) == (self.me == 1) else 0.0          # tree.py:71-81: the farmers win together

    # ------------------------------------------------------------------ the tree (host)
    def _expand(self, node):
        i = int(self.rng.integers(len(node.untried)))
        mv = node.untried.pop(i)
        hands, recent = node.hands.copy(), node.recent.copy()
        hands[node.cur] -= mv
        recent[node.cur] = mv
        winner = node.cur if mv.any() and not hands[node.cur].any() else -1
        child = _Node(node, hands, recent, (node.cur + 1) % 3, winner, mv)
        node.children.append(child)
        return child

    def _best_child(self, node):
        visit = np.array([ch.visit for ch in node.children], np.float64)
        reward = np.array([ch.reward for ch in node.children], np.float64)
        values = reward / visit + self.c * np.sqrt(2.0 * math.log(node.visit) / visit)
        return node.children[self._pick(values, values.max() if node.cur == self.me else values.min())]

    def _pick(self, values, target):
        """index of the entry equal to `target`; a random one of them when several tie (get_bestchild.py:8-17)"""
        tied = np.flatnonzero(values == target)
        return int(tied[0] if len(tied) == 1 else tied[self.rng.integers(len(tied))])

    def _tree_policy(self):
        node = self.root
        while node.winner < 0:
            if node.untried is None:
                moves = self._legal_moves(node)
                node.untried, node.nmoves = [m for m in moves], len(moves)
            if len(node.children) < node.nmoves:
                return self._expand(node)
            node = self._best_child(node)
        return node

    def run(self, computation_budget=1000):
        for _ in range(int(computation_budget)):
            node = self._tree_policy()
            reward = self._default_policy(node, self.iterations)
            while node is not None:                      # backup.py
                node.visit += self.width
                node.reward += reward
                node = node.parent
            self.iterations += 1
        return self

    def root_table(self):
        """(moves int64 [n,15], visits [n], win rate [n]) of the root's children in expansion order"""
        ch = self.root.children
        return (np.stack([c.action for c in ch]), np.array([c.visit for c in ch]),
                np.array([c.reward / c.visit for c in ch]))

    def best_move(self):
        """get_bestchild_: the root child with the best reward / visit (a random one of them on ties, get_bestchild.py:35-42);
        counts int64 [15].  Consumes the generator when there is a tie: call it once."""
        moves, _, rate = self.root_table()
        return moves[self._pick(rate, rate.max())]


# ---------------------------------------------------------------------------------------------------- batched search
def _ln_table(n, device):
    """float64 [>= n + 1] on `device`: ln_table[k] = math.log(k) (the C library's log, correctly rounded where the device's
    is not; entry 0 is never read and holds 0)"""
    t = _LN.get(device)
    if t is None or t.numel() < n + 1:
        t = torch.tensor([0.0] + [math.log(k) for k in range(1, n + 1)], dtype=torch.float64, device=device)
        _LN[device] = t
    return t


def _workspace(nbytes, device, stream):
    """the cached workspace of `stream`: one per stream, because a launch owns its workspace until it ends, so searches
    on two concurrent streams must not share one"""
    key = (device, stream)
    t = _WS.get(key)
    if t is None or t.numel() < nbytes:
        _WS.pop(key, None)
        t = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=device)
        _WS[key] = t
    return t


def release_workspaces():
    """free the workspaces uct_search keeps for reuse: (B x (budget + 1) x 160 bytes each, e.g. 5.2 GB after a search
    of 32 768 roots at budget 1000)"""
    _WS.clear()


def _check_budget(computation_budget, width):
    """(budget, width) as ints, or ValueError outside ddz_uct_search's bounds"""
    budget, width = int(computation_budget), int(width)
    if not (1 <= budget <= N.UCT_MAX_BUDGET and 1 <= width <= N.UCT_MAX_WIDTH and budget * width <= N.UCT_MAX_PLAYOUTS):
        raise ValueError("need 1 <= budget <= %d, 1 <= width <= %d and budget * width <= %d"
                         % (N.UCT_MAX_BUDGET, N.UCT_MAX_WIDTH, N.UCT_MAX_PLAYOUTS))
    return budget, width


def _device_mask(env_mask, B, dev):
    """env_mask (bool [B] or None) as a contiguous uint8 tensor on `dev`"""
    mask = None if env_mask is None else torch.as_tensor(env_mask).to(dev, torch.bool).to(torch.uint8).contiguous()
    if mask is not None and mask.numel() != B:
        raise ValueError("env_mask must have B entries")
    return mask


def _p(t):
    return None if t is None else t.data_ptr()


def uct_search(env, computation_budget=1000, width=1, prune=True, c=UCB_C, seed=1, env_mask=None, root_table=False,
               workspace=None):
    """The search bot for every env of a BatchedEnv* in ONE launch (ddz_uct_search): root b is env b's position (all three
    hands: full information), the searching player its role to move.  `computation_budget` iterations of the reference's
    UCT (the same algorithm as UctSearch: UCB1 max for the searching player and min for the others, one expansion per
    iteration, `width` random playouts of the expanded node, back-up, answer = root child with the best win rate), with
    the bot's pruned move lists unless prune=False.  Every draw comes from Philox keyed by (seed, env.env0 + b), so a batch
    split into chunks by env0 searches the same trees.  env_mask (bool [B]): only those envs are searched.
    Returns (choice int32 [B], moves int64 [B]): the index of the chosen move in env.valid_actions() -- feed it to
    env.step() -- and the packed move; -1 / ~0 for an env that is finished or masked out.  root_table=True adds
    (root_n int32 [B], root_moves int64 [B,S], root_visits int32 [B,S], root_wins int32 [B,S]), the root's children in
    expansion order (S = min(budget, 512)).  The env's state, step counter and lists are left as they are.
    The search tree lives in a workspace of ddz_uct_workspace_bytes(B, budget) bytes: `workspace` (a device uint8 tensor
    of at least that size, owned by the caller) or, by default, one cached per stream and kept for the next call (free
    the cache with release_workspaces())."""
    budget, width = _check_budget(computation_budget, width)
    B, dev = env.B, env.device
    with torch.cuda.device(dev):
        ln = _ln_table(budget * width, dev)
        stream = torch.cuda.current_stream(dev)
        need = N.lib.ddz_uct_workspace_bytes(B, budget)
        if workspace is None:
            ws = _workspace(need, dev, stream.cuda_stream)
        else:
            ws = workspace
            if ws.device != dev or ws.dtype != torch.uint8 or not ws.is_contiguous() or ws.numel() < need:
                raise ValueError("workspace must be a contiguous uint8 tensor of at least %d bytes on %s" % (need, dev))
        mask = _device_mask(env_mask, B, dev)
        choice = torch.empty(B, dtype=torch.int32, device=dev)
        moves = torch.empty(B, dtype=torch.int64, device=dev)
        S = min(budget, N.MAX_LEGAL)
        tab = None
        if root_table:
            tab = (torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros((B, S), dtype=torch.int64, device=dev),
                   torch.zeros((B, S), dtype=torch.int32, device=dev), torch.zeros((B, S), dtype=torch.int32, device=dev))
        N.check(N.lib.ddz_uct_search(_p(env._state), _p(mask), ws.data_ptr(), budget, width, int(bool(prune)), float(c),
                                     ln.data_ptr(), int(seed), env.env0, choice.data_ptr(), moves.data_ptr(),
                                     *(_p(t) for t in (tab or (None,) * 4)), S if root_table else 0, B,
                                     stream.cuda_stream), "ddz_uct_search")
    return (choice, moves) + ((tab,) if root_table else ())


# ---------------------------------------------------------------------------------------------------- determinized search
def _check_determinizations(determinizations, B):
    D = int(determinizations)
    if not 1 <= D <= N.PIMC_MAX_DETERMINIZATIONS:
        raise ValueError("need 1 <= determinizations <= %d" % N.PIMC_MAX_DETERMINIZATIONS)
    if B * D > 2 ** 31 - 1:
        raise ValueError("B x determinizations must stay below 2^31")
    return D


def _state_slice(env, b0, n):
    """a state buffer of its own holding envs b0 .. b0 + n - 1 of env (the state is struct-of-arrays, so a range of envs
    is not a contiguous part of it); the whole state when the range is the whole batch"""
    if b0 == 0 and n == env.B:
        return env._state
    out = torch.empty(N.lib.ddz_state_bytes(n) // 4, dtype=torch.int32, device=env.device)
    f, meta = env._fields()
    out[: 18 * n].view(torch.int64).view(9, n).copy_(f[:, b0:b0 + n])
    out[18 * n: 19 * n].copy_(meta[b0:b0 + n])
    return out


def determinize(env, determinizations, seed=1, env_mask=None):
    """ddz_determinize: the raw state (int32 tensor of ddz_state_bytes(B * D) bytes) of B * D full-information envs, env
    b * D + d being determinization d of env b -- its mover's hand, hist, recent and meta, the two hidden hands replaced by
    a uniformly random split of the cards the mover has not seen (Philox keyed by (seed, (env.env0 + b) * D + d)).
    Masked-out and finished envs are copied unchanged; envs no deal agrees with are copied as finished with the sticky error
    bit and counted in env.stats[7]."""
    B, dev = env.B, env.device
    D = _check_determinizations(determinizations, B)
    with torch.cuda.device(dev):
        out = torch.empty(N.lib.ddz_state_bytes(B * D) // 4, dtype=torch.int32, device=dev)
        mask = _device_mask(env_mask, B, dev)
        N.check(N.lib.ddz_determinize(env._state.data_ptr(), _p(mask), D, int(seed), env.env0, out.data_ptr(),
                                      env.stats.data_ptr(), B, torch.cuda.current_stream(dev).cuda_stream), "ddz_determinize")
    return out


def pimc_search(env, determinizations=16, computation_budget=1000, width=1, prune=True, c=UCB_C, seed=1, env_mask=None,
                pooled_table=False, max_workspace_bytes=2 ** 31):
    """The search bot from the player's own view (determinized UCT, perfect-information Monte Carlo): for every env of a
    BatchedEnv*, `determinizations` (D) complete deals that agree with what the player to move has seen -- its own hand,
    the cards every role has played, the last hand-outs and the sizes of the other two hands -- each searched as a
    full-information game by uct_search's algorithm, and the root statistics added up per move.  The real hidden hands
    are never read: two envs that show the same view get the same answer.
    Returns (choice int32 [B], moves int64 [B]) with uct_search's conventions (feed choice to env.step(); -1 / ~0 for an
    env that is masked out, finished, or whose view no deal agrees with -- the last are counted in env.stats[7]);
    pooled_table=True adds (pooled_visits, pooled_wins), int32 [B, 512] in the order of env.valid_actions().  The answer is
    the move with the best pooled wins / visits, the lowest list index on exact ties.
    Roots are searched in chunks of Bc, Bc x D x (budget + 1) x 160 <= max_workspace_bytes (at least one root per chunk);
    the results do not depend on the chunking.  The env's state, step counter and lists are left as they are."""
    budget, width = _check_budget(computation_budget, width)
    B, dev = env.B, env.device
    D = _check_determinizations(determinizations, 1)
    if D * budget * width > 2 ** 31 - 1:
        raise ValueError("determinizations x budget x width must stay below 2^31 (pooled int32 counts)")
    Bc = max(1, min(B, int(max_workspace_bytes) // (D * (budget + 1) * N.UCT_NODE_BYTES), (2 ** 31 - 1) // D))
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        ln = _ln_table(budget * width, dev)
        mask = _device_mask(env_mask, B, dev)
        ws = _workspace(N.lib.ddz_uct_workspace_bytes(Bc * D, budget), dev, stream)
        sub = torch.empty(N.lib.ddz_state_bytes(Bc * D) // 4, dtype=torch.int32, device=dev)
        tree_choice = torch.empty(Bc * D, dtype=torch.int32, device=dev)
        choice = torch.empty(B, dtype=torch.int32, device=dev)
        moves = torch.empty(B, dtype=torch.int64, device=dev)
        tab = None
        if pooled_table:
            tab = tuple(torch.empty((B, N.MAX_LEGAL), dtype=torch.int32, device=dev) for _ in range(2))
        for b0 in range(0, B, Bc):
            n = min(Bc, B - b0)
            m = None if mask is None else mask[b0:b0 + n]
            env0 = (env.env0 + b0) & (2 ** 64 - 1)
            N.check(N.lib.ddz_determinize(_state_slice(env, b0, n).data_ptr(), _p(m), D, int(seed), env0, sub.data_ptr(),
                                          env.stats.data_ptr(), n, stream), "ddz_determinize")
            N.check(N.lib.ddz_uct_search(sub.data_ptr(), _p(None if m is None else m.repeat_interleave(D)), ws.data_ptr(),
                                         budget, width, int(bool(prune)), float(c), ln.data_ptr(), int(seed),
                                         (env0 * D) & (2 ** 64 - 1), tree_choice.data_ptr(), None, None, None, None, None,
                                         0, n * D, stream), "ddz_uct_search")
            N.check(N.lib.ddz_uct_pool(ws.data_ptr(), budget, D, choice[b0:].data_ptr(), moves[b0:].data_ptr(),
                                       *(None if t is None else t[b0:].data_ptr() for t in (tab or (None, None))), n,
                                       stream), "ddz_uct_pool")
    return (choice, moves) + ((tab,) if pooled_table else ())
