"""Batched UCT search on the device (ddz_uct_search, search.uct_search, ingest.mcts_batch): the reference's search bot
(server/mcts/interface.py:37-45) for a whole batch of positions in one launch, with Philox draws.

CPU: the readable restatement (uct_philox_reference.uct) and the C port over the oracle (ddz_ref_uct_batch) build identical
trees; the argument checks of both entry points.  GPU: the kernel's whole trees, read back from the workspace, equal the C
port's bit for bit, over many position families, widths, budgets and batch shapes; the Python entry points; an end-to-end
match against random farmers."""
import numpy as np
import pytest

from uct_philox_reference import ref_uct_batch, uct

Z = np.zeros((3, 15), np.int64)
DECK = np.array([i // 4 for i in range(52)] + [13, 14])


# ------------------------------------------------------------------ positions (hands [3,15], recent [3,15], role)
def uct_test_positions():
    """the four positions of test_uct_search_equals_reference_algorithm_on_oracle"""
    out = []
    h = np.zeros((3, 15), np.int64); h[1, [0, 1, 2, 3, 4, 9]] = [1, 1, 1, 1, 1, 2]; h[2, [5, 6]] = 2; h[0, [10, 11, 12]] = [1, 2, 1]
    out.append((h, Z.copy(), 1))
    h2 = np.zeros((3, 15), np.int64); h2[2, [7, 8, 12]] = [2, 1, 1]; h2[0, [0, 3]] = [1, 2]; h2[1, [1, 5, 13]] = [1, 1, 1]
    last = Z.copy(); last[1, 6] = 2
    out.append((h2, last, 2))
    rng = np.random.default_rng(4)
    p = rng.permutation(DECK)[:21]
    out.append((np.stack([np.bincount(p[a:b], minlength=15) for a, b in ((0, 7), (7, 15), (15, 21))]).astype(np.int64), Z.copy(), 0))
    p = rng.permutation(DECK)[:45]
    out.append((np.stack([np.bincount(p[a:b], minlength=15) for a, b in ((0, 14), (14, 31), (31, 45))]).astype(np.int64), Z.copy(), 1))
    return out


def random_positions(oracle, rng, n, lo=2, hi=12, follow=0.5):
    """n positions: three random hands of lo..hi-1 cards, a random role to move; with probability `follow` the previous
    player's last hand-out is a random move of its list from the lead (the role to move must beat it or pass)"""
    out = []
    while len(out) < n:
        sizes = rng.integers(lo, hi, 3)
        p = rng.permutation(DECK)
        hands = np.stack([np.bincount(p[s:s + k], minlength=15) for s, k in zip((0, 20, 40), sizes)]).astype(np.int64)
        role = int(rng.integers(3))
        recent = Z.copy()
        if rng.random() < follow:
            prev = (role + 2) % 3
            mv = oracle.get_moves(hands[prev], np.zeros(15, np.int8), fast=True)
            m = mv[rng.integers(len(mv))].astype(np.int64)
            if m.sum() and (hands[prev] - m).sum():          # a real hand-out that leaves the previous player in the game
                recent[prev] = m
                hands[prev] -= m
        out.append((hands, recent, role))
    return out


def run_python(oracle, positions, budget, width, prune, seed, env0=0):
    res = []
    for b, (hands, recent, role) in enumerate(positions):
        best, nodes = uct(oracle, role, hands, recent, budget, width=width, seed=seed, prune=prune, env=env0 + b)
        ids = {id(n): k for k, n in enumerate(nodes)}
        res.append({"best": best, "nodes": nodes, "ids": ids})
    return res


def sibling_pos(parent):
    pos, seen = np.zeros(len(parent), np.int64), {}
    for k, p in enumerate(parent):
        pos[k] = seen.get(p, 0)
        seen[p] = pos[k] + 1
    return pos


def assert_python_equals_c(oracle, positions, budget, width, prune, seed):
    B = len(positions)
    hands = np.stack([p[0] for p in positions]); recent = np.stack([p[1] for p in positions])
    cur = np.array([p[2] for p in positions]); live = np.ones(B, bool)
    got = ref_uct_batch(hands, recent, cur, live, budget, width=width, prune=prune, seed=seed)
    want = run_python(oracle, positions, budget, width, prune, seed)
    for b, w in enumerate(want):
        nodes = w["nodes"]
        n = len(nodes)
        assert got["nnodes"][b] == n, (b, budget, width, prune)
        parent = np.array([-1] + [w["ids"][id(x.parent)] for x in nodes[1:]])
        where = (b, budget, width, prune)
        assert np.array_equal(got["parent"][b, :n], parent), where
        assert np.array_equal(sibling_pos(got["parent"][b, :n]), sibling_pos(parent)), where
        assert np.array_equal(got["visits"][b, :n], [x.visit for x in nodes]), where
        assert np.array_equal(got["wins"][b, :n], [x.reward for x in nodes]), where
        assert np.array_equal(got["index"][b, :n], [x.index for x in nodes]), where
        moves = [0] + [oracle.pack(x.state.action) for x in nodes[1:]]
        assert np.array_equal(got["node_move"][b, :n], np.array(moves, np.uint64)), where
        root = nodes[0]
        assert got["root_n"][b] == len(root.children), where
        assert np.array_equal(got["parent"][b, 1:1 + len(root.children)], np.zeros(len(root.children))), where
        assert got["move"][b] == oracle.pack(w["best"]), where
        best = next(x for x in root.children if np.array_equal(x.state.action, w["best"]))
        assert got["choice"][b] == best.index, where
    return got


# ------------------------------------------------------------------ CPU
def test_python_restatement_equals_c_port(oracle):
    """uct_philox_reference.uct (Python over the oracle) and ddz_ref_uct_batch (C over the oracle): identical trees (parent,
    move, visits, wins, canonical index, position among siblings), root tables and answers"""
    rng = np.random.default_rng(20)
    positions = uct_test_positions()[:3] + random_positions(oracle, rng, 13)
    assert any(p[1].any() for p in positions) and any(not p[1].any() for p in positions)
    assert {p[2] for p in positions} == {0, 1, 2}
    for budget in (1, 7, 60):
        for width in (1, 3):
            for prune in (True, False):
                assert_python_equals_c(oracle, positions, budget, width, prune, seed=3 + budget)


def test_c_port_prunes_long_lists(oracle):
    """a mid-game position whose lists are longer than 10 moves: the pruned and the full search differ at the root"""
    h, recent, role = uct_test_positions()[3]
    assert len(oracle.get_moves(h[role], np.zeros(15, np.int8), fast=True)) > 10
    got = {prune: assert_python_equals_c(oracle, [(h, recent, role)], 12, 1, prune, seed=5) for prune in (True, False)}
    assert got[True]["root_n"][0] == 12 and got[False]["root_n"][0] == 12
    assert not np.array_equal(got[True]["node_move"][0, 1:13], got[False]["node_move"][0, 1:13])


def test_uct_argument_checks():
    """both entry points check their arguments before any CUDA call (DDZ_E_ARG without a device)"""
    import ddz_b200 as D
    L, E = D.native.lib, D.native.E_ARG
    node = D.native.UCT_NODE_BYTES
    assert node == 160
    for B, budget in ((1, 1), (3, 7), (1000, 1000), (65, 65536)):
        assert L.ddz_uct_workspace_bytes(B, budget) == (4 * B + 255) // 256 * 256 + B * (budget + 1) * node
    assert L.ddz_uct_workspace_bytes(0, 10) == 0 and L.ddz_uct_workspace_bytes(4, 0) == 0
    assert L.ddz_uct_workspace_bytes(4, 65537) == 0

    def call(state=1, mask=None, ws=1, budget=10, width=1, prune=1, c=0.7, ln=1, choice=1, root_n=None, rm=None, rv=None,
             rw=None, stride=0, B=4):
        return L.ddz_uct_search(state, mask, ws, budget, width, prune, c, ln, 1, 0, choice, None, root_n, rm, rv, rw, stride,
                                B, None)
    assert call(state=None) == E and call(ws=None) == E and call(ln=None) == E and call(choice=None) == E
    assert call(B=0) == E and call(B=-3) == E
    assert call(budget=0) == E and call(budget=65537) == E
    assert call(width=0) == E and call(width=1025) == E
    assert call(budget=65536, width=257) == E and call(budget=16385, width=1024) == E     # budget * width > 2^24
    assert call(c=float("nan")) == E and call(c=float("inf")) == E
    assert call(root_n=1) == E and call(root_n=1, rm=1, rv=1, rw=1, stride=0) == E and call(root_n=1, rm=1, rv=None, rw=1, stride=4) == E


# ------------------------------------------------------------------ GPU
NODE = np.dtype([("untried", "<u4", 16), ("hand", "<u8", 3), ("recent", "<u8", 3), ("move", "<u8"), ("parent", "<i4"),
                 ("first_child", "<i4"), ("last_child", "<i4"), ("nchild", "<i4"), ("visits", "<i4"), ("wins", "<i4"),
                 ("nentries", "<i2"), ("remaining", "<i2"), ("index", "<i2"), ("cur", "i1"), ("winner", "i1"),
                 ("pad", "<i4", 2)])
assert NODE.itemsize == 160


@pytest.fixture(scope="module")
def D():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


def env_of(D, positions, env0=0, seed=None):
    """a BatchedEnv whose env b is positions[b] (hands, recent, role)"""
    B = len(positions)
    hands = np.stack([p[0] for p in positions]); recent = np.stack([p[1] for p in positions])
    role = np.array([p[2] for p in positions])
    return D.env_from_arrays(role, hands[np.arange(B), role], np.zeros((B, 3, 15), np.int64), recent, hands.sum(2),
                             env_cls=D.BatchedEnv, hands=hands, env0=env0, seed=seed)


def positions_of(D, env):
    """(hands int [B,3,15], recent [B,3,15], cur [B], done [B]) of a BatchedEnv"""
    f, meta = env._fields()
    u = D.unpack_counts(f.t().contiguous()).cpu().numpy()                    # [B, 9, 15]
    meta = meta.cpu().numpy()
    return u[:, 0:3], u[:, 6:9], (meta & 3).astype(np.int32), ((meta >> 2) & 1).astype(bool)


def device_run(D, env, budget, width, prune, seed, mask=None, c=0.7, env0=None, stride=None):
    """ddz_uct_search through the C-ABI on env's state; returns the outputs and every root's tree read from the workspace"""
    import torch
    from importlib import import_module
    S = import_module("doudizhu-rl_b200.search")
    N = D.native
    B, dev = env.B, env.device
    ws = torch.zeros(N.lib.ddz_uct_workspace_bytes(B, budget), dtype=torch.uint8, device=dev)
    ws.fill_(0xA5)
    ln = S._ln_table(budget * width, dev)
    stride = stride or min(budget, 512)
    out = {"choice": torch.full((B,), 7, dtype=torch.int32, device=dev), "move": torch.zeros(B, dtype=torch.int64, device=dev),
           "root_n": torch.full((B,), 9, dtype=torch.int32, device=dev),
           "root_moves": torch.zeros((B, stride), dtype=torch.int64, device=dev),
           "root_visits": torch.zeros((B, stride), dtype=torch.int32, device=dev),
           "root_wins": torch.zeros((B, stride), dtype=torch.int32, device=dev)}
    m = None if mask is None else torch.as_tensor(np.asarray(mask, np.uint8)).to(dev)
    p = lambda t: None if t is None else t.data_ptr()
    N.check(N.lib.ddz_uct_search(p(env._state), p(m), ws.data_ptr(), budget, width, int(prune), c, ln.data_ptr(), seed,
                                 env.env0 if env0 is None else env0, p(out["choice"]), p(out["move"]), p(out["root_n"]),
                                 p(out["root_moves"]), p(out["root_visits"]), p(out["root_wins"]), stride, B,
                                 torch.cuda.current_stream(dev).cuda_stream), "ddz_uct_search")
    torch.cuda.synchronize()
    r = {k: v.cpu().numpy() for k, v in out.items()}
    r["move"] = r["move"].view(np.uint64)
    r["root_moves"] = r["root_moves"].view(np.uint64)
    raw = ws.cpu().numpy()
    hdr = (4 * B + 255) // 256 * 256
    r["nnodes"] = raw[:4 * B].view(np.int32)
    r["tree"] = raw[hdr:].view(NODE).reshape(B, budget + 1)
    return r


def ref_of(D, env, budget, width, prune, seed, mask=None, c=0.7):
    hands, recent, cur, done = positions_of(D, env)
    live = ~done if mask is None else (~done & np.asarray(mask, bool))
    return ref_uct_batch(hands, recent, cur, live, budget, width=width, prune=prune, c=c, seed=seed, env0=env.env0)


def assert_trees_equal(dev, ref, where=""):
    """whole trees bit for bit: every node's parent, move, visits, wins and canonical index; outputs; root tables"""
    assert np.array_equal(dev["nnodes"], ref["nnodes"]), where
    B, n1 = ref["parent"].shape
    used = np.arange(n1)[None, :] < ref["nnodes"][:, None]
    t = dev["tree"]
    for k, d in (("parent", t["parent"]), ("visits", t["visits"]), ("wins", t["wins"]), ("index", t["index"]),
                 ("node_move", t["move"])):
        bad = np.argwhere(used & (d != ref[k]))
        assert len(bad) == 0, (where, k, bad[:5])
    assert np.array_equal(dev["choice"], ref["choice"]), where
    assert np.array_equal(dev["move"], ref["move"]), where
    assert np.array_equal(dev["root_n"], ref["root_n"]), where
    S = dev["root_moves"].shape[1]
    for b in range(B):
        k = min(int(ref["root_n"][b]), S)
        assert np.array_equal(dev["root_moves"][b, :k], ref["node_move"][b, 1:1 + k]), (where, b)
        assert np.array_equal(dev["root_visits"][b, :k], ref["visits"][b, 1:1 + k]), (where, b)
        assert np.array_equal(dev["root_wins"][b, :k], ref["wins"][b, 1:1 + k]), (where, b)
        # the tree's own bookkeeping agrees with its parent links
        n = int(ref["nnodes"][b])
        if n:
            kids = np.flatnonzero(t["parent"][b, :n] == 0)
            assert np.array_equal(kids, np.arange(1, 1 + len(kids))) and t["nchild"][b, 0] == len(kids), (where, b)


def rollout_env(D, B, seed, steps, env0=0):
    """B dealt envs after a seeded random rollout of a per-env random number of steps (0..steps-1)"""
    import torch
    perm, lord = D.random_deals(B, seed=seed)
    env = D.BatchedEnv(B, seed=seed, env0=env0)
    env.prepare(perm, lord)
    k = np.random.default_rng(seed).integers(0, steps, B)
    for t in range(steps):
        env.observe()
        mask = torch.as_tensor(k > t, device=env.device)
        n = (env.offsets[1:] - env.offsets[:-1]).cpu().numpy()
        ch = np.where(k > t, np.random.default_rng(seed * 1000 + t).integers(0, 1 << 30, B) % np.maximum(n, 1), 0)
        # envs whose rollout is over replay their state: step everybody, then restore the ones that stopped
        f, meta = env._fields()
        keep_f, keep_m = f.clone(), meta.clone()
        env.step(ch.astype(np.int32))
        f, meta = env._fields()
        f.copy_(torch.where(mask[None, :], f, keep_f)); meta.copy_(torch.where(mask, meta, keep_m))
        env._fresh = False
    return env


def family_positions(oracle, rng):
    """position families, each asserted on the input: (name, positions)"""
    fam = [("uct test", uct_test_positions())]
    lf = random_positions(oracle, rng, 48, 5, 18, follow=0.5)
    assert {(p[2], bool(p[1].any())) for p in lf} == {(r, f) for r in range(3) for f in (False, True)}
    fam.append(("leads and follows", lf))
    # lists longer than 10 moves with rocket-kicker moves that the pruning drops
    rk = []
    while len(rk) < 12:
        p = random_positions(oracle, rng, 1, 12, 20, follow=0.0)[0]
        h = p[0][p[2]]
        if h[13] and h[14] and (h >= 3).any():
            full = oracle.get_moves(h, np.zeros(15, np.int8), fast=True)
            kept = {oracle.pack(m) for m in oracle.mcts_moves(h, np.zeros(15, np.int8))}
            rocket_kick = [m for m in full if m[13] and m[14] and m.sum() > 2 and (m >= 3).any()]
            if len(full) > 10 and rocket_kick and all(oracle.pack(m) not in kept for m in rocket_kick):
                rk.append(p)
    fam.append(("pruned with rocket kickers", rk))
    # A pruned list repeats entries only when fewer moves are kept than its 2 (n / 3 + 1) slots, i.e. when the rocket-kicker
    # drop removes about a third of a list; no hand of one deck does that (a search over 20 000 random hands holding the
    # rocket found none), so there is no duplicate-entry family.
    # a root move ends the game: the role to move holds one playable move (a pair, a trio, a straight, a solo, the rocket);
    # the other two hands are dealt from the rest of the deck, so every position is a consistent deal
    term = []
    for hand in ([0, 0], [5, 5, 5], [0, 1, 2, 3, 4], [11], [13, 14]):
        for role in range(3):
            rest = list(DECK)
            for r in hand:
                rest.remove(r)
            p = rng.permutation(np.array(rest))
            h = np.zeros((3, 15), np.int64)
            h[role] = np.bincount(hand, minlength=15)
            others = [q for q in range(3) if q != role]
            k = rng.integers(3, 10, 2)
            h[others[0]] = np.bincount(p[:k[0]], minlength=15)
            h[others[1]] = np.bincount(p[k[0]:k[0] + k[1]], minlength=15)
            term.append((h, Z.copy(), role))
    for h, _, role in term:
        assert (h.sum(0) <= np.bincount(DECK, minlength=15)).all()
    for h, _, role in term:
        assert any(oracle.pack(m) == oracle.pack(h[role]) for m in oracle.get_moves(h[role], np.zeros(15, np.int8), fast=True))
    fam.append(("terminal root children", term))
    return fam


@pytest.mark.gpu
def test_device_trees_equal_c_port_on_position_families(D, oracle):
    """every family x widths 1, 8, 31, 32, 33, 100 x pruned / full lists: whole trees bit for bit"""
    rng = np.random.default_rng(31)
    fam = family_positions(oracle, rng)
    mid = rollout_env(D, 96, seed=5, steps=40)
    _, _, _, done = positions_of(D, mid)
    assert not done.all()
    roots = 0
    for width, budget in ((1, 300), (8, 100), (31, 40), (32, 40), (33, 40), (100, 20)):
        for prune in (True, False):
            for name, pos in fam:
                env = env_of(D, pos, env0=17)
                dev = device_run(D, env, budget, width, prune, seed=width + 11)
                assert_trees_equal(dev, ref_of(D, env, budget, width, prune, seed=width + 11), (name, width, budget, prune))
                roots += len(pos)
                if name == "terminal root children":
                    assert (dev["tree"]["winner"][:, 1:] >= 0).any()
            if width <= 8:
                dev = device_run(D, mid, budget, width, prune, seed=3)
                assert_trees_equal(dev, ref_of(D, mid, budget, width, prune, seed=3), ("mid-game", width, budget, prune))
                roots += mid.B
    assert roots >= 600


@pytest.mark.gpu
def test_device_small_budgets(D, oracle):
    """budget 1, and budgets below the root's entry count (the root is never fully expanded)"""
    rng = np.random.default_rng(32)
    pos = random_positions(oracle, rng, 40, 8, 18)
    n_entries = np.array([len(oracle.mcts_moves(h[r], r_[(r + 2) % 3] if r_[(r + 2) % 3].any() else r_[(r + 1) % 3]))
                          for h, r_, r in pos])
    env = env_of(D, pos)
    for budget in (1, 2, 5):
        assert (n_entries > budget).sum() >= 20
        for prune, width in ((True, 1), (False, 3)):
            dev = device_run(D, env, budget, width, prune, seed=9)
            assert_trees_equal(dev, ref_of(D, env, budget, width, prune, seed=9), (budget, prune))
            assert (dev["root_n"] == np.minimum(budget, dev["tree"]["nentries"][:, 0])).all()


@pytest.mark.gpu
def test_device_reference_configuration(D, oracle):
    """the reference's configuration: budget 1000, width 1, pruned lists, 64 roots"""
    env = rollout_env(D, 64, seed=8, steps=20)
    dev = device_run(D, env, 1000, 1, True, seed=1)
    assert_trees_equal(dev, ref_of(D, env, 1000, 1, True, seed=1), "reference configuration")


@pytest.mark.gpu
def test_device_batch_shapes(D, oracle):
    """B = 1, B not a multiple of the CTA's 4 warps, B = 4096"""
    rng = np.random.default_rng(33)
    pos = random_positions(oracle, rng, 7, 6, 18)
    for B in (1, 7):
        env = env_of(D, pos[:B])
        assert_trees_equal(device_run(D, env, 50, 2, True, seed=4), ref_of(D, env, 50, 2, True, seed=4), B)
    env = rollout_env(D, 4096, seed=9, steps=30)
    assert_trees_equal(device_run(D, env, 24, 1, True, seed=4), ref_of(D, env, 24, 1, True, seed=4), 4096)


@pytest.mark.gpu
def test_mask_finished_envs_and_env0_chunks(D, oracle):
    """masked-out and finished envs keep their sentinels and take no draw (the other roots' trees do not move);
    two calls over halves with their env0 equal one call; the state is not changed"""
    import torch
    env = rollout_env(D, 64, seed=12, steps=200)          # long rollouts: some games are over
    _, _, _, done = positions_of(D, env)
    assert done.any() and not done.all()
    before = env._state.clone()
    mask = np.random.default_rng(1).random(64) < 0.7
    full = device_run(D, env, 40, 2, True, seed=6)
    masked = device_run(D, env, 40, 2, True, seed=6, mask=mask)
    assert torch.equal(env._state, before)
    assert_trees_equal(masked, ref_of(D, env, 40, 2, True, seed=6, mask=mask), "masked")
    off = ~mask | done
    assert (masked["choice"][off] == -1).all() and (masked["move"][off] == np.uint64(2 ** 64 - 1)).all()
    assert (masked["root_n"][off] == 0).all() and (masked["nnodes"][off] == 0).all()
    on = ~off
    for k in ("choice", "move", "root_n", "nnodes"):
        assert np.array_equal(masked[k][on], full[k][on]), k
    assert masked["tree"][on].tobytes() == full["tree"][on].tobytes()
    # env0 chunking: the two halves as envs of their own, with their global env0
    hands, recent, cur, _ = positions_of(D, env)
    pos = [(hands[b].astype(np.int64), recent[b].astype(np.int64), int(cur[b])) for b in range(64)]
    live = ~done
    halves = []
    for lo in (0, 32):
        e = env_of(D, [pos[b] for b in range(lo, lo + 32)], env0=env.env0 + lo)
        e_f, e_m = e._fields()
        e_m.copy_(env._fields()[1][lo:lo + 32])                  # keep the finished flags
        halves.append(device_run(D, e, 40, 2, True, seed=6))
    for k in ("choice", "move", "root_n", "nnodes"):
        assert np.array_equal(np.concatenate([h[k] for h in halves]), full[k]), k
    assert np.concatenate([h["tree"] for h in halves])[live].tobytes() == full["tree"][live].tobytes()


@pytest.mark.gpu
def test_uct_search_choice_is_legal_and_steps(D):
    """uct_search: choice is the index of the move in env.valid_actions(); env.step(choice) raises no sticky error; the
    env's state and step counter are untouched; the root table matches the workspace run"""
    import torch
    env = rollout_env(D, 200, seed=14, steps=30)
    before, stepno = env._state.clone(), env._stepno
    choice, moves, tab = D.uct_search(env, computation_budget=60, width=4, seed=2, root_table=True)
    assert torch.equal(env._state, before) and env._stepno == stepno
    dev = device_run(D, env, 60, 4, True, seed=2)
    assert np.array_equal(choice.cpu().numpy(), dev["choice"]) and np.array_equal(moves.cpu().numpy().view(np.uint64), dev["move"])
    assert np.array_equal(tab[0].cpu().numpy(), dev["root_n"])
    assert np.array_equal(tab[2].cpu().numpy(), dev["root_visits"])
    packed, off = env.actions_packed.cpu().numpy().view(np.uint64), env.offsets.cpu().numpy()
    ch, mv = choice.cpu().numpy(), moves.cpu().numpy().view(np.uint64)
    done = positions_of(D, env)[3]
    for b in range(env.B):
        if done[b]:
            assert ch[b] == -1
            continue
        assert 0 <= ch[b] < off[b + 1] - off[b] and packed[off[b] + ch[b]] == mv[b]
    # a caller-owned workspace gives the same search as the per-stream cache
    ws = torch.empty(D.native.lib.ddz_uct_workspace_bytes(env.B, 60), dtype=torch.uint8, device=env.device)
    c2, m2 = D.uct_search(env, computation_budget=60, width=4, seed=2, workspace=ws)
    assert torch.equal(c2, choice) and torch.equal(m2, moves)
    with pytest.raises(ValueError):
        D.uct_search(env, computation_budget=60, width=4, seed=2, workspace=ws[:-1])
    env.step(np.where(ch < 0, 0, ch).astype(np.int32))
    assert int(env.stats[7].item()) == 0


@pytest.mark.gpu
def test_mcts_batch(D):
    """mcts_batch(payloads) == uct_search on the equivalent env; legal on the payloads of test_mcts_entry_point"""
    payloads = [{"role_id": 1, "hand_card": {0: [13, 14, 14, 15], 1: [3, 4, 5, 6, 7], 2: [8, 8, 9, 9]},
                 "last_taken": {0: [], 1: [], 2: []}},
                {"role_id": 2, "hand_card": {"0": [3], "1": [4], "2": [10, 10, 11]},
                 "last_taken": {"0": [], "1": [9, 9], "2": []}}]
    rng = np.random.default_rng(3)
    deck = [min(i // 4 + 3, 15) if i < 52 else 16 + (i - 52) for i in range(54)]
    cards = [int(c) for c in rng.permutation(deck)[:31]]
    payloads.append({"role_id": 1, "hand_card": {0: sorted(cards[:10]), 1: sorted(cards[10:22]), 2: sorted(cards[22:31])},
                     "last_taken": {0: [], 1: [], 2: []}})
    got = D.mcts_batch(payloads, computation_budget=400, seed=3)
    assert got[0] == [3, 4, 5, 6, 7]                          # the straight wins on the spot
    assert got[1] in ([10, 10], [])                           # beat the 9s with the pair, or pass
    hand = payloads[2]["hand_card"][1]
    assert all(got[2].count(v) <= hand.count(v) for v in got[2]) and got[2]
    # the same as uct_search on the env the payloads describe
    pos = []
    for p in payloads:
        g = lambda d, q: d[q] if q in d else d[str(q)]
        h = np.stack([np.bincount(np.array(g(p["hand_card"], q), int) - 3, minlength=15) for q in range(3)])
        r = np.stack([np.bincount(np.array(g(p["last_taken"], q), int) - 3, minlength=15) for q in range(3)])
        pos.append((h, r, int(p["role_id"])))
    env = env_of(D, pos)
    ch, mv = D.uct_search(env, computation_budget=400, seed=3)
    want = [[r + 3 for r in range(15) for _ in range(int((m >> (4 * r)) & 15))] for m in mv.cpu().numpy().view(np.uint64).tolist()]
    assert got == want


@pytest.mark.gpu
def test_searched_landlord_beats_random_landlord(D):
    """512 seeded games, the landlord searched (budget 200) and the farmers random, played to the end through env.step;
    the same deals with a random landlord.  Every game finishes without a sticky error and the searched landlord wins
    more.  The run is deterministic: the two win counts are pinned."""
    import torch
    B = 512
    perm, lord = D.random_deals(B, seed=21)
    wins = {}
    for searched in (True, False):
        env = D.BatchedEnv(B, seed=4)
        env.prepare(perm, lord)
        rng = np.random.default_rng(7)
        for t in range(200):
            f, meta = env._fields()
            done = ((meta >> 2) & 1).bool()
            if bool(done.all()):
                break
            env.observe()
            n = (env.offsets[1:] - env.offsets[:-1]).cpu().numpy()
            ch = (rng.integers(0, 1 << 30, B) % np.maximum(n, 1)).astype(np.int32)
            if searched:
                lord_turn = ((meta & 3) == 1) & ~done
                if bool(lord_turn.any()):
                    c, _ = D.uct_search(env, computation_budget=200, seed=t + 1, env_mask=lord_turn)
                    c = c.cpu().numpy()
                    ch = np.where(lord_turn.cpu().numpy(), c, ch).astype(np.int32)
            env.step(ch)
        meta = env._fields()[1].cpu().numpy()
        assert ((meta >> 2) & 1).all() and int(env.stats[7].item()) == 0
        wins[searched] = int((((meta >> 3) & 3) == 1).sum())
    print("landlord wins: searched %d, random %d" % (wins[True], wins[False]))
    assert wins[True] > wins[False], wins
    assert (wins[True], wins[False]) == PINNED_LORD_WINS, wins


PINNED_LORD_WINS = (482, 176)      # (searched landlord, random landlord) wins out of 512, measured on a B200
