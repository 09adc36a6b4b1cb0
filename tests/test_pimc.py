"""Determinized search (ddz_determinize, ddz_uct_pool, search.pimc_search, ingest.pimc_batch, BatchedGame's search seat):
the search bot playing from the player's own view -- D deals of the unseen cards, one UCT tree each, root statistics
pooled per canonical move index.

CPU: the argument checks of both entry points; the draw rule's distribution (exact enumeration); the pooling rule on
hand-built trees; the numpy Philox of the reference.  GPU: determinized states, choices, moves and pooled tables bit for
bit against tests/pimc_reference.py (a CPU pipeline over the oracle); the invariants of every determinization; the
device's split distribution; no information leak; chunking; inconsistent roots; payloads; seeded games."""
import numpy as np
import pytest

from pimc_reference import DECK, MAX_LEGAL, determinize, philox_np, pimc_reference, pool
from test_uct_batch import env_of, rollout_env

NONE = np.uint64(2 ** 64 - 1)


# ------------------------------------------------------------------ CPU
def test_pimc_argument_checks():
    """both entry points return DDZ_E_ARG before any CUDA call"""
    import ddz_b200 as D
    L, E = D.native.lib, D.native.E_ARG
    assert D.native.PIMC_MAX_DETERMINIZATIONS == 4096

    def det(state=1, mask=None, Dn=4, out=1, B=4):
        return L.ddz_determinize(state, mask, Dn, 1, 0, out, None, B, None)
    assert det(state=None) == E and det(out=None) == E
    assert det(B=0) == E and det(B=-1) == E
    assert det(Dn=0) == E and det(Dn=-2) == E and det(Dn=4097) == E
    assert det(Dn=4096, B=524288) == E                                 # B * D = 2^31
    assert det(Dn=2, B=2 ** 30) == E

    def pl(ws=1, budget=10, Dn=4, choice=1, B=4):
        return L.ddz_uct_pool(ws, budget, Dn, choice, None, None, None, B, None)
    assert pl(ws=None) == E and pl(choice=None) == E
    assert pl(B=0) == E and pl(B=-5) == E
    assert pl(budget=0) == E and pl(budget=65537) == E
    assert pl(Dn=0) == E and pl(Dn=4097) == E
    assert pl(Dn=4096, B=524288) == E                                  # B * D > INT_MAX


def test_reference_philox_equals_oracle(oracle):
    rng = np.random.default_rng(0)
    env = rng.integers(0, 2 ** 63, 300, dtype=np.uint64)
    step = rng.integers(0, 2 ** 32, 300, dtype=np.uint64)
    for seed in (0, 1, 2 ** 40 + 7, 2 ** 64 - 1):
        want = np.array([oracle.philox(seed, int(e), int(s)) for e, s in zip(env, step)], np.uint32)
        assert np.array_equal(philox_np(seed, env, step), want), seed


def one_root(unseen, na, m=1, hist=None):
    """one position of role m whose unseen cards are `unseen` (counts [15]) and whose next role holds na of them"""
    hist = np.zeros((3, 15), np.int64) if hist is None else hist
    hands = np.zeros((3, 15), np.int64)
    hands[m] = DECK - unseen - hist.sum(0)
    a, c = (m + 1) % 3, (m + 2) % 3
    U = int(unseen.sum())
    hands[a, 0], hands[c, 0] = na, U - na          # placeholders of the right sizes: never read
    return hands, hist


def test_draw_rule_is_hypergeometric():
    """unseen {3,3,4,5,J} split 2 / 3: every split of the five distinguishable cards is equally likely, so the next role's
    pair is {3,3} 1/10, {3,4} 2/10, {3,5} 2/10, {3,J} 2/10, {4,5} 1/10, {4,J} 1/10, {5,J} 1/10 -- 20 000 reference draws"""
    from itertools import combinations
    from scipy.stats import chisquare
    unseen = np.bincount([0, 0, 1, 2, 8], minlength=15)
    hands, hist = one_root(unseen, 2)
    Dn = 20000
    h, _, _, meta, nbad = determinize(hands[None], hist[None], np.zeros((1, 3, 15)), np.array([1], np.uint32), Dn, seed=11)
    assert nbad == 0 and not ((meta >> 2) & 1).any()
    a_hands = h[:, 2]
    assert (h[:, 2] + h[:, 0] == unseen).all() and (a_hands.sum(1) == 2).all() and (h[:, 1] == hands[1]).all()
    cards = [0, 0, 1, 2, 8]
    expect = {}
    for pair in combinations(range(5), 2):
        key = tuple(sorted(cards[i] for i in pair))
        expect[key] = expect.get(key, 0) + 1
    keys = sorted(expect)
    got = {k: 0 for k in keys}
    for row in a_hands:
        got[tuple(np.repeat(np.arange(15), row))] += 1
    obs = np.array([got[k] for k in keys])
    exp = np.array([expect[k] / 10 * Dn for k in keys])
    stat, p = chisquare(obs, exp)
    assert obs.sum() == Dn and p > 1e-3, (obs, exp, p)


def test_pool_on_hand_built_trees():
    """duplicate indices in one tree add up, trees add up, exact ties go to the lowest index, an unsearched tree adds
    nothing and a root with no searched tree answers -1"""
    n = 6
    parent = np.array([[-1, 0, 0, 0, 1, 0],      # tree 0: root children 1, 2, 3, 5 (4 is a grandchild)
                       [-1, 0, 0, 2, 0, 0],      # tree 1: root children 1, 2, 4, 5
                       [-1, 0, 0, 0, 0, 0],      # tree 2: not searched (nnodes 0)
                       [-1, 0, 0, 0, 0, 0],      # tree 3: not searched
                       [-1, 0, 0, 0, 0, 0],      # tree 4: ties
                       [-1, 0, 0, 0, 0, 0]])
    index = np.array([[-1, 7, 3, 7, 9, 4],       # duplicate pruned entries of index 7
                      [-1, 3, 4, 1, 9, 0],
                      [-1, 1, 2, 3, 4, 5],
                      [-1, 1, 2, 3, 4, 5],
                      [-1, 5, 2, 9, 0, 0],
                      [-1, 0, 0, 0, 0, 0]])
    visits = np.array([[9, 2, 3, 1, 1, 3], [9, 2, 2, 5, 1, 4], [0] * 6, [0] * 6, [8, 2, 4, 1, 1, 0], [0] * 6])
    wins = np.array([[5, 1, 1, 1, 1, 2], [5, 2, 0, 5, 1, 1], [0] * 6, [0] * 6, [4, 1, 2, 0, 0, 0], [0] * 6])
    nnodes = np.array([6, 6, 0, 0, 5, 0])
    trees = {"parent": parent, "index": index, "visits": visits, "wins": wins, "nnodes": nnodes}
    choice, pv, pw = pool(trees, 2)
    # root 0 = trees 0 + 1: index 7: 2 + 1 = 3 visits, 1 + 1 = 2 wins; 3: 3 + 2; 4: 3 + 2; 9: 1 (tree 1); 0: 4
    assert pv[0, 7] == 3 and pw[0, 7] == 2
    assert pv[0, 3] == 5 and pw[0, 3] == 3
    assert pv[0, 4] == 5 and pw[0, 4] == 2
    assert pv[0, 9] == 1 and pw[0, 9] == 1 and pv[0, 0] == 4 and pw[0, 0] == 1 and pv[0, 1] == 0
    assert pv[0].sum() == 18 and choice[0] == 9                 # 1 / 1
    assert choice[1] == -1 and not pv[1].any()                  # trees 2 and 3 were not searched
    # root 2 = tree 4 (5 nodes) + unsearched tree 5: indices 5 (1/2), 2 (2/4), 9 (0/1), 0 (0/1) -> the tie goes to 2
    assert choice[2] == 2 and pv[2, 5] == 2 and pv[2, 2] == 4 and pv[2, 0] == 1
    # an index whose pooled rate equals a lower index's loses
    trees2 = {"parent": np.array([[-1, 0, 0]]), "index": np.array([[-1, 8, 6]]), "visits": np.array([[6, 2, 4]]),
              "wins": np.array([[3, 1, 2]]), "nnodes": np.array([3])}
    assert pool(trees2, 1)[0][0] == 6


def test_search_seat_needs_a_free_role():
    """a role cannot have a net and a search entry; unknown roles are refused"""
    import ddz_b200 as D
    with pytest.raises(ValueError):
        D.BatchedGame(D.BatchedEnv, {"lord": object}, {"lord": object}, search_dict={"lord": {"determinizations": 2}})
    with pytest.raises(ValueError):
        D.BatchedGame(D.BatchedEnv, {}, {}, search_dict={"boss": {}})


def test_unseen_mismatch_on_core_payloads(golden):
    """every core payload (the server/client.py examples included) is consistent: unseen = the other two `left` counts"""
    from importlib import import_module
    I = import_module("doudizhu-rl_b200.ingest")
    g = golden.core_payloads
    assert len(I.unseen_mismatch(g["role"], g["hand"], g["history"], g["left"])) == 0
    left = g["left"].astype(np.int64).copy()
    left[5, (g["role"][5] + 1) % 3] += 1
    assert I.unseen_mismatch(g["role"], g["hand"], g["history"], left).tolist() == [5]


# ------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def D():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


def S():
    from importlib import import_module
    return import_module("doudizhu-rl_b200.search")


def state_arrays(D, state, n):
    """(hands, hist, recent int [n,3,15], meta uint32 [n]) of a raw state tensor of n envs"""
    f = state[: 18 * n].view(__import__("torch").int64).view(9, n)
    u = D.unpack_counts(f.t().contiguous()).cpu().numpy().astype(np.int64)
    meta = state[18 * n: 19 * n].cpu().numpy().view(np.uint32)
    return u[:, 0:3], u[:, 3:6], u[:, 6:9], meta


def env_arrays(D, env):
    return state_arrays(D, env._state, env.B)


def make_env(D, hands, hist, recent, role, env0=0):
    B = len(role)
    return D.env_from_arrays(role, hands[np.arange(B), role], hist, recent, hands.sum(2), env_cls=D.BatchedEnv,
                             hands=hands, env0=env0)


def forced_positions(rng, n):
    """positions whose unseen cards are copies of one rank: every determinization is the true deal"""
    out_h, out_hist, out_role = [], [], []
    deck = np.repeat(np.arange(15), DECK)
    while len(out_role) < n:
        r = int(rng.integers(13))
        k = int(rng.integers(2, 5))
        k1 = int(rng.integers(1, k))
        rest = list(deck)
        for _ in range(k):
            rest.remove(r)
        rest = rng.permutation(np.array(rest))
        m = int(rng.integers(3))
        s = int(rng.integers(1, 12))
        hands = np.zeros((3, 15), np.int64)
        hands[m] = np.bincount(rest[:s], minlength=15)
        hands[(m + 1) % 3, r], hands[(m + 2) % 3, r] = k1, k - k1
        owner = rng.integers(3, size=len(rest) - s)
        hist = np.stack([np.bincount(rest[s:][owner == q], minlength=15) for q in range(3)])
        out_h.append(hands); out_hist.append(hist); out_role.append(m)
    return np.stack(out_h), np.stack(out_hist), np.array(out_role)


def assert_determinized(D, env, Dn, seed, mask=None):
    """ddz_determinize == pimc_reference.determinize over every output env, and the invariants"""
    import torch
    hands, hist, recent, meta = env_arrays(D, env)
    before = env.stats[7].item()
    out = S().determinize(env, Dn, seed=seed, env_mask=mask)
    torch.cuda.synchronize()
    got = state_arrays(D, out, env.B * Dn)
    want = determinize(hands, hist, recent, meta, Dn, seed, env0=env.env0, mask=mask)
    for k, (g, w) in enumerate(zip(got, want[:4])):
        assert np.array_equal(g, w), (k, np.argwhere(g != w)[:5])
    assert env.stats[7].item() - before == want[4]
    # invariants: mover's hand, hist, recent, meta unchanged; hidden sizes unchanged; hidden = unseen
    h, hs, rc, mt = got
    rep = lambda x: np.repeat(x, Dn, axis=0)
    ar = np.arange(env.B * Dn)
    m = (mt & 3).astype(np.int64)
    assert np.array_equal(h[ar, m], rep(hands)[ar, m])
    assert np.array_equal(hs, rep(hist)) and np.array_equal(rc, rep(recent))
    ok = ((mt >> 5) & 1) == 0
    assert np.array_equal(mt[ok], rep(meta)[ok])
    assert np.array_equal(h.sum(2), rep(hands).sum(2))
    live = ok & (((rep(meta) >> 2) & 1) == 0)
    if mask is not None:
        live &= np.repeat(np.asarray(mask, bool), Dn)
    unseen = DECK[None, :] - h[ar, m] - hs.sum(1)
    assert np.array_equal((h[ar, (m + 1) % 3] + h[ar, (m + 2) % 3])[live], unseen[live])
    assert np.array_equal(h[~live], rep(hands)[~live])
    return got, want


@pytest.mark.gpu
def test_determinized_states_equal_reference(D, golden):
    """fresh deals, mid-game rollouts, the core payloads and forced splits; D = 1, 7, 64; B = 1, 7, 4096; masks, finished
    envs and env0 chunks"""
    import torch
    rng = np.random.default_rng(40)
    fresh = D.BatchedEnv(4096, seed=3)
    fresh.prepare(*D.random_deals(4096, seed=41))
    for Dn in (1, 7, 64):
        assert_determinized(D, fresh, Dn, seed=Dn + 2)
    mid = rollout_env(D, 512, seed=42, steps=120, env0=1000)
    done = ((env_arrays(D, mid)[3] >> 2) & 1).astype(bool)
    assert done.any() and not done.all()
    mask = rng.random(512) < 0.6
    for Dn in (1, 7, 64):
        assert_determinized(D, mid, Dn, seed=9)
        assert_determinized(D, mid, Dn, seed=9, mask=mask)
    g = golden.core_payloads
    pay = D.env_from_arrays(g["role"], g["hand"], g["history"], g["last_taken"], g["left"], env_cls=D.BatchedEnv)
    got, _ = assert_determinized(D, pay, 7, seed=5)
    assert not ((got[3] >> 5) & 1).any()
    h, hs, role = forced_positions(rng, 7)
    env = make_env(D, h, hs, np.zeros((7, 3, 15), np.int64), role)
    for B in (1, 7):
        one = make_env(D, h[:B], hs[:B], np.zeros((B, 3, 15), np.int64), role[:B])
        got, _ = assert_determinized(D, one, 64, seed=3)
        assert np.array_equal(got[0], np.repeat(h[:B], 64, axis=0))             # the only deal there is
    # env0 chunks: two raw launches over halves with their env0 == one launch
    N = D.native
    Dn = 7
    whole = S().determinize(mid, Dn, seed=4)
    parts = []
    for lo in (0, 200):
        n = 200 if lo == 0 else 312
        st = S()._state_slice(mid, lo, n)
        out = torch.empty(N.lib.ddz_state_bytes(n * Dn) // 4, dtype=torch.int32, device=mid.device)
        N.check(N.lib.ddz_determinize(st.data_ptr(), None, Dn, 4, mid.env0 + lo, out.data_ptr(), None, n,
                                      torch.cuda.current_stream().cuda_stream), "ddz_determinize")
        parts.append(state_arrays(D, out, n * Dn))
    for k, w in enumerate(state_arrays(D, whole, 512 * Dn)):
        assert np.array_equal(np.concatenate([p[k] for p in parts]), w), k


@pytest.mark.gpu
def test_device_split_distribution(D):
    """2^20 determinizations of one opening (the lord's view: 34 unseen cards, 17 / 17): each rank's count in the next
    role's hand follows its hypergeometric marginal (chi-square, seed pinned)"""
    from scipy.stats import chisquare, hypergeom
    deck = np.repeat(np.arange(15), DECK)
    p = np.random.default_rng(7).permutation(deck)
    h = np.stack([np.bincount(p[a:b], minlength=15) for a, b in ((0, 17), (17, 37), (37, 54))])
    B, Dn = 256, 4096
    env = make_env(D, np.repeat(h[None], B, 0), np.zeros((B, 3, 15), np.int64), np.zeros((B, 3, 15), np.int64),
                   np.ones(B, np.int64))
    import torch
    n = B * Dn
    out = S().determinize(env, Dn, seed=2024)
    f = out[: 18 * n].view(torch.int64).view(9, n)
    unseen = DECK - h[1]
    U, na = int(unseen.sum()), int(h[2].sum())
    assert U == 34 and na == 17 and n == 2 ** 20
    assert torch.equal(D.unpack_counts(f[2]) + D.unpack_counts(f[0]), torch.as_tensor(unseen, device=f.device).expand(n, 15))
    assert torch.equal(f[1], f[1, :1].expand(n))
    a_hand = D.unpack_counts(f[2]).cpu().numpy()
    pvals = []
    for r in np.flatnonzero(unseen):
        ks = np.arange(int(unseen[r]) + 1)
        exp = hypergeom(U, int(unseen[r]), na).pmf(ks) * 2 ** 20
        obs = np.bincount(a_hand[:, r], minlength=len(ks))
        assert obs.sum() == 2 ** 20 and len(obs) == len(ks)
        keep = exp >= 5
        obs2 = np.append(obs[keep], obs[~keep].sum()) if (~keep).any() else obs
        exp2 = np.append(exp[keep], exp[~keep].sum()) if (~keep).any() else exp
        pvals.append(chisquare(obs2, exp2 * obs2.sum() / exp2.sum()).pvalue)
    assert min(pvals) > 1e-4, pvals


def run_pimc(D, env, Dn, budget, width=1, prune=True, seed=1, mask=None, **kw):
    ch, mv, (pv, pw) = D.pimc_search(env, determinizations=Dn, computation_budget=budget, width=width, prune=prune,
                                     seed=seed, env_mask=mask, pooled_table=True, **kw)
    return {"choice": ch.cpu().numpy(), "move": mv.cpu().numpy().view(np.uint64), "pooled_visits": pv.cpu().numpy(),
            "pooled_wins": pw.cpu().numpy()}


def assert_pimc_equals_reference(D, oracle, env, Dn, budget, width=1, prune=True, seed=1, mask=None, where=""):
    hands, hist, recent, meta = env_arrays(D, env)
    got = run_pimc(D, env, Dn, budget, width, prune, seed, mask)
    want = pimc_reference(oracle, hands, hist, recent, meta, Dn, budget, width=width, prune=prune, seed=seed,
                          env0=env.env0, mask=mask)
    for k in ("choice", "move", "pooled_visits", "pooled_wins"):
        assert np.array_equal(got[k], want[k]), (where, k, np.argwhere(got[k] != want[k])[:5])
    return got


@pytest.mark.gpu
def test_pimc_search_equals_reference(D, oracle):
    """choice, move and pooled tables == determinize -> C port -> pool: D = 1, 4, 16; budgets 1, 50, 1000; widths 1 and 16;
    pruned and full lists; B = 1, 7, 512"""
    mid = rollout_env(D, 512, seed=44, steps=40, env0=3)
    h7 = env_arrays(D, mid)
    live = np.flatnonzero(((h7[3] >> 2) & 1) == 0)[:7]
    small = make_env(D, h7[0][live], h7[1][live], h7[2][live], (h7[3][live] & 3).astype(np.int64), env0=11)
    one = make_env(D, h7[0][live[:1]], h7[1][live[:1]], h7[2][live[:1]], (h7[3][live[:1]] & 3).astype(np.int64))
    for Dn, budget, width, prune in ((1, 1, 1, True), (4, 1, 16, False), (16, 50, 1, True), (4, 50, 16, True),
                                     (16, 50, 1, False), (1, 50, 16, False)):
        assert_pimc_equals_reference(D, oracle, small, Dn, budget, width, prune, seed=budget + Dn, where=(Dn, budget, width))
    assert_pimc_equals_reference(D, oracle, one, 16, 1000, 1, True, seed=2, where="B=1 budget 1000")
    assert_pimc_equals_reference(D, oracle, small, 4, 1000, 1, True, seed=3, where="B=7 budget 1000")
    mask = np.random.default_rng(2).random(512) < 0.8
    got = assert_pimc_equals_reference(D, oracle, mid, 4, 50, 1, True, seed=6, mask=mask, where="B=512")
    off = ~mask | (((h7[3] >> 2) & 1) == 1)
    assert (got["choice"][off] == -1).all() and (got["move"][off] == NONE).all() and not got["pooled_visits"][off].any()
    assert (got["choice"][~off] >= 0).all()
    # the answer is the legal move at that index
    mid.observe()
    packed, offs = mid.actions_packed.cpu().numpy().view(np.uint64), mid.offsets.cpu().numpy()
    for b in np.flatnonzero(~off):
        assert packed[offs[b] + got["choice"][b]] == got["move"][b]


@pytest.mark.gpu
def test_no_information_leak(D):
    """two batches with the same views (own hand, hist, recent, hand sizes) but different hidden hands: identical
    determinizations, choices and pooled tables"""
    import torch
    mid = rollout_env(D, 256, seed=45, steps=30)
    hands, hist, recent, meta = env_arrays(D, mid)
    live = np.flatnonzero(((meta >> 2) & 1) == 0)
    hands, hist, recent, role = hands[live], hist[live], recent[live], (meta[live] & 3).astype(np.int64)
    other = hands.copy()
    rng = np.random.default_rng(46)
    changed = 0
    for b, m in enumerate(role):
        a, c = (m + 1) % 3, (m + 2) % 3
        cards = rng.permutation(np.repeat(np.arange(15), hands[b, a] + hands[b, c]))
        na = int(hands[b, a].sum())
        other[b, a] = np.bincount(cards[:na], minlength=15)
        other[b, c] = np.bincount(cards[na:], minlength=15)
        changed += not np.array_equal(other[b, a], hands[b, a])
    assert changed >= len(role) // 2
    x = make_env(D, hands, hist, recent, role)
    y = make_env(D, other, hist, recent, role)
    assert not torch.equal(x._state, y._state)
    assert torch.equal(S().determinize(x, 8, seed=3), S().determinize(y, 8, seed=3))
    gx, gy = run_pimc(D, x, 8, 60, seed=4), run_pimc(D, y, 8, 60, seed=4)
    for k in gx:
        assert np.array_equal(gx[k], gy[k]), k
    # the full-information search does see the difference
    cx, _ = D.uct_search(x, computation_budget=60, seed=4)
    cy, _ = D.uct_search(y, computation_budget=60, seed=4)
    assert not torch.equal(cx, cy)


@pytest.mark.gpu
def test_one_determinization_of_a_forced_split_is_uct_search(D):
    """on positions whose unseen cards allow one deal only, D = 1 searches uct_search's own tree: the pooled tables are
    its root table folded by canonical index, and the choice is the same where the best rate has no tie"""
    rng = np.random.default_rng(47)
    h, hs, role = forced_positions(rng, 64)
    env = make_env(D, h, hs, np.zeros((64, 3, 15), np.int64), role, env0=5)
    got = run_pimc(D, env, 1, 200, seed=8)
    ch, mv, (rn, rm, rv, rw) = D.uct_search(env, computation_budget=200, seed=8, root_table=True)
    env.observe()
    packed, offs = env.actions_packed.cpu().numpy().view(np.uint64), env.offsets.cpu().numpy()
    rn, rm, rv, rw = rn.cpu().numpy(), rm.cpu().numpy().view(np.uint64), rv.cpu().numpy(), rw.cpu().numpy()
    ch = ch.cpu().numpy()
    untied = 0
    for b in range(64):
        lst = packed[offs[b]:offs[b + 1]]
        fv, fw = np.zeros(MAX_LEGAL, np.int64), np.zeros(MAX_LEGAL, np.int64)
        for k in range(rn[b]):
            i = int(np.flatnonzero(lst == rm[b, k])[0])
            fv[i] += rv[b, k]; fw[i] += rw[b, k]
        assert np.array_equal(got["pooled_visits"][b], fv) and np.array_equal(got["pooled_wins"][b], fw), b
        rate = np.where(fv > 0, fw / np.maximum(fv, 1), -1.0)
        if (rate == rate.max()).sum() == 1:
            untied += 1
            assert got["choice"][b] == ch[b], b
    assert untied >= 32


@pytest.mark.gpu
def test_chunking_does_not_change_results(D):
    """one root per chunk (a tiny max_workspace_bytes), three roots per chunk with a mask, and one call: equal results"""
    env = rollout_env(D, 23, seed=48, steps=30, env0=77)
    mask = np.random.default_rng(3).random(23) < 0.7
    for m in (None, mask):
        whole = run_pimc(D, env, 6, 40, width=2, seed=5, mask=m)
        per_root = 6 * 41 * 160
        for cap in (1, 3 * per_root + 100):
            part = run_pimc(D, env, 6, 40, width=2, seed=5, mask=m, max_workspace_bytes=cap)
            for k in whole:
                assert np.array_equal(part[k], whole[k]), (cap, k)


@pytest.mark.gpu
def test_inconsistent_roots(D):
    """a full-information env with zero hist (mcts_batch's form) shows a view no deal agrees with: -1, counted once per
    root in stats[7]; a payload whose `left` does not match its unseen cards makes pimc_batch raise"""
    rng = np.random.default_rng(49)
    deck = np.repeat(np.arange(15), DECK)
    pos = []
    for _ in range(9):
        p = rng.permutation(deck)
        pos.append((np.stack([np.bincount(p[a:b], minlength=15) for a, b in ((0, 5), (5, 12), (12, 20))]),
                    np.zeros((3, 15), np.int64), int(rng.integers(3))))
    env = env_of(D, pos)
    before = int(env.stats[7].item())
    ch, mv = D.pimc_search(env, determinizations=5, computation_budget=20)
    assert (ch.cpu().numpy() == -1).all() and (mv.cpu().numpy().view(np.uint64) == NONE).all()
    assert int(env.stats[7].item()) - before == 9
    out = state_arrays(D, S().determinize(env, 3), 27)[3]
    assert (((out >> 2) & 1) == 1).all() and (((out >> 5) & 1) == 1).all()
    payloads = core_payload_dicts(D, 4)
    payloads[2] = dict(payloads[2], left={q: v + (q == (payloads[2]["role_id"] + 1) % 3) for q, v in payloads[2]["left"].items()})
    with pytest.raises(ValueError, match=r"\[2\]"):
        D.pimc_batch(payloads, determinizations=2, computation_budget=5)


def cards_of(c):
    return [r + 3 for r in range(15) for _ in range(int(c[r]))]


def core_payload_dicts(D, n=None):
    g = np.load(__import__("os").path.join(__import__("os").path.dirname(__file__), "golden", "core_payloads.npz"))
    n = len(g["role"]) if n is None else n
    return [{"role_id": int(g["role"][b]), "cur_cards": cards_of(g["hand"][b]),
             "history": {q: cards_of(g["history"][b, q]) for q in range(3)},
             "last_taken": {q: cards_of(g["last_taken"][b, q]) for q in range(3)},
             "left": {q: int(g["left"][b, q]) for q in range(3)}} for b in range(n)]


def as_cards(choice, moves):
    out = []
    for ch, mv in zip(choice.tolist(), moves.tolist()):
        out.append(cards_of([(mv >> (4 * r)) & 15 for r in range(15)]) if ch >= 0 else [])
    return out


@pytest.mark.gpu
def test_pimc_batch(D):
    """the 591 core payloads: legal answers, equal to pimc_search on env_from_payloads; payloads cut from live games equal
    pimc_search on the live env, which holds the true hidden hands"""
    payloads = core_payload_dicts(D)
    got = D.pimc_batch(payloads, determinizations=4, computation_budget=30, seed=6)
    env = D.env_from_payloads(payloads, env_cls=D.BatchedEnv)
    ch, mv = D.pimc_search(env, determinizations=4, computation_budget=30, seed=6)
    assert got == as_cards(ch, mv)
    ch = ch.cpu().numpy()
    assert (ch >= 0).all()
    acts, offs = env.valid_actions()
    packed, offs = env.actions_packed.cpu().numpy().view(np.uint64), offs.cpu().numpy()
    assert (ch < offs[1:] - offs[:-1]).all()
    assert np.array_equal(packed[offs[:-1] + ch], mv.cpu().numpy().view(np.uint64))
    # live games
    mid = rollout_env(D, 128, seed=50, steps=40)
    hands, hist, recent, meta = env_arrays(D, mid)
    live = np.flatnonzero(((meta >> 2) & 1) == 0)
    role = (meta[live] & 3).astype(np.int64)
    live_env = make_env(D, hands[live], hist[live], recent[live], role)
    pl = [{"role_id": int(role[i]), "cur_cards": cards_of(hands[b, role[i]]),
           "history": {q: cards_of(hist[b, q]) for q in range(3)}, "last_taken": {q: cards_of(recent[b, q]) for q in range(3)},
           "left": {q: int(hands[b, q].sum()) for q in range(3)}} for i, b in enumerate(live)]
    ch, mv = D.pimc_search(live_env, determinizations=4, computation_budget=50, seed=7)
    assert D.pimc_batch(pl, determinizations=4, computation_budget=50, seed=7) == as_cards(ch, mv)


def lord_games(D, search, B=512, steps=200):
    """test_searched_landlord_beats_random_landlord's games: its deals, its farmers' draws; search(env, t, lord_turn) ->
    the landlord's choices, or None for a random landlord"""
    import torch
    perm, lord = D.random_deals(B, seed=21)
    env = D.BatchedEnv(B, seed=4)
    env.prepare(perm, lord)
    rng = np.random.default_rng(7)
    for t in range(steps):
        f, meta = env._fields()
        done = ((meta >> 2) & 1).bool()
        if bool(done.all()):
            break
        env.observe()
        n = (env.offsets[1:] - env.offsets[:-1]).cpu().numpy()
        ch = (rng.integers(0, 1 << 30, B) % np.maximum(n, 1)).astype(np.int32)
        lord_turn = ((meta & 3) == 1) & ~done
        if search is not None and bool(lord_turn.any()):
            c = search(env, t, lord_turn).cpu().numpy()
            ch = np.where(lord_turn.cpu().numpy(), c, ch).astype(np.int32)
        env.step(ch)
    meta = env._fields()[1].cpu().numpy()
    assert ((meta >> 2) & 1).all() and int(env.stats[7].item()) == 0
    return int((((meta >> 3) & 3) == 1).sum())


@pytest.mark.gpu
def test_pimc_landlord_beats_random_landlord(D):
    """512 seeded games, a pimc_search landlord (D = 8, budget 125) against random farmers on the deals of
    test_searched_landlord_beats_random_landlord (random landlord: 176 wins, full-information search: 482).  Every game
    ends without a sticky error; the run is deterministic, so the win count is pinned."""
    wins = lord_games(D, lambda env, t, m: D.pimc_search(env, determinizations=8, computation_budget=125, seed=t + 1,
                                                          env_mask=m)[0])
    print("pimc landlord wins: %d of 512" % wins)
    assert wins > 176
    assert wins == PINNED_PIMC_LORD_WINS, wins


@pytest.mark.gpu
def test_compete_with_a_search_seat(D):
    """BatchedGame.compete with a searched landlord, from its own view and with full information: both beat the random
    landlord of the same seeded run"""
    kw = dict(total=256, num_envs=128, seed=5, debug=False)
    rand = D.BatchedGame.compete(D.BatchedEnv, {}, {}, None, **kw)
    pimc = D.BatchedGame.compete(D.BatchedEnv, {}, {}, None, search_dict={"lord": {"determinizations": 4,
                                                                                   "computation_budget": 60}}, **kw)
    full = D.BatchedGame.compete(D.BatchedEnv, {}, {}, None, search_dict={"lord": {"determinizations": 0,
                                                                                   "computation_budget": 60}}, **kw)
    print("compete lord wins: random %d, pimc %d, full information %d" % (rand["lord"], pimc["lord"], full["lord"]))
    for w in (rand, pimc, full):
        assert w["lord"] + w["up"] + w["down"] >= 256
    assert pimc["lord"] > rand["lord"] and full["lord"] > rand["lord"]


PINNED_PIMC_LORD_WINS = 499     # pimc landlord wins out of 512 (D = 8, budget 125), measured on a B200
