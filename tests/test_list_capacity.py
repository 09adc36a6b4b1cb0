"""Legal-move lists that do not fit their buffer, against an oracle model of the capacity rule (include/ddz_b200.h,
ddz_observe / ddz_rollout_step; DESIGN.md "Errors").

The launches are called through the C-ABI with buffers this file allocates, so the capacity `cap` is exactly what each case
names.  The model, over oracle.RefBatch:
  observe at cap   the complete offsets; moves [0, min(cap, total)) and their one-hot rows stored, nothing after them; the
                   face always complete; stats[7] += (total > cap), stats[8] += total;
  fused step       full = diff(off), cnt = clip(min(full, cap - off[:-1]), 0): the move is picked among the cnt stored
                   entries (INDEX: choice, MOD: uint32(choice) % cnt, PHILOX: philox(seed, env0 + b, stepno) % cnt, MOVE: its
                   position in the stored part); a live env with cnt == 0 < full sits the step out (stats[7], no sticky
                   bit), any other index outside [0, cnt) is illegal (stats[7] and the sticky bit).
Every list buffer holds the complete lists plus a guard whatever `cap` is, and is refilled with sentinels before every
launch; offsets, results and face have guard slots too.  A kernel that wrote past `cap` would leave a non-sentinel word
there.  Before a fused step the part of the previous lists that was not stored is filled with the true moves of the
complete lists: a kernel that read past `cap` would then apply a real move (a state the comparison catches) rather than a
sentinel word as a move.  Everything is compared bit for bit after every launch."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SENT_U64 = np.uint64(0xA5A5A5A5A5A5A5A5)     # nibbles > 4: never a legal move
SENT_BYTE = 0x5C                              # offsets, r, done, cat
GUARD = 256                                   # moves past the complete lists
GUARD_ENVS = 8                                # offset / result / face slots past B
INDEX, MOD, PHILOX, MOVE = range(4)
HEAVY, WIN, EMIT_WIN = 32, 320, 896           # kHeavy; the window of the observe kernel and of ddz_legal_emit


@pytest.fixture(scope="module")
def D():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


@pytest.fixture
def tile_order(D):
    prev = D.native.set_tile_order("auto")
    yield D.native.set_tile_order
    D.native.set_tile_order(prev)


def _p(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------ the oracle model
class Model:
    """oracle.RefBatch plus the capacity rule; `cap` is the capacity of the lists the next fused step reads."""

    def __init__(self, O, ref):
        self.O, self.ref, self.cap = O, ref, None
        self.counts = np.zeros(3, np.int64)    # env-steps played from a complete / cut / dropped list

    def observe(self, cap, want_f32=True, want_face=True):
        off, au, af, face = self.ref.observe(want_f32=want_f32, want_face=want_face)
        total = int(off[-1])
        self.ref.stats[7] += total > cap
        self.ref.stats[8] += total
        self.cap = cap
        return off, au, af, face

    def stored(self):
        off = self.ref.offsets.astype(np.int64)
        full = np.diff(off)
        return full, np.clip(np.minimum(full, self.cap - off[:-1]), 0, None)

    def step(self, mode, choice=None, seed=0, env0=0, stepno=0, perm=None, lord=None, G=1):
        ref, B = self.ref, self.ref.B
        off = ref.offsets.astype(np.int64)
        full, cnt = self.stored()
        live = ref.envs["done"] == 0
        if mode == INDEX:
            idx = np.asarray(choice).astype(np.int64)
        elif mode == MOD:
            ent = np.asarray(choice).view(np.uint32).astype(np.int64)
            idx = np.where(cnt > 0, ent % np.maximum(cnt, 1), -1)
        elif mode == PHILOX:
            idx = np.array([self.O.philox(seed, env0 + b, stepno) % cnt[b] if cnt[b] > 0 and live[b] else -1
                            for b in range(B)], np.int64)
        else:
            want = np.asarray(choice).view(np.uint64)
            idx = np.full(B, -1, np.int64)
            for b in np.nonzero(live & (cnt > 0))[0]:
                hit = np.nonzero(ref.actions_u64[off[b]:off[b] + cnt[b]] == want[b])[0]
                if len(hit):
                    idx[b] = hit[0]
        sit = live & (cnt == 0) & (full > 0)
        idx[(idx < 0) | (idx >= cnt) | sit] = -1
        self.counts += [np.sum(live & (cnt == full)), np.sum(live & (cnt > 0) & (cnt < full)), np.sum(sit)]
        err = ref.envs["err"].copy()
        res = ref.step(idx.astype(np.int32), mode=0)       # -1: no-op, sticky bit and stats[7]
        ref.envs["err"][sit] = err[sit]                     # ... but an env that sat out keeps its bit
        if perm is not None:
            ref.deal(perm, lord, only_done=True, pool_games=G)
        return [np.array(a) for a in res]


# ------------------------------------------------------------------ device buffers
def _state_bytes(ref):
    f, meta = ref.export()
    return np.concatenate([f.reshape(-1).view(np.uint8), meta.view(np.uint8)])


def _state_to_dev(ref):
    return torch.as_tensor(_state_bytes(ref)).cuda()


def _check_state(state, ref, what):
    got = state.cpu().numpy()
    f, meta = ref.export()
    B = ref.B
    assert np.array_equal(got[:72 * B].view(np.uint64).reshape(9, B), f), "state fields, %s" % what
    assert np.array_equal(got[72 * B:].view(np.uint32), meta), "meta, %s" % what


class Lists:
    """offsets [B+1] + guard, packed moves and one-hot rows for `n` moves (the complete lists) + guard"""

    def __init__(self, B, n, f32=True):
        self.B = B
        self.offsets = torch.empty(B + 1 + GUARD_ENVS, dtype=torch.int32, device="cuda")
        self.u64 = torch.empty(n + GUARD, dtype=torch.int64, device="cuda")
        self.f32 = torch.empty((n + GUARD, 15, 4), dtype=torch.float32, device="cuda") if f32 else None

    def fill(self):
        self.offsets.view(torch.uint8).fill_(SENT_BYTE)
        self.u64.view(torch.uint8).fill_(0xA5)
        if self.f32 is not None:
            self.f32.fill_(float("nan"))

    def fill_unstored(self, au, cap):
        """the part of the complete lists that was not stored gets the true moves (see the module docstring)"""
        keep = min(cap, len(au))
        if keep < len(au):
            self.u64[keep:len(au)] = torch.as_tensor(au[keep:].view(np.int64)).cuda()

    def check(self, off, au, af, cap, what):
        """offsets, the stored prefix (and its one-hot rows when af is given) and the sentinels after it, on the device"""
        B, total = self.B, int(off[-1])
        keep = min(cap, total)
        o = self.offsets.cpu().numpy()
        assert np.array_equal(o[:B + 1], off), "offsets, %s" % what
        assert (o[B + 1:].view(np.uint8) == SENT_BYTE).all(), "offsets guard, %s" % what
        assert torch.equal(self.u64[:keep], torch.as_tensor(au[:keep].view(np.int64)).cuda()), "stored moves, %s" % what
        bad = int((self.u64[keep:] != int(SENT_U64.view(np.int64))).sum().item())
        assert bad == 0, "%d moves written past the stored part, %s" % (bad, what)
        if self.f32 is not None:
            if af is not None:
                assert torch.equal(self.f32[:keep], torch.as_tensor(af[:keep]).cuda()), "one-hot rows, %s" % what
            assert bool(torch.isnan(self.f32[keep:]).all()), "one-hot rows past the stored part, %s" % what


class Outs:
    """face and step results of B envs, each with guard slots"""

    def __init__(self, B, C):
        self.B, self.C = B, C
        self.face = torch.empty((B + GUARD_ENVS, C, 15, 4), dtype=torch.float32, device="cuda")
        self.r = torch.empty(B + GUARD_ENVS, dtype=torch.int8, device="cuda")
        self.done = torch.empty(B + GUARD_ENVS, dtype=torch.uint8, device="cuda")
        self.cat = torch.empty(B + GUARD_ENVS, dtype=torch.int8, device="cuda")
        self.reward = torch.empty((B + GUARD_ENVS, 3), dtype=torch.float32, device="cuda")

    def fill(self):
        self.face.fill_(float("nan"))
        self.reward.fill_(float("nan"))
        for t in (self.r, self.done, self.cat):
            t.view(torch.uint8).fill_(SENT_BYTE)

    def check_face(self, face, what):
        f = self.face.cpu().numpy()
        assert np.array_equal(f[:self.B], face), "face, %s" % what
        assert np.isnan(f[self.B:]).all(), "face guard, %s" % what

    def check_results(self, want, what):
        B = self.B
        for name, t, w in zip(("r", "done", "cat"), (self.r, self.done, self.cat), want[:3]):
            g = t.cpu().numpy()
            assert np.array_equal(g[:B], w), "%s, %s" % (name, what)
            assert (g[B:].view(np.uint8) == SENT_BYTE).all(), "%s guard, %s" % (name, what)
        rw = self.reward.cpu().numpy()
        assert np.array_equal(rw[:B], want[3]), "reward, %s" % what
        assert np.isnan(rw[B:]).all(), "reward guard, %s" % what


def _check_stats(stats, ref, what):
    got = stats.cpu().numpy()
    assert np.array_equal(got[:10], ref.stats[:10]), "stats %s != model %s, %s" % (got[:10], ref.stats[:10], what)


# ------------------------------------------------------------------ positions and capacities
def _adversarial_env(ref, b, hand, rng):
    """env b: the lord (to move, leading) holds `hand`, the other 54 - 20 cards go to the farmers, 17 each"""
    deck = np.array([4] * 13 + [1, 1])
    rest = np.repeat(np.arange(15), deck - hand)
    rng.shuffle(rest)
    e = ref.envs[b]
    e["hand"][:] = 0
    e["hist"][:] = 0
    e["recent"][:] = 0
    e["hand"][1] = hand
    e["hand"][0] = np.bincount(rest[:17], minlength=15)
    e["hand"][2] = np.bincount(rest[17:], minlength=15)
    e["cur"], e["done"], e["winner"], e["err"] = 1, 0, -1, 0


def _positions(D, O, B, variant, seed=1, G=2):
    """B envs: random deals played a few oracle steps on (leads and follows mixed), some envs replaced by adversarial
    leads (all of tile 2) -- env 37 (B > 37) or 0 holds the 497-move hand.  Returns the model, the 497 env and the deal pool."""
    rng = np.random.default_rng(seed)
    perm, lord = D.random_deals(B, seed=seed, pool_games=G)
    ref = O.RefBatch(B, variant)
    ref.deal(perm, lord, pool_games=G)
    for t in range(3):
        ref.observe(want_f32=False, want_face=False)
        ref.step(mode=2, seed=seed, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=G)
    big = 37 if B > 37 else 0
    _adversarial_env(ref, big, D.ADVERSARIAL_POOL[0], rng)
    for b in sorted(set(range(5, B, 97)) | set(range(64, min(B, 96)))):   # tile 2 (envs 64..95): leads only, many windows
        if b != big:
            _adversarial_env(ref, b, D.ADVERSARIAL_POOL[rng.integers(1, len(D.ADVERSARIAL_POOL))], rng)
    ref.stats[:] = 0
    return Model(O, ref), big, perm, lord


def _caps(off, big, win):
    """capacities that hit the boundaries the capacity rule has, for the lists `off` of B envs"""
    off = np.asarray(off, np.int64)
    B, total = len(off) - 1, int(off[-1])
    full = np.diff(off)
    caps = {0, 1, 2, total - 1, total, total + 1, 160 * B, 512 * B}
    heavy = [b for b in np.nonzero(full > HEAVY)[0] if b != big]
    for b in ([heavy[len(heavy) // 2]] if heavy else []) + [big]:
        caps |= {off[b] - 1, off[b], off[b] + 1, off[b] + full[b] // 2, off[b + 1]}
    nt = (B + 31) // 32
    tiles = off[np.minimum(np.arange(nt + 1) * 32, B)]
    for k in (1, nt // 2, nt - 1):
        if 0 < k < nt:
            caps |= {tiles[k] - 1, tiles[k], tiles[k] + 1}
    fat = [k for k in range(nt) if tiles[k + 1] - tiles[k] > 2 * win]
    for k in fat[:2]:
        for j in sorted({1, 2, int((tiles[k + 1] - tiles[k] - 1) // win)}):
            caps |= {tiles[k] + win * j - 1, tiles[k] + win * j, tiles[k] + win * j + 1}
    caps.add(tiles[nt - 1] + (total - tiles[nt - 1]) // 2)      # inside the last (partial) tile
    return sorted(int(c) for c in caps if c >= 0), bool(fat)


def _choice(mode, rng, model, B):
    """per-mode choices that hit every branch: indices inside the stored part, past it (inside the complete list) and past
    the list; moves in the stored part, only in the cut-off tail, and not in the list at all"""
    off = model.ref.offsets.astype(np.int64)
    full = np.diff(off)
    if mode == INDEX:
        c = rng.integers(0, np.maximum(full, 1)).astype(np.int64)
        c[rng.random(B) < 0.05] += 1000
        return c.astype(np.int32)
    if mode == MOD:
        return rng.integers(0, 1 << 32, B, dtype=np.uint64).astype(np.uint32).view(np.int32)
    if mode == PHILOX:
        return None
    au = model.ref.actions_u64
    mv = np.full(B, 0x1111, np.uint64)                              # a pair of 3s, 4s, 5s, 6s: rarely legal, never here
    for b in np.nonzero(full > 0)[0]:
        if rng.random() < 0.9:
            mv[b] = au[off[b] + rng.integers(0, full[b])]
    return mv.view(np.int64)


# ------------------------------------------------------------------ launchers
def _observe(D, variant, state, ws, lists, outs, cap, stats, B, emit=False):
    lists.fill()
    if outs is not None:
        outs.fill()
    if emit:
        rc = D.native.lib.ddz_legal_emit(_p(state), _p(ws), _p(lists.offsets), _p(lists.u64), cap, _p(stats), B, _stream())
    else:
        rc = D.native.lib.ddz_observe(_p(state), _p(ws), variant, _p(lists.offsets), _p(lists.u64), _p(lists.f32), cap,
                                      _p(outs.face), _p(stats), B, _stream())
    assert rc == 0, rc
    torch.cuda.synchronize()


def _rollout_step(D, variant, state, ws, prev, nxt, outs, mode, choice, seed, env0, stepno, perm, lord, G, cap, stats, B):
    nxt.fill()
    outs.fill()
    ch = None if choice is None else torch.as_tensor(choice).cuda()
    rc = D.native.lib.ddz_rollout_step(
        _p(state), _p(ws), variant, _p(prev.offsets), _p(prev.u64), _p(ch), mode, seed, env0, stepno, None,
        _p(perm), _p(lord), G, _p(outs.r), _p(outs.done), _p(outs.cat), _p(outs.reward),
        _p(nxt.offsets), _p(nxt.u64), _p(nxt.f32), cap, _p(outs.face), _p(stats), B, _stream())
    assert rc == 0, rc
    torch.cuda.synchronize()


def _single_launch_cases(D, oracle, variant, B, order, tile_order, modes):
    tile_order(order)
    model, big, perm, lord = _positions(D, oracle, B, variant, seed=B + variant)
    ref = model.ref
    G = 2
    perm_d, lord_d = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    base_envs = ref.envs.copy()
    off0, au0, af0, face0 = ref.observe()
    total = int(off0[-1])
    caps, fat = _caps(off0, big, WIN)
    assert fat or B < 64, "no tile with more than two windows of moves"
    assert int(np.diff(off0)[big]) == 497
    C = ref.C
    state0 = _state_to_dev(ref)
    ws = torch.zeros(D.native.lib.ddz_workspace_bytes(B) // 4, dtype=torch.int32, device="cuda")
    stats = torch.zeros(16, dtype=torch.int64, device="cuda")
    prev, outs = Lists(B, total), Outs(B, C)
    seen = {"cut": 0, "dropped": 0, "sticky": 0}
    rng = np.random.default_rng(7)
    for ci, cap in enumerate(caps):
        what = "variant %d, B %d, %s tiles, cap %d of %d" % (variant, B, order, cap, total)
        ref.envs[:] = base_envs
        ref.stats[:] = 0
        stats.zero_()
        state = state0.clone()
        off, au, af, face = model.observe(cap)
        _observe(D, variant, state, ws, prev, outs, cap, stats, B)
        prev.check(off, au, af, cap, "observe, " + what)
        outs.check_face(face, "observe, " + what)
        _check_stats(stats, ref, "observe, " + what)
        _check_state(state, ref, "observe, " + what)
        prev.fill_unstored(au, cap)
        envs_obs, lists_obs = ref.envs.copy(), (ref.offsets, ref.actions_u64)
        for mode in modes:
            wm = "mode %d, %s" % (mode, what)
            ref.envs[:] = envs_obs
            ref.offsets, ref.actions_u64 = lists_obs
            model.cap = cap
            ref.stats[:] = 0
            stats.zero_()
            st = state.clone()
            full, cnt = model.stored()
            seen["cut"] += int(np.sum((cnt > 0) & (cnt < full)))
            seen["dropped"] += int(np.sum((cnt == 0) & (full > 0)))
            choice = _choice(mode, rng, model, B)
            env0, stepno = (1 << 33) + 11, 5 + mode
            want = model.step(mode, choice, seed=4242, env0=env0, stepno=stepno, perm=perm, lord=lord, G=G)
            seen["sticky"] += int(np.sum(ref.envs["err"]))
            rows = (mode == ci % 4)                     # one-hot rows of the new lists: one mode per capacity
            off2, au2, af2, face2 = model.observe(cap, want_f32=rows)
            nxt = Lists(B, int(off2[-1]))
            _rollout_step(D, variant, st, ws, prev, nxt, outs, mode, choice, 4242, env0, stepno, perm_d, lord_d, G, cap,
                          stats, B)
            outs.check_results(want, wm)
            _check_state(st, ref, wm)
            nxt.check(off2, au2, af2, cap, wm)
            outs.check_face(face2, wm)
            _check_stats(stats, ref, wm)
    return seen


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("variant,order", [(0, "auto"), (1, "auto"), (2, "auto"), (3, "auto"), (2, "ticket")])
def test_observe_and_fused_step_at_every_capacity(D, oracle, tile_order, variant, order):
    """ddz_observe at B = 1000 (not a multiple of 32) at every boundary capacity, each followed by ddz_rollout_step from
    the lists it cut in all four choice modes"""
    seen = _single_launch_cases(D, oracle, variant, 1000, order, tile_order, (INDEX, MOD, PHILOX, MOVE))
    assert seen["cut"] > 0 and seen["dropped"] > 1000 and seen["sticky"] > 0, seen


@pytest.mark.parametrize("order", ["auto", "ticket"])
def test_single_env_at_every_capacity(D, oracle, tile_order, order):
    """B = 1: the 497-move lead cut at every capacity from 0 to past its end, in all four variants and choice modes"""
    for variant in range(4):
        seen = _single_launch_cases(D, oracle, variant, 1, order, tile_order, (INDEX, MOD, PHILOX, MOVE))
        assert seen["cut"] > 0 and seen["dropped"] > 0, seen


@pytest.mark.parametrize("order", ["auto", "ticket"])
def test_legal_emit_at_every_capacity(D, oracle, tile_order, order):
    """ddz_legal_emit stages 896 moves per window instead of 320: its window boundaries, and the rest of the caps"""
    tile_order(order)
    for B in (1000, 1):
        model, big, _, _ = _positions(D, oracle, B, 0, seed=50 + B)
        ref = model.ref
        off0 = ref.observe(want_f32=False, want_face=False)[0]
        caps, fat = _caps(off0, big, EMIT_WIN)
        assert fat or B == 1, "no tile with more than two emit windows of moves"
        state = _state_to_dev(ref)
        ws = torch.zeros(D.native.lib.ddz_workspace_bytes(B) // 4, dtype=torch.int32, device="cuda")
        stats = torch.zeros(16, dtype=torch.int64, device="cuda")
        lists = Lists(B, int(off0[-1]), f32=False)
        for cap in caps:
            ref.stats[:] = 0
            stats.zero_()
            off, au, _, _ = model.observe(cap, want_f32=False, want_face=False)
            _observe(D, 0, state, ws, lists, None, cap, stats, B, emit=True)
            what = "emit, B %d, %s tiles, cap %d of %d" % (B, order, cap, int(off[-1]))
            lists.check(off, au, None, cap, what)
            _check_stats(stats, ref, what)
            _check_state(state, ref, what)


@pytest.mark.parametrize("variant,mode,steps", [(2, PHILOX, 48), (0, MOD, 40)])
def test_fused_steps_on_cut_lists(D, oracle, variant, mode, steps):
    """4096 envs stepped 40+ times by ddz_rollout_step at a capacity that about half of the launches overflow (the fresh
    deals' leads need about 320 000 moves, later steps about 20 000): every step against the model (results, state, lists,
    rows, face, stats).  Cut lists, dropped lists and complete lists must all be played."""
    B, G, seed, env0, cap = 4096, 4, 31 + variant, 12345, 30000
    perm, lord = D.random_deals(B, seed=seed, pool_games=G)
    perm_d, lord_d = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    rng = np.random.default_rng(seed)
    ents = [rng.integers(0, 1 << 32, B, dtype=np.uint64).astype(np.uint32).view(np.int32) for _ in range(steps)]
    ref = oracle.RefBatch(B, variant)
    ref.deal(perm, lord, pool_games=G)
    model = Model(oracle, ref)
    state = _state_to_dev(ref)
    ws = torch.zeros(D.native.lib.ddz_workspace_bytes(B) // 4, dtype=torch.int32, device="cuda")
    stats = torch.zeros(16, dtype=torch.int64, device="cuda")
    outs = Outs(B, ref.C)
    off, au, af, face = model.observe(cap)
    prev = Lists(B, int(off[-1]))
    _observe(D, variant, state, ws, prev, outs, cap, stats, B)
    prev.check(off, au, af, cap, "first observe")
    overflowed = int(off[-1]) > cap
    for t in range(steps):
        prev.fill_unstored(au, cap)
        choice = ents[t] if mode == MOD else None
        want = model.step(mode, choice, seed=seed, env0=env0, stepno=t, perm=perm, lord=lord, G=G)
        off, au, af, face = model.observe(cap, want_f32=(t % 4 == 0))
        overflowed += int(off[-1]) > cap
        nxt = Lists(B, int(off[-1]))
        _rollout_step(D, variant, state, ws, prev, nxt, outs, mode, choice, seed, env0, t, perm_d, lord_d, G, cap, stats, B)
        what = "step %d, cap %d of %d" % (t, cap, int(off[-1]))
        outs.check_results(want, what)
        _check_state(state, ref, what)
        nxt.check(off, au, af, cap, what)
        outs.check_face(face, what)
        _check_stats(stats, ref, what)
        prev = nxt
    complete, cut, dropped = (int(x) for x in model.counts)
    print("variant %d, cap %d: env-steps from complete lists %d, cut lists %d, dropped lists %d; launches that overflowed "
          "%d of %d" % (variant, cap, complete, cut, dropped, overflowed, steps + 1))
    # a launch cuts at most one list (the one that straddles cap), so cut lists are counted per launch
    assert complete >= 300 and dropped >= 300 and cut >= 10, model.counts
    assert 5 <= overflowed <= steps - 4, overflowed


def _rollout_steps_case(D, oracle, variant, mode, B, K, cap, seed=61, steps_before=2):
    """ddz_rollout_steps: K slices against the model, slice by slice, with guard memory after the last slice"""
    G, env0, stepno0 = 3, 777, 100
    perm, lord = D.random_deals(B, seed=seed, pool_games=G)
    perm_d, lord_d = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    ref = oracle.RefBatch(B, variant)
    ref.deal(perm, lord, pool_games=G)
    for t in range(steps_before):                      # mid-game positions: leads and follows mixed
        ref.observe(want_f32=False, want_face=False)
        ref.step(mode=2, seed=seed, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=G)
    ref.stats[:] = 0
    model, C = Model(oracle, ref), ref.C
    state = _state_to_dev(ref)
    ws = torch.zeros(D.native.lib.ddz_workspace_bytes(B) // 4, dtype=torch.int32, device="cuda")
    stats = torch.zeros(16, dtype=torch.int64, device="cuda")
    off, au, af, face = model.observe(cap)
    prev, outs = Lists(B, int(off[-1])), Outs(B, C)
    _observe(D, variant, state, ws, prev, outs, cap, stats, B)
    prev.check(off, au, af, cap, "observe before the launch")
    _check_stats(stats, ref, "observe before the launch")
    prev.fill_unstored(au, cap)
    rng = np.random.default_rng(seed)
    ent = rng.integers(0, 1 << 32, (K, B), dtype=np.uint64).astype(np.uint32).view(np.int32) if mode == MOD else None
    want = []
    for s in range(K):                                  # the model's trajectory first: it sizes the buffers
        res = model.step(mode, None if ent is None else ent[s], seed=seed, env0=env0, stepno=stepno0 + s, perm=perm,
                         lord=lord, G=G)
        want.append((res, model.observe(cap)))
    tail = max(int(w[1][0][-1]) for w in want) + GUARD  # room for the complete lists after the last slice
    n = K * cap + tail
    u64 = torch.empty(n, dtype=torch.int64, device="cuda").view(torch.uint8).fill_(0xA5).view(torch.int64)
    f32 = torch.full((n, 15, 4), float("nan"), dtype=torch.float32, device="cuda")
    offs = torch.empty(K * (B + 1) + GUARD_ENVS, dtype=torch.int32, device="cuda")
    offs.view(torch.uint8).fill_(SENT_BYTE)
    r, done, cat = (torch.empty(K * B + GUARD_ENVS, dtype=dt, device="cuda") for dt in (torch.int8, torch.uint8, torch.int8))
    for t in (r, done, cat):
        t.view(torch.uint8).fill_(SENT_BYTE)
    reward = torch.full((K * B + GUARD_ENVS, 3), float("nan"), dtype=torch.float32, device="cuda")
    facebuf = torch.full((K * B + GUARD_ENVS, C, 15, 4), float("nan"), dtype=torch.float32, device="cuda")
    ch = None if ent is None else torch.as_tensor(ent).cuda()
    rc = D.native.lib.ddz_rollout_steps(
        _p(state), _p(ws), variant, K, _p(prev.offsets), _p(prev.u64), _p(ch), mode, seed, env0, stepno0, None,
        _p(perm_d), _p(lord_d), G, _p(r), _p(done), _p(cat), _p(reward), _p(offs), _p(u64), _p(f32), cap, _p(facebuf),
        _p(stats), B, _stream())
    assert rc == 0, "ddz_rollout_steps returned %d at cap %d" % (rc, cap)
    torch.cuda.synchronize()
    exp_u = np.full(n, SENT_U64, np.uint64)
    exp_f = np.full((n, 15, 4), np.nan, np.float32)
    for s in range(K):                                  # later slices overwrite nothing of earlier ones: stride cap
        au_s, af_s = want[s][1][1], want[s][1][2]
        keep = min(cap, len(au_s))
        exp_u[s * cap:s * cap + keep] = au_s[:keep]
        exp_f[s * cap:s * cap + keep] = af_s[:keep]
    got_u = u64.cpu().numpy().view(np.uint64)
    for s in range(K):
        (rr, rd, rcat, rrew), (off_s, _, _, face_s) = want[s]
        what = "slice %d of %d, mode %d, cap %d" % (s, K, mode, cap)
        sl = slice(s * B, (s + 1) * B)
        assert np.array_equal(offs[s * (B + 1):(s + 1) * (B + 1)].cpu().numpy(), off_s), "offsets, " + what
        assert np.array_equal(r[sl].cpu().numpy(), rr) and np.array_equal(done[sl].cpu().numpy(), rd), "r / done, " + what
        assert np.array_equal(cat[sl].cpu().numpy(), rcat), "cat, " + what
        assert np.array_equal(reward[sl].cpu().numpy(), rrew), "reward, " + what
        assert np.array_equal(facebuf[sl].cpu().numpy(), face_s), "face, " + what
        assert np.array_equal(got_u[s * cap:(s + 1) * cap], exp_u[s * cap:(s + 1) * cap]), "moves, " + what
    assert np.array_equal(got_u, exp_u), "moves after the last slice"
    assert torch.equal(f32.view(torch.int32), torch.as_tensor(exp_f).cuda().view(torch.int32)), "one-hot rows"
    for name, t in (("offsets", offs[K * (B + 1):]), ("r", r[K * B:]), ("done", done[K * B:]), ("cat", cat[K * B:])):
        assert (t.cpu().numpy().view(np.uint8) == SENT_BYTE).all(), name + " guard"
    assert bool(torch.isnan(reward[K * B:]).all()) and bool(torch.isnan(facebuf[K * B:]).all()), "reward / face guard"
    _check_state(state, ref, "after %d slices" % K)
    _check_stats(stats, ref, "after %d slices" % K)
    return model


@pytest.mark.parametrize("variant,mode", [(2, PHILOX), (3, MOD)])
def test_multi_step_launch_on_cut_lists(D, oracle, variant, mode):
    B, K = 2048 + 37, 8
    model = _rollout_steps_case(D, oracle, variant, mode, B, K, cap=9 * B)
    complete, cut, dropped = (int(x) for x in model.counts)
    assert complete > 0 and cut > 0 and dropped > 0, model.counts


@pytest.mark.parametrize("mode", [PHILOX, MOD])
def test_capacity_zero_multi_step_launch(D, oracle, mode):
    """ddz_rollout_steps at cap = 0 runs all K = 3 steps, and every live env sits each of them out"""
    B = 1000
    model = _rollout_steps_case(D, oracle, 2, mode, B, 3, cap=0)
    assert model.counts[0] == model.counts[1] == 0 and model.counts[2] == 3 * B


@pytest.mark.parametrize("mode", [PHILOX, MOD])
def test_capacity_zero(D, oracle, mode):
    """cap = 0 is accepted by every launcher: ddz_observe writes the offsets and the face, nothing else, and every live env
    sits a ddz_rollout_step from such lists out"""
    B = 1000
    model, _, _, _ = _positions(D, oracle, B, 2, seed=13)
    ref = model.ref
    before = ref.export()
    state = _state_to_dev(ref)
    ws = torch.zeros(D.native.lib.ddz_workspace_bytes(B) // 4, dtype=torch.int32, device="cuda")
    stats = torch.zeros(16, dtype=torch.int64, device="cuda")
    ref.stats[:] = 0
    off, au, af, face = model.observe(0)
    prev, nxt, outs = Lists(B, int(off[-1])), Lists(B, int(off[-1])), Outs(B, ref.C)
    _observe(D, 2, state, ws, prev, outs, 0, stats, B)
    prev.check(off, au, af, 0, "observe at cap 0")
    outs.check_face(face, "observe at cap 0")
    prev.fill_unstored(au, 0)
    rng = np.random.default_rng(3)
    choice = rng.integers(0, 1 << 31, B).astype(np.int32) if mode == MOD else None
    want = model.step(mode, choice, seed=9, env0=0, stepno=0)
    off, au, af, face = model.observe(0)
    _rollout_step(D, 2, state, ws, prev, nxt, outs, mode, choice, 9, 0, 0, None, None, 1, 0, stats, B)
    outs.check_results(want, "rollout_step at cap 0")
    nxt.check(off, au, af, 0, "rollout_step at cap 0")
    outs.check_face(face, "rollout_step at cap 0")
    _check_state(state, ref, "rollout_step at cap 0")
    _check_stats(stats, ref, "rollout_step at cap 0")
    assert all(np.array_equal(a, b) for a, b in zip(before, ref.export()))
    assert (want[2] == -1).all() and int(ref.stats[4]) == 0 and int(ref.stats[7]) == B + 2   # B envs sat out, two observations overflowed


def test_host_rollout_groups_at_a_small_capacity(D, oracle):
    """HostRolloutGroups (two groups) with max_actions_per_env = 12: host r | done | cat of every step and the final state
    against one model per group (each group has its own lists and capacity)"""
    B, P, NG, per_env, steps = 2048, 2, 2, 12, 60
    Bg = B // NG
    rng = np.random.default_rng(17)
    perm, lord = D.random_deals(B, seed=23, pool_games=P)
    ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=NG, seed=3, max_actions_per_env=per_env)
    ge.prepare(perm, lord, pool_games=P)
    host = D.HostRolloutGroups(ge)
    pp, lp = perm.reshape(P, B, 54), lord.reshape(P, B)
    models, pools = [], []
    for g in range(NG):
        pg = np.ascontiguousarray(pp[:, g * Bg:(g + 1) * Bg]).reshape(-1, 54)
        lg = np.ascontiguousarray(lp[:, g * Bg:(g + 1) * Bg]).reshape(-1)
        ref = oracle.RefBatch(Bg, 2)
        ref.deal(pg, lg, pool_games=P)
        m = Model(oracle, ref)
        m.observe(ge.envs[g].cap, want_f32=False, want_face=False)
        models.append(m)
        pools.append((pg, lg))
    ents = [torch.as_tensor(rng.integers(0, 1 << 31, B).astype(np.int32)).pin_memory() for _ in range(4)]
    for t in range(steps):
        got = D.HostRolloutGroups.wait(host.step(ents[t % 4]))
        for g, m in enumerate(models):
            rr, rd, rc, _ = m.step(MOD, ents[t % 4].numpy()[g * Bg:(g + 1) * Bg], perm=pools[g][0], lord=pools[g][1], G=P)
            m.observe(ge.envs[g].cap, want_f32=False, want_face=False)
            assert np.array_equal(got.r[g], rr) and np.array_equal(got.done[g], rd) and np.array_equal(got.cat[g], rc), (t, g)
    ge.join()
    torch.cuda.synchronize()
    for g, (e, m) in enumerate(zip(ge.envs, models)):
        f, meta = m.ref.export()
        ef, emeta = e._fields()
        assert np.array_equal(ef.cpu().numpy().view(np.uint64), f) and np.array_equal(emeta.cpu().numpy().view(np.uint32), meta), g
    want_stats = sum(m.ref.stats for m in models)
    assert np.array_equal(ge.stats.cpu().numpy()[:10], want_stats[:10])
    counts = sum(m.counts for m in models)
    assert counts[1] > 0 and counts[2] > 0 and counts[0] > 0, counts


def test_eager_layer_after_cut_lists(D, oracle):
    """after fused steps that cut lists, valid_actions() grows the buffers and observes again, and step_random() plays the
    complete list (ddz_step: capacity unknown = lists complete)"""
    B, G, seed = 512, 2, 5
    perm, lord = D.random_deals(B, seed=8, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvCooperation(B, seed=seed, max_actions_per_env=8)
    env.prepare(pd, ld, pool_games=G)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=G)
    model = Model(oracle, ref)
    cap0 = env.cap
    for t in range(6):
        model.observe(cap0, want_f32=False, want_face=False)
        want = model.step(PHILOX, seed=seed, env0=0, stepno=t, perm=perm, lord=lord, G=G)
        r, done, cat = env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)
        assert np.array_equal(r.cpu().numpy(), want[0]) and np.array_equal(cat.cpu().numpy(), want[2]), t
    assert model.counts[1] > 0 and model.counts[2] > 0, model.counts
    off, au, af, face = model.observe(cap0)
    assert int(off[-1]) > cap0                          # the fused step's lists of this state were cut
    model.ref.stats[8] += int(off[-1])                  # ... and valid_actions() observes them once more, complete
    rows, offsets = env.valid_actions()
    assert env.cap >= int(off[-1]) > cap0
    assert np.array_equal(offsets.cpu().numpy(), off) and np.array_equal(rows.cpu().numpy(), af)
    assert np.array_equal(env.actions_packed.cpu().numpy().view(np.uint64), au)
    assert np.array_equal(env.face.cpu().numpy(), face)
    model.cap = env.cap
    want = model.step(PHILOX, seed=seed, env0=0, stepno=6)
    r, done, cat = env.step_random()
    assert np.array_equal(r.cpu().numpy(), want[0]) and np.array_equal(done.cpu().numpy(), want[1])
    assert np.array_equal(cat.cpu().numpy(), want[2]) and np.array_equal(env.reward.cpu().numpy(), want[3])
    torch.cuda.synchronize()
    f, meta = ref.export()
    ef, emeta = env._fields()
    assert np.array_equal(ef.cpu().numpy().view(np.uint64), f) and np.array_equal(emeta.cpu().numpy().view(np.uint32), meta)
    assert np.array_equal(env.stats.cpu().numpy()[:10], ref.stats[:10])
