"""Action ids (include/ddz_b200.h: ddz_move_ids, ddz_moves_of_ids, ddz_legal_mask; D.move_ids / moves_of_ids / action_space,
BatchedEnv.legal_ids / legal_mask / step_ids): a fixed index per move in the universe of 13 551 moves, which is the
reference's action space (card.py) plus the 24 rocket-kicker moves of r.get_moves, in oracle.universe() order.

CPU: the product's id code compiled for the host (tests/host_harness/ids_host.cpp) against the oracle's universe and its
ddz_ref_classify, the generated block table against card_space.npz, the argument checks, the kernels' register counts.
GPU (-m gpu): the kernels bit for bit against the same references, the reference's own masks (legal_sets.npz), mid-game
lists of all four env classes, capacities that cut and drop lists, step_ids against step(index), and a fixed-head policy."""
import ctypes as C
import os
import re
import shutil
import subprocess
import sys
from math import comb

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "doudizhu-rl_b200", "csrc")
NIDS, WORDS = 13551, 424
INVALID = np.uint64(0xFFFFFFFFFFFFFFFF)
SENT = 0x5C


# ------------------------------------------------------------------ references
@pytest.fixture(scope="module")
def uni(oracle):
    """(packed uint64 [13551] in id order, is_extra [13551], sorted packed, id of each sorted entry)"""
    cnt, _, _, _, extra = oracle.universe()
    packed = oracle.pack(cnt).astype(np.uint64)
    order = np.argsort(packed)
    return packed, extra.astype(bool), packed[order], order.astype(np.int32)


def ref_ids(uni, moves):
    """universe index of every packed move (-1 when it is not in the universe)"""
    _, _, srt, idx = uni
    m = np.asarray(moves, np.uint64)
    pos = np.clip(np.searchsorted(srt, m), 0, len(srt) - 1)
    return np.where(srt[pos] == m, idx[pos], -1).astype(np.int32)


def near_misses(oracle):
    """every universe move with one card added at each rank, or removed at each rank that has one (counts may exceed 4)"""
    cnt = oracle.universe()[0].astype(np.int16)
    out = []
    for r in range(15):
        for d in (1, -1):
            x = cnt.copy()
            x[:, r] += d
            out.append(x[x[:, r] >= 0])
    v = np.concatenate(out)
    packed = (v.astype(np.uint64) << (np.arange(15, dtype=np.uint64) * np.uint64(4))).sum(1, dtype=np.uint64)
    want = np.array([oracle.classify(row)[0] for row in v.astype(np.int8)], np.int32)
    return packed, want


def random_values(rng, n):
    """random 64-bit values (nibbles 0..15, so mostly nibbles above 4) and random count vectors with counts 0..4"""
    raw = rng.integers(0, 2 ** 64, n, dtype=np.uint64)
    low = rng.integers(0, 5, (n, 15)) * (rng.random((n, 15)) < 0.2)
    packed = (low.astype(np.uint64) << (np.arange(15, dtype=np.uint64) * np.uint64(4))).sum(1, dtype=np.uint64)
    return np.concatenate([raw, raw >> np.uint64(4), packed]), low.astype(np.int8)


# ------------------------------------------------------------------ CPU: the id code compiled for the host
@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("ids_host") / "libids_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wno-unknown-pragmas", "-o", lib,
                           os.path.join(HERE, "host_harness", "ids_host.cpp")])
    L = C.CDLL(lib)
    L.ids_host_move_ids.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p]
    L.ids_host_moves_of_ids.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p]
    L.ids_host_blocks.argtypes = [C.c_void_p]
    return L


def host_ids(L, moves):
    m = np.ascontiguousarray(moves, np.uint64)
    out = np.full(len(m), -7, np.int32)
    L.ids_host_move_ids(m.ctypes.data, len(m), out.ctypes.data)
    return out


def host_moves(L, ids):
    i = np.ascontiguousarray(ids, np.int32)
    out = np.zeros(len(i), np.uint64)
    L.ids_host_moves_of_ids(i.ctypes.data, len(i), out.ctypes.data)
    return out


def test_host_ids_of_the_universe(harness, uni):
    packed = uni[0]
    assert np.array_equal(host_ids(harness, packed), np.arange(NIDS))
    assert np.array_equal(host_moves(harness, np.arange(NIDS)), packed)
    bad = np.array([-1, -2 ** 31, NIDS, NIDS + 1, 2 ** 31 - 1], np.int32)
    assert (host_moves(harness, bad) == INVALID).all()


def test_host_ids_of_near_misses(harness, oracle):
    packed, want = near_misses(oracle)
    assert len(packed) > 280000 and (want >= 0).any()
    assert np.array_equal(host_ids(harness, packed), want)


def test_host_ids_of_random_values(harness, oracle, uni):
    rng = np.random.default_rng(11)
    vals, low = random_values(rng, 100000)
    got = host_ids(harness, vals)
    assert np.array_equal(got, ref_ids(uni, vals))
    big = vals[:200000]
    nib = (big[:, None] >> (np.arange(16, dtype=np.uint64) * np.uint64(4))) & np.uint64(15)
    assert (got[:200000][(nib > 4).any(1)] == -1).all()
    sample = np.array([oracle.classify(row)[0] for row in low[:5000]], np.int32)
    assert np.array_equal(got[200000:205000], sample)


def _load_generator():
    sys.path.insert(0, CSRC)
    try:
        import make_action_ids
    finally:
        sys.path.remove(CSRC)
    return make_action_ids


def test_block_table_restates_card_py(harness, golden, uni):
    gen = _load_generator()
    words, cat_first, line_first, n = gen.table()
    assert n == NIDS
    table = np.zeros(512, np.uint64)
    nb = harness.ids_host_blocks(table.ctypes.data)
    assert nb == len(words) and [int(w) for w in table[:nb]] == words           # the compiled table is the generated one
    out = subprocess.run([sys.executable, os.path.join(CSRC, "make_action_ids.py")], capture_output=True, text=True, check=True)
    assert out.stdout == open(os.path.join(CSRC, "ddz_action_ids.inc")).read()   # and the committed file is current
    # expand every block: main part + each kicker subset of the pool in itertools.combinations order
    from itertools import combinations
    moves, extra = [], []
    for w in words:
        first, main, pool = w & 0xFFFF, (w >> 16) & 0x7FFF, (w >> 32) & 0x7FFF
        mult, kmult, k = (w >> 48) & 7, (w >> 52) & 7, (w >> 56) & 7
        assert first == len(moves)
        ranks = [r for r in range(15) if pool >> r & 1]
        for ks in combinations(ranks, k):
            c = np.zeros(15, np.int8)
            c[[r for r in range(15) if main >> r & 1]] = mult
            c[list(ks)] = kmult
            moves.append(c)
            extra.append(k == 2 and 13 in ks and 14 in ks and (w >> 60) in (10, 13))
        assert len(moves) - first == comb(len(ranks), k)
    moves, extra = np.array(moves), np.array(extra)
    assert np.array_equal(moves[~extra], golden.card_space["counts"])            # card.py's 13 527 moves, in order
    assert np.array_equal(extra, uni[1]) and extra.sum() == 24


def test_argument_checks_before_any_cuda_call():
    import ddz_b200 as D
    L, E = D.native.lib, D.native.E_ARG
    assert L.ddz_move_ids(None, 4, None, None) == E and L.ddz_move_ids(8, 4, None, None) == E
    assert L.ddz_move_ids(8, -1, 8, None) == E and L.ddz_move_ids(None, 0, None, None) == 0        # n = 0: no launch
    assert L.ddz_moves_of_ids(None, 4, 8, None) == E and L.ddz_moves_of_ids(8, 4, None, None) == E
    assert L.ddz_moves_of_ids(8, -5, 8, None) == E and L.ddz_moves_of_ids(None, 0, None, None) == 0
    ok = dict(offsets=16, actions=16, cap=64, layout=D.native.MASK_BITS, out=16, B=4)

    def mask(**kw):
        a = dict(ok, **kw)
        return L.ddz_legal_mask(a["offsets"], a["actions"], a["cap"], a["layout"], a["out"], None, a["B"], None)
    for bad in (dict(offsets=None), dict(out=None), dict(actions=None), dict(cap=-1), dict(B=0), dict(B=-3),
                dict(layout=2), dict(layout=-1), dict(out=17)):
        assert mask(**bad) == E, bad
    assert mask(actions=None, cap=0, out=None) == E
    assert D.native.NUM_ACTION_IDS == NIDS and D.native.MASK_WORDS == WORDS
    hdr = open(os.path.join(ROOT, "include", "ddz_b200.h")).read()
    for name, val in (("DDZ_NUM_ACTION_IDS", "13551"), ("DDZ_MASK_WORDS", "424"), ("DDZ_MASK_BITS", "0"), ("DDZ_MASK_BYTES", "1"),
                      ("DDZ_MOVE_INVALID", "0xFFFFFFFFFFFFFFFFull")):
        assert re.search(r"#define %s %s\b" % (name, val), hdr), name


# register counts of the kernels that existed before action ids (one entry per instantiation), and of the new ones
REGS_BEFORE = {"k_determinize": [74], "k_encode_actions": [32], "k_env": [55] + [72] * 10, "k_face": [27, 32, 32, 37],
               "k_face_gather": [28, 28, 32, 32, 34, 34, 38, 38], "k_kth_moves": [31], "k_legal_count": [28],
               "k_legal_flat": [72], "k_mcts_moves": [46], "k_playout": [64, 72],
               "k_q_features": [121] * 4 + [124] * 4 + [127] * 8, "k_reset": [51], "k_select_actions": [26],
               "k_state_actions": [27, 32, 34, 39], "k_uct": [128], "k_uct_pool": [32]}
REGS_NEW = {"k_move_ids": [24], "k_moves_of_ids": [20], "k_legal_mask": [30, 30]}


def test_register_counts():
    import ddz_b200 as D
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-res-usage", D.native.LIB_PATH], capture_output=True, text=True).stdout
    regs, stack = {}, {}
    for name, reg, st, local in re.findall(r"Function _ZN3ddz\d+(k_[a-z_]+?)[IE]\S*:\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)", out):
        regs.setdefault(name, []).append(int(reg))
        stack.setdefault(name, []).append(int(st) + int(local))
    assert {k: sorted(v) for k, v in regs.items()} == dict(REGS_BEFORE, **REGS_NEW)
    for k in REGS_NEW:
        assert set(stack[k]) == {0}, k                                           # no stack, no spills


# ------------------------------------------------------------------ GPU
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def D():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


CLASSES = (("BatchedEnv", 0), ("BatchedEnvComplicated", 1), ("BatchedEnvCooperation", 2), ("BatchedEnvCooperationSimplify", 3))


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def expected_masks(offsets, ids, B):
    """bool [B, 13551] and int32 [B, 424] rows of the CSR ids (on the device)"""
    off = torch.as_tensor(np.asarray(offsets, np.int64), device="cuda")
    ids = torch.as_tensor(np.asarray(ids, np.int64), device="cuda")
    owner = torch.repeat_interleave(torch.arange(B, device="cuda"), off[1:] - off[:-1], output_size=len(ids))
    m = torch.zeros((B, NIDS), dtype=torch.bool, device="cuda")
    m[owner, ids] = True
    return m, bits_of(m)


def bits_of(m):
    pad = torch.zeros((m.shape[0], WORDS * 32), dtype=torch.int64, device=m.device)
    pad[:, :NIDS] = m.to(torch.int64)
    return (pad.view(-1, WORDS, 32) << torch.arange(32, device=m.device)).sum(-1)      # the uint32 words, as int64


def run_mask(D, offsets, actions, cap, layout, B, stats=None, shift=0):
    """ddz_legal_mask into a sentinel-filled buffer with guard bytes before and after (bytes rows start `shift` bytes past a
    16-byte boundary); returns the rows and asserts the guards are untouched"""
    nbytes = B * (NIDS if layout == D.native.MASK_BYTES else 4 * WORDS)
    g = 64
    buf = torch.full((nbytes + 2 * g + 16,), SENT, dtype=torch.uint8, device="cuda")
    s = g + shift
    rc = D.native.lib.ddz_legal_mask(offsets.data_ptr(), None if actions is None else actions.data_ptr(), cap, layout,
                                     buf.data_ptr() + s, None if stats is None else stats.data_ptr(), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    assert (buf[:s] == SENT).all() and (buf[s + nbytes:] == SENT).all()
    rows = buf[s:s + nbytes]
    if layout == D.native.MASK_BYTES:
        rows = rows.view(B, NIDS)
        assert ((rows == 0) | (rows == 1)).all()                                   # every byte was written
        return rows.to(torch.bool)
    return rows.clone().view(torch.int32).view(B, WORDS).to(torch.int64).bitwise_and(0xFFFFFFFF)


@pytest.mark.gpu
def test_ids_of_the_universe_on_the_device(D, oracle, uni):
    packed = uni[0]
    got = D.move_ids(packed)
    assert got.dtype == torch.int32 and np.array_equal(got.cpu().numpy(), np.arange(NIDS))
    back = D.moves_of_ids(torch.arange(NIDS, dtype=torch.int32, device="cuda"))
    assert back.dtype == torch.int64 and np.array_equal(_u64(back), packed)
    assert np.array_equal(D.move_ids(back).cpu().numpy(), np.arange(NIDS))         # round trip
    bad = torch.tensor([-1, -2 ** 31, NIDS, NIDS + 7, 2 ** 31 - 1], dtype=torch.int32)
    assert (_u64(D.moves_of_ids(bad)) == INVALID).all()
    nm, want = near_misses(oracle)
    assert np.array_equal(D.move_ids(nm).cpu().numpy(), want)
    vals, _ = random_values(np.random.default_rng(5), 300000)
    assert np.array_equal(D.move_ids(vals).cpu().numpy(), ref_ids(uni, vals))
    sp = D.action_space()
    assert np.array_equal(_u64(sp.moves), packed)
    cp = sp.card_py_index.cpu().numpy()
    assert np.array_equal(cp < 0, uni[1]) and np.array_equal(cp[~uni[1]], np.arange(13527))
    assert np.array_equal(sp.id_of_card_py.cpu().numpy(), np.nonzero(~uni[1])[0])
    assert D.move_ids(torch.zeros((3, 0), dtype=torch.int64, device="cuda")).shape == (3, 0)


@pytest.mark.gpu
def test_ids_and_masks_of_get_mask_onehot60(D, golden):
    g = golden.legal_sets
    moves, off = D.get_moves(g["hands"], g["lasts"])
    ids = D.move_ids(moves).cpu().numpy()
    assert np.array_equal(off.cpu().numpy().astype(np.int64), g["legal_off"]) and np.array_equal(ids, g["legal_idx"])
    B = len(g["hands"])
    want_b, want_w = expected_masks(g["legal_off"], g["legal_idx"], B)
    for shift in (0, 3):
        assert torch.equal(run_mask(D, off, moves, moves.numel(), D.native.MASK_BYTES, B, shift=shift), want_b)
    assert torch.equal(run_mask(D, off, moves, moves.numel(), D.native.MASK_BITS, B), want_w)


def _mirrored_rollout(D, O, cls_name, variant, B, steps, seed):
    env = getattr(D, cls_name)(B, seed=seed)
    perm, lord = D.random_deals(B, seed=seed + 1)
    env.prepare(perm, lord)
    ref = O.RefBatch(B, variant)
    ref.deal(perm, lord)
    for t in range(steps):
        ref.observe(want_f32=False, want_face=False)
        env.step_random()
        ref.step(mode=2, seed=seed, env0=0, step=t)
    return env, ref


def check_env_ids(D, env, ref, uni):
    off, au, _, _ = ref.observe(fast=False, want_f32=False, want_face=False)   # the definitional generator
    B = env.B
    assert np.array_equal(env.offsets.cpu().numpy(), off) and np.array_equal(_u64(env.actions_packed), au)
    want = ref_ids(uni, au)
    got = env.legal_ids().cpu().numpy()
    assert np.array_equal(got, want) and (want >= 0).all()
    inner = np.ones(len(got), bool)
    inner[off[:-1][off[:-1] < len(got)]] = False
    assert (np.diff(got.astype(np.int64))[inner[1:]] > 0).all()                 # strictly increasing within each list
    want_b, want_w = expected_masks(off, want, B)
    mb, mw = env.legal_mask("bool"), env.legal_mask("bits")
    assert mb.dtype == torch.bool and mb.shape == (B, NIDS) and mw.dtype == torch.int32 and mw.shape == (B, WORDS)
    assert torch.equal(mb, want_b) and torch.equal(mw.to(torch.int64).bitwise_and(0xFFFFFFFF), want_w)
    o, a = env.offsets, env._actions_u64[env._cur]
    for shift in (0, 5, 15):
        assert torch.equal(run_mask(D, o, a, env.cap, D.native.MASK_BYTES, B, shift=shift), want_b)
    assert torch.equal(run_mask(D, o, a, env.cap, D.native.MASK_BITS, B), want_w)
    finished = np.diff(off) == 0
    assert not mb[torch.as_tensor(finished, device="cuda")].any()
    return int(finished.sum())


@pytest.mark.gpu
@pytest.mark.parametrize("cls_name,variant", CLASSES)
@pytest.mark.parametrize("B", [1, 7, 4096])
def test_legal_ids_and_masks_mid_game(D, oracle, uni, cls_name, variant, B):
    finished = 0
    for steps in (0, 9, 40, 90):
        env, ref = _mirrored_rollout(D, oracle, cls_name, variant, B, steps, seed=100 + B + variant)
        finished += check_env_ids(D, env, ref, uni)
        assert int(env.stats[7].item()) == 0
    if B == 4096:
        assert finished > 0


@pytest.mark.gpu
def test_legal_ids_and_masks_at_131072_envs(D, oracle, uni):
    env, ref = _mirrored_rollout(D, oracle, "BatchedEnvCooperation", 2, 131072, 12, seed=77)
    check_env_ids(D, env, ref, uni)


@pytest.mark.gpu
def test_masks_of_cut_and_dropped_lists(D, oracle, uni):
    B = 300
    env, ref = _mirrored_rollout(D, oracle, "BatchedEnvComplicated", 1, B, 30, seed=9)
    off_np, au, _, _ = ref.observe(want_f32=False, want_face=False)
    off_np = off_np.astype(np.int64)
    total = int(off_np[-1])
    off = torch.as_tensor(off_np.astype(np.int32), device="cuda")
    actions = torch.as_tensor(np.concatenate([au, np.full(64, 0xA5A5A5A5A5A5A5A5, np.uint64)]).view(np.int64), device="cuda")
    ids = ref_ids(uni, au)
    full = np.diff(off_np)
    for cap in sorted({0, 1, 2, 5, total // 3, total // 2 + 1, total - 1, total, total + 64}):
        stored = np.clip(np.minimum(full, cap - off_np[:-1]), 0, None)
        keep = np.concatenate([np.arange(off_np[b], off_np[b] + stored[b]) for b in range(B)]).astype(np.int64)
        st_off = np.concatenate([[0], np.cumsum(stored)])
        want_b, want_w = expected_masks(st_off, ids[keep], B)
        for layout, want in ((D.native.MASK_BYTES, want_b), (D.native.MASK_BITS, want_w)):
            stats = torch.zeros(16, dtype=torch.int64, device="cuda")
            got = run_mask(D, off, actions if cap else None, cap, layout, B, stats=stats, shift=7 if layout else 0)
            assert torch.equal(got, want), (cap, layout)
            assert int(stats[7].item()) == int((stored < full).sum()), (cap, layout)


@pytest.mark.gpu
def test_ids_of_config5_lists(D, uni):
    hands, lasts = D.adversarial_pairs(16384)
    moves, off = D.get_moves(D.unpack_counts(torch.as_tensor(hands.view(np.int64))).numpy(),
                             D.unpack_counts(torch.as_tensor(lasts.view(np.int64))).numpy())
    got = D.move_ids(moves).cpu().numpy()
    assert len(got) > 100000
    assert np.array_equal(got, ref_ids(uni, _u64(moves)))
    o = off.cpu().numpy()
    inner = np.ones(len(got), bool)
    inner[o[:-1][o[:-1] < len(got)]] = False
    assert (np.diff(got.astype(np.int64))[inner[1:]] > 0).all()


def _state(env):
    return env._state.clone()


@pytest.mark.gpu
@pytest.mark.parametrize("cls_name,variant", CLASSES)
def test_step_ids_equals_step_index(D, cls_name, variant):
    B, K = 4096, 60
    perm, lord = D.random_deals(B, seed=31)
    a, b = (getattr(D, cls_name)(B, seed=3) for _ in range(2))
    a.prepare(perm, lord)
    b.prepare(perm, lord)
    rng = np.random.default_rng(variant)
    for _ in range(K):
        off = a.offsets.cpu().numpy()
        cnt = np.diff(off)
        choice = (rng.integers(0, 1 << 30, B) % np.maximum(cnt, 1)).astype(np.int32)
        ids = b.legal_ids().cpu().numpy()
        pick = np.where(cnt > 0, ids[np.minimum(off[:-1] + choice, len(ids) - 1)], 0)
        ra = [t.clone() for t in a.step(choice)]
        rb = [t.clone() for t in b.step_ids(pick)]
        assert all(torch.equal(x, y) for x, y in zip(ra, rb)) and torch.equal(a.reward, b.reward)
        assert torch.equal(_state(a), _state(b))
        a.prepare(perm, lord, only_done=True)
        b.prepare(perm, lord, only_done=True)
    assert torch.equal(a.stats, b.stats) and int(a.stats[7].item()) == 0 and int(a.stats[4].item()) > 0


@pytest.mark.gpu
def test_illegal_and_out_of_range_ids(D, oracle, uni):
    B = 64
    env = D.BatchedEnvCooperation(B, seed=4)
    perm, lord = D.random_deals(B, seed=8)
    env.prepare(perm, lord)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord)
    ref.observe(want_f32=False, want_face=False)
    off = env.offsets.cpu().numpy()
    ids = env.legal_ids().cpu().numpy()
    legal = [set(ids[off[k]:off[k + 1]].tolist()) for k in range(B)]
    choice = ids[off[:-1]].copy()                                              # legal: the first move of each list
    rng = np.random.default_rng(2)
    kinds = rng.integers(0, 4, B)
    for k in range(B):
        if kinds[k] == 1:
            choice[k] = next(i for i in range(NIDS) if i not in legal[k])          # a move, but not legal here
        elif kinds[k] == 2:
            choice[k] = -1 - int(rng.integers(0, 1000))
        elif kinds[k] == 3:
            choice[k] = NIDS + int(rng.integers(0, 1000))
    before = _state(env)
    r, done, cat = env.step_ids(choice)
    # the oracle's model of a DDZ_CHOICE_MOVE step: the move's position in the env's list, -1 (illegal) when it is not there
    moves = np.where((choice >= 0) & (choice < NIDS), uni[0][np.clip(choice, 0, NIDS - 1)], INVALID)
    roff = ref.offsets
    pos = np.full(B, -1, np.int32)
    for k in range(B):
        hit = np.nonzero(ref.actions_u64[roff[k]:roff[k + 1]] == moves[k])[0]
        if len(hit):
            pos[k] = hit[0]
    assert np.array_equal(pos >= 0, kinds == 0)
    rr, rd, rc, _ = ref.step(choice=pos, mode=0)
    assert np.array_equal(r.cpu().numpy(), rr) and np.array_equal(done.cpu().numpy(), rd) and np.array_equal(cat.cpu().numpy(), rc)
    f, meta = ref.export()
    fields, m = env._fields()
    assert np.array_equal(fields.cpu().numpy().view(np.uint64), f) and np.array_equal(m.cpu().numpy().view(np.uint32), meta)
    bad = kinds != 0
    assert int(env.stats[7].item()) == int(bad.sum()) == int(ref.stats[7])
    assert ((m.cpu().numpy()[bad] >> 5) & 1 == 1).all()
    after = _state(env)
    fb, fa = before[:18 * B].view(torch.int64).view(9, B), after[:18 * B].view(torch.int64).view(9, B)
    assert torch.equal(fb[:, torch.as_tensor(bad, device="cuda")], fa[:, torch.as_tensor(bad, device="cuda")])
    dbg = D.BatchedEnvCooperation(4, seed=4, debug=True)
    dbg.prepare(*D.random_deals(4, seed=8))
    with pytest.raises(D.native.DdzError):
        dbg.step_ids([NIDS, 0, 0, 0])


@pytest.mark.gpu
def test_fixed_head_policy_end_to_end(D):
    """logits [B, 13551] masked by legal_mask and argmaxed, played by id, against the same logits gathered at legal_ids,
    picked by ddz_select_actions and played by list index: identical trajectories, only legal moves"""
    B, T = 4096, 300
    a, b = D.BatchedEnvCooperation(B, seed=1), D.BatchedEnvCooperation(B, seed=1)
    a.prepare()
    b.prepare()
    gen = torch.Generator(device="cuda").manual_seed(0)
    choice = torch.empty(B, dtype=torch.int32, device="cuda")
    finished = 0
    for t in range(T):
        logits = torch.randn((B, NIDS), device="cuda", generator=gen)
        mask = a.legal_mask("bool")
        ids = logits.masked_fill(~mask, float("-inf")).argmax(1).to(torch.int32)
        off = b.offsets.to(torch.int64)
        owner = torch.repeat_interleave(torch.arange(B, device="cuda"), off[1:] - off[:-1], output_size=b.num_actions)
        q = logits[owner, b.legal_ids().to(torch.int64)].contiguous()
        D.native.check(D.native.lib.ddz_select_actions(q.data_ptr(), b.offsets.data_ptr(), 0.0, 0, 0, 0, choice.data_ptr(),
                                                       B, _stream()), "ddz_select_actions")
        ra = [x.clone() for x in a.step_ids(ids)]
        rb = [x.clone() for x in b.step(choice)]
        assert all(torch.equal(x, y) for x, y in zip(ra, rb))
        assert torch.equal(_state(a), _state(b))
        finished += int(ra[1].sum().item())
        a.prepare(only_done=True)
        b.prepare(only_done=True)
    assert int(a.stats[7].item()) == 0 and torch.equal(a.stats, b.stats) and finished > B


@pytest.mark.gpu
def test_form_b_build_ids():
    lib_b = os.path.join(ROOT, "doudizhu-rl_b200", "libddz_b200_formB.so")
    if not os.path.exists(lib_b):
        import __graft_entry__
        __graft_entry__.build()
    out = subprocess.run([sys.executable, os.path.join(HERE, "form_b_ids_check.py")],
                         env=dict(os.environ, DDZ_LIB=lib_b), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "form B ids ok" in out.stdout
