"""ddz_q_features (csrc/ddz_kernels.cu, k_q_features) row by row against the network's own first layer in float64.

The kernel computes the four rank convolutions + max-pool and the line convolution of net.py:91-97 from the packed state
and move lists through the tables of agent.q_tables.  The reference here is the module itself: QNetLike(...).double()'s
rank_convs (max over k) and line_conv applied to env.state_actions() in float64 -- that input is pinned bit-exact to the
oracle elsewhere (test_gpu_parity.py, form_b_check.py) -- permuted to the kernel's rank-major row [15][W] | [W][4].

Error bound (float32 round-to-nearest, unit roundoff 2^-24): a feature is a sum of n terms, each a table entry rounded to
float32 once (and, for a probability plane, multiplied by its scale: one more rounding), added up in float32, so

    |got - ref| <= (n + 2) * 2^-24 * A,     n = C + 2 (rank feature), 15 (C + 1) + 1 (line feature)

with A the same convolutions on |x| with |weights| and |bias|; a rank feature takes max_k A_k (max-pool is 1-Lipschitz).
A missing or misplaced term is ~1e-2 with Conv2d's default init, 1e3-1e4 times the bound.

tests/form_b_q_features_check.py runs the row checks (fp32, bf16, edge positions) against the -DDDZ_PROB_FORM_B build."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from qnet_like import QNetLike

CLASSES = [("BatchedEnv", 4), ("BatchedEnvComplicated", 7), ("BatchedEnvCooperation", 9), ("BatchedEnvCooperationSimplify", 6)]
WIDTHS = [4, 36, 100, 252, 256]          # below one warp, not a multiple of 32, and both instantiations (W = 256 is compiled in)
U32 = 2.0 ** -24
CHUNK = 8192                             # rows per float64 reference batch
SENTINEL32, SENTINEL16 = 0x7FBADBAD, 0x7FDB      # NaN bit patterns no kernel writes


@pytest.fixture(scope="module")
def D():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


@pytest.fixture(scope="module")
def envs(D):
    """envs("BatchedEnv", "mid" | "finished" | "edge"), built once per module"""
    make = {"mid": midgame_env, "finished": finished_mix_env, "edge": edge_env}
    cache = {}

    def get(cls, kind):
        if (cls, kind) not in cache:
            cache[cls, kind] = make[kind](D, cls)
        return cache[cls, kind]
    return get


# ------------------------------------------------------------------------------------------------ inputs
def midgame_env(D, cls, B=2000, steps=23, seed=3):
    perm, lord = D.random_deals(B, seed=seed, pool_games=2)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = getattr(D, cls)(B, seed=seed)
    env.prepare(pd, ld, pool_games=2)
    for _ in range(steps):
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=2)
    env.num_actions
    return env


def finished_mix_env(D, cls, B=600, steps=40, seed=4):
    """no re-deal: games end one by one, so some envs are finished and have no legal moves"""
    perm, lord = D.random_deals(B, seed=seed)
    env = getattr(D, cls)(B, seed=seed)
    env.prepare(torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda())
    for _ in range(steps):
        env.rollout_step()
    env.observe()
    assert 0 < int(env.is_done.sum()) < env.B
    assert int((env.offsets[1:] - env.offsets[:-1]).min()) == 0
    env.num_actions
    return env


def _counts(cards):
    c = np.zeros(15, np.int64)
    for v in cards:                      # card values 3..17 (16 = small joker, 17 = big joker)
        c[v - 3] += 1
    return c


# (role to move, its hand, history per role, last hand-out per role ([] = pass / none), cards left per role);
# role 0 = up, 1 = lord, 2 = down; the previous player of role s is (s + 2) % 3
EDGE_POSITIONS = [
    (1, [3, 4, 5, 6, 7, 7, 8, 9, 10, 11, 12, 13, 14, 15], {2: [17]}, {}, [17, 14, 16]),   # a history of the big joker only
    (1, [3, 4, 5, 6, 7, 7, 8, 9, 10, 11, 12, 13, 14, 15], {0: [16]}, {}, [16, 14, 17]),   # ... of the small joker only
    (1, [5, 5, 5, 5, 8, 9], {0: [17]}, {0: [17]}, [16, 6, 17]),      # following the big joker: pass or a bomb
    (1, [17], {0: [3, 3, 4], 2: [5]}, {}, [14, 1, 16]),               # the mover holds the big joker only
    (1, [3, 4, 5, 6, 9, 9, 16, 17], {}, {}, [17, 8, 17]),             # the rocket in hand, untouched history
    (0, [6, 6, 6, 6, 8, 8, 11, 14], {1: [3, 4]}, {}, [8, 18, 17]),    # a four-of-a-kind
    (2, [4, 8, 8, 12, 15], {0: [3], 1: [7]}, {1: [7]}, [16, 19, 5]),  # following a single: the pass move is in the list
    (1, [3, 5, 9], {0: [10, 10, 11]}, {}, [5, 3, 0]),                 # probability scales 0 (next player) and 1
    (1, [3, 5, 9], {2: [10, 10, 11]}, {}, [0, 3, 7]),                 # ... and 1 and 0
    (1, [3, 3, 3, 4, 4, 4, 5, 5, 5, 6, 6, 6, 7, 7, 7, 8, 8, 8, 9, 9], {}, {}, [17, 20, 17]),   # 260 moves: more than a CTA
]


def edge_env(D, cls):
    """the positions above via ingest.env_from_arrays; asserts that each special case is really in the input"""
    B = len(EDGE_POSITIONS)
    role = np.array([p[0] for p in EDGE_POSITIONS])
    hand = np.stack([_counts(p[1]) for p in EDGE_POSITIONS])
    hist = np.stack([[_counts(p[2].get(q, [])) for q in range(3)] for p in EDGE_POSITIONS])
    last = np.stack([[_counts(p[3].get(q, [])) for q in range(3)] for p in EDGE_POSITIONS])
    left = np.array([p[4] for p in EDGE_POSITIONS])
    assert ((hand + hist.sum(1)) <= np.array([4] * 13 + [1, 1])).all()
    env = D.env_from_arrays(role, hand, hist, last, left, env_cls=getattr(D, cls))
    C = env.C
    counts = (env.offsets[1:] - env.offsets[:-1]).cpu()
    x = env.state_actions()[0]
    nz = (x[:, :C - 2] != 0).any(-1)                  # [n, count planes, 15]: the rank is non-empty
    assert bool((nz[..., 14] & ~nz[..., :14].any(-1)).any()), "no plane holding the big joker only"
    assert bool((nz[..., 13] & ~nz[..., :13].any(-1) & ~nz[..., 14]).any()), "no plane holding the small joker only"
    assert bool((~nz.any(-1)).any()), "no empty plane"
    mv = x[:, C]
    assert bool((mv == 0).all(-1).all(-1).any()), "no pass move"
    assert bool((mv[:, :13, 3] == 1).any()), "no bomb (nibble 4)"
    assert bool(((mv[:, 13, 0] == 1) & (mv[:, 14, 0] == 1)).any()), "no rocket"
    assert int(counts.max()) > 256, "no list longer than a CTA"
    p = x[:, C - 2:C].amax((2, 3))                      # the two probability planes' scales (their rows are not empty here)
    assert bool(((p[:, 0] == 0) & (p[:, 1] == 1)).any()) and bool(((p[:, 0] == 1) & (p[:, 1] == 0)).any()), "no scale 0 / 1"
    return env


# ------------------------------------------------------------------------------------------------ kernel and reference
def tables_of(net):
    """the kernel's float32 tables, built by the library's own agent.q_tables from the network's weights"""
    import ddz_b200.agent as agent
    convs, line, _, _ = agent.net_parts(net)
    return agent.q_tables(convs, line)


def q_features(D, env, tables, W, out, bf16, mask=None, dst=None, env_begin=0, env_count=None, row_base=0):
    T, rb, L, lb = tables
    off = env._offsets[env._cur]
    D.native.check(D.native.lib.ddz_q_features(env._state.data_ptr(), env.VARIANT, off.data_ptr(),
                                               env._actions_u64[env._cur].data_ptr(), None if mask is None else mask.data_ptr(),
                                               None if dst is None else dst.data_ptr(), env_begin,
                                               env.B - env_begin if env_count is None else env_count, row_base,
                                               T.data_ptr(), rb.data_ptr(), L.data_ptr(), lb.data_ptr(), W, out.data_ptr(),
                                               int(bf16), env.B, env._stream()), "ddz_q_features")


def kernel_rows(D, env, tables, W, dtype):
    """one call over every env, rows in the order of the CSR move list"""
    out = torch.empty((env.num_actions, 19 * W), dtype=dtype, device=env.device)
    if out.shape[0]:
        q_features(D, env, tables, W, out, dtype == torch.bfloat16)
    return out


def first_layer64(net, x):
    """[n, 19 W] in the kernel's layout: max_k rank_convs[k](x) rank-major (r * W + o), then line_conv(x) (o * 4 + j)"""
    r = torch.cat([c(x) for c in net.rank_convs], -1).max(-1).values          # [n, W, 15]
    return torch.cat([r.transpose(1, 2).flatten(1), net.line_conv(x).flatten(1)], 1)


def abs_net(net):
    a = copy.deepcopy(net)
    with torch.no_grad():
        for p in a.parameters():
            p.abs_()
    return a


def net64(C, W, seed, device, hidden=8):
    return QNetLike(C, W, hidden, seed=seed).double().to(device)


def check_rows(D, env, C, W, seed):
    """every fp32 row against float64 within the derived bound; returns (rows, x, largest err / bound)"""
    net = net64(C, W, seed, env.device)
    got = kernel_rows(D, env, tables_of(net), W, torch.float32)
    x = env.state_actions()[0]
    assert got.shape[0] == x.shape[0] == env.num_actions
    assert bool(torch.isfinite(got).all())
    terms = torch.cat([torch.full((15 * W,), C + 2.0), torch.full((4 * W,), 15.0 * (C + 1) + 1)]).to(env.device, torch.float64)
    absn = abs_net(net)
    worst = 0.0
    with torch.no_grad():
        for lo in range(0, x.shape[0], CHUNK):
            xs = x[lo:lo + CHUNK].double()
            err = (got[lo:lo + CHUNK].double() - first_layer64(net, xs)).abs()
            bound = (terms + 2) * U32 * first_layer64(absn, xs.abs())
            worst = max(worst, float((err / bound).max()))
    assert worst <= 1.0, "W=%d: largest |got - ref| / bound = %.3g" % (W, worst)
    return got, x, worst


def check_bf16_rows(D, env, C, W, seed, rows32):
    """bfloat16 rows == the float32 rows rounded to nearest-even, bit for bit (same arithmetic, only the store differs)"""
    net = net64(C, W, seed, env.device)
    got = kernel_rows(D, env, tables_of(net), W, torch.bfloat16)
    want = rows32.to(torch.bfloat16)
    diff = int((got.view(torch.int16) != want.view(torch.int16)).sum())
    assert diff == 0, "W=%d: %d of %d bfloat16 elements differ from round-to-nearest-even of the float32 rows" % (W, diff, got.numel())


def check_env(D, env, C, W, seed):
    rows32, x, worst = check_rows(D, env, C, W, seed)
    check_bf16_rows(D, env, C, W, seed, rows32)
    return x, worst


# ------------------------------------------------------------------------------------------------ GPU tests
@pytest.mark.gpu
@pytest.mark.parametrize("W", WIDTHS)
@pytest.mark.parametrize("cls,C", CLASSES)
def test_fp32_rows_within_float64_bound(D, envs, cls, C, W):
    """every element of every row of mid-game envs and of a batch with finished envs, within the bound of the docstring"""
    worst = 0.0
    for env in (envs(cls, "mid"), envs(cls, "finished")):
        _, x, w = check_rows(D, env, C, W, seed=W + C)
        worst = max(worst, w)
        prob = x[:, C - 2:C]
        # the scale multiply is exercised: probability slots strictly between 0 and 1 occur, and so do empty ones
        assert bool(((prob > 0) & (prob < 1)).any()) and bool((prob == 0).any())
    print("fp32 rows %s W=%d: largest err/bound %.3g" % (cls, W, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("W", WIDTHS)
@pytest.mark.parametrize("cls,C", CLASSES)
def test_bf16_rows_are_fp32_rows_rounded(D, envs, cls, C, W):
    for env in (envs(cls, "mid"), envs(cls, "finished")):
        net = net64(C, W, W + C, env.device)
        check_bf16_rows(D, env, C, W, W + C, kernel_rows(D, env, tables_of(net), W, torch.float32))


@pytest.mark.gpu
@pytest.mark.parametrize("W", WIDTHS)
@pytest.mark.parametrize("cls,C", CLASSES)
def test_edge_positions(D, envs, cls, C, W):
    """jokers alone in a plane, the rocket, bombs, the pass move, empty planes, scales 0 and 1, 260 moves in one env"""
    env = envs(cls, "edge")
    _, worst = check_env(D, env, C, W, seed=3 * W + C)
    print("edge rows %s W=%d: largest err/bound %.3g" % (cls, W, worst))


def _sentinel(rows, W, dtype, device):
    buf = torch.empty((rows, 19 * W), dtype=dtype, device=device)
    if dtype == torch.bfloat16:
        buf.view(torch.int16).fill_(SENTINEL16)
    else:
        buf.view(torch.int32).fill_(SENTINEL32)
    return buf


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("W", WIDTHS)
@pytest.mark.parametrize("cls,C", CLASSES)
def test_rows_land_where_the_offsets_say(D, envs, cls, C, W):
    """Each env writes exactly its own rows: into a NaN-filled buffer with guard rows, unmasked and masked, at the CSR
    offsets, at compacted offsets and at offsets with a gap after every env; finished and masked-out envs write nothing;
    three uneven (env_begin, env_count, row_base) chunks give the same bits as one call, in float32 and bfloat16."""
    env = envs(cls, "finished")
    dev, B, G = env.device, env.B, 3
    off = env.offsets.to(torch.int64)
    cnt = off[1:] - off[:-1]
    off_h = off.tolist()
    assert int((cnt == 0).sum()) > 0                                        # finished envs
    mask = torch.rand(B, generator=torch.Generator().manual_seed(W), device="cpu").to(dev) < 0.6
    mask8 = mask.to(torch.uint8)
    compact = torch.zeros(B + 1, dtype=torch.int64, device=dev)
    compact[1:] = torch.cumsum(cnt * mask, 0)
    gapped = off + torch.arange(B + 1, device=dev)                          # one unowned row after every env's block
    net = net64(C, W, 5, dev)
    tables = tables_of(net)
    bounds = [0, B // 7, B // 7 + B // 2, B]                                # uneven chunks
    for dtype in (torch.float32, torch.bfloat16):
        plain = kernel_rows(D, env, tables, W, dtype)
        for masked, dst in ((False, None), (False, gapped), (True, None), (True, compact), (True, gapped)):
            start = (off if dst is None else dst).tolist()
            live = ((cnt > 0) & mask if masked else cnt > 0).tolist()
            nrows = start[B]
            want = _sentinel(nrows + 2 * G, W, dtype, dev)
            for b in range(B):
                if live[b]:
                    want[G + start[b]:G + start[b] + off_h[b + 1] - off_h[b]] = plain[off_h[b]:off_h[b + 1]]
            dst32 = None if dst is None else dst.to(torch.int32)
            m8 = mask8 if masked else None
            got = _sentinel(nrows + 2 * G, W, dtype, dev)
            q_features(D, env, tables, W, got[G:], dtype == torch.bfloat16, mask=m8, dst=dst32)
            what = "%s masked=%s offsets=%s" % (dtype, masked, "csr" if dst is None else "compact" if dst is compact else "gapped")
            assert torch.equal(_bits(got), _bits(want)), what
            for b_lo, b_hi in zip(bounds[:-1], bounds[1:]):
                lo, hi = start[b_lo], start[b_hi]
                part = _sentinel(hi - lo + 2 * G, W, dtype, dev)
                q_features(D, env, tables, W, part[G:], dtype == torch.bfloat16, mask=m8, dst=dst32, env_begin=b_lo,
                           env_count=b_hi - b_lo, row_base=lo)
                assert torch.equal(_bits(part[G:G + hi - lo]), _bits(want[G + lo:G + hi])), (what, b_lo, b_hi)
                assert torch.equal(_bits(part[:G]), _bits(want[:G])) and torch.equal(_bits(part[-G:]), _bits(want[:G])), \
                    (what, b_lo, b_hi)


@pytest.mark.gpu
def test_form_b_build_rows():
    """the row checks above (fp32, bf16, edge positions) against the -DDDZ_PROB_FORM_B build, in a subprocess"""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_b = os.path.join(root, "doudizhu-rl_b200", "libddz_b200_formB.so")
    if not os.path.exists(lib_b):
        import __graft_entry__
        __graft_entry__.build()
    out = subprocess.run([sys.executable, os.path.join(root, "tests", "form_b_q_features_check.py")],
                         env=dict(os.environ, DDZ_LIB=lib_b), capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "form B q features ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    print(out.stdout.strip())


def q_bound64(net, x, u):
    """float64 Q of net on x [m, C+1, 15, 4] and, per move, the bound on |q - q64| of a fc1 whose operands are rounded to
    a relative u (features, fc1's weights and bias) and whose output is rounded to u; fc2 in float32:
        2 sum_k |w2_k| (u |h_k| + 2u (sum_i |f_i| |w1_ki| + |b1_k|)) + (H + 2) 2^-24 (sum_k |w2_k h_k| + |b2|)
    (the factor 2 in front covers the float32 accumulation inside fc1 and the float32 rows' own error)"""
    w1, b1 = net.fc1.weight, net.fc1.bias
    w2, b2 = net.fc2.weight[0], net.fc2.bias[0]
    r = torch.cat([c(x) for c in net.rank_convs], -1).max(-1).values.flatten(1)
    f = torch.cat([r, net.line_conv(x).flatten(1)], 1)                        # net.py:93-97's layout
    h = torch.relu(f @ w1.t() + b1)
    q = h @ w2 + b2
    S = f.abs() @ w1.abs().t() + b1.abs()
    bound = 2 * ((u * h + 2 * u * S) * w2.abs()).sum(1) + (w2.numel() + 2) * U32 * ((h * w2).abs().sum(1) + b2.abs())
    return q, bound


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("W,H", [(32, 64), (256, 256)])
@pytest.mark.parametrize("cls,C", CLASSES)
def test_reduced_precision_q_within_derived_bound(D, envs, cls, C, W, H, precision):
    """FusedQScorer in tf32 / bf16, every scored move against the float64 network, unmasked and masked, each cut into
    about five chunks.  u = 2^-8 (bf16: rows, fc1's weights and hidden layer stored in bfloat16) or 2^-10 (TF32 keeps 10
    mantissa bits; whether the GEMM rounds or truncates its float32 operands, their relative error stays below 2^-10)."""
    env = envs(cls, "mid")
    u = 2.0 ** -8 if precision == "bf16" else 2.0 ** -10
    net = QNetLike(C, W, H, seed=17 + W).eval().to(env.device)
    n64 = copy.deepcopy(net).double()
    total = env.num_actions
    worst = 0.0
    for mask in (None, env.get_role_ID() == 2):                            # every move; the landlord's decisions only
        x, rows = env.state_actions(mask)
        q = D.FusedQScorer(net, C, precision=precision, chunk_rows=x.shape[0] // 5).q_values(env, mask)
        assert q.shape == (total,)
        if rows is not None:
            assert 0 < rows.numel() < total
            rest = torch.ones(total, dtype=torch.bool, device=env.device)
            rest[rows] = False
            assert not bool(q[rest].any())                                 # moves outside the mask stay 0
            q = q[rows]
        with torch.no_grad():
            for lo in range(0, x.shape[0], CHUNK):
                want, bound = q_bound64(n64, x[lo:lo + CHUNK].double(), u)
                err = (q[lo:lo + CHUNK].double() - want).abs()
                worst = max(worst, float((err / bound).max()))
    assert worst <= 1.0, "largest |q - q64| / bound = %.3g" % worst
    print("Q %s %s W=%d: largest err/bound %.3g" % (precision, cls, W, worst))


# ------------------------------------------------------------------------------------------------ CPU
def test_reference_features_cover_form_b_rows():
    """qscore_reference.features on form-B-shaped inputs (right-aligned rows in ranks 0..12 of the two probability planes,
    the jokers' single left slot) == the network's float64 convolutions"""
    from qscore_reference import features, nibbles_of
    import ddz_b200.agent as agent
    rng = np.random.default_rng(8)
    for C in (4, 7, 9, 6):
        n = 64
        net = QNetLike(C, 36, 8, seed=C).double()
        counts = rng.integers(0, 5, (n, C + 1, 15))
        counts[:, :, 13:] = rng.integers(0, 2, (n, C + 1, 2))
        x = (counts[..., None] > np.arange(4)).astype(np.float64)
        x[:, C - 2:C, :13] = x[:, C - 2:C, :13, ::-1].copy()                     # right-aligned
        scale = rng.random((n, 2))
        scale[:4] = [[0.0, 1.0], [1.0, 0.0], [0.25, 0.75], [1.0, 1.0]]
        x[:, C - 2:C] *= scale[:, :, None, None]
        nib, sc = nibbles_of(x)
        live = counts[:, C - 2:C, :13] * (scale[:, :, None] > 0)
        assert ((nib[:, C - 2:C, :13] >= 9) == ((live > 0) & (live < 4))).all()
        convs, line, _, _ = agent.net_parts(net)
        T, rb, L, lb = agent.q_tables(convs, line, dtype=torch.float64)
        got = features(nib, sc, T.numpy(), rb.numpy(), L.numpy(), lb.numpy())
        with torch.no_grad():
            xt = torch.from_numpy(x.copy())
            r = torch.cat([c(xt) for c in net.rank_convs], -1).max(-1).values.flatten(1)
            want = torch.cat([r, net.line_conv(xt).flatten(1)], 1).numpy()
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12, err_msg="C=%d" % C)
