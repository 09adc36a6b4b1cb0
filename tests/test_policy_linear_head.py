"""Linear policy heads evaluated only at the legal ids (include/ddz_b200.h: ddz_policy_linear_logits, _sample, _logprob,
_backward, _grad_weight; D.LinearPolicyHead, D.HeadedPolicy).

CPU: argument checks before any CUDA call, the workspace size, and the register counts of the new kernels (no stack, no
spills).
GPU (-m gpu): the legal logits against float64 W[id] . h + b within the float32 bound; sampling, log-probability, entropy
and the per-entry gradient bit for bit against the dense kernels run on a row that holds the kernel's own legal logits;
the hidden, weight and bias gradients against float64 sums (including a batch whose pass id has more than 60 000
entries) and a repeated call bit for bit; LinearPolicyHead.log_prob's autograd against float64 autograd of the dense
masked log_softmax; the peak memory of a training step at 131 072 envs; a landlord trained by REINFORCE through the head;
BatchedGame and compete with a HeadedPolicy seat."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NIDS = 13551
SENT = 0x5C
U32 = 2.0 ** -24                    # unit roundoff of float32
U16 = 2.0 ** -8                     # of bfloat16 (the rounding of a bfloat16 output)


def gamma(k, u=U32):
    """gamma_k = k u / (1 - k u), the bound of a k-term float sum (Higham)"""
    return k * u / (1 - k * u)


# ------------------------------------------------------------------ CPU
def test_argument_checks_before_any_cuda_call():
    import ddz_b200 as D
    L, E, N = D.native.lib, D.native.E_ARG, D.native
    F32, BF = N.DTYPE_F32, N.DTYPE_BF16
    ok = dict(state=None, off=16, act=16, cap=64, h=256, W=512, b=1024, dtype=F32, H=64, ld=64, T=1.0, out=16, B=4)

    def head(a):
        return (a["h"], a["W"], a["b"], a["dtype"], a["H"], a["ld"])

    bad_head = (dict(h=None), dict(W=None), dict(dtype=2), dict(dtype=-1), dict(H=0), dict(H=-4), dict(H=1028),
                dict(H=1032, ld=1032), dict(H=6, ld=8), dict(ld=60), dict(ld=66), dict(H=8, ld=12, dtype=BF),
                dict(H=12, ld=16, dtype=BF), dict(h=264), dict(W=520), dict(b=1026), dict(h=258, dtype=BF),
                dict(b=1025, dtype=BF), dict(B=0), dict(B=-3), dict(off=None), dict(cap=-1), dict(act=None))

    def logits(**kw):
        a = dict(ok, **kw)
        return L.ddz_policy_linear_logits(a["off"], a["act"], a["cap"], *head(a), a["out"], None, a["B"], None)
    for bad in bad_head + (dict(out=None),):
        assert logits(**bad) == E, bad

    def sample(**kw):
        a = dict(ok, **kw)
        return L.ddz_policy_linear_sample(a["state"], a["off"], a["act"], a["cap"], *head(a), a["T"], 0, 0, 0, None,
                                          a.get("choice", 16), a.get("ids", 16), a.get("logp", 16), a.get("ent", 16), None,
                                          a["B"], None)
    for bad in bad_head + (dict(choice=None), dict(ids=None), dict(logp=None), dict(ent=None), dict(T=-0.5),
                           dict(T=float("nan")), dict(T=float("inf"))):
        assert sample(**bad) == E, bad

    def logprob(**kw):
        a = dict(ok, **kw)
        return L.ddz_policy_linear_logprob(a["off"], a["act"], a["cap"], *head(a), a.get("ids", 16), a.get("logp", 16),
                                           a.get("ent", 16), None, None, a["B"], None)
    for bad in bad_head + (dict(ids=None), dict(logp=None), dict(ent=None)):
        assert logprob(**bad) == E, bad

    def backward(**kw):
        a = dict(ok, **kw)
        return L.ddz_policy_linear_backward(a["off"], a["act"], a["cap"], *head(a), a.get("ids", 16), a.get("lse", 16), None,
                                            None, a.get("gl", 16), a.get("gh", 2048), a.get("ldg", 64), a["B"], None)
    for bad in bad_head + (dict(ids=None), dict(lse=None), dict(gl=None), dict(gh=None), dict(gh=2056), dict(ldg=60),
                           dict(ldg=66), dict(ldg=12, dtype=BF, H=8, ld=8)):
        assert backward(**bad) == E, bad

    def grad_weight(**kw):
        a = dict(dict(ok, n=100, gl=16, order=16, ido=16, gw=4096, gb=8192, ws=16384), **kw)
        return L.ddz_policy_linear_grad_weight(a["off"], a["n"], a["h"], a["dtype"], a["H"], a["ld"], a["gl"], a["order"],
                                               a["ido"], a["gw"], a["gb"], a["ws"], a["B"], None)
    for bad in (dict(off=None), dict(n=-1), dict(h=None), dict(gw=None), dict(gl=None), dict(order=None), dict(ido=None),
                dict(ws=None), dict(B=0), dict(dtype=3), dict(H=0), dict(H=1028), dict(H=6, ld=8), dict(ld=60), dict(h=264),
                dict(gw=4100), dict(gb=8194), dict(ws=16388), dict(H=12, ld=16, dtype=BF)):
        assert grad_weight(**bad) == E, bad

    # the workspace: two slots of H + 4 floats per 128 entries of the sorted order
    W = L.ddz_policy_linear_workspace_bytes
    assert W(0, 64) == 0 and W(-5, 64) == 0 and W(10, 0) == 0 and W(10, 1028) == 0
    assert W(1, 64) == 2 * 68 * 4 and W(128, 64) == 2 * 68 * 4 and W(129, 64) == 4 * 68 * 4
    assert W(580000, 256) == 2 * ((580000 + 127) // 128) * 260 * 4
    hdr = open(os.path.join(ROOT, "include", "ddz_b200.h")).read()
    assert re.search(r"#define DDZ_ABI_VERSION 3\b", hdr) and N.LINEAR_MAX_HIDDEN == 1024


def test_head_module_layout():
    """nn.Linear's parameters and layout, both ways; the fused paths reject widths they do not take"""
    torch = pytest.importorskip("torch")
    import ddz_b200 as D
    lin = torch.nn.Linear(24, NIDS)
    head = D.LinearPolicyHead(24)
    head.load_state_dict(lin.state_dict())
    assert torch.equal(head.weight, lin.weight) and torch.equal(head.bias, lin.bias)
    h = torch.randn(3, 24)
    assert torch.equal(head(h), lin(h))
    head2 = D.LinearPolicyHead.from_linear(lin)
    assert torch.equal(head2.weight, lin.weight) and head2.weight.data_ptr() != lin.weight.data_ptr()
    lin.load_state_dict(head2.state_dict())
    nb = D.LinearPolicyHead(8, bias=False, dtype=torch.bfloat16)
    assert nb.bias is None and nb.weight.dtype == torch.bfloat16 and tuple(nb.weight.shape) == (NIDS, 8)
    with pytest.raises(ValueError):
        D.LinearPolicyHead.from_linear(torch.nn.Linear(8, 100))
    with pytest.raises(ValueError):
        D.LinearPolicyHead(6).log_prob(torch.zeros(1, 6), torch.zeros(2, dtype=torch.int32), torch.zeros(0), [0])
    with pytest.raises(ValueError):
        D.LinearPolicyHead(12, dtype=torch.bfloat16).log_prob(torch.zeros(1, 12), torch.zeros(2, dtype=torch.int32),
                                                              torch.zeros(0), [0])
    with pytest.raises(TypeError):
        D.HeadedPolicy(torch.nn.Flatten(), torch.nn.Linear(8, NIDS))
    pol = D.HeadedPolicy(torch.nn.Flatten(), D.LinearPolicyHead(60))
    assert tuple(pol(torch.zeros(2, 1, 15, 4)).shape) == (2, NIDS)


# one entry per instantiation (float32, bfloat16), sorted
REGS_LINEAR = {"k_linear_logits": [32, 40], "k_linear_sample": [40, 48], "k_linear_logprob": [38, 40],
               "k_linear_backward": [40, 40], "k_linear_grad_chunks": [58, 63], "k_linear_grad_combine": [64, 80]}


def test_register_counts():
    import ddz_b200 as D
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([tool, "-res-usage", D.native.LIB_PATH], capture_output=True, text=True).stdout
    regs, stack = {}, {}
    pat = r"Function _ZN3ddz11linear_head\d+(k_[a-z_]+?)I\S*:\s*REG:(\d+) STACK:(\d+) SHARED:\d+ LOCAL:(\d+)"
    for name, reg, st, local in re.findall(pat, out):
        regs.setdefault(name, []).append(int(reg))
        stack.setdefault(name, []).append(int(st) + int(local))
    assert {k: sorted(v) for k, v in regs.items()} == REGS_LINEAR
    for k in REGS_LINEAR:
        assert set(stack[k]) == {0}, k                                           # no stack, no spills


# ------------------------------------------------------------------ GPU
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def D():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


CLASSES = ("BatchedEnv", "BatchedEnvComplicated", "BatchedEnvCooperation", "BatchedEnvCooperationSimplify")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _dt(D, t):
    return D.native.DTYPE_F32 if t.dtype == torch.float32 else D.native.DTYPE_BF16


def _p(t):
    return None if t is None else t.data_ptr()


class Guarded:
    """an output buffer of n elements with sentinel-filled guard memory before and after it"""

    def __init__(self, n, dtype, g=64):
        self.buf = torch.empty(n + 2 * g, dtype=dtype, device="cuda")
        self.buf.view(torch.uint8).fill_(SENT)
        self.g, self.n = g, n
        self.t = self.buf[g:g + n]

    def ptr(self):
        return self.t.data_ptr()

    def check(self):
        u8 = self.buf.view(torch.uint8)
        es = self.buf.element_size()
        assert (u8[:self.g * es] == SENT).all() and (u8[(self.g + self.n) * es:] == SENT).all()
        return self.t


class Head:
    """hidden [B, H] (a view of rows of ld elements), weight [13551, H], bias [13551] or None, one dtype"""

    def __init__(self, B, H, dtype, gen, ld=None, bias=True, scale=1.0):
        ld = ld or H
        self.h = (torch.randn((B, ld), device="cuda", generator=gen)).to(dtype)[:, :H]
        self.W = (torch.randn((NIDS, H), device="cuda", generator=gen) * (scale / H ** 0.5)).to(dtype)
        self.b = (torch.randn(NIDS, device="cuda", generator=gen) * 0.5).to(dtype) if bias else None
        self.B, self.H, self.dtype = B, H, dtype

    def args(self, D):
        return (self.h.data_ptr(), self.W.data_ptr(), _p(self.b), _dt(D, self.h), self.H, self.h.stride(0))

    def reference(self, owner, ids):
        """float64 W[id] . h + b of every entry, and the float32 bound gamma_{H+1} (sum |W h| + |b|)"""
        prod = self.W.to(torch.float64)[ids] * self.h.to(torch.float64)[owner]
        b = self.b.to(torch.float64)[ids] if self.b is not None else torch.zeros(len(ids), dtype=torch.float64, device="cuda")
        return prod.sum(1) + b, gamma(self.H + 1) * (prod.abs().sum(1) + b.abs())


def _lists(env):
    """(offsets, the whole list buffer, cap) of an env's current lists (an empty slice has no pointer)"""
    return env.offsets, env._actions_u64[env._cur], env.cap


def csr_of(off, ids, B):
    off = off.to(torch.int64)
    owner = torch.repeat_interleave(torch.arange(B, device="cuda"), off[1:] - off[:-1], output_size=int(off[-1].item()))
    return owner, ids.to(torch.int64)


def _mirrored(D, cls_name, B, steps, seed):
    env = getattr(D, cls_name)(B, seed=seed)
    env.prepare(*D.random_deals(B, seed=seed + 1))
    for _ in range(steps):
        env.step_random()
    return env


def logits_raw(D, off, act, cap, hd, stats=None):
    B = off.numel() - 1
    out = Guarded(cap, torch.float32)
    rc = D.native.lib.ddz_policy_linear_logits(off.data_ptr(), _p(act), cap, *hd.args(D), out.ptr(), _p(stats), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return out.check()


def lsample_raw(D, off, act, cap, hd, T, seed=0, env0=0, stepno=0, mask=None, state=None, stats=None):
    B = off.numel() - 1
    outs = [Guarded(B, torch.int32), Guarded(B, torch.int32), Guarded(B, torch.float32), Guarded(B, torch.float32)]
    rc = D.native.lib.ddz_policy_linear_sample(_p(state), off.data_ptr(), _p(act), cap, *hd.args(D), float(T), seed, env0,
                                               stepno, _p(mask), *[o.ptr() for o in outs], _p(stats), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return [o.check() for o in outs]


def dsample_raw(D, off, act, cap, dense, T, seed=0, env0=0, stepno=0, mask=None, state=None, stats=None):
    B = off.numel() - 1
    outs = [Guarded(B, torch.int32), Guarded(B, torch.int32), Guarded(B, torch.float32), Guarded(B, torch.float32)]
    rc = D.native.lib.ddz_policy_sample(_p(state), off.data_ptr(), _p(act), cap, dense.data_ptr(), D.native.DTYPE_F32,
                                        dense.stride(0), float(T), seed, env0, stepno, _p(mask), *[o.ptr() for o in outs],
                                        _p(stats), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return [o.check() for o in outs]


def llogprob_raw(D, off, act, cap, hd, ids, stats=None):
    B = off.numel() - 1
    outs = [Guarded(B, torch.float32) for _ in range(3)]
    rc = D.native.lib.ddz_policy_linear_logprob(off.data_ptr(), _p(act), cap, *hd.args(D), ids.data_ptr(),
                                                *[o.ptr() for o in outs], _p(stats), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return [o.check() for o in outs]


def dlogprob_raw(D, off, act, cap, dense, ids, stats=None):
    B = off.numel() - 1
    outs = [Guarded(B, torch.float32) for _ in range(3)]
    rc = D.native.lib.ddz_policy_logprob(off.data_ptr(), _p(act), cap, dense.data_ptr(), D.native.DTYPE_F32, dense.stride(0),
                                         ids.data_ptr(), *[o.ptr() for o in outs], _p(stats), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return [o.check() for o in outs]


def lbackward_raw(D, off, act, cap, hd, ids, lse, glp, gent, ld_g=None):
    """(grad_legal [cap], grad_hidden [B, H]) with guard memory, and the padding of grad_hidden's rows untouched"""
    B, H = off.numel() - 1, hd.H
    ld_g = ld_g or H
    gl = Guarded(cap, torch.float32)
    gh = Guarded(B * ld_g, hd.dtype)
    rc = D.native.lib.ddz_policy_linear_backward(off.data_ptr(), _p(act), cap, *hd.args(D), ids.data_ptr(), lse.data_ptr(),
                                                 _p(glp), _p(gent), gl.ptr(), gh.ptr(), ld_g, B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    rows = gh.check().view(B, ld_g)
    assert (rows[:, H:].contiguous().view(torch.uint8) == SENT).all()
    return gl.check(), rows[:, :H]


def dbackward_raw(D, off, act, cap, dense, ids, lse, glp, gent):
    B = off.numel() - 1
    g = torch.empty((B, NIDS), dtype=torch.float32, device="cuda")
    rc = D.native.lib.ddz_policy_logprob_backward(off.data_ptr(), _p(act), cap, dense.data_ptr(), D.native.DTYPE_F32,
                                                  dense.stride(0), ids.data_ptr(), lse.data_ptr(), _p(glp), _p(gent),
                                                  g.data_ptr(), NIDS, B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return g


def sort_by_id(D, act, n):
    """order int32 [n] (entries sorted by id, stable) and id_offsets int32 [13552], as the header asks"""
    key = D.move_ids(act[:n]).to(torch.int64)
    key = torch.where(key < 0, NIDS, key)
    keys, order = torch.sort(key, stable=True)
    id_offsets = torch.searchsorted(keys, torch.arange(NIDS + 1, device="cuda"))
    return order.to(torch.int32), id_offsets.to(torch.int32), key


def grad_weight_raw(D, off, n, hd, grad_legal, order, id_offsets, bias=True):
    B, H = off.numel() - 1, hd.H
    gw = Guarded(NIDS * H, hd.dtype)
    gb = Guarded(NIDS, hd.dtype) if bias else None
    ws = torch.empty(max(1, D.native.lib.ddz_policy_linear_workspace_bytes(n, H) // 4), dtype=torch.float32, device="cuda")
    ws.fill_(float("nan"))                                                       # nothing in it is read before written
    rc = D.native.lib.ddz_policy_linear_grad_weight(off.data_ptr(), n, hd.h.data_ptr(), _dt(D, hd.h), H, hd.h.stride(0),
                                                    _p(grad_legal), _p(order), _p(id_offsets), gw.ptr(),
                                                    None if gb is None else gb.ptr(), ws.data_ptr(), B, _stream())
    assert rc == 0
    torch.cuda.synchronize()
    return gw.check().view(NIDS, H), None if gb is None else gb.check()


def bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


# ------------------------------------------------------------------ the legal logits
def _check_logits(D, env, hd):
    off, act, cap = _lists(env)
    B = off.numel() - 1
    stats = torch.zeros(16, dtype=torch.int64, device="cuda")
    got = logits_raw(D, off, act, cap, hd, stats=stats)
    owner, ids = csr_of(off, env.legal_ids(), B)
    want, tol = hd.reference(owner, ids)
    n = len(ids)
    assert bool(((got[:n].to(torch.float64) - want).abs() <= tol).all())
    assert int(stats[7].item()) == 0
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("cls_name", CLASSES)
@pytest.mark.parametrize("B", [1, 7, 4096])
def test_logits_against_float64(D, cls_name, B):
    """every width path (one, a few and many 16-byte pieces per lane), both dtypes, padded rows; fresh, mid-game and
    finished envs (mid-game batches are not re-dealt)"""
    gen = torch.Generator(device="cuda").manual_seed(B + len(cls_name))
    seen = 0
    for k, (steps, dtype, H, pad) in enumerate(((0, torch.float32, 4, 0), (9, torch.bfloat16, 8, 8), (25, torch.float32, 24, 4),
                                                (40, torch.bfloat16, 24, 0), (15, torch.float32, 256, 12),
                                                (70, torch.bfloat16, 256, 8), (30, torch.float32, 1024, 0),
                                                (5, torch.bfloat16, 1024, 16))):
        env = _mirrored(D, cls_name, B, steps, seed=300 + B + k)
        seen += _check_logits(D, env, Head(B, H, dtype, gen, ld=H + pad, bias=k % 3 != 2))
    assert seen > 0


@pytest.mark.gpu
def test_logits_at_131072_envs_and_config5_lists(D):
    gen = torch.Generator(device="cuda").manual_seed(3)
    env = _mirrored(D, "BatchedEnvCooperation", 131072, 12, seed=77)
    assert _check_logits(D, env, Head(131072, 256, torch.bfloat16, gen)) > 500000
    hands, lasts = D.adversarial_pairs(2048)
    moves, off = D.get_moves(D.unpack_counts(torch.as_tensor(hands.view(np.int64))).numpy(),
                             D.unpack_counts(torch.as_tensor(lasts.view(np.int64))).numpy())
    B = off.numel() - 1
    assert int((off[1:] - off[:-1]).max().item()) >= 400
    owner, ids = csr_of(off, D.move_ids(moves), B)
    for dtype, H in ((torch.float32, 256), (torch.bfloat16, 64)):
        hd = Head(B, H, dtype, gen, ld=H + 8)
        got = logits_raw(D, off, moves, moves.numel(), hd)
        want, tol = hd.reference(owner, ids)
        assert bool(((got.to(torch.float64) - want).abs() <= tol).all())


# ------------------------------------------------------------------ bit for bit against the dense kernels
def _special_head(B, H, dtype, gen):
    """a head whose legal logits include NaN (NaN hidden rows), +-inf and NaN (infinite hidden entries against weights of
    both signs) and -inf (bias -inf at 2 % of the ids and at id 0, the pass)"""
    hd = Head(B, H, dtype, gen, ld=H + 8)
    rows = torch.arange(B, device="cuda")
    hd.h[rows % 13 == 5, 1] = float("nan")
    hd.h[rows % 17 == 6, 0] = float("inf")
    drop = torch.rand(NIDS, device="cuda", generator=gen) < 0.02
    drop[0] = True
    hd.b[drop] = float("-inf")
    return hd


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_bit_exact_to_the_dense_kernels(D, dtype):
    """the kernel's own legal logits scattered into a dense float32 row of -inf: ddz_policy_sample / _logprob /
    _logprob_backward on it give the linear kernels' outputs bit for bit, with env_mask, finished envs, illegal ids, and
    cut and dropped lists"""
    dtype = getattr(torch, dtype)
    B = 4096
    gen = torch.Generator(device="cuda").manual_seed(11)
    env = _mirrored(D, "BatchedEnvComplicated", B, 30, seed=21)
    off, act, cap = _lists(env)
    total = int(off[-1].item())
    owner, ids = csr_of(off, env.legal_ids(), B)
    hd = _special_head(B, 64, dtype, gen)
    legal = logits_raw(D, off, act, cap, hd)[:total]
    assert torch.isnan(legal).any() and torch.isneginf(legal).any() and torch.isposinf(legal).any()
    dense = torch.full((B, NIDS), float("-inf"), device="cuda")
    dense[owner, ids] = legal
    emask = (torch.rand(B, device="cuda", generator=gen) < 0.8).to(torch.uint8)
    full = (off[1:] - off[:-1]).to(torch.int64)
    caps = (total, total // 2 + 3, 17, 0)
    cut_seen = 0
    for cap_k in caps:
        a_k = act if cap_k else None
        stored = (cap_k - off[:-1].to(torch.int64)).clamp(min=0).minimum(full)
        cut = stored < full
        cut_seen += int(cut.sum().item())
        for T in (0.0, 0.5, 1.0, 2.0):
            for mask in (None, emask):
                sa, sb = torch.zeros(16, dtype=torch.int64, device="cuda"), torch.zeros(16, dtype=torch.int64, device="cuda")
                st_a, st_b = env._state.clone(), env._state.clone()
                kw = dict(seed=99, env0=5, stepno=int(T * 4) + 1, mask=mask)
                want = dsample_raw(D, off, a_k, cap_k, dense, T, state=st_a, stats=sa, **kw)
                got = lsample_raw(D, off, a_k, cap_k, hd, T, state=st_b, stats=sb, **kw)
                assert all(torch.equal(bits(x), bits(y)) for x, y in zip(got, want)), (cap_k, T)
                assert torch.equal(sa, sb) and torch.equal(st_a, st_b)
        # the training forward on sampled ids, a fifth of them replaced by ids off the list
        chosen = lsample_raw(D, off, act, total, hd, 1.0, seed=3)[1].clone()
        swap = torch.rand(B, device="cuda", generator=gen) < 0.2
        chosen[swap] = torch.tensor([-1, NIDS, NIDS + 7, 5000], device="cuda", dtype=torch.int32)[
            torch.randint(0, 4, (int(swap.sum().item()),), device="cuda", generator=gen)]
        sa, sb = torch.zeros(16, dtype=torch.int64, device="cuda"), torch.zeros(16, dtype=torch.int64, device="cuda")
        want = dlogprob_raw(D, off, a_k, cap_k, dense, chosen, stats=sa)
        got = llogprob_raw(D, off, a_k, cap_k, hd, chosen, stats=sb)
        assert all(torch.equal(bits(x), bits(y)) for x, y in zip(got, want)) and torch.equal(sa, sb), cap_k
        # the per-entry gradient: the dense row at the legal ids, exactly 0 for empty, cut and dropped lists
        lse = got[2]
        glp = torch.randn(B, device="cuda", generator=gen)
        gent = torch.randn(B, device="cuda", generator=gen)
        for gl_in, ge_in in ((glp, gent), (glp, None), (None, gent)):
            row = dbackward_raw(D, off, a_k, cap_k, dense, chosen, lse, gl_in, ge_in)
            gl, _ = lbackward_raw(D, off, a_k, cap_k, hd, chosen, lse, gl_in, ge_in)
            n_st = min(cap_k, total)
            keep = ~cut[owner[:n_st]]
            assert torch.equal(bits(gl[:n_st][keep]), bits(row[owner[:n_st], ids[:n_st]][keep])), cap_k
            assert (bits(gl[:n_st][~keep]) == 0).all()
            assert (row[cut] == 0).all()
    assert cut_seen > 0


# ------------------------------------------------------------------ gradients against float64
def _check_grads(D, off, act, n, hd, gl, gh, owner, ids, key, order, id_offsets):
    """grad_hidden, grad_weight and grad_bias of the kernels against float64 sums over the kernel's own grad_legal"""
    B, H = off.numel() - 1, hd.H
    g64 = gl[:n].to(torch.float64)
    W64, h64 = hd.W.to(torch.float64), hd.h.to(torch.float64)
    half = U16 if hd.dtype == torch.bfloat16 else 0.0
    cnt = torch.bincount(owner, minlength=B).to(torch.float64)
    # grad_hidden[b] = sum_i g_i W[id_i]: gamma_N sum |g W| (N = the list's length) + the output rounding
    t = g64[:, None] * W64[ids]
    want = torch.zeros((B, H), dtype=torch.float64, device="cuda").index_add_(0, owner, t)
    mag = torch.zeros((B, H), dtype=torch.float64, device="cuda").index_add_(0, owner, t.abs())
    tol = (cnt * U32 / (1 - cnt * U32))[:, None] * mag + want.abs() * half
    assert bool(((gh.to(torch.float64) - want).abs() <= tol).all())
    # grad_weight[id] = sum_e g_e h[env(e)], grad_bias[id] = sum_e g_e: gamma_n (n = the id's entries)
    gw, gb = grad_weight_raw(D, off, n, hd, gl[:n], order, id_offsets)
    valid = key < NIDS
    ki, oi, gv = key[valid], owner[valid], g64[valid]
    t = gv[:, None] * h64[oi]
    want = torch.zeros((NIDS, H), dtype=torch.float64, device="cuda").index_add_(0, ki, t)
    mag = torch.zeros((NIDS, H), dtype=torch.float64, device="cuda").index_add_(0, ki, t.abs())
    per = torch.bincount(ki, minlength=NIDS).to(torch.float64)
    gam = (per * U32 / (1 - per * U32))
    assert bool(((gw.to(torch.float64) - want).abs() <= gam[:, None] * mag + want.abs() * half).all())
    wb = torch.zeros(NIDS, dtype=torch.float64, device="cuda").index_add_(0, ki, gv)
    mb = torch.zeros(NIDS, dtype=torch.float64, device="cuda").index_add_(0, ki, gv.abs())
    assert bool(((gb.to(torch.float64) - wb).abs() <= gam * mb + wb.abs() * half).all())
    nowhere = per == 0
    assert int(nowhere.sum().item()) > 0
    assert (gw[nowhere].view(torch.uint8) == 0).all()                           # +0.0 exactly
    assert (gb[nowhere].view(torch.uint8) == 0).all()
    # no atomics: a second call gives the same bits
    gw2, gb2 = grad_weight_raw(D, off, n, hd, gl[:n], order, id_offsets)
    assert torch.equal(gw.view(torch.uint8), gw2.view(torch.uint8)) and torch.equal(gb.view(torch.uint8), gb2.view(torch.uint8))
    return int(per[0].item())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_gradients_against_float64(D, dtype):
    dtype = getattr(torch, dtype)
    gen = torch.Generator(device="cuda").manual_seed(5)
    for cls_name, B, steps, H in (("BatchedEnvCooperationSimplify", 4096, 25, 24), ("BatchedEnv", 7, 3, 256),
                                  ("BatchedEnvComplicated", 1, 0, 1024)):
        env = _mirrored(D, cls_name, B, steps, seed=40 + B)
        off, act, cap = _lists(env)
        n = int(off[-1].item())
        owner, ids = csr_of(off, env.legal_ids(), B)
        hd = Head(B, H, dtype, gen, ld=H + 8)
        chosen = lsample_raw(D, off, act, cap, hd, 1.0, seed=1)[1]
        lse = llogprob_raw(D, off, act, cap, hd, chosen)[2]
        glp = torch.randn(B, device="cuda", generator=gen)
        gent = torch.randn(B, device="cuda", generator=gen)
        gl, gh = lbackward_raw(D, off, act, cap, hd, chosen, lse, glp, gent, ld_g=H + 16)
        gl2, gh2 = lbackward_raw(D, off, act, cap, hd, chosen, lse, glp, gent)
        assert torch.equal(bits(gl), bits(gl2))                                # padded rows or not: the same bits
        assert torch.equal(gh.contiguous().view(torch.uint8), gh2.contiguous().view(torch.uint8))
        order, id_offsets, key = sort_by_id(D, act, n)
        _check_grads(D, off, act, n, hd, gl, gh, owner, ids, key, order, id_offsets)


@pytest.mark.gpu
def test_weight_gradient_of_a_long_pass_segment(D):
    """131 072 mid-game envs: the pass (id 0) has more than 60 000 entries, spread over hundreds of chunks"""
    B, H = 131072, 32
    gen = torch.Generator(device="cuda").manual_seed(8)
    env = _mirrored(D, "BatchedEnvCooperation", B, 6, seed=5)
    off, act, cap = _lists(env)
    n = int(off[-1].item())
    owner, ids = csr_of(off, env.legal_ids(), B)
    hd = Head(B, H, torch.float32, gen)
    chosen = lsample_raw(D, off, act, cap, hd, 1.0, seed=2)[1]
    lse = llogprob_raw(D, off, act, cap, hd, chosen)[2]
    gl, gh = lbackward_raw(D, off, act, cap, hd, chosen, lse, torch.randn(B, device="cuda", generator=gen),
                           torch.randn(B, device="cuda", generator=gen))
    order, id_offsets, key = sort_by_id(D, act, n)
    passes = _check_grads(D, off, act, n, hd, gl, gh, owner, ids, key, order, id_offsets)
    print("entries of the pass id: %d of %d" % (passes, n))
    assert passes > 60000


@pytest.mark.gpu
def test_grad_weight_without_entries(D):
    """n = 0 writes every row and bias element once, as exact zeros"""
    B, H = 4, 16
    hd = Head(B, H, torch.float32, torch.Generator(device="cuda").manual_seed(0))
    off = torch.zeros(B + 1, dtype=torch.int32, device="cuda")
    gw, gb = grad_weight_raw(D, off, 0, hd, None, None, None)
    assert (gw.view(torch.int32) == 0).all() and (gb.view(torch.int32) == 0).all()


# ------------------------------------------------------------------ the module, end to end
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "bfloat16"])
def test_log_prob_autograd_against_float64(D, dtype):
    """LinearPolicyHead.log_prob's gradients of h, weight and bias against float64 autograd through the dense forward and
    a masked log_softmax.  Tolerance: a legal logit is within delta = gamma_{H+1} (sum |W h| + |b|) of the exact one, so p
    within about 2 delta relative; on top of the float32 softmax bound of the dense kernels' test, each entry's gradient
    g_e is within tg_e = (4 e (3 N + 12 + 2 |log S| + |l - m|) + 4 delta_env) (|g_lp| + |g_ent| (2 + |H|)); then
    grad_h within sum tg |W| + gamma_N sum |g W|, grad_W within sum tg |h| + gamma_n sum |g h|, grad_b within
    sum tg + gamma_n sum |g|, plus a bfloat16 output's half ulp"""
    dtype = getattr(torch, dtype)
    B, H = 2048, 64
    gen = torch.Generator(device="cuda").manual_seed(31)
    env = _mirrored(D, "BatchedEnvCooperation", B, 20, seed=9)
    off, act = env.offsets, env.actions_packed
    owner, ids = csr_of(off, env.legal_ids(), B)
    head = D.LinearPolicyHead(H, device="cuda", dtype=dtype)
    with torch.no_grad():
        head.weight.copy_(torch.randn((NIDS, H), device="cuda", generator=gen) * 0.5)
        head.bias.copy_(torch.randn(NIDS, device="cuda", generator=gen))
    h = torch.randn((B, H), device="cuda", generator=gen).to(dtype)
    chosen = head.sample(env, h, temperature=1.0, seed=4)[1]
    # the Python outputs are the raw entry points'
    hd = Head(B, H, dtype, gen)
    hd.h, hd.W, hd.b = h, head.weight.detach(), head.bias.detach()
    raw_logits = logits_raw(D, off, env._actions_u64[env._cur], env.cap, hd)[:len(ids)]
    assert torch.equal(bits(head.legal_logits(h, off, act)), bits(raw_logits))
    assert torch.equal(chosen, lsample_raw(D, off, env._actions_u64[env._cur], env.cap, hd, 1.0, seed=4, env0=env.env0,
                                           stepno=env._stepno)[1])
    glp = torch.randn(B, device="cuda", generator=gen)
    gent = torch.randn(B, device="cuda", generator=gen)
    hh = h.clone().requires_grad_(True)
    lp, ent = head.log_prob(hh, off, act, chosen)
    (glp * lp + gent * ent).sum().backward()
    # float64 autograd of the dense path
    mask = torch.zeros((B, NIDS), dtype=torch.bool, device="cuda")
    mask[owner, ids] = True
    live = chosen >= 0
    h64 = h.detach().to(torch.float64).requires_grad_(True)
    W64 = head.weight.detach().to(torch.float64).requires_grad_(True)
    b64 = head.bias.detach().to(torch.float64).requires_grad_(True)
    x = torch.nn.functional.linear(h64, W64, b64)
    logp = torch.log_softmax(x.masked_fill(~mask, -1e300), 1)
    zero = torch.zeros(B, dtype=torch.float64, device="cuda")
    lp_c = torch.where(live, logp.gather(1, chosen.clamp(min=0).to(torch.int64)[:, None])[:, 0], zero)
    Hs = torch.where(live, -torch.where(mask, logp.exp() * logp, torch.zeros_like(logp)).sum(1), zero)
    (glp.double() * lp_c + gent.double() * Hs).sum().backward()
    # the tolerance
    xl = x.detach()[owner, ids]
    _, delta = hd.reference(owner, ids)
    m = torch.full((B,), float("-inf"), dtype=torch.float64, device="cuda").scatter_reduce(0, owner, xl, "amax")
    lse = torch.logsumexp(x.detach().masked_fill(~mask, float("-inf")), 1)
    d_env = torch.zeros(B, dtype=torch.float64, device="cuda").scatter_reduce(0, owner, delta, "amax")
    N = torch.bincount(owner, minlength=B).to(torch.float64)
    e = U32
    tol_p = 4 * e * (3 * N[owner] + 12 + 2 * (lse - m)[owner].abs() + (xl - m[owner]).abs()) + 4 * d_env[owner]
    tg = tol_p * (glp.double().abs() + gent.double().abs() * (2 + Hs.detach().abs()))[owner]
    p = (xl - lse[owner]).exp()
    g_ex = (glp.double()[owner] * ((ids == chosen.to(torch.int64)[owner]).double() - p)
            - gent.double()[owner] * p * ((xl - lse[owner]) + Hs.detach()[owner])).abs() + tg   # >= |g_e| of the kernel
    half = U16 if dtype == torch.bfloat16 else 0.0
    Wl, hl = W64.detach()[ids], h64.detach()[owner]
    gam_N = (N * e / (1 - N * e))
    tol_h = torch.zeros((B, H), dtype=torch.float64, device="cuda").index_add_(0, owner, tg[:, None] * Wl.abs()) + \
        gam_N[:, None] * torch.zeros((B, H), dtype=torch.float64, device="cuda").index_add_(0, owner, g_ex[:, None] * Wl.abs())
    per = torch.bincount(ids, minlength=NIDS).to(torch.float64)
    gam_n = per * e / (1 - per * e)
    tol_w = torch.zeros((NIDS, H), dtype=torch.float64, device="cuda").index_add_(0, ids, tg[:, None] * hl.abs()) + \
        gam_n[:, None] * torch.zeros((NIDS, H), dtype=torch.float64, device="cuda").index_add_(0, ids, g_ex[:, None] * hl.abs())
    tol_b = torch.zeros(NIDS, dtype=torch.float64, device="cuda").index_add_(0, ids, tg) + \
        gam_n * torch.zeros(NIDS, dtype=torch.float64, device="cuda").index_add_(0, ids, g_ex)
    for got, want, tol in ((hh.grad, h64.grad, tol_h), (head.weight.grad, W64.grad, tol_w), (head.bias.grad, b64.grad, tol_b)):
        assert got.dtype == dtype
        err = (got.to(torch.float64) - want).abs()
        assert bool((err <= tol + want.abs() * half).all()), float((err - tol - want.abs() * half).max())
    assert (head.weight.grad[per == 0] == 0).all() and (head.bias.grad[per == 0] == 0).all()


@pytest.mark.gpu
def test_training_step_memory_at_131072_envs(D):
    """forward + backward of -(adv * logp).sum() - 0.01 * H.sum() at B = 131 072, H = 256: the peak extra memory stays under
    a bound from shapes -- grad_h and the hidden copy a bfloat16 cast would make (2 B H 4), 128 bytes per list entry (ids,
    sort keys and indices, order, grad_legal, the sort's scratch), three weight-sized tensors (grad_W, the workspace, slack)
    and 64 bytes per env -- far under one [B, 13551] float32 tensor"""
    B, H = 131072, 256
    env = _mirrored(D, "BatchedEnvCooperation", B, 24, seed=7)
    off, act = env.offsets, env.actions_packed
    head = D.LinearPolicyHead(H, device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(1)
    h = torch.randn((B, H), device="cuda", generator=gen).requires_grad_(True)
    adv = torch.randn(B, device="cuda", generator=gen)
    ids = head.sample(env, h.detach(), seed=3)[1]
    n = act.numel()

    def step():
        lp, ent = head.log_prob(h, off, act, ids)
        (-(adv * lp).sum() - 0.01 * ent.sum()).backward()

    step()                                                                       # the gradients' own storage exists now
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    step()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    bound = 2 * B * H * 4 + 128 * n + 3 * NIDS * H * 4 + 64 * B
    print("peak extra memory %.1f MB, bound %.1f MB, a dense [B, 13551] float32 tensor %.1f MB"
          % (peak / 2 ** 20, bound / 2 ** 20, B * NIDS * 4 / 2 ** 20))
    assert peak <= bound and bound < B * NIDS * 4 // 10
    assert int(env.stats[7].item()) == 0


def _landlord_games(D, policy, B, deal_seed, rng_seed, learn):
    """B seeded games, the landlord seat played by the HeadedPolicy `policy` through head.sample (T = 1 while learning, else
    argmax; None: a uniformly random landlord), farmers uniformly random.  Returns (landlord wins, the landlord's decisions
    (states, faces, ids, env index), won)."""
    env = D.BatchedEnvCooperation(B, seed=rng_seed)
    env.prepare(*D.random_deals(B, seed=deal_seed))
    gen = torch.Generator(device="cuda").manual_seed(rng_seed)
    won = torch.zeros(B, dtype=torch.bool, device="cuda")
    over = torch.zeros(B, dtype=torch.bool, device="cuda")
    trace = []
    while not bool(over.all()):
        cnt = (env.offsets[1:] - env.offsets[:-1]).to(torch.int64)
        lord = (env.get_role_ID() == 2) & ~over
        rnd = torch.randint(0, 1 << 30, (B,), device="cuda", generator=gen) % cnt.clamp(min=1)
        if policy is None:
            pick = rnd
        else:
            with torch.no_grad():
                h = policy.trunk(env.face)
            choice, ids, _, _ = policy.head.sample(env, h, temperature=1.0 if learn else 0.0, seed=rng_seed, env_mask=lord)
            pick = torch.where(lord, choice.to(torch.int64), rnd)
            if learn and bool(lord.any()):
                idx = torch.nonzero(lord).flatten()
                trace.append((D.gather_states(env, idx), env.face[idx].clone(), ids[idx], idx))
        env.step(pick.to(torch.int32))
        newly = env.is_done & ~over
        won |= newly & (env.winner == 1)
        over |= newly
    assert int(env.stats[7].item()) == 0
    return int(won.sum().item()), trace, won


def _zero_policy(D, C=9):
    head = D.LinearPolicyHead(C * 60, device="cuda")
    torch.nn.init.zeros_(head.weight)
    torch.nn.init.zeros_(head.bias)
    return D.HeadedPolicy(torch.nn.Flatten(), head)


@pytest.mark.gpu
def test_reinforce_landlord_learns(D):
    """A HeadedPolicy landlord (flattened face -> LinearPolicyHead) trained by REINFORCE with a mean baseline through
    head.sample + head.log_prob on the re-derived lists of its recorded states wins clearly more of the same seeded deals
    against random farmers than a random landlord"""
    torch.manual_seed(0)
    policy = _zero_policy(D)
    opt = torch.optim.Adam(policy.parameters(), lr=0.01)
    B = 2048
    for it in range(40):
        _, trace, won = _landlord_games(D, policy, B, deal_seed=1000 + it, rng_seed=it + 1, learn=True)
        R = won.to(torch.float32) * 2 - 1
        adv = R - R.mean()
        loss = 0.0
        for st, face, ids, idx in trace:
            off, act = D.legal_lists_of_states(st)
            logp, _ = policy.head.log_prob(policy.trunk(face), off, act, ids)
            loss = loss - (adv[idx] * logp).sum() / B
        opt.zero_grad()
        loss.backward()
        opt.step()
    eval_B = 4096
    trained, _, _ = _landlord_games(D, policy, eval_B, deal_seed=5, rng_seed=99, learn=False)
    rand, _, _ = _landlord_games(D, None, eval_B, deal_seed=5, rng_seed=99, learn=False)
    print("landlord wins of %d seeded deals: trained %d, random %d" % (eval_B, trained, rand))
    assert trained > rand + eval_B // 20


@pytest.mark.gpu
def test_game_and_compete_with_a_headed_policy_seat(D):
    policy = _zero_policy(D)
    torch.nn.init.normal_(policy.head.weight, std=0.01)
    calls = []
    real = policy.head._sample

    def spy(*a, **kw):
        calls.append(1)
        return real(*a, **kw)
    policy.head._sample = spy
    wins = D.BatchedGame.compete(D.BatchedEnvCooperation, {}, {}, None, total=512, num_envs=256, debug=False, seed=3,
                                 policy_dict={"lord": policy})
    assert sum(wins.values()) >= 512 and calls
    g = D.BatchedGame(D.BatchedEnvCooperation, {}, {}, num_envs=256, seed=3, policy_dict={"lord": policy})
    g.play(256)
    assert int(g.env.stats[7].item()) == 0 and g.episodes >= 256
