"""Fixed-head policies over the action ids (include/ddz_b200.h: ddz_policy_sample, ddz_policy_logprob,
ddz_policy_logprob_backward), and linear heads evaluated only at the legal ids (ddz_policy_linear_*: LinearPolicyHead,
HeadedPolicy).

A fixed-head policy maps a state to logits [B, 13551], one per action id (move_ids).  Its softmax is restricted to the
legal ids of each env, and these kernels read only those logits (mean 5.6, at most 512 per env): no dense mask, no
masked_fill, no full-size log_softmax or saved tensors.  Sampling at decision time, and log-probability + entropy with
their gradient at training time, each take one launch; the gradient row is written once, zero off the legal set.
"""
import math

import torch
import torch.nn.functional as F

from . import _native as N

_DTYPES = {torch.float32: N.DTYPE_F32, torch.bfloat16: N.DTYPE_BF16}


def _head(logits, B, device):
    """(logits, dtype code, row stride) of a float32 / bfloat16 [B, 13551] head on `device` (rows may be padded)"""
    if not isinstance(logits, torch.Tensor) or logits.dim() != 2 or tuple(logits.shape) != (B, N.NUM_ACTION_IDS):
        raise ValueError("logits must be a [%d, %d] tensor" % (B, N.NUM_ACTION_IDS))
    if logits.dtype not in _DTYPES:
        raise ValueError("logits must be float32 or bfloat16, not %s" % (logits.dtype,))
    if logits.device != torch.device(device):
        raise ValueError("logits are on %s, the lists on %s" % (logits.device, device))
    if logits.stride(1) != 1 or logits.stride(0) < N.NUM_ACTION_IDS:
        logits = logits.contiguous()
    return logits, _DTYPES[logits.dtype], logits.stride(0)


def policy_sample(env, logits, temperature=1.0, seed=0, env_mask=None):
    """One move per env of a batched env from its fixed-head logits [B, 13551] (float32 or bfloat16), softmax over the
    env's legal ids at `temperature` (ddz_policy_sample).  The draw of env b is Philox-keyed (seed, env.env0 + b, the step
    number of the env's next step).  temperature = 0: argmax (lowest id on ties, NaN first, as torch.argmax), with logp and
    entropy of temperature 1.  env_mask bool [B] (optional): only those envs.
    Returns (choice int32 [B] = index in the env's legal list, feeds env.step; ids int32 [B]; logp float32 [B] = log-
    probability of the chosen move; entropy float32 [B]).  Finished and masked-out envs get -1 / -1 / 0 / 0.  An env whose
    legal logits are all -inf (or, at temperature > 0, include NaN or +inf) is not drawn from: -1, its sticky error bit is
    set and env.stats[7] counts it (debug=True raises)."""
    out = _sample(env, logits, temperature, seed, env_mask, record=True)
    env._check_errors("policy_sample")
    return out


def _sample(env, logits, temperature, seed, env_mask, record):
    """ddz_policy_sample over the env's current lists; record=False leaves the sticky bit and stats[7] of an env that is not
    drawn from to the step that follows (its choice -1 is an illegal choice there), so that it is counted once"""
    env.num_actions                                   # complete lists: the buffers grow if they have to
    B, dev = env.B, env.device
    logits, dt, ld = _head(logits, B, dev)
    mask8 = None if env_mask is None else torch.as_tensor(env_mask, device=dev).reshape(B).to(torch.uint8).contiguous()
    choice = torch.empty(B, dtype=torch.int32, device=dev)
    ids = torch.empty(B, dtype=torch.int32, device=dev)
    logp = torch.empty(B, dtype=torch.float32, device=dev)
    entropy = torch.empty(B, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_policy_sample(env._state.data_ptr() if record else None, env._offsets[env._cur].data_ptr(),
                                        env._actions_u64[env._cur].data_ptr(), env.cap, logits.data_ptr(), dt, ld,
                                        float(temperature), int(seed) & 0xFFFFFFFFFFFFFFFF, env.env0, env._stepno,
                                        None if mask8 is None else mask8.data_ptr(), choice.data_ptr(), ids.data_ptr(),
                                        logp.data_ptr(), entropy.data_ptr(), env.stats.data_ptr() if record else None, B,
                                        env._stream()), "ddz_policy_sample")
    return choice, ids, logp, entropy


class _PolicyLogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, offsets, actions, ids, stats):
        B, dev = offsets.numel() - 1, offsets.device
        head, dt, ld = _head(logits, B, dev)
        logp = torch.empty(B, dtype=torch.float32, device=dev)
        entropy = torch.empty(B, dtype=torch.float32, device=dev)
        lse = torch.empty(B, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.ddz_policy_logprob(offsets.data_ptr(), actions.data_ptr(), actions.numel(), head.data_ptr(), dt, ld,
                                             ids.data_ptr(), logp.data_ptr(), entropy.data_ptr(), lse.data_ptr(),
                                             None if stats is None else stats.data_ptr(), B,
                                             torch.cuda.current_stream(dev).cuda_stream), "ddz_policy_logprob")
        ctx.save_for_backward(head, offsets, actions, ids, lse)
        ctx.set_materialize_grads(False)
        return logp, entropy

    @staticmethod
    def backward(ctx, g_logp, g_entropy):
        head, offsets, actions, ids, lse = ctx.saved_tensors
        B, dev = offsets.numel() - 1, offsets.device
        grad = torch.empty((B, N.NUM_ACTION_IDS), dtype=head.dtype, device=dev)
        g_logp = None if g_logp is None else g_logp.to(torch.float32).contiguous()
        g_entropy = None if g_entropy is None else g_entropy.to(torch.float32).contiguous()
        with torch.cuda.device(dev):
            N.check(N.lib.ddz_policy_logprob_backward(offsets.data_ptr(), actions.data_ptr(), actions.numel(), head.data_ptr(),
                                                      _DTYPES[head.dtype], head.stride(0), ids.data_ptr(), lse.data_ptr(),
                                                      None if g_logp is None else g_logp.data_ptr(),
                                                      None if g_entropy is None else g_entropy.data_ptr(), grad.data_ptr(),
                                                      N.NUM_ACTION_IDS, B, torch.cuda.current_stream(dev).cuda_stream),
                    "ddz_policy_logprob_backward")
        return grad, None, None, None, None


def policy_log_prob(logits, offsets, actions_packed, ids, stats=None):
    """Training-time forward of a fixed-head policy (ddz_policy_logprob), differentiable in `logits`: for the chosen action
    ids (int32 [B], e.g. from replay) over the lists offsets int32 [B+1] / actions_packed int64 [sumN] (env.offsets /
    env.actions_packed, or legal_lists_of_states of replayed states), returns (logp, entropy), float32 [B] each, of the
    softmax over each env's legal ids (temperature 1).  An id not in its env's list gives logp = -inf; legal logits with no
    softmax (all -inf, or a NaN or +inf among them) give NaN, as torch's log_softmax does; both are counted in stats[7]
    when an int64 [16] stats tensor is given.  backward writes the full [B, 13551] gradient row once, exactly 0
    off the legal set (ddz_policy_logprob_backward)."""
    dev = logits.device
    offsets = offsets.to(device=dev, dtype=torch.int32).contiguous()
    actions = actions_packed.to(device=dev, dtype=torch.int64).contiguous()
    ids = torch.as_tensor(ids, device=dev).to(torch.int32).contiguous()
    if ids.numel() != offsets.numel() - 1:
        raise ValueError("ids must have one entry per env (%d), not %d" % (offsets.numel() - 1, ids.numel()))
    return _PolicyLogProb.apply(logits, offsets, actions, ids, stats)


def legal_lists_of_states(packed_states, device=None):
    """The legal-move lists of library states (int32 [19 n], e.g. trainer.gather_states of a replay minibatch), re-derived on
    the device (ddz_legal_count, then ddz_legal_emit): (offsets int32 [n+1], actions_packed int64 [sumN]), the lists the
    envs had when those states were observed -- so a replayed minibatch can be re-scored without storing masks."""
    dev = torch.device(device) if device is not None else packed_states.device
    if dev.type != "cuda":
        raise N.DdzError("legal lists are built on a CUDA device")
    state = packed_states.to(device=dev, dtype=torch.int32).contiguous()
    n = state.numel() // N.STATE_WORDS
    if n <= 0 or state.numel() != n * N.STATE_WORDS:
        raise ValueError("packed_states must hold int32 [19 n] with n > 0")
    stream = torch.cuda.current_stream(dev).cuda_stream
    counts = torch.empty(n, dtype=torch.int32, device=dev)
    offsets = torch.empty(n + 1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        N.check(N.lib.ddz_legal_count(state.data_ptr(), counts.data_ptr(), n, stream), "ddz_legal_count")
        total = int(counts.sum().item())
        actions = torch.empty(max(total, 1), dtype=torch.int64, device=dev)
        ws = torch.zeros(max(1, N.lib.ddz_workspace_bytes(n) // 4), dtype=torch.int32, device=dev)
        N.check(N.lib.ddz_legal_emit(state.data_ptr(), ws.data_ptr(), offsets.data_ptr(), actions.data_ptr(), total, None, n,
                                     stream), "ddz_legal_emit")
    return offsets, actions[:total]


# ------------------------------------------------------------------ linear heads evaluated at the legal ids
def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


def _ptr(t):
    return None if t is None or t.numel() == 0 else t.data_ptr()


def _hidden_rows(h, weight, B):
    """(h, dtype code, H, ld) of hidden vectors [B, H] in the dtype and on the device of `weight`, with rows the kernels
    read: whole 16-byte pieces, 16-byte aligned (copied when they are not)"""
    if not isinstance(h, torch.Tensor) or h.dim() != 2 or tuple(h.shape) != (B, weight.shape[1]):
        raise ValueError("hidden must be a [%d, %d] tensor" % (B, weight.shape[1]))
    if h.dtype != weight.dtype or h.device != weight.device:
        raise ValueError("hidden is %s on %s, the head %s on %s" % (h.dtype, h.device, weight.dtype, weight.device))
    vec = 16 // h.element_size()
    if h.stride(1) != 1 or h.stride(0) < h.shape[1] or h.stride(0) % vec or h.data_ptr() % 16:
        h = h.clone(memory_format=torch.contiguous_format)
    return h, _DTYPES[h.dtype], int(h.shape[1]), h.stride(0)


def _indexed(dev):
    """a device with its index ("cuda" -> "cuda:<current>")"""
    dev = torch.device(dev)
    return torch.device(dev.type, torch.cuda.current_device()) if dev.type == "cuda" and dev.index is None else dev


def _move_ids(actions):
    ids = torch.empty(actions.numel(), dtype=torch.int32, device=actions.device)
    if actions.numel():
        N.check(N.lib.ddz_move_ids(actions.data_ptr(), actions.numel(), ids.data_ptr(), _stream(actions.device)),
                "ddz_move_ids")
    return ids


def _weight_grads(h, dt, H, ld, offsets, actions, grad_legal, dtype, with_bias):
    """(grad_weight [13551, H], grad_bias [13551] or None) from the per-entry gradients (ddz_policy_linear_grad_weight).
    The entries sorted by id, stable, and the start of every id's segment: the order of each sum is fixed by the lists."""
    dev, n, B = h.device, actions.numel(), offsets.numel() - 1
    key = _move_ids(actions)
    key = torch.where(key < 0, N.NUM_ACTION_IDS, key)              # entries that are not moves go last, and are ignored
    keys, order = torch.sort(key, stable=True)
    order = order.to(torch.int32)
    id_offsets = torch.searchsorted(keys, torch.arange(N.NUM_ACTION_IDS + 1, dtype=torch.int32, device=dev), out_int32=True)
    ws = torch.empty(max(1, N.lib.ddz_policy_linear_workspace_bytes(n, H) // 4), dtype=torch.float32, device=dev)
    gw = torch.empty((N.NUM_ACTION_IDS, H), dtype=dtype, device=dev)
    gb = torch.empty(N.NUM_ACTION_IDS, dtype=dtype, device=dev) if with_bias else None
    N.check(N.lib.ddz_policy_linear_grad_weight(offsets.data_ptr(), n, h.data_ptr(), dt, H, ld, _ptr(grad_legal),
                                                _ptr(order), _ptr(id_offsets), gw.data_ptr(), _ptr(gb), ws.data_ptr(), B,
                                                _stream(dev)), "ddz_policy_linear_grad_weight")
    return gw, gb


class _LinearLogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, weight, bias, offsets, actions, ids, stats):
        B, dev = offsets.numel() - 1, offsets.device
        w = weight.detach().contiguous()
        b = None if bias is None else bias.detach().contiguous()
        h, dt, H, ld = _hidden_rows(h.detach(), w, B)
        logp = torch.empty(B, dtype=torch.float32, device=dev)
        entropy = torch.empty(B, dtype=torch.float32, device=dev)
        lse = torch.empty(B, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.ddz_policy_linear_logprob(offsets.data_ptr(), _ptr(actions), actions.numel(), h.data_ptr(),
                                                    w.data_ptr(), _ptr(b), dt, H, ld, ids.data_ptr(), logp.data_ptr(),
                                                    entropy.data_ptr(), lse.data_ptr(),
                                                    None if stats is None else stats.data_ptr(), B, _stream(dev)),
                    "ddz_policy_linear_logprob")
        ctx.save_for_backward(h, w, b, offsets, actions, ids, lse)
        ctx.set_materialize_grads(False)
        return logp, entropy

    @staticmethod
    def backward(ctx, g_logp, g_entropy):
        h, w, b, offsets, actions, ids, lse = ctx.saved_tensors
        B, dev, n = offsets.numel() - 1, offsets.device, actions.numel()
        dt, H, ld = _DTYPES[h.dtype], int(h.shape[1]), h.stride(0)
        g_logp = None if g_logp is None else g_logp.to(torch.float32).contiguous()
        g_entropy = None if g_entropy is None else g_entropy.to(torch.float32).contiguous()
        grad_legal = torch.empty(n, dtype=torch.float32, device=dev)
        grad_h = torch.empty((B, H), dtype=h.dtype, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.ddz_policy_linear_backward(offsets.data_ptr(), _ptr(actions), n, h.data_ptr(), w.data_ptr(), _ptr(b),
                                                     dt, H, ld, ids.data_ptr(), lse.data_ptr(), _ptr(g_logp),
                                                     _ptr(g_entropy), _ptr(grad_legal), grad_h.data_ptr(), H, B,
                                                     _stream(dev)), "ddz_policy_linear_backward")
            gw = gb = None
            if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:
                gw, gb = _weight_grads(h, dt, H, ld, offsets, actions, grad_legal, h.dtype,
                                       b is not None and ctx.needs_input_grad[2])
        return (grad_h if ctx.needs_input_grad[0] else None, gw if ctx.needs_input_grad[1] else None, gb,
                None, None, None, None)


class LinearPolicyHead(torch.nn.Module):
    """The last layer of a fixed-head policy, logits = h W^T + bias over the 13 551 action ids, evaluated only at the legal
    ids of each env (ddz_policy_linear_*): sampling, log-probability, entropy and the gradients of h, W and bias never make
    a [B, 13551] tensor.  weight [13551, in_features] and bias [13551] are nn.Linear's parameters in nn.Linear's layout, so
    load_state_dict from an nn.Linear(in_features, 13551) works (from_linear).  float32 or bfloat16; the fused paths need
    in_features a multiple of 4 (float32) or 8 (bfloat16), at most 1024.  forward(h) is the dense F.linear, so the head
    still works wherever a dense head does (policy_sample, policy_log_prob)."""

    def __init__(self, in_features, bias=True, device=None, dtype=None):
        super().__init__()
        kw = {"device": device, "dtype": dtype}
        self.in_features, self.out_features = int(in_features), N.NUM_ACTION_IDS
        self.weight = torch.nn.Parameter(torch.empty((N.NUM_ACTION_IDS, self.in_features), **kw))
        if bias:
            self.bias = torch.nn.Parameter(torch.empty(N.NUM_ACTION_IDS, **kw))
        else:
            self.register_parameter("bias", None)
        self.reset_parameters()

    def reset_parameters(self):
        """nn.Linear's initialisation"""
        torch.nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        if self.bias is not None:
            bound = 1 / math.sqrt(self.in_features) if self.in_features > 0 else 0
            torch.nn.init.uniform_(self.bias, -bound, bound)

    @classmethod
    def from_linear(cls, linear):
        """a head holding a copy of the parameters of nn.Linear(in_features, 13551)"""
        if linear.out_features != N.NUM_ACTION_IDS:
            raise ValueError("an nn.Linear with %d outputs, not %d" % (linear.out_features, N.NUM_ACTION_IDS))
        head = cls(linear.in_features, bias=linear.bias is not None, device=linear.weight.device, dtype=linear.weight.dtype)
        head.load_state_dict(linear.state_dict())
        return head

    def extra_repr(self):
        return "in_features=%d, out_features=%d, bias=%s" % (self.in_features, self.out_features, self.bias is not None)

    def forward(self, h):
        """the dense logits [B, 13551]"""
        return F.linear(h, self.weight, self.bias)

    def _check_fused(self):
        if self.weight.dtype not in _DTYPES:
            raise ValueError("the head must be float32 or bfloat16, not %s" % (self.weight.dtype,))
        vec = 16 // self.weight.element_size()
        if self.in_features % vec or not 0 < self.in_features <= N.LINEAR_MAX_HIDDEN:
            raise ValueError("in_features must be a multiple of %d in [%d, %d] for the fused paths, not %d"
                             % (vec, vec, N.LINEAR_MAX_HIDDEN, self.in_features))

    def _params(self, B, h):
        """(weight, bias, h, dtype code, H, ld) for a launch"""
        self._check_fused()
        w = self.weight.detach().contiguous()
        b = None if self.bias is None else self.bias.detach().contiguous()
        return (w, b) + _hidden_rows(h.detach().to(w.dtype), w, B)

    def legal_logits(self, h, offsets, actions_packed):
        """the legal logits W[id] . h_b + bias[id] of every entry of the lists offsets int32 [B+1] / actions_packed int64
        [sumN], float32 [sumN] in CSR order (ddz_policy_linear_logits; not differentiable).  An entry of a list longer than
        512 gets NaN."""
        dev = self.weight.device
        offsets = offsets.to(device=dev, dtype=torch.int32).contiguous()
        actions = actions_packed.to(device=dev, dtype=torch.int64).contiguous()
        w, b, hd, dt, H, ld = self._params(offsets.numel() - 1, h)
        out = torch.empty(actions.numel(), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.ddz_policy_linear_logits(offsets.data_ptr(), _ptr(actions), actions.numel(), hd.data_ptr(),
                                                   w.data_ptr(), _ptr(b), dt, H, ld, _ptr(out), None, offsets.numel() - 1,
                                                   _stream(dev)), "ddz_policy_linear_logits")
        return out

    def sample(self, env, h, temperature=1.0, seed=0, env_mask=None):
        """policy_sample(env, self(h), temperature, seed, env_mask) without the dense logits (ddz_policy_linear_sample):
        the same draw, outputs and error handling.  Returns (choice, ids, logp, entropy), int32 / int32 / float32 / float32
        [B]."""
        out = self._sample(env, h, temperature, seed, env_mask, record=True)
        env._check_errors("LinearPolicyHead.sample")
        return out

    def _sample(self, env, h, temperature, seed, env_mask, record):
        """policy._sample with the head's logits"""
        env.num_actions                                   # complete lists: the buffers grow if they have to
        B, dev = env.B, env.device
        if _indexed(dev) != _indexed(self.weight.device):
            raise ValueError("the head is on %s, the env on %s" % (self.weight.device, dev))
        w, b, hd, dt, H, ld = self._params(B, h)
        mask8 = None if env_mask is None else torch.as_tensor(env_mask, device=dev).reshape(B).to(torch.uint8).contiguous()
        choice = torch.empty(B, dtype=torch.int32, device=dev)
        ids = torch.empty(B, dtype=torch.int32, device=dev)
        logp = torch.empty(B, dtype=torch.float32, device=dev)
        entropy = torch.empty(B, dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            N.check(N.lib.ddz_policy_linear_sample(env._state.data_ptr() if record else None, env._offsets[env._cur].data_ptr(),
                                                   env._actions_u64[env._cur].data_ptr(), env.cap, hd.data_ptr(), w.data_ptr(),
                                                   _ptr(b), dt, H, ld, float(temperature), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                                   env.env0, env._stepno, None if mask8 is None else mask8.data_ptr(),
                                                   choice.data_ptr(), ids.data_ptr(), logp.data_ptr(), entropy.data_ptr(),
                                                   env.stats.data_ptr() if record else None, B, env._stream()),
                    "ddz_policy_linear_sample")
        return choice, ids, logp, entropy

    def log_prob(self, h, offsets, actions_packed, ids, stats=None):
        """policy_log_prob(self(h), offsets, actions_packed, ids, stats) without the dense logits
        (ddz_policy_linear_logprob): (logp, entropy) float32 [B], differentiable in h, weight and bias.  The backward
        writes grad_h [B, H] and the weight and bias gradients from the per-entry gradients
        (ddz_policy_linear_backward, ddz_policy_linear_grad_weight); nothing of size [B, 13551] is made or saved."""
        dev = self.weight.device
        offsets = offsets.to(device=dev, dtype=torch.int32).contiguous()
        actions = actions_packed.to(device=dev, dtype=torch.int64).contiguous()
        ids = torch.as_tensor(ids, device=dev).to(torch.int32).contiguous()
        if ids.numel() != offsets.numel() - 1:
            raise ValueError("ids must have one entry per env (%d), not %d" % (offsets.numel() - 1, ids.numel()))
        self._check_fused()
        return _LinearLogProb.apply(h.to(self.weight.dtype), self.weight, self.bias, offsets, actions, ids, stats)


class HeadedPolicy(torch.nn.Module):
    """A fixed-head policy whose last layer is a LinearPolicyHead: forward(face) = head(trunk(face)), the dense logits.
    BatchedGame(policy_dict=...) and compete sample such a seat through head.sample(env, trunk(face)), without the dense
    logits; train it through head.log_prob(trunk(face), ...)."""

    def __init__(self, trunk, head):
        super().__init__()
        if not isinstance(head, LinearPolicyHead):
            raise TypeError("head must be a LinearPolicyHead, not %s" % type(head).__name__)
        self.trunk, self.head = trunk, head

    def forward(self, face):
        return self.head(self.trunk(face))
