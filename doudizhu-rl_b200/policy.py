"""Fixed-head policies over the action ids (include/ddz_b200.h: ddz_policy_sample, ddz_policy_logprob,
ddz_policy_logprob_backward).

A fixed-head policy maps a state to logits [B, 13551], one per action id (move_ids).  Its softmax is restricted to the
legal ids of each env, and these kernels read only those logits (mean 5.6, at most 512 per env): no dense mask, no
masked_fill, no full-size log_softmax or saved tensors.  Sampling at decision time, and log-probability + entropy with
their gradient at training time, each take one launch; the gradient row is written once, zero off the legal set.
"""
import torch

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
