"""Fixed-head policy over the action ids: the fused path (ddz_policy_sample, ddz_policy_logprob + backward) against the
dense torch path a user writes today, at B = 4 096 and 131 072 envs on mid-game lists (EnvCooperation, 24 random steps
from seeded deals), fp32 logits [B, 13551]:

  * sample: dense = legal_mask("bool") + masked_fill(-inf) + log_softmax + multinomial + gather of the chosen log-prob;
            fused = D.policy_sample (one launch);
  * train:  forward + backward of the loss -(g * log p(chosen)).sum() - 0.01 * H.sum();
            dense = legal_mask + masked_fill + log_softmax + gather + entropy, torch autograd;
            fused = D.policy_log_prob (one launch each way).

The logits themselves are made outside the timed window (the network's cost is the same on both paths).  Device time from
CUDA events around --reps calls, median of --rounds; peak memory = torch.cuda.max_memory_allocated above what was
allocated before the call (the logits, lists and env), after reset_peak_memory_stats.  A dense path that does not fit in
memory is recorded as such.  Writes one JSON document (stdout, and --out)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ddz_b200 as D

NIDS = 13551


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:                     # noqa: BLE001 -- recorded, not fatal
        info["power_limit"] = "unknown (%s)" % e
    return info


def measure(fn, reps, rounds):
    """(median ms of one fn() call, peak bytes above the allocation before it) or the out-of-memory error"""
    try:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        fn()
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        out = []
        for _ in range(rounds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                fn()
            b.record()
            b.synchronize()
            out.append(a.elapsed_time(b) / reps)
        return {"ms": float(np.median(out)), "peak_extra_bytes": int(peak)}
    except torch.OutOfMemoryError as e:
        torch.cuda.empty_cache()
        return {"ms": None, "does_not_fit": str(e).splitlines()[0]}


def bench(B, reps, rounds):
    env = D.BatchedEnvCooperation(B, seed=7)
    env.prepare(*D.random_deals(B, seed=8))
    for _ in range(24):
        env.step_random()
    off, act = env.offsets, env.actions_packed
    gen = torch.Generator(device="cuda").manual_seed(1)
    logits = torch.randn((B, NIDS), device="cuda", generator=gen)
    g = torch.randn(B, device="cuda", generator=gen)
    ids = D.policy_sample(env, logits)[1]
    res = {"B": B, "legal_moves": int(env.num_actions), "logits_bytes": logits.numel() * 4}

    def dense_sample():
        mask = env.legal_mask("bool")
        lp = torch.log_softmax(logits.masked_fill(~mask, float("-inf")), 1)
        live = mask.any(1)                                        # finished envs: a dummy row, as a user must
        pick = torch.multinomial(torch.where(live[:, None], lp.exp(), torch.ones((), device="cuda")), 1)
        return pick[:, 0], lp.gather(1, pick)[:, 0]

    def fused_sample():
        return D.policy_sample(env, logits, 1.0, seed=3)

    def dense_train():
        x = logits.detach().requires_grad_(True)
        mask = env.legal_mask("bool")
        lp = torch.log_softmax(x.masked_fill(~mask, float("-inf")), 1)
        live = mask.any(1)
        chosen = torch.where(live, lp.gather(1, ids.clamp(min=0).to(torch.int64)[:, None])[:, 0], 0.0)
        ent = -torch.where(mask, lp.exp() * lp, torch.zeros((), device="cuda")).sum(1)
        ent = torch.where(live, ent, 0.0)
        (-(g * chosen).sum() - 0.01 * ent.sum()).backward()
        return x.grad

    def fused_train():
        x = logits.detach().requires_grad_(True)
        lp, ent = D.policy_log_prob(x, off, act, ids)
        (-(g * lp).sum() - 0.01 * ent.sum()).backward()
        return x.grad

    for name, fn in (("fused_sample", fused_sample), ("dense_sample", dense_sample), ("fused_train", fused_train),
                     ("dense_train", dense_train)):
        res[name] = measure(fn, reps, rounds)
        print(json.dumps({"B": B, name: res[name]}), file=sys.stderr, flush=True)
    assert int(env.stats[7].item()) == 0
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="4096,131072")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"config": {"envs": args.envs, "reps": args.reps, "rounds": args.rounds, "logits": "float32 [B, 13551]",
                      "positions": "EnvCooperation, 24 random steps from random_deals(seed=8)"},
           "device": gpu_info(), "runs": [bench(int(b), args.reps, args.rounds) for b in args.envs.split(",")]}
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
