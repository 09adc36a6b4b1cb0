"""Linear policy head evaluated at the legal ids (LinearPolicyHead) against the best dense path a user has today, at
B = 4 096 and 131 072 envs on mid-game lists (EnvCooperation, 24 random steps from seeded deals), hidden width H = 256,
float32 and bfloat16 (hidden, weight and bias in one dtype):

  * sample: dense = nn.Linear(H, 13551) (cuBLAS) + D.policy_sample;  fused = LinearPolicyHead.sample (one launch);
  * train:  forward + backward of -(adv * log p(chosen)).sum() - 0.01 * H.sum(), with the gradients of h, W and bias;
            dense = nn.Linear + D.policy_log_prob;  fused = LinearPolicyHead.log_prob.

Both arms hold the same parameters and hidden vectors, made outside the timed window.  Device time from CUDA events
around --reps calls, median of --rounds; peak memory = torch.cuda.max_memory_allocated above what was allocated before the
call, after reset_peak_memory_stats.  Also recorded: how many argmax ids (T = 0) and how close the log-probabilities of the
two arms are (their logits differ by the rounding of the two dot products).  Writes one JSON document (stdout, and --out)."""
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
        fn()                                                      # warm-up: libraries pick their algorithms
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
        return {"ms": float(np.median(out)), "ms_rounds": [round(x, 4) for x in out], "peak_extra_bytes": int(peak)}
    except torch.OutOfMemoryError as e:
        torch.cuda.empty_cache()
        return {"ms": None, "does_not_fit": str(e).splitlines()[0]}


def bench(B, H, dtype, reps, rounds):
    env = D.BatchedEnvCooperation(B, seed=7)
    env.prepare(*D.random_deals(B, seed=8))
    for _ in range(24):
        env.step_random()
    off, act = env.offsets, env.actions_packed
    torch.manual_seed(1)
    dense = torch.nn.Linear(H, NIDS, device="cuda", dtype=dtype)
    fused = D.LinearPolicyHead.from_linear(dense)
    gen = torch.Generator(device="cuda").manual_seed(2)
    h = torch.randn((B, H), device="cuda", generator=gen).to(dtype)
    adv = torch.randn(B, device="cuda", generator=gen)
    ids = fused.sample(env, h, seed=3)[1]
    res = {"B": B, "H": H, "dtype": str(dtype).replace("torch.", ""), "legal_moves": int(env.num_actions),
           "dense_logits_bytes": B * NIDS * h.element_size()}

    def dense_sample():
        with torch.no_grad():
            return D.policy_sample(env, dense(h), 1.0, seed=3)

    def fused_sample():
        return fused.sample(env, h, 1.0, seed=3)

    def train(model, logp_fn):
        def step():
            for p in model.parameters():
                p.grad = None
            x = h.detach().requires_grad_(True)
            lp, ent = logp_fn(x)
            (-(adv * lp).sum() - 0.01 * ent.sum()).backward()
            return x.grad
        return step

    dense_train = train(dense, lambda x: D.policy_log_prob(dense(x), off, act, ids))
    fused_train = train(fused, lambda x: fused.log_prob(x, off, act, ids))
    for name, fn in (("fused_sample", fused_sample), ("dense_sample", dense_sample), ("fused_train", fused_train),
                     ("dense_train", dense_train)):
        res[name] = measure(fn, reps, rounds)
        print(json.dumps({"B": B, "dtype": res["dtype"], name: res[name]}), file=sys.stderr, flush=True)
    # agreement of the two arms: argmax ids, and log-probabilities of the same ids
    with torch.no_grad():
        a0 = D.policy_sample(env, dense(h), 0.0)[1]
        b0 = fused.sample(env, h, 0.0)[1]
        la = D.policy_log_prob(dense(h), off, act, ids)[0]
        lb = fused.log_prob(h, off, act, ids)[0]
    live = ids >= 0
    res["argmax_ids_equal"] = "%d of %d" % (int((a0 == b0).sum().item()), B)
    res["max_abs_logp_difference"] = float((la[live] - lb[live]).abs().max().item())
    assert int(env.stats[7].item()) == 0
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="4096,131072")
    ap.add_argument("--hidden", type=int, default=256)
    ap.add_argument("--dtypes", default="float32,bfloat16")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"config": {"envs": args.envs, "hidden": args.hidden, "dtypes": args.dtypes, "reps": args.reps,
                      "rounds": args.rounds, "positions": "EnvCooperation, 24 random steps from random_deals(seed=8)",
                      "float32_matmul_precision": torch.get_float32_matmul_precision()},
           "device": gpu_info(),
           "runs": [bench(int(b), args.hidden, getattr(torch, dt), args.reps, args.rounds)
                    for dt in args.dtypes.split(",") for b in args.envs.split(",")]}
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
