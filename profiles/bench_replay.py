"""Packed replay (trainer.PackedReplayBuffer, ddz_encode_face_gather) against the float ring (trainer.ReplayBuffer):

  * bytes per transition of both, for C = 4 / 6 / 7 / 9, from the buffers' own tensors;
  * sample() time at batch 256 / 4 096 / 65 536 from a full buffer of --capacity transitions (EnvCooperation, C = 9): the
    float ring's index gather against the packed decode, which writes the same rows but reads 176 B a transition instead of
    4 808 B.  Both buffers are larger than the 126 MB L2 at the default capacity, and sampled rows are uniformly random, so
    the reads come from HBM.  Device time from CUDA events around --reps calls, median of --rounds, the two buffers
    alternating;
  * BatchedGame.step time with a learning landlord (QNetLike width = hidden = 64, farmers random, one TD step a decision,
    --step-capacity slots) at B = 16 384 and 131 072, float against packed: host clock around --steps decisions (step()
    synchronises), after --warmup decisions; and the largest capacity each mode fits in the device memory left free
    by that game (free bytes / bytes per transition).

The buffers are filled with the states and moves of real mid-game positions (128 steps of 4 096 random games).
Writes one JSON document (stdout, and --out)."""
import argparse
import functools
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ddz_b200 as D
from qnet_like import QNetLike

N = D.native


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:                     # noqa: BLE001 -- recorded, not fatal
        info["power_limit"] = "unknown (%s)" % e
    return info


def bytes_per_transition():
    out = {}
    for cls, C in (("BatchedEnv", 4), ("BatchedEnvCooperationSimplify", 6), ("BatchedEnvComplicated", 7),
                   ("BatchedEnvCooperation", 9)):
        v = getattr(D, cls).VARIANT
        rb, pb = D.ReplayBuffer(1024, C, "cuda"), D.PackedReplayBuffer(1024, v, "cuda")
        fb = sum(t.nbytes for t in (rb.s0, rb.a0, rb.r, rb.s1, rb.a1, rb.done)) / 1024
        pk = sum(t.nbytes for t in (pb.state, pb.moves, pb.r, pb.done)) / 1024
        assert pk == pb.bytes_per_transition
        out["C=%d" % C] = {"float": fb, "packed": pk, "ratio": round(fb / pk, 2)}
        del rb, pb
    return out


def source_transitions(B=4096, steps=128):
    """packed (state, move) pairs of real positions: every env after each of `steps` random decisions"""
    env = D.BatchedEnvCooperation(B, seed=5)
    perm, lord = D.random_deals(B, seed=5, pool_games=4)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env.prepare(pd, ld, pool_games=4)
    states, moves = [], []
    idx = torch.arange(B, device="cuda")
    for _ in range(steps):
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=4)
        off = env.offsets.to(torch.int64)
        au = env.actions_packed
        states.append(D.gather_states(env, idx))
        moves.append(au[off[:-1].clamp(max=au.numel() - 1)] * ((off[1:] - off[:-1]) > 0))
    return env, states, moves


def fill(cap, env, states, moves):
    """a float and a packed buffer holding the same `cap` transitions"""
    rb = D.ReplayBuffer(cap, env.C, "cuda")
    pb = D.PackedReplayBuffer(cap, env.VARIANT, "cuda")
    B, k, n = env.B, 0, 0
    while n < cap:
        s0, s1 = states[k % len(states)], states[(k + 1) % len(states)]
        a0, a1 = moves[k % len(moves)], moves[(k + 1) % len(moves)]
        r = torch.zeros(B, device="cuda")
        done = torch.zeros(B, device="cuda")
        pb.append(s0, a0, r, s1, a1, done)
        idx = torch.arange(B, device="cuda")
        f0, m0 = D.decode_rows(s0, env.VARIANT, idx, a0)
        f1, m1 = D.decode_rows(s1, env.VARIANT, idx, a1)
        rb.append(f0, m0, r, f1, m1, done)
        n += B
        k += 1
    return rb, pb


def time_sample(buf, batch, reps, gen):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        buf.sample(batch, gen)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / reps


def sample_times(rb, pb, batches, reps, rounds):
    out = {}
    g = torch.Generator(device="cuda")
    g.manual_seed(1)
    for bs in batches:
        for buf in (rb, pb):
            time_sample(buf, bs, 3, g)                 # warm-up: every shape of the timed window
        tf, tp = [], []
        for _ in range(rounds):
            tf.append(time_sample(rb, bs, reps, g))
            tp.append(time_sample(pb, bs, reps, g))
        f, p = float(np.median(tf)), float(np.median(tp))
        rows = 2 * bs * (rb.s0.shape[1] + 1) * 240 + 8 * bs       # bytes of the 6-tuple both return
        out[str(bs)] = {"float_ms": round(f, 4), "packed_ms": round(p, 4), "packed_over_float": round(p / f, 3),
                        "float_spread_ms": [round(min(tf), 4), round(max(tf), 4)],
                        "packed_spread_ms": [round(min(tp), 4), round(max(tp), 4)],
                        "bytes_returned": rows, "float_GBps_written": round(rows / f / 1e6, 1),
                        "packed_GBps_written": round(rows / p / 1e6, 1)}
        print(json.dumps({"sample": bs, **out[str(bs)]}), file=sys.stderr, flush=True)
    return out


def step_times(B, replay, capacity, warmup, steps):
    torch.manual_seed(0)
    net = lambda: QNetLike(9, width=64, hidden=64)
    dqn = functools.partial(D.BatchedDQN, replay_size=capacity)
    game = D.BatchedGame(D.BatchedEnvCooperation, {"lord": net, "down": None, "up": None}, {"lord": dqn, "down": None, "up": None},
                         train_dict={"lord": True, "down": False, "up": False}, seed=1, num_envs=B, replay=replay)
    for _ in range(warmup):
        game.step()
    torch.cuda.synchronize()
    n0 = len(game.lord.replay_buffer)
    t0 = time.perf_counter()
    for _ in range(steps):
        game.step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    added = len(game.lord.replay_buffer) - n0
    rb = game.lord.replay_buffer
    per = rb.bytes_per_transition if replay == "packed" else \
        sum(t.nbytes for t in (rb.s0, rb.a0, rb.r, rb.s1, rb.a1, rb.done)) / rb.capacity
    free, total = torch.cuda.mem_get_info()
    res = {"B": B, "replay": replay, "ms_per_step": round(dt * 1e3, 3), "transitions_per_step": round(added / steps, 1),
           "bytes_per_transition": per, "free_bytes_after_build": free,
           "largest_capacity_fits": int((free + rb.capacity * per) // per)}
    print(json.dumps(res), file=sys.stderr, flush=True)
    del game
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--capacity", type=int, default=1 << 20)
    ap.add_argument("--batches", default="256,4096,65536")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--step-envs", default="16384,131072")
    ap.add_argument("--step-capacity", type=int, default=1 << 20)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_replay.py measures on the GPU: no CUDA device")
    config = {k: v for k, v in vars(a).items() if k != "out"}       # where the document is written is not part of the run
    res = {"config": config, **gpu_info(), "bytes_per_transition": bytes_per_transition()}
    env, states, moves = source_transitions()
    rb, pb = fill(a.capacity, env, states, moves)
    g1, g2 = torch.Generator(device="cuda"), torch.Generator(device="cuda")
    g1.manual_seed(3)
    g2.manual_seed(3)
    same = all(torch.equal(x, y) for x, y in zip(rb.sample(4096, g1), pb.sample(4096, g2)))
    res["sample_outputs_bit_equal"] = same
    res["sample_ms"] = sample_times(rb, pb, [int(x) for x in a.batches.split(",")], a.reps, a.rounds)
    del rb, pb, states, moves, env
    torch.cuda.empty_cache()
    res["step"] = [step_times(int(B), replay, a.step_capacity, a.warmup, a.steps)
                   for B in a.step_envs.split(",") for replay in ("float", "packed")]
    out = json.dumps(res, indent=1)
    print(out)
    if a.out:
        with open(a.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
