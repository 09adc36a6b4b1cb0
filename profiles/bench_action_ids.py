"""Action ids (ddz_move_ids, ddz_legal_mask, BatchedEnv.step_ids):

  * ddz_move_ids over the lists of one config-5 call (ddz_legal_moves on 131 072 adversarial (hand, last) pairs, about
    18 M moves: 144 MB read, 72 MB written, more than the 126 MB L2);
  * ddz_legal_mask at B = 4 096 and 131 072 in both layouts (bits: 1 696 B a row, bytes: 13 551 B a row) over the lists of
    mid-game positions (EnvCooperation, 24 random steps from seeded deals);
  * a decision at 131 072 envs played by id (moves_of_ids + the DDZ_CHOICE_MOVE step) against the same decision played by
    list index (ddz_step with DDZ_CHOICE_INDEX), on two envs in the same state, alternating.

Device time from CUDA events around --reps launches, median of --rounds.  Writes one JSON document (stdout, and --out)."""
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


def timed(fn, reps, rounds):
    """median over rounds of the mean device time (ms) of one fn() call, CUDA events around reps calls"""
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / reps)
    return float(np.median(out))


def stream():
    return torch.cuda.current_stream().cuda_stream


def bench_move_ids(pairs, reps, rounds):
    hands, lasts = D.adversarial_pairs(pairs, seed=5)
    h = torch.as_tensor(hands.view(np.int64), device="cuda")
    l = torch.as_tensor(lasts.view(np.int64), device="cuda")
    ws = torch.zeros(max(1, N.lib.ddz_workspace_bytes(pairs) // 4), dtype=torch.int32, device="cuda")
    off = torch.zeros(pairs + 1, dtype=torch.int32, device="cuda")
    cap = pairs * N.MAX_LEGAL
    moves = torch.zeros(cap, dtype=torch.int64, device="cuda")
    N.check(N.lib.ddz_legal_moves(h.data_ptr(), l.data_ptr(), ws.data_ptr(), off.data_ptr(), moves.data_ptr(), cap, None,
                                  pairs, stream()), "ddz_legal_moves")
    n = int(off[pairs].item())
    ids = torch.empty(n, dtype=torch.int32, device="cuda")
    ms = timed(lambda: N.check(N.lib.ddz_move_ids(moves.data_ptr(), n, ids.data_ptr(), stream()), "ddz_move_ids"), reps, rounds)
    assert int((ids < 0).sum().item()) == 0
    return {"pairs": pairs, "moves": n, "ms": ms, "moves_per_s": n / ms * 1e3, "GB_per_s": n * 12 / ms / 1e6}


def midgame_env(B, steps=24):
    env = D.BatchedEnvCooperation(B, seed=7)
    env.prepare(*D.random_deals(B, seed=3))
    for _ in range(steps):
        env.step_random()
    env.num_actions
    return env


def bench_mask(B, reps, rounds):
    env = midgame_env(B)
    res = {"B": B, "moves": env.num_actions}
    for name, lay, shape, dt in (("bits", N.MASK_BITS, (B, N.MASK_WORDS), torch.int32),
                                 ("bool", N.MASK_BYTES, (B, N.NUM_ACTION_IDS), torch.bool)):
        out = torch.empty(shape, dtype=dt, device="cuda")
        off, acts = env.offsets, env._actions_u64[env._cur]

        def run():
            N.check(N.lib.ddz_legal_mask(off.data_ptr(), acts.data_ptr(), env.cap, lay, out.data_ptr(), None, B, stream()),
                    "ddz_legal_mask")
        ms = timed(run, reps, rounds)
        nbytes = out.numel() * out.element_size()
        res[name] = {"ms": ms, "bytes_stored": nbytes, "GB_per_s_stored": nbytes / ms / 1e6}
    return res


def bench_step(B, reps, rounds):
    """one decision by id against one by index; both envs are restored to the same state before every call, and that
    copy is timed on its own and subtracted"""
    a = midgame_env(B)
    state0 = a._state.clone()
    off = a.offsets.cpu().numpy()
    cnt = np.diff(off)
    choice = np.zeros(B, np.int32)
    ids = a.legal_ids().cpu().numpy()
    pick = np.where(cnt > 0, ids[np.minimum(off[:-1], len(ids) - 1)], 0).astype(np.int32)
    choice_d = torch.as_tensor(choice, device="cuda")
    pick_d = torch.as_tensor(pick, device="cuda")
    off_d, acts = a.offsets, a._actions_u64[a._cur]
    moves = torch.empty(B, dtype=torch.int64, device="cuda")
    rw = a._rewards.data_ptr()

    def restore():
        a._state.copy_(state0)

    def by_index():
        restore()
        N.check(N.lib.ddz_step(a._state.data_ptr(), off_d.data_ptr(), acts.data_ptr(), choice_d.data_ptr(), N.CHOICE_INDEX,
                               0, 0, 0, rw, None, None, None, None, None, B, stream()), "ddz_step")

    def by_id():
        restore()
        N.check(N.lib.ddz_moves_of_ids(pick_d.data_ptr(), B, moves.data_ptr(), stream()), "ddz_moves_of_ids")
        N.check(N.lib.ddz_step(a._state.data_ptr(), off_d.data_ptr(), acts.data_ptr(), moves.data_ptr(), N.CHOICE_MOVE,
                               0, 0, 0, rw, None, None, None, None, None, B, stream()), "ddz_step")
    res = {"B": B}
    copy_ms, idx, ids_ms = [], [], []
    for _ in range(rounds):      # alternate the two paths
        copy_ms.append(timed(restore, reps, 1))
        idx.append(timed(by_index, reps, 1))
        ids_ms.append(timed(by_id, reps, 1))
    c = float(np.median(copy_ms))
    res["state_copy_ms"] = c
    res["step_index_ms"] = float(np.median(idx)) - c
    res["step_ids_ms"] = float(np.median(ids_ms)) - c
    by_index()
    s_idx = a._state.clone()
    by_id()
    assert torch.equal(s_idx, a._state), "the two paths must play the same moves"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=131072)
    ap.add_argument("--mask-envs", default="4096,131072")
    ap.add_argument("--step-envs", type=int, default=131072)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a GPU"
    res = {"bench": "action ids (ddz_move_ids / ddz_legal_mask / step_ids)", "device": gpu_info(),
           "config": {k: v for k, v in vars(args).items() if k != "out"}}
    res["move_ids"] = bench_move_ids(args.pairs, args.reps, args.rounds)
    print(json.dumps(res["move_ids"]), file=sys.stderr, flush=True)
    res["legal_mask"] = [bench_mask(int(b), args.reps, args.rounds) for b in args.mask_envs.split(",")]
    print(json.dumps(res["legal_mask"]), file=sys.stderr, flush=True)
    res["step"] = bench_step(args.step_envs, args.reps, args.rounds)
    out = json.dumps(res, indent=1)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(out + "\n")


if __name__ == "__main__":
    main()
