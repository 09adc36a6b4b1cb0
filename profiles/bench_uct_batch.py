"""Batched UCT search on the device (search.uct_search / ddz_uct_search): roots searched per second at B = 1, 512, 4096 and
32 768, budget 1000 (the reference's, server/mcts/interface.py:37), playout widths 1 / 16 / 256, the bot's pruned lists and
the full lists -- against the host-tree UctSearch (mcts(payload), the timings of bench_mcts.py) measured in the same run.

Roots: env b is the mid-game position of bench_mcts.py when b % 4 == 0, its opening when b % 4 == 1, and otherwise a
position from a seeded random rollout (12 Philox moves from a random deal).  Device time from CUDA events around the one
launch.  Runs whose playout count (B x budget x width) exceeds --max-playouts are not run and are listed as not measured.
The largest timed run at width 1 is checked against the C port over the oracle (tests/host_harness/uct_oracle.c) on 64 of
its roots.  Writes one JSON document (stdout, and --out)."""
import argparse
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
from importlib import import_module

S = import_module("doudizhu-rl_b200.search")


def bench_payloads():
    """the two positions of bench_mcts.py"""
    rng = np.random.default_rng(3)
    deck = [min(i // 4 + 3, 15) if i < 52 else 16 + (i - 52) for i in range(54)]
    cards = [int(c) for c in rng.permutation(deck)[:31]]
    mid = {"role_id": 1, "hand_card": {0: sorted(cards[:10]), 1: sorted(cards[10:22]), 2: sorted(cards[22:31])},
           "last_taken": {0: [], 1: [], 2: []}}
    cards = [int(c) for c in rng.permutation(deck)]
    opening = {"role_id": 1, "hand_card": {0: sorted(cards[:17]), 1: sorted(cards[17:37]), 2: sorted(cards[37:54])},
               "last_taken": {0: [], 1: [], 2: []}}
    return [("mid-game 10/12/9 cards", mid), ("opening 17/20/17 cards", opening)]


def counts(cards):
    c = np.zeros(15, np.int64)
    for v in cards:
        c[int(v) - 3] += 1
    return c


def roots(B, seed=1):
    """(hands [B,3,15], recent [B,3,15], role [B]) of the mixed batch described above"""
    env = D.BatchedEnv(B, seed=seed)
    perm, lord = D.random_deals(B, seed=seed)
    env.prepare(perm, lord)
    for _ in range(12):
        env.step_random()
    f, meta = env._fields()
    u = D.unpack_counts(f.t().contiguous()).cpu().numpy()
    hands, recent, role = u[:, 0:3].astype(np.int64), u[:, 6:9].astype(np.int64), (meta.cpu().numpy() & 3).astype(np.int64)
    done = ((meta.cpu().numpy() >> 2) & 1).astype(bool)
    for k, (_, p) in enumerate(bench_payloads()):
        sel = np.arange(k, B, 4)
        hands[sel] = np.stack([counts(p["hand_card"][q]) for q in range(3)])
        recent[sel] = 0
        role[sel] = p["role_id"]
        done[sel] = False
    return hands, recent, role, done


def make_env(hands, recent, role, done):
    B = len(role)
    env = D.env_from_arrays(role, hands[np.arange(B), role], np.zeros((B, 3, 15), np.int64), recent, hands.sum(2),
                            env_cls=D.BatchedEnv, hands=hands)
    meta = env._fields()[1]
    meta.copy_(meta | torch.as_tensor(done.astype(np.int32) << 2, device=env.device))
    return env


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:                     # noqa: BLE001 -- recorded, not fatal
        info["power_limit"] = "unknown (%s)" % e
    return info


def uct_search_timings():
    """mcts(payload) with the host tree (UctSearch), as bench_mcts.py runs it"""
    out = []
    pl = bench_payloads()
    D.mcts(pl[0][1], computation_budget=50)
    D.mcts(pl[0][1], computation_budget=50, prune=False)
    for name, p in pl:
        for prune in (True, False):
            for width in (1, 16, 256):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                D.mcts(p, computation_budget=1000, width=width, seed=5, prune=prune)
                torch.cuda.synchronize()
                out.append({"position": name, "pruned_lists": prune, "width": width, "seconds": time.perf_counter() - t0})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--budget", type=int, default=1000)
    ap.add_argument("--batches", default="1,512,4096,32768")
    ap.add_argument("--widths", default="1,16,256")
    ap.add_argument("--max-playouts", type=float, default=2 ** 28)
    ap.add_argument("--check-roots", type=int, default=64)
    ap.add_argument("--lists", default="pruned,full", help="which move lists to search: pruned, full or both")
    ap.add_argument("--skip-host-tree", action="store_true", help="do not time UctSearch (no speed-up column)")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_uct_batch.py needs a CUDA device")
    batches = [int(x) for x in a.batches.split(",")]
    widths = [int(x) for x in a.widths.split(",")]
    budget = a.budget
    dev = torch.device("cuda:0")
    res = {"workload": "batched UCT search, budget %d" % budget, **gpu_info(), "runs": [], "not_measured": []}
    res["library"] = os.path.basename(D.native.LIB_PATH)
    res["uct_search_host_tree"] = [] if a.skip_host_tree else uct_search_timings()
    ws = torch.empty(D.native.lib.ddz_uct_workspace_bytes(max(batches), budget), dtype=torch.uint8, device=dev)   # untimed
    S._ln_table(budget * max(widths), dev)
    pos = roots(max(batches))
    warm = make_env(*(x[:8] for x in pos))
    largest = None
    for prune in [{"pruned": True, "full": False}[x] for x in a.lists.split(",")]:
        for width in widths:
            D.uct_search(warm, computation_budget=4, width=width, prune=prune, workspace=ws)
            for B in batches:
                if B * budget * width > a.max_playouts:
                    res["not_measured"].append({"B": B, "width": width, "pruned_lists": prune,
                                                "reason": "B x budget x width over --max-playouts"})
                    continue
                env = make_env(*(x[:B] for x in pos))
                live = int((~pos[3][:B]).sum())
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                s0.record()
                choice, moves = D.uct_search(env, computation_budget=budget, width=width, prune=prune, seed=7, workspace=ws)
                s1.record()
                torch.cuda.synchronize()
                sec = s0.elapsed_time(s1) / 1e3
                run = {"B": B, "live_roots": live, "width": width, "pruned_lists": prune, "seconds": sec,
                       "roots_per_s": live / sec, "playouts_per_s": live * budget * width / sec}
                res["runs"].append(run)
                print(json.dumps(run), file=sys.stderr, flush=True)
                if width == 1 and prune and (largest is None or B > largest[0]):
                    largest = (B, choice.cpu().numpy(), moves.cpu().numpy().view(np.uint64))
    # the host-tree rate at the reference configuration (pruned lists, width 1): the mean over the two positions
    host = [r["seconds"] for r in res["uct_search_host_tree"] if r["pruned_lists"] and r["width"] == 1]
    if host:
        host_rate = len(host) / sum(host)
        res["host_tree_roots_per_s_pruned_width1"] = host_rate
        for r in res["runs"]:
            if r["pruned_lists"] and r["width"] == 1:
                r["speedup_vs_host_tree"] = r["roots_per_s"] / host_rate
    if largest is not None:
        from uct_philox_reference import ref_uct_batch
        B, choice, moves = largest
        b0 = max(0, B // 2 - a.check_roots // 2)
        b1 = min(B, b0 + a.check_roots)
        ref = ref_uct_batch(pos[0][b0:b1], pos[1][b0:b1], pos[2][b0:b1], ~pos[3][b0:b1], budget, width=1, prune=True,
                            seed=7, env0=b0)
        ok = bool(np.array_equal(ref["choice"], choice[b0:b1]) and np.array_equal(ref["move"], moves[b0:b1]))
        res["oracle_check"] = {"run_B": B, "roots": [b0, b1], "equal": ok}
    out = json.dumps(res, indent=1)
    print(out)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(out + "\n")
    if largest is not None and not res["oracle_check"]["equal"]:
        raise SystemExit("the device search differs from the oracle port")


if __name__ == "__main__":
    main()
