"""Determinized search on the device (search.pimc_search: ddz_determinize -> ddz_uct_search over B x D roots ->
ddz_uct_pool): roots searched per second at B = 1, 512, 4096, D = 1, 8, 32 determinizations, budget 125 and 1000, width 1,
the bot's pruned lists; the time of each of the three launches on its own; and the landlord's win count over 2048 seeded
deals against random farmers, all on the same deals and the same farmer draws: a random landlord, pimc_search (D = 8 and
D = 32, budget 125) and the full-information uct_search (budget 1000), which sees the farmers' cards.

Roots: mid-game positions of real games (random deals, 12 Philox moves), so every view has a consistent set of unseen
cards.  Device time from CUDA events; every run fits one chunk (the workspace cap is raised to --max-workspace-gb), so a
run is one launch of each kernel.  Writes one JSON document (stdout, and --out)."""
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
from importlib import import_module

S = import_module("doudizhu-rl_b200.search")
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


def mid_game(B, seed=1):
    env = D.BatchedEnv(B, seed=seed)
    env.prepare(*D.random_deals(B, seed=seed))
    for _ in range(12):
        env.step_random()
    return env


def events(n):
    return [torch.cuda.Event(enable_timing=True) for _ in range(n)]


def stage_times(env, Dn, budget, seed):
    """seconds of ddz_determinize, ddz_uct_search (B x D roots) and ddz_uct_pool, each launch between two events"""
    B, dev = env.B, env.device
    s = torch.cuda.current_stream(dev).cuda_stream
    ws = S._workspace(N.lib.ddz_uct_workspace_bytes(B * Dn, budget), dev, s)
    ln = S._ln_table(budget, dev)
    sub = torch.empty(N.lib.ddz_state_bytes(B * Dn) // 4, dtype=torch.int32, device=dev)
    tc = torch.empty(B * Dn, dtype=torch.int32, device=dev)
    choice = torch.empty(B, dtype=torch.int32, device=dev)
    moves = torch.empty(B, dtype=torch.int64, device=dev)
    e = events(4)
    torch.cuda.synchronize()
    e[0].record()
    N.check(N.lib.ddz_determinize(env._state.data_ptr(), None, Dn, seed, env.env0, sub.data_ptr(), None, B, s), "det")
    e[1].record()
    N.check(N.lib.ddz_uct_search(sub.data_ptr(), None, ws.data_ptr(), budget, 1, 1, S.UCB_C, ln.data_ptr(), seed,
                                 env.env0 * Dn, tc.data_ptr(), None, None, None, None, None, 0, B * Dn, s), "uct")
    e[2].record()
    N.check(N.lib.ddz_uct_pool(ws.data_ptr(), budget, Dn, choice.data_ptr(), moves.data_ptr(), None, None, B, s), "pool")
    e[3].record()
    torch.cuda.synchronize()
    return [e[i].elapsed_time(e[i + 1]) / 1e3 for i in range(3)], choice


def lord_wins(B, search, seed=21):
    """games on B seeded deals, random farmers (one numpy stream shared by every arm), the landlord random or searched"""
    env = D.BatchedEnv(B, seed=4)
    env.prepare(*D.random_deals(B, seed=seed))
    rng = np.random.default_rng(7)
    for t in range(300):
        meta = env._fields()[1]
        done = ((meta >> 2) & 1).bool()
        if bool(done.all()):
            break
        env.observe()
        n = (env.offsets[1:] - env.offsets[:-1]).cpu().numpy()
        ch = (rng.integers(0, 1 << 30, B) % np.maximum(n, 1)).astype(np.int32)
        lord_turn = ((meta & 3) == 1) & ~done
        if search is not None and bool(lord_turn.any()):
            c = search(env, t, lord_turn).cpu().numpy()
            ch = np.where(lord_turn.cpu().numpy(), c, ch).astype(np.int32)
        env.step(ch)
    meta = env._fields()[1].cpu().numpy()
    assert ((meta >> 2) & 1).all() and int(env.stats[7].item()) == 0
    return int((((meta >> 3) & 3) == 1).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="1,512,4096")
    ap.add_argument("--determinizations", default="1,8,32")
    ap.add_argument("--budgets", default="125,1000")
    ap.add_argument("--games", type=int, default=2048)
    ap.add_argument("--max-workspace-gb", type=float, default=32.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pimc.py needs a CUDA device")
    batches = [int(x) for x in a.batches.split(",")]
    dets = [int(x) for x in a.determinizations.split(",")]
    budgets = [int(x) for x in a.budgets.split(",")]
    cap = int(a.max_workspace_gb * 2 ** 30)
    dev = torch.device("cuda:0")
    res = {"workload": "determinized UCT search (pimc_search), width 1, pruned lists", **gpu_info(), "runs": []}
    res["library"] = os.path.basename(N.LIB_PATH)
    big = max(batches) * max(dets)
    S._workspace(N.lib.ddz_uct_workspace_bytes(big, max(budgets)), dev, torch.cuda.current_stream(dev).cuda_stream)
    pool = mid_game(max(batches))
    warm = mid_game(8, seed=2)
    D.pimc_search(warm, determinizations=2, computation_budget=4, max_workspace_bytes=cap)
    for budget in budgets:
        for B in batches:
            env = mid_game(B) if B != max(batches) else pool
            live = int((~env.is_done).sum().item())
            for Dn in dets:
                if B * Dn * (budget + 1) * N.UCT_NODE_BYTES > cap:
                    res["runs"].append({"B": B, "D": Dn, "budget": budget, "not_measured": "over --max-workspace-gb"})
                    continue
                e = events(2)
                torch.cuda.synchronize()
                e[0].record()
                choice, _ = D.pimc_search(env, determinizations=Dn, computation_budget=budget, seed=9,
                                          max_workspace_bytes=cap)
                e[1].record()
                torch.cuda.synchronize()
                sec = e[0].elapsed_time(e[1]) / 1e3
                (t_det, t_uct, t_pool), c2 = stage_times(env, Dn, budget, 9)
                run = {"B": B, "D": Dn, "budget": budget, "live_roots": live, "seconds": sec, "roots_per_s": live / sec,
                       "trees_per_s": live * Dn / sec, "determinize_s": t_det, "search_s": t_uct, "pool_s": t_pool,
                       "stages_equal_pimc_search": bool(torch.equal(choice, c2))}
                res["runs"].append(run)
                print(json.dumps(run), file=sys.stderr, flush=True)
    G = a.games
    arms = [("random landlord", None),
            ("pimc_search D=8 budget 125", lambda env, t, m: D.pimc_search(env, determinizations=8, computation_budget=125,
                                                                            seed=t + 1, env_mask=m)[0]),
            ("pimc_search D=32 budget 125", lambda env, t, m: D.pimc_search(env, determinizations=32, computation_budget=125,
                                                                             seed=t + 1, env_mask=m)[0]),
            ("uct_search budget 1000 (full information)",
             lambda env, t, m: D.uct_search(env, computation_budget=1000, seed=t + 1, env_mask=m)[0])]
    res["games"] = {"deals": G, "farmers": "uniformly random legal moves", "landlord_wins": {}}
    for name, fn in arms:
        res["games"]["landlord_wins"][name] = lord_wins(G, fn)
        print(name, res["games"]["landlord_wins"][name], file=sys.stderr, flush=True)
    out = json.dumps(res, indent=1)
    print(out)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(out + "\n")
    if not all(r.get("stages_equal_pimc_search", True) for r in res["runs"]):
        raise SystemExit("the staged launches differ from pimc_search")


if __name__ == "__main__":
    main()
