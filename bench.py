#!/usr/bin/env python
"""bench.py -- the batched Doudizhu env on B200: env-steps/sec (legal moves + state/action encode + step + re-deal).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 4|5|3]

--config 4 (default; BASELINE.json configs[3], the config the metric is quoted on): 131 072 envs per GPU (weak scaling),
    EnvCooperation face (C=9, reference train.py:4-5), every seat plays a uniformly random legal move from the Philox
    index stream (config 2's lord-vs-random policy), synthetic random deals.  One "step" = one fused env-step of every env
    of the rank's slice (ddz_rollout_step: apply the chosen move, re-deal finished envs, generate the legal moves of the
    new state, write face [B,9,15,4] and the action one-hots).  A step writes ~0.5 GB, more than the 126 MB L2: no flush
    between iterations is needed.
--config 2 (configs[1]): the same rollout with 4096 envs in one chain of launches (latency-bound; its parity test is
    tests/test_gpu_parity.py::test_fused_rollout_bit_exact).
--config 5 (configs[4]): legal-move microbench, 131 072 adversarial (hand, last) pairs per GPU (SURVEY.md 8d C5), one
    "step" = one ddz_legal_moves call over all pairs; value = legal moves/s.
--config 3 (configs[2]): 65 536 envs, the landlord = argmax Q over its legal moves with a NetCooperation-shaped 256-wide
    torch network (the reference's consumer, net.py:125-139 / dqn.py:63-71 -- not part of the hot path), farmers random;
    reports how a step splits between the env kernels and the network.  Single GPU.

--impl reference times the CPU restatement of the reference env (oracle/, kind "port": the reference's own native
modules are not shipped, DESIGN.md) on all host cores over a bounded sample of the same workload.  That arm never loads
the product package or its library.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned to its caller as DIR/<name>.npy
(float32, or float64 where an integer needs it): for a fixed seeded sample of the envs (config 5: pairs) the step
results r / done / cat / reward, the face and the legal moves of the new state (one-hot rows and count per env; config 3
also the Q-values of the scored lists with their counts, and the chosen move index of the step; config 5 the move lists
as per-rank card counts).  Lists are written whole: the sample ends before the first env whose lists would pass the row
limit, and env_index (pair_index) lists the envs written.  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.  Under torchrun every rank writes its own share of the sample with a
_rank<r> suffix; all ranks together stay within 64 MB.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec (legal moves + state encode)"
UNIT = "env-steps/s"
VARIANT, CHANNELS = 2, 9            # EnvCooperation
STATE_BYTES = 76                    # 9 x uint64 + uint32 per env (include/ddz_b200.h)
POOL_GAMES = 8
SEED = 20260101
# the reference's own Python wrapper (unmodified envi.EnvCooperation: face + valid_actions + step_random per decision) over
# the oracle-backed natives, one core, measured in the build container where /root/reference exists
# (profiles/time_reference_envi.py -> profiles/r1n_reference_envi_python_timing.json); it cannot run on the GPU box
REFERENCE_PYTHON_ENVI = {"value": 1.96e3, "unit": UNIT, "cores": 1, "kind": "reference-python-over-port",
                         "where": "build container (the reference tree does not travel to the GPU box)",
                         "source": "profiles/r1n_reference_envi_python_timing.json"}


def load_deals():
    """doudizhu-rl_b200/deals.py by path: numpy only, shared by both arms (importing the package loads the library)"""
    spec = importlib.util.spec_from_file_location("ddz_deals", os.path.join(ROOT, "doudizhu-rl_b200", "deals.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=4, choices=[2, 3, 4, 5], help="BASELINE.json config number (1-based)")
    ap.add_argument("--envs", type=int, default=None, help="envs (config 5: pairs) per GPU; default 131072 (config 3: 65536)")
    ap.add_argument("--prefill", type=int, default=150, help="untimed env-steps that bring the games to their steady-state mix")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--groups", type=int, default=None, help="stream-parallel env groups per GPU (default 4; config 2: 1 = one chain of launches)")
    ap.add_argument("--steps-per-graph", type=int, default=2, help="env-steps captured in one CUDA graph per env group (even)")
    ap.add_argument("--no-single", action="store_true", help="skip the single-chain information run")
    ap.add_argument("--no-verify", action="store_true", help="skip the post-run check of a 512-env sample against the oracle")
    ap.add_argument("--stats-every", type=int, default=64, help="env-steps between two statistics all-reduces (multi-GPU)")
    ap.add_argument("--clock-interval-ms", type=int, default=20, help="nvidia-smi polling interval of the clock sampler (0 = off)")
    ap.add_argument("--net-precision", default="fp32", choices=["fp32", "tf32", "bf16"], help="config 3: the consumer network")
    ap.add_argument("--scoring", default="fused", choices=["fused", "module"],
                    help="config 3: how the landlord's legal moves are scored -- fused: ddz_q_features (the network's first layer "
                         "from the packed state and lists, no input tensor) + two library GEMMs; module: the torch module on the "
                         "[n, C+1, 15, 4] input written by ddz_encode_state_actions")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (a fixed sample, at most 64 MB) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    if args.envs is None:
        args.envs = {2: 4096, 3: 65536}.get(args.config, 131072)
    if args.groups is None:
        args.groups = 1 if args.config == 2 else 4
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def ncu_traffic(key):
    """DRAM bytes per step from the committed steady-state measurement (profiles/r2_traffic.json), or None"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        return d[key]["traffic_bytes_per_step"]
    except Exception:
        return None


def bytes_per_env_step(nbar, C=CHANNELS):
    """ALGORITHMIC bytes of one env-step = one env's share of one k_env launch (DESIGN.md): state read + write,
    previous offsets (2 x 4) and chosen move (8) read, r/done/cat/reward (15) written, new offset (4), packed list
    (8 N) and one-hot rows (240 N) written, face (240 C) written.  Deck permutations of re-dealt envs (55 B x ~1.6 %)
    and the look-back words are not counted."""
    return 2 * STATE_BYTES + 8 + 8 + 15 + 4 + 240 * C + 248 * nbar


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, interval_ms=20):
        self.gpu, self.proc, self.lines, self.interval = gpu_index, None, [], int(interval_ms)

    def start(self):
        if self.interval <= 0:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", str(self.interval)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(names, f[4:8]):
                if val == "Active":
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------- CPU arm
def workload_text(args):
    if args.config == 5:
        return ("BASELINE config 5: legal-move generation on adversarial hands, %d (hand, last) pairs per GPU from the "
                "committed pool (497-move hand, 5-trio airplanes, bombs + rocket, 12-straights + pairs), 50 %% lead / 50 %% "
                "follow a legal lead move; one step = r.get_moves for every pair (packed CSR lists)" % args.envs)
    if args.config == 3:
        return ("BASELINE config 3: %d envs on 1 GPU, landlord = argmax Q over its legal moves (NetCooperation-shaped 256-wide "
                "torch network, random-init), farmers uniform random; EnvCooperation face C=9" % args.envs)
    if args.config == 2:
        return ("BASELINE config 2: %d batched envs on 1 GPU, lord-vs-random rollout (all seats uniform random legal move, Philox "
                "stream), EnvCooperation face C=9, fused step+redeal+legal+encode -- the latency-bound regime (less than one warp "
                "per SM)" % args.envs)
    return ("BASELINE config 4 per-GPU slice: %d envs/GPU, lord-vs-random rollout (all seats uniform random legal move, "
            "Philox stream), EnvCooperation face C=9, fused step+redeal+legal+encode" % args.envs)


def cpu_rollout(envs, warm, steps, threads):
    from oracle import ddz_oracle as O
    perm, lord = load_deals().random_deals(envs, seed=SEED, pool_games=POOL_GAMES)
    n, sec, stats, cs = O.rollout(envs, warm, steps, VARIANT, SEED, perm, lord, POOL_GAMES, threads)
    return n, sec, stats


def cpu_baseline(target_seconds):
    """oracle port timed on this box's host cores over a bounded sample of the config-4 workload"""
    threads = os.cpu_count() or 1
    envs = 4096 * threads
    n, sec, _ = cpu_rollout(envs, 100, 20, threads)                 # calibration
    rate = n / max(sec, 1e-9)
    steps = max(20, min(int(target_seconds * rate / envs), 20000))
    n, sec, stats = cpu_rollout(envs, 100, steps, threads)
    return {"value": n / sec, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "%d envs x %d env-steps after 100 warm-up steps (%.1f s), C oracle (oracle/ddz_oracle.c), "
                      "mean legal moves %.2f" % (envs, steps, sec, stats[8] / max(n, 1)),
            "reference_python_envi": REFERENCE_PYTHON_ENVI}


def cpu_moves(pairs, reps, threads):
    from oracle import ddz_oracle as O
    h, l = load_deals().adversarial_pairs(pairs, seed=5)
    n, sec, counts, cs = O.get_moves_batch(h, l, reps=reps, nthreads=threads)
    return n, sec, float(counts.mean())


def cpu_baseline_moves(target_seconds):
    threads = os.cpu_count() or 1
    pairs = 1024 * threads
    n, sec, _ = cpu_moves(pairs, 2, threads)
    reps = max(2, min(int(target_seconds * (n / max(sec, 1e-9)) / max(n // 2, 1)), 5000))
    n, sec, nbar = cpu_moves(pairs, reps, threads)
    return {"value": n / sec, "unit": "moves/s", "cores": threads, "kind": "port",
            "sample": "%d adversarial pairs x %d passes (%.1f s), oracle constructive generator ddz_ref_get_moves_fast, every "
                      "move packed; mean %.1f moves per pair" % (pairs, reps, sec, nbar)}


def run_reference(args):
    """Reference arm: the reference's CPU path = the oracle port on all host threads (its natives are absent).  Loads
    numpy and oracle/libddz_oracle.so only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = os.cpu_count() or 1
    note = ("CPU arm: the reference's natives are absent, so this is the C oracle port of the same work on all host "
            "threads, over a bounded sample of the workload")
    if args.config == 5:
        pairs = 1024 * threads
        cpu_moves(pairs, max(1, args.warmup), threads)
        n, sec, nbar = cpu_moves(pairs, args.steps, threads)
        value, unit, metric = n / sec, "moves/s", "legal moves/sec (adversarial hands)"
        sample = "%d pairs (of the %d-per-GPU workload) x %d passes, oracle ddz_ref_get_moves_fast, %d threads" % (pairs, args.envs, args.steps, threads)
        cfg = {"workload": workload_text(args), "pairs_per_gpu": args.envs, "sample_pairs": pairs, "mean_moves_per_pair": nbar, "note": note}
    else:
        envs = 4096 * threads
        n, sec, stats = cpu_rollout(envs, 100 + args.warmup, args.steps, threads)
        value, unit, metric = n / sec, UNIT, METRIC
        sample = "%d envs (of the %d-per-GPU workload) x %d env-steps, C oracle port, %d threads" % (envs, args.envs, args.steps, threads)
        cfg = {"workload": workload_text(args), "envs_per_gpu": args.envs, "face_channels": CHANNELS, "sample_envs": envs,
               "mean_legal_moves": stats[8] / max(n, 1), "prefill_steps": 100, "pool_games": POOL_GAMES, "note": note}
        if args.config == 3:
            cfg["note"] += "; the env work only: the reference's Q-network runs in torch on either arm and is not part of the CPU port"
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port", "sample": sample,
                             "reference_python_envi": REFERENCE_PYTHON_ENVI},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- GPU arm: shared pieces
def setup_rank():
    import torch
    import ddz_b200 as D
    os.environ.setdefault("NCCL_PROTO", "LL")       # the only collective is a 128-byte all-reduce: latency protocol
    rank, local, world = D.sharding.init_distributed()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the env has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    return D, torch, rank, local, world, torch.device("cuda", local)


def make_barrier(torch, dev, world):
    import torch.distributed as dist

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    return barrier


def verify_slice(D, torch, dev, rank, B):
    """After the timed regions: a 512-env sample of THIS rank's slice (its global env ids, its Philox streams, its deal rows)
    stepped 48 times on this GPU and compared, every output of every step, with the oracle.  Outside any timed region."""
    import numpy as np
    from oracle import ddz_oracle as O
    n, G, steps = 512, 4, 48
    env0 = rank * B
    perm, lord = D.random_deals(n, seed=SEED + 31 * rank + 7, pool_games=G)
    env = D.BatchedEnvCooperation(n, seed=SEED, device=dev, env0=env0)
    pd, ld = torch.as_tensor(perm).to(dev), torch.as_tensor(lord).to(dev)
    env.prepare(pd, ld, pool_games=G)
    ref = O.RefBatch(n, variant=VARIANT)
    ref.deal(perm, lord, pool_games=G)
    env.observe()
    for t in range(steps):
        off, au, af, face = ref.observe()
        ok = (np.array_equal(env.offsets.cpu().numpy(), off)
              and np.array_equal(env.actions_packed.cpu().numpy().view(np.uint64), au)
              and np.array_equal(env.valid_actions()[0].cpu().numpy(), af)
              and np.array_equal(env.face.cpu().numpy(), face))
        r, done, cat = env.rollout_step(mode=D.native.CHOICE_PHILOX, perm=pd, lord_pile=ld, pool_games=G)
        rr, rd, rc, rrew = ref.step(mode=2, seed=SEED, env0=env0, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=G)
        ok = ok and np.array_equal(r.cpu().numpy(), rr) and np.array_equal(done.cpu().numpy(), rd) \
            and np.array_equal(cat.cpu().numpy(), rc) and np.array_equal(env.reward.cpu().numpy(), rrew)
        if not ok:
            return "MISMATCH at step %d on rank %d" % (t, rank)
    st = env.stats.cpu().numpy()
    if st[7] != 0 or st[4] != ref.stats[4] or st[0] != ref.stats[0]:
        return "stats mismatch on rank %d" % rank
    return "ok"


def verify_timed_run(timed_state, B, rank, perm, lord, P):
    """The timed run ITSELF, at full size: every env of this rank's slice was dealt, prefilled, warmed up and timed with moves
    from its own Philox stream, so the oracle can replay all of it (ddz_ref_rollout_export, all host threads, about a second)
    and the complete state of every env right after the timed region, and the counters, must be equal."""
    import numpy as np
    from oracle import ddz_oracle as O
    fields, meta, stats, steps, listed = timed_state
    n, ostats, f, m = O.rollout_export(B, steps, VARIANT, SEED, perm, lord, P, os.cpu_count() or 1, env0=rank * B)
    if n != B * steps:
        return "oracle replay failed on rank %d" % rank
    st = stats.cpu().numpy()
    same = (np.array_equal(fields.cpu().numpy().view(np.uint64), f) and np.array_equal(meta.cpu().numpy().view(np.uint32), m)
            and np.array_equal(st[[0, 1, 2, 3, 4, 5, 6, 9]], ostats[[0, 1, 2, 3, 4, 5, 6, 9]]) and st[8] - listed == ostats[8])
    return "ok" if same else "MISMATCH of the timed run's final state on rank %d" % rank


def all_ranks_ok(D, torch, dev, world, verdict):
    import torch.distributed as dist
    bad = torch.tensor([0 if verdict == "ok" else 1], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(bad)
    return verdict if verdict != "ok" else ("ok" if int(bad.item()) == 0 else "MISMATCH on another rank")


# ---------------------------------------------------------------------------------------------- --dump-outputs
# The limits are for all ranks together: under torchrun each rank dumps 1/world of the sample and of the rows.
DUMP_BYTES = 64 << 20               # all arrays of one dump, over all ranks
DUMP_ENVS = 8192                    # sampled envs: 17.7 MB of face
DUMP_ROWS = 1 << 16                 # legal-move rows of the sampled envs (15.7 MB of one-hots; 5-8 moves per env in configs 3/4)
DUMP_PAIRS = 1024                   # config 5: sampled pairs (~140 moves each)
DUMP_MOVES = 1 << 18                # ... and their moves as 15 card counts each (15.7 MB)


def dump_sample(n, k, limit, *offsets):
    """sorted indices of the envs (pairs) of n whose outputs are dumped: k of them drawn with a fixed seed (the same in
    every run of the same size), then only the leading ones whose lists, under every CSR offsets given (host int [n+1]),
    hold at most `limit` rows together -- lists are dumped whole, never cut"""
    import numpy as np
    idx = np.arange(n) if n <= k else np.sort(np.random.default_rng(SEED).choice(n, k, replace=False))
    keep = len(idx)
    for off in offsets:
        keep = min(keep, int(np.searchsorted(np.cumsum(off[idx + 1] - off[idx]), limit, side="right")))
    return idx[:keep]


def list_rows(offsets, idx):
    """indices of the rows of the CSR lists idx (offsets: host int [n+1]), in list order"""
    import numpy as np
    return np.concatenate([np.arange(offsets[i], offsets[i + 1], dtype=np.int64) for i in idx] + [np.zeros(0, np.int64)])


def batch_offsets(torch, envs):
    """host int64 [B+1]: the legal-move offsets of the batch the env objects `envs` (the groups of a GroupedEnv, or one
    env) make together"""
    import numpy as np
    counts = torch.cat([e.offsets[1:] - e.offsets[:-1] for e in envs]).cpu().numpy()
    return np.concatenate([[0], np.cumsum(counts, dtype=np.int64)])


def env_outputs(torch, envs, idx, off):
    """What a caller of the fused env-step holds after it, for the envs idx of the batch `envs` (legal-move offsets off,
    batch_offsets): the step's r / done / cat / reward, and the new state's face and legal moves (the one-hot rows of the
    listed envs, in order, and each env's count)."""
    import numpy as np
    dev = envs[0].device
    sel = torch.as_tensor(idx, device=dev)
    rows = torch.as_tensor(list_rows(off, idx), device=dev)
    batch = lambda f: torch.cat([f(e) for e in envs])
    host = lambda t: t.cpu().numpy().astype(np.float32)
    return {"env_index": idx.astype(np.float64), "r": host(batch(lambda e: e.r)[sel]), "done": host(batch(lambda e: e.done)[sel]),
            "cat": host(batch(lambda e: e.cat)[sel]), "reward": host(batch(lambda e: e.reward)[sel]),
            "face": host(batch(lambda e: e.face)[sel]), "legal_counts": np.diff(off)[idx].astype(np.float32),
            "legal_actions": host(batch(lambda e: e.valid_actions()[0])[rows])}


def write_dump(out_dir, arrays, rank, world):
    import numpy as np
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES // world:
        raise SystemExit("--dump-outputs: %d bytes on rank %d exceed its share of the %d-byte limit" % (total, rank, DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ("_rank%d" % rank if world > 1 else "") + ".npy"), a)


# ---------------------------------------------------------------------------------------------- config 4
def run_config4(args):
    import numpy as np
    import torch.distributed as dist
    D, torch, rank, local, world, dev = setup_rank()
    B, K, W, P, NG = args.envs, args.steps, args.warmup, POOL_GAMES, args.groups
    env0 = rank * B                                   # global env ids keep results independent of the GPU count
    perm, lord = D.random_deals(B, seed=SEED + 1000 * rank, pool_games=P)
    barrier = make_barrier(torch, dev, world)

    sampler = ClockSampler(local, args.clock_interval_ms)       # samples from here to the end of the e2e region: the same kernel runs throughout
    if rank == 0:
        sampler.start()

    # ---------------- the rank's envs as NG stream-parallel groups (DESIGN.md 4: one group's load-only prologue and tail
    # overlap the other group's store phase); device-resident deal pool, Philox moves on the device; ONE stats vector
    ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=NG, seed=SEED, device=dev, env0=env0, max_actions_per_env=160)
    compressed = hasattr(ge.envs[0]._face, "_ddz_rows")          # row buffers in compressible memory (the default where supported)
    ge.prepare(perm, lord, pool_games=P)
    for _ in range(args.prefill):
        ge.rollout_step()
    SPG = args.steps_per_graph if (args.steps_per_graph % 2 == 0 and K % args.steps_per_graph == 0) else 2
    ge.capture(steps_per_graph=SPG)     # the loop is launch-bound from Python: replay SPG steps per group as one CUDA graph
    warm_replays = max(-(-max(W, 3) // SPG), 2)
    for _ in range(warm_replays):
        ge.replay()
    ge.join()
    torch.cuda.synchronize(dev)
    if int(ge.stats[7].item()):
        raise SystemExit("env reported errors during warm-up")

    # ---------------- timed region: exactly K env-steps of every env, CUDA events on the launching (current) stream
    stats0 = ge.stats.clone()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    side = torch.cuda.Stream(dev) if world > 1 else None
    snap = torch.zeros_like(ge.stats)   # preallocated all-reduce buffer
    snap_ready = torch.cuda.Event()
    if side is not None:                # warm the collective up on its stream
        with torch.cuda.stream(side):
            dist.all_reduce(snap)
        side.synchronize()
    half = K // SPG                     # graph replays in the window
    every = max(1, args.stats_every // SPG)
    coll_ev = []                        # (issued, done) events of every exchange, on the side stream: where the window's time goes
    barrier()
    e0.record()
    ge._fork()
    exchanges = 0
    for i in range(half):
        ge.replay()                     # per group: two launches of k_env<cooperation, step+observe>
        # the path's only collective: the win/return statistics, all-reduced on a side stream while the envs keep stepping
        # (reference game.py:209-226 logs these counters every log_every episodes).  It is issued from the MIDDLE of each
        # interval, never straight after the barrier: whatever skew the ranks have leaving the barrier is absorbed by the
        # steps already queued, instead of landing on the rank that arrives first.
        if side is not None and (i == (half - 1) // 2 if half <= every else i % every == every // 2):
            snap_ready.record(ge.streams[0])
            side.wait_event(snap_ready)
            with torch.cuda.stream(side):
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record()
                snap.copy_(ge.stats)    # one 128-byte device copy of the vector all groups add to
                dist.all_reduce(snap)
                c1.record()
                coll_ev.append((c0, c1))
            exchanges += 1
    for _ in range(K - half * SPG):
        ge.rollout_step()
    ge.join()
    if side is not None:
        torch.cuda.current_stream(dev).wait_stream(side)
    e1.record()
    barrier()
    total_ms = e0.elapsed_time(e1)
    dstats_t = (ge.stats - stats0).clone()
    dstats = dstats_t.cpu().numpy()
    if int(ge.stats[7].item()):
        raise SystemExit("env reported errors during the timed region")
    local_steps = int(dstats[4])
    assert local_steps == B * K, (local_steps, B * K)   # every env applied one move per step (finished ones re-dealt)
    nbar = float(dstats[8]) / local_steps
    # what the timed run left behind, for verify_timed_run below (a 10 MB device copy, outside every timed region)
    timed_state = None if args.no_verify else (
        torch.cat([e._fields()[0] for e in ge.envs], dim=1).clone(), torch.cat([e._fields()[1] for e in ge.envs]).clone(),
        ge.stats.clone(), int(ge.envs[0]._stepno), sum(int(e.num_actions) for e in ge.envs))
    if args.dump_outputs:               # before the regions below step the same envs further
        off = batch_offsets(torch, ge.envs)
        idx = dump_sample(B, DUMP_ENVS // world, DUMP_ROWS // world, off)
        write_dump(args.dump_outputs, env_outputs(torch, ge.envs, idx, off), rank, world)

    # ---------------- for information: one chain of launches over all envs (no groups), graph replay and eager Python loop
    info = {}
    if NG > 1 and not args.no_single:
        perm_d, lord_d = torch.as_tensor(perm).to(dev), torch.as_tensor(lord).to(dev)
        one = D.BatchedEnvCooperation(B, seed=SEED, device=dev, env0=env0, max_actions_per_env=160)
        one.prepare(perm_d, lord_d, pool_games=P)
        kw = dict(perm=perm_d, lord_pile=lord_d, pool_games=P)
        for _ in range(args.prefill):
            one.rollout_step(**kw)
        gr = D.GraphedRollout(one, perm_d, lord_d, P)
        for _ in range(3):
            gr.replay()
        g0, g1, g2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        torch.cuda.synchronize(dev)
        g0.record()
        for _ in range(max(1, K // 2)):
            gr.replay()
        g1.record()
        for _ in range(K):
            one.rollout_step(**kw)
        g2.record()
        torch.cuda.synchronize(dev)
        info = {"single_chain_graph_ms_per_step": g0.elapsed_time(g1) / (2 * max(1, K // 2)),
                "single_chain_eager_python_ms_per_step": g1.elapsed_time(g2) / K}
        del one, gr, perm_d, lord_d
        torch.cuda.empty_cache()

    # ---------------- e2e: the same env-step through the host-facing API (HostRolloutGroups: ONE native call per step of
    # all groups) with HOST buffers every step: H2D of the step's entropy (int32 [B], pinned) and of the deal-pool refill
    # (one slot of host-made permutations every REFILL steps = about one game length, the rate at which deals are
    # consumed), D2H of the step's results (r, done, cat) into pinned memory.  All copies are inside the timed region.
    R, REFILL = 4, 64
    rng = np.random.default_rng(SEED + rank)
    ent_h = [torch.as_tensor(rng.integers(0, 1 << 31, B, dtype=np.int64).astype(np.int32)).pin_memory() for _ in range(R)]
    pool_h = []
    for i in range(2):
        pp, ll = D.random_deals(B, seed=SEED + 77 + i + 1000 * rank)
        pool_h.append((torch.as_tensor(pp).pin_memory(), torch.as_tensor(ll).pin_memory()))
    ge.join()
    torch.cuda.synchronize(dev)
    host = D.HostRolloutGroups(ge)
    sink = [0]
    DEPTH = D.native.PIPE_DEPTH                                   # the host reads step i's results while step i+3 is issued
    pending = [None] * DEPTH

    def e2e_step(i):
        old = pending[i % DEPTH]
        if old is not None:                                       # the host reads the results of step i-DEPTH
            D.HostRolloutGroups.wait(old)
            sink[0] += int(old.done[0][0]) + int(old.r[-1][-1])
        pending[i % DEPTH] = host.step(ent_h[i % R])
        if i % REFILL == 0:                                       # after the step is on its way: the GPU never waits for it
            pp, ll = pool_h[(i // REFILL) % 2]
            host.refill((i // REFILL) % P, pp, ll)

    # warm-up: one untimed pass of the same shape (a pool upload and the steps that carry its chunks), then flush it, so
    # that no upload is half-way when the window opens and the first-use costs of the pinned pool buffers are paid
    for i in range(max(W, 24)):
        e2e_step(i)
    host.flush()
    for res in pending:
        if res is not None:
            D.HostRolloutGroups.wait(res)
    ge.join()
    barrier()
    stats_e0 = ge.stats.clone()
    x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    x0.record()
    ge._fork()
    for i in range(K):
        e2e_step(i)
    ge.join()
    host.join()                         # ... and the D2H of the last step's results: the window ends on the device
    x1.record()
    for res in pending:                 # the host reads the last results (already on their way when x1 is recorded)
        if res is not None:
            D.HostRolloutGroups.wait(res)
            sink[0] += int(res.done[0][0])
    barrier()
    clocks = sampler.stop()
    e2e_ms = x0.elapsed_time(x1)
    e2e_steps = int((ge.stats - stats_e0)[4].item())
    assert e2e_steps == B * K and sink[0] > -(1 << 40)
    h2d = host.h2d_bytes + (55 * B * ((K + REFILL - 1) // REFILL)) // K
    d2h = host.d2h_bytes
    if int(ge.stats[7].item()):
        raise SystemExit("env reported errors during the e2e region")

    # ---------------- after the timed regions: this rank's sample against the oracle
    verdict = "skipped" if args.no_verify else verify_slice(D, torch, dev, rank, B)
    if verdict == "ok" and timed_state is not None:
        verdict = verify_timed_run(timed_state, B, rank, perm, lord, P)
    if not args.no_verify:
        verdict = all_ranks_ok(D, torch, dev, world, verdict)

    # ---------------- reduce over ranks: MAX of the device times, SUM of the work
    trace = None
    if world > 1:                       # every rank's window and where its exchanges sat in it (ms from the window start)
        mine = torch.tensor([total_ms] + [x for c0, c1 in coll_ev[:4] for x in (e0.elapsed_time(c0), e0.elapsed_time(c1))],
                            dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        trace = {"per_rank_window_ms": [round(float(t[0]), 4) for t in allr],
                 "per_rank_exchange_issued_done_ms": [[round(float(x), 4) for x in t[1:]] for t in allr]}
    total_ms = D.sharding.max_over_ranks(total_ms, dev)
    e2e_ms = D.sharding.max_over_ranks(e2e_ms, dev)
    gstats = D.sharding.allreduce_stats(dstats_t, side_stream=torch.cuda.Stream(dev) if world > 1 else None)
    torch.cuda.synchronize(dev)
    all_steps = int(gstats[4].item())

    if rank == 0:
        peak, peak_src = peaks()
        eb = bytes_per_env_step(nbar)
        value = all_steps / (total_ms * 1e-3)
        step_ms = total_ms / K
        kern_gbs = B * eb / (step_ms * 1e-3) / 1e9
        single = info.get("single_chain_graph_ms_per_step")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": dict({"workload": workload_text(args), "baseline_config": args.config,
                            "envs_per_gpu": B, "env_groups_per_gpu": NG, "face_channels": CHANNELS, "mean_legal_moves": nbar,
                            "prefill_steps": args.prefill, "warmup_env_steps": warm_replays * SPG, "pool_games": P,
                            "parallelism": "env-shard x%d" % world,
                            "launch": "CUDA graph replay, %d env-steps per graph, one chain per env group" % SPG,
                            "collectives": ("none (single GPU)" if world == 1 else
                                            "stats all-reduce (int64[16], NCCL LL) %d time(s) in the timed region, every %d steps "
                                            "from the middle of the interval, on a side stream" % (exchanges, SPG * every)),
                            "l2_policy": ("per-step output (%.0f MB) exceeds the 126 MB L2; no flush" % (B * eb / 1e6) if B * eb > 126e6 else
                                          "per-step output (%.0f MB) FITS the 126 MB L2 and is not flushed between steps: a latency "
                                          "measurement of the launch chain, not a bandwidth line" % (B * eb / 1e6)),
                            "row_buffers": ("compressible device memory (CU_MEM_ALLOCATION_COMP_GENERIC: the L2 compresses "
                                            "the 0/1 thermometer rows on their way to HBM)" if compressed else "plain device memory"),
                            "games_finished": int(gstats[0].item()),
                            "lord_win_rate": float(gstats[1].item()) / max(1, int(gstats[0].item())),
                            "window_trace": trace}, **info),
            "roofline": {"bound": "hbm", "kernel": "k_env<2,step+observe>", "achieved": kern_gbs, "peak": peak,
                         "unit": "GB/s", "frac": kern_gbs / peak, "frac_of_nominal_8000_GBs": kern_gbs / 8000.0,
                         "frac_single_chain": (B * eb / (single * 1e-3) / 1e9 / peak) if single else None,
                         "traffic": ncu_traffic("config4_%dgroups%s" % (NG, "" if compressed else "_plain")),
                         "peak_source": peak_src, "algorithmic_bytes_per_env": eb,
                         "algorithmic_bytes_per_step": B * eb, "ms_per_step": step_ms, "launches_in_flight": NG,
                         "row_buffers_compressed": bool(compressed),
                         "note": "achieved = ALGORITHMIC bytes of one step of all envs / wall time per step, frac = that / the "
                                 "measured copy peak -- not a DRAM-utilisation figure: with the row buffers in compressible "
                                 "memory the DRAM traffic (`traffic`, steady state over >= 10 steps with all groups in flight, "
                                 "profiles/r2_traffic.json) is well below the algorithmic bytes.  The step is %d concurrent "
                                 "launches of the same kernel (one per env group); frac_single_chain is one launch over all %d "
                                 "envs in one chain of launches" % (NG, B)},
            "e2e": {"value": B * K * world / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K, "steps": K,
                    "api": "HostRolloutGroups.step(entropy_host): ONE native call per env-step of all groups (ddz_mpipe_step: one "
                           "H2D of the pinned entropy, one k_env launch per group on its stream, one D2H of r/done/cat -- the "
                           "reference step's return tuple -- on copy streams), results of step t-4 read by the host every step "
                           "(rings of 4 buffers on both sides), refill(slot, perm_host, lord_host) uploads host-made deals "
                           "every %d steps" % REFILL},
            "gpu_launches": K * NG,
            "verify": verdict,
            "verify_scope": "after the timed regions, on every rank: (1) a 512-env sample of its slice, every output of 48 steps "
                            "against the oracle; (2) the timed run itself -- the complete state of ALL its envs and the counters "
                            "right after the timed region against the oracle's replay of the same deals and Philox streams "
                            "(prefill + warm-up + timed steps from the deal, ddz_ref_rollout_export)",
            "clocks": clocks,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if verdict not in ("ok", "skipped"):
        raise SystemExit("verification against the oracle failed: " + verdict)


# ---------------------------------------------------------------------------------------------- config 5
def run_config5(args):
    import numpy as np
    import torch.distributed as dist
    D, torch, rank, local, world, dev = setup_rank()
    n, K, W = args.envs, args.steps, max(args.warmup, 3)
    barrier = make_barrier(torch, dev, world)
    sampler = ClockSampler(local, args.clock_interval_ms)
    if rank == 0:
        sampler.start()
    hands_np, lasts_np = D.adversarial_pairs(n, seed=5 + rank)
    hands = torch.as_tensor(hands_np.view(np.int64)).to(dev)
    lasts = torch.as_tensor(lasts_np.view(np.int64)).to(dev)
    gen = D.MoveGenerator(n, device=dev)
    for _ in range(W):
        gen.generate(hands, lasts)
    torch.cuda.synchronize(dev)
    total = int(gen.offsets[n].item())
    if int(gen.stats[7].item()) or total > gen.cap:
        raise SystemExit("the generator reported errors during warm-up")

    # ---------------- timed region: K calls over all pairs; each call writes 8 * total bytes (145 MB > the 126 MB L2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K):
        gen.generate(hands, lasts)
    e1.record()
    barrier()
    total_ms = e0.elapsed_time(e1)
    if args.dump_outputs:               # the lists of the last call: per-pair counts, and the moves as per-rank card counts
        off = gen.offsets.cpu().numpy().astype(np.int64)
        idx = dump_sample(n, DUMP_PAIRS // world, DUMP_MOVES // world, off)
        rows = torch.as_tensor(list_rows(off, idx), device=dev)
        write_dump(args.dump_outputs, {"pair_index": idx.astype(np.float64), "moves_total": np.array([off[n]], np.float64),
                                       "move_counts": np.diff(off)[idx].astype(np.float32),
                                       "moves": D.unpack_counts(gen.actions[rows]).cpu().numpy().astype(np.float32)}, rank, world)

    # ---------------- e2e: pinned host (hand, last) arrays in, the packed CSR lists (offsets + moves) back in pinned memory
    hh, lh = torch.as_tensor(hands_np.view(np.int64)).pin_memory(), torch.as_tensor(lasts_np.view(np.int64)).pin_memory()
    hd, ld = torch.empty_like(hands), torch.empty_like(lasts)
    off_h = torch.empty(n + 1, dtype=torch.int32).pin_memory()
    mv_h = torch.empty(total, dtype=torch.int64).pin_memory()

    def e2e_call():
        hd.copy_(hh, non_blocking=True); ld.copy_(lh, non_blocking=True)
        acts, offs = gen.generate(hd, ld)
        off_h.copy_(offs, non_blocking=True)
        mv_h.copy_(acts[:total], non_blocking=True)     # the list length of this fixed input is known from the warm-up

    Ke = max(3, min(K, 50))
    for _ in range(2):
        e2e_call()
    torch.cuda.synchronize(dev)
    x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    x0.record()
    for _ in range(Ke):
        e2e_call()
    x1.record()
    barrier()
    clocks = sampler.stop()
    e2e_ms = x0.elapsed_time(x1)
    assert int(off_h[n]) == total and int(gen.stats[7].item()) == 0

    # ---------------- verification (outside the timed regions): a 512-pair sample of this rank, list by list, against the oracle
    verdict = "skipped"
    if not args.no_verify:
        from oracle import ddz_oracle as O
        off = off_h.numpy()
        mv = mv_h.numpy().view(np.uint64)
        verdict = "ok"
        for i in np.random.default_rng(rank).choice(n, 512, replace=False):
            want = np.atleast_1d(O.pack(O.get_moves(O.unpack(hands_np[i]), O.unpack(lasts_np[i]), fast=True)))
            if not np.array_equal(mv[off[i]:off[i + 1]], want):
                verdict = "MISMATCH at pair %d on rank %d" % (i, rank)
                break
        if verdict == "ok":
            # ... and ALL lists of this rank (the ones the e2e region brought back): lengths and an order-sensitive digest of every
            # move against the oracle's generator
            moves, counts, un, od = O.get_moves_digest(hands_np, lasts_np)
            if moves != total or not np.array_equal(np.diff(off), counts) or O.lists_digest(mv, off) != (un, od):
                verdict = "MISMATCH of the full-size digest on rank %d" % rank
        verdict = all_ranks_ok(D, torch, dev, world, verdict)

    total_ms = D.sharding.max_over_ranks(total_ms, dev)
    e2e_ms = D.sharding.max_over_ranks(e2e_ms, dev)
    tot_t = torch.tensor([total, n], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot_t)
    all_moves, all_pairs = int(tot_t[0].item()), int(tot_t[1].item())
    if rank == 0:
        peak, peak_src = peaks()
        step_ms = total_ms / K
        alg = 20.0 * n + 8.0 * total                      # hand + last (16) + offset (4) per pair, 8 per move
        gbs = alg / (step_ms * 1e-3) / 1e9
        line = {"metric": "legal moves/sec (adversarial hands)", "value": all_moves / (step_ms * 1e-3), "unit": "moves/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u64", "data": "synthetic",
                "config": {"workload": workload_text(args), "baseline_config": 5, "pairs_per_gpu": n,
                           "mean_moves_per_pair": total / n, "pairs_per_s": all_pairs / (step_ms * 1e-3),
                           "parallelism": "pair-shard x%d, no collective on the data path" % world,
                           "l2_policy": "each call writes %.0f MB of lists, more than the 126 MB L2; no flush" % (8 * total / 1e6)},
                "roofline": {"bound": "hbm", "kernel": "k_legal_flat", "achieved": gbs, "peak": peak, "unit": "GB/s",
                             "frac": gbs / peak, "frac_of_nominal_8000_GBs": gbs / 8000.0, "traffic": ncu_traffic("config5"),
                             "peak_source": peak_src,
                             "algorithmic_bytes_per_pair": alg / n, "algorithmic_bytes_per_step": alg,
                             "note": "algorithmic bytes = 16 (hand, last) + 4 (offset) per pair + 8 per move; the kernel is "
                                     "issue-bound (integer work per move), far from the HBM roofline"},
                "e2e": {"value": all_moves / (e2e_ms / Ke * 1e-3), "unit": "moves/s", "h2d_bytes_per_step": 16 * n, "d2h_bytes_per_step": 4 * (n + 1) + 8 * total,
                        "ms_per_step": e2e_ms / Ke, "steps": Ke,
                        "api": "MoveGenerator.generate on pinned host (hand, last) arrays: H2D pairs, ddz_legal_moves, D2H of the "
                               "offsets and of every packed move list into pinned memory -- PCIe-bound (the lists are %.0f MB per call)"
                               % (8 * total / 1e6)},
                "gpu_launches": K, "verify": verdict, "clocks": clocks}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_moves(args.cpu_seconds)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if verdict not in ("ok", "skipped"):
        raise SystemExit("verification against the oracle failed: " + verdict)


# ---------------------------------------------------------------------------------------------- config 3
def run_config3(args):
    import numpy as np
    D, torch, rank, local, world, dev = setup_rank()
    if world != 1:
        raise SystemExit("config 3 is a single-GPU configuration (BASELINE.json configs[2])")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from qnet_like import QNetLike                    # the reference's NetCooperation contract (net.py:125-139), random-init
    B, K, W, P = args.envs, args.steps, max(args.warmup, 3), POOL_GAMES
    torch.manual_seed(0)
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = (args.net_precision == "tf32")
    net = QNetLike(CHANNELS, width=256, hidden=256).to(dev).eval()
    if args.scoring == "fused":
        policy = D.BatchedGreedyPolicy(net, fused=True, precision=args.net_precision)
    elif args.net_precision == "bf16":
        inner = net

        class Autocast(torch.nn.Module):
            def forward_state_action(self, x):
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    return inner.forward_state_action(x).float()
        net = Autocast()
    if args.scoring == "module":
        policy = D.BatchedGreedyPolicy(net, chunk_actions=1 << 16)
    sampler = ClockSampler(local, args.clock_interval_ms)
    sampler.start()
    perm, lord = D.random_deals(B, seed=SEED, pool_games=P)
    pd, ld = torch.as_tensor(perm).to(dev), torch.as_tensor(lord).to(dev)
    # other kernels (the network's) share the GPU with the env launches: tiles by ticket, not by launch position
    D.native.set_tile_order("ticket")
    env = D.BatchedEnvCooperation(B, seed=SEED, device=dev, max_actions_per_env=160)
    env.prepare(pd, ld, pool_games=P)
    for _ in range(min(args.prefill, 60)):
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=P)
    gen = torch.Generator(device=dev); gen.manual_seed(1)
    scored = [0]
    last = {}                                              # the last timed step's scores and decisions, for --dump-outputs

    def step(timed):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if timed else None
        if timed:
            ev[0].record()
        is_lord = env.get_role_ID() == 2
        q = policy.q_values(env, is_lord)                  # ddz_q_features + GEMMs, or ddz_encode_state_actions -> the module
        greedy = policy.select(env, q)                     # ddz_select_actions (segmented argmax)
        off = env.offsets
        cnt = off[1:] - off[:-1]
        ent = torch.randint(0, 1 << 30, (B,), device=dev, dtype=torch.int32, generator=gen)
        choice = torch.where(is_lord, greedy, ent % cnt.clamp(min=1)).to(torch.int32)
        if timed:
            ev[1].record()
        env.rollout_step(choice, mode=D.native.CHOICE_INDEX, perm=pd, lord_pile=ld, pool_games=P)
        if timed:
            ev[2].record()
            scored[0] += int(q.numel())
            if args.dump_outputs:
                last.update(q=q, offsets=off, choice=choice)
        return ev

    for _ in range(W):
        step(False)
    torch.cuda.synchronize(dev)
    st0 = env.stats.clone()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    evs = [step(True) for _ in range(K)]
    e1.record()
    torch.cuda.synchronize(dev)
    clocks = sampler.stop()
    total_ms = e0.elapsed_time(e1)
    net_ms = sum(a.elapsed_time(b) for a, b, _ in evs) / K
    env_ms = sum(b.elapsed_time(c) for _, b, c in evs) / K
    if args.dump_outputs:
        # + what the step decided on: the Q-values of the sampled envs' moves in the scored (pre-step) lists, 0 where the
        # landlord is not to move, with each env's count in those lists (q_counts), and the chosen move indices
        off, off0 = batch_offsets(torch, [env]), last["offsets"].cpu().numpy().astype(np.int64)
        idx = dump_sample(B, DUMP_ENVS, DUMP_ROWS, off, off0)
        out = env_outputs(torch, [env], idx, off)
        out["q_counts"] = np.diff(off0)[idx].astype(np.float32)
        out["q_values"] = last["q"][torch.as_tensor(list_rows(off0, idx), device=dev)].cpu().numpy().astype(np.float32)
        out["choice"] = last["choice"][torch.as_tensor(idx, device=dev)].cpu().numpy().astype(np.float32)
        write_dump(args.dump_outputs, out, 0, 1)
    st = (env.stats - st0).cpu().numpy()
    if int(env.stats[7].item()):
        raise SystemExit("env reported errors")
    assert int(st[4]) == B * K
    nbar = float(st[8]) / (B * K)
    peak, peak_src = peaks()
    eb = bytes_per_env_step(nbar)
    gbs = B * eb / (env_ms * 1e-3) / 1e9
    verdict = "skipped" if args.no_verify else verify_slice(D, torch, dev, 0, B)
    line = {"metric": METRIC, "value": B * K / (total_ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": workload_text(args), "baseline_config": 3, "envs_per_gpu": B, "face_channels": CHANNELS,
                       "mean_legal_moves": nbar, "network": "QNetLike(9+1 channels, width 256, hidden 256) = NetCooperation's layer sizes (net.py:125-139), %s, "
                       "torch.manual_seed(0) random init (no checkpoint ships)" % args.net_precision,
                       "scoring": ("fused: ddz_q_features computes the network's first layer (four rank convolutions, max-pool, line "
                                   "convolution, net.py:91-97) for every legal move of the landlord from the packed state and move lists "
                                   "-- the [n, C+1, 15, 4] input is never built --, fc1 / fc2 are two library GEMMs; same weights, same Q "
                                   "values as the torch module within float32 rounding (tests/test_consumer_contract.py)")
                       if args.scoring == "fused" else
                       "module: the torch module on the [n, C+1, 15, 4] input written in place by ddz_encode_state_actions",
                       "network_and_selection_ms_per_step": net_ms, "env_kernel_ms_per_step": env_ms,
                       "actions_scored_per_step": scored[0] / K,
                       "games_finished": int(st[0]), "lord_win_rate": float(st[1]) / max(1, int(st[0])),
                       "note": "the network is the reference's consumer (SURVEY 8 a16: the contract is its torch module, which "
                               "--scoring module runs unchanged); the hot path contributes the env kernel, the Q-scoring kernels "
                               "(ddz_q_features or the in-place [n,C+1,15,4] encoder) and the segmented argmax"},
            "roofline": {"bound": "hbm", "kernel": "k_env<2,step+observe>", "achieved": gbs, "peak": peak, "unit": "GB/s",
                         "frac": gbs / peak, "frac_of_nominal_8000_GBs": gbs / 8000.0, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_env": eb,
                         "note": "the env kernel alone (env_kernel_ms_per_step), one launch over %d envs between two network "
                                 "passes; the step as a whole is network-bound" % B},
            "e2e": {"value": B * K / (total_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "config 3 keeps observations and decisions on the device (that is its point); there is no host copy "
                            "to time -- see config 4 for the host-buffer path"},
            "gpu_launches": 3 * K, "verify": verdict, "clocks": clocks}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(min(args.cpu_seconds, 6.0))
    print(json.dumps(line), flush=True)


def ensure_built():
    """a fresh checkout has no built artefacts (*.so are git-ignored): build them in-tree before importing the package"""
    if not os.path.exists(os.path.join(ROOT, "doudizhu-rl_b200", "libddz_b200.so")):
        import __graft_entry__
        __graft_entry__.build()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        ensure_built()
    else:                                   # the other ranks wait for rank 0's build instead of racing it
        lib = os.path.join(ROOT, "doudizhu-rl_b200", "libddz_b200.so")
        for _ in range(600):
            if os.path.exists(lib) and time.time() - os.path.getmtime(lib) > 2.0:
                break
            time.sleep(0.5)
    {2: run_config4, 4: run_config4, 5: run_config5, 3: run_config3}[args.config](args)


if __name__ == "__main__":
    main()
