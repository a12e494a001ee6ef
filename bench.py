#!/usr/bin/env python
"""Benchmark of the geodesic-guidance hot path (BASELINE.json metric: geodesic maps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One step = one pass of the hot path (FPS seeds -> kNN graph -> geodesic maps) over one synthetic scene of the
workload (default c2: 100k points, 256 seeds, k=16, radius 0.5, 32 levels).  The library call is batched like the
reference's own (cal_geodesic_vectorize takes a batch of scenes): --batch B scenes per call, so K steps are K/B
calls, replayed as CUDA graphs on two alternating streams (the FPS / graph construction of one batch runs under
the propagation of the previous one).
  value     whole-job maps/s with the scenes already resident in HBM: EXACTLY K steps between two CUDA events,
            barrier + synchronize on both sides, max over ranks; --repeats R times the K-step region R times and
            reports the MEDIAN region, all regions listed in `repeats_ms`
  e2e       the same through the host-buffer C-ABI call gf_guidance_host: pinned host points in,
            seeds + maps back in pinned host memory, copies inside the timed region
  roofline  the propagation kernel (geo_bfs_batch_kernel, one launch per batch): algorithmic bytes of SURVEY 8(d)
            x the scenes of a launch / its CUDA-event duration inside the timed region (external event nodes of the
            replayed graphs), against the measured HBM peak (MEASURED_PEAKS.json); `*_alone` = the same launch
            with nothing else running
  cpu_baseline  the CPU oracle port (oracle/) on this box's host cores, bounded sample (N=1 only)
--impl reference times that CPU port as the reference arm on all host cores (the reference's own torch code
cannot travel to the GPU box and its kNN is faiss-gpu, absent everywhere; see DESIGN.md).
--dump-outputs DIR writes what the last timed step returned (the seeds and the maps of one scene) as .npy files, so
that two builds can be compared output for output: the scenes are generated from fixed seeds, so the same arguments
give the same inputs on every run.
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# hardware work queues: the pipeline keeps ~20 streams busy (two batches in flight x (4 FPS + 4 kNN lanes), copy lanes
# of the host path); with the default of 8 connections unrelated streams share a queue and wait for each other
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

N_SCENES = 8  # rotating scenes per rank (both arms)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c1", "c2", "c4"])
    ap.add_argument("--max-step", type=int, default=None, help="override the workload's level bound")
    ap.add_argument("--batch", type=int, default=20, help="scenes per library call (reduced to a divisor of --steps)")
    ap.add_argument("--repeats", type=int, default=1,
                    help="repetitions of the K-step timed region, median reported (0 = automatic, 5 to 21)")
    ap.add_argument("--runners", type=int, default=2, help="batches in flight (alternating CUDA streams)")
    ap.add_argument("--no-graph", action="store_true", help="plain launches instead of CUDA-graph replay")
    ap.add_argument("--seed-sharded", default=None, choices=["shard", "nccl", "fused"],
                    help="ONE scene split by seed blocks over the ranks (SURVEY 8(e), strong scaling): row blocks "
                         "exchanged by an NCCL all-gather, or stored into the peers by the propagation kernel itself")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-threads", type=int, default=2, help="blocking host-buffer calls in flight")
    ap.add_argument("--e2e-batch", type=int, default=4, help="scenes per host-buffer call")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip epilogues / eval setting / model setting records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the seeds and geodesic maps of the last timed step to DIR/*.npy (default arm only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.seed_sharded):
        ap.error("--dump-outputs needs the default arm (--impl ours, no --seed-sharded)")
    return args


def workload(args):
    from geoformer_b200.scenes import CONFIGS

    cfg = dict(CONFIGS[args.workload])
    if args.max_step is not None:
        cfg["max_step"] = args.max_step
    return cfg


def make_scene(cfg, index):
    from geoformer_b200 import scenes

    gen = scenes.scene if cfg["gen"] == "scene" else scenes.room
    return gen(cfg["n"], cfg["seed"] + index)


def config_block(cfg, args):
    """identical in both arms: only what defines the workload"""
    n_sc = N_SCENES if cfg["n"] <= 200_000 else 2
    return {"workload": "%s: %s(n=%d), Q=%d seeds, k=%d, radius=%.3g, max_step=%d" % (
        args.workload, cfg["gen"], cfg["n"], cfg["Q"], cfg["k"], cfg["radius"], cfg["max_step"]),
        "N": cfg["n"], "Q": cfg["Q"], "k": cfg["k"], "radius": cfg["radius"], "max_step": cfg["max_step"],
        "inputs": "%d rotating synthetic scenes per rank (generator seeds %d..%d), %.0f MB of maps each: far above "
                  "the 126 MB L2 in total, no explicit flush" % (n_sc, cfg["seed"], cfg["seed"] + n_sc - 1,
                                                                 4e-6 * cfg["Q"] * cfg["n"])}


def n_scenes_for(cfg):
    return N_SCENES if cfg["n"] <= 200_000 else 2


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload_name, max_step, batch):
    """per-launch DRAM bytes of the propagation kernel from the committed ncu capture of the same configuration
    (profiles/geo_traffic.json: {"<workload>:<max_step>:B<batch>": {"dram_bytes_per_launch": .., "captured": ..}})"""
    p = os.path.join(ROOT, "profiles", "geo_traffic.json")
    try:
        rec = json.load(open(p)).get("%s:%d:B%d" % (workload_name, max_step, batch))
        return (rec["dram_bytes_per_launch"], rec.get("captured")) if rec else (None, None)
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """samples SM clock and throttle reasons of one GPU through NVML while the timed regions run (100 Hz: the
    timed loop only replays a few graphs per region, the poller does not compete with it for the driver)"""

    def __init__(self, index, period=0.01):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if bit and (r & bit):
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples),
                "window": "the repeated timed regions, sampled at %.0f Hz" % (1.0 / self.period)}


# ------------------------------------------------------------------------------------------------
# CPU port (oracle) timing: used for cpu_baseline and for --impl reference.  The ONLY place bench.py
# touches oracle/.
# ------------------------------------------------------------------------------------------------
def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


class CpuPort:
    """FPS + exact kNN + propagation of whole scenes on the host cores (OpenMP team = every core this process may
    run on, set explicitly: torch.distributed.run exports OMP_NUM_THREADS=1).  Nothing is sampled or extrapolated
    unless a whole scene would take longer than `max_step_s` (few-core hosts); then the kNN query rows are cut to
    a prefix and the record says so."""

    def __init__(self, cfg, max_step_s=12.0):
        import numpy as np

        import oracle

        oracle.build()
        self.np, self.oracle, self.cfg = np, oracle, cfg
        self.cores = oracle.set_num_threads(host_cores())
        self.xs = [make_scene(cfg, s).numpy() for s in range(n_scenes_for(cfg))]
        self.N, self.Q, self.k = cfg["n"], cfg["Q"], cfg["k"]
        rows = min(self.N, 2048)
        t0 = time.perf_counter()
        oracle.knn_sq(self.xs[0], self.k, self.xs[0][:rows])
        est = (time.perf_counter() - t0) / rows * self.N
        self.rows = self.N if est <= max_step_s else max(2048, int(self.N * max_step_s / est))
        self.full = self.rows >= self.N
        self.graph = None
        if not self.full:  # the propagation needs the whole graph: built once, untimed
            self.graph = [oracle.find_knn(x, self.k) for x in self.xs[:1]]
        self.sample = ("whole scenes: FPS + exact kNN of all %d rows + propagation, %d OpenMP threads" % (self.N, self.cores)
                       if self.full else
                       "FPS whole + kNN on the first %d of %d query rows (NOT extrapolated: the step is shorter than a "
                       "whole scene) + propagation whole on a prebuilt graph, %d OpenMP threads" % (self.rows, self.N, self.cores))

    def step(self, i=0):
        """seconds of one step and the per-stage split"""
        o, np = self.oracle, self.np
        x = self.xs[i % len(self.xs)] if self.full else self.xs[0]
        t0 = time.perf_counter()
        seeds = o.furthest_point_sampling(x[None], self.Q)[0]
        t1 = time.perf_counter()
        if self.full:
            D2, I = o.knn_sq(x, self.k)
            D = np.sqrt(D2)
        else:
            o.knn_sq(x, self.k, x[: self.rows])
            D, I = self.graph[0]
        t2 = time.perf_counter()
        o.geodesic(D, I, seeds, self.cfg["radius"], self.cfg["max_step"])
        t3 = time.perf_counter()
        return t3 - t0, {"fps_s": t1 - t0, "knn_s": t2 - t1, "geodesic_s": t3 - t2}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = workload(args)
    port = CpuPort(cfg)
    for i in range(args.warmup):
        port.step(i)
    t_wall0 = time.perf_counter()
    total, parts = 0.0, []
    for i in range(args.steps):
        t, p = port.step(args.warmup + i)
        total += t
        parts.append(p)
    wall = time.perf_counter() - t_wall0
    ms = 1e3 * total / max(1, args.steps)
    value = cfg["Q"] / (ms * 1e-3)
    line = {
        "impl": "reference", "metric": "geodesic maps/sec", "value": value, "unit": "maps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_block(cfg, args),
        "arm": "CPU port of the reference path (oracle/oracle.c, OpenMP) on rank 0's host cores",
        "cpu_baseline": {"value": value, "unit": "maps/s", "cores": port.cores, "kind": "port", "sample": port.sample},
        "e2e": {"value": value, "unit": "maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "stage_s": {k: statistics.mean(p[k] for p in parts) for k in parts[0]} if parts else {},
        "whole_scene_per_step": port.full, "wall_s": wall,
    }
    print(json.dumps(line), flush=True)
    return 0


def bind_to_gpu_numa_node(local):
    """Multi-rank runs only: keep this rank's host threads (and therefore the first-touch placement of its
    pinned buffers) on the CPUs NVML reports as local to its GPU, so that several ranks' D2H copies do not
    all land in one socket's memory.  Best effort: any failure leaves the affinity as it was."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w in range(len(mask)) for b in range(64) if (int(mask[w]) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if len(cpus) >= 4:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------
def seed_sharded_record(cfg4, mode, steps, dist, dev, rank, world):
    """One c4 scene (1M points, 512 seeds) split by seed blocks over the ranks (SURVEY 8(e) row c4), next to the
    same scene on ONE GPU measured in the same process.  mode "shard": every rank keeps its (Q/G, N) block, no
    exchange (the mode that scales); "fused" / "nccl": the full matrix on every rank, rows stored into the peers by
    the propagation kernel / gathered by NCCL.  Returns the sub-record (identical on all ranks)."""
    import torch

    from geoformer_b200.guidance import GuidanceRunner
    from geoformer_b200.parallel import (SeedShardedRows, seed_sharded_guidance, seed_sharded_guidance_fused,
                                         shard_seeds)

    N, Q, k = cfg4["n"], cfg4["Q"], cfg4["k"]
    x = make_scene(cfg4, 0).to(dev)

    def timed(fn, n):
        for _ in range(3):
            out = fn()
        dist.barrier()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out

    one = GuidanceRunner(N, Q, k, cfg4["radius"], cfg4["max_step"], device=dev)
    ms_one, out_one = timed(lambda: one.run(x), steps)
    q0, q1 = shard_seeds(Q, rank, world)
    want = out_one[1][q0:q1].clone()
    del one, out_one
    torch.cuda.empty_cache()
    rec = {"workload": "c4: room(n=%d), Q=%d, k=%d, radius=%.3g, max_step=%d" % (N, Q, k, cfg4["radius"], cfg4["max_step"]),
           "world": world, "steps": steps, "one_gpu_ms_per_scene": ms_one}
    for m in (["shard", mode] if mode != "shard" else ["shard"]):
        rows = SeedShardedRows(Q, N) if m == "fused" else None
        if m == "shard":
            fn = lambda: seed_sharded_guidance(x, Q, k, cfg4["radius"], cfg4["max_step"], gather=False)  # noqa: E731
        elif m == "fused":
            fn = lambda: seed_sharded_guidance_fused(x, Q, k, cfg4["radius"], cfg4["max_step"], rows)  # noqa: E731
        else:
            fn = lambda: seed_sharded_guidance(x, Q, k, cfg4["radius"], cfg4["max_step"])  # noqa: E731
        ms, out = timed(fn, steps)
        mine = out[1] if m == "shard" else out[1][q0:q1]
        same = torch.tensor([1 if torch.equal(mine, want) else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        rec[m] = {"ms_per_scene": ms, "maps_per_s": Q / (ms * 1e-3), "speedup_vs_one_gpu": ms_one / ms,
                  "rows_identical_to_the_one_gpu_run_on_all_ranks": bool(same.item())}
        del out, mine
        if rows is not None:
            rows.close()
        torch.cuda.empty_cache()
    return rec


def run_seed_sharded(args):
    """One scene, seed blocks per rank (strong scaling).  Not the driver's default line: an extra mode
    for the c4 row of SURVEY 8(e); prints the same JSON shape."""
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29511")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    cfg = workload(args)
    K = args.steps
    sampler = ClockSampler(local)
    sampler.start()
    rec = seed_sharded_record(cfg, args.seed_sharded, K, dist, dev, rank, world)
    clocks = sampler.stop()
    if rank == 0:
        main = rec[args.seed_sharded]
        print(json.dumps({
            "metric": "geodesic maps/sec", "value": main["maps_per_s"], "unit": "maps/s", "n_gpus": world, "steps": K,
            "warmup": 3, "ms_per_step": main["ms_per_scene"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_block(cfg, args),
            "parallelism": "seed-sharded x%d, exchange: %s" % (world, args.seed_sharded), "clocks": clocks,
            "seed_sharded": rec,
        }), flush=True)
    dist.destroy_process_group()
    return 0


def pick_batch(K, want):
    """largest batch size <= want that divides K (K steps must be whole calls)"""
    for b in range(max(1, min(want, 32)), 0, -1):
        if K % b == 0:
            return b
    return 1


DUMP_MAX_VALUES = 8 << 20  # 32 MB of f32 maps per dump


def dump_outputs(out_dir, seeds, geo):
    """seeds.npy (Q,) f64 and geo.npy (Q, M) f32: all N columns of the (Q, N) maps when Q*N <= DUMP_MAX_VALUES, else
    M = DUMP_MAX_VALUES // Q columns drawn with a fixed seed; geo_columns.npy (M,) f64 lists which."""
    import numpy as np
    import torch

    Q, N = geo.shape
    cols = np.arange(N)
    if Q * N > DUMP_MAX_VALUES:
        cols = np.sort(np.random.default_rng(0).choice(N, DUMP_MAX_VALUES // Q, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "seeds.npy"), seeds.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "geo.npy"), geo[:, torch.from_numpy(cols).to(geo.device)].cpu().numpy())
    np.save(os.path.join(out_dir, "geo_columns.npy"), cols.astype(np.float64))


def run_ours(args):
    import torch

    from geoformer_b200 import _capi as C
    from geoformer_b200.guidance import BATCH_MAX_POINTS, BatchGuidanceRunner, GuidanceRunner, HostGuidance

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    numa_cpus = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = workload(args)
    N, Q, k = cfg["n"], cfg["Q"], cfg["k"]
    K = args.steps
    L = C.lib()
    batched = N <= BATCH_MAX_POINTS
    B = pick_batch(K, args.batch) if batched else 1
    calls = K // B
    n_run = max(1, min(args.runners, calls))
    S = n_scenes_for(cfg)
    # every rank runs the same S scenes: weak scaling with an identical per-GPU workload (with different scenes
    # per rank the max-over-ranks time measures which rank drew the heaviest scenes: +-10 % between scene sets)
    scenes_host = [make_scene(cfg, s) for s in range(S)]
    xs = [x.to(dev) for x in scenes_host]
    stream = torch.cuda.current_stream(dev)
    side = [torch.cuda.Stream(device=dev) for _ in range(n_run)]

    if batched:
        runners = [BatchGuidanceRunner(N, B, Q, k, cfg["radius"], cfg["max_step"], device=dev,
                                       graph=not args.no_graph, stage_events=True) for _ in range(n_run)]
        for i, r in enumerate(runners):  # runner i always holds the same B scenes: together they rotate over all S
            r.load([xs[(i * B + b) % S] for b in range(B)], side[i])
    else:  # scenes beyond the on-chip bitmaps (c4): one scene per call, plain launches
        runners = [GuidanceRunner(N, Q, k, cfg["radius"], cfg["max_step"], device=dev) for _ in range(n_run)]

    def launch(c):
        r, st = runners[c % n_run], side[c % n_run]
        if batched:
            r.replay(st)
        else:
            r.run(xs[c % S], st)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # warm-up: W steps, and at least three calls of every (runner, stream) pair: graph capture, auxiliary streams
    # and events, kernel attributes and the clocks are all settled before the first timed region
    warm_calls = max(-(-max(3, args.warmup) // B), 3 * n_run)
    for c in range(warm_calls):
        launch(c)
    torch.cuda.synchronize(dev)
    if batched:
        reach = [int(v) for r in runners for v in r.stats[:, 0].tolist()]
        levels = [int(v) for r in runners for v in r.stats[:, 1].tolist()]
        launches_per_call = runners[0].launches_per_run
    else:
        reach = [int(r.stats[0].item()) for r in runners]
        levels = [int(r.stats[1].item()) for r in runners]
        C.reset_launch_count()
        launch(0)
        torch.cuda.synchronize(dev)
        launches_per_call = C.launch_count()

    # ---- device-resident timed regions -----------------------------------------------------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def region():
        barrier()
        e0.record(stream)
        for st_ in side:
            st_.wait_event(e0)
        t_host0 = time.perf_counter()
        for c in range(calls):
            launch(c)
        host_ms = 1e3 * (time.perf_counter() - t_host0)
        for st_ in side:
            done = torch.cuda.Event()
            done.record(st_)
            stream.wait_event(done)
        e1.record(stream)
        barrier()
        prop = [r.propagation_ms() for r in runners] if batched else []
        return e0.elapsed_time(e1), host_ms, [p for p in prop if p]

    probe_ms, _, _ = region()  # untimed: sizes the number of repetitions
    R = args.repeats if args.repeats > 0 else int(max(5, min(21, 60.0 / max(probe_ms, 0.05))))
    if dist is not None:  # the same count on every rank
        t = torch.tensor([R], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        R = int(t.item())
    sampler = ClockSampler(local)
    sampler.start()
    reps, host_reps, prop_in_region = [], [], []
    for _ in range(R):
        ms, host_ms, prop = region()
        reps.append(ms)
        host_reps.append(host_ms)
        prop_in_region += prop
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:  # the last step: the last scene of the last call
        last = runners[(calls - 1) % n_run]
        dump_outputs(args.dump_outputs, *((last.seeds[-1], last.geo[-1]) if batched else (last.seeds, last.geo)))
    if dist is not None:
        t = torch.tensor(reps, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)  # per repetition: the slowest rank
        reps = [float(v) for v in t.tolist()]
    ms_total = statistics.median(reps)
    ms_step = ms_total / K
    value = world * K * Q / (ms_total * 1e-3)
    spread = (max(reps) - min(reps)) / ms_total

    # ---- one batch alone (nothing else on the GPU): the propagation launch and the whole call ------------------
    alone = {}
    if batched:
        r0 = runners[0]
        ts, ps = [], []
        for _ in range(6):
            torch.cuda.synchronize(dev)
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(side[0])
            r0.replay(side[0])
            b_.record(side[0])
            torch.cuda.synchronize(dev)
            ts.append(a_.elapsed_time(b_))
            ps.append(r0.propagation_ms())
        alone = {"call_ms": statistics.median(ts[1:]), "propagation_ms": statistics.median(ps[1:]), "scenes": B}

    # ---- per-stage times of ONE scene alone (plain launches, stage events of the library) ---------------------
    stage_ms_serial = None
    try:
        r1 = GuidanceRunner(N, Q, k, cfg["radius"], cfg["max_step"], device=dev)
        Ks = 10
        ev_s = [[L.gf_event_create() for _ in range(5)] for _ in range(Ks)]
        arr_s = [(ctypes.c_void_p * 5)(*e) for e in ev_s]
        for i in range(Ks):
            L.gf_set_stage_events(arr_s[i], 5)
            r1.run(xs[i % S], stream)
        torch.cuda.synchronize(dev)

        def stage_serial(a, b):
            v = [L.gf_event_elapsed_ms(e[a], e[b]) for e in ev_s[3:]]
            v = [x for x in v if x >= 0]
            return statistics.median(v) if v else None

        stage_ms_serial = {"knn_grid_build": stage_serial(0, 1), "knn_query_and_fps_join": stage_serial(1, 2),
                           "geodesic_propagation": stage_serial(3, 4), "whole_call": stage_serial(0, 4)}
        for e in ev_s:
            for h in e:
                L.gf_event_destroy(h)
        del r1
    except Exception as ex:
        stage_ms_serial = {"error": repr(ex)}

    # ---- roofline of the propagation launch ----------------------------------------------------------
    Kn = k - 1
    R_pairs = statistics.mean(reach) if reach else 0
    b_geo = 4.0 * Q * N + (R_pairs + Q) * Kn * 12.0 + 4.0 * R_pairs  # SURVEY 8(d): per reached pair 12K+4 B, + dense output
    peak, peak_src = measured_peak()
    per_launch = b_geo * B
    t_in = statistics.median(prop_in_region) if prop_in_region else None
    t_alone = alone.get("propagation_ms") if alone else (stage_ms_serial or {}).get("geodesic_propagation")
    if not batched:
        t_in = t_in or t_alone
    achieved = per_launch / (t_in * 1e-3) / 1e9 if t_in else None
    achieved_alone = per_launch / (t_alone * 1e-3) / 1e9 if t_alone else None
    traffic, traffic_date = ncu_traffic(args.workload, cfg["max_step"], B)
    roofline = {"bound": "hbm", "kernel": "geo_bfs_batch_kernel" if batched else "geo_seed_bfs_kernel",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": traffic, "traffic_captured": traffic_date, "peak_source": peak_src,
                "scenes_per_launch": B, "algorithmic_bytes_per_launch": per_launch,
                "algorithmic_bytes_per_scene": b_geo, "reached_pairs_R_per_scene": R_pairs,
                "levels": max(levels) if levels else None,
                "kernel_ms": t_in, "kernel_ms_samples": len(prop_in_region), "kernel_ms_alone": t_alone,
                "achieved_alone": achieved_alone, "frac_alone": (achieved_alone / peak) if achieved_alone else None,
                "note": "kernel_ms = duration of the propagation launch (one per batch of %d scenes) between two event "
                        "nodes of the replayed graph, inside the timed regions (with more than one call per region the "
                        "next batch's FPS / kNN kernels share the SMs); *_alone = the same launch in a call of its own"
                        % B,
                "compulsory_bytes_per_scene": 12.0 * N + 8.0 * N * k + 4.0 * Q * N}

    extras = {}
    if not args.no_extras and world == 1:
        extras = extra_records(args, cfg, xs, dev, stream, peak)

    # ---- end to end through the host-buffer C-ABI call ------------------------------------------
    e2e = None
    if not args.no_e2e:
        from geoformer_b200.guidance import HostBatchGuidance

        pinned = [x.pin_memory() for x in scenes_host]
        Be = max(1, min(args.e2e_batch, 16)) if batched else 1
        nthreads = max(1, args.e2e_threads)  # blocking calls in flight (a call overlaps its own copies and compute)
        if batched:
            hgs = [HostBatchGuidance(N, Be, Q, k, cfg["radius"], cfg["max_step"], device=dev) for _ in range(nthreads)]
            run_one = lambda h, c: h.run([pinned[(c * Be + b) % S] for b in range(Be)])  # noqa: E731
            call_name = "gf_guidance_batch_host (%d scenes per call" % Be
        else:
            hgs = [HostGuidance(N, Q, k, cfg["radius"], cfg["max_step"], device=dev) for _ in range(nthreads)]
            run_one = lambda h, c: h.run(pinned[c % S])  # noqa: E731
            call_name = "gf_guidance_host (1 scene per call"
        Ke = (40 // Be) * Be if batched else 8  # scenes: the copy of the maps is the bound; a fixed count keeps fill / drain small
        ncalls = Ke // Be
        for h in hgs:
            run_one(h, 0)

        def worker(tid):
            torch.cuda.set_device(local)
            for c in range(tid, ncalls, nthreads):
                run_one(hgs[tid], c)

        barrier()
        t0 = time.perf_counter()
        th = [threading.Thread(target=worker, args=(t,)) for t in range(nthreads)]
        for t_ in th:
            t_.start()
        for t_ in th:
            t_.join()
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        # what the link alone gives: the same maps copied device -> pinned host, nothing else running
        link = None
        try:
            src = torch.empty((Q, N), dtype=torch.float32, device=dev)
            dst = hgs[0].geo_host[0] if batched else hgs[0].geo_host
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize(dev)
            a_.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            b_.record()
            torch.cuda.synchronize(dev)
            link = 4.0 * Q * N * 4 / (a_.elapsed_time(b_) * 1e-3) / 1e9
            del src
        except Exception:
            pass
        e2e = {"value": world * Ke * Q / dt, "unit": "maps/s", "h2d_bytes_per_step": hgs[0].h2d_bytes,
               "d2h_link_GBps": link,
               "d2h_achieved_GBps": hgs[0].d2h_bytes * Ke / dt / 1e9,
               "d2h_bytes_per_step": hgs[0].d2h_bytes, "steps": Ke, "ms_per_step": 1e3 * dt / Ke,
               "call": call_name + ", pinned host buffers, %d overlapped host threads)" % nthreads}
        del hgs

    # ---- one large scene split by seed blocks over the ranks (SURVEY 8(e) row c4), multi-rank runs only --------
    sharded = None
    if dist is not None and args.workload == "c2":
        try:
            from geoformer_b200.scenes import CONFIGS

            for r in runners:
                if batched:
                    r.close()
            runners = []
            torch.cuda.empty_cache()
            sharded = seed_sharded_record(dict(CONFIGS["c4"]), "fused", 6, dist, dev, rank, world)
            if rank != 0:
                sharded = None
        except Exception as ex:
            sharded = {"error": repr(ex)}

    # ---- CPU baseline (rank 0, N=1 only) ------------------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            port = CpuPort(cfg)
            ts = [port.step(i)[0] for i in range(3)]
            cpu = {"value": Q / min(ts), "unit": "maps/s", "cores": port.cores, "kind": "port", "sample": port.sample}
        except Exception as ex:  # the benchmark itself must not depend on the checker
            cpu = {"value": None, "unit": "maps/s", "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}

    if rank == 0:
        line = {
            "metric": "geodesic maps/sec", "value": value, "unit": "maps/s", "n_gpus": world, "steps": K,
            "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_block(cfg, args),
            "parallelism": "scene-parallel x%d (one scene per rank per step, no collective; every rank runs the same "
                           "%d scenes)" % (world, S),
            "pipeline": {"scenes_per_call": B, "calls_per_region": calls, "calls_in_flight": n_run,
                         "cuda_graph_replay": bool(batched and not args.no_graph), "kernels_per_call": launches_per_call},
            "repeats_ms": reps, "repeats": R, "repeat_spread": spread,
            "e2e": e2e, "gpu_launches": calls * (launches_per_call or 0), "clocks": clocks, "roofline": roofline,
            "cpu_baseline": cpu, "one_batch_alone": alone, "stage_ms_serial": stage_ms_serial,
            "scenes_per_s": value / Q, "host_enqueue_ms_per_step": statistics.median(host_reps) / K,
            "host_cpus_bound_to_gpu_node": numa_cpus, "seed_sharded_c4": sharded,
        }
        line.update(extras)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def extra_records(args, cfg, xs, dev, stream, peak):
    """N=1 only, all outside the timed regions: the reference's evaluation and model settings, the two epilogues."""
    import torch

    from geoformer_b200 import _capi as C
    from geoformer_b200.guidance import BatchGuidanceRunner, GuidanceRunner

    L = C.lib()
    N, Q, k = cfg["n"], cfg["Q"], cfg["k"]
    S = len(xs)
    out = {}

    def batch_alone(kk, radius, max_step, B):
        r = BatchGuidanceRunner(N, B, Q, kk, radius, max_step, device=dev, stage_events=True)
        r.load([xs[b % S] for b in range(B)])
        ts, ps = [], []
        for _ in range(5):
            torch.cuda.synchronize(dev)
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(stream)
            r.replay(stream)
            b_.record(stream)
            torch.cuda.synchronize(dev)
            ts.append(a_.elapsed_time(b_))
            ps.append(r.propagation_ms())
        reached = float(r.stats[:, 0].double().mean().item())
        lev = int(r.stats[:, 1].max().item())
        r.close()
        return statistics.median(ts[1:]), statistics.median(ps[1:]), reached, lev

    # ---- the reference's evaluation setting (max_step = 256, geoformer_fs.py:502; SURVEY 8: "additionally
    #      report max_step=256") and the model's own call (neighbor=64, radius=0.05, max_step=256, :497-506) -------
    if args.workload == "c2" and cfg["max_step"] == 32:
        for name, kk, rad, ms in (("eval_setting_max_step_256", k, cfg["radius"], 256),
                                  ("model_setting_k64_r005_ms256", 64, 0.05, 256)):
            try:
                B = 4
                call, prop, reached, lev = batch_alone(kk, rad, ms, B)
                b_s = 4.0 * Q * N + (reached + Q) * (kk - 1) * 12.0 + 4.0 * reached
                out[name] = {"neighbor": kk, "radius": rad, "max_step": ms, "scenes_per_call": B, "levels_run": lev,
                             "reached_pairs_R_per_scene": reached, "call_ms_per_scene_alone": call / B,
                             "propagation_ms_per_scene_alone": prop / B, "maps_per_s_alone": Q * B / (call * 1e-3),
                             "algorithmic_bytes_per_scene": b_s, "achieved_alone": b_s * B / (prop * 1e-3) / 1e9,
                             "frac_alone": b_s * B / (prop * 1e-3) / 1e9 / peak}
            except Exception as ex:
                out[name] = {"error": repr(ex)}

    # ---- config 5: the post-backbone few-shot forward (stub backbone, random weights) with the library's kernels vs
    #      the reference's torch formulation of the same pieces, at the model's shapes --------------------------------
    if args.workload == "c2":
        try:
            from geoformer_b200.harness import FewShotForward

            torch.manual_seed(5)
            net = FewShotForward().to(dev)  # m=16, dec_dim 64, 4 layers, 2048 contexts, 256 queries (test config)
            locs = xs[0][None].contiguous()
            feats = torch.randn(1, N, 16, device=dev)
            support = torch.randn(1, 32, device=dev)

            def run(impl):
                return net(locs, feats, support, impl=impl)  # neighbor 64, radius 0.05, max_step 256 (:497-506)

            def timeit_h(impl, reps=4):
                run(impl)
                torch.cuda.synchronize(dev)
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record(stream)
                for _ in range(reps):
                    o = run(impl)
                b_.record(stream)
                torch.cuda.synchronize(dev)
                return a_.elapsed_time(b_) / reps, o

            t_b, o_b = timeit_h("b200")
            t_t, o_t = timeit_h("torch")
            scale = o_t[0][0].abs().max().item()
            out["config5_harness"] = {
                "what": "geoformer_fs.py:424-596 after the backbone (stub): aggregator -> geodesic (k=64, r=0.05, 256 levels) "
                        "-> 4 decoder layers -> mask head, 100k foreground points, 2048 contexts, 256 queries, random init",
                "ms_forward_b200_path": t_b, "ms_forward_torch_formulation": t_t, "speedup": t_t / t_b,
                "mask_logit_max_abs_diff": (o_b[0][0] - o_t[0][0]).abs().max().item(), "mask_logit_scale": scale,
                "note": "both share the geodesic maps' kernel (the reference's torch level loop needs tens of GB at this "
                        "size) and the plain torch.nn layers; the difference is the fused aggregator, the fused "
                        "embedding + cross-attention and the mask-head epilogue"}
            del net, o_b, o_t
        except Exception as ex:
            out["config5_harness"] = {"error": repr(ex)}

    # ---- the two distance -> bias epilogues (SURVEY a10 / a11), timed on their own ---------------------
    try:
        from geoformer_b200.bias import decoder_relative_embedding, decoder_relative_pos, mask_head_relative_coords
        from geoformer_b200.pointnet2 import _ext as p2

        Cn = 2048  # contexts of the real model (geoformer_fs.py:630-645); the seeds are their prefix
        ctx = p2.furthest_point_sampling(xs[0][None].contiguous(), Cn)
        r1 = GuidanceRunner(N, Q, k, cfg["radius"], cfg["max_step"], device=dev)
        geo0 = r1.run(xs[0], stream)[1]
        ctx_xyz = xs[0][ctx[0].long()][None].contiguous()
        q_xyz = ctx_xyz[:, :Q].contiguous()
        torch.cuda.synchronize(dev)

        def timeit(fn, reps=10):
            fn()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record(stream)
            for _ in range(reps):
                fn()
            b_.record(stream)
            torch.cuda.synchronize(dev)
            return a_.elapsed_time(b_) / reps

        t_dec = timeit(lambda: decoder_relative_pos([geo0], ctx, q_xyz, ctx_xyz))
        t_mask = timeit(lambda: mask_head_relative_coords(geo0, xs[0], q_xyz[0]))
        rmax0 = r1.row_max.clone()
        t_mask1 = timeit(lambda: mask_head_relative_coords(geo0, xs[0], q_xyz[0], row_max=rmax0))
        gauss_B = torch.randn(3, 32, device=dev)  # d_pos = 64 (config dec_dim), pos_embedding.py:38-41
        pc = [xs[0].min(0)[0][None].contiguous(), xs[0].max(0)[0][None].contiguous()]
        t_four = timeit(lambda: decoder_relative_embedding([geo0], ctx, q_xyz, ctx_xyz, gauss_B, pc))
        b_four = 4.0 * Q * Cn * (1 + 64)          # gather + (B,Q,C,64) write; the (B,Q,C,3) tensor never exists
        b_dec = 4.0 * Q * Cn * (1 + 3)            # SURVEY 8(d): gather + (B,Q,C,3) write
        b_mask = 4.0 * Q * N * (1 + 3) + 12.0 * N  # one read of geo + (Q,3,N) write + coords
        out["epilogues"] = {
            "decoder_bias": {"ms": t_dec, "algorithmic_bytes": b_dec, "GBps": b_dec / t_dec / 1e6},
            "decoder_bias_fourier": {"ms": t_four, "algorithmic_bytes": b_four, "GBps": b_four / t_four / 1e6,
                                     "frac_of_hbm_peak": b_four / t_four / 1e6 / peak},
            "mask_head_bias": {"ms": t_mask, "algorithmic_bytes": b_mask, "GBps": b_mask / t_mask / 1e6,
                               "frac_of_hbm_peak": b_mask / t_mask / 1e6 / peak},
            "mask_head_bias_with_row_max": {"ms": t_mask1, "algorithmic_bytes": b_mask, "GBps": b_mask / t_mask1 / 1e6,
                                            "frac_of_hbm_peak": b_mask / t_mask1 / 1e6 / peak},
        }
        del r1
    except Exception as ex:
        out["epilogues"] = {"error": repr(ex)}
    return out


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        sys.exit(run_reference(a))
    sys.exit(run_seed_sharded(a) if a.seed_sharded else run_ours(a))
