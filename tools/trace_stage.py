"""Where the FPS / kNN-graph stage of one batched guidance call spends its time.

    python tools/trace_stage.py [--workload c2] [--batch 20] [--calls 3] [--out stage.json]
    GF_LIB=geoformer_b200/libgeoformer_b200_x.so python tools/trace_stage.py ...

Replays single batched calls (plain launches, no CUDA graph, nothing else in flight) under torch.profiler with CUDA
activities and reads every kernel's start and end from the trace.  The stage of a call runs from its first kernel's
start to the start of the propagation launch (geo_bfs_batch_kernel).  Printed per call:
  streams      each stream's kernels, start and end in microseconds from the stage start
  fps_lanes    the FPS chain per stream: its span, busy time and the gaps between consecutive FPS launches
  knn_lanes    the span of each stream's kNN work (build and query kernels) and its busy time
  no_query     the share of the stage in which no kNN query kernel runs
The JSON written to --out holds every call; the last line printed is the summary (median over the calls).
"""
import argparse
import json
import os
import statistics
import sys
import tempfile

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from geoformer_b200.guidance import BatchGuidanceRunner  # noqa: E402
from geoformer_b200.scenes import CONFIGS, scene  # noqa: E402


def kind(name):
    if "fps_" in name:
        return "fps"
    if "knn_grid_query" in name:
        return "query"
    if "knn_" in name:
        return "build"
    if "geo_bfs_batch" in name:
        return "propagation"
    return "other"


def union_us(intervals):
    tot, end = 0.0, None
    for a, b in sorted(intervals):
        if end is None or a > end:
            tot += b - a
            end = b
        elif b > end:
            tot += b - end
            end = b
    return tot


def one_call(runner, xs):
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            runner.run(xs)
            torch.cuda.synchronize()
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    kern = [e for e in trace["traceEvents"] if e.get("cat") == "kernel" and e.get("ph") == "X"]
    kern.sort(key=lambda e: e["ts"])
    prop = [e for e in kern if kind(e["name"]) == "propagation"]
    if not prop:
        raise SystemExit("no propagation launch in the trace: is this the batched call?")
    t0, t1 = kern[0]["ts"], prop[0]["ts"]
    stage = t1 - t0
    streams = {}
    for e in kern:
        s = str(e.get("args", {}).get("stream", e.get("tid")))
        short = e["name"].split("(")[0].replace("void ", "")
        streams.setdefault(s, []).append((short, kind(e["name"]), e["ts"] - t0, e["ts"] + e["dur"] - t0))
    fps_lanes, knn_lanes = {}, {}
    for s, ks in streams.items():
        f = [k for k in ks if k[1] == "fps"]
        if f:
            gaps = [round(b[2] - a[3], 2) for a, b in zip(f, f[1:])]
            fps_lanes[s] = {"launches": len(f), "start_us": round(f[0][2], 2), "end_us": round(f[-1][3], 2),
                            "busy_us": round(sum(k[3] - k[2] for k in f), 2), "gaps_us": gaps}
        g = [k for k in ks if k[1] in ("build", "query")]
        if g:
            knn_lanes[s] = {"launches": len(g), "start_us": round(g[0][2], 2), "end_us": round(g[-1][3], 2),
                            "busy_us": round(union_us([(k[2], k[3]) for k in g]), 2),
                            "query_us": round(sum(k[3] - k[2] for k in g if k[1] == "query"), 2)}
    query_iv = [(k[2], min(k[3], stage)) for ks in streams.values() for k in ks if k[1] == "query" and k[2] < stage]
    knn_iv = [(k[2], min(k[3], stage)) for ks in streams.values() for k in ks if k[1] in ("build", "query")]
    fps_iv = [(k[2], min(k[3], stage)) for ks in streams.values() for k in ks if k[1] == "fps"]
    counts = {}
    for ks in streams.values():
        for k in ks:
            counts[k[1]] = counts.get(k[1], 0) + 1
    return {
        "stage_us": round(stage, 2),
        "propagation_us": round(prop[0]["dur"], 2),
        "kernels": counts,
        "kernels_total": len(kern),
        "knn_end_us": round(max(b for _, b in knn_iv), 2),
        "fps_end_us": round(max(b for _, b in fps_iv), 2),
        "knn_busy_us": round(union_us(knn_iv), 2),
        "query_busy_us": round(union_us(query_iv), 2),
        "no_query_share": round(1.0 - union_us(query_iv) / stage, 4),
        "fps_lanes": fps_lanes,
        "knn_lanes": knn_lanes,
        "streams": {s: [[n, round(a, 2), round(b, 2)] for n, _, a, b in ks] for s, ks in streams.items()},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=20)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "trace_stage needs a GPU"
    cfg = CONFIGS[a.workload]
    dev = torch.device("cuda:0")
    xs = [scene(cfg["n"], cfg["seed"] + s).to(dev) for s in range(a.batch)]
    r = BatchGuidanceRunner(cfg["n"], a.batch, cfg["Q"], cfg["k"], cfg["radius"], cfg["max_step"], device=dev)
    for _ in range(4):
        r.run(xs)
    torch.cuda.synchronize()
    calls = [one_call(r, xs) for _ in range(a.calls)]
    for i, c in enumerate(calls):
        print("call %d: stage %.1f us (FPS ends %.1f, kNN ends %.1f), kNN busy %.1f us, query busy %.1f us, "
              "no query CTA running in %.1f %% of the stage, kernels %s" % (
                  i, c["stage_us"], c["fps_end_us"], c["knn_end_us"], c["knn_busy_us"], c["query_busy_us"],
                  100 * c["no_query_share"], c["kernels"]))
        for s, l in c["fps_lanes"].items():
            print("  stream %s FPS chain: %d launches %.1f..%.1f us, busy %.1f us, gaps %s" % (
                s, l["launches"], l["start_us"], l["end_us"], l["busy_us"], l["gaps_us"]))
        for s, l in c["knn_lanes"].items():
            print("  stream %s kNN: %d launches %.1f..%.1f us, busy %.1f us, query %.1f us" % (
                s, l["launches"], l["start_us"], l["end_us"], l["busy_us"], l["query_us"]))
    med = {key: statistics.median(c[key] for c in calls)
           for key in ("stage_us", "fps_end_us", "knn_end_us", "knn_busy_us", "query_busy_us", "no_query_share",
                       "propagation_us")}
    summary = {"library": os.environ.get("GF_LIB", "libgeoformer_b200.so"), "workload": a.workload,
               "scenes": a.batch, "calls": a.calls, "median": med, "kernels_per_call": calls[-1]["kernels_total"]}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"summary": summary, "calls": calls}, f, indent=1)
    print(json.dumps(summary))


if __name__ == "__main__":
    main()
