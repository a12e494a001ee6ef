"""The set aggregator on ragged batches (scenes of different sizes, flat points + offsets): the model's module (2048
centres, r = 0.2, nsample 64, widths 19 -> 32 -> 32 -> 32, max pooling) timed with CUDA events after warm-up, with
the peak memory of each arm, on batches of B in {1, 4, 8, 16} scenes of 60k-150k points (scenes.scene, fixed seeds)
and one batch with a 250k-point scene (beyond one cluster).  Arms:

    inference (eval mode, no grad)
        loop       aggregate() per scene + cat (what a caller without aggregate_batch does)
        torch      the reference's formulation: per-scene FPS / gather / ball query / group, cat, one mlp, max pool
        batch      aggregate_batch
    training forward + backward (train mode, gradient to the features)
        torch      the formulation above under autograd
        batch      aggregate_batch
    FPS alone: B single-scene launches against one ragged call

The card's name, power limit and max SM clock are read in the same run.  Writes OUT/aggregate_batch.json.

    python tools/measure_aggregate_batch.py [--reps 5] [--out profiles/r11]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from geoformer_b200 import aggregate as agg  # noqa: E402
from geoformer_b200.harness import FewShotForward  # noqa: E402
from geoformer_b200.pointnet2 import _ext  # noqa: E402
from geoformer_b200.scenes import scene  # noqa: E402


def timed(fn, reps):
    """ms per call (median of reps, each one call between events) and peak memory above the start, MiB"""
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return {"ms": float(np.median(ms)), "ms_all": ms,
            "peak_mib": (torch.cuda.max_memory_allocated() - base) / 2 ** 20}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False  # the torch arm in fp32, as the library computes
    torch.manual_seed(0)
    net = FewShotForward(m=16).to(dev)  # its aggregator is the model's: 2048 centres, r 0.2, ns 64, 19 -> 32 x 3
    batches = {}
    for B in (1, 4, 8, 16):
        batches["B%d" % B] = np.random.default_rng(B).integers(60_000, 150_001, size=B).tolist()
    batches["B4_with_250k"] = [250_000] + np.random.default_rng(40).integers(60_000, 150_001, size=3).tolist()
    res = {"card": card(), "module": "2048 centres, r 0.2, nsample 64, widths 19-32-32-32, max", "batches": {}}
    print(res["card"])
    for name, Ns in batches.items():
        locs = torch.cat([scene(n, 500 + i) for i, n in enumerate(Ns)]).to(dev)
        feats = torch.randn(sum(Ns), 16, device=dev)
        off = [0] + np.cumsum(Ns).tolist()
        r = {"N": Ns}

        def loop():
            outs = [net.forward_aggregator(locs[s:e][None], feats[s:e][None], "b200") for s, e in zip(off, off[1:])]
            return [torch.cat(t) for t in zip(*outs)]

        net.eval()
        with torch.no_grad():
            r["infer_loop"] = timed(loop, a.reps)
            r["infer_torch"] = timed(lambda: net.forward_aggregator_batch(locs, feats, off, "torch"), a.reps)
            r["infer_batch"] = timed(lambda: net.forward_aggregator_batch(locs, feats, off, "b200"), a.reps)
            same = all(torch.equal(x, y) for x, y in zip(loop(), net.forward_aggregator_batch(locs, feats, off, "b200")))
            r["infer_batch_equals_loop"] = bool(same)
        net.train()
        f = feats.clone().requires_grad_()

        def train(impl):
            def step():
                _, out, _ = net.forward_aggregator_batch(locs, f, off, impl)
                out.sum().backward()
            return step

        r["train_torch"] = timed(train("torch"), a.reps)
        r["train_batch"] = timed(train("b200"), a.reps)
        net.zero_grad(set_to_none=True)
        r["fps_single_launches"] = timed(
            lambda: [_ext.furthest_point_sampling(locs[s:e][None], 2048) for s, e in zip(off, off[1:])], a.reps)
        r["fps_ragged_call"] = timed(lambda: agg.furthest_point_sampling_batch(locs, off, 2048), a.reps)
        res["batches"][name] = r
        print("%-13s loop %7.2f  torch %7.2f  batch %7.2f ms | train torch %7.2f  batch %7.2f ms | "
              "fps %7.2f -> %7.2f ms | peak MiB train torch %.0f batch %.0f" % (
                  name, r["infer_loop"]["ms"], r["infer_torch"]["ms"], r["infer_batch"]["ms"], r["train_torch"]["ms"],
                  r["train_batch"]["ms"], r["fps_single_launches"]["ms"], r["fps_ragged_call"]["ms"],
                  r["train_torch"]["peak_mib"], r["train_batch"]["peak_mib"]), flush=True)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "aggregate_batch.json"), "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
