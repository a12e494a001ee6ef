"""The fused mask head on ragged batches: B single-scene calls (the loop FewShotForward.mask_logits ran per scene)
against one mask_heads_forward_batch call, timed with CUDA events (median of repeated calls after warm-up), with the
per-call library launches of the forward and the peak memory of each arm, on batches of B in {1, 4, 8, 16} scenes:

    fwd_q256        forward (no grad), Q = 256, scenes of 60k-150k points (scenes.scene, fixed seeds)
    train_q128      forward + backward, Q = 128, scenes of 60k-150k points
    train_q128_30k  forward + backward, Q = 128, 30k-point scenes (the training shape of DESIGN 4.5d)

The maps are synthetic (30 % unreachable); the kernels' work does not depend on their values.  Both arms compute
bitwise-equal logits (checked here).  The card's name, power limit and max SM clock are read in the same run.
Writes OUT/mask_head_batch.json.

    python tools/measure_mask_head_batch.py [--reps 10] [--out profiles/r15]
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
from geoformer_b200 import _capi  # noqa: E402
from geoformer_b200 import mask_head as mh  # noqa: E402
from geoformer_b200.scenes import scene  # noqa: E402

M = 16


def timed(fn, reps):
    """ms per call (median of reps, each one call between events), library launches of one call on this thread (the
    forward: autograd runs the backward on a thread of its own), and peak memory above the start, MiB"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    _capi.reset_launch_count()
    fn()
    torch.cuda.synchronize()
    launches = _capi.launch_count()
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
    return {"ms": float(np.median(ms)), "ms_all": ms, "fwd_launches": launches,
            "peak_mib": (torch.cuda.max_memory_allocated() - base) / 2 ** 20}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def inputs(Ns, Q, seed, dev):
    gen = torch.Generator().manual_seed(seed)
    B, off = len(Ns), [0] + np.cumsum(Ns).tolist()
    coords = torch.cat([scene(n, 700 + seed + i) for i, n in enumerate(Ns)]).to(dev)
    geo = []
    for n in Ns:
        g = torch.rand(Q, n, generator=gen) * 3
        g[torch.rand(Q, n, generator=gen) < 0.3] = -1.0
        geo.append(g.to(dev))
    feats = torch.randn(off[-1], M, generator=gen).to(dev)
    w0 = (torch.randn(B * Q * M, M + 3, 1, generator=gen) * 0.3).to(dev)
    w1 = (torch.randn(B * Q, M, 1, generator=gen) * 0.3).to(dev)
    b0 = (torch.randn(B * Q * M, generator=gen) * 0.1).to(dev)
    b1 = (torch.randn(B * Q, generator=gen) * 0.1).to(dev)
    seeds = torch.stack([coords[off[b]:off[b + 1]][:Q] for b in range(B)]).contiguous()
    return geo, feats, off, [w0, w1], [b0, b1], coords, seeds


def arms(geo, feats, off, weights, biases, coords, seeds):
    """loop(): the per-scene calls; batch(): the batched call"""
    B, Q = seeds.shape[:2]
    (w0, w1), (b0, b1) = weights, biases

    def loop():
        return [mh.mask_heads_forward(geo[b], feats[s:e], [w0[b * Q * M:(b + 1) * Q * M], w1[b * Q:(b + 1) * Q]],
                                      [b0[b * Q * M:(b + 1) * Q * M], b1[b * Q:(b + 1) * Q]], Q, coords[s:e],
                                      seeds[b]) for b, (s, e) in enumerate(zip(off, off[1:]))]

    def batch():
        return mh.mask_heads_forward_batch(geo, feats, off, weights, biases, coords, seeds)

    return loop, batch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r15"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    res = {"card": card(), "sms": torch.cuda.get_device_properties(dev).multi_processor_count, "shapes": {}}
    print(res["card"], flush=True)
    for shape, Q, train, big in (("fwd_q256", 256, False, True), ("train_q128", 128, True, True),
                                 ("train_q128_30k", 128, True, False)):
        res["shapes"][shape] = {}
        for B in (1, 4, 8, 16):
            Ns = np.random.default_rng(B).integers(60_000, 150_001, size=B).tolist() if big else [30_000] * B
            geo, feats, off, weights, biases, coords, seeds = inputs(Ns, Q, B, dev)
            r = {"N": Ns, "Q": Q}
            if train:
                feats.requires_grad_()
                for t in weights + biases:
                    t.requires_grad_()
                params = [feats] + weights + biases
                wl = [torch.randn(Q, n, device=dev) for n in Ns]
                loop, batch = arms(geo, feats, off, weights, biases, coords, seeds)

                def step(fn):
                    def run():
                        out = fn()
                        torch.autograd.grad(sum((o * w).sum() for o, w in zip(out, wl)), params)
                    return run

                r["loop"], r["batch"] = timed(step(loop), a.reps), timed(step(batch), a.reps)
                with torch.no_grad():
                    same = all(torch.equal(x, y) for x, y in zip(loop(), batch()))
            else:
                loop, batch = arms(geo, feats, off, weights, biases, coords, seeds)
                with torch.no_grad():
                    r["loop"], r["batch"] = timed(loop, a.reps), timed(batch, a.reps)
                    same = all(torch.equal(x, y) for x, y in zip(loop(), batch()))
            r["batch_equals_loop"] = bool(same)
            r["speedup"] = r["loop"]["ms"] / r["batch"]["ms"]
            res["shapes"][shape]["B%d" % B] = r
            print("%-15s B=%2d loop %8.2f ms (%3d fwd launches)  batch %8.2f ms (%d fwd launches)  x%.3f  equal %s  "
                  "peak MiB %.0f / %.0f" % (shape, B, r["loop"]["ms"], r["loop"]["fwd_launches"], r["batch"]["ms"],
                                            r["batch"]["fwd_launches"], r["speedup"], same, r["loop"]["peak_mib"],
                                            r["batch"]["peak_mib"]), flush=True)
            del geo, feats, weights, biases, coords, seeds, loop, batch
            torch.cuda.empty_cache()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "mask_head_batch.json"), "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
