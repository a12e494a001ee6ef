"""Forward + backward of the decoder vector cross-attention at the training shape (Q=128 queries, C=2048 contexts,
B=1 and 4) and the eval shape (Q=256, C=2048, B=1): the library (embedding given / fused) against the torch
formulation (oracle.attention's op sequence under autograd, fp32, same GPU).  Per arm: fwd+bwd time from CUDA events
after warm-up, peak memory (torch.cuda.max_memory_allocated, reset between arms, inputs included), and the max error
of every gradient against the torch arm relative to its scale; then the backward kernel alone from torch.profiler.

    python tools/measure_attention_backward.py --out <dir>      -> <dir>/attention_backward.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import attention as oatt  # noqa: E402

from geoformer_b200 import _capi  # noqa: E402
from geoformer_b200.attention import rel_cross_attention, rel_cross_attention_fused  # noqa: E402
from geoformer_b200.bias import decoder_relative_embedding  # noqa: E402
from geoformer_b200.scenes import scene  # noqa: E402

WN = ("w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo")


def make_case(Q, Cn, B, dev, N=100_000):
    gen = torch.Generator().manual_seed(Q + 10 * B)
    w = {k: (torch.randn(64, 64, generator=gen) * 0.125 if k[0] == "w" else torch.randn(64, generator=gen) * 0.1).to(dev)
         for k in WN}
    geos, inds, ctxs = [], [], []
    pmin, pmax = [], []
    for b in range(B):
        x = scene(N, 1234 + b)
        g = torch.rand(Q, N, generator=gen) * 4
        g[torch.rand(Q, N, generator=gen) < 0.5] = -1
        geos.append(g.to(dev))
        i = torch.randperm(N, generator=gen)[:Cn].int()
        inds.append(i)
        ctxs.append(x[i.long()])
        pmin.append(x.min(0)[0])
        pmax.append(x.max(0)[0])
    ctx = torch.stack(ctxs).contiguous()
    args = (geos, torch.stack(inds).to(dev), ctx[:, :Q].contiguous().to(dev), ctx.to(dev),
            torch.randn(3, 32, generator=gen).to(dev), [torch.stack(pmin).to(dev), torch.stack(pmax).to(dev)])
    tgt2 = torch.randn(Q, B, 64, generator=gen).to(dev)
    mem = torch.randn(Cn, B, 64, generator=gen).to(dev)
    dy = torch.randn(Q, B, 64, generator=gen).to(dev)
    emb = decoder_relative_embedding(*args).contiguous()
    return w, args, tgt2, mem, dy, emb


def arm(kind, w, args, tgt2, mem, dy, emb):
    """one forward + backward; returns the gradients of tgt2, memory and the weights"""
    wl = {k: v.detach().clone().requires_grad_() for k, v in w.items()}
    t, m = tgt2.detach().clone().requires_grad_(), mem.detach().clone().requires_grad_()
    if kind == "library":
        y = rel_cross_attention(t, m, emb, wl)
    elif kind == "library_fused":
        y = rel_cross_attention_fused(t, m, *args, wl)
    else:
        y = oatt.rel_cross_attention(t, m, emb, wl)
    g = torch.autograd.grad(y, [t, m] + [wl[k] for k in WN], dy)
    return dict(zip(("tgt2", "memory") + WN, g))


def time_ms(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        info["nvidia_smi"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                                            capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def backward_kernel_us(case, fused, reps=5):
    """the tcgen05 backward kernel alone (torch.profiler, CUDA activity), mean over `reps` backward passes"""
    from torch.profiler import ProfilerActivity, profile

    w, args, tgt2, mem, dy, emb = case
    kind = "library_fused" if fused else "library"
    arm(kind, *case)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            arm(kind, *case)
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            tot[e.name] = tot.get(e.name, 0.0) + e.device_time
    out = {n.split("(")[0][:80]: round(v / reps, 2) for n, v in tot.items()
           if "rel_cross_attention" in n or n.startswith("att_")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    opt = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    res = {"gpu": gpu_info(), "shapes": []}
    for Q, Cn, B in ((128, 2048, 1), (128, 2048, 4), (256, 2048, 1)):
        case = make_case(Q, Cn, B, dev)
        row = {"Q": Q, "C": Cn, "B": B}
        grads = {}
        for kind in ("torch", "library", "library_fused"):
            torch.cuda.synchronize()
            _capi.workspace = _capi.Workspace()  # each arm pays for its own scratch buffers
            torch.cuda.empty_cache()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            grads[kind] = arm(kind, *case)
            torch.cuda.synchronize()
            row["peak_mb_" + kind] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)
            row["fwd_bwd_ms_" + kind] = round(time_ms(lambda: arm(kind, *case), opt.reps if kind != "torch" else 5), 4)
        for kind in ("library", "library_fused"):
            row["max_rel_err_" + kind] = {k: float((grads[kind][k] - g).abs().max() / g.abs().max().clamp_min(1e-30))
                                          for k, g in grads["torch"].items() if k != "b2"}
        with torch.no_grad():
            wd = case[0]
            row["fwd_ms_library"] = round(time_ms(lambda: rel_cross_attention(case[2], case[3], case[5], wd), opt.reps), 4)
            row["fwd_ms_library_fused"] = round(time_ms(lambda: rel_cross_attention_fused(case[2], case[3], *case[1], wd),
                                                        opt.reps), 4)
        row["backward_kernels_us_library"] = backward_kernel_us(case, False)
        row["backward_kernels_us_library_fused"] = backward_kernel_us(case, True)
        row["speedup_fwd_bwd_fused_vs_torch"] = round(row["fwd_bwd_ms_torch"] / row["fwd_bwd_ms_library_fused"], 2)
        print(json.dumps(row), flush=True)
        res["shapes"].append(row)
        del case, grads
    res["note"] = ("peak_mb: torch.cuda.max_memory_allocated during one fwd+bwd above what was allocated before it "
                   "(the library's workspace included); errors relative to the max |g| of "
                   "the fp32 torch arm")
    os.makedirs(opt.out, exist_ok=True)
    with open(os.path.join(opt.out, "attention_backward.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
