"""The set aggregator in training form (geoformer_b200.aggregate.group_mlp_pool_train) against torch autograd, on one GPU.

  * Model shape: N = 100k foreground points (scenes.scene), 2048 FPS centres, r = 0.2, ns = 64, SharedMLP
    19 -> 32 -> 32 -> 32 with batch norm in training mode, max pooling, B = 1 and 4 scenes.
  * forward (training mode: batch statistics, running statistics updated) and forward + backward (gradients of the
    weights, gamma, beta and the features), library op vs the reference formulation in torch: the library's
    ball_query / grouping_operation (autograd through group_points_grad), then train-mode nn.Conv2d / BatchNorm2d /
    ReLU modules (cuDNN with torch's default settings) and max_pool2d.  Time and peak memory of each.
  * share of the issue bound: warp instructions counted from shapes -- 64 per sample and layer evaluated (32 SHFL +
    32 FFMA), 94 per sample and layer backpropagated (the transposing warp reduction: 31 SHFL + 31 FADD + 32 FMUL),
    64 per sample for the weight-gradient accumulation of a backward pass -- over 148 SMs x 4 schedulers x the max SM
    clock.  Every sample is counted in every pass (batch statistics make every sample carry gradient).
  * one FewShotForward.forward_train step + backward (n_query_points = 128, max_step = 128, B = 1, N = 100k) with each
    impl.
The ball query is computed once per shape, outside the timed calls (it is the same call in both formulations; its
time is reported on its own).  Each case: CUDA events over repeated calls after warm-up; peak =
torch.cuda.max_memory_allocated during one call minus what was allocated before it; the library's grow-only workspace
(allocated by the warm-up call) is reported as library_workspace_mb and added to its peak in the peak ratio.  The card's name, power limit and max SM clock are read in the same run.

    python tools/measure_aggregate_train.py --out <dir>      -> <dir>/aggregate_train.json
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch
import torch.nn as nn
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from geoformer_b200 import _capi as C  # noqa: E402
from geoformer_b200 import pointnet2_utils as pu  # noqa: E402
from geoformer_b200.aggregate import group_mlp_pool_train  # noqa: E402
from geoformer_b200.harness import FewShotForward  # noqa: E402
from geoformer_b200.pointnet2 import _ext  # noqa: E402
from geoformer_b200.scenes import scene  # noqa: E402

N, M_CENTRES, NS, CF, R = 100_000, 2048, 64, 16, 0.2
WIDTHS = [19, 32, 32, 32]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, reps, dev):
    fn()
    torch.cuda.synchronize(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    fn()
    torch.cuda.synchronize(dev)
    peak = torch.cuda.max_memory_allocated(dev) - base
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize(dev)
    return {"ms": a.elapsed_time(b) / reps, "peak_mb": peak / 2**20}


def issue_instructions(B, L=3):
    """warp instructions of the library's passes at the model shape, counted from shapes (see the module docstring)"""
    samples = B * M_CENTRES * NS
    fwd = 64 * (sum(l + 1 for l in range(L)) + L)  # statistics pass l evaluates l + 1 layers, then the output pass
    bwd = 0
    for p in range(L, -1, -1):
        bwd += 64 * L + (64 * L if p == L else 0)  # recompute (and the argmax loop of pass L)
        bwd += 94 * (L - p) + (64 if p < L else 0)  # backpropagation to layer p, dW_p
    return {"forward": fwd * samples, "backward": bwd * samples}


def mlp_module(dev):
    def conv_bn(cin, cout):
        return nn.Sequential(nn.Conv2d(cin, cout, 1, bias=False), nn.Sequential(nn.BatchNorm2d(cout)), nn.ReLU())

    return nn.Sequential(*[conv_bn(WIDTHS[i], WIDTHS[i + 1]) for i in range(3)]).to(dev).train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    dev = torch.device("cuda:0")
    info = card()
    clock_hz = float(info["max_sm_clock"].split()[0]) * 1e6
    issue_rate = torch.cuda.get_device_properties(dev).multi_processor_count * 4 * clock_hz
    res = {"card": info, "shape": {"N": N, "m": M_CENTRES, "nsample": NS, "radius": R, "widths": WIDTHS,
                                   "pooling": "max"}, "cases": []}
    torch.manual_seed(0)
    for B in (1, 4):
        xyz = torch.stack([scene(N, 10 + b) for b in range(B)]).to(dev).contiguous()
        feats = torch.randn(B, CF, N, device=dev)
        inds = _ext.furthest_point_sampling(xyz, M_CENTRES)
        new_xyz = _ext.gather_points(xyz.transpose(1, 2).contiguous(), inds).transpose(1, 2).contiguous()
        mod = mlp_module(dev)
        layers = [(l[0], l[1][0]) for l in mod]

        idx = _ext.ball_query(new_xyz, xyz, R, NS)

        def lib_fwd(f):
            return group_mlp_pool_train(xyz, new_xyz, f, idx, R, True, True, [c.weight for c, _ in layers], None,
                                        [b.weight for _, b in layers], [b.bias for _, b in layers],
                                        [b.running_mean for _, b in layers], [b.running_var for _, b in layers], True,
                                        momentum=0.1, num_batches_tracked=[b.num_batches_tracked for _, b in layers])

        def torch_fwd(f):
            g_xyz = pu.grouping_operation(xyz.transpose(1, 2).contiguous(), idx)
            g_xyz = (g_xyz - new_xyz.transpose(1, 2).unsqueeze(-1)) / R
            x = mod(torch.cat([g_xyz, pu.grouping_operation(f, idx)], dim=1))
            return F.max_pool2d(x, kernel_size=[1, x.size(3)]).squeeze(-1)

        fr = feats.clone().requires_grad_()
        dy = torch.randn(B, 32, M_CENTRES, device=dev)
        params = [fr] + list(mod.parameters())
        lib = C.lib()
        ws_mb = (lib.gf_group_mlp_pool_train_workspace_bytes(B, M_CENTRES)
                 + lib.gf_group_mlp_pool_backward_workspace_bytes(B, N, M_CENTRES, NS, CF)) / 2**20
        case = {"B": B, "ball_query": timed(lambda: _ext.ball_query(new_xyz, xyz, R, NS), args.reps, dev),
                "library_workspace_mb": ws_mb}
        for name, fwd in (("library", lib_fwd), ("torch", torch_fwd)):
            def f_only():
                with torch.no_grad():
                    fwd(feats)

            def f_b():
                torch.autograd.grad(fwd(fr), params, dy)

            case[name] = {"forward": timed(f_only, args.reps, dev), "forward_backward": timed(f_b, args.reps, dev)}
        ins = issue_instructions(B)
        bound_f = ins["forward"] / issue_rate * 1e3
        bound_fb = (ins["forward"] + ins["backward"]) / issue_rate * 1e3
        case["issue_bound"] = {"warp_instructions": ins, "forward_ms": bound_f, "forward_backward_ms": bound_fb,
                               "share_forward": bound_f / case["library"]["forward"]["ms"],
                               "share_forward_backward": bound_fb / case["library"]["forward_backward"]["ms"]}
        case["speedup_forward_backward"] = case["torch"]["forward_backward"]["ms"] / case["library"]["forward_backward"]["ms"]
        # the library's grow-only workspace is allocated by the warm-up call: counted here on top of the peak
        case["peak_ratio_forward_backward"] = (case["torch"]["forward_backward"]["peak_mb"]
                                               / (case["library"]["forward_backward"]["peak_mb"] + ws_mb))
        print(json.dumps(case))
        res["cases"].append(case)
        del xyz, feats, fr

    # one training step of the post-backbone path
    base = FewShotForward(n_query_points=128).to(dev).train()
    locs = scene(N, 77)[None].to(dev).contiguous()
    out_feats = torch.randn(1, N, 16, device=dev)
    se = torch.randn(1, 32, device=dev)
    wl = torch.randn(128, N, device=dev)
    step = {}
    for impl in ("b200", "torch"):
        model = copy.deepcopy(base)

        def one():
            logits, _, _ = model.forward_train(locs, out_feats, se, impl=impl, max_step=128)
            ((logits[0] * wl).sum() / N).backward()

        step[impl] = timed(one, max(3, args.reps // 4), dev)
    res["forward_train_step"] = {"B": 1, "N": N, "n_query_points": 128, "max_step": 128, **step}
    print(json.dumps(res["forward_train_step"]))
    with open(os.path.join(args.out, "aggregate_train.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
