"""The fused mask head (geoformer_b200.mask_head) against the torch formulation, on one GPU.

  * config5_stage_split: FewShotForward (the config5_harness of bench.py: c2 scene, 100k points, Q = 256) timed per
    stage with CUDA events: aggregator, geodesic (k = 64, r = 0.05, 256 levels), decoder, mask head; the mask head
    both as the previous library ran it (epilogue a11 kernel + repeat / cat / two grouped conv1d in torch) and fused.
  * forward: Q = 256, m = 16 at N = 100k (the maps of that c2 scene) and N = 250k (synthetic maps): library op vs the
    torch formulation (epilogue in torch + the conv chain), time, peak memory, the share of the HBM bound (maps +
    features + coordinates read, logits written) and of the epilogue issue bound (6 instructions per (q, j, n)).
  * forward + backward: Q = 128 at N = 30k and 100k, library op vs torch autograd through the reference formulation.
Each case: CUDA events over repeated calls after warm-up; peak = torch.cuda.max_memory_allocated during one call
minus what was allocated before it.  The card's name, power limit and SM clock are read in the same run.

    python tools/measure_mask_head.py --out <dir>      -> <dir>/mask_head.json
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from geoformer_b200 import bias as gbias  # noqa: E402
from geoformer_b200.geodesic_utils import cal_geodesic_vectorize  # noqa: E402
from geoformer_b200.harness import FewShotForward, torch_mask_head_relative_coords  # noqa: E402
from geoformer_b200.mask_head import mask_heads_forward  # noqa: E402
from geoformer_b200.scenes import scene  # noqa: E402

M = 16


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


def torch_formulation(geo, feats, w, bs, coords, seeds, a11=False, row_max=None):
    """the reference's chain (:269-297): relative coordinates (torch, or the a11 kernel as the previous library did),
    repeat, cat, two grouped conv1d"""
    Q, N = geo.shape
    if a11:
        rel = gbias.mask_head_relative_coords(geo, coords, seeds, row_max=row_max)
    else:
        rel = torch_mask_head_relative_coords(geo, coords, seeds)
    x = torch.cat([rel, feats.t()[None].repeat(Q, 1, 1)], dim=1).reshape(1, -1, N)
    x = F.relu(F.conv1d(x, w[0], bias=bs[0], groups=Q))
    return F.conv1d(x, w[1], bias=bs[1], groups=Q).reshape(Q, N)


def params(Q, N, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    feats = torch.randn(N, M, generator=g).to(dev)
    w = [(torch.randn(Q * M, M + 3, 1, generator=g) * 0.3).to(dev), (torch.randn(Q, M, 1, generator=g) * 0.3).to(dev)]
    bs = [(torch.randn(Q * M, generator=g) * 0.1).to(dev), (torch.randn(Q, generator=g) * 0.1).to(dev)]
    return feats, w, bs


def bounds(Q, N, ms, clock_mhz, sms):
    hbm = (4 * Q * N + 4 * N * M + 4 * N * 3 + 4 * Q * N) / 6.5e12 * 1e3  # measured copy peak of the card
    issue = Q * N * M * 6 / (sms * 4 * 32 * clock_mhz * 1e6) * 1e3
    return {"hbm_bound_ms_at_6.5TBps": hbm, "epilogue_issue_bound_ms": issue, "share_of_hbm_bound": hbm / ms,
            "share_of_issue_bound": issue / ms, "binding_bound": "issue" if issue > hbm else "hbm"}


def stage_split(dev, reps):
    torch.manual_seed(5)
    net = FewShotForward().to(dev)
    N = 100_000
    locs = scene(N, 1234)[None].contiguous().to(dev)
    feats = torch.randn(1, N, 16, device=dev)
    support = torch.randn(1, 32, device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    acc = {k: 0.0 for k in ("aggregator", "geodesic", "decoder", "mask_head_previous", "mask_head_fused")}
    with torch.no_grad():
        for it in range(reps + 1):
            B = 1
            ev[0].record()
            pc_dims = [locs.min(dim=1)[0], locs.max(dim=1)[0]]
            mask_features = net.mask_tower(feats.transpose(1, 2)).transpose(1, 2)
            context_locs, context_feats, pre_enc_inds = net.forward_aggregator(locs, feats, "b200")
            query_locs = context_locs[:, : net.Q, :].contiguous()
            ev[1].record()
            offsets = torch.arange(B + 1, dtype=torch.int32) * N
            geo = cal_geodesic_vectorize(None, pre_enc_inds, locs.reshape(-1, 3).contiguous(), offsets, max_step=256,
                                         neighbor=64, radius=0.05, n_queries=net.Q)
            ev[2].record()
            se = support.unsqueeze(1)
            aggregation = torch.cat([context_feats * se, context_feats - se, context_feats], dim=2)
            dec = net.forward_decoder(context_locs, aggregation, query_locs, pc_dims, geo, pre_enc_inds, "b200")
            ev[3].record()
            # the previous library's mask head: a11 kernel + the torch chain
            pk = dec[-1].transpose(0, 1).flatten(0, 1)
            ctl = net.controller(net.before_embedding_tower(pk.unsqueeze(2))).squeeze(2).reshape(B, net.Q, -1)
            w0, w1, b0, b1 = torch.split_with_sizes(ctl[0], net.weight_nums + net.bias_nums, dim=1)
            w = [w0.reshape(net.Q * M, -1, 1), w1.reshape(net.Q, -1, 1)]
            bs = [b0.reshape(net.Q * M), b1.reshape(net.Q)]
            prev = torch_formulation(geo[0], mask_features[0], w, bs, locs[0], query_locs[0], a11=True)
            ev[4].record()
            new = net.mask_logits(geo, dec[-1], mask_features, locs, query_locs, None, "b200")[0]
            ev[5].record()
            torch.cuda.synchronize(dev)
            if it == 0:
                continue
            for k, (i, j) in zip(acc, [(0, 1), (1, 2), (2, 3), (3, 4), (4, 5)]):
                acc[k] += ev[i].elapsed_time(ev[j]) / reps
    acc["mask_logit_max_abs_diff_fused_vs_previous"] = (new - prev).abs().max().item()
    acc["mask_logit_scale"] = prev.abs().max().item()
    acc["b200_path_previous_ms"] = acc["aggregator"] + acc["geodesic"] + acc["decoder"] + acc["mask_head_previous"]
    acc["b200_path_fused_ms"] = acc["aggregator"] + acc["geodesic"] + acc["decoder"] + acc["mask_head_fused"]
    acc["mask_head_share_previous"] = acc["mask_head_previous"] / acc["b200_path_previous_ms"]
    acc["note"] = ("stages of FewShotForward.forward, impl='b200', one c2 scene; the mask head includes the controller "
                   "(before_embedding_tower + controller convs) in both arms")
    return acc, geo[0], locs[0], query_locs[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = card()
    clock = float(info["max_sm_clock"].split()[0])
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    res = {"card": info, "sms": sms, "torch": torch.__version__,
           "cudnn_conv_tf32": torch.backends.cudnn.allow_tf32}
    split, geo_c2, locs_c2, seeds_c2 = stage_split(dev, 5)
    res["config5_stage_split"] = split
    print(json.dumps(split), flush=True)

    fwd = {}
    for N in (100_000, 250_000):
        Q = 256
        feats, w, bs = params(Q, N, dev)
        if N == 100_000:
            geo, coords, seeds, src = geo_c2, locs_c2, seeds_c2, "maps of the c2 scene, k=64 r=0.05 256 levels"
        else:
            g = torch.Generator().manual_seed(1)
            coords = scene(N, 99).to(dev)
            geo = (torch.rand(Q, N, generator=g) * 3).to(dev)
            geo[(torch.rand(Q, N, generator=g) < 0.4).to(dev)] = -1
            seeds = coords[:Q].contiguous()
            src = "synthetic maps, 40 % unreachable"
        lib = timed(lambda: mask_heads_forward(geo, feats, w, bs, Q, coords, seeds), args.reps, dev)
        ref = timed(lambda: torch_formulation(geo, feats, w, bs, coords, seeds), max(3, args.reps // 4), dev)
        a = mask_heads_forward(geo, feats, w, bs, Q, coords, seeds)
        b = torch_formulation(geo, feats, w, bs, coords, seeds)
        lib.update(bounds(Q, N, lib["ms"], clock, sms))
        fwd["Q%d_N%d" % (Q, N)] = {"maps": src, "library": lib, "torch_formulation": ref, "speedup": ref["ms"] / lib["ms"],
                                   "max_abs_diff": (a - b).abs().max().item(), "scale": b.abs().max().item()}
        print(json.dumps(fwd["Q%d_N%d" % (Q, N)]), flush=True)
        del a, b
    res["forward"] = fwd

    fb = {}
    for N in (30_000, 100_000):
        Q = 128
        feats, w, bs = params(Q, N, dev, seed=2)
        g = torch.Generator().manual_seed(3)
        coords = scene(N, 5).to(dev)
        geo = (torch.rand(Q, N, generator=g) * 3).to(dev)
        geo[(torch.rand(Q, N, generator=g) < 0.4).to(dev)] = -1
        seeds = coords[:Q].contiguous()
        dl = torch.randn(Q, N, generator=g).to(dev)
        leaves = [t.clone().requires_grad_() for t in [feats] + w + bs]

        def lib_fb():
            y = mask_heads_forward(geo, leaves[0], leaves[1:3], leaves[3:5], Q, coords, seeds)
            return torch.autograd.grad(y, leaves, dl)

        def ref_fb():
            y = torch_formulation(geo, leaves[0], leaves[1:3], leaves[3:5], coords, seeds)
            return torch.autograd.grad(y, leaves, dl)

        lib = timed(lib_fb, args.reps, dev)
        ref = timed(ref_fb, max(3, args.reps // 2), dev)
        ga, gb = lib_fb(), ref_fb()
        errs = {n: ((x - y).norm() / y.norm()).item() for n, x, y in zip(("feats", "w0", "w1", "b0", "b1"), ga, gb)}
        fb["Q%d_N%d" % (Q, N)] = {"library": lib, "torch_autograd": ref, "speedup": ref["ms"] / lib["ms"],
                                  "grad_rel_frobenius_vs_torch": errs}
        print(json.dumps(fb["Q%d_N%d" % (Q, N)]), flush=True)
    res["forward_backward"] = fb
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "mask_head.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
