"""Propagation over the caller's own kNN graphs (the faiss layout: sqrt'ed f32 distances, int64 indices), for batches
of B scenes, three arms timed alternately with CUDA events (median of the repeated calls after warm-up):

    loop    one geodesic_from_graph call per scene (what cal_geodesic_vectorize ran for a foreign index before)
    orig    one gf_geodesic_batch call in the ORIGINAL point numbering: a development build of the library
            (GF_GEO_ORIGINAL_ORDER: no grid build, rank / order null), loaded next to the product library
    cell    one gf_geodesic_batch call in the cell order of a kNN grid over the scene's points (the product)

and cal_geodesic_vectorize end to end with a stand-in index (add / search / reset, not a FlatL2Index, so it takes the
index branch): `before` restates that branch's per-scene loop, `after` is the current function.  Workloads:

    c2      scenes.scene(100_000, s), Q = 256, k = 16, r = 0.5, 32 levels              B in {1, 4, 8, 20}
    eval    60k-150k-point scenes (as tools/measure_mask_head_batch.py), Q = 256, k = 64, r = 0.05, max_step 256
                                                                                        B in {1, 4, 8}
    train   the same scenes, Q = 128, k = 64, r = 0.05, max_step 128                    B in {4, 8}

Graphs come from knn_graph (int64) and are built outside the timed region; seeds are random points of each scene.
The maps of all arms are compared bitwise.  Peak memory above the start of each arm (outputs, and for
cal_geodesic_vectorize the B graphs alive at once) and the workspace of the batched call are reported.  The card's
name, power limit and max SM clock are read in the same run.  Writes OUT/geodesic_graph_batch.json.

    python -m geoformer_b200.build --variant=orignum -DGF_GEO_ORIGINAL_ORDER    # the development build
    python tools/measure_geodesic_graph_batch.py [--reps 10] [--out profiles/r16]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from geoformer_b200 import _capi as C  # noqa: E402
from geoformer_b200 import geodesic_utils as gu  # noqa: E402
from geoformer_b200.scenes import scene  # noqa: E402

ORIG_LIB = os.path.join(ROOT, "geoformer_b200", "libgeoformer_b200_orignum.so")


def load_variant(path):
    h = ctypes.CDLL(path)
    for name, (res, args) in C.SIGNATURES.items():
        fn = getattr(h, name)
        fn.restype = res
        fn.argtypes = args
    return h


class StandIn:
    """an index with the faiss protocol that is not a FlatL2Index: cal_geodesic_vectorize takes the index branch"""

    def __init__(self):
        self._ix = gu.FlatL2Index()

    def add(self, x):
        self._ix.add(x)

    def search(self, q, k, D, I):
        return self._ix.search(q, k, D, I)

    def reset(self):
        self._ix.reset()


def cal_before(index, pre, locs, offs, max_step, neighbor, radius, n_queries):
    """cal_geodesic_vectorize's index branch as it was: kNN then propagation, scene after scene"""
    out = []
    for b in range(len(offs) - 1):
        x = locs[offs[b]:offs[b + 1]].contiguous()
        D, I = gu.find_knn(index, x, neighbor=neighbor)
        out.append(gu.geodesic_from_graph(D, I, pre[b][:n_queries], radius, max_step))
    return out


def timed_alternating(arms, reps):
    """arms: name -> (fn, lib).  ms per call (median), launches of one call, peak MiB above the start of a call"""
    res = {}
    for name, (fn, lib) in arms.items():  # warm-up (module loads, kernel attributes, workspace growth)
        C._lib = lib
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        lib.gf_reset_launch_count()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = fn()
        torch.cuda.synchronize()
        res[name] = {"launches": int(lib.gf_launch_count()),
                     "peak_mib": (torch.cuda.max_memory_allocated() - base) / 2 ** 20, "ms_all": [], "out": out}
    for _ in range(reps):
        for name, (fn, lib) in arms.items():
            C._lib = lib
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            res[name]["ms_all"].append(a.elapsed_time(b))
    for r in res.values():
        r["ms"] = float(np.median(r["ms_all"]))
    return res


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r16"))
    ap.add_argument("--orig-lib", default=ORIG_LIB)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda:0")
    prod, orig = C.lib(), load_variant(a.orig_lib)
    res = {"card": card(), "sms": torch.cuda.get_device_properties(dev).multi_processor_count, "workloads": {}}
    print(res["card"], flush=True)
    workloads = (("c2", 256, 16, 0.5, 32, (1, 4, 8, 20)), ("eval", 256, 64, 0.05, 256, (1, 4, 8)),
                 ("train", 128, 64, 0.05, 128, (4, 8)))
    for wl, Q, k, r, ms, Bs in workloads:
        res["workloads"][wl] = {}
        for B in Bs:
            if wl == "c2":
                Ns = [100_000] * B
                pts = [scene(100_000, 1234 + i).to(dev) for i in range(B)]
            else:
                Ns = np.random.default_rng(B).integers(60_000, 150_001, size=B).tolist()
                pts = [scene(n, 700 + B + i).to(dev) for i, n in enumerate(Ns)]
            gen = torch.Generator().manual_seed(B)
            seeds = [torch.randint(0, n, (Q,), generator=gen).int().to(dev) for n in Ns]
            graphs = [gu.knn_graph(x, k) for x in pts]
            torch.cuda.synchronize()

            def loop():
                return [gu.geodesic_from_graph(D, I, s, r, ms) for (D, I), s in zip(graphs, seeds)]

            def batch():
                return gu.geodesic_from_graph_batch(pts, graphs, seeds, r, ms)

            t = timed_alternating({"loop": (loop, prod), "orig": (batch, orig), "cell": (batch, prod)}, a.reps)
            C._lib = prod
            same = all(torch.equal(x, y) for arm in ("orig", "cell") for x, y in zip(t["loop"]["out"], t[arm]["out"]))
            for v in t.values():
                del v["out"]
            Nc = (ctypes.c_int * B)(*Ns)
            rec = {"N": Ns, "Q": Q, "k": k, "radius": r, "max_step": ms, "arms": t, "maps_equal": bool(same),
                   "workspace_mib": prod.gf_geodesic_batch_workspace_bytes(Nc, B, Q, k) / 2 ** 20}
            del graphs
            torch.cuda.empty_cache()
            # cal_geodesic_vectorize end to end over the stand-in index
            locs = torch.cat(pts).contiguous()
            offs = [0] + np.cumsum(Ns).tolist()
            pre = torch.stack(seeds)
            ix = StandIn()
            e2e = timed_alternating({
                "before": (lambda: cal_before(ix, pre, locs, offs, ms, k, r, Q), prod),
                "after": (lambda: gu.cal_geodesic_vectorize(ix, pre, locs, torch.tensor(offs), max_step=ms,
                                                            neighbor=k, radius=r, n_queries=Q), prod)}, a.reps)
            rec["cal_equal"] = all(torch.equal(x, y) for x, y in zip(e2e["before"]["out"], e2e["after"]["out"]))
            for v in e2e.values():
                del v["out"]
            rec["cal_geodesic_vectorize"] = e2e
            res["workloads"][wl]["B%d" % B] = rec
            print("%-5s B=%2d loop %8.3f ms (%3d launches, %6.0f MiB)  orig %8.3f ms (%d)  cell %8.3f ms (%d, %6.0f MiB, "
                  "ws %5.0f MiB)  equal %s | cal_geodesic_vectorize before %8.3f ms (%5.0f MiB)  after %8.3f ms "
                  "(%5.0f MiB)  equal %s" % (
                      wl, B, t["loop"]["ms"], t["loop"]["launches"], t["loop"]["peak_mib"], t["orig"]["ms"],
                      t["orig"]["launches"], t["cell"]["ms"], t["cell"]["launches"], t["cell"]["peak_mib"],
                      rec["workspace_mib"], same, e2e["before"]["ms"], e2e["before"]["peak_mib"], e2e["after"]["ms"],
                      e2e["after"]["peak_mib"], rec["cal_equal"]), flush=True)
            del pts, seeds, locs, pre
            torch.cuda.empty_cache()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "geodesic_graph_batch.json"), "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
