"""A/B of furthest point sampling alone between two builds of the library, loaded side by side in one process and
timed alternately (A B B A ...) with CUDA events around back-to-back calls on one room() scene.  Prints and writes
DIR/ab_fps.json: ms per call of each build per repeat, the card's name and power limit, and whether the two builds
returned the same seeds.

    python tools/ab_fps.py OLD.so NEW.so [--n 1000000] [--m 512] [--repeats 6] [--calls 20] [--out DIR]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from geoformer_b200.scenes import room  # noqa: E402


def load(path):
    L = ctypes.CDLL(os.path.abspath(path))
    L.gf_fps_workspace_bytes.restype = ctypes.c_size_t
    L.gf_fps_workspace_bytes.argtypes = [ctypes.c_int] * 3
    L.gf_furthest_point_sampling.restype = ctypes.c_int
    L.gf_furthest_point_sampling.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                             ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    return L


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs=2)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--m", type=int, default=512)
    ap.add_argument("--repeats", type=int, default=6)
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    x = room(a.n, 4321)[None].to(dev).contiguous()
    st = torch.cuda.current_stream(dev)
    runs = []
    for path in a.libs:
        L = load(path)
        nbytes = L.gf_fps_workspace_bytes(1, a.n, a.m)
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=dev)
        out = torch.empty((1, a.m), dtype=torch.int32, device=dev)

        def call(L=L, ws=ws, nbytes=nbytes, out=out):
            rc = L.gf_furthest_point_sampling(x.data_ptr(), 1, a.n, a.m, out.data_ptr(), ws.data_ptr(), nbytes,
                                              st.cuda_stream)
            assert rc == 0, rc

        runs.append(dict(lib=path, call=call, out=out, ms=[]))
    for r in runs:  # warm-up: module load, cluster-size probe
        for _ in range(3):
            r["call"]()
    torch.cuda.synchronize()
    same = bool(torch.equal(runs[0]["out"], runs[1]["out"]))
    for rep in range(a.repeats):
        for r in (runs if rep % 2 == 0 else runs[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            for _ in range(a.calls):
                r["call"]()
            e1.record(st)
            e1.synchronize()
            r["ms"].append(e0.elapsed_time(e1) / a.calls)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    res = dict(what="furthest_point_sampling alone, B=1, room(n, 4321), CUDA events around %d back-to-back calls per "
               "repeat, builds alternated A B B A" % a.calls, n=a.n, m=a.m, card=card, same_seeds=same,
               builds=[dict(lib=os.path.basename(r["lib"]), ms_per_call=r["ms"], median_ms=sorted(r["ms"])[len(r["ms"]) // 2],
                            us_per_round=1e3 * sorted(r["ms"])[len(r["ms"]) // 2] / (a.m - 1)) for r in runs])
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "ab_fps.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
