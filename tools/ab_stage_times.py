"""A/B of libraries (GF_LIB, read once per process => one subprocess per combination).
Prints per-stage CUDA-event times of the fused hot path, one scene in flight, for a workload.

    python tools/ab_stage_times.py c2 "" "GF_LIB=geoformer_b200/libgeoformer_b200_x.so"
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import ctypes, json, statistics, sys
import torch
sys.path.insert(0, %(root)r)
from geoformer_b200 import _capi as C
from geoformer_b200.guidance import GuidanceRunner
from geoformer_b200.scenes import CONFIGS, scene, room
cfg = dict(CONFIGS[%(wl)r])
if %(ms)d > 0: cfg["max_step"] = %(ms)d
dev = torch.device("cuda:0")
gen = scene if cfg["gen"] == "scene" else room
xs = [gen(cfg["n"], cfg["seed"] + s).to(dev) for s in range(3)]
L = C.lib()
r = GuidanceRunner(cfg["n"], cfg["Q"], cfg["k"], cfg["radius"], cfg["max_step"], device=dev)
st = torch.cuda.current_stream(dev)
K = 14
ev = [[L.gf_event_create() for _ in range(5)] for _ in range(K)]
arr = [(ctypes.c_void_p * 5)(*e) for e in ev]
for i in range(K):
    L.gf_set_stage_events(arr[i], 5)
    r.run(xs[i %% 3], st)
torch.cuda.synchronize()
def stage(a, b):
    return statistics.median(L.gf_event_elapsed_ms(e[a], e[b]) for e in ev[4:])
print(json.dumps({"build": stage(0, 1), "query_join": stage(1, 2), "pack": stage(2, 3), "bfs": stage(3, 4),
                  "whole": stage(0, 4), "reached": int(r.stats[0].item()), "levels": int(r.stats[1].item()),
                  "checksum": float(r.geo.double().sum().item())}))
"""


def main():
    wl = sys.argv[1]
    ms = 0
    if ":" in wl:
        wl, ms = wl.split(":")
        ms = int(ms)
    for combo in sys.argv[2:] or [""]:
        env = dict(os.environ)
        for kv in combo.split():
            k, v = kv.split("=")
            env[k] = v
        out = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT, "wl": wl, "ms": ms}], env=env, cwd=ROOT,
                             capture_output=True, text=True, timeout=600)
        line = out.stdout.strip().splitlines()[-1] if out.stdout.strip() else out.stderr[-600:]
        print("%-44s %s" % (combo or "(default)", line), flush=True)


if __name__ == "__main__":
    main()
