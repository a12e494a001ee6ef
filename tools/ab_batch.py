"""A/B of the batched hot path: ms per scene for batches of B scenes of a workload, one batch in flight, per
combination of batch size and library (one subprocess each).

    python tools/ab_batch.py c2 "B=1" "B=8" "B=8 GF_LIB=geoformer_b200/libgeoformer_b200_x.so" ...
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import json, statistics, sys
import torch
sys.path.insert(0, %(root)r)
from geoformer_b200.guidance import BatchGuidanceRunner
from geoformer_b200.scenes import CONFIGS, scene, room
cfg = dict(CONFIGS[%(wl)r])
if %(ms)d > 0: cfg["max_step"] = %(ms)d
B, graph, two = %(B)d, %(graph)d, %(two)d
dev = torch.device("cuda:0")
gen = scene if cfg["gen"] == "scene" else room
xs = [gen(cfg["n"], cfg["seed"] + s).to(dev) for s in range(8)]
rs = [BatchGuidanceRunner(cfg["n"], B, cfg["Q"], cfg["k"], cfg["radius"], cfg["max_step"], device=dev, graph=bool(graph),
                          stage_events=True) for _ in range(2 if two else 1)]
sts = [torch.cuda.Stream(device=dev) for _ in rs]
for i, r in enumerate(rs):
    r.load([xs[(i * B + b) %% 8] for b in range(B)])
for r, st in zip(rs, sts):
    for _ in range(3):
        r.replay(st)
torch.cuda.synchronize()
K = 12
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
cur = torch.cuda.current_stream(dev)
e0.record(cur)
for st in sts: st.wait_event(e0)
prop = []
for i in range(K):
    rs[i %% len(rs)].replay(sts[i %% len(rs)])
for st in sts:
    ev = torch.cuda.Event(); ev.record(st); cur.wait_event(ev)
e1.record(cur)
torch.cuda.synchronize()
prop = [r.propagation_ms() for r in rs]
ms = e0.elapsed_time(e1) / (K * B)
print(json.dumps({"ms_per_scene": round(ms, 4), "maps_per_s": round(cfg["Q"] / ms * 1e3), "prop_ms_per_scene": [round(p / B, 4) for p in prop],
                  "launches": rs[0].launches_per_run, "checksum": float(rs[0].geo[0].double().sum().item())}))
"""


def main():
    wl = sys.argv[1]
    ms = 0
    if ":" in wl:
        wl, ms = wl.split(":")
        ms = int(ms)
    for combo in sys.argv[2:] or ["B=1"]:
        env = dict(os.environ)
        opts = {"B": 1, "GRAPH": 0, "TWO": 0}
        for kv in combo.split():
            k, v = kv.split("=")
            if k in opts:
                opts[k] = int(v)
            else:
                env[k] = v
        out = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT, "wl": wl, "ms": ms, "B": opts["B"],
                                                             "graph": opts["GRAPH"], "two": opts["TWO"]}],
                             env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
        line = out.stdout.strip().splitlines()[-1] if out.stdout.strip() else out.stderr[-800:]
        print("%-52s %s" % (combo, line), flush=True)


if __name__ == "__main__":
    main()
