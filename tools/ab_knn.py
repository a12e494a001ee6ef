"""A/B of kNN query kernel variants, each built into its own library (one subprocess per library): ms per kNN graph
and a checksum of the index / distance tables, so that two variants can be compared for equality at a glance.

    python tools/ab_knn.py "" "GF_LIB=geoformer_b200/libgeoformer_b200_x.so"
"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import hashlib, json, sys
import torch
sys.path.insert(0, %(root)r)
from geoformer_b200.scenes import room, scene
from geoformer_b200.geodesic_utils import knn_graph
dev = torch.device("cuda", 0)
def t(fn, reps=10):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps
out = {}
for name, x in (("c2", scene(100_000, 1234).to(dev)), ("c1", scene(50_000, 1234).to(dev)), ("c4", room(1_000_000, 4321).to(dev))):
    for k in (8, 16, 64):
        if name == "c4" and k == 64: continue
        D, I = knn_graph(x, k, index_dtype=torch.int32)
        h = hashlib.sha1(I.cpu().numpy().tobytes() + D.cpu().numpy().tobytes()).hexdigest()[:10]
        out["%%s_k%%d" %% (name, k)] = [round(t(lambda: knn_graph(x, k, index_dtype=torch.int32)), 4), h]
print(json.dumps(out))
"""


def main():
    for combo in sys.argv[1:] or [""]:
        env = dict(os.environ)
        for kv in combo.split():
            key, val = kv.split("=", 1)
            env[key] = val
        r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}], env=env, capture_output=True, text=True)
        print(combo or "(default)", "->", r.stdout.strip() or r.stderr.strip()[-600:], flush=True)


if __name__ == "__main__":
    main()
