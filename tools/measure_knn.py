"""kNN graph time at c1 / c2 / c4 for k = 8, 16, 32; GF_LIB selects another build of the library.

    python tools/measure_knn.py
    GF_LIB=geoformer_b200/libgeoformer_b200_x.so python tools/measure_knn.py
"""
import os, sys, torch
sys.path.insert(0, ".")
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
for name, x in (("c2", scene(100_000, 1234).to(dev)), ("c1", scene(50_000, 1234).to(dev)), ("c4", room(1_000_000, 4321).to(dev))):
    for k in (8, 16, 32):
        print(os.environ.get("GF_LIB", "libgeoformer_b200.so"), name, "k", k, "knn ms %.4f" % t(lambda: knn_graph(x, k, index_dtype=torch.int32)))
