"""Batched kNN graphs: one launch of each grid-build kernel and one query launch for all scenes of a call
(gf_knn.cu: knn_grid_build_batch, knn_grid_query_batch).  A block of those launches belongs to exactly one scene, so
every scene's tables must equal what the single-scene call computes for it, bit for bit, whatever the other scenes
are: scenes of different sizes (fewer points than a 128-query block, sizes that are not a multiple of it, a single
point), scenes whose query lists overflow (duplicate clusters, a lattice) next to ordinary ones, and k on both query
kernels (the count-then-collect one up to k = 32, the warp-synchronous one at k = 64)."""
import ctypes
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from geoformer_b200.scenes import scene  # noqa: E402

KS = [8, 16, 17, 64]


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _lattice(seed):
    """a 20 x 20 x 10 lattice of spacing 0.25: every distance is tied many times"""
    g = np.random.default_rng(seed)
    ax = [np.arange(n, dtype=np.float32) * np.float32(0.25) for n in (20, 20, 10)]
    x = np.stack(np.meshgrid(*ax, indexing="ij"), -1).reshape(-1, 3)
    return np.ascontiguousarray(x[g.permutation(len(x))])


def _duplicate_clusters(seed):
    """clusters of 40 .. 200 copies of one point: more candidates at d2 = 0 than a query's list holds"""
    g = np.random.default_rng(seed)
    x = scene(6000, seed).numpy().copy()
    at = 0
    for n in (40, 90, 200):
        x[at:at + n] = x[at + n + 7]
        at += n + 10
    return np.ascontiguousarray(x[g.permutation(len(x))])


def _sizes():
    """different N: a single point, fewer than 128, exactly 128, not multiples of 128, a c2 scene"""
    g = np.random.default_rng(5)
    one = (g.random((1, 3)) * 2.0).astype(np.float32)
    return [one, scene(37, 2).numpy(), scene(128, 3).numpy(), scene(1001, 4).numpy(), scene(100_000, 1234).numpy(),
            scene(4999, 6).numpy()]


def _mixed():
    """list-overflow scenes between c2-like ones"""
    return [scene(100_000, 1235).numpy(), _duplicate_clusters(7), scene(30_000, 8).numpy(), _lattice(9),
            scene(100_000, 1236).numpy()]


CASES = {"sizes": (_sizes, 3), "mixed": (_mixed, 3)}  # the scene that is also checked against the CPU oracle


def _knn_batch(xs, k):
    """gf_knn_batch over the scenes xs (CUDA (N,3) f32) -> [(sqrt distances (N,k) f32, indices (N,k) i32)]"""
    from geoformer_b200 import _capi as C

    L = C.lib()
    B = len(xs)
    Ns = (ctypes.c_int * B)(*[x.shape[0] for x in xs])
    D = [torch.empty((x.shape[0], k), dtype=torch.float32, device=x.device) for x in xs]
    I = [torch.empty((x.shape[0], k), dtype=torch.int32, device=x.device) for x in xs]
    nbytes = L.gf_knn_batch_workspace_bytes(Ns, B)
    assert nbytes > 0
    ws = torch.empty(nbytes, dtype=torch.uint8, device=xs[0].device)

    def arr(ts):
        return (ctypes.c_void_p * B)(*[t.data_ptr() for t in ts])

    C.check(L.gf_knn_batch(arr(xs), Ns, B, k, 1, arr(D), arr(I), ctypes.c_void_p(ws.data_ptr()), nbytes,
                           ctypes.c_void_p(torch.cuda.current_stream(xs[0].device).cuda_stream)), "knn_batch")
    torch.cuda.synchronize()
    return list(zip(D, I))


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("case", sorted(CASES))
def test_knn_batch_equals_single_scene_calls(oracle_lib, dev, case, k):
    from geoformer_b200.geodesic_utils import knn_graph

    make, checked = CASES[case]
    xs_np = make()
    xs = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in xs_np]
    got = _knn_batch(xs, k)
    for i, x in enumerate(xs):
        D1, I1 = knn_graph(x, k, index_dtype=torch.int32)
        assert torch.equal(got[i][1], I1), (case, k, i)
        assert torch.equal(got[i][0], D1), (case, k, i)
    rD, rI = oracle_lib.find_knn(xs_np[checked], k)
    assert np.array_equal(got[checked][1].cpu().numpy(), rI.astype(np.int32))
    assert np.array_equal(got[checked][0].cpu().numpy(), rD)


def test_knn_batch_alone_and_in_company(dev):
    """a scene's tables do not depend on the scenes batched with it, nor on its place in the batch"""
    xs = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in _mixed()]
    alone = _knn_batch([xs[1]], 16)[0]
    for order in ([0, 1, 2, 3, 4], [4, 3, 2, 1, 0]):
        got = _knn_batch([xs[j] for j in order], 16)
        D, I = got[order.index(1)]
        assert torch.equal(I, alone[1]) and torch.equal(D, alone[0]), order


@pytest.mark.parametrize("k", [16, 17])
def test_guidance_batch_of_different_sizes(oracle_lib, dev, k):
    """the fused hot path over scenes of different N, list-overflow scenes among them: each scene's seeds and maps
    equal its single-scene call, one of them also the oracle's"""
    from geoformer_b200.guidance import geodesic_guidance, geodesic_guidance_batch

    xs_np = [scene(300, 11).numpy(), _duplicate_clusters(12), scene(1001, 13).numpy(), _lattice(14),
             scene(20_000, 15).numpy()]
    xs = [torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in xs_np]
    Q, r, ms = 24, 0.5, 24
    seeds, geos = geodesic_guidance_batch(xs, Q, k, r, ms)
    for i, x in enumerate(xs):
        s1, g1 = geodesic_guidance(x, Q, k, r, ms)
        assert torch.equal(seeds[i], s1) and torch.equal(geos[i], g1), i
    rs = oracle_lib.furthest_point_sampling(xs_np[3][None], Q)[0]
    rD, rI = oracle_lib.find_knn(xs_np[3], k)
    assert np.array_equal(geos[3].cpu().numpy(), oracle_lib.geodesic(rD, rI, rs, r, ms))


def _kernel_names(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = []
    for e in prof.events():  # demangled "gf::knn_scan_kernel(...)" or mangled "_ZN2gf15knn_scan_kernel..."
        m = re.search(r"(fps_\w+?_kernel|knn_\w+?_kernel|geo_\w+?_kernel)", e.name)
        if m:
            names.append(m.group(1))
    return names


def test_guidance_batch_launch_count(dev):
    """one batched call of B scenes, more than the four FPS lanes, launches B FPS kernels, the five grid-build kernels
    once, one query and one propagation: B + 7 kernels"""
    from geoformer_b200.guidance import geodesic_guidance_batch

    B = 6
    xs = [scene(20_000, 40 + b).to(dev) for b in range(B)]
    geodesic_guidance_batch(xs, 32, 16, 0.5, 8)  # warm-up: lanes, workspace
    torch.cuda.synchronize()
    names = _kernel_names(lambda: geodesic_guidance_batch(xs, 32, 16, 0.5, 8))
    count = {n: names.count(n) for n in set(names)}
    assert sum(v for n, v in count.items() if n.startswith("fps_")) == B, count
    assert count.get("knn_bbox_kernel") == 1 and count.get("knn_count_kernel") == 2, count
    assert count.get("knn_scan_kernel") == 1 and count.get("knn_scatter_kernel") == 1, count
    assert count.get("knn_grid_query_kernel") == 1, count
    assert count.get("geo_bfs_batch_kernel") == 1, count
    assert len(names) == B + 7, count


def test_batch_guidance_runner_with_batched_graphs(dev):
    """BatchGuidanceRunner: plain and CUDA-graph replay give the bits of the per-scene call; the two stage events
    that bracket the propagation launch are stamped by every replay (external event record nodes).  With more scenes
    than FPS lanes the graphs are batched: B FPS launches, the five grid-build kernels and the query once, one
    propagation launch."""
    from geoformer_b200.guidance import BatchGuidanceRunner, geodesic_guidance

    N, B, Q, k = 30000, 6, 48, 16
    xa = [scene(N, 60 + i).to(dev) for i in range(B)]
    xb = [scene(N, 70 + i).to(dev) for i in range(B)]
    want = {id(x): geodesic_guidance(x, Q, k, 0.5, 20) for x in xa + xb}
    side = torch.cuda.Stream(device=dev)
    for graph in (False, True):
        r = BatchGuidanceRunner(N, B, Q, k, 0.5, 20, device=dev, graph=graph, stage_events=True)
        for xs in (xa, xb, xa):
            seeds, geo = r.run(xs, side)
            side.synchronize()
            for b, x in enumerate(xs):
                assert torch.equal(seeds[b], want[id(x)][0]) and torch.equal(geo[b], want[id(x)][1]), (graph, b)
                assert torch.equal(r.row_max[b], want[id(x)][1].max(dim=1).values)
            ms = r.propagation_ms()
            assert ms is not None and 0.0 < ms < 50.0, ms
        assert r.launches_per_run == B + 7, r.launches_per_run
        r.close()

