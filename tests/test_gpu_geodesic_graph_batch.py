"""The propagation of a batch of scenes over the caller's own kNN graphs (gf_geodesic_batch, geodesic_from_graph_batch
and the index branch of cal_geodesic_vectorize): every map bitwise equal to the oracle and to geodesic_from_graph on
the scene alone, whatever numbering the points passed in choose, with a fixed number of kernels per call."""
import ctypes

import numpy as np
import pytest
import torch

from geoformer_b200.scenes import scene
from test_gpu_workspace_layouts import _check_layout

pytestmark = pytest.mark.gpu

GF_ERR_INVALID = 1


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _points(n, seed):
    if n > 50:
        return scene(n, seed).numpy()
    return np.random.default_rng(seed).uniform(0, 1, (n, 3)).astype(np.float32)


def _batch(oracle_lib, Ns, Q, k, seed):
    """points, oracle graphs (int64) and Q random seeds per scene"""
    g = np.random.default_rng(seed)
    pts, graphs, seeds = [], [], []
    for i, n in enumerate(Ns):
        x = _points(n, seed * 100 + i)
        D, I = oracle_lib.find_knn(x, k)
        s = g.integers(0, n, Q).astype(np.int32)
        pts.append(x), graphs.append((D, I)), seeds.append(s)
    return pts, graphs, seeds


def _to(dev, pts, graphs, seeds, idt=np.int64):
    return ([torch.from_numpy(x).to(dev) for x in pts],
            [(torch.from_numpy(D).to(dev), torch.from_numpy(I.astype(idt)).to(dev)) for D, I in graphs],
            [torch.from_numpy(s).to(dev) for s in seeds])


def _singles(graphs, seeds, r, ms):
    from geoformer_b200.geodesic_utils import geodesic_from_graph

    out = []
    for (D, I), s in zip(graphs, seeds):
        rm = torch.empty(s.numel(), dtype=torch.float32, device=D.device)
        geo, st = geodesic_from_graph(D, I, s, r, ms, return_stats=True, row_max=rm)
        out.append((geo, st, rm))
    return out


def _check(oracle_lib, dev, pts, graphs, seeds, r, ms, xyz=None):
    """batched call == oracle == per-scene op, maps, stats and row maxima, with int64 and int32 indices"""
    from geoformer_b200.geodesic_utils import geodesic_from_graph_batch

    refs = [oracle_lib.geodesic(D, I, s, r, ms) for (D, I), s in zip(graphs, seeds)]
    for idt in (np.int64, np.int32):
        x, gr, sd = _to(dev, pts, graphs, seeds, idt)
        if xyz is not None:
            x = xyz
        geo, stats, rmax = geodesic_from_graph_batch(x, gr, sd, r, ms, row_max=True, return_stats=True)
        single = _singles(gr, sd, r, ms)
        for b, ref in enumerate(refs):
            assert np.array_equal(geo[b].cpu().numpy(), ref), (idt, b)
            assert torch.equal(geo[b], single[b][0]), (idt, b)
            assert torch.equal(stats[b], single[b][1]), (idt, b)
            assert torch.equal(rmax[b], single[b][2]), (idt, b)


@pytest.mark.parametrize("B", [1, 2, 5, 32, 33])
def test_batch_matches_oracle_and_per_scene_op(oracle_lib, dev, B):
    g = np.random.default_rng(B)
    Ns = g.choice([1, 2, 37, 800, 3000, 6000], size=B).tolist()
    Ns[0] = 40_000 if B < 32 else Ns[0]
    Ns[-1] = 17_000
    pts, graphs, seeds = _batch(oracle_lib, Ns, 24, 8, B)
    _check(oracle_lib, dev, pts, graphs, seeds, 0.3, 24)


@pytest.mark.parametrize("k", [1, 2, 16, 64, 100])
def test_foreign_graph_quirks(oracle_lib, dev, k):
    """-1 padded entries, self loops with non-zero length, a column 0 that is not the point, duplicate points, a seed
    given twice, radius cut-offs"""
    g = np.random.default_rng(k)
    Ns = [4000, 1500, 2500]
    pts, graphs, seeds = _batch(oracle_lib, Ns, 16, k, 50 + k)
    pts[1][10:20] = pts[1][0:10]  # duplicates: a seed in its own neighbour row
    graphs[1] = oracle_lib.find_knn(pts[1], k)
    seeds[1][:3] = [12, 12, 2]
    D, I = graphs[0]
    D, I = D.copy(), I.copy()
    I[g.random(I.shape) < 0.15] = -1
    if k > 3:
        loops = g.integers(0, Ns[0], 50)
        I[loops, 3], D[loops, 3] = loops, 0.01
        seeds[0][:4] = loops[:4]
    I[:, 0] = g.integers(0, Ns[0], Ns[0])  # column 0 is dropped, whatever it holds
    graphs[0] = (D, I)
    _check(oracle_lib, dev, pts, graphs, seeds, 0.3, 30)
    _check(oracle_lib, dev, pts, graphs, seeds, 0.05, 30)  # most edges cut off by the radius
    _check(oracle_lib, dev, pts, graphs, seeds, 0.3, 0)  # max_step 0: only the seed entries


def test_out_of_range_seeds_leave_their_row_empty(oracle_lib, dev):
    from geoformer_b200.geodesic_utils import geodesic_from_graph_batch

    pts, graphs, seeds = _batch(oracle_lib, [3000, 700], 8, 8, 7)
    seeds[0][[1, 4]] = [3000, -5]
    seeds[1][2] = 1 << 30
    x, gr, sd = _to(dev, pts, graphs, seeds)
    geo, stats, rmax = geodesic_from_graph_batch(x, gr, sd, 0.3, 20, row_max=True, return_stats=True)
    single = _singles(gr, sd, 0.3, 20)
    for b in range(2):
        assert torch.equal(geo[b], single[b][0]) and torch.equal(stats[b], single[b][1])
        assert torch.equal(rmax[b], single[b][2])
    assert bool((geo[0][[1, 4]] == -1).all()) and bool((geo[1][2] == -1).all())
    assert float(rmax[0][1]) == -1.0 and float(rmax[1][2]) == -1.0


def test_numbering_does_not_change_the_maps(oracle_lib, dev):
    """xyz only chooses the cell order: permuted points, another scene's points of the same N, or all zeros"""
    Ns = [5000, 5000, 3000]
    pts, graphs, seeds = _batch(oracle_lib, Ns, 16, 16, 9)
    perm = np.random.default_rng(0).permutation(5000)
    others = [torch.from_numpy(pts[0][perm]).to(dev), torch.from_numpy(pts[0]).to(dev),
              torch.zeros(3000, 3, device=dev)]
    _check(oracle_lib, dev, pts, graphs, seeds, 0.5, 32)
    _check(oracle_lib, dev, pts, graphs, seeds, 0.5, 32, xyz=others)


def _call(L, dev, xs, Ds, Is, i64, Ns, B, k, seeds, Q, geo, ws_bytes=None):
    """gf_geodesic_batch called directly: (status, kernels launched)"""
    Nc = (ctypes.c_int * len(Ns))(*Ns) if Ns is not None else None
    nbytes = ws_bytes if ws_bytes is not None else L.gf_geodesic_batch_workspace_bytes(Nc, max(B, 1), Q, k)
    ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
    before = L.gf_launch_count()
    rc = L.gf_geodesic_batch(xs, Ds, Is, i64, Nc, B, k, seeds, Q, ctypes.c_float(0.3), 16, geo, None, None,
                             ws.data_ptr(), nbytes, torch.cuda.current_stream(dev).cuda_stream)
    torch.cuda.synchronize()
    return rc, L.gf_launch_count() - before


def test_scene_too_large_for_the_batched_kernel(oracle_lib, dev):
    from geoformer_b200 import _capi as C
    from geoformer_b200.geodesic_utils import geodesic_from_graph, geodesic_from_graph_batch, knn_graph
    from geoformer_b200.guidance import _ptr_array

    Ns = [3000, 910_000, 2000]
    x = [torch.from_numpy(_points(n, 80 + i)).to(dev) for i, n in enumerate(Ns)]
    gr = [knn_graph(p, 8) for p in x]
    sd = [torch.randint(0, n, (4,), generator=torch.Generator().manual_seed(i)).int().to(dev)
          for i, n in enumerate(Ns)]
    geo, stats = geodesic_from_graph_batch(x, gr, sd, 0.5, 3, return_stats=True)
    for b in range(3):
        g1, s1 = geodesic_from_graph(*gr[b], sd[b], 0.5, 3, return_stats=True)
        assert torch.equal(geo[b], g1) and torch.equal(stats[b], s1), b
    L = C.lib()
    out = [torch.empty(4, n, device=dev) for n in Ns]
    rc, launched = _call(L, dev, _ptr_array(x), _ptr_array([D for D, _ in gr]), _ptr_array([I for _, I in gr]), 1, Ns,
                         3, 8, _ptr_array(sd), 4, _ptr_array(out), ws_bytes=1 << 20)
    assert rc == GF_ERR_INVALID and launched == 0
    assert "gf_geodesic" in L.gf_last_error().decode()


def test_argument_checks_launch_nothing(dev):
    from geoformer_b200 import _capi as C
    from geoformer_b200.guidance import _ptr_array

    L = C.lib()
    Ns = [500, 300]
    x = [torch.from_numpy(_points(n, i)).to(dev) for i, n in enumerate(Ns)]
    D = [torch.zeros(n, 8, device=dev) for n in Ns]
    I = [torch.zeros(n, 8, dtype=torch.int64, device=dev) for n in Ns]
    s = [torch.zeros(4, dtype=torch.int32, device=dev) for _ in Ns]
    geo = [torch.empty(4, n, device=dev) for n in Ns]
    P = _ptr_array
    ok = dict(xs=P(x), Ds=P(D), Is=P(I), i64=1, Ns=Ns, B=2, k=8, seeds=P(s), Q=4, geo=P(geo))
    assert _call(L, dev, **ok) == (0, 7)
    bad = [dict(B=0), dict(B=33, Ns=Ns * 17), dict(xs=None), dict(Ds=None), dict(Is=None), dict(seeds=None),
           dict(geo=None), dict(Ns=None), dict(Ns=[500, 0]), dict(Ns=[500, -3]), dict(k=0), dict(k=257), dict(Q=0),
           dict(i64=2), dict(i64=-1), dict(xs=P([x[0], None])), dict(Ds=P([None, D[1]])), dict(geo=P([geo[0], None]))]
    for change in bad:
        args = dict(ok, **change)
        rc, launched = _call(L, dev, ws_bytes=1 << 22, **args)
        assert (rc, launched) == (GF_ERR_INVALID, 0), change


def test_launch_count_does_not_grow_with_the_batch(dev):
    from geoformer_b200 import _capi as C
    from geoformer_b200.geodesic_utils import geodesic_from_graph_batch, knn_graph

    counts = []
    for B in (2, 5, 32):
        x = [torch.from_numpy(_points(n, i)).to(dev) for i, n in enumerate([700 + 13 * i for i in range(B)])]
        gr = [knn_graph(p, 8) for p in x]
        sd = [torch.arange(6, dtype=torch.int32, device=dev) for _ in x]
        geodesic_from_graph_batch(x, gr, sd, 0.3, 10)
        torch.cuda.synchronize()
        before = C.launch_count()
        geodesic_from_graph_batch(x, gr, sd, 0.3, 10)
        counts.append(C.launch_count() - before)
    assert counts == [7, 7, 7], counts


class _StandIn:
    """an index with the faiss protocol that is not a FlatL2Index: brute-force kNN with some neighbours dropped"""

    def __init__(self):
        from geoformer_b200.geodesic_utils import FlatL2Index

        self._ix = FlatL2Index(algo="brute")

    def add(self, x):
        self._ix.add(x)

    def search(self, q, k, D, I):
        self._ix.search(q, k, D, I)
        drop = torch.arange(I.numel(), device=I.device).view_as(I) % 7 == 3
        I[drop] = -1
        D[drop] = float("inf")

    def reset(self):
        self._ix.reset()


def _reference(oracle_lib, pre, locs, offs, ms, k, r, Q, drop_some):
    """the oracle scene by scene (an empty scene gets an empty map), over its kNN graph with the stand-in's drops"""
    out = []
    for b in range(len(offs) - 1):
        if offs[b + 1] == offs[b]:
            out.append(np.empty((Q, 0), dtype=np.float32))
            continue
        D, I = oracle_lib.find_knn(locs[offs[b]:offs[b + 1]], k)
        if drop_some:
            drop = np.arange(I.size).reshape(I.shape) % 7 == 3
            I, D = I.copy(), D.copy()
            I[drop], D[drop] = -1, np.inf
        out.append(oracle_lib.geodesic(D, I, pre[b][:Q], r, ms))
    return out


def test_cal_geodesic_vectorize_over_a_foreign_index(oracle_lib, dev):
    from geoformer_b200.geodesic_utils import FlatL2Index, cal_geodesic_vectorize

    sizes = [3000, 0, 1, 4500, 2200]
    locs = np.concatenate([_points(n, 90 + i) for i, n in enumerate(sizes)]).astype(np.float32)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    pre = np.stack([np.random.default_rng(i).integers(0, max(n, 1), 40) for i, n in enumerate(sizes)]).astype(np.int32)
    Q, k = 16, 8
    for index, drop_some in ((_StandIn(), True), (FlatL2Index(algo="brute"), False)):
        ref = _reference(oracle_lib, pre, locs, offs, 20, k, 0.3, Q, drop_some)
        out = cal_geodesic_vectorize(index, torch.from_numpy(pre).to(dev), torch.from_numpy(locs).to(dev),
                                     torch.from_numpy(offs).to(dev), max_step=20, neighbor=k, radius=0.3, n_queries=Q)
        assert len(out) == len(sizes)
        for o, r in zip(out, ref):
            assert o.shape == r.shape and o.dtype == torch.float32 and o.is_cuda
            assert np.array_equal(o.cpu().numpy(), r)


def test_streams_and_repeated_calls_stay_exact(dev):
    from geoformer_b200.geodesic_utils import cal_geodesic_vectorize, find_knn, geodesic_from_graph

    sizes = [20000, 35000, 1, 27000, 0, 22000, 40000]
    pts = [torch.from_numpy(_points(n, 70 + i)) for i, n in enumerate(sizes)]
    locs = torch.cat(pts).to(dev)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    Q = 32
    gen = torch.Generator().manual_seed(3)
    pre = torch.stack([torch.randint(0, max(n, 1), (48,), generator=gen) for n in sizes]).int().to(dev)
    singles = []
    for b, n in enumerate(sizes):
        lb = locs[int(offs[b]):int(offs[b + 1])].contiguous()
        singles.append(geodesic_from_graph(*find_knn(_StandIn(), lb, 16), pre[b][:Q], 0.5, 24) if n > 0 else None)
    torch.cuda.synchronize()
    user = torch.cuda.Stream(device=dev)
    for rep in range(3):
        with torch.cuda.stream(user):
            out = cal_geodesic_vectorize(_StandIn(), pre, locs, torch.from_numpy(offs).to(dev), max_step=24,
                                         neighbor=16, radius=0.5, n_queries=Q)
            sums = [o.sum() if o.numel() else None for o in out]  # consumed on the caller's stream at once
        user.synchronize()
        for b, n in enumerate(sizes):
            assert out[b].shape == (Q, n)
            if n > 0:
                assert torch.equal(out[b], singles[b]), (rep, b)
                assert torch.equal(sums[b], singles[b].sum())


@pytest.mark.parametrize("Ns,k", [([3000], 8), ([5000, 1, 2500, 12000, 700, 3000], 16), ([4000, 900], 100)])
def test_workspace_layout(dev, Ns, k):
    """one scene; scenes of many sizes (the largest sets the propagation scratch); k above the grid's 64"""
    from geoformer_b200.geodesic_utils import geodesic_from_graph_batch, knn_graph

    x = [torch.from_numpy(_points(n, 30 + i)).to(dev) for i, n in enumerate(Ns)]
    gr = [knn_graph(p, min(k, 64)) for p in x]
    if k > 64:  # a wider graph than our kNN serves: padded with missing neighbours
        gr = [(torch.cat([D, torch.full((D.size(0), k - 64), float("inf"), device=dev)], 1).contiguous(),
               torch.cat([I, torch.full((I.size(0), k - 64), -1, dtype=I.dtype, device=dev)], 1).contiguous())
              for D, I in gr]
    sd = [torch.randint(0, n, (12,), generator=torch.Generator().manual_seed(i)).int().to(dev)
          for i, n in enumerate(Ns)]
    _check_layout(dev, "gf_geodesic_batch",
                  lambda: geodesic_from_graph_batch(x, gr, sd, 0.5, 16, row_max=True, return_stats=True))
