"""GPU parity tests: every CUDA entry point of libgeoformer_b200.so against the CPU oracle on the
same seeded inputs.  Index / integer results must be bit-exact; the geodesic is compared bit-exact
as well (one fp32 add per reached pair in both) with the north_star bound (1e-5 relative, identical
unreachable sets) as the stated tolerance.  Run on the B200 box:  pytest -m gpu
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from geoformer_b200.scenes import scene  # noqa: E402
from test_gpu_ops_launch_shapes import (assert_atomic_sum, gather_grad_terms, group_grad_terms,  # noqa: E402
                                        interpolate_grad_terms)


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _tied_cloud(n, seed):
    """points on a coarse lattice: many exactly tied distances, some points inside the |p|^2<1e-3 ball"""
    g = np.random.default_rng(seed)
    x = g.integers(-3, 4, size=(n, 3)).astype(np.float32) * 0.25
    x[g.integers(0, n, size=max(1, n // 50))] = 0.0
    x[g.integers(0, n, size=max(1, n // 50))] = np.float32(0.01)
    return x


def _check_knn_against_kdtree(x, rows, I_rows, D_rows, k):
    """Independent exact kNN: scipy's cKDTree on the float64 copies of the points (a different algorithm, different
    arithmetic, no code shared with the library or the oracle).  Tie-gap rule: position by position the float64
    distance of OUR neighbour must equal the tree's within 2e-6 relative (fp32 rounding of d2 is ~3e-7), so an
    index may differ from the tree's only where the two candidates are that close to a tie; the reported fp32
    distances must be the float64 ones within 1e-6 relative.  Returns the number of rows whose index lists differ."""
    from scipy.spatial import cKDTree

    x64 = x.astype(np.float64)
    d_ref, i_ref = cKDTree(x64).query(x64[rows], k=k)
    d_ours = np.linalg.norm(x64[rows][:, None, :] - x64[I_rows.astype(np.int64)], axis=2)
    np.testing.assert_allclose(d_ours, d_ref, rtol=2e-6, atol=1e-9)
    np.testing.assert_allclose(D_rows.astype(np.float64), d_ours, rtol=1e-6, atol=1e-9)
    assert (d_ours[:, 1:] >= d_ours[:, :-1] - 2e-6 * d_ours[:, 1:] - 1e-9).all()
    return int((I_rows.astype(np.int64) != i_ref).any(axis=1).sum())


# ------------------------------------------------------------------------------------------ FPS
@pytest.mark.parametrize("B,N,m", [(1, 1, 1), (1, 2, 2), (2, 7, 5), (1, 300, 64), (3, 511, 100), (1, 512, 128),
                                   (2, 1000, 256), (1, 5000, 512), (2, 20000, 300), (1, 70000, 128)])
def test_fps_scene(oracle_lib, dev, B, N, m):
    from geoformer_b200.pointnet2 import _ext

    xyz = torch.stack([scene(N, 100 + b) for b in range(B)]) if N >= 50 else torch.randn(B, N, 3)
    ref = oracle_lib.furthest_point_sampling(xyz.numpy(), m)
    out = _ext.furthest_point_sampling(xyz.to(dev), m).cpu().numpy()
    assert out.dtype == np.int32 and np.array_equal(out, ref)


@pytest.mark.parametrize("N,m", [(64, 64), (500, 200), (513, 300), (4096, 512), (9000, 256)])
def test_fps_ties_and_skip_rule(oracle_lib, dev, N, m):
    from geoformer_b200.pointnet2 import _ext

    xyz = _tied_cloud(N, N)[None]
    ref = oracle_lib.furthest_point_sampling(xyz, m)
    out = _ext.furthest_point_sampling(torch.from_numpy(xyz).to(dev), m).cpu().numpy()
    assert np.array_equal(out, ref)


def test_fps_all_points_skipped(oracle_lib, dev):
    from geoformer_b200.pointnet2 import _ext

    xyz = np.full((1, 100, 3), 0.001, dtype=np.float32)  # |p|^2 = 3e-6: nothing is eligible
    ref = oracle_lib.furthest_point_sampling(xyz, 10)
    out = _ext.furthest_point_sampling(torch.from_numpy(xyz).to(dev), 10).cpu().numpy()
    assert np.array_equal(out, ref) and (out == 0).all()


def test_fps_config_c2_and_model_shape(oracle_lib, dev):
    """c2 (100k points, 256 seeds) and the model's 2048-context draw; prefix consistency (F8)."""
    from geoformer_b200.pointnet2 import _ext

    xyz = scene(100_000, 1234)[None]
    out = _ext.furthest_point_sampling(xyz.to(dev), 2048).cpu().numpy()
    ref = oracle_lib.furthest_point_sampling(xyz.numpy(), 512)
    assert np.array_equal(out[:, :512], ref)
    out256 = _ext.furthest_point_sampling(xyz.to(dev), 256).cpu().numpy()
    assert np.array_equal(out256, out[:, :256])
    assert len(set(out[0].tolist())) == 2048


@pytest.mark.parametrize("B,N,m", [(1, 400_000, 24), (2, 250_000, 12), (1, 1_000_000, 16), (1, 1_300_000, 6)])
def test_fps_whole_gpu_variants_large_scene(oracle_lib, dev, B, N, m):
    """N above one cluster's register capacity: the cooperative whole-GPU kernel (points in registers up
    to 1.2 M, streaming from L2 above), including a batch of two scenes."""
    from geoformer_b200.pointnet2 import _ext
    from geoformer_b200.scenes import room

    xyz = torch.stack([room(N, 4321 + b) for b in range(B)])
    ref = oracle_lib.furthest_point_sampling(xyz.numpy(), m)
    out = _ext.furthest_point_sampling(xyz.to(dev), m).cpu().numpy()
    assert np.array_equal(out, ref)


# --------------------------------------------------------------------------- gather / group / ball
def test_gather_and_grad(oracle_lib, dev):
    from geoformer_b200.pointnet2 import _ext

    g = torch.Generator().manual_seed(0)
    feats = torch.randn(2, 5, 700, generator=g)
    idx = torch.randint(0, 700, (2, 300), generator=g, dtype=torch.int32)
    out = _ext.gather_points(feats.to(dev), idx.to(dev)).cpu().numpy()
    assert np.array_equal(out, oracle_lib.gather_points(feats.numpy(), idx.numpy()))
    go = torch.randn(2, 5, 300, generator=g)
    gr = _ext.gather_points_grad(go.to(dev), idx.to(dev), 700).cpu().numpy()
    assert_atomic_sum(gr, *gather_grad_terms(go.numpy(), idx.numpy(), 700))


def test_group_and_grad(oracle_lib, dev):
    from geoformer_b200.pointnet2 import _ext

    g = torch.Generator().manual_seed(1)
    feats = torch.randn(2, 19, 900, generator=g)
    idx = torch.randint(0, 900, (2, 128, 16), generator=g, dtype=torch.int32)
    out = _ext.group_points(feats.to(dev), idx.to(dev)).cpu().numpy()
    assert np.array_equal(out, oracle_lib.group_points(feats.numpy(), idx.numpy()))
    go = torch.randn(2, 19, 128, 16, generator=g)
    gr = _ext.group_points_grad(go.to(dev), idx.to(dev), 900).cpu().numpy()
    assert_atomic_sum(gr, *group_grad_terms(go.numpy(), idx.numpy(), 900))


@pytest.mark.parametrize("N,m,r,ns", [(3000, 200, 0.2, 64), (20000, 512, 0.2, 64), (20000, 300, 0.05, 16),
                                      (5000, 40, 1e-4, 8), (100, 7, 10.0, 200), (4097, 33, 0.3, 1)])
def test_ball_query(oracle_lib, dev, N, m, r, ns):
    from geoformer_b200.pointnet2 import _ext

    xyz = scene(N, 7)[None]
    centres = xyz[:, torch.randperm(N, generator=torch.Generator().manual_seed(2))[:m]].contiguous()
    centres[0, 0] += 100.0  # a centre with no point in range -> all-zero row
    ref = oracle_lib.ball_query(centres.numpy(), xyz.numpy(), r, ns)
    out = _ext.ball_query(centres.to(dev), xyz.to(dev), r, ns).cpu().numpy()
    assert np.array_equal(out, ref)
    assert (out[0, 0] == 0).all()


def test_three_nn_and_interpolate(oracle_lib, dev):
    from geoformer_b200.pointnet2 import _ext

    g = torch.Generator().manual_seed(3)
    unknown, known = scene(3000, 11)[None], scene(1500, 12)[None]
    d2, idx = _ext.three_nn(unknown.to(dev), known.to(dev))
    rd2, ridx = oracle_lib.three_nn(unknown.numpy(), known.numpy())
    assert np.array_equal(idx.cpu().numpy(), ridx) and np.array_equal(d2.cpu().numpy(), rd2)
    feats = torch.randn(1, 6, 1500, generator=g)
    w = torch.rand(1, 3000, 3, generator=g)
    out = _ext.three_interpolate(feats.to(dev), idx, w.to(dev)).cpu().numpy()
    assert np.array_equal(out, oracle_lib.three_interpolate(feats.numpy(), ridx, w.numpy()))
    go = torch.randn(1, 6, 3000, generator=g)
    gr = _ext.three_interpolate_grad(go.to(dev), idx, w.to(dev), 1500).cpu().numpy()
    assert_atomic_sum(gr, *interpolate_grad_terms(go.numpy(), ridx, w.numpy(), 1500))
    # fewer than three known points: +inf / index 0 (interpolate_gpu.cu:31-32,56-61)
    d2s, idxs = _ext.three_nn(unknown[:, :10].contiguous().to(dev), known[:, :2].contiguous().to(dev))
    rd2s, ridxs = oracle_lib.three_nn(unknown[:, :10].numpy(), known[:, :2].numpy())
    assert np.array_equal(idxs.cpu().numpy(), ridxs) and np.array_equal(d2s.cpu().numpy(), rd2s)


def test_operator_preconditions(dev):
    """bindings raise RuntimeError like the reference's AT_ASSERTs (utils.h:8-28, sampling.cpp:35-37)."""
    from geoformer_b200.pointnet2 import _ext

    with pytest.raises(RuntimeError):
        _ext.furthest_point_sampling(torch.zeros(1, 10, 3), 4)  # CPU not supported
    with pytest.raises(RuntimeError):
        _ext.furthest_point_sampling(torch.zeros(1, 10, 3, dtype=torch.float64, device=dev), 4)
    with pytest.raises(RuntimeError):
        _ext.gather_points(torch.zeros(1, 3, 10, device=dev), torch.zeros(1, 4, dtype=torch.int64, device=dev))
    with pytest.raises(RuntimeError):
        _ext.ball_query(torch.zeros(1, 4, 3, device=dev).transpose(1, 2), torch.zeros(1, 10, 3, device=dev), 0.1, 4)


# ------------------------------------------------------------------------------------------ kNN
@pytest.mark.parametrize("N,k,algo", [(5, 8, "grid"), (17, 16, "brute"), (1000, 8, "grid"), (1000, 8, "brute"),
                                      (20000, 16, "grid"), (20000, 16, "brute"), (20000, 64, "grid"),
                                      (20000, 33, "grid"), (50000, 8, "grid"), (5000, 33, "brute"),
                                      (5000, 64, "brute"), (40, 64, "brute"), (20, 33, "brute")])
def test_knn_matches_oracle(oracle_lib, dev, N, k, algo):
    from geoformer_b200.geodesic_utils import knn_graph

    xyz = scene(N, 21) if N >= 50 else torch.randn(N, 3)
    D, I = knn_graph(xyz.to(dev), k, algo=algo)
    rD, rI = oracle_lib.find_knn(xyz.numpy(), k)
    assert I.dtype == torch.int64
    assert np.array_equal(I.cpu().numpy(), rI)
    assert np.array_equal(D.cpu().numpy(), rD)  # sqrtf is correctly rounded on both sides


def test_knn_duplicates_and_lattice_ties(oracle_lib, dev):
    from geoformer_b200.geodesic_utils import knn_graph

    x = _tied_cloud(6000, 5)
    x[100:200] = x[0:100]  # exact duplicates
    for algo in ("grid", "brute"):
        D, I = knn_graph(torch.from_numpy(x).to(dev), 16, algo=algo)
        rD, rI = oracle_lib.find_knn(x, 16)
        assert np.array_equal(I.cpu().numpy(), rI), algo
        assert np.array_equal(D.cpu().numpy(), rD), algo


def test_knn_degenerate_shapes(oracle_lib, dev):
    from geoformer_b200.geodesic_utils import knn_graph

    g = np.random.default_rng(9)
    line = np.zeros((3000, 3), np.float32)
    line[:, 0] = g.random(3000, dtype=np.float32) * 50
    plane = g.random((4000, 3), dtype=np.float32)
    plane[:, 2] = 1.5
    same = np.ones((300, 3), np.float32)
    outlier = scene(5000, 3).numpy().copy()
    outlier[17] = [900.0, -700.0, 300.0]
    for x in (line, plane, same, outlier):
        D, I = knn_graph(torch.from_numpy(x).to(dev), 8)
        rD, rI = oracle_lib.find_knn(x, 8)
        assert np.array_equal(I.cpu().numpy(), rI)
        assert np.array_equal(D.cpu().numpy(), rD)


def test_flat_index_protocol(oracle_lib, dev):
    """faiss-shaped boundary: add / search into pre-allocated tensors (squared distances) / reset."""
    from geoformer_b200.geodesic_utils import FlatL2Index, find_knn

    x = scene(8000, 31)
    q = scene(500, 32)
    index = FlatL2Index()
    index.add(x.to(dev))
    D = torch.zeros(500, 8, device=dev)
    I = torch.zeros(500, 8, dtype=torch.int64, device=dev)
    index.search(q.to(dev), 8, D, I)
    rD2, rI = oracle_lib.knn_sq(x.numpy(), 8, q.numpy())
    assert np.array_equal(I.cpu().numpy(), rI) and np.array_equal(D.cpu().numpy(), rD2)
    index.reset()
    assert index.ntotal == 0
    Dk, Ik = find_knn(FlatL2Index(), x.to(dev), neighbor=8)
    rD, rI = oracle_lib.find_knn(x.numpy(), 8)
    assert np.array_equal(Ik.cpu().numpy(), rI) and np.array_equal(Dk.cpu().numpy(), rD)


def test_flat_index_copies_its_points_and_streams_do_not_share_scratch(dev):
    """faiss copies on add(): mutating the caller's tensor afterwards must not change the index; find_knn refuses an
    index that still holds points (the reference resets it after every call).  Two streams running the hot path at
    the same time get scratch of their own (Workspace is keyed by stream and thread)."""
    from geoformer_b200.geodesic_utils import FlatL2Index, find_knn, knn_graph
    from geoformer_b200.guidance import geodesic_guidance

    x = scene(6000, 5).to(dev)
    keep = x.clone()
    index = FlatL2Index()
    index.add(x)
    x.mul_(3.0)  # the caller's tensor changes after add()
    D = torch.zeros(6000, 8, device=dev)
    I = torch.zeros(6000, 8, dtype=torch.int64, device=dev)
    index.search(keep, 8, D, I)
    rD, rI = knn_graph(keep, 8)
    assert torch.equal(I, rI) and torch.equal(torch.sqrt(D), rD)
    with pytest.raises(RuntimeError):
        find_knn(index, keep, neighbor=8)
    index.reset()
    Dk, Ik = find_knn(index, keep, neighbor=8)
    assert torch.equal(Ik, rI) and torch.equal(Dk, rD)
    xa, xb = scene(30000, 6).to(dev), scene(45000, 7).to(dev)
    want_a, want_b = geodesic_guidance(xa, 40, 16, 0.5, 20), geodesic_guidance(xb, 40, 16, 0.5, 20)
    torch.cuda.synchronize()
    sa, sb = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    for _ in range(4):
        with torch.cuda.stream(sa):
            ga = geodesic_guidance(xa, 40, 16, 0.5, 20)
        with torch.cuda.stream(sb):
            gb = geodesic_guidance(xb, 40, 16, 0.5, 20)
        torch.cuda.synchronize()
        assert torch.equal(ga[0], want_a[0]) and torch.equal(ga[1], want_a[1])
        assert torch.equal(gb[0], want_b[0]) and torch.equal(gb[1], want_b[1])


def test_knn_grid_equals_brute_at_full_size(dev):
    """c2 size (too slow for the CPU oracle in a unit test): the two GPU algorithms must agree."""
    from geoformer_b200.geodesic_utils import knn_graph

    x = scene(100_000, 1234).to(dev)
    Dg, Ig = knn_graph(x, 16, algo="grid")
    Db, Ib = knn_graph(x, 16, algo="brute")
    assert torch.equal(Ig, Ib) and torch.equal(Dg, Db)
    assert (Ig[:, 0] == torch.arange(100_000, device=dev)).all()  # distinct points: self is nearest
    assert (Dg[:, 1:] >= Dg[:, :-1]).all()  # sortedness


# ------------------------------------------------------------------------------------- geodesic
def _check_geodesic(oracle_lib, dev, x, Q, k, r, ms):
    from geoformer_b200.geodesic_utils import geodesic_from_graph, geodesic_from_points

    xn = x.numpy() if isinstance(x, torch.Tensor) else x
    xt = torch.from_numpy(np.ascontiguousarray(xn))
    seeds = oracle_lib.furthest_point_sampling(xn[None], Q)[0]
    rD, rI = oracle_lib.find_knn(xn, k)
    ref, R, lev = oracle_lib.geodesic(rD, rI, seeds, r, ms, return_stats=True)
    st = torch.from_numpy(seeds).to(dev)
    # (a) propagation only, on the oracle's graph, int64 indices (the faiss layout)
    geo_a, stats = geodesic_from_graph(torch.from_numpy(rD).to(dev), torch.from_numpy(rI).to(dev), st, r, ms,
                                       return_stats=True)
    # (b) fused kNN + propagation with the spatial renumbering
    geo_b = geodesic_from_points(xt.to(dev), st, k, r, ms)
    for geo in (geo_a, geo_b):
        g = geo.cpu().numpy()
        assert np.array_equal(g < 0, ref < 0), "unreachable sets differ"
        np.testing.assert_allclose(g, ref, rtol=1e-5, atol=0)  # north_star tolerance
        assert np.array_equal(g, ref), "expected bit-exact distances"
    assert int(stats[0]) == R and int(stats[1]) == lev
    return R


@pytest.mark.parametrize("N,Q,k,r,ms", [(400, 8, 6, 0.15, 4), (400, 8, 6, 10.0, 3), (2000, 16, 8, 0.2, 64),
                                        (3000, 32, 16, 0.5, 1), (3000, 33, 16, 0.3, 7), (20000, 64, 8, 0.5, 32),
                                        (20000, 64, 16, 0.1, 256), (20000, 300, 16, 0.5, 16),
                                        (5000, 8, 2, 0.5, 50), (5000, 8, 1, 0.5, 50), (5000, 8, 8, 0.5, 0),
                                        # many seeds per CTA: the claim / distance array is never reset between seeds
                                        (3000, 2500, 8, 0.3, 12), (6000, 3000, 16, 0.25, 40)])
def test_geodesic_matches_oracle(oracle_lib, dev, N, Q, k, r, ms):
    _check_geodesic(oracle_lib, dev, scene(N, 40 + N % 7), Q, k, r, ms)


def test_geodesic_config_c1(oracle_lib, dev):
    """BASELINE config 1: 50k points, 128 seeds, k=8, radius 0.5, max_step 32 (reach 9.1 %)."""
    R = _check_geodesic(oracle_lib, dev, scene(50_000, 1234), 128, 8, 0.5, 32)
    assert abs(R / (128 * 50_000) - 0.0910) < 5e-4


def test_geodesic_duplicate_points_and_seeds(oracle_lib, dev):
    """exact duplicates put a seed in its own neighbour row (the level-1 'no visited filter' quirk,
    geodesic_utils.py:123) and two queries on the same point must give identical rows"""
    from geoformer_b200.geodesic_utils import geodesic_from_graph

    x = scene(3000, 77).numpy().copy()
    x[10:20] = x[0:10]
    x[5] = x[2999]
    rD, rI = oracle_lib.find_knn(x, 8)
    seeds = np.array([12, 5, 2999, 0, 2, 12, 10, 700], dtype=np.int32)
    ref = oracle_lib.geodesic(rD, rI, seeds, 0.2, 40)
    geo = geodesic_from_graph(torch.from_numpy(rD).to(dev), torch.from_numpy(rI).to(dev), torch.from_numpy(seeds).to(dev),
                              0.2, 40).cpu().numpy()
    assert np.array_equal(geo, ref)
    assert np.array_equal(geo[0], geo[5])


def test_geodesic_foreign_graph_with_missing_neighbours(oracle_lib, dev):
    """a graph from a foreign index: -1 padded rows, int32 indices, self loops with non-zero length"""
    from geoformer_b200.geodesic_utils import geodesic_from_graph

    g = np.random.default_rng(4)
    N, k = 4000, 10
    rD, rI = oracle_lib.find_knn(scene(N, 9).numpy(), k)
    rI = rI.copy()
    rD = rD.copy()
    drop = g.random((N, k)) < 0.15
    rI[drop] = -1
    loops = g.integers(0, N, 50)
    rI[loops, 3] = loops
    rD[loops, 3] = 0.01
    seeds = np.concatenate([loops[:4], g.integers(0, N, 12)]).astype(np.int32)
    ref = oracle_lib.geodesic(rD, rI, seeds, 0.3, 30)
    geo = geodesic_from_graph(torch.from_numpy(rD).to(dev), torch.from_numpy(rI.astype(np.int32)).to(dev),
                              torch.from_numpy(seeds).to(dev), 0.3, 30).cpu().numpy()
    assert np.array_equal(geo, ref)


def test_cal_geodesic_vectorize_batch_api(oracle_lib, dev):
    """the reference entry point: ragged batch, list of (Q, N_b) tensors (geodesic_utils.py:91-164)"""
    from geoformer_b200.geodesic_utils import FlatL2Index, cal_geodesic_vectorize

    sizes = [3000, 1, 4500]
    pts = [scene(n, 60 + i) if n > 50 else torch.zeros(n, 3) for i, n in enumerate(sizes)]
    locs = torch.cat(pts)
    offsets = torch.tensor([0, 3000, 3001, 7501], dtype=torch.int32)
    Q = 16
    pre = np.zeros((3, 40), dtype=np.int32)
    pre[0] = oracle_lib.furthest_point_sampling(pts[0][None].numpy(), 40)[0]
    pre[2] = oracle_lib.furthest_point_sampling(pts[2][None].numpy(), 40)[0]
    ref = oracle_lib.cal_geodesic_vectorize(pre, locs.numpy(), offsets.numpy(), max_step=20, neighbor=8, radius=0.3,
                                            n_queries=Q)
    out = cal_geodesic_vectorize(FlatL2Index(), torch.from_numpy(pre).to(dev), locs.to(dev), offsets.to(dev),
                                 max_step=20, neighbor=8, radius=0.3, n_queries=Q)
    assert len(out) == 3
    for o, r in zip(out, ref):
        assert o.shape == r.shape and o.dtype == torch.float32 and o.is_cuda
        assert np.array_equal(o.cpu().numpy(), r)


def test_cal_geodesic_vectorize_batch_overlaps_scenes_and_stays_exact(dev):
    """A batch of 8 scenes runs on side streams inside cal_geodesic_vectorize: every map must equal the
    one-scene-at-a-time result, repeatedly (stream / workspace hazards would show up as differences), also
    when the caller consumes the result on its own non-default stream right away."""
    from geoformer_b200.geodesic_utils import cal_geodesic_vectorize, geodesic_from_points

    sizes = [20000, 35000, 1, 27000, 31000, 0, 22000, 40000]
    pts = [scene(n, 70 + i) if n > 50 else torch.zeros(n, 3) for i, n in enumerate(sizes)]
    locs = torch.cat(pts).to(dev)
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    Q = 32
    gen = torch.Generator().manual_seed(3)
    pre = torch.stack([torch.randint(0, max(n, 1), (48,), generator=gen) for n in sizes]).int().to(dev)
    singles = []
    for b, n in enumerate(sizes):
        lb = locs[int(offs[b]):int(offs[b + 1])].contiguous()
        singles.append(geodesic_from_points(lb, pre[b][:Q], 16, 0.5, 24) if n > 0 else None)
    torch.cuda.synchronize()
    user = torch.cuda.Stream(device=dev)
    for rep in range(3):
        with torch.cuda.stream(user):
            out = cal_geodesic_vectorize(None, pre, locs, torch.from_numpy(offs).to(dev), max_step=24, neighbor=16,
                                         radius=0.5, n_queries=Q)
            sums = [o.sum() if o.numel() else None for o in out]  # consumed on the caller's stream at once
        user.synchronize()
        for b, n in enumerate(sizes):
            assert out[b].shape == (Q, n)
            if n > 0:
                assert torch.equal(out[b], singles[b]), (rep, b)
                assert torch.equal(sums[b], singles[b].sum())


def test_full_size_config_c2(oracle_lib, dev):
    """BASELINE config 2 at full size (100k points, 256 seeds, k=16, radius 0.5, 32 levels) through the
    fused entry point: seeds == oracle FPS; kNN == oracle on ALL rows and == an independent float64 k-d tree;
    geodesic == oracle propagation on that graph, bit for bit; plus the size-independent properties (seed
    entries 0, unreachable exactly -1, idempotence, reach 13.1 %)."""
    from geoformer_b200.guidance import geodesic_guidance

    xc = scene(100_000, 1234)
    x = xc.to(dev)
    seeds, geo, D, I, stats = geodesic_guidance(x, 256, 16, 0.5, 32, return_graph=True, return_stats=True)
    seeds2, geo2 = geodesic_guidance(x, 256, 16, 0.5, 32)
    assert torch.equal(seeds, seeds2) and torch.equal(geo, geo2)  # idempotent / deterministic
    assert np.array_equal(seeds.cpu().numpy(), oracle_lib.furthest_point_sampling(xc[None].numpy(), 256)[0])
    # kNN: ALL 100k rows against the oracle (brute force, fp32, (d2, index) order: bit-exact) and against an
    # independent float64 k-d tree (tie-gap rule in _check_knn_against_kdtree)
    rD2, rI = oracle_lib.knn_sq(xc.numpy(), 16)
    assert np.array_equal(I.cpu().numpy(), rI.astype(np.int32))
    assert np.array_equal(D.cpu().numpy(), np.sqrt(rD2))
    differing = _check_knn_against_kdtree(xc.numpy(), np.arange(100_000), I.cpu().numpy(), D.cpu().numpy(), 16)
    assert differing < 100, differing  # only near-ties may be listed in another order (App. C scenes: a handful)
    ref, R, lev = oracle_lib.geodesic(D.cpu().numpy(), I.cpu().numpy().astype(np.int64), seeds.cpu().numpy(), 0.5, 32,
                                      return_stats=True)
    g = geo.cpu().numpy()
    assert np.array_equal(g < 0, ref < 0)
    np.testing.assert_allclose(g, ref, rtol=1e-5, atol=0)
    assert np.array_equal(g, ref)
    assert int(stats[0]) == R and int(stats[1]) == lev == 32
    q = torch.arange(256, device=dev)
    assert (geo[q, seeds.long()] == 0).all()
    assert (geo[geo < 0] == -1).all()
    assert abs(R / (256 * 100_000) - 0.131) < 2e-3  # SURVEY App. B


def test_full_size_config_c4(oracle_lib, dev):
    """BASELINE config 4 at full size (one 1M-point room, 512 seeds, k=16, radius 0.5, 32 levels): all 512 FPS
    seeds == oracle (whole-GPU FPS variant); 20 000 sampled kNN rows == oracle and == the float64 k-d tree; the
    propagation (the layout without on-chip bitmaps, which only scenes of this size select) == oracle
    propagation on the GPU's graph for ALL 512 seeds, bit for bit; row maxima; statistics."""
    from geoformer_b200.guidance import geodesic_guidance
    from geoformer_b200.scenes import room

    N, Q, k = 1_000_000, 512, 16
    xc = room(N, 4321)
    x = xc.to(dev)
    rm = torch.zeros(Q, device=dev)
    seeds, geo, D, I, stats = geodesic_guidance(x, Q, k, 0.5, 32, return_graph=True, return_stats=True, row_max=rm)
    xn = xc.numpy()
    assert np.array_equal(seeds.cpu().numpy(), oracle_lib.furthest_point_sampling(xn[None], Q)[0])
    rows = np.sort(np.random.default_rng(4).choice(N, 20_000, replace=False))
    In, Dn = I.cpu().numpy(), D.cpu().numpy()
    rD2, rI = oracle_lib.knn_sq(xn, k, xn[rows])
    assert np.array_equal(In[rows], rI.astype(np.int32))
    assert np.array_equal(Dn[rows], np.sqrt(rD2))
    assert _check_knn_against_kdtree(xn, rows, In[rows], Dn[rows], k) < 50
    ref, R, lev = oracle_lib.geodesic(Dn, In.astype(np.int64), seeds.cpu().numpy(), 0.5, 32, return_stats=True)
    g = geo.cpu().numpy()
    assert np.array_equal(g, ref)
    assert int(stats[0]) == R and int(stats[1]) == lev
    assert np.array_equal(rm.cpu().numpy(), ref.max(axis=1))


# ----------------------------------------------------------------------------------------- bias
def test_bias_epilogues(oracle_lib, dev):
    from oracle import bias as obias

    from geoformer_b200.bias import decoder_relative_pos, mask_head_relative_coords
    from geoformer_b200.geodesic_utils import geodesic_from_points

    B, Q, Cn = 2, 32, 256
    geos, pres, qlocs, clocs, xs = [], [], [], [], []
    for b in range(B):
        x = scene(6000 + 500 * b, 90 + b)
        pre = torch.from_numpy(oracle_lib.furthest_point_sampling(x[None].numpy(), Cn)[0])
        geo = geodesic_from_points(x.to(dev), pre[:Q].to(dev), 8, 0.3, 6 if b == 0 else 0)
        geos.append(geo)
        pres.append(pre)
        clocs.append(x[pre.long()])
        qlocs.append(x[pre[:Q].long()])
        xs.append(x)
    pre_t, ql, cl = torch.stack(pres), torch.stack(qlocs), torch.stack(clocs)
    out = decoder_relative_pos(geos, pre_t.to(dev), ql.to(dev), cl.to(dev)).cpu()
    ref = obias.decoder_relative_pos([g.cpu() for g in geos], pre_t, ql, cl)
    assert out.shape == (B, Q, Cn, 3)
    torch.testing.assert_close(out, ref, rtol=1e-6, atol=0)
    assert torch.equal(out, ref)
    # synthetic maps that exercise the "row without any reachable entry takes the global max" branch
    gsyn = [torch.rand(Q, x.shape[0], generator=torch.Generator().manual_seed(5)) for x in xs]
    for gsy in gsyn:
        gsy[torch.rand(gsy.shape, generator=torch.Generator().manual_seed(6)) < 0.6] = -1.0
        gsy[3] = -1.0
        gsy[17] = -1.0
    out = decoder_relative_pos([gg.to(dev) for gg in gsyn], pre_t.to(dev), ql.to(dev), cl.to(dev)).cpu()
    assert torch.equal(out, obias.decoder_relative_pos(gsyn, pre_t, ql, cl))
    msyn = mask_head_relative_coords(gsyn[0].to(dev), xs[0].to(dev), ql[0].to(dev)).cpu()
    assert torch.equal(msyn, obias.mask_head_relative_coords(gsyn[0], xs[0], ql[0]))
    for b in range(B):
        m = mask_head_relative_coords(geos[b], xs[b].to(dev), ql[b].to(dev)).cpu()
        rm = obias.mask_head_relative_coords(geos[b].cpu(), xs[b], ql[b])
        assert m.shape == (Q, 3, xs[b].shape[0])
        torch.testing.assert_close(m, rm, rtol=1e-6, atol=0)
        assert torch.equal(m, rm)


def test_guidance_runner_cuda_graph(dev):
    """The fused path (forked FPS stream included) captured into a CUDA graph replays to the same bits, also
    when run() is handed another scene than the one it was captured with; the caller's tensors are never
    written (the graph reads a private staging buffer)."""
    from geoformer_b200.guidance import GuidanceRunner, geodesic_guidance

    xa, xb = scene(40000, 31).to(dev), scene(40000, 32).to(dev)
    keep = {id(xa): xa.clone(), id(xb): xb.clone()}
    want = {id(x): geodesic_guidance(x, 64, 16, 0.5, 20) for x in (xa, xb)}
    torch.cuda.synchronize()
    r = GuidanceRunner(40000, 64, 16, 0.5, 20, device=dev, graph=True)
    side = torch.cuda.Stream(device=dev)
    for x in (xa, xb, xa, xb):
        seeds, geo = r.run(x, side)
        side.synchronize()
        assert torch.equal(x, keep[id(x)]), "run() must not write the caller's points"
        ref_seeds, ref_geo = want[id(x)]
        assert torch.equal(seeds, ref_seeds) and torch.equal(geo, ref_geo)
        assert torch.equal(r.row_max, ref_geo.max(dim=1).values)
    assert not torch.equal(want[id(xa)][1], want[id(xb)][1])
    # bbox+plan | coarse count+plan | count | scan | scatter | query (+ edge table) | propagation | FPS
    assert r.launches_per_run == 8


def test_guidance_batch_equals_per_scene_calls_and_oracle(oracle_lib, dev):
    """gf_guidance_batch (graphs side by side, ONE propagation launch over all (scene, seed) pairs) on a ragged
    batch: bit-identical to the per-scene call for every scene, to the oracle for two of them; seeds given or
    sampled; row maxima and per-scene statistics."""
    from geoformer_b200.guidance import geodesic_guidance, geodesic_guidance_batch

    sizes = [20000, 31111, 12345, 50000, 777, 20000, 16384]
    xs = [scene(n, 40 + i).to(dev) for i, n in enumerate(sizes)]
    Q, k, r, ms = 40, 16, 0.5, 24
    seeds, geos, stats, rmax = geodesic_guidance_batch(xs, Q, k, r, ms, return_stats=True, row_max=True)
    for i, x in enumerate(xs):
        s1, g1, st1 = geodesic_guidance(x, Q, k, r, ms, return_stats=True)
        assert torch.equal(seeds[i], s1) and torch.equal(geos[i], g1), i
        assert torch.equal(stats[i], st1), (i, stats[i], st1)
        assert torch.equal(rmax[i], g1.max(dim=1).values), i
    for i in (2, 4):
        xn = xs[i].cpu().numpy()
        rs = oracle_lib.furthest_point_sampling(xn[None], Q)[0]
        rD, rI = oracle_lib.find_knn(xn, k)
        assert np.array_equal(seeds[i].cpu().numpy(), rs)
        assert np.array_equal(geos[i].cpu().numpy(), oracle_lib.geodesic(rD, rI, rs, r, ms))
    # seeds given (the body of cal_geodesic_vectorize), more scenes than one library call takes (32): a full call + 3
    many = [xs[i % len(xs)] for i in range(35)]
    given = [torch.randperm(x.size(0), generator=torch.Generator().manual_seed(j))[:Q].int() for j, x in enumerate(many)]
    _, geos2 = geodesic_guidance_batch(many, Q, k, r, ms, seeds=given)
    from geoformer_b200.geodesic_utils import geodesic_from_points
    for j, x in enumerate(many):
        assert torch.equal(geos2[j], geodesic_from_points(x, given[j].to(dev), k, r, ms)), j


def test_batch_guidance_runner_graph_and_stage_events(dev):
    """BatchGuidanceRunner: plain and CUDA-graph replay give the bits of the per-scene call; the two stage events
    that bracket the propagation launch are stamped by every replay (external event record nodes)."""
    from geoformer_b200.guidance import BatchGuidanceRunner, geodesic_guidance

    N, B, Q, k = 30000, 3, 48, 16
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
        # per scene: bbox | coarse count | count | scan | scatter | query (+ edge table), FPS; one propagation launch
        assert r.launches_per_run == 7 * B + 1, r.launches_per_run
        r.close()


def test_batch_host_entry_point_equals_device_path(dev):
    """gf_guidance_batch_host: pinned host points in, seeds + maps back in pinned host memory == the device path"""
    from geoformer_b200.guidance import HostBatchGuidance, geodesic_guidance

    N, B, Q, k = 25000, 3, 32, 16
    xs = [scene(N, 80 + i) for i in range(B)]
    h = HostBatchGuidance(N, B, Q, k, 0.5, 18, device=dev)
    for rep in range(2):
        seeds, geo = h.run([x.pin_memory() for x in xs])
        for b, x in enumerate(xs):
            rs, rg = geodesic_guidance(x.to(dev), Q, k, 0.5, 18)
            assert torch.equal(seeds[b], rs.cpu()) and torch.equal(geo[b], rg.cpu()), (rep, b)


def test_row_max_by_product(oracle_lib, dev):
    """The propagation can hand out the maximum of every row (what both epilogues start from); it must be
    exactly geo.max(dim=1), also for rows that stay empty, and the mask-head epilogue fed with it must
    produce the same bits as when it reduces the maps itself."""
    from geoformer_b200.bias import mask_head_relative_coords
    from geoformer_b200.geodesic_utils import geodesic_from_graph, geodesic_from_points, knn_graph
    from geoformer_b200.guidance import geodesic_guidance

    x = scene(30000, 21).to(dev)
    for ms in (0, 1, 2, 7, 40):
        rm = torch.full((48,), 123.0, device=dev)
        seeds, geo = geodesic_guidance(x, 48, 16, 0.5, ms, row_max=rm)
        assert torch.equal(rm, geo.max(dim=1).values), ms
        out_a = mask_head_relative_coords(geo, x, x[seeds.long()].contiguous(), row_max=rm)
        out_b = mask_head_relative_coords(geo, x, x[seeds.long()].contiguous())
        assert torch.equal(out_a, out_b), ms
    # seeded entry points, out-of-range seeds (rows stay -1), duplicate seeds, unaligned N
    x2 = scene(10001, 22).to(dev)
    D, I = knn_graph(x2, 8)
    seeds = torch.tensor([5, -1, 10001, 5, 9999, 0], dtype=torch.int32, device=dev)
    rm = torch.zeros(6, device=dev)
    geo = geodesic_from_graph(D, I, seeds, 0.3, 12, row_max=rm)
    assert torch.equal(rm, geo.max(dim=1).values) and rm[1] == -1 and rm[2] == -1
    rm2 = torch.zeros(6, device=dev)
    geo2 = geodesic_from_points(x2, seeds, 8, 0.3, 12, row_max=rm2)
    assert torch.equal(geo2, geo) and torch.equal(rm2, rm)
    sx = x2[seeds.clamp(0, 10000).long()].contiguous()
    assert torch.equal(mask_head_relative_coords(geo, x2, sx, row_max=rm), mask_head_relative_coords(geo, x2, sx))


def test_epilogues_match_reference_lines_fixture(dev):
    """both epilogue kernels against tests/golden/bias_golden.npz = outputs of the reference's OWN statements
    (geoformer_fs.py:263-300, :680-702 executed from source, oracle/ref_bias.py).  Bit-exact incl. the NaN case."""
    import os

    from geoformer_b200.bias import decoder_relative_pos, mask_head_relative_coords

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bias_golden.npz"))
    T = lambda a: torch.from_numpy(np.array(a)).to(dev)  # noqa: E731
    for i in range(int(g["n_mask"])):
        geo = T(g["m%d_geo" % i])
        out = mask_head_relative_coords(geo, T(g["m%d_coords" % i]), T(g["m%d_seed_xyz" % i]))
        assert np.array_equal(out.cpu().numpy(), g["m%d_out" % i], equal_nan=True), i
        out2 = mask_head_relative_coords(geo, T(g["m%d_coords" % i]), T(g["m%d_seed_xyz" % i]),
                                         row_max=geo.max(dim=1).values.contiguous())
        assert np.array_equal(out2.cpu().numpy(), g["m%d_out" % i], equal_nan=True), i
    for i in range(int(g["n_dec"])):
        B = int(g["d%d_B" % i])
        out = decoder_relative_pos([T(g["d%d_geo%d" % (i, b)]) for b in range(B)], T(g["d%d_inds" % i]),
                                   T(g["d%d_qry" % i]), T(g["d%d_ctx" % i]))
        assert np.array_equal(out.cpu().numpy(), g["d%d_out" % i], equal_nan=True), i


def test_decoder_fourier_embedding(dev):
    """geoformer_fs.py:680-712 fused (gather -> fill -> normalise -> 3x32 projection -> sin|cos) against the
    fixture produced by the reference's own PositionEmbeddingCoordsSine, and against the torch restatement
    at the model's shapes.  Tolerance 2e-5 absolute: the order of the 3-term dot product (torch.mm) and the
    last ulp of sinf/cosf at arguments of up to ~50 rad."""
    import os

    from oracle import bias as obias

    from geoformer_b200.bias import decoder_relative_embedding

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fourier_golden.npz"))
    t = {k: torch.from_numpy(g[k]) for k in g.files}
    out = decoder_relative_embedding([t["geo0"].to(dev), t["geo1"].to(dev)], t["inds"].to(dev), t["qry"].to(dev),
                                     t["ctx"].to(dev), t["gauss_B"].to(dev), [t["pc_min"].to(dev), t["pc_max"].to(dev)])
    assert out.shape == (12, 40, 2, 64) and out.stride() == (40 * 64, 64, 12 * 40 * 64, 1)  # the reference's view
    torch.testing.assert_close(out.cpu().contiguous(), t["emb"], rtol=0, atol=2e-5)
    # model shapes: B=1, Q=256 queries, C=2048 contexts, d_pos=64; ragged context count and a narrower embedding too
    # ... and embeddings whose half width d_out is below 32 or not a multiple of 32 (dec_dim = 32 -> d_out = 16,
    # num_channels = 96 -> d_out = 48): lanes without a frequency must still take part in the warp's shuffles
    for Q, Cn, d_pos, nch in ((256, 2048, 64, None), (37, 301, 64, None), (16, 100, 96, 64), (19, 77, 32, None),
                              (23, 130, 96, None), (8, 33, 128, 96)):
        gen = torch.Generator().manual_seed(Q)
        N = 20000
        geo = torch.rand(Q, N, generator=gen) * 4.0
        geo[torch.rand(Q, N, generator=gen) < 0.5] = -1.0
        geo[1] = -1.0
        x = scene(N, 3)
        inds = torch.randperm(N, generator=gen)[:Cn].int()[None]
        ctx = x[inds[0].long()][None].contiguous()
        qry = ctx[:, :Q].contiguous()
        gb = torch.randn(3, d_pos // 2, generator=gen)
        pc = [x.min(0)[0][None].contiguous(), x.max(0)[0][None].contiguous()]
        ours = decoder_relative_embedding([geo.to(dev)], inds.to(dev), qry.to(dev), ctx.to(dev), gb.to(dev),
                                          [pc[0].to(dev), pc[1].to(dev)], num_channels=nch).cpu()
        ref = obias.decoder_relative_embedding([geo], inds, qry, ctx, gb if nch is None else gb[:, : nch // 2], pc)
        assert ours.shape == ref.shape
        torch.testing.assert_close(ours.contiguous(), ref.contiguous(), rtol=0, atol=2e-5)


# ------------------------------------------------------------------------- python surface / e2e
def test_group_points_pipeline_and_autograd(oracle_lib, dev):
    """set_aggregator.group_points chain (pointnet2_modules.py:200-226): FPS -> gather -> ball query ->
    group -> centre -> concat, and gradients through gather / group."""
    from geoformer_b200 import pointnet2_utils as pu

    x = scene(5000, 5)[None]
    feats = torch.randn(1, 16, 5000, generator=torch.Generator().manual_seed(0))
    grouper = pu.QueryAndGroup(0.2, 64, use_xyz=True, ret_grouped_xyz=True, normalize_xyz=True)
    fd = feats.to(dev).requires_grad_(True)
    new_xyz, gf, gx, inds = pu.group_points(x.to(dev), fd, grouper, 128)
    r_inds = oracle_lib.furthest_point_sampling(x.numpy(), 128)
    assert np.array_equal(inds.cpu().numpy(), r_inds)
    r_new = oracle_lib.gather_points(x.transpose(1, 2).contiguous().numpy(), r_inds).transpose(0, 2, 1)
    assert np.array_equal(new_xyz.cpu().numpy(), r_new)
    r_idx = oracle_lib.ball_query(np.ascontiguousarray(r_new), x.numpy(), 0.2, 64)
    r_gx = oracle_lib.group_points(x.transpose(1, 2).contiguous().numpy(), r_idx)
    r_gx_raw = torch.from_numpy(r_gx) - torch.from_numpy(np.ascontiguousarray(r_new)).transpose(1, 2).unsqueeze(-1)
    r_gx = r_gx_raw / 0.2
    # torch's CUDA `/= scalar` multiplies by the reciprocal (not our kernel): allow its 1-ulp difference
    torch.testing.assert_close(gx.cpu(), r_gx, rtol=1e-6, atol=1e-7)
    grouper_raw = pu.QueryAndGroup(0.2, 64, use_xyz=True, ret_grouped_xyz=True, normalize_xyz=False)
    _, _, gx_raw, _ = pu.group_points(x.to(dev), fd, grouper_raw, 128)
    assert torch.equal(gx_raw.cpu(), r_gx_raw)
    assert gf.shape == (1, 19, 128, 64)
    assert np.array_equal(gf[:, 3:].detach().cpu().numpy(), oracle_lib.group_points(feats.numpy(), r_idx))
    gf.sum().backward()
    counts = np.bincount(r_idx.reshape(-1), minlength=5000).astype(np.float32)
    np.testing.assert_allclose(fd.grad[0, 0].cpu().numpy(), counts, rtol=0, atol=0)


def test_host_entry_point_equals_device_path(oracle_lib, dev):
    from geoformer_b200.guidance import HostGuidance, geodesic_guidance

    x = scene(30_000, 8)
    hg = HostGuidance(30_000, 64, 8, 0.5, 16)
    seeds_h, geo_h = hg.run(x)
    seeds_d, geo_d = geodesic_guidance(x.to(dev), 64, 8, 0.5, 16)
    assert torch.equal(seeds_h, seeds_d.cpu()) and torch.equal(geo_h, geo_d.cpu())
    assert np.array_equal(seeds_h.numpy(), oracle_lib.furthest_point_sampling(x[None].numpy(), 64)[0])
    rD, rI = oracle_lib.find_knn(x.numpy(), 8)
    assert np.array_equal(geo_h.numpy(), oracle_lib.geodesic(rD, rI, seeds_h.numpy(), 0.5, 16))
