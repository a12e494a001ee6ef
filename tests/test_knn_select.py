"""The grid kNN query selects each query's candidates in its first shell by counting them into distance bins and
inserting only those at or below the bin that holds the k-th (gf_knn.cu, knn_grid_query_kernel).  These inputs aim
at that selection: many candidates tied at the threshold distance, more tied candidates than the per-lane list
holds (the query then offers every candidate), shells holding fewer than k points, flat and line-like scenes, and
k that is not a power of two (the general edge-table path of the fused hot path).  Every result must equal the CPU
oracle and the brute-force kernel bit for bit."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from geoformer_b200.scenes import scene  # noqa: E402

KS = [1, 8, 15, 16, 17, 32]


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _lattice(seed):
    """a 24 x 24 x 12 lattice of spacing 0.25 (every distance is tied many times) with a few jittered points"""
    g = np.random.default_rng(seed)
    ax = [np.arange(n, dtype=np.float32) * np.float32(0.25) for n in (24, 24, 12)]
    x = np.stack(np.meshgrid(*ax, indexing="ij"), -1).reshape(-1, 3)
    x = x[g.permutation(len(x))]
    x[:50] += g.random((50, 3), dtype=np.float32) * np.float32(0.01)
    return np.ascontiguousarray(x)


def _duplicate_clusters(seed):
    """a scene with clusters of 10 .. 200 copies of one point: more points at d2 = 0 than a query's list holds"""
    g = np.random.default_rng(seed)
    x = scene(8000, seed).numpy().copy()
    at = 0
    for n in (10, 40, 49, 80, 200):
        x[at:at + n] = x[at + n + 7]
        at += n + 10
    return x[g.permutation(len(x))]


def _sparse_outliers(seed):
    """a dense scene plus points scattered far from it and from each other: their first shell holds fewer than k"""
    g = np.random.default_rng(seed)
    x = scene(6000, seed).numpy()
    far = (g.random((60, 3)) * 400.0 - 200.0).astype(np.float32)
    pairs = far[:10] + np.float32(0.003)  # a few outliers with one close companion
    return np.ascontiguousarray(np.concatenate([x, far, pairs])[g.permutation(len(x) + 70)])


def _flat(seed):
    g = np.random.default_rng(seed)
    x = g.random((7000, 3), dtype=np.float32) * np.float32(3.0)
    x[:, 1] = np.float32(-0.5)
    return x


def _line(seed):
    g = np.random.default_rng(seed)
    x = np.zeros((5000, 3), np.float32)
    x[:, 2] = g.random(5000, dtype=np.float32) * np.float32(20.0)
    x[::3, 0] = np.float32(1e-3)  # a second, parallel line very close to the first
    return x


SCENES = {"lattice": _lattice, "duplicates": _duplicate_clusters, "outliers": _sparse_outliers, "flat": _flat,
          "line": _line}


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("name", sorted(SCENES))
def test_knn_select_matches_oracle_and_brute(oracle_lib, dev, name, k):
    from geoformer_b200.geodesic_utils import knn_graph

    x = SCENES[name](11)
    xt = torch.from_numpy(x).to(dev)
    D, I = knn_graph(xt, k, algo="grid")
    Db, Ib = knn_graph(xt, k, algo="brute")
    assert torch.equal(I, Ib) and torch.equal(D, Db)
    rD, rI = oracle_lib.find_knn(x, k)
    assert np.array_equal(I.cpu().numpy(), rI)
    assert np.array_equal(D.cpu().numpy(), rD)


@pytest.mark.parametrize("k", [8, 17])
def test_knn_select_external_queries(oracle_lib, dev, k):
    """queries that are not the indexed points (FlatL2Index.search): some inside the lattice, some far outside"""
    from geoformer_b200.geodesic_utils import FlatL2Index

    x = _lattice(3)
    g = np.random.default_rng(4)
    q = np.concatenate([x[:300] + np.float32(0.125), (g.random((40, 3)) * 30.0 - 15.0).astype(np.float32)])
    index = FlatL2Index()
    index.add(torch.from_numpy(x).to(dev))
    D = torch.zeros(len(q), k, device=dev)
    I = torch.zeros(len(q), k, dtype=torch.int64, device=dev)
    index.search(torch.from_numpy(q).to(dev), k, D, I)
    rD2, rI = oracle_lib.knn_sq(x, k, q)
    assert np.array_equal(I.cpu().numpy(), rI) and np.array_equal(D.cpu().numpy(), rD2)


def test_knn_select_more_than_65535_tied_points(dev):
    """one point repeated 66000 times: a shell too large for the 16-bit bin counts is offered candidate by candidate"""
    from geoformer_b200.geodesic_utils import knn_graph

    x = scene(3000, 8).numpy()
    x = np.concatenate([np.repeat(x[:1], 66000, axis=0), x])
    xt = torch.from_numpy(x).to(dev)
    D, I = knn_graph(xt, 16, algo="grid")
    Db, Ib = knn_graph(xt, 16, algo="brute")
    assert torch.equal(I, Ib) and torch.equal(D, Db)
    assert (I[:66000] == torch.arange(16, device=dev)).all()  # ties broken by index


@pytest.mark.parametrize("k", [15, 16, 17])
def test_guidance_batch_on_select_scenes(oracle_lib, dev, k):
    """the fused hot path (kNN edge table written by the query kernel, one propagation launch for the batch) on the
    scenes above: bit-identical to the per-scene call, and to the oracle's maps"""
    from geoformer_b200.guidance import geodesic_guidance, geodesic_guidance_batch

    xs_np = [SCENES[n](21) for n in sorted(SCENES)]
    xs = [torch.from_numpy(x).to(dev) for x in xs_np]
    Q, r, ms = 24, 0.5, 24
    seeds, geos = geodesic_guidance_batch(xs, Q, k, r, ms)
    for i, x in enumerate(xs):
        s1, g1 = geodesic_guidance(x, Q, k, r, ms)
        assert torch.equal(seeds[i], s1) and torch.equal(geos[i], g1), i
        rs = oracle_lib.furthest_point_sampling(xs_np[i][None], Q)[0]
        rD, rI = oracle_lib.find_knn(xs_np[i], k)
        assert np.array_equal(seeds[i].cpu().numpy(), rs), i
        assert np.array_equal(geos[i].cpu().numpy(), oracle_lib.geodesic(rD, rI, rs, r, ms)), i
