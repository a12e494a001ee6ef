"""CPU tests (no GPU): the oracle against the committed golden fixtures and against independent
restatements, so that the checker itself is pinned before it is used to judge the CUDA path."""
import glob
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLD, "geodesic_*.npz"))), ids=os.path.basename)
def test_oracle_geodesic_matches_reference_fixture(oracle_lib, path):
    """fixtures = the reference's own cal_geodesic_vectorize on CPU (tests/golden/make_golden.py)"""
    g = np.load(path)
    D, I = oracle_lib.find_knn(g["xyz"], int(g["k"]))
    assert np.array_equal(I, g["knn_idx"]) and np.array_equal(D, g["knn_dist"])
    geo = oracle_lib.geodesic(D, I, g["seeds"], float(g["radius"]), int(g["max_step"]))
    assert np.array_equal(geo < 0, g["geo"] < 0)
    assert np.array_equal(geo, g["geo"])


def test_golden_fixtures_exist():
    assert len(glob.glob(os.path.join(GOLD, "geodesic_*.npz"))) >= 4


def _fps_by_key_rule(xyz, m, rank=None):
    """Independent restatement of FPS through the closed-form tie rule of SURVEY F6(b): among equal maxima
    the winner is the k with the smallest (bitrev_L(k mod bs), k div bs).  `rank` (n,) replaces that order
    with another one (smallest rank wins), e.g. np.arange(n) for the lowest index.  Exact wherever the float64
    emulation of sq3 is, which includes every input on a coarse lattice."""
    n = xyz.shape[0]
    L = 0
    while (2 << L) <= n and L < 9:
        L += 1
    bs = 1 << L
    x, y, z = (xyz[:, i].astype(np.float32) for i in range(3))
    f32 = np.float32

    def sq3(a, b, c):  # fma(c,c, fma(a,a, b*b)) emulated in float64 -> float32 (exact for fp32 inputs)
        bb = (b.astype(np.float64) * b.astype(np.float64)).astype(f32)
        t = (a.astype(np.float64) * a.astype(np.float64) + bb.astype(np.float64)).astype(f32)
        return (c.astype(np.float64) * c.astype(np.float64) + t.astype(np.float64)).astype(f32)

    elig = ~(sq3(x, y, z).astype(np.float64) <= 1e-3)
    temp = np.full(n, 1e10, dtype=f32)
    if rank is None:
        k = np.arange(n, dtype=np.int64)
        rev = sum(((k % bs >> b) & 1) << (L - 1 - b) for b in range(L)) if L else np.zeros(n, dtype=np.int64)
        rank = (rev << 23) | (k // bs)
    rank = np.asarray(rank, dtype=np.int64)
    idx = np.zeros(m, dtype=np.int32)
    old = 0
    for j in range(1, m):
        d = sq3(x - x[old], y - y[old], z - z[old])
        temp = np.where(elig, np.minimum(d, temp), temp)
        if not elig.any():
            old = 0
        else:
            best = temp[elig].max()
            cand = np.nonzero(elig & (temp == best))[0]
            old = int(cand[np.argmin(rank[cand])])
        idx[j] = old
    return idx


@pytest.mark.parametrize("n,m,lattice", [(5, 5, False), (200, 40, False), (777, 60, True), (3000, 64, True)])
def test_oracle_fps_against_closed_form_tie_rule(oracle_lib, n, m, lattice):
    g = np.random.default_rng(n)
    if lattice:  # many exact ties and points inside the |p|^2 <= 1e-3 ball
        xyz = g.integers(-3, 4, size=(n, 3)).astype(np.float32) * 0.25
        xyz[g.integers(0, n, size=n // 20)] = 0.0
    else:
        xyz = g.normal(size=(n, 3)).astype(np.float32)
    assert np.array_equal(oracle_lib.furthest_point_sampling(xyz[None], m)[0], _fps_by_key_rule(xyz, m))


def test_oracle_knn_against_numpy(oracle_lib):
    g = np.random.default_rng(1)
    x = g.normal(size=(700, 3)).astype(np.float32)
    x[50:60] = x[40:50]  # duplicates: ordering by index among equal distances
    D2, I = oracle_lib.knn_sq(x, 9)
    d = (x[None, :, :] - x[:, None, :]).astype(np.float64)  # the differences are rounded to fp32 first
    # fma(dz,dz, fma(dx,dx, dy*dy)) in float64 -> float32 steps
    t = ((d[..., 1] * d[..., 1]).astype(np.float32).astype(np.float64) + d[..., 0] * d[..., 0]).astype(np.float32)
    d2 = (t.astype(np.float64) + d[..., 2] * d[..., 2]).astype(np.float32)
    order = np.lexsort((np.broadcast_to(np.arange(700), d2.shape), d2), axis=1)[:, :9]
    assert np.array_equal(I, order)
    assert np.array_equal(D2, np.take_along_axis(d2, order, axis=1))
    # fewer points than k: -1 / +inf padding
    D2s, Is = oracle_lib.knn_sq(x[:4], 6)
    assert (Is[:, 4:] == -1).all() and np.isinf(D2s[:, 4:]).all() and (Is[:, :4] >= 0).all()


def test_oracle_ball_query_and_grouping_semantics(oracle_lib):
    g = np.random.default_rng(2)
    xyz = g.random((1, 500, 3)).astype(np.float32)
    centres = xyz[:, :7].copy()
    centres[0, 0] += 50  # nothing in range
    idx = oracle_lib.ball_query(centres, xyz, 0.2, 16)
    assert (idx[0, 0] == 0).all()
    for j in range(1, 7):
        d2 = ((xyz[0] - centres[0, j]) ** 2).sum(1)
        hits = np.nonzero(d2 < 0.2 * 0.2 - 1e-6)[0][:16]
        row = idx[0, j]
        assert np.array_equal(row[: len(hits)], hits[: len(row)]) or len(hits) == 16
        assert (row[len(hits):] == row[0]).all() or len(hits) >= 16
    feats = g.normal(size=(1, 4, 500)).astype(np.float32)
    grouped = oracle_lib.group_points(feats, idx)
    assert np.array_equal(grouped[0, 2, 3], feats[0, 2, idx[0, 3]])
    gathered = oracle_lib.gather_points(feats, idx[:, :, 0].copy())
    assert np.array_equal(gathered[0, 1], feats[0, 1, idx[0, :, 0]])


def test_oracle_geodesic_level_semantics(oracle_lib):
    """hand-built graph: first-visit wins, smallest parent index wins inside a level, radius filter,
    -1 neighbours, max_step bound"""
    inf = np.float32(9.0)
    #          self  n1   n2
    I = np.array([[0, 1, 2], [1, 3, -1], [2, 3, 4], [3, 5, -1], [4, 5, -1], [5, -1, -1]], dtype=np.int64)
    D = np.array([[0, 1.0, 1.5], [0, 1.0, inf], [0, 0.25, 1.0], [0, 1.0, inf], [0, 0.5, inf], [0, inf, inf]],
                 dtype=np.float32)
    geo = oracle_lib.geodesic(D, I, np.array([0]), 2.0, 10)[0]
    # level 1: 1 (1.0), 2 (1.5).  level 2: 3 is offered by 1 (2.0) and 2 (1.75): parent 1 wins (smaller index),
    # although 2's path is shorter -> NOT a shortest path.  4 via 2 (2.5).  level 3: 5 via 3 (3.0), not via 4 (3.0)
    assert geo.tolist() == [0.0, 1.0, 1.5, 2.0, 2.5, 3.0]
    geo2 = oracle_lib.geodesic(D, I, np.array([0]), 2.0, 2)[0]
    assert geo2.tolist() == [0.0, 1.0, 1.5, 2.0, 2.5, -1.0]
    geo3 = oracle_lib.geodesic(D, I, np.array([0]), 1.2, 10)[0]  # the 1.5 edge is outside the radius
    assert geo3.tolist() == [0.0, 1.0, -1.0, 2.0, -1.0, 3.0]


# ---- fixtures produced by the reference's own CUDA kernels on the GPU box ----------------------------
# (tests/golden/make_golden_ref_ext.py; oracle/_ref = lib/pointnet2/_ext_src compiled unmodified)
@pytest.fixture(scope="module")
def ref_ext_golden():
    path = os.path.join(GOLD, "ref_ext_golden.npz")
    if not os.path.exists(path):
        pytest.skip("ref_ext_golden.npz not generated yet")
    return np.load(path)


def test_oracle_fps_matches_reference_kernel_fixture(oracle_lib, ref_ext_golden):
    g = ref_ext_golden
    names = sorted(k[4:-4] for k in g.files if k.startswith("fps_") and k.endswith("_idx"))
    assert len(names) >= 6
    for name in names:
        xyz, m, idx = g["fps_%s_xyz" % name], int(g["fps_%s_m" % name]), g["fps_%s_idx" % name]
        assert np.array_equal(oracle_lib.furthest_point_sampling(xyz, m), idx), name


def test_oracle_ball_query_group_gather_match_reference_kernel_fixture(oracle_lib, ref_ext_golden):
    g = ref_ext_golden
    for tag in ("a", "b"):
        out = oracle_lib.ball_query(g["bq_centres"], g["bq_xyz"], float(g["bq_%s_r" % tag]), int(g["bq_%s_ns" % tag]))
        assert np.array_equal(out, g["bq_%s_idx" % tag]), tag
    assert np.array_equal(oracle_lib.group_points(g["grp_feats"], g["bq_a_idx"]), g["grp_out"])
    assert np.array_equal(oracle_lib.gather_points(g["grp_feats"], np.ascontiguousarray(g["bq_a_idx"][:, :, 0])), g["gat_out"])


def test_oracle_three_nn_interpolate_match_reference_kernel_fixture(oracle_lib, ref_ext_golden):
    g = ref_ext_golden
    d2, idx = oracle_lib.three_nn(g["tnn_unknown"], g["tnn_known"])
    assert np.array_equal(idx, g["tnn_idx"]) and np.array_equal(d2, g["tnn_d2"])
    assert np.array_equal(oracle_lib.three_interpolate(g["ti_feats"], idx, g["ti_w"]), g["ti_out"])
    d2s, idxs = oracle_lib.three_nn(g["tnn_unknown"][:, :10], g["tnn_known"][:, :2])
    assert np.array_equal(idxs, g["tnn_small_idx"]) and np.array_equal(d2s, g["tnn_small_d2"])


# ---- decoder relative-position embedding (geoformer_fs.py:680-712) ----------------------------------
# fixture = the reference's own PositionEmbeddingCoordsSine applied on CPU (tests/golden/make_golden_fourier.py)
def _fourier_fixture():
    import torch

    g = np.load(os.path.join(GOLD, "fourier_golden.npz"))
    t = {k: torch.from_numpy(g[k]) for k in g.files}
    return t


def test_oracle_fourier_embedding_matches_reference_module_fixture():
    import torch

    from oracle import bias as obias

    t = _fourier_fixture()
    emb = obias.decoder_relative_embedding([t["geo0"], t["geo1"]], t["inds"], t["qry"], t["ctx"], t["gauss_B"],
                                           [t["pc_min"], t["pc_max"]])
    assert emb.shape == t["emb"].shape == (12, 40, 2, 64)
    # same torch ops on the same platform class (CPU); allow the last ulps of sin/cos across torch builds
    torch.testing.assert_close(emb.contiguous(), t["emb"], rtol=0, atol=2e-6)
    # the [sin | cos] halves are consistent
    s, c = emb[..., :32], emb[..., 32:]
    torch.testing.assert_close(s * s + c * c, torch.ones_like(s), rtol=0, atol=1e-5)


def _bias_golden():
    import torch

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bias_golden.npz"))
    return g, (lambda a: torch.from_numpy(np.array(a)))


def test_bias_oracle_matches_reference_lines_fixture():
    """oracle/bias.py against tests/golden/bias_golden.npz = outputs of the reference's OWN epilogue statements
    (geoformer_fs.py:263-300 and :680-702, executed from source by oracle/ref_bias.py).  Bit-exact, NaN included
    (a matrix with nothing reachable makes the reference take sqrt(-1))."""
    import torch

    from oracle import bias as obias

    g, T = _bias_golden()
    assert tuple(g["mask_lines"]) == (263, 300) and tuple(g["dec_lines"]) == (680, 702)
    for i in range(int(g["n_mask"])):
        out = obias.mask_head_relative_coords(T(g["m%d_geo" % i]), T(g["m%d_coords" % i]), T(g["m%d_seed_xyz" % i]))
        assert np.array_equal(out.numpy(), g["m%d_out" % i], equal_nan=True), i
    for i in range(int(g["n_dec"])):
        B = int(g["d%d_B" % i])
        geos = [T(g["d%d_geo%d" % (i, b)]) for b in range(B)]
        out = obias.decoder_relative_pos(geos, T(g["d%d_inds" % i]), T(g["d%d_qry" % i]), T(g["d%d_ctx" % i]))
        assert np.array_equal(out.numpy(), g["d%d_out" % i], equal_nan=True), i


def test_attention_oracle_matches_reference_layer_fixture():
    """oracle/attention.py against tests/golden/attention_golden.npz = what the reference's OWN
    TransformerDecoderLayer.forward_pre_rel computes in its cross-attention block (transformer_detr.py:443-454),
    captured by forward hooks (tests/golden/make_golden_attention.py).  Same fp32 torch ops: 1e-6."""
    import torch

    from oracle import attention as oatt

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "attention_golden.npz"))
    T = lambda a: torch.from_numpy(np.array(a))  # noqa: E731
    for i in range(int(g["n"])):
        w = {k: T(g["c%d_%s" % (i, k)]) for k in ("w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo")}
        out = oatt.rel_cross_attention(T(g["c%d_tgt2" % i]), T(g["c%d_memory" % i]), T(g["c%d_rel" % i]), w)
        np.testing.assert_allclose(out.numpy(), g["c%d_out" % i], rtol=1e-5, atol=1e-6)


def _aggregate_case(g, i):
    import torch

    T = lambda a: torch.from_numpy(np.array(a))  # noqa: E731
    layers = []
    l = 0
    while "c%d_w%d" % (i, l) in g.files:
        layers.append({"w": T(g["c%d_w%d" % (i, l)]), "gamma": T(g["c%d_gamma%d" % (i, l)]), "beta": T(g["c%d_beta%d" % (i, l)]),
                       "mean": T(g["c%d_mean%d" % (i, l)]), "var": T(g["c%d_var%d" % (i, l)])})
        l += 1
    radius, ns, norm = g["c%d_meta" % i]
    xyz, feats, inds = T(g["c%d_xyz" % i]), T(g["c%d_feats" % i]), T(g["c%d_inds" % i])
    new_xyz = torch.stack([xyz[b][inds[b].long()] for b in range(xyz.shape[0])])
    return xyz, new_xyz, feats, T(g["c%d_idx" % i]), float(radius), bool(norm), layers


def test_aggregate_oracle_matches_reference_module_fixture():
    """oracle/aggregate.py against tests/golden/aggregate_golden.npz = what the reference's OWN
    PointnetSAModuleVotesSeparate.mlp returns on CPU (tests/golden/make_golden_aggregate.py)"""
    from oracle import aggregate as oagg

    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "aggregate_golden.npz"))
    for i in range(int(g["n"])):
        xyz, new_xyz, feats, idx, radius, norm, layers = _aggregate_case(g, i)
        for pooling in ("max", "avg"):
            out = oagg.group_mlp_pool(xyz, new_xyz, feats, idx, radius, norm, True, layers, pooling=pooling)
            np.testing.assert_allclose(out.numpy(), g["c%d_%s" % (i, pooling)], rtol=1e-5, atol=1e-6)
