"""The culled FPS on the kNN grid (fps_cells_kernel, gf_fps.cu) that samples the seeds of a batched guidance call with
more scenes than FPS lanes: bit for bit the seeds of the single-scene FPS and of the oracle, on c2-size scenes, ragged
batches, more seeds than points, ties, points on both sides of the |p|^2 <= 1e-3 rule and a scene without an eligible
point, at B = 5 and B = 32.  The CPU test checks the rule a skipped block rests on: the lower bound of sq3(p - c) over
a box never exceeds the computed sq3(p - c) of a point inside it."""
import re

import numpy as np
import pytest
import torch

from geoformer_b200.scenes import scene

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev(cuda_lib):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _single_scene_fps(x, Q, dev):
    from geoformer_b200.pointnet2._ext import furthest_point_sampling

    return furthest_point_sampling(torch.from_numpy(x)[None].to(dev), Q)[0].cpu().numpy()


def _check_batch(oracle_lib, dev, xs, Q):
    """one batched call over the scenes xs (list of (N, 3) float32 arrays): the culled FPS ran once per scene, and
    every scene's seeds are the single-scene FPS's and the oracle's"""
    from geoformer_b200.guidance import geodesic_guidance_batch

    assert len(xs) > 4
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        seeds, _ = geodesic_guidance_batch([torch.from_numpy(x).to(dev) for x in xs], Q, 8, 0.5, 4)
        torch.cuda.synchronize()
    names = [m.group(1) for e in prof.events() for m in [re.search(r"(fps_\w+?_kernel)", e.name)] if m]
    assert names == ["fps_cells_kernel"] * len(xs), names
    for b, (x, s) in enumerate(zip(xs, seeds)):
        got = s.cpu().numpy()
        want = oracle_lib.furthest_point_sampling(x[None], Q)[0]
        assert np.array_equal(got, want), (b, len(x), np.nonzero(got != want)[0][:8])
        assert np.array_equal(got, _single_scene_fps(x, Q, dev)), (b, len(x))


def _lattice(N, seed, sites=4):
    """points on sites^3 lattice sites, so most of them are duplicates: ties at every distance"""
    g = np.random.default_rng(seed)
    return (g.integers(0, sites, size=(N, 3)) - (sites - 1) / 2).astype(np.float32) * np.float32(0.5)


def _near_origin(N, seed, share):
    """a c2-like scene with a share of its points moved inside |p|^2 <= 1e-3 (never eligible), some of them on the
    float32 boundary of the rule, and point 0 at the origin"""
    g = np.random.default_rng(seed)
    x = scene(N, seed).numpy()
    k = g.choice(N, size=int(share * N), replace=False)
    x[k] = g.uniform(-0.018, 0.018, size=(len(k), 3)).astype(np.float32)
    on = np.float32(np.sqrt(np.float32(1e-3)))
    x[k[:8], :] = 0.0
    x[k[:8], 0] = on  # |p|^2 in float32 = 1e-3 or one ulp off: both sides of the rule
    x[0] = 0.0
    return x


@gpu
def test_c2_scenes(oracle_lib, dev):
    _check_batch(oracle_lib, dev, [scene(100_000, 1234 + s).numpy() for s in range(5)], 256)


@gpu
def test_ragged_batch(oracle_lib, dev):
    Ns = [1, 2, 300, 511, 777, 20_000, 200_000]
    _check_batch(oracle_lib, dev, [scene(n, 500 + i).numpy() for i, n in enumerate(Ns)], 96)


@gpu
def test_more_seeds_than_points(oracle_lib, dev):
    Ns = [1, 2, 300, 511, 600]
    _check_batch(oracle_lib, dev, [scene(n, 600 + i).numpy() for i, n in enumerate(Ns)], 640)


@gpu
def test_duplicates_and_lattice(oracle_lib, dev):
    xs = [_lattice(n, 700 + i, sites) for i, (n, sites) in enumerate([(5000, 4), (20_000, 5), (777, 3), (64, 2),
                                                                     (30_000, 6)])]
    xs.append(np.repeat(scene(3000, 77).numpy(), 3, axis=0))  # every point three times
    _check_batch(oracle_lib, dev, xs, 160)


@gpu
def test_points_near_the_origin_and_no_eligible_point(oracle_lib, dev):
    g = np.random.default_rng(9)
    none = g.uniform(-0.018, 0.018, size=(5000, 3)).astype(np.float32)  # |p|^2 <= 1e-3 everywhere
    xs = [_near_origin(50_000, 10, 0.3), _near_origin(8000, 11, 0.9), none, _near_origin(777, 12, 0.5),
          _near_origin(20_000, 13, 0.01)]
    _check_batch(oracle_lib, dev, xs, 64)


@gpu
def test_thirty_two_scenes(oracle_lib, dev):
    g = np.random.default_rng(32)
    Ns = g.integers(500, 40_000, size=32)
    _check_batch(oracle_lib, dev, [scene(int(n), 800 + i).numpy() for i, n in enumerate(Ns)], 64)


# ------------------------------------------------------------------------------------------ CPU
SHRINK = np.float32(1.0 - 2.0 ** -20)  # FPS_CELLS_SHRINK


def _fma32(a, b, c):
    """float32 fma, correctly rounded: a * b is exact in float64, the sum is rounded to odd, then to float32"""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    fix = (err != 0) & ((s.view(np.int64) & 1) == 0)
    s = np.where(fix, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def _sq3(x, y, z):
    """gf::sq3: fma(z, z, fma(x, x, y * y))"""
    return _fma32(z, z, _fma32(x, x, (y * y).astype(np.float32)))


def test_fma32_mirror_is_correctly_rounded():
    from fractions import Fraction

    g = np.random.default_rng(1)
    a, c = g.standard_normal((2, 2000)).astype(np.float32)
    exact = np.array([np.float32(float(Fraction(float(x)) ** 2 + Fraction(float(z)))) for x, z in zip(a, c)],
                     np.float32)
    assert np.array_equal(_fma32(a, a, c), exact)


def test_box_lower_bound_never_exceeds_the_computed_distance():
    """fps_cells_kernel skips a block when the bound is not below its largest running minimum: exact only if the
    bound never exceeds sq3(px - cx, py - cy, pz - cz) as the kernel computes it, for every point of the box"""
    g = np.random.default_rng(2)
    for trial in range(200):
        scale = np.float32(10.0 ** g.uniform(-3, 2))
        lo = (g.standard_normal(3) * scale).astype(np.float32)
        hi = (lo + np.abs(g.standard_normal(3)) * scale * g.uniform(0, 1)).astype(np.float32)
        p = (lo + (hi - lo) * g.uniform(0, 1, size=(2000, 3))).astype(np.float32)
        p = np.clip(p, lo, hi)
        p[:6] = [lo, hi, [lo[0], hi[1], lo[2]], [hi[0], lo[1], hi[2]], [lo[0], lo[1], hi[2]], [hi[0], hi[1], lo[2]]]
        box_lo, box_hi = p.min(0), p.max(0)  # the tight box, as the kernel builds it
        cs = [(lo + (hi - lo) * g.uniform(-1, 2, size=3)).astype(np.float32) for _ in range(16)]
        cs += [box_lo, box_hi, p[7].copy(), np.nextafter(box_lo, np.float32(-np.inf))]  # touching the box
        for c in cs:
            gap = np.maximum(np.maximum(box_lo - c, c - box_hi), np.float32(0))
            lb = (_sq3(gap[0:1], gap[1:2], gap[2:3]) * SHRINK).astype(np.float32)[0]
            d = _sq3(p[:, 0] - c[0], p[:, 1] - c[1], p[:, 2] - c[2])
            assert lb <= d.min(), (trial, c, lb, d.min())
