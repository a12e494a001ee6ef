"""Every furthest-point-sampling kernel the library can launch, reached through the rule that chooses it from N, the
largest co-schedulable cluster and the SM count (plan_fps, gf_fps.cu), bit for bit against the oracle, with a check of
which kernel ran:

    fps_cluster_kernel<256, P>   one cluster of 1..16 CTAs per scene, P points per thread in registers,
                                 P in 1, 2, 4, 8, 12, 16, 20, 25, 32 (N up to 16 x 256 x 32 = 131072 on a B200)
    fps_cluster_kernel<512, 24>  the largest cluster with 512-thread CTAs (N up to 196608 on a B200)
    fps_grid_kernel<P>           one CTA per SM (cooperative launch), P in 8, 16, 24, 32 points per thread
    fps_grid_kernel<0>           the same, streaming the points and their running minimum from L2

The case families, each at the instances where it can go wrong:
  * both ends of every interval of N with one launch shape, with the last point far out (padding at capacity);
  * points on a few lattice sites, more seeds than sites: ties inside and across CTAs at every multi-CTA instance;
  * all eligible points in one CTA, and a scene with no eligible point at all;
  * points on both sides of the |p|^2 <= 1e-3 skip rule, exactly at the float32 boundary;
  * batches of different scenes, m at its edges, and the batched hot path.
The CPU tests at the end prove on the oracle that the tie and skip-boundary inputs tell a wrong kernel apart."""
import re

import numpy as np
import pytest
import torch

from test_oracle_golden import _fps_by_key_rule

P256 = (1, 2, 4, 8, 12, 16, 20, 25, 32)  # kFpsP256
GRID_P = (8, 16, 24, 32)
GRID_T = 256  # FPS_GRID_T
MAX_GRID_CTAS = 160  # FPS_MAX_GRID_CTAS
B200 = (16, 148)  # (largest cluster, SMs) of a B200: the shape the CPU checks are made for

INSTANCES = [("cluster", 256, p) for p in P256] + [("cluster", 512, 24)] + [("grid", p) for p in GRID_P + (0,)]


def _id(inst):
    return "%s<%s>" % (inst[0], ",".join(str(v) for v in inst[1:]))


def _grid_ctas(sms):
    return min(sms & ~1, MAX_GRID_CTAS)


def _plan(N, max_cs, sms):
    """plan_fps (gf_fps.cu:453-469) restated -> (("cluster", T, P) or ("grid", P), CTAs per scene)"""
    if N < 512:
        return ("cluster", 256, 1 if N <= 256 else 2), 1
    cs = max_cs
    while cs > 2 and cs // 2 * 256 * 4 >= N:
        cs //= 2
    for p in P256:
        if cs * 256 * p >= N:
            return ("cluster", 256, p), cs
    if max_cs * 512 * 24 >= N:
        return ("cluster", 512, 24), max_cs
    ctas = _grid_ctas(sms)
    for p in GRID_P:
        if ctas * GRID_T * p >= N:
            return ("grid", p), ctas
    return ("grid", 0), ctas


def _tiers(max_cs, sms):
    """[(first N, last N, instance, CTAs)] for every interval of N with one launch shape; the streaming interval has
    no last N (None).  The cuts are every threshold _plan compares N with."""
    pow2 = [1 << i for i in range(1, 5) if 1 << i <= max_cs]
    cuts = {256, 511, max_cs * 512 * 24}
    cuts |= {c * 512 for c in pow2} | {c * 256 * p for c in pow2 for p in P256}
    cuts |= {_grid_ctas(sms) * GRID_T * p for p in GRID_P}
    tiers, lo = [], 1
    for hi in sorted(cuts) + [None]:
        shape = _plan(lo, max_cs, sms)
        if tiers and tuple(tiers[-1][2:]) == shape:
            tiers[-1][1] = hi
        else:
            tiers.append([lo, hi, *shape])
        if hi is not None:
            lo = hi + 1
    return [tuple(t) for t in tiers]


def _reachable(max_cs, sms):
    return {t[2] for t in _tiers(max_cs, sms)}


def _largest(inst, max_cs, sms, min_ctas=1):
    """the largest N the instance takes with at least min_ctas CTAs (the streaming kernel: its first N + 37 000)"""
    ts = [t for t in _tiers(max_cs, sms) if t[2] == inst and t[3] >= min_ctas]
    if not ts:
        return None
    lo, hi = ts[-1][:2]
    return hi if hi is not None else lo + 37_000


def _cta_of(k, N, inst, ctas):
    """CTA that holds point k in the register-resident kernels: thread u = g*bs + c owns k = c + bs*(g*P + i)"""
    L = 0
    while (2 << L) <= N and L < 9:
        L += 1
    bs = 1 << L
    T, P = (inst[1], inst[2]) if inst[0] == "cluster" else (GRID_T, inst[1])
    assert P > 0
    return ((k // bs) // P * bs + k % bs) // T


# ------------------------------------------------------------------------------------------ inputs
def _boundary_scene(N, seed):
    """scene() with its last point far out: the first seed after 0 is N - 1, the last slot of the padded layout"""
    from geoformer_b200.scenes import scene

    x = scene(N, seed).numpy()
    if N > 1:
        x[N - 1] = (40.0, -30.0, 20.0)
    return x


def _lattice(N, seed):
    """27 lattice sites (multiples of 0.25), the origin ineligible and point 0 on it: ties at every distance,
    and all-zero ties once every site has a seed"""
    x = np.random.default_rng(seed).integers(-1, 2, size=(N, 3)).astype(np.float32) * np.float32(0.25)
    x[0] = 0.0
    return x


TIE_M = 40  # > 27 sites


def _in_ball(n, g):
    """points with |p|^2 <= 3 * 0.015^2 < 1e-3: never eligible"""
    return g.uniform(-0.015, 0.015, size=(n, 3)).astype(np.float32)


def _one_cta_eligible(N, inst, ctas, seed):
    """every point inside the skip ball except six, all held by one CTA"""
    g = np.random.default_rng(seed)
    x = _in_ball(N, g)
    k = np.arange(1, N)
    mine = k[_cta_of(k, N, inst, ctas) == ctas // 2 + 1]
    pick = g.choice(mine, size=6, replace=False)
    x[pick] = g.uniform(0.5, 2.0, size=(6, 3)).astype(np.float32) * g.choice([-1, 1], size=(6, 3))
    return x, pick


def _sq3(x):
    """the oracle's fma(z,z, fma(x,x, y*y)) in float64 -> float32 steps (exact for these magnitudes)"""
    x = x.astype(np.float64)
    yy = (x[..., 1] * x[..., 1]).astype(np.float32).astype(np.float64)
    t = (x[..., 0] * x[..., 0] + yy).astype(np.float32).astype(np.float64)
    return (x[..., 2] * x[..., 2] + t).astype(np.float32)


def _skip_boundary_points():
    """(on, below): 16 points each whose sq3 is float32(1e-3) (above 1e-3 in double: eligible) and the float below it
    (ineligible); two points each, with all eight sign patterns"""
    lim = np.float32(1e-3)
    below = np.nextafter(lim, np.float32(0))
    a = np.float32(np.sqrt(1e-3 / 3))
    steps = np.arange(-96, 97, dtype=np.float32) * np.spacing(a)
    xs, ys = np.meshgrid(a + steps, a + steps, indexing="ij")
    pts = np.stack([xs.ravel(), ys.ravel(), np.full(xs.size, a, np.float32)], axis=1)
    s = _sq3(pts)
    signs = np.array([[sx, sy, sz] for sx in (1, -1) for sy in (1, -1) for sz in (1, -1)], dtype=np.float32)
    out = []
    for want in (lim, below):
        base = pts[s == want][[0, -1]]
        assert len(base) == 2 and not np.array_equal(base[0], base[1])
        out.append((base[:, None, :] * signs[None]).reshape(-1, 3))
    return out


def _skip_boundary_scene(N, seed):
    """a scene inside the skip ball with the boundary points spread over it -> xyz, indices of on, of below"""
    g = np.random.default_rng(seed)
    x = _in_ball(N, g)
    on, below = _skip_boundary_points()
    where = g.choice(np.arange(1, N), size=len(on) + len(below), replace=False)
    x[where[:len(on)]] = on
    x[where[len(on):]] = below
    return x, where[:len(on)], where[len(on):]


SKIP_M = 24  # > the 16 eligible points


# ------------------------------------------------------------------------------------------ GPU
_SEEN = set()  # instances whose launch a test below has asserted


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _launched(fn):
    """fn() under the profiler -> its result and the FPS kernel instances it launched, in launch order"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    found = []
    for e in prof.events():  # demangled "fps_grid_kernel<8>(...)" or mangled "fps_grid_kernelILi8EE..."
        m = re.search(r"fps_(cluster|grid)_kernel(?:<([-\d, ]+)>|I((?:Li-?\d+E)+)E)", e.name)
        if m:
            found.append((m.group(1),) + tuple(int(v) for v in re.findall(r"-?\d+", m.group(2) or m.group(3))))
    return out, found


def _fps(xyz, m, dev):
    from geoformer_b200.pointnet2 import _ext

    x = torch.from_numpy(np.ascontiguousarray(xyz, dtype=np.float32)).to(dev)
    out, kernels = _launched(lambda: _ext.furthest_point_sampling(x, m))
    return out.cpu().numpy(), kernels


@pytest.fixture(scope="module")
def shape(dev):
    """(largest cluster, SMs) of this device: N = 65537 runs <256,20> with clusters of 16, <512,24> with clusters of 8"""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    _, kernels = _fps(np.random.default_rng(0).normal(size=(1, 65537, 3)), 2, dev)
    max_cs = {("cluster", 256, 20): 16, ("cluster", 512, 24): 8}[kernels[0]]
    assert kernels == [_plan(65537, max_cs, sms)[0]]
    return max_cs, sms


def _check(oracle_lib, dev, shape, xyz, m):
    """the library's seeds of xyz (B, N, 3) == the oracle's, from the kernel the plan mirror predicts -> the seeds"""
    xyz = np.ascontiguousarray(xyz, dtype=np.float32)
    inst = _plan(xyz.shape[1], *shape)[0]
    got, kernels = _fps(xyz, m, dev)
    assert kernels == [inst], (xyz.shape, m)
    _SEEN.add(inst)
    want = oracle_lib.furthest_point_sampling(xyz, m)
    assert got.dtype == np.int32 and got.shape == want.shape
    bad = np.argwhere(got != want)
    assert bad.size == 0, "%d wrong seeds, first at (scene, round) %s: %d, oracle %d" % (
        len(bad), tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])])
    return want


def _need(inst, shape):
    if inst not in _reachable(*shape):
        pytest.skip("%s is not reachable on this device" % _id(inst))


@pytest.mark.gpu
@pytest.mark.parametrize("inst", INSTANCES, ids=_id)
def test_fps_tier_boundaries(oracle_lib, dev, shape, inst):
    """the first and last N of every interval this instance takes: padding exactly at capacity and one point over"""
    _need(inst, shape)
    for lo, hi, _, ctas in (t for t in _tiers(*shape) if t[2] == inst):
        for N in sorted({lo, hi or lo}):
            want = _check(oracle_lib, dev, shape, _boundary_scene(N, N)[None], 64)
            assert N == 1 or want[0, 1] == N - 1, "the far point is the first seed after 0"


@pytest.mark.gpu
@pytest.mark.parametrize("inst", INSTANCES, ids=_id)
def test_fps_ties_across_ctas(oracle_lib, dev, shape, inst):
    N = _largest(inst, *shape, min_ctas=2)
    if N is None:
        pytest.skip("%s never runs with more than one CTA on this device" % _id(inst))
    _check(oracle_lib, dev, shape, _lattice(N, N)[None], TIE_M)


NOBODY = [("cluster", 256, 16), ("cluster", 512, 24), ("grid", 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("inst", NOBODY, ids=_id)
def test_fps_ctas_without_eligible_points(oracle_lib, dev, shape, inst):
    """all CTAs but one publish the empty key in every round; then a scene where every CTA does"""
    _need(inst, shape)
    N = _largest(inst, *shape, min_ctas=2)
    ctas = _plan(N, *shape)[1]
    assert inst[0] == "grid" or ctas == shape[0]
    x, pick = _one_cta_eligible(N, inst, ctas, N)
    want = _check(oracle_lib, dev, shape, x[None], 12)
    assert set(want[0, 1:7]) == set(pick.tolist())
    want = _check(oracle_lib, dev, shape, _in_ball(N, np.random.default_rng(1))[None], 8)
    assert (want == 0).all()


SKIP_AT = [("cluster", 256, 1), ("cluster", 256, 16), ("cluster", 512, 24), ("grid", 8)]


@pytest.mark.gpu
@pytest.mark.parametrize("inst", SKIP_AT, ids=_id)
def test_fps_skip_rule_boundary(oracle_lib, dev, shape, inst):
    _need(inst, shape)
    N = _largest(inst, *shape)
    x, on, below = _skip_boundary_scene(N, N)
    want = _check(oracle_lib, dev, shape, x[None], SKIP_M)
    assert set(want[0].tolist()) == {0} | set(on.tolist())


BATCHED = [("cluster", 256, 16), ("cluster", 256, 32), ("cluster", 512, 24), ("grid", 24), ("grid", 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("inst", BATCHED, ids=_id)
def test_fps_batch_of_different_scenes(oracle_lib, dev, shape, inst):
    """each scene of a launch has its own seeds: a kernel that reused one scene's points, running minima or
    exchange slots for the next would give one scene's answer twice"""
    from geoformer_b200.scenes import scene

    _need(inst, shape)
    if inst == ("grid", 0):
        B, N, m = 2, 1_250_000, 24  # each scene has its own running-minimum area
        assert _plan(N, *shape)[0] == inst
    else:
        B, N, m = 3 if inst[0] == "cluster" else 2, _largest(inst, *shape), 64
    xyz = np.stack([scene(N, 700 + b).numpy() for b in range(B)])
    want = _check(oracle_lib, dev, shape, xyz, m)
    assert all(not np.array_equal(want[a], want[b]) for a in range(B) for b in range(a))


@pytest.mark.gpu
@pytest.mark.parametrize("inst", [("cluster", 256, 16), ("grid", 8)], ids=_id)
@pytest.mark.parametrize("m", [1, 2])
def test_fps_one_and_two_seeds(oracle_lib, dev, shape, inst, m):
    from geoformer_b200.scenes import scene

    _need(inst, shape)
    N = _largest(inst, *shape)
    xyz = np.stack([scene(N, 800 + b).numpy() for b in range(2)])
    _check(oracle_lib, dev, shape, xyz, m)


@pytest.mark.gpu
@pytest.mark.parametrize("N", [257, 512])
def test_fps_more_seeds_than_points(oracle_lib, dev, shape, N):
    """N = 512 is <256,1> on two CTAs"""
    from geoformer_b200.scenes import scene

    _check(oracle_lib, dev, shape, scene(N, 5)[None].numpy(), N + 40)


@pytest.mark.gpu
def test_fps_seeds_of_the_batched_hot_path(oracle_lib, dev, shape):
    """geodesic_guidance_batch samples every scene's seeds on its own lane; the cluster tiers only (whether two
    cooperative grids on concurrent lanes can be co-resident is another question)"""
    from geoformer_b200.guidance import geodesic_guidance_batch
    from geoformer_b200.scenes import scene

    Ns = [n for n in (777, 50_000, 120_000, 150_000) if _plan(n, *shape)[0][0] == "cluster"]
    xs = [scene(n, 900 + i) for i, n in enumerate(Ns)]
    Q = 64
    (seeds, _), kernels = _launched(lambda: geodesic_guidance_batch([x.to(dev) for x in xs], Q, 8, 0.5, 8))
    assert sorted(kernels) == sorted(_plan(n, *shape)[0] for n in Ns)
    _SEEN.update(kernels)
    for x, s in zip(xs, seeds):
        assert np.array_equal(s.cpu().numpy(), oracle_lib.furthest_point_sampling(x[None].numpy(), Q)[0])


@pytest.mark.gpu
def test_fps_every_reachable_instance_ran(shape):
    """runs after the tests above (file order): together they launched every instance the plan can choose here"""
    assert _SEEN == _reachable(*shape), sorted(_reachable(*shape) ^ _SEEN)


# ------------------------------------------------------------------------------------------ CPU
def test_plan_mirror_covers_every_instance_on_b200():
    tiers = _tiers(*B200)
    assert {t[2] for t in tiers} == set(INSTANCES)
    assert [t[0] for t in tiers[1:]] == [t[1] + 1 for t in tiers[:-1]]
    for lo, hi, inst, ctas in tiers:
        for N in (lo, hi or lo + 10_000):
            assert _plan(N, *B200) == (inst, ctas)
    assert _plan(50_000, *B200)[0] == ("cluster", 256, 16) and _plan(1_000_000, *B200)[0] == ("grid", 32)


@pytest.mark.parametrize("inst", INSTANCES, ids=_id)
def test_tied_inputs_tell_the_lowest_index_rule_apart(oracle_lib, inst):
    """the reference's tie order and the lowest index give different seeds on the tie test's input"""
    N = _largest(inst, *B200, min_ctas=2)
    x = _lattice(N, N)
    want = oracle_lib.furthest_point_sampling(x[None], TIE_M)[0]
    assert np.array_equal(_fps_by_key_rule(x, TIE_M), want)
    lowest = _fps_by_key_rule(x, TIE_M, rank=np.arange(N))
    assert not np.array_equal(lowest, want)


def test_skip_boundary_points_sit_on_the_float32_boundary():
    on, below = _skip_boundary_points()
    assert (_sq3(on) == np.float32(1e-3)).all() and float(np.float32(1e-3)) > 1e-3
    assert (_sq3(below) == np.nextafter(np.float32(1e-3), np.float32(0))).all()
    assert len({tuple(p) for p in on}) == len(on) == 16 and len({tuple(p) for p in below}) == 16


@pytest.mark.parametrize("inst", SKIP_AT, ids=_id)
def test_skip_boundary_inputs_tell_a_float32_compare_apart(oracle_lib, inst):
    """the oracle selects exactly the points on the boundary; compared in float32 they would be skipped, as if they
    sat at the origin, and the seeds differ"""
    N = _largest(inst, *B200)
    x, on, below = _skip_boundary_scene(N, N)
    want = oracle_lib.furthest_point_sampling(x[None], SKIP_M)[0]
    assert set(want.tolist()) == {0} | set(on.tolist())
    y = x.copy()
    y[on] = 0.0
    assert not np.array_equal(oracle_lib.furthest_point_sampling(y[None], SKIP_M)[0], want)
