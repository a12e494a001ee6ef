"""The generic kernels that cap their grid at a multiple of the SM count and walk the rest of their work in a grid-stride
loop, driven past one grid pass and onto their tile edges, against the oracle (oracle.c, oracle/bias.py,
oracle/aggregate_train.py) and, where the answer has a closed form, against that too:

    kernel                          launch rule (restated below)                       work unit of the loop
    ball_query_kernel               min(B ceil(m/4), 8 SMs) CTAs                       4 centres (a CTA)
    three_nn_kernel                 min(B ceil(n/256), 8 SMs) CTAs                     256 unknown points (a CTA)
    gather / group / three_interpolate and their gradients
                                    grid_for: min(ceil(total/256), 32 SMs) CTAs        one element (a thread)
    bias_ctx_rowmax_kernel          (4 if C >= 1024 else 1, Q) CTAs                    --
    bias_ctx_write_kernel           min(ceil(QC/256), 8 SMs) CTAs                      one (query, context) (a thread)
    bias_mask_rowmax_kernel<VEC>    Q x chunks CTAs, chunks = ceil(8 SMs / Q) capped   --
    bias_mask_write_kernel<VEC>     (min(ceil(work/256), ceil(16 SMs / Q)), Q) CTAs    4 points (VEC) or 1 (a thread)
    group_mlp_pool_kernel<L>        min(ceil(Bm/8), 8 SMs) CTAs of 8 warps             one centre (a warp)
    knn_brute_kernel<KT>            ceil(nq/128) CTAs, KT = 8, 16, 32, 64 for k up to it

Each large case is sized from the rule and this device's SM count so that it takes at least two full passes and a
partial one, which is asserted before it runs; the kernel name and the grid are then read from the profiler's trace
and compared with the rule.  The last GPU test asserts that together the cases reached every (kernel, regime) pair.

Scatter-add gradients (atomicAdd in an order that changes from run to run) are checked against the float64 sum of
their terms with a bound that scales with the number of contributors c of each entry: exactly 0 at c = 0, exactly the
term at c = 1, and |got - exact| <= (c - 1) 2^-24 sum|terms| otherwise (each add after the first into zero rounds
once, by at most 2^-24 of a partial sum).  The CPU tests at the end show that the oracle's serial sum meets the bound
and that a sum with one term dropped, doubled or sent to the neighbouring entry does not.  The bound is a worst case:
for an entry with thousands of contributors it is wider than a fixed relative tolerance, and wider than any one term.
So every large gradient case also asserts that its index pattern keeps contributor counts low enough that the bound
resolves single terms (bound_resolution below).  Float32 atomic adds flush subnormal inputs to zero, so the exact
rule at c = 1 holds for normal terms only; the check refuses inputs with subnormal terms."""
import json
import os
import re
import tempfile

import numpy as np
import pytest
import torch

U = 2.0 ** -24  # unit roundoff of float32


# ------------------------------------------------------------------------------------------ launch rules, restated
def _cdiv(a, b):
    return -(-a // b)


def ball_query_launch(B, m, sms):
    """gf_ball_query (gf_pointops.cu): -> (grid, work units = groups of 4 centres, units per pass)"""
    groups = B * _cdiv(m, 4)
    return min(groups, 8 * sms), groups, min(groups, 8 * sms)


def three_nn_launch(B, n, sms):
    """gf_three_nn: one CTA of 256 threads per 256 unknown points"""
    blocks = B * _cdiv(n, 256)
    return min(blocks, 8 * sms), blocks, min(blocks, 8 * sms)


def elementwise_launch(total, sms):
    """grid_for (gf_pointops.cu): gather, group, three_interpolate and their gradients, one thread per element"""
    grid = max(1, min(_cdiv(total, 256), 32 * sms))
    return grid, total, grid * 256


def ctx_rowmax_launch(Q, C):
    """bias_ctx_rowmax_kernel (gf_bias.cu): (chunks, Q); chunk k holds the contexts c with (c // 256) % chunks == k"""
    return (4 if C >= 1024 else 1), Q


def ctx_write_launch(Q, C, sms):
    grid = min(_cdiv(Q * C, 256), 8 * sms)
    return grid, Q * C, grid * 256


def mask_is_vec(N, aligned):
    return N % 4 == 0 and aligned


def mask_rowmax_launch(Q, N, vec, sms):
    """bias_mask_rowmax: -> (CTAs, chunks per row)"""
    work = N // 4 if vec else N
    chunks = max(1, _cdiv(8 * sms, Q))
    chunks = max(1, min(chunks, _cdiv(work, 1024)))
    return Q * chunks, chunks


def mask_write_launch(Q, N, vec, sms):
    """bias_mask_write_kernel: -> (gx, work units of a row, units per pass); the grid is (gx, Q)"""
    work = N // 4 if vec else N
    gx = min(_cdiv(work, 256), max(1, _cdiv(16 * sms, Q)))
    return gx, work, gx * 256


def aggregate_launch(B, m, sms):
    """gf_group_mlp_pool: 8 warps a CTA, one warp per centre"""
    blocks = min(_cdiv(B * m, 8), 8 * sms)
    return blocks, B * m, blocks * 8


def passes(launch):
    _, work, per_pass = launch
    return _cdiv(work, per_pass)


def assert_past_two_passes(launch):
    """two full passes and a partial one"""
    _, work, per_pass = launch
    assert work > 2 * per_pass and work % per_pass != 0, launch


def past_two_passes(per_pass, unit=1):
    """the smallest multiple of `unit` past 2.5 passes that leaves the last pass partial"""
    w = _cdiv(5 * per_pass // 2 + 1, unit) * unit
    while w % per_pass == 0:
        w += unit
    return w


# the (kernel, regime) pairs the cases below must reach together
REGIMES = {
    ("ball_query_kernel", "past two passes"),
    ("three_nn_kernel", "past two passes"),
    ("gather_points_kernel", "past two passes"),
    ("gather_points_grad_kernel", "past two passes"),
    ("group_points_kernel", "past two passes"),
    ("group_points_grad_kernel", "past two passes"),
    ("three_interpolate_kernel", "past two passes"),
    ("three_interpolate_grad_kernel", "past two passes"),
    ("bias_ctx_rowmax_kernel", "4 chunks"),
    ("bias_ctx_write_kernel", "past two passes"),
    ("bias_mask_rowmax_kernel<true>", "several chunks"),
    ("bias_mask_rowmax_kernel<false>", "several chunks"),
    ("bias_mask_write_kernel<true>", "past two passes"),
    ("bias_mask_write_kernel<false>", "past two passes"),
    ("group_mlp_pool_kernel<1>", "past two passes"),
    ("group_mlp_pool_kernel<3>", "past two passes"),
    ("group_mlp_pool_kernel<4>", "past two passes"),
    ("knn_brute_kernel<64>", "k in 33..64"),
}
_REACHED = set()

_KERNELS = sorted({k.split("<")[0] for k, _ in REGIMES} | {"bias_init_kernel", "bias_zero_kernel",
                                                           "bias_rowmax_import_kernel"}, key=len, reverse=True)


def _kernel_id(name):
    """trace name (demangled or not) -> "base<args>" for the kernels above, else None"""
    for base in _KERNELS:
        m = re.search(r"(?<![A-Za-z_])" + base + r"(?:<([^<>]*)>|I((?:L[a-z]-?\d+E)+)E)?", name)
        if m:
            if m.group(1) is not None:
                return "%s<%s>" % (base, m.group(1).replace(" ", ""))
            if m.group(2) is not None:
                args = [{"b1": "true", "b0": "false"}.get(a, a[1:]) for a in re.findall(r"L([a-z]-?\d+)E", m.group(2))]
                return "%s<%s>" % (base, ",".join(args))
            return base
    return None


def _launched(fn):
    """fn() under the profiler -> its result and [(kernel id, grid)] of the kernels above it launched, in order; the
    grid is read from the exported trace"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    found = []
    for e in sorted((e for e in events if str(e.get("cat", "")).lower() == "kernel"), key=lambda e: e["ts"]):
        k = _kernel_id(e["name"])
        if k is not None:
            found.append((k, tuple(int(v) for v in e["args"]["grid"])))
    return out, found


def _expect(kernels, want):
    assert kernels == want, (kernels, want)


# ------------------------------------------------------------------------------------------ scatter-add bound
def gather_grad_terms(grad_out, idx, n):
    """gather_points_grad: grad_points[b,c,idx[b,j]] += grad_out[b,c,j] -> (flat destinations, terms)"""
    grad_out, idx = np.asarray(grad_out, np.float32), np.asarray(idx, np.int64)
    B, C, m = grad_out.shape
    dest = (np.arange(B * C).reshape(B, C, 1) * n + idx[:, None, :]).ravel()
    return dest, grad_out.ravel()


def group_grad_terms(grad_out, idx, n):
    """group_points_grad: grad_points[b,c,idx[b,j,s]] += grad_out[b,c,j,s]"""
    grad_out, idx = np.asarray(grad_out, np.float32), np.asarray(idx, np.int64)
    B, C = grad_out.shape[:2]
    dest = (np.arange(B * C).reshape(B, C, 1, 1) * n + idx[:, None]).ravel()
    return dest, grad_out.ravel()


def interpolate_grad_terms(grad_out, idx, weight, m):
    """three_interpolate_grad: grad_points[b,c,idx[b,j,k]] += fl(grad_out[b,c,j] * weight[b,j,k]) (__fmul_rn)"""
    grad_out, idx = np.asarray(grad_out, np.float32), np.asarray(idx, np.int64)
    weight = np.asarray(weight, np.float32)
    B, C, n = grad_out.shape
    dest = (np.arange(B * C).reshape(B, C, 1, 1) * m + idx[:, None]).ravel()
    terms = grad_out[:, :, :, None] * weight[:, None]  # float32 x float32: one rounding, as __fmul_rn
    assert terms.dtype == np.float32
    return dest, terms.ravel()


def atomic_sum_violations(got, dest, terms):
    """flat indices of `got` that break the bound of the module docstring"""
    got = np.asarray(got, np.float32).ravel()
    size = got.size
    assert not ((terms != 0) & (np.abs(terms) < np.finfo(np.float32).tiny)).any(), "subnormal terms: atomics flush them"
    t = terms.astype(np.float64)
    exact = np.bincount(dest, weights=t, minlength=size)
    mag = np.bincount(dest, weights=np.abs(t), minlength=size)
    cnt = np.bincount(dest, minlength=size)
    assert len(exact) == size, "a destination outside the result"
    g = got.astype(np.float64)
    bad = (cnt == 0) & (g != 0.0)
    bad |= (cnt == 1) & (g != exact)  # one term: exact in float64, and stored exactly
    bad |= (cnt >= 2) & ~(np.abs(g - exact) <= (cnt - 1) * U * mag)
    return np.flatnonzero(bad)


def bound_resolution(dest, terms, size):
    """-> (fraction of the nonzero terms whose loss, doubling or misrouting the bound is sure to catch, median number of
    contributors of an entry that has any).  A term t of an entry with c >= 2 contributors is caught when
    |t| > 2 (c - 1) 2^-24 sum|terms|: the result may itself sit a full bound from the exact sum.  At c = 1 every nonzero
    term is caught (the exact rule)."""
    t = terms.astype(np.float64)
    cnt = np.bincount(dest, minlength=size)
    bound = np.maximum(cnt - 1, 0) * U * np.bincount(dest, weights=np.abs(t), minlength=size)
    nz = terms != 0
    return float(np.mean(np.abs(t[nz]) > 2 * bound[dest[nz]])), float(np.median(cnt[cnt > 0]))


def assert_bound_resolves_terms(dest, terms, size, at_least=0.98):
    frac, med = bound_resolution(dest, terms, size)
    assert frac >= at_least, "the bound resolves only %.4f of the single terms (median %g contributors)" % (frac, med)


def assert_atomic_sum(got, dest, terms):
    bad = atomic_sum_violations(got, dest, terms)
    if bad.size:
        got = np.asarray(got, np.float32).ravel()
        cnt = np.bincount(dest, minlength=got.size)
        exact = np.bincount(dest, weights=terms.astype(np.float64), minlength=got.size)
        i = bad[0]
        raise AssertionError("%d entries outside the atomic-sum bound; first: flat %d, %d contributors, got %r, "
                             "exact %r" % (bad.size, i, cnt[i], float(got[i]), float(exact[i])))


# ------------------------------------------------------------------------------------------ planted ball queries
R = 0.5  # r^2 = 0.25 exactly
# offsets of a hit from its centre: multiples of 1/32 up to 1/8 per axis, |offset| <= 0.22 < R; exact in float32 next to
# centres up to 2^16
OFFS = np.array([(a, b, c) for a in range(-4, 5) for b in range(-4, 5) for c in range(-4, 5)], np.float32) / 32
BELOW = np.float32(0.5) - np.float32(2.0 ** -25)  # nextafter(0.5, 0) pairs with 2^-13 to squared distance just below r^2
TINY = np.float32(2.0 ** -13)


def _sq3(d):
    """the kernels' fmaf(z,z, fmaf(x,x, y*y)) in float64 steps rounded to float32 (exact for these magnitudes)"""
    d = d.astype(np.float64)
    yy = (d[..., 1] * d[..., 1]).astype(np.float32).astype(np.float64)
    t = (d[..., 0] * d[..., 0] + yy).astype(np.float32).astype(np.float64)
    return (d[..., 2] * d[..., 2] + t).astype(np.float32)


def _centres(m):
    """centre j at (4j, 0, 0): no point within R of one centre is within R of another"""
    c = np.zeros((m, 3), np.float32)
    c[:, 0] = 4 * np.arange(m)
    return c


def _plant(N, m, hits, seed):
    """N points far from every centre (all coordinates in [-60, -50]) except those of hits[j] (disjoint index lists),
    which lie at exact offsets within 0.22 of centre j -> centres (m,3), xyz (N,3)"""
    g = np.random.default_rng(seed)
    xyz = g.uniform(-60, -50, size=(N, 3)).astype(np.float32)
    c = _centres(m)
    used = np.concatenate([np.asarray(h, np.int64) for h in hits.values()] + [np.zeros(0, np.int64)])
    assert len(np.unique(used)) == len(used) and (used < N).all(), "hit lists must be disjoint and inside the scene"
    for j, h in hits.items():
        h = np.asarray(h, np.int64)
        xyz[h] = c[j] + OFFS[g.integers(0, len(OFFS), len(h))]
    return c, xyz


def _rows(hits, m, ns):
    """the expected rows: the first ns hits in index order, then the first hit repeated; no hit: zeros"""
    out = np.zeros((m, ns), np.int32)
    for j, h in hits.items():
        h = np.sort(np.asarray(h, np.int64))
        if len(h):
            out[j] = h[0]
            out[j, :min(ns, len(h))] = h[:ns]
    return out


def _case_edges():
    """hits on the quarter (511/512) and tile (2047/2048) edges, only the last point, the first hit in quarter 3 of
    tile 2, none; m = 5 leaves a CTA with one live centre"""
    N = 3 * 2048 + 1
    hits = {0: [511, 512], 1: [2047, 2048], 2: [N - 1], 3: [2 * 2048 + 3 * 512 + 17, 6000], 4: []}
    return N, 5, 4, [hits]


NS_CUTS = (1, 31, 32, 33, 64, 600)


def _case_cut(ns):
    """four centres of one CTA with ns - 1, ns, ns + 1 and 2 ns + 5 hits, interleaved with stride 4 from index 400: the
    four share the quarters their hits reach (one quarter at ns = 1, up to the third tile at ns = 600), and each full
    row is cut inside a quarter"""
    N = 3 * 2048 + 1
    counts = (ns - 1, ns, ns + 1, 2 * ns + 5)
    hits = {a: [400 + 4 * i + a for i in range(c)] for a, c in enumerate(counts)}
    return N, 4, ns, [hits]


BQ_SIZES = (1, 31, 33, 511, 512, 513, 2047, 2048, 2049, 6145)


def _case_size(N):
    rest = [i for i in range(N - 1)]
    hits = {0: [N - 1], 1: rest[0::3], 2: rest[1::3], 3: [], 4: rest[2::3][:5]}
    return N, 5, 32, [hits]


def _case_mixed():
    """CTA 0: a centre that fills in tile 0 (more hits later that must not appear), one whose last hit is the single
    point of the last tile, one that never fills, one without hits.  CTA 1: all four fill in tile 0 (the CTA-wide early
    exit) with more hits in tile 1"""
    N = 3 * 2048 + 1
    hits = {0: [4 * k for k in range(16)] + [2048 + 4 * k for k in range(10)] + [4096 + 4 * k for k in range(10)],
            1: [4 * k + 1 for k in range(15)] + [N - 1],
            2: [2048 + 4 * k + 2 for k in range(5)],
            3: []}
    for a in range(4):
        hits[4 + a] = [1000 + 4 * k + a for k in range(20)] + [3000 + 4 * k + a for k in range(5)]
    return N, 8, 16, [hits]


def _case_batch():
    """three scenes with different hit layouts; m = 7"""
    N, m, ns = 5000, 7, 8
    layouts = []
    for b in range(3):
        g = np.random.default_rng(50 + b)
        perm = g.permutation(N)
        counts = g.integers(0, 13, size=m)
        counts[b] = 0  # a different centre without hits in every scene
        starts = np.concatenate([[0], np.cumsum(counts)])
        layouts.append({j: perm[starts[j]:starts[j + 1]] for j in range(m)})
    return N, m, ns, layouts


def _case_grid(B, sms):
    """B scenes, m centres each, past two passes of the grid; every point belongs to a random centre or to nobody"""
    grid = 8 * sms
    groups = past_two_passes(grid, B)
    m = 4 * (groups // B) - 1  # not a multiple of 4: the last group of every scene has a dead slot
    N = 40000 if B == 1 else 15000
    layouts = []
    for b in range(B):
        owner = np.random.default_rng(60 + b).integers(-(m // 2), m, size=N)
        layouts.append({j: np.flatnonzero(owner == j) for j in np.unique(owner[owner >= 0])})
    return N, m, 4, layouts


def _radius_scene():
    """centre 0 at the origin with six points at squared distance exactly r^2 (outside) and four at the float below it
    (inside); centre 1 with two ordinary hits"""
    N, m, ns = 3000, 2, 8
    on_at, below_at = [10, 700, 1500, 2047, 2048, 2999], [5, 1023, 1024, 2500]
    c, xyz = _plant(N, m, {1: [3, 4]}, 7)
    on = np.array([(R, 0, 0), (-R, 0, 0), (0, R, 0), (0, -R, 0), (0, 0, R), (0, 0, -R)], np.float32)
    below = np.array([(BELOW, TINY, 0), (-BELOW, -TINY, 0), (0, BELOW, TINY), (0, -BELOW, -TINY)], np.float32)
    xyz[on_at], xyz[below_at] = on, below
    return c, xyz, ns, {0: below_at, 1: [3, 4]}, on, below


def _bq_inputs(N, m, ns, layouts):
    cs, xs, rows = [], [], []
    for b, hits in enumerate(layouts):
        c, x = _plant(N, m, hits, 100 + b)
        cs.append(c), xs.append(x), rows.append(_rows(hits, m, ns))
    return np.stack(cs), np.stack(xs), np.stack(rows)


BQ_CASES = {"edges": _case_edges, "mixed": _case_mixed, "batch": _case_batch}
BQ_CASES.update({"cut%d" % ns: (lambda ns=ns: _case_cut(ns)) for ns in NS_CUTS})
BQ_CASES.update({"size%d" % n: (lambda n=n: _case_size(n)) for n in BQ_SIZES})


# ------------------------------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def sms(dev):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ------------------------------------------------------------------------------------------ ball query
def _ball_query(oracle_lib, dev, centres, xyz, ns, want):
    from geoformer_b200.pointnet2 import _ext

    out, kernels = _launched(lambda: _ext.ball_query(_t(centres, dev), _t(xyz, dev), R, ns))
    out = out.cpu().numpy()
    ref = oracle_lib.ball_query(centres, xyz, R, ns)
    assert np.array_equal(ref, want), "the planted rows disagree with the oracle"
    bad = np.argwhere((out != want).any(axis=2))
    assert bad.size == 0, "%d wrong rows, first (scene, centre) %s: %s, want %s" % (
        len(bad), tuple(bad[0]), out[tuple(bad[0])][:12], want[tuple(bad[0])][:12])
    return kernels


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(BQ_CASES))
def test_ball_query_planted_rows(oracle_lib, dev, sms, case):
    N, m, ns, layouts = BQ_CASES[case]()
    centres, xyz, want = _bq_inputs(N, m, ns, layouts)
    kernels = _ball_query(oracle_lib, dev, centres, xyz, ns, want)
    _expect(kernels, [("ball_query_kernel", (ball_query_launch(len(layouts), m, sms)[0], 1, 1))])


@pytest.mark.gpu
def test_ball_query_radius_boundary(oracle_lib, dev):
    c, xyz, ns, hits, _, _ = _radius_scene()
    _ball_query(oracle_lib, dev, c[None], xyz[None], ns, _rows(hits, 2, ns)[None])


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 3])
def test_ball_query_grid_stride(oracle_lib, dev, sms, B):
    N, m, ns, layouts = _case_grid(B, sms)
    launch = ball_query_launch(B, m, sms)
    assert_past_two_passes(launch)
    centres, xyz, want = _bq_inputs(N, m, ns, layouts)
    assert (want[:, :, 0] == 0).any() and (want[:, :, -1] != want[:, :, 0]).any()  # rows without hits and full rows
    kernels = _ball_query(oracle_lib, dev, centres, xyz, ns, want)
    _expect(kernels, [("ball_query_kernel", (launch[0], 1, 1))])
    _REACHED.add(("ball_query_kernel", "past two passes"))


# ------------------------------------------------------------------------------------------ three_nn / interpolate
def _three_nn(oracle_lib, dev, unknown, known):
    from geoformer_b200.pointnet2 import _ext

    (d2, idx), kernels = _launched(lambda: _ext.three_nn(_t(unknown, dev), _t(known, dev)))
    rd2, ridx = oracle_lib.three_nn(unknown, known)
    d2, idx = d2.cpu().numpy(), idx.cpu().numpy()
    bad = np.argwhere((idx != ridx).any(axis=2) | (d2.view(np.int32) != rd2.view(np.int32)).any(axis=2))
    assert bad.size == 0, "%d wrong rows, first %s: %s %s, oracle %s %s" % (
        len(bad), tuple(bad[0]), idx[tuple(bad[0])], d2[tuple(bad[0])], ridx[tuple(bad[0])], rd2[tuple(bad[0])])
    return idx, d2, kernels


@pytest.mark.gpu
@pytest.mark.parametrize("m", [0, 1, 2, 3, 4, 1023, 1024, 1025, 3000])
def test_three_nn_known_set_sizes(oracle_lib, dev, sms, m):
    g = np.random.default_rng(m)
    unknown = g.uniform(-1, 1, size=(1, 700, 3)).astype(np.float32)
    known = g.uniform(-1, 1, size=(1, m, 3)).astype(np.float32)
    idx, d2, kernels = _three_nn(oracle_lib, dev, unknown, known)
    _expect(kernels, [("three_nn_kernel", (three_nn_launch(1, 700, sms)[0], 1, 1))])
    if m < 3:
        assert (idx[..., m:] == 0).all() and np.isinf(d2[..., m:]).all()


def _tie_scene():
    """3000 known points: exact duplicates whose copy lies in a later tile; around (5,5,5) two nearer points and a tie of
    the 3rd and 4th candidates at indices 1023 / 1024 (and 1025); around (-5,-5,-5) six points at squared distance
    exactly 0.25, spread over the tiles"""
    g = np.random.default_rng(8)
    known = g.uniform(-1, 1, size=(3000, 3)).astype(np.float32)
    known[1100:1140] = known[0:40]
    known[2100:2140] = known[600:640]
    p = np.float32(5)
    known[[1021, 1022, 1023, 1024, 1025]] = p + np.array(
        [(0.125, 0, 0), (0, 0.125, 0), (0.25, 0, 0), (0, 0.25, 0), (0, 0, 0.25)], np.float32)
    axis_at = [45, 1000, 1030, 2047, 2048, 2999]
    known[axis_at] = -p + np.array([(0.5, 0, 0), (-0.5, 0, 0), (0, 0.5, 0), (0, -0.5, 0), (0, 0, 0.5), (0, 0, -0.5)],
                                   np.float32)
    near = lambda a: a + g.uniform(-1e-3, 1e-3, size=a.shape).astype(np.float32)  # noqa: E731
    unknown = np.concatenate([g.uniform(-1, 1, size=(300, 3)).astype(np.float32), near(known[0:40]),
                              near(known[600:640]), known[0:10], np.full((2, 3), p, np.float32),
                              np.full((2, 3), -p, np.float32)])
    return unknown, known, axis_at


@pytest.mark.gpu
def test_three_nn_ties(oracle_lib, dev):
    unknown, known, axis_at = _tie_scene()
    idx, d2, _ = _three_nn(oracle_lib, dev, unknown[None], known[None])
    assert (idx[0, -4:-2] == [1021, 1022, 1023]).all() and (d2[0, -4:-2] == [1 / 64, 1 / 64, 1 / 16]).all()
    assert (idx[0, -2:] == axis_at[:3]).all() and (d2[0, -2:] == 0.25).all()


@pytest.mark.gpu
def test_three_nn_batch_of_different_known_sets(oracle_lib, dev, sms):
    g = np.random.default_rng(9)
    unknown = g.uniform(-1, 1, size=(3, 900, 3)).astype(np.float32)
    known = g.uniform(-1, 1, size=(3, 1500, 3)).astype(np.float32)
    idx, _, kernels = _three_nn(oracle_lib, dev, unknown, known)
    _expect(kernels, [("three_nn_kernel", (three_nn_launch(3, 900, sms)[0], 1, 1))])
    assert not np.array_equal(idx[0], idx[1])


@pytest.mark.gpu
def test_three_nn_and_interpolate_grid_stride(oracle_lib, dev, sms):
    from geoformer_b200.pointnet2 import _ext

    n = 256 * past_two_passes(8 * sms) - 100
    launch = three_nn_launch(1, n, sms)
    assert_past_two_passes(launch)
    g = np.random.default_rng(10)
    unknown = g.uniform(-1, 1, size=(1, n, 3)).astype(np.float32)
    known = g.uniform(-1, 1, size=(1, 64, 3)).astype(np.float32)
    idx, _, kernels = _three_nn(oracle_lib, dev, unknown, known)
    _expect(kernels, [("three_nn_kernel", (launch[0], 1, 1))])
    _REACHED.add(("three_nn_kernel", "past two passes"))

    # interpolation from as many known points as unknown ones, random indices: about 3 contributors per gradient entry
    # (three_nn's 64 known points would give each entry tens of thousands, and a bound wider than any single term)
    C = _cdiv(past_two_passes(32 * sms * 256), n)
    ilaunch = elementwise_launch(C * n, sms)
    assert_past_two_passes(ilaunch)
    m = n
    iidx = g.integers(0, m, size=(1, n, 3)).astype(np.int32)
    feats = g.standard_normal(size=(1, C, m)).astype(np.float32)
    w = g.uniform(0, 1, size=(1, n, 3)).astype(np.float32)
    out, kernels = _launched(lambda: _ext.three_interpolate(_t(feats, dev), _t(iidx, dev), _t(w, dev)))
    _expect(kernels, [("three_interpolate_kernel", (ilaunch[0], 1, 1))])
    assert np.array_equal(out.cpu().numpy(), oracle_lib.three_interpolate(feats, iidx, w))
    _REACHED.add(("three_interpolate_kernel", "past two passes"))

    go = g.standard_normal(size=(1, C, n)).astype(np.float32)
    dest, terms = interpolate_grad_terms(go, iidx, w, m)
    assert_bound_resolves_terms(dest, terms, C * m)
    gr, kernels = _launched(lambda: _ext.three_interpolate_grad(_t(go, dev), _t(iidx, dev), _t(w, dev), m))
    _expect(kernels, [("three_interpolate_grad_kernel", (ilaunch[0], 1, 1))])
    assert_atomic_sum(gr.cpu().numpy(), dest, terms)
    _REACHED.add(("three_interpolate_grad_kernel", "past two passes"))


# ------------------------------------------------------------------------------------------ gather / group
@pytest.mark.gpu
def test_gather_and_group_grid_stride(oracle_lib, dev, sms):
    """B = 2, odd C, a ragged N; the indices of a real ball query, whose padding gives some points many contributors"""
    from geoformer_b200.pointnet2 import _ext
    from geoformer_b200.scenes import scene

    B, N, C, ns = 2, 20011, 5, 32
    npoint = _cdiv(past_two_passes(32 * sms * 256, B * ns), B * ns)
    glaunch = elementwise_launch(B * npoint * ns, sms)
    assert_past_two_passes(glaunch)
    xyz = torch.stack([scene(N, 30 + b) for b in range(B)]).to(dev)
    pick = torch.randint(0, N, (B, npoint), generator=torch.Generator().manual_seed(3))
    centres = torch.stack([xyz[b, pick[b].to(dev)] for b in range(B)]).contiguous()
    idx = _ext.ball_query(centres, xyz, 0.2, ns)
    idx_np = idx.cpu().numpy()
    cnt = np.bincount(idx_np[0].ravel(), minlength=N)
    assert cnt.max() > 64 and (cnt == 0).any()
    g = np.random.default_rng(11)
    feats = g.standard_normal(size=(B, C, N)).astype(np.float32)

    out, kernels = _launched(lambda: _ext.group_points(_t(feats, dev), idx))
    _expect(kernels, [("group_points_kernel", (glaunch[0], 1, 1))])
    assert np.array_equal(out.cpu().numpy(), oracle_lib.group_points(feats, idx_np))
    _REACHED.add(("group_points_kernel", "past two passes"))
    go = g.standard_normal(size=(B, C, npoint, ns)).astype(np.float32)
    dest, terms = group_grad_terms(go, idx_np, N)
    assert_bound_resolves_terms(dest, terms, B * C * N)
    gr, kernels = _launched(lambda: _ext.group_points_grad(_t(go, dev), idx, N))
    _expect(kernels, [("group_points_grad_kernel", (glaunch[0], 1, 1))])
    assert_atomic_sum(gr.cpu().numpy(), dest, terms)
    _REACHED.add(("group_points_grad_kernel", "past two passes"))

    mg = _cdiv(past_two_passes(32 * sms * 256, B * C), B * C)
    alaunch = elementwise_launch(B * C * mg, sms)
    assert_past_two_passes(alaunch)
    gidx = idx.reshape(B, -1)[:, :mg].contiguous()
    gidx_np = gidx.cpu().numpy()
    out, kernels = _launched(lambda: _ext.gather_points(_t(feats, dev), gidx))
    _expect(kernels, [("gather_points_kernel", (alaunch[0], 1, 1))])
    assert np.array_equal(out.cpu().numpy(), oracle_lib.gather_points(feats, gidx_np))
    _REACHED.add(("gather_points_kernel", "past two passes"))
    go = g.standard_normal(size=(B, C, mg)).astype(np.float32)
    dest, terms = gather_grad_terms(go, gidx_np, N)
    assert_bound_resolves_terms(dest, terms, B * C * N)
    gr, kernels = _launched(lambda: _ext.gather_points_grad(_t(go, dev), gidx, N))
    _expect(kernels, [("gather_points_grad_kernel", (alaunch[0], 1, 1))])
    assert_atomic_sum(gr.cpu().numpy(), dest, terms)
    _REACHED.add(("gather_points_grad_kernel", "past two passes"))


# ------------------------------------------------------------------------------------------ distance epilogues
def _decoder(dev, geos, inds, qry, ctx):
    from oracle import bias as obias

    from geoformer_b200.bias import decoder_relative_pos

    out, kernels = _launched(lambda: decoder_relative_pos([g.to(dev) for g in geos], inds.to(dev), qry.to(dev),
                                                          ctx.to(dev)))
    ref = obias.decoder_relative_pos(geos, inds, qry, ctx)
    out = out.cpu()
    bad = (out.view(torch.int32) != ref.view(torch.int32)).nonzero()
    assert bad.numel() == 0, "%d wrong values, first at %s: %r, want %r" % (
        len(bad), tuple(bad[0].tolist()), float(out[tuple(bad[0])]), float(ref[tuple(bad[0])]))
    return kernels


def _decoder_inputs(Q, C, Ns, seed):
    g = torch.Generator().manual_seed(seed)
    geos, inds = [], []
    for n in Ns:
        geo = torch.rand(Q, n, generator=g) * 20
        geo[torch.rand(Q, n, generator=g) < 0.5] = -1.0
        geos.append(geo)
        inds.append(torch.randperm(n, generator=g)[:C].int() if n >= C else torch.randint(0, n, (C,), generator=g,
                                                                                           dtype=torch.int32))
    B = len(Ns)
    return geos, torch.stack(inds), torch.rand(B, Q, 3, generator=g) * 8, torch.rand(B, C, 3, generator=g) * 8


def _decoder_kernels(B, Q, C, sms):
    chunks, _ = ctx_rowmax_launch(Q, C)
    return ([("bias_zero_kernel", (_cdiv(B * Q + 1, 256), 1, 1))] + [("bias_ctx_rowmax_kernel", (chunks, Q, 1))] * B
            + [("bias_ctx_write_kernel", (ctx_write_launch(Q, C, sms)[0], 1, 1))] * B)


@pytest.mark.gpu
def test_decoder_two_scenes_past_two_passes(dev, sms):
    """C = 2048: four row-maximum chunks; a row without a reachable context (global maximum) and a row whose reachable
    contexts all lie in the last chunk"""
    C = 2048
    Q = max(256, _cdiv(past_two_passes(8 * sms * 256, C), C))
    launch = ctx_write_launch(Q, C, sms)
    assert_past_two_passes(launch)
    chunks, _ = ctx_rowmax_launch(Q, C)
    assert chunks == 4
    geos, inds, qry, ctx = _decoder_inputs(Q, C, (5000, 7001), 12)
    geos[0][3, inds[0].long()] = -1.0
    chunk = (torch.arange(C) // 256) % chunks
    last = inds[1][chunk == chunks - 1].long()
    geos[1][5, inds[1].long()] = -1.0
    geos[1][5, last] = torch.linspace(0.5, 3.0, len(last))
    kernels = _decoder(dev, geos, inds, qry, ctx)
    _expect(kernels, _decoder_kernels(2, Q, C, sms))
    _REACHED.add(("bias_ctx_rowmax_kernel", "4 chunks"))
    _REACHED.add(("bias_ctx_write_kernel", "past two passes"))


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [0, 1])
def test_decoder_one_pass_and_one_element_more(dev, sms, extra):
    """Q C = one write pass exactly (Q = 256, C = 8 SMs), and one element more (Q = 1)"""
    Q, C = (256, 8 * sms) if extra == 0 else (1, 8 * sms * 256 + 1)
    _, work, per_pass = ctx_write_launch(Q, C, sms)
    assert work == per_pass + extra
    geos, inds, qry, ctx = _decoder_inputs(Q, C, (C + 17,), 13)
    _expect(_decoder(dev, geos, inds, qry, ctx), _decoder_kernels(1, Q, C, sms))


def _mask(dev, geo, coords, seeds, row_max=None):
    from geoformer_b200.bias import mask_head_relative_coords

    rm = None if row_max is None else row_max.to(dev)
    return _launched(lambda: mask_head_relative_coords(geo, coords.to(dev), seeds.to(dev), row_max=rm))


def _mask_inputs(Q, N, seed):
    g = torch.Generator().manual_seed(seed)
    geo = torch.rand(Q, N, generator=g) * 10
    geo[torch.rand(Q, N, generator=g) < 0.4] = -1.0
    if Q > 2:
        geo[Q // 2] = -1.0  # a row with nothing reachable: the global maximum
    return geo, torch.rand(N, 3, generator=g) * 8 - 4, torch.rand(Q, 3, generator=g) * 8 - 4


def _mask_kernels(Q, N, vec, sms, with_row_max):
    tag = "<true>" if vec else "<false>"
    gx = mask_write_launch(Q, N, vec, sms)[0]
    first = ([("bias_rowmax_import_kernel", (1, 1, 1))] if with_row_max else
             [("bias_init_kernel", (1, 1, 1)), ("bias_mask_rowmax_kernel" + tag, (mask_rowmax_launch(Q, N, vec, sms)[0],
                                                                                 1, 1))])
    return first + [("bias_mask_write_kernel" + tag, (gx, Q, 1))]


def _assert_bits(out, ref):
    out, ref = out.cpu().numpy(), ref.numpy()
    bad = np.argwhere(out.view(np.int32) != ref.view(np.int32))
    assert bad.size == 0, "%d wrong values, first at %s: %r, want %r" % (
        len(bad), tuple(bad[0]), out[tuple(bad[0])], ref[tuple(bad[0])])


def _record_mask(Q, N, vec, sms, with_row_max):
    tag = "<true>" if vec else "<false>"
    if not with_row_max and mask_rowmax_launch(Q, N, vec, sms)[1] > 1:
        _REACHED.add(("bias_mask_rowmax_kernel" + tag, "several chunks"))
    launch = mask_write_launch(Q, N, vec, sms)
    if passes(launch) > 2 and launch[1] % launch[2]:
        _REACHED.add(("bias_mask_write_kernel" + tag, "past two passes"))


MASK_SHAPES = [(1, 100_000), (1, 100_003), (3, 16_388), (256, 100_000), (256, 100_001)]


@pytest.mark.gpu
@pytest.mark.parametrize("Q,N", MASK_SHAPES)
def test_mask_head_shapes(dev, sms, Q, N):
    from oracle import bias as obias

    geo, coords, seeds = _mask_inputs(Q, N, Q + N)
    ref = obias.mask_head_relative_coords(geo, coords, seeds)
    vec = mask_is_vec(N, True)
    if Q == 256:
        assert_past_two_passes(mask_write_launch(Q, N, vec, sms))
    geo_d = geo.to(dev)
    for row_max in (None, geo.max(dim=1).values):
        out, kernels = _mask(dev, geo_d, coords, seeds, row_max)
        _expect(kernels, _mask_kernels(Q, N, vec, sms, row_max is not None))
        _assert_bits(out, ref)
        _record_mask(Q, N, vec, sms, row_max is not None)


@pytest.mark.gpu
def test_mask_head_unaligned_maps_equal_aligned(dev, sms):
    """the (256, 100 000) maps copied to a base one float past a 16-byte boundary: the scalar kernels at N % 4 == 0,
    with the bits of the vector kernels"""
    Q, N = 256, 100_000
    geo, coords, seeds = _mask_inputs(Q, N, 14)
    aligned = geo.to(dev)
    buf = torch.empty(Q * N + 1, device=dev)
    unaligned = buf[1:].view(Q, N)
    unaligned.copy_(aligned)
    assert unaligned.data_ptr() % 16 != 0
    assert_past_two_passes(mask_write_launch(Q, N, False, sms))
    for row_max in (None, geo.max(dim=1).values):
        want, kernels = _mask(dev, aligned, coords, seeds, row_max)
        _expect(kernels, _mask_kernels(Q, N, True, sms, row_max is not None))
        got, kernels = _mask(dev, unaligned, coords, seeds, row_max)
        _expect(kernels, _mask_kernels(Q, N, False, sms, row_max is not None))
        assert torch.equal(got, want)
        _record_mask(Q, N, False, sms, row_max is not None)


@pytest.mark.gpu
def test_mask_head_every_row_unreachable(dev, sms):
    """nothing reachable anywhere: sqrt of the maximum -1 is NaN, and every output is NaN, as in the reference"""
    from oracle import bias as obias

    Q, N = 5, 4099
    geo, coords, seeds = _mask_inputs(Q, N, 15)
    geo[:] = -1.0
    ref = obias.mask_head_relative_coords(geo, coords, seeds)
    assert torch.isnan(ref).all()
    for row_max in (None, geo.max(dim=1).values):
        out, kernels = _mask(dev, geo.to(dev), coords, seeds, row_max)
        _expect(kernels, _mask_kernels(Q, N, False, sms, row_max is not None))
        assert torch.isnan(out).all()


# ------------------------------------------------------------------------------------------ inference aggregator
@pytest.mark.gpu
@pytest.mark.parametrize("work", ["one more than a pass", "past two passes"])
@pytest.mark.parametrize("L", [1, 3, 4])
def test_aggregator_grid_stride(oracle_lib, dev, sms, L, work):
    """against the float64 oracle; every scene of the batch equals a call on that scene alone, bit for bit (a warp's
    arithmetic does not depend on the grid)"""
    from test_aggregate_train import assert_fwd, layers_of, mlp, oracle64

    from geoformer_b200.aggregate import fold_shared_mlp, group_mlp_pool
    from geoformer_b200.pointnet2 import _ext
    from geoformer_b200.scenes import scene

    per_pass = 8 * 8 * sms
    if work == "one more than a pass":
        B, m = 1, per_pass + 1
    else:
        B = 3
        m = past_two_passes(per_pass, B) // B
    launch = aggregate_launch(B, m, sms)
    if work == "past two passes":
        assert_past_two_passes(launch)
    else:
        assert launch[1] == launch[2] + 1
    N, Cf, ns, radius = 20000, 16, 16, 0.2
    widths = {1: [19, 32], 3: [19, 32, 32, 32], 4: [19, 32, 24, 32, 17]}[L]
    xyz = torch.stack([scene(N, 40 + b) for b in range(B)]).to(dev)
    pick = torch.stack([torch.randperm(N, generator=torch.Generator().manual_seed(b))[:m] for b in range(B)])
    new_xyz = torch.stack([xyz[b, pick[b].to(dev)] for b in range(B)]).contiguous()
    feats = torch.randn(B, Cf, N, generator=torch.Generator().manual_seed(L)).to(dev)
    idx = _ext.ball_query(new_xyz, xyz, radius, ns)
    net = mlp(widths, torch.Generator().manual_seed(20 + L)).eval()
    w, Ws, scs, shs = fold_shared_mlp(net)
    assert w == widths
    run = lambda sl: group_mlp_pool(xyz[sl], new_xyz[sl], feats[sl], idx[sl], radius, True, True, w, Ws, scs,  # noqa
                                    shs)
    out, kernels = _launched(lambda: run(slice(None)))
    _expect(kernels, [("group_mlp_pool_kernel<%d>" % L, (launch[0], 1, 1))])
    (ref, _), _ = oracle64(xyz, new_xyz, feats, idx, radius, True, True, layers_of(net, torch.float64), False)
    assert out.shape == (B, widths[-1], m)
    assert_fwd(out, ref)
    for b in range(B):
        assert torch.equal(run(slice(b, b + 1))[0], out[b]), b
    if work == "past two passes":
        _REACHED.add(("group_mlp_pool_kernel<%d>" % L, "past two passes"))


# ------------------------------------------------------------------------------------------ brute-force kNN, KT = 64
@pytest.mark.gpu
@pytest.mark.parametrize("k", [33, 64])
def test_knn_brute_kt64_launch(dev, k):
    """the launch only: both ends of 33..64 select knn_brute_kernel<64>.  Its results are compared with the oracle in
    test_gpu_parity.py::test_knn_matches_oracle (k = 33, 64, and N < k)"""
    from geoformer_b200.geodesic_utils import knn_graph
    from geoformer_b200.scenes import scene

    x = scene(300, 23).to(dev)
    _, kernels = _launched(lambda: knn_graph(x, k, algo="brute"))
    _expect(kernels, [("knn_brute_kernel<64>", (_cdiv(300, 128), 1, 1))])
    _REACHED.add(("knn_brute_kernel<64>", "k in 33..64"))


def _runs_every_gpu_test_here(request):
    """whether this session runs every GPU test of this file in this process (not a -k subset, not a distributed
    worker's share): only then can their launches add up to the whole table"""
    if hasattr(request.config, "workerinput"):
        return False
    want = 0
    for name, fn in vars(request.module).items():
        marks = getattr(fn, "pytestmark", []) if name.startswith("test_") and callable(fn) else []
        if name == request.function.__name__ or not any(mk.name == "gpu" for mk in marks):
            continue
        n = 1
        for mk in marks:
            if mk.name == "parametrize":
                n *= len(mk.args[1])
        want += n
    ran = sum(1 for it in request.session.items
              if getattr(it, "module", None) is request.module and it.get_closest_marker("gpu") is not None
              and it.nodeid != request.node.nodeid)
    return ran == want


@pytest.mark.gpu
def test_every_kernel_regime_reached(request):
    """runs after the tests above (file order): together they reached every (kernel, regime) pair"""
    if not _runs_every_gpu_test_here(request):
        pytest.skip("needs every GPU test of this file in one session and process")
    assert _REACHED == REGIMES, sorted(REGIMES - _REACHED)


# ------------------------------------------------------------------------------------------ CPU
B200_SMS = 148


def test_launch_rules_on_b200():
    """the thresholds where a second pass starts on 148 SMs"""
    s = B200_SMS
    assert passes(ball_query_launch(1, 4 * 1184, s)) == 1 and passes(ball_query_launch(1, 4 * 1184 + 1, s)) == 2
    assert passes(three_nn_launch(1, 1184 * 256, s)) == 1 and passes(three_nn_launch(1, 1184 * 256 + 1, s)) == 2
    assert passes(elementwise_launch(1_212_416, s)) == 1 and passes(elementwise_launch(1_212_417, s)) == 2
    assert passes(ctx_write_launch(1, 303_104, s)) == 1 and passes(ctx_write_launch(1, 303_105, s)) == 2
    assert ctx_rowmax_launch(256, 1023)[0] == 1 and ctx_rowmax_launch(256, 1024)[0] == 4
    assert passes(aggregate_launch(1, 9472, s)) == 1 and passes(aggregate_launch(1, 9473, s)) == 2
    assert mask_write_launch(256, 100_000, True, s) == (10, 25_000, 2560)
    assert mask_rowmax_launch(256, 100_000, True, s) == (1280, 5)
    assert not mask_is_vec(100_001, True) and not mask_is_vec(100_000, False)


@pytest.mark.parametrize("sms", [100, 132, 148, 160])
def test_large_cases_take_two_passes_and_a_part(sms):
    """the sizes the GPU tests derive from the SM count land past two passes on any of these devices"""
    for B in (1, 3):
        N, m, _, layouts = _case_grid(B, sms)
        assert len(layouts) == B and m % 4
        assert_past_two_passes(ball_query_launch(B, m, sms))
    n = 256 * past_two_passes(8 * sms) - 100
    assert_past_two_passes(three_nn_launch(1, n, sms))
    assert_past_two_passes(elementwise_launch(_cdiv(past_two_passes(32 * sms * 256), n) * n, sms))
    B, ns, C = 2, 32, 5
    assert_past_two_passes(elementwise_launch(B * ns * _cdiv(past_two_passes(32 * sms * 256, B * ns), B * ns), sms))
    assert_past_two_passes(elementwise_launch(B * C * _cdiv(past_two_passes(32 * sms * 256, B * C), B * C), sms))
    Q = max(256, _cdiv(past_two_passes(8 * sms * 256, 2048), 2048))
    assert_past_two_passes(ctx_write_launch(Q, 2048, sms))
    assert_past_two_passes(aggregate_launch(3, past_two_passes(64 * sms, 3) // 3, sms))
    for N, vec in ((100_000, True), (100_001, False), (100_000, False)):
        assert_past_two_passes(mask_write_launch(256, N, vec, sms))
        assert mask_rowmax_launch(256, N, vec, sms)[1] > 1


def test_kernel_names_from_traces():
    assert _kernel_id("void gf::bias_mask_write_kernel<true>(float const*, float*)") == "bias_mask_write_kernel<true>"
    assert _kernel_id("_ZN2gf22bias_mask_write_kernelILb0EEEvPKfS2_") == "bias_mask_write_kernel<false>"
    assert _kernel_id("void gf::group_mlp_pool_kernel<3>(gf::AggArgs)") == "group_mlp_pool_kernel<3>"
    assert _kernel_id("void gf::knn_brute_kernel<64>(float const*, int)") == "knn_brute_kernel<64>"
    assert _kernel_id("gf::three_interpolate_grad_kernel(float const*)") == "three_interpolate_grad_kernel"
    assert _kernel_id("gf::group_points_kernel(float const*)") == "group_points_kernel"
    assert _kernel_id("void gf::knn_grid_query_kernel<16>(gf::KnnQueryArgs)") is None


@pytest.mark.parametrize("case", sorted(BQ_CASES))
def test_planted_rows_equal_the_oracle(oracle_lib, case):
    """the closed-form rows of the planted scenes are the oracle's"""
    N, m, ns, layouts = BQ_CASES[case]()
    centres, xyz, want = _bq_inputs(N, m, ns, layouts)
    assert np.array_equal(oracle_lib.ball_query(centres, xyz, R, ns), want)


def test_radius_boundary_points_sit_on_and_below_r2(oracle_lib):
    c, xyz, ns, hits, on, below = _radius_scene()
    r2 = np.float32(R) * np.float32(R)
    assert (_sq3(-on) == r2).all()
    assert (_sq3(-below) == np.nextafter(r2, np.float32(0))).all()
    assert np.array_equal(oracle_lib.ball_query(c[None], xyz[None], R, ns)[0], _rows(hits, 2, ns))


def _grad_cases(oracle_lib):
    """op -> (the oracle's serial float32 result, flat destinations, terms in the oracle's order) on small inputs with
    the index patterns of a ball query: sorted rows, the first hit repeated as padding"""
    g = np.random.default_rng(16)
    B, C, N, npoint, ns = 2, 3, 300, 40, 16
    idx = np.stack([np.sort(g.integers(0, N // 2, size=(npoint, ns)), axis=1) for _ in range(B)]).astype(np.int32)
    idx[:, :, ns // 2:] = idx[:, :, :1]
    gidx = np.ascontiguousarray(idx.reshape(B, -1))
    go4 = g.standard_normal(size=(B, C, npoint, ns)).astype(np.float32)
    go3 = g.standard_normal(size=(B, C, npoint * ns)).astype(np.float32)
    n = 500
    tidx = g.integers(0, N, size=(B, n, 3)).astype(np.int32)
    tidx[:, :40] = 7  # an entry with many contributors
    w = g.uniform(0, 1, size=(B, n, 3)).astype(np.float32)
    gi = g.standard_normal(size=(B, C, n)).astype(np.float32)
    return {
        "gather": (oracle_lib.gather_points_grad(go3, gidx, N),) + gather_grad_terms(go3, gidx, N),
        "group": (oracle_lib.group_points_grad(go4, idx, N),) + group_grad_terms(go4, idx, N),
        "interpolate": (oracle_lib.three_interpolate_grad(gi, tidx, w, N),) + interpolate_grad_terms(gi, tidx, w, N),
    }


def _serial_sum(dest, terms, size):
    """float32 adds in list order (np.add.at is unbuffered): the oracle's loop"""
    out = np.zeros(size, np.float32)
    np.add.at(out, dest, terms)
    return out


@pytest.mark.parametrize("op", ["gather", "group", "interpolate"])
def test_bound_holds_for_the_serial_oracle(oracle_lib, op):
    ref, dest, t = _grad_cases(oracle_lib)[op]
    assert atomic_sum_violations(ref, dest, t).size == 0
    assert np.array_equal(_serial_sum(dest, t, ref.size), ref.ravel())
    cnt = np.bincount(dest, minlength=ref.size)
    assert (cnt == 0).any() and (cnt == 1).any() and cnt.max() >= 16  # every rule of the bound is exercised


def test_bound_resolution_flags_many_contributors():
    """interpolation gradients over 100 000 unknown points: into 64 entries (tens of thousands of contributors each)
    the bound is wider than nearly every single term; into 100 000 entries (about 3 each) it resolves nearly all"""
    g = np.random.default_rng(17)
    n = 100_000
    go = g.standard_normal(size=(1, 2, n)).astype(np.float32)
    w = g.uniform(0, 1, size=(1, n, 3)).astype(np.float32)
    for m, lo, hi in ((64, 0.0, 0.2), (n, 0.99, 1.0)):
        idx = g.integers(0, m, size=(1, n, 3)).astype(np.int32)
        frac, _ = bound_resolution(*interpolate_grad_terms(go, idx, w, m), 2 * m)
        assert lo <= frac <= hi, (m, frac)
    with pytest.raises(AssertionError):
        assert_bound_resolves_terms(*interpolate_grad_terms(go, g.integers(0, 64, size=(1, n, 3)).astype(np.int32), w,
                                                            64), 2 * 64)


def test_subnormal_terms_are_refused():
    terms = np.array([1.0, np.float32(1e-40)], np.float32)
    with pytest.raises(AssertionError, match="subnormal"):
        atomic_sum_violations(np.zeros(2, np.float32), np.array([0, 1]), terms)


@pytest.mark.parametrize("fault", ["dropped", "doubled", "neighbour"])
@pytest.mark.parametrize("op", ["gather", "group", "interpolate"])
def test_bound_rejects_a_wrong_sum(oracle_lib, op, fault):
    """the serial sum with one term dropped, counted twice or sent to the next entry of its row fails the bound, for the
    largest term of an entry with many contributors and for the smallest nonzero term of an entry with one"""
    ref, dest, t = _grad_cases(oracle_lib)[op]
    cnt = np.bincount(dest, minlength=ref.size)
    many = np.flatnonzero(cnt[dest] >= 8)
    one = np.flatnonzero((cnt[dest] == 1) & (t != 0))
    for k in (many[np.argmax(np.abs(t[many]))], one[np.argmin(np.abs(t[one]))]):
        d2, t2 = dest.copy(), t.copy()
        if fault == "dropped":
            d2, t2 = np.delete(d2, k), np.delete(t2, k)
        elif fault == "doubled":
            d2, t2 = np.append(d2, d2[k]), np.append(t2, t2[k])
        else:
            d2[k] += 1
        assert atomic_sum_violations(_serial_sum(d2, t2, ref.size), dest, t).size > 0, k
