"""The training kernels of the set aggregator (gf_aggregate_train.cu) at the size of a training batch, against the
float64 oracle (oracle/aggregate_train.py) through the helpers and bounds of test_aggregate_train.py.

A training step runs group_mlp_pool_train once over every scene's centres, so its kernels see B m in the tens of
thousands, B m ns in the millions and B N (the keys of the feature gradient) around 2^20.  Each kernel caps its grid and
walks the rest of its work in a loop, or, for the scan of tile totals, in chunks:

    kernel                              launch rule (restated below)                        one pass covers
    agg_stats_kernel<K> (K = 0..3)      min(ceil(Bm/8), 8 SMs) CTAs, one centre a warp      64 SMs centres
    group_mlp_pool_kernel<L>            the same rule (the output pass)                     64 SMs centres
    agg_backward_kernel<L> (L = 1..4)   min(ceil(Bm/8), 2 SMs) CTAs, one centre a warp      16 SMs centres
    agg_count_kernel, agg_place_kernel  min(ceil(Bm ns/256), 16 SMs) CTAs, one entry a thread  4096 SMs entries
    agg_scan_totals_kernel              1 CTA, a carry over chunks of 1024 tiles of 1024 keys  2^20 keys
    agg_segment_sum_kernel              one thread a key: insertion sort, then a serial sum  --
    agg_stats_finish_kernel             1 CTA; sums the statistics kernel's grid of partial rows
    agg_backward_finish_kernel          ceil(1120/128) CTAs; sums the backward kernel's grid of partial rows

Each case is sized from this device's SM count to take two full passes and a partial one (or, for the scan, two full
chunks and a partial one), which is asserted before it runs; every launch and its grid is then read from the
profiler's trace and compared with the rules.  The last GPU test asserts that together the cases reached every
(kernel, regime) pair of REGIMES.

1. Statistics and backward past two passes, for every template instance: batch statistics in every layer, L = 1..4
   with max pooling and L = 3 with avg pooling, three scenes of 20k points with ~8k centres each.  Output, batch and
   running statistics, every gradient; two calls bitwise equal.
2. The feature gradient over more than 2 * 2^20 keys (three scan chunks, the last partial) and past two count / place
   passes, on a synthetic idx: most keys referenced by no entry (their gradient must be exactly 0), entries in every
   chunk, and planted points at the chunk edges referenced by 1000..4000 entries each (long segments).
3. aggregate_batch in training at a model batch: 8 ragged scenes of 61k..150k points, m = 2048, ns = 32, against the
   float64 evaluation of the reference's formulation.  2^20 < sum N: the realistic path crosses the first chunk edge.

Bounds: MAX_REL / FRO_REL of test_aggregate_train, unchanged, with its exclusion rule.  Measured on a B200 (1000 W
power limit, 1965 MHz) the worst ratios over every case are 1.05e-5 (max, the feature gradient of L = 3 with max
pooling) and 3.5e-6 (Frobenius).  The CPU tests at the end show, in float64 on the inputs the GPU cases build for 148
SMs, that the faults a wrong loop bound, a lost CTA partial or a wrong carry would produce miss those bounds: batch
statistics without the last partial statistics pass (by 400x or more), a dW without one CTA's partial row (the weakest
CTA: 5000x), dfeatures shifted by one key past the first chunk (1e5x), one segment's sum dropped (the longest: 800x;
the one of median magnitude: 3x; MAX_REL resolves the loss of 84 % of the nonempty segments).

On that B200 the GPU tests of this file take about 15 s; the float64 reference of case 3 brings the test process to a
peak of 3.6 GB resident host memory.
"""
import copy
import resource

import numpy as np
import pytest
import torch

from test_aggregate_train import FRO_REL, MAX_REL, assert_fwd, check_backward, excluded_pools, layers_of, lib_call, \
    mlp, oracle64, rel_errs
from test_gpu_ops_launch_shapes import B200_SMS, _cdiv, _expect, _kernel_id, _launched, _runs_every_gpu_test_here, \
    assert_past_two_passes, passes, past_two_passes

# ------------------------------------------------------------------------------------------ launch rules, restated
WARPS = 8  # AGT_THREADS / 32: centres a CTA takes per pass
SCAN = 1024  # AGT_SCAN_THREADS: keys a tile, tiles a chunk of the carried scan


def stats_launch(Bm, sms):
    """agg_stats_kernel<K> and the output pass: -> (grid, centres, centres a pass)"""
    grid = max(1, min(_cdiv(Bm, WARPS), 8 * sms))
    return grid, Bm, grid * WARPS


def backward_launch(Bm, sms):
    """agg_backward_kernel<L>"""
    grid = max(1, min(_cdiv(Bm, WARPS), 2 * sms))
    return grid, Bm, grid * WARPS


def entries_launch(ent, sms):
    """agg_count_kernel, agg_place_kernel: one (scene, centre, sample) entry a thread"""
    grid = min(_cdiv(ent, 256), 16 * sms)
    return grid, ent, grid * 256


def scan_launch(keys):
    """-> (tiles: agg_scan_tiles_kernel's grid, chunks agg_scan_totals_kernel carries over)"""
    tiles = _cdiv(keys, SCAN)
    return tiles, _cdiv(tiles, SCAN)


BACKWARD_FINISH_GRID = _cdiv(32 * 32 + 32 + 2 * 32, 128)  # dW and dbias, then the two sums of the layer below


def train_launches(B, N, m, ns, L, sms):
    """[(kernel, grid)] of one forward + backward of group_mlp_pool_train with batch statistics in every layer"""
    sg, bg = stats_launch(B * m, sms)[0], backward_launch(B * m, sms)[0]
    out = []
    for k in range(L):
        out += [("agg_stats_kernel<%d>" % k, (sg, 1, 1)), ("agg_stats_finish_kernel", (1, 1, 1))]
    out.append(("group_mlp_pool_kernel<%d>" % L, (sg, 1, 1)))
    finish = ("agg_backward_finish_kernel", (BACKWARD_FINISH_GRID, 1, 1))
    out += [("agg_backward_kernel<%d>" % L, (bg, 1, 1)), finish] * (L + 1)
    eg, tiles, keys = entries_launch(B * m * ns, sms)[0], scan_launch(B * N)[0], B * N
    return out + [("agg_count_kernel", (eg, 1, 1)), ("agg_scan_tiles_kernel", (tiles, 1, 1)),
                  ("agg_scan_totals_kernel", (1, 1, 1)), ("agg_scan_add_kernel", (_cdiv(keys, 256), 1, 1)),
                  ("agg_place_kernel", (eg, 1, 1)), ("agg_segment_sum_kernel", (_cdiv(keys, 256), 1, 1))]


KERNELS = sorted(["agg_stats_kernel", "agg_stats_finish_kernel", "group_mlp_pool_kernel", "agg_backward_kernel",
                  "agg_backward_finish_kernel", "agg_count_kernel", "agg_scan_tiles_kernel", "agg_scan_totals_kernel",
                  "agg_scan_add_kernel", "agg_place_kernel", "agg_segment_sum_kernel"], key=len, reverse=True)

# the (kernel, regime) pairs the cases below must reach together
REGIMES = {("agg_stats_kernel<%d>" % k, "past two passes") for k in range(4)} | {
    ("agg_backward_kernel<%d>" % L, "past two passes") for L in range(1, 5)} | {
    ("agg_count_kernel", "past two passes"),
    ("agg_place_kernel", "past two passes"),
    ("agg_scan_totals_kernel", "past two chunks"),
    ("agg_segment_sum_kernel", "segments of 1000..4000 entries"),
}
_REACHED = set()


def _assert_past_two_chunks(keys):
    tiles, chunks = scan_launch(keys)
    assert chunks >= 3 and tiles % SCAN != 0, (keys, tiles)


def _peak_rss_gb():
    """this process's peak resident set so far (Linux: ru_maxrss in KiB)"""
    return resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 2 ** 20


# ------------------------------------------------------------------------------------------ case 1: statistics
RADIUS = 0.2
STATS_B, STATS_N, STATS_NS, STATS_CF = 3, 20_000, 16, 16
WIDTHS = {1: [19, 32], 2: [19, 32, 32], 3: [19, 32, 32, 32], 4: [19, 32, 24, 32, 17]}
STATS_CASES = [(1, "max"), (2, "max"), (3, "max"), (4, "max"), (3, "avg")]


def stats_case_m(sms):
    """centres a scene: B m past 2.5 statistics passes, the last statistics and backward passes partial"""
    m = past_two_passes(8 * WARPS * sms, STATS_B) // STATS_B
    while (STATS_B * m) % (8 * WARPS * sms) == 0 or (STATS_B * m) % (2 * WARPS * sms) == 0:
        m += 1
    return m


def stats_case_inputs(m, ball_query):
    """three scenes.scene clouds, m centres each picked from the points, their ball query -> CPU (xyz, new_xyz, feats,
    idx); ball_query(new_xyz, xyz) is the library's or the oracle's (bitwise equal, test_gpu_parity)"""
    from geoformer_b200.scenes import scene

    xyz = torch.stack([scene(STATS_N, 40 + b) for b in range(STATS_B)])
    pick = [torch.randperm(STATS_N, generator=torch.Generator().manual_seed(b))[:m] for b in range(STATS_B)]
    new_xyz = torch.stack([xyz[b, pick[b]] for b in range(STATS_B)]).contiguous()
    feats = torch.randn(STATS_B, STATS_CF, STATS_N, generator=torch.Generator().manual_seed(41))
    return xyz, new_xyz, feats, ball_query(new_xyz, xyz)


def stats_case_layers(L):
    return layers_of(mlp(WIDTHS[L], torch.Generator().manual_seed(30 + L), bias=True), torch.float64)


# ------------------------------------------------------------------------------------------ case 2: feature gradient
CARRY_B, CARRY_N, CARRY_NS, CARRY_CF = 2, 1_100_000, 64, 2
CARRY_WIDTHS = [5, 8, 8]
CARRY_RADIUS = 0.5
# planted keys b N + p at the scan's chunk edges and the last key, with the entries that reference them
PLANTED = {(0, SCAN * SCAN - 1): 1000, (0, SCAN * SCAN): 2500, (1, 2 * SCAN * SCAN - CARRY_N): 4000,
           (1, CARRY_N - 1): 1500}


def carry_case_m(sms):
    """centres a scene: B m ns past 2.5 count / place passes, the last partial"""
    return past_two_passes(256 * 16 * sms, CARRY_B * CARRY_NS) // (CARRY_B * CARRY_NS)


def carry_case_inputs(m):
    """points uniform in a unit box; every centre samples a random quarter of its scene's points, and each planted
    point takes one random sample of each of PLANTED[key] centres (no centre holds two planted points); a centre sits
    on its first sample.
    -> CPU (xyz, new_xyz, feats, idx)"""
    B, N, ns = CARRY_B, CARRY_N, CARRY_NS
    g = np.random.default_rng(90)
    xyz = g.uniform(0, 1, size=(B, N, 3)).astype(np.float32)
    feats = g.standard_normal(size=(B, CARRY_CF, N)).astype(np.float32)
    idx = np.empty((B, m, ns), np.int32)
    for b in range(B):
        pool = np.sort(g.choice(N, N // 4, replace=False))
        rows = pool[g.integers(0, len(pool), size=(m, ns))]
        centres, at = g.permutation(m), 0
        for (pb, p), c in PLANTED.items():
            if pb == b:
                rows[centres[at:at + c], g.integers(0, ns, size=c)] = p
                at += c
        idx[b] = rows
    new_xyz = np.stack([xyz[b, idx[b, :, 0]] for b in range(B)])
    return tuple(torch.from_numpy(np.ascontiguousarray(a)) for a in (xyz, new_xyz, feats, idx))


def carry_case_keys(idx):
    """-> entries a key (B N,), with the key b N + idx[b, j, s] of every entry"""
    B = idx.shape[0]
    keys = (np.arange(B)[:, None, None] * CARRY_N + idx.numpy()).ravel()
    return np.bincount(keys, minlength=B * CARRY_N)


def assert_carry_layout(idx, sms):
    """the properties case 2 relies on, asserted before it runs"""
    B, m, ns = idx.shape
    assert_past_two_passes(entries_launch(B * m * ns, sms))
    _assert_past_two_chunks(B * CARRY_N)
    cnt = carry_case_keys(idx)
    chunk = SCAN * SCAN
    assert all(cnt[c * chunk:(c + 1) * chunk].sum() > 0 for c in range(scan_launch(B * CARRY_N)[1])), \
        "a scan chunk without entries"
    assert (cnt == 0).mean() > 0.7, "most keys must have no entry"
    planted = np.array([b * CARRY_N + p for b, p in PLANTED])
    assert (cnt[planted] >= np.array(list(PLANTED.values()))).all()
    rest = np.delete(cnt, planted)
    assert rest.max() < 20 and cnt[planted].min() >= 1000 and cnt[planted].max() < 4100
    for b, p in PLANTED:  # spread over many centres
        assert (idx[b] == p).any(dim=1).sum() >= PLANTED[(b, p)]
    return cnt


# ------------------------------------------------------------------------------------------ case 3: aggregate_batch
BATCH_NS = [150_000, 61_000, 149_000, 143_000, 137_000, 150_000, 131_000, 128_000]  # sum 1,049,000 > 2^20
BATCH_M, BATCH_NSAMPLE, BATCH_WIDTHS = 2048, 32, [19, 32, 32, 32]


# ------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def sms(dev):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _train_twice(xyz, new_xyz, feats, idx, radius, layers, pooling, dy):
    """two forward + backward calls at momentum 1 (running statistics = the batch mean and the unbiased batch
    variance) -> [output, gradients of features and every parameter, running statistics] of each"""
    res = []
    for _ in range(2):
        f = feats.clone().requires_grad_()
        out, p, run = lib_call(xyz, new_xyz, f, idx, radius, True, True, copy.deepcopy(layers), True, pooling,
                               momentum=1.0)
        grads = torch.autograd.grad(out, [f] + [q[k] for q in p for k in ("w", "b", "gamma", "beta")], dy)
        res.append([out] + list(grads) + [r[k] for r in run for k in ("mean", "var")])
    return res


def _check_running_statistics(res, stats, n, L):
    """the running statistics of a momentum-1 call against the oracle's batch statistics"""
    run = res[-2 * L:]
    for l, (mean, var) in enumerate(stats):
        torch.testing.assert_close(run[2 * l].cpu().double(), mean, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(run[2 * l + 1].cpu().double(), var * n / (n - 1), rtol=1e-5, atol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("L,pooling", STATS_CASES)
def test_statistics_and_backward_past_two_passes(dev, sms, L, pooling):
    from geoformer_b200.pointnet2 import _ext

    m = stats_case_m(sms)
    Bm = STATS_B * m
    assert_past_two_passes(stats_launch(Bm, sms))
    assert_past_two_passes(backward_launch(Bm, sms))
    xyz, new_xyz, feats, idx = [t.to(dev) for t in stats_case_inputs(
        m, lambda c, x: _ext.ball_query(c.to(dev), x.to(dev), RADIUS, STATS_NS))]
    layers = stats_case_layers(L)

    # gradients against the float64 oracle; every launch and grid of the forward and the backward
    worst, kernels = _launched(lambda: check_backward(xyz, new_xyz, feats, idx, RADIUS, True, True,
                                                      copy.deepcopy(layers), True, pooling), KERNELS)
    _expect(kernels, train_launches(STATS_B, STATS_N, m, STATS_NS, L, sms))
    print("L=%d %s: worst gradient errors %s; peak host RSS %.2f GB" % (L, pooling, worst, _peak_rss_gb()))

    # output, batch statistics (the running statistics at momentum 1); two calls bitwise equal
    (ref, stats), _ = oracle64(xyz, new_xyz, feats, idx, RADIUS, True, True, copy.deepcopy(layers), True, pooling,
                               momentum=1.0)
    dy = torch.randn(ref.shape, generator=torch.Generator().manual_seed(L)).to(dev)
    a, b = _train_twice(xyz, new_xyz, feats, idx, RADIUS, layers, pooling, dy)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    assert_fwd(a[0], ref)
    _check_running_statistics(a, stats, Bm * STATS_NS, L)
    for k in range(L):
        _REACHED.add(("agg_stats_kernel<%d>" % k, "past two passes"))
    _REACHED.add(("agg_backward_kernel<%d>" % L, "past two passes"))


@pytest.mark.gpu
def test_feature_gradient_across_scan_chunks_and_entry_passes(dev, sms):
    m = carry_case_m(sms)
    xyz, new_xyz, feats, idx = carry_case_inputs(m)
    cnt = assert_carry_layout(idx, sms)
    xyz, new_xyz, feats, idx = [t.to(dev) for t in (xyz, new_xyz, feats, idx)]
    layers = layers_of(mlp(CARRY_WIDTHS, torch.Generator().manual_seed(91), bias=True), torch.float64)

    worst, kernels = _launched(lambda: check_backward(xyz, new_xyz, feats, idx, CARRY_RADIUS, True, True,
                                                      copy.deepcopy(layers), True), KERNELS)
    _expect(kernels, train_launches(CARRY_B, CARRY_N, m, CARRY_NS, len(CARRY_WIDTHS) - 1, sms))
    print("worst gradient errors %s; peak host RSS %.2f GB" % (worst, _peak_rss_gb()))

    # keys without an entry get exactly 0; two calls bitwise equal
    dy = torch.randn(CARRY_B, CARRY_WIDTHS[-1], m, generator=torch.Generator().manual_seed(92)).to(dev)
    a, b = _train_twice(xyz, new_xyz, feats, idx, CARRY_RADIUS, layers, "max", dy)
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    df = a[1].cpu().numpy().transpose(1, 0, 2).reshape(CARRY_CF, -1)  # (C, B N): key-major per channel
    assert (df[:, cnt == 0] == 0).all()
    assert (df[:, cnt > 0] != 0).mean() > 0.99
    for k in ("agg_count_kernel", "agg_place_kernel"):
        _REACHED.add((k, "past two passes"))
    _REACHED.add(("agg_scan_totals_kernel", "past two chunks"))
    _REACHED.add(("agg_segment_sum_kernel", "segments of 1000..4000 entries"))


@pytest.mark.gpu
def test_aggregate_batch_training_at_a_model_batch(oracle_lib, dev, sms):
    """as test_gpu_aggregate_batch.py::test_aggregate_batch_training_against_float64_reference, at 8 scenes"""
    from oracle import aggregate_train as ot
    from test_gpu_aggregate_batch import _global_idx, _grouped_ref, _module, _per_scene, _ragged

    from geoformer_b200.aggregate import aggregate_batch

    B, m, ns = len(BATCH_NS), BATCH_M, BATCH_NSAMPLE
    assert passes(stats_launch(B * m, sms)) >= 2 and passes(backward_launch(B * m, sms)) > 2
    assert scan_launch(sum(BATCH_NS))[1] == 2
    gen = torch.Generator().manual_seed(93)
    net = mlp(BATCH_WIDTHS, gen)
    layers = layers_of(net, torch.float64)  # float64 CPU copies for the reference
    net = net.to(dev).train()
    locs, feats, off = _ragged(BATCH_NS, 300, dev)

    def step():
        f = feats.clone().requires_grad_()
        _, out, inds = aggregate_batch(_module(net, m, ns=ns), locs, f, off)
        return out, f, inds

    (out, f, inds), kernels = _launched(step, KERNELS)
    _expect(kernels, train_launches(1, sum(BATCH_NS), B * m, ns, 3, sms)[:7])  # the forward
    rss0 = _peak_rss_gb()
    new_xyz = torch.stack([locs[off[b]:off[b + 1]][inds[b].long()] for b in range(B)])
    f64 = feats.detach().cpu().double().requires_grad_()
    x = _grouped_ref(locs, feats, off, new_xyz, inds, 0.2, ns, feats_ref=f64)
    ref, _ = ot.shared_mlp_pool(x, layers, "max", True)
    assert_fwd(out, _per_scene(ref, B))
    for l, ly in zip(net, layers):  # running statistics updated once, over the whole batch
        assert int(l[1][0].num_batches_tracked) == 1
        torch.testing.assert_close(l[1][0].running_mean.cpu().double(), ly["mean"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(l[1][0].running_var.cpu().double(), ly["var"], rtol=1e-5, atol=1e-6)
    dy = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    dy[excluded_pools(x.detach(), layers, True, _global_idx(x), "max")] = 0
    lib_t = [p for l in net for p in (l[0].weight, l[1][0].weight, l[1][0].bias)] + [f]
    ref_t = [t for ly in layers for t in (ly["w"], ly["gamma"], ly["beta"])] + [f64]
    g_lib, kernels = _launched(lambda: torch.autograd.grad(out, lib_t, _per_scene(dy, B).float().to(dev).contiguous()),
                               KERNELS)
    _expect(kernels, train_launches(1, sum(BATCH_NS), B * m, ns, 3, sms)[7:])  # the backward
    g_ref = torch.autograd.grad(ref, ref_t, dy)
    print("peak host RSS before the float64 reference %.2f GB, after %.2f GB" % (rss0, _peak_rss_gb()))
    for i, (a, b) in enumerate(zip(g_lib, g_ref)):
        assert bool(torch.isfinite(a).all()), i
        emax, efro = rel_errs(a.reshape(b.shape), b)
        print("gradient %d: max %.2e fro %.2e" % (i, emax, efro))
        assert emax <= MAX_REL and efro <= FRO_REL, (i, emax, efro)


@pytest.mark.gpu
def test_every_kernel_regime_reached(request):
    """runs after the tests above (file order): together they reached every (kernel, regime) pair"""
    if not _runs_every_gpu_test_here(request):
        pytest.skip("needs every GPU test of this file in one session and process")
    assert _REACHED == REGIMES, sorted(REGIMES - _REACHED)


# ------------------------------------------------------------------------------------------ CPU: rules and sizes
def test_launch_rules_on_b200():
    """the thresholds where a second pass or a second chunk starts on 148 SMs"""
    s = B200_SMS
    assert passes(stats_launch(9472, s)) == 1 and passes(stats_launch(9473, s)) == 2
    assert passes(backward_launch(2368, s)) == 1 and passes(backward_launch(2369, s)) == 2
    assert passes(entries_launch(606_208, s)) == 1 and passes(entries_launch(606_209, s)) == 2
    assert scan_launch(2 ** 20) == (1024, 1) and scan_launch(2 ** 20 + 1) == (1025, 2)
    assert scan_launch(2 ** 21 + 1)[1] == 3 and BACKWARD_FINISH_GRID == 9
    assert stats_launch(1, s)[0] == 1 and backward_launch(1, s)[0] == 1
    # the model training batch of the issue's arithmetic: 8 scenes of 2048 centres, 64 samples
    assert passes(stats_launch(16_384, s)) == 2 and passes(backward_launch(16_384, s)) == 7
    assert passes(entries_launch(16_384 * 64, s)) == 2


@pytest.mark.parametrize("sms", [100, 132, 148, 160])
def test_cases_take_two_passes_and_a_part(sms):
    """the sizes the GPU cases derive from the SM count land past two passes on any of these devices"""
    m = stats_case_m(sms)
    assert_past_two_passes(stats_launch(STATS_B * m, sms))
    assert_past_two_passes(backward_launch(STATS_B * m, sms))
    assert m < STATS_N
    m = carry_case_m(sms)
    assert_past_two_passes(entries_launch(CARRY_B * m * CARRY_NS, sms))
    assert all(sum(c for (pb, _), c in PLANTED.items() if pb == b) <= m for b in range(CARRY_B))
    _assert_past_two_chunks(CARRY_B * CARRY_N)
    assert all(0 <= p < CARRY_N for _, p in PLANTED)
    assert passes(backward_launch(len(BATCH_NS) * BATCH_M, sms)) > 2
    assert all(60_000 <= n <= 150_000 for n in BATCH_NS) and scan_launch(sum(BATCH_NS))[1] == 2


def test_kernel_names_from_traces():
    assert _kernel_id("void gf::agg_stats_kernel<2>(gf::AgtArgs)", KERNELS) == "agg_stats_kernel<2>"
    assert _kernel_id("_ZN2gf19agg_backward_kernelILi4EEEvN2gf7AgtArgsEi", KERNELS) == "agg_backward_kernel<4>"
    assert _kernel_id("gf::agg_stats_finish_kernel(double const*, int)", KERNELS) == "agg_stats_finish_kernel"
    assert _kernel_id("gf::agg_backward_finish_kernel(float const*)", KERNELS) == "agg_backward_finish_kernel"
    assert _kernel_id("gf::agg_scan_totals_kernel(int*, int, int*)", KERNELS) == "agg_scan_totals_kernel"
    assert _kernel_id("void gf::group_mlp_pool_kernel<3>(gf::AggArgs)", KERNELS) == "group_mlp_pool_kernel<3>"
    assert _kernel_id("void gf::ball_query_kernel(float const*)", KERNELS) is None


def test_carry_case_layout():
    """the synthetic idx of case 2 at 148 SMs has the properties the GPU case asserts"""
    cnt = assert_carry_layout(carry_case_inputs(carry_case_m(B200_SMS))[3], B200_SMS)
    print("keys without an entry: %.3f; planted segments %s" % ((cnt == 0).mean(),
                                                                 [int(cnt[b * CARRY_N + p]) for b, p in PLANTED]))


# ------------------------------------------------------------------------------------------ CPU: the faults miss
class _ConvCapture(torch.overrides.TorchFunctionMode):
    """records (input, output) of every conv2d the oracle runs; the outputs keep their gradient"""

    def __init__(self):
        super().__init__()
        self.io = []

    def __torch_function__(self, func, types, args=(), kwargs=None):
        out = func(*args, **(kwargs or {}))
        if func is torch.nn.functional.conv2d or func is torch.conv2d:
            out.retain_grad()
            self.io.append((args[0], out))
        return out


def _miss(bad, good):
    """by how much `bad` misses the gradient bounds: > 1 fails check_backward"""
    emax, efro = rel_errs(bad, good)
    return max(emax / MAX_REL, efro / FRO_REL)


@pytest.fixture(scope="module")
def stats_oracle(oracle_lib):
    """case 1 (L = 3, max pooling) at 148 SMs in float64: the conv inputs and outputs with their gradients, dW"""
    from oracle import aggregate_train as ot

    m = stats_case_m(B200_SMS)
    xyz, new_xyz, feats, idx = stats_case_inputs(m, lambda c, x: torch.from_numpy(
        oracle_lib.ball_query(c.numpy(), x.numpy(), RADIUS, STATS_NS)))
    layers = stats_case_layers(3)
    x = ot.grouped_input(xyz.double(), new_xyz.double(), feats.double(), idx, RADIUS, True, True)
    with _ConvCapture() as cap:
        ref, _ = ot.shared_mlp_pool(x, copy.deepcopy(layers), "max", True)
    dy = torch.randn(ref.shape, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    dy[excluded_pools(x, layers, True, idx, "max")] = 0
    ref.backward(dy)
    return m, cap.io


def test_statistics_without_the_last_partial_pass_miss(stats_oracle):
    """each layer's batch mean and variance over the centres of the full statistics passes only: the running
    statistics check (rtol 1e-5, atol 1e-6) fails"""
    m, io = stats_oracle
    Bm = STATS_B * m
    _, _, per_pass = stats_launch(Bm, B200_SMS)
    keep = torch.arange(Bm) < (passes(stats_launch(Bm, B200_SMS)) - 1) * per_pass
    assert 0 < int((~keep).sum()) < per_pass
    for l, (_, z) in enumerate(io):
        z = z.detach().transpose(0, 1).reshape(z.shape[1], Bm, -1)  # (C, B m, ns): centre cj = b m + j
        n, nk = z[0].numel(), z[:, keep].shape[1] * z.shape[2]
        for want, got in ((z.mean(dim=(1, 2)), z[:, keep].mean(dim=(1, 2))),
                          (z.var(dim=(1, 2), unbiased=False) * n / (n - 1),
                           z[:, keep].var(dim=(1, 2), unbiased=False) * nk / (nk - 1))):
            miss = ((got - want).abs() / (1e-6 + 1e-5 * want.abs())).max().item()
            print("layer %d: statistics without the last partial pass miss the bound by %.0fx" % (l, miss))
            assert miss > 10, (l, miss)


def test_dw_without_one_cta_partial_row_misses(stats_oracle):
    """dW of each layer without the partial row of one backward CTA (CTA k sums the centres cj with
    (cj mod 8 grid) // 8 == k): the weakest CTA of every layer still misses MAX_REL / FRO_REL"""
    m, io = stats_oracle
    Bm = STATS_B * m
    grid = backward_launch(Bm, B200_SMS)[0]
    cta = (torch.arange(Bm) % (grid * WARPS)) // WARPS
    for l, (h, z) in enumerate(io):
        dz = z.grad.transpose(0, 1).reshape(z.shape[1], Bm, -1)
        prev = h.detach().transpose(0, 1).reshape(h.shape[1], Bm, -1)
        per_centre = torch.einsum("ocs,ics->coi", dz, prev)
        rows = torch.zeros((grid,) + per_centre.shape[1:], dtype=torch.float64).index_add_(0, cta, per_centre)
        dw = rows.sum(dim=0)
        miss = min(_miss(dw - rows[k], dw) for k in range(grid))
        print("layer %d: dW without the weakest CTA's row misses the bounds by %.0fx" % (l, miss))
        assert miss > 10, (l, miss)


@pytest.fixture(scope="module")
def carry_oracle():
    """case 2 at 148 SMs in float64: the feature gradient, key-major per channel (C, B N), and entries a key"""
    from oracle import aggregate_train as ot

    xyz, new_xyz, feats, idx = carry_case_inputs(carry_case_m(B200_SMS))
    layers = layers_of(mlp(CARRY_WIDTHS, torch.Generator().manual_seed(91), bias=True), torch.float64)
    f64 = feats.double().requires_grad_()
    x = ot.grouped_input(xyz.double(), new_xyz.double(), f64, idx, CARRY_RADIUS, True, True)
    ref, _ = ot.shared_mlp_pool(x, layers, "max", True)
    dy = torch.randn(ref.shape, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    dy[excluded_pools(x.detach(), layers, True, idx, "max")] = 0
    (g,) = torch.autograd.grad(ref, [f64], dy)
    return g.transpose(0, 1).reshape(CARRY_CF, -1), carry_case_keys(idx)


def test_dfeatures_shifted_past_the_first_chunk_miss(carry_oracle):
    """the keys past the first chunk read their neighbour's segment (an off-by-one carry): the bounds fail, and keys
    without an entry get a nonzero gradient"""
    g, cnt = carry_oracle
    bad = g.clone()
    bad[:, SCAN * SCAN:] = g[:, SCAN * SCAN - 1:-1]
    miss = _miss(bad, g)
    nonzero = int(((bad != 0).any(dim=0) & torch.from_numpy(cnt == 0)).sum())
    print("a carry off by one key misses the bounds by %.0fx; %d keys without an entry get a gradient"
          % (miss, nonzero))
    assert miss > 10 and nonzero > 0


def test_one_segment_dropped_misses(carry_oracle):
    """one key's segment sum dropped: the longest (a planted point) and the one of median magnitude miss the bounds.
    MAX_REL resolves the loss of a segment whose sum exceeds MAX_REL of the largest key's; the fraction of the nonempty
    segments that holds for is printed"""
    g, cnt = carry_oracle
    mag = g.abs().amax(dim=0)
    nonempty = np.flatnonzero(cnt > 0)
    resolved = (mag[nonempty] > MAX_REL * mag.max()).double().mean().item()
    med = nonempty[np.argsort(mag[nonempty].numpy())[len(nonempty) // 2]]
    for key in (int(np.argmax(cnt)), int(med)):
        bad = g.clone()
        bad[:, key] = 0
        miss = _miss(bad, g)
        print("segment of key %d (%d entries) dropped: misses the bounds by %.0fx" % (key, cnt[key], miss))
        assert miss > 1, (key, miss)
    print("the bounds resolve the loss of %.4f of the nonempty segments" % resolved)
