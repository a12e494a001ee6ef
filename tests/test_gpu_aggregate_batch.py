"""The set aggregator over a ragged batch (geoformer_b200.aggregate.aggregate_batch): scenes of different sizes held as
one flat point array plus offsets, as forward_aggregator (geoformer_fs.py:619-660) holds them.

FPS (gf_furthest_point_sampling_batch): every row equals the single-scene call and the oracle bit for bit, for scene
sizes across every size rule (1 point .. beyond one cluster), for the tie, skip-boundary and no-eligible-point inputs
of test_gpu_fps_variants placed inside ragged batches, and for B = 1, 32 and 33; the profiler shows one cluster launch
per 32 cluster-sized scenes, of the instance the largest one plans, plus one whole-GPU launch per larger scene.

Ball query (gf_ball_query_batch): overlapping rooms (another scene's points lie inside a centre's ball), sizes that
are not multiples of the 2048-point tile, hits on tile edges, empty and padded rows; bit-exact against the
single-scene call and the oracle.

aggregate_batch: inference bitwise equal to aggregate() per scene and on a stacked batch of equal scenes, and within
the oracle tolerance at the model's shape; training against a float64 evaluation of the reference's formulation
(per-scene grouping, cat, conv / batch norm / ReLU, max pool) with the bounds and exclusion rule of
test_aggregate_train; deterministic; per-scene statistics are told apart; malformed inputs raise.

Harness: FewShotForward on a ragged batch, impl "b200" against "torch"."""
import numpy as np
import pytest
import torch

from test_aggregate_train import FRO_REL, MAX_REL, assert_fwd, excluded_pools, layers_of, mlp, rel_errs
from test_gpu_fps_variants import _in_ball, _lattice, _launched, _plan, _skip_boundary_scene, SKIP_M, TIE_M

pytestmark = pytest.mark.gpu

MODEL = dict(m=2048, radius=0.2, ns=64, widths=[19, 32, 32, 32])


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def shape(dev):
    """(largest cluster, SMs): the size rules' inputs, read from the kernel a 65,537-point scene runs"""
    from geoformer_b200.pointnet2 import _ext

    sms = torch.cuda.get_device_properties(0).multi_processor_count
    x = torch.randn(1, 65537, 3, device=dev)
    _, kernels = _launched(lambda: _ext.furthest_point_sampling(x, 2))
    return {("cluster", 256, 20): 16, ("cluster", 512, 24): 8}[kernels[0]], sms


def _flat(scenes):
    """list of (N_b,3) arrays -> flat CUDA (sum N,3) f32, offsets list"""
    off = np.concatenate([[0], np.cumsum([len(s) for s in scenes])]).astype(int).tolist()
    return torch.from_numpy(np.ascontiguousarray(np.concatenate(scenes), dtype=np.float32)).cuda(), off


def _expected_launches(Ns, shape):
    """plan restated: one cluster launch per 32 cluster-sized scenes (instance of the largest), then one whole-GPU
    launch per larger scene"""
    cap = shape[0] * 512 * 24
    small = [n for n in Ns if n <= cap]
    out = []
    if small:
        out += [("cluster_batch",) + _plan(max(small), *shape)[0][1:]] * ((len(small) + 31) // 32)
    return out + [_plan(n, *shape)[0] for n in Ns if n > cap]


def _launched_batch(fn):
    """fn() under the profiler -> result, FPS kernels in launch order with the ragged cluster kernel named
    'cluster_batch'"""
    import re

    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    found = []
    for e in prof.events():
        m = re.search(r"fps_(cluster_batch|cluster|grid)_kernel(?:<([-\d, ]+)>|I((?:Li-?\d+E)+)E)", e.name)
        if m:
            found.append((m.group(1),) + tuple(int(v) for v in re.findall(r"-?\d+", m.group(2) or m.group(3))))
    return out, found


def _check_fps(oracle_lib, shape, scenes, m):
    """ragged call == single-scene call == oracle for every scene; launches as planned"""
    from geoformer_b200.aggregate import furthest_point_sampling_batch
    from geoformer_b200.pointnet2 import _ext

    xyz, off = _flat(scenes)
    got, kernels = _launched_batch(lambda: furthest_point_sampling_batch(xyz, off, m))
    assert kernels == _expected_launches([len(s) for s in scenes], shape)
    got = got.cpu().numpy()
    assert got.shape == (len(scenes), m) and got.dtype == np.int32
    for b, s in enumerate(scenes):
        x = torch.from_numpy(np.ascontiguousarray(s, dtype=np.float32))[None]
        single = _ext.furthest_point_sampling(x.cuda(), m).cpu().numpy()[0]
        want = oracle_lib.furthest_point_sampling(x.numpy(), m)[0]
        assert np.array_equal(single, want), b
        bad = np.flatnonzero(got[b] != want)
        assert bad.size == 0, "scene %d (N=%d): %d wrong seeds, first at round %d" % (b, len(s), bad.size, bad[0])
    return got


# ---- FPS --------------------------------------------------------------------------------------------------------------
SIZES = [1, 37, 300, 511, 512, 4097, 100_000, 196_608, 196_609, 250_000]


def test_fps_batch_every_size_rule(oracle_lib, shape):
    from geoformer_b200.scenes import scene

    scenes = [scene(n, 1000 + i).numpy() for i, n in enumerate(SIZES)]
    _check_fps(oracle_lib, shape, scenes, 2048)  # m > N for the first five scenes


@pytest.mark.parametrize("Ns", [[1, 37, 300, 511], [300, 511, 4097], [511, 100_000]], ids=str)
def test_fps_batch_ties_in_a_larger_cluster(oracle_lib, shape, Ns):
    """lattice scenes (ties at every distance) below 512 points run on the cluster the largest scene plans"""
    _check_fps(oracle_lib, shape, [_lattice(n, 7 + n) for n in Ns], TIE_M)


def test_fps_batch_skip_boundary_and_no_eligible_point(oracle_lib, shape):
    from geoformer_b200.scenes import scene

    skip = [_skip_boundary_scene(n, n)[0] for n in (300, 5000, 120_000)]
    nobody = [_in_ball(n, np.random.default_rng(n)) for n in (256, 9000)]
    got = _check_fps(oracle_lib, shape, [skip[0], nobody[0], scene(20_000, 3).numpy(), skip[1], nobody[1], skip[2]],
                     SKIP_M)
    assert (got[1] == 0).all() and (got[4] == 0).all()


@pytest.mark.parametrize("B", [1, 32, 33])
def test_fps_batch_chunks(oracle_lib, shape, B):
    from geoformer_b200.scenes import scene

    rng = np.random.default_rng(B)
    Ns = rng.integers(200, 6000, size=B).tolist()
    _check_fps(oracle_lib, shape, [scene(n, 50 + i).numpy() for i, n in enumerate(Ns)], 128)


# ---- ball query -------------------------------------------------------------------------------------------------------
def test_ball_query_batch_overlapping_scenes(oracle_lib, dev):
    from geoformer_b200.aggregate import ball_query_batch
    from geoformer_b200.pointnet2 import _ext
    from geoformer_b200.scenes import scene

    Ns = [3001, 2048, 6143, 4097, 700]  # not multiples of the 2048-point tile, and tile-sized
    scenes = [scene(n, 300 + i, L=(3.0, 2.5, 2.0), nbox=4).numpy() for i, n in enumerate(Ns)]
    m, r, ns = 300, 0.1, 24
    rng = np.random.default_rng(5)
    centres = []
    for s in scenes:
        c = s[rng.choice(len(s), m, replace=False)].copy()
        edge = [k for k in (0, 2047, 2048, 4095, 4096, len(s) - 1) if k < len(s)]
        c[:len(edge)] = s[edge]  # hits on tile edges
        c[8:12] = (40.0, 40.0, 40.0)  # nothing in range: an all-zero row
        centres.append(c)
    new_xyz = torch.from_numpy(np.stack(centres)).to(dev)
    xyz, off = _flat(scenes)
    got = ball_query_batch(new_xyz, xyz, off, r, ns).cpu().numpy()
    # some centre has another scene's point inside its ball: a search across scene boundaries would differ
    x = xyz.cpu().numpy()
    cross = 0
    for b in range(len(Ns)):
        other = np.concatenate([x[off[a]:off[a + 1]] for a in range(len(Ns)) if a != b])
        d2 = ((centres[b][:40, None, :] - other[None, ::7, :]) ** 2).sum(-1)
        cross += int((d2 < r * r).any(axis=1).sum())
    assert cross > 0
    for b, s in enumerate(scenes):
        single = _ext.ball_query(new_xyz[b:b + 1].contiguous(), torch.from_numpy(s)[None].to(dev), r, ns).cpu().numpy()
        want = oracle_lib.ball_query(centres[b][None], s[None], r, ns)
        assert np.array_equal(single, want), b
        assert np.array_equal(got[b], want[0]), b
    assert (got[:, 8:12] == 0).all()
    padded = (got[:, :, -1] == got[:, :, 0]) & (got[:, :, 1] != got[:, :, 0])
    assert padded.any(), "some row has fewer than nsample hits"
    assert (got[:, :, -1] != got[:, :, 0]).any(), "some row is full"


def test_ball_query_batch_chunks(oracle_lib, dev):
    from geoformer_b200.aggregate import ball_query_batch
    from geoformer_b200.scenes import scene

    scenes = [scene(n, 400 + i).numpy() for i, n in enumerate(np.random.default_rng(2).integers(50, 3000, 33))]
    xyz, off = _flat(scenes)
    rng = np.random.default_rng(3)
    centres = np.stack([s[rng.integers(0, len(s), 64)] for s in scenes])
    got = ball_query_batch(torch.from_numpy(centres).to(dev), xyz, off, 0.3, 16).cpu().numpy()
    for b, s in enumerate(scenes):
        assert np.array_equal(got[b], oracle_lib.ball_query(centres[b][None], s[None], 0.3, 16)[0]), b


# ---- aggregate_batch --------------------------------------------------------------------------------------------------
class _Grouper:
    pass


def _module(mlp_module, m, radius=0.2, ns=64):
    class M:
        pass

    mod = M()
    mod.npoint, mod.pooling, mod.mlp_module = m, "max", mlp_module
    mod.grouper = _Grouper()
    mod.grouper.radius, mod.grouper.nsample, mod.grouper.normalize_xyz, mod.grouper.use_xyz = radius, ns, True, True
    return mod


def _ragged(Ns, seed, dev, Cf=16):
    from geoformer_b200.scenes import scene

    locs = torch.cat([scene(n, seed + i) for i, n in enumerate(Ns)]).to(dev)
    feats = torch.randn(sum(Ns), Cf, generator=torch.Generator().manual_seed(seed)).to(dev)
    off = np.concatenate([[0], np.cumsum(Ns)]).astype(int).tolist()
    return locs, feats, off


def test_aggregate_batch_inference_equals_per_scene_calls(dev):
    from geoformer_b200.aggregate import aggregate, aggregate_batch

    gen = torch.Generator().manual_seed(3)
    net = mlp(MODEL["widths"], gen).to(dev).eval()
    mod = _module(net, 512)
    locs, feats, off = _ragged([7000, 12_345, 3001, 9000], 70, dev)
    with torch.no_grad():
        cx, cf, ci = aggregate_batch(mod, locs, feats, torch.tensor(off))
        for b in range(4):
            x, f = locs[off[b]:off[b + 1]][None], feats[off[b]:off[b + 1]].t()[None].contiguous()
            nx, nf, ni = aggregate(mod, x, f)
            assert torch.equal(ci[b], ni[0]) and torch.equal(cx[b], nx[0]) and torch.equal(cf[b], nf[0]), b
        # B equally sized scenes: the stacked (B,N,3) call
        locs, feats, off = _ragged([8000] * 3, 80, dev)
        cx, cf, ci = aggregate_batch(mod, locs, feats, off)
        nx, nf, ni = aggregate(mod, locs.reshape(3, 8000, 3), feats.reshape(3, 8000, -1).transpose(1, 2).contiguous())
        assert torch.equal(ci, ni) and torch.equal(cx, nx) and torch.equal(cf, nf)


def test_aggregate_batch_inference_model_shape_oracle(dev):
    from oracle import aggregate_train as ot

    from geoformer_b200.aggregate import aggregate_batch

    gen = torch.Generator().manual_seed(4)
    net = mlp(MODEL["widths"], gen).to(dev).eval()
    locs, feats, off = _ragged([60_000, 100_000, 150_000], 90, dev)
    with torch.no_grad():
        cx, cf, ci = aggregate_batch(_module(net, MODEL["m"]), locs, feats, off)
    layers = layers_of(net.cpu(), torch.float64)
    x = _grouped_ref(locs, feats, off, cx, ci, MODEL["radius"], MODEL["ns"])
    ref, _ = ot.shared_mlp_pool(x, layers, "max", False)
    torch.testing.assert_close(cf.cpu().double(), _per_scene(ref, 3), rtol=1e-4, atol=1e-5)


def _grouped_ref(locs, feats, off, new_xyz, inds, radius, ns, dtype=torch.float64, feats_ref=None):
    """the reference's grouping per scene (oracle ball query on the scene alone), concatenated along the centres:
    (1, 3+C, B*m, ns) -- a batch of B*m centres, as one module.mlp call sees it"""
    import oracle
    from oracle import aggregate_train as ot

    B = len(off) - 1
    f_all = feats_ref if feats_ref is not None else feats.detach().cpu().to(dtype)
    xs = []
    for b in range(B):
        s = locs[off[b]:off[b + 1]].cpu().numpy()
        c = new_xyz[b].cpu().numpy()
        assert np.array_equal(c, s[inds[b].long().cpu().numpy()])
        idx = torch.from_numpy(oracle.ball_query(c[None], s[None], radius, ns))
        xs.append(ot.grouped_input(torch.from_numpy(s)[None].to(dtype), torch.from_numpy(c)[None].to(dtype),
                                   f_all[off[b]:off[b + 1]].t()[None], idx, radius, True, True))
    return torch.cat(xs, dim=2)


def _per_scene(out, B):
    """(1, C, B*m) -> (B, C, m)"""
    return out[0].reshape(out.shape[1], B, -1).transpose(0, 1)


TRAIN_NS = [5000, 8000, 11_000]


def _train_step(net, locs, feats, off, m, ns):
    """aggregate_batch with a gradient wanted for the features -> out, the features leaf, seeds"""
    from geoformer_b200.aggregate import aggregate_batch

    f = feats.clone().requires_grad_()
    _, out, inds = aggregate_batch(_module(net, m, ns=ns), locs, f, off)
    return out, f, inds


def test_aggregate_batch_training_against_float64_reference(dev):
    from oracle import aggregate_train as ot

    gen = torch.Generator().manual_seed(6)
    net = mlp(MODEL["widths"], gen)
    layers = layers_of(net, torch.float64)  # float64 CPU copies for the reference
    net = net.to(dev).train()
    for ly in layers:
        ly["mean0"], ly["var0"] = ly["mean"].clone(), ly["var"].clone()
    m, ns = 256, 32
    locs, feats, off = _ragged(TRAIN_NS, 100, dev)
    out, f, inds = _train_step(net, locs, feats, off, m, ns)
    new_xyz = torch.stack([locs[off[b]:off[b + 1]][inds[b].long()] for b in range(3)])
    f64 = feats.detach().cpu().double().requires_grad_()
    x = _grouped_ref(locs, feats, off, new_xyz, inds, 0.2, ns, feats_ref=f64)
    ref, stats = ot.shared_mlp_pool(x, layers, "max", True)
    assert_fwd(out, _per_scene(ref, 3))
    for l, ly in zip(net, layers):  # running statistics updated once, over the whole batch
        assert int(l[1][0].num_batches_tracked) == 1
        torch.testing.assert_close(l[1][0].running_mean.cpu().double(), ly["mean"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(l[1][0].running_var.cpu().double(), ly["var"], rtol=1e-5, atol=1e-6)
    dy = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    ex = excluded_pools(x.detach(), layers, True, _global_idx(x), "max")
    dy[ex] = 0
    lib_t = [p for l in net for p in (l[0].weight, l[1][0].weight, l[1][0].bias)] + [f]
    ref_t = [t for ly in layers for t in (ly["w"], ly["gamma"], ly["beta"])] + [f64]
    g_lib = torch.autograd.grad(out, lib_t, _per_scene(dy, 3).float().to(dev).contiguous())
    g_ref = torch.autograd.grad(ref, ref_t, dy)
    for i, (a, b) in enumerate(zip(g_lib, g_ref)):
        assert bool(torch.isfinite(a).all()), i
        emax, efro = rel_errs(a.reshape(b.shape), b)
        assert emax <= MAX_REL and efro <= FRO_REL, (i, emax, efro)


def _global_idx(x):
    """excluded_pools compares sample identities by index; distinct (m, s) entries of the grouped input with equal
    columns are the padded duplicates: identify samples by their grouped column"""
    cols = x.detach()[0].permute(1, 2, 0).reshape(-1, x.shape[1])
    _, inv = torch.unique(cols, dim=0, return_inverse=True)
    return inv.reshape(1, x.shape[2], x.shape[3]).int()


def test_aggregate_batch_running_statistics_two_steps_and_determinism(dev):
    import copy

    from oracle import aggregate_train as ot

    gen = torch.Generator().manual_seed(7)
    net = mlp(MODEL["widths"], gen)
    layers = layers_of(net, torch.float64)  # float64 CPU copies for the reference
    net = net.to(dev).train()
    twin = copy.deepcopy(net)
    m, ns = 256, 32
    results = []
    for step in range(2):
        locs, feats, off = _ragged(TRAIN_NS, 200 + 10 * step, dev)
        for which in (net, twin):
            out, f, inds = _train_step(which, locs, feats, off, m, ns)
            g = torch.autograd.grad(out, [p for p in which.parameters()] + [f], torch.ones_like(out))
            results.append((out.detach(), g))
        new_xyz = torch.stack([locs[off[b]:off[b + 1]][inds[b].long()] for b in range(3)])
        ot.shared_mlp_pool(_grouped_ref(locs, feats, off, new_xyz, inds, 0.2, ns), layers, "max", True)
        # two calls give bitwise-equal outputs and gradients
        (o1, g1), (o2, g2) = results[-2], results[-1]
        assert torch.equal(o1, o2) and all(torch.equal(a, b) for a, b in zip(g1, g2))
    for l, t, ly in zip(net, twin, layers):
        assert torch.equal(l[1][0].running_mean, t[1][0].running_mean)
        assert torch.equal(l[1][0].running_var, t[1][0].running_var)
        assert int(l[1][0].num_batches_tracked) == 2
        torch.testing.assert_close(l[1][0].running_mean.cpu().double(), ly["mean"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(l[1][0].running_var.cpu().double(), ly["var"], rtol=1e-5, atol=1e-6)


def test_per_scene_statistics_miss_the_bounds(dev):
    """aggregate() per scene in training mode, concatenated: each scene normalised with its own statistics -- the
    forward misses the tolerance the one-pass call meets"""
    from oracle import aggregate_train as ot

    from geoformer_b200.aggregate import aggregate

    gen = torch.Generator().manual_seed(6)
    net = mlp(MODEL["widths"], gen)
    layers = layers_of(net, torch.float64)  # float64 CPU copies for the reference
    net = net.to(dev).train()
    m, ns = 256, 32
    locs, feats, off = _ragged(TRAIN_NS, 100, dev)
    outs, cs, ids = [], [], []
    with torch.no_grad():
        for b in range(3):
            nx, nf, ni = aggregate(_module(net, m, ns=ns), locs[off[b]:off[b + 1]][None],
                                   feats[off[b]:off[b + 1]].t()[None].contiguous())
            outs.append(nf), cs.append(nx[0]), ids.append(ni[0])
    ref, _ = ot.shared_mlp_pool(_grouped_ref(locs, feats, off, torch.stack(cs), torch.stack(ids), 0.2, ns), layers,
                                "max", True)
    with pytest.raises(AssertionError):
        assert_fwd(torch.cat(outs), _per_scene(ref, 3))


def test_aggregate_batch_rejects_malformed_input(dev):
    from geoformer_b200 import _capi as C
    from geoformer_b200.aggregate import aggregate_batch

    net = mlp(MODEL["widths"], torch.Generator().manual_seed(1)).to(dev).eval()
    mod = _module(net, 64)
    locs, feats, off = _ragged([3000, 2000], 5, dev)
    cases = [
        (locs, feats, [0, 3000, 3000, 5000]),  # an empty scene
        (locs, feats, [0, 3000, 2000, 5000]),  # offsets fall
        (locs, feats, [0, 3000, 4000]),  # do not end at sum N
        (locs, feats, [1, 3000, 5000]),  # do not start at 0
        (locs, feats[:-1], off),  # feature rows != sum N
        (locs.cpu(), feats, off),  # CPU tensors
        (locs, feats.cpu(), off),
    ]
    torch.cuda.synchronize()
    C.reset_launch_count()
    for l, f, o in cases:
        with torch.no_grad(), pytest.raises(RuntimeError):
            aggregate_batch(mod, l, f, o)
    assert C.launch_count() == 0


# ---- harness ----------------------------------------------------------------------------------------------------------
def test_few_shot_forward_on_a_ragged_batch(dev):
    from geoformer_b200.harness import FewShotForward
    from geoformer_b200.scenes import scene

    torch.manual_seed(12)
    Ns, m = [12_000, 20_000, 31_000], 16
    net = FewShotForward(m=m, nlayers=2, n_decode_point=512, n_query_points=64).to(dev)
    locs = torch.cat([scene(n, 60 + b, L=(4.0, 3.0, 2.0), nbox=6) for b, n in enumerate(Ns)]).to(dev)
    feats = torch.randn(sum(Ns), m, device=dev)
    support = torch.randn(3, 2 * m, device=dev)
    off = torch.tensor([0] + np.cumsum(Ns).tolist())
    kw = dict(max_step=48, neighbor=16, geo_radius=0.2, batch_offsets=off)
    la, ga, ia = net(locs, feats, support, impl="b200", **kw)
    lb, gb, ib = net(locs, feats, support, impl="torch", **kw)
    assert torch.equal(ia, ib)
    for b, n in enumerate(Ns):
        assert torch.equal(ga[b], gb[b]) and ga[b].shape == (64, n)
        assert la[b].shape == (64, n) and torch.isfinite(la[b]).all()
        scale = lb[b].abs().max().item()
        assert (la[b] - lb[b]).abs().max().item() <= 0.02 * scale + 1e-6, b
    net.train()
    logits, _, _ = net.forward_train(locs, feats, support, impl="b200", **kw)
    sum(l.square().mean() for l in logits).backward()
    for name, p in net.named_parameters():
        if p.requires_grad:
            assert p.grad is not None and bool(torch.isfinite(p.grad).all()), name
