"""The set aggregator in training form (geoformer_b200.aggregate.group_mlp_pool_train, gf_aggregate_train.cu).

CPU: the float64 oracle (oracle.aggregate_train) equals nn.Conv2d + nn.BatchNorm2d + ReLU + max/avg pool modules built
like the harness's conv_bn, in training and eval mode, momentum 0.1 and None: output, batch statistics, running
statistics after one and two steps, autograd gradients; the C entries validate their arguments before any CUDA call.

GPU: forward output and batch statistics against the float64 oracle at the model shape and at ragged shapes; running
statistics after two steps; no_grad with a training-mode module; the eval-mode forward is bitwise gf_group_mlp_pool;
gradients against autograd through the float64 oracle; determinism; data inputs refuse gradients; unfused forms
still raise; peak memory; FewShotForward trained through both impls.

Forward tolerance: fp32 products and fp32 per-layer rounding against float64: |got - ref| <= 1e-4 |ref| + 1e-4 (the
outputs are O(1) after batch norm); batch statistics 1e-5 relative.

Backward tolerance.  With a random-sign upstream gradient, a pooled maximum whose top two samples lie within fp32
rounding can flip its argmax, moving a row of dW_L by about 1/sqrt(B m) of its size.  So the upstream gradient is
zeroed at the pools whose float64 top-two gap (over distinct points: padded duplicates are exact ties in both paths
and map to the same point), or whose argmax sample's |y_l| at any layer and channel, is below DELTA = 1e-4; a ReLU
whose input lies that close to its kink may set its mask differently in fp32.  Then every gradient is checked as
max |g - g_ref| / max |g_ref| <= 2e-5 and ||g - g_ref|| / ||g_ref|| <= 1e-5 (the conv bias in batch mode, whose exact
gradient is zero, against 1e-3 of gamma's gradient scale).  Measured on a B200 (1000 W, 1965 MHz) the worst ratios
over every case below are 2.4e-6 (max) and 1.4e-6 (Frobenius).  test_bounds_catch_a_wrong_backward shows that the oracle's gradient with the batch-norm mean
term or the sum(dy xhat) term dropped misses these bounds by orders of magnitude, so the bounds can catch a wrong
backward."""
import copy
import ctypes

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

DELTA = 1e-4
MAX_REL, FRO_REL = 2e-5, 1e-5


# ---- fixtures and helpers --------------------------------------------------------------------------------------------
def conv_bn(cin, cout, gen, bias=False, bn=True):
    """pytorch_utils.Conv2d(bn=True) as the harness builds it, with non-trivial parameters and running statistics"""
    conv = nn.Conv2d(cin, cout, 1, bias=bias)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(cout, cin, 1, 1, generator=gen) / np.sqrt(cin))
        if bias:
            conv.bias.copy_(torch.randn(cout, generator=gen) * 0.2)
    if not bn:
        return nn.Sequential(conv, nn.ReLU())
    b = nn.BatchNorm2d(cout)
    with torch.no_grad():
        b.weight.uniform_(0.5, 1.5, generator=gen)
        b.bias.normal_(0, 0.2, generator=gen)
        b.running_mean.normal_(0, 0.3, generator=gen)
        b.running_var.uniform_(0.5, 1.5, generator=gen)
    return nn.Sequential(conv, nn.Sequential(b), nn.ReLU())


def mlp(widths, gen, bias=False, bn=True):
    return nn.Sequential(*[conv_bn(widths[i], widths[i + 1], gen, bias, bn) for i in range(len(widths) - 1)])


def layers_of(module, dtype=None):
    """oracle layer dicts of an nn SharedMLP (parameters as leaves of `dtype` requiring grad)"""
    out = []
    for layer in module:
        conv, bn = layer[0], (layer[1][0] if len(layer) == 3 else None)
        cv = lambda t: None if t is None else t.detach().to(dtype or t.dtype).clone().requires_grad_()  # noqa: E731
        ly = {"w": cv(conv.weight.reshape(conv.out_channels, -1)), "b": cv(conv.bias)}
        if bn is not None:
            ly.update(gamma=cv(bn.weight), beta=cv(bn.bias),
                      mean=bn.running_mean.detach().to(dtype or torch.float32).clone(),
                      var=bn.running_var.detach().to(dtype or torch.float32).clone(),
                      nbt=bn.num_batches_tracked.detach().clone())
        out.append(ly)
    return out


def lib_call(xyz, new_xyz, feats, idx, radius, norm, use_xyz, layers, batch, pooling="max", momentum=0.1):
    """group_mlp_pool_train on the oracle layer dicts (fp32 CUDA copies as leaves requiring grad)"""
    from geoformer_b200.aggregate import group_mlp_pool_train

    dev = xyz.device
    cv = lambda t: None if t is None else t.detach().float().to(dev).clone().requires_grad_()  # noqa: E731
    p = [{k: cv(ly.get(k)) for k in ("w", "b", "gamma", "beta")} for ly in layers]
    run = [{k: (ly[k].detach().float().to(dev).clone() if ly.get(k) is not None else None) for k in ("mean", "var", "nbt")}
           for ly in layers]
    out = group_mlp_pool_train(xyz, new_xyz, feats, idx, radius, norm, use_xyz, [q["w"] for q in p], [q["b"] for q in p],
                               [q["gamma"] for q in p], [q["beta"] for q in p], [r["mean"] for r in run],
                               [r["var"] for r in run], batch, momentum=momentum, pooling=pooling,
                               num_batches_tracked=[r["nbt"] for r in run])
    return out, p, run


def scene_case(B, N, m, ns, Cf, radius, seed, dev, outliers=0):
    """B scenes.scene point clouds, FPS centres, ball query: (xyz, new_xyz, feats, idx) on dev"""
    from geoformer_b200.pointnet2 import _ext
    from geoformer_b200.scenes import scene

    xyz = torch.stack([scene(N, seed + b) for b in range(B)])
    if outliers:
        xyz[:, -outliers:] = xyz[:, -outliers:] + 50.0 + torch.arange(outliers, dtype=torch.float32)[:, None] * 7.0
    xyz = xyz.to(dev).contiguous()
    gen = torch.Generator().manual_seed(seed)
    feats = torch.randn(B, Cf, N, generator=gen).to(dev) if Cf else None
    inds = _ext.furthest_point_sampling(xyz, m)
    new_xyz = _ext.gather_points(xyz.transpose(1, 2).contiguous(), inds).transpose(1, 2).contiguous()
    idx = _ext.ball_query(new_xyz, xyz, radius, ns)
    return xyz, new_xyz, feats, idx


def oracle64(xyz, new_xyz, feats, idx, radius, norm, use_xyz, layers, batch, pooling="max", momentum=0.1, drop=()):
    from oracle import aggregate_train as ot

    x = ot.grouped_input(xyz.double().cpu(), new_xyz.double().cpu(), feats.double().cpu() if feats is not None else None,
                         idx.cpu(), radius, norm, use_xyz)
    return ot.shared_mlp_pool(x, layers, pooling, batch, momentum, drop=drop), x


def assert_fwd(got, ref):
    ref = ref.detach().float()
    err = (got.detach().cpu() - ref).abs()
    assert bool((err <= 1e-4 * ref.abs() + 1e-4).all()), float(err.max())


def rel_errs(g, r):
    g, r = g.detach().double().cpu(), r.detach().double().cpu()
    d = g - r
    return (d.abs().max() / r.abs().max().clamp_min(1e-30)).item(), (d.norm() / r.norm().clamp_min(1e-30)).item()


def excluded_pools(x, layers, batch, idx, pooling):
    """(B, C_out, m) bool: pools whose float64 top-two gap over distinct points, or whose argmax sample's |y| at any
    layer, is below DELTA (see the module docstring)"""
    with torch.no_grad():
        ys, h = [], x
        for ly in layers:
            z = F.conv2d(h, ly["w"].detach()[:, :, None, None], None if ly.get("b") is None else ly["b"].detach())
            if ly.get("gamma") is not None:
                if batch:
                    mean, var = z.mean(dim=(0, 2, 3)), z.var(dim=(0, 2, 3), unbiased=False)
                else:
                    mean, var = ly["mean0"], ly["var0"]
                z = (z - mean[None, :, None, None]) / torch.sqrt(var + 1e-5)[None, :, None, None]
                z = z * ly["gamma"].detach()[None, :, None, None] + ly["beta"].detach()[None, :, None, None]
            ys.append(z)
            h = F.relu(z)
        B, Co, m, ns = h.shape
        if pooling != "max":
            near = torch.stack([y.abs().amin(dim=1) for y in ys]).amin(dim=0).amin(dim=2) < DELTA  # (B, m)
            return near[:, None, :].expand(B, Co, m)
        top, arg = h.max(dim=3)
        same = idx.long().cpu()[:, None, :, :].expand(B, Co, m, ns) == \
            torch.gather(idx.long().cpu()[:, None].expand(B, Co, m, ns), 3, arg[..., None])
        second = torch.where(same, torch.full_like(h, -1.0), h).max(dim=3)[0]
        ex = (top - second) < DELTA
        for y in ys:  # |y| of every channel at the argmax sample of each output channel
            ya = y.abs().permute(0, 2, 3, 1)  # (B, m, ns, C_l)
            at = torch.gather(ya, 2, arg.permute(0, 2, 1)[..., None].expand(B, m, Co, ya.shape[3]))  # (B,m,Co,C_l)
            ex |= (at.amin(dim=3) < DELTA).permute(0, 2, 1)
        return ex


# ---- CPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("pooling", ["max", "avg"])
@pytest.mark.parametrize("momentum", [0.1, None])
def test_oracle_equals_torch_modules_float64(training, pooling, momentum):
    from oracle import aggregate_train as ot

    gen = torch.Generator().manual_seed(1)
    B, m, ns, widths = 2, 24, 8, [7, 12, 9, 10]
    mod = mlp(widths, gen).double()
    for layer in mod:
        layer[1][0].momentum = momentum
    mod.train(training)
    ly = layers_of(mod, torch.float64)
    for step in range(2):
        x = torch.randn(B, widths[0], m, ns, generator=gen, dtype=torch.float64)
        x_ref, x_or = x.clone().requires_grad_(), x.clone().requires_grad_()
        inputs, h = [], x_ref
        for layer in mod:
            inputs.append(layer[0](h))
            h = layer[2](layer[1](inputs[-1]))
        want = (F.max_pool2d(h, [1, ns]) if pooling == "max" else F.avg_pool2d(h, [1, ns])).squeeze(-1)
        got, stats = ot.shared_mlp_pool(x_or, ly, pooling, training, momentum)
        torch.testing.assert_close(got, want, rtol=1e-12, atol=1e-12)
        for i, layer in enumerate(mod):
            bn = layer[1][0]
            torch.testing.assert_close(ly[i]["mean"], bn.running_mean, rtol=1e-12, atol=1e-14)
            torch.testing.assert_close(ly[i]["var"], bn.running_var, rtol=1e-12, atol=1e-14)
            if training:
                z = inputs[i].detach()
                torch.testing.assert_close(stats[i][0], z.mean(dim=(0, 2, 3)), rtol=1e-12, atol=1e-14)
                torch.testing.assert_close(stats[i][1], z.var(dim=(0, 2, 3), unbiased=False), rtol=1e-12, atol=1e-14)
        dy = torch.randn(want.shape, generator=gen, dtype=torch.float64)
        gw = torch.autograd.grad(want, [x_ref] + [p for layer in mod for p in layer.parameters()], dy)
        go = torch.autograd.grad(got, [x_or] + [ly[i][k] for i in range(len(ly)) for k in ("w", "gamma", "beta")], dy)
        for a, b in zip(go, gw):
            torch.testing.assert_close(a, b.reshape(a.shape), rtol=1e-10, atol=1e-12)


def test_entries_validate_before_any_cuda_call(cuda_lib):
    L = cuda_lib
    assert L.gf_group_mlp_pool_train_workspace_bytes(0, 10) == 0 and L.gf_group_mlp_pool_train_workspace_bytes(1, 64) > 0
    assert L.gf_group_mlp_pool_backward_workspace_bytes(1, 100, 64, 8, 16) >= 64 * 8 * 16 * 4
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below fails its checks first
    P = ctypes.c_void_p * 4
    ptrs = P(fake, fake, fake, fake)
    widths = (ctypes.c_int * 4)(19, 32, 32, 32)
    batch = (ctypes.c_int * 3)(1, 1, 1)
    eps = (ctypes.c_float * 3)(1e-5, 1e-5, 1e-5)

    def train(B=1, N=100, m=8, ns=4, C=16, use_xyz=1, nl=3, w=widths, out=fake, gam=ptrs, bat=batch):
        return L.gf_group_mlp_pool_train(fake, fake, fake, fake, B, N, m, ns, C, 0.2, 1, use_xyz, nl, w, ptrs, gam,
                                         ptrs, eps, bat, fake, 0, out, fake, 1 << 20, None)

    assert train(B=-1) == 1 and b"bad sizes" in L.gf_last_error()
    assert train(nl=5) == 1 and b"5 layers" in L.gf_last_error()
    assert train(C=15) == 1 and b"first width" in L.gf_last_error()
    assert train(out=None) == 1 and b"null pointer" in L.gf_last_error()
    assert train(w=(ctypes.c_int * 4)(19, 33, 32, 32)) == 1 and b"width 33" in L.gf_last_error()
    assert train(gam=P(fake, None, fake, fake)) == 1 and b"layer 1 needs gamma" in L.gf_last_error()

    def bwd(B=1, ns=4, nl=3, dout=fake, dws=ptrs):
        return L.gf_group_mlp_pool_backward(fake, fake, fake, fake, B, 100, 8, ns, 16, 0.2, 1, 1, nl, widths, ptrs,
                                            batch, fake, 0, dout, fake, dws, fake, fake, 1 << 20, None)

    assert bwd(ns=0) == 1 and b"bad sizes" in L.gf_last_error()
    assert bwd(nl=0) == 1 and b"0 layers" in L.gf_last_error()
    assert bwd(dout=None) == 1 and b"null pointer" in L.gf_last_error()
    assert bwd(dws=P(fake, fake, None, fake)) == 1 and b"null dweights of layer 2" in L.gf_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev(cuda_lib):
    return torch.device("cuda:0")


MODEL = dict(N=100_000, m=2048, ns=64, Cf=16, radius=0.2)


def check_backward(xyz, new_xyz, feats, idx, radius, norm, use_xyz, layers, batch, pooling="max", seed=0):
    """gradients of the library op against autograd through the float64 oracle, with the exclusion rule; returns the
    worst (max, Frobenius) ratios per gradient"""
    for ly in layers:
        if ly.get("gamma") is not None:
            ly["mean0"], ly["var0"] = ly["mean"].clone(), ly["var"].clone()
    feats_l = feats.clone().requires_grad_() if feats is not None else None
    out, p, _ = lib_call(xyz, new_xyz, feats_l, idx, radius, norm, use_xyz, layers, batch, pooling)
    f64 = feats.double().cpu().requires_grad_() if feats is not None else None
    from oracle import aggregate_train as ot

    x = ot.grouped_input(xyz.double().cpu(), new_xyz.double().cpu(), f64, idx.cpu(), radius, norm, use_xyz)
    for ly in layers:  # the oracle's running-statistics form reads them, batch form updates them: use copies
        if ly.get("gamma") is not None:
            ly["mean"], ly["var"] = ly["mean0"].clone(), ly["var0"].clone()
    ref, _ = ot.shared_mlp_pool(x, layers, pooling, batch)
    assert_fwd(out, ref)
    gen = torch.Generator().manual_seed(seed)
    dy = torch.randn(ref.shape, generator=gen, dtype=torch.float64)
    dy[excluded_pools(x.detach(), layers, batch, idx, pooling)] = 0
    names, lib_t, ref_t = [], [], []
    for i, (ly, q) in enumerate(zip(layers, p)):
        for k in ("w", "b", "gamma", "beta"):
            if ly.get(k) is not None:
                names.append("%s%d" % (k, i)), lib_t.append(q[k]), ref_t.append(ly[k])
    if feats is not None:
        names.append("features"), lib_t.append(feats_l), ref_t.append(f64)
    g_lib = torch.autograd.grad(out, lib_t, dy.float().to(out.device))
    g_ref = torch.autograd.grad(ref, ref_t, dy)
    worst = {}
    gscale = max([g.abs().max().item() for n, g in zip(names, g_ref) if n.startswith("gamma")] + [0.0])
    for n, a, b in zip(names, g_lib, g_ref):
        assert bool(torch.isfinite(a).all()), n
        if n.startswith("b") and not n.startswith("beta") and batch and layers[int(n[1:])].get("gamma") is not None:
            err = (a.detach().double().cpu() - b).abs().max().item()
            print("%-9s |g| %.2e (exact gradient 0)" % (n, a.abs().max().item()))
            assert err <= 1e-3 * gscale, (n, err, gscale)
            continue
        emax, efro = rel_errs(a, b)
        worst[n] = (emax, efro)
        print("%-9s max %.2e fro %.2e" % (n, emax, efro))
        assert emax <= MAX_REL and efro <= FRO_REL, (n, emax, efro)
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 3])
def test_forward_and_batch_statistics_model_shape(dev, B):
    gen = torch.Generator().manual_seed(B)
    xyz, new_xyz, feats, idx = scene_case(B, MODEL["N"], MODEL["m"], MODEL["ns"], MODEL["Cf"], MODEL["radius"], 11, dev)
    layers = layers_of(mlp([19, 32, 32, 32], gen), torch.float64)
    # momentum 1: the running statistics become the batch mean and the unbiased batch variance
    out, _, run = lib_call(xyz, new_xyz, feats, idx, MODEL["radius"], True, True, layers, True, momentum=1.0)
    (ref, stats), _ = oracle64(xyz, new_xyz, feats, idx, MODEL["radius"], True, True, layers, True, momentum=1.0)
    assert out.shape == (B, 32, MODEL["m"])
    assert_fwd(out, ref)
    n = B * MODEL["m"] * MODEL["ns"]
    for r, (mean, var) in zip(run, stats):
        torch.testing.assert_close(r["mean"].cpu().double(), mean, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(r["var"].cpu().double(), var * n / (n - 1), rtol=1e-5, atol=1e-6)


RAGGED = {  # name: (widths, Cf, use_xyz, normalize, pooling, ns, m, bias, bn)
    "L1": ([19, 32], 16, True, True, "max", 16, 256, False, True),
    "L4": ([19, 32, 32, 32, 32], 16, True, True, "max", 16, 256, False, True),
    "w5_7_32": ([5, 7, 32], 2, True, True, "max", 16, 256, True, True),
    "no_xyz": ([16, 24, 32], 16, False, True, "max", 16, 256, False, True),
    "no_normalize": ([19, 32, 32], 16, True, False, "max", 16, 256, False, True),
    "avg": ([19, 32, 32, 32], 16, True, True, "avg", 16, 256, False, True),
    "ns1": ([19, 32, 32], 16, True, True, "max", 1, 256, False, True),
    "m_odd": ([19, 32, 32], 16, True, True, "max", 16, 203, False, True),
    "no_bn_bias": ([19, 32, 20], 16, True, True, "max", 16, 256, True, False),
}


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [True, False])
@pytest.mark.parametrize("case", sorted(RAGGED))
def test_ragged_forward_and_backward(dev, case, batch):
    widths, Cf, use_xyz, norm, pooling, ns, m, bias, bn = RAGGED[case]
    gen = torch.Generator().manual_seed(5)
    xyz, new_xyz, feats, idx = scene_case(2, 6000, m, ns, Cf, 0.2, 21, dev)
    layers = layers_of(mlp(widths, gen, bias, bn), torch.float64)
    check_backward(xyz, new_xyz, feats, idx, 0.2, norm, use_xyz, layers, batch, pooling)


@pytest.mark.gpu
def test_sparse_outliers_pad_and_dead_channel(dev):
    """centres on far outliers: their balls hold only themselves, padded with duplicates of the first hit; one channel
    of the second layer is dead for every sample (gamma 0, beta < 0)"""
    gen = torch.Generator().manual_seed(8)
    xyz, new_xyz, feats, idx = scene_case(2, 6000, 256, 32, 16, 0.2, 31, dev, outliers=40)
    assert bool((idx[:, :, 1:] == idx[:, :, :1]).all(dim=2).any())
    layers = layers_of(mlp([19, 32, 32, 32], gen), torch.float64)
    with torch.no_grad():
        layers[1]["gamma"][3] = 0.0
        layers[1]["beta"][3] = -1.0
    for batch in (True, False):
        check_backward(xyz, new_xyz, feats, idx, 0.2, True, True, copy.deepcopy(layers), batch)


@pytest.mark.gpu
@pytest.mark.parametrize("momentum", [0.1, None])
def test_running_statistics_after_two_steps(dev, momentum):
    gen = torch.Generator().manual_seed(9)
    layers = layers_of(mlp([19, 32, 32], gen), torch.float64)
    lib_layers = copy.deepcopy(layers)
    for step in range(2):
        xyz, new_xyz, feats, idx = scene_case(2, 6000, 256, 32, 16, 0.2, 40 + step, dev)
        _, _, run = lib_call(xyz, new_xyz, feats, idx, 0.2, True, True, lib_layers, True, momentum=momentum)
        for ly, r in zip(lib_layers, run):
            ly["mean"], ly["var"], ly["nbt"] = r["mean"].cpu().double(), r["var"].cpu().double(), r["nbt"].cpu()
        oracle64(xyz, new_xyz, feats, idx, 0.2, True, True, layers, True, momentum=momentum)
    for a, b in zip(lib_layers, layers):
        torch.testing.assert_close(a["mean"], b["mean"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(a["var"], b["var"], rtol=1e-5, atol=1e-6)
        assert int(a["nbt"]) == int(b["nbt"]) == 2


class _Grouper:
    pass


def _module(mlp_module, m, pooling="max", npoint=True):
    class M:
        pass

    mod = M()
    mod.npoint, mod.pooling, mod.mlp_module = (m if npoint else None), pooling, mlp_module
    mod.grouper = _Grouper()
    mod.grouper.radius, mod.grouper.nsample, mod.grouper.normalize_xyz, mod.grouper.use_xyz = 0.2, 32, True, True
    return mod


@pytest.mark.gpu
def test_aggregate_routes_training_modules_and_keeps_eval_bitwise(dev):
    from geoformer_b200.aggregate import aggregate

    gen = torch.Generator().manual_seed(12)
    xyz, _, feats, _ = scene_case(2, 6000, 256, 32, 16, 0.2, 50, dev)
    net = mlp([19, 32, 32, 32], gen).to(dev)
    mod = _module(net, 256)
    # eval module: under no_grad the inference entry; under grad the op, bitwise the same output, with a grad_fn
    net.eval()
    with torch.no_grad():
        _, want, inds = aggregate(mod, xyz, feats)
    _, got, _ = aggregate(mod, xyz, feats, inds=inds)
    assert got.grad_fn is not None and want.grad_fn is None
    assert torch.equal(got, want)
    # training module under no_grad: batch statistics, running statistics updated
    net.train()
    before = [l[1][0].running_mean.clone() for l in net]
    with torch.no_grad():
        _, out, _ = aggregate(mod, xyz, feats, inds=inds)
    assert all(not torch.equal(b, l[1][0].running_mean) for b, l in zip(before, net))
    assert all(int(l[1][0].num_batches_tracked) == 1 for l in net)
    assert not torch.equal(out, want)


@pytest.mark.gpu
@pytest.mark.parametrize("batch", [True, False])
def test_backward_model_shape(dev, batch):
    gen = torch.Generator().manual_seed(13)
    xyz, new_xyz, feats, idx = scene_case(1, MODEL["N"], MODEL["m"], MODEL["ns"], MODEL["Cf"], MODEL["radius"], 60, dev)
    layers = layers_of(mlp([19, 32, 32, 32], gen, bias=True), torch.float64)
    check_backward(xyz, new_xyz, feats, idx, MODEL["radius"], True, True, layers, batch)


@pytest.mark.gpu
def test_bounds_catch_a_wrong_backward(dev):
    """the float64 oracle's gradients with the batch-norm mean term, or the sum(dy xhat) term, dropped are compared
    with the true ones under the same exclusion: both miss MAX_REL / FRO_REL by more than 10x"""
    from oracle import aggregate_train as ot

    gen = torch.Generator().manual_seed(13)
    xyz, new_xyz, feats, idx = scene_case(1, 20_000, 1024, MODEL["ns"], MODEL["Cf"], MODEL["radius"], 61, dev)
    layers = layers_of(mlp([19, 32, 32, 32], gen), torch.float64)
    x = ot.grouped_input(xyz.double().cpu(), new_xyz.double().cpu(), feats.double().cpu(), idx.cpu(), 0.2, True, True)
    dy = torch.randn((1, 32, 1024), generator=gen, dtype=torch.float64)
    dy[excluded_pools(x, layers, True, idx, "max")] = 0
    params = [ly[k] for ly in layers for k in ("w", "gamma")]
    good = torch.autograd.grad(ot.shared_mlp_pool(x, layers, "max", True)[0], params, dy)
    for drop in (("mean",), ("var",)):
        lys = copy.deepcopy(layers)
        bad = torch.autograd.grad(ot.shared_mlp_pool(x, lys, "max", True, drop=drop)[0],
                                  [ly[k] for ly in lys for k in ("w", "gamma")], dy)
        worst = max(max(rel_errs(b, g)[0] / MAX_REL, rel_errs(b, g)[1] / FRO_REL) for b, g in zip(bad, good))
        print("drop %s: worst error / bound %.1f" % (drop, worst))
        assert worst > 10, (drop, worst)


@pytest.mark.gpu
def test_deterministic(dev):
    gen = torch.Generator().manual_seed(14)
    xyz, new_xyz, feats, idx = scene_case(2, 20_000, 1024, 64, 16, 0.2, 70, dev)
    layers = layers_of(mlp([19, 32, 32, 32], gen, bias=True), torch.float64)
    dy = torch.randn(2, 32, 1024, generator=gen).to(dev)
    res = []
    for _ in range(2):
        f = feats.clone().requires_grad_()
        out, p, run = lib_call(xyz, new_xyz, f, idx, 0.2, True, True, layers, True)
        grads = torch.autograd.grad(out, [f] + [q[k] for q in p for k in ("w", "b", "gamma", "beta")], dy)
        res.append([out] + list(grads) + [r[k] for r in run for k in ("mean", "var")])
    assert all(torch.equal(a, b) for a, b in zip(*res))


@pytest.mark.gpu
def test_data_inputs_refuse_gradients_and_unfused_forms_raise(dev):
    from geoformer_b200.aggregate import aggregate

    gen = torch.Generator().manual_seed(15)
    xyz, new_xyz, feats, idx = scene_case(1, 3000, 64, 16, 16, 0.2, 80, dev)
    layers = layers_of(mlp([19, 32], gen), torch.float64)
    for which in ("xyz", "new_xyz"):
        a = xyz.clone().requires_grad_() if which == "xyz" else xyz
        b = new_xyz.clone().requires_grad_() if which == "new_xyz" else new_xyz
        with pytest.raises(RuntimeError, match="no gradient"):
            lib_call(a, b, feats, idx, 0.2, True, True, layers, True)
    net = mlp([19, 32], gen).to(dev).train()
    with pytest.raises(RuntimeError, match="rbf"):
        aggregate(_module(net, 64, pooling="rbf"), xyz, feats)
    with pytest.raises(RuntimeError, match="GroupAll"):
        aggregate(_module(net, 64, npoint=False), xyz, feats)


@pytest.mark.gpu
def test_peak_memory_model_shape_b4(dev):
    """forward + backward at B = 4 allocates under 100 MB above its inputs (70 MB measured on a B200): the per-sample
    input gradient (B m ns C fp32 = 34 MB), the inverse index (~6 MB), the feature gradient (26 MB) and the other
    workspaces.  torch autograd through the reference formulation peaks at 551 MB at this shape
    (tools/measure_aggregate_train.py, profiles/r06)."""
    gen = torch.Generator().manual_seed(16)
    xyz, new_xyz, feats, idx = scene_case(4, MODEL["N"], MODEL["m"], MODEL["ns"], MODEL["Cf"], MODEL["radius"], 90, dev)
    layers = layers_of(mlp([19, 32, 32, 32], gen), torch.float64)
    f = feats.clone().requires_grad_()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out, p, _ = lib_call(xyz, new_xyz, f, idx, MODEL["radius"], True, True, layers, True)
    out.backward(torch.ones_like(out))
    torch.cuda.synchronize()
    peak = (torch.cuda.max_memory_allocated() - base) / 1e6
    print("peak above inputs: %.1f MB" % peak)
    assert peak < 100, peak


# ---- harness -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_forward_aggregator_trains_through_both_impls(dev):
    """FewShotForward.forward_aggregator in training mode: the mlp_module gradients and running statistics of
    impl="b200" and impl="torch" (cuDNN without TF32) agree.  Both are fp32; the few pools whose argmax differs
    between the two move a gradient row by ~1/sqrt(B m): Frobenius 2e-2, max 5e-2 relative."""
    from geoformer_b200.harness import FewShotForward
    from geoformer_b200.scenes import scene

    torch.manual_seed(0)
    base = FewShotForward(n_query_points=128).to(dev).train()
    B, N = 2, 50_000
    locs = torch.stack([scene(N, 100 + b) for b in range(B)]).to(dev)
    feats = torch.randn(B, N, 16, generator=torch.Generator().manual_seed(1)).to(dev)
    wl = torch.randn(B, 2048, 32, generator=torch.Generator().manual_seed(2)).to(dev)
    res = {}
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        for impl in ("b200", "torch"):
            model = copy.deepcopy(base)
            _, cf, _ = model.forward_aggregator(locs, feats, impl)
            params = list(model.mlp_module.parameters())
            grads = torch.autograd.grad((cf * wl).sum(), params)
            run = [t for l in model.mlp_module for t in (l[1][0].running_mean, l[1][0].running_var)]
            res[impl] = (grads, run)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    for i, (a, b) in enumerate(zip(res["b200"][0], res["torch"][0])):
        emax, efro = rel_errs(a, b)
        print("mlp param %d: max %.2e fro %.2e" % (i, emax, efro))
        assert efro <= 2e-2 and emax <= 5e-2, (i, emax, efro)
    for a, b in zip(res["b200"][1], res["torch"][1]):
        torch.testing.assert_close(a, b, rtol=1e-4, atol=1e-5)


@pytest.mark.gpu
def test_forward_train_step_both_impls(dev):
    """one forward_train step (model with n_query_points=128, max_step=128) with a loss on the mask logits: every
    parameter that gets a gradient on the torch path gets a finite one on the b200 path, and they agree within
    0.5 max / 0.2 Frobenius relative.  The chain passes through the TF32 decoder and mask head and, on the torch path,
    cuDNN's TF32 convolutions of the aggregator, whose argmax flips differ from the fp32 kernel's: the decoder test's
    scale (0.15 max / 0.1 Frobenius) is the expectation.  Measured on a B200 (1000 W, 1965 MHz): Frobenius <= 0.07
    for all but two small bias vectors of the second decoder layer (norm3.bias 0.135, linear1.bias 0.124), max
    <= 0.32 (linear1.bias); the weights of the aggregator's SharedMLP <= 0.06 Frobenius.  A wrong gradient anywhere
    in the chain shows as O(1).  Gradients that are zero by construction (the last bias of each attn_mlp: the softmax is
    shift invariant) are checked to stay below 1e-5 of the largest gradient norm instead."""
    from geoformer_b200.harness import FewShotForward
    from geoformer_b200.scenes import scene

    torch.manual_seed(0)
    base = FewShotForward(n_query_points=128).to(dev).train()
    B, N = 2, 20_000
    locs = torch.stack([scene(N, 200 + b) for b in range(B)]).to(dev)
    feats = torch.randn(B, N, 16, generator=torch.Generator().manual_seed(1)).to(dev)
    se = torch.randn(B, 32, generator=torch.Generator().manual_seed(2)).to(dev)
    wl = [torch.randn(128, N, generator=torch.Generator().manual_seed(3 + b)).to(dev) for b in range(B)]
    grads = {}
    for impl in ("b200", "torch"):
        model = copy.deepcopy(base)
        logits, _, _ = model.forward_train(locs, feats, se, impl=impl, max_step=128)
        loss = sum((lg * w).sum() for lg, w in zip(logits, wl)) / N
        names = [n for n, _ in model.named_parameters()]
        gs = torch.autograd.grad(loss, list(model.parameters()), allow_unused=True)
        grads[impl] = dict(zip(names, gs))
    scale = max(b.norm().item() for b in grads["torch"].values() if b is not None)
    bad = []
    for n, b in grads["torch"].items():
        if b is None:
            continue
        a = grads["b200"][n]
        assert a is not None and bool(torch.isfinite(a).all()), n
        if b.norm().item() <= 1e-5 * scale:  # zero by construction (attn_mlp's last bias: softmax shift invariance)
            print("%-50s |g| %.1e, torch %.1e (zero gradient)" % (n, a.norm().item(), b.norm().item()))
            if a.norm().item() > 1e-5 * scale:
                bad.append(n)
            continue
        emax, efro = rel_errs(a, b)
        print("%-50s max %.2e fro %.2e" % (n, emax, efro))
        if not (emax <= 0.5 and efro <= 0.2):
            bad.append(n)
    assert not bad, bad
