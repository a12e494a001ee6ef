"""The fused mask head over a ragged batch (geoformer_b200.mask_head.mask_heads_forward_batch,
gf_mask_head_logits_batch(_backward)): persistent CTAs take 128-point tiles from the tiles of all scenes.

CPU: both entries and both workspace queries refuse bad input before any CUDA call; the Python op refuses CPU tensors,
mismatched shapes and data that requires grad; the new kernels multiply on the tensor cores.

GPU: every logit is bitwise the single-scene op's on its scene (ragged sizes across tile edges, Q across query groups,
B past one C call, unaligned bases); given row maxima give the computed result and each scene keeps its own global
maximum; dfeats is bitwise the single-scene op's and the weight gradients lie within the TF32-exact bound of
oracle/tf32.mask_head_backward at the batched call's reduction depth; the launch count does not grow with B; no
(B, Q, >1, N) temporary; FewShotForward's batched mask head equals its per-scene loop."""
import ctypes
import subprocess

import pytest
import torch

M = 16


# ---- inputs -------------------------------------------------------------------------------------------------------
def _batch(sizes, Q, seed, scale=3.0):
    """a ragged batch: maps (list of (Q, N_b)), flat feats and coords, stacked w0 (B*Q*16, 19), b0, w1 (B*Q, 16), b1,
    seeds (B, Q, 3), offsets; about 30 % of every map unreachable"""
    gen = torch.Generator().manual_seed(seed)
    B, n = len(sizes), sum(sizes)
    geo = []
    for N in sizes:
        g = torch.rand(Q, N, generator=gen) * scale
        g[torch.rand(Q, N, generator=gen) < 0.3] = -1.0
        geo.append(g)
    feats = torch.randn(n, M, generator=gen)
    w0 = torch.randn(B * Q * M, M + 3, generator=gen) * 0.3
    b0 = torch.randn(B * Q * M, generator=gen) * 0.1
    w1 = torch.randn(B * Q, M, generator=gen) * 0.3
    b1 = torch.randn(B * Q, generator=gen) * 0.1
    coords = (torch.rand(n, 3, generator=gen) - 0.5) * 8
    seeds = (torch.rand(B, Q, 3, generator=gen) - 0.5) * 8
    offsets = [0]
    for N in sizes:
        offsets.append(offsets[-1] + N)
    return geo, feats, w0, b0, w1, b1, coords, seeds, offsets


def _to(case, dev):
    geo, *rest, offsets = case
    return [[g.to(dev) for g in geo]] + [t.to(dev) for t in rest] + [offsets]


def _batch_call(geo, feats, w0, b0, w1, b1, coords, seeds, offsets, row_max=None):
    from geoformer_b200.mask_head import mask_heads_forward_batch

    return mask_heads_forward_batch(geo, feats, offsets, [w0[:, :, None], w1[:, :, None]], [b0, b1], coords, seeds,
                                    row_max=row_max)


def _scene_call(geo, feats, w0, b0, w1, b1, coords, seeds, offsets, b, row_max=None):
    """the single-scene op on scene b of the batch"""
    from geoformer_b200.mask_head import mask_heads_forward

    Q = seeds.shape[1]
    s, e, q = offsets[b], offsets[b + 1], slice(b * Q, (b + 1) * Q)
    qm = slice(b * Q * M, (b + 1) * Q * M)
    return mask_heads_forward(geo[b], feats[s:e], [w0[qm].reshape(Q * M, M + 3, 1), w1[q].reshape(Q, M, 1)],
                              [b0[qm], b1[q]], Q, coords[s:e], seeds[b], row_max=row_max)


def _bits(t):
    return t.contiguous().view(torch.int32)  # bitwise, NaN included


def _segments(sizes, sms):
    """the batched backward's partition (gf_mask_head.cu, mh_batch_plan): per scene its number of (CTA, scene)
    segments and the most tiles one of them sums"""
    tiles = [(n + 127) // 128 for n in sizes]
    T = sum(tiles)
    g = min(T, sms)
    start = lambda c: c * T // g  # noqa: E731
    owner = lambda t: ((t + 1) * g - 1) // T  # noqa: E731
    out, t0 = [], 0
    for nt in tiles:
        c0, c1 = owner(t0), owner(t0 + nt - 1)
        longest = max(min(start(c + 1), t0 + nt) - max(start(c), t0) for c in range(c0, c1 + 1))
        out.append((c1 - c0 + 1, longest))
        t0 += nt
    return out


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_segments_cover_every_tile_once():
    for sizes, sms in (([1, 127, 128, 129, 5000, 30_000, 100_003], 148), ([30_000] * 4, 148), ([1] * 32, 148),
                       ([100] * 3, 2), ([128 * 148 + 1], 148)):
        segs = _segments(sizes, sms)
        tiles = [(n + 127) // 128 for n in sizes]
        assert sum(s for s, _ in segs) <= min(sum(tiles), sms) + len(sizes) - 1
        for (ns, longest), nt in zip(segs, tiles):
            assert 1 <= longest <= nt and ns * longest >= nt


def test_batch_entries_validate_before_any_cuda_call(cuda_lib):
    L = cuda_lib
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below fails its checks first

    def offs(*v):
        return (ctypes.c_int * len(v))(*v)

    def maps(n, null=None):
        return (ctypes.c_void_p * n)(*[None if i == null else 256 for i in range(n)])

    good = offs(0, 5, 300)
    for q in (L.gf_mask_head_batch_workspace_bytes, L.gf_mask_head_batch_backward_workspace_bytes):
        assert q(good, 0, 4) == 0 and q(offs(*range(34)), 33, 4) == 0
        assert q(offs(1, 5, 300), 2, 4) == 0 and q(offs(0, 5, 5), 2, 4) == 0 and q(good, 2, 0) == 0
        assert q(None, 2, 4) == 0
    assert L.gf_mask_head_batch_workspace_bytes(good, 2, 4) >= (2 * 4 + 2) * 4
    assert L.gf_mask_head_batch_backward_workspace_bytes(good, 2, 4) >= 2 * 4 * 384 * 4  # >= one segment per scene

    p8 = [fake] * 8  # feats, w0, b0, w1, b1, coords, seed_xyz, row_max
    big = 1 << 30

    def fwd(geo, o, B, m=16, feats=fake, out=fake, ws=fake, nbytes=big):
        return L.gf_mask_head_logits_batch(geo, o, B, 4, m, feats, *p8[1:], out, ws, nbytes, None)

    def bwd(geo, o, B, m=16, feats=fake, dw1=fake, ws=fake, nbytes=big):
        return L.gf_mask_head_logits_batch_backward(geo, o, B, 4, m, feats, *p8[1:], fake, fake, fake, fake, dw1,
                                                    fake, ws, nbytes, None)

    for call in (fwd, bwd):
        assert call(maps(2), good, 0) == 1 and b"B=0" in L.gf_last_error()
        assert call(maps(33), offs(*range(34)), 33) == 1 and b"B=33" in L.gf_last_error()
        assert call(maps(2), offs(1, 5, 300), 2) == 1 and b"offsets[0]=1" in L.gf_last_error()
        assert call(maps(2), offs(0, 5, 5), 2) == 1 and b"scene 1 is empty" in L.gf_last_error()
        assert call(maps(2), good, 2, m=8) == 1 and b"m=8" in L.gf_last_error()
        assert call(None, good, 2) == 1 and b"null pointer" in L.gf_last_error()
        assert call(maps(2), None, 2) == 1 and b"null pointer" in L.gf_last_error()
        assert call(maps(2, null=1), good, 2) == 1 and b"geo[1]" in L.gf_last_error()
        assert call(maps(2), good, 2, feats=None) == 1 and b"null pointer" in L.gf_last_error()
        assert call(maps(2), good, 2, nbytes=16) == 3 and b"too small" in L.gf_last_error()
        assert call(maps(2), good, 2, ws=ctypes.c_void_p(260)) == 3 and b"aligned" in L.gf_last_error()
    assert fwd(maps(2), good, 2, out=None) == 1 and b"null pointer" in L.gf_last_error()
    assert bwd(maps(2), good, 2, dw1=None) == 1 and b"null pointer" in L.gf_last_error()


def test_batch_op_refuses_bad_input(cuda_lib):
    geo, feats, w0, b0, w1, b1, coords, seeds, offsets = _batch([5, 7], 3, 0)
    with pytest.raises(RuntimeError, match="CPU not supported"):
        _batch_call(geo, feats, w0, b0, w1, b1, coords, seeds, offsets)
    with pytest.raises(RuntimeError, match=r"geo_dists\[1\] must be"):
        _batch_call([geo[0], geo[1][:, :6]], feats, w0, b0, w1, b1, coords, seeds, offsets)
    with pytest.raises(RuntimeError, match="w0 must be"):
        _batch_call(geo, feats, w0[:-1], b0, w1, b1, coords, seeds, offsets)
    with pytest.raises(RuntimeError, match="fps_sampling_coords must be"):
        _batch_call(geo, feats, w0, b0, w1, b1, coords, seeds[:1], offsets)
    with pytest.raises(RuntimeError, match="mask_features must be"):
        _batch_call(geo, feats[:-1], w0, b0, w1, b1, coords, seeds, offsets)
    with pytest.raises(RuntimeError, match="empty"):
        _batch_call(geo, feats, w0, b0, w1, b1, coords, seeds, [0, 12, 12])
    with pytest.raises(RuntimeError, match="row_max must be"):
        _batch_call(geo, feats, w0, b0, w1, b1, coords, seeds, offsets, row_max=torch.zeros(3))
    for i in range(3):
        data = [[g.clone() for g in geo], coords.clone(), seeds.clone()]
        (data[0][1] if i == 0 else data[i]).requires_grad_()
        with pytest.raises(RuntimeError, match="they are data"):
            _batch_call(data[0], feats, w0, b0, w1, b1, data[1], data[2], offsets)


def test_batch_kernels_run_on_the_tensor_cores(cuda_lib):
    from geoformer_b200 import _capi

    tool = "cuobjdump" if subprocess.run(["which", "cuobjdump"], capture_output=True).returncode == 0 \
        else "/usr/local/cuda/bin/cuobjdump"
    sass = subprocess.run([tool, "-sass", _capi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    per_fn, cur = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            per_fn[cur] = 0
        elif cur and "UTCHMMA" in line:
            per_fn[cur] += 1
    k = {f: n for f, n in per_fn.items() if "mask_head_batch_kernel" in f}
    assert len(k) == 2 and all(n > 0 for n in k.values()), k


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev(cuda_lib):
    return torch.device("cuda:0")


SEVEN = [1, 127, 128, 129, 5000, 30_000, 100_003]
FORWARD_CASES = {  # name: (Q, scene sizes)
    "B1": (16, [5000]),
    "B2_Q1": (1, [1, 129]),
    "B7_Q17_tile_edges": (17, SEVEN),
    "B7_Q15": (15, SEVEN[::-1]),
    "B5_Q16": (16, [128, 1, 127, 30_000, 129]),
    "B4_Q128": (128, [30_000, 5000, 129, 30_000]),
    "B3_Q256": (256, [100_003, 1, 30_000]),
    "B32_Q17": (17, [int(v) for v in torch.randint(1, 4000, (32,), generator=torch.Generator().manual_seed(32))]),
    "B33_Q16": (16, [int(v) for v in torch.randint(1, 3000, (33,), generator=torch.Generator().manual_seed(33))]),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FORWARD_CASES))
def test_forward_bitwise_equals_single_scene_op(dev, name):
    Q, sizes = FORWARD_CASES[name]
    args = _to(_batch(sizes, Q, len(sizes) * 100 + Q), dev)
    with torch.no_grad():
        got = _batch_call(*args)
        assert len(got) == len(sizes)
        for b in range(len(sizes)):
            assert got[b].shape == (Q, sizes[b])
            assert torch.equal(_bits(got[b]), _bits(_scene_call(*args, b))), (name, b)


def _unaligned(t):
    """the same values at a base 4 bytes past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


@pytest.mark.gpu
def test_forward_unaligned_bases(dev):
    sizes, Q = [4099, 128, 4100], 17
    geo, *rest, offsets = _to(_batch(sizes, Q, 7), dev)
    ua = [[_unaligned(g) for g in geo]] + [_unaligned(t) for t in rest] + [offsets]
    with torch.no_grad():
        want = _batch_call(geo, *rest, offsets)
        got = _batch_call(*ua)
        for b in range(len(sizes)):
            assert torch.equal(_bits(got[b]), _bits(want[b])), b
            assert torch.equal(_bits(got[b]), _bits(_scene_call(*ua, b))), b


@pytest.mark.gpu
def test_row_max_given_is_bitwise_equal(dev):
    sizes, Q = [9001, 129, 30_000], 40
    geo, *rest, offsets = _to(_batch(sizes, Q, 9), dev)
    geo[0][3] = -1.0  # a row with nothing reachable takes its scene's maximum
    rm = torch.stack([g.max(dim=1)[0] for g in geo]).contiguous()
    with torch.no_grad():
        a = _batch_call(geo, *rest, offsets)
        c = _batch_call(geo, *rest, offsets, row_max=rm)
    for b in range(len(sizes)):
        assert torch.equal(_bits(a[b]), _bits(c[b])), b


@pytest.mark.gpu
def test_each_scene_keeps_its_own_global_maximum(dev):
    """scene 0: maxima about 3 and one unreachable row; scene 1: maxima about 1e4 and one unreachable row; scene 2:
    nothing reachable (NaN logits, as alone).  A maximum shared across scenes would move scene 0's unreachable row by
    sqrt(1e4) and make scene 2 finite."""
    sizes, Q = [5003, 4099, 700], 33
    geo, *rest, offsets = _to(_batch(sizes, Q, 13), dev)
    geo[0][5] = -1.0
    geo[1] = geo[1] * 1e4 / 3
    geo[1][geo[1] < 0] = -1.0
    geo[1][7] = -1.0
    geo[2][:] = -1.0
    with torch.no_grad():
        got = _batch_call(geo, *rest, offsets)
        for b in range(len(sizes)):
            alone = _scene_call(geo, *rest, offsets, b)
            assert torch.equal(_bits(got[b]), _bits(alone)), b
    assert torch.isnan(got[2]).all() and torch.isfinite(got[0]).all() and torch.isfinite(got[1]).all()


GNAMES = ("feats", "w0", "b0", "w1", "b1")


def _batch_grads(args, dls):
    geo, feats, w0, b0, w1, b1, coords, seeds, offsets = args
    leaves = [t.clone().requires_grad_() for t in (feats, w0, b0, w1, b1)]
    ys = _batch_call(geo, *leaves, coords, seeds, offsets)
    return dict(zip(GNAMES, torch.autograd.grad(ys, leaves, dls))), ys


@pytest.mark.gpu
@pytest.mark.parametrize("Q,sizes", [(17, [129, 5000, 1, 30_000, 4099, 128]), (128, [30_000, 30_000, 5000])])
def test_backward_against_single_scene_op_and_tf32_oracle(dev, Q, sizes):
    from oracle import tf32

    case = _batch(sizes, Q, Q + len(sizes))
    for g in case[0]:
        g[:, 0] = 0.5  # a reachable point in every row: no NaN scene here
    args = _to(case, dev)
    geo, feats, w0, b0, w1, b1, coords, seeds, offsets = args
    gen = torch.Generator().manual_seed(5)
    dls = [torch.randn(Q, n, generator=gen).to(dev) for n in sizes]
    # the upstream gradient zeroed where some hidden value lies within TF32 rounding of ReLU's kink (the oracle's rule)
    emu = []
    for b in range(len(sizes)):
        s, e, q, qm = offsets[b], offsets[b + 1], slice(b * Q, (b + 1) * Q), slice(b * Q * M, (b + 1) * Q * M)
        emu.append(tf32.mask_head_forward(geo[b], feats[s:e], w0[qm], b0[qm], w1[q], b1[q], coords[s:e], seeds[b]))
        dls[b] = torch.where(emu[b]["kink"], torch.zeros_like(dls[b]), dls[b])
    got, ys = _batch_grads(args, dls)
    again, ys2 = _batch_grads(args, dls)
    with torch.no_grad():
        ys0 = _batch_call(*args)
    for k in GNAMES:
        assert torch.equal(got[k], again[k]), k  # deterministic
    for b in range(len(sizes)):
        assert torch.equal(_bits(ys[b]), _bits(ys0[b])) and torch.equal(_bits(ys2[b]), _bits(ys0[b])), b
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    ratios = {k: 0.0 for k in GNAMES}
    for b, (nseg, longest) in enumerate(_segments(sizes, sms)):
        s, e, q, qm = offsets[b], offsets[b + 1], slice(b * Q, (b + 1) * Q), slice(b * Q * M, (b + 1) * Q * M)
        # dfeats: per point, in the fixed (q, j) order whatever the partition: bitwise the single-scene op's
        leaves = [t.clone().requires_grad_() for t in (feats[s:e], w0[qm], b0[qm], w1[q], b1[q])]
        y = _scene_one(geo[b], leaves, coords[s:e], seeds[b])
        alone = torch.autograd.grad(y, leaves, dls[b])
        assert torch.equal(got["feats"][s:e], alone[0]), b
        # the weight sums of the scene: its segments' tiles (at most `longest` each) then nseg segments in order;
        # n_ctas = nseg + longest makes the oracle's depth (ceil(tiles / n_ctas) + n_ctas) cover both
        want = tf32.mask_head_backward(emu[b], feats[s:e], w0[qm], w1[q], dls[b], nseg + longest)
        for k, g in (("feats", got["feats"][s:e]), ("w0", got["w0"][qm]), ("b0", got["b0"][qm]), ("w1", got["w1"][q]),
                     ("b1", got["b1"][q])):
            err = (g.double() - want[k]).abs()
            r = torch.where(err == 0, torch.zeros_like(err), err / want["e_" + k])
            ratios[k] = max(ratios[k], r.max().item())
    print("Q=%d sizes=%s |err| / bound %s" % (Q, sizes, " ".join("%s %.3g" % kv for kv in ratios.items())))
    assert max(ratios.values()) <= 0.5, ratios


def _scene_one(geo, leaves, coords, seeds):
    from geoformer_b200.mask_head import mask_heads_forward

    feats, w0, b0, w1, b1 = leaves
    Q = geo.shape[0]
    return mask_heads_forward(geo, feats, [w0.reshape(Q * M, M + 3, 1), w1.reshape(Q, M, 1)], [b0, b1], Q, coords,
                              seeds)


@pytest.mark.gpu
def test_launches_do_not_grow_with_the_batch(dev):
    from geoformer_b200 import _capi
    from geoformer_b200 import mask_head as mh

    counts = {}
    for B in (2, 8, 32):
        args = _to(_batch([3000 + 37 * b for b in range(B)], 16, B), dev)
        for rm in (False, True):
            extra = {"row_max": torch.stack([g.max(dim=1)[0] for g in args[0]])} if rm else {}
            with torch.no_grad():
                _batch_call(*args, **extra)  # first call: workspace allocation
                torch.cuda.synchronize()
                _capi.reset_launch_count()
                _batch_call(*args, **extra)
                fwd = _capi.launch_count()
            # the backward entry called on this thread (the launch counter is per thread; autograd's backward
            # runs on a thread of its own)
            geo, feats, w0, b0, w1, b1, coords, seeds, offsets = args
            dl = torch.ones(16 * offsets[-1], device=dev)
            grads = [torch.empty_like(t) for t in (feats, w0, b0, w1, b1)]
            torch.cuda.synchronize()
            _capi.reset_launch_count()
            mh._launch_batch(geo, offsets, feats, w0, b0, w1, b1, coords, seeds, extra.get("row_max"), dlogit=dl,
                             grads=grads)
            counts[(B, rm)] = (fwd, _capi.launch_count())
    print(counts)
    for rm in (False, True):
        assert counts[(2, rm)] == counts[(8, rm)] == counts[(32, rm)], counts
    assert counts[(2, False)] == (3, 4) and counts[(2, True)] == (2, 3), counts


@pytest.mark.gpu
def test_no_large_temporaries(dev):
    sizes, Q = [60_000, 45_000, 30_001, 50_000], 128
    args = _to(_batch(sizes, Q, 4), dev)
    with torch.no_grad():
        _batch_call(*args)  # workspace allocated once
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base = torch.cuda.memory_allocated(dev)
        out = _batch_call(*args)
        torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    logits = sum(o.numel() for o in out) * 4
    print("peak increase %.1f MB (logits %.1f MB)" % (peak / 2**20, logits / 2**20))
    assert peak < 1.5 * logits


def _per_scene_batch(geo_dists, mask_features, batch_offsets, weights, biases, coords, fps_sampling_coords,
                     row_max=None):
    """mask_heads_forward_batch as the per-scene loop FewShotForward.mask_logits ran before it"""
    from geoformer_b200.mask_head import mask_heads_forward

    B, Q = fps_sampling_coords.shape[:2]
    (w0, w1), (b0, b1) = weights, biases
    out = []
    for b, (s, e) in enumerate(zip(batch_offsets, batch_offsets[1:])):
        q, qm = slice(b * Q, (b + 1) * Q), slice(b * Q * M, (b + 1) * Q * M)
        out.append(mask_heads_forward(geo_dists[b], mask_features[s:e], [w0[qm], w1[q]], [b0[qm], b1[q]], Q,
                                      coords[s:e].contiguous(), fps_sampling_coords[b].contiguous()))
    return out


@pytest.mark.gpu
def test_few_shot_forward_ragged_batch(dev, monkeypatch):
    from geoformer_b200 import mask_head as mh
    from geoformer_b200.harness import FewShotForward
    from geoformer_b200.scenes import scene

    torch.manual_seed(11)
    sizes = [20_000, 7001, 12_345]
    net = FewShotForward(m=16, nlayers=2, n_decode_point=512, n_query_points=64).to(dev)
    locs = torch.cat([scene(n, 70 + b, L=(4.0, 3.0, 2.0), nbox=6) for b, n in enumerate(sizes)]).to(dev)
    feats = torch.randn(sum(sizes), 16, device=dev)
    support = torch.randn(len(sizes), 32, device=dev)
    off = [0, sizes[0], sizes[0] + sizes[1], sum(sizes)]
    kw = dict(max_step=48, neighbor=16, geo_radius=0.2, batch_offsets=off)
    la, ga, _ = net(locs, feats, support, impl="b200", **kw)
    lt, _, _ = net(locs, feats, support, impl="torch", **kw)
    monkeypatch.setattr(mh, "mask_heads_forward_batch", _per_scene_batch)
    ll, gl, _ = net(locs, feats, support, impl="b200", **kw)
    for b, n in enumerate(sizes):
        assert torch.equal(ga[b], gl[b]) and la[b].shape == (64, n)
        assert torch.equal(_bits(la[b]), _bits(ll[b])), b
        scale = lt[b].abs().max().item()
        err = (la[b] - lt[b]).abs().max().item()
        assert err <= 0.02 * scale + 1e-6, (b, err, scale)


@pytest.mark.gpu
def test_forward_train_batched_equals_per_scene_path(dev, monkeypatch):
    """one forward_train step at B = 2: the logits are bitwise those of the per-scene path, so every ReLU mask is the
    same; the gradients differ only in how the mask head's weight sums are grouped over the points (fp32 rounding,
    checked against the TF32-exact bound in the backward test above).  Carried back through the controller and the
    decoder, where random loss weights make the sums cancel, that rounding reached 7.5e-5 of the scale below (measured
    on a B200); the limit is 1e-3 of the larger of that norm and 1e-2 of the largest one, so that a
    gradient that is zero up to rounding (a bias in front of a batch-statistics batch norm) is held to the scale of
    the others."""
    from geoformer_b200 import mask_head as mh
    from geoformer_b200.harness import FewShotForward
    from geoformer_b200.scenes import scene

    torch.manual_seed(5)
    B, N = 2, 12_000
    net = FewShotForward(m=16, nlayers=2, n_decode_point=256, n_query_points=128).to(dev)
    net.train()
    locs = torch.stack([scene(N, 40 + b, L=(4.0, 3.0, 2.0), nbox=6) for b in range(B)]).to(dev)
    feats = torch.randn(B, N, 16, device=dev)
    support = torch.randn(B, 32, device=dev)
    wl = torch.randn(B, 128, N, device=dev)
    params = [p for p in net.parameters() if p.requires_grad]
    grads, logits = {}, {}
    for path in ("batch", "loop"):
        if path == "loop":
            monkeypatch.setattr(mh, "mask_heads_forward_batch", _per_scene_batch)
        torch.manual_seed(6)
        lg, _, _ = net.forward_train(locs, feats, support, impl="b200", max_step=48, neighbor=16, geo_radius=0.2)
        loss = sum((l * w).sum() for l, w in zip(lg, wl))
        grads[path] = torch.autograd.grad(loss, params, allow_unused=True)
        logits[path] = [l.detach() for l in lg]
    for b in range(B):
        assert torch.equal(_bits(logits["batch"][b]), _bits(logits["loop"][b])), b
    big = max(c.norm().item() for c in grads["loop"] if c is not None)
    checked, worst = 0, 0.0
    for i, (a, c) in enumerate(zip(grads["batch"], grads["loop"])):
        if a is None or c is None:
            assert a is None and c is None, i
            continue
        checked += 1
        err = ((a - c).norm() / max(c.norm().item(), 1e-2 * big)).item()
        worst = max(worst, err)
        assert err <= 1e-3, (i, err, c.norm().item(), big)
    print("%d parameter gradients, worst scaled Frobenius difference %.2e" % (checked, worst))
    assert checked > 10
