"""Every entry that takes a workspace, at shapes that reach each branch of its layout, called through the package's
own wrappers with the workspace swapped at the library boundary:
- exact: the reported size, carved from a larger buffer whose tail holds a canary.  The outputs equal those of an
  ordinary call and the canary is untouched.
- too small: the reported size minus 256.  The entry returns GF_ERR_WORKSPACE and has launched nothing.
- misaligned: the base 16 bytes past a 256-byte boundary.  The entry returns GF_ERR_WORKSPACE.  The kernels need at
  most 16-byte alignment, so a build that failed to reject this base would still run correctly instead of faulting."""
import ctypes
import contextlib

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GF_ERR_WORKSPACE = 3
CANARY = 0xA5
TAIL = 1 << 16


@pytest.fixture(scope="module")
def dev(cuda_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


class _Swap:
    """The library, with the workspace of every call to `entry` replaced by place(reported bytes) -> (pointer,
    bytes).  Records the status of each such call and the kernels it launched."""

    def __init__(self, real, entry, place):
        self._real, self._entry, self._place = real, entry, place
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(self._real, name)
        if name != self._entry:
            return fn

        def call(*args):
            args = list(args)
            args[-3], args[-2] = self._place(int(args[-2]))  # every entry ends with (workspace, bytes, stream)
            before = self._real.gf_launch_count()
            rc = fn(*args)
            self.calls.append((rc, self._real.gf_launch_count() - before))
            return rc

        return call


@contextlib.contextmanager
def _swapped(entry, place):
    from geoformer_b200 import _capi as C

    real = C.lib()
    sw = _Swap(real, entry, place)
    C._lib = sw
    try:
        yield sw
    finally:
        C._lib = real


def _flat(out):
    if isinstance(out, torch.Tensor):
        return [out]
    return [t for o in out if o is not None for t in _flat(o)]


def _check_layout(dev, entry, run):
    """run() calls the wrappers and returns its outputs (copies of any buffer a later call would overwrite)"""
    want = [t.clone() for t in _flat(run())]
    torch.cuda.synchronize()

    bufs = []

    def buffer(n):
        b = torch.full((n + TAIL,), CANARY, dtype=torch.uint8, device=dev)
        assert b.data_ptr() % 256 == 0
        bufs.append((b, n))
        return b

    def exact(n):
        return buffer(n).data_ptr(), n

    def too_small(n):
        assert n >= 256, "%s: reported %d bytes" % (entry, n)
        return buffer(n).data_ptr(), n - 256

    def misaligned(n):
        return buffer(n).data_ptr() + 16, n

    with _swapped(entry, exact) as sw:
        got = _flat(run())
    torch.cuda.synchronize()
    assert sw.calls and all(rc == 0 for rc, _ in sw.calls), (entry, sw.calls)
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert torch.equal(g, w), (entry, i)
    for b, n in bufs:
        assert bool((b[n:] == CANARY).all()), "%s wrote past its %d-byte workspace" % (entry, n)

    for place, says in ((too_small, "too small"), (misaligned, "256-byte aligned")):
        with _swapped(entry, place) as sw:
            with pytest.raises(RuntimeError, match=says):
                run()
        torch.cuda.synchronize()
        assert sw.calls == [(GF_ERR_WORKSPACE, 0)], (entry, place.__name__, sw.calls)


# ---- the point operators and the hot path ---------------------------------------------------------------------------
def _scene(N, seed, dev):
    from geoformer_b200.scenes import scene

    return scene(N, seed).to(dev)


def test_fps_whole_gpu(dev):
    """a scene above the cluster capacity: the whole-GPU kernel's exchange slots and running minima"""
    from geoformer_b200.pointnet2._ext import furthest_point_sampling

    x = _scene(250_000, 3, dev)[None].contiguous()
    _check_layout(dev, "gf_furthest_point_sampling", lambda: furthest_point_sampling(x, 64))


def test_fps_ragged_batch_with_a_scene_above_the_cluster_capacity(dev):
    from geoformer_b200.aggregate import furthest_point_sampling_batch

    Ns = [3000, 250_000, 5000]
    x = torch.cat([_scene(n, 10 + i, dev) for i, n in enumerate(Ns)]).contiguous()
    offsets = np.concatenate([[0], np.cumsum(Ns)]).tolist()
    _check_layout(dev, "gf_furthest_point_sampling_batch", lambda: furthest_point_sampling_batch(x, offsets, 64))


def test_knn(dev):
    from geoformer_b200.geodesic_utils import knn_graph

    x = _scene(30_000, 4, dev)
    _check_layout(dev, "gf_knn", lambda: knn_graph(x, 16, index_dtype=torch.int32))


def test_knn_batch(dev):
    from geoformer_b200 import _capi as C

    xs = [_scene(n, 20 + i, dev) for i, n in enumerate([5000, 37, 20_000])]
    B, k = len(xs), 16
    Ns = (ctypes.c_int * B)(*[x.shape[0] for x in xs])

    def run():
        L = C.lib()
        D = [torch.empty((x.shape[0], k), dtype=torch.float32, device=dev) for x in xs]
        I = [torch.empty((x.shape[0], k), dtype=torch.int32, device=dev) for x in xs]
        nbytes = L.gf_knn_batch_workspace_bytes(Ns, B)
        ws = C.workspace.get(dev, "knn_batch", nbytes)
        arr = lambda ts: (ctypes.c_void_p * B)(*[t.data_ptr() for t in ts])  # noqa: E731
        C.check(L.gf_knn_batch(arr(xs), Ns, B, k, 1, arr(D), arr(I), C.ptr(ws), nbytes, C.stream_of(dev)), "knn_batch")
        return D + I

    _check_layout(dev, "gf_knn_batch", run)


def test_geodesic(dev):
    from geoformer_b200.geodesic_utils import geodesic_from_graph, knn_graph

    x = _scene(20_000, 5, dev)
    D, I = knn_graph(x, 16, index_dtype=torch.int32)
    seeds = torch.arange(0, 20_000, 625, dtype=torch.int32, device=dev)
    _check_layout(dev, "gf_geodesic", lambda: geodesic_from_graph(D, I, seeds, 0.5, 16, return_stats=True))


def test_guidance(dev):
    from geoformer_b200.guidance import geodesic_guidance

    x = _scene(20_000, 6, dev)
    _check_layout(dev, "gf_guidance",
                  lambda: geodesic_guidance(x, 64, 16, 0.5, 16, return_graph=True, return_stats=True))


@pytest.mark.parametrize("B", [3, 6])
def test_guidance_batch(dev, B):
    """B <= 4: a lane per scene and the cluster FPS; B > 4: the batched graphs and the culled FPS"""
    from geoformer_b200.guidance import geodesic_guidance_batch

    xs = [_scene(8000 + 1000 * b, 30 + b, dev) for b in range(B)]
    _check_layout(dev, "gf_guidance_batch",
                  lambda: geodesic_guidance_batch(xs, 64, 16, 0.5, 16, return_stats=True, row_max=True))


def test_guidance_host(dev):
    from geoformer_b200 import guidance

    x = _scene(20_000, 7, dev).cpu().contiguous()
    _check_layout(dev, "gf_guidance_host",
                  lambda: guidance.HostGuidance(20_000, 64, 16, 0.5, 16, device=dev, pinned=False).run(x))


def test_guidance_batch_host(dev):
    from geoformer_b200 import guidance

    xs = [_scene(10_000, 40 + b, dev).cpu().contiguous() for b in range(3)]
    _check_layout(dev, "gf_guidance_batch_host",
                  lambda: guidance.HostBatchGuidance(10_000, 3, 64, 16, 0.5, 16, device=dev, pinned=False).run(xs))


# ---- the epilogues, the cross-attention, the mask head -------------------------------------------------------------
def _decoder_case(dev, Q=64, Cn=512, B=2):
    gen = torch.Generator().manual_seed(11)
    Ns = [3000 + 500 * b for b in range(B)]
    xs = [_scene(n, 80 + b, dev).cpu() for b, n in enumerate(Ns)]
    geos = []
    for n in Ns:
        g = torch.rand(Q, n, generator=gen) * 4.0
        g[torch.rand(Q, n, generator=gen) < 0.5] = -1.0
        geos.append(g.to(dev))
    inds = torch.stack([torch.randperm(n, generator=gen)[:Cn] for n in Ns]).int()
    ctx = torch.stack([x[i.long()] for x, i in zip(xs, inds)]).contiguous()
    qry = ctx[:, :Q].contiguous()
    gb = torch.randn(3, 32, generator=gen)
    pc = [torch.stack([x.min(0)[0] for x in xs]).to(dev), torch.stack([x.max(0)[0] for x in xs]).to(dev)]
    return [geos, inds.to(dev), qry.to(dev), ctx.to(dev), gb.to(dev), pc]


def test_bias_decoder(dev):
    from geoformer_b200.bias import decoder_relative_pos

    geos, inds, qry, ctx, _, _ = _decoder_case(dev)
    _check_layout(dev, "gf_bias_decoder", lambda: decoder_relative_pos(geos, inds, qry, ctx))


def test_bias_decoder_fourier(dev):
    from geoformer_b200.bias import decoder_relative_embedding

    geos, inds, qry, ctx, gb, pc = _decoder_case(dev)
    _check_layout(dev, "gf_bias_decoder_fourier", lambda: decoder_relative_embedding(geos, inds, qry, ctx, gb, pc))


def test_bias_mask_head(dev):
    from geoformer_b200.bias import mask_head_relative_coords

    geos, _, qry, _, _, _ = _decoder_case(dev)
    x = _scene(3000, 80, dev)
    _check_layout(dev, "gf_bias_mask_head", lambda: mask_head_relative_coords(geos[0], x, qry[0]))


def _attention_inputs(dev, Q=64, Cn=512, B=2):
    gen = torch.Generator().manual_seed(12)
    w = {}
    for k in ("w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo"):
        w[k] = (torch.randn((64, 64) if k[0] == "w" else (64,), generator=gen) * 0.125).to(dev)
    tgt2 = torch.randn(Q, B, 64, generator=gen).to(dev)
    mem = torch.randn(Cn, B, 64, generator=gen).to(dev)
    rel = torch.randn(Q, Cn, B, 64, generator=gen).to(dev)
    return tgt2, mem, rel, w


@pytest.mark.parametrize("fused", [False, True])
def test_attention_forward(dev, fused):
    from geoformer_b200.attention import rel_cross_attention, rel_cross_attention_fused

    tgt2, mem, rel, w = _attention_inputs(dev)
    case = _decoder_case(dev)
    with torch.no_grad():
        if fused:
            _check_layout(dev, "gf_rel_cross_attention_fused", lambda: rel_cross_attention_fused(tgt2, mem, *case, w))
        else:
            _check_layout(dev, "gf_rel_cross_attention", lambda: rel_cross_attention(tgt2, mem, rel, w))


@pytest.mark.parametrize("fused", [False, True])
def test_attention_backward(dev, fused):
    """the saving forward and the backward"""
    from geoformer_b200.attention import rel_cross_attention, rel_cross_attention_fused

    tgt2, mem, rel, w = _attention_inputs(dev)
    case = _decoder_case(dev)
    dy = torch.randn(tgt2.shape, generator=torch.Generator().manual_seed(13)).to(dev)

    def run():
        leaves = [t.detach().requires_grad_(True) for t in (tgt2, mem)]
        wl = {k: v.detach().requires_grad_(True) for k, v in w.items()}
        if fused:
            y = rel_cross_attention_fused(*leaves, *case, wl)
        else:
            y = rel_cross_attention(*leaves, rel, wl)
        y.backward(dy)
        return [y.detach()] + [t.grad for t in leaves] + [wl[k].grad for k in sorted(wl)]

    name = "gf_rel_cross_attention_fused" if fused else "gf_rel_cross_attention"
    _check_layout(dev, name + "_save", run)
    _check_layout(dev, name + "_backward", run)


def _mask_head_inputs(dev, Q=32, N=20_000):
    gen = torch.Generator().manual_seed(14)
    M = 16
    geo = torch.rand(Q, N, generator=gen) * 3.0
    geo[torch.rand(Q, N, generator=gen) < 0.3] = -1.0
    x = _scene(N, 90, dev)
    seeds = x[torch.randperm(N, generator=gen)[:Q].to(dev)].contiguous()
    feats = torch.randn(N, M, generator=gen)
    w0 = torch.randn(Q * M, M + 3, generator=gen) * 0.3
    b0 = torch.randn(Q * M, generator=gen) * 0.1
    w1 = torch.randn(Q, M, generator=gen) * 0.3
    b1 = torch.randn(Q, generator=gen) * 0.1
    return geo.to(dev), x, seeds, [t.to(dev) for t in (feats, w0, b0, w1, b1)]


def _mask_logits(geo, x, seeds, feats, w0, b0, w1, b1):
    from geoformer_b200.mask_head import mask_heads_forward

    Q, M = w1.shape
    return mask_heads_forward(geo, feats, [w0.reshape(Q * M, M + 3, 1), w1.reshape(Q, M, 1)], [b0, b1], Q, x, seeds)


def test_mask_head_forward(dev):
    geo, x, seeds, p = _mask_head_inputs(dev)
    with torch.no_grad():
        _check_layout(dev, "gf_mask_head_logits", lambda: _mask_logits(geo, x, seeds, *p))


def test_mask_head_backward(dev):
    geo, x, seeds, p = _mask_head_inputs(dev)
    dl = torch.randn(geo.shape, generator=torch.Generator().manual_seed(15)).to(dev)

    def run():
        leaves = [t.detach().requires_grad_(True) for t in p]
        _mask_logits(geo, x, seeds, *leaves).backward(dl)
        return [t.grad for t in leaves]

    _check_layout(dev, "gf_mask_head_logits_backward", run)


# ---- the aggregator's training forward and backward -----------------------------------------------------------------
def _aggregator_inputs(dev, B=2, N=4000, m=64, ns=16, Cn=13):
    gen = torch.Generator().manual_seed(16)
    xyz = torch.rand(B, N, 3, generator=gen).to(dev)
    new_xyz = xyz[:, :m].contiguous()
    idx = torch.randint(0, N, (B, m, ns), generator=gen, dtype=torch.int32).to(dev)
    feats = torch.randn(B, Cn, N, generator=gen).to(dev)
    widths = [3 + Cn, 32, 32]
    Ws = [(torch.randn(widths[l + 1], widths[l], generator=gen) * 0.3).to(dev) for l in range(2)]
    gammas = [(1.0 + 0.1 * torch.randn(w, generator=gen)).to(dev) for w in widths[1:]]
    betas = [(0.1 * torch.randn(w, generator=gen)).to(dev) for w in widths[1:]]
    dout = torch.randn(B, widths[-1], m, generator=gen).to(dev)
    return xyz, new_xyz, idx, feats, Ws, gammas, betas, dout


def test_aggregator_train(dev):
    from geoformer_b200.aggregate import group_mlp_pool_train

    xyz, new_xyz, idx, feats, Ws, gammas, betas, _ = _aggregator_inputs(dev)
    with torch.no_grad():
        _check_layout(dev, "gf_group_mlp_pool_train",
                      lambda: group_mlp_pool_train(xyz, new_xyz, feats, idx, 0.3, False, True, Ws, gammas=gammas,
                                                   betas=betas))


@pytest.mark.parametrize("dfeatures", [False, True])
def test_aggregator_backward(dev, dfeatures):
    from geoformer_b200.aggregate import group_mlp_pool_train

    xyz, new_xyz, idx, feats, Ws, gammas, betas, dout = _aggregator_inputs(dev)

    def run():
        f = feats.detach().requires_grad_(dfeatures)
        leaves = [t.detach().requires_grad_(True) for t in Ws + gammas + betas]
        y = group_mlp_pool_train(xyz, new_xyz, f, idx, 0.3, False, True, leaves[:2], gammas=leaves[2:4],
                                 betas=leaves[4:])
        y.backward(dout)
        return [t.grad for t in leaves] + ([f.grad] if dfeatures else [])

    _check_layout(dev, "gf_group_mlp_pool_backward", run)
