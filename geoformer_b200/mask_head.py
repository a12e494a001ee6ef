"""The mask head of GeoFormerFS (model/geoformer/geoformer_fs.py:263-300, mask_heads_forward) as one tcgen05 kernel.

The reference builds the relative coordinates (Q,3,N), repeats the mask features to (Q,m,N), concatenates them to
(Q,m+3,N) and runs two grouped conv1d (about 7 GB of temporaries at Q = 256, N = 100k).  Here the maps are read once
and the (Q,N) logits written once: the feature part of the first dynamic conv runs on the tensor cores (TF32, fp32
accumulation, as the reference's cuDNN conv runs in TF32 by default), the relative coordinates (epilogue a11, the
same code as bias.mask_head_relative_coords) and the second layer in fp32.  Only m = 16.

It is an autograd op: gradients flow to the mask features and the dynamic weights and biases (into the controller
and the decoder).  The maps, coordinates and row maxima are data; asking for their gradient raises.  The backward
recomputes the hidden layer with the forward's products and sums in a fixed order: deterministic gradients.

mask_heads_forward_batch takes a ragged batch as the model holds it (flat points and offsets, stacked dynamic
weights) and computes every scene's logits in one launch, each bitwise what mask_heads_forward gives on the scene.
"""
import ctypes

import torch

from . import _capi as C
from .aggregate import batch_offsets_list

M = 16
BATCH_MAX = 32  # scenes per C call (gf_mask_head_logits_batch); larger batches go through consecutive calls


def _launch_forward(geo, feats, w0, b0, w1, b1, coords, seeds, row_max, out):
    Q, N = geo.shape
    dev = geo.device
    L = C.lib()
    with torch.cuda.device(dev):
        nbytes = L.gf_mask_head_workspace_bytes(Q, N)
        ws = C.workspace.get(dev, "mask_head", nbytes)
        C.check(L.gf_mask_head_logits(C.ptr(geo), C.ptr(feats), C.ptr(w0), C.ptr(b0), C.ptr(w1), C.ptr(b1),
                                      C.ptr(coords), C.ptr(seeds), C.ptr(row_max), Q, N, M, C.ptr(out), C.ptr(ws),
                                      nbytes, C.stream_of(dev)), "mask_head")
    return out


class _MaskHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, w0, b0, w1, b1, data):
        geo, coords, seeds, row_max = data
        out = torch.empty(geo.shape, dtype=torch.float32, device=geo.device)
        _launch_forward(geo, feats, w0, b0, w1, b1, coords, seeds, row_max, out)
        ctx.save_for_backward(feats, w0, b0, w1, b1)
        ctx.data = data
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dlogit):
        feats, w0, b0, w1, b1 = ctx.saved_tensors
        geo, coords, seeds, row_max = ctx.data
        Q, N = geo.shape
        dev = geo.device
        dlogit = dlogit.to(torch.float32).contiguous()
        grads = [torch.empty_like(t) for t in (feats, w0, b0, w1, b1)]
        L = C.lib()
        with torch.cuda.device(dev):
            nbytes = L.gf_mask_head_backward_workspace_bytes(Q, N)
            ws = C.workspace.get(dev, "mask_head_backward", nbytes)
            C.check(L.gf_mask_head_logits_backward(C.ptr(geo), C.ptr(feats), C.ptr(w0), C.ptr(b0), C.ptr(w1),
                                                   C.ptr(b1), C.ptr(coords), C.ptr(seeds), C.ptr(row_max), Q, N, M,
                                                   C.ptr(dlogit), *[C.ptr(g) for g in grads], C.ptr(ws), nbytes,
                                                   C.stream_of(dev)), "mask_head_backward")
        return tuple(grads) + (None,)


def mask_heads_forward(geo_dist, mask_features, weights, biases, num_insts, coords, fps_sampling_coords, row_max=None):
    """The reference method's arguments minus `self`, for one scene:
    geo_dist (Q,N) f32 maps, mask_features (N,m) or (N,m,1), weights = [w0 (Q*m, m+3, 1), w1 (Q, m, 1)],
    biases = [b0 (Q*m), b1 (Q)], num_insts = Q, coords (N,3), fps_sampling_coords (Q,3); row_max: optional (Q,) row
    maxima of the maps as the propagation produces them (bias.mask_head_relative_coords takes them too).
    Returns the (Q,N) mask logits.  m = 16 only."""
    C.check_cuda_f32(geo_dist, "geo_dist")
    C.check_cuda_f32(coords, "coords")
    C.check_cuda_f32(fps_sampling_coords, "fps_sampling_coords")
    C.require(geo_dist.dim() == 2, "geo_dist must be (Q, N)")
    Q, N = geo_dist.shape
    C.require(int(num_insts) == Q, "num_insts must equal geo_dist.shape[0]")
    C.require(tuple(coords.shape) == (N, 3) and tuple(fps_sampling_coords.shape) == (Q, 3), "shape mismatch")
    if row_max is not None:
        C.check_cuda_f32(row_max, "row_max")
        C.require(tuple(row_max.shape) == (Q,), "row_max must be (Q,)")
    C.require(len(weights) == 2 and len(biases) == 2, "weights and biases must be two tensors each")
    feats = mask_features
    C.require(isinstance(feats, torch.Tensor) and feats.is_cuda and feats.dtype == torch.float32
              and feats.device == geo_dist.device, "mask_features must be a float CUDA tensor on the maps' device")
    if feats.dim() == 3:
        C.require(feats.size(2) == 1, "mask_features must be (N, m) or (N, m, 1)")
        feats = feats.squeeze(2)
    C.require(feats.dim() == 2 and feats.size(0) == N, "mask_features must be (N, m)")
    m = feats.size(1)
    if m != M:
        raise RuntimeError("mask_heads_forward: m=%d, only m = 16 is supported" % m)
    w0, w1 = weights
    b0, b1 = biases
    for t, name in ((w0, "w0"), (w1, "w1"), (b0, "b0"), (b1, "b1")):
        C.require(isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.device == geo_dist.device,
                  "%s must be a float CUDA tensor on the maps' device" % name)
    C.require(w0.numel() == Q * M * (M + 3) and w0.size(0) == Q * M, "w0 must be (Q*m, m+3, 1)")
    C.require(w1.numel() == Q * M and w1.size(0) == Q, "w1 must be (Q, m, 1)")
    C.require(b0.numel() == Q * M and b1.numel() == Q, "b0 must be (Q*m) and b1 (Q)")
    data = [t for t in (geo_dist, coords, fps_sampling_coords, row_max) if t is not None]
    if torch.is_grad_enabled() and any(t.requires_grad for t in data):
        raise RuntimeError("mask_heads_forward: no gradient for geo_dist, coords, fps_sampling_coords or row_max "
                           "(they are data)")
    dev = geo_dist.device
    if Q == 0 or N == 0:
        out = torch.empty((Q, N), dtype=torch.float32, device=dev)
        params = (mask_features, w0, w1, b0, b1)
        if torch.is_grad_enabled() and any(t.requires_grad for t in params):  # keep the graph: zero gradients
            out = out + sum(t.sum() * 0 for t in params)
        return out
    shaped = [w0.reshape(Q * M, M + 3), b0.reshape(Q * M), w1.reshape(Q, M), b1.reshape(Q)]
    if torch.is_grad_enabled() and any(t.requires_grad for t in (feats, w0, b0, w1, b1)):
        args = [feats.contiguous()] + [t.contiguous() for t in shaped]
        out = _MaskHead.apply(*args, (geo_dist, coords, fps_sampling_coords, row_max))
        return out
    out = torch.empty((Q, N), dtype=torch.float32, device=dev)
    return _launch_forward(geo_dist, feats.detach().contiguous(), *[t.detach().contiguous() for t in shaped], coords,
                           fps_sampling_coords, row_max, out)


def _at(t, elems):
    """the device address `elems` floats into t, or None"""
    return t.data_ptr() + 4 * elems if t is not None else None


def _launch_batch(geo, offsets, feats, w0, b0, w1, b1, coords, seeds, row_max, out=None, dlogit=None, grads=None):
    """the forward (out) or the backward (dlogit, grads = dfeats, dw0, db0, dw1, db1) over every scene, in calls of
    at most BATCH_MAX scenes whose pointers start at their first scene"""
    Q = seeds.shape[1]
    dev = feats.device
    L = C.lib()
    with torch.cuda.device(dev):
        for s in range(0, len(geo), BATCH_MAX):
            e = min(s + BATCH_MAX, len(geo))
            n, p0, q0 = e - s, offsets[s], s * Q
            offs = (ctypes.c_int * (n + 1))(*[o - p0 for o in offsets[s:e + 1]])
            maps = (ctypes.c_void_p * n)(*[g.data_ptr() for g in geo[s:e]])
            args = [maps, offs, n, Q, M, _at(feats, p0 * M), _at(w0, q0 * M * (M + 3)), _at(b0, q0 * M),
                    _at(w1, q0 * M), _at(b1, q0), _at(coords, p0 * 3), _at(seeds, q0 * 3), _at(row_max, q0)]
            if grads is None:
                nbytes = L.gf_mask_head_batch_workspace_bytes(offs, n, Q)
                ws = C.workspace.get(dev, "mask_head_batch", nbytes)
                C.check(L.gf_mask_head_logits_batch(*args, _at(out, Q * p0), C.ptr(ws), nbytes, C.stream_of(dev)),
                        "mask_head_batch")
            else:
                dfeats, dw0, db0, dw1, db1 = grads
                nbytes = L.gf_mask_head_batch_backward_workspace_bytes(offs, n, Q)
                ws = C.workspace.get(dev, "mask_head_batch_backward", nbytes)
                C.check(L.gf_mask_head_logits_batch_backward(
                    *args, _at(dlogit, Q * p0), _at(dfeats, p0 * M), _at(dw0, q0 * M * (M + 3)), _at(db0, q0 * M),
                    _at(dw1, q0 * M), _at(db1, q0), C.ptr(ws), nbytes, C.stream_of(dev)), "mask_head_batch_backward")


def _split(flat, offsets, Q):
    """scene b's (Q, N_b) block of the flat logits, as a view"""
    return [flat[Q * a:Q * b].view(Q, b - a) for a, b in zip(offsets, offsets[1:])]


class _MaskHeadBatch(torch.autograd.Function):
    @staticmethod
    def forward(ctx, feats, w0, b0, w1, b1, data):
        geo, offsets, coords, seeds, row_max = data
        Q = seeds.shape[1]
        out = torch.empty(Q * offsets[-1], dtype=torch.float32, device=feats.device)
        _launch_batch(geo, offsets, feats, w0, b0, w1, b1, coords, seeds, row_max, out=out)
        ctx.save_for_backward(feats, w0, b0, w1, b1)
        ctx.data = data
        return tuple(_split(out, offsets, Q))

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *dlogits):
        feats, w0, b0, w1, b1 = ctx.saved_tensors
        geo, offsets, coords, seeds, row_max = ctx.data
        dlogit = torch.cat([(g if g is not None else torch.zeros_like(m)).to(torch.float32).reshape(-1)
                            for g, m in zip(dlogits, geo)])
        grads = [torch.empty_like(t) for t in (feats, w0, b0, w1, b1)]
        _launch_batch(geo, offsets, feats, w0, b0, w1, b1, coords, seeds, row_max, dlogit=dlogit, grads=grads)
        return tuple(grads) + (None,)


def mask_heads_forward_batch(geo_dists, mask_features, batch_offsets, weights, biases, coords, fps_sampling_coords,
                             row_max=None):
    """mask_heads_forward over a ragged batch of B scenes with Q queries each, in one launch per 32 scenes:
    geo_dists B maps (Q, N_b) f32, mask_features (sum N, m) or (sum N, m, 1) flat, batch_offsets (B+1) tensor or
    sequence from 0 rising strictly, weights = [w0 (B*Q*m, m+3, 1), w1 (B*Q, m, 1)] and biases = [b0 (B*Q*m),
    b1 (B*Q)] stacked scene after scene (the controllers' split of the whole batch), coords (sum N, 3),
    fps_sampling_coords (B, Q, 3); row_max: optional (B, Q) row maxima of the maps.
    Returns B (Q, N_b) logits, views of one buffer, each bitwise mask_heads_forward of its scene.  m = 16 only."""
    tensors = [coords, fps_sampling_coords, mask_features] + list(weights) + list(biases)
    C.require(all(isinstance(t, torch.Tensor) for t in tensors), "every argument but batch_offsets must be a tensor")
    offsets = batch_offsets_list(batch_offsets, coords.shape[0])
    B = len(offsets) - 1
    sizes = [b - a for a, b in zip(offsets, offsets[1:])]
    C.require(coords.dim() == 2 and coords.size(1) == 3, "coords must be (sum N, 3)")
    C.require(fps_sampling_coords.dim() == 3 and fps_sampling_coords.shape[0] == B and fps_sampling_coords.shape[2] == 3,
              "fps_sampling_coords must be (B, Q, 3)")
    Q = fps_sampling_coords.shape[1]
    geo = list(geo_dists)
    C.require(len(geo) == B, "geo_dists must hold one map per scene (%d), not %d" % (B, len(geo)))
    for b, g in enumerate(geo):
        C.require(isinstance(g, torch.Tensor) and tuple(g.shape) == (Q, sizes[b]),
                  "geo_dists[%d] must be (Q, N_b) = (%d, %d)" % (b, Q, sizes[b]))
    C.require(row_max is None or tuple(row_max.shape) == (B, Q), "row_max must be (B, Q)")
    C.require(len(weights) == 2 and len(biases) == 2, "weights and biases must be two tensors each")
    feats = mask_features
    if feats.dim() == 3:
        C.require(feats.size(2) == 1, "mask_features must be (sum N, m) or (sum N, m, 1)")
        feats = feats.squeeze(2)
    C.require(feats.dim() == 2 and feats.size(0) == offsets[-1], "mask_features must be (sum N, m)")
    if feats.size(1) != M:
        raise RuntimeError("mask_heads_forward_batch: m=%d, only m = 16 is supported" % feats.size(1))
    w0, w1 = weights
    b0, b1 = biases
    BQ = B * Q
    C.require(w0.numel() == BQ * M * (M + 3) and w0.size(0) == BQ * M, "w0 must be (B*Q*m, m+3, 1)")
    C.require(w1.numel() == BQ * M and w1.size(0) == BQ, "w1 must be (B*Q, m, 1)")
    C.require(b0.numel() == BQ * M and b1.numel() == BQ, "b0 must be (B*Q*m) and b1 (B*Q)")
    data = [t for t in geo + [coords, fps_sampling_coords, row_max] if t is not None]
    if torch.is_grad_enabled() and any(t.requires_grad for t in data):
        raise RuntimeError("mask_heads_forward_batch: no gradient for geo_dists, coords, fps_sampling_coords or "
                           "row_max (they are data)")
    dev = coords.device
    for t, name in [(coords, "coords"), (fps_sampling_coords, "fps_sampling_coords"), (row_max, "row_max")] + \
            [(g, "geo_dists[%d]" % b) for b, g in enumerate(geo)]:
        if t is not None:
            C.check_cuda_f32(t, name)
            C.require(t.device == dev, "%s must be on the coordinates' device" % name)
    for t, name in ((feats, "mask_features"), (w0, "w0"), (w1, "w1"), (b0, "b0"), (b1, "b1")):
        C.require(t.is_cuda and t.dtype == torch.float32 and t.device == dev,
                  "%s must be a float CUDA tensor on the coordinates' device" % name)
    params = (mask_features, w0, w1, b0, b1)
    grad = torch.is_grad_enabled() and any(t.requires_grad for t in params)
    if Q == 0:
        out = _split(torch.empty(0, dtype=torch.float32, device=dev), offsets, 0)
        if grad:  # keep the graph: zero gradients
            out = [o + sum(t.sum() * 0 for t in params) for o in out]
        return out
    shaped = [w0.reshape(BQ * M, M + 3), b0.reshape(BQ * M), w1.reshape(BQ, M), b1.reshape(BQ)]
    data = (geo, offsets, coords, fps_sampling_coords, row_max)
    if grad:
        return list(_MaskHeadBatch.apply(feats.contiguous(), *[t.contiguous() for t in shaped], data))
    out = torch.empty(Q * offsets[-1], dtype=torch.float32, device=dev)
    _launch_batch(geo, offsets, feats.detach().contiguous(), *[t.detach().contiguous() for t in shaped], coords,
                  fps_sampling_coords, row_max, out=out)
    return _split(out, offsets, Q)
