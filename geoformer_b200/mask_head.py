"""The mask head of GeoFormerFS (model/geoformer/geoformer_fs.py:263-300, mask_heads_forward) as one tcgen05 kernel.

The reference builds the relative coordinates (Q,3,N), repeats the mask features to (Q,m,N), concatenates them to
(Q,m+3,N) and runs two grouped conv1d (about 7 GB of temporaries at Q = 256, N = 100k).  Here the maps are read once
and the (Q,N) logits written once: the feature part of the first dynamic conv runs on the tensor cores (TF32, fp32
accumulation, as the reference's cuDNN conv runs in TF32 by default), the relative coordinates (epilogue a11, the
same code as bias.mask_head_relative_coords) and the second layer in fp32.  Only m = 16.

It is an autograd op: gradients flow to the mask features and the dynamic weights and biases (into the controller
and the decoder).  The maps, coordinates and row maxima are data; asking for their gradient raises.  The backward
recomputes the hidden layer with the forward's products and sums in a fixed order: deterministic gradients.
"""
import torch

from . import _capi as C

M = 16


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
