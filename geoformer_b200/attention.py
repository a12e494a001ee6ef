"""The decoder's vector cross-attention over the geodesic relative-position embedding
(model/transformer_detr.py:443-454 with the MLPs of :384-396) as one tcgen05 kernel per call.

rel_cross_attention        : takes the embedding tensor (Q,C,B,64) the reference passes as `relative_pos`
rel_cross_attention_fused  : takes the geodesic maps instead and builds the embedding on the fly (decoder epilogue
                             a10 + Fourier features, geoformer_fs.py:680-712), so the (Q,C,B,64) tensor never exists
Both return out_mlp(sum_c softmax_c(attn_mlp(tgt2 - memory + rel) / 8) * v_mlp(memory + rel)), shape (Q,B,64):
what TransformerDecoderLayer.forward_pre_rel assigns to `tgt` at :453, before the residual of :456.
Products run on the tensor cores in TF32 with fp32 accumulation (the reference is plain fp32): agreement is 2e-3
of the output scale (tests/test_gpu_attention.py), not bit-exact.

Both are autograd ops.  Under grad mode, when an input requires grad, the forward also saves o and lse (Q,B,64) and
the backward kernel recomputes the scores tile by tile: gradients flow to tgt2, memory, the eight weights (through
layer_weights, into the layer's parameters) and, unfused, relative_pos.  The fused variant's embedding ingredients
are data (gauss_B is a buffer in the reference); asking for their gradient raises.  Otherwise the inference entry
runs unchanged.
"""
import ctypes

import torch

from . import _capi as C


def layer_weights(layer):
    """the eight tensors of a reference TransformerDecoderLayer(use_rel=True) this path uses"""
    return {"w1": layer.attn_mlp[0].weight, "b1": layer.attn_mlp[0].bias, "w2": layer.attn_mlp[2].weight,
            "b2": layer.attn_mlp[2].bias, "wv": layer.v_mlp[0].weight, "bv": layer.v_mlp[0].bias,
            "wo": layer.out_mlp[0].weight, "bo": layer.out_mlp[0].bias}


_WNAMES = ("w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo")


def _weights(w, dev):
    """the eight weights as f32 contiguous tensors on `dev`; differentiable, so that gradients reach w's tensors"""
    out = {}
    for k in _WNAMES:
        t = w[k].to(device=dev, dtype=torch.float32).contiguous()
        C.require(tuple(t.shape) == ((64, 64) if k[0] == "w" else (64,)), "%s must be %s" % (k, "(64, 64)" if k[0] == "w" else "(64,)"))
        out[k] = t
    return out


def _common(tgt2, memory):
    C.check_cuda_f32(tgt2, "tgt2")
    C.check_cuda_f32(memory, "memory")
    C.require(tgt2.dim() == 3 and memory.dim() == 3 and tgt2.size(2) == 64 and memory.size(2) == 64 and
              tgt2.size(1) == memory.size(1), "tgt2 must be (Q, B, 64) and memory (C, B, 64)")
    return tgt2.size(0), memory.size(0), tgt2.size(1)


def _wants_grad(*tensors):
    return torch.is_grad_enabled() and any(t.requires_grad for t in tensors)


def _grads_out(dev, Q, Cn, B):
    """gradient buffers: dtgt2, dmemory and one per weight"""
    z = lambda *shape: torch.empty(shape, dtype=torch.float32, device=dev)  # noqa: E731
    return z(Q, B, 64), z(Cn, B, 64), {k: z(64, 64) if k[0] == "w" else z(64) for k in _WNAMES}


def _wptrs(w):
    """the eight weights (or their gradients) in the order of the C entries"""
    return [C.ptr(w[k]) for k in _WNAMES]


def _save_buffers(Q, B, dev):
    return [torch.empty((Q, B, 64), dtype=torch.float32, device=dev) for _ in range(3)]  # out, o, lse


class _RelCrossAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tgt2, memory, relative_pos, *wts):
        Q, Cn, B = tgt2.size(0), memory.size(0), tgt2.size(1)
        dev = tgt2.device
        out, o, lse = _save_buffers(Q, B, dev)
        L = C.lib()
        with torch.cuda.device(dev):
            nbytes = L.gf_rel_cross_attention_workspace_bytes(Q, Cn, B)
            ws = C.workspace.get(dev, "attention", nbytes)
            C.check(L.gf_rel_cross_attention_save(C.ptr(tgt2), C.ptr(memory), C.ptr(relative_pos), Q, Cn, B,
                                                  *[C.ptr(t) for t in wts], C.ptr(out), C.ptr(o), C.ptr(lse),
                                                  C.ptr(ws), nbytes, C.stream_of(dev)), "rel_cross_attention")
        ctx.save_for_backward(tgt2, memory, relative_pos, out, o, lse, *wts)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        tgt2, memory, rel, out, o, lse, *wts = ctx.saved_tensors
        w = dict(zip(_WNAMES, wts))
        Q, Cn, B = tgt2.size(0), memory.size(0), tgt2.size(1)
        dev = tgt2.device
        dy = dy.to(torch.float32).contiguous()
        dt, dm, g = _grads_out(dev, Q, Cn, B)
        drel = torch.empty_like(rel) if ctx.needs_input_grad[2] else None
        L = C.lib()
        with torch.cuda.device(dev):
            nbytes = L.gf_rel_cross_attention_backward_workspace_bytes(Q, Cn, B)
            ws = C.workspace.get(dev, "attention_backward", nbytes)
            C.check(L.gf_rel_cross_attention_backward(C.ptr(tgt2), C.ptr(memory), C.ptr(rel), Q, Cn, B, *_wptrs(w),
                                                      C.ptr(out), C.ptr(o), C.ptr(lse), C.ptr(dy), C.ptr(dt),
                                                      C.ptr(dm), C.ptr(drel), *_wptrs(g), C.ptr(ws), nbytes,
                                                      C.stream_of(dev)), "rel_cross_attention_backward")
        return (dt, dm, drel) + tuple(g[k] for k in _WNAMES)


class _RelCrossAttentionFused(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tgt2, memory, emb_args, *wts):
        ptrs, lds, inds, qry, cl, gb, pc_min, pc_max, keep = emb_args
        Q, Cn, B = tgt2.size(0), memory.size(0), tgt2.size(1)
        dev = tgt2.device
        out, o, lse = _save_buffers(Q, B, dev)
        L = C.lib()
        with torch.cuda.device(dev):
            nbytes = L.gf_rel_cross_attention_workspace_bytes(Q, Cn, B)
            ws = C.workspace.get(dev, "attention", nbytes)
            C.check(L.gf_rel_cross_attention_fused_save(C.ptr(tgt2), C.ptr(memory), ptrs, lds, C.ptr(inds), C.ptr(qry),
                                                        C.ptr(cl), C.ptr(gb), gb.stride(0), C.ptr(pc_min),
                                                        C.ptr(pc_max), Q, Cn, B, *[C.ptr(t) for t in wts], C.ptr(out),
                                                        C.ptr(o), C.ptr(lse), C.ptr(ws), nbytes, C.stream_of(dev)),
                    "rel_cross_attention_fused")
        ctx.save_for_backward(tgt2, memory, out, o, lse, *wts)
        ctx.emb_args = emb_args  # the geodesic maps and the pointer table that refers to them stay alive with ctx
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dy):
        tgt2, memory, out, o, lse, *wts = ctx.saved_tensors
        ptrs, lds, inds, qry, cl, gb, pc_min, pc_max, keep = ctx.emb_args
        w = dict(zip(_WNAMES, wts))
        Q, Cn, B = tgt2.size(0), memory.size(0), tgt2.size(1)
        dev = tgt2.device
        dy = dy.to(torch.float32).contiguous()
        dt, dm, g = _grads_out(dev, Q, Cn, B)
        L = C.lib()
        with torch.cuda.device(dev):
            nbytes = L.gf_rel_cross_attention_backward_workspace_bytes(Q, Cn, B)
            ws = C.workspace.get(dev, "attention_backward", nbytes)
            C.check(L.gf_rel_cross_attention_fused_backward(C.ptr(tgt2), C.ptr(memory), ptrs, lds, C.ptr(inds),
                                                            C.ptr(qry), C.ptr(cl), C.ptr(gb), gb.stride(0),
                                                            C.ptr(pc_min), C.ptr(pc_max), Q, Cn, B, *_wptrs(w),
                                                            C.ptr(out), C.ptr(o), C.ptr(lse), C.ptr(dy), C.ptr(dt),
                                                            C.ptr(dm), *_wptrs(g), C.ptr(ws), nbytes,
                                                            C.stream_of(dev)), "rel_cross_attention_fused_backward")
        return (dt, dm, None) + tuple(g[k] for k in _WNAMES)


def rel_cross_attention(tgt2, memory, relative_pos, weights):
    """tgt2 (Q,B,64) f32 CUDA (= norm2(tgt)), memory (C,B,64), relative_pos (Q,C,B,64) contiguous -> (Q,B,64)"""
    Q, Cn, B = _common(tgt2, memory)
    C.check_cuda_f32(relative_pos, "relative_pos")
    C.require(tuple(relative_pos.shape) == (Q, Cn, B, 64), "relative_pos must be (Q, C, B, 64)")
    dev = tgt2.device
    w = _weights(weights, dev)
    if _wants_grad(tgt2, memory, relative_pos, *w.values()):
        return _RelCrossAttention.apply(tgt2, memory, relative_pos, *[w[k] for k in _WNAMES])
    out = torch.empty((Q, B, 64), dtype=torch.float32, device=dev)
    L = C.lib()
    with torch.cuda.device(dev):
        nbytes = L.gf_rel_cross_attention_workspace_bytes(Q, Cn, B)
        ws = C.workspace.get(dev, "attention", nbytes)
        C.check(L.gf_rel_cross_attention(C.ptr(tgt2), C.ptr(memory), C.ptr(relative_pos), Q, Cn, B, C.ptr(w["w1"]),
                                         C.ptr(w["b1"]), C.ptr(w["w2"]), C.ptr(w["b2"]), C.ptr(w["wv"]), C.ptr(w["bv"]),
                                         C.ptr(w["wo"]), C.ptr(w["bo"]), C.ptr(out), C.ptr(ws), nbytes,
                                         C.stream_of(dev)), "rel_cross_attention")
    return out


def rel_cross_attention_fused(tgt2, memory, geo_dists, pre_enc_inds, query_locs, context_locs, gauss_B, pc_dims, weights):
    """The same with the embedding built on the fly: geo_dists list of B (Q,N_b) maps, pre_enc_inds (B,C) i32,
    query_locs (B,Q,3), context_locs (B,C,3), gauss_B (3, >= 32), pc_dims = [pc_min (B,3), pc_max (B,3)]
    (the arguments of bias.decoder_relative_embedding) -> (Q,B,64).  Differentiable with respect to tgt2, memory and
    the weights; the embedding's ingredients are data and must not require grad."""
    Q, Cn, B = _common(tgt2, memory)
    dev = tgt2.device
    C.check_cuda_i32(pre_enc_inds, "pre_enc_inds")
    C.check_cuda_f32(query_locs, "query_locs")
    C.check_cuda_f32(context_locs, "context_locs")
    C.check_cuda_f32(gauss_B, "gauss_B")
    C.require(len(geo_dists) == B and tuple(pre_enc_inds.shape) == (B, Cn) and tuple(query_locs.shape) == (B, Q, 3)
              and tuple(context_locs.shape) == (B, Cn, 3), "batch / query / context mismatch")
    C.require(gauss_B.dim() == 2 and gauss_B.size(0) == 3 and gauss_B.size(1) >= 32, "gauss_B must be (3, >= 32)")
    for g in geo_dists:
        C.check_cuda_f32(g, "geo_dists[b]")
        C.require(g.size(0) == Q, "geo_dists[b] must have Q rows")
    pc_min, pc_max = [t.to(device=dev, dtype=torch.float32).contiguous() for t in pc_dims]
    C.require(tuple(pc_min.shape) == (B, 3) and tuple(pc_max.shape) == (B, 3), "pc_dims must be two (B, 3) tensors")
    w = _weights(weights, dev)
    ptrs = (ctypes.c_void_p * B)(*[g.data_ptr() for g in geo_dists])
    lds = (ctypes.c_int * B)(*[g.stride(0) for g in geo_dists])
    data = list(geo_dists) + [query_locs, context_locs, gauss_B] + list(pc_dims)
    C.require(not _wants_grad(*[t for t in data if isinstance(t, torch.Tensor)]),
              "rel_cross_attention_fused: no gradient for geo_dists, the locations, gauss_B or pc_dims (they are "
              "data); build the embedding with bias.decoder_relative_embedding and use rel_cross_attention")
    if _wants_grad(tgt2, memory, *w.values()):
        emb_args = (ptrs, lds, pre_enc_inds, query_locs, context_locs, gauss_B, pc_min, pc_max, list(geo_dists))
        return _RelCrossAttentionFused.apply(tgt2, memory, emb_args, *[w[k] for k in _WNAMES])
    out = torch.empty((Q, B, 64), dtype=torch.float32, device=dev)
    L = C.lib()
    with torch.cuda.device(dev):
        nbytes = L.gf_rel_cross_attention_workspace_bytes(Q, Cn, B)
        ws = C.workspace.get(dev, "attention", nbytes)
        C.check(L.gf_rel_cross_attention_fused(C.ptr(tgt2), C.ptr(memory), ptrs, lds, C.ptr(pre_enc_inds),
                                               C.ptr(query_locs), C.ptr(context_locs), C.ptr(gauss_B), gauss_B.stride(0),
                                               C.ptr(pc_min), C.ptr(pc_max), Q, Cn, B, C.ptr(w["w1"]), C.ptr(w["b1"]),
                                               C.ptr(w["w2"]), C.ptr(w["b2"]), C.ptr(w["wv"]), C.ptr(w["bv"]),
                                               C.ptr(w["wo"]), C.ptr(w["bo"]), C.ptr(out), C.ptr(ws), nbytes,
                                               C.stream_of(dev)), "rel_cross_attention_fused")
    return out
