"""ctypes binding of libgeoformer_b200.so (include/geoformer_b200.h).

This is the only place the shared library is loaded.  There is NO fallback: if the library is
missing or a tensor is not on a CUDA device the call raises RuntimeError (the reference raises
through AT_ASSERT "CPU not supported", sampling.cpp:35-37).
"""
import ctypes
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# GF_LIB: development builds of the same library (python -m geoformer_b200.build --variant=trace -DGF_TRACE)
LIB_PATH = os.environ.get("GF_LIB") or os.path.join(_HERE, "libgeoformer_b200.so")

_lib = None
_lock = threading.Lock()

c_int, c_float, c_size_t, c_void_p, c_int64 = ctypes.c_int, ctypes.c_float, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_int64

# name -> (restype, argtypes); mirrors include/geoformer_b200.h one to one
_P = c_void_p
SIGNATURES = {
    "gf_last_error": (ctypes.c_char_p, []),
    "gf_version": (c_int, []),
    "gf_launch_count": (c_int64, []),
    "gf_reset_launch_count": (None, []),
    "gf_set_stage_events": (c_int, [_P, c_int]),
    "gf_event_create": (c_void_p, []),
    "gf_event_destroy": (None, [_P]),
    "gf_event_elapsed_ms": (c_float, [_P, _P]),
    "gf_fps_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gf_furthest_point_sampling": (c_int, [_P, c_int, c_int, c_int, _P, _P, c_size_t, _P]),
    "gf_fps_batch_workspace_bytes": (c_size_t, [_P, c_int, c_int]),
    "gf_furthest_point_sampling_batch": (c_int, [_P, _P, c_int, c_int, _P, _P, c_size_t, _P]),
    "gf_gather_points": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "gf_gather_points_grad": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "gf_ball_query": (c_int, [_P, _P, c_int, c_int, c_int, c_float, c_int, _P, _P]),
    "gf_ball_query_batch": (c_int, [_P, _P, _P, c_int, c_int, c_float, c_int, _P, _P]),
    "gf_group_points": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "gf_group_points_grad": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "gf_three_nn": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P]),
    "gf_three_interpolate": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "gf_three_interpolate_grad": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "gf_knn_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "gf_knn": (c_int, [_P, c_int, _P, c_int, c_int, c_int, _P, _P, _P, c_int, _P, c_size_t, _P]),
    "gf_knn_batch_workspace_bytes": (c_size_t, [_P, c_int]),
    "gf_knn_batch": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "gf_geodesic_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gf_geodesic": (c_int, [_P, _P, c_int, c_int, c_int, _P, c_int, c_float, c_int, _P, _P, _P, _P, c_size_t, _P]),
    "gf_geodesic_batch_workspace_bytes": (c_size_t, [_P, c_int, c_int, c_int]),
    "gf_geodesic_batch": (c_int, [_P, _P, _P, c_int, _P, c_int, c_int, _P, c_int, c_float, c_int, _P, _P, _P, _P,
                                  c_size_t, _P]),
    "gf_bias_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gf_bias_decoder": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, _P, _P, c_size_t, _P]),
    "gf_bias_decoder_fourier": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, _P, c_int, c_int, _P, _P, _P, _P,
                                        c_size_t, _P]),
    "gf_bias_mask_head": (c_int, [_P, _P, _P, c_int, c_int, _P, _P, _P, c_size_t, _P]),
    "gf_rel_cross_attention_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gf_rel_cross_attention": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gf_rel_cross_attention_fused": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, c_int, c_int, c_int,
                                             _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gf_rel_cross_attention_save": (c_int, [_P, _P, _P, c_int, c_int, c_int] + [_P] * 12 + [c_size_t, _P]),
    "gf_rel_cross_attention_fused_save": (c_int, [_P] * 8 + [c_int, _P, _P, c_int, c_int, c_int] + [_P] * 12
                                          + [c_size_t, _P]),
    "gf_rel_cross_attention_backward_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gf_rel_cross_attention_backward": (c_int, [_P, _P, _P, c_int, c_int, c_int] + [_P] * 24 + [c_size_t, _P]),
    "gf_rel_cross_attention_fused_backward": (c_int, [_P] * 8 + [c_int, _P, _P, c_int, c_int, c_int] + [_P] * 23
                                              + [c_size_t, _P]),
    "gf_mask_head_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gf_mask_head_logits": (c_int, [_P] * 9 + [c_int, c_int, c_int, _P, _P, c_size_t, _P]),
    "gf_mask_head_backward_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gf_mask_head_logits_backward": (c_int, [_P] * 9 + [c_int, c_int, c_int] + [_P] * 7 + [c_size_t, _P]),
    "gf_mask_head_batch_workspace_bytes": (c_size_t, [_P, c_int, c_int]),
    "gf_mask_head_logits_batch": (c_int, [_P, _P, c_int, c_int, c_int] + [_P] * 9 + [_P, c_size_t, _P]),
    "gf_mask_head_batch_backward_workspace_bytes": (c_size_t, [_P, c_int, c_int]),
    "gf_mask_head_logits_batch_backward": (c_int, [_P, _P, c_int, c_int, c_int] + [_P] * 14 + [_P, c_size_t, _P]),
    "gf_group_mlp_pool": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_int, _P, _P,
                                  _P, _P, c_int, _P, _P]),
    "gf_group_mlp_pool_train_workspace_bytes": (c_size_t, [c_int, c_int]),
    "gf_group_mlp_pool_train": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int, c_int,
                                        _P, _P, _P, _P, _P, _P, _P, c_int, _P, _P, c_size_t, _P]),
    "gf_group_mlp_pool_backward_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "gf_group_mlp_pool_backward": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_int,
                                           c_int, _P, _P, _P, _P, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gf_guidance_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gf_guidance": (c_int, [_P, c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gf_guidance_seeded": (c_int, [_P, c_int, _P, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gf_guidance_batch_workspace_bytes": (c_size_t, [_P, c_int, c_int, c_int]),
    "gf_guidance_batch": (c_int, [_P, _P, c_int, c_int, c_int, c_float, c_int, _P, c_int, _P, _P, _P, _P, c_size_t, _P]),
    "gf_guidance_shard": (c_int, [_P, c_int, c_int, c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P, _P, c_size_t, _P]),
    "gf_geodesic_scatter": (c_int, [_P, _P, c_int, c_int, c_int, _P, c_int, c_float, c_int, _P, _P, c_int, _P, _P,
                                    c_size_t, _P]),
    "gf_guidance_seeded_scatter": (c_int, [_P, c_int, _P, c_int, c_int, c_float, c_int, _P, _P, c_int, _P, _P,
                                           c_size_t, _P]),
    "gf_peer_alloc": (c_int, [_P, c_size_t]),
    "gf_peer_free": (c_int, [_P]),
    "gf_peer_export": (c_int, [_P, _P]),
    "gf_peer_open": (c_int, [_P, _P]),
    "gf_peer_close": (c_int, [_P]),
    "gf_guidance_batch_host_workspace_bytes": (c_size_t, [_P, c_int, c_int, c_int]),
    "gf_guidance_batch_host": (c_int, [_P, _P, c_int, c_int, c_int, c_float, c_int, _P, _P, _P, c_size_t, _P]),
    "gf_guidance_host_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "gf_guidance_host": (c_int, [_P, c_int, c_int, c_int, c_float, c_int, _P, _P, _P, c_size_t, _P]),
}


def lib():
    """Load the CUDA library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "geoformer_b200: %s is missing; build it with `python -m geoformer_b200.build` "
                        "(there is no CPU or PyTorch fallback)" % LIB_PATH)
                h = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(h, name)  # AttributeError = header / library mismatch
                    fn.restype = res
                    fn.argtypes = args
                _lib = h
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().gf_last_error()
        raise RuntimeError("%s failed (status %d): %s" % (what, rc, msg.decode() if msg else "?"))


def launch_count():
    return int(lib().gf_launch_count())


def reset_launch_count():
    lib().gf_reset_launch_count()


# ---- tensor plumbing ------------------------------------------------------------------------------
def ptr(t):
    # plain ints / None convert to void* through the declared argtypes; no ctypes object per argument
    return t.data_ptr() if t is not None else None


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_of(device):
    """the current CUDA stream of `device` as a raw cudaStream_t value"""
    if _raw_stream is not None:
        return _raw_stream(device.index if device.index is not None else torch.cuda.current_device())
    return torch.cuda.current_stream(device).cuda_stream


def require(cond, msg):
    # the reference's AT_ASSERT surfaces in Python as RuntimeError (utils.h:8-28)
    if not cond:
        raise RuntimeError(msg)


def check_cuda_f32(x, name):
    require(isinstance(x, torch.Tensor), "%s must be a tensor" % name)
    require(x.is_cuda, "%s: CPU not supported (must be a CUDA tensor)" % name)
    require(x.is_contiguous(), "%s must be a contiguous tensor" % name)
    require(x.dtype == torch.float32, "%s must be a float tensor" % name)


def check_cuda_i32(x, name):
    require(isinstance(x, torch.Tensor), "%s must be a tensor" % name)
    require(x.is_cuda, "%s: CPU not supported (must be a CUDA tensor)" % name)
    require(x.is_contiguous(), "%s must be a contiguous tensor" % name)
    require(x.dtype == torch.int32, "%s must be an int tensor" % name)


class Workspace:
    """Grow-only scratch buffers, one per (device, tag, CUDA stream, host thread): two streams or two threads that
    call the same operator never share scratch (the whole-GPU FPS keeps polled tag slots there, the propagation its
    claim arrays).  A buffer that is outgrown is kept alive (kernels launched earlier may still be using it)."""

    def __init__(self):
        self._bufs = {}
        self._retired = []
        self._lock = threading.Lock()

    def get(self, device, tag, nbytes):
        nbytes = int(nbytes)
        dev = device.index if device.index is not None else torch.cuda.current_device()
        key = (dev, tag, stream_of(device), threading.get_ident())
        with self._lock:
            buf = self._bufs.get(key)
            if buf is None or buf.numel() < nbytes:
                if buf is not None:
                    self._retired.append(buf)
                buf = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=device)
                self._bufs[key] = buf
            return buf


workspace = Workspace()
