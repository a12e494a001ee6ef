"""Drop-in for model/geoformer/geodesic_utils.py (find_knn, cal_geodesic_vectorize,
unique_with_inds) plus the index object that stands where faiss.GpuIndexFlatL2 stood
(geoformer_fs.py:170-175).  All arithmetic runs in the sm_100a library; there is no torch
fallback path for the propagation.
"""
import ctypes

import torch

from . import _capi as C
from .guidance import BATCH_MAX, BATCH_MAX_POINTS, _ptr_array, geodesic_guidance_batch


class FlatL2Index:
    """Exact L2 index over 3-D points with the faiss protocol used by the reference
    (geodesic_utils.py:18-21): add(x) / search(x, k, D_out, I_out) / reset().
    search() writes SQUARED distances (float32) and int64 indices into the pre-allocated
    tensors, ordered by (distance, index); missing neighbours are (-1, +inf)."""

    def __init__(self, algo="grid"):
        self.algo = {"grid": 0, "brute": 1}[algo]
        self._x = None
        self._src = None

    @property
    def ntotal(self):
        return 0 if self._x is None else self._x.shape[0]

    def add(self, x):
        C.check_cuda_f32(x, "x")
        C.require(x.dim() == 2 and x.size(1) == 3, "x must be (N, 3)")
        # faiss copies what it is given: later changes of the caller's tensor must not change the index
        self._x = x.detach().clone() if self._x is None else torch.cat([self._x, x]).contiguous()
        self._src = (x.data_ptr(), tuple(x.shape)) if self.ntotal == x.size(0) else None

    def reset(self):
        self._x = None
        self._src = None

    def search(self, q, k, D_out, I_out):
        C.require(self._x is not None, "search on an empty index")
        C.check_cuda_f32(q, "q")
        C.check_cuda_f32(D_out, "D_out")
        C.require(I_out.is_cuda and I_out.is_contiguous() and I_out.dtype == torch.int64, "I_out must be int64 CUDA")
        nq = q.size(0)
        C.require(tuple(D_out.shape) == (nq, k) and tuple(I_out.shape) == (nq, k), "output shape must be (nq, k)")
        x = self._x
        # the reference searches a scene against itself right after adding it (geodesic_utils.py:18-19): then the
        # self-query path (no second copy of the points) applies
        same = self._src == (q.data_ptr(), tuple(q.shape))
        _knn_into(x, None if same else q, int(k), False, D_out, I_out, None, self.algo)
        return D_out, I_out


def _knn_into(x, queries, k, sqrt_out, dist, idx64, idx32, algo):
    L = C.lib()
    N = x.size(0)
    nq = N if queries is None else queries.size(0)
    with torch.cuda.device(x.device):
        nbytes = L.gf_knn_workspace_bytes(N, nq, k, algo)
        ws = C.workspace.get(x.device, "knn", nbytes) if nbytes else None
        C.check(L.gf_knn(C.ptr(x), N, C.ptr(queries), nq, k, 1 if sqrt_out else 0, C.ptr(dist), C.ptr(idx64),
                         C.ptr(idx32), algo, C.ptr(ws), nbytes, C.stream_of(x.device)), "knn")


def knn_graph(locs, neighbor, algo="grid", index_dtype=torch.int64):
    """kNN of a scene against itself: (sqrt distances (N,k) f32, indices (N,k) int64 or int32)."""
    C.check_cuda_f32(locs, "locs")
    N = locs.size(0)
    D = torch.empty((N, neighbor), dtype=torch.float32, device=locs.device)
    I = torch.empty((N, neighbor), dtype=index_dtype, device=locs.device)
    a = {"grid": 0, "brute": 1}[algo]
    if index_dtype == torch.int64:
        _knn_into(locs, None, int(neighbor), True, D, I, None, a)
    else:
        _knn_into(locs, None, int(neighbor), True, D, None, I, a)
    return D, I


@torch.no_grad()
def find_knn(gpu_index, locs, neighbor=32):
    """geodesic_utils.py:11-24: (sqrt distances (N,k) f32, indices (N,k) i64) through the index
    protocol.  With our own FlatL2Index the sqrt is fused into the search kernel."""
    if isinstance(gpu_index, FlatL2Index) or gpu_index is None:
        # the reference adds the scene, searches it against itself and resets the index (:18-21): points added
        # earlier would take part in the search, so an index that is not empty is an error here, not ignored
        C.require(gpu_index is None or gpu_index.ntotal == 0,
                  "find_knn: the index already holds %d points (the reference resets it after every call)"
                  % (0 if gpu_index is None else gpu_index.ntotal))
        algo = "grid" if gpu_index is None or gpu_index.algo == 0 else "brute"
        return knn_graph(locs.contiguous(), neighbor, algo=algo)
    n_points = locs.shape[0]
    D = torch.zeros(n_points, neighbor, device=locs.device, dtype=torch.float32)
    I = torch.zeros(n_points, neighbor, device=locs.device, dtype=torch.int64)
    gpu_index.add(locs)
    gpu_index.search(locs, neighbor, D, I)
    gpu_index.reset()
    return torch.sqrt(D), I


def unique_with_inds(x, dim=-1):
    """geodesic_utils.py:4-8: unique slices along `dim` and, for each, the index of its FIRST
    occurrence.  The reference relies on scatter_ with duplicate indices (last write wins), which is
    only deterministic on CPU; this version is deterministic on CUDA too (amin reduction).  It is
    not used by our propagation kernel -- kept because it is part of the module's surface."""
    unique, inverse = torch.unique(x, return_inverse=True, dim=dim)
    perm = torch.arange(inverse.size(0), dtype=inverse.dtype, device=inverse.device)
    first = torch.full((unique.size(dim),), inverse.size(0), dtype=inverse.dtype, device=inverse.device)
    first.scatter_reduce_(0, inverse, perm, reduce="amin", include_self=True)
    return unique, first


def geodesic_from_graph(D, I, seeds, radius, max_step, return_stats=False, row_max=None):
    """Propagation only (geodesic_utils.py:109-163) on a given kNN graph: D (N,k) sqrt'ed f32,
    I (N,k) int64/int32, seeds (Q,) int32/int64 -> (Q,N) f32, -1 = unreachable."""
    C.check_cuda_f32(D, "D")
    C.require(I.is_cuda and I.is_contiguous() and I.dtype in (torch.int64, torch.int32), "I must be int64/int32 CUDA")
    N, k = D.shape
    seeds = seeds.to(device=D.device, dtype=torch.int32).contiguous()
    Q = seeds.numel()
    geo = torch.empty((Q, N), dtype=torch.float32, device=D.device)
    stats = torch.zeros(2, dtype=torch.int64, device=D.device) if return_stats else None
    L = C.lib()
    with torch.cuda.device(D.device):
        nbytes = L.gf_geodesic_workspace_bytes(N, k, Q)
        ws = C.workspace.get(D.device, "geodesic", nbytes) if nbytes else None
        C.check(L.gf_geodesic(C.ptr(D), C.ptr(I), 1 if I.dtype == torch.int64 else 0, N, k, C.ptr(seeds), Q,
                              ctypes.c_float(float(radius)), int(max_step), C.ptr(geo), C.ptr(stats), C.ptr(row_max),
                              C.ptr(ws), nbytes, C.stream_of(D.device)), "geodesic")
    return (geo, stats) if return_stats else geo


def geodesic_from_graph_batch(locs, graphs, seeds, radius, max_step, row_max=False, return_stats=False):
    """geodesic_from_graph for a BATCH of scenes: one library call per <= 32 scenes (gf_geodesic_batch, seven kernels
    whatever the number of scenes), every map bitwise the one geodesic_from_graph gives for its scene alone.
    locs: list of (N_b, 3) f32 CUDA tensors.  They only choose the numbering the propagation runs in (the cell order
    of a kNN grid over them): the maps do not depend on them, the scene's own points make the call fastest.
    graphs: list of (D (N_b,k) sqrt'ed f32, I (N_b,k) int64 or int32), one k and one index dtype for all.
    seeds: list of (Q,) int tensors, one Q for all.
    Returns the list of (Q, N_b) f32 maps, or (maps[, stats (B,2) i64][, row_max list of (Q,) f32]) when asked.
    Scenes too large for the batched kernel run through geodesic_from_graph one at a time; a scene without points
    gets a (Q, 0) map (row maxima -1), a call without seeds (0, N_b) maps."""
    B = len(graphs)
    C.require(B > 0 and len(locs) == B and len(seeds) == B, "one point set and one seed tensor per graph")
    dev = graphs[0][0].device
    k, idt = graphs[0][0].shape[-1], graphs[0][1].dtype
    C.require(idt in (torch.int64, torch.int32), "I must be int64/int32 CUDA")
    for x, (D, I) in zip(locs, graphs):
        C.check_cuda_f32(D, "D")
        C.check_cuda_f32(x, "locs")
        C.require(I.is_cuda and I.is_contiguous() and I.dtype == idt, "I must be contiguous CUDA, one dtype for all")
        C.require(D.dim() == 2 and D.size(1) == k and tuple(I.shape) == tuple(D.shape), "graphs must be (N_b, k), one k")
        C.require(tuple(x.shape) == (D.size(0), 3) and x.device == dev and D.device == dev and I.device == dev,
                  "locs must be (N_b, 3), on the graphs' device")
    seeds = [s.to(device=dev, dtype=torch.int32).contiguous() for s in seeds]
    Q = seeds[0].numel()
    C.require(all(s.numel() == Q for s in seeds), "one (Q,) seed tensor per scene, one Q for all")
    Ns = [D.size(0) for D, _ in graphs]
    geo = [torch.empty((Q, n), dtype=torch.float32, device=dev) for n in Ns]
    rmax = [torch.full((Q,), -1.0, dtype=torch.float32, device=dev) for _ in Ns] if row_max else None
    stats = torch.zeros((B, 2), dtype=torch.int64, device=dev) if return_stats else None
    batch = [b for b in range(B) if Q > 0 and 0 < Ns[b] <= BATCH_MAX_POINTS]
    for b in range(B):
        if Q > 0 and Ns[b] > BATCH_MAX_POINTS:
            out = geodesic_from_graph(*graphs[b], seeds[b], radius, max_step, return_stats=return_stats,
                                      row_max=rmax[b] if rmax else None)
            geo[b] = out[0] if return_stats else out
            if return_stats:
                stats[b] = out[1]
    L = C.lib()
    with torch.cuda.device(dev):
        st = C.stream_of(dev)
        for b0 in range(0, len(batch), BATCH_MAX):
            sub = batch[b0:b0 + BATCH_MAX]
            n = len(sub)
            Nc = (ctypes.c_int * n)(*[Ns[b] for b in sub])
            nbytes = L.gf_geodesic_batch_workspace_bytes(Nc, n, Q, k)
            C.require(nbytes > 0, "geodesic_batch: bad sizes")
            ws = C.workspace.get(dev, "geodesic_batch", nbytes)
            st_call = torch.empty((n, 2), dtype=torch.int64, device=dev) if return_stats else None
            C.check(L.gf_geodesic_batch(_ptr_array([locs[b] for b in sub]), _ptr_array([graphs[b][0] for b in sub]),
                                        _ptr_array([graphs[b][1] for b in sub]), 1 if idt == torch.int64 else 0, Nc,
                                        n, k, _ptr_array([seeds[b] for b in sub]), Q, ctypes.c_float(float(radius)),
                                        int(max_step), _ptr_array([geo[b] for b in sub]),
                                        _ptr_array([rmax[b] for b in sub]) if rmax else None, C.ptr(st_call),
                                        C.ptr(ws), nbytes, st), "geodesic_batch")
            if return_stats:
                stats.index_copy_(0, torch.tensor(sub, device=dev), st_call)
    if not (return_stats or row_max):
        return geo
    out = [geo]
    if return_stats:
        out.append(stats)
    if row_max:
        out.append(rmax)
    return tuple(out)


def geodesic_from_points(locs, seeds, neighbor, radius, max_step, return_graph=False, return_stats=False,
                         row_max=None, ws_tag="guidance"):
    """kNN graph + propagation of one scene in one library call (the body of the reference loop,
    geodesic_utils.py:98-163)."""
    C.check_cuda_f32(locs, "locs")
    N = locs.size(0)
    seeds = seeds.to(device=locs.device, dtype=torch.int32).contiguous()
    Q = seeds.numel()
    geo = torch.empty((Q, N), dtype=torch.float32, device=locs.device)
    D = torch.empty((N, neighbor), dtype=torch.float32, device=locs.device) if return_graph else None
    I = torch.empty((N, neighbor), dtype=torch.int32, device=locs.device) if return_graph else None
    stats = torch.zeros(2, dtype=torch.int64, device=locs.device) if return_stats else None
    L = C.lib()
    with torch.cuda.device(locs.device):
        nbytes = L.gf_guidance_workspace_bytes(N, Q, int(neighbor))
        ws = C.workspace.get(locs.device, ws_tag, nbytes)
        C.check(L.gf_guidance_seeded(C.ptr(locs), N, C.ptr(seeds), Q, int(neighbor), ctypes.c_float(float(radius)),
                                     int(max_step), C.ptr(geo), C.ptr(D), C.ptr(I), C.ptr(stats), C.ptr(row_max),
                                     C.ptr(ws), nbytes, C.stream_of(locs.device)), "guidance_seeded")
    out = [geo]
    if return_graph:
        out += [D, I]
    if return_stats:
        out.append(stats)
    return out[0] if len(out) == 1 else tuple(out)


@torch.no_grad()
def cal_geodesic_vectorize(gpu_index, pre_enc_inds, locs_float_, batch_offset_, max_step=128, neighbor=64,
                           radius=0.05, n_queries=128):
    """geodesic_utils.py:91-164, same signature and return value: a list over the batch of
    (n_queries, N_b) float32 tensors on locs_float_.device, -1 = unreachable.

    gpu_index: a FlatL2Index (or None) -> kNN and propagation run fused in the library;
               any other object with add/search/reset (e.g. a real faiss GpuIndexFlatL2) -> its
               neighbours are used as they are and only the propagation runs here."""
    batch_size = pre_enc_inds.shape[0]
    offsets = batch_offset_.tolist() if isinstance(batch_offset_, torch.Tensor) else list(batch_offset_)
    own_index = gpu_index is None or isinstance(gpu_index, FlatL2Index)
    fused = own_index and (gpu_index is None or gpu_index.algo == 0)
    dev = locs_float_.device
    geo_dists = [None] * batch_size
    batch = []  # (b, points, seeds) of the scenes that go through the batched library call
    graphs = []  # (b, points, (D, I), seeds) of the scenes whose graph comes from the caller's index
    for b in range(batch_size):
        start, end = int(offsets[b]), int(offsets[b + 1])
        seeds = pre_enc_inds[b][:n_queries]
        if end - start == 0:
            geo_dists[b] = torch.empty((seeds.numel(), 0), dtype=torch.float32, device=dev)
            continue
        locs_b = locs_float_[start:end].contiguous()
        if fused and end - start <= BATCH_MAX_POINTS and seeds.numel() > 0:
            batch.append((b, locs_b, seeds))
        elif fused:
            geo_dists[b] = geodesic_from_points(locs_b, seeds, neighbor, radius, max_step)
        else:
            # the index protocol answers one scene per call (:18-21); the graphs are propagated together below
            graphs.append((b, locs_b, find_knn(gpu_index, locs_b, neighbor=neighbor), seeds))
    # The scenes of a batch are independent (the reference loops over them, :98): their graphs are built side by
    # side and ALL their (scene, seed) pairs are propagated by one launch (gf_guidance_batch) -- the per-seed runs
    # are chains of dependent latencies, so the GPU is only filled by many of them at once.  Graphs from the caller's
    # index take the same launch after one pass that packs them all (gf_geodesic_batch).
    # Scenes with the same number of seeds share a call (pre_enc_inds is one (B, >= n_queries) tensor: all of them).
    groups = {}
    for b, locs_b, seeds in batch:
        groups.setdefault(seeds.numel(), []).append((b, locs_b, seeds))
    for q_n, items in groups.items():
        _, geos = geodesic_guidance_batch([x for _, x, _ in items], q_n, neighbor, radius, max_step,
                                          seeds=[s for _, _, s in items])
        for (b, _, _), g in zip(items, geos):
            geo_dists[b] = g
    groups = {}
    for item in graphs:
        groups.setdefault(item[3].numel(), []).append(item)
    for items in groups.values():
        if len(items) == 1:
            # one scene: the grid build of the batched call costs more than its cell order saves (DESIGN 4.3)
            b, _, (D, I), seeds = items[0]
            geo_dists[b] = geodesic_from_graph(D, I, seeds, radius, max_step)
            continue
        geos = geodesic_from_graph_batch([x for _, x, _, _ in items], [g for _, _, g, _ in items],
                                         [s for _, _, _, s in items], radius, max_step)
        for (b, _, _, _), g in zip(items, geos):
            geo_dists[b] = g
    return geo_dists


_MAX_SCENES_IN_FLIGHT = 4
_lane_streams = {}


def _side_streams(device, n):
    """up to n cached side streams of `device` (created once per device and thread of first use)"""
    key = (device.index if device.index is not None else torch.cuda.current_device())
    have = _lane_streams.setdefault(key, [])
    while len(have) < n:
        have.append(torch.cuda.Stream(device=device))
    return have[:n]
