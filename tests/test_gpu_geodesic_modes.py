"""Every propagation kernel the library can launch, reached through the rules that choose it from N, Q and the SM
count, bit for bit against the oracle, with a check of which kernel ran:

    geo_bfs_batch_kernel<1024>   scenes whose two bitmaps fit on chip, at most two seeds per SM
    geo_bfs_batch_kernel<512>    the same with more seeds
    geo_seed_bfs_kernel<2>       both bitmaps on chip: seed-sharded scenes (peers given: always the per-scene kernel)
    geo_seed_bfs_kernel<1>       visited bitmap only: scenes too large for both bitmaps (N > ~860k), Q <= SM count
    geo_seed_bfs_kernel<0>       no on-chip state: the same with more seeds (test_full_size_config_c4: k = 16)

Each kernel also runs a case whose frontiers spill beyond the on-chip queue into the global overflow area.  The
oracle's statistics show it: R reached pairs over Q seeds and levels + 1 levels (the seed's included) average more
than the queue holds, so some level's frontier was larger."""
import ctypes
import functools
import re

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

QUEUE = 4096  # frontier entries of the on-chip queue (the batched kernel's queue is at most this long)

SCENES = {  # N, points
    "n30k": (30000, "scene"),
    # on the surfaces of `scene` a frontier grows linearly with the level and stays below the queue in any scene the
    # batched kernel takes; in a filled volume it grows with the square of the level
    "volume400k": (400_000, "volume"),
    "n4097": (4097, "small_room"),  # N just over a queue
    "n20k": (20000, "room_2x1.5"),
    "room1m": (1_000_000, "room_1m"),
}
# scene, Q (a number or a function of the SM count), k, radius, max_step, entry point, kernel, spills beyond the queue.
# The batched and one-peer runs of a case are adjacent: they share one graph and one oracle result.
CASES = {}
for name, q, k, r, ms, spills in [
        ("n30k", 8, 16, 0.5, 40, False),
        ("volume400k", 6, 64, 10.0, 24, True),
        ("n4097", 5, 33, 10.0, 4, False),  # K = 32 exactly (KP = 32)
        ("n20k", lambda sms: 2 * sms + 4, 8, 0.2, 300, False)]:  # a persistent loop over the seeds, deep
    many = callable(q)
    CASES["batched_%s" % name] = (name, q, k, r, ms, "geodesic", ("bfs_batch", 512 if many else 1024), spills)
    CASES["one_peer_%s" % name] = (name, q, k, r, ms, "one_peer", ("seed_bfs", 2), spills)
CASES["visited_only_k16"] = ("room1m", 8, 16, 0.5, 32, "geodesic", ("seed_bfs", 1), False)
CASES["visited_only_k64"] = ("room1m", 8, 64, 10.0, 96, "geodesic", ("seed_bfs", 1), True)
CASES["no_on_chip_state_k64"] = ("room1m", lambda sms: sms + 1, 64, 10.0, 80, "geodesic", ("seed_bfs", 0), True)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _points(n, gen):
    from geoformer_b200.scenes import room, scene

    if gen == "volume":
        return torch.rand(n, 3, generator=torch.Generator().manual_seed(17))  # the unit cube, filled
    if gen == "room_1m":
        return room(n, 4321)
    shape = {"scene": {}, "small_room": dict(L=(1.0, 1.0, 0.5), nbox=2), "room_2x1.5": dict(L=(2.0, 1.5, 1.0), nbox=4)}
    return scene(n, 17, **shape[gen])


@functools.lru_cache(maxsize=1)
def _inputs(scene_name, Q, k, r, ms, oracle):
    """the kNN graph on the device, FPS seeds, and the oracle's maps and statistics"""
    from geoformer_b200.geodesic_utils import knn_graph

    x = _points(*SCENES[scene_name])
    seeds = oracle.furthest_point_sampling(x[None].numpy(), Q)[0]
    D, I = knn_graph(x.to("cuda:0"), k)
    want, R, lev = oracle.geodesic(D.cpu().numpy(), I.cpu().numpy(), seeds, r, ms, return_stats=True)
    return D, I, torch.from_numpy(seeds).to("cuda:0"), want, R, lev


def _launched(fn):
    """fn() under the profiler -> its result and the propagation kernels it launched, as (kernel, template argument)"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    found = (re.search(r"geo_(bfs_batch|seed_bfs)_kernel(?:<|ILi)(\d+)", e.name) for e in prof.events())
    return out, [(m.group(1), int(m.group(2))) for m in found if m]


def _geodesic(D, I, seeds, r, ms):
    from geoformer_b200.geodesic_utils import geodesic_from_graph

    rm = torch.zeros(seeds.numel(), device=D.device)
    geo, stats = geodesic_from_graph(D, I, seeds, r, ms, return_stats=True, row_max=rm)
    return geo, stats, rm


def _geodesic_one_peer(D, I, seeds, r, ms):
    """gf_geodesic_scatter with one peer matrix on the same device: the finished rows are also stored there"""
    from geoformer_b200 import _capi as C

    N, k = D.shape
    Q = seeds.numel()
    seeds = seeds.to(torch.int32).contiguous()
    geo = torch.empty((Q, N), dtype=torch.float32, device=D.device)
    peer = torch.full_like(geo, float("nan"))
    stats = torch.zeros(2, dtype=torch.int64, device=D.device)
    peers = (ctypes.c_void_p * 1)(peer.data_ptr())
    L = C.lib()
    with torch.cuda.device(D.device):
        nbytes = L.gf_geodesic_workspace_bytes(N, k, Q)
        ws = C.workspace.get(D.device, "geodesic", nbytes)
        C.check(L.gf_geodesic_scatter(C.ptr(D), C.ptr(I), 1 if I.dtype == torch.int64 else 0, N, k, C.ptr(seeds), Q,
                                      ctypes.c_float(r), ms, C.ptr(geo), ctypes.cast(peers, ctypes.c_void_p), 1,
                                      C.ptr(stats), C.ptr(ws), nbytes, C.stream_of(D.device)), "geodesic_scatter")
    return geo, peer, stats


@pytest.mark.parametrize("case", list(CASES))
def test_geodesic_state_layouts_and_overflow(cuda_lib, oracle_lib, case):
    scene_name, Q, k, r, ms, entry, kernel, spills = CASES[case]
    Q = Q(_sms()) if callable(Q) else Q
    D, I, seeds, want, R, lev = _inputs(scene_name, Q, k, r, ms, oracle_lib)
    if entry == "geodesic":
        (geo, stats, rm), kernels = _launched(lambda: _geodesic(D, I, seeds, r, ms))
    else:
        (geo, peer, stats), kernels = _launched(lambda: _geodesic_one_peer(D, I, seeds, r, ms))
    assert kernels == [kernel]
    got = geo.cpu().numpy()
    assert np.array_equal(got, want), int((got != want).sum())
    if entry == "geodesic":
        assert np.array_equal(rm.cpu().numpy(), want.max(axis=1)), "row_max by-product"
    else:  # the seed-sharded entry point has no row-maximum output
        assert torch.equal(peer, geo)
    assert (int(stats[0]), int(stats[1])) == (R, lev)
    if spills:
        assert R / (Q * (lev + 1)) > QUEUE, (R, Q, lev)
