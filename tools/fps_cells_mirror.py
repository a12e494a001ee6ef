"""CPU mirror of the culled FPS on the kNN grid's cell order (fps_cells_kernel, gf_fps.cu): exact FPS that updates only
the blocks of cell-ordered points a new seed can reach.  It checks the seeds against oracle.furthest_point_sampling and
counts the work of every round.

    python tools/fps_cells_mirror.py [--scenes 2] [--n 100000] [--m 256] [--S 32 64 128]

Cell order: the points are counting-sorted into a uniform grid, x fastest, with a cell edge that puts about 0.45 k
points (k = 16) in the average point's cell, as the kNN grid does; inside a cell the order is arbitrary.  Blocks are
S consecutive points of that order with the tight box of their eligible points.  A round updates a block only if
the lower bound of sq3(p - c) over its box, shrunk by 2^-20, is below the block's largest running minimum.
Every float32 operation is the library's: sq3 = fma(z, z, fma(x, x, y * y)) (gf::sq3), emulated exactly with
round-to-odd.
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHRINK = np.float32(1.0 - 2.0 ** -20)


def fma32(a, b, c):
    """float32 fma(a, b, c), correctly rounded: a * b is exact in float64, the float64 sum is rounded to odd, and
    rounding that to float32 is then the correctly rounded result (53 >= 24 + 2 bits)."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    even = (s.view(np.int64) & 1) == 0
    fix = (err != 0) & even
    s = np.where(fix, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def sq3(x, y, z):
    return fma32(z, z, fma32(x, x, (y * y).astype(np.float32)))


def lower_bound(lo, hi, c):
    """a lower bound of the computed sq3(p - c) over the box [lo, hi] (arrays (..., 3) float32, c (3,) float32)"""
    g = np.maximum(np.maximum(lo - c, c - hi), np.float32(0))
    return (sq3(g[..., 0], g[..., 1], g[..., 2]) * SHRINK).astype(np.float32)


def ref_log2_block(n):
    L = 0
    while (2 << L) <= n and L < 9:
        L += 1
    return L


def brev32(v):
    v = v.astype(np.uint32)
    out = np.zeros_like(v)
    for b in range(32):
        out |= ((v >> np.uint32(b)) & np.uint32(1)) << np.uint32(31 - b)
    return out


def rank_of(i, L):
    i = i.astype(np.uint32)
    return brev32(i & np.uint32((1 << L) - 1)) | (i >> np.uint32(L))


def decode(rk, L):
    rk = int(rk)
    if L == 0:
        return rk
    lo = rk & ((1 << (32 - L)) - 1)
    hi = rk >> (32 - L)
    return (lo << L) | int(brev32(np.array([hi], np.uint32))[0] >> np.uint32(32 - L))


def cell_order(xyz, k=16, seed=0):
    lo, hi = xyz.min(0), xyz.max(0)
    ext = np.maximum(hi - lo, 1e-6)
    h = float(np.cbrt(np.prod(ext) * 0.45 * k / len(xyz)))
    for _ in range(40):  # occupancy ~ h^2 on surfaces: rescale until sum(c^2) / N is about 0.45 k
        d = (np.floor(ext / h) + 1).astype(np.int64)
        c = np.minimum(np.floor((xyz - lo) / h).astype(np.int64), d - 1)
        cell = (c[:, 2] * d[1] + c[:, 1]) * d[0] + c[:, 0]
        occ = np.bincount(cell).astype(np.float64)
        f = float(np.sqrt(0.45 * k / max((occ ** 2).sum() / len(xyz), 1e-3)))
        if abs(f - 1) < 0.02:
            break
        h *= min(max(f, 0.5), 2.0)
    shuffle = np.random.default_rng(seed).permutation(len(xyz))
    return shuffle[np.argsort(cell[shuffle], kind="stable")]


def fps_cells(xyz, m, S, order):
    """seeds of the culled FPS and, per round, (blocks updated, points updated)"""
    N = len(xyz)
    L = ref_log2_block(N)
    nb = (N + S - 1) // S
    pad = nb * S - N
    pts = np.concatenate([xyz[order], np.zeros((pad, 3), np.float32)])
    ids = np.concatenate([order, np.zeros(pad, np.int64)]).astype(np.uint32)
    elig = ~(sq3(pts[:, 0], pts[:, 1], pts[:, 2]).astype(np.float64) <= 1e-3)
    elig[N:] = False
    t = np.where(elig, np.float32(1e10), np.float32(-1)).astype(np.float32)
    lo_key = np.where(elig, ~rank_of(ids, L), np.uint32(0)).astype(np.uint32)
    P = pts.reshape(nb, S, 3)
    E = elig.reshape(nb, S)
    box_lo = np.where(E[..., None], P, np.float32(np.inf)).min(1)
    box_hi = np.where(E[..., None], P, np.float32(-np.inf)).max(1)

    def block_keys(bl):
        tb = t.reshape(nb, S)[bl]
        v = np.where(tb >= 0, tb.view(np.uint32), np.uint32(0)).astype(np.uint64)
        key = (v << np.uint64(32)) | lo_key.reshape(nb, S)[bl].astype(np.uint64)
        return key.max(1)

    bkey = block_keys(np.arange(nb))
    idx = np.zeros(m, np.int64)
    c = xyz[0].copy()
    work = []
    for j in range(1, m):
        bmax = np.where(bkey > 0, (bkey >> np.uint64(32)).astype(np.uint32).view(np.float32), np.float32(-1))
        upd = np.nonzero(lower_bound(box_lo, box_hi, c) < bmax)[0]
        if len(upd):
            q = (upd[:, None] * S + np.arange(S)).ravel()
            d = sq3(pts[q, 0] - c[0], pts[q, 1] - c[1], pts[q, 2] - c[2])
            t[q] = np.minimum(d, t[q])
            bkey[upd] = block_keys(upd)
        work.append((len(upd), len(upd) * S))
        w = bkey.max()
        if w == 0:
            idx[j] = 0
        else:
            idx[j] = decode(~np.uint32(int(w) & 0xFFFFFFFF), L)
        c = xyz[idx[j]].copy()
    return idx, np.array(work).reshape(-1, 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scenes", type=int, default=2)
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--m", type=int, default=256)
    ap.add_argument("--S", type=int, nargs="+", default=[32, 64, 128])
    a = ap.parse_args()
    import oracle
    from geoformer_b200.scenes import scene

    oracle.build()
    for s in range(a.scenes):
        x = scene(a.n, 1234 + s).numpy()
        want = oracle.furthest_point_sampling(x[None], a.m)[0]
        order = cell_order(x)
        for S in a.S:
            got, work = fps_cells(x, a.m, S, order)
            full = (a.m - 1) * a.n
            pts = int(work[:, 1].sum())
            print("scene %d S=%d: seeds %s the oracle; points updated %d = %.4f of %d x N (rounds 1-10: %d, "
                  "11-255: %d), blocks updated %d of %d x %d, per round after round 10: mean %.1f max %d" % (
                      s, S, "equal" if np.array_equal(got, want) else "DIFFER FROM", pts, pts / full, a.m - 1,
                      int(work[:10, 1].sum()), int(work[10:, 1].sum()), int(work[:, 0].sum()), a.m - 1,
                      (a.n + S - 1) // S, work[10:, 0].mean(), work[10:, 0].max()))


if __name__ == "__main__":
    main()
