"""Kernel-faithful float64 references of the three tensor-core kernels -- TEST INFRASTRUCTURE ONLY.

The decoder cross-attention (forward and backward, gf_attention.cu) and the mask head (gf_mask_head.cu) read raw
fp32 operands from shared memory and multiply them as tcgen05 kind::tf32.  Everything else they compute is plain
fp32 whose order can be read from the code.  The functions below round exactly the operands the kernels hand to the
tensor cores to TF32 (10 explicit mantissa bits, `tf32_round`) and compute everything else in float64, so that what
remains between a kernel and its emulation is fp32 accumulation, __expf and rare one-TF32-ulp flips of rounded
intermediates.  Each function also returns an elementwise bound of that remainder, built from
  * the tensor-core accumulation, K * 2^-23 * sum |terms| (TC below),
  * sequential fp32 sums, n * 2^-24 * sum |terms| (U below),
  * the __expf error, (2 + 2 |x|) * 2^-23 relative (the CUDA guide states 2 + 1.16 |x| ulp; the argument x = s - max
    is itself one fp32 subtraction),
  * the flips: an intermediate the kernel computes in fp32 and then hands to the tensor cores (h, g, dv, dh) can
    round to the TF32 neighbour of the emulated value when it lies within its fp32 error of a rounding boundary.
    The kernel's operand lies in [T(lo), T(hi)] for the interval [lo, hi] its fp32 value can take (rounding is
    monotone), so the width of that interval enters the bound, and is zero away from a boundary.
The tests (tests/test_tf32_reference.py) calibrate a margin on these bounds; the near-kink sets returned here state
which gradient entries a ReLU mask may set differently in fp32.

Works on float tensors on any device (the GPU tests run it on the GPU); results are float64.  The keyword mutations
(drop_last_context, no_rescale, lse_half0, b2_unscaled, no_tf32, drop_feature_channel) emulate specific wrong kernels;
only the sensitivity test uses them.
"""
import math

import torch
import torch.nn.functional as F

U = 2.0 ** -24   # fp32 unit roundoff
TC = 2.0 ** -23  # per-term allowance of the tensor core's fp32 accumulation (truncating alignment included)
F64 = torch.float64

# How kind::tf32 treats the 13 low mantissa bits of a raw fp32 operand, measured on a B200 by
# tests/test_tf32_reference.py::test_tf32_rounding_mode_probe (DESIGN section 4).
KERNEL_TF32_MODE = "rz"


def tf32_round(x, mode=KERNEL_TF32_MODE):
    """x cast to fp32, then rounded to TF32 (10 explicit mantissa bits), as float64.  mode: "rz" drops the 13 low
    bits, "rne" rounds to nearest with ties to even, "rna" with ties away from zero; None leaves x as it is (in
    float64), which turns the emulation into a plain float64 evaluation."""
    if mode is None:
        return x.to(F64)
    x32 = x.to(torch.float32)
    b = x32.contiguous().view(torch.int32)
    low = b & 0x1FFF
    kept = b & ~0x1FFF
    if mode == "rz":
        up = torch.zeros_like(low, dtype=torch.bool)
    elif mode == "rne":
        up = (low > 0x1000) | ((low == 0x1000) & ((kept & 0x2000) != 0))
    elif mode == "rna":
        up = low >= 0x1000
    else:
        raise ValueError("mode must be rz, rne, rna or None")
    r = (kept + up.to(torch.int32) * 0x2000).view(torch.float32)
    return torch.where(torch.isfinite(x32), r, x32).to(F64)


def _operand_interval(v, err, mode, relu=False):
    """the emulated TF32 operand of an fp32 intermediate with exact value v and fp32 error bound err, and the width
    of the interval the kernel's operand can lie in"""
    lo, hi = v - err, v + err
    if relu:
        v, lo, hi = F.relu(v), F.relu(lo), F.relu(hi)
    return tf32_round(v, mode), tf32_round(hi, mode) - tf32_round(lo, mode)


def _gamma(n):
    return n * U


# ---- decoder vector cross-attention ---------------------------------------------------------------------------------
def _att_prepare(tgt2, memory, rel, w, mode):
    d = lambda t: t.to(F64)  # noqa: E731
    W = {k: d(v) for k, v in w.items()}
    t, m, r = d(tgt2), d(memory), d(rel)
    T = {k: tf32_round(w[k], mode) for k in ("w1", "w2", "wv")}
    rt = tf32_round(rel, mode)
    # tables (att_tables_kernel): 64-term fp32 FMA chains, then + b1 / + bv
    aq = t @ W["w1"].t() + W["b1"]
    p1 = m @ W["w1"].t()
    pv = m @ W["wv"].t() + W["bv"]
    e_aq = _gamma(66) * (t.abs() @ W["w1"].abs().t() + W["b1"].abs())
    e_p1 = _gamma(65) * (m.abs() @ W["w1"].abs().t())
    e_pv = _gamma(66) * (m.abs() @ W["wv"].abs().t() + W["bv"].abs())
    # product 1: [Wv; W1] x rel on the tensor cores
    d1h, d1v = rt @ T["w1"].t(), rt @ T["wv"].t()
    s1h, s1v = rt.abs() @ T["w1"].abs().t(), rt.abs() @ T["wv"].abs().t()
    hp = d1h + aq[:, None] - p1[None]  # (Q,C,B,64)
    e_hp = 64 * TC * s1h + e_aq[:, None] + e_p1[None] + 2 * U * (d1h.abs() + aq.abs()[:, None] + p1.abs()[None])
    v = d1v + pv[None]
    e_v = 64 * TC * s1v + e_pv[None] + U * (d1v.abs() + pv.abs()[None])
    return W, T, t, m, r, rt, hp, e_hp, v, e_v


def attention_forward(tgt2, memory, rel, w, mode=KERNEL_TF32_MODE, *, near_kink=False, drop_last_context=False,
                      no_rescale=False, lse_half0=False, b2_unscaled=False, no_tf32=False):
    """rel_cross_attention_kernel (the unfused, saving variant) in float64 with its TF32 operands.
    tgt2 (Q,B,64), memory (C,B,64), rel (Q,C,B,64), w the eight weights -> dict with
      out, o, lse (Q,B,64) and their bounds e_out, e_o, e_lse;
      with near_kink: kink_h (Q,C,B,64), the pairs and hidden channels whose pre-activation lies within its fp32
      error of ReLU's kink, and kink_out (Q,B,64), the outputs whose out_mlp pre-activation lies within e_out of it;
      and the intermediates the backward emulation reuses (key "_ctx")."""
    if no_tf32:
        mode = None
    Q, C, B, _ = rel.shape
    W, T, t, m, r, rt, hp, e_hp, v, e_v = _att_prepare(tgt2, memory, rel, w, mode)
    # hidden tile: relu in fp32, handed to product 2 as a TF32 operand
    ht, wd_h = _operand_interval(hp, e_hp, mode, relu=True)
    d2 = ht @ T["w2"].t()
    e_d2 = 64 * TC * (ht.abs() @ T["w2"].abs().t()) + wd_h @ T["w2"].abs().t()
    s = (d2 / 8 + W["b2"]) if b2_unscaled else (d2 + W["b2"]) / 8
    e_s = (e_d2 + U * (d2.abs() + W["b2"].abs())) / 8
    if drop_last_context:
        s = s.clone()
        s[:, C - 1] = -math.inf
    M = s.max(1).values  # (Q,B,64)
    ex = torch.exp(s - M[:, None])
    S = ex.sum(1)
    a = ex / S[:, None]
    o = (a * v).sum(1)
    lse = M + torch.log(S)
    if no_rescale or lse_half0:
        o, lse = _softmax_mutant(s, v, no_rescale, lse_half0)
    # bounds: score and v errors, __expf, the fp32 sums of the online softmax (per column half, with the rescales)
    nt = (C + 63) // 64
    srange = M - s.masked_fill(torch.isinf(s), math.inf).min(1).values
    eps = 2.0 ** -23 * (2 + 2 * (M[:, None] - s)) + 2.0 ** -23 * (2 * (nt + 2) + 2 * srange)[:, None]
    eps = torch.where(torch.isinf(s), torch.zeros_like(s), eps)
    dev = (v - o[:, None]).abs()
    gam = _gamma(34 * nt + 8)
    e_o = 1.01 * ((a * (e_s + eps) * dev).sum(1) + (a * e_v).sum(1)) + gam * ((a * v.abs()).sum(1) + o.abs())
    e_lse = 1.01 * (a * (e_s + eps)).sum(1) + gam + 2.0 ** -22 * (M.abs() + torch.log(S).abs() + 1)
    y = o @ W["wo"].t() + W["bo"]
    e_out = e_o @ W["wo"].abs().t() + _gamma(66) * (o.abs() @ W["wo"].abs().t() + W["bo"].abs())
    res = {"out": F.relu(y), "o": o, "lse": lse, "e_out": e_out, "e_o": e_o, "e_lse": e_lse}
    if near_kink:
        res["kink_h"] = hp.abs() <= e_hp
        res["kink_out"] = y.abs() <= e_out
    res["_ctx"] = dict(W=W, T=T, t=t, m=m, r=r, rt=rt, hp=hp, e_hp=e_hp, ht=ht, wd_h=wd_h, v=v, e_v=e_v, s=s,
                       e_s=e_s, a=a, o=o, y=y, e_o=e_o, e_out=e_out, mode=mode)
    return res


def _softmax_mutant(s, v, no_rescale, lse_half0):
    """the online softmax of the kernel, per column half and context tile, with one of two defects:
    no_rescale keeps each tile's partial sums at that tile's running maximum; lse_half0 takes half 0's maximum"""
    Q, C, B, D = s.shape
    nt = (C + 63) // 64
    pad = nt * 64 - C
    sp = F.pad(s, (0, 0, 0, 0, 0, pad), value=-math.inf).reshape(Q, nt, 2, 32, B, D)
    vp = F.pad(v, (0, 0, 0, 0, 0, pad)).reshape(Q, nt, 2, 32, B, D)
    tmax = sp.max(3).values  # (Q,nt,2,B,D)
    run = torch.cummax(tmax, 1).values  # running maximum after each tile
    mh = run[:, -1]  # (Q,2,B,D)
    ref = run if no_rescale else mh[:, None].expand_as(run)
    ex = torch.exp(sp - ref[:, :, :, None])
    ex = torch.where(torch.isinf(sp), torch.zeros_like(ex), ex)
    sh, ah = ex.sum((1, 3)), (ex * vp).sum((1, 3))  # (Q,2,B,D) at each half's (claimed) maximum mh
    mx = mh.max(1).values
    e = torch.where(torch.isinf(mh), torch.zeros_like(mh), torch.exp(mh - mx[:, None]))
    S, A = (sh * e).sum(1), (ah * e).sum(1)
    o = A / S
    lse = (mh[:, 0] if lse_half0 else mx) + torch.log(S)
    return o, lse


def attention_backward(fwd, dy):
    """rel_cross_attention_bwd_kernel and its finishing kernels in float64 with the TF32 operands of P1-P5, for the
    forward emulation `fwd` (attention_forward(..., near_kink=True)) and the upstream gradient dy (Q,B,64).
    The kernel's saved o and lse are those of the forward (their emulation is used here; their kernel-vs-emulation
    difference is in e_o / e_lse).  dy must be zero where fwd["kink_out"] is set (the caller's exclusion).
    A pair whose hidden channel lies at ReLU's kink (fwd["kink_h"]) may carry W2^T g or 0 there in the kernel: its
    whole contribution enters the bounds of every gradient it reaches.
    -> dict of the gradients tgt2, memory, rel, w1, b1, w2, b2, wv, bv, wo, bo and a bound "e_<name>" for each."""
    c = fwd["_ctx"]
    W, T, mode = c["W"], c["T"], c["mode"]
    t, m, r, rt, hp, e_hp, ht, v, e_v, a, o = (c[k] for k in ("t", "m", "r", "rt", "hp", "e_hp", "ht", "v", "e_v",
                                                               "a", "o"))
    dy = dy.to(F64)
    y = c["y"]
    dz = dy * (y > 0)
    do = dz @ W["wo"]  # prologue: 64-term fp32 chain
    e_do = _gamma(64) * (dz.abs() @ W["wo"].abs())
    lse, e_lse = fwd["lse"], fwd["e_lse"]
    # P2 gives the forward's s bit for bit: a = exp(s - lse) with the saved lse
    e_s = c["e_s"]
    e_a = a * (e_s + e_lse[:, None] + 2.0 ** -23 * (2 + 2 * (lse[:, None] - c["s"]).abs()) + 2 * U)
    e_a = torch.nan_to_num(e_a)
    dv = a * do[:, None]
    e_dv = e_a * do.abs()[:, None] + a * e_do[:, None] + U * dv.abs()
    vo = v - o[:, None]
    e_vo = e_v + c["e_o"][:, None] + U * vo.abs()
    g = dv * vo / 8
    e_g = (e_dv * vo.abs() + dv.abs() * e_vo) / 8 + U * g.abs()
    # P3: W2^T g with g a TF32 operand; dh = (W2^T g) [hp > 0]
    gt, wd_g = _operand_interval(g, e_g, mode)
    w2t = T["w2"]
    dhp = gt @ w2t
    e_dhp = 64 * TC * (gt.abs() @ w2t.abs()) + wd_g @ w2t.abs()
    on = hp > 0
    kink_h = fwd["kink_h"]
    dh = dhp * on
    # a pair whose hidden channel is at the kink may carry dhp or 0 in the kernel
    e_dh = e_dhp * (on | kink_h) + dhp.abs() * kink_h
    # P4: dW2 = sum_c g h^T with both TF32 operands (h^T is the forward's hidden tile)
    Q, C, B, _ = hp.shape
    outer = lambda x, y: torch.einsum("...i,...j->ij", x, y)  # noqa: E731
    dW2 = outer(gt, ht)
    e_w2 = (C * TC + _gamma(Q * B + 16)) * outer(gt.abs(), ht.abs()) + outer(wd_g, ht.abs()) \
        + outer(gt.abs(), c["wd_h"])
    # P5: [dWv; dW1] r-terms = sum_c [dv; dh] r^T with dv, dh, r as TF32 operands
    dvt, wd_dv = _operand_interval(dv, e_dv, mode)
    dht, wd_dh = _operand_interval(dh, e_dh, mode)
    rabs = rt.abs()
    dWv_r, dW1_r = outer(dvt, rt), outer(dht, rt)
    e_wv_r = (C * TC + _gamma(Q * B + 16)) * outer(dvt.abs(), rabs) + outer(wd_dv, rabs)
    e_w1_r = (C * TC + _gamma(Q * B + 16)) * outer(dht.abs(), rabs) + outer(wd_dh, rabs)
    # fp32 finishing sums (att_bwd_rows_kernel, att_bwd_weights_kernel, att_bwd_drel_kernel) of the fp32 pairs
    hsum, DH, DV = dh.sum(1), dh.sum(0), dv.sum(0)
    e_hsum = e_dh.sum(1) + _gamma(C) * dh.abs().sum(1)
    e_DH = e_dh.sum(0) + _gamma(Q) * dh.abs().sum(0)
    e_DV = e_dv.sum(0) + _gamma(Q) * dv.abs().sum(0)
    W1, Wv, Wo = W["w1"].abs(), W["wv"].abs(), W["wo"].abs()
    n_ws = lambda n: _gamma(n // 8 + 1 + 8)  # noqa: E731  (8 fixed slices, added in slice order)
    res = {
        "tgt2": hsum @ W["w1"],
        "e_tgt2": e_hsum @ W1 + _gamma(64) * (hsum.abs() @ W1),
        "memory": DV @ W["wv"] - DH @ W["w1"],
        "e_memory": e_DV @ Wv + e_DH @ W1 + _gamma(65) * (DV.abs() @ Wv + DH.abs() @ W1),
        "rel": dh @ W["w1"] + dv @ W["wv"],
        "e_rel": e_dh @ W1 + e_dv @ Wv + _gamma(65) * (dh.abs() @ W1 + dv.abs() @ Wv),
        "w1": dW1_r + outer(hsum, t) - outer(DH, m),
        "e_w1": e_w1_r + outer(e_hsum, t.abs()) + outer(e_DH, m.abs())
        + n_ws(3 * Q * B + C * B) * (outer(dht.abs(), rabs) + outer(hsum.abs(), t.abs()) + outer(DH.abs(), m.abs())),
        "b1": hsum.sum((0, 1)),
        "e_b1": e_hsum.sum((0, 1)) + n_ws(Q * B) * hsum.abs().sum((0, 1)),
        "w2": dW2, "e_w2": e_w2 + n_ws(Q * B) * outer(gt.abs(), ht.abs()),
        "b2": torch.zeros(64, dtype=F64, device=dW2.device), "e_b2": torch.zeros(64, dtype=F64, device=dW2.device),
        "wv": dWv_r + outer(DV, m),
        "e_wv": e_wv_r + outer(e_DV, m.abs()) + n_ws(Q * B + C * B) * (outer(dvt.abs(), rabs) + outer(DV.abs(), m.abs())),
        "bv": do.sum((0, 1)), "e_bv": e_do.sum((0, 1)) + n_ws(Q * B) * do.abs().sum((0, 1)),
        "wo": outer(dz, o), "e_wo": outer(dz.abs(), c["e_o"]) + n_ws(Q * B) * outer(dz.abs(), o.abs()),
        "bo": dz.sum((0, 1)), "e_bo": n_ws(Q * B) * dz.abs().sum((0, 1)),
    }
    return res


# ---- mask head ------------------------------------------------------------------------------------------------------
def _mh_relative_coords(geo, coords, seeds):
    """epilogue a11 as mask_head_kernel computes it: fp32 subtractions and the fp32 push of unreachable points
    (correctly rounded ops: bit-identical to the kernel).  (Q,3,N) float32"""
    geo, coords, seeds = geo.to(torch.float32), coords.to(torch.float32), seeds.to(torch.float32)
    d = seeds[:, :, None] - coords.t()[None]  # (Q,3,N)
    mx = geo.max(1).values
    mx = torch.where(mx < 0, mx.max(), mx)
    sq = torch.sqrt(mx.to(F64)).to(torch.float32)  # sqrt is correctly rounded through float64
    pushed = d + sq[:, None, None] * torch.sign(d)
    return torch.where((geo < 0)[:, None], pushed, d)


def mask_head_forward(geo, feats, w0, b0, w1, b1, coords, seeds, mode=KERNEL_TF32_MODE, *, no_tf32=False,
                      drop_feature_channel=None):
    """mask_head_kernel<false> in float64 with its TF32 operands (feats and w0[:, 3:]).
    geo (Q,N), feats (N,16), w0 (Q*16,19), b0 (Q*16), w1 (Q,16), b1 (Q), coords (N,3), seeds (Q,3)
    -> dict with out (Q,N), its bound e_out, h (Q,16,N), e_h, kink (Q,N: some hidden value within e_h of the kink)
    and the relative coordinates rel (Q,3,N)."""
    if no_tf32:
        mode = None
    Q, N = geo.shape
    M = feats.shape[1]
    rel = _mh_relative_coords(geo, coords, seeds).to(F64)
    ft = tf32_round(feats, mode)
    W0 = w0.to(F64).reshape(Q, M, M + 3)
    wf = tf32_round(w0.reshape(Q, M, M + 3)[:, :, 3:], mode)
    if drop_feature_channel is not None:
        ft = ft.clone()
        ft[:, drop_feature_channel] = 0
    d = torch.einsum("qjc,nc->qjn", wf, ft)
    sf = torch.einsum("qjc,nc->qjn", wf.abs(), ft.abs())
    B0 = b0.to(F64).reshape(Q, M, 1)
    wr = torch.einsum("qja,qan->qjn", W0[:, :, :3], rel)
    swr = torch.einsum("qja,qan->qjn", W0[:, :, :3].abs(), rel.abs())
    h = d + B0 + wr
    e_h = M * TC * sf + 4 * U * (sf + B0.abs() + swr)
    W1 = w1.to(F64).reshape(Q, M, 1)
    out = (W1 * F.relu(h)).sum(1) + b1.to(F64)[:, None]
    e_out = (W1.abs() * e_h).sum(1) + _gamma(M + 1) * ((W1.abs() * F.relu(h)).sum(1) + b1.to(F64).abs()[:, None])
    kink = (h.abs() <= e_h).any(1)
    return {"out": out, "e_out": e_out, "h": h, "e_h": e_h, "kink": kink, "rel": rel}


def mask_head_backward(fwd, feats, w0, w1, dlogit, n_ctas):
    """mask_head_kernel<true> and mask_head_bwd_finish_kernel in float64 for the forward emulation `fwd` and dlogit
    (Q,N), zero where fwd["kink"] is set (the caller's exclusion).  Only dw1 sees the TF32 product (through h); the
    ReLU masks, dfeats (raw fp32 w0[:, 3:]) and the other sums are fp32.  n_ctas: the backward's grid size.
    -> dict feats (N,16), w0 (Q*16,19), b0 (Q*16), w1 (Q,16), b1 (Q) and their bounds e_<name>."""
    h, e_h, rel = fwd["h"], fwd["e_h"], fwd["rel"]
    Q, M, N = h.shape
    g = dlogit.to(F64)
    W0 = w0.to(F64).reshape(Q, M, M + 3)
    W1 = w1.to(F64).reshape(Q, M, 1)
    f = feats.to(F64)
    x = torch.cat([rel, f.t()[None].expand(Q, M, N)], 1)  # (Q,19,N)
    dh = g[:, None] * W1 * (h > 0)
    rh = F.relu(h)
    # reduction depth over the points: warp tree, lane quarters, the CTA's tiles, the CTAs
    tiles = (N + 127) // 128
    n_pts = 5 + 3 + (tiles + n_ctas - 1) // n_ctas + n_ctas + 2
    gw = _gamma(n_pts)
    dh_abs = dh.abs()
    return {
        "feats": torch.einsum("qjn,qjc->nc", dh, W0[:, :, 3:]),
        "e_feats": (_gamma(M * Q + 4) + U) * torch.einsum("qjn,qjc->nc", dh_abs, W0[:, :, 3:].abs()),
        "w0": torch.einsum("qjn,qcn->qjc", dh, x).reshape(Q * M, M + 3),
        "e_w0": (gw + U) * torch.einsum("qjn,qcn->qjc", dh_abs, x.abs()).reshape(Q * M, M + 3),
        "b0": dh.sum(2).reshape(Q * M), "e_b0": gw * dh_abs.sum(2).reshape(Q * M),
        "w1": torch.einsum("qn,qjn->qj", g, rh),
        "e_w1": torch.einsum("qn,qjn->qj", g.abs(), e_h) + (gw + U) * torch.einsum("qn,qjn->qj", g.abs(), rh),
        "b1": g.sum(1), "e_b1": gw * g.abs().sum(1),
    }
