"""The three tensor-core kernels against their kernel-faithful float64 emulation (oracle/tf32.py).

The cross-attention forward and backward (gf_attention.cu) and the mask head (gf_mask_head.cu) multiply raw fp32
operands as TF32.  Their other tests compare against plain fp32 or float64 references, with tolerances that absorb the
whole TF32 error.  Here the reference rounds exactly the kernel's tensor-core operands to TF32 and computes the rest in
float64, and every output is held elementwise to |got - emul| <= LIMIT * bound, where the bound (oracle/tf32.py)
adds up the tensor-core accumulation, the kernel's sequential fp32 sums, __expf and the possible one-ulp TF32 flips of
rounded intermediates.  Only the backward needs an exclusion: dy is zeroed where out_mlp's pre-activation lies within
its bound of the kink (dz = dy [out > 0] could switch), and the dlogit of the mask head where a hidden value does.
Hidden-layer kinks of the attention backward need none: such a pair's whole contribution enters the bounds.

CPU: tf32_round on crafted bit patterns; with rounding off the emulations equal oracle.attention / oracle.mask_head
and autograd through them to 1e-12 in float64; each mutation of the emulation changes its result.

GPU: the rounding mode of kind::tf32 on raw fp32 operands (probe); forward out, o and lse at the context-tile
boundaries in six score regimes (flat as the other tests draw them, peaked, ascending and descending ramps, a spike in
the last tile, a spike in column half 1 of a tile); the fused forward; every gradient of the backward; mask head
forward and backward across the 16-query groups and 128-point tiles; the bounds reject emulations of wrong kernels.

Measured on a B200 (1000 W power limit, 1965 MHz max SM clock): kind::tf32 truncates raw fp32 operands (round toward
zero), on both operand sides of both kernels.  Worst |got - emul| / bound over every case below:
  attention forward   out 0.10, o 0.60, lse 0.89 (fused out 0.001)
  attention backward  drel 0.98, dmemory 0.86, dWo 0.21, dbo 0.19, the others <= 0.08
  mask head           logits 0.10; dfeats 0.22, dw0 0.21, db0 0.17, dw1 0.09, db1 0.05
A ratio near 1 is a realised flip: the allowance of a flip is the exact width of the kernel's possible operands, so one
flip that dominates an entry's bound uses it up.  The attention bounds are therefore asserted as they are (LIMIT 1),
the mask head's with a margin of about 2.5x above the worst measured ratio.  The emulated wrong kernels miss these
limits by 176x (TF32 operands not rounded) to 1e5x; the file's GPU tests take about 20 s.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import tf32

WNAMES = ("w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo")
ANAMES = ("tgt2", "memory", "rel") + WNAMES
MNAMES = ("feats", "w0", "b0", "w1", "b1")
M = 16
REGIMES = ("flat", "peaked", "ascending", "descending", "spike_last", "spike_half1")
# worst |got - emul| / bound accepted per kernel (the bounds are meant to be sound: a ratio above 1 is a finding)
LIMITS = {"att_fwd": 1.0, "att_bwd": 1.0, "mh_fwd": 0.25, "mh_bwd": 0.5}


# ---- inputs ---------------------------------------------------------------------------------------------------------
def attention_case(Q, C, B, regime, seed, dtype=torch.float32):
    """weights, tgt2, memory, rel, dy of one attention case in score regime `regime`"""
    gen = torch.Generator().manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=gen, dtype=dtype)  # noqa: E731
    w = {k: rn(64, 64) * 0.125 if k[0] == "w" else rn(64) * 0.1 for k in WNAMES}
    tgt2, mem, dy = rn(Q, B, 64), rn(C, B, 64), rn(Q, B, 64)
    rel = torch.rand(Q, C, B, 64, generator=gen, dtype=dtype) * 2 - 1
    if regime == "peaked":  # scores spanning tens of units
        w["w2"] = w["w2"] * 60
    elif regime != "flat":  # non-negative first and second layer: the scores grow with rel
        w["w1"], w["w2"] = w["w1"].abs(), w["w2"].abs()
        tgt2, mem = tgt2 * 0.1, mem * 0.1
        noise = torch.rand(Q, C, B, 64, generator=gen, dtype=dtype) * 0.05
        if regime in ("ascending", "descending"):
            ramp = torch.arange(C, dtype=dtype) * (2.0 / max(C - 1, 1))
            if regime == "descending":
                ramp = ramp.flip(0)
            rel = ramp[None, :, None, None] + noise
        else:
            rel = noise * 4
            c = C - 1 if regime == "spike_last" else max([c for c in range(C) if c % 64 >= 32], default=C - 1)
            rel[:, c] += 3.0
    return w, tgt2, mem, rel.contiguous(), dy


def mask_head_case(Q, N, seed, pattern="mixed", scale=3.0):
    gen = torch.Generator().manual_seed(seed)
    feats = torch.randn(N, M, generator=gen)
    w0 = torch.randn(Q * M, M + 3, generator=gen) * 0.3
    b0 = torch.randn(Q * M, generator=gen) * 0.1
    w1 = torch.randn(Q, M, generator=gen) * 0.3
    b1 = torch.randn(Q, generator=gen) * 0.1
    geo = torch.rand(Q, N, generator=gen) * scale
    if pattern == "mixed":
        geo[torch.rand(Q, N, generator=gen) < 0.3] = -1.0
    elif pattern == "all_but_seed":
        geo[:] = -1.0
        geo[torch.arange(Q), torch.randint(0, N, (Q,), generator=gen)] = 0.0
    elif pattern == "all":
        geo[:] = -1.0
    coords = (torch.rand(N, 3, generator=gen) - 0.5) * 8
    seeds = (torch.rand(Q, 3, generator=gen) - 0.5) * 8
    dl = torch.randn(Q, N, generator=gen)
    return geo, feats, w0, b0, w1, b1, coords, seeds, dl


def _ratio(got, want, bound, skip_nan=False):
    """max |got - want| / bound; entries with got == want count 0"""
    err = (got.to(torch.float64) - want).abs()
    if skip_nan:
        err = torch.nan_to_num(err, nan=0.0)
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return r.max().item() if r.numel() else 0.0


# ---- CPU --------------------------------------------------------------------------------------------------------------
def _bits(x):
    return torch.tensor(np.array(x, dtype=np.uint32).view(np.float32))


@pytest.mark.parametrize("mode", ["rz", "rne", "rna"])
def test_tf32_round_on_crafted_bit_patterns(mode):
    one, ulp = 0x3F800000, 0x2000  # 1.0 and one TF32 ulp in its bit pattern
    cases = {  # bits -> expected bits per mode (rz, rne, rna)
        one + 0x1800: (one, one + ulp, one + ulp),                          # 1 + 0.75 ulp
        one + 0x1000: (one, one, one + ulp),                                # exactly half, even last kept bit
        one + ulp + 0x1000: (one + ulp, one + 2 * ulp, one + 2 * ulp),      # exactly half, odd last kept bit
        one + 0x0FFF: (one, one, one),                                      # just below half
        one + ulp + 0x1001: (one + ulp, one + 2 * ulp, one + 2 * ulp),      # just above half
        0x80000000 | (one + 0x1800): (0x80000000 | one,) + (0x80000000 | (one + ulp),) * 2,  # negative
        0x80000000 | (one + 0x1000): (0x80000000 | one, 0x80000000 | one, 0x80000000 | (one + ulp)),
        one + 5 * ulp: (one + 5 * ulp,) * 3,                                # already TF32
        0x40490000: (0x40490000,) * 3,                                      # 3.140625, already TF32
        0x00000FFF: (0, 0, 0),                                              # subnormal below half an ulp
        0x00001001: (0, 0x2000, 0x2000),                                    # subnormal above half an ulp
        0x7F7FFFFF: (0x7F7FE000, 0x7F800000, 0x7F800000),                   # the largest float rounds up to inf
    }
    k = ("rz", "rne", "rna").index(mode)
    x = _bits(list(cases))
    want = _bits([v[k] for v in cases.values()]).double()
    got = tf32.tf32_round(x, mode)
    assert torch.equal(got, want), [(hex(a), float(g), float(w)) for a, g, w in zip(cases, got, want) if g != w]
    assert torch.equal(tf32.tf32_round(x.double(), mode), got)  # float64 input: cast to fp32 first
    assert torch.isnan(tf32.tf32_round(torch.tensor([float("nan")]), mode)).all()


def _att_oracle_grads(tgt2, mem, rel, w, dy):
    from oracle import attention as oatt

    leaves = [t.clone().requires_grad_() for t in (tgt2, mem, rel)] + [w[k].clone().requires_grad_() for k in WNAMES]
    y = oatt.rel_cross_attention(*leaves[:3], dict(zip(WNAMES, leaves[3:])))
    return y.detach(), dict(zip(ANAMES, torch.autograd.grad(y, leaves, dy)))


@pytest.mark.parametrize("Q,C,B,regime", [(3, 1, 1, "flat"), (5, 70, 2, "peaked"), (4, 33, 3, "ascending"),
                                          (2, 129, 1, "spike_half1")])
def test_attention_emulation_without_rounding_equals_oracle(Q, C, B, regime):
    w, tgt2, mem, rel, dy = attention_case(Q, C, B, regime, Q + C, torch.float64)
    y, want = _att_oracle_grads(tgt2, mem, rel, w, dy)
    fwd = tf32.attention_forward(tgt2, mem, rel, w, None, near_kink=True)
    scale = lambda t: max(1.0, t.abs().max().item())  # noqa: E731
    assert (fwd["out"] - y).abs().max().item() <= 1e-12 * scale(y)
    s = F.linear(F.relu(F.linear(tgt2[:, None] - mem[None] + rel, w["w1"], w["b1"])), w["w2"], w["b2"]) / 8
    v = F.linear(mem[None] + rel, w["wv"], w["bv"])
    o, lse = (torch.softmax(s, 1) * v).sum(1), torch.logsumexp(s, 1)
    assert (fwd["o"] - o).abs().max().item() <= 1e-12 * scale(o)
    assert (fwd["lse"] - lse).abs().max().item() <= 1e-12 * scale(lse)
    got = tf32.attention_backward(fwd, dy)
    for k in ANAMES:
        assert got[k].shape == want[k].shape, k
        err = (got[k] - want[k]).abs().max().item()
        assert err <= 1e-12 * scale(want[k]), (k, err)


def _dyadic_mask_head_case(Q, N, seed):
    """coordinates on a 2^-8 grid and row maxima 4 or 9: the kernel's fp32 relative coordinates are exact, so the
    float64 oracle and the emulation see the same values"""
    geo, feats, w0, b0, w1, b1, _, _, dl = mask_head_case(Q, N, seed)
    gen = torch.Generator().manual_seed(seed + 1)
    coords = torch.randint(-1024, 1024, (N, 3), generator=gen).float() / 256
    seeds = torch.randint(-1024, 1024, (Q, 3), generator=gen).float() / 256
    geo[:, 0] = torch.where(torch.arange(Q) % 2 == 0, 4.0, 9.0)
    return geo, feats, w0, b0, w1, b1, coords, seeds, dl


@pytest.mark.parametrize("Q,N", [(1, 1), (3, 70), (17, 129)])
def test_mask_head_emulation_without_rounding_equals_oracle(Q, N):
    from oracle.mask_head import mask_heads_forward

    geo, feats, w0, b0, w1, b1, coords, seeds, dl = _dyadic_mask_head_case(Q, N, Q * 10 + N)
    d = torch.float64
    leaves = [t.to(d).requires_grad_() for t in (feats, w0, b0, w1, b1)]
    y = mask_heads_forward(geo.to(d), leaves[0], [leaves[1].reshape(Q * M, M + 3, 1), leaves[3].reshape(Q, M, 1)],
                           [leaves[2], leaves[4]], Q, coords.to(d), seeds.to(d))
    want = dict(zip(MNAMES, torch.autograd.grad(y, leaves, dl.to(d))))
    fwd = tf32.mask_head_forward(geo, feats, w0, b0, w1, b1, coords, seeds, None)
    assert (fwd["out"] - y).abs().max().item() <= 1e-12 * max(1.0, y.abs().max().item())
    got = tf32.mask_head_backward(fwd, feats, w0, w1, dl, 1)
    for k in MNAMES:
        assert got[k].shape == want[k].shape, k
        err = (got[k] - want[k]).abs().max().item()
        assert err <= 1e-12 * max(1.0, want[k].abs().max().item()), (k, err)


ATT_MUTATIONS = {  # mutation -> (Q, C, B, regime) on which it must miss the bounds
    "drop_last_context": [(4, 33, 1, "flat"), (4, 65, 1, "flat"), (4, 129, 2, "flat")],
    "no_rescale": [(4, 300, 1, "ascending")],
    "lse_half0": [(4, 129, 1, "spike_half1")],
    "b2_unscaled": [(4, 129, 1, "flat")],
    "no_tf32": [(4, 129, 1, "spike_last")],  # non-negative operands: truncation errors add up
}
MH_MUTATIONS = {"drop_feature_channel": 5, "no_tf32": True}


@pytest.mark.parametrize("mutation", list(ATT_MUTATIONS))
def test_each_attention_mutation_changes_the_result(mutation):
    for Q, C, B, regime in ATT_MUTATIONS[mutation]:
        w, tgt2, mem, rel, _ = attention_case(Q, C, B, regime, C)
        a = tf32.attention_forward(tgt2, mem, rel, w)
        b = tf32.attention_forward(tgt2, mem, rel, w, **{mutation: True})
        assert not torch.equal(a["o"], b["o"]) or not torch.equal(a["lse"], b["lse"]), (mutation, C)


@pytest.mark.parametrize("mutation", list(MH_MUTATIONS))
def test_each_mask_head_mutation_changes_the_result(mutation):
    geo, feats, w0, b0, w1, b1, coords, seeds, _ = mask_head_case(17, 300, 3)
    a = tf32.mask_head_forward(geo, feats, w0, b0, w1, b1, coords, seeds)
    b = tf32.mask_head_forward(geo, feats, w0, b0, w1, b1, coords, seeds, **{mutation: MH_MUTATIONS[mutation]})
    assert not torch.equal(a["out"], b["out"])


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev(cuda_lib):
    return torch.device("cuda:0")


def att_save(tgt2, mem, rel, w, dev):
    """gf_rel_cross_attention_save: out, o, lse of the kernel"""
    from geoformer_b200 import _capi as C

    Q, Cn, B = tgt2.shape[0], mem.shape[0], tgt2.shape[1]
    f = lambda t: t.to(dev, torch.float32).contiguous()  # noqa: E731
    tgt2, mem, rel = f(tgt2), f(mem), f(rel)
    w = {k: f(v) for k, v in w.items()}
    out, o, lse = [torch.empty(Q, B, 64, device=dev) for _ in range(3)]
    L = C.lib()
    nbytes = L.gf_rel_cross_attention_workspace_bytes(Q, Cn, B)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    C.check(L.gf_rel_cross_attention_save(C.ptr(tgt2), C.ptr(mem), C.ptr(rel), Q, Cn, B, *[C.ptr(w[k]) for k in WNAMES],
                                          C.ptr(out), C.ptr(o), C.ptr(lse), C.ptr(ws), nbytes, C.stream_of(dev)),
            "rel_cross_attention_save")
    torch.cuda.synchronize(dev)
    return out, o, lse


def _mh_call(geo, feats, w0, b0, w1, b1, coords, seeds):
    from geoformer_b200.mask_head import mask_heads_forward

    Q = geo.shape[0]
    return mask_heads_forward(geo, feats, [w0.reshape(Q * M, M + 3, 1), w1.reshape(Q, M, 1)], [b0, b1], Q, coords,
                              seeds)


def _observed_mode(got, x):
    """which rounding of x the kernel's values `got` are (x: the probed fp32 values)"""
    found = [m for m in ("rz", "rne", "rna") if torch.equal(got.double().cpu(), tf32.tf32_round(x, m))]
    assert len(found) == 1, (got.tolist(), found)
    return found[0]


PROBE = _bits([0x3F800000 + 0x1800, 0x3F800000 + 0x1000, 0x3F800000 + 0x3000, 0xBF800000 + 0x1800,
               0xBF800000 + 0x1000, 0xBF800000 + 0x3000])  # 1 + 0.75, 0.5, 1.5 ulp and their negatives


@pytest.mark.gpu
def test_tf32_rounding_mode_probe(dev):
    """One directed call per operand side settles how kind::tf32 treats the 13 low bits of a raw fp32 operand: with
    C = 1 the softmax weight is exactly 1, so o = Wv rel + bv, read back exactly through the saved o."""
    n = PROBE.numel()
    modes = []
    for side in ("rel", "wv"):
        w = {k: torch.zeros(64, 64) if k[0] == "w" else torch.zeros(64) for k in WNAMES}
        w["wo"] = torch.eye(64)
        rel = torch.zeros(1, 1, 1, 64)
        for i in range(n):  # channel i of v reads operand entry (i, 10 + i)
            if side == "rel":
                w["wv"][i, 10 + i], rel[0, 0, 0, 10 + i] = 1.0, PROBE[i]
            else:
                w["wv"][i, 10 + i], rel[0, 0, 0, 10 + i] = PROBE[i], 1.0
        _, o, _ = att_save(torch.zeros(1, 1, 64), torch.zeros(1, 1, 64), rel, w, dev)
        modes.append(_observed_mode(o[0, 0, :n], PROBE))
    for side in ("feats", "w0"):  # mask head: one-hot weight rows, w1 = 1, everything else zero
        Q, N = 1, n
        feats, w0 = torch.zeros(N, M), torch.zeros(Q * M, M + 3)
        for i in range(n):  # point i reads feature channel i; hidden channel i of the one query takes it
            if side == "feats":
                feats[i, i], w0[i, 3 + i] = PROBE[i].abs(), 1.0
            else:
                feats[i, i], w0[i, 3 + i] = 1.0, PROBE[i].abs()
        w1 = torch.zeros(Q, M)
        w1[0, :n] = 1.0
        z = lambda *s: torch.zeros(*s, device=dev)  # noqa: E731
        out = _mh_call(torch.ones(Q, N, device=dev), feats.to(dev), w0.to(dev), z(Q * M), w1.to(dev), z(Q),
                       z(N, 3), z(Q, 3))
        modes.append(_observed_mode(out[0], PROBE.abs()))
    print("kind::tf32 rounding of raw fp32 operands (rel, Wv, feats, w0):", modes)
    assert modes == [tf32.KERNEL_TF32_MODE] * 4, modes


ATT_C = (1, 31, 32, 33, 63, 64, 65, 127, 128, 129, 2048, 2049)
ATT_QB = ((1, 1), (3, 3), (37, 1), (256, 3))


def _check_att_forward(w, tgt2, mem, rel, dev, what):
    out, o, lse = att_save(tgt2, mem, rel, w, dev)
    e = tf32.attention_forward(*[t.to(dev) for t in (tgt2, mem, rel)], {k: v.to(dev) for k, v in w.items()})
    r = {k: _ratio(g, e[k], e["e_" + k]) for k, g in (("out", out), ("o", o), ("lse", lse))}
    print("%s: |err| / bound out %.3g o %.3g lse %.3g" % (what, r["out"], r["o"], r["lse"]))
    assert max(r.values()) <= LIMITS["att_fwd"], (what, r)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("C", ATT_C)
def test_attention_forward_matches_tf32_emulation(dev, C, regime):
    for Q, B in ATT_QB:
        w, tgt2, mem, rel, _ = attention_case(Q, C, B, regime, Q * 1000 + C)
        _check_att_forward(w, tgt2, mem, rel, dev, "Q=%d C=%d B=%d %s" % (Q, C, B, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 8])
def test_fused_attention_forward_matches_tf32_emulation(dev, B):
    """the fused kernel builds the embedding the library's decoder_relative_embedding writes, bit for bit
    (test_gpu_attention.py), so that tensor is the emulation's rel"""
    from geoformer_b200.attention import rel_cross_attention_fused
    from geoformer_b200.bias import decoder_relative_embedding
    from geoformer_b200.scenes import scene

    Q, Cn = 40, 300
    gen = torch.Generator().manual_seed(B)
    Ns = [3000 + 500 * b for b in range(B)]
    xs = [scene(n, 80 + b) for b, n in enumerate(Ns)]
    geos = []
    for n in Ns:
        g = torch.rand(Q, n, generator=gen) * 4.0
        g[torch.rand(Q, n, generator=gen) < 0.5] = -1.0
        g[1] = -1.0
        geos.append(g.to(dev))
    inds = torch.stack([torch.randperm(n, generator=gen)[:Cn] for n in Ns]).int().to(dev)
    ctx = torch.stack([x[i.long().cpu()] for x, i in zip(xs, inds)]).contiguous().to(dev)
    qry = ctx[:, :Q].contiguous()
    gb = torch.randn(3, 32, generator=gen).to(dev)
    pc = [torch.stack([x.min(0)[0] for x in xs]).to(dev), torch.stack([x.max(0)[0] for x in xs]).to(dev)]
    w = {k: v.to(dev) for k, v in attention_case(1, 1, 1, "flat", B)[0].items()}
    tgt2, mem = torch.randn(Q, B, 64, generator=gen).to(dev), torch.randn(Cn, B, 64, generator=gen).to(dev)
    with torch.no_grad():
        out = rel_cross_attention_fused(tgt2, mem, geos, inds, qry, ctx, gb, pc, w)
        emb = decoder_relative_embedding(geos, inds, qry, ctx, gb, pc).contiguous()
    e = tf32.attention_forward(tgt2, mem, emb, w)
    r = _ratio(out, e["out"], e["e_out"])
    print("fused B=%d: |err| / bound out %.3g" % (B, r))
    assert r <= LIMITS["att_fwd"], r


def _att_kernel_grads(w, tgt2, mem, rel, dy, dev):
    from geoformer_b200.attention import rel_cross_attention

    leaves = {k: v.to(dev).clone().requires_grad_() for k, v in w.items()}
    ins = [t.to(dev).clone().requires_grad_() for t in (tgt2, mem, rel)]
    y = rel_cross_attention(*ins, leaves)
    return dict(zip(ANAMES, torch.autograd.grad(y, ins + [leaves[k] for k in WNAMES], dy.to(dev))))


def _check_att_backward(w, tgt2, mem, rel, dy, dev, what):
    wd = {k: v.to(dev) for k, v in w.items()}
    fwd = tf32.attention_forward(tgt2.to(dev), mem.to(dev), rel.to(dev), wd, near_kink=True)
    dy = torch.where(fwd["kink_out"], torch.zeros_like(dy.to(dev)), dy.to(dev))
    want = tf32.attention_backward(fwd, dy)
    del fwd
    got = _att_kernel_grads(w, tgt2, mem, rel, dy.float(), dev)
    r = {}
    for k in ANAMES:
        if k == "b2":
            assert not got[k].any(), "db2 must be exactly zero"
            continue
        r[k] = _ratio(got[k], want[k], want["e_" + k])
    print("%s: |err| / bound %s" % (what, " ".join("%s %.3g" % kv for kv in r.items())))
    assert max(r.values()) <= LIMITS["att_bwd"], (what, r)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("regime", REGIMES)
@pytest.mark.parametrize("C", ATT_C)
def test_attention_backward_matches_tf32_emulation(dev, C, regime):
    for Q, B in ((3, 3), (37, 1)):
        w, tgt2, mem, rel, dy = attention_case(Q, C, B, regime, Q * 1000 + C + 1)
        _check_att_backward(w, tgt2, mem, rel, dy, dev, "Q=%d C=%d B=%d %s" % (Q, C, B, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["full", "rel0", "mem0"])
def test_attention_backward_training_shape_matches_tf32_emulation(dev, case):
    Q, C, B = 128, 2048, 4
    w, tgt2, mem, rel, dy = attention_case(Q, C, B, "flat", 7)
    if case == "rel0":
        rel.zero_()
    if case == "mem0":
        mem.zero_()
    _check_att_backward(w, tgt2, mem, rel, dy, dev, "training shape %s" % case)


MH_Q = (1, 15, 16, 17, 31, 32, 33, 256, 257)
MH_N = (1, 127, 128, 129, 4099, 100_003)


def _check_mh(case, dev, what, backward=True, nan_expected=False):
    geo, feats, w0, b0, w1, b1, coords, seeds, dl = [t.to(dev) for t in case]
    args = (feats, w0, b0, w1, b1)
    with torch.no_grad():
        out = _mh_call(geo, *args, coords, seeds)
    e = tf32.mask_head_forward(geo, *args, coords, seeds)
    nan_g, nan_w = torch.isnan(out), torch.isnan(e["out"])
    assert torch.equal(nan_g, nan_w), (what, nan_g.sum().item(), nan_w.sum().item())
    if nan_expected:
        assert bool(nan_w.all()), what
        return {}
    r = {"out": _ratio(out, e["out"], e["e_out"], skip_nan=True)}
    if backward:
        dl = torch.where(e["kink"], torch.zeros_like(dl), dl)
        leaves = [t.clone().requires_grad_() for t in args]
        y = _mh_call(geo, *leaves, coords, seeds)
        got = dict(zip(MNAMES, torch.autograd.grad(y, leaves, dl)))
        n_ctas = min((geo.shape[1] + 127) // 128, torch.cuda.get_device_properties(dev).multi_processor_count)
        want = tf32.mask_head_backward(e, feats, w0, w1, dl, n_ctas)
        for k in MNAMES:
            r[k] = _ratio(got[k], want[k], want["e_" + k])
    print("%s: |err| / bound %s" % (what, " ".join("%s %.3g" % kv for kv in r.items())))
    assert r["out"] <= LIMITS["mh_fwd"], (what, r)
    assert max([v for k, v in r.items() if k != "out"], default=0.0) <= LIMITS["mh_bwd"], (what, r)
    return r


@pytest.mark.gpu
@pytest.mark.parametrize("N", MH_N)
def test_mask_head_matches_tf32_emulation(dev, N):
    for Q in MH_Q:
        if Q * N > 257 * 5000 and Q not in (17, 33):
            continue  # the largest scenes at two query counts, one of them a partial group
        _check_mh(mask_head_case(Q, N, Q * 7 + N), dev, "Q=%d N=%d" % (Q, N))


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["none", "all_but_seed", "mixed_large_rowmax", "all"])
def test_mask_head_unreachable_patterns_match_tf32_emulation(dev, pattern):
    Q, N = 37, 5003
    if pattern == "mixed_large_rowmax":  # sqrt(rowmax) = 100 against coordinates within 4 m
        case = mask_head_case(Q, N, 5, "mixed", scale=1e4)
    else:
        case = mask_head_case(Q, N, 5, pattern)
    case = list(case)
    case[7] = case[6][torch.randint(0, N, (Q,), generator=torch.Generator().manual_seed(6))].contiguous()
    if pattern != "all":
        case[0][:, 0] = case[0][:, 0].abs()  # a reachable point in every row for the backward
    _check_mh(case, dev, pattern, backward=pattern != "all", nan_expected=pattern == "all")


# ---- the bounds catch wrong kernels ------------------------------------------------------------------------------------
OLD_ATT_TOL = dict(rtol=4e-3, atol=4e-3)  # test_gpu_attention.py against the fp32 oracle


@pytest.mark.gpu
@pytest.mark.parametrize("mutation", list(ATT_MUTATIONS))
def test_bounds_reject_attention_mutations(dev, mutation):
    """the emulation of a wrong kernel misses the new bounds by at least 10x LIMIT; whether it would have passed the
    fp32-oracle tolerance of test_gpu_attention.py is printed, not asserted"""
    from oracle import attention as oatt

    for Q, C, B, regime in ATT_MUTATIONS[mutation]:
        w, tgt2, mem, rel, _ = attention_case(Q, C, B, regime, C)
        ins = [t.to(dev) for t in (tgt2, mem, rel)]
        wd = {k: v.to(dev) for k, v in w.items()}
        e = tf32.attention_forward(*ins, wd)
        bad = tf32.attention_forward(*ins, wd, **{mutation: True})
        bad_out = F.relu(bad["o"] @ e["_ctx"]["W"]["wo"].t() + e["_ctx"]["W"]["bo"])
        factor = max(_ratio(bad["o"], e["o"], e["e_o"]), _ratio(bad["lse"], e["lse"], e["e_lse"]),
                     _ratio(bad_out, e["out"], e["e_out"])) / LIMITS["att_fwd"]
        ref = oatt.rel_cross_attention(*[t.float() for t in ins], {k: v.float() for k, v in wd.items()}).double()
        old_pass = bool(((bad_out - ref).abs() <= OLD_ATT_TOL["atol"] + OLD_ATT_TOL["rtol"] * ref.abs()).all())
        print("mutation %s C=%d %s: misses the new bound by %.3g x; old fp32-oracle tolerance would %s it"
              % (mutation, C, regime, factor, "accept" if old_pass else "reject"))
        assert factor >= 10, (mutation, C, factor)


@pytest.mark.gpu
@pytest.mark.parametrize("mutation", list(MH_MUTATIONS))
def test_bounds_reject_mask_head_mutations(dev, mutation):
    Q, N = 33, 4099
    geo, feats, w0, b0, w1, b1, coords, seeds, _ = [t.to(dev) for t in mask_head_case(Q, N, 3)]
    e = tf32.mask_head_forward(geo, feats, w0, b0, w1, b1, coords, seeds)
    bad = tf32.mask_head_forward(geo, feats, w0, b0, w1, b1, coords, seeds, **{mutation: MH_MUTATIONS[mutation]})
    factor = _ratio(bad["out"], e["out"], e["e_out"]) / LIMITS["mh_fwd"]
    # the float64 bound of test_mask_head.py: 4e-3 S_f + 1e-5 S + 1e-6
    d = torch.float64
    rel = e["rel"]
    W0, f, a1 = w0.to(d).reshape(Q, M, M + 3), feats.to(d), w1.to(d).reshape(Q, M, 1).abs()
    ref = F.relu(torch.einsum("qjc,nc->qjn", W0[:, :, 3:], f) + torch.einsum("qja,qan->qjn", W0[:, :, :3], rel)
                 + b0.to(d).reshape(Q, M, 1))
    ref = (w1.to(d).reshape(Q, M, 1) * ref).sum(1) + b1.to(d)[:, None]
    sf = (a1 * torch.einsum("qjc,nc->qjn", W0[:, :, 3:].abs(), f.abs())).sum(1)
    s = sf + (a1 * (b0.to(d).reshape(Q, M, 1).abs() + torch.einsum("qja,qan->qjn", W0[:, :, :3].abs(), rel.abs()))).sum(1)
    old_pass = bool(((bad["out"] - ref).abs() <= 4e-3 * sf + 1e-5 * (s + b1.to(d).abs()[:, None]) + 1e-6).all())
    print("mutation %s: misses the new bound by %.3g x; old float64 tolerance would %s it"
          % (mutation, factor, "accept" if old_pass else "reject"))
    assert factor >= 10, (mutation, factor)
