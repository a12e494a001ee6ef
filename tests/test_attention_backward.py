"""Backward of the decoder's vector cross-attention.

CPU: the factored backward oracle (rel_cross_attention_backward below, test infrastructure) equals autograd through
the forward oracle oracle.attention.rel_cross_attention (pinned to the reference layer) in float64; the new C entries validate their arguments before any CUDA call; the
backward kernel multiplies on the tensor cores (UTCHMMA in its SASS).

GPU: every gradient of the tcgen05 backward against the fp32 oracle, including the cases rel = 0 and memory = 0 in
which the per-pair terms and the factored t / m terms of dW1 / dWv dominate in turn; determinism; the saving forward
is bitwise the inference forward; fused == unfused; the decoder of FewShotForward trained through both paths.
Tolerance (max |g - g_ref| / max |g_ref|, relative Frobenius error), measured on a B200 over the oracle cases below
with dy zeroed where the two forwards disagree on out_mlp's ReLU (_same_relu_side):
  memory, w2, wv, bv, wo, bo   <= 9.7e-3, 2.0e-3     asserted at 2e-2, 5e-3
  tgt2, b1, w1                 <= 3.0e-2, 1.5e-2     asserted at 6e-2, 3e-2
  rel                          <= 4.9e-2, 1.4e-3     asserted at 1e-1, 5e-3
The products are TF32 (10 mantissa bits) like the forward's, whose error is 2e-3 of the output scale.  tgt2, b1 and
w1 go through Hsum_q = sum_c dh, a sum over the contexts of terms that largely cancel (sum_c a (v - o) = 0 exactly),
so their relative error is that of the terms times the cancellation.  rel is per pair: a pair whose hidden
pre-activation lies within TF32 rounding of ReLU's kink flips its mask, a few isolated entries (hence the small
Frobenius error).  A missing term gives errors of order 1; the rel = 0 and memory = 0 cases make each term of dW1 /
dWv dominant in turn.  These tolerances tie the backward to the reference model; its arithmetic is pinned by elementwise
bounds against the TF32-exact float64 emulation oracle/tf32.py (tests/test_tf32_reference.py)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
NAMES = ("tgt2", "memory", "rel", "w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo")
WNAMES = NAMES[3:]
TOL = {"tgt2": (6e-2, 3e-2), "b1": (6e-2, 3e-2), "w1": (6e-2, 3e-2), "rel": (1e-1, 5e-3)}  # (max, Frobenius)
TOL_DEFAULT = (2e-2, 5e-3)


def rel_cross_attention_backward(tgt2, memory, relative_pos, w, dy):
    """Gradients of oracle.attention.rel_cross_attention for the upstream gradient dy (Q,B,64), written in the
    factored form the backward kernel computes (the t and m parts of x = t - m + r summed out of the per-pair sums):
        dz = dy [y > 0], do = Wo^T dz, dv = a do, g = a do (v - o) / 8, dh = (W2^T g) [hp > 0]
        Hsum_q = sum_c dh, DH_c = sum_q dh, DV_c = sum_q dv
        dtgt2 = W1^T Hsum, dmemory = Wv^T DV - W1^T DH, drel = W1^T dh + Wv^T dv
        dW1 = sum dh r^T + sum_q Hsum t^T - sum_c DH m^T, dWv = sum dv r^T + sum_c DV m^T, dW2 = sum g h^T
    -> dict with tgt2, memory, rel and the eight weight names.  db2 = sum g is zero up to rounding (the softmax is
    shift invariant per channel); it is returned as computed."""
    t, m, r = tgt2[:, None], memory[None], relative_pos
    hp = F.linear(t - m + r, w["w1"], w["b1"])
    h = F.relu(hp)
    a = F.softmax(F.linear(h, w["w2"], w["b2"]) / 8, dim=1)
    v = F.linear(m + r, w["wv"], w["bv"])
    o = (a * v).sum(1)  # (Q,B,64)
    y = F.relu(F.linear(o, w["wo"], w["bo"]))
    dz = dy * (y > 0)
    do = dz @ w["wo"]
    dv = a * do[:, None]
    g = dv * (v - o[:, None]) / 8
    dh = (g @ w["w2"]) * (hp > 0)
    hsum, DH, DV = dh.sum(1), dh.sum(0), dv.sum(0)
    outer = lambda x, y: torch.einsum("...i,...j->ij", x, y)  # noqa: E731
    return {"tgt2": hsum @ w["w1"], "memory": DV @ w["wv"] - DH @ w["w1"], "rel": dh @ w["w1"] + dv @ w["wv"],
            "w1": outer(dh, r) + outer(hsum, tgt2) - outer(DH, memory), "b1": hsum.sum((0, 1)),
            "w2": outer(g, h), "b2": g.sum((0, 1, 2)),
            "wv": outer(dv, r) + outer(DV, memory), "bv": do.sum((0, 1)),
            "wo": outer(dz, o), "bo": dz.sum((0, 1))}


def _rand_weights(gen, scale=0.125, dtype=torch.float32):
    return {k: (torch.randn(64, 64, generator=gen, dtype=dtype) * scale if k[0] == "w"
                else torch.randn(64, generator=gen, dtype=dtype) * 0.1) for k in WNAMES}


def _autograd_grads(tgt2, mem, rel, w, dy):
    from oracle import attention as oatt

    leaves = [t.clone().requires_grad_() for t in (tgt2, mem, rel)] + [w[k].clone().requires_grad_() for k in WNAMES]
    y = oatt.rel_cross_attention(*leaves[:3], dict(zip(WNAMES, leaves[3:])))
    return dict(zip(NAMES, torch.autograd.grad(y, leaves, dy)))


def _assert_oracle_equals_autograd(tgt2, mem, rel, w, dy):
    want = _autograd_grads(tgt2, mem, rel, w, dy)
    got = rel_cross_attention_backward(tgt2, mem, rel, w, dy)
    for k in NAMES:
        assert got[k].shape == want[k].shape, k
        err = (got[k] - want[k]).abs().max().item()
        assert err <= 1e-10 * max(1.0, want[k].abs().max().item()), (k, err)


def test_oracle_backward_equals_autograd_on_reference_fixture():
    g = np.load(os.path.join(HERE, "golden", "attention_golden.npz"))
    T = lambda a: torch.from_numpy(np.array(a)).double()  # noqa: E731
    gen = torch.Generator().manual_seed(3)
    for i in range(int(g["n"])):
        w = {k: T(g["c%d_%s" % (i, k)]) for k in WNAMES}
        tgt2, mem, rel = T(g["c%d_tgt2" % i]), T(g["c%d_memory" % i]), T(g["c%d_rel" % i])
        dy = torch.randn(tgt2.shape, generator=gen, dtype=torch.float64)
        _assert_oracle_equals_autograd(tgt2, mem, rel, w, dy)


@pytest.mark.parametrize("Q,C,B", [(1, 1, 1), (3, 70, 2), (9, 5, 3), (17, 33, 1)])
def test_oracle_backward_equals_autograd_ragged(Q, C, B):
    gen = torch.Generator().manual_seed(Q * 100 + C)
    d = torch.float64
    w = _rand_weights(gen, dtype=d)
    tgt2, mem = torch.randn(Q, B, 64, generator=gen, dtype=d), torch.randn(C, B, 64, generator=gen, dtype=d)
    rel = torch.rand(Q, C, B, 64, generator=gen, dtype=d) * 2 - 1
    _assert_oracle_equals_autograd(tgt2, mem, rel, w, torch.randn(Q, B, 64, generator=gen, dtype=d))


def test_backward_entries_validate_before_any_cuda_call(cuda_lib):
    L = cuda_lib
    assert L.gf_rel_cross_attention_backward_workspace_bytes(0, 10, 1) == 0
    assert L.gf_rel_cross_attention_backward_workspace_bytes(4, 10, 2) >= 4 * 4 * 2 * 10 * 128
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below fails its checks first
    w = [fake] * 8
    rc = L.gf_rel_cross_attention_backward(fake, fake, fake, 0, 5, 1, *w, fake, fake, fake, fake, fake, fake, None,
                                           *w, fake, 1 << 20, None)
    assert rc == 1 and b"Q, C, B >= 1" in L.gf_last_error()
    rc = L.gf_rel_cross_attention_backward(fake, fake, fake, 2, 5, 1, *w, fake, None, fake, fake, fake, fake, None,
                                           *w, fake, 1 << 20, None)
    assert rc == 1 and b"null pointer" in L.gf_last_error()
    rc = L.gf_rel_cross_attention_backward(fake, fake, None, 2, 5, 1, *w, fake, fake, fake, fake, fake, fake, None,
                                           *w, fake, 1 << 20, None)
    assert rc == 1 and b"null relative_pos" in L.gf_last_error()
    geo = [fake] * 8
    rc = L.gf_rel_cross_attention_fused_backward(*geo, 32, fake, fake, 2, 5, 9, *w, fake, fake, fake, fake, fake, fake,
                                                 *w, fake, 1 << 20, None)
    assert rc == 1 and b"at most 8" in L.gf_last_error()
    rc = L.gf_rel_cross_attention_fused_backward(*geo, 32, fake, fake, 2, 5, 1, *w, fake, fake, None, fake, fake, fake,
                                                 *w, fake, 1 << 20, None)
    assert rc == 1 and b"null pointer" in L.gf_last_error()
    rc = L.gf_rel_cross_attention_save(fake, fake, fake, 2, 5, 1, *w, fake, None, fake, fake, 1 << 20, None)
    assert rc == 1 and b"null pointer" in L.gf_last_error()
    rc = L.gf_rel_cross_attention_fused_save(*geo, 16, fake, fake, 2, 5, 1, *w, fake, fake, fake, fake, 1 << 20, None)
    assert rc == 1 and b"32 frequencies" in L.gf_last_error()


def test_backward_kernel_runs_on_the_tensor_cores(cuda_lib):
    from geoformer_b200 import _capi

    tool = "cuobjdump" if subprocess.run(["which", "cuobjdump"], capture_output=True).returncode == 0 \
        else "/usr/local/cuda/bin/cuobjdump"
    sass = subprocess.run([tool, "-sass", _capi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    per_fn, cur = {}, None
    for line in sass.splitlines():
        if "Function :" in line:
            cur = line.split("Function :")[1].strip()
            per_fn[cur] = 0
        elif cur and "UTCHMMA" in line:
            per_fn[cur] += 1
    bwd = {f: n for f, n in per_fn.items() if "rel_cross_attention_bwd_kernel" in f}
    assert len(bwd) == 2 and all(n > 0 for n in bwd.values()), bwd


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev(cuda_lib):
    return torch.device("cuda:0")


def _assert_grad_close(k, got, want, what="", tol=None):
    tol_max, tol_fro = tol or TOL.get(k, TOL_DEFAULT)
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    scale = want.abs().max().item()
    emax = (got - want).abs().max().item() / scale
    efro = ((got - want).norm() / want.norm()).item()
    print("%s %-6s max %.2e fro %.2e scale %.3g" % (what, k, emax, efro, scale))
    assert emax <= tol_max and efro <= tol_fro, (what, k, emax, efro)


def _kernel_grads(tgt2, mem, rel, w, dy, dev, fused_args=None):
    """all gradients of the library op via autograd, on `dev`"""
    from geoformer_b200.attention import rel_cross_attention, rel_cross_attention_fused

    leaves = {k: v.to(dev).clone().requires_grad_() for k, v in w.items()}
    t, m = tgt2.to(dev).requires_grad_(), mem.to(dev).requires_grad_()
    if fused_args is None:
        r = rel.to(dev).requires_grad_()
        y = rel_cross_attention(t, m, r, leaves)
        ins = [t, m, r]
    else:
        y = rel_cross_attention_fused(t, m, *fused_args, leaves)
        ins = [t, m]
    g = torch.autograd.grad(y, ins + [leaves[k] for k in WNAMES], dy.to(dev))
    return dict(zip(NAMES if fused_args is None else NAMES[:2] + WNAMES, g)), y


def _inputs(Q, C, B, seed):
    gen = torch.Generator().manual_seed(seed)
    w = _rand_weights(gen)
    tgt2, mem = torch.randn(Q, B, 64, generator=gen), torch.randn(C, B, 64, generator=gen)
    rel = torch.rand(Q, C, B, 64, generator=gen) * 2 - 1
    return w, tgt2, mem, rel, torch.randn(Q, B, 64, generator=gen)


def _same_relu_side(dy, tgt2, mem, rel, w, dev):
    """dy with zeros where the TF32 forward and the fp32 oracle put the output on different sides of out_mlp's ReLU:
    there dz = dy [y > 0] switches between dy and 0, a difference of the size of dy that says nothing about the
    backward (a handful of the Q*B*64 outputs lie within the forward's 2e-3 of the kink)"""
    from oracle import attention as oatt

    from geoformer_b200.attention import rel_cross_attention

    with torch.no_grad():
        y = rel_cross_attention(tgt2.to(dev), mem.to(dev), rel.to(dev), {k: v.to(dev) for k, v in w.items()}).cpu()
    return torch.where((y > 0) == (oatt.rel_cross_attention(tgt2, mem, rel, w) > 0), dy, torch.zeros_like(dy))


@pytest.mark.gpu
@pytest.mark.parametrize("Q,C,B", [(256, 2048, 1), (37, 301, 2), (3, 1, 1), (5, 129, 3)])
@pytest.mark.parametrize("case", ["full", "rel0", "mem0"])
def test_backward_matches_fp32_oracle(dev, Q, C, B, case):
    w, tgt2, mem, rel, dy = _inputs(Q, C, B, Q * 7 + C)
    if case == "rel0":
        rel.zero_()
    if case == "mem0":
        mem.zero_()
    dy = _same_relu_side(dy, tgt2, mem, rel, w, dev)
    want = rel_cross_attention_backward(tgt2, mem, rel, w, dy)
    got, _ = _kernel_grads(tgt2, mem, rel, w, dy, dev)
    for k in NAMES:
        if k == "b2":
            assert not got[k].any(), "db2 must be exactly zero"
            assert want[k].abs().max().item() <= 1e-5 * want["w2"].abs().max().item() + 1e-6
            continue
        if case == "rel0" and k == "rel" or want[k].abs().max().item() == 0:
            continue
        _assert_grad_close(k, got[k], want[k], "%s %s" % ((Q, C, B), case))


@pytest.mark.gpu
def test_backward_is_deterministic_and_forward_unchanged(dev):
    from geoformer_b200.attention import rel_cross_attention

    w, tgt2, mem, rel, dy = _inputs(64, 700, 2, 11)
    a, ya = _kernel_grads(tgt2, mem, rel, w, dy, dev)
    b, yb = _kernel_grads(tgt2, mem, rel, w, dy, dev)
    for k in NAMES:
        assert torch.equal(a[k], b[k]), k
    with torch.no_grad():
        y0 = rel_cross_attention(tgt2.to(dev), mem.to(dev), rel.to(dev), {k: v.to(dev) for k, v in w.items()})
    assert torch.equal(ya.detach(), y0) and torch.equal(yb.detach(), y0)


def _fused_case(dev, Q, Cn, B, gen):
    from geoformer_b200.scenes import scene

    Ns = [3000 + 500 * b for b in range(B)]
    xs = [scene(n, 80 + b) for b, n in enumerate(Ns)]
    geos = []
    for n in Ns:
        gq = torch.rand(Q, n, generator=gen) * 4.0
        gq[torch.rand(Q, n, generator=gen) < 0.5] = -1.0
        gq[1] = -1.0  # a query that reaches nothing: the embedding falls back to the coordinate distances
        geos.append(gq.to(dev))
    inds = torch.stack([torch.randperm(n, generator=gen)[:Cn] for n in Ns]).int()
    ctx = torch.stack([x[i.long()] for x, i in zip(xs, inds)]).contiguous()
    qry = ctx[:, :Q].contiguous()
    gb = torch.randn(3, 32, generator=gen)
    pc = [torch.stack([x.min(0)[0] for x in xs]).to(dev), torch.stack([x.max(0)[0] for x in xs]).to(dev)]
    return [geos, inds.to(dev), qry.to(dev), ctx.to(dev), gb.to(dev), pc]


@pytest.mark.gpu
@pytest.mark.parametrize("Q,Cn,B", [(40, 300, 8), (256, 2048, 1)])
def test_fused_backward_equals_unfused_on_our_embedding(dev, Q, Cn, B):
    from geoformer_b200.bias import decoder_relative_embedding

    gen = torch.Generator().manual_seed(Q + B)
    args = _fused_case(dev, Q, Cn, B, gen)
    w = _rand_weights(gen)
    tgt2, mem, dy = torch.randn(Q, B, 64, generator=gen), torch.randn(Cn, B, 64, generator=gen), torch.randn(Q, B, 64, generator=gen)
    emb = decoder_relative_embedding(*args).contiguous()
    a, ya = _kernel_grads(tgt2, mem, emb, w, dy, dev)
    f, yf = _kernel_grads(tgt2, mem, None, w, dy, dev, fused_args=args)
    torch.testing.assert_close(yf, ya, rtol=1e-5, atol=1e-5)
    for k in NAMES[:2] + WNAMES:
        torch.testing.assert_close(f[k], a[k], rtol=1e-5, atol=1e-5 * a[k].abs().max().item(), msg=k)


@pytest.mark.gpu
def test_fused_refuses_gradients_of_the_embedding_inputs(dev):
    from geoformer_b200.attention import rel_cross_attention_fused

    gen = torch.Generator().manual_seed(5)
    args = _fused_case(dev, 8, 50, 1, gen)
    w = {k: v.to(dev) for k, v in _rand_weights(gen).items()}
    tgt2, mem = torch.randn(8, 1, 64, device=dev, requires_grad=True), torch.randn(50, 1, 64, device=dev)
    for i in (2, 3, 4):  # query locations, context locations, gauss_B
        a = list(args)
        a[i] = a[i].clone().requires_grad_()
        with pytest.raises(RuntimeError, match="no gradient"):
            rel_cross_attention_fused(tgt2, mem, *a, w)


@pytest.mark.gpu
def test_decoder_trains_through_the_b200_path(dev):
    """FewShotForward.forward_decoder under grad, impl="b200" (fused kernel) vs impl="torch" (the reference's ops):
    the gradients of every decoder-layer parameter and of the two projections agree, so dtgt2 and dmemory flow
    through the stacked layers.  Measured on a B200: max 7.6e-2, Frobenius 5.8e-2 (layer 0, whose gradients pass
    through both layers' TF32 forwards and every ReLU mask of the chain); asserted at 0.15 / 0.1.  A missing dtgt2
    or dmemory path gives errors of order 1."""
    from geoformer_b200.harness import FewShotForward

    torch.manual_seed(0)
    Q, Cn, B = 64, 512, 2
    model = FewShotForward(nlayers=2, n_decode_point=Cn, n_query_points=Q).to(dev)
    gen = torch.Generator().manual_seed(21)
    geos, inds, qry, ctx, gb, pc = _fused_case(dev, Q, Cn, B, gen)
    agg = torch.randn(B, Cn, 96, generator=gen).to(dev)
    proj = torch.randn(2, Q, B, 64, generator=gen).to(dev)
    params = [(n, p) for n, p in model.named_parameters()
              if n.startswith(("layers.", "encoder_to_decoder_projection.", "query_projection."))]
    grads = {}
    for impl in ("b200", "torch"):
        model.zero_grad()
        out = model.forward_decoder(ctx, agg, qry, pc, geos, inds, impl)
        (out * proj).sum().backward()
        grads[impl] = {n: p.grad.clone() for n, p in params}
    for n, _ in params:
        if n.endswith("attn_mlp.2.bias"):  # db2: exactly zero against rounding level
            assert not grads["b200"][n].any() and grads["torch"][n].abs().max() < 1e-5
            continue
        _assert_grad_close(n, grads["b200"][n], grads["torch"][n], "decoder", tol=(0.15, 0.1))
