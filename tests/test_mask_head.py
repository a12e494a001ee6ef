"""The fused mask head (geoformer_b200.mask_head.mask_heads_forward, gf_mask_head.cu).

CPU: the oracle (oracle.mask_head) equals the harness's torch formulation in float64 and its relative coordinates
equal the reference fixture bias_golden.npz; the factored backward formulas (mask_head_backward below, test
infrastructure) equal autograd through the oracle in float64; the C entries validate their arguments before any
CUDA call; the kernel multiplies on the tensor cores (UTCHMMA in its SASS).

GPU: forward against the float64 oracle at ragged shapes, on maps of the library's guidance and on synthetic maps with
controlled unreachable patterns; row_max given or not gives bitwise-equal logits; no (Q, >=2, N) temporary; the
backward against autograd through the float64 oracle, deterministic, its forward bitwise the inference forward; the
data inputs refuse gradients; FewShotForward.mask_logits trained through both paths.

Tolerance.  The feature part of the first layer, sum_c w0[q,j,3+c] f[n,c], is a TF32 product (operands rounded to
10 mantissa bits, fp32 accumulation), the rest is fp32.  Each logit is therefore checked elementwise against
    |got - ref| <= 4e-3 * S_f + 1e-5 * S + 1e-6,
    S_f = sum_j |w1_j| sum_c |w0f_jc f_c|,   S = |b1| + sum_j |w1_j| (|b0_j| + sum_c |w0_jc x_c|)
(4e-3 ~ 2^-8 covers two operand roundings of 2^-11 each with room; measured on a B200 the worst |err| / bound over
the cases below is 0.13).  A wrong unreachable decision moves a logit by |w1 w0r| sqrt(rowmax); the cases with sqrt(rowmax) = 100
against coordinates of a few metres make that two orders of magnitude above the bound.  The gradients pass through
sums over up to N points of such terms; they are checked as max |g - g_ref| / max |g_ref| <= 1e-2 and relative
Frobenius error <= 3e-3, with the upstream gradient zeroed at the (q, n) where some hidden value lies within the
forward's bound of ReLU's kink: there the mask may be set differently from the float64 one, and with random dlogit
the sums over the points cancel enough for those few flips to reach 1.5e-2 of the result.  Measured on a B200 with
that exclusion: dfeats, dw0, db0, db1 <= 4.3e-7 (max) and dw1 <= 2.6e-4 (max), 4.3e-4 (Frobenius): dw1 sums
g relu(h), which carries the TF32 error of h itself, the others only its ReLU mask."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
M = 16
GNAMES = ("feats", "w0", "b0", "w1", "b1")


def mask_head_backward(geo, feats, w0, b0, w1, b1, coords, seeds, dlogit):
    """Gradients of oracle.mask_head.mask_heads_forward for dlogit (Q,N), in the factored form the kernel computes:
        db1 = sum_n g, dw1 = sum_n g relu(h), dh = g w1 [h > 0], db0 = sum_n dh, dw0 = sum_n dh x^T,
        dfeats = sum_{q,j} dh w0[., 3:]
    w0 (Q*16, 19), b0 (Q*16), w1 (Q, 16), b1 (Q) -> dict in those shapes"""
    from oracle.bias import mask_head_relative_coords

    Q, N = geo.shape
    rel = mask_head_relative_coords(geo, coords, seeds).to(feats.dtype)
    x = torch.cat([rel, feats.t()[None].expand(Q, M, N)], dim=1)  # (Q,19,N)
    W0 = w0.reshape(Q, M, M + 3)
    h = torch.einsum("qjc,qcn->qjn", W0, x) + b0.reshape(Q, M, 1)
    g = dlogit
    dh = g[:, None] * w1.reshape(Q, M, 1) * (h > 0)
    return {"feats": torch.einsum("qjn,qjc->nc", dh, W0[:, :, 3:]), "w0": torch.einsum("qjn,qcn->qjc", dh, x).reshape(Q * M, M + 3),
            "b0": dh.sum(2).reshape(Q * M), "w1": torch.einsum("qn,qjn->qj", g, F.relu(h)), "b1": g.sum(1)}


def _params(Q, N, gen, dtype=torch.float32, wscale=0.3):
    feats = torch.randn(N, M, generator=gen, dtype=dtype)
    w0 = torch.randn(Q * M, M + 3, generator=gen, dtype=dtype) * wscale
    b0 = torch.randn(Q * M, generator=gen, dtype=dtype) * 0.1
    w1 = torch.randn(Q, M, generator=gen, dtype=dtype) * wscale
    b1 = torch.randn(Q, generator=gen, dtype=dtype) * 0.1
    return feats, w0, b0, w1, b1


def _oracle(geo, feats, w0, b0, w1, b1, coords, seeds):
    from oracle.mask_head import mask_heads_forward

    Q = geo.shape[0]
    return mask_heads_forward(geo, feats, [w0.reshape(Q * M, M + 3, 1), w1.reshape(Q, M, 1)], [b0, b1], Q, coords, seeds)


def _maps(Q, N, gen, pattern="mixed", scale=3.0):
    geo = torch.rand(Q, N, generator=gen) * scale
    if pattern == "mixed":
        geo[torch.rand(Q, N, generator=gen) < 0.3] = -1.0
    elif pattern == "all_but_seed":
        geo[:] = -1.0
        geo[torch.arange(Q), torch.randint(0, N, (Q,), generator=gen)] = 0.0
    elif pattern == "all":
        geo[:] = -1.0
    return geo


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_oracle_equals_harness_torch_formulation_float64():
    from geoformer_b200.harness import FewShotForward
    from oracle.mask_head import mask_heads_forward

    torch.manual_seed(0)
    model = FewShotForward(n_query_points=9).double()
    gen = torch.Generator().manual_seed(1)
    B, Q, N = 2, 9, 301
    locs = torch.rand(B, N, 3, generator=gen, dtype=torch.float64) * 4
    query_locs = locs[:, :Q].clone()
    geo = [_maps(Q, N, gen).double() for _ in range(B)]
    feats = torch.randn(B, N, M, generator=gen, dtype=torch.float64)
    dec = torch.randn(Q, B, 64, generator=gen, dtype=torch.float64)
    with torch.no_grad():
        got = model.mask_logits(geo, dec, feats, locs, query_locs, None, "torch")
        ctl = model.controller(model.before_embedding_tower(dec.transpose(0, 1).flatten(0, 1).unsqueeze(2)))
        ctl = ctl.squeeze(2).reshape(B, Q, -1)
        for b in range(B):
            w0, w1, b0, b1 = torch.split_with_sizes(ctl[b], model.weight_nums + model.bias_nums, dim=1)
            want = mask_heads_forward(geo[b], feats[b], [w0.reshape(Q * M, -1, 1), w1.reshape(Q, -1, 1)],
                                      [b0.reshape(Q * M), b1.reshape(Q)], Q, locs[b], query_locs[b])
            err = (got[b] - want).abs().max().item() / want.abs().max().item()
            assert err <= 1e-12, err


def test_oracle_relative_coordinates_equal_reference_fixture():
    """weights that copy the three coordinate channels through the two layers: logit_j = rel_j + 1000"""
    from oracle.mask_head import mask_heads_forward

    g = np.load(os.path.join(HERE, "golden", "bias_golden.npz"))
    for i in range(int(g["n_mask"])):
        geo, coords, seeds = [torch.from_numpy(np.array(g["m%d_%s" % (i, k)])) for k in ("geo", "coords", "seed_xyz")]
        want = torch.from_numpy(np.array(g["m%d_out" % i])).double()  # (Q,3,N)
        Q, N = geo.shape
        feats = torch.randn(N, M, dtype=torch.float64)
        for a in range(3):
            w0 = torch.zeros(Q * M, M + 3, 1, dtype=torch.float64)
            w0[torch.arange(Q) * M, a, 0] = 1.0
            b0 = torch.zeros(Q * M, dtype=torch.float64)
            b0[torch.arange(Q) * M] = 1000.0
            w1 = torch.zeros(Q, M, 1, dtype=torch.float64)
            w1[:, 0, 0] = 1.0
            b1 = torch.full((Q,), -1000.0, dtype=torch.float64)
            got = mask_heads_forward(geo, feats, [w0, w1], [b0, b1], Q, coords, seeds)
            np.testing.assert_allclose(got.numpy(), want[:, a].numpy(), rtol=0, atol=1e-9)


@pytest.mark.parametrize("Q,N", [(1, 1), (3, 70), (17, 33)])
def test_factored_backward_equals_autograd_float64(Q, N):
    gen = torch.Generator().manual_seed(Q * 100 + N)
    feats, w0, b0, w1, b1 = _params(Q, N, gen, torch.float64)
    geo = _maps(Q, N, gen)
    coords = torch.rand(N, 3, generator=gen) * 4
    seeds = torch.rand(Q, 3, generator=gen) * 4
    dl = torch.randn(Q, N, generator=gen, dtype=torch.float64)
    leaves = [t.clone().requires_grad_() for t in (feats, w0, b0, w1, b1)]
    y = _oracle(geo, *leaves, coords, seeds)
    want = dict(zip(GNAMES, torch.autograd.grad(y, leaves, dl)))
    got = mask_head_backward(geo, feats, w0, b0, w1, b1, coords, seeds, dl)
    for k in GNAMES:
        assert got[k].shape == want[k].shape, k
        err = (got[k] - want[k]).abs().max().item()
        assert err <= 1e-10 * max(1.0, want[k].abs().max().item()), (k, err)


def test_entries_validate_before_any_cuda_call(cuda_lib):
    L = cuda_lib
    assert L.gf_mask_head_workspace_bytes(0, 10) == 0 and L.gf_mask_head_workspace_bytes(4, 10) >= 4 * 4 + 4
    assert L.gf_mask_head_backward_workspace_bytes(4, 0) == 0
    assert L.gf_mask_head_backward_workspace_bytes(4, 1000) >= 4 * 384 * 4
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below fails its checks first
    p9 = [fake] * 9
    rc = L.gf_mask_head_logits(*p9, -1, 10, 16, fake, fake, 1 << 20, None)
    assert rc == 1 and b"negative" in L.gf_last_error()
    rc = L.gf_mask_head_logits(*p9, 4, 10, 8, fake, fake, 1 << 20, None)
    assert rc == 1 and b"m=8" in L.gf_last_error()
    rc = L.gf_mask_head_logits(fake, None, *p9[2:], 4, 10, 16, fake, fake, 1 << 20, None)
    assert rc == 1 and b"null pointer" in L.gf_last_error()
    rc = L.gf_mask_head_logits(*p9, 4, 10, 16, None, fake, 1 << 20, None)
    assert rc == 1 and b"null pointer" in L.gf_last_error()
    g7 = [fake] * 7
    rc = L.gf_mask_head_logits_backward(*p9, 4, -2, 16, *g7, 1 << 20, None)
    assert rc == 1 and b"negative" in L.gf_last_error()
    rc = L.gf_mask_head_logits_backward(*p9, 4, 10, 17, *g7, 1 << 20, None)
    assert rc == 1 and b"m=17" in L.gf_last_error()
    rc = L.gf_mask_head_logits_backward(*p9, 4, 10, 16, fake, fake, None, fake, fake, fake, fake, 1 << 20, None)
    assert rc == 1 and b"null pointer" in L.gf_last_error()


def test_python_op_refuses_cpu_tensors_and_other_m(cuda_lib):
    from geoformer_b200.mask_head import mask_heads_forward

    Q, N = 2, 5
    w = [torch.zeros(Q * M, M + 3, 1), torch.zeros(Q, M, 1)]
    b = [torch.zeros(Q * M), torch.zeros(Q)]
    with pytest.raises(RuntimeError):
        mask_heads_forward(torch.zeros(Q, N), torch.zeros(N, M), w, b, Q, torch.zeros(N, 3), torch.zeros(Q, 3))


def test_kernel_runs_on_the_tensor_cores(cuda_lib):
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
    k = {f: n for f, n in per_fn.items() if "mask_head_kernel" in f}
    assert len(k) == 2 and all(n > 0 for n in k.values()), k


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev(cuda_lib):
    return torch.device("cuda:0")


def _ref64(geo, feats, w0, b0, w1, b1, coords, seeds):
    """float64 reference logits and the elementwise bound of the module docstring, computed on the inputs' device
    (the relative coordinates by the harness's torch statement of :271-288, which the CPU tests tie to the oracle)"""
    from geoformer_b200.harness import torch_mask_head_relative_coords

    d = torch.float64
    Q, N = geo.shape
    rel = torch_mask_head_relative_coords(geo.to(d), coords.to(d), seeds.to(d))  # (Q,3,N)
    W0 = w0.to(d).reshape(Q, M, M + 3)
    f = feats.to(d)
    hf = torch.einsum("qjc,nc->qjn", W0[:, :, 3:], f)
    h = hf + torch.einsum("qja,qan->qjn", W0[:, :, :3], rel) + b0.to(d).reshape(Q, M, 1)
    a1 = w1.to(d).reshape(Q, M, 1).abs()
    out = torch.einsum("qj,qjn->qn", w1.to(d).reshape(Q, M), F.relu(h)) + b1.to(d)[:, None]
    sf = (a1 * torch.einsum("qjc,nc->qjn", W0[:, :, 3:].abs(), f.abs())).sum(1)
    s = sf + (a1 * (b0.to(d).reshape(Q, M, 1).abs() + torch.einsum("qja,qan->qjn", W0[:, :, :3].abs(), rel.abs()))).sum(1)
    s = s + b1.to(d).abs()[:, None]
    return out, 4e-3 * sf + 1e-5 * s + 1e-6


def _call(geo, feats, w0, b0, w1, b1, coords, seeds, row_max=None):
    from geoformer_b200.mask_head import mask_heads_forward

    Q = geo.shape[0]
    return mask_heads_forward(geo, feats, [w0.reshape(Q * M, M + 3, 1), w1.reshape(Q, M, 1)], [b0, b1], Q, coords,
                              seeds, row_max=row_max)


def _check_forward(geo, feats, w0, b0, w1, b1, coords, seeds, what, nan_expected=False):
    got = _call(geo, feats, w0, b0, w1, b1, coords, seeds)
    torch.cuda.synchronize()
    want, bound = _ref64(geo, feats, w0, b0, w1, b1, coords, seeds)
    nan_g, nan_w = torch.isnan(got), torch.isnan(want)
    assert torch.equal(nan_g, nan_w), (what, nan_g.sum().item(), nan_w.sum().item())
    if nan_expected:
        assert bool(nan_w.all()), what
        return
    ratio = ((got.double() - want).abs() / bound).max().item() if got.numel() else 0.0
    print("%s: max |err| / bound = %.3f" % (what, ratio))
    assert ratio <= 1.0, (what, ratio)


def _unaligned(t):
    """the same values at a base 4 bytes past a 16-byte boundary"""
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    return v


@pytest.mark.gpu
@pytest.mark.parametrize("Q,N", [(1, 1), (15, 127), (16, 4099), (17, 4099), (17, 1), (256, 100_003), (33, 100_000)])
def test_forward_matches_float64_oracle(dev, Q, N):
    gen = torch.Generator().manual_seed(Q * 7 + N)
    feats, w0, b0, w1, b1 = [t.to(dev) for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen).to(dev)
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = ((torch.rand(Q, 3, generator=gen) - 0.5) * 8).to(dev)
    _check_forward(geo, feats, w0, b0, w1, b1, coords, seeds, "Q=%d N=%d" % (Q, N))


@pytest.mark.gpu
def test_forward_unaligned_bases(dev):
    Q, N = 17, 4099
    gen = torch.Generator().manual_seed(11)
    args = [t.to(dev) for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen).to(dev)
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = ((torch.rand(Q, 3, generator=gen) - 0.5) * 8).to(dev)
    ua = [_unaligned(t) for t in [geo] + args + [coords, seeds]]
    _check_forward(*ua, what="unaligned")
    assert torch.equal(_call(*ua), _call(geo, *args, coords, seeds))


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", ["none", "all_but_seed", "mixed_large_rowmax", "all"])
def test_forward_unreachable_patterns(dev, pattern):
    Q, N = 37, 5003
    gen = torch.Generator().manual_seed(5)
    args = [t.to(dev) for t in _params(Q, N, gen)]
    if pattern == "mixed_large_rowmax":  # sqrt(rowmax) = 100 against coordinates within 4 m
        geo = _maps(Q, N, gen, "mixed", scale=1e4)
    else:
        geo = _maps(Q, N, gen, pattern)
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = coords[torch.randint(0, N, (Q,), generator=gen).to(dev)].contiguous()
    _check_forward(geo.to(dev), *args, coords, seeds, pattern, nan_expected=pattern == "all")


@pytest.mark.gpu
def test_forward_on_guidance_maps(dev):
    """maps of the library's propagation (the model's setting k = 64, r = 0.05) on a synthetic ScanNet scene"""
    from geoformer_b200 import scenes
    from geoformer_b200.geodesic_utils import cal_geodesic_vectorize

    N, Q = 20_000, 64
    locs = scenes.scene(N, 7).to(dev)
    gen = torch.Generator().manual_seed(2)
    seeds_idx = torch.randperm(N, generator=gen)[:Q].int()[None].to(dev)
    geo = cal_geodesic_vectorize(None, seeds_idx, locs, torch.tensor([0, N], dtype=torch.int32), max_step=256,
                                 neighbor=64, radius=0.05, n_queries=Q)[0]
    assert (geo < 0).any() and (geo >= 0).any()
    args = [t.to(dev) for t in _params(Q, N, gen)]
    _check_forward(geo.contiguous(), *args, locs, locs[seeds_idx[0].long()].contiguous(), "guidance maps")


@pytest.mark.gpu
def test_row_max_given_is_bitwise_equal(dev):
    Q, N = 40, 9001
    gen = torch.Generator().manual_seed(9)
    args = [t.to(dev) for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen).to(dev)
    geo[3] = -1.0  # a row with nothing reachable takes the global maximum
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = ((torch.rand(Q, 3, generator=gen) - 0.5) * 8).to(dev)
    a = _call(geo, *args, coords, seeds)
    b = _call(geo, *args, coords, seeds, row_max=geo.max(dim=1)[0].contiguous())
    assert torch.equal(a, b)


@pytest.mark.gpu
def test_no_large_temporaries(dev):
    Q, N = 256, 100_000
    gen = torch.Generator().manual_seed(4)
    args = [t.to(dev) for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen).to(dev)
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = ((torch.rand(Q, 3, generator=gen) - 0.5) * 8).to(dev)
    _call(geo, *args, coords, seeds)  # workspace allocated once
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(dev)
    base = torch.cuda.memory_allocated(dev)
    out = _call(geo, *args, coords, seeds)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    print("peak increase %.1f MB (logits %.1f MB)" % (peak / 2**20, out.numel() * 4 / 2**20))
    assert peak < 2 * Q * N * 4


def _lib_grads(geo, feats, w0, b0, w1, b1, coords, seeds, dl):
    leaves = [t.clone().requires_grad_() for t in (feats, w0, b0, w1, b1)]
    y = _call(geo, *leaves, coords, seeds)
    return dict(zip(GNAMES, torch.autograd.grad(y, leaves, dl))), y


@pytest.mark.gpu
@pytest.mark.parametrize("Q,N", [(1, 1), (17, 4099), (128, 30_000)])
def test_backward_matches_float64_oracle(dev, Q, N):
    gen = torch.Generator().manual_seed(Q + N)
    args = [t.to(dev) for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen)
    geo[:, 0] = 0.5  # a reachable point in every row: no NaN scene here (sqrt(-1), see the forward tests)
    geo = geo.to(dev)
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = ((torch.rand(Q, 3, generator=gen) - 0.5) * 8).to(dev)
    dl = torch.randn(Q, N, generator=gen).to(dev)
    d = torch.float64
    from geoformer_b200.harness import torch_mask_head_relative_coords

    rel = torch_mask_head_relative_coords(geo.to(d), coords.to(d), seeds.to(d))
    W0 = args[1].to(d).reshape(Q, M, M + 3)
    f = args[0].to(d)
    h = torch.einsum("qjc,nc->qjn", W0[:, :, 3:], f) + torch.einsum("qja,qan->qjn", W0[:, :, :3], rel) \
        + args[2].to(d).reshape(Q, M, 1)
    bound = 4e-3 * torch.einsum("qjc,nc->qjn", W0[:, :, 3:].abs(), f.abs()) + 1e-5 * (
        args[2].to(d).abs().reshape(Q, M, 1) + torch.einsum("qja,qan->qjn", W0[:, :, :3].abs(), rel.abs())) + 1e-6
    near_kink = (h.abs() <= bound).any(1)  # (q, n) whose ReLU masks the TF32 forward may set differently
    print("Q=%d N=%d: %d of %d (q, n) near a ReLU kink, their dlogit zeroed" % (Q, N, int(near_kink.sum()), Q * N))
    dl = torch.where(near_kink, torch.zeros_like(dl), dl)
    got, y = _lib_grads(geo, *args, coords, seeds, dl)
    leaves = [t.to(d).requires_grad_() for t in args]
    x = torch.cat([rel, leaves[0].t()[None].expand(Q, M, N)], 1).reshape(1, -1, N)
    x = F.relu(F.conv1d(x, leaves[1].reshape(Q * M, M + 3, 1), leaves[2], groups=Q))
    ref = F.conv1d(x, leaves[3].reshape(Q, M, 1), leaves[4], groups=Q).reshape(Q, N)
    want = dict(zip(GNAMES, torch.autograd.grad(ref, leaves, dl.to(d))))
    errs = {}
    for k in GNAMES:
        g, w = got[k].double(), want[k]
        assert g.shape == w.shape, k
        scale = max(w.abs().max().item(), 1e-30)
        errs[k] = ((g - w).abs().max().item() / scale, ((g - w).norm() / max(w.norm().item(), 1e-30)).item())
        print("Q=%d N=%d %-5s max %.2e fro %.2e scale %.3g" % (Q, N, k, errs[k][0], errs[k][1], scale))
    for k, (emax, efro) in errs.items():
        assert emax <= 1e-2 and efro <= 3e-3, (k, emax, efro)


@pytest.mark.gpu
def test_backward_deterministic_and_forward_unchanged(dev):
    Q, N = 64, 20_011
    gen = torch.Generator().manual_seed(21)
    args = [t.to(dev) for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen).to(dev)
    coords = ((torch.rand(N, 3, generator=gen) - 0.5) * 8).to(dev)
    seeds = ((torch.rand(Q, 3, generator=gen) - 0.5) * 8).to(dev)
    dl = torch.randn(Q, N, generator=gen).to(dev)
    g1, y1 = _lib_grads(geo, *args, coords, seeds, dl)
    g2, y2 = _lib_grads(geo, *args, coords, seeds, dl)
    for k in GNAMES:
        assert torch.equal(g1[k], g2[k]), k
    with torch.no_grad():
        y0 = _call(geo, *args, coords, seeds)
    assert torch.equal(y1, y0) and torch.equal(y2, y0)


@pytest.mark.gpu
def test_data_inputs_refuse_gradients(dev):
    Q, N = 4, 100
    gen = torch.Generator().manual_seed(1)
    args = [t.to(dev).requires_grad_() for t in _params(Q, N, gen)]
    geo = _maps(Q, N, gen).to(dev)
    coords = torch.rand(N, 3).to(dev)
    seeds = torch.rand(Q, 3).to(dev)
    for i in range(3):
        data = [geo.clone(), coords.clone(), seeds.clone()]
        data[i].requires_grad_()
        with pytest.raises(RuntimeError):
            _call(data[0], *args, data[1], data[2])


@pytest.mark.gpu
def test_mask_logits_trains_through_both_paths(dev):
    """loss on FewShotForward.mask_logits: gradients of the mask tower, the before-embedding tower, the controller
    and the decoder output agree between impl="b200" and impl="torch" (both TF32 on the first layer's products).
    Relative Frobenius error <= 5e-2: with random loss weights the sums over the points cancel, so the (q, n) whose
    hidden values lie within TF32 rounding of ReLU's kink, and flip their mask in one of the two paths, weigh in
    with the square root of their share (about 1.5e-2 measured on a B200)."""
    from geoformer_b200.harness import FewShotForward

    torch.manual_seed(0)
    B, N, Q = 2, 5000, 32
    model = FewShotForward(n_query_points=Q).to(dev)
    gen = torch.Generator().manual_seed(3)
    locs = ((torch.rand(B, N, 3, generator=gen) - 0.5) * 6).to(dev)
    query_locs = locs[:, :Q].contiguous()
    geo = [_maps(Q, N, gen).to(dev) for _ in range(B)]
    out_feats = torch.randn(B, N, M, generator=gen).to(dev)
    dec = torch.randn(Q, B, 64, generator=gen).to(dev)
    wl = [torch.randn(Q, N, generator=gen).to(dev) for _ in range(B)]
    params = list(model.mask_tower.parameters()) + list(model.before_embedding_tower.parameters()) + \
        list(model.controller.parameters())
    grads = {}
    for impl in ("b200", "torch"):
        d = dec.clone().requires_grad_()
        mf = model.mask_tower(out_feats.transpose(1, 2)).transpose(1, 2)
        logits = model.mask_logits(geo, d, mf, locs, query_locs, None, impl)
        loss = sum((lg * w).sum() for lg, w in zip(logits, wl))
        grads[impl] = torch.autograd.grad(loss, params + [d])
    for i, (a, b) in enumerate(zip(grads["b200"], grads["torch"])):
        efro = ((a - b).norm() / b.norm()).item()
        print("param %d fro %.2e" % (i, efro))
        assert efro <= 5e-2, (i, efro)
