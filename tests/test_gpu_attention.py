"""GPU tests of the decoder's vector cross-attention kernel (tcgen05, TF32 products, fp32 accumulation) against
  * the fixture produced by the reference's OWN TransformerDecoderLayer.forward_pre_rel (tests/golden/attention_golden.npz),
  * the fp32 CPU restatement oracle/attention.py at the model's shapes (Q=256, C=2048) and ragged ones,
  * and, for the fused variant, the unfused kernel fed with the embedding our own Fourier epilogue writes.
Tolerance: the reference is fp32; TF32 rounds the operands of the three 64-wide products to 10 mantissa bits
(relative 5e-4 each).  Measured: max |diff| <= 2e-3 of the output scale; asserted at 4e-3 absolute + 4e-3 relative.
That tolerance ties the kernel to the reference model.  The kernel's own arithmetic (out, o and lse, every score
regime and context-tile boundary) is pinned much tighter against the TF32-exact float64 emulation oracle/tf32.py in
tests/test_tf32_reference.py, which also shows wrong kernels this tolerance would accept."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
TOL = dict(rtol=4e-3, atol=4e-3)


@pytest.fixture(scope="module")
def dev(cuda_lib):
    return torch.device("cuda:0")


def _rand_weights(gen, scale=0.125):
    return {"w1": torch.randn(64, 64, generator=gen) * scale, "b1": torch.randn(64, generator=gen) * 0.1,
            "w2": torch.randn(64, 64, generator=gen) * scale, "b2": torch.randn(64, generator=gen) * 0.1,
            "wv": torch.randn(64, 64, generator=gen) * scale, "bv": torch.randn(64, generator=gen) * 0.1,
            "wo": torch.randn(64, 64, generator=gen) * scale, "bo": torch.randn(64, generator=gen) * 0.1}


def test_cross_attention_matches_reference_layer_fixture(dev):
    from geoformer_b200.attention import rel_cross_attention

    g = np.load(os.path.join(HERE, "golden", "attention_golden.npz"))
    T = lambda a: torch.from_numpy(np.array(a)).to(dev)  # noqa: E731
    for i in range(int(g["n"])):
        w = {k: T(g["c%d_%s" % (i, k)]) for k in ("w1", "b1", "w2", "b2", "wv", "bv", "wo", "bo")}
        out = rel_cross_attention(T(g["c%d_tgt2" % i]), T(g["c%d_memory" % i]), T(g["c%d_rel" % i]), w)
        want = g["c%d_out" % i]
        assert out.shape == want.shape
        err = np.abs(out.cpu().numpy() - want).max()
        np.testing.assert_allclose(out.cpu().numpy(), want, err_msg="case %d max err %g" % (i, err), **TOL)


@pytest.mark.parametrize("Q,C,B", [(256, 2048, 1), (37, 301, 2), (3, 1, 1), (5, 129, 3)])
def test_cross_attention_matches_fp32_oracle(dev, Q, C, B):
    from oracle import attention as oatt

    from geoformer_b200.attention import rel_cross_attention

    gen = torch.Generator().manual_seed(Q * 7 + C)
    w = _rand_weights(gen)
    tgt2 = torch.randn(Q, B, 64, generator=gen)
    mem = torch.randn(C, B, 64, generator=gen)
    rel = torch.rand(Q, C, B, 64, generator=gen) * 2 - 1
    want = oatt.rel_cross_attention(tgt2, mem, rel, w)
    out = rel_cross_attention(tgt2.to(dev), mem.to(dev), rel.to(dev), w).cpu()
    err = (out - want).abs().max().item()
    torch.testing.assert_close(out, want, msg="max err %g" % err, **TOL)
    assert (out >= 0).all()  # out_mlp ends in a ReLU


def test_fused_variant_equals_unfused_on_our_embedding(dev):
    """the fused kernel builds the Fourier embedding itself (a10 + :704-712); the unfused one is fed the tensor our
    epilogue kernel writes for the same inputs.  Same arithmetic for the embedding (bit-identical sin / cos), same
    products: equal to 1e-5."""
    from geoformer_b200.attention import rel_cross_attention, rel_cross_attention_fused
    from geoformer_b200.bias import decoder_relative_embedding
    from geoformer_b200.scenes import scene

    gen = torch.Generator().manual_seed(9)
    for Q, Cn, B in ((64, 300, 2), (256, 2048, 1)):
        Ns = [20000 + 1000 * b for b in range(B)]
        xs = [scene(n, 50 + b) for b, n in enumerate(Ns)]
        geos = []
        for n in Ns:
            gq = torch.rand(Q, n, generator=gen) * 4.0
            gq[torch.rand(Q, n, generator=gen) < 0.5] = -1.0
            gq[1] = -1.0
            geos.append(gq.to(dev))
        inds = torch.stack([torch.randperm(n, generator=gen)[:Cn] for n in Ns]).int()
        ctx = torch.stack([x[i.long()] for x, i in zip(xs, inds)]).contiguous()
        qry = ctx[:, :Q].contiguous()
        gb = torch.randn(3, 32, generator=gen)
        pc = [torch.stack([x.min(0)[0] for x in xs]), torch.stack([x.max(0)[0] for x in xs])]
        w = _rand_weights(gen)
        tgt2 = torch.randn(Q, B, 64, generator=gen).to(dev)
        mem = torch.randn(Cn, B, 64, generator=gen).to(dev)
        emb = decoder_relative_embedding(geos, inds.to(dev), qry.to(dev), ctx.to(dev), gb.to(dev),
                                         [pc[0].to(dev), pc[1].to(dev)])  # (Q, C, B, 64) view
        a = rel_cross_attention(tgt2, mem, emb.contiguous(), w)
        f = rel_cross_attention_fused(tgt2, mem, geos, inds.to(dev), qry.to(dev), ctx.to(dev), gb.to(dev),
                                      [pc[0].to(dev), pc[1].to(dev)], w)
        torch.testing.assert_close(f, a, rtol=1e-5, atol=1e-5)
