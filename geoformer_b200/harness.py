"""BASELINE.json config 5 (SURVEY 8(f) rank 4): the few-shot inference forward of GeoFormer AFTER its backbone, random
init, with the B200 path swapped in -- model/geoformer/geoformer_fs.py:424-596 with the sparse-conv U-Net replaced by
a stub that produces `output_feats` / `semantic_preds` of the right shapes (:460-475; spconv, PG_OP and faiss do not
exist in this image).  What runs is the real chain

    forward_aggregator (:619-660)  ->  queries (:494)  ->  cal_geodesic_vectorize (:497-506, the model's setting:
    neighbor 64, radius 0.05, max_step 256)  ->  forward_decoder (:662-723: position embeddings, relative geodesic
    embedding, four pre-norm decoder layers with the vector cross-attention of transformer_detr.py:422-463)  ->
    get_mask_prediction / mask_heads_forward (:302-360, :263-300: dynamic convolutions on [relative coords | mask features])

Every piece of the hot path has two implementations selected by `impl`:
    "b200"   the library: fused aggregator, batched geodesic guidance, fused cross-attention (embedding never
             materialised), fused mask head (relative coordinates + both dynamic convolutions in one kernel)
    "torch"  the reference's formulation with plain torch ops on the same device (group -> conv/bn/relu -> pool; the
             level loop of cal_geodesic_vectorize is NOT rerun in torch: the maps are shared, they are bit-exact
             anyway; relative_pos materialised; three (Q,C,B,64) temporaries; boolean-mask indexing in the mask head)
The surrounding torch layers (self-attention, layer norms, feed-forward, projections, controller) are ordinary
torch.nn modules shared by both, built with the reference's shapes (config/geoformer_fs_scannet.yaml: m = 16,
dec_dim 64, 4 heads, 4 layers, ffn 64, 2048 contexts, 128 queries at training / 256 at test).
"""
import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import aggregate as agg
from . import attention as att
from . import mask_head as mh
from .geodesic_utils import cal_geodesic_vectorize
from .pointnet2 import _ext


def fourier_embedding(xyz, gauss_B, pc_dims):
    """PositionEmbeddingCoordsSine.get_fourier_embeddings, normalize=True (pos_embedding.py:88-114 + utils_pc.py:35-61):
    xyz (B,n,3) -> (B, d_pos, n)"""
    mn, mx = pc_dims
    x = (xyz - mn[:, None, :]) / (mx[:, None, :] - mn[:, None, :])
    x = x * (2 * np.pi)
    proj = torch.matmul(x.reshape(-1, 3), gauss_B).reshape(xyz.shape[0], xyz.shape[1], -1)
    return torch.cat([proj.sin(), proj.cos()], dim=2).permute(0, 2, 1)


class DecoderLayer(nn.Module):
    """TransformerDecoderLayer(use_rel=True, normalize_before=True), transformer_detr.py:361-463, inference form"""

    def __init__(self, d=64, nhead=4, ffn=64):
        super().__init__()
        self.self_attn = nn.MultiheadAttention(d, nhead)
        self.norm1, self.norm2, self.norm3 = nn.LayerNorm(d), nn.LayerNorm(d), nn.LayerNorm(d)
        self.linear1, self.linear2 = nn.Linear(d, ffn), nn.Linear(ffn, d)
        self.attn_mlp = nn.Sequential(nn.Linear(d, d), nn.ReLU(), nn.Linear(d, d))
        self.v_mlp = nn.Sequential(nn.Linear(d, d))
        self.out_mlp = nn.Sequential(nn.Linear(d, d), nn.ReLU())

    def forward(self, tgt, memory, query_pos, cross):
        tgt2 = self.norm1(tgt)  # :431-435
        qk = tgt2 + query_pos
        tgt = tgt + self.self_attn(qk, qk, value=tgt2)[0]
        tgt2 = self.norm2(tgt)
        tgt = cross(self, tgt2, memory) + tgt2  # :443-456 (the reference adds tgt2, not tgt, back: kept)
        tgt2 = self.norm3(tgt)
        return tgt + self.linear2(F.relu(self.linear1(tgt2)))  # :457-459


class FewShotForward(nn.Module):
    def __init__(self, m=16, dec_dim=64, nhead=4, nlayers=4, ffn=64, n_decode_point=2048, n_query_points=256,
                 radius=0.2, nsample=64):
        super().__init__()
        self.m, self.dec_dim, self.C, self.Q = m, dec_dim, n_decode_point, n_query_points
        self.radius, self.nsample = radius, nsample

        def conv_bn(cin, cout):  # pytorch_utils.Conv2d(bn=True): conv without bias + BatchNorm2d + ReLU
            return nn.Sequential(nn.Conv2d(cin, cout, 1, bias=False), nn.Sequential(nn.BatchNorm2d(cout)), nn.ReLU())

        self.mlp_module = nn.Sequential(conv_bn(m + 3, 2 * m), conv_bn(2 * m, 2 * m), conv_bn(2 * m, 2 * m))  # :105-113
        self.register_buffer("gauss_B", torch.randn(3, dec_dim // 2))  # pos_embedding.py:38-41
        d_agg = 2 * m * 3
        self.encoder_to_decoder_projection = nn.Sequential(  # GenericMLP :139-149
            nn.Conv1d(d_agg, d_agg, 1, bias=False), nn.BatchNorm1d(d_agg), nn.ReLU(),
            nn.Conv1d(d_agg, dec_dim, 1, bias=False), nn.BatchNorm1d(dec_dim), nn.ReLU())
        self.query_projection = nn.Sequential(nn.Conv1d(dec_dim, dec_dim, 1), nn.ReLU(), nn.Conv1d(dec_dim, dec_dim, 1), nn.ReLU())
        self.layers = nn.ModuleList([DecoderLayer(dec_dim, nhead, ffn) for _ in range(nlayers)])
        self.mask_tower = nn.Sequential(nn.Conv1d(m, m, 1), nn.ReLU(), nn.Conv1d(m, m, 1))  # stands for :62-67
        self.before_embedding_tower = nn.Sequential(nn.Conv1d(dec_dim, m, 1), nn.BatchNorm1d(m), nn.ReLU())
        self.weight_nums, self.bias_nums = [(m + 3) * m, m], [m, 1]  # :77-96
        self.controller = nn.Conv1d(m, sum(self.weight_nums) + sum(self.bias_nums), 1)
        nn.init.normal_(self.controller.weight, std=0.01)
        nn.init.constant_(self.controller.bias, 0)
        for mod in self.modules():  # non-trivial running statistics so that the folded batch norm is exercised
            if isinstance(mod, (nn.BatchNorm1d, nn.BatchNorm2d)):
                mod.running_mean.normal_(0, 0.2)
                mod.running_var.uniform_(0.6, 1.4)
        self.eval()

    # ---- :619-660 ---------------------------------------------------------------------------------------
    def _aggregator_module(self):
        """the set aggregator's attributes aggregate() / aggregate_batch() read"""
        class _G:
            radius, nsample, normalize_xyz, use_xyz = self.radius, self.nsample, True, True

        class _M:
            npoint, pooling, grouper, mlp_module = self.C, "max", _G, self.mlp_module

        return _M

    def _group_torch(self, xyz, f):
        """group_points of the reference (pointnet2_modules.py:200-232): xyz (B,N,3), f (B,m,N) -> centres (B,C,3),
        grouped input (B, 3+m, C, nsample), seeds (B,C) i32"""
        inds = _ext.furthest_point_sampling(xyz, self.C)
        new_xyz = _ext.gather_points(xyz.transpose(1, 2).contiguous(), inds).transpose(1, 2).contiguous()
        idx = _ext.ball_query(new_xyz, xyz, self.radius, self.nsample)
        g_xyz = _ext.group_points(xyz.transpose(1, 2).contiguous(), idx)  # pointnet2_utils.py:330-341
        g_xyz = (g_xyz - new_xyz.transpose(1, 2).unsqueeze(-1)) / self.radius
        return new_xyz, torch.cat([g_xyz, _ext.group_points(f, idx)], dim=1), inds

    def _mlp_pool_torch(self, x):
        x = self.mlp_module(x)
        return F.max_pool2d(x, kernel_size=[1, x.size(3)]).squeeze(-1).transpose(1, 2)

    def forward_aggregator(self, locs, feats, impl):
        """locs (B,N,3), feats (B,N,m) -> context_locs (B,C,3), context_feats (B,C,2m), pre_enc_inds (B,C) i32"""
        xyz = locs.contiguous()
        f = feats.transpose(1, 2).contiguous()
        if impl == "b200":
            new_xyz, out, inds = agg.aggregate(self._aggregator_module(), xyz, f)
            return new_xyz, out.transpose(1, 2), inds
        new_xyz, x, inds = self._group_torch(xyz, f)
        return new_xyz, self._mlp_pool_torch(x), inds

    def forward_aggregator_batch(self, locs, feats, offsets, impl):
        """the ragged form of :619-660: locs (sum N,3), feats (sum N,m), offsets (B+1) ints -> as forward_aggregator.
        "torch" groups every scene on its own, concatenates the groups and runs ONE mlp over them (:643-657)."""
        if impl == "b200":
            new_xyz, out, inds = agg.aggregate_batch(self._aggregator_module(), locs, feats, offsets)
            return new_xyz, out.transpose(1, 2), inds
        groups = [self._group_torch(locs[a:b][None].contiguous(), feats[a:b].t()[None].contiguous())
                  for a, b in zip(offsets, offsets[1:])]
        new_xyz, x, inds = (torch.cat(t, dim=0) for t in zip(*groups))
        return new_xyz, self._mlp_pool_torch(x), inds

    # ---- :662-723 ---------------------------------------------------------------------------------------
    def forward_decoder(self, context_locs, aggregation, query_locs, pc_dims, geo_dists, pre_enc_inds, impl):
        B = context_locs.shape[0]
        context_pos = fourier_embedding(context_locs, self.gauss_B, pc_dims)
        ctx = self.encoder_to_decoder_projection(aggregation.permute(0, 2, 1))  # (B, d, C)
        query_pos = self.query_projection(fourier_embedding(query_locs, self.gauss_B, pc_dims))
        tgt = ctx[:, :, : self.Q].permute(2, 0, 1).contiguous()
        memory = ctx.permute(2, 0, 1).contiguous()
        query_pos = query_pos.permute(2, 0, 1).contiguous()
        del context_pos  # the reference passes it as `pos`; forward_pre_rel never uses it
        if impl == "b200":
            def cross(layer, tgt2, mem):
                return att.rel_cross_attention_fused(tgt2.contiguous(), mem, geo_dists, pre_enc_inds, query_locs,
                                                     context_locs, self.gauss_B, pc_dims, att.layer_weights(layer))
        else:
            rel = gbias_torch_decoder_relative_pos(geo_dists, pre_enc_inds, query_locs, context_locs)  # :680-702
            emb = fourier_embedding(rel.reshape(B, self.Q * self.C, 3), self.gauss_B, pc_dims)
            relative_pos = emb.reshape(B, -1, self.Q, self.C).permute(2, 3, 0, 1)  # :704-712

            def cross(layer, tgt2, mem):  # transformer_detr.py:443-453
                n_q, n_c = relative_pos.shape[0], relative_pos.shape[1]
                t_e = tgt2[:, None, :, :].repeat(1, n_c, 1, 1)
                m_e = mem[None, :, :, :].repeat(n_q, 1, 1, 1)
                sim = layer.attn_mlp(t_e - m_e + relative_pos)
                attn = F.softmax(sim / math.sqrt(sim.shape[-1]), dim=1)
                return layer.out_mlp(torch.einsum("qcbf,qcbf->qbf", attn, layer.v_mlp(m_e + relative_pos)))
        outs = []
        for layer in self.layers:
            tgt = layer(tgt, memory, query_pos, cross)
            outs.append(tgt)
        return torch.stack(outs)  # (layers, Q, B, d)

    # ---- :302-360, :263-300 -----------------------------------------------------------------------------------
    def mask_logits(self, geo_dists, dec_out, mask_features, locs, query_locs, row_max, impl):
        """dec_out (Q,B,d) -> list of (Q, N_b) logits"""
        Qn, B, _ = dec_out.shape
        pk = dec_out.transpose(0, 1).flatten(0, 1)
        controllers = self.controller(self.before_embedding_tower(pk.unsqueeze(2))).squeeze(2).reshape(B, Qn, -1)
        m = self.m
        out = []
        for b in range(B):
            w0, w1, b0, b1 = torch.split_with_sizes(controllers[b], self.weight_nums + self.bias_nums, dim=1)
            weights = [w0.reshape(Qn * m, -1, 1), w1.reshape(Qn, -1, 1)]
            biases = [b0.reshape(Qn * m), b1.reshape(Qn)]
            feats_b = mask_features[b]  # (N, m)
            if impl == "b200":  # :263-300 in one kernel: no (Q, >1, N) temporary
                out.append(mh.mask_heads_forward(geo_dists[b], feats_b, weights, biases, Qn, locs[b].contiguous(),
                                                 query_locs[b].contiguous(),
                                                 row_max=row_max[b] if row_max is not None else None))
                continue
            rel = torch_mask_head_relative_coords(geo_dists[b], locs[b], query_locs[b])
            x = feats_b.t()[None].repeat(Qn, 1, 1)  # :269
            x = torch.cat([rel, x], dim=1).reshape(1, -1, feats_b.shape[0])  # :291-293
            for i, (w, bb) in enumerate(zip(weights, biases)):
                x = F.conv1d(x, w, bias=bb, stride=1, padding=0, groups=Qn)  # :294-297
                if i < len(weights) - 1:
                    x = F.relu(x)
            out.append(x.squeeze(0))
        return out

    @torch.no_grad()
    def forward(self, locs, output_feats, support_embedding, impl="b200", max_step=256, neighbor=64, geo_radius=0.05,
                batch_offsets=None):
        """locs (B,N,3) foreground points of B equally sized scenes, output_feats (B,N,m) the stub backbone's point
        features, support_embedding (B, 2m).  Returns (list of (Q,N) mask logits, geo_dists, pre_enc_inds).
        batch_offsets (B+1), tensor or list: a ragged batch as the model holds it, locs (sum N,3) and output_feats
        (sum N,m) flat; the logits are then (Q, N_b) per scene."""
        return self._chain(locs, output_feats, support_embedding, impl, max_step, neighbor, geo_radius, batch_offsets)

    def forward_train(self, locs, output_feats, support_embedding, impl="b200", max_step=128, neighbor=64,
                      geo_radius=0.05, batch_offsets=None):
        """forward with autograd: one training step of the post-backbone path (the training setting of SURVEY 3.1 is a
        model built with n_query_points=128 and max_step=128).  Call model.train() first for batch-statistics batch
        norm.  Gradients reach every parameter through the aggregator, decoder and mask head of either impl; the
        geodesic maps are data.  batch_offsets: as in forward."""
        return self._chain(locs, output_feats, support_embedding, impl, max_step, neighbor, geo_radius, batch_offsets)

    def _chain(self, locs, output_feats, support_embedding, impl, max_step, neighbor, geo_radius, batch_offsets=None):
        if batch_offsets is not None:
            return self._chain_ragged(locs, output_feats, support_embedding, impl, max_step, neighbor, geo_radius,
                                      agg.batch_offsets_list(batch_offsets, locs.shape[0]))
        B, N, _ = locs.shape
        pc_dims = [locs.min(dim=1)[0], locs.max(dim=1)[0]]
        mask_features = self.mask_tower(output_feats.transpose(1, 2)).transpose(1, 2)  # :477-483
        context_locs, context_feats, pre_enc_inds = self.forward_aggregator(locs, output_feats, impl)
        query_locs = context_locs[:, : self.Q, :].contiguous()  # :494
        offsets = torch.arange(B + 1, dtype=torch.int32) * N
        geo_dists = cal_geodesic_vectorize(None, pre_enc_inds, locs.reshape(-1, 3).contiguous(), offsets,
                                           max_step=max_step, neighbor=neighbor, radius=geo_radius, n_queries=self.Q)
        se = support_embedding.unsqueeze(1)
        aggregation = torch.cat([context_feats * se, context_feats - se, context_feats], dim=2)  # :543-548
        dec = self.forward_decoder(context_locs, aggregation, query_locs, pc_dims, geo_dists, pre_enc_inds, impl)
        logits = self.mask_logits(geo_dists, dec[-1], mask_features, locs, query_locs, None, impl)
        return logits, geo_dists, pre_enc_inds

    def _chain_ragged(self, locs, output_feats, support_embedding, impl, max_step, neighbor, geo_radius, offsets):
        """_chain on the flat (sum N, .) arrays of a ragged batch: per-scene extents, mask features and mask heads"""
        scenes = [slice(a, b) for a, b in zip(offsets, offsets[1:])]
        pc_dims = [torch.stack([locs[s].min(dim=0)[0] for s in scenes]), torch.stack([locs[s].max(dim=0)[0] for s in scenes])]
        mask_features = self.mask_tower(output_feats.t()[None])[0].t()  # a 1x1 conv: per point
        context_locs, context_feats, pre_enc_inds = self.forward_aggregator_batch(locs, output_feats, offsets, impl)
        query_locs = context_locs[:, : self.Q, :].contiguous()
        geo_dists = cal_geodesic_vectorize(None, pre_enc_inds, locs.contiguous(), offsets, max_step=max_step,
                                           neighbor=neighbor, radius=geo_radius, n_queries=self.Q)
        se = support_embedding.unsqueeze(1)
        aggregation = torch.cat([context_feats * se, context_feats - se, context_feats], dim=2)
        dec = self.forward_decoder(context_locs, aggregation, query_locs, pc_dims, geo_dists, pre_enc_inds, impl)
        logits = self.mask_logits(geo_dists, dec[-1], [mask_features[s] for s in scenes], [locs[s] for s in scenes],
                                  query_locs, None, impl)
        return logits, geo_dists, pre_enc_inds


def gbias_torch_decoder_relative_pos(geo_dists, pre_enc_inds, query_locs, context_locs):
    """geoformer_fs.py:680-702 with torch ops on the tensors' device"""
    B = context_locs.shape[0]
    rel = torch.abs(query_locs[:, :, None, :] - context_locs[:, None, :, :])
    Q, Cn = rel.shape[1], rel.shape[2]
    g = torch.stack([geo_dists[b][:, pre_enc_inds[b].long()] for b in range(B)], dim=0)
    mx = torch.max(g, dim=2)[0]
    mx[mx < 0] = torch.max(mx)
    mx = mx[:, :, None, None].expand(B, Q, Cn, 3)
    g = g[:, :, :, None].repeat(1, 1, 1, 3)
    cond = g < 0
    g[cond] = mx[cond] + rel[cond]
    return g


def torch_mask_head_relative_coords(geo_dist, coords, fps_sampling_coords):
    """geoformer_fs.py:271-288 with torch ops on the tensors' device"""
    rel = fps_sampling_coords[:, None, :] - coords[None, :, :]
    Qn, Nn = geo_dist.shape
    mx = torch.max(geo_dist, dim=1)[0]
    mx[mx < 0] = torch.max(mx)
    mx = torch.sqrt(mx)[:, None, None].expand(Qn, Nn, 3)
    cond = (geo_dist < 0).unsqueeze(-1).expand(Qn, Nn, 3)
    rel[cond] = rel[cond] + mx[cond] * torch.sign(rel[cond])
    return rel.permute(0, 2, 1)
