"""set_aggregator (PointnetSAModuleVotesSeparate, lib/pointnet2/pointnet2_modules.py:150-249) with its grouping and its
SharedMLP fused into one kernel: FPS -> gather -> ball_query on the library's operators, then gf_group_mlp_pool
instead of group_points x2 + three Conv2d/BatchNorm2d/ReLU layers + a pooling op.

Two forms.  group_mlp_pool takes folded constants (batch norm with running statistics) and has nothing to
differentiate.  group_mlp_pool_train takes the unfolded parameters and is an autograd op: batch norm with batch
statistics where torch's would use them (training mode, or no running statistics), the running statistics updated as
nn.BatchNorm2d updates them, and a deterministic backward to the conv weights and biases, gamma, beta and the
features (gf_aggregate_train.cu).  aggregate() picks the form from the module's mode and whether a gradient is wanted.

aggregate_batch() takes a ragged batch (flat points + offsets, scenes of different sizes) the way forward_aggregator
holds it: ragged FPS and ball query (gf_furthest_point_sampling_batch, gf_ball_query_batch), then one MLP call over
the whole batch.
"""
import ctypes

import torch

from . import _capi as C
from .pointnet2 import _ext


def _shared_mlp_layers(mlp_module):
    """(conv, bn or None) per layer of a reference SharedMLP (pytorch_utils.py:9-32): Conv2d 1x1 [+ BatchNorm2d] [+ ReLU]"""
    layers = []
    for layer in mlp_module:
        conv = bn = None
        for sub in layer:
            if isinstance(sub, torch.nn.Conv2d):
                conv = sub
            elif isinstance(sub, torch.nn.Sequential) or isinstance(sub, torch.nn.BatchNorm2d):
                bn = sub[0] if isinstance(sub, torch.nn.Sequential) else sub
        C.require(conv is not None and conv.kernel_size == (1, 1), "SharedMLP layers must be 1x1 convolutions")
        layers.append((conv, bn))
    return layers


def _fold(W, bias, bn):
    """scale, shift of y = scale * (W x) + shift; bn: (gamma, beta, running_mean, running_var, eps) or None"""
    if bn is not None:
        gamma, beta, running_mean, running_var, eps = bn
        scale = (gamma.detach() / torch.sqrt(running_var.detach() + eps)).float()
        shift = (beta.detach() - running_mean.detach() * scale).float()
    else:
        scale = torch.ones(W.shape[0], device=W.device)
        shift = torch.zeros(W.shape[0], device=W.device)
    if bias is not None:
        shift = shift + bias.detach().float() * scale
    return scale, shift


def fold_shared_mlp(mlp_module):
    """(widths, weights, scales, shifts) of a reference SharedMLP (pytorch_utils.py:9-32) in eval mode: every layer is
    Conv2d 1x1 [+ BatchNorm2d] [+ ReLU]; batch norm folds into y = scale * (W x) + shift"""
    widths, Ws, scs, shs = [], [], [], []
    for conv, bn in _shared_mlp_layers(mlp_module):
        W = conv.weight.detach().reshape(conv.out_channels, conv.in_channels).float()
        if bn is not None:
            C.require(not bn.training, "fused aggregator: batch norm must be in eval mode (running statistics)")
        scale, shift = _fold(W, conv.bias, (bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
                             if bn is not None else None)
        if not widths:
            widths.append(conv.in_channels)
        widths.append(conv.out_channels)
        Ws.append(W.contiguous()), scs.append(scale.contiguous()), shs.append(shift.contiguous())
    return widths, Ws, scs, shs


def group_mlp_pool(xyz, new_xyz, features, idx, radius, normalize_xyz, use_xyz, widths, weights, scales, shifts,
                   pooling="max"):
    """xyz (B,N,3), new_xyz (B,m,3), features (B,C,N) or None, idx (B,m,nsample) i32 -> (B, widths[-1], m)"""
    C.check_cuda_f32(xyz, "xyz")
    C.check_cuda_f32(new_xyz, "new_xyz")
    C.check_cuda_i32(idx, "idx")
    C.require(pooling in ("max", "avg"), "pooling must be 'max' or 'avg' (rbf pooling is not fused)")
    B, N, _ = xyz.shape
    m, ns = idx.shape[1], idx.shape[2]
    Cn = 0
    if features is not None:
        C.check_cuda_f32(features, "features")
        C.require(features.shape[0] == B and features.shape[2] == N, "features must be (B, C, N)")
        Cn = features.shape[1]
    dev = xyz.device
    L = len(weights)
    ws = [w.to(device=dev, dtype=torch.float32).contiguous() for w in weights]
    sc = [s.to(device=dev, dtype=torch.float32).contiguous() for s in scales]
    sh = [s.to(device=dev, dtype=torch.float32).contiguous() for s in shifts]
    out = torch.empty((B, widths[-1], m), dtype=torch.float32, device=dev)
    arr = lambda ts: (ctypes.c_void_p * L)(*[t.data_ptr() for t in ts])  # noqa: E731
    with torch.cuda.device(dev):
        C.check(C.lib().gf_group_mlp_pool(C.ptr(xyz), C.ptr(new_xyz), C.ptr(features), C.ptr(idx), B, N, m, ns, Cn,
                                          ctypes.c_float(float(radius)), 1 if normalize_xyz else 0, 1 if use_xyz else 0,
                                          L, (ctypes.c_int * (L + 1))(*widths), arr(ws), arr(sc), arr(sh),
                                          1 if pooling == "avg" else 0, C.ptr(out), C.stream_of(dev)), "group_mlp_pool")
    return out


class _Spec:
    """the non-differentiable part of one group_mlp_pool_train call: data tensors, sizes, modes, constants"""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def _arr(ts):
    return (ctypes.c_void_p * len(ts))(*[C.ptr(t) for t in ts])


class _GroupMlpPool(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sp, features, *params):
        L = sp.L
        Ws, gammas, betas = params[:L], params[2 * L:3 * L], params[3 * L:]
        dev = sp.xyz.device
        B, N = sp.xyz.shape[0], sp.xyz.shape[1]
        m, ns = sp.idx.shape[1], sp.idx.shape[2]
        out = torch.empty((B, sp.widths[-1], m), dtype=torch.float32, device=dev)
        lib = C.lib()
        with torch.cuda.device(dev):
            nbytes = lib.gf_group_mlp_pool_train_workspace_bytes(B, m)
            ws = C.workspace.get(dev, "group_mlp_pool_train", nbytes)
            C.check(lib.gf_group_mlp_pool_train(
                C.ptr(sp.xyz), C.ptr(sp.new_xyz), C.ptr(features), C.ptr(sp.idx), B, N, m, ns, sp.Cn,
                ctypes.c_float(float(sp.radius)), 1 if sp.normalize_xyz else 0, 1 if sp.use_xyz else 0, L,
                (ctypes.c_int * (L + 1))(*sp.widths), _arr(Ws), _arr(gammas), _arr(betas),
                (ctypes.c_float * L)(*sp.eps), (ctypes.c_int * L)(*sp.batch), C.ptr(sp.consts), sp.pool_avg,
                C.ptr(out), C.ptr(ws), nbytes, C.stream_of(dev)), "group_mlp_pool_train")
        ctx.sp = sp
        ctx.save_for_backward(features, *Ws)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dout):
        sp = ctx.sp
        L = sp.L
        features, *Ws = ctx.saved_tensors
        dev = sp.xyz.device
        B, N = sp.xyz.shape[0], sp.xyz.shape[1]
        m, ns = sp.idx.shape[1], sp.idx.shape[2]
        dout = dout.to(torch.float32).contiguous()
        dWs = [torch.empty_like(w) for w in Ws]
        dvec = torch.empty((L, 3, 32), dtype=torch.float32, device=dev)
        want_df = features is not None and ctx.needs_input_grad[1]
        dfeat = torch.empty_like(features) if want_df else None
        lib = C.lib()
        with torch.cuda.device(dev):
            nbytes = lib.gf_group_mlp_pool_backward_workspace_bytes(B, N, m, ns, sp.Cn)
            ws = C.workspace.get(dev, "group_mlp_pool_backward", nbytes)
            C.check(lib.gf_group_mlp_pool_backward(
                C.ptr(sp.xyz), C.ptr(sp.new_xyz), C.ptr(features), C.ptr(sp.idx), B, N, m, ns, sp.Cn,
                ctypes.c_float(float(sp.radius)), 1 if sp.normalize_xyz else 0, 1 if sp.use_xyz else 0, L,
                (ctypes.c_int * (L + 1))(*sp.widths), _arr(Ws), (ctypes.c_int * L)(*sp.batch), C.ptr(sp.consts),
                sp.pool_avg, C.ptr(dout), C.ptr(dfeat), _arr(dWs), C.ptr(dvec), C.ptr(ws), nbytes,
                C.stream_of(dev)), "group_mlp_pool_backward")
        w = sp.widths[1:]
        dbias = [dvec[l, 0, :w[l]] for l in range(L)]
        dgamma = [dvec[l, 1, :w[l]] for l in range(L)]
        dbeta = [dvec[l, 2, :w[l]] for l in range(L)]
        return (None, dfeat, *dWs, *dbias, *dgamma, *dbeta)


def group_mlp_pool_train(xyz, new_xyz, features, idx, radius, normalize_xyz, use_xyz, weights, biases=None, gammas=None,
                         betas=None, running_means=None, running_vars=None, batch_stats=True, momentum=0.1, eps=1e-5,
                         pooling="max", num_batches_tracked=None):
    """group_mlp_pool with the SharedMLP's own parameters, differentiable.  Layer l is conv (weights[l] (out, in) or
    (out, in, 1, 1), biases[l] or None), then batch norm when gammas[l] is not None (gammas[l], betas[l], running
    statistics running_means[l] / running_vars[l] / num_batches_tracked[l] or None), then ReLU.  biases, gammas,
    betas, running_*, num_batches_tracked: lists with None entries (None: none for any layer); batch_stats, momentum,
    eps: one value or one per layer.  A batch norm with batch_stats normalises with the mean and biased variance of
    its input over all B * m * nsample elements and, when it has running statistics, updates them as nn.BatchNorm2d
    does in training mode (momentum None: cumulative average); otherwise it uses its running statistics.
    Gradients: weights, biases, gammas, betas, features.  xyz, new_xyz and idx are data.  Parameters on another
    device are copied to xyz's (differentiably; the constants of running-statistics layers are folded where the
    parameters live, as fold_shared_mlp folds them).  -> (B, C_out, m)"""
    C.check_cuda_f32(xyz, "xyz")
    C.check_cuda_f32(new_xyz, "new_xyz")
    C.check_cuda_i32(idx, "idx")
    C.require(pooling in ("max", "avg"), "pooling must be 'max' or 'avg' (rbf pooling is not fused)")
    if torch.is_grad_enabled() and (xyz.requires_grad or new_xyz.requires_grad):
        raise RuntimeError("group_mlp_pool_train: no gradient for xyz or new_xyz (they are data)")
    L = len(weights)
    C.require(1 <= L <= 4, "group_mlp_pool_train: 1..4 layers are fused")

    def per(v):
        return list(v) if isinstance(v, (list, tuple)) else [v] * L

    biases, gammas, betas = per(biases), per(gammas), per(betas)
    running_means, running_vars, nbt = per(running_means), per(running_vars), per(num_batches_tracked)
    batch_stats, momentum, eps = per(batch_stats), per(momentum), [float(e) for e in per(eps)]
    C.require(all(len(v) == L for v in (biases, gammas, betas, running_means, running_vars, nbt, batch_stats,
                                        momentum, eps)), "group_mlp_pool_train: one entry per layer")
    B, N, _ = xyz.shape
    m, ns = idx.shape[1], idx.shape[2]
    C.require(new_xyz.shape[0] == B and idx.shape[0] == B and new_xyz.shape[1] == m, "xyz, new_xyz, idx mismatch")
    dev = xyz.device
    Cn = 0
    if features is not None:
        C.check_cuda_f32(features, "features")
        C.require(features.shape[0] == B and features.shape[2] == N, "features must be (B, C, N)")
        Cn = features.shape[1]
    folded_W = [w.reshape(w.shape[0], -1) for w in weights]  # on the parameters' own device, as fold_shared_mlp
    widths = [folded_W[0].shape[1]] + [w.shape[0] for w in folded_W]
    C.require(widths[0] == (3 if use_xyz else 0) + Cn, "first layer takes %d channels, the input has %d"
              % (widths[0], (3 if use_xyz else 0) + Cn))
    C.require(all(folded_W[l + 1].shape[1] == widths[l + 1] for l in range(L - 1)), "layer widths do not chain")
    C.require(max(widths) <= 32, "widths above 32 are not fused")
    for t in folded_W + [t for t in biases + gammas + betas if t is not None]:
        C.require(isinstance(t, torch.Tensor) and t.is_floating_point(), "parameters must be float tensors")

    def on_dev(t):  # differentiable: the gradient goes back to the parameter's own device
        return t.to(device=dev, dtype=torch.float32) if t is not None else None
    batch = [bool(batch_stats[l]) and gammas[l] is not None for l in range(L)]
    consts = torch.zeros((L, 5, 32), dtype=torch.float32, device=dev)
    for l in range(L):
        if batch[l]:
            continue
        bn = (gammas[l], betas[l], running_means[l], running_vars[l], eps[l]) if gammas[l] is not None else None
        scale, shift = _fold(folded_W[l], biases[l], bn)
        w = widths[l + 1]
        consts[l, 0, :w], consts[l, 1, :w] = scale, shift
        if bn is not None:  # xhat = (W x - mean) * invstd for the gradient of gamma
            mean = running_means[l].detach().float().to(dev)
            consts[l, 2, :w] = mean - biases[l].detach().float().to(dev) if biases[l] is not None else mean
            consts[l, 3, :w] = torch.rsqrt(running_vars[l].detach().float().to(dev) + eps[l])
    zeros = [torch.zeros(w, device=dev) for w in widths[1:]]
    sp = _Spec(xyz=xyz, new_xyz=new_xyz, idx=idx, L=L, Cn=Cn, radius=radius, normalize_xyz=normalize_xyz,
               use_xyz=use_xyz, widths=widths, batch=[1 if b else 0 for b in batch], eps=eps, consts=consts,
               pool_avg=1 if pooling == "avg" else 0)
    params = ([on_dev(w).contiguous() for w in folded_W] + [on_dev(b) if b is not None else z for b, z in zip(biases, zeros)]
              + [on_dev(g) if g is not None else z for g, z in zip(gammas, zeros)]
              + [on_dev(b) if b is not None else z for b, z in zip(betas, zeros)])
    out = _GroupMlpPool.apply(sp, features, *params)
    n = B * m * ns
    with torch.no_grad():
        for l in range(L):
            if not batch[l] or running_means[l] is None:
                continue
            w = widths[l + 1]
            rm, rv = running_means[l], running_vars[l]
            mean = (consts[l, 2, :w] + (on_dev(biases[l]).detach() if biases[l] is not None else 0)).to(rm)
            var = (consts[l, 4, :w] * (n / (n - 1) if n > 1 else 1.0)).to(rv)
            if nbt[l] is not None:
                nbt[l].add_(1)
            f = momentum[l] if momentum[l] is not None else 1.0 / nbt[l].to(rm)
            rm.mul_(1 - f).add_(mean * f)
            rv.mul_(1 - f).add_(var * f)
    return out


def aggregate(module, xyz, features, inds=None, npoint_new=None, pooling=None):
    """module.group_points(...) followed by module.mlp(...) of a reference PointnetSAModuleVotesSeparate (the calls of
    geoformer_fs.py:643-657 / :413-416), fused: returns (new_xyz (B,m,3), new_features (B,C_out,m), inds (B,m) i32).
    xyz (B,N,3), features (B,C,N)."""
    npoint = npoint_new if npoint_new is not None else module.npoint
    C.require(npoint is not None, "GroupAll aggregators (npoint=None) are not fused")
    if inds is None:
        inds = _ext.furthest_point_sampling(xyz.contiguous(), int(npoint))
    else:
        C.require(inds.shape[1] == npoint, "inds must have npoint columns")
    new_xyz = _ext.gather_points(xyz.transpose(1, 2).contiguous(), inds).transpose(1, 2).contiguous()
    g = module.grouper
    idx = _ext.ball_query(new_xyz, xyz.contiguous(), float(g.radius), int(g.nsample))
    return new_xyz, _mlp(module, xyz, new_xyz, features, idx, pooling), inds


def _mlp(module, xyz, new_xyz, features, idx, pooling):
    """module.mlp on the groups of idx, in the form the module's mode and the gradient wanted choose: the folded
    inference kernel, or group_mlp_pool_train"""
    g = module.grouper
    pooling = pooling if pooling is not None else module.pooling
    features = features.contiguous() if features is not None else None
    layers = _shared_mlp_layers(module.mlp_module)
    batch = [bn is not None and (bn.training or not bn.track_running_stats) for _, bn in layers]
    params = [t for conv, bn in layers for t in (conv.weight, conv.bias) + ((bn.weight, bn.bias) if bn else ())
              if t is not None]
    wants_grad = torch.is_grad_enabled() and any(t.requires_grad for t in params + [xyz, features] if t is not None)
    if not any(batch) and not wants_grad:
        widths, Ws, scs, shs = fold_shared_mlp(module.mlp_module)
        return group_mlp_pool(xyz.contiguous(), new_xyz, features, idx, g.radius, g.normalize_xyz, g.use_xyz, widths,
                              Ws, scs, shs, pooling=pooling)

    def ones_if_none(t, bn, value):  # BatchNorm2d(affine=False)
        return t if t is not None else torch.full((bn.num_features,), value, device=xyz.device)

    return group_mlp_pool_train(
        xyz.contiguous(), new_xyz, features, idx, g.radius, g.normalize_xyz, g.use_xyz,
        [conv.weight for conv, _ in layers], [conv.bias for conv, _ in layers],
        [ones_if_none(bn.weight, bn, 1.0) if bn else None for _, bn in layers],
        [ones_if_none(bn.bias, bn, 0.0) if bn else None for _, bn in layers],
        [bn.running_mean if bn else None for _, bn in layers], [bn.running_var if bn else None for _, bn in layers],
        batch, [bn.momentum if bn else None for _, bn in layers], [bn.eps if bn else 1e-5 for _, bn in layers],
        pooling=pooling,
        num_batches_tracked=[bn.num_batches_tracked if bn is not None and bn.training and bn.track_running_stats
                             else None for _, bn in layers])


def batch_offsets_list(batch_offsets, n_points):
    """batch_offsets (B+1) tensor or sequence -> list of ints, checked: starts at 0, rises strictly (no empty scene)
    and ends at n_points"""
    off = [int(v) for v in (batch_offsets.tolist() if isinstance(batch_offsets, torch.Tensor) else batch_offsets)]
    C.require(len(off) >= 2 and off[0] == 0, "batch_offsets must start at 0 and describe at least one scene")
    C.require(all(b > a for a, b in zip(off, off[1:])), "batch_offsets must rise strictly (a scene is empty)")
    C.require(off[-1] == n_points, "batch_offsets end at %d, the batch has %d points" % (off[-1], n_points))
    return off


def furthest_point_sampling_batch(xyz, offsets, m):
    """xyz (sum N, 3) f32 flat, offsets (B+1) host ints -> (B, m) i32 scene-local seeds; row b equals
    _ext.furthest_point_sampling of scene b alone"""
    C.check_cuda_f32(xyz, "xyz")
    B = len(offsets) - 1
    out = torch.empty((B, int(m)), dtype=torch.int32, device=xyz.device)
    offs = (ctypes.c_int * (B + 1))(*offsets)
    lib = C.lib()
    with torch.cuda.device(xyz.device):
        nbytes = lib.gf_fps_batch_workspace_bytes(offs, B, int(m))
        ws = C.workspace.get(xyz.device, "fps", nbytes) if nbytes else None
        C.check(lib.gf_furthest_point_sampling_batch(C.ptr(xyz), offs, B, int(m), C.ptr(out), C.ptr(ws), nbytes,
                                                     C.stream_of(xyz.device)), "furthest_point_sampling_batch")
    return out


def ball_query_batch(new_xyz, xyz, offsets, radius, nsample):
    """new_xyz (B, m, 3), xyz (sum N, 3) flat, offsets (B+1) host ints -> (B, m, nsample) i32 scene-local; row b
    equals _ext.ball_query of scene b alone"""
    C.check_cuda_f32(new_xyz, "new_xyz")
    C.check_cuda_f32(xyz, "xyz")
    B, m = new_xyz.shape[0], new_xyz.shape[1]
    C.require(B == len(offsets) - 1, "new_xyz has %d scenes, offsets %d" % (B, len(offsets) - 1))
    out = torch.empty((B, m, int(nsample)), dtype=torch.int32, device=new_xyz.device)
    with torch.cuda.device(new_xyz.device):
        C.check(C.lib().gf_ball_query_batch(C.ptr(new_xyz), C.ptr(xyz), (ctypes.c_int * (B + 1))(*offsets), B, m,
                                            float(radius), int(nsample), C.ptr(out), C.stream_of(new_xyz.device)),
                "ball_query_batch")
    return out


def aggregate_batch(module, locs_float_, features_, batch_offsets_, inds=None, npoint_new=None, pooling=None):
    """aggregate() over a RAGGED batch, as forward_aggregator (geoformer_fs.py:619-660) holds it: locs_float_ (sum N, 3),
    features_ (sum N, C) point-major or None, batch_offsets_ (B+1) tensor or list.  One FPS launch and one ball-query
    launch (per 32 scenes) for all scenes, then ONE group_mlp_pool[_train] call over the whole batch as a single scene
    of sum N points and B * m centres: batch statistics cover all B * m * nsample samples, as the reference's one
    module.mlp call over the concatenated groups.  inds (B, m) i32 scene-local seeds skip the FPS.
    Returns (context_locs (B, m, 3), context_feats (B, C_out, m), pre_enc_inds (B, m) i32)."""
    npoint = int(npoint_new if npoint_new is not None else module.npoint)
    C.check_cuda_f32(locs_float_, "locs_float_")
    C.require(locs_float_.dim() == 2 and locs_float_.shape[1] == 3, "locs_float_ must be (sum N, 3)")
    n_points = locs_float_.shape[0]
    off = batch_offsets_list(batch_offsets_, n_points)
    B = len(off) - 1
    dev = locs_float_.device
    if features_ is not None:
        C.require(isinstance(features_, torch.Tensor) and features_.is_cuda, "features_: CPU not supported")
        C.require(features_.dtype == torch.float32, "features_ must be a float tensor")
        C.require(features_.dim() == 2 and features_.shape[0] == n_points,
                  "features_ must be (sum N, C) with sum N = %d rows" % n_points)
    if inds is None:
        inds = furthest_point_sampling_batch(locs_float_, off, npoint)
    else:
        C.check_cuda_i32(inds, "inds")
        C.require(tuple(inds.shape) == (B, npoint), "inds must be (B, npoint)")
    start = torch.tensor(off[:-1], dtype=torch.int32, device=dev)
    new_xyz = locs_float_.detach()[(inds + start[:, None]).long()]
    g = module.grouper
    idx = ball_query_batch(new_xyz, locs_float_, off, g.radius, g.nsample)
    # the whole batch as one scene: global indices, features channel-major once
    idx1 = (idx + start[:, None, None]).reshape(1, B * npoint, -1)
    feats1 = features_.t().unsqueeze(0).contiguous() if features_ is not None else None
    out = _mlp(module, locs_float_.unsqueeze(0), new_xyz.reshape(1, B * npoint, 3), feats1, idx1, pooling)
    return new_xyz, out[0].reshape(out.shape[1], B, npoint).transpose(0, 1).contiguous(), inds
