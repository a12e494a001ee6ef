"""CPU restatement of set_aggregator's grouping + SharedMLP + pooling in TRAINING form -- TEST INFRASTRUCTURE ONLY.
Torch ops in the caller's dtype (float64 in the tests), so that autograd through it is the gradient oracle of
geoformer_b200.aggregate.group_mlp_pool_train.  The grouping follows lib/pointnet2/pointnet2_utils.py:330-341 as
oracle.aggregate.group_mlp_pool does; every layer is 1x1 conv [+ bias] [+ batch norm] + ReLU (pytorch_utils.py:59-104),
where a batch norm with batch statistics takes the mean and biased variance over (B, m, nsample) and updates its
running statistics as nn.BatchNorm2d does in training mode.  PINNED by tests/test_aggregate_train.py against
nn.Conv2d + nn.BatchNorm2d + ReLU + max_pool2d / avg_pool2d modules in float64."""
import torch
import torch.nn.functional as F


def grouped_input(xyz, new_xyz, features, idx, radius, normalize_xyz, use_xyz):
    """(B, 3+C, m, ns) tensor of QueryAndGroup (pointnet2_utils.py:330-341)"""
    B = idx.shape[0]
    ii = idx.long()
    xyz_t = xyz.transpose(1, 2)
    g_xyz = torch.stack([xyz_t[b][:, ii[b]] for b in range(B)]) - new_xyz.transpose(1, 2).unsqueeze(-1)
    if normalize_xyz:
        g_xyz = g_xyz / radius
    if features is None:
        return g_xyz
    g_f = torch.stack([features[b][:, ii[b]] for b in range(B)])
    return torch.cat([g_xyz, g_f], dim=1) if use_xyz else g_f


def shared_mlp_pool(x, layers, pooling="max", batch_stats=True, momentum=0.1, eps=1e-5, drop=()):
    """x (B, C, m, ns); layers: dicts with `w` (out, in), optional `b` (conv bias) and, for a batch norm, `gamma`,
    `beta` and running statistics `mean`, `var` (None: untracked) and `nbt` (num_batches_tracked).  With batch_stats
    the running statistics are updated in place (momentum None: cumulative average).  drop: "mean" and / or "var"
    stop autograd through the batch mean / variance (wrong gradients, to show what the tests' bounds catch).
    -> (out (B, C_out, m), [(batch mean, biased batch variance) or None per layer])"""
    stats = []
    for ly in layers:
        x = F.conv2d(x, ly["w"][:, :, None, None], ly.get("b"))
        if ly.get("gamma") is None:
            stats.append(None)
        elif batch_stats:
            n = x.numel() // x.shape[1]
            mean = x.mean(dim=(0, 2, 3))
            var = x.var(dim=(0, 2, 3), unbiased=False)
            stats.append((mean.detach(), var.detach()))
            mean = mean.detach() if "mean" in drop else mean
            var = var.detach() if "var" in drop else var
            if ly.get("mean") is not None:
                with torch.no_grad():
                    if ly.get("nbt") is not None:
                        ly["nbt"].add_(1)
                    f = momentum if momentum is not None else 1.0 / float(ly["nbt"])
                    ly["mean"].mul_(1 - f).add_(mean.detach() * f)
                    ly["var"].mul_(1 - f).add_(var.detach() * (n / (n - 1)) * f)
            x = (x - mean[None, :, None, None]) / torch.sqrt(var + eps)[None, :, None, None]
            x = x * ly["gamma"][None, :, None, None] + ly["beta"][None, :, None, None]
        else:
            stats.append(None)
            x = F.batch_norm(x, ly["mean"], ly["var"], ly["gamma"], ly["beta"], training=False, eps=eps)
        x = F.relu(x)
    if pooling == "max":
        x = F.max_pool2d(x, kernel_size=[1, x.size(3)])
    else:
        x = F.avg_pool2d(x, kernel_size=[1, x.size(3)])
    return x.squeeze(-1), stats
