"""CPU restatement of the mask head (model/geoformer/geoformer_fs.py:263-300, mask_heads_forward) -- TEST
INFRASTRUCTURE ONLY.  Torch ops in any dtype: the relative coordinates of oracle.bias.mask_head_relative_coords
(pinned to the reference's own statements by tests/golden/bias_golden.npz), then the concatenation with the mask
features and the two grouped conv1d of :291-297, written as the torch path of geoformer_b200/harness.py writes them.
Differentiable with respect to the mask features and the dynamic weights and biases."""
import torch
import torch.nn.functional as F

from .bias import mask_head_relative_coords


def mask_heads_forward(geo_dist, mask_features, weights, biases, num_insts, coords, fps_sampling_coords):
    """geo_dist (Q,N), mask_features (N,m) or (N,m,1), weights = [w0 (Q*m, m+3, 1), w1 (Q, m, 1)],
    biases = [b0 (Q*m), b1 (Q)], coords (N,3), fps_sampling_coords (Q,3) -> (Q,N) logits"""
    feats = mask_features.reshape(mask_features.shape[0], -1)
    rel = mask_head_relative_coords(geo_dist, coords, fps_sampling_coords).to(feats.dtype)  # :271-289
    x = feats.t()[None].repeat(num_insts, 1, 1)  # :269
    x = torch.cat([rel, x], dim=1).reshape(1, -1, feats.shape[0])  # :291-293
    for i, (w, b) in enumerate(zip(weights, biases)):
        x = F.conv1d(x, w, bias=b, stride=1, padding=0, groups=num_insts)  # :294-297
        if i < len(weights) - 1:
            x = F.relu(x)
    return x.reshape(num_insts, -1)
