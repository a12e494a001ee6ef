"""unique_with_inds (model/geoformer/geodesic_utils.py:4-8, SURVEY 8(a) row a8): the drop-in against
  * the definition (every unique column once, lexicographic order, index of its FIRST occurrence), checked by a
    plain numpy scan;
  * the committed fixture of the reference's own function's outputs, run on CPU (the only device where its
    scatter_ with duplicate indices is deterministic, SURVEY F2): tests/golden/unique_golden.npz;
on CPU tensors here and on CUDA tensors under -m gpu (where the reference itself is nondeterministic)."""
import os

import numpy as np
import pytest
import torch

from geoformer_b200.geodesic_utils import unique_with_inds

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden", "unique_golden.npz")


def _cases():
    g = torch.Generator().manual_seed(77)
    out = []
    for M, hi in ((1, 3), (17, 2), (500, 6), (4000, 40), (3000, 3)):
        out.append(torch.stack([torch.randint(0, hi, (M,), generator=g), torch.randint(0, hi, (M,), generator=g)]))
    out.append(torch.tensor([[5, 5, 5, 5], [1, 1, 1, 1]]))
    out.append(torch.zeros((2, 0), dtype=torch.int64))
    return out


def _definition(x):
    xn = x.numpy()
    cols = {}
    for i in range(xn.shape[1]):
        cols.setdefault((int(xn[0, i]), int(xn[1, i])), i)
    keys = sorted(cols)
    uniq = np.array(keys, dtype=np.int64).reshape(-1, 2).T
    return uniq, np.array([cols[k] for k in keys], dtype=np.int64)


def _check(device):
    gold = np.load(GOLD)
    for i, x in enumerate(_cases()):
        u, first = unique_with_inds(x.to(device), dim=-1)
        wu, wf = _definition(x)
        assert np.array_equal(u.cpu().numpy(), wu) and np.array_equal(first.cpu().numpy(), wf), i
        assert np.array_equal(u.cpu().numpy(), gold["u%d" % i]) and np.array_equal(first.cpu().numpy(), gold["f%d" % i]), i


def test_unique_with_inds_cpu_matches_definition_and_fixture():
    _check("cpu")


@pytest.mark.gpu
def test_unique_with_inds_cuda_is_deterministic_and_equal(cuda_lib):
    _check("cuda:0")
    x = _cases()[3].to("cuda:0")
    a = unique_with_inds(x)
    for _ in range(5):
        b = unique_with_inds(x)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


def make_golden():
    """python tests/test_unique_with_inds.py  (build container: outputs of the reference's own function on CPU)"""
    from oracle import ref_geodesic

    ref = ref_geodesic.load_reference_module().unique_with_inds
    out = {}
    for i, x in enumerate(_cases()):
        if x.size(1) == 0:
            u, f = _definition(x)
            out["u%d" % i], out["f%d" % i] = u.reshape(2, 0), f
            continue
        u, f = ref(x, dim=-1)
        out["u%d" % i], out["f%d" % i] = u.numpy(), f.numpy()
    np.savez_compressed(GOLD, **out)
    print("wrote", GOLD)


if __name__ == "__main__":
    import sys

    sys.path.insert(0, os.path.dirname(HERE))
    make_golden()
