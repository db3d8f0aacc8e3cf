"""CPU test of the SparseToDense return type (sparseeventid_b200/scn/dense_view.py): the interception logic is
exercised with pure-torch stand-ins for the two CUDA kernels, and must be indistinguishable from the dense tensor."""
import numpy as np
import torch
import torch.nn.functional as F

from helpers import random_sites
from sparseeventid_b200.scn.dense_view import SparseDenseTensor


def make(n=60, grid=(4, 5, 6), batch=3, c=7, seed=0):
    coords = torch.as_tensor(random_sites(n, grid, batch, seed))
    feats = torch.randn(coords.shape[0], c, requires_grad=True)
    keys = (coords[:, 3] << 48) | (coords[:, 0] << 32) | (coords[:, 1] << 16) | coords[:, 2]

    def materialize(f):
        d = torch.zeros((batch, c) + grid)
        return d.index_put((coords[:, 3], slice(None), coords[:, 0], coords[:, 1], coords[:, 2]), f.float()) \
            if False else _dense(f, coords, grid, batch)

    def pooled(f, b_of_row, nb, vol):
        out = torch.zeros(nb, f.shape[1])
        return out.index_add(0, b_of_row.long(), f) / vol
    return feats, coords, SparseDenseTensor(feats, keys, batch, grid, materialize, pooled), grid, batch


def _dense(f, coords, grid, batch):
    d = torch.zeros((batch, f.shape[1]) + tuple(grid))
    idx = (coords[:, 3], coords[:, 0], coords[:, 1], coords[:, 2])
    dperm = d.permute(0, 2, 3, 4, 1).contiguous()
    dperm = dperm.index_put(idx, f.float())
    return dperm.permute(0, 4, 1, 2, 3)


def test_metadata_and_fallback_ops():
    feats, coords, x, grid, batch = make()
    dense = _dense(feats, coords, grid, batch)
    assert tuple(x.shape) == (batch, 7) + grid and x.dim() == 5 and x.dtype == torch.float32 and x.requires_grad
    assert x.size(1) == 7 and x.numel() == dense.numel()
    assert torch.equal((x * 2 + 1).detach(), (dense * 2 + 1).detach())        # arithmetic materialises
    assert torch.equal(x[1, :, 2].detach(), dense[1, :, 2].detach())          # indexing materialises
    assert torch.allclose(x.sum(), dense.sum())
    assert torch.equal(F.avg_pool3d(x, 2).detach(), F.avg_pool3d(dense, 2).detach())   # not the full extent
    assert torch.equal(torch.sigmoid(x).detach(), torch.sigmoid(dense).detach())       # sigmoid(0) != 0


def test_reference_head_path_matches_dense_and_backpropagates():
    feats, coords, x, grid, batch = make()
    head = torch.nn.Sequential(torch.nn.AvgPool3d(list(grid)), torch.nn.Flatten(1, -1), torch.nn.Linear(7, 3))
    y = head(torch.tanh(x))                     # exactly what Encoder.forward + classification head do
    assert x._dense is None, "tanh + full-extent AvgPool3d must not materialise the dense tensor"
    feats2 = feats.detach().clone().requires_grad_(True)
    y_ref = head(torch.tanh(_dense(feats2, coords, grid, batch)))
    assert torch.allclose(y, y_ref, atol=1e-6)
    y.sum().backward()
    y_ref.sum().backward()
    assert torch.allclose(feats.grad, feats2.grad, atol=1e-6)
    z = torch.tanh(x)
    assert isinstance(z, SparseDenseTensor)
    assert torch.allclose(z.dense(), torch.tanh(_dense(feats, coords, grid, batch)))


def test_batch_indices_above_32767_decode_unsigned():
    """The batch field is the top 16 bits of an int64 key: batch 32768..65534 makes the key negative, and the row's
    sample must still come out as that index (not index - 65536) on the pooled head path."""
    grid, c, batch = (2, 2, 3), 3, 65535
    coords = torch.as_tensor(random_sites(30, grid, 3, seed=5))
    coords[:, 3] = torch.tensor([32767, 32768, 65534])[coords[:, 3]]
    feats = torch.randn(coords.shape[0], c, requires_grad=True)
    keys = (coords[:, 3] << 48) | (coords[:, 0] << 32) | (coords[:, 1] << 16) | coords[:, 2]
    assert bool((keys[coords[:, 3] >= 32768] < 0).all())

    def pooled(f, b_of_row, nb, vol):
        return torch.zeros(nb, f.shape[1]).index_add(0, b_of_row.long(), f) / vol
    x = SparseDenseTensor(feats, keys, batch, grid, lambda f: _dense(f, coords, grid, batch), pooled)
    assert torch.equal(x._batch_index().long(), coords[:, 3])
    y = F.avg_pool3d(torch.tanh(x), list(grid))
    assert x._dense is None
    feats2 = feats.detach().clone().requires_grad_(True)
    y_ref = F.avg_pool3d(_dense(torch.tanh(feats2), coords, grid, batch), list(grid))
    assert torch.allclose(y, y_ref, atol=1e-6)
    w = torch.randn(y.shape)
    (y * w).sum().backward()
    (y_ref * w).sum().backward()
    assert torch.allclose(feats.grad, feats2.grad, atol=1e-6)
