"""The two oracles pin each other: the plain-C restatement (oracle/scn_oracle_c.c: chained hash map, explicit loops)
and the Python one (oracle/scn_oracle.py: sorted arrays + searchsorted, index_add_) were written independently from
the same published semantics (SURVEY.md App. A) and must agree exactly on the integer work -- InputLayer row numbering,
submanifold and strided rulebooks -- and to fp64 round-off on a rulebook convolution.  (Both remain PARITY UNPINNED
against SparseConvNet itself.)"""
import numpy as np
import pytest
import torch

from helpers import blob_sites, random_sites
from oracle import c_oracle as OC
from oracle import scn_oracle as O


def sites(kind, seed):
    if kind == "blob":
        return blob_sites(250, (20, 16, 24), 3, seed=seed)
    return random_sites(400, (20, 16, 24), 2, seed=seed)


@pytest.mark.parametrize("dup", [0, 57])
def test_input_layer_row_numbering(dup):
    c = sites("rand", 1)
    if dup:
        rng = np.random.default_rng(3)
        c = np.concatenate([c, c[rng.integers(0, c.shape[0], dup)]], 0)[rng.permutation(c.shape[0] + dup)]
    rows_py, active_py = O.input_layer_rules(c)
    rows_c, active_c = OC.input_rules(c)
    assert np.array_equal(rows_py, rows_c) and np.array_equal(active_py, active_c)


@pytest.mark.parametrize("filt", [(3, 3, 3), (1, 3, 3), (5, 5, 5), (1, 1, 1)])
@pytest.mark.parametrize("kind,seed", [("blob", 4), ("rand", 5)])
def test_submanifold_rulebook(filt, kind, seed):
    _, active = O.input_layer_rules(sites(kind, seed))
    want = O.submanifold_rulebook(active, filt)
    got, _ = OC.subm_rules(active, filt)
    assert len(got) == len(want)
    for a, b in zip(O.normalize_rulebook(got, active, active), O.normalize_rulebook(want, active, active)):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("stride,grid,batch0", [((2, 2, 2), (20, 16, 24), 0), ((1, 2, 2), (3, 16, 24), 0),
                                                ((2, 2, 2), (20, 16, 24), 32767), ((1, 2, 2), (3, 16, 24), 32767)],
                         ids=["stride0-grid0", "stride1-grid1", "stride0-grid0-batch32767", "stride1-grid1-batch32767"])
def test_strided_rulebook(stride, grid, batch0):
    """batch0 = 32767: the samples 32767 and 32768 straddle the top bit of the packed key, whose order is unsigned."""
    rng = np.random.default_rng(8)
    b = batch0 + rng.integers(0, 2, 500)
    pts = np.unique(np.stack([rng.integers(0, grid[a], 500) for a in range(3)] + [b], 1), axis=0)
    _, active = O.input_layer_rules(pts.astype(np.int64))
    out_py, rules_py, _ = O.strided_rulebook(active, stride, stride, grid)
    out_c, rules_c = OC.strided_rules(active, stride)
    k = O.pack_keys(out_py)
    assert np.array_equal(out_py, out_c) and np.all(k[1:] > k[:-1])
    assert np.array_equal(np.unique(out_py[:, 3]), np.unique(active[:, 3]))
    for a, b in zip(O.normalize_rulebook(rules_c, active, out_c), O.normalize_rulebook(rules_py, active, out_py)):
        assert np.array_equal(a, b)


def test_rulebook_convolution_fp64():
    _, active = O.input_layer_rules(sites("blob", 9))
    n, cin, cout = active.shape[0], 5, 7
    rules, raw = OC.subm_rules(active, (3, 3, 3))
    g = torch.Generator().manual_seed(0)
    x = torch.randn(n, cin, generator=g, dtype=torch.float64)
    W = torch.randn(27, cin, cout, generator=g, dtype=torch.float64)
    bias = torch.randn(cout, generator=g, dtype=torch.float64)
    want = O.conv_forward(x, W, bias, O.submanifold_rulebook(active, (3, 3, 3)), n)
    got = OC.conv_forward(x.numpy(), W.numpy(), bias.numpy(), raw, n)
    assert np.allclose(got, want.numpy(), rtol=1e-12, atol=1e-12)
