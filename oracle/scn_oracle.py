"""CPU oracle: a restatement of SparseConvNet's (SCN) CPU algorithms.

TEST INFRASTRUCTURE ONLY.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import this file.
The product path (``sparseeventid_b200`` / ``sparseconvnet``) never does.

PARITY UNPINNED: the arithmetic of the reference's hot path lives in the third-party
``sparseconvnet`` package (facebookresearch/SparseConvNet, version un-pinned by the
reference: ``requirements.txt`` is empty, ``README.md:20-21``).  It is absent from
``/root/reference`` and from this image, and the reference ships no tests or golden
vectors, so this restatement cannot be checked against SCN output.  It follows SCN's
published algorithm (SURVEY.md App. A) and is pinned instead by independent dense
identities (``tests/test_oracle_dense.py``: ``torch.nn.functional.conv3d``,
``F.batch_norm``), brute-force dictionary rulebooks, and float64 ``gradcheck``.

Every function cites the reference call site (relative to /root/reference) whose
behaviour it restates.
"""
from __future__ import annotations

import itertools
from typing import List, Sequence, Tuple

import numpy as np
import torch

# ----------------------------------------------------------------------------
# coordinates / keys
# ----------------------------------------------------------------------------


def as_triple(v, dimension: int = 3) -> Tuple[int, ...]:
    """SCN accepts int / list / tuple / tensor for sizes (src/networks/resnet.py:26-36)."""
    if isinstance(v, torch.Tensor):
        v = v.tolist()
    if isinstance(v, np.ndarray):
        v = v.tolist()
    if isinstance(v, (int, np.integer)):
        return tuple(int(v) for _ in range(dimension))
    v = tuple(int(x) for x in v)
    assert len(v) == dimension
    return v


def pack_keys(coords: np.ndarray) -> np.ndarray:
    """(x0..x_{D-1}, batch) int rows -> one uint64 key (batch | x0 | x1 | x2), 16 bits each.

    Lexicographic order of (batch, x0, x1, x2) == numeric order of the key.  The key is unsigned, as on the device:
    batch indices 32768..65534 set the top bit and must still sort after batch 0.
    """
    coords = np.asarray(coords, dtype=np.int64).astype(np.uint64)
    d = coords.shape[1] - 1
    key = coords[:, d]
    for a in range(3):
        key = key << np.uint64(16)
        if a < d:
            key = key | coords[:, a]
    return key


def unpack_keys(keys: np.ndarray, dimension: int = 3) -> np.ndarray:
    """uint64 (or int64 bit pattern) keys -> int64 rows (x0..x_{D-1}, batch)."""
    keys = np.asarray(keys).astype(np.uint64)
    field = [((keys >> np.uint64(s)) & np.uint64(0xFFFF)).astype(np.int64) for s in (32, 16, 0, 48)]
    return np.stack(field[:dimension] + [field[3]], axis=1)


# ----------------------------------------------------------------------------
# InputLayer  (src/networks/resnet.py:26-29,40-43,143)
# ----------------------------------------------------------------------------


def input_layer_rules(coords: np.ndarray, mode: int = 3):
    """Row assignment of scn.InputLayer [SCN-recalled, SURVEY App. A.2].

    coords: int64 [N, D+1], batch index LAST (src/io/data_transforms.py:43-46).
    Rows are numbered in first-appearance order with one counter over the whole batch.
    Returns (row_of_input [N] int64, active_coords [N0, D+1] int64).
    mode 0: caller guarantees no duplicates; 1: last wins; 2: first wins; 3: sum; 4: mean.
    """
    coords = np.asarray(coords, dtype=np.int64)
    n = coords.shape[0]
    if n == 0:
        return np.zeros((0,), np.int64), coords.reshape(0, coords.shape[1])
    keys = pack_keys(coords)
    uniq, first_idx, inverse = np.unique(keys, return_index=True, return_inverse=True)
    order = np.argsort(first_idx, kind="stable")      # unique keys by first appearance
    rank = np.empty_like(order)
    rank[order] = np.arange(order.shape[0])
    row_of_input = rank[inverse]
    active = coords[first_idx[order]]
    return row_of_input.astype(np.int64), active


def input_layer_forward(features: torch.Tensor, row_of_input: np.ndarray, n_active: int, mode: int = 3):
    rows = torch.as_tensor(row_of_input, dtype=torch.long)
    n, c = features.shape
    out = torch.zeros((n_active, c), dtype=features.dtype)
    if mode in (0, 3, 4):
        out.index_add_(0, rows, features)
        if mode == 4:
            cnt = torch.zeros((n_active,), dtype=features.dtype)
            cnt.index_add_(0, rows, torch.ones((n,), dtype=features.dtype))
            out = out / cnt[:, None]
    elif mode == 1:      # last wins
        for i in range(n):
            out[rows[i]] = features[i]
    elif mode == 2:      # first wins
        seen = set()
        for i in range(n):
            r = int(rows[i])
            if r not in seen:
                seen.add(r)
                out[r] = features[i]
    else:
        raise ValueError(mode)
    return out


def input_layer_backward(dout: torch.Tensor, row_of_input: np.ndarray, mode: int = 3):
    rows = torch.as_tensor(row_of_input, dtype=torch.long)
    if mode in (0, 3):
        return dout.index_select(0, rows)
    if mode == 4:
        cnt = torch.zeros((dout.shape[0],), dtype=dout.dtype)
        cnt.index_add_(0, rows, torch.ones((rows.shape[0],), dtype=dout.dtype))
        return dout.index_select(0, rows) / cnt.index_select(0, rows)[:, None]
    raise NotImplementedError("backward for modes 1/2 not needed by the reference")


def output_layer_forward(features: torch.Tensor, row_of_input: np.ndarray):
    """scn.OutputLayer: inverse of InputLayer, duplicates replicated (SURVEY App. A.7)."""
    return features.index_select(0, torch.as_tensor(row_of_input, dtype=torch.long))


def output_layer_backward(dout: torch.Tensor, row_of_input: np.ndarray, n_active: int):
    out = torch.zeros((n_active, dout.shape[1]), dtype=dout.dtype)
    out.index_add_(0, torch.as_tensor(row_of_input, dtype=torch.long), dout)
    return out


# ----------------------------------------------------------------------------
# rulebooks
# ----------------------------------------------------------------------------


def filter_offsets(filter_size: Sequence[int]) -> np.ndarray:
    """Row-major, last axis fastest, box [-f/2, +f/2] per axis (SURVEY App. A.3)."""
    f = tuple(int(x) for x in filter_size)
    assert all(fa % 2 == 1 for fa in f), "submanifold filters are odd on every axis"
    offs = list(itertools.product(*[range(-(fa // 2), fa // 2 + 1) for fa in f]))
    return np.asarray(offs, dtype=np.int64)


def _lookup(sorted_keys: np.ndarray, sorted_rows: np.ndarray, query: np.ndarray):
    pos = np.searchsorted(sorted_keys, query)
    pos_c = np.minimum(pos, sorted_keys.shape[0] - 1)
    hit = sorted_keys[pos_c] == query
    return np.where(hit, sorted_rows[pos_c], -1)


def submanifold_rulebook(coords: np.ndarray, filter_size: Sequence[int]) -> List[np.ndarray]:
    """scn.SubmanifoldConvolution rulebook (sparse_building_blocks.py:29-34) [SCN-recalled App. A.3].

    coords: active sites int64 [N, 4] = (x0,x1,x2,batch) in row order.
    Returns K arrays [P_k, 2] of (in_row, out_row): in = row(p + d_k), out = row(p).
    Pair order inside one k is by out row (SCN's is hash-iteration order; compare as sets).
    """
    coords = np.asarray(coords, dtype=np.int64)
    n = coords.shape[0]
    offs = filter_offsets(filter_size)
    rules = []
    if n == 0:
        return [np.zeros((0, 2), np.int64) for _ in offs]
    keys = pack_keys(coords)
    order = np.argsort(keys, kind="stable")
    skeys = keys[order]
    rows = np.arange(n, dtype=np.int64)
    for d in offs:
        q = coords.copy()
        q[:, :3] += d[None, :]
        ok = np.all((q[:, :3] >= 0) & (q[:, :3] < 65536), axis=1)
        qk = pack_keys(np.where(ok[:, None], q, 0))
        j = _lookup(skeys, order, qk)
        j = np.where(ok, j, -1)
        m = j >= 0
        rules.append(np.stack([j[m], rows[m]], axis=1))
    return rules


def submanifold_rulebook_bruteforce(coords, filter_size) -> List[List[Tuple[int, int]]]:
    """Pure-python dictionary version (small cases only) used to pin the vectorised one."""
    table = {tuple(int(v) for v in c): i for i, c in enumerate(np.asarray(coords))}
    offs = filter_offsets(filter_size)
    rules = [[] for _ in offs]
    for i, c in enumerate(np.asarray(coords)):
        for k, d in enumerate(offs):
            q = (int(c[0] + d[0]), int(c[1] + d[1]), int(c[2] + d[2]), int(c[3]))
            j = table.get(q)
            if j is not None:
                rules[k].append((j, i))
    return rules


def strided_rulebook(coords: np.ndarray, filter_size, filter_stride, in_spatial):
    """scn.Convolution rulebook + output grid (sparse_building_blocks.py:110-117) [App. A.4].

    out_spatial = (in - f)/s + 1 (asserted exact).  Input p reaches outputs q with
    ceil((p-f+1)/s) <= q <= floor(p/s), clipped to [0, out); offset index = rowmajor(p - q*s).
    Output rows: this restatement numbers them sorted by (batch, x0, x1, x2); SCN's own order
    is implementation-defined (hash iteration) and every consumer is permutation-invariant.
    Returns (out_coords [M,4], rules: K arrays [P_k,2] of (in_row,out_row), out_spatial).
    """
    f = as_triple(filter_size)
    s = as_triple(filter_stride)
    in_spatial = as_triple(in_spatial)
    out_spatial = []
    for a in range(3):
        assert (in_spatial[a] - f[a]) % s[a] == 0, "spatial size not compatible with filter/stride"
        out_spatial.append((in_spatial[a] - f[a]) // s[a] + 1)
    coords = np.asarray(coords, dtype=np.int64)
    n = coords.shape[0]
    K = f[0] * f[1] * f[2]
    cand_in, cand_k, cand_q = [], [], []
    # enumerate per-axis candidate outputs; (f/s rounded up)^3 candidates per input
    per_axis = [(f[a] + s[a] - 1) // s[a] for a in range(3)]
    for t in itertools.product(*[range(m) for m in per_axis]):
        q = np.empty((n, 3), np.int64)
        ok = np.ones((n,), bool)
        for a in range(3):
            qa = coords[:, a] // s[a] - t[a]
            off = coords[:, a] - qa * s[a]
            ok &= (qa >= 0) & (qa < out_spatial[a]) & (off < f[a])
            q[:, a] = qa
        offv = coords[:, :3] - q * np.asarray(s)[None, :]
        k = (offv[:, 0] * f[1] + offv[:, 1]) * f[2] + offv[:, 2]
        idx = np.nonzero(ok)[0]
        cand_in.append(idx)
        cand_k.append(k[idx])
        cand_q.append(np.concatenate([q[idx], coords[idx, 3:4]], axis=1))
    cin = np.concatenate(cand_in) if cand_in else np.zeros((0,), np.int64)
    ck = np.concatenate(cand_k) if cand_k else np.zeros((0,), np.int64)
    cq = np.concatenate(cand_q) if cand_q else np.zeros((0, 4), np.int64)
    if cq.shape[0] == 0:
        return np.zeros((0, 4), np.int64), [np.zeros((0, 2), np.int64) for _ in range(K)], tuple(out_spatial)
    qkeys = pack_keys(cq)
    ukeys, inv = np.unique(qkeys, return_inverse=True)
    out_coords = unpack_keys(ukeys)
    rules = []
    for k in range(K):
        m = ck == k
        pr = np.stack([cin[m], inv[m]], axis=1)
        pr = pr[np.lexsort((pr[:, 0], pr[:, 1]))]
        rules.append(pr)
    return out_coords, rules, tuple(out_spatial)


def normalize_rulebook(rules, in_coords, out_coords):
    """Order-normalised form (SURVEY App. A.3): per offset k, the sorted int64 array of
    (batch, in_coord[3], out_coord[3]) rows.  Two rulebooks are bit-exact iff these agree."""
    in_coords = np.asarray(in_coords, dtype=np.int64)
    out_coords = np.asarray(out_coords, dtype=np.int64)
    norm = []
    for r in rules:
        r = np.asarray(r, dtype=np.int64).reshape(-1, 2)
        if r.shape[0] == 0:
            norm.append(np.zeros((0, 7), np.int64))
            continue
        ic = in_coords[r[:, 0]]
        oc = out_coords[r[:, 1]]
        t = np.concatenate([ic[:, 3:4], ic[:, :3], oc[:, :3]], axis=1)
        assert np.array_equal(ic[:, 3], oc[:, 3]), "rule crosses batch samples"
        t = t[np.lexsort(t.T[::-1])]
        norm.append(t)
    return norm


# ----------------------------------------------------------------------------
# convolution arithmetic (SCN CPU path: per offset index_select -> mm -> index_add_)
# ----------------------------------------------------------------------------


def conv_forward(x: torch.Tensor, weight: torch.Tensor, bias, rules, n_out: int):
    """out = bias + sum_k scatter_add(x[rules[k].in] @ W[k] -> rules[k].out)  (App. A.3/A.4).

    weight: [K, Cin, Cout] (4-D SCN layouts [K,1,Cin,Cout] are viewed to 3-D by the caller).
    """
    K, cin, cout = weight.shape
    out = torch.zeros((n_out, cout), dtype=x.dtype)
    if bias is not None:
        out += bias[None, :]
    for k in range(K):
        r = rules[k]
        if len(r) == 0:
            continue
        r = torch.as_tensor(np.asarray(r), dtype=torch.long)
        out.index_add_(0, r[:, 1], x.index_select(0, r[:, 0]) @ weight[k])
    return out


def conv_backward(x, weight, has_bias, rules, dout):
    """dW[k] = x[in]^T @ dout[out]; dx[in] += dout[out] @ W[k]^T; dbias = dout.sum(0)."""
    K, cin, cout = weight.shape
    dx = torch.zeros_like(x)
    dw = torch.zeros_like(weight)
    for k in range(K):
        r = rules[k]
        if len(r) == 0:
            continue
        r = torch.as_tensor(np.asarray(r), dtype=torch.long)
        xi = x.index_select(0, r[:, 0])
        do = dout.index_select(0, r[:, 1])
        dw[k] = xi.t() @ do
        dx.index_add_(0, r[:, 0], do @ weight[k].t())
    db = dout.sum(0) if has_bias else None
    return dx, dw, db


def swap_rules(rules):
    """Deconvolution uses the strided rulebook with the columns swapped (App. A.7)."""
    return [np.asarray(r).reshape(-1, 2)[:, ::-1].copy() for r in rules]


# ----------------------------------------------------------------------------
# AveragePooling (sparse_building_blocks.py:150-154, the non-default ``Pooling`` down-sampling branch)
# ----------------------------------------------------------------------------


def average_pooling_forward(x: torch.Tensor, rules, n_out: int, volume: int, n_drop: int = 0):
    """out[o] = (1/volume) * sum over (i,o) in the strided rulebook of x[i, n_drop:]  [SCN-recalled].

    SCN's AveragePooling walks the same rulebook as a Convolution with filter == pool_size, stride == pool_stride and
    divides by the pool volume -- inactive sites count as zeros, which is what makes it equal to a dense
    ``avg_pool3d`` on the zero-filled volume at every active output site.  The first ``n_drop`` feature planes are
    skipped (SCN ``nFeaturesToDrop``)."""
    out = torch.zeros((n_out, x.shape[1] - n_drop), dtype=x.dtype)
    for r in rules:
        if len(r) == 0:
            continue
        r = torch.as_tensor(np.asarray(r), dtype=torch.long)
        out.index_add_(0, r[:, 1], x.index_select(0, r[:, 0])[:, n_drop:])
    return out / volume


def average_pooling_backward(dout: torch.Tensor, rules, n_in: int, volume: int, n_drop: int = 0):
    """dx[i, n_drop:] = dout[o] / volume for the (single) pair (i,o) of every input row; dropped planes get zeros."""
    dx = torch.zeros((n_in, dout.shape[1] + n_drop), dtype=dout.dtype)
    for r in rules:
        if len(r) == 0:
            continue
        r = torch.as_tensor(np.asarray(r), dtype=torch.long)
        dx[:, n_drop:].index_add_(0, r[:, 0], dout.index_select(0, r[:, 1]) / volume)
    return dx


# ----------------------------------------------------------------------------
# BatchNormalization (+ fused leaky ReLU)  (sparse_building_blocks.py:39,122)
# ----------------------------------------------------------------------------

BN_EPS = 1e-4
BN_MOMENTUM = 0.9


def batchnorm_forward(x, gamma, beta, running_mean, running_var, training: bool,
                      eps: float = BN_EPS, momentum: float = BN_MOMENTUM, leakiness: float = 1.0):
    """SCN BatchNormalization [App. A.5].  Updates running stats in place when training.
    Returns (out, save_mean, save_invstd)."""
    n = x.shape[0]
    if training:
        mean = x.mean(0) if n > 0 else torch.zeros_like(running_mean)
        s = ((x - mean[None, :]) ** 2).sum(0)
        with torch.no_grad():
            running_mean.mul_(momentum).add_((1 - momentum) * mean.to(running_mean.dtype))
            # SCN divides by (N-1); N==1 would give 0/0 (App. A.5 edge case).  Documented guard,
            # shared with the CUDA path: the divisor is max(N-1, 1).
            unbiased = s / max(n - 1, 1)
            running_var.mul_(momentum).add_((1 - momentum) * unbiased.to(running_var.dtype))
        invstd = (s / max(n, 1) + eps) ** -0.5
    else:
        mean = running_mean.to(x.dtype)
        invstd = (running_var.to(x.dtype) + eps) ** -0.5
    y = (x - mean[None, :]) * invstd[None, :]
    if gamma is not None:
        y = y * gamma[None, :] + beta[None, :]
    if leakiness != 1.0:
        y = torch.where(y > 0, y, y * leakiness)
    return y, mean, invstd


def batchnorm_backward(x, out, gamma, mean, invstd, dout, training: bool, leakiness: float = 1.0):
    """Backward of the above; d = dout * (out>0 ? 1 : leak)  [App. A.5]."""
    d = dout
    if leakiness != 1.0:
        d = torch.where(out > 0, dout, dout * leakiness)
    xhat = (x - mean[None, :]) * invstd[None, :]
    dbeta = d.sum(0)
    dgamma = (d * xhat).sum(0)
    g = gamma if gamma is not None else torch.ones_like(mean)
    if training:
        n = x.shape[0]
        dx = g[None, :] * invstd[None, :] * (d - dbeta[None, :] / n - xhat * dgamma[None, :] / n)
    else:
        dx = g[None, :] * invstd[None, :] * d
    return dx, dgamma, dbeta


# ----------------------------------------------------------------------------
# activations / AddTable  (sparse_building_blocks.py:45,76-82,96-98,128)
# ----------------------------------------------------------------------------

LEAK_DEFAULT = 1.0 / 3.0


def leaky_relu_forward(x, leak=LEAK_DEFAULT):
    return torch.where(x > 0, x, x * leak)


def leaky_relu_backward(x, dout, leak=LEAK_DEFAULT):
    return torch.where(x > 0, dout, dout * leak)


def add_table_forward(xs):
    out = xs[0].clone()
    for t in xs[1:]:
        out = out + t
    return out


# ----------------------------------------------------------------------------
# SparseToDense  (src/networks/resnet.py:123-125)
# ----------------------------------------------------------------------------


def sparse_to_dense_forward(x, coords, spatial, batch_size: int):
    """zeros([B, C, *spatial]); out[b, :, p] = x[row]  [App. A.8]."""
    spatial = as_triple(spatial)
    c = x.shape[1]
    out = torch.zeros((batch_size, c) + spatial, dtype=x.dtype)
    if x.shape[0]:
        co = torch.as_tensor(np.asarray(coords), dtype=torch.long)
        out[co[:, 3], :, co[:, 0], co[:, 1], co[:, 2]] = x
    return out


def sparse_to_dense_backward(dout, coords):
    co = torch.as_tensor(np.asarray(coords), dtype=torch.long)
    return dout[co[:, 3], :, co[:, 0], co[:, 1], co[:, 2]]
