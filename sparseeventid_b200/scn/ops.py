"""Thin tensor-level wrappers over the C ABI (include/scn_b200.h).  No autograd here.

Every function takes CUDA tensors, allocates outputs with torch's caching allocator on the
current stream, and calls libscn_b200.so through ctypes.  Nothing here computes on the host.
"""
from __future__ import annotations

import torch

from .. import _lib as L


class Profiler:
    """CUDA-event timing of individual C-ABI calls on the launching stream (bench.py's roofline pass)."""

    def __init__(self):
        self.recs = []

    def begin(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def end(self, e0, **meta):
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        meta["_e0"], meta["_e1"] = e0, e1
        self.recs.append(meta)

    def finish(self):
        torch.cuda.synchronize()
        pairs = {}
        out = []
        for r in self.recs:
            r = dict(r)
            r["ms"] = r.pop("_e0").elapsed_time(r.pop("_e1"))
            nbr = r.pop("nbr", None)
            if nbr is not None:
                key = (nbr.data_ptr(), tuple(nbr.shape))
                if key not in pairs:
                    pairs[key] = int((nbr >= 0).sum().item())
                r["pairs"] = pairs[key]
            out.append(r)
        return out


_profiler = None


def set_profiler(p):
    global _profiler
    _profiler = p


def profiling() -> bool:
    return _profiler is not None


_scratch = {}


def stats_scratch(device, c: int) -> torch.Tensor:
    """fp64 [2*C] scratch of the column reductions: one buffer per device shared by every layer (stream-ordered)."""
    t = _scratch.get(device)
    if t is None or t.numel() < 2 * c:
        t = torch.empty((max(2 * c, 2048),), dtype=torch.float64, device=device)
        _scratch[device] = t
    return t


def _i32(n, device):
    return torch.empty((n,), dtype=torch.int32, device=device)


def pad128(n: int) -> int:
    return (n + 127) // 128 * 128


# ---------------------------------------------------------------------------- hash / rulebooks


def pack_coords(coords: torch.Tensor, dimension: int, info: torch.Tensor = None) -> torch.Tensor:
    """info: optional zeroed int32[4] device tensor; [1] is set when a coordinate / batch index does not fit its 16-bit
    key field, [2] receives the largest batch index (see scn_pack_coords_checked)."""
    L.require_cuda(coords, "pack_coords")
    if coords.dtype not in L.COORD_CODES:
        coords = coords.long()
    coords = coords.contiguous()
    n, ncols = coords.shape
    keys = torch.empty((n,), dtype=torch.int64, device=coords.device)
    L.check(L.lib().scn_pack_coords_checked(L.ptr(coords), L.COORD_CODES[coords.dtype], n, ncols, dimension, L.ptr(keys),
                                            L.ptr(info), L.stream()), "scn_pack_coords_checked")
    return keys


def unpack_keys(keys: torch.Tensor) -> torch.Tensor:
    n = keys.shape[0]
    out = torch.empty((n, 4), dtype=torch.int32, device=keys.device)
    L.check(L.lib().scn_unpack_keys(L.ptr(keys), n, L.ptr(out), L.stream()), "scn_unpack_keys")
    return out


def new_table(n: int, device):
    cap = int(L.lib().scn_hash_capacity(n))
    tk = torch.empty((cap,), dtype=torch.int64, device=device)
    tv = torch.empty((cap,), dtype=torch.int32, device=device)
    return tk, tv, cap


def hash_build(keys: torch.Tensor):
    n = keys.shape[0]
    tk, tv, cap = new_table(n, keys.device)
    L.check(L.lib().scn_hash_build(L.ptr(keys), n, L.ptr(tk), L.ptr(tv), cap, L.stream()), "scn_hash_build")
    return tk, tv, cap


def hash_lookup(queries: torch.Tensor, tk, tv, cap) -> torch.Tensor:
    n = queries.shape[0]
    out = _i32(n, queries.device)
    L.check(L.lib().scn_hash_lookup(L.ptr(queries), n, L.ptr(tk), L.ptr(tv), cap, L.ptr(out), L.stream()),
            "scn_hash_lookup")
    return out


def input_layer_rules(keys_in: torch.Tensor, info: torch.Tensor = None):
    """-> (row_of_input int32 [n], keys_out int64 [n_active], table_keys, table_vals, cap, info list).  One D2H sync:
    `info` (the int32[4] tensor pack_coords filled) comes back as [n_active, range violation flag, max batch index, 0]."""
    n = keys_in.shape[0]
    dev = keys_in.device
    tk, tv, cap = new_table(n, dev)
    rows = _i32(n, dev)
    keys_out = torch.empty((n,), dtype=torch.int64, device=dev)
    n_active = info if info is not None else torch.zeros((4,), dtype=torch.int32, device=dev)
    ws_bytes = int(L.lib().scn_input_rules_workspace(n))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_input_layer_rules(L.ptr(keys_in), n, L.ptr(tk), L.ptr(tv), cap, L.ptr(rows), L.ptr(keys_out),
                                          L.ptr(n_active), L.ptr(ws), ws_bytes, L.stream()), "scn_input_layer_rules")
    if p:
        p.end(e0, kind="rulebook_input", bytes=20.0 * n, rows=n)
    got = n_active.tolist()
    na = int(got[0])
    return rows, keys_out[:na], tk, tv, cap, got


def subm_rulebook(keys, tk, tv, cap, filt) -> torch.Tensor:
    n = keys.shape[0]
    n_pad = pad128(n)
    K = filt[0] * filt[1] * filt[2]
    nbr = torch.empty((K, n_pad), dtype=torch.int32, device=keys.device)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_subm_rulebook(L.ptr(keys), n, L.ptr(tk), L.ptr(tv), cap, filt[0], filt[1], filt[2],
                                      L.ptr(nbr), n_pad, L.stream()), "scn_subm_rulebook")
    if p:
        p.end(e0, kind="rulebook_subm", bytes=8.0 * n + 4.0 * K * n_pad, K=K, rows=n)
    return nbr


def strided_rulebook(keys_in, stride):
    """-> (keys_out int64 [n_out] in first-appearance order, out_row_of_in int32 [n], off_of_in int32 [n],
    (table_keys, table_vals, cap) = the coarse level's hash table).  One D2H sync."""
    n = keys_in.shape[0]
    dev = keys_in.device
    keys_out = torch.empty((n,), dtype=torch.int64, device=dev)
    out_row = _i32(n, dev)
    off = _i32(n, dev)
    n_out = torch.zeros((1,), dtype=torch.int32, device=dev)
    tk, tv, cap = new_table(n, dev)
    ws_bytes = int(L.lib().scn_strided_hash_workspace(n))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_strided_rulebook_hash(L.ptr(keys_in), n, stride[0], stride[1], stride[2], L.ptr(tk), L.ptr(tv), cap,
                                              L.ptr(keys_out), L.ptr(out_row), L.ptr(off), L.ptr(n_out), L.ptr(ws), ws_bytes,
                                              L.stream()), "scn_strided_rulebook_hash")
    if p:
        p.end(e0, kind="rulebook_strided", bytes=24.0 * n, rows=n)
    m = int(n_out.item())
    return keys_out[:m], out_row, off, (tk, tv, cap)


def strided_tables(out_row, off, K, n_in, n_out):
    dev = out_row.device
    down = torch.empty((K, pad128(n_out)), dtype=torch.int32, device=dev)
    up = torch.empty((K, pad128(n_in)), dtype=torch.int32, device=dev)
    L.check(L.lib().scn_strided_tables(L.ptr(out_row), L.ptr(off), n_in, K, L.ptr(down), pad128(n_out), L.ptr(up),
                                       pad128(n_in), L.stream()), "scn_strided_tables")
    return down, up


def rulebook_pairs(nbr: torch.Tensor, n: int):
    """SCN-format rulebook: list of K int32 [P_k, 2] (in,out) tensors, pairs sorted by out row."""
    K, n_pad = nbr.shape
    dev = nbr.device
    counts = torch.zeros((K,), dtype=torch.int32, device=dev)
    L.check(L.lib().scn_rulebook_count(L.ptr(nbr), K, n, n_pad, L.ptr(counts), L.stream()), "scn_rulebook_count")
    total = int(counts.sum().item())
    pin, pout = _i32(max(total, 1), dev), _i32(max(total, 1), dev)
    offs = _i32(K + 1, dev)
    ws_bytes = int(L.lib().scn_rulebook_workspace(K, n_pad))
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    L.check(L.lib().scn_rulebook_pairs(L.ptr(nbr), K, n, n_pad, L.ptr(pin), L.ptr(pout), L.ptr(offs), L.ptr(ws),
                                       ws_bytes, L.stream()), "scn_rulebook_pairs")
    o = offs.cpu().tolist()
    return [torch.stack([pin[o[k]:o[k + 1]], pout[o[k]:o[k + 1]]], 1) for k in range(K)]


# ---------------------------------------------------------------------------- convolution


_DT = {torch.float32: L.SCN_F32, torch.bfloat16: L.SCN_BF16}


def conv_path(K, n_in, n_out, prec, feat_dtype) -> int:
    """0 = exact fp32 FMA kernels, 1 = mma.sync tensor cores, 2 = tcgen05 tensor cores (see scn_b200.h)."""
    return int(L.lib().scn_conv_path(K, n_in, n_out, prec, _DT[feat_dtype]))


def prep_weights(w3: torch.Tensor, transpose: bool, mirror: bool, prec: int, feat_dtype) -> torch.Tensor:
    """w3: fp32 [K, Cin, Cout] -> B_k laid out for the kernel family that will run on feat_dtype features."""
    K, cin, cout = w3.shape
    n_in, n_out = (cout, cin) if transpose else (cin, cout)
    nbytes = int(L.lib().scn_conv_prep_bytes(K, n_in, n_out, prec, _DT[feat_dtype]))
    out = torch.empty((nbytes,), dtype=torch.uint8, device=w3.device)
    L.check(L.lib().scn_conv_prep_weights(L.ptr(w3), K, cin, cout, int(transpose), int(mirror), prec, _DT[feat_dtype],
                                          L.ptr(out), L.stream()), "scn_conv_prep_weights")
    return out


def conv_forward(x, nbr, n_out_rows, n_in, n_out, bprep, bias, prec, out_dtype, kind="conv_fwd") -> torch.Tensor:
    K, n_pad = nbr.shape
    tc = conv_path(K, n_in, n_out, prec, out_dtype) > 0
    if tc and x.dtype != out_dtype:
        x = convert(x, out_dtype)
    out = torch.empty((n_out_rows, n_out), dtype=out_dtype, device=x.device)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_conv_forward(L.ptr(x), L.dtype_code(x), x.shape[0], L.ptr(nbr), K, n_out_rows, n_pad, n_in,
                                     n_out, L.ptr(bprep), L.ptr(bias), prec, L.ptr(out), L.dtype_code(out),
                                     L.stream()), "scn_conv_forward")
    if p:
        p.end(e0, kind=kind, K=K, n_in=n_in, n_out=n_out, rows_in=x.shape[0], rows_out=n_out_rows, nbr=nbr, tc=tc)
    return out


def conv_wgrad(x, dout, nbr, n_rows, n_in, n_out, prec) -> torch.Tensor:
    K, n_pad = nbr.shape
    tc = conv_path(K, n_in, n_out, prec, dout.dtype) > 0
    if tc and x.dtype != dout.dtype:
        x = convert(x, dout.dtype)
    dw = torch.zeros((K, n_in, n_out), dtype=torch.float32, device=x.device)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_conv_wgrad(L.ptr(x), L.dtype_code(x), L.ptr(dout), L.dtype_code(dout), L.ptr(nbr), K, n_rows,
                                   n_pad, n_in, n_out, prec, L.ptr(dw), L.stream()), "scn_conv_wgrad")
    if p:
        p.end(e0, kind="conv_wgrad", K=K, n_in=n_in, n_out=n_out, rows_in=x.shape[0], rows_out=n_rows, nbr=nbr, tc=tc)
    return dw


def conv_prep_bytes(K, n_in, n_out, prec, feat_dtype) -> int:
    return int(L.lib().scn_conv_prep_bytes(K, n_in, n_out, prec, _DT[feat_dtype]))


def conv_module_forward(x, weight, bias, nbr, n_out_rows, K, cin, cout, prec, out_dtype, wimg, skip_prep) -> torch.Tensor:
    """One C-ABI call: weight re-layout into `wimg` (unless skip_prep) + out = bias + conv(x).  weight/bias fp32."""
    out = torch.empty((n_out_rows, cout), dtype=out_dtype, device=x.device)
    L.check(L.lib().scn_conv_module_forward(x.data_ptr(), _DT[x.dtype], x.shape[0], nbr.data_ptr(), K, n_out_rows,
                                            nbr.shape[1], cin, cout, weight.data_ptr(),
                                            None if bias is None else bias.data_ptr(), prec, wimg.data_ptr(),
                                            int(skip_prep), out.data_ptr(), _DT[out_dtype], L.stream()),
            "scn_conv_module_forward")
    return out


def conv_module_backward(x, dout, weight, nbr_fwd, nbr_bwd, n_out_rows, K, cin, cout, mirror, prec, wimg_t, skip_prep,
                         need_dx, dw, zero_dw, dbias, accumulate_dbias, dout_colsum=None):
    """One C-ABI call: dx (returned, or None), dW accumulated into `dw`, dbias (+)= column sums of dout (taken from
    `dout_colsum` when the caller already has them).  Any part may be None."""
    dx = torch.empty((x.shape[0], cin), dtype=x.dtype, device=x.device) if need_dx else None
    ws = stats_scratch(x.device, cout) if dbias is not None else None
    L.check(L.lib().scn_conv_module_backward_colsum(
        x.data_ptr(), _DT[x.dtype], x.shape[0], dout.data_ptr(), _DT[dout.dtype], n_out_rows,
        nbr_fwd.data_ptr(), nbr_fwd.shape[1], nbr_bwd.data_ptr(), nbr_bwd.shape[1], K, cin, cout, weight.data_ptr(),
        int(mirror), prec, None if wimg_t is None else wimg_t.data_ptr(), int(skip_prep),
        None if dx is None else dx.data_ptr(), None if dw is None else dw.data_ptr(), int(zero_dw),
        None if dbias is None else dbias.data_ptr(), int(accumulate_dbias),
        None if dout_colsum is None else dout_colsum.data_ptr(), None if ws is None else ws.data_ptr(),
        L.stream()), "scn_conv_module_backward_colsum")
    return dx


def col_sum(x) -> torch.Tensor:
    n, c = x.shape
    ws = torch.empty((2 * c,), dtype=torch.float64, device=x.device)
    out = torch.empty((c,), dtype=torch.float32, device=x.device)
    L.check(L.lib().scn_col_sum_acc(L.ptr(x), L.dtype_code(x), n, c, L.ptr(ws), L.ptr(out), 0, L.stream()),
            "scn_col_sum_acc")
    return out


# ---------------------------------------------------------------------------- bandwidth layers


def bn_forward(x, gamma, beta, rm, rv, training, eps, momentum, leak):
    """-> (out, stats) with stats fp32 [2, C] = (mean, invstd) used by the backward."""
    n, c = x.shape
    dev = x.device
    stats = torch.empty((2, c), dtype=torch.float32, device=dev)
    ws = stats_scratch(dev, c)
    out = torch.empty_like(x)
    p = _profiler
    e0 = p.begin() if p else None
    sp = stats.data_ptr()
    L.check(L.lib().scn_bn_forward(x.data_ptr(), _DT[x.dtype], n, c, L.ptr(gamma), L.ptr(beta), rm.data_ptr(),
                                   rv.data_ptr(), int(training), eps, momentum, leak, sp, sp + 4 * c, ws.data_ptr(),
                                   out.data_ptr(), L.stream()), "scn_bn_forward")
    if p:   # stats pass reads x, apply pass reads x and writes out
        p.end(e0, kind="bn_fwd", bytes=3.0 * x.numel() * x.element_size())
    return out, stats


def bn_backward(x, dout, gamma, beta, stats, training, leak, dgamma=None, dbeta=None, want_colsum=False):
    """-> (dx, dgamma, dbeta) or, with want_colsum, (dx, dgamma, dbeta, column sums of dx [C] fp32).  When dgamma/dbeta
    buffers are given the parameter gradients are ACCUMULATED into them."""
    n, c = x.shape
    dev = x.device
    ws = stats_scratch(dev, c)
    dx = torch.empty_like(x)
    accumulate = dgamma is not None
    if not accumulate:
        both = torch.empty((2, c), dtype=torch.float32, device=dev)
        dgamma, dbeta = both[0], both[1]
    colsum = torch.empty((c,), dtype=torch.float32, device=dev) if want_colsum else None
    p = _profiler
    e0 = p.begin() if p else None
    sp = stats.data_ptr()
    L.check(L.lib().scn_bn_backward_colsum(x.data_ptr(), dout.data_ptr(), _DT[x.dtype], n, c, L.ptr(gamma), L.ptr(beta),
                                           sp, sp + 4 * c, int(training), leak, ws.data_ptr(), dx.data_ptr(),
                                           dgamma.data_ptr(), dbeta.data_ptr(), int(accumulate), L.ptr(colsum), L.stream()),
            "scn_bn_backward_colsum")
    if p:   # reduce pass reads x,dout; apply pass reads x,dout and writes dx
        p.end(e0, kind="bn_bwd", bytes=5.0 * x.numel() * x.element_size())
    if want_colsum:
        return dx, dgamma, dbeta, colsum
    return dx, dgamma, dbeta


def leaky_forward(x, leak):
    out = torch.empty_like(x)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_leaky_forward(L.ptr(x), L.dtype_code(x), x.numel(), leak, L.ptr(out), L.stream()),
            "scn_leaky_forward")
    if p:
        p.end(e0, kind="leaky_fwd", bytes=2.0 * x.numel() * x.element_size())
    return out


def leaky_backward(x, dout, leak):
    dx = torch.empty_like(x)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_leaky_backward(L.ptr(x), L.ptr(dout), L.dtype_code(x), x.numel(), leak, L.ptr(dx),
                                       L.stream()), "scn_leaky_backward")
    if p:
        p.end(e0, kind="leaky_bwd", bytes=3.0 * x.numel() * x.element_size())
    return dx


def add_forward(a, b, leak=1.0):
    out = torch.empty_like(a)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_add_forward(L.ptr(a), L.ptr(b), L.dtype_code(a), a.numel(), leak, L.ptr(out), L.stream()),
            "scn_add_forward")
    if p:
        p.end(e0, kind="add", bytes=3.0 * a.numel() * a.element_size())
    return out


def convert(x, dtype):
    if x.dtype == dtype:
        return x
    out = torch.empty(x.shape, dtype=dtype, device=x.device)
    if x.numel():
        L.check(L.lib().scn_rows_gather(L.ptr(x), L.dtype_code(x), None, x.numel(), 1, L.ptr(out), L.dtype_code(out),
                                        L.stream()), "scn_rows_gather(convert)")
    return out


def input_layer_forward(feats, rows, n_active, mode):
    n_in, c = feats.shape
    dev = feats.device
    out = torch.empty((n_active, c), dtype=torch.float32, device=dev)
    cnt = torch.empty((n_active,), dtype=torch.float32, device=dev) if mode == 4 else None
    L.check(L.lib().scn_input_layer_forward(L.ptr(feats), L.ptr(rows), n_in, n_active, c, mode, L.ptr(out), L.SCN_F32,
                                            L.ptr(cnt), L.stream()), "scn_input_layer_forward")
    return out


def rows_gather(src, rows, out_dtype):
    n = rows.shape[0]
    c = src.shape[1]
    out = torch.empty((n, c), dtype=out_dtype, device=src.device)
    L.check(L.lib().scn_rows_gather(L.ptr(src), L.dtype_code(src), L.ptr(rows), n, c, L.ptr(out), L.dtype_code(out),
                                    L.stream()), "scn_rows_gather")
    return out


def rows_scatter_add(src, rows, n_out):
    c = src.shape[1]
    out = torch.zeros((n_out, c), dtype=torch.float32, device=src.device)
    L.check(L.lib().scn_rows_scatter_add(L.ptr(src), L.dtype_code(src), L.ptr(rows), rows.shape[0], c, L.ptr(out),
                                         L.stream()), "scn_rows_scatter_add")
    return out


def pool_rows(x, nbr, n_rows, scale, col0=0, ncol=None):
    """out[r] = scale * sum_k x[nbr[k][r], col0:col0+ncol] over existing table entries (AveragePooling fwd / bwd)."""
    L.require_cuda(x, "AveragePooling")
    assert x.dim() == 2 and x.stride(1) == 1 and nbr.dtype == torch.int32
    K, n_pad = nbr.shape
    c = x.shape[1] - col0 if ncol is None else ncol
    out = torch.empty((n_rows, c), dtype=x.dtype, device=x.device)
    src = x[:, col0:] if col0 else x
    L.check(L.lib().scn_pool_rows(src.data_ptr(), L.dtype_code(x), x.stride(0), L.ptr(nbr), K, n_rows, n_pad, c,
                                  float(scale), L.ptr(out), L.stream()), "scn_pool_rows")
    return out


def sparse_to_dense_forward(x, keys, batch, spatial):
    n, c = x.shape
    dense = torch.empty((batch, c) + tuple(spatial), dtype=torch.float32, device=x.device)
    p = _profiler
    e0 = p.begin() if p else None
    L.check(L.lib().scn_sparse_to_dense_forward(L.ptr(x), L.dtype_code(x), L.ptr(keys), n, c, batch, spatial[0],
                                                spatial[1], spatial[2], L.ptr(dense), L.stream()),
            "scn_sparse_to_dense_forward")
    if p:
        p.end(e0, kind="sparse_to_dense_fwd", bytes=4.0 * dense.numel() + x.numel() * x.element_size())
    return dense


def sparse_to_dense_backward(ddense, keys, n, c, batch, spatial, dtype):
    dx = torch.empty((n, c), dtype=dtype, device=ddense.device)
    L.check(L.lib().scn_sparse_to_dense_backward(L.ptr(ddense), L.ptr(keys), n, c, batch, spatial[0], spatial[1],
                                                 spatial[2], L.ptr(dx), L.dtype_code(dx), L.stream()),
            "scn_sparse_to_dense_backward")
    return dx
