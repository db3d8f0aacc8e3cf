"""autograd.Function wrappers: the host-side mirror of SCN's ``X_updateOutput`` / ``X_backward``
pairs (SURVEY.md §8b).  Forward and backward both run on the C ABI; nothing is computed by torch.
The hot modules use the C++ functions of csrc_torch/scn_torch.cpp instead, except under ops.Profiler and for
parameters that are not contiguous fp32 (modules._native).
"""
from __future__ import annotations

import torch
from torch.autograd import Function

from . import config, ops


def _w3(weight):
    """SCN stores [K, groups=1, Cin, Cout] (newer) or [K, Cin, Cout] (2018-19); kernels take 3-D."""
    return weight.detach().reshape(weight.shape[0], weight.shape[-2], weight.shape[-1]).contiguous().float()


def _direct_grad(param):
    """The gradient buffer to accumulate into in place, when the owner of the parameter asked for it
    (trainer.FlatGradArena marks parameters with ``_scn_direct_grad``): saves the separate dW tensor, its zero fill and
    autograd's AccumulateGrad add for every parameter of the sparse network."""
    if param is None or not getattr(param, "_scn_direct_grad", False):
        return None
    g = param.grad
    if g is None or g.dtype != torch.float32 or not g.is_contiguous() or g.device != param.device:
        return None
    return g


def _grad_ready(param):
    cb = getattr(param, "_scn_grad_ready", None)
    if cb is not None:
        cb(param)


class ConvWorkspace:
    """Per-module device workspaces of the convolution kernels: the buffers of the re-laid weight images (forward and
    dgrad) and the kernel family chosen for this shape.  The images are rebuilt on every call (modules._ConvBase._conv)
    unless a trainer has prepared all of them for the current step in one launch (prepare_weight_images below)."""

    __slots__ = ("fwd", "bwd", "fwd_key", "bwd_key", "path", "prepared", "shape")

    def __init__(self, K, cin, cout, prec, dtype, device):
        self.fwd = torch.zeros((ops.conv_prep_bytes(K, cin, cout, prec, dtype),), dtype=torch.uint8, device=device)
        self.bwd = None
        self.fwd_key = self.bwd_key = None
        self.path = ops.conv_path(K, cin, cout, prec, dtype)
        self.prepared = -1          # value of the global epoch for which both images are current
        self.shape = (K, cin, cout, prec, dtype, device)

    def bwd_buffer(self, K, cin, cout, prec, dtype, device):
        if self.bwd is None:
            self.bwd = torch.zeros((ops.conv_prep_bytes(K, cout, cin, prec, dtype),), dtype=torch.uint8, device=device)
        return self.bwd


# ---- all weight images of a model in one launch ------------------------------------------------------------------
# A training step re-lays 56 forward and 56 dgrad weight images; per module that is 112 launches of a ~3 us kernel.
# A trainer that knows when the parameters change (after optimizer.step()) has them all built at once:
#     token = prepare_weight_images(modules)   # at the start of a step
#     ... forward / backward (the modules pass skip_prep) ...
#     release_weight_images()                  # before the optimizer updates the parameters
_epoch = [0]
_active = [False]


def weight_images_current(ws) -> bool:
    return _active[0] and ws.prepared == _epoch[0]


def release_weight_images() -> None:
    _active[0] = False


class _ImagePlan:
    __slots__ = ("descs", "n", "total", "workspaces", "key")


_plans = {}


def prepare_weight_images(modules) -> int:
    """modules: the convolution modules of a model (objects with .weight, .mirror_dgrad and .workspace()).  Builds the
    forward and dgrad images of every module on the tcgen05 path in ONE launch; the other paths keep their per-call
    re-layout.  Returns the number of images built."""
    from .. import _lib as L
    mods = [m for m in modules if m.weight.is_cuda and m.weight.dtype == torch.float32 and m.weight.is_contiguous()]
    if not mods:
        return 0
    prec, fdt = config.precision_code(), config.feature_dtype()
    key = (id(mods[0]), len(mods), prec, fdt) + tuple(m.weight.data_ptr() for m in mods)
    plan = _plans.get(key)
    if plan is None:
        rows, wss, first = [], [], 0
        for m in mods:
            w = m.weight
            K, cin, cout = w.shape[0], w.shape[-2], w.shape[-1]
            ws = m.workspace(K, cin, cout, prec, fdt, w.device)
            if ws.path != 2 or ops.conv_path(K, cout, cin, prec, fdt) != 2:
                continue
            bwd = ws.bwd_buffer(K, cin, cout, prec, fdt, w.device)
            rows.append([w.data_ptr(), ws.fwd.data_ptr(), K, cin, cout, 0, first, prec])
            first += K * cin * cout
            rows.append([w.data_ptr(), bwd.data_ptr(), K, cin, cout, 1 | (2 if m.mirror_dgrad else 0), first, prec])
            first += K * cin * cout
            wss.append(ws)
        plan = _ImagePlan()
        plan.n, plan.total, plan.workspaces = len(rows), first, wss
        plan.descs = torch.tensor(rows, dtype=torch.int64, device=mods[0].weight.device) if rows else None
        _plans.clear()              # one model at a time
        _plans[key] = plan
    _epoch[0] += 1
    if plan.n:
        L.check(L.lib().scn_conv_prep_weights_batched(plan.descs.data_ptr(), plan.n, plan.total, L.stream()),
                "scn_conv_prep_weights_batched")
        for ws in plan.workspaces:
            ws.prepared = _epoch[0]
    _active[0] = True
    return plan.n


class ConvFn(Function):
    """out[o] = bias + sum_k x[nbr_fwd[k][o]] @ W[k], with weight re-layout, contraction, dgrad, wgrad and bias gradient
    each a C-ABI call of its own (so that ops.Profiler times each kernel).

    mirror=True  (submanifold): dgrad uses the same table with B_k = W[K-1-k]^T.
    mirror=False (strided / deconvolution): dgrad uses nbr_bwd (the transposed table) with W[k]^T.
    """

    @staticmethod
    def forward(ctx, x, weight, bias, nbr_fwd, nbr_bwd, n_out_rows, mirror):
        x = x.contiguous()
        prec = config.precision_code()
        fdt = config.feature_dtype()
        cin, cout = weight.shape[-2], weight.shape[-1]
        bprep = ops.prep_weights(_w3(weight), False, False, prec, fdt)
        b = bias.detach().float().contiguous() if bias is not None else None
        out = ops.conv_forward(x, nbr_fwd, n_out_rows, cin, cout, bprep, b, prec, fdt)
        ctx.save_for_backward(x, weight, bias)
        ctx.nbr_fwd, ctx.nbr_bwd, ctx.mirror, ctx.prec = nbr_fwd, nbr_bwd, mirror, prec
        ctx.n_out_rows = n_out_rows
        return out

    @staticmethod
    def backward(ctx, dout):
        x, weight, bias = ctx.saved_tensors
        dout = dout.contiguous()
        cin, cout = weight.shape[-2], weight.shape[-1]
        dx = dw = db = None
        w3 = _w3(weight)
        if ctx.needs_input_grad[0]:
            bt = ops.prep_weights(w3, True, ctx.mirror, ctx.prec, x.dtype)
            dx = ops.conv_forward(dout, ctx.nbr_bwd, x.shape[0], cout, cin, bt, None, ctx.prec, x.dtype,
                                  kind="conv_dgrad")
        if ctx.needs_input_grad[1]:
            dw = ops.conv_wgrad(x, dout, ctx.nbr_fwd, ctx.n_out_rows, cin, cout, ctx.prec).view_as(weight)
            dw = dw.to(weight.dtype)
        if bias is not None and ctx.needs_input_grad[2]:
            db = ops.col_sum(dout)
        return dx, dw, db, None, None, None, None


class BatchNormFn(Function):
    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, training, eps, momentum, leak):
        x = x.contiguous()
        lean = weight is None or (weight.dtype == torch.float32 and weight.is_contiguous()
                                  and bias.dtype == torch.float32 and bias.is_contiguous())
        g = weight if lean else weight.detach().float().contiguous()
        b = bias if lean else bias.detach().float().contiguous()
        out, stats = ops.bn_forward(x, g, b, running_mean, running_var, training, eps, momentum, leak)
        ctx.save_for_backward(x, g, b, stats)
        ctx.params = (weight, bias) if lean and weight is not None else None
        ctx.training, ctx.leak, ctx.affine = training, leak, weight is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        x, g, b, stats = ctx.saved_tensors
        gw = gb = None
        if ctx.params is not None and ctx.needs_input_grad[1] and ctx.needs_input_grad[2]:
            gw, gb = _direct_grad(ctx.params[0]), _direct_grad(ctx.params[1])
            if gw is None or gb is None:
                gw = gb = None
        # column sums unused here, but the profiled pass must time the BatchNorm kernel a training step runs (scn_torch.cpp)
        colsum = ctx.training and x.shape[0] > 0
        dx, dg, db = ops.bn_backward(x, dout.contiguous(), g, b, stats, ctx.training, ctx.leak, gw, gb, colsum)[:3]
        if gw is not None:
            _grad_ready(ctx.params[0])
            _grad_ready(ctx.params[1])
            dg = db = None
        if not ctx.affine:
            dg = db = None
        return dx, dg, db, None, None, None, None, None, None


class LeakyReLUFn(Function):
    @staticmethod
    def forward(ctx, x, leak):
        x = x.contiguous()
        ctx.save_for_backward(x)
        ctx.leak = leak
        return ops.leaky_forward(x, leak)

    @staticmethod
    def backward(ctx, dout):
        (x,) = ctx.saved_tensors
        return ops.leaky_backward(x, dout.contiguous(), ctx.leak), None


class AddFn(Function):
    @staticmethod
    def forward(ctx, a, b):
        return ops.add_forward(a.contiguous(), b.contiguous())

    @staticmethod
    def backward(ctx, dout):
        return dout, dout


class AddLeakyFn(Function):
    """out = leaky(a + b): AddTable followed by LeakyReLU in one kernel (reference ResidualBlock tail,
    src/networks/sparse_building_blocks.py:96-98)."""

    @staticmethod
    def forward(ctx, a, b, leak):
        out = ops.add_forward(a.contiguous(), b.contiguous(), leak)
        ctx.save_for_backward(out)
        ctx.leak = leak
        return out

    @staticmethod
    def backward(ctx, dout):
        (out,) = ctx.saved_tensors
        # sign(out) == sign(a + b) for leak > 0; for leak == 0 (ReLU) out > 0 <=> a + b > 0 as well
        d = ops.leaky_backward(out, dout.contiguous(), ctx.leak)
        return d, d, None


class InputLayerFn(Function):
    @staticmethod
    def forward(ctx, feats, rows, n_active, mode):
        ctx.rows, ctx.mode, ctx.in_dtype = rows, mode, feats.dtype
        return ops.input_layer_forward(feats.detach().float().contiguous(), rows, n_active, mode)

    @staticmethod
    def backward(ctx, dout):
        if ctx.mode not in (0, 3):
            raise NotImplementedError("InputLayer backward is implemented for modes 0 and 3")
        return ops.rows_gather(dout.contiguous(), ctx.rows, ctx.in_dtype if ctx.in_dtype in (torch.float32, torch.bfloat16) else torch.float32), None, None, None


class OutputLayerFn(Function):
    @staticmethod
    def forward(ctx, feats, rows):
        ctx.rows, ctx.n, ctx.dtype = rows, feats.shape[0], feats.dtype
        return ops.rows_gather(feats.contiguous(), rows, feats.dtype)

    @staticmethod
    def backward(ctx, dout):
        acc = ops.rows_scatter_add(dout.contiguous(), ctx.rows, ctx.n)
        return ops.convert(acc, ctx.dtype), None


class AveragePoolingFn(Function):
    """features of scn.AveragePooling: out[q] = (1 / pool volume) * sum of the input rows of output site q."""

    @staticmethod
    def forward(ctx, x, down, up, n_out, volume, drop):
        if x.stride(-1) != 1:
            x = x.contiguous()
        ctx.up, ctx.n_in, ctx.c_in, ctx.drop, ctx.scale = up, x.shape[0], x.shape[1], drop, 1.0 / volume
        return ops.pool_rows(x, down, n_out, ctx.scale, col0=drop)

    @staticmethod
    def backward(ctx, dout):
        d = ops.pool_rows(dout.contiguous(), ctx.up, ctx.n_in, ctx.scale)
        if ctx.drop:                       # dropped leading features get no gradient
            d = torch.cat([d.new_zeros((ctx.n_in, ctx.drop)), d], 1)
        return d, None, None, None, None, None


class SparseToDenseFn(Function):
    @staticmethod
    def forward(ctx, x, keys, batch, spatial):
        x = x.contiguous()
        ctx.keys, ctx.batch, ctx.spatial = keys, batch, spatial
        ctx.n, ctx.c, ctx.dtype = x.shape[0], x.shape[1], x.dtype
        return ops.sparse_to_dense_forward(x, keys, batch, spatial)

    @staticmethod
    def backward(ctx, ddense):
        dx = ops.sparse_to_dense_backward(ddense.contiguous().float(), ctx.keys, ctx.n, ctx.c, ctx.batch, ctx.spatial,
                                          ctx.dtype)
        return dx, None, None, None
