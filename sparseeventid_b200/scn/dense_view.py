"""What ``scn.SparseToDense`` returns: a tensor that IS the dense ``[B, C, *spatial]`` fp32 tensor to every
consumer, but keeps the sparse rows it was built from (SURVEY.md §8f rank 1, "fused sparse head ... exposed
behind the same modules").

The reference follows ``scn.SparseToDense`` with ``torch.tanh`` (src/networks/resnet.py:156-159) and four
``torch.nn.AvgPool3d(full spatial extent)`` heads (src/networks/classification_head.py:19-28).  On the dense
tensor ([64,128,32,16,40] fp32 = 671 MB at batch 64) those cost ~16 ms per training step on a B200, nearly
all of it moving zeros.  Both commute with sparsity: ``tanh(0) == 0`` and the mean over the full extent is
``sum over active rows / V``.  ``SparseDenseTensor`` intercepts exactly those calls through
``__torch_function__`` and evaluates them on the ``[N, C]`` rows; ANY other use (indexing, arithmetic, printing,
a pooling window that is not the full extent, ...) first materialises the real dense tensor with the
SparseToDense kernel, so semantics never change.  ``scn.set_lazy_dense(False)`` turns the mechanism off.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F_torch
from torch.autograd import Function

from . import ops

_state = {"lazy": True}


def set_lazy_dense(flag: bool) -> None:
    _state["lazy"] = bool(flag)


def lazy_dense_enabled() -> bool:
    return _state["lazy"]


class _PooledMeanFn(Function):
    """[N, C] rows -> [B, C] mean over the FULL dense extent (zeros included): sum over the sample's rows / V."""

    @staticmethod
    def forward(ctx, feats, batch_of_row, batch, volume):
        ctx.batch_of_row, ctx.volume, ctx.dtype = batch_of_row, volume, feats.dtype
        acc = ops.rows_scatter_add(feats.contiguous(), batch_of_row, batch)
        return acc / float(volume)

    @staticmethod
    def backward(ctx, dout):
        g = (dout.float() / float(ctx.volume)).contiguous()
        return ops.rows_gather(g, ctx.batch_of_row, ctx.dtype), None, None, None


# elementwise maps with f(0) == 0 that may be applied to the rows instead of the dense tensor
_ZERO_PRESERVING = {torch.tanh, torch.Tensor.tanh, torch.relu, torch.Tensor.relu, F_torch.relu, F_torch.leaky_relu,
                    F_torch.tanh}
_PROPERTIES = {"shape", "dtype", "device", "ndim", "requires_grad", "is_cuda", "layout", "is_sparse", "grad_fn",
               "is_leaf", "names", "is_quantized", "is_meta", "grad"}
_METHODS = {"size", "dim", "numel", "nelement", "ndimension", "is_floating_point", "element_size", "get_device"}
_POOLS = {F_torch.avg_pool3d: 3, F_torch.avg_pool2d: 2, F_torch.avg_pool1d: 1}


def _pooled_mean_cuda(feats, batch_of_row, batch, volume):
    return _PooledMeanFn.apply(feats, batch_of_row, batch, volume)


class SparseDenseTensor(torch.Tensor):
    @staticmethod
    def __new__(cls, feats, keys, batch, spatial, materialize, pooled_mean=_pooled_mean_cuda):
        c = feats.shape[1]
        r = torch.Tensor._make_wrapper_subclass(cls, (batch, c) + tuple(spatial), dtype=torch.float32,
                                                device=feats.device, requires_grad=feats.requires_grad)
        r._feats = feats            # [N, C] rows (autograd-tracked), any feature dtype
        r._keys = keys              # int64 [N] packed (batch|x0|x1|x2)
        r._batch = batch
        r._spatial = tuple(spatial)
        r._materialize = materialize    # feats -> dense [B, C, *spatial] fp32 (the SparseToDense kernel)
        r._pooled_mean = pooled_mean
        r._dense = None
        r._batch_of_row = None
        r._pooled_cache = None
        return r

    # -- helpers -------------------------------------------------------------------------------
    def dense(self) -> torch.Tensor:
        """The real dense tensor (built once, on first need)."""
        if self._dense is None:
            self._dense = self._materialize(self._feats)
        return self._dense

    def _rows_f32(self):
        f = self._feats
        return f if f.dtype == torch.float32 else f.float()

    def _like(self, feats):
        return SparseDenseTensor(feats, self._keys, self._batch, self._spatial, self._materialize, self._pooled_mean)

    def _batch_index(self):
        if self._batch_of_row is None:
            # keys are int64 and the shift is arithmetic: mask so that batch indices >= 32768 stay non-negative
            self._batch_of_row = ((self._keys >> 48) & 0xFFFF).to(torch.int32).contiguous()
        return self._batch_of_row

    def _full_extent(self, nd, kernel_size, stride, padding, ceil_mode, count_include_pad, divisor_override):
        if nd != len(self._spatial):
            return False
        tup = lambda v: (v,) * nd if isinstance(v, int) else tuple(v)
        if tup(kernel_size) != self._spatial:
            return False
        if stride is not None and stride != [] and stride != () and tup(stride) != self._spatial:
            return False
        return all(p == 0 for p in tup(padding)) and not ceil_mode and count_include_pad and divisor_override is None

    # -- interception --------------------------------------------------------------------------
    @classmethod
    def __torch_function__(cls, func, types, args=(), kwargs=None):
        kwargs = kwargs or {}
        name = getattr(func, "__name__", "")
        owner = getattr(getattr(func, "__self__", None), "__name__", "")
        if (name == "__get__" and owner in _PROPERTIES) or name in _METHODS:
            with torch._C.DisableTorchFunctionSubclass():
                return func(*args, **kwargs)
        self = args[0] if args and isinstance(args[0], SparseDenseTensor) else None
        if self is not None:
            if func in _ZERO_PRESERVING and not kwargs.get("inplace", False):
                with torch._C.DisableTorchFunctionSubclass():
                    return self._like(func(self._rows_f32(), *args[1:], **kwargs))
            if func in _POOLS:
                names = ["kernel_size", "stride", "padding", "ceil_mode", "count_include_pad", "divisor_override"]
                cfg = {"stride": None, "padding": 0, "ceil_mode": False, "count_include_pad": True,
                       "divisor_override": None}
                cfg.update(dict(zip(names, args[1:])))
                cfg.update(kwargs)
                if "kernel_size" in cfg and self._full_extent(_POOLS[func], **cfg):
                    vol = 1
                    for v in self._spatial:
                        vol *= v
                    # the reference applies one full-extent pool per head (classification_head.py:19-28: four heads on the
                    # same tensor): the pooled mean is computed once and shared (autograd sums the heads' gradients)
                    pooled = self._pooled_cache
                    if pooled is None:
                        pooled = self._pooled_cache = self._pooled_mean(self._rows_f32(), self._batch_index(), self._batch, vol)
                    return pooled.view((self._batch, pooled.shape[1]) + (1,) * len(self._spatial))

        # anything else: behave exactly like the dense tensor
        def unwrap(a):
            if isinstance(a, SparseDenseTensor):
                return a.dense()
            if isinstance(a, (list, tuple)):
                return type(a)(unwrap(x) for x in a)
            return a
        with torch._C.DisableTorchFunctionSubclass():
            return func(*[unwrap(a) for a in args], **{k: unwrap(v) for k, v in kwargs.items()})

    @classmethod
    def __torch_dispatch__(cls, func, types, args=(), kwargs=None):
        # safety net for anything that reaches the dispatcher without passing __torch_function__
        def unwrap(a):
            if isinstance(a, SparseDenseTensor):
                return a.dense()
            if isinstance(a, (list, tuple)):
                return type(a)(unwrap(x) for x in a)
            return a
        return func(*[unwrap(a) for a in args], **{k: unwrap(v) for k, v in (kwargs or {}).items()})

    def __repr__(self):
        return f"SparseDenseTensor(shape={tuple(self.shape)}, rows={self._feats.shape[0]})"
