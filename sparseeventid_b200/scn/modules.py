"""nn.Module surface of ``sparseconvnet`` used by the reference (SURVEY.md §2.3), B200-backed.

Constructor forms, parameter/buffer names, shapes and initialisation follow SCN (SURVEY.md
App. A) so the reference's ``src/networks/*.py`` run unchanged and checkpoints round-trip.
Every forward runs hand-written sm_100a kernels through libscn_b200.so; there is no CPU path.
"""
from __future__ import annotations

import math

import torch
from torch import nn

from .. import _lib as L
from . import _ext, config, core, dense_view, ops
from . import functional as F
from .core import Metadata, Pending, SparseConvNetTensor, as_tuple


def _volume(t):
    v = 1
    for x in t:
        v *= x
    return v


def _mark(*params):
    """Tags parameters whose gradients the kernels can accumulate in place (see trainer.FlatGradArena)."""
    for p in params:
        if p is not None:
            p._scn_param = True


def _native(x, *params):
    """The C++ autograd functions (csrc_torch/scn_torch.cpp) that run a module forward / backward in one native call,
    or None where functional.py's per-kernel functions run instead: under ops.Profiler, which times every kernel on its
    own, and for parameters that are not contiguous fp32."""
    ext = _ext.get()
    L.require_cuda(x, "sparse module")
    if ops.profiling():
        return None
    for p in params:
        if p is not None and (p.dtype != torch.float32 or not p.is_contiguous()):
            return None
    return ext


def _new_like(input, features, spatial_size=None):
    if spatial_size is None:
        return SparseConvNetTensor(features, input.metadata, input.spatial_size, None, input._spc)
    return SparseConvNetTensor(features, input.metadata, spatial_size)


class InputLayer(nn.Module):
    """scn.InputLayer(dimension, spatial_size, mode=3)  -- reference src/networks/resnet.py:26-29,40-43.

    forward((coords, features[, batch_size])): coords [N, dimension(+1)] of any dtype, batch index
    in the LAST column (src/io/data_transforms.py:43-46,242); features [N, C].
    mode 0: no duplicates promised, 3: sum duplicates (default), 4: mean.  (1/2 = last/first wins
    are not implemented on the GPU; the reference never selects them.)
    """

    def __init__(self, dimension, spatial_size, mode=3):
        super().__init__()
        self.dimension = dimension
        self.spatial_size = torch.LongTensor(list(as_tuple(spatial_size, dimension)))
        self.mode = mode

    def forward(self, input):
        coords, feats = input[0], input[1]
        batch_size = int(input[2]) if len(input) > 2 and input[2] is not None else 0
        coords = torch.as_tensor(coords)
        feats = torch.as_tensor(feats)
        L.require_cuda(feats, "InputLayer(features)")
        if not coords.is_cuda:
            coords = coords.to(feats.device, non_blocking=True)
        if coords.dim() != 2 or coords.shape[1] not in (self.dimension, self.dimension + 1):
            raise ValueError(f"coords must be [N, {self.dimension}] or [N, {self.dimension + 1}]")
        sp = tuple(int(v) for v in self.spatial_size)
        md = core.take_prefetched(coords, self.dimension, sp)        # built ahead by scn.prefetch() for this very tensor?
        if md is None:
            md = Metadata(self.dimension, feats.device)
            lvl = md.build_input(coords, sp)
        else:
            lvl = md.levels[sp]
        rows = md.row_of_input
        keys_out = lvl.keys
        self._last_plan = md.plan                                    # filled as the network asks for rulebooks
        # SCN: batch size = max(argument, largest batch index + 1); the index came back with the row count (no extra sync)
        md.batch_size = max(batch_size, md.max_batch_index + 1)
        out = SparseConvNetTensor(None, md, self.spatial_size)
        out.features = F.InputLayerFn.apply(feats, rows, lvl.n, self.mode)
        return out

    def __repr__(self):
        return f"InputLayer(dimension={self.dimension}, spatial_size={self.spatial_size.tolist()}, mode={self.mode})"


class OutputLayer(nn.Module):
    """scn.OutputLayer(dimension): features back in the original input-row order (App. A.7)."""

    def __init__(self, dimension):
        super().__init__()
        self.dimension = dimension

    def forward(self, input):
        return F.OutputLayerFn.apply(input.features, input.metadata.row_of_input)


class _ConvBase(nn.Module):
    mirror_dgrad = False         # dgrad weights: W[K-1-k]^T (submanifold) or W[k]^T (strided / deconvolution)

    def _init_params(self, nIn, nOut, bias):
        k = self.filter_volume
        w = torch.empty(k, 1, nIn, nOut)
        w.normal_(0, math.sqrt(2.0 / (nIn * k)))
        self.weight = nn.Parameter(w)
        self.bias = nn.Parameter(torch.zeros(nOut)) if bias else None
        _mark(self.weight, self.bias)

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        # accept SCN 2018-19 checkpoints whose conv weights are [K, Cin, Cout]
        key = prefix + "weight"
        if key in state_dict and state_dict[key].dim() == 3:
            w = state_dict[key]
            state_dict[key] = w.reshape(w.shape[0], 1, w.shape[1], w.shape[2])
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    def workspace(self, K, cin, cout, prec, dtype, device):
        """Device workspaces of this module's kernels (weight images), created on first use; not part of state_dict."""
        table = self.__dict__.setdefault("_scn_ws", {})
        key = (prec, dtype, device)
        ws = table.get(key)
        if ws is None:
            ws = table[key] = F.ConvWorkspace(K, cin, cout, prec, dtype, device)
        return ws

    def _conv(self, x, nbr_fwd, nbr_bwd, n_out_rows, mirror):
        """out = bias + conv(x)."""
        w, b = self.weight, self.bias
        ext = _native(x, w, b)
        if ext is not None:
            prec, fdt = config.precision_code(), config.feature_dtype()
            K, cin, cout = w.shape[0], w.shape[-2], w.shape[-1]
            ws = self.workspace(K, cin, cout, prec, fdt, x.device)
            if ws.path > 0 and x.dtype != fdt:
                x = ops.convert(x, fdt)
            # The weight image is rebuilt on every call: there is no reliable "weights changed" signal (fused
            # optimizers update parameters without bumping Tensor._version), and the re-layout is a ~4 us kernel --
            # unless a trainer has just built every image of the model in one launch (F.prepare_weight_images).
            skip = F.weight_images_current(ws)
            wimg_t = None
            if x.requires_grad and torch.is_grad_enabled():
                wimg_t = ws.bwd_buffer(K, cin, cout, prec, x.dtype, x.device)
            return ext.conv(x, w, b, nbr_fwd, nbr_bwd, n_out_rows, mirror, prec, L.SCN_BF16 if fdt == torch.bfloat16
                            else L.SCN_F32, ws.fwd, wimg_t, skip, getattr(w, "_scn_direct_grad", False),
                            b is not None and getattr(b, "_scn_direct_grad", False))
        return F.ConvFn.apply(x, w, b, nbr_fwd, nbr_bwd, n_out_rows, mirror)

    def _check(self, input):
        assert input.features.nelement() == 0 or input.features.size(1) == self.nIn, \
            f"expected {self.nIn} input planes, got {input.features.size(1)}"


class SubmanifoldConvolution(_ConvBase):
    """scn.SubmanifoldConvolution(dimension, nIn, nOut, filter_size, bias, groups=1)
    -- reference src/networks/sparse_building_blocks.py:29-34, src/networks/resnet.py:30-36,44-50,105-110."""
    mirror_dgrad = True

    def __init__(self, dimension, nIn, nOut, filter_size, bias, groups=1):
        super().__init__()
        assert groups == 1, "groups > 1 is not used by the reference"
        self.dimension, self.nIn, self.nOut = dimension, nIn, nOut
        self.filter_size = as_tuple(filter_size, dimension)
        assert all(f % 2 == 1 for f in self.filter_size), "submanifold filters must be odd"
        self.filter_volume = _volume(self.filter_size)
        self._init_params(nIn, nOut, bias)

    def forward(self, input):
        self._check(input)
        md = input.metadata
        nbr = md.subm_table(input._sp(), self.filter_size)
        n = md.levels[input._sp()].n
        feats = self._conv(input.features, nbr, nbr, n, True)
        return _new_like(input, feats)

    def __repr__(self):
        return f"SubmanifoldConvolution {self.nIn}->{self.nOut} C{list(self.filter_size)}"


class Convolution(_ConvBase):
    """scn.Convolution(dimension, nIn, nOut, filter_size, filter_stride, bias)
    -- reference src/networks/sparse_building_blocks.py:110-117."""

    def __init__(self, dimension, nIn, nOut, filter_size, filter_stride, bias, groups=1):
        super().__init__()
        assert groups == 1
        self.dimension, self.nIn, self.nOut = dimension, nIn, nOut
        self.filter_size = as_tuple(filter_size, dimension)
        self.filter_stride = as_tuple(filter_stride, dimension)
        self.filter_volume = _volume(self.filter_size)
        self._init_params(nIn, nOut, bias)

    def forward(self, input):
        self._check(input)
        md = input.metadata
        rule = md.strided_rule(input._sp(), self.filter_size, self.filter_stride)
        feats = self._conv(input.features, rule.down, rule.up, rule.n_out, False)
        return _new_like(input, feats, torch.LongTensor(list(rule.out_spatial)))

    def __repr__(self):
        return f"Convolution {self.nIn}->{self.nOut} C{list(self.filter_size)}/{list(self.filter_stride)}"


class Deconvolution(_ConvBase):
    """scn.Deconvolution(dimension, nIn, nOut, filter_size, filter_stride, bias)
    -- reference src/networks/sparse_building_blocks.py:207-213.  The fine grid must already exist
    in the metadata (App. A.7)."""

    def __init__(self, dimension, nIn, nOut, filter_size, filter_stride, bias, groups=1):
        super().__init__()
        assert groups == 1
        self.dimension, self.nIn, self.nOut = dimension, nIn, nOut
        self.filter_size = as_tuple(filter_size, dimension)
        self.filter_stride = as_tuple(filter_stride, dimension)
        self.filter_volume = _volume(self.filter_size)
        self._init_params(nIn, nOut, bias)

    def forward(self, input):
        self._check(input)
        md = input.metadata
        sp = input._sp()
        fine = tuple((sp[a] - 1) * self.filter_stride[a] + self.filter_size[a] for a in range(self.dimension))
        if fine not in md.levels:
            raise RuntimeError("Deconvolution needs the fine grid to exist in the metadata")
        rule = md.strided_rule(fine, self.filter_size, self.filter_stride)
        feats = self._conv(input.features, rule.up, rule.down, rule.n_in, False)
        return _new_like(input, feats, torch.LongTensor(list(fine)))


class AveragePooling(nn.Module):
    """scn.AveragePooling(dimension, pool_size, pool_stride, nFeaturesToDrop=0) -- the ``Pooling`` down-sampling branch,
    reference src/networks/sparse_building_blocks.py:150-154 (non-default ``encoder.downsampling``).  Output sites and
    rows are those of a Convolution with the same size/stride; features are the SUM of the window's active inputs
    divided by the pool volume (SparseConvNet's convention: inactive sites count as zeros), the first nFeaturesToDrop
    channels left out.  No parameters."""

    def __init__(self, dimension, pool_size, pool_stride, nFeaturesToDrop=0):
        super().__init__()
        self.dimension = dimension
        self.pool_size = as_tuple(pool_size, dimension)
        self.pool_stride = as_tuple(pool_stride, dimension)
        self.pool_volume = _volume(self.pool_size)
        self.nFeaturesToDrop = int(nFeaturesToDrop)

    def forward(self, input):
        md = input.metadata
        feats = input.features
        assert feats.shape[1] > self.nFeaturesToDrop, "nFeaturesToDrop leaves no feature planes"
        rule = md.strided_rule(input._sp(), self.pool_size, self.pool_stride)
        out = F.AveragePoolingFn.apply(feats, rule.down, rule.up, rule.n_out, self.pool_volume, self.nFeaturesToDrop)
        return _new_like(input, out, torch.LongTensor(list(rule.out_spatial)))

    def __repr__(self):
        return f"AveragePooling {list(self.pool_size)}/{list(self.pool_stride)}"


class BatchNormalization(nn.Module):
    """scn.BatchNormalization(nPlanes, eps=1e-4, momentum=0.9, affine=True, leakiness=1)
    -- reference src/networks/sparse_building_blocks.py:39,122.  SCN conventions (App. A.5)."""

    def __init__(self, nPlanes, eps=1e-4, momentum=0.9, affine=True, leakiness=1):
        super().__init__()
        self.nPlanes, self.eps, self.momentum, self.affine, self.leakiness = nPlanes, eps, momentum, affine, leakiness
        self.register_buffer("running_mean", torch.zeros(nPlanes))
        self.register_buffer("running_var", torch.ones(nPlanes))
        if affine:
            self.weight = nn.Parameter(torch.ones(nPlanes))
            self.bias = nn.Parameter(torch.zeros(nPlanes))
            _mark(self.weight, self.bias)
        else:
            self.register_parameter("weight", None)
            self.register_parameter("bias", None)

    def forward(self, input):
        x = input.features
        assert x.nelement() == 0 or x.size(1) == self.nPlanes
        training = self.training

        def run(leak=float(self.leakiness), second=False):
            # second=True: the same layer evaluated again for another consumer of a tensor whose first evaluation was
            # fused into a following activation -- the running statistics were updated by the first one
            rm = self.running_mean.clone() if second and training else self.running_mean
            rv = self.running_var.clone() if second and training else self.running_var
            w, b = self.weight, self.bias
            ext = _native(x, w, b)
            if ext is not None:
                return ext.batch_norm(x, w, b, rm, rv, training, float(self.eps),
                                      float(self.momentum), leak,
                                      w is not None and getattr(w, "_scn_direct_grad", False)
                                      and getattr(b, "_scn_direct_grad", False))
            return F.BatchNormFn.apply(x, w, b, rm, rv, training, float(self.eps), float(self.momentum), leak)
        if float(self.leakiness) == 1.0:
            # defer by one module: a following LeakyReLU/ReLU becomes the fused leakiness of this same kernel
            return SparseConvNetTensor(None, input.metadata, input.spatial_size, Pending("bn", run, run, lambda: run(second=True)), input._spc)
        return _new_like(input, run())

    def __repr__(self):
        return (f"BatchNorm({self.nPlanes},eps={self.eps},momentum={self.momentum},affine={self.affine}"
                f",leakiness={self.leakiness})")


class BatchNormReLU(BatchNormalization):
    def __init__(self, nPlanes, eps=1e-4, momentum=0.9):
        super().__init__(nPlanes, eps, momentum, True, 0)


class BatchNormLeakyReLU(BatchNormalization):
    def __init__(self, nPlanes, eps=1e-4, momentum=0.9, leakiness=0.333):
        super().__init__(nPlanes, eps, momentum, True, leakiness)


class LeakyReLU(nn.Module):
    """scn.LeakyReLU(leak=1/3) -- reference sparse_building_blocks.py:20,45,80,128."""

    def __init__(self, leak=1.0 / 3.0):
        super().__init__()
        self.leak = leak

    def forward(self, input):
        pend = input.take_pending() if isinstance(input, SparseConvNetTensor) else None
        if pend is not None:
            return _new_like(input, pend.fuse(float(self.leak)))
        x = input.features
        ext = _native(x)
        if ext is not None:
            return _new_like(input, ext.leaky(x, float(self.leak)))
        return _new_like(input, F.LeakyReLUFn.apply(x, float(self.leak)))


class ReLU(LeakyReLU):
    def __init__(self):
        super().__init__(0.0)


class Tanh(nn.Module):
    def forward(self, input):
        return _new_like(input, torch.tanh(input.features))


class Sigmoid(nn.Module):
    def forward(self, input):
        return _new_like(input, torch.sigmoid(input.features))


class Identity(nn.Module):
    def forward(self, input):
        return input


class AddTable(nn.Module):
    """scn.AddTable(): features = sum of the list's features (rows aligned) -- sparse_building_blocks.py:82,96."""

    def forward(self, input):
        if len(input) == 2:
            a, b = input[0].features, input[1].features

            def run():
                return F.AddFn.apply(a, b)

            def fuse(leak):
                ext = _native(a)
                if ext is not None:
                    return ext.add_leaky(a, b, leak)
                return F.AddLeakyFn.apply(a, b, leak)
            return SparseConvNetTensor(None, input[0].metadata, input[0].spatial_size, Pending("add", run, fuse),
                                       input[0]._spc)
        feats = input[0].features
        for t in input[1:]:
            feats = F.AddFn.apply(feats, t.features)
        return _new_like(input[0], feats)


class SparseToDense(nn.Module):
    """scn.SparseToDense(dimension, nPlanes) -> dense [B, C, *spatial] fp32 -- src/networks/resnet.py:123-125."""

    def __init__(self, dimension, nPlanes):
        super().__init__()
        self.dimension, self.nPlanes = dimension, nPlanes

    def forward(self, input):
        md = input.metadata
        sp = input._sp()
        lvl = md.levels[sp]
        sp3 = tuple(sp) + (1,) * (3 - len(sp))
        batch, c = md.batch_size, input.features.shape[1]

        def materialize(feats):
            return F.SparseToDenseFn.apply(feats, lvl.keys, batch, sp3).view((batch, c) + tuple(sp))
        # the dense tensor to every consumer, but tanh / full-extent average pooling run on the rows
        return dense_view.SparseDenseTensor(input.features, lvl.keys, batch, tuple(sp), materialize)


class Sequential(nn.Sequential):
    """scn.Sequential: torch's container plus SparseConvNet's chaining `.add(module)`."""

    def add(self, module):
        self._modules[str(len(self._modules))] = module
        return self


class SparseGroupNorm(nn.Module):
    """scn.SparseGroupNorm(num_groups, num_channels, eps=1e-5, affine=True) -- named by the reference's non-default
    normalisation branches (src/networks/sparse_building_blocks.py:12,42,125,220: `encoder.normalization` = group /
    instance / InputNorm).  SparseConvNet itself has no such class (those branches raise AttributeError on the real
    package), so there is no upstream algorithm to restate; it is DEFINED here as torch.nn.GroupNorm restricted to the
    active sites: per sample and channel group, mean / biased variance over (active rows of the sample) x (channels of
    the group), then a per-channel affine.  Off the benchmarked path: segment sums with torch ops on the device (fp32),
    no dedicated kernel."""

    def __init__(self, num_groups, num_channels, eps=1e-5, affine=True):
        super().__init__()
        assert num_channels % num_groups == 0, "num_channels must be divisible by num_groups"
        self.num_groups, self.num_channels, self.eps, self.affine = num_groups, num_channels, eps, affine
        if affine:
            self.weight = nn.Parameter(torch.ones(num_channels))
            self.bias = nn.Parameter(torch.zeros(num_channels))
        else:
            self.register_parameter("weight", None)
            self.register_parameter("bias", None)

    def forward(self, input):
        x = input.features
        L.require_cuda(x, "SparseGroupNorm")
        md = input.metadata
        n, c = x.shape
        assert c == self.num_channels
        g, cg = self.num_groups, c // self.num_groups
        b = ((md.levels[input._sp()].keys >> 48) & 0xFFFF).long()             # sample of every active row (int64 keys)
        nb = max(int(md.batch_size), 1)
        xf = x.float().view(n, g, cg)
        cnt = torch.zeros(nb, device=x.device).index_add_(0, b, torch.ones(n, device=x.device)).clamp_min(1.0) * cg
        mean = torch.zeros(nb, g, device=x.device).index_add_(0, b, xf.sum(2)) / cnt[:, None]
        d = xf - mean[b][:, :, None]
        var = torch.zeros(nb, g, device=x.device).index_add_(0, b, (d * d).sum(2)) / cnt[:, None]
        y = (d * torch.rsqrt(var + self.eps)[b][:, :, None]).view(n, c)
        if self.affine:
            y = y * self.weight + self.bias
        return _new_like(input, y.to(x.dtype))

    def __repr__(self):
        return f"SparseGroupNorm({self.num_groups}, {self.num_channels}, eps={self.eps}, affine={self.affine})"
