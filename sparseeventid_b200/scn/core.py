"""SparseConvNetTensor + device-resident Metadata (SURVEY.md App. A.1, §8b "Ownership").

SCN keeps per-sample sparsehash grids and vectors of rule vectors on the host; here one
Metadata object owns, per spatial size, the packed site keys in row order plus one open-
addressing hash table, and caches one neighbour table per (spatial size, filter[, stride]).
It is shared by reference by every tensor derived from one InputLayer call.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Tuple

import torch

from . import ops


def as_tuple(v, dimension: int) -> Tuple[int, ...]:
    """SCN accepts int / list / tuple / tensor for sizes (reference src/networks/resnet.py:26-36)."""
    if isinstance(v, torch.Tensor):
        v = v.tolist()
    if hasattr(v, "tolist"):
        v = v.tolist()
    if isinstance(v, int):
        return tuple(v for _ in range(dimension))
    v = tuple(int(x) for x in v)
    if len(v) != dimension:
        raise ValueError(f"expected {dimension} values, got {v}")
    return v


def pad3(t: Tuple[int, ...], fill: int) -> Tuple[int, int, int]:
    return tuple(t) + (fill,) * (3 - len(t))


@dataclass
class Level:
    keys: torch.Tensor          # int64 [n]: packed (batch|x0|x1|x2) in row order
    n: int
    table_keys: torch.Tensor
    table_vals: torch.Tensor
    cap: int

    @property
    def n_pad(self):
        return ops.pad128(self.n)


@dataclass
class StridedRule:
    out_spatial: Tuple[int, ...]
    down: torch.Tensor          # [K, n_out_pad]
    up: torch.Tensor            # [K, n_in_pad]
    K: int
    n_in: int
    n_out: int


_side_streams: Dict[torch.device, "torch.cuda.Stream"] = {}


class _RulebookStream:
    """Context: hash / rulebook work runs on a per-device side stream.

    Rulebooks depend only on coordinates, never on features, but sizing the next level needs a row count on the
    host.  On the caller's stream that read-back waits for every feature kernel queued so far (milliseconds of
    convolutions) and the GPU then idles until the host has refilled the queue; on a side stream it waits for the
    rulebook kernels alone, and those overlap the feature kernels.  On exit the caller's stream is made to wait for
    the side stream's event, and every tensor produced inside is registered with the caller's stream
    (``record_stream``) so the caching allocator does not recycle it while feature kernels still read it."""

    def __init__(self, md, join_first=False):
        self.md, self.join_first = md, join_first

    def __enter__(self):
        md = self.md
        self.main = torch.cuda.current_stream(md.device)
        self.prefetch = md._prefetch is not None
        side = _side_streams.get(md.device)
        if side is None:
            side = _side_streams[md.device] = torch.cuda.Stream(device=md.device)
        self.side = side
        if self.join_first:
            if not self.prefetch:        # the coordinates were produced on the caller's stream
                side.wait_stream(self.main)
            elif md._prefetch["ready"] is not None:      # ... or by a copy whose completion event we were given
                side.wait_event(md._prefetch["ready"])
        torch.cuda.set_stream(side)
        return self

    def publish(self, *tensors):
        for t in tensors:
            if t is not None:
                if self.prefetch:        # the consuming stream is not known yet: registered when the metadata is taken
                    self.md._prefetch["tensors"].append(t)
                else:
                    t.record_stream(self.main)
        return tensors[0] if len(tensors) == 1 else tensors

    def __exit__(self, *exc):
        ev = self.side.record_event()
        torch.cuda.set_stream(self.main)
        if self.prefetch:
            self.md._prefetch["event"] = ev      # nobody waits yet: that is the point of prefetching
        else:
            self.main.wait_event(ev)
        return False


class Metadata:
    def __init__(self, dimension: int, device):
        self.dimension = dimension
        self.device = torch.device(device)
        self.levels: Dict[Tuple[int, ...], Level] = {}
        self.subm: Dict[tuple, torch.Tensor] = {}
        self.strided: Dict[tuple, StridedRule] = {}
        self.row_of_input = None        # int32 [n_input]
        self.max_batch_index = -1       # largest batch index among the input rows (read back with n_active)
        self.n_input = 0
        self.batch_size = 0
        self.input_spatial = None
        self.plan = []                  # rulebooks in the order the network asked for them (replayed by prefetch())
        self._prefetch = None           # while being built ahead of use: {"ready", "event", "tensors"}

    # -- input ---------------------------------------------------------------------------------
    def build_input(self, coords, spatial):
        """InputLayer rules: packed keys, first-appearance row numbering, hash table of the input level."""
        spatial = tuple(spatial)
        with self.rulebook_stream(join_first=True) as rs:
            info = torch.zeros((4,), dtype=torch.int32, device=coords.device)
            keys = ops.pack_coords(coords, self.dimension, info)
            rows, keys_out, tk, tv, cap, got = ops.input_layer_rules(keys, info)
            lvl = self.add_level(spatial, keys_out, (tk, tv, cap))
            rs.publish(rows, keys_out, tk, tv)
        if got[1]:
            raise ValueError("InputLayer: coordinates must lie in [0, 65535] and batch indices in [0, 65534] "
                             "(16-bit fields of the packed site keys); got values outside that range")
        self.max_batch_index = int(got[2]) if keys.shape[0] else -1
        self.row_of_input = rows
        self.n_input = int(keys.shape[0])
        self.input_spatial = spatial
        return lvl

    def adopt(self):
        """A prefetched metadata becomes the current one: its tensors (allocated on the rulebook stream) are registered
        with the consuming stream, which waits for the rulebook stream's last event."""
        pf, self._prefetch = self._prefetch, None
        if pf is None:
            return self
        main = torch.cuda.current_stream(self.device)
        for t in pf["tensors"]:
            t.record_stream(main)
        if pf["event"] is not None:
            main.wait_event(pf["event"])
        return self

    # -- levels ------------------------------------------------------------------------------
    def rulebook_stream(self, join_first=False) -> _RulebookStream:
        return _RulebookStream(self, join_first)

    def add_level(self, spatial, keys, table=None):
        n = int(keys.shape[0])
        if table is None:
            table = ops.hash_build(keys)
        self.levels[tuple(spatial)] = Level(keys, n, table[0], table[1], table[2])
        return self.levels[tuple(spatial)]

    def coords(self, spatial) -> torch.Tensor:
        """int64 [n, dimension+1] (coords..., batch) in row order == get_spatial_locations()."""
        lvl = self.levels[tuple(spatial)]
        c = ops.unpack_keys(lvl.keys).long()
        if self.dimension < 3:
            c = torch.cat([c[:, : self.dimension], c[:, 3:4]], 1)
        return c

    # -- rulebooks ---------------------------------------------------------------------------
    def subm_table(self, spatial, filt) -> torch.Tensor:
        key = (tuple(spatial), tuple(filt))
        if key not in self.subm:
            lvl = self.levels[tuple(spatial)]
            self.plan.append(("subm", tuple(spatial), tuple(filt)))
            with self.rulebook_stream() as rs:
                self.subm[key] = rs.publish(
                    ops.subm_rulebook(lvl.keys, lvl.table_keys, lvl.table_vals, lvl.cap, pad3(filt, 1)))
        return self.subm[key]

    def strided_rule(self, spatial, filt, stride) -> StridedRule:
        spatial, filt, stride = tuple(spatial), tuple(filt), tuple(stride)
        key = (spatial, filt, stride)
        if key in self.strided:
            return self.strided[key]
        if filt != stride:
            raise NotImplementedError(
                "strided Convolution/Deconvolution is implemented for filter_size == filter_stride "
                "(every use in the reference: [2,2,2], [1,2,2], 2)")
        out_spatial = []
        for a in range(len(spatial)):
            if (spatial[a] - filt[a]) % stride[a] != 0:
                raise AssertionError(f"spatial size {spatial} not compatible with filter {filt} / stride {stride}")
            out_spatial.append((spatial[a] - filt[a]) // stride[a] + 1)
        out_spatial = tuple(out_spatial)
        lvl = self.levels[spatial]
        self.plan.append(("strided", spatial, filt, stride))
        with self.rulebook_stream() as rs:
            keys_out, out_row, off, table = ops.strided_rulebook(lvl.keys, pad3(stride, 1))
            if out_spatial in self.levels:
                # coarse grid already exists (e.g. built through another path): re-index onto its rows
                have = self.levels[out_spatial]
                remap = ops.hash_lookup(keys_out, have.table_keys, have.table_vals, have.cap)
                out_row = remap[out_row.long()].contiguous()
                n_out = have.n
            else:
                new = self.add_level(out_spatial, keys_out.clone(), table)      # the rulebook left the level's hash table behind
                rs.publish(new.keys, new.table_keys, new.table_vals)
                n_out = int(keys_out.shape[0])
            K = 1
            for f in filt:
                K *= f
            down, up = rs.publish(*ops.strided_tables(out_row, off, K, lvl.n, n_out))
        rule = StridedRule(out_spatial, down, up, K, lvl.n, n_out)
        self.strided[key] = rule
        return rule


# ---------------------------------------------------------------------------------------------
# Rulebook prefetch: rulebooks depend on coordinates only, so a data pipeline that knows its next batch can have them
# built on the rulebook stream while the current step's backward runs (the stem's 125-offset table alone is ~1.2 ms of
# otherwise exposed time at the start of a step).  Explicit and identity-based: the prefetched metadata is used only
# if InputLayer later receives THE SAME coordinate tensor object.
# ---------------------------------------------------------------------------------------------
_prefetched = {}


def prefetch(coords, dimension, spatial_size, plan, ready_event=None):
    """Builds InputLayer rules and the rulebooks listed in `plan` (a previous Metadata.plan) for `coords` ahead of use.
    `ready_event`: CUDA event after which `coords` is valid (e.g. the end of its host->device copy), or None if it
    already is."""
    coords = torch.as_tensor(coords)
    if not coords.is_cuda:
        return None
    md = Metadata(dimension, coords.device)
    md._prefetch = {"ready": ready_event, "event": None, "tensors": []}
    md.build_input(coords, tuple(int(v) for v in spatial_size))
    for item in list(plan):
        try:
            if item[0] == "subm":
                md.subm_table(item[1], item[2])
            else:
                md.strided_rule(item[1], item[2], item[3])
        except KeyError:            # a level the plan expects does not exist for this input: leave the rest to the forward
            break
    _prefetched.clear()             # one batch ahead
    _prefetched[id(coords)] = (coords, md, dimension, tuple(int(v) for v in spatial_size))
    return md


def take_prefetched(coords, dimension, spatial):
    hit = _prefetched.pop(id(coords), None)
    if hit is None or hit[0] is not coords or hit[2] != dimension or hit[3] != tuple(spatial):
        return None
    return hit[1].adopt()


class Pending:
    """A bandwidth-bound layer whose launch is deferred by one module so that the NEXT module can fuse with it:
    BatchNormalization -> LeakyReLU/ReLU and AddTable -> LeakyReLU/ReLU run as ONE kernel each (forward and
    backward) instead of two.  Any other consumer reads ``.features``, which runs the deferred layer unfused."""

    __slots__ = ("kind", "run", "fuse", "rerun")

    def __init__(self, kind, run, fuse, rerun=None):
        self.kind = kind        # "bn" | "add"
        self.run = run          # () -> features, the layer as written
        self.fuse = fuse        # (leak) -> features of layer followed by leaky ReLU
        self.rerun = rerun or run   # the layer as written, evaluated a SECOND time (no side effects: running statistics)


class SparseConvNetTensor:
    """features [nActive, C] + shared metadata + spatial_size (LongTensor), as in SCN."""

    def __init__(self, features=None, metadata=None, spatial_size=None, pending=None, _sp=None):
        self._features = features
        self._pending = pending
        self._taken = None
        self.metadata = metadata
        self._spatial_size = spatial_size
        self._spc = _sp            # spatial_size as a tuple of ints (reading a LongTensor element-wise costs microseconds)

    @property
    def spatial_size(self):
        return self._spatial_size

    @spatial_size.setter
    def spatial_size(self, value):
        self._spatial_size = value
        self._spc = None

    @property
    def features(self):
        if self._pending is not None:
            self._features = self._pending.run()
            self._pending = None
        elif self._features is None and self._taken is not None:
            # a second consumer of a tensor whose layer was fused into a following activation: run it as written
            self._features = self._taken.rerun()
            self._taken = None
        return self._features

    @features.setter
    def features(self, value):
        self._features = value
        self._pending = None

    def take_pending(self):
        """Hands the deferred layer to a fusing consumer (the tensor then owns no features of its own)."""
        pend, self._pending = self._pending, None
        self._taken = pend
        return pend

    def _sp(self):
        c = self._spc
        if c is None:
            c = self._spc = tuple(int(v) for v in self._spatial_size)
        return c

    def get_spatial_locations(self, spatial_size=None):
        sp = self._sp() if spatial_size is None else tuple(int(v) for v in spatial_size)
        return self.metadata.coords(sp).cpu()

    def batch_size(self):
        return self.metadata.batch_size

    def to(self, *args, **kwargs):
        self.features = self.features.to(*args, **kwargs)
        return self

    def type(self, t=None):
        if t is None:
            return self.features.type()
        self.features = self.features.type(t)
        return self

    def cuda(self):
        self.features = self.features.cuda()
        return self

    def cpu(self):
        out = SparseConvNetTensor(self.features.cpu(), self.metadata, self.spatial_size)
        return out

    def detach(self):
        return SparseConvNetTensor(self.features.detach(), self.metadata, self.spatial_size)

    @property
    def requires_grad(self):
        return self.features.requires_grad

    def __repr__(self):
        return (f"SparseConvNetTensor<b200>(features={tuple(self.features.shape)}, dtype={self.features.dtype}, "
                f"spatial_size={self._sp()})")
