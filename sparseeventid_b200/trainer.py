"""Event-sharded data-parallel training step for the sparse ResNet (SURVEY.md §8e, §8f rank 3).

Replaces, for this path only, the reference's Lightning DDPStrategy / Horovod DistributedOptimizer
(src/utils/create_trainer.py:46-60, src/utils/torch/distributed_trainer.py:95): one process per GPU,
events are independent so the batch is split by event, BatchNorm statistics stay per rank (no SyncBN in
the reference), and the only exchange is the gradient mean -- done here on ONE flat fp32 gradient arena,
all-reduced bucket by bucket from autograd hooks so NCCL (NVLink 5 / NVSwitch) overlaps the rest of
the backward.  Loss / optimizer follow src/utils/supervised_eventID.py:168-207 and
src/utils/training_utils.py:13 (Adam lr=1.0 x schedule, eps 1e-6, betas (0.8, 0.9), weight decay 1e-6).
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import torch
import torch.distributed as dist

from . import networks


class FlatGradArena:
    """All parameter gradients as views into one fp32 buffer; bucketed async all-reduce from hooks."""

    def __init__(self, params: List[torch.nn.Parameter], bucket_bytes: int = 32 << 20, process_group=None,
                 overlap: bool = False):
        """overlap=False (default): ONE all-reduce of the whole arena after the backward.  The convolution kernels
        are persistent (one CTA per SM, 220 KB of shared memory each): a NCCL kernel that runs concurrently takes SMs
        away and every overlapped convolution then needs a second wave -- measured at 2 GPUs, bucketed overlap cost
        2.8 ms per step against ~0.5 ms for the exposed single all-reduce (83.5 MB over NVLink 5).
        overlap=True: bucketed asynchronous all-reduces launched from gradient-ready hooks (DDP style)."""
        self.params = [p for p in params if p.requires_grad]
        self.group = process_group
        self.overlap = overlap
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        total = sum(p.numel() for p in self.params)
        dev = self.params[0].device
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        # parameters are laid out in REVERSE registration order: the backward produces gradients roughly
        # from the last layer to the first, so bucket 0 fills first and its all-reduce starts earliest
        self.buckets = []            # (start, end, n_params)
        self._bucket_of: Dict[int, int] = {}
        off = 0
        b_start, b_count = 0, 0
        for p in reversed(self.params):
            n = p.numel()
            p.grad = self.flat[off:off + n].view_as(p)
            self._bucket_of[id(p)] = len(self.buckets)
            off += n
            b_count += 1
            if (off - b_start) * 4 >= bucket_bytes:
                self.buckets.append((b_start, off, b_count))
                b_start, b_count = off, 0
        if b_count:
            self.buckets.append((b_start, off, b_count))
        self._views = [p.grad for p in self.params]
        self._pending = [0] * len(self.buckets)
        self._works = []
        self._hooks = []
        # Parameters of the sparse modules get their gradients ACCUMULATED IN PLACE by the kernels (wgrad atomics,
        # BatchNorm / bias column sums) straight into the arena: no dW temporaries, no zero fills, no AccumulateGrad
        # adds (218 small launches per step).  Those never reach autograd's accumulation hook, so the functions call
        # `_scn_grad_ready` themselves; every other parameter (the dense heads) uses the normal hook.
        self._param_of_ptr = {}
        for p in self.params:
            if getattr(p, "_scn_param", False):
                p._scn_direct_grad = True
                if self.world > 1 and overlap:
                    p._scn_grad_ready = self._on_grad
                    self._param_of_ptr[p.data_ptr()] = p
            elif self.world > 1 and overlap:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._on_grad))
        if self.world > 1 and overlap:
            from .scn import _ext
            ext = _ext.get()
            if ext is not None:      # the C++ autograd functions report completed in-place gradients through this
                ext.set_grad_ready_callback(lambda t: self._on_grad(self._param_of_ptr[t.data_ptr()]))

    def _bind(self):
        """(Re-)points every parameter's .grad at its slice of the arena.  optimizer.zero_grad() / model.zero_grad()
        default to set_to_none=True: autograd would then allocate fresh gradient tensors, the kernels' in-place
        accumulation would fall back, and finish() would all-reduce a stale buffer (ranks silently diverge)."""
        for p, view in zip(self.params, self._views):        # identity test: ~50 ns per parameter
            if p.grad is not view:
                p.grad = view

    def zero(self):
        self._bind()
        self.flat.zero_()
        self._pending = [c for (_, _, c) in self.buckets]
        self._works = []

    def _on_grad(self, p):
        b = self._bucket_of[id(p)]
        self._pending[b] -= 1
        if self._pending[b] == 0:
            s, e, _ = self.buckets[b]
            self._works.append(dist.all_reduce(self.flat[s:e], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def finish(self):
        """Waits for the in-flight bucket all-reduces and turns the sums into means."""
        if self.world == 1:
            return
        for p, view in zip(self.params, self._views):        # a gradient that left the arena would never be averaged
            if p.grad is not view:
                raise RuntimeError("FlatGradArena: a parameter's .grad no longer points into the arena (zero_grad with "
                                   "set_to_none=True after arena.zero()?); call arena.zero() at the start of every step")
        if not self.overlap:
            if dist.get_backend(self.group) == "nccl":
                dist.all_reduce(self.flat, op=dist.ReduceOp.AVG, group=self.group)
            else:
                dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=self.group)
                self.flat.mul_(1.0 / self.world)
            return
        for b, left in enumerate(self._pending):      # parameters that received no gradient this step
            if left > 0:
                s, e, _ = self.buckets[b]
                self._works.append(dist.all_reduce(self.flat[s:e], op=dist.ReduceOp.SUM, group=self.group,
                                                   async_op=True))
                self._pending[b] = 0
        for w in self._works:
            w.wait()
        self._works = []
        self.flat.mul_(1.0 / self.world)


def warmup_flat_lr(step: int, peak: float = 3e-3, warmup_steps: int = 100) -> float:
    """First two segments of WarmupFlatDecay (src/utils/learning_rate_scheduler.py:92-126)."""
    if step < warmup_steps:
        return 1e-5 + (peak - 1e-5) * step / max(warmup_steps, 1)
    return peak


# ------------------------------------------------------------------------------------------------
# Checkpoints in the reference's (pytorch_lightning) layout: {"state_dict": {"encoder....", "head...."}, ...}.
# src/utils/create_trainer.py:83-115: ModelCheckpoint every 50 steps; restore = the whole module, or with
# mode.restore_encoder_only the encoder alone (keys containing "encoder", prefix stripped) which is then FROZEN.
# ------------------------------------------------------------------------------------------------


LIGHTNING_VERSION = "2.0.0"      # the envelope below is the one pytorch_lightning 2.x writes and validates on resume


def checkpoint_dict(model: torch.nn.Module, optimizer=None, scheduler=None, global_step: int = 0, epoch: int = 0) -> dict:
    """A checkpoint the reference can resume from: `pl.Trainer.fit(ckpt_path=...)` (create_trainer.py:107-115) reads
    "state_dict", "optimizer_states", "lr_schedulers", "epoch", "global_step", "pytorch-lightning_version", "loops" and
    "callbacks"; the last three are written as the minimal envelope Lightning accepts (loop progress restarts from the
    recorded global step, callback state empty)."""
    ck = {"state_dict": {k: v.detach().cpu() for k, v in model.state_dict().items()}, "global_step": int(global_step),
          "epoch": int(epoch), "pytorch-lightning_version": LIGHTNING_VERSION, "loops": {}, "callbacks": {},
          "optimizer_states": [], "lr_schedulers": []}
    if optimizer is not None:
        ck["optimizer_states"] = [optimizer.state_dict()]
    if scheduler is not None:
        ck["lr_schedulers"] = [scheduler.state_dict()]
    return ck


def restore_checkpoint(model: torch.nn.Module, checkpoint: dict, encoder_only: bool = False, optimizer=None,
                       scheduler=None) -> int:
    """Loads a Lightning-layout checkpoint (this repo's or the reference's) into `model`; returns its global step.
    encoder_only mirrors create_trainer.py:94-106: only the encoder's tensors are loaded and the encoder is frozen.
    A reference checkpoint may carry tensors of the LightningModule that are not part of the networks (e.g.
    `criterion.weight` with loss_balance_scheme=even, supervised_eventID.py): keys outside `encoder.` / `head.` are
    ignored; a key the model needs and the checkpoint lacks is an error."""
    sd = checkpoint["state_dict"]
    if encoder_only:
        enc = {k.replace("encoder.", ""): v for k, v in sd.items() if "encoder" in k}
        model.encoder.load_state_dict(enc)
        for p in model.encoder.parameters():
            p.requires_grad = False
        return int(checkpoint.get("global_step", 0))
    own = {k: v for k, v in sd.items() if k.startswith("encoder.") or k.startswith("head.")}
    missing, unexpected = model.load_state_dict(own, strict=False)
    if missing or unexpected:
        raise KeyError(f"checkpoint does not match the model: missing {list(missing)[:5]}, unexpected {list(unexpected)[:5]}")
    if optimizer is not None and checkpoint.get("optimizer_states"):
        optimizer.load_state_dict(checkpoint["optimizer_states"][0])
    if scheduler is not None and checkpoint.get("lr_schedulers"):
        scheduler.load_state_dict(checkpoint["lr_schedulers"][0])
    return int(checkpoint.get("global_step", 0))


class Trainer:
    def __init__(self, scn, dataset: str = "dune3d", device="cuda", cfg: Optional[networks.EncoderConfig] = None,
                 seed: int = 0, weight_decay: float = 1e-6, peak_lr: float = 3e-3, fused_adam: Optional[bool] = None):
        torch.manual_seed(seed)
        self.scn, self._convs = scn, None
        enc, head = networks.build_networks(scn, dataset, cfg)
        self.model = networks.EventIDModel(enc, head).to(device)
        self.device = torch.device(device)
        self.distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if self.distributed:      # rank 0's initial weights everywhere (distributed_trainer.py:127-133)
            for t in list(self.model.parameters()) + list(self.model.buffers()):
                dist.broadcast(t.data, src=0)
        self.arena = FlatGradArena(list(self.model.parameters()))
        if fused_adam is None:
            fused_adam = self.device.type == "cuda"
        self.opt = torch.optim.Adam(self.model.parameters(), lr=1.0, eps=1e-6, betas=(0.8, 0.9),
                                    weight_decay=weight_decay, fused=fused_adam)
        self.sched = torch.optim.lr_scheduler.LambdaLR(self.opt, lambda s: warmup_flat_lr(s, peak_lr))
        self.peak_lr = peak_lr
        self.global_step = 0
        self.graph_head = os.environ.get("SCN_B200_GRAPH_HEAD", "1") not in ("0", "false", "False")
        self._head_graphs = {}
        self.model.train()

    def save_checkpoint(self, path: str) -> None:
        """Lightning-layout checkpoint (rank 0 writes under data parallelism: every rank holds the same state)."""
        if not self.distributed or dist.get_rank() == 0:
            torch.save(checkpoint_dict(self.model, self.opt, self.sched, self.global_step), path)

    def load_checkpoint(self, path: str, encoder_only: bool = False) -> None:
        ck = torch.load(path, map_location="cpu", weights_only=False)
        self.global_step = restore_checkpoint(self.model, ck, encoder_only, None if encoder_only else self.opt,
                                              None if encoder_only else self.sched)
        if encoder_only:      # frozen parameters leave the optimizer and the gradient arena
            live = [p for p in self.model.parameters() if p.requires_grad]
            self.arena = FlatGradArena(live)
            self.opt = torch.optim.Adam(live, lr=1.0, eps=1e-6, betas=(0.8, 0.9),
                                        weight_decay=self.opt.param_groups[0]["weight_decay"],
                                        fused=self.opt.param_groups[0].get("fused") or False)
            self.sched = torch.optim.lr_scheduler.LambdaLR(self.opt, lambda s: warmup_flat_lr(s, self.peak_lr))

    def prefetch_rulebooks(self, next_batch, ready_event=None):
        """Has the rulebooks of the NEXT batch built on the rulebook stream now (they depend on coordinates only), so
        they overlap this step's backward instead of stalling the start of the next step.  A no-op until one forward
        has recorded which rulebooks the network asks for, or on modules without the mechanism (oracle shim)."""
        il = getattr(self, "_input_layer", None)
        if il is None:
            cands = [m for m in self.model.modules() if hasattr(m, "_last_plan")]
            il = self._input_layer = cands[0] if cands else False
        if not il or not getattr(il, "_last_plan", None):
            return
        from .scn import core
        core.prefetch(next_batch[0], il.dimension, il.spatial_size, il._last_plan, ready_event)

    # ---- dense heads + focal loss as ONE CUDA graph per direction ------------------------------------------------------
    # classification_head.py:19-28 + supervised_eventID.py:168-196 on a [B, 128] pooled tensor are ~90 tiny torch launches
    # forward and ~150 backward, a few microseconds each with a launch gap after every one.  Their shapes are static (batch
    # size, channel count), so they are captured once with torch.cuda.make_graphed_callables (dropout included: the
    # capture registers the CUDA generator, every replay draws fresh random numbers) and replayed; the encoder -- whose
    # level sizes are data-dependent -- stays eager.  Eager fallback for anything unexpected (a different batch size, CPU,
    # a head that does not start with the full-extent pool, SCN_B200_GRAPH_HEAD=0).
    def _graphed_head_loss(self, feat, labels):
        if not self.graph_head or self.device.type != "cuda" or not isinstance(feat, torch.Tensor):
            return None
        heads = getattr(self.model.head, "classification_head", None)
        if heads is None or any(not isinstance(h[0], torch.nn.AvgPool3d) for h in heads.values()):
            return None
        keys = list(heads.keys())
        if any(k not in labels for k in keys):
            return None
        first = heads[keys[0]][0]
        pooled = first(feat)                                    # [B, C, 1, 1, 1]; the lazy dense view pools the sparse rows
        labs = tuple(labels[k] for k in keys)
        sig = (tuple(pooled.shape), pooled.dtype) + tuple((tuple(l.shape), l.dtype) for l in labs)
        g = self._head_graphs.get(sig)
        if g is None:
            if len(self._head_graphs) >= 4:
                return None

            class HeadLoss(torch.nn.Module):
                def __init__(self, heads, keys):
                    super().__init__()
                    self.tails = torch.nn.ModuleList([heads[k][1:] for k in keys])

                def forward(self, pooled, *labs):
                    loss = 0.0
                    for tail, lab in zip(self.tails, labs):
                        logits = tail(pooled)
                        y = torch.nn.functional.one_hot(lab, logits.size(-1))
                        p = torch.nn.functional.softmax(logits, dim=-1).clamp(1e-7, 1.0 - 1e-7)
                        loss = loss + (-y * torch.log(p) * (1 - p) ** 2).sum(dim=-1).mean()
                    return loss

            try:
                mod = HeadLoss(heads, keys)
                mod.train(self.model.head.training)
                sample = (pooled.detach().clone().requires_grad_(True),) + tuple(l.clone() for l in labs)
                g = torch.cuda.make_graphed_callables(mod, sample)
            except Exception:                                   # capture is an optimisation, never a requirement
                self.graph_head = False
                return None
            self._head_graphs[sig] = g
        return g(pooled, *labs)

    def step(self, batch, labels, prefetch=None, prefetch_ready=None):
        """batch: (coords [N,4], features [N,1], batch_size) on self.device; labels: dict of int64 [B].
        prefetch: the next step's batch tuple (same tensor objects that will be passed then), optional."""
        self.arena.zero()
        prep = getattr(self.scn, "prepare_weight_images", None)        # every conv weight image of the step in one launch
        if prep is not None and self.device.type == "cuda":
            if self._convs is None:
                self._convs = [m for m in self.model.modules() if hasattr(m, "mirror_dgrad") and hasattr(m, "workspace")]
            prep(self._convs)
        try:
            feat = self.model.encoder(batch)
            loss = self._graphed_head_loss(feat, labels)
            if loss is None:
                loss = networks.focal_loss(labels, self.model.head(feat))
            if prefetch is not None:
                self.prefetch_rulebooks(prefetch, prefetch_ready)
            loss.backward()
        finally:
            if prep is not None:
                self.scn.release_weight_images()                       # the optimizer is about to change the parameters
        self.arena.finish()
        self.opt.step()
        self.sched.step()
        self.global_step += 1
        return loss
