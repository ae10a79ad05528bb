"""Public training-step API: ``StudentTrainer``.

One object owns the model, the elastic data-parallel engine, the flat fused optimizer, the per-step
scratch arena and (on CUDA) a captured CUDA graph of the WHOLE step:

    zero grads/arena -> forward -> fused soft-CE -> backward (+ overlapped fused all-reduce buckets)
    -> fused SGD-momentum

so a replay costs one graph launch instead of ~600 kernel launches from Python.  The user-facing
call is ``trainer.step(images, targets)`` with *host* (pinned) tensors: the H2D copies, the graph
replay and the D2H read of the loss are what the end-to-end benchmark times.

This is the B200 counterpart of the reference's ``train_exe.run(train_prog, feed=data)`` hot loop
(example/distill/resnet/train_with_fleet.py:468-524).
"""
from __future__ import annotations

from typing import Callable, Optional

import torch
import torch.distributed as dist

from . import ops
from .models.resnet_vd import ConvBNAct
from .parallel import ElasticDataParallel


class LossHandle:
    """Result of ``StudentTrainer.step``: the loss of one step, readable once its asynchronous device ->
    pinned-host copy has landed.  At most ``StudentTrainer._LOSS_SLOTS`` unread handles are live at a time
    (a handle that was never read is overwritten ``_LOSS_SLOTS`` steps later)."""

    __slots__ = ("_ev", "_host", "_value")

    def __init__(self, ev, host, value=None):
        self._ev, self._host, self._value = ev, host, value

    def item(self) -> float:
        if self._value is None:
            self._ev.synchronize()
            self._value = float(self._host[0])
        return self._value

    def __float__(self) -> float:
        return self.item()

    def __format__(self, spec) -> str:
        return format(self.item(), spec)

    def __repr__(self) -> str:
        return "LossHandle(%s)" % ("pending" if self._value is None else "%.6f" % self._value)


class StepArena:
    """One flat fp32 scratch buffer holding every BN layer's forward (sum, sum^2) and backward
    (dbeta, dgamma) accumulators; zeroed with a single memset per step."""

    def __init__(self, model: torch.nn.Module, device):
        units = [m for m in model.modules() if isinstance(m, ConvBNAct)]
        total = sum(4 * u.cout + 4 for u in units)
        self.buf = torch.zeros(max(total, 4), dtype=torch.float32, device=device)
        off = 0
        for u in units:
            u.fwd_stats = self.buf[off:off + 2 * u.cout]
            off += 2 * u.cout
            bwd = self.buf[off:off + 2 * u.cout]
            off += 2 * u.cout
            sync = self.buf[off:off + 4].view(torch.int32)   # grid-barrier counters (fwd, bwd)
            off += 4
            u.bn.ws = (u.fwd_stats, bwd, sync)

    def zero(self):
        self.buf.zero_()


class StudentTrainer:
    def __init__(self, model: torch.nn.Module, batch_size: int, image_shape=(3, 224, 224),
                 num_classes: int = 1000, lr: float = 0.1, momentum: float = 0.9,
                 weight_decay: float = 1e-4, target_kind: str = "probs",
                 group: Optional[dist.ProcessGroup] = None, use_graph: bool = True,
                 bucket_cap_mb: float = 16.0, comm_blocks: int = 32, algo: str = "auto",
                 overlap: bool = True, dtype=torch.bfloat16, input_dtype=None,
                 loss_fn: Optional[Callable] = None, loss_scaling: Optional[float] = None,
                 dynamic_loss_scaling: bool = True, optimizer: Optional[Callable] = None,
                 fabric=None, clip_norm: Optional[float] = None, fused_optimizer: Optional[bool] = None,
                 comm_timeout_s: Optional[float] = None):
        self.model = model
        self.device = next(model.parameters()).device
        self.cuda = self.device.type == "cuda"
        self.batch_size = batch_size
        self.dtype = dtype
        self.target_kind = target_kind
        self.loss_fn = loss_fn
        if comm_timeout_s is None:
            # in-place elastic mode: a dead peer must surface within seconds (the kernels' barrier timeout raises the
            # fabric's error word, every later barrier then gives up at once); otherwise be patient
            import os
            comm_timeout_s = float(os.environ.get("EDL_COMM_TIMEOUT", "10" if os.environ.get(
                "EDL_RESCALE_MODE", "").lower() == "inplace" else "60"))
        self.dp = ElasticDataParallel(model, group=group, bucket_cap_mb=bucket_cap_mb, timeout_s=comm_timeout_s,
                                      comm_blocks=comm_blocks, algo=algo, overlap=overlap,
                                      check_finite=loss_scaling is not None, fabric=fabric, clip_norm=clip_norm)
        if optimizer is not None:
            self.opt = optimizer(self.dp.flat)
        else:
            self.opt = ops.FlatSGDMomentum(self.dp.flat, lr=lr, momentum=momentum,
                                           weight_decay=weight_decay)
        # fp16-style loss scaling (reference: mixed_precision.decorate(init_loss_scaling,
        # use_dynamic_loss_scaling), example/distill/resnet/train_with_fleet.py:324-327); bf16 runs
        # leave it off
        self.scaler = None
        if loss_scaling is not None:
            self.scaler = ops.DynamicLossScaler(
                self.device, init_scale=loss_scaling,
                growth_interval=1000 if dynamic_loss_scaling else (1 << 30),
                backoff_factor=0.5 if dynamic_loss_scaling else 1.0)
            self.scaler.found_inf = self.dp.found_inf
            self.scaler.attach(self.opt, self.dp)
        self._guard_comm_error()
        # the optimizer rides in the bucket hook of the data-parallel engine when nothing needs to see every
        # gradient first (loss scaling, clipping): fused reduce-scatter -> SGD -> all-gather kernel on > 1 GPU,
        # per-bucket optimizer launches on the side stream on one (parallel/ddp.py:attach_optimizer)
        self._fused_optimizer = fused_optimizer
        if isinstance(self.opt, (ops.FlatSGDMomentum, ops.FlatLARS, ops.FlatLAMB)):
            self.dp.attach_optimizer(self.opt, fused=fused_optimizer)
        # recompute runs every block's forward twice: the pre-zeroed accumulate-into arena slices would
        # be summed twice, so those runs let each op allocate its own scratch
        self.arena = StepArena(model, self.device) if self.cuda and not getattr(model, "recompute", False) else None
        in_dtype = input_dtype if input_dtype is not None else dtype
        self.static_x = torch.zeros((batch_size,) + tuple(image_shape), dtype=in_dtype,
                                    device=self.device).contiguous(memory_format=torch.channels_last)
        if target_kind == "labels":
            self.static_t = torch.zeros(batch_size, dtype=torch.int64, device=self.device)
        else:
            self.static_t = torch.zeros(batch_size, num_classes, dtype=dtype, device=self.device)
        self.static_loss = torch.zeros((), dtype=torch.float32, device=self.device)
        self.use_graph = use_graph and self.cuda
        self.graph = None
        self.steps_done = 0
        # ONE stream per module for every optimizer step, eager or captured, of every trainer that ever
        # drives it.  autograd pins each parameter's gradient-accumulator node to the stream of its first
        # use and joins those "leaf streams" at the end of every backward -- a CUDA-graph capture on any
        # other stream then fails with "dependency created on uncaptured work in another stream"
        # (tools/diag_seq.py reproduces it with two trainers on one model).  High priority: the step is the
        # critical chain, weight gradients run below it (parallel/ddp.py).
        self._cap_stream = None
        if self.cuda:
            self._cap_stream = getattr(model, "_edl_step_stream", None)
            if self._cap_stream is None:
                self._cap_stream = torch.cuda.Stream(device=self.device, priority=-1)
                model._edl_step_stream = self._cap_stream

    # ------------------------------------------------------------------ one step on device
    def _step_body(self):
        self.dp.zero_grad()
        if self.arena is not None:
            self.arena.zero()
        x = self.static_x
        if x.dtype != self.dtype:
            x = x.to(self.dtype)
        logits = self.model(x)
        if self.loss_fn is not None:
            loss = self.loss_fn(logits, self.static_t)
        else:
            loss = ops.soft_cross_entropy(logits, self.static_t, target_kind=self.target_kind)
        (self.scaler.scale_loss(loss) if self.scaler is not None else loss).backward()
        self.dp.finish()
        self.opt.step()
        if self.scaler is not None:
            self.scaler.update()
        self.static_loss.copy_(loss.detach())

    def capture(self, warmup: int = 3):
        """Warm up on a side stream (cuDNN autotune, allocator) then capture the step graph."""
        if not self.use_graph:
            return
        # the step is captured on a HIGH-priority stream: its kernels are the critical chain, the
        # weight-gradient side stream (parallel/ddp.py) runs at low priority underneath it
        s = self._cap_stream
        s.wait_stream(torch.cuda.current_stream(self.device))
        self.dp.warming = True                 # eager collectives of the warm-up wait patiently for slower ranks
        try:
            with torch.cuda.stream(s):
                for _ in range(warmup):
                    self._step_body()
            torch.cuda.current_stream(self.device).wait_stream(s)
            torch.cuda.synchronize(self.device)
        finally:
            self.dp.warming = False
        self.dp.barrier()
        self.graph = torch.cuda.CUDAGraph()
        before = ops.launches()
        with torch.cuda.graph(self.graph, stream=s):
            self._step_body()
        self.launches_per_step = ops.launches() - before
        torch.cuda.synchronize(self.device)
        self.dp.barrier()                      # every rank replays its first step within milliseconds of the others

    def step_device(self):
        """Run one optimizer step on whatever is currently in the static input buffers."""
        if self.use_graph:
            if self.graph is None:
                self.capture()
            self.graph.replay()
            ops.count_launch(self.launches_per_step)
        elif self._cap_stream is not None:
            cur = torch.cuda.current_stream(self.device)
            self._cap_stream.wait_stream(cur)            # inputs were copied on the caller's stream
            with torch.cuda.stream(self._cap_stream):
                self._step_body()
            cur.wait_stream(self._cap_stream)
        else:
            self._step_body()
        self.steps_done += 1
        return self.static_loss

    def step(self, images: torch.Tensor, targets: torch.Tensor, sync: bool = False):
        """Public per-step call.  ``images`` / ``targets`` may live on the host (ideally pinned).

        Default (``sync=False``): the double-buffered feed of ``step_pipelined`` -- the host -> device copy of this
        batch is staged on a copy stream while the previous step still runs, and the returned ``LossHandle`` is
        readable (``.item()`` / ``float()``) once its asynchronous device -> host copy has landed; read it one step
        late and the host never stalls the GPU.  ``sync=True``: copy on the caller's stream, run, and return the
        device-resident scalar loss tensor (the round-1 behaviour)."""
        if not sync:
            return self.step_pipelined(images, targets)
        self.static_x.copy_(images, non_blocking=True)
        self.static_t.copy_(targets, non_blocking=True)
        return self.step_device()

    # ------------------------------------------------------------------ double-buffered feed
    def _pipe_init(self):
        self._copy_stream = torch.cuda.Stream(device=self.device)
        self._stage_x = [torch.empty_like(self.static_x) for _ in range(2)]
        self._stage_t = [torch.empty_like(self.static_t) for _ in range(2)]
        self._stage_ready = [torch.cuda.Event() for _ in range(2)]
        self._stage_free = [torch.cuda.Event() for _ in range(2)]
        cur = torch.cuda.current_stream(self.device)
        for ev in self._stage_free:
            ev.record(cur)
        self._loss_host = torch.zeros(self._LOSS_SLOTS, dtype=torch.float32).pin_memory()
        self._loss_ev = [torch.cuda.Event() for _ in range(self._LOSS_SLOTS)]
        self._pipe_i = 0

    _LOSS_SLOTS = 4

    def step_pipelined(self, images: torch.Tensor, targets: torch.Tensor) -> "LossHandle":
        """``step()`` with the host work taken off the critical path (the reference feeds its trainers through
        a double-buffered reader: ``use_double_buffer`` of the Paddle data loader used by
        example/distill/resnet/train_with_fleet.py).

        The pinned-host -> device copy of THIS batch goes to one of two staging buffers on a copy stream, so
        it overlaps the previous step still running on the GPU; the step stream then moves it into the
        graph's static input (device-to-device) and replays the step.  The loss is copied to pinned host
        memory asynchronously; the returned handle's ``item()`` waits for that copy only -- read it one step
        late (``h = step_pipelined(b[i+1]); prev.item()``) and the host never stalls the GPU."""
        if not self.cuda:
            return LossHandle(None, None, float(self.step(images, targets, sync=True)))
        if getattr(self, "_copy_stream", None) is None:
            self._pipe_init()
        k = self._pipe_i % 2
        j = self._pipe_i % self._LOSS_SLOTS
        self._pipe_i += 1
        cs = self._copy_stream
        cs.wait_event(self._stage_free[k])           # the slot's previous contents were consumed two steps ago
        with torch.cuda.stream(cs):
            self._stage_x[k].copy_(images, non_blocking=True)
            self._stage_t[k].copy_(targets, non_blocking=True)
            self._stage_ready[k].record(cs)
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(self._stage_ready[k])
        self.static_x.copy_(self._stage_x[k], non_blocking=True)
        self.static_t.copy_(self._stage_t[k], non_blocking=True)
        self._stage_free[k].record(cur)
        self.step_device()
        self._loss_host[j:j + 1].copy_(self.static_loss.view(1), non_blocking=True)
        self._loss_ev[j].record(cur)
        return LossHandle(self._loss_ev[j], self._loss_host[j:j + 1])

    def set_lr(self, lr: float):
        self.opt.set_lr(lr)

    @torch.no_grad()
    def evaluate(self, batches):
        """Per-rank evaluation + all-reduce of the counters (the reference evaluates on trainer 0 with a
        single-process multi-GPU ``CompiledProgram.with_data_parallel``,
        example/distill/resnet/train_with_fleet.py:403-404,537-575).  ``batches`` yields (images, int64
        labels); returns {"acc1", "acc5", "n"} over all ranks."""
        was_training = self.model.training
        self.model.eval()
        counts = torch.zeros(3, device=self.device, dtype=torch.float32)
        for images, labels in batches:
            x = images.to(self.device, non_blocking=True)
            if x.dtype != self.dtype:
                x = x.to(self.dtype)
            if x.dim() == 4:
                x = x.contiguous(memory_format=torch.channels_last)
            labels = labels.to(self.device, non_blocking=True).view(-1)
            hits = ops.topk_accuracy(self.model(x), labels)
            counts[:2] += hits.to(counts.device)
            counts[2] += labels.numel()
        if self.dp.world > 1:
            counts = self.dp.allreduce_scalars(counts)
        self.model.train(was_training)
        n = max(1.0, float(counts[2]))
        return {"acc1": float(counts[0]) / n, "acc5": float(counts[1]) / n, "n": int(counts[2])}

    # ------------------------------------------------------------------ elastic
    def _guard_comm_error(self):
        """In-place elastic mode: make the fused optimizer skip its update on device while the fabric's error word is
        set.  A peer that died mid-step makes our all-reduce kernels time out with partial sums in the gradient buffer;
        with the optimizer's ``found_inf`` pointer aimed at that word, every step from the broken one on is a no-op --
        no host round trip, graph replays included -- until ``ElasticContext.poll(agree=dp.agree)`` notices, ``recover()``
        rebuilds the group and the parameters are still those of the last good step."""
        import os

        if (os.environ.get("EDL_RESCALE_MODE", "").lower() != "inplace" or self.scaler is not None
                or self.dp.pool is None or not hasattr(self.opt, "set_found_inf")):
            return
        w = ops.native().comm_error_word_offset()
        self.opt.set_found_inf(self.dp.pool.sig_tensor()[w:w + 1], comm_error=True)

    def prepare_rescale(self):
        """Collective over the OLD stage, before a planned membership change (``ElasticContext.poll()`` said switch):
        with the fused optimizer every rank only kept its slices of master weights / momentum current."""
        self.dp.consolidate_optimizer_state()

    def consolidate(self):
        """Collective: make this rank's optimizer state complete (call on every rank before rank 0 checkpoints)."""
        self.dp.consolidate_optimizer_state()

    def rebuild(self, group=None, fabric=None, failed: bool = False):
        """World-size change: re-plan the communication, drop the captured graph.  ``failed=True``: the old stage
        broke (a peer died); the sharded optimizer state is completed locally instead of collectively."""
        self.graph = None
        if failed:
            self.dp.localize_optimizer_state()
        self.dp.rebuild(group, fabric=fabric)
        if self.scaler is None and hasattr(self.opt, "set_found_inf"):
            self.opt.set_found_inf(None)          # the old pool (and its error word) is gone
        self._guard_comm_error()
        if getattr(self, "_copy_stream", None) is not None:
            torch.cuda.synchronize(self.device)

    @torch.no_grad()
    def sync_from(self, root: int = 0):
        """After a join: take parameters, fp32 masters, optimizer state (tensors AND step counters / learning rate)
        and the module buffers (BatchNorm running statistics) from ``root`` over the fabric (NVSwitch broadcast
        kernel) instead of re-reading the checkpoint from the file system."""
        self.dp.broadcast_parameters(root)
        for st in getattr(self.opt, "state", {}).values():
            for v in st.values():
                if torch.is_tensor(v):
                    self.dp.broadcast_tensor(v, root)
        for name in ("step_t", "lr_t"):
            v = getattr(self.opt, name, None)
            if torch.is_tensor(v):
                self.dp.broadcast_tensor(v, root)
        if hasattr(self.opt, "lr_t"):
            self.opt.lr = float(self.opt.lr_t.item())
        bufs = [b for b in self.model.buffers() if torch.is_tensor(b) and b.numel() > 0]
        by_dtype = {}
        for b in bufs:
            by_dtype.setdefault(b.dtype, []).append(b)
        for dt, group in by_dtype.items():              # one broadcast per dtype, not one per BatchNorm layer
            flat = torch.cat([b.reshape(-1) for b in group])
            self.dp.broadcast_tensor(flat, root)
            off = 0
            for b in group:
                b.copy_(flat[off:off + b.numel()].view_as(b))
                off += b.numel()
        if self.cuda:
            torch.cuda.synchronize(self.device)

    def state_dict(self):
        if self.dp.state_sharded and not self.dp.state_complete:
            raise RuntimeError("the optimizer state is sharded across ranks (fused optimizer): call "
                               "trainer.consolidate() on EVERY rank before state_dict()")
        return {"model": {k: v for k, v in self.model.state_dict().items()},
                "optim": self.opt.state_dict(), "steps_done": self.steps_done}

    def load_state_dict(self, sd):
        self.model.load_state_dict(sd["model"])
        self.dp.flat.sync_master_from_params()
        self.opt.load_state_dict(sd["optim"])
        self.steps_done = sd.get("steps_done", 0)
        self.graph = None
