"""ElasticDataParallel -- the B200-native replacement for Paddle fleet collective DP.

Reference behaviour being replaced: ``fleet.distributed_optimizer(opt, strategy).minimize(loss)``
inserts fused (<=16 MB) NCCL all-reduces after backward (example/distill/resnet/
train_with_fleet.py:332-333,353-364; scripts/train_gpu.sh:67-70) and every membership change
restarts all trainer processes (utils/launcher.py:221-244).

Here:
* gradients live in ONE flat buffer per dtype inside NVSwitch-symmetric memory (``FlatParams``);
  buckets are zero-copy windows of it, planned from (world size, bucket cap) -- re-planned by
  ``rebuild()`` on every elastic stage change without touching model or optimizer state;
* as soon as autograd (or a fused op writing straight into its gradient sink) has produced every
  gradient of a bucket, the bucket's fused all-reduce kernel (csrc/allreduce.cu: P2P two-shot /
  NVLS multimem, fp32 accumulate, 1/world scale, finite check, squared-norm) is enqueued on a side
  stream so it overlaps the rest of backward; the whole thing is CUDA-graph capturable;
* with an attached ``FlatSGDMomentum`` the bucket kernel becomes gradient reduce-scatter -> SGD-momentum on the
  owned slice -> parameter all-gather (``allreduce_sgd_kernel``): one kernel per bucket instead of all-reduce +
  stream join + a separate optimizer pass, optimizer state traffic divided by the world size; on ONE GPU the same
  hook runs the optimizer per bucket on the side stream while backward is still going;
* global-norm gradient clipping (``clip_norm``): the bucket kernels accumulate sum(g^2) of the slices they reduce,
  one scalar all-gather kernel + one tiny kernel turn the partials into the device-resident clip factor the
  optimizer kernel multiplies into the gradients -- no extra pass over the gradients;
* the ranks of a stage meet either through a ``torch.distributed`` group or -- in-place elastic mode on GPUs --
  through a ``Fabric`` (store + rank + world, parallel/symm.py): no process group, no NCCL communicator at all;
* CPU / gloo groups (the fit_a_line plumbing config) fall back to ``dist.all_reduce``.
"""
from __future__ import annotations

import os
import weakref
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional

import torch
import torch.distributed as dist

from .flat import FlatParams


def _host_id() -> str:
    """Identity of the NVSwitch domain a rank lives in: host name + boot id (containers of one machine share both)."""
    import socket

    boot = ""
    try:
        with open("/proc/sys/kernel/random/boot_id") as f:
            boot = f.read().strip()
    except OSError:
        pass
    return socket.gethostname() + ":" + boot


class _NullCtx:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


@dataclass
class Bucket:
    dtype: torch.dtype
    start: int                 # element offset inside the group's flat gradient
    numel: int
    entry_ids: List[int] = field(default_factory=list)
    order: int = 0             # launch order (position of the last-ready parameter)
    pending: int = 0
    launched: bool = False
    algo: str = "twoshot"
    fused_opt: bool = False    # the bucket kernel also runs the optimizer (and, on > 1 rank, all-gathers parameters)


def plan_buckets(flat: FlatParams, cap_bytes: int, tail_bytes: int = 512 * 1024) -> List[Bucket]:
    """Cut each dtype group's flat gradient into contiguous buckets of ~cap_bytes.

    Flat layout is reverse registration order, so entry 0 of a group is the *last* layer: buckets are
    produced in the order their gradients become ready."""
    buckets: List[Bucket] = []
    eid = 0
    # global readiness order = interleaving of the dtype groups in reverse-registration order
    order_of: Dict[int, int] = {i: e.order for i, (_, e) in enumerate(flat.entries())}
    for g in flat.groups.values():
        esz = g.grad.element_size()
        # the LAST bucket (the first layers' parameters, whose gradients are produced at the very end of backward) is
        # kept small: its reduction / optimizer kernel cannot overlap anything and is exposed 1 : 1 at the end of the step
        tail_from = len(g.entries)
        if tail_bytes > 0 and len(g.entries) > 1 and g.numel * esz > 8 * tail_bytes:
            acc = 0
            while tail_from > 1 and acc < tail_bytes:
                tail_from -= 1
                acc += g.entries[tail_from].numel * esz
            if acc >= cap_bytes or tail_from <= 0:
                tail_from = len(g.entries)            # the group is small anyway: one greedy pass
        cur: Optional[Bucket] = None
        for idx, e in enumerate(g.entries):
            if cur is None:
                cur = Bucket(dtype=g.dtype, start=e.offset, numel=0)
            cur.entry_ids.append(eid)
            cur.numel = e.offset + e.numel - cur.start
            cur.order = max(cur.order, order_of[eid])
            eid += 1
            if cur.numel * esz >= cap_bytes or idx + 1 == tail_from:
                buckets.append(cur)
                cur = None
        if cur is not None:
            buckets.append(cur)
        # every bucket runs up to the start of the next one (entries start on 128-element boundaries, the alignment
        # gap behind a bucket's last tensor rides with it: kernels want multiples of 16 bytes), and the tail padding
        # of the group rides with the last bucket so the buffer is fully covered
        mine = sorted((b for b in buckets if b.dtype == g.dtype), key=lambda b: b.start)
        for b, nxt in zip(mine, mine[1:]):
            b.numel = nxt.start - b.start
        mine[-1].numel = g.numel - mine[-1].start
    buckets.sort(key=lambda b: b.order)
    return buckets


def choose_algo(nbytes: int, world: int, has_multicast: bool, prefer: str = "auto") -> str:
    """Planner rule.  NVSwitch gives every peer full bandwidth, so the crossover is about launch /
    barrier latency, not link count: NVLS (in-switch reduce, half the NVLink traffic) whenever the
    multicast alias exists, P2P two-shot otherwise; tiny out-of-place reductions use one-shot."""
    if prefer in ("twoshot", "multimem", "nccl"):
        return prefer if (prefer != "multimem" or has_multicast) else "twoshot"
    if world <= 1:
        return "none"
    if has_multicast and nbytes >= 64 * 1024:
        return "multimem"
    return "twoshot"


class ElasticDataParallel:
    def __init__(self, module: torch.nn.Module, group: Optional[dist.ProcessGroup] = None,
                 bucket_cap_mb: float = 16.0, overlap: bool = True, comm_blocks: int = 32,
                 algo: str = "auto", timeout_s: float = 60.0, average: bool = True,
                 check_finite: bool = False, track_sqnorm: bool = False, hierarchical: str = "auto",
                 fabric=None, clip_norm: Optional[float] = None):
        # one engine per module: a second engine on the same parameters would leave the first one's
        # autograd hooks installed (they would fire, and launch reductions, during the new engine's backward)
        old = getattr(module, "_edl_dp_engine", None)
        if old is not None and old() is not None:
            old().detach()
        module._edl_dp_engine = weakref.ref(self)
        self.module = module
        self.bucket_cap = int(bucket_cap_mb * (1 << 20))
        self.overlap = overlap
        self.comm_blocks = comm_blocks
        self.algo_pref = os.environ.get("EDL_ALLREDUCE_ALGO", algo)
        self.timeout_s = timeout_s
        # eager warm-up steps of a (re)built stage: ranks reach their first kernels seconds apart (cold caches, lazy
        # module loading on a fresh joiner); those launches wait patiently, the captured steady-state step does not
        self.warm_timeout_s = max(timeout_s, float(os.environ.get("EDL_COMM_WARM_TIMEOUT", "120")))
        self.warming = False
        self.average = average
        self.device = next(module.parameters()).device
        self.pool = None
        self.slices = {}
        self.found_inf = None
        self.sqnorm = None
        self.clip_norm = float(clip_norm) if clip_norm else None
        self.param_slices = {}
        self.opt = None                 # attach_optimizer()
        self.bucket_opt = False         # optimizer runs per bucket inside / right after the reduction
        self.state_sharded = False      # fused mode on > 1 rank: every rank only updates its slices of master / momentum
        self.state_complete = True      # False between a fused step and the next consolidate / localize
        self.last_algos = []            # what the last step actually launched: (algo, bytes, fused)
        if check_finite:
            self.found_inf = torch.zeros(1, dtype=torch.int32, device=self.device)
        if (track_sqnorm or self.clip_norm) and self.device.type == "cuda":
            self.sqnorm = torch.zeros(1, dtype=torch.float32, device=self.device)
            self.clip_scale_t = torch.ones(1, dtype=torch.float32, device=self.device)
            self.grad_norm_t = torch.zeros(1, dtype=torch.float32, device=self.device)
        # "auto": two-level reduction as soon as the ranks span more than one host (NVSwitch domain); "off": never
        # (one flat group; across hosts that means the library path); the reference's use_hierarchical_allreduce knob
        self.hierarchical = os.environ.get("EDL_HIERARCHICAL_ALLREDUCE", hierarchical)
        self.overlap_wgrad = os.environ.get("EDL_OVERLAP_WGRAD", "1") == "1"
        self.enabled = True     # False: gradients stay local (DGC exchanges them itself)
        self._bind_group(group, fabric)
        self.flat = FlatParams(module, grad_alloc=self._grad_alloc if self.pool is not None else None)
        self._plan()
        self._install_hooks()
        self.comm_launches = 0

    # ------------------------------------------------------------------ group / memory
    def _bind_group(self, group, fabric=None):
        self.group = group
        self.fabric = fabric
        if fabric is not None:
            # no process group: the stage's members meet in a key-value store, everything that moves between GPUs
            # moves through our own kernels over the symmetric slab (in-place elastic mode on one NVSwitch domain)
            self.world, self.rank = fabric.world, fabric.rank
            self.backend = "fabric" if self.world > 1 else "none"
            self.hier, self.local_group, self.cross_group = False, None, None
            self.local_world, self.local_rank = self.world, self.rank
        else:
            if dist.is_available() and dist.is_initialized():
                self.world = dist.get_world_size(group)
                self.rank = dist.get_rank(group)
            else:
                self.world, self.rank = 1, 0
            self.backend = dist.get_backend(group) if self.world > 1 else "none"
            self._plan_hierarchy(group)
        symm_world = self.local_world if self.hier else self.world
        self.use_symm = (symm_world > 1 and self.device.type == "cuda"
                         and self.algo_pref != "nccl")
        self.pool = None
        if self.use_symm:
            from .symm import SymmetricPool

            need = 0
            for p in self.module.parameters():
                if p.requires_grad:
                    # gradients + (fused optimizer) the bf16 parameter shadow every rank stores into
                    need += (p.numel() + 256) * p.element_size() * (2 if p.element_size() == 2 else 1)
            need += 4 << 20
            self.pool = SymmetricPool(need, group=self.local_group if self.hier else group, device=self.device,
                                      fabric=fabric)
        if self.device.type == "cuda" and getattr(self, "comm_stream", None) is None:
            # all-reduce kernels: high priority (few CTAs, on the critical path of the optimizer step);
            # weight-gradient kernels: LOW priority -- they only have to finish before their bucket is
            # reduced, and must not take SMs from the dgrad / BN-backward chain of the main stream
            self.comm_stream = torch.cuda.Stream(device=self.device, priority=-1)
            self.wgrad_stream = torch.cuda.Stream(device=self.device, priority=0)
            # a second one: the weight gradients of consecutive layers alternate between the two (ops/gemm.py)
            self.wgrad_stream2 = (torch.cuda.Stream(device=self.device, priority=0)
                                  if os.environ.get("EDL_WGRAD_STREAMS", "2") == "2" else None)
            self._main_stream = None
            self._comm_used = False

    def _plan_hierarchy(self, group):
        """Peer memory only reaches the GPUs of one NVSwitch domain.  When the ranks span several hosts the
        reduction becomes two-level (the reference's ``use_hierarchical_allreduce``, example/distill/resnet/
        train_with_fleet.py:90-91,360-362): our kernels inside a host, the library collective across hosts on 1/L of
        every bucket per rank.  Hosts must hold the same number of ranks; otherwise one flat library group."""
        self.hier, self.local_group, self.cross_group = False, group, None
        self.local_world, self.local_rank = self.world, self.rank
        if self.world <= 1 or self.hierarchical == "off":
            return
        fake = os.environ.get("EDL_FAKE_HOST")
        if not fake and os.environ.get("LOCAL_WORLD_SIZE") == str(self.world) and group is None:
            return                       # torchrun started every rank of the job on this host: nothing to find out
        me = fake or _host_id()
        hosts = [None] * self.world
        dist.all_gather_object(hosts, me, group=group)
        if len(set(hosts)) <= 1:
            return
        nodes: Dict[str, List[int]] = {}
        for r, h in enumerate(hosts):
            nodes.setdefault(h, []).append(r)
        sizes = {len(v) for v in nodes.values()}
        if len(sizes) != 1:
            self.algo_pref = "nccl"          # uneven hosts: flat library all-reduce
            return
        to_global = (lambda r: dist.get_global_rank(group, r)) if group is not None else (lambda r: r)
        L = sizes.pop()
        node_lists = list(nodes.values())
        # every member creates every subgroup in the same order (local synchronisation: ranks outside `group`,
        # e.g. the teachers of a distill job, do not take part)
        for members in node_lists:
            g = dist.new_group(ranks=[to_global(r) for r in members], use_local_synchronization=True) \
                if self.rank in members else None
            if g is not None:
                self.local_group, self.local_rank = g, members.index(self.rank)
        for l in range(L):
            members = [n[l] for n in node_lists]
            if self.rank in members:
                self.cross_group = dist.new_group(ranks=[to_global(r) for r in members], use_local_synchronization=True)
        self.local_world, self.hier = L, True

    def _grad_alloc(self, numel, dtype, device):
        sl = self.pool.alloc(numel, dtype)
        self.slices[dtype] = sl
        return sl.tensor

    def _plan(self):
        self.entries = list(self.flat.entries())
        self.buckets = plan_buckets(self.flat, self.bucket_cap)
        has_mc = self.pool.has_multicast if self.pool is not None else False
        for b in self.buckets:
            esz = 2 if b.dtype in (torch.bfloat16, torch.float16) else 4
            b.algo = choose_algo(b.numel * esz, self.local_world if self.hier else self.world, has_mc, self.algo_pref) \
                if self.use_symm else ("nccl" if self.world > 1 else "none")
        self.bucket_of = {}
        for bi, b in enumerate(self.buckets):
            for eid in b.entry_ids:
                self.bucket_of[eid] = bi
        self._plan_bucket_optimizer()
        self._reset_pending()

    # ------------------------------------------------------------------ optimizer inside the bucket hook
    def attach_optimizer(self, opt, fused: Optional[bool] = None):
        """Let the engine run ``opt`` (a ``FlatSGDMomentum`` on this engine's flat buffers) bucket by bucket: inside
        the reduction kernel on > 1 rank, right behind the bucket's last gradient on one.  ``FlatLARS`` /
        ``FlatLAMB`` run bucket by bucket on one rank only (``step_range``).  ``fused=None`` follows
        ``EDL_FUSED_OPT`` (default on).  Not used with loss scaling, clipping (both need every gradient before any
        update), the hierarchical or library reduction paths, or weight-decay masks on a single rank."""
        self.opt = opt
        if fused is None:
            fused = os.environ.get("EDL_FUSED_OPT", "1") == "1"
        self._want_bucket_opt = bool(fused)
        opt.skip_dtype = self._opt_skips
        self._plan_bucket_optimizer()

    def _opt_skips(self, dtype) -> bool:
        """Asked by ``opt.step()``: was this dtype group already updated by the bucket kernels of this step?"""
        return self.bucket_opt and self.enabled and dtype in self._fused_dtypes

    def _plan_bucket_optimizer(self):
        self._fused_dtypes = set()
        was_sharded = self.state_sharded
        self.bucket_opt = False
        opt = self.opt
        # per-tensor-norm optimizers (LARS, LAMB: ``step_range``) ride along on ONE rank only: a bucket holds whole
        # tensors, so their update per bucket is exact; the fused multi-rank kernel is SGD-momentum's
        layerwise = hasattr(opt, "step_range")
        ok = (opt is not None and getattr(self, "_want_bucket_opt", False) and self.device.type == "cuda"
              and (type(opt).__name__ == "FlatSGDMomentum" or (layerwise and self.world == 1))
              and opt.found_inf_is_comm_error()
              and opt.grad_scale_t is None and self.clip_norm is None and self.found_inf is None
              and not self.hier and (self.world == 1 or self.use_symm))
        if ok:
            for dt, g in self.flat.groups.items():
                # > 1 rank: bf16 groups with fp32 masters (the kernel stores bf16 parameters into every rank's
                # shadow); 1 rank: any group (plain per-bucket optimizer launches)
                if self.world > 1 and not (dt == torch.bfloat16 and g.master is not None):
                    continue
                if self.world > 1 and any(b.algo not in ("twoshot", "multimem") for b in self.buckets if b.dtype == dt):
                    continue
                self._fused_dtypes.add(dt)
            self.bucket_opt = bool(self._fused_dtypes)
        for b in self.buckets:
            b.fused_opt = self.bucket_opt and b.dtype in self._fused_dtypes
        if layerwise and self.bucket_opt:
            # chunk tables of every bucket, uploaded now: never inside the captured step
            opt.plan_ranges([(b.dtype, b.start, b.numel) for b in self.buckets if b.fused_opt])
        if self.bucket_opt and self.world > 1:
            if not self.param_slices:
                self.flat.rebind_params(self._param_alloc, dtypes=self._fused_dtypes)
            self.state_sharded = True
        elif was_sharded:
            self.state_sharded = False

    def _param_alloc(self, numel, dtype, device):
        sl = self.pool.alloc(numel, dtype)
        self.param_slices[dtype] = sl
        return sl.tensor

    def _reset_pending(self):
        for b in self.buckets:
            b.pending = len(b.entry_ids)
            b.launched = False
        self._next = 0
        self._works = []
        self._seen = [False] * len(self.entries)

    def _install_hooks(self):
        self._hook_handles = []
        for eid, (g, e) in enumerate(self.entries):
            cb = self._make_ready(eid)
            e.param._edl_grad_ready = cb
            self._hook_handles.append(
                e.param.register_post_accumulate_grad_hook(lambda p, _cb=cb: _cb()))

    def detach(self):
        """Remove this engine's autograd hooks (another engine is taking over the module)."""
        for h in getattr(self, "_hook_handles", []):
            h.remove()
        self._hook_handles = []

    def _make_ready(self, eid) -> Callable[[], None]:
        def ready():
            # idempotent per step: a parameter may be reported both by a fused op writing into its
            # gradient sink and by autograd's post-accumulate hook
            if self._seen[eid]:
                return
            self._seen[eid] = True
            b = self.buckets[self.bucket_of[eid]]
            b.pending -= 1
            if b.pending == 0 and self.overlap:
                self._launch_ready()
        return ready

    # ------------------------------------------------------------------ launching
    def _launch_ready(self):
        while self._next < len(self.buckets) and self.buckets[self._next].pending <= 0:
            self._launch(self.buckets[self._next])
            self._next += 1

    def _timeout(self) -> float:
        return self.warm_timeout_s if self.warming else self.timeout_s

    def _join_producers(self):
        """The bucket's gradients were written on the main stream (BN, pools, ...) and on the weight-gradient
        stream: whatever consumes them on the communication stream waits for both."""
        for st in {torch.cuda.current_stream(self.device), self._main_stream,
                   self.wgrad_stream if self.overlap_wgrad else None,
                   self.wgrad_stream2 if self.overlap_wgrad else None}:
            if st is not None and st != self.comm_stream:
                ev = torch.cuda.Event()
                ev.record(st)
                self.comm_stream.wait_event(ev)
        self._comm_used = True

    def _bucket_optimizer_local(self, b: Bucket, g):
        """One rank: the optimizer of this bucket right behind its last gradient, on the side stream, while the
        rest of backward still runs (the separate whole-model optimizer pass at the end of the step disappears)."""
        from ..ops import native, count_launch

        opt = self.opt
        self._join_producers()
        if hasattr(opt, "step_range"):                 # LARS / LAMB: norm pass + update pass over the bucket
            with torch.cuda.stream(self.comm_stream):
                opt.step_range(b.dtype, b.start, b.numel)
            self.last_algos.append(("local_" + type(opt).__name__.lower(), b.numel * g.grad.element_size(), True))
            return
        st = opt.state[b.dtype]
        lo, hi = b.start, b.start + b.numel
        master = g.master if g.master is not None else g.param
        lp = g.param[lo:hi] if g.master is not None else None
        with torch.cuda.stream(self.comm_stream):
            native().sgd_momentum(lp, master[lo:hi], st["mom"][lo:hi], g.grad[lo:hi],
                                  st["wd_mask"][lo:hi] if st["wd_mask"] is not None else None, opt.lr_t, None,
                                  opt.found_inf_t, opt.momentum, opt.weight_decay, opt.nesterov)
        count_launch()
        self.last_algos.append(("local_sgd", b.numel * g.grad.element_size(), True))

    def _launch(self, b: Bucket):
        if b.launched or not self.enabled:
            b.launched = True
            return
        b.launched = True
        g = self.flat.groups[b.dtype]
        if self.world <= 1:
            if b.fused_opt:
                self._bucket_optimizer_local(b, g)
            return
        scale = 1.0 / self.world if self.average else 1.0
        if self.hier:
            return self._launch_hier(b, g, scale)
        if b.algo in ("twoshot", "multimem"):
            from ..ops import native, count_launch

            sl = self.slices[b.dtype]
            esz = g.grad.element_size()
            off = b.start * esz
            self._join_producers()
            with torch.cuda.stream(self.comm_stream):
                if b.fused_opt:
                    opt, st, ps = self.opt, self.opt.state[b.dtype], self.param_slices[b.dtype]
                    lo, hi = b.start, b.start + b.numel
                    self.state_complete = False
                    native().allreduce_sgd(
                        [p + off for p in sl.data_ptrs], sl.sig_ptrs, (sl.mc_ptr + off) if sl.mc_ptr else 0,
                        [p + off for p in ps.data_ptrs], (ps.mc_ptr + off) if ps.mc_ptr else 0, self.rank,
                        g.master[lo:hi], st["mom"][lo:hi], st["wd_mask"][lo:hi] if st["wd_mask"] is not None else None,
                        opt.lr_t, scale, None, self.sqnorm, opt.found_inf_t, opt.momentum, opt.weight_decay,
                        opt.nesterov, b.algo == "multimem", self.comm_blocks, self._timeout())
                else:
                    native().allreduce_twoshot(
                        [p + off for p in sl.data_ptrs], sl.sig_ptrs, (sl.mc_ptr + off) if sl.mc_ptr else 0,
                        self.rank, g.grad, b.numel, scale, self.found_inf, self.sqnorm,
                        b.algo == "multimem", self.comm_blocks, self._timeout())
            count_launch()
            self.comm_launches += 1
            self.last_algos.append((b.algo + ("+sgd" if b.fused_opt else ""), b.numel * esz, b.fused_opt))
        else:  # nccl / gloo baseline path
            self.last_algos.append((self.backend, b.numel * g.grad.element_size(), False))
            view = g.grad[b.start:b.start + b.numel]
            if self.device.type == "cuda":
                w = dist.all_reduce(view, group=self.group, async_op=True)
                self._works.append((w, view, scale))
            else:
                dist.all_reduce(view, group=self.group)
                if self.average:
                    view.mul_(scale)

    def _local_allreduce(self, b: Bucket, g, scale: float, final: bool):
        """Sum (x scale) of the bucket over the ranks of this host: our kernel over peer memory, or the library on CPU."""
        view = g.grad[b.start:b.start + b.numel]
        if self.local_world <= 1:
            if scale != 1.0:
                view.mul_(scale)
            return
        if self.use_symm:
            from ..ops import native, count_launch

            sl = self.slices[b.dtype]
            off = b.start * g.grad.element_size()
            native().allreduce_twoshot(
                [p + off for p in sl.data_ptrs], sl.sig_ptrs, (sl.mc_ptr + off) if sl.mc_ptr else 0,
                self.local_rank, g.grad, b.numel, scale, self.found_inf if final else None,
                self.sqnorm if final else None, b.algo == "multimem", self.comm_blocks, self.timeout_s)
            count_launch()
            self.comm_launches += 1
        else:
            dist.all_reduce(view, group=self.local_group)
            if scale != 1.0:
                view.mul_(scale)

    def _launch_hier(self, b: Bucket, g, scale: float):
        """Two-level all-reduce of one bucket: (1) sum inside the host, (2) rank l of every host all-reduces slice l
        across hosts (1/L of the bucket per NIC), (3) the slices are put back together inside the host by a second
        local sum over buffers that are zero outside the owned slice, with the 1/world scale and the finite check."""
        L = self.local_world
        per = -(-b.numel // L)
        per = -(-per // 8) * 8                                  # slices stay 16-byte aligned
        lo = min(b.numel, self.local_rank * per)
        hi = min(b.numel, lo + per)
        view = g.grad[b.start:b.start + b.numel]
        cuda = self.device.type == "cuda"
        if cuda:
            for st in {torch.cuda.current_stream(self.device), self._main_stream,
                       self.wgrad_stream if self.overlap_wgrad else None,
                       self.wgrad_stream2 if self.overlap_wgrad else None}:
                if st is not None and st != self.comm_stream:
                    ev = torch.cuda.Event()
                    ev.record(st)
                    self.comm_stream.wait_event(ev)
            self._comm_used = True
        ctx = torch.cuda.stream(self.comm_stream) if cuda else _NullCtx()
        with ctx:
            self._local_allreduce(b, g, 1.0, final=False)
            if hi > lo:
                dist.all_reduce(view[lo:hi], group=self.cross_group)
            if L > 1:
                if lo > 0:
                    view[:lo].zero_()
                if hi < b.numel:
                    view[hi:].zero_()
            self._local_allreduce(b, g, scale, final=True)

    def finish(self):
        """Call after ``backward()``: flush buckets whose parameters received no gradient, then make
        the compute stream wait for the communication stream."""
        for b in self.buckets:
            b.pending = 0
        self._launch_ready()
        if self.clip_norm is not None and self.enabled and self.device.type == "cuda":
            self._launch_clip()
        if self.device.type == "cuda" and (self.world > 1 or self.overlap_wgrad or self._comm_used):
            if self.use_symm or self.overlap_wgrad or self.hier or self._comm_used:
                cur = torch.cuda.current_stream(self.device)
                # only streams that took part in this step (a stream without forked work is not part
                # of a CUDA-graph capture and must not be joined into it)
                if self._comm_used:
                    cur.wait_stream(self.comm_stream)
                if self.overlap_wgrad:
                    cur.wait_stream(self.wgrad_stream)
                    if self.wgrad_stream2 is not None:
                        cur.wait_stream(self.wgrad_stream2)
                from ..ops import gemm as _gemm
                _gemm.release_wgrad_keepalive()
            for w, view, scale in self._works:
                w.wait()
                if self.average:
                    view.mul_(scale)
        if self.clip_norm is not None and self.enabled and self.device.type != "cuda":
            self._clip_cpu()
        if self.found_inf is not None and not (self.use_symm and self.world > 1):
            # the fused all-reduce epilogue raises the flag itself; without it (one rank, NCCL / gloo
            # path) the gradients are scanned here.  Summed gradients carry every rank's inf/nan, so
            # all ranks agree without another collective.
            for g in self.flat.groups.values():
                bad = (~torch.isfinite(g.grad).all()).to(torch.int32).view(1)
                self.found_inf.copy_(torch.maximum(self.found_inf, bad))
        self._reset_pending()

    # ------------------------------------------------------------------ global-norm clipping (SURVEY K9)
    def _launch_clip(self):
        """After the last bucket: turn the squared-norm partials into the clip factor the optimizer kernel multiplies
        into the gradients.  Symmetric path: every rank's bucket kernels summed g^2 over the slices THAT RANK
        reduced, so the global norm is the sum over ranks (one scalar all-gather kernel); otherwise every rank holds
        the complete reduced gradient and one streaming reduction gives the norm."""
        from ..ops import native, count_launch

        C = native()
        symm = self.use_symm and self.world > 1 and not self.hier and any(
            b.algo in ("twoshot", "multimem") for b in self.buckets)
        if symm:
            self._comm_used = True
            with torch.cuda.stream(self.comm_stream):
                # groups that did not go through our kernels (none today) would be added here
                sl = max(self.slices.values(), key=lambda x: x.tensor.numel())
                if getattr(self, "_norm_parts", None) is None or self._norm_parts.numel() != self.world:
                    self._norm_parts = torch.zeros(self.world, device=self.device, dtype=torch.float32)
                C.comm_allgather_scalars(sl.data_ptrs, sl.sig_ptrs, self.rank, self.sqnorm, self._norm_parts,
                                         self.timeout_s)
                C.clip_scale(self._norm_parts, self.world, 1, self.clip_norm, self.clip_scale_t, self.grad_norm_t)
            count_launch(2)
        else:
            # one rank, or the library / hierarchical paths: join the producers / async works first
            for w, view, scale in self._works:
                w.wait()
                if self.average:
                    view.mul_(scale)
            self._works = []
            if self.overlap_wgrad or self._comm_used:
                cur = torch.cuda.current_stream(self.device)
                if self._comm_used:
                    cur.wait_stream(self.comm_stream)
                if self.overlap_wgrad:
                    cur.wait_stream(self.wgrad_stream)
                    if self.wgrad_stream2 is not None:
                        cur.wait_stream(self.wgrad_stream2)
            self.sqnorm.zero_()
            for g in self.flat.groups.values():
                C.grad_sqnorm(g.grad, self.sqnorm)
            C.clip_scale(self.sqnorm, 1, 1, self.clip_norm, self.clip_scale_t, self.grad_norm_t)
            count_launch(1 + len(self.flat.groups))
        if self.opt is not None:
            self.opt.set_grad_scale(self.clip_scale_t)

    def _clip_cpu(self):
        total = sum(float(g.grad.float().pow(2).sum()) for g in self.flat.groups.values()) ** 0.5
        if total > self.clip_norm:
            for g in self.flat.groups.values():
                g.grad.mul_(self.clip_norm / (total + 1e-6))
        self.last_grad_norm = total

    # ------------------------------------------------------------------ sharded optimizer state
    def owned_ranges(self, dtype, rank: Optional[int] = None, world: Optional[int] = None):
        """Element ranges of the dtype group's flat buffers whose master weights / momentum THIS rank keeps
        current in fused mode (slice ``rank`` of every bucket, csrc/allreduce.cu slice rule)."""
        rank = self.rank if rank is None else rank
        world = self.world if world is None else world
        out = []
        for b in self.buckets:
            if b.dtype != dtype or not b.fused_opt:
                continue
            nvec = b.numel // 8
            cap = -(-nvec // world)
            lo = min(nvec, cap * rank)
            hi = min(nvec, lo + cap)
            if hi > lo:
                out.append((b.start + lo * 8, b.start + hi * 8))
        return out

    @torch.no_grad()
    def consolidate_optimizer_state(self):
        """Collective over the current stage: bring master weights and momentum of the fused groups up to date on
        EVERY rank (each rank only maintained its slices).  Called before a checkpoint is written and before a
        planned stage change.  Exact: every element is owned by exactly one rank, the others contribute zeros to an
        fp32 sum that rides on the two-shot kernel through the (idle) gradient slab."""
        if not (self.state_sharded and self.world > 1):
            return
        from ..ops import native, count_launch

        torch.cuda.synchronize(self.device)
        for dt in self._fused_dtypes:
            g = self.flat.groups[dt]
            sl = self.slices[dt]
            stage = sl.tensor.view(torch.uint8)
            cap = stage.numel() // 4 // 1024 * 1024                       # fp32 elements per round
            fstage = stage[:cap * 4].view(torch.float32)
            own = self.owned_ranges(dt)
            for t in (g.master, self.opt.state[dt]["mom"]):
                for off in range(0, t.numel(), cap):
                    n = min(cap, t.numel() - off)
                    n8 = -(-n // 4) * 4
                    fstage[:n8].zero_()
                    for lo, hi in own:
                        a, b_ = max(lo, off), min(hi, off + n)
                        if b_ > a:
                            fstage[a - off:b_ - off].copy_(t[a:b_])
                    native().allreduce_twoshot(sl.data_ptrs, sl.sig_ptrs, 0, self.rank, fstage, n8, 1.0, None, None,
                                               False, self.comm_blocks, self.timeout_s)
                    count_launch()
                    t[off:off + n].copy_(fstage[:n])
            sl.tensor.zero_()
        torch.cuda.synchronize(self.device)
        self.state_complete = True

    @torch.no_grad()
    def localize_optimizer_state(self):
        """After a FAILED collective (a peer died, its slices are gone): make this rank's optimizer state complete
        without any communication -- master weights outside the owned slices are re-derived from the bf16
        parameters (those are replicated and current as of the last good step), momentum there keeps its last
        consolidated value.  The elastic recovery then takes the root's state for everybody."""
        if not self.state_sharded:
            return
        for dt in self._fused_dtypes:
            g = self.flat.groups[dt]
            keep = torch.zeros(g.numel, dtype=torch.bool, device=self.device)
            for lo, hi in self.owned_ranges(dt):
                keep[lo:hi] = True
            g.master.copy_(torch.where(keep, g.master, g.param.float()))
        self.state_complete = True

    # ------------------------------------------------------------------ user-facing
    def __call__(self, *a, **kw):
        return self.module(*a, **kw)

    def zero_grad(self):
        if self.device.type == "cuda":
            from ..ops import gemm as _gemm
            # the zeroing memsets run on the main stream: the side stream must not start writing
            # gradients before them
            self.flat.zero_grad()
            self._main_stream = torch.cuda.current_stream(self.device)
            self._comm_used = False
            if self.overlap_wgrad:
                self.wgrad_stream.wait_stream(self._main_stream)
                if self.wgrad_stream2 is not None:
                    self.wgrad_stream2.wait_stream(self._main_stream)
                _gemm.set_wgrad_stream([self.wgrad_stream, self.wgrad_stream2])
            else:
                _gemm.set_wgrad_stream(None)
            if self.found_inf is not None:
                self.found_inf.zero_()
            if self.sqnorm is not None:
                self.sqnorm.zero_()
            self.last_algos = []
            return
        self.flat.zero_grad()
        if self.found_inf is not None:
            self.found_inf.zero_()
        if self.sqnorm is not None:
            self.sqnorm.zero_()

    def check_comm_error(self) -> int:
        return self.pool.check_error() if self.pool is not None else 0

    def agree(self, flag: float):
        """(max of ``flag`` over the ranks, comm error word).  The agreement ``ElasticContext.poll`` needs, routed
        through our own scalar all-gather kernel when the ranks share symmetric memory: unlike a library
        all-reduce it has the ``globaltimer`` timeout, so a DEAD peer shows up as a non-zero error word a few
        seconds later instead of a hung process -- the trigger for ``ElasticContext.recover()`` on GPUs."""
        if self.world <= 1:
            return float(flag), 0
        if self.use_symm and self.slices and not self.hier:
            from ..ops import native, count_launch

            sl = max(self.slices.values(), key=lambda x: x.tensor.numel())
            inp = torch.tensor([float(flag), 0.0], device=self.device, dtype=torch.float32)
            out = torch.zeros(self.world * 2, device=self.device, dtype=torch.float32)
            native().comm_allgather_scalars(sl.data_ptrs, sl.sig_ptrs, self.rank, inp, out, min(self.timeout_s, 10.0))
            count_launch()
            err = self.check_comm_error()                     # host sync: the kernel above has finished
            return float(out.view(self.world, 2)[:, 0].max().item()), err
        t = torch.tensor([float(flag)], device=self.device if self.device.type == "cuda" else "cpu")
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return float(t.item()), 0

    def allreduce_scalars(self, t: torch.Tensor) -> torch.Tensor:
        """Sum of a tiny fp32 tensor (<= 8 values: evaluation counters, flags) over the ranks; our scalar all-gather
        kernel when the ranks share symmetric memory, else the library."""
        if self.world <= 1:
            return t
        if self.use_symm and self.slices and not self.hier and t.numel() <= 8 and t.is_cuda:
            from ..ops import native, count_launch

            sl = max(self.slices.values(), key=lambda x: x.tensor.numel())
            inp = t.detach().to(torch.float32).contiguous().view(-1)
            out = torch.zeros(self.world * inp.numel(), device=self.device, dtype=torch.float32)
            native().comm_allgather_scalars(sl.data_ptrs, sl.sig_ptrs, self.rank, inp, out, min(self.timeout_s, 30.0))
            count_launch()
            return out.view(self.world, -1).sum(0).view_as(t).to(t.dtype)
        t = t.clone()
        dist.all_reduce(t, group=self.group)
        return t

    def rebuild(self, group: Optional[dist.ProcessGroup] = None, fabric=None):
        """Elastic stage change: new group (or fabric) => new symmetric slab, new bucket plan.  Parameters,
        master weights and optimizer state stay where they are (no process restart).  With a sharded optimizer
        state call ``consolidate_optimizer_state()`` (planned change, old stage still intact) or
        ``localize_optimizer_state()`` (a peer died) BEFORE this."""
        if self.state_sharded and not self.state_complete:
            raise RuntimeError("the optimizer state is sharded across the ranks of the old stage: call "
                               "consolidate_optimizer_state() (planned change, collective over the OLD stage) or "
                               "localize_optimizer_state() (a peer died) before rebuild()")
        for h in self._hook_handles:
            h.remove()
        old_pool = self.pool
        had_param_shadow = bool(self.param_slices)
        self.slices = {}
        self.param_slices = {}
        self.state_sharded = False
        self._norm_parts = None
        self._bind_group(group, fabric)
        if self.pool is not None:
            self.flat.rebind_grads(self._grad_alloc)
        else:
            self.flat.rebind_grads(lambda n, dt, dev: torch.zeros(n, dtype=dt, device=dev))
        self._plan()            # re-homes the bf16 parameters into the new slab when the fused optimizer is on
        if had_param_shadow and not self.param_slices:
            # the fused path is off in the new stage (one rank left, library path): parameters leave the old slab
            self.flat.rebind_params(lambda n, dt, dev: torch.empty(n, dtype=dt, device=dev),
                                    dtypes=[dt for dt, g in self.flat.groups.items() if g.master is not None])
        del old_pool
        self._install_hooks()

    def barrier(self):
        """Host-side barrier of the stage's ranks (store barrier of the pool, else the library's)."""
        if self.world <= 1:
            return
        if self.pool is not None and not self.hier:
            self.pool.barrier()
        else:
            dist.barrier(self.group)

    @torch.no_grad()
    def broadcast_parameters(self, root: int = 0):
        """Bring every rank's parameters (and fp32 masters) in sync with ``root`` -- used after a
        join so that the newcomer does not need to read the checkpoint from the file system."""
        if self.world <= 1:
            return
        for g in self.flat.groups.values():
            src = g.master if g.master is not None else g.param
            if self.use_symm and not self.hier:
                self._broadcast_tensor(src, root)
                if g.master is not None:
                    g.param.copy_(g.master.to(g.param.dtype))
            else:
                dist.broadcast(src, src=dist.get_global_rank(self.group, root) if self.group else root,
                               group=self.group)
                if g.master is not None:
                    g.param.copy_(g.master.to(g.param.dtype))

    @torch.no_grad()
    def broadcast_tensor(self, t: torch.Tensor, root: int = 0):
        """Broadcast any contiguous device tensor (e.g. optimizer state) from ``root`` of the current group."""
        if self.world <= 1:
            return
        if self.use_symm and not self.hier:
            self._broadcast_tensor(t, root)
        else:
            dist.broadcast(t, src=dist.get_global_rank(self.group, root) if self.group else root, group=self.group)

    def _broadcast_tensor(self, t: torch.Tensor, root: int):
        """Chunked broadcast through the gradient slab (it is idle outside backward)."""
        from ..ops import native, count_launch

        flat = t.view(-1).view(torch.uint8)
        sl = max(self.slices.values(), key=lambda s: s.tensor.numel() * s.tensor.element_size())
        stage = sl.tensor.view(torch.uint8)
        cap = stage.numel() // 16 * 16
        for off in range(0, flat.numel(), cap):
            n = min(cap, flat.numel() - off)
            if self.rank == root:
                stage[:n].copy_(flat[off:off + n])
            native().comm_broadcast(sl.data_ptrs, sl.sig_ptrs, self.rank, root, n, self.comm_blocks,
                                    self.timeout_s, sl.tensor)
            count_launch()
            if self.rank != root:
                flat[off:off + n].copy_(stage[:n])
        sl.tensor.zero_()
