#!/usr/bin/env python
"""Flagship benchmark: ResNet50_vd student training throughput (img/s, whole job), bf16,
per-GPU batch 32 (= the reference's "total batch 256 on 8 GPUs", README.md:81-83), synthetic
ImageNet-shaped data, random-init weights.

    python bench.py --gpus 1 --steps 50 --warmup 5
    python bench.py --gpus 1 --steps 50 --warmup 5 --dump-outputs DIR  # + one step's outputs as DIR/*.npy
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...   # the unmodified reference (unavailable offline: see DESIGN.md)
    python bench.py --impl torch ...       # our own PyTorch-DDP + cuDNN + NCCL comparator (baseline/)

Prints ONE JSON line on rank 0.  `value` is device-timed (CUDA events, max over ranks) with inputs
resident on the device; `e2e` runs the same steps through the public `StudentTrainer.step()` API
with a pinned-host -> device copy of every batch and a device -> host read of a step's loss each step.  On N > 1 GPUs the
line also carries what the all-reduce path really launched (`allreduce`), a cross-check of our kernel against NCCL,
`exposed_comm_ms`, the in-place `rescale` recovery times and the `distill` service throughput (BASELINE.json's metric).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

BASELINE_IMG_S = 1828.0  # BASELINE.md P1: ResNet50_vd pure train, 8xV100, total batch 256


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="edl", choices=["edl", "reference", "torch"])
    ap.add_argument("--batch-per-gpu", type=int, default=32)
    ap.add_argument("--mode", default="pure", choices=["pure", "distill"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--conv-impl", default="auto", choices=["auto", "cudnn"])
    ap.add_argument("--algo", default="auto")
    ap.add_argument("--bucket-mb", type=float, default=16.0)
    ap.add_argument("--comm-blocks", type=int, default=32)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--layers", type=int, default=50)
    ap.add_argument("--kineto", type=str, default="", help="write a torch.profiler per-kernel table of 5 replayed steps here")
    ap.add_argument("--teacher", default="resnext101_32x16d", choices=["resnext101_32x16d", "resnext50_32x4d"])
    ap.add_argument("--teacher-fp8", action="store_true", help="distill mode: e4m3 tcgen05 GEMMs for the teacher's 1x1 convs")
    ap.add_argument("--no-fused-bn", action="store_true", help="A/B: disable the SM-resident fused BN kernels")
    ap.add_argument("--no-stream-bn", action="store_true", help="A/B: disable the cp.async.bulk BN kernels")
    ap.add_argument("--teacher-fuse-res", action="store_true",
                    help="A/B (experimental, distill mode): residual add of the teacher's blocks inside the GEMM epilogue")
    ap.add_argument("--fuse-bn-bwd", type=int, default=0, choices=[0, 1, 2],
                    help="A/B (experimental): BatchNorm-backward reduction inside the dgrad epilogues; 1 = shuffle "
                         "version of round 1, 2 = column-loop version (EDL_FUSE_BN_BWD=1 + EDL_BNR_MODE)")
    ap.add_argument("--own-stem1", action="store_true", help="A/B (experimental): direct kernel for the first stem convolution")
    ap.add_argument("--conv3-s2", action="store_true",
                    help="A/B (experimental): stride-2 3x3 forward convolutions on the tcgen05 kernel (student and teacher)")
    ap.add_argument("--pdl", action="store_true", help="A/B (experimental): programmatic dependent launch of the hot kernels")
    ap.add_argument("--own-wgrad3", action="store_true", help="A/B (experimental): tcgen05 3x3 weight-gradient kernel")
    ap.add_argument("--no-library", action="store_true",
                    help="every convolution of the student on our own kernels (3x3 wgrad v2, stride-2 backward, pixel-pair "
                         "stem convolutions): no cuDNN / cuBLAS kernel in the step; `library_fallbacks` must come out empty")
    ap.add_argument("--no-fused-opt", action="store_true",
                    help="A/B: plain all-reduce kernels + one optimizer pass instead of the fused reduce-scatter -> "
                         "SGD -> all-gather buckets")
    ap.add_argument("--clip-norm", type=float, default=0.0,
                    help="global-norm gradient clipping (0 = off, the reference's config)")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the extra metric terms of BASELINE.json at N > 1 (exposed comm, rescale recovery, "
                         "distill service)")
    ap.add_argument("--extras-budget-s", type=float, default=240.0,
                    help="wall-clock budget of the extra sections; when it runs out the headline line is printed without them")
    ap.add_argument("--distill-steps", type=int, default=40)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed runs, reset the model to its seeded initial state, run the timed step (the "
                         "captured graph) once on a seeded batch and write its loss, updated parameters and BatchNorm "
                         "running statistics as DIR/<name>.npy, so that two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.mode != "pure" or args.impl != "edl" or args.gpus != 1):
        ap.error("--dump-outputs supports --mode pure --impl edl --gpus 1 only")
    return args


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []          # (host arrival time, csv line)
        self.windows = []        # [t_begin, t_end] of the timed regions (host clock)

    def begin(self):
        self.windows.append([time.perf_counter(), None])

    def end(self):
        self.windows[-1][1] = time.perf_counter()

    def in_window_samples(self) -> int:
        return sum(1 for t, _ in list(self.lines) if any(a <= t <= (b or 1e30) for a, b in self.windows))

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], 0, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        # nvidia-smi was started before the warm-up (its start-up takes longer than a short timed region);
        # only samples that arrived inside a timed window count
        for t, ln in list(self.lines):
            if self.windows and not any(a <= t <= (b or 1e30) for a, b in self.windows):
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = max(smax, float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax or None,
                "power_w_max": max(power) if power else None, "samples": len(sm),
                "reasons": sorted(reasons)}


def reference_arm(args):
    """The reference cannot run offline: record why (details in DESIGN.md)."""
    why = ("reference needs paddlepaddle-gpu==1.8 + paddle-serving + etcd3 + grpc_tools codegen; none are "
           "in the image/wheelhouse (pure-Python `edl` wheel installs into baseline/_ref but "
           "`import edl.utils.launcher` fails on missing *_pb2 / paddle)")
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


def distill_main(args, world, rank, dev):
    out = distill_run(args, world, rank, dev, args.steps, with_clocks=True)
    import torch.distributed as dist

    if rank == 0:
        print(json.dumps(out))
    dist.barrier()
    dist.destroy_process_group()
    return 0


def distill_run(args, world, rank, dev, steps, with_clocks=False):
    """Distill-service mode: ranks [0, N/2) are students, [N/2, N) teachers (ResNeXt101_32x16d); the
    images go student -> teacher and the logits teacher -> student through NVSwitch peer memory.
    Returns the result record (complete on rank 0)."""
    import torch
    import torch.distributed as dist

    import edl_b200.ops as ops
    from edl_b200.distill.device_feed import DeviceDistillLink, pool_bytes_needed
    from edl_b200.distill.device_trainer import DistillStudentTrainer, TeacherWorker, split_roles
    from edl_b200.models import ResNetVd, to_train_dtype
    from edl_b200.models.resnext import ResNeXt101_32x16d, ResNeXt50_32x4d, to_inference_dtype
    from edl_b200.parallel.symm import SymmetricPool

    B = args.batch_per_gpu
    n_students, students, teachers = split_roles(world)
    sgroup = dist.new_group(ranks=students)
    dist.new_group(ranks=teachers)
    pool = SymmetricPool(pool_bytes_needed(B, slots=2) + (8 << 20), device=dev)
    is_student = rank < n_students
    peer = rank + n_students if is_student else rank - n_students
    link = DeviceDistillLink(pool, peer, "student" if is_student else "teacher", B, slots=2, timeout_s=120.0)
    if is_student:
        model = to_train_dtype(ResNetVd(args.layers, impl=args.conv_impl), torch.bfloat16, dev).train()
        trainer = DistillStudentTrainer(model, B, link, lr=0.1 * B * n_students / 256.0, use_graph=not args.no_graph,
                                        group=sgroup, bucket_cap_mb=args.bucket_mb,
                                        comm_blocks=args.comm_blocks, algo=args.algo)
    else:
        tm = ResNeXt50_32x4d() if args.teacher == "resnext50_32x4d" else ResNeXt101_32x16d()
        tm = to_inference_dtype(tm, torch.bfloat16, dev)
        if args.teacher_fp8:
            calib = torch.randn(B, 3, 224, 224, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
            tm.enable_fp8(calib)
        worker = TeacherWorker(tm, link, use_graph=not args.no_graph)
    pool_n = 4
    host_x = [torch.randn(B, 3, 224, 224).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).pin_memory()
              for _ in range(pool_n)] if is_student else None

    def sync_all():
        dist.barrier()
        torch.cuda.synchronize(dev)

    def run(n, e2e):
        last = 0.0
        for i in range(n):
            if is_student:
                if e2e:
                    last = float(trainer.step(host_x[i % pool_n]).item())
                else:
                    trainer.step_device()
            else:
                worker.step()
        return last

    warm = max(args.warmup, 7)      # 4 eager protocol steps + one graph capture per ring slot + one replay
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if with_clocks:
        sampler.start()
    run(warm, True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    sampler.begin()
    ops.reset_launches()
    ev0.record()
    run(steps, False)
    ev1.record()
    sync_all()
    sampler.end()
    launches = ops.launches()
    t = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())
    e2e = None
    if not args.no_e2e:
        sync_all()
        t0 = time.perf_counter()
        last = run(steps, True)
        torch.cuda.synchronize(dev)
        t = torch.tensor([(time.perf_counter() - t0) * 1e3], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
        e2e = {"value": B * n_students * steps / (e2e_ms / 1e3), "unit": "img/s", "ms_per_step": e2e_ms / steps,
               "h2d_bytes_per_step": B * 3 * 224 * 224 * 2, "d2h_bytes_per_step": 4, "last_loss": last,
               "timing": "host wall clock around K public-API steps (student: pinned H2D images + loss.item())"}
    flag = torch.tensor([1.0 if (with_clocks and sampler.proc is not None and sampler.in_window_samples() < 3) else 0.0],
                        device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)              # all ranks take the same decision: pairs step in lockstep
    if float(flag.item()) > 0.5:
        sampler.begin()
        run(60, False)
        torch.cuda.synchronize(dev)
        sampler.end()
    clocks = sampler.stop() if with_clocks else None
    err = link.check_error()
    value = B * n_students * steps / (dev_ms / 1e3)
    if True:
        return ({
            "metric": "ResNet50_vd student img/s with same-box distill service (teacher logits over NVSwitch)",
            "value": value, "unit": "img/s", "n_gpus": world, "steps": steps, "warmup": warm,
            "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": value / 1514.0, "dtype": "bf16",
            "data": "synthetic images, random-init student and teacher", "impl": "edl",
            "config": {"model": "ResNet%d_vd student + %s teacher" % (args.layers, args.teacher),
                       "students": n_students, "teachers": n_students, "batch_per_gpu": B,
                       "global_batch": B * n_students,
                       "transport": "peer_ship + GEMM->peer-ship epilogue over NVSwitch peer memory, "
                                    "student/teacher pipelined by one batch",
                       "teacher_dtype": "e4m3 1x1 convs + bf16" if args.teacher_fp8 else "bf16",
                       "teacher_fuse_res": bool(__import__("edl_b200.models.resnext", fromlist=["x"]).FUSE_RESIDUAL),
                       "conv3_s2": bool(ops.gemm.CONV3_S2), "pdl": bool(args.pdl),
                       "parallelism": "dp%d + %d teacher GPUs" % (n_students, n_students),
                       "baseline_note": "vs_baseline divides by the published 1514 img/s (8xV100 + 40xP4, BASELINE.md P3)"},
            "clocks": clocks, "gpu_launches": launches, "e2e": e2e, "link_error": err})


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    if os.environ.get("EDL_FAKE_HOST_SPLIT"):  # A/B of the hierarchical all-reduce: ranks [0, k) and [k, N) play two hosts
        os.environ["EDL_FAKE_HOST"] = "node%d" % (int(os.environ.get("RANK", "0")) // int(os.environ["EDL_FAKE_HOST_SPLIT"]))
    if args.pdl:
        os.environ["EDL_PDL"] = "1"            # read when the extension is loaded
    if args.no_library:
        for k in ("EDL_OWN_WGRAD3", "EDL_OWN_S2_BWD", "EDL_OWN_STEM23"):
            os.environ[k] = "1"                # read when edl_b200.ops.gemm is imported
    if args.own_wgrad3:
        os.environ["EDL_OWN_WGRAD3"] = "1"     # read when edl_b200.ops.gemm is imported
    if args.fuse_bn_bwd:
        os.environ["EDL_FUSE_BN_BWD"] = "1"        # read when edl_b200.ops.gemm is imported
        os.environ["EDL_BNR_MODE"] = str(args.fuse_bn_bwd)   # read when the extension is loaded
    if args.own_stem1:
        os.environ["EDL_OWN_STEM1"] = "1"          # read when edl_b200.ops.gemm is imported
    if args.conv3_s2:
        os.environ["EDL_CONV3_S2"] = "1"           # read when edl_b200.ops.gemm is imported
    if args.teacher_fuse_res:
        os.environ["EDL_TEACHER_FUSE_RES"] = "1"   # read when edl_b200.models.resnext is imported

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device", "impl": args.impl}))
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "launch with torchrun for --gpus > 1"

    torch.manual_seed(1234 + rank)
    B = args.batch_per_gpu
    if args.mode == "distill":
        return distill_main(args, world, rank, dev)
    if args.impl == "torch":
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from baseline.torch_ddp import TorchDDPTrainer

        trainer = TorchDDPTrainer(B, dev, layers=args.layers, use_graph=not args.no_graph)
        import edl_b200.ops as ops
    else:
        import edl_b200.ops as ops
        from edl_b200.models import ResNetVd, to_train_dtype
        from edl_b200.trainer import StudentTrainer

        if args.no_fused_bn:
            ops.set_fused_bn(False)
        if args.no_stream_bn:
            ops.native().bn_set_stream_kernels(False)
        model = to_train_dtype(ResNetVd(args.layers, impl=args.conv_impl), torch.bfloat16, dev)
        model.train()
        trainer = StudentTrainer(model, B, lr=0.1 * B * world / 256.0, use_graph=not args.no_graph,
                                 bucket_cap_mb=args.bucket_mb, comm_blocks=args.comm_blocks,
                                 algo=args.algo, target_kind="probs",
                                 fused_optimizer=False if args.no_fused_opt else None,
                                 clip_norm=args.clip_norm or None)
        initial = snapshot(trainer) if args.dump_outputs else None

    # synthetic host data (pinned): a small pool of distinct batches, cycled
    pool = 4
    host_x = [torch.randn(B, 3, 224, 224).to(torch.bfloat16).contiguous(
        memory_format=torch.channels_last).pin_memory() for _ in range(pool)]
    host_t = [torch.softmax(torch.randn(B, 1000) * 2.0, -1).to(torch.bfloat16).pin_memory()
              for _ in range(pool)]
    h2d_bytes = host_x[0].numel() * 2 + host_t[0].numel() * 2
    d2h_bytes = 4

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- one-off proof, before any training step: OUR all-reduce kernel on a real gradient bucket against
    #      NCCL's all-reduce of the same data (the gradient slab is idle before the first step)
    crosscheck = None
    if world > 1 and args.impl == "edl" and getattr(trainer.dp, "use_symm", False):
        crosscheck = allreduce_crosscheck(trainer.dp, dev, world)

    sampler = ClockSampler(local_rank)
    sampler.start()              # streams samples from now on; only those inside the timed windows are used
    # ---- warm-up (also captures the CUDA graph) ----
    loss = None
    for i in range(max(args.warmup, 3)):
        loss = trainer.step(host_x[i % pool], host_t[i % pool])
    loss0 = float(loss.item())

    # ---- device-timed region: K steps, inputs resident on device ----
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    sampler.begin()
    ops.reset_launches()
    ev0.record()
    for _ in range(args.steps):
        trainer.step_device()
    ev1.record()
    sync_all()
    sampler.end()
    launches = ops.launches()
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1))

    if args.kineto and rank == 0:
        # per-kernel device times inside the REAL pipelined execution (graph replays, warm caches) --
        # complements ncu, whose serialised cold-cache timings overstate small kernels
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(5):
                trainer.step_device()
            torch.cuda.synchronize(dev)
        with open(args.kineto, "w") as fh:
            fh.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=60, max_name_column_width=90))
        # timeline of ONE replayed step for tools/trace_timeline.py (stream overlap / idle-gap analysis)
        with profile(activities=[ProfilerActivity.CUDA]) as prof1:
            trainer.step_device()
            torch.cuda.synchronize(dev)
        prof1.export_chrome_trace(args.kineto + ".trace.json")
    if args.kineto and world > 1:
        for _ in range(6):                  # the other ranks keep their collectives in step with rank 0's profiled steps
            if rank != 0:
                trainer.step_device()
        torch.cuda.synchronize(dev)

    # ---- end-to-end region: the public API (`trainer.step(host images, host targets)`), every step with its
    #      pinned-host -> device input copy and a device -> host read of a step's loss.  The public default is the
    #      double-buffered feed: the loss handle of step i is read while step i+1 runs (one D2H read per step).
    e2e = None
    if not args.no_e2e:
        def e2e_loop(sync_mode):
            sync_all()
            sampler.begin()
            t0 = time.perf_counter()
            last, prev = 0.0, None
            for i in range(args.steps):
                if sync_mode:
                    last = float((trainer.step(host_x[i % pool], host_t[i % pool], sync=True) if args.impl == "edl"
                                  else trainer.step(host_x[i % pool], host_t[i % pool])).item())
                else:
                    h = trainer.step(host_x[i % pool], host_t[i % pool])
                    if prev is not None:
                        last = prev.item()
                    prev = h
            if prev is not None:
                last = prev.item()
            torch.cuda.synchronize(dev)
            ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
            sampler.end()
            return ms, last

        if hasattr(trainer, "step_pipelined"):
            for i in range(3):
                trainer.step(host_x[i % pool], host_t[i % pool]).item()
            e2e_ms, last = e2e_loop(False)
            api = ("StudentTrainer.step(images, targets) -> LossHandle (default: staged H2D on a copy stream, loss of "
                   "step i read while step i+1 runs)")
        else:
            e2e_ms, last = e2e_loop(True)
            api = "trainer.step(images, targets); loss.item()"
        e2e = {"value": B * world * args.steps / (e2e_ms / 1e3), "unit": "img/s",
               "ms_per_step": e2e_ms / args.steps, "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": d2h_bytes, "api": api,
               "timing": "host wall clock around K public-API steps, each with a pinned H2D input copy and a D2H loss "
                         "read; max over ranks", "last_loss": last}
        if hasattr(trainer, "step_pipelined"):
            s_ms, s_last = e2e_loop(True)
            e2e["sync"] = {"value": B * world * args.steps / (s_ms / 1e3), "unit": "img/s",
                           "ms_per_step": s_ms / args.steps, "last_loss": s_last,
                           "note": "step(..., sync=True) + loss.item() inside every step (host stalls the GPU)"}
    clocks_note = "samples inside the timed regions"

    def few_samples_somewhere() -> bool:      # every rank must take the same decision (collectives inside a step)
        if sampler.proc is None:              # no nvidia-smi on this box: nothing to wait for
            return False
        return max_over_ranks(1.0 if sampler.in_window_samples() < 3 else 0.0) > 0.5

    if few_samples_somewhere():
        # K steps can be shorter than nvidia-smi's 100 ms period: keep the same load running (untimed, after
        # the measurement) until a few samples exist, so that a throttled or clock-locked GPU is still caught
        sampler.begin()
        for _ in range(8):
            for _ in range(25):
                trainer.step_device()
            torch.cuda.synchronize(dev)
            if not few_samples_somewhere():
                break
        sampler.end()
        clocks_note = "timed regions + identical untimed steps right after them (timed region < sampling period)"
    clocks = sampler.stop()
    if args.dump_outputs:
        restore(trainer, initial)
        torch.manual_seed(4321)
        x = torch.randn(B, 3, 224, 224).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        t = torch.softmax(torch.randn(B, 1000) * 2.0, -1).to(torch.bfloat16)
        dump_outputs(args.dump_outputs, trainer.step(x, t, sync=True), trainer.model)
    clocks["window"] = clocks_note

    value = B * world * args.steps / (dev_ms / 1e3)
    dp = getattr(trainer, "dp", None)
    out = {
        "metric": "ResNet50_vd student train throughput (pure data-parallel, no teacher)",
        "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": value / BASELINE_IMG_S,
        "dtype": "bf16", "data": "synthetic (random 3x224x224 images, random soft labels; random-init weights)",
        "impl": args.impl,
        "config": {"model": "ResNet%d_vd" % args.layers, "global_batch": B * world,
                   "batch_per_gpu": B, "seq_len": None, "image": "3x224x224 NHWC bf16",
                   "parallelism": "dp%d" % world, "optimizer": "SGD-momentum 0.9 wd 1e-4 (fused, fp32 master)",
                   "loss": "soft-label cross-entropy (teacher-score shaped targets)",
                   "cuda_graph": not args.no_graph, "conv_impl": args.conv_impl,
                   "pdl": bool(args.pdl), "own_wgrad3": ops.gemm.OWN_WGRAD3 if args.impl == "edl" else None,
                   "conv3_s2": ops.gemm.CONV3_S2 if args.impl == "edl" else None,
                   "own_stem1": ops.gemm.OWN_STEM1 if args.impl == "edl" else None,
                   "fuse_bn_bwd": (ops.native().get_bnr_mode() if ops.gemm.FUSE_BN_BWD else 0) if args.impl == "edl" else None,
                   "clip_norm": args.clip_norm or None, "no_library": bool(args.no_library),
                   "l2": "per-step working set (~GBs of activations) >> 126 MB L2, no explicit flush",
                   "baseline_note": "vs_baseline divides by the published 8xV100 1828 img/s (BASELINE.md P1)"},
        "clocks": clocks, "gpu_launches": launches, "e2e": e2e, "loss_after_warmup": loss0,
        "library_fallbacks": ops.fallbacks() if hasattr(ops, "fallbacks") else None,
    }
    if dp is not None:
        out["allreduce"] = allreduce_report(dp, crosscheck)
        out["config"]["allreduce"] = out["allreduce"]["algos"]

    # ---- the other terms of the BASELINE.json metric, each bounded in time; the headline above never waits for them
    #      longer than --extras-budget-s (a watchdog prints it alone and exits)
    if args.impl == "edl" and world > 1 and not args.no_extras:
        def bail():
            if rank == 0:
                out["extras_error"] = "extra sections exceeded %.0f s: printed without them" % args.extras_budget_s
                print(json.dumps(out), flush=True)
            os._exit(0)

        wd = threading.Timer(args.extras_budget_s, bail)
        wd.daemon = True
        wd.start()
        for name, fn in (("exposed_comm", lambda: exposed_comm(trainer, args, dev, world, max_over_ranks, sync_all, dev_ms)),
                         ("rescale", lambda: rescale_section(trainer, args, dev, world, rank, host_x[0], host_t[0])),
                         ("distill", lambda: distill_section(args, world, rank, dev))):
            try:
                t0 = time.perf_counter()
                out[name] = fn()
                if isinstance(out[name], dict):
                    out[name]["section_s"] = round(time.perf_counter() - t0, 2)
            except Exception as exc:  # noqa: BLE001 - an extra term must not cost the headline
                out[name] = {"error": repr(exc)[:400]}
                break                  # the ranks may no longer be in step: stop here
        wd.cancel()
        if isinstance(out.get("exposed_comm"), dict) and "exposed_comm_ms" in out["exposed_comm"]:
            out["exposed_comm_ms"] = out["exposed_comm"]["exposed_comm_ms"]
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


DUMP_PARAM_SAMPLE = 4 << 20  # float32 elements (16 MB): ResNet50_vd has 25.6 M parameters


def snapshot(trainer):
    """Copies of everything a training step changes: parameters, BatchNorm buffers, fp32 masters, momentum."""
    model = {k: v.detach().clone() for k, v in trainer.model.state_dict().items()}
    opt = trainer.opt.state_dict()
    return model, {"lr": opt["lr"], "momentum": {k: v.clone() for k, v in opt["momentum"].items()},
                   "master": {k: v.clone() for k, v in opt["master"].items()}}


def restore(trainer, state):
    """Copies ``snapshot()`` back in place, so that the captured step graph still points at the live tensors."""
    import torch

    with torch.no_grad():
        trainer.model.load_state_dict(state[0])
        trainer.opt.load_state_dict(state[1])


def dump_outputs(out_dir, loss, model):
    """What one training step hands its caller: the loss and the model it updated in place.  Writes ``loss.npy``,
    ``params.npy`` (all parameters in ``named_parameters()`` order, or a fixed seeded sample of
    ``DUMP_PARAM_SAMPLE`` of them, sorted by position) and ``bn_running_stats.npy`` (every floating-point buffer),
    all float32."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    params = torch.cat([p.detach().float().flatten() for _, p in model.named_parameters()]).cpu().numpy()
    if params.size > DUMP_PARAM_SAMPLE:
        params = params[np.sort(np.random.default_rng(0).choice(params.size, DUMP_PARAM_SAMPLE, replace=False))]
    bufs = [b.detach().float().flatten() for _, b in model.named_buffers() if b.is_floating_point()]
    arrays = {"loss": loss.detach().float().reshape(1).cpu().numpy(), "params": params,
              "bn_running_stats": torch.cat(bufs).cpu().numpy() if bufs else np.zeros(0, np.float32)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def allreduce_crosscheck(dp, dev, world):
    """max |own all-reduce - NCCL all-reduce| on the largest real gradient bucket, filled with random data."""
    import torch
    import torch.distributed as dist

    from edl_b200.ops import native

    b = max(dp.buckets, key=lambda bb: bb.numel)
    g = dp.flat.groups[b.dtype]
    sl = dp.slices[b.dtype]
    view = g.grad[b.start:b.start + b.numel]
    torch.manual_seed(4321 + dp.rank)
    view.copy_((torch.randn(b.numel, device=dev) * 0.5).to(view.dtype))
    ref = view.float().clone()
    dist.all_reduce(ref)                                        # NCCL, fp32
    ref /= world
    torch.cuda.synchronize(dev)
    dist.barrier()
    off = b.start * view.element_size()
    algo = b.algo if b.algo in ("twoshot", "multimem") else "twoshot"
    native().allreduce_twoshot([p + off for p in sl.data_ptrs], sl.sig_ptrs, (sl.mc_ptr + off) if sl.mc_ptr else 0,
                               dp.rank, g.grad, b.numel, 1.0 / world, None, None, algo == "multimem", dp.comm_blocks, 30.0)
    torch.cuda.synchronize(dev)
    diff = (view.float() - ref).abs().max()
    dist.all_reduce(diff, op=dist.ReduceOp.MAX)
    scale = float(ref.abs().max())
    err = dp.check_comm_error()
    g.grad.zero_()
    torch.cuda.synchronize(dev)
    dist.barrier()
    return {"maxdiff": float(diff), "ref_absmax": scale, "bucket_bytes": b.numel * view.element_size(), "algo": algo,
            "dtype": str(view.dtype).replace("torch.", ""), "comm_error": err,
            "note": "own kernel (bf16 in, fp32 accumulate, bf16 out) vs NCCL fp32 all-reduce of the same data, max over ranks"}


def allreduce_report(dp, crosscheck):
    """What the data-parallel engine actually launched in the captured step (facts, not preferences)."""
    algos = [{"algo": a, "bytes": n, "optimizer_fused": f} for a, n, f in dp.last_algos]
    rep = {"algos": sorted({a["algo"] for a in algos}) or (["none"] if dp.world <= 1 else ["?"]),
           "buckets": algos, "comm_launches_per_step": sum(1 for a in algos if a["algo"] not in ("local_sgd", "none")),
           "has_multicast": bool(dp.pool.has_multicast) if dp.pool is not None else False,
           "fused_optimizer": bool(dp.bucket_opt), "world": dp.world,
           "bootstrap": dp.pool.describe() if dp.pool is not None else None}
    if crosscheck is not None:
        rep["crosscheck"] = crosscheck
        rep["maxdiff"] = crosscheck["maxdiff"]
    return rep


def exposed_comm(trainer, args, dev, world, max_over_ranks, sync_all, dev_ms_on):
    """Exposed communication per step: the captured step as benchmarked (bucket kernels overlapped with backward)
    minus the same step re-captured with communication disabled (gradients stay local, plain optimizer pass)."""
    import torch

    K = args.steps

    def timed():
        for _ in range(3):
            trainer.step_device()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        ev0.record()
        for _ in range(K):
            trainer.step_device()
        ev1.record()
        sync_all()
        return max_over_ranks(ev0.elapsed_time(ev1)) / K

    on = timed()
    trainer.dp.consolidate_optimizer_state()
    trainer.dp.enabled = False
    trainer.graph = None
    off = timed()
    trainer.dp.enabled = True
    trainer.graph = None
    trainer.sync_from(0)                      # the replicas drifted apart while they did not communicate
    on2 = timed()
    return {"exposed_comm_ms": max(0.0, min(on, on2) - off), "ms_per_step_comm_on": min(on, on2), "ms_per_step_comm_off": off,
            "ms_per_step_comm_on_runs": [on, on2], "headline_ms_per_step": dev_ms_on / K,
            "method": "device-timed A/B of the same captured step, dp.enabled True/False, %d steps each, max over ranks" % K}


def rescale_section(trainer, args, dev, world, rank, x, t):
    """Rescale recovery time after -1 / +1 GPU, in place (BASELINE.json: "rescale recovery time after +-1 pod"):
    from "the new membership is known" to "the first optimizer step at the new world size is done on every member",
    host wall clock, max over ranks.  The stop-resume path of the reference (checkpoint reload into fresh trainers,
    process start-up excluded) is timed next to it by tools/bench_rescale.py."""
    import torch
    import torch.distributed as dist

    from edl_b200.ops.optim import scaled_lr

    B = args.batch_per_gpu
    survivors = list(range(world - 1))
    small = dist.new_group(ranks=survivors)
    solo = [dist.new_group(ranks=[r]) for r in range(world)][rank]
    alive = rank in survivors

    def wall_max(t0, group=None):
        tt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX, group=group)
        return float(tt.item())

    res = {"from": world, "to": world - 1}
    torch.cuda.synchronize(dev)
    dist.barrier()
    t0 = time.perf_counter()
    trainer.prepare_rescale()
    trainer.rebuild(small if alive else solo)
    if alive:
        trainer.set_lr(scaled_lr(0.1, B, len(survivors)))
        float(trainer.step(x, t).item())
        res["leave_inplace_s"] = wall_max(t0, small)
        if len(survivors) > 1:
            res["bootstrap_small"] = trainer.dp.pool.describe()
    torch.cuda.synchronize(dev)
    dist.barrier()
    t0 = time.perf_counter()
    if alive:
        trainer.prepare_rescale()
    trainer.rebuild(None)
    trainer.sync_from(0)
    trainer.set_lr(scaled_lr(0.1, B, world))
    float(trainer.step(x, t).item())
    res["join_inplace_s"] = wall_max(t0)
    res["bootstrap_full"] = trainer.dp.pool.describe()
    flat = torch.cat([g.param.flatten().float() for g in trainer.dp.flat.groups.values()])
    ref = flat.clone()
    dist.broadcast(ref, src=0)
    same = torch.tensor([1.0 if torch.equal(flat, ref) else 0.0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    res["replicas_identical_after_join"] = bool(same.item() > 0.5)
    res["comm_error"] = trainer.dp.check_comm_error()
    res["lr_rescaled"] = [scaled_lr(0.1, B, world - 1), scaled_lr(0.1, B, world)]
    res["note"] = ("in-place: survivors keep process, CUDA context, parameters and optimizer state; new symmetric slab "
                   "through the store (no NCCL communicator), bucket re-plan, graph re-capture, joiner state over NVLink")
    return res


def distill_section(args, world, rank, dev):
    """The distill-service term of the metric on the same N GPUs (N/2 students + N/2 teachers)."""
    if world % 2 != 0:
        return {"skipped": "needs an even number of GPUs"}
    import torch

    torch.cuda.empty_cache()
    rec = distill_run(args, world, rank, dev, args.distill_steps)
    keep = ("metric", "value", "unit", "ms_per_step", "steps", "vs_baseline", "config", "e2e", "link_error", "gpu_launches")
    return {k: rec[k] for k in keep if k in rec}


if __name__ == "__main__":
    sys.exit(main())
