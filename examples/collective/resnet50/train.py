#!/usr/bin/env python
"""Elastic ResNet training (reference workload: example/collective/resnet50/train_with_fleet.py,
launched through ``python -m paddle_edl.collective.launch``, train_pretrain.sh:36-61).

With ``--rescale_mode inplace`` on the launcher (``EDL_RESCALE_MODE=inplace``) the trainer is NOT restarted on a
membership change: it re-rendezvouses through the store (``edl_b200.elastic.ElasticContext``), re-plans the fused
all-reduce for the new world (``StudentTrainer.rebuild``), hands parameters / momentum / step counters to joiners
over the fabric (``sync_from``) and rescales the LR.  Otherwise, the reference's stop-resume:

Every (re)start: join the stage's process group, reload the newest atomic checkpoint, rescale the
learning rate to the world size (``lr = base_lr * batch * world / 256`` -- the reference's rule,
:129-141) and continue from ``train_status.next()``.  Data is synthetic unless ``--data_dir`` points
at a directory of ``.pt`` shards (uint8 NHWC images + int64 labels).

    python -m paddle_edl.collective.launch --nodes_range 1:8 --nproc_per_node 8 --etcd_endpoints H:P \
        --job_id rn50 --hdfs_path /ckpt/rn50 examples/collective/resnet50/train.py --epochs 90
"""
import argparse
import json
import os
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, ROOT)

import edl_b200 as edl  # noqa: E402
from edl_b200 import elastic, ops  # noqa: E402
from edl_b200.checkpoint import LocalFS, TrainStatus, load_check_point, save_check_point  # noqa: E402
from edl_b200.models import VGG, ResNet, ResNetVd, to_train_dtype  # noqa: E402
from edl_b200.ops.optim import (cosine_decay_with_warmup, piecewise_decay_with_warmup,  # noqa: E402
                                polynomial_decay_with_warmup, scaled_lr)
from edl_b200.trainer import StudentTrainer  # noqa: E402
from edl_b200.utils import train_status as edl_train_status  # noqa: E402
from edl_b200.utils.metrics import StepMeter, write_benchmark_log  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="ResNet50_vd", help="ResNet{18,34,50,101,152}[_vd] or VGG{11,13,16,19}")
    ap.add_argument("--layers", type=int, default=0, help="deprecated: overrides the depth in --model")
    ap.add_argument("--epochs", type=int, default=90)
    ap.add_argument("--batch_size", type=int, default=32, help="per trainer")
    ap.add_argument("--total_batch_size", type=int, default=0, help="if set, per-trainer batch = total / world")
    ap.add_argument("--lr", type=float, default=0.1)
    ap.add_argument("--lr_strategy", default="cosine_decay_with_warmup",
                    choices=["cosine_decay_with_warmup", "piecewise_decay", "polynomial_decay"])
    ap.add_argument("--optimizer", default="momentum", choices=["momentum", "lars", "lamb"],
                    help="momentum SGD (the reference's default), LARS or LAMB (large global batches); LARS / LAMB "
                         "leave 1-D parameters (BatchNorm scale / shift, biases) out of weight decay")
    ap.add_argument("--lars_coeff", type=float, default=0.001)
    ap.add_argument("--lars_weight_decay", type=float, default=5e-4)
    ap.add_argument("--steps_per_epoch", type=int, default=0, help="0 = total_images / (batch * world)")
    ap.add_argument("--total_images", type=int, default=1281167)
    ap.add_argument("--class_dim", type=int, default=1000)
    ap.add_argument("--image_size", type=int, default=224)
    ap.add_argument("--label_smoothing", type=float, default=0.0)
    ap.add_argument("--width_mult", type=float, default=1.0)
    ap.add_argument("--ckpt", default=os.environ.get("PADDLE_EDL_HDFS_PATH") or "./resnet_ckpt")
    ap.add_argument("--max_steps", type=int, default=0, help="stop an epoch early (smoke runs)")
    ap.add_argument("--inject_fault_file", default=os.environ.get("RESNET_INJECT_FAULT_FILE", ""),
                    help="testing: once this file exists, rank 1 reports ONE failed collective although every pod is alive "
                         "(a false alarm: exercises the soft reset of ElasticContext.recover())")
    ap.add_argument("--data_dir", default=None,
                    help="ImageNet-style directory with train_list.txt ('relative/path.jpg label' per line); synthetic if unset")
    ap.add_argument("--use_dali", type=lambda v: str(v).lower() in ("1", "true", "yes"), default=False,
                    help="the reference's flag for GPU-side decoding: JPEGs are decoded by nvJPEG and cropped / resized / "
                         "normalised by one kernel on the training GPU (ImageBatchLoader(decode='nvjpeg')); default: "
                         "OpenCV worker threads + uint8 H2D + normalize_u8")
    ap.add_argument("--reader_threads", type=int, default=8)
    ap.add_argument("--solo_step_sleep", type=float, default=0.0,
                    help="elastic demos / tests: seconds to sleep per step while the job has ONE trainer, so that a "
                         "second pod has time to join whatever the speed of the box")
    return ap.parse_args()


def file_feed(args, bs, rank, world, epoch, skip, dev, dtype, cuda):
    """Batches of the ImageNet-style file list for this rank and epoch, ``skip`` batches in (resume / in-place rescale
    mid-epoch).  Reference: the DALI / cv2 readers of example/collective/resnet50/train_with_fleet.py (--use_dali)."""
    if not args.data_dir:
        return None
    from edl_b200.utils import image_pipeline as ip

    samples = ip.read_file_list(os.path.join(args.data_dir, "train_list.txt"))
    ld = ip.ImageBatchLoader(samples, bs, size=args.image_size, train=True, rank=rank, world=world, seed=0,
                             threads=args.reader_threads, decode="nvjpeg" if (args.use_dali and cuda) else "cpu")
    ld.set_epoch(epoch)

    def gen():
        for i, batch in enumerate(ld):
            if i >= skip:
                yield ip.to_device_batch(batch, dev, dtype)
    return gen()


def make_optimizer(args, lr):
    """``StudentTrainer(optimizer=...)`` factory for ``--optimizer`` (None: the trainer's momentum SGD)."""
    if args.optimizer == "momentum":
        return None
    no_decay = lambda name, p: p.dim() <= 1                  # noqa: E731  (BatchNorm scale / shift, biases)
    if args.optimizer == "lars":
        return lambda flat: ops.FlatLARS(flat, lr=lr, lars_coeff=args.lars_coeff,
                                         lars_weight_decay=args.lars_weight_decay, exclude=no_decay)
    return lambda flat: ops.FlatLAMB(flat, lr=lr, exclude=no_decay)


def learning_rate(args, step, base_lr, steps_per_epoch):
    if args.lr_strategy.startswith("cosine"):
        return cosine_decay_with_warmup(step, base_lr, steps_per_epoch, args.epochs)
    if args.lr_strategy == "polynomial_decay":
        return polynomial_decay_with_warmup(step, base_lr, steps_per_epoch, args.epochs, warmup_epochs=5)
    return piecewise_decay_with_warmup(step, base_lr, steps_per_epoch, [30, 60, 80])


def main():
    args = parse()
    ctx = info = None
    if elastic.inplace_requested():
        ctx = elastic.ElasticContext(check_every=int(os.environ.get("EDL_INPLACE_CHECK_EVERY", "20")))
        info = ctx.start()
        env, world, rank = ctx.env, info.size, info.rank
    else:
        env = edl.init_distributed()
        world, rank = env.size, env.global_rank
    cuda = torch.cuda.is_available()
    if args.data_dir:
        from edl_b200.utils import image_pipeline
        args.total_images = len(image_pipeline.read_file_list(os.path.join(args.data_dir, "train_list.txt")))
    dev = torch.device("cuda", torch.cuda.current_device()) if cuda else torch.device("cpu")
    bs = args.batch_size if not args.total_batch_size else max(1, args.total_batch_size // world)
    torch.manual_seed(0)
    dtype = torch.bfloat16 if cuda else torch.float32
    depth = args.layers or int("".join(ch for ch in args.model.split("_")[0] if ch.isdigit()))
    if args.model.upper().startswith("VGG"):
        net = VGG(depth, args.class_dim, width_mult=args.width_mult, image_size=args.image_size)
    elif args.model.endswith("_vd"):
        net = ResNetVd(depth, args.class_dim, width_mult=args.width_mult)
    else:
        net = ResNet(depth, args.class_dim, width_mult=args.width_mult)
    model = to_train_dtype(net, dtype, dev).train()
    base_lr = scaled_lr(args.lr, bs, world)
    tr = StudentTrainer(model, bs, image_shape=(3, args.image_size, args.image_size), num_classes=args.class_dim,
                        lr=base_lr, target_kind="labels", use_graph=cuda, dtype=dtype,
                        fabric=ctx.fabric if ctx is not None else None,   # GPUs in place: no process group at all
                        optimizer=make_optimizer(args, base_lr),
                        loss_fn=lambda z, t: ops.soft_cross_entropy(z, t, "labels", label_smoothing=args.label_smoothing))
    fs = LocalFS()

    def take_cursor_from(root, cursor):
        """Parameters, momentum and the (epoch, iteration, step) cursor of ``root``: the in-place state handoff."""
        if world <= 1:
            return cursor
        tr.sync_from(root)
        if ctx is not None:
            return tuple(ctx.broadcast_object(cursor, root))
        box = [cursor]
        dist.broadcast_object_list(box, src=root)
        return box[0]

    if ctx is not None and info.root is not None:
        epoch, it0, step = take_cursor_from(info.root, None)        # joined a running job: nothing is read from disk
    else:
        tensors, ts, _ = load_check_point(args.ckpt, fs, trainer_id=rank, map_location=dev)
        if tensors is not None:
            tr.load_state_dict(tensors)
        epoch, it0, step = ts.next(), 0, ts.global_step
    steps_per_epoch = args.steps_per_epoch or max(1, args.total_images // (bs * world))
    etcd = None
    if env.etcd_endpoints:
        from edl_b200.discovery.etcd_client import EtcdClient
        etcd = EtcdClient(env.etcd_endpoints, root=env.job_id)
        etcd.init()
    meter = StepMeter(bs, world)
    lr = base_lr
    progress = os.environ.get("EDL_PROGRESS_FILE", "")
    injected = False
    while epoch < args.epochs:
        g = torch.Generator().manual_seed(epoch * 1000 + rank)       # pass_id as seed: reproducible after resume
        t0, seen = time.time(), 0
        n_steps = steps_per_epoch if not args.max_steps else min(steps_per_epoch, args.max_steps)
        it = it0
        it0 = 0
        switch, failed = False, ""
        feed = file_feed(args, bs, rank, world, epoch, it, dev, dtype, cuda)
        while it < n_steps:
            lr = learning_rate(args, step, base_lr, steps_per_epoch)
            tr.set_lr(lr)
            if (ctx is not None and world > 1 and rank == 1 and not injected and args.inject_fault_file
                    and os.path.exists(args.inject_fault_file)):
                injected = True
                failed = "injected collective fault (testing the soft reset)"
                break
            if feed is not None:
                try:
                    x, y = next(feed)                                # already on the device (or CPU tensors without one)
                except StopIteration:
                    break                                            # this rank's shard is exhausted: epoch over
            else:
                x = torch.randn(bs, 3, args.image_size, args.image_size, generator=g).to(dtype)
                x = x.contiguous(memory_format=torch.channels_last)
                y = torch.randint(0, args.class_dim, (bs,), generator=g)
                if cuda:
                    x, y = x.pin_memory(), y.pin_memory()
            try:
                loss = tr.step(x, y)
            except RuntimeError as e:
                # library collectives (gloo / NCCL process group) RAISE when a peer is gone; the fabric kernels time out
                # into an error word instead and the poll below reports it
                if ctx is None:
                    raise
                failed = str(e).splitlines()[0][:200]
                break
            step += 1
            it += 1
            seen += bs
            meter.step()
            if args.solo_step_sleep and world == 1:
                time.sleep(args.solo_step_sleep)
            if progress and rank == 0 and step % 5 == 0:
                with open(progress, "a") as fh:       # machine-readable heartbeat (tools/bench_elastic_launch.py)
                    fh.write(json.dumps({"t": time.time(), "step": step, "epoch": epoch, "world": world,
                                         "pid": os.getpid(), "loss": float(loss)}) + "\n")
            if (it - 1) % 10 == 0 and rank == 0:
                print("Pass %d trainbatch %d loss %.4f lr %.5f speed %.1f img/s" % (
                    epoch, it - 1, float(loss), lr, seen * world / max(1e-6, time.time() - t0)), flush=True)
            try:
                if ctx is not None and ctx.poll(agree=tr.dp.agree):
                    switch = True
                    break
            except RuntimeError as e:                            # a collective timed out: a peer is gone
                failed = str(e)
                break
        if ctx is not None and not switch and not failed:
            try:
                switch = ctx.poll(force=True, agree=tr.dp.agree)
            except RuntimeError as e:
                failed = str(e)
        if switch or failed:
            try:
                if failed:
                    # hot recovery: the steps since the failure were device-side no-ops (the fused optimizer skips
                    # its update while the fabric's error word is set), the parameters are those of the last good step
                    print("rank %d: %s -- recovering in place" % (rank, failed), flush=True)
                    info = ctx.recover()
                else:
                    tr.prepare_rescale()                        # sharded optimizer state made complete (old stage)
                    info = ctx.rescale()
            except elastic.EdlEvicted:
                print("rank %d: pod left the job (scale-in); exiting" % rank, flush=True)
                ctx.close()
                return
            old_world, world, rank = world, info.size, info.rank
            # new symmetric slab + bucket plan; graph re-captured lazily
            tr.rebuild(None, fabric=ctx.fabric, failed=bool(failed))
            failed = ""
            epoch, it0, step = take_cursor_from(info.root, (epoch, it, step))
            base_lr = scaled_lr(args.lr, bs, world)             # lr = base * batch * world / 256
            steps_per_epoch = args.steps_per_epoch or max(1, args.total_images // (bs * world))
            meter = StepMeter(bs, world)
            print("rescaled in place: world %d -> %d, rank %d, pid %d, rendezvous %.2fs" % (
                old_world, world, rank, os.getpid(), info.rendezvous_s), flush=True)
            # back to the top with the agreed cursor -- survivors AND joiners then run exactly the same code from
            # here on (a switch that landed on the epoch boundary included: the step loop is empty, the forced poll,
            # the checkpoint and the barrier below follow on every rank in the same order)
            continue
        if etcd is not None and epoch >= args.epochs - 2 and env.pod_id:
            edl_train_status.save_to_etcd(etcd, env.pod_id, edl_train_status.TrainStatus.NEARTHEEND)   # no more scale-out
        tr.consolidate()                 # fused optimizer: every rank's slices of master / momentum -> complete state
        if rank == 0:
            save_check_point(args.ckpt, tr.state_dict(), TrainStatus(epoch, step), fs, trainer_id=0,
                             state_json=json.dumps({"world": world, "lr": lr}))
        if ctx is not None:
            ctx.barrier()
        elif world > 1:
            dist.barrier()
        epoch += 1
    write_benchmark_log(rank, dict(meter.summary(), model=args.model, batch_size=bs))   # reference: benchmark_logs/log_<id>
    if ctx is not None:
        ctx.close()
    elif world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
