#!/usr/bin/env python
"""Optimizer cost on one GPU: momentum SGD vs LARS vs LAMB on ResNet50_vd's flat layout.

Part 1 -- the whole-model optimizer step alone (``opt.step()`` over both dtype groups: 167 tensors, 25.6 M
parameters), CUDA events around each step, the L2 overwritten between steps (a 256 MB memset) so every step
streams from HBM.  Reports the median time, the bytes the update has to move (from the shapes: what each kernel
reads and writes per parameter) and that traffic's share of the 7.7 TB/s data-sheet bandwidth.

Part 2 -- the full captured training step (batch 32 per GPU, bf16, one rank: SGD and LARS / LAMB all run per
bucket on the side stream during backward), one trainer per optimizer in the same process, timed in alternating
rounds, in img/s.

Writes one JSON document (stdout and ``--out``) with the GPU name and power limit read in the same run.

    python tools/bench_optim.py --out bench_optim.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from edl_b200 import ops  # noqa: E402
from edl_b200.models import ResNetVd, to_train_dtype  # noqa: E402
from edl_b200.parallel import FlatParams  # noqa: E402

HBM_BYTES_PER_S = 7.7e12     # B200 data sheet, one GPU


def no_decay(name, p):
    return p.dim() <= 1


def make_opt(kind, flat, lr):
    if kind == "sgd":
        return ops.FlatSGDMomentum(flat, lr=lr, momentum=0.9, weight_decay=1e-4)
    if kind == "lars":
        return ops.FlatLARS(flat, lr=lr, exclude=no_decay)
    return ops.FlatLAMB(flat, lr=lr * 1e-2, exclude=no_decay)


def bytes_moved(kind, flat):
    """Bytes per step from the shapes: every kernel's reads + writes of grad (bf16 / fp32), fp32 master and state,
    and the bf16 model copy.  SGD streams each group's padded buffer, LARS / LAMB the tensors' chunks."""
    total = 0
    for g in flat.groups.values():
        gb = g.grad.element_size()
        lp = 2 if g.master is not None else 0          # bf16 model copy written next to the fp32 master
        if kind == "sgd":
            n = g.numel
            per = gb + 4 + 4 + 4 + 4 + lp               # grad, master r/w, momentum r/w, model copy
        else:
            n = sum(e.numel for e in g.entries)
            if kind == "lars":
                per = (4 + gb) + (gb + 4 + 4 + 4 + 4 + lp)          # norms: w, g;  update: g, w r/w, v r/w, copy
            else:
                per = (gb + 4 * 3 + 4 * 2) + (4 * 3 + 4 + lp)      # moments: g, m, v, w, m/v out;  update: m, v, w, w out
        total += n * per
    return total


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, clk = [s.strip() for s in out.strip().split(",")[:2]]
        info.update(power_limit_w=float(pl), sm_max_mhz=float(clk))
    except Exception as e:  # noqa: BLE001 - reported, not hidden
        info["power_limit_w"] = "unavailable (%s)" % e
    return info


def part1(dev, iters):
    torch.manual_seed(0)
    model = to_train_dtype(ResNetVd(50), torch.bfloat16, dev)
    flat = FlatParams(model)
    n_tensors = sum(len(g.entries) for g in flat.groups.values())
    n_params = sum(e.numel for g in flat.groups.values() for e in g.entries)
    for g in flat.groups.values():
        g.grad.copy_((torch.randn(g.numel, device=dev) * 1e-2).to(g.grad.dtype))
    opts = {k: make_opt(k, flat, 1e-3) for k in ("sgd", "lars", "lamb")}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    times = {k: [] for k in opts}
    launches = {}
    for k, o in opts.items():                           # warm-up: module load, tables, first launches
        ops.reset_launches()
        o.step()
        launches[k] = ops.launches()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters * 3)]
    i = 0
    for _ in range(iters):
        for k, o in opts.items():                       # alternate the optimizers
            flush.zero_()
            a, b = evs[i]
            a.record()
            o.step()
            b.record()
            times[k].append((a, b))
            i += 1
    torch.cuda.synchronize()
    res = {"tensors": n_tensors, "params": n_params,
           "groups": {str(dt): {"tensors": len(g.entries), "params": sum(e.numel for e in g.entries)}
                      for dt, g in flat.groups.items()}}
    for k in opts:
        ms = [a.elapsed_time(b) for a, b in times[k]]
        us = statistics.median(ms) * 1e3
        nbytes = bytes_moved(k, flat)
        res[k] = {"us_median": round(us, 2), "us_min": round(min(ms) * 1e3, 2), "launches": launches[k],
                  "bytes": nbytes, "bytes_per_param": round(nbytes / n_params, 2),
                  "hbm_fraction_of_datasheet": round(nbytes / (us * 1e-6) / HBM_BYTES_PER_S, 3)}
    for k in ("lars", "lamb"):
        res[k]["vs_sgd"] = round(res[k]["us_median"] / res["sgd"]["us_median"], 3)
    return res


def part2(dev, batch, steps, rounds):
    from edl_b200.trainer import StudentTrainer

    x = torch.randn(batch, 3, 224, 224).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).pin_memory()
    t = torch.softmax(torch.randn(batch, 1000) * 2.0, -1).to(torch.bfloat16).pin_memory()
    trainers = {}
    for k in ("sgd", "lars", "lamb"):
        torch.manual_seed(1234)
        model = to_train_dtype(ResNetVd(50), torch.bfloat16, dev).train()
        lr = 0.1 * batch / 256.0
        factory = None if k == "sgd" else (lambda f, k=k, lr=lr: make_opt(k, f, lr))
        tr = StudentTrainer(model, batch, lr=lr, target_kind="probs", optimizer=factory)
        for _ in range(3):
            tr.step(x, t, sync=True)                    # warm-up + capture
        trainers[k] = tr
    torch.cuda.synchronize()
    per = {k: [] for k in trainers}
    for _ in range(rounds):
        for k, tr in trainers.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                tr.step_device()
            b.record()
            torch.cuda.synchronize()
            per[k].append(batch * steps / (a.elapsed_time(b) * 1e-3))
    res = {"batch": batch, "steps_per_round": steps, "rounds": rounds}
    for k, tr in trainers.items():
        res[k] = {"img_s_median": round(statistics.median(per[k]), 1),
                  "img_s_min": round(min(per[k]), 1), "img_s_max": round(max(per[k]), 1),
                  "launches_per_step": tr.launches_per_step, "bucket_optimizer": bool(tr.dp.bucket_opt),
                  "loss_finite": bool(torch.isfinite(tr.static_loss).item())}
    for k in ("lars", "lamb"):
        res[k]["vs_sgd"] = round(res[k]["img_s_median"] / res["sgd"]["img_s_median"], 4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50, help="part 1: timed steps per optimizer")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=100, help="part 2: steps per timed round")
    ap.add_argument("--rounds", type=int, default=5, help="part 2: alternating rounds")
    ap.add_argument("--skip-train", action="store_true", help="part 1 only")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}))
        return 1
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "optimizer_step": part1(dev, args.iters)}
    if not args.skip_train:
        res["train_step"] = part2(dev, args.batch, args.steps, args.rounds)
    doc = json.dumps(res, indent=1)
    print(doc)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(doc + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
