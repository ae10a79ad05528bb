"""LARS and LAMB on the flat buffers (``ops.FlatLARS`` / ``ops.FlatLAMB``, csrc/optim_layerwise.cu).

Every numeric check compares against the per-tensor fp32 implementation below, written from the update rules
alone (it shares no code with the classes' CPU branch).  CPU cases run everywhere; CUDA cases need a GPU."""
import math
import os
import subprocess
import sys

import pytest
import torch

from edl_b200 import ops
from edl_b200.ops.optim import CHUNK_ELEMS, polynomial_decay_with_warmup
from edl_b200.parallel import FlatParams
from edl_b200.parallel.ddp import plan_buckets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEVICES = ["cpu", pytest.param("cuda", marks=pytest.mark.gpu)]
KINDS = ["lars", "lamb"]

LARS_KW = dict(lr=1.0, momentum=0.9, lars_coeff=0.05, lars_weight_decay=5e-3, epsilon=1e-9)
LAMB_KW = dict(lr=0.05, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.01)


def _no_decay(name, p):
    return p.dim() == 1


# ---------------------------------------------------------------------------------------------- reference
def _ref_lars(w, v, g, lr, momentum, lars_coeff, lars_weight_decay, epsilon, decay):
    wd = lars_weight_decay if decay else 0.0
    wn, gn = w.norm().item(), g.norm().item()
    local_lr = lr * lars_coeff * wn / (gn + wd * wn + epsilon) if (wd > 0 and wn > 0 and gn > 0) else lr
    v = momentum * v + local_lr * (g + wd * w)
    return w - v, v


def _ref_lamb(w, m, v, g, t, lr, betas, eps, weight_decay, decay):
    b1, b2 = betas
    wd = weight_decay if decay else 0.0
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    r = (m / (1 - b1 ** t)) / ((v / (1 - b2 ** t)).sqrt() + eps) + wd * w
    wn, rn = w.norm().item(), r.norm().item()
    trust = wn / rn if wn > 0 and rn > 0 else 1.0
    return w - lr * trust * r, m, v


class _Mixed(torch.nn.Module):
    """bf16 matrices and fp32 vectors: one tensor spans several chunks and is not a multiple of 8 long, 1-D tensors
    are excluded from decay, and two tensors never receive a gradient (LARS / LAMB trust-ratio fallbacks)."""

    ZERO_GRAD = ("frozen", "still")

    def __init__(self, dev):
        super().__init__()
        gen = torch.Generator().manual_seed(0)
        big = (203, 130)
        assert big[0] * big[1] > 3 * CHUNK_ELEMS and big[0] * big[1] % 8 != 0
        mk = lambda shape, dt: torch.nn.Parameter(torch.randn(*shape, generator=gen).to(dt).to(dev))  # noqa: E731
        self.big = mk(big, torch.bfloat16)
        self.small = mk((7, 9), torch.bfloat16)
        self.frozen = mk((16, 8), torch.bfloat16)        # decayed, zero gradient
        self.mat32 = mk((5, 12), torch.float32)
        self.bias = mk((130,), torch.float32)            # excluded
        self.still = mk((33,), torch.float32)            # excluded, zero gradient


def _grads(model, step):
    gen = torch.Generator().manual_seed(100 + step)
    out = {}
    for n, p in model.named_parameters():
        g = torch.randn(p.shape, generator=gen)
        out[n] = torch.zeros(p.shape) if n in _Mixed.ZERO_GRAD else g
    return out


def _make(kind, dev):
    model = _Mixed(dev)
    flat = FlatParams(model)
    opt = (ops.FlatLARS(flat, exclude=_no_decay, **LARS_KW) if kind == "lars"
           else ops.FlatLAMB(flat, exclude=_no_decay, **LAMB_KW))
    return model, flat, opt


def _load_grads(model, flat, grads):
    flat.zero_grad()
    for n, p in model.named_parameters():
        p.grad.copy_(grads[n].to(p.dtype))


def _masters(flat):
    """name -> fp32 master view of every tensor."""
    out = {}
    for g, e in flat.entries():
        master = g.master if g.master is not None else g.param
        out[e.name] = master[e.offset:e.offset + e.numel].view(e.param.shape)
    return out


def _snapshot(flat, opt):
    out = [g.param.clone() for g in flat.groups.values()]
    out += [g.master.clone() for g in flat.groups.values() if g.master is not None]
    out += [t.clone() for st in opt.state.values() for t in st.values()]
    if hasattr(opt, "step_t"):
        out.append(opt.step_t.clone())
    return out


def _run(kind, dev, steps=5, grad_scale=0.5, bucket_cap=None):
    """``steps`` optimizer steps on _Mixed; whole-model ``step()``, or ``step_range`` bucket by bucket."""
    model, flat, opt = _make(kind, dev)
    opt.set_grad_scale(torch.full((1,), grad_scale, device=dev))
    buckets = plan_buckets(flat, bucket_cap) if bucket_cap else None
    if buckets:
        assert len(buckets) > 2
        opt.skip_dtype = lambda dt: True             # what ElasticDataParallel does when it owns the update
    for s in range(steps):
        _load_grads(model, flat, _grads(model, s))
        if buckets:
            for b in buckets:
                opt.step_range(b.dtype, b.start, b.numel)
        opt.step()
    if dev == "cuda":
        torch.cuda.synchronize()
    return model, flat, opt


def _reference(kind, dev, steps=5, grad_scale=0.5):
    model = _Mixed("cpu")
    w = {n: p.detach().float().clone() for n, p in model.named_parameters()}
    s1 = {n: torch.zeros_like(t) for n, t in w.items()}
    s2 = {n: torch.zeros_like(t) for n, t in w.items()}
    decay = {n: not _no_decay(n, p) for n, p in model.named_parameters()}
    for s in range(steps):
        grads = _grads(model, s)
        for n, p in model.named_parameters():
            g = grads[n].to(p.dtype).float() * grad_scale
            if kind == "lars":
                w[n], s1[n] = _ref_lars(w[n], s1[n], g, decay=decay[n], **LARS_KW)
            else:
                w[n], s1[n], s2[n] = _ref_lamb(w[n], s1[n], s2[n], g, s + 1, decay=decay[n], **LAMB_KW)
    return w


def _rel(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


# ---------------------------------------------------------------------------------------------- numerics
@pytest.mark.parametrize("dev", DEVICES)
@pytest.mark.parametrize("kind", KINDS)
def test_matches_per_tensor_reference(kind, dev):
    model, flat, opt = _run(kind, dev)
    ref = _reference(kind, dev)
    masters = _masters(flat)
    for n, p in model.named_parameters():
        assert _rel(masters[n], ref[n]) <= 1e-5, (n, _rel(masters[n], ref[n]))
        if p.dtype == torch.bfloat16:
            assert torch.equal(p.detach(), masters[n].to(torch.bfloat16)), n
    # the rules did something: every tensor moved except the excluded one without a gradient (no decay term either)
    init = _Mixed("cpu")
    for n, p in init.named_parameters():
        moved = _rel(masters[n], p.detach().float()) > 1e-3
        assert moved == (n != "still"), n
    if kind == "lamb":
        assert float(opt.step_t.item()) == 5.0


@pytest.mark.parametrize("dev", DEVICES)
@pytest.mark.parametrize("kind", KINDS)
def test_deterministic_and_bucketwise_bitwise_equal(kind, dev):
    _, flat_a, opt_a = _run(kind, dev)
    _, flat_b, opt_b = _run(kind, dev)
    _, flat_c, opt_c = _run(kind, dev, bucket_cap=256)
    a, b, c = _snapshot(flat_a, opt_a), _snapshot(flat_b, opt_b), _snapshot(flat_c, opt_c)
    assert all(torch.equal(x, y) for x, y in zip(a, b)), "two runs differ"
    assert all(torch.equal(x, y) for x, y in zip(a, c)), "bucket-by-bucket differs from the whole-model step"


@pytest.mark.parametrize("dev", DEVICES)
@pytest.mark.parametrize("kind", KINDS)
def test_found_inf_skips_the_step(kind, dev):
    model, flat, opt = _run(kind, dev, steps=1)
    before = _snapshot(flat, opt)
    _load_grads(model, flat, _grads(model, 7))
    flag = torch.ones(1, dtype=torch.int32, device=dev)
    opt.set_found_inf(flag)
    opt.step()
    after = _snapshot(flat, opt)
    assert all(torch.equal(x, y) for x, y in zip(before, after))
    flag.zero_()                                      # the same flag cleared: the step applies again
    opt.step()
    assert not all(torch.equal(x, y) for x, y in zip(before, _snapshot(flat, opt)))
    if kind == "lamb":
        assert float(opt.step_t.item()) == 2.0


def test_range_must_hold_whole_tensors():
    model, flat, opt = _make("lars", "cpu")
    g = flat.groups[torch.bfloat16]
    e = g.entries[0]
    with pytest.raises(ValueError):
        opt.step_range(torch.bfloat16, e.offset, e.numel // 2)


def test_polynomial_decay_with_warmup():
    f = lambda s: polynomial_decay_with_warmup(s, 8.0, 10, 5, 1, power=2.0, end_lr=1e-4)  # noqa: E731
    assert f(0) == 0.0 and f(5) == 4.0 and math.isclose(f(10), 8.0)
    assert math.isclose(f(30), (8.0 - 1e-4) * (1 - 20 / 40) ** 2 + 1e-4)
    assert math.isclose(f(50), 1e-4) and math.isclose(f(80), 1e-4)
    assert all(f(s) >= f(s + 1) for s in range(10, 60))


# ---------------------------------------------------------------------------------------------- trainer
def _trainer(kind, dev, graph=False, seed=0, **kw):
    from edl_b200.models import ResNetVd, to_train_dtype
    from edl_b200.trainer import StudentTrainer

    dt = torch.bfloat16 if dev == "cuda" else torch.float32
    torch.manual_seed(seed)
    m = to_train_dtype(ResNetVd(18, class_dim=10, width_mult=0.25), dt, torch.device(dev)).train()
    factory = {"lars": lambda f: ops.FlatLARS(f, lr=0.5, lars_coeff=0.02, exclude=_no_decay),
               "lamb": lambda f: ops.FlatLAMB(f, lr=0.01, exclude=_no_decay)}[kind]
    return StudentTrainer(m, batch_size=8, image_shape=(3, 32, 32), num_classes=10, lr=0.5, use_graph=graph,
                          dtype=dt, optimizer=factory, **kw)


def _batch(dev, seed=0):
    gen = torch.Generator().manual_seed(seed)
    dt = torch.bfloat16 if dev == "cuda" else torch.float32
    x = torch.randn(8, 3, 32, 32, generator=gen).to(dt).contiguous(memory_format=torch.channels_last)
    t = torch.softmax(torch.randn(8, 10, generator=gen), -1).to(dt)
    if dev == "cuda":
        x, t = x.pin_memory(), t.pin_memory()
    return x, t


def _flat_masters(tr):
    return [(g.master if g.master is not None else g.param).clone() for g in tr.dp.flat.groups.values()]


def _clone(obj):
    if torch.is_tensor(obj):
        return obj.detach().clone()
    if isinstance(obj, dict):
        return {k: _clone(v) for k, v in obj.items()}
    return obj


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_trainer_rides_the_bucket_hook_and_graph_matches_eager(kind):
    x, t = _batch("cuda")
    eager, graph = _trainer(kind, "cuda", graph=False), _trainer(kind, "cuda", graph=True)
    # one rank, no loss scaling / clipping: the update runs per bucket on the side stream
    assert eager.dp.bucket_opt and graph.dp.bucket_opt
    w0 = _flat_masters(eager)
    le = [float(eager.step(x, t, sync=True)) for _ in range(4)]       # == the graph trainer's 3 warm-ups + 1 replay
    lg = [float(graph.step(x, t, sync=True))]
    assert any(a[0].startswith("local_" + type(eager.opt).__name__.lower()) for a in eager.dp.last_algos)
    le.append(float(eager.step(x, t, sync=True)))
    lg.append(float(graph.step(x, t, sync=True)))
    torch.cuda.synchronize()
    assert all(math.isfinite(v) for v in le + lg)
    assert abs(le[-1] - lg[-1]) <= 1e-2 * max(1.0, abs(le[-1])), (le, lg)
    for a, b, w in zip(_flat_masters(eager), _flat_masters(graph), w0):
        assert _rel(b, a) < 1e-2
        assert _rel(b - w, a - w) < 0.15                              # the updates themselves, bf16 tolerance
    if kind == "lamb":
        assert float(eager.opt.step_t.item()) == 5.0 and float(graph.opt.step_t.item()) == 5.0


@pytest.mark.gpu
def test_graph_reads_the_learning_rate_from_the_device():
    x, t = _batch("cuda")
    tr = _trainer("lars", "cuda", graph=True)
    tr.step(x, t, sync=True)                                         # capture + first replay
    tr.set_lr(0.0)
    for st in tr.opt.state.values():
        st["mom"].zero_()                                            # v = 0.9 * 0 + 0 * (...): nothing moves
    torch.cuda.synchronize()
    before = [g.param.clone() for g in tr.dp.flat.groups.values()] + _flat_masters(tr)
    tr.step(x, t, sync=True)
    torch.cuda.synchronize()
    after = [g.param.clone() for g in tr.dp.flat.groups.values()] + _flat_masters(tr)
    assert all(torch.equal(a, b) for a, b in zip(before, after))
    tr.set_lr(0.5)
    tr.step(x, t, sync=True)
    torch.cuda.synchronize()
    assert not all(torch.equal(a, b) for a, b in zip(after, _flat_masters(tr)))


@pytest.mark.gpu
def test_clipped_step_matches_reference_on_clipped_gradients():
    x, t = _batch("cuda")
    tr = _trainer("lars", "cuda", graph=True, clip_norm=0.05)
    assert not tr.dp.bucket_opt                                      # clipping needs every gradient first
    tr.step(x, t, sync=True)
    torch.cuda.synchronize()
    flat = tr.dp.flat
    w_before = {dt: (g.master if g.master is not None else g.param).clone() for dt, g in flat.groups.items()}
    v_before = {dt: st["mom"].clone() for dt, st in tr.opt.state.items()}
    tr.step(x, t, sync=True)
    torch.cuda.synchronize()
    scale = float(tr.dp.clip_scale_t.item())
    assert 0 < scale < 1, scale
    opt = tr.opt
    for dt, g in flat.groups.items():
        master = g.master if g.master is not None else g.param
        for e in g.entries:
            sl = slice(e.offset, e.offset + e.numel)
            decay = not _no_decay(e.name, e.param)
            want, _ = _ref_lars(w_before[dt][sl].cpu(), v_before[dt][sl].cpu(), g.grad[sl].float().cpu() * scale,
                                lr=opt.lr, momentum=opt.momentum, lars_coeff=opt.lars_coeff,
                                lars_weight_decay=opt.lars_weight_decay, epsilon=opt.epsilon, decay=decay)
            assert _rel(master[sl], want) <= 1e-5, (e.name, _rel(master[sl], want))


@pytest.mark.parametrize("dev", DEVICES)
@pytest.mark.parametrize("kind", KINDS)
def test_checkpoint_resumes_exactly(kind, dev):
    x, t = _batch(dev)
    a = _trainer(kind, dev)
    for _ in range(2):
        a.step(x, t, sync=True)
    sd = _clone(a.state_dict())
    b = _trainer(kind, dev, seed=1)
    b.load_state_dict(sd)
    a.step(x, t, sync=True)
    b.step(x, t, sync=True)
    if dev == "cuda":
        torch.cuda.synchronize()
    tol = 1e-3 if dev == "cuda" else 1e-6                           # BatchNorm atomics on the GPU
    for wa, wb in zip(_flat_masters(a), _flat_masters(b)):
        assert _rel(wb, wa) <= tol
    if kind == "lamb":
        assert float(b.opt.step_t.item()) == 3.0


# ---------------------------------------------------------------------------------------------- example
def _example(args, timeout=300):
    e = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    p = subprocess.run([sys.executable, "examples/collective/resnet50/train.py"] + args, cwd=ROOT, env=e,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=timeout, text=True)
    assert p.returncode == 0, p.stdout[-3000:]
    losses = [float(line.split(" loss ")[1].split()[0]) for line in p.stdout.splitlines() if " loss " in line]
    assert losses and all(math.isfinite(v) for v in losses), p.stdout[-3000:]
    return p.stdout


@pytest.mark.parametrize("flags", [["--optimizer", "lars", "--lr_strategy", "polynomial_decay"],
                                   ["--optimizer", "lamb", "--lr", "0.5"]])
def test_resnet_example_with_layerwise_optimizer(tmp_path, flags):
    base = ["--model", "ResNet18_vd", "--width_mult", "0.125", "--image_size", "32", "--class_dim", "10",
            "--batch_size", "4", "--steps_per_epoch", "3", "--ckpt", str(tmp_path / "ck")] + flags
    out = _example(base + ["--epochs", "1"])
    assert "Pass 0 trainbatch 0" in out
    out = _example(base + ["--epochs", "2"])                        # resumes from the epoch-0 checkpoint
    assert "Pass 1 trainbatch 0" in out and "Pass 0 trainbatch" not in out


# ---------------------------------------------------------------------------------------------- two ranks
def _two_rank_worker(rank, world, port, q):
    try:
        import torch.distributed as dist

        from edl_b200.parallel import ElasticDataParallel

        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        model = _Mixed(dev)
        dp = ElasticDataParallel(model)
        opt = ops.FlatLARS(dp.flat, exclude=_no_decay, **LARS_KW)
        ref_model = _Mixed(dev)
        ref_flat = FlatParams(ref_model)
        ref_opt = ops.FlatLARS(ref_flat, exclude=_no_decay, **LARS_KW)
        for s in range(3):
            per_rank = [_grads(model, 10 * s + r) for r in range(world)]
            dp.zero_grad()
            for n, p in model.named_parameters():
                p.grad.copy_(per_rank[rank][n].to(p.dtype))
            dp.finish()                                      # every bucket through the all-reduce kernels
            opt.step()
            avg = {n: sum(g[n].to(p.dtype).float() for g in per_rank) / world for n, p in model.named_parameters()}
            _load_grads(ref_model, ref_flat, avg)
            ref_opt.step()
        torch.cuda.synchronize()
        got, want = _masters(dp.flat), _masters(ref_flat)
        errs = {n: _rel(got[n], want[n]) for n in got}
        assert all(v <= 1e-5 for v in errs.values()), errs
        if rank == 0:
            q.put(("ok", errs))
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:  # noqa
        import traceback

        q.put(("fail", "rank %d: %s\n%s" % (rank, e, traceback.format_exc())))
        raise


@pytest.mark.gpu
@pytest.mark.multigpu
def test_two_rank_allreduce_then_lars_equals_single_rank_on_averaged_gradients():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29400 + os.getpid() % 1000
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    status, payload = q.get(timeout=300)
    for p in procs:
        p.join(60)
    assert status == "ok", payload
