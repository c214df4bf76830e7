#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): samples/sec, whole box, device-timed, max over ranks, for
ResNet-50 data-parallel training in bf16 at 1/2/4/8 B200.

  python bench.py --gpus 1 --steps 30 --warmup 5                       # this framework
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P bench.py --gpus N --steps K --warmup W           # N > 1
  python bench.py --impl reference ...                                 # the UNMODIFIED reference from baseline/_ref
  python bench.py ... --dump-outputs DIR                               # + the last timed step's loss and parameters as .npy

Workload (identical in both arms; weak scaling - per-GPU work fixed):
  ResNet-50, random init, bf16 compute; per-GPU batch 32 (the reference's --per_gpu_train_batch_size default,
  ddp.py:298); synthetic ImageNet-shaped data held in host memory the way the reference's dataset.py holds its
  data: x fp32 [3,224,224], y fp32 [1000] (dense one-hot, because the reference's train() hard-codes nn.MSELoss,
  ddp.py:164); SGD lr 1e-3, clip_grad_norm 1000, linear warmup/decay schedule; every step includes the optimizer.

Arms:
  ours       b200ddp public API: BatchLoader (pinned) -> DevicePrefetcher (H2D on a copy stream) -> TrainStep
             (CUDA-graph captured fwd + fused loss + bwd + native DDP reducer kernels + fused clip/SGD).
             "value" times K steps on device-resident (already prefetched) batches; "e2e" times K steps through
             the loader including the pinned->device copy of every batch and a D2H read of every step's loss.
  reference  baseline/_ref/ddp.py's own setup()/train()/cleanup() (stock torch DDP + NCCL, DataLoader,
             blocking H2D, 2x loss.item() per step, clip_grad_norm_, SGD).  train() takes the model as an
             argument (ResNet-50 under autocast bf16, channels_last); the dataset is injected by rebinding the
             module global ``FooDataset`` (the template's intended customisation point is dataset.py) - no
             reference source line is edited.  Its loop is inherently end to end, so value == e2e there.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
# the image exports NCCL_DEBUG=VERSION, which makes NCCL print a banner on stdout; stdout carries the JSON line
os.environ["NCCL_DEBUG"] = os.environ.get("B200DDP_NCCL_DEBUG", "WARN")
BASELINE_PUBLISHED = None   # the reference publishes no number (BASELINE.md) -> vs_baseline = null

MODEL_CHOICES = ("resnet50", "resnet152", "foo", "bert-base")


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=30)
    p.add_argument("--warmup", type=int, default=8)
    p.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "stock"],
                   help="ours | reference (unmodified template from baseline/_ref) | stock (torch DDP + NCCL + cuBLAS/cuDNN loop for the non-headline BASELINE configs)")
    p.add_argument("--model", type=str, default="resnet50", choices=MODEL_CHOICES)
    p.add_argument("--per_gpu_batch", type=int, default=None, help="default: 32 (resnet/foo, the reference default), 16 (bert-base, seq 512)")
    p.add_argument("--image_size", type=int, default=224)
    p.add_argument("--samples", type=int, default=1024, help="synthetic samples held in host memory per rank")
    p.add_argument("--backend", type=str, default="auto", choices=["auto", "b200", "nccl"])
    p.add_argument("--no_graph", action="store_true")
    p.add_argument("--bucket_cap_mb", type=float, default=None)
    p.add_argument("--wire_dtype", type=str, default=None)
    p.add_argument("--gradient_as_bucket_view", action="store_true")
    p.add_argument("--find_unused_parameters", action="store_true")
    p.add_argument("--skip_e2e", action="store_true")
    p.add_argument("--stock_graph", action="store_true", help="--impl stock: replay the whole stock step (fwd + bwd + DDP/NCCL + clip + SGD) from one CUDA graph")
    p.add_argument("--no_comm", action="store_true", help="diagnostic: N ranks, gradient communication disabled")
    p.add_argument("--profile_range", action="store_true", help="cudaProfilerStart/Stop around the device-timed loop (ncu --profile-from-start off)")
    p.add_argument("--trace_dir", type=str, default=None, help="after the timed loops: 4 more steps under the CUPTI profiler, one chrome trace per rank "
                                                                  "(<dir>/rank<r>.json) for tools/trace_digest.py; never a timing source")
    p.add_argument("--no_broadcast_buffers", action="store_true", help="diagnostic: DDP without the per-step buffer broadcast")
    p.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                   help="--impl ours: after the timed loops, write what the last timed step left for its caller (the loss it returned "
                        "and the updated parameters) as DIR/loss.npy and DIR/params.npy, so two builds can be compared output for output")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs is only implemented for --impl ours")
    if args.per_gpu_batch is None:
        args.per_gpu_batch = 16 if args.model.startswith("bert") else 32
    return args


# --------------------------------------------------------------------------------------------------
# clocks / throttle sampling during the timed region (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc = None
        self.lines = []
        self.gpu_index = gpu_index
        self._thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.lines.append(line.strip())
        self._thread = threading.Thread(target=pump, daemon=True)
        self._thread.start()

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [c for c, w in zip(sm, power) if w > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(busy), "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local_rank, world


def emit(obj: dict) -> None:
    sys.stdout.write(json.dumps(obj) + "\n")
    sys.stdout.flush()


# --------------------------------------------------------------------------------------------------
# shared workload pieces
# --------------------------------------------------------------------------------------------------
def make_dataset(args):
    import torch
    sys.path.insert(0, ROOT)
    from b200ddp.data import FooDataset, SyntheticImageNet, SyntheticTokens
    if args.model.startswith("resnet"):
        return SyntheticImageNet(samples=args.samples, size=args.image_size, image_dtype=torch.float32, dense_target=True)
    if args.model == "foo":
        return FooDataset(100000)
    return SyntheticTokens(samples=min(args.samples, 256))


def opt_ins(model):
    """Non-default kernel choices switched on through the environment (none by default) - recorded so a run is
    reproducible from its JSON line."""
    out = {}
    for key in ("B200DDP_GEMM_GROUP_M", "B200DDP_GEMM_TMA_STORE", "B200DDP_GEMM_CTAS", "B200DDP_CONV", "B200DDP_CONV_WGRAD", "B200DDP_DISABLE_TC",
                "B200DDP_STEM", "B200DDP_STEM_WGRAD", "B200DDP_STEM_RESIDENT", "B200DDP_BLOCK_FUSE", "B200DDP_PDL", "B200DDP_BN_FUSED", "B200DDP_DDP_SERIAL",
                "B200DDP_COMM_BLOCKS", "B200DDP_TAIL_BLOCKS", "B200DDP_TAIL_BUCKET_MB", "B200DDP_TAIL_ONE_SHOT_MAX_MB"):
        if os.environ.get(key):
            out[key] = os.environ[key]
    return {"opt_in": out} if out else {}


DUMP_SAMPLE = 1 << 22      # elements kept per array (16 MB): positions drawn from a fixed seed, the same in every build


def dump_outputs(out_dir, loss, model):
    """What the caller of a training step holds after it, as float32 arrays: the loss the step returned (loss.npy) and
    the parameters it updated, flattened and concatenated in module order (params.npy), reduced to a seeded sample of
    DUMP_SAMPLE elements when longer.  Gradients and BatchNorm running statistics are not written: on a randomly
    initialised bf16 ResNet two runs of the same build already disagree on them (the gradients below the head
    entirely, the last stage's running statistics by a few percent), so they cannot tell two builds apart."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, tensors in (("loss", [loss]), ("params", list(model.parameters()))):
        flat = torch.cat([t.detach().reshape(-1).float() for t in tensors])
        if flat.numel() > DUMP_SAMPLE:
            idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(out_dir, name + ".npy"), flat.cpu().numpy())


def config_dict(args, world, extra=None):
    cfg = {"model": args.model, "global_batch": args.per_gpu_batch * world, "per_gpu_batch": args.per_gpu_batch,
           "image_size": args.image_size if args.model.startswith("resnet") else None,
           "seq_len": 512 if args.model.startswith("bert") else None,
           "parallelism": f"dp{world}", "loss": "mse(dense one-hot target)" if not args.model.startswith("bert") else "ce",
           "optimizer": "sgd lr1e-3 + clip_grad_norm 1000 + linear warmup/decay",
           "l2": "per-step working set (bf16 activations + weights + grads, > 2 GB at batch 32) exceeds the 126 MB L2; "
                 "input batches rotate over distinct pinned host batches"}
    if extra:
        cfg.update(extra)
    return cfg


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from b200ddp import _ext
    from b200ddp.data import BatchLoader, DevicePrefetcher
    from b200ddp.engine.step import TrainStep
    from b200ddp.models import build_model
    from b200ddp.ops import CrossEntropyLoss, MSELoss
    from b200ddp.optim import FusedSGD, get_linear_schedule_with_warmup
    from b200ddp.parallel import DistributedDataParallel, EndlessSampler, ShardedSampler
    from b200ddp.utils import to_mixed_bf16

    rank, local_rank, world = dist_env()
    assert world == args.gpus, f"WORLD_SIZE={world} but --gpus {args.gpus}: launch with torchrun --nproc-per-node {args.gpus}"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    C = _ext.get()
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    torch.manual_seed(42)
    torch.backends.cudnn.benchmark = True

    is_image = args.model.startswith("resnet")
    model = build_model(args.model).to(dev)
    if args.model != "foo":
        model = to_mixed_bf16(model)
    if is_image:
        model = model.to(memory_format=torch.channels_last)
    compute_dtype = torch.float32 if args.model == "foo" else torch.bfloat16
    inner = model
    backend = args.backend
    if world > 1:
        model = DistributedDataParallel(model, device_ids=[local_rank], find_unused_parameters=args.find_unused_parameters,
                                        gradient_as_bucket_view=args.gradient_as_bucket_view, backend=backend,
                                        bucket_cap_mb=args.bucket_cap_mb, wire_dtype=args.wire_dtype,
                                        broadcast_buffers=not args.no_broadcast_buffers)
        backend = model.backend_name
        if args.no_comm:
            model.require_backward_grad_sync = False
            backend += "(comm disabled: diagnostic)"
    else:
        backend = "single"
    opt = FusedSGD(inner.parameters(), lr=1e-3, max_grad_norm=1000.0)     # after the wrap-time broadcast
    sched = get_linear_schedule_with_warmup(opt, num_warmup_steps=100, num_training_steps=100000)
    criterion = CrossEntropyLoss() if args.model.startswith("bert") else MSELoss()

    # input pipeline kernel: raw fp32 NCHW batch -> bf16 channels_last, straight into the graph's input buffer
    mean = torch.zeros(3, device=dev)
    inv_std = torch.ones(3, device=dev)
    static_in = {}

    def input_transform(x):
        if not is_image:
            return x if x.dtype == compute_dtype or not x.is_floating_point() else x.to(compute_dtype)
        shape = tuple(x.shape)
        buf = step.static_inputs()[0]          # after capture: write straight into the graph's input buffer
        if buf is None or tuple(buf.shape) != shape:
            buf = static_in.get("x")
        if buf is None or tuple(buf.shape) != shape:
            buf = torch.empty(shape, dtype=compute_dtype, device=dev).contiguous(memory_format=torch.channels_last)
            static_in["x"] = buf
        C.normalize_to_channels_last(x, buf, mean, inv_std, 1.0)
        return buf

    def target_transform(y):
        return y.to(compute_dtype) if y.is_floating_point() and y.dtype != compute_dtype else y

    step = TrainStep(model, criterion, opt, dev, use_graph=not args.no_graph, input_transform=input_transform,
                     target_transform=target_transform)

    dataset = make_dataset(args)
    sampler = ShardedSampler(dataset, num_replicas=world, rank=rank, shuffle=True, seed=0) if world > 1 else \
        torch.utils.data.RandomSampler(dataset)
    # an endless index stream: with a small synthetic dataset sharded over 8 ranks an epoch is only 4 batches, and
    # draining the prefetch pipeline at every epoch boundary would be an artefact of the benchmark, not of training
    loader = BatchLoader(dataset, batch_size=args.per_gpu_batch, sampler=EndlessSampler(sampler), drop_last=True, pin_memory=True)

    def batches():
        feed = DevicePrefetcher(loader, dev)
        for b in feed:
            yield b, feed

    stream = batches()

    def sync_all():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    # ---- warm-up (includes cuDNN autotune, graph capture) -------------------------------------------
    for _ in range(max(args.warmup, 5)):
        (x, y), _feed = next(stream)
        step(x, y)
        sched.step()
    torch.cuda.synchronize(dev)

    # ---- (1) device-timed loop: batches already resident on the device -------------------------------
    resident = []
    for _ in range(4):
        (x, y), _feed = next(stream)
        resident.append((x.clone(), y.clone()))
    sync_all()
    sampler_clk = ClockSampler(local_rank)
    if rank == 0:
        sampler_clk.start()
    c0 = C.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all()
    if args.profile_range:
        torch.cuda.profiler.start()
    ev0.record()
    for i in range(args.steps):
        x, y = resident[i % len(resident)]
        loss = step(x, y)
        sched.step()
    ev1.record()
    sync_all()
    if args.profile_range:
        torch.cuda.profiler.stop()
    eager_launches = C.launch_count() - c0
    ms_dev = ev0.elapsed_time(ev1)
    clocks = sampler_clk.stop() if rank == 0 else {}

    # ---- (2) end-to-end loop through the public loader API: H2D every step + D2H loss read every step ---
    e2e = None
    if not args.skip_e2e:
        loss_ring = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(4)]
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        e0.record()
        h2d_bytes = 0
        d2h_bytes = 0
        wait_s = 0.0
        for i in range(args.steps):
            t_w = time.perf_counter()
            (x, y), feed = next(stream)
            wait_s += time.perf_counter() - t_w
            h2d_bytes += x.numel() * x.element_size() + y.numel() * y.element_size()
            loss = step(x, y)
            sched.step()
            slot = loss_ring[i % len(loss_ring)]
            slot.copy_(loss.detach().float().reshape(()), non_blocking=True)     # D2H read of this step's loss
            d2h_bytes += 4
        e1.record()
        sync_all()
        ms_e2e = e0.elapsed_time(e1)
        last_loss = float(loss_ring[(args.steps - 1) % len(loss_ring)])
        e2e = {"ms": ms_e2e, "h2d": h2d_bytes / args.steps, "d2h": d2h_bytes / args.steps, "last_loss": last_loss,
               "loader_wait_ms": wait_s * 1e3 / args.steps}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, inner)         # `loss`: what the last timed step returned

    # ---- reduce over ranks (max time) ---------------------------------------------------------------
    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    ms_dev = max_over_ranks(ms_dev)
    if e2e:
        e2e["ms"] = max_over_ranks(e2e["ms"])
    per_step_graph = step.captured_native_launches
    gpu_launches = int(eager_launches + (per_step_graph * args.steps if step.graph is not None else 0))
    global_batch = args.per_gpu_batch * world
    value = global_batch * args.steps / (ms_dev / 1e3)
    stats = model.ddp_stats() if hasattr(model, "ddp_stats") else {}
    if rank == 0:
        out = {"metric": "samples/sec (whole box, device-timed, max over ranks) for ResNet-50 DDP at 1/2/4/8 B200"
               if args.model == "resnet50" else f"samples/sec {args.model}",
               "impl": "ours", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": (value / BASELINE_PUBLISHED) if BASELINE_PUBLISHED else None,
               "dtype": "bf16" if compute_dtype == torch.bfloat16 else "fp32",
               "data": "synthetic (random-init weights, random ImageNet-shaped batches in pinned host memory)",
               "config": config_dict(args, world, {"transport": backend, "cuda_graph": step.graph is not None,
                                                   "ddp": stats, **opt_ins(inner)}),
               "clocks": clocks, "gpu_launches": gpu_launches,
               "native_launches_per_step": per_step_graph if step.graph is not None else eager_launches / max(1, args.steps)}
        if e2e:
            out["e2e"] = {"value": global_batch * args.steps / (e2e["ms"] / 1e3), "unit": "samples/s",
                          "ms_per_step": e2e["ms"] / args.steps, "h2d_bytes_per_step": e2e["h2d"],
                          "d2h_bytes_per_step": e2e["d2h"], "last_loss": e2e["last_loss"],
                          "host_wait_for_batch_ms_per_step": e2e["loader_wait_ms"]}
        emit(out)
    if args.trace_dir:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(args.trace_dir, exist_ok=True)
        sync_all()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for i in range(4):
                x, y = resident[i % len(resident)]
                step(x, y)
                sched.step()
            sync_all()
        prof.export_chrome_trace(os.path.join(args.trace_dir, f"rank{rank}.json"))
    stream.close()                      # stops the loader's helper thread before interpreter shutdown
    if world > 1:
        try:
            from b200ddp.parallel.peer import PeerCollectives
            PeerCollectives.shutdown_all()
        except Exception:
            pass
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# reference arm: the unmodified template from baseline/_ref
# --------------------------------------------------------------------------------------------------
def run_reference(args):
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isfile(os.path.join(ref_dir, "ddp.py")):
        emit({"impl": "reference", "unavailable": "baseline/_ref is missing: run baseline/install_reference.sh"})
        return
    rank, local_rank, world = dist_env()
    smi_index = str(local_rank)
    if args.gpus == 1 and "LOCAL_RANK" not in os.environ:
        # The reference would otherwise wrap the model in DataParallel over every visible GPU (ddp.py:96-98,189-191).
        # Narrow visibility to ONE device whatever the incoming value is (on an 8-GPU box the variable may already list
        # all eight, so setdefault was a no-op in round 1); must happen before torch initialises CUDA.
        first = (os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[0].strip()) or "0"
        os.environ["CUDA_VISIBLE_DEVICES"] = first
        smi_index = first                      # nvidia-smi -i takes the physical index or the UUID
    import torch
    import torch.nn as nn
    if not torch.cuda.is_available():
        emit({"impl": "reference", "unavailable": "no CUDA device visible"})
        return
    # make `import ddp` resolve to the reference modules, not this repo's same-named entry scripts
    sys.path = [p for p in sys.path if os.path.abspath(p or ".") != ROOT]
    sys.path.insert(0, ref_dir)
    for name in ("ddp", "model", "dataset", "utils"):
        sys.modules.pop(name, None)
    import ddp as ref          # noqa: E402  (reference ddp.py, unmodified)
    assert os.path.abspath(ref.__file__).startswith(ref_dir), ref.__file__
    import torch.utils.data
    import torchvision

    # nothing from this repository's package is imported in this arm: the data set below is the "user's dataset.py"
    # (plain tensors + __getitem__), the model is stock torchvision, the loop / DDP / loader / optimizer are the reference's

    W, K = args.warmup, args.steps
    state = {"calls": 0, "t0": None, "t1": None, "h2d": 0}

    class RefWorkload(nn.Module):
        """User model handed to the reference's train(): stock torchvision ResNet-50, channels_last, bf16 autocast."""

        def __init__(self):
            super().__init__()
            if args.model == "resnet50":
                self.net = torchvision.models.resnet50()
            elif args.model == "resnet152":
                self.net = torchvision.models.resnet152()
            else:
                raise SystemExit("reference arm supports resnet50/resnet152")
            self.net = self.net.to(memory_format=torch.channels_last)

        def forward(self, x):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                return self.net(x.contiguous(memory_format=torch.channels_last)).float()

    def pre_hook(module, inputs):
        # step boundaries = successive forward calls: K full reference steps lie between call W and call W+K
        idx = state["calls"]
        state["calls"] += 1
        if idx == W or idx == W + K:
            if world > 1:
                torch.distributed.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
            # both events on this process' training device (a DataParallel replica thread may have another one current)
            with torch.cuda.device(ns.device if getattr(ns, "device", None) is not None and ns.device.type == "cuda" else torch.cuda.current_device()):
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
            state["t0" if idx == W else "t1"] = ev
            if idx == W:
                state["clock"] = ClockSampler(smi_index)
                if rank == 0:
                    state["clock"].start()
            else:
                torch.cuda.synchronize()
                state["clocks"] = state["clock"].stop() if rank == 0 else {}
        if W <= idx < W + K:
            x = inputs[0]
            state["h2d"] += x.numel() * x.element_size()

    class RefDataset(torch.utils.data.Dataset):
        """ImageNet-shaped synthetic samples with the dense one-hot target the reference's hard-coded MSELoss needs
        (same generator, seed and shapes as b200ddp.data.SyntheticImageNet, re-stated here so this arm imports nothing of ours)."""

        def __init__(self, samples):   # the reference calls FooDataset(100000)
            g = torch.Generator().manual_seed(1234)
            n, size, classes = int(args.samples), int(args.image_size), 1000
            self.X = torch.randn(n, 3, size, size, generator=g)
            labels = torch.randint(0, classes, (n,), generator=g)
            self.Y = torch.zeros(n, classes)
            self.Y[torch.arange(n), labels] = 1.0

        def __len__(self):
            return self.X.shape[0]

        def __getitem__(self, index):
            return self.X[index], self.Y[index]

    if args.model != "foo":
        ref.FooDataset = RefDataset    # dataset.py is the template's customisation point; no source edit

    ns = argparse.Namespace(**{"global_step": 0, "no_cuda": False, "output_dir": "/tmp/ref_outputs", "seed": 42,
                               "gradient_accumulation_steps": 1, "per_gpu_train_batch_size": args.per_gpu_batch,
                               "max_steps": W + K + 1, "logging_steps": 10 ** 9, "save_steps": 0, "num_train_epochs": 10,
                               "warmup_steps": 100, "max_grad_norm": 1000.0, "local_rank": -1, "fp16": False,
                               "loss_scale": 0, "fp16_opt_level": "O2"})
    torch.backends.cudnn.benchmark = True
    cwd = os.getcwd()
    os.makedirs("/tmp/ref_run", exist_ok=True)
    os.chdir("/tmp/ref_run")           # SummaryWriter() writes ./runs
    with contextlib.redirect_stdout(sys.stderr):
        ref.setup(ns)
        if args.model == "foo":
            import model as ref_model_mod          # the reference's own model.py (FooModel) and dataset.py, untouched
            model = ref_model_mod.FooModel()
        else:
            model = RefWorkload()
        model.register_forward_pre_hook(pre_hook)
        ref.train(ns, model)
    os.chdir(cwd)
    ms = state["t0"].elapsed_time(state["t1"])
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t)
    with contextlib.redirect_stdout(sys.stderr):
        ref.cleanup(ns)
    global_batch = args.per_gpu_batch * world
    value = global_batch * K / (ms / 1e3)
    target_bytes = args.per_gpu_batch * (5 if args.model == "foo" else 1000) * 4
    if rank == 0:
        emit({"metric": "samples/sec (whole box, device-timed, max over ranks) for ResNet-50 DDP at 1/2/4/8 B200",
              "impl": "reference", "model": args.model, "value": value, "unit": "samples/s", "n_gpus": world, "steps": K, "warmup": W,
              "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
              "data": "synthetic (random-init weights, random ImageNet-shaped batches via the reference DataLoader, pin_memory)",
              "config": config_dict(args, world, {"transport": "nccl (stock torch DDP)" if world > 1 else "single",
                                                  "cuda_graph": False, "amp": "torch.autocast bf16, fp32 params"}),
              "clocks": state.get("clocks", {}), "gpu_launches": 0,
              "e2e": {"value": value, "unit": "samples/s", "ms_per_step": ms / K,
                      "h2d_bytes_per_step": state["h2d"] / K + target_bytes, "d2h_bytes_per_step": 8,
                      "note": "the reference loop is end to end by construction (DataLoader, blocking .to(device), 2x loss.item())"}})



# --------------------------------------------------------------------------------------------------
# stock arm: plain torch DDP + NCCL + library kernels on the same workload (BASELINE configs 3 and 4)
# --------------------------------------------------------------------------------------------------
def run_stock(args):
    """Competent stock loop (the honest bar next to the host-bound reference loop): torch DDP + NCCL + cuDNN/cuBLAS on
    device-resident batches, bf16 autocast, clip + SGD every step; ``--stock_graph`` additionally captures the whole
    step into one CUDA graph following torch's whole-network-capture recipe for DDP (side-stream construction, 11 eager
    DDP iterations before capture, NCCL async error handling off)."""
    if args.stock_graph:
        os.environ["TORCH_NCCL_ASYNC_ERROR_HANDLING"] = "0"
        os.environ["NCCL_ASYNC_ERROR_HANDLING"] = "0"
    import torch
    import torch.distributed as dist
    import torch.nn as nn
    rank, local_rank, world = dist_env()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=dev)
    torch.manual_seed(42)
    torch.backends.cudnn.benchmark = True
    is_bert = args.model.startswith("bert")
    if is_bert:
        from transformers import BertConfig, BertForMaskedLM
        model = BertForMaskedLM(BertConfig(vocab_size=30528, attn_implementation="sdpa", hidden_dropout_prob=0.0,
                                           attention_probs_dropout_prob=0.0)).to(dev)   # dropout off in both arms
    else:
        import torchvision
        model = getattr(torchvision.models, args.model)().to(dev).to(memory_format=torch.channels_last)
    side = torch.cuda.Stream()
    if world > 1:
        kw = {}
        if args.bucket_cap_mb is not None:
            kw["bucket_cap_mb"] = args.bucket_cap_mb
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            model = nn.parallel.DistributedDataParallel(model, device_ids=[local_rank], gradient_as_bucket_view=args.gradient_as_bucket_view,
                                                        find_unused_parameters=args.find_unused_parameters, **kw)
        torch.cuda.current_stream().wait_stream(side)
    opt = torch.optim.SGD(model.parameters(), lr=1e-3)
    B = args.per_gpu_batch
    if is_bert:
        xs = [torch.randint(0, 30522, (B, 512), device=dev) for _ in range(4)]
        ys = [torch.where(torch.rand(B, 512, device=dev) < 0.15, torch.randint(0, 30522, (B, 512), device=dev), torch.full((B, 512), -100, device=dev)) for _ in range(4)]
    else:
        xs = [torch.randn(B, 3, args.image_size, args.image_size, device=dev) for _ in range(4)]
        ys = [torch.zeros(B, 1000, device=dev) for _ in range(4)]

    def fwd_bwd_step(x, y):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if is_bert:
                loss = model(input_ids=x, labels=y).loss
            else:
                out = model(x.contiguous(memory_format=torch.channels_last)).float()
        if not is_bert:
            loss = nn.functional.mse_loss(out, y)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1000.0)
        opt.step()

    def one(i):
        fwd_bwd_step(xs[i % 4], ys[i % 4])
        opt.zero_grad(set_to_none=True)

    graph, graph_error = None, None
    if args.stock_graph:
        try:
            sx, sy = xs[0].clone(), ys[0].clone()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(max(args.warmup, 12)):          # >= 11 DDP-enabled eager iterations before capture
                    fwd_bwd_step(sx, sy)
                    opt.zero_grad(set_to_none=True)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fwd_bwd_step(sx, sy)
            torch.cuda.synchronize()

            def one(i):                                        # noqa: F811  (replay: copy the batch into the static buffers)
                sx.copy_(xs[i % 4]); sy.copy_(ys[i % 4])
                graph.replay()
        except Exception as exc:
            graph, graph_error = None, f"{type(exc).__name__}: {exc}"[:200]
            raise SystemExit(f"stock CUDA-graph capture failed: {graph_error}")

    for i in range(max(args.warmup, 5)):
        one(i)
    if world > 1:
        dist.barrier(device_ids=[local_rank])
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        one(i)
    e1.record()
    if world > 1:
        dist.barrier(device_ids=[local_rank])
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
        dist.destroy_process_group()
    if rank == 0:
        gb = B * world
        emit({"metric": f"samples/sec {args.model} DDP bf16", "impl": "stock", "value": gb * args.steps / (ms / 1e3), "unit": "samples/s",
              "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
              "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic, device-resident",
              "config": config_dict(args, world, {"transport": "nccl (stock torch DDP)", "bucket_cap_mb": args.bucket_cap_mb,
                                                  "gradient_as_bucket_view": args.gradient_as_bucket_view,
                                                  "find_unused_parameters": args.find_unused_parameters,
                                                  "cuda_graph": graph is not None, "amp": "torch.autocast bf16, fp32 params"})})


def main():
    args = parse_args()
    if args.impl == "reference":
        try:
            run_reference(args)
        except Exception as exc:  # the driver expects a JSON line and exit 0 when the arm cannot run
            import traceback
            traceback.print_exc()
            rank, _, _ = dist_env()
            if rank == 0:
                emit({"impl": "reference", "unavailable": f"{type(exc).__name__}: {exc}"[:300]})
    elif args.impl == "stock":
        run_stock(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
