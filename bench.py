#!/usr/bin/env python
"""bench.py -- train samples/sec of the ViT-B/16 224px bf16 training step (BASELINE.json configs[1] / [2]).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # the B200-native arm (this repo)
  python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU path (oracle port), host cores
  torchrun ... bench.py --gpus N ...                              # one rank per GPU, weak scaling (256 images / GPU)

One step = forward + cross-entropy + backward + (N > 1: bucketed gradient all-reduce) + Adam step on one batch of
synthetic images (randn, fp32 NCHW) and labels (uniform int64), random-init weights of the named architecture.
Rank 0 prints ONE JSON line.  ``value`` is measured with inputs resident in HBM; ``e2e`` goes through the public
module API with pinned HOST buffers, the host->device copy of every step's batch and a device->host read of the loss
inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

FLOP_PER_IMAGE_FWD_BWD = 105_382_969_344  # BASELINE.md section 2 (GEMM-only, 3x forward)
CLIP_FLOP_PER_PAIR_FWD_BWD = 3 * 14_780_000_000  # SURVEY.md 8a row a16: 14.78 GFLOP / pair forward (vision 8.82 + text 5.96)
CONFIG_NAME = "vit_b16"
PER_GPU_BATCH = 256
# N > 1 gradient exchange used by default ("graph" once validated on real multi-GPU boxes; see --dp-mode)
DEFAULT_DP_MODE = "auto"  # graph (in-graph bucketed exchange) for N <= 2, flat (one uncapped all-reduce behind the graph) for N >= 3: see --dp-mode


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(burst=p["bf16_tflops"], sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), hbm=p["hbm_gbs"], source="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, source="fallback")


# ------------------------------------------------------------------------------------------------------------------
# multi-GPU watchdog: a collective that never completes (a dead peer, a rank that took another code path) would otherwise sit in
# an NCCL kernel until the caller's own limit; say where it happened and leave, so the launcher tears the other ranks down
# ------------------------------------------------------------------------------------------------------------------
class Watchdog:
    def __init__(self, seconds: float, rank: int):
        self.phase, self.rank, self.seconds = "start", rank, seconds
        self._timer = None
        if seconds > 0:
            self._timer = threading.Timer(seconds, self._fire)
            self._timer.daemon = True
            self._timer.start()

    def _fire(self):
        sys.stderr.write(f"bench.py: rank {self.rank} made no progress for {self.seconds:.0f} s in phase '{self.phase}' -- aborting "
                         f"(B200_BENCH_WATCHDOG_S=0 disables; --dp-mode flat / torch select other gradient-exchange schedules)\n")
        sys.stderr.flush()
        os._exit(3)

    def enter(self, phase: str):
        self.phase = phase
        if self._timer is not None:  # every phase gets the full allowance
            self._timer.cancel()
            self._timer = threading.Timer(self.seconds, self._fire)
            self._timer.daemon = True
            self._timer.start()

    def done(self):
        if self._timer is not None:
            self._timer.cancel()
            self._timer = None


# ------------------------------------------------------------------------------------------------------------------
# clocks sampler (pynvml; nvidia-smi fields of the profiling recipe)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # pragma: no cover
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle (pinned bit-for-bit to the reference) on the host cores
# ------------------------------------------------------------------------------------------------------------------
def cpu_reference_samples_per_sec(steps: int, warmup: int, budget_s: float):
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vit_oracle as vo

    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        usable = os.cpu_count() or 1
    cfg = vo.vit_config(CONFIG_NAME)
    # "all the host threads it can use": on the shared GPU hosts 128 logical CPUs are visible but oversubscribing them
    # is slower than using fewer, so a few short probes pick the fastest thread count (reported as `cores`)
    cores = usable
    if usable > 16:
        probe_sd = vo.init_state_dict(cfg, seed=0, perturb=False)
        px, py = vo.synthetic_batch(cfg, 4, seed=0)
        best = None
        for n in sorted({usable, max(1, usable // 2), max(1, usable // 4), 16}, reverse=True):
            torch.set_num_threads(n)
            pp = {k: v.clone().requires_grad_(True) for k, v in probe_sd.items()}
            vo.cross_entropy(vo.classifier_forward(pp, px, cfg), py).backward()  # warm
            t0 = time.perf_counter()
            vo.cross_entropy(vo.classifier_forward(pp, px, cfg), py).backward()
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, n)
        cores = best[1]
    torch.set_num_threads(cores)
    sd = vo.init_state_dict(cfg, seed=0, perturb=False)
    params = [v.clone().requires_grad_(True) for v in sd.values()]
    keys = list(sd.keys())
    opt = torch.optim.Adam(params, lr=1e-3)

    def step(x, y):
        # fp32: CPU bf16 autocast is slower than fp32 (SURVEY.md section 6), so fp32 is the reference's best CPU path
        pd = dict(zip(keys, params))
        loss = vo.cross_entropy(vo.classifier_forward(pd, x, cfg), y)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    # calibrate the bounded sample (micro-batch) so that (steps + warmup) steps fit the time budget
    x, y = vo.synthetic_batch(cfg, 16, seed=0)
    step(x, y)  # cold step (thread pool spin-up, allocator): not representative
    t0 = time.perf_counter()
    step(x, y)
    per_img = (time.perf_counter() - t0) / 16
    # many-core hosts need a reasonably large micro-batch to use their threads; keep it within the time budget
    mb = int(max(8, min(64, budget_s / max(1e-6, per_img * (steps + warmup)))))
    x, y = vo.synthetic_batch(cfg, mb, seed=1)
    for _ in range(warmup):
        step(x, y)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(x, y)
    dt = time.perf_counter() - t0
    return mb * steps / dt, dt / steps * 1e3, mb, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    v, ms, mb, cores = cpu_reference_samples_per_sec(args.steps, max(1, args.warmup), budget_s=150.0)
    sample = f"micro-batch {mb} images x {args.steps} steps, fp32, torch CPU, {cores} threads"
    line = {
        "impl": "reference", "metric": "train samples/sec, ViT-B/16 224px, fwd+bwd+adam step", "value": round(v, 3),
        "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "ViT-B/16 classifier 224x224, 1000 classes (BASELINE.json configs[1])", "micro_batch": mb},
        "cpu_baseline": {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": round(v, 3), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# N > 1: gradient parity of the data-parallel path that is about to be timed (small config, every run)
# ------------------------------------------------------------------------------------------------------------------
def dp_gradient_parity(comm, rank, world, dev, flat=False):
    """Runs the SAME graphed DP step the bench times (in-graph bucketed all-reduce over the native communicator) on a small
    ViT with each rank's shard of a global batch, and compares the averaged gradients with a single-process run over the
    whole batch on rank 0 (SURVEY.md 8e: all-reduced grads == global-batch mean-loss grads).  Returns the relative L2
    difference (rank 0; other ranks None) -- bf16 rounding of shard-wise weight gradients sets a floor of ~2e-3."""
    import torch
    import torch.distributed as dist

    from cflearn_b200 import dp, registry
    from cflearn_b200.optim import ArenaAdam, GraphedTrainStep

    cfgs = dict(in_channels=3, num_classes=24, img_size=64, latent_dim=256, encoder="vit", encoder_config=dict(patch_size=16, num_layers=3))
    per_rank = 8
    gen = torch.Generator().manual_seed(77)
    x = torch.randn(per_rank * world, 3, 64, 64, generator=gen)
    y = torch.randint(0, 24, (per_rank * world, 1), generator=gen)
    torch.manual_seed(5)
    m = registry.build_module("cv_clf", config=cfgs).to(dev)
    with torch.no_grad():  # biases / LayerNorm parameters off their 0 / 1 initial values
        for k, p in m.named_arena_parameters():
            if k.endswith("bias") or "norm" in k:
                p.add_(0.05 * torch.randn_like(p))
    dp.broadcast_parameters(m)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    opt = ArenaAdam(m, lr=0.0, capturable=True)  # lr 0: the step leaves the parameters alone, the gradient arena is what we read
    gs = GraphedTrainStep(m, opt, per_rank, comm=comm, flat=flat)
    idx = list(dp.shard_indices(per_rank * world, rank, world))
    gs.step(x[idx].to(dev), y[idx].to(dev))
    torch.cuda.synchronize()
    g_dp = m.arena.grad.clone()
    ref = g_dp.clone()
    dist.broadcast(ref, src=0)
    same = torch.equal(ref, g_dp)
    flags = torch.tensor([1.0 if same else 0.0], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if flags.item() != 1.0:
        raise SystemExit("bench.py: ranks disagree on the all-reduced gradients")
    rel = None
    if rank == 0:
        single = registry.build_module("cv_clf", config=cfgs).to(dev)
        single.load_state_dict(sd, strict=True)
        single.train_step(x.to(dev), y.to(dev))
        torch.cuda.synchronize()
        g_one = single.arena.grad
        rel = ((g_dp - g_one).norm() / g_one.norm()).item()
        if not rel < 5e-3:
            raise SystemExit(f"bench.py: data-parallel gradient parity failed: rel L2 {rel:.3e} >= 5e-3")
    m.engine.reducer = None
    gs.release()  # (a graph that captured the communicator must be gone before the communicator is closed)
    del gs, m
    return rel


# ------------------------------------------------------------------------------------------------------------------
# the real bar (BASELINE.md section 3): the reference path in PyTorch eager on the SAME GPU(s), torch DDP at N > 1
# ------------------------------------------------------------------------------------------------------------------
def eager_gpu_leg(rank, world, dev, steps, warmup):
    """The oracle port (pinned bit-for-bit to the reference's modules, oracle/vit_oracle.py) under torch.autocast(bf16) on
    CUDA: forward + cross-entropy + backward + torch's fused Adam, batch 256 per GPU, CUDA events; at N > 1 wrapped in
    torch DistributedDataParallel over NCCL (what accelerate.prepare gives the reference, cflearn/trainer.py:266-273).
    A BASELINE leg: nothing of the product is on this path, and the product never imports the oracle."""
    import torch
    import torch.distributed as dist

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vit_oracle as vo

    cfg = vo.vit_config(CONFIG_NAME)
    sd = vo.init_state_dict(cfg, seed=0, perturb=False)
    keys = list(sd.keys())

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.ps = torch.nn.ParameterList([torch.nn.Parameter(sd[k].clone()) for k in keys])

        def forward(self, x):
            return vo.classifier_forward(dict(zip(keys, self.ps)), x, cfg)

    net = Net().to(dev)
    mod = torch.nn.parallel.DistributedDataParallel(net, device_ids=[dev.index]) if world > 1 else net
    opt = torch.optim.Adam(net.parameters(), lr=1e-3, fused=True)
    B = PER_GPU_BATCH
    x = torch.randn(B, 3, 224, 224, device=dev)
    y = torch.randint(0, 1000, (B, 1), device=dev)

    def step():
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            loss = vo.cross_entropy(mod(x), y)
        loss.backward()
        opt.step()

    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    del mod, net, opt, x, y
    torch.cuda.empty_cache()
    return {"value": round(world * B * steps / (ms / 1e3), 1), "unit": "samples/s", "ms_per_step": round(ms / steps, 3), "steps": steps,
            "impl": "oracle port of the reference modules (pinned bit-for-bit), PyTorch eager, bf16 autocast, fused torch Adam"
                    + (", torch DDP over NCCL" if world > 1 else ""), "torch": torch.__version__}


# ------------------------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step handed its caller, for output-for-output comparison of two builds
# ------------------------------------------------------------------------------------------------------------------
DUMP_SAMPLE = 1 << 21  # values kept per dumped array (8 MB in float32); at most 6 arrays -> under 64 MB in all


def dump_outputs(out_dir, loss, arenas):
    """Writes ``loss.npy`` (the step's loss) and, per parameter arena ``name``, ``<name>params.npy`` (the parameters after the
    step's Adam update) and ``<name>grads.npy`` (the step's gradients), all float32.  An arena longer than DUMP_SAMPLE is
    cut to DUMP_SAMPLE values at positions drawn from a fixed seed, the same positions on every run."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss.detach().reshape(1)}
    for name, a in arenas:
        arrays[f"{name}params"], arrays[f"{name}grads"] = a.flat, a.grad
    for name, t in arrays.items():
        t = t.detach().reshape(-1)
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    import cflearn_b200  # noqa: F401
    from cflearn_b200 import _cabi, dp, ops, registry
    from cflearn_b200.optim import ArenaAdam

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU path)")
    if not _cabi.available():
        raise SystemExit(f"bench.py: {_cabi.load_error()}")
    info = dp.ddp_info()
    rank, world, local = info if info is not None else (0, 1, 0)
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py: --gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # N > 1 only: no phase of a healthy run takes anywhere near this long, even on a cold box
    dog = Watchdog(float(os.environ.get("B200_BENCH_WATCHDOG_S", "300")) if world > 1 else 0.0, rank)
    if world > 1:
        dog.enter("init_process_group")
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)
    is_clip = args.config == "clip"
    if is_clip:  # BASELINE.json configs[3]: CLIP() defaults = ViT-B/32 vision tower + 12 x 512 text tower, context 77, vocab 49,408
        model = registry.build_module("clip").to(dev)
    else:
        model = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=1000, img_size=224, latent_dim=768, encoder="vit",
                                                            encoder_config=dict(patch_size=16, num_layers=12))).to(dev)
    for a in (model.arenas() if is_clip else [model.arena]):
        a.ensure()
    comm = None
    dp_parity = None
    if world > 1:
        # the library's own NCCL communicator (csrc/comm.cu): its all-reduces are plain stream operations, so the bucketed
        # exchange is captured INSIDE the step's CUDA graph on a forked stream, overlapped with the remaining backward
        # (flat: nothing overlaps the all-reduce, so the communicator is not capped to a few CTAs)
        dog.enter("communicator init + gradient parity check")
        comm = (dp.TorchComm(rank, world, dev) if args.dp_mode == "torch" else
                dp.NativeComm(rank, world, dev, max_ctas=0 if args.dp_mode == "flat" and "B200_COMM_CTAS" not in os.environ else None))
        dp.broadcast_parameters(model)
        dp_parity = dp_gradient_parity(comm, rank, world, dev, flat=args.flat_allreduce)  # (the ViT path's reducer; CLIP reuses it per tower)
    use_graph = not args.no_graph
    opt = ArenaAdam(model, lr=1e-3, capturable=use_graph)
    B = PER_GPU_BATCH
    g = torch.Generator(device="cpu").manual_seed(1000 + rank)  # rank r uses its own data seed (BASELINE.md section 4)
    n_host = 2
    host_x = [torch.randn(B, 3, 224, 224, generator=g).pin_memory() for _ in range(n_host)]
    if is_clip:  # SURVEY.md 8d config 4: ids uniform in [1, V-2], EOS (= V-1, the arg-max id) forced at a random position >= 1
        host_y = []
        for _ in range(n_host):
            ids = torch.randint(1, 49407, (B, 77), generator=g)
            ids[torch.arange(B), torch.randint(1, 77, (B,), generator=g)] = 49407
            host_y.append(ids.pin_memory())
    else:
        host_y = [torch.randint(0, 1000, (B, 1), generator=g).pin_memory() for _ in range(n_host)]
    dev_x = [h.to(dev) for h in host_x]
    dev_y = [h.to(dev) for h in host_y]

    dog.enter("graph capture")
    gstep = None
    if use_graph:  # zero_grad + fwd + loss + bwd + (N > 1: per-block bucket all-reduces on a forked stream) + Adam as ONE CUDA graph
        from cflearn_b200.optim import GraphedTrainStep

        static_inputs = [torch.zeros_like(dev_x[0]), torch.zeros_like(dev_y[0])] if is_clip else None
        gstep = GraphedTrainStep(model, opt, B, comm=comm, flat=args.flat_allreduce, inputs=static_inputs)
    elif world > 1:
        dp.attach_native_reducers(model, comm)

    def do_step(x, y):
        if gstep is not None:
            return gstep.step(x, y)
        opt.zero_grad()  # schema.py:984 (backward then overwrites the gradient arena instead of accumulating)
        loss = model.train_step(x, y)  # N > 1: the native bucket reducer all-reduces inside backward
        opt.step()
        return loss

    def step_resident(i):
        return do_step(dev_x[i % n_host], dev_y[i % n_host])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    # ---- device-resident timing ---------------------------------------------------------------------------------
    dog.enter("warm-up + timed steps")
    for i in range(args.warmup):
        step_resident(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = _cabi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = step_resident(i)
    e1.record()
    barrier()
    launches = _cabi.launch_count() - launches0  # (flat / torch exchange: the Adam launches behind each replay are counted here)
    if gstep is not None:  # graph replays launch the captured kernels without going through the host-side counter
        launches += gstep.launches_per_replay * args.steps
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop()
    ms_step = ms_total / args.steps
    value = world * B * args.steps / (ms_total / 1e3)
    final_loss = loss.item()
    if not (final_loss == final_loss and abs(final_loss) < 1e4):
        raise SystemExit(f"bench.py: loss diverged ({final_loss})")
    if args.dump_outputs and rank == 0:  # before the end-to-end steps below move the parameters on
        dump_outputs(args.dump_outputs, loss, zip(("vit_", "text_", "glue_"), model.arenas()) if is_clip else [("", model.arena)])

    dog.enter("end-to-end steps")
    # ---- end to end: pinned host batches -> H2D on a copy stream (prefetched one step ahead) -> step -> loss D2H --
    copy_stream = torch.cuda.Stream()
    stage_x = [torch.empty_like(dev_x[0]) for _ in range(2)]
    stage_y = [torch.empty_like(dev_y[0]) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            stage_x[s].copy_(host_x[i % n_host], non_blocking=True)
            stage_y[s].copy_(host_y[i % n_host], non_blocking=True)
            ready[s].record(copy_stream)

    loss_dev = [torch.zeros(1, device=dev) for _ in range(2)]
    loss_pinned = [torch.zeros(1).pin_memory() for _ in range(2)]
    losses_seen = []

    def e2e_loop(n):
        pending = None
        for s in range(2):
            consumed[s].record(torch.cuda.current_stream())
        prefetch(0)
        for i in range(n):
            s = i % 2
            if i + 1 < n:
                prefetch(i + 1)
            torch.cuda.current_stream().wait_event(ready[s])
            ls = do_step(stage_x[s], stage_y[s])
            consumed[s].record(torch.cuda.current_stream())
            # device->host read of the loss every step (the reference's per-step .item(), models/common.py:42); the
            # read of step i is waited for after step i+1 has been queued so the GPU never idles on the host
            loss_dev[i % 2].copy_(ls.reshape(1))
            if pending is not None:
                pending[0].synchronize()
                losses_seen.append(float(loss_pinned[pending[1]][0]))
            loss_pinned[i % 2].copy_(loss_dev[i % 2], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            pending = (ev, i % 2)
        if pending is not None:
            pending[0].synchronize()
            losses_seen.append(float(loss_pinned[pending[1]][0]))

    e2e_loop(max(1, min(3, args.warmup)))
    barrier()
    t0 = time.perf_counter()
    e0.record()
    e2e_loop(args.steps)
    e1.record()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), wall_ms))
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)
    h2d = host_x[0].numel() * 4 + host_y[0].numel() * 8
    d2h = 4

    flop_per_sample = CLIP_FLOP_PER_PAIR_FWD_BWD if is_clip else FLOP_PER_IMAGE_FWD_BWD
    # ---- roofline: every heavy kernel of the step timed ALONE at its bench shape (CUDA events on the launching stream);
    # `roofline` proper names the top-time kernel of the step's launch list (profiles/r0X_step_launches.md): the split-K
    # weight-gradient GEMM gemm_bf16_kernel<EPI_PARTIAL_F32> at the FeedForward shape; the others are listed beside it ------
    peaks = _peaks()
    M, D_, FF_, H_ = B * 197, 768, 3072, 12

    def bf(*shape, scale=1.0):
        return (torch.randn(*shape, device=dev) * scale).to(torch.bfloat16)

    x768, x3072, hpre = bf(M, D_), bf(M, FF_), bf(M, FF_)
    w_qkv, w_1, w_2 = bf(3 * D_, D_, scale=0.02), bf(FF_, D_, scale=0.02), bf(D_, FF_, scale=0.02)
    b_qkv, b_1, b_o = bf(3 * D_, scale=0.02), bf(FF_, scale=0.02), bf(D_, scale=0.02)
    resid = torch.randn(M, D_, device=dev)
    o_qkv = torch.empty(M, 3 * D_, device=dev, dtype=torch.bfloat16)
    o_ff0, o_ff1 = torch.empty(M, FF_, device=dev, dtype=torch.bfloat16), torch.empty(M, FF_, device=dev, dtype=torch.bfloat16)
    o_res = torch.empty(M, D_, device=dev, dtype=torch.float32)
    splits = ops.pick_splits(FF_, D_, M)
    part = torch.empty(splits, FF_, D_, device=dev, dtype=torch.float32)
    qkv = bf(B, 197, 3 * D_)
    att_o, att_lse = ops.attention_fwd(qkv, B, 197, H_)
    att_do = bf(M, D_)
    att_dqkv = torch.empty(M, 3 * D_, device=dev, dtype=torch.bfloat16)

    def time_kernel(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(reps):
            fn()
        k1.record()
        torch.cuda.synchronize()
        return k0.elapsed_time(k1) / reps

    gf = 2.0 * M * FF_ * D_
    kernels = [
        ("gemm_bf16_kernel<EPI_PARTIAL_F32> wgrad dW1 = dh^T.ln2 3072x768x50432 split-K", gf,
         lambda: ops.gemm(x3072, x768, a_mn_major=True, b_mn_major=True, epilogue=ops.EPI_PARTIAL_F32, out0=part, splits=splits)),
        ("gemm_bf16_kernel<EPI_BIAS_BF16> qkv 50432x2304x768", 2.0 * M * 3 * D_ * D_, lambda: ops.gemm(x768, w_qkv, bias=b_qkv, out0=o_qkv)),
        ("gemm_bf16_kernel<EPI_BIAS_GELU_BF16> ff1 50432x3072x768", gf,
         lambda: ops.gemm(x768, w_1, bias=b_1, epilogue=ops.EPI_BIAS_GELU_BF16, out0=o_ff0, out1=o_ff1)),
        ("gemm_bf16_kernel<EPI_BIAS_RESID_F32> ff2 50432x768x3072", gf,
         lambda: ops.gemm(x3072, w_2, bias=b_o, epilogue=ops.EPI_BIAS_RESID_F32, aux=resid, out0=o_res)),
        ("gemm_bf16_kernel<EPI_DGELU_BF16> ff2-dgrad 50432x3072x768", gf,
         lambda: ops.gemm(x768, w_2, b_mn_major=True, epilogue=ops.EPI_DGELU_BF16, aux=hpre, out0=o_ff0)),
        ("attn_fwd2_kernel B256 T197 H12 (per-shape default)", 4.0 * B * H_ * 197 * 197 * 64, lambda: ops.attention_fwd(qkv, B, 197, H_)),
        ("attn_bwd2_kernel<PP=false> B256 T197 H12 (per-shape default)", 10.0 * B * H_ * 197 * 197 * 64,
         lambda: ops.attention_bwd(qkv, att_o, att_do, att_lse, B, 197, H_, dqkv=att_dqkv)),
    ]
    timed = []
    for name, flops, fn in kernels:
        k_ms = time_kernel(fn)
        tf = flops / (k_ms * 1e-3) / 1e12
        timed.append({"kernel": name, "kernel_ms": round(k_ms, 4), "achieved": round(tf, 1), "frac": round(tf / peaks["burst"], 4)})
    del x768, x3072, hpre, o_qkv, o_ff0, o_ff1, o_res, part, qkv, att_o, att_do, att_dqkv
    step_tflops = flop_per_sample * B / (ms_step * 1e-3) / 1e12
    traffic, traffic_note = None, "no ncu --set full capture of this build's kernel committed yet"
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")  # written from the committed capture by tools/ncu_summary.py
    if os.path.isfile(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic, traffic_note = tj.get("wgrad_ff1_bytes_per_launch"), tj.get("note", "")
    top = timed[0]
    roofline = {
        "bound": "tensor", "kernel": top["kernel"], "achieved": top["achieved"], "peak": peaks["burst"], "unit": "TFLOP/s",
        "frac": top["frac"], "kernel_ms": top["kernel_ms"],
        "why_this_kernel": "top-time kernel of the step's ncu launch list (profiles/): the split-K wgrad GEMM variant",
        "traffic": traffic, "traffic_note": traffic_note,
        "peak_source": f"{peaks['source']} MEASURED_PEAKS.json bf16_tflops (burst; kernel timed alone)",
        "others": timed[1:],
        "step": {"achieved": round(step_tflops, 1), "peak": peaks["sustained"], "frac": round(step_tflops / peaks["sustained"], 4),
                 "note": f"whole step, GEMM-only FLOPs {flop_per_sample / 1e9:.2f} GFLOP/sample (3x forward), vs sustained cuBLAS bf16 peak"},
    }

    # ---- the real bar: the reference path in PyTorch eager on the same GPU(s) (DDP at N > 1), same run ---------------
    dog.enter("per-kernel timing + eager DDP leg")
    eager = None
    if not args.no_eager_baseline and not is_clip:
        if gstep is not None:
            gstep.release()
            gstep = None  # free the graph's private pool (~17 GB) before eager allocates its ~40 GB of activations
        torch.cuda.empty_cache()
        eager = eager_gpu_leg(rank, world, dev, steps=min(args.steps, 10), warmup=3)
        eager["speedup_of_value"] = round(value / eager["value"], 3)

    # ---- CPU baseline (rank 0, N == 1 only): the oracle on the host cores, bounded sample -------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, ms, mb, cores = cpu_reference_samples_per_sec(2, 1, budget_s=20.0)
        cpu = {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": "port",
               "sample": f"micro-batch {mb} images x 2 steps (fp32 oracle port of the reference path, torch CPU, {cores} threads)"}

    if rank == 0:
        line = {
            "metric": ("train pairs/sec, CLIP ViT-B/32 + text transformer, contrastive fwd+bwd+adam step" if is_clip else
                       "train samples/sec, ViT-B/16 224px, fwd+bwd+adam step"), "value": round(value, 1), "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": ("CLIP ViT-B/32 + 12x512 text transformer (ctx 77, vocab 49408), symmetric cross-entropy over the local batch, "
                                    "256 image-text pairs per GPU (BASELINE.json configs[3])" if is_clip else
                                    "ViT-B/16 classifier 224x224, 1000 classes, batch 256 per GPU (BASELINE.json configs[1]/[2])"),
                       "global_batch": world * B, "seq_len": "50 / 77" if is_clip else 197, "parallelism": f"dp{world}",
                       "optimizer": "adam (fused arena kernel, inside the timed region)",
                       "cuda_graph": bool(use_graph),
                       "gradient_exchange": (None if world == 1 else {
                           "graph": "per-block bucket all-reduces (library-owned NCCL communicator) captured inside the step graph on a forked stream",
                           "flat": "one flat all-reduce on the library-owned NCCL communicator behind the graph",
                           "torch": "one flat torch.distributed all-reduce behind the graph"}[args.dp_mode]),
                       "l2": "per-step working set (> 15 GB of activations) exceeds the 126 MB L2; no explicit flush needed"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": round(e2e_value, 1), "unit": "samples/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": round(e2e_ms / args.steps, 3)},
            "roofline": roofline, "cpu_baseline": cpu, "eager_gpu": eager, "dp_parity_rel": dp_parity, "loss": round(final_loss, 4),
        }
        print(json.dumps(line), flush=True)
    dog.enter("teardown")
    if gstep is not None:  # ncclCommDestroy waits for every graph that captured the communicator: destroy the graph first
        gstep.release()
        gstep = None
    if comm is not None:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        comm.close()
    if world > 1:
        dist.destroy_process_group()
    dog.done()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="vit", choices=["vit", "clip"], help="vit: BASELINE.json configs[1]/[2] (the metric); clip: configs[3]")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--dp-mode", default=os.environ.get("B200_DP_MODE", DEFAULT_DP_MODE), choices=["auto", "graph", "flat", "torch"],
                    help="N > 1 gradient exchange: graph = per-block bucket all-reduces on the library's own NCCL communicator, captured "
                         "inside the step graph and overlapped with backward; flat = same communicator (uncapped), ONE all-reduce behind the "
                         "graph; torch = torch.distributed, one all-reduce behind the graph (round 1's schedule); auto = graph for N <= 2, "
                         "flat for N >= 3 (measured: graph 0.990 at N = 2 but 0.894 at N = 8, DESIGN.md section 4)")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the PyTorch-eager-on-GPU baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss, updated parameters and gradients to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dp_mode == "auto":
        args.dp_mode = "graph" if int(os.environ.get("WORLD_SIZE", "1")) <= 2 else "flat"
    args.flat_allreduce = args.dp_mode in ("flat", "torch")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
