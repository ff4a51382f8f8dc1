#!/usr/bin/env python
"""bench.py -- headline benchmark of the ray-marched NeRF step (BASELINE.json: train rays/s & render Msamples/s on a
lego-shape 800x800 synthetic scene at 1/2/4/8 B200, % of roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); training shards RAYS (4096 per GPU, weak scaling) with one
exchange of the hash-grid + MLP gradients per step.  A "step" is one full training step of configs[1]:
near/far -> march_rays_train -> hash-grid encode -> sigma MLP -> SH -> colour MLP -> composite -> MSE -> backward of
all of it -> Adam, under fp16 autocast exactly as `-O` runs it.  One JSON line is printed by rank 0.

Besides the headline (`value`, `e2e`, `roofline`, `cpu_baseline`) the line carries
  render          one 800x800 view on the reference's round schedule (bit-identical sample positions), the fast schedule beside it
  configs         BASELINE.json configs 3-5: flower-shape training (ray-sharded at N > 1), bonsai-shape bound-16 test view
                  (tile-sharded), edit stage (view-sharded distillation renders + data-parallel style-network steps)
  gpu_reference   the reference's OWN stack on the same GPU in the same process: its Python callers (nerf/renderer.py run_cuda,
                  network_ff.py / network.py, staged untouched under oracle/_ref/py) on its own extensions (oracle/_ref/*.so) --
                  the `--ff` stack, the default `-O` stack (nn.Linear MLPs) and the host-loop render -- with `vs_gpu_reference`
  roofline_large  march / encode / composite at 65 536 rays (~4 M samples), the regime where an HBM roofline is meaningful

`--impl reference` times the CPU arm: the PyTorch-CPU restatement of the reference's non-cuda_ray renderer
(oracle/cpu_renderer.py, BASELINE.json configs[0]) on the host cores, same metric and unit, exactly K timed steps.

`--dump-outputs DIR` writes what the last of the K timed steps returned -- loss, image, depth (of the rays that enter the box),
weights_sum, nears, num_points -- as DIR/<name>.npy.  Scenes, batches and initial weights are seeded, so two builds run with the
same arguments can be compared output for output (up to the run-to-run order of the fp16 atomic gradient sums).  The step is the
graph-replayed one that `value` times, so with the look-ahead pipeline (the default) the loss and per-ray results are those of
the batch handed to the step before the last, and with N > 1 they are rank 0's shard of the rays.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_RAYS = 4096
_OUT = sys.stdout
WORKLOAD = "lego-shape 800x800 hash-grid NeRF training step (16 levels, 2^19 table, 4096 rays/GPU, cuda_ray, fp16 autocast, Adam)"

# algorithmic bytes / FLOPs per unit (SURVEY.md section 8d; restated in DESIGN.md section 8)
ALGO = {
    "lnrf_march_rays_train": dict(bound="hbm", per_ray=48, per_sample=32),
    "lnrf_march_rays_train_clipped": dict(bound="hbm", per_ray=48, per_sample=32),   # the same kernel, rays ending at the occupied box
    "lnrf_grid_encode_forward": dict(bound="hbm", per_ray=0, per_sample_padded=588),
    "lnrf_grid_encode_backward": dict(bound="hbm", per_ray=0, per_sample_padded=588),
    "lnrf_grid_encode_forward_world": dict(bound="hbm", per_ray=0, per_sample_padded=588),   # same kernels, world-coordinate inputs
    "lnrf_grid_encode_backward_world": dict(bound="hbm", per_ray=0, per_sample_padded=588),
    "lnrf_composite_rays_train_forward": dict(bound="hbm", per_ray=32, per_sample=24),
    "lnrf_composite_rays_train_backward": dict(bound="hbm", per_ray=44, per_sample=40),
    # row f-5: composite + blend + depth normalisation + MSE in one launch (gt 12 + image_raw 12 + nears/fars 8 B/ray on top)
    "lnrf_composite_loss_train_forward": dict(bound="hbm", per_ray=64, per_sample=24),
    "lnrf_composite_loss_train_backward": dict(bound="hbm", per_ray=60, per_sample=40),
    # forward + backward of the tail in one launch: the samples are read once from DRAM (24 B), the gradients written (16 B)
    "lnrf_composite_loss_train_forward_backward": dict(bound="hbm", per_ray=64, per_sample=40),
    "lnrf_ffmlp_forward": dict(bound="tensor", flops_per_sample_padded=36864 / 2),   # mean of sigma (14336) and colour (22528) nets
    "lnrf_ffmlp_backward": dict(bound="tensor", flops_per_sample_padded=73728 / 2),
    "lnrf_sh_encode_forward": dict(bound="hbm", per_ray=0, per_sample_padded=12 + 64),
    "lnrf_near_far_from_aabb": dict(bound="hbm", per_ray=32, per_sample=0),
    # fused rows f-1 / f-4 (one C-ABI call each)
    "lnrf_nerf_forward": dict(bound="tensor", flops_per_sample_padded=36864),
    "lnrf_nerf_backward": dict(bound="tensor", flops_per_sample_padded=73728),
    # round 2: lean forward (keeps only h) + recompute backward (csrc/nerfbwd.cu); the algorithmic FLOPs stay the contract's figures
    # (the recomputed forward layers are overhead, not credited)
    "lnrf_nerf_forward_lean": dict(bound="tensor", flops_per_sample_padded=36864),
    "lnrf_nerf_backward_recompute": dict(bound="tensor", flops_per_sample_padded=73728),
    "lnrf_adam_step": dict(bound="hbm", per_param=30),            # g16 R+W 4, p/m/v R+W 24, p16 W 2
    "lnrf_grad_nonfinite_check": dict(bound="hbm", per_param=2),
    "lnrf_grad_nonfinite_check_amp_update": dict(bound="hbm", per_param=2),   # the same pass + GradScaler.update() by the last block
}


# The unit that bounds a kernel when it is neither of the two the contract's `bound` can name; figures from the ncu captures under
# profiles/ (DESIGN.md sections 4, 5, 11)
LIMITERS = {
    "lnrf_nerf_backward_recompute": "TMEM read port (64 B/clk/SM, B300_MICROARCH.md): every MMA step's 128 x 64 fp32 accumulator leaves TMEM through it "
                                    "(512 cycles); 37.9 B/clk/SM sustained over the kernel = 84 % of the two-tile-set roofline inside the tile loop "
                                    "(scripts/diag_bwd_steps.py); tensor pipe 22 %, DRAM 65 MB per call (profiles/r2a_stalls_nerf_bwd.txt, r2e_kernels.txt)",
    "lnrf_nerf_forward_lean": "TMEM read port: 634 cycles per 64-column step against a floor of 512; tensor pipe 24 % (profiles/r2e_kernels.txt)",
    "lnrf_grid_encode_backward_world": "L2 atomic units: ~16 M sector reductions (red.global.add.f16x2 / .v2.f16x2) per call at ~88 per clock, L2 hit 62 %, "
                                       "DRAM 39 MB (5 % of peak), issue 35 % (profiles/r2e_kernels.txt); `frac` is the algorithmic 588 B/sample over HBM peak",
    "lnrf_grid_encode_forward_world": "L1TEX gather rate: 128 gathers per sample, issue 57 %, 82 % warps active, DRAM 24 MB per call (profiles/r2e_kernels.txt)",
    "lnrf_march_rays_train_clipped": "issue / latency of the longest ray of a block (one warp per ray, issue 47 %, 38 % warps active); moves 8 MB: not a bandwidth kernel",
    "lnrf_composite_loss_train_forward_backward": "latency: 4096 warps in one wave, three dependent round trips per ray; 6 MB of DRAM traffic per call",
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=float(d["hbm_gbs"]), tensor_burst=float(d["bf16_tflops"]), tensor=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])),
                    source="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


class TimedLib:
    """Proxy around the ctypes library that brackets selected entry points with CUDA events on the launching stream
    (per-kernel durations measured live inside the timed region, as the roofline contract asks)."""

    def __init__(self, lib, names, torch):
        self._lib, self._names, self._torch = lib, set(names), torch
        self.events = {n: [] for n in names}
        self.enabled = False

    def reset(self):
        self.events = {n: [] for n in self._names}

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name not in self._names:
            return fn

        def wrapped(*a):
            if not self.enabled:
                return fn(*a)
            torch = self._torch
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a)
            e1.record()
            self.events[name].append((e0, e1))
            return r
        return wrapped

    def summary(self):
        out = {}
        for n, ev in self.events.items():
            if ev:
                ms = [a.elapsed_time(b) for a, b in ev]
                out[n] = dict(calls=len(ms), mean_ms=sum(ms) / len(ms), total_ms=sum(ms))
        return out


def base_config(world):
    """The static part of `config` (identical in both arms)."""
    return {"workload": WORKLOAD, "rays_per_gpu": N_RAYS,
            "l2": "no explicit flush: one step touches ~245 MB (fp32 table + grads + Adam moments + fp16 copies) > 126 MB L2",
            "parallelism": (f"ray-sharded dp{world}: the fp16 hash-grid + MLP gradients are averaged over NVLink peer memory, Adam runs on a "
                            f"1/{world} slice per rank, the new fp16 values are stored into every rank's table (ZeRO-1 style, one kernel)")
            if world > 1 else "single GPU"}


def run_reference(args, rank, world):
    """CPU arm: oracle/cpu_renderer.py (PyTorch-CPU port of NeRFRenderer.run + nn.Linear NeRFNetwork, freq encodings), all host
    cores, EXACTLY --steps timed steps after --warmup untimed ones, each step a bounded sample of the 4096-ray batch."""
    if rank != 0:
        return
    import torch
    from cases import scene_rays
    from oracle import cpu_renderer
    steps, warm = args.steps, args.warmup
    # ~0.15 ms per ray-step on 16 cores: keep the whole run near 30 s whatever K is
    n = int(os.environ.get("LNRF_CPU_RAYS", str(max(256, min(2048, int(200_000 / max(1, steps + warm)) // 128 * 128)))))
    sc, ro, rd, rng = scene_rays("lego", n, 0)
    gt = torch.rand(n, 3, generator=torch.Generator().manual_seed(0))
    sec, threads, used = cpu_renderer.time_train_steps(torch.from_numpy(ro), torch.from_numpy(rd), gt, steps=steps, warmup=warm,
                                                       num_steps=512, bound=sc.bound, min_near=sc.min_near)
    value = used / sec
    sample = (f"{used} rays x 512 uniform samples/ray per step (the rays of a {n}-ray draw that hit the box; non-cuda_ray renderer "
              f"nerf/renderer.py:128-256 + nerf/network.py with frequency encodings restated in oracle/cpu_renderer.py), {steps} timed + {warm} warm-up "
              f"steps, fp32, ONE host whatever --gpus is")
    cfg = base_config(1)
    cfg["arm"] = "cpu port of the reference's non-cuda_ray path; bounded sample of the workload (see cpu_baseline.sample)"
    line = {"impl": "reference", "metric": "train_rays_per_s", "value": value, "unit": "rays/s", "n_gpus": 1, "requested_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": "rays/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), file=_OUT, flush=True)


# =====================================================================================================================
class Ctx:
    """Process-wide handles shared by the measurement functions."""

    def __init__(self, args, torch, dist, rank, world, local, timed):
        self.args, self.torch, self.dist, self.rank, self.world, self.local, self.timed = args, torch, dist, rank, world, local, timed
        self.dev = torch.device("cuda", local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed_loop(self, fn, n):
        """n calls of fn(i) bracketed by barrier + synchronize, CUDA events, max over ranks -> total ms."""
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))

    def max_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def make_model(ctx, name, n_poses=8):
    from laenerf_b200.nerf import NeRFNetwork
    from laenerf_b200.scene import make_scene
    torch = ctx.torch
    sc = make_scene(name, seed=0, n_poses=n_poses)
    torch.manual_seed(0)
    model = NeRFNetwork(bound=sc.bound, min_near=sc.min_near, density_thresh=sc.density_thresh).to(ctx.dev)
    model.set_density_grid(torch.from_numpy(sc.density_grid).to(ctx.dev), thresh=10.0)
    return sc, model


def make_batches(ctx, sc, n_batches=8, seed=1000):
    import numpy as np
    from laenerf_b200.scene import get_rays_np
    torch = ctx.torch
    rng = np.random.default_rng(seed + ctx.rank)
    host = []
    for b in range(n_batches):
        ro, rd, _ = get_rays_np(sc.poses[b % len(sc.poses)], sc.intrinsics, sc.H, sc.W, N=N_RAYS, rng=rng)
        gt = rng.random((N_RAYS, 3), dtype=np.float32)
        host.append(tuple(torch.from_numpy(x).pin_memory() for x in (ro, rd, gt)))
    return host, [tuple(x.to(ctx.dev) for x in hb) for hb in host]


def size_sample_buffer(model, step, dev_batches):
    """The reference sizes the sample buffer from a running mean of the last <= 16 counters (renderer.py:643-647) and silently drops
    the rays that overflow it.  A timed pass must not drop work it is credited for: every batch is marched once, the buffer is
    sized for the largest one plus 3 % for the march noise, and mean_count stays fixed afterwards."""
    counts = []
    model.mean_count = 0
    for b in dev_batches:
        model.local_step = 0
        step(*b)  # mean_count <= 0: exact size from the counter (one host sync per step, as in the reference's first epoch)
        counts.append(int(model.step_counter[0, 0].item()))
    model.mean_count = int(max(counts) * 1.03) + 128
    model.local_step = 0
    return counts


def train_config(ctx, name, headline):
    """Training step of one scene: eager pass with per-kernel events, graph pass (`value`), end-to-end pass; headline adds the
    occupancy-update variant."""
    from laenerf_b200 import _native
    from laenerf_b200.nerf import GraphedTrainStep, TrainStep
    torch, args, world, timed = ctx.torch, ctx.args, ctx.world, ctx.timed
    sc, model = make_model(ctx, name)
    step = TrainStep(model, world_size=world)
    host_batches, dev_batches = make_batches(ctx, sc)
    nb = len(dev_batches)
    for i in range(max(args.warmup - nb, 0)):
        step(*dev_batches[i % nb])
    counts = size_sample_buffer(model, step, dev_batches)
    for i in range(3):
        step(*dev_batches[i % nb])
    ctx.barrier()
    steps = args.steps if headline else max(10, args.steps // 2)

    # ---- pass 1 (eager, Python-issued launches): per-kernel CUDA events live on the launching stream ------------------
    points = []
    timed.reset()
    timed.enabled = True
    l0 = _native.launch_count()
    model.local_step = 0
    eager_ms = ctx.timed_loop(lambda i: points.append(step(*dev_batches[i % nb])[1]["num_points"]), steps)
    timed.enabled = False
    eager_launches = _native.launch_count() - l0
    rows = int(points[0])
    seen = model.step_counter[: min(16, steps), 0].tolist()
    actual = int(sum(seen) / len(seen))
    dropped_samples = int(sum(max(0, c - rows) for c in seen))
    kern = timed.summary()

    # ---- pass 2 (product path): the whole step replayed from one CUDA graph; device-resident inputs ----------------------
    lookahead = os.environ.get("LNRF_LOOKAHEAD", "1") == "1"
    gstep, graph_note = None, "cuda graph (one capture per sample-buffer size)" + (
        "; software-pipelined: the occupancy march of batch k runs on a second stream beside the backward of batch k-1 (two sample-buffer "
        "sets, two graphs; every replay = one batch marched + one full forward/backward/optimizer step, loss one call late)" if lookahead else "")
    if os.environ.get("LNRF_NO_GRAPH", "0") != "1":
        try:
            gstep = GraphedTrainStep(step, N_RAYS, lookahead=lookahead)
            gstep.capture(*dev_batches[0])
            for i in range(3):
                gstep(*dev_batches[i % nb])
        except Exception as e:  # never silently: the JSON line says which path was timed
            gstep, graph_note = None, f"eager (graph capture failed: {type(e).__name__}: {e})"[:300]
            torch.cuda.synchronize()
    run = gstep if gstep is not None else (lambda *b: step(*b))
    last = [None]

    def timed_step(i):
        last[0] = run(*dev_batches[i % nb])

    clocks = ClockSampler(ctx.local).start() if ctx.rank == 0 else None
    ms = ctx.timed_loop(timed_step, steps)
    clk = clocks.stop() if clocks else None
    if headline and args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, *last[0])
    graph_seen = model.step_counter[: min(16, steps), 0].tolist()
    graph_rows = int(gstep.out["num_points"]) if gstep is not None else rows
    dropped_samples += int(sum(max(0, c - graph_rows) for c in graph_seen))
    in_sync = None
    if world > 1 and step.fused_optimizer:  # every rank must hold the same fp16 table after the sharded optimizer steps
        chk = model.encoder._shadow_f16.float().abs().sum().double().reshape(1)
        lo_, hi_ = chk.clone(), chk.clone()
        ctx.dist.all_reduce(lo_, op=ctx.dist.ReduceOp.MIN)
        ctx.dist.all_reduce(hi_, op=ctx.dist.ReduceOp.MAX)
        in_sync = bool(lo_.item() == hi_.item())
    value = world * N_RAYS * steps / (ms * 1e-3)
    res = dict(scene=name, image=[sc.H, sc.W], bound=sc.bound, cascades=model.cascade, ms_per_step=ms / steps, value=value, unit="rays/s",
               steps=steps, samples_per_step=actual, samples_per_ray=actual / N_RAYS, sample_rows_eager=rows, sample_rows_graph=graph_rows,
               samples_per_batch_at_sizing=counts, dropped_samples=dropped_samples, dropped_rays=0 if dropped_samples == 0 else None,
               train_msamples_per_s=world * actual * steps / (ms * 1e-3) / 1e6, occupancy=sc.occupancy_fraction(),
               eager_ms_per_step=eager_ms / steps, step_mode=graph_note, replicas_in_sync=in_sync, clocks=clk)
    if world > 1 and step.fused_optimizer:
        opt = step.optimizer
        res["exchange"] = ("one fused kernel over NVLink peer memory (torch symmetric memory): mean of the ranks' fp16 gradients + Adam on a 1/N "
                           "slice + store of the new fp16 values into every rank's table" if opt.p2p is not None else
                           "NCCL reduce-scatter + Adam on a 1/N slice + NCCL all-gather (symmetric memory unavailable: " +
                           str(getattr(opt, "p2p_error", "disabled")) + ")")
        res["exchange_sync"] = (None if opt.p2p is None else "inside the kernels (signal + poll on peer-mapped flag words)" if opt.inkernel_sync
                                else "two symmetric-memory barrier launches around the kernel")
        if os.environ.get("LNRF_TIME_EXCHANGE", "1") == "1":
            res["exchange_timing_us"] = opt.exchange_timing()

    # ---- per-kernel roofline (events recorded live inside the eager timed region) -------------------------------------
    peaks = measured_peaks()
    n_params = sum(p.numel() for p in model.parameters())
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    traffic = json.load(open(traffic_file)) if os.path.exists(traffic_file) else {}
    table = {}
    for kname, k in kern.items():
        a = ALGO[kname]
        calls_per_step = k["calls"] / steps
        if a["bound"] == "hbm":
            byts = (a.get("per_ray", 0) * N_RAYS + a.get("per_sample", 0) * actual + a.get("per_sample_padded", 0) * rows +
                    a.get("per_param", 0) * (n_params // world))  # sharded optimizer: each rank updates 1/world of the table
            ach = byts / (k["mean_ms"] * 1e-3) / 1e9
            table[kname] = dict(bound="hbm", achieved=ach, peak=peaks["hbm"], unit="GB/s", frac=ach / peaks["hbm"], mean_ms=k["mean_ms"],
                                calls_per_step=calls_per_step, algorithmic_bytes=byts, traffic=traffic.get(kname))
        else:
            fl = a["flops_per_sample_padded"] * rows
            ach = fl / (k["mean_ms"] * 1e-3) / 1e12
            table[kname] = dict(bound="tensor", achieved=ach, peak=peaks["tensor"], unit="TFLOP/s", frac=ach / peaks["tensor"],
                                mean_ms=k["mean_ms"], calls_per_step=calls_per_step, algorithmic_flops=fl, traffic=traffic.get(kname))
    dominant = max(table, key=lambda n: kern[n]["total_ms"]) if table else None
    roofline = None
    if dominant:
        d = table[dominant]
        roofline = dict(bound=d["bound"], achieved=d["achieved"], peak=d["peak"], unit=d["unit"], frac=d["frac"], traffic=d["traffic"],
                        kernel=dominant, mean_ms=d["mean_ms"], peak_source=peaks["source"] + (" (sustained)" if d["bound"] == "tensor" else ""),
                        share_of_step=kern[dominant]["total_ms"] / sum(k["total_ms"] for k in kern.values()),
                        timing="CUDA events around each C-ABI launch during the eager pass of the same step (graph replays cannot be bracketed)")
        # what actually limits the kernel when it is neither HBM nor the tensor pipe (ncu evidence under profiles/, DESIGN.md section 11)
        roofline["limiter"] = LIMITERS.get(dominant)
    for kname, lim in LIMITERS.items():
        if kname in table:
            table[kname]["limiter"] = lim
    res.update(roofline=roofline, kernels=table, gpu_launches=int(eager_launches))

    if headline:
        # ---- end-to-end: pinned host inputs -> H2D -> step -> D2H loss, every step ------------------------------------
        # Every step: three pinned host tensors -> device (147 456 B), the step, and the step's loss -> a pinned host word (4 B), which
        # the host READS one step later (event-synchronised) -- the way a training loop logs its loss without stalling the device
        # between steps.  `e2e_blocking` beside it: `loss.item()` right after every step.
        host_loss = torch.zeros(2, dtype=torch.float32).pin_memory()
        loss_ready = [torch.cuda.Event(), torch.cuda.Event()]
        seen_losses = []

        def e2e_iter(i, blocking=False):
            hb = host_batches[i % nb]
            if gstep is not None:
                loss, _ = gstep(*hb)  # static device buffers are filled straight from pinned memory (non_blocking copies)
            else:
                loss, _ = step(*(x.to(ctx.dev, non_blocking=True) for x in hb))
            if blocking:
                seen_losses.append(float(loss.item()))
                return
            slot = i & 1
            host_loss[slot:slot + 1].copy_(loss.detach().reshape(1), non_blocking=True)
            loss_ready[slot].record()
            if i > 0:
                loss_ready[slot ^ 1].synchronize()
                seen_losses.append(float(host_loss[slot ^ 1]))

        e2e_ms = ctx.timed_loop(e2e_iter, steps)
        e2e_blocking_ms = ctx.timed_loop(lambda i: e2e_iter(i, True), steps)
        assert all(math.isfinite(x) for x in seen_losses) and len(seen_losses) >= 2 * steps - 1
        res["e2e"] = {"value": world * N_RAYS * steps / (e2e_ms * 1e-3), "unit": "rays/s",
                      "h2d_bytes_per_step": sum(x.numel() * x.element_size() for x in host_batches[0]), "d2h_bytes_per_step": 4,
                      "loss_read": "every step's loss is copied to pinned host memory inside the timed region and read by the host one step "
                                   "later (event-synchronised)",
                      "blocking_read_value": world * N_RAYS * steps / (e2e_blocking_ms * 1e-3)}

        # ---- with the occupancy maintenance the reference pays every 16 steps (nerf/utils.py:1465-1467, renderer.py:556-649) ---------
        # The synthetic scene IS its procedural occupancy grid: letting a random-init network rewrite it would change the workload
        # (every cell becomes occupied).  So the update runs for real -- point generation, encoder, sigma net, scatter, EMA, mean,
        # packbits -- and the grid / bitfield are restored from a copy right after (8.6 MB of device copies, inside the timed region).
        try:
            keep = (model.density_grid.clone(), model.density_bitfield.clone(), model.mean_count)

            def occ_update(full):
                model.iter_density = 0 if full else 16
                with torch.autocast("cuda", dtype=torch.float16):
                    model.update_extra_state()
                model.density_grid.copy_(keep[0]); model.density_bitfield.copy_(keep[1])
                model.mean_count, model.local_step = keep[2], 0

            occ_ms = {}
            for full in (True, False):
                occ_update(full)
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                ev0.record()
                for _ in range(3):
                    occ_update(full)
                ev1.record()
                torch.cuda.synchronize()
                occ_ms["full" if full else "partial"] = ev0.elapsed_time(ev1) / 3

            def with_occ(i):
                if i % 16 == 0:
                    occ_update(False)
                    if gstep is not None:
                        gstep.remarch()  # look-ahead: the batch in flight goes through the updated bitfield again
                run(*dev_batches[i % nb])

            k16 = max(16, steps // 16 * 16)
            oms = ctx.timed_loop(with_occ, k16)
            res["value_with_occupancy_update"] = {
                "value": world * N_RAYS * k16 / (oms * 1e-3), "unit": "rays/s", "ms_per_step": oms / k16, "steps": k16, "update_every": 16,
                "update_ms": occ_ms, "note": "steady-state (partial) update_extra_state every 16 steps inside the timed region; the grid is restored "
                                             "after each update so the workload stays the procedural scene (full updates run only in the first 256 steps)"}
        except Exception as e:
            res["value_with_occupancy_update"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    res["_model"], res["_sc"], res["_step"], res["_batches"] = model, sc, step, (host_batches, dev_batches)
    return res


def dump_outputs(out_dir, loss, out):
    """What the last timed step returned to its caller -- the loss, the per-ray image / depth / weights_sum / nears and the sample
    count -- as DIR/<name>.npy (float32; the count float64).  Called right after the timed loop: the later passes of the benchmark
    replay the graph again, which overwrites these buffers.

    `depth` holds the rays that enter the scene box only.  A ray that misses it has near == far == FLT_MAX (raymarching.cu:122), and
    the depth normalisation of renderer.py:328 gives it 0 / 0 = NaN, a value that says nothing about the build; which rays miss is
    fixed by the inputs and visible in `nears`."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = dict(out, loss=loss)
    arrays["depth"] = out["depth"][out["nears"] < torch.finfo(torch.float32).max]
    for name, v in arrays.items():
        a = v.detach().float().cpu().numpy() if torch.is_tensor(v) else np.float64(v)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def count_real_samples(ctx, model, ro_d, rd_d):
    """Occupied-cell samples of these rays (the slots of a round include the zero padding the API mandates): counted once, outside
    the timed region, by the one-shot marcher without a sample budget."""
    from laenerf_b200 import raymarching as _rm
    torch = ctx.torch
    real = 0
    with torch.no_grad():
        for c0 in range(0, ro_d.shape[0], 65536):
            o_, d_ = ro_d[c0:c0 + 65536].contiguous(), rd_d[c0:c0 + 65536].contiguous()
            ne_, fa_ = _rm.near_far_from_aabb(o_, d_, model.aabb_infer, model.min_near)
            cnt_ = torch.zeros(2, dtype=torch.int32, device=ctx.dev)
            # force_all_rays with a 128-row token buffer would allocate N x 1024 rows: march with mean_count = 128 instead (counters are exact)
            _rm.march_rays_train(o_, d_, model.bound, model.density_bitfield, model.cascade, model.grid_size, ne_, fa_, cnt_, 128, False, -1, False, 0, 1024)
            real += int(cnt_[0].item())
    return real


def render_config(ctx, model, sc, pose_index=0, frames=3):
    """One full view, tile-sharded over ranks (no collective but the final gather), on both round schedules.  `value` is the
    reference schedule: bit-identical sample positions to nerf/renderer.py:335-387 (tests/test_gpu_refstack.py, test_gpu_fused.py)."""
    import numpy as np
    from laenerf_b200.parallel import gather_tiles, tile_shard_indices
    from laenerf_b200.scene import get_rays_np
    torch, world, rank = ctx.torch, ctx.world, ctx.rank
    ro, rd, _ = get_rays_np(sc.poses[pose_index], sc.intrinsics, sc.H, sc.W)
    # N > 1: 32 x 32 pixel tiles dealt round-robin over the ranks (contiguous row ranges leave the object to the middle ranks)
    tile = int(os.environ.get("LNRF_RENDER_TILE", "16"))  # 16 x 16: 2500 tiles of the 800 x 800 view, ~312 per rank at N = 8 (32 x 32 left the
    # ranks 20 % apart: the frame is as slow as its slowest share)
    mine = tile_shard_indices(sc.H, sc.W, rank, world, tile).numpy() if world > 1 else np.arange(sc.H * sc.W)
    ro_d, rd_d = torch.from_numpy(ro[mine]).to(ctx.dev), torch.from_numpy(rd[mine]).to(ctx.dev)
    model.eval()
    real = ctx.sum_over_ranks(count_real_samples(ctx, model, ro_d, rd_d))
    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for schedule in ("auto", "reference", "fast"):
        model.render_schedule = schedule
        model._auto_fast_ok = True
        marks, slots = [], 0
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            for _ in range(2):  # warm-up frames, final gather included (the first collective of a shape pays NCCL's lazy set-up)
                gather_tiles(model.render(ro_d, rd_d, perturb=False, bg_color=1)["image"], sc.H, sc.W, rank, world, tile)
            ctx.barrier()
            e0, e1 = ev(), ev()
            e0.record()
            for _ in range(frames):
                a, b, c = ev(), ev(), ev()
                a.record()
                o = model.render(ro_d, rd_d, perturb=False, bg_color=1)
                b.record()
                img = gather_tiles(o["image"], sc.H, sc.W, rank, world, tile)
                c.record()
                marks.append((a, b, c))
                slots += o["num_points"]
            e1.record()
            ctx.barrier()
        rms = ctx.max_over_ranks(e0.elapsed_time(e1))
        loop_ms = ctx.max_over_ranks(sum(a.elapsed_time(b) for a, b, _ in marks) / frames)
        gather_ms = ctx.max_over_ranks(sum(b.elapsed_time(c) for _, b, c in marks) / frames)
        slots_all = ctx.sum_over_ranks(slots)
        out[schedule] = dict(value=real * frames / (rms * 1e-3) / 1e6, unit="Msamples/s", ms_per_frame=rms / frames, render_loop_ms=loop_ms,
                             gather_ms=gather_ms, rounds=o.get("rounds"), resolved_schedule=o.get("schedule"), sample_slots_per_frame=slots_all / frames,
                             slots_msamples_per_s=slots_all / (rms * 1e-3) / 1e6, rays_per_s=ro.shape[0] * frames / (rms * 1e-3))
    model.render_schedule = "auto"
    model._auto_fast_ok = True
    model.train()
    res = dict(out["auto"])
    res.update(scene=sc.name, image_shape=list(img.shape), rays_per_frame=int(ro.shape[0]), samples_per_frame=real, schedule="auto",
               note=("value counts REAL samples (occupied-cell samples of the frame's rays; slots include the zero padding of every round).  "
                     "schedule 'auto': up to 32 samples per ray per round after the first WHEN the marcher proves the frame's bits cannot depend "
                     "on the round boundaries (every emitted delta exactly representable, checked per sample on the device), else the frame is "
                     "rendered on the reference's n_step rule -- either way image / depth / weights are bit-identical to the reference schedule "
                     "(tests/test_gpu_fused.py); `reference_schedule` and `fast_schedule` are the two fixed schedules for context (fast alone is "
                     "NOT bit-identical on scenes with cameras inside the volume)"),
               reference_schedule=out["reference"], fast_schedule=out["fast"],
               sharding=("32x32-pixel tiles dealt round-robin over the ranks; all_gather + index_select by the known index lists"
                         if world > 1 else "single GPU, row-major rays"))
    return res


def edit_config(ctx, flower):
    """BASELINE.json configs[4]: the recolor/style stage on the flower shape.  (1) EditDataset construction: one full-image
    run_cuda_distill per training view against the edit grid, VIEWS sharded over ranks (editing/edit_dataset.py:74-234);
    (2) style-network training: StyleTrainStep on the masked points of a view, data parallel over views (nerf/utils.py:953-1055)."""
    import numpy as np
    from laenerf_b200.parallel import shard_range
    from laenerf_b200.scene import get_rays_np
    from laenerf_b200.style_encoder import LAENeRF, StyleTrainStep
    torch, world, rank, dev = ctx.torch, ctx.world, ctx.rank, ctx.dev
    sc, model = flower["_sc"], flower["_model"]
    model.eval()
    model.render_schedule = "auto"
    n_views = max(8, world)
    lo, hi = shard_range(n_views, rank, world)
    views = []
    for v in range(lo, hi):
        ro, rd, _ = get_rays_np(sc.poses[v % len(sc.poses)], sc.intrinsics, sc.H, sc.W)
        views.append((torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)))
    # edit grid: the occupied cells of two quarters of the Morton range of each cascade (same layout as the density bitfield)
    edit = model.density_bitfield.clone()
    edit[edit.numel() // 4: edit.numel() // 2] = 0
    edit[3 * edit.numel() // 4:] = 0
    outs = []

    def distill_all(_):
        outs.clear()
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            for ro, rd in views:
                outs.append(model.run_cuda_distill(ro, rd, edit, perturb=False))

    distill_all(0)
    ms = ctx.timed_loop(distill_all, 2) / 2
    o, (ro, rd) = outs[0], views[0]
    mask = o["weights_edit"] > 0.05
    x_term, d = o["x_term"][mask].contiguous(), rd[mask].contiguous()
    masked = int(x_term.shape[0])
    # the reference's fp16 regularisers overflow beyond ~75k points (sum of (1 - max w) in half, style_encoder.py:185-189): one
    # iteration trains on a view's worth of at most 49 152 masked points
    x_term, d = x_term[:49152].contiguous(), d[:49152].contiguous()
    K = int(x_term.shape[0])
    params = SimpleNamespace(bound=sc.bound, num_palette_bases=8, style_weight=0.0, weight_loss_uniform=1e-6, weight_loss_non_uniform=1e-6,
                             offset_loss=1e-6, palette_loss_valid=1e-3, palette_loss_distinct=1e-3)
    res = dict(scene="flower", image=[sc.H, sc.W], views=n_views, views_per_rank=hi - lo, distill_ms_per_view_set=ms,
               distill_views_per_s=n_views / (ms * 1e-3), distill_rays_per_s=n_views * sc.H * sc.W / (ms * 1e-3),
               masked_points_of_view=masked, points_per_style_step=K)
    model.train()
    if K < 128:
        res["style"] = {"error": "edit grid hit by fewer than 128 pixels"}
        return res
    target = torch.rand(K, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(rank))
    timings = {}
    for fused in (True, False):
        torch.manual_seed(1)
        style = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
        st = StyleTrainStep(style, params, fused_optimizer=fused, world_size=world, rank=rank)
        losses = []
        for _ in range(5):
            st(x_term, d, target)
        sms = ctx.timed_loop(lambda i: losses.append(st(x_term, d, target)[0]), 20) / 20
        l = [float(x) for x in losses]
        timings["fused_adam" if fused else "torch_adam"] = dict(ms_per_step=sms, points_per_s=world * K / (sms * 1e-3), loss_first=l[0], loss_last=l[-1])
        if fused and world == 1:  # the same step replayed from one CUDA graph (the eager iteration is bound by the interpreter)
            try:
                from laenerf_b200.style_encoder import GraphedStyleTrainStep
                gst = GraphedStyleTrainStep(st, K)
                gst.capture(x_term, d, target)
                gl = []
                for _ in range(3):
                    gst(x_term, d, target)
                gms = ctx.timed_loop(lambda i: gl.append(gst(x_term, d, target)[0].clone()), 50) / 50
                timings["graph"] = dict(ms_per_step=gms, points_per_s=K / (gms * 1e-3), loss_last=float(gl[-1]))
                del gst
            except Exception as e:
                timings["graph"] = {"error": f"{type(e).__name__}: {e}"[:200]}
        del style, st
    res["style"] = dict(timings["fused_adam"], torch_adam=timings["torch_adam"], cuda_graph=timings.get("graph"),
                        note="StyleTrainStep: hash grid fwd/bwd (fp32 table, as the reference runs it without autocast), SH-3, two FFMLP nets on tcgen05, "
                             "palette mix, MSE + regularisers, GradScaler + Adam; `torch_adam` = the same step with torch.optim.Adam + torch GradScaler; "
                             "N > 1: one view per rank per step, gradients averaged over ranks")
    return res


def roofline_large(ctx, model, sc):
    """march / encode / composite at 65 536 rays (~4 M samples): the regime where the >= 60 %-of-HBM target is meaningful
    (SURVEY.md 8d: the 4096-ray launches move 6-130 MB and are latency-bound)."""
    import numpy as np
    from laenerf_b200 import raymarching
    from laenerf_b200.scene import get_rays_np
    torch, dev = ctx.torch, ctx.dev
    HBM = measured_peaks()["hbm"]
    N = 65536

    not_captured = []

    def timed(fn, n=8, warm=2):
        """n back-to-back calls captured in ONE CUDA graph and replayed: device time per call.  (Issued from Python, the 20-100 us
        kernels of this table are bound by the wrapper -- autograd Function, output allocation, ctypes: 40-100 us per call -- which is
        what rounds 1 and 2a reported for the compositing kernels by mistake.)"""
        for _ in range(warm):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        try:
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_, stream=cap):
                for _ in range(n):
                    fn()
            g_.replay()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                g_.replay()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / (3 * n)
        except Exception as e:  # say so instead of reporting a host-bound number silently
            torch.cuda.synchronize()
            not_captured.append(f"{type(e).__name__}: {e}"[:160])
            if os.environ.get("LNRF_BENCH_DEBUG"):
                import traceback
                traceback.print_exc()
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

    # everything below runs on ONE side stream, which is also the capture stream: autograd graphs built outside a capture and
    # differentiated inside it must not cross streams (the legacy stream cannot wait for a capturing one)
    cap = torch.cuda.Stream()
    cap.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cap):
        out = _roofline_large_on(ctx, model, sc, cap, N=N, HBM=HBM, timed=timed, not_captured=not_captured)
    torch.cuda.current_stream().wait_stream(cap)
    return out


def _roofline_large_on(ctx, model, sc, cap, N, HBM, timed, not_captured):
    import numpy as np
    from laenerf_b200 import raymarching
    from laenerf_b200.scene import get_rays_np
    torch, dev = ctx.torch, ctx.dev
    ro, rd, _ = get_rays_np(sc.poses[0], sc.intrinsics, sc.H, sc.W, N=N, rng=np.random.default_rng(0))
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    nears, fars = raymarching.near_far_from_aabb(ro, rd, model.aabb_train, model.min_near)
    counter = torch.zeros(2, dtype=torch.int32, device=dev)
    raymarching.march_rays_train(ro, rd, model.bound, model.density_bitfield, model.cascade, model.grid_size, nears, fars, counter, 128, True, -1, False, 0, 1024)
    M_real = int(counter[0].item())
    mean_count = int(M_real * 1.02)

    def march():
        counter.zero_()
        return raymarching.march_rays_train(ro, rd, model.bound, model.density_bitfield, model.cascade, model.grid_size, nears, fars, counter,
                                            mean_count, True, 128, False, 0, 1024)

    clocks = ClockSampler(ctx.local).start()
    xyzs, dirs, deltas, rays = march()
    M = int(xyzs.shape[0])
    out = {"rays": N, "samples": M_real, "rows": M, "hbm_peak_gbs": HBM, "kernels": {}}

    def rec(name, ms, byts):
        out["kernels"][name] = dict(ms=ms, algorithmic_bytes=byts, achieved_gbs=byts / ms / 1e6, frac=byts / ms / 1e6 / HBM)
        if not_captured:
            out["kernels"][name]["timing"] = "eager from Python (host-bound below ~100 us): graph capture failed: " + not_captured.pop()

    rec("march_rays_train", timed(march), 48 * N + 32 * M_real)
    enc = model.encoder
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        rec("grid_encode_forward", timed(lambda: enc(xyzs, bound=model.bound)), 588 * M)
    g = torch.randn(M, 32, device=dev).half() * 1e-3
    enc._grad_f16.zero_() if enc._grad_f16 is not None else None
    with torch.autocast("cuda", dtype=torch.float16):
        f2 = enc(xyzs, bound=model.bound)

    def enc_bwd():
        enc.embeddings.grad = None
        f2.backward(g, retain_graph=True)

    rec("grid_encode_backward", timed(enc_bwd), 588 * M)
    if enc._grad_f16 is not None:
        enc._grad_f16.zero_()
    sig = torch.rand(M, device=dev) * 20
    rgb = torch.rand(M, 3, device=dev)
    rec("composite_rays_train_forward", timed(lambda: raymarching.composite_rays_train(sig, rgb, deltas, rays, 1e-4)), 32 * N + 24 * M_real)
    gt = torch.rand(N, 3, device=dev)
    sg, rg = sig.clone().requires_grad_(True), rgb.clone().requires_grad_(True)
    loss, _, _, _ = raymarching.composite_loss_train(sg, rg, deltas, rays, gt, 1, nears, fars, 1e-4)

    def comp_bwd():
        sg.grad = rg.grad = None
        loss.backward(retain_graph=True)

    rec("composite_loss_train_forward", timed(lambda: raymarching.composite_loss_train(sig, rgb, deltas, rays, gt, 1, nears, fars, 1e-4)), 64 * N + 24 * M_real)
    rec("composite_loss_train_backward", timed(comp_bwd), 60 * N + 40 * M_real)
    scale = torch.tensor(1024.0, device=dev)

    from laenerf_b200 import _native as NL
    lib = NL.lib()
    o_ws, o_d, o_img, o_raw = torch.empty(N, device=dev), torch.empty(N, device=dev), torch.empty(N, 3, device=dev), torch.empty(N, 3, device=dev)
    o_loss, o_gs, o_gc = torch.empty((), device=dev), torch.empty_like(sig), torch.empty_like(rgb)
    nb = lib.lnrf_composite_loss_scratch_bytes(N)
    scr = torch.zeros((nb + 7) // 8, dtype=torch.int64, device=dev)

    def comp_both():  # the training step's entry point, straight through the C ABI (autograd would add the leaf-gradient copies)
        NL.check(lib.lnrf_composite_loss_train_forward_backward(
            scale.data_ptr(), sig.data_ptr(), rgb.data_ptr(), deltas.data_ptr(), rays.data_ptr(), gt.data_ptr(), None, 1.0, nears.data_ptr(),
            fars.data_ptr(), M, N, 1e-4, o_ws.data_ptr(), o_d.data_ptr(), o_img.data_ptr(), o_raw.data_ptr(), o_loss.data_ptr(), o_gs.data_ptr(),
            o_gc.data_ptr(), scr.data_ptr(), nb, NL.stream()))

    rec("composite_loss_train_forward_backward", timed(comp_both), 64 * N + 40 * M_real)
    out["timing"] = "8 calls captured in one CUDA graph, 3 replays, CUDA events: device time per call"
    out["clocks"] = clocks.stop()
    return out


def gpu_reference(ctx, lego, render):
    """The reference's OWN stack on this GPU, in this process (VERDICT r1: the >= 10x target needs driver-side evidence):
    nerf/renderer.py + nerf/network_ff.py (`--ff`) / nerf/network.py (default `-O`: nn.Linear MLPs on cuBLAS) of the reference, untouched,
    on the reference's wrapper packages and compiled extensions (oracle/_ref), driven like Trainer.train_step + the `-O` optimizer recipe
    (nerf/utils.py:535-642, 1474-1484; main_nerf.py:223).  Same scene, same 4096-ray batches, same sample-buffer size, CUDA events."""
    import ref_stack
    torch, args, dev = ctx.torch, ctx.args, ctx.dev
    if not ref_stack.available("reference"):
        return {"unavailable": "oracle/_ref (reference extensions + staged python) not built: python oracle/build_ref.py"}
    sc, ours = lego["_sc"], lego["_model"]
    _, dev_batches = lego["_batches"]
    nb = len(dev_batches)
    steps = max(5, min(args.steps, 20))
    out = {"what": "reference Python callers + reference CUDA extensions (sm_100a build of the untouched sources), eager as its trainer issues them",
           "steps": steps}
    clocks = ClockSampler(ctx.local).start()
    for variant in ("ff", "default"):
        try:
            m = ref_stack.make_model("reference", variant, device=dev, bound=sc.bound, density_scale=1, min_near=sc.min_near, density_thresh=10.0)
            with torch.no_grad():
                m.density_grid.copy_(ours.density_grid)
                m.density_bitfield.copy_(ours.density_bitfield)
            m.mean_count, m.local_step = ours.mean_count, 0
            m.train()
            opt = torch.optim.Adam(m.get_params(1e-2), betas=(0.9, 0.99), eps=1e-15)
            scaler = torch.amp.GradScaler("cuda")
            pts = []

            def one(i):
                ro, rd, gt = dev_batches[i % nb]
                opt.zero_grad()
                with torch.autocast("cuda", dtype=torch.float16):
                    o = m.render(ro[None], rd[None], staged=False, bg_color=1, perturb=True, force_all_rays=False, dt_gamma=0, max_steps=1024)
                    loss = torch.nn.functional.mse_loss(o["image"], gt[None], reduction="none").mean(-1).mean()
                scaler.scale(loss).backward()
                scaler.step(opt)
                scaler.update()
                m.local_step = 0

            for i in range(3):
                one(i)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                one(i)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            rec = dict(ms_per_step=ms, rays_per_s=N_RAYS / (ms * 1e-3), sample_rows=int(ours.mean_count),
                       stack=("--ff: nerf/network_ff.py (FFMLP extension, CUTLASS split-K wgrad)" if variant == "ff" else
                              "default -O: nerf/network.py (nn.Linear on cuBLAS) + raymarching / gridencoder / shencoder extensions"))
            if variant == "ff":  # the occupancy update and the host-loop render of the same 800 x 800 view, on this stack
                m.iter_density = 16
                keep = (m.density_grid.clone(), m.density_bitfield.clone())
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
                    m.update_extra_state()
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    m.iter_density = 16
                    m.update_extra_state()
                    torch.cuda.synchronize()
                rec["occupancy_partial_update_ms"] = (time.perf_counter() - t0) * 1e3
                with torch.no_grad():
                    m.density_grid.copy_(keep[0]); m.density_bitfield.copy_(keep[1])
                if render is not None:
                    from laenerf_b200.scene import get_rays_np
                    ro, rd, _ = get_rays_np(sc.poses[0], sc.intrinsics, sc.H, sc.W)
                    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
                    m.eval()
                    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
                        m.render(ro[None], rd[None], staged=False, bg_color=1, perturb=False, dt_gamma=0, max_steps=1024, T_thresh=1e-4, scale_depth=True)
                        torch.cuda.synchronize()
                        e0.record()
                        for _ in range(2):
                            m.render(ro[None], rd[None], staged=False, bg_color=1, perturb=False, dt_gamma=0, max_steps=1024, T_thresh=1e-4, scale_depth=True)
                        e1.record()
                        torch.cuda.synchronize()
                    rms = e0.elapsed_time(e1) / 2
                    out["render"] = dict(ms_per_frame=rms, value=render["samples_per_frame"] / (rms * 1e-3) / 1e6, unit="Msamples/s",
                                         note="NeRFRenderer.run_cuda inference loop (renderer.py:335-387, one host sync per round) on the same view")
            out[variant] = rec
            del m, opt
        except Exception as e:
            out[variant] = {"error": f"{type(e).__name__}: {e}"[:400]}
    out["clocks"] = clocks.stop()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-render", action="store_true", help="skip the full-image render measurement")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-gpu-ref", action="store_true", help="skip the gpu_reference leg")
    ap.add_argument("--no-configs", action="store_true", help="skip BASELINE configs 3-5")
    ap.add_argument("--no-large", action="store_true", help="skip the large-batch kernel roofline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed training step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3)

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    # ONE JSON line on stdout, whatever the libraries print (NCCL writes its version banner to fd 1): keep the real stdout aside
    # and point fd 1 at stderr for the rest of the process
    global _OUT
    sys.stdout.flush()
    _OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from laenerf_b200 import _native
    from laenerf_b200.parallel import init_distributed

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback for the product path)")
    if world > 1:
        os.environ.setdefault("LNRF_TIME_EXCHANGE", "1")
    rank, world, local = init_distributed()
    torch.cuda.set_device(torch.device("cuda", local))
    timed = TimedLib(_native.lib(), list(ALGO), torch)
    _native._lib = timed
    ctx = Ctx(args, torch, dist, rank, world, local, timed)

    def guarded(fn, *a):
        """Secondary records never take the headline down: an exception becomes {"error": ...} on every rank alike."""
        try:
            return fn(*a)
        except Exception as e:
            torch.cuda.synchronize()
            return {"error": f"{type(e).__name__}: {e}"[:400]}

    # ---- headline: configs[1], lego-shape training step ----------------------------------------------------------------
    lego = train_config(ctx, "lego", headline=True)
    render = None if args.no_render else guarded(render_config, ctx, lego["_model"], lego["_sc"])

    # ---- BASELINE configs 3-5 ----------------------------------------------------------------------------------------------
    configs = {}
    if not args.no_configs:
        flower = guarded(train_config, ctx, "flower", False)
        configs["flower_train"] = {k: v for k, v in flower.items() if not k.startswith("_") and k != "kernels"}
        if "_model" in flower:
            configs["flower_train"]["kernels_ms"] = {k: round(v["mean_ms"], 5) for k, v in flower["kernels"].items()}
            configs["edit_stage"] = guarded(edit_config, ctx, flower)

        def bonsai_render():
            sc_b, model_b = make_model(ctx, "bonsai")
            return render_config(ctx, model_b, sc_b, frames=2)
        configs["bonsai_render"] = guarded(bonsai_render)

    if rank != 0:
        _finish(world)
        return

    large = None if (args.no_large or world > 1) else guarded(roofline_large, ctx, lego["_model"], lego["_sc"])
    gref = None if (args.no_gpu_ref or world > 1) else guarded(gpu_reference, ctx, lego, render if render and "error" not in render else None)
    vs_gref = None
    if gref and "error" not in gref and "unavailable" not in gref:
        vs_gref = {}
        for k in ("ff", "default"):
            if isinstance(gref.get(k), dict) and "ms_per_step" in gref[k]:
                vs_gref[k] = gref[k]["ms_per_step"] / lego["ms_per_step"]
        if isinstance(gref.get("render"), dict) and render and "ms_per_frame" in render:
            vs_gref["render"] = gref["render"]["ms_per_frame"] / render["ms_per_frame"]
        vs_gref["target"] = ">= 10x the reference's own extensions on one B200 (BASELINE.json north_star)"

    # ---- CPU baseline beside it (rank 0, N = 1 only; bounded sample) ---------------------------------------------------
    cpu = None
    if world == 1 and not args.no_cpu:
        from oracle import cpu_renderer
        n = int(os.environ.get("LNRF_CPU_RAYS", "1024"))
        hb = lego["_batches"][0][0]
        sc = lego["_sc"]
        sec, threads, used = cpu_renderer.time_train_steps(hb[0][:n].clone(), hb[1][:n].clone(), hb[2][:n].clone(), steps=2, warmup=1,
                                                           num_steps=512, bound=sc.bound, min_near=sc.min_near)
        cpu = dict(value=used / sec, unit="rays/s", cores=threads, kind="port",
                   sample=f"{used} rays x 512 uniform samples/ray per step (non-cuda_ray renderer restated in oracle/cpu_renderer.py), 2 timed + 1 warm-up steps")

    cfg = base_config(world)
    for k in ("samples_per_step", "samples_per_ray", "sample_rows_eager", "sample_rows_graph", "dropped_rays", "dropped_samples", "step_mode",
              "replicas_in_sync", "exchange", "exchange_sync", "exchange_timing_us"):
        if k in lego:
            cfg[k] = lego[k]
    cfg["scene_occupancy"] = lego["occupancy"]
    cfg["occupancy_update"] = "excluded from `value` (fixed procedural grid); included in `value_with_occupancy_update`"
    if vs_gref:
        cfg["vs_gpu_reference"] = {k: (round(v, 2) if isinstance(v, float) else v) for k, v in vs_gref.items()}
    if render and "value" in render:
        cfg["render_msamples_per_s"] = round(render["value"], 1)
    line = {
        "metric": "train_rays_per_s", "value": lego["value"], "unit": "rays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": lego["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": cfg, "clocks": lego["clocks"], "e2e": lego.get("e2e"), "gpu_launches": lego["gpu_launches"], "roofline": lego["roofline"],
        "cpu_baseline": cpu,
        "eager": {"ms_per_step": lego["eager_ms_per_step"], "value": world * N_RAYS / (lego["eager_ms_per_step"] * 1e-3), "unit": "rays/s",
                  "note": "same step issued launch by launch from Python (the drop-in modules without graph capture)"},
        "value_with_occupancy_update": lego.get("value_with_occupancy_update"),
        "train_msamples_per_s": lego["train_msamples_per_s"],
        "kernels": lego["kernels"], "render": render, "configs": configs, "roofline_large": large,
        "gpu_reference": gref, "vs_gpu_reference": vs_gref,
    }
    print(json.dumps(line), file=_OUT, flush=True)
    _finish(world)


def _finish(world):
    """Multi-rank runs leave without tearing NCCL down: destroy_process_group() with captured collectives still alive in
    CUDA graphs was observed to hang until the launcher's timeout (2-GPU run of round 1).  All collectives are complete
    (every rank passed the final barrier + synchronize), so the processes simply exit."""
    if world > 1:
        import torch
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
