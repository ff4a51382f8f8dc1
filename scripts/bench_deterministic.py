#!/usr/bin/env python
"""What torch.use_deterministic_algorithms(True) costs (GPU only).  In one call, flag off against flag on:

  train_step      lego, 4096 rays, GraphedTrainStep(lookahead=True) as bench.py runs it: one model and graph per mode (each captured
                  under its own flag), the two modes alternating over `--rounds` rounds of `--steps` replays, CUDA events
  encoder_bwd     the hash-grid backward alone at the training shape (a seeded lego march, fp16 table): the atomic kernel
                  (lnrf_grid_encode_backward_world) against the fixed-point kernel (lnrf_grid_encode_backward_world_det), and the
                  finish kernel (lnrf_grid_det_finish) on its own; each captured `--reps` times in a CUDA graph
  occupancy       one partial update_extra_state (iter_density >= 16), host clock around a synchronised call
  style_step      the edit-stage style step (flower bound, 8 palette bases, 49 152 points) replayed from GraphedStyleTrainStep

Every number is the median and the spread (min, max) of the per-round means.  The card, power limit and SM clock are read in the
same call.  The style step multiplies the palette with cuBLAS, which under the flag needs CUBLAS_WORKSPACE_CONFIG=:4096:8: the
script sets it before CUDA starts.

    python scripts/bench_deterministic.py --out /tmp/det
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _machine():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        return {"query": q, "gpus": [l.strip() for l in out.strip().splitlines()]}
    except Exception as e:  # the measurement stands without it, but says so
        return {"query": q, "error": f"{type(e).__name__}: {e}"}


def stat(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="output directory (bench_deterministic.json)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()

    import numpy as np
    import torch

    from laenerf_b200 import _native as N
    from laenerf_b200.gridencoder import _offsets_host
    from laenerf_b200.nerf import GraphedTrainStep, NeRFNetwork, TrainStep
    from laenerf_b200.scene import get_rays_np, make_scene

    if not torch.cuda.is_available():
        raise SystemExit("bench_deterministic: needs a GPU")
    dev = torch.device("cuda", 0)
    lib = N.lib()
    modes = (False, True)
    sc = make_scene("lego", seed=0, n_poses=2)
    ro, rd, _ = get_rays_np(sc.poses[0], sc.intrinsics, sc.H, sc.W, N=4096, rng=np.random.default_rng(0))
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    gt = torch.rand(4096, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def model():
        torch.manual_seed(0)
        m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
        m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
        return m

    # ---- graphed training step -------------------------------------------------------------------------------------------------
    runs = {}
    for det in modes:
        torch.use_deterministic_algorithms(det)
        m = model()
        g = GraphedTrainStep(TrainStep(m), 4096, lookahead=True)
        for _ in range(10):
            g(ro, rd, gt)
        runs[det] = (m, g)
    step_ms = {det: [] for det in modes}
    for _ in range(args.rounds):
        for det in modes:
            torch.use_deterministic_algorithms(det)
            g = runs[det][1]
            g(ro, rd, gt)
            e0.record()
            for _ in range(args.steps):
                g(ro, rd, gt)
            e1.record()
            torch.cuda.synchronize()
            step_ms[det].append(e0.elapsed_time(e1) / args.steps)

    # ---- encoder backward alone + finish -----------------------------------------------------------------------------------------
    torch.use_deterministic_algorithms(False)
    m = runs[False][0]
    mr = m.march_train(ro, rd, perturb=True)
    xyzs, cnt = mr["xyzs"], mr["counter"]
    M = xyzs.shape[0]
    enc = m.encoder
    L, S, H = enc.num_levels, float(np.log2(enc.per_level_scale)), enc.base_resolution
    off_h = _offsets_host(enc.offsets)
    E = enc.embeddings.shape[0]
    dy = (torch.randn(M, L * 2, device=dev, generator=torch.Generator(device=dev).manual_seed(1)) * 1e-2).half()
    gemb = torch.zeros(E, 2, dtype=torch.half, device=dev)
    acc = torch.zeros(E, 2, dtype=torch.int64, device=dev)
    flags = torch.zeros(E, dtype=torch.int32, device=dev)

    def s():
        return torch.cuda.current_stream().cuda_stream

    kernels = {
        "atomic_bwd": lambda: N.check(lib.lnrf_grid_encode_backward_world(N.ptr(dy), N.ptr(xyzs), float(sc.bound), N.ptr(off_h), N.ptr(gemb),
                                                                          M, N.ptr(cnt), L, S, H, 0, 0, 0, N.F16, s())),
        "det_bwd": lambda: N.check(lib.lnrf_grid_encode_backward_world_det(N.ptr(dy), N.ptr(xyzs), float(sc.bound), N.ptr(off_h), N.ptr(acc),
                                                                           N.ptr(flags), None, M, N.ptr(cnt), L, S, H, 0, 0, 0, N.F16, s())),
        "det_finish": lambda: N.check(lib.lnrf_grid_det_finish(N.ptr(acc), N.ptr(flags), None, M, N.ptr(gemb), E, 2, N.F16, s())),
    }
    kernels["det_bwd_plus_finish"] = lambda: (kernels["det_bwd"](), kernels["det_finish"]())
    graphs = {}
    for k, fn in kernels.items():
        warm = torch.cuda.Stream()
        warm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(warm):
            fn()
            kernels["det_finish"]()  # leaves acc / flags re-armed
        torch.cuda.current_stream().wait_stream(warm)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(args.reps):
                fn()
        graphs[k] = gr
    kern_us = {k: [] for k in kernels}
    for _ in range(args.rounds):
        for k, gr in graphs.items():
            gr.replay()
            e0.record()
            gr.replay()
            e1.record()
            torch.cuda.synchronize()
            kern_us[k].append(e0.elapsed_time(e1) * 1e3 / args.reps)
            if k == "det_bwd":  # the sums of reps backwards: clear them before the next window
                kernels["det_finish"]()
    acc.zero_()
    flags.zero_()

    # ---- one partial occupancy update --------------------------------------------------------------------------------------------
    occ_ms = {det: [] for det in modes}
    for _ in range(args.rounds):
        for det in modes:
            torch.use_deterministic_algorithms(det)
            mm = runs[det][0]
            mm.iter_density = max(mm.iter_density, 16)
            torch.cuda.synchronize()
            t = time.perf_counter()
            mm.update_extra_state()
            torch.cuda.synchronize()
            occ_ms[det].append((time.perf_counter() - t) * 1e3)

    # ---- graphed style step --------------------------------------------------------------------------------------------------
    from types import SimpleNamespace

    from laenerf_b200.style_encoder import GraphedStyleTrainStep, LAENeRF, StyleTrainStep
    params = SimpleNamespace(bound=2.0, num_palette_bases=8, style_weight=0.0, weight_loss_uniform=1e-6, weight_loss_non_uniform=1e-6,
                             offset_loss=1e-6, palette_loss_valid=1e-3, palette_loss_distinct=1e-3)
    K = 49152
    gs = torch.Generator(device=dev).manual_seed(4)
    view = ((torch.rand(K, 3, device=dev, generator=gs) - 0.5) * 3.0, torch.nn.functional.normalize(torch.randn(K, 3, device=dev, generator=gs), dim=-1),
            torch.rand(K, 3, device=dev, generator=gs))
    styles = {}
    for det in modes:
        torch.use_deterministic_algorithms(det)
        torch.manual_seed(1)
        st = GraphedStyleTrainStep(StyleTrainStep(LAENeRF(params, dir_encoding="sphere_harmonics").to(dev), params), K)
        for _ in range(5):
            st(*view)
        styles[det] = st
    style_ms = {det: [] for det in modes}
    for _ in range(args.rounds):
        for det in modes:
            torch.use_deterministic_algorithms(det)
            e0.record()
            for _ in range(args.steps // 4):
                styles[det](*view)
            e1.record()
            torch.cuda.synchronize()
            style_ms[det].append(e0.elapsed_time(e1) / (args.steps // 4))
    torch.use_deterministic_algorithms(False)

    name = {False: "flag_off", True: "flag_on"}
    out = {"what": "torch.use_deterministic_algorithms(True) against the default, alternating rounds", "machine": _machine(),
           "rounds": args.rounds, "train_steps_per_round": args.steps, "kernel_reps_per_graph": args.reps,
           "train_step_ms": {name[d]: stat(step_ms[d]) for d in modes},
           "encoder_bwd_us": {k: stat(v) for k, v in kern_us.items()},
           "encoder_bwd_shape": {"scene": "lego", "sample_rows": M, "live_samples": int(cnt[0]), "levels": L, "entries": E, "table": "fp16",
                                 "acc_bytes": acc.numel() * 8},
           "occupancy_update_ms": {name[d]: stat(occ_ms[d]) for d in modes},
           "style_step_ms": {name[d]: stat(style_ms[d]) for d in modes}}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_deterministic.json"), "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
