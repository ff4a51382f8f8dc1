#!/usr/bin/env python
"""Can the hash-table Adam update overlap the hash-grid backward?  Go/no-go measurement for running Adam on a second stream beside
the encoder backward (GPU only; today's kernels, nothing new).

Training shape: lego, a seeded 4096-ray march from a model warmed up by six TrainSteps (so the sample buffer and its live-row count
are the real ones), 16 levels, 2^19 entries, fp16 table.  Every variant is captured in a CUDA graph that repeats its pattern `--reps`
times and is replayed `--replays` times between two CUDA events:

  serial      lnrf_grid_encode_backward_world, then lnrf_adam_step, on one stream (today's order, without the inf check between them)
  concurrent  the same two launches on two streams with no dependency between them
  bwd_alone   the backward only
  adam_alone  Adam only

Adam runs on a CLONE of the optimizer state (parameters, moments, fp16 shadow, gradient), so what it computes does not matter and
there is no data dependency on the backward.  The knobs tried: LNRF_GRID_CAP (the backward's CTAs per SM) and the priority of the
Adam stream.  The variants alternate over `--rounds` rounds; every number is the median and the spread (min, max) of the per-round
means.  The card, power limit and SM clock are read in the same call.

    python scripts/bench_adam_overlap.py --out /tmp/adam_overlap.json

Result on one B200 at a 1000 W power limit (`profiles/r3b_adam_overlap.json`, DESIGN.md §11): two streams save at most 4.4 us of the
159 us serial pair, so Adam is not overlapped with the backward.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--replays", type=int, default=5)
    ap.add_argument("--caps", default="16,8,4", help="LNRF_GRID_CAP backward CTAs per SM to try")
    args = ap.parse_args()

    import ctypes as C

    import numpy as np
    import torch

    from laenerf_b200 import _native as N
    from laenerf_b200.gridencoder import _offsets_host
    from laenerf_b200.nerf import NeRFNetwork, TrainStep
    from laenerf_b200.scene import get_rays_np, make_scene

    if not torch.cuda.is_available():
        raise SystemExit("bench_adam_overlap: needs a GPU")
    dev = torch.device("cuda", 0)
    lib = N.lib()
    torch.manual_seed(0)
    sc = make_scene("lego", seed=0, n_poses=2)
    m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
    m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    ro, rd, _ = get_rays_np(sc.poses[0], sc.intrinsics, sc.H, sc.W, N=4096, rng=np.random.default_rng(0))
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    gt = torch.rand(4096, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    step = TrainStep(m)
    for _ in range(3):
        step(ro, rd, gt)
    m.update_mean_count()
    for _ in range(3):
        step(ro, rd, gt)
    mr = m.march_train(ro, rd, perturb=True)
    xyzs, cnt = mr["xyzs"], mr["counter"]
    M = xyzs.shape[0]
    live = int(cnt[0])
    enc = m.encoder
    L, S, H = enc.num_levels, float(np.log2(enc.per_level_scale)), enc.base_resolution
    off_h = _offsets_host(enc.offsets)
    g = torch.Generator(device=dev).manual_seed(1)
    dy = (torch.randn(M, L * 2, device=dev, generator=g) * 1e-2).half()  # d loss / d features at the encoder's output
    gemb = torch.zeros_like(enc._shadow_f16)

    # Adam on a clone of the optimizer state: same sizes, same layout, no dependency on gemb
    opt = step.optimizer
    keep = []
    arr = (N.OptTensor * len(opt.owners))()
    for i, (o, st) in enumerate(zip(opt.owners, opt.state)):
        p, ea, es = o.param.data.clone(), st["exp_avg"].clone(), st["exp_avg_sq"].clone()
        sh = o.module._shadow_f16.clone()
        gr = (torch.randn(p.shape, device=dev, generator=g) * 1e-3).half()
        keep += [p, ea, es, sh, gr]
        arr[i].params, arr[i].exp_avg, arr[i].exp_avg_sq = p.data_ptr(), ea.data_ptr(), es.data_ptr()
        arr[i].grad, arr[i].params_f16, arr[i].n, arr[i].grad_dtype = gr.data_ptr(), sh.data_ptr(), p.numel(), N.F16
    snap = torch.tensor([0.0, 65536.0, 10.0, 0.0], device=dev)  # {found_inf, scale, step}
    lr_scale = torch.ones(1, device=dev)
    n_params = sum(o.param.numel() for o in opt.owners)

    def s():
        return torch.cuda.current_stream().cuda_stream

    def bwd():
        N.check(lib.lnrf_grid_encode_backward_world(N.ptr(dy), N.ptr(xyzs), float(sc.bound), N.ptr(off_h), N.ptr(gemb), M, N.ptr(cnt), L, S,
                                                    H, 0, 0, 0, N.F16, s()))

    def adam():
        base = snap.data_ptr()
        N.check(lib.lnrf_adam_step(C.cast(arr, C.c_void_p), len(opt.owners), 1e-2, 0.9, 0.99, 1e-15, 0.0, base + 4, base, base + 8,
                                   N.ptr(lr_scale), s()))

    def capture(kind, cap, prio):
        os.environ["LNRF_GRID_CAP"] = f"16,{cap}"  # read by the launch wrapper at capture time
        side = torch.cuda.Stream(priority=prio)
        warm = torch.cuda.Stream()
        warm.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(warm):
            bwd(); adam()
        torch.cuda.current_stream().wait_stream(warm)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            main = torch.cuda.current_stream()
            for _ in range(args.reps):
                if kind == "serial":
                    bwd(); adam()
                elif kind == "concurrent":
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        adam()
                    bwd()
                    main.wait_stream(side)
                elif kind == "bwd_alone":
                    bwd()
                else:
                    adam()
        os.environ.pop("LNRF_GRID_CAP", None)
        return gr

    caps = [int(c) for c in args.caps.split(",")]
    lo, hi = torch.cuda.Stream.priority_range()  # (least, greatest): greatest is the numerically lowest
    variants = [("adam_alone", 16, 0)]
    for cap in caps:
        variants += [("bwd_alone", cap, 0), ("serial", cap, 0), ("concurrent", cap, 0), ("concurrent", cap, hi)]
    graphs = {v: capture(*v) for v in variants}
    for gr in graphs.values():
        gr.replay()
    torch.cuda.synchronize()

    times = {v: [] for v in variants}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.rounds):
        for v in variants:
            graphs[v].replay()  # one untimed replay: the same L2 state before every timed window
            e0.record()
            for _ in range(args.replays):
                graphs[v].replay()
            e1.record()
            torch.cuda.synchronize()
            times[v].append(e0.elapsed_time(e1) * 1e3 / (args.replays * args.reps))

    def stat(xs):
        xs = sorted(xs)
        return {"median_us": xs[len(xs) // 2], "min_us": xs[0], "max_us": xs[-1]}

    res = {f"{k}|cap={c}|adam_prio={'high' if p == hi and p != 0 else 'normal'}": stat(times[(k, c, p)]) for k, c, p in variants}
    a = stat(times[("adam_alone", 16, 0)])["median_us"]
    verdict = {}
    for cap in caps:
        ser = stat(times[("serial", cap, 0)])["median_us"]
        best = min(stat(times[("concurrent", cap, p)])["median_us"] for p in (0, hi))
        verdict[f"cap={cap}"] = {"serial_us": ser, "best_concurrent_us": best, "saving_us": ser - best,
                                 "bwd_alone_plus_adam_alone_us": stat(times[("bwd_alone", cap, 0)])["median_us"] + a}
    out = {"what": "hash-grid backward + Adam, serial vs two streams, CUDA graph replay, per pattern", "scene": "lego", "rays": 4096,
           "sample_rows": M, "live_samples": live, "levels": L, "table_params": enc.embeddings.numel(), "adam_params": n_params,
           "rounds": args.rounds, "reps_per_graph": args.reps, "replays": args.replays, "stream_priority_range": [lo, hi],
           "machine": _machine(), "results": res, "summary": verdict}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
