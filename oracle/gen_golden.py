#!/usr/bin/env python
"""Freeze golden vectors from the reference's OWN CUDA extensions (TEST INFRASTRUCTURE; needs a B200).

Run on the GPU box (`gpurun -- python oracle/gen_golden.py`): evaluates every case of tests/cases.py with
tests/backends.RefBackend -- the untouched reference sources compiled for sm_100a by oracle/build_ref.py into
oracle/_ref/ -- and writes gpurun_out/golden/ref_<case>.npz.  The files are then committed under tests/golden/
so that later rounds (and the CPU-only test tier) check parity without the reference or a GPU.  The per-level
hash-grid scales as the device evaluates exp2f are stored next to the grid cases ("in_scales_*").
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


MARCH_MILLION = [("lego", 1 << 20, 0.0), ("flower", 1 << 20, 0.0), ("bonsai", 1 << 20, 0.0), ("bonsai", 1 << 18, 1.0 / 256)]


def march_million(out_dir):
    """ref_march_million.json: digests of the reference's march_rays_train on the inputs of
    tests/test_gpu_live_reference.py::test_march_train_counts_bit_exact_on_a_million_rays (its helpers, the reference kernel)."""
    import torch
    import ref_step
    import test_gpu_live_reference as T
    dev = torch.device("cuda", 0)
    rm = ref_step.backend("_raymarching")
    out = {}
    for name, n, dt_gamma in MARCH_MILLION:
        sc, ro, rd = T._all_rays(name, n, 11, dev)
        n = ro.shape[0]
        bits = torch.from_numpy(sc.density_bitfield).to(dev)
        nears, fars = torch.empty(n, device=dev), torch.empty(n, device=dev)
        rm.near_far_from_aabb(ro, rd, torch.from_numpy(sc.aabb).to(dev), n, float(sc.min_near), nears, fars)
        noises = torch.rand(n, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
        _, _, _, rays, cnt = T._march_ref(rm, sc, ro, rd, bits, nears, fars, noises, 128, dt_gamma)
        counts = rays[torch.argsort(rays[:, 0].long())][:, 2]
        k = min(65536, n)
        sub = [x[:k].contiguous() for x in (ro, rd, nears, fars, noises)]
        xr, dr, lr, rr, c2 = T._march_ref(rm, sc, sub[0], sub[1], bits, sub[2], sub[3], sub[4], int(counts[:k].sum()) + 128, dt_gamma)
        cnt_b, (xb, db, lb) = T._canonical(rr, xr, dr, lr)
        out[f"{name}_{n}_{dt_gamma:g}"] = dict(near_far=T._digest(nears, fars), counter=cnt.tolist(), counts=T._digest(counts),
                                               subset_counter=c2.tolist(), subset_counts=T._digest(cnt_b), subset_xyzs=T._digest(xb),
                                               subset_dirs=T._digest(db), subset_deltas=T._digest(lb))
    with open(os.path.join(out_dir, "ref_march_million.json"), "w") as f:
        json.dump(out, f, indent=1)


def main():
    import torch  # noqa: F401  (libtorch symbols must be loaded before the extension modules)
    from backends import OursBackend, RefBackend
    from cases import CASES, grid_config, run_case

    out_dir = os.path.join(ROOT, "gpurun_out", "golden")
    os.makedirs(out_dir, exist_ok=True)
    want = sys.argv[1:] or list(CASES) + ["march_million"]
    if "march_million" in want:
        march_million(out_dir)
        want.remove("march_million")
    ref = RefBackend()
    ours = None
    try:
        ours = OursBackend()
    except Exception as e:  # the golden vectors do not depend on our library, only the scale hook does
        print("[gen_golden] our library unavailable for the scale hook:", e)
    report = {}
    for name in want:
        t0 = time.time()
        try:
            res = run_case(name, ref)
        except Exception as e:
            report[name] = f"FAILED: {type(e).__name__}: {e}"
            print(f"[gen_golden] {name}: FAILED {e}", flush=True)
            continue
        if name.startswith("grid") and ours is not None:
            L, H = (8, 16) if name == "grid_small" else (4, 16)
            _, pls = grid_config(8, 2, 3, 16, 12, 512) if name == "grid_small" else grid_config(4, 4, 2, 16, 10, 128)
            res[f"in_scales_{L}_{H}"] = ours.grid_level_scales(L, pls, H)
        np.savez_compressed(os.path.join(out_dir, f"ref_{name}.npz"), **res)
        report[name] = {k: list(np.asarray(v).shape) for k, v in res.items()}
        print(f"[gen_golden] {name}: {len(res)} arrays in {time.time() - t0:.1f}s", flush=True)
    with open(os.path.join(out_dir, "report.json"), "w") as f:
        json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
