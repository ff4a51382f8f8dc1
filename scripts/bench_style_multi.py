"""Edit-stage style-network step, data parallel over views: ms per step at N = 1, 2, 4, 8 GPUs, eager and replayed from a CUDA graph,
for the symmetric-memory exchange (StyleTrainStep(world_size=N) -> ShardedFlatAdam: one exchange + Adam kernel over NVLink) against
the NCCL all-reduce path it replaces (AmpAdam with one all-reduce per gradient tensor and the full Adam on every rank), eagerly and
with the collectives captured in the graph.

Inputs are bench.py's edit stage: the flower shape, one distillation render per rank's view against the same edit grid, at most
49 152 masked points per rank per step (repeated up to that count when a view has fewer, reported as `masked_points`).  The variants
are timed in the same process, alternating, over `--repeats` rounds of `--steps` steps each; every number is the median and the
spread (min, max) of the per-round means.  The card name, power limit and SM clock are read in the same call.  N above the number
of visible GPUs is reported as not measured.

    python scripts/bench_style_multi.py --out /tmp/style_multi.json
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
K_MAX = 49152


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _machine():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        return [dict(zip(q.split(","), [x.strip() for x in line.split(",")])) for line in out.strip().splitlines()]
    except Exception as e:  # reported, not guessed
        return {"error": f"{type(e).__name__}: {e}"}


def _inputs(torch, dev, rank, world):
    """bench.py edit_config's inputs for this rank's view: flower shape, distillation render against the edit grid, masked points."""
    from types import SimpleNamespace
    from cases import scene
    from laenerf_b200.nerf import NeRFNetwork
    from laenerf_b200.scene import get_rays_np
    sc = scene("flower")
    torch.manual_seed(0)
    model = NeRFNetwork(bound=sc.bound, min_near=sc.min_near, density_thresh=sc.density_thresh).to(dev)
    model.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    model.eval()
    edit = model.density_bitfield.clone()
    edit[edit.numel() // 4: edit.numel() // 2] = 0
    edit[3 * edit.numel() // 4:] = 0
    ro, rd, _ = get_rays_np(sc.poses[rank % len(sc.poses)], sc.intrinsics, sc.H, sc.W)
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        o = model.run_cuda_distill(ro, rd, edit, perturb=False)
    mask = o["weights_edit"] > 0.05
    x, d = o["x_term"][mask].float().contiguous(), rd[mask].contiguous()
    masked = int(x.shape[0])
    if masked < 128:
        raise RuntimeError(f"rank {rank}: the edit grid hit {masked} pixels of the view")
    idx = torch.arange(K_MAX, device=dev) % masked
    x, d = x[idx][:K_MAX].contiguous(), d[idx][:K_MAX].contiguous()
    target = torch.rand(K_MAX, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(rank))
    params = SimpleNamespace(bound=sc.bound, num_palette_bases=8, style_weight=0.0, weight_loss_uniform=1e-6, weight_loss_non_uniform=1e-6,
                             offset_loss=1e-6, palette_loss_valid=1e-3, palette_loss_distinct=1e-3)
    del model
    return params, (x, d, target), masked


def _worker(rank, world, port, args, q):
    import torch
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from laenerf_b200.style_encoder import GraphedStyleTrainStep, LAENeRF, StyleTrainStep
    res = {"n_gpus": world}
    try:
        params, batch, masked = _inputs(torch, dev, rank, world)
        res["masked_points_rank0"] = masked
        runs = {}

        def make(kind):
            torch.manual_seed(1)
            style = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
            if kind == "exchange":   # what StyleTrainStep selects (at N = 1: the single-GPU step)
                st = StyleTrainStep(style, params, world_size=world, rank=rank)
                res["exchange"] = st.exchange if world > 1 else "local"
                if st.p2p_error:
                    res["p2p_error"] = st.p2p_error
            else:                    # the NCCL all-reduce path: AmpAdam, one all-reduce per gradient tensor, full Adam on every rank
                st = StyleTrainStep(style, params, world_size=1, rank=rank)
                st.optimizer.world = world
            return st

        kinds = ["exchange"] + (["allreduce"] if world > 1 else [])
        for kind in kinds:
            st = make(kind)
            for _ in range(3):
                st(*batch)
            runs[f"{kind}_eager"] = st
            try:
                gst = GraphedStyleTrainStep(make(kind), K_MAX)
                gst.capture(*batch)
                for _ in range(3):
                    gst(*batch)
                runs[f"{kind}_graph"] = gst
            except Exception as e:
                res[f"{kind}_graph_error"] = f"{type(e).__name__}: {e}"[:300]
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        times = {k: [] for k in runs}
        for _ in range(args.repeats):   # variants alternate inside every round
            for k, fn in runs.items():
                if dist is not None:
                    dist.barrier()
                torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.steps):
                    fn(*batch)
                b.record()
                torch.cuda.synchronize()
                ms = torch.tensor([a.elapsed_time(b) / args.steps], device=dev)
                if dist is not None:
                    dist.all_reduce(ms, op=dist.ReduceOp.MAX)   # the step of the slowest rank
                times[k].append(float(ms))
        for k, v in times.items():
            s = sorted(v)
            res[k] = {"ms_per_step_median": s[len(s) // 2], "min": s[0], "max": s[-1], "rounds": v}
        if world > 1 and "exchange_eager" in runs:   # the replicas hold the same parameters
            opt = runs["exchange_eager"].optimizer
            if hasattr(opt, "param_flat"):
                full = torch.empty(world, opt.param_flat.numel(), device=dev)
                dist.all_gather_into_tensor(full, opt.param_flat.clone())
                res["replicas_identical"] = all(bool(torch.equal(full[r], full[0])) for r in range(world))
    except Exception as e:
        res["error"] = f"{type(e).__name__}: {e}"[:500]
    if rank == 0:
        q.put(res)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    os._exit(0)   # symmetric memory / captured collectives: leave without tearing NCCL down (as bench.py does)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--gpus", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available():
        raise SystemExit("bench_style_multi: no CUDA device (this measurement needs B200s)")
    visible = torch.cuda.device_count()
    out = {"machine": _machine(), "visible_gpus": visible, "steps_per_round": args.steps, "rounds": args.repeats,
           "points_per_rank_per_step": K_MAX, "results": []}
    ctx = mp.get_context("spawn")
    for n in [int(x) for x in args.gpus.split(",")]:
        if n > visible:
            out["results"].append({"n_gpus": n, "not_measured": f"{visible} GPU(s) visible"})
            continue
        q = ctx.Queue()
        port = _free_port()
        procs = [ctx.Process(target=_worker, args=(r, n, port, args, q)) for r in range(n)]
        for p in procs:
            p.start()
        out["results"].append(q.get(timeout=1800))
        for p in procs:
            p.join(timeout=120)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
