"""Seeded training runs under torch.use_deterministic_algorithms(True), shared by tests/test_gpu_deterministic.py.

Each run returns {name: tensor} of everything that must be bit-identical between two runs from the same seed.  Run as a
script, one run per process, it prints the sha256 digest of that state:
    python tests/det_driver.py nerf graphed|eager [lookahead] [noperturb]
    python tests/det_driver.py style graphed|eager
The style step multiplies the palette with cuBLAS, which under the flag needs CUBLAS_WORKSPACE_CONFIG=:4096:8 in the
environment before CUDA starts.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_RAYS = 4096


def digest(state: dict) -> str:
    h = hashlib.sha256()
    for k in sorted(state):
        t = state[k].detach().contiguous().cpu()
        h.update(k.encode())
        h.update(t.view(torch.uint8).numpy().tobytes() if t.numel() else b"")
    return h.hexdigest()


def nerf_run(form="graphed", lookahead=True, perturb=True, steps=20, update_after=10, seed=0):
    """lego, `steps` training batches of 4096 rays with one partial occupancy update (iter_density >= 16) after batch
    `update_after`.  form "eager": TrainStep calls that mirror what GraphedTrainStep(...).capture(b0, warmup=1) runs eagerly."""
    from cases import scene, scene_rays
    from laenerf_b200.nerf import GraphedTrainStep, NeRFNetwork, TrainStep
    torch.use_deterministic_algorithms(True)
    dev = torch.device("cuda", 0)
    sc = scene("lego")
    torch.manual_seed(seed)
    m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
    with torch.no_grad():
        m.encoder.embeddings.uniform_(-0.5, 0.5, generator=torch.Generator(device=dev).manual_seed(seed + 1))
    m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    m.iter_density = 16  # partial updates: random cells with repeats
    batches = []
    for k in range(steps):
        _, ro, rd, _ = scene_rays("lego", N_RAYS, 200 + k)
        gt = torch.rand(N_RAYS, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(300 + k))
        batches.append((torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev), gt))
    step = TrainStep(m)
    losses = []

    def occupancy_update():
        # as bench.py does it: under autocast, and the sample buffer keeps its size (the captured graphs' buffers stay valid)
        keep = m.mean_count
        with torch.autocast("cuda", dtype=torch.float16):
            m.update_extra_state()
        m.mean_count = keep

    if form == "eager":
        step(*batches[0], perturb=perturb)        # sizes the sample buffer (capture does the same when mean_count is 0)
        m.update_mean_count()
        step(*batches[0], perturb=perturb)        # capture's warm-up step
        for k, b in enumerate(batches):
            losses.append(step(*b, perturb=perturb)[0].detach().clone())
            if k == update_after:
                occupancy_update()
    else:
        g = GraphedTrainStep(step, N_RAYS, perturb=perturb, lookahead=lookahead)
        g.capture(*batches[0], warmup=1)
        for k, b in enumerate(batches):
            if lookahead and k == 0:
                continue                          # batch 0 is in flight since the capture
            loss = g(*b)[0]
            losses.append(loss.detach().clone())
            trained = k - 1 if lookahead else k
            if trained == update_after:
                occupancy_update()
                g.remarch()                       # lookahead: the batch in flight was marched through the old bitfield
        if lookahead:
            losses.append(g.flush()[0].detach().clone())
    torch.cuda.synchronize()
    opt = step.optimizer
    state = {"loss": torch.stack([l.float().reshape(()) for l in losses]), "density_grid": m.density_grid.clone(),
             "bitfield": m.density_bitfield.clone(), "scale": opt._scale.clone(), "step": opt.step_count.clone()}
    for k, v in m.named_parameters():
        state["param." + k] = v.detach().clone()
    for i, s in enumerate(opt.state):
        for k, v in s.items():
            state[f"opt.{i}.{k}"] = v.clone()
    return state


def style_run(form="graphed", steps=8, seed=0):
    """The edit-stage style network (flower bound, 8 palette bases), `steps` iterations over 4 views of 49 152 points."""
    from types import SimpleNamespace
    from laenerf_b200.style_encoder import GraphedStyleTrainStep, LAENeRF, StyleTrainStep
    torch.use_deterministic_algorithms(True)
    dev = torch.device("cuda", 0)
    params = SimpleNamespace(bound=2.0, num_palette_bases=8, style_weight=0.0, weight_loss_uniform=1e-6, weight_loss_non_uniform=1e-6,
                             offset_loss=1e-6, palette_loss_valid=1e-3, palette_loss_distinct=1e-3)
    g = torch.Generator(device=dev).manual_seed(seed + 4)
    K = 49152
    views = [((torch.rand(K, 3, device=dev, generator=g) - 0.5) * 3.0, torch.nn.functional.normalize(torch.randn(K, 3, device=dev, generator=g), dim=-1),
              torch.rand(K, 3, device=dev, generator=g)) for _ in range(4)]
    torch.manual_seed(seed + 1)
    style = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
    st = StyleTrainStep(style, params)
    run = GraphedStyleTrainStep(st, K) if form == "graphed" else st
    losses = []
    for k in range(steps):
        losses.append(run(*views[k % len(views)])[0].detach().float().clone())
    torch.cuda.synchronize()
    opt = st.optimizer
    state = {"loss": torch.stack(losses), "scale": opt._scale.clone(), "step": opt.step_count.clone(),
             "palette": style.color_palette.detach().clone()}
    for k, v in style.named_parameters():
        state["param." + k] = v.detach().clone()
    for i, s in enumerate(opt.state):
        for k, v in s.items():
            state[f"opt.{i}.{k}"] = v.clone()
    return state


if __name__ == "__main__":
    what, form = sys.argv[1], sys.argv[2]
    if what == "nerf":
        st = nerf_run(form, lookahead="lookahead" in sys.argv[3:], perturb="noperturb" not in sys.argv[3:])
    else:
        st = style_run(form)
    assert all(np.isfinite(st["loss"].cpu().numpy())), st["loss"]
    print(digest(st))
