"""GPU tier, needs >= 2 GPUs (skipped below): data-parallel training of the edit-stage style network through the symmetric-memory
exchange (StyleTrainStep(world_size=2) -> laenerf_b200.optim.ShardedFlatAdam), eager and then replayed from a CUDA graph.

Each rank trains on its own view's points.  The twin is a single-GPU run whose loss is the mean of the two views' losses: every term
of the style loss is a mean or a sum per view, so its gradient is the mean of the per-rank gradients, and the two runs differ only
by the order of the encoder backward's fp32 atomics and by the fp32 rounding of the two-term mean.  An Adam step moves an entry by
at most about lr whatever its gradient's size, so an entry whose gradient is near zero can step the other way in one run: the
bound on a single entry is steps x lr (x 2 for the palette), while the mean difference must stay at the level of rounding.
"""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STEPS = 6
K = 16384


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _views(dev):
    from types import SimpleNamespace
    params = SimpleNamespace(bound=2.0, num_palette_bases=8, style_weight=0.0, weight_loss_uniform=1e-6, weight_loss_non_uniform=1e-6,
                             offset_loss=1e-6, palette_loss_valid=1e-3, palette_loss_distinct=1e-3)
    g = torch.Generator(device=dev).manual_seed(21)
    views = [((torch.rand(K, 3, device=dev, generator=g) - 0.5) * 3.0, torch.nn.functional.normalize(torch.randn(K, 3, device=dev, generator=g), dim=-1),
              torch.rand(K, 3, device=dev, generator=g)) for _ in range(2)]
    return params, views


def _twin(dev, params, views, steps):
    """Single GPU, loss = mean of the two views' losses (StyleTrainStep's terms), today's optimizer."""
    from laenerf_b200.style_encoder import LAENeRF, StyleTrainStep
    torch.manual_seed(1)
    style = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
    st = StyleTrainStep(style, params)
    m, p, opt = style, params, st.optimizer
    for _ in range(steps):
        m.train()
        opt.zero_grad()
        total = 0
        for x, d, t in views:
            pc, pw, po = m.forward_train(x=x, d=d)
            loss = st.loss_fct(input=pc, target=t.half()) + m.weights_loss(pw, p).half() + m.offset_loss(po, p).half() + m.palet_loss(p).half()
            total = total + loss
        opt.scale(total * 0.5).backward()
        opt.step()
    return style


def _worker(rank, world, port, out):
    import torch.distributed as dist
    from laenerf_b200.style_encoder import GraphedStyleTrainStep, LAENeRF, StyleTrainStep
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    params, views = _views(dev)
    res = {}

    def flat_equal_everywhere(opt):
        full = torch.empty(world, opt.P_pad, device=dev)
        dist.all_gather_into_tensor(full, opt.param_flat.clone())
        return all(torch.equal(full[r], full[0]) for r in range(world))

    for mode in ("eager", "graph"):
        torch.manual_seed(1)
        style = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
        st = StyleTrainStep(style, params, world_size=world, rank=rank)
        res[f"{mode}_exchange"] = st.exchange
        if st.exchange != "p2p":
            res["p2p_error"] = st.p2p_error
            break
        run = st if mode == "eager" else GraphedStyleTrainStep(st, K)
        if mode == "graph":
            run.capture(*views[rank], warmup=1)   # one eager step (lazy allocations stay outside the capture): STEPS + 1 in all
        in_sync = True
        losses = []
        for _ in range(STEPS):
            losses.append(float(run(*views[rank])[0]))
            in_sync &= flat_equal_everywhere(st.optimizer)
        res[f"{mode}_in_sync"] = in_sync
        res[f"{mode}_losses"] = losses
        sd = style.state_dict()
        res[f"{mode}_state_dict_live"] = all(torch.equal(sd[k], v.detach()) for k, v in style.named_parameters())
        res[f"{mode}_moments_slice"] = st.optimizer.state[0]["exp_avg"].numel() == st.optimizer.P_pad // world
        if rank == 0:
            res[f"{mode}_params"] = [style.encoder.embeddings.detach().clone(), style.weight_net.weights.detach().clone(),
                                     style.offset_net.weights.detach().clone(), style.color_palette.detach().clone()]
        dist.barrier()
        torch.cuda.synchronize()
    if rank == 0:
        for mode, steps in (("eager", STEPS), ("graph", STEPS + 1)):
            if f"{mode}_params" in res:
                twin = _twin(dev, params, views, steps)
                ref = [twin.encoder.embeddings.detach(), twin.weight_net.weights.detach(), twin.offset_net.weights.detach(),
                       twin.color_palette.detach()]
                got = res.pop(f"{mode}_params")
                res[f"{mode}_err_max"] = [float((a - b).abs().max()) for a, b in zip(got, ref)]
                res[f"{mode}_err_mean"] = [float((a - b).abs().mean()) for a, b in zip(got, ref)]
        out.put(res)
    dist.barrier()
    torch.cuda.synchronize()
    os._exit(0)   # symmetric memory / captured barriers: leave without tearing NCCL down (see bench.py _finish)


def test_data_parallel_style_training_tracks_the_mean_loss_twin():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = out.get(timeout=600)
    for p in procs:
        p.join(timeout=60)
    assert res["eager_exchange"] == "p2p", res
    for mode in ("eager", "graph"):
        assert res[f"{mode}_in_sync"] and res[f"{mode}_state_dict_live"] and res[f"{mode}_moments_slice"], (mode, res)
        assert all(np.isfinite(res[f"{mode}_losses"])), res
        emax, emean = res[f"{mode}_err_max"], res[f"{mode}_err_mean"]
        bound = (STEPS + (mode == "graph")) * 1e-3 * 1.1   # steps x lr, with 10 % for Adam's early steps slightly above lr
        assert max(emax[:3]) < bound and emax[3] < 2 * bound, (mode, res)
        assert emean[0] < 2e-5 and emean[1] < 2e-4 and emean[2] < 2e-4, (mode, res)
