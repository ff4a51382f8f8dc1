"""Ray-sharded graphed training under torch.use_deterministic_algorithms(True), one rank per GPU (started by
torch.distributed.run with 2 processes).  Each rank prints `replica <sha256>` of the state every replica must share (parameters,
density grid, bitfield, AMP scale and step) and `digest <rank> <sha256>` of everything it holds, losses and its Adam slice included."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def main():
    import torch.distributed as dist
    from cases import scene, scene_rays
    from det_driver import digest
    from laenerf_b200.nerf import GraphedTrainStep, NeRFNetwork, TrainStep
    torch.use_deterministic_algorithms(True)
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    sc = scene("lego")
    torch.manual_seed(0)
    m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
    with torch.no_grad():
        m.encoder.embeddings.uniform_(-0.5, 0.5, generator=torch.Generator(device=dev).manual_seed(1))
    m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    step = TrainStep(m, world_size=world)
    g = GraphedTrainStep(step, 4096, perturb=False, lookahead=True)
    losses = []
    for k in range(12):
        _, ro, rd, _ = scene_rays("lego", 4096, 500 + 16 * k + rank)   # every rank its own rays
        gt = torch.rand(4096, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(600 + 16 * k + rank))
        loss = g(torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev), gt)[0]
        if loss is not None:
            losses.append(loss.detach().float().clone())
    losses.append(g.flush()[0].detach().float().clone())
    m.train(False)   # brings the fp32 parameters up to date from the replicated fp16 shadow
    torch.cuda.synchronize()
    opt = step.optimizer
    shared = {"density_grid": m.density_grid, "bitfield": m.density_bitfield, "scale": opt._scale, "step": opt.step_count}
    shared.update({"param." + k: v for k, v in m.named_parameters()})
    mine = dict(shared, loss=torch.stack([l.reshape(()) for l in losses]))
    for i, s in enumerate(opt.state):
        for k, v in s.items():
            mine[f"opt.{i}.{k}"] = v
    print(f"replica {digest(shared)}", flush=True)
    print(f"digest {rank} {digest(mine)}", flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
