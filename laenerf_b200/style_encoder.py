"""Host-side mirror of the edit-stage CALLER of the hot path (SURVEY.md section 8, row a-13): LAENeRF's style / recolouring
network `editing/style_encoder.py:21-158` and the loop body of `Trainer.train_LAENeRF_step` (nerf/utils.py:953-1045).

What runs on the hot-path kernels here: the stage's own hash grid (`GridEncoder`, L=16, F=2, T=2^19, res 2048*bound -- the same
shape as the NeRF's, editing/style_encoder.py:36-38) forward/backward, the degree-3 SH direction encoding, and the two small
MLPs.  The reference builds those two MLPs with tiny-cuda-nn (`tcnn.Network`, FullyFusedMLP, ReLU, 64 neurons,
`n_hidden_layers = num_layers - 1`, style_encoder.py:65-88), a third-party dependency that is neither vendored nor pinned
(README.md:31-34) -- SURVEY.md section 8c: *parity unpinned* for it.  tcnn's `n_hidden_layers = k` is k+1 matmuls, which is the
topology of `FFMLP(num_layers = k)`; both pad the input width to a multiple of 16 and the output width to 16.  So the nets here
are `FFMLP(num_layers = num_layers - 1)` on the tcgen05 kernels, checked against fp32 torch math (tests/test_gpu_modules.py).
The initialisation is FFMLP's (U(+-sqrt(3/64)), seed 42), not tcnn's Xavier draw.

Out of scope (SURVEY.md section 8: VGG style losses, datasets, GUI): `StyleNetwork` (VGG19 style loss, style_encoder.py:59-61),
the TV / depth-guided image-space losses that need the EditDataset's per-view crops, `distill_color_palettes`' dataset walk.
`style_weight > 0` therefore raises instead of silently training without the style term.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .ffmlp import FFMLP
from .gridencoder import GridEncoder
from .shencoder import SHEncoder


def _attr(params, name, default):
    return getattr(params, name, default) if params is not None else default


class LAENeRF(nn.Module):
    """editing/style_encoder.py:21-158.  `params` is the reference's option namespace (only `bound`, `num_palette_bases`,
    `style_weight` and the loss weights are read)."""

    def __init__(self, params=None, encoding="hashgrid", dir_encoding=None, num_layers=3, hidden_dim=64, color_palette=None,
                 size=256, style_img=None, device="cuda"):
        super().__init__()
        if encoding != "hashgrid":
            raise RuntimeError("LAENeRF: only the hash-grid encoding of the reference configs is built (encoding.py:68-70)")
        self.opt = params
        self.bound = _attr(params, "bound", 2)
        self.encoder = GridEncoder(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=19,
                                   desired_resolution=2048 * self.bound, gridtype="hash", align_corners=False)
        self.in_dim = self.encoder.output_dim
        self.num_layers = num_layers
        self.hidden_dim = hidden_dim
        self.num_color_bases = int(_attr(params, "num_palette_bases", 4))
        if not 1 <= self.num_color_bases <= 16:
            raise RuntimeError("LAENeRF: num_palette_bases must be in [1, 16] (one 16-wide output tile)")
        dev = torch.device(device)
        self.active_palets = torch.ones(self.num_color_bases, dtype=torch.bool, device=dev)
        if color_palette is not None:
            self.color_palette = color_palette
        else:
            self.color_palette = torch.rand((self.num_color_bases, 3), dtype=torch.float32, device=dev)
        self.color_palette.requires_grad = True  # a plain leaf tensor, not an nn.Parameter (style_encoder.py:46-50)
        self.original_color_palette = None
        self.size = size
        self.dir_encoding, self.in_dim_dir = None, 0
        if dir_encoding is not None:
            if dir_encoding != "sphere_harmonics":
                raise RuntimeError("LAENeRF: only the SH direction encoding is built")
            self.dir_encoding = SHEncoder(input_dim=3, degree=3)  # get_encoder(dir_encoding, degree=3), style_encoder.py:57
            self.in_dim_dir = self.dir_encoding.output_dim
        if _attr(params, "style_weight", 0) > 0:
            raise RuntimeError("LAENeRF: the VGG style loss (editing/style_network.py) is out of scope of laenerf_b200")
        # tcnn pads the 32 (+9) inputs to a multiple of 16 with zeros; FFMLP wants the padded width up front
        self.offset_in_dim = (self.in_dim + self.in_dim_dir + 15) // 16 * 16
        self.offset_net = FFMLP(input_dim=self.offset_in_dim, output_dim=3, hidden_dim=hidden_dim, num_layers=num_layers - 1)
        self.weight_net = FFMLP(input_dim=self.in_dim, output_dim=self.num_color_bases, hidden_dim=hidden_dim, num_layers=num_layers - 1)

    # ---- style_encoder.py:93-158 --------------------------------------------------------------------------------------
    def _offset_input(self, x, d):
        offset_in = x
        if self.dir_encoding is not None:
            assert d is not None
            enc_d = self.dir_encoding(d)
            offset_in = torch.cat([offset_in, enc_d.to(x.dtype)], dim=-1)
        pad = self.offset_in_dim - offset_in.shape[-1]
        if pad > 0:
            offset_in = torch.cat([offset_in, torch.zeros(offset_in.shape[0], pad, dtype=offset_in.dtype, device=offset_in.device)], dim=-1)
        return offset_in

    def _active(self):
        """Integer indices of the active palette entries.  The reference indexes with the boolean mask itself (style_encoder.py:95,
        123, 132): every such index is a nonzero() and a device->host synchronisation, three per training iteration.  The indices are
        cached and re-derived when the mask is replaced or written to (its version counter)."""
        m = self.active_palets
        key = (id(m), m._version)
        if getattr(self, "_active_key", None) != key:
            self._active_idx = torch.nonzero(m).flatten()
            self._active_key = key
        return self._active_idx

    def get_weights(self, x):
        x = self.encoder(x, bound=self.bound)
        w_hat = self.weight_net(x)[:, self._active()]
        return torch.softmax(w_hat, -1)

    def get_offsets(self, x, d):
        x = self.encoder(x, bound=self.bound)
        return self.offset_net(self._offset_input(x, d))

    def forward_train(self, x, d=None):
        # x: [N, 3] in [-bound, bound] (the distilled termination points `x_term` of run_cuda_distill); d: [N, 3] unit
        x = self.encoder(x, bound=self.bound)
        act = self._active()
        w_hat = self.weight_net(x)[:, act]
        o_hat = self.offset_net(self._offset_input(x, d))
        o_hat = torch.tanh(o_hat)
        w_hat = torch.softmax(w_hat, -1)
        pred_colors = w_hat @ self.color_palette[act].half() + o_hat
        return torch.clamp(pred_colors, 0, 1), w_hat, o_hat

    def forward(self, x, d=None):
        return self.forward_train(x, d)[0]

    def get_color_palette(self):
        return self.color_palette[self._active()]

    def set_color_palette(self, palet):
        if self.original_color_palette is None:
            self.original_color_palette = self.color_palette.detach().clone()
        with torch.no_grad():
            self.color_palette[self.active_palets] = palet

    # ---- regularisers (style_encoder.py:185-203) ------------------------------------------------------------------------
    def weights_loss(self, pred_bary_weights, params):
        uniform_loss = torch.sum(pred_bary_weights, dim=0).max()
        non_uniform_loss = (1 - pred_bary_weights.max(dim=-1).values).sum()
        return uniform_loss * _attr(params, "weight_loss_uniform", 0.0) + non_uniform_loss * _attr(params, "weight_loss_non_uniform", 0.0)

    def palet_loss(self, params):
        dists = (torch.pow(self.color_palette[:, None, :] - self.color_palette, 2)).sum(-1)
        dist_loss = (1 - dists / dists.max()).mean()
        valid_loss = (torch.floor(self.color_palette) * self.color_palette).sum()
        return valid_loss * _attr(params, "palette_loss_valid", 0.0) + dist_loss * _attr(params, "palette_loss_distinct", 0.0)

    def offset_loss(self, pred_offsets, params):
        return torch.pow(pred_offsets, 2).sum() * _attr(params, "offset_loss", 0.0)

    def get_params(self, lr):  # style_encoder.py:247-255
        return [{"params": self.encoder.parameters(), "lr": lr}, {"params": self.weight_net.parameters(), "lr": lr},
                {"params": self.offset_net.parameters(), "lr": lr}, {"params": self.color_palette, "lr": 2 * lr}]

    def get_params_but_dont_learn_palette(self, lr):
        p = self.get_params(lr)
        p[3]["lr"] = 0
        return p


class StyleTrainStep:
    """One iteration of the loop in `Trainer.train_LAENeRF_step` (nerf/utils.py:983-1034) without the image-space style / TV
    terms: forward_train on one view's masked points, MSE against the recoloured target + the weight / offset / palette
    regularisers, GradScaler backward, Adam(lr 1e-3; palette 2e-3) -- the reference's "naive Adam" (:969-971).

    fused_optimizer (default): `laenerf_b200.optim.AmpAdam` over the style network's own 12.2 M-entry table, the two MLPs and the
    palette -- inf check + unscale + Adam for all four tensors in 2 + 2 launches instead of torch's GradScaler + Adam passes
    (the reference's precision is kept: no autocast around the encoder, fp32 table and fp32 gradients, as nerf/utils.py:983 runs it).
    world_size > 1 = data parallel over VIEWS (SURVEY.md 8e): every rank trains on the masked points of its own view, gradients
    are averaged across ranks inside optimizer.step().  With the fused optimizer that is `laenerf_b200.optim.ShardedFlatAdam`: the
    parameters become views of one peer-mapped fp32 vector, the table gradient accumulates straight into a peer-mapped gradient
    vector, and one kernel averages each rank's slice over NVLink, runs Adam on it and stores the result into every rank's
    parameters.  Where torch symmetric memory is unavailable the gradients are all-reduced with NCCL instead, one collective per
    tensor, and every rank runs the full Adam.  `exchange` records which path runs ("local", "p2p" or "allreduce"; for the last,
    `p2p_error` says why)."""

    def __init__(self, style_encoder: LAENeRF, params=None, lr: float = 1e-3, fused_optimizer: bool = True, world_size: int = 1, rank: int = 0):
        self.model, self.params = style_encoder, params
        self.world = int(world_size)
        self.fused_optimizer = bool(fused_optimizer)
        self.exchange, self.p2p_error = "local", None
        if self.fused_optimizer:
            from .optim import AmpAdam, ShardedFlatAdam
            m = style_encoder
            # get_params(): palette at 2 lr; the table's gradient reaches the sharded optimizer without autograd (persistent)
            owners = [(m.encoder, m.encoder.embeddings, 1.0, False, 0), (m.weight_net, m.weight_net.weights, 1.0, False, 1),
                      (m.offset_net, m.offset_net.weights, 1.0, False, 2), (m, m.color_palette, 2.0, False, 3)]
            self.optimizer = None
            if self.world > 1:
                try:
                    self.optimizer = ShardedFlatAdam([(o[0], o[1], o[2], o[0] is m.encoder, o[4]) for o in owners], lr=lr, betas=(0.9, 0.999),
                                                     eps=1e-8, world_size=self.world, rank=rank, n_groups=4)
                    self.exchange = "p2p"
                except Exception as e:  # never silently: the caller can report which exchange path ran
                    self.p2p_error = f"{type(e).__name__}: {e}"[:300]
            if self.optimizer is None:
                self.optimizer = AmpAdam(None, lr=lr, betas=(0.9, 0.999), eps=1e-8, fp16=True, world_size=1, rank=rank, owners=owners,
                                         n_groups=4)
                self.optimizer.world = self.world  # fp32 tensors only: plain mean all-reduce of the gradients, replicated update
                if self.world > 1:
                    self.exchange = "allreduce"
                    self.optimizer.p2p_error = self.p2p_error
            self.scaler = None
        else:
            self.optimizer = torch.optim.Adam(style_encoder.get_params(lr))
            self.scaler = torch.amp.GradScaler("cuda")
        self.loss_fct = nn.MSELoss()
        self.style_step = 0

    def __call__(self, x_term, d, target):
        m, p = self.model, self.params
        m.train()
        self.style_step += 1
        self.optimizer.zero_grad()
        pred_colors, pred_weight, pred_offset = m.forward_train(x=x_term, d=d)
        loss = self.loss_fct(input=pred_colors, target=target.half())
        loss = loss + m.weights_loss(pred_weight, p).half()
        loss = loss + m.offset_loss(pred_offset, p).half()
        loss = loss + m.palet_loss(p).half()
        if self.fused_optimizer:
            self.optimizer.scale(loss).backward()
            self.optimizer.step()
        else:
            self.scaler.scale(loss).backward()
            if self.world > 1:
                from .parallel import allreduce_gradients
                allreduce_gradients([q for g in self.optimizer.param_groups for q in g["params"]], self.world)
            self.scaler.step(self.optimizer)
            self.scaler.update()
        return loss.detach(), pred_colors.detach()


class GraphedStyleTrainStep:
    """A StyleTrainStep replayed from ONE CUDA graph per point count: forward_train, the four loss terms, the scaled backward and the
    optimizer are ~60 launches of a few microseconds each, so issued from Python the iteration is bound by the interpreter (2.5 ms for
    49 152 points; the kernels take a fraction of that).  Inputs are copied into static device buffers; `loss` / `pred` are views of
    graph-owned memory that the next replay overwrites.  The point count is fixed per capture -- a view's masked points are padded or
    chunked by the caller (the reference feeds one view's mask per step, nerf/utils.py:983-1034).  At world_size > 1 the step must
    use the symmetric-memory exchange (`step.exchange == "p2p"`): the graph then holds the inf check, the two barriers around the
    exchange kernel and the kernel itself, as GraphedTrainStep does for the NeRF; the NCCL fallback all-reduces eagerly and is
    refused."""

    def __init__(self, step: StyleTrainStep, n_points: int):
        if step.world > 1 and step.exchange != "p2p":
            raise RuntimeError("GraphedStyleTrainStep: at world_size > 1 the step must run the symmetric-memory exchange "
                               f"(StyleTrainStep.exchange is {step.exchange!r}: {step.p2p_error})")
        self.step = step
        dev = next(step.model.parameters()).device
        self.x = torch.zeros(n_points, 3, device=dev)
        self.d = torch.zeros(n_points, 3, device=dev)
        self.t = torch.zeros(n_points, 3, device=dev)
        self.graph = None
        self.loss = self.pred = None

    def capture(self, x_term, d, target, warmup: int = 3):
        self.x.copy_(x_term); self.d.copy_(d); self.t.copy_(target)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.step(self.x, self.d, self.t)
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss, self.pred = self.step(self.x, self.d, self.t)

    def __call__(self, x_term, d, target):
        if self.graph is None:
            self.capture(x_term, d, target)
        self.x.copy_(x_term, non_blocking=True); self.d.copy_(d, non_blocking=True); self.t.copy_(target, non_blocking=True)
        self.graph.replay()
        self.step.style_step += 1
        return self.loss, self.pred
