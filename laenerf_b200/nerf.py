"""Host-side mirror of the reference CALLERS of the hot path, so that tests and bench.py drive the kernels exactly
the way LAENeRF does: `NeRFNetwork.forward/density` (nerf/network_ff.py:11-100) and the `cuda_ray` branches of
`NeRFRenderer.run_cuda` / `run_cuda_distill` (nerf/renderer.py:259-392, 394-480), plus the `Trainer.train_step`
loss/optimizer recipe (nerf/utils.py:535-642, main_nerf.py:223).  This is plumbing around the drop-in modules, not
a re-implementation of the reference's trainer, GUI, datasets or checkpointing (out of scope, SURVEY.md section 8).
"""
from __future__ import annotations

import ctypes as C
import math
import os

import numpy as np
import torch
import torch.nn as nn
from torch.autograd import Function
from torch.amp import custom_bwd, custom_fwd

from . import _native as N
from . import raymarching
from ._shadow import half_of, shadow_f16
from .ffmlp import FFMLP, backward_deterministic
from .gridencoder import GridEncoder
from .shencoder import SHEncoder


class _trunc_exp(Function):  # activation.py:5-17
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return torch.exp(x)

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, g):
        x = ctx.saved_tensors[0]
        return g * torch.exp(x.clamp(-15, 15))


trunc_exp = _trunc_exp.apply


def _recompute_ok(ns, nc) -> bool:
    """Round-2 pair (lean forward + recompute backward, csrc/nerfbwd.cu); LNRF_MLP_RECOMPUTE=0 selects the round-1 save/reload pair."""
    return os.environ.get("LNRF_MLP_RECOMPUTE", "1") != "0" and bool(N.lib().lnrf_nerf_backward_recompute_supported(int(ns), int(nc)))


_WGRAD_SIDE = os.environ.get("LNRF_WGRAD_SIDE", "1") == "1"  # A/B switch: weight-gradient reduction beside the hash-grid backward
_wgrad_scratch_cache = {}


def _wgrad_scratch(dev, nbytes):
    key = (dev.index, nbytes)
    t = _wgrad_scratch_cache.get(key)
    if t is None:
        t = _wgrad_scratch_cache[key] = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    return t


before_network_backward = None  # GraphedTrainStep(lookahead=True) forks the next batch's march here


class _fused_network(Function):
    """NeRFNetwork.forward after the hash-grid encoder (network_ff.py:57-79 + `density_scale * sigma`, renderer.py:299)
    as ONE kernel and its backward as one more (+ the weight-gradient reduction): row f-1 of SURVEY.md section 8.
    Inputs/outputs and every fp16 rounding point are those of the module-by-module path below; the ~25 elementwise /
    cat / cast launches between the MLP kernels are gone.  Training keeps only h = sigma_net(enc) [M,16] fp16 for the backward,
    which recomputes the hidden activations on the tensor cores (lnrf_nerf_forward_lean / lnrf_nerf_backward_recompute).
    m_dev: optional device int32 holding the number of live samples (the marcher's counter): padding rows are skipped."""

    @staticmethod
    def forward(ctx, enc, dirs, w_sigma, w_color, ns, nc, density_scale, train, w_sigma_f16, w_color_f16, gw_sigma_f16, gw_color_f16,
                m_dev=None):
        M = enc.shape[0]
        enc = enc.contiguous()
        dirs = dirs.contiguous().float()
        ws = w_sigma_f16 if w_sigma_f16 is not None else w_sigma.detach().half()
        wc = w_color_f16 if w_color_f16 is not None else w_color.detach().half()
        dev = enc.device
        lean = _recompute_ok(ns, nc)
        if m_dev is not None and not lean:
            m_dev = None
        # with a device-side count the tiles past it are never written; the compositor only indexes live samples, the backward
        # kernels honour the same count
        sigmas = torch.empty(M, dtype=torch.float32, device=dev)
        rgbs = torch.empty(M, 3, dtype=torch.float32, device=dev)
        lib = N.lib()
        if lean:
            h = torch.empty(M, 16, dtype=torch.half, device=dev) if train else None
            N.check(lib.lnrf_nerf_forward_lean(N.ptr(enc), N.ptr(dirs), N.ptr(ws), N.ptr(wc), M, N.ptr(m_dev), ns, nc, float(density_scale),
                                               N.ptr(h), N.ptr(sigmas), N.ptr(rgbs), N.stream()))
            if train:
                ctx.save_for_backward(enc, dirs, ws, wc, h, rgbs, m_dev)
        else:
            fb = cin = h0 = None
            if train:
                fb = torch.empty(ns + nc, M, 64, dtype=torch.half, device=dev)
                cin = torch.empty(M, 32, dtype=torch.half, device=dev)
                h0 = torch.empty(M, dtype=torch.half, device=dev)
            N.check(lib.lnrf_nerf_forward(N.ptr(enc), N.ptr(dirs), N.ptr(ws), N.ptr(wc), M, ns, nc, float(density_scale), int(train),
                                          N.ptr(fb), N.ptr(cin), N.ptr(h0), N.ptr(sigmas), N.ptr(rgbs), N.stream()))
            if train:
                ctx.save_for_backward(enc, ws, wc, fb, cin, h0, rgbs)
        if train:
            ctx.lean = lean
            ctx.cfg = (ns, nc, float(density_scale))
            ctx.gw = (gw_sigma_f16, gw_color_f16)
        return sigmas, rgbs

    @staticmethod
    def backward(ctx, grad_sigmas, grad_rgbs):
        if before_network_backward is not None:
            before_network_backward()
        ns, nc, density_scale = ctx.cfg
        lib = N.lib()
        if ctx.lean:
            enc, dirs, ws, wc, h, rgbs, m_dev = ctx.saved_tensors
        else:
            enc, ws, wc, fb, cin, h0, rgbs = ctx.saved_tensors
            m_dev = None
        M = enc.shape[0]
        dev = enc.device
        grad_sigmas = torch.zeros(M, dtype=torch.float32, device=dev) if grad_sigmas is None else grad_sigmas.contiguous().float()
        grad_rgbs = torch.zeros(M, 3, dtype=torch.float32, device=dev) if grad_rgbs is None else grad_rgbs.contiguous().float()
        grad_enc = torch.empty_like(enc)
        persistent = ctx.gw[0] is not None
        gws = ctx.gw[0] if persistent else torch.empty_like(ws)
        gwc = ctx.gw[1] if persistent else torch.empty_like(wc)
        nbytes = lib.lnrf_nerf_wgrad_scratch_bytes(ns, nc)
        # persistent gradients (AmpAdam): the fixed-order reduction of the per-CTA partial sums runs on a side stream BESIDE the hash-grid
        # backward -- neither depends on the other -- and AmpAdam.step() joins it (N.join_pending); the partial sums then live in a
        # scratch that outlives this call (two streams touch it: no allocator recycling in between)
        side_reduce = persistent and ctx.lean and _WGRAD_SIDE
        scratch = _wgrad_scratch(dev, nbytes) if side_reduce else torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
        if ctx.lean:
            N.check(lib.lnrf_nerf_backward_recompute(N.ptr(grad_sigmas), N.ptr(grad_rgbs), N.ptr(rgbs), N.ptr(h), N.ptr(enc), N.ptr(dirs),
                                                     N.ptr(ws), N.ptr(wc), M, N.ptr(m_dev), ns, nc, density_scale, N.ptr(grad_enc), N.ptr(gws),
                                                     N.ptr(gwc), int(persistent) | (2 if side_reduce else 0), N.ptr(scratch), nbytes, N.stream()))
            if side_reduce:
                with torch.cuda.stream(N.defer_to_side_stream(dev)):
                    N.check(lib.lnrf_nerf_wgrad_reduce(N.ptr(scratch), nbytes, M, ns, nc, N.ptr(gws), N.ptr(gwc), 1, N.stream()))
        else:
            if torch.are_deterministic_algorithms_enabled() and not backward_deterministic(32, 16, 64, ns, 0):
                N.alert_not_deterministic(f"fused NeRF backward with a {ns}-layer sigma net (lnrf_nerf_backward, float-atomics weight gradient)")
            dh = torch.empty(M, 16, dtype=torch.half, device=dev)
            N.check(lib.lnrf_nerf_backward(N.ptr(grad_sigmas), N.ptr(grad_rgbs), N.ptr(rgbs), N.ptr(h0), N.ptr(enc), N.ptr(cin), N.ptr(ws),
                                           N.ptr(wc), N.ptr(fb), M, ns, nc, density_scale, N.ptr(grad_enc), N.ptr(gws), N.ptr(gwc),
                                           int(persistent), N.ptr(dh), N.ptr(scratch), nbytes, N.stream()))
        if persistent:  # AmpAdam reads (and clears) the persistent fp16 buffers; autograd sees no weight gradient
            gws = gwc = None
        return grad_enc, None, gws, gwc, None, None, None, None, None, None, None, None, None


fused_network = _fused_network.apply


class NeRFNetwork(nn.Module):
    """network_ff.NeRFNetwork + the state NeRFRenderer keeps for cuda_ray (renderer.py:72-126)."""

    def __init__(self, bound=1, num_layers=2, hidden_dim=64, geo_feat_dim=15, num_layers_color=3, hidden_dim_color=64,
                 density_scale=1, min_near=0.2, density_thresh=0.01, grid_size=128):
        super().__init__()
        self.bound = bound
        self.cascade = 1 + math.ceil(math.log2(bound))
        self.grid_size = grid_size
        self.density_scale = density_scale
        self.min_near = min_near
        self.density_thresh = density_thresh
        self.bg_radius = -1
        aabb = torch.FloatTensor([-bound, -bound, -bound, bound, bound, bound])
        self.register_buffer("aabb_train", aabb)
        self.register_buffer("aabb_infer", aabb.clone())
        self.register_buffer("density_grid", torch.zeros([self.cascade, grid_size ** 3]))
        self.register_buffer("density_bitfield", torch.zeros(self.cascade * grid_size ** 3 // 8, dtype=torch.uint8))
        self.register_buffer("step_counter", torch.zeros(16, 2, dtype=torch.int32))
        self._mean_host, self._mean_dev = 0.0, None  # behind the mean_density property
        self._tmp_grid = self._occ_scratch = self._occ_mean = self._occ_winner = None
        self.iter_density = 0
        self.mean_count = 0
        self.local_step = 0

        self.geo_feat_dim = geo_feat_dim
        self.encoder = GridEncoder(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=19,
                                   desired_resolution=2048 * bound, gridtype="hash", align_corners=False)  # encoding.py:68-70
        self.in_dim = self.encoder.output_dim
        self.sigma_net = FFMLP(input_dim=self.in_dim, output_dim=1 + geo_feat_dim, hidden_dim=hidden_dim, num_layers=num_layers)
        self.encoder_dir = SHEncoder(input_dim=3, degree=4)
        self.in_dim_color = self.encoder_dir.output_dim + geo_feat_dim + 1  # padded to 32 (network_ff.py:43)
        self.color_net = FFMLP(input_dim=self.in_dim_color, output_dim=3, hidden_dim=hidden_dim_color, num_layers=num_layers_color)
        # fused = True: forward()/the sigma scaling run as the fused kernels of csrc/nerfnet.cu whenever the call has the shape
        # they are built for (fp16 autocast, hidden 64, 16+15+1 colour inputs, sample count a multiple of 128)
        self.fused = True
        self.device_loop = True  # row f-3: inference rounds driven from the device (falls back to the host loop when not fused)
        # round schedule of the device loop.  "reference": run_cuda's n_step rule.  "fast": 8x the sample-buffer memory for ~5x fewer
        # rounds, same per-sample arithmetic.  "auto" (default): "fast" whenever the marcher PROVES the frame's bits do not depend on
        # the round boundaries (every emitted delta exactly representable -- csrc/raymarch.cu, kCtlInexact), otherwise the frame is
        # rendered again on the reference schedule and later frames of this model go there directly: always the reference's bits
        self.render_schedule = "auto"
        self._auto_fast_ok = True
        self.render_samples_per_round = 64  # "fast" only: cap on the samples a ray takes per round after the first
        self.render_clip_far = os.environ.get("LNRF_RENDER_CLIP", "1") == "1"  # device loop: rays end where they leave occupied_box()
        self._occ_box = self._occ_box_key = self._occ_box_work = None
        self.render_row_budget = int(os.environ.get("LNRF_RENDER_ROW_BUDGET", "24"))  # "fast" only: sample-buffer rows per ray of the frame
        self._amp_adam = None  # weak reference to the AmpAdam that owns the fp16 shadows, if any
        self._fused_ok = (hidden_dim == 64 and hidden_dim_color == 64 and geo_feat_dim == 15 and self.in_dim == 32 and
                          self.in_dim_color == 32 and self.encoder_dir.degree == 4)

    def train(self, mode: bool = True):
        # ray-sharded AmpAdam keeps the fp32 masters as per-rank slices: bring the modules' fp32 parameters up to date (from the
        # local fp16 shadow, no collective) before anything evaluates or serialises them
        opt = getattr(self, "_amp_adam", None)
        opt = opt() if opt is not None else None
        if opt is not None and not mode:
            opt.refresh_params()
        return super().train(mode)

    def _use_fused(self, x):
        return (self.fused and self._fused_ok and x.is_cuda and x.dim() == 2 and x.shape[0] > 0 and x.shape[0] % 128 == 0 and
                torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.float16)

    def forward_scaled(self, x, d, m_dev=None):
        """(density_scale * sigma, rgb): what run_cuda feeds the compositor (renderer.py:298-299, 363-364).
        m_dev: optional device int32 with the number of LIVE samples among the rows of x (the training marcher's counter): the
        sample buffer is sized for the largest batch, the rows past the count are zero padding that the reference pushes through
        encoder and MLPs like real samples (SURVEY.md Appendix C-7); with the count the fused kernels skip those 128-row tiles
        (their sigma / rgb rows stay unwritten -- no ray refers to them -- and they receive no gradient)."""
        if self._use_fused(x):
            sn, cn = self.sigma_net, self.color_net
            if m_dev is not None and not (_recompute_ok(sn.num_layers, cn.num_layers) and os.environ.get("LNRF_DEVICE_COUNT", "1") != "0"):
                m_dev = None
            enc = self.encoder(x, bound=self.bound, b_dev=m_dev)
            train = torch.is_grad_enabled() and (enc.requires_grad or self.sigma_net.weights.requires_grad)
            return fused_network(enc, d, sn.weights, cn.weights, sn.num_layers, cn.num_layers, self.density_scale, train,
                                 shadow_f16(sn, sn.weights), shadow_f16(cn, cn.weights),
                                 getattr(sn, "_grad_f16", None), getattr(cn, "_grad_f16", None), m_dev)
        sigmas, rgbs = self(x, d)
        return self.density_scale * sigmas, rgbs

    # ---- network_ff.py:51-79 -------------------------------------------------------------------------------
    def forward(self, x, d):
        x = self.encoder(x, bound=self.bound)
        h = self.sigma_net(x)
        sigma = trunc_exp(h[..., 0])
        geo_feat = h[..., 1:]
        d = self.encoder_dir(d)
        p = torch.zeros_like(geo_feat[..., :1])
        h = torch.cat([d, geo_feat, p], dim=-1)
        h = self.color_net(h)
        rgb = torch.sigmoid(h)
        return sigma, rgb

    def density(self, x):  # network_ff.py:81-95
        x = self.encoder(x, bound=self.bound)
        h = self.sigma_net(x)
        return {"sigma": trunc_exp(h[..., 0]), "geo_feat": h[..., 1:]}

    # ---- occupancy state ---------------------------------------------------------------------------------------
    def set_density_grid(self, density_grid: torch.Tensor, thresh: float | None = None):
        """Install a [C, H^3] Morton-ordered density grid and derive the bitfield (renderer.py:640-641)."""
        self.density_grid.copy_(density_grid)
        self.mean_density = float(self.density_grid.clamp(min=0).mean().item())
        t = min(self.mean_density, self.density_thresh) if thresh is None else thresh
        raymarching.packbits(self.density_grid, t, self.density_bitfield)
        self._bitfield_written()

    # ---- renderer.py:556-649 (row f-2) ----------------------------------------------------------------------------
    def _density_scaled(self, xyzs):
        """density_scale * sigma of `xyzs` ([M,3] world coordinates): the fused encode + sigma-net path when available."""
        M = xyzs.shape[0]
        if self.fused and self._fused_ok and xyzs.is_cuda and torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.float16:
            from .gridencoder import _offsets_host
            enc, sn = self.encoder, self.sigma_net
            emb, ws = half_of(enc, enc.embeddings), half_of(sn, sn.weights)
            Mp = (M + 127) // 128 * 128
            if Mp != M:
                xyzs = torch.cat([xyzs, torch.zeros(Mp - M, 3, dtype=xyzs.dtype, device=xyzs.device)], 0)
            feat = torch.empty(Mp, 32, dtype=torch.half, device=xyzs.device)
            sig = torch.empty(Mp, dtype=torch.float32, device=xyzs.device)
            lib, st = N.lib(), N.stream()
            N.check(lib.lnrf_grid_encode_forward_world(N.ptr(xyzs), float(self.bound), N.ptr(emb), N.ptr(_offsets_host(enc.offsets)), N.ptr(feat),
                                                       Mp, None, int(enc.num_levels), float(np.log2(enc.per_level_scale)),
                                                       int(enc.base_resolution), int(enc.gridtype_id), int(bool(enc.align_corners)),
                                                       int(enc.interp_id), N.F16, st))
            N.check(lib.lnrf_nerf_density(N.ptr(feat), N.ptr(ws), Mp, int(sn.num_layers), float(self.density_scale), N.ptr(sig), st))
            return sig[:M]
        sig = self.density(xyzs)["sigma"].reshape(-1).detach().float()
        return sig * self.density_scale

    @property
    def mean_density(self):
        """mean(clamp(density_grid, 0)) of the last update; kept on the device, read (one sync) only when somebody asks."""
        if self._mean_dev is not None:
            self._mean_host = float(self._mean_dev[0].item())
            self._mean_dev = None
        return self._mean_host

    @mean_density.setter
    def mean_density(self, v):
        self._mean_host, self._mean_dev = float(v), None

    @torch.no_grad()
    def update_extra_state(self, decay=0.95, S=128):
        """NeRFRenderer.update_extra_state (renderer.py:556-649): re-sample the density grid (all cells for the first 16
        updates, then H^3/4 random + H^3/4 occupied cells per cascade), EMA-max it into `density_grid`, rebuild the
        bitfield from min(mean density, density_thresh), refresh `mean_count`.  The random numbers are drawn with the
        reference's torch calls in the reference's order; everything else runs in csrc/occupancy.cu, and nothing on the
        path waits for the device (the reference's mean().item() becomes a device-side threshold)."""
        H, Cc = self.grid_size, self.cascade
        dev = self.density_bitfield.device
        lib, st = N.lib(), N.stream()
        if self._tmp_grid is None or self._tmp_grid.device != dev:
            self._tmp_grid = -torch.ones_like(self.density_grid)
            self._occ_scratch = torch.empty(lib.lnrf_occupancy_scratch_bytes() // 4, dtype=torch.float32, device=dev)
            self._occ_mean = torch.zeros(2, dtype=torch.float32, device=dev)
        tmp = self._tmp_grid
        for cas in range(Cc):
            bound_c = min(2 ** cas, self.bound)
            if self.iter_density < 16:  # full update
                n = H ** 3
                coords = None
                indices = torch.empty(n, dtype=torch.int32, device=dev)
            else:  # partial update: random cells + random occupied cells
                n4 = H ** 3 // 4
                coords = torch.randint(0, H, (n4, 3), device=dev)
                occ_indices = torch.nonzero(self.density_grid[cas] > 0).squeeze(-1)
                rand_mask = torch.randint(0, occ_indices.shape[0], [n4], dtype=torch.long, device=dev)
                occ_coords = raymarching.morton3D_invert(occ_indices[rand_mask])
                coords = torch.cat([coords.int(), occ_coords], dim=0).contiguous()
                n = coords.shape[0]
                indices = torch.empty(n, dtype=torch.int32, device=dev)
            u = torch.rand(n, 3, device=dev)  # rand_like(cas_xyzs)
            xyzs = torch.empty(n, 3, dtype=torch.float32, device=dev)
            N.check(lib.lnrf_occupancy_points(N.ptr(coords), N.ptr(u), n, H, float(bound_c), N.ptr(xyzs), N.ptr(indices), st))
            sig = self._density_scaled(xyzs).contiguous()
            if torch.are_deterministic_algorithms_enabled():  # partial updates draw cells with repeats: the last occurrence wins
                if self._occ_winner is None or self._occ_winner.device != dev:
                    self._occ_winner = torch.full((H ** 3,), -1, dtype=torch.int32, device=dev)  # re-armed by the kernel
                N.check(lib.lnrf_occupancy_scatter_det(N.ptr(sig), N.ptr(indices), n, N.ptr(tmp[cas]), N.ptr(self._occ_winner), H ** 3, st))
            else:
                N.check(lib.lnrf_occupancy_scatter(N.ptr(sig), N.ptr(indices), n, N.ptr(tmp[cas]), st))
        N.check(lib.lnrf_occupancy_ema(N.ptr(self.density_grid), N.ptr(tmp), self.density_grid.numel(), float(decay), float(self.density_thresh),
                                       N.ptr(self._occ_mean), N.ptr(self._occ_scratch), self._occ_scratch.numel() * 4, st))
        self._mean_dev = self._occ_mean
        self.iter_density += 1
        N.check(lib.lnrf_packbits_dev(N.ptr(self.density_grid), self.density_bitfield.numel(), N.ptr(self._occ_mean[1:]),
                                      N.ptr(self.density_bitfield), st))
        self._bitfield_written()  # written through a raw pointer: torch's version counter does not see it (occupied_box)
        self.update_mean_count()

    @torch.no_grad()
    def mark_untrained_grid(self, poses, intrinsic, S=64, filter_close_point=False):
        """NeRFRenderer.mark_untrained_grid (renderer.py:483-554, the other half of row f-2): cells of every cascade that no
        training camera sees (or that lie closer than `min_near` to one) get density -1, so update_extra_state never revives
        them.  Same predicate per (cell, camera) as the reference; evaluated for all H^3 cells of a cascade at once in Morton
        order (one `morton3D` call instead of the reference's 8 x 8 x 8 Python block loop), cameras in chunks of S."""
        if isinstance(poses, np.ndarray):
            poses = torch.from_numpy(poses)
        dev = self.density_bitfield.device
        H = self.grid_size
        fx, fy, cx, cy = (float(v) for v in intrinsic)
        poses = poses.to(dev).float()
        ar = torch.arange(H, dtype=torch.int32, device=dev)
        coords = torch.stack(torch.meshgrid(ar, ar, ar, indexing="ij"), dim=-1).reshape(-1, 3).contiguous()  # [H^3, 3] in [0, H)
        indices = raymarching.morton3D(coords).long()
        world = 2 * coords.float() / (H - 1) - 1  # [-1, 1]
        count = torch.zeros_like(self.density_grid)
        too_close = torch.zeros_like(self.density_grid)
        chunk = max(1, min(int(S), 16))  # [chunk, H^3, 3] fp32 temporaries
        for cas in range(self.cascade):
            bound = min(2 ** cas, self.bound)
            half_grid_size = bound / H
            cas_world = (world * (bound - half_grid_size)).unsqueeze(0)
            seen = torch.zeros(H ** 3, dtype=torch.float32, device=dev)
            close = torch.zeros(H ** 3, dtype=torch.float32, device=dev)
            for head in range(0, poses.shape[0], chunk):
                P = poses[head:head + chunk]
                cam = (cas_world - P[:, :3, 3].unsqueeze(1)) @ P[:, :3, :3]  # world -> camera (poses are c2w)
                z = cam[:, :, 2]
                inside = (z > 0) & (cam[:, :, 0].abs() < cx / fx * z + half_grid_size * 2) & (cam[:, :, 1].abs() < cy / fy * z + half_grid_size * 2)
                seen += inside.sum(0)
                close += ((z < self.min_near) & inside).sum(0)
                if filter_close_point:
                    close += (cam.norm(dim=-1) < self.min_near).sum(0)
            count[cas, indices] = seen
            too_close[cas, indices] = close
        count = count * (too_close == 0)
        self.density_grid[count == 0] = -1
        return int((count == 0).sum().item())

    def update_mean_count(self):
        """The step-counter part of update_extra_state (renderer.py:643-647)."""
        total_step = min(16, self.local_step)
        if total_step > 0:
            self.mean_count = int(self.step_counter[:total_step, 0].sum().item() / total_step)
        self.local_step = 0

    @torch.no_grad()
    def occupied_box(self):
        """Device float[6] {lo xyz, hi xyz}: a world-space box around every occupied cell of density_bitfield on every cascade, two
        cells of margin (include/laenerf_b200.h lnrf_occupied_box).  One launch into a PERSISTENT buffer (CUDA graphs that captured
        its address keep seeing the current box) whenever the bitfield changed: torch's version counter for torch writes, an explicit
        invalidation where this module writes it through a raw pointer (set_density_grid, update_extra_state)."""
        bf = self.density_bitfield
        key = (bf.data_ptr(), bf._version)
        if self._occ_box_key != key:
            dev, H, Cn = bf.device, int(self.grid_size), int(self.cascade)
            if self._occ_box is None or self._occ_box.device != dev:
                self._occ_box = torch.empty(6, dtype=torch.float32, device=dev)
                self._occ_box_work = torch.tensor([H, H, H, -1, -1, -1] * Cn + [0], dtype=torch.int32, device=dev)
            N.check(N.lib().lnrf_occupied_box(bf.data_ptr(), Cn, H, float(self.bound), self._occ_box_work.data_ptr(), self._occ_box.data_ptr(),
                                              N.stream()))
            self._occ_box_key = key
        return self._occ_box

    def _bitfield_written(self):
        """density_bitfield was rewritten through a raw pointer: refresh the box now (eagerly: replays of a captured step read it)."""
        self._occ_box_key = None
        if self.render_clip_far and self.density_bitfield.is_cuda:
            self.occupied_box()

    # ---- row f-3: the inference loop of run_cuda / run_cuda_distill driven from the device -----------------------------
    def _render_rounds_device(self, rays_o, rays_d, nears, fars, dens_grid, edit_bitfield, dt_gamma, perturb, max_steps, T_thresh,
                              rounds_per_call: int = 8):
        """The device loop on self.render_schedule.  "auto" renders on the fast schedule and makes the result the reference
        schedule's, bit for bit:

          * no ray emitted an inexact delta after round 0 (csrc/raymarch.cu, kCtlInexact): the round boundaries leave no trace -- done;
          * some rays did (cameras inside the volume): only THEIR results depend on where the boundaries fall.  Every other ray dies at
            the same sample on any schedule, and the fast pass recorded that sample index for all rays (`ray_steps`), so the reference's
            n_step sequence -- a function of how many rays are alive after each round -- follows from the histogram of those indices
            (`_reference_sequence`).  The flagged rays alone are rendered again with that sequence prescribed (`nstep_seq`), i.e. exactly
            as the reference's full-frame loop would render them, and take their places in the outputs.  Their own death indices may
            move in that pass; the sequence is recomputed and the pass repeated until it reproduces itself (a fixed point IS the
            reference's run: by induction over the rounds both make the same n_step decisions) -- in practice at once;
          * the max_steps cap cut rays off, or no fixed point after three passes: the frame is rendered on the reference schedule."""
        sched = self.render_schedule
        args = (rays_o, rays_d, nears, fars, dens_grid, edit_bitfield, dt_gamma, perturb, max_steps, T_thresh, rounds_per_call)
        if sched != "auto":
            return self._render_rounds_on(sched, *args)
        if self._auto_fast_ok and not perturb:
            t = self._render_rounds_on("fast", *args, track=True)
            if not t["schedule_dependent"]:
                t["schedule"] = "fast (proven bit-identical to the reference schedule for this frame)"
                return t
            fixed = self._fix_schedule_dependent_rays(t, *args) if (t["inexact_rays"] > 0 and not t["cap_cut"]) else None
            if fixed is not None:
                return fixed
            self._auto_fast_ok = False  # the cap cut rays off / no fixed point: this scene goes to the reference schedule directly
        t = self._render_rounds_on("reference", *args)
        t["schedule"] = "reference"
        return t

    @staticmethod
    def _reference_sequence(hist, n_rays, max_steps):
        """n_step of every round of the reference loop (renderer.py:353-379) from the histogram of the rays' death sample indices:
        a ray that completes k samples in total is alive at the start of a round iff the rounds before it handed out <= k samples."""
        alive_from = np.concatenate([np.cumsum(hist[::-1])[::-1], [0]])  # alive_from[b] = rays with k >= b
        seq, b = [], 0
        while b < max_steps:
            alive = int(alive_from[min(b, len(alive_from) - 1)])
            if alive <= 0:
                break
            n = max(min(n_rays // alive, 8), 1)
            seq.append(n)
            b += n
        return seq

    def _fix_schedule_dependent_rays(self, t, rays_o, rays_d, nears, fars, dens_grid, edit_bitfield, dt_gamma, perturb, max_steps, T_thresh,
                                     rounds_per_call):
        """Re-render the rays the fast pass flagged on the reference's n_step sequence -- all rounds in ONE pass
        (lnrf_march_rays_prescribed -> network -> lnrf_composite_rays_prescribed, see include/laenerf_b200.h) -- and put the results
        in their places.  LNRF_FIXUP_ROUNDS=1 runs the same sequence round by round through lnrf_render_rounds instead."""
        n_rays = rays_o.shape[0]
        dev = rays_o.device
        cap = int(max_steps) + 72
        idx = t["ray_flags"].nonzero().flatten()
        nf = int(idx.numel())
        if nf == 0:
            return None
        steps = t["ray_steps"].long().clamp_(max=cap)
        hist = torch.bincount(steps, minlength=cap + 1).cpu().numpy().astype(np.int64)
        sub_steps = steps[idx]
        sub = [x[idx].contiguous() for x in (rays_o, rays_d, nears, fars)]
        by_rounds = os.environ.get("LNRF_FIXUP_ROUNDS", "0") == "1"
        use_caps = os.environ.get("LNRF_FIXUP_CAPS", "1") == "1"
        distill = edit_bitfield is not None
        lib, st = N.lib(), N.stream()
        for _ in range(4):
            seq = self._reference_sequence(hist, n_rays, max_steps)
            if not seq:
                return None
            seq_dev = torch.tensor(seq, dtype=torch.int32, device=dev)
            if by_rounds:
                t2 = self._render_rounds_on("prescribed", *sub, dens_grid, edit_bitfield, dt_gamma, perturb, max_steps, T_thresh, rounds_per_call,
                                            track=True, seq=seq_dev)
                rounds2, slots2 = t2["rounds"], t2["slots"]
            else:
                so, sd, sn_, sf = sub
                counts = torch.empty(nf, dtype=torch.int32, device=dev)
                box = t.get("occupied_box")
                geo = (float(self.bound), float(dt_gamma), int(max_steps), int(self.cascade), int(self.grid_size), dens_grid.data_ptr(),
                       edit_bitfield.data_ptr() if distill else None, seq_dev.data_ptr(), len(seq))
                f32 = dict(dtype=torch.float32, device=dev)

                def march(caps):
                    """Samples of the flagged rays on `seq`, back to back.  caps: most samples per ray (offsets = their prefix sum: one
                    marching pass); None: a counting pass first, every ray to its far end."""
                    if caps is None:
                        N.check(lib.lnrf_march_rays_prescribed(nf, so.data_ptr(), sd.data_ptr(), sn_.data_ptr(), sf.data_ptr(), *geo, None,
                                                               counts.data_ptr(), None, None, None, None, None, N.ptr(box), st))
                        sizes = counts
                    else:
                        sizes = caps
                    ends = torch.cumsum(sizes, 0, dtype=torch.int32)
                    offsets = (ends - sizes).contiguous()
                    total = int(ends[-1].item())
                    rows = total + 128 - total % 128  # raymarching.py:331-332 padding rule; unused rows are zeros
                    bufs = (torch.zeros(rows, 3, **f32), torch.zeros(rows, 3, **f32), torch.zeros(rows, 2, **f32),
                            torch.zeros(rows, dtype=torch.uint8, device=dev) if distill else None)
                    N.check(lib.lnrf_march_rays_prescribed(nf, so.data_ptr(), sd.data_ptr(), sn_.data_ptr(), sf.data_ptr(), *geo, offsets.data_ptr(),
                                                           counts.data_ptr(), bufs[0].data_ptr(), bufs[1].data_ptr(), bufs[2].data_ptr(),
                                                           N.ptr(bufs[3]), N.ptr(caps), N.ptr(box), st))
                    return offsets, rows, bufs

                # the fast pass knows where each ray died; on the reference's sequence it dies within a few samples of that
                seq_total = int(sum(seq))
                caps = (sub_steps + 96).clamp(max=seq_total).int().contiguous() if use_caps else None
                offsets, rows, (xyzs, dirs, deltas, edit_occ) = march(caps)
                sigmas, rgbs = self.forward_scaled(xyzs, dirs)
                sigmas, rgbs = sigmas.float().contiguous(), rgbs.float().contiguous()
                t2 = dict(weights_sum=torch.empty(nf, **f32), depth=torch.empty(nf, **f32), image=torch.empty(nf, 3, **f32),
                          wes=torch.empty(nf, **f32) if distill else None, de=torch.empty(nf, **f32) if distill else None,
                          ray_steps=torch.empty(nf, dtype=torch.int32, device=dev))
                N.check(lib.lnrf_composite_rays_prescribed(nf, float(T_thresh), offsets.data_ptr(), counts.data_ptr(), sn_.data_ptr(),
                                                           sigmas.data_ptr(), rgbs.data_ptr(), deltas.data_ptr(), N.ptr(edit_occ),
                                                           t2["weights_sum"].data_ptr(), N.ptr(t2["wes"]), t2["depth"].data_ptr(), N.ptr(t2["de"]),
                                                           t2["image"].data_ptr(), t2["ray_steps"].data_ptr(), st))
                rounds2, slots2 = len(seq), rows
                if caps is not None:
                    # a ray that used up its cap without dying (neither T_thresh nor the end of its samples) was cut short: redo the
                    # pass without caps (never seen on the three scene shapes; the margin is 96 samples)
                    cut = (t2["ray_steps"] == counts) & (counts == caps) & (caps < seq_total)
                    if bool(cut.any().item()):
                        use_caps = False
                        continue
            new_steps = t2["ray_steps"].long().clamp_(max=cap)
            hist = hist - torch.bincount(sub_steps, minlength=cap + 1).cpu().numpy() + torch.bincount(new_steps, minlength=cap + 1).cpu().numpy()
            sub_steps = new_steps
            seq2 = self._reference_sequence(hist, n_rays, max_steps)
            # the flagged rays only see the rounds up to the death of the last of them
            last, b, need = int(new_steps.max().item()), 0, 0
            for need, n in enumerate(seq2, 1):
                b += n
                if b > last:
                    break
            if seq2[:need] == seq[:need]:
                for k in ("weights_sum", "depth", "image", "wes", "de"):
                    if t.get(k) is not None:
                        t[k][idx] = t2[k]
                t["schedule"] = (f"fast + {nf} schedule-dependent rays re-rendered on the reference's n_step sequence "
                                 f"({len(seq)} rounds, from the histogram of the rays' death samples" +
                                 ("" if by_rounds else "; all rounds in one pass") + "): bit-identical to the reference schedule")
                t["rounds_fixup"], t["slots"] = rounds2, t["slots"] + slots2
                return t
        return None

    def _render_rounds_on(self, schedule, rays_o, rays_d, nears, fars, dens_grid, edit_bitfield, dt_gamma, perturb, max_steps, T_thresh,
                          rounds_per_call: int = 8, track: bool = False, seq=None):
        """renderer.py:335-387 (and :425-470 with an edit grid) without a host synchronisation per round: the kernels read
        n_alive / n_step from a control block in device memory that the compaction kernel updates (csrc/render.cu); the
        host queues `rounds_per_call` rounds at a time and only then looks at the `finished` flag.  Same kernels, same
        order, same per-round geometry as the host loop -- the results are bit-identical to it."""
        from .gridencoder import _offsets_host
        n_rays = rays_o.shape[0]
        dev = rays_o.device
        f32 = dict(dtype=torch.float32, device=dev)
        # "reference": n_step = clamp(n_rays / n_alive, 1, 8), buffers of n_rays + 128 rows (renderer.py:357) -- bit-identical to the
        # host loop.  "fast": buffers of 8 n_rays + 128 rows; the first round (n_step = 1) weeds out the rays that miss, every later
        # round takes up to render_samples_per_round samples per ray -- several times fewer rounds, each of which costs ~90 us of
        # latency whatever its size
        fast = schedule == "fast"
        # "fast": a round's row budget is render_row_budget (24) x n_rays -- rounds >= 1 are compact (csrc/raymarch.cu
        # k_march_infer_compact: no empty slots), so the budget only bounds the worst case and what it costs is address space --, or -- for the small ray sets a rank renders when a frame is tile-sharded over many
        # GPUs -- up to 4 M rows: every round costs ~100 us of latency whatever its size (march of the longest gap + four dependent
        # launches), so a small ray set should finish in as few rounds as possible (up to 64 samples per ray per round)
        rows = (max(self.render_row_budget * n_rays, min(64 * n_rays, 1 << 22)) if fast else n_rays) + 128
        if schedule == "prescribed":  # n_step per round from `seq` (at most 8): a subset of a frame on the full frame's schedule
            rows = 8 * n_rays + 128
        distill = edit_bitfield is not None
        enc, sn, cn = self.encoder, self.sigma_net, self.color_net
        emb, ws, wc = half_of(enc, enc.embeddings), half_of(sn, sn.weights), half_of(cn, cn.weights)
        t = dict(
            ctl=torch.zeros(32, dtype=torch.int32, device=dev),
            ray_steps=torch.empty(n_rays, dtype=torch.int32, device=dev) if track else None,
            ray_flags=torch.empty(n_rays, dtype=torch.uint8, device=dev) if track else None,
            alive0=torch.empty(n_rays, dtype=torch.int32, device=dev), alive1=torch.empty(n_rays, dtype=torch.int32, device=dev),
            rays_t=torch.empty(n_rays, **f32), xyzs=torch.empty(rows, 3, **f32), dirs=torch.empty(rows, 3, **f32),
            deltas=torch.empty(rows, 2, **f32), enc=torch.empty(rows, 32, dtype=torch.half, device=dev),
            sigmas=torch.empty(rows, **f32), rgbs=torch.empty(rows, 3, **f32),
            weights_sum=torch.empty(n_rays, **f32), depth=torch.empty(n_rays, **f32), image=torch.empty(n_rays, 3, **f32),
            noises=torch.rand(n_rays, **f32) if perturb else None,
            edit_occ=torch.empty(rows, dtype=torch.uint8, device=dev) if distill else None,
            wes=torch.empty(n_rays, **f32) if distill else None, de=torch.empty(n_rays, **f32) if distill else None,
        )
        lib = N.lib()
        nbytes = lib.lnrf_render_scratch_bytes(n_rays)
        t["scratch"] = torch.zeros((nbytes + 7) // 8, dtype=torch.int64, device=dev)
        off_h = _offsets_host(enc.offsets)
        d = N.RenderDesc()
        d.ctl, d.n_rays, d.max_steps = t["ctl"].data_ptr(), n_rays, int(max_steps)
        d.rays_o, d.rays_d, d.nears, d.fars = rays_o.data_ptr(), rays_d.data_ptr(), nears.data_ptr(), fars.data_ptr()
        d.density_bitfield = dens_grid.data_ptr()
        d.edit_bitfield = edit_bitfield.data_ptr() if distill else None
        d.bound, d.dt_gamma, d.T_thresh = float(self.bound), float(dt_gamma), float(T_thresh)
        d.cascade, d.grid_size = int(self.cascade), int(self.grid_size)
        d.first_round_noises = N.ptr(t["noises"])
        d.embeddings_f16, d.offsets_host = emb.data_ptr(), off_h.data_ptr()
        d.num_levels, d.base_resolution = int(enc.num_levels), int(enc.base_resolution)
        d.gridtype, d.interpolation, d.align_corners = int(enc.gridtype_id), int(enc.interp_id), int(bool(enc.align_corners))
        d.level_scale_log2 = float(np.log2(enc.per_level_scale))
        d.w_sigma_f16, d.w_color_f16 = ws.data_ptr(), wc.data_ptr()
        d.num_layers_sigma, d.num_layers_color, d.density_scale = int(sn.num_layers), int(cn.num_layers), float(self.density_scale)
        d.rays_alive[0], d.rays_alive[1], d.rays_t = t["alive0"].data_ptr(), t["alive1"].data_ptr(), t["rays_t"].data_ptr()
        d.xyzs, d.dirs, d.deltas = t["xyzs"].data_ptr(), t["dirs"].data_ptr(), t["deltas"].data_ptr()
        d.edit_occ, d.enc_f16 = N.ptr(t["edit_occ"]), t["enc"].data_ptr()
        d.sigmas, d.rgbs = t["sigmas"].data_ptr(), t["rgbs"].data_ptr()
        d.weights_sum, d.depth, d.image = t["weights_sum"].data_ptr(), t["depth"].data_ptr(), t["image"].data_ptr()
        d.weights_edit_sum, d.depth_edit = N.ptr(t["wes"]), N.ptr(t["de"])
        d.scratch, d.scratch_bytes = t["scratch"].data_ptr(), nbytes
        d.sample_rows = rows if (fast or seq is not None) else 0
        d.samples_per_round = int(self.render_samples_per_round) if fast else (8 if seq is not None else 0)
        d.ray_steps, d.ray_flags = N.ptr(t["ray_steps"]), N.ptr(t["ray_flags"])
        d.nstep_seq, d.nstep_len = (seq.data_ptr(), int(seq.numel())) if seq is not None else (None, 0)
        # every schedule: a ray ends where it leaves the box around the occupied cells (exact: nothing is ever sampled beyond it)
        t["occupied_box"] = self.occupied_box() if (self.render_clip_far and dens_grid is self.density_bitfield) else None
        d.occupied_box = N.ptr(t["occupied_box"])
        st = N.stream()
        N.check(lib.lnrf_render_begin(C.byref(d), st))
        launched = 0
        if seq is not None:
            rounds_per_call = 32  # a prescribed schedule is run for a few thousand rays: tiny rounds, fewer host look-ups
        max_rounds = int(max_steps)  # n_step >= 1: the reference loop cannot run more rounds than this
        while launched < max_rounds:
            # fast schedule: a frame takes ~8-10 rounds, the last of them tiny; rounds queued behind the end of the frame are no-ops
            # that still cost five launches (~40 us) each, so after the first batch the host looks more often
            k = min(rounds_per_call if (launched == 0 or not fast) else max(2, rounds_per_call // 3), max_rounds - launched)
            N.check(lib.lnrf_render_rounds(C.byref(d), launched, k, st))
            launched += k
            ctl = t["ctl"].tolist()  # the one synchronisation per batch of rounds
            if ctl[6]:
                break
        t["rounds"], t["steps"], t["slots"] = ctl[7], ctl[2], ctl[9]
        t["schedule_dependent"] = bool(ctl[12])
        t["inexact_rays"] = int(ctl[13])
        t["cap_cut"] = bool(ctl[14])
        t["schedule"] = schedule
        return t

    def _device_loop_ok(self, rays_o):
        return (self.fused and self._fused_ok and rays_o.is_cuda and rays_o.shape[0] > 0 and torch.is_autocast_enabled() and
                torch.get_autocast_dtype("cuda") == torch.float16 and not torch.is_grad_enabled())

    # ---- the training branch of run_cuda (renderer.py:284-333) in two halves: everything that depends only on the rays
    # (near/far + occupancy-grid march) and everything that depends on the parameters (network, compositing).  run_cuda runs
    # them back to back; GraphedTrainStep(lookahead=True) runs the first half of the NEXT batch beside the second half of
    # the current one.
    def _march_train_from(self, rays_o, rays_d, nears, fars, dens_grid, perturb, force_all_rays, dt_gamma, max_steps, into=None):
        """`into`: a dict of a previous march of the same shape (and its own `counter`) to overwrite -- the second sample buffer of a
        software-pipelined loop; the step counter history is then the caller's business."""
        if into is not None:
            counter = into["counter"]
        else:
            counter = self.step_counter[self.local_step % 16]
            self.local_step += 1
        counter.zero_()
        out = None if into is None else (into["xyzs"], into["dirs"], into["deltas"], into["rays"])
        box = self.occupied_box() if (self.render_clip_far and dens_grid is self.density_bitfield) else None
        xyzs, dirs, deltas, rays = raymarching.march_rays_train(rays_o, rays_d, self.bound, dens_grid, self.cascade,
                                                                self.grid_size, nears, fars, counter, self.mean_count, perturb,
                                                                128, force_all_rays, dt_gamma, max_steps, out, box)
        if into is not None:
            into["nears"].copy_(nears)
            into["fars"].copy_(fars)
            return into
        return dict(xyzs=xyzs, dirs=dirs, deltas=deltas, rays=rays, nears=nears, fars=fars, counter=counter)

    def march_train(self, rays_o, rays_d, perturb=True, force_all_rays=False, dt_gamma=0, max_steps=1024, edit_grid=None, into=None):
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, self.aabb_train, self.min_near)
        dens_grid = edit_grid if edit_grid is not None else self.density_bitfield
        return self._march_train_from(rays_o, rays_d, nears, fars, dens_grid, perturb, force_all_rays, dt_gamma, max_steps, into)

    def shade_train(self, marched, bg_color=1, T_thresh=1e-4, prefix=None, scale_depth=True):
        xyzs, dirs, deltas, rays, nears, fars = (marched[k] for k in ("xyzs", "dirs", "deltas", "rays", "nears", "fars"))
        prefix = (rays.shape[0],) if prefix is None else prefix
        sigmas, rgbs = self.forward_scaled(xyzs, dirs, marched.get("counter"))
        weights_sum, depth, image = raymarching.composite_rays_train(sigmas, rgbs, deltas, rays, T_thresh)
        image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
        if scale_depth:
            depth = torch.clamp(depth - nears, min=0) / (fars - nears)
        return {"image": image.view(*prefix, 3), "depth": depth.view(*prefix), "weights_sum": weights_sum, "nears": nears,
                "num_points": xyzs.shape[0]}

    def shade_loss_train(self, marched, gt_rgb, bg_color=1, T_thresh=1e-4, prefix=None, scale_depth=True, grad_scale=None):
        """shade_train + the trainer's MSE (nerf/utils.py:592,633) with the whole tail behind the network -- compositing,
        background blend, depth normalisation, loss -- as one launch each way (row f-5, raymarching.composite_loss_train).
        Returns (loss, results) with the same `results` dict as shade_train."""
        xyzs, dirs, deltas, rays, nears, fars = (marched[k] for k in ("xyzs", "dirs", "deltas", "rays", "nears", "fars"))
        prefix = (rays.shape[0],) if prefix is None else prefix
        sigmas, rgbs = self.forward_scaled(xyzs, dirs, marched.get("counter"))
        loss, weights_sum, depth, image = raymarching.composite_loss_train(
            sigmas, rgbs, deltas, rays, gt_rgb, bg_color, nears if scale_depth else None, fars if scale_depth else None, T_thresh, grad_scale)
        return loss, {"image": image.view(*prefix, 3), "depth": depth.view(*prefix), "weights_sum": weights_sum, "nears": nears,
                      "num_points": xyzs.shape[0]}

    # ---- renderer.py:259-392 ---------------------------------------------------------------------------------
    def run_cuda(self, rays_o, rays_d, dt_gamma=0, bg_color=None, perturb=False, force_all_rays=False, max_steps=1024,
                 T_thresh=1e-4, scale_depth=True, edit_grid=None, **kwargs):
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        dens_grid = edit_grid if edit_grid is not None else self.density_bitfield
        n_rays = rays_o.shape[0]
        device = rays_o.device
        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, self.aabb_train if self.training else self.aabb_infer,
                                                     self.min_near)
        if bg_color is None:
            bg_color = 1
        results = {}
        if self.training:
            marched = self._march_train_from(rays_o, rays_d, nears, fars, dens_grid, perturb, force_all_rays, dt_gamma, max_steps)
            results = self.shade_train(marched, bg_color, T_thresh, prefix, scale_depth=not kwargs.get("distill", False))
            depth, image = results["depth"], results["image"]
        elif self.device_loop and self._device_loop_ok(rays_o):
            t = self._render_rounds_device(rays_o, rays_d, nears, fars, dens_grid, None, dt_gamma, perturb, max_steps, T_thresh)
            weights_sum, depth, image = t["weights_sum"], t["depth"], t["image"]
            image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
            if scale_depth:
                depth = torch.clamp(depth - nears, min=0) / (fars - nears)
            else:
                results["t"] = weights_sum
            image = image.view(*prefix, 3)
            depth = depth.view(*prefix)
            results["num_points"] = t["slots"]
            results["rounds"] = t["rounds"]
            results["schedule"] = t["schedule"]
        else:
            weights_sum = torch.zeros(n_rays, dtype=torch.float32, device=device)
            depth = torch.zeros(n_rays, dtype=torch.float32, device=device)
            image = torch.zeros(n_rays, 3, dtype=torch.float32, device=device)
            n_alive = n_rays
            rays_alive = torch.arange(n_alive, dtype=torch.int32, device=device)
            spare = torch.empty_like(rays_alive)
            count = torch.empty(1, dtype=torch.int32, device=device)
            rays_t = nears.clone()
            step = 0
            total_samples = 0
            while step < max_steps:
                if n_alive <= 0:
                    break
                n_step = max(min(n_rays // n_alive, 8), 1)
                xyzs, dirs, deltas = raymarching.march_rays(n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, self.bound,
                                                            dens_grid, self.cascade, self.grid_size, nears, fars, 128,
                                                            perturb if step == 0 else False, dt_gamma, max_steps)
                sigmas, rgbs = self.forward_scaled(xyzs, dirs)
                raymarching.composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image,
                                           T_thresh)
                total_samples += xyzs.shape[0]
                # rays_alive = rays_alive[rays_alive >= 0] (renderer.py:375), compacted on the device
                raymarching.compact_alive(rays_alive, n_alive, spare, count)
                rays_alive, spare = spare, rays_alive
                n_alive = int(count.item())
                step += n_step
            image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
            if scale_depth:
                depth = torch.clamp(depth - nears, min=0) / (fars - nears)
            else:
                results["t"] = weights_sum
            image = image.view(*prefix, 3)
            depth = depth.view(*prefix)
            results["num_points"] = total_samples
        results["depth"] = depth
        results["image"] = image
        return results

    # ---- renderer.py:394-480 (edit-grid distillation render used to build LAENeRF's EditDataset) --------------
    @torch.no_grad()
    def run_cuda_distill(self, rays_o, rays_d, edit_bitfield, dt_gamma=0, bg_color=None, perturb=False, force_all_rays=False,
                         max_steps=1024, T_thresh=1e-4, perturb_depth=False, grow_grid=False, **kwargs):
        """Same result dict as the reference (renderer.py:466-480): the UN-blended composite `image`, `depth`, `depth_edit`,
        `x_term = rays_o + depth * rays_d`, `weights_edit`, `weights`, `min_near` (+ `weights_sum` / `weights_edit_sum` aliases)."""
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        n_rays = rays_o.shape[0]
        device = rays_o.device
        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, self.aabb_train if self.training else self.aabb_infer, self.min_near)
        dens_bitfield = edit_bitfield if grow_grid else self.density_bitfield  # renderer.py:410-413

        def finish(weights_sum, weights_edit_sum, depth, depth_edit, image):
            if perturb_depth:  # renderer.py:463-464
                depth = depth + (torch.rand(depth.shape, device=device) - 0.5) * (depth.max() - depth.min()) / max_steps
            return {"depth": depth.view(*prefix), "depth_edit": depth_edit, "image": image.view(*prefix, 3),
                    "x_term": rays_o + depth[..., None] * rays_d, "weights_edit": weights_edit_sum, "weights": weights_sum,
                    "min_near": nears.min(), "weights_sum": weights_sum, "weights_edit_sum": weights_edit_sum}

        if self.device_loop and self._device_loop_ok(rays_o):
            t = self._render_rounds_device(rays_o, rays_d, nears, fars, dens_bitfield, edit_bitfield, dt_gamma, perturb, max_steps, T_thresh)
            return finish(t["weights_sum"], t["wes"], t["depth"], t["de"], t["image"])
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=device)
        weights_sum, weights_edit_sum, depth, depth_edit, image = z(n_rays), z(n_rays), z(n_rays), z(n_rays), z(n_rays, 3)
        n_alive = n_rays
        rays_alive = torch.arange(n_alive, dtype=torch.int32, device=device)
        spare = torch.empty_like(rays_alive)
        count = torch.empty(1, dtype=torch.int32, device=device)
        rays_t = nears.clone()
        step = 0
        while step < max_steps and n_alive > 0:
            n_step = max(min(n_rays // n_alive, 8), 1)
            xyzs, dirs, deltas, edit_occ = raymarching.march_rays_distill(
                n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, self.bound, dens_bitfield, edit_bitfield, self.cascade,
                self.grid_size, nears, fars, 128, perturb if step == 0 else False, dt_gamma, max_steps)
            sigmas, rgbs = self.forward_scaled(xyzs, dirs)
            raymarching.composite_rays_distill(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum,
                                               weights_edit_sum, depth, depth_edit, image, edit_occ, T_thresh)
            raymarching.compact_alive(rays_alive, n_alive, spare, count)
            rays_alive, spare = spare, rays_alive
            n_alive = int(count.item())
            step += n_step
        return finish(weights_sum, weights_edit_sum, depth, depth_edit, image)

    def render(self, rays_o, rays_d, **kwargs):
        return self.run_cuda(rays_o, rays_d, **kwargs)

    def get_params(self, lr):  # network_ff.py:139-153
        return [{"params": self.encoder.parameters(), "lr": lr}, {"params": self.sigma_net.parameters(), "lr": lr},
                {"params": self.encoder_dir.parameters(), "lr": lr}, {"params": self.color_net.parameters(), "lr": lr}]


class TrainStep:
    """One NeRF training step as `Trainer.train_one_epoch` runs it under `-O` (nerf/utils.py:1474-1484):
    fp16 autocast forward, MSE on RGB, GradScaler backward, Adam(lr 1e-2, betas (0.9, 0.99), eps 1e-15)."""

    def __init__(self, model: NeRFNetwork, lr: float = 1e-2, fp16: bool = True, world_size: int = 1, fused_optimizer: bool = True,
                 fused_loss: bool = True):
        self.model = model
        self.fp16 = fp16
        self.world_size = world_size
        self.fused_loss = bool(fused_loss)
        self.fused_tail = os.environ.get("LNRF_FUSED_TAIL", "1") == "1"  # forward + backward of the compositing tail in one launch
        self.fused_optimizer = bool(fused_optimizer) and fp16 and model.fused and model._fused_ok
        if self.fused_optimizer:
            # row f-4: inf check + unscale + Adam + fp16 shadow rewrite + gradient clear in two launches (optim.py)
            from .optim import AmpAdam
            rank = 0
            if world_size > 1:
                import torch.distributed as dist
                rank = dist.get_rank()
            # world_size > 1: reduce-scatter + per-rank Adam on a 1/N table slice + all-gather of the fp16 shadow (optim.py)
            self.optimizer = AmpAdam(model, lr=lr, betas=(0.9, 0.99), eps=1e-15, fp16=True, world_size=world_size, rank=rank)
            self.scaler = None
        else:
            # torch path.  fused=True: one multi-tensor kernel that also consumes GradScaler's scale / found_inf on the
            # device, so the step has no host synchronisation and can be captured into a CUDA graph (GraphedTrainStep)
            self.optimizer = torch.optim.Adam(model.get_params(lr), betas=(0.9, 0.99), eps=1e-15, fused=True, capturable=True)
            self.scaler = torch.amp.GradScaler("cuda", enabled=fp16)

    def __call__(self, rays_o, rays_d, gt_rgb, bg_color=1, perturb=True):
        return self.train_on(self.march(rays_o, rays_d, perturb), gt_rgb, bg_color)

    def march(self, rays_o, rays_d, perturb=True, into=None):
        """The parameter-independent half of the step (near/far + occupancy march); see NeRFNetwork.march_train."""
        self.model.train()
        return self.model.march_train(rays_o, rays_d, perturb=perturb, force_all_rays=False, dt_gamma=0, max_steps=1024, into=into)

    def train_on(self, marched, gt_rgb, bg_color=1):
        loss, out = self.forward_backward(marched, gt_rgb, bg_color)
        self.reduce_and_step()
        return loss, out

    def forward_backward(self, marched, gt_rgb, bg_color=1):
        """Network + compositing + loss + backward of one marched batch: gradients are left in the optimizer's buffers."""
        self.model.train()
        self.optimizer.zero_grad(set_to_none=True)
        if self.fused_loss and self.fused_optimizer:
            # row f-5: composite + blend + MSE in one launch; the AMP scale enters the backward as a device scalar, so
            # `scale(loss).backward()` costs no launch of its own
            scale = self.optimizer._scale.view(())
            with torch.autocast(device_type="cuda", dtype=torch.float16, enabled=self.fp16):
                loss, out = self.model.shade_loss_train(marched, gt_rgb, bg_color, grad_scale=scale if self.fused_tail else None)
            torch.autograd.backward(loss, grad_tensors=scale)
            return loss, out
        with torch.autocast(device_type="cuda", dtype=torch.float16, enabled=self.fp16):
            out = self.model.shade_train(marched, bg_color)
            loss = torch.nn.functional.mse_loss(out["image"], gt_rgb, reduction="none").mean(-1).mean()
        (self.optimizer if self.fused_optimizer else self.scaler).scale(loss).backward()
        return loss, out

    def reduce_and_step(self):
        """The exchange step of ray-sharded training (SURVEY.md 8e) followed by the identical Adam step on every rank."""
        if self.fused_optimizer:
            self.optimizer.step()  # includes the exchange when world_size > 1 (AmpAdam._exchange_gradients)
            return
        if self.world_size > 1:
            from .parallel import allreduce_gradients
            allreduce_gradients([p for g in self.optimizer.param_groups for p in g["params"]], self.world_size)
        self.scaler.step(self.optimizer)
        self.scaler.update()


def _check_mode(captured: bool, who: str) -> None:
    """A graph replays the kernels of the mode it was captured in: never the other one silently."""
    if captured != torch.are_deterministic_algorithms_enabled():
        raise RuntimeError(f"{who}: captured with torch.are_deterministic_algorithms_enabled() == {captured}, but the flag is now "
                           f"{not captured}; call capture() again (needs_recapture() reports the change)")


class GraphedTrainStep:
    """The same training step replayed from ONE CUDA graph (march -> encode -> MLPs -> composite -> loss -> backward
    -> Adam): the 4096-ray step is launch-bound when issued from Python (SURVEY.md section 7, "hard parts"), so the
    steady state is captured once per sample-buffer size and replayed.  Inputs are copied into static device buffers;
    `loss` / `out` are views of graph-owned memory that the next replay overwrites.

    lookahead=True software-pipelines consecutive steps: near/far + the occupancy march depend only on the rays and the
    occupancy bitfield, never on the parameters, and the march is latency-bound (a few warps per SM busy walking the grid),
    while the hash-grid backward is bound by the L2 atomic units with its warps waiting.  So the graph marches the batch handed
    to call k on a second stream BESIDE the backward (MLP backward onwards) of the batch handed to call k-1.  Two
    sample-buffer sets and two graphs alternate (train on set p, march into set 1-p): nothing is copied between steps.
    Forking earlier -- beside the persistent MLP kernels, which need a whole SM's shared memory and registers -- or only
    beside Adam measured slower than no overlap.  Every call still consumes one batch and performs one full optimizer step;
    the returned loss is that of the previous call's batch (one-step delay, `flush()` trains the last one).  After an
    occupancy update call `remarch()`: the batch in flight was marched through the old bitfield."""

    def __init__(self, step: TrainStep, n_rays: int, bg_color=1, perturb=True, lookahead: bool = False):
        self.step, self.model = step, step.model
        dev = next(self.model.parameters()).device
        self.ro = torch.zeros(n_rays, 3, device=dev)
        self.rd = torch.zeros(n_rays, 3, device=dev)
        self.gt = torch.zeros(n_rays, 3, device=dev)
        self.bg_color, self.perturb, self.lookahead = bg_color, perturb, bool(lookahead)
        self.graph = None
        self.captured_mean_count = 0
        self.loss = self.out = None
        self._pipe_opt = False
        self.sets = self.graphs = None  # lookahead: the two marched-batch buffer sets (with their targets) and the two graphs
        self.phase = 0                  # lookahead: the set the next replay trains on
        self.deterministic = None       # torch.are_deterministic_algorithms_enabled() at capture: the graph holds that mode's kernels

    def _load(self, rays_o, rays_d, gt_rgb):
        self.ro.copy_(rays_o, non_blocking=True)
        self.rd.copy_(rays_d, non_blocking=True)
        self.gt.copy_(gt_rgb, non_blocking=True)

    def _capture_pipelined(self, p):
        """Graph p: train on set p; beside its backward (from the MLP backward on), march the loaded batch into set 1-p."""
        from . import gridencoder as _ge
        cur, nxt = self.sets[p], self.sets[1 - p]
        if self._pipe_opt:  # ray-sharded: graph p accumulates into gradient buffer p and clears buffer 1 - p inside its exchange kernel
            self.step.optimizer.select_phase(p)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            main = torch.cuda.current_stream()

            def fork():  # runs on the autograd thread, right before the encoder backward is queued
                self._side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(self._side):
                    self.step.march(self.ro, self.rd, self.perturb, into=nxt)
                    nxt["gt"].copy_(self.gt)

            # where the side stream forks (A/B switch; measured on one B200, ms/step: none 0.405 | start 0.401 | adam 0.409 |
            # enc_bwd 0.380 | nerf_bwd 0.375): the march cannot share an SM with the persistent MLP kernels (registers, shared memory),
            # so forked at nerf_bwd it starts on each SM the moment that kernel's CTA retires -- ahead of the hash-grid backward
            at = os.environ.get("LNRF_LOOKAHEAD_AT", "nerf_bwd")
            import laenerf_b200.nerf as _me
            if at == "start":
                fork()
            elif at == "nerf_bwd":
                _me.before_network_backward = fork
            elif at == "enc_bwd":
                _ge.before_backward = fork
            try:
                loss, out = self.step.forward_backward(cur, cur["gt"], self.bg_color)
            finally:
                _ge.before_backward = None
                _me.before_network_backward = None
            if at == "adam":
                fork()
            self.step.reduce_and_step()
            main.wait_stream(self._side)
        if self._pipe_opt:
            self.step.optimizer.select_phase(None)
        return g, loss, out

    def capture(self, rays_o, rays_d, gt_rgb, warmup: int = 3):
        """Warm up, then capture the step (lookahead: both graphs; the given batch becomes the batch in flight).  A RE-capture with
        lookahead discards the batch that was in flight: call flush() first if it must be trained on."""
        m = self.model
        self._load(rays_o, rays_d, gt_rgb)
        if m.mean_count <= 0:  # the first (eager) steps size the sample buffer, as in the reference
            self.step(self.ro, self.rd, self.gt, self.bg_color, self.perturb)
            m.update_mean_count()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.step(self.ro, self.rd, self.gt, self.bg_color, self.perturb)
        torch.cuda.current_stream().wait_stream(side)
        m.local_step = 0  # the captured march always counts into step_counter[0]; rotated after each replay
        opt = self.step.optimizer
        self._pipe_opt = bool(self.lookahead and self.step.fused_optimizer and getattr(opt, "can_pipeline", False) and
                              os.environ.get("LNRF_PIPELINED_EXCHANGE", "1") == "1")
        if self._pipe_opt:
            opt._settle_buffers()  # a re-capture starts from two clean gradient buffers
        if self.lookahead:
            # prime the pipeline: march the capture batch eagerly into set 0; set 1 is a same-shape twin
            first = self.step.march(self.ro, self.rd, self.perturb)
            m.local_step = 0
            self.sets = [{k: v.clone() for k, v in first.items()} for _ in range(2)]
            for s_ in self.sets:
                s_["gt"] = self.gt.clone()
            self._side = torch.cuda.Stream(priority=int(os.environ.get("LNRF_LOOKAHEAD_PRIO", "0")))
            self.graphs, self._results = [], []
            for p in range(2):
                g, loss, out = self._capture_pipelined(p)
                self.graphs.append(g)
                self._results.append((loss, out))
            self.graph, self.phase = self.graphs[0], 0
            # the captures ran no kernels: set 0 still holds the capture batch, marched eagerly above
        else:
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.loss, self.out = self.step(self.ro, self.rd, self.gt, self.bg_color, self.perturb)
        self.captured_mean_count = m.mean_count
        self.deterministic = torch.are_deterministic_algorithms_enabled()
        m.local_step = 0
        self._replays = 0

    def needs_recapture(self) -> bool:
        """After update_mean_count(): re-capture when the running mean outgrew the captured buffer or shrank by > 1/8, or when
        torch.use_deterministic_algorithms was switched since the capture."""
        mc, cap = self.model.mean_count, self.captured_mean_count
        return (self.graph is None or mc > cap or mc < cap - cap // 8 or
                self.deterministic != torch.are_deterministic_algorithms_enabled())

    def __call__(self, rays_o, rays_d, gt_rgb):
        if self.graph is None:
            self.capture(rays_o, rays_d, gt_rgb)
            if self.lookahead:  # the capture batch is in flight; its loss arrives with the next call
                return None, None
        _check_mode(self.deterministic, "GraphedTrainStep")
        self._load(rays_o, rays_d, gt_rgb)
        m = self.model
        if m.render_clip_far:
            m.occupied_box()  # the captured marcher reads the box from a persistent buffer: refresh it if the bitfield changed
        row = self._replays % 16
        if self.lookahead:
            p = self.phase
            self.graphs[p].replay()
            self.loss, self.out = self._results[p]
            self.phase = 1 - p
            if self._pipe_opt:
                self.step.optimizer._dirty_buf = p  # what the replay left for its successor (or an eager step) to clear
            # keep the 16-entry counter history the occupancy update averages (renderer.py:643-647)
            m.step_counter[row].copy_(self.sets[1 - p]["counter"], non_blocking=True)
        else:
            self.graph.replay()
            if row:
                m.step_counter[row].copy_(m.step_counter[0], non_blocking=True)
        self._replays += 1
        m.local_step = min(16, self._replays)
        return self.loss, self.out

    def remarch(self):
        """lookahead, after an occupancy update: march the batch in flight again (eagerly) through the new bitfield, as the
        un-pipelined loop would have."""
        if self.lookahead and self.sets is not None:
            keep = self.model.local_step
            self.step.march(self.ro, self.rd, self.perturb, into=self.sets[self.phase])
            self.model.local_step = keep

    def flush(self):
        """lookahead: train on the batch that is still in flight (eagerly); returns its (loss, out)."""
        if not self.lookahead or self.sets is None:
            return None, None
        cur = self.sets[self.phase]
        return self.step.train_on(cur, cur["gt"], self.bg_color)  # eager, one gradient buffer: settles what the last replay left
