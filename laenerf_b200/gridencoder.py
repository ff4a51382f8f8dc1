"""Drop-in for the reference's `gridencoder` package (gridencoder/grid.py:24-185) on liblaenerf_b200.so.

Same module/function names, constructor arguments, parameter names and shapes (`embeddings [sum(entries), C]`
fp32, `offsets [L+1]` int32 buffer -> checkpoints interchange), same AMP behaviour (fp16 table copy under autocast
when C is even).  The kernel writes the `[B, L*C]` layout the API returns directly and reads gradients in that
layout, so the reference's two permute copies (grid.py:57, 75) do not exist here.
"""
from __future__ import annotations

import weakref

import numpy as np
import torch
import torch.nn as nn
from torch.autograd import Function
from torch.amp import custom_bwd, custom_fwd

from . import _native as N
from ._shadow import shadow_f16

_gridtype_to_id = {"hash": 0, "tiled": 1}
_interp_to_id = {"linear": 0, "smoothstep": 1}

_host_offsets = {}  # id(device offsets tensor) -> (weakref to it, its _version, int32 host copy)


def _offsets_host(offsets: torch.Tensor) -> torch.Tensor:
    """The C ABI takes the L+1 level offsets from the host (they are launch geometry, not data).  The cache entry is tied
    to the tensor OBJECT (weak reference): a freed tensor whose address is reused by another model must not hit it."""
    if not offsets.is_cuda:
        return offsets.contiguous().to(torch.int32)
    key = id(offsets)
    hit = _host_offsets.get(key)
    if hit is not None and hit[0]() is offsets and hit[1] == offsets._version:
        return hit[2]
    h = offsets.detach().to("cpu", torch.int32).contiguous()
    if len(_host_offsets) > 64:  # drop entries whose tensor is gone
        for k in [k for k, v in _host_offsets.items() if v[0]() is None]:
            del _host_offsets[k]
    _host_offsets[key] = (weakref.ref(offsets), offsets._version, h)
    return h


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.float16:
        return N.F16
    if t.dtype == torch.float32:
        return N.F32
    raise RuntimeError(f"GridEncoder: unsupported embedding dtype {t.dtype} (float32 or float16)")


class _grid_encode(Function):
    @staticmethod
    @custom_fwd(device_type="cuda")
    def forward(ctx, inputs, embeddings, offsets, per_level_scale, base_resolution, calc_grad_inputs=False, gridtype=0,
                align_corners=False, interpolation=0, shadow_f16=None, grad_f16=None, world_bound=0.0, b_dev=None, grad_f32=None):
        # b_dev: optional device int32 with the number of live rows (world_bound > 0 only): whole 128-row tiles past it are neither
        # encoded nor differentiated -- their output rows stay unwritten, which is fine for a consumer that honours the same count
        # world_bound > 0: `inputs` are world coordinates and the kernel applies GridEncoder.forward's (x + bound) / (2 * bound)
        # itself (hot shape only: D = 3, C = 2, no input gradients) -- two elementwise passes over [B, 3] less per call
        inputs = inputs.contiguous().float()
        B, D = inputs.shape
        L = offsets.shape[0] - 1
        C = embeddings.shape[1]
        S = float(np.log2(per_level_scale))
        H = int(base_resolution)
        ctx.grad_buf = None
        if torch.is_autocast_enabled() and C % 2 == 0:  # grid.py:43-44
            if shadow_f16 is not None:  # laenerf_b200.optim.AmpAdam keeps embeddings.half() up to date: no cast pass
                embeddings = shadow_f16
                ctx.grad_buf = grad_f16
            else:
                embeddings = embeddings.to(torch.half)
        elif grad_f32 is not None and embeddings.dtype == torch.float32:
            ctx.grad_buf = grad_f32  # the fp32 table read directly (no autocast) with a persistent fp32 gradient buffer
        embeddings = embeddings.contiguous()
        off_h = _offsets_host(offsets)
        outputs = torch.empty(B, L * C, device=inputs.device, dtype=embeddings.dtype)
        dy_dx = torch.empty(B, L * D * C, device=inputs.device, dtype=embeddings.dtype) if calc_grad_inputs else None
        if b_dev is not None and not world_bound > 0:
            raise RuntimeError("GridEncoder: a device-side row count needs the world-coordinate kernel (D = 3, C = 2, no input gradients)")
        if world_bound > 0:
            N.check(N.lib().lnrf_grid_encode_forward_world(N.ptr(inputs), float(world_bound), N.ptr(embeddings), N.ptr(off_h), N.ptr(outputs),
                                                           B, N.ptr(b_dev), L, S, H, int(gridtype), int(bool(align_corners)), int(interpolation),
                                                           _dt(embeddings), N.stream()))
        else:
            N.check(N.lib().lnrf_grid_encode_forward(N.ptr(inputs), N.ptr(embeddings), N.ptr(off_h), N.ptr(outputs), B, D, C, L, S, H,
                                                     N.ptr(dy_dx), int(gridtype), int(bool(align_corners)), int(interpolation),
                                                     _dt(embeddings), N.GRID_BLC, N.stream()))
        ctx.save_for_backward(inputs, embeddings, offsets, dy_dx, b_dev)
        ctx.dims = [B, D, C, L, S, H, gridtype, interpolation]
        ctx.world_bound = float(world_bound)
        ctx.align_corners = align_corners
        return outputs

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, grad):
        if before_backward is not None:  # GraphedTrainStep(lookahead="bwd"): fork the next batch's march beside this kernel
            before_backward()
        inputs, embeddings, offsets, dy_dx, b_dev = ctx.saved_tensors
        B, D, C, L, S, H, gridtype, interpolation = ctx.dims
        grad = grad.contiguous().to(embeddings.dtype)
        # with AmpAdam the gradient accumulates straight into its persistent fp16 buffer (cleared by the optimizer kernel); with
        # ShardedFlatAdam into this rank's fp32 gradient vector, which the other ranks read over NVLink
        grad_embeddings = ctx.grad_buf if ctx.grad_buf is not None else torch.zeros_like(embeddings)
        grad_inputs = torch.zeros_like(inputs, dtype=embeddings.dtype) if dy_dx is not None else None
        if ctx.world_bound > 0:
            N.check(N.lib().lnrf_grid_encode_backward_world(N.ptr(grad), N.ptr(inputs), ctx.world_bound, N.ptr(_offsets_host(offsets)),
                                                            N.ptr(grad_embeddings), B, N.ptr(b_dev), L, S, H, int(gridtype),
                                                            int(bool(ctx.align_corners)), int(interpolation), _dt(embeddings), N.stream()))
        else:
            N.check(N.lib().lnrf_grid_encode_backward(N.ptr(grad), N.ptr(inputs), N.ptr(embeddings), N.ptr(_offsets_host(offsets)),
                                                      N.ptr(grad_embeddings), B, D, C, L, S, H, N.ptr(dy_dx), N.ptr(grad_inputs),
                                                      int(gridtype), int(bool(ctx.align_corners)), int(interpolation),
                                                      _dt(embeddings), N.GRID_BLC, N.stream()))
        if dy_dx is not None:
            grad_inputs = grad_inputs.to(inputs.dtype)
        if ctx.grad_buf is not None:
            grad_embeddings = None
        return grad_inputs, grad_embeddings, None, None, None, None, None, None, None, None, None, None, None, None


grid_encode = _grid_encode.apply
before_backward = None


class GridEncoder(nn.Module):
    def __init__(self, input_dim=3, num_levels=16, level_dim=2, per_level_scale=2, base_resolution=16, log2_hashmap_size=19,
                 desired_resolution=None, gridtype="hash", align_corners=False, interpolation="linear"):
        super().__init__()
        if desired_resolution is not None:  # grid.py:101-102
            per_level_scale = np.exp2(np.log2(desired_resolution / base_resolution) / (num_levels - 1))
        self.input_dim = input_dim
        self.num_levels = num_levels
        self.level_dim = level_dim
        self.per_level_scale = per_level_scale
        self.log2_hashmap_size = log2_hashmap_size
        self.base_resolution = base_resolution
        self.output_dim = num_levels * level_dim
        self.gridtype = gridtype
        self.gridtype_id = _gridtype_to_id[gridtype]
        self.interpolation = interpolation
        self.interp_id = _interp_to_id[interpolation]
        self.align_corners = align_corners

        offsets, offset = [], 0
        self.max_params = 2 ** log2_hashmap_size
        for i in range(num_levels):  # grid.py:121-126
            resolution = int(np.ceil(base_resolution * per_level_scale ** i))
            params_in_level = min(self.max_params, (resolution if align_corners else resolution + 1) ** input_dim)
            params_in_level = int(np.ceil(params_in_level / 8) * 8)
            offsets.append(offset)
            offset += params_in_level
        offsets.append(offset)
        self.register_buffer("offsets", torch.from_numpy(np.array(offsets, dtype=np.int32)))
        self.n_params = offsets[-1] * level_dim
        self.embeddings = nn.Parameter(torch.empty(offset, level_dim))
        self.reset_parameters()
        # set by laenerf_b200.optim.AmpAdam: fp16 shadow of the table + persistent fp16 gradient (row f-4)
        self._shadow_f16 = None
        self._grad_f16 = None
        # set by laenerf_b200.optim.ShardedFlatAdam: persistent fp32 gradient of the fp32 table, used when no autocast casts it
        self._grad_f32 = None

    def reset_parameters(self):
        std = 1e-4
        self.embeddings.data.uniform_(-std, std)

    def __repr__(self):
        return (f"GridEncoder: input_dim={self.input_dim} num_levels={self.num_levels} level_dim={self.level_dim} "
                f"resolution={self.base_resolution} -> {int(round(self.base_resolution * self.per_level_scale ** (self.num_levels - 1)))} "
                f"per_level_scale={self.per_level_scale:.4f} params={tuple(self.embeddings.shape)} gridtype={self.gridtype} "
                f"align_corners={self.align_corners} interpolation={self.interpolation}")

    def forward(self, inputs, bound=1, b_dev=None):
        # hot shape on the GPU: the kernel maps to [0, 1] itself (same IEEE add + divide as the line below)
        in_kernel = (inputs.is_cuda and self.input_dim == 3 and self.level_dim == 2 and not inputs.requires_grad and
                     inputs.dtype == torch.float32 and bound > 0)
        if not in_kernel:
            b_dev = None
        if not in_kernel:
            inputs = (inputs + bound) / (2 * bound)  # map to [0, 1]
        prefix_shape = list(inputs.shape[:-1])
        inputs = inputs.view(-1, self.input_dim)
        outputs = grid_encode(inputs, self.embeddings, self.offsets, self.per_level_scale, self.base_resolution,
                              inputs.requires_grad, self.gridtype_id, self.align_corners, self.interp_id,
                              shadow_f16(self, self.embeddings), self._grad_f16, float(bound) if in_kernel else 0.0, b_dev,
                              self._grad_f32)
        return outputs.view(prefix_shape + [self.output_dim])

    @torch.autocast(device_type="cuda", enabled=False)
    def grad_total_variation(self, weight=1e-7, inputs=None, bound=1, B=1000000):
        D, C, L = self.input_dim, self.embeddings.shape[1], self.offsets.shape[0] - 1
        S, H = float(np.log2(self.per_level_scale)), self.base_resolution
        if inputs is None:
            inputs = torch.rand(B, self.input_dim, device=self.embeddings.device)
        else:
            inputs = ((inputs + bound) / (2 * bound)).view(-1, self.input_dim)
            B = inputs.shape[0]
        if self.embeddings.grad is None:
            raise ValueError("grad is None, should be called after loss.backward() and before optimizer.step()!")
        inputs = inputs.contiguous().to(self.embeddings.dtype)
        N.check(N.lib().lnrf_grad_total_variation(N.ptr(inputs), N.ptr(self.embeddings), N.ptr(self.embeddings.grad),
                                                  N.ptr(_offsets_host(self.offsets)), float(weight), B, D, C, L, S, H,
                                                  self.gridtype_id, int(bool(self.align_corners)), _dt(self.embeddings), N.stream()))
