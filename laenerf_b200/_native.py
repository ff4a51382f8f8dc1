"""ctypes loader for liblaenerf_b200.so -- the C-ABI boundary of the package (include/laenerf_b200.h).

PyTorch only supplies device memory and streams: every call passes raw `data_ptr()` addresses, sizes and the
current CUDA stream.  There is NO fallback: if the shared library is missing, or a call fails, a RuntimeError is
raised (the reference raises RuntimeError through TORCH_CHECK / std::runtime_error, SURVEY.md section 8b).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "liblaenerf_b200.so")
_lib = None

vp, u32, i32, f32, f64, sz, u64 = C.c_void_p, C.c_uint32, C.c_int, C.c_float, C.c_double, C.c_size_t, C.c_uint64


class OptTensor(C.Structure):
    """lnrf_opt_tensor (include/laenerf_b200.h): one parameter tensor of the fused Adam / AMP step."""
    _fields_ = [("params", vp), ("exp_avg", vp), ("exp_avg_sq", vp), ("grad", vp), ("params_f16", vp), ("n", u64),
                ("grad_dtype", i32)]


# name -> (restype, argtypes); must list every symbol include/laenerf_b200.h declares (tests/test_abi.py checks)
SIGNATURES = {
    "lnrf_last_error": (C.c_char_p, []),
    "lnrf_version": (i32, []),
    "lnrf_compiled_arch": (i32, []),
    "lnrf_launch_count": (u64, []),
    "lnrf_sizeof_render_desc": (sz, []),
    "lnrf_sizeof_opt_tensor": (sz, []),
    "lnrf_near_far_from_aabb": (i32, [vp, vp, vp, u32, f32, vp, vp, vp]),
    "lnrf_sph_from_ray": (i32, [vp, vp, f32, u32, vp, vp]),
    "lnrf_morton3D": (i32, [vp, u32, vp, vp]),
    "lnrf_morton3D_invert": (i32, [vp, u32, vp, vp]),
    "lnrf_packbits": (i32, [vp, u32, f32, vp, vp]),
    "lnrf_march_rays_train_scratch_bytes": (sz, [u32]),
    "lnrf_march_rays_train": (i32, [vp, vp, vp, f32, f32, u32, u32, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "lnrf_march_rays_train_clipped": (i32, [vp, vp, vp, f32, f32, u32, u32, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
    "lnrf_composite_rays_train_forward": (i32, [vp, vp, vp, vp, u32, u32, f32, vp, vp, vp, vp]),
    "lnrf_composite_rays_train_backward": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, u32, u32, f32, vp, vp, i32, vp]),
    "lnrf_composite_loss_scratch_bytes": (sz, [u32]),
    "lnrf_composite_loss_train_forward": (i32, [vp, vp, vp, vp, vp, vp, f32, vp, vp, u32, u32, f32, vp, vp, vp, vp, vp, vp, sz, vp]),
    "lnrf_composite_loss_train_backward": (i32, [vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, vp, u32, u32, f32, vp, vp, vp]),
    "lnrf_composite_loss_train_forward_backward": (i32, [vp, vp, vp, vp, vp, vp, vp, f32, vp, vp, u32, u32, f32, vp, vp, vp, vp, vp, vp, vp,
                                                         vp, sz, vp]),
    "lnrf_march_rays": (i32, [u32, u32, vp, vp, vp, vp, f32, f32, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp, u32, vp]),
    "lnrf_march_rays_distill": (i32, [u32, u32, vp, vp, vp, vp, f32, f32, u32, u32, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp, u32, vp]),
    "lnrf_composite_rays": (i32, [u32, u32, f32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "lnrf_composite_rays_distill": (i32, [u32, u32, f32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "lnrf_march_rays_prescribed": (i32, [u32, vp, vp, vp, vp, f32, f32, u32, u32, u32, vp, vp, vp, u32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "lnrf_composite_rays_prescribed": (i32, [u32, f32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "lnrf_compact_alive_scratch_bytes": (sz, [u32]),
    "lnrf_compact_alive": (i32, [vp, u32, vp, vp, vp, sz, vp]),
    "lnrf_grid_encode_forward": (i32, [vp, vp, vp, vp, u32, u32, u32, u32, f32, u32, vp, u32, i32, u32, i32, i32, vp]),
    "lnrf_grid_encode_backward": (i32, [vp, vp, vp, vp, vp, u32, u32, u32, u32, f32, u32, vp, vp, u32, i32, u32, i32, i32, vp]),
    "lnrf_grad_total_variation": (i32, [vp, vp, vp, vp, f32, u32, u32, u32, u32, f32, u32, u32, i32, i32, vp]),
    "lnrf_grid_level_scales": (i32, [u32, f32, u32, vp, vp]),
    "lnrf_ffmlp_forward": (i32, [vp, vp, u32, u32, u32, u32, u32, u32, u32, vp, vp, vp]),
    "lnrf_ffmlp_inference": (i32, [vp, vp, u32, u32, u32, u32, u32, u32, u32, vp, vp, vp]),
    "lnrf_ffmlp_wgrad_scratch_bytes": (sz, [u32, u32, u32, u32]),
    "lnrf_ffmlp_backward": (i32, [vp, vp, vp, vp, u32, u32, u32, u32, u32, u32, u32, i32, vp, vp, vp, vp, sz, vp]),
    "lnrf_allocate_splitk": (i32, [sz]),
    "lnrf_free_splitk": (i32, []),
    "lnrf_sh_encode_forward": (i32, [vp, vp, u32, u32, vp, i32, vp]),
    "lnrf_sh_encode_backward": (i32, [vp, u32, u32, vp, vp, vp]),
    "lnrf_grid_encode_forward_world": (i32, [vp, f32, vp, vp, vp, u32, vp, u32, f32, u32, u32, i32, u32, i32, vp]),
    "lnrf_grid_encode_backward_world": (i32, [vp, vp, f32, vp, vp, u32, vp, u32, f32, u32, u32, i32, u32, i32, vp]),
    "lnrf_render_scratch_bytes": (sz, [u32]),
    "lnrf_render_begin": (i32, [vp, vp]),
    "lnrf_render_rounds": (i32, [vp, u32, u32, vp]),
    "lnrf_occupancy_points": (i32, [vp, vp, u32, u32, f32, vp, vp, vp]),
    "lnrf_occupancy_scatter": (i32, [vp, vp, u32, vp, vp]),
    "lnrf_occupancy_fill": (i32, [vp, u32, f32, vp]),
    "lnrf_occupancy_scratch_bytes": (sz, []),
    "lnrf_occupancy_ema": (i32, [vp, vp, u32, f32, f32, vp, vp, sz, vp]),
    "lnrf_packbits_dev": (i32, [vp, u32, vp, vp, vp]),
    "lnrf_occupied_box_work_ints": (sz, [u32]),
    "lnrf_occupied_box": (i32, [vp, u32, u32, f32, vp, vp, vp]),
    "lnrf_nerf_density": (i32, [vp, vp, u32, u32, f32, vp, vp]),
    "lnrf_nerf_forward": (i32, [vp, vp, vp, vp, u32, u32, u32, f32, i32, vp, vp, vp, vp, vp, vp]),
    "lnrf_nerf_wgrad_scratch_bytes": (sz, [u32, u32]),
    "lnrf_nerf_backward": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, u32, u32, u32, f32, vp, vp, vp, i32, vp, vp, sz, vp]),
    "lnrf_nerf_forward_lean": (i32, [vp, vp, vp, vp, u32, vp, u32, u32, f32, vp, vp, vp, vp]),
    "lnrf_nerf_backward_recompute_supported": (i32, [u32, u32]),
    "lnrf_nerf_backward_recompute": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, u32, vp, u32, u32, f32, vp, vp, vp, i32, vp, sz, vp]),
    "lnrf_nerf_wgrad_reduce": (i32, [vp, sz, u32, u32, u32, vp, vp, i32, vp]),
    "lnrf_grad_nonfinite_check": (i32, [vp, u32, vp, vp]),
    "lnrf_adam_step": (i32, [vp, u32, f64, f64, f64, f64, f64, vp, vp, vp, vp, vp]),
    "lnrf_adam_step_sharded": (i32, [vp, vp, vp, u32, u64, u64, vp, vp, vp, f64, f64, f64, f64, f64, vp, vp, vp, vp, vp]),
    "lnrf_adam_step_sharded_f32": (i32, [vp, vp, vp, u32, u32, u64, u64, vp, vp, u32, vp, vp, f64, f64, f64, f64, f64, vp, vp, vp, vp, vp]),
    "lnrf_adam_step_sharded_pipelined": (i32, [vp, vp, vp, u32, u64, u64, vp, vp, vp, f64, f64, f64, f64, f64, vp, vp, vp, u64, vp, vp, vp, vp, vp,
                                               f32, f32, i32, vp]),
    "lnrf_grad_nonfinite_check_snapshot": (i32, [vp, u32, vp, vp, vp, vp, vp]),
    "lnrf_adam_step_sharded_sync": (i32, [vp, vp, vp, u32, u32, u64, u64, vp, vp, vp, f64, f64, f64, f64, f64, vp, vp, vp, vp, vp, vp]),
    "lnrf_exchange_finish": (i32, [vp, u32, vp, vp, u64, vp]),
    "lnrf_adam_amp_step": (i32, [vp, u32, f64, f64, f64, f64, f64, vp, vp, vp, vp, vp, f32, f32, i32, vp, vp]),
    "lnrf_exchange_tail": (i32, [vp, u64, vp, vp, vp, vp, f32, f32, i32, vp]),
    "lnrf_amp_update": (i32, [vp, vp, vp, vp, f32, f32, i32, vp]),
    "lnrf_grad_nonfinite_check_amp_update": (i32, [vp, u32, vp, vp, vp, vp, f32, f32, i32, vp, vp]),
    "lnrf_grid_encode_backward_det": (i32, [vp, vp, vp, vp, vp, vp, u32, u32, u32, u32, f32, u32, vp, vp, u32, i32, u32, i32, i32, vp]),
    "lnrf_grid_encode_backward_world_det": (i32, [vp, vp, f32, vp, vp, vp, vp, u32, vp, u32, f32, u32, u32, i32, u32, i32, vp]),
    "lnrf_grid_det_finish": (i32, [vp, vp, vp, u32, vp, u32, u32, i32, vp]),
    "lnrf_ffmlp_backward_deterministic": (i32, [u32, u32, u32, u32, u32, u32]),
    "lnrf_occupancy_scatter_det": (i32, [vp, vp, u32, vp, vp, u32, vp]),
}

class RenderDesc(C.Structure):
    """lnrf_render_desc (include/laenerf_b200.h): everything one device-driven inference frame needs."""
    _fields_ = [
        ("ctl", vp), ("n_rays", u32), ("max_steps", u32),
        ("rays_o", vp), ("rays_d", vp), ("nears", vp), ("fars", vp),
        ("density_bitfield", vp), ("edit_bitfield", vp),
        ("bound", f32), ("dt_gamma", f32), ("T_thresh", f32),
        ("cascade", u32), ("grid_size", u32),
        ("first_round_noises", vp),
        ("embeddings_f16", vp), ("offsets_host", vp),
        ("num_levels", u32), ("base_resolution", u32), ("gridtype", u32), ("interpolation", u32),
        ("align_corners", i32), ("level_scale_log2", f32),
        ("w_sigma_f16", vp), ("w_color_f16", vp),
        ("num_layers_sigma", u32), ("num_layers_color", u32), ("density_scale", f32),
        ("rays_alive", vp * 2), ("rays_t", vp),
        ("xyzs", vp), ("dirs", vp), ("deltas", vp), ("edit_occ", vp), ("enc_f16", vp), ("sigmas", vp), ("rgbs", vp),
        ("weights_sum", vp), ("depth", vp), ("image", vp), ("weights_edit_sum", vp), ("depth_edit", vp),
        ("scratch", vp), ("scratch_bytes", sz),
        ("sample_rows", u32), ("samples_per_round", u32),
        ("ray_steps", vp), ("ray_flags", vp), ("nstep_seq", vp), ("nstep_len", u32), ("occupied_box", vp)
    ]


F32, F16 = 0, 1  # lnrf_dtype
GRID_LBC, GRID_BLC = 0, 1  # lnrf_grid_layout


def build(verbose: bool = False) -> str:
    """Compile liblaenerf_b200.so in-tree with nvcc for sm_100a (seconds; no torch headers involved)."""
    subprocess.run(["make", "-s", "-C", os.path.join(_HERE, "csrc"), "-j8"], check=True,
                   stdout=None if verbose else subprocess.DEVNULL)
    return SO_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"laenerf_b200: {SO_PATH} is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(make -C laenerf_b200/csrc).  There is no CPU or PyTorch fallback for this package.")
        l = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype, fn.argtypes = res, args
        if l.lnrf_sizeof_render_desc() != C.sizeof(RenderDesc) or l.lnrf_sizeof_opt_tensor() != C.sizeof(OptTensor):
            raise RuntimeError("laenerf_b200: the ctypes mirrors of lnrf_render_desc / lnrf_opt_tensor do not match "
                               f"{SO_PATH} (stale build?) -- rebuild with `make -C laenerf_b200/csrc`")
        _lib = l
    return _lib


def check(status: int) -> None:
    if status != 0:
        raise RuntimeError(lib().lnrf_last_error().decode("utf-8", "replace"))


def alert_not_deterministic(op: str) -> None:
    """What torch does for its own ops without a deterministic kernel: under torch.use_deterministic_algorithms(True) raise a
    RuntimeError naming the op, or warn when warn_only=True; nothing when the flag is off."""
    import torch
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = (f"{op} does not have a deterministic implementation, but you set 'torch.use_deterministic_algorithms(True)'. "
           "You can turn off determinism just for this operation, or you can use the 'warn_only=True' option, if that's "
           "acceptable for your application.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        import warnings
        warnings.warn(msg, UserWarning, stacklevel=3)
    else:
        raise RuntimeError(msg)


def ptr(t):
    """Device (or host) address of a tensor, None -> NULL."""
    return None if t is None else t.data_ptr()


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


# Work queued on side streams whose results the optimizer reads (the weight-gradient reduction of the fused network runs beside the
# hash-grid backward): AmpAdam.step() makes the current stream wait for them first.
_pending_streams = []


def defer_to_side_stream(dev):
    """A cached side stream for `dev`, made to wait for the current stream; the caller launches on it and it is joined by join_pending()."""
    import torch
    key = (dev.index if dev.index is not None else torch.cuda.current_device())
    s = _side_streams.get(key)
    if s is None:
        s = _side_streams[key] = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream())
    if s not in _pending_streams:
        _pending_streams.append(s)
    return s


_side_streams = {}


def join_pending():
    import torch
    while _pending_streams:
        torch.cuda.current_stream().wait_stream(_pending_streams.pop())


def launch_count() -> int:
    return int(lib().lnrf_launch_count())
