"""torch.use_deterministic_algorithms(True) on the device: the fixed-point hash-grid backward against the CPU oracle within its
derived bound, bit-identical results across calls, launch geometries and processes, non-finite handling, the deterministic
occupancy scatter, whole NeRF and style training runs, graph mode switching and the paths that refuse to run under the flag.

Bound of the deterministic backward (DESIGN.md section 4): with s the exact sum of an entry's contributions, n_e their number
and q the quantum, |r - s| <= (n_e + 2) u A_e  (fp32 run sums, as test_gpu_grid_encoder.check_backward)  + n_e q / 2
(one rounding to the quantum per flush) + 1/2 ulp of the output dtype at r (+ 1/2 ulp more when accumulating into a non-zero
buffer) + 2^-50 |s| (the int64 -> fp64 conversion and the fp64 add before the final rounding).
"""
import os
import subprocess
import sys
import warnings
import zlib

import numpy as np
import pytest

from cases import grid_config, scene, scene_rays
from oracle import pyoracle as O
from test_gpu_grid_encoder import (U, _config, _env, _h, _path_inputs, _ray_runs, _to_unit, _training_case, _within, corner_entries,
                                   touched_counts)

torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def be(ours_backend):
    return ours_backend


@pytest.fixture
def det():
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(False)


def quantum(grad, B, half):
    lb = int(np.ceil(np.log2(max(B, 1)))) if B > 1 else 0
    if half:
        E = 16
    else:
        g = np.abs(np.asarray(grad, np.float32))
        g = g[np.isfinite(g)]
        m = float(g.max()) if g.size else 0.0
        E = max(int(np.frexp(np.float32(m))[1]), -60) if m > 0 else -60
    return 2.0 ** (E + lb + 1 - 62)


def det_bwd(be, g, x, offsets, C, pls, H, half, gridtype=0, align=False, interp=0, layout=1, base=None, world=None, count=None):
    """Deterministic backward + finish through the C ABI; world = bound: x are world coordinates (lnrf_*_world_det)."""
    N, p = be.N, be.N.ptr
    xt = be.f32(x)
    gt = be.f16(g) if half else be.f32(g)
    off = torch.from_numpy(np.asarray(offsets, np.int32))
    B = xt.shape[0]
    D = xt.shape[1]
    L = off.shape[0] - 1
    E = int(offsets[-1])
    ge = torch.zeros(E, C, dtype=gt.dtype, device=be.dev) if base is None else (be.f16(base) if half else be.f32(base))
    acc = torch.zeros(E, C, dtype=torch.int64, device=be.dev)
    flags = torch.zeros(E, dtype=torch.int32, device=be.dev)
    gmax = None if half else torch.zeros(1, dtype=torch.int32, device=be.dev)
    dt = N.F16 if half else N.F32
    S = float(np.log2(pls))
    if world is not None:
        bd = None if count is None else torch.tensor([count], dtype=torch.int32, device=be.dev)
        N.check(be.lib.lnrf_grid_encode_backward_world_det(p(gt), p(xt), float(world), p(off), p(acc), p(flags), p(gmax), B, p(bd), L, S, H,
                                                           gridtype, int(align), interp, dt, None))
    else:
        N.check(be.lib.lnrf_grid_encode_backward_det(p(gt), p(xt), p(off), p(acc), p(flags), p(gmax), B, D, C, L, S, H, None, None, gridtype,
                                                     int(align), interp, dt, layout, None))
    if B > 0:
        N.check(be.lib.lnrf_grid_det_finish(p(acc), p(flags), p(gmax), B, p(ge), E, C, dt, None))
    torch.cuda.synchronize()
    assert not acc.any() and not flags.any(), "the finish kernel must re-arm the fixed-point sums and flags"
    return ge


def det_check(ge, g, x, offsets, scales, half, counts, B, gridtype=0, align=False, interp=0, layout=1, base=None, what="det backward"):
    C = ge.shape[1]
    got = ge.float().cpu().numpy().astype(np.float64)
    kw = dict(gridtype=gridtype, align_corners=align, interp=interp, scales=scales, grad_layout=layout)
    want = O.grid_encode_backward(g, x, offsets, C, 0.0, 0, **kw).astype(np.float64)
    a = O.grid_encode_backward(np.abs(g), x, offsets, C, 0.0, 0, **kw).astype(np.float64)
    if base is not None:
        want = want + np.asarray(base, np.float64)
    n = counts[:, None].astype(np.float64)
    q = quantum(g, B, half)
    spacing = (lambda v: np.spacing(np.abs(v).astype(np.float16)).astype(np.float64)) if half else \
              (lambda v: np.spacing(np.abs(v).astype(np.float32)).astype(np.float64))
    ulp = np.maximum(spacing(got), spacing(want))
    bound = (n + 2) * U * a + n * q / 2 + (1.0 if base is not None else 0.5) * ulp + 2.0 ** -50 * np.abs(want)
    _within(got, want, bound, what)
    return want


# ---------------------------------------------------------------------------------------------------------------------------
# 1. oracle bound
@pytest.mark.gpu
@pytest.mark.parametrize("align", [False, True], ids=["noalign", "align"])
@pytest.mark.parametrize("gridtype", [0, 1], ids=["hash", "tiled"])
@pytest.mark.parametrize("interp", [0, 1], ids=["linear", "smooth"])
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
@pytest.mark.parametrize("cfg", ["mixed", "custom"])
def test_det_tile_kernel_within_bound(be, cfg, half, interp, gridtype, align):
    offsets, pls, H, D = _config(cfg, align)
    L = len(offsets) - 1
    rng = np.random.default_rng(zlib.crc32(repr((cfg, half, interp, gridtype, align)).encode()))
    scales = be.grid_level_scales(L, pls, H)
    x = _path_inputs(rng, D, scales, align)
    g = (rng.standard_normal((x.shape[0], 2 * L)) * 0.05).astype(np.float32)
    g = _h(g) if half else g
    n = touched_counts(x, offsets, scales, gridtype, align, interp)
    kw = dict(gridtype=gridtype, align=align, interp=interp)
    ge = det_bwd(be, g, x, offsets, 2, pls, H, half, **kw)
    det_check(ge, g, x, offsets, scales, half, n, x.shape[0], gridtype, align, interp)
    base = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
    base = _h(base) if half else base
    ge = det_bwd(be, g, x, offsets, 2, pls, H, half, base=base, **kw)
    det_check(ge, g, x, offsets, scales, half, n, x.shape[0], gridtype, align, interp, base=base, what="det backward into a base")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [1, 0], ids=["BLC", "LBC"])
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
@pytest.mark.parametrize("C", [1, 2, 4, 8])
@pytest.mark.parametrize("D", [2, 3])
def test_det_generic_kernel_within_bound(be, D, C, half, layout):
    rng = np.random.default_rng(2000 + 100 * D + 10 * C + 2 * half + layout)
    for gridtype, interp, align in ((0, 0, False), (1, 1, True)):
        offsets, pls = grid_config(5, C, D, 8, 11 if D == 3 else 8, 96, align)
        H, L = 8, len(offsets) - 1
        scales = be.grid_level_scales(L, pls, H)
        x = _path_inputs(rng, D, scales, align, B=900)
        B = x.shape[0]
        gshape = (B, L * C) if layout == 1 else (L, B, C)
        g = (rng.standard_normal(gshape) * 0.05).astype(np.float32)
        g = _h(g) if half else g
        ge = det_bwd(be, g, x, offsets, C, pls, H, half, gridtype, align, interp, layout)
        det_check(ge, g, x, offsets, scales, half, touched_counts(x, offsets, scales, gridtype, align, interp), B, gridtype, align, interp,
                  layout)


@pytest.mark.gpu
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
def test_det_run_merging_within_bound(be, half):
    """Same-cell runs, A-B-A runs, zero rows and out-of-range samples inside runs, runs across item and tile boundaries."""
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    scales = be.grid_level_scales(L, pls, H)
    rng = np.random.default_rng(11)
    a = np.array([0.31, 0.52, 0.77], np.float32)
    b = np.array([0.62, 0.18, 0.41], np.float32)
    jit = lambda p, k: (p + rng.uniform(0, 1e-4, size=(k, 3))).astype(np.float32)  # noqa: E731
    x = np.concatenate([jit(a, 45), np.stack([a, a, b, b, a, a, b, a, b, a, a, a, b]), jit(b, 3),
                        np.array([[0.62, 1.2, 0.41], [-0.1, 0.18, 0.41]], np.float32), jit(b, 4), jit(a, 5),
                        _ray_runs(rng, 3, 70, 3, 1 / 400), jit(b, 300)]).astype(np.float32)
    g = (rng.standard_normal((x.shape[0], 2 * L)) * 0.05).astype(np.float32)
    g[50:53] = 0.0
    g[5::9, 0::2] = 0.0
    g = _h(g) if half else g
    ge = det_bwd(be, g, x, offsets, 2, pls, H, half)
    det_check(ge, g, x, offsets, scales, half, touched_counts(x, offsets, scales), x.shape[0])


@pytest.mark.gpu
@pytest.mark.parametrize("count", [0, 1, 300, 5000, -3])
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
def test_det_device_side_count(be, half, count):
    """Rows at or past ceil128(count) are never read, by the max pre-pass either: they hold NaN here."""
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    scales = be.grid_level_scales(L, pls, H)
    rng = np.random.default_rng(20)
    cap, bound = 2560, 2.0
    xw = ((_ray_runs(rng, 20, 128, 3, 1 / 300)[:cap] * 2 - 1) * bound).astype(np.float32)
    g = _h(rng.standard_normal((cap, 2 * L)) * 0.05)
    live = min(-(-max(count, 0) // 128) * 128, cap)
    g[live:] = np.nan
    ge = det_bwd(be, g, xw, offsets, 2, pls, H, half, world=bound, count=count)
    if live == 0:
        assert not ge.any()
        return
    x01 = _to_unit(xw[:live], bound)
    det_check(ge, g[:live], x01, offsets, scales, half, touched_counts(x01, offsets, scales), cap)


@pytest.mark.gpu
def test_det_training_shape_within_bound_and_reproducible(be):
    """lego at the training shape through both entry points, fp16 and fp32; then every launch geometry bit-identical."""
    case = _training_case("lego")
    off, pls, bound = case["offsets"], case["pls"], case["bound"]
    scales = be.grid_level_scales(16, pls, 16)
    n = touched_counts(case["x01"], off, scales)
    B = case["xw"].shape[0]
    for half in (True, False):
        g = case["g16"] if half else case["g32"]
        ref = det_bwd(be, g, case["x01"], off, 2, pls, 16, half)
        det_check(ref, g, case["x01"], off, scales, half, n, B, what=f"lego half={half}")
        world = det_bwd(be, g, case["xw"], off, 2, pls, 16, half, world=bound)
        det_check(world, g, case["x01"], off, scales, half, n, B, what=f"lego world half={half}")
        for cap in (None, "4,4", "1,1"):
            for pair in (0, 2):
                with _env("LNRF_GRID_PAIR", pair), _env("LNRF_GRID_CAP", cap or "16,16"):
                    for _ in range(2):
                        assert torch.equal(det_bwd(be, g, case["x01"], off, 2, pls, 16, half), ref), (half, cap, pair)
                        assert torch.equal(det_bwd(be, g, case["xw"], off, 2, pls, 16, half, world=bound), world), (half, cap, pair)
                    assert torch.equal(det_bwd(be, g, case["xw"], off, 2, pls, 16, half, world=bound, count=B), world)


# ---------------------------------------------------------------------------------------------------------------------------
# 3. non-finite values
@pytest.mark.gpu
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
def test_det_nonfinite_gradients_flag_exactly_their_entries(be, half):
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    scales = be.grid_level_scales(L, pls, H)
    rng = np.random.default_rng(31)
    x = np.concatenate([_ray_runs(rng, 6, 64, 3, 1 / 300), rng.random((500, 3), dtype=np.float32)]).astype(np.float32)
    x = np.clip(x, 0.0, 1.0)
    B = x.shape[0]
    g = _h(rng.standard_normal((B, 2 * L)) * 0.05)
    bad = [(17, 0, np.inf), (18, 0, np.inf), (200, 3, -np.inf), (401, 1, np.nan), (402, 5, np.nan)]
    gp = g.copy()
    clean = g.copy()
    want_nan = np.zeros(int(offsets[-1]), bool)
    per_level = list(corner_entries(x, offsets, scales))
    for s, level, v in bad:
        gp[s, 2 * level: 2 * level + 2] = v
        clean[s, 2 * level: 2 * level + 2] = 0.0
        want_nan[per_level[level][0][s]] = True
    ge = det_bwd(be, gp, x, offsets, 2, pls, H, half).float().cpu().numpy()
    got_nan = np.isnan(ge)
    assert (got_nan[:, 0] == got_nan[:, 1]).all() and np.array_equal(got_nan[:, 0], want_nan)
    ok = ~want_nan
    ge_clean = det_bwd(be, clean, x, offsets, 2, pls, H, half).float().cpu().numpy()
    if half:  # q depends only on B: the untouched entries are the clean run's, bit for bit
        assert np.array_equal(ge[ok], ge_clean[ok])
    else:
        want = O.grid_encode_backward(clean, x, offsets, 2, 0.0, 0, scales=scales).astype(np.float64)
        a = O.grid_encode_backward(np.abs(clean), x, offsets, 2, 0.0, 0, scales=scales).astype(np.float64)
        n = touched_counts(x, offsets, scales)[:, None].astype(np.float64)
        bound = (n + 2) * U * a + n * quantum(gp, B, False) / 2 + np.spacing(np.abs(want).astype(np.float32)) + 2.0 ** -50 * np.abs(want)
        _within(ge[ok], want[ok], bound[ok], "untouched entries")


@pytest.mark.gpu
def test_det_fp16_overflow_gives_inf_only_beyond_the_range(be):
    """Gradients near the fp16 maximum on one point: entries whose exact sum leaves the fp16 range become +-inf, others stay finite."""
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    scales = be.grid_level_scales(L, pls, H)
    x = np.tile(np.array([[0.3137, 0.5521, 0.7713]], np.float32), (6, 1))
    g = np.full((6, 2 * L), 60000.0, np.float32)
    g[:, 1::2] = -30000.0
    g[:, 2:4] = 1000.0
    ge = det_bwd(be, g, x, offsets, 2, pls, H, True).float().cpu().numpy()
    s = O.grid_encode_backward(g, x, offsets, 2, 0.0, 0, scales=scales).astype(np.float64)
    over = np.abs(s) > 65520.0 * (1 + 1e-3)
    inside = np.abs(s) < 65504.0
    assert over.any() and inside.any()
    assert np.isinf(ge[over]).all() and (np.sign(ge[over]) == np.sign(s[over])).all()
    assert np.isfinite(ge[inside]).all()


@pytest.mark.gpu
def test_det_amp_adam_skips_a_step_on_overflowing_gradients(det):
    from laenerf_b200.nerf import NeRFNetwork, TrainStep
    dev = torch.device("cuda", 0)
    sc = scene("lego")
    torch.manual_seed(0)
    m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
    m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    step = TrainStep(m)
    _, ro, rd, _ = scene_rays("lego", 2048, 3)
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    gt = torch.rand(2048, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    step(ro, rd, gt)
    m.update_mean_count()
    before = {k: v.detach().clone() for k, v in m.named_parameters()}
    step.optimizer._scale.fill_(2.0 ** 60)    # scaled gradients leave the fp16 range
    count = step.optimizer.step_count.clone()
    step(ro, rd, gt)
    torch.cuda.synchronize()
    assert float(step.optimizer._scale) == 2.0 ** 59
    assert torch.equal(step.optimizer.step_count, count)
    for k, v in m.named_parameters():
        assert torch.equal(v.detach(), before[k]), k


# ---------------------------------------------------------------------------------------------------------------------------
# 4. occupancy scatter
@pytest.mark.gpu
def test_det_occupancy_scatter_matches_torch_index_put(be, det):
    N, p = be.N, be.N.ptr
    dev = be.dev
    cells = 4096
    gen = torch.Generator(device=dev).manual_seed(3)
    for n in (1, 1000, 50000):
        idx = torch.randint(0, 300, (n,), device=dev, generator=gen, dtype=torch.int32)
        sig = torch.rand(n, device=dev, generator=gen)
        want = torch.full((cells,), -1.0, device=dev)
        want[idx.long()] = sig                     # torch's deterministic index_put_
        got = torch.full((cells,), -1.0, device=dev)
        winner = torch.full((cells,), -1, dtype=torch.int32, device=dev)
        N.check(be.lib.lnrf_occupancy_scatter_det(p(sig), p(idx), n, p(got), p(winner), cells, None))
        torch.cuda.synchronize()
        assert torch.equal(got, want), n
        assert bool((winner == -1).all())
        last = {}  # and that is the last occurrence of each index
        for i, j in enumerate(idx.cpu().tolist()):
            last[j] = i
        js = torch.tensor(list(last), device=dev)
        assert torch.equal(want[js], sig[torch.tensor(list(last.values()), device=dev)])


@pytest.mark.gpu
def test_det_partial_occupancy_updates_are_reproducible(det):
    from laenerf_b200.nerf import NeRFNetwork
    dev = torch.device("cuda", 0)
    sc = scene("lego")
    outs = []
    for _ in range(2):
        torch.manual_seed(0)
        m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
        with torch.no_grad():
            m.encoder.embeddings.uniform_(-0.5, 0.5, generator=torch.Generator(device=dev).manual_seed(1))
        m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
        m.iter_density = 16
        torch.manual_seed(5)
        m.update_extra_state()
        m.update_extra_state()
        torch.cuda.synchronize()
        outs.append((m.density_grid.clone(), m.density_bitfield.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


# ---------------------------------------------------------------------------------------------------------------------------
# 5-7. whole training runs
def _equal_states(a, b):
    assert a.keys() == b.keys()
    diff = [(k, int((a[k] != b[k]).sum()), a[k].numel()) for k in a if not torch.equal(a[k], b[k])]
    assert not diff, diff


@pytest.mark.gpu
def test_det_nerf_training_runs_are_bit_identical():
    import det_driver
    try:
        a = det_driver.nerf_run("graphed", lookahead=True)
        b = det_driver.nerf_run("graphed", lookahead=True)
    finally:
        torch.use_deterministic_algorithms(False)
    _equal_states(a, b)
    assert bool((a["loss"] > 0).all()) and bool(torch.isfinite(a["loss"]).all())


@pytest.mark.gpu
def test_det_nerf_eager_graphed_and_lookahead_agree():
    """perturb=False: no RNG stream is involved, so eager, graphed and pipelined steps train the same batches bit for bit."""
    import det_driver
    try:
        eager = det_driver.nerf_run("eager", perturb=False)
        plain = det_driver.nerf_run("graphed", lookahead=False, perturb=False)
        look = det_driver.nerf_run("graphed", lookahead=True, perturb=False)
    finally:
        torch.use_deterministic_algorithms(False)
    _equal_states(eager, plain)
    _equal_states(plain, look)


def _digest(*args):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "det_driver.py"), *args], env=env, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return r.stdout.strip().splitlines()[-1]


@pytest.mark.gpu
def test_det_nerf_training_across_processes():
    d = [_digest("nerf", "graphed", "lookahead") for _ in range(2)]
    assert d[0] == d[1] and len(d[0]) == 64


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["eager", "graphed"])
def test_det_style_training_across_processes(form):
    d = [_digest("style", form) for _ in range(2)]
    assert d[0] == d[1] and len(d[0]) == 64


# ---------------------------------------------------------------------------------------------------------------------------
# 8. mode switching
@pytest.mark.gpu
def test_det_flag_flip_after_capture_never_replays_the_other_mode():
    from laenerf_b200.nerf import GraphedTrainStep, NeRFNetwork, TrainStep
    dev = torch.device("cuda", 0)
    sc = scene("lego")
    m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
    m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    _, ro, rd, _ = scene_rays("lego", 1024, 9)
    b = (torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev), torch.rand(1024, 3, device=dev))
    g = GraphedTrainStep(TrainStep(m), 1024)
    g(*b)
    assert g.deterministic is False and not g.needs_recapture()
    try:
        torch.use_deterministic_algorithms(True)
        assert g.needs_recapture()
        with pytest.raises(RuntimeError, match="capture"):
            g(*b)
        g.capture(*b)
        assert g.deterministic is True and not g.needs_recapture()
        g(*b)
    finally:
        torch.use_deterministic_algorithms(False)
    assert g.needs_recapture()
    with pytest.raises(RuntimeError, match="capture"):
        g(*b)


# ---------------------------------------------------------------------------------------------------------------------------
# 9. paths without a deterministic implementation
@pytest.mark.gpu
def test_det_unsupported_paths_raise_or_warn():
    from laenerf_b200.ffmlp import FFMLP
    from laenerf_b200.gridencoder import GridEncoder
    dev = torch.device("cuda", 0)
    enc = GridEncoder(num_levels=4, log2_hashmap_size=10).to(dev)
    enc(torch.rand(256, 3, device=dev)).float().sum().backward()
    net = FFMLP(32, 16, 64, 2, activation="sigmoid").to(dev)   # not ReLU: the float-atomics backward
    x = torch.rand(256, 32, device=dev)
    try:
        torch.use_deterministic_algorithms(True)
        with pytest.raises(RuntimeError, match="grad_total_variation"):
            enc.grad_total_variation()
        with pytest.raises(RuntimeError, match="FFMLP"):
            net(x).float().sum().backward()
        torch.use_deterministic_algorithms(True, warn_only=True)
        with pytest.warns(UserWarning, match="grad_total_variation"):
            enc.grad_total_variation()
        with pytest.warns(UserWarning, match="FFMLP"):
            net(x).float().sum().backward()
    finally:
        torch.use_deterministic_algorithms(False)


@pytest.mark.gpu
def test_det_laenerf_nets_take_fixed_order_backward_kernels(det):
    """The NeRF sigma and colour nets (module and fused tier) and the style network's weight_net and offset_net (input 48)."""
    from laenerf_b200.ffmlp import backward_deterministic
    from laenerf_b200.nerf import NeRFNetwork
    from laenerf_b200.style_encoder import LAENeRF
    dev = torch.device("cuda", 0)
    m = NeRFNetwork(bound=1).to(dev)
    style = LAENeRF(None, dir_encoding="sphere_harmonics").to(dev)
    nets = [m.sigma_net, m.color_net, style.weight_net, style.offset_net]
    assert style.offset_net.input_dim == 48
    for net in nets:
        assert backward_deterministic(net.input_dim, net.padded_output_dim, net.hidden_dim, net.num_layers, net.activation), net
        x = torch.rand(256, net.input_dim, device=dev, requires_grad=True)
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            net(x).float().sum().backward()
    # the fused tier: forward_scaled + backward through the fused kernels, no raise
    m.train()
    x = torch.rand(1024, 3, device=dev) * 2 - 1
    d = torch.nn.functional.normalize(torch.randn(1024, 3, device=dev), dim=-1)
    with torch.autocast("cuda", dtype=torch.float16):
        s, rgb = m.forward_scaled(x, d)
    (s.float().sum() + rgb.float().sum()).backward()
    assert m.encoder.embeddings.grad is not None and torch.isfinite(m.encoder.embeddings.grad).all()


# ---------------------------------------------------------------------------------------------------------------------------
# 10. rendering
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lego", "bonsai"])
def test_det_render_matches_flag_off(name):
    from laenerf_b200.nerf import NeRFNetwork
    dev = torch.device("cuda", 0)
    sc = scene(name)
    torch.manual_seed(0)
    m = NeRFNetwork(bound=sc.bound, min_near=sc.min_near).to(dev)
    with torch.no_grad():
        m.encoder.embeddings.uniform_(-0.5, 0.5, generator=torch.Generator(device=dev).manual_seed(1))
    m.set_density_grid(torch.from_numpy(sc.density_grid).to(dev), thresh=10.0)
    m.eval()
    _, ro, rd, _ = scene_rays(name, 5003, 41)
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    outs = []
    for flag in (False, True):
        torch.use_deterministic_algorithms(flag)
        try:
            m.render_schedule, m._auto_fast_ok = "auto", True
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
                outs.append(m.run_cuda(ro, rd, perturb=False, bg_color=1, dt_gamma=1.0 / 128 if name == "bonsai" else 0))
        finally:
            torch.use_deterministic_algorithms(False)
    for k in ("image", "depth"):
        a, b = outs[0][k], outs[1][k]   # rays that end with zero weight have a NaN depth in both modes
        assert torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(), b.nan_to_num()), k


# ---------------------------------------------------------------------------------------------------------------------------
# 11. two GPUs
@pytest.mark.gpu
def test_det_sharded_training_on_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    r = [subprocess.run([sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc_per_node=2",
                         os.path.join(ROOT, "tests", "det_driver_multi.py")], capture_output=True, text=True, timeout=900)
         for _ in range(2)]
    for x in r:
        assert x.returncode == 0, x.stderr[-3000:]
    replicas = [[ln for ln in x.stdout.splitlines() if ln.startswith("replica ")] for x in r]
    digests = [sorted(ln for ln in x.stdout.splitlines() if ln.startswith("digest ")) for x in r]
    assert len(replicas[0]) == 2 and len(set(replicas[0])) == 1, replicas   # the replicas agree
    assert len(digests[0]) == 2 and digests[0] == digests[1], digests      # and the two runs, rank by rank
