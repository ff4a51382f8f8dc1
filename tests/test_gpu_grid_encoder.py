"""The hash-grid encoder (laenerf_b200/csrc/gridenc.cu) against the CPU oracle (oracle/oracle.c), entry by entry, on every
kernel path: the tile kernels at the training shape and at small sizes, the generic kernel, input gradients, the total-variation
gradient, the device-side row count of the world-coordinate kernels and the grid-stride loop.  Nothing here needs the
reference's extensions.

Our side goes through the C ABI (tests/backends.py OursBackend, or ctypes directly for the world-coordinate entry points); the
reference side is oracle/pyoracle.py, given the level scales the device computes (lnrf_grid_level_scales) so that exp2f
differences cannot move a point into another cell.

Tolerances are derived from the arithmetic, not fitted.  u = 2^-24.  A is the same sum over absolute values (the oracle run on
|table| for the forward, on |grad| for the backward; the interpolation weights are >= 0) and n_e is the number of
(sample, corner) contributions with a nonzero weight to table entry e (touched_counts, a numpy restatement of the cell and
corner index):
  * fp32 forward:   |ours - oracle| <= 16 u A                (eight fma / mul+add steps on each side)
  * fp16 forward:   one fp16 ulp of the oracle value + 16 u A + 2^-24 (fp32 accumulation, one rounding to fp16)
  * fp32 backward:  (n_e + 2) u A_e                          (n_e fp32 additions, one product rounding in the oracle)
  * fp16 backward:  n_e 2^-10 A_e + n_e 2^-25 + (n_e + 2) u A_e  (per flush: one rounding to fp16, one fp16 addition)
Each check records the largest ratio of error to bound; run with -s to see them.
"""
import functools
import os
import zlib

import numpy as np
import pytest

from cases import grid_config, scene_rays
from oracle import pyoracle as O

U = 2.0 ** -24
P1, P2 = np.uint32(2654435761), np.uint32(805459861)


# ---------------------------------------------------------------------------------------------------------------------------
# helpers
def corner_entries(x, offsets, scales, gridtype=0, align=False, interp=0):
    """Per level: (table entries [n, 2^D], corner weights [n, 2^D]) of the in-range samples, in the kernels' corner order.
    Restates gridencoder.cu's cell (fma(x, scale, 0.5) rounded once), corner weights (fp32 products in the kernel's order) and
    index (dense strides while they fit the level, else the uint32 xor hash; then modulo the level size)."""
    x = np.asarray(x, np.float32)
    inside = ((x >= 0) & (x <= 1)).all(1)
    x64 = x[inside].astype(np.float64)
    D = x.shape[1]
    for level in range(len(offsets) - 1):
        hs = int(offsets[level + 1] - offsets[level])
        scale = float(np.float32(scales[level]))
        res = int(np.ceil(np.float32(scale))) + 1
        step = res if align else res + 1
        p = (x64 * scale + (0.0 if align else 0.5)).astype(np.float32)  # exact product, one rounding: fmaf
        pg = np.floor(p).astype(np.uint32)
        f = p - pg.astype(np.float32)
        if interp == 1:
            f = f * f * (np.float32(3.0) - np.float32(2.0) * f)
        strides, stride = [], 1
        for d in range(D):
            if stride > hs:
                break
            strides.append(np.uint32(stride))
            stride = (stride * step) & 0xFFFFFFFF
        hashed = gridtype == 0 and stride > hs
        entries, weights = [], []
        for c in range(1 << D):
            w = np.ones(len(x64), np.float32)
            corner = []
            for d in range(D):
                up = (c >> d) & 1
                w = w * (f[:, d] if up else np.float32(1.0) - f[:, d])
                corner.append(pg[:, d] + np.uint32(up))
            if hashed:
                idx = corner[0].copy()
                if D > 1:
                    idx ^= corner[1] * P1
                if D > 2:
                    idx ^= corner[2] * P2
            else:
                idx = np.zeros(len(x64), np.uint32)
                for d, s in enumerate(strides):
                    idx += corner[d] * s
            entries.append(int(offsets[level]) + (idx % np.uint32(hs)).astype(np.int64))
            weights.append(w)
        yield np.stack(entries, 1), np.stack(weights, 1)


def touched_counts(x, offsets, scales, gridtype=0, align=False, interp=0):
    """n_e: (sample, corner) contributions with a nonzero interpolation weight to each table entry."""
    counts = np.zeros(int(offsets[-1]), np.int64)
    for e, w in corner_entries(x, offsets, scales, gridtype, align, interp):
        counts += np.bincount(e[w != 0], minlength=counts.shape[0])
    return counts


def base_entries(x, offsets, scales, gridtype=0, align=False):
    """[n_inside, L] the entry of each in-range sample's base (lower) corner on every level: where its TV gradient goes."""
    return np.stack([e[:, 0] for e, _ in corner_entries(x, offsets, scales, gridtype, align)], 1)


def _spacing16(v):
    """One fp16 ulp at |v| (2^-24 in the subnormal range)."""
    return np.spacing(np.abs(np.asarray(v, np.float64)).astype(np.float16)).astype(np.float64)


def _h(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


RATIOS = {}


def _within(got, want, bound, what):
    got, want, bound = (np.asarray(a, np.float64) for a in (got, want, bound))
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = np.abs(got - want)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} outside the bound; first at {np.argwhere(bad)[0]}: "
                           f"got {got[bad][0]!r} want {want[bad][0]!r} bound {bound[bad][0]:.3e}")
    if not err.size:
        return 0.0
    r = err / np.where(bound > 0, bound, 1.0)
    i = np.unravel_index(np.argmax(r), r.shape)
    test = os.environ.get("PYTEST_CURRENT_TEST", "?").split(" ")[0]
    if r[i] >= RATIOS.get(test, (-1.0,))[0]:
        RATIOS[test] = (float(r[i]), what, float(want[i]), float(got[i]), float(bound[i]))
    return float(r[i])


@pytest.fixture(scope="module", autouse=True)
def _report_ratios():
    yield
    for k, (r, what, want, got, bound) in RATIOS.items():
        print(f"max error / bound  {r:.3g}  {k}  [{what}: oracle {want:.6g} ours {got:.6g} bound {bound:.3g}]")


def check_forward(got, x, emb, offsets, scales, half, gridtype=0, align=False, interp=0, layout=1, what="forward"):
    """got: our forward output (as float); oracle on the same (fp16-rounded when half) table."""
    emb = _h(emb) if half else np.asarray(emb, np.float32)
    kw = dict(gridtype=gridtype, align_corners=align, interp=interp, scales=scales, out_layout=layout)
    want = O.grid_encode_forward(x, emb, offsets, 0.0, 0, **kw)
    a = O.grid_encode_forward(x, np.abs(emb), offsets, 0.0, 0, **kw)
    bound = 16 * U * a.astype(np.float64)
    if half:
        bound += _spacing16(want) + 2.0 ** -24
    _within(got, want, bound, what)
    return want


def check_backward(got, grad, x, offsets, scales, half, counts, gridtype=0, align=False, interp=0, layout=1, what="backward"):
    """got: our grad_embeddings (as float); grad: what our kernel read (fp16-representable when half)."""
    C = got.shape[1]
    kw = dict(gridtype=gridtype, align_corners=align, interp=interp, scales=scales, grad_layout=layout)
    want = O.grid_encode_backward(grad, x, offsets, C, 0.0, 0, **kw)
    a = O.grid_encode_backward(np.abs(grad), x, offsets, C, 0.0, 0, **kw)
    n = counts[:, None].astype(np.float64)
    bound = (n + 2) * U * a
    if half:
        bound += n * 2.0 ** -10 * a + n * 2.0 ** -25
    _within(got, want, bound, what)
    return want


@pytest.fixture(scope="module")
def be(ours_backend):
    return ours_backend


def _scales(be, L, pls, H):
    return be.grid_level_scales(L, pls, H)


class _env:
    """Set an environment variable for the duration of a block (the grid launchers read LNRF_GRID_PAIR / LNRF_GRID_CAP on
    every call) and restore what was there."""

    def __init__(self, key, value):
        self.key, self.value = key, str(value)

    def __enter__(self):
        self.old = os.environ.get(self.key)
        os.environ[self.key] = self.value

    def __exit__(self, *a):
        if self.old is None:
            os.environ.pop(self.key, None)
        else:
            os.environ[self.key] = self.old


def _world_fwd(be, xw, bound, emb, offsets, S, H, half, gridtype=0, align=False, interp=0, count=None, sentinel=float("nan")):
    N, p, torch = be.N, be.N.ptr, be.torch
    x = be.f32(xw)
    e = be.f16(emb) if half else be.f32(emb)
    off = torch.from_numpy(np.asarray(offsets, np.int32))
    B, L = x.shape[0], off.shape[0] - 1
    out = torch.full((B, 2 * L), sentinel, dtype=e.dtype, device=be.dev)
    bd = None if count is None else torch.tensor([count], dtype=torch.int32, device=be.dev)
    N.check(be.lib.lnrf_grid_encode_forward_world(p(x), float(bound), p(e), p(off), p(out), B, p(bd), L, float(S), H, gridtype,
                                                  int(align), interp, N.F16 if half else N.F32, None))
    be._done()
    return be.n(out)


def _world_bwd(be, grad, xw, bound, offsets, S, H, half, gridtype=0, align=False, interp=0, count=None):
    N, p, torch = be.N, be.N.ptr, be.torch
    x = be.f32(xw)
    g = be.f16(grad) if half else be.f32(grad)
    off = torch.from_numpy(np.asarray(offsets, np.int32))
    B, L = x.shape[0], off.shape[0] - 1
    ge = torch.zeros(int(offsets[-1]), 2, dtype=g.dtype, device=be.dev)
    bd = None if count is None else torch.tensor([count], dtype=torch.int32, device=be.dev)
    N.check(be.lib.lnrf_grid_encode_backward_world(p(g), p(x), float(bound), p(off), p(ge), B, p(bd), L, float(S), H, gridtype,
                                                   int(align), interp, N.F16 if half else N.F32, None))
    be._done()
    return be.n(ge)


def _to_unit(xw, bound):
    """(x + bound) / (2 * bound) with the two fp32 roundings torch and the world-coordinate kernels use."""
    return ((np.asarray(xw, np.float32) + np.float32(bound)) * (np.float32(1.0) / np.float32(2.0 * bound))).astype(np.float32)


def _edge_points(D, scales, align, coarse=3):
    """Coordinates 0, 0.5, 1, 1 - 2^-24, -eps / 1 + eps in one coordinate at a time, and points on the cell boundaries of the
    coarse levels."""
    rng = np.random.default_rng(101)
    vals = np.array([0.0, 0.5, 1.0, 1.0 - 2.0 ** -24], np.float32)
    pts = [np.full(D, v, np.float32) for v in vals]
    pts += [rng.choice(vals, size=D).astype(np.float32) for _ in range(24)]
    for d in range(D):
        for bad in (np.nextafter(np.float32(0), np.float32(-1)), np.float32(-1e-7), np.nextafter(np.float32(1), np.float32(2)),
                    np.float32(1 + 1e-6)):
            q = rng.random(D).astype(np.float32)
            q[d] = bad
            pts.append(q)
    for level in range(min(coarse, len(scales))):
        s = float(scales[level])
        for k in range(0, int(np.ceil(s)) + 2):
            v = np.float32(k / s if align else (k - 0.5) / s)
            if 0 <= v <= 1:
                q = rng.random(D).astype(np.float32)
                q[k % D] = v
                pts.append(q)
                pts.append(np.full(D, v, np.float32))
    return np.stack(pts).astype(np.float32)


def _ray_runs(rng, n_rays, steps, D, dt):
    """Samples marching along random rays with a fixed step: consecutive samples share cells on the coarse levels."""
    o = rng.uniform(0.05, 0.95, size=(n_rays, 1, D))
    d = rng.standard_normal((n_rays, 1, D))
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    t = np.arange(steps)[None, :, None] * dt
    return np.clip(o + d * t, 0.0, 1.0).reshape(-1, D).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------------
# CPU tier: the index restatement behind the tolerances
@pytest.mark.parametrize("cfg", ["mixed", "custom"])
def test_touched_counts_match_the_oracle_support(cfg):
    """touched_counts must name exactly the entries the oracle's backward writes with an all-ones gradient (weights >= 0)."""
    rng = np.random.default_rng(1)
    for gridtype in (0, 1):
        for align in (False, True):
            for interp in (0, 1):
                offsets, pls, H, D = _config(cfg, align)
                L = len(offsets) - 1
                scales = O.grid_level_scales(L, float(np.log2(pls)), H)
                x = np.concatenate([rng.random((700, D), dtype=np.float32), _ray_runs(rng, 4, 40, D, 1 / 300),
                                    _edge_points(D, scales, align)])
                n = touched_counts(x, offsets, scales, gridtype, align, interp)
                ones = O.grid_encode_backward(np.ones((x.shape[0], L * 2), np.float32), x, offsets, 2, 0.0, 0, gridtype=gridtype,
                                              align_corners=align, interp=interp, scales=scales)
                assert np.array_equal(n > 0, (ones != 0).any(1)), (cfg, gridtype, align, interp)
                assert n.sum() > 0 and (n > 0).sum() < n.shape[0]


# ---------------------------------------------------------------------------------------------------------------------------
# level configurations of the small-size path matrix (D = 3, C = 2)
CONFIGS = ["dense", "mixed", "small_table", "custom"]


def _config(name, align=False):
    """-> (offsets, per_level_scale, base_resolution, D)
    dense:        every level dense and in range (x = 1 with align_corners wraps level 0's far corner)
    mixed:        dense coarse levels + hashed power-of-two tables (tiled: dense index wrapped by the mask)
    small_table:  every level larger than its 2^10 table (hash: hashed; tiled: wrapped by the mask)
    custom:       caller-supplied offsets: odd level sizes and odd bases, a non-power-of-two hashed table -> unpaired accesses
                  and the modulo paths"""
    if name == "dense":
        return (*grid_config(3, 2, 3, 8, 16, 32, align), 8, 3)
    if name == "mixed":
        return (*grid_config(6, 2, 3, 8, 12, 128, align), 8, 3)
    if name == "small_table":
        return (*grid_config(4, 2, 3, 16, 10, 64, align), 16, 3)
    if name == "custom":
        # base 4, scale 2: steps 5, 9, 17, 33 (align: 4, 8, 16, 32).  Level 0: 125 = 5^3 entries, dense; level 1: 731 > 9^3,
        # dense; level 2: 1001 < 17^3 (hashed / modulo-wrapped); level 3: 2047, same
        return np.cumsum([0, 125, 731, 1001, 2047]).astype(np.int32), 2.0, 4, 3
    raise KeyError(name)


def _path_inputs(rng, D, scales, align, B=1100):
    x = np.concatenate([_ray_runs(rng, 8, 48, D, 1 / 200), _edge_points(D, scales, align)])
    return np.concatenate([x, rng.random((B - x.shape[0], D), dtype=np.float32)])


@pytest.mark.gpu
@pytest.mark.parametrize("align", [False, True], ids=["noalign", "align"])
@pytest.mark.parametrize("gridtype", [0, 1], ids=["hash", "tiled"])
@pytest.mark.parametrize("interp", [0, 1], ids=["linear", "smooth"])
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
@pytest.mark.parametrize("cfg", CONFIGS)
def test_tile_kernels_path_matrix(be, cfg, half, interp, gridtype, align):
    """k_grid_fwd_tile / k_grid_bwd_tile, paired (LNRF_GRID_PAIR=3) and unpaired (0) table accesses, against the oracle."""
    offsets, pls, H, D = _config(cfg, align)
    L = len(offsets) - 1
    rng = np.random.default_rng(zlib.crc32(repr((cfg, half, interp, gridtype, align)).encode()))
    scales = _scales(be, L, pls, H)
    x = _path_inputs(rng, D, scales, align)
    emb = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
    g = (rng.standard_normal((x.shape[0], 2 * L)) * 0.05).astype(np.float32)
    g = _h(g) if half else g
    n = touched_counts(x, offsets, scales, gridtype, align, interp)
    kw = dict(gridtype=gridtype, align=align, interp=interp)
    for pair in (0, 3):
        with _env("LNRF_GRID_PAIR", pair):
            out = be.grid_fwd(x, emb, offsets, pls, H, half=half, **kw)
            ge = be.grid_bwd(g, x, offsets, 2, pls, H, half=half, **kw)
        check_forward(out, x, emb, offsets, scales, half, gridtype, align, interp, what=f"forward pair={pair}")
        check_backward(ge, g, x, offsets, scales, half, n, gridtype, align, interp, what=f"backward pair={pair}")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [1, 0], ids=["BLC", "LBC"])
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
@pytest.mark.parametrize("C", [1, 2, 4, 8])
@pytest.mark.parametrize("D", [2, 3])
def test_generic_kernel_path_matrix(be, D, C, half, layout):
    """k_grid_fwd_generic (forced by asking for dy_dx) / k_grid_bwd_generic / k_grid_input_bwd against the oracle: outputs,
    dy_dx, table gradients and input gradients, for a hashed linear and a tiled smoothstep align_corners setting."""
    rng = np.random.default_rng(1000 + 100 * D + 10 * C + 2 * half + layout)
    for gridtype, interp, align in ((0, 0, False), (1, 1, True)):
        offsets, pls = grid_config(5, C, D, 8, 11 if D == 3 else 8, 96, align)
        H, L = 8, len(offsets) - 1
        scales = _scales(be, L, pls, H)
        x = _path_inputs(rng, D, scales, align, B=900)
        B = x.shape[0]
        emb = rng.uniform(-1, 1, size=(int(offsets[-1]), C)).astype(np.float32)
        embq = _h(emb) if half else emb
        kw = dict(gridtype=gridtype, align=align, interp=interp)
        out, dd = be.grid_fwd(x, emb, offsets, pls, H, half=half, dy_dx=True, layout=layout, **kw)
        want = check_forward(out, x, emb, offsets, scales, half, gridtype, align, interp, layout, what="forward")
        # dy_dx: sum over 2^(D-1) corner pairs of w * (v_r - v_l) * pos_deriv, sum_w = scale, |v_r - v_l| <= 2 max|table|,
        # pos_deriv <= 1.5 (smoothstep) -> A <= 3 scale max|table| per (sample, level)
        _, dd_want = O.grid_encode_forward(x, embq, offsets, 0.0, 0, True, gridtype, align, interp, scales, layout)
        a = (3.0 * np.abs(embq).max() * scales.astype(np.float64))[None, :, None].repeat(B, 0).repeat(D * C, 2).reshape(B, -1)
        bound = 16 * U * a + ((_spacing16(dd_want) + 2.0 ** -24) if half else 0.0)
        _within(dd, dd_want, bound, "dy_dx")
        assert np.abs(want).max() > 0.1 and np.abs(dd_want).max() > 1.0
        gshape = (B, L * C) if layout == 1 else (L, B, C)
        g = (rng.standard_normal(gshape) * 0.05).astype(np.float32)
        g = _h(g) if half else g
        ge, gi = be.grid_bwd(g, x, offsets, C, pls, H, half=half, layout=layout, dy_dx=dd, **kw)
        n = touched_counts(x, offsets, scales, gridtype, align, interp)
        check_backward(ge, g, x, offsets, scales, half, n, gridtype, align, interp, layout, what="backward")
        # input gradients from OUR dy_dx: the same L*C-term fp32 sum on both sides
        _, gi_want = O.grid_encode_backward(g, x, offsets, C, 0.0, 0, dd, gridtype, align, interp, scales, layout)
        gb = g.reshape(B, L, 1, C) if layout == 1 else g.transpose(1, 0, 2).reshape(B, L, 1, C)
        a = (np.abs(gb).astype(np.float64) * np.abs(dd.reshape(B, L, D, C))).sum((1, 3))
        bound = (L * C + 2) * U * a + ((_spacing16(gi_want) + 2.0 ** -24) if half else 0.0)
        _within(gi, gi_want, bound, "grad_inputs")
        assert np.abs(gi_want).max() > 0.1


# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
@pytest.mark.parametrize("cfg", ["dense", "custom"])
def test_input_edges(be, cfg, half):
    """Edge coordinates alone, both align_corners settings; out-of-range points give exact zeros and no gradient."""
    for align in (False, True):
        offsets, pls, H, D = _config(cfg, align)
        L = len(offsets) - 1
        scales = _scales(be, L, pls, H)
        x = _edge_points(D, scales, align, coarse=L)
        rng = np.random.default_rng(7)
        emb = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
        g = (rng.standard_normal((x.shape[0], 2 * L)) * 0.05).astype(np.float32)
        g = _h(g) if half else g
        for interp in (0, 1):
            out = be.grid_fwd(x, emb, offsets, pls, H, half=half, align=align, interp=interp)
            check_forward(out, x, emb, offsets, scales, half, 0, align, interp)
            outside = ~((x >= 0) & (x <= 1)).all(1)
            assert outside.sum() == 4 * D and not out[outside].any()
            ge = be.grid_bwd(g, x, offsets, 2, pls, H, half=half, align=align, interp=interp)
            check_backward(ge, g, x, offsets, scales, half, touched_counts(x, offsets, scales, 0, align, interp), 0, align, interp)
            g_in = np.where(outside[:, None], g, 0).astype(np.float32)
            assert not be.grid_bwd(g_in, x, offsets, 2, pls, H, half=half, align=align, interp=interp).any()


@pytest.mark.gpu
@pytest.mark.parametrize("B", [0, 1, 127, 128, 129, 1000 + 37])
def test_batch_sizes(be, B):
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    S = float(np.log2(pls))
    scales = _scales(be, L, pls, H)
    rng = np.random.default_rng(B)
    x = rng.random((B, 3), dtype=np.float32)
    emb = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
    g = _h(rng.standard_normal((B, 2 * L)) * 0.05)
    n = touched_counts(x, offsets, scales)
    for half in (True, False):
        out = be.grid_fwd(x, emb, offsets, pls, H, half=half)
        assert out.shape == (B, 2 * L)
        ge = be.grid_bwd(g, x, offsets, 2, pls, H, half=half)
        xw = (x * 2.0 - 1.0).astype(np.float32)  # bound 1
        outw = _world_fwd(be, xw, 1.0, emb, offsets, S, H, half)
        gew = _world_bwd(be, g, xw, 1.0, offsets, S, H, half)
        if B == 0:
            assert not ge.any() and not gew.any()
            continue
        check_forward(out, x, emb, offsets, scales, half)
        check_forward(outw, _to_unit(xw, 1.0), emb, offsets, scales, half, what="forward_world")
        check_backward(ge, g, x, offsets, scales, half, n)
        check_backward(gew, g, _to_unit(xw, 1.0), offsets, scales, half, touched_counts(_to_unit(xw, 1.0), offsets, scales),
                       what="backward_world")


@pytest.mark.gpu
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
def test_backward_run_merging(be, half):
    """k_grid_bwd_tile sums the samples of one cell in registers and flushes when the cell changes: long same-cell runs, runs
    that leave a cell and come back (A, B, A), out-of-range samples and zero gradient rows inside a run, runs across the
    8-sample boundaries of the per-thread work items and across tiles."""
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    scales = _scales(be, L, pls, H)
    rng = np.random.default_rng(11)
    a = np.array([0.31, 0.52, 0.77], np.float32)
    b = np.array([0.62, 0.18, 0.41], np.float32)
    jit = lambda p, k: (p + rng.uniform(0, 1e-4, size=(k, 3))).astype(np.float32)  # noqa: E731
    parts = [
        jit(a, 45),                                                      # one long run, crosses several 8-sample items
        np.stack([a, a, b, b, a, a, b, a, b, a, a, a, b]),               # A, B, A
        jit(b, 3), np.array([[0.62, 1.2, 0.41], [-0.1, 0.18, 0.41]], np.float32), jit(b, 4),  # out of range inside a run
        jit(a, 5),                                                       # starts at item offset 4, crosses the 8 boundary
        _ray_runs(rng, 3, 70, 3, 1 / 400),                               # ray-like
        jit(b, 300),                                                     # across tile boundaries
    ]
    x = np.concatenate(parts).astype(np.float32)
    B = x.shape[0]
    g = (rng.standard_normal((B, 2 * L)) * 0.05).astype(np.float32)
    g[50:53] = 0.0                                                       # zero rows inside the A,B,A part
    g[70:72] = -0.0                                                      # and inside the out-of-range run
    g[5::9, 0::2] = 0.0                                                  # one channel zero, the other not
    g = _h(g) if half else g
    n = touched_counts(x, offsets, scales)
    for pair in (0, 3):
        with _env("LNRF_GRID_PAIR", pair):
            ge = be.grid_bwd(g, x, offsets, 2, pls, H, half=half)
        check_backward(ge, g, x, offsets, scales, half, n, what=f"backward pair={pair}")


@pytest.mark.gpu
@pytest.mark.parametrize("count", [0, 1, 300, 1280, 5000, -3])
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
def test_world_kernels_device_side_count(be, half, count):
    """B_dev (the training marcher's counter): forward rows below ceil128(count) equal the full-batch result and the rest keep
    their sentinel; the backward equals the backward over the first ceil128(count) rows.  5000 exceeds the 2560-row capacity
    the way an overflowing marcher counter does."""
    offsets, pls, H, D = _config("mixed")
    L = len(offsets) - 1
    S = float(np.log2(pls))
    scales = _scales(be, L, pls, H)
    rng = np.random.default_rng(20)
    cap, bound = 2560, 2.0
    xw = ((_ray_runs(rng, 20, 128, 3, 1 / 300)[:cap] * 2 - 1) * bound).astype(np.float32)
    emb = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
    g = _h(rng.standard_normal((cap, 2 * L)) * 0.05)
    live = min(-(-max(count, 0) // 128) * 128, cap)
    full = _world_fwd(be, xw, bound, emb, offsets, S, H, half)
    out = _world_fwd(be, xw, bound, emb, offsets, S, H, half, count=count, sentinel=7.0)
    assert np.array_equal(out[:live], full[:live]) and (out[live:] == 7.0).all()
    ge = _world_bwd(be, g, xw, bound, offsets, S, H, half, count=count)
    x01 = _to_unit(xw[:live], bound)
    if live == 0:
        assert not ge.any()
        return
    check_backward(ge, g[:live], x01, offsets, scales, half, touched_counts(x01, offsets, scales))


# ---------------------------------------------------------------------------------------------------------------------------
# training shape: 16 levels x 2^19 entries, desired resolution 2048 * bound, ray-ordered samples of a seeded march
@functools.lru_cache(maxsize=1)
def _training_case(name):
    from backends import OracleBackend, canonicalize
    orc = OracleBackend()
    sc, ro, rd, rng = scene_rays(name, 4096, 0)
    nears, fars = orc.near_far(ro, rd, sc.aabb, sc.min_near)
    noises = rng.random(4096, dtype=np.float32)
    xyzs, dirs, deltas, rays, counter = orc.march_train(ro, rd, sc.density_bitfield, sc.bound, 0.0, sc.max_steps, sc.cascade,
                                                        128, 4096 * sc.max_steps, nears, fars, noises)
    xw = np.ascontiguousarray(canonicalize(xyzs, dirs, deltas, rays)[1])
    offsets, pls = grid_config(16, 2, 3, 16, 19, 2048 * sc.bound)
    rng = np.random.default_rng(5)
    emb = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
    g = (rng.standard_normal((xw.shape[0], 32)) * 0.05).astype(np.float32)
    return dict(bound=sc.bound, xw=xw, x01=_to_unit(xw, sc.bound), offsets=offsets, pls=pls, emb=emb, g32=g, g16=_h(g), memo={})


def _training_expect(case, be):
    """Oracle results and bounds of one training case (computed once, reused by the grid-stride test)."""
    m = case["memo"]
    if not m:
        off, x01 = case["offsets"], case["x01"]
        m["scales"] = _scales(be, 16, case["pls"], 16)
        m["n"] = touched_counts(x01, off, m["scales"])
        for half in (True, False):
            emb = _h(case["emb"]) if half else case["emb"]
            g = case["g16"] if half else case["g32"]
            want = O.grid_encode_forward(x01, emb, off, 0.0, 0, scales=m["scales"])
            bound = 16 * U * O.grid_encode_forward(x01, np.abs(emb), off, 0.0, 0, scales=m["scales"]).astype(np.float64)
            if half:
                bound += _spacing16(want) + 2.0 ** -24
            m["fwd", half] = (want, bound)
            want = O.grid_encode_backward(g, x01, off, 2, 0.0, 0, scales=m["scales"])
            a = O.grid_encode_backward(np.abs(g), x01, off, 2, 0.0, 0, scales=m["scales"])
            n = m["n"][:, None].astype(np.float64)
            bound = (n + 2) * U * a + ((n * 2.0 ** -10 * a + n * 2.0 ** -25) if half else 0.0)
            m["bwd", half] = (want, bound)
    return m


def _training_run(be, case, tag):
    m = _training_expect(case, be)
    off, pls, bound = case["offsets"], case["pls"], case["bound"]
    S = float(np.log2(pls))
    for half in (True, False):
        g = case["g16"] if half else case["g32"]
        unit = be.grid_fwd(case["x01"], case["emb"], off, pls, 16, half=half)
        world = _world_fwd(be, case["xw"], bound, case["emb"], off, S, 16, half)
        _within(unit, *m["fwd", half], f"{tag} forward half={half}")
        assert np.array_equal(world, unit), "world-coordinate forward differs from the [0, 1] forward"
        for what, ge in (("backward", be.grid_bwd(g, case["x01"], off, 2, pls, 16, half=half)),
                         ("backward_world", _world_bwd(be, g, case["xw"], bound, off, S, 16, half))):
            _within(ge, *m["bwd", half], f"{tag} {what} half={half}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["lego", "bonsai", "flower"])  # flower last: the grid-stride test below reuses its oracle results
def test_training_shape(be, name):
    case = _training_case(name)
    assert case["xw"].shape[0] > 200_000
    m = _training_expect(case, be)
    assert m["n"][: case["offsets"][5]].max() > 100  # coarse levels: many samples per entry
    _training_run(be, case, name)


@pytest.mark.gpu
def test_training_shape_grid_stride_loop(be):
    """LNRF_GRID_CAP=1,1: 148 CTAs for flower's ~4 900 tiles, every CTA loops over many tiles in both directions."""
    case = _training_case("flower")
    assert case["xw"].shape[0] > 148 * 128 * 8
    with _env("LNRF_GRID_CAP", "1,1"):
        _training_run(be, case, "flower cap=1,1")


# ---------------------------------------------------------------------------------------------------------------------------
# input gradients through the module, total variation
@pytest.mark.gpu
@pytest.mark.parametrize("autocast", [False, True], ids=["fp32", "autocast"])
def test_grid_encoder_input_gradient_end_to_end(be, autocast):
    """GridEncoder with inputs.requires_grad (generic forward with dy_dx, tile backward + k_grid_input_bwd, torch's
    (x + bound) / (2 bound)) against the oracle's input gradient times the 1 / (2 bound) chain factor."""
    import torch
    from laenerf_b200.gridencoder import GridEncoder
    bound, dev = 2.0, be.dev
    torch.manual_seed(0)
    enc = GridEncoder(num_levels=6, base_resolution=8, log2_hashmap_size=12, desired_resolution=128).to(dev)
    rng = np.random.default_rng(30)
    with torch.no_grad():
        enc.embeddings.copy_(torch.from_numpy(rng.uniform(-1, 1, size=tuple(enc.embeddings.shape)).astype(np.float32)))
    xw = ((_ray_runs(rng, 6, 100, 3, 1 / 300) * 2 - 1) * bound).astype(np.float32)
    xw[::97] *= 1.3  # some points outside the box
    G = _h(rng.standard_normal((xw.shape[0], 12)) * 0.05)
    inputs = torch.from_numpy(xw).to(dev).requires_grad_(True)
    with torch.autocast("cuda", enabled=autocast):
        out = enc(inputs, bound=bound)
    (out.float() * torch.from_numpy(G).to(dev)).sum().backward()
    torch.cuda.synchronize()
    assert out.dtype == (torch.float16 if autocast else torch.float32)
    got = inputs.grad.cpu().numpy()
    x01 = ((inputs.detach() + bound) / (2 * bound)).cpu().numpy()
    off, L, C = enc.offsets.cpu().numpy(), 6, 2
    scales = _scales(be, L, enc.per_level_scale, 8)
    emb = enc.embeddings.detach().cpu().numpy()
    emb = _h(emb) if autocast else emb
    _, dd = O.grid_encode_forward(x01, emb, off, 0.0, 0, True, scales=scales)
    _, gi = O.grid_encode_backward(G, x01, off, C, 0.0, 0, dd, scales=scales)
    B = x01.shape[0]
    # dy_dx error (see test_generic_kernel_path_matrix), carried through the sum over levels and channels, then that sum's own
    # L*C fp32 additions, the fp16 rounding of grad_inputs under autocast, and the chain factor's two roundings
    a_dd = (3.0 * np.abs(emb).max() * scales.astype(np.float64))[None, :, None].repeat(B, 0).repeat(3 * C, 2).reshape(B, -1)
    e_dd = 16 * U * a_dd + ((_spacing16(dd) + 2.0 ** -24) if autocast else 0.0)
    gb = np.abs(G).astype(np.float64).reshape(B, L, 1, C)
    carried = (gb * e_dd.reshape(B, L, 3, C)).sum((1, 3))
    a_gi = (gb * np.abs(dd.reshape(B, L, 3, C))).sum((1, 3))
    e_gi = carried + (L * C + 2) * U * a_gi + ((_spacing16(gi) + 2.0 ** -24) if autocast else 0.0)
    chain = 1.0 / (2 * bound)
    want = gi.astype(np.float64) * chain
    _within(got, want, e_gi * chain + 2 * U * np.abs(want), "grad_inputs (world)")
    assert np.abs(want).max() > 0.1 and not got[~((x01 >= 0) & (x01 <= 1)).all(1)].any()


def _tv(be, x, emb, offsets, weight, pls, H, half, gridtype=0, align=False):
    N, p, torch = be.N, be.N.ptr, be.torch
    xi = be.f16(x) if half else be.f32(x)
    e = be.f16(emb) if half else be.f32(emb)
    off = torch.from_numpy(np.asarray(offsets, np.int32))
    grad = torch.zeros_like(e)
    B, D = x.shape
    N.check(be.lib.lnrf_grad_total_variation(p(xi), p(e), p(grad), p(off), float(weight), B, D, e.shape[1], off.shape[0] - 1,
                                             float(np.log2(pls)), H, gridtype, int(align), N.F16 if half else N.F32, None))
    be._done()
    return be.n(grad)


@pytest.mark.gpu
@pytest.mark.parametrize("half", [True, False], ids=["f16", "f32"])
def test_total_variation(be, half):
    """lnrf_grad_total_variation against pyoracle.grad_total_variation.  First with points whose base cells are distinct on
    every level (each entry holds one rounded value on both sides), then with random points.  |results| / sqrt(idelta) <=
    sqrt(2D) (Cauchy-Schwarz over at most 2D neighbours), so one contribution is at most weight / sqrt(2D) in magnitude."""
    weight = 0.05
    for cfg, gridtype, align in (("mixed", 0, False), ("custom", 1, True), ("small_table", 0, True)):
        offsets, pls, H, D = _config(cfg, align)
        L = len(offsets) - 1
        scales = _scales(be, L, pls, H)
        rng = np.random.default_rng(40)
        emb = rng.uniform(-1, 1, size=(int(offsets[-1]), 2)).astype(np.float32)
        embq = _h(emb) if half else emb
        cand = np.concatenate([_edge_points(D, scales, align), rng.random((3000, D), dtype=np.float32)])
        cand = _h(cand) if half else cand
        cand = cand[((cand >= 0) & (cand <= 1)).all(1)]
        base = base_entries(cand, offsets, scales, gridtype, align)
        used, keep = set(), []
        for i, row in enumerate(base.tolist()):
            if not used.intersection(row):
                used.update(row)
                keep.append(i)
        single = cand[keep]
        assert len(keep) > 30
        for x, tag in ((single, "single"), (cand, "random")):
            got = _tv(be, x, emb, offsets, weight, pls, H, half, gridtype, align)
            want = O.grad_total_variation(x, embq, np.zeros_like(emb), offsets, weight, 0.0, 0, gridtype, align, scales)
            n = np.bincount(base_entries(x, offsets, scales, gridtype, align).ravel(), minlength=emb.shape[0])
            n = n[:, None].astype(np.float64)
            if tag == "single":
                assert n.max() == 1
                # per value: rsqrtf (2 ulp) vs 1 / sqrtf, fma vs mul+add in idelta, two products: <= 14 u relative
                bound = 16 * U * np.abs(want) + ((_spacing16(want) + 2.0 ** -24) if half else 0.0)
            else:
                a = n * weight / np.sqrt(2 * D)
                bound = (n + 16) * U * a + ((n * 2.0 ** -10 * a + n * 2.0 ** -25) if half else 0.0)
            _within(got, want, bound, f"tv {cfg} {tag}")
            assert np.abs(want).max() > weight / 20
