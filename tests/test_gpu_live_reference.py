"""GPU tier, LIVE comparisons with the reference's own extensions (oracle/_ref, present on the GPU box) at the sizes BASELINE.json
names -- the parity holes VERDICT round 1 listed under "No oracle comparison at the BASELINE shapes":

  * march_rays_train sample counts over >= 10^6 rays, bit-exact, on lego (C=1), flower (C=2) and bonsai (C=5, dt_gamma = 0:
    the fast-forward path) + sample positions of a 65 536-ray subset bit for bit (SURVEY.md Appendix A);
  * march_rays / composite_rays rounds of a full bonsai-shape view (404 301 rays, bound 16, 5 cascades) with the reference's
    n_step rule: positions, deltas, rays_t and the kill pattern round by round;
  * grid_encode forward / backward at 16 levels x 2^19 x resolution 2048 * bound on ~228 k ray-ordered samples: forward against
    the reference kernel, backward against the reference kernel run with an fp32 table (an fp32-accumulated oracle made of the
    reference's own code) with the reference's fp16 atomic-order noise measured beside it;
  * lnrf_nerf_backward (the dominant call of the step) against the CPU oracle's composition of network_ff.py:51-79.

Everything goes through the C ABI (ctypes) on our side and through the pybind11 modules on the reference side.

The grid encoder is also checked without the reference: tests/test_gpu_grid_encoder.py compares every kernel path (the training
shape of lego, flower and bonsai included) entry by entry with the CPU oracle, under tolerances derived from the arithmetic.
"""
import ctypes as C
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from cases import scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def ref():
    import ref_step
    if not ref_step.ref_available():
        pytest.skip("oracle/_ref not built")
    return {k: ref_step.backend(k) for k in ("_raymarching", "_gridencoder", "_ffmlp", "_shencoder")}


def _N():
    from laenerf_b200 import _native as N
    return N


def _all_rays(name, n, seed, dev):
    """n rays drawn from ALL pixels of the scene's 4 cameras (a single view has fewer than 10^6 pixels)."""
    from laenerf_b200.scene import get_rays_np
    sc = scene(name)
    ros, rds = [], []
    for p in sc.poses:
        ro, rd, _ = get_rays_np(p, sc.intrinsics, sc.H, sc.W)
        ros.append(ro); rds.append(rd)
    ro, rd = np.concatenate(ros), np.concatenate(rds)
    pick = np.random.default_rng(seed).choice(ro.shape[0], size=min(n, ro.shape[0]), replace=False)
    return sc, torch.from_numpy(ro[pick]).to(dev), torch.from_numpy(rd[pick]).to(dev)


def _near_far_ours(sc, ro, rd):
    N = _N()
    n = ro.shape[0]
    aabb = torch.from_numpy(sc.aabb).to(ro.device)
    nears, fars = torch.empty(n, device=ro.device), torch.empty(n, device=ro.device)
    N.check(N.lib().lnrf_near_far_from_aabb(N.ptr(ro), N.ptr(rd), N.ptr(aabb), n, float(sc.min_near), N.ptr(nears), N.ptr(fars), None))
    return nears, fars


def _march_ours(sc, ro, rd, bits, nears, fars, noises, M, dt_gamma):
    N = _N()
    n, dev = ro.shape[0], ro.device
    xyzs, dirs, deltas = (torch.full((M, 3), float("nan"), device=dev), torch.full((M, 3), float("nan"), device=dev),
                          torch.full((M, 2), float("nan"), device=dev))
    rays = torch.full((n, 3), -7, dtype=torch.int32, device=dev)
    cnt = torch.zeros(2, dtype=torch.int32, device=dev)
    nbytes = N.lib().lnrf_march_rays_train_scratch_bytes(n)
    scratch = torch.zeros((nbytes + 7) // 8, dtype=torch.int64, device=dev)
    N.check(N.lib().lnrf_march_rays_train(N.ptr(ro), N.ptr(rd), N.ptr(bits), float(sc.bound), float(dt_gamma), int(sc.max_steps), n,
                                          int(sc.cascade), 128, M, N.ptr(nears), N.ptr(fars), N.ptr(xyzs), N.ptr(dirs), N.ptr(deltas),
                                          N.ptr(rays), N.ptr(cnt), N.ptr(noises), N.ptr(scratch), nbytes, None))
    torch.cuda.synchronize()
    return xyzs, dirs, deltas, rays, cnt


def _march_ref(rm, sc, ro, rd, bits, nears, fars, noises, M, dt_gamma):
    n, dev = ro.shape[0], ro.device
    xyzs, dirs, deltas = torch.zeros(M, 3, device=dev), torch.zeros(M, 3, device=dev), torch.zeros(M, 2, device=dev)
    rays = torch.empty(n, 3, dtype=torch.int32, device=dev)
    cnt = torch.zeros(2, dtype=torch.int32, device=dev)
    rm.march_rays_train(ro, rd, bits, float(sc.bound), float(dt_gamma), int(sc.max_steps), n, int(sc.cascade), 128, M, nears, fars, xyzs,
                        dirs, deltas, rays, cnt, noises)
    torch.cuda.synchronize()
    return xyzs, dirs, deltas, rays, cnt


def _canonical(rays, *bufs):
    """Per-ray segments gathered into ray-id order on the device (the reference hands segments out in atomic arrival order)."""
    order = torch.argsort(rays[:, 0].long(), stable=True)
    r = rays[order].long()
    counts, offs = r[:, 2], r[:, 1]
    total = int(counts.sum())
    starts = torch.cumsum(counts, 0) - counts
    seg = torch.repeat_interleave(torch.arange(r.shape[0], device=rays.device), counts, output_size=total)
    idx = offs[seg] + (torch.arange(total, device=rays.device) - starts[seg])
    return counts, [b[idx] for b in bufs]


def _bits_equal(a, b):
    return bool(((a.view(torch.int32) == b.view(torch.int32)) | ((a == 0) & (b == 0))).all())


def _digest(*tensors):
    """sha256 of the bits of the tensors (floats with -0 folded into +0, which _bits_equal does not tell apart)."""
    h = hashlib.sha256()
    for t in tensors:
        t = t + 0.0 if t.is_floating_point() else t
        h.update(t.contiguous().cpu().numpy().tobytes())
    return h.hexdigest()


@pytest.fixture(scope="module")
def march_golden():
    with open(os.path.join(ROOT, "tests", "golden", "ref_march_million.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("name,n,dt_gamma", [("lego", 1 << 20, 0.0), ("flower", 1 << 20, 0.0), ("bonsai", 1 << 20, 0.0),
                                             ("bonsai", 1 << 18, 1.0 / 256)])
def test_march_train_counts_bit_exact_on_a_million_rays(dev, march_golden, name, n, dt_gamma):
    """Against the reference's march_rays_train on the same rays, bit for bit.  The reference's results are stored as digests in
    tests/golden/ref_march_million.json (near/far, per-ray counts of every ray, positions / directions / deltas of a 65 536-ray
    subset, in ray-id order); where oracle/_ref is built the reference kernel is also run live."""
    import ref_step
    sc, ro, rd = _all_rays(name, n, 11, dev)
    n = ro.shape[0]
    assert n >= 750_000 or dt_gamma > 0 or name == "flower"  # flower: 4 x 190 512 pixels exist in total
    gold = march_golden[f"{name}_{n}_{dt_gamma:g}"]
    rm = ref_step.backend("_raymarching") if ref_step.ref_available() else None
    bits = torch.from_numpy(sc.density_bitfield).to(dev)
    nears, fars = _near_far_ours(sc, ro, rd)
    assert _digest(nears, fars) == gold["near_far"]
    if rm is not None:
        rn, rf = torch.empty_like(nears), torch.empty_like(fars)
        rm.near_far_from_aabb(ro, rd, torch.from_numpy(sc.aabb).to(dev), n, float(sc.min_near), rn, rf)
        assert _bits_equal(nears, rn) and _bits_equal(fars, rf)
    noises = torch.rand(n, device=dev, generator=torch.Generator(device=dev).manual_seed(5))
    # pass 1 with a token buffer: every ray overflows (nothing is written) but `rays` rows and the counters are complete
    _, _, _, rays_o_, cnt_o = _march_ours(sc, ro, rd, bits, nears, fars, noises, 128, dt_gamma)
    assert cnt_o.tolist() == gold["counter"] and cnt_o[1].item() == n
    co = rays_o_[torch.argsort(rays_o_[:, 0].long())][:, 2]
    assert _digest(co) == gold["counts"], "per-ray sample counts differ from the reference's"
    if rm is not None:
        _, _, _, rays_r_, cnt_r = _march_ref(rm, sc, ro, rd, bits, nears, fars, noises, 128, dt_gamma)
        assert cnt_o.tolist() == cnt_r.tolist()
        cr = rays_r_[torch.argsort(rays_r_[:, 0].long())][:, 2]
        assert torch.equal(co, cr), f"{int((co != cr).sum())} of {n} per-ray sample counts differ"
    assert int(co.sum()) == int(cnt_o[0]) and int(co.max()) > 8
    # pass 2 on a 65 536-ray subset with room for every sample: positions, directions and deltas bit for bit
    k = min(65536, n)
    sro, srd, sn, sf, sno = ro[:k].contiguous(), rd[:k].contiguous(), nears[:k].contiguous(), fars[:k].contiguous(), noises[:k].contiguous()
    M = int(co[:k].sum()) + 128
    xo, do_, lo, ro_rows, c2 = _march_ours(sc, sro, srd, bits, sn, sf, sno, M, dt_gamma)
    total = int(c2[0])
    assert bool((xo[total:] == 0).all()) and bool((lo[total:] == 0).all())  # self-zeroed tail == torch.zeros + reference kernel
    cnt_a, (xa, da, la) = _canonical(ro_rows, xo, do_, lo)
    assert c2.tolist() == gold["subset_counter"] and _digest(cnt_a) == gold["subset_counts"]
    assert _digest(xa) == gold["subset_xyzs"] and _digest(da) == gold["subset_dirs"] and _digest(la) == gold["subset_deltas"]
    if rm is not None:
        xr, dr, lr, rr_rows, c3 = _march_ref(rm, sc, sro, srd, bits, sn, sf, sno, M, dt_gamma)
        assert c2.tolist() == c3.tolist()
        cnt_b, (xb, db, lb) = _canonical(rr_rows, xr, dr, lr)
        assert torch.equal(cnt_a, cnt_b)
        assert _bits_equal(xa, xb) and _bits_equal(da, db) and _bits_equal(la, lb)


class _OracleRaymarching:
    """march_rays / composite_rays of the CPU oracle (oracle/oracle.c, raymarching.cu restated; tests/test_oracle_golden.py holds it
    to the reference's golden vectors bit for bit) behind the reference module's in-place signatures (raymarching/src/bindings.cpp)."""

    def __init__(self):
        from oracle import pyoracle
        self.o = pyoracle

    @staticmethod
    def _h(t):
        return t.cpu().numpy()

    def march_rays(self, n_alive, n_step, alive, rays_t, ro, rd, bound, dt_gamma, max_steps, C, H, bits, nears, fars, xyzs, dirs, deltas,
                   noises):
        h = self._h
        out = self.o.march_rays(n_alive, n_step, h(alive), h(rays_t), h(ro), h(rd), bound, h(bits), C, H, h(nears), h(fars), h(noises),
                                xyzs.shape[0], dt_gamma, max_steps)
        for dst, src in zip((xyzs, dirs, deltas), out):
            dst.copy_(torch.from_numpy(src))

    def composite_rays(self, n_alive, n_step, T_thresh, alive, rays_t, sigmas, rgbs, deltas, ws, depth, image):
        h = self._h
        out = self.o.composite_rays(n_alive, n_step, h(alive), h(rays_t), h(sigmas), h(rgbs), h(deltas), h(ws), h(depth), h(image),
                                    T_thresh)
        for dst, src in zip((alive, rays_t, ws, depth, image), out):
            dst.copy_(torch.from_numpy(src))


@pytest.fixture(scope="module")
def raymarching_ref():
    """The reference's raymarching extension where oracle/_ref is built, else the CPU oracle that restates it."""
    import ref_step
    return ref_step.backend("_raymarching") if ref_step.ref_available() else _OracleRaymarching()


def test_inference_rounds_bonsai_full_view_bit_exact(dev, raymarching_ref):
    """The loop of run_cuda (renderer.py:335-387) on a full bonsai-shape view (bound 16, C = 5): in every round the SAME state
    (rays_alive, rays_t) goes through the reference's march_rays and ours, then through both compositors with synthetic
    densities; the reference's results carry the state forward.  Positions / deltas bit-exact, kill pattern exact.  Without
    oracle/_ref the reference side is the CPU oracle's restatement of the same two kernels."""
    from laenerf_b200.scene import get_rays_np
    N, rm = _N(), raymarching_ref
    sc = scene("bonsai")
    ro, rd, _ = get_rays_np(sc.poses[1], sc.intrinsics, sc.H, sc.W)
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    n = ro.shape[0]
    assert n == 779 * 519
    bits = torch.from_numpy(sc.density_bitfield).to(dev)
    nears, fars = _near_far_ours(sc, ro, rd)
    alive = torch.arange(n, dtype=torch.int32, device=dev)
    rays_t = nears.clone()
    ws, depth, image = torch.zeros(n, device=dev), torch.zeros(n, device=dev), torch.zeros(n, 3, device=dev)
    step, rounds, compared = 0, 0, 0
    while step < sc.max_steps and alive.shape[0] > 0 and rounds < 40:
        n_alive = alive.shape[0]
        n_step = max(min(n // n_alive, 8), 1)
        rows = n_alive * n_step
        rows += 128 - rows % 128
        noises = torch.zeros(n_alive, device=dev)
        xr, dr, lr = torch.zeros(rows, 3, device=dev), torch.zeros(rows, 3, device=dev), torch.zeros(rows, 2, device=dev)
        rm.march_rays(n_alive, n_step, alive, rays_t, ro, rd, float(sc.bound), 0.0, int(sc.max_steps), int(sc.cascade), 128, bits, nears, fars,
                      xr, dr, lr, noises)
        xo, do_, lo = (torch.full((rows, 3), float("nan"), device=dev), torch.full((rows, 3), float("nan"), device=dev),
                       torch.full((rows, 2), float("nan"), device=dev))
        N.check(N.lib().lnrf_march_rays(n_alive, n_step, N.ptr(alive), N.ptr(rays_t), N.ptr(ro), N.ptr(rd), float(sc.bound), 0.0,
                                        int(sc.max_steps), int(sc.cascade), 128, N.ptr(bits), N.ptr(nears), N.ptr(fars), N.ptr(xo), N.ptr(do_),
                                        N.ptr(lo), N.ptr(noises), rows, None))
        torch.cuda.synchronize()
        assert _bits_equal(xo, xr) and _bits_equal(do_, dr) and _bits_equal(lo, lr), f"round {rounds} (n_alive {n_alive}, n_step {n_step})"
        compared += rows
        # synthetic densities: a deterministic function of the position, strong enough to terminate rays over the rounds
        sig = (40.0 * (torch.sin(7.0 * xr[:, 0]) * torch.cos(5.0 * xr[:, 1]) + 1.0)).contiguous()
        rgb = torch.sigmoid(xr).contiguous()
        a2, t2, w2, d2, i2 = alive.clone(), rays_t.clone(), ws.clone(), depth.clone(), image.clone()
        rm.composite_rays(n_alive, n_step, 1e-4, alive, rays_t, sig, rgb, lr, ws, depth, image)
        N.check(N.lib().lnrf_composite_rays(n_alive, n_step, 1e-4, N.ptr(a2), N.ptr(t2), N.ptr(sig), N.ptr(rgb), N.ptr(lo), N.ptr(w2),
                                            N.ptr(d2), N.ptr(i2), None))
        torch.cuda.synchronize()
        assert torch.equal(a2, alive), f"kill pattern differs in round {rounds}"
        assert torch.allclose(t2, rays_t, rtol=1e-6, atol=1e-7) and torch.allclose(w2, ws, rtol=2e-6, atol=1e-6)
        assert torch.allclose(i2, image, rtol=2e-6, atol=1e-6) and torch.allclose(d2, depth, rtol=2e-6, atol=1e-6)
        alive = alive[alive >= 0]
        step += n_step
        rounds += 1
    assert rounds >= 8 and compared > 2 * n


def _ray_ordered_samples(dev, name="lego", n_rays=4096):
    """xyzs of one training batch as the marcher emits them (ray-ordered: neighbouring samples share cells)."""
    from laenerf_b200.scene import get_rays_np
    sc = scene(name)
    ro, rd, _ = get_rays_np(sc.poses[0], sc.intrinsics, sc.H, sc.W, N=n_rays, rng=np.random.default_rng(3))
    ro, rd = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    bits = torch.from_numpy(sc.density_bitfield).to(dev)
    nears, fars = _near_far_ours(sc, ro, rd)
    noises = torch.rand(n_rays, device=dev, generator=torch.Generator(device=dev).manual_seed(9))
    _, _, _, _, cnt = _march_ours(sc, ro, rd, bits, nears, fars, noises, 128, 0.0)
    M = int(cnt[0])
    M += 128 - M % 128
    xyzs, _, _, _, _ = _march_ours(sc, ro, rd, bits, nears, fars, noises, M, 0.0)
    return sc, xyzs


@pytest.mark.parametrize("name", ["lego", "flower"])
def test_grid_encode_baseline_shape_against_the_reference_kernels(dev, ref, name):
    """16 levels, 2^19 entries, desired resolution 2048 * bound, ~2.3e5 ray-ordered samples (the bench's own launch)."""
    from laenerf_b200.gridencoder import GridEncoder
    N, ge = _N(), ref["_gridencoder"]
    sc, xyzs = _ray_ordered_samples(dev, name)
    B = xyzs.shape[0]
    assert B > 150_000
    torch.manual_seed(1)
    enc = GridEncoder(desired_resolution=2048 * sc.bound).to(dev)
    with torch.no_grad():
        enc.embeddings.uniform_(-1.0, 1.0)
    L, S, H = 16, float(np.log2(enc.per_level_scale)), 16
    x01 = ((xyzs + sc.bound) / (2 * sc.bound)).contiguous()
    emb16 = enc.embeddings.detach().half().contiguous()
    off_h = enc.offsets.cpu().contiguous()
    # ---- forward: ours ([B, L*C] direct) vs the reference kernel ([L, B, C] + permute) on the same fp16 table
    out_o = torch.full((B, 32), float("nan"), dtype=torch.half, device=dev)
    N.check(N.lib().lnrf_grid_encode_forward(N.ptr(x01), N.ptr(emb16), N.ptr(off_h), N.ptr(out_o), B, 3, 2, L, S, H, None, 0, 0, 0, N.F16,
                                             N.GRID_BLC, None))
    out_r = torch.empty(L, B, 2, dtype=torch.half, device=dev)
    ge.grid_encode_forward(x01, emb16, enc.offsets, out_r, B, 3, 2, L, S, H, None, 0, False, 0)
    out_r = out_r.permute(1, 0, 2).reshape(B, 32)
    torch.cuda.synchronize()
    err = (out_o.float() - out_r.float()).abs()
    assert bool((err <= 2.0 ** -9 * out_r.float().abs().clamp(min=1.0)).all()), float(err.max())  # SURVEY 8c: the reference rounds 8x per level
    # same through the world-coordinate entry point the product path uses
    out_w = torch.empty_like(out_o)
    N.check(N.lib().lnrf_grid_encode_forward_world(N.ptr(xyzs), float(sc.bound), N.ptr(emb16), N.ptr(off_h), N.ptr(out_w), B, None, L, S, H, 0, 0, 0,
                                                   N.F16, None))
    torch.cuda.synchronize()
    assert torch.equal(out_w, out_o)
    # ---- backward: fp16 gradients into an fp16 table.  Oracle = the reference kernel with an fp32 table (fp32 atomics).
    g = (torch.randn(B, 32, device=dev, generator=torch.Generator(device=dev).manual_seed(2)) * 0.05).half()
    g_lbc = g.view(B, L, 2).permute(1, 0, 2).contiguous()
    emb32 = enc.embeddings.detach().contiguous()
    ge32 = torch.zeros_like(emb32)
    ge.grid_encode_backward(g_lbc.float(), x01, emb32, enc.offsets, ge32, B, 3, 2, L, S, H, None, None, 0, False, 0)
    runs = []
    for _ in range(2):
        t = torch.zeros_like(emb16)
        ge.grid_encode_backward(g_lbc, x01, emb16, enc.offsets, t, B, 3, 2, L, S, H, None, None, 0, False, 0)
        runs.append(t.float())
    ge_o = torch.zeros_like(emb16)
    N.check(N.lib().lnrf_grid_encode_backward(N.ptr(g), N.ptr(x01), None, N.ptr(off_h), N.ptr(ge_o), B, 3, 2, L, S, H, None, None, 0, 0, 0, N.F16,
                                              N.GRID_BLC, None))
    torch.cuda.synchronize()
    assert bool(torch.isfinite(ge_o).all())
    scale = float(ge32.abs().max())
    err_ours = float((ge_o.float() - ge32).abs().max()) / scale
    err_ref = float((runs[0] - ge32).abs().max()) / scale          # the reference's own fp16 accumulation error
    run_noise = float((runs[0] - runs[1]).abs().max()) / scale      # the reference's atomic-order noise between two runs
    # ours sums runs of same-cell samples in fp32 registers before the fp16 reduction: it must not be further from the fp32
    # result than the reference's own fp16 path is (plus one fp16 ulp of the largest element)
    assert err_ours <= max(err_ref, run_noise) + 2.0 ** -10, (err_ours, err_ref, run_noise)
    # per-level mass: every level received the same total gradient as the oracle (guards the privatised coarse levels)
    for l in range(L):
        a, b = int(off_h[l]), int(off_h[l + 1])
        so, sr = ge_o[a:b].float().sum(0), ge32[a:b].sum(0)
        tol = 5e-3 * ge32[a:b].abs().sum(0) + 1e-3
        assert bool(((so - sr).abs() <= tol).all()), (l, so.tolist(), sr.tolist())
    # and the fp32-table variant of ours against the same oracle, tightly
    ge_o32 = torch.zeros_like(emb32)
    N.check(N.lib().lnrf_grid_encode_backward(N.ptr(g.float()), N.ptr(x01), None, N.ptr(off_h), N.ptr(ge_o32), B, 3, 2, L, S, H, None, None, 0, 0, 0,
                                              N.F32, N.GRID_BLC, None))
    torch.cuda.synchronize()
    assert float((ge_o32 - ge32).abs().max()) <= 1e-4 * scale


def _h(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float32)


@pytest.mark.parametrize("M,ns,nc,variant", [(8192, 2, 3, "saved"), (1152, 3, 2, "saved"), (8192, 2, 3, "recompute"), (1280, 2, 2, "recompute"),
                                             (640, 3, 3, "recompute"), (128 * 301, 2, 3, "recompute")])
def test_nerf_backward_matches_oracle_composition(dev, oracle_backend, M, ns, nc, variant):
    """lnrf_nerf_backward (colour-net backward with the glue fused + sigma-net backward + weight-gradient reduction) against the
    CPU oracle composed the way autograd composes network_ff.py:51-79: sigmoid', FFMLP backward, cat split, trunc_exp backward
    (activation.py:13-16), FFMLP backward."""
    N = _N()
    rng = np.random.default_rng(M)
    enc = _h(rng.standard_normal((M, 32)) * 0.5)
    dirs = rng.standard_normal((M, 3)).astype(np.float32)
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    amp = 0.25
    ws = _h(rng.uniform(-amp, amp, 64 * (32 + 64 * (ns - 1) + 16)))
    wc = _h(rng.uniform(-amp, amp, 64 * (32 + 64 * (nc - 1) + 16)))
    ds = 1.5
    gsig = (rng.standard_normal(M) * 1e-2).astype(np.float32)
    grgb = (rng.standard_normal((M, 3)) * 1e-1).astype(np.float32)
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a)).to(dev).to(dt)
    enc_d, dirs_d, ws_d, wc_d = t(enc, torch.half), t(dirs, torch.float32), t(ws, torch.half), t(wc, torch.half)
    sig, rgb = torch.empty(M, device=dev), torch.empty(M, 3, device=dev)
    lib = N.lib()
    genc = torch.full((M, 32), float("nan"), dtype=torch.half, device=dev)
    gws, gwc = torch.full_like(ws_d, float("nan")), torch.full_like(wc_d, float("nan"))
    nbytes = lib.lnrf_nerf_wgrad_scratch_bytes(ns, nc)
    scratch = torch.full((nbytes // 4,), float("nan"), device=dev)
    gsig_d, grgb_d = t(gsig, torch.float32), t(grgb, torch.float32)  # named: a temporary would be freed (and its block reused) before the launch
    dh = None
    if variant == "saved":   # round-1 pair: hidden activations saved by the forward, read back by two backward launches
        fb = torch.empty(ns + nc, M, 64, dtype=torch.half, device=dev)
        cin = torch.empty(M, 32, dtype=torch.half, device=dev)
        h0 = torch.empty(M, dtype=torch.half, device=dev)
        N.check(lib.lnrf_nerf_forward(N.ptr(enc_d), N.ptr(dirs_d), N.ptr(ws_d), N.ptr(wc_d), M, ns, nc, ds, 1, N.ptr(fb), N.ptr(cin), N.ptr(h0),
                                      N.ptr(sig), N.ptr(rgb), None))
        dh = torch.empty(M, 16, dtype=torch.half, device=dev)
        N.check(lib.lnrf_nerf_backward(N.ptr(gsig_d), N.ptr(grgb_d), N.ptr(rgb), N.ptr(h0), N.ptr(enc_d), N.ptr(cin), N.ptr(ws_d), N.ptr(wc_d),
                                       N.ptr(fb), M, ns, nc, ds, N.ptr(genc), N.ptr(gws), N.ptr(gwc), 0, N.ptr(dh), N.ptr(scratch), nbytes, None))
    else:                    # round-2 pair: only h is kept; the backward recomputes the hidden activations (csrc/nerfbwd.cu)
        assert lib.lnrf_nerf_backward_recompute_supported(ns, nc) == 1
        hbuf = torch.full((M, 16), float("nan"), dtype=torch.half, device=dev)
        N.check(lib.lnrf_nerf_forward_lean(N.ptr(enc_d), N.ptr(dirs_d), N.ptr(ws_d), N.ptr(wc_d), M, None, ns, nc, ds, N.ptr(hbuf), N.ptr(sig),
                                           N.ptr(rgb), None))
        N.check(lib.lnrf_nerf_backward_recompute(N.ptr(gsig_d), N.ptr(grgb_d), N.ptr(rgb), N.ptr(hbuf), N.ptr(enc_d), N.ptr(dirs_d), N.ptr(ws_d),
                                                 N.ptr(wc_d), M, None, ns, nc, ds, N.ptr(genc), N.ptr(gws), N.ptr(gwc), 0, N.ptr(scratch), nbytes,
                                                 None))
    torch.cuda.synchronize()
    # ---- oracle composition ----
    ob = oracle_backend
    h, fb_s = ob.ffmlp_fwd(enc, ws, 32, 16, 64, ns)
    h = _h(h)
    sh = _h(ob.sh(dirs, 4))
    cin_o = np.concatenate([sh, h[:, 1:], np.zeros((M, 1), np.float32)], axis=1)
    hc, fb_c = ob.ffmlp_fwd(cin_o, wc, 32, 16, 64, nc)
    rgb_o = _h(1.0 / (1.0 + np.exp(-_h(hc[:, :3]))))
    dy = np.zeros((M, 16), np.float32)
    dy[:, :3] = _h(_h(grgb) * ((1.0 - rgb_o) * rgb_o))       # torch.sigmoid backward on the half tensor
    gwc_o, gi_c = ob.ffmlp_bwd(dy, cin_o, wc, fb_c, 32, 16, 64, nc, 0, True)
    dh_o = np.zeros((M, 16), np.float32)
    dh_o[:, 0] = gsig * ds * np.exp(np.clip(h[:, 0], -15, 15))
    dh_o[:, 1:] = np.asarray(gi_c)[:, 16:31]
    dh_o = _h(dh_o)
    gws_o, gi_s = ob.ffmlp_bwd(dh_o, enc, ws, fb_s, 32, 16, 64, ns, 0, True)

    def relmax(a, b):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return np.abs(a - b).max() / np.abs(b).max()

    def rows_off(a, b, tol):   # fraction of rows further than tol * max|b| from the oracle (see the ReLU-mask note below)
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        return float(((np.abs(a - b).max(axis=1) / np.abs(b).max()) > tol).mean())

    if dh is not None:
        assert rows_off(dh.float().cpu().numpy(), dh_o, 3e-3) <= 1e-3
    else:
        assert np.allclose(hbuf.float().cpu().numpy(), h, rtol=2e-3, atol=2e-3)   # the one tensor the lean forward keeps
    assert bool(torch.isfinite(genc).all()) and bool(torch.isfinite(gws).all()) and bool(torch.isfinite(gwc).all())
    # dL/denc row by row: a hidden unit whose pre-activation is within an fp32 summation-order ulp of zero has its ReLU mask flipped
    # between the tensor-core sum and the oracle's sequential sum, which changes that ROW by a few per cent of the largest element;
    # measured: < 1e-4 of the rows at M = 8192.  Everything else agrees to fp16 rounding.
    ge, go = genc.float().cpu().numpy().astype(np.float64), np.asarray(gi_s, np.float64)
    row_err = np.abs(ge - go).max(axis=1) / np.abs(go).max()
    assert float((row_err > 5e-3).mean()) <= 1e-3, float((row_err > 5e-3).mean())
    assert float(np.median(row_err)) <= 1e-3 and float(row_err.max()) <= 0.2
    # weight gradients sum over all rows: the handful of mask-flipped rows moves them by a fraction of a per cent of the largest element
    assert relmax(gwc.float().cpu().numpy(), gwc_o) <= 1e-2, relmax(gwc.float().cpu().numpy(), gwc_o)
    assert relmax(gws.float().cpu().numpy(), gws_o) <= 1e-2, relmax(gws.float().cpu().numpy(), gws_o)


def test_recompute_pair_equals_saved_pair_and_honours_the_device_side_count(dev):
    """Round-2 kernels against the round-1 kernels on the same inputs: same MMAs and rounding points, so dL/denc is bit-identical and
    the weight gradients differ only by the order of the fp32 partial sums; with a device-side sample count the rows past it are
    skipped (outputs untouched, gradients as if those rows carried zero gradient)."""
    N = _N()
    lib = N.lib()
    M, ns, nc, ds = 128 * 77, 2, 3, 1.0
    g = torch.Generator(device=dev).manual_seed(3)
    enc = (torch.randn(M, 32, device=dev, generator=g) * 0.5).half()
    dirs = torch.nn.functional.normalize(torch.randn(M, 3, device=dev, generator=g), dim=-1)
    ws = ((torch.rand(64 * (32 + 64 * (ns - 1) + 16), device=dev, generator=g) - 0.5) * 0.5).half()
    wc = ((torch.rand(64 * (32 + 64 * (nc - 1) + 16), device=dev, generator=g) - 0.5) * 0.5).half()
    gsig = torch.randn(M, device=dev, generator=g) * 1e-2
    grgb = torch.randn(M, 3, device=dev, generator=g) * 1e-1
    nbytes = lib.lnrf_nerf_wgrad_scratch_bytes(ns, nc)
    scratch = torch.empty(nbytes // 4, device=dev)

    def saved():
        sig, rgb = torch.empty(M, device=dev), torch.empty(M, 3, device=dev)
        fb, cin, h0 = (torch.empty(ns + nc, M, 64, dtype=torch.half, device=dev), torch.empty(M, 32, dtype=torch.half, device=dev),
                       torch.empty(M, dtype=torch.half, device=dev))
        N.check(lib.lnrf_nerf_forward(N.ptr(enc), N.ptr(dirs), N.ptr(ws), N.ptr(wc), M, ns, nc, ds, 1, N.ptr(fb), N.ptr(cin), N.ptr(h0), N.ptr(sig),
                                      N.ptr(rgb), None))
        genc, gws, gwc, dh = torch.empty_like(enc), torch.empty_like(ws), torch.empty_like(wc), torch.empty(M, 16, dtype=torch.half, device=dev)
        N.check(lib.lnrf_nerf_backward(N.ptr(gsig), N.ptr(grgb), N.ptr(rgb), N.ptr(h0), N.ptr(enc), N.ptr(cin), N.ptr(ws), N.ptr(wc), N.ptr(fb), M, ns, nc,
                                       ds, N.ptr(genc), N.ptr(gws), N.ptr(gwc), 0, N.ptr(dh), N.ptr(scratch), nbytes, None))
        torch.cuda.synchronize()
        return sig, rgb, genc, gws, gwc

    def lean(m_dev=None, gs=gsig, gr=grgb):
        sig, rgb = torch.full((M,), -7.0, device=dev), torch.full((M, 3), -7.0, device=dev)
        h = torch.empty(M, 16, dtype=torch.half, device=dev)
        N.check(lib.lnrf_nerf_forward_lean(N.ptr(enc), N.ptr(dirs), N.ptr(ws), N.ptr(wc), M, N.ptr(m_dev), ns, nc, ds, N.ptr(h), N.ptr(sig), N.ptr(rgb),
                                           None))
        genc, gws, gwc = torch.full_like(enc, -7.0), torch.empty_like(ws), torch.empty_like(wc)
        N.check(lib.lnrf_nerf_backward_recompute(N.ptr(gs), N.ptr(gr), N.ptr(rgb), N.ptr(h), N.ptr(enc), N.ptr(dirs), N.ptr(ws), N.ptr(wc), M, N.ptr(m_dev),
                                                 ns, nc, ds, N.ptr(genc), N.ptr(gws), N.ptr(gwc), 0, N.ptr(scratch), nbytes, None))
        torch.cuda.synchronize()
        return sig, rgb, genc, gws, gwc

    a, b = saved(), lean()
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])
    for x, y in ((a[3], b[3]), (a[4], b[4])):
        assert float((x.float() - y.float()).abs().max()) <= 2e-3 * float(x.float().abs().max())
    # device-side count: 5000 live samples -> 40 tiles of 128 rows are processed, the other 37 are left alone
    live = 5000
    m_dev = torch.tensor([live, 0], dtype=torch.int32, device=dev)
    rows = (live + 127) // 128 * 128
    gs2, gr2 = gsig.clone(), grgb.clone()
    gs2[live:] = 0
    gr2[live:] = 0     # what composite_rays_train's backward leaves for rows no ray owns
    c = lean(m_dev, gs2, gr2)
    assert torch.equal(c[0][:rows], b[0][:rows]) and bool((c[0][rows:] == -7.0).all()) and bool((c[2][rows:] == -7.0).all())
    d = lean(None, gs2, gr2)
    assert torch.equal(c[2][:rows], d[2][:rows])
    for x, y in ((c[3], d[3]), (c[4], d[4])):
        assert float((x.float() - y.float()).abs().max()) <= 2e-3 * float(y.float().abs().max()) + 1e-6
