"""GPU tier, one GPU: the fp32 sharded exchange of the edit-stage style network (csrc/optim.cu `k_adam_step_p2p<float, float>`,
`lnrf_adam_step_sharded_f32`; laenerf_b200.optim.ShardedFlatAdam).  The kernel sees only per-rank device POINTERS (fp32 gradient
vector, fp32 parameter vector, flag buffer of every rank), so R local buffer sets emulate R ranks exactly, as in
test_gpu_sharded_optimizer.py for the fp16 form.  Checked against `lnrf_adam_step` (itself checked against torch.optim.Adam +
GradScaler in test_gpu_fused.py) on the fp32 mean of the R gradients, one call per learning-rate segment:

  * result == single-GPU Adam on the mean gradient with per-segment learning rates, R = 2 and R = 8, over 4 steps;
  * every "rank" ends with the same bits in its parameter vector; a rerun on the same inputs gives the same bits;
  * a non-finite gradient on one rank skips the update on every rank and backs the loss scale off once;
  * the moments of a rank are written only inside its slice;
  * StyleTrainStep with ShardedFlatAdam at R = 1 follows today's StyleTrainStep (AmpAdam) within fp32 rounding.
"""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

HYPER = (1e-3, 0.9, 0.999, 1e-8, 0.0)   # the style network's Adam
AMP = (2.0, 0.5, 2000)                  # GradScaler growth, back-off, interval
GUARD = 64                              # sentinel words behind every moment slice


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)


class _Ranks32:
    """R emulated ranks: full fp32 gradient / parameter / flag buffers each, moments for the owned slice only (plus a guard), and a
    GradScaler state per rank (every rank keeps its own copy; they must stay identical)."""

    def __init__(self, dev, R, Sz, segs, seed=0):
        from laenerf_b200 import _native as N
        self.N, self.R, self.Sz, self.P = N, R, Sz, R * Sz
        self.seg_start = [s for s, _ in segs]
        self.seg_mult = [m for _, m in segs]
        g = torch.Generator(device=dev).manual_seed(seed)
        self.p0 = torch.rand(self.P, device=dev, generator=g) - 0.5
        self.grad = [torch.zeros(self.P, device=dev) for _ in range(R)]
        self.param = [self.p0.clone() for _ in range(R)]
        self.flag = [torch.zeros(32, device=dev) for _ in range(R)]
        self.m = [torch.full((Sz + GUARD,), 7.0, device=dev) for _ in range(R)]
        self.v = [torch.full((Sz + GUARD,), 7.0, device=dev) for _ in range(R)]
        for t in self.m + self.v:
            t[:Sz] = 0.0
        self.scale = [torch.full((1,), 1024.0, device=dev) for _ in range(R)]
        self.tracker = [torch.zeros(1, dtype=torch.int32, device=dev) for _ in range(R)]
        self.step_count = [torch.ones(1, device=dev) for _ in range(R)]
        self.found = [torch.zeros(1, device=dev) for _ in range(R)]
        mk = lambda ts: (C.c_void_p * R)(*[t.data_ptr() for t in ts])
        self.arrays = (mk(self.grad), mk(self.param), mk(self.flag))

    def fill_grads(self, seed, bad_rank=None):
        dev = self.p0.device
        g = torch.Generator(device=dev).manual_seed(seed)
        for r in range(self.R):
            self.grad[r].copy_(torch.randn(self.P, device=dev, generator=g) * 8.0)   # "scaled" gradients, |g| ~ 8
        if bad_rank is not None:
            self.grad[bad_rank][12345 % self.P] = float("inf")

    def mean_grad(self):
        acc = torch.zeros(self.P, device=self.p0.device)
        for r in range(self.R):  # the kernel's order: rank 0, 1, ... added in fp32, then one multiply by 1/R
            acc += self.grad[r]
        return acc * (1.0 / self.R)

    def step(self):
        """Every rank: inf check into its flag, the exchange kernel, then clear + GradScaler.update() (ShardedFlatAdam.step)."""
        N, lib = self.N, self.N.lib()
        for r in range(self.R):
            self.flag[r][0] = 0.0
            arr = (N.OptTensor * 1)()
            arr[0].grad, arr[0].n, arr[0].grad_dtype = self.grad[r].data_ptr(), self.P, N.F32
            N.check(lib.lnrf_grad_nonfinite_check(C.cast(arr, C.c_void_p), 1, N.ptr(self.flag[r]), None))
        g, p, f = self.arrays
        starts = (C.c_uint64 * len(self.seg_start))(*self.seg_start)
        mults = (C.c_double * len(self.seg_mult))(*self.seg_mult)
        for r in range(self.R):
            N.check(lib.lnrf_adam_step_sharded_f32(C.cast(g, C.c_void_p), C.cast(p, C.c_void_p), C.cast(f, C.c_void_p), self.R, r, r * self.Sz,
                                                   self.Sz, starts, mults, len(self.seg_start), N.ptr(self.m[r]), N.ptr(self.v[r]), *HYPER,
                                                   N.ptr(self.scale[r]), N.ptr(self.found[r]), N.ptr(self.step_count[r]), None, None))
        for r in range(self.R):
            N.check(lib.lnrf_exchange_tail(N.ptr(self.grad[r]), 2 * self.P, N.ptr(self.scale[r]), N.ptr(self.tracker[r]), N.ptr(self.found[r]),
                                           N.ptr(self.step_count[r]), *AMP, None))
        torch.cuda.synchronize()


class _Single:
    """lnrf_adam_step on the full fp32 vector, one descriptor per learning-rate segment at lr x mult: the comparison target."""

    def __init__(self, ranks):
        self.N, self.ranks = ranks.N, ranks
        self.p = ranks.p0.clone()
        self.m, self.v = torch.zeros_like(self.p), torch.zeros_like(self.p)
        self.scale = torch.full((1,), 1024.0, device=self.p.device)
        self.step_count = torch.ones(1, device=self.p.device)

    def step(self, grad):
        N, rk = self.N, self.ranks
        g = grad.clone()
        bounds = rk.seg_start + [rk.P]
        for s, mult in enumerate(rk.seg_mult):
            a, b = bounds[s], bounds[s + 1]
            arr = (N.OptTensor * 1)()
            arr[0].params, arr[0].exp_avg, arr[0].exp_avg_sq = self.p[a:].data_ptr(), self.m[a:].data_ptr(), self.v[a:].data_ptr()
            arr[0].grad, arr[0].params_f16, arr[0].n, arr[0].grad_dtype = g[a:].data_ptr(), None, b - a, N.F32
            lr = HYPER[0] * mult
            N.check(N.lib().lnrf_adam_step(C.cast(arr, C.c_void_p), 1, lr, *HYPER[1:], N.ptr(self.scale), None, N.ptr(self.step_count), None, None))
        self.step_count += 1.0
        torch.cuda.synchronize()


def _segs(P):
    # table-like bulk at lr, a middle part at 0.5 lr, a palette-sized tail at 2 lr (the style network's layout has the first and last)
    return [(0, 1.0), (P // 2 // 8 * 8 + 8, 0.5), (P - 32, 2.0)]


@pytest.mark.parametrize("R", [2, 8])
def test_fp32_exchange_equals_single_gpu_adam_on_the_mean_gradient(dev, R):
    Sz = 8 * 1000 * 13  # a multiple of 8 that is not a multiple of the 2048-element chunk
    ranks = _Ranks32(dev, R, Sz, _segs(R * Sz), seed=R)
    single = _Single(ranks)
    for it in range(4):
        ranks.fill_grads(100 + it)
        mean = ranks.mean_grad()
        ranks.step()
        single.step(mean)
        for r in range(R):
            assert torch.equal(ranks.param[r], ranks.param[0]), (it, r)            # replicas identical, bit for bit
            assert float(ranks.found[r]) == 0.0 and float(ranks.step_count[r]) == it + 2
            assert float(ranks.grad[r].abs().max()) == 0.0                         # cleared for the next backward
        got = ranks.param[0]
        assert torch.allclose(got, single.p, rtol=0, atol=2e-7), float((got - single.p).abs().max())
        assert torch.allclose(torch.cat([m[:Sz] for m in ranks.m]), single.m, rtol=1e-6, atol=1e-9)
        assert torch.allclose(torch.cat([v[:Sz] for v in ranks.v]), single.v, rtol=1e-6, atol=1e-12)
    # the segments took their own learning rates: Adam's first steps move an entry by ~lr x mult
    moved = (ranks.param[0] - ranks.p0).abs()
    P = R * Sz
    assert float(moved[:P // 2 - 64].max()) > 3e-3 and float(moved[P - 32:].max()) > 2.5e-3 and float(moved[P // 2 + 64:P - 64].max()) < 2.1e-3
    for r in range(R):  # moments written inside the owned slice only
        assert bool((ranks.m[r][Sz:] == 7.0).all()) and bool((ranks.v[r][Sz:] == 7.0).all())


def test_fp32_exchange_is_deterministic(dev):
    R, Sz = 4, 8 * 3000
    runs = []
    for _ in range(2):
        ranks = _Ranks32(dev, R, Sz, _segs(R * Sz), seed=9)
        for it in range(3):
            ranks.fill_grads(700 + it)
            ranks.step()
        runs.append((ranks.param[0].clone(), torch.cat([m[:Sz] for m in ranks.m]), torch.cat([v[:Sz] for v in ranks.v])))
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_fp32_nonfinite_gradient_on_one_rank_skips_everywhere_and_backs_off_once(dev):
    R, Sz = 4, 8 * 4096
    ranks = _Ranks32(dev, R, Sz, _segs(R * Sz), seed=5)
    ranks.fill_grads(7, bad_rank=2)
    before = ranks.param[0].clone()
    ranks.step()
    for r in range(R):
        assert float(ranks.flag[r][0]) == (1.0 if r == 2 else 0.0)
        assert torch.equal(ranks.param[r], before) and float(ranks.m[r][:Sz].abs().sum()) == 0.0
        assert float(ranks.scale[r]) == 512.0 and float(ranks.step_count[r]) == 1.0   # backed off once, step not counted
        assert float(ranks.grad[r].abs().max()) == 0.0
    ranks.fill_grads(8)   # the next step with clean gradients proceeds normally (at the new scale)
    ranks.step()
    assert all(float(s) == 512.0 for s in ranks.scale) and all(float(c) == 2.0 for c in ranks.step_count)
    assert float((ranks.param[0] - before).abs().max()) > 5e-4


def _edit_stage_inputs(dev, K=49152):
    """The edit stage's step shape (bench.py edit_config): flower bound, at most 49 152 masked points a view, its loss weights."""
    from types import SimpleNamespace
    params = SimpleNamespace(bound=2.0, num_palette_bases=8, style_weight=0.0, weight_loss_uniform=1e-6, weight_loss_non_uniform=1e-6,
                             offset_loss=1e-6, palette_loss_valid=1e-3, palette_loss_distinct=1e-3)
    g = torch.Generator(device=dev).manual_seed(4)
    views = [((torch.rand(K, 3, device=dev, generator=g) - 0.5) * 3.0, torch.nn.functional.normalize(torch.randn(K, 3, device=dev, generator=g), dim=-1),
              torch.rand(K, 3, device=dev, generator=g)) for _ in range(6)]
    return params, views


def _owners(m):
    """StyleTrainStep's owners for ShardedFlatAdam: the table's gradient arrives in the flat vector (persistent), palette at 2 lr."""
    return [(m.encoder, m.encoder.embeddings, 1.0, True, 0), (m.weight_net, m.weight_net.weights, 1.0, False, 1),
            (m.offset_net, m.offset_net.weights, 1.0, False, 2), (m, m.color_palette, 2.0, False, 3)]


def test_style_step_on_the_sharded_optimizer_follows_todays_step(dev):
    """R = 1: the table gradient goes straight into the flat vector, the nets' and palette's are copied in; over six steps the
    parameters stay within fp32 rounding (plus the encoder backward's fp32-atomic order) of today's StyleTrainStep."""
    from laenerf_b200.optim import ShardedFlatAdam
    from laenerf_b200.style_encoder import LAENeRF, StyleTrainStep
    params, views = _edit_stage_inputs(dev)
    runs = []
    for sharded in (False, True):
        torch.manual_seed(1)
        style = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
        st = StyleTrainStep(style, params)
        if sharded:
            st.optimizer = ShardedFlatAdam(_owners(style), lr=1e-3, betas=(0.9, 0.999), eps=1e-8, n_groups=4)
            opt = st.optimizer
            assert opt.state[0]["exp_avg"].numel() == opt.P_pad and style.color_palette.is_leaf and style.color_palette.requires_grad
            assert style.color_palette.data_ptr() == opt.param_flat[opt._offsets[3]:].data_ptr()
        losses = [float(st(*v)[0]) for v in views]
        if sharded:
            assert style.encoder.embeddings.grad is None   # no autograd gradient for the table: it went into the flat vector
            # checkpoints round-trip: the module's parameters ARE the flat vector; the optimizer's state has torch.optim.Adam's layout
            sd = style.state_dict()
            assert torch.equal(sd["encoder.embeddings"], style.encoder.embeddings.detach())
            osd = opt.state_dict()
            assert torch.equal(osd["state"][0]["exp_avg"].reshape(-1), opt.state[0]["exp_avg"][:style.encoder.embeddings.numel()])
            assert osd["param_groups"][3]["lr"] == 2e-3
            style2 = LAENeRF(params, dir_encoding="sphere_harmonics").to(dev)
            opt2 = ShardedFlatAdam(_owners(style2), n_groups=4)
            style2.load_state_dict(sd)
            opt2.load_state_dict(osd)
            assert torch.equal(style2.encoder.embeddings.detach(), style.encoder.embeddings.detach())
            for k in ("exp_avg", "exp_avg_sq"):
                assert torch.equal(opt2.state[0][k][:opt._offsets[3]], opt.state[0][k][:opt._offsets[3]])
            assert float(opt2.step_count) == float(opt.step_count)
        runs.append((losses, style.encoder.embeddings.detach().clone(), style.weight_net.weights.detach().clone(),
                     style.color_palette.detach().clone()))
    (la, ea, wa, pa), (lb, eb, wb, pb) = runs
    assert all(np.isfinite(la)) and np.allclose(la, lb, rtol=2e-3), (la, lb)
    # six Adam steps of lr 1e-3 move an entry by <= 6e-3: where the fp32 atomics of the encoder backward land in another order, an entry
    # with a near-zero gradient can step the other way -- a few entries, never the bulk (the bound test_gpu_modules uses for the graph)
    assert float((ea - eb).abs().max()) < 7e-3 and float((ea - eb).abs().mean()) < 2e-5
    assert float((wa - wb).abs().max()) < 7e-3 and float((pa - pb).abs().max()) < 1e-3
    assert la[-1] < la[0]
