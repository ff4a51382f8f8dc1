"""CPU tier of the deterministic hash-grid backward (torch.use_deterministic_algorithms): the fixed-point quantum rule cannot
wrap an int64 sum, integer sums of quantised flushes do not depend on their order and stay within the stated bound, the finish
rule's NaN / overflow handling, and argument validation of the new entry points (which fails before any device access)."""
import ctypes as C
import os

import numpy as np
import pytest

FAKE = 1 << 20   # a 16-byte-aligned address that is never dereferenced: every call below fails validation first


def qexp(B, E):
    """q = 2^qexp, qexp = E + ceil(log2 B) + 1 - 62 (gridenc.cu det_qexp; 2^E >= max |g|)."""
    lb = int(np.ceil(np.log2(B))) if B > 1 else 0
    return E + lb + 1 - 62


def quantise(p, qe):
    """round(p / q) to nearest even, as __float2ll_rn(p * 2^-qe) -- exact for a power-of-two q."""
    return np.rint(np.ldexp(np.asarray(p, np.float64), -qe)).astype(np.int64)


def finish(base, acc, flag, qe, dtype):
    """k_det_finish: RN_T(base + acc * q), NaN where flagged."""
    v = base.astype(np.float64) + np.ldexp(acc.astype(np.float64), qe)
    with np.errstate(over="ignore"):
        out = v.astype(dtype)
    return np.where(flag, np.array(np.nan, dtype), out)


@pytest.mark.parametrize("B", [1, 2, 1000, 268_288, 1 << 24, (1 << 31) - 1])
@pytest.mark.parametrize("E", [16, 0, -20, 40])
def test_quantum_rule_cannot_wrap(B, E):
    """Worst case: every sample puts its whole weight (sum 1 per level) on one entry with |g| at the bound 2^E."""
    qe = qexp(B, E)
    worst = B * 2.0 ** E * (1 + 2.0 ** -20)   # corner weights are fp32 products: their sum is 1 within a few ulp
    per_flush = quantise(2.0 ** E * (1 + 2.0 ** -20), qe)
    assert worst < 2.0 ** 62 * 2.0 ** qe
    assert int(per_flush) * B < 2 ** 63


def test_lego_quantum_is_finer_than_fp16_subnormals():
    assert qexp(268_288, 16) == -26 and 2.0 ** -26 < 2.0 ** -24


def test_quantised_sums_are_order_independent_and_bounded():
    rng = np.random.default_rng(0)
    B = 4096
    qe = qexp(B, 16)
    flushes = (rng.standard_normal(B) * rng.choice([1e-6, 1e-2, 1.0, 30.0], B)).astype(np.float32)
    exact = float(np.sum(flushes.astype(np.float64)))
    results = set()
    for _ in range(8):
        perm = rng.permutation(B)
        acc = np.int64(0)
        for v in quantise(flushes[perm], qe):
            acc += v
        results.add(int(acc))
    assert len(results) == 1
    acc = np.array([results.pop()])
    for dtype in (np.float16, np.float32):
        r = finish(np.zeros(1, dtype), acc, np.zeros(1, bool), qe, dtype)[0]
        ulp = float(np.spacing(np.abs(np.array(r, dtype))))
        assert abs(float(r) - exact) <= B * 2.0 ** qe / 2 + ulp / 2 + 2.0 ** -50 * abs(exact), dtype


def test_finish_rule_nan_and_overflow():
    qe = qexp(1000, 16)
    q = 2.0 ** qe
    acc = np.array([int(70000 / q), int(-70000 / q), int(65000 / q), 0, int(1.5 / q)])
    flag = np.array([False, False, False, True, False])
    r = finish(np.zeros(5, np.float16), acc, flag, qe, np.float16)
    assert r[0] == np.inf and r[1] == -np.inf and np.isfinite(r[2]) and np.isnan(r[3]) and r[4] == np.float16(1.5)
    r = finish(np.full(5, np.float16(65000)), acc, np.zeros(5, bool), qe, np.float16)
    assert r[2] == np.inf and r[1] == np.float16(float(np.float16(65000)) - 70000)


@pytest.fixture(scope="module")
def lib():
    from laenerf_b200 import _native as N
    if not os.path.exists(N.SO_PATH):
        N.build()
    return N.lib()


OFFS = (C.c_int32 * 3)(0, 64, 128)


def test_backward_det_arguments_are_checked(lib):
    f = lib.lnrf_grid_encode_backward_det
    assert f(FAKE, FAKE, OFFS, None, FAKE, None, 16, 3, 2, 2, 1.0, 4, None, None, 0, 0, 0, 1, 1, None) != 0
    assert b"acc / flags is null" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, OFFS, FAKE, FAKE, None, 16, 3, 2, 2, 1.0, 4, None, None, 0, 0, 0, 0, 1, None) != 0
    assert b"gmax" in lib.lnrf_last_error()                              # fp32 without the max word
    assert f(FAKE, FAKE, OFFS, FAKE + 8, FAKE, None, 16, 3, 2, 2, 1.0, 4, None, None, 0, 0, 0, 1, 1, None) != 0
    assert b"aligned" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, OFFS, FAKE, FAKE, None, 16, 3, 3, 2, 1.0, 4, None, None, 0, 0, 0, 1, 1, None) != 0
    assert b"C must be" in lib.lnrf_last_error()
    assert f(None, FAKE, OFFS, FAKE, FAKE, None, 16, 3, 2, 2, 1.0, 4, None, None, 0, 0, 0, 1, 1, None) != 0
    assert b"null pointer" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, OFFS, FAKE, FAKE, None, 16, 3, 2, 2, 1.0, 4, None, None, 0, 0, 0, 7, 1, None) != 0
    assert b"dtype" in lib.lnrf_last_error()


def test_backward_world_det_arguments_are_checked(lib):
    f = lib.lnrf_grid_encode_backward_world_det
    assert f(FAKE, FAKE, 0.0, OFFS, FAKE, FAKE, None, 16, None, 2, 1.0, 4, 0, 0, 0, 1, None) != 0
    assert b"bound" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, 1.0, OFFS, FAKE, None, None, 16, None, 2, 1.0, 4, 0, 0, 0, 1, None) != 0
    assert b"acc / flags" in lib.lnrf_last_error()


def test_finish_arguments_are_checked(lib):
    f = lib.lnrf_grid_det_finish
    assert f(FAKE, FAKE, None, 16, FAKE, 64, 3, 1, None) != 0 and b"C must be" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, None, 16, None, 64, 2, 1, None) != 0 and b"null" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, None, 16, FAKE, 64, 2, 0, None) != 0 and b"gmax" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, None, 0, FAKE, 64, 2, 1, None) != 0 and b"B must be" in lib.lnrf_last_error()


def test_occupancy_scatter_det_arguments_are_checked(lib):
    f = lib.lnrf_occupancy_scatter_det
    assert f(FAKE, FAKE, 16, FAKE, None, 64, None) != 0 and b"null pointer" in lib.lnrf_last_error()
    assert f(FAKE, FAKE, 16, FAKE, FAKE, 0, None) != 0 and b"cells" in lib.lnrf_last_error()
    assert f(None, None, 0, None, None, 0, None) == 0   # nothing to do


def test_ffmlp_backward_deterministic_predicate(lib):
    assert lib.lnrf_ffmlp_backward_deterministic(32, 16, 64, 2, 0, 6) == 1    # LAENeRF's sigma net / weight_net
    assert lib.lnrf_ffmlp_backward_deterministic(32, 16, 64, 3, 0, 6) == 1    # colour net
    assert lib.lnrf_ffmlp_backward_deterministic(48, 16, 64, 2, 0, 6) == 1    # offset_net
    assert lib.lnrf_ffmlp_backward_deterministic(32, 16, 64, 2, 3, 6) == 0    # sigmoid: the float-atomics kernel
    assert lib.lnrf_ffmlp_backward_deterministic(32, 16, 48, 2, 0, 6) < 0     # a shape lnrf_ffmlp_backward rejects
