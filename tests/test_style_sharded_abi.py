"""CPU tier: argument validation of the fp32 sharded exchange (`lnrf_adam_step_sharded_f32`) fails loudly before anything touches a
device -- world size, rank, peer pointers and the learning-rate segment table."""
import ctypes as C
import os

import pytest

HYPER = (1e-3, 0.9, 0.999, 1e-8, 0.0)
FAKE = 1 << 20   # a 16-byte-aligned address that is never dereferenced: every call below fails validation first


@pytest.fixture(scope="module")
def lib():
    from laenerf_b200 import _native as N
    if not os.path.exists(N.SO_PATH):
        N.build()
    return N.lib()


def _call(lib, world=1, rank=0, starts=(0,), mults=(1.0,), peer=FAKE, n=64):
    ptrs = (C.c_void_p * 8)(*([peer] * 8))
    p = C.cast(ptrs, C.c_void_p)
    return lib.lnrf_adam_step_sharded_f32(p, p, p, world, rank, 0, n, (C.c_uint64 * len(starts))(*starts), (C.c_double * len(mults))(*mults),
                                          len(starts), FAKE, FAKE, *HYPER, None, FAKE, FAKE, None, None)


def test_world_and_rank_are_checked(lib):
    assert _call(lib, world=0) != 0 and b"ranks" in lib.lnrf_last_error()
    assert _call(lib, world=9) != 0 and b"ranks" in lib.lnrf_last_error()
    assert _call(lib, world=2, rank=2) != 0 and b"rank 2" in lib.lnrf_last_error()


def test_null_peers_are_rejected(lib):
    assert _call(lib, peer=None) != 0 and b"null peer" in lib.lnrf_last_error()


def test_segment_table_is_checked(lib):
    assert _call(lib, starts=(0, 16, 8), mults=(1.0, 1.0, 2.0)) != 0 and b"ascend" in lib.lnrf_last_error()
    assert _call(lib, starts=(8,)) != 0 and b"ascend" in lib.lnrf_last_error()
    assert _call(lib, starts=(0, 12), mults=(1.0, 2.0)) != 0 and b"multiple of 8" in lib.lnrf_last_error()
    assert _call(lib, starts=tuple(range(0, 72, 8)), mults=(1.0,) * 9) != 0 and b"segments" in lib.lnrf_last_error()
    assert _call(lib, starts=(0, 8), mults=(1.0, -1.0)) != 0 and b"multiplier" in lib.lnrf_last_error()


def test_slice_must_be_whole_vectors(lib):
    assert _call(lib, n=60) != 0 and b"multiples of 8" in lib.lnrf_last_error()
