"""CPU tests of the host side of warm-up stream pools (koe_stream_pool_create_ex2 with KOE_POOL_WARMUP): the flags
word, the pool geometry, open / close, the refusal of push misuse before the argument block is read, the export and the
Python option -- none of which touches a device."""
import ctypes as C

import numpy as np
import pytest
import torch

WARMUP = 1  # KOE_POOL_WARMUP


@pytest.fixture
def lib():
    from koemorph_b200 import _lib
    return _lib.load()


@pytest.fixture(params=[1, 4], ids=["max_hops=1", "max_hops=4"])
def pool(lib, request):
    h = C.c_void_p()
    assert lib.koe_stream_pool_create_ex2(3, 533, 256, 512, request.param, WARMUP, C.byref(h)) == 0 and h.value
    yield h, request.param
    assert lib.koe_stream_pool_destroy(h) == 0


def test_create_ex2_is_exported(lib):
    from koemorph_b200 import _lib
    assert "koe_stream_pool_create_ex2" in _lib.exported_symbols()
    assert getattr(lib, "koe_stream_pool_create_ex2", None) is not None
    assert _lib.POOL_WARMUP == WARMUP


def test_create_ex2_flags_and_geometry(lib):
    h = C.c_void_p()
    for flags in (0, WARMUP):
        for hop, window in ((533, 256), (266, 512)):
            for max_hops in (1, 2, 30):
                assert lib.koe_stream_pool_create_ex2(4, hop, window, 512, max_hops, flags, C.byref(h)) == 0 and h.value
                assert lib.koe_stream_pool_destroy(h) == 0
    for flags in (2, 3, 1 << 8, -1, -(1 << 31)):
        h = C.c_void_p()
        assert lib.koe_stream_pool_create_ex2(4, 533, 256, 512, 1, flags, C.byref(h)) == -1
        assert h.value is None
    assert b"unknown flags" in lib.koe_last_error()
    # the geometry checks of koe_stream_pool_create_ex hold with the flag
    h = C.c_void_p()
    for max_hops in (0, -1):
        assert lib.koe_stream_pool_create_ex2(4, 533, 256, 512, max_hops, WARMUP, C.byref(h)) == -1
    assert lib.koe_stream_pool_create_ex2(1 << 20, 533, 256, 512, 16, WARMUP, C.byref(h)) == 0
    assert lib.koe_stream_pool_destroy(h) == 0
    h = C.c_void_p()
    assert lib.koe_stream_pool_create_ex2(1 << 20, 533, 256, 512, 17, WARMUP, C.byref(h)) == -1
    assert lib.koe_stream_pool_create_ex2(0, 533, 256, 512, 1, WARMUP, C.byref(h)) == -1
    assert lib.koe_stream_pool_create_ex2(4, 100, 256, 512, 1, WARMUP, C.byref(h)) == -1  # 6 edge frames per side
    assert lib.koe_stream_pool_create_ex2(4, 533, 0, 512, 1, WARMUP, C.byref(h)) == -1
    assert lib.koe_stream_pool_create_ex2(4, 533, 256, 512, 1, WARMUP, None) == -1
    assert h.value is None


def test_open_and_close_work_on_a_warmup_pool(lib, pool):
    h, _ = pool
    s = torch.full((3,), -7, dtype=torch.int32)
    assert lib.koe_stream_pool_open(h, 3, s.data_ptr()) == 0 and s.tolist() == [0, 1, 2]
    assert lib.koe_stream_pool_open(h, 1, s.data_ptr()) == -1           # full
    assert lib.koe_stream_pool_close(h, 1) == 0
    assert lib.koe_stream_pool_close(h, 1) == -1                         # not open
    assert lib.koe_stream_pool_open(h, 1, s.data_ptr()) == 0 and s[0].item() == 1


def test_push_misuse_is_refused_before_the_arguments_are_read(lib, pool):
    """On a warm-up pool both push entries run the burst path: slot and count checks come first, so with an empty
    argument block nothing else is looked at (and no device is needed)."""
    from koemorph_b200 import _lib
    h, max_hops = pool
    s = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(h, 2, s.data_ptr()) == 0
    args = _lib.StreamPoolArgs()
    emitted = torch.full((12,), -3, dtype=torch.int32)
    hops = torch.full((12,), -3, dtype=torch.int64)
    n = C.c_int(-5)
    for slots in ([2], [0, 0], [3], [-1], [0, 1, 2, 0]):
        t = torch.tensor(slots, dtype=torch.int32)
        assert lib.koe_stream_pool_push(h, C.byref(args), t.data_ptr(), len(slots), emitted.data_ptr(), C.byref(n),
                                        None) == -1, slots
        assert n.value == 0
        n.value = -5
        c = torch.ones(len(slots), dtype=torch.int32)
        assert lib.koe_stream_pool_push_hops(h, C.byref(args), t.data_ptr(), c.data_ptr(), len(slots), emitted.data_ptr(),
                                             hops.data_ptr(), C.byref(n), None) == -1, slots
        assert n.value == 0
        n.value = -5
    for counts in ([0], [max_hops + 1], [-1]):
        t = torch.tensor([0], dtype=torch.int32)
        c = torch.tensor(counts, dtype=torch.int32)
        assert lib.koe_stream_pool_push_hops(h, C.byref(args), t.data_ptr(), c.data_ptr(), 1, emitted.data_ptr(),
                                             hops.data_ptr(), C.byref(n), None) == -1, counts
        assert n.value == 0
    assert f"outside [1, {max_hops}]".encode() in lib.koe_last_error()
    # NULL outputs, and an empty call is a no-op
    t = torch.tensor([0], dtype=torch.int32)
    assert lib.koe_stream_pool_push(h, C.byref(args), t.data_ptr(), 1, None, C.byref(n), None) == -1
    assert lib.koe_stream_pool_push(h, C.byref(args), None, 0, emitted.data_ptr(), C.byref(n), None) == 0
    assert n.value == 0
    # with every slot right, the first thing looked at is the argument block itself: its NULL frontend is refused
    assert lib.koe_stream_pool_push(h, C.byref(args), t.data_ptr(), 1, emitted.data_ptr(), C.byref(n), None) == -1
    assert b"NULL frontend" in lib.koe_last_error()


@pytest.mark.parametrize("bad", [1, 0, None, "yes", 1.0, np.bool_(True), torch.tensor(True)])
def test_stream_pool_rejects_a_non_bool_warmup(bad):
    from koemorph_b200.streaming import StreamPool
    with pytest.raises(ValueError, match="warmup must be a bool"):
        StreamPool(None, 4, warmup=bad)      # (checked before the model is looked at)
