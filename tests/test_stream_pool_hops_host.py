"""CPU tests of the host side of stream-pool bursts (koe_stream_pool_create_ex / koe_stream_pool_push_hops): the pool
geometry, the refusal of misuse before the argument block is read, and the exports -- none of which touches a device."""
import ctypes as C

import pytest
import torch


@pytest.fixture
def lib():
    from koemorph_b200 import _lib
    return _lib.load()


@pytest.fixture
def pool(lib):
    h = C.c_void_p()
    assert lib.koe_stream_pool_create_ex(3, 533, 256, 512, 4, C.byref(h)) == 0 and h.value
    yield h
    assert lib.koe_stream_pool_destroy(h) == 0


def test_new_entry_points_are_exported(lib):
    from koemorph_b200 import _lib
    for name in ("koe_stream_pool_create_ex", "koe_stream_pool_push_hops"):
        assert name in _lib.exported_symbols()
        assert getattr(lib, name, None) is not None, name


def test_create_ex_geometry(lib):
    h = C.c_void_p()
    for max_hops in (1, 2, 30):
        assert lib.koe_stream_pool_create_ex(4, 533, 256, 512, max_hops, C.byref(h)) == 0 and h.value
        assert lib.koe_stream_pool_destroy(h) == 0
    for max_hops in (0, -1, -(1 << 31)):
        h = C.c_void_p()
        assert lib.koe_stream_pool_create_ex(4, 533, 256, 512, max_hops, C.byref(h)) == -1
        assert h.value is None
    assert b"max_hops" in lib.koe_last_error()
    # capacity * max_hops is bounded like the capacity itself
    assert lib.koe_stream_pool_create_ex(1 << 20, 533, 256, 512, 16, C.byref(h)) == 0
    assert lib.koe_stream_pool_destroy(h) == 0
    h = C.c_void_p()
    assert lib.koe_stream_pool_create_ex(1 << 20, 533, 256, 512, 17, C.byref(h)) == -1 and h.value is None
    # the geometry checks of koe_stream_pool_create hold for every max_hops
    assert lib.koe_stream_pool_create_ex(0, 533, 256, 512, 2, C.byref(h)) == -1
    assert lib.koe_stream_pool_create_ex(4, 100, 256, 512, 2, C.byref(h)) == -1   # 6 edge frames per window side
    assert lib.koe_stream_pool_create_ex(4, 533, 0, 512, 2, C.byref(h)) == -1
    assert lib.koe_stream_pool_create_ex(4, 533, 256, 512, 2, None) == -1
    assert h.value is None


def test_open_and_close_work_on_a_burst_pool(lib, pool):
    s = torch.full((3,), -7, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 3, s.data_ptr()) == 0 and s.tolist() == [0, 1, 2]
    assert lib.koe_stream_pool_close(pool, 1) == 0
    assert lib.koe_stream_pool_open(pool, 1, s.data_ptr()) == 0 and s[0].item() == 1


def _push_hops(lib, pool, args, slots, counts):
    s = torch.tensor(slots, dtype=torch.int32)
    c = torch.tensor(counts, dtype=torch.int32)
    emitted = torch.full((12,), -3, dtype=torch.int32)
    hops = torch.full((12,), -3, dtype=torch.int64)
    n = C.c_int(-5)
    rc = lib.koe_stream_pool_push_hops(pool, C.byref(args), s.data_ptr(), c.data_ptr(), len(slots), emitted.data_ptr(),
                                       hops.data_ptr(), C.byref(n), None)
    return rc, n.value


def test_push_hops_misuse_is_refused_before_the_arguments_are_read(lib, pool):
    """Slot and count checks come first: with an empty argument block nothing else is looked at (and no device is
    needed)."""
    from koemorph_b200 import _lib
    s = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == 0
    args = _lib.StreamPoolArgs()
    cases = [
        ([2], [1]),             # closed
        ([0, 0], [1, 1]),       # listed twice
        ([3], [1]), ([-1], [1]),  # out of range
        ([0], [0]),             # count 0
        ([0], [5]),             # count > max_hops
        ([0, 1], [2, -1]),      # a negative count
        ([0, 1, 2, 0], [1, 1, 1, 1]),
    ]
    for slots, counts in cases:
        rc, n = _push_hops(lib, pool, args, slots, counts)
        assert rc == -1, (slots, counts)
        assert n == 0
    _push_hops(lib, pool, args, [0], [5])
    assert b"count 5 for slot 0 outside [1, 4]" in lib.koe_last_error()
    # NULL counts and NULL outputs
    t = torch.tensor([0], dtype=torch.int32)
    emitted = torch.empty(4, dtype=torch.int32)
    hops = torch.empty(4, dtype=torch.int64)
    n = C.c_int(0)
    assert lib.koe_stream_pool_push_hops(pool, C.byref(args), t.data_ptr(), None, 1, emitted.data_ptr(), hops.data_ptr(),
                                         C.byref(n), None) == -1
    c = torch.tensor([1], dtype=torch.int32)
    assert lib.koe_stream_pool_push_hops(pool, C.byref(args), t.data_ptr(), c.data_ptr(), 1, emitted.data_ptr(), None,
                                         C.byref(n), None) == -1
    # an empty call is a no-op
    assert lib.koe_stream_pool_push_hops(pool, C.byref(args), None, None, 0, emitted.data_ptr(), hops.data_ptr(),
                                         C.byref(n), None) == 0
    assert n.value == 0


def test_push_on_a_burst_pool_refuses_misuse_like_push_hops(lib, pool):
    """koe_stream_pool_push on a pool with max_hops > 1 runs the burst path with counts of 1; its slot checks are the
    same."""
    from koemorph_b200 import _lib
    s = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == 0
    args = _lib.StreamPoolArgs()
    emitted = torch.empty(3, dtype=torch.int32)
    n = C.c_int(-5)
    for slots in ([2], [0, 0], [3], [-1]):
        t = torch.tensor(slots, dtype=torch.int32)
        assert lib.koe_stream_pool_push(pool, C.byref(args), t.data_ptr(), len(slots), emitted.data_ptr(), C.byref(n),
                                        None) == -1, slots
        assert n.value == 0
    assert lib.koe_stream_pool_push(pool, C.byref(args), None, 0, emitted.data_ptr(), C.byref(n), None) == 0
