"""CPU tests of the stream pool's host side: the ctypes mirror of koe_stream_pool_args and the slot bookkeeping of the
native pool object (open / close / misuse), none of which touches a device."""
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
    assert lib.koe_stream_pool_create(3, 533, 256, 512, C.byref(h)) == 0 and h.value
    yield h
    assert lib.koe_stream_pool_destroy(h) == 0


def test_pool_args_mirror_has_the_size_of_the_c_struct(lib):
    from koemorph_b200 import _lib
    assert lib.koe_sizeof_struct(5) == C.sizeof(_lib.StreamPoolArgs)
    assert lib.koe_sizeof_struct(99) == -1


def test_create_rejects_bad_geometry(lib):
    h = C.c_void_p()
    assert lib.koe_stream_pool_create(0, 533, 256, 512, C.byref(h)) == -1
    assert lib.koe_stream_pool_create(4, 100, 256, 512, C.byref(h)) == -1   # 6 edge frames per window side
    assert lib.koe_stream_pool_create(4, 533, 0, 512, C.byref(h)) == -1
    assert h.value is None


def test_open_takes_the_lowest_free_slots_and_close_frees_them(lib, pool):
    s = torch.full((3,), -7, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == 0 and s[:2].tolist() == [0, 1]
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == -1              # one slot free
    assert b"1 of 3 slots free" in lib.koe_last_error()
    assert lib.koe_stream_pool_close(pool, 0) == 0
    assert lib.koe_stream_pool_close(pool, 0) == -1                          # not open any more
    assert lib.koe_stream_pool_close(pool, 3) == -1 and lib.koe_stream_pool_close(pool, -1) == -1
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == 0 and s[:2].tolist() == [0, 2]


def test_push_misuse_is_refused_before_the_arguments_are_read(lib, pool):
    """Slot checks come first: with an empty argument block nothing else is looked at (and no device is needed)."""
    from koemorph_b200 import _lib
    s = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == 0
    args = _lib.StreamPoolArgs()
    emitted = torch.empty(3, dtype=torch.int32)
    n = C.c_int(-5)
    for slots in ([2], [0, 0], [3], [-1], [0, 1, 2, 0]):
        t = torch.tensor(slots, dtype=torch.int32)
        assert lib.koe_stream_pool_push(pool, C.byref(args), t.data_ptr(), len(slots), emitted.data_ptr(), C.byref(n),
                                        None) == -1, slots
        assert n.value == 0
        assert lib.koe_stream_pool_set_egemaps(pool, C.byref(args), t.data_ptr(), len(slots), None, None) == -1, slots
    # an empty push is a no-op
    assert lib.koe_stream_pool_push(pool, C.byref(args), None, 0, emitted.data_ptr(), C.byref(n), None) == 0
