"""CPU tests of the host side of stream-pool snapshots (koe_stream_pool_state_floats / koe_stream_pool_snapshot /
koe_stream_pool_restore, StreamSnapshot): the record size, the refusal of misuse before the argument block is read, the
exports and the geometry checks of StreamPool.restore -- none of which touches a device."""
import ctypes as C
import io
import re

import pytest
import torch

HEADER = __import__("pathlib").Path(__file__).resolve().parents[1] / "include" / "koemorph_b200.h"
NEW = ("koe_stream_pool_state_floats", "koe_stream_pool_snapshot", "koe_stream_pool_restore")


@pytest.fixture
def lib():
    from koemorph_b200 import _lib
    return _lib.load()


def _create(lib, capacity, hop, window, max_hops, warmup):
    h = C.c_void_p()
    assert lib.koe_stream_pool_create_ex2(capacity, hop, window, 512, max_hops, 1 if warmup else 0, C.byref(h)) == 0
    return h


@pytest.fixture
def pool(lib):
    h = _create(lib, 3, 533, 256, 4, False)
    yield h
    assert lib.koe_stream_pool_destroy(h) == 0


def test_new_entry_points_are_exported_and_declared(lib):
    from koemorph_b200 import _lib
    header = HEADER.read_text()
    for name in NEW:
        assert name in _lib.exported_symbols()
        assert getattr(lib, name, None) is not None, name
        assert re.search(r"\bint " + name + r"\(", header), name
    assert lib.koe_version() >= 101


def _layout_floats(hop, window):
    n_edge = -(-512 // hop)
    P = window - n_edge                            # W - 1 - lag frames a later window can still read
    f = (1 + n_edge) * P * 80 + (1 + n_edge) * P + (512 + n_edge * hop) + 1 + 52
    return -(-f // 4) * 4


@pytest.mark.parametrize("fps,hop,window", [(30, 533, 256), (60, 266, 512)])
@pytest.mark.parametrize("max_hops", [1, 8])
@pytest.mark.parametrize("warmup", [False, True])
def test_state_floats_is_the_layout(lib, fps, hop, window, max_hops, warmup):
    h = _create(lib, 5, hop, window, max_hops, warmup)
    try:
        got = lib.koe_stream_pool_state_floats(h)
        assert got == _layout_floats(hop, window) and got % 4 == 0
        assert got == {30: 42408, 60: 125028}[fps]     # the sizes the header states
    finally:
        lib.koe_stream_pool_destroy(h)
    assert lib.koe_stream_pool_state_floats(None) == -1


def _snapshot(lib, pool, args, slots, records=1 << 20, hops=True):
    s = torch.tensor(slots, dtype=torch.int32)
    h = torch.full((max(1, len(slots)),), -9, dtype=torch.int64)
    rc = lib.koe_stream_pool_snapshot(pool, C.byref(args), s.data_ptr(), len(slots), records,
                                      h.data_ptr() if hops else None, None)
    return rc, h


def _restore(lib, pool, args, hops, records=1 << 20, slots_out=True, n=None):
    h = torch.tensor(hops, dtype=torch.int64)
    s = torch.full((max(1, len(hops)),), -9, dtype=torch.int32)
    rc = lib.koe_stream_pool_restore(pool, C.byref(args), records, h.data_ptr() if len(hops) else None,
                                     len(hops) if n is None else n, s.data_ptr() if slots_out else None, None)
    return rc, s


def _free_slots(lib, pool, capacity):
    """The pool's free slots, found by opening them all (and closing them again)."""
    s = torch.empty(capacity, dtype=torch.int32)
    for k in range(capacity, -1, -1):
        if lib.koe_stream_pool_open(pool, k, s.data_ptr()) == 0:
            free = s[:k].tolist()
            for x in free:
                assert lib.koe_stream_pool_close(pool, x) == 0
            return free
    raise AssertionError("unreachable")


def test_snapshot_misuse_is_refused_before_the_arguments_are_read(lib, pool):
    """Slot checks and NULL outputs come first: with an empty argument block (NULL rings) nothing else is looked at, and
    the hops output is not written."""
    from koemorph_b200 import _lib
    s = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 2, s.data_ptr()) == 0     # slots 0, 1 open; 2 closed
    args = _lib.StreamPoolArgs()
    for slots in ([2], [0, 0], [3], [-1], [1, 0, 1]):
        rc, h = _snapshot(lib, pool, args, slots)
        assert rc == -1, slots
        assert (h == -9).all()
    assert b"listed twice" in (_snapshot(lib, pool, args, [0, 0])[0] == -1 and lib.koe_last_error())
    assert _snapshot(lib, pool, args, [0], records=0)[0] == -1                  # NULL records
    assert _snapshot(lib, pool, args, [0], hops=False)[0] == -1                 # NULL hops
    assert _snapshot(lib, pool, args, [0], records=(1 << 20) + 4)[0] == -1      # not 16-byte aligned
    assert _snapshot(lib, pool, args, [0, 1])[0] == -1                          # NULL rings
    assert b"NULL buffer" in lib.koe_last_error()
    assert lib.koe_stream_pool_snapshot(pool, None, s.data_ptr(), 1, 1 << 20, s.data_ptr(), None) == -1
    # an empty call is a no-op
    assert lib.koe_stream_pool_snapshot(pool, C.byref(args), None, 0, None, None, None) == 0
    # nothing moved: the same slots are open
    assert _free_slots(lib, pool, 3) == [2]


def test_restore_misuse_is_refused_before_the_arguments_are_read(lib, pool):
    """Free-slot, hops and NULL checks come first; a refused restore opens no slot and writes no slot output."""
    from koemorph_b200 import _lib
    s = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool, 1, s.data_ptr()) == 0     # slot 0 open; 1, 2 free
    args = _lib.StreamPoolArgs()
    for hops in ([5, 6, 7], [0, 0, 0, 0]):                        # more records than free slots
        rc, out = _restore(lib, pool, args, hops)
        assert rc == -1 and (out == -9).all(), hops
    assert b"2 of 3 slots free" in lib.koe_last_error()
    rc, out = _restore(lib, pool, args, [3, -1])                   # a negative hops
    assert rc == -1 and (out == -9).all()
    assert b"-1 hops" in lib.koe_last_error()
    assert _restore(lib, pool, args, [3], records=0)[0] == -1      # NULL records
    assert _restore(lib, pool, args, [3], slots_out=False)[0] == -1
    assert lib.koe_stream_pool_restore(pool, C.byref(args), 1 << 20, None, 1, s.data_ptr(), None) == -1
    assert _restore(lib, pool, args, [3], records=(1 << 20) + 8)[0] == -1
    assert _restore(lib, pool, args, [3, 4])[0] == -1               # NULL rings
    assert b"NULL buffer" in lib.koe_last_error()
    assert _restore(lib, pool, args, [], n=-1)[0] == -1
    assert lib.koe_stream_pool_restore(pool, None, 1 << 20, s.data_ptr(), 1, s.data_ptr(), None) == -1
    # an empty call is a no-op
    assert lib.koe_stream_pool_restore(pool, C.byref(args), None, None, 0, None, None) == 0
    # no slot was taken
    assert _free_slots(lib, pool, 3) == [1, 2]


def _cpu_pool(hop=533, window=256, warmup=False, max_hops=1):
    from koemorph_b200.streaming import StreamPool
    p = StreamPool.__new__(StreamPool)
    p.hop, p.W, p.half, p.warmup, p.max_hops = hop, window, 512, warmup, max_hops
    p.dev = torch.device("cpu")                   # (records are checked against the pool's device)
    p.state_floats = _layout_floats(hop, window)
    p._h = None
    return p


def _snap(hop=533, window=256, half=512, warmup=False, k=2, floats=None, dtype=torch.float32, hops_dtype=torch.int64):
    from koemorph_b200.streaming import StreamSnapshot
    floats = _layout_floats(hop, window) if floats is None else floats
    return StreamSnapshot(hop, window, half, warmup, torch.arange(k, dtype=hops_dtype), torch.zeros(k, floats, dtype=dtype))


def test_restore_checks_the_snapshot_before_any_native_call():
    p = _cpu_pool()
    r, h = p._check_snapshot(_snap())
    assert r.shape == (2, p.state_floats) and h.tolist() == [0, 1]
    bad = [
        _snap(hop=266, window=256),                 # another hop
        _snap(window=512),                          # another window
        _snap(half=256),                            # another FFT size
        _snap(warmup=True),                         # a warm-up pool's streams
        _snap(floats=_layout_floats(533, 256) - 4),
        _snap(dtype=torch.float64),
        _snap(hops_dtype=torch.int32),
    ]
    for s in bad:
        with pytest.raises(ValueError):
            p.restore(s)                            # (p has no native pool: it must fail before any native call)
    s = _snap()
    s.hops[1] = -3
    with pytest.raises(ValueError):
        p.restore(s)
    s = _snap()
    s.records = s.records[:1]
    with pytest.raises(ValueError, match="records must be"):
        p.restore(s)
    with pytest.raises(ValueError):
        p.restore((s.hops, s.records))
    with pytest.raises(ValueError, match="warmup"):
        _cpu_pool(warmup=True).restore(_snap())


def test_snapshot_to_and_torch_save_round_trip():
    from koemorph_b200.streaming import StreamSnapshot
    s = _snap(k=3)
    s.records.normal_()
    t = s.to("cpu")
    assert t is not s and t.records.data_ptr() != s.records.data_ptr() and torch.equal(t.records, s.records)
    buf = io.BytesIO()
    torch.save(t, buf)
    buf.seek(0)
    u = torch.load(buf)                             # (the default, weights-only loader)
    assert isinstance(u, StreamSnapshot) and len(u) == 3
    assert (u.hop, u.window_frames, u.half_fft, u.warmup) == (533, 256, 512, False)
    assert torch.equal(u.hops, s.hops) and torch.equal(u.records, s.records)
    assert u.hops.dtype == torch.int64 and u.records.dtype == torch.float32
