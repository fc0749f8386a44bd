"""CPU tests of the host side of packed warm-up batches (koe_forward_varlen_ex / koe_forward_varlen_size_ex with
KOE_VARLEN_WARMUP): the exports, flags 0 as the plain entries, the row count against a Python count of grid hops, the
refusal of unknown flags and of clips without a grid hop before any buffer is read, and the Python option -- none of
which touches a device."""
import ctypes as C

import numpy as np
import pytest
import torch

WARMUP = 1  # KOE_VARLEN_WARMUP
HOP = {30: 533, 60: 266}
WIN = {30: 256, 60: 512}


@pytest.fixture
def lib():
    from koemorph_b200 import _lib
    return _lib.load()


def _args(lengths, fps=30, stride=1):
    from koemorph_b200 import _lib
    lens = torch.tensor(lengths, dtype=torch.int64)
    a = _lib.ForwardVarlenArgs()
    a.lengths_host, a.n_clips = lens.data_ptr(), len(lengths)
    a.hop, a.window_frames, a.stride_frames, a.half_fft = HOP[fps], WIN[fps], stride, 512
    return a, lens


def _size_ex(lib, a, flags):
    n_win, n_frames, ws = C.c_int64(-1), C.c_int64(-1), C.c_int64(-1)
    rc = lib.koe_forward_varlen_size_ex(C.byref(a), flags, C.byref(n_win), C.byref(n_frames), C.byref(ws))
    return rc, n_win.value, n_frames.value, ws.value


def _size(lib, a):
    n_win, n_frames, ws = C.c_int64(-1), C.c_int64(-1), C.c_int64(-1)
    rc = lib.koe_forward_varlen_size(C.byref(a), C.byref(n_win), C.byref(n_frames), C.byref(ws))
    return rc, n_win.value, n_frames.value, ws.value


def _grid_rows(L, fps, stride):
    """Rows of one clip, counted hop by hop: the hops h = W - 1 (mod stride), h >= 0, that the clip completes."""
    W, n = WIN[fps], L // HOP[fps]
    return sum(1 for h in range(n) if (h - (W - 1)) % stride == 0)


def _lengths(fps):
    hop, W = HOP[fps], WIN[fps]
    return [hop, hop + 1, (W - 1) * hop, W * hop - 1, W * hop, W * hop + hop - 1, (W + 1) * hop, 60 * 16000]


def test_warmup_entries_are_exported(lib):
    from koemorph_b200 import _lib
    for name in ("koe_forward_varlen_ex", "koe_forward_varlen_size_ex"):
        assert name in _lib.exported_symbols()
        assert getattr(lib, name, None) is not None
    assert _lib.VARLEN_WARMUP == WARMUP
    assert lib.koe_sizeof_struct(6) == C.sizeof(_lib.ForwardVarlenArgs)


@pytest.mark.parametrize("fps,stride", [(30, 1), (30, 3), (60, 1), (60, 2)])
def test_flags_zero_is_the_plain_sizing(lib, fps, stride):
    """The length sets of the plain sizing test: flags 0 gives exactly koe_forward_varlen_size's answer."""
    hop, W = HOP[fps], WIN[fps]
    lengths = [0, 1, 511, 512, 1024, W * hop - 1, W * hop, W * hop + 1, (W + 1) * hop, (W + 1) * hop + 5,
               (W + 31) * hop, (W + 32) * hop - 1, (W + 64) * stride * hop, 60 * 16000]
    for i in range(len(lengths)):
        sub = lengths[i:] + lengths[:i][:3]
        a, _ = _args(sub, fps, stride)
        plain = _size(lib, a)
        assert plain[0] == 0, lib.koe_last_error()
        assert _size_ex(lib, a, 0) == plain
    a, _ = _args([])
    assert _size_ex(lib, a, 0) == _size(lib, a) == (0, 0, 0, _size(lib, a)[3])


@pytest.mark.parametrize("fps,stride", [(30, 1), (30, 2), (30, 3), (60, 1), (60, 2), (60, 3)])
def test_warmup_rows_are_the_grid_hops(lib, fps, stride):
    """With KOE_VARLEN_WARMUP the row count is one per grid hop each clip completes, the global frames are the plain
    call's, and the workspace grows by the lead rows of the n_edge window-end buffers only."""
    from koemorph_b200.model.sequential_dual_stream_model import SequentialDualStreamModel
    m = SequentialDualStreamModel.__new__(SequentialDualStreamModel)
    m.hop_length, m.window_frames, m.stride_frames = HOP[fps], WIN[fps], stride
    hop, W = HOP[fps], WIN[fps]
    r = (W - 1) % stride
    lengths = [L for L in _lengths(fps) if L >= (r + 1) * hop]
    n_edge = -(-512 // hop)
    for i in range(len(lengths)):
        sub = lengths[i:] + lengths[:i][:2]
        a, lens = _args(sub, fps, stride)
        rc, rows, n_frames, ws = _size_ex(lib, a, WARMUP)
        assert rc == 0, lib.koe_last_error()
        want = [_grid_rows(L, fps, stride) for L in sub]
        assert rows == sum(want)
        assert m.varlen_rows(lens, warmup=True).tolist() == want
        plain = _size(lib, a)
        assert n_frames == plain[2]
        leads = sum(sum(1 for h in range(L // hop) if h <= W - 2 and (h - (W - 1)) % stride == 0) for L in sub)
        assert plain[3] + n_edge * leads * 81 * 4 <= ws <= plain[3] + n_edge * leads * 81 * 4 + 16 * (4 * n_edge + 1) + \
            4 * (3 * len(sub) + 3)


def test_warmup_rows_of_a_short_batch(lib):
    """Every clip shorter than one window: no padded window, only lead rows (one per hop at stride 1)."""
    a, _ = _args([533, 16000, 136000 - 1])
    rc, rows, n_frames, _ = _size_ex(lib, a, WARMUP)
    assert rc == 0 and rows == 1 + 16000 // 533 + 255 and n_frames == 3 * 257


@pytest.mark.parametrize("fps,stride", [(30, 1), (30, 3), (60, 2)])
def test_a_clip_without_a_grid_hop_is_refused(lib, fps, stride):
    hop, W = HOP[fps], WIN[fps]
    r = (W - 1) % stride
    for short in (0, hop - 1, (r + 1) * hop - 1):
        a, _ = _args([60 * 16000, short, hop * (r + 1)], fps, stride)
        assert _size_ex(lib, a, WARMUP)[0] == -1
        assert b"completes no hop of the output grid" in lib.koe_last_error()
        assert _size_ex(lib, a, 0)[0] == 0                 # the plain call gives it its padded window
        # refused before any buffer (all NULL here) or the frontend / weights are looked at
        assert lib.koe_forward_varlen_ex(C.byref(a), WARMUP, None) == -1
        assert b"completes no hop of the output grid" in lib.koe_last_error()


def test_unknown_flags_are_refused(lib):
    a, _ = _args([16000, 160000])
    for flags in (2, 3, 1 << 8, -1, -(1 << 31)):
        assert _size_ex(lib, a, flags)[0] == -1
        assert b"unknown flags" in lib.koe_last_error()
        assert lib.koe_forward_varlen_ex(C.byref(a), flags, None) == -1
        assert b"unknown flags" in lib.koe_last_error()
    a, _ = _args([])
    assert lib.koe_forward_varlen_ex(C.byref(a), 2, None) == -1
    assert lib.koe_forward_varlen_ex(C.byref(a), WARMUP, None) == 0   # an empty batch is a no-op


def test_warmup_sizing_keeps_the_plain_checks(lib):
    for lengths in ([5000, -1], [1 << 30]):
        a, _ = _args(lengths)
        assert _size_ex(lib, a, WARMUP)[0] == -1
        assert b"outside [0, 2^30)" in lib.koe_last_error()
    a, _ = _args([16000])
    a.hop = 100                                        # 6 edge frames per window side
    assert _size_ex(lib, a, WARMUP)[0] == -1
    n_win = C.c_int64()
    a, _ = _args([16000])
    assert lib.koe_forward_varlen_size_ex(C.byref(a), WARMUP, C.byref(n_win), None, None) == -1


@pytest.mark.parametrize("bad", [1, 0, None, "yes", 1.0, np.bool_(True), torch.tensor(True)])
def test_forward_varlen_rejects_a_non_bool_warmup(bad):
    from koemorph_b200.model.sequential_dual_stream_model import SequentialDualStreamModel
    m = SequentialDualStreamModel.__new__(SequentialDualStreamModel)
    with pytest.raises(ValueError, match="warmup must be a bool"):
        m.forward_varlen(None, [1], warmup=bad)      # (checked before anything else is looked at)


def test_python_refuses_a_clip_without_a_grid_hop():
    from koemorph_b200.model.sequential_dual_stream_model import SequentialDualStreamModel
    m = SequentialDualStreamModel.__new__(SequentialDualStreamModel)
    m.hop_length, m.window_frames, m.stride_frames = 533, 256, 3      # r = 0
    lens = torch.tensor([16000, 532], dtype=torch.int64)
    with pytest.raises(ValueError, match="clip 1 of 532 samples completes no hop"):
        m.varlen_rows(lens, warmup=True)
    assert m.varlen_rows(lens).tolist() == [1, 1]
    m.hop_length, m.window_frames, m.stride_frames = 266, 512, 2      # r = 1: two hops
    with pytest.raises(ValueError, match="clip 0"):
        m.varlen_rows(torch.tensor([2 * 266 - 1]), warmup=True)
    assert m.varlen_rows(torch.tensor([2 * 266]), warmup=True).tolist() == [1]
