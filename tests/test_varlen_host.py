"""CPU tests of the packed variable-length forward's host side: the ctypes mirror of koe_forward_varlen_args, the sizing
entry (the library's per-clip geometry against SequentialDualStreamModel.num_output_frames) and its validation, none of
which touches a device."""
import ctypes as C

import pytest
import torch

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


def _size(lib, a):
    n_win, n_frames, ws = C.c_int64(-1), C.c_int64(-1), C.c_int64(-1)
    rc = lib.koe_forward_varlen_size(C.byref(a), C.byref(n_win), C.byref(n_frames), C.byref(ws))
    return rc, n_win.value, n_frames.value, ws.value


def test_varlen_args_mirror_has_the_size_of_the_c_struct(lib):
    from koemorph_b200 import _lib
    assert lib.koe_sizeof_struct(6) == C.sizeof(_lib.ForwardVarlenArgs)


def test_varlen_symbols_are_exported():
    from koemorph_b200 import _lib
    names = _lib.exported_symbols()
    assert "koe_forward_varlen" in names and "koe_forward_varlen_size" in names


@pytest.mark.parametrize("fps,stride", [(30, 1), (30, 3), (60, 1), (60, 2)])
def test_sizing_agrees_with_num_output_frames(lib, fps, stride):
    """Total windows and frames for a sweep of lengths around every rule of the per-clip geometry, and a workspace that
    holds the mel rows of the plain frames and of every edge variant."""
    from koemorph_b200.model.sequential_dual_stream_model import SequentialDualStreamModel
    m = SequentialDualStreamModel.__new__(SequentialDualStreamModel)
    m.hop_length, m.window_frames, m.stride_frames = HOP[fps], WIN[fps], stride
    hop, W = HOP[fps], WIN[fps]
    lengths = [0, 1, 511, 512, 1024, W * hop - 1, W * hop, W * hop + 1, (W + 1) * hop, (W + 1) * hop + 5,
               (W + 31) * hop, (W + 32) * hop - 1, (W + 64) * stride * hop, 60 * 16000]
    n_edge = -(-512 // hop)
    for i in range(len(lengths)):
        sub = lengths[i:] + lengths[:i][:3]
        a, _ = _args(sub, fps, stride)
        rc, n_win, n_frames, ws = _size(lib, a)
        assert rc == 0, lib.koe_last_error()
        outs = [m.num_output_frames(L) for L in sub]
        assert n_win == sum(outs)
        assert n_frames == sum((n - 1) * stride + W + 1 for n in outs)
        with_edges = any(not (n == 1 and L <= W * hop) for n, L in zip(outs, sub))
        floats = n_frames * 81 + (2 * n_edge * n_win * 81 if with_edges else 0)
        assert floats * 4 <= ws <= floats * 4 + 16 * 12 + 4 * (8 * len(sub) + 4) + 16


def test_all_short_clips_need_no_edge_rows(lib):
    a, _ = _args([136000, 16000, 0])
    rc, n_win, n_frames, ws = _size(lib, a)
    assert rc == 0 and n_win == 3 and n_frames == 3 * 257
    assert ws < 3 * 257 * 81 * 4 + 1024


def test_sizing_rejects_misuse(lib):
    for lengths in ([5, -1], [1 << 30]):
        a, _ = _args(lengths)
        assert _size(lib, a)[0] == -1
        assert b"outside [0, 2^30)" in lib.koe_last_error()
    a, _ = _args([16000] * 4, fps=30, stride=0)
    assert _size(lib, a)[0] == -1
    a, _ = _args([16000])
    a.hop = 100                                        # 6 edge frames per window side
    assert _size(lib, a)[0] == -1
    a, _ = _args([(1 << 30) - 1] * 1100)               # more than 2^31 frames in one call
    assert _size(lib, a)[0] == -1
    a, _ = _args([])
    assert _size(lib, a)[:3] == (0, 0, 0)


def test_forward_varlen_refuses_misuse_before_reading_buffers(lib):
    """Length misuse is refused by the library before any buffer or device is looked at."""
    a, _ = _args([16000, -3])
    assert lib.koe_forward_varlen(C.byref(a), None) == -1
    a, _ = _args([])
    assert lib.koe_forward_varlen(C.byref(a), None) == 0   # an empty batch is a no-op


def test_python_length_validation():
    from koemorph_b200.model.sequential_dual_stream_model import SequentialDualStreamModel as M
    assert M._check_lengths([3, 0, 4], 7).tolist() == [3, 0, 4]
    assert M._check_lengths(torch.tensor([2, 5], dtype=torch.int32), 7).dtype == torch.int64
    for bad, n in (([3, 4], 8), ([5, -1], 4), ([1.5, 2], 3), (torch.tensor([1.0, 2.0]), 3)):
        with pytest.raises(ValueError):
            M._check_lengths(bad, n)
