"""Every mel row of every frontend path against the float64 model of the frontend (oracle/logmel_model.py), with the
per-band gates derived from the fp32 error bound of its pair-packed FFT.

test_gpu_parity.py gates bands within 60 dB of the clip peak at 8.7e-4 dB and every other band only at 2e-6 of the
clip peak in power, which lets a band 70 dB down be off by some 13 dB; several paths are only compared bit for bit
with another path.  Here each band of each row the library computes is held to its own gate: the rounding of an fp32
transform of that frame and its pair partner, times 4.  On a failure the message names the clip (or stream and hop),
the row, the frame, the band and the pair partner.  The model takes the library's own float32 bank
(LogMelFrontend.filterbank()), which is checked against the float64 banks on its own.

Paths: LogMelFrontend.power (default bank on the warp-specialised kernel, a generic bank on the lock-step kernel,
split pairs, constant and reflect padding, a grid of frame offsets / steps / sample offsets / masks / output rows);
koe_forward_windows with test-owned workspace buffers (plain rows and every edge-variant buffer, batches up to 2100
clips including the early-released launch); koe_forward_varlen_ex (plain, steady and lead variant rows read from the
workspace as include/koemorph_b200.h lays it out); StreamingEngine rings after every hop; StreamPool (one hop per push,
bursts of up to 8 hops, warm-up) rings and staging; the two reference extractors; koe_logmel_normalise.

Largest error / gate measured on a B200 (power limit 1000 W), the worst input kind of logmel_model.KINDS per path
(G = 4, so 0.25 is the fp32 bound itself):
  LogMelFrontend.power   default bank 0.28, generic bank 0.27, split pairs 0.28, ragged grid constant 0.20 / reflect 0.19
  koe_forward_windows    sequences: plain 0.29, window-start 0.26, window-end 0.23; batches of 1-2100 clips
                         (early-released launch): plain 0.46 at 30 fps, 0.30 at 60 fps
  koe_forward_varlen(_ex) plain 0.26, steady variants 0.11, lead window-end variants 0.29
  StreamingEngine        rings and window-end rows 0.28 (30 fps), 0.30 (60 fps)
  StreamPool             default, max_hops 8 and warm-up alike: 0.27 (30 fps), 0.30 (60 fps)
  extractors             MelSlidingWindowExtractor 0.15 (n_fft 512 and 1024), MelSpectrogramExtractor 0.30
No path exceeded its gate.  tests/test_logmel_model.py shows each mutation of logmel_model.MUTATIONS (frame shifted by a
sample, symmetric Hann, a dropped bank bin at each run boundary, partner leak, fp16 input, off-by-one masks, symmetric
padding, frame max over 79 bands) at least 5x over the same gates on the CPU.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O
from oracle import logmel_model as M

pytestmark = pytest.mark.gpu

KINDS = M.KINDS
WORST = {}   # path -> largest error / gate seen


@pytest.fixture(scope="module")
def K():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import koemorph_b200
    from koemorph_b200 import _lib
    _lib.load()
    yield koemorph_b200
    for path in sorted(WORST):   # the largest error / gate per path of this run (run with -s to see it)
        print(f"logmel worst {path:60s} {WORST[path]:.3f}")


def _frontend(**kw):
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    return LogMelFrontend.get("cuda", **kw)


def _audio(n_clips, n_samples, seed=0):
    """(B, L) float32: clip b is of kind KINDS[b % len(KINDS)]."""
    out = np.empty((n_clips, n_samples), np.float32)
    for i, kind in enumerate(KINDS):
        idx = np.arange(i, n_clips, len(KINDS))
        if len(idx):
            out[idx] = M.make_audio(kind, len(idx), n_samples, seed=seed + i)
    return out


def _np(t):
    return t.detach().cpu().double().numpy()


def _record(path, ratio):
    WORST[path] = max(WORST.get(path, 0.0), float(ratio))
    print(f"logmel {path:50s} max error / gate {WORST[path]:.3f}")


def _check(path, log, fmax, ref, clip_names=None):
    """log (B, R, 80) / fmax (B, R) as the library stored them against the model rows `ref` of the same shape."""
    log, fmax = np.asarray(log, np.float64), np.asarray(fmax, np.float64)
    assert log.shape == ref["log"].shape, f"{path}: shape {log.shape} vs model {ref['log'].shape}"
    bad = np.argwhere(fmax != log.max(-1))
    assert len(bad) == 0, f"{path}: frame max of clip {bad[0][0]}, row {bad[0][1]} is not its row's largest band"
    r = M.excess(log, ref)
    _record(path, r.max() if r.size else 0.0)
    if r.size and r.max() > 1:
        b, j, m = np.unravel_index(int(np.argmax(r)), r.shape)
        name = clip_names[b] if clip_names is not None else f"clip {b} ({KINDS[b % len(KINDS)]})"
        raise AssertionError(
            f"{path}: {name}, row {j} = frame {int(ref['frame'][j])}, band {m}: got {log[b, j, m]:.7g}, model "
            f"{ref['log'][b, j, m]:.7g}, {r[b, j, m]:.3g} x the gate (pair partner row {int(ref['partner'][j])}, "
            f"{int((r > 1).sum())} bands over the gate)")


def _bank(fe):
    return fe.filterbank().astype(np.float64)


# ---- 1. LogMelFrontend.power ----------------------------------------------------------------------------------------------
def test_banks_against_float64(K):
    """The library's float32 banks against the float64 formulas: Slaney (the default and a generic one) and HTK."""
    for kw, ref in ((dict(), M.slaney_bank()), (dict(f_min=60.0, f_max=7600.0), M.slaney_bank(fmin=60.0, fmax=7600.0)),
                    (dict(n_fft=512, mel_scale="htk", window_normalized=True, log_mode="ln", log_eps=1e-8),
                     M.htk_bank(n_fft=512))):
        fb = _frontend(**kw).filterbank()
        assert np.abs(fb - ref).max() <= 1.2e-7 * ref.max(), kw
        assert ((fb > 0) == (ref > 0)).all(), kw


@pytest.mark.parametrize("bank", ["default", "generic"])
@pytest.mark.parametrize("hop,n_frames", [(533, 257), (266, 512), (533, 255)])
def test_power_every_kind(K, bank, hop, n_frames):
    """One clip per input kind, 136000 samples: the bench geometry (frames 255, 256 run past the clip), 60 fps, odd."""
    fe = _frontend() if bank == "default" else _frontend(f_min=60.0, f_max=7600.0)
    assert fe.uses_unrolled_bank() == (bank == "default")
    audio = _audio(len(KINDS), 136000, seed=hop)
    db, fmax = fe.power(torch.from_numpy(audio).cuda(), hop, n_frames)
    ref = M.launch(audio, hop, n_frames, _bank(fe))
    _check(f"power {bank} bank", _np(db), _np(fmax), ref)


@pytest.mark.parametrize("bank", ["default", "generic"])
def test_power_split_pairs(K, bank):
    """out_b: the pairs' second frames in their own buffer (the streaming step's launch)."""
    fe = _frontend() if bank == "default" else _frontend(f_min=60.0, f_max=7600.0)
    audio = _audio(len(KINDS), 40000, seed=5)
    B, n = audio.shape[0], 75
    pb = torch.empty((B, n // 2, 80), device="cuda")
    fb = torch.empty((B, n // 2), device="cuda")
    db, fmax = fe.power(torch.from_numpy(audio).cuda(), 533, n, out_b=(pb, fb))
    ref = M.launch(audio, 533, n, _bank(fe))
    even = {k: (v[:, 0::2] if k not in ("frame", "partner") else v[0::2]) for k, v in ref.items()}
    odd = {k: (v[:, 1::2] if k not in ("frame", "partner") else v[1::2]) for k, v in ref.items()}
    _check(f"power split pairs {bank} bank", _np(db)[:, 0::2], _np(fmax)[:, 0::2], even)
    _check(f"power split pairs {bank} bank", _np(pb), _np(fb), odd)


RAGGED_SHAPES = [  # L, hop, n_frames, frame_offset, pad_mode (test_gpu_parity.RAGGED_SHAPES, plus hop 532)
    (136000, 533, 257, 0, "constant"), (136000, 533, 256, 0, "constant"), (20000, 533, 38, 0, "constant"),
    (20000, 533, 5, 3, "constant"), (3000, 533, 6, 0, "constant"), (700, 533, 2, 0, "constant"),
    (1500, 533, 1, 1, "constant"), (20000, 266, 76, 0, "constant"), (20000, 533, 38, 0, "reflect"),
    (20000, 532, 38, 0, "reflect"), (136000, 532, 256, 0, "constant"), (3000, 532, 7, 0, "reflect"),
]
# frame_step, sample_offset, lo_rel, hi_rel, out_row (masks: constant padding only)
VARIANTS = [(1, 0, None, None, 0), (3, 100, 0, None, 2), (2, 0, None, 1, 1), (1, 37, -1, 2, 0), (1, 0, None, 0, 3)]


@pytest.mark.parametrize("L,hop,n_frames,frame_offset,pad_mode", RAGGED_SHAPES)
def test_power_ragged_grid(K, L, hop, n_frames, frame_offset, pad_mode):
    fe = _frontend()
    audio = _audio(4, L, seed=L + hop)
    x = torch.from_numpy(audio).cuda()
    for step, s_off, lo, hi, out_row in VARIANTS:
        if pad_mode == "reflect" and (lo is not None or hi is not None):
            continue
        R = out_row + n_frames + 1
        out = (torch.full((4, R, 80), 7.0, device="cuda"), torch.full((4, R), 7.0, device="cuda"))
        db, fmax = fe.power(x, hop, n_frames, frame_offset=frame_offset, frame_step=step, sample_offset=s_off,
                            lo_rel=lo, hi_rel=hi, pad_mode=pad_mode, out=out, out_row=out_row)
        db, fmax = _np(db), _np(fmax)
        assert (db[:, :out_row] == 7.0).all() and (db[:, out_row + n_frames:] == 7.0).all(), "rows outside the launch written"
        ref = M.launch(audio, hop, n_frames, _bank(fe), frame_offset=frame_offset, frame_step=step, sample_offset=s_off,
                       lo_rel=lo, hi_rel=hi, pad_mode=pad_mode)
        _check(f"power ragged grid {pad_mode}", db[:, out_row:out_row + n_frames], fmax[:, out_row:out_row + n_frames], ref)


# ---- 2. koe_forward_windows -----------------------------------------------------------------------------------------------
_models = {}


def _model(K, fps, stride=None):
    key = (fps, stride)
    if key not in _models:
        w = O.make_weights(21, fps, style="stress")
        kw = dict(target_fps=fps, mel_sequence_length=256 if fps == 30 else 512)
        m = K.SimplifiedDualStreamModel(**kw) if stride is None else K.SequentialDualStreamModel(stride_frames=stride, **kw)
        m.load_state_dict(O.model_state_dict(w), strict=True)
        m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
        m = m.cuda().eval()
        m.precision = "bf16"
        _models[key] = m
    return _models[key]


def _forward_windows(K, m, audio, n_frames, T, stride, n_out, n_edge):
    """koe_forward_windows with workspace buffers owned here, laid out as include/koemorph_b200.h documents."""
    from koemorph_b200 import _lib
    B, L = audio.shape
    f32 = dict(dtype=torch.float32, device="cuda")
    power = [torch.full((B, n_frames, 80), 7.0, **f32)] + [torch.full((B, n_out, 80), 7.0, **f32) for _ in range(2 * n_edge)]
    fmax = [torch.full(p.shape[:2], 7.0, **f32) for p in power]
    eg = torch.randn(B, 264, device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
    expr, out = torch.empty(B, **f32), torch.empty(B, n_out, 52, **f32)
    w = m.dual_stream_attention.kernel_weights(m._compression)
    a = _lib.ForwardArgs()
    a.frontend, a.weights = m._frontend(audio.device)._h, C.addressof(w.struct)
    a.audio, a.audio_stride = audio.data_ptr(), audio.stride(0)
    a.n_clips, a.n_samples, a.hop = B, L, m.hop_length
    a.n_frames, a.frames_per_window, a.stride_frames, a.n_out, a.n_edge = n_frames, T, stride, n_out, n_edge
    a.egemaps = eg.data_ptr()
    for j, (p, f) in enumerate(zip(power, fmax)):
        a.power[j], a.frame_max[j] = p.data_ptr(), f.data_ptr()
    a.expr_sigmoid, a.out = expr.data_ptr(), out.data_ptr()
    a.sigmoid_out = a.attn_out = None
    a.alpha, a.smooth, a.precision = 0.0, 0, 2
    _lib.check(_lib.load().koe_forward_windows(C.byref(a), _lib.stream_ptr(audio.device)), "koe_forward_windows")
    return [_np(p) for p in power], [_np(f) for f in fmax]


def _check_windows(path, fe, audio_np, power, fmax, hop, n_frames, T, stride, n_out, n_edge):
    bank = _bank(fe)
    B = audio_np.shape[0]
    for c0 in range(0, B, 256):   # (the model, in chunks of clips)
        sl = slice(c0, c0 + 256)
        a = audio_np[sl]
        names = [f"clip {c} ({KINDS[c % len(KINDS)]})" for c in range(c0, c0 + len(a))]
        _check(f"{path}: plain rows", power[0][sl], fmax[0][sl], M.launch(a, hop, n_frames, bank), names)
        for m in range(n_edge):
            ref = M.launch(a, hop, n_out, bank, frame_offset=m, frame_step=stride, lo_rel=-m)
            _check(f"{path}: window-start variant {m}", power[1 + 2 * m][sl], fmax[1 + 2 * m][sl], ref, names)
            ref = M.launch(a, hop, n_out, bank, frame_offset=T - 1 - m, frame_step=stride, hi_rel=m)
            _check(f"{path}: window-end variant {m}", power[2 + 2 * m][sl], fmax[2 + 2 * m][sl], ref, names)


# fps, stride, extra samples past the last complete window (window-count boundaries)
SEQUENCES = [(30, 1, 0), (30, 1, 532), (30, 3, 533 * 2 + 1), (30, 3, 533 * 3), (60, 1, 265), (60, 1, 266),
             (60, 3, 3 * 266 + 1), (60, 3, 2 * 266 + 265)]


@pytest.mark.parametrize("fps,stride,extra", SEQUENCES)
def test_forward_windows_sequences(K, fps, stride, extra):
    m = _model(K, fps, stride)
    hop, W = m.hop_length, m.window_frames
    L = (W + 4 * stride) * hop + extra
    n_out = m.num_output_frames(L)
    T = W + 1
    n_frames = (n_out - 1) * stride + T
    n_edge = -(-512 // hop)
    audio = _audio(len(KINDS), L, seed=fps + stride + extra)
    power, fmax = _forward_windows(K, m, torch.from_numpy(audio).cuda(), n_frames, T, stride, n_out, n_edge)
    _check_windows(f"forward_windows {fps} fps", m._frontend("cuda"), audio, power, fmax, hop, n_frames, T, stride, n_out,
                   n_edge)


@pytest.mark.parametrize("fps,n_clips", [(30, 1), (30, 149), (30, 512), (30, 2100), (60, 512)])
def test_forward_windows_batches(K, fps, n_clips):
    """One window per clip, bf16, no edge variants: above one round of windows the core is released early by the
    frontend (the launch the benchmark measures)."""
    m = _model(K, fps, 1)
    hop, T = m.hop_length, m.window_frames + 1
    audio = _audio(n_clips, 136000, seed=n_clips)
    power, fmax = _forward_windows(K, m, torch.from_numpy(audio).cuda(), T, T, 1, 1, 0)
    _check_windows(f"forward_windows batch {fps} fps", m._frontend("cuda"), audio, power, fmax, hop, T, T, 1, 1, 0)


# ---- 3. koe_forward_varlen / _ex ------------------------------------------------------------------------------------------
def _align16(x):
    return (x + 15) // 16 * 16


@pytest.mark.parametrize("warmup", [False, True])
@pytest.mark.parametrize("fps,stride", [(30, 1), (60, 2), (30, 3)])
def test_forward_varlen_rows(K, fps, stride, warmup):
    """The plain, steady and lead variant rows of a packed batch, read from the workspace at the offsets the header
    documents for koe_forward_varlen_size."""
    from koemorph_b200 import _lib
    m = _model(K, fps, stride)
    hop, W, s = m.hop_length, m.window_frames, stride
    T, n_edge, r = W + 1, -(-512 // hop), (W - 1) % stride
    lengths = [136000, 20 * hop + 5, (W + 3 * s) * hop + 17, (r + 1) * hop, W * hop, W * hop + hop - 1, 3 * hop + 100,
               40000, (W - 1) * hop + 3, 5 * hop, 70001]
    B = len(lengths)
    clips = [M.make_audio(KINDS[c % len(KINDS)], 1, n, seed=c + fps)[0] for c, n in enumerate(lengths)]
    flat = torch.from_numpy(np.concatenate(clips)).cuda()
    lens = torch.tensor(lengths, dtype=torch.int64)
    eg = torch.randn(B, 264, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))
    # per-clip geometry (header: koe_forward_varlen, KOE_VARLEN_WARMUP)
    n_out = [max(1, (n // hop - W) // s + 1) for n in lengths]
    n_frames = [(o - 1) * s + W + 1 for o in n_out]
    plain = [o == 1 and n <= W * hop for o, n in zip(n_out, lengths)]
    leads = []
    for n in lengths:
        last = min(W - 2, n // hop - 1)
        leads.append(0 if not warmup or last < r else (last - r) // s + 1)
    rows = [k + (o if n // hop >= W else 0) if warmup else o for k, o, n in zip(leads, n_out, lengths)]
    E = n_edge if (not all(plain) or sum(leads) > 0) else 0
    N = sum(n_out) if not all(plain) else 0
    F, Kt = sum(n_frames), sum(leads)
    var_rows = [F] + [N + (Kt if j % 2 == 0 else 0) for j in range(1, 2 * E + 1)]
    off, offs_p, offs_f = 0, [], []
    for n in var_rows:
        offs_p.append(off)
        off += _align16(n * 80 * 4)
    for n in var_rows:
        offs_f.append(off)
        off += _align16(n * 4)
    w = m.dual_stream_attention.kernel_weights(m._compression)
    a = _lib.ForwardVarlenArgs()
    a.frontend, a.weights = m._frontend("cuda")._h, C.addressof(w.struct)
    a.audio, a.lengths_host, a.n_clips = flat.data_ptr(), lens.data_ptr(), B
    a.hop, a.window_frames, a.stride_frames, a.half_fft = hop, W, s, 512
    a.smooth, a.precision, a.alpha = 0, 2, 0.0
    flags = _lib.VARLEN_WARMUP if warmup else 0
    n_win, n_fr, ws_bytes = C.c_int64(), C.c_int64(), C.c_int64()
    lib = _lib.load()
    _lib.check(lib.koe_forward_varlen_size_ex(C.byref(a), flags, C.byref(n_win), C.byref(n_fr), C.byref(ws_bytes)))
    assert n_win.value == sum(rows) and n_fr.value == F and off <= ws_bytes.value
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device="cuda")
    out = torch.empty(n_win.value, 52, device="cuda")
    a.egemaps, a.workspace, a.workspace_bytes, a.out = eg.data_ptr(), ws.data_ptr(), ws_bytes.value, out.data_ptr()
    a.sigmoid_out = a.attn_out = None
    _lib.check(lib.koe_forward_varlen_ex(C.byref(a), flags, _lib.stream_ptr(flat.device)), "koe_forward_varlen_ex")
    torch.cuda.synchronize()

    def region(j, n):
        p = ws[offs_p[j]:offs_p[j] + n * 320].view(torch.float32).view(n, 80)
        f = ws[offs_f[j]:offs_f[j] + n * 4].view(torch.float32)
        return _np(p), _np(f)

    bank = _bank(m._frontend("cuda"))
    regions = [region(j, n) for j, n in enumerate(var_rows)]
    fb = wb = lb = 0
    tag = f"forward_varlen{'_ex warm-up' if warmup else ''} {fps} fps stride {s}"
    for c, n in enumerate(lengths):
        x = clips[c][None, :]
        name = f"clip {c} ({KINDS[c % len(KINDS)]}, {n} samples)"
        p, f = regions[0]
        _check(f"{tag}: plain rows", p[None, fb:fb + n_frames[c]], f[None, fb:fb + n_frames[c]],
               M.launch(x, hop, n_frames[c], bank), [name])
        if not plain[c]:
            for mm in range(n_edge):
                p, f = regions[1 + 2 * mm]
                _check(f"{tag}: window-start variant {mm}", p[None, wb:wb + n_out[c]], f[None, wb:wb + n_out[c]],
                       M.launch(x, hop, n_out[c], bank, frame_offset=mm, frame_step=s, lo_rel=-mm), [name])
                p, f = regions[2 + 2 * mm]
                _check(f"{tag}: window-end variant {mm}", p[None, wb:wb + n_out[c]], f[None, wb:wb + n_out[c]],
                       M.launch(x, hop, n_out[c], bank, frame_offset=T - 1 - mm, frame_step=s, hi_rel=mm), [name])
        if leads[c]:
            for mm in range(n_edge):
                p, f = regions[2 + 2 * mm]
                rows_c = slice(N + lb, N + lb + leads[c])
                _check(f"{tag}: lead window-end variant {mm}", p[None, rows_c], f[None, rows_c],
                       M.launch(x, hop, leads[c], bank, frame_offset=r + 1 - mm, frame_step=s, hi_rel=mm), [name])
        fb, wb, lb = fb + n_frames[c], wb + n_out[c], lb + leads[c]


# ---- 4. StreamingEngine, 5. StreamPool ------------------------------------------------------------------------------------
def _hop_rows(x, n, hop, n_edge, bank):
    """Model rows of the variants a stream computes at its hop n from its audio so far x (1, (n + 1) * hop): V rows in
    the staging order plain, window-start 0, window-end 0, window-start 1, window-end 1 (koe_stream_push)."""
    g = n - (n_edge - 1)
    pair = M.launch(x, hop, 2, bank, frame_offset=g)           # plain frame g and frame g + 1: one pair
    pick = lambda ref, j: {k: (v[:, j:j + 1] if k not in ("frame", "partner") else v[j:j + 1]) for k, v in ref.items()}
    rows = [pick(pair, 0), M.launch(x, hop, 1, bank, frame_offset=g, lo_rel=0)]
    if n_edge == 1:
        rows.append(pick(pair, 1))
    else:
        rows += [M.launch(x, hop, 1, bank, frame_offset=g + 2), M.launch(x, hop, 1, bank, frame_offset=g, lo_rel=-1),
                 pick(pair, 1)]
    return g, rows


def _check_row(path, got, gmax, ref, what):
    """One stored row (80,) and its frame max against a one-row model launch."""
    r = M.excess(got[None, None], ref)[0, 0]
    _record(path, r.max())
    assert gmax == got.max(), f"{path}: {what}: frame max {gmax} is not the row's largest band {got.max()}"
    if r.max() > 1:
        mb = int(np.argmax(r))
        raise AssertionError(f"{path}: {what}, band {mb}: got {got[mb]:.7g}, model {ref['log'][0, 0, mb]:.7g}, "
                             f"{r.max():.3g} x the gate")


class _Ring:
    """Model of a ring buffer [streams][rows][80]: what each row written so far must hold, checked all at once."""

    def __init__(self, n_streams, n_rows):
        self.log = np.zeros((n_streams, n_rows, 80))
        self.gate = np.ones((n_streams, n_rows, 80))
        self.frame = np.full((n_streams, n_rows), -10 ** 9)
        self.written = np.zeros((n_streams, n_rows), bool)

    def put(self, s, row, ref):
        self.log[s, row], self.gate[s, row] = ref["log"][0, 0], ref["gate_log"][0, 0]
        self.frame[s, row], self.written[s, row] = ref["frame"][0], True

    def check(self, path, ring, fmax, what):
        ring, fmax = _np(ring), _np(fmax)
        w = self.written
        assert (fmax[w] == ring[w].max(-1)).all(), f"{path}: {what}: a frame max is not its row's largest band"
        r = np.where(w[..., None], np.abs(ring - self.log) / self.gate, 0.0)
        _record(path, r.max())
        if r.max() > 1:
            s, row, mb = np.unravel_index(int(np.argmax(r)), r.shape)
            raise AssertionError(f"{path}: {what}: stream {s}, ring row {row} (frame {self.frame[s, row]}), band {mb}: "
                                 f"got {ring[s, row, mb]:.7g}, model {self.log[s, row, mb]:.7g}, {r.max():.3g} x the gate")


@pytest.mark.parametrize("fps", [30, 60])
def test_streaming_engine_rings_every_hop(K, fps):
    """koe_stream_push: after each of W + 5 hops, every ring row written so far and the window-end rows, against the
    model on each stream's audio so far (the tail-based frontend pairs frame g with frame g + 1)."""
    from koemorph_b200.streaming import StreamingEngine
    m = _model(K, fps)
    m.use_temporal_smoothing = False
    S = len(KINDS)
    eng = StreamingEngine(m, S)
    hop, W, n_edge = eng.hop, eng.W, eng.n_edge
    bank = _bank(eng._fe)
    n_hops = W + 5
    audio = _audio(S, n_hops * hop, seed=fps + 1)
    x = torch.from_numpy(audio).cuda()
    eng.set_egemaps(torch.randn(S, 264, device="cuda"))
    rings = [("ring_f", "fmax_f", 0), ("ring_r", "fmax_r", 1)] + ([("ring_r2", "fmax_r2", 3)] if n_edge == 2 else [])
    rows_l = [("row_l", "fmax_l", 2)] + ([("row_l2", "fmax_l2", 4)] if n_edge == 2 else [])
    model = {name: _Ring(S, W) for name, _, _ in rings}
    path = f"StreamingEngine {fps} fps"
    for n in range(n_hops):
        eng.step(x[:, n * hop:(n + 1) * hop])
        for s in range(S):
            g, rows = _hop_rows(audio[s:s + 1, :(n + 1) * hop], n, hop, n_edge, bank)
            for name, _, v in rings:
                model[name].put(s, g % W, rows[v])
            for name, fname, v in rows_l:
                _check_row(path, _np(getattr(eng, name)[s, 0]), float(_np(getattr(eng, fname)[s, 0])), rows[v],
                           f"stream {s} ({KINDS[s]}), hop {n}, {name}")
        for name, fname, _ in rings:
            model[name].check(path, getattr(eng, name), getattr(eng, fname), f"after hop {n}, {name}")


@pytest.mark.parametrize("mode", ["default", "max_hops 8", "warmup"])
@pytest.mark.parametrize("fps", [30, 60])
def test_stream_pool_rings_and_staging(K, fps, mode):
    """StreamPool: every staged row of every push (per-hop tails with bursts of up to 8 hops; warm-up, whose window-end
    rows see zeros past the audio so far) and every ring row written so far, after each push."""
    from koemorph_b200.streaming import StreamPool
    m = _model(K, fps)
    m.use_temporal_smoothing = False
    S = len(KINDS)
    H = 8 if mode == "max_hops 8" else 1
    pool = StreamPool(m, S, max_hops=H, warmup=mode == "warmup")
    hop, W, n_edge, R = pool.hop, pool.W, pool.n_edge, pool.ring_frames
    V = 1 + 2 * n_edge
    bank = _bank(pool._fe)
    n_hops = W + 5
    audio = _audio(S, (n_hops + H) * hop, seed=fps + 7)
    x = torch.from_numpy(audio).cuda()
    slots = pool.open(torch.randn(S, 264, device="cuda"))
    rng = np.random.default_rng(fps)
    done = [0] * S
    ring_of = {0: ("ring_f", "fmax_f"), 1: ("ring_r", "fmax_r"), 3: ("ring_r2", "fmax_r2")}
    ring_of = {v: ring_of[v] for v in (0, 1, 3)[:1 + n_edge]}
    model = {v: _Ring(S, R) for v in ring_of}
    path = f"StreamPool {mode} {fps} fps"
    while min(done) < n_hops:
        act = [s for s in range(S) if done[s] < n_hops]           # streams still pushing, in call order
        counts = [1] * S if H == 1 else [int(c) for c in rng.integers(1, H + 1, S)]
        hops = torch.cat([x[s, done[s] * hop:(done[s] + counts[s]) * hop] for s in act])
        if H == 1:
            pool.push([slots[s] for s in act], hops.view(len(act), hop))
        else:
            pool.push_hops([slots[s] for s in act], hops, [counts[s] for s in act])
        stage, stage_max = _np(pool.stage), _np(pool.stage_max)
        e = 0
        for s in act:
            for n in range(done[s], done[s] + counts[s]):
                g, rows = _hop_rows(audio[s:s + 1, :(n + 1) * hop], n, hop, n_edge, bank)
                for v in range(V):
                    _check_row(path, stage[e, v], float(stage_max[e, v]), rows[v],
                               f"stream {s} ({KINDS[s]}), hop {n}, staged hop {e}, stage variant {v}")
                for v in model:
                    model[v].put(slots[s], g % R, rows[v])
                e += 1
            done[s] += counts[s]
        for v, (name, fname) in ring_of.items():
            model[v].check(path, getattr(pool, name), getattr(pool, fname), f"after push {pool.pushes}, {name}")
        if mode == "default":   # the window-end rows of the push: the staged rows, copied
            for v, (name, fname) in ((2, ("row_l", "fmax_l")), (4, ("row_l2", "fmax_l2")))[:n_edge]:
                got, fm = _np(getattr(pool, name)), _np(getattr(pool, fname))
                for i, s in enumerate(act):
                    assert np.array_equal(got[slots[s]], stage[i, v]) and fm[slots[s]] == stage_max[i, v], (name, s)


# ---- 6. the extractors ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_fft,win_length", [(512, None), (1024, None), (512, 400)])
def test_mel_sliding_window_extractor(K, n_fft, win_length):
    """process_audio_batch: dB relative to the clip max, clamped at -80 (reflect padding, hop 532).  The gate of a band is
    its own plus that of the clip's loudest band, plus the rounding of the subtraction."""
    from koemorph_b200.features.mel_sliding_window import MelSlidingWindowExtractor
    ex = MelSlidingWindowExtractor(n_fft=n_fft, win_length=win_length, device="cuda")
    bank = ex._fe.filterbank().astype(np.float64)
    for c, kind in enumerate(KINDS):
        a = M.make_audio(kind, 1, 40000, seed=c)
        got = _np(ex.process_audio_batch(a[0], as_tensor=True))
        ref = M.launch(a, ex.hop_length, 1 + a.shape[1] // ex.hop_length, bank, pad_mode="reflect", n_fft=n_fft,
                       win_length=win_length)
        y = ref["log"][0]
        i = np.unravel_index(int(np.argmax(y)), y.shape)
        want = np.maximum(y - y[i], -80.0)
        gate = ref["gate_log"][0] + ref["gate_log"][0][i] + 2 * np.spacing(np.abs(want).astype(np.float32))
        r = np.abs(got - want) / gate
        _record(f"MelSlidingWindowExtractor n_fft {n_fft}", r.max())
        assert r.max() <= 1, f"{kind}: {M.worst(r)}"


def test_mel_spectrogram_extractor(K):
    """torchaudio flavour: HTK bank, 512-point frame, window-power normalisation, ln(p + 1e-8), reflect padding,
    truncated / last-row-padded to int(L / sr * fps) frames."""
    from koemorph_b200.features.stft import MelSpectrogramExtractor
    ex = MelSpectrogramExtractor().cuda()
    for L in (40000, 16000 * 3 + 7):
        audio = _audio(len(KINDS), L, seed=L)
        got = _np(ex(torch.from_numpy(audio).cuda()))
        fe = ex._frontend(torch.device("cuda"))
        n = 1 + L // ex.hop_length
        ref = M.launch(audio, ex.hop_length, n, _bank(fe), pad_mode="reflect", n_fft=512, window_normalized=True,
                       log_mode="ln", log_eps=ex.eps)
        T = got.shape[1]
        assert T == int(L / 16000 * 30)
        k = min(T, n)
        r = M.excess(got[:, :k], {k2: (v[:, :k] if k2 not in ("frame", "partner") else v) for k2, v in ref.items()})
        _record("MelSpectrogramExtractor", r.max())
        assert r.max() <= 1, M.worst(r)
        assert (got[:, k:] == got[:, k - 1:k]).all()


# ---- 7. koe_logmel_normalise ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 2, 3, 4, 257])
def test_normalise_against_float64(K, T):
    """Long-term rows within 2 ulp of (max(d, -80) + 80) / 80 in float64 from the kernel's own dB rows, d = dB - clip
    max: the difference is taken as float32 rounds it (correctly rounded, and 80 dB below the peak one of its ulps is
    thousands of ulps of the result, so no kernel could match a float64 difference there).  Short-term rows are the last
    three long-term rows, zero padded below three frames; every frame max is its row's largest band."""
    fe = _frontend()
    audio = _audio(len(KINDS) + 1, max(T - 1, 1) * 533 + 100, seed=T)
    audio[-1] = 0.0                                              # digital silence: every band on the floor
    db, fmax = fe.power(torch.from_numpy(audio).cuda(), 533, T)
    lt, st = fe.normalise(db, fmax)
    assert torch.equal(fmax, db.max(-1).values)
    db32, cmax = db.cpu().numpy(), fmax.cpu().numpy().max(1)
    d = (db32 - cmax[:, None, None]).astype(np.float32).astype(np.float64)
    ref = (np.maximum(d, -80.0) + 80.0) / 80.0
    lt, st = _np(lt), _np(st)
    ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
    err = np.abs(lt - ref) / ulp
    assert err.max() <= 2, f"long-term: {M.worst(err)} (ulp)"
    want = np.zeros((ref.shape[0], 3, 80))
    want[:, :min(T, 3)] = lt[:, T - min(T, 3):]
    np.testing.assert_array_equal(st, want)
