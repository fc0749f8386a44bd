"""Float64 model of the log-mel frontend (csrc/logmel.cu) and the error bound its fp32 arithmetic must meet.

TEST INFRASTRUCTURE ONLY, like the rest of ``oracle/``: numpy / scipy, no torch, no device.

Rows.  ``launch`` computes, in float64 from the float32 audio, the rows one ``koe_logmel_power_ex`` launch writes: row j
of clip b is frame g = frame_offset + j * frame_step, the 1024-sample frame centred on sample_offset + g * hop, with
samples outside [lo, hi) read as zero (lo = max(0, sample_offset + (g + lo_rel) * hop), hi = min(L, sample_offset +
(g + hi_rel) * hop) when the masks are given) or, with ``pad_mode="reflect"``, reflected about the first / last sample.
The window is the periodic Hann of ``win_length`` points centred in the ``n_fft`` frame, centred in turn in the
1024-point transform (a 512-point frame is the middle of a zero-extended 1024-point one: its bin k is bin 2k of the
larger transform).  Mel power P = s * sum_k w_k |X_k|^2 with the bank passed in (s = 1 / sum(window^2) with
``window_normalized``, else 1), then ``10 log10(max(P, 1e-10))`` (``log_mode="db"``) or ``ln(P + log_eps)``, and the
frame max over the bands.  Taking the bank as an argument lets a GPU test pass the library's own float32 bank
(``LogMelFrontend.filterbank()``), which keeps bank construction out of the comparison; ``slaney_bank`` / ``htk_bank``
build the float64 banks it is checked against separately.

Error bound.  The kernel transforms the two frames of a pair (rows 2j and 2j + 1 of a launch's frame list, per clip) as
one complex FFT z = a + i b and separates them with the conjugate-symmetric partner, so its rounding scales with the
pair's combined norm.  With x_t the windowed samples of frame t and x_u those of its partner (zero for the unpaired last
row of an odd launch), the per-bin error scale is

    delta_t = eps32 * sqrt(log2 1024) * sqrt(|x_t|^2 + |x_u|^2)

and the band gate, in power, is

    gate = G * (8 eps32 P + s * (2 delta_t sum_k w_k |X_k| + delta_t^2 sum_k w_k)),    G = 4.

In dB it is |d dB| <= 10 / ln 10 * gate / max(P, 1e-10), in ``ln`` mode |d| <= gate / (P + eps).  The log itself is
evaluated with a 2-ulp log2 and stored as float32, so the log gates add 4 ulp of the stored value (at most 3e-5 dB for
any value the clamp allows); that floor is far below every bug below.

``fp32_emulation=True`` computes the rows the way the kernel's arithmetic does, not in its operation order: float32
windowed samples, the pair packed into one complex64 ``scipy.fft.fft``, separated with the conjugate-symmetric partner,
|X|^2 and the bank sum in float32.  On every input kind of the tests it stays under a quarter of the gate.

Mutations (``mutate=``), each a plausible kernel bug that the gate must reject by at least 5x on some input:
  frame_shift      every frame starts one sample late
  symmetric_hann   the symmetric instead of the periodic Hann window
  drop_bin:K       bin K of the bank is skipped (K = each of the 15 interior run boundaries of the default bank,
                   ``kDefRunBin`` in csrc/melbank_default.inc: ``DROP_BINS``)
  partner_leak     3e-4 of the pair partner's windowed samples leak into each frame (a wrong pair separation)
  fp16_input       the input samples are rounded to fp16
  mask_off_by_one  the lo_rel / hi_rel masks start one sample late (sample lo is zeroed, sample hi is read)
  symmetric_pad    numpy "symmetric" instead of "reflect" padding
  max_79_bands     the frame max is taken over the first 79 bands only

Not caught: twiddles with 1e-6 relative error reach only 2.6-4.8 times the bound (G = 1), at most 1.2x the gate, which
is no margin.  The bound is not tightened for them: twiddle accuracy is not observable through the ABI, and a gate that
catches them would also reject legitimate fp32 rounding on some inputs.
"""
from __future__ import annotations

import math
import os
import re
from typing import Dict, Optional, Sequence

import numpy as np
import scipy.fft
import scipy.signal

from . import koemorph_oracle as O

EPS32 = float(np.finfo(np.float32).eps)
G = 4.0
AMIN = 1e-10
FRAME = 1024                       # the kernel's transform length
DB_PER_LN = 10.0 / math.log(10.0)  # d(10 log10 P) = DB_PER_LN * dP / P
LOG_ULPS = 4.0                     # log2 within 2 ulp, the scale by 10 log10 2 and the float32 store


def _default_run_bins() -> np.ndarray:
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "koemorph_b200", "csrc",
                        "melbank_default.inc")
    with open(path) as f:
        m = re.search(r"kDefRunBin\[17\]\s*=\s*\{([^}]*)\}", f.read())
    return np.array([int(v) for v in m.group(1).split(",")])


DEF_RUN_BIN = _default_run_bins()
DROP_BINS = tuple(int(k) for k in DEF_RUN_BIN[1:-1])   # the 15 interior run boundaries
MUTATIONS = ("frame_shift", "symmetric_hann", *[f"drop_bin:{k}" for k in DROP_BINS], "partner_leak", "fp16_input",
             "mask_off_by_one", "symmetric_pad", "max_79_bands")


# ---- banks --------------------------------------------------------------------------------------------------------------
def slaney_bank(sr: int = 16000, n_fft: int = 1024, n_mels: int = 80, fmin: float = 80.0, fmax: float = 8000.0) -> np.ndarray:
    """librosa.filters.mel(htk=False, norm="slaney") in float64: (n_mels, 1 + n_fft // 2)."""
    fftfreqs = np.fft.rfftfreq(n=n_fft, d=1.0 / sr)
    mel_f = O.mel_to_hz(np.linspace(O.hz_to_mel(fmin), O.hz_to_mel(fmax), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fftfreqs)
    lower = -ramps[:-2] / fdiff[:-1, None]
    upper = ramps[2:] / fdiff[1:, None]
    w = np.maximum(0.0, np.minimum(lower, upper))
    return w * (2.0 / (mel_f[2:] - mel_f[:-2]))[:, None]


def htk_bank(sr: int = 16000, n_fft: int = 512, n_mels: int = 80, fmin: float = 80.0, fmax: float = 8000.0) -> np.ndarray:
    """torchaudio.functional.melscale_fbanks(mel_scale="htk", norm=None) in float64, transposed: (n_mels, 1 + n_fft // 2)."""
    all_freqs = np.linspace(0.0, sr // 2, n_fft // 2 + 1)
    m_min, m_max = 2595.0 * np.log10(1.0 + fmin / 700.0), 2595.0 * np.log10(1.0 + fmax / 700.0)
    f_pts = 700.0 * (10.0 ** (np.linspace(m_min, m_max, n_mels + 2) / 2595.0) - 1.0)
    f_diff = np.diff(f_pts)
    slopes = f_pts[None, :] - all_freqs[:, None]
    down = -slopes[:, :-2] / f_diff[:-1]
    up = slopes[:, 2:] / f_diff[1:]
    return np.maximum(0.0, np.minimum(down, up)).T


# ---- frames -------------------------------------------------------------------------------------------------------------
def window(n_fft: int = 1024, win_length: Optional[int] = None, symmetric: bool = False) -> np.ndarray:
    """The 1024-point analysis window: periodic Hann of win_length points centred in the n_fft frame, centred in 1024."""
    wl = n_fft if win_length in (None, 0) else int(win_length)
    w = np.zeros(FRAME)
    start = (FRAME - n_fft) // 2 + (n_fft - wl) // 2
    w[start:start + wl] = scipy.signal.get_window("hann", wl, fftbins=not symmetric)
    return w


def frame_samples(clip: np.ndarray, centres: np.ndarray, lo: np.ndarray, hi: np.ndarray, pad_mode: str = "constant",
                  symmetric_pad: bool = False) -> np.ndarray:
    """(R, 1024) float64 samples of the frames centred on `centres` of one clip: zero outside [lo, hi), or reflected."""
    n = len(clip)
    idx = centres[:, None] - FRAME // 2 + np.arange(FRAME)[None, :]
    if pad_mode == "reflect":
        last = n - 1
        if symmetric_pad:
            idx = np.where(idx < 0, -idx - 1, np.where(idx > last, 2 * last + 1 - idx, idx))
        else:
            idx = np.where(idx < 0, -idx, np.where(idx > last, 2 * last - idx, idx))
        ok = (idx >= 0) & (idx <= last)
    else:
        ok = (idx >= lo[:, None]) & (idx < hi[:, None])
    src = np.asarray(clip, np.float64)
    return np.where(ok, src[np.clip(idx, 0, max(n - 1, 0))] if n > 0 else 0.0, 0.0)


def _pair_partner(n_rows: int) -> np.ndarray:
    """Row index of each row's pair partner (rows 2j, 2j + 1), -1 for the unpaired last row of an odd launch."""
    p = np.arange(n_rows) ^ 1
    p[p >= n_rows] = -1
    return p


# ---- one launch -----------------------------------------------------------------------------------------------------------
def launch(audio: np.ndarray, hop: int, n_frames: int, bank: np.ndarray, *, frame_offset: int = 0, frame_step: int = 1,
           sample_offset: int = 0, lo_rel: Optional[int] = None, hi_rel: Optional[int] = None, pad_mode: str = "constant",
           n_fft: int = 1024, win_length: Optional[int] = None, window_normalized: bool = False, log_mode: str = "db",
           log_eps: float = 0.0, partner: str = "pair", fp32_emulation: bool = False,
           mutate: Optional[str] = None) -> Dict[str, np.ndarray]:
    """The rows of one koe_logmel_power_ex launch over the clips of `audio` (B, L) float32.

    Returns float64 arrays: ``power`` (B, n_frames, n_mels), ``log`` (the stored value, dB or ln), ``frame_max``
    (B, n_frames), the gates ``gate_power`` / ``gate_log`` (same shape as ``power``) and ``norm`` (B, n_frames), each
    frame's windowed-sample norm.  ``partner``: "pair" (rows 2j, 2j + 1 of the launch) or "neighbour" (the larger norm
    of the two adjacent rows, for launches whose pairing is not the plain one)."""
    audio = np.atleast_2d(np.asarray(audio, np.float32))
    if mutate is not None and mutate not in MUTATIONS:
        raise ValueError(f"unknown mutation {mutate!r}")
    if mutate == "fp16_input":
        audio = audio.astype(np.float16).astype(np.float32)
    B, L = audio.shape
    n_mels = bank.shape[0]
    sub = FRAME // n_fft
    bank = np.asarray(bank, np.float64)
    assert bank.shape[1] == n_fft // 2 + 1, "bank must be (n_mels, 1 + n_fft // 2)"
    if mutate is not None and mutate.startswith("drop_bin:"):
        bank = bank.copy()
        bank[:, int(mutate.split(":")[1])] = 0.0
    win = window(n_fft, win_length, symmetric=mutate == "symmetric_hann")
    scale = 1.0 / float(np.sum(win ** 2)) if window_normalized else 1.0
    g = frame_offset + np.arange(n_frames) * frame_step
    centres = sample_offset + g * hop + (1 if mutate == "frame_shift" else 0)
    lo = np.zeros(n_frames, np.int64)
    hi = np.full(n_frames, L, np.int64)
    shift = 1 if mutate == "mask_off_by_one" else 0
    if lo_rel is not None:
        lo = np.maximum(lo, sample_offset + (g + lo_rel) * hop + shift)
    if hi_rel is not None:
        hi = np.minimum(hi, sample_offset + (g + hi_rel) * hop + shift)
    out = {k: np.zeros((B, n_frames, n_mels)) for k in ("power", "log", "gate_power", "gate_log")}
    out["frame_max"] = np.zeros((B, n_frames))
    out["norm"] = np.zeros((B, n_frames))
    pidx = _pair_partner(n_frames)
    out["frame"], out["partner"] = g, pidx
    for b in range(B):
        x = frame_samples(audio[b], centres, lo, hi, pad_mode, symmetric_pad=mutate == "symmetric_pad") * win[None, :]
        norm = np.sqrt(np.sum(x * x, axis=1))
        if mutate == "partner_leak":
            xp = np.where(pidx[:, None] >= 0, x[np.maximum(pidx, 0)], 0.0)
            x = x + 3e-4 * xp
        X = np.abs(np.fft.rfft(x, axis=1))[:, ::sub]                        # (R, 1 + n_fft // 2)
        if fp32_emulation:
            P = _fp32_rows(audio[b], centres, lo, hi, pad_mode, win, pidx, bank, sub, scale)
        else:
            P = scale * ((X * X) @ bank.T)
        if partner == "pair":
            nu = np.where(pidx >= 0, norm[np.maximum(pidx, 0)], 0.0)
        else:
            nu = np.maximum(np.concatenate([[0.0], norm[:-1]]), np.concatenate([norm[1:], [0.0]]))
        delta = EPS32 * math.sqrt(math.log2(FRAME)) * np.sqrt(norm ** 2 + nu ** 2)
        # the gate of the exact P (fp32 emulation: of the float64 row it emulates)
        Pref = scale * ((X * X) @ bank.T)
        gate = G * (8 * EPS32 * Pref + scale * (2 * delta[:, None] * (X @ bank.T) + delta[:, None] ** 2 * bank.sum(1)[None, :]))
        if log_mode == "db":
            y = DB_PER_LN * np.log(np.maximum(P, AMIN))
            glog = DB_PER_LN * gate / np.maximum(Pref, AMIN)
        else:
            y = np.log(P + log_eps)
            glog = gate / (Pref + log_eps)
        if fp32_emulation:
            y = y.astype(np.float32).astype(np.float64)
        glog = glog + LOG_ULPS * np.spacing(np.abs(y).astype(np.float32)).astype(np.float64)
        out["power"][b], out["log"][b], out["gate_power"][b], out["gate_log"][b] = P, y, gate, glog
        out["frame_max"][b] = y[:, :79].max(axis=1) if mutate == "max_79_bands" else y.max(axis=1)
        out["norm"][b] = norm
    return out


def _fp32_rows(clip, centres, lo, hi, pad_mode, win, pidx, bank, sub, scale) -> np.ndarray:
    """Mel power the way the kernel's arithmetic computes it: float32 windowed samples, each pair packed into one
    complex64 FFT and separated with the conjugate-symmetric partner, |X|^2 and the bank sum in float32."""
    x = (frame_samples(clip, centres, lo, hi, pad_mode).astype(np.float32) * win.astype(np.float32)[None, :])
    R = x.shape[0]
    P = np.zeros((R, bank.shape[0]))
    bank32 = bank.astype(np.float32)
    k = np.arange(FRAME // 2 + 1)
    for j in range(0, R, 2):
        a = x[j]
        b = x[j + 1] if j + 1 < R else np.zeros_like(a)
        Z = scipy.fft.fft((a + 1j * b).astype(np.complex64))
        Zc = np.conj(Z[(-k) % FRAME])
        A, Bs = (Z[k] + Zc) * np.float32(0.5), (Z[k] - Zc) * np.complex64(-0.5j)
        for r, S in ((j, A), (j + 1, Bs)):
            if r >= R:
                continue
            S = S[::sub].astype(np.complex64)
            p2 = (S.real * S.real + S.imag * S.imag).astype(np.float32)
            P[r] = (bank32 @ p2).astype(np.float32) * np.float32(scale)
    return P.astype(np.float32).astype(np.float64)


# ---- comparison ---------------------------------------------------------------------------------------------------------
def excess(got_log: np.ndarray, ref: Dict[str, np.ndarray]) -> np.ndarray:
    """|got - model| / gate per band (the stored log values); <= 1 passes."""
    return np.abs(np.asarray(got_log, np.float64) - ref["log"]) / ref["gate_log"]


def frame_max_excess(got_max: np.ndarray, ref: Dict[str, np.ndarray]) -> np.ndarray:
    """|got - model| / gate of each frame's loudest band."""
    arg = ref["log"].argmax(axis=-1)
    gate = np.take_along_axis(ref["gate_log"], arg[..., None], axis=-1)[..., 0]
    return np.abs(np.asarray(got_max, np.float64) - ref["frame_max"]) / gate


def worst(ratio: np.ndarray) -> str:
    """Where the largest ratio of a (B, R, M) array sits, for assertion messages."""
    i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    names = ("clip", "row", "band")[-len(i):] if len(i) <= 3 else [f"axis{a}" for a in range(len(i))]
    return ", ".join(f"{n} {int(v)}" for n, v in zip(names, i)) + f": {float(ratio[i]):.3g} x gate"


# ---- inputs ---------------------------------------------------------------------------------------------------------------
KINDS = ("noise", "silence_burst", "sine", "level_step", "speechlike", "loud_next_to_silence", "clipping", "tiny",
         "dc_offset", "chirp", "int16_speech")


def make_audio(kind: str, batch: int, n_samples: int, seed: int = 0) -> np.ndarray:
    """(B, L) float32 test audio: the kinds of oracle.make_inputs plus edge cases of the frontend's arithmetic."""
    if kind in ("noise", "silence_burst", "sine", "level_step", "speechlike", "silence"):
        return O.make_inputs(seed, batch, n_samples, kind)[0]
    rng = np.random.default_rng(seed + 7)
    t = np.arange(n_samples) / O.SAMPLE_RATE
    clips = []
    for b in range(batch):
        if kind == "loud_next_to_silence":
            # loud bursts a few hops long between stretches of digital silence: pairs of a loud and a silent frame
            a = np.zeros(n_samples)
            period = 533 * (5 + b)
            for s in range(period // 2, n_samples, period):
                w = min(533 * 2 + 17 * b, n_samples - s)
                a[s:s + w] = 0.9 * rng.standard_normal(w)
        elif kind == "clipping":
            a = np.clip(3.0 * np.sin(2 * np.pi * (300.0 + 50 * b) * t) + 0.5 * rng.standard_normal(n_samples), -1.0, 1.0)
        elif kind == "tiny":
            a = 1e-6 * (rng.standard_normal(n_samples) * (1 + 0.5 * np.sin(2 * np.pi * 0.7 * t + b)))
        elif kind == "dc_offset":
            a = 0.4 + 0.05 * rng.standard_normal(n_samples) + 0.1 * np.sin(2 * np.pi * 220.0 * t)
        elif kind == "chirp":
            a = 0.5 * scipy.signal.chirp(t, f0=0.0, t1=max(t[-1], 1e-3), f1=8000.0, method="linear", phi=90 * b)
        elif kind == "int16_speech":
            s = O.make_inputs(seed + b, 1, n_samples, "speechlike")[0][0].astype(np.float64)
            a = np.round(np.clip(s / max(np.abs(s).max(), 1e-9) * 0.7, -1, 1) * 32767) / 32768.0
        else:
            raise ValueError(kind)
        clips.append(a)
    return np.stack(clips).astype(np.float32)
