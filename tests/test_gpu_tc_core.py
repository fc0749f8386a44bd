"""The bf16 tensor-core core (dual_stream_tc_kernel) against the float64 model of its own arithmetic
(oracle/tc_core_model.py), on every window: mouth blendshapes, pre-fusion mouth sigmoid and head-averaged attention.

test_gpu_parity.py compares this core with the fp32 reference at gates wide enough for the bf16 design error; here the
model rounds where the kernel rounds, so what is left is the kernel's fp32 accumulation order and its fast exp / rsqrt
flipping single bf16 roundings, and the gates (oracle.tc_core_model.GATES) sit just above that floor.  The forward cases
feed the model the kernel's own frontend rows (plain rows, edge variants and frame maxima), so the frontend's own
error stays out of the comparison.

Largest deviations measured on a B200 (power limit 1000 W), per weight style and case group (out / sigmoid / attention):
  stress  standalone 5.9e-6 / 1.2e-4 / 1.3e-4   windows 3.6e-6 / 9.7e-5 / 5.5e-5   batches 6.4e-6 / 1.7e-4 / 5.6e-5
  init    standalone 1.9e-7 / 1.0e-5 / 8.5e-8   windows 3.7e-7 / 1.9e-5 / 1.4e-7   batches 4.9e-7 / 2.5e-5 / 2.4e-7
  offset  standalone 1.3e-5 / 3.8e-4 / 7.5e-4   windows 1.1e-5 / 3.6e-4 / 2.8e-4   batches 1.0e-5 / 2.2e-4 / 6.8e-5
The offset style's excess over stress comes from the kernel's one-pass LayerNorm variance, E[z^2] - mean^2 in fp32,
which cancels when the encoder output sits off zero mean; windows of one to three frames show it most.  With the
activations truncated to bf16 instead of rounded (pack8_bf16), this test fails on every stress and init case group
(stress up to 1.7e-4 / 2.5e-3 / 2.2e-3, init 6.0e-6 / 3.2e-4 / 1.8e-6) while the tests of
test_gpu_parity.py that run the bf16 core still pass.
"""
import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O
from oracle import tc_core_model as M

pytestmark = pytest.mark.gpu

MOUTH = O.MOUTH_INDICES
# weight style: (seed, make_weights style, added to the encoder bias); the offset moves every encoder output away from
# zero mean, where the LayerNorm variance loses the most to cancellation
STYLES = {"stress": (21, "stress", 0.0), "init": (1234, "init", 0.0), "offset": (21, "stress", 3.0)}


@pytest.fixture(scope="module")
def K():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import koemorph_b200
    from koemorph_b200 import _lib
    _lib.load()
    return koemorph_b200


_cache = {}


def _weights(style, fps):
    key = (style, fps)
    if key not in _cache:
        seed, base, offset = STYLES[style]
        w = O.make_weights(seed, fps, style=base)
        w["dual_stream_attention.mel_channel_encoder.bias"] = w["dual_stream_attention.mel_channel_encoder.bias"] + np.float32(offset)
        _cache[key] = (w, M.tc_weights(w, device="cuda"))
    return _cache[key]


def _check(style, case, got, want):
    """got / want: (sigmoid, blendshapes, attention) over the same windows, mouth entries only; None: not compared."""
    dev = [0.0 if g is None else float((g.double() - x).abs().max()) for g, x in zip(got, want)]
    sig, out, att = dev
    print(f"tc-core {style:6s} {case:40s} out {out:.3e} sig {sig:.3e} att {att:.3e}")
    gates = M.GATES[style]
    assert out <= gates[0] and sig <= gates[1] and att <= gates[2], \
        f"{case}: out {out:.3e} sig {sig:.3e} att {att:.3e} against gates {gates}"


def _model(K, w, fps, stride=None):
    """The sequence model with this stride, or (None) the single-window model; bf16 core."""
    kw = dict(target_fps=fps, mel_sequence_length=256 if fps == 30 else 512)
    m = K.SimplifiedDualStreamModel(**kw) if stride is None else K.SequentialDualStreamModel(stride_frames=stride, **kw)
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m = m.cuda().eval()
    m.precision = "bf16"
    return m


def _window_rows(power, fmax, n_out, stride, T, n_edge):
    """The rows the kernel reads for each window (koe_dual_stream_windows): [B * n_out, T, 80] dB and [B * n_out, T]."""
    k = torch.arange(n_out, device=power[0].device)[:, None] * stride + torch.arange(T, device=power[0].device)
    db, fm = power[0][:, k].clone(), fmax[0][:, k].clone()               # [B, n_out, T, (80)]
    for m in range(n_edge):
        db[:, :, m], fm[:, :, m] = power[1 + 2 * m], fmax[1 + 2 * m]
        db[:, :, T - 1 - m], fm[:, :, T - 1 - m] = power[2 + 2 * m], fmax[2 + 2 * m]
    return db.reshape(-1, T, 80), fm.reshape(-1, T)


def _core_windows(m, audio, eg, n_out, stride, T, n_edge):
    """The frontend buffers a forward builds, then the core on them through koe_dual_stream_windows (with attention)."""
    fe, hop = m._frontend(audio.device), m.hop_length
    n_frames = (n_out - 1) * stride + T
    p0, f0 = fe.power(audio, hop, n_frames)
    power, fmax = [p0], [f0]
    for j in range(n_edge):
        for off, lo, hi in ((j, -j, None), (T - 1 - j, None, j)):
            p, f = fe.power(audio, hop, n_out, frame_offset=off, frame_step=stride, lo_rel=lo, hi_rel=hi)
            power.append(p)
            fmax.append(f)
    B = audio.shape[0]
    out, sig, attn = m._core_windows(power, fmax, n_edge, B, n_frames, n_out, stride, T,
                                     m._check_egemaps(eg, B, audio.device), True)
    db, fm = _window_rows(power, fmax, n_out, stride, T, n_edge)
    return (sig[..., MOUTH].reshape(-1, 28), out[..., MOUTH].reshape(-1, 28), attn.reshape(-1, 28, 80)), db, fm


STANDALONE = [(256, T) for T in (1, 2, 3, 13, 47, 48, 49, 255, 256, 300)] + [(512, T) for T in (1, 3, 97, 511, 512, 700)]


@pytest.mark.parametrize("style", list(STYLES))
@pytest.mark.parametrize("mel_seq,T", STANDALONE)
def test_standalone_core_vs_model(K, style, mel_seq, T):
    """koe_dual_stream_features (prenormalised features, staged by the SIMT warps): windows shorter than the short-term
    detail, around the 8-frame K chunks and the 48-row stages, equal to and longer than mel_sequence_length."""
    w, W = _weights(style, 30 if mel_seq == 256 else 60)
    core = K.DualStreamCrossAttention(mel_sequence_length=mel_seq).cuda().eval()
    core.load_state_dict({k[len("dual_stream_attention."):]: v for k, v in O.model_state_dict(w).items()
                          if k.startswith("dual_stream_attention.")})
    core.precision = "bf16"
    g = torch.Generator(device="cuda").manual_seed(mel_seq + T)
    lt = torch.rand(5, T, 80, device="cuda", generator=g)
    st = torch.rand(5, 3, 80, device="cuda", generator=g)
    res = core(lt, st, torch.randn(5, 256, device="cuda", generator=g), return_attention=True)
    got = (res["mel_blendshapes"][:, MOUTH], res["blendshapes"][:, MOUTH], res["mel_attention_weights"])
    _check(style, f"standalone K={mel_seq + 3} T={T}", got, M.forward(W, lt, st))


# fps, stride, audio kind, "seq": n windows of a sequence / "single": one window over a whole clip of n frames
FORWARD = [
    (30, 1, "speechlike", "seq", 6), (30, 3, "noise", "seq", 5), (60, 1, "speechlike", "seq", 6), (60, 3, "sine", "seq", 4),
    (30, 2, "level_step", "seq", 5), (60, 1, "silence_burst", "seq", 3), (30, 1, "silence", "seq", 2),
    (30, 1, "quiet", "seq", 3),
    (30, 1, "speechlike", "single", 1), (30, 1, "speechlike", "single", 2), (30, 1, "noise", "single", 3),
    (30, 1, "speechlike", "single", 13), (30, 1, "level_step", "single", 97), (30, 1, "silence", "single", 150),
    (60, 1, "speechlike", "single", 2), (60, 1, "noise", "single", 203), (60, 1, "quiet", "single", 400),
]


@pytest.mark.parametrize("style", list(STYLES))
@pytest.mark.parametrize("fps,stride,kind,shape,n", FORWARD, ids=[f"{a}fps-s{b}-{c}-{d}{e}" for a, b, c, d, e in FORWARD])
def test_windows_core_vs_model(K, style, fps, stride, kind, shape, n):
    """koe_dual_stream_windows (mel rows by TMA in 48-row stages, normalised in the kernel): sequences with one (30 fps)
    and two (60 fps) edge variants per side and strides that overlap windows; single windows over whole clips of n frames
    (a partial last stage, row counts that are not a multiple of 8, fewer than three frames); silence, quiet clips and
    level steps, where frames sit on the -80 dB floor."""
    w, W = _weights(style, fps)
    hop, win = 16000 // fps, 256 if fps == 30 else 512
    if shape == "seq":
        m = _model(K, w, fps, stride)
        L = (win + (n - 1) * stride) * hop + 100
        n_out, T, n_edge = n, win + 1, -(-512 // hop)
        assert m.num_output_frames(L) == n_out
    else:
        m = _model(K, w, fps)
        L = (n - 1) * hop + 100
        n_out, T, n_edge = 1, n, 0
    audio, eg = O.make_inputs(fps + n, 3, L, "noise" if kind == "quiet" else kind)
    if kind == "quiet":
        audio *= 1e-4
    got, db, fm = _core_windows(m, torch.from_numpy(audio).cuda(), torch.from_numpy(eg).cuda(), n_out, stride, T, n_edge)
    _check(style, f"windows {fps} fps stride {stride} {kind} {shape} {n}", got, M.forward(W, db=db, fmax=fm))


@pytest.mark.parametrize("style", list(STYLES))
@pytest.mark.parametrize("fps,n_clips", [(30, 512), (30, 2100), (60, 512)])
def test_large_batches_vs_model(K, style, fps, n_clips):
    """Several windows per CTA (the next window staged under the S / VT GEMMs at 30 fps), and the fused forward, whose
    core starts its first rounds of windows on the frontend's early-release flag: every window against the model, run
    in float64 on the device."""
    w, W = _weights(style, fps)
    m = _model(K, w, fps, 1)
    T = m.window_frames + 1
    g = torch.Generator(device="cuda").manual_seed(n_clips + fps)
    audio = 0.1 * torch.randn(n_clips, 136000, device="cuda", generator=g)
    audio[::7] *= 1e-3
    eg = torch.randn(n_clips, 264, device="cuda", generator=g)
    got, db, fm = _core_windows(m, audio, eg, 1, 1, T, 0)
    want = M.forward(W, db=db, fmax=fm)
    _check(style, f"batch {n_clips} at {fps} fps, windows", got, want)
    fused = m(audio, egemaps=eg)["blendshapes"][:, 0, MOUTH]
    _check(style, f"batch {n_clips} at {fps} fps, fused forward", (None, fused, None), want)
