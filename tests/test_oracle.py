"""CPU tests: pin the oracle (oracle/koemorph_oracle.py) against

* the committed golden vectors produced by the unmodified reference
  (tests/golden/make_golden.py), and
* independent implementations of the librosa stage (torchaudio Slaney filterbank,
  torch.stft), because the reference has no fixture for that stage (parity unpinned there).
"""
import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O


def _run_oracle(spec, **kw):
    w = O.make_weights(spec["wseed"], spec["fps"], style=spec["style"])
    audio, eg = O.make_inputs(spec["iseed"], spec["B"], spec["L"], spec["kind"])
    if spec["mode"] == "single":
        return O.forward_single(w, audio, eg, fps=spec["fps"], return_attention=True, **kw)
    return O.forward_sequence(w, audio, eg, fps=spec["fps"], stride_frames=spec.get("stride", 1),
                              return_attention=True, **kw)


SINGLE = ["single_noise_init", "single_speech_stress", "single_burst_stress", "single_sine_stress",
          "single_step_stress", "single_silence_init", "single_short_clip", "single_long_clip", "single_60fps"]
SEQ = ["seq_clip_T1", "seq_13_frames", "seq_stride3", "seq_60fps", "seq_burst_edge"]


@pytest.mark.parametrize("name", SINGLE)
def test_oracle_matches_reference_single(golden, name):
    cases, data = golden
    out = _run_oracle(cases[name])
    np.testing.assert_allclose(out["blendshapes"].numpy(), data[f"{name}/blendshapes"], rtol=0, atol=2e-7)
    np.testing.assert_allclose(out["mel_attention_weights"].numpy(), data[f"{name}/mel_attention_weights"],
                               rtol=0, atol=2e-7)
    np.testing.assert_allclose(out["logmel"].numpy(), data[f"{name}/logmel"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(out["logmel_short"].numpy(), data[f"{name}/logmel_short"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(out["mel_blendshapes"].numpy(), data[f"{name}/mel_blendshapes"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(out["emotion_blendshapes"].numpy(), data[f"{name}/emotion_blendshapes"],
                               rtol=0, atol=1e-6)


@pytest.mark.parametrize("name", SEQ)
def test_oracle_matches_reference_sequence(golden, name):
    cases, data = golden
    out = _run_oracle(cases[name])
    ref = data[f"{name}/blendshapes"]
    assert out["blendshapes"].shape == ref.shape
    np.testing.assert_allclose(out["blendshapes"].numpy(), ref, rtol=0, atol=2e-7)
    n = data[f"{name}/mel_attention_weights"].shape[1]
    np.testing.assert_allclose(out["mel_attention_weights"].numpy()[:, :n], data[f"{name}/mel_attention_weights"],
                               rtol=0, atol=2e-7)


def test_oracle_matches_reference_20s_prefix(golden):
    """20 s clip (T_out = 345): the oracle recomputes the first 24 frames (the whole clip takes ~25 s)."""
    cases, data = golden
    spec = cases["seq_20s"]
    assert data["seq_20s/blendshapes"].shape == (1, 345, 52)
    w = O.make_weights(spec["wseed"], spec["fps"], style=spec["style"])
    audio, eg = O.make_inputs(spec["iseed"], spec["B"], spec["L"], spec["kind"])
    out = O.forward_sequence(w, audio, eg, max_frames=24)
    np.testing.assert_allclose(out["blendshapes"].numpy(), data["seq_20s/blendshapes"][:, :24], rtol=0, atol=2e-7)


def test_streaming_mel_matches_reference(golden):
    _, data = golden
    hop = int(data["streaming/hop"])
    assert hop == 532  # int(16000 / (1 / 0.0333)), mel_sliding_window.py:49-50 (SURVEY.md section 3.5)
    audio, _ = O.make_inputs(4242, 1, hop * 300, "speechlike")
    # after 300 hops of 532 the 136000-sample ring holds the last 136000 samples written, in order
    ring = audio[0, hop * 300 - 136000:]
    got = O.streaming_mel(ring, hop_length=hop)
    np.testing.assert_allclose(got, data["streaming/features"], rtol=0, atol=2e-5)
    got_b = O.power_to_db(O.melspectrogram(audio[0, :136000], hop_length=hop, pad_mode="reflect")).T
    np.testing.assert_allclose(got_b, data["streaming/batch_features"], rtol=0, atol=2e-5)


# ---- independent cross-checks of the librosa restatement (parity unpinned at this boundary) ----
def test_filterbank_vs_torchaudio():
    ta = pytest.importorskip("torchaudio")
    fb = O.mel_filterbank()
    assert fb.shape == (80, 513) and fb.dtype == np.float32
    ref = ta.functional.melscale_fbanks(513, 80.0, 8000.0, 80, 16000, norm="slaney", mel_scale="slaney").T.numpy()
    assert np.abs(fb - ref).max() < 5e-7
    assert int((fb > 0).sum()) == 992  # SURVEY.md section 7 probe
    # every bin feeds at most two (adjacent) filters: the triangle structure the CUDA epilogue relies on
    assert int((fb > 0).sum(axis=0).max()) == 2


def test_stft_vs_torch():
    audio, _ = O.make_inputs(3, 1, 20000, "speechlike")
    spec = O.stft(audio[0], hop_length=533)
    ref = torch.stft(torch.from_numpy(audio[0]).double(), 1024, hop_length=533,
                     window=torch.hann_window(1024, periodic=True, dtype=torch.float64), center=True,
                     pad_mode="constant", return_complex=True).numpy()
    assert spec.shape == ref.shape == (513, 1 + 20000 // 533)
    assert np.abs(spec - ref).max() < 1e-5 * np.abs(ref).max()


def test_frame_counts():
    # SURVEY.md section 8(a1): 30 fps clip -> 256 frames, window -> 257; 60 fps -> 512 / 513
    assert O.melspectrogram(np.zeros(136000, np.float32), hop_length=533).shape == (80, 256)
    assert O.melspectrogram(np.zeros(256 * 533, np.float32), hop_length=533).shape == (80, 257)
    assert O.melspectrogram(np.zeros(136000, np.float32), hop_length=266).shape == (80, 512)
    assert O.melspectrogram(np.zeros(512 * 266, np.float32), hop_length=266).shape == (80, 513)


def test_known_answers():
    # silence: every value hits amin, ref == amin too -> 0 dB everywhere -> normalised 1.0
    lt, st = O.extract_mel_features(np.zeros((1, 136000), np.float32))
    assert np.all(lt == 1.0) and np.all(st == 1.0)
    # pure 1 kHz tone: the loudest band is the one whose centre is nearest 1 kHz, max is exactly 1.0,
    # and far-away bands sit on the -80 dB clamp (normalised 0.0)
    t = np.arange(136000) / 16000.0
    lt, _ = O.extract_mel_features((0.5 * np.sin(2 * np.pi * 1000.0 * t)).astype(np.float32)[None])
    centres = O.mel_to_hz(np.linspace(O.hz_to_mel(80.0), O.hz_to_mel(8000.0), 82))[1:-1]
    assert lt.max() == 1.0
    assert abs(int(lt[0, 100].argmax()) - int(np.abs(centres - 1000.0).argmin())) <= 1
    assert lt[0, 100].min() == 0.0
    # index tables (dual_stream_attention.py:44-45)
    assert O.MOUTH_INDICES == list(range(14, 41)) + [51] and len(O.EXPRESSION_INDICES) == 24


def test_fp64_oracle_agrees_with_fp32():
    w = O.make_weights(5, 30, style="stress")
    audio, eg = O.make_inputs(6, 2, 136000, "speechlike")
    a = O.forward_single(w, audio, eg)
    b = O.forward_single(w, audio, eg, dtype=torch.float64)
    assert (a["blendshapes"].double() - b["blendshapes"]).abs().max() < 1e-6
    assert (a["sigmoid"].double() - b["sigmoid"]).abs().max() < 1e-5


def test_librosa_stage_vs_transformers_audio_utils():
    """A third independent implementation of the librosa stage: transformers.audio_utils (numpy; written to reproduce
    librosa's Slaney filterbank, centred STFT and power_to_db for the Whisper-family feature extractors).  Filterbank,
    mel power and the dB conversion of the oracle's restatement against it, on a speech-like clip."""
    A = pytest.importorskip("transformers.audio_utils")
    fb = A.mel_filter_bank(num_frequency_bins=513, num_mel_filters=80, min_frequency=80.0, max_frequency=8000.0,
                           sampling_rate=16000, norm="slaney", mel_scale="slaney")            # (513, 80) float64
    ours = O.mel_filterbank().astype(np.float64)                                              # (80, 513) float32 weights
    assert np.abs(ours - fb.T).max() <= 2e-7 * fb.max()
    assert ((ours > 0) == (fb.T > 1e-12)).all()

    audio, _ = O.make_inputs(17, 1, 40000, "speechlike")
    y = audio[0]
    window = A.window_function(1024, "hann", periodic=True) if hasattr(A, "window_function") else O.hann_window(1024)
    mel = A.spectrogram(y.astype(np.float64), window, frame_length=1024, hop_length=533, power=2.0, center=True,
                        pad_mode="constant", mel_filters=fb, mel_floor=0.0, dtype=np.float64)    # (80, T)
    ref = O.melspectrogram(y, hop_length=533, exact=True)                                       # float64 restatement
    assert mel.shape == ref.shape == (80, 1 + 40000 // 533)
    # (librosa -- and the restatement -- keep the filterbank in float32; audio_utils keeps float64: 6e-8 relative)
    assert np.abs(mel - ref).max() <= 2e-7 * ref.max()

    db = A.power_to_db(mel, reference=mel.max(), min_value=1e-10, db_range=80.0)
    ours_db = O.power_to_db(ref.astype(np.float64))
    assert np.abs(db - ours_db).max() <= 2e-5   # dB; 2e-7 relative in power is 1e-6 dB, the rest is the -80 dB clamp edge
