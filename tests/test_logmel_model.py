"""The float64 model of the log-mel frontend (oracle/logmel_model.py) on the CPU: with its mutations off it is the
reference (librosa's STFT + mel restated in oracle.koemorph_oracle, float64 torch.stft for the torchaudio flavour,
explicit zeroing for the window-edge masks), its gates pass fp32 arithmetic with a factor 4 to spare, and each
plausible kernel bug of logmel_model.MUTATIONS exceeds them by at least 5x on some input.  tests/test_gpu_logmel.py
applies the same gates to every row the library computes."""
import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O
from oracle import logmel_model as M

BANK = O.mel_filterbank()   # the float32 Slaney bank the library builds (checked against it on the GPU)


@pytest.mark.parametrize("pad_mode", ["constant", "reflect"])
@pytest.mark.parametrize("hop", [533, 266, 532])
def test_model_is_the_float64_reference(pad_mode, hop):
    audio = M.make_audio("speechlike", 2, 30001, seed=hop)
    n = 1 + audio.shape[1] // hop
    got = M.launch(audio, hop, n, BANK, pad_mode=pad_mode)
    for b in range(2):
        ref = O.melspectrogram(audio[b], hop_length=hop, pad_mode=pad_mode, exact=True).T
        assert np.abs(got["power"][b] - ref).max() <= 1e-12 * ref.max(), (b, "power")
        rel = np.abs(got["power"][b] - ref) / ref
        assert rel.max() <= 1e-12, f"clip {b}: relative {rel.max():.3e}"
        db = 10 * np.log10(np.maximum(ref, 1e-10))
        assert np.abs(got["log"][b] - db).max() <= 1e-12 * np.abs(db).max()
        np.testing.assert_array_equal(got["frame_max"][b], got["log"][b].max(axis=1))


def test_model_of_the_512_point_htk_flavour_is_torch_stft():
    """n_fft 512 centred in the 1024-point transform, a 400-point window centred in the 512-point frame, the power
    normalised by sum(window^2), the HTK bank, ln(p + eps): float64 torch.stft with reflect padding times the bank."""
    hop, eps = 533, 1e-8
    audio = M.make_audio("chirp", 2, 20000, seed=1)
    bank = M.htk_bank(n_fft=512)
    n = 1 + audio.shape[1] // hop
    got = M.launch(audio, hop, n, bank, pad_mode="reflect", n_fft=512, win_length=400, window_normalized=True,
                   log_mode="ln", log_eps=eps)
    win = torch.hann_window(400, periodic=True, dtype=torch.float64)
    spec = torch.stft(torch.from_numpy(audio).double(), 512, hop, 400, win, center=True, pad_mode="reflect",
                      return_complex=True)
    ref = (torch.from_numpy(bank) @ (spec.abs() ** 2 / (win ** 2).sum())).transpose(1, 2).numpy()
    assert np.abs(got["power"] - ref).max() <= 1e-12 * ref.max()
    np.testing.assert_allclose(got["log"], np.log(ref + eps), rtol=0, atol=1e-10)


def test_banks_are_the_library_formulas():
    """slaney_bank is librosa's bank (the oracle's float32 one, within float32 rounding); htk_bank is torchaudio's."""
    np.testing.assert_allclose(M.slaney_bank(), O.mel_filterbank(), rtol=0, atol=1.2e-7 * O.mel_filterbank().max())
    torchaudio = pytest.importorskip("torchaudio")
    dtype = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)     # torchaudio builds the bank in the default dtype
    try:
        ref = torchaudio.functional.melscale_fbanks(257, 80.0, 8000.0, 80, 16000, norm=None, mel_scale="htk")
    finally:
        torch.set_default_dtype(dtype)
    assert ref.dtype == torch.float64
    np.testing.assert_allclose(M.htk_bank(n_fft=512), ref.numpy().T, rtol=0, atol=1e-12)


@pytest.mark.parametrize("lo_rel,hi_rel", [(0, None), (-1, None), (None, 0), (None, 1), (-1, 2)])
def test_masks_equal_explicit_zeroing(lo_rel, hi_rel):
    """lo_rel / hi_rel: each frame sees zeros before (g + lo_rel) * hop and from (g + hi_rel) * hop on."""
    hop, off, step = 266, 3, 5
    audio = M.make_audio("noise", 1, 20000, seed=2)
    got = M.launch(audio, hop, 6, BANK, frame_offset=off, frame_step=step, sample_offset=40, lo_rel=lo_rel, hi_rel=hi_rel)
    for j in range(6):
        g = off + j * step
        a = audio.copy()
        if lo_rel is not None:
            a[:, :max(0, 40 + (g + lo_rel) * hop)] = 0
        if hi_rel is not None:
            a[:, max(0, 40 + (g + hi_rel) * hop):] = 0
        one = M.launch(a, hop, 1, BANK, frame_offset=g, sample_offset=40)
        np.testing.assert_allclose(got["power"][0, j], one["power"][0, 0], rtol=1e-12, atol=0)


# launch geometries of the GPU suite (keyword arguments of M.launch besides audio / bank), on 136000-sample clips
GEOMETRIES = {
    "plain 533": dict(hop=533, n_frames=256),
    "plain 266 odd": dict(hop=266, n_frames=511),
    "window start": dict(hop=533, n_frames=40, frame_offset=0, frame_step=3, lo_rel=0),
    "window end 60 fps": dict(hop=266, n_frames=40, frame_offset=510, frame_step=2, hi_rel=1),
    "reflect 532": dict(hop=532, n_frames=256, pad_mode="reflect"),
}
HTK = dict(hop=533, n_frames=256, pad_mode="reflect", n_fft=512, window_normalized=True, log_mode="ln", log_eps=1e-8)


def _bank(geom):
    return M.htk_bank(n_fft=512).astype(np.float32) if geom.get("n_fft") == 512 else BANK


@pytest.mark.parametrize("kind", M.KINDS)
def test_fp32_emulation_stays_under_a_quarter_of_the_gate(kind):
    audio = M.make_audio(kind, 1, 136000, seed=11)
    for name, geom in [*GEOMETRIES.items(), ("htk ln 512", HTK)]:
        base = M.launch(audio, bank=_bank(geom), **geom)
        emu = M.launch(audio, bank=_bank(geom), fp32_emulation=True, **geom)
        r = M.excess(emu["log"], base)
        assert r.max() <= 0.25, f"{kind}, {name}: {M.worst(r)}"


# which launches can show a mutation at all (the mask bug needs masks, the padding bug reflect padding)
_MUTATION_GEOMS = {"mask_off_by_one": ("window start", "window end 60 fps"), "symmetric_pad": ("reflect 532",)}


@pytest.mark.parametrize("mutation", M.MUTATIONS)
def test_each_mutation_exceeds_the_gate_fivefold(mutation):
    geoms = _MUTATION_GEOMS.get(mutation, ("plain 533", "plain 266 odd"))
    best = (0.0, "")
    for kind in M.KINDS:
        audio = M.make_audio(kind, 1, 136000, seed=11)
        for name in geoms:
            geom = GEOMETRIES[name]
            base = M.launch(audio, bank=BANK, **geom)
            mut = M.launch(audio, bank=BANK, mutate=mutation, **geom)
            r = M.frame_max_excess(mut["frame_max"], base) if mutation == "max_79_bands" else M.excess(mut["log"], base)
            if r.max() > best[0]:
                best = (float(r.max()), f"{kind}, {name}")
            if best[0] >= 5:
                return
    pytest.fail(f"{mutation}: at most {best[0]:.3g} x the gate ({best[1]})")
