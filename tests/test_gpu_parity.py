"""GPU parity tests (-m gpu): the CUDA path, reached through the C ABI, against the CPU oracle and the
golden vectors of the unmodified reference.

Tolerances (BASELINE.md section 5 / north_star):
  * log-mel, normalised (dB + 80) / 80:   |d| <= 1e-4 * |ref| + 2e-5   (1e-4 relative; the absolute floor
    covers values on the -80 dB clamp where "relative" is undefined)
  * blendshapes, fp32 path:               |d| <= 1e-3 absolute (north_star) -- and, because random-init outputs are
    ~0.01, the tighter gates we add: <= 2e-6 on the output, <= 2e-5 on the pre-fusion sigmoid, <= 2e-5 on the
    head-averaged attention weights.
"""
import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O

pytestmark = pytest.mark.gpu

LOGMEL_RTOL, LOGMEL_ATOL = 1e-4, 2e-5
OUT_ATOL, SIG_ATOL, ATTN_ATOL = 2e-6, 2e-5, 2e-5


@pytest.fixture(scope="module")
def K():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import koemorph_b200
    from koemorph_b200 import _lib
    _lib.load()  # fails loudly if the CUDA library is missing
    return koemorph_b200


def _model(K, spec, sequential):
    w = O.make_weights(spec["wseed"], spec["fps"], style=spec["style"])
    kw = dict(target_fps=spec["fps"], mel_sequence_length=256 if spec["fps"] == 30 else 512)
    m = (K.SequentialDualStreamModel(stride_frames=spec.get("stride", 1), **kw) if sequential
         else K.SimplifiedDualStreamModel(**kw))
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    return m.cuda().eval(), w


def _inputs(spec):
    audio, eg = O.make_inputs(spec["iseed"], spec["B"], spec["L"], spec["kind"])
    return torch.from_numpy(audio).cuda(), torch.from_numpy(eg).cuda()


def _close(got, ref, rtol, atol, what):
    got = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, np.float64)
    ref = ref.detach().cpu().double().numpy() if torch.is_tensor(ref) else np.asarray(ref, np.float64)
    assert got.shape == ref.shape, f"{what}: shape {got.shape} vs {ref.shape}"
    err = np.abs(got - ref) - (atol + rtol * np.abs(ref))
    assert err.max() <= 0, f"{what}: max |d| = {np.abs(got - ref).max():.3e} (excess {err.max():.3e})"


SINGLE = ["single_noise_init", "single_speech_stress", "single_burst_stress", "single_sine_stress",
          "single_step_stress", "single_silence_init", "single_short_clip", "single_long_clip", "single_60fps"]
SEQ = ["seq_clip_T1", "seq_13_frames", "seq_20s", "seq_stride3", "seq_60fps", "seq_burst_edge"]


def test_filterbank_matches_oracle(K):
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    fb = LogMelFrontend.get("cuda").filterbank()
    ref = O.mel_filterbank()
    assert np.abs(fb - ref).max() <= 1.2e-7 * ref.max()
    assert ((fb > 0) == (ref > 0)).all()


def test_default_bank_is_unrolled_and_generic_bank_agrees(K):
    """The path's filterbank takes the unrolled kernel (a silent fall-back to the generic loops would only show up as a
    slower bench); a bank with other band edges takes the generic kernel, and both agree with the float64 oracle."""
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    assert LogMelFrontend.get("cuda").uses_unrolled_bank()
    other = LogMelFrontend.get("cuda", f_min=60.0, f_max=7600.0)
    assert not other.uses_unrolled_bank()
    audio, _ = O.make_inputs(77, 2, 40000, "speechlike")
    for fe, (fmin, fmax) in ((LogMelFrontend.get("cuda"), (80.0, 8000.0)), (other, (60.0, 7600.0))):
        db, fmx = fe.power(torch.from_numpy(audio).cuda(), 533, 76)
        db = db.cpu().double().numpy()
        fb = O.mel_filterbank(fmin=fmin, fmax=fmax).astype(np.float64)
        assert np.abs(fe.filterbank() - fb).max() <= 1.2e-7 * fb.max()
        for b in range(2):
            spec = np.abs(O.stft(audio[b], hop_length=533, exact=True)) ** 2
            ref = (fb @ spec).T
            big = ref > 1e-6 * ref.max()
            assert np.abs(db[b] - 10 * np.log10(np.maximum(ref, 1e-10)))[big].max() < 8.7e-4
            np.testing.assert_allclose(fmx[b].cpu().numpy(), db[b].max(axis=1), rtol=1e-6)


@pytest.mark.parametrize("name", SINGLE)
def test_logmel_vs_golden(K, golden, name):
    cases, data = golden
    spec = cases[name]
    m, _ = _model(K, spec, False)
    audio, _ = _inputs(spec)
    lt, st = m.extract_mel_features(audio)
    _close(lt, data[f"{name}/logmel"], LOGMEL_RTOL, LOGMEL_ATOL, "long-term log-mel")
    _close(st, data[f"{name}/logmel_short"], LOGMEL_RTOL, LOGMEL_ATOL, "short-term log-mel")


@pytest.mark.parametrize("kind", ["noise", "speechlike", "level_step", "sine", "silence_burst"])
def test_mel_power_vs_float64_oracle(K, kind):
    """koe_logmel_power (mel power in dB, before the reference is subtracted) against the float64 restatement."""
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    audio, _ = O.make_inputs(31, 3, 136000, kind)
    fe = LogMelFrontend.get("cuda")
    db, fmax = fe.power(torch.from_numpy(audio).cuda(), 533, 256)
    db = db.cpu().double().numpy()
    for b in range(3):
        ref = O.melspectrogram(audio[b], hop_length=533, exact=True).T
        ref_db = 10 * np.log10(np.maximum(ref, 1e-10))
        # bands within 60 dB of the clip peak: 2e-4 relative in power = 8.7e-4 dB
        big = ref > 1e-6 * ref.max()
        assert np.abs(db[b] - ref_db)[big].max() < 8.7e-4
        # everything else: absolute error in power below 2e-6 of the clip peak
        assert np.abs(10 ** (db[b] / 10) - np.maximum(ref, 1e-10)).max() <= 2e-6 * max(ref.max(), 1e-10)
        np.testing.assert_allclose(fmax[b].cpu().numpy(), db[b].max(axis=1), rtol=1e-6)


@pytest.mark.parametrize("name", SINGLE)
def test_forward_single_vs_golden(K, golden, name):
    cases, data = golden
    spec = cases[name]
    m, _ = _model(K, spec, False)
    audio, eg = _inputs(spec)
    out = m(audio, return_attention=True, egemaps=eg)
    _close(out["blendshapes"], data[f"{name}/blendshapes"], 0, OUT_ATOL, "blendshapes")
    _close(out["mel_blendshapes"], data[f"{name}/mel_blendshapes"], 0, SIG_ATOL, "mel_blendshapes")
    _close(out["emotion_blendshapes"], data[f"{name}/emotion_blendshapes"], 0, SIG_ATOL, "emotion_blendshapes")
    _close(out["mel_attention_weights"], data[f"{name}/mel_attention_weights"], 0, ATTN_ATOL, "mel attention")
    assert out["emotion_attention_weights"].shape == (spec["B"], 24, 1)
    assert bool((out["emotion_attention_weights"] == 1).all())
    # without return_attention only the blendshapes come back, and they are identical
    m.reset_temporal_state()
    out2 = m(audio, egemaps=eg)
    assert set(out2) == {"blendshapes"} and torch.equal(out2["blendshapes"], out["blendshapes"])


@pytest.mark.parametrize("name", SEQ)
def test_forward_sequence_vs_golden(K, golden, name):
    cases, data = golden
    spec = cases[name]
    m, _ = _model(K, spec, True)
    audio, eg = _inputs(spec)
    out = m(audio, return_attention=True, egemaps=eg)
    ref = data[f"{name}/blendshapes"]
    assert out["num_frames"] == ref.shape[1] and out["fps"] == spec["fps"]
    _close(out["blendshapes"], ref, 0, OUT_ATOL, "sequence blendshapes")
    n = data[f"{name}/mel_attention_weights"].shape[1]
    _close(out["mel_attention_weights"][:, :n], data[f"{name}/mel_attention_weights"], 0, ATTN_ATOL, "mel attention")
    assert out["emotion_attention_weights"].shape == (spec["B"], ref.shape[1], 24, 1)


def test_core_standalone_vs_oracle(K):
    """DualStreamCrossAttention.forward on ready-made features, T shorter / equal / longer than 256."""
    w = O.make_weights(21, 30, style="stress")
    core = K.DualStreamCrossAttention().cuda().eval()
    core.load_state_dict({k[len("dual_stream_attention."):]: v for k, v in O.model_state_dict(w).items()
                          if k.startswith("dual_stream_attention.")})
    rng = np.random.default_rng(5)
    for T in (100, 256, 300):
        lt = rng.uniform(0, 1, (4, T, 80)).astype(np.float32)
        st = rng.uniform(0, 1, (4, 3, 80)).astype(np.float32)
        emo = rng.standard_normal((4, 256)).astype(np.float32)
        ref = O.dual_stream_core(w, lt, st, emo, return_attention=True)
        out = core(torch.from_numpy(lt).cuda(), torch.from_numpy(st).cuda(), torch.from_numpy(emo).cuda(),
                   return_attention=True)
        _close(out["blendshapes"], ref["blendshapes"], 0, OUT_ATOL, f"core T={T}")
        _close(out["mel_attention_weights"], ref["mel_attention_weights"], 0, ATTN_ATOL, f"attn T={T}")
        _close(out["mel_blendshapes"], ref["mel_blendshapes"], 0, SIG_ATOL, f"sigmoid T={T}")


@pytest.mark.parametrize("T", [1, 2, 31, 32, 33, 345, 1000])
def test_ema_scan_vs_oracle(K, T):
    from koemorph_b200 import _lib
    x = torch.rand(5, T, 52, dtype=torch.float32)
    alpha = 0.6899744811276125
    ref = O.ema_smooth(x.double(), alpha)
    y = x.cuda().clone()
    state = torch.zeros(5, 52, device="cuda")
    _lib.check(_lib.load().koe_ema_scan(y.data_ptr(), 5, T, alpha, state.data_ptr(), 0, _lib.stream_ptr()))
    _close(y, ref, 1e-6, 1e-7, "ema scan")
    _close(state, ref[:, -1], 1e-6, 1e-7, "ema state")
    # continuing from a state == one long scan
    y2 = x.cuda().clone()
    cut = max(1, T // 3)
    st = torch.zeros(5, 52, device="cuda")
    a, b = y2[:, :cut].contiguous(), y2[:, cut:].contiguous()
    _lib.check(_lib.load().koe_ema_scan(a.data_ptr(), 5, cut, alpha, st.data_ptr(), 0, _lib.stream_ptr()))
    if T - cut > 0:
        _lib.check(_lib.load().koe_ema_scan(b.data_ptr(), 5, T - cut, alpha, st.data_ptr(), 1, _lib.stream_ptr()))
    _close(torch.cat([a, b], 1), ref, 1e-6, 1e-7, "ema scan with carried state")


def test_stateful_smoothing_across_calls(K, golden):
    """SimplifiedDualStreamModel keeps an EMA across forward calls (reference :341-368)."""
    cases, _ = golden
    spec = cases["single_speech_stress"]
    m, w = _model(K, spec, False)
    audio, eg = _inputs(spec)
    a2, e2 = O.make_inputs(999, spec["B"], spec["L"], "noise")
    r1 = O.forward_single(w, audio.cpu().numpy(), eg.cpu().numpy())["blendshapes"]
    r2 = O.forward_single(w, a2, e2)["blendshapes"]
    alpha = O.smoothing_alpha(w)
    o1 = m(audio, egemaps=eg)["blendshapes"]
    o2 = m(torch.from_numpy(a2).cuda(), egemaps=torch.from_numpy(e2).cuda())["blendshapes"]
    _close(o1, r1, 0, OUT_ATOL, "first call passes through")
    _close(o2, alpha * r2 + (1 - alpha) * r1, 0, OUT_ATOL, "second call is smoothed")
    m.reset_temporal_state()
    _close(m(torch.from_numpy(a2).cuda(), egemaps=torch.from_numpy(e2).cuda())["blendshapes"], r2, 0, OUT_ATOL,
           "reset")


def test_full_size_properties(K):
    """BASELINE config 1 size (512 clips x 8.5 s): properties that need no oracle run.

    * clips are independent: a clip's output does not depend on its batch neighbours or position;
    * the dB reference is the clip's own max, so scaling a clip by 2^k changes nothing up to the rounding of
      log10f(16 p) - log10f(16 ref) versus log10f(p) - log10f(ref);
    * a small batch cut out of the big one is checked against the oracle."""
    spec = dict(wseed=1235, style="stress", fps=30)
    m, w = _model(K, spec, True)
    B = 512
    g = torch.Generator(device="cuda").manual_seed(7)
    audio = 0.1 * torch.randn(B, 136000, device="cuda", generator=g)
    eg = torch.randn(B, 264, device="cuda", generator=g)
    out = m(audio, egemaps=eg)["blendshapes"]
    assert out.shape == (B, 1, 52) and bool(torch.isfinite(out).all()) and float(out.min()) >= 0 and float(out.max()) <= 1
    perm = torch.randperm(B, device="cuda", generator=g)
    out_p = m(audio[perm].contiguous(), egemaps=eg[perm].contiguous())["blendshapes"]
    assert torch.equal(out_p, out[perm])
    out_s = m((audio * 4.0).contiguous(), egemaps=eg)["blendshapes"]
    _close(out_s, out, 0, 5e-7, "scale invariance")
    sub = [0, 17, 255, 511]
    ref = O.forward_sequence(w, audio[sub].cpu().numpy(), eg[sub].cpu().numpy())["blendshapes"]
    _close(out[sub], ref, 0, OUT_ATOL, "full-size batch vs oracle")


def test_argument_validation(K):
    m = K.SequentialDualStreamModel().cuda()
    a = torch.zeros(2, 136000, device="cuda")
    with pytest.raises(RuntimeError, match="egemaps is required"):
        m(a)
    with pytest.raises(TypeError):
        m(a.double(), egemaps=torch.zeros(2, 264, device="cuda"))
    with pytest.raises(ValueError):
        m(a, egemaps=torch.zeros(3, 264, device="cuda"))
    with pytest.raises(ValueError):
        m(torch.zeros(136000, device="cuda"), egemaps=torch.zeros(1, 264, device="cuda"))
    out = m(a, egemaps=torch.zeros(2, 3, 88, device="cuda"))
    assert out["blendshapes"].shape == (2, 1, 52)


# ---- tcgen05 path (precision "bf16": bf16 operands, fp32 accumulation in TMEM) -----------------------------------
# north_star states the bf16 tolerance separately from fp32: blendshapes <= 1e-3 absolute.  Measured on B200 the
# error is ~1e-5 on the outputs; we gate at 1e-4 (outputs), 2e-3 (pre-fusion sigmoid), 2e-3 (attention weights).
BF16_OUT_ATOL, BF16_SIG_ATOL, BF16_ATTN_ATOL = 1e-4, 2e-3, 2e-3


@pytest.mark.parametrize("name", ["single_noise_init", "single_speech_stress", "single_burst_stress",
                                  "single_silence_init", "single_short_clip", "single_long_clip", "single_60fps"])
def test_bf16_tensor_path_single(K, golden, name):
    cases, data = golden
    spec = cases[name]
    m, _ = _model(K, spec, False)
    m.precision = "bf16"
    audio, eg = _inputs(spec)
    out = m(audio, return_attention=True, egemaps=eg)
    _close(out["blendshapes"], data[f"{name}/blendshapes"], 0, BF16_OUT_ATOL, "bf16 blendshapes")
    _close(out["mel_blendshapes"], data[f"{name}/mel_blendshapes"], 0, BF16_SIG_ATOL, "bf16 sigmoid")
    _close(out["emotion_blendshapes"], data[f"{name}/emotion_blendshapes"], 0, SIG_ATOL, "emotion stream stays fp32")
    _close(out["mel_attention_weights"], data[f"{name}/mel_attention_weights"], 0, BF16_ATTN_ATOL, "bf16 attention")
    rows = out["mel_attention_weights"].sum(-1)
    assert float((rows - 1).abs().max()) < 1e-2


@pytest.mark.parametrize("name", ["seq_clip_T1", "seq_13_frames", "seq_20s", "seq_stride3", "seq_burst_edge", "seq_60fps"])
def test_bf16_tensor_path_sequence(K, golden, name):
    cases, data = golden
    spec = cases[name]
    m, _ = _model(K, spec, True)
    m.precision = "bf16"
    audio, eg = _inputs(spec)
    out = m(audio, egemaps=eg)
    _close(out["blendshapes"], data[f"{name}/blendshapes"], 0, BF16_OUT_ATOL, "bf16 sequence blendshapes")


def test_bf16_tensor_path_full_batch_consistency(K):
    """512 windows through the persistent tcgen05 kernel: every CTA / pipeline wrap gives the same answer as the
    fp32 kernel within the bf16 tolerance, and results do not depend on which CTA handled the clip."""
    spec = dict(wseed=1235, style="stress", fps=30)
    m, _ = _model(K, spec, True)
    g = torch.Generator(device="cuda").manual_seed(11)
    audio = 0.1 * torch.randn(512, 136000, device="cuda", generator=g)
    eg = torch.randn(512, 264, device="cuda", generator=g)
    ref = m(audio, egemaps=eg)["blendshapes"]
    m.precision = "bf16"
    out = m(audio, egemaps=eg)["blendshapes"]
    _close(out, ref, 0, BF16_OUT_ATOL, "bf16 vs fp32 kernel, 512 windows")
    perm = torch.randperm(512, device="cuda", generator=g)
    out_p = m(audio[perm].contiguous(), egemaps=eg[perm].contiguous())["blendshapes"]
    assert torch.equal(out_p, out[perm])
    # ... and against the CPU oracle on clips spread over the batch (first / last CTA round, middle): the full-size run is
    # checked by something other than the repo's own kernels
    w = O.make_weights(spec["wseed"], 30, style=spec["style"])
    pick = [0, 1, 147, 148, 295, 444, 510, 511]
    want = O.forward_sequence(w, audio[pick].cpu().numpy(), eg[pick].cpu().numpy())["blendshapes"]
    _close(ref[pick], want, 0, OUT_ATOL, "fp32 kernel at batch 512 vs oracle")
    _close(out[pick], want, 0, BF16_OUT_ATOL, "bf16 kernel at batch 512 vs oracle")


def test_bf16_unsupported_geometry_is_refused_not_faked(K):
    """The tensor path is built for K = 259 (30 fps) and 515 (60 fps); any other window length has no pre-tiled bf16
    weights and must raise instead of silently running something else."""
    m = K.SequentialDualStreamModel(target_fps=30, mel_sequence_length=128).cuda()
    m.precision = "bf16"
    with pytest.raises(RuntimeError, match="tc_bf16 is missing|30 fps"):
        m(torch.zeros(1, 136000, device="cuda"), egemaps=torch.zeros(1, 264, device="cuda"))


def test_pcm16_conversion_is_exact_and_host_pipeline_accepts_it(K):
    """int16 PCM -> float is sample / 32768 (libsndfile's normalisation behind sf.read(dtype="float32"),
    src/data/io.py:71), bit for bit, including the < 8-sample tail; the host-buffer pipeline fed int16 returns exactly
    what it returns for the same samples as float32."""
    from koemorph_b200.features.mel_frontend import pcm16_to_float
    from koemorph_b200.infer import HostPipeline
    rng = np.random.default_rng(5)
    for n in (0, 1, 7, 8, 4099, 136000 * 3 + 5):
        pcm = rng.integers(-32768, 32768, size=n, dtype=np.int16)
        if n >= 2:
            pcm[0], pcm[-1] = -32768, 32767
        got = pcm16_to_float(torch.from_numpy(pcm).cuda()).cpu().numpy()
        assert np.array_equal(got, pcm.astype(np.float32) / np.float32(32768.0))
    with pytest.raises(TypeError):
        pcm16_to_float(torch.zeros(8, device="cuda"))

    spec = dict(wseed=3, fps=30, style="stress", B=5, L=136000, iseed=11, kind="speechlike")
    m, _ = _model(K, spec, sequential=True)
    audio, eg = O.make_inputs(spec["iseed"], spec["B"], spec["L"], spec["kind"])
    pcm = np.clip(np.round(audio * 32768.0), -32768, 32767).astype(np.int16)
    as_float = torch.from_numpy(pcm.astype(np.float32) / np.float32(32768.0))
    pipe = HostPipeline(m, chunk_clips=2)  # 3 chunks, the last one ragged
    want = pipe(as_float.pin_memory(), torch.from_numpy(eg).pin_memory()).clone()
    got = pipe(torch.from_numpy(pcm).pin_memory(), torch.from_numpy(eg).pin_memory())
    assert torch.equal(got, want)
    ref = m(as_float.cuda(), egemaps=torch.from_numpy(eg).cuda())["blendshapes"].cpu()
    assert torch.equal(want, ref)
    with pytest.raises(ValueError):
        pipe(torch.zeros(2, 136000, dtype=torch.float64), torch.from_numpy(eg[:2]))


RAGGED_SHAPES = [  # L, hop, n_frames, frame_offset, pad_mode
    (136000, 533, 257, 0, "constant"),   # bench shape: frame 255 and 256 run past the clip (three edge pairs)
    (136000, 533, 256, 0, "constant"),
    (20000, 533, 38, 0, "constant"),     # short clip: 1 + L // hop frames
    (20000, 533, 5, 3, "constant"),      # a few interior frames only (no edge pair at either end)
    (3000, 533, 6, 0, "constant"),       # shorter than two frames: every pair touches an edge
    (700, 533, 2, 0, "constant"),        # shorter than one frame
    (1500, 533, 1, 1, "constant"),       # a single frame = a single half-empty pair
    (20000, 266, 76, 0, "constant"),     # 60 fps hop: two leading / trailing edge frames
    (20000, 533, 38, 0, "reflect"),      # MelSlidingWindowExtractor padding
]


@pytest.mark.parametrize("L,hop,n_frames,frame_offset,pad_mode", RAGGED_SHAPES)
def test_logmel_launch_order_over_ragged_shapes(K, L, hop, n_frames, frame_offset, pad_mode):
    """The frontend launches a clip's padding-touching frame pairs ahead of its interior ones (they take masked loads);
    whatever the split -- no edge pairs, only edge pairs, odd frame counts, several clips -- every output row must still be
    the frame it is documented to be: compared with the float64 restatement of librosa's STFT + mel."""
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    B = 5
    audio, _ = O.make_inputs(1000 + L + n_frames, B, L, "speechlike")
    fe = LogMelFrontend.get("cuda")
    db, fmax = fe.power(torch.from_numpy(audio).cuda(), hop, n_frames, frame_offset=frame_offset, pad_mode=pad_mode)
    db = db.cpu().double().numpy()
    assert db.shape == (B, n_frames, 80)
    for b in range(B):
        full = O.melspectrogram(audio[b], hop_length=hop, pad_mode=pad_mode, exact=True).T   # (1 + L // hop, 80)
        have = min(n_frames, max(0, full.shape[0] - frame_offset))
        ref = full[frame_offset:frame_offset + have]
        got = 10 ** (db[b, :have] / 10)
        assert np.abs(got - np.maximum(ref, 1e-10)).max() <= 2e-6 * max(full.max(), 1e-10)
        big = ref > 1e-6 * full.max()
        if big.any():
            assert np.abs(db[b, :have] - 10 * np.log10(np.maximum(ref, 1e-10)))[big].max() < 8.7e-4
        np.testing.assert_allclose(fmax[b].cpu().numpy(), db[b].max(axis=1), rtol=1e-6)


@pytest.mark.parametrize("bank", ["default", "generic"])
@pytest.mark.parametrize("L,hop,n_frames,frame_offset",
                         [s[:4] for s in RAGGED_SHAPES if s[4] == "constant" and s[2] >= 2])
def test_logmel_split_pairs_equal_plain_frames(K, L, hop, n_frames, frame_offset, bank):
    """The two organisations of the frontend kernel compute the same rows bit for bit.  A plain launch runs the
    warp-specialised kernel for the default bank and the lock-step kernel for any other; a launch that sends each pair's
    second frame to its own buffer (out_b, the streaming step) runs the lock-step kernel for both."""
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    B = 5
    audio, _ = O.make_inputs(1000 + L + n_frames, B, L, "speechlike")
    audio = torch.from_numpy(audio).cuda()
    fe = LogMelFrontend.get("cuda") if bank == "default" else LogMelFrontend.get("cuda", f_min=60.0, f_max=7600.0)
    assert fe.uses_unrolled_bank() == (bank == "default")
    db, fmax = fe.power(audio, hop, n_frames, frame_offset=frame_offset)
    db_b = torch.empty((B, n_frames // 2, 80), dtype=torch.float32, device="cuda")
    fmax_b = torch.empty((B, n_frames // 2), dtype=torch.float32, device="cuda")
    db_a, fmax_a = fe.power(audio, hop, n_frames, frame_offset=frame_offset, out_b=(db_b, fmax_b))
    assert torch.equal(db_a[:, 0::2], db[:, 0::2])
    assert torch.equal(fmax_a[:, 0::2], fmax[:, 0::2])
    assert torch.equal(db_b, db[:, 1::2])
    assert torch.equal(fmax_b, fmax[:, 1::2])


# ---- round 2: host pipeline state handling, fused native forward, public emotion entry, weight-cache invalidation --------
def test_host_pipeline_with_the_single_frame_model_matches_one_forward(K):
    """HostPipeline(SimplifiedDualStreamModel): chunking must not change the result.  forward() blends every call with the
    previous call's output (reference :341-368); a chunked run has to apply that once over the whole batch."""
    from koemorph_b200.infer import HostPipeline
    spec = dict(fps=30, wseed=1235, style="stress", iseed=77, kind="speechlike", B=11, L=60000)
    m, _ = _model(K, spec, False)
    audio, eg = _inputs(spec)
    audio2 = torch.roll(audio, 1, 0).contiguous()
    want1 = m(audio, egemaps=eg)["blendshapes"].clone()
    want2 = m(audio2, egemaps=eg)["blendshapes"].clone()         # second call: EMA against the first
    m.reset_temporal_state()
    pipe = HostPipeline(m, chunk_clips=4)                         # 3 chunks: 4 + 4 + 3 clips on two streams
    got1 = pipe(audio.cpu().pin_memory(), eg.cpu().pin_memory()).clone()
    got2 = pipe(audio2.cpu().pin_memory(), eg.cpu().pin_memory()).clone()
    assert got1.shape == (11, 52)
    assert torch.equal(got1, want1.cpu()) and torch.equal(got2, want2.cpu())
    assert not torch.equal(got1, got2)


def test_host_pipeline_leaves_the_sequence_models_state(K):
    from koemorph_b200.infer import HostPipeline
    spec = dict(fps=30, wseed=1235, style="stress", iseed=78, kind="noise", B=5, L=136000 + 3 * 533)
    m, _ = _model(K, spec, True)
    audio, eg = _inputs(spec)
    want = m(audio, egemaps=eg)["blendshapes"].clone()
    state = m.prev_blendshapes.clone()
    m.reset_temporal_state()
    got = HostPipeline(m, chunk_clips=2)(audio.cpu().pin_memory(), eg.cpu().pin_memory())
    assert torch.equal(got, want.cpu())
    assert torch.equal(m.prev_blendshapes, state)
    # the state a later single-frame call smooths against is the last frame, whatever its memory layout
    nxt = m.forward_single_frame(audio[:, :136000].contiguous(), egemaps=eg)["blendshapes"]
    alpha = torch.sigmoid(m.smoothing_alpha).item()
    raw = m._single_frames(audio[:, :136000].contiguous(), eg, False)[0]
    _close(nxt, alpha * raw + (1 - alpha) * want[:, -1], 0, 1e-7, "single frame after a sequence")
    assert torch.equal(want, m(audio, egemaps=eg)["blendshapes"]), "the earlier result tensor was modified"


def test_forward_out_argument_and_fused_call_equal_the_separate_entry_points(K):
    """koe_forward_windows (one native call, programmatic dependent launch inside) against the same kernels issued one by
    one through the public single-kernel entries."""
    spec = dict(fps=30, wseed=1235, style="stress", iseed=79, kind="speechlike", B=3, L=136000 + 7 * 533)
    m, _ = _model(K, spec, True)
    audio, eg = _inputs(spec)
    for precision in ("fp32", "bf16"):
        m.precision = precision
        res = m(audio, egemaps=eg, return_attention=True)
        n_out, W = m.num_output_frames(audio.shape[1]), 256
        assert n_out == 7
        buf = torch.full((3, n_out, 52), float("nan"), device="cuda")
        res2 = m(audio, egemaps=eg, out=buf)
        assert res2["blendshapes"].data_ptr() == buf.data_ptr() and torch.equal(buf, res["blendshapes"])
        # the decomposed path: frontend launches, emotion stream, core, EMA through the public entries
        fe = m._frontend(audio.device)
        n_frames = n_out - 1 + W + 1
        power, fmax = fe.power(audio, 533, n_frames)
        lo = fe.power(audio, 533, n_out, frame_offset=0, frame_step=1, lo_rel=0)
        hi = fe.power(audio, 533, n_out, frame_offset=W, frame_step=1, hi_rel=0)
        out, sig, attn = m._core_windows([power, lo[0], hi[0]], [fmax, lo[1], hi[1]], 1, 3, n_frames, n_out, 1, W + 1, eg, True)
        assert torch.equal(sig, res["mel_blendshapes"] + res["emotion_blendshapes"])
        _close(attn, res["mel_attention_weights"], 0, 1e-6, "attention weights")  # head average accumulated with atomics
        from koemorph_b200 import _lib
        alpha = float(torch.sigmoid(m.smoothing_alpha.detach()))
        _lib.check(_lib.load().koe_ema_scan(out.data_ptr(), 3, n_out, alpha, None, 0, _lib.stream_ptr(out.device)))
        assert torch.equal(out, res["blendshapes"])
    with pytest.raises(ValueError):
        m(audio, egemaps=eg, out=torch.empty(3, 8, 52, device="cuda"))


def test_public_emotion_entry_sees_the_previous_kernels_writes(K):
    """koe_emotion_stream from the public ABI keeps full stream order: its input may be produced by the kernel queued just
    before it (ADVICE r1: it used to start early under programmatic dependent launch)."""
    import ctypes as C
    from koemorph_b200 import _lib
    spec = dict(fps=30, wseed=1235, style="stress", iseed=80, kind="noise", B=4096, L=1)
    m, _ = _model(K, spec, False)
    w = m.dual_stream_attention.kernel_weights(m._compression)
    lib = _lib.load()
    eg = torch.randn(4096, 264, device="cuda")
    want = torch.empty(4096, device="cuda")
    _lib.check(lib.koe_emotion_stream(C.byref(w.struct), eg.data_ptr(), 4096, want.data_ptr(), _lib.stream_ptr(eg.device)))
    torch.cuda.synchronize()
    big = torch.randn(64, 1 << 20, device="cuda")
    for _ in range(5):
        src = torch.zeros_like(eg)
        got = torch.empty(4096, device="cuda")
        big.mul_(1.0001)                       # keep the device busy so that the next kernels queue up
        src.copy_(eg)                          # producer of the input: the kernel right before the emotion stream
        _lib.check(lib.koe_emotion_stream(C.byref(w.struct), src.data_ptr(), 4096, got.data_ptr(), _lib.stream_ptr(eg.device)))
        assert torch.equal(got, want)


def test_extract_emotion_features_is_the_compression_layer(K):
    spec = dict(fps=30, wseed=1235, style="stress", iseed=81, kind="noise", B=7, L=1)
    m, w = _model(K, spec, False)
    eg = torch.randn(7, 264, device="cuda")
    got, meta = m.extract_emotion_features(egemaps=eg)
    ref = eg.double().cpu() @ torch.from_numpy(w["compression.weight"]).double().t() + torch.from_numpy(w["compression.bias"]).double()
    _close(got, ref, 1e-5, 1e-6, "264 -> 256 compression")
    assert meta["backend_used"] == "egemaps_input"
    got3, _ = m.extract_emotion_features(egemaps=eg.view(7, 3, 88))
    assert torch.equal(got3, got)


def test_folded_weights_follow_in_place_edits_after_invalidate(K):
    spec = dict(fps=30, wseed=1234, style="init", iseed=82, kind="noise", B=2, L=136000)
    m, _ = _model(K, spec, False)
    audio, eg = _inputs(spec)
    a = m(audio, egemaps=eg)["blendshapes"].clone()
    m.reset_temporal_state()
    m.dual_stream_attention.mel_weights.data.mul_(2.0)            # .data edit: no version bump
    m.dual_stream_attention.invalidate_kernel_weights()
    b = m(audio, egemaps=eg)["blendshapes"].clone()
    assert not torch.equal(a, b)
    m.reset_temporal_state()
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    sd["dual_stream_attention.mel_weights"] /= 2.0
    m.load_state_dict(sd)                                          # post hook invalidates
    assert torch.equal(m(audio, egemaps=eg)["blendshapes"], a)
    with pytest.raises(ValueError):
        m.precision = "tf32"


def test_forward_is_cuda_graph_capturable(K):
    """The whole forward (one native call: six launches chained with programmatic dependent launch, one workspace
    allocation) can be captured in a CUDA graph and replayed: same bits as the eager call, also after the inputs change."""
    spec = dict(fps=30, wseed=1235, style="stress", iseed=83, kind="speechlike", B=4, L=136000 + 3 * 533)
    m, _ = _model(K, spec, True)
    m.precision = "bf16"
    audio, eg = _inputs(spec)
    out = torch.empty(4, m.num_output_frames(audio.shape[1]), 52, device="cuda")
    want = m(audio, egemaps=eg)["blendshapes"].clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m(audio, egemaps=eg, out=out)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m(audio, egemaps=eg, out=out)
    out.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)
    audio.copy_(torch.roll(audio, 1, 0))            # new clips in the captured buffers
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, m(audio, egemaps=eg)["blendshapes"])


@pytest.mark.parametrize("L", [0, 1, 100, 532, 533, 1599, 136447, 136448, 136449])
def test_tiny_and_boundary_clip_lengths_vs_oracle(K, L):
    """Ragged edges of the geometry: empty audio, clips shorter than a hop / than three frames (the reference zero-pads the
    short-term detail, simplified_dual_stream_model.py:206-212), lengths just below / at / above one full window."""
    spec = dict(fps=30, wseed=1235, style="stress", iseed=90 + L % 7, kind="noise", B=2, L=max(L, 1))
    m, w = _model(K, spec, True)
    audio, eg = O.make_inputs(spec["iseed"], 2, max(L, 1), "noise")
    audio = audio[:, :L]
    want = O.forward_sequence(w, audio, eg)["blendshapes"]
    a, e = torch.from_numpy(np.ascontiguousarray(audio)).cuda(), torch.from_numpy(eg).cuda()
    for prec, tol in (("fp32", OUT_ATOL), ("bf16", BF16_OUT_ATOL)):
        m.precision = prec
        got = m(a, egemaps=e)["blendshapes"]
        assert got.shape == want.shape == (2, 1 if L < 136448 + 533 else 2, 52)
        _close(got, want, 0, tol, f"L = {L}, {prec}")
    single = K.SimplifiedDualStreamModel().cuda().eval()
    single.load_state_dict(O.model_state_dict(w), strict=True)
    single.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    lt, st = single.extract_mel_features(a)
    ref_lt, ref_st = O.extract_mel_features(audio)
    _close(lt, ref_lt, LOGMEL_RTOL, LOGMEL_ATOL, f"log-mel, L = {L}")
    _close(st, ref_st, LOGMEL_RTOL, LOGMEL_ATOL, f"short-term log-mel, L = {L}")


def test_empty_batch(K):
    m, _ = _model(K, dict(fps=30, wseed=1234, style="init"), True)
    out = m(torch.zeros(0, 136000, device="cuda"), egemaps=torch.zeros(0, 264, device="cuda"))
    assert out["blendshapes"].shape == (0, 1, 52) and out["num_frames"] == 1
    from koemorph_b200.infer import HostPipeline
    host = HostPipeline(m)(torch.zeros(0, 136000).pin_memory(), torch.zeros(0, 264).pin_memory())
    assert host.shape == (0, 1, 52)


@pytest.mark.parametrize("fps,W,stride,extra", [(60, 512, 1, 0), (60, 512, 1, 265), (60, 512, 1, 266), (60, 512, 2, 3 * 266 + 1),
                                                (30, 256, 4, 7 * 533), (30, 256, 7, 20 * 533 + 532)])
def test_window_count_boundaries_vs_oracle(K, fps, W, stride, extra):
    """T_out = max(1, (L // hop - W) // stride + 1) at its boundaries, both frame rates, strides that do not divide the
    surplus (reference sequential_dual_stream_model.py:84-96)."""
    hop = 16000 // fps
    L = W * hop + extra
    spec = dict(fps=fps, wseed=1236, style="stress", iseed=200 + extra % 11, kind="speechlike", B=2, L=L, stride=stride)
    m, w = _model(K, spec, True)
    audio, eg = O.make_inputs(spec["iseed"], 2, L, "speechlike")
    want = O.forward_sequence(w, audio, eg, fps=fps, stride_frames=stride)["blendshapes"]
    a, e = torch.from_numpy(audio).cuda(), torch.from_numpy(eg).cuda()
    n_out = max(1, (L // hop - W) // stride + 1)
    assert want.shape == (2, n_out, 52) and m.num_output_frames(L) == n_out
    for prec, tol in (("fp32", OUT_ATOL), ("bf16", BF16_OUT_ATOL)):
        m.precision = prec
        _close(m(a, egemaps=e)["blendshapes"], want, 0, tol, f"{fps} fps stride {stride} extra {extra} {prec}")


def test_core_standalone_degenerate_shapes(K):
    """DualStreamCrossAttention.forward with one / two long-term frames, far more than the window (truncated, reference
    dual_stream_attention.py:192-202), and an empty batch."""
    w = O.make_weights(1235, 30, style="stress")
    core = K.DualStreamCrossAttention().cuda().eval()
    core.load_state_dict({k[len("dual_stream_attention."):]: v for k, v in O.model_state_dict(w).items()
                          if k.startswith("dual_stream_attention.")})
    rng = np.random.default_rng(6)
    for T in (1, 2, 700):
        lt = rng.uniform(0, 1, (3, T, 80)).astype(np.float32)
        st = rng.uniform(0, 1, (3, 3, 80)).astype(np.float32)
        emo = rng.standard_normal((3, 256)).astype(np.float32)
        want = O.dual_stream_core(w, lt, st, emo)["blendshapes"]
        for prec, tol in (("fp32", OUT_ATOL), ("bf16", BF16_OUT_ATOL)):
            core.precision = prec
            got = core(torch.from_numpy(lt).cuda(), torch.from_numpy(st).cuda(), torch.from_numpy(emo).cuda())["blendshapes"]
            _close(got, want, 0, tol, f"core T = {T} {prec}")
    core.precision = "fp32"
    out = core(torch.zeros(0, 5, 80, device="cuda"), torch.zeros(0, 3, 80, device="cuda"), torch.zeros(0, 256, device="cuda"))
    assert out["blendshapes"].shape == (0, 52)


@pytest.mark.parametrize("n_clips", [1, 7, 8, 9, 61, 2049, 2061])
def test_emotion_stream_clip_counts_vs_oracle(K, n_clips):
    """koe_emotion_stream over ragged clip counts: a partly filled last CTA, one clip, and the sixteen-clips-per-CTA kernel
    that large batches take (> 2048 clips); expression sigmoid against the oracle's emotion stream
    (reference dual_stream_attention.py:234-240)."""
    import ctypes as C
    from koemorph_b200 import _lib
    w = O.make_weights(1237, 30, style="stress")
    core = K.DualStreamCrossAttention().cuda().eval()
    core.load_state_dict({k[len("dual_stream_attention."):]: v for k, v in O.model_state_dict(w).items()
                          if k.startswith("dual_stream_attention.")})
    rng = np.random.default_rng(n_clips)
    emo = rng.standard_normal((n_clips, 256)).astype(np.float32)
    pick = sorted(set([0, n_clips - 1, n_clips // 2, min(n_clips - 1, 2047), min(n_clips - 1, 2048)]))
    lt = np.full((len(pick), 4, 80), 0.5, np.float32)
    st = np.full((len(pick), 3, 80), 0.5, np.float32)
    want = O.dual_stream_core(w, lt, st, emo[pick], return_attention=True)["emotion_blendshapes"]
    kw = core.kernel_weights()
    expr = torch.full((n_clips,), float("nan"), device="cuda")
    e = torch.from_numpy(emo).cuda()
    _lib.check(_lib.load().koe_emotion_stream(C.byref(kw.struct), e.data_ptr(), n_clips, expr.data_ptr(),
                                              _lib.stream_ptr(e.device)), "koe_emotion_stream")
    got = expr.cpu().numpy()
    assert np.isfinite(got).all()
    idx = [i for i in range(52) if i not in O.MOUTH_INDICES]
    for j, c in enumerate(pick):
        ref = want[j].numpy() if torch.is_tensor(want) else np.asarray(want[j])
        assert np.abs(ref[idx] - got[c]).max() <= SIG_ATOL, (c, ref[idx][:3], got[c])


@pytest.mark.parametrize("n_clips", [24, 512])
def test_back_to_back_forwards_do_not_interfere(K, n_clips):
    """The forward's kernels are chained with programmatic dependent launch (a kernel's CTAs start while the previous
    kernel's last CTAs still run) and successive forwards reuse the same workspace addresses: thirty forwards queued
    without a synchronisation, alternating between two different inputs, must each equal the result of the same forward
    run alone -- bit for bit, for both cores."""
    spec = dict(fps=30, wseed=1238, style="stress")
    m, _ = _model(K, spec, True)
    g = torch.Generator(device="cuda").manual_seed(n_clips)
    L = 136000
    inputs = [(0.1 * torch.randn(n_clips, L, device="cuda", generator=g), torch.randn(n_clips, 264, device="cuda", generator=g))
              for _ in range(2)]
    for prec in ("bf16", "fp32"):
        m.precision = prec
        alone = []
        for a, e in inputs:
            torch.cuda.synchronize()
            alone.append(m(a, egemaps=e)["blendshapes"].clone())
            torch.cuda.synchronize()
        assert not torch.equal(alone[0], alone[1])
        n = 30 if prec == "bf16" else 6
        kept = torch.full((n, n_clips, 1, 52), float("nan"), device="cuda")
        for i in range(n):
            a, e = inputs[i & 1]
            m(a, egemaps=e, out=kept[i])
        torch.cuda.synchronize()
        for i in range(n):
            assert torch.equal(kept[i], alone[i & 1]), f"{prec}: forward {i} of the queue differs from the same forward run alone"


@pytest.mark.parametrize("fps,n_clips", [(30, 149), (30, 297), (30, 445), (30, 512), (30, 700), (30, 2100), (60, 300), (60, 512)])
def test_early_released_core_equals_the_plain_chain(K, fps, n_clips):
    """Batches of more than one round of windows take the early-release chain (the core starts its first rounds on a flag
    of the frontend instead of waiting for the whole frontend, csrc/session.cu).  Its result must equal, bit for bit, the
    same kernels issued one by one through the public entries (plain stream order, no flag), on repeated calls."""
    spec = dict(fps=fps, wseed=1239, style="stress")
    m, _ = _model(K, spec, True)
    m.precision = "bf16"
    hop, T = m.hop_length, m.window_frames + 1
    g = torch.Generator(device="cuda").manual_seed(n_clips)
    audio = 0.1 * torch.randn(n_clips, 136000, device="cuda", generator=g)
    audio[::7] *= 1e-3                                    # quiet clips: a stale (zero / garbage) row would move their dB reference
    eg = torch.randn(n_clips, 264, device="cuda", generator=g)
    fe = m._frontend(audio.device)
    power, fmax = fe.power(audio, hop, T)
    want, _, _ = m._core_windows([power], [fmax], 0, n_clips, T, 1, 1, T, m._check_egemaps(eg, n_clips, audio.device), False)
    torch.cuda.synchronize()
    for rep in range(4):
        got = m(audio, egemaps=eg)["blendshapes"]
        assert torch.equal(got.reshape(want.shape), want), f"call {rep}: early-released forward differs from the plain chain"


def test_early_released_core_in_a_replayed_cuda_graph(K):
    """Three forwards of a batch that takes the early-release chain, captured in one CUDA graph: every replay must leave
    the release flag cleared for the next one (the last core CTA out clears it) and reproduce the eager results bit for
    bit, also interleaved with eager calls on the same stream."""
    spec = dict(fps=30, wseed=1240, style="stress")
    m, _ = _model(K, spec, True)
    m.precision = "bf16"
    n = 300
    g = torch.Generator(device="cuda").manual_seed(9)
    audio = 0.1 * torch.randn(n, 136000, device="cuda", generator=g)
    eg = torch.randn(n, 264, device="cuda", generator=g)
    want = m(audio, egemaps=eg)["blendshapes"].clone()     # eager (allocates the flag words outside any capture)
    outs = torch.zeros(3, n, 1, 52, device="cuda")
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for i in range(3):
            m(audio, egemaps=eg, out=outs[i])
    for rep in range(4):
        outs.zero_()
        graph.replay()
        if rep % 2:
            assert torch.equal(m(audio, egemaps=eg)["blendshapes"], want)   # an eager forward between replays
        torch.cuda.synchronize()
        for i in range(3):
            assert torch.equal(outs[i], want), f"replay {rep}, forward {i}"


def test_early_released_core_on_two_streams(K):
    """Forwards that take the early-release chain, queued on two streams at once (each stream has its own flag words):
    results equal the same forwards run alone."""
    spec = dict(fps=30, wseed=1241, style="stress")
    m, _ = _model(K, spec, True)
    m.precision = "bf16"
    n = 300
    g = torch.Generator(device="cuda").manual_seed(10)
    ins = [(0.1 * torch.randn(n, 136000, device="cuda", generator=g), torch.randn(n, 264, device="cuda", generator=g)) for _ in range(2)]
    want = [m(a, egemaps=e)["blendshapes"].clone() for a, e in ins]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = torch.zeros(2, 4, n, 1, 52, device="cuda")
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    for i in range(4):
        for k, s in enumerate(streams):
            with torch.cuda.stream(s):
                m._forward_frames(ins[k][0], m._check_egemaps(ins[k][1], n, ins[k][0].device), False, out=outs[k, i])
    for s in streams:
        torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    for k in range(2):
        for i in range(4):
            assert torch.equal(outs[k, i], want[k]), f"stream {k}, forward {i}"
