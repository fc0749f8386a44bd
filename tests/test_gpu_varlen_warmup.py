"""GPU tests (-m gpu) of packed warm-up batches (SequentialDualStreamModel.forward_varlen(..., warmup=True)): a row at
every hop of the output grid of every clip, from its first hop on.  Before hop W - 1 a row is
SimplifiedDualStreamModel.forward on the clip's audio up to that hop; from hop W - 1 on it is bit for bit the row of
warmup=False (smoothing off); the smoothing runs over all of a clip's rows."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O

pytestmark = pytest.mark.gpu

HOP = {30: 533, 60: 266}
WIN = {30: 256, 60: 512}
GATE = {"fp32": 2e-6, "bf16": 1e-4}          # against the fp32 forward, as tests/test_gpu_stream_pool_warmup.py
PARITY = {"fp32": 2e-5, "bf16": 2e-3}        # sigmoid and attention rows, as tests/test_gpu_parity.py
# (fps, precision, stride): stride 3 at 30 fps has r = 0, stride 2 at 60 fps r = 1
CONFIGS = [(30, "fp32", 1), (30, "bf16", 1), (60, "fp32", 1), (60, "bf16", 1), (30, "bf16", 3), (60, "fp32", 2)]


def _model(fps, precision, stride=1, smoothing=False, seed=1235):
    import koemorph_b200 as K
    w = O.make_weights(seed, fps, style="stress")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length=WIN[fps], stride_frames=stride).cuda().eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = precision
    m.use_temporal_smoothing = smoothing
    return m


def _grid(fps, stride):
    W = WIN[fps]
    return (W - 1) % stride, W


def _lengths(fps, stride, seed, long_clip=60 * 16000):
    """Lengths around every boundary of the warm-up rows, plus random ones, in random order; none without a grid hop."""
    hop, (r, W) = HOP[fps], _grid(fps, stride)
    fixed = [hop, hop + 1, 2 * hop, 5 * hop + 7, (W - 1) * hop, W * hop - 1, W * hop, W * hop + hop - 1, (W + 1) * hop,
             (W + 7) * hop + 3, long_clip]
    rng = np.random.default_rng(seed)
    lens = [L for L in fixed if L >= (r + 1) * hop] + [int(x) for x in rng.integers((r + 1) * hop, 2 * W * hop, 6)]
    rng.shuffle(lens)
    return lens


def _pack(lens, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    audio = (torch.rand(sum(lens), generator=g, device="cuda") * 2 - 1) * 0.3
    eg = torch.randn(len(lens), 264, generator=g, device="cuda")
    return audio, eg


def _clip(audio, lens, c, n=None):
    s = sum(lens[:c])
    return audio[s:s + (lens[c] if n is None else n)]


def _hops(L, fps, stride):
    """The grid hops of a clip of L samples: its rows, in order."""
    r, W = _grid(fps, stride)
    return list(range(r, L // HOP[fps], stride))


def _max_diff(a, b):
    return (a.double() - b.double()).abs().max().item()


@functools.lru_cache(maxsize=None)
def _run(fps, precision, stride):
    m = _model(fps, precision, stride)
    lens = _lengths(fps, stride, 80 + fps + stride)
    audio, eg = _pack(lens, 21 + fps + stride)
    warm = m.forward_varlen(audio, lens, egemaps=eg, return_attention=True, warmup=True)
    plain = m.forward_varlen(audio, lens, egemaps=eg, return_attention=True)
    torch.cuda.synchronize()
    return lens, audio, eg, warm, plain


@pytest.mark.parametrize("fps,precision,stride", CONFIGS)
def test_lead_rows_are_the_forward_on_the_audio_so_far(fps, precision, stride):
    """Every lead row of the longest clip and hops {0, 1, 2, W/2, W - 3, W - 2} (where on the grid) of the others against
    the fp32 SimplifiedDualStreamModel.forward on the clip's first (h + 1) hops; sigmoid and attention too."""
    from koemorph_b200.model.simplified_dual_stream_model import SimplifiedDualStreamModel
    lens, audio, eg, warm, _ = _run(fps, precision, stride)
    ref = _model(fps, "fp32", stride)
    hop, (r, W) = HOP[fps], _grid(fps, stride)
    off = warm["frame_offsets"]
    assert [int(off[c + 1] - off[c]) for c in range(len(lens))] == [len(_hops(L, fps, stride)) for L in lens]
    assert warm["blendshapes"].shape == (int(off[-1]), 52) and warm["num_frames"] == int(off[-1])
    longest = max(range(len(lens)), key=lambda c: lens[c])
    some = {0, 1, 2, W // 2, W - 3, W - 2}
    worst, checked = 0.0, 0
    for h in range(r, W - 1, stride):
        clips = [c for c, L in enumerate(lens) if L // hop > h and (c == longest or h in some)]
        if not clips:
            continue
        rows = torch.tensor([int(off[c]) + (h - r) // stride for c in clips])
        prefix = torch.stack([_clip(audio, lens, c, (h + 1) * hop) for c in clips])
        want = SimplifiedDualStreamModel.forward(ref, prefix, return_attention=True, egemaps=eg[clips])
        d = _max_diff(warm["blendshapes"][rows], want["blendshapes"])
        worst = max(worst, d)
        assert d <= GATE[precision], f"hop {h}: max |d| = {d:.3e}"
        for key in ("mel_blendshapes", "mel_attention_weights"):
            d = _max_diff(warm[key][rows], want[key])
            assert d <= PARITY[precision], f"hop {h} {key}: max |d| = {d:.3e}"
        checked += len(clips)
    assert checked >= (W - 1 - r) // stride
    print(f"{fps} fps {precision} stride {stride}: largest deviation {worst:.3e} over {checked} lead rows")


@pytest.mark.parametrize("fps,precision,stride", CONFIGS)
def test_steady_rows_equal_the_plain_call(fps, precision, stride):
    """Rows at hops >= W - 1 are bit for bit warmup=False's rows of the same batch; a clip of fewer than W hops has no
    steady row (its padded window is not a warm-up row)."""
    lens, _, _, warm, plain = _run(fps, precision, stride)
    hop, (r, W) = HOP[fps], _grid(fps, stride)
    ow, op = warm["frame_offsets"], plain["frame_offsets"]
    for c, L in enumerate(lens):
        leads = len([h for h in _hops(L, fps, stride) if h < W - 1])
        steady = slice(int(ow[c]) + leads, int(ow[c + 1]))
        if L // hop < W:
            assert steady.start == steady.stop, c
            continue
        sl = slice(int(op[c]), int(op[c + 1]))
        for key in ("blendshapes", "mel_blendshapes", "emotion_blendshapes"):
            assert torch.equal(warm[key][steady], plain[key][sl]), (c, L, key)
        if precision == "fp32":
            assert torch.equal(warm["mel_attention_weights"][steady], plain["mel_attention_weights"][sl]), c
        else:  # the tensor-core kernel averages the heads with atomics: the order of the eight additions varies
            torch.testing.assert_close(warm["mel_attention_weights"][steady], plain["mel_attention_weights"][sl],
                                       rtol=0, atol=1e-6)


@pytest.mark.parametrize("fps,precision,stride", CONFIGS)
def test_lead_window_equals_the_public_core_on_its_rows(fps, precision, stride):
    """A lead window's T rows rebuilt with the public frontend -- the clip's plain rows (the plan's frame count) and the
    lead window-end variants (frame_offset r + 1 - m, frame_step stride, hi_rel m, K_c frames) -- run through
    koe_dual_stream_windows as one clip without edge variants give the packed row bit for bit."""
    from koemorph_b200 import _lib
    from koemorph_b200.features.mel_frontend import LogMelFrontend
    lens, audio, eg, warm, _ = _run(fps, precision, stride)
    m = _model(fps, precision, stride)
    hop, (r, W) = HOP[fps], _grid(fps, stride)
    n_edge = -(-512 // hop)
    fe = LogMelFrontend.get(audio.device)
    lib = _lib.load()
    w = m.dual_stream_attention.kernel_weights(m._compression)
    st = torch.cuda.current_stream().cuda_stream
    n_buf = 1 + 2 * _lib.MAX_EDGE
    off = warm["frame_offsets"]
    checked = 0
    for c in sorted(range(len(lens)), key=lambda c: lens[c])[::3]:
        L = lens[c]
        clip = _clip(audio, lens, c)[None].contiguous()
        n_out = m.num_output_frames(L)
        plain_rows, plain_max = fe.power(clip, hop, (n_out - 1) * stride + W + 1)
        lead_hops = [h for h in _hops(L, fps, stride) if h < W - 1]
        K = len(lead_hops)
        var = [fe.power(clip, hop, K, frame_offset=r + 1 - mm, frame_step=stride, hi_rel=mm) for mm in range(n_edge)]
        expr = torch.empty(1, device="cuda")
        _lib.check(lib.koe_emotion_stream(C.byref(w.struct), eg[c:c + 1].contiguous().data_ptr(), 1, expr.data_ptr(), st))
        for j in sorted({0, 1, K // 2, K - 2, K - 1} & set(range(K))):
            T = lead_hops[j] + 2
            k_plain = T - n_edge
            power = torch.cat([plain_rows[0, :k_plain]] + [var[T - 1 - k][0][0, j:j + 1] for k in range(k_plain, T)])
            fmax = torch.cat([plain_max[0, :k_plain]] + [var[T - 1 - k][1][0, j:j + 1] for k in range(k_plain, T)])
            power, fmax = power.contiguous(), fmax.contiguous()
            out = torch.full((1, 52), float("nan"), device="cuda")
            pw = (C.c_void_p * n_buf)(power.data_ptr(), *[None] * (n_buf - 1))
            fm = (C.c_void_p * n_buf)(fmax.data_ptr(), *[None] * (n_buf - 1))
            _lib.check(lib.koe_dual_stream_windows(C.byref(w.struct), pw, fm, 0, 1, T, 1, 1, T, expr.data_ptr(),
                                                   out.data_ptr(), None, None, _lib.PRECISIONS[precision], st),
                       "koe_dual_stream_windows")
            assert torch.equal(out[0], warm["blendshapes"][int(off[c]) + j]), f"clip {c}, hop {lead_hops[j]} (T = {T})"
            checked += 1
    assert checked > 0


@pytest.mark.parametrize("fps,precision,stride", CONFIGS)
def test_rows_agree_with_a_warmup_stream_pool(fps, precision, stride):
    """A warm-up StreamPool fed the same clips one hop per call emits, at the grid hops, the packed rows within 2 GATE
    (smoothing off)."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, stride)
    hop, (r, W) = HOP[fps], _grid(fps, stride)
    lens = [L for L in (hop, 7 * hop + 5, (W - 1) * hop, W * hop + hop - 1, (W + 9) * hop + 3) if L >= (r + 1) * hop]
    audio, eg = _pack(lens, 31 + fps)
    res = m.forward_varlen(audio, lens, egemaps=eg, warmup=True)
    off = res["frame_offsets"]
    pool = StreamPool(m, len(lens), warmup=True)
    slots = pool.open(eg)
    got = {c: [] for c in range(len(lens))}
    for h in range(max(L // hop for L in lens)):
        live = [c for c, L in enumerate(lens) if L // hop > h]
        x = torch.stack([_clip(audio, lens, c)[h * hop:(h + 1) * hop] for c in live])
        emitted, frames = pool.push([slots[c] for c in live], x)
        assert emitted.tolist() == [slots[c] for c in live]
        for i, c in enumerate(live):
            if h >= r and (h - r) % stride == 0:
                got[c].append(frames[i].clone())
    worst = 0.0
    for c in range(len(lens)):
        want = torch.stack(got[c])
        d = _max_diff(res["blendshapes"][int(off[c]):int(off[c + 1])], want)
        worst = max(worst, d)
        assert d <= 2 * GATE[precision], f"clip {c}: max |d| = {d:.3e}"
    print(f"{fps} fps {precision} stride {stride}: largest deviation from the pool {worst:.3e}")


@pytest.mark.parametrize("fps,precision,stride", [(30, "bf16", 1), (60, "fp32", 2)])
def test_smoothing_restarts_at_each_clip_and_runs_over_its_rows(fps, precision, stride):
    from koemorph_b200 import _lib
    lens = _lengths(fps, stride, 90 + fps, long_clip=(WIN[fps] + 40) * HOP[fps])
    audio, eg = _pack(lens, 41 + fps)
    raw = _model(fps, precision, stride, smoothing=False).forward_varlen(audio, lens, egemaps=eg, warmup=True)
    m = _model(fps, precision, stride, smoothing=True)
    res = m.forward_varlen(audio, lens, egemaps=eg, warmup=True)
    off = res["frame_offsets"]
    assert torch.equal(off, raw["frame_offsets"])
    lib = _lib.load()
    alpha = torch.sigmoid(m.smoothing_alpha.detach().float()).item()
    last = m.prev_blendshapes
    assert last.shape == (len(lens), 52)
    for c in range(len(lens)):
        want = raw["blendshapes"][int(off[c]):int(off[c + 1])].clone()
        _lib.check(lib.koe_ema_scan(want.data_ptr(), 1, want.shape[0], alpha, None, 0, _lib.stream_ptr(want.device)))
        got = res["blendshapes"][int(off[c]):int(off[c + 1])]
        assert torch.equal(got, want), c
        assert torch.equal(last[c], got[-1]), c
        if want.shape[0] > 1:
            assert not torch.equal(got[1:], raw["blendshapes"][int(off[c]) + 1:int(off[c + 1])])


@pytest.mark.parametrize("fps", [30, 60])
def test_launch_counts(fps):
    """The plain call's launches plus n_edge lead-variant launches when a clip has a lead window; an all-short batch has
    no steady edge launches; an empty batch queues nothing."""
    from koemorph_b200 import _lib
    m = _model(fps, "bf16", smoothing=True)
    hop, W = HOP[fps], WIN[fps]
    n_edge = -(-512 // hop)
    # (plain call, warm-up call): frontend, steady edge variants, [lead variants,] emotion, core, EMA
    cases = [([W * hop + 9 * hop, 20000, 5 * hop], 1 + 2 * n_edge + 1 + 1 + 1, 1 + 2 * n_edge + n_edge + 1 + 1 + 1),
             ([20000, 5 * hop], 1 + 1 + 1, 1 + n_edge + 1 + 1 + 1)]   # all short: no steady edge variants
    for lens, plain, warm in cases:
        audio, eg = _pack(lens, 3)
        for warmup, want in ((False, plain), (True, warm)):
            torch.cuda.synchronize()
            _lib.reset_launch_count()
            m.forward_varlen(audio, lens, egemaps=eg, warmup=warmup)
            assert _lib.launch_count() == want, (lens, warmup)
    _lib.reset_launch_count()
    res = m.forward_varlen(torch.zeros(0, device="cuda"), [], egemaps=torch.zeros(0, 264, device="cuda"), warmup=True)
    assert _lib.launch_count() == 0 and res["blendshapes"].shape == (0, 52) and res["frame_offsets"].tolist() == [0]


def test_misuse_raises_and_queues_nothing():
    from koemorph_b200 import _lib
    m = _model(30, "bf16", stride=3)
    lens = [20000, 300, 30000]                      # clip 1 completes no hop
    audio, eg = _pack(lens, 4)
    _lib.reset_launch_count()
    with pytest.raises(ValueError, match="clip 1 of 300 samples completes no hop"):
        m.forward_varlen(audio, lens, egemaps=eg, warmup=True)
    with pytest.raises(ValueError, match="warmup must be a bool"):
        m.forward_varlen(audio, lens, egemaps=eg, warmup=1)
    assert _lib.launch_count() == 0


def test_interleaved_with_plain_packed_forwards_on_one_and_two_streams():
    """Warm-up and plain packed forwards queued back to back (the per-call tables' staging is reused while earlier
    calls are still queued) give what each call gives run alone."""
    m = _model(30, "bf16", smoothing=True)
    hop, W = HOP[30], WIN[30]
    calls = []
    for i in range(6):
        lens = [int(x) for x in np.random.default_rng(i).integers(hop, 2 * W * hop, 5 + i)]
        calls.append((lens,) + _pack(lens, 40 + i) + (i % 2 == 0,))
    alone = [m.forward_varlen(a, l, egemaps=e, warmup=wu)["blendshapes"].clone() for l, a, e, wu in calls]
    torch.cuda.synchronize()
    got = [m.forward_varlen(a, l, egemaps=e, warmup=wu)["blendshapes"] for l, a, e, wu in calls]   # one stream
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream()), s2.wait_stream(torch.cuda.current_stream())
    got2 = []
    for i, (l, a, e, wu) in enumerate(calls):                                                       # two streams
        with torch.cuda.stream(s1 if i % 2 == 0 else s2):
            got2.append((m.forward_varlen(a, l, egemaps=e, warmup=wu)["blendshapes"],
                         m.forward_varlen(a, l, egemaps=e, warmup=not wu)["blendshapes"]))
    torch.cuda.synchronize()
    other = [m.forward_varlen(a, l, egemaps=e, warmup=not wu)["blendshapes"] for l, a, e, wu in calls]
    for i in range(len(calls)):
        assert torch.equal(got[i], alone[i]), i
        assert torch.equal(got2[i][0], alone[i]) and torch.equal(got2[i][1], other[i]), i
