"""GPU tests (-m gpu) of SequentialDualStreamModel.forward_varlen: a packed batch of clips of different lengths as one
native forward.  The reference for every clip is forward() on that clip alone; its rows must match it bit for bit."""
import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O

pytestmark = pytest.mark.gpu

HOP = {30: 533, 60: 266}
WIN = {30: 256, 60: 512}


def _model(fps, precision, stride=1, seed=1235):
    import koemorph_b200 as K
    w = O.make_weights(seed, fps, style="stress")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length=WIN[fps], stride_frames=stride).cuda().eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = precision
    return m, w


def _lengths(fps, stride, seed):
    """Every boundary the issue of per-clip geometry has, plus random lengths, in random order."""
    hop, W = HOP[fps], WIN[fps]
    n_out_len = lambda n, extra=0: (W + (n - 1) * stride) * hop + extra   # a clip with n output frames
    fixed = [0, 1, 300, 511, 5 * hop, 5 * hop + 7, W * hop - 1, W * hop, W * hop + 1, (W + 1) * hop, (W + 1) * hop + 1,
             n_out_len(2), n_out_len(3, hop - 1), n_out_len(31), n_out_len(32, 17), n_out_len(33), n_out_len(64, hop - 1),
             60 * 16000]
    rng = np.random.default_rng(seed)
    lens = fixed + [int(x) for x in rng.integers(0, 3 * W * hop, 24)]
    rng.shuffle(lens)
    return lens


def _pack(lens, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    audio = (torch.rand(sum(lens), generator=g, device="cuda") * 2 - 1) * 0.3
    eg = torch.randn(len(lens), 264, generator=g, device="cuda")
    return audio, eg


def _clip(audio, lens, c):
    s = sum(lens[:c])
    return audio[s:s + lens[c]][None]


@pytest.mark.parametrize("fps,precision,stride", [(30, "fp32", 1), (30, "bf16", 1), (30, "fp32", 3), (30, "bf16", 3),
                                                  (60, "fp32", 1), (60, "bf16", 1), (60, "fp32", 3), (60, "bf16", 3)])
def test_mixed_lengths_equal_each_clips_forward(fps, precision, stride):
    m, _ = _model(fps, precision, stride)
    lens = _lengths(fps, stride, 70 + fps + stride)
    audio, eg = _pack(lens, 11 + fps)
    res = m.forward_varlen(audio, lens, egemaps=eg)
    off = res["frame_offsets"]
    assert off.dtype == torch.int64 and off.device.type == "cpu" and off.shape == (len(lens) + 1,)
    assert [int(off[c + 1] - off[c]) for c in range(len(lens))] == [m.num_output_frames(L) for L in lens]
    assert res["blendshapes"].shape == (int(off[-1]), 52) and res["num_frames"] == int(off[-1]) > 148
    assert res["fps"] == fps and res["emotion_backend"] == "egemaps_input"
    got = res["blendshapes"].clone()
    last = m.prev_blendshapes.clone()
    assert last.shape == (len(lens), 52)
    for c, L in enumerate(lens):
        want = m(_clip(audio, lens, c), egemaps=eg[c:c + 1])["blendshapes"][0]
        assert torch.equal(got[off[c]:off[c + 1]], want), f"clip {c}: length {L}"
        assert torch.equal(last[c], want[-1])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_attention_and_sigmoid_slices(precision):
    m, _ = _model(30, precision)
    hop, W = HOP[30], WIN[30]
    lens = [W * hop + 5 * hop, 16000, 0, W * hop + 1, W * hop + 40 * hop]
    audio, eg = _pack(lens, 5)
    res = m.forward_varlen(audio, lens, egemaps=eg, return_attention=True)
    off = res["frame_offsets"]
    N = int(off[-1])
    assert res["mel_attention_weights"].shape == (N, 28, 80) and res["mel_blendshapes"].shape == (N, 52)
    for c in range(len(lens)):
        want = m(_clip(audio, lens, c), egemaps=eg[c:c + 1], return_attention=True)
        sl = slice(int(off[c]), int(off[c + 1]))
        for key in ("blendshapes", "mel_blendshapes", "emotion_blendshapes"):
            assert torch.equal(res[key][sl], want[key][0]), (c, key)
        if precision == "fp32":
            assert torch.equal(res["mel_attention_weights"][sl], want["mel_attention_weights"][0]), c
        else:  # the tensor-core kernel averages the heads with atomics: the order of the eight additions varies
            torch.testing.assert_close(res["mel_attention_weights"][sl], want["mel_attention_weights"][0], rtol=0, atol=1e-6)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_one_clip_and_equal_lengths_match_forward(precision):
    m, _ = _model(30, precision)
    L = WIN[30] * HOP[30] + 45 * HOP[30] + 100
    audio, eg = _pack([L] * 6, 9)
    one = m.forward_varlen(audio[:L], [L], egemaps=eg[:1])
    assert torch.equal(one["blendshapes"], m(audio[:L][None], egemaps=eg[:1])["blendshapes"][0])
    res = m.forward_varlen(audio, torch.tensor([L] * 6), egemaps=eg.reshape(6, 3, 88))
    want = m(audio.view(6, L), egemaps=eg)["blendshapes"]
    assert torch.equal(res["blendshapes"], want.reshape(-1, 52))


def test_against_the_cpu_oracle():
    m, w = _model(30, "fp32")
    hop, W = HOP[30], WIN[30]
    lens = [W * hop + 7 * hop + 11, 40000, W * hop]
    clips, egs = [], []
    for i, L in enumerate(lens):
        a, e = O.make_inputs(300 + i, 1, L, "speechlike")
        clips.append(a[0]), egs.append(e[0])
    audio = torch.from_numpy(np.concatenate(clips)).cuda()
    eg = torch.from_numpy(np.stack(egs)).cuda()
    res = m.forward_varlen(audio, lens, egemaps=eg)
    off = res["frame_offsets"]
    for c in range(len(lens)):
        want = np.asarray(O.forward_sequence(w, clips[c][None], egs[c][None])["blendshapes"][0])
        got = res["blendshapes"][off[c]:off[c + 1]].cpu().numpy()
        assert got.shape == want.shape and np.abs(got - want).max() <= 2e-6, c


def test_interleaved_with_uniform_forwards_on_one_and_two_streams():
    """Packed and uniform forwards queued back to back (the per-call tables' staging is reused while earlier calls are
    still queued) give what each call gives run alone."""
    m, _ = _model(30, "bf16")
    hop, W = HOP[30], WIN[30]
    batches = []
    for i in range(6):
        lens = [int(x) for x in np.random.default_rng(i).integers(0, 2 * W * hop, 5 + i)]
        batches.append((lens,) + _pack(lens, 40 + i))
    ua, ue = _pack([W * hop + 30 * hop] * 4, 99)
    ua = ua.view(4, -1)
    alone = [m.forward_varlen(a, l, egemaps=e)["blendshapes"].clone() for l, a, e in batches]
    u_alone = m(ua, egemaps=ue)["blendshapes"].clone()
    torch.cuda.synchronize()
    got, ugot = [], []
    for l, a, e in batches:                  # one stream
        got.append(m.forward_varlen(a, l, egemaps=e)["blendshapes"])
        ugot.append(m(ua, egemaps=ue)["blendshapes"])
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream()), s2.wait_stream(torch.cuda.current_stream())
    got2 = []
    for i, (l, a, e) in enumerate(batches):  # two streams
        with torch.cuda.stream(s1 if i % 2 == 0 else s2):
            got2.append((m.forward_varlen(a, l, egemaps=e)["blendshapes"], m(ua, egemaps=ue)["blendshapes"]))
    torch.cuda.synchronize()
    for i in range(len(batches)):
        assert torch.equal(got[i], alone[i]) and torch.equal(ugot[i], u_alone), i
        assert torch.equal(got2[i][0], alone[i]) and torch.equal(got2[i][1], u_alone), i


@pytest.mark.parametrize("fps", [30, 60])
def test_launch_counts(fps):
    from koemorph_b200 import _lib
    m, _ = _model(fps, "bf16")
    hop, W = HOP[fps], WIN[fps]
    n_edge = -(-512 // hop)
    cases = [([W * hop + 9 * hop, 20000, 0], 1 + 2 * n_edge + 1 + 1 + 1),   # frontend, edge variants, emotion, core, EMA
             ([W * hop + 1, 20000], 1 + 2 * n_edge + 1 + 1),                # one frame per clip: nothing to smooth
             ([W * hop, 16000, 0], 1 + 1 + 1)]                              # single windows over whole clips: no edges
    for lens, want in cases:
        audio, eg = _pack(lens, 3)
        torch.cuda.synchronize()
        _lib.reset_launch_count()
        m.forward_varlen(audio, lens, egemaps=eg)
        assert _lib.launch_count() == want, lens
    _lib.reset_launch_count()
    res = m.forward_varlen(torch.zeros(0, device="cuda"), [], egemaps=torch.zeros(0, 264, device="cuda"))
    assert _lib.launch_count() == 0 and res["blendshapes"].shape == (0, 52) and res["frame_offsets"].tolist() == [0]


def test_misuse_raises_and_queues_nothing():
    from koemorph_b200 import _lib
    m, _ = _model(30, "bf16")
    lens = [20000, 30000]
    audio, eg = _pack(lens, 4)
    bad = [dict(audio=audio, lengths=[20000, 29999], egemaps=eg),         # lengths do not add up
           dict(audio=audio, lengths=[50001, -1], egemaps=eg),            # negative length
           dict(audio=audio, lengths=lens, egemaps=eg[:1]),               # egemaps rows
           dict(audio=audio.cpu(), lengths=lens, egemaps=eg),             # audio on the host
           dict(audio=audio.view(1, -1), lengths=lens, egemaps=eg),       # not 1-D
           dict(audio=audio, lengths=torch.tensor(lens).cuda(), egemaps=eg),
           dict(audio=audio, lengths=lens, egemaps=eg, out=torch.empty(3, 52, device="cuda"))]
    _lib.reset_launch_count()
    for kw in bad:
        a = kw.pop("audio")
        with pytest.raises(ValueError):
            m.forward_varlen(a, **kw)
    assert _lib.launch_count() == 0
