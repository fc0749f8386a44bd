"""GPU tests (-m gpu) of StreamPool: streams that open, close and advance on their own clocks.  The reference for every
stream is a one-stream StreamingEngine fed the same hops from the moment the stream was opened; every frame must match
it bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O

pytestmark = pytest.mark.gpu

HOP = {30: 533, 60: 266}
WIN = {30: 256, 60: 512}


def _model(fps, precision, seed=1235):
    import koemorph_b200 as K
    w = O.make_weights(seed, fps, style="stress")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length=WIN[fps]).cuda().eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = precision
    return m


def _clips(seed, n, n_hops, fps):
    audio, eg = O.make_inputs(seed, n, n_hops * HOP[fps], "speechlike")
    return torch.from_numpy(audio).cuda(), torch.from_numpy(eg).cuda()


def _solo(m, clip, eg, fps, egemaps_at=None):
    """Frames of a one-stream StreamingEngine fed `clip` hop by hop: {hop index: (52,) frame}.  egemaps_at: {hop index:
    (264,) eGeMAPS set before that hop}."""
    from koemorph_b200.streaming import StreamingEngine
    hop = HOP[fps]
    eng = StreamingEngine(m, 1)
    eng.set_egemaps(eg[None])
    frames = {}
    for n in range(clip.shape[0] // hop):
        if egemaps_at and n in egemaps_at:
            eng.set_egemaps(egemaps_at[n][None])
        o = eng.step(clip[None, n * hop:(n + 1) * hop].contiguous())
        if o is not None:
            frames[n] = o[0].clone()
    return frames


def _hops(clip, hop_indices, fps):
    hop = HOP[fps]
    return torch.stack([clip[j][n * hop:(n + 1) * hop] for j, n in hop_indices]) if hop_indices else \
        torch.empty(0, hop, device="cuda")


@pytest.mark.parametrize("fps,precision", [(30, "fp32"), (30, "bf16"), (60, "fp32"), (60, "bf16")])
def test_staggered_opens(fps, precision):
    """Six streams open at pool calls 0, 1, 37, 255, 256 and 300 and each push W + 20 hops (their rings wrap): every
    emitted frame equals the stream's solo engine bit for bit and emission starts at the stream's own W-th hop."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision)
    W = WIN[fps]
    n_hops = W + 20
    opens = [0, 1, 37, 255, 256, 300]
    audio, eg = _clips(4100 + fps, len(opens), n_hops, fps)
    pool = StreamPool(m, 8)
    slot_of, got = {}, {j: {} for j in range(len(opens))}
    for call in range(opens[-1] + n_hops):
        for j, c0 in enumerate(opens):
            if c0 == call:
                slot_of[j] = pool.open(eg[j:j + 1])[0]
        live = [j for j in slot_of if call - opens[j] < n_hops]
        emitted, frames = pool.push([slot_of[j] for j in live], _hops(audio, [(j, call - opens[j]) for j in live], fps))
        by_slot = {slot_of[j]: j for j in live}
        for row, s in enumerate(emitted.tolist()):
            j = by_slot[s]
            got[j][call - opens[j]] = frames[row].clone()
        for j in live:
            if call - opens[j] == n_hops - 1:
                pool.close(slot_of[j])
    for j in range(len(opens)):
        want = _solo(m, audio[j], eg[j], fps)
        assert sorted(got[j]) == list(range(W - 1, n_hops)), f"stream {j} emitted at the wrong hops"
        assert sorted(want) == sorted(got[j])
        for n in want:
            assert torch.equal(got[j][n], want[n]), f"stream {j} (opened at call {opens[j]}), hop {n}"
    if precision == "fp32":
        # the pool against the golden-pinned sequence forward, once: stream 2's frames on its whole clip
        ref = m(audio[2:3], egemaps=eg[2:3])["blendshapes"][0]
        pool_frames = torch.stack([got[2][n] for n in range(W - 1, n_hops)])
        assert ref.shape == pool_frames.shape
        assert (pool_frames - ref).abs().max().item() <= 2e-6


@pytest.mark.parametrize("fps,precision", [(30, "fp32"), (60, "bf16")])
def test_independent_clocks(fps, precision):
    """In every call a seeded random ~60 % of the open streams push: each stream's sequence of frames equals its solo
    engine's."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, seed=77)
    W = WIN[fps]
    n_hops = W + 12
    S = 5
    audio, eg = _clips(4200 + fps, S, n_hops, fps)
    pool = StreamPool(m, S)
    slots = pool.open(eg)
    rng = np.random.default_rng(fps)
    pushed = [0] * S
    got = {j: [] for j in range(S)}
    while min(pushed) < n_hops:
        live = [j for j in range(S) if pushed[j] < n_hops and rng.random() < 0.6]
        rng.shuffle(live)
        emitted, frames = pool.push([slots[j] for j in live], _hops(audio, [(j, pushed[j]) for j in live], fps))
        rows = {s: r for r, s in enumerate(emitted.tolist())}
        for j in live:
            assert (slots[j] in rows) == (pushed[j] >= W - 1)
            if slots[j] in rows:
                got[j].append(frames[rows[slots[j]]].clone())
            pushed[j] += 1
    for j in range(S):
        want = _solo(m, audio[j], eg[j], fps)
        assert len(got[j]) == len(want) == n_hops - W + 1
        for i, n in enumerate(sorted(want)):
            assert torch.equal(got[j][i], want[n]), f"stream {j}, frame {i}"


def test_slot_reuse_carries_nothing_over():
    """A loud stream wraps its rings, smooths and closes; a new stream opened into the same slot starts silent.  It must
    equal a fresh solo engine bit for bit from its first (pass-through) frame on, while a neighbour keeps pushing."""
    from koemorph_b200.streaming import StreamPool
    fps, W = 30, WIN[30]
    m = _model(fps, "fp32")
    audio, eg = _clips(4300, 3, 2 * W + 40, fps)
    loud = audio[0] * 8.0
    quiet = audio[1].clone()
    quiet[: (W // 2) * HOP[fps]] = 0.0
    pool = StreamPool(m, 2)
    s_old, s_nb = pool.open(eg[0:1])[0], pool.open(eg[2:3])[0]
    nb_frames = []
    t = 0
    for n in range(W + 30):
        emitted, frames = pool.push([s_old, s_nb], _hops(torch.stack([loud, audio[2]]), [(0, n), (1, t)], fps))
        t += 1
        if emitted.numel():
            nb_frames.append(frames[emitted.tolist().index(s_nb)].clone())
    pool.close(s_old)
    s_new = pool.open(eg[1:2])[0]
    assert s_new == s_old
    got = {}
    for n in range(W + 10):
        emitted, frames = pool.push([s_nb, s_new], _hops(torch.stack([audio[2], quiet]), [(0, t), (1, n)], fps))
        t += 1
        rows = emitted.tolist()
        nb_frames.append(frames[rows.index(s_nb)].clone())
        if s_new in rows:
            got[n] = frames[rows.index(s_new)].clone()
    want = _solo(m, quiet[: (W + 10) * HOP[fps]], eg[1], fps)
    assert sorted(got) == sorted(want) == list(range(W - 1, W + 10))
    for n in want:
        assert torch.equal(got[n], want[n]), f"reused slot, hop {n}"
    want_nb = _solo(m, audio[2][: t * HOP[fps]], eg[2], fps)
    assert len(nb_frames) == len(want_nb)
    for f, n in zip(nb_frames, sorted(want_nb)):
        assert torch.equal(f, want_nb[n]), f"neighbour, hop {n}"


def test_set_egemaps_on_a_subset():
    """set_egemaps on two of four streams: only their expression entries change (as in their solo engines given the same
    update); their mouth entries and the other streams stay bitwise unchanged."""
    import koemorph_b200 as K
    from koemorph_b200.streaming import StreamPool
    fps, W = 30, WIN[30]
    m = _model(fps, "fp32")
    S, n_hops, t_set = 4, W + 4, W + 1
    audio, eg = _clips(4400, S, n_hops, fps)
    _, eg_new = O.make_inputs(4401, S, HOP[fps], "speechlike")
    eg_new = torch.from_numpy(eg_new).cuda()
    changed = [1, 3]
    pool = StreamPool(m, S)
    slots = pool.open(eg)
    got = {j: {} for j in range(S)}
    for n in range(n_hops):
        if n == t_set:
            pool.set_egemaps([slots[j] for j in changed], eg_new[changed])
        emitted, frames = pool.push(slots, _hops(audio, [(j, n) for j in range(S)], fps))
        for j in range(S):
            if slots[j] in emitted.tolist():
                got[j][n] = frames[emitted.tolist().index(slots[j])].clone()
    mouth, expr = list(K.MOUTH_INDICES), list(K.EXPRESSION_INDICES)
    for j in range(S):
        plain = _solo(m, audio[j], eg[j], fps)
        want = _solo(m, audio[j], eg[j], fps, {t_set: eg_new[j]}) if j in changed else plain
        for n in want:
            assert torch.equal(got[j][n], want[n]), f"stream {j}, hop {n}"
            assert torch.equal(got[j][n][mouth], plain[n][mouth])
            if j in changed and n >= t_set:
                assert not torch.equal(got[j][n][expr], plain[n][expr])
            else:
                assert torch.equal(got[j][n], plain[n])


@pytest.mark.parametrize("fps,counts", [(30, (6, 4, 0)), (60, (8, 6, 0))])
def test_launch_counts(fps, counts):
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, "fp32")
    assert m.use_temporal_smoothing
    W, hop = WIN[fps], HOP[fps]
    pool = StreamPool(m, 3)
    a = pool.open(torch.zeros(1, 264, device="cuda"))[0]
    x = torch.randn(2, hop, device="cuda") * 0.1
    for _ in range(W - 1):
        pool.push([a], x[:1])
    b = pool.open(torch.zeros(1, 264, device="cuda"))[0]
    torch.cuda.synchronize()
    seen = []
    for slots in ([a, b], [b], []):
        _lib.reset_launch_count()
        emitted, frames = pool.push(slots, x[:len(slots)])
        seen.append(_lib.launch_count())
        assert emitted.tolist() == ([a] if slots == [a, b] else [])
        assert emitted.dtype == torch.int64 and frames.shape == (emitted.numel(), 52) and frames.is_cuda
    assert tuple(seen) == counts


def test_misuse_is_refused_before_any_kernel():
    """A push to a closed slot, a slot listed twice, a slot >= capacity, a wrong hop_audio shape and an open beyond
    capacity all raise; the native entries return KOE_E_INVALID and the clocks do not move."""
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    fps, W, hop = 30, WIN[30], HOP[30]
    m = _model(fps, "fp32")
    pool = StreamPool(m, 3)
    a, b = pool.open(torch.zeros(2, 264, device="cuda"))
    pool.close(b)
    x = torch.zeros(2, hop, device="cuda")
    with pytest.raises(ValueError):
        pool.push([b], x[:1])                      # closed
    with pytest.raises(ValueError):
        pool.push([a, a], x)                       # listed twice
    with pytest.raises(ValueError):
        pool.push([3], x[:1])                      # slot >= capacity
    with pytest.raises(ValueError):
        pool.push([a], x)                          # hop_audio rows != slots
    with pytest.raises(ValueError):
        pool.push([a], torch.zeros(1, hop + 1, device="cuda"))
    with pytest.raises(ValueError):
        pool.push([a], x[:1].double())
    with pytest.raises(ValueError):
        pool.open(torch.zeros(3, 264, device="cuda"))   # 2 slots free
    with pytest.raises(ValueError):
        pool.set_egemaps([b], torch.zeros(1, 264, device="cuda"))
    lib = _lib.load()
    pool._current_args()
    pool._args.hop_audio = x.data_ptr()
    n_emitted = C.c_int(0)
    st = torch.cuda.current_stream().cuda_stream

    def native_push(slots):
        s = torch.tensor(slots, dtype=torch.int32)
        return lib.koe_stream_pool_push(pool._h, pool._args_ref, s.data_ptr(), len(slots), pool._emitted.data_ptr(),
                                        C.byref(n_emitted), st)
    _lib.reset_launch_count()
    assert native_push([b]) == -1
    assert native_push([a, a]) == -1
    assert native_push([3]) == -1
    assert native_push([-1]) == -1
    buf = torch.empty(3, dtype=torch.int32)
    assert lib.koe_stream_pool_open(pool._h, 3, buf.data_ptr()) == -1
    assert _lib.launch_count() == 0
    # the refused calls moved no clock: stream a still emits first at its own W-th hop
    for n in range(W):
        emitted, _ = pool.push([a], x[:1])
        assert emitted.tolist() == ([a] if n == W - 1 else [])
