"""GPU tests (-m gpu) of StreamPool.push_hops: streams that advance by several hops in one call.  The reference for
every stream is a one-stream StreamingEngine fed the same hops one at a time from the moment the stream was opened;
every frame must match it bit for bit, whatever the counts of the calls were."""
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


class _Driver:
    """Feeds stream j of `audio` (its own clip, from its hop 0) to a pool and keeps every frame by (stream, hop)."""

    def __init__(self, pool, audio, eg, fps):
        self.pool, self.audio, self.eg, self.hop, self.W = pool, audio, eg, HOP[fps], WIN[fps]
        self.slot, self.pushed, self.got = {}, {}, {}

    def open(self, j):
        self.slot[j] = self.pool.open(self.eg[j:j + 1])[0]
        self.pushed[j], self.got[j] = 0, {}
        return self.slot[j]

    def close(self, j):
        self.pool.close(self.slot.pop(j))

    def _audio(self, plan):
        hop = self.hop
        parts = [self.audio[j][self.pushed[j] * hop:(self.pushed[j] + c) * hop] for j, c in plan]
        return torch.cat(parts) if parts else torch.empty(0, device="cuda")

    def _keep(self, plan, rows):
        want = [(self.slot[j], h) for j, c in plan for h in range(self.pushed[j], self.pushed[j] + c) if h >= self.W - 1]
        assert [(s, h) for s, h, _ in rows] == want, "rows not grouped by stream in call order, hops ascending"
        by_slot = {self.slot[j]: j for j, _ in plan}
        for s, h, f in rows:
            self.got[by_slot[s]][h] = f.clone()
        for j, c in plan:
            self.pushed[j] += c

    def push_hops(self, plan, flat=True):
        """plan: [(stream, count)] in call order."""
        x = self._audio(plan)
        slots, hops, frames = self.pool.push_hops([self.slot[j] for j, _ in plan], x if flat else x.view(-1, self.hop),
                                                  [c for _, c in plan])
        assert slots.dtype == hops.dtype == torch.int64 and not slots.is_cuda and not hops.is_cuda
        assert frames.shape == (slots.numel(), 52) and frames.is_cuda
        self._keep(plan, list(zip(slots.tolist(), hops.tolist(), frames)))

    def push(self, js):
        plan = [(j, 1) for j in js]
        x = self._audio(plan).view(-1, self.hop)
        emitted, frames = self.pool.push([self.slot[j] for j in js], x)
        by_slot = {self.slot[j]: j for j in js}
        self._keep(plan, [(s, self.pushed[by_slot[s]], f) for s, f in zip(emitted.tolist(), frames)])

    def check(self, m, fps, j, egemaps_at=None, eg=None, audio=None):
        clip = (self.audio[j] if audio is None else audio)[: self.pushed[j] * self.hop]
        want = _solo(m, clip, self.eg[j] if eg is None else eg, fps, egemaps_at)
        assert sorted(self.got[j]) == sorted(want) == list(range(self.W - 1, self.pushed[j])), f"stream {j}: wrong hops"
        for n in want:
            assert torch.equal(self.got[j][n], want[n]), f"stream {j}, hop {n}"


def _random_plan(rng, d, live, n_hops, max_hops, straddled, p_push=0.8):
    """A seeded burst per live stream (count in [1, max_hops]); where a burst can take a stream across its hop W - 1
    from before it, the first such burst does."""
    plan = []
    for j in live:
        left = n_hops - d.pushed[j]
        if left == 0 or rng.random() > p_push:
            continue
        c = min(int(rng.integers(1, max_hops + 1)), left)
        p = d.pushed[j]
        if j not in straddled and p < d.W - 1 < p + min(max_hops, left):
            c = max(c, d.W - p)                   # hops p .. W - 1: the window completes part-way through
            straddled.add(j)
        elif j not in straddled and p + c == d.W - 1 and c > 1:
            c -= 1                                # (a burst starting at hop W - 1 would not cross it)
        plan.append((j, c))
    rng.shuffle(plan)
    return plan


@pytest.mark.parametrize("fps,precision", [(30, "fp32"), (30, "bf16"), (60, "fp32"), (60, "bf16")])
def test_staggered_bursts(fps, precision):
    """Six streams open at pool calls 0, 1, 7, 19, 20 and 33 and are driven for W + 3 max_hops hops with seeded counts in
    [1, max_hops]; a burst takes each stream across its first window.  Every frame equals the solo engine's."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision)
    W, H = WIN[fps], 8
    n_hops = W + 3 * H
    opens = [0, 1, 7, 19, 20, 33]
    audio, eg = _clips(5100 + fps, len(opens), n_hops, fps)
    pool = StreamPool(m, 8, max_hops=H)
    d = _Driver(pool, audio, eg, fps)
    rng = np.random.default_rng(fps * 10 + len(precision))
    straddled = set()
    call = 0
    while call <= opens[-1] or any(d.pushed[j] < n_hops for j in d.pushed):
        for j, c0 in enumerate(opens):
            if c0 == call:
                d.open(j)
        d.push_hops(_random_plan(rng, d, list(d.slot), n_hops, H, straddled), flat=call % 2 == 0)
        call += 1
    assert straddled == set(range(len(opens)))
    for j in range(len(opens)):
        d.check(m, fps, j)
    if precision == "fp32" and fps == 30:
        # against the golden-pinned sequence forward, once: stream 2's frames on its whole clip
        ref = m(audio[2:3], egemaps=eg[2:3])["blendshapes"][0]
        frames = torch.stack([d.got[2][n] for n in range(W - 1, n_hops)])
        assert ref.shape == frames.shape
        assert (frames - ref).abs().max().item() <= 2e-6


@pytest.mark.parametrize("fps,precision", [(30, "bf16"), (60, "fp32")])
def test_max_hops_one_equals_the_default_pool(fps, precision):
    """A pool of max_hops = 1 driven by push_hops and a default pool driven by push give the same frames."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, seed=91)
    W = WIN[fps]
    S, n_hops = 3, W + 6
    audio, eg = _clips(5200 + fps, S, n_hops, fps)
    a, b = StreamPool(m, S, max_hops=1), StreamPool(m, S)
    assert a.ring_frames == b.ring_frames == W and a.out.shape == b.out.shape and a.tables.shape == b.tables.shape
    da, db = _Driver(a, audio, eg, fps), _Driver(b, audio, eg, fps)
    rng = np.random.default_rng(3)
    for j in range(S):
        da.open(j), db.open(j)
    while min(da.pushed.values()) < n_hops:
        live = [j for j in range(S) if da.pushed[j] < n_hops and (rng.random() < 0.7 or da.pushed[j] == 0)]
        da.push_hops([(j, 1) for j in live])
        db.push(live)
    for j in range(S):
        assert sorted(da.got[j]) == sorted(db.got[j]) == list(range(W - 1, n_hops))
        for n in da.got[j]:
            assert torch.equal(da.got[j][n], db.got[j][n]), f"stream {j}, hop {n}"
    da.check(m, fps, 0)


@pytest.mark.parametrize("fps,precision", [(30, "bf16"), (60, "bf16")])
def test_push_and_push_hops_interleaved(fps, precision):
    """On a pool of max_hops = 4, plain pushes and bursts alternate call by call: each stream's frames equal its solo
    engine's."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, seed=92)
    W, H = WIN[fps], 4
    S, n_hops = 3, W + 3 * H
    audio, eg = _clips(5300 + fps, S, n_hops, fps)
    pool = StreamPool(m, S, max_hops=H)
    d = _Driver(pool, audio, eg, fps)
    for j in range(S):
        d.open(j)
    rng = np.random.default_rng(4)
    straddled = set()
    call = 0
    while min(d.pushed.values()) < n_hops:
        if call % 2:
            d.push([j for j in range(S) if d.pushed[j] < n_hops])
        else:
            d.push_hops(_random_plan(rng, d, range(S), n_hops, H, straddled, p_push=1.0))
        call += 1
    for j in range(S):
        d.check(m, fps, j)


@pytest.mark.parametrize("fps,precision,max_hops", [(30, "bf16", 2), (30, "fp32", 8), (60, "bf16", 8), (30, "bf16", 30)])
def test_every_count_at_max_hops(fps, precision, max_hops):
    """Every burst is max_hops long -- the longest reach back into the rings (W + max_hops - 1 - lag rows).  Stream 1
    opens one call later and stream 2 has an odd start, so bursts cross the first window at different offsets."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, seed=93)
    W, H = WIN[fps], max_hops
    n_hops = W + 3 * H + (-(W + 3 * H)) % H        # a whole number of bursts
    audio, eg = _clips(5400 + fps + H, 3, n_hops + H, fps)
    pool = StreamPool(m, 3, max_hops=H)
    d = _Driver(pool, audio, eg, fps)
    d.open(0)
    d.push_hops([(0, H)])
    d.open(1)
    d.open(2)
    d.push_hops([(2, 1)])                          # stream 2 is then one hop off the H grid
    while d.pushed[1] < n_hops:
        d.push_hops([(j, H) for j in range(3) if d.pushed[j] + H <= n_hops + 1])
    for j in range(3):
        d.check(m, fps, j)


def test_slot_reuse_then_burst():
    """A loud stream wraps its rings, smooths and closes mid-burst-sequence; a new stream opened into the same slot takes
    its first window in one burst.  It equals a fresh solo engine from its first frame on; a neighbour keeps going."""
    from koemorph_b200.streaming import StreamPool
    fps, W, H = 30, WIN[30], 8
    m = _model(fps, "fp32")
    audio, eg = _clips(5500, 3, 2 * W + 5 * H, fps)
    audio[0] *= 8.0
    audio[1, : (W // 2) * HOP[fps]] = 0.0          # the new stream starts silent
    pool = StreamPool(m, 2, max_hops=H)
    d = _Driver(pool, audio, eg, fps)
    s_old = d.open(0)
    d.open(2)
    while d.pushed[0] < W + 3 * H:
        d.push_hops([(0, H), (2, 3)])
    d.close(0)
    assert d.open(1) == s_old
    d.push_hops([(2, 1), (1, H)])
    while d.pushed[1] < W - 3:
        d.push_hops([(1, H), (2, 5)] if d.pushed[1] + H <= W - 3 else [(1, W - 3 - d.pushed[1])])
    d.push_hops([(2, 2), (1, H)])                  # hops W - 3 .. W + 4: the first window completes in this burst
    d.push_hops([(1, H)])
    d.check(m, fps, 1)
    d.check(m, fps, 2)


@pytest.mark.parametrize("smoothing", [True, False])
def test_set_egemaps_on_a_subset_between_bursts(smoothing):
    """set_egemaps on two of four streams between two bursts: their frames from the next burst on follow the new
    expression input (as their solo engines given the same update before that hop), the others stay unchanged; with and
    without temporal smoothing."""
    import koemorph_b200 as K
    from koemorph_b200.streaming import StreamPool
    fps, W, H = 30, WIN[30], 6
    m = _model(fps, "bf16")
    m.use_temporal_smoothing = smoothing
    S, n_hops = 4, W + 4 * H
    audio, eg = _clips(5600, S, n_hops, fps)
    _, eg_new = O.make_inputs(5601, S, HOP[fps], "speechlike")
    eg_new = torch.from_numpy(eg_new).cuda()
    changed = [1, 3]
    pool = StreamPool(m, S, max_hops=H)
    d = _Driver(pool, audio, eg, fps)
    for j in range(S):
        d.open(j)
    t_set = {}
    while min(d.pushed.values()) < n_hops:
        if not t_set and d.pushed[1] >= W + H:
            pool.set_egemaps([d.slot[j] for j in changed], eg_new[changed])
            t_set = {j: d.pushed[j] for j in changed}
        d.push_hops([(j, min(H if j % 2 else H - 1, n_hops - d.pushed[j])) for j in range(S) if d.pushed[j] < n_hops])
    mouth, expr = list(K.MOUTH_INDICES), list(K.EXPRESSION_INDICES)
    for j in range(S):
        if j in changed:
            d.check(m, fps, j, egemaps_at={t_set[j]: eg_new[j]})
            plain = _solo(m, audio[j], eg[j], fps)
            n_after = [n for n in plain if n >= t_set[j]]
            assert n_after and all(torch.equal(d.got[j][n][mouth], plain[n][mouth]) for n in plain)
            assert not any(torch.equal(d.got[j][n][expr], plain[n][expr]) for n in n_after)
        else:
            d.check(m, fps, j)


@pytest.mark.parametrize("fps,counts", [(30, (6, 4, 5)), (60, (8, 6, 7))])
def test_launch_counts_do_not_depend_on_the_counts(fps, counts):
    """6 kernels per call at 30 fps (8 at 60) when a frame completes, 4 (6) when none does, one fewer without smoothing
    -- for bursts of any length; none for an empty call."""
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, "bf16")
    assert m.use_temporal_smoothing
    W, hop, H = WIN[fps], HOP[fps], 5
    emit, quiet, unsmoothed = counts
    pool = StreamPool(m, 3, max_hops=H)
    a = pool.open(torch.zeros(1, 264, device="cuda"))[0]
    x = torch.randn(3 * H * hop, device="cuda") * 0.1
    pushed_a = 0
    while W - 1 - pushed_a > H:
        pool.push_hops([a], x[:H * hop], [H])
        pushed_a += H
    left = W - 1 - pushed_a                       # a's first frame completes at its (left + 1)-th next hop
    assert 1 <= left <= H
    b, c = pool.open(torch.zeros(2, 264, device="cuda"))
    torch.cuda.synchronize()
    for slots, cnt, want in (([b, c], [H, 1], quiet), ([b], [2], quiet), ([b, a], [1, left], quiet),
                             ([a, b, c], [1, H, 3], emit), ([a], [H], emit), ([c, a], [2, 1], emit)):
        _lib.reset_launch_count()
        slots_out, _, _ = pool.push_hops(slots, x[:sum(cnt) * hop], cnt)
        assert _lib.launch_count() == want, (slots, cnt)
        assert (slots_out.numel() > 0) == (want == emit)
    m.use_temporal_smoothing = False
    _lib.reset_launch_count()
    slots_out, _, _ = pool.push_hops([a, b], x[:(H + 4) * hop], [H, 4])
    assert slots_out.tolist() == [a] * H and _lib.launch_count() == unsmoothed
    _lib.reset_launch_count()
    assert pool.push_hops([], x[:0], [])[0].numel() == 0 and _lib.launch_count() == 0


def test_misuse_is_refused_before_any_kernel():
    """Counts of 0 or above max_hops, counts and slots of different lengths, audio of the wrong length, a slot listed
    twice and a closed slot all raise; the native entry returns KOE_E_INVALID, no kernel is queued and no clock moves."""
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    fps, W, hop, H = 30, WIN[30], HOP[30], 4
    m = _model(fps, "fp32")
    pool = StreamPool(m, 3, max_hops=H)
    a, b = pool.open(torch.zeros(2, 264, device="cuda"))
    pool.close(b)
    x = torch.zeros(2 * H * hop, device="cuda")
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    for slots, counts, n in (([a], [0], 0), ([a], [H + 1], H + 1), ([a], [1, 1], 2), ([a], [2], 3), ([a], [2], 1),
                             ([a, a], [1, 1], 2), ([b], [1], 1), ([3], [1], 1), ([a], [-1], 0)):
        with pytest.raises(ValueError):
            pool.push_hops(slots, x[:n * hop], counts)
    with pytest.raises(ValueError):
        pool.push_hops([a], x[:hop].double(), [1])
    with pytest.raises(ValueError):
        pool.push_hops([a], x[:hop], torch.ones(1))              # float counts
    with pytest.raises(ValueError):
        pool.push_hops([a], x[:2 * hop].view(2, hop).t().contiguous(), [2])   # (hop, 2): not (2, hop)
    lib = _lib.load()
    pool._current_args()
    pool._args.hop_audio = x.data_ptr()
    n_emitted = C.c_int(0)
    st = torch.cuda.current_stream().cuda_stream

    def native(slots, counts):
        s, c = torch.tensor(slots, dtype=torch.int32), torch.tensor(counts, dtype=torch.int32)
        return lib.koe_stream_pool_push_hops(pool._h, pool._args_ref, s.data_ptr(), c.data_ptr(), len(slots),
                                             pool._emitted.data_ptr(), pool._emitted_hop.data_ptr(), C.byref(n_emitted),
                                             st)
    for slots, counts in (([a], [0]), ([a], [H + 1]), ([a, a], [1, 1]), ([b], [1]), ([3], [1]), ([-1], [1])):
        assert native(slots, counts) == -1
        assert n_emitted.value == 0
    assert _lib.launch_count() == 0
    # the refused calls moved no clock: stream a still emits first at its own hop W - 1
    pushed = 0
    while pushed < W + H:
        c = min(H, W + H - pushed)
        slots, hops, _ = pool.push_hops([a], x[:c * hop], [c])
        assert hops.tolist() == [h for h in range(pushed, pushed + c) if h >= W - 1]
        pushed += c
