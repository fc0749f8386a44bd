"""GPU tests (-m gpu) of warm-up stream pools (StreamPool(..., warmup=True)): every pushed hop emits, from each stream's
hop 0 on.  Before hop W - 1 a frame is SimplifiedDualStreamModel.forward on the audio heard so far; from hop W - 1 on
it is bit for bit the frame of a pool without warm-up (smoothing off); the smoothing runs over every frame since the
stream opened."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O

pytestmark = pytest.mark.gpu

HOP = {30: 533, 60: 266}
WIN = {30: 256, 60: 512}
GATE = {"fp32": 2e-6, "bf16": 1e-4}   # against the fp32 forward, as tests/test_gpu_streaming.py
CONFIGS = [(30, "fp32"), (30, "bf16"), (60, "fp32"), (60, "bf16")]


def _model(fps, precision, smoothing, seed=1235):
    import koemorph_b200 as K
    w = O.make_weights(seed, fps, style="stress")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length=WIN[fps]).cuda().eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = precision
    m.use_temporal_smoothing = smoothing
    return m


def _clips(seed, n, n_hops, fps):
    audio, eg = O.make_inputs(seed, n, n_hops * HOP[fps], "speechlike")
    return torch.from_numpy(audio).cuda(), torch.from_numpy(eg).cuda()


class _Driver:
    """Feeds stream j of `audio` (its own clip, from its hop 0) to a pool and keeps every frame by (stream, hop)."""

    def __init__(self, pool, audio, eg):
        self.pool, self.audio, self.eg, self.hop, self.W = pool, audio, eg, pool.hop, pool.W
        self.slot, self.pushed, self.got = {}, {}, {}

    def open(self, j, eg=None):
        self.slot[j] = self.pool.open(self.eg[j:j + 1] if eg is None else eg[None])[0]
        self.pushed[j], self.got[j] = 0, {}
        return self.slot[j]

    def close(self, j):
        self.pool.close(self.slot.pop(j))

    def _keep(self, plan, rows):
        # a warm-up pool emits at every hop: rows grouped by stream in call order, hops ascending
        want = [(self.slot[j], h) for j, c in plan for h in range(self.pushed[j], self.pushed[j] + c)
                if self.pool.warmup or h >= self.W - 1]
        assert [(s, h) for s, h, _ in rows] == want
        by_slot = {self.slot[j]: j for j, _ in plan}
        for s, h, f in rows:
            self.got[by_slot[s]][h] = f.clone()
        for j, c in plan:
            self.pushed[j] += c

    def push(self, js):
        """One hop of each stream js, by StreamPool.push."""
        plan = [(j, 1) for j in js]
        x = torch.stack([self.audio[j][self.pushed[j] * self.hop:(self.pushed[j] + 1) * self.hop] for j in js]) if js \
            else torch.empty(0, self.hop, device="cuda")
        emitted, frames = self.pool.push([self.slot[j] for j in js], x)
        by_slot = {self.slot[j]: j for j in js}
        self._keep(plan, [(s, self.pushed[by_slot[s]], f) for s, f in zip(emitted.tolist(), frames)])

    def push_hops(self, plan):
        """plan: [(stream, count)] in call order, by StreamPool.push_hops."""
        parts = [self.audio[j][self.pushed[j] * self.hop:(self.pushed[j] + c) * self.hop] for j, c in plan]
        x = torch.cat(parts) if parts else torch.empty(0, device="cuda")
        slots, hops, frames = self.pool.push_hops([self.slot[j] for j, _ in plan], x, [c for _, c in plan])
        self._keep(plan, list(zip(slots.tolist(), hops.tolist(), frames)))


def _max_diff(a, b):
    return (a.double() - b.double()).abs().max().item()


@functools.lru_cache(maxsize=None)
def _staggered(fps, precision):
    """Four streams opened at pool calls 0, 1, 6 and 17 of a warm-up pool and of a plain pool (smoothing off), one hop
    per stream and call, until each has pushed W + 3 hops."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, smoothing=False)
    W = WIN[fps]
    opens, n_hops = [0, 1, 6, 17], W + 3
    audio, eg = _clips(6100 + fps, len(opens), n_hops, fps)
    warm = _Driver(StreamPool(m, 6, warmup=True), audio, eg)
    plain = _Driver(StreamPool(m, 6), audio, eg)
    call = 0
    while call <= opens[-1] or any(p < n_hops for p in warm.pushed.values()):
        for d in (warm, plain):
            for j, c0 in enumerate(opens):
                if c0 == call:
                    d.open(j)
            d.push([j for j in d.slot if d.pushed[j] < n_hops])
        call += 1
    return audio, eg, n_hops, warm.got, plain.got


@pytest.mark.parametrize("fps,precision", CONFIGS)
def test_frame_at_every_hop_is_the_forward_on_the_audio_so_far(fps, precision):
    """Hop h < W - 1: SimplifiedDualStreamModel.forward on the first (h + 1) hops (T = h + 2 frames: T = 2, T < 3, and
    T = 255 .. 257 around mel_seq at 30 fps); hop h >= W - 1: the last frame of the sequence forward on them."""
    audio, eg, n_hops, got, _ = _staggered(fps, precision)
    ref = _model(fps, "fp32", smoothing=False)
    hop, W, S = HOP[fps], WIN[fps], audio.shape[0]
    worst = 0.0
    for j in range(S):
        assert sorted(got[j]) == list(range(n_hops)), f"stream {j} did not emit at every hop"
    for h in range(n_hops):
        prefix = audio[:, :(h + 1) * hop].contiguous()
        frames = torch.stack([got[j][h] for j in range(S)])
        wants = []
        if h <= W - 1:
            wants.append(ref.forward_single_frame(prefix, egemaps=eg)["blendshapes"])
        if h >= W - 1:
            wants.append(ref(prefix, egemaps=eg)["blendshapes"][:, -1])
        for want in wants:
            d = _max_diff(frames, want)
            worst = max(worst, d)
            assert d <= GATE[precision], f"hop {h}: max |d| = {d:.3e}"
    print(f"{fps} fps {precision}: largest deviation {worst:.3e} over {n_hops} hops")


@pytest.mark.parametrize("fps,precision", CONFIGS)
def test_frames_from_hop_w_minus_1_equal_a_plain_pool(fps, precision):
    _, _, n_hops, warm, plain = _staggered(fps, precision)
    W = WIN[fps]
    for j in warm:
        assert sorted(plain[j]) == list(range(W - 1, n_hops))
        for h in plain[j]:
            assert torch.equal(warm[j][h], plain[j][h]), f"stream {j}, hop {h}"


@pytest.mark.parametrize("fps,precision", CONFIGS)
def test_warmup_window_equals_the_public_core_on_its_rows(fps, precision):
    """After a push, a warm-up window's T rows -- the plain ring rows, then the hop's window-end staging rows -- run
    through koe_dual_stream_windows as one clip without edge variants give the pool's frame bit for bit."""
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, smoothing=False)
    W, n_edge = WIN[fps], -(-512 // HOP[fps])
    check = {0, 1, 2, 3, W // 2, W - 3, W - 2}
    audio, eg = _clips(6200 + fps, 2, W, fps)
    pool = StreamPool(m, 3, warmup=True)
    d = _Driver(pool, audio, eg)
    d.open(0)
    lib = _lib.load()
    w = m.dual_stream_attention.kernel_weights(m._compression)
    st = torch.cuda.current_stream().cuda_stream
    n_buf = 1 + 2 * _lib.MAX_EDGE
    checked = 0
    while True:
        if 1 not in d.slot and d.pushed[0] == 1:
            d.open(1)                              # stream 1 runs one hop behind stream 0
        js = [j for j in d.slot if d.pushed[j] < W - 1]
        if not js:
            break
        d.push(js)
        for e, j in enumerate(js):                 # staged hop e of this call is stream js[e]'s
            h = d.pushed[j] - 1
            if h not in check:
                continue
            s, T = d.slot[j], h + 2
            k_ring = T - n_edge                    # frames 0 .. T - 1 - n_edge: ring rows 0 .. (frame g in row g)
            variants = [2 + 2 * (T - 1 - k) for k in range(k_ring, T)]
            power = torch.cat([pool.ring_f[s, :k_ring], pool.stage[e, variants]]).contiguous()
            fmax = torch.cat([pool.fmax_f[s, :k_ring], pool.stage_max[e, variants]]).contiguous()
            out = torch.full((1, 52), float("nan"), device="cuda")
            pw = (C.c_void_p * n_buf)(power.data_ptr(), *[None] * (n_buf - 1))
            fm = (C.c_void_p * n_buf)(fmax.data_ptr(), *[None] * (n_buf - 1))
            _lib.check(lib.koe_dual_stream_windows(C.byref(w.struct), pw, fm, 0, 1, T, 1, 1, T,
                                                   pool.expr[s:s + 1].data_ptr(), out.data_ptr(), None, None,
                                                   _lib.PRECISIONS[precision], st), "koe_dual_stream_windows")
            assert torch.equal(out[0], d.got[j][h]), f"stream {j}, hop {h} (T = {T})"
            checked += 1
    assert checked == 2 * len(check)


def _burst_plan(rng, d, n_hops, max_hops, straddled):
    """A seeded burst per live stream; where a burst can take a stream across its hop W - 1 from before it, the first
    such burst does."""
    plan = []
    for j in list(d.slot):
        left = n_hops - d.pushed[j]
        if left == 0 or rng.random() > 0.8:
            continue
        c = min(int(rng.integers(1, max_hops + 1)), left)
        p = d.pushed[j]
        if j not in straddled and p < d.W - 1 < p + min(max_hops, left):
            c = max(c, d.W - p)
            straddled.add(j)
        elif j not in straddled and p + c == d.W - 1 and c > 1:
            c -= 1                                 # (a burst starting at hop W - 1 would not cross it)
        plan.append((j, c))
    rng.shuffle(plan)
    return plan


@pytest.mark.parametrize("fps,precision,max_hops", [(30, "bf16", 2), (30, "fp32", 8), (60, "bf16", 8), (30, "bf16", 30)])
def test_bursts_equal_one_push_per_hop(fps, precision, max_hops):
    """Seeded bursts from hop 0 on, across hop W - 1 and in steady state, with streams in warm-up and in steady state
    in the same calls (smoothing on): every frame equals that of one push per hop on a max_hops = 1 warm-up pool."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, smoothing=True)
    W, H = WIN[fps], max_hops
    n_hops = W + 3 * H
    audio, eg = _clips(6300 + fps + H, 4, n_hops, fps)
    d = _Driver(StreamPool(m, 5, max_hops=H, warmup=True), audio, eg)
    d.open(0)
    d.open(1)
    rng = np.random.default_rng(fps + H)
    straddled, mixed, call = set(), 0, 0
    while len(d.slot) < 4 or any(p < n_hops for p in d.pushed.values()):
        if 2 not in d.slot and d.pushed[0] >= W:
            d.open(2)                              # opens while stream 0 is past its warm-up
        if 3 not in d.slot and call == 3:
            d.open(3)
        plan = _burst_plan(rng, d, n_hops, H, straddled)
        states = {d.pushed[j] >= W - 1 for j, _ in plan}
        mixed += len(states) == 2
        d.push_hops(plan)
        call += 1
    assert straddled == {0, 1, 2, 3} and mixed > 0
    ref = _Driver(StreamPool(m, 4, warmup=True), audio, eg)
    for j in range(4):
        ref.open(j)
    for _ in range(n_hops):
        ref.push(list(range(4)))
    for j in range(4):
        assert sorted(d.got[j]) == sorted(ref.got[j]) == list(range(n_hops))
        for h in range(n_hops):
            assert torch.equal(d.got[j][h], ref.got[j][h]), f"stream {j}, hop {h}"


@pytest.mark.parametrize("fps,precision", [(30, "bf16"), (60, "fp32")])
def test_smoothing_runs_from_hop_0(fps, precision):
    """With smoothing on, the frames are the float32 chain y = fmaf(1 - a, y, a x) from hop 0 over the smoothing-off
    frames (within 1 ulp: the chain is evaluated in float64 here, which may round twice)."""
    from koemorph_b200.streaming import StreamPool
    W = WIN[fps]
    n_hops = W + 4
    audio, eg = _clips(6400 + fps, 2, n_hops, fps)
    runs = {}
    for smoothing in (True, False):
        m = _model(fps, precision, smoothing=smoothing)
        d = _Driver(StreamPool(m, 2, max_hops=3, warmup=True), audio, eg)
        d.open(0)
        d.push_hops([(0, 2)])
        d.open(1)
        while min(d.pushed.values()) < n_hops:
            d.push_hops([(j, min(1 + (d.pushed[j] % 3), n_hops - d.pushed[j])) for j in (1, 0) if d.pushed[j] < n_hops])
        runs[smoothing] = d.got
    alpha = np.float32(torch.sigmoid(m.smoothing_alpha.detach().float()).item())
    one_minus = np.float32(1.0) - alpha
    for j in (0, 1):
        x = torch.stack([runs[False][j][h] for h in range(n_hops)]).cpu().numpy()
        got = torch.stack([runs[True][j][h] for h in range(n_hops)]).cpu().numpy()
        want = np.empty_like(x)
        y = x[0]
        want[0] = y
        for h in range(1, n_hops):
            y = (np.float64(one_minus) * y.astype(np.float64) + (alpha * x[h]).astype(np.float64)).astype(np.float32)
            want[h] = y
        assert np.array_equal(got[0], x[0]), "the hop-0 frame passes the smoothing unchanged"
        ulps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))
        assert ulps.max() <= 1, f"stream {j}: {ulps.max()} ulp"
        assert not np.array_equal(got[1:], x[1:])


def test_slot_reuse_and_set_egemaps():
    """A stream closed mid-warm-up and a new one opened into its slot: the new stream's frames are those of a fresh pool.
    set_egemaps on one of two streams between pushes changes that stream's expression entries only."""
    import koemorph_b200 as K
    from koemorph_b200.streaming import StreamPool
    fps, W = 30, WIN[30]
    m = _model(fps, "bf16", smoothing=True)
    n_hops = W + 3
    audio, eg = _clips(6500, 3, n_hops, fps)
    audio[0] *= 8.0                                # the closed stream is loud
    _, eg_new = O.make_inputs(6501, 1, HOP[fps], "speechlike")
    eg_new = torch.from_numpy(eg_new).cuda()[0]
    t_set = W // 2
    d = _Driver(StreamPool(m, 2, warmup=True), audio, eg)
    s_old = d.open(0)
    d.open(1)
    for _ in range(W // 3):
        d.push([0, 1])
    d.close(0)
    assert d.open(2) == s_old
    while d.pushed[2] < n_hops:
        if d.pushed[1] == t_set:
            d.pool.set_egemaps([d.slot[1]], eg_new[None])
        d.push([j for j in (1, 2) if d.pushed[j] < n_hops])

    def fresh(j, set_at=None):
        r = _Driver(StreamPool(m, 1, warmup=True), audio, eg)
        r.open(j)
        while r.pushed[j] < n_hops:
            if r.pushed[j] == set_at:
                r.pool.set_egemaps([r.slot[j]], eg_new[None])
            r.push([j])
        return r.got[j]
    for j, want in ((2, fresh(2)), (1, fresh(1, set_at=t_set))):
        assert sorted(d.got[j]) == sorted(want) == list(range(n_hops))
        for h in want:
            assert torch.equal(d.got[j][h], want[h]), f"stream {j}, hop {h}"
    unchanged = fresh(1)
    mouth, expr = list(K.MOUTH_INDICES), list(K.EXPRESSION_INDICES)
    assert all(torch.equal(d.got[1][h][mouth], unchanged[h][mouth]) for h in range(n_hops))
    assert all(torch.equal(d.got[1][h][expr], unchanged[h][expr]) for h in range(t_set))
    assert not any(torch.equal(d.got[1][h][expr], unchanged[h][expr]) for h in range(t_set, n_hops))


@pytest.mark.parametrize("fps,per_push", [(30, 6), (60, 8)])
def test_launch_counts(fps, per_push):
    """6 kernels per call at 30 fps (8 at 60) whenever a stream is pushed -- every pushed stream emits -- for push on
    max_hops = 1 and max_hops = 4 pools and for bursts; one fewer without smoothing, none for an empty call."""
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, "bf16", smoothing=True)
    hop, W = HOP[fps], WIN[fps]
    x = torch.randn(8 * hop, device="cuda") * 0.1
    def push(pool, slots):
        _lib.reset_launch_count()
        emitted, _ = pool.push(slots, x[:len(slots) * hop].view(-1, hop))
        assert _lib.launch_count() == per_push and emitted.tolist() == slots

    for max_hops in (1, 4):
        pool = StreamPool(m, 3, max_hops=max_hops, warmup=True)
        a = pool.open(torch.zeros(1, 264, device="cuda"))[0]
        torch.cuda.synchronize()
        push(pool, [a])                            # hop 0 emits
        push(pool, [a])
        b, c = pool.open(torch.zeros(2, 264, device="cuda"))
        torch.cuda.synchronize()
        push(pool, [a, b])
        push(pool, [b])
        push(pool, [a, b, c])
        if max_hops > 1:
            _lib.reset_launch_count()
            slots, hops, _ = pool.push_hops([b, a], x[:7 * hop], [4, 3])
            assert _lib.launch_count() == per_push and slots.tolist() == [b] * 4 + [a] * 3
        m.use_temporal_smoothing = False
        _lib.reset_launch_count()
        assert pool.push([c], x[:hop].view(1, hop))[0].tolist() == [c] and _lib.launch_count() == per_push - 1
        m.use_temporal_smoothing = True
        _lib.reset_launch_count()
        assert pool.push([], x[:0].view(0, hop))[0].numel() == 0 and _lib.launch_count() == 0
    assert W > 8                                   # (every push above was in warm-up)
