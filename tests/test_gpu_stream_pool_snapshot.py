"""GPU tests (-m gpu) of StreamPool.snapshot / StreamPool.restore: streams that leave their pool with their whole state
and continue in another one -- of another capacity or max_hops, after a trip through host memory, on another GPU.  A
restored stream pushed the same hops as the original must give bit for bit the original's frames and hops; both must
equal a one-stream StreamingEngine fed the whole clip."""
import io

import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O

pytestmark = pytest.mark.gpu

HOP = {30: 533, 60: 266}
WIN = {30: 256, 60: 512}


def _model(fps, precision, smoothing=True, seed=1236):
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


def _solo(m, clip, eg, fps, egemaps_at=None):
    """Frames of a one-stream StreamingEngine fed `clip` hop by hop: {hop: (52,) frame}."""
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
    """Feeds stream j of `audio` (its own clip) to one pool and keeps every frame it emits by (stream, hop)."""

    def __init__(self, pool, audio, eg, fps):
        self.pool, self.audio, self.eg, self.hop, self.W = pool, audio, eg, HOP[fps], WIN[fps]
        self.first = 0 if pool.warmup else self.W - 1          # the hop of a stream's first frame
        self.slot, self.pushed, self.got = {}, {}, {}

    def open(self, j):
        self.adopt(j, self.pool.open(self.eg[j:j + 1])[0], 0)
        return self.slot[j]

    def adopt(self, j, slot, pushed):
        """stream j continues in `slot` (a restore) from its hop `pushed`"""
        self.slot[j], self.pushed[j], self.got[j] = slot, pushed, {}

    def _audio(self, plan):
        parts = [self.audio[j][self.pushed[j] * self.hop:(self.pushed[j] + c) * self.hop] for j, c in plan]
        return torch.cat(parts) if parts else torch.empty(0, device=self.audio.device)

    def _keep(self, plan, rows):
        want = [(self.slot[j], h) for j, c in plan for h in range(self.pushed[j], self.pushed[j] + c) if h >= self.first]
        assert [(s, h) for s, h, _ in rows] == want, "rows not those of the pushed hops"
        by_slot = {self.slot[j]: j for j, _ in plan}
        for s, h, f in rows:
            self.got[by_slot[s]][h] = f.clone()
        for j, c in plan:
            self.pushed[j] += c

    def push_hops(self, plan):
        if not plan:
            return
        slots, hops, frames = self.pool.push_hops([self.slot[j] for j, _ in plan], self._audio(plan), [c for _, c in plan])
        self._keep(plan, list(zip(slots.tolist(), hops.tolist(), frames)))

    def push(self, js):
        if not js:
            return
        plan = [(j, 1) for j in js]
        emitted, frames = self.pool.push([self.slot[j] for j in js], self._audio(plan).view(-1, self.hop))
        by_slot = {self.slot[j]: j for j in js}
        self._keep(plan, [(s, self.pushed[by_slot[s]], f) for s, f in zip(emitted.tolist(), frames)])

    def drive(self, rng, targets, max_hops):
        """Seeded bursts until stream j has pushed targets[j] hops."""
        while any(self.pushed[j] < t for j, t in targets.items()):
            plan = [(j, min(int(rng.integers(1, max_hops + 1)), t - self.pushed[j]))
                    for j, t in targets.items() if self.pushed[j] < t]
            rng.shuffle(plan)
            self.push_hops(plan)


def _continue(rng, drivers, targets, max_hops):
    """Pushes every driver the same seeded plans -- single-hop pushes and bursts of up to max_hops, mixed -- until
    stream j has pushed targets[j] hops in each."""
    d0 = drivers[0]
    while any(d0.pushed[j] < t for j, t in targets.items()):
        live = [j for j, t in targets.items() if d0.pushed[j] < t]
        if rng.random() < 0.4:
            for d in drivers:
                d.push(live)
        else:
            plan = [(j, min(int(rng.integers(1, max_hops + 1)), targets[j] - d0.pushed[j])) for j in live]
            rng.shuffle(plan)
            for d in drivers:
                d.push_hops(plan)


def _same(a, b, j, since):
    """stream j's frames in drivers a and b from hop `since` on: the same hops, torch.equal frames"""
    hops = sorted(h for h in a.got[j] if h >= since)
    assert hops == sorted(b.got[j]) and hops, f"stream {j}: hops {hops[:3]}.. vs {sorted(b.got[j])[:3]}.."
    for h in hops:
        assert torch.equal(a.got[j][h], b.got[j][h]), f"stream {j}, hop {h}"


def _ages(W):
    return [0, 1, W - 2, W - 1, W, W + 37, 3 * W + 5]


def _stale(pool, fps, hops, seed):
    """Fills every slot of `pool` with a loud stream that runs `hops` hops (its rings wrap), then closes them all."""
    audio, eg = _clips(seed, pool.capacity, hops, fps)
    d = _Driver(pool, 4.0 * audio, eg, fps)
    for j in range(pool.capacity):
        d.open(j)
    d.drive(np.random.default_rng(seed), {j: hops for j in range(pool.capacity)}, pool.max_hops)
    for j in range(pool.capacity):
        pool.close(d.slot[j])


@pytest.mark.parametrize("fps,precision,smoothing", [(30, "fp32", True), (30, "bf16", False), (60, "fp32", False),
                                                     (60, "bf16", True)])
def test_twin_streams(fps, precision, smoothing):
    """Seven streams of pool A at ages 0, 1, W - 2, W - 1, W, W + 37 and 3 W + 5 hops (rings wrapped) are snapshotted in
    one call and restored into pool B (another capacity and max_hops, slots that held loud streams for more than R
    hops).  Pushed the same hops from there -- pushes and bursts mixed -- every frame and hop of B equals A's, and both
    equal a solo StreamingEngine fed the whole clip."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, smoothing)
    W = WIN[fps]
    ages = _ages(W)
    end = 3 * W + 5 + 19
    audio, eg = _clips(7100 + fps, len(ages), end, fps)
    a = StreamPool(m, 8, max_hops=8)
    b = StreamPool(m, 9, max_hops=4)
    _stale(b, fps, b.ring_frames + 5, 7200 + fps)
    da, db = _Driver(a, audio, eg, fps), _Driver(b, audio, eg, fps)
    for j in range(len(ages)):
        da.open(j)
    da.drive(np.random.default_rng(fps), dict(enumerate(ages)), 8)
    order = [3, 0, 6, 1, 5, 2, 4]                                   # (not slot order)
    snap = a.snapshot([da.slot[j] for j in order])
    assert snap.hops.tolist() == [ages[j] for j in order]
    assert snap.records.shape == (len(ages), a.state_floats) and snap.records.device == a.dev
    if not smoothing:
        # without smoothing the records carry a zero smoothing row, and a restore leaves the slots' own rows alone
        o = (1 + a.n_edge) * (W - a.n_edge) * 81 + a.tail_len + 1
        assert not snap.records[:, o:o + 52].any()
        b.state.fill_(7.0)
    slots = b.restore(snap)
    assert slots == list(range(len(ages)))                          # the lowest free slots
    if not smoothing:
        assert (b.state == 7.0).all()
    for j, s in zip(order, slots):
        db.adopt(j, s, ages[j])
    _continue(np.random.default_rng(fps + 1), [da, db], {j: end for j in range(len(ages))}, 4)
    for j, age in enumerate(ages):
        _same(da, db, j, age)
        want = _solo(m, audio[j], eg[j], fps)
        got = {**{h: f for h, f in da.got[j].items() if h < age}, **db.got[j]}
        assert sorted(got) == sorted(want) == list(range(W - 1, end))
        for h in want:
            assert torch.equal(got[h], want[h]), f"stream {j}, hop {h}"


@pytest.mark.parametrize("fps,precision", [(30, "bf16"), (60, "fp32")])
def test_resize(fps, precision):
    """A pool of max_hops = 1 moves into a larger one of max_hops = 8 and is driven with bursts; that pool's streams
    move back into a pool of max_hops = 1 and are driven one hop per push.  Bursts end right at both snapshot points and
    start right after them.  Every frame bit for bit the solo engine's."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision)
    W = WIN[fps]
    ages = [W - 3, W + 2, 2 * W + 1]
    mid = [a + 21 for a in ages]
    end = [x + 11 for x in mid]
    audio, eg = _clips(7300 + fps, 3, max(end), fps)
    small = StreamPool(m, 3)
    big = StreamPool(m, 16, max_hops=8)
    small2 = StreamPool(m, 4)
    d1, d2, d3 = (_Driver(p, audio, eg, fps) for p in (small, big, small2))
    for j in range(3):
        d1.open(j)
    d1.drive(np.random.default_rng(0), dict(enumerate(ages)), 1)
    for j, s in enumerate(big.restore(small.snapshot([d1.slot[j] for j in range(3)]))):
        d2.adopt(j, s, ages[j])
    d2.push_hops([(j, 8) for j in range(3)])                         # a burst right after the snapshot point
    d2.drive(np.random.default_rng(1), dict(enumerate(mid)), 8)   # (ends with bursts up to the next snapshot point)
    snap = big.snapshot([d2.slot[j] for j in (2, 0, 1)])
    assert snap.hops.tolist() == [mid[2], mid[0], mid[1]]
    for j, s in zip((2, 0, 1), small2.restore(snap)):
        d3.adopt(j, s, mid[j])
    rng = np.random.default_rng(2)
    while any(d3.pushed[j] < end[j] for j in range(3)):
        d3.push([j for j in range(3) if d3.pushed[j] < end[j] and (rng.random() < 0.8 or d3.pushed[j] == mid[j])])
    for j in range(3):
        want = _solo(m, audio[j][:end[j] * HOP[fps]], eg[j], fps)
        got = {**{h: f for h, f in d1.got[j].items()}, **d2.got[j], **d3.got[j]}
        assert sorted(got) == sorted(want) == list(range(W - 1, end[j]))
        for h in want:
            assert torch.equal(got[h], want[h]), f"stream {j}, hop {h}"


@pytest.mark.parametrize("fps,precision", [(30, "fp32"), (60, "bf16")])
def test_warmup_pools(fps, precision):
    """Warm-up pools: streams snapshotted before, at and after hop W - 1 and restored into a warm-up pool of another
    max_hops give every frame of the original from there on, smoothing chain included (it runs from hop 0)."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, precision, smoothing=True)
    W = WIN[fps]
    ages = [0, 1, 5, W - 2, W - 1, W, W + 9]
    end = W + 25
    audio, eg = _clips(7400 + fps, len(ages), end, fps)
    a = StreamPool(m, 8, max_hops=4, warmup=True)
    b = StreamPool(m, 7, max_hops=1, warmup=True)
    _stale(b, fps, b.ring_frames + 3, 7500 + fps)
    da, db = _Driver(a, audio, eg, fps), _Driver(b, audio, eg, fps)
    for j in range(len(ages)):
        da.open(j)
    da.drive(np.random.default_rng(5), dict(enumerate(ages)), 4)
    for j, s in zip(range(len(ages)), b.restore(a.snapshot([da.slot[j] for j in range(len(ages))]))):
        db.adopt(j, s, ages[j])
    _continue(np.random.default_rng(6), [da, db], {j: end for j in range(len(ages))}, 1)
    for j, age in enumerate(ages):
        _same(da, db, j, age)
        assert sorted(h for h in da.got[j]) == list(range(end))
    # a snapshot of a warm-up pool does not go into a plain one, nor the other way round
    plain = StreamPool(m, 2)
    with pytest.raises(ValueError, match="warmup"):
        plain.restore(a.snapshot([da.slot[0]]))
    with pytest.raises(ValueError, match="warmup"):
        b.restore(plain.snapshot([]))


def test_snapshot_is_read_only():
    """A pool that takes snapshots mid-stream (of some streams, twice) gives exactly the frames of an identical pool
    that never takes one."""
    from koemorph_b200.streaming import StreamPool
    fps, W = 30, WIN[30]
    m = _model(fps, "bf16")
    audio, eg = _clips(7600, 4, W + 40, fps)
    a, c = StreamPool(m, 4, max_hops=3), StreamPool(m, 4, max_hops=3)
    da, dc = _Driver(a, audio, eg, fps), _Driver(c, audio, eg, fps)
    for j in range(4):
        da.open(j), dc.open(j)
    rng = np.random.default_rng(8)
    for target, snap in ((W - 1, [0, 2]), (W + 13, [3, 2, 1, 0]), (W + 40, None)):
        _continue(rng, [da, dc], {j: target for j in range(4)}, 3)
        if snap:
            a.snapshot([da.slot[j] for j in snap])
    for j in range(4):
        _same(da, dc, j, 0)


def test_expression_is_carried():
    """A restored stream's first frame needs no set_egemaps; a set_egemaps after the restore changes the restored
    stream only -- not its original, and not the other restored stream."""
    import koemorph_b200 as K
    from koemorph_b200.streaming import StreamPool
    fps, W = 30, WIN[30]
    m = _model(fps, "fp32")
    age, end = W + 4, W + 30
    audio, eg = _clips(7700, 2, end, fps)
    _, eg_new = O.make_inputs(7701, 1, HOP[fps], "speechlike")
    eg_new = torch.from_numpy(eg_new).cuda()
    a, b = StreamPool(m, 2), StreamPool(m, 2, max_hops=2)
    da, db = _Driver(a, audio, eg, fps), _Driver(b, audio, eg, fps)
    for j in range(2):
        da.open(j)
    da.drive(np.random.default_rng(9), {0: age, 1: age}, 1)
    for j, s in enumerate(b.restore(a.snapshot([da.slot[0], da.slot[1]]))):
        db.adopt(j, s, age)
    assert torch.equal(b.expr[:2], a.expr[[da.slot[0], da.slot[1]]])
    _continue(np.random.default_rng(10), [da, db], {0: age + 1, 1: age + 1}, 1)
    b.set_egemaps([db.slot[0]], eg_new)
    _continue(np.random.default_rng(11), [da, db], {0: end, 1: end}, 1)
    _same(da, db, 1, age)
    solo_a = _solo(m, audio[0], eg[0], fps)
    solo_b = _solo(m, audio[0], eg[0], fps, egemaps_at={age + 1: eg_new[0]})
    expr = list(K.EXPRESSION_INDICES)
    for h in range(W - 1, end):
        assert torch.equal(da.got[0][h], solo_a[h]), h
    for h in range(age, end):
        assert torch.equal(db.got[0][h], solo_b[h]), h
    assert torch.equal(db.got[0][age], da.got[0][age])
    assert not any(torch.equal(db.got[0][h][expr], da.got[0][h][expr]) for h in range(age + 1, end))


@pytest.mark.parametrize("fps", [30, 60])
def test_record_layout(fps):
    """Record row i of variant v is ring row (a + 1 - W + i) mod R of the plain / window-start rings for frames >= 0 and
    zero for frames < 0; then the maxima, the tail, the expression value, the smoothing row and zero padding.  A
    restored stream with hops > 0 keeps its tail through its next hop (its first hop in the new pool is not a first
    hop)."""
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, "bf16")
    W, hop = WIN[fps], HOP[fps]
    n_edge = -(-512 // hop)
    P, Vr = W - n_edge, 1 + n_edge
    ages = [0, 3, W - 2, W + 1, 2 * W + 7]
    audio, eg = _clips(7800 + fps, len(ages), max(ages) + 1, fps)
    a = StreamPool(m, len(ages), max_hops=5)
    d = _Driver(a, audio, eg, fps)
    for j in range(len(ages)):
        d.open(j)
    d.drive(np.random.default_rng(12), dict(enumerate(ages)), 5)
    slots = [d.slot[j] for j in range(len(ages))]
    snap = a.snapshot(slots)
    torch.cuda.synchronize()
    R = a.ring_frames
    rings = [(a.ring_f, a.fmax_f), (a.ring_r, a.fmax_r)] + ([(a.ring_r2, a.fmax_r2)] if n_edge == 2 else [])
    assert len(rings) == Vr
    for j, (s, age) in enumerate(zip(slots, ages)):
        rec = snap.records[j]
        rows = rec[:Vr * P * 80].view(Vr, P, 80)
        maxima = rec[Vr * P * 80:Vr * P * 81].view(Vr, P)
        o = Vr * P * 81
        frames = torch.arange(P) + age + 1 - W
        ok = frames >= 0
        ring_rows = (frames % R).cuda()
        for v, (ring, fmax) in enumerate(rings):
            assert torch.equal(rows[v][ok.cuda()], ring[s][ring_rows][ok.cuda()]), (age, v)
            assert torch.equal(maxima[v][ok.cuda()], fmax[s][ring_rows][ok.cuda()]), (age, v)
            assert not rows[v][~ok.cuda()].any() and not maxima[v][~ok.cuda()].any()
        assert torch.equal(rec[o:o + a.tail_len], a.tail[s])
        assert torch.equal(rec[o + a.tail_len], a.expr[s])
        assert torch.equal(rec[o + a.tail_len + 1:o + a.tail_len + 53], a.state[s])
        assert not rec[o + a.tail_len + 53:].any() and rec.numel() == a.state_floats
    # restored: the tail goes back in, and the next hop extends it instead of starting from zeros
    b = StreamPool(m, len(ages) + 2, max_hops=2)
    db = _Driver(b, audio, eg, fps)
    for j, s in enumerate(b.restore(snap)):
        db.adopt(j, s, ages[j])
    torch.cuda.synchronize()
    for j in range(len(ages)):
        assert torch.equal(b.tail[db.slot[j]], a.tail[d.slot[j]])
    plan = [(j, 1) for j in range(len(ages))]
    d.push_hops(plan)
    db.push_hops(plan)
    torch.cuda.synchronize()
    for j, age in enumerate(ages):
        if age > 0:
            assert torch.equal(b.tail[db.slot[j]], a.tail[d.slot[j]]), age
            assert b.tail[db.slot[j]][:-hop].any()


def test_host_round_trip():
    """The snapshot through host memory and torch.save / torch.load restores bit for bit."""
    from koemorph_b200.streaming import StreamPool, StreamSnapshot
    fps, W = 60, WIN[60]
    m = _model(fps, "bf16")
    ages = [W - 4, W + 3]
    end = W + 20
    audio, eg = _clips(7900, 2, end, fps)
    a, b = StreamPool(m, 2, max_hops=2), StreamPool(m, 3)
    da, db = _Driver(a, audio, eg, fps), _Driver(b, audio, eg, fps)
    for j in range(2):
        da.open(j)
    da.drive(np.random.default_rng(13), dict(enumerate(ages)), 2)
    host = a.snapshot([da.slot[0], da.slot[1]]).to("cpu")
    assert host.records.device.type == "cpu"
    buf = io.BytesIO()
    torch.save(host, buf)
    buf.seek(0)
    loaded = torch.load(buf)
    assert isinstance(loaded, StreamSnapshot)
    for j, s in enumerate(b.restore(loaded.to("cuda"))):
        db.adopt(j, s, ages[j])
    _continue(np.random.default_rng(14), [da, db], {0: end, 1: end}, 1)
    for j in range(2):
        _same(da, db, j, ages[j])


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two visible GPUs (restore on cuda:1)")
def test_cross_device():
    """Streams of a pool on cuda:0 continue in a pool on cuda:1, bit for bit."""
    from koemorph_b200.streaming import StreamPool
    fps, W = 30, WIN[30]
    m0 = _model(fps, "bf16")
    m1 = _model(fps, "bf16")
    m1.to("cuda:1")
    ages = [W - 2, W + 30]
    end = W + 50
    audio, eg = _clips(8000, 2, end, fps)
    a = StreamPool(m0, 2, max_hops=4)
    b = StreamPool(m1, 4)
    da = _Driver(a, audio, eg, fps)
    db = _Driver(b, audio.to("cuda:1"), eg.to("cuda:1"), fps)
    for j in range(2):
        da.open(j)
    da.drive(np.random.default_rng(15), dict(enumerate(ages)), 4)
    snap = a.snapshot([da.slot[0], da.slot[1]])
    moved = snap.to("cuda:1")
    torch.cuda.synchronize("cuda:0")
    torch.cuda.synchronize("cuda:1")
    with torch.cuda.device(1):
        slots = b.restore(moved)
    for j, s in enumerate(slots):
        db.adopt(j, s, ages[j])
    while any(da.pushed[j] < end for j in range(2)):
        js = [j for j in range(2) if da.pushed[j] < end]
        da.push(js)
        with torch.cuda.device(1):
            db.push(js)
    for j in range(2):
        hops = sorted(h for h in da.got[j] if h >= ages[j])
        assert hops == sorted(db.got[j])
        for h in hops:
            assert torch.equal(da.got[j][h], db.got[j][h].to("cuda:0")), (j, h)


@pytest.mark.parametrize("fps", [30, 60])
def test_launch_counts_and_misuse(fps):
    """Snapshot and restore queue one kernel each; misuse raises ValueError, queues none and moves no clock."""
    from koemorph_b200 import _lib
    from koemorph_b200.streaming import StreamPool
    m = _model(fps, "bf16")
    W = WIN[fps]
    audio, eg = _clips(8100 + fps, 3, W + 8, fps)
    a, b = StreamPool(m, 4, max_hops=4), StreamPool(m, 2, max_hops=4)
    d = _Driver(a, audio, eg, fps)
    for j in range(3):
        d.open(j)
    d.drive(np.random.default_rng(17), {0: W - 1, 1: 2, 2: W + 3}, 4)
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    snap = a.snapshot([d.slot[2], d.slot[0], d.slot[1]])
    assert _lib.launch_count() == 1
    _lib.reset_launch_count()
    two = type(snap)(snap.hop, snap.window_frames, snap.half_fft, snap.warmup, snap.hops[:2].clone(),
                     snap.records[:2].clone())
    torch.cuda.synchronize()
    _lib.reset_launch_count()
    slots = b.restore(two)
    assert _lib.launch_count() == 1 and slots == [0, 1]
    _lib.reset_launch_count()
    closed = a.open(eg[:1])[0]
    a.close(closed)
    _lib.reset_launch_count()
    for bad in ([closed], [d.slot[0], d.slot[0]], [4], [-1]):
        with pytest.raises(ValueError):
            a.snapshot(bad)
    with pytest.raises(ValueError, match="slots free"):
        b.restore(two)                                              # b is full
    c = StreamPool(m, 4)
    with pytest.raises(ValueError):
        c.restore(type(snap)(snap.hop, snap.window_frames, snap.half_fft, snap.warmup, snap.hops, snap.records.double()))
    neg = snap.hops.clone()
    neg[1] = -1
    with pytest.raises(ValueError):
        c.restore(type(snap)(snap.hop, snap.window_frames, snap.half_fft, snap.warmup, neg, snap.records))
    assert _lib.launch_count() == 0
    assert c.restore(type(snap)(snap.hop, snap.window_frames, snap.half_fft, snap.warmup, snap.hops[:0],
                                snap.records[:0])) == [] and _lib.launch_count() == 0
    # the refused calls moved no clock: b's streams continue at hops W + 3 and W - 1, c's slots are all free
    dd = _Driver(b, audio, eg, fps)
    dd.adopt(2, slots[0], W + 3)
    dd.adopt(0, slots[1], W - 1)
    dd.push_hops([(2, 2), (0, 1)])
    assert sorted(dd.got[2]) == [W + 3, W + 4] and sorted(dd.got[0]) == [W - 1]
    assert c.restore(snap) == [0, 1, 2]
