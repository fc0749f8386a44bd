"""Hop-aligned streaming inference for many concurrent streams (BASELINE.json configs[3]).

The reference's real-time loop (``scripts/rt.py:465-519`` + ``SimplifiedDualStreamModel.process_audio_frame_realtime``,
``src/model/simplified_dual_stream_model.py:452-500``) recomputes the whole 8.5 s mel for every 33 ms hop.  A window
of ``SequentialDualStreamModel`` that starts at hop i only differs from the previous one by (SURVEY.md section 8,
note E; 30 fps geometry, hop 533 >= n_fft / 2):

* one new plain frame           F[n]    centred on sample n*hop,
* one new "window starts here"  R[n]    the same frame with everything before n*hop zeroed (frame 0 of window n),
* one "window ends here" frame  L[n+1]  centred on (n+1)*hop with everything from (n+1)*hop on zeroed,

so a step costs 3 FFTs per stream, not 257.  At 60 fps (hop 266 < n_fft / 2) two frames per window side are edge
frames: the newest complete plain frame is F[n-1], and a step adds its two window-start variants R0[n-1] (nothing before
(n-1)*hop) and R1[n-1] (nothing before (n-2)*hop) plus the last two frames of the window that ends now, L1[n] and
L0[n+1] -- 5 FFTs per hop against 513.  F and R rows go into per-stream rings of ``W`` mel rows in HBM
(164 KB per stream), the only audio kept is the last ``n_fft/2 + hop`` samples, and the core kernel addresses the
rings directly (``koe_dual_stream_ring``).  After the 256th hop every step emits the frame that
``SequentialDualStreamModel.forward`` would produce for the window ending at the newest sample, EMA included.
All streams of a StreamingEngine advance in lockstep (one hop per step each); in a StreamPool every stream opens,
closes and advances on its own clock, by one hop per push or by several in one push_hops, and a warm-up StreamPool
emits from each stream's first hop on, computed on the audio heard so far.
"""
from __future__ import annotations

import ctypes as C
import operator
from typing import Optional

import torch

from . import _lib


class StreamingEngine:
    def __init__(self, model, n_streams: int):
        self.model = model
        self.S = int(n_streams)
        self.dev = next(model.parameters()).device
        if self.dev.type != "cuda":
            raise RuntimeError("StreamingEngine needs the model on a CUDA device")
        self._dev_index = self.dev.index if self.dev.index is not None else torch.cuda.current_device()
        self.hop = model.hop_length
        self.W = model.mel_sequence_length
        self.half = model.n_fft // 2
        # frames within n_fft/2 of a window edge see zeros beyond it: one per side at 30 fps (hop 533 >= 512), two at 60 fps
        # (hop 266): frames 0, 1 and W-1, W of every window are edge variants (SURVEY.md section 8 note E: 5 FFTs per hop)
        self.n_edge = -(-self.half // self.hop)
        if self.n_edge > _lib.MAX_EDGE:
            raise NotImplementedError(f"hop {self.hop} needs {self.n_edge} edge frames per window side (max {_lib.MAX_EDGE})")
        self.lag = self.n_edge - 1                         # the newest complete plain frame is global frame n - lag
        self.tail_len = self.half + self.n_edge * self.hop  # samples [ (n+1)hop - tail_len, (n+1)hop )
        f32 = dict(dtype=torch.float32, device=self.dev)
        self._tails = [torch.zeros(self.S, self.tail_len, **f32) for _ in range(2)]   # ping-pong (koe_stream_push)
        self.ring_f = torch.zeros(self.S, self.W, 80, **f32)
        self.ring_r = torch.zeros(self.S, self.W, 80, **f32)
        self.fmax_f = torch.zeros(self.S, self.W, **f32)
        self.fmax_r = torch.zeros(self.S, self.W, **f32)
        self.row_l = torch.zeros(self.S, 1, 80, **f32)
        self.fmax_l = torch.zeros(self.S, 1, **f32)
        if self.n_edge == 2:
            self.ring_r2 = torch.zeros(self.S, self.W, 80, **f32)
            self.fmax_r2 = torch.zeros(self.S, self.W, **f32)
            self.row_l2 = torch.zeros(self.S, 1, 80, **f32)
            self.fmax_l2 = torch.zeros(self.S, 1, **f32)
        else:
            self.ring_r2 = self.fmax_r2 = self.row_l2 = self.fmax_l2 = None
        self.expr = torch.zeros(self.S, **f32)
        self.state = torch.zeros(self.S, 52, **f32)
        self.out = torch.zeros(self.S, 52, **f32)
        self.n = 0                                          # hops pushed so far
        self.emitted = 0
        self._fe = model._frontend(self.dev)
        self._alpha, self._alpha_key = 0.0, None
        self._args, self._args_key, self._w_tensors = None, None, []
        self.native = True                                  # one koe_stream_push per step (False: call by call from Python)

    def reset(self):
        for t in (*self._tails, self.ring_f, self.ring_r, self.fmax_f, self.fmax_r, self.state, self.ring_r2, self.fmax_r2):
            if t is not None:
                t.zero_()
        self.n = 0
        self.emitted = 0
        self._args = None                                   # the next step walks the module's weights again

    @torch.no_grad()
    def set_egemaps(self, egemaps: torch.Tensor) -> None:
        """(S, 264) eGeMAPS windows; the reference refreshes them every 300 ms, not every frame
        (src/features/opensmile_extractor.py:168)."""
        eg = self.model._check_egemaps(egemaps, self.S, self.dev)
        self._args = None                                   # (a natural point to pick up replaced weights, too)
        w = self.model.dual_stream_attention.kernel_weights(self.model._compression)
        with torch.cuda.device(self.dev):
            _lib.check(_lib.load().koe_emotion_stream(C.byref(w.struct), eg.data_ptr(), self.S, self.expr.data_ptr(),
                                                      _lib.stream_ptr(self.dev)), "koe_emotion_stream")

    @torch.no_grad()
    def step(self, hop_audio: torch.Tensor) -> Optional[torch.Tensor]:
        """hop_audio (S, hop) float32 CUDA: the next hop of every stream.  Returns (S, 52) smoothed blendshapes once
        the 8.5 s context is full (from the W-th hop on), else None.  The returned tensor is reused by the next step."""
        x = _lib.require_cuda(hop_audio, "hop_audio")
        if x.shape != (self.S, self.hop):
            raise ValueError(f"hop_audio must be ({self.S}, {self.hop}), got {tuple(x.shape)}")
        if not self.native:
            return self._step_python(x)
        # the whole step -- tail shift, the three new frames F[n], R[n], L[n+1] into the rings, the window that ends at
        # the newest sample through the core, the smoothing -- is one native call that queues five kernels
        # (host time before the first launch is latency nobody hides: the argument block is built once, a step only
        # updates what changes)
        m = self.model
        a = self._args
        # the folded weights are re-validated against the module's parameters by their in-place version counters every
        # step, and by the full walk over the module (replaced tensors: .to(), new Parameters) every 256th
        key = (m.precision, m.use_temporal_smoothing, tuple(t._version for t in self._w_tensors))
        if a is None or self._args_key != key or (self.n & 255) == 0:
            a = self._args = self._build_args()
            self._args_key = (m.precision, m.use_temporal_smoothing, tuple(t._version for t in self._w_tensors))
        if m.use_temporal_smoothing:
            # sigmoid(smoothing_alpha) is read back once per parameter version, not once per hop (a device sync)
            ver = (m.smoothing_alpha.data_ptr(), m.smoothing_alpha._version)
            if self._alpha_key != ver:
                self._alpha = float(torch.sigmoid(m.smoothing_alpha.detach().float()))
                self._alpha_key = ver
            a.alpha = self._alpha
        a.hop_audio = x.data_ptr()
        a.has_state = 1 if self.emitted > 0 else 0
        a.step = self.n
        emitted = self._emitted_flag
        if torch.cuda.current_device() == self._dev_index:
            rc = self._push(self._args_ref, self._emitted_ref, torch.cuda.current_stream(self.dev).cuda_stream)
        else:
            with torch.cuda.device(self.dev):
                rc = self._push(self._args_ref, self._emitted_ref, torch.cuda.current_stream(self.dev).cuda_stream)
        _lib.check(rc, "koe_stream_push")
        self.n += 1
        if not emitted.value:
            return None
        self.emitted += 1
        return self.out

    def _build_args(self):
        m = self.model
        self._weights = m.dual_stream_attention.kernel_weights(m._compression)   # (kept alive: the block points into it)
        att = m.dual_stream_attention
        self._w_tensors = [t for _, t in att.named_parameters()] + [t for _, t in att.named_buffers()] + \
            ([] if m._compression is None else [m._compression["weight"], m._compression["bias"]])
        a = _lib.StreamArgs()
        a.frontend, a.weights = self._fe._h, C.cast(C.pointer(self._weights.struct), C.c_void_p)
        a.n_streams, a.hop, a.window_frames, a.half_fft = self.S, self.hop, self.W, self.half
        a.tail[0], a.tail[1] = self._tails[0].data_ptr(), self._tails[1].data_ptr()
        a.ring_f, a.fmax_f = self.ring_f.data_ptr(), self.fmax_f.data_ptr()
        a.ring_r, a.fmax_r = self.ring_r.data_ptr(), self.fmax_r.data_ptr()
        a.row_l, a.fmax_l = self.row_l.data_ptr(), self.fmax_l.data_ptr()
        if self.n_edge == 2:
            a.ring_r2, a.fmax_r2 = self.ring_r2.data_ptr(), self.fmax_r2.data_ptr()
            a.row_l2, a.fmax_l2 = self.row_l2.data_ptr(), self.fmax_l2.data_ptr()
        a.expr_sigmoid, a.out = self.expr.data_ptr(), self.out.data_ptr()
        a.ema_state, a.alpha = (self.state.data_ptr(), self._alpha) if m.use_temporal_smoothing else (None, 1.0)
        a.precision = _lib.PRECISIONS[m.precision]
        self._args_ref = C.byref(a)
        self._emitted_flag = C.c_int(0)
        self._emitted_ref = C.byref(self._emitted_flag)
        self._push = _lib.load().koe_stream_push
        return a

    def _step_python(self, x: torch.Tensor) -> Optional[torch.Tensor]:
        """The same step issued call by call from Python (``native = False``): the readable statement of what
        koe_stream_push does, kept as its cross-check (tests/test_gpu_streaming.py)."""
        n, hop, W, half = self.n, self.hop, self.W, self.half
        # slide the audio tail: drop the oldest hop, append the new one
        tail = self._tails[(n + 1) & 1]
        torch.cat([self._tails[n & 1][:, hop:], x], dim=1, out=tail)
        slot = (n - self.lag) % W                           # ring slot of the newest complete frame g = n - lag
        fe = self._fe
        # frame g and the frame one hop later are consecutive frames of the tail: one launch, g into the ring slot, the
        # pair's second frame into its own row -- at 30 fps that is L (centred on the tail's end, beyond which the clip
        # reads as zeros), at 60 fps the last-but-one frame of the window that ends now
        second = (self.row_l, self.fmax_l) if self.n_edge == 1 else (self.row_l2, self.fmax_l2)
        fe.power(tail, hop, 2, sample_offset=half, out=(self.ring_f, self.fmax_f), out_row=slot, out_b=second)
        if self.n_edge == 2:                                # the frame centred on the tail's end: the window's last frame
            fe.power(tail, hop, 1, frame_offset=2, sample_offset=half, out=(self.row_l, self.fmax_l))
        # window-start variants of frame g: nothing before its centre; at 60 fps also nothing before frame g-1's centre
        fe.power(tail, hop, 1, sample_offset=half, lo_rel=0, out=(self.ring_r, self.fmax_r), out_row=slot)
        if self.n_edge == 2:
            fe.power(tail, hop, 1, sample_offset=half, lo_rel=-1, out=(self.ring_r2, self.fmax_r2), out_row=slot)
        self.n += 1
        if self.n < W:
            return None
        base = self.n - W                                    # first frame of the window that ends now
        m = self.model
        w = m.dual_stream_attention.kernel_weights(m._compression)
        lib = _lib.load()
        with torch.cuda.device(self.dev):
            st = _lib.stream_ptr(self.dev)
            bufs = [self.ring_f, self.ring_r, self.row_l] + ([self.ring_r2, self.row_l2] if self.n_edge == 2 else [])
            fmx = [self.fmax_f, self.fmax_r, self.fmax_l] + ([self.fmax_r2, self.fmax_l2] if self.n_edge == 2 else [])
            n_buf = 1 + 2 * _lib.MAX_EDGE
            pw = (C.c_void_p * n_buf)(*[t.data_ptr() for t in bufs] + [None] * (n_buf - len(bufs)))
            fm = (C.c_void_p * n_buf)(*[t.data_ptr() for t in fmx] + [None] * (n_buf - len(fmx)))
            _lib.check(lib.koe_dual_stream_ring_edges(
                C.byref(w.struct), pw, fm, self.n_edge, self.S, W, base % W, W + 1, self.expr.data_ptr(),
                self.out.data_ptr(), None, None, _lib.PRECISIONS[m.precision], st), "koe_dual_stream_ring_edges")
            if m.use_temporal_smoothing:
                # sigmoid(smoothing_alpha) is read back once per parameter version, not once per hop (a device sync)
                ver = (m.smoothing_alpha.data_ptr(), m.smoothing_alpha._version)
                if self._alpha_key != ver:
                    self._alpha = float(torch.sigmoid(m.smoothing_alpha.detach().float()))
                    self._alpha_key = ver
                alpha = self._alpha
                _lib.check(lib.koe_ema_scan(self.out.data_ptr(), self.S, 1, alpha, self.state.data_ptr(),
                                            1 if self.emitted > 0 else 0, st), "koe_ema_scan")
        self.emitted += 1
        return self.out


class StreamSnapshot:
    """The state of k streams of a :class:`StreamPool` (:meth:`StreamPool.snapshot`), to continue them in another pool
    (:meth:`StreamPool.restore`): a pool of another capacity or ``max_hops``, on another GPU, or in a later process.

    * ``hop``, ``window_frames``, ``half_fft``, ``warmup``: the geometry of the pool it was taken from; a pool restores
      only a snapshot of its own geometry and warm-up flag;
    * ``hops``: CPU int64 ``[k]``, each stream's hops since it was opened;
    * ``records``: float32 ``[k][state_floats]``, one record per stream (layout in ``koe_stream_pool_snapshot``,
      include/koemorph_b200.h), on the source pool's device until moved with :meth:`to`.

    Tensors and ints only: ``torch.save`` / ``torch.load`` keep it as it is."""

    def __init__(self, hop: int, window_frames: int, half_fft: int, warmup: bool, hops: torch.Tensor,
                 records: torch.Tensor):
        self.hop, self.window_frames, self.half_fft, self.warmup = int(hop), int(window_frames), int(half_fft), bool(warmup)
        self.hops, self.records = hops, records

    def __len__(self) -> int:
        return int(self.hops.numel())

    def to(self, device) -> "StreamSnapshot":
        """A copy with the records on `device` (another GPU, or "cpu" to keep them in host memory)."""
        return StreamSnapshot(self.hop, self.window_frames, self.half_fft, self.warmup, self.hops.clone(),
                              self.records.to(device, copy=True))


# Intended, process-wide: importing the package adds StreamSnapshot to torch's weights-only allowlist, so that
# torch.load(path) with its default weights_only=True loads a saved snapshot.  The class holds tensors and ints only, so
# the allowlist admits nothing that could run code on load.
torch.serialization.add_safe_globals([StreamSnapshot])


class StreamPool:
    """Up to ``capacity`` concurrent streams that open, close and advance on their own clocks (``koe_stream_pool_*`` in
    include/koemorph_b200.h): a real-time service whose users connect and leave at any time and whose packets arrive
    late.  Every stream of the pool computes bit for bit what a one-stream :class:`StreamingEngine` computes when fed
    the same hops from the moment the stream was opened, whatever the other streams do and whatever its slot held
    before: it emits from its own W-th hop on (256 at 30 fps, 512 at 60 fps), its first frame passes the smoothing
    unchanged, and a reused slot carries nothing over.  The clocks live in the native pool object; this class owns the
    device buffers and checks what it hands over.

    ``max_hops`` > 1 lets :meth:`push_hops` advance a stream by up to that many hops in one call (late packets after a
    jitter buffer drains, chunked audio, a backlog): the rings then hold ``W + max_hops - 1`` rows, and the per-call
    buffers are sized for ``capacity * max_hops`` hops.

    ``warmup=True`` makes every pushed hop of every stream emit a frame from the stream's hop 0 on, instead of after
    8.5 s (``KOE_POOL_WARMUP``):

    * at hops h >= W - 1 the unsmoothed frame is bit for bit the one a pool without warm-up gives;
    * at hops h < W - 1 it is :meth:`SimplifiedDualStreamModel.forward` (smoothing off) on the audio heard so far, the
      stream's first ``(h + 1) * hop`` samples (up to the frontend's rounding): ``h + 2`` frames, the long-term part
      those frames zero-padded, the short-term detail their last three;
    * the temporal smoothing runs over every frame since the stream opened: its hop-0 frame passes unchanged and each
      later frame is smoothed onto the one before, so with smoothing on the frames from hop W - 1 on are the smoothing
      of this pool's own frames and differ from those of a pool without warm-up.

    :meth:`push` on a warm-up pool runs the burst path with counts of 1, whatever ``max_hops`` is.

    :meth:`snapshot` and :meth:`restore` move streams with their whole state (audio tail, mel rings, expression input,
    smoothing state) into another pool: one of another capacity or ``max_hops``, on another GPU, or in a later process."""

    def __init__(self, model, capacity: int, max_hops: int = 1, warmup: bool = False):
        self.model = model
        self.capacity = int(capacity)
        if self.capacity < 1:
            raise ValueError(f"capacity must be >= 1, got {capacity}")
        try:
            self.max_hops = operator.index(max_hops)
        except TypeError:
            raise ValueError(f"max_hops must be an integer, got {type(max_hops).__name__}") from None
        if isinstance(max_hops, bool) or self.max_hops < 1:
            raise ValueError(f"max_hops must be an integer >= 1, got {max_hops!r}")
        if not isinstance(warmup, bool):
            raise ValueError(f"warmup must be a bool, got {type(warmup).__name__}")
        self.warmup = warmup
        self.dev = next(model.parameters()).device
        if self.dev.type != "cuda":
            raise RuntimeError("StreamPool needs the model on a CUDA device")
        self._dev_index = self.dev.index if self.dev.index is not None else torch.cuda.current_device()
        self.hop = model.hop_length
        self.W = model.mel_sequence_length
        self.half = model.n_fft // 2
        self.n_edge = -(-self.half // self.hop)            # edge frames per window side (StreamingEngine)
        if self.n_edge > _lib.MAX_EDGE:
            raise NotImplementedError(f"hop {self.hop} needs {self.n_edge} edge frames per window side (max {_lib.MAX_EDGE})")
        self.tail_len = self.half + self.n_edge * self.hop
        cap, V = self.capacity, 1 + 2 * self.n_edge
        hops = cap * self.max_hops                          # hops one call may push
        self.ring_frames = R = self.W + self.max_hops - 1
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.tail = torch.zeros(cap, self.tail_len, **f32)
        self.tail_compact = torch.empty(hops, self.tail_len, **f32)
        self.stage = torch.empty(hops, V, 80, **f32)
        self.stage_max = torch.empty(hops, V, **f32)
        self.ring_f = torch.zeros(cap, R, 80, **f32)
        self.ring_r = torch.zeros(cap, R, 80, **f32)
        self.fmax_f = torch.zeros(cap, R, **f32)
        self.fmax_r = torch.zeros(cap, R, **f32)
        self.row_l = torch.zeros(cap, 80, **f32)
        self.fmax_l = torch.zeros(cap, **f32)
        if self.n_edge == 2:
            self.ring_r2 = torch.zeros(cap, R, 80, **f32)
            self.fmax_r2 = torch.zeros(cap, R, **f32)
            self.row_l2 = torch.zeros(cap, 80, **f32)
            self.fmax_l2 = torch.zeros(cap, **f32)
        else:
            self.ring_r2 = self.fmax_r2 = self.row_l2 = self.fmax_l2 = None
        self.expr = torch.zeros(cap, **f32)
        self.expr_compact = torch.empty(cap, **f32)
        self.state = torch.zeros(cap, 52, **f32)
        self.out = torch.zeros(hops, 52, **f32)
        self.tables = torch.empty((7 if warmup else 6) * hops, dtype=torch.int32, device=self.dev)
        self._emitted = torch.empty(hops, dtype=torch.int32)     # host: the slots of the last push's frames
        self._emitted_hop = torch.empty(hops, dtype=torch.int64)  # host: the hop of each (push_hops)
        self._n_emitted = C.c_int(0)
        self._n_emitted_ref = C.byref(self._n_emitted)
        self._lib = _lib.load()
        h = C.c_void_p()
        flags = _lib.POOL_WARMUP if warmup else 0
        self._check(self._lib.koe_stream_pool_create_ex2(cap, self.hop, self.W, self.half, self.max_hops, flags,
                                                         C.byref(h)), "koe_stream_pool_create_ex2")
        self._h = h
        self.state_floats = self._lib.koe_stream_pool_state_floats(h)   # floats per StreamSnapshot record
        if self.state_floats < 0:
            self._check(self.state_floats, "koe_stream_pool_state_floats")
        self._fe = model._frontend(self.dev)
        self._alpha, self._alpha_key = 0.0, None
        self._args, self._args_key, self._w_tensors = None, None, []
        self.pushes = 0

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.koe_stream_pool_destroy(h)
            self._h = None

    # ---- public API -------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def open(self, egemaps: torch.Tensor) -> list:
        """Opens k streams for egemaps (k, 264) (or (k, 3, 88)); returns their slots.  Their clocks start at zero."""
        eg = self._egemaps(egemaps)
        k = eg.shape[0]
        slots = torch.empty(k, dtype=torch.int32)
        self._check(self._lib.koe_stream_pool_open(self._h, k, slots.data_ptr()), "koe_stream_pool_open")
        try:
            self._set_egemaps(slots, eg)
        except BaseException:
            for s in slots.tolist():
                self._lib.koe_stream_pool_close(self._h, s)
            raise
        return slots.tolist()

    def close(self, slot: int) -> None:
        """Frees the slot of an open stream; the next stream opened there starts from silence."""
        slot = int(slot)
        if not 0 <= slot < self.capacity:
            raise ValueError(f"slot {slot} out of range [0, {self.capacity})")
        self._check(self._lib.koe_stream_pool_close(self._h, slot), "koe_stream_pool_close")

    @torch.no_grad()
    def set_egemaps(self, slots, egemaps: torch.Tensor) -> None:
        """Refreshes the expression input of the listed open streams only: egemaps row i belongs to slots[i]."""
        s = self._slots(slots)
        eg = self._egemaps(egemaps)
        if eg.shape[0] != s.numel():
            raise ValueError(f"egemaps has {eg.shape[0]} rows for {s.numel()} slots")
        self._set_egemaps(s, eg)

    @torch.no_grad()
    def push(self, slots, hop_audio: torch.Tensor):
        """Advances exactly the listed open streams by one hop each: hop_audio (n, hop) float32 on the model's device,
        row i the next hop of slots[i].  Returns (emitted_slots, frames): a CPU int64 tensor of the streams that emitted
        a frame in this call, in call order, and their (k, 52) smoothed frames -- a view reused by the next call.  A
        stream emits from its hop W - 1 on; on a warm-up pool every listed stream emits, from its hop 0 on."""
        s = self._slots(slots)
        n = s.numel()
        if not isinstance(hop_audio, torch.Tensor):
            raise ValueError(f"hop_audio must be a torch.Tensor, got {type(hop_audio).__name__}")
        if hop_audio.device != self.dev or hop_audio.dtype != torch.float32:
            raise ValueError(f"hop_audio must be float32 on {self.dev}, got {hop_audio.dtype} on {hop_audio.device}")
        if tuple(hop_audio.shape) != (n, self.hop):
            raise ValueError(f"hop_audio must be ({n}, {self.hop}) for {n} slots, got {tuple(hop_audio.shape)}")
        x = hop_audio.contiguous()
        a = self._current_args()
        a.hop_audio = x.data_ptr()
        self._call(self._lib.koe_stream_pool_push, self._h, self._args_ref, s.data_ptr(), n, self._emitted.data_ptr(),
                   self._n_emitted_ref, what="koe_stream_pool_push")
        self.pushes += 1
        k = self._n_emitted.value
        return self._emitted[:k].to(torch.int64), self.out[:k]

    @torch.no_grad()
    def push_hops(self, slots, audio: torch.Tensor, counts):
        """Advances each listed open stream by several hops in one call: slots[i] by counts[i] hops, 1 <= counts[i] <=
        max_hops (host integers).  audio: float32 on the model's device, the sum(counts) hops back to back, stream by
        stream in call order -- a 1-D tensor of sum(counts) * hop samples or an (sum(counts), hop) tensor.  Every frame
        is bit for bit what one :meth:`push` per hop gives.  Returns (slots, hops, frames): two CPU int64 tensors and a
        (k, 52) view reused by the next call; row r is the frame of stream slots[r] that completes at its hop hops[r]
        (counted from 0 since the stream was opened; its first frame comes at hop W - 1, or at hop 0 on a warm-up pool,
        where every hop emits).  Rows are grouped by stream in call order, hops ascending.  All frames of the call use each stream's expression input as it is now."""
        s = self._slots(slots)
        n = s.numel()
        c = counts if isinstance(counts, torch.Tensor) else torch.as_tensor(counts, dtype=torch.int64)
        if c.device.type != "cpu":
            raise ValueError("counts must be host (CPU) integers")
        if c.dim() != 1 or c.is_floating_point() or c.is_complex() or c.dtype == torch.bool:
            raise ValueError(f"counts must be a 1-D sequence of integers, got {c.dtype} of shape {tuple(c.shape)}")
        if c.numel() != n:
            raise ValueError(f"{c.numel()} counts for {n} slots")
        if n and (int(c.min()) < 1 or int(c.max()) > self.max_hops):
            raise ValueError(f"counts must lie in [1, {self.max_hops}] (max_hops)")
        c = c.to(torch.int32).contiguous()
        total = int(c.sum()) if n else 0
        if not isinstance(audio, torch.Tensor):
            raise ValueError(f"audio must be a torch.Tensor, got {type(audio).__name__}")
        if audio.device != self.dev or audio.dtype != torch.float32:
            raise ValueError(f"audio must be float32 on {self.dev}, got {audio.dtype} on {audio.device}")
        if tuple(audio.shape) not in ((total * self.hop,), (total, self.hop)):
            raise ValueError(f"audio must hold sum(counts) = {total} hops of {self.hop} samples: ({total * self.hop},) or "
                             f"({total}, {self.hop}), got {tuple(audio.shape)}")
        x = audio.contiguous()
        a = self._current_args()
        a.hop_audio = x.data_ptr()
        self._call(self._lib.koe_stream_pool_push_hops, self._h, self._args_ref, s.data_ptr(), c.data_ptr(), n,
                   self._emitted.data_ptr(), self._emitted_hop.data_ptr(), self._n_emitted_ref,
                   what="koe_stream_pool_push_hops")
        self.pushes += 1
        k = self._n_emitted.value
        return self._emitted[:k].to(torch.int64), self._emitted_hop[:k].clone(), self.out[:k]

    @torch.no_grad()
    def snapshot(self, slots) -> StreamSnapshot:
        """The state of the listed open streams after every call queued so far on the current stream (where the
        snapshot is queued, as :meth:`push`).  The streams stay open and unchanged.  Restored into a pool of the same
        geometry and warm-up flag that runs the same weights at the same precision, each of them gives bit for bit the
        frames and hops it gives here when both are pushed the same audio from here on, with :meth:`push` or
        :meth:`push_hops` in any mix.  Without temporal smoothing the records carry a zero smoothing state."""
        s = self._slots(slots)
        k = s.numel()
        records = torch.empty(k, self.state_floats, dtype=torch.float32, device=self.dev)
        hops = torch.zeros(k, dtype=torch.int64)
        self._current_args()
        self._call(self._lib.koe_stream_pool_snapshot, self._h, self._args_ref, s.data_ptr(), k, records.data_ptr(),
                   hops.data_ptr(), what="koe_stream_pool_snapshot")
        return StreamSnapshot(self.hop, self.W, self.half, self.warmup, hops, records)

    @torch.no_grad()
    def restore(self, snapshot: StreamSnapshot) -> list:
        """Opens one stream per record of `snapshot` in the lowest free slots and returns them, in record order: each
        continues from its recorded hop with its recorded state, expression input included (no :meth:`set_egemaps`
        needed).  The equality of :meth:`snapshot` holds whatever this pool's capacity and ``max_hops`` are and
        whatever its slots held before.  The restore is queued on the current stream: records written on another CUDA
        stream (a snapshot there, a copy from another device) need the caller's synchronisation first.  Raises
        ValueError for a snapshot of another hop, window, FFT size or warm-up flag, records that are not float32 on
        this pool's device or whose shapes disagree, or more records than free slots -- before anything is queued."""
        records, hops = self._check_snapshot(snapshot)
        k = hops.numel()
        slots = torch.empty(k, dtype=torch.int32)
        self._current_args()
        self._call(self._lib.koe_stream_pool_restore, self._h, self._args_ref, records.data_ptr(), hops.data_ptr(), k,
                   slots.data_ptr(), what="koe_stream_pool_restore")
        return slots.tolist()

    # ---- helpers ----------------------------------------------------------------------------------------------------
    def _check_snapshot(self, snap):
        if not isinstance(snap, StreamSnapshot):
            raise ValueError(f"restore takes a StreamSnapshot, got {type(snap).__name__}")
        mine = (self.hop, self.W, self.half, self.warmup)
        theirs = (snap.hop, snap.window_frames, snap.half_fft, snap.warmup)
        if theirs != mine:
            raise ValueError(f"snapshot of a pool with (hop, window_frames, half_fft, warmup) = {theirs}, this pool has "
                             f"{mine}")
        h, r = snap.hops, snap.records
        if not isinstance(h, torch.Tensor) or h.device.type != "cpu" or h.dtype != torch.int64 or h.dim() != 1:
            raise ValueError("snapshot hops must be a 1-D CPU int64 tensor")
        if not isinstance(r, torch.Tensor) or r.device != self.dev or r.dtype != torch.float32:
            raise ValueError(f"snapshot records must be float32 on {self.dev}, got "
                             f"{getattr(r, 'dtype', type(r).__name__)} on {getattr(r, 'device', None)}")
        if tuple(r.shape) != (h.numel(), self.state_floats):
            raise ValueError(f"snapshot records must be ({h.numel()}, {self.state_floats}) for {h.numel()} hops, got "
                             f"{tuple(r.shape)}")
        if h.numel() and int(h.min()) < 0:
            raise ValueError("snapshot hops must be >= 0")
        return r.contiguous(), h.contiguous()

    def _check(self, rc: int, what: str) -> None:
        if rc == -1:   # KOE_E_INVALID: misuse (slot out of range / not open / listed twice, pool full)
            msg = self._lib.koe_last_error()
            raise ValueError(f"{what}: {msg.decode() if msg else 'invalid argument'}")
        _lib.check(rc, what)

    def _call(self, fn, *args, what: str) -> None:
        if torch.cuda.current_device() == self._dev_index:
            rc = fn(*args, torch.cuda.current_stream(self.dev).cuda_stream)
        else:
            with torch.cuda.device(self.dev):
                rc = fn(*args, torch.cuda.current_stream(self.dev).cuda_stream)
        self._check(rc, what)

    def _slots(self, slots) -> torch.Tensor:
        s = slots if isinstance(slots, torch.Tensor) else torch.as_tensor(slots, dtype=torch.int64)
        if s.device.type != "cpu":
            raise ValueError("slots must be host (CPU) indices")
        if s.dim() != 1 or s.is_floating_point() or s.is_complex() or s.dtype == torch.bool:
            raise ValueError(f"slots must be a 1-D sequence of integers, got {s.dtype} of shape {tuple(s.shape)}")
        if s.dtype == torch.int32:        # (the library checks the range of every slot itself)
            return s.contiguous()
        if s.numel() and (int(s.min()) < 0 or int(s.max()) >= self.capacity):
            raise ValueError(f"slots must lie in [0, {self.capacity})")
        return s.to(torch.int32)

    def _egemaps(self, egemaps) -> torch.Tensor:
        if not isinstance(egemaps, torch.Tensor):
            raise ValueError(f"egemaps must be a torch.Tensor, got {type(egemaps).__name__}")
        if egemaps.device != self.dev or egemaps.dtype != torch.float32:
            raise ValueError(f"egemaps must be float32 on {self.dev}, got {egemaps.dtype} on {egemaps.device}")
        eg = egemaps.reshape(egemaps.shape[0], -1) if egemaps.dim() == 3 else egemaps
        if eg.dim() != 2 or eg.shape[1] != 264:
            raise ValueError(f"egemaps must be (k, 264) or (k, 3, 88), got {tuple(egemaps.shape)}")
        return eg.contiguous()

    def _set_egemaps(self, s: torch.Tensor, eg: torch.Tensor) -> None:
        self._current_args()
        self._call(self._lib.koe_stream_pool_set_egemaps, self._h, self._args_ref, s.data_ptr(), s.numel(), eg.data_ptr(),
                   what="koe_stream_pool_set_egemaps")

    def _current_args(self):
        # the folded weights are re-validated against the module's parameters by their in-place version counters every
        # call, and by the full walk over the module (replaced tensors: .to(), new Parameters) every 256th push
        m = self.model
        a = self._args
        key = (m.precision, m.use_temporal_smoothing, tuple(t._version for t in self._w_tensors))
        if a is None or self._args_key != key or (self.pushes & 255) == 0:
            a = self._args = self._build_args()
            self._args_key = (m.precision, m.use_temporal_smoothing, tuple(t._version for t in self._w_tensors))
        if m.use_temporal_smoothing:
            # sigmoid(smoothing_alpha) is read back once per parameter version, not once per hop (a device sync)
            ver = (m.smoothing_alpha.data_ptr(), m.smoothing_alpha._version)
            if self._alpha_key != ver:
                self._alpha = float(torch.sigmoid(m.smoothing_alpha.detach().float()))
                self._alpha_key = ver
            a.alpha = self._alpha
        return a

    def _build_args(self):
        m = self.model
        self._weights = m.dual_stream_attention.kernel_weights(m._compression)   # (kept alive: the block points into it)
        att = m.dual_stream_attention
        self._w_tensors = [t for _, t in att.named_parameters()] + [t for _, t in att.named_buffers()] + \
            ([] if m._compression is None else [m._compression["weight"], m._compression["bias"]])
        a = _lib.StreamPoolArgs()
        a.frontend, a.weights = self._fe._h, C.cast(C.pointer(self._weights.struct), C.c_void_p)
        a.tail, a.tail_compact = self.tail.data_ptr(), self.tail_compact.data_ptr()
        a.stage, a.stage_max = self.stage.data_ptr(), self.stage_max.data_ptr()
        a.ring_f, a.fmax_f = self.ring_f.data_ptr(), self.fmax_f.data_ptr()
        a.ring_r, a.fmax_r = self.ring_r.data_ptr(), self.fmax_r.data_ptr()
        a.row_l, a.fmax_l = self.row_l.data_ptr(), self.fmax_l.data_ptr()
        if self.n_edge == 2:
            a.ring_r2, a.fmax_r2 = self.ring_r2.data_ptr(), self.fmax_r2.data_ptr()
            a.row_l2, a.fmax_l2 = self.row_l2.data_ptr(), self.fmax_l2.data_ptr()
        a.expr_sigmoid, a.expr_compact, a.out = self.expr.data_ptr(), self.expr_compact.data_ptr(), self.out.data_ptr()
        a.ema_state, a.alpha = (self.state.data_ptr(), self._alpha) if m.use_temporal_smoothing else (None, 1.0)
        a.tables = self.tables.data_ptr()
        a.precision = _lib.PRECISIONS[m.precision]
        self._args_ref = C.byref(a)
        return a
