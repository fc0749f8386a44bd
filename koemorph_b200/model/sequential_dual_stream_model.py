"""B200 drop-in for the reference's ``src/model/sequential_dual_stream_model.py``.

The reference slides a window of ``mel_sequence_length`` hops over the clip and, for EVERY output
frame, recomputes the whole window's librosa mel (``:101-120``) before running the core and the EMA.
Here each STFT frame is computed once: frame k of window i is global frame i*stride + k, except the
frames within n_fft/2 of a window edge, which see zeros beyond the edge (SURVEY.md section 8, note E).
Those are produced as separate "edge variants" by ``koe_logmel_power`` (lo_rel_hops / hi_rel_hops) on
the window grid; the dB reference of a window is the max over ITS frames, taken inside the core kernel.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional

import numpy as np
import torch

from .. import _lib
from .dual_stream_attention import _package
from .simplified_dual_stream_model import SimplifiedDualStreamModel


class SequentialDualStreamModel(SimplifiedDualStreamModel):
    """audio (B, L) -> blendshapes (B, T_out, 52), T_out = max(1, (L // hop - W) // stride + 1)."""

    def __init__(self, d_model: int = 256, num_heads: int = 8, num_blendshapes: int = 52, sample_rate: int = 16000,
                 target_fps: int = 30, mel_sequence_length: int = 256, emotion_config: Optional[Dict] = None,
                 device: str = "cuda", real_time_mode: bool = False, stride_frames: int = 1):
        super().__init__(d_model=d_model, num_heads=num_heads, num_blendshapes=num_blendshapes,
                         sample_rate=sample_rate, target_fps=target_fps, mel_sequence_length=mel_sequence_length,
                         emotion_config=emotion_config, device=device, real_time_mode=real_time_mode)
        if stride_frames < 1:
            raise ValueError("stride_frames must be >= 1")
        self.stride_frames = stride_frames
        self.window_frames = mel_sequence_length
        self.window_samples = self.window_frames * self.hop_length
        self.stride_samples = self.stride_frames * self.hop_length

    def num_output_frames(self, audio_length: int) -> int:
        """reference :84,96."""
        return max(1, (audio_length // self.hop_length - self.window_frames) // self.stride_frames + 1)

    def _forward_frames(self, audio, eg, return_attention, out=None):
        """The stateless part of forward(): (B, T_out, 52) smoothed blendshapes (+ sigmoid, attention)."""
        B, L = audio.shape
        hop, W, stride = self.hop_length, self.window_frames, self.stride_frames
        n_out = self.num_output_frames(L)
        T_w = W + 1                                        # librosa: 1 + (W * hop) // hop frames per window
        n_frames = (n_out - 1) * stride + T_w              # global frames touched
        # a single window that already spans the whole (zero padded) clip has no interior edges
        n_edge = 0 if (n_out == 1 and L <= self.window_samples) else math.ceil((self.n_fft // 2) / hop)
        if n_edge > _lib.MAX_EDGE:
            raise NotImplementedError(f"hop {hop} needs {n_edge} edge variants per side (max {_lib.MAX_EDGE})")
        return self._forward_windows(audio, eg, n_frames, T_w, stride, n_out, n_edge, self.use_temporal_smoothing,
                                     return_attention, out=out)

    @torch.no_grad()
    def forward(self, audio: torch.Tensor, return_attention: bool = False,
                egemaps: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """reference :63-167.  ``out`` (extension): a preallocated contiguous (B, T_out, 52) float32 CUDA tensor that
        receives the blendshapes (a corpus sweep lets every batch write where the results will be gathered)."""
        audio = self._check_audio(audio)
        B, L = audio.shape
        eg = self._check_egemaps(egemaps, B, audio.device)
        out, sig, attn = self._forward_frames(audio, eg, return_attention, out=out)
        # the reference leaves the smoothing state at the last frame of the sequence (:99,136): a view, like its .detach()
        self.prev_blendshapes = out[:, -1] if self.use_temporal_smoothing else None
        res = _package(out, sig, attn, return_attention)
        res["num_frames"] = out.shape[1]
        res["fps"] = self.target_fps
        res["emotion_backend"] = "egemaps_input"
        res["emotion_processing_time"] = 0.0
        return res

    @torch.no_grad()
    def forward_varlen(self, audio: torch.Tensor, lengths, egemaps: Optional[torch.Tensor] = None,
                       return_attention: bool = False, out: Optional[torch.Tensor] = None,
                       warmup: bool = False) -> Dict[str, torch.Tensor]:
        """A packed batch of clips of different lengths as one native forward (koe_forward_varlen).

        ``audio``: 1-D float32 CUDA tensor with the clips back to back, ``audio.numel() == sum(lengths)``; ``lengths``:
        host sequence or CPU integer tensor, one entry >= 0 per clip; ``egemaps``: (B, 264) or (B, 3, 88).  Clip c's
        ``num_output_frames(lengths[c])`` frames are rows ``frame_offsets[c]:frame_offsets[c + 1]`` of ``blendshapes``
        (N, 52) (and of the attention / sigmoid outputs), each equal to ``forward`` on that clip alone, smoothing
        included.  ``out``: a preallocated contiguous (N, 52) float32 tensor.  Afterwards ``prev_blendshapes`` holds every
        clip's last frame, (B, 52).

        ``warmup=True`` (koe_forward_varlen_ex with KOE_VARLEN_WARMUP) gives the frames a warm-up ``StreamPool`` would
        emit for each clip, from its first hop on.  With W = ``mel_sequence_length``, s = ``stride_frames`` and
        n = ``lengths[c] // hop`` complete hops, clip c gets one row per hop h = W - 1 (mod s) that it completes: h = r,
        r + s, ... <= n - 1 with r = (W - 1) % s (every hop 0 .. n - 1 when s = 1), ascending.  Rows at h >= W - 1 are,
        with smoothing off, bit for bit the rows of ``warmup=False``; rows at h < W - 1 are
        ``SimplifiedDualStreamModel.forward`` on the clip's first (h + 1) * hop samples.  A clip of fewer than W hops
        gets no padded window.  Smoothing restarts at each clip's first row and runs over all of its rows, so with
        smoothing on the rows from W - 1 on are the smoothing of these rows, not those of ``warmup=False``.  A clip that
        completes no grid hop (``lengths[c] < (r + 1) * hop``) raises ``ValueError``."""
        if not isinstance(warmup, bool):
            raise ValueError(f"warmup must be a bool, got {type(warmup).__name__}")
        if not isinstance(audio, torch.Tensor) or not audio.is_cuda:
            raise ValueError("audio must be a 1-D float32 CUDA tensor holding the clips back to back")
        audio = _lib.require_cuda(audio, "audio")
        if audio.dim() != 1:
            raise ValueError(f"audio must be 1-D (the clips back to back), got {tuple(audio.shape)}")
        lens = self._check_lengths(lengths, audio.numel())
        B = lens.numel()
        dev = audio.device
        eg = self._check_egemaps(egemaps, B, dev)
        hop, W, stride = self.hop_length, self.window_frames, self.stride_frames
        n_out = self.varlen_rows(lens, warmup)
        offsets = torch.zeros(B + 1, dtype=torch.int64)
        torch.cumsum(n_out, 0, out=offsets[1:])
        N = int(offsets[-1])
        if out is None:
            out = torch.empty(N, 52, dtype=torch.float32, device=dev)
        elif out.shape != (N, 52) or out.dtype != torch.float32 or not out.is_contiguous() or out.device != dev:
            raise ValueError(f"out must be a contiguous float32 ({N}, 52) tensor on {dev}")
        sig = torch.empty(N, 52, dtype=torch.float32, device=dev) if return_attention else None
        attn = torch.empty(N, 28, 80, dtype=torch.float32, device=dev) if return_attention else None
        if B > 0:
            lib = _lib.load()
            w = self.dual_stream_attention.kernel_weights(self._compression)
            a = _lib.ForwardVarlenArgs()
            a.frontend, a.weights = self._frontend(dev)._h, C.addressof(w.struct)
            # (a batch of empty clips reads no sample, but the ABI wants a pointer)
            src = audio if audio.numel() > 0 else torch.zeros(1, dtype=torch.float32, device=dev)
            a.audio, a.lengths_host, a.n_clips = src.data_ptr(), lens.data_ptr(), B
            a.hop, a.window_frames, a.stride_frames, a.half_fft = hop, W, stride, self.n_fft // 2
            a.smooth = 1 if self.use_temporal_smoothing else 0
            a.alpha = self._alpha() if self.use_temporal_smoothing else 0.0
            a.precision = _lib.PRECISIONS[self.precision]
            flags = _lib.VARLEN_WARMUP if warmup else 0
            n_win, n_frames, ws_bytes = C.c_int64(), C.c_int64(), C.c_int64()
            _lib.check(lib.koe_forward_varlen_size_ex(C.byref(a), flags, C.byref(n_win), C.byref(n_frames),
                                                      C.byref(ws_bytes)), "koe_forward_varlen_size_ex")
            if n_win.value != N:
                raise RuntimeError(f"koe_forward_varlen_size_ex: {n_win.value} windows, the model counts {N}")
            ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
            a.egemaps, a.workspace, a.workspace_bytes = eg.data_ptr(), ws.data_ptr(), ws_bytes.value
            a.out = out.data_ptr()
            a.sigmoid_out = sig.data_ptr() if sig is not None else None
            a.attn_out = attn.data_ptr() if attn is not None else None
            with torch.cuda.device(dev):
                _lib.check(lib.koe_forward_varlen_ex(C.byref(a), flags, _lib.stream_ptr(dev)), "koe_forward_varlen_ex")
        # as forward: the smoothing state is each clip's last frame
        self.prev_blendshapes = None
        if self.use_temporal_smoothing:
            # (the row indices go up from pinned memory: a pageable copy would hold the host until the forward is done)
            self.prev_blendshapes = out[(offsets[1:] - 1).pin_memory().to(dev, non_blocking=True)]
        res = _package(out, sig, attn, return_attention)
        res["frame_offsets"] = offsets
        res["num_frames"] = N
        res["fps"] = self.target_fps
        res["emotion_backend"] = "egemaps_input"
        res["emotion_processing_time"] = 0.0
        return res

    def varlen_rows(self, lengths: torch.Tensor, warmup: bool = False) -> torch.Tensor:
        """Output rows of each clip of ``forward_varlen`` for the CPU int64 ``lengths``: ``num_output_frames`` per clip,
        or with ``warmup`` the hops h = W - 1 (mod stride) from r = (W - 1) % stride on that the clip completes (raises
        ``ValueError`` for a clip that completes none)."""
        hop, W, stride = self.hop_length, self.window_frames, self.stride_frames
        n_out = torch.clamp((lengths // hop - W) // stride + 1, min=1)     # num_output_frames, per clip
        if not warmup:
            return n_out
        r = (W - 1) % stride
        n_hops = lengths // hop
        last_lead = torch.clamp(n_hops - 1, max=W - 2)                  # the last hop a lead window can end on
        leads = torch.where(last_lead >= r, torch.div(last_lead - r, stride, rounding_mode="floor") + 1, 0)
        rows = leads + torch.where(n_hops >= W, n_out, 0)
        if rows.numel() > 0 and int(rows.min()) == 0:
            c = int(torch.nonzero(rows == 0)[0, 0])
            raise ValueError(f"clip {c} of {int(lengths[c])} samples completes no hop of the output grid: warm-up rows "
                             f"start at {r + 1} complete hops of {hop} samples")
        return rows

    @staticmethod
    def _check_lengths(lengths, n_samples: int) -> torch.Tensor:
        """Clip lengths as a contiguous CPU int64 tensor; they must be >= 0 and add up to the packed audio."""
        if isinstance(lengths, torch.Tensor):
            if lengths.device.type != "cpu" or lengths.is_floating_point() or lengths.is_complex() or lengths.dtype == torch.bool:
                raise ValueError("lengths must be a host sequence or a CPU integer tensor")
            lens = lengths.to(torch.int64).reshape(-1).contiguous()
        else:
            arr = np.asarray(lengths)
            if arr.size > 0 and arr.dtype.kind not in "iu":
                raise ValueError(f"lengths must be integers, got {arr.dtype}")
            lens = torch.from_numpy(arr.astype(np.int64).reshape(-1))
        if lens.numel() > 0 and int(lens.min()) < 0:
            raise ValueError(f"lengths must be >= 0, got {int(lens.min())}")
        if int(lens.sum()) != n_samples:
            raise ValueError(f"lengths add up to {int(lens.sum())} samples, audio holds {n_samples}")
        return lens

    @torch.no_grad()
    def forward_single_frame(self, audio: torch.Tensor, frame_idx: int = None,
                             egemaps: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        """reference :169-181."""
        return SimplifiedDualStreamModel.forward(self, audio, return_attention=False, egemaps=egemaps)
