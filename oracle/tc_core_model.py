"""Float64 model of the bf16 tensor-core core (``dual_stream_tc_kernel``, koemorph_b200/csrc/dual_stream_tc.cu).

TEST INFRASTRUCTURE ONLY, like ``koemorph_oracle``.  The oracle's ``dual_stream_core`` is the reference arithmetic; this
module is the arithmetic the tensor-core kernel is *designed* to perform: the same operation with its operands rounded
to bf16 (round to nearest even) at the kernel's rounding points and everything else exact.  The kernel accumulates in
fp32, so it sits within a small floor of this model, far closer than to the reference, whose distance is the bf16
design error.  A test can then gate the kernel just above that floor.

Rounding points:

* A operand (``stage_window``): ``bf16(fmaf(max(db - ref_db, -80), 1/80, 1))`` computed in fp32, ``ref_db`` the
  maximum of the window's frame maxima; prenormalised features: ``bf16(x)``.  Long-term rows past
  ``min(T, mel_seq)`` are 0; the short-term frames are ``T-3 .. T-1`` (missing ones, T < 3, are 0); column ``k_mel``
  is 1 and meets the encoder bias.
* weights (pre-tiled by ``model/folding.py``, rebuilt here from the state dict): ``bf16([Wc | bc])``,
  ``bf16(Qk_h diag(ln_g))``, ``bf16(Wv diag(ln_g))``, ``bf16(W1 Wmo Wo)``; ``tc_bv = fp32(Wv ln_b + bv)``, ``ba``
  and ``coef`` in fp32.
* ``enc = bf16(LayerNorm(z))`` without affine (mel_norm's affine lives in the weights).
* softmax unrounded; ``P`` rounded to bf16 for the PV product, the attention output is the head mean of unrounded P.
* ``vT = bf16(Wv' enc^T + tc_bv)``; ``O = bf16(P_bf16 vT)``.
* decoder tail: ``H = O Wa'^T``, ``logit = sum relu(H + ba) w2 + b2``, ``sigmoid``, ``clamp(coef y, 0, 1)``.

``rounding=False`` drops every rounding point (the model is then the folded reference, exactly); ``accum=torch.float32``
carries the arithmetic in fp32 instead of float64, a stand-in for the kernel's own accumulation.  ``mutate`` applies
one of ``MUTATIONS``, plausible kernel bugs, so that a test can show a gate would catch them.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import numpy as np
import torch

from .koemorph_oracle import MOUTH_INDICES

MUTATIONS = (
    "truncate",            # activation conversions to bf16 truncate instead of rounding to nearest even
    "no_value_bias_head",  # the value bias (tc_bv) is missing for the last head
    "softmax_79",          # the softmax denominator sums 79 of the 80 tokens
    "drop_last_short",     # the last short-term frame is dropped from the A operand
    "drop_tail_chunk",     # the last 8-frame K chunk of long-term frames is left zero
)

# Gates of the kernel against this model (tests/test_gpu_tc_core.py), per weight style: max |d| on the mouth
# blendshapes, the pre-fusion mouth sigmoid and the head-averaged attention.  Set at 1.1-2x the largest deviation
# measured on a B200 (1000 W) over every case of that test (the maxima are listed there); tests/test_tc_core_model.py
# checks on the CPU that each mutation above moves the model by more than 5x these on at least one output, and fp32
# accumulation by less than a quarter of them.
GATES = {
    "stress": (1.25e-5, 3.3e-4, 2.6e-4),
    "init": (1e-6, 2.8e-5, 5e-7),
    "offset": (2.7e-5, 7.7e-4, 1.5e-3),
}

_P = "dual_stream_attention."


def _bf16(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.bfloat16).to(x.dtype)


def _bf16_truncated(x: torch.Tensor) -> torch.Tensor:
    bits = x.to(torch.float32).view(torch.int32) & ~0xFFFF
    return bits.view(torch.float32).to(x.dtype)


def _f32(x: torch.Tensor) -> torch.Tensor:
    return x.to(torch.float32).to(x.dtype)


def tc_weights(weights, device="cpu", rounding: bool = True) -> Dict[str, torch.Tensor]:
    """The kernel's weights in float64, built from a ``make_weights``-style state dict (keys prefixed
    ``dual_stream_attention.``) without going through ``model/folding.py``."""
    g = lambda k: torch.as_tensor(np.asarray(weights[_P + k]), dtype=torch.float64, device=device)
    b16, f32 = (_bf16, _f32) if rounding else (lambda x: x, lambda x: x)
    d, nh = 256, 8
    hd = d // nh
    wc, bc = g("mel_channel_encoder.weight"), g("mel_channel_encoder.bias")
    inw, inb = g("mel_attention.in_proj_weight"), g("mel_attention.in_proj_bias")
    wq, wk, wv, bq, bv = inw[:d], inw[d:2 * d], inw[2 * d:], inb[:d], inb[2 * d:]
    ln_g, ln_b = g("mel_norm.weight"), g("mel_norm.bias")
    qt = (g("mouth_queries") @ wq.T + bq) / math.sqrt(hd)
    # scores = Qt_h (Wk_h (ln_g enc + ln_b) + bk_h): the terms without enc are constant along the keys
    qk = torch.stack([qt[:, h * hd:(h + 1) * hd] @ wk[h * hd:(h + 1) * hd] * ln_g for h in range(nh)])
    w1, b1 = g("blendshape_decoder.0.weight"), g("blendshape_decoder.0.bias")
    wo, bo = g("mel_attention.out_proj.weight"), g("mel_attention.out_proj.bias")
    wmo, bmo = g("mel_output_proj.weight"), g("mel_output_proj.bias")
    coef = 0.5 * (torch.softmax(g("mel_weights"), 0) + torch.softmax(g("emotion_weights"), 0))
    return {
        "wc": b16(torch.cat([wc, bc[:, None]], 1)),          # [256, k_mel + 1]
        "qk": b16(qk),                                       # [8, 28, 256]
        "wv": b16(wv * ln_g),                                # [256, 256]
        "wa": b16(w1 @ wmo @ wo),                            # [128, 256]
        "bv": f32(wv @ ln_b + bv),
        "ba": f32(w1 @ (wmo @ bo + bmo) + b1),
        "w2": g("blendshape_decoder.3.weight").reshape(-1),
        "b2": g("blendshape_decoder.3.bias").reshape(-1),
        "coef": f32(coef[MOUTH_INDICES]),
    }


def _normalise(db: torch.Tensor, ref_db: torch.Tensor, rounding: bool) -> torch.Tensor:
    """``fmaf(fmaxf(db - ref_db, -80), 1/80, 1)`` in fp32 (one rounding after the exact product and sum)."""
    if not rounding:
        return torch.clamp(db - ref_db, min=-80.0) / 80.0 + 1.0
    x = torch.clamp(_f32(db - ref_db), min=-80.0)
    return _f32(x * float(np.float32(1.0 / 80.0)) + 1.0)


def forward(W: Dict[str, torch.Tensor], mel_long: Optional[torch.Tensor] = None, mel_short: Optional[torch.Tensor] = None,
            db: Optional[torch.Tensor] = None, fmax: Optional[torch.Tensor] = None, rounding: bool = True,
            accum: torch.dtype = torch.float64, mutate: Optional[str] = None,
            eps: float = 1e-5) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """One window per row of the batch -> (mouth sigmoid [B, 28], mouth blendshapes [B, 28], attention [B, 28, 80]).

    Either prenormalised features, ``mel_long`` [B, T, 80] and ``mel_short`` [B, 3, 80] (koe_dual_stream_features), or
    a window's mel rows in dB, ``db`` [B, T, 80] (frame k already taken from the edge variant the kernel reads for it),
    with their frame maxima ``fmax`` [B, T] (koe_dual_stream_windows)."""
    if mutate is not None and mutate not in MUTATIONS:
        raise ValueError(f"unknown mutation {mutate!r}")
    r = (_bf16_truncated if mutate == "truncate" else _bf16) if rounding else (lambda x: x)
    mel_seq = W["wc"].shape[1] - 4
    dt, dev = torch.float64, W["wc"].device
    if db is not None:
        db = db.to(device=dev, dtype=dt)
        B, T = db.shape[:2]
        xn = _normalise(db, fmax.to(device=dev, dtype=dt).amax(1)[:, None, None], rounding)
        n3 = min(T, 3)
        short = torch.zeros(B, 3, 80, dtype=dt, device=dev)
        short[:, :n3] = xn[:, T - n3:]
        long = xn[:, :mel_seq]
    else:
        long, short = mel_long.to(device=dev, dtype=dt)[:, :mel_seq], mel_short.to(device=dev, dtype=dt)
        B = long.shape[0]
    Tl = long.shape[1]
    X = torch.zeros(B, 80, mel_seq + 4, dtype=dt, device=dev)
    X[:, :, :Tl] = r(long).transpose(1, 2)
    X[:, :, mel_seq:mel_seq + 3] = r(short).transpose(1, 2)
    X[:, :, mel_seq + 3] = 1.0
    if mutate == "drop_last_short":
        X[:, :, mel_seq + 2] = 0.0
    if mutate == "drop_tail_chunk" and Tl > 0:
        X[:, :, 8 * ((Tl - 1) // 8):Tl] = 0.0

    X = X.to(accum)
    w = {k: v.to(accum) for k, v in W.items()}
    z = X @ w["wc"].T                                                    # [B, 80, 256]
    # the kernel's one-pass variance (exact in float64; with accum=float32 it is the kernel's own cancellation)
    mean = z.mean(-1, keepdim=True)
    var = torch.clamp((z * z).mean(-1, keepdim=True) - mean * mean, min=0.0)
    enc = r((z - mean) * torch.rsqrt(var + eps))
    s = torch.einsum("hqk,btk->bhqt", w["qk"], enc)                     # [B, 8, 28, 80]
    if mutate == "softmax_79":
        e = torch.exp(s - s.amax(-1, keepdim=True))
        p = e / e[..., :79].sum(-1, keepdim=True)
    else:
        p = torch.softmax(s, -1)
    attn = p.mean(1)
    bv = w["bv"].clone()
    if mutate == "no_value_bias_head":
        bv[224:] = 0.0
    vt = r(enc @ w["wv"].T + bv)                                         # [B, 80 tokens, 256 = 32 h + d]
    o = r(torch.einsum("bhqt,bthd->bqhd", r(p), vt.reshape(B, 80, 8, 32)).reshape(B, 28, 256))
    h = o @ w["wa"].T + w["ba"]
    y = torch.sigmoid(torch.relu(h) @ w["w2"] + w["b2"])
    return y.to(dt), torch.clamp(w["coef"] * y, 0.0, 1.0).to(dt), attn.to(dt)
