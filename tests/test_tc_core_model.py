"""The float64 model of the bf16 tensor-core core (oracle/tc_core_model.py) on the CPU: it is the reference when its
rounding is switched off, its weights are exactly the ones the kernel streams, and the gates that
tests/test_gpu_tc_core.py applies with it would catch plausible kernel bugs."""
import numpy as np
import pytest
import torch

from oracle import koemorph_oracle as O
from oracle import tc_core_model as M

_P = "dual_stream_attention."


def _reference(w, lt, st, mel_seq):
    ref = O.dual_stream_core(w, lt, st, np.zeros((lt.shape[0], 256)), mel_sequence_length=mel_seq,
                             return_attention=True, dtype=torch.float64)
    return ref["sigmoid"][:, O.MOUTH_INDICES], ref["blendshapes"][:, O.MOUTH_INDICES], ref["mel_attention_weights"]


def _max_dev(a, b):
    return [float((x - y).abs().max()) for x, y in zip(a, b)]


@pytest.mark.parametrize("fps", [30, 60])
def test_model_without_rounding_is_the_reference(fps):
    """With every rounding point switched off the model is the folded algebra of the reference core, on prenormalised
    features and on dB rows (window shorter than three frames, shorter than, equal to and longer than mel_seq)."""
    S = 256 if fps == 30 else 512
    rng = np.random.default_rng(fps)
    for style, seed in (("stress", 21), ("init", 1234)):
        w = O.make_weights(seed, fps, style=style)
        W = M.tc_weights(w, rounding=False)
        for T in (2, 100, S, S + 44):
            lt, st = rng.uniform(0, 1, (3, T, 80)), rng.uniform(0, 1, (3, 3, 80))
            got = M.forward(W, torch.from_numpy(lt), torch.from_numpy(st), rounding=False)
            assert max(_max_dev(got, _reference(w, lt, st, S))) < 1e-10, (style, T)
            # dB rows: the window's dB reference is its loudest frame, the floor 80 dB below it, short-term = last 3 frames
            db = rng.uniform(-130.0, -10.0, (3, T, 80))
            db[0, :, :40] = -200.0                       # far below the floor
            fmax = db.max(-1)
            x = (np.maximum(db - fmax.max(1)[:, None, None], -80.0) + 80.0) / 80.0
            short = np.zeros((3, 3, 80))
            short[:, :min(T, 3)] = x[:, T - min(T, 3):]
            got = M.forward(W, db=torch.from_numpy(db), fmax=torch.from_numpy(fmax), rounding=False)
            assert max(_max_dev(got, _reference(w, x, short, S))) < 1e-10, (style, T, "dB rows")


def _untile(flat, rows, k, rows_per_stage, k_per_stage):
    """Inverse of the pre-tiled stage images: element (r, k) of a stage sits at bf16 index
    ((r//8)*(chunks*128) + (k//8)*128 + (r%8)*16 + (k%8)*2) / 2, stages cut rows-outer, K-inner."""
    r = torch.arange(rows_per_stage)[:, None]
    c = torch.arange(k_per_stage)[None, :]
    idx = ((r // 8) * (k_per_stage // 8 * 128) + (c // 8) * 128 + (r % 8) * 16 + (c % 8) * 2) // 2
    stages = flat.view(-1, 8192)
    out = torch.empty(rows, k, dtype=flat.dtype)
    i = 0
    for r0 in range(0, rows, rows_per_stage):
        for k0 in range(0, k, k_per_stage):
            out[r0:r0 + rows_per_stage, k0:k0 + k_per_stage] = stages[i][idx]
            i += 1
    assert i == stages.shape[0]
    return out


@pytest.mark.parametrize("k_mel,n_stages", [(259, 29), (515, 37)])
def test_weight_pack_is_the_models_bf16_weights(k_mel, n_stages):
    """The pre-tiled bf16 stages that the kernel streams, untiled, equal the model's weights bit for bit: stage count,
    zero K padding up to the half-full last stage of the first GEMM, the encoder-bias column, zero query rows 28..31
    of every head, and the value bias."""
    from koemorph_b200.model.folding import fold
    w = O.make_weights(7, 30 if k_mel == 259 else 60, style="stress")
    sd = {k[len(_P):]: torch.from_numpy(np.array(v)) for k, v in w.items() if k.startswith(_P)}
    cw = fold(sd, 8, 1.0, "cpu")
    pack = cw.tensors["tc_bf16"]
    assert pack.dtype == torch.bfloat16 and pack.numel() * 2 == n_stages * 16384 and cw.struct.tc_stages == n_stages
    W = M.tc_weights(w)
    n_g1 = n_stages - 20
    g1, rest = pack[:n_g1 * 8192], pack[n_g1 * 8192:]
    wc = _untile(g1, 256, 32 * n_g1, 256, 32)
    assert torch.equal(wc[:, :k_mel + 1], W["wc"].to(torch.bfloat16))
    assert not wc[:, k_mel + 1:].any()
    qk = _untile(rest[:8 * 8192], 256, 256, 128, 64).view(8, 32, 256)
    assert torch.equal(qk[:, :28], W["qk"].to(torch.bfloat16)) and not qk[:, 28:].any()
    assert torch.equal(_untile(rest[8 * 8192:16 * 8192], 256, 256, 128, 64), W["wv"].to(torch.bfloat16))
    assert torch.equal(_untile(rest[16 * 8192:], 128, 256, 128, 64), W["wa"].to(torch.bfloat16))
    assert torch.equal(cw.tensors["tc_bv"], W["bv"].to(torch.float32))
    assert torch.equal(cw.tensors["ba"], W["ba"].to(torch.float32))


@pytest.mark.parametrize("style,seed", [("stress", 21), ("init", 1234)])
def test_gates_catch_the_mutations_and_pass_fp32_accumulation(style, seed):
    """Each kernel bug of MUTATIONS moves the model by more than 5x the GPU test's gate on at least one output, while
    carrying the arithmetic in fp32 (as the kernel accumulates) stays under a quarter of every gate."""
    w = O.make_weights(seed, 30, style=style)
    W = M.tc_weights(w)
    rng = np.random.default_rng(5)
    lt = torch.from_numpy(rng.uniform(0, 1, (6, 256, 80)).astype(np.float32))
    st = torch.from_numpy(rng.uniform(0, 1, (6, 3, 80)).astype(np.float32))
    gates = M.GATES[style]
    # outputs in the order of GATES: blendshapes, sigmoid, attention
    order = lambda r: (r[1], r[0], r[2])
    base = order(M.forward(W, lt, st))
    dev = _max_dev(order(M.forward(W, lt, st, accum=torch.float32)), base)
    assert all(d < g / 4 for d, g in zip(dev, gates)), f"fp32 accumulation: {dev} against gates {gates}"
    for mutation in M.MUTATIONS:
        dev = _max_dev(order(M.forward(W, lt, st, mutate=mutation)), base)
        assert max(d / g for d, g in zip(dev, gates)) > 5, f"{mutation}: {dev} against gates {gates}"
