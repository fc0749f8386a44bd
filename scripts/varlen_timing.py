"""Time of SequentialDualStreamModel.forward_varlen (one packed batch of clips of different lengths) against the ways a
user handles such clips without it, bf16, arms alternated call by call in one process, CUDA events, p50 over --calls:

  utterances   512 clips of 1-8.5 s, 30 fps: every clip is one 257-frame window, so the reference arm is forward on
               512 x 8.5 s clips (the same windows and frames).                                      target <= 1.10x
  recordings   256 clips of 10-60 s, 30 fps, stride 1: packed; one forward per clip; padded to the longest clip (rows
               past each clip's own frames thrown away); a uniform batch at the mean length (about the same windows
               and frames).                                                        target <= 1.10x the uniform batch
  recordings60 the recordings workload at 60 fps with 64 clips.

Every shape is warmed up first.  Per-kernel times of the packed and the uniform arm come from a separate torch.profiler
run.  Lengths are seeded.

    python scripts/varlen_timing.py [--calls 20] [--out profiles/varlen_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import koemorph_b200 as K
from oracle import koemorph_oracle as O  # weight generator only


def make_model(fps):
    w = O.make_weights(1234, fps, style="init")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length={30: 256, 60: 512}[fps]).cuda().eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = "bf16"
    return m


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def race(arms, calls):
    """p50 (ms) of every arm, the arms alternated call by call after one warm-up call each."""
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(calls):
        for k, fn in arms.items():
            times[k].append(event_ms(fn))
    return {k: round(float(np.median(v)), 4) for k, v in times.items()}


def kernel_times(fn):
    """Device time per kernel name (us) of one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.device_time_total > 0:
            out[e.key[:90]] = round(e.device_time_total, 1)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def workload(m, lens, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    audio = (torch.rand(sum(lens), generator=g, device="cuda") * 2 - 1) * 0.3
    eg = torch.randn(len(lens), 264, generator=g, device="cuda")
    return audio, eg


def utterances(calls):
    m = make_model(30)
    lens = [int(x) for x in np.random.default_rng(1).integers(16000, 136000 + 1, 512)]
    audio, eg = workload(m, lens, 2)
    full = (torch.rand(512, 136000, device="cuda") * 2 - 1) * 0.3
    arms = {"packed": lambda: m.forward_varlen(audio, lens, egemaps=eg),
            "uniform_8.5s": lambda: m(full, egemaps=eg)}
    t = race(arms, calls)
    return {"clips": 512, "windows": len(lens), "p50_ms": t, "ratio_packed_vs_uniform": round(t["packed"] / t["uniform_8.5s"], 3),
            "target": 1.10, "kernels_us": {"packed": kernel_times(arms["packed"]), "uniform_8.5s": kernel_times(arms["uniform_8.5s"])}}


def recordings(calls, fps, n_clips, seed):
    m = make_model(fps)
    lens = [int(x) for x in np.random.default_rng(seed).integers(10 * 16000, 60 * 16000 + 1, n_clips)]
    audio, eg = workload(m, lens, seed + 1)
    offs = np.concatenate([[0], np.cumsum(lens)])
    clips = [audio[offs[c]:offs[c + 1]][None] for c in range(n_clips)]
    L_max, L_mean = max(lens), int(round(np.mean(lens)))
    padded = torch.zeros(n_clips, L_max, device="cuda")
    for c in range(n_clips):
        padded[c, :lens[c]] = audio[offs[c]:offs[c + 1]]
    uniform = (torch.rand(n_clips, L_mean, device="cuda") * 2 - 1) * 0.3
    windows = sum(m.num_output_frames(L) for L in lens)
    arms = {"packed": lambda: m.forward_varlen(audio, lens, egemaps=eg),
            "per_clip": lambda: [m(clips[c], egemaps=eg[c:c + 1]) for c in range(n_clips)],
            "padded": lambda: m(padded, egemaps=eg),
            "uniform_mean": lambda: m(uniform, egemaps=eg)}
    t = race(arms, calls)
    return {"clips": n_clips, "fps": fps, "windows": windows, "windows_padded": n_clips * m.num_output_frames(L_max),
            "windows_uniform_mean": n_clips * m.num_output_frames(L_mean), "p50_ms": t,
            "ratio_packed_vs_uniform_mean": round(t["packed"] / t["uniform_mean"], 3),
            "ratio_per_clip_vs_packed": round(t["per_clip"] / t["packed"], 3),
            "ratio_padded_vs_packed": round(t["padded"] / t["packed"], 3), "target": 1.10,
            "kernels_us": {"packed": kernel_times(arms["packed"]), "uniform_mean": kernel_times(arms["uniform_mean"])}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default="profiles/varlen_timing.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("varlen_timing.py needs a CUDA device")
    with torch.no_grad():
        res = {"gpu": gpu_info(), "calls": args.calls, "precision": "bf16",
               "utterances": utterances(args.calls),
               "recordings": recordings(args.calls, 30, 256, 3),
               "recordings60": recordings(args.calls, 60, 64, 5)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v if k in ("gpu",) else {kk: vv for kk, vv in v.items() if kk != "kernels_us"})
                      for k, v in res.items() if isinstance(v, dict)}, indent=1))


if __name__ == "__main__":
    main()
