"""Time of packed warm-up batches (SequentialDualStreamModel.forward_varlen(..., warmup=True)) against the other ways to
get a frame at every hop of every clip, bf16, arms alternated call by call in one process:

  utterances    512 clips of 1-8.5 s (the utterances of varlen_timing.py), 30 fps: warmup=True; the warm-up stream-pool
                route (one StreamPool of capacity 512 with warm-up, every clip opened, drained with push_hops of up to
                max_hops hops per stream and call, the frames copied out, the streams closed); warmup=False (512 rows)
  recordings    256 clips of 10-60 s, 30 fps, stride 1: warmup=True against warmup=False
  utterances60  the utterances at 60 fps

Latency = host submit of the call -> its rows complete on the device (host sync), p50 / p99 over --calls calls after one
warm-up call per arm; the table also gives the time per output row.  Before timing, with smoothing off, the arms' rows
are compared: the steady rows (hops >= W - 1) of warmup=True with warmup=False's (torch.equal), and warmup=True with
the pool route's frames (max |d|, within 2e-4).  The timed calls run with smoothing on.  A separate torch.profiler run
gives per-kernel device time, and the core's time per lead window (utterances: every row is a lead window) against
per steady window (recordings, warmup=False: every row is a steady window).

    python scripts/varlen_warmup_timing.py [--calls 20] [--out profiles/varlen_warmup_timing.json]
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np
import torch

from koemorph_b200.streaming import StreamPool
from varlen_timing import gpu_info, kernel_times, make_model, workload

POOL_MAX_HOPS = 32
POOL_GATE = 2e-4   # two bf16 gates against the fp32 forward (tests/test_gpu_varlen_warmup.py)


def pct(xs):
    xs = sorted(xs)
    p = lambda q: xs[min(len(xs) - 1, int(q * len(xs)))]
    return {"p50": round(p(0.50), 4), "p99": round(p(0.99), 4), "calls": len(xs)}


def race(arms, calls):
    """Host submit -> device sync (ms) of every arm, the arms alternated call by call after one warm-up call each."""
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(calls):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3)
    return {k: pct(v) for k, v in times.items()}


def pool_route(m, audio, lens, eg):
    """A callable that computes every clip's frames with a warm-up StreamPool: (N, 52) rows in forward_varlen's order."""
    hop = m.hop_length
    n_hops = [L // hop for L in lens]
    offs = np.concatenate([[0], np.cumsum(lens)])
    B = len(lens)
    pool = StreamPool(m, B, max_hops=POOL_MAX_HOPS, warmup=True)

    def run():
        slots = pool.open(eg)
        pushed = [0] * B
        got = [[] for _ in range(B)]
        while True:
            plan = [(c, min(POOL_MAX_HOPS, n_hops[c] - pushed[c])) for c in range(B) if pushed[c] < n_hops[c]]
            if not plan:
                break
            x = torch.cat([audio[offs[c] + pushed[c] * hop:offs[c] + (pushed[c] + k) * hop] for c, k in plan])
            _, _, frames = pool.push_hops([slots[c] for c, _ in plan], x, [k for _, k in plan])
            frames = frames.clone()
            r = 0
            for c, k in plan:
                got[c].append(frames[r:r + k])
                pushed[c] += k
                r += k
        for s in slots:
            pool.close(s)
        return torch.cat([torch.cat(g) for g in got])
    return run


def check_rows(m, audio, lens, eg, with_pool):
    """Smoothing off: steady rows of warmup=True against warmup=False (equal), and warmup=True against the pool route."""
    m.use_temporal_smoothing = False
    hop, W = m.hop_length, m.window_frames
    warm = m.forward_varlen(audio, lens, egemaps=eg, warmup=True)
    plain = m.forward_varlen(audio, lens, egemaps=eg)
    ow, op = warm["frame_offsets"], plain["frame_offsets"]
    steady = 0
    for c, L in enumerate(lens):
        if L // hop >= W:
            n = int(op[c + 1] - op[c])
            assert torch.equal(warm["blendshapes"][int(ow[c + 1]) - n:int(ow[c + 1])], plain["blendshapes"][op[c]:op[c + 1]]), c
            steady += n
    out = {"rows": int(ow[-1]), "steady_rows_equal": steady}
    if with_pool:
        d = (warm["blendshapes"].double() - pool_route(m, audio, lens, eg)().double()).abs().max().item()
        assert d <= POOL_GATE, d
        out["max_abs_diff_vs_pool"] = d
    m.use_temporal_smoothing = True
    return out


def core_us(kernels):
    return sum(v for k, v in kernels.items() if "dual_stream_tc_kernel" in k)


def utterances(calls, fps):
    m = make_model(fps)
    lens = [int(x) for x in np.random.default_rng(1).integers(16000, 136000 + 1, 512)]
    audio, eg = workload(m, lens, 2)
    checked = check_rows(m, audio, lens, eg, with_pool=True)
    route = pool_route(m, audio, lens, eg)
    arms = {"warmup": lambda: m.forward_varlen(audio, lens, egemaps=eg, warmup=True),
            "pool_route": route,
            "plain": lambda: m.forward_varlen(audio, lens, egemaps=eg)}
    t = race(arms, calls)
    rows = {"warmup": checked["rows"], "pool_route": checked["rows"], "plain": len(lens)}
    res = {"clips": len(lens), "fps": fps, "rows": rows, "checked": checked, "latency_ms": t,
           "us_per_row_p50": {k: round(1e3 * t[k]["p50"] / rows[k], 4) for k in t},
           "ratio_pool_route_vs_warmup": round(t["pool_route"]["p50"] / t["warmup"]["p50"], 3)}
    kt = kernel_times(arms["warmup"])        # (a profiled call of its own, after the timed ones)
    res["kernels_us_warmup"] = kt
    res["core_us_per_lead_window"] = round(core_us(kt) / checked["rows"], 4)   # every row is a lead window
    return res


def recordings(calls):
    m = make_model(30)
    lens = [int(x) for x in np.random.default_rng(3).integers(10 * 16000, 60 * 16000 + 1, 256)]
    audio, eg = workload(m, lens, 4)
    checked = check_rows(m, audio, lens, eg, with_pool=False)
    arms = {"warmup": lambda: m.forward_varlen(audio, lens, egemaps=eg, warmup=True),
            "plain": lambda: m.forward_varlen(audio, lens, egemaps=eg)}
    t = race(arms, calls)
    rows = {"warmup": checked["rows"], "plain": sum(m.num_output_frames(L) for L in lens)}
    res = {"clips": len(lens), "fps": 30, "rows": rows, "checked": checked, "latency_ms": t,
           "us_per_row_p50": {k: round(1e3 * t[k]["p50"] / rows[k], 4) for k in t},
           "ratio_warmup_vs_plain": round(t["warmup"]["p50"] / t["plain"]["p50"], 3)}
    kw, kp = kernel_times(arms["warmup"]), kernel_times(arms["plain"])
    res["kernels_us"] = {"warmup": kw, "plain": kp}
    res["core_us_per_steady_window"] = round(core_us(kp) / rows["plain"], 4)   # warmup=False: every row is steady
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--out", default="profiles/varlen_warmup_timing.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("varlen_warmup_timing.py needs a CUDA device")
    if args.calls < 20:
        sys.exit("--calls must be at least 20")
    with torch.no_grad():
        res = {"gpu": gpu_info(), "calls": args.calls, "precision": "bf16", "pool_max_hops": POOL_MAX_HOPS}
        res["utterances"] = utterances(args.calls, 30)
        res["recordings"] = recordings(args.calls)
        res["utterances60"] = utterances(args.calls, 60)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not kk.startswith("kernels")} if isinstance(v, dict) else v)
                      for k, v in res.items()}, indent=1))


if __name__ == "__main__":
    main()
