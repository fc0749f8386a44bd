"""Per-call latency of StreamPool.push against StreamingEngine.step (30 fps, 8.5 s context), pool and engine alternated
call by call in one process:

  a) capacity 4096, all 4096 streams pushing every call      vs StreamingEngine(4096)
  b) capacity 4096, a rotating 1024 of them pushing per call  vs StreamingEngine(1024)
  c) capacity 256, all pushing                                vs StreamingEngine(256)
  d) host time of one push / step at 4096 streams (the call alone, issued on an idle device)

Latency = host submit of one hop for every listed stream -> all outputs complete on the device (host sync), as in
scripts/bench_configs.py c4.  Every stream is warmed past its W-th hop first, so every timed call emits.  In (a) the pool
and the engine are fed the same hops: their frames are compared bit for bit after every call.

    python scripts/pool_timing.py [--calls 300] [--precision bf16] [--out profiles/pool_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import koemorph_b200 as K
from koemorph_b200.streaming import StreamingEngine, StreamPool
from oracle import koemorph_oracle as O  # weight generator only


def make_model(dev, precision):
    w = O.make_weights(1234, 30, style="init")
    m = K.SequentialDualStreamModel().to(dev).eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = precision
    return m


def pct(xs):
    xs = sorted(xs)
    p = lambda q: xs[min(len(xs) - 1, int(q * len(xs)))]
    return {"p50": round(p(0.50), 4), "p99": round(p(0.99), 4), "max": round(xs[-1], 4), "calls": len(xs)}


def timed_call(fn):
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=300)
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = make_model(dev, args.precision)
    W, hop = m.mel_sequence_length, m.hop_length
    hops = [0.1 * torch.randn(4096, hop, device=dev) for _ in range(8)]
    eg = torch.randn(4096, 264, device=dev)
    res = {"gpu": gpu_info(), "precision": args.precision, "fps": 30, "calls": args.calls,
           "note": "latency = host submit -> device sync, ms per call; pool and engine alternated call by call"}

    def warm(eng, pool, slot_sets):
        for i in range(W + 4):
            if eng is not None:
                eng.step(hops[i % 8][:eng.S])
            for s in slot_sets:
                pool.push(s, hops[i % 8][:s.numel()])
        torch.cuda.synchronize()

    # ---- (a) 4096 of 4096, and (d) host time
    pool = StreamPool(m, 4096)
    slots = torch.tensor(pool.open(eg), dtype=torch.int32)
    assert slots.tolist() == list(range(4096))
    eng = StreamingEngine(m, 4096)
    eng.set_egemaps(eg)
    warm(eng, pool, [slots])
    t_pool, t_eng, mismatches = [], [], 0
    for i in range(args.calls):
        x = hops[i % 8]
        dt, (emitted, frames) = timed_call(lambda: pool.push(slots, x))
        t_pool.append(dt)
        dt, out = timed_call(lambda: eng.step(x))
        t_eng.append(dt)
        mismatches += int(emitted.numel() != 4096 or not torch.equal(frames, out))
    res["a_4096_of_4096"] = {"pool": pct(t_pool), "engine_4096": pct(t_eng),
                             "ratio_p50": round(pct(t_pool)["p50"] / pct(t_eng)["p50"], 4),
                             "frames_differing_from_engine": mismatches}
    h_pool, h_eng = [], []
    for i in range(100):
        x = hops[i % 8]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        pool.push(slots, x)
        h_pool.append((time.perf_counter() - t0) * 1e3)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.step(x)
        h_eng.append((time.perf_counter() - t0) * 1e3)
    torch.cuda.synchronize()
    res["d_host_ms_per_call_4096"] = {"pool": pct(h_pool), "engine": pct(h_eng)}

    # ---- (b) a rotating 1024 of the same 4096 (all warmed above)
    del eng
    eng = StreamingEngine(m, 1024)
    eng.set_egemaps(eg[:1024])
    warm(eng, pool, [])
    quarters = [slots[q * 1024:(q + 1) * 1024].clone() for q in range(4)]
    t_pool, t_eng = [], []
    for i in range(args.calls):
        x = hops[i % 8][:1024]
        dt, (emitted, _) = timed_call(lambda: pool.push(quarters[i % 4], x))
        assert emitted.numel() == 1024
        t_pool.append(dt)
        dt, _ = timed_call(lambda: eng.step(x))
        t_eng.append(dt)
    res["b_1024_of_4096_rotating"] = {"pool": pct(t_pool), "engine_1024": pct(t_eng),
                                      "ratio_p50": round(pct(t_pool)["p50"] / pct(t_eng)["p50"], 4)}
    del pool, eng
    torch.cuda.empty_cache()

    # ---- (c) 256 of 256
    pool = StreamPool(m, 256)
    slots = torch.tensor(pool.open(eg[:256]), dtype=torch.int32)
    eng = StreamingEngine(m, 256)
    eng.set_egemaps(eg[:256])
    warm(eng, pool, [slots])
    t_pool, t_eng = [], []
    for i in range(args.calls):
        x = hops[i % 8][:256]
        dt, _ = timed_call(lambda: pool.push(slots, x))
        t_pool.append(dt)
        dt, _ = timed_call(lambda: eng.step(x))
        t_eng.append(dt)
    res["c_256_of_256"] = {"pool": pct(t_pool), "engine_256": pct(t_eng),
                           "ratio_p50": round(pct(t_pool)["p50"] / pct(t_eng)["p50"], 4)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
