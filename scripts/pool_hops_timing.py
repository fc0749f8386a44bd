"""Per-call latency of StreamPool.push_hops (several hops per stream in one call) against draining the same hops with
StreamPool.push (one hop per stream per call), bf16, 30 fps, 8.5 s context; the two arms alternate call by call in one
process, each on its own pool fed the same audio:

  a) 1024 streams x 8 hops:  one push_hops              vs 8 pushes of all 1024 streams
  b) 4096 streams, a seeded 25 % carry 2-4 hops, the rest 1:
                             one push_hops              vs pushes until every stream is drained (4 pushes: all, then those
                                                           with >= 2, >= 3, 4 hops left)
  c) 256 streams x 30 hops (1 s chunks): one push_hops  vs 30 pushes

Latency = host submit of the whole backlog -> all its frames complete on the device (host sync); `host` is the time until
the last call returns (enqueue only).  Every stream is warmed past its W-th hop first, so every hop emits a frame.  The
first calls of each scenario are not timed: there the frames of both arms are compared with torch.equal (each stream's
frames in hop order).

    python scripts/pool_hops_timing.py [--calls 40] [--out profiles/pool_hops_timing.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import koemorph_b200 as K
from koemorph_b200.streaming import StreamPool
from oracle import koemorph_oracle as O  # weight generator only

VERIFY_CALLS = 3


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


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi (name, power.limit, clocks.max.sm)": q[0] if q else "unavailable"}


class Scenario:
    """n streams open in a burst pool (max_hops = max(counts)) and in a default pool; call i feeds both the same audio:
    stream s's counts[s] next hops."""

    def __init__(self, m, counts, eg, hops_pool):
        self.m, self.dev = m, eg.device
        self.counts = torch.as_tensor(counts, dtype=torch.int64)
        self.n, self.H = len(counts), int(self.counts.max())
        self.hop, self.W = m.hop_length, m.mel_sequence_length
        self.total = int(self.counts.sum())
        self.hops_pool = hops_pool                                     # [P, hop] random hops, indexed cyclically
        self.burst = StreamPool(m, self.n, max_hops=self.H)
        self.plain = StreamPool(m, self.n)
        self.slots = torch.tensor(self.burst.open(eg[:self.n]), dtype=torch.int32)
        assert self.plain.open(eg[:self.n]) == self.slots.tolist()
        # stream s's hops of a call are rows offset[s] .. offset[s] + counts[s] of the call's audio; drain r of the plain
        # arm pushes hop r of every stream with counts > r
        self.offset = torch.cumsum(self.counts, 0) - self.counts
        self.drains = [torch.nonzero(self.counts > r).flatten() for r in range(self.H)]
        self.drain_slots = [self.slots[d].contiguous() for d in self.drains]
        self.call = 0

    def audio(self):
        P = self.hops_pool.shape[0]
        idx = (torch.arange(self.total, device=self.dev) * 7 + self.call * 131) % P
        self.call += 1
        x = self.hops_pool[idx]                                        # (total, hop), stream-major
        rows = [(self.offset[d] + r).to(self.dev) for r, d in enumerate(self.drains)]
        return x, [x[r].contiguous() for r in rows]

    def warm(self):
        need = -(-(self.W + 1) // int(self.counts.min()))             # calls until every stream is past its W-th hop
        while self.call < need:
            x, per_drain = self.audio()
            self.burst.push_hops(self.slots, x, self.counts)
            for s, xr in zip(self.drain_slots, per_drain):
                self.plain.push(s, xr)
        torch.cuda.synchronize()

    def run_burst(self, x):
        return self.burst.push_hops(self.slots, x, self.counts)

    def run_plain(self, per_drain, keep=False):
        out = []
        for s, xr in zip(self.drain_slots, per_drain):
            emitted, frames = self.plain.push(s, xr)
            if keep:
                out.append((emitted, frames.clone()))
        return out

    def verify(self):
        x, per_drain = self.audio()
        slots, hops, frames = self.run_burst(x)
        frames = frames.clone()
        drained = self.run_plain(per_drain, keep=True)
        torch.cuda.synchronize()
        assert slots.numel() == self.total, "every hop of a warmed stream emits"
        ok = True
        for r, (emitted, f) in enumerate(drained):
            assert torch.equal(emitted.to(torch.int32), self.drain_slots[r])
            ok &= torch.equal(frames[(self.offset[self.drains[r]] + r).to(self.dev)], f)
        return ok

    def time(self, calls):
        t = {"push_hops": [], "push": [], "push_hops_host": [], "push_host": []}
        mismatches = 0
        for _ in range(VERIFY_CALLS):
            mismatches += int(not self.verify())
        for i in range(calls):
            x, per_drain = self.audio()
            arms = [("push_hops", lambda: self.run_burst(x)), ("push", lambda: self.run_plain(per_drain))]
            for name, fn in (arms if i % 2 == 0 else arms[::-1]):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                t1 = time.perf_counter()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                t[name].append((t2 - t0) * 1e3)
                t[name + "_host"].append((t1 - t0) * 1e3)
        res = {k: pct(v) for k, v in t.items()}
        res["ratio_p50 (push_hops / push)"] = round(res["push_hops"]["p50"] / res["push"]["p50"], 4)
        res["hops"], res["streams"], res["push_calls_per_backlog"] = self.total, self.n, len(self.drains)
        res["verified_calls"], res["verified_calls_with_differing_frames"] = VERIFY_CALLS, mismatches
        return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=40)
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"])
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                   "profiles", "pool_hops_timing.json"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    m = make_model(dev, args.precision)
    hops_pool = 0.1 * torch.randn(4099, m.hop_length, device=dev)
    eg = torch.randn(4096, 264, device=dev)
    res = {"gpu": gpu_info(), "precision": args.precision, "fps": 30, "timed_calls": args.calls,
           "note": "latency = host submit of the backlog -> device sync, ms; *_host = until the last call returns; "
                   "arms alternated call by call"}
    rng = np.random.default_rng(0)
    mixed = np.ones(4096, dtype=np.int64)
    late = rng.random(4096) < 0.25
    mixed[late] = rng.integers(2, 5, int(late.sum()))
    for key, counts in (("a_1024_streams_x_8_hops", [8] * 1024), ("b_4096_streams_25pct_2to4_hops", mixed.tolist()),
                        ("c_256_streams_x_30_hops", [30] * 256)):
        sc = Scenario(m, counts, eg, hops_pool)
        sc.warm()
        res[key] = sc.time(args.calls)
        print(key, json.dumps(res[key]), flush=True)
        del sc
        torch.cuda.empty_cache()
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
