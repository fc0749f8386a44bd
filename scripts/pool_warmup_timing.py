"""Per-push latency of warm-up stream pools (StreamPool(..., warmup=True)) against pools without warm-up, bf16, 8.5 s
context; every push advances each of its streams by one hop, and the arms of a workload alternate (rotate) call by call
in one process, each on its own pool:

  n streams (4096 and 256), four arms:
    warmup      a warm-up pool whose streams are all in warm-up (ages spread over hops 0 .. W - 2 - calls, so that they
                stay there): every push runs n windows of 2 .. W frames
    warm_steady a warm-up pool whose streams are all past hop W - 1
    plain       a default pool (max_hops = 1) in steady state
    plain_hops  a pool with max_hops = 2 in steady state (the burst path, which a warm-up pool always runs)
  churn: 4096 streams, a seeded 1/8 of them in warm-up and the rest in steady state, on a warm-up pool (churn_warmup:
  4096 frames per push) and on a default pool fed the same (churn_plain: only the steady streams emit)

Latency = host submit of the push -> its frames complete on the device (host sync); `host` is the time until the push
returns (enqueue only).  Before the timed calls, with smoothing off, the frames of the arms that must be equal are
compared with torch.equal: warm_steady, plain and plain_hops (bit for bit the same from hop W - 1 on), and the steady
streams of churn_warmup and churn_plain.  The timed calls run with smoothing on.  Time to first frame: the audio a new
stream must send before its first frame (hop_length * (first emitting hop + 1) samples), plus the p50 latency of the
push that computes it.

    python scripts/pool_warmup_timing.py [--calls 40] [--fps 30 60] [--out profiles/pool_warmup_timing.json]
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
SAMPLE_RATE = 16000


def make_model(dev, fps, precision):
    w = O.make_weights(1234, fps, style="init")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length=256 if fps == 30 else 512).to(dev).eval()
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


class Arm:
    """A pool with n open streams at the given ages (hops pushed since open); each push feeds every stream one hop of
    the arm's own audio sequence (arms built with the same `seed` and ages get the same audio)."""

    def __init__(self, m, n, eg, hops_pool, ages, seed, **pool_kw):
        self.pool = StreamPool(m, n, **pool_kw)
        self.slots = torch.tensor(self.pool.open(eg[:n]), dtype=torch.int32)
        self.n, self.hops_pool, self.seed, self.call = n, hops_pool, seed, 0
        self.ages = np.asarray(ages, dtype=np.int64)
        for r in range(int(self.ages.max())):               # bring every stream to its age
            sel = torch.from_numpy(np.nonzero(self.ages > r)[0])
            self.pool.push(self.slots[sel].contiguous(), self.audio()[sel.to(hops_pool.device)])
        torch.cuda.synchronize()

    def audio(self):
        P = self.hops_pool.shape[0]
        idx = (torch.arange(self.n, device=self.hops_pool.device) * 7 + self.call * 131 + self.seed) % P
        self.call += 1
        return self.hops_pool[idx]

    def push(self):
        return self.pool.push(self.slots, self.audio())


def rows_by_slot(emitted, frames):
    return {s: frames[i] for i, s in enumerate(emitted.tolist())}


def run(arms, equal_groups, calls, m):
    """Verify (smoothing off), then time the arms alternating call by call (smoothing on)."""
    mismatches = 0
    m.use_temporal_smoothing = False
    for _ in range(VERIFY_CALLS):
        out = {k: a.push() for k, a in arms.items()}
        out = {k: (e, f.clone()) for k, (e, f) in out.items()}
        torch.cuda.synchronize()
        for group in equal_groups:
            rows = [rows_by_slot(*out[k]) for k in group]
            common = set.intersection(*(set(r) for r in rows))
            assert common, group
            mismatches += sum(not torch.equal(rows[0][s], r[s]) for r in rows[1:] for s in common)
    m.use_temporal_smoothing = True
    names = list(arms)
    t = {k: [] for k in names}
    t.update({k + "_host": [] for k in names})
    emitted = {}
    for i in range(calls):
        order = names[i % len(names):] + names[:i % len(names)]
        for k in order:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e, _ = arms[k].push()
            t1 = time.perf_counter()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            t[k].append((t2 - t0) * 1e3)
            t[k + "_host"].append((t1 - t0) * 1e3)
            emitted[k] = e.numel()
    res = {k: pct(v) for k, v in t.items()}
    res["frames_per_push"] = emitted
    res["verified_calls"], res["verified_frames_that_differ"] = VERIFY_CALLS, mismatches
    return res


def first_frame(m, eg, hops_pool, **pool_kw):
    """The hop at which a new stream's first frame comes (pushing one hop at a time)."""
    pool = StreamPool(m, 1, **pool_kw)
    s = pool.open(eg[:1])
    for h in range(4 * m.mel_sequence_length):
        e, _ = pool.push(s, hops_pool[h % hops_pool.shape[0]][None])
        if e.numel():
            return h
    raise RuntimeError("no frame")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=40)
    ap.add_argument("--fps", type=int, nargs="+", default=[30], choices=[30, 60])
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"])
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                   "profiles", "pool_warmup_timing.json"))
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    res = {"gpu": gpu_info(), "precision": args.precision, "timed_calls": args.calls,
           "note": "latency = host submit of one push -> device sync, ms; *_host = until the push returns; arms rotated "
                   "call by call; verified with smoothing off, timed with smoothing on"}
    for fps in args.fps:
        m = make_model(dev, fps, args.precision)
        W, hop = m.mel_sequence_length, m.hop_length
        hops_pool = 0.1 * torch.randn(4099, hop, device=dev)
        eg = torch.randn(4096, 264, device=dev)
        rng = np.random.default_rng(fps)
        young = W - 2 - args.calls - VERIFY_CALLS            # the oldest age that stays in warm-up
        r = {"W": W, "hop": hop}
        for n in (4096, 256):
            arms = {"warmup": Arm(m, n, eg, hops_pool, rng.integers(0, young + 1, n), 1, warmup=True),
                    "warm_steady": Arm(m, n, eg, hops_pool, [W] * n, 2, warmup=True),
                    "plain": Arm(m, n, eg, hops_pool, [W] * n, 2),
                    "plain_hops": Arm(m, n, eg, hops_pool, [W] * n, 2, max_hops=2)}
            r[f"{n}_streams"] = run(arms, [("warm_steady", "plain", "plain_hops")], args.calls, m)
            print(fps, n, json.dumps(r[f"{n}_streams"]), flush=True)
            del arms
            torch.cuda.empty_cache()
        ages = np.full(4096, W, dtype=np.int64)
        churn = rng.random(4096) < 1 / 8
        ages[churn] = rng.integers(0, young + 1, int(churn.sum()))
        arms = {"churn_warmup": Arm(m, 4096, eg, hops_pool, ages, 3, warmup=True),
                "churn_plain": Arm(m, 4096, eg, hops_pool, ages, 3)}
        r["churn_4096_streams"] = run(arms, [("churn_warmup", "churn_plain")], args.calls, m)
        r["churn_4096_streams"]["streams_in_warmup"] = int(churn.sum())
        print(fps, "churn", json.dumps(r["churn_4096_streams"]), flush=True)
        del arms
        torch.cuda.empty_cache()
        ttff = {}
        for name, kw, n in (("plain", {}, 4096), ("warmup", {"warmup": True}, 4096)):
            h = first_frame(m, eg, hops_pool, **kw)
            audio_ms = 1e3 * (h + 1) * hop / SAMPLE_RATE
            push_ms = r[f"{n}_streams"][name]["p50"]
            ttff[name] = {"first_frame_hop": h, "audio_ms": round(audio_ms, 1),
                          "audio_plus_p50_push_at_4096_streams_ms": round(audio_ms + push_ms, 2)}
        r["time_to_first_frame"] = ttff
        print(fps, "ttff", json.dumps(ttff), flush=True)
        res[f"{fps}fps"] = r
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
