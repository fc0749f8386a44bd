"""Device and host time of StreamPool.snapshot / StreamPool.restore (one kernel each), bf16 weights, against the only
other way to rebuild a stream's state: opening it afresh and pushing the last W - 1 hops of its audio with push_hops.

  a) 4096 streams at 30 fps (records of 42,408 floats)
  b) 1024 streams at 60 fps (records of 125,028 floats)

Every stream is pushed past W + max_hops hops first, so its rings are full and wrapped.  Three figures per call:

  kernel_ms   the duration of pool_snapshot_kernel / pool_restore_kernel from torch.profiler (CUDA activity), p50 over
              --calls launches after --warm untimed calls of the same shape; bandwidth = 2 * streams * state_floats * 4
              bytes (the record bytes written or read plus as many bytes of pool state read or written) / kernel_ms --
              the kernel figure, against the HBM data-sheet 7.7 TB/s and the project's measured 6,541 GB/s (SURVEY.md 8d);
  call_ms     CUDA events recorded on an idle stream just before the host call and just after it returns: the host path
              before the launch (argument checks, table building), the table upload and the kernel -- what one call
              costs a caller that waits for it;
  host_ms     until the call returns (enqueue only).

The working set (pool state + records, >= 1 GB) is far larger than the 126 MB L2, so every call streams from HBM.  Before
timing, one restored copy of every stream is pushed one more hop beside its original and the frames are compared with
torch.equal.  With two visible GPUs, StreamSnapshot.to("cuda:1") and a restore there are timed too (host clock, synced).

    python scripts/pool_snapshot_timing.py [--calls 50] [--out profiles/pool_snapshot_timing.json]
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
from koemorph_b200.streaming import StreamPool
from oracle import koemorph_oracle as O  # weight generator only

HBM_DATASHEET_GBS = 7700.0
HBM_MEASURED_GBS = 6541.0   # SURVEY.md section 8d
L2_BYTES = 126 * 2 ** 20
MAX_HOPS = 8
REBUILD_MAX_HOPS = 16


def make_model(dev, fps):
    w = O.make_weights(1234, fps, style="init")
    m = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length={30: 256, 60: 512}[fps]).to(dev).eval()
    m.load_state_dict(O.model_state_dict(w), strict=True)
    m.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    m.precision = "bf16"
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
    return {"device": torch.cuda.get_device_name(0), "visible_gpus": torch.cuda.device_count(),
            "nvidia_smi (name, power.limit, clocks.max.sm)": q if q else "unavailable"}


def kernel_ms(fn, name, calls, between=None):
    """durations (ms) of the launches of kernel `name` over `calls` calls of fn, from torch.profiler"""
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            if between:
                between()
            fn()
        torch.cuda.synchronize()
    d = [e.time_range.elapsed_us() / 1e3 for e in prof.events()
         if e.device_type == DeviceType.CUDA and name in e.name]
    assert len(d) == calls, (name, len(d), calls)
    return pct(d)


def timed(fn, calls, warm, between=None):
    """(call ms from CUDA events around the host call on an idle stream, host ms per call) over `calls` calls after
    `warm` untimed ones"""
    dev, host = [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(warm + calls):
        if between:
            between()
        torch.cuda.synchronize()
        e0.record()
        t0 = time.perf_counter()
        fn()
        t1 = time.perf_counter()
        e1.record()
        torch.cuda.synchronize()
        if i >= warm:
            dev.append(e0.elapsed_time(e1))
            host.append((t1 - t0) * 1e3)
    return pct(dev), pct(host)


def scenario(fps, n, calls, warm):
    dev = torch.device("cuda", 0)
    m = make_model(dev, fps)
    hop, W = m.hop_length, m.mel_sequence_length
    g = torch.Generator(device=dev).manual_seed(fps)
    hops_pool = 0.1 * torch.randn(4099, hop, device=dev, generator=g)
    eg = torch.randn(n, 264, device=dev, generator=g)
    a = StreamPool(m, n, max_hops=MAX_HOPS)
    b = StreamPool(m, n, max_hops=MAX_HOPS)
    slots = a.open(eg)
    counts = [MAX_HOPS] * n
    pushed = 0
    while pushed < W + MAX_HOPS:                          # rings full and wrapped
        idx = (torch.arange(n * MAX_HOPS, device=dev) * 7 + pushed * 131) % hops_pool.shape[0]
        a.push_hops(slots, hops_pool[idx], counts)
        pushed += MAX_HOPS
    torch.cuda.synchronize()

    # ---- equality check: one restored copy against its original, one more hop each
    snap = a.snapshot(slots)
    got = b.restore(snap)
    x = hops_pool[torch.arange(n, device=dev) % hops_pool.shape[0]]
    _, fa = a.push(slots, x)
    fa = fa.clone()
    _, fb = b.push(got, x)
    equal = bool(torch.equal(fa, fb))
    for s in got:
        b.close(s)
    torch.cuda.synchronize()

    sf = a.state_floats
    record_bytes = n * sf * 4
    traffic = 2 * record_bytes
    snap_dev, snap_host = timed(lambda: a.snapshot(slots), calls, warm)
    keep = a.snapshot(slots)

    def free_b():
        for s in range(n):
            if s in opened:
                b.close(s)
        opened.clear()
    opened = set()

    def restore():
        opened.update(b.restore(keep))
    rest_dev, rest_host = timed(restore, calls, warm, between=free_b)
    free_b()
    snap_k = kernel_ms(lambda: a.snapshot(slots), "pool_snapshot_kernel", calls)
    rest_k = kernel_ms(restore, "pool_restore_kernel", calls, between=free_b)
    free_b()

    # ---- the alternative: open fresh streams and push the last W - 1 hops of audio (no frame completes)
    c = StreamPool(m, n, max_hops=REBUILD_MAX_HOPS)
    audio = hops_pool[(torch.arange(n * (W - 1), device=dev) * 5) % hops_pool.shape[0]].view(n, W - 1, hop)
    plan = []
    for h0 in range(0, W - 1, REBUILD_MAX_HOPS):
        k = min(REBUILD_MAX_HOPS, W - 1 - h0)
        plan.append((k, audio[:, h0:h0 + k].reshape(-1).contiguous()))
    c_slots = []

    def rebuild():
        c_slots[:] = c.open(eg)
        for k, xs in plan:
            c.push_hops(c_slots, xs, [k] * n)

    def close_c():
        for s in c_slots:
            c.close(s)
        c_slots.clear()
    reb_dev, reb_host = timed(rebuild, max(5, calls // 5), 2, between=close_c)
    close_c()

    def kernel_fig(t):
        gbs = traffic / (t["p50"] * 1e-3) / 1e9
        return {"bytes_per_call": traffic, "achieved_GB_per_s (kernel figure, p50)": round(gbs, 1),
                "fraction_of_datasheet_7.7TBps": round(gbs / HBM_DATASHEET_GBS, 3),
                "fraction_of_measured_6541GBps": round(gbs / HBM_MEASURED_GBS, 3)}

    res = {"fps": fps, "streams": n, "state_floats": sf, "record_bytes_per_stream": sf * 4,
           "records_bytes": record_bytes, "pool_max_hops": MAX_HOPS,
           "working_set_exceeds_L2": 2 * record_bytes > L2_BYTES,
           "restored_copies_push_equal_frames": equal,
           "snapshot_kernel_ms": snap_k, "snapshot_kernel_bandwidth": kernel_fig(snap_k),
           "snapshot_call_ms (host path + table upload + kernel)": snap_dev, "snapshot_host_ms": snap_host,
           "restore_kernel_ms": rest_k, "restore_kernel_bandwidth": kernel_fig(rest_k),
           "restore_call_ms (host path + table upload + kernel)": rest_dev, "restore_host_ms": rest_host,
           f"rebuild_by_push_hops_call_ms (open + {W - 1} hops per stream, max_hops {REBUILD_MAX_HOPS}, "
           f"{len(plan)} calls)": reb_dev,
           "rebuild_by_push_hops_host_ms": reb_host,
           "ratio_p50 (snapshot + restore calls) / rebuild": round((snap_dev["p50"] + rest_dev["p50"]) / reb_dev["p50"], 4)}

    if torch.cuda.device_count() >= 2:
        m1 = make_model(torch.device("cuda", 1), fps)
        d = StreamPool(m1, n, max_hops=MAX_HOPS)
        t_copy, t_rest = [], []
        for _ in range(warm + max(5, calls // 5)):
            torch.cuda.synchronize(0)
            torch.cuda.synchronize(1)
            t0 = time.perf_counter()
            moved = keep.to("cuda:1")
            torch.cuda.synchronize(0)
            torch.cuda.synchronize(1)
            t1 = time.perf_counter()
            with torch.cuda.device(1):
                s1 = d.restore(moved)
                torch.cuda.synchronize(1)
            t2 = time.perf_counter()
            for s in s1:
                d.close(s)
            t_copy.append((t1 - t0) * 1e3)
            t_rest.append((t2 - t1) * 1e3)
        res["to_cuda1_copy_ms (host clock, synced)"] = pct(t_copy[warm:])
        res["restore_on_cuda1_ms (host clock, synced)"] = pct(t_rest[warm:])
        res["to_cuda1_GB_per_s (p50)"] = round(record_bytes / (res["to_cuda1_copy_ms (host clock, synced)"]["p50"] * 1e-3) / 1e9, 1)
    else:
        res["cross_device"] = "not measured: one visible GPU"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--warm", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                   "profiles", "pool_snapshot_timing.json"))
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "precision": "bf16", "timed_calls": args.calls,
           "note": "kernel ms = torch.profiler duration of the one kernel per call; call ms = CUDA events on an idle "
                   "stream from before the host call to after it returns (host path before the launch + table upload + "
                   "kernel); host ms = until the call returns; bandwidth = 2 * record bytes (read + written) / p50 "
                   "kernel ms; p50 after warm-up; the working set exceeds the 126 MB L2 in every scenario, but up to 126 MB of a "
                   "kernel's last writes can still sit in L2 when it ends, so a write-heavy figure may read a few per "
                   "cent above what HBM sustains"}
    for key, fps, n in (("a_30fps_4096_streams", 30, 4096), ("b_60fps_1024_streams", 60, 1024)):
        res[key] = scenario(fps, n, args.calls, args.warm)
        print(key, json.dumps(res[key]), flush=True)
        torch.cuda.empty_cache()
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
