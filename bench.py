#!/usr/bin/env python
"""Benchmark of the hot path: batched audio -> blendshape inference (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision fp32|bf16] [--dump-outputs DIR]

One step = ``SequentialDualStreamModel.forward`` (the public call) over 512 synthetic 8.5 s clips (16 kHz, 30 fps, one
output frame per clip) per GPU.  BASELINE.json quotes configs[1] in "fp32 and bf16": the line's value / dtype are the
bf16-operand tensor-core core (log-mel frontend in fp32 either way), ``other_precision`` carries the all-fp32 path of the
same run.  Prints ONE JSON line (see the task contract): ``value`` is the whole-job audio-seconds per second with inputs
resident in HBM; ``e2e`` is the same metric through the host-buffer API (pinned host audio -> H2D -> kernels -> D2H) next
to the bare host->device copy rate measured in the same run; ``roofline`` describes the dominant kernel (timed in its own
short leg so that the timed region keeps its programmatic dependent launches); ``configs`` holds the other workloads of
BASELINE.json (60 fps, 4096 streams, corpus sweep); ``cpu_baseline`` / ``--impl reference`` time the reference's own CPU
forward (the unmodified modules staged under oracle/_ref) on this box's host cores.
``--dump-outputs DIR`` writes the blendshapes the last timed step returned to ``DIR/blendshapes.npy`` (float32; the inputs
are seeded, so two builds can be compared output for output).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the benchmark may run from a read-only checkout: it writes nothing into the tree, compiled bytecode included
sys.dont_write_bytecode = True

CLIPS_PER_GPU = 512
CLIP_SAMPLES = 136000          # 8.5 s at 16 kHz
CLIP_SECONDS = 8.5
METRIC = "audio-seconds/sec (30fps, 8.5s ctx)"
UNIT = "audio-s/s"
WORKLOAD = "512 x 8.5 s clips @16 kHz per GPU, 30 fps, 256x80 mel context, 1 frame/clip (BASELINE.json configs[1])"
# the same dict in both arms' lines; "l2": how the GPU arm keeps its timed iterations cache-cold
CONFIG = {"workload": WORKLOAD, "clips_per_step_per_gpu": CLIPS_PER_GPU,
          "l2": "inputs 278.5 MB per GPU > 126 MB L2, no flush needed"}


# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on the first
# collective when NCCL_DEBUG asks for it), so the real stdout is set aside at start-up and everything else goes to stderr.
_REAL_STDOUT = None


def _claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


# ----------------------------------------------------------------------------- CPU arm: the reference's own forward
_G = {}


def _cpu_init(clips_per_worker, kind):
    """Per-process set-up (not timed): weights, synthetic clips, one warm-up forward.  kind "reference": the unmodified
    SequentialDualStreamModel of the reference (oracle/_ref or /root/reference); "port": the oracle restatement."""
    import torch
    from oracle import koemorph_oracle as O
    torch.set_num_threads(1)
    w = O.make_weights(1234, 30, style="init")
    audio, eg = O.make_inputs(1000 + os.getpid() % 1000, clips_per_worker, CLIP_SAMPLES, "noise")
    if kind == "reference":
        from oracle import run_reference as R
        model = R.build_reference_model(w, 30, sequential=True)
        model.set_egemaps(eg)
        ta = torch.from_numpy(audio)

        def fwd():
            with torch.no_grad():
                return model(ta)["blendshapes"]
    else:
        def fwd():
            return O.forward_sequence(w, audio, eg)
    fwd()
    _G.update(fwd=fwd)


def _cpu_pass(reps):
    t0 = time.perf_counter()
    for _ in range(reps):
        _G["fwd"]()
    return time.perf_counter() - t0


def _cpu_pool(clips_per_worker, kind):
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    # one single-threaded worker per core: without this every worker's BLAS/OpenMP runtime spawns a thread per core and
    # the oversubscribed pool runs ~50x slower (which would flatter the GPU numbers)
    saved = {k: os.environ.get(k) for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS")}
    os.environ.update({k: "1" for k in saved})
    try:
        pool = mp.get_context("spawn").Pool(cores, initializer=_cpu_init, initargs=(clips_per_worker, kind))
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    pool.map(_cpu_pass, [0] * cores, chunksize=1)  # make sure every worker is up
    return pool, cores


def _cpu_kind():
    from oracle import run_reference as R
    return "reference" if R.reference_available() else "port"


def _cpu_note(kind):
    from oracle import run_reference as R
    if kind == "reference":
        return (f"the reference's unmodified SequentialDualStreamModel.forward ({R.reference_kind()} copy: {R.REFERENCE_ROOT}), "
                "one single-threaded process per host core, clips split over the processes; librosa / opensmile are absent "
                "from the image, so its librosa calls run the numpy restatement in oracle/koemorph_oracle.py and the eGeMAPS "
                "extraction is replaced by the synthetic 264-D input (excluded on both sides)")
    return ("oracle.forward_sequence (port of the reference forward, per-clip Python loop, one single-threaded process per "
            "core); eGeMAPS extraction excluded (synthetic input); mel stage is the librosa restatement, not librosa")


def _pool_throughput(kind, target_seconds, clips_per_worker=4):
    pool, cores = _cpu_pool(clips_per_worker, kind)
    with pool:
        t_probe = max(pool.map(_cpu_pass, [1] * cores, chunksize=1))
        reps = max(1, int(target_seconds / max(t_probe, 1e-3)))
        t0 = time.perf_counter()
        pool.map(_cpu_pass, [reps] * cores, chunksize=1)
        wall = time.perf_counter() - t0
    n = cores * clips_per_worker * reps
    return n * CLIP_SECONDS / wall, cores, f"{n} clips of 8.5 s ({cores} processes x {clips_per_worker} clips x {reps} passes, {wall:.1f} s wall)"


def _reference_single_process():
    """BASELINE.md section 4: config C1 (B = 1, median of >= 20 runs, all host threads for torch), B = 32, and the mel vs
    attention split -- the reference as a user runs it, one process."""
    import torch
    from oracle import koemorph_oracle as O
    from oracle import run_reference as R
    if not R.reference_available():
        return None
    res = {"torch_threads": os.cpu_count()}
    torch.set_num_threads(os.cpu_count() or 1)
    w = O.make_weights(1234, 30, style="init")
    model = R.build_reference_model(w, 30, sequential=True)

    def timed(B, runs):
        audio, eg = O.make_inputs(5678, B, CLIP_SAMPLES, "noise")
        model.set_egemaps(eg)
        ta = torch.from_numpy(audio)
        with torch.no_grad():
            for _ in range(3):
                model(ta)
            ts = []
            for _ in range(runs):
                t0 = time.perf_counter()
                model(ta)
                ts.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            for _ in range(5):
                model.extract_mel_features(ta)
            mel = (time.perf_counter() - t0) / 5
        med = statistics.median(ts)
        return {"B": B, "runs": runs, "median_ms": med * 1e3, "audio_s_per_s": B * CLIP_SECONDS / med,
                "mel_share": min(1.0, mel / med)}

    res["c1_B1"] = timed(1, 20)
    res["B32"] = timed(32, 5)
    # the same with one torch thread: on a box whose cores are busy / virtual, torch's own thread pool can be the slower one
    torch.set_num_threads(1)
    res["c1_B1_one_thread"] = timed(1, 20)
    return res


def cpu_baseline(target_seconds=10.0):
    kind = _cpu_kind()
    value, cores, sample = _pool_throughput(kind, target_seconds)
    out = {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample + " through " + _cpu_note(kind)}
    if kind == "reference":
        port_value, _, port_sample = _pool_throughput("port", 4.0)
        out["port"] = {"value": port_value, "unit": UNIT, "sample": port_sample + " through " + _cpu_note("port")}
        out["single_process"] = _reference_single_process()
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    kind = _cpu_kind()
    clips_per_worker = 4
    pool, cores = _cpu_pool(clips_per_worker, kind)
    # one step = the GPU arm's step: every worker forwards its 4 clips `reps` times, ~512 clips in all
    reps = max(1, -(-CLIPS_PER_GPU // (cores * clips_per_worker)))
    times = []
    with pool:
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            pool.map(_cpu_pass, [reps] * cores, chunksize=1)
            if i >= args.warmup:
                times.append(time.perf_counter() - t0)
    n = cores * clips_per_worker * reps
    step = sum(times) / len(times)
    value = n * CLIP_SECONDS / step
    sample = f"{n} clips of 8.5 s per step ({cores} processes x {clips_per_worker} clips x {reps} passes) through " + _cpu_note(kind)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": dict(CONFIG),
            "details": {"step_sample": f"{n} clips per step"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if kind == "reference":
        line["cpu_baseline"]["single_process"] = _reference_single_process()
    emit(line)


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._go = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _loop(self):
        nv = self._nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        # Samples are taken INSIDE the timed region but only once the host has queued all of its steps (release()): an NVML
        # query holds a driver lock for a millisecond or two, and a kernel launch of the main thread that waits for it
        # drains the GPU's queue -- 8 us per step of a 20-step region with the sampler polling from the start, 5 us when
        # it started a millisecond in.  The GPU is still working through the queued steps (the host submits a step in
        # ~75 us, the GPU runs it in ~200 us) while the clocks and throttle reasons are read.
        self._go.wait()
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                break
            time.sleep(0.001)

    def start(self):
        if self._nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def release(self):
        self._go.set()

    def stop(self):
        self._stop.set()
        self._go.set()
        if self._thread is not None:
            self._thread.join()
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ----------------------------------------------------------------------------- GPU arm
def dump_outputs(directory, arrays):
    """Write each tensor of ``arrays`` to ``directory/<name>.npy`` as float32."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), t.float().cpu().numpy())


def _make_model(K, O, torch, dev, fps, precision):
    w = O.make_weights(1234, fps, style="init")
    model = K.SequentialDualStreamModel(target_fps=fps, mel_sequence_length=256 if fps == 30 else 512).to(dev).eval()
    model.load_state_dict(O.model_state_dict(w), strict=True)
    model.set_compression_layer(torch.from_numpy(w["compression.weight"]), torch.from_numpy(w["compression.bias"]))
    model.precision = precision
    return model


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import koemorph_b200 as K
    from koemorph_b200 import _lib
    from koemorph_b200.infer import HostPipeline, bind_host_thread_to_gpu_node
    from oracle import koemorph_oracle as O  # weights generator + cpu_baseline only (never on the timed path)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: koemorph_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_node = bind_host_thread_to_gpu_node(local) if world > 1 else None   # before any pinned allocation
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()
    torch.set_grad_enabled(False)

    model = _make_model(K, O, torch, dev, 30, args.precision)
    B, K_steps = CLIPS_PER_GPU, args.steps

    def inputs_of(r):
        g = torch.Generator(device=dev).manual_seed(5678 + r)
        a = 0.1 * torch.randn(B, CLIP_SAMPLES, device=dev, generator=g)       # 278.5 MB > 126 MB L2
        return a, torch.randn(B, 264, device=dev, generator=g)

    audio, eg = inputs_of(rank)
    # every step's frames land directly in their slot of the buffer that is gathered at the end (forward's `out=`)
    kept = torch.empty(K_steps, B, 1, 52, device=dev)
    gathered = torch.empty(world * K_steps, B, 1, 52, device=dev) if world > 1 else None
    tiny = torch.zeros(1, device=dev)

    def step(i):
        return model(audio, egemaps=eg, out=kept[i % K_steps])["blendshapes"]

    def gather_all():
        # the path's only collective (north_star: "NCCL over NVLink used only for the final output gather"): every
        # rank's results of all the steps, once, inside the timed region
        if world > 1:
            dist.all_gather_into_tensor(gathered, kept)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def device_gate():
        # after the host barrier the ranks' streams still start up to a few hundred microseconds apart (host skew), which
        # the closing collective turns into waiting time of the early ranks.  A tiny all-reduce on the compute stream is a
        # device-side rendezvous: every rank's start event is recorded right behind it.
        if world > 1:
            dist.all_reduce(tiny)

    sampler = ClockSampler(local)   # (NVML initialisation takes tens of milliseconds: before the warm-up, not between it
    #                                  and the timed region, where it would leave the GPU idle right before the first step)
    for i in range(max(args.warmup, 3)):
        step(i)
    gather_all()  # warm-up covers the collective too (first use sets up NCCL's channels for this size)
    device_gate()
    # The ranks reach the first barrier milliseconds apart (process start-up, first-use initialisation), and a GPU that
    # idles that long answers its next kernels slowly: with one barrier the first timed step of a multi-GPU run took
    # 406 us instead of 260 us and the next four were still 2-5 % slow (scripts/multi_gpu_step_profile.py).  So the ranks
    # meet once, run three more untimed steps -- now aligned -- and meet again: that second barrier, the one that brackets
    # the timed region, is then a matter of microseconds.
    barrier()
    for i in range(3):
        step(i)
    _lib.reset_launch_count()
    barrier()
    sampler.start()
    t0, t1, g0 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    device_gate()
    h0 = time.perf_counter()
    t0.record()
    for i in range(K_steps):
        step(i)
    host_submit_ms = (time.perf_counter() - h0) * 1e3
    sampler.release()
    g0.record()
    gather_all()
    t1.record()
    barrier()
    clocks = sampler.stop()
    launches = _lib.launch_count()
    # what the timed path handed its caller in the last step (every rank's block, as gathered), set aside before the legs
    # below write into `kept` again
    last_step = None
    if args.dump_outputs:
        last_step = (gathered.view(world, K_steps, B, 1, 52)[:, -1] if world > 1 else kept[-1]).reshape(-1, 1, 52).clone()
    mine_ms, gather_ms = t0.elapsed_time(t1), g0.elapsed_time(t1)
    per_rank = torch.tensor([mine_ms, gather_ms, host_submit_ms], device=dev)
    all_ranks = per_rank.clone().unsqueeze(0)
    if world > 1:
        all_ranks = torch.empty(world, 3, device=dev)
        dist.all_gather_into_tensor(all_ranks, per_rank)
    all_ranks = all_ranks.cpu()
    elapsed_ms = float(all_ranks[:, 0].max())
    value = world * B * CLIP_SECONDS * K_steps / (elapsed_ms * 1e-3)
    rank_stats = {"elapsed_ms": {"min": float(all_ranks[:, 0].min()), "median": float(all_ranks[:, 0].median()),
                                 "max": elapsed_ms},
                  "gather_ms": {"min": float(all_ranks[:, 1].min()), "median": float(all_ranks[:, 1].median()),
                                "max": float(all_ranks[:, 1].max())},
                  "host_submit_ms_per_step_max": float(all_ranks[:, 2].max()) / K_steps}

    # ---- outside the timed region: the gathered block of rank r is rank r's result, and equals a 1-rank run of r's clips ----
    gather_check = None
    if world > 1:
        blocks = gathered.view(world, K_steps, B, 1, 52)
        for r in range(world):
            theirs = kept.clone()
            dist.broadcast(theirs, src=r)
            assert torch.equal(blocks[r], theirs), f"gathered block {r} differs from rank {r}'s local result"
        if rank == 0:
            a_r, e_r = inputs_of(world - 1)
            alone = model(a_r, egemaps=e_r)["blendshapes"]
            assert torch.equal(blocks[world - 1][0], alone), "N-rank result differs from the 1-rank run of the same clips"
            del a_r, e_r
        gather_check = f"all {world} gathered blocks equal their ranks' local results; rank {world - 1}'s block equals a " \
                       "single-GPU forward of the same clips on rank 0 (bitwise)"
        barrier()

    # ---- the same K steps captured once in a CUDA graph and replayed (no host work between the launches) ----
    graph_leg = None
    try:
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            step(0)
        torch.cuda.current_stream(dev).wait_stream(side)
        want = kept.clone()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(K_steps):
                step(i)
        graph.replay()
        barrier()
        assert torch.equal(kept, want), "graph replay of forward() differs from the eager steps"
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        device_gate()
        q0.record()
        graph.replay()
        q1.record()
        barrier()
        tq = torch.tensor([q0.elapsed_time(q1)], device=dev)
        if world > 1:
            dist.all_reduce(tq, op=dist.ReduceOp.MAX)
        graph_leg = {"ms_per_step": float(tq.item()) / K_steps, "unit": UNIT,
                     "value": world * B * CLIP_SECONDS * K_steps / (float(tq.item()) * 1e-3),
                     "note": f"the {K_steps} forward() calls of the timed region captured in one CUDA graph and replayed "
                             "(bitwise the same results; no gather inside); the headline value above is the eager loop"}
        del graph, want
    except Exception as e:  # capture is an extra: the contract line does not depend on it
        graph_leg = {"error": f"{type(e).__name__}: {e}"[:300]}
        torch.cuda.synchronize()

    # ---- roofline leg: the dominant kernel (log-mel power) alone, one event pair per launch ----
    fe = model._frontend(dev)
    n_frames = model.window_frames + 1
    pw = fe.power(audio, model.hop_length, n_frames)
    for _ in range(3):
        fe.power(audio, model.hop_length, n_frames, out=pw)
    torch.cuda.synchronize()
    pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(20)]
    for e0, e1 in pairs:
        e0.record()
        fe.power(audio, model.hop_length, n_frames, out=pw)
        e1.record()
    torch.cuda.synchronize()
    k1_ms = statistics.mean(a.elapsed_time(b) for a, b in pairs)
    del pw

    # ---- the other precision of BASELINE.json configs[1] ("fp32 and bf16"), same workload, device-resident ----
    other = None
    if not args.no_other_precision:
        other_name = "bf16" if args.precision == "fp32" else "fp32"
        model.precision = other_name
        for i in range(3):
            step(i)
        barrier()
        o0, o1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_other = max(3, min(K_steps, 20))
        o0.record()
        for i in range(n_other):
            step(i)
        o1.record()
        barrier()
        to = torch.tensor([o0.elapsed_time(o1)], device=dev)
        if world > 1:
            dist.all_reduce(to, op=dist.ReduceOp.MAX)
        other = {"precision": other_name, "value": world * B * CLIP_SECONDS * n_other / (float(to.item()) * 1e-3),
                 "unit": UNIT, "ms_per_step": float(to.item()) / n_other, "steps": n_other}
        model.precision = args.precision

    # ---- end to end through the host-buffer API (pinned host -> H2D -> kernels -> D2H) ----
    e2e = None
    if not args.no_e2e:
        pipe = HostPipeline(model, chunk_clips=64)
        audio_h = torch.empty(B, CLIP_SAMPLES, dtype=torch.float32, pin_memory=True)
        audio_h.copy_(audio)
        eg_h = torch.empty(B, 264, dtype=torch.float32, pin_memory=True)
        eg_h.copy_(eg)
        out_h = torch.empty(B, 1, 52, dtype=torch.float32, pin_memory=True)
        e2e_steps = max(3, min(K_steps, 20))

        def time_region(fn):
            barrier()
            ts = time.perf_counter()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(e2e_steps):
                fn()
            e1.record()
            barrier()
            ms = max(e0.elapsed_time(e1), (time.perf_counter() - ts) * 1e3)
            te = torch.tensor([ms], device=dev)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return float(te.item()) / e2e_steps

        for _ in range(2):
            pipe(audio_h, eg_h, out_h)
        expect = step(0).clone()
        barrier()
        assert torch.allclose(out_h, expect.cpu(), atol=1e-7), "host pipeline diverges from the device path"
        e2e_ms = time_region(lambda: pipe(audio_h, eg_h, out_h))

        # the ceiling of that leg: the same chunks copied host -> device (one cudaMemcpyAsync per 64-clip chunk on the
        # pipeline's two streams) with no kernels at all
        def bare_copy():
            cur = torch.cuda.current_stream(dev)
            for s in pipe._streams:
                s.wait_stream(cur)
            for ci, c0 in enumerate(range(0, B, pipe.chunk)):
                n = min(pipe.chunk, B - c0)
                a_dev, e_dev = pipe._buffers(ci & 1, n, CLIP_SAMPLES)
                with torch.cuda.stream(pipe._streams[ci & 1]):
                    a_dev.copy_(audio_h[c0:c0 + n], non_blocking=True)
                    e_dev.copy_(eg_h[c0:c0 + n], non_blocking=True)
            for s in pipe._streams:
                cur.wait_stream(s)
            cur.synchronize()

        bare_copy()
        h2d_ms = time_region(bare_copy)
        h2d_bytes = B * (CLIP_SAMPLES + 264) * 4

        # the same clips handed over as 16-bit PCM (the samples' format in a WAV file): half the PCIe bytes.  Reported
        # beside the float32 number, not instead of it; checked against the float path fed the same quantised samples.
        pcm_h = torch.empty(B, CLIP_SAMPLES, dtype=torch.int16, pin_memory=True)
        pcm_h.copy_((audio.clamp(-1.0, 32767.0 / 32768.0) * 32768.0).round().to(torch.int16))
        audio_h.copy_(pcm_h.to(torch.float32) / 32768.0)
        pipe(audio_h, eg_h, out_h)
        want = out_h.clone()
        for _ in range(2):
            pipe(pcm_h, eg_h, out_h)
        barrier()
        assert torch.equal(out_h, want), "PCM16 host path differs from the float path on the same samples"
        pcm_ms = time_region(lambda: pipe(pcm_h, eg_h, out_h))
        per_s = lambda ms: world * B * CLIP_SECONDS / (ms * 1e-3)
        e2e = {"value": per_s(e2e_ms), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": B * 52 * 4,
               "steps": e2e_steps, "ms_per_step": e2e_ms,
               "api": "koemorph_b200.infer.HostPipeline (pinned host tensors, 64-clip chunks, 2 streams)",
               "h2d_ceiling": {"gbytes_per_s_per_gpu": h2d_bytes / (h2d_ms * 1e-3) / 1e9, "ms_per_step": h2d_ms,
                               "value": per_s(h2d_ms), "unit": UNIT,
                               "how": "the same pinned chunks copied host -> device with no kernels, same streams, same run "
                                      "(max over ranks)"},
               "frac_of_h2d_ceiling": h2d_ms / e2e_ms,
               "host_numa_node_rank0": numa_node,
               "pcm16_input": {"value": per_s(pcm_ms), "unit": UNIT, "h2d_bytes_per_step": B * (CLIP_SAMPLES * 2 + 264 * 4),
                               "note": "same API, audio handed over as int16 PCM and converted on the device "
                                       "(bit-identical results); the headline e2e above is float32 host audio"}}
        del audio_h, pcm_h

    # ---- the other workloads of BASELINE.json (short legs; not the headline) ----
    configs = None
    if not args.no_configs:
        configs = other_configs(args, torch, dist, K, O, dev, rank, world, barrier)

    if rank == 0:
        peaks, peak_src = None, "fallback"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
            peak_src = "measured"
        except Exception:
            pass
        hbm_peak = float(peaks["hbm_gbs"]) if peaks else 6650.0
        # algorithmic bytes of one step's frontend launch (SURVEY.md section 8(d)): audio + eGeMAPS read, 52 floats written,
        # per clip -- the mel rows the kernel materialises between itself and the core are NOT counted
        k1_bytes = B * (CLIP_SAMPLES * 4 + 264 * 4 + 52 * 4)
        achieved = k1_bytes / (k1_ms * 1e-3) / 1e9
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
                traffic = json.load(f).get("logmel_power_kernel_dram_bytes_per_launch")
        except Exception:
            pass
        ms_per_step = elapsed_ms / K_steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K_steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "bf16": "bf16"}[args.precision],
            "data": "synthetic",
            # (the same dict as the reference arm's, so that the two lines compare as the same configuration)
            "config": dict(CONFIG),
            "details": {"parallelism": f"clip-shard x{world}", "precision": args.precision,
                        "timed_call": "SequentialDualStreamModel.forward(audio, egemaps=, out=)",
                        "collective": f"one all_gather of the ({K_steps},B,1,52) results at the end of the timed region; "
                                      "start events behind a device-side rendezvous (tiny all-reduce)" if world > 1 else "none",
                        },
            "clocks": clocks,
            "ranks": rank_stats,
            "e2e": e2e if e2e is not None else {"value": None, "unit": UNIT},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "logmel_power_ws_kernel", "bound": "hbm", "achieved": achieved, "peak": hbm_peak,
                         "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                         "peak_source": peak_src, "kernel_ms": k1_ms, "share_of_step": k1_ms / ms_per_step,
                         "algorithmic_bytes_per_launch": k1_bytes,
                         "how": "mean of 20 launches, one CUDA-event pair each, in a leg of their own after the timed region "
                                "(inputs 278.5 MB > L2); bytes = SURVEY section 8(d) per-clip figure x 512",
                         "whole_step_frac_of_hbm": k1_bytes / (ms_per_step * 1e-3) / 1e9 / hbm_peak},
        }
        if graph_leg is not None:
            line["cuda_graph"] = graph_leg
        if gather_check is not None:
            line["gather_check"] = gather_check
        if other is not None:
            line["other_precision"] = other
        if configs is not None:
            line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        if last_step is not None:
            dump_outputs(args.dump_outputs, {"blendshapes": last_step})
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def other_configs(args, torch, dist, K, O, dev, rank, world, barrier):
    """BASELINE.json configs[2] (60 fps), [3] (4096 streams) on rank 0's GPU and [4] (corpus sweep) over all ranks: short
    device-timed legs, reported under `configs` (scripts/bench_configs.py runs them at full length)."""
    from koemorph_b200.parallel import gather_outputs, shard_range
    from koemorph_b200.streaming import StreamingEngine
    res = {}

    def timed(fn, steps, warmup=3):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    B = CLIPS_PER_GPU
    if rank == 0:
        # c3: 60 fps (hop 266, 512-frame window, K = 515), 512 clips, one frame per clip
        m60 = _make_model(K, O, torch, dev, 60, args.precision)
        audio = 0.1 * torch.randn(B, CLIP_SAMPLES, device=dev)
        eg = torch.randn(B, 264, device=dev)
        ms = timed(lambda: m60(audio, egemaps=eg), 10)
        res["c3_60fps"] = {"workload": "512 x 8.5 s clips, 60 fps (hop 266, 512-frame window, K = 515), 1 frame/clip",
                           "precision": args.precision, "ms_per_step": ms, "value": B * CLIP_SECONDS / (ms * 1e-3), "unit": UNIT}
        del m60, audio, eg
        # c4: 4096 concurrent streams, stride one hop, 8.5 s context; per-hop latency host submit -> outputs complete
        m30 = _make_model(K, O, torch, dev, 30, args.precision)
        for S in (4096, 256):
            eng = StreamingEngine(m30, S)
            eng.set_egemaps(torch.randn(S, 264, device=dev))
            hops = [0.1 * torch.randn(S, m30.hop_length, device=dev) for _ in range(4)]
            for i in range(m30.mel_sequence_length + 8):
                eng.step(hops[i & 3])
            torch.cuda.synchronize()
            lat = []
            for i in range(200):
                t0 = time.perf_counter()
                out = eng.step(hops[i & 3])
                torch.cuda.synchronize()
                lat.append((time.perf_counter() - t0) * 1e3)
                assert out is not None
            lat.sort()
            res[f"c4_streams_{S}"] = {"workload": f"{S} concurrent streams, one 533-sample hop per stream per step, 8.5 s context",
                                      "precision": args.precision, "latency_ms": {"p50": lat[100], "p99": lat[197], "max": lat[-1]},
                                      "steps": 200, "real_time_factor_p99": (m30.hop_length / 16000.0 * 1e3) / lat[197],
                                      "driver": "koe_stream_push (one native call per hop)"}
            del eng, hops
        del m30
    # c5: corpus sweep sharded by clip over the ranks, one gather at the end (a bounded 100k-clip sample of the 1M corpus)
    N = 102400 * world if world > 1 else 102400
    model = _make_model(K, O, torch, dev, 30, args.precision)
    lo, hi = shard_range(N, rank, world)
    pool = [(0.1 * torch.randn(B, CLIP_SAMPLES, device=dev), torch.randn(B, 264, device=dev)) for _ in range(2)]
    out = torch.empty(hi - lo, 1, 52, device=dev)

    def sweep():
        for i, c0 in enumerate(range(0, hi - lo, B)):
            n = min(B, hi - lo - c0)
            a, e = pool[i & 1]
            model(a[:n], egemaps=e[:n], out=out[c0:c0 + n])
        return gather_outputs(out, N) if world > 1 else out

    sweep()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    full = sweep()
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    assert full.shape[0] == N
    res["c5_corpus"] = {"workload": f"{N} synthetic 8.5 s clips sharded by clip over {world} GPU(s), 512-clip batches, one "
                                    "all_gather of (N,1,52) at the end (bounded sample of the 1M-clip sweep: weak scaling, "
                                    "102,400 clips per GPU)",
                        "precision": args.precision, "seconds": float(t.item()) * 1e-3,
                        "value": N * CLIP_SECONDS / (float(t.item()) * 1e-3), "unit": UNIT}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="koemorph_b200", choices=["koemorph_b200", "reference"])
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"],
                    help="core kernel: bf16 = tcgen05 tensor path (bf16 operands, fp32 accumulation; default), fp32 = CUDA-core FMA; "
                         "the other one is timed too and reported under other_precision")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--no-other-precision", action="store_true", help="skip the secondary (bf16 / fp32) leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the 60 fps / streaming / corpus legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the blendshapes of the last timed step to DIR/blendshapes.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "koemorph_b200":
        ap.error("--dump-outputs applies to the koemorph_b200 path")
    _claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
