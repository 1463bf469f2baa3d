#!/usr/bin/env python
"""Benchmark of the B200 MWF beamforming hot path (BASELINE.json metric: beamformed frames/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|...]
                    [--shard utterances|nodes] [--masks oracle|crnn] [--dump-outputs DIR]

One "step" = one pass of the whole two-step Tango path (STFT -> masked SCM -> per-bin GEVD-MWF
-> filter-and-sum, twice) over one batch of synthetic utterances, in DEPLOYMENT mode: the mixture y
and the two masks are the inputs, yf / z / zn the outputs (no clean components, no diagnostics) --
the same work in the GPU arm and in the CPU arm.  Default workload = BASELINE configs[1]: 1 node x
4 mics, batch = 64 x 10 s @ 16 kHz per GPU, 512-pt STFT, device-resident masks.  Frame unit
(SURVEY.md 8d): one STFT frame of one node's beamformed output, so a step produces B*K*T frames per
GPU.  N > 1: utterances shard over ranks, no data-path collective (weak scaling); --shard nodes
instead gives every rank K/N nodes of every utterance and exchanges the compressed signals z with
one NCCL all-gather per batch chunk (reference tango.py:379-386), overlapped with step 1 of the next
chunk.  Timing = max over ranks of CUDA-event time between barriers.

The JSON line also carries
  roofline      the dominant kernel of the step (algorithmic bytes / CUDA-event time vs the measured
                HBM peak) and, under "kernels", the same for EVERY kernel of the step
  e2e           the same metric through the public API with pinned HOST buffers (H2D of signals and
                masks, D2H of the beamformed STFT inside the timed region); --masks crnn: only the
                signals cross PCIe (int16 PCM), the masks come from the reference's CRNN on device
  cpu_baseline  the oracle port of the reference (oracle/tango_np.py, per-frame np.outer loops
                like tango.py:357-374) on the host cores, bounded sample
--impl reference times only that CPU path (the reference is pure Python/NumPy and cannot travel to
the GPU box; its restatement is pinned to the reference's outputs by tests/test_oracle.py).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (B per GPU, K nodes, C mics, L samples, n_fft, description)
    "cfg1": (1, 1, 2, 64000, 512, "1 node x 2 mics, 4 s, 512-pt STFT (BASELINE configs[0])"),
    "cfg2": (64, 1, 4, 160000, 512, "1 node x 4 mics, batch=64 x 10 s per GPU, 512-pt STFT, DNN mask (BASELINE configs[1])"),
    "cfg3": (64, 4, 4, 160000, 512, "4 nodes x 4 mics, batch=64 x 10 s per GPU (BASELINE configs[2] shape)"),
    "cfg5": (64, 8, 2, 160000, 512, "8 nodes x 2 mics, batch=64 x 10 s per GPU (BASELINE configs[4] shape)"),
    "cfg4_256": (128, 1, 8, 160000, 256, "8 mics, 256-pt STFT, batch=128 x 10 s per GPU (BASELINE configs[3] sweep point)"),
    "cfg4_512": (128, 1, 8, 160000, 512, "8 mics, 512-pt STFT, batch=128 x 10 s per GPU (BASELINE configs[3] sweep point)"),
    "cfg4_1024": (128, 1, 8, 160000, 1024, "8 mics, 1024-pt STFT, batch=128 x 10 s per GPU (BASELINE configs[3] sweep point)"),
}
METRIC = "beamformed frames/sec (16kHz, 512-pt STFT)"
DUMP_BUDGET = 48 << 20       # bytes written by --dump-outputs, all arrays together


def dump_outputs(out_dir, arrays, budget=DUMP_BUDGET, seed=0):
    """Write every output tensor as out_dir/<name>.npy in float32; complex tensors gain a trailing (re, im) axis.
    When the arrays together exceed `budget` bytes, each one is replaced by the same fixed, seeded sample of its
    flattened elements (a share of the budget proportional to its size), so that two runs or two builds can be
    compared element for element."""
    import torch
    nbytes = lambda t: t.numel() * (8 if t.is_complex() else 4)
    total = sum(nbytes(t) for t in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if total > budget:
            n = max(1, nbytes(t) * budget // total // (8 if t.is_complex() else 4))
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(seed))[:n].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = torch.view_as_real(t) if t.is_complex() else t
        np.save(os.path.join(out_dir, name + ".npy"), a.to(torch.float32).cpu().numpy())


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference in deployment mode (masks given), bounded sample,
# one utterance per host process (exp/ex1/loop_tango.sh launches one process per utterance)
# ----------------------------------------------------------------------------------------------
def _cpu_one(args):
    seed, K, C, L, n_fft, gran = args
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    from disco_b200.synth import make_utterance
    from oracle import librosa_np, tango_np
    y, s, n = make_utterance(seed, K, C, L)
    hop = n_fft // 2
    # masks are an INPUT of the timed path (they come from the DNN in deployment): computed outside the clock
    S = [librosa_np.stft(s[k, 0], n_fft, hop) for k in range(K)]
    N = [librosa_np.stft(n[k, 0], n_fft, hop) for k in range(K)]
    mz = [tango_np.tf_mask(S[k], N[k], "irm1") for k in range(K)]
    mw = [tango_np.tf_mask(S[k], N[k], "irm2") for k in range(K)]
    t0 = time.perf_counter()
    tango_np.offline_tango(list(y), None, None, masks=(mz, mw), n_fft=n_fft, n_hop=hop, granularity=gran)
    return time.perf_counter() - t0


def _cpu_warm(_):
    import scipy.linalg  # noqa: F401
    from oracle import tango_np  # noqa: F401
    time.sleep(0.2)
    return 0


def usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota, capped at 64
    workers so the bounded sample stays bounded."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, min(n, 64))


class CpuArm:
    """Pool of host processes (started and warmed once); sample() times one bounded sample."""

    def __init__(self, K, C, L, n_fft, procs=None):
        import multiprocessing as mp
        self.K, self.C, self.L, self.n_fft = K, C, L, n_fft
        self.cores = procs or usable_cores()
        os.environ["OMP_NUM_THREADS"] = "1"          # inherited by the workers: one thread per process
        os.environ["OPENBLAS_NUM_THREADS"] = "1"
        os.environ["MKL_NUM_THREADS"] = "1"
        self.pool = mp.get_context("spawn").Pool(self.cores)
        self.pool.map(_cpu_warm, range(self.cores), chunksize=1)      # interpreter + NumPy/SciPy imports: untimed
        self.seed = 1000

    def sample(self, budget_s, granularity="frame"):
        K, C, L, n_fft = self.K, self.C, self.L, self.n_fft
        # bound the sample: shorten the utterance so one of them takes <~ budget (the reference runs ~120 frames/s/core)
        est_rate = 150.0 if granularity == "frame" else 20000.0
        max_frames = max(64, int(budget_s * est_rate / K))
        Ls = min(L, (max_frames - 1) * (n_fft // 2))
        Ts = 1 + Ls // (n_fft // 2)
        jobs = [(self.seed + i, K, C, Ls, n_fft, granularity) for i in range(self.cores)]
        self.seed += self.cores
        t0 = time.perf_counter()
        self.pool.map(_cpu_one, jobs, chunksize=1)
        wall = time.perf_counter() - t0
        return {"value": self.cores * K * Ts / wall, "unit": "frames/s", "cores": self.cores, "kind": "port",
                "sample": "%d utterances (one per process) x %d node(s) x %d mics x %.2f s (%d frames), oracle/tango_np.py "
                          "deployment mode (masks given; yf, z, zn), granularity=%s, workers pre-started"
                          % (self.cores, K, C, Ls / 16000.0, Ts, granularity),
                "seconds": wall, "frames": self.cores * K * Ts}

    def close(self):
        self.pool.close()
        self.pool.join()


# ----------------------------------------------------------------------------------------------
def _nvml_handle(gpu_index):
    import pynvml as nv
    nv.nvmlInit()
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
    return nv, nv.nvmlDeviceGetHandleByIndex(phys)


def bind_host_to_gpu(gpu_index):
    """Multi-GPU runs: keep this rank's host threads -- and therefore the first touch of its pinned staging
    buffers -- on the CPUs of the GPU's NUMA node (NVML's affinity mask).  Round 2 measured the host-to-host leg at
    31 M frames/s on 8 GPUs against 8 x 8.2 M alone with unbound ranks (4 of the 8 GPUs hang off the other socket).
    Any failure (no NVML, restricted cpuset) leaves the process as it was.  Returns the CPU count bound to, or None."""
    try:
        nv, h = _nvml_handle(gpu_index)
        allowed = os.sched_getaffinity(0)
        words = nv.nvmlDeviceGetCpuAffinity(h, max(allowed) // 64 + 1)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1} & allowed
        if cpus and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def clock_sampler(stop, out, gpu_index):
    """Sample SM clock and throttle reasons through NVML every ~2 ms while the timed region runs."""
    try:
        nv, h = _nvml_handle(gpu_index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not stop.is_set():
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            out.append([str(sm), str(mx)] + ["Active" if r & bits[k] else "Not Active" for k in
                                             ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")])
            stop.wait(0.002)
        return
    except Exception:
        pass
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    while not stop.is_set():
        try:
            r = subprocess.run(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=5)
            parts = [p.strip() for p in r.stdout.strip().split(",")]
            if len(parts) >= 6:
                out.append(parts)
        except Exception:
            pass
        stop.wait(0.1)


def summarize_clocks(samples):
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    sm = sorted(float(s[0]) for s in samples)
    reasons = []
    for i, nm in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
        if any(s[2 + i].lower().startswith("active") for s in samples):
            reasons.append(nm)
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(samples[0][1]), "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# Per-kernel accounting: algorithmic bytes of every op of the step (DESIGN.md section 4), from the
# shapes of the tensors it is called with
# ----------------------------------------------------------------------------------------------
def _op_models(n_fft):
    F = n_fft // 2 + 1

    def dims(Y):
        C, T = Y.shape[-3], Y.shape[-2]
        return Y.numel() // (C * T * F), C, T          # groups, channels, frames

    def stft_scm(a, k, nm):
        x = a[0]
        G, C, L = x.shape
        T = 1 + L // (n_fft // 2)
        keep = k.get("keep_partials", False) or nm == 2
        return ("stft_scm_kernel<%d,%d,%d>" % (n_fft, C, nm),
                G * (4 * C * L + nm * 4 * F * T + 8 * C * F * T + nm * 16 * F * C * C), 1 if keep else 2)

    def solve(n_mat, D):
        return n_mat * (16 * D * D + 16 * D)

    def filter_sum(a, k):
        W, Y = a[0], a[1]
        Z = a[2] if len(a) > 2 else k.get("Z")
        G, C, T = dims(Y)
        D = W.shape[-1]
        resid = k.get("ref") is not None
        if Z is not None and k.get("out_layout", "TF") in ("TF", 0) and k.get("node_sel") is None:
            Kn = Z.shape[1]   # all-nodes pass: Y and every z read once
            return ("filter_sum_multi_kernel<%d,%d>" % (C, Kn), (G // Kn) * (8 * Kn * C * F * T + 16 * Kn * F * T + 8 * Kn * F * D), 1)
        return ("filter_sum<%d>" % D, G * (8 * D * F * T + 8 * F * D + (16 if resid else 8) * F * T), 1)

    def masked_scm(a, k):
        Y = a[0]
        Z = a[2] if len(a) > 2 else k.get("Z")
        G, C, T = dims(Y)
        D = C + (Z.shape[1] - 1 if Z is not None else 0)
        return ("masked_scm<%d>" % D, G * (8 * D * F * T + 4 * F * T + 16 * F * D * D), 1)

    def filter_sum_scm(a, k):
        G, C, T = dims(a[1])
        return ("masked_scm<%d,ZF>" % C, G * (8 * C * F * T + 4 * F * T + 16 * F * T + 16 * F * C * C), 1)

    def tango_mid(a, k):
        Y = a[1]
        B, Kn, C, T, _ = Y.shape
        D = C + Kn - 1
        return ("tango_mid_kernel<%d,%d>" % (C, Kn), B * (8 * Kn * C * F * T + 4 * Kn * F * T + 16 * Kn * F * T + 16 * Kn * F * D * D), 1)

    def filter_dual(a, k):
        G, C, T = dims(a[2])
        return ("filter_dual_kernel<%d>" % C, G * (8 * C * F * T + 24 * F * T + 16 * F * C), 1)

    def stft(a, k):
        x = a[0]
        L = x.shape[-1]
        n = x.numel() // L
        return ("stft_scm_kernel<%d,*,0>" % n_fft, n * (4 * L + 8 * F * (1 + L // (n_fft // 2))), 1)

    return {
        "stft": stft,
        "stft_scm": lambda a, k: stft_scm(a, k, 1),
        "stft_scm2": lambda a, k: stft_scm(a, k, 2),
        "mwf_solve_workspace": lambda a, k: ("mwf_solve_kernel<%d,partials>" % a[2], solve(a[1] * F, a[2]), 1),
        "mwf_solve_workspace2": lambda a, k: ("mwf_solve_kernel<%d,partials,2 sets>" % a[2], solve(2 * a[1] * F, a[2]), 1),
        "mwf_solve": lambda a, k: ("mwf_solve_kernel<%d>" % a[0].shape[-1], solve(a[0].numel() // a[0].shape[-1] ** 2, a[0].shape[-1]), 1),
        "filter_sum": filter_sum,
        "masked_scm": masked_scm,
        "filter_sum_scm": filter_sum_scm,
        "tango_mid": tango_mid,
        "filter_dual": filter_dual,
    }


class KernelTimer:
    """Wraps the ops the pipeline calls with CUDA events on their launch stream (eager steps only)."""

    def __init__(self, ops_mod, n_fft):
        import torch
        self.torch, self.ops = torch, ops_mod
        self.models = _op_models(n_fft)
        self.orig = {}
        self.calls = []          # (key, name, bytes, launches, ev0, ev1) of the CURRENT step
        self.steps = []
        self.on = False

    def __enter__(self):
        for name, model in self.models.items():
            fn = getattr(self.ops, name)
            self.orig[name] = fn
            setattr(self.ops, name, self._wrap(name, fn, model))
        return self

    def _wrap(self, name, fn, model):
        def timed(*a, **k):
            if not self.on:
                return fn(*a, **k)
            label, nbytes, launches = model(a, k)
            e0, e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            self.calls.append(("%d:%s" % (len(self.calls), name), label, nbytes, launches, e0, e1))
            return r
        return timed

    def step(self, fn):
        self.on, self.calls = True, []
        fn()
        self.on = False
        self.steps.append(self.calls)

    def __exit__(self, *exc):
        for name, fn in self.orig.items():
            setattr(self.ops, name, fn)

    def summary(self, peak_gbs):
        self.torch.cuda.synchronize()
        rows = {}
        for calls in self.steps:
            for key, label, nbytes, launches, e0, e1 in calls:
                r = rows.setdefault(key, {"kernel": label, "bytes": nbytes, "launches": launches, "ms": []})
                r["ms"].append(e0.elapsed_time(e1))
        out = []
        for key in sorted(rows, key=lambda k: int(k.split(":")[0])):
            r = rows[key]
            ms = float(np.mean(r["ms"]))
            gbs = r["bytes"] / (ms / 1e3) / 1e9
            out.append({"op": key.split(":")[1], "kernel": r["kernel"], "launches": r["launches"], "us": 1e3 * ms,
                        "algorithmic_bytes": int(r["bytes"]), "achieved_gbs": gbs, "frac": gbs / peak_gbs})
        return out


# ----------------------------------------------------------------------------------------------
# Node-sharded distributed MWF (BASELINE configs[2] / [4] as stated: the array nodes live on different GPUs and
# exchange their compressed signals): rank r owns K / N nodes of EVERY utterance of the global batch.
# ----------------------------------------------------------------------------------------------
NODE_BATCH = {"cfg3": 256, "cfg5": 512}          # global utterances per step (BASELINE: 256 over 4 GPUs, 512 over 8)


def synth_on_device(B, Kl, C, L, seed, dev, taps=32):
    """Coherent source through a random decaying FIR per microphone + white noise, generated on the device
    (same recipe as disco_b200/synth.py; the node-sharded batches are too large to synthesise on the host)."""
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    src = 0.1 * torch.randn((B, 1, L + taps - 1), generator=g, device=dev)
    h = torch.randn((Kl * C, 1, taps), generator=g, device=dev) * torch.exp(-torch.arange(taps, device=dev) / 6.0)
    s = torch.nn.functional.conv1d(src, h.flip(-1)).view(B, Kl, C, L)
    n = 0.05 * torch.randn((B, Kl, C, L), generator=g, device=dev)
    return s + n, s, n


def main_nodes(args):
    import torch
    import torch.distributed as dist
    from disco_b200 import ops
    from disco_b200.dist import tango_node_sharded
    B, K, C, L, n_fft, desc = WORKLOADS[args.workload]
    B = args.batch or NODE_BATCH.get(args.workload, B)
    T, F = 1 + L // (n_fft // 2), n_fft // 2 + 1
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert K % world == 0, "--shard nodes needs the number of ranks to divide the number of nodes (%d)" % K
    Kl = K // world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29533")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        os.environ.pop("NCCL_DEBUG")             # keep NCCL's version banner out of stdout (one JSON line)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    ops.init(n_fft)
    # measured (DESIGN.md section 6): chunking pays only when the step is one CUDA graph; eager launches cost more
    # than the overlap returns (4 GPUs: 3.98 ms unchunked, 4.19 ms with 4 chunks)
    chunks = args.chunks if args.chunks > 0 else (4 if args.graph else 1)
    # this rank's nodes of every utterance; masks from the clean components of the reference microphone
    y = torch.empty((B, Kl, C, L), dtype=torch.float32, device=dev)
    mz = torch.empty((B, Kl, T, F), dtype=torch.float32, device=dev)
    mw = torch.empty_like(mz)
    for lo in range(0, B, 32):
        yb, sb, nb = synth_on_device(min(32, B - lo), Kl, C, L, 7919 * rank + lo, dev)
        y[lo:lo + 32] = yb
        S, N = ops.stft(sb[:, :, 0].contiguous(), n_fft), ops.stft(nb[:, :, 0].contiguous(), n_fft)
        mz[lo:lo + 32], mw[lo:lo + 32] = ops.tf_mask(S, N, "irm1"), ops.tf_mask(S, N, "irm2")
    del yb, sb, nb, S, N
    torch.cuda.empty_cache()

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    stats = {}

    def eager_step(st=stats):
        return tango_node_sharded(y, mz, mw, chunks=chunks, stats=st, n_fft=n_fft, out_layout="TF",
                                  reserve_sms=None if args.reserve_sms < 0 else args.reserve_sms)
    for _ in range(max(3, args.warmup)):
        eager_step()
    barrier()
    # optional: the whole step (compute kernels, stream forks / joins, NCCL gathers) as ONE CUDA graph -- the eager step
    # costs ~10 Python-level launches per chunk, which is what limits fine chunking
    graph, execution = None, "eager launches (no CUDA graph)"
    if args.graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                eager_step(None)
            torch.cuda.current_stream(dev).wait_stream(side)
            barrier()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                graph_out = eager_step(None)
            barrier()
            for _ in range(3):
                graph.replay()
            barrier()
            execution = "CUDA graph of the whole step (kernels + NCCL all-gathers)"
        except Exception as exc:           # capture of collectives not possible here: stay eager, say so
            graph, execution = None, "eager launches (CUDA-graph capture failed: %s)" % str(exc).splitlines()[0][:120]
            barrier()

    def step():
        if graph is not None:
            graph.replay()
        else:
            eager_step()
    samples, stop = [], threading.Event()
    th = threading.Thread(target=clock_sampler, args=(stop, samples, local_rank), daemon=True)
    if rank == 0:
        th.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gathers = []
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
        gathers.append(stats["gathers"])           # (graph replay: the events of the last eager warm-up step)
    e1.record()
    barrier()
    stop.set()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    g_ms = float(np.mean([sum(t0.elapsed_time(t1) for t0, t1, _ in gs) for gs in gathers]))
    g_bytes = sum(nb for _, _, nb in gathers[0])
    gt = torch.tensor([g_ms], device=dev)
    dist.all_reduce(gt, op=dist.ReduceOp.MAX)
    # the same step without the exchange being waited for is not observable from outside; what is: the compute
    # kernels alone (one chunk, gather result reused), timed on this rank
    frames = B * K * T * args.steps
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        res = {"metric": METRIC, "value": frames / (ms / 1e3), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "f32 (c64 spectra, f32 SCM accumulation, f64 per-bin solve)", "data": "synthetic",
               "config": {"workload": "%s: %s" % (args.workload, desc), "nodes": K, "mics_per_node": C,
                          "utterance_s": L / 16000.0, "n_fft": n_fft, "hop": n_fft // 2, "global_batch": B,
                          "frames_per_step": B * K * T,
                          "parallelism": "node-sharded: %d node(s) of every utterance per rank x %d ranks; compressed signals z "
                                         "all-gathered over NCCL in %d batch chunks, gather(i) overlapped with step 1(i+1), "
                                         "node-major Z read in place by step 2" % (Kl, world, chunks),
                          "mode": "deployment: mixture + masks in, yf / z out", "execution": execution,
                          "reserved_sms": "library default (16 while gathers are in flight)" if args.reserve_sms < 0 else args.reserve_sms,
                          "l2": "inputs larger than L2 (y %.0f MB, Y %.0f MB per GPU)" % (B * Kl * C * L * 4 / 1e6, B * Kl * C * T * F * 8 / 1e6)},
               "clocks": summarize_clocks(samples),
               "exchange": {"collective": "ncclAllGather (all_gather_into_tensor), %d per step" % chunks,
                            "bytes_received_per_rank_per_step": int(g_bytes), "gather_ms_per_step": float(gt.item()),
                            "gather_gbs_per_rank": g_bytes / (float(gt.item()) / 1e3) / 1e9 if g_bytes else None,
                            "nvlink_reference_gbs": 770.0,
                            "note": "gather time is measured on the communication stream (CUDA events), max over ranks; it "
                                    "overlaps step 1 of the next chunk" + ("; under the CUDA graph it is the figure of the last "
                                    "eager warm-up step" if graph is not None else "")},
               "gpu_launches": None, "roofline": None}
        print(json.dumps(res), flush=True)
    if graph is not None:
        # measured on 8 GPUs (round 2): tearing down the process group after a CUDA graph holding NCCL kernels was
        # replayed hangs until the launcher's timeout; the line is out, every rank is past the last barrier -> leave
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="override utterances per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=8, help="batch slices of the host-to-host pipeline")
    ap.add_argument("--chunks", type=int, default=0, help="batch chunks captured on parallel graph branches (0 = auto)")
    ap.add_argument("--shard", default="utterances", choices=["utterances", "nodes"])
    ap.add_argument("--masks", default="oracle", choices=["oracle", "crnn"],
                    help="e2e leg: masks uploaded from the host (oracle) or predicted on device by the reference CRNN")
    ap.add_argument("--graph", action="store_true", help="--shard nodes: capture the step (kernels + NCCL gathers) in a CUDA graph")
    ap.add_argument("--reserve-sms", type=int, default=-1, help="--shard nodes: SMs left free for NCCL (-1 = library default)")
    ap.add_argument("--crnn-exact", action="store_true", help="run the CRNN in IEEE float32 (default: TF32)")
    ap.add_argument("--crnn-bf16", action="store_true", help="run the CRNN under bf16 autocast (throughput only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32; a fixed, "
                         "seeded sample of %d MiB in all when larger)" % (DUMP_BUDGET >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.shard != "utterances"):
        ap.error("--dump-outputs writes the outputs of --impl ours --shard utterances")
    B, K, C, L, n_fft, desc = WORKLOADS[args.workload]
    if args.batch:
        B = args.batch
    T, F = 1 + L // (n_fft // 2), n_fft // 2 + 1
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.shard == "nodes":
        return main_nodes(args)                      # node-sharded distributed MWF (all-gather of z)
    chunks = args.chunks if args.chunks > 0 else (2 if K > 1 else 1)
    chunks = max(1, min(chunks, B))
    config = {"workload": "%s: %s" % (args.workload, desc), "nodes": K, "mics_per_node": C, "utterance_s": L / 16000.0,
              "n_fft": n_fft, "hop": n_fft // 2, "batch_per_gpu": B, "global_batch": B * world, "frames_per_step": B * K * T * world,
              "mode": "deployment: inputs = mixture y + masks (mask_z, mask_w), outputs = yf, z, zn; same work in the CPU arm",
              "inputs": "%d distinct synthetic utterances per GPU (coherent source + white noise, disco_b200/synth.py)" % B,
              "mask": "device-resident masks, frame-major (T,F): mask_z = irm1, mask_w = irm2 of the clean components' "
                      "reference channel (tf_mask, dnn/utils.py:44-71)",
              "parallelism": "utterance-sharded x%d, no collective" % world,
              "execution": "CUDA graph, %d batch chunk(s) on parallel branches" % chunks,
              "l2": "inputs larger than L2 (y %.0f MB, Y %.0f MB per GPU)" % (B * K * C * L * 4 / 1e6, B * K * C * T * F * 8 / 1e6)}

    if args.impl == "reference":
        if rank != 0:
            return
        arm = CpuArm(K, C, L, n_fft)
        steps = max(1, args.steps)
        budget = max(2.0, min(15.0, 150.0 / (steps + min(args.warmup, 1))))     # whole run within a few minutes
        if args.warmup > 0:
            arm.sample(min(budget, 3.0))                                       # one untimed warm-up sample
        t_all, frames, last = 0.0, 0, None
        for _ in range(steps):            # each step = one bounded sample on all host cores
            last = arm.sample(budget)
            t_all += last["seconds"]
            frames += last["frames"]
        arm.close()
        val = frames / t_all
        last = dict(last, value=val, seconds=t_all, frames=frames,
                    sample=last["sample"] + "; %d such samples" % steps)
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": val,
                          "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": min(args.warmup, 1),
                          "ms_per_step": 1e3 * t_all / steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "c64 SCM/cggev, c128 filters (reference dtype flow)", "data": "synthetic",
                          "config": config, "cpu_baseline": last,
                          "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    from disco_b200 import ops
    from disco_b200.tango import tango_batched
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        bound = bind_host_to_gpu(local_rank)     # before the pinned buffers are allocated
        config["host_affinity"] = ("rank bound to the %d CPUs of its GPU's NUMA node" % bound) if bound else "unbound"
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            os.environ.pop("NCCL_DEBUG")         # keep NCCL's version banner out of stdout (one JSON line)
        dist.init_process_group("nccl", device_id=dev)

    # ---- synthetic inputs (seeded): B distinct utterances; masks from the clean components on the device
    from disco_b200.synth import make_utterance
    ops.init(n_fft)
    y_host = torch.empty((B, K, C, L), dtype=torch.float32).pin_memory()
    mz = torch.empty((B, K, T, F), dtype=torch.float32, device=dev)
    mw = torch.empty_like(mz)
    s_ref = torch.empty((B, K, L), dtype=torch.float32)
    n_ref = torch.empty((B, K, L), dtype=torch.float32)
    for b in range(B):
        yb, sb, nb = make_utterance(100000 * rank + b, K, C, L)
        y_host[b] = torch.from_numpy(yb)
        s_ref[b], n_ref[b] = torch.from_numpy(sb[:, 0]), torch.from_numpy(nb[:, 0])
    for lo in range(0, B, 32):          # a few launches for the whole batch (keeps profiler launch lists short)
        S, N = ops.stft(s_ref[lo:lo + 32].to(dev), n_fft), ops.stft(n_ref[lo:lo + 32].to(dev), n_fft)
        mz[lo:lo + 32], mw[lo:lo + 32] = ops.tf_mask(S, N, "irm1"), ops.tf_mask(S, N, "irm2")
    del S, N, s_ref, n_ref
    mz_host, mw_host = mz.cpu().pin_memory(), mw.cpu().pin_memory()
    y = y_host.to(dev)
    from disco_b200.plan import TangoGraph
    plan = TangoGraph(B, K, C, L, n_fft=n_fft, chunks=chunks, device=dev)   # CUDA graph of the whole step
    plan.load(y, mz, mw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed region 1: whole-path throughput, inputs resident in HBM (graph replays)
    for _ in range(max(3, args.warmup)):
        plan.run()
    barrier()
    samples, stop = [], threading.Event()
    th = threading.Thread(target=clock_sampler, args=(stop, samples, local_rank), daemon=True)
    if rank == 0:
        th.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(args.steps):
        plan.run()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    tmax = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms = float(tmax.item())
    frames = B * K * T * world * args.steps
    value = frames / (ms / 1e3)
    if args.dump_outputs and rank == 0:           # the plan's static output buffers still hold the last timed step
        dump_outputs(args.dump_outputs, {nm: plan.output(nm) for nm in plan.outputs[0]})

    # ---- timed region 2: every kernel of the step, CUDA events on the launch stream inside eager steps
    import disco_b200.tango as tango_mod

    def eager_step():
        return tango_batched(y, masks=(mz, mw), n_fft=n_fft, out_layout="TF", diagnostics=False)
    for _ in range(3):
        eager_step()
    barrier()
    n_k = min(args.steps, 30)
    with KernelTimer(tango_mod.ops, n_fft) as kt:
        for i in range(n_k):
            kt.step(eager_step)
        barrier()

    # ---- e2e: pinned host buffers in, beamformed STFT out, through the public API
    e2e = None
    if not args.no_e2e:
        yf_host = torch.empty((B, K, T, F), dtype=torch.complex64).pin_memory()
        if args.masks == "crnn" and K == 1:
            from disco_b200.plan import CrnnTangoPipeline
            pipe = CrnnTangoPipeline(B, C, L, n_fft, args.e2e_chunks, dev, exact=args.crnn_exact, bf16=args.crnn_bf16,
                                     cudnn_benchmark=args.crnn_bf16)
            y_i16 = pipe.to_pcm(y_host)

            def e2e_step():   # int16 PCM H2D -> CRNN masks on device -> the whole path -> D2H of yf
                pipe.process(y_i16, yf_host)
            h2d, how = int(y_i16.numel() * 2), pipe.how
        else:
            from disco_b200.plan import TangoPipeline
            pipe = TangoPipeline(B, K, C, L, n_fft=n_fft, chunks=args.e2e_chunks, device=dev)

            def e2e_step():   # H2D of signals + masks, the whole path, D2H of yf -- overlapped across batch slices
                pipe.process(y_host, mz_host, mw_host, yf_host)
            h2d = int(y_host.numel() * 4 + 2 * mz_host.numel() * 4)
            how = "TangoPipeline: %d batch slices, per-slice H2D -> graph replay -> D2H on its own stream (pinned host buffers)" % args.e2e_chunks
        for _ in range(3):
            e2e_step()
        barrier()
        n_e2e = max(3, min(args.steps // 4, 50))
        e0.record()
        for _ in range(n_e2e):
            e2e_step()
        e1.record()
        barrier()
        t2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e = {"value": B * K * T * world * n_e2e / (float(t2.item()) / 1e3), "unit": "frames/s",
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": int(yf_host.numel() * 8), "steps": n_e2e, "how": how}
        if args.masks == "crnn" and K == 1:
            e2e["crnn"] = pipe.report()
    stop.set()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        kernels = kt.summary(peak)
        step_us = sum(k["us"] for k in kernels)
        for k in kernels:
            k["share_of_step"] = k["us"] / step_us
        dom = max(kernels, key=lambda k: k["us"])
        traffic = None       # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, from the committed ncu capture
        try:
            norm = lambda t: t.replace("void", "").strip().split("<")[0].split("(")[0]      # kernel base name
            tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            for ent in tj.values():
                if ent.get("workload") == args.workload and not args.batch and norm(ent["kernel"]) == norm(dom["kernel"]):
                    traffic = ent["dram_bytes_per_launch"]
        except Exception:
            pass
        roof = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": dom["frac"], "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                "algorithmic_bytes_per_launch": dom["algorithmic_bytes"], "kernel_ms": dom["us"] / 1e3,
                "share_of_step": dom["share_of_step"],
                "timed": "CUDA events around every op in %d eager steps (the throughput region replays a CUDA graph)" % n_k,
                "step_algorithmic_bytes": int(sum(k["algorithmic_bytes"] for k in kernels)),
                "step_frac": sum(k["algorithmic_bytes"] for k in kernels) / (ms / args.steps / 1e3) / 1e9 / peak,
                "kernels": kernels}
        res = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world,
               "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f32 (c64 spectra, f32 SCM accumulation, f64 per-bin solve)",
               "data": "synthetic", "config": config, "clocks": summarize_clocks(samples),
               "gpu_launches": sum(k["launches"] for k in kernels) * chunks * args.steps, "roofline": roof}
        if e2e:
            res["e2e"] = e2e
        if not args.no_cpu and world == 1:      # the CPU leg is an N = 1 measurement (rank 0 owns the whole host)
            arm = CpuArm(K, C, L, n_fft)
            res["cpu_baseline"] = arm.sample(12.0)
            res["cpu_baseline_vectorized"] = arm.sample(6.0, granularity="bin")
            arm.close()
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
