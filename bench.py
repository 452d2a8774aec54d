#!/usr/bin/env python
"""bench.py - CTR inferences/s of the DIN forward path (BASELINE.json configs[2]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

What is scored: DIN ranking instances (T=50, E=32, MovieLens-20M-shaped vocabularies, synthetic
Zipf inputs, seeded random-init weights of the reference architecture) in batches of `--batch`
(4096) rows, ONE fused-kernel launch per batch.

A *step* is one `model.predict(dataset)` pass (DIN.py:185: Keras iterates the dataset batch by
batch) over a resident dataset of R distinct 4096-row batches - R launches - so that K = 20 steps
are a timed region of a few hundred milliseconds, not a few hundred microseconds.  R and the
number of launches are in the line (`step`, `gpu_launches`).

* `value`  : rows scored per second with the dataset already resident in HBM, device-timed with
             CUDA events around exactly K steps (K replays of a CUDA graph of the R launches),
             max over ranks.  The dataset's footprint far exceeds the 126 MB L2, so every
             launch's ids / numerics come from HBM; the 21 MB of embedding tables stay L2
             resident by size (that is the workload's nature, see `detail.l2`).
* `e2e`    : the same metric through the reference-facing C-ABI call with HOST buffers: one
             `srs_predict_host_batches` call per step over a pinned host dataset (H2D of each
             batch, kernel, D2H of its scores, pipelined over the library's slots), wall clock
             around K calls, max over ranks.  `e2e` carries the reference's own wire types (int32
             ids); `e2e_hist16` is the same leg with the history ids as uint16
             (`srs_batch::hist16`, opt-in in the Python surface too).
* `roofline`: algorithmic bytes per launch (SURVEY.md 8d: 7160 B/row) / device time per launch
             (timed region / launches), against the measured HBM copy bandwidth in
             MEASURED_PEAKS.json.
* `cpu_baseline`: the CPU restatement of the Keras graph (TensorFlow is not installable here)
             timed on this box's host cores on a bounded sample: oracle/ctr_oracle_c.c (plain C,
             OpenMP over rows) for DIN, the row-chunked numpy oracle for the other models.

`--impl reference` times that CPU restatement as the reference arm (rank 0 only): thread-count
sweep, >= 20 timed iterations, median / p10 / p90, plus the batch-12 and batch-128 lines of
BASELINE.md section 2.
Multi-GPU (`torchrun`, one rank per GPU): rows shard by rank, weights replicate, no data-path
collective (weak scaling: 4096 rows per GPU per launch); `--gather` adds the exchange of scores
that a ranking call spanning GPUs needs (`--gather nccl`: torch NCCL all-gather per launch;
`--gather fused`: the kernel's epilogue stores its scores into every peer's gather buffer over
NVLink).  Each rank binds to the CPUs of its GPU's NUMA node before it allocates pinned memory.
`--workload cfg5_din` (10^8-row table) launches directly instead of replaying a graph (`--graph`
restores the replay; why: DESIGN.md section 6).  stdout carries the one JSON line and nothing else;
an outer `timeout` (SIGTERM) makes the script dump its Python stacks to stderr first.
`--dump-outputs DIR` writes the scores of the last timed step to DIR/scores.npy ([batches, rows], float32;
`scores_rank<r>.npy` per rank with N > 1): the inputs are seeded, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# OpenMP workers of the CPU arm sleep when idle (set before anything loads an OpenMP runtime): a
# thread-count sweep otherwise leaves the larger teams spinning on the cores the next measurement needs
for _k, _v in (("OMP_WAIT_POLICY", "PASSIVE"), ("GOMP_SPINCOUNT", "0"), ("OMP_PROC_BIND", "false"),
               ("OMP_DYNAMIC", "false")):
    os.environ.setdefault(_k, _v)

METRIC = "CTR inferences/sec (DIN, batch=4096, hist_len=50)"
WORKLOAD = "cfg3_din"
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 64 << 20                   # --dump-outputs: at most this much in all, a seeded sample of batches above
DTYPE = "bf16x3 (fp32 accumulate)"      # every MMA operand is split hi + lo, three products, fp32 accumulators

# BASELINE.json configs -> (default rows per GPU per launch, metric label).  cfg3_din is the
# configuration the headline metric is quoted on (the default); the others are the remaining
# rows of SURVEY.md section 8d and run with `--workload <name>`.
WORKLOADS = {
    "cfg1_embeddingmlp": (128, "EmbeddingMLP, MovieLens-1K vocab, batch=128"),
    "cfg2_deepfm": (4096, "DeepFM, ML-20M vocab, emb_dim=16, batch=4096"),
    "cfg2_deepfm_v2": (4096, "DeepFM_v2, ML-20M vocab, emb_dim=16, batch=4096"),
    "cfg3_din": (4096, "DIN, batch=4096, hist_len=50"),
    "cfg4_widendeep": (8192, "Wide&Deep, batch=65536 over 8 GPUs = 8192 per GPU"),
    "cfg4_neuralcf": (8192, "NeuralCF, batch=65536 over 8 GPUs = 8192 per GPU"),
    "cfg4_twotowers": (8192, "two towers, batch=65536 over 8 GPUs = 8192 per GPU"),
    "cfg5_din": (8192, "DIN, 100M-item vocab, emb_dim=64, hist_len=200, batch=8192"),
    # not a BASELINE.json config: the reference's DIEN.py shape (SURVEY.md section 8f row 4)
    "ref_dien": (4096, "DIEN, MovieLens-1K vocab, emb_dim=10, hist_len=5, batch=4096"),
}
FP32_WORKLOADS = ("cfg2_deepfm_v2", "cfg4_neuralcf", "cfg4_twotowers", "ref_dien")   # CUDA-core fp32 kernels


def metric_name(workload):
    return METRIC if workload == WORKLOAD else "CTR inferences/sec (%s)" % WORKLOADS[workload][1]


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="rows per GPU per launch")
    ap.add_argument("--workload", default=WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--dataset-batches", type=int, default=None,
                    help="R: distinct batches of the resident dataset = launches per step (default: "
                         "512, more if needed to exceed the L2, fewer if 1.5 GB of inputs is exceeded)")
    ap.add_argument("--host-batches", type=int, default=None,
                    help="batches of the pinned host dataset of the e2e leg = batches per step (default 256, "
                         "fewer if 512 MB of pinned memory is exceeded)")
    ap.add_argument("--gather", nargs="?", const="nccl", default=None, choices=["nccl", "fused"],
                    help="exchange the scores after every launch (N > 1): torch NCCL all-gather, or the "
                         "kernel storing into the peers' gather buffers (fused)")
    ap.add_argument("--no-graph", action="store_true", help="launch directly instead of CUDA graphs")
    ap.add_argument("--graph", action="store_true",
                    help="cfg5_din only: replay a CUDA graph although that is off by default there (see below)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--streams", type=int, default=None,
                    help="S > 1: consecutive batches run side by side on S branches of the CUDA graph "
                         "(default: 2 for the headline workload, 1 for cfg 5, 4 otherwise)")
    ap.add_argument("--sm-limit", type=int, default=None,
                    help="CTAs per launch with --streams S > 1 (default: SMs/S for kernels that hold a whole "
                         "SM per CTA, 0 = no limit for kernels that fit two CTAs per SM)")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--history", default=None, choices=["uniform", "zipf"],
                    help="distribution of the history ids (default: uniform for cfg 5 - the L2-defeating worst case "
                         "BASELINE.md asks for - Zipf(1.05) otherwise)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the scores of the last timed step to DIR/scores.npy")
    args = ap.parse_args(argv)
    if args.dump_outputs and (args.impl != "ours" or args.gather == "fused"):
        ap.error("--dump-outputs writes the scores of --impl ours without --gather fused")
    if args.batch is None:
        args.batch = WORKLOADS[args.workload][0]
    # cfg 5 launches directly: CUDA-graph replays of din_rt64_kernel on the 10^8-row table did not finish in
    # 11 of 18 runs on the B200 (direct launches: 4 of 4 finished, same throughput; profiles/r02/rt64_hang/)
    if args.workload == "cfg5_din" and not args.graph:
        args.no_graph = True
    if args.streams is None:
        # batches in flight side by side (BASELINE.md section 3 (iii): steady-state throughput is quoted
        # with batches in flight, single-call latency separately).  cfg 5 launches fill the machine.
        args.streams = 1 if args.workload == "cfg5_din" else (2 if args.workload == WORKLOAD else 4)
    return args


def dist_env():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")),
            int(os.environ.get("WORLD_SIZE", "1")))


def workload_desc(name, spec, batch):
    if spec.model == "din":
        return ("%s: DIN forward, hist_len=%d, emb_dim=%d, batch=%d per GPU, V_movie=%d, V_user=%d, "
                "activation unit 4E->32->1 sigmoid-gated sum pooling, top MLP %d->128->64->1"
                % (name, spec.hist_len, spec.emb_dim, batch, spec.n_movies, spec.n_users,
                   5 * spec.emb_dim + 7))
    return ("%s: %s forward, emb_dim=%d, batch=%d per GPU, V_movie=%d, V_user=%d, hidden=%s"
            % (name, spec.model, spec.emb_dim, batch, spec.n_movies, spec.n_users, list(spec.hidden)))


def shared_config(args, spec, world):
    """The `config` object: identical in both arms (what is computed, not how)."""
    return {"workload": workload_desc(args.workload, spec, args.batch), "batch_per_gpu": args.batch,
            "global_batch": world * args.batch,
            "inputs": "synthetic MovieLens-20M-shaped rows (seeded): %s movie ids, history 0-padded to T "
                      "(padding included, as in the reference), random-init weights of the reference "
                      "architecture (seed 2)" % ("uniform" if ((args.history == "uniform") if args.history
                                                                 else args.workload == "cfg5_din") else "Zipf(1.05)")}


def make_weights(spec, device=None):
    """Seeded random-init weights of the reference architecture.  The 25.6 GB movie table of
    cfg 5 is generated in place in HBM (srs_fill_uniform) and handed over without a copy; on
    the CPU side a 10^6-row surrogate of the same formula is used for timing only."""
    from sparrowrecsys_b200.weights import init_weights
    big = spec.model == "din" and spec.n_movies > 10_000_000
    if not big:
        return init_weights(spec, 2), None
    W = init_weights(spec, 2, skip=("embedding",))
    if device is None:
        return W, None
    import torch
    from sparrowrecsys_b200 import _lib
    table = torch.empty(spec.n_movies, spec.emb_dim, dtype=torch.float32, device=device)
    _lib.check(_lib.load().srs_fill_uniform(table.data_ptr(), table.numel(), 1234, -0.05, 0.05,
                                            device.index, None))
    torch.cuda.synchronize(device)
    W["embedding"] = table
    return W, table


def cpu_spec_and_weights(spec):
    """Spec/weights the CPU restatement can hold (cfg 5: 10^6-row surrogate vocabulary)."""
    from dataclasses import replace
    from sparrowrecsys_b200.weights import init_weights
    from oracle import ctr_oracle as O
    if spec.model == "din" and spec.n_movies > 10_000_000:
        small = replace(spec, n_movies=1_000_000)
        W = init_weights(small, 2, skip=("embedding",))
        W["embedding"] = O.fill_uniform(np.arange(small.n_movies * small.emb_dim), 1234, -0.05,
                                        0.05).reshape(small.n_movies, small.emb_dim)
        return small, W, " (10^6-row surrogate movie table for the CPU timing)"
    return spec, init_weights(spec, 2), ""


# ----------------------------------------------------------------------------------------
def gpu_cpu_affinity(index):
    """CPUs of the NUMA node GPU `index` hangs off (NVML nvmlDeviceGetCpuAffinity), or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")
        if visible:
            index = int(visible.split(",")[index])
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = (ncpu + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        return [c for c in cpus if c < ncpu] or None
    except Exception:
        return None


def bind_to_gpu_numa(local_rank):
    """Pin this process (and the pinned host memory it allocates from now on: first touch) to the
    CPUs next to its GPU.  Returns (previous affinity, description)."""
    try:
        before = os.sched_getaffinity(0)
    except Exception:
        return None, "sched_getaffinity unavailable"
    cpus = gpu_cpu_affinity(local_rank)
    if not cpus:
        return before, "NVML gave no CPU affinity for the GPU: not bound"
    try:
        allowed = sorted(set(cpus) & before) or sorted(cpus)
        os.sched_setaffinity(0, allowed)
        return before, "bound to the %d CPUs of GPU %d's NUMA node (%d..%d)" % (
            len(allowed), local_rank, allowed[0], allowed[-1])
    except Exception as e:                                   # pragma: no cover
        return before, "sched_setaffinity failed: %r" % (e,)


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed
    region runs (nvidia-smi reads the same counters)."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap",
               0x8: "hw_slowdown", 0x10: "sync_boost", 0x20: "sw_thermal_slowdown",
               0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
               0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons = [], set()
        self.ok = False
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            if visible:
                index = int(visible.split(",")[index])
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                                   # pragma: no cover
            self.err = repr(e)

    def sample(self):
        if not self.ok:
            return
        try:
            nv = self.nv
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in self.REASONS.items():
                if mask & bit and name != "gpu_idle":
                    self.reasons.add(name)
        except Exception:
            pass

    def start(self, period=0.02):
        def run():
            while not self._stop.is_set():
                self.sample()
                self._stop.wait(period)
        self._thread = threading.Thread(target=run, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": float(self.max_mhz),
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s; MEASURED_PEAKS.json absent)"


def ncu_traffic(workload, kernel_name, batch):
    """dram read+write bytes per launch of the dominant kernel from the committed ncu summary of this
    workload (profiles/ncu_bench_summary.json, written by profiles/summarize_r02.py from one
    `ncu --set full` capture of `bench.py --workload W`), or None when the capture was of another
    kernel or batch size."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_bench_summary.json")) as f:
            rec = json.load(f)[workload]
        if rec.get("kernel") != kernel_name or int(rec.get("batch", -1)) != int(batch):
            return None
        return rec.get("dram_bytes_per_launch")
    except Exception:
        return None


# ----------------------------------------------------------------------------------------
# CPU arm: the restatement of the Keras graph on the host cores
# ----------------------------------------------------------------------------------------
def cpu_forward(spec, W):
    """(fn(feats, threads) -> scores, description, thread counts worth sweeping)."""
    cores = os.cpu_count() or 1
    if spec.model == "din":
        from oracle import ctr_oracle_cext as OC
        fwd = OC.din_predictor(spec, W, cores)
        return (lambda feats, th: fwd(feats, th)), \
            "oracle/ctr_oracle_c.c: plain-C restatement of DIN.py:125-167, OpenMP over batch rows " \
            "(gcc -O3 -mavx2 -mfma), feature-column encoding in numpy", \
            sorted({t for t in (8, 16, 32, 64, cores // 2, cores) if 1 <= t <= cores})
    from oracle import ctr_oracle_torch as OT
    cache = {}

    def run(feats, th):
        if th not in cache:
            cache[th] = OT._chunked_numpy(spec, W, th)
        return cache[th](feats)
    return run, "numpy oracle (oracle/ctr_oracle.py) over 256-row chunks on a thread pool, 1 BLAS thread each", \
        sorted({t for t in (8, 32, cores) if 1 <= t <= cores})


def time_calls(fn, min_iters, max_seconds, min_seconds=0.0):
    """Per-call seconds of fn(): at least `min_iters` calls (and `min_seconds` of them), stopping
    early only if `max_seconds` is exceeded after 3 calls."""
    ts = []
    t_start = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
        el = time.perf_counter() - t_start
        if (len(ts) >= min_iters and el >= min_seconds) or (len(ts) >= 3 and el > max_seconds):
            break
    return np.array(ts)


def best_threads(run, feats, candidates, seconds_each=1.5):
    """Thread count with the best single call, candidates visited up and then down again (the first
    configuration a process runs and the one right after a larger team are the ones that measure low)."""
    sweep = {}
    order = list(candidates) + list(reversed(candidates))[1:]
    for th in order:
        run(feats, th)                                            # warm-up (thread team, caches)
        ts = time_calls(lambda: run(feats, th), 4, seconds_each / 2)
        v = round(len(feats["movieId"]) / float(np.min(ts)), 1)   # best call: picks the count, not the value
        sweep[str(th)] = max(v, sweep.get(str(th), 0.0))
    best = max(candidates, key=lambda th: sweep[str(th)])
    return best, sweep


def cpu_baseline_block(args, spec, feats_full):
    """cpu_baseline of the GPU arm: bounded sample (about --cpu-seconds of CPU work)."""
    from sparrowrecsys_b200.features import synthetic_features
    cspec, cW, cnote = cpu_spec_and_weights(spec)
    n_cpu = min(args.batch, 4096)
    feats = {k: np.asarray(v)[:n_cpu] for k, v in feats_full.items()}
    if cspec is not spec:
        feats = synthetic_features(cspec, n_cpu, seed=7, uniform_history=True)
    run, how, cands = cpu_forward(cspec, cW)
    th, sweep = best_threads(run, feats, cands, seconds_each=min(1.5, args.cpu_seconds / (2 * len(cands))))
    ts = time_calls(lambda: run(feats, th), 20, args.cpu_seconds / 2)
    v = n_cpu / float(np.median(ts))
    return {"value": v, "unit": "inferences/s", "cores": th, "host_cpus": os.cpu_count() or 1, "kind": "port",
            "p10": n_cpu / float(np.quantile(ts, 0.9)), "p90": n_cpu / float(np.quantile(ts, 0.1)),
            "thread_sweep": sweep,
            "sample": "%d x %d-row batch of the same workload, median; %s; TF2 is not installable here%s"
                      % (len(ts), n_cpu, how, cnote)}


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path.  TensorFlow is not
    installed / installable on this image, so this is the CPU restatement of the Keras graph
    (see cpu_forward), same workload, each step a bounded sample of the batch."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    from sparrowrecsys_b200.features import synthetic_features
    from sparrowrecsys_b200.spec import baseline_spec
    full_spec = baseline_spec(args.workload)
    spec, W, note = cpu_spec_and_weights(full_spec)
    feats = synthetic_features(spec, args.batch, seed=2, uniform_history=args.workload == "cfg5_din")
    run, how, cands = cpu_forward(spec, W)
    th, sweep = best_threads(run, feats, cands)
    # per-step sample: the whole batch unless steps + warmup would exceed ~2 minutes
    t_batch = float(np.median(time_calls(lambda: run(feats, th), 3, 10.0)))
    budget, total = 120.0, args.steps + args.warmup
    rows = args.batch
    if t_batch * total > budget:
        rows = int(max(16, min(args.batch, args.batch * budget / (t_batch * total))))
    sample = {k: np.asarray(v)[:rows] for k, v in feats.items()}
    for _ in range(args.warmup):
        run(sample, th)
    ts = np.array([0.0] * args.steps)
    t0 = time.perf_counter()
    for i in range(args.steps):
        t1 = time.perf_counter()
        run(sample, th)
        ts[i] = time.perf_counter() - t1
    dt = time.perf_counter() - t0
    value = rows * args.steps / dt
    # BASELINE.md section 2: batch 12 (what the reference scripts use) and batch 128 (cfg 1) lines,
    # >= 20 timed iterations after 3 warm-ups, median and p10 / p90
    small = {}
    for bs in (12, 128):
        if bs >= args.batch:
            continue
        fb = {k: np.asarray(v)[:bs] for k, v in feats.items()}
        best = None
        for t in sorted({1, min(8, th), th}):
            for _ in range(3):
                run(fb, t)
            tb = time_calls(lambda: run(fb, t), 20, 5.0)
            r = {"threads": t, "median_inf_s": round(bs / float(np.median(tb)), 1),
                 "p10_inf_s": round(bs / float(np.quantile(tb, 0.9)), 1),
                 "p90_inf_s": round(bs / float(np.quantile(tb, 0.1)), 1),
                 "median_ms_per_call": round(1e3 * float(np.median(tb)), 4), "iterations": len(tb)}
            if best is None or r["median_inf_s"] > best["median_inf_s"]:
                best = r
        small["batch_%d" % bs] = best
    line = {
        "impl": "reference", "metric": metric_name(args.workload), "value": value, "unit": "inferences/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args, full_spec, world),
        "step": {"rows": rows, "what": "one CPU forward over a %d-row sample of the %d-row batch%s"
                                       % (rows, args.batch, note)},
        "cpu_baseline": {"value": value, "unit": "inferences/s", "cores": th, "host_cpus": os.cpu_count() or 1,
                         "kind": "port",
                         "median": rows / float(np.median(ts)) if args.steps else None,
                         "p10": rows / float(np.quantile(ts, 0.9)) if args.steps else None,
                         "p90": rows / float(np.quantile(ts, 0.1)) if args.steps else None,
                         "thread_sweep": sweep, "small_batches": small,
                         "sample": "%d of %d rows per step, %s; best of the thread sweep; TF2 itself is "
                                   "not installable here" % (rows, args.batch, how)},
        "e2e": {"value": value, "unit": "inferences/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------------------
def tile_encoded(enc, reps, rng):
    """`reps` row-permuted replicas of an encoded dataset (distinct batches at distinct addresses
    without generating reps x as many synthetic rows on the host)."""
    from sparrowrecsys_b200.features import EncodedBatch
    if reps <= 1:
        return enc
    perms = [np.arange(enc.B)] + [rng.permutation(enc.B) for _ in range(reps - 1)]
    cat = lambda a: None if a is None else np.ascontiguousarray(np.concatenate([a[p] for p in perms], axis=0))
    return EncodedBatch(enc.B * reps, cat(enc.movie_id), cat(enc.user_id), cat(enc.hist),
                        cat(enc.movie_genre), cat(enc.user_genre), cat(enc.numerics))


def dump_outputs(directory, name, scores, limit):
    """Write `scores` ([batches, rows], on the device) to directory/name.npy as float32: all of it, or when that
    exceeds `limit` bytes a seeded sample of whole batches, the same batches on every run."""
    import torch
    os.makedirs(directory, exist_ok=True)
    n, rows = scores.shape
    keep = min(n, max(1, limit // (4 * rows)))
    if keep < n:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        scores = scores[torch.from_numpy(idx).to(scores.device)]
    np.save(os.path.join(directory, name + ".npy"), scores.float().cpu().numpy())


def run_ours(args):
    rank, local_rank, world = dist_env()
    prev_affinity, numa_note = (None, "not bound (--no-numa-bind)") if args.no_numa_bind \
        else bind_to_gpu_numa(local_rank)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from sparrowrecsys_b200 import _lib
    from sparrowrecsys_b200.features import encode_batch, synthetic_features
    from sparrowrecsys_b200.model import CTRModel
    from sparrowrecsys_b200.spec import baseline_spec

    lib = _lib.load()
    spec = baseline_spec(args.workload)
    B = args.batch
    W, _table = make_weights(spec, dev)               # same weights on every rank (replicated)
    model = CTRModel(spec, W, device=local_rank)
    T = model.hist_cols
    uniform_hist = (args.history == "uniform") if args.history else args.workload == "cfg5_din"   # worst case for the 25.6 GB table: defeats L2

    # ---- resident dataset: R distinct batches, footprint >> L2 ----------------------
    probe = encode_batch(spec, synthetic_features(spec, 8, seed=0))
    cols = [a for a in (probe.movie_id, probe.user_id, probe.hist, probe.movie_genre,
                        probe.user_genre, probe.numerics) if a is not None]
    bytes_per_row = sum(a.nbytes for a in cols) // 8 + 4          # inputs + the score written back
    bytes_per_batch = B * bytes_per_row
    min_ring = max(2, int(np.ceil(1.25 * L2_BYTES / bytes_per_batch)))
    if args.dataset_batches:
        ring = max(2, args.dataset_batches)
    else:
        ring = min(4096, max(min_ring, min(512, int(1.5e9 // bytes_per_batch))))
    gen = min(ring, max(2, min(min_ring, 160)))                   # batches generated on the host, then tiled
    reps = (ring + gen - 1) // gen
    feats = synthetic_features(spec, gen * B, seed=1000 + rank, uniform_history=uniform_hist)
    enc0 = encode_batch(spec, feats)                  # each rank scores its own user-batches
    enc = tile_encoded(enc0, reps, np.random.default_rng(77 + rank))
    d = model.to_device(enc)                          # one big device allocation per column
    out = torch.empty(ring, B, dtype=torch.float32, device=dev)
    ptr = lambda t, lo, width: None if t is None else t.data_ptr() + 4 * lo * width
    structs = []
    for i in range(ring):
        lo = i * B
        structs.append(_lib.SrsBatch(B, T, ptr(d.movie_id, lo, 1), ptr(d.user_id, lo, 1),
                                     ptr(d.hist, lo, max(T, 1)), ptr(d.movie_genre, lo, 3),
                                     ptr(d.user_genre, lo, 5), ptr(d.numerics, lo, 7)))
    out_ptrs = [out[i].data_ptr() for i in range(ring)]
    handle = model._h

    def launch(i, stream_ptr):
        rc = lib.srs_predict_device(handle, C.byref(structs[i % ring]), out_ptrs[i % ring], None,
                                    stream_ptr)
        if rc != 0:
            _lib.check(rc)

    gather_mode = args.gather if distributed else None
    gather_buf = None
    gather_note = "no data-path collective"
    extra_launches_per_batch = 0
    if gather_mode == "nccl":
        gather_buf = torch.empty(world * B, dtype=torch.float32, device=dev)
        gather_note = "torch NCCL all_gather_into_tensor of the scores after every launch"
    elif gather_mode == "fused":
        from sparrowrecsys_b200 import sharding
        fused = sharding.FusedScoreGather(model, B, dev)           # symmetric buffers + peer pointers
        gather_note = fused.describe()
        extra_launches_per_batch = 1                               # the one-warp wait kernel

        # The forward kernels run back to back on the launch stream; the wait for the N slices of step i - what a
        # consumer of the gathered scores does - runs on a second stream.  Forward i + 2 reuses the gather buffer
        # of step i, so it waits for that step's wait (two buffers alternate).
        wait_stream = torch.cuda.Stream(device=dev)
        fwd_done = [torch.cuda.Event() for _ in range(2)]
        waited = [torch.cuda.Event() for _ in range(2)]
        fused_state = {"n": 0}

        def launch(i, stream_ptr):                                 # noqa: F811 - the gathering launch
            n = fused_state["n"]
            cur = torch.cuda.current_stream()
            if n >= 2:
                cur.wait_event(waited[n & 1])                      # the consumer is done with this buffer
            fused.predict(structs[i % ring], stream_ptr, wait=False)
            fwd_done[n & 1].record(cur)
            wait_stream.wait_event(fwd_done[n & 1])
            fused.wait(wait_stream.cuda_stream)
            waited[n & 1].record(wait_stream)
            fused_state["n"] = n + 1

    stream = torch.cuda.Stream(device=dev)
    S = max(1, args.streams) if gather_mode is None else 1
    n_sms = torch.cuda.get_device_properties(dev).multi_processor_count
    side = [torch.cuda.Stream(device=dev) for _ in range(S - 1)]
    half_sm_kernel = False                                         # (no kernel fits two CTAs per SM at present)
    if args.sm_limit is not None:
        sm_limit = args.sm_limit
    else:
        sm_limit = 0 if (half_sm_kernel or S == 1) else max(1, n_sms // S)
    if S > 1:
        model.set_sm_limit(sm_limit)
    graph = None
    launch_mode = "%d direct launches per step" % ring
    with torch.cuda.stream(stream):
        for i in range(min(8, ring)):                 # first touches / module load
            launch(i, stream.cuda_stream)
            if gather_buf is not None:
                dist.all_gather_into_tensor(gather_buf, out[i % ring])     # communicator set-up outside the capture
        stream.synchronize()
        if not args.no_graph and gather_mode != "nccl":   # (capturing the NCCL all-gathers hung on the box: direct launches)
            try:
                g = torch.cuda.CUDAGraph()
                if gather_mode == "fused":
                    torch.cuda.synchronize()
                    fused_state["n"] = 0                  # no waits on events recorded outside the capture
                with torch.cuda.graph(g, stream=stream):
                    cur = torch.cuda.current_stream()
                    for sd in side:                       # fork: S branches, batch i on branch i % S
                        sd.wait_stream(cur)
                    branches = [cur] + side
                    for i in range(ring):
                        launch(i, branches[i % S].cuda_stream)
                        if gather_buf is not None:
                            dist.all_gather_into_tensor(gather_buf, out[i % ring])
                    for sd in side:                       # join
                        cur.wait_stream(sd)
                    if gather_mode == "fused":
                        cur.wait_stream(wait_stream)
                graph = g
                launch_mode = "one replay per step of a CUDA graph of %d launches (one per batch of the dataset)" % ring
                if S > 1:
                    launch_mode += (", %d parallel branches, %s"
                                    % (S, "each launch limited to %d of %d SMs" % (sm_limit, n_sms) if sm_limit > 0
                                       else "no SM limit (two CTAs of this kernel share an SM)"))
            except Exception as e:                    # pragma: no cover
                sys.stderr.write("graph capture failed (%r); launching directly\n" % (e,))
                torch.cuda.synchronize()

        def run_steps(n):
            for _ in range(n):
                if graph is not None:
                    graph.replay()
                    continue
                for sd in side:
                    sd.wait_stream(stream)
                for i in range(ring):
                    launch(i, ([stream] + side)[i % S].cuda_stream)
                    if gather_buf is not None:
                        dist.all_gather_into_tensor(gather_buf, out[i % ring])
                for sd in side:
                    stream.wait_stream(sd)
                if gather_mode == "fused":
                    stream.wait_stream(wait_stream)

        run_steps(max(args.warmup, 3))
        stream.synchronize()

        sampler = ClockSampler(local_rank)
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.start()
        ev0.record(stream)
        run_steps(args.steps)
        ev1.record(stream)
        sampler.sample()                               # GPU still draining the queue
        stream.synchronize()
        sampler.sample()
        sampler.stop()
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
    model.status()                                     # no id was out of range
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "scores" if world == 1 else "scores_rank%d" % rank, out, DUMP_BYTES // world)
    if S > 1:
        model.set_sm_limit(0)                          # the host legs below are single launches again

    # ---- e2e through the C ABI with host buffers ----------------------------------
    n_slots = model.num_slots()
    e2e = {}
    latency = None
    if not args.no_e2e:
        host_b = args.host_batches or max(8, min(256, int(512e6 // max(bytes_per_batch, 1))))
        host_b = min(host_b, gen)
        hout = torch.empty(host_b, B, dtype=torch.float32).pin_memory()
        d2h = B * 4 + 4
        can_narrow = T > 0 and spec.n_movies <= 65536 and spec.model in ("din", "dien")

        def e2e_leg(narrow):
            pinned = []

            def pinned_arena(nbytes):
                t = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
                pinned.append(t)
                return t.numpy()

            hstructs = []
            hp = lambda a: None if a is None else a.ctypes.data
            for i in range(host_b):
                e = encode_batch(spec, {k: np.asarray(v)[i * B:(i + 1) * B] for k, v in feats.items()},
                                 arena_alloc=pinned_arena, narrow_ids=narrow)
                hstructs.append(_lib.SrsBatch(B, T, hp(e.movie_id), hp(e.user_id), None if narrow else hp(e.hist),
                                              hp(e.movie_genre), hp(e.user_genre), hp(e.numerics),
                                              hp(e.hist) if narrow else None))
            h2d = sum(t.numel() for t in pinned) // host_b         # bytes of one packed host batch
            arr = (_lib.SrsBatch * host_b)(*hstructs)
            outs = (C.c_void_p * host_b)(*[hout[i].data_ptr() for i in range(host_b)])

            def steps(n):
                # one library call per step scores the host dataset (the predict-over-a-dataset loop):
                # H2D / kernel / D2H of consecutive batches overlapped over the library's slots
                for _ in range(n):
                    _lib.check(lib.srs_predict_host_batches(handle, host_b, arr, outs, None))

            steps(max(2, min(args.warmup, 5)))
            if distributed:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            steps(args.steps)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            # scores that came back over PCIe equal the device-path scores of the same rows
            chk = torch.empty(B, dtype=torch.float32, device=dev)
            lib.srs_predict_device(handle, C.byref(structs[0]), chk.data_ptr(), None, None)
            torch.cuda.synchronize()
            if args.steps >= 1 and not np.array_equal(chk.cpu().numpy(), hout[0].numpy()):
                raise SystemExit("e2e scores differ from device-path scores")
            return dt, h2d, hstructs, pinned

        dt32, h2d32, hstructs32, keep32 = e2e_leg(False)
        e2e["int32"] = (dt32, h2d32)
        # ---- single-call latency (not part of the metric): one synchronous srs_predict_host ----
        try:
            lat = []
            for i in range(80):
                t1 = time.perf_counter()
                rc = lib.srs_predict_host(handle, C.byref(hstructs32[i % host_b]), hout[i % host_b].data_ptr(), None)
                lat.append((time.perf_counter() - t1) * 1e6)
                if rc != 0:
                    _lib.check(rc)
            lat = np.sort(np.array(lat[20:]))
            latency = {"median": round(float(np.median(lat)), 1), "p99": round(float(lat[-1]), 1),
                       "what": "one synchronous srs_predict_host call on a %d-row pinned host batch "
                               "(H2D, kernel, D2H, wait), nothing else in flight" % B}
        except Exception as e:                              # pragma: no cover - never fail the line for this
            sys.stderr.write("latency probe failed: %r\n" % (e,))
        del hstructs32, keep32
        if can_narrow:
            dt16, h2d16, _, _ = e2e_leg(True)
            e2e["hist16"] = (dt16, h2d16)

    # ---- reduce over ranks ------------------------------------------------------------
    times = [ms] + [v[0] for v in e2e.values()]
    if distributed:
        t = torch.tensor(times, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times = [float(x) for x in t]
    ms = times[0]
    for k, tv in zip(list(e2e), times[1:]):
        e2e[k] = (tv, e2e[k][1])
    launches = args.steps * ring
    total_rows = world * B * launches
    value = total_rows / (ms * 1e-3)

    if rank == 0:
        if prev_affinity:
            try:
                os.sched_setaffinity(0, prev_affinity)     # the CPU baseline may use every core again
            except Exception:
                pass
        peak, peak_src = measured_peaks()
        bpi = model.bytes_per_inference
        launch_us = 1e3 * ms / max(launches, 1)
        achieved = bpi * B / (launch_us * 1e-6) / 1e9
        line = {
            "metric": metric_name(args.workload), "value": value, "unit": "inferences/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.workload in FP32_WORKLOADS else DTYPE,
            "data": "synthetic",
            "config": shared_config(args, spec, world),
            "step": {"batches": ring, "rows": ring * B,
                     "what": "one predict pass over a resident dataset of %d distinct %d-row batches "
                             "(one kernel launch per batch)" % (ring, B)},
            "detail": {
                "parallelism": "dp%d: rows sharded by user-batch, weights replicated, %s" % (world, gather_note),
                "kernel": model.kernel_name, "launch": launch_mode,
                "l2": "the dataset (%d batches, %.0f MB) exceeds the 126 MB L2: ids / numerics are read from "
                      "HBM every launch; embedding tables total %.1f MB (%s)"
                      % (ring, ring * bytes_per_batch / 1e6,
                         4 * spec.emb_dim * (spec.n_movies + spec.n_users) / 1e6,
                         "L2-resident by size" if spec.n_movies < 10_000_000 else "HBM-resident, uniform ids"),
                "dataset": "%d batches generated on the host, %d row-permuted replicas" % (gen, reps),
                "numa": numa_note,
            },
            "gpu_launches": launches + extra_launches_per_batch * launches,
            "single_call_latency_us": latency,
            "clocks": sampler.summary(),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak,
                         "traffic": ncu_traffic(args.workload, model.kernel_name, B),
                         "algorithmic_bytes_per_launch": bpi * B, "launch_us": launch_us,
                         "peak_source": peak_src},
        }
        if S > 1:
            line["roofline"]["concurrency"] = (
                "%d launches in flight; launch_us is the timed region / launches (device time per "
                "batch), a single launch lasts about %d times that" % (S, S))
        if e2e:
            host_b_ = host_b

            def e2e_obj(key, what):
                dt, h2d = e2e[key]
                return {"value": world * B * host_b_ * args.steps / dt, "unit": "inferences/s",
                        "h2d_bytes_per_step": h2d * host_b_, "d2h_bytes_per_step": d2h * host_b_,
                        "h2d_bytes_per_batch": h2d, "d2h_bytes_per_batch": d2h,
                        "steps": args.steps, "batches_per_step": host_b_, "seconds": dt,
                        "how": "one srs_predict_host_batches call per step over %d pinned %d-row host batches "
                               "(pipelined over %d slots), %s, wall clock" % (host_b_, B, n_slots, what)}
            line["e2e"] = e2e_obj("int32", "int32 ids (the reference's wire types)")
            if "hist16" in e2e:
                line["e2e_hist16"] = e2e_obj("hist16", "history ids as uint16 (srs_batch::hist16) widened on "
                                                       "the device")
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block(args, spec, feats)
        emit(line)
    model.close()
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


_JSON_FD = None


def emit(line):
    """The ONE line of stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    global _JSON_FD
    # a run that an outer `timeout` ends leaves the Python stacks of all threads on stderr
    import faulthandler
    import signal
    faulthandler.register(signal.SIGTERM, all_threads=True, chain=True)
    args = parse_args()
    # stdout carries the JSON line and nothing else: whatever libraries print there (NCCL's version banner
    # comes from C code) goes to stderr instead
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
