#!/usr/bin/env python
"""bench.py -- loghisto hot path on B200: samples/s, HBM roofline fraction, CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3] [--impl b200|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic float64
samples: ingest (bucket index + increment) of the whole batch, then the
snapshot (double-buffer swap, bucket-array all-reduce when N > 1) and the
bucket->percentile reduction, result read back to the host.

  value      whole-job samples/s with the batch already resident in HBM
  e2e        same steps fed from pinned HOST memory through lh_ingest_f64_host
             (H2D copies inside the timed region)
  roofline   the dominant kernel (K1 ingest) alone: 8 B/sample (10 B for c3)
             over its CUDA-event duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the CPU oracle port of metrics.go:273-295 timed on this box's
             host cores over a bounded sample (N=1, rank 0 only)

--impl reference times that CPU port alone (the Go reference cannot be built
here: no Go toolchain in the image; see DESIGN.md).

--dump-outputs DIR writes what the last timed step returned (counts, sums,
avgs, pkeys, pvals of every histogram) as DIR/<name>.npy, float64.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0x10C415C0
PERCENTILES = [0.0, 0.5, 0.75, 0.9, 0.95, 0.99, 0.999, 0.9999, 1.0]   # metrics.go:145-155
PUBLISHED_SAMPLES_PER_S = 2.0171025e7   # readme.md:34, the reference's only published ingest rate
FALLBACK_HBM_GBS = 6650.0               # /opt/skills/guides/B200_PROFILING.md


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c3", "c5", "c4x1"],
                    help="c2 = configs[1] (default), c3 = configs[2] (1024 keyed), c5 = configs[4] (mixed ops), "
                         "c4x1 = the north-star target: the 1e10-sample stream of configs[3] resident on ONE GPU (80 GB)")
    ap.add_argument("--stream", default="U", choices=["U", "L", "S", "C", "Z"])
    ap.add_argument("--n", "--samples-per-gpu", dest="n", type=int, default=0, help="samples per GPU per step (default: BASELINE config)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps for the host-fed leg (default min(steps, 5))")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-api", action="store_true", help="skip the per-call API leg (MetricSystem.Histogram / StartTimer+Stop)")
    ap.add_argument("--no-parity", action="store_true", help="skip the bucket-for-bucket oracle check after the timed legs")
    ap.add_argument("--sustain-seconds", type=float, default=-1.0,
                    help="extra leg of back-to-back steps for at least this long (default 2 s for c2/c4x1 at N=1, else 0)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--k1-grid-mult", type=int, default=0, help="override the K1 waves-per-launch tuning")
    ap.add_argument("--k1-variant", type=int, default=-1)
    ap.add_argument("--pipeline-depth", type=int, default=-1,
                    help="snapshots in flight behind the next ingest: 0 = blocking snapshot after every batch, 1, 2 (default 2)")
    ap.add_argument("--collective", default="peer", choices=["nccl", "peer"],
                    help="N>1: peer (default) = the library's own peer-memory all-reduce kernel behind the C ABI "
                         "(lh_comm_*); nccl = torch.distributed all-reduce of the frozen arrays, kept for comparison "
                         "(and the automatic fallback if the peer mappings cannot be made)")
    ap.add_argument("--keyed-mode", type=int, default=-1)
    ap.add_argument("--debug-steps", action="store_true", help="print every timed step's kernel time to stderr")
    ap.add_argument("--nccl-defaults", action="store_true", help="do not set NCCL_MAX_NCHANNELS / NCCL_CGA_CLUSTER_SIZE")
    ap.add_argument("--reserve-sms", type=int, default=-1, help="SMs K1 leaves free for the snapshot stream (default: 0 at N=1, 2 at N>1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (the reduction of every "
                         "histogram) as DIR/<name>.npy in float64; the inputs are a function of the arguments only, "
                         "so two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl b200: the reference arm hands no arrays back")
    return a


def measured_traffic(workload, n):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, if one matches this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f).get(workload)
        if t and int(t["samples"]) == int(n):
            return int(t["bytes"]), t["source"]
    except Exception:
        pass
    return None, None


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock, power and throttle reasons through NVML every ~2 ms while the timed region runs
    (nvidia-smi -lms cannot resolve a region this short)."""

    def __init__(self, device_index):
        import threading
        self.rows = []
        self.stop_flag = False
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            idx = device_index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[device_index])
                except Exception:
                    idx = device_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                self.rows.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.ok:
            return out
        self.stop_flag = True
        self.t.join(timeout=2)
        nv = self.nv
        rows = self.rows
        if not rows:
            out["sm_max_mhz"] = self.max_sm
            return out
        sm = sorted(r[0] for r in rows)
        flags = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        reasons = sorted(k for k, bit in flags.items() if any(r[2] & bit for r in rows))
        out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=self.max_sm, reasons=reasons, samples=len(rows),
                   power_w_max=max(r[1] for r in rows), sm_mhz_min=sm[0])
        return out


# ----------------------------------------------------------------- CPU arm
def cpu_quota_cores():
    """CPU time this container may use, in cores (cgroup v2 cpu.max; the pool's boxes show 128 CPUs under a 16-core
    quota), or the CPU count when there is no quota."""
    ncpu = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            return max(1, min(ncpu, int(round(int(quota) / int(period)))))
    except Exception:
        pass
    return ncpu


def _thread_ladder():
    ncpu = os.cpu_count() or 1
    q = cpu_quota_cores()
    return sorted({1, min(2, ncpu), min(4, ncpu), min(16, ncpu), min(q, ncpu), min(2 * q, ncpu), ncpu})


def _calibrate_cpu_port(o, kind, n_hist, names):
    """The port's shared reader count and bucket cells ping-pong between cores (as the reference's RWMutex and
    atomics do), so more threads is not always faster: probe a ladder of thread counts and keep the best."""
    # long enough (>= 0.25 s) that the scheduler has spread the threads over distinct cores
    probe = 8_000_000
    vals = o.gen_stream(kind, probe, SEED)
    ids = o.gen_ids(0, probe, n_hist, SEED) if n_hist > 1 else None
    best = (0.0, 1)
    ladder = {}
    for t in _thread_ladder():
        ms = o.OracleMetricSystem()
        ms.bench_ingest(vals[:100_000], ids[:100_000] if ids is not None else None, names, t)   # create the cells
        dt = ms.bench_ingest(vals, ids, names, t)
        ms.close()
        ladder[t] = probe / dt
    top = max(ladder.values())
    # ties go to the smaller thread count: short probes can flatter contended runs (the scheduler has not yet
    # spread the threads over distinct cores), and fewer threads is never slower for this lock-bound port
    threads = min(t for t, r in ladder.items() if r >= 0.95 * top)
    best = (ladder[threads], threads)
    return best[0], best[1], ladder


def cpu_port_rate(n_hist, stream_kind, seconds):
    """Times the oracle's structure-faithful port of MetricSystem.Histogram (metrics.go:273-295: Go-style
    RWMutex + name->map[int16] lookups + atomic add, Go-exact compress) on a bounded sample of the same
    synthetic stream, at the thread count that runs fastest on this host.
    Returns (samples_per_s, threads, n_sample, dense_rate, ladder)."""
    from oracle import oracle as o
    o.build()
    names = ["histogram%d" % i for i in range(n_hist)]
    rate, threads, ladder = _calibrate_cpu_port(o, stream_kind, n_hist, names)
    n = int(min(max(rate * seconds, 1_000_000), 400_000_000))
    vals = o.gen_stream(stream_kind, n, SEED)
    ids = o.gen_ids(0, n, n_hist, SEED) if n_hist > 1 else None
    ms = o.OracleMetricSystem()
    dt = ms.bench_ingest(vals, ids, names, threads)
    ms.close()
    # "best-case CPU" (dense private arrays, no locks/maps, every core) for context
    m = min(n, 50_000_000)
    t0 = time.perf_counter()
    o.ingest(vals[:m], threads=os.cpu_count() or 1)
    dense = m / (time.perf_counter() - t0)
    return n / dt, threads, n, dense, ladder


def run_reference(a):
    """--impl reference: the reference's CPU implementation of the path on the host cores, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as o
    o.build()
    n_hist = 1024 if a.workload in ("c3", "c5") else 1
    kind = {"U": 0, "L": 1, "S": 2, "C": 3, "Z": 4}[a.stream]
    names = ["histogram%d" % i for i in range(n_hist)]
    rate, threads, ladder = _calibrate_cpu_port(o, kind, n_hist, names)
    n = int(min(max(rate * 1.0, 1_000_000), 200_000_000))     # about 1 s of CPU work per step
    vals = o.gen_stream(kind, n, SEED)
    ids = o.gen_ids(0, n, n_hist, SEED) if n_hist > 1 else None
    ms = o.OracleMetricSystem()
    for _ in range(a.warmup):
        ms.bench_ingest(vals, ids, names, threads)
        ms.collect_and_process()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        ms.bench_ingest(vals, ids, names, threads)
        ms.collect_and_process()          # snapshot + percentile reduction, like one b200 step
    dt = time.perf_counter() - t0
    ms.close()
    value = n * a.steps / dt
    unit = "samples/s"
    print(json.dumps({
        "impl": "reference", "metric": "histogram ingest throughput (samples/s)", "value": value, "unit": unit,
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": value / PUBLISHED_SAMPLES_PER_S,
        "dtype": "f64", "data": "synthetic",
        # the same config object as the b200 arm prints for this N; the CPU arm processes a bounded sample of that
        # workload per step and reports a RATE (samples/s), hence rate_normalised
        "config": workload_config(a, a.n or default_n(a.workload, a.gpus), a.gpus),
        "rate_normalised": True, "sample": "bounded sample of %d samples per step (about 1 s of CPU work)" % n,
        "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port",
                         "host_cpus": os.cpu_count(), "cpu_quota_cores": cpu_quota_cores(), "thread_ladder_samples_per_s": ladder,
                         "sample": "%d samples/step x %d steps, stream %s, %d name(s); C port of "
                                   "metrics.go:273-295 incl. Go's RWMutex algorithm (Go toolchain absent), run at "
                                   "the fastest thread count of the ladder" % (n, a.steps, a.stream, n_hist)},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def workload_config(a, n_per_gpu, n_gpus):
    if a.workload == "c2":
        name = ("BASELINE configs[1]: 1 GPU, 1 histogram, 1e9-sample synthetic float64 stream" if n_gpus == 1 else
                "BASELINE configs[3] slice: %d GPU(s), 1 histogram, %d samples per GPU, bucket-array all-reduce "
                "before percentiles" % (n_gpus, n_per_gpu))
    elif a.workload == "c4x1":
        name = ("north_star target: the 1e10-sample synthetic float64 stream of BASELINE configs[3] resident on ONE GPU "
                "(80 GB), 1 histogram, bit-exact bucket counts")
    elif a.workload == "c5":
        name = ("BASELINE configs[4]: mixed ops, 50% Histogram (u16 id, f64) / 25% Timer (u16 id, int64 ns) / 25% Counter "
                "(u16 id, u64 amount 1..16) over 1024 names, one percentile snapshot per batch of ops "
                "(1e8 ops = 100 ms of traffic at the nominal 1e9 ops/s)")
    else:
        name = "BASELINE configs[2]: 1024 keyed histograms, (uint16 id, float64 value) pairs"
    single = a.workload in ("c2", "c4x1")
    return {"workload": name, "stream": a.stream, "samples_per_gpu_per_step": n_per_gpu,
            "histograms": 1 if single else 1024, "percentiles": len(PERCENTILES),
            "l2": "inputs (%.1f GB per GPU) are larger than the 126 MB L2; no flush needed"
                  % (n_per_gpu * (8 if single else 10) / 1e9),
            "published_ref": "readme.md:34 (2014, unnamed CPU, Timer path incl. two time.Now() per sample)"}


# ----------------------------------------------------------------- parity
def oracle_parity(a, eng, sharded, ingest, world, rank, n, H, kind, timed_red):
    """Bucket-for-bucket check of the device path against the CPU oracle at the FULL size of this run, outside
    every timed region.  All ranks ingest their batch once more and take a snapshot with export (the same
    kernels, the same collective); rank 0 regenerates the whole index range on every host core with the oracle
    (oracle/loghisto_oracle.c: compress = metrics.go:316-322, Histogram = :273-295, Counter = :251-269,
    processHistograms/percentile = :336-418) and compares every bucket of every histogram, every counter, and the
    percentile bucket keys -- of the verification step AND of the last timed step."""
    import numpy as np
    mixed = a.workload == "c5"
    keyed = a.workload == "c3"
    t0 = time.perf_counter()
    ingest(None)
    red, sp = sharded.snapshot(PERCENTILES, export=True, counters=mixed)
    if rank != 0:
        return None
    from oracle import oracle as o
    o.build()
    got = np.zeros((H, 65536), dtype=np.uint64)
    ent_h = np.repeat(np.arange(H), np.diff(sp.offsets.astype(np.int64)))
    got[ent_h, sp.keys.view(np.uint16)] = sp.counts
    t1 = time.perf_counter()
    counters_equal = None
    if mixed:
        nh, nt = n // 2, n // 4
        nc = n - nh - nt
        want = np.zeros((H, 65536), dtype=np.uint64)
        want_c = np.zeros(1024, dtype=np.uint64)
        for r in range(world):
            b = r * n
            o.stream_ingest_keyed(kind, nh, H, SEED, val_start=b, ids_start=b, counts=want)
            o.stream_ingest_keyed(o.STREAM_TIMER_NS, nt, H, SEED, val_start=b + nh, ids_start=b + nh, as_i64=True, counts=want)
            o.stream_counter(nc, 1024, SEED, val_start=b + nh + nt, ids_start=b + nh + nt, counters=want_c)
        counters_equal = bool((sp.counter_deltas == want_c).all())
        n_checked = n * world
    elif keyed:
        want = o.stream_ingest_keyed(kind, n * world, H, SEED, val_start=0, ids_start=0)
        n_checked = n * world
    else:
        want = o.stream_ingest(kind, n * world, SEED, start=0).reshape(1, 65536)
        n_checked = n * world
    t2 = time.perf_counter()
    buckets_equal = bool((got == want).all())
    pkeys_equal = True
    counts_equal = True
    pvals_equal = True
    for h in range(H):
        ref = o.process_histogram(want[h], PERCENTILES)
        for r_ in (red, timed_red):
            if int(r_.counts[h]) != ref["total"]:
                counts_equal = False
            if ref["total"] and not (r_.pkeys[h] == ref["pkeys"]).all():
                pkeys_equal = False
            if ref["total"] and not (r_.pvals[h].view(np.uint64) == ref["pvals"].view(np.uint64)).all():
                pvals_equal = False
    out = {"buckets_equal": buckets_equal, "pkeys_equal": pkeys_equal, "counts_equal": counts_equal,
           "pvals_bit_equal": pvals_equal, "n_checked": n_checked, "histograms_checked": H,
           "nonempty_buckets": int((want != 0).sum()), "mismatching_buckets": int((got != want).sum()),
           "oracle": "oracle/loghisto_oracle.c regenerating indices [0, %d) on %d host threads (%.1f s); device side: "
                     "one more step of the same batch + snapshot export after the all-reduce, and the percentile keys "
                     "of the last timed step" % (n_checked, os.cpu_count() or 1, t2 - t1),
           "seconds": time.perf_counter() - t0}
    if counters_equal is not None:
        out["counters_equal"] = counters_equal
    out["ok"] = bool(buckets_equal and pkeys_equal and counts_equal and pvals_equal and counters_equal is not False)
    return out


# ----------------------------------------------------------------- per-call API leg
def api_leg(device, kind):
    """The reference's one published number (readme.md:34: 2.0171e7 timer samples/s) is a PER-CALL rate: goroutines
    looping StartTimer/Stop (print_benchmark.go:59-67).  This leg drives the same loop, and a plain
    Histogram(name, value)-per-sample loop, through the C++ MetricSystem mirror above the C ABI (one OS thread per
    goroutine; thread-local name cache, one pinned staging shard per thread, batches committed to the GPU)."""
    from loghisto_b200.metric_system import MetricSystem, timer_loop
    ncpu = os.cpu_count() or 1
    out = {"published_reference_samples_per_s": PUBLISHED_SAMPLES_PER_S,
           "published_reference_source": "readme.md:34 (StartTimer/Stop from 100 goroutines, 2014, unnamed CPU)"}
    rate, calls, reported = timer_loop("benchmark1234", 100, 3.0, 0.1, device)
    out["timer_loop"] = {"value": rate, "unit": "calls/s", "threads": 100, "op": "StartTimer + Stop (print_benchmark.go:59-67, empty op)",
                         "calls": calls, "reported_count": reported, "count_ok": float(calls) == reported, "host_cpus": ncpu}
    n_api = 1_000_000_000
    # twice the CPU quota: enough runnable threads to use every core the container is allowed, not so many that the
    # quota throttles them in bursts (measured: profiles/r02/api_probe_r02h.txt)
    ncpu = min(ncpu, 2 * cpu_quota_cores())
    out["cpu_quota_cores"] = cpu_quota_cores()
    ms = MetricSystem(3600.0, False, device=device, max_histograms=16, max_counters=16)
    k = kind if kind in (0, 1) else 0
    # pass 0 warms the staging ring up (every shard pins its slots on first use: cudaMallocHost is slow); pass 1 is reported
    passes = []
    for i in range(2):
        wall, in_calls = ms.histogram_stream_timed(["benchmark1234"], k, SEED, i * n_api, n_api, ncpu)
        raw, metrics = ms.collect_and_process()
        got = sum(raw["Histograms"].get("benchmark1234", {}).values())
        passes.append({"calls_per_s": n_api / wall, "call_loops_only": n_api / in_calls, "count_ok": got == n_api})
    out["histogram_calls"] = {"value": passes[1]["calls_per_s"], "unit": "calls/s", "threads": ncpu, "calls": n_api,
                              "op": "MetricSystem.Histogram(name, value), one call per sample, 1 name",
                              "timed": "wall clock over all threads, the synthetic value generator included",
                              "call_loops_only_calls_per_s": passes[1]["call_loops_only"],
                              "call_loops_only_timed": "largest per-thread time inside the Histogram() call loops (blocks of 1024 "
                                                       "pre-generated samples): the API path without the generator",
                              "count_ok": all(p_["count_ok"] for p_ in passes), "warmup_pass_calls_per_s": passes[0]["calls_per_s"],
                              "dropped": ms.dropped()}
    ms.close()
    return out


# ----------------------------------------------------------------- GPU arm
def dump_outputs(out_dir, red):
    """Writes the Reduced of one snapshot, every field as float64: H x (at most 32 percentiles) values, far below 64 MB,
    so nothing is sampled.  int32 keys convert exactly, and so do the uint64 counts (below 2^53 at any bench size)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name in ("counts", "sums", "avgs", "pkeys", "pvals"):
        np.save(os.path.join(out_dir, name + ".npy"), getattr(red, name).astype(np.float64))


def default_n(workload, world):
    if workload == "c5":
        return 100_000_000
    if workload == "c4x1":
        return 10_000_000_000
    if workload == "c3" or world == 1:
        return 1_000_000_000
    return 1_250_000_000


def run_b200(a):
    import numpy as np
    import torch
    import loghisto_b200 as lh

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("bench.py --gpus %d must be launched with torch.distributed.run (one rank per GPU)" % a.gpus)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the b200 arm has no CPU fallback (use --impl reference)")
    if a.workload == "c4x1" and world != 1:
        raise SystemExit("bench.py: c4x1 is the single-GPU 1e10-sample run; use c2 with --gpus N for the sharded form")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")   # the bucket all-reduce outranks the ingest kernel
        # Measured (profiles/r01/scaling_r01.txt): up to 4 ranks the 512 KiB all-reduce is fastest with few channels
        # and no CTA clusters (its CTAs then fit the 2 SMs the ingest kernel leaves free); with 8 ranks those limits
        # turn pathological (3.37 ms/step) and NCCL's own choices plus 8 free SMs are best (1.58 ms/step).
        if a.collective == "nccl" and not a.nccl_defaults and world <= 4:
            os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
            os.environ.setdefault("NCCL_CGA_CLUSTER_SIZE", "0")
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    keyed = a.workload == "c3"
    mixed = a.workload == "c5"
    single = not (keyed or mixed)
    n = a.n or default_n(a.workload, world)
    H = 1 if single else 1024
    kind = {"U": 0, "L": 1, "S": 2, "C": 3, "Z": 4}[a.stream]
    bytes_per_sample = 8 if single else 10

    eng = lh.Engine(device=local, max_histograms=H, max_counters=1024 if mixed else 1)
    if a.k1_grid_mult:
        eng.tune("k1_grid_mult", a.k1_grid_mult)
    if a.k1_variant >= 0:
        eng.tune("k1", a.k1_variant)
    if a.keyed_mode >= 0:
        eng.tune("keyed_mode", a.keyed_mode)
    depth = a.pipeline_depth if a.pipeline_depth >= 0 else 2
    peer = world > 1 and a.collective == "peer"
    # SMs the ingest kernels leave to the snapshot stream: 1 with the peer collective (its small-payload form needs
    # one; its large-payload form goes wide for ~0.2 ms between two ingest kernels instead of hiding on a few SMs, where
    # an SM's ~4 GB/s of NVLink loads would make it slower than the step).  NCCL needs 2 (N <= 4) or 8 SMs.
    if a.reserve_sms >= 0:
        reserve = a.reserve_sms
    elif depth == 0:
        reserve = 0
    elif world == 1:
        reserve = 1
    elif peer:
        reserve = 1
    else:
        reserve = 2 if world <= 4 else 8
    if reserve:
        eng.tune("k1_reserve_sms", reserve)
    # launch on the context's own non-blocking ingest stream (torch's legacy default stream serialises against
    # other streams); torch only wraps it so that torch.cuda.Event can time the region on the launching stream
    stream = torch.cuda.ExternalStream(eng.ingest_stream, device=local)
    d_vals = eng.alloc(n, np.float64)
    slab = 1_000_000_000
    for off in range(0, n, slab):        # generated in 1e9-sample slabs (identical bits: the stream is a function of the index)
        m = min(slab, n - off)
        eng._check(eng.lib.lh_gen_stream_f64(eng.h, kind, SEED, rank * n + off, m, d_vals.offset(off), stream.cuda_stream))
    d_ids = eng.gen_ids_u16(0, n, H, SEED, start=rank * n, stream=stream) if (keyed or mixed) else None
    nh = nt = nc = 0
    if mixed:
        # one batch = n ops: [0, n/2) Histogram, [n/2, 3n/4) Timer (int64 ns), [3n/4, n) Counter; ids cover all three
        nh, nt = n // 2, n // 4
        nc = n - nh - nt
        d_ns = eng.alloc(nt, np.int64)
        eng._check(eng.lib.lh_gen_stream_f64(eng.h, 6, SEED, rank * n + nh, nt, d_ns.ptr, stream.cuda_stream))
        d_amt = eng.alloc(nc, np.uint64)
        eng._check(eng.lib.lh_gen_stream_f64(eng.h, 7, SEED, rank * n + nh + nt, nc, d_amt.ptr, stream.cuda_stream))
    torch.cuda.synchronize()

    from loghisto_b200.distributed import ShardedEngine
    sharded = ShardedEngine(eng, local, collective=a.collective if world > 1 else "none")
    kernel_ms = []
    allreduce_ms = []
    launches_per_step = 2 if mixed else 1

    def ingest(host_src=None):
        if mixed and host_src is not None:
            hv_, hi_, hns_, hamt_ = host_src
            eng.ingest_keyed_f64_u16_host(hi_[:nh], hv_, nh)
            eng.ingest_keyed_i64ns_u16_host(hi_[nh:nh + nt], hns_, nt)
            eng.counter_add_u16_host(hi_[nh + nt:], hamt_, nc)
            return
        if mixed:   # Histogram + Timer samples in one call (one launch of the write-combining kernel), then the counter ops
            eng.ingest_keyed_pair_u16(d_ids, d_vals, nh, d_ids.offset(nh), d_ns, nt, stream=stream)
            eng.counter_add_u16(d_ids.offset(nh + nt), d_amt, nc, stream=stream)
            return
        if host_src is None:
            if keyed:
                eng.ingest_keyed_f64_u16(d_ids, d_vals, n, stream=stream)
            else:
                eng.ingest_f64(0, d_vals, n, stream=stream)
        else:
            if keyed:
                eng.ingest_keyed_f64_u16_host(host_src[1], host_src[0], n)
            else:
                eng.ingest_f64_host(0, host_src, n)

    def run_steps(k, host_src=None, record=False):
        """k steps.  Step i = ingest of batch i, then its snapshot (buffer swap, all-reduce, percentile
        reduction, D2H of the results).  Snapshots are only ENQUEUED (high-priority stream, the frozen one of the
        two buffers); the host launches batch i+1 right away and collects snapshot i-1's results, so the GPU
        never idles on a host round trip -- the same overlap loghisto's reaper gets by handing processMetrics
        to a worker (metrics.go:583-587).  Device-side ordering keeps the semantics exact: batch i+2 waits
        (event) until snapshot i has drained and zeroed its buffer.  All k ingests and all k snapshots complete
        inside the call."""
        red = None
        pending = []          # (handle, ingest seq) of snapshots whose results are still on their way

        def collect(entry):
            h, seq = entry
            r = sharded.result(h)
            if record and host_src is None:
                # CUDA events around that batch's ingest kernel(s); the mixed batch is three launches
                kernel_ms.append(sum(eng.kernel_ms(seq - j) for j in range(launches_per_step)))
                if world > 1:
                    allreduce_ms.append(sharded.allreduce_ms(h))
            return r

        if depth == 0:
            # blocking form: ingest, then the whole snapshot, then the next ingest (nothing overlaps)
            for i in range(k):
                ingest(host_src)
                red = collect((sharded.snapshot_async(PERCENTILES, counters=mixed), eng.ingest_seq()))
            return red
        ingest(host_src)
        for i in range(k):
            seq = eng.ingest_seq()
            nxt = (lambda: ingest(host_src)) if i + 1 < k else None     # batch i+1 goes out right after the swap
            pending.append((sharded.snapshot_async(PERCENTILES, counters=mixed, after_swap=nxt), seq))
            if len(pending) >= depth:
                red = collect(pending.pop(0))
        while pending:
            red = collect(pending.pop(0))
        return red

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(k, host_src=None, record=False):
        """k steps bracketed by barrier + synchronize on both sides; device events on the launching stream and the
        host clock both cover the region (the snapshot leg ends host-synchronously), the larger one is reported;
        max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        red = run_steps(k, host_src, record)
        e1.record(stream)
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        return red, max_over_ranks(max(e0.elapsed_time(e1), wall))

    # ---- device-resident leg
    run_steps(max(a.warmup, 3))
    del allreduce_ms[:]
    del kernel_ms[:]
    launches0 = eng.stats()["kernel_launches"]
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    red, total_ms = timed(a.steps, record=True)
    clk = clocks.stop() if clocks else None
    launches = eng.stats()["kernel_launches"] - launches0
    kms = sum(kernel_ms) / len(kernel_ms)
    if a.debug_steps and rank == 0:
        sys.stderr.write("kernel_ms per step: %s\ntotal_ms %.3f\n" % (" ".join("%.3f" % x for x in kernel_ms), total_ms))
    ar_ms = (sum(allreduce_ms) / len(allreduce_ms)) if allreduce_ms else 0.0
    count_ok = int(red.counts.sum()) == (n - nc if mixed else n) * world

    # ---- sustained leg: back-to-back steps for >= S seconds; the rate over the SECOND half is the sustained figure
    sus = None
    s_seconds = a.sustain_seconds if a.sustain_seconds >= 0 else (2.0 if (single and world == 1) else 0.0)
    if s_seconds > 0:
        ms_step = total_ms / a.steps
        half = max(4, int(s_seconds * 500.0 / ms_step) + 1)
        del kernel_ms[:]
        _, ms_a = timed(half, record=False)
        clocks2 = ClockSampler(local) if rank == 0 else None
        _, ms_b = timed(half, record=True)
        clk2 = clocks2.stop() if clocks2 else None
        kms_s = sum(kernel_ms) / len(kernel_ms)
        sus = {"seconds": (ms_a + ms_b) / 1e3, "steps": 2 * half, "ms_per_step_first_half": ms_a / half,
               "ms_per_step": ms_b / half, "kernel_ms": kms_s, "clocks": clk2}
        del kernel_ms[:]

    # ---- host-fed leg (e2e)
    e2e = None
    paced = None
    if not a.no_e2e and a.workload != "c4x1":
        ksteps = a.e2e_steps or min(a.steps, 5)
        pinned_bufs = []

        def to_host(dev, count, dtype):
            h_ = eng.pinned(count, dtype)
            eng._check(eng.lib.lh_memcpy_d2h(eng.h, h_.ptr, dev.ptr, count * np.dtype(dtype).itemsize))
            pinned_bufs.append(h_)
            return h_.array
        if mixed:
            hsrc = (to_host(d_vals, nh, np.float64), to_host(d_ids, n, np.uint16), to_host(d_ns, nt, np.int64), to_host(d_amt, nc, np.uint64))
            api_name = "lh_ingest_keyed_f64_u16_host + lh_ingest_keyed_i64ns_u16_host + lh_counter_add_u16_host + lh_snapshot_*"
        elif keyed:
            hsrc = (to_host(d_vals, n, np.float64), to_host(d_ids, n, np.uint16))
            api_name = "lh_ingest_keyed_f64_u16_host + lh_snapshot_* (pinned host buffers)"
        else:
            hsrc = to_host(d_vals, n, np.float64)
            api_name = "lh_ingest_f64_host + lh_snapshot_* (pinned host buffers)"
        run_steps(2, hsrc)
        red_h, e2e_ms = timed(ksteps, hsrc)
        d2h = H * 8 * 3 + H * len(PERCENTILES) * 12
        e2e = {"value": n * world * ksteps / (e2e_ms / 1e3), "unit": "ops/s" if mixed else "samples/s",
               "h2d_bytes_per_step": n * bytes_per_sample, "d2h_bytes_per_step": d2h, "steps": ksteps,
               "ms_per_step": e2e_ms / ksteps, "api": api_name,
               "count_ok": int(red_h.counts.sum()) == (n - nc if mixed else n) * world,
               "same_result_as_device_leg": bool((red_h.pkeys == red.pkeys).all() and (red_h.counts == red.counts).all())}
        if mixed and world == 1:
            # BASELINE configs[4] as stated: 1e9 ops/s SUSTAINED with a percentile snapshot every 100 ms.  50 intervals
            # paced by the wall clock; every interval feeds its 1e8 ops from pinned host memory through the host-fed
            # entry points and enqueues its snapshot; the previous interval's results are collected meanwhile.
            period, intervals = 0.1, 50
            feed_ms, late, pend = [], 0, None
            barrier()
            t_start = time.perf_counter()
            for k_ in range(intervals):
                while time.perf_counter() < t_start + k_ * period:
                    time.sleep(0.0005)
                t_a = time.perf_counter()
                ingest(hsrc)
                h_ = sharded.snapshot_async(PERCENTILES, counters=True)
                if pend is not None:
                    sharded.result(pend)
                pend = h_
                feed_ms.append((time.perf_counter() - t_a) * 1e3)
                if feed_ms[-1] > period * 1e3:
                    late += 1
            last = sharded.result(pend)
            wall = time.perf_counter() - t_start
            paced = {"intervals": intervals, "interval_ms": period * 1e3, "ops_per_interval": n,
                     "nominal_ops_per_s": n / period, "achieved_ops_per_s": n * intervals / max(wall, intervals * period),
                     "feed_and_snapshot_ms_per_interval_mean": sum(feed_ms) / len(feed_ms),
                     "feed_and_snapshot_ms_per_interval_max": max(feed_ms), "late_intervals": late, "keeps_up": late == 0,
                     "headroom": period * 1e3 / (sum(feed_ms) / len(feed_ms)),
                     "last_interval_count_ok": int(last.counts.sum()) == n - nc,
                     "fed_from": "pinned host memory, H2D inside every interval"}
        for h_ in pinned_bufs:
            h_.free()

    # ---- per-call API leg: the path an instrumented service uses (one Histogram / StartTimer+Stop call per sample)
    api = None
    if a.workload == "c2" and world == 1 and not a.no_api:
        api = api_leg(local, kind)

    # ---- parity (outside every timed region)
    parity = None
    if not a.no_parity:
        parity = oracle_parity(a, eng, sharded, ingest, world, rank, n, H, kind, red)

    rc = 0
    if rank == 0:
        peak, peak_src = peak_hbm()
        achieved = n * bytes_per_sample / (kms / 1e3) / 1e9
        traffic, traffic_src = measured_traffic(a.workload, n)
        value = n * world * a.steps / (total_ms / 1e3)
        line = {
            "metric": "mixed op throughput (ops/s)" if mixed else "histogram ingest throughput (samples/s)",
            "value": value, "unit": "ops/s" if mixed else "samples/s",
            "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": total_ms / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": value / PUBLISHED_SAMPLES_PER_S,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(a, n, world),
            "gpu_launches": launches, "count_ok": count_ok, "clocks": clk,
            "pipeline": {"snapshots_in_flight": depth, "sms_left_free_by_ingest": reserve},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": n * bytes_per_sample,
                         "peak_source": peak_src,
                         "kernel": ("keyed ingest x2 + k_counter_add_smem (%s)" % eng.keyed_kernel_name()) if mixed else
                                   eng.keyed_kernel_name() if keyed else "k_ingest_single (%s)" % eng.k1_variant_name(),
                         "kernel_ms": kms, "bytes_per_sample": bytes_per_sample},
        }
        if world > 1:
            line["collective"] = {"kind": sharded.collective, "allreduce_ms": ar_ms,
                                  "timed": "CUDA events around the collective on the snapshot stream, one pair per step, "
                                           "warm-up pairs discarded",
                                  "bytes": sharded.allreduce_bytes()}
            if getattr(sharded, "fallback_reason", None):
                line["collective"]["fallback_from_peer"] = sharded.fallback_reason
            line["allreduce_ms"] = ar_ms
        if sus:
            v_s = n * world / (sus["ms_per_step"] / 1e3)
            a_s = n * bytes_per_sample / (sus["kernel_ms"] / 1e3) / 1e9
            line["value_sustained"] = v_s
            line["roofline"]["achieved_sustained"] = a_s
            line["roofline"]["frac_sustained"] = a_s / peak
            line["sustained"] = sus
        if e2e:
            line["e2e"] = e2e
        if paced:
            line["paced"] = paced
        if api:
            line["api_e2e"] = api
        if parity:
            line["parity"] = parity
            if not parity["ok"]:
                rc = 3
        if world == 1 and not a.no_cpu_baseline:
            rate, threads, ns, dense, ladder = cpu_port_rate(H, kind, a.cpu_seconds)
            line["cpu_baseline"] = {
                "value": rate, "unit": "samples/s", "cores": threads, "kind": "port",
                "sample": ("(mixed workload: the Histogram calls only -- Counter ops are cheaper in the reference) " if mixed else "") +
                          "%d samples of the same stream; C port of metrics.go:273-295 (RWMutex + maps + atomic add, "
                          "Go-exact compress) at the fastest rung of a thread ladder (= `cores`; more threads are slower, "
                          "the shared reader count ping-pongs as in the reference); the Go toolchain is absent so the "
                          "reference itself cannot run" % ns,
                "host_cpus": os.cpu_count(), "cpu_quota_cores": cpu_quota_cores(), "thread_ladder_samples_per_s": ladder,
                "dense_private_arrays_all_cores_value": dense}
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, red)
        print(json.dumps(line))
        sys.stdout.flush()
    eng.close()
    if dist is not None:
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
