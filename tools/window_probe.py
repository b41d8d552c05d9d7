"""Device cost of the window (lh_window_*) per snapshot.

For H = 1 (one histogram, lh_ingest_f64) and H = 1024 (keyed, uniform ids): every histogram touched, 1e8 pairs of
stream U per interval, windows of K = 60 intervals (timed once the window is full, so every fold also evicts) and
lifetime (K = 0).  CUDA events on the snapshot stream bracket

  fold    lh_window_fold: capture (K3 non-empty counts, scan, the one host synchronisation that sizes the slot,
          k_export into the slot) + k_window_apply.  The host round trip of that synchronisation is included.
  reduce  lh_window_reduce with 9 percentiles (H2D of the percentiles, K3 over the accumulator, the packed D2H)
  snap    lh_snapshot_reduce of the same snapshot, for comparison

Prints the card name and power limit read in the same run, then one line per configuration.

    python tools/window_probe.py [--intervals 8] [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import loghisto_b200 as lh  # noqa: E402

PS = [0.0, 0.5, 0.75, 0.9, 0.95, 0.99, 0.999, 0.9999, 1.0]
N = 100_000_000


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:   # report what could be read
        q = "nvidia-smi unavailable (%s)" % ex
    return "%s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), q)


def run(H, K, timed):
    import torch
    with lh.Engine(device=0, max_histograms=H, max_counters=1) as e:
        d_v = e.gen_stream(lh.STREAM_U, N, lh.DEFAULT_SEED)
        d_i = e.gen_ids_u16(0, N, H, lh.DEFAULT_SEED) if H > 1 else None
        e.window_configure(K)
        warm = (K if K else 2) + 1
        ext, fold, red, snap = None, [], [], []
        for it in range(warm + timed):
            if H > 1:
                e.ingest_keyed_f64_u16(d_i, d_v, N)
            else:
                e.ingest_f64(0, d_v, N)
            e.snapshot_begin()
            v = e.snapshot_device()
            if ext is None:
                ext = torch.cuda.ExternalStream(int(v.stream), device=0)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
            ev[0].record(ext)
            e.snapshot_reduce(PS)
            ev[1].record(ext)
            ev[2].record(ext)
            e.window_fold()
            ev[3].record(ext)
            ev[4].record(ext)
            r = e.window_reduce(PS)
            ev[5].record(ext)
            e.snapshot_end()
            ev[5].synchronize()
            if it >= warm:
                snap.append(ev[0].elapsed_time(ev[1]))
                fold.append(ev[2].elapsed_time(ev[3]))
                red.append(ev[4].elapsed_time(ev[5]))
        info = e.window_info()
        held = info["held"]
        assert int(r.counts.sum()) == held * N, (int(r.counts.sum()), held * N)
        assert int((r.counts != 0).sum()) == H
        return fold, red, snap, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--intervals", type=int, default=8, help="timed snapshots per configuration")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = ["card: " + card(),
             "pairs per interval: %d (stream U, every histogram touched); times in ms, median [min, max] of %d snapshots"
             % (N, a.intervals)]
    for H in (1, 1024):
        for K in (60, 0):
            fold, red, snap, info = run(H, K, a.intervals)
            f = lambda x: "%.4f [%.4f, %.4f]" % (float(np.median(x)), min(x), max(x))
            lines.append("H=%-4d K=%-8s fold %s | window_reduce %s | snapshot_reduce %s | held %d, entries_held %d, device %.1f MB"
                         % (H, K if K else "lifetime", f(fold), f(red), f(snap), info["held"], info["entries_held"],
                            info["device_bytes"] / 1e6))
    text = "\n".join(lines)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
