"""Bandwidth of the tracking-quality kernel (sgx_track_quality) on a config-4 shard's tracking output.

    python tools/quick_quality_bench.py [--window 40] [--reps 20]

The input is a device-resident float64 [32, 8, 13, 37 000] tracking result (985 MB; the I_P / Q_P rows the kernel
reads are 152 MB, more than the 126 MB L2), filled with a 45 dB-Hz carrier plus Gaussian noise in I_P / Q_P so that
every estimate takes the full arithmetic path.  Each timed call has device outputs (no host synchronisation inside
the call) and is preceded, outside the timed interval, by a 256 MB device fill that evicts L2.  Time: CUDA events
around the call, median of --reps runs after 3 warm-up calls.

Algorithmic bytes: I_P + Q_P of every whole window (2 x 8 B per channel-ms) plus 17 B of outputs per window.
Reported against the data-sheet 7.7 TB/s of HBM3e and the 6 452 GB/s this project measured with a bare device copy,
with the card's name and power limit read in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

R, C, MS = 32, 8, 37000
DATASHEET_GBS = 7700.0
MEASURED_GBS = 6452.0


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=int, default=40)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    from softgnss_python_b200 import _native
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import FIELDS, track_quality_batch
    L = _native.lib()
    L.require_device()
    W = args.window
    g = torch.Generator(device="cuda").manual_seed(1)
    out = torch.zeros((R, C, len(FIELDS), MS), dtype=torch.float64, device="cuda")
    a = np.sqrt(2 * 10 ** 4.5 * 1e-3) * 1000.0
    ph = torch.rand((R, C, 1), generator=g, device="cuda", dtype=torch.float64) * 2 * np.pi + \
        torch.arange(MS, device="cuda", dtype=torch.float64) * 1e-3
    for f, trig in (("I_P", torch.cos), ("Q_P", torch.sin)):
        out[:, :, FIELDS.index(f)] = a * trig(ph) + 1000.0 * torch.randn((R, C, MS), generator=g, device="cuda",
                                                                         dtype=torch.float64)
    s = Settings(CNoVSMinterval=W)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(3):
        res = track_quality_batch(out, None, s)
    torch.cuda.synchronize()
    times = []
    for it in range(args.reps):
        flush.fill_(it & 0xff)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = track_quality_batch(out, None, s)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    t = float(np.median(times))
    n_win = MS // W
    nbytes = R * C * n_win * (2 * 8 * W + 17)
    gbs = nbytes / t / 1e9
    cn0 = res["cn0"].cpu().numpy()
    line = dict(kernel="sgx_track_quality", shape=[R, C, len(FIELDS), MS], window_ms=W, windows=R * C * n_win,
                median_s=t, min_s=float(min(times)), max_s=float(max(times)), reps=args.reps, algorithmic_bytes=nbytes,
                gb_per_s=gbs, share_datasheet_7700=gbs / DATASHEET_GBS, share_measured_6452=gbs / MEASURED_GBS,
                median_cn0_dbhz=float(np.nanmedian(cn0)), device=torch.cuda.get_device_name(0),
                power_limit_w=power_limit(), l2_flush_bytes=flush.numel())
    print(json.dumps(line))


if __name__ == "__main__":
    main()
