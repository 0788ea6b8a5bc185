"""Time of the velocity stage (sgx_nav_velocity) chained after the navigation solution (sgx_nav_solve) on a
device-resident tracking result of 32 recordings x 8 channels x 37 000 ms (63 epochs each).

    python tools/quick_velocity_bench.py [--reps 50]

The input is the synthetic chain case of tests/cases.py (seeds 2 and 7 alternating: LNAV streams in I_P, the geometry
in absoluteSample) with carrFreq = IF + the scenario's Doppler + hash noise, as one float64 [32, 8, 13, 37 000] CUDA
tensor (985 MB).  post_navigate_batch runs the chain up to the fix once; then two kinds of velocity call are timed
with CUDA events, median of --reps after 3 warm-up calls:
  * device:  active / sol already on the device, device outputs (what a caller that keeps the chain on the GPU pays;
             the call still copies the small per-recording inputs and has no host synchronisation inside);
  * host:    nav_velocity_batch as the Python layer calls it: host active / sol / outputs, synchronous.
The card's name and power limit are read in the same run.  Prints one JSON line.
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


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out.splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        return None


def timed(fn, reps):
    import torch
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    return float(np.median(times)), float(min(times)), float(max(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    import torch
    from softgnss_python_b200 import _native, postnav
    from softgnss_python_b200.settings import Settings
    from tests.cases import _hash_noise, build_chain_case
    L = _native.lib()
    L.require_device()
    s = Settings(numberOfChannels=C, msToProcess=float(MS))
    cases = []
    for seed in (2, 7):
        tr, prn, truth = build_chain_case(seed=seed, ms=MS)
        for c in range(C):
            tr[c, 2] = s.IF + truth["doppler"][c] + 0.01 * _hash_noise(seed * 1000 + c, MS)
        cases.append((tr, prn))
    dev = torch.empty((R, C, 13, MS), dtype=torch.float64, device="cuda")
    prn = np.zeros((R, C), dtype=np.int64)
    for r in range(R):
        dev[r] = torch.from_numpy(cases[r % 2][0]).cuda()
        prn[r] = cases[r % 2][1]
    nav = postnav.post_navigate_batch(dev, prn, s)
    assert (nav["n_epochs"] == 63).all(), nav["n_epochs"]
    rows = np.stack([postnav.eph_rows(nav["eph"][r], np.where(nav["ready"][r] > 0, prn[r], 0)) for r in range(R)])
    E = nav["sol"].shape[1]
    vs = postnav.vel_settings(s)
    act_d, sol_d = torch.from_numpy(nav["active"]).cuda(), torch.from_numpy(nav["sol"]).cuda()
    z = lambda shp: torch.empty(shp, dtype=torch.float64, device="cuda")
    out_d = dict(vel=z((R, E, 8)), doppler=z((R, E, C)), rrResid=z((R, E, C)))
    carr = dev.data_ptr() + 8 * 2 * MS

    def device_call():
        L.nav_velocity(carr, 13 * MS, R, C, MS, None, nav["subFrameStart"], rows, nav["tow"],
                       nav["n_epochs"], act_d, sol_d, vs, out=out_d)

    def host_call():
        return postnav.nav_velocity_batch(dev, nav, nav["subFrameStart"], rows, nav["tow"], s)

    t_dev = timed(device_call, args.reps)
    t_host = timed(host_call, args.reps)
    res = host_call()
    assert np.array_equal(out_d["vel"].cpu().numpy(), res["vel"], equal_nan=True)
    vel = res["vel"]
    line = dict(kernel="sgx_nav_velocity", recordings=R, channels=C, ms=MS, epochs=int(nav["n_epochs"].sum()),
                doppler_avg_ms=vs.doppler_avg_ms, device_call_median_s=t_dev[0], device_call_min_s=t_dev[1],
                device_call_max_s=t_dev[2], host_call_median_s=t_host[0], host_call_min_s=t_host[1],
                host_call_max_s=t_host[2], epochs_per_s_device=float(nav["n_epochs"].sum() / t_dev[0]),
                median_speed_ms=float(np.nanmedian(np.sqrt((vel[..., :3] ** 2).sum(-1)))), reps=args.reps,
                device=torch.cuda.get_device_name(0), power_limit_w=power_limit())
    print(json.dumps(line))


if __name__ == "__main__":
    main()
