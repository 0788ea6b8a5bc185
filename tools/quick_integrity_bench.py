"""Time of the integrity stage (sgx_nav_integrity) after the navigation solution (sgx_nav_solve) on a device-resident
tracking result of 32 recordings x 8 channels x 37 000 ms (63 epochs each).

    python tools/quick_integrity_bench.py [--reps 50]

The input is the synthetic chain case of tests/cases.py (seeds 2 and 7 alternating), as one float64 [32, 8, 13, 37 000]
CUDA tensor (985 MB); every fourth recording carries a 300 m range error on one channel from epoch 20, so the exclusion
path (Gauss-Newton on the remaining channels) runs on a quarter of the warps after that epoch.  post_navigate_batch runs
the chain up to the fix once; then two kinds of integrity call are timed with CUDA events, median of --reps after 3
warm-up calls:
  * device:  rawP / active / sol already on the device, device outputs (no host synchronisation inside the call);
  * host:    nav_integrity_batch as the Python layer calls it: host inputs and outputs, synchronous.
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
    from tests.cases import build_chain_case
    L = _native.lib()
    L.require_device()
    s = Settings(numberOfChannels=C, msToProcess=float(MS), useTropCorr=False)
    cases = [build_chain_case(seed=seed, ms=MS)[:2] for seed in (2, 7)]
    dev = torch.empty((R, C, 13, MS), dtype=torch.float64, device="cuda")
    prn = np.zeros((R, C), dtype=np.int64)
    for r in range(R):
        tr = cases[r % 2][0].copy()
        if r % 4 == 3:                                   # 300 m on channel r % 8 from epoch 20
            ch = r % C
            tr[ch, 0, 5200 + 500 * 20 - 250:] += 300.0 * 1000.0 * s.samplesPerCode / s.c
        dev[r] = torch.from_numpy(tr).cuda()
        prn[r] = cases[r % 2][1]
    nav = postnav.post_navigate_batch(dev, prn, s)
    assert (nav["n_epochs"] == 63).all(), nav["n_epochs"]
    rows = np.stack([postnav.eph_rows(nav["eph"][r], np.where(nav["ready"][r] > 0, prn[r], 0)) for r in range(R)])
    E = nav["sol"].shape[1]
    ns, ist = postnav.nav_settings(s), postnav.integ_settings(s)
    raw_d, act_d, sol_d = (torch.from_numpy(nav[k]).cuda() for k in ("rawP", "active", "sol"))
    z = lambda shp: torch.empty(shp, dtype=torch.float64, device="cuda")
    out_d = dict(integ=z((R, E, len(_native.NAV_INTEG_FIELDS))), normResid=z((R, E, C)))

    def device_call():
        L.nav_integrity(raw_d, act_d, sol_d, nav["n_epochs"], rows, nav["tow"], ns, ist, out=out_d)

    def host_call():
        return postnav.nav_integrity_batch(nav, rows, nav["tow"], s)

    t_dev = timed(device_call, args.reps)
    t_host = timed(host_call, args.reps)
    res = host_call()
    assert out_d["integ"].cpu().numpy().tobytes() == res["integ"].tobytes()
    integ = res["integ"]
    status = np.bincount(integ[..., 13].astype(int).ravel(), minlength=len(_native.INTEG_STATUS))
    line = dict(kernel="sgx_nav_integrity", recordings=R, channels=C, ms=MS, epochs=int(nav["n_epochs"].sum()),
                status_counts=dict(zip(_native.INTEG_STATUS, status.tolist())), device_call_median_s=t_dev[0],
                device_call_min_s=t_dev[1], device_call_max_s=t_dev[2], host_call_median_s=t_host[0],
                host_call_min_s=t_host[1], host_call_max_s=t_host[2],
                epochs_per_s_device=float(nav["n_epochs"].sum() / t_dev[0]),
                median_hpl_m=float(np.nanmedian(integ[..., 11])), median_vpl_m=float(np.nanmedian(integ[..., 12])),
                reps=args.reps, device=torch.cuda.get_device_name(0), power_limit_w=power_limit())
    print(json.dumps(line))


if __name__ == "__main__":
    main()
