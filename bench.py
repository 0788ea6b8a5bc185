#!/usr/bin/env python
"""Benchmark of the two hot paths on B200 (one JSON line on stdout, rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Primary line  : tracking channel-ms/s on BASELINE.json config 4 ("batched tracking: 8 channels x 256
                independent recordings (37 s each) sharded across 1/2/4/8 GPUs"): every GPU holds
                256/8 = 32 recordings (45 GB of int8 samples, generated on the device), i.e. weak
                scaling; N = 8 is the whole configuration.  A step = one pass of sgx_track over the
                rank's shard (32 x 8 channels x 37000 code periods), input and output resident in HBM.
`e2e`         : the same shard through the same C-ABI call with HOST (pinned) buffers: the int8
                recordings are copied host->device and the 13 result series device->host inside the
                timed region.
`secondary`   : acquisition search cells/s (config 1 settings, a batch of 11 ms recordings per GPU).
`tertiary`    : preamble search / nav-bit summation on the tracking result (SURVEY.md 8(f) row 3), channels/s.
`quaternary`  : navigation solution (pseudoranges, satellite positions, least-squares fix per measurement epoch;
                SURVEY.md 8(f) row 4) for one recording per tracked recording of the shard, fixes/s.
`roofline`    : tracking kernel, algorithmic bytes (38192 B in + 104 B out per channel-ms,
                SURVEY.md section 8(d)) / CUDA-event duration vs the measured HBM copy bandwidth.
`cpu_baseline`: the numpy oracle (a restatement of the reference's loops, oracle/gnss_oracle.py) timed
                on one host core on a bounded sample.
`--impl reference` times that CPU path on all host cores (one process per channel / PRN group).
`--dump-outputs DIR` writes, after the timed steps, what the last timed step of each GPU leg returned (rank 0's
                shard) as DIR/<name>.npy in float64: a fixed, seeded sample of the tracking output's code periods
                and the acquisition, preamble-search, navigation and config-3 results, each leg within a fixed
                share of 60 MB (a leg whose output is larger keeps its first recordings).  The inputs are generated
                from fixed seeds, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                 # the tree may be read-only; leave no __pycache__ in it
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, "1")

import numpy as np  # noqa: E402

N_CODE = 38192
REC_PER_GPU = 32
CHANNELS = 8
MS = 37000
ACQ_REC_PER_GPU = 32
BYTES_PER_CHANNEL_MS = 38192 + 13 * 8          # SURVEY.md 8(d)
FLOP_PER_CELL = 330.0                          # reference formulation, SURVEY.md 8(d)
TRACK_CPU_MS = 1000                            # bounded CPU sample (code periods per channel)
# --dump-outputs: float64 bytes per leg, fixed in advance so that what one leg dumps never depends on another leg's
# outputs; 60 MB in all, under 64 MB with the npy headers
DUMP_BUDGET = {"track": 40 * 10 ** 6, "acq": 2 * 10 ** 6, "preamble": 8 * 10 ** 6, "nav": 8 * 10 ** 6, "c3": 2 * 10 ** 6}


_RESULT_FD = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def track_sample(out, budget):
    """Tracking output [R, C, 13, ms] at a fixed, seeded set of code periods (every channel, every series) and
    those periods, as many as fit `budget` bytes in float64; all of it when it fits whole."""
    import torch
    r, c, f, ms = out.shape
    n = max(1, min(ms, budget // ((r * c * f + 1) * 8)))
    t = np.sort(np.random.default_rng(0).choice(ms, n, replace=False)) if n < ms else np.arange(ms)
    return out[..., torch.from_numpy(t).to(out.device)].cpu().numpy(), t


def leading_rows(arrays, budget):
    """The arrays of one leg (name -> array, axis 0 = recording or channel), cut to the same first rows so that
    they fit `budget` bytes in float64; whole when they fit."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    per_row = sum(a[:1].size * 8 for a in arrays.values())
    n = max(1, budget // max(1, per_row))
    return {k: a[:n] for k, a in arrays.items()}


def dump_outputs(path, arrays):
    """arrays: name -> numeric array; written as path/<name>.npy in float64."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= sum(DUMP_BUDGET.values()), "output dump of %d bytes exceeds the budget" % total
    os.makedirs(path, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        return len(self.rows)

    def stop(self, lo=0, hi=None):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = self.rows[lo:hi] or self.rows
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------ workloads
def make_specs(first_seed, count, lnav=False):
    """Synthetic 8-satellite recordings.  lnav=True: valid LNAV frames, Kepler geometry and range-consistent delays
    (navsynth.build_scenario) -- the tracking workload, so that the preamble search and the navigation chain that
    follow it in the bench find what postNavigation needs; lnav=False: random Doppler / code phase / data bits (the
    11 ms acquisition batches)."""
    from softgnss_python_b200 import navsynth, synth
    if lnav:
        return [navsynth.build_scenario(seed=first_seed + r)[0] for r in range(count)]
    return [synth.RecordingSpec(synth.default_constellation(first_seed + r, CHANNELS), seed=first_seed + r)
            for r in range(count)]


def channel_truth(specs):
    """Channel table as preRun would hand it to tracking: PRN, carrier (with the fine search's -36 Hz
    bias, SURVEY.md A.1-8) and the code phase the acquisition reports (start + 1, A.1-9)."""
    prn, freq, cph = [], [], []
    for sp in specs:
        for i, s in enumerate(sp.sats):
            prn.append(s.prn)
            freq.append(sp.true_carr_freq(i) - 36.0)
            cph.append(float((s.code_phase + 1) % N_CODE))
    return prn, freq, cph


def run_gpu(args, rank, world):
    import torch
    import torch.distributed as dist
    from softgnss_python_b200 import _native, synth
    from softgnss_python_b200.acquisition import acquire_batch
    from softgnss_python_b200.settings import Settings, to_pod

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = _native.lib()
    L.require_device()
    L.check(L.dll.sgx_set_device(local))
    stream = torch.cuda.current_stream().cuda_stream
    chips, lut = _native.ca_chips_int8(), synth.cos_lut()

    recs, ms = args.recordings, args.ms
    settings = Settings(msToProcess=float(ms))
    pod = to_pod(settings)
    specs = make_specs(2000 + rank * recs, recs, lnav=True)
    n = (ms + 2) * N_CODE
    stride = (n + 15) // 16 * 16
    dev = torch.empty((recs, stride), dtype=torch.int8, device="cuda")
    sp, bits = _native.make_synth_specs(specs)
    for r0 in range(0, recs, 8):                       # generate on the device, 8 recordings per launch
        r1 = min(recs, r0 + 8)
        sub = (_native.SgxSynthSpec * (r1 - r0))(*[sp[i] for i in range(r0, r1)])
        L.synth(dev[r0:r1], stride, n, 0, sub, np.ascontiguousarray(bits[r0:r1]), lut, chips, stream)
    chans = _native.make_channels(*channel_truth(specs))
    out = torch.empty((recs, CHANNELS, 13, ms), dtype=torch.float64, device="cuda")
    rec_len = [n] * recs
    units = recs * CHANNELS * ms

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev():
        rc, done = L.track(dev, stride, rec_len, chans, pod, chips, out, stream)
        L.check(rc)
        return done

    # ---- device-resident timing (value, roofline) -------------------------------------------------
    clocks = ClockSampler(local) if rank == 0 else None     # started early: nvidia-smi needs ~1 s to spin up
    for _ in range(args.warmup):
        step_dev()
    barrier()
    l0 = L.launches()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    c0 = clocks.mark() if clocks else 0
    ev[0].record()
    for k in range(args.steps):
        done = step_dev()
        ev[k + 1].record()
    barrier()
    c1 = clocks.mark() if clocks else 0
    launches = L.launches() - l0
    total_ms = ev[0].elapsed_time(ev[-1])
    assert int(done.min()) == ms
    t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = world * units / (ms_per_step / 1e3)
    kernel_ms = float(np.mean([ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]))
    lock = out[:, :, 3, 500:].abs().mean().item() / max(out[:, :, 7, 500:].abs().mean().item(), 1e-9) if ms > 600 else None
    dump = {} if args.dump_outputs and rank == 0 else None     # name -> what the last timed step of a leg returned

    # ---- end to end through the C ABI with host buffers --------------------------------------------
    e2e = None
    if not args.no_e2e:
        try:
            # host buffers: keep the pinned allocation within half of the free host RAM shared by the ranks
            import psutil
            per_rec = stride + CHANNELS * 13 * ms * 8
            budget = 0.5 * psutil.virtual_memory().available / max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
            erecs = int(max(1, min(recs, budget // per_rec)))
            host = torch.empty((erecs, stride), dtype=torch.int8, pin_memory=True)
            host.copy_(dev[:erecs])
            hout = torch.empty((erecs, CHANNELS, 13, ms), dtype=torch.float64, pin_memory=True)
            del dev
            torch.cuda.empty_cache()
            hin, hres = host.numpy(), hout.numpy()
            # ceiling of this box: every rank copies pinned host memory to its GPU at the same time (bare copies)
            probe = torch.empty(min(1 << 30, host.numel()), dtype=torch.int8, device="cuda")
            barrier()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(3):
                probe.copy_(host.view(-1)[:probe.numel()], non_blocking=True)
            h1.record()
            barrier()
            th = torch.tensor([h0.elapsed_time(h1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(th, op=dist.ReduceOp.MAX)
            h2d_gbs = 3 * probe.numel() / (float(th.item()) / 1e3) / 1e9      # per GPU, slowest rank
            del probe
            echans = _native.make_channels(*channel_truth(specs[:erecs]))
            eunits = erecs * CHANNELS * ms

            def step_host():
                rc, d = L.track(hin, stride, rec_len[:erecs], echans, pod, chips, hres, stream)
                L.check(rc)

            for _ in range(max(1, min(args.warmup, 2))):
                step_host()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ksteps = args.steps
            e0.record()
            for _ in range(ksteps):
                step_host()
            e1.record()
            barrier()
            tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_ms = float(tt.item()) / ksteps
            e2e = {"value": world * eunits / (e2e_ms / 1e3), "unit": "channel-ms/s",
                   "h2d_bytes_per_step": int(erecs * n), "d2h_bytes_per_step": int(hres.nbytes),
                   "ms_per_step": e2e_ms, "steps": ksteps, "recordings_per_gpu": erecs,
                   "h2d_ceiling_gbs_per_gpu": h2d_gbs, "h2d_ceiling_gbs_all_gpus": h2d_gbs * world,
                   "h2d_achieved_gbs_per_gpu": erecs * n / (e2e_ms / 1e3) / 1e9,
                   "frac_of_h2d_ceiling": (erecs * n / (e2e_ms / 1e3) / 1e9) / h2d_gbs,
                   "h2d_note": "ceiling = concurrent bare cudaMemcpyAsync of 1 GiB pinned buffers on all ranks (slowest "
                               "rank); the e2e step cannot be faster than its input bytes / this rate",
                   "path": "sgx_track with host pointers: chunked H2D on a copy stream overlapped with the kernel, "
                           "results D2H at the end"}
            del host, hout
        except Exception as exc:  # pinned allocation can fail on a small host
            e2e = {"value": None, "unit": "channel-ms/s", "error": str(exc)[:200]}

    # ---- secondary: acquisition ----------------------------------------------------------------------
    acq = None
    if not args.no_acq:
        areq = args.acq_recordings
        aspecs = make_specs(1000 + rank * areq, areq)
        an = 11 * N_CODE
        adev = torch.empty((areq, an), dtype=torch.int8, device="cuda")
        asp, abits = _native.make_synth_specs(aspecs)
        L.synth(adev, an, an, 0, asp, abits, lut, chips, stream)
        aset = Settings()
        cells = areq * 32 * 29 * N_CODE
        for _ in range(args.warmup):
            res = acquire_batch(adev, aset, stream=stream)
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        al0 = L.launches()
        a0.record()
        for _ in range(args.steps):
            res = acquire_batch(adev, aset, stream=stream)
        a1.record()
        barrier()
        alaunch = L.launches() - al0
        ta = torch.tensor([a0.elapsed_time(a1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ta, op=dist.ReduceOp.MAX)
        a_ms = float(ta.item()) / args.steps
        if dump is not None:
            dump.update(leading_rows({"acq_" + k: v for k, v in res.items()}, DUMP_BUDGET["acq"]))
        ahost = torch.empty((areq, an), dtype=torch.int8, pin_memory=True)
        ahost.copy_(adev)
        ah = ahost.numpy()
        acquire_batch(ah, aset, stream=stream)
        barrier()
        a0.record()
        for _ in range(args.steps):
            acquire_batch(ah, aset, stream=stream)
        a1.record()
        barrier()
        tb = torch.tensor([a0.elapsed_time(a1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        ae_ms = float(tb.item()) / args.steps
        truth = sum(len(s.sats) for s in aspecs)
        # config 1 itself: ONE 11 ms recording (latency of acquisition(longSignal, settings) with the signal in HBM)
        for _ in range(2):
            acquire_batch(adev[:1], aset, stream=stream)
        barrier()
        a0.record()
        for _ in range(args.steps):
            acquire_batch(adev[:1], aset, stream=stream)
        a1.record()
        barrier()
        a1_ms = a0.elapsed_time(a1) / args.steps
        fp32_peak = L.fp32_peak(stream)                       # FFMA burn on this GPU, TFLOP/s (SURVEY.md 8(d))
        acq_tflops = cells * FLOP_PER_CELL / (a_ms / 1e3) / 1e12
        acq_traffic = None      # DRAM bytes of the search kernel per launch, from the committed ncu capture of this workload
        try:
            with open(os.path.join(ROOT, "profiles", "acq_traffic_r2.json")) as f:
                acq_traffic = json.load(f).get("dram_bytes_per_launch") if areq == 32 else None
        except (OSError, ValueError):
            pass
        acq = {"metric": "acq search cells/s", "value": world * cells / (a_ms / 1e3), "unit": "cells/s",
               "ms_per_step": a_ms, "gpu_launches": int(alaunch),
               "config": {"workload": "config 1 settings (32 PRN x 29 bins x 38192 code phases + fine search), "
                                      "%d x 11 ms recordings per GPU, 8 satellites each at 45 dB-Hz" % areq,
                          "detected": int((res["carrFreq"] > 0).sum()), "present": truth},
               "e2e": {"value": world * cells / (ae_ms / 1e3), "unit": "cells/s",
                       "h2d_bytes_per_step": int(areq * an), "d2h_bytes_per_step": int(areq * 32 * 3 * 8)},
               "single_recording": {"ms": a1_ms, "cells_per_s": 32 * 29 * N_CODE / (a1_ms / 1e3),
                                    "note": "config 1 as written: one 11 ms recording, 32 PRN x 29 bins + fine search"},
               "roofline": {"bound": "fp32 (CUDA-core FFT; not HBM: 0.3 B/cell)",
                            "achieved": acq_tflops, "peak": fp32_peak, "unit": "TFLOP/s",
                            "frac": acq_tflops / fp32_peak, "frac_of_nominal_74.5": acq_tflops / 74.5,
                            "traffic": acq_traffic, "kernel": "sgx::pfa::pfa_search_kernel (68 % of the call)",
                            "note": "reference-formulation FLOPs (330/cell, SURVEY.md 8(d)); peak = FP32 FMA burn "
                                    "measured on this GPU in this run (sgx_fp32_peak; nominal 74.5)"}}
        if rank == 0 and not args.no_cpu:
            from oracle import gnss_oracle as orc
            one = adev[0].cpu().numpy()
            t0 = time.perf_counter()
            oref = orc.acquire(one, aset)
            dt = time.perf_counter() - t0
            acq["cpu_baseline"] = {"value": 32 * 29 * N_CODE / dt, "unit": "cells/s", "cores": 1, "kind": "port",
                                   "sample": "one of the %d recordings in full (32 PRN x 29 bins + fine search), "
                                             "oracle/gnss_oracle.py acquire (numpy restatement of acquisition.py:49-204 with "
                                             "the carrier wipe-off hoisted out of the PRN loop), %.1f s" % (areq, dt)}
            assert np.array_equal(oref["carrFreq"] > 0, res["carrFreq"][0] > 0), "acquisition differs from the oracle"
            assert np.array_equal(oref["codePhase"], res["codePhase"][0])

    # ---- tertiary: preamble search / bit summation on the device-resident tracking result (8(f) row 3) ----
    bsync = None
    if not args.no_acq and ms >= 160:
        from softgnss_python_b200 import postnav
        ipv = out.view(recs * CHANNELS, 13 * ms)[:, 3 * ms:4 * ms]      # I_P rows, row stride 13 * ms
        for _ in range(args.warmup):
            postnav.find_preambles_batch(ipv, stream=stream)
        barrier()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        bl0 = L.launches()
        b0.record()
        for _ in range(args.steps):
            first, nbits, nvalid = postnav.find_preambles_batch(ipv, stream=stream)
        b1.record()
        barrier()
        tb = torch.tensor([b0.elapsed_time(b1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tb, op=dist.ReduceOp.MAX)
        b_ms = float(tb.item()) / args.steps
        if dump is not None:
            dump.update(leading_rows(dict(preamble_first=first, preamble_bits=nbits, preamble_valid=nvalid),
                                     DUMP_BUDGET["preamble"]))
        nch = recs * CHANNELS
        bsync = {"metric": "preamble search channels/s", "value": world * nch / (b_ms / 1e3), "unit": "channels/s",
                 "ms_per_step": b_ms, "gpu_launches": int(L.launches() - bl0),
                 "config": {"workload": "sign bits + 160-tap preamble correlation at %d lags + parity verification + "
                                        "1501 nav bits for %d channels per GPU (I_P of the tracking step above, "
                                        "device resident; results copied to the host inside the timed region)" % (ms, nch),
                            "channels_with_preamble": int((first > 0).sum())},
                 "roofline": {"bound": "hbm", "achieved": nch * ms * 8 / (b_ms / 1e3) / 1e9, "peak": peaks()[0],
                              "unit": "GB/s", "frac": nch * ms * 8 / (b_ms / 1e3) / 1e9 / peaks()[0],
                              "note": "algorithmic bytes = 8 B per ms per channel (I_P read once)"}}
        if rank == 0 and not args.no_cpu:
            from oracle import gnss_oracle as orc
            hip = [x.copy() for x in ipv[:CHANNELS].cpu().numpy()]
            t0 = time.perf_counter()
            of, _ = orc.find_preambles(hip)
            for c in range(CHANNELS):
                if of[c] and of[c] + 30000 <= ms:
                    orc.nav_bits(hip[c], int(of[c]))
            dt = time.perf_counter() - t0
            bsync["cpu_baseline"] = {"value": CHANNELS / dt, "unit": "channels/s", "cores": 1, "kind": "port",
                                     "sample": "%d channels x %d ms, oracle/gnss_oracle.py find_preambles (160-tap sliding "
                                               "window; the reference's own M x M np.correlate takes ~0.24 s per channel)"
                                               % (CHANNELS, ms)}
            assert np.array_equal(of, first[:CHANNELS]), "bit sync differs from the oracle"

    # ---- quaternary: preamble search -> ephemeris decoding -> measurement loop on the tracking result (8(f) rows 3-4) ----
    navb = None
    if not args.no_acq and ms >= 36000:
        from softgnss_python_b200 import postnav
        nset = Settings(msToProcess=float(ms))
        nset.useTropCorr = False                       # the synthetic geometry has no troposphere
        prn_arr = np.array(channel_truth(specs)[0], dtype=np.int64).reshape(recs, CHANNELS)
        for _ in range(args.warmup):
            postnav.post_navigate_batch(out, prn_arr, nset, stream=stream)
        barrier()
        q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ql0 = L.launches()
        q0.record()
        for _ in range(args.steps):
            nout = postnav.post_navigate_batch(out, prn_arr, nset, stream=stream)
        q1.record()
        barrier()
        tq = torch.tensor([q0.elapsed_time(q1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tq, op=dist.ReduceOp.MAX)
        q_ms = float(tq.item()) / args.steps
        if dump is not None:
            dump.update(leading_rows({"nav_" + k: v for k, v in nout.items() if isinstance(v, np.ndarray)},
                                     DUMP_BUDGET["nav"]))
        n_fix = int(nout["n_epochs"].sum())
        from softgnss_python_b200 import navsynth
        rx = navsynth.build_scenario(seed=2000 + rank * recs)[1]["rx"]
        sol0 = nout["sol"][0, :int(nout["n_epochs"][0])]
        err0 = np.sqrt(((sol0[:, :3] - rx) ** 2).sum(1))
        navb = {"metric": "navigation epochs/s", "value": world * n_fix / (q_ms / 1e3), "unit": "epochs/s",
                "ms_per_step": q_ms, "gpu_launches": int(L.launches() - ql0),
                "config": {"workload": "postNavigate chain on the tracking result of the step above (device resident, %d "
                                       "recordings x %d channels per GPU): preamble search + 1501 nav bits per channel "
                                       "(device), ephemeris decoding (host bit slicing), pseudoranges / satpos / 7-iteration "
                                       "least-squares fix / DOP / cart2geo for %d measurement epochs per recording (device); "
                                       "solutions copied to the host inside the timed region"
                                       % (recs, CHANNELS, int(nout["n_epochs"][0])),
                           "epochs_with_fix": int(np.isfinite(nout["sol"][:, :, 0]).sum()),
                           "recordings_with_solution": int((nout["n_epochs"] > 0).sum()),
                           "median_3d_error_to_true_antenna_m": float(np.median(err0))},
                "roofline": {"bound": "latency (one warp per recording, epochs sequential through the elevation mask; "
                                      "float64 dependency chain)", "frac": None}}
        if rank == 0 and not args.no_cpu:
            from oracle import gnss_oracle as orc
            trk0 = out[0].cpu().numpy()
            t0 = time.perf_counter()
            of, oa = orc.find_preambles([trk0[c, 3] for c in range(CHANNELS)])
            eph, tow, ready = [None] * 32, None, []
            for c in oa:
                if of[c] + 30000 > ms:
                    continue
                b = orc.nav_bits(trk0[c, 3], int(of[c]))
                e, tow = orc.ephemeris(b[1:], b[0])
                eph[int(prn_arr[0, c]) - 1] = e
                if e["IODC"] is not None and e["IODE_sf2"] is not None and e["IODE_sf3"] is not None:
                    ready.append(c)
            o = orc.nav_solve([trk0[c, 0] for c in range(CHANNELS)], prn_arr[0], of, ready, eph, tow, float(ms), N_CODE,
                              elevation_mask=nset.elevationMask, use_trop_corr=nset.useTropCorr)
            dt = time.perf_counter() - t0
            navb["cpu_baseline"] = {"value": o["n_epochs"] / dt, "unit": "epochs/s", "cores": 1, "kind": "port",
                                    "sample": "the same chain for recording 0 (8 channels x %d ms, %d epochs) with "
                                              "oracle/gnss_oracle.py: find_preambles, nav_bits, ephemeris, nav_solve"
                                              % (ms, o["n_epochs"])}
            assert o["n_epochs"] == int(nout["n_epochs"][0])
            assert np.abs(sol0[:, 0] - o["X"]).max() <= 1e-5 and np.abs(sol0[:, 2] - o["Z"]).max() <= 1e-5, "nav chain differs"

    # ---- config 3 (weak-signal acquisition, 141 bins): 10 ms coherent and 10 x 1 ms blocks, split by PRN over the ranks ----
    c3 = None
    if not args.no_acq and args.c3_recordings > 0:
        from softgnss_python_b200 import dist as sd
        c3 = {}
        c3n = args.c3_recordings
        c3specs = make_specs(1000, c3n)                      # every rank holds the same recordings: the split is by PRN
        c3dev = torch.empty((c3n, 11 * N_CODE), dtype=torch.int8, device="cuda")
        c3sp, c3bits = _native.make_synth_specs(c3specs)
        L.synth(c3dev, 11 * N_CODE, 11 * N_CODE, 0, c3sp, c3bits, lut, chips, stream)
        for name, ext in (("coherent_10ms", dict(acqCoherentMs=10, acqNonCoherentBlocks=1, acqDopplerStep=100.0)),
                          ("blocks_10x1ms", dict(acqCoherentMs=1, acqNonCoherentBlocks=10, acqDopplerStep=100.0))):
            cs = Settings(**ext)
            sd.acquire_sharded(c3dev, cs, stream=stream)
            barrier()
            z0, z1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            z0.record()
            for _ in range(args.steps):
                r3 = sd.acquire_sharded(c3dev, cs, stream=stream)
            z1.record()
            barrier()
            tz = torch.tensor([z0.elapsed_time(z1) / args.steps], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(tz, op=dist.ReduceOp.MAX)
            if dump is not None:
                dump.update(leading_rows({"c3_%s_%s" % (name, k): v for k, v in r3.items()}, DUMP_BUDGET["c3"] // 2))
            cells3 = c3n * 32 * 141 * N_CODE
            c3[name] = {"value": cells3 / (float(tz.item()) / 1e3), "unit": "cells/s", "ms_per_step": float(tz.item()),
                        "recordings": c3n, "bins": 141, "prn_per_rank": 32 // world,
                        "detected": int((r3["carrFreq"] > 0).sum())}
        c3["note"] = ("BASELINE config 3 settings on %d recordings at 45 dB-Hz, 32 PRNs split by PRN over the ranks "
                      "(dist.acquire_sharded, results gathered over NCCL); parity at 30-43 dB-Hz: tests/test_gpu_config3.py" % c3n)
        del c3dev

    # ---- collectives (world > 1): PRN-split acquisition of one batch and the result gathers, timed separately ----------
    coll = None
    if world > 1 and not args.no_acq:
        from softgnss_python_b200 import dist as sd
        coll = {}
        sd.acquire_sharded(adev, aset, stream=stream)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            rs = sd.acquire_sharded(adev, aset, stream=stream)
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1) / args.steps], dtype=torch.float64, device="cuda")
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        coll["acquire_sharded_by_prn"] = {"ms": float(tg.item()), "cells_per_s": areq * 32 * 29 * N_CODE / (float(tg.item()) / 1e3),
                                           "note": "the SAME %d recordings on every rank, 32/%d PRNs each, gather included"
                                                   % (areq, world)}
        packed = torch.zeros((3, areq, 32 // world), dtype=torch.float64, device="cuda")
        sd.gather_results(packed, 32 // world * world, axis=2)
        barrier()
        g0.record()
        for _ in range(args.steps):
            sd.gather_results(packed, 32 // world * world, axis=2)
        g1.record()
        barrier()
        coll["acq_results_gather"] = {"ms": g0.elapsed_time(g1) / args.steps, "bytes_per_rank": int(packed.numel() * 8),
                                      "note": "latency only (SURVEY.md 8(e))"}
        sd.gather_results(out[:1], world, axis=0)
        barrier()
        g0.record()
        for _ in range(args.steps):
            full = None                                              # at most one gathered copy alive
            full = sd.gather_results(out, world * recs, axis=0)      # trackResults of all ranks, GPU to GPU
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1) / args.steps], dtype=torch.float64, device="cuda")
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        nbytes = int(out.numel() * 8)
        coll["track_results_gather"] = {"ms": float(tg.item()), "bytes_per_rank": nbytes, "total_bytes": nbytes * world,
                                         "bus_gbs_per_gpu": nbytes * (world - 1) / (float(tg.item()) / 1e3) / 1e9,
                                         "note": "all_gather_into_tensor of the device-resident [R][C][13][ms] float64 results "
                                                 "(NCCL over NVLink); bus bandwidth = bytes received per GPU / time"}
        assert torch.equal(full[rank * recs:(rank + 1) * recs], out)
        del full

    ck = clocks.stop(c0, c1) if clocks else None
    if world > 1:
        counts = [None] * world
        dist.all_gather_object(counts, int(done.sum()))
        dist.destroy_process_group()
    if rank != 0:
        return
    if dump is not None:
        # `out` still holds the last timed tracking step: the later legs only read it
        dump["track_ms_done"] = done
        dump["track_out_sample"], dump["track_out_sample_ms"] = track_sample(out, DUMP_BUDGET["track"] - done.size * 8)
        dump_outputs(args.dump_outputs, dump)
    peak, how = peaks()
    achieved = units * BYTES_PER_CHANNEL_MS / (kernel_ms / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "track_traffic.json")
    if os.path.exists(tp):
        tj = json.load(open(tp))
        if tj.get("recordings") == recs and tj.get("ms") == ms:
            traffic = tj.get("dram_bytes_per_launch")
    line = {
        "metric": "tracking channel-ms/s", "value": value, "unit": "channel-ms/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int8 x Q38 fixed-point correlators (exact int32 dot products), f64 rotors / accumulation / loop filters", "data": "synthetic",
        "realtime_factor": value / 1000.0,
        "config": {"workload": "BASELINE config 4 shard: %d recordings x %d channels x %d ms per GPU "
                               "(int8 IF, fs 38.192 MHz, generated on device); x%d GPUs" % (recs, CHANNELS, ms, world),
                   "recordings_per_gpu": recs, "channels": CHANNELS, "ms": ms,
                   "l2": "inputs (%.1f GB per GPU) far exceed L2; no flush needed" % (recs * n / 1e9),
                   "lock_check_mean_absIP_over_absQP": lock},
        "gpu_launches": int(launches),
        "e2e": e2e,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "sgx::track_kernel", "kernel_ms": kernel_ms,
                     "algorithmic_bytes_per_channel_ms": BYTES_PER_CHANNEL_MS, "peak_source": how},
        "clocks": ck,
        "secondary": acq,
        "tertiary": bsync,
        "quaternary": navb,
        "config3": c3,
        "collectives": coll,
        # the acquisition half of BASELINE.json's metric, lifted so that per-N records keep it
        "acq_value": acq["value"] if acq else None,
        "acq_unit": "cells/s",
        "acq_ms_per_step": acq["ms_per_step"] if acq else None,
        "acq_roofline_frac": acq["roofline"]["frac"] if acq else None,
        "acq_e2e_value": acq["e2e"]["value"] if acq else None,
    }
    if not args.no_cpu:
        line["cpu_baseline"] = cpu_track_baseline(TRACK_CPU_MS, 1)
    emit(line)


# ------------------------------------------------------------------------------------------ CPU arms
_CPU = {}


def _cpu_prepare(ms):
    """One config-4 recording (seed 2000) long enough for `ms` code periods; shared with forked workers."""
    if _CPU.get("ms") == ms:
        return
    from softgnss_python_b200 import synth
    from softgnss_python_b200.settings import Settings
    spec = make_specs(2000, 1, lnav=True)[0]
    _CPU.update(ms=ms, data=synth.generate_cpu(spec, (ms + 2) * N_CODE), truth=channel_truth([spec]),
                settings=Settings(msToProcess=float(ms)))


def _cpu_track_one(ch):
    from oracle import gnss_oracle as orc
    prn, freq, cph = _CPU["truth"]
    t = time.perf_counter()
    _, done = orc.track_channel(_CPU["data"], prn[ch], freq[ch], cph[ch], _CPU["settings"], _CPU["ms"])
    assert done == _CPU["ms"]
    return time.perf_counter() - t


def cpu_track_baseline(ms, procs):
    """Oracle tracking (numpy restatement of tracking.py:132-275).  procs == 1: the 8 channels of one
    recording one after the other on one core (as the reference does); procs > 1: one channel per process."""
    import multiprocessing as mp
    _cpu_prepare(ms)
    if procs == 1:
        dt = sum(_cpu_track_one(c) for c in range(CHANNELS))
        n_ch = CHANNELS
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            pool.map(_cpu_track_one, [0] * procs)      # start the workers before timing
            t = time.perf_counter()
            pool.map(_cpu_track_one, [c % CHANNELS for c in range(procs)], chunksize=1)
            dt = time.perf_counter() - t
        n_ch = procs
    return {"value": n_ch * ms / dt, "unit": "channel-ms/s", "cores": procs, "kind": "port",
            "sample": "%d channel(s) x %d ms of config-4 recording seed 2000, oracle/gnss_oracle.py "
                      "(numpy restatement of the reference loop; numpy %s)" % (n_ch, ms, np.__version__)}


def _cpu_acq_one(seed):
    from oracle import gnss_oracle as orc
    from softgnss_python_b200 import synth
    from softgnss_python_b200.settings import Settings
    spec = make_specs(seed, 1)[0]
    data = synth.generate_cpu(spec, 11 * N_CODE)
    t = time.perf_counter()
    r = orc.acquire(data, Settings())
    return time.perf_counter() - t, int((r["carrFreq"] > 0).sum())


def cpu_acq_baseline(procs):
    """Oracle acquisition (numpy restatement of acquisition.py:49-204), one full config-1 recording per process."""
    import multiprocessing as mp
    with mp.get_context("fork").Pool(procs) as pool:
        t = time.perf_counter()
        res = pool.map(_cpu_acq_one, [1000 + i for i in range(procs)], chunksize=1)
        dt = time.perf_counter() - t
    return {"value": procs * 32 * 29 * N_CODE / dt, "unit": "cells/s", "cores": procs, "kind": "port",
            "ms_per_step": dt * 1e3, "detected": int(sum(x[1] for x in res)),
            "sample": "%d config-1 recordings (11 ms, 32 PRN x 29 bins + fine search), one per process, "
                      "oracle/gnss_oracle.py acquire; recording generation excluded from the per-process time but the "
                      "wall clock of the pool is what is reported" % procs}


def run_reference(args, rank):
    """--impl reference: the reference's CPU algorithm (oracle port) on all host cores."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(cores, 64))
    vals = []
    for k in range(args.warmup + args.steps):
        r = cpu_track_baseline(args.ref_ms, procs)
        if k >= args.warmup:
            vals.append(r)
    v = float(np.mean([x["value"] for x in vals]))
    base = vals[-1]
    base["value"] = v
    line = {"impl": "reference", "metric": "tracking channel-ms/s", "value": v, "unit": "channel-ms/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": procs * args.ref_ms / v * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "BASELINE config 4 shard: %d recordings x %d channels x %d ms per GPU; CPU arm "
                                   "runs a bounded sample of it" % (REC_PER_GPU, CHANNELS, MS)},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": "channel-ms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if not args.no_acq:
        a = cpu_acq_baseline(procs)
        line["secondary"] = {"metric": "acq search cells/s", "value": a["value"], "unit": "cells/s",
                             "ms_per_step": a["ms_per_step"], "cpu_baseline": a,
                             "config": {"workload": "config 1 settings, one 11 ms recording per host core"}}
        line["acq_value"] = a["value"]
        line["acq_unit"] = "cells/s"
        line["acq_ms_per_step"] = a["ms_per_step"]
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--recordings", type=int, default=REC_PER_GPU, help="recordings per GPU")
    ap.add_argument("--ms", type=int, default=MS)
    ap.add_argument("--acq-recordings", type=int, default=ACQ_REC_PER_GPU)
    ap.add_argument("--c3-recordings", type=int, default=2, help="recordings of the config-3 leg (0 = skip)")
    ap.add_argument("--ref-ms", type=int, default=400, help="code periods per channel per CPU step")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-acq", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of every GPU leg to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    # stdout carries exactly one JSON line: everything else that libraries write to fd 1 (NCCL prints its
    # version banner there) goes to stderr
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    run_gpu(args, rank, world)


if __name__ == "__main__":
    main()
