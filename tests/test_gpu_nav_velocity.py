"""Receiver velocity and clock drift from the PLL's Doppler (sgx_nav_velocity, csrc/sgx_nav.cu) against the float64
oracle (tests/velocity_oracle.py), against the geometry the inputs were made from, and end to end on the config-2
recording.

The parity tests run on two backends, as in test_gpu_track_quality.py:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).
The inputs are the synthetic chain cases of tests/cases.py (LNAV streams in I_P, the geometry in absoluteSample) with a
carrFreq series written into field 2: IF plus the Doppler of a receiver that moves at V_TRUTH with a clock drift of
DRIFT_TRUTH, plus hash noise.  The fix and its channel lists come from sgx_nav_solve on the same backend.
"""
import ctypes
import os

import numpy as np
import pytest

from tests import velocity_oracle as vor
from tests.cases import NAV_MS, _hash_noise, build_chain_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
SGX_OK, SGX_ERR_ARG, SGX_ERR_NODEV = 0, -2, -4
IF = 9548000.0
C_LIGHT = 299792458.0
F_L1 = 1575.42e6
V_TRUTH = np.array([12.0, -7.0, 3.0])
DRIFT_TRUTH = 150.0                       # m/s (c times the receiver clock drift)
SEEDS = ((2, ()), (5, (1, 4, 6, 7, 2)), (7, (3,)))      # seed 5 keeps three satellites: no fix at all
ELEV_MASK = 25.0                          # drops the satellites between the scenario's 15 degrees and 25 degrees
NOISE_HZ = 0.01                           # Hz per unit of hash noise (sigma 209 units: ~2 Hz rms per code period)


def _vs(n=100, period=500.0, c=C_LIGHT, f_l1=F_L1, if_hz=IF):
    from softgnss_python_b200 import _native
    return _native.SgxVelSettings(IF=if_hz, c=c, f_L1=f_l1, nav_sol_period=period, doppler_avg_ms=n, reserved=0)


def _settings(mask=ELEV_MASK):
    from softgnss_python_b200.settings import Settings
    return Settings(numberOfChannels=8, msToProcess=float(NAV_MS), elevationMask=mask)


# ---------------------------------------------------------------------------------------------- inputs
def truth_range_rate(e, t, rx, v, h=0.01):
    """Range rate at transmit time t of a receiver passing through rx with velocity v: central difference of
    navsynth.geometric_range over +-h."""
    from softgnss_python_b200 import navsynth
    rp, _ = navsynth.geometric_range(e, t + h, rx + v * h)
    rm, _ = navsynth.geometric_range(e, t - h, rx - v * h)
    return (rp - rm) / (2 * h)


def _carr_freq(track, truth, seed, noise=True, grid_ms=250):
    """carrFreq series [C, ms] of the chain case: channel c's subframe at tow arrives at ms k0 (cases.build_chain_case),
    so ms k carries transmit time tow + (k - k0) / 1000.  The range rate is evaluated every grid_ms and interpolated
    linearly (its curvature over 250 ms is far below a micrometre per second)."""
    n_ch, _, ms = track.shape
    k = np.arange(ms, dtype=np.float64)
    out = np.empty((n_ch, ms))
    grid = np.arange(-grid_ms, ms + 2 * grid_ms, grid_ms, dtype=np.float64)
    for c in range(n_ch):
        k0 = 5200 + (3 * c) % 7
        rr = np.array([truth_range_rate(truth["eph"][c], truth["tow"] + (g - k0) / 1000.0, truth["rx"], V_TRUTH)
                       for g in grid])
        d = -(np.interp(k, grid, rr) + DRIFT_TRUTH) * F_L1 / C_LIGHT
        out[c] = IF + d + (NOISE_HZ * _hash_noise(seed * 1000 + c, ms) if noise else 0.0)
    return out


def _chain_inputs(seed, drop, noise=True):
    """(track [C, 13, ms] with carrFreq in field 2, prn, truth, sub_frame_start, ready, eph rows, tow, n_epochs) with
    the preamble search and ephemeris decoding of the oracle (the same bits and values as the device chain)."""
    from oracle import gnss_oracle as orc
    from softgnss_python_b200 import postnav
    track, prn, truth = build_chain_case(seed=seed, drop=drop)
    track[:, 2] = _carr_freq(track, truth, seed, noise)
    n_ch, _, ms = track.shape
    first, active = orc.find_preambles([track[c, 3] for c in range(n_ch)])
    eph, tow, ready = [None] * 32, 0.0, []
    for ch in active:
        if first[ch] + 30000 > ms:
            continue
        b = orc.nav_bits(track[ch, 3], int(first[ch]))
        e, t = orc.ephemeris(b[1:], b[0])
        eph[int(prn[ch]) - 1] = e
        if e["IODC"] is not None and e["IODE_sf2"] is not None and e["IODE_sf3"] is not None:
            ready.append(ch)
            tow = t
    rdy = np.zeros(n_ch, dtype=np.uint8)
    n_ep = 0
    if len(ready) >= 4:
        rdy[ready] = 1
        n_ep = postnav.nav_epochs(_settings(), np.asarray(first))
    rows = postnav.eph_rows(eph, np.where(rdy > 0, prn, 0))
    return dict(track=track, prn=prn, truth=truth, sfs=np.asarray(first, dtype=np.int32), ready=rdy, eph=rows,
                tow=float(tow), n_ep=n_ep)


_CACHE = {}


def chain_batch(noise=True):
    """The three chain cases stacked: dict with [R, ...] arrays."""
    if noise not in _CACHE:
        cs = [_chain_inputs(s, d, noise) for s, d in SEEDS]
        _CACHE[noise] = dict(track=np.ascontiguousarray(np.stack([c["track"] for c in cs])),
                             sfs=np.stack([c["sfs"] for c in cs]), ready=np.stack([c["ready"] for c in cs]),
                             eph=np.stack([c["eph"] for c in cs]), tow=np.array([c["tow"] for c in cs]),
                             n_ep=np.array([c["n_ep"] for c in cs], dtype=np.int32), truth=[c["truth"] for c in cs])
    return _CACHE[noise]


def ragged_done(b, nav):
    """ms_done [R, C]: all ms except for the first channel of recording 0 that is active at every epoch (it stops after
    the period of epoch 30, so epoch 30 is the last it takes part in) and the last such channel of recording 2 (it
    stops at the period of epoch 10, which it therefore misses)."""
    done = np.full(b["sfs"].shape, NAV_MS, dtype=np.int32)
    c0 = int(np.flatnonzero(nav["active"][0].all(axis=0))[0])
    c2 = int(np.flatnonzero(nav["active"][2].all(axis=0))[-1])
    done[0, c0] = b["sfs"][0, c0] + 500 * 30 + 1
    done[2, c2] = b["sfs"][2, c2] + 500 * 10
    return done, c0, c2


# ---------------------------------------------------------------------------------------------- backends
class Backend(object):
    def __init__(self, name, lib):
        self.name = name
        self.lib = lib
        self._nav = {}

    def nav(self, b, key="noise", mask=ELEV_MASK):
        """sgx_nav_solve on this backend for the batch (host operands), elevation mask `mask`."""
        from softgnss_python_b200 import postnav
        if key not in self._nav:
            tr = b["track"]
            r, c, nf, ms = tr.shape
            self._nav[key] = self.lib.nav_solve(tr, nf * ms, r, c, ms, b["sfs"], b["ready"], b["eph"], b["tow"], b["n_ep"],
                                                postnav.nav_settings(_settings(mask)))
        return self._nav[key]

    def velocity(self, b, nav, vs, ms_done=None, host_in=True, host_out=True, track=None, sl=slice(None)):
        """sgx_nav_velocity on recordings `sl` of the batch; returns numpy outputs (with satVel, satClkDrift)."""
        tr = np.ascontiguousarray(b["track"][sl] if track is None else track)
        r, c, nf, ms = tr.shape
        args = [b["sfs"][sl], b["eph"][sl], b["tow"][sl], b["n_ep"][sl]]
        active, sol = np.ascontiguousarray(nav["active"][sl]), np.ascontiguousarray(nav["sol"][sl])
        done = None if ms_done is None else np.ascontiguousarray(ms_done[sl])
        shp = active.shape
        if self.name == "gpu" and not (host_in and host_out):
            import torch
            keep = []
            if not host_in:
                tr_d = torch.from_numpy(tr).cuda()
                active_d, sol_d = torch.from_numpy(active).cuda(), torch.from_numpy(sol).cuda()
                carr, keep = tr_d.data_ptr() + 16 * ms, [tr_d]
            else:
                active_d, sol_d, carr = active, sol, tr.ctypes.data + 16 * ms
            out = None
            if not host_out:
                z = lambda s: torch.full(s, -1.0, dtype=torch.float64, device="cuda")
                out = dict(vel=z(shp[:2] + (8,)), doppler=z(shp), rrResid=z(shp), satVel=z(shp + (3,)), satClkDrift=z(shp))
            res = self.lib.nav_velocity(carr, nf * ms, r, c, ms, done, *args, active_d, sol_d, vs, want_sat=True,
                                        out=out)
            torch.cuda.synchronize()
            del keep
            return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in res.items()}
        return self.lib.nav_velocity(tr.ctypes.data + 16 * ms, nf * ms, r, c, ms, done, *args, active, sol, vs,
                                     want_sat=True)

    def last_error(self):
        return self.lib.dll.sgx_last_error().decode()


@pytest.fixture(scope="module", params=[pytest.param("gpu", marks=pytest.mark.gpu),
                                        pytest.param("emul", marks=pytest.mark.emul)])
def backend(request):
    from softgnss_python_b200 import _native
    if request.param == "gpu":
        L = _native.lib()
        L.require_device()
        return Backend("gpu", L)
    if os.environ.get("SGX_EMUL_TESTS") != "1" or not os.path.exists(EMUL_LIB):
        pytest.skip("CPU emulator tests: set SGX_EMUL_TESTS=1 and build %s with tools/cpu_emul/build_emul.sh" % EMUL_LIB)
    return Backend("emul", _native.Lib(EMUL_LIB))


@pytest.fixture(autouse=True)
def default_env(monkeypatch):
    monkeypatch.delenv("SGX_EMUL_HOST", raising=False)


def oracle_batch(b, nav, ms_done=None, **kw):
    """Oracle outputs stacked over the recordings of the batch."""
    r, c, _, ms = b["track"].shape
    outs = []
    for i in range(r):
        done = np.full(c, ms) if ms_done is None else ms_done[i]
        outs.append(vor.nav_velocity(b["track"][i, :, 2], done, b["sfs"][i], b["eph"][i], b["tow"][i], int(b["n_ep"][i]),
                                     nav["active"][i], nav["sol"][i], IF, **kw))
    return {k: np.stack([o[k] for o in outs]) for k in outs[0]}


# Tolerances: 10x the largest deviation from the oracle over the three chain cases, ragged ms_done included (CPU
# emulator; the B200 values are in DESIGN.md K10).  The velocity error of a rounding-level difference in the normal
# equations grows with their condition number, i.e. with GDOP^2: recording 2 keeps four satellites at GDOP ~900 under
# the 25 degree mask.  Observed |dv| / GDOP^2 <= 1.8e-13 (1.7e-11 m/s at GDOP 9.7, 7.1e-8 m/s at GDOP 995).
TOL_VEL_PER_GDOP2 = 2e-12  # m/s
TOL_DOPPLER = 0.0          # Hz: the same sum in the same order
TOL_SATVEL = 3e-11         # m/s (observed 2.6e-12)
TOL_SATCLK = 1e-20         # s/s (observed 0; the values are ~1e-12)
TOL_RESID = 1e-9           # m/s (observed 8.6e-11)


def compare(got, want, gdop, label):
    """NaN patterns identical, values within the tolerances (velocity: per epoch, TOL_VEL_PER_GDOP2 * GDOP^2 with gdop
    [R, E]); returns the largest deviation per output (velocity: as a ratio to GDOP^2)."""
    worst = {}
    for k, tol in (("vel", None), ("doppler", TOL_DOPPLER), ("rrResid", TOL_RESID), ("satVel", TOL_SATVEL),
                   ("satClkDrift", TOL_SATCLK)):
        g, w = got[k], want[k]
        assert g.shape == w.shape, (label, k, g.shape, w.shape)
        assert np.array_equal(np.isnan(g), np.isnan(w)), "%s %s: NaN pattern" % (label, k)
        fin = np.isfinite(w)
        if k == "vel":
            assert np.array_equal(g[..., 7], w[..., 7]), label + " channels used"
            d = np.where(fin, np.abs(g - w), 0.0)[..., :7].max(-1)
            ratio = d / np.maximum(gdop, 1.0) ** 2
            worst[k] = float(ratio.max())
            assert worst[k] <= TOL_VEL_PER_GDOP2, "%s vel: |dv| / GDOP^2 = %.3g > %.3g (|dv| %.3g)" % (
                label, worst[k], TOL_VEL_PER_GDOP2, d.max())
            continue
        worst[k] = float(np.abs(g[fin] - w[fin]).max()) if fin.any() else 0.0
        assert worst[k] <= tol, "%s %s: max deviation %.3g > %.3g" % (label, k, worst[k], tol)
    return worst


# ---------------------------------------------------------------------------------------------- 1. oracle parity
@pytest.mark.parametrize("ragged", [False, True])
def test_parity_with_oracle(backend, ragged):
    """Every output against the oracle on the three chain cases: all ms tracked, and ragged ms_done; the elevation mask
    drops channels, seed 5 has no fix, and recordings 0 and 2 have epochs past their n_epochs only if the counts differ
    (the NaN rows of recording 1 cover that)."""
    b = chain_batch()
    nav = backend.nav(b)
    done, c0, c2 = ragged_done(b, nav) if ragged else (None, 0, 0)
    got = backend.velocity(b, nav, _vs(), ms_done=done)
    want = oracle_batch(b, nav, ms_done=done)
    worst = compare(got, want, nav["sol"][..., 4], "%s ragged=%s" % (backend.name, ragged))
    print(backend.name, "ragged" if ragged else "all ms", {k: "%.2g" % v for k, v in worst.items()})
    vel = got["vel"]
    assert b["n_ep"].tolist() == [63, 0, 63]
    assert np.isnan(vel[1, :, :7]).all() and (vel[1, :, 7] == 0).all()               # no fix: past n_epochs
    fixed = vel[[0, 2]]
    enough = fixed[..., 7] >= 4                              # recording 2 keeps 4 channels; ragged ms_done leaves 3
    assert np.isfinite(fixed[enough][:, :7]).all() and np.isnan(fixed[~enough][:, :7]).all()
    assert enough.all() != ragged
    masked = b["ready"][:, None, :].astype(bool) & (nav["active"] == 0)
    assert masked[[0, 2], 1:].any(), "the elevation mask drops no channel"
    assert np.isnan(got["doppler"][masked]).all()
    if ragged:
        assert np.isfinite(got["doppler"][0, :31, c0]).all() and np.isnan(got["doppler"][0, 31:, c0]).all()
        assert np.isfinite(got["doppler"][2, :10, c2]).all() and np.isnan(got["doppler"][2, 10:, c2]).all()


# ---------------------------------------------------------------------------------------------- 2. truth recovery
# Noise-free carrFreq of a receiver moving at V_TRUTH with drift DRIFT_TRUTH, under the default 10 degree mask (8 and
# 7 satellites, GDOP <= 6.9).  Largest error observed over the 126 epochs of seeds 2 and 7 (CPU emulator): 0.0071 m/s
# in velocity, 0.0047 m/s in drift.  What the model leaves out: the 100 ms window trails the epoch by 49.5 ms (Doppler
# rates here <= 0.7 Hz/s: < 7 mm/s per channel), the ignored Sagnac rate (< 1 cm/s) and the fix error of 12-23 m
# (a line-of-sight change of ~1e-6 rad).  The bound allows each of them to reach 1-2 cm/s through the geometry.
# (Under the 25 degree mask seed 7 keeps four satellites at GDOP ~900, which scales these mm/s to m/s.)
TRUTH_VEL_MS = 0.05


def test_truth_recovery(backend):
    b = chain_batch(noise=False)
    nav = backend.nav(b, key="clean", mask=10.0)
    got = backend.velocity(b, nav, _vs())
    for r in (0, 2):
        vel = got["vel"][r]
        err_v = np.abs(vel[:, :3] - V_TRUTH).max()
        err_d = np.abs(vel[:, 3] - DRIFT_TRUTH).max()
        print("recording %d: max |v - truth| %.3g m/s, max |drift - truth| %.3g m/s" % (r, err_v, err_d))
        assert err_v < TRUTH_VEL_MS and err_d < TRUTH_VEL_MS
        enu_speed = np.sqrt((vel[:, 4:7] ** 2).sum(1))
        assert np.abs(enu_speed - np.linalg.norm(V_TRUTH)).max() < TRUTH_VEL_MS


def test_satellite_velocity_is_the_derivative_of_satpos():
    """Analytic velocity and clock drift of the oracle against a +-10 ms central difference of oracle satpos, with
    clock terms that are not zero."""
    from oracle import gnss_oracle as orc
    b = chain_batch()
    for r in (0, 2):
        for c in range(8):
            if not b["ready"][r, c]:
                continue
            e = dict(zip(orc.EPH_FIELDS, b["eph"][r, c]))
            e.update(a_f0=1.2e-4, a_f1=3.5e-11, a_f2=1e-18, t_oc=e["t_oe"] - 1000.0)
            for dt in (0.0, 17.3, 31.0):
                t = b["tow"][r] + dt
                _, _, v, clk_drift = vor.sat_state(t, e)
                pp, cp = orc.satpos(t + 0.01, [1], [e])
                pm, cm = orc.satpos(t - 0.01, [1], [e])
                num = (pp[:, 0] - pm[:, 0]) / 0.02
                assert np.abs(v - num).max() < 1e-4, (r, c, v - num)
                assert abs(clk_drift - (cp[0] - cm[0]) / 0.02) < 1e-13


# ---------------------------------------------------------------------------------------------- 4. determinism
def test_deterministic_and_operand_kinds(backend):
    b = chain_batch()
    nav = backend.nav(b)
    done = ragged_done(b, nav)[0]
    kinds = [(True, True)] + ([(False, False), (True, False), (False, True)] if backend.name == "gpu" else [])
    ref = backend.velocity(b, nav, _vs(), ms_done=done)
    for host_in, host_out in kinds + kinds[:1]:
        got = backend.velocity(b, nav, _vs(), ms_done=done, host_in=host_in, host_out=host_out)
        for k in ref:
            assert got[k].tobytes() == ref[k].tobytes(), (k, host_in, host_out)
    for r in range(3):                                       # a recording alone equals its row of the batch
        one = backend.velocity(b, nav, _vs(), ms_done=done, sl=slice(r, r + 1))
        for k in ref:
            assert one[k][0].tobytes() == ref[k][r].tobytes(), (r, k)


# ---------------------------------------------------------------------------------------------- 5. errors, NaN rules
def test_invalid_arguments(backend):
    b = chain_batch()
    nav = backend.nav(b)
    L = backend.lib
    for vs in (_vs(n=0), _vs(n=-5), _vs(period=0.5), _vs(period=float("nan")), _vs(c=0.0), _vs(c=float("inf")),
               _vs(f_l1=-1.0), _vs(f_l1=float("nan")), _vs(if_hz=float("nan"))):
        with pytest.raises(Exception) as ex:
            backend.velocity(b, nav, vs)
        assert getattr(ex.value, "code", None) == SGX_ERR_ARG, backend.last_error()
    tr = b["track"]
    r, c, nf, ms = tr.shape
    out = [np.zeros((r, 63, 8)), np.zeros((r, 63, c)), np.zeros((r, 63, c))]
    common = (b["sfs"].ctypes.data, np.ascontiguousarray(b["eph"]).ctypes.data, b["tow"].ctypes.data,
              b["n_ep"].ctypes.data, 63, nav["active"].ctypes.data, nav["sol"].ctypes.data)

    def call(carr=tr.ctypes.data, stride=nf * ms, n_rec=r, n_ch=c, n_ms=ms, done=None, vs=None, outs=out):
        return L.dll.sgx_nav_velocity(carr, stride, n_rec, n_ch, n_ms, None if done is None else done.ctypes.data,
                                      *common, ctypes.byref(vs or _vs()), *(o.ctypes.data if o is not None else None
                                                                           for o in outs), None, None, None)
    assert call() == SGX_OK
    assert call(n_ch=0) == SGX_ERR_ARG and call(n_ch=33) == SGX_ERR_ARG
    assert call(n_ms=0) == SGX_ERR_ARG and call(stride=ms - 1, n_ms=ms) == SGX_ERR_ARG
    assert call(carr=None) == SGX_ERR_ARG
    assert call(outs=[out[0], None, out[2]]) == SGX_ERR_ARG
    for bad in (-1, ms + 1):
        done = np.full((r, c), ms, dtype=np.int32)
        done[1, 2] = bad
        assert call(done=done) == SGX_ERR_ARG


def test_nan_rules(backend):
    """An epoch whose fix is NaN, or that has fewer than 4 usable channels, is NaN; a Doppler window that starts before
    ms 0 or reaches ms_done excludes the channel."""
    b = chain_batch()
    nav = dict(backend.nav(b))
    nav["sol"] = nav["sol"].copy()
    nav["active"] = nav["active"].copy()
    nav["sol"][0, 5, :3] = np.nan                            # no fix at epoch 5 of recording 0
    act = np.flatnonzero(nav["active"][0, 7])
    nav["active"][0, 7, act[3:]] = 0                         # three channels left at epoch 7
    got = backend.velocity(b, nav, _vs())
    want = oracle_batch(b, nav)
    compare(got, want, nav["sol"][..., 4], backend.name + " NaN rules")
    assert np.isnan(got["vel"][0, 5, :7]).all() and got["vel"][0, 5, 7] == len(np.flatnonzero(nav["active"][0, 5]))
    assert np.isnan(got["rrResid"][0, 5]).all() and np.isfinite(got["doppler"][0, 5, nav["active"][0, 5] > 0]).all()
    assert np.isnan(got["vel"][0, 7, :7]).all() and got["vel"][0, 7, 7] == 3
    assert np.isfinite(got["vel"][0, [4, 6, 8], :7]).all()
    # the window of channel ch at epoch 0 starts at sfs - N + 1: N = sfs + 1 starts at 0 (used), N = sfs + 2 at -1
    ch = int(np.flatnonzero(nav["active"][0, 0])[0])
    sfs = int(b["sfs"][0, ch])
    ok = backend.velocity(b, nav, _vs(n=sfs + 1))
    early = backend.velocity(b, nav, _vs(n=sfs + 2))
    assert np.isfinite(ok["doppler"][0, 0, ch]) and np.isnan(early["doppler"][0, 0, ch])
    assert np.isfinite(early["doppler"][0, 1, ch])
    # ms_done = m excludes epoch 0 (the window would end on a period that was not tracked), m + 1 includes it
    for extra, finite in ((0, False), (1, True)):
        done = np.full(b["sfs"].shape, NAV_MS, dtype=np.int32)
        done[0, ch] = sfs + extra
        g = backend.velocity(b, nav, _vs(), ms_done=done)
        assert np.isfinite(g["doppler"][0, 0, ch]) == finite
        assert np.isnan(g["doppler"][0, 1:, ch]).all()


# ---------------------------------------------------------------------------------------------- 3. end to end (GPU)
# Config 2 (navsynth.build_scenario(seed=2), 37 100 ms, static receiver, no clock drift), tracked on the device and
# solved with post_navigate_batch(velocity=True).  See DESIGN.md K10 for the values measured on a B200.
E2E_EPOCH0_MS = 1.0           # |v| at epoch 0, m/s
E2E_VS_TRUTH_DOPPLER_MS = 1.0  # |v(tracked Doppler) - v(truth Doppler)| at every epoch, m/s


@pytest.mark.gpu
def test_config2_end_to_end():
    import torch
    from softgnss_python_b200 import _native, navsynth, postnav, synth
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import FIELDS, track_batch
    g = np.load(os.path.join(ROOT, "tests", "golden", "c2_full.npz"), allow_pickle=False)
    N = 38192
    ms, total = int(g["ms"]), int(g["total_ms"]) * N
    spec, truth = navsynth.build_scenario(seed=int(g["seed"]))
    L = _native.lib()
    stride = (total + 15) // 16 * 16
    dev = torch.empty((1, stride), dtype=torch.int8, device="cuda")
    sp, bits = _native.make_synth_specs([spec])
    L.synth(dev, stride, total, 0, sp, bits, synth.cos_lut(), _native.ca_chips_int8(), 0)
    s = Settings(msToProcess=float(ms), numberOfChannels=8)
    s.useTropCorr = False
    ch = np.rec.fromarrays([g["ch_PRN"], g["ch_acquiredFreq"], g["ch_codePhase"], ['T'] * len(g["ch_PRN"])],
                           names="PRN,acquiredFreq,codePhase,status")
    out = torch.zeros((1, len(ch), len(FIELDS), ms), dtype=torch.float64, device="cuda")
    rc, out, done = track_batch(dev, [total], [ch], s, out=out)
    assert rc == 0
    prn = np.asarray(g["ch_PRN"]).reshape(1, -1)
    res = postnav.post_navigate_batch(out, prn, s, velocity=True, ms_done=done)
    n_ep = int(res["n_epochs"][0])
    assert n_ep > 50
    vel = res["vel"][0, :n_ep]
    assert np.isfinite(vel[:, :7]).all() and (vel[:, 7] >= 4).all()
    truth_dop = np.array([truth["doppler"][truth["prn"].index(int(p))] for p in prn[0]])
    dop = res["doppler"][0, :n_ep]
    used = np.isfinite(dop)
    err = (dop - truth_dop[None, :])[used]
    rms = float(np.sqrt(np.mean(err ** 2)))
    speed0 = float(np.linalg.norm(vel[0, :3]))
    # the oracle fed with the truth Doppler (constant, as the synthesiser holds it) at the device's fixes
    carr = np.broadcast_to(IF + truth_dop[:, None], (len(ch), ms)).copy()
    want = vor.nav_velocity(carr, done[0], res["subFrameStart"][0], postnav.eph_rows(res["eph"][0], np.where(
        res["ready"][0] > 0, prn[0], 0)), res["tow"][0], n_ep, res["active"][0], res["sol"][0], s.IF, s.c)
    dv = np.sqrt(((vel[:, :3] - want["vel"][:n_ep, :3]) ** 2).sum(1))
    print("config 2: %d epochs; Doppler rms vs truth %.3f Hz (max %.3f); |v| at epoch 0 %.3f m/s (drift %.3f m/s); "
          "|v - v(truth Doppler)| rms %.3f max %.3f m/s; drift vs truth-Doppler drift max %.3f m/s"
          % (n_ep, rms, np.abs(err).max(), speed0, vel[0, 3], np.sqrt(np.mean(dv ** 2)), dv.max(),
             np.abs(vel[:, 3] - want["vel"][:n_ep, 3]).max()))
    assert speed0 < E2E_EPOCH0_MS
    assert dv.max() < E2E_VS_TRUTH_DOPPLER_MS
    assert np.abs(vel[:, 3] - want["vel"][:n_ep, 3]).max() < E2E_VS_TRUTH_DOPPLER_MS


@pytest.mark.gpu
def test_recarray_surface_matches_batch():
    """postNavigateVelocity on a recarray and post_navigate_batch(velocity=True) on the same numbers agree bit for
    bit; post_navigate_batch without velocity returns what it always did."""
    from softgnss_python_b200 import postnav
    from softgnss_python_b200.tracking import RESULT_DTYPE
    b = chain_batch()
    tr = b["track"][0]
    prn = np.array([int(p) for p in build_chain_case(seed=2)[1]])
    s = _settings()
    batch = postnav.post_navigate_batch(tr[None], prn[None], s, velocity=True)
    plain = postnav.post_navigate_batch(tr[None], prn[None], s)
    assert "vel" not in plain and "doppler" not in plain
    for k in ("sol", "rawP", "active"):
        assert np.array_equal(plain[k], batch[k], equal_nan=True)
    recs = np.rec.fromrecords([(b'T',) + tuple(tr[c, f].copy() for f in range(13)) + (int(prn[c]),) for c in range(8)],
                              dtype=RESULT_DTYPE)
    nav, eph, v = postnav.postNavigateVelocity(recs, s)
    assert nav is not None
    for i, f in enumerate(("VX", "VY", "VZ", "clkDrift", "VE", "VN", "VU", "nUsed")):
        assert np.asarray(v[0][f], dtype=np.float64).tobytes() == batch["vel"][0, :, i].tobytes(), f
    assert np.asarray(v[0].doppler).tobytes() == batch["doppler"][0].T.copy().tobytes()
    assert np.array_equal(nav[0].X, batch["sol"][0, :, 0], equal_nan=True)


# ---------------------------------------------------------------------------------------------- 6. CPU only
def test_settings_struct_size():
    from softgnss_python_b200 import _native
    assert ctypes.sizeof(_native.SgxVelSettings) == 40


def test_settings_defaults_and_foreign_settings():
    from softgnss_python_b200.postnav import vel_settings
    from softgnss_python_b200.settings import Settings
    s = Settings()
    assert (s.dopplerAvgMs, s.L1Freq) == (100, 1575.42e6)

    class Foreign(object):                    # the reference's Settings has IF, c and navSolPeriod but no extensions
        IF, c, navSolPeriod = 9548000.0, 299792458.0, 500.0
    for obj in (s, Foreign()):
        v = vel_settings(obj)
        assert (v.doppler_avg_ms, v.f_L1, v.IF, v.c, v.nav_sol_period) == (100, 1575.42e6, 9548000.0, 299792458.0,
                                                                           500.0)
    v = vel_settings(Settings(dopplerAvgMs=20, L1Freq=1575.0e6))
    assert (v.doppler_avg_ms, v.f_L1) == (20, 1575.0e6)


def test_export_and_no_cpu_fallback():
    from softgnss_python_b200 import _native
    assert "sgx_nav_velocity" in _native.EXPORTS
    L = _native.lib()
    assert hasattr(L.dll, "sgx_nav_velocity")
    if L.dll.sgx_device_count() > 0:
        pytest.skip("a CUDA device is present")
    rc = L.dll.sgx_nav_velocity(None, 0, 0, 0, 0, None, None, None, None, None, 0, None, None, ctypes.byref(_vs()),
                                None, None, None, None, None, None)
    assert rc == SGX_ERR_NODEV
    from softgnss_python_b200 import postnav
    with pytest.raises(_native.NativeError):
        postnav.nav_velocity_batch(np.zeros((1, 8, 13, 100)), dict(n_epochs=np.zeros(1, dtype=np.int32),
                                   active=np.zeros((1, 1, 8), dtype=np.uint8), sol=np.zeros((1, 1, 12))),
                                   np.zeros((1, 8)), np.zeros((1, 8, 21)), [0.0], _settings())
