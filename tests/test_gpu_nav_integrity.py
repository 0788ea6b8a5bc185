"""RAIM fault detection and exclusion with protection levels (sgx_nav_integrity, csrc/sgx_nav.cu) against the float64
oracle (tests/integrity_oracle.py), against injected faults of known size, and end to end on the config-2 recording.

The kernel tests run on two backends, as in test_gpu_nav_velocity.py:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).
The inputs are the synthetic chain cases of tests/cases.py, with the fix (sgx_nav_solve) computed on the same backend.
Their pseudoranges are whole-sample quantised (c/fs = 7.85 m, sigma 2.27 m), so a fault-free fix lies metres from the
truth and every bound below is written for that noise floor.  A fault of B metres on channel ch from epoch k on adds
B*1000*samplesPerCode/c samples to that channel's absoluteSample from 250 ms before the code period of epoch k.
"""
import ctypes
import os

import numpy as np
import pytest

from tests import integrity_oracle as ior
from tests.cases import NAV_MS, build_chain_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
SGX_OK, SGX_ERR_ARG, SGX_ERR_NODEV = 0, -2, -4
C_LIGHT = 299792458.0
FS = 38.192e6
SPC = 38192
SIGMA = 5.0
ONSET = 20                                   # first faulted epoch in the detection tests
THRESH, PBIAS = ior.tables()


def _settings(mask=10.0, trop=False, sigma=SIGMA):
    from softgnss_python_b200.settings import Settings
    return Settings(numberOfChannels=8, msToProcess=float(NAV_MS), elevationMask=mask, useTropCorr=trop,
                    raimSigma=sigma)


def _is(sigma=SIGMA, thresh=THRESH, pbias=PBIAS):
    from softgnss_python_b200 import _native
    st = _native.SgxIntegSettings()
    st.sigma = sigma
    st.thresh[:] = list(thresh)
    st.pbias[:] = list(pbias)
    return st


# ---------------------------------------------------------------------------------------------- inputs
_CHAIN = {}


def chain(seed, drop=()):
    """Fault-free chain case: absoluteSample [C, ms], sfs, ready, eph rows, tow, n_epochs, truth; preamble search and
    ephemeris decoding by the oracle (the same bits and values as the device chain)."""
    key = (seed, tuple(drop))
    if key not in _CHAIN:
        from oracle import gnss_oracle as orc
        from softgnss_python_b200 import postnav
        track, prn, truth = build_chain_case(seed=seed, drop=drop)
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
        _CHAIN[key] = dict(abs=np.ascontiguousarray(track[:, 0]), sfs=np.asarray(first, dtype=np.int32), ready=rdy,
                           eph=postnav.eph_rows(eph, np.where(rdy > 0, prn, 0)), tow=float(tow), n_ep=n_ep, truth=truth,
                           prn=prn, track=track)
    return _CHAIN[key]


def faulted(case, ch, bias_m, onset=ONSET):
    """absoluteSample of `case` with a range error of bias_m metres on channel ch from epoch `onset` on."""
    ab = case["abs"].copy()
    if bias_m:
        start = max(int(case["sfs"][ch]) + 500 * onset - 250, 0)
        ab[ch, start:] += bias_m * 1000.0 * SPC / C_LIGHT
    return ab


def relativity_consistent(case):
    """absoluteSample with the satellite's relativistic clock term F e sqrtA sin E taken out of the epochs' samples.
    build_chain_case synthesises geometric ranges without it, but the fix adds the satellite clock correction (which
    includes it) to every pseudorange, so each satellite carries a bias of up to several metres that is nearly constant
    over the recording.  Without it only the quantisation noise is left."""
    from oracle import gnss_oracle as orc
    ab = case["abs"].copy()
    for c in np.flatnonzero(case["ready"]):
        e = dict(zip(orc.EPH_FIELDS, case["eph"][c]))
        e0 = dict(e, a_f0=0.0, a_f1=0.0, a_f2=0.0, T_GD=0.0)
        for ep in range(case["n_ep"]):
            ab[c, int(case["sfs"][c]) + 500 * ep] -= orc.satpos(case["tow"] + 0.5 * ep, [1], [e0])[1][0] * FS
    return ab


def batch(case, abs_list):
    """Recordings of one chain case that differ only in absoluteSample."""
    r = len(abs_list)
    rep = lambda x: np.ascontiguousarray(np.repeat(np.asarray(x)[None], r, axis=0))
    return dict(abs=np.ascontiguousarray(np.stack(abs_list)), sfs=rep(case["sfs"]), ready=rep(case["ready"]),
                eph=rep(case["eph"]), tow=np.full(r, case["tow"]), n_ep=np.full(r, case["n_ep"], dtype=np.int32))


def stack(batches):
    return {k: np.ascontiguousarray(np.concatenate([b[k] for b in batches])) for k in batches[0]}


# ---------------------------------------------------------------------------------------------- backends
class Backend(object):
    def __init__(self, name, lib):
        self.name = name
        self.lib = lib

    def nav(self, b, mask=10.0, trop=False):
        from softgnss_python_b200 import postnav
        r, c, ms = b["abs"].shape
        return self.lib.nav_solve(b["abs"], ms, r, c, ms, b["sfs"], b["ready"], b["eph"], b["tow"], b["n_ep"],
                                  postnav.nav_settings(_settings(mask, trop)), want_sat=False)

    def integrity(self, b, nav, trop=False, st=None, host_in=True, host_out=True, sl=slice(None)):
        """sgx_nav_integrity on recordings `sl`; numpy outputs."""
        from softgnss_python_b200 import postnav
        ns = postnav.nav_settings(_settings(trop=trop))
        st = st or _is()
        ins = [np.ascontiguousarray(nav[k][sl]) for k in ("rawP", "active", "sol")]
        rest = (b["n_ep"][sl], b["eph"][sl], b["tow"][sl])
        if self.name == "gpu" and not (host_in and host_out):
            import torch
            if not host_in:
                ins = [torch.from_numpy(x).cuda() for x in ins]
            out = None
            if not host_out:
                shp = ins[1].shape
                z = lambda s: torch.full(s, -1.0, dtype=torch.float64, device="cuda")
                out = dict(integ=z(tuple(shp[:2]) + (16,)), normResid=z(tuple(shp)))
            res = self.lib.nav_integrity(*ins, *rest, ns, st, out=out)
            torch.cuda.synchronize()
            return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in res.items()}
        return self.lib.nav_integrity(*ins, *rest, ns, st)

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


def oracle(b, nav, sigma=SIGMA, trop=False, recs=None):
    """Oracle integ [R, E, 16], norm_resid [R, E, C] and per-epoch details on the backend's fixes."""
    recs = range(b["abs"].shape[0]) if recs is None else recs
    res = [ior.nav_integrity(nav["rawP"][i], nav["active"][i], nav["sol"][i], b["eph"][i], b["tow"][i],
                             int(b["n_ep"][i]), sigma, THRESH, PBIAS, use_trop_corr=trop) for i in recs]
    return np.stack([x[0] for x in res]), np.stack([x[1] for x in res]), [x[2] for x in res]


def assert_clear_margins(details, label):
    """The cases must not sit on a decision edge: every q at least 1e-6 T from its threshold, and where an exclusion is
    considered, the two smallest SSE_(j) 1e-6 apart (relative) and the smallest 1e-6 T1 from its threshold."""
    for r, rec in enumerate(details):
        for ep, d in enumerate(rec):
            if not d:
                continue
            assert abs(d["q"] - d["T"]) >= 1e-6 * d["T"], "%s rec %d ep %d: q %.9g at T %.9g" % (label, r, ep, d["q"], d["T"])
            if "T1" in d:
                s = np.sort(d["t0"]["sse_j"])
                assert s[1] - s[0] >= 1e-6 * abs(s[1]), "%s rec %d ep %d: SSE_(j) tie %r" % (label, r, ep, s[:2])
                q1 = s[0] / SIGMA ** 2
                assert abs(q1 - d["T1"]) >= 1e-6 * d["T1"], "%s rec %d ep %d: SSE_(j*) at T1" % (label, r, ep)


def rel_dev(got, want):
    """max |got - want| / |want| over the finite entries (same pattern asserted by the caller)."""
    fin = np.isfinite(want)
    if not fin.any():
        return 0.0
    return float((np.abs(got[fin] - want[fin]) / np.abs(want[fin])).max())


# Tolerances against the oracle.  A prefit residual is the difference of two ~2.6e7 m quantities (one ulp: 3.7e-9 m), and
# the device's satpos agrees with numpy's to ~2e-8 m (tests/nav_util.py), so residual-level values are held to
# EPS_RESID_M in metres of residual rather than to a relative bar: w_j through e_j = w_j sigma sqrt(1 - h_j), and q
# through |dSSE| <= 2 sqrt(n SSE) EPS_RESID_M.  Observed on the CPU emulator: 5.9e-9 m (q 4.1e-9 and 7.0e-9 relative).
# HPL and VPL depend on the geometry only, but 1 - h_j cancels for a channel with little redundancy (5 channels at
# GDOP 23): observed 4.6e-10 relative.
EPS_RESID_M = 5e-8
TOL_REL = 1e-9                 # T; and the relative part of q, qFinal
TOL_PL_REL = 1e-8              # HPL, VPL
TOL_FIX_M = 1e-5               # nav_util.POS_M: the exclusion fix (observed 1.6e-8 m)
TOL_ANGLE_DEG = 1e-9           # its latitude and longitude


def compare(got, want, label):
    """Statuses, exclusions and NaN / inf patterns identical; values within the tolerances.  Returns the deviations:
    relative for T, HPL, VPL; in metres of residual for q, qFinal (dSSE / (2 sqrt(n SSE))) and w (sigma sqrt(1-h) dw)."""
    gi, wi = got["integ"], want[0]
    gw, ww = got["normResid"], want[1]
    assert gi.shape == wi.shape and gw.shape == ww.shape, label
    for k in (13, 14, 15, 9):
        assert np.array_equal(gi[..., k], wi[..., k], equal_nan=True), "%s %s:\n%r\n%r" % (
            label, ior.FIELDS[k], gi[..., k], wi[..., k])
    for name, g, w in (("integ", gi, wi), ("normResid", gw, ww)):
        assert np.array_equal(np.isnan(g), np.isnan(w)), "%s %s: NaN pattern" % (label, name)
        assert np.array_equal(np.isinf(g), np.isinf(w)), "%s %s: inf pattern" % (label, name)
    dev = dict(T=rel_dev(gi[..., 8], wi[..., 8]), HPL=rel_dev(gi[..., 11], wi[..., 11]),
               VPL=rel_dev(gi[..., 12], wi[..., 12]), q_m=0.0, qFinal_m=0.0, w_m=0.0)
    for r, rec in enumerate(want[2]):
        for ep, d in enumerate(rec):
            if not d:
                continue
            ch, t0 = d["chans"], d["t0"]
            n = len(ch)
            de = np.abs(gw[r, ep, ch] - ww[r, ep, ch]) * SIGMA_OF[label] * np.sqrt(t0["omh"])
            dev["w_m"] = max(dev["w_m"], float(np.nanmax(np.where(t0["testable"], de, 0.0))))
            for k, key, sse, m in ((7, "q_m", t0["sse"], n), (10, "qFinal_m", d.get("t1", t0)["sse"], n - ("t1" in d))):
                dq = abs(gi[r, ep, k] - wi[r, ep, k]) * SIGMA_OF[label] ** 2
                dev[key] = max(dev[key], dq / (2 * np.sqrt(m * sse)))
                assert dq <= TOL_REL * sse + 2 * np.sqrt(m * sse) * EPS_RESID_M, (label, r, ep, ior.FIELDS[k], dq)
    fin = np.isfinite(wi[..., 0])
    dev["fix_m"] = float(np.abs(gi[..., :4][fin] - wi[..., :4][fin]).max(initial=0.0))
    dev["fix_deg"] = float(np.abs(gi[..., 4:6][fin] - wi[..., 4:6][fin]).max(initial=0.0))
    dev["height_m"] = float(np.abs(gi[..., 6][fin] - wi[..., 6][fin]).max(initial=0.0))
    assert dev["T"] == 0.0, label
    assert dev["HPL"] <= TOL_PL_REL and dev["VPL"] <= TOL_PL_REL, (label, dev)
    assert dev["w_m"] <= EPS_RESID_M, (label, dev)
    assert dev["fix_m"] <= TOL_FIX_M and dev["height_m"] <= TOL_FIX_M, (label, dev)
    assert dev["fix_deg"] <= TOL_ANGLE_DEG, (label, dev)
    return dev


SIGMA_OF = {}                  # label -> sigma of the run compared


# ---------------------------------------------------------------------------------------------- 1. oracle parity
def _parity_cases(backend):
    """(label, batch, mask, trop): fault-free and faulted seeds 2 and 7 and seed 5 with three satellites (no fix) under
    the default mask with the troposphere model on; seed 7 under a 25 degree mask, which keeps 5 channels (a fault there
    can only be flagged), and seed 7 without channel 3, which keeps 4 (no statistic)."""
    s2, s7, s5 = chain(2), chain(7), chain(5, (1, 4, 6, 7, 2))
    b10 = stack([batch(s2, [s2["abs"], faulted(s2, 3, 300.0)]), batch(s7, [s7["abs"], faulted(s7, 5, 300.0)]),
                 batch(s5, [s5["abs"]])])
    s7d = chain(7, (3,))
    nav7 = backend.nav(batch(s7, [s7["abs"]]), mask=25.0)
    ch5 = int(np.flatnonzero(nav7["active"][0].all(axis=0))[0])
    b25 = stack([batch(s7, [faulted(s7, ch5, 1000.0)]), batch(s7d, [s7d["abs"]])])
    return [("mask 10, trop on", b10, 10.0, True), ("mask 25", b25, 25.0, False)]


def test_parity_with_oracle(backend):
    seen = set()
    for label, b, mask, trop in _parity_cases(backend):
        nav = backend.nav(b, mask=mask, trop=trop)
        got = backend.integrity(b, nav, trop=trop)
        want = oracle(b, nav, trop=trop)
        assert_clear_margins(want[2], label)
        SIGMA_OF["%s %s" % (backend.name, label)] = SIGMA
        dev = compare(got, want, "%s %s" % (backend.name, label))
        print(backend.name, label, {k: "%.2g" % v for k, v in dev.items()})
        seen |= set(np.unique(got["integ"][..., 13]).astype(int).tolist())
        if mask == 25.0:
            assert set(got["integ"][0, 1:63, 15].tolist()) == {5.0} and set(got["integ"][1, 1:63, 15].tolist()) == {4.0}
            assert (got["integ"][0, ONSET + 1:63, 13] == ior.FAULT).all()
            assert (got["integ"][1, 1:63, 13] == ior.UNAVAILABLE).all()     # epoch 0 is unmasked (5 channels)
            assert np.isnan(got["integ"][1, 1:63][:, [7, 8, 10, 11, 12]]).all()
    assert seen == {ior.NO_FIX, ior.UNAVAILABLE, ior.OK, ior.EXCLUDED, ior.FAULT}, seen


# ---------------------------------------------------------------------------------------------- 2. detection truth
BIASES = (300.0, 1000.0)


def _detection_runs(backend):
    """Per seed: fault-free run plus one recording per (B, channel), fix and integrity on the backend, and the oracle
    on the same fixes."""
    runs = {}
    for seed in (2, 7):
        case = chain(seed)
        abs_list = [case["abs"]] + [faulted(case, ch, bias) for bias in BIASES for ch in range(8)]
        b = batch(case, abs_list)
        nav = backend.nav(b)
        runs[seed] = (b, nav, backend.integrity(b, nav), oracle(b, nav))
    return runs


def test_detection_and_exclusion(backend):
    runs = _detection_runs(backend)
    for bi, bias in enumerate(BIASES):
        separable = []
        for seed, (b, nav, got, want) in runs.items():
            gi, base = got["integ"], got["integ"][0]
            assert (base[:63, 13] == ior.OK).all(), "B = 0 must be OK at every epoch"
            for ch in range(8):
                r = 1 + 8 * bi + ch
                # before the onset the recording is the fault-free one, bit for bit
                assert gi[r, :ONSET].tobytes() == base[:ONSET].tobytes(), (seed, ch, bias)
                assert got["normResid"][r, :ONSET].tobytes() == got["normResid"][0, :ONSET].tobytes()
                sep = True
                for ep in range(ONSET, 63):
                    d = want[2][r][ep]
                    k = list(d["chans"]).index(ch)
                    others = np.delete(d["t0"]["sse_j"], k) / SIGMA ** 2
                    sep &= bool(d["q"] > d["T"] and d["t0"]["sse_j"][k] / SIGMA ** 2 <= d["T1"] and (others > d["T1"]).all())
                if sep:
                    separable.append((seed, ch))
                    assert (gi[r, ONSET:63, 13] == ior.EXCLUDED).all() and (gi[r, ONSET:63, 14] == ch).all(), (
                        seed, ch, bias, gi[r, ONSET:63, 13], gi[r, ONSET:63, 14])
        print("%s: B = %g m: %d of 16 faults separable at every epoch from onset: %s" % (
            backend.name, bias, len(separable), separable))
        assert len(separable) >= 8
    # the exclusion fix does not depend on the size of the excluded error (its position; dt may differ by whole
    # milliseconds of c when the faulted channel moves the minimum travel time that the pseudoranges are relative to)
    for seed, (b, nav, got, want) in runs.items():
        gi = got["integ"]
        for ch in range(8):
            r3, r10 = 1 + ch, 9 + ch
            both = (gi[r3, ONSET:63, 13] == ior.EXCLUDED) & (gi[r10, ONSET:63, 13] == ior.EXCLUDED) & \
                   (gi[r3, ONSET:63, 14] == ch) & (gi[r10, ONSET:63, 14] == ch)
            d = np.abs(gi[r3, ONSET:63, :3] - gi[r10, ONSET:63, :3])[both]
            assert d.size == 0 or d.max() <= 1e-3, (seed, ch, d.max())


# ---------------------------------------------------------------------------------------------- 3. protection levels
PL_BIASES = tuple(np.arange(0.0, 101.0, 5.0))


def _enu(sol):
    lat, lon = np.radians(sol[..., 9]), np.radians(sol[..., 10])
    sl, cl, sb, cb = np.sin(lon), np.cos(lon), np.sin(lat), np.cos(lat)
    return np.stack([np.stack([-sl, cl, 0 * sl], -1), np.stack([-sb * cl, -sb * sl, cb], -1),
                     np.stack([cb * cl, cb * sl, sb], -1)], -2)


def test_protection_levels_bound_the_error(backend):
    """At every OK epoch with a fault of 0..100 m on one channel (from epoch 0), the fix's horizontal and vertical
    displacement from the fault-free fix are within HPL and VPL.  Holds by construction when the fault-free parity
    residual sqrt(SSE) is below sigma (sqrt(lambda) - sqrt(T)); that premise is asserted on the oracle."""
    worst = 0.0
    n_ok = 0
    for seed in (2, 7):
        case = chain(seed)
        base_b = batch(case, [case["abs"]])
        base_nav = backend.nav(base_b)
        wi = oracle(base_b, base_nav)[0][0]
        dof = wi[:63, 9].astype(int)
        margin = SIGMA * (PBIAS[dof - 1] - np.sqrt(THRESH[dof - 1]))
        parity = SIGMA * np.sqrt(wi[:63, 7])
        assert (parity < margin).all(), (seed, parity.max(), margin.min())
        rot = _enu(base_nav["sol"][0])
        for ch in range(8):
            b = batch(case, [faulted(case, ch, bias, onset=0) for bias in PL_BIASES])
            nav = backend.nav(b)
            gi = backend.integrity(b, nav)["integ"]
            ok = gi[:, :63, 13] == ior.OK
            dx = gi[:, :63, :3] - base_nav["sol"][0, None, :63, :3]
            enu = np.einsum("eij,rej->rei", rot[:63], dx)
            h, v = np.hypot(enu[..., 0], enu[..., 1]), np.abs(enu[..., 2])
            assert (h[ok] <= gi[:, :63, 11][ok]).all() and (v[ok] <= gi[:, :63, 12][ok]).all(), (seed, ch)
            n_ok += int(ok.sum())
            worst = max(worst, float(np.max(np.maximum(h / gi[:, :63, 11], v / gi[:, :63, 12])[ok])))
    print("%s: %d OK epochs, largest displacement / protection level %.3f" % (backend.name, n_ok, worst))


# ---------------------------------------------------------------------------------------------- 4. statistic scaling
SIGMA_Q = C_LIGHT / FS / np.sqrt(12)          # the quantisation sigma of the synthetic pseudoranges


def test_statistic_scaling(backend):
    """With the true sigma the mean of q / dof over the fault-free epochs is near 1: catches sigma versus sigma^2 and
    an off-by-one in dof.  The satellites' relativistic clock term is made consistent first (see relativity_consistent;
    with it left in, the oracle gives 1.77 and 1.25 for seeds 2 and 7)."""
    qd = []
    for seed in (2, 7):
        case = chain(seed)
        b = batch(case, [relativity_consistent(case)])
        nav = backend.nav(b)
        got = backend.integrity(b, nav, st=_is(sigma=SIGMA_Q))["integ"][0, :63]
        want = oracle(b, nav, sigma=SIGMA_Q)[0][0, :63]
        assert 0.7 <= np.mean(want[:, 7] / want[:, 9]) <= 1.3           # the premise, on the oracle
        qd.append(got[:, 7] / got[:, 9])
    m = float(np.mean(np.concatenate(qd)))
    print("%s: mean q/dof %.3f (seed 2 %.3f, seed 7 %.3f)" % (backend.name, m, qd[0].mean(), qd[1].mean()))
    assert 0.7 <= m <= 1.3


# ---------------------------------------------------------------------------------------------- 5. determinism
def test_deterministic_and_operand_kinds(backend):
    s2, s7 = chain(2), chain(7)
    b = stack([batch(s2, [faulted(s2, 3, 300.0)]), batch(s7, [s7["abs"], faulted(s7, 1, 1000.0)])])
    nav = backend.nav(b)
    kinds = [(True, True)] + ([(False, False), (True, False), (False, True)] if backend.name == "gpu" else [])
    ref = backend.integrity(b, nav)
    for host_in, host_out in kinds + kinds[:1]:
        got = backend.integrity(b, nav, host_in=host_in, host_out=host_out)
        for k in ref:
            assert got[k].tobytes() == ref[k].tobytes(), (k, host_in, host_out)
    for r in range(3):                                       # a recording alone equals its row of the batch
        one = backend.integrity(b, nav, sl=slice(r, r + 1))
        for k in ref:
            assert one[k][0].tobytes() == ref[k][r].tobytes(), (r, k)


# ---------------------------------------------------------------------------------------------- 6. arguments
def test_invalid_arguments(backend):
    from softgnss_python_b200 import postnav
    case = chain(2)
    b = batch(case, [case["abs"]])
    nav = backend.nav(b)
    L = backend.lib
    bad_tables = []
    for arr in ("thresh", "pbias"):
        for v in (0.0, -1.0, float("nan"), float("inf")):
            t, p = THRESH.copy(), PBIAS.copy()
            (t if arr == "thresh" else p)[7] = v
            bad_tables.append(_is(thresh=t, pbias=p))
    for st in [_is(sigma=v) for v in (0.0, -5.0, float("nan"), float("inf"))] + bad_tables:
        with pytest.raises(Exception) as ex:
            backend.integrity(b, nav, st=st)
        assert getattr(ex.value, "code", None) == SGX_ERR_ARG, backend.last_error()
    r, e, c = nav["active"].shape
    integ, res = np.zeros((r, e, 16)), np.zeros((r, e, c))
    ns = postnav.nav_settings(_settings())
    ptr = lambda x: None if x is None else x.ctypes.data

    def call(raw=nav["rawP"], act=nav["active"], sol=nav["sol"], n_rec=r, n_ch=c, e_max=e, nep=b["n_ep"], eph=b["eph"],
             tow=b["tow"], st=ns, ist=None, outs=(integ, res)):
        return L.dll.sgx_nav_integrity(ptr(raw), ptr(act), ptr(sol), n_rec, n_ch, e_max, ptr(nep), ptr(eph), ptr(tow),
                                       None if st is None else ctypes.byref(st),
                                       ctypes.byref(ist or _is()), ptr(outs[0]), ptr(outs[1]), None)
    assert call() == SGX_OK
    assert call(n_ch=0) == SGX_ERR_ARG and call(n_ch=33) == SGX_ERR_ARG
    assert call(e_max=-1) == SGX_ERR_ARG and call(n_rec=-1) == SGX_ERR_ARG
    assert call(n_rec=0) == SGX_OK and call(e_max=0) == SGX_OK
    for kw in (dict(raw=None), dict(act=None), dict(sol=None), dict(nep=None), dict(eph=None), dict(tow=None),
               dict(st=None), dict(outs=(None, res)), dict(outs=(integ, None))):
        assert call(**kw) == SGX_ERR_ARG, kw
    for period, cl in ((0.5, C_LIGHT), (float("nan"), C_LIGHT), (500.0, 0.0), (500.0, float("inf"))):
        s = postnav.nav_settings(_settings())
        s.nav_sol_period, s.c = period, cl
        assert call(st=s) == SGX_ERR_ARG, (period, cl)


def test_settings_struct_size():
    from softgnss_python_b200 import _native
    assert ctypes.sizeof(_native.SgxIntegSettings) == 8 + 2 * 8 * 28
    assert len(_native.NAV_INTEG_FIELDS) == 16 and _native.INTEG_STATUS == ior.STATUS
    assert _native.NAV_INTEG_FIELDS == ior.FIELDS


def test_settings_defaults_and_foreign_settings():
    from softgnss_python_b200.postnav import integ_settings
    from softgnss_python_b200.settings import Settings
    s = Settings()
    assert (s.raimSigma, s.raimPfa, s.raimPmd) == (5.0, 1e-5, 1e-3)

    class Foreign(object):                    # the reference's Settings has none of the extension attributes
        pass
    for obj in (s, Foreign()):
        st = integ_settings(obj)
        assert st.sigma == 5.0
        assert np.abs(np.array(st.thresh) / THRESH - 1).max() < 1e-10
        assert np.abs(np.array(st.pbias) / PBIAS - 1).max() < 1e-10
    st = integ_settings(Settings(raimSigma=3.0, raimPfa=1e-3, raimPmd=1e-2))
    t, p = ior.tables(1e-3, 1e-2)
    assert st.sigma == 3.0 and np.abs(np.array(st.thresh) / t - 1).max() < 1e-10


def test_raim_tables_match_scipy():
    from scipy.stats import chi2, ncx2
    from softgnss_python_b200 import postnav
    dof = np.arange(1, 29)
    for pfa, pmd in ((1e-5, 1e-3), (1e-3, 1e-2), (1e-7, 1e-4)):
        t, p = postnav.raim_tables(pfa, pmd)
        assert t.shape == p.shape == (28,)
        assert np.abs(t / chi2.isf(pfa, dof) - 1).max() <= 1e-10, (pfa, t)
        assert np.abs(ncx2.cdf(t, dof, p ** 2) / pmd - 1).max() <= 1e-10, (pmd, p)
        _, p_ref = ior.tables(pfa, pmd)
        assert np.abs(p / p_ref - 1).max() <= 1e-10
    t, p = postnav.raim_tables(1e-5, 1e-3)
    assert abs(t[3] - 28.473) < 1e-3 and abs(p[3] - 8.200) < 1e-3


def test_export_and_no_cpu_fallback():
    from softgnss_python_b200 import _native, postnav
    assert "sgx_nav_integrity" in _native.EXPORTS
    L = _native.lib()
    assert hasattr(L.dll, "sgx_nav_integrity")
    if L.dll.sgx_device_count() > 0:
        pytest.skip("a CUDA device is present")
    rc = L.dll.sgx_nav_integrity(None, None, None, 0, 0, 0, None, None, None, None, ctypes.byref(_is()), None, None,
                                 None)
    assert rc == SGX_ERR_NODEV
    nav = dict(rawP=np.zeros((1, 1, 8)), active=np.zeros((1, 1, 8), dtype=np.uint8), sol=np.zeros((1, 1, 12)),
               n_epochs=np.zeros(1, dtype=np.int32))
    with pytest.raises(_native.NativeError):
        postnav.nav_integrity_batch(nav, np.zeros((1, 8, 21)), [0.0], _settings())


# ---------------------------------------------------------------------------------------------- 7. end to end (GPU)
def _config2_tracked():
    import torch
    from softgnss_python_b200 import _native, navsynth, synth
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import FIELDS, track_batch
    g = np.load(os.path.join(ROOT, "tests", "golden", "c2_full.npz"), allow_pickle=False)
    ms, total = int(g["ms"]), int(g["total_ms"]) * SPC
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
    return out, np.asarray(g["ch_PRN"]).reshape(1, -1), s, truth


def synth_model_spread(truth, n_ep, period_s=0.5):
    """Per epoch, the spread over the satellites of the config-2 synthesiser's range-model error.  build_scenario holds
    each satellite's Doppler at its value at tow, so the synthetic code phase follows rho0 + rhodot0 * t while the
    ephemeris range curves away by ~rhoddot t^2 / 2; the common part goes into the clock, the spread stays in the
    residuals."""
    from softgnss_python_b200 import navsynth
    err = []
    for e, rho0 in zip(truth["eph"], truth["range"]):
        r1 = navsynth.geometric_range(e, truth["tow"] + 1.0, truth["rx"])[0]
        err.append([navsynth.geometric_range(e, truth["tow"] + t, truth["rx"])[0] - (rho0 + (r1 - rho0) * t)
                    for t in period_s * np.arange(n_ep)])
    err = np.array(err)
    return err.max(0) - err.min(0)


E2E_CLEAN_M = 3.0              # epochs whose synthesiser model spread is below this are held to the defaults
E2E_ONSET = 8                  # first epoch of the injected 300 m step


@pytest.mark.gpu
def test_config2_end_to_end():
    """Config 2 synthesised, tracked and solved on the device with post_navigate_batch(integrity=True) at the default
    raimSigma / raimPfa / raimPmd.  Every epoch whose synthesiser model spread is below E2E_CLEAN_M is OK; the later
    epochs are flagged because the synthesiser's constant-Doppler ranges drift from the ephemeris by up to ~19 m across
    the satellites (synth_model_spread), and the printout reports them.  A 300 m step written into one channel's
    absoluteSample in the CUDA tracking tensor is excluded at every such epoch from its onset."""
    from softgnss_python_b200 import postnav
    out, prn, s, truth = _config2_tracked()
    res = postnav.post_navigate_batch(out, prn, s, integrity=True)
    n_ep = int(res["n_epochs"][0])
    assert n_ep > 50
    integ = res["integ"][0, :n_ep]
    spread = synth_model_spread(truth, n_ep)
    clean = spread < E2E_CLEAN_M
    qd = integ[:, 7] / integ[:, 9]
    print("config 2: %d epochs, status counts %s (first not OK: %s); q/dof min %.3f median %.3f max %.3f, over the %d "
          "epochs with model spread < %g m: median %.3f max %.3f; median HPL %.1f m, VPL %.1f m; dof %s" % (
              n_ep, np.bincount(integ[:, 13].astype(int), minlength=5).tolist(),
              np.flatnonzero(integ[:, 13] != ior.OK)[:1].tolist(), np.nanmin(qd), np.nanmedian(qd), np.nanmax(qd),
              int(clean.sum()), E2E_CLEAN_M, np.median(qd[clean]), qd[clean].max(), np.nanmedian(integ[:, 11]),
              np.nanmedian(integ[:, 12]), np.unique(integ[:, 9]).tolist()))
    assert clean[:20].all()
    assert (integ[clean, 13] == ior.OK).all()
    ch = int(np.flatnonzero(res["active"][0, :n_ep].all(axis=0))[0])
    start = int(res["subFrameStart"][0, ch]) + 500 * E2E_ONSET - 250
    out[0, ch, 0, start:] += 300.0 * 1000.0 * s.samplesPerCode / s.c
    bad = postnav.post_navigate_batch(out, prn, s, integrity=True)["integ"][0, :n_ep]
    sel = clean & (np.arange(n_ep) >= E2E_ONSET)
    print("config 2 with 300 m on channel %d from epoch %d: statuses %s, excluded %s at the %d clean epochs" % (
        ch, E2E_ONSET, np.unique(bad[sel, 13]).tolist(), np.unique(bad[sel, 14]).tolist(), int(sel.sum())))
    assert (bad[sel, 13] == ior.EXCLUDED).all() and (bad[sel, 14] == ch).all()
    assert bad[:E2E_ONSET].tobytes() == integ[:E2E_ONSET].tobytes()


# ---------------------------------------------------------------------------------------------- 8. recarray form
@pytest.mark.gpu
def test_recarray_surface_matches_batch():
    """postNavigateIntegrity on a recarray and post_navigate_batch(integrity=True) on the same numbers agree bit for
    bit; post_navigate_batch without integrity returns what it always did."""
    from softgnss_python_b200 import postnav
    from softgnss_python_b200.tracking import RESULT_DTYPE
    case = chain(2)
    tr = case["track"].copy()
    tr[3, 0] = faulted(case, 3, 300.0)[3]
    prn = np.asarray(case["prn"])
    s = _settings()
    b = postnav.post_navigate_batch(tr[None], prn[None], s, integrity=True)
    plain = postnav.post_navigate_batch(tr[None], prn[None], s)
    assert "integ" not in plain and "normResid" not in plain
    for k in ("sol", "rawP", "active"):
        assert np.array_equal(plain[k], b[k], equal_nan=True)
    assert (b["integ"][0, ONSET:63, 13] == ior.EXCLUDED).any()
    recs = np.rec.fromrecords([(b'T',) + tuple(tr[c, f].copy() for f in range(13)) + (int(prn[c]),) for c in range(8)],
                              dtype=RESULT_DTYPE)
    nav, eph, g = postnav.postNavigateIntegrity(recs, s)
    assert nav is not None
    from softgnss_python_b200 import _native
    for i, f in enumerate(_native.NAV_INTEG_FIELDS):
        assert np.asarray(g[0][f], dtype=np.float64).tobytes() == b["integ"][0, :, i].tobytes(), f
    assert np.asarray(g[0].normResid).tobytes() == b["normResid"][0].T.copy().tobytes()
    assert np.array_equal(nav[0].X, b["sol"][0, :, 0], equal_nan=True)
