"""The three stages between tracking and the position fix against the float64 oracle (oracle/gnss_oracle.py), at the
shapes and edges where they can go wrong:
  K6 sgx_find_preambles  (bitsync_kernel)     -- exact: first subframe, the 1501 nav bits, nav_bits_valid;
  K7 sgx_pseudoranges    (pseudorange_kernel) -- bit-identical to calculate_pseudoranges;
  K8 sgx_nav_solve       (nav_solve_kernel)   -- channel lists and rawP exact, everything else within the measured
                                                 bounds below; plus the whole chain (post_navigate_batch).

The kernel tests run on two backends, as in test_gpu_nav_velocity.py:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).
"""
import ctypes
import itertools
import os

import numpy as np
import pytest

from oracle import gnss_oracle as orc
from tests.cases import NAV_MS, _hash_noise, _lnav_ms, build_chain_case, oracle_chain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
SGX_ERR_RANGE = -5
C_LIGHT = 299792458.0
OMEGA_E = 7.2921151467e-5            # satpos's Earth rotation rate
HALF_WEEK = 302400.0
MAX_PREAMBLE_MS = 819072             # longest record sgx_find_preambles accepts (200 KB of shared memory)
PRE_MS = np.repeat(orc.PREAMBLE_BITS, 20)

# K8 bounds: the largest deviation from the oracle a run may show.  Observed maxima over every case of this file, on a
# B200 at 1000 W | under the CPU emulator:
#   POS_M          X, Y, Z, dt, height, correctedP (m)                       7.4e-8 | 6.6e-8
#   POS_PER_GDOP2  the same in the high-GDOP case, over GDOP^2 (m)           1.5e-10 | 1.7e-10
#   ANGLE_DEG      latitude, longitude, el, az (degrees)                     2.2e-12 | 1.7e-12
#   DOP_REL        GDOP .. TDOP, relative                                    4.4e-13 | 5.0e-13
#   SAT_M          satellite ECEF position (m)                               2.4e-8 | 2.4e-8
#   CLK_S          satellite clock correction (s)                            2.7e-23 | 0
# Each bound is within 10x of the larger of the two.  The position error of a rounding-level difference in the normal
# equations grows with their condition number, i.e. with GDOP^2: the high-GDOP case (four satellites, GDOP 51-59)
# reaches 5.1e-7 m under the emulator, so there the position bound is per GDOP^2, as in test_gpu_nav_velocity.py.
# tests/nav_util.py keeps the looser bounds of the older tests.
POS_M = 5e-7
POS_PER_GDOP2 = 1.7e-9
ANGLE_DEG = 2e-11
DOP_REL = 4e-12
SAT_M = 2e-7
CLK_S = 2e-22
BOUNDS = dict(pos=POS_M, pos_gdop2=POS_PER_GDOP2, angle=ANGLE_DEG, dop=DOP_REL, sat=SAT_M, clk=CLK_S)
WORST = {}


# ---------------------------------------------------------------------------------------------- backends
class Backend(object):
    def __init__(self, name, lib):
        self.name = name
        self.lib = lib

    def preambles(self, rows, ms, want_bits=True):
        """sgx_find_preambles on the rows of a [n, stride] array (stride >= ms)."""
        return self.lib.find_preambles(rows, rows.shape[1], rows.shape[0], ms, want_bits=want_bits)

    def nav(self, abs_s, sfs, ready, eph, tow, n_ep, st, max_epochs=None):
        """sgx_nav_solve on [R, C, ms] absoluteSample rows; every output starts as -7 so that a column the kernel leaves
        unwritten shows."""
        from softgnss_python_b200 import _native
        abs_s = np.ascontiguousarray(abs_s, dtype=np.float64)
        r, c, ms = abs_s.shape
        n_ep = np.ascontiguousarray(n_ep, dtype=np.int32).reshape(r)
        e_max = int(n_ep.max()) if max_epochs is None else int(max_epochs)
        shp = (r, e_max, c)
        out = dict(rawP=np.full(shp, -7.0), correctedP=np.full(shp, -7.0), el=np.full(shp, -7.0), az=np.full(shp, -7.0),
                   satPositions=np.full(shp + (3,), -7.0), satClkCorr=np.full(shp, -7.0),
                   active=np.full(shp, 7, dtype=np.uint8), sol=np.full((r, e_max, 12), -7.0))
        args = [np.ascontiguousarray(sfs, dtype=np.int32).reshape(r, c),
                np.ascontiguousarray(ready, dtype=np.uint8).reshape(r, c),
                np.ascontiguousarray(eph, dtype=np.float64).reshape(r, c, 21),
                np.ascontiguousarray(tow, dtype=np.float64).reshape(r), n_ep]
        p = _native._ptr
        self.lib.check(self.lib.dll.sgx_nav_solve(
            p(abs_s), ms, r, c, ms, *[p(a) for a in args], e_max, ctypes.byref(st),
            *[p(out[k]) for k in ("rawP", "correctedP", "el", "az", "satPositions", "satClkCorr", "active", "sol")], None))
        out["n_epochs"] = n_ep
        return out


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


@pytest.fixture(scope="module", autouse=True)
def report_worst():
    """Prints the largest K8 deviations seen per backend (run with -s to see them)."""
    yield
    for (name, k), (v, where) in sorted(WORST.items()):
        print("nav matrix worst %s %-5s %.3g (bound %.3g) at %s" % (name, k, v, BOUNDS[k], where))


# ---------------------------------------------------------------------------------------------- K6 reference
def _corr(i_p):
    """orc.preamble_correlation without its [ms, 160] product: lags 0..M-1 of the signs (NaN, 0 -> -1) against the
    preamble pattern, taps past the end of the record dropped."""
    bits = np.where(np.asarray(i_p, dtype=np.float64) > 0, 1, -1).astype(np.int32)
    padded = np.concatenate([bits, np.zeros(PRE_MS.size, dtype=np.int32)])
    return np.correlate(padded, PRE_MS.astype(np.int32), "valid")[:bits.size]


def ref_preambles(rows, ms):
    """(first, nav_bits [n, 1501], nav_bits_valid) of the oracle for the first ms values of each row."""
    mp = pytest.MonkeyPatch()
    mp.setattr(orc, "preamble_correlation", _corr)
    try:
        first, _ = orc.find_preambles([r[:ms] for r in rows])
    finally:
        mp.undo()
    valid = np.array([f != 0 and f + 30000 <= ms for f in first], dtype=np.int32)
    bits = np.zeros((len(rows), 1501), dtype=np.uint8)
    for i, f in enumerate(first):
        if valid[i]:
            bits[i] = orc.nav_bits(rows[i][:ms], int(f))
    return first, bits, valid


def check_preambles(backend, rows, ms, expect_first=None, want_bits=True):
    """Device against the oracle, exactly; optionally against the first subframe the case was built for."""
    first, bits, valid = backend.preambles(rows, ms, want_bits)
    rf, rb, rv = ref_preambles(rows, ms)
    assert first.tolist() == rf.tolist(), "%s first subframe, ms %d" % (backend.name, ms)
    if want_bits:
        assert valid.tolist() == rv.tolist(), "nav_bits_valid, ms %d" % ms
        assert np.array_equal(bits, rb), "nav bits, ms %d, rows %s" % (ms, np.flatnonzero((bits != rb).any(1)))
    else:
        assert bits is None and valid is None
    if expect_first is not None:
        assert rf.tolist() == list(expect_first), "the case does not exercise what it was built for"
    return first, valid


_LNAV = {}


def lnav_ip(ms, boundary, seed, pol=1, amp=4000.0, noise=1):
    """I_P of an LNAV stream whose subframe boundary lies at ms `boundary` (0..6000), plus hash noise of sigma
    209*noise; the +0.25 keeps every 20 ms sum away from zero."""
    n_sf = (ms + 6000 - boundary) // 6000 + 2
    if _LNAV.get(seed, (0, None))[0] < n_sf:
        _LNAV[seed] = (n_sf, _lnav_ms(seed, n_subframes=n_sf)[0])
    per = _LNAV[seed][1]
    w0 = 6000 - boundary
    return per[w0:w0 + ms] * (amp * pol) + _hash_noise(seed, ms) * noise + 0.25


def rows_of(chans, stride=None, fill=np.inf):
    """[n, stride] array whose first ms columns are the channels; the rest is `fill` (never to be read)."""
    ms = len(chans[0])
    out = np.full((len(chans), stride or ms), fill)
    for i, c in enumerate(chans):
        out[i, :ms] = c
    return out


# ---------------------------------------------------------------------------------------------- K6 tests
def test_correlation_helper_matches_oracle():
    """The np.correlate form used for long records equals the oracle's own, special values and short records
    included (CPU only)."""
    for m in (1, 20, 159, 160, 161, 191, 5000):
        x = _hash_noise(40 + m, m).astype(np.float64)
        x[::7] = 0.0
        x[3::11] = np.nan
        x[5::13] = -0.0
        x[6::17] = np.inf
        x[8::19] = -np.inf
        if m >= 400:
            x[200:360] = np.repeat(orc.PREAMBLE_BITS, 20) * 5.0
        assert np.array_equal(_corr(x), orc.preamble_correlation(x)), m


@pytest.mark.parametrize("ms", [160, 190, 191, 188288, 188289, 196448, 196449, 196480, 196481, MAX_PREAMBLE_MS])
def test_record_lengths(backend, ms):
    """160..191: word 0 changes from the partial-tap path to the full-tap path at ms = 191 (32*w + 31 + 160 <= ms).
    Above that, the dynamic shared memory is two words per 32 ms plus 8 padding words, and a block needs the opt-in
    attribute once it and the kernel's static shared memory pass 48 KB: 188 288 / 188 289 are either side of that with
    the 2 KB static part of the sm_100a build, 196 448 / 196 449 with the 4 bytes of `best` alone, 196 480 / 196 481
    with the dynamic part alone.  819 072: the longest record accepted (200 KB)."""
    if ms < 6000:
        chans = [lnav_ip(ms, b, 11 + i, pol) for i, (b, pol) in enumerate(((0, 1), (20, -1), (31, 1)))]
        chans.append(np.tile(PRE_MS * 100.0 + 0.5, 2)[:ms])        # a full-strength preamble at k = 0 and k = 160
        check_preambles(backend, rows_of(chans), ms, expect_first=[0] * 4)
        return
    chans = [lnav_ip(ms, 3655, 7), lnav_ip(ms, 1234, 8, pol=-1), lnav_ip(ms, 39, 9)]
    check_preambles(backend, rows_of(chans, ms + 5), ms, expect_first=[3655, 1234, 6039])


def test_record_too_long(backend):
    """One millisecond past the limit: SGX_ERR_RANGE before anything is launched or written."""
    n = 2
    ms = MAX_PREAMBLE_MS + 1
    ip = np.zeros((n, ms))
    first = np.full(n, -1, dtype=np.int32)
    bits = np.full((n, 1501), 9, dtype=np.uint8)
    valid = np.full(n, -1, dtype=np.int32)
    L = backend.lib
    before = L.launches()
    rc = L.dll.sgx_find_preambles(ip.ctypes.data, ms, n, ms, first.ctypes.data, bits.ctypes.data, valid.ctypes.data, None)
    assert rc == SGX_ERR_RANGE
    assert "819 072" in L.dll.sgx_last_error().decode()
    assert L.launches() == before
    assert (first == -1).all() and (bits == 9).all() and (valid == -1).all()


def test_preamble_positions(backend):
    """Winners at k mod 32 = 0, 1 and 31 (lanes 0, 1 and 31 of a sign word), at k = 39 (passed over: the reference
    would read I_P[-1:]; k + 6000 wins) and k = 40 (the first lag that is read), in both polarities."""
    ms = NAV_MS
    cases = [(3200, 1), (3201, -1), (3231, 1), (39, -1), (40, 1), (32, 1), (63, -1), (5999, 1)]
    chans = [lnav_ip(ms, b, 20 + i, pol) for i, (b, pol) in enumerate(cases)]
    expect = [b if b >= 40 else b + 6000 for b, _ in cases]
    check_preambles(backend, rows_of(chans, ms + 3), ms, expect_first=expect)


@pytest.mark.parametrize("n_taps", [154, 153, 30])
def test_partner_in_the_last_160_ms(backend, n_taps):
    """The partner of the only complete preamble lies n taps before the end of the record (partial-tap path): with
    n >= 154 it is a candidate, below it is not and nothing is found.  n = 30 is where taps past the end, if they
    were counted as zeros, would agree with 100 - n of the pattern's -1 bits and make the partner a candidate."""
    b = 3000
    ms = b + 6000 + n_taps
    chans = [lnav_ip(ms, b, 31 + i, pol) for i, pol in enumerate((1, -1))]
    expect = [b if n_taps >= 154 else 0] * 2
    check_preambles(backend, rows_of(chans, ms + 1), ms, expect_first=expect)


@pytest.mark.parametrize("extra", [0, -1])
def test_nav_bits_valid_edge(backend, extra):
    """The 1501 bits need first - 20 .. first + 30000: valid at first + 30000 == ms, not at ms - 1."""
    b = 3000
    ms = b + 30000 + extra
    chans = [lnav_ip(ms, b, 41, 1), lnav_ip(ms, b + 17, 42, -1)]
    first, valid = check_preambles(backend, rows_of(chans), ms, expect_first=[b, b + 17])
    assert valid.tolist() == ([1, 0] if extra == 0 else [0, 0])


@pytest.mark.parametrize("pol", [1, -1])
def test_parity_failing_candidates(backend, pol):
    """Eight preamble/partner pairs that fail the parity check, one in a word of each of the eight verification warps
    (word 8 + 9i goes to warp i), with alternating signs, all before the valid subframe at 5000 (word 156)."""
    ms = 17000
    b = 5000
    ip = lnav_ip(ms, b, 50, pol)
    fakes = []
    for i in range(8):
        k = 32 * (8 + 9 * i) + (7 * i) % 32
        s = pol * (1 if i % 2 else -1)
        for kk in (k, k + 6000):
            ip[kk:kk + 160] = s * PRE_MS * 4000.0 + 0.25
        fakes.append(k)
    assert sorted({(k >> 5) % 8 for k in fakes}) == list(range(8))
    corr = _corr(ip)
    assert all(abs(corr[k]) > 153 and abs(corr[k + 6000]) > 153 for k in fakes)
    check_preambles(backend, rows_of([ip], ms + 9), ms, expect_first=[b])


def test_special_values(backend):
    """NaN, +-0 and +-inf in I_P: in the sign bits NaN and both zeros count as -1; in the 20 ms sums a NaN or
    inf - inf gives bit 0 and a lone inf its sign.  Rows of all NaN and all inf find nothing."""
    ms = NAV_MS
    b = 3655
    pre = lnav_ip(ms, b, 61)
    pre[b + 3] = np.nan                               # two taps of the preamble and two of its partner; the NaN
    pre[b + 150] = 0.0                                # also makes one bit of the TLM word 0
    pre[b + 6001] = -0.0
    pre[b + 6100] = np.nan
    ip = lnav_ip(ms, b, 60)
    for j, vals in ((100, (np.inf,)), (200, (-np.inf,)), (300, (np.inf, -np.inf)), (400, (np.nan,)),
                    (500, (0.0, -0.0)), (1499, (np.nan, np.inf))):
        s = b - 20 + 20 * j + 3
        ip[s:s + len(vals)] = vals
    chans = [ip, -ip, pre, -pre, np.full(ms, np.nan), np.full(ms, np.inf), np.zeros(ms)]
    first, _ = check_preambles(backend, rows_of(chans, ms + 2), ms)
    assert first[[0, 1, 4, 5, 6]].tolist() == [b, b, 0, 0, 0] and first[2] in (b, b + 6000, b + 12000)
    bits = backend.preambles(rows_of(chans, ms + 2), ms)[1]
    assert bits[0, 100] == 1 and bits[0, 200] == 0 and bits[0, 300] == 0 and bits[0, 400] == 0


@pytest.mark.parametrize("n_ch", [1, 149, 1000])
@pytest.mark.parametrize("want_bits", [True, False])
def test_batches(backend, n_ch, want_bits):
    """More channels than SMs, rows `stride` > ms apart with +inf between them; every channel against the oracle.
    Channels differ in boundary, polarity, noise and seed; every seventh carries noise only."""
    ms = NAV_MS if n_ch < 1000 else 8000
    chans, expect = [], []
    for i in range(n_ch):
        b = (53 * i) % (5960 if ms == NAV_MS else 1800) + 40
        pol = -1 if i % 5 == 2 else 1
        if i % 7 == 6:
            chans.append(_hash_noise(9000 + i, ms) * 10.0 + 0.25)
            expect.append(None)
        else:
            chans.append(lnav_ip(ms, b, 100 + i % 23, pol, noise=1 + i % 3))
            expect.append(b)
    first, _ = check_preambles(backend, rows_of(chans, ms + 7), ms, want_bits=want_bits)
    for f, e in zip(first, expect):
        assert e is None or f == e


# ---------------------------------------------------------------------------------------------- K7
PR_UNITS = [(1, 1), (1, 7), (2, 4), (3, 3), (33, 9)]      # R x E = 1, 7, 8, 9, 297 (= 8*37 + 1) warps
PR_SPC = [4092, 16368, 38192, 64000]


def _pr_case(n_rec, n_ch, n_ep, spc, ms, seed):
    """absoluteSample rows (integer-valued, one code period per ms with a drift), ms_index and active."""
    noise = _hash_noise(seed, n_rec * n_ch * ms).reshape(n_rec, n_ch, ms)
    start = 1000 + 977 * np.arange(n_rec * n_ch).reshape(n_rec, n_ch, 1) * 13
    abs_s = (start + np.cumsum(spc + noise % 5 - 2, axis=2)).astype(np.float64)
    h = np.abs(_hash_noise(seed + 1, n_rec * n_ep * n_ch)).reshape(n_rec, n_ep, n_ch)
    idx = (h * 7919 % ms).astype(np.int64)
    active = ((h >> 3) % 4 != 0).astype(np.uint8)
    idx[:, 0, 0] = 0
    idx[:, -1, -1] = ms - 1
    active[:, 0, 0] = active[:, -1, -1] = 1
    if n_ep > 2:
        active[:, 1] = 0                                                   # empty list: inf - inf = NaN everywhere
        active[:, 2] = 0
        active[:, 2, n_ch - 1] = 1                                         # a single channel
    if n_ep > 3 and n_ch > 4:
        bad = np.array([-1, ms, -2 ** 31, 2 ** 31 - 1])                     # outside [0, ms): counts as not listed
        idx[:, 3, :4] = bad
        active[:, 3, :] = 1
    return abs_s, idx, active


@pytest.mark.parametrize("n_ch", [1, 5, 31, 32])
@pytest.mark.parametrize("units", PR_UNITS, ids=["%dx%d" % u for u in PR_UNITS])
def test_pseudoranges(backend, n_ch, units):
    n_rec, n_ep = units
    spc = PR_SPC[(n_ch + n_rec + n_ep) % len(PR_SPC)]
    ms = 2500
    start_offset = 12.345
    abs_s, idx, active = _pr_case(n_rec, n_ch, n_ep, spc, ms, seed=n_ch * 100 + n_rec + n_ep)
    track = np.zeros((n_rec, n_ch, 13, ms))
    track[:, :, 0] = abs_s
    track[:, :, 1:] = np.nan                                   # only field 0 may be read
    got = backend.lib.pseudoranges(track, n_rec, n_ch, ms, idx.astype(np.int32), active, spc, start_offset, C_LIGHT)
    for r in range(n_rec):
        for e in range(n_ep):
            listed = [c for c in range(n_ch) if active[r, e, c] and 0 <= idx[r, e, c] < ms]
            want = orc.calculate_pseudoranges(abs_s[r], idx[r, e], listed, n_ch, float(spc), start_offset, C_LIGHT)
            assert got[r, e].tobytes() == want.tobytes(), (backend.name, r, e, got[r, e], want)
    if n_ep > 3 and n_ch > 4:
        assert np.isinf(got[:, 3, :4]).all() and np.isfinite(got[:, 3, 4:]).all()


# ---------------------------------------------------------------------------------------------- K8 cases
def _eph_dict(row):
    return dict(zip(orc.EPH_FIELDS, row))


def _abs_sample(eph, tow, rx, fs, n_code, ms, sfs):
    """absoluteSample rows of channels whose subframe at transmit time `tow` arrives at ms sfs[c] (the quadratic model
    of cases.build_chain_case, from navsynth.geometric_range at tow, tow + 18 s, tow + 36 s)."""
    from softgnss_python_b200 import navsynth
    rho = np.array([[navsynth.geometric_range(e, tow + kk, rx)[0] for kk in (0.0, 18.0, 36.0)] for e in eph])
    rho_min = rho[:, 0].min()
    k = np.arange(ms, dtype=np.float64)
    out = np.zeros((len(eph), ms))
    for c in range(len(eph)):
        s = (rho[c] - rho_min) / navsynth.C * fs
        p2 = ((s[2] - s[0]) - 2 * (s[1] - s[0])) / (2 * 18000.0 ** 2)
        p1 = (s[1] - s[0]) / 18000.0 - p2 * 18000.0
        kr = k - sfs[c]
        out[c] = np.round(sfs[0] * n_code + s[0] + kr * n_code + p1 * kr + p2 * kr * kr)
    return out


def _rebase(e, toe, toc=None):
    """The same orbit with t_oe moved to `toe`: omega_0 absorbs OMEGA_E * (toe - t_oe), so at transmit time t the
    satellite stands where the original stood at t_oe + check_t(t - toe)."""
    e = dict(e)
    e["omega_0"] = e["omega_0"] + OMEGA_E * (toe - e["t_oe"])
    e["t_oe"] = float(toe)
    e["t_oc"] = float(toe if toc is None else toc)
    return e


_SCEN = {}


def _scenario(seed, n_sats, min_elev, rx_llh):
    from softgnss_python_b200 import navsynth
    key = (seed, n_sats, min_elev, rx_llh)
    if key not in _SCEN:
        _SCEN[key] = navsynth.build_scenario(seed=seed, n_sats=n_sats, min_elev=min_elev, rx_llh=rx_llh)[1]
    return _SCEN[key]


def _gdop_subset(truth, n):
    """The n satellites of the scenario whose GDOP at the receiver is closest to 60."""
    from softgnss_python_b200 import navsynth
    rx = truth["rx"]
    u = []
    for e in truth["eph"]:
        d = navsynth.sat_ecef(e, truth["tow"]) - rx
        u.append(d / np.linalg.norm(d))
    best = None
    for sub in itertools.combinations(range(len(u)), n):
        g = np.array([np.append(-u[i], 1.0) for i in sub])
        gd = float(np.sqrt(np.trace(np.linalg.inv(g.T @ g))))
        if best is None or abs(np.log(gd / 60.0)) < abs(np.log(best[0] / 60.0)):
            best = (gd, list(sub))
    return best[1]


# name: build_scenario seed / n_sats / min_elev, padding channels, rate, period, mask, tropo, time base, edits
K8_CASES = {
    "ch4": dict(seed=3, n_sats=4),
    "ch5": dict(seed=4, n_sats=5),
    "ch12": dict(seed=5, n_sats=12, min_elev=5.0),
    "ch31_padded": dict(seed=6, n_sats=12, min_elev=5.0, pad=19),
    "ch32": dict(seed=(7, 19, 23, 29), min_elev=-90.0, mask=0.0),   # PRNs 1..32, half of them below the horizon
    "fs16368_p100": dict(seed=8, fs=16.368e6, period=100.0, mask=0.0),
    "fs64000_p1000": dict(seed=9, fs=64e6, period=1000.0, mask=25.0, rx=(-33.9, 18.4, 30.0)),
    "notrop_mask25": dict(seed=10, n_sats=10, min_elev=5.0, trop=False, mask=25.0),
    "mask90": dict(seed=11, mask=90.0),
    "week_end": dict(seed=12, tow=604795.0, toe=16.0),       # t_oe / t_oc of the next week
    "week_start": dict(seed=13, tow=3.0, toe=604784.0),      # t_oe / t_oc of the week before
    "toc_half_week": dict(seed=14, toc_offset=-HALF_WEEK),   # transmit_time - t_oc == 302400 at epoch 0: no wrap
    "eccentric": dict(seed=15, n_sats=12, min_elev=5.0, ecc=True, rx=(60.0, 25.0, 100.0)),
    "duplicate": dict(seed=16, n_sats=3, dup=True),          # 4 listed channels, 3 satellites: rank 3, zero fix
    "high_gdop": dict(seed=17, n_sats=12, min_elev=5.0, gdop4=True, mask=0.0),
    "three": dict(seed=18, n_sats=3, pad=2),                 # 3 listed channels: no fix
}


def build_nav_case(name):
    """Inputs of sgx_nav_solve for one recording and the oracle's output for them."""
    from softgnss_python_b200 import _native, navsynth
    k = K8_CASES[name]
    fs = k.get("fs", 38.192e6)
    n_code = int(round(fs / 1000.0))
    seeds = k["seed"] if isinstance(k["seed"], tuple) else (k["seed"],)
    truths = [_scenario(sd, k.get("n_sats", 8), k.get("min_elev", 15.0), k.get("rx", (40.0, -105.0, 1600.0)))
              for sd in seeds]
    truth = truths[0]
    ephs = [dict(e) for t in truths for e in t["eph"]]
    tow = float(k.get("tow", truth["tow"]))
    if "gdop4" in k:
        ephs = [ephs[i] for i in _gdop_subset(truth, 4)]
    rng = np.random.default_rng(seeds[0])
    for c, e in enumerate(ephs):
        e.update(a_f0=rng.uniform(-2e-8, 2e-8), a_f1=rng.uniform(-5e-12, 5e-12), a_f2=1e-19 * (c % 3),
                 T_GD=-4.7e-9 * (c % 2), C_rs=12.0 * c, C_rc=-90.0 + 20 * c, C_us=2e-6, C_uc=-1e-6, C_is=6e-8,
                 C_ic=-4e-8, iDot=2e-10, t_oc=e["t_oe"])
        if "toe" in k:
            ephs[c] = e = _rebase(e, k["toe"])
        if "toc_offset" in k:
            e["t_oc"] = tow + k["toc_offset"]
        if k.get("ecc"):
            e["e"] = 0.02 + 0.01 * ((c * 0.37) % 1.0)
            while c == 0 and _kepler_iterations(e, tow) < 10:      # move satellite 0 to where the loop runs to the end
                e["M_0"] += 2e-3
    prn = np.array(truth["prn"] if len(seeds) == 1 else np.arange(1, len(ephs) + 1), dtype=np.int64)
    if "gdop4" in k:
        prn = np.array([truth["prn"][i] for i in _gdop_subset(truth, 4)], dtype=np.int64)
    if k.get("dup"):
        ephs.append(dict(ephs[0]))
        prn = np.append(prn, prn[0])
    sfs = np.array([5200 + (3 * c) % 7 for c in range(len(ephs))], dtype=np.int32)
    abs_s = _abs_sample(ephs, tow, truth["rx"], fs, n_code, NAV_MS, sfs)
    rows = np.array([[e[f] for f in _native.EPH_FIELDS] for e in ephs])
    ready = np.ones(len(ephs), dtype=np.uint8)
    pad = k.get("pad", 0)
    if pad:
        abs_s = np.concatenate([abs_s, _hash_noise(seeds[0], pad * NAV_MS).reshape(pad, NAV_MS) * 1e3 + 5e8])
        sfs = np.concatenate([sfs, np.arange(pad, dtype=np.int32) * 11])
        ready = np.concatenate([ready, np.zeros(pad, dtype=np.uint8)])
        rows = np.concatenate([rows, np.zeros((pad, 21))])
        prn = np.concatenate([prn, np.zeros(pad, dtype=np.int64)])
    st = dict(samples_per_code=float(n_code), start_offset=68.802 + 0.5 * (seeds[0] % 3), c=C_LIGHT,
              nav_sol_period=k.get("period", 500.0), elevation_mask=k.get("mask", 10.0), use_trop_corr=int(k.get("trop", True)))
    n_ep = int(np.fix(NAV_MS - sfs.max()) / st["nav_sol_period"])
    case = dict(name=name, abs=abs_s, prn=prn, sfs=sfs, ready=ready, eph=rows, tow=tow, n_ep=n_ep, st=st)
    case["ref"] = oracle_nav(case)
    return case


def oracle_nav(case, check_t=None):
    st = case["st"]
    eph = [None] * 32
    for c in np.flatnonzero(case["ready"]):
        eph[int(case["prn"][c]) - 1] = _eph_dict(case["eph"][c])
    mp = pytest.MonkeyPatch()
    if check_t is not None:
        mp.setattr(orc, "check_t", check_t)
    try:
        return orc.nav_solve(list(case["abs"]), case["prn"], case["sfs"], np.flatnonzero(case["ready"]), eph, case["tow"],
                             float(NAV_MS), st["samples_per_code"], nav_sol_period=st["nav_sol_period"],
                             elevation_mask=st["elevation_mask"], use_trop_corr=bool(st["use_trop_corr"]),
                             start_offset=st["start_offset"], c=st["c"])
    finally:
        mp.undo()


def nav_settings(st):
    from softgnss_python_b200 import _native
    return _native.SgxNavSettings(st["samples_per_code"], st["start_offset"], st["c"], st["nav_sol_period"],
                                  st["elevation_mask"], st["use_trop_corr"], 0)


_CASES = {}


def nav_case(name):
    if name not in _CASES:
        _CASES[name] = build_nav_case(name)
    return _CASES[name]


def assert_clear_mask(ref, ready, mask):
    """Every elevation the oracle computed for a ready channel is at least 1e-6 degrees from the mask, so that the
    channel lists do not hang on the last digits of el."""
    el = ref["el"][np.flatnonzero(ready)]
    fin = np.isfinite(el)
    assert (np.abs(el[fin] - mask) >= 1e-6).all(), "an elevation lies on the mask"


def compare_nav(out, r, ref, label, backend_name, gdop_scale=False):
    """Channel lists and rawP exactly, the rest within the K8 bounds; epochs past n_epochs hold the initial values."""
    n_ep = int(ref["n_epochs"])
    assert out["n_epochs"][r] == n_ep, label
    act = out["active"][r, :n_ep].T
    assert np.array_equal(act > 0, ref["PRN"] > 0) and set(np.unique(act)) <= {0, 1}, label + " channel lists"
    assert np.array_equal(out["rawP"][r, :n_ep].T, ref["rawP"], equal_nan=True), label + " rawP"
    sol = out["sol"][r, :n_ep]
    gd = np.where(ref["DOP"][0] > 0, ref["DOP"][0], 1.0) if gdop_scale else None

    def close(got, want, kind, name):
        assert got.shape == want.shape, (label, name)
        assert np.array_equal(np.isnan(got), np.isnan(want)), "%s %s: NaN pattern" % (label, name)
        fin = np.isfinite(want)
        err = np.where(fin, np.abs(np.where(fin, got, 0.0) - np.where(fin, want, 0.0)), 0.0)
        if kind == "dop":
            err = err / np.where(fin & (want != 0), np.abs(want), 1.0)
        if gd is not None and kind == "pos":
            err = err / np.maximum(gd, 1.0) ** 2 if err.ndim == 1 else err / np.maximum(gd, 1.0)[None] ** 2
            kind = "pos_gdop2"
        worst = float(err.max()) if err.size else 0.0
        key = (backend_name, kind)
        if worst >= WORST.get(key, (0.0, ""))[0]:
            WORST[key] = (worst, "%s %s" % (label, name))
        assert worst <= BOUNDS[kind], "%s %s: max deviation %.3g > %.3g" % (label, name, worst, BOUNDS[kind])

    for i, name in enumerate(("X", "Y", "Z", "dt")):
        close(sol[:, i], ref[name], "pos", name)
    close(sol[:, 11], ref["height"], "pos", "height")
    close(sol[:, 9], ref["latitude"], "angle", "latitude")
    close(sol[:, 10], ref["longitude"], "angle", "longitude")
    close(sol[:, 4:9].T, ref["DOP"], "dop", "DOP")
    close(out["el"][r, :n_ep].T, ref["el"], "angle", "el")
    close(out["az"][r, :n_ep].T, ref["az"], "angle", "az")
    close(out["correctedP"][r, :n_ep].T, ref["correctedP"], "pos", "correctedP")
    close(out["satPositions"][r, :n_ep].transpose(1, 0, 2), ref["satPositions"], "sat", "satPositions")
    close(out["satClkCorr"][r, :n_ep].T, ref["satClkCorr"], "clk", "satClkCorr")
    # epochs past n_epochs: NaN, no channel, DOP 0 (the reference's initial values)
    pad = slice(n_ep, None)
    for k in ("rawP", "correctedP", "el", "az", "satClkCorr", "satPositions"):
        assert np.isnan(out[k][r, pad]).all(), "%s %s past n_epochs" % (label, k)
    assert (out["active"][r, pad] == 0).all()
    p = out["sol"][r, pad]
    assert np.isnan(p[:, [0, 1, 2, 3, 9, 10, 11]]).all() and (p[:, 4:9] == 0).all(), label + " sol past n_epochs"


def run_case(backend, case, max_epochs=None):
    return backend.nav(case["abs"][None], case["sfs"][None], case["ready"][None], case["eph"][None], [case["tow"]],
                       [case["n_ep"]], nav_settings(case["st"]), max_epochs=max_epochs)


# ---------------------------------------------------------------------------------------------- K8 tests
@pytest.mark.parametrize("name", sorted(K8_CASES))
def test_nav_solve_case(backend, name):
    case = nav_case(name)
    ref = case["ref"]
    assert_clear_mask(ref, case["ready"], case["st"]["elevation_mask"])
    out = run_case(backend, case, max_epochs=case["n_ep"] + 2)
    compare_nav(out, 0, ref, "%s %s" % (backend.name, name), backend.name, gdop_scale=name == "high_gdop")
    fix = np.isfinite(ref["X"]) & (ref["X"] != 0)
    listed = (ref["PRN"] > 0).sum(0)
    if name == "mask90":
        assert listed[0] == len(case["prn"]) and (listed[1:] == 0).all()
    elif name == "duplicate":                                 # el stays 0 after the zero fix: nothing listed after it
        assert listed[0] == 4 and ref["X"][0] == 0 and (out["sol"][0, 0, :4] == 0).all()
    elif name == "three":
        assert (listed == 3).all() and np.isnan(ref["X"]).all()
    else:
        assert fix.all(), "every epoch has a fix"
    if name == "high_gdop":
        assert ref["DOP"][0].min() > 20, ref["DOP"][0]
    if name.startswith("ch"):
        assert out["active"].shape[2] == int(name[2:4])


@pytest.mark.parametrize("name", ["week_end", "week_start", "toc_half_week"])
def test_week_crossover_is_exercised(name):
    """On the oracle side: check_t wraps both t - t_oc and t - t_oe in the two crossover cases, and nothing wraps when
    transmit_time - t_oc is exactly 302 400 s (the test is t > 302400, not >=) (CPU only)."""
    seen = []

    def spy(t):
        seen.append(t)
        return _check_t(t)
    case = nav_case(name)
    oracle_nav(case, check_t=spy)
    wrapped = [t for t in seen if abs(t) > HALF_WEEK]
    if name == "toc_half_week":
        # epoch 0 meets the edge once per listed satellite; later epochs are past it and wrap
        assert seen.count(HALF_WEEK) == (case["ref"]["PRN"][:, 0] > 0).sum() > 0
    else:
        n_sat = (case["ref"]["PRN"] > 0).sum()
        assert len(wrapped) == 2 * n_sat, (len(wrapped), n_sat)        # t_oc and t_oe of every listed satellite


def _check_t(t):
    if t > HALF_WEEK:
        return t - 2 * HALF_WEEK
    if t < -HALF_WEEK:
        return t + 2 * HALF_WEEK
    return t


def _kepler_iterations(e, t):
    """Iterations of satpos's Kepler loop for ephemeris e at transmit time t (the oracle's expressions)."""
    gps_pi, gm = 3.14159265359, 3.986005e+14
    e = {k: np.float64(v) for k, v in e.items()}
    dt = _check_t(t - e["t_oc"])
    clk = (e["a_f2"] * dt + e["a_f1"]) * dt + e["a_f0"] - e["T_GD"]
    a = e["sqrtA"] * e["sqrtA"]
    tk = _check_t(t - clk - e["t_oe"])
    m = np.remainder(e["M_0"] + (np.sqrt(gm / a ** 3) + e["deltan"]) * tk + 2 * gps_pi, 2 * gps_pi)
    ea = m
    for i in range(10):
        old = ea
        ea = m + e["e"] * np.sin(ea)
        if abs(np.remainder(ea - old, 2 * gps_pi)) < 1e-12:
            return i + 1
    return 10


def test_eccentric_case_runs_the_whole_kepler_loop():
    """The eccentric case has a satellite whose Kepler loop stops early and one that runs all ten iterations (CPU
    only)."""
    case = nav_case("eccentric")
    its = [_kepler_iterations(_eph_dict(row), case["tow"]) for row in case["eph"]]
    assert min(its) < 10 and max(its) == 10, its
    assert all(0.02 <= row[9] <= 0.03 for row in case["eph"])


BATCH_KINDS = [("ch5", 5200), ("ch5", 9100), ("ch5", 15003), ("ch5", 5200), ("ch5", 20000)]


def _batch_member(i):
    """Recording i of a batch: the ch5 case with its first subframe moved, which changes n_epochs; every fifth
    recording is given n_epochs = 0 (fewer than four satellites decoded)."""
    base = nav_case("ch5")
    key = ("batch", i % 5)
    if key not in _CASES:
        shift = BATCH_KINDS[i % 5][1] - 5200
        c = dict(base, sfs=base["sfs"] + shift, abs=np.roll(base["abs"], shift, axis=1), name="batch%d" % (i % 5))
        c["n_ep"] = int(np.fix(NAV_MS - c["sfs"].max()) / c["st"]["nav_sol_period"])
        c["tow"] = base["tow"] + 0.5 * (i % 5)
        c["ref"] = oracle_nav(c)
        _CASES[key] = c
    c = dict(_CASES[key])
    if i % 5 == 3:
        c["n_ep"] = 0
    return c


@pytest.mark.parametrize("n_rec", [1, 4, 5, 33])
def test_batch_ragged_epochs(backend, n_rec):
    """R recordings with ragged n_epochs (0 included) and max_epochs past the largest: each recording matches the
    oracle, epochs past its n_epochs hold the initial values, and its row equals its solo run bit for bit."""
    members = [_batch_member(i) for i in range(n_rec)]
    max_ep = max(m["n_ep"] for m in members) + 3
    out = backend.nav(np.stack([m["abs"] for m in members]), np.stack([m["sfs"] for m in members]),
                      np.stack([m["ready"] for m in members]), np.stack([m["eph"] for m in members]),
                      [m["tow"] for m in members], [m["n_ep"] for m in members], nav_settings(members[0]["st"]),
                      max_epochs=max_ep)
    for r, m in enumerate(members):
        ref = m["ref"] if m["n_ep"] else dict(m["ref"], n_epochs=0, **{k: m["ref"][k][..., :0] for k in (
            "PRN", "el", "az", "rawP", "correctedP", "DOP", "X", "Y", "Z", "dt", "latitude", "longitude", "height",
            "satClkCorr")}, satPositions=m["ref"]["satPositions"][:, :0])
        compare_nav(out, r, ref, "%s batch %d rec %d" % (backend.name, n_rec, r), backend.name)
        solo = run_case(backend, m, max_epochs=max_ep)
        for k in ("rawP", "correctedP", "el", "az", "satPositions", "satClkCorr", "active", "sol"):
            assert solo[k][0].tobytes() == out[k][r].tobytes(), (r, k)
    n_eps = {m["n_ep"] for m in members}
    assert n_rec < 4 or (0 in n_eps and len(n_eps) >= 4)


def test_chain_at_16_3676_mhz(backend, monkeypatch):
    """post_navigate_batch (preamble search, ephemeris decoding, measurement loop) against the oracle chain at
    16.3676 MHz, where samplesPerCode is the rounded 16 368."""
    from softgnss_python_b200 import _native, postnav
    from softgnss_python_b200.settings import Settings
    monkeypatch.setattr(_native, "_LIB", backend.lib)
    fs = 16.3676e6
    s = Settings(numberOfChannels=8, msToProcess=float(NAV_MS), samplingFreq=fs)
    assert s.samplesPerCode == 16368
    tr, prn, _ = build_chain_case(seed=2, n_code=s.samplesPerCode, fs=fs)
    out = postnav.post_navigate_batch(tr[None], prn[None], s)
    first, ref = oracle_chain(tr, prn, dict(elevation_mask=s.elevationMask, use_trop_corr=s.useTropCorr),
                              samples_per_code=s.samplesPerCode)
    assert out["subFrameStart"][0].tolist() == list(first)
    assert ref is not None and ref["n_epochs"] > 50
    assert_clear_mask(ref, np.ones(len(prn)), s.elevationMask)
    compare_nav(out, 0, ref, backend.name + " chain 16.3676 MHz", backend.name)
