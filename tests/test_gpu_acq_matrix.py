"""Acquisition against the float64 oracle at every transform shape, exclusion-window edge, Doppler-grid edge, block
choice, fine-search seam and batch size, on the default path and on every path the library's SGX_* settings select.

Every run is checked in full (_check): the detected set, codePhase, frqBin, finePeakIndex and carrFreq equal the
oracle's (oracle.gnss_oracle.acquire(..., clamp_window=True, return_debug=True)) exactly, and peakMetric stays within
the bound of its path (PRECISION), which is set from the precision the kernels reach.  Exact comparisons are only fair
when the float64 winner is clear of its runner-up by far more than float32 error, so every case asserts that on the
oracle's values first (_assert_clear_decisions): best Doppler bin against the next, winning block against the other
blocks at that bin, code phase against every other, fine bin against every other, peakMetric against the threshold;
and no nav-bit sign change inside the 10 ms of the fine search.  Each case also asserts that it contains what it
claims (the code phase at the window edge, the block that wins, the fine bin at the seam).

Which kernel each shape reaches (sgx_acq.cu, sgx_pfa.cu, sgx_fine.cu; fine sub-transform radices from fft::build_plan):
  38.192 MHz   N = 38 192 = 31*7*16*11   prime-factor search (pfa p2 = 7); fine 2^22: fine::run (2048 x 2048)
  16.3676 MHz  N = 16 368 = 31*3*16*11   prime-factor search (pfa p2 = 3); fine 2^21: Stockham 64*64*64 (16x4 kernels)
  4.092 MHz    N = 4 092                 Stockham search; fine 2^19: Stockham 256*256 (16x16 kernels)
  8.184 MHz    N = 8 184                 Stockham search; fine 2^20: Stockham 64*64*32 (16x4 kernels + generic)
  32.736 MHz   N = 32 736                Stockham search; fine 2^22: fine::run
  64 MHz       N = 64 000                Stockham search; fine 2^23: Stockham 128*128*64 (16x8 and 16x4 kernels)
  acqCoherentMs = 2 at 38.192 MHz: N = 76 384, Stockham search (the prime-factor shapes are 1 ms only)

Every test runs on two backends:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).
The forced-path tests run tests/acq_matrix_worker.py in a subprocess per setting, because the library caches several
of them per process.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
WORKER = os.path.join(ROOT, "tests", "acq_matrix_worker.py")

# Largest |peakMetric / oracle - 1| a run may show, per path.  Observed maxima over every run of this file, on a
# B200 at 1000 W | under the CPU emulator:
#   pfa (38 192 and 16 368 points, default path)     6.2e-7 | 4.2e-7
#   stockham (every other shape, default path)       4.6e-7 | 4.1e-7
#   SGX_ACQ_PFA=0                                    5.3e-7 | 3.9e-7
#   SGX_ACQ_PFA_FWD=0                                4.0e-7 | 5.4e-7
#   SGX_ACQ_ASYNC=0, SGX_FFT_GENERIC=1               5.4e-7 | 4.2e-7
#   SGX_ACQ_FINE2=0                                  4.0e-7 | 4.2e-7
#   SGX_ACQ_CHUNK_MB=1, SGX_ACQ_FINE_CHUNK_MB=1      5.4e-7 | 4.2e-7
#   SGX_PFA_CFG = 62, 121, 43                        4.4e-7 | 4.0e-7
#   SGX_PFA_CFG = 643, 143, 543                      4.0e-7 | 4.2e-7
# Each bound is within 10x of its maximum (the kernels are float32 throughout, so every path lands in the same
# range).  The tolerance the older tests use, 1e-5, would pass a kernel 20x less precise.
PRECISION = {"pfa": 3e-6, "stockham": 3e-6}
FORCED_PRECISION = 3e-6
# Smallest relative lead of a float64 decision over its runner-up for an exact comparison to be fair: about 100x the
# largest peakMetric deviation above.  (The closest decision of the bench workload, a code phase, leads by 7.8e-5.)
MARGIN = 5e-5


class Backend(object):
    """One library (device build or CPU emulator)."""

    def __init__(self, name, lib, path):
        self.name = name
        self.lib = lib
        self.path = path

    def acquire(self, data, s, **kw):
        from softgnss_python_b200 import _native
        from softgnss_python_b200.acquisition import acquire_batch
        saved = _native._LIB
        _native._LIB = self.lib
        try:
            return acquire_batch(data, s, diagnostics=True, **kw)
        finally:
            _native._LIB = saved


@pytest.fixture(scope="module", params=[pytest.param("gpu", marks=pytest.mark.gpu),
                                        pytest.param("emul", marks=pytest.mark.emul)])
def backend(request):
    from softgnss_python_b200 import _native
    if request.param == "gpu":
        L = _native.lib()
        L.require_device()
        return Backend("gpu", L, None)
    if os.environ.get("SGX_EMUL_TESTS") != "1" or not os.path.exists(EMUL_LIB):
        pytest.skip("CPU emulator tests: set SGX_EMUL_TESTS=1 and build %s with tools/cpu_emul/build_emul.sh" % EMUL_LIB)
    return Backend("emul", _native.Lib(EMUL_LIB), EMUL_LIB)


KNOBS = ("SGX_ACQ_PFA", "SGX_ACQ_PFA_FWD", "SGX_ACQ_ASYNC", "SGX_FFT_GENERIC", "SGX_ACQ_FINE2", "SGX_ACQ_CHUNK_MB",
         "SGX_ACQ_FINE_CHUNK_MB", "SGX_PFA_CFG")


@pytest.fixture(autouse=True)
def default_path(monkeypatch):
    """Every in-process run below takes the default path."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)


# ---------------------------------------------------------------------------------------------------- cases
def _n(fs):
    return int(np.round(fs / 1e3))


def _nfft(n):
    """Length of the fine transform for N samples per code (acquisition.py:179)."""
    return 8 * 2 ** int(np.ceil(np.log2(10 * n)))


def _chip(fs):
    return int(round(fs / 1.023e6))


def _fine_bin_doppler(fs, f_if, doppler):
    """The Doppler nearest to `doppler` that puts the carrier on a bin centre of the fine search."""
    w = fs / _nfft(_n(fs))
    return round((f_if + doppler) / w) * w - f_if


# sample at which the synthesiser starts a code period, relative to the code phase the acquisition reports there
# (the chip index rule of make_ca_table puts the correlation peak 0 or 1 sample after it)
START_LAG = {38192: 1, 16368: 1, 4092: 0, 8184: 0, 32736: 0, 64000: 1}


class Case(object):
    """Recordings [R, n_samples] of one sampling rate and settings; oracle results cached per case."""

    def __init__(self, name, fs, f_if, recs, nprn, clean_fine=True, **ext):
        """recs: list of (SatSpec list, noise seed).  clean_fine=False: some satellite has a nav-bit sign change in the
        10 ms of its fine search on purpose (its fine bin is still held to MARGIN)."""
        self.name, self.fs, self.f_if, self.recs, self.nprn, self.clean_fine = name, fs, f_if, recs, nprn, clean_fine
        self.ext = ext
        self._data = self._specs = None
        self._ref = {}

    @property
    def n(self):
        return _n(self.fs)

    def settings(self):
        from softgnss_python_b200.settings import Settings
        s = Settings(samplingFreq=self.fs, IF=self.f_if, **self.ext)
        s.acqSatelliteList = range(1, self.nprn + 1)
        return s

    def settings_dict(self):
        return dict(samplingFreq=self.fs, IF=self.f_if, **self.ext)

    def data(self):
        if self._data is None:
            from softgnss_python_b200 import synth
            s = self.settings()
            ns = max(11, s.acqCoherentMs * s.acqNonCoherentBlocks) * self.n
            self._specs = [synth.RecordingSpec(sats, fs=self.fs, f_if=self.f_if, seed=seed) for sats, seed in self.recs]
            self._data = np.stack([synth.generate_cpu(sp, ns) for sp in self._specs])
        return self._data

    def specs(self):
        self.data()
        return self._specs

    def oracle(self, r):
        """Oracle result of recording r; its decisions are asserted clear on first use."""
        if r not in self._ref:
            from oracle import gnss_oracle as orc
            s = self.settings()
            ref = orc.acquire(self.data()[r], s, coherent_ms=s.acqCoherentMs, noncoh_blocks=s.acqNonCoherentBlocks,
                              doppler_step=s.acqDopplerStep, return_debug=True, clamp_window=True)
            _assert_clear_decisions(self, r, ref)
            self._ref[r] = ref
        return self._ref[r]


def _lead(best, others):
    """Relative lead of `best` over the largest of `others`."""
    others = np.asarray(others, dtype=np.float64)
    return 1.0 if others.size == 0 else (best - others.max()) / best


def _period_amplitude(spec, i, periods):
    """Signed amplitude (amplitude x nav bit) of satellite i in the given code periods."""
    return np.array([int(spec.amp[i]) * int(spec.nav_bit_at_period(i, p)) for p in periods])


def _code_period(spec, i, sample):
    return ((int(spec.cp0[i]) + sample * int(spec.dcp[i])) >> 32) // 1023


def _assert_clear_decisions(case, r, ref):
    """Every exact comparison with this oracle result is fair: each float64 decision leads its runner-up by MARGIN."""
    s = case.settings()
    n1 = case.n
    spec = case.specs()[r]
    label = "%s rec %d" % (case.name, r)
    for p in range(case.nprn):
        d = ref["debug"][p]
        prn = "%s PRN %d" % (label, p + 1)
        assert abs(ref["peakMetric"][p] / s.acqThreshold - 1) > MARGIN, prn + ": peakMetric at the threshold"
        if ref["carrFreq"][p] == 0:
            continue
        b = d["bin"]
        assert _lead(d["binMax"][b], np.delete(d["binMax"], b)) > MARGIN, prn + ": Doppler bin not clear"
        blk = d["blockMax"][b]
        assert _lead(blk.max(), np.sort(blk)[:-1]) > MARGIN, prn + ": block choice not clear"
        cp = d["codePhase"]
        assert _lead(d["colMax"][cp], np.delete(d["colMax"], cp)) > MARGIN, prn + ": code phase not clear"
        assert (d["finePeak"] - d["fineRunnerUp"]) / d["finePeak"] > MARGIN, prn + ": fine bin not clear"
        if case.clean_fine:
            # satellites of this PRN whose code is aligned with the detection: their summed signed amplitude keeps one
            # sign over the code periods of the fine search (samples cp .. cp + 10 N - 1)
            own = [i for i, x in enumerate(spec.sats) if x.prn == p + 1 and
                   min((cp - x.code_phase) % n1, (x.code_phase - cp) % n1) <= _chip(case.fs)]
            assert own, prn + ": detection of a satellite that is not in the recording"
            lo = min(_code_period(spec, i, cp) for i in own)
            hi = max(_code_period(spec, i, cp + 10 * n1 - 1) for i in own)
            amp = sum(_period_amplitude(spec, i, range(lo, hi + 1)) for i in own)
            assert (amp > 0).all() or (amp < 0).all(), prn + ": nav-bit sign change inside the fine search"


def _sat(prn, doppler, cp, case_fs, f_if, cn0=50.0, **kw):
    """A satellite whose correlation peak is at code phase `cp` and whose carrier is on a fine-search bin centre."""
    from softgnss_python_b200 import synth
    n = _n(case_fs)
    kw.setdefault("bit_offset_ms", 5)
    return synth.SatSpec(prn, _fine_bin_doppler(case_fs, f_if, doppler), (cp - START_LAG[n]) % n, cn0=cn0, **kw)


DOPPLERS = (-6000.0, -3500.0, -1000.0, 1500.0, 4000.0, 6500.0, -5000.0, 2500.0, -2000.0, 5500.0, 500.0, -4500.0)


def _plain_case(name, fs, f_if, seed, nsat=8, nprn=10, **ext):
    """nsat satellites among PRN 1..nprn (the rest absent), code phases spread over the code, Dopplers on the grid."""
    n = _n(fs)
    rng = np.random.default_rng(seed)
    prns = np.sort(rng.choice(np.arange(1, nprn + 1), nsat, replace=False))
    cps = [int(x) for x in rng.integers(2 * _chip(fs), n - 2 * _chip(fs), nsat)]
    sats = [_sat(int(p), DOPPLERS[i], cps[i], fs, f_if, bit_offset_ms=int(rng.integers(1, 11)))
            for i, p in enumerate(prns)]
    return Case(name, fs, f_if, [(sats, seed)], nprn, **ext)


# -- shapes: one rate per transform family
SHAPES = {
    "38.192MHz-pfa7-fine2": (38.192e6, 9.548e6, {}),
    "16.3676MHz-pfa3": (16.3676e6, 4.1304e6, {}),
    "4.092MHz": (4.092e6, 1.023e6, {}),
    "8.184MHz": (8.184e6, 2.046e6, {}),
    "32.736MHz": (32.736e6, 8.184e6, {}),
    "64MHz": (64e6, 16e6, {}),
    "38.192MHz-coherent2ms": (38.192e6, 9.548e6, dict(acqCoherentMs=2)),
}
EDGE_RATES = {"chip37": (38.192e6, 9.548e6), "chip16": (16.3676e6, 4.1304e6), "chip4": (4.092e6, 1.023e6)}
EDGE_CN0 = 63.0
ECHO_OFFSETS = ("+chip", "-chip", "+(chip-1)", "-(chip-1)")


def _edge_mains(n, w):
    """Main code phases: mid-code; lo = 1 - w and lo = -1 (window wraps past 0); lo = 1 (last index of the low part);
    hi = n - 1 (a = -1, numpy's last element); hi = n - 2 + w (window wraps past n - 1)."""
    return [n // 2 + 3, 1, w - 1, w + 1, n - 1 - w, n - 2]


def _edge_case(key):
    """Four recordings, one per echo offset: six PRNs, each a main signal at a window-edge code phase and an echo at
    -6 dB with the same Doppler, offset by +-chip (a second-peak candidate: peakMetric ~ main / echo) or by
    +-(chip - 1) (inside the exclusion window).  PRN 7 and 8 are absent."""
    fs, f_if = EDGE_RATES[key]
    n, w = _n(fs), _chip(fs)
    recs = []
    for j, off in enumerate(ECHO_OFFSETS):
        d = {"+chip": w, "-chip": -w, "+(chip-1)": w - 1, "-(chip-1)": 1 - w}[off]
        sats = []
        for i, cp in enumerate(_edge_mains(n, w)):
            sats.append(_sat(i + 1, DOPPLERS[i], cp, fs, f_if, cn0=EDGE_CN0))
            sats.append(_sat(i + 1, DOPPLERS[i], (cp + d) % n, fs, f_if, cn0=EDGE_CN0 - 6.0))
        recs.append((sats, 140 + j))
    return Case("edge-" + key, fs, f_if, recs, 8)


PFA_SHAPES = {"pfa7": (38.192e6, 9.548e6, (31, 7, 16, 11)), "pfa3": (16.3676e6, 4.1304e6, (31, 3, 16, 11))}


def _crt(res, mods):
    n = int(np.prod(mods))
    x = 0
    for r, m in zip(res, mods):
        q = n // m
        x += r * q * pow(q, -1, m)
    return x % n


def _residue_cps(key):
    """The 16 code phases whose residues modulo the four factors are all 0 or P - 1."""
    mods = PFA_SHAPES[key][2]
    return [_crt([(m - 1) * ((bits >> b) & 1) for b, m in enumerate(mods)], mods) for bits in range(16)]


def _residue_case(key):
    """Two recordings of eight satellites (PRN 1..8; 9 and 10 absent) at the 16 residue code phases."""
    fs, f_if, _ = PFA_SHAPES[key]
    cps = _residue_cps(key)
    recs = [([_sat(i + 1, DOPPLERS[i], cps[8 * j + i], fs, f_if, cn0=EDGE_CN0) for i in range(8)], 60 + j)
            for j in range(2)]
    return Case("residue-" + key, fs, f_if, recs, 10)


FINE_SEAM_OFFSETS = (-513, -512, -511, 511, 512, 513)   # k mod 2048 = 2047, 0, 1, 1023, 1024, 1025


def _fine_seam_case(key):
    """38.192 MHz: the IF moved to fine bin 2^20 + 512, so that carriers 511 .. 513 bins either side sit at
    k mod 2048 in {2047, 0, 1} (mirrored row 1, direct rows 0 and 1) and {1023, 1024, 1025} (direct rows 1023 and 1024,
    mirrored row 1023).  16.3676 MHz (generic fine transform, 8 sub-transforms of 2^18): carriers around the IF bin
    and the sub-transform boundaries, k mod 8 = 0 .. 7."""
    if key == "fine2":
        fs = 38.192e6
        w = fs / _nfft(_n(fs))
        f_if = (2 ** 20 + 512) * w
        offs = FINE_SEAM_OFFSETS
    else:
        fs, f_if = 16.3676e6, 4.1304e6
        w = fs / _nfft(_n(fs))
        offs = (-1, 0, 1, 2, 3, -4, -3, 7, 600, -601)
    n = _n(fs)
    base = round(f_if / w)
    cps = [1111 + 2711 * i for i in range(len(offs))]
    sats = []
    for i, k in enumerate(offs):
        sats.append(_sat(i + 1, 0.0, cps[i] % n, fs, f_if))
        sats[-1].doppler = (base + k) * w - f_if
    return Case("fineseam-" + key, fs, f_if, [(sats, 70)], len(offs) + 1)


def _grid_case(key):
    """Satellites in the first and the last Doppler bin; 129 bins (the last one is a second iteration of thread 0 of
    select_kernel's 128); a single bin."""
    if key == "edges":
        fs, f_if = 38.192e6, 9.548e6
        sats = [_sat(1, -7000.0, 9000, fs, f_if), _sat(2, 7000.0, 21000, fs, f_if), _sat(3, 500.0, 30000, fs, f_if)]
        return Case("grid-edges", fs, f_if, [(sats, 80)], 4)
    if key == "129bins":
        fs, f_if = 4.092e6, 1.023e6
        sats = [_sat(1, 7000.0, 1000, fs, f_if), _sat(2, -7000.0, 2000, fs, f_if), _sat(3, 0.0, 3000, fs, f_if)]
        return Case("grid-129bins", fs, f_if, [(sats, 81)], 4, acqDopplerStep=14000.0 / 128)
    fs, f_if = 38.192e6, 9.548e6
    sats = [_sat(1, 0.0, 12000, fs, f_if), _sat(2, 3000.0, 25000, fs, f_if)]
    return Case("grid-1bin", fs, f_if, [(sats, 82)], 3, acqSearchBand=0.0)


def _block_case(key):
    """Which block wins (acquisition.py:129-133).  PRN 1: a nav-bit sign change at the start of code period 1, in the
    middle of block 0 (code phase N/2): block 1 wins.  PRN 2: three copies of the signal, one of them changing sign at
    the start of period 2 (middle of block 1): periods 0 and 1 carry amplitude 3, later ones 1, block 0 wins.  With
    three blocks, PRN 1 is three copies whose signed sum is 1 in period 0, 3 in periods 1 and 2 and 1 from period 3
    on: blocks 0 and 2 are half as strong as block 1, the middle one wins."""
    fs, f_if = 38.192e6, 9.548e6
    n = _n(fs)
    alt = [1, -1] + [-1] * 8
    pos = [1, -1] + [-1] * 8
    if key == "2blocks":
        sats = [_sat(1, 2000.0, n // 2, fs, f_if, bit_offset_ms=0, nav_bits=alt),
                _sat(2, -3000.0, n // 2 + 777, fs, f_if, cn0=45.0, bit_offset_ms=5, nav_bits=[1] * 10),
                _sat(2, -3000.0, n // 2 + 777, fs, f_if, cn0=45.0, bit_offset_ms=19, nav_bits=pos),
                _sat(2, -3000.0, n // 2 + 777, fs, f_if, cn0=45.0, bit_offset_ms=5, nav_bits=[1] * 10),
                _sat(3, 4500.0, 5000, fs, f_if)]
        return Case("blocks-2", fs, f_if, [(sats, 90)], 4)
    # A constant; B: -1 in period 0, +1 later (change at period 1: bit_offset 0); C: +1 up to period 2, -1 from
    # period 3 (bit_offset 18)
    sats = [_sat(1, 1000.0, n // 2, fs, f_if, cn0=45.0, bit_offset_ms=5, nav_bits=[1] * 10),
            _sat(1, 1000.0, n // 2, fs, f_if, cn0=45.0, bit_offset_ms=0, nav_bits=[-1] + [1] * 9),
            _sat(1, 1000.0, n // 2, fs, f_if, cn0=45.0, bit_offset_ms=18, nav_bits=[1] + [-1] * 9),
            _sat(2, -2500.0, 3000, fs, f_if)]
    return Case("blocks-3", fs, f_if, [(sats, 91)], 3, acqNonCoherentBlocks=3)


def _batch_case(key):
    """12 satellites (PRN 1..12) per recording: 12 recordings at 38.192 MHz (144 detections, fine::run takes 127 per
    chunk) or 5 at 16.3676 MHz (60 detections, the generic fine path takes 51 per chunk)."""
    fs, f_if, nrec = (38.192e6, 9.548e6, 12) if key == "12x38MHz" else (16.3676e6, 4.1304e6, 5)
    n = _n(fs)
    rng = np.random.default_rng(100)
    recs = []
    for r in range(nrec):
        dop = rng.permutation(DOPPLERS)
        cps = rng.integers(2 * _chip(fs), n - 2 * _chip(fs), 12)
        sats = [_sat(p + 1, dop[p], int(cps[p]), fs, f_if, cn0=float(rng.uniform(48, 53)),
                     bit_offset_ms=int(rng.integers(1, 10))) for p in range(12)]
        recs.append((sats, 200 + r))
    return Case("batch-" + key, fs, f_if, recs, 12)


_CASES = {}


def case(key):
    if key not in _CASES:
        kind, sub = key.split(":", 1)
        if kind == "shape":
            fs, f_if, ext = SHAPES[sub]
            _CASES[key] = _plain_case("shape-" + sub, fs, f_if, 10 + list(SHAPES).index(sub), **ext)
        else:
            _CASES[key] = dict(edge=_edge_case, residue=_residue_case, fine=_fine_seam_case, grid=_grid_case,
                               block=_block_case, batch=_batch_case)[kind](sub)
    return _CASES[key]


# ---------------------------------------------------------------------------------------------------- checks
OBSERVED = {}     # path -> largest peakMetric deviation seen in this process (for refreshing PRECISION)


def _path(c):
    n = c.n * c.settings().acqCoherentMs
    return "pfa" if n in (38192, 16368) else "stockham"


def _check(got, c, path, bound, rows=None, label=""):
    """Results of acquire_batch(diagnostics=True) for the recordings `rows` of case c against the oracle."""
    s = c.settings()
    nfft = _nfft(c.n)
    rows = range(c.data().shape[0]) if rows is None else rows
    worst = 0.0
    for j, r in enumerate(rows):
        ref = c.oracle(r)
        lab = "%s %s rec %d" % (label or path, c.name, r)
        det = ref["carrFreq"][:c.nprn] > 0
        dbg = ref["debug"]
        assert np.array_equal(got["carrFreq"][j] > 0, det), lab + ": detected set"
        assert np.array_equal(got["codePhase"][j], ref["codePhase"][:c.nprn]), lab + ": codePhase"
        assert np.array_equal(got["frqBin"][j][det], [dbg[p]["bin"] for p in np.nonzero(det)[0]]), lab + ": frqBin"
        fine = np.array([dbg[p]["fineIndex"] if det[p] else -1 for p in range(c.nprn)])
        assert np.array_equal(got["finePeakIndex"][j], fine), lab + ": finePeakIndex"
        assert np.array_equal(got["carrFreq"][j], ref["carrFreq"][:c.nprn]), lab + ": carrFreq"
        assert np.array_equal(got["carrFreq"][j][det], fine[det] * s.samplingFreq / nfft)
        worst = max(worst, float(np.abs(got["peakMetric"][j] / ref["peakMetric"][:c.nprn] - 1).max()))
    OBSERVED[path] = max(OBSERVED.get(path, 0.0), worst)
    assert worst <= bound, "%s %s: peakMetric deviation %.3g (bound %.3g)" % (label or path, c.name, worst, bound)


def _run(backend, key):
    c = case(key)
    got = backend.acquire(c.data(), c.settings())
    path = _path(c)
    _check(got, c, path, PRECISION[path], label=backend.name)
    return c, got


# ---------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("shape", list(SHAPES))
def test_shapes(backend, shape):
    _run(backend, "shape:" + shape)


@pytest.mark.parametrize("key", list(EDGE_RATES))
def test_exclusion_window_edges(backend, key):
    """Every main code phase of _edge_mains, every echo offset.  Noise moves a correlation peak by a sample now and
    then, so the fixture's claims are checked on the code phases the oracle found: in most cases the second peak sits
    on the window boundary on the echo's side (the echo itself, or the first candidate next to an excluded echo), and
    the windows take every branch of second_peak_candidate."""
    c, _ = _run(backend, "edge:" + key)
    n, w = c.n, _chip(c.fs)
    on_boundary, branches = 0, set()
    for j, off in enumerate(ECHO_OFFSETS):
        ref = c.oracle(j)
        side = w if off[0] == "+" else -w
        for i in range(len(_edge_mains(n, w))):
            dbg = ref["debug"][i]
            cp = dbg["codePhase"]
            branches.add("lo<=0" if cp - w <= 0 else "hi=n-1" if cp + w == n - 1 else "hi>n-1" if cp + w > n - 1
                         else "mid")
            on_boundary += (dbg["secondIndex"] - cp) % n == side % n
    assert on_boundary >= 14, "%s: the second peak on the window boundary in only %d of 24 cases" % (c.name, on_boundary)
    assert branches == {"lo<=0", "hi=n-1", "hi>n-1", "mid"}, branches


@pytest.mark.parametrize("key", list(PFA_SHAPES))
def test_pfa_output_residues(backend, key):
    c, _ = _run(backend, "residue:" + key)
    got = [c.oracle(r)["debug"][i]["codePhase"] for r in range(2) for i in range(8)]
    hit = sum(a == b for a, b in zip(got, _residue_cps(key)))
    assert hit >= 12, "%s: %d of the 16 residue code phases realised" % (key, hit)
    for m in PFA_SHAPES[key][2]:
        assert {0, m - 1} <= {x % m for x in got}


@pytest.mark.parametrize("key", ["fine2", "generic"])
def test_fine_search_seams(backend, key):
    c, _ = _run(backend, "fine:" + key)
    if key == "fine2":
        ref = c.oracle(0)
        k = [ref["debug"][i]["fineIndex"] + 4 for i in range(len(FINE_SEAM_OFFSETS))]
        assert [x % 2048 for x in k] == [2047, 0, 1, 1023, 1024, 1025], k


@pytest.mark.parametrize("key", ["edges", "129bins", "1bin"])
def test_doppler_grid(backend, key):
    c, got = _run(backend, "grid:" + key)
    ref = c.oracle(0)
    want = {"edges": {0: 0, 1: 28}, "129bins": {0: 128, 1: 0}, "1bin": {0: 0}}[key]
    for p, b in want.items():
        assert ref["carrFreq"][p] > 0 and ref["debug"][p]["bin"] == b, (key, p)


@pytest.mark.parametrize("key,winners", [("2blocks", {0: 1, 1: 0}), ("3blocks", {0: 1})])
def test_block_choice(backend, key, winners):
    c, _ = _run(backend, "block:" + key)
    ref = c.oracle(0)
    for p, blk in winners.items():
        d = ref["debug"][p]
        assert ref["carrFreq"][p] > 0 and d["blockMax"][d["bin"]].argmax() == blk, (key, p, d["blockMax"][d["bin"]])


@pytest.mark.parametrize("key", ["12x38MHz", "5x16MHz"])
def test_batch_chunks_and_invariance(backend, key):
    """One call for the whole batch crosses the chunk boundaries of the fine search.  Each recording acquired alone,
    and each PRN shard of the batch, equal their part of it bit for bit (multi-GPU sharding relies on it).  The first,
    a middle and the last recording (whose detections fall in the last fine chunk) against the oracle."""
    c = case("batch:" + key)
    data, s = c.data(), c.settings()
    whole = backend.acquire(data, s)
    assert int((whole["carrFreq"] > 0).sum()) > (127 if c.n == 38192 else 51)
    for r in range(data.shape[0]):
        one = backend.acquire(data[r:r + 1], s)
        for f in whole:
            assert np.array_equal(one[f][0], whole[f][r]), (key, r, f)
    for first, count in ((0, 5), (5, 7)):
        part = backend.acquire(data, s, prn_first=first, prn_count=count)
        for f in whole:
            assert np.array_equal(part[f], whole[f][:, first:first + count]), (key, first, f)
    rows = [0, data.shape[0] // 2, data.shape[0] - 1]
    path = _path(c)
    _check({f: v[rows] for f, v in whole.items()}, c, path, PRECISION[path], rows=rows, label=backend.name)


def test_bench_workload_against_oracle(backend):
    """The acquisition batch of bench.py (32 recordings of bench.make_specs, 32 PRNs), every recording against the
    oracle.  Random Doppler and data bits: the fine search of some satellites spans a nav-bit change, so only the
    margins of the decisions are asserted for it."""
    if backend.name != "gpu":
        pytest.skip("the oracle takes about two minutes for this batch")
    from softgnss_python_b200 import synth
    from softgnss_python_b200.settings import Settings
    specs = [synth.RecordingSpec(synth.default_constellation(1000 + r, 8), seed=1000 + r) for r in range(32)]
    c = Case("bench", 38.192e6, 9.548e6, [(sp.sats, sp.seed) for sp in specs], 32, clean_fine=False)
    assert c.settings().acqThreshold == Settings().acqThreshold
    got = backend.acquire(c.data(), c.settings())
    _check(got, c, "pfa", PRECISION["pfa"], label=backend.name)


# -- forced paths: each setting in a worker process of its own, on the edge, residue and fine-seam cases
FORCED_CASES = ["edge:chip37", "edge:chip16", "edge:chip4", "residue:pfa7", "residue:pfa3", "fine:fine2",
                "fine:generic"]
PFA7_CASES = ["edge:chip37", "residue:pfa7", "fine:fine2"]
FORCED = [("SGX_ACQ_PFA", "0", FORCED_CASES), ("SGX_ACQ_PFA_FWD", "0", FORCED_CASES),
          ("SGX_ACQ_ASYNC", "0", FORCED_CASES), ("SGX_FFT_GENERIC", "1", FORCED_CASES),
          ("SGX_ACQ_FINE2", "0", PFA7_CASES), ("SGX_ACQ_CHUNK_MB", "1", FORCED_CASES),
          ("SGX_ACQ_FINE_CHUNK_MB", "1", FORCED_CASES)] + \
         [("SGX_PFA_CFG", str(v), PFA7_CASES) for v in (62, 121, 43, 643, 143, 543)]


@pytest.mark.parametrize("knob,value,keys", FORCED, ids=["%s=%s" % (k, v) for k, v, _ in FORCED])
def test_forced_path(backend, knob, value, keys, tmp_path):
    cases = [case(k) for k in keys]
    inp, out = str(tmp_path / "in.npz"), str(tmp_path / "out.npz")
    meta = [dict(settings=c.settings_dict(), nprn=c.nprn) for c in cases]
    np.savez(inp, meta=json.dumps(meta), **{"data%d" % i: c.data() for i, c in enumerate(cases)})
    env = dict(os.environ)
    for k in KNOBS:
        env.pop(k, None)
    env[knob] = value
    cmd = [sys.executable, WORKER, inp, out] + ([backend.path] if backend.path else [])
    p = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    z = np.load(out)
    path = "%s=%s" % (knob, value)
    for i, c in enumerate(cases):
        got = {f: z["%s%d" % (f, i)] for f in ("carrFreq", "codePhase", "peakMetric", "frqBin", "finePeakIndex")}
        _check(got, c, path, FORCED_PRECISION, label="%s %s" % (backend.name, path))
