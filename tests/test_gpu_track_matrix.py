"""The exact tracking correlator against the float64 oracle at every compiled segment width, window alignment and
recording edge.

The default correlator (exact integer segment sums, sgx_track.cu) is compiled for NW = 1 .. 8 words per half-chip
segment, NW = (ceil(fs / (2 * 1.023e6) + 0.25) + 3) / 4 (track_core).  NW <= 5 quantises the carrier twiddles to Q38
(five signed base-256 digits), NW >= 6 to Q30 (four digits).  That precision is the variant's purpose: DESIGN.md
section 5 relies on it to keep absoluteSample identical over 37 000 ms.  So besides compare_tracking(strict=True),
whose 1e-5 of full scale would pass a kernel that had lost a whole twiddle digit, every exact run here is held to a
bound per digit count that is set from the precision the kernel reaches (PRECISION below).

Inputs are built as in test_gpu_tracking.test_fresh_seed_against_oracle: a synthetic recording at fs with the IF at
fs / 4, and channels taken from the synthesiser's truth (carrier 30 Hz off, code phase + 1), so any sampling rate
works without acquisition.  The Doppler of +-7 kHz makes the code drift by 0.02 (4.092 MHz) to 0.3 (64 MHz) samples
per period, so the window offsets, word selects and funnel shifts of the segment loads move during a run.

Every test runs on two backends:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).  It runs the whole file in
            seconds without a GPU, which is the way to check a kernel change, or a deliberately broken kernel, against
            this suite.
"""
import math
import os

import numpy as np
import pytest

from tests.gpu_util import compare_tracking

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
IQ = ("I_P", "I_E", "I_L", "Q_E", "Q_P", "Q_L")
STAGES = ("bulk", "cpasync")

# (fs, NW): one rate per compiled width.  30.69 and 49.104 MHz give exactly 15 and 24 samples per half chip, so in
# period 0 every threshold falls on a sample instant and settle_boundary runs at NW 4 and 7 as well.
RATES = [(4.092e6, 1), (8.184e6, 2), (16.3676e6, 3), (30.69e6, 4), (38.192e6, 5), (45.0e6, 6), (49.104e6, 7),
         (64.0e6, 8)]

# Largest deviation from the oracle an exact run may show, per number of twiddle digits: max |d| over the six I/Q
# fields relative to their full scale, and max |d| of carrFreq / codeFreq in Hz.  Observed maxima over every exact run
# of this file (rate matrix, alignment sweep, recording end; both staging paths) on a B200 at 1000 W, identical
# under the CPU emulator:
#   NW       1        2        3        4        5     |    6        7        8
#   I/Q   1.5e-12  1.3e-12  9.9e-13  9.1e-13  8.7e-12  | 1.8e-10  1.6e-10  1.4e-10
#   carr  1.2e-10  0        4.7e-10  9.3e-10  1.9e-9   | 7.5e-9   7.5e-9   7.5e-9    (1 - 4 ulp)
#   code  0        0        0        0        1.2e-10  | 5.8e-10  3.5e-10  3.5e-10   (1 - 5 ulp)
# Each bound is within 10x of its maximum.  Zeroing the lowest twiddle digit (8 bits of every twiddle) fails every
# exact test here, with I/Q deviations from 1.2e-10 (Q38, 38.192 MHz) and from 2.2e-8 (Q30, 45 MHz) of full scale.
PRECISION = {5: dict(IQ_REL=5e-11, CARR_HZ=1e-8, CODE_HZ=1e-9),
             4: dict(IQ_REL=1e-9, CARR_HZ=5e-8, CODE_HZ=5e-9)}


def _nw(fs):
    """Words per segment of the exact correlator at fs (track_core)."""
    return (math.ceil(fs / (2 * 1.023e6) + 0.25) + 3) // 4


def _digits(nw):
    return 5 if nw <= 5 else 4


class Backend(object):
    """One library (device build or CPU emulator) and how a recording is put where the kernel reads it."""

    def __init__(self, name, lib):
        self.name = name
        self.lib = lib

    def track(self, rec, rec_len, channels, settings, resident=True):
        """rec: int8 [R, stride] on the host.  resident=True: the recordings are in device memory (the kernel reads
        them in place, bytes beyond rec_len included); False: they are streamed from host memory in chunks.
        Returns (rc, out float64 [R, C, 13, ms], ms_done [R, C])."""
        from softgnss_python_b200 import _native
        from softgnss_python_b200.settings import to_pod
        pod = to_pod(settings)
        r, stride = rec.shape
        out = np.zeros((r, int(settings.numberOfChannels), len(_native.TRACK_FIELDS), pod.msToProcess))
        chans = _native.make_channels(*[np.tile(x, r) for x in channels])
        host_env = os.environ.pop("SGX_EMUL_HOST", None)
        try:
            if self.name == "gpu":
                import torch
                buf = torch.from_numpy(rec).cuda() if resident else np.ascontiguousarray(rec)
            else:
                # the emulator takes every pointer for a device pointer unless SGX_EMUL_HOST is set; device
                # recordings must be 16-byte aligned
                raw = np.zeros(rec.size + 16, dtype=np.int8)
                o = (-raw.ctypes.data) % 16
                buf = raw[o:o + rec.size].reshape(rec.shape)
                buf[...] = rec
                if not resident:
                    os.environ["SGX_EMUL_HOST"] = "1"
            rc, done = self.lib.track(buf, stride, list(rec_len), chans, pod, _native.ca_chips_int8(), out)
        finally:
            os.environ.pop("SGX_EMUL_HOST", None)
            if host_env is not None:
                os.environ["SGX_EMUL_HOST"] = host_env
        return rc, out, done

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
def default_kernel(monkeypatch):
    """Every run below is the default correlator selection unless a test says otherwise."""
    for k in ("SGX_TRK_KERNEL", "SGX_TRK_STAGE", "SGX_TRK_CHUNK_MS", "SGX_EMUL_HOST"):
        monkeypatch.delenv(k, raising=False)


_CASES = {}


def _case(fs, ms, skip=0, spacing=0.5):
    """(data, settings, channels (prn, freq, codePhase), oracle fields [C, ms]) of a two-satellite recording at fs;
    cached, the oracle is the slow part."""
    key = (fs, ms, skip, spacing)
    if key not in _CASES:
        from oracle import gnss_oracle as orc
        from softgnss_python_b200 import _native, synth
        from softgnss_python_b200.settings import Settings
        s = Settings(samplingFreq=fs, IF=fs / 4, numberOfChannels=2, msToProcess=float(ms), skipNumberOfBytes=skip,
                     dllCorrelatorSpacing=spacing)
        n = s.samplesPerCode
        sats = [synth.SatSpec(2, 6900.0, n // 3, cn0=52.0, bit_offset_ms=3),
                synth.SatSpec(5, -7000.0, n - 7, cn0=52.0, bit_offset_ms=11)]
        spec = synth.RecordingSpec(sats, fs=fs, f_if=fs / 4, seed=11)
        data = synth.generate_cpu(spec, (ms + 3) * n + skip)
        prn = np.array([x.prn for x in sats], dtype=np.int64)
        freq = np.array([spec.true_carr_freq(i) - 30.0 for i in range(len(sats))])
        cph = np.array([(x.code_phase + 1) % n for x in sats], dtype=np.float64)
        recs = orc.track(data, dict(PRN=prn, acquiredFreq=freq, codePhase=cph, status=['T'] * len(sats)), s)
        ref = {f: np.stack([r[2][f] for r in recs]) for f in _native.TRACK_FIELDS}
        _CASES[key] = (data, s, (prn, freq, cph), ref)
    return _CASES[key]


def _fields(out):
    """out [C, 13, ms] -> dict field -> [C, ms]"""
    from softgnss_python_b200._native import TRACK_FIELDS
    return {f: out[:, i, :] for i, f in enumerate(TRACK_FIELDS)}


def _deviation(got, ref):
    """(max |d| of the six I/Q fields relative to their full scale, max |d| carrFreq, max |d| codeFreq)"""
    scale = max(np.abs(ref[f]).max() for f in IQ)
    iq = max(np.abs(got[f] - ref[f]).max() for f in IQ) / scale
    return (iq, np.abs(got["carrFreq"] - ref["carrFreq"]).max(), np.abs(got["codeFreq"] - ref["codeFreq"]).max())


def _check_exact(out, ref, fs, label):
    """An exact-correlator result [C, 13, ms] against the oracle: no chip reassignment, and the precision bound of its
    digit count."""
    got = _fields(out)
    compare_tracking(got, ref, label, strict=True)
    iq, carr, code = _deviation(got, ref)
    b = PRECISION[_digits(_nw(fs))]
    assert iq <= b["IQ_REL"], "%s: I/Q deviation %.3g of full scale (bound %.3g)" % (label, iq, b["IQ_REL"])
    assert carr <= b["CARR_HZ"], "%s: carrFreq deviation %.3g Hz (bound %.3g)" % (label, carr, b["CARR_HZ"])
    assert code <= b["CODE_HZ"], "%s: codeFreq deviation %.3g Hz (bound %.3g)" % (label, code, b["CODE_HZ"])


def _both_stages(backend, monkeypatch, rec, rec_len, channels, s):
    """Run with the bulk-copy and the cp.async staging; the two must agree bit for bit.  Returns (rc, out, done)."""
    res = {}
    for stage in STAGES:
        monkeypatch.setenv("SGX_TRK_STAGE", stage)
        res[stage] = backend.track(rec, rec_len, channels, s)
    (rc0, out0, done0), (rc1, out1, done1) = res["bulk"], res["cpasync"]
    assert rc0 == rc1 and np.array_equal(done0, done1)
    assert np.array_equal(out0, out1), "bulk and cp.async staging differ"
    return rc0, out0, done0


@pytest.mark.parametrize("fs,nw", RATES, ids=["%gMHz-NW%d" % (fs / 1e6, nw) for fs, nw in RATES])
def test_rate_matrix(backend, fs, nw, monkeypatch):
    """One sampling rate per compiled width, 20 ms of two channels, both staging paths."""
    assert _nw(fs) == nw
    ms = 20
    data, s, ch, ref = _case(fs, ms)
    rc, out, done = _both_stages(backend, monkeypatch, data[None], [data.size], ch, s)
    assert rc == 0 and (done == ms).all()
    _check_exact(out[0], ref, fs, "%s fs=%g NW=%d" % (backend.name, fs, nw))


@pytest.mark.parametrize("skip", range(16))
@pytest.mark.parametrize("fs", [38.192e6, 45.0e6])
def test_window_alignment(backend, fs, skip, monkeypatch):
    """skipNumberOfBytes = 0 .. 15 puts the first window of each channel at every offset from the 16-byte staging
    base, and so every word select and funnel shift of the segment loads (38192 is a multiple of 16, so at the
    default rate the offset otherwise moves only with code drift).  A Q38 and a Q30 width."""
    ms = 8
    data, s, ch, ref = _case(fs, ms, skip=skip)
    rc, out, done = _both_stages(backend, monkeypatch, data[None], [data.size], ch, s)
    assert rc == 0 and (done == ms).all()
    _check_exact(out[0], ref, fs, "%s fs=%g skip=%d" % (backend.name, fs, skip))


@pytest.mark.parametrize("fs", [38.192e6, 45.0e6])
def test_recording_end(backend, fs, monkeypatch):
    """A device recording that ends exactly at the last sample the channels read completes every period; one byte
    shorter, the channel that reads it stops with the short-recording error after ms - 1 periods.  rec_len is not a
    multiple of 16, so the staging copies of the last window take bytes beyond it (up to the 16-byte rounded length):
    whatever those bytes hold (0 or 0x7f here, also past the rounded length) must not change a result."""
    from softgnss_python_b200._native import SGX_ERR_SHORT
    ms = 12
    data, s, ch, ref = _case(fs, ms)
    last = ref["absoluteSample"][:, -1].astype(np.int64)
    end = int(last.max())
    assert end % 16 != 0 and last.min() < end - 1
    rc, full, done = _both_stages(backend, monkeypatch, data[None], [data.size], ch, s)
    assert rc == 0 and (done == ms).all()
    _check_exact(full[0], ref, fs, "%s fs=%g full recording" % (backend.name, fs))
    for rec_len in (end, end - 1):
        want = np.where(last <= rec_len, ms, ms - 1)
        runs = []
        for fill in (0, 0x7f):
            rec = np.full((1, (rec_len + 15) // 16 * 16 + 64), fill, dtype=np.int8)
            rec[0, :rec_len] = data[:rec_len]
            label = "%s fs=%g rec_len=%d fill=%#x" % (backend.name, fs, rec_len, fill)
            rc, out, done = _both_stages(backend, monkeypatch, rec, [rec_len], ch, s)
            assert rc == (0 if rec_len == end else SGX_ERR_SHORT), label
            if rc:
                assert "Not able to read the specified number of samples" in backend.last_error()
            assert np.array_equal(done[0], want), label + " ms_done %s" % done[0]
            for c in range(len(want)):          # the completed periods are those of the full recording
                assert np.array_equal(out[0, c, :, :want[c]], full[0, c, :, :want[c]]), label + " ch%d" % c
            runs.append(out)
        for c in range(len(want)):
            assert np.array_equal(runs[0][0, c, :, :want[c]], runs[1][0, c, :, :want[c]])


@pytest.mark.parametrize("chunk_ms", ["1", "7"])
def test_streamed_resume_45mhz(backend, chunk_ms, monkeypatch):
    """Host recordings streamed in chunks of 1 / 7 code periods at NW 6: 45000 samples per code is not a multiple of
    16, so the chunk edges (rounded to 16 bytes) drift against the periods and channels pause at every window offset.
    Two recordings, the second shifted by 5 samples and shorter.  The result must equal the device-resident run bit
    for bit."""
    ms = 20
    data, s, ch, _ = _case(45.0e6, ms)
    n = data.size
    rec_len = [n, n - 5]
    rec = np.zeros((2, (n + 15) // 16 * 16), dtype=np.int8)
    rec[0, :n] = data
    rec[1, :n - 5] = data[5:]
    rc0, out0, done0 = backend.track(rec, rec_len, ch, s, resident=True)
    monkeypatch.setenv("SGX_TRK_CHUNK_MS", chunk_ms)
    rc1, out1, done1 = backend.track(rec, rec_len, ch, s, resident=False)
    assert rc0 == 0 and rc1 == 0 and (done0 == ms).all() and np.array_equal(done0, done1)
    assert np.array_equal(out0, out1)


@pytest.mark.parametrize("fs", [4.092e6, 16.3676e6])
def test_group_kernel_low_rates(backend, fs, monkeypatch):
    """dllCorrelatorSpacing = 0.25 selects the aligned 16-sample-group correlator.  At 2 (4.092 MHz) and 8 (16.3676
    MHz) samples per half chip most groups hold several chip boundaries and take the per-sample walk.  Tolerances of
    test_gpu_configs.test_non_default_correlator_spacing_uses_group_kernel (float32 correlator)."""
    ms = 15
    data, s, ch, ref = _case(fs, ms, spacing=0.25)
    rc, out, done = _both_stages(backend, monkeypatch, data[None], [data.size], ch, s)
    assert rc == 0 and (done == ms).all()
    compare_tracking(_fields(out[0]), ref, "%s spacing 0.25 fs=%g" % (backend.name, fs))
