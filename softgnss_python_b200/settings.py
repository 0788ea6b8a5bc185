"""Receiver settings and the signal-definition helpers of the hot path.

Host-side mirror of the reference's ``Settings`` object: the same attribute
names and defaults (reference ``initialize.py:80-173``) so that code written
against the reference -- ``main.py``, ``Settings.postProcessing``,
``postNavigation`` -- can hand either object to :func:`acquisition` /
:func:`tracking`.  Only the four helpers the hot path calls are implemented
(SURVEY.md section 8(a) rows A1-A3, T1):

* ``samplesPerCode``      -- reference ``initialize.py:183-185``
* ``generateCAcode(prn)`` -- reference ``initialize.py:234-302`` (bit-level LFSRs here)
* ``makeCaTable()``       -- reference ``initialize.py:188-231`` (same float64 index rule)
* ``calcLoopCoef``        -- reference ``initialize.py:304-328``

Extension attributes (not in the reference; defaults reproduce it):
``acqDopplerStep`` (500 Hz, literal at ``acquisition.py:101``),
``acqCoherentMs`` (1) and ``acqNonCoherentBlocks`` (2, the pick-max of two 1 ms
blocks at ``acquisition.py:129-133``).
Tracking-quality extensions, read by ``tracking.cno_vsm`` / ``track_quality_batch`` (with these defaults when an
object lacks them): ``CNoVSMinterval`` (40 code periods per C/N0 estimate, Matlab ``settings.CNo.VSMinterval``),
``CNoAccTime`` (0.001 s per prompt sample, ``settings.CNo.accTime``), ``lockCNoMin`` (30.0 dB-Hz) and ``lockPllMin``
(0.5, cos 2 dphi): a window counts as locked when its C/N0 and its carrier-lock indicator reach both.
Velocity extensions, read by ``postnav.nav_velocity_batch`` / ``postNavigateVelocity`` (same defaults for an object
without them): ``dopplerAvgMs`` (100 code periods of carrFreq averaged per Doppler) and ``L1Freq`` (1575.42e6 Hz).
Integrity (RAIM) extensions, read by ``postnav.nav_integrity_batch`` / ``postNavigateIntegrity`` (same defaults for an
object without them): ``raimSigma`` (5.0 m, the standard deviation assumed for one pseudorange error -- a judgement, not
a measurement of tracked-range noise), ``raimPfa`` (1e-5, false-alarm probability of the residual test) and ``raimPmd``
(1e-3, missed-detection probability behind the protection levels).
"""
import ctypes

import numpy as np

# G2 output delay (chips) selecting the PRN, IS-GPS-200 table 3-I; the reference
# carries the same 32 values (plus SBAS ones it never uses) at initialize.py:251-255.
_G2_DELAY = (5, 6, 7, 8, 17, 18, 139, 140, 141, 251, 252, 254, 255, 256, 257, 258,
             469, 470, 471, 472, 473, 474, 509, 512, 513, 514, 515, 516, 859, 860, 861, 862)


def _lfsr_sequence(taps):
    """1023 output bits of a 10-stage Fibonacci LFSR, all-ones start, output = stage 10."""
    state = 0x3FF  # bit i-1 holds stage i
    out = np.empty(1023, dtype=np.uint8)
    for n in range(1023):
        out[n] = (state >> 9) & 1
        fb = 0
        for t in taps:
            fb ^= (state >> (t - 1)) & 1
        state = ((state << 1) | fb) & 0x3FF
    return out


_G1_BITS = _lfsr_sequence((3, 10))
_G2_BITS = _lfsr_sequence((2, 3, 6, 8, 9, 10))


def ca_code_bits(prn0):
    """C/A chips of PRN ``prn0+1`` as 0/1 bits (chip 1 <-> +1 in the reference's convention)."""
    if prn0 not in range(32):
        raise AssertionError("prn index must be 0..31")
    return _G1_BITS ^ np.roll(_G2_BITS, _G2_DELAY[prn0])


class TruePosition(object):
    """Placeholder with E/N/U attributes (reference ``initialize.py:49-77``); unused by the hot path."""

    def __init__(self):
        self.E = None
        self.N = None
        self.U = None


class Settings(object):
    """Same public fields as the reference ``Settings`` (``initialize.py:80-173``)."""

    _DEFAULTS = dict(
        msToProcess=37000.0, numberOfChannels=8, skipNumberOfBytes=0,
        fileName='', dataType='int8',
        IF=9548000.0, samplingFreq=38192000.0, codeFreqBasis=1023000.0, codeLength=1023,
        skipAcquisition=False, acqSearchBand=14.0, acqThreshold=2.5,
        dllDampingRatio=0.7, dllNoiseBandwidth=2.0, dllCorrelatorSpacing=0.5,
        pllDampingRatio=0.7, pllNoiseBandwidth=25.0,
        navSolPeriod=500.0, elevationMask=10.0, useTropCorr=True, plotTracking=True,
        # extensions (defaults == reference behaviour)
        acqDopplerStep=500.0, acqCoherentMs=1, acqNonCoherentBlocks=2,
        CNoVSMinterval=40, CNoAccTime=0.001, lockCNoMin=30.0, lockPllMin=0.5,
        dopplerAvgMs=100, L1Freq=1575.42e6, raimSigma=5.0, raimPfa=1e-5, raimPmd=1e-3,
    )

    def __init__(self, **overrides):
        for k, v in self._DEFAULTS.items():
            setattr(self, k, v)
        self.acqSatelliteList = range(1, 33)
        self.truePosition = TruePosition()
        self._c = 299792458.0
        self._startOffset = 68.802
        for k, v in overrides.items():
            setattr(self, k, v)

    @property
    def c(self):
        return self._c

    @property
    def startOffset(self):
        return self._startOffset

    @property
    def samplesPerCode(self):
        return samples_per_code(self)

    def generateCAcode(self, prn):
        return generate_ca_code(prn)

    def makeCaTable(self):
        return make_ca_table(self)

    @staticmethod
    def calcLoopCoef(LBW, zeta, k):
        return calc_loop_coef(LBW, zeta, k)


def samples_per_code(settings):
    """A1: ``round(fs / (codeFreqBasis / codeLength))`` (reference ``initialize.py:185``)."""
    return int(np.round(settings.samplingFreq / (settings.codeFreqBasis / settings.codeLength)))


def generate_ca_code(prn0):
    """A2: float64[1023] of +-1 for 0-based PRN index (reference ``initialize.py:234-302``)."""
    return ca_code_bits(prn0).astype(np.float64) * 2.0 - 1.0


def ca_table_index(settings):
    """The float64 sample->chip index rule of ``initialize.py:223-226`` (A3); int64[N].

    Kept in float64 on the host on purpose: at 24 of 38192 positions the rounded
    product differs from exact rational arithmetic (SURVEY.md appendix A.1-9) and
    the acquisition code phase depends on it.
    """
    n = samples_per_code(settings)
    ts = 1.0 / settings.samplingFreq
    tc = 1.0 / settings.codeFreqBasis
    idx = (np.ceil(ts * np.arange(1, n + 1) / tc) - 1).astype(np.int64)
    idx[-1] = settings.codeLength - 1
    return idx


def make_ca_table(settings):
    """A3: float64[32, samplesPerCode] of +-1 (reference ``initialize.py:188-231``)."""
    idx = ca_table_index(settings)
    return np.stack([generate_ca_code(p)[idx] for p in range(32)])


def fine_code_index(settings, n_ms=10):
    """A10 chip index for the code-stripped fine search: ``floor(ts*(1..n_ms*N)/tc) % 1023``
    in float64 exactly as ``acquisition.py:172-174``; uint16[n_ms*N]."""
    n = samples_per_code(settings)
    ts = 1.0 / settings.samplingFreq
    idx = np.floor(ts * np.arange(1, n_ms * n + 1) / (1.0 / settings.codeFreqBasis))
    return (idx % settings.codeLength).astype(np.uint16)


def calc_loop_coef(LBW, zeta, k):
    """T1: second-order loop time constants (reference ``initialize.py:306-328``)."""
    wn = LBW * 8.0 * zeta / (4.0 * zeta ** 2 + 1)
    return k / (wn * wn), 2.0 * zeta / wn


class SgxSettings(ctypes.Structure):
    """POD mirror of ``sgx_settings`` in ``include/softgnss_b200.h``."""
    _fields_ = [
        ("samplingFreq", ctypes.c_double), ("IF", ctypes.c_double),
        ("codeFreqBasis", ctypes.c_double),
        ("acqSearchBand", ctypes.c_double), ("acqThreshold", ctypes.c_double),
        ("acqDopplerStep", ctypes.c_double),
        ("dllCorrelatorSpacing", ctypes.c_double),
        ("tau1code", ctypes.c_double), ("tau2code", ctypes.c_double),
        ("tau1carr", ctypes.c_double), ("tau2carr", ctypes.c_double),
        ("PDIcode", ctypes.c_double), ("PDIcarr", ctypes.c_double),
        ("skipNumberOfBytes", ctypes.c_int64),
        ("codeLength", ctypes.c_int32), ("samplesPerCode", ctypes.c_int32),
        ("numAcqSatellites", ctypes.c_int32), ("numFrqBins", ctypes.c_int32),
        ("acqCoherentMs", ctypes.c_int32), ("acqNonCoherentBlocks", ctypes.c_int32),
        ("samplesPerCodeChip", ctypes.c_int32), ("fineMs", ctypes.c_int32),
        ("msToProcess", ctypes.c_int32), ("numberOfChannels", ctypes.c_int32),
    ]


def to_pod(settings):
    """Marshal a (reference or local) settings object into the C-ABI struct.

    Derived integers are computed here with the reference's own float64 expressions
    (``acquisition.py:68``, ``:145``; ``tracking.py:42-52``) so the device never
    re-derives a rounding-sensitive quantity.
    """
    g = lambda name, default: getattr(settings, name, default)
    tau1code, tau2code = calc_loop_coef(settings.dllNoiseBandwidth, settings.dllDampingRatio, 1.0)
    tau1carr, tau2carr = calc_loop_coef(settings.pllNoiseBandwidth, settings.pllDampingRatio, 0.25)
    step = float(g("acqDopplerStep", 500.0))
    nbins = int(np.round(settings.acqSearchBand * 1000.0 / step) + 1)
    return SgxSettings(
        samplingFreq=float(settings.samplingFreq), IF=float(settings.IF),
        codeFreqBasis=float(settings.codeFreqBasis),
        acqSearchBand=float(settings.acqSearchBand), acqThreshold=float(settings.acqThreshold),
        acqDopplerStep=step,
        dllCorrelatorSpacing=float(settings.dllCorrelatorSpacing),
        tau1code=tau1code, tau2code=tau2code, tau1carr=tau1carr, tau2carr=tau2carr,
        PDIcode=0.001, PDIcarr=0.001,
        skipNumberOfBytes=int(settings.skipNumberOfBytes),
        codeLength=int(settings.codeLength), samplesPerCode=samples_per_code(settings),
        numAcqSatellites=len(settings.acqSatelliteList), numFrqBins=nbins,
        acqCoherentMs=int(g("acqCoherentMs", 1)),
        acqNonCoherentBlocks=int(g("acqNonCoherentBlocks", 2)),
        samplesPerCodeChip=int(round(settings.samplingFreq / settings.codeFreqBasis)),
        fineMs=10,
        msToProcess=int(settings.msToProcess), numberOfChannels=int(settings.numberOfChannels),
    )
