"""The reference's downstream consumer (``postNavigation.py``) on the B200: preamble search and navigation-bit
extraction (SURVEY.md section 8(f) row 3), relative pseudoranges, satellite positions and the least-squares
fix (row 4), with the ephemeris bit-field decoding in between on the host.

Mirrors, with the reference's names and conventions:

* ``findPreambles(trackResults, settings)`` -> ``(firstSubFrame, activeChnList)``
  (``NavigationResult.findPreambles``, postNavigation.py:524-631);
* ``navBitsBin(trackResults, firstSubFrame, channelNr)`` -> list of ``'0'``/``'1'`` strings
  (postNavigation.py:125-139), ready for ``ephemeris.ephemeris(bits[1:], bits[0])``.

Extension (no reference behaviour): receiver velocity and clock drift from the PLL's Doppler at the same epochs
(``nav_velocity_batch``, ``post_navigate_batch(..., velocity=True)``, ``postNavigateVelocity``), computed by
``sgx_nav_velocity`` (csrc/sgx_nav.cu).  Receiver autonomous integrity monitoring of the fix: a residual test, exclusion of
one faulty channel and horizontal / vertical protection levels (``raim_tables``, ``nav_integrity_batch``,
``post_navigate_batch(..., integrity=True)``, ``postNavigateIntegrity``), computed by ``sgx_nav_integrity``.

``find_preambles_batch`` is the batched entry point over a float64 ``[channels, ms]`` array or CUDA tensor
(e.g. field 3 of ``track_batch``'s device-resident output).  There is no CPU implementation here: the
work is done by ``sgx_find_preambles`` (csrc/sgx_bitsync.cu) and the call fails without a CUDA device.
"""
import math

import numpy as np

from . import _native

NAV_BITS = 1501


def find_preambles_batch(i_p, ms=None, stride=None, want_bits=True, stream=0):
    """``i_p``: float64 ``[n, ms]`` numpy array or CUDA tensor (rows ``stride`` elements apart).
    Returns ``(first int32[n], bits uint8[n, 1501] | None, valid int32[n] | None)``."""
    if isinstance(i_p, np.ndarray):
        i_p = np.ascontiguousarray(i_p, dtype=np.float64)
        n = i_p.shape[0]
        ms = i_p.shape[1] if ms is None else int(ms)
        stride = i_p.shape[1] if stride is None else int(stride)
    else:                                   # torch tensor
        import torch
        assert i_p.dtype == torch.float64 and i_p.stride(-1) == 1
        n = i_p.shape[0]
        ms = i_p.shape[1] if ms is None else int(ms)
        stride = i_p.stride(0) if stride is None else int(stride)
    return _native.lib().find_preambles(i_p, stride, n, ms, want_bits=want_bits, stream=stream)


def _tracked_ip(trackResults):
    active = (trackResults.status != '-').nonzero()[0] if trackResults.status.dtype.kind != 'S' \
        else (trackResults.status != b'-').nonzero()[0]
    # (the reference indexes trackResults with range(len(activeChnList)), postNavigation.py:563)
    rows = [np.asarray(trackResults[c].I_P, dtype=np.float64) for c in range(len(active))]
    return active, (np.stack(rows) if rows else np.zeros((0, 1)))


def findPreambles(trackResults, settings, return_bits=False):
    """postNavigation.py:524-631.  ``firstSubFrame`` has ``settings.numberOfChannels`` entries (0 = none);
    ``activeChnList`` lists the channels with a verified preamble."""
    assert isinstance(trackResults, np.recarray)
    firstSubFrame = np.zeros(settings.numberOfChannels, dtype=int)
    activeChnList, i_p = _tracked_ip(trackResults)
    bits = valid = None
    if len(activeChnList):
        first, bits, valid = find_preambles_batch(i_p)
        firstSubFrame[:len(first)] = first
    for channelNr in range(len(activeChnList)):
        if firstSubFrame[channelNr] == 0:
            activeChnList = np.setdiff1d(activeChnList, channelNr)
            print('Could not find valid preambles in channel %2d !' % channelNr)
    if return_bits:
        return firstSubFrame, activeChnList, bits, valid
    return firstSubFrame, activeChnList


def navBitsBin(bits_row):
    """The ``navBitsBin`` list of postNavigation.py:134-137 from one row of the device's hard bits."""
    return [str(int(b)) for b in bits_row]


def calculatePseudoranges(trackResults, msOfTheSignal, channelList, settings):
    """postNavigation.py:27-72 for one measurement epoch (function-style form of the reference method)."""
    n_ch = settings.numberOfChannels
    # the reference calls this once per measurement epoch: hand the device only the one sample per channel it reads
    # (a [1, C, 13, 1] view of the tracking result, epoch index 0), not the whole 30 MB result
    trk = np.zeros((1, n_ch, len(_native.TRACK_FIELDS), 1))
    idx = np.zeros((1, 1, n_ch), dtype=np.int32)
    act = np.zeros((1, 1, n_ch), dtype=np.uint8)
    for c in channelList:
        trk[0, c, 0, 0] = trackResults[c].absoluteSample[int(msOfTheSignal[c])]
        act[0, 0, c] = 1
    return pseudoranges_batch(trk, idx, act, settings)[0, 0]


def pseudoranges_batch(track_out, ms_index, active, settings, stream=0):
    """``track_out``: float64 ``[R, C, 13, ms]`` numpy array or CUDA tensor (``track_batch``'s output);
    ``ms_index`` / ``active``: ``[R, E, C]``.  Returns metres, float64 ``[R, E, C]``."""
    r, c, _, ms = track_out.shape
    return _native.lib().pseudoranges(track_out, r, c, ms, ms_index, active, settings.samplesPerCode,
                                      settings.startOffset, settings.c, stream=stream)


# ---- ephemeris decoding (ephemeris.py:98-196): host-side integer bit slicing between the two device stages ----------
EPH_ALL = ("weekNumber", "accuracy", "health", "T_GD", "IODC", "t_oc", "a_f2", "a_f1", "a_f0", "IODE_sf2", "C_rs",
           "deltan", "M_0", "C_uc", "e", "C_us", "sqrtA", "t_oe", "C_ic", "omega_0", "C_is", "i_0", "C_rc", "omega",
           "omegaDot", "IODE_sf3", "iDot")
_GPS_PI = 3.1415926535898                      # ephemeris.py:113
#  field: (subframe ID, bit ranges inside the subframe, signed, power of two, times pi)   -- ephemeris.py:139-176
_EPH_LAYOUT = {
    "weekNumber": (1, ((60, 70),), False, 0, False), "accuracy": (1, ((72, 76),), False, 0, False),
    "health": (1, ((76, 82),), False, 0, False), "T_GD": (1, ((195, 204),), True, -31, False),
    "IODC": (1, ((82, 84), (196, 204)), False, 0, False), "t_oc": (1, ((218, 234),), False, 4, False),
    "a_f2": (1, ((240, 248),), True, -55, False), "a_f1": (1, ((248, 264),), True, -43, False),
    "a_f0": (1, ((270, 292),), True, -31, False),
    "IODE_sf2": (2, ((60, 68),), False, 0, False), "C_rs": (2, ((68, 84),), True, -5, False),
    "deltan": (2, ((90, 106),), True, -43, True), "M_0": (2, ((106, 114), (120, 144)), True, -31, True),
    "C_uc": (2, ((150, 166),), True, -29, False), "e": (2, ((166, 174), (180, 204)), False, -33, False),
    "C_us": (2, ((210, 226),), True, -29, False), "sqrtA": (2, ((226, 234), (240, 264)), False, -19, False),
    "t_oe": (2, ((270, 286),), False, 4, False),
    "C_ic": (3, ((60, 76),), True, -29, False), "omega_0": (3, ((76, 84), (90, 114)), True, -31, True),
    "C_is": (3, ((120, 136),), True, -29, False), "i_0": (3, ((136, 144), (150, 174)), True, -31, True),
    "C_rc": (3, ((180, 196),), True, -5, False), "omega": (3, ((196, 204), (210, 234)), True, -31, True),
    "omegaDot": (3, ((240, 264),), True, -43, True), "IODE_sf3": (3, ((270, 278),), False, 0, False),
    "iDot": (3, ((278, 292),), True, -43, True),
}


def _field(sf, ranges, signed):
    v, n = 0, 0
    for lo, hi in ranges:
        for b in sf[lo:hi]:
            v = (v << 1) | int(b)
        n += hi - lo
    if signed and v >> (n - 1):
        v -= 1 << n
    return v


def ephemeris(bits, d30star):
    """``ephemeris.ephemeris(bits, D30Star)`` of the reference (ephemeris.py:98-196) on hard bits: ``bits`` holds
    1500 values 0/1 (or the characters '0'/'1') starting at a subframe boundary, ``d30star`` the bit before them.
    Returns (dict keyed by ``EPH_ALL``, TOW); fields of a subframe ID that does not occur stay ``None`` (the
    reference raises ``UnboundLocalError`` there, the caller's ``is None`` checks at postNavigation.py:142-146
    are what they feed)."""
    b = np.array([int(x) for x in bits[:1500]], dtype=np.uint8)
    if b.size < 1500:
        raise TypeError('The parameter BITS must contain 1500 bits!')                      # ephemeris.py:101
    words = b.reshape(50, 30).copy()
    prev = np.concatenate([[int(d30star)], words[:-1, 29]])                                 # parity bits are never inverted
    words[:, :24] ^= prev[:, None].astype(np.uint8)                                         # checkPhase, :122-127
    out = dict.fromkeys(EPH_ALL)
    for i in range(5):
        sf = words[10 * i:10 * i + 10].reshape(300)
        sid = _field(sf, ((49, 52),), False)                                                # :133
        for name, (fid, ranges, signed, p2, pi) in _EPH_LAYOUT.items():
            if fid == sid:
                v = _field(sf, ranges, signed)
                if name == "weekNumber":
                    v += 1024                                                                # :139
                if p2 or pi:
                    v = v * 2 ** p2
                    if pi:
                        v = v * _GPS_PI
                out[name] = v
    tow = _field(words[40:50].reshape(300), ((30, 47),), False) * 6 - 30                     # :190
    return out, tow


def nav_settings(settings):
    """The settings the measurement loop reads (initialize.py:144-181) as the C-ABI struct."""
    return _native.SgxNavSettings(float(settings.samplesPerCode), float(settings.startOffset), float(settings.c),
                                  float(settings.navSolPeriod), float(settings.elevationMask),
                                  int(bool(settings.useTropCorr)), 0)


def nav_epochs(settings, sub_frame_start):
    """Number of measurement epochs, postNavigation.py:199."""
    return int(np.fix(settings.msToProcess - np.max(sub_frame_start)) / settings.navSolPeriod)


def nav_solve_batch(abs_sample, sub_frame_start, ready, eph, tow, settings, stride=None, ms=None, want_sat=True,
                    stream=0):
    """Measurement loops of R independent recordings in one launch (postNavigation.py:159-301).

    ``abs_sample``: float64 ``[R, C, ms]`` numpy array, or ``track_batch``'s ``[R, C, 13, ms]`` output (numpy or CUDA
    tensor; field 0 is read in place); ``sub_frame_start`` / ``ready`` ``[R, C]``; ``eph`` ``[R, C, 21]`` in
    ``_native.EPH_FIELDS`` order (row c = ephemeris of channel c's PRN); ``tow`` ``[R]``.
    Returns a dict: ``rawP, correctedP, el, az, active`` ``[R, E, C]``, ``satPositions`` ``[R, E, C, 3]``,
    ``satClkCorr``, ``sol`` ``[R, E, 12]`` (``_native.NAV_SOL_FIELDS``), ``n_epochs`` ``[R]``."""
    shape = tuple(abs_sample.shape)
    r, c = shape[0], shape[1]
    if ms is None:
        ms = shape[-1]
    if stride is None:
        stride = int(np.prod(shape[2:]))
    sub_frame_start = np.asarray(sub_frame_start).reshape(r, c)
    n_ep = np.array([nav_epochs(settings, sub_frame_start[i]) for i in range(r)], dtype=np.int32)
    if isinstance(abs_sample, np.ndarray):
        abs_sample = np.ascontiguousarray(abs_sample, dtype=np.float64)
    return _native.lib().nav_solve(abs_sample, stride, r, c, ms, sub_frame_start, ready, eph, tow, n_ep,
                                   nav_settings(settings), want_sat=want_sat, stream=stream)


def vel_settings(settings):
    """``sgx_vel_settings`` from ``IF``, ``c``, ``navSolPeriod`` and the extension attributes ``L1Freq`` and
    ``dopplerAvgMs``; an object without the latter (the reference's own Settings) gets 1575.42e6 Hz and 100."""
    return _native.SgxVelSettings(IF=float(settings.IF), c=float(settings.c),
                                  f_L1=float(getattr(settings, "L1Freq", 1575.42e6)),
                                  nav_sol_period=float(settings.navSolPeriod),
                                  doppler_avg_ms=int(getattr(settings, "dopplerAvgMs", 100)), reserved=0)


def nav_velocity_batch(track_out, nav_out, sub_frame_start, eph, tow, settings, ms_done=None, want_sat=False, stream=0):
    """Receiver velocity and clock drift at the epochs of ``nav_out`` from the Doppler the PLL tracked, computed by
    ``sgx_nav_velocity`` (csrc/sgx_nav.cu; contract in include/softgnss_b200.h).

    ``track_out``: ``track_batch``'s float64 ``[R, C, 13, ms]`` output, numpy array or contiguous CUDA tensor (carrFreq,
    field 2, is read in place), or a ``[R, C, ms]`` carrFreq array.  ``nav_out``: the dict of :func:`nav_solve_batch` or
    :func:`post_navigate_batch` (``active``, ``sol``, ``n_epochs`` are read).  ``sub_frame_start`` ``[R, C]``, ``eph``
    ``[R, C, 21]`` and ``tow`` ``[R]``: what the fix was computed from.  ``ms_done`` ``[R, C]``: periods tracked
    (``track_batch``'s third result), None for all.  Returns numpy ``vel`` ``[R, E, 8]`` (``_native.NAV_VEL_FIELDS``),
    ``doppler`` and ``rrResid`` ``[R, E, C]``, and with ``want_sat`` ``satVel`` ``[R, E, C, 3]`` and ``satClkDrift``.
    There is no host implementation: without a device this raises NativeError."""
    L = _native.lib()
    L.require_device()
    shape = tuple(track_out.shape)
    r, c, ms = shape[0], shape[1], shape[-1]
    if len(shape) == 4:
        carr, stride, keep = _native.track_field(track_out, "carrFreq")
    else:                                                    # [R, C, ms] carrFreq rows
        carr = keep = track_out if hasattr(track_out, "data_ptr") else np.ascontiguousarray(track_out, dtype=np.float64)
        stride = ms
    out = L.nav_velocity(carr, stride, r, c, ms, ms_done, sub_frame_start, eph, tow, nav_out["n_epochs"],
                         nav_out["active"], nav_out["sol"], vel_settings(settings), want_sat=want_sat, stream=stream)
    if not want_sat:
        out.pop("satVel"), out.pop("satClkDrift")
    return out


# ---- RAIM tables: chi-square and noncentral chi-square in float64 with math only (scipy is not a dependency) -------------
def _gamma_pq(a, x):
    """Regularised incomplete gamma functions (P(a, x), Q(a, x)): series for x < a + 1, else Lentz's continued fraction
    for Q (each accurate to a few ulp relative; the complement then to a few ulp absolute)."""
    if x <= 0.0:
        return 0.0, 1.0
    lead = math.exp(a * math.log(x) - x - math.lgamma(a))
    if x < a + 1.0:
        term = s = 1.0 / a
        n = 1
        while term > s * 1e-17:
            term *= x / (a + n)
            s += term
            n += 1
        p = s * lead
        return p, 1.0 - p
    tiny = 1e-300
    b = x + 1.0 - a
    c, d = 1.0 / tiny, 1.0 / b
    h = d
    for i in range(1, 10000):
        an = -i * (i - a)
        b += 2.0
        d = an * d + b
        d = tiny if abs(d) < tiny else d
        c = b + an / c
        c = tiny if abs(c) < tiny else c
        d = 1.0 / d
        delta = d * c
        h *= delta
        if abs(delta - 1.0) < 1e-16:
            break
    q = lead * h
    return 1.0 - q, q


def _ncx2_cdf(x, k, lam):
    """Noncentral chi-square CDF: sum_j Poisson(j; lam/2) P(k/2 + j, x/2), with P(a + 1, y) = P(a, y) - y^a e^-y /
    Gamma(a + 1) from one accurate P(k/2, x/2)."""
    y, a, m = 0.5 * x, 0.5 * k, 0.5 * lam
    p = _gamma_pq(a, y)[0]
    g = math.exp(a * math.log(y) - y - math.lgamma(a + 1.0))           # y^a e^-y / Gamma(a + 1)
    total, j = 0.0, 0
    while True:
        w = math.exp(-m + (j * math.log(m) if m > 0 else 0.0) - math.lgamma(j + 1.0)) if (m > 0 or j == 0) else 0.0
        total += w * p
        if (j > m and w * p < 1e-20 * total) or p <= 0.0 or j > 100000:
            return total
        p = max(p - g, 0.0)
        g *= y / (a + j + 1.0)
        j += 1


def _bisect(f, lo, hi):
    """Root of a decreasing f on [lo, hi] (f(lo) > 0 > f(hi)) to the last bit."""
    while True:
        mid = 0.5 * (lo + hi)
        if mid <= lo or mid >= hi:
            return mid
        if f(mid) > 0:
            lo = mid
        else:
            hi = mid


def raim_tables(pfa, pmd, max_dof=_native.INTEG_MAX_DOF):
    """``(thresh, pbias)``, float64 ``[max_dof]``, entry k for dof = k + 1: the chi-square threshold T with upper tail
    ``pfa`` (false alarm) and sqrt(lambda) of the noncentrality lambda whose noncentral chi-square CDF at T is ``pmd``
    (missed detection).  The inputs of ``sgx_integ_settings``."""
    assert 0 < pfa < 1 and 0 < pmd < 1 and max_dof >= 1
    thresh, pbias = np.empty(max_dof), np.empty(max_dof)
    for k in range(1, max_dof + 1):
        hi = 2.0 * k + 10.0
        while _gamma_pq(0.5 * k, 0.5 * hi)[1] > pfa:
            hi *= 2.0
        t = _bisect(lambda v: _gamma_pq(0.5 * k, 0.5 * v)[1] - pfa, 0.0, hi)
        hi = t + 10.0
        while _ncx2_cdf(t, k, hi) > pmd:
            hi *= 2.0
        lam = _bisect(lambda v: _ncx2_cdf(t, k, v) - pmd, 0.0, hi)
        thresh[k - 1], pbias[k - 1] = t, math.sqrt(lam)
    return thresh, pbias


_TABLES = {}


def integ_settings(settings):
    """``sgx_integ_settings`` from the extension attributes ``raimSigma``, ``raimPfa`` and ``raimPmd``; an object without
    them (the reference's own Settings) gets 5.0 m, 1e-5 and 1e-3."""
    pfa, pmd = float(getattr(settings, "raimPfa", 1e-5)), float(getattr(settings, "raimPmd", 1e-3))
    if (pfa, pmd) not in _TABLES:
        _TABLES[(pfa, pmd)] = raim_tables(pfa, pmd)
    thresh, pbias = _TABLES[(pfa, pmd)]
    st = _native.SgxIntegSettings()
    st.sigma = float(getattr(settings, "raimSigma", 5.0))
    st.thresh[:] = thresh.tolist()
    st.pbias[:] = pbias.tolist()
    return st


def nav_integrity_batch(nav_out, eph, tow, settings, stream=0):
    """RAIM at the epochs of ``nav_out`` (the dict of :func:`nav_solve_batch` or :func:`post_navigate_batch`; ``rawP``,
    ``active``, ``sol`` and ``n_epochs`` are read), computed by ``sgx_nav_integrity`` (csrc/sgx_nav.cu; contract in
    include/softgnss_b200.h).  ``eph`` ``[R, C, 21]`` and ``tow`` ``[R]``: what the fix was computed from.  Returns numpy
    ``integ`` ``[R, E, 16]`` (``_native.NAV_INTEG_FIELDS``; status values index ``_native.INTEG_STATUS``) and
    ``normResid`` ``[R, E, C]``.  There is no host implementation: without a device this raises NativeError."""
    L = _native.lib()
    L.require_device()
    return L.nav_integrity(nav_out["rawP"], nav_out["active"], nav_out["sol"], nav_out["n_epochs"], eph, tow,
                           nav_settings(settings), integ_settings(settings), stream=stream)


def eph_rows(eph, prn):
    """Rows of ``_native.EPH_FIELDS`` for the channels' PRNs from the reference's ephemeris recarray
    (postNavigation.py:120-140: ``eph[PRN - 1].<field>``); channels without an ephemeris get zeros."""
    rows = np.zeros((len(prn), len(_native.EPH_FIELDS)))
    for ch, p in enumerate(prn):
        if p <= 0:
            continue
        rec = eph[int(p) - 1]
        if rec is None:
            continue
        vals = [rec[k] if isinstance(rec, dict) else getattr(rec, k) for k in _native.EPH_FIELDS]
        if all(v is not None for v in vals):
            rows[ch] = vals
    return rows


def navSolutions(trackResults, subFrameStart, readyChnList, eph, TOW, settings):
    """The measurement loop of ``postNavigate`` for one recording in the reference's own result layout
    (postNavigation.py:176-197): returns (navSolutions, channel) -- ``navSolutions.X/Y/Z/dt/latitude/longitude/
    height`` of length E, ``.DOP`` ``[5, E]``; ``channel.PRN/el/az/rawP/correctedP`` ``[numberOfChannels, E]``.
    UTM fields (``E, N, U, utmZone``) are left to the reference's ``cart2utm``."""
    nav, channel, _ = _nav_solutions(trackResults, subFrameStart, readyChnList, eph, TOW, settings)
    return nav, channel


def _nav_solutions(trackResults, subFrameStart, readyChnList, eph, TOW, settings):
    """navSolutions plus the dict of nav_solve_batch and the inputs it was given (``subFrameStart``, ``ephRows``,
    ``tow``)."""
    n_ch = settings.numberOfChannels
    ms = len(trackResults[0].absoluteSample)
    abs_sample = np.zeros((1, n_ch, ms))
    prn = np.zeros(n_ch, dtype=np.int64)
    for c in range(min(n_ch, len(trackResults))):
        abs_sample[0, c] = trackResults[c].absoluteSample
        prn[c] = trackResults[c].PRN
    ready = np.zeros((1, n_ch), dtype=np.uint8)
    ready[0, np.asarray(readyChnList, dtype=int)] = 1
    rows = eph_rows(eph, prn)[None]
    out = nav_solve_batch(abs_sample, np.asarray(subFrameStart)[None, :n_ch], ready, rows, [float(TOW)], settings)
    sol = out["sol"][0]
    channel = np.rec.array([(np.where(out["active"][0].T > 0, prn[:, None], 0).astype(np.float64), out["el"][0].T.copy(),
                             out["az"][0].T.copy(), out["rawP"][0].T.copy(), out["correctedP"][0].T.copy())],
                           formats=['O'] * 5, names='PRN,el,az,rawP,correctedP')
    nav = np.rec.array([(channel, sol[:, 4:9].T.copy(), sol[:, 0].copy(), sol[:, 1].copy(), sol[:, 2].copy(),
                         sol[:, 3].copy(), sol[:, 9].copy(), sol[:, 10].copy(), sol[:, 11].copy())],
                       formats=['O'] * 9, names='channel,DOP,X,Y,Z,dt,latitude,longitude,height')
    out.update(subFrameStart=np.asarray(subFrameStart)[None, :n_ch], ephRows=rows, tow=np.array([float(TOW)]))
    return nav, channel, out


def _decode_channels(bits, valid, first, prn, candidates):
    """Ephemeris decoding of the channels in ``candidates`` (postNavigation.py:120-146).  Returns
    (eph list indexed by PRN-1, TOW of the last decoded channel, channels that keep a complete ephemeris)."""
    eph = [None] * 32
    tow = None
    ready = []
    for ch in candidates:
        if first[ch] == 0 or not valid[ch]:          # five subframes do not fit after the preamble (the reference raises)
            continue
        e, tow = ephemeris(bits[ch][1:], bits[ch][0])                                        # :140
        eph[int(prn[ch]) - 1] = e
        if e["IODC"] is None or e["IODE_sf2"] is None or e["IODE_sf3"] is None:              # :142-146
            continue
        ready.append(ch)
    return eph, tow, np.array(ready, dtype=int)


def postNavigate(trackResults, settings):
    """``NavigationResult.postNavigate`` (postNavigation.py:75-301) on the B200 stages: preamble search and bit
    summation (``sgx_find_preambles``), ephemeris decoding (host bit slicing), measurement loop
    (``sgx_nav_solve``).  Returns ``(navSolutions, eph)`` -- ``(None, None)`` with the reference's messages when
    the record is too short or fewer than four satellites have an ephemeris.  ``navSolutions`` is the recarray of
    :func:`navSolutions` (no UTM fields); ``eph`` a list of 32 dicts/None indexed by PRN-1."""
    r = _post_navigate(trackResults, settings)
    return (None, None) if r is None else (r[0], r[1])


def _post_navigate(trackResults, settings):
    """postNavigate's chain; (navSolutions, eph, nav_solve dict) or None with the reference's messages."""
    tracked = (trackResults.status != '-') if trackResults.status.dtype.kind != 'S' else (trackResults.status != b'-')
    if settings.msToProcess < 36000 or int(tracked.sum()) < 4:                                # :104-111
        print('Record is to short or too few satellites tracked. Exiting!')
        return None
    subFrameStart, activeChnList, bits, valid = findPreambles(trackResults, settings, return_bits=True)   # :115
    prn = [int(trackResults[c].PRN) for c in range(len(trackResults))]
    eph, TOW, ready = _decode_channels(bits, valid, subFrameStart, prn, activeChnList) if bits is not None \
        else ([None] * 32, None, np.zeros(0, dtype=int))
    if ready.size < 4:                                                                        # :149-156
        print('Too few satellites with ephemeris data for position calculations. Exiting!')
        return None
    nav, _, out = _nav_solutions(trackResults, subFrameStart, ready, eph, TOW, settings)
    return nav, eph, out


def postNavigateVelocity(trackResults, settings):
    """:func:`postNavigate` plus the receiver velocity and clock drift of every measurement epoch (extension; no
    reference behaviour).  Returns ``(navSolutions, eph, navVelocities)``, ``(None, None, None)`` where postNavigate
    returns ``(None, None)``.  ``navVelocities`` is a one-record recarray with the length-E fields ``VX VY VZ`` (ECEF,
    m/s), ``clkDrift`` (m/s), ``VE VN VU`` (m/s, at the fix's latitude and longitude), ``nUsed`` (channels in the
    solution) and ``doppler`` ``[numberOfChannels, E]`` (Hz, NaN for channels not used).  The Doppler of a channel is
    the mean carrFreq of the ``settings.dopplerAvgMs`` code periods that end at the epoch, minus ``settings.IF``."""
    r = _post_navigate(trackResults, settings)
    if r is None:
        return None, None, None
    nav, eph, out = r
    n_ch = settings.numberOfChannels
    ms = len(trackResults[0].carrFreq)
    carr = np.zeros((1, n_ch, ms))
    for c in range(min(n_ch, len(trackResults))):
        carr[0, c] = trackResults[c].carrFreq
    v = nav_velocity_batch(carr, out, out["subFrameStart"], out["ephRows"], out["tow"], settings)
    vel = v["vel"][0]
    cols = [vel[:, k].copy() for k in range(len(_native.NAV_VEL_FIELDS))]
    velocities = np.rec.array([tuple(cols) + (v["doppler"][0].T.copy(),)], formats=['O'] * 9,
                              names=','.join(_native.NAV_VEL_FIELDS) + ',doppler')
    return nav, eph, velocities


def postNavigateIntegrity(trackResults, settings):
    """:func:`postNavigate` plus the integrity of every measurement epoch (extension; no reference behaviour).  Returns
    ``(navSolutions, eph, navIntegrity)``, ``(None, None, None)`` where postNavigate returns ``(None, None)``.
    ``navIntegrity`` is a one-record recarray with the length-E fields of ``_native.NAV_INTEG_FIELDS`` -- the final fix
    ``X Y Z dt latitude longitude height`` (K8's unless a channel was excluded), the all-in-view statistic ``q``, its
    threshold ``T`` and ``dof``, ``qFinal``, the protection levels ``HPL VPL`` (m), ``status`` (index into
    ``_native.INTEG_STATUS``), ``excluded`` (channel, -1 for none), ``nUsed`` -- and ``normResid``
    ``[numberOfChannels, E]``.  Settings: ``raimSigma`` (m), ``raimPfa``, ``raimPmd``."""
    r = _post_navigate(trackResults, settings)
    if r is None:
        return None, None, None
    nav, eph, out = r
    g = nav_integrity_batch(out, out["ephRows"], out["tow"], settings)
    integ = g["integ"][0]
    cols = [integ[:, k].copy() for k in range(len(_native.NAV_INTEG_FIELDS))]
    integrity = np.rec.array([tuple(cols) + (g["normResid"][0].T.copy(),)], formats=['O'] * 17,
                             names=','.join(_native.NAV_INTEG_FIELDS) + ',normResid')
    return nav, eph, integrity


def post_navigate_batch(track_out, prn, settings, stream=0, velocity=False, ms_done=None, integrity=False):
    """The same chain for R recordings whose tracking result ``track_out`` (float64 ``[R, C, 13, ms]``, numpy or
    CUDA tensor as written by ``track_batch``) stays where it is: ``I_P`` and ``absoluteSample`` are read in
    place by the two device stages; only the 1501 hard bits per channel and the solutions cross to the host.
    ``prn``: int ``[R, C]`` (0 = channel not tracked).  Returns the dict of :func:`nav_solve_batch` plus
    ``subFrameStart`` ``[R, C]``, ``ready`` ``[R, C]``, ``tow`` ``[R]`` and ``eph`` (R lists indexed by PRN-1);
    recordings with fewer than four usable satellites get ``n_epochs = 0``.  With ``velocity=True`` the dict also
    carries ``vel``, ``doppler`` and ``rrResid`` of :func:`nav_velocity_batch` (carrFreq read in place; ``ms_done``
    ``[R, C]`` as returned by ``track_batch``, None for all ms).  With ``integrity=True`` it also carries ``integ`` and
    ``normResid`` of :func:`nav_integrity_batch`."""
    r, c, _, ms = track_out.shape
    prn = np.asarray(prn).reshape(r, c)
    L = _native.lib()
    ip, stride, track_out = _native.track_field(track_out, "I_P")
    first, bits, valid = L.find_preambles(ip, stride, r * c, ms, stream=stream)
    first = first.reshape(r, c)
    first[prn == 0] = 0
    ready = np.zeros((r, c), dtype=np.uint8)
    rows = np.zeros((r, c, len(_native.EPH_FIELDS)))
    tow = np.zeros(r)
    ephs = []
    n_ep = np.zeros(r, dtype=np.int32)
    for i in range(r):
        cand = [ch for ch in range(c) if prn[i, ch] > 0 and first[i, ch] > 0]
        eph, t, rdy = _decode_channels(bits[i * c:(i + 1) * c], valid[i * c:(i + 1) * c], first[i], prn[i], cand)
        ephs.append(eph)
        if rdy.size >= 4 and settings.msToProcess >= 36000:
            ready[i, rdy] = 1
            rows[i] = eph_rows(eph, np.where(ready[i] > 0, prn[i], 0))
            tow[i] = t
            n_ep[i] = nav_epochs(settings, first[i])
    abs_sample = _native.track_field(track_out, "absoluteSample")[0]
    out = L.nav_solve(abs_sample, stride, r, c, ms, first, ready, rows, tow, n_ep, nav_settings(settings), stream=stream)
    out.update(subFrameStart=first, ready=ready, tow=tow, eph=ephs)
    if velocity:
        out.update(nav_velocity_batch(track_out, out, first, rows, tow, settings, ms_done=ms_done, stream=stream))
    if integrity:
        out.update(nav_integrity_batch(out, rows, tow, settings, stream=stream))
    return out


def install(navigation_result_cls):
    """Bind the B200 preamble search into the reference's own class (see INTEGRATION.md):
    ``NavigationResult.findPreambles`` keeps its signature and return value."""
    def _find(self):
        return findPreambles(self._results, self._settings)
    def _pseudo(self, msOfTheSignal, channelList):
        return calculatePseudoranges(self._results, msOfTheSignal, channelList, self._settings)
    navigation_result_cls.findPreambles = _find
    navigation_result_cls.calculatePseudoranges = _pseudo
    return navigation_result_cls
