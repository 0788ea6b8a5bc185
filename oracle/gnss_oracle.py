"""CPU oracle for the acquisition and tracking hot paths  --  TEST INFRASTRUCTURE ONLY.

A float64 numpy restatement of what the reference computes (it is *not* shipped and
the product never imports it: only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may).  Every function
cites the reference lines it follows (paths relative to the reference repo).

Pinning: the reference has no tests or golden vectors of its own (SURVEY.md section 4),
so this restatement is pinned against the reference itself, run in the build
container through the mechanical Python-3 shim (``oracle/make_ref_shim.py``):

* ``tests/golden/*.npz`` -- outputs of the shimmed reference on seeded synthetic
  recordings, produced by ``tests/golden/make_golden.py`` (committed with the data);
* ``tests/test_oracle_vs_reference.py`` -- live diff when ``/root/reference`` exists.

Arithmetic that the reference delegates to numpy (pocketfft ``np.fft``, ufuncs) is
delegated to the same numpy calls here (numpy 2.3.5 in this image; the reference
pins no version, README.md:7-10).

The ``coherent_ms`` / ``noncoh_blocks`` / ``doppler_step`` arguments of
:func:`acquire` are extensions with *no* reference behaviour (BASELINE.json configs 3
and 5); at their defaults (1, 2, 500.0) the function reduces to the reference.
"""
import numpy as np

TWO_PI = 2 * np.pi

_G2S = [5, 6, 7, 8, 17, 18, 139, 140, 141, 251, 252, 254, 255, 256, 257, 258, 469, 470, 471,
        472, 473, 474, 509, 512, 513, 514, 515, 516, 859, 860, 861, 862]


# --------------------------------------------------------------------------- helpers
def samples_per_code(s):
    """initialize.py:183-185."""
    return int(np.round(s.samplingFreq / (s.codeFreqBasis / s.codeLength)))


def ca_code(prn0):
    """initialize.py:234-302 -- +-1 register arithmetic as the reference does it."""
    assert 0 <= prn0 < 32

    def run(tap_idx):
        reg = -np.ones(10)
        seq = np.zeros(1023)
        for i in range(1023):
            seq[i] = reg[9]
            fb = np.prod(reg[tap_idx])
            reg[1:] = reg[:-1].copy()
            reg[0] = fb
        return seq

    g1 = run([2, 9])                      # :272
    g2 = run([1, 2, 5, 7, 8, 9])          # :290
    sh = _G2S[prn0]
    g2 = np.concatenate((g2[1023 - sh:], g2[:1023 - sh]))   # :298
    return -g1 * g2                       # :301


_CODE_CACHE = {}


def ca_code_cached(prn0):
    if prn0 not in _CODE_CACHE:
        _CODE_CACHE[prn0] = ca_code(prn0)
    return _CODE_CACHE[prn0]


def ca_table(s):
    """initialize.py:188-231."""
    n = samples_per_code(s)
    ts = 1.0 / s.samplingFreq
    tc = 1.0 / s.codeFreqBasis
    idx = np.ceil(ts * np.arange(1, n + 1) / tc) - 1        # :223
    idx = idx.astype(np.int64)
    idx[-1] = 1022                                          # :226
    return np.array([ca_code_cached(p)[idx] for p in range(32)])


def loop_coef(lbw, zeta, k):
    """initialize.py:306-328."""
    wn = lbw * 8.0 * zeta / (4.0 * zeta ** 2 + 1)
    return k / (wn * wn), 2.0 * zeta / wn


# --------------------------------------------------------------------------- acquisition
def _exclusion_range(code_phase, chip_samples, n):
    """acquisition.py:147-159 -- candidate indices for the second peak (may contain
    negative values, which index from the end exactly as numpy does there)."""
    lo = code_phase - chip_samples
    hi = code_phase + chip_samples
    if lo <= 0:
        return np.arange(hi, n + lo + 1)
    if hi >= n - 1:
        return np.arange(hi - n, lo)
    return np.concatenate((np.arange(0, lo + 1), np.arange(hi, n)))


def acquire(long_signal, s, coherent_ms=1, noncoh_blocks=2, doppler_step=500.0,
            return_debug=False, clamp_window=False):
    """acquisition.py:49-204.  Returns dict(carrFreq, codePhase, peakMetric) (float64[32]).

    ``clamp_window=True`` drops the out-of-range index the reference generates when
    codePhase == samplesPerCodeChip (its IndexError, SURVEY.md appendix A.1-6) --
    that is the behaviour the CUDA path implements for that one case.
    """
    n1 = samples_per_code(s)
    n = n1 * coherent_ms
    x = np.asarray(long_signal)
    blocks = [x[b * n:(b + 1) * n] for b in range(noncoh_blocks)]          # :55-57
    x0 = x - x.mean()                                                      # :59
    ts = 1.0 / s.samplingFreq
    phase_pts = np.arange(n) * 2 * np.pi * ts                              # :65
    if doppler_step == 500.0:
        nbins = int(np.round(s.acqSearchBand * 2) + 1)                     # :68
    else:
        nbins = int(np.round(s.acqSearchBand * 1000.0 / doppler_step) + 1)
    table = ca_table(s)                                                    # :71
    if coherent_ms > 1:
        table = np.tile(table, (1, coherent_ms))
    nprn = len(s.acqSatelliteList)                                         # :92 (length only)
    carr = np.zeros(32)
    cph = np.zeros(32)
    metric = np.zeros(32)
    dbg = {}
    freqs = np.array([s.IF - s.acqSearchBand / 2 * 1000 + doppler_step * k
                      for k in range(nbins)])                              # :99-101
    # Carrier wipe-off does not depend on the PRN; do it once per (bin, block).
    spec = np.empty((noncoh_blocks, nbins, n), dtype=np.complex128)
    for k in range(nbins):
        sin_c = np.sin(freqs[k] * phase_pts)                               # :103
        cos_c = np.cos(freqs[k] * phase_pts)                               # :105
        for b in range(noncoh_blocks):
            spec[b, k] = np.fft.fft(sin_c * blocks[b] + 1j * (cos_c * blocks[b]))  # :107-117
    for prn in range(nprn):
        code_f = np.fft.fft(table[prn]).conj()                             # :95
        results = np.zeros((nbins, n1))
        block_max = np.zeros((nbins, noncoh_blocks))
        for k in range(nbins):
            best = None
            for b in range(noncoh_blocks):
                r = abs(np.fft.ifft(spec[b, k] * code_f)) ** 2             # :120-126
                if coherent_ms > 1:
                    r = r[:n1]      # extension: the correlation repeats every code period; search one
                block_max[k, b] = r.max()
                # :129-133 keep block 1 only if strictly larger, later blocks win ties
                if best is None or not (best.max() > r.max()):
                    best = r
            results[k] = best
        fbin = results.max(1).argmax()                                     # :140
        peak = results.max(0).max()                                        # :142
        cp = int(results.max(0).argmax())                                  # :143
        chip = int(round(s.samplingFreq / s.codeFreqBasis))                # :145
        rng = _exclusion_range(cp, chip, n1)
        if clamp_window:
            rng = rng[rng < n1]
        second = results[fbin, rng].max()                                  # :162
        metric[prn] = peak / second                                        # :164
        if return_debug:
            # besides the decisions, what a test needs to see how clear they are: the block maxima of every bin, the
            # row maxima (bin decision), the column maxima (code phase), the winning row and where its second peak is
            dbg[prn] = dict(bin=int(fbin), codePhase=cp, peak=peak, second=second,
                            secondIndex=int(rng[results[fbin, rng].argmax()]) % n1, blockMax=block_max,
                            binMax=results.max(1), colMax=results.max(0), row=results[fbin].copy())
        if peak / second > s.acqThreshold:                                 # :166
            code = ca_code_cached(prn)
            idx = np.floor(ts * np.arange(1, 10 * n1 + 1) / (1.0 / s.codeFreqBasis))   # :172
            long_code = code[(idx % 1023).astype(np.int64)]                # :174
            xc = x0[cp:cp + 10 * n1] * long_code                           # :177
            nfft = int(8 * 2 ** (np.ceil(np.log2(len(xc)))))               # :179
            mag = np.abs(np.fft.fft(xc, nfft))                             # :182
            uniq = int(np.ceil((nfft + 1) / 2.0))                          # :184
            imax = mag[4:uniq - 5].argmax()                                # :187 (slice-relative!)
            bins = np.arange(uniq) * s.samplingFreq / nfft                 # :189
            carr[prn] = bins[imax]                                         # :191
            cph[prn] = cp                                                  # :193
            if return_debug:
                dbg[prn]["fineIndex"] = int(imax)
                dbg[prn]["fineRunnerUp"] = float(np.delete(mag[4:uniq - 5], imax).max())
                dbg[prn]["finePeak"] = float(mag[4 + imax])
    out = dict(carrFreq=carr, codePhase=cph, peakMetric=metric)
    if return_debug:
        out["debug"] = dbg
    return out


def pre_run(acq, s):
    """acquisition.py:259-306 -> dict(PRN int64[C], acquiredFreq, codePhase, status list)."""
    c = s.numberOfChannels
    prn = np.zeros(c, dtype=np.int64)
    freq = np.zeros(c)
    cph = np.zeros(c)
    status = ['-'] * c
    order = sorted(enumerate(acq["peakMetric"]), key=lambda t: t[-1], reverse=True)   # :288
    for i in range(min(c, int(np.sum(acq["carrFreq"] > 0)))):             # :294
        j = order[i][0]
        prn[i] = j + 1
        freq[i] = acq["carrFreq"][j]
        cph[i] = acq["codePhase"][j]
        status[i] = 'T'
    return dict(PRN=prn, acquiredFreq=freq, codePhase=cph, status=status)


# --------------------------------------------------------------------------- tracking
TRACK_FIELDS = ("absoluteSample", "codeFreq", "carrFreq", "I_P", "I_E", "I_L", "Q_E", "Q_P",
                "Q_L", "dllDiscr", "dllDiscrFilt", "pllDiscr", "pllDiscrFilt")


def track_channel(data, prn, acquired_freq, code_phase, s, ms=None):
    """tracking.py:99-283 for one channel.  ``data`` is the whole int8 recording (the
    reference reads the same bytes through fid.seek/np.fromfile).  Returns
    (dict of 13 float64[ms] series, ms_done); ms_done < ms means the short-read exit
    at tracking.py:159-163 fired."""
    ms = int(s.msToProcess) if ms is None else int(ms)
    fs = s.samplingFreq
    spc = s.dllCorrelatorSpacing
    t1c, t2c = loop_coef(s.dllNoiseBandwidth, s.dllDampingRatio, 1.0)      # :45
    t1p, t2p = loop_coef(s.pllNoiseBandwidth, s.pllDampingRatio, 0.25)     # :52
    pdi = 0.001
    out = {k: (np.zeros(ms) if k in ("absoluteSample", "I_P", "I_E", "I_L", "Q_E", "Q_P", "Q_L")
               else np.inf * np.ones(ms)) for k in TRACK_FIELDS}           # :65-94
    pos = int(s.skipNumberOfBytes + code_phase)                            # :107
    c = ca_code_cached(int(prn) - 1)
    code = np.concatenate(([c[-1]], c, [c[0]]))                            # :111
    code_freq = s.codeFreqBasis
    rem_code = 0.0
    carr_freq = acquired_freq
    carr_basis = acquired_freq
    rem_carr = 0.0
    old_code_nco = old_code_err = old_carr_nco = old_carr_err = 0.0
    done = 0
    for k in range(ms):
        step = code_freq / fs                                              # :148
        blk = int(np.ceil((s.codeLength - rem_code) / step))               # :150
        raw = data[pos:pos + blk]
        if len(raw) != blk:                                                # :159
            break
        pos += blk

        def replica(off):
            t = np.linspace(rem_code + off, blk * step + rem_code + off, blk, endpoint=False)
            return code[np.ceil(t).astype(np.int64)], t

        early, _ = replica(-spc)                                           # :166-172
        late, _ = replica(+spc)                                            # :174-180
        t = np.linspace(rem_code, blk * step + rem_code, blk, endpoint=False)
        prompt = code[np.ceil(t).astype(np.int64)]                         # :182-188
        rem_code = t[blk - 1] + step - 1023.0                              # :190
        tm = np.arange(0, blk + 1) / fs                                    # :193
        arg = carr_freq * 2.0 * np.pi * tm + rem_carr                      # :195
        rem_carr = arg[blk] % (2 * np.pi)                                  # :197
        q_bb = np.cos(arg[:blk]) * raw                                     # :199,205
        i_bb = np.sin(arg[:blk]) * raw                                     # :201,207
        ie, qe = (early * i_bb).sum(), (early * q_bb).sum()                # :209-211
        ip, qp = (prompt * i_bb).sum(), (prompt * q_bb).sum()              # :213-215
        il, ql = (late * i_bb).sum(), (late * q_bb).sum()                  # :217-219
        with np.errstate(divide="ignore", invalid="ignore"):
            carr_err = np.arctan(qp / ip) / 2.0 / np.pi                    # :223
        carr_nco = old_carr_nco + t2p / t1p * (carr_err - old_carr_err) + carr_err * (pdi / t1p)
        old_carr_nco, old_carr_err = carr_nco, carr_err                    # :225-231
        carr_freq = carr_basis + carr_nco                                  # :233
        e_mag = np.sqrt(ie * ie + qe * qe)
        l_mag = np.sqrt(il * il + ql * ql)
        with np.errstate(divide="ignore", invalid="ignore"):
            code_err = (e_mag - l_mag) / (e_mag + l_mag)                   # :238
        code_nco = old_code_nco + t2c / t1c * (code_err - old_code_err) + code_err * (pdi / t1c)
        old_code_nco, old_code_err = code_nco, code_err                    # :241-247
        code_freq = s.codeFreqBasis - code_nco                             # :249
        out["absoluteSample"][k] = pos                                     # :255 (fid.tell())
        out["codeFreq"][k] = code_freq
        out["carrFreq"][k] = carr_freq
        out["dllDiscr"][k] = code_err
        out["dllDiscrFilt"][k] = code_nco
        out["pllDiscr"][k] = carr_err
        out["pllDiscrFilt"][k] = carr_nco
        out["I_E"][k], out["I_P"][k], out["I_L"][k] = ie, ip, il
        out["Q_E"][k], out["Q_P"][k], out["Q_L"][k] = qe, qp, ql
        done += 1
    return out, done


def track(data, channels, s, ms=None):
    """tracking.py:59-295 -- list of (PRN, status, series dict) for channels with PRN != 0,
    or None if any channel hits the short-read exit (tracking.py:159-163)."""
    recs = []
    for ch in range(s.numberOfChannels):
        if channels["PRN"][ch] == 0:                                       # :99
            continue
        series, done = track_channel(data, channels["PRN"][ch], channels["acquiredFreq"][ch],
                                     channels["codePhase"][ch], s, ms)
        want = int(s.msToProcess) if ms is None else int(ms)
        if done != want:
            return None
        recs.append((int(channels["PRN"][ch]), channels["status"][ch], series))
    return recs


# ---------------------------------------------------------------------------------------------
# SURVEY.md section 8(f) row 3: preamble search / bit synchronisation (postNavigation.py:524-631)
# and the 20 ms bit summation of the caller (postNavigation.py:125-134).
# ---------------------------------------------------------------------------------------------
PREAMBLE_BITS = np.array([1, -1, -1, -1, 1, -1, 1, 1])                     # postNavigation.py:554


def nav_party_chk(ndat):
    """postNavigation.py:441-521 on a copy of 32 values of +-1: D29*, D30*, d1..d24, D25..D30.
    Returns -D30* (+1 / -1) when the six parity equations hold, else 0."""
    d = np.array(ndat, dtype=np.float64)
    if d[1] != 1:                                                         # :469
        d[2:26] *= -1
    taps = ((0, 2, 3, 4, 6, 7, 11, 12, 13, 14, 15, 18, 19, 21, 24),       # :480-504, indices into ndat
            (1, 3, 4, 5, 7, 8, 12, 13, 14, 15, 16, 19, 20, 22, 25),
            (0, 2, 4, 5, 6, 8, 9, 13, 14, 15, 16, 17, 20, 21, 23),
            (1, 3, 5, 6, 7, 9, 10, 14, 15, 16, 17, 18, 21, 22, 24),
            (1, 2, 4, 6, 7, 8, 10, 11, 15, 16, 17, 18, 19, 22, 23, 25),
            (0, 4, 6, 7, 9, 10, 11, 12, 14, 16, 20, 23, 24, 25))
    parity = np.array([np.prod(d[list(t)]) for t in taps])
    if (parity == d[26:]).sum() == 6:                                     # :507
        return -1 * d[1]
    return 0


def sum20(i_p, start, n_bits):
    """``I_P[start:start+20*n_bits].reshape(20, -1, order='F').sum(0)`` (postNavigation.py:596-598,
    :127-129) -- numpy's own reduction, so the rounding order is the reference's by construction."""
    seg = np.array(i_p[start:start + 20 * n_bits], dtype=np.float64)
    return seg.reshape(20, -1, order="F").sum(0)


def preamble_correlation(i_p):
    """Lags 0..M-1 of ``np.correlate(bits, zero-padded preamble_ms, 'full')`` (postNavigation.py:571-584).
    The reference evaluates the full M x M product; the 160 non-zero taps give the same integers."""
    bits = np.where(np.asarray(i_p, dtype=np.float64) > 0, 1, -1).astype(np.int32)   # :567-569 (NaN, 0 -> -1)
    pat = np.kron(PREAMBLE_BITS, np.ones(20, dtype=np.int32)).astype(np.int32)       # :558
    m = bits.size
    padded = np.concatenate([bits, np.zeros(pat.size, dtype=np.int32)])
    win = np.lib.stride_tricks.sliding_window_view(padded, pat.size)[:m]
    return win @ pat


def find_preambles(i_p_list, skip_unreadable=True):
    """postNavigation.py:524-631 for the tracked channels (status != '-') in result order.

    Returns (firstSubFrame int array, activeChnList).  ``skip_unreadable``: a candidate nearer than
    40 ms to the start of the record makes the reference read ``I_P[negative:positive]`` (an empty
    slice) and crash in ``navPartyChk``; with the flag such candidates are passed over (the only
    deviation, analogous to ``acquire(clamp_window=True)``)."""
    n_ch = len(i_p_list)
    first = np.zeros(n_ch, dtype=int)
    for ch in range(n_ch):
        i_p = np.asarray(i_p_list[ch], dtype=np.float64)
        corr = preamble_correlation(i_p)
        index = (np.abs(corr) > 153).nonzero()[0]                         # :584 (searchStartOffset = 0)
        cand = set(index.tolist())
        for k in index:
            if (k + 6000) not in cand:                                    # :593-595
                continue
            if k < 40:
                if skip_unreadable:
                    continue
                raise IndexError("reference reads I_P[%d:%d]" % (k - 40, k + 1200))
            if k + 1200 > i_p.size:                                       # unreachable: k + 6000 is a candidate
                continue
            s = sum20(i_p, k - 40, 62)                                    # :594-598
            bits = np.where(s > 0, 1, -1)                                 # :600-602
            if nav_party_chk(bits[:32]) != 0 and nav_party_chk(bits[30:62]) != 0:   # :604
                first[ch] = k
                break
    active = np.array([ch for ch in range(n_ch) if first[ch] != 0], dtype=int)      # :612-618
    return first, active


def nav_bits(i_p, sub_frame_start):
    """postNavigation.py:125-134: 1501 hard bits (0/1) of the five subframes that start at
    ``sub_frame_start``, preceded by the last bit of the subframe before."""
    s = sum20(i_p, sub_frame_start - 20, 1501)
    return (s > 0).astype(np.uint8)


# ---------------------------------------------------------------------------------------------
# SURVEY.md section 8(f) row 4, first half: relative pseudoranges (postNavigation.py:27-72)
# ---------------------------------------------------------------------------------------------
def calculate_pseudoranges(abs_sample, ms_of_the_signal, channel_list, n_channels, samples_per_code,
                           start_offset=68.802, c=299792458.0):
    """postNavigation.py:52-72.  ``abs_sample[ch]`` is the absoluteSample series of channel ch."""
    travel = np.inf * np.ones(n_channels)                                  # :52
    for ch in channel_list:                                                 # :58-61
        travel[ch] = abs_sample[ch][int(ms_of_the_signal[ch])] / samples_per_code
    with np.errstate(invalid="ignore"):
        minimum = np.floor(travel.min())                                    # :64
        travel = travel - minimum + start_offset                            # :66
        return travel * c / 1000                                            # :71


# ---------------------------------------------------------------------------------------------
# SURVEY.md section 8(f) row 4, second half: satellite positions, least-squares fix and the
# measurement-epoch loop of postNavigate (postNavigation.py:159-301, geoFunctions/__init__.py).
# Scalar float64 arithmetic in the reference's own operation order (np.float64 scalars, numpy ufuncs).
# ---------------------------------------------------------------------------------------------
EPH_FIELDS = ("t_oc", "a_f2", "a_f1", "a_f0", "T_GD", "sqrtA", "t_oe", "deltan", "M_0", "e", "omega",
              "C_uc", "C_us", "C_rc", "C_rs", "i_0", "iDot", "C_ic", "C_is", "omega_0", "omegaDot")


def check_t(time):
    """geoFunctions/__init__.py:745-771: week crossover."""
    half_week = 302400.0
    if time > half_week:
        return time - 2 * half_week
    if time < -half_week:
        return time + 2 * half_week
    return time


def satpos(transmit_time, prn_list, eph):
    """geoFunctions/__init__.py:779-885.  ``eph[prn-1]`` is a mapping with the EPH_FIELDS keys.
    Returns (satPositions float64 [3, n], satClkCorr float64 [n])."""
    n_sat = len(prn_list)
    gps_pi = 3.14159265359                                                  # :798
    omegae_dot = 7.2921151467e-05                                           # :803
    gm = 3.986005e+14                                                       # :805
    f_rel = -4.442807633e-10                                                # :808
    clk = np.zeros(n_sat)
    pos = np.zeros((3, n_sat))
    for k in range(n_sat):
        e = {key: np.float64(eph[int(prn_list[k]) - 1][key]) for key in EPH_FIELDS}
        dt = check_t(transmit_time - e["t_oc"])                             # :823
        clk[k] = (e["a_f2"] * dt + e["a_f1"]) * dt + e["a_f0"] - e["T_GD"]  # :825
        time = transmit_time - clk[k]                                       # :827
        a = e["sqrtA"] * e["sqrtA"]                                         # :831
        tk = check_t(time - e["t_oe"])                                      # :833
        n0 = np.sqrt(gm / a ** 3)                                           # :835
        n = n0 + e["deltan"]
        m = e["M_0"] + n * tk
        m = np.remainder(m + 2 * gps_pi, 2 * gps_pi)                        # :841
        ea = m
        for _ in range(10):                                                 # :845-853
            ea_old = ea
            ea = m + e["e"] * np.sin(ea)
            d_e = np.remainder(ea - ea_old, 2 * gps_pi)
            if abs(d_e) < 1e-12:
                break
        ea = np.remainder(ea + 2 * gps_pi, 2 * gps_pi)                      # :855
        dtr = f_rel * e["e"] * e["sqrtA"] * np.sin(ea)                      # :857
        nu = np.arctan2(np.sqrt(1 - e["e"] ** 2) * np.sin(ea), np.cos(ea) - e["e"])   # :859
        phi = nu + e["omega"]
        phi = np.remainder(phi, 2 * gps_pi)                                 # :863
        u = phi + e["C_uc"] * np.cos(2 * phi) + e["C_us"] * np.sin(2 * phi)            # :865
        r = a * (1 - e["e"] * np.cos(ea)) + e["C_rc"] * np.cos(2 * phi) + e["C_rs"] * np.sin(2 * phi)
        inc = e["i_0"] + e["iDot"] * tk + e["C_ic"] * np.cos(2 * phi) + e["C_is"] * np.sin(2 * phi)
        om = e["omega_0"] + (e["omegaDot"] - omegae_dot) * tk - omegae_dot * e["t_oe"]   # :871
        om = np.remainder(om + 2 * gps_pi, 2 * gps_pi)
        pos[0, k] = np.cos(u) * r * np.cos(om) - np.sin(u) * r * np.cos(inc) * np.sin(om)   # :875
        pos[1, k] = np.cos(u) * r * np.sin(om) + np.sin(u) * r * np.cos(inc) * np.cos(om)
        pos[2, k] = np.sin(u) * r * np.sin(inc)
        clk[k] = (e["a_f2"] * dt + e["a_f1"]) * dt + e["a_f0"] - e["T_GD"] + dtr        # :882
    return pos, clk


def e_r_corr(traveltime, x_sat):
    """geoFunctions/__init__.py:491-521: rotate by the Earth's rotation during the flight."""
    omegatau = 7.292115147e-05 * traveltime                                 # :508-511 (this constant, not satpos's)
    r3 = np.array([[np.cos(omegatau), np.sin(omegatau), 0.0],
                   [-np.sin(omegatau), np.cos(omegatau), 0.0],
                   [0.0, 0.0, 1.0]])
    return r3.dot(x_sat)


def togeod(a, finv, x, y, z):
    """geoFunctions/__init__.py:892-1000: geodetic latitude/longitude (degrees) and height."""
    h = 0.0
    tolsq = 1e-10
    maxit = 10
    rtd = 180 / np.pi
    esq = 0.0 if finv < 1e-20 else (2 - 1 / finv) / finv
    oneesq = 1 - esq
    p = np.sqrt(x ** 2 + y ** 2)
    dlambda = np.arctan2(y, x) * rtd if p > 1e-20 else 0.0
    if dlambda < 0:
        dlambda = dlambda + 360
    r = np.sqrt(p ** 2 + z ** 2)
    sinphi = z / r if r > 1e-20 else 0.0
    dphi = np.arcsin(sinphi)
    if r < 1e-20:
        return dphi, dlambda, 0.0
    h = r - a * (1 - sinphi * sinphi / finv)
    for _ in range(maxit):
        sinphi = np.sin(dphi)
        cosphi = np.cos(dphi)
        n_phi = a / np.sqrt(1 - esq * sinphi * sinphi)
        d_p = p - (n_phi + h) * cosphi
        d_z = z - (n_phi * oneesq + h) * sinphi
        h = h + sinphi * d_z + cosphi * d_p
        dphi = dphi + (cosphi * d_z - sinphi * d_p) / (n_phi + h)
        if (d_p * d_p + d_z * d_z) < tolsq:
            break
    dphi *= rtd
    return dphi, dlambda, h


def topocent(x, dx):
    """geoFunctions/__init__.py:1003-1063: azimuth, elevation (degrees) and length of dx seen from x."""
    dtr = np.pi / 180
    phi, lambda_, _ = togeod(6378137, 298.257223563, x[0], x[1], x[2])
    cl = np.cos(lambda_ * dtr)
    sl = np.sin(lambda_ * dtr)
    cb = np.cos(phi * dtr)
    sb = np.sin(phi * dtr)
    f = np.array([[-sl, -sb * cl, cb * cl], [cl, -sb * sl, cb * sl], [0.0, cb, sb]])
    local = f.T.dot(dx)
    e, n, u = local[0], local[1], local[2]
    hor_dis = np.sqrt(e ** 2 + n ** 2)
    if hor_dis < 1e-20:
        az, el = 0.0, 90.0
    else:
        az = np.arctan2(e, n) / dtr
        el = np.arctan2(u, hor_dis) / dtr
    if az < 0:
        az = az + 360
    d = np.sqrt(dx[0] ** 2 + dx[1] ** 2 + dx[2] ** 2)
    return az, el, d


def tropo(sinel, hsta, p, tkel, hum, hp, htkel, hhum):
    """geoFunctions/__init__.py:1071-1169: Goad-Goodman tropospheric delay in metres."""
    a_e = 6378.137
    b0 = 7.839257e-05
    tlapse = -6.5
    tkhum = tkel + tlapse * (hhum - htkel)
    atkel = 7.5 * (tkhum - 273.15) / (237.3 + tkhum - 273.15)
    e0 = 0.0611 * hum * 10 ** atkel
    tksea = tkel - tlapse * htkel
    em = -978.77 / (2870400.0 * tlapse * 1e-05)
    tkelh = tksea + tlapse * hhum
    e0sea = e0 * (tksea / tkelh) ** (4 * em)
    tkelp = tksea + tlapse * hp
    psea = p * (tksea / tkelp) ** em
    if sinel < 0:
        sinel = 0
    tropo_ = 0.0
    done = False
    refsea = 7.7624e-05 / tksea
    htop = 1.1385e-05 / refsea
    refsea = refsea * psea
    ref = refsea * ((htop - hsta) / htop) ** 4
    while 1:
        rtop = (a_e + htop) ** 2 - (a_e + hsta) ** 2 * (1 - sinel ** 2)
        if rtop < 0:
            rtop = 0
        rtop = np.sqrt(rtop) - (a_e + hsta) * sinel
        a = -sinel / (htop - hsta)
        b = -b0 * (1 - sinel ** 2) / (htop - hsta)
        rn = np.zeros(8)
        for i in range(8):
            rn[i] = rtop ** (i + 2)
        alpha = np.array([2 * a, 2 * a ** 2 + 4 * b / 3, a * (a ** 2 + 3 * b),
                          a ** 4 / 5 + 2.4 * a ** 2 * b + 1.2 * b ** 2,
                          2 * a * b * (a ** 2 + 3 * b) / 3,
                          b ** 2 * (6 * a ** 2 + 4 * b) * 0.1428571, 0, 0])
        if b ** 2 > 1e-35:
            alpha[6] = a * b ** 3 / 2
            alpha[7] = b ** 4 / 9
        dr = rtop
        dr = dr + alpha.dot(rn)
        tropo_ += dr * ref * 1000
        if done:
            return tropo_
        done = True
        refsea = (0.3719 / tksea - 1.292e-05) / tksea
        htop = 1.1385e-05 * (1255.0 / tksea + 0.05) / refsea
        ref = refsea * e0sea * ((htop - hsta) / htop) ** 4


def least_square_pos(satpos_, obs, c=299792458.0, use_trop_corr=True):
    """geoFunctions/__init__.py:636-739.  Returns (pos[4], el[n], az[n], dop[5]).
    Quirks kept: the design-matrix rows are divided by obs[i] (not by the geometric range, :706-709);
    ``trop = 2`` in the first iteration (:683); DOP from the last iteration's A (:726)."""
    dtr = np.pi / 180
    pos = np.zeros(4)
    x_all = satpos_.copy()
    n = satpos_.shape[1]
    a_mat = np.zeros((n, 4))
    omc = np.zeros(n)
    az = np.zeros(n)
    el = np.zeros(n)
    dop = np.zeros(5)
    for it in range(7):                                                      # :659
        for i in range(n):
            if it == 0:
                rot_x = x_all[:, i].copy()
                trop = 2
            else:
                rho2 = (x_all[0, i] - pos[0]) ** 2 + (x_all[1, i] - pos[1]) ** 2 + (x_all[2, i] - pos[2]) ** 2
                traveltime = np.sqrt(rho2) / c
                rot_x = e_r_corr(traveltime, x_all[:, i])
                az[i], el[i], _ = topocent(pos[0:3], rot_x - pos[0:3])
                if use_trop_corr:
                    trop = tropo(np.sin(el[i] * dtr), 0.0, 1013.0, 293.0, 50.0, 0.0, 0.0, 0.0)
                else:
                    trop = 0
            omc[i] = obs[i] - np.linalg.norm(rot_x - pos[0:3]) - pos[3] - trop          # :704
            a_mat[i, :] = np.array([-(rot_x[0] - pos[0]) / obs[i], -(rot_x[1] - pos[1]) / obs[i],
                                    -(rot_x[2] - pos[2]) / obs[i], 1])
        if np.linalg.matrix_rank(a_mat) != 4:                                # :712-715
            return np.zeros(4), el, az, dop
        x = np.linalg.lstsq(a_mat, omc, rcond=None)[0]                       # :717
        pos = pos + x.flatten()
    q = np.linalg.inv(a_mat.T.dot(a_mat))                                    # :726
    dop[0] = np.sqrt(np.trace(q))
    dop[1] = np.sqrt(q[0, 0] + q[1, 1] + q[2, 2])
    dop[2] = np.sqrt(q[0, 0] + q[1, 1])
    dop[3] = np.sqrt(q[2, 2])
    dop[4] = np.sqrt(q[3, 3])
    return pos, el, az, dop


def cart2geo(x, y, z, i=4):
    """geoFunctions/__init__.py:7-77 (ellipsoid 4 = WGS84): latitude, longitude (degrees), height."""
    a = np.array([6378388.0, 6378160.0, 6378135.0, 6378137.0, 6378137.0])
    f = np.array([1 / 297, 1 / 298.247, 1 / 298.26, 1 / 298.257222101, 1 / 298.257223563])
    lambda_ = np.arctan2(y, x)
    ex2 = (2 - f[i]) * f[i] / ((1 - f[i]) ** 2)
    c = a[i] * np.sqrt(1 + ex2)
    phi = np.arctan(z / (np.sqrt(x ** 2 + y ** 2) * (1 - (2 - f[i])) * f[i]))
    h = 0.1
    oldh = 0
    iterations = 0
    while abs(h - oldh) > 1e-12:
        oldh = h
        n = c / np.sqrt(1 + ex2 * np.cos(phi) ** 2)
        phi = np.arctan(z / (np.sqrt(x ** 2 + y ** 2) * (1 - (2 - f[i]) * f[i] * n / (n + h))))
        h = np.sqrt(x ** 2 + y ** 2) / np.cos(phi) - n
        iterations += 1
        if iterations > 100:
            break
    return phi * (180 / np.pi), lambda_ * (180 / np.pi), h


def nav_solve(abs_sample, prn, sub_frame_start, ready, eph, tow, ms_to_process, samples_per_code,
              nav_sol_period=500.0, elevation_mask=10.0, use_trop_corr=True, start_offset=68.802,
              c=299792458.0):
    """The measurement loop of postNavigate (postNavigation.py:159-301) for one recording.

    ``abs_sample[ch]``: absoluteSample series; ``prn[ch]``; ``sub_frame_start[ch]`` (0 for channels
    without a preamble); ``ready``: channel indices with a decoded ephemeris (readyChnList, :166);
    ``eph[prn-1]``: mapping with EPH_FIELDS; ``tow``: transmitTime of the first epoch (:168).
    Returns a dict of arrays with one column per measurement epoch."""
    n_ch = len(prn)
    sub_frame_start = np.asarray(sub_frame_start)
    ready = np.asarray(ready, dtype=int)
    prn = np.asarray(prn)
    n_ep = int(np.fix(ms_to_process - sub_frame_start.max()) / nav_sol_period)          # :199
    nan = np.nan
    out = dict(PRN=np.zeros((n_ch, n_ep)), el=nan * np.ones((n_ch, n_ep)), az=nan * np.ones((n_ch, n_ep)),
               rawP=nan * np.ones((n_ch, n_ep)), correctedP=nan * np.ones((n_ch, n_ep)),
               DOP=np.zeros((5, n_ep)), X=nan * np.ones(n_ep), Y=nan * np.ones(n_ep), Z=nan * np.ones(n_ep),
               dt=nan * np.ones(n_ep), latitude=nan * np.ones(n_ep), longitude=nan * np.ones(n_ep),
               height=nan * np.ones(n_ep), satPositions=nan * np.ones((n_ch, n_ep, 3)),
               satClkCorr=nan * np.ones((n_ch, n_ep)), n_epochs=n_ep)
    sat_elev = np.inf * np.ones(n_ch)                                        # :159
    transmit_time = tow                                                      # :168
    for m in range(n_ep):
        with np.errstate(invalid="ignore"):
            active = np.intersect1d((sat_elev >= elevation_mask).nonzero()[0], ready)   # :201
        out["PRN"][active, m] = prn[active]                                  # :203
        out["rawP"][:, m] = calculate_pseudoranges(abs_sample, sub_frame_start + nav_sol_period * m, active,
                                                   n_ch, samples_per_code, start_offset, c)   # :212-214
        sat_positions, sat_clk = satpos(transmit_time, prn[active], eph)     # :217
        out["satPositions"][active, m, :] = sat_positions.T
        out["satClkCorr"][active, m] = sat_clk
        if active.size > 3:                                                  # :222
            xyzdt, el, az, dop = least_square_pos(sat_positions, out["rawP"][active, m] + sat_clk * c, c,
                                                  use_trop_corr)             # :224-231
            out["el"][active, m] = el
            out["az"][active, m] = az
            out["DOP"][:, m] = dop
            out["X"][m], out["Y"][m], out["Z"][m], out["dt"][m] = xyzdt
            sat_elev = out["el"][:, m]                                       # :241
            out["correctedP"][active, m] = out["rawP"][active, m] + sat_clk * c + out["dt"][m]   # :243-245
            out["latitude"][m], out["longitude"][m], out["height"][m] = cart2geo(out["X"][m], out["Y"][m],
                                                                                out["Z"][m], 4)   # :249-254
        else:                                                                # :264-291
            out["DOP"][:, m] = 0.0
            out["az"][active, m] = nan
            out["el"][active, m] = nan
        transmit_time += nav_sol_period / 1000                               # :298
    return out


# ---------------------------------------------------------------------------------------------
# Ephemeris decoding (ephemeris.py:98-196): the host-side stage between the preamble search and the
# measurement loop.  Integer restatement on 0/1 arrays (the reference slices character strings).
# ---------------------------------------------------------------------------------------------
EPH_ALL = ("weekNumber", "accuracy", "health", "T_GD", "IODC", "t_oc", "a_f2", "a_f1", "a_f0", "IODE_sf2", "C_rs",
           "deltan", "M_0", "C_uc", "e", "C_us", "sqrtA", "t_oe", "C_ic", "omega_0", "C_is", "i_0", "C_rc", "omega",
           "omegaDot", "IODE_sf3", "iDot")                                    # ephemeris.py:191-194, in order


def _u(b):
    return int("".join(str(int(x)) for x in b), 2)                          # bin2dec, ephemeris.py:1-8


def _s(b):
    v = _u(b)                                                               # twosComp2dec, ephemeris.py:30-41
    return v - (1 << len(b)) if int(b[0]) == 1 else v


def ephemeris(bits, d30star):
    """ephemeris.py:98-196.  ``bits``: 1500 values 0/1 (five subframes from a subframe start), ``d30star``:
    the bit before them.  Returns (dict with EPH_ALL keys -- None for fields whose subframe is absent --, TOW)."""
    bits = [int(b) for b in bits]
    assert len(bits) >= 1500
    gps_pi = 3.1415926535898                                                 # :113
    d30 = int(d30star)
    out = dict.fromkeys(EPH_ALL)
    sf = None
    for i in range(5):
        sf = bits[300 * i:300 * (i + 1)]
        for j in range(10):                                                  # :122-127 checkPhase: data bits inverted by D30*
            if d30 == 1:
                for k in range(30 * j, 30 * j + 24):
                    sf[k] ^= 1
            d30 = sf[30 * j + 29]
        sid = _u(sf[49:52])                                                  # :133
        if sid == 1:                                                         # :139-150
            out.update(weekNumber=_u(sf[60:70]) + 1024, accuracy=_u(sf[72:76]), health=_u(sf[76:82]),
                       T_GD=_s(sf[195:204]) * 2 ** (-31), IODC=_u(sf[82:84] + sf[196:204]), t_oc=_u(sf[218:234]) * 2 ** 4,
                       a_f2=_s(sf[240:248]) * 2 ** (-55), a_f1=_s(sf[248:264]) * 2 ** (-43), a_f0=_s(sf[270:292]) * 2 ** (-31))
        elif sid == 2:                                                       # :152-163
            out.update(IODE_sf2=_u(sf[60:68]), C_rs=_s(sf[68:84]) * 2 ** (-5), deltan=_s(sf[90:106]) * 2 ** (-43) * gps_pi,
                       M_0=_s(sf[106:114] + sf[120:144]) * 2 ** (-31) * gps_pi, C_uc=_s(sf[150:166]) * 2 ** (-29),
                       e=_u(sf[166:174] + sf[180:204]) * 2 ** (-33), C_us=_s(sf[210:226]) * 2 ** (-29),
                       sqrtA=_u(sf[226:234] + sf[240:264]) * 2 ** (-19), t_oe=_u(sf[270:286]) * 2 ** 4)
        elif sid == 3:                                                       # :165-176
            out.update(C_ic=_s(sf[60:76]) * 2 ** (-29), omega_0=_s(sf[76:84] + sf[90:114]) * 2 ** (-31) * gps_pi,
                       C_is=_s(sf[120:136]) * 2 ** (-29), i_0=_s(sf[136:144] + sf[150:174]) * 2 ** (-31) * gps_pi,
                       C_rc=_s(sf[180:196]) * 2 ** (-5), omega=_s(sf[196:204] + sf[210:234]) * 2 ** (-31) * gps_pi,
                       omegaDot=_s(sf[240:264]) * 2 ** (-43) * gps_pi, IODE_sf3=_u(sf[270:278]),
                       iDot=_s(sf[278:292]) * 2 ** (-43) * gps_pi)
    tow = _u(sf[30:47]) * 6 - 30                                             # :190 (HOW of the fifth subframe)
    return out, tow
