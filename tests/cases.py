"""Seeded synthetic test cases shared by the golden generator, the CPU oracle tests and the
GPU parity tests.  Inputs are always regenerated from these specs (never stored)."""
import numpy as np

from softgnss_python_b200 import synth

N = 38192  # samplesPerCode at the reference's default fs


def _sats(lst, cn0=47.0):
    return [synth.SatSpec(p, d, c, cn0=k.get("cn0", cn0), bit_offset_ms=k.get("bo", 3 * p % 20),
                          carrier_phase=(0.137 * p) % 1.0)
            for (p, d, c, k) in [(x[0], x[1], x[2], x[3] if len(x) > 3 else {}) for x in lst]]


CASES = {
    # BASELINE.json config 1: default acquisition on an 11 ms recording, 8 satellites
    "acq_c1": dict(seed=1, ms=0, n_ms=11, sats=_sats([
        (1, 1500.0, 1000), (3, -3250.0, 12345), (7, -2500.0, 40), (11, 6200.0, 38000),
        (14, 250.0, 20000), (19, -6400.0, 5), (22, 4000.0, 38181), (31, -7000.0, 27001)], cn0=45.0)),
    # code phases around the second-peak window branches (acquisition.py:147-159); the
    # reference reports start+1 (appendix A.1-9), 37 is its IndexError and is avoided here
    "acq_edges": dict(seed=2, ms=0, n_ms=11, sats=_sats([
        (2, 0.0, 0), (5, 3000.0, 35), (9, -3000.0, 37), (12, 7000.0, N - 40),
        (17, -500.0, N - 39), (25, 500.0, N - 2)], cn0=50.0)),
    # acquisition + preRun + 300 ms of tracking on 4 channels out of 5 satellites
    "trk_small": dict(seed=3, ms=300, n_ms=303, settings=dict(numberOfChannels=4), sats=_sats([
        (4, 2100.0, 777), (8, -4300.0, 30011), (15, 5600.0, 15000, dict(cn0=50.0)),
        (21, -900.0, 38100, dict(cn0=44.0)), (30, 3333.0, 9000)], cn0=47.0)),
    # non-zero skipNumberOfBytes and a weak satellite near the detection threshold
    "trk_skip": dict(seed=4, ms=120, n_ms=125, settings=dict(numberOfChannels=3, skipNumberOfBytes=5000),
                     sats=_sats([(6, -1234.0, 100), (13, 4321.0, 22222),
                                 (27, 600.0, 31000, dict(cn0=39.0))], cn0=48.0)),
}


def build_recording(case):
    spec = synth.RecordingSpec(case["sats"], seed=case["seed"])
    data = synth.generate_cpu(spec, case["n_ms"] * N)
    return spec, data


class SettingsLike(object):
    """Minimal settings bag for the oracle (same attribute names as the reference)."""

    def __init__(self, **kw):
        from softgnss_python_b200.settings import Settings
        base = Settings(**kw)
        self.__dict__.update(base.__dict__)
        self.acqSatelliteList = range(1, 33)


def case_settings(case):
    from softgnss_python_b200.settings import Settings
    s = Settings(**case.get("settings", {}))
    s.msToProcess = float(case["ms"])
    return s


# ---------------------------------------------------------------------------------------------
# Bit-sync cases (SURVEY.md section 8(f) row 3): prompt in-phase series I_P built directly from an
# LNAV bit stream with integer-only noise (exactly reproducible from the seed on any numpy).
# ---------------------------------------------------------------------------------------------
BITSYNC_MS = 37000


def _hash_noise(seed, n):
    """Irwin-Hall noise as in softgnss_python_b200.synth: sum of the 8 bytes of splitmix64, mean removed."""
    from softgnss_python_b200 import synth
    i = np.arange(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h = synth._splitmix64(np.uint64(seed) + i * np.uint64(synth.GOLDEN))
    return h.view(np.uint8).reshape(-1, 8).sum(axis=1).astype(np.int64) - 1020     # sigma 209


def _lnav_ms(seed, n_subframes=9, first_sf_id=1):
    """+-1 per millisecond of `n_subframes` consecutive valid LNAV subframes."""
    from softgnss_python_b200 import navsynth
    rng = np.random.default_rng(seed)
    e = dict(sqrtA=5153.6, e=0.004 + 0.001 * (seed % 3), i_0=np.radians(55.0), omega_0=0.3 * (seed % 7) - 1.0,
             omega=-1.0, M_0=2.0, omegaDot=-8.0e-9, iDot=0.0, deltan=4.5e-9, t_oe=388800.0, weekNumber=2100,
             IODE=int(rng.integers(1, 255)))
    bits01 = navsynth.encode_stream(navsynth.quantize_ephemeris(e), first_sf_id, 388800 - 6, n_subframes)
    return np.repeat(bits01.astype(np.int64) * 2 - 1, 20), bits01


#  name: (first subframe boundary in ms, amplitude, noise scale, polarity, kind)
BITSYNC_CHANNELS = [
    dict(name="clean", boundary=3655, amp=4000, noise=6, pol=1),
    dict(name="inverted", boundary=977, amp=4000, noise=6, pol=-1),
    dict(name="random", boundary=0, amp=4000, noise=6, pol=1, random_bits=True),
    dict(name="noisy", boundary=2222, amp=430, noise=1, pol=1),             # ~2 % of the ms have the wrong sign
    dict(name="tlm_parity_broken", boundary=1500, amp=4000, noise=6, pol=1, flip_bit=12),   # first valid = +6000
    dict(name="zeros", boundary=5999, amp=3000, noise=1, pol=-1, integer_ties=True),         # exact zeros -> -1
    dict(name="late", boundary=41, amp=4000, noise=6, pol=1),
    dict(name="weak", boundary=4321, amp=120, noise=1, pol=1),              # sign errors ~28 %: nothing found
]
BITSYNC_EARLY = dict(name="early", boundary=20, amp=4000, noise=6, pol=1)   # the reference crashes on this one


def build_bitsync_channel(ch, seed):
    ms, bits01 = _lnav_ms(seed)
    if ch.get("random_bits"):
        rng_bits = (_hash_noise(seed + 99, len(bits01)) & 1) * 2 - 1
        ms = np.repeat(rng_bits, 20)
    if "flip_bit" in ch:                       # corrupt one data bit of the first complete subframe's TLM word
        b = 300 + ch["flip_bit"]
        ms = ms.copy()
        ms[20 * b:20 * b + 20] *= -1
    w0 = 6000 - ch["boundary"]                 # subframe 2 of the stream starts at ms `boundary` of the window
    sig = ms[w0:w0 + BITSYNC_MS] * ch["amp"] * ch["pol"]
    noise = _hash_noise(seed, BITSYNC_MS) * ch["noise"]
    ip = (sig + noise).astype(np.float64)
    if ch.get("integer_ties"):
        ip[::97] = 0.0                          # I_P == 0 counts as a -1 (postNavigation.py:569)
        b0 = ch["boundary"] + 20 * 70           # one data bit whose 20 ms sum is exactly 0 -> bit 0 (:131)
        ip[b0:b0 + 20] = np.tile([500.0, -500.0], 10)
    else:
        ip += 0.25                              # keep the 20 ms sums away from exact zero
    return ip


def build_bitsync_case(channels=None, seed0=500):
    channels = BITSYNC_CHANNELS if channels is None else channels
    return [build_bitsync_channel(ch, seed0 + i) for i, ch in enumerate(channels)]


# ---------------------------------------------------------------------------------------------
# Pseudorange cases (SURVEY.md section 8(f) row 4, first half)
# ---------------------------------------------------------------------------------------------
def build_pseudo_case(n_ch=8, ms=2000, n_epochs=6, seed=77):
    """absoluteSample-like series (integer-valued float64, one code period per ms with a slow drift),
    msOfTheSignal per epoch/channel and channel lists of varying size (including an empty one)."""
    noise = _hash_noise(seed, n_ch * ms).reshape(n_ch, ms)
    start = 1000 + 4000 * np.arange(n_ch)[:, None] + (_hash_noise(seed + 1, n_ch)[:, None] % 977)
    drift = np.cumsum(38192 + (noise % 3) - 1, axis=1)
    abs_sample = (start + drift).astype(np.float64)
    sub = 40 + (np.abs(_hash_noise(seed + 2, n_ch)) % 900)                     # "subFrameStart" per channel
    ms_index = (sub[None, :] + 150 * np.arange(n_epochs)[:, None]).astype(np.int32)
    active = np.ones((n_epochs, n_ch), dtype=np.uint8)
    active[1, [2, 5]] = 0
    active[2, :] = 0
    active[2, [0, 3, 4, 7]] = 1
    active[3, :] = 0                                                           # empty list: all inf - inf = nan
    active[4, 1:] = 0                                                          # a single channel
    return abs_sample, ms_index, active


# ---------------------------------------------------------------------------------------------
# Navigation-solution cases (SURVEY.md section 8(f) row 4, second half).  The float inputs (ephemerides,
# polynomial coefficients of the code-period arrival samples) are stored in tests/golden/nav.npz by
# tests/golden/make_golden_nav.py; the absoluteSample series are expanded from them with integer arithmetic.
# ---------------------------------------------------------------------------------------------
NAV_MS = 37000
NAV_FIELDS = ("t_oc", "a_f2", "a_f1", "a_f0", "T_GD", "sqrtA", "t_oe", "deltan", "M_0", "e", "omega",
              "C_uc", "C_us", "C_rc", "C_rs", "i_0", "iDot", "C_ic", "C_is", "omega_0", "omegaDot")


def nav_abs_sample(coef, n_code=38192, ms=NAV_MS):
    """coef int64 [C][4] = (b, k0, p1, p2): absoluteSample[i] = b + k*n_code + ((p1*k + p2*k*k) >> 40), k = i - k0."""
    coef = np.asarray(coef, dtype=np.int64)
    i = np.arange(ms, dtype=np.int64)[None, :]
    k = i - coef[:, 1:2]
    return (coef[:, 0:1] + k * n_code + ((coef[:, 2:3] * k + coef[:, 3:4] * k * k) >> 40)).astype(np.float64)


def load_nav_cases():
    """List of dicts (one per golden recording): inputs of the measurement loop + the reference's outputs."""
    import os
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "nav.npz"))
    cases = []
    for r in range(int(z["n_cases"])):
        g = lambda name: z["c%d_%s" % (r, name)]
        eph_arr = g("eph_arr")                                                # [C][21] in NAV_FIELDS order
        prn = g("prn")
        eph = [None] * 32
        for c in range(len(prn)):
            eph[int(prn[c]) - 1] = dict(zip(NAV_FIELDS, eph_arr[c]))
        cases.append(dict(coef=g("coef"), prn=prn, eph_arr=eph_arr, eph=eph, sub_frame_start=g("sub_frame_start"),
                          ready=g("ready"), tow=float(g("tow")), elevation_mask=float(g("elevation_mask")),
                          use_trop_corr=bool(g("use_trop_corr")), rx=g("rx"),
                          ref={k: g("ref_" + k) for k in ("rawP", "el", "az", "correctedP", "DOP", "X", "Y", "Z", "dt",
                                                          "latitude", "longitude", "height", "PRN")}))
    return cases


# ---------------------------------------------------------------------------------------------
# Ephemeris-decoding cases: 1501 hard bits (bit 0 = D30* of the word before the first subframe)
# ---------------------------------------------------------------------------------------------
def build_ephemeris_cases():
    """uint8 [n][1501].  Rows 0-4: LNAV streams of navsynth's encoder (one per starting subframe ID, alternating
    polarity of the preceding bit); rows 5-9: hash-random bits with the subframe IDs forced to 1..5 in rotation, so
    that every field (clock terms, T_GD, IODC, signs) takes arbitrary values."""
    from softgnss_python_b200 import navsynth
    rows = []
    for k in range(5):
        e = dict(sqrtA=5153.6 + 0.1 * k, e=0.002 + 0.001 * k, i_0=np.radians(54.0 + k), omega_0=-2.5 + 1.2 * k,
                 omega=2.9 - 1.4 * k, M_0=-3.0 + 1.5 * k, omegaDot=-8.0e-9 * (k - 2), iDot=1e-10 * (k - 2), deltan=1.5e-9 * (k - 1),
                 t_oe=388800.0 + 16 * k, weekNumber=2100 + k, IODE=10 + k, C_rs=-50.0 + 30 * k, C_rc=200.0 - 90 * k,
                 C_uc=1e-6 * (k - 2), C_us=-2e-6 * (k - 1), C_ic=5e-8 * (k - 3), C_is=-4e-8 * k)
        bits = navsynth.encode_stream(navsynth.quantize_ephemeris(e), 1 + k, 388800 - 6, 7)
        rows.append(bits[299:1800].astype(np.uint8))          # last bit of the first subframe + the five after it
    for k in range(5):
        b = (_hash_noise(900 + k, 1501) & 1).astype(np.uint8)
        for i in range(5):
            sid = (k + i) % 5 + 1
            base = 1 + 300 * i
            inv = b[base + 29]                                 # D30 of word 1 decides the inversion of word 2
            for j, bit in enumerate(((sid >> 2) & 1, (sid >> 1) & 1, sid & 1)):
                b[base + 49 + j] = bit ^ inv
        rows.append(b)
    return np.stack(rows)


# ---------------------------------------------------------------------------------------------
# Whole downstream chain (preamble search -> ephemeris decoding -> measurement loop) on a synthetic tracking
# result: I_P carries the LNAV stream of each satellite, absoluteSample the geometry of navsynth.build_scenario.
# ---------------------------------------------------------------------------------------------
def build_chain_case(seed=2, ms=NAV_MS, n_code=38192, fs=38.192e6, first_boundary_ms=5200, drop=()):
    """Returns (track float64 [C, 13, ms], prn int64 [C], truth).  Channels in ``drop`` carry noise only."""
    from softgnss_python_b200 import navsynth
    _, truth = navsynth.build_scenario(seed=seed)
    n_ch = len(truth["prn"])
    track = np.zeros((n_ch, 13, ms))
    rho_min = min(truth["range"])
    k = np.arange(ms, dtype=np.float64)
    for c in range(n_ch):
        e = truth["eph"][c]
        q = navsynth.quantize_ephemeris(dict(e, weekNumber=2100, IODE=40 + c))
        sid = 1 + (c % 5)                                                     # subframe that starts at `tow`
        bits01 = navsynth.encode_stream(q, (sid - 2) % 5 + 1, truth["tow"] - 6, 8)
        k0 = first_boundary_ms + (3 * c) % 7                                  # index of that boundary in the series
        per_ms = np.repeat(bits01.astype(np.float64) * 2 - 1, 20)            # stream starts one subframe (6000 ms) earlier
        idx = np.arange(ms) - k0 + 6000
        ip = np.where((idx >= 0) & (idx < per_ms.size), per_ms[np.clip(idx, 0, per_ms.size - 1)], 1.0)
        noise = _hash_noise(seed * 100 + c, ms) * 2.0
        track[c, 3] = (0.0 if c in drop else 3000.0) * ip * (1 if c % 2 else -1) + noise + 0.25
        s = []
        for kk in (0.0, 18000.0, 36000.0):
            rho, _ = navsynth.geometric_range(e, truth["tow"] + kk * 1e-3, truth["rx"])
            s.append((rho - rho_min) / navsynth.C * fs)
        p2 = ((s[2] - s[0]) - 2 * (s[1] - s[0])) / (2 * 18000.0 ** 2)
        p1 = (s[1] - s[0]) / 18000.0 - p2 * 18000.0
        kr = k - k0
        track[c, 0] = np.round(first_boundary_ms * n_code + s[0] + kr * n_code + p1 * kr + p2 * kr * kr)
    return track, np.array(truth["prn"], dtype=np.int64), truth


def oracle_chain(track, prn, settings_kw, samples_per_code=38192):
    """The same chain with the oracle: find_preambles, nav_bits, ephemeris, nav_solve.  Returns (first, nav dict | None).
    ``samples_per_code``: settings.samplesPerCode of the rate the absoluteSample series was made for."""
    from oracle import gnss_oracle as orc
    n_ch, _, ms = track.shape
    first, active = orc.find_preambles([track[c, 3] for c in range(n_ch)])
    eph, tow, ready = [None] * 32, None, []
    for ch in active:
        if first[ch] + 30000 > ms:
            continue
        b = orc.nav_bits(track[ch, 3], int(first[ch]))
        e, tow = orc.ephemeris(b[1:], b[0])
        eph[int(prn[ch]) - 1] = e
        if e["IODC"] is not None and e["IODE_sf2"] is not None and e["IODE_sf3"] is not None:
            ready.append(ch)
    if len(ready) < 4:
        return first, None
    return first, orc.nav_solve([track[c, 0] for c in range(n_ch)], prn, first, ready, eph, tow, float(ms), samples_per_code,
                                  **settings_kw)
