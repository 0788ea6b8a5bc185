"""Per-window C/N0 (variance-summing method) and carrier-lock detection of tracked channels (sgx_track_quality,
csrc/sgx_quality.cu) against the float64 oracle (tests/quality_oracle.py) and against the truth of the
synthetic recording generator.

The parity tests run on two backends, as in test_gpu_track_matrix.py:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).  The emulator treats every
            pointer as device memory unless SGX_EMUL_HOST is set, so there host and device operands can only be
            switched together.
The tests that track a recording first need the device tracker and run on the gpu backend only.
"""
import ctypes
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
SGX_ERR_ARG = -2
T = 0.001


def _qs(W, acc_time=T, cn0_min=30.0, pll_min=0.5):
    from softgnss_python_b200 import _native
    return _native.SgxQualitySettings(acc_time=acc_time, cn0_min=cn0_min, pll_lock_min=pll_min, window_ms=W)


class Backend(object):
    """One library (device build or CPU emulator) and where it finds its operands."""

    def __init__(self, name, lib):
        self.name = name
        self.lib = lib

    def quality(self, i_p, q_p, stride, n, ms, ms_done, qs, host_in=True, host_out=True):
        """i_p, q_p: float64 host arrays whose rows are `stride` apart (views into one buffer are fine).  Returns
        (rc, cn0, pll_lock, locked) as host arrays [n, ms // W]."""
        n_win = ms // qs.window_ms if qs.window_ms >= 2 else 0
        shape = (n, max(n_win, 1))
        host_env = os.environ.pop("SGX_EMUL_HOST", None)
        try:
            if self.name == "gpu":
                import torch
                if host_in:
                    a_i, a_q = i_p.ctypes.data, q_p.ctypes.data
                    keep = (i_p, q_p)
                else:
                    keep = (torch.from_numpy(np.ascontiguousarray(i_p)).cuda(),
                            torch.from_numpy(np.ascontiguousarray(q_p)).cuda())
                    a_i, a_q = keep[0].data_ptr(), keep[1].data_ptr()
                if host_out:
                    outs = [np.full(shape, -1.0), np.full(shape, -1.0), np.full(shape, 7, dtype=np.uint8)]
                else:
                    outs = [torch.full(shape, -1.0, dtype=torch.float64, device="cuda"),
                            torch.full(shape, -1.0, dtype=torch.float64, device="cuda"),
                            torch.full(shape, 7, dtype=torch.uint8, device="cuda")]
                rc = self.lib.track_quality(a_i, a_q, stride, n, ms, ms_done, qs, *outs)
                if not host_out:
                    torch.cuda.synchronize()
                    outs = [o.cpu().numpy() for o in outs]
                del keep
            else:
                assert host_in == host_out, "the emulator switches host / device operands together"
                if host_in:
                    os.environ["SGX_EMUL_HOST"] = "1"
                outs = [np.full(shape, -1.0), np.full(shape, -1.0), np.full(shape, 7, dtype=np.uint8)]
                rc = self.lib.track_quality(i_p.ctypes.data, q_p.ctypes.data, stride, n, ms, ms_done, qs, *outs)
        finally:
            os.environ.pop("SGX_EMUL_HOST", None)
            if host_env is not None:
                os.environ["SGX_EMUL_HOST"] = host_env
        return (rc,) + tuple(o[:, :n_win] for o in outs)

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
    for k in ("SGX_TRK_KERNEL", "SGX_TRK_STAGE", "SGX_TRK_CHUNK_MS", "SGX_EMUL_HOST"):
        monkeypatch.delenv(k, raising=False)


# ---------------------------------------------------------------------------------------------- oracle comparison
def _oracle(i, q, W, done, cn0_min=30.0, pll_min=0.5):
    """Expected (cn0, pll_lock, locked) of one row from the oracle, windows past `done` invalid."""
    from tests import quality_oracle as orc
    cn0, pll = orc.cno_vsm(i, q, W, T), orc.pll_lock(i, q, W)
    with np.errstate(invalid="ignore"):
        locked = ((cn0 >= cn0_min) & (pll >= pll_min)).astype(np.uint8)
    invalid = (np.arange(len(cn0)) + 1) * W > done
    cn0[invalid], pll[invalid], locked[invalid] = np.nan, np.nan, 0
    return cn0, pll, locked


def _well_posed(i, q, W):
    """Windows whose Zm^2 - Zv is at least 1e-6 Zm^2: there the NaN decision and cn0 do not hinge on rounding."""
    n = len(i) // W
    z = (i[:n * W] ** 2 + q[:n * W] ** 2).reshape(n, W)
    zm, zv = z.mean(axis=1), z.var(axis=1, ddof=1)
    return zm ** 2 - zv >= 1e-6 * zm ** 2


def check_against_oracle(i_rows, q_rows, W, ms_done, got, label, cn0_min=30.0, pll_min=0.5):
    """got = (cn0, pll, locked) [n, n_win]: NaN pattern and cn0 within 1e-9 dB on well-posed windows, pll_lock
    within 1e-12 everywhere, locked identical wherever neither value is within 1e-9 of its threshold."""
    cn0, pll, locked = got
    for c in range(len(i_rows)):
        ec, ep, el = _oracle(i_rows[c], q_rows[c], W, ms_done[c], cn0_min, pll_min)
        lab = "%s row %d W=%d" % (label, c, W)
        wp = _well_posed(i_rows[c], q_rows[c], W)
        assert np.array_equal(np.isnan(cn0[c][wp]), np.isnan(ec[wp])), lab + " cn0 NaN pattern"
        fin = wp & np.isfinite(ec) & np.isfinite(cn0[c])
        if fin.any():
            d = np.abs(cn0[c][fin] - ec[fin]).max()
            assert d <= 1e-9, "%s: |d cn0| = %.3g dB" % (lab, d)
        assert np.array_equal(np.isnan(pll[c]), np.isnan(ep)), lab + " pll_lock NaN pattern"
        fp = np.isfinite(ep)
        if fp.any():
            d = np.abs(pll[c][fp] - ep[fp]).max()
            assert d <= 1e-12, "%s: |d pll_lock| = %.3g" % (lab, d)
        with np.errstate(invalid="ignore"):
            clear = ~(np.abs(ec - cn0_min) <= 1e-9) & ~(np.abs(ep - pll_min) <= 1e-9)
        assert np.array_equal(locked[c][clear], el[clear]), lab + " locked"
        invalid = (np.arange(cn0.shape[1]) + 1) * W > ms_done[c]
        assert np.isnan(cn0[c][invalid]).all() and np.isnan(pll[c][invalid]).all() and (locked[c][invalid] == 0).all()


MS = 3517                      # not a multiple of any W below
WINDOWS = (2, 20, 40, 1000)
CN0S = (25.0, 30.0, 35.0, 40.0, 45.0, 50.0, 55.0)


def _synthetic_rows(ms=MS, seed=3):
    """float64 prompt rows [n, ms]: a carrier at each C/N0 of CN0S with nav-bit flips, phase wander and unit-variance
    Gaussian noise per component (scaled by 1000, roughly the tracker's magnitude); noise only; all zeros; constant
    power (I, Q) in {(3, 4), (5, 0), (0, -5), (-4, 3)} so that Z = 25 exactly and Zv = 0."""
    rng = np.random.default_rng(seed)
    rows_i, rows_q = [], []
    for cn in CN0S:
        a = np.sqrt(2 * 10 ** (cn / 10) * T)
        ph = rng.uniform(0, 2 * np.pi) + np.cumsum(rng.normal(0, 0.02, ms))
        bits = np.repeat(rng.choice([-1.0, 1.0], ms // 20 + 1), 20)[:ms]
        rows_i.append(1000 * (a * bits * np.cos(ph) + rng.normal(0, 1, ms)))
        rows_q.append(1000 * (a * bits * np.sin(ph) + rng.normal(0, 1, ms)))
    rows_i.append(1000 * rng.normal(0, 1, ms))
    rows_q.append(1000 * rng.normal(0, 1, ms))
    rows_i.append(np.zeros(ms))
    rows_q.append(np.zeros(ms))
    pat = np.array([(3, 4), (5, 0), (0, -5), (-4, 3)], dtype=np.float64)[rng.integers(0, 4, ms)]
    rows_i.append(pat[:, 0].copy())
    rows_q.append(pat[:, 1].copy())
    return np.stack(rows_i), np.stack(rows_q)


def _strided(i_rows, q_rows, pad=5):
    """The rows in one buffer laid out like sgx_track's output, [n][2][ms + pad] with NaN padding, so a kernel that
    reads past ms or ignores the stride sees NaN.  Returns (buffer, i_p view, q_p view, stride)."""
    n, ms = i_rows.shape
    stride = 2 * (ms + pad)
    buf = np.full((n, 2, ms + pad), np.nan)
    buf[:, 0, :ms] = i_rows
    buf[:, 1, :ms] = q_rows
    flat = buf.reshape(-1)
    return buf, flat[0:], flat[ms + pad:], stride


def _ragged_done(n, ms, W):
    """ms_done per row: all, none, one short of all, a window edge exactly, and values in between."""
    base = [ms, 0, ms - 1, (ms // W) * W, ms // 2, 1, W - 1, W, 2 * W + 1, ms]
    return np.array([min(max(b, 0), ms) for b in (base * (n // len(base) + 1))[:n]], dtype=np.int32)


@pytest.mark.parametrize("W", WINDOWS)
def test_parity_with_oracle(backend, W):
    """Signal plus noise at 25 .. 55 dB-Hz, noise only, all zeros and constant power, read through a row stride,
    with all periods valid and with a ragged ms_done."""
    i_rows, q_rows = _synthetic_rows()
    n = len(i_rows)
    buf, ip, qp, stride = _strided(i_rows, q_rows)
    for done, label in ((None, "all ms"), (_ragged_done(n, MS, W), "ragged ms_done")):
        rc, cn0, pll, locked = backend.quality(ip, qp, stride, n, MS, done, _qs(W))
        assert rc == 0, backend.last_error()
        assert cn0.shape == (n, MS // W)
        d = np.full(n, MS) if done is None else done
        check_against_oracle(i_rows, q_rows, W, d, (cn0, pll, locked), "%s %s" % (backend.name, label))
    # the special rows: noise-only windows are often undefined; zero and constant-power rows always are
    rc, cn0, pll, locked = backend.quality(ip, qp, stride, n, MS, None, _qs(W))
    assert np.isnan(cn0[-2]).all() and np.isnan(pll[-2]).all() and (locked[-2] == 0).all()
    assert np.isnan(cn0[-1]).all() and (locked[-1] == 0).all()
    assert np.isfinite(cn0[len(CN0S) - 1]).all()                  # 55 dB-Hz: defined everywhere


def test_thresholds_and_acc_time(backend):
    """Non-default thresholds and accumulation time reach the kernel: cn0 moves by 10 log10(ratio of T), and the
    locked flags follow the thresholds given."""
    i_rows, q_rows = _synthetic_rows(ms=800, seed=5)
    n = len(i_rows)
    ip, qp = np.ascontiguousarray(i_rows), np.ascontiguousarray(q_rows)
    rc, c1, p1, l1 = backend.quality(ip, qp, 800, n, 800, None, _qs(40))
    assert rc == 0
    rc, c2, p2, l2 = backend.quality(ip, qp, 800, n, 800, None, _qs(40, acc_time=0.002, cn0_min=38.0, pll_min=0.9))
    assert rc == 0
    assert np.array_equal(p1, p2, equal_nan=True)
    ok = np.isfinite(c1)
    assert np.array_equal(ok, np.isfinite(c2))
    assert np.abs((c1[ok] - c2[ok]) - 10 * np.log10(2.0)).max() < 1e-9
    check_against_oracle(i_rows, q_rows, 40, np.full(n, 800), (c2 + 10 * np.log10(2.0), p2, l2), backend.name,
                         cn0_min=38.0 + 10 * np.log10(2.0), pll_min=0.9)


def test_deterministic_and_operand_kinds(backend):
    """Two runs, host vs device inputs and host vs device outputs give bit-identical results."""
    i_rows, q_rows = _synthetic_rows(ms=1234, seed=9)
    n = len(i_rows)
    buf, ip, qp, stride = _strided(i_rows, q_rows)
    done = _ragged_done(n, 1234, 40)
    kinds = [(True, True), (False, False)] + ([(True, False), (False, True)] if backend.name == "gpu" else [])
    runs = []
    for host_in, host_out in kinds + kinds[:1]:
        rc, cn0, pll, locked = backend.quality(ip, qp, stride, n, 1234, done, _qs(40), host_in, host_out)
        assert rc == 0, backend.last_error()
        runs.append((cn0, pll, locked))
    ref = runs[0]
    for (host_in, host_out), got in zip(kinds + kinds[:1], runs):
        for a, b in zip(got, ref):
            assert a.tobytes() == b.tobytes(), "host_in=%s host_out=%s" % (host_in, host_out)


def test_invalid_arguments(backend):
    i_rows, q_rows = _synthetic_rows(ms=200, seed=1)
    n = len(i_rows)
    ip, qp = np.ascontiguousarray(i_rows), np.ascontiguousarray(q_rows)
    for qs in (_qs(1), _qs(0), _qs(-40), _qs(40, acc_time=0.0), _qs(40, acc_time=-1e-3),
               _qs(40, acc_time=float("inf")), _qs(40, acc_time=float("nan"))):
        rc = backend.quality(ip, qp, 200, n, 200, None, qs)[0]
        assert rc == SGX_ERR_ARG, (qs.window_ms, qs.acc_time)
    assert backend.quality(ip, qp, 199, n, 200, None, _qs(40))[0] == SGX_ERR_ARG               # stride < ms
    for bad in (-1, 201):
        done = np.full(n, 100, dtype=np.int32)
        done[3] = bad
        assert backend.quality(ip, qp, 200, n, 200, done, _qs(40))[0] == SGX_ERR_ARG
    out = [np.zeros((n, 5)), np.zeros((n, 5)), np.zeros((n, 5), dtype=np.uint8)]
    L = backend.lib
    assert L.track_quality(None, qp, 200, n, 200, None, _qs(40), *out) == SGX_ERR_ARG
    assert L.track_quality(ip, None, 200, n, 200, None, _qs(40), *out) == SGX_ERR_ARG
    assert L.track_quality(ip, qp, 200, n, 200, None, _qs(40), None, out[1], out[2]) == SGX_ERR_ARG
    assert L.track_quality(ip, qp, 200, n, 200, None, _qs(40), out[0], out[1], None) == SGX_ERR_ARG
    # fewer periods than one window: nothing to do, and that is not an error
    rc, cn0, pll, locked = backend.quality(ip, qp, 200, n, 39, None, _qs(40))
    assert rc == 0 and cn0.shape == (n, 0)
    if backend.name == "gpu":                                  # mixed host / device operands
        import torch
        dq = torch.from_numpy(qp).cuda()
        assert L.track_quality(ip, dq, 200, n, 200, None, _qs(40), *out) == SGX_ERR_ARG
        dc = torch.zeros((n, 5), dtype=torch.float64, device="cuda")
        assert L.track_quality(ip, qp, 200, n, 200, None, _qs(40), dc, out[1], out[2]) == SGX_ERR_ARG
        assert L.track_quality(ip, qp, 200, n, 200, None, _qs(40), out[0], dc, out[2]) == SGX_ERR_ARG


# ---------------------------------------------------------------------------------------------- on tracked channels
FS = 38.192e6


def _track_case(ms, sats, extra, seed, n_rec=1):
    """A recording at 38.192 MHz with `sats` (synth.SatSpec), on the device, and channels taken from the truth as
    test_gpu_track_matrix._case builds them (carrier 30 Hz off, code phase + 1), followed by `extra` channels
    (prn, freq, codePhase).  n_rec recordings: the same channels on recordings with seeds seed, seed + 1, ...
    Returns (dev [n_rec, stride] int8 tensor, total samples, settings, channel recarray, RecordingSpec of seed)."""
    import torch
    from softgnss_python_b200 import _native, synth
    from softgnss_python_b200.settings import Settings
    s = Settings(numberOfChannels=len(sats) + len(extra), msToProcess=float(ms))
    n = s.samplesPerCode
    total = (ms + 3) * n
    stride = (total + 15) // 16 * 16
    dev = torch.zeros((n_rec, stride), dtype=torch.int8, device="cuda")
    specs = [synth.RecordingSpec(sats, fs=FS, f_if=FS / 4, seed=seed + r) for r in range(n_rec)]
    sp, bits = _native.make_synth_specs(specs)
    L = _native.lib()
    L.synth(dev, stride, total, 0, sp, bits, synth.cos_lut(), _native.ca_chips_int8(), 0)
    torch.cuda.synchronize()
    spec = specs[0]
    prn = [x.prn for x in sats] + [e[0] for e in extra]
    freq = [spec.true_carr_freq(i) - 30.0 for i in range(len(sats))] + [e[1] for e in extra]
    cph = [float((x.code_phase + 1) % n) for x in sats] + [float(e[2]) for e in extra]
    ch = np.rec.fromarrays([np.array(prn, dtype=np.int64), np.array(freq), np.array(cph), ['T'] * len(prn)],
                           names="PRN,acquiredFreq,codePhase,status")
    return dev, total, s, ch, spec


def _two_sats():
    from softgnss_python_b200 import synth
    return [synth.SatSpec(4, 2300.0, 5100, cn0=44.0, bit_offset_ms=6),
            synth.SatSpec(17, -3900.0, 30011, cn0=36.0, bit_offset_ms=13)]


@pytest.mark.gpu
def test_in_place_on_track_output():
    """track_quality_batch on a device-resident [R, C, 13, ms] tensor reads I_P / Q_P through the field strides; the
    result equals the oracle applied to out[:, :, 3] and out[:, :, 7] copied to the host."""
    import torch
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import FIELDS, track_batch, track_quality_batch
    ms = 600
    dev, total, s, ch, _ = _track_case(ms, _two_sats(), [(9, 9.548e6 + 1000.0, 777.0), (0, 0.0, 0.0)], seed=21,
                                       n_rec=2)
    out = torch.zeros((2, len(ch), len(FIELDS), ms), dtype=torch.float64, device="cuda")
    rc, out, done = track_batch(dev, [total, total], [ch, ch], s, out=out)
    assert rc == 0
    assert (done[:, :3] == ms).all() and (done[:, 3] == 0).all()
    res = track_quality_batch(out, done, Settings())
    torch.cuda.synchronize()
    assert res["cn0"].is_cuda and tuple(res["cn0"].shape) == (2, len(ch), ms // 40)
    assert np.array_equal(res["index"], 40 * np.arange(1, ms // 40 + 1))
    host = out.cpu().numpy()
    i_p, q_p = host[:, :, FIELDS.index("I_P")], host[:, :, FIELDS.index("Q_P")]
    got = [res[k].cpu().numpy().reshape(-1, ms // 40) for k in ("cn0", "pllLock", "locked")]
    check_against_oracle(i_p.reshape(-1, ms), q_p.reshape(-1, ms), 40, done.reshape(-1), got, "in place")
    # the numpy path on the same result is bit-identical
    res_np = track_quality_batch(host, done, Settings())
    for k, g in zip(("cn0", "pllLock", "locked"), got):
        assert res_np[k].reshape(g.shape).tobytes() == g.tobytes(), k


TRUTH_MS = 3000
TRUTH_CN0 = (35.0, 40.0, 45.0, 50.0)
ABSENT_PRN = 9


def _truth_sats():
    from softgnss_python_b200 import synth
    return [synth.SatSpec(3, 3100.0, 1200, cn0=35.0, bit_offset_ms=2),
            synth.SatSpec(11, -1800.0, 14000, cn0=40.0, bit_offset_ms=9),
            synth.SatSpec(19, 600.0, 25555, cn0=45.0, bit_offset_ms=15),
            synth.SatSpec(27, -4400.0, 33333, cn0=50.0, bit_offset_ms=19)]


def _generated_cn0(spec, i):
    """C/N0 of satellite i as the generator's integers realise it: carrier amplitude A = amp / 256 LSB against
    the hash noise (sigma = noise_k * 209.0215 / 2^22 LSB) plus the output rounding (1/12 LSB^2)."""
    from softgnss_python_b200.synth import HASH_SIGMA, OUT_SHIFT
    a = spec.amp[i] / 256.0
    var = (spec.noise_k * HASH_SIGMA / 2.0 ** OUT_SHIFT) ** 2 + 1.0 / 12
    return 10 * np.log10(a * a * spec.fs / (4 * var))


# The same recording through the float64 oracle tracker (oracle.gnss_oracle.track) and the oracle VSM on the CPU,
# W = 40, windows 5 .. 74:
#   PRN                        3        11       19       27      | absent PRN 9
#   truth (generator), dB-Hz   35.01    39.96    45.01    49.99   |
#   median cn0 - truth, dB     -1.03    +0.11    +0.00    -0.41   | median cn0 28.3, 27 of 70 windows NaN
#   per-window std, dB         1.98     1.45     1.00     1.26    |
#   median pll_lock            0.678    0.882    0.962    0.987   | -0.020
#   windows locked             60/70    70/70    70/70    70/70   | 0/70
# Noise alone bounds pll_lock by (C/N0 T) / (C/N0 T + 1): 0.76 at 35 dB-Hz, 0.91 at 40 dB-Hz; the loop's phase
# jitter lowers it further.  At 35 dB-Hz 6 windows fall below pll_lock 0.5 and 4 below 30 dB-Hz (none both), so
# the tracker locks 86 % of them there, and the bound is 80 %.
LOCKED_SHARE_35 = 0.8


@pytest.mark.gpu
def test_ground_truth_from_synthesiser():
    """Four satellites at 35 .. 50 dB-Hz, a channel on a PRN the recording does not contain and an idle channel,
    tracked for 3000 ms.  From window 5 on (after 200 ms of pull-in): the median C/N0 of each satellite is within
    1 dB of the generator's (1.5 dB at 35 dB-Hz); every window is locked at >= 40 dB-Hz and >= 80 % at 35 dB-Hz; the
    absent PRN has |median pll_lock| < 0.2 and <= 2 % of its windows locked; the idle channel is all NaN and 0."""
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import track_batch, track_quality_batch
    sats = _truth_sats()
    dev, total, s, ch, spec = _track_case(TRUTH_MS, sats, [(ABSENT_PRN, 9.548e6 + 1500.0, 4321.0), (0, 0.0, 0.0)],
                                          seed=77)
    rc, out, done = track_batch(dev, [total], [ch], s)
    assert rc == 0
    assert (done[0, :5] == TRUTH_MS).all() and done[0, 5] == 0
    res = track_quality_batch(out, done, Settings())
    cn0, pll, locked = res["cn0"][0], res["pllLock"][0], res["locked"][0]
    report = []
    for i, x in enumerate(sats):
        truth = _generated_cn0(spec, i)
        assert abs(truth - x.cn0) < 0.05
        med = np.nanmedian(cn0[i, 5:])
        tol = 1.5 if x.cn0 < 37 else 1.0
        report.append("PRN %d truth %.2f median %.2f locked %.3f" % (x.prn, truth, med, locked[i, 5:].mean()))
        assert abs(med - truth) <= tol, report[-1]
        if x.cn0 >= 40:
            assert locked[i, 5:].all(), report[-1]
        else:
            assert locked[i, 5:].mean() >= LOCKED_SHARE_35, report[-1]
    a = len(sats)
    assert abs(np.nanmedian(pll[a, 5:])) < 0.2, pll[a, 5:]
    assert locked[a, 5:].mean() <= 0.02
    assert np.isnan(cn0[a + 1]).all() and np.isnan(pll[a + 1]).all() and (locked[a + 1] == 0).all()
    print("; ".join(report))


@pytest.mark.gpu
def test_short_recording():
    """A recording cut so that tracking stops with the short-recording error: windows that end at or before a
    channel's ms_done are bit-identical to the full-length run, later windows are NaN, NaN, 0."""
    from softgnss_python_b200._native import SGX_ERR_SHORT
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import track_batch, track_quality_batch
    ms = 500
    dev, total, s, ch, _ = _track_case(ms, _two_sats(), [], seed=31)
    rc, full, done_full = track_batch(dev, [total], [ch], s)
    assert rc == 0 and (done_full == ms).all()
    cut = 331 * s.samplesPerCode + 5000
    rc, part, done = track_batch(dev, [cut], [ch], s)
    assert rc == SGX_ERR_SHORT
    assert (done < ms).all() and (done > 200).all()
    qs = Settings(CNoVSMinterval=20)
    a = track_quality_batch(full, done_full, qs)
    b = track_quality_batch(part, done, qs)
    for c in range(len(ch)):
        k = int(done[0, c]) // 20
        for key in ("cn0", "pllLock", "locked"):
            assert a[key][0, c, :k].tobytes() == b[key][0, c, :k].tobytes(), (c, key)
        assert np.isnan(b["cn0"][0, c, k:]).all() and np.isnan(b["pllLock"][0, c, k:]).all()
        assert (b["locked"][0, c, k:] == 0).all()


@pytest.mark.gpu
def test_recarray_mirror():
    """cno_vsm(trackResults, Settings()) on tracking()'s recarray equals track_quality_batch on track_batch's output;
    the drop-in module exports it."""
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import cno_vsm, track_batch, track_quality_batch, tracking
    ms = 400
    dev, total, s, ch, _ = _track_case(ms, _two_sats(), [(0, 0.0, 0.0)], seed=41)
    data = dev[0, :total].cpu().numpy()
    res, _ = tracking(data, ch, s)
    q = cno_vsm(res, Settings())
    assert list(q.PRN) == [4, 17] and q.PRN.dtype == np.int64
    rc, out, done = track_batch(data[None], [total], [ch], s)
    assert rc == 0
    b = track_quality_batch(out, done, Settings())
    for k in range(2):
        assert np.array_equal(q[k].VSMIndex, b["index"])
        assert q[k].VSMValue.tobytes() == b["cn0"][0, k].tobytes()
        assert q[k].pllLock.tobytes() == b["pllLock"][0, k].tobytes()
        assert q[k].locked.tobytes() == b["locked"][0, k].tobytes()
    import importlib.util
    spec = importlib.util.spec_from_file_location("dropin_tracking", os.path.join(ROOT, "dropin", "tracking.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert mod.cno_vsm is cno_vsm


# ---------------------------------------------------------------------------------------------- CPU only
def test_settings_struct_size():
    from softgnss_python_b200 import _native
    assert ctypes.sizeof(_native.SgxQualitySettings) == 32


def test_settings_defaults_and_foreign_settings():
    """The extension attributes have the Matlab defaults; an object without them (the reference's own Settings) gets
    the same values."""
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import quality_pod
    s = Settings()
    assert (s.CNoVSMinterval, s.CNoAccTime, s.lockCNoMin, s.lockPllMin) == (40, 0.001, 30.0, 0.5)
    for obj in (s, object(), None):
        q = quality_pod(obj)
        assert (q.window_ms, q.acc_time, q.cn0_min, q.pll_lock_min) == (40, 0.001, 30.0, 0.5)
    q = quality_pod(Settings(CNoVSMinterval=20, lockCNoMin=35.0))
    assert (q.window_ms, q.cn0_min) == (20, 35.0)


def test_no_cpu_fallback():
    from softgnss_python_b200 import _native
    if _native.lib().dll.sgx_device_count() > 0:
        pytest.skip("a CUDA device is present")
    from softgnss_python_b200.settings import Settings
    from softgnss_python_b200.tracking import RESULT_DTYPE, cno_vsm, track_quality_batch
    with pytest.raises(_native.NativeError):
        track_quality_batch(np.zeros((1, 2, 13, 400)), None, Settings())
    rec = np.rec.fromrecords([(b'T',) + tuple(np.zeros(400) for _ in range(13)) + (5,)], dtype=RESULT_DTYPE)
    with pytest.raises(_native.NativeError):
        cno_vsm(rec, Settings())


def test_oracle_known_answer():
    """Noiseless two-level power: (I, Q) alternating (3, 0) and (0, 1), so Z alternates 9 and 1.  W = 4: Zm = 5,
    Zv = 4 * 4^2 / 3 = 64/3, Pav = sqrt(25 - 64/3) = sqrt(11/3), Nv = (5 - sqrt(11/3)) / 2, and
    cn0 = 10 log10(sqrt(11/3) / ((5 - sqrt(11/3)) * 0.001)) = 27.9286 dB-Hz; pll_lock = (18 - 2) / 20 = 0.8.
    W = 2: Zv = 32 > Zm^2 = 25, so no estimate."""
    from tests import quality_oracle as orc
    i = np.tile([3.0, 0.0], 6)
    q = np.tile([0.0, 1.0], 6)
    pav = np.sqrt(11.0 / 3.0)
    want = 10 * np.log10(pav / ((5 - pav) * 0.001))
    assert abs(want - 27.9286002) < 1e-6
    got = orc.cno_vsm(i, q, 4, 0.001)
    assert got.shape == (3,) and np.allclose(got, want, rtol=0, atol=1e-12)
    assert np.allclose(orc.pll_lock(i, q, 4), 0.8, rtol=0, atol=1e-15)
    assert np.isnan(orc.cno_vsm(i, q, 2, 0.001)).all()
    assert np.allclose(orc.pll_lock(i, q, 2), 0.8, rtol=0, atol=1e-15)
    # 5 samples with W = 4: one window, the trailing sample is not used
    assert orc.cno_vsm(i[:5], q[:5], 4, 0.001).shape == (1,)
