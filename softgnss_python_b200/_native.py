"""ctypes binding of the C ABI declared in include/softgnss_b200.h.

The library is the in-tree ``libsoftgnss_b200.so`` built by ``build.py`` (nvcc, sm_100a).  There is
no CPU fallback: every compute entry point raises :class:`NativeError` when the library or a CUDA
device is missing.
"""
import ctypes
import os

import numpy as np

from .settings import SgxSettings

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsoftgnss_b200.so")
MAX_SATS = 12
TRACK_FIELDS = ("absoluteSample", "codeFreq", "carrFreq", "I_P", "I_E", "I_L", "Q_E", "Q_P", "Q_L",
                "dllDiscr", "dllDiscrFilt", "pllDiscr", "pllDiscrFilt")
SGX_ERR_SHORT = -3


def track_field(track_out, field):
    """Rows of one field of a ``[R, C, 13, ms]`` tracking result, for the entry points that take a channel's series as
    (address, stride): a numpy array (made contiguous float64) or a contiguous float64 CUDA tensor.  Returns
    ``(address, row stride in elements, object to keep alive while the address is in use)``."""
    r, c, nf, ms = track_out.shape
    assert nf == len(TRACK_FIELDS), "a tracking result is [R, C, %d, ms]" % len(TRACK_FIELDS)
    if hasattr(track_out, "data_ptr"):
        import torch
        assert track_out.is_cuda and track_out.dtype == torch.float64 and track_out.is_contiguous()
        base = track_out.data_ptr()
    else:
        track_out = np.ascontiguousarray(track_out, dtype=np.float64)
        base = track_out.ctypes.data
    return base + 8 * TRACK_FIELDS.index(field) * ms, nf * ms, track_out

EXPORTS = ("sgx_abi_version", "sgx_last_error", "sgx_device_count", "sgx_set_device", "sgx_fp32_peak",
           "sgx_kernel_launch_count", "sgx_acquire", "sgx_track", "sgx_track_file", "sgx_synth_generate", "sgx_fft_c2c",
           "sgx_find_preambles", "sgx_pseudoranges", "sgx_nav_solve", "sgx_track_quality", "sgx_nav_velocity")


class NativeError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "softgnss_b200 error %d: %s" % (code, msg))
        self.code = code


class SgxChannel(ctypes.Structure):
    _fields_ = [("prn", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("acquiredFreq", ctypes.c_double), ("codePhase", ctypes.c_double)]


EPH_FIELDS = ("t_oc", "a_f2", "a_f1", "a_f0", "T_GD", "sqrtA", "t_oe", "deltan", "M_0", "e", "omega",
              "C_uc", "C_us", "C_rc", "C_rs", "i_0", "iDot", "C_ic", "C_is", "omega_0", "omegaDot")   # sgx_eph, in order
NAV_SOL_FIELDS = ("X", "Y", "Z", "dt", "GDOP", "PDOP", "HDOP", "VDOP", "TDOP", "latitude", "longitude", "height")
NAV_VEL_FIELDS = ("VX", "VY", "VZ", "clkDrift", "VE", "VN", "VU", "nUsed")                  # SGX_NAV_VEL_FIELDS


class SgxNavSettings(ctypes.Structure):
    _fields_ = [("samples_per_code", ctypes.c_double), ("start_offset", ctypes.c_double), ("c", ctypes.c_double),
                ("nav_sol_period", ctypes.c_double), ("elevation_mask", ctypes.c_double),
                ("use_trop_corr", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class SgxQualitySettings(ctypes.Structure):
    _fields_ = [("acc_time", ctypes.c_double), ("cn0_min", ctypes.c_double), ("pll_lock_min", ctypes.c_double),
                ("window_ms", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class SgxVelSettings(ctypes.Structure):
    _fields_ = [("IF", ctypes.c_double), ("c", ctypes.c_double), ("f_L1", ctypes.c_double),
                ("nav_sol_period", ctypes.c_double), ("doppler_avg_ms", ctypes.c_int32), ("reserved", ctypes.c_int32)]


class SgxSynthSpec(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("n_sats", ctypes.c_int32), ("noise_k", ctypes.c_int32),
                ("n_bits", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("prn", ctypes.c_int32 * MAX_SATS), ("amp", ctypes.c_int32 * MAX_SATS),
                ("per0", ctypes.c_int32 * MAX_SATS),
                ("phi0", ctypes.c_uint64 * MAX_SATS), ("dphi", ctypes.c_uint64 * MAX_SATS),
                ("cp0", ctypes.c_uint64 * MAX_SATS), ("dcp", ctypes.c_uint64 * MAX_SATS)]


def _ptr(x):
    """Raw address of a numpy array, a torch tensor, a ctypes object or an int."""
    if x is None:
        return None
    if isinstance(x, int):
        return ctypes.c_void_p(x)
    if isinstance(x, np.ndarray):
        assert x.flags["C_CONTIGUOUS"]
        return ctypes.c_void_p(x.ctypes.data)
    if hasattr(x, "data_ptr"):
        return ctypes.c_void_p(x.data_ptr())
    return ctypes.cast(x, ctypes.c_void_p)


class Lib(object):
    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise NativeError(-100, "%s not built -- run `python -m softgnss_python_b200.build` "
                                    "(needs nvcc; there is no CPU fallback)" % path)
        self.path = path
        self.dll = ctypes.CDLL(path)
        vp, i32, i64, f64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_double
        d = self.dll
        d.sgx_abi_version.restype = ctypes.c_int
        d.sgx_last_error.restype = ctypes.c_char_p
        d.sgx_device_count.restype = ctypes.c_int
        d.sgx_set_device.argtypes = [ctypes.c_int]
        d.sgx_fp32_peak.argtypes = [vp, vp]
        d.sgx_kernel_launch_count.restype = i64
        d.sgx_acquire.argtypes = [vp, i64, i64, i32, ctypes.POINTER(SgxSettings), vp, vp, vp, i32, i32,
                                  vp, vp, vp, vp, vp, vp]
        d.sgx_track.argtypes = [vp, i64, vp, i32, vp, i32, ctypes.POINTER(SgxSettings), vp, vp, vp, vp]
        d.sgx_track_file.argtypes = [ctypes.c_char_p, i32, vp, i32, ctypes.POINTER(SgxSettings), vp, vp, vp, i64, vp, vp]
        d.sgx_synth_generate.argtypes = [vp, i64, i64, i64, i32, vp, vp, vp, vp, vp]
        d.sgx_fft_c2c.argtypes = [vp, vp, i32, i32, i32, vp]
        d.sgx_find_preambles.argtypes = [vp, i64, i32, i32, vp, vp, vp, vp]
        d.sgx_pseudoranges.argtypes = [vp, i32, i32, i32, vp, vp, i32, f64, f64, f64, vp, vp]
        d.sgx_track_quality.argtypes = [vp, vp, i64, i32, i32, vp, ctypes.POINTER(SgxQualitySettings), vp, vp, vp, vp]
        d.sgx_nav_solve.argtypes = [vp, i64, i32, i32, i32, vp, vp, vp, vp, vp, i32, ctypes.POINTER(SgxNavSettings),
                                    vp, vp, vp, vp, vp, vp, vp, vp, vp]
        d.sgx_nav_velocity.argtypes = [vp, i64, i32, i32, i32, vp, vp, vp, vp, vp, i32, vp, vp,
                                       ctypes.POINTER(SgxVelSettings), vp, vp, vp, vp, vp, vp]

    def check(self, rc):
        if rc != 0:
            raise NativeError(rc, self.dll.sgx_last_error().decode())

    def require_device(self):
        if self.dll.sgx_device_count() <= 0:
            raise NativeError(-4, "no CUDA device visible; the B200 path has no CPU fallback")

    def launches(self):
        return int(self.dll.sgx_kernel_launch_count())

    def fp32_peak(self, stream=0):
        """Measured FP32 FMA-burn throughput of the current device, TFLOP/s."""
        self.require_device()
        v = ctypes.c_double(0.0)
        self.check(self.dll.sgx_fp32_peak(ctypes.byref(v), ctypes.c_void_p(stream)))
        return float(v.value)

    # ------------------------------------------------------------------ tracking
    def track(self, rec, rec_stride, rec_len, channels, pod, ca_chips, out, stream=0):
        """rec: int8 numpy [R, stride] / torch cuda tensor / address; channels: SgxChannel array [R*C];
        out: float64 numpy or cuda tensor [R, C, 13, ms].  Returns (rc, ms_done[R, C])."""
        self.require_device()
        rec_len = np.ascontiguousarray(rec_len, dtype=np.int64)
        r = len(rec_len)
        c = len(channels) // r
        ms_done = np.zeros((r, c), dtype=np.int32)
        rc = self.dll.sgx_track(_ptr(rec), int(rec_stride), _ptr(rec_len), r, _ptr(channels), c,
                                ctypes.byref(pod), _ptr(ca_chips), _ptr(out), _ptr(ms_done),
                                ctypes.c_void_p(stream))
        return rc, ms_done

    def track_file(self, path, sample_bytes, channels, pod, ca_chips, out, chunk_samples=0, stream=0):
        """One recording streamed from a file (pread -> pinned double buffer -> HBM).  Returns
        (rc, ms_done[1, C], (first sample, samples) of the window that was read)."""
        self.require_device()
        c = len(channels)
        ms_done = np.zeros((1, c), dtype=np.int32)
        window = np.zeros(2, dtype=np.int64)
        rc = self.dll.sgx_track_file(os.fsencode(path), int(sample_bytes), _ptr(channels), c, ctypes.byref(pod),
                                     _ptr(ca_chips), _ptr(out), _ptr(ms_done), int(chunk_samples), _ptr(window),
                                     ctypes.c_void_p(stream))
        return rc, ms_done, (int(window[0]), int(window[1]))

    def fft(self, x, inverse=False, stream=0, persistent=False):
        """Unnormalised FFT of the rows of complex64 x through the acquisition FFT engine (test hook);
        ``persistent``: passes after the first use the persistent pass kernels of the search."""
        self.require_device()
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.complex64)
        out = np.empty_like(x)
        self.check(self.dll.sgx_fft_c2c(_ptr(x), _ptr(out), x.shape[1], x.shape[0], int(bool(inverse)) | (2 if persistent else 0),
                                        ctypes.c_void_p(stream)))
        return out

    # ------------------------------------------------------------------ bit synchronisation
    def find_preambles(self, i_p, stride, n_channels, ms, want_bits=True, stream=0):
        """i_p: float64 [n_channels][stride] (numpy or CUDA tensor).  Returns (first int32[n], bits uint8[n,1501]
        or None, valid int32[n] or None) as numpy arrays."""
        self.require_device()
        first = np.zeros(n_channels, dtype=np.int32)
        bits = np.zeros((n_channels, 1501), dtype=np.uint8) if want_bits else None
        valid = np.zeros(n_channels, dtype=np.int32) if want_bits else None
        self.check(self.dll.sgx_find_preambles(_ptr(i_p), int(stride), int(n_channels), int(ms), _ptr(first),
                                               _ptr(bits), _ptr(valid), ctypes.c_void_p(stream)))
        return first, bits, valid

    def pseudoranges(self, track_out, n_rec, n_ch, ms, ms_index, active, samples_per_code, start_offset, c, stream=0):
        """track_out: float64 [n_rec][n_ch][13][ms] (numpy or CUDA tensor); ms_index int32 / active uint8
        [n_rec][n_epochs][n_ch].  Returns float64 [n_rec][n_epochs][n_ch]."""
        self.require_device()
        ms_index = np.ascontiguousarray(ms_index, dtype=np.int32).reshape(n_rec, -1, n_ch)
        active = np.ascontiguousarray(active, dtype=np.uint8).reshape(n_rec, -1, n_ch)
        n_ep = ms_index.shape[1]
        out = np.empty((n_rec, n_ep, n_ch), dtype=np.float64)
        self.check(self.dll.sgx_pseudoranges(_ptr(track_out), n_rec, n_ch, int(ms), _ptr(ms_index), _ptr(active), n_ep,
                                             float(samples_per_code), float(start_offset), float(c), _ptr(out),
                                             ctypes.c_void_p(stream)))
        return out

    def track_quality(self, i_p, q_p, stride, n_channels, ms, ms_done, qs, cn0, pll_lock, locked, stream=0):
        """Per-window C/N0 / carrier lock (sgx_track_quality).  i_p, q_p: float64 numpy arrays, CUDA tensors or
        addresses whose channel rows are `stride` apart; ms_done: int32 [n_channels] or None; qs: SgxQualitySettings;
        cn0, pll_lock (float64) and locked (uint8) [n_channels][ms // qs.window_ms], written in place.  Returns rc."""
        self.require_device()
        if ms_done is not None:
            ms_done = np.ascontiguousarray(ms_done, dtype=np.int32).reshape(-1)
            assert ms_done.size == n_channels
        return self.dll.sgx_track_quality(_ptr(i_p), _ptr(q_p), int(stride), int(n_channels), int(ms), _ptr(ms_done),
                                          ctypes.byref(qs), _ptr(cn0), _ptr(pll_lock), _ptr(locked),
                                          ctypes.c_void_p(stream))

    def nav_solve(self, abs_sample, stride, n_rec, n_ch, ms, sub_frame_start, ready, eph, tow, n_epochs, nav_settings,
                  want_sat=True, stream=0):
        """abs_sample: float64 numpy array / CUDA tensor whose channel rows are `stride` apart; sub_frame_start int32 /
        ready uint8 [n_rec][n_ch]; eph float64 [n_rec][n_ch][21] (EPH_FIELDS order); tow float64 [n_rec]; n_epochs
        int32 [n_rec].  Returns a dict of numpy arrays with the epoch axis second ([R][E][C] / [R][E][12])."""
        self.require_device()
        sub_frame_start = np.ascontiguousarray(sub_frame_start, dtype=np.int32).reshape(n_rec, n_ch)
        ready = np.ascontiguousarray(ready, dtype=np.uint8).reshape(n_rec, n_ch)
        eph = np.ascontiguousarray(eph, dtype=np.float64).reshape(n_rec, n_ch, len(EPH_FIELDS))
        tow = np.ascontiguousarray(tow, dtype=np.float64).reshape(n_rec)
        n_epochs = np.ascontiguousarray(n_epochs, dtype=np.int32).reshape(n_rec)
        e_max = int(n_epochs.max()) if n_rec else 0
        shp = (n_rec, e_max, n_ch)
        out = dict(rawP=np.empty(shp), correctedP=np.empty(shp), el=np.empty(shp), az=np.empty(shp),
                   satPositions=np.empty(shp + (3,)) if want_sat else None, satClkCorr=np.empty(shp) if want_sat else None,
                   active=np.empty(shp, dtype=np.uint8), sol=np.empty((n_rec, e_max, len(NAV_SOL_FIELDS))))
        self.check(self.dll.sgx_nav_solve(_ptr(abs_sample), int(stride), n_rec, n_ch, int(ms), _ptr(sub_frame_start),
                                          _ptr(ready), _ptr(eph), _ptr(tow), _ptr(n_epochs), e_max,
                                          ctypes.byref(nav_settings), _ptr(out["rawP"]), _ptr(out["correctedP"]),
                                          _ptr(out["el"]), _ptr(out["az"]), _ptr(out["satPositions"]),
                                          _ptr(out["satClkCorr"]), _ptr(out["active"]), _ptr(out["sol"]),
                                          ctypes.c_void_p(stream)))
        out["n_epochs"] = n_epochs
        return out

    def nav_velocity(self, carr_freq, stride, n_rec, n_ch, ms, ms_done, sub_frame_start, eph, tow, n_epochs, active, sol,
                     vel_settings, want_sat=False, out=None, stream=0):
        """Velocity and clock drift per epoch (sgx_nav_velocity).  carr_freq: float64 numpy array, CUDA tensor or address
        whose channel rows are `stride` apart; ms_done int32 [n_rec][n_ch] or None; sub_frame_start / eph / tow /
        n_epochs as for nav_solve; active uint8 [n_rec][E][n_ch] and sol float64 [n_rec][E][12]: nav_solve's outputs
        (numpy or CUDA tensors).  ``out``: optional dict of preallocated outputs (vel, doppler, rrResid and, with
        want_sat, satVel, satClkDrift; numpy or CUDA tensors); by default numpy arrays are allocated.  Returns that dict."""
        self.require_device()
        if ms_done is not None:
            ms_done = np.ascontiguousarray(ms_done, dtype=np.int32).reshape(n_rec, n_ch)
        sub_frame_start = np.ascontiguousarray(sub_frame_start, dtype=np.int32).reshape(n_rec, n_ch)
        eph = np.ascontiguousarray(eph, dtype=np.float64).reshape(n_rec, n_ch, len(EPH_FIELDS))
        tow = np.ascontiguousarray(tow, dtype=np.float64).reshape(n_rec)
        n_epochs = np.ascontiguousarray(n_epochs, dtype=np.int32).reshape(n_rec)
        if isinstance(active, np.ndarray):
            active = np.ascontiguousarray(active, dtype=np.uint8)
        if isinstance(sol, np.ndarray):
            sol = np.ascontiguousarray(sol, dtype=np.float64)
        e_max = int(sol.shape[1])
        assert tuple(active.shape) == (n_rec, e_max, n_ch) and tuple(sol.shape) == (n_rec, e_max, len(NAV_SOL_FIELDS))
        shp = (n_rec, e_max, n_ch)
        if out is None:
            out = dict(vel=np.empty((n_rec, e_max, len(NAV_VEL_FIELDS))), doppler=np.empty(shp), rrResid=np.empty(shp),
                       satVel=np.empty(shp + (3,)) if want_sat else None, satClkDrift=np.empty(shp) if want_sat else None)
        self.check(self.dll.sgx_nav_velocity(_ptr(carr_freq), int(stride), n_rec, n_ch, int(ms), _ptr(ms_done),
                                             _ptr(sub_frame_start), _ptr(eph), _ptr(tow), _ptr(n_epochs), e_max,
                                             _ptr(active), _ptr(sol), ctypes.byref(vel_settings), _ptr(out["vel"]),
                                             _ptr(out["doppler"]), _ptr(out["rrResid"]), _ptr(out.get("satVel")),
                                             _ptr(out.get("satClkDrift")), ctypes.c_void_p(stream)))
        return out

    # ------------------------------------------------------------------ synthetic recordings
    def synth(self, out, rec_stride, n_samples, start, specs, bits, lut, ca_chips, stream=0):
        self.require_device()
        self.check(self.dll.sgx_synth_generate(_ptr(out), int(rec_stride), int(n_samples), int(start),
                                               len(specs), _ptr(specs), _ptr(bits), _ptr(lut),
                                               _ptr(ca_chips), ctypes.c_void_p(stream)))


_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        _LIB = Lib()
    return _LIB


def ca_chips_int8():
    from .settings import ca_code_bits
    return np.ascontiguousarray(np.stack([ca_code_bits(p) for p in range(32)]).astype(np.int8) * 2 - 1)


def make_channels(prn, freq, cph):
    n = len(prn)
    arr = (SgxChannel * n)()
    for i in range(n):
        arr[i].prn = int(prn[i])
        arr[i].acquiredFreq = float(freq[i])
        arr[i].codePhase = float(cph[i])
    return arr


def make_synth_specs(specs):
    """list of synth.RecordingSpec -> (SgxSynthSpec array, bits int8 [R, MAX_SATS, n_bits])."""
    n = len(specs)
    arr = (SgxSynthSpec * n)()
    nb = specs[0].n_bits
    bits = np.ones((n, MAX_SATS, nb), dtype=np.int8)
    for r, sp in enumerate(specs):
        a = arr[r]
        a.seed = sp.seed & ((1 << 64) - 1)
        a.n_sats = len(sp.prn)
        a.noise_k = sp.noise_k
        a.n_bits = nb
        for i in range(len(sp.prn)):
            a.prn[i] = int(sp.prn[i]); a.amp[i] = int(sp.amp[i]); a.per0[i] = int(sp.per0[i])
            a.phi0[i] = int(sp.phi0[i]); a.dphi[i] = int(sp.dphi[i])
            a.cp0[i] = int(sp.cp0[i]); a.dcp[i] = int(sp.dcp[i])
        bits[r, :len(sp.prn)] = sp.bits
    return arr, bits
