"""Tracking stage: same call surface as the reference, computed by the sm_100a kernel.

Reference surface (``tracking.py:6-295``):
    ``TrackingResult(acqResult).track(fid)`` then ``.results`` / ``.channels`` / ``.settings``;
the Matlab-style function the reference keeps as a comment (``tracking.py:18``):
    ``trackResults, channel = tracking(fid, channel, settings)``.

Both are provided.  ``fid`` may be an open binary file (the reference's only form), a path, an int8
numpy array holding the file's bytes, or an int8 CUDA tensor already resident in HBM.  The result is
the reference's recarray (``tracking.py:285-294``): one record per channel whose PRN != 0, fields
``status`` ('S1'), thirteen float64[msToProcess] series as object fields, ``PRN`` int64.
On a short recording the reference prints a message and returns None (``tracking.py:159-163``);
so does this.

Extension (no reference behaviour): the per-channel C/N0 and lock detector of the later Matlab SoftGNSS releases
(``CNoVSM``), as ``track_quality_batch`` on a batched tracking result and ``cno_vsm`` on the recarray.
"""
import numpy as np

from . import _native
from .settings import to_pod

FIELDS = _native.TRACK_FIELDS
FILE_CHUNK_SAMPLES = 0          # samples per staging buffer of the file ingest (0: the library's default, 1024 code periods)
RESULT_DTYPE = [('status', 'S1')] + [(f, 'object') for f in FIELDS] + [('PRN', 'int64')]


class Result(object):
    """Base of the stage objects (reference ``initialize.py:20-46``)."""

    def __init__(self, settings):
        self._settings = settings
        self._results = None
        self._channels = None

    @property
    def settings(self):
        return self._settings

    @property
    def channels(self):
        assert isinstance(self._channels, np.recarray)
        return self._channels

    @property
    def results(self):
        assert isinstance(self._results, np.recarray)
        return self._results

    @results.setter
    def results(self, records):
        assert isinstance(records, np.recarray)
        self._results = records

    def plot(self):
        pass


SAMPLE_BYTES = {"int8": 1, "b": 1, "schar": 1, "int16": 2, "short": 2}


def _sample_bytes(settings):
    """``settings.dataType`` (initialize.py:102) -> bytes per sample; anything but int8 / int16 is rejected."""
    dt = str(getattr(settings, "dataType", "int8"))
    if dt not in SAMPLE_BYTES:
        raise _native.NativeError(-2, "dataType %r is not supported (int8, int16)" % dt)
    return SAMPLE_BYTES[dt]


def _file_path(fid):
    """Path of a recording given as a path or as an open file object (the reference's form), else None."""
    import os
    if isinstance(fid, (str, bytes, os.PathLike)):
        return os.fspath(fid)
    name = getattr(fid, "name", None)
    if isinstance(name, (str, bytes)) and os.path.exists(name):
        return name
    return None


def _load_recording(fid, settings=None):
    """In-memory forms of a recording: an int8 numpy array, a CUDA tensor (passed through), or a file-like object
    without a path (read once).  Files with a path never come here: they are streamed (``sgx_track_file``)."""
    if hasattr(fid, "data_ptr"):            # torch tensor
        return fid
    if isinstance(fid, np.ndarray):
        assert fid.dtype == np.int8 and fid.ndim == 1
        return np.ascontiguousarray(fid)
    fid.seek(0)
    raw = fid.read()
    if settings is not None and _sample_bytes(settings) == 2:
        x = np.frombuffer(raw, dtype="<i2")
        if x.size and (x.min() < -128 or x.max() > 127):
            raise _native.NativeError(-2, "int16 sample outside the int8 range of the correlators")
        return x.astype(np.int8)
    return np.frombuffer(raw, dtype=np.int8)


def track_batch(recordings, rec_len, channel_sets, settings, out=None, stream=0):
    """Batched entry: ``recordings`` int8 [R, stride] (numpy or CUDA tensor), ``channel_sets`` a list of
    R channel recarrays (``preRun`` output).  Returns (rc, out[R, C, 13, ms], ms_done[R, C])."""
    L = _native.lib()
    pod = to_pod(settings)
    r = len(channel_sets)
    c = int(settings.numberOfChannels)
    prn, freq, cph = [], [], []
    for ch in channel_sets:
        for i in range(c):
            prn.append(int(ch.PRN[i])); freq.append(float(ch.acquiredFreq[i])); cph.append(float(ch.codePhase[i]))
    chans = _native.make_channels(prn, freq, cph)
    ms = pod.msToProcess
    if out is None:
        out = np.empty((r, c, len(FIELDS), ms), dtype=np.float64)
    stride = recordings.stride(0) if hasattr(recordings, "data_ptr") else recordings.strides[0]
    rc, done = L.track(recordings, stride, rec_len, chans, pod, _native.ca_chips_int8(), out, stream)
    return rc, out, done


QUALITY_DTYPE = [('PRN', 'int64'), ('VSMValue', 'object'), ('VSMIndex', 'object'), ('pllLock', 'object'),
                 ('locked', 'object')]


def quality_pod(settings=None):
    """``sgx_quality_settings`` from the extension attributes ``CNoVSMinterval``, ``CNoAccTime``, ``lockCNoMin`` and
    ``lockPllMin``; an object without them (the reference's own Settings, or None) gets their defaults."""
    g = lambda name, default: getattr(settings, name, default)
    return _native.SgxQualitySettings(acc_time=float(g("CNoAccTime", 0.001)), cn0_min=float(g("lockCNoMin", 30.0)),
                                      pll_lock_min=float(g("lockPllMin", 0.5)),
                                      window_ms=int(g("CNoVSMinterval", 40)), reserved=0)


def track_quality_batch(track_out, ms_done=None, settings=None, stream=0):
    """C/N0 (variance-summing method) and carrier lock per window of ``settings.CNoVSMinterval`` code periods for
    every channel of a tracking result, computed by ``sgx_track_quality`` (csrc/sgx_quality.cu).

    ``track_out``: float64 ``[R, C, 13, ms]`` as ``track_batch`` returns it, a numpy array or a contiguous CUDA
    tensor; the I_P and Q_P fields are read in place.  ``ms_done``: ``[R, C]`` periods completed (``track_batch``'s
    third result) or None for all ``ms``.  Returns ``dict(cn0, pllLock, locked, index)``: the first three ``[R, C,
    n_win]`` (float64, float64, uint8; numpy for a numpy input, CUDA tensors on the input's device otherwise, written
    asynchronously on ``stream``), ``index`` int64 ``[n_win]`` = ``(w + 1) * W``, the period count at which window w
    is complete (Matlab's ``VSMIndex``).  There is no host implementation: without a device this raises NativeError."""
    L = _native.lib()
    L.require_device()
    qs = quality_pod(settings)
    r, c, _, ms = track_out.shape
    i_p, stride, track_out = _native.track_field(track_out, "I_P")
    q_p = _native.track_field(track_out, "Q_P")[0]
    n_win = ms // qs.window_ms if qs.window_ms >= 2 else 0   # W < 2 is refused by the library
    if hasattr(track_out, "data_ptr"):
        import torch
        res = dict(cn0=torch.empty((r, c, n_win), dtype=torch.float64, device=track_out.device),
                   pllLock=torch.empty((r, c, n_win), dtype=torch.float64, device=track_out.device),
                   locked=torch.empty((r, c, n_win), dtype=torch.uint8, device=track_out.device))
    else:
        res = dict(cn0=np.empty((r, c, n_win)), pllLock=np.empty((r, c, n_win)),
                   locked=np.empty((r, c, n_win), dtype=np.uint8))
    done = None if ms_done is None else np.ascontiguousarray(ms_done, dtype=np.int32).reshape(r * c)
    if n_win or qs.window_ms < 2:           # (an empty CUDA tensor has no address to pass)
        L.check(L.track_quality(i_p, q_p, stride, r * c, ms, done, qs, res["cn0"], res["pllLock"], res["locked"],
                                stream))
    res["index"] = (np.arange(n_win, dtype=np.int64) + 1) * qs.window_ms
    return res


def cno_vsm(trackResults, settings):
    """Function-style mirror of the Matlab SoftGNSS ``CNoVSM`` stage on the tracking recarray: one record per tracked
    channel with ``PRN`` and the object fields ``VSMValue`` (C/N0 per window, dB-Hz, NaN where undefined),
    ``VSMIndex`` (``(w + 1) * CNoVSMinterval``), ``pllLock`` (cos 2 dphi per window) and ``locked`` (uint8).  Computed
    on the device by ``sgx_track_quality``; raises NativeError without one."""
    L = _native.lib()
    L.require_device()
    qs = quality_pod(settings)
    n = len(trackResults)
    if n == 0:
        return np.recarray((0,), dtype=QUALITY_DTYPE)
    i_p = np.ascontiguousarray(np.stack([np.asarray(trackResults[k].I_P, dtype=np.float64) for k in range(n)]))
    q_p = np.ascontiguousarray(np.stack([np.asarray(trackResults[k].Q_P, dtype=np.float64) for k in range(n)]))
    ms = i_p.shape[1]
    n_win = ms // qs.window_ms if qs.window_ms >= 2 else 0   # W < 2 is refused by the library
    cn0, pll, locked = np.empty((n, n_win)), np.empty((n, n_win)), np.empty((n, n_win), dtype=np.uint8)
    L.check(L.track_quality(i_p, q_p, ms, n, ms, None, qs, cn0, pll, locked))
    index = (np.arange(n_win, dtype=np.int64) + 1) * qs.window_ms
    recs = [(int(trackResults[k].PRN), cn0[k], index.copy(), pll[k], locked[k]) for k in range(n)]
    return np.rec.fromrecords(recs, dtype=QUALITY_DTYPE)


def tracking(fid, channel, settings):
    """``[trackResults, channel] = tracking(fid, channel, settings)`` (reference tracking.py:13-295)."""
    path = _file_path(fid)
    if path is not None:
        # on-disk recording: pread -> two pinned staging buffers -> HBM, overlapped with tracking; only the window the
        # channels can touch is read (tracking.py:107, :154; initialize.py:102, :466-481)
        L = _native.lib()
        pod = to_pod(settings)
        c = int(settings.numberOfChannels)
        chans = _native.make_channels([int(channel.PRN[i]) for i in range(c)],
                                      [float(channel.acquiredFreq[i]) for i in range(c)],
                                      [float(channel.codePhase[i]) for i in range(c)])
        out = np.zeros((1, c, len(FIELDS), pod.msToProcess), dtype=np.float64)
        rc, done, _ = L.track_file(path, _sample_bytes(settings), chans, pod, _native.ca_chips_int8(), out,
                                   chunk_samples=FILE_CHUNK_SAMPLES)
    else:
        data = _load_recording(fid, settings)
        n = int(data.numel() if hasattr(data, "data_ptr") else data.size)
        rec = data.reshape(1, n) if not hasattr(data, "data_ptr") else data.view(1, n)
        rc, out, done = track_batch(rec, [n], [channel], settings)
    if rc == _native.SGX_ERR_SHORT:
        print('Not able to read the specified number of samples for tracking, exiting!')
        if hasattr(fid, "close"):
            fid.close()
        return None, channel
    _native.lib().check(rc)
    recs = []
    for i in range(int(settings.numberOfChannels)):
        if channel.PRN[i] == 0:           # tracking.py:99, :280-283 -- idle channels produce no record
            continue
        series = tuple(np.array(out[0, i, f]) for f in range(len(FIELDS)))
        recs.append((channel.status[i],) + series + (int(channel.PRN[i]),))
    if recs:
        res = np.rec.fromrecords(recs, dtype=RESULT_DTYPE)
    else:
        res = np.recarray((0,), dtype=RESULT_DTYPE)
    return res, channel


class TrackingResult(Result):
    """Drop-in for the reference class of the same name (``tracking.py:6-13``)."""

    def __init__(self, acqResult):
        self._results = None
        self._channels = acqResult.channels
        self._settings = acqResult.settings

    def track(self, fid):
        res, _ = tracking(fid, self._channels, self._settings)
        if res is None:
            return None
        self._results = res
        return
