"""Host and device operands of the five post-tracking entry points (sgx_find_preambles, sgx_pseudoranges,
sgx_track_quality, sgx_nav_solve, sgx_nav_velocity), which all stage them through the helpers of csrc/sgx_common.cuh:

  * host and device operands give bit-identical results;
  * a series read as one field of a [R, C, 13, ms] tracking result (stride 13 * ms) gives the same result as the
    same rows packed;
  * host staging reads nothing outside the documented rows (CPU emulator only: the tracking result is put right
    before an inaccessible page, in a child process so that a fault fails one test);
  * sgx_find_preambles leaves nav_bits_valid untouched when nav_bits is NULL.

Two backends, as in test_gpu_track_quality.py:
  * gpu  -- the sm_100a library on the device (marker gpu);
  * emul -- the same CUDA sources under the CPU fiber emulator (marker emul, opt-in: SGX_EMUL_TESTS=1 and
            tools/cpu_emul/libsoftgnss_emul.so, built by tools/cpu_emul/build_emul.sh).  The emulator treats every
            pointer as device memory unless SGX_EMUL_HOST is set, so there host and device operands can only be
            switched together.
"""
import ctypes
import mmap
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import nav_util
from tests.cases import NAV_MS, _hash_noise, build_bitsync_case, load_nav_cases, nav_abs_sample

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_LIB = os.path.join(ROOT, "tools", "cpu_emul", "libsoftgnss_emul.so")
ENTRY_POINTS = ("find_preambles", "pseudoranges", "track_quality", "nav_solve", "nav_velocity")
NF = 13
IF = 9548000.0
N_EPOCHS = 6                       # pseudorange epochs
QUALITY_W = 40
FIELD = dict(absoluteSample=0, carrFreq=2, I_P=3, Q_P=7)        # where the series of each stage are read


# ---------------------------------------------------------------------------------------------- inputs
_INPUTS = {}


def inputs():
    """One [R, C, 13, ms] tracking result for all five stages, R = 2 golden navigation cases of 8 channels: field 0
    absoluteSample, 2 carrFreq, 3 I_P (preamble-search channels), 7 Q_P; every other field NaN, so that a stage
    reading the wrong rows, or between them, sees NaN.  Plus the per-stage inputs, all host arrays."""
    if not _INPUTS:
        from softgnss_python_b200 import postnav
        cases = [load_nav_cases()[i] for i in (0, 2)]
        r, c, ms = len(cases), 8, NAV_MS
        # one spare row of all fields after the array: a stage that over-reads the last row fails the guarded test
        # below instead of faulting here
        trk = np.full(r * c * NF * ms + NF * ms, np.nan)[:r * c * NF * ms].reshape(r, c, NF, ms)
        k = np.arange(ms)
        for i, case in enumerate(cases):
            trk[i, :, 0] = nav_abs_sample(case["coef"])
            trk[i, :, 3] = np.stack(build_bitsync_case(seed0=500 + 100 * i))
            for ch in range(c):
                trk[i, ch, 2] = IF + 800.0 * np.sin(k / 9000.0 + ch) + 0.01 * _hash_noise(40 + 10 * i + ch, ms)
                trk[i, ch, 7] = 3.0 * _hash_noise(70 + 10 * i + ch, ms)
        settings = nav_util.settings_for(cases[0], c, ms)
        sfs = np.stack([nav_util.case_inputs(cs)[0] for cs in cases])
        n_ep = np.array([postnav.nav_epochs(settings, sfs[i]) for i in range(r)], dtype=np.int32)
        rng = np.random.default_rng(11)
        done = np.full(r * c, ms, dtype=np.int32)
        done[[1, 6, 12]] = (ms - 1, 4000, 25000)
        _INPUTS.update(
            trk=trk, r=r, c=c, ms=ms, sfs=sfs, n_ep=n_ep, max_ep=int(n_ep.max()),
            ready=np.stack([nav_util.case_inputs(cs)[1] for cs in cases]),
            eph=np.ascontiguousarray(np.stack([nav_util.case_inputs(cs)[2] for cs in cases]), dtype=np.float64),
            tow=np.array([cs["tow"] for cs in cases]), nav_settings=postnav.nav_settings(settings), ms_done=done,
            ms_index=rng.integers(-2, ms + 2, (r, N_EPOCHS, c)).astype(np.int32),
            active=(rng.random((r, N_EPOCHS, c)) < 0.8).astype(np.uint8))
    return _INPUTS


def _rows(trk, field, packed):
    """(array, element offset, stride) of one field's rows: in place in trk, or packed [R*C, ms]."""
    ms = trk.shape[-1]
    if packed:
        return np.ascontiguousarray(trk[:, :, field]), 0, ms
    return trk, field * ms, NF * ms


# ---------------------------------------------------------------------------------------------- backends
class Backend(object):
    """One library (device build or CPU emulator) and where it puts the operands of a call."""

    def __init__(self, name, lib):
        self.name = name
        self.lib = lib
        self._nav = None
        # (host inputs, host outputs) of the calls compared with all-host operands
        self.kinds = [(True, True), (False, False)] + ([(True, False), (False, True)] if name == "gpu" else [])

    def run(self, entry, packed=False, host_in=True, host_out=True):
        """Calls `entry` on the shared inputs; returns its outputs as host arrays."""
        env = os.environ.pop("SGX_EMUL_HOST", None)
        try:
            if self.name == "emul":
                assert host_in == host_out, "the emulator switches host / device operands together"
                if host_in:
                    os.environ["SGX_EMUL_HOST"] = "1"
            ops = _Operands(self.name == "gpu", host_in, host_out)
            outs = CALLS[entry](self, ops, inputs(), packed)
            return ops.fetch(outs)
        finally:
            os.environ.pop("SGX_EMUL_HOST", None)
            if env is not None:
                os.environ["SGX_EMUL_HOST"] = env

    def nav(self):
        """sgx_nav_solve's active and sol on all-host operands: inputs of sgx_nav_velocity."""
        if self._nav is None:
            self._nav = self.run("nav_solve", packed=True)
        return self._nav

    def check(self, rc):
        assert rc == 0, self.lib.dll.sgx_last_error().decode()


class _Operands(object):
    """Host operands are numpy arrays; device operands (gpu backend) CUDA copies of them."""

    def __init__(self, gpu, host_in, host_out):
        self.gpu, self.host_in, self.host_out = gpu, host_in, host_out
        self.keep = []

    def _place(self, a, host):
        if host or not self.gpu:
            return a
        import torch
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.keep.append(t)
        return t

    def addr(self, a, host, offset=0):
        """Address of element `offset` of a, placed as `host` says."""
        if a is None:
            return None
        skip = a.itemsize * offset
        a = self._place(a, host)
        return (a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data) + skip

    def inp(self, a, offset=0):
        return self.addr(a, self.host_in, offset)

    def out(self, shape, dtype=np.float64, fill=-1):
        a = self._place(np.full(shape, fill, dtype=dtype), self.host_out)
        return a, self.addr(a, True)

    def fetch(self, outs):
        if self.gpu:
            import torch
            torch.cuda.synchronize()
        return [o.cpu().numpy() if hasattr(o, "cpu") else o for o in outs]


def _find_preambles(b, ops, d, packed):
    a, off, stride = _rows(d["trk"], FIELD["I_P"], packed)
    n = d["r"] * d["c"]
    (first, p1), (bits, p2), (valid, p3) = ops.out(n, np.int32), ops.out((n, 1501), np.uint8, 7), ops.out(n, np.int32)
    b.check(b.lib.dll.sgx_find_preambles(ops.inp(a, off), stride, n, d["ms"], p1, p2, p3, None))
    return [first, bits, valid]


def _pseudoranges(b, ops, d, packed):
    trk = d["trk"]
    if packed:                                   # field 0 alone: every other value NaN
        trk = np.full_like(trk, np.nan)
        trk[:, :, 0] = d["trk"][:, :, 0]
    pr, p = ops.out(d["ms_index"].shape)
    b.check(b.lib.dll.sgx_pseudoranges(ops.inp(trk), d["r"], d["c"], d["ms"], ops.inp(d["ms_index"]),
                                       ops.inp(d["active"]), N_EPOCHS, 38192.0, 68.802, 299792458.0, p, None))
    return [pr]


def _track_quality(b, ops, d, packed):
    from softgnss_python_b200 import _native
    a_i, off_i, stride = _rows(d["trk"], FIELD["I_P"], packed)
    a_q, off_q, _ = _rows(d["trk"], FIELD["Q_P"], packed)
    n, ms = d["r"] * d["c"], d["ms"]
    qs = _native.SgxQualitySettings(acc_time=0.001, cn0_min=30.0, pll_lock_min=0.5, window_ms=QUALITY_W)
    shape = (n, ms // QUALITY_W)
    (cn0, p1), (pll, p2), (locked, p3) = ops.out(shape), ops.out(shape), ops.out(shape, np.uint8, 7)
    b.check(b.lib.dll.sgx_track_quality(ops.inp(a_i, off_i), ops.inp(a_q, off_q), stride, n, ms, d["ms_done"].ctypes.data,
                                        ctypes.byref(qs), p1, p2, p3, None))
    return [cn0, pll, locked]


def _nav_solve(b, ops, d, packed):
    a, off, stride = _rows(d["trk"], FIELD["absoluteSample"], packed)
    r, c, e = d["r"], d["c"], d["max_ep"]
    outs = [ops.out((r, e, c)) for _ in range(4)] + [ops.out((r, e, c, 3)), ops.out((r, e, c)),
                                                     ops.out((r, e, c), np.uint8, 7), ops.out((r, e, 12))]
    b.check(b.lib.dll.sgx_nav_solve(ops.inp(a, off), stride, r, c, d["ms"], ops.inp(d["sfs"]), ops.inp(d["ready"]),
                                    ops.inp(d["eph"]), ops.inp(d["tow"]), ops.inp(d["n_ep"]), e,
                                    ctypes.byref(d["nav_settings"]), *[p for _, p in outs], None))
    return [o for o, _ in outs]


def _nav_velocity(b, ops, d, packed):
    from softgnss_python_b200 import _native
    nav = b.nav()
    active, sol = nav[6], nav[7]
    a, off, stride = _rows(d["trk"], FIELD["carrFreq"], packed)
    r, c, e = d["r"], d["c"], d["max_ep"]
    vs = _native.SgxVelSettings(IF=IF, c=299792458.0, f_L1=1575.42e6, nav_sol_period=500.0, doppler_avg_ms=100)
    outs = [ops.out((r, e, 8)), ops.out((r, e, c)), ops.out((r, e, c)), ops.out((r, e, c, 3)), ops.out((r, e, c))]
    b.check(b.lib.dll.sgx_nav_velocity(ops.inp(a, off), stride, r, c, d["ms"], d["ms_done"].ctypes.data,
                                       ops.inp(d["sfs"]), ops.inp(d["eph"]), ops.inp(d["tow"]), ops.inp(d["n_ep"]), e,
                                       ops.inp(active), ops.inp(sol), ctypes.byref(vs), *[p for _, p in outs], None))
    return [o for o, _ in outs]


CALLS = dict(find_preambles=_find_preambles, pseudoranges=_pseudoranges, track_quality=_track_quality,
             nav_solve=_nav_solve, nav_velocity=_nav_velocity)


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
    monkeypatch.delenv("SGX_EMUL_HOST", raising=False)


def _same(got, want, label):
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape and g.tobytes() == w.tobytes(), "%s: output %d differs" % (label, k)


# ---------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_host_and_device_operands_agree(backend, entry):
    """Every host / device combination of inputs and outputs the entry point accepts gives the all-host result bit
    for bit, with the series read in place from the tracking result."""
    ref = backend.run(entry)
    if entry == "find_preambles":
        assert (ref[0] > 0).sum() >= 8, "too few preambles found to compare"
    if entry == "nav_solve":
        assert np.isfinite(ref[7][..., 0]).sum() >= 20, "too few fixes to compare"
    for host_in, host_out in backend.kinds:
        _same(backend.run(entry, host_in=host_in, host_out=host_out), ref,
              "%s %s host_in=%s host_out=%s" % (backend.name, entry, host_in, host_out))


@pytest.mark.parametrize("entry", ENTRY_POINTS)
def test_field_view_equals_packed_rows(backend, entry):
    """A series taken as one field of the [R, C, 13, ms] result (stride 13 * ms) gives the result of the same rows
    packed (for sgx_pseudoranges: of an array that holds field 0 and NaN elsewhere), host and device operands."""
    for host in (True, False):
        _same(backend.run(entry, packed=False, host_in=host, host_out=host),
              backend.run(entry, packed=True, host_in=host, host_out=host),
              "%s %s host=%s" % (backend.name, entry, host))


@pytest.mark.gpu
def test_find_preambles_without_bits_leaves_valid_untouched():
    """nav_bits = NULL: nav_bits_valid (here host memory) is not written, and the call succeeds."""
    from softgnss_python_b200 import _native
    L = _native.lib()
    L.require_device()
    _check_find_preambles_without_bits(L, inputs()["trk"])


def _check_find_preambles_without_bits(L, trk):
    ms = trk.shape[-1]
    n = trk.shape[0] * trk.shape[1]
    first = np.full(n, -1, dtype=np.int32)
    valid = np.full(n, 7, dtype=np.int32)
    rc = L.dll.sgx_find_preambles(trk.ctypes.data + 8 * 3 * ms, NF * ms, n, ms, first.ctypes.data, None,
                                  valid.ctypes.data, None)
    assert rc == 0, L.dll.sgx_last_error().decode()
    assert (valid == 7).all() and (first > 0).any()


@pytest.mark.emul
def test_host_staging_reads_only_the_documented_rows():
    """CPU emulator, host operands: the tracking result ends right before an inaccessible page and every row-taking
    entry point reads a field view of it (plus sgx_find_preambles without nav_bits).  Run in a child process: a read
    past the documented rows kills the child, not the session."""
    if os.environ.get("SGX_EMUL_TESTS") != "1" or not os.path.exists(EMUL_LIB):
        pytest.skip("CPU emulator tests: set SGX_EMUL_TESTS=1 and build %s with tools/cpu_emul/build_emul.sh" % EMUL_LIB)
    env = dict(os.environ, SGX_EMUL_HOST="1")
    p = subprocess.run([sys.executable, "-c", "from tests import test_operand_staging as t; t._guarded_calls()"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    assert p.returncode == 0, "child exited with %d\n%s%s" % (p.returncode, p.stdout, p.stderr[-4000:])
    assert p.stdout.strip().endswith("all calls returned")


def _guarded_calls():
    """Child process of the test above (SGX_EMUL_HOST=1, emulator library only: a bounds check on host memory)."""
    assert os.environ.get("SGX_EMUL_HOST") == "1"
    from softgnss_python_b200 import _native
    L = _native.Lib(EMUL_LIB)
    d = inputs()
    page = mmap.PAGESIZE
    nbytes = d["trk"].nbytes
    size = (nbytes + page - 1) // page * page
    buf = mmap.mmap(-1, size + page)
    base = ctypes.addressof(ctypes.c_char.from_buffer(buf))
    libc = ctypes.CDLL(None, use_errno=True)
    libc.mprotect.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    assert libc.mprotect(base + size, page, 0) == 0, os.strerror(ctypes.get_errno())       # PROT_NONE
    guarded = np.frombuffer(buf, dtype=np.float64, count=nbytes // 8, offset=size - nbytes).reshape(d["trk"].shape)
    trk = d["trk"]
    b = Backend("emul", L)
    b.nav()                                      # sgx_nav_velocity's active and sol
    # each stage's series moved to the last fields, so that the last row of each ends right at the inaccessible page
    moves = (("find_preambles", dict(I_P=NF - 1)), ("pseudoranges", {}), ("track_quality", dict(I_P=NF - 2, Q_P=NF - 1)),
             ("nav_solve", dict(absoluteSample=NF - 1)), ("nav_velocity", dict(carrFreq=NF - 1)))
    home = dict(FIELD)
    for entry, moved in moves:
        FIELD.update(home, **moved)
        guarded[...] = np.nan
        for name, f in FIELD.items():
            guarded[:, :, f] = trk[:, :, home[name]]
        d["trk"] = guarded
        b.run(entry)
        print(entry, "ok", flush=True)
    _check_find_preambles_without_bits(L, guarded)       # I_P is field 3 again after nav_velocity's move
    print("all calls returned", flush=True)
