"""The drop-in modules resolve under the reference's module names and expose the surface its caller
uses (initialize.py:456-507, postNavigation.py:9-12).  CPU only, no compute."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_module_names_resolve_in_a_clean_interpreter(tmp_path):
    code = ("import sys; sys.path.insert(0, %r); import acquisition, tracking; "
            "a = acquisition.AcquisitionResult; t = tracking.TrackingResult; "
            "print(all(hasattr(a, m) for m in ('acquire','preRun','showChannelStatus','plot','carrFreq','codePhase','peakMetric','channels','settings','results')), "
            "all(hasattr(t, m) for m in ('track','plot','results','channels','settings')), "
            "callable(acquisition.acquisition), callable(acquisition.preRun), callable(tracking.tracking))"
            % os.path.join(ROOT, "dropin"))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr
    assert out.stdout.split() == ["True"] * 5


def test_prerun_matches_reference_semantics():
    """acquisition.py:278-304: strongest detected PRNs first, idle channels PRN 0 / '-'."""
    from oracle import gnss_oracle as orc
    from softgnss_python_b200.acquisition import preRun
    from softgnss_python_b200.settings import Settings
    rng = np.random.default_rng(3)
    metric = rng.uniform(1, 10, 32)
    carr = np.where(metric > 6.0, 9.5e6 + rng.uniform(-5e3, 5e3, 32), 0.0)
    cph = np.where(carr > 0, rng.integers(0, 38192, 32).astype(float), 0.0)
    acq = np.rec.fromarrays([carr, cph, metric], names="carrFreq,codePhase,peakMetric")
    for nch in (4, 8, 16):
        s = Settings(numberOfChannels=nch)
        ch = preRun(acq, s)
        ref = orc.pre_run(dict(carrFreq=carr, codePhase=cph, peakMetric=metric), s)
        assert np.array_equal(ch.PRN, ref["PRN"]) and ch.PRN.dtype == np.int64
        assert np.array_equal(ch.acquiredFreq, ref["acquiredFreq"])
        assert np.array_equal(ch.codePhase, ref["codePhase"])
        assert list(ch.status) == ref["status"]


def test_results_setter_accepts_loaded_recarray():
    """initialize.py:504 assigns a np.load()ed recarray to TrackingResult.results."""
    from softgnss_python_b200.tracking import RESULT_DTYPE, TrackingResult

    class Acq(object):
        channels = np.rec.fromarrays([[1], [9.5e6], [0.0], ['T']], names="PRN,acquiredFreq,codePhase,status")
        settings = None
    t = TrackingResult(Acq())
    rec = np.recarray((0,), dtype=RESULT_DTYPE)
    t.results = rec
    assert t.results is rec
    try:
        t.results = [1, 2]
        raise RuntimeError("expected an AssertionError")
    except AssertionError:
        pass
