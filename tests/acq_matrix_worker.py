"""Worker of tests/test_gpu_acq_matrix.py: acquires the recordings of an input npz in a process of its own, with the
SGX_* path settings of its environment (the library reads several of them once per process, or only when it rebuilds
its plan), and writes the results into an output npz.

    python tests/acq_matrix_worker.py IN.npz OUT.npz [LIBRARY]

IN.npz holds `meta` (JSON: one dict(settings=..., nprn=...) per case) and `data<i>` (int8 [R, n_samples]); OUT.npz
gets `<field><i>` for every field of acquire_batch(..., diagnostics=True).  LIBRARY (optional) is the shared library
to load instead of the package's own, e.g. the CPU emulator build."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(inp, out, lib_path=None):
    from softgnss_python_b200 import _native
    from softgnss_python_b200.acquisition import acquire_batch
    from softgnss_python_b200.settings import Settings
    if lib_path:
        _native._LIB = _native.Lib(lib_path)
    z = np.load(inp)
    res = {}
    for i, m in enumerate(json.loads(str(z["meta"]))):
        s = Settings(**m["settings"])
        s.acqSatelliteList = range(1, m["nprn"] + 1)
        for f, v in acquire_batch(z["data%d" % i], s, diagnostics=True).items():
            res["%s%d" % (f, i)] = v
    np.savez(out, **res)


if __name__ == "__main__":
    main(*sys.argv[1:])
