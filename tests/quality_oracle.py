"""Float64 oracle of the tracking-quality stage (sgx_track_quality, csrc/sgx_quality.cu)  --  TEST INFRASTRUCTURE ONLY.

An EXTENSION with no reference behaviour: the Python reference has neither a C/N0 estimator nor a lock detector
(later Matlab SoftGNSS releases compute the same variance-summing estimator in CNoVSM.m).  So, unlike
oracle/gnss_oracle.py, which restates the reference and is pinned against it, this module is a literal numpy
statement of the contract in include/softgnss_b200.h, for one channel row.
"""
import numpy as np


def cno_vsm(i, q, W, T):
    """Variance-summing-method C/N0 (dB-Hz) of every whole window of W prompt samples: Z = I^2 + Q^2,
    Zm = mean(Z), Zv = var(Z, ddof=1), Pav = sqrt(Zm^2 - Zv), Nv = 0.5 (Zm - Pav),
    cn0 = 10 log10(Pav / (2 Nv T)); NaN unless Zm^2 - Zv > 0 and Nv > 0."""
    i, q = np.asarray(i, dtype=np.float64), np.asarray(q, dtype=np.float64)
    n = len(i) // W
    z = (i[:n * W] ** 2 + q[:n * W] ** 2).reshape(n, W)
    zm = z.mean(axis=1)
    zv = z.var(axis=1, ddof=1)
    p2 = zm ** 2 - zv
    cn0 = np.full(n, np.nan)
    with np.errstate(invalid="ignore", divide="ignore"):
        pav = np.sqrt(p2)
        nv = 0.5 * (zm - pav)
        ok = (p2 > 0) & (nv > 0)
        cn0[ok] = 10 * np.log10(pav[ok] / (2 * nv[ok] * T))
    return cn0


def pll_lock(i, q, W):
    """Narrow-band carrier-lock indicator cos(2 dphi) of every whole window of W prompt samples:
    sum(I^2 - Q^2) / sum(I^2 + Q^2); NaN when the denominator is 0."""
    i, q = np.asarray(i, dtype=np.float64), np.asarray(q, dtype=np.float64)
    n = len(i) // W
    num = (i[:n * W] ** 2 - q[:n * W] ** 2).reshape(n, W).sum(axis=1)
    den = (i[:n * W] ** 2 + q[:n * W] ** 2).reshape(n, W).sum(axis=1)
    out = np.full(n, np.nan)
    ok = den != 0
    out[ok] = num[ok] / den[ok]
    return out
