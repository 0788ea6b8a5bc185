"""Float64 numpy statement of the RAIM contract of sgx_nav_integrity (include/softgnss_b200.h).

It lives under tests/ rather than in oracle/gnss_oracle.py, which restates the reference and is pinned against it: the
reference has no integrity monitoring.  Satellite positions, the Earth-rotation correction, togeod, tropo and cart2geo
are that oracle's; the 4x4 solves are LU (numpy.linalg.solve) and the tables come from scipy.
"""
import numpy as np

from oracle import gnss_oracle as orc

STATUS = ("NO_FIX", "UNAVAILABLE", "OK", "EXCLUDED", "FAULT")
NO_FIX, UNAVAILABLE, OK, EXCLUDED, FAULT = range(5)
FIELDS = ("X", "Y", "Z", "dt", "latitude", "longitude", "height", "q", "T", "dof", "qFinal", "HPL", "VPL", "status",
          "excluded", "nUsed")
MAX_DOF = 28


def tables(pfa=1e-5, pmd=1e-3, max_dof=MAX_DOF):
    """(thresh, pbias) with scipy: chi2.isf and the root of ncx2.cdf(T, dof, lambda) = pmd."""
    from scipy.optimize import brentq
    from scipy.stats import chi2, ncx2
    dof = np.arange(1, max_dof + 1)
    thresh = chi2.isf(pfa, dof)
    lam = np.array([brentq(lambda v: ncx2.cdf(thresh[k - 1], k, v) - pmd, 1e-6, 1e4, xtol=1e-13, rtol=1e-15)
                    for k in dof])
    return thresh, np.sqrt(lam)


def model(p, xs, obs, c, use_trop_corr):
    """(y, row) of one channel at p = (x, dt): the measurement model of the contract."""
    dtr = np.pi / 180
    x = p[:3]
    rot = orc.e_r_corr(np.linalg.norm(xs - x) / c, xs)
    trop = 0.0
    if use_trop_corr:
        _, el, _ = orc.topocent(x, rot - x)
        trop = orc.tropo(np.sin(el * dtr), 0.0, 1013.0, 293.0, 50.0, 0.0, 0.0, 0.0)
    d = rot - x
    rho = np.linalg.norm(d)
    return obs - rho - p[3] - trop, np.concatenate([-d / rho, [1.0]])


def residual_test(h, y, sigma, pbias, lat, lon):
    """Test of one set: dict(sse, e, omh (1 - h_j), w, sse_j, hpl, vpl, testable)."""
    n_mat = h.T.dot(h)
    xh = np.linalg.solve(n_mat, h.T.dot(y))
    e = y - h.dot(xh)
    sse = float(e.dot(e))
    z = np.linalg.solve(n_mat, h.T)                                   # [4, n]: columns N^-1 a_j
    omh = 1.0 - np.einsum("ij,ji->i", h, z)
    testable = omh > 1e-12
    s = np.sqrt(np.where(testable, omh, 1.0))
    sl, cl, sb, cb = np.sin(np.radians(lon)), np.cos(np.radians(lon)), np.sin(np.radians(lat)), np.cos(np.radians(lat))
    ze = -sl * z[0] + cl * z[1]
    zn = -sb * cl * z[0] - sb * sl * z[1] + cb * z[2]
    zu = cb * cl * z[0] + cb * sl * z[1] + sb * z[2]
    dof = h.shape[0] - 4
    scale = sigma * pbias[dof - 1] if dof >= 1 else np.nan
    if testable.all():
        hpl, vpl = scale * np.max(np.sqrt(ze ** 2 + zn ** 2) / s), scale * np.max(np.abs(zu) / s)
    else:
        hpl = vpl = np.inf
    w = np.where(testable, e / (sigma * s), np.nan)
    sse_j = np.where(testable, sse - e ** 2 / np.where(testable, omh, 1.0), np.inf)
    return dict(sse=sse, e=e, omh=omh, w=w, sse_j=sse_j, hpl=hpl, vpl=vpl, testable=testable, x=xh)


def epoch(raw_p, active, sol, eph, t, sigma, thresh, pbias, c=299792458.0, use_trop_corr=False):
    """One epoch.  raw_p, active [C]; sol [12]; eph [C, 21].  Returns (integ [16], norm_resid [C], detail dict with the
    all-in-view test ``t0`` and the candidate exclusion ``sse_j`` for margin checks)."""
    n_ch = len(active)
    out = np.full(16, np.nan)
    w_out = np.full(n_ch, np.nan)
    if not np.isfinite(sol[:4]).all():
        out[13:] = (NO_FIX, -1, 0)
        return out, w_out, {}
    chans = np.flatnonzero(active)
    n = len(chans)
    xs, obs = {}, {}
    for ch in chans:
        pos, clk = orc.satpos(t, [1], [dict(zip(orc.EPH_FIELDS, eph[ch]))])
        xs[ch], obs[ch] = pos[:, 0], raw_p[ch] + clk[0] * c
    out[:7] = sol[[0, 1, 2, 3, 9, 10, 11]]
    out[9] = n - 4
    out[13:] = (UNAVAILABLE, -1, n)
    if n < 5:
        return out, w_out, {}
    lat, lon = sol[9], sol[10]

    def evaluate(p, cs):
        ys, rows = zip(*[model(p, xs[ch], obs[ch], c, use_trop_corr) for ch in cs])
        return np.array(ys), np.array(rows)

    p0 = sol[:4].copy()
    y, h = evaluate(p0, chans)
    t0 = residual_test(h, y, sigma, pbias, lat, lon)
    dof = n - 4
    q = t0["sse"] / sigma ** 2
    out[7], out[8], out[10], out[11], out[12] = q, thresh[dof - 1], q, t0["hpl"], t0["vpl"]
    w_out[chans] = t0["w"]
    detail = dict(t0=t0, chans=chans, q=q, T=thresh[dof - 1])
    if q <= thresh[dof - 1]:
        out[13] = OK
        return out, w_out, detail
    out[13] = FAULT
    if n < 6:
        return out, w_out, detail
    k = int(np.argmin(t0["sse_j"]))                                   # first minimum: lowest channel
    detail["T1"] = thresh[dof - 2]
    if not t0["sse_j"][k] / sigma ** 2 <= thresh[dof - 2]:
        return out, w_out, detail
    s1 = np.delete(chans, k)
    p = p0.copy()
    for _ in range(6):
        y1, h1 = evaluate(p, s1)
        dx = np.linalg.solve(h1.T.dot(h1), h1.T.dot(y1))
        p = p + dx
        if np.linalg.norm(dx[:3]) < 1e-4:
            break
    y1, h1 = evaluate(p, s1)
    t1 = residual_test(h1, y1, sigma, pbias, lat, lon)
    out[:4] = p
    out[4:7] = orc.cart2geo(p[0], p[1], p[2], 4)
    out[10], out[11], out[12] = t1["sse"] / sigma ** 2, t1["hpl"], t1["vpl"]
    out[13:] = (EXCLUDED, chans[k], n - 1)
    detail["t1"] = t1
    return out, w_out, detail


def nav_integrity(raw_p, active, sol, eph, tow, n_epochs, sigma, thresh, pbias, c=299792458.0, nav_sol_period=500.0,
                  use_trop_corr=False):
    """One recording: raw_p, active [E, C]; sol [E, 12]; eph [C, 21].  Returns (integ [E, 16], norm_resid [E, C],
    details [E])."""
    n_ep_max, n_ch = active.shape
    integ = np.full((n_ep_max, 16), np.nan)
    integ[:, 13:] = (NO_FIX, -1, 0)
    w = np.full((n_ep_max, n_ch), np.nan)
    details = [{} for _ in range(n_ep_max)]
    t = tow
    for ep in range(min(n_epochs, n_ep_max)):
        integ[ep], w[ep], details[ep] = epoch(raw_p[ep], active[ep], sol[ep], eph, t, sigma, thresh, pbias, c,
                                              use_trop_corr)
        t += nav_sol_period / 1000
    return integ, w, details
