"""Float64 numpy statement of the receiver velocity / clock-drift contract of sgx_nav_velocity (include/softgnss_b200.h).

It lives under tests/ rather than in oracle/gnss_oracle.py, which restates the reference and is pinned against it: the
reference computes no velocity.  Satellite positions come from that oracle's ``satpos``; their time derivatives are
written out here.
"""
import numpy as np

from oracle import gnss_oracle as orc

OMEGAE_DOT = 7.2921151467e-05     # satpos (geoFunctions/__init__.py:803)
OMEGA_TAU = 7.292115147e-05       # e_r_corr (geoFunctions/__init__.py:508)
F_REL = -4.442807633e-10
VEL_FIELDS = ("VX", "VY", "VZ", "clkDrift", "VE", "VN", "VU", "nUsed")


def sat_state(transmit_time, e):
    """Position, clock correction, velocity and clock drift of one satellite.  ``e``: mapping with the EPH_FIELDS keys.
    Returns (pos [3], clk, vel [3], clk_drift)."""
    pos, clk = orc.satpos(transmit_time, [1], [e])
    e = {k: np.float64(e[k]) for k in orc.EPH_FIELDS}
    gps_pi = 3.14159265359
    dt = orc.check_t(transmit_time - e["t_oc"])
    c0 = (e["a_f2"] * dt + e["a_f1"]) * dt + e["a_f0"] - e["T_GD"]
    a = e["sqrtA"] * e["sqrtA"]
    tk = orc.check_t(transmit_time - c0 - e["t_oe"])
    n = np.sqrt(3.986005e+14 / a ** 3) + e["deltan"]
    m = np.remainder(e["M_0"] + n * tk + 2 * gps_pi, 2 * gps_pi)
    ea = m
    for _ in range(10):
        old = ea
        ea = m + e["e"] * np.sin(ea)
        if abs(np.remainder(ea - old, 2 * gps_pi)) < 1e-12:
            break
    ea = np.remainder(ea + 2 * gps_pi, 2 * gps_pi)
    nu = np.arctan2(np.sqrt(1 - e["e"] ** 2) * np.sin(ea), np.cos(ea) - e["e"])
    phi = np.remainder(nu + e["omega"], 2 * gps_pi)
    c2, s2 = np.cos(2 * phi), np.sin(2 * phi)
    u = phi + e["C_uc"] * c2 + e["C_us"] * s2
    r = a * (1 - e["e"] * np.cos(ea)) + e["C_rc"] * c2 + e["C_rs"] * s2
    inc = e["i_0"] + e["iDot"] * tk + e["C_ic"] * c2 + e["C_is"] * s2
    om = np.remainder(e["omega_0"] + (e["omegaDot"] - OMEGAE_DOT) * tk - OMEGAE_DOT * e["t_oe"] + 2 * gps_pi, 2 * gps_pi)
    # derivatives
    ea_dot = n / (1 - e["e"] * np.cos(ea))
    nu_dot = ea_dot * np.sqrt(1 - e["e"] ** 2) / (1 - e["e"] * np.cos(ea))
    u_dot = nu_dot * (1 + 2 * (e["C_us"] * c2 - e["C_uc"] * s2))
    r_dot = a * e["e"] * np.sin(ea) * ea_dot + 2 * nu_dot * (e["C_rs"] * c2 - e["C_rc"] * s2)
    i_dot = e["iDot"] + 2 * nu_dot * (e["C_is"] * c2 - e["C_ic"] * s2)
    om_dot = e["omegaDot"] - OMEGAE_DOT
    xp, yp = r * np.cos(u), r * np.sin(u)
    xp_dot = r_dot * np.cos(u) - r * np.sin(u) * u_dot
    yp_dot = r_dot * np.sin(u) + r * np.cos(u) * u_dot
    co, so, ci, si = np.cos(om), np.sin(om), np.cos(inc), np.sin(inc)
    vel = np.array([xp_dot * co - xp * so * om_dot - yp_dot * ci * so + yp * si * i_dot * so - yp * ci * co * om_dot,
                    xp_dot * so + xp * co * om_dot + yp_dot * ci * co - yp * si * i_dot * co - yp * ci * so * om_dot,
                    yp_dot * si + yp * ci * i_dot])
    clk_drift = e["a_f1"] + 2 * e["a_f2"] * dt + F_REL * e["e"] * e["sqrtA"] * np.cos(ea) * ea_dot
    return pos[:, 0], clk[0], vel, clk_drift


def nav_velocity(carr_freq, ms_done, sub_frame_start, eph, tow, n_epochs, active, sol, IF, c=299792458.0,
                 f_l1=1575.42e6, nav_sol_period=500.0, doppler_avg_ms=100):
    """One recording.  ``carr_freq`` [C, ms]; ``ms_done`` [C]; ``sub_frame_start`` [C]; ``eph`` [C, 21] in EPH_FIELDS
    order; ``active`` [E, C] and ``sol`` [E, 12]: the fix's outputs.  Returns dict(vel [E, 8], doppler [E, C],
    rrResid [E, C], satVel [E, C, 3], satClkDrift [E, C])."""
    carr_freq = np.asarray(carr_freq, dtype=np.float64)
    n_ch, ms = carr_freq.shape
    n_ep_max = sol.shape[0]
    nan = np.nan
    vel = np.full((n_ep_max, 8), nan)
    vel[:, 7] = 0.0
    out = dict(vel=vel, doppler=np.full((n_ep_max, n_ch), nan), rrResid=np.full((n_ep_max, n_ch), nan),
               satVel=np.full((n_ep_max, n_ch, 3), nan), satClkDrift=np.full((n_ep_max, n_ch), nan))
    transmit_time = tow
    for ep in range(min(n_epochs, n_ep_max)):
        rows, ys, used = [], [], []
        x_r = sol[ep, :3]
        for ch in range(n_ch):
            if not active[ep, ch]:
                continue
            e = dict(zip(orc.EPH_FIELDS, eph[ch]))
            xs, _, vs, clk_drift = sat_state(transmit_time, e)
            out["satVel"][ep, ch] = vs
            out["satClkDrift"][ep, ch] = clk_drift
            m = int(sub_frame_start[ch]) + int(nav_sol_period) * ep
            first = m - doppler_avg_ms + 1
            if first < 0 or m >= ms_done[ch]:
                continue
            s = 0.0
            for k in range(first, m + 1):                                   # increasing index order
                s += carr_freq[ch, k]
            d = s / doppler_avg_ms - IF
            if not np.isfinite(d):
                continue
            out["doppler"][ep, ch] = d
            used.append(ch)
            if np.isnan(x_r).any():
                continue
            tau = np.linalg.norm(xs - x_r) / c
            xs_rot = orc.e_r_corr(tau, xs)
            vs_rot = orc.e_r_corr(tau, vs)
            u = (xs_rot - x_r) / np.linalg.norm(xs_rot - x_r)
            rr = -(c / f_l1) * d
            rows.append(np.concatenate([-u, [1.0]]))
            ys.append(rr - u.dot(vs_rot) + c * clk_drift)
        vel[ep, 7] = len(used)
        if np.isnan(x_r).any() or len(used) < 4:
            transmit_time += nav_sol_period / 1000
            continue
        h = np.array(rows)
        y = np.array(ys)
        x = np.linalg.solve(h.T.dot(h), h.T.dot(y))
        lat, lon = np.radians(sol[ep, 9]), np.radians(sol[ep, 10])
        sl, cl, sb, cb = np.sin(lon), np.cos(lon), np.sin(lat), np.cos(lat)
        vel[ep, :4] = x
        vel[ep, 4] = -sl * x[0] + cl * x[1]
        vel[ep, 5] = -sb * cl * x[0] - sb * sl * x[1] + cb * x[2]
        vel[ep, 6] = cb * cl * x[0] + cb * sl * x[1] + sb * x[2]
        out["rrResid"][ep, used] = y - h.dot(x)
        transmit_time += nav_sol_period / 1000
    return out
