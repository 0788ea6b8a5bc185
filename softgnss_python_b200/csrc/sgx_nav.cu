// Navigation solution on the device (SURVEY.md section 8(f) row 4, second half): the measurement loop of
// NavigationResult.postNavigate, batched over independent recordings.
//
// Replaces, for every recording and every measurement epoch,
//   postNavigation.py:199-301   elevation mask, channel list, transmit-time stepping, result bookkeeping
//   postNavigation.py:27-72     calculatePseudoranges (same expression order as pseudorange_kernel)
//   geoFunctions/__init__.py:779-885   satpos  (broadcast-ephemeris orbit + clock correction)
//   geoFunctions/__init__.py:636-739   leastSquarePos (7 Gauss-Newton iterations, DOP)
//   geoFunctions/__init__.py:491-521   e_r_corr, :892-1000 togeod, :1003-1063 topocent, :1071-1169 tropo
//   geoFunctions/__init__.py:7-77      cart2geo (WGS84)
//
// Mapping: one warp per recording, lane = channel (n_channels <= 32).  Satellite positions, Earth-rotation
// correction, topocentric angles and the tropospheric delay of the channels run in parallel on the lanes; the
// 4x4 normal equations are formed with warp reductions and solved redundantly by every lane.  Epochs are
// sequential inside a recording because the elevation mask of epoch k uses the elevations of epoch k-1
// (postNavigation.py:201, :241); recordings are independent, so the batch fills the GPU with warps.
// All arithmetic is float64 in the reference's operation order (the translation unit is built with
// -fmad=false); what differs from numpy is the last-ulp rounding of sin/cos/atan2/pow and the solver of the
// 8x4 least-squares step (Cholesky on the normal equations instead of LAPACK gelsd) -- see DESIGN.md for
// the tolerance this gives (1e-5 m on the fix).
//
// nav_velocity_kernel (K10, an extension with no reference behaviour) reuses satpos_one and the helpers above: receiver
// velocity and clock drift at the same epochs from the PLL's carrier frequency, one warp per (recording, epoch).
// nav_integrity_kernel (K11, likewise an extension) runs a RAIM residual test on each fix, excludes one faulty channel
// and gives protection levels, one warp per (recording, epoch), post hoc (nothing feeds back into K8).
#include <math.h>

#include "sgx_common.cuh"

namespace sgx {

struct NavArgs {
  const double* abs_sample;   // row (r, c) = abs_sample + (r*n_ch + c)*stride, ms values
  long long stride;
  const int* sub_frame_start; // [R][C]
  const unsigned char* ready; // [R][C]
  const sgx_eph* eph;         // [R][C]
  const double* tow;          // [R]
  const int* n_epochs;        // [R]
  int n_rec, n_ch, ms, max_epochs;
  sgx_nav_settings st;
  double* raw_p;              // [R][E][C]
  double* corrected_p;        // [R][E][C]
  double* el;                 // [R][E][C]
  double* az;                 // [R][E][C]
  double* sat_pos;            // [R][E][C][3] or null
  double* sat_clk;            // [R][E][C] or null
  unsigned char* active;      // [R][E][C]
  double* sol;                // [R][E][SGX_NAV_SOL_FIELDS]
};

__device__ __forceinline__ double nan_f64() { return __longlong_as_double(0x7ff8000000000000LL); }
__device__ __forceinline__ double inf_f64() { return __longlong_as_double(0x7ff0000000000000LL); }

// numpy.remainder for a positive divisor: result in [0, y)
__device__ __forceinline__ double py_mod(double x, double y) {
  double r = fmod(x, y);
  if (r != 0.0 && r < 0.0) r += y;
  return r;
}

__device__ __forceinline__ double check_t(double t) {   // geoFunctions/__init__.py:745-771
  const double half_week = 302400.0;
  if (t > half_week) return t - 2 * half_week;
  if (t < -half_week) return t + 2 * half_week;
  return t;
}

// geoFunctions/__init__.py:779-885 for one satellite
__device__ void satpos_one(double transmit_time, const sgx_eph& e, double xs[3], double& clk) {
  const double gps_pi = 3.14159265359, omegae_dot = 7.2921151467e-05, gm = 3.986005e+14, f_rel = -4.442807633e-10;
  const double two_pi = 2 * gps_pi;
  const double dt = check_t(transmit_time - e.t_oc);
  clk = (e.a_f2 * dt + e.a_f1) * dt + e.a_f0 - e.T_GD;
  const double time = transmit_time - clk;
  const double a = e.sqrtA * e.sqrtA;
  const double tk = check_t(time - e.t_oe);
  const double n0 = sqrt(gm / (a * a * a));
  const double n = n0 + e.deltan;
  double m = e.M_0 + n * tk;
  m = py_mod(m + two_pi, two_pi);
  double ea = m;
  for (int i = 0; i < 10; ++i) {
    const double old = ea;
    ea = m + e.e * sin(ea);
    const double d = py_mod(ea - old, two_pi);
    if (fabs(d) < 1e-12) break;
  }
  ea = py_mod(ea + two_pi, two_pi);
  double se, ce;
  sincos(ea, &se, &ce);
  const double dtr = f_rel * e.e * e.sqrtA * se;
  const double nu = atan2(sqrt(1 - e.e * e.e) * se, ce - e.e);
  double phi = nu + e.omega;
  phi = py_mod(phi, two_pi);
  double s2, c2;
  sincos(2 * phi, &s2, &c2);
  const double u = phi + e.C_uc * c2 + e.C_us * s2;
  const double r = a * (1 - e.e * ce) + e.C_rc * c2 + e.C_rs * s2;
  const double inc = e.i_0 + e.iDot * tk + e.C_ic * c2 + e.C_is * s2;
  double om = e.omega_0 + (e.omegaDot - omegae_dot) * tk - omegae_dot * e.t_oe;
  om = py_mod(om + two_pi, two_pi);
  double su, cu, so, co, si, ci;
  sincos(u, &su, &cu);
  sincos(om, &so, &co);
  sincos(inc, &si, &ci);
  xs[0] = cu * r * co - su * r * ci * so;
  xs[1] = cu * r * so + su * r * ci * co;
  xs[2] = su * r * si;
  clk = (e.a_f2 * dt + e.a_f1) * dt + e.a_f0 - e.T_GD + dtr;
}

// geoFunctions/__init__.py:892-1000 with a = 6378137, finv = 298.257223563; degrees out
__device__ void togeod(double x, double y, double z, double& dphi, double& dlambda, double& h) {
  const double a = 6378137.0, finv = 298.257223563, rtd = 180 / 3.141592653589793;
  const double esq = (2 - 1 / finv) / finv, oneesq = 1 - esq;
  const double p = sqrt(x * x + y * y);
  dlambda = p > 1e-20 ? atan2(y, x) * rtd : 0.0;
  if (dlambda < 0) dlambda += 360;
  const double r = sqrt(p * p + z * z);
  double sinphi = r > 1e-20 ? z / r : 0.0;
  dphi = asin(sinphi);
  if (r < 1e-20) { h = 0.0; return; }
  h = r - a * (1 - sinphi * sinphi / finv);
  for (int i = 0; i < 10; ++i) {
    double cosphi;
    sincos(dphi, &sinphi, &cosphi);
    const double n_phi = a / sqrt(1 - esq * sinphi * sinphi);
    const double d_p = p - (n_phi + h) * cosphi;
    const double d_z = z - (n_phi * oneesq + h) * sinphi;
    h = h + sinphi * d_z + cosphi * d_p;
    dphi = dphi + (cosphi * d_z - sinphi * d_p) / (n_phi + h);
    if (d_p * d_p + d_z * d_z < 1e-10) break;
  }
  dphi *= rtd;
}

// geoFunctions/__init__.py:1071-1169 called as tropo(sinel, 0, 1013, 293, 50, 0, 0, 0) (:697)
__device__ double tropo(double sinel, double hsta, double p, double tkel, double hum, double hp, double htkel,
                        double hhum) {
  const double a_e = 6378.137, b0 = 7.839257e-05, tlapse = -6.5;
  const double tkhum = tkel + tlapse * (hhum - htkel);
  const double atkel = 7.5 * (tkhum - 273.15) / (237.3 + tkhum - 273.15);
  const double e0 = 0.0611 * hum * pow(10.0, atkel);
  const double tksea = tkel - tlapse * htkel;
  const double em = -978.77 / (2870400.0 * tlapse * 1e-05);
  const double tkelh = tksea + tlapse * hhum;
  const double e0sea = e0 * pow(tksea / tkelh, 4 * em);
  const double tkelp = tksea + tlapse * hp;
  const double psea = p * pow(tksea / tkelp, em);
  if (sinel < 0) sinel = 0;
  double total = 0.0;
  double refsea = 7.7624e-05 / tksea;
  double htop = 1.1385e-05 / refsea;
  refsea = refsea * psea;
  double q = (htop - hsta) / htop;
  double ref = refsea * ((q * q) * (q * q));
  for (int pass = 0; pass < 2; ++pass) {
    double rtop = (a_e + htop) * (a_e + htop) - (a_e + hsta) * (a_e + hsta) * (1 - sinel * sinel);
    if (rtop < 0) rtop = 0;
    rtop = sqrt(rtop) - (a_e + hsta) * sinel;
    const double a = -sinel / (htop - hsta);
    const double b = -b0 * (1 - sinel * sinel) / (htop - hsta);
    const double a2 = a * a, b2 = b * b;
    double alpha[8];
    alpha[0] = 2 * a;
    alpha[1] = 2 * a2 + 4 * b / 3;
    alpha[2] = a * (a2 + 3 * b);
    alpha[3] = (a2 * a2) / 5 + 2.4 * a2 * b + 1.2 * b2;
    alpha[4] = 2 * a * b * (a2 + 3 * b) / 3;
    alpha[5] = b2 * (6 * a2 + 4 * b) * 0.1428571;
    alpha[6] = 0;
    alpha[7] = 0;
    if (b2 > 1e-35) {
      alpha[6] = a * (b2 * b) / 2;
      alpha[7] = (b2 * b2) / 9;
    }
    double rn = rtop * rtop, dot = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      dot += alpha[i] * rn;
      rn *= rtop;
    }
    const double dr = rtop + dot;
    total += dr * ref * 1000;
    if (pass == 0) {
      refsea = (0.3719 / tksea - 1.292e-05) / tksea;
      htop = 1.1385e-05 * (1255.0 / tksea + 0.05) / refsea;
      q = (htop - hsta) / htop;
      ref = refsea * e0sea * ((q * q) * (q * q));
    }
  }
  return total;
}

// geoFunctions/__init__.py:7-77, ellipsoid 4 (WGS84)
__device__ void cart2geo(double x, double y, double z, double& lat, double& lon, double& hh) {
  const double a = 6378137.0, f = 1 / 298.257223563, rtd = 180 / 3.141592653589793;
  const double lambda = atan2(y, x);
  const double ex2 = (2 - f) * f / ((1 - f) * (1 - f));
  const double c = a * sqrt(1 + ex2);
  const double pxy = sqrt(x * x + y * y);
  double phi = atan(z / (pxy * (1 - (2 - f)) * f));
  double h = 0.1, oldh = 0;
  int it = 0;
  while (fabs(h - oldh) > 1e-12) {
    oldh = h;
    const double cp = cos(phi);
    const double n = c / sqrt(1 + ex2 * (cp * cp));
    phi = atan(z / (pxy * (1 - (2 - f) * f * n / (n + h))));
    h = pxy / cos(phi) - n;
    if (++it > 100) break;
  }
  lat = phi * rtd;
  lon = lambda * rtd;
  hh = h;
}

__device__ __forceinline__ double warp_add(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

// Solve the symmetric positive definite 4x4 system n x = b (upper triangle in n[10]: 00 01 02 03 11 12 13 22 23 33)
// by Cholesky; optionally returns the diagonal of n^-1.  false when a pivot is not positive (rank < 4).
__device__ bool chol4(const double n[10], const double b[4], double x[4], double qdiag[4]) {
  double l[4][4];
  const double m[4][4] = {{n[0], n[1], n[2], n[3]}, {n[1], n[4], n[5], n[6]}, {n[2], n[5], n[7], n[8]}, {n[3], n[6], n[8], n[9]}};
  const double tiny = 1e-13 * (n[0] + n[4] + n[7] + n[9]);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double d = m[j][j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= l[j][k] * l[j][k];
    if (!(d > tiny)) return false;
    l[j][j] = sqrt(d);
#pragma unroll
    for (int i = j + 1; i < 4; ++i) {
      double s = m[i][j];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= l[i][k] * l[j][k];
      l[i][j] = s / l[j][j];
    }
  }
  double y[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    double s = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) s -= l[i][k] * y[k];
    y[i] = s / l[i][i];
  }
#pragma unroll
  for (int i = 3; i >= 0; --i) {
    double s = y[i];
#pragma unroll
    for (int k = i + 1; k < 4; ++k) s -= l[k][i] * x[k];
    x[i] = s / l[i][i];
  }
  if (qdiag) {
    // columns of L^-1 (lower triangular); diag(n^-1)[i] = sum_k Linv[k][i]^2
    double li[4][4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        if (r < c) { li[r][c] = 0.0; continue; }
        double s = (r == c) ? 1.0 : 0.0;
#pragma unroll
        for (int k = c; k < r; ++k) s -= l[r][k] * li[k][c];
        li[r][c] = s / l[r][r];
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double s = 0.0;
#pragma unroll
      for (int k = i; k < 4; ++k) s += li[k][i] * li[k][i];
      qdiag[i] = s;
    }
  }
  return true;
}

__global__ void __launch_bounds__(128) nav_solve_kernel(NavArgs a) {
  const int rec = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (rec >= a.n_rec) return;
  const int C = a.n_ch;
  const bool mine = lane < C;
  const long long rc = (long long)rec * C + lane;
  const double* abs_row = a.abs_sample + rc * a.stride;
  const int sfs = mine ? a.sub_frame_start[rc] : 0;
  const bool ready = mine && a.ready[rc] != 0;
  sgx_eph e;
  if (ready) e = a.eph[rc];
  const int n_ep = min(a.n_epochs[rec], a.max_epochs);
  const double c_light = a.st.c, dtr_deg = 3.141592653589793 / 180;
  const int period = (int)a.st.nav_sol_period;
  double sat_elev = inf_f64();                       // postNavigation.py:159
  double transmit_time = a.tow[rec];                 // :168

  for (int ep = 0; ep < a.max_epochs; ++ep) {
    const long long o = ((long long)rec * a.max_epochs + ep) * C + lane;
    double* sol = a.sol + ((long long)rec * a.max_epochs + ep) * SGX_NAV_SOL_FIELDS;
    if (ep >= n_ep) {                                // columns the reference leaves at their initial values
      if (mine) {
        a.raw_p[o] = nan_f64(); a.corrected_p[o] = nan_f64(); a.el[o] = nan_f64(); a.az[o] = nan_f64();
        a.active[o] = 0;
        if (a.sat_clk) a.sat_clk[o] = nan_f64();
        if (a.sat_pos) { a.sat_pos[o * 3] = nan_f64(); a.sat_pos[o * 3 + 1] = nan_f64(); a.sat_pos[o * 3 + 2] = nan_f64(); }
      }
      if (lane < SGX_NAV_SOL_FIELDS) sol[lane] = (lane >= 4 && lane < 9) ? 0.0 : nan_f64();
      continue;
    }
    // ---- :201 channel list of this epoch ---------------------------------------------------------
    const int idx = sfs + period * ep;
    const bool act = ready && (sat_elev >= a.st.elevation_mask) && idx >= 0 && idx < a.ms;
    const unsigned act_mask = __ballot_sync(0xffffffffu, act);
    const int n_act = __popc(act_mask);
    // ---- :212 calculatePseudoranges (postNavigation.py:52-71) -------------------------------------
    double t = inf_f64();
    if (act) t = abs_row[idx] / a.st.samples_per_code;
    double mn = t;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, d));
    const double raw_p = ((t - floor(mn)) + a.st.start_offset) * c_light / 1000.0;
    // ---- :217 satpos --------------------------------------------------------------------------------
    double xs[3] = {0.0, 0.0, 0.0}, clk = 0.0;
    if (act) satpos_one(transmit_time, e, xs, clk);
    double el = nan_f64(), az = nan_f64(), corrected = nan_f64();
    double pos[4] = {0.0, 0.0, 0.0, 0.0}, dop[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
    double lat = nan_f64(), lon = nan_f64(), hgt = nan_f64();
    bool fix = false;
    if (n_act > 3) {                                   // :222
      // ---- leastSquarePos (geoFunctions/__init__.py:636-739) ---------------------------------------
      const double obs = raw_p + clk * c_light;        // :228-230
      double el_i = 0.0, az_i = 0.0;                   // np.zeros (:652-654)
      double nrm[10], rhs[4], arow[4] = {0.0, 0.0, 0.0, 0.0};
      bool ok = true;
      for (int it = 0; it < 7 && ok; ++it) {
        double omc = 0.0;
        if (act) {
          double rot[3], trop;
          if (it == 0) {
            rot[0] = xs[0]; rot[1] = xs[1]; rot[2] = xs[2];
            trop = 2;                                  // :683
          } else {
            const double dx0 = xs[0] - pos[0], dx1 = xs[1] - pos[1], dx2 = xs[2] - pos[2];
            const double rho2 = dx0 * dx0 + dx1 * dx1 + dx2 * dx2;
            const double traveltime = sqrt(rho2) / c_light;
            const double omegatau = 7.292115147e-05 * traveltime;      // e_r_corr's own constant (:508)
            double so, co;
            sincos(omegatau, &so, &co);
            rot[0] = co * xs[0] + so * xs[1] + 0.0 * xs[2];
            rot[1] = -so * xs[0] + co * xs[1] + 0.0 * xs[2];
            rot[2] = 0.0 * xs[0] + 0.0 * xs[1] + 1.0 * xs[2];
            // topocent(pos, rot - pos)
            double phi, lam, hh;
            togeod(pos[0], pos[1], pos[2], phi, lam, hh);
            double sl, cl, sb, cb;
            sincos(lam * dtr_deg, &sl, &cl);
            sincos(phi * dtr_deg, &sb, &cb);
            const double d0 = rot[0] - pos[0], d1 = rot[1] - pos[1], d2 = rot[2] - pos[2];
            const double E = -sl * d0 + cl * d1 + 0.0 * d2;
            const double N = (-sb * cl) * d0 + (-sb * sl) * d1 + cb * d2;
            const double U = (cb * cl) * d0 + (cb * sl) * d1 + sb * d2;
            const double hor = sqrt(E * E + N * N);
            if (hor < 1e-20) { az_i = 0.0; el_i = 90.0; }
            else { az_i = atan2(E, N) / dtr_deg; el_i = atan2(U, hor) / dtr_deg; }
            if (az_i < 0) az_i += 360;
            trop = a.st.use_trop_corr ? tropo(sin(el_i * dtr_deg), 0.0, 1013.0, 293.0, 50.0, 0.0, 0.0, 0.0) : 0.0;
          }
          const double d0 = rot[0] - pos[0], d1 = rot[1] - pos[1], d2 = rot[2] - pos[2];
          omc = obs - sqrt(d0 * d0 + d1 * d1 + d2 * d2) - pos[3] - trop;          // :704
          arow[0] = -d0 / obs; arow[1] = -d1 / obs; arow[2] = -d2 / obs; arow[3] = 1.0;   // :706-709 (divided by obs)
        }
        int k = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
#pragma unroll
          for (int j = i; j < 4; ++j) nrm[k++] = warp_add(arow[i] * arow[j]);
          rhs[i] = warp_add(arow[i] * omc);
        }
        double x[4];
        ok = chol4(nrm, rhs, x, nullptr);               // :712-717
        if (ok) {
#pragma unroll
          for (int i = 0; i < 4; ++i) pos[i] = pos[i] + x[i];
        }
      }
      if (ok) {
        double x[4], q[4];
        ok = chol4(nrm, rhs, x, q);                     // Q = inv(A'A) of the last iteration (:726)
        dop[0] = sqrt(q[0] + q[1] + q[2] + q[3]);
        dop[1] = sqrt(q[0] + q[1] + q[2]);
        dop[2] = sqrt(q[0] + q[1]);
        dop[3] = sqrt(q[2]);
        dop[4] = sqrt(q[3]);
      } else {                                          // rank-deficient geometry: pos = 0, dop = 0 (:712-715)
        pos[0] = pos[1] = pos[2] = pos[3] = 0.0;
      }
      if (act) { el = el_i; az = az_i; }
      fix = true;
      sat_elev = el;                                    // :241 (NaN for channels outside the list)
      if (act) corrected = raw_p + clk * c_light + pos[3];   // :243-245
      cart2geo(pos[0], pos[1], pos[2], lat, lon, hgt);  // :249-254
    }
    // ---- results ---------------------------------------------------------------------------------
    if (mine) {
      a.raw_p[o] = raw_p;
      a.corrected_p[o] = corrected;
      a.el[o] = el;
      a.az[o] = az;
      a.active[o] = act ? 1 : 0;
      if (a.sat_clk) a.sat_clk[o] = act ? clk : nan_f64();
      if (a.sat_pos) {
        a.sat_pos[o * 3] = act ? xs[0] : nan_f64();
        a.sat_pos[o * 3 + 1] = act ? xs[1] : nan_f64();
        a.sat_pos[o * 3 + 2] = act ? xs[2] : nan_f64();
      }
    }
    if (lane == 0) {
      sol[0] = fix ? pos[0] : nan_f64(); sol[1] = fix ? pos[1] : nan_f64(); sol[2] = fix ? pos[2] : nan_f64();
      sol[3] = fix ? pos[3] : nan_f64();
#pragma unroll
      for (int i = 0; i < 5; ++i) sol[4 + i] = dop[i];
      sol[9] = lat; sol[10] = lon; sol[11] = hgt;
    }
    transmit_time += a.st.nav_sol_period / 1000;        // :298
  }
}

// ---- K10: receiver velocity and clock drift from the PLL's Doppler (extension; contract in softgnss_b200.h) -------
struct VelArgs {
  const double* carr_freq;    // row (r, c) = carr_freq + (r*n_ch + c)*stride, ms values
  long long stride;
  const int* ms_done;         // [R][C] or null (all ms)
  const int* sub_frame_start; // [R][C]
  const sgx_eph* eph;         // [R][C]
  const double* tow;          // [R]
  const int* n_epochs;        // [R]
  const unsigned char* active;// [R][E][C]
  const double* sol;          // [R][E][SGX_NAV_SOL_FIELDS]
  int n_rec, n_ch, ms, max_epochs;
  sgx_vel_settings st;
  double* vel;                // [R][E][SGX_NAV_VEL_FIELDS]
  double* doppler;            // [R][E][C]
  double* rr_resid;           // [R][E][C]
  double* sat_vel;            // [R][E][C][3] or null
  double* sat_clk_drift;      // [R][E][C] or null
};

// Time derivatives of satpos_one's position and clock at the same transmit time: its anomaly chain recomputed with the
// same expressions, then every term of the ECEF formulas differentiated (dt/dt of the transmit time taken as 1).
__device__ void satvel_one(double transmit_time, const sgx_eph& e, double vs[3], double& clk_drift) {
  const double gps_pi = 3.14159265359, omegae_dot = 7.2921151467e-05, gm = 3.986005e+14, f_rel = -4.442807633e-10;
  const double two_pi = 2 * gps_pi;
  const double dt = check_t(transmit_time - e.t_oc);
  double clk = (e.a_f2 * dt + e.a_f1) * dt + e.a_f0 - e.T_GD;
  const double time = transmit_time - clk;
  const double a = e.sqrtA * e.sqrtA;
  const double tk = check_t(time - e.t_oe);
  const double n = sqrt(gm / (a * a * a)) + e.deltan;
  double m = e.M_0 + n * tk;
  m = py_mod(m + two_pi, two_pi);
  double ea = m;
  for (int i = 0; i < 10; ++i) {
    const double old = ea;
    ea = m + e.e * sin(ea);
    const double d = py_mod(ea - old, two_pi);
    if (fabs(d) < 1e-12) break;
  }
  ea = py_mod(ea + two_pi, two_pi);
  double se, ce;
  sincos(ea, &se, &ce);
  const double nu = atan2(sqrt(1 - e.e * e.e) * se, ce - e.e);
  const double phi = py_mod(nu + e.omega, two_pi);
  double s2, c2;
  sincos(2 * phi, &s2, &c2);
  const double u = phi + e.C_uc * c2 + e.C_us * s2;
  const double r = a * (1 - e.e * ce) + e.C_rc * c2 + e.C_rs * s2;
  const double inc = e.i_0 + e.iDot * tk + e.C_ic * c2 + e.C_is * s2;
  double om = e.omega_0 + (e.omegaDot - omegae_dot) * tk - omegae_dot * e.t_oe;
  om = py_mod(om + two_pi, two_pi);
  const double one_m_ecose = 1 - e.e * ce;
  const double ea_dot = n / one_m_ecose;
  const double nu_dot = ea_dot * sqrt(1 - e.e * e.e) / one_m_ecose;
  const double u_dot = nu_dot * (1 + 2 * (e.C_us * c2 - e.C_uc * s2));
  const double r_dot = a * e.e * se * ea_dot + 2 * nu_dot * (e.C_rs * c2 - e.C_rc * s2);
  const double i_dot = e.iDot + 2 * nu_dot * (e.C_is * c2 - e.C_ic * s2);
  const double om_dot = e.omegaDot - omegae_dot;
  double su, cu, so, co, si, ci;
  sincos(u, &su, &cu);
  sincos(om, &so, &co);
  sincos(inc, &si, &ci);
  const double xp = r * cu, yp = r * su;                       // position in the orbital plane
  const double xp_dot = r_dot * cu - r * su * u_dot, yp_dot = r_dot * su + r * cu * u_dot;
  vs[0] = xp_dot * co - xp * so * om_dot - yp_dot * ci * so + yp * si * i_dot * so - yp * ci * co * om_dot;
  vs[1] = xp_dot * so + xp * co * om_dot + yp_dot * ci * co - yp * si * i_dot * co - yp * ci * so * om_dot;
  vs[2] = yp_dot * si + yp * ci * i_dot;
  clk_drift = e.a_f1 + 2 * e.a_f2 * dt + f_rel * e.e * e.sqrtA * ce * ea_dot;
}

// One warp per (recording, epoch), lane = channel.  Epochs are independent: K8's `active` already carries the
// elevation feedback between them.
__global__ void __launch_bounds__(128) nav_velocity_kernel(VelArgs a) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= (long long)a.n_rec * a.max_epochs) return;
  const int rec = (int)(warp / a.max_epochs), ep = (int)(warp % a.max_epochs);
  const int C = a.n_ch;
  const bool mine = lane < C;
  const long long o = warp * C + lane;                           // [R][E][C] index of (rec, ep, lane)
  double* vel = a.vel + warp * SGX_NAV_VEL_FIELDS;
  const int n_ep = min(a.n_epochs[rec], a.max_epochs);
  if (ep >= n_ep) {
    if (mine) {
      a.doppler[o] = nan_f64(); a.rr_resid[o] = nan_f64();
      if (a.sat_clk_drift) a.sat_clk_drift[o] = nan_f64();
      if (a.sat_vel) { a.sat_vel[o * 3] = nan_f64(); a.sat_vel[o * 3 + 1] = nan_f64(); a.sat_vel[o * 3 + 2] = nan_f64(); }
    }
    if (lane < SGX_NAV_VEL_FIELDS) vel[lane] = lane == 7 ? 0.0 : nan_f64();
    return;
  }
  const double* sol = a.sol + warp * SGX_NAV_SOL_FIELDS;
  const double c_light = a.st.c, dtr_deg = 3.141592653589793 / 180;
  double transmit_time = a.tow[rec];                             // advanced as nav_solve_kernel does, bit for bit
  for (int k = 0; k < ep; ++k) transmit_time += a.st.nav_sol_period / 1000;
  const bool act = mine && a.active[o] != 0;
  // ---- Doppler: mean of the N carrFreq values ending at the epoch's code period, summed in index order ------------
  double dop = nan_f64();
  if (act) {
    const long long rc = (long long)rec * C + lane;
    const int idx = a.sub_frame_start[rc] + (int)a.st.nav_sol_period * ep;
    const int first = idx - a.st.doppler_avg_ms + 1;
    const int done = a.ms_done ? a.ms_done[rc] : a.ms;
    if (first >= 0 && idx < done) {
      const double* row = a.carr_freq + rc * a.stride;
      double s = 0.0;
      for (int k = first; k <= idx; ++k) s += row[k];
      dop = s / a.st.doppler_avg_ms - a.st.IF;
    }
  }
  // ---- satellite state --------------------------------------------------------------------------------------------
  double xs[3] = {0.0, 0.0, 0.0}, vs[3] = {0.0, 0.0, 0.0}, clk = 0.0, clk_drift = 0.0;
  if (act) {
    const sgx_eph e = a.eph[(long long)rec * C + lane];
    satpos_one(transmit_time, e, xs, clk);
    satvel_one(transmit_time, e, vs, clk_drift);
  }
  const bool use = act && isfinite(dop);
  const int n_used = __popc(__ballot_sync(0xffffffffu, use));
  const double px = sol[0], py = sol[1], pz = sol[2];
  const bool fix = !isnan(px) && !isnan(py) && !isnan(pz);
  // ---- least squares on the 4x4 normal equations ------------------------------------------------------------------
  double row[4] = {0.0, 0.0, 0.0, 0.0}, y = 0.0, x[4] = {0.0, 0.0, 0.0, 0.0};
  bool ok = false;
  if (fix && n_used >= 4) {
    if (use) {
      const double d0 = xs[0] - px, d1 = xs[1] - py, d2 = xs[2] - pz;
      const double omegatau = 7.292115147e-05 * (sqrt(d0 * d0 + d1 * d1 + d2 * d2) / c_light);   // e_r_corr's constant
      double so, co;
      sincos(omegatau, &so, &co);
      const double rx0 = co * xs[0] + so * xs[1], rx1 = -so * xs[0] + co * xs[1], rx2 = xs[2];
      const double rv0 = co * vs[0] + so * vs[1], rv1 = -so * vs[0] + co * vs[1], rv2 = vs[2];
      const double l0 = rx0 - px, l1 = rx1 - py, l2 = rx2 - pz;
      const double rho = sqrt(l0 * l0 + l1 * l1 + l2 * l2);
      const double u0 = l0 / rho, u1 = l1 / rho, u2 = l2 / rho;
      const double rr = -(c_light / a.st.f_L1) * dop;
      y = rr - (u0 * rv0 + u1 * rv1 + u2 * rv2) + c_light * clk_drift;
      row[0] = -u0; row[1] = -u1; row[2] = -u2; row[3] = 1.0;
    }
    double nrm[10], rhs[4];
    int k = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int j = i; j < 4; ++j) nrm[k++] = warp_add(row[i] * row[j]);
      rhs[i] = warp_add(row[i] * y);
    }
    ok = chol4(nrm, rhs, x, nullptr);
  }
  // ---- results ------------------------------------------------------------------------------------------------------
  if (mine) {
    a.doppler[o] = use ? dop : nan_f64();
    a.rr_resid[o] = (ok && use) ? y - (row[0] * x[0] + row[1] * x[1] + row[2] * x[2] + row[3] * x[3]) : nan_f64();
    if (a.sat_clk_drift) a.sat_clk_drift[o] = act ? clk_drift : nan_f64();
    if (a.sat_vel) {
      a.sat_vel[o * 3] = act ? vs[0] : nan_f64();
      a.sat_vel[o * 3 + 1] = act ? vs[1] : nan_f64();
      a.sat_vel[o * 3 + 2] = act ? vs[2] : nan_f64();
    }
  }
  if (lane == 0) {
    if (ok) {
      double sl, cl, sb, cb;
      sincos(sol[10] * dtr_deg, &sl, &cl);
      sincos(sol[9] * dtr_deg, &sb, &cb);
      vel[0] = x[0]; vel[1] = x[1]; vel[2] = x[2]; vel[3] = x[3];
      vel[4] = -sl * x[0] + cl * x[1];
      vel[5] = (-sb * cl) * x[0] + (-sb * sl) * x[1] + cb * x[2];
      vel[6] = (cb * cl) * x[0] + (cb * sl) * x[1] + sb * x[2];
    } else {
      for (int i = 0; i < 7; ++i) vel[i] = nan_f64();
    }
    vel[7] = (double)n_used;
  }
}

// ---- K11: RAIM fault detection and exclusion, protection levels (extension; contract in softgnss_b200.h) ----------
struct IntegArgs {
  const double* raw_p;         // [R][E][C]
  const unsigned char* active; // [R][E][C]
  const double* sol;           // [R][E][SGX_NAV_SOL_FIELDS]
  const int* n_epochs;         // [R]
  const sgx_eph* eph;          // [R][C]
  const double* tow;           // [R]
  int n_rec, n_ch, max_epochs;
  sgx_nav_settings st;
  sgx_integ_settings is;
  double* integ;               // [R][E][SGX_NAV_INTEG_FIELDS]
  double* norm_resid;          // [R][E][C]
};

// Prefit residual y and row a = [-(xs_rot - x)/rho, 1] of one channel at p = (x, dt).  Unlike K8 the row is a true
// unit vector (K8 divides by obs, leastSquarePos's quirk), so N^-1 and the slopes below are those of the geometry.
__device__ void integ_model(const double p[4], const double xs[3], double obs, double c_light, bool trop_on, double& y,
                            double row[4]) {
  const double dtr_deg = 3.141592653589793 / 180;
  const double dx0 = xs[0] - p[0], dx1 = xs[1] - p[1], dx2 = xs[2] - p[2];
  const double omegatau = 7.292115147e-05 * (sqrt(dx0 * dx0 + dx1 * dx1 + dx2 * dx2) / c_light);   // e_r_corr
  double so, co;
  sincos(omegatau, &so, &co);
  const double r0 = co * xs[0] + so * xs[1], r1 = -so * xs[0] + co * xs[1], r2 = xs[2];
  const double d0 = r0 - p[0], d1 = r1 - p[1], d2 = r2 - p[2];
  double trop = 0.0;
  if (trop_on) {                                       // K8's topocent and tropo at x
    double phi, lam, hh;
    togeod(p[0], p[1], p[2], phi, lam, hh);
    double sl, cl, sb, cb;
    sincos(lam * dtr_deg, &sl, &cl);
    sincos(phi * dtr_deg, &sb, &cb);
    const double E = -sl * d0 + cl * d1;
    const double N = (-sb * cl) * d0 + (-sb * sl) * d1 + cb * d2;
    const double U = (cb * cl) * d0 + (cb * sl) * d1 + sb * d2;
    const double hor = sqrt(E * E + N * N);
    const double el = hor < 1e-20 ? 90.0 : atan2(U, hor) / dtr_deg;
    trop = tropo(sin(el * dtr_deg), 0.0, 1013.0, 293.0, 50.0, 0.0, 0.0, 0.0);
  }
  const double rho = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
  y = obs - rho - p[3] - trop;
  row[0] = -d0 / rho; row[1] = -d1 / rho; row[2] = -d2 / rho; row[3] = 1.0;
}

// N = sum a a^T and the solution of N x = sum a y over the lanes (lanes outside the set pass a = 0, y = 0).
__device__ __forceinline__ bool integ_normal(const double row[4], double y, double nrm[10], double x[4]) {
  double rhs[4];
  int k = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int j = i; j < 4; ++j) nrm[k++] = warp_add(row[i] * row[j]);
    rhs[i] = warp_add(row[i] * y);
  }
  return chol4(nrm, rhs, x, nullptr);
}

__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, d));
  return v;
}

// Residual test of the channel set {lanes with `use`} at the point the rows were evaluated at.  Per lane: the
// post-fit residual e and 1 - h (h = a . N^-1 a); for the set: SSE and the protection levels (+inf when a channel of
// the set is not testable).  ENU at (sl, cl) = sin, cos of the longitude and (sb, cb) of the latitude.  false when
// a Cholesky pivot of N is not above 1e-13 of its trace.
struct IntegTest {
  double sse, e, omh, hpl, vpl;
};

__device__ bool integ_test(bool use, double y, const double row[4], double sigma_pb, double sl, double cl, double sb,
                           double cb, IntegTest& t) {
  double nrm[10], xh[4], z[4];
  if (!integ_normal(row, y, nrm, xh)) return false;
  t.e = use ? y - (row[0] * xh[0] + row[1] * xh[1] + row[2] * xh[2] + row[3] * xh[3]) : 0.0;
  t.sse = warp_add(t.e * t.e);
  chol4(nrm, row, z, nullptr);                         // z = N^-1 a: column of (H^T H)^-1 H^T
  t.omh = 1.0 - (row[0] * z[0] + row[1] * z[1] + row[2] * z[2] + row[3] * z[3]);
  const bool testable = use && t.omh > 1e-12;
  double hs = 0.0, vs = 0.0;
  if (testable) {
    const double ze = -sl * z[0] + cl * z[1];
    const double zn = (-sb * cl) * z[0] + (-sb * sl) * z[1] + cb * z[2];
    const double zu = (cb * cl) * z[0] + (cb * sl) * z[1] + sb * z[2];
    const double s = sqrt(t.omh);
    hs = sqrt(ze * ze + zn * zn) / s;
    vs = fabs(zu) / s;
  }
  const bool untestable = __ballot_sync(0xffffffffu, use && !testable) != 0;
  hs = warp_max(hs);
  vs = warp_max(vs);
  t.hpl = untestable ? inf_f64() : sigma_pb * hs;
  t.vpl = untestable ? inf_f64() : sigma_pb * vs;
  return true;
}

// One warp per (recording, epoch), lane = channel, after K8 and independent of K8's next epoch (post hoc).
__global__ void __launch_bounds__(128) nav_integrity_kernel(IntegArgs a) {
  const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= (long long)a.n_rec * a.max_epochs) return;
  const int rec = (int)(warp / a.max_epochs), ep = (int)(warp % a.max_epochs);
  const int C = a.n_ch;
  const bool mine = lane < C;
  const long long o = warp * C + lane;
  double* out = a.integ + warp * SGX_NAV_INTEG_FIELDS;
  const double* sol = a.sol + warp * SGX_NAV_SOL_FIELDS;
  const int n_ep = min(a.n_epochs[rec], a.max_epochs);
  if (ep >= n_ep || !(isfinite(sol[0]) && isfinite(sol[1]) && isfinite(sol[2]) && isfinite(sol[3]))) {
    if (mine) a.norm_resid[o] = nan_f64();
    if (lane < SGX_NAV_INTEG_FIELDS)
      out[lane] = lane == 13 ? (double)SGX_INTEG_NO_FIX : lane == 14 ? -1.0 : lane == 15 ? 0.0 : nan_f64();
    return;
  }
  const double c_light = a.st.c, sigma = a.is.sigma, dtr_deg = 3.141592653589793 / 180;
  const bool trop_on = a.st.use_trop_corr != 0;
  double transmit_time = a.tow[rec];                   // advanced as nav_solve_kernel does, bit for bit
  for (int k = 0; k < ep; ++k) transmit_time += a.st.nav_sol_period / 1000;
  const bool use0 = mine && a.active[o] != 0;
  const int n = __popc(__ballot_sync(0xffffffffu, use0));
  double xs[3] = {0.0, 0.0, 0.0}, obs = 0.0;
  if (use0) {
    double clk;
    satpos_one(transmit_time, a.eph[(long long)rec * C + lane], xs, clk);
    obs = a.raw_p[o] + clk * c_light;
  }
  double fix[7] = {sol[0], sol[1], sol[2], sol[3], sol[9], sol[10], sol[11]};
  double q = nan_f64(), thr = nan_f64(), q_final = nan_f64(), hpl = nan_f64(), vpl = nan_f64(), w = nan_f64();
  int status = SGX_INTEG_UNAVAILABLE, excluded = -1, n_used = n;
  const int dof = n - 4;
  double sl, cl, sb, cb;
  sincos(sol[10] * dtr_deg, &sl, &cl);
  sincos(sol[9] * dtr_deg, &sb, &cb);
  const double sigma_pb = dof >= 1 ? sigma * a.is.pbias[dof - 1] : 0.0;
  double y = 0.0, row[4] = {0.0, 0.0, 0.0, 0.0};
  IntegTest t0;
  if (n >= 5) {
    const double p0[4] = {sol[0], sol[1], sol[2], sol[3]};
    if (use0) integ_model(p0, xs, obs, c_light, trop_on, y, row);
    if (integ_test(use0, y, row, sigma_pb, sl, cl, sb, cb, t0)) {
      const bool testable = use0 && t0.omh > 1e-12;
      q = t0.sse / (sigma * sigma);
      thr = a.is.thresh[dof - 1];
      q_final = q; hpl = t0.hpl; vpl = t0.vpl;
      if (testable) w = t0.e / (sigma * sqrt(t0.omh));
      if (q <= thr) {
        status = SGX_INTEG_OK;
      } else {
        status = SGX_INTEG_FAULT;
        if (n >= 6) {
          // SSE without channel j, argmin with ties to the lowest channel
          double smin = testable ? t0.sse - (t0.e * t0.e) / t0.omh : inf_f64();
          int jstar = lane;
#pragma unroll
          for (int d = 16; d > 0; d >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, smin, d);
            const int oj = __shfl_xor_sync(0xffffffffu, jstar, d);
            if (ov < smin || (ov == smin && oj < jstar)) { smin = ov; jstar = oj; }
          }
          if (smin / (sigma * sigma) <= a.is.thresh[dof - 2]) {
            // Gauss-Newton on S1 = S0 \ {j*} from K8's fix, the model re-evaluated at every iterate
            const bool use1 = use0 && lane != jstar;
            const double sigma_pb1 = sigma * a.is.pbias[dof - 2];
            double p[4] = {p0[0], p0[1], p0[2], p0[3]};
            bool ok = true;
            for (int it = 0; it < 6 && ok; ++it) {
              double y1 = 0.0, row1[4] = {0.0, 0.0, 0.0, 0.0}, nrm[10], dx[4];
              if (use1) integ_model(p, xs, obs, c_light, trop_on, y1, row1);
              ok = integ_normal(row1, y1, nrm, dx);
              if (ok) {
#pragma unroll
                for (int i = 0; i < 4; ++i) p[i] = p[i] + dx[i];
                if (sqrt(dx[0] * dx[0] + dx[1] * dx[1] + dx[2] * dx[2]) < 1e-4) break;
              }
            }
            double y1 = 0.0, row1[4] = {0.0, 0.0, 0.0, 0.0};
            IntegTest t1;
            if (ok && use1) integ_model(p, xs, obs, c_light, trop_on, y1, row1);
            if (ok && integ_test(use1, y1, row1, sigma_pb1, sl, cl, sb, cb, t1)) {
              status = SGX_INTEG_EXCLUDED;
              excluded = jstar;
              n_used = n - 1;
              q_final = t1.sse / (sigma * sigma);
              hpl = t1.hpl; vpl = t1.vpl;
              fix[0] = p[0]; fix[1] = p[1]; fix[2] = p[2]; fix[3] = p[3];
              cart2geo(p[0], p[1], p[2], fix[4], fix[5], fix[6]);
            }
          }
        }
      }
    }
  }
  if (mine) a.norm_resid[o] = w;
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < 7; ++i) out[i] = fix[i];
    out[7] = q; out[8] = thr; out[9] = (double)dof; out[10] = q_final; out[11] = hpl; out[12] = vpl;
    out[13] = (double)status; out[14] = (double)excluded; out[15] = (double)n_used;
  }
}

}  // namespace sgx

using namespace sgx;

extern "C" int sgx_nav_solve(const double* abs_sample, int64_t stride, int32_t n_recordings, int32_t n_channels,
                             int32_t ms, const int32_t* sub_frame_start, const uint8_t* ready, const sgx_eph* eph,
                             const double* tow, const int32_t* n_epochs, int32_t max_epochs,
                             const sgx_nav_settings* st, double* raw_p, double* corrected_p, double* el, double* az,
                             double* sat_pos, double* sat_clk, uint8_t* active, double* sol, void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_nav_solve", "no CUDA device");
  SGX_API_GUARD();
  if (!abs_sample || !sub_frame_start || !ready || !eph || !tow || !n_epochs || !st || !raw_p || !corrected_p || !el ||
      !az || !active || !sol || n_channels < 1 || n_channels > 32 || ms <= 0 || stride < ms || n_recordings < 0 ||
      max_epochs < 0 || !(st->nav_sol_period >= 1.0) || !(st->samples_per_code > 0))
    return fail(SGX_ERR_ARG, "sgx_nav_solve", "bad argument (1..32 channels, stride >= ms, period >= 1 ms)");
  if (n_recordings == 0 || max_epochs == 0) return SGX_OK;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  static DevBuf b_abs, b_sfs, b_ready, b_eph, b_tow, b_nep, b_raw, b_cor, b_el, b_az, b_pos, b_clk, b_act, b_sol;
  const size_t rc = (size_t)n_recordings * n_channels, rec = (size_t)n_recordings * max_epochs * n_channels;
  NavArgs a;
  StagedOutputs out;
  int r;
  if ((r = stage_rows_in(abs_sample, stride, ms, rc, b_abs, a.abs_sample, a.stride, s)) ||
      (r = stage_in(sub_frame_start, rc, b_sfs, a.sub_frame_start, s)) || (r = stage_in(ready, rc, b_ready, a.ready, s)) ||
      (r = stage_in(eph, rc, b_eph, a.eph, s)) || (r = stage_in(tow, (size_t)n_recordings, b_tow, a.tow, s)) ||
      (r = stage_in(n_epochs, (size_t)n_recordings, b_nep, a.n_epochs, s)))
    return r;
  if ((r = out.add(raw_p, rec, b_raw, a.raw_p)) || (r = out.add(corrected_p, rec, b_cor, a.corrected_p)) ||
      (r = out.add(el, rec, b_el, a.el)) || (r = out.add(az, rec, b_az, a.az)) ||
      (r = out.add(sat_pos, rec * 3, b_pos, a.sat_pos)) || (r = out.add(sat_clk, rec, b_clk, a.sat_clk)) ||
      (r = out.add(active, rec, b_act, a.active)) ||
      (r = out.add(sol, (size_t)n_recordings * max_epochs * SGX_NAV_SOL_FIELDS, b_sol, a.sol)))
    return r;
  a.n_rec = n_recordings; a.n_ch = n_channels; a.ms = ms; a.max_epochs = max_epochs; a.st = *st;
  const int threads = 128;                            // 4 recordings per CTA
  const unsigned blocks = (unsigned)(((long long)n_recordings * 32 + threads - 1) / threads);
  SGX_COUNTED_LAUNCH(nav_solve_kernel, dim3(blocks), dim3(threads), 0, s, a);
  SGX_CUDA(cudaGetLastError());
  return out.finish(s);
}

extern "C" int sgx_nav_velocity(const double* carr_freq, int64_t stride, int32_t n_recordings, int32_t n_channels,
                                int32_t ms, const int32_t* ms_done, const int32_t* sub_frame_start, const sgx_eph* eph,
                                const double* tow, const int32_t* n_epochs, int32_t max_epochs, const uint8_t* active,
                                const double* sol, const sgx_vel_settings* vs, double* vel, double* doppler,
                                double* rr_resid, double* sat_vel, double* sat_clk_drift, void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_nav_velocity", "no CUDA device");
  SGX_API_GUARD();
  if (!carr_freq || !sub_frame_start || !eph || !tow || !n_epochs || !active || !sol || !vs || !vel || !doppler ||
      !rr_resid || n_channels < 1 || n_channels > 32 || ms <= 0 || stride < ms || n_recordings < 0 || max_epochs < 0)
    return fail(SGX_ERR_ARG, "sgx_nav_velocity", "bad argument (NULL pointer, 1..32 channels, ms > 0, stride >= ms)");
  if (vs->doppler_avg_ms < 1 || !(vs->nav_sol_period >= 1.0) || !isfinite(vs->nav_sol_period) || !isfinite(vs->c) ||
      !(vs->c > 0) || !isfinite(vs->f_L1) || !(vs->f_L1 > 0) || !isfinite(vs->IF))
    return fail(SGX_ERR_ARG, "sgx_nav_velocity",
                "bad settings (doppler_avg_ms >= 1, nav_sol_period >= 1, c and f_L1 finite and > 0, IF finite)");
  const size_t rc = (size_t)n_recordings * n_channels;
  if (ms_done)
    for (size_t i = 0; i < rc; ++i)
      if (ms_done[i] < 0 || ms_done[i] > ms) return fail(SGX_ERR_ARG, "sgx_nav_velocity", "ms_done outside [0, ms]");
  if (n_recordings == 0 || max_epochs == 0) return SGX_OK;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  static DevBuf b_carr, b_done, b_sfs, b_eph, b_tow, b_nep, b_act, b_sol, b_vel, b_dop, b_res, b_svel, b_sclk;
  const size_t rec = rc * max_epochs, n_sol = (size_t)n_recordings * max_epochs;
  VelArgs a;
  StagedOutputs out;
  int r;
  if ((r = stage_rows_in(carr_freq, stride, ms, rc, b_carr, a.carr_freq, a.stride, s)) ||
      (r = stage_in(ms_done, rc, b_done, a.ms_done, s)) ||          // NULL: every channel completed all ms periods
      (r = stage_in(sub_frame_start, rc, b_sfs, a.sub_frame_start, s)) || (r = stage_in(eph, rc, b_eph, a.eph, s)) ||
      (r = stage_in(tow, (size_t)n_recordings, b_tow, a.tow, s)) ||
      (r = stage_in(n_epochs, (size_t)n_recordings, b_nep, a.n_epochs, s)) ||
      (r = stage_in(active, rec, b_act, a.active, s)) || (r = stage_in(sol, n_sol * SGX_NAV_SOL_FIELDS, b_sol, a.sol, s)))
    return r;
  if ((r = out.add(vel, n_sol * SGX_NAV_VEL_FIELDS, b_vel, a.vel)) || (r = out.add(doppler, rec, b_dop, a.doppler)) ||
      (r = out.add(rr_resid, rec, b_res, a.rr_resid)) || (r = out.add(sat_vel, rec * 3, b_svel, a.sat_vel)) ||
      (r = out.add(sat_clk_drift, rec, b_sclk, a.sat_clk_drift)))
    return r;
  a.n_rec = n_recordings; a.n_ch = n_channels; a.ms = ms; a.max_epochs = max_epochs; a.st = *vs;
  const int threads = 128;                            // 4 (recording, epoch) warps per CTA
  const unsigned blocks = (unsigned)(((long long)n_recordings * max_epochs * 32 + threads - 1) / threads);
  SGX_COUNTED_LAUNCH(nav_velocity_kernel, dim3(blocks), dim3(threads), 0, s, a);
  SGX_CUDA(cudaGetLastError());
  return out.finish(s);
}

extern "C" int sgx_nav_integrity(const double* raw_p, const uint8_t* active, const double* sol, int32_t n_recordings,
                                 int32_t n_channels, int32_t max_epochs, const int32_t* n_epochs, const sgx_eph* eph,
                                 const double* tow, const sgx_nav_settings* st, const sgx_integ_settings* is,
                                 double* integ, double* norm_resid, void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_nav_integrity", "no CUDA device");
  SGX_API_GUARD();
  if (!raw_p || !active || !sol || !n_epochs || !eph || !tow || !st || !is || !integ || !norm_resid || n_channels < 1 ||
      n_channels > 32 || n_recordings < 0 || max_epochs < 0)
    return fail(SGX_ERR_ARG, "sgx_nav_integrity", "bad argument (NULL pointer, 1..32 channels, counts >= 0)");
  if (!(st->nav_sol_period >= 1.0) || !isfinite(st->nav_sol_period) || !(st->c > 0) || !isfinite(st->c) ||
      !(is->sigma > 0) || !isfinite(is->sigma))
    return fail(SGX_ERR_ARG, "sgx_nav_integrity", "bad settings (nav_sol_period >= 1, c and sigma finite and > 0)");
  for (int k = 0; k < SGX_INTEG_MAX_DOF; ++k)
    if (!(is->thresh[k] > 0) || !isfinite(is->thresh[k]) || !(is->pbias[k] > 0) || !isfinite(is->pbias[k]))
      return fail(SGX_ERR_ARG, "sgx_nav_integrity", "thresh and pbias entries must be finite and > 0");
  if (n_recordings == 0 || max_epochs == 0) return SGX_OK;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  static DevBuf b_raw, b_act, b_sol, b_nep, b_eph, b_tow, b_integ, b_res;
  const size_t rc = (size_t)n_recordings * n_channels, rec = rc * max_epochs, n_sol = (size_t)n_recordings * max_epochs;
  IntegArgs a;
  StagedOutputs out;
  int r;
  if ((r = stage_in(raw_p, rec, b_raw, a.raw_p, s)) || (r = stage_in(active, rec, b_act, a.active, s)) ||
      (r = stage_in(sol, n_sol * SGX_NAV_SOL_FIELDS, b_sol, a.sol, s)) ||
      (r = stage_in(n_epochs, (size_t)n_recordings, b_nep, a.n_epochs, s)) || (r = stage_in(eph, rc, b_eph, a.eph, s)) ||
      (r = stage_in(tow, (size_t)n_recordings, b_tow, a.tow, s)))
    return r;
  if ((r = out.add(integ, n_sol * SGX_NAV_INTEG_FIELDS, b_integ, a.integ)) ||
      (r = out.add(norm_resid, rec, b_res, a.norm_resid)))
    return r;
  a.n_rec = n_recordings; a.n_ch = n_channels; a.max_epochs = max_epochs; a.st = *st; a.is = *is;
  const int threads = 128;                            // 4 (recording, epoch) warps per CTA
  const unsigned blocks = (unsigned)(((long long)n_recordings * max_epochs * 32 + threads - 1) / threads);
  SGX_COUNTED_LAUNCH(nav_integrity_kernel, dim3(blocks), dim3(threads), 0, s, a);
  SGX_CUDA(cudaGetLastError());
  return out.finish(s);
}
