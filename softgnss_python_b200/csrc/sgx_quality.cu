// Per-window C/N0 (variance-summing method) and carrier-lock indicator of tracked channels, on the device.
//
// Reads the prompt correlator series I_P / Q_P where they already are (e.g. fields 3 and 7 of sgx_track's output,
// rows SGX_TRACK_FIELDS * ms apart) and reduces every window of W code periods to three numbers:
//   Z_k = I_k^2 + Q_k^2,  Zm = sum(Z) / W,  Zv = sum((Z_k - Zm)^2) / (W - 1)          (two passes, unbiased)
//   Pav = sqrt(Zm^2 - Zv),  Nv = 0.5 * (Zm - Pav),  cn0 = 10 * log10(Pav / (2 * Nv * T))   dB-Hz
//   pll_lock = sum(I_k^2 - Q_k^2) / sum(Z_k)                                               (cos 2 dphi)
//   locked = cn0 >= cn0_min && pll_lock >= pll_lock_min
// cn0 is NaN unless Zm^2 - Zv > 0 and Nv > 0 (the Matlab CNoVSM takes abs() of the complex result instead);
// pll_lock is NaN when sum(Z) == 0; a window that ends after ms_done[c] gets NaN, NaN, 0.
//
// Layout: one warp per (channel, window); lane l takes periods l, l + 32, ... of the window, so every load of the
// warp reads contiguous bytes of both rows.  Four such loads per row are issued before any is used.  The second
// pass re-reads the window, which the first pass has just brought into L1.  Lane sums are combined by a fixed xor
// butterfly, so the result does not depend on scheduling: two runs, and host or device operands, agree bit for bit.
// float64 throughout, no atomics.
#include <math.h>

#include "sgx_common.cuh"

namespace sgx {

constexpr int Q_THREADS = 256;        // 8 windows per CTA
constexpr int Q_UNROLL = 4;           // loads in flight per lane and row

struct QualityArgs {
  const double* ip;
  const double* qp;
  long long stride;                   // elements between channel rows
  const int* ms_done;                 // [n_ch] or nullptr (all ms)
  double* cn0;                        // [n_ch][n_win]
  double* pll;
  unsigned char* locked;
  long long n_units;                  // n_ch * n_win
  int n_win, W, ms;
  double acc_time, cn0_min, pll_min;
};

__global__ void __launch_bounds__(Q_THREADS) quality_kernel(QualityArgs a) {
  const long long unit = ((long long)blockIdx.x * Q_THREADS + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (unit >= a.n_units) return;                          // whole warps only: n_units is counted in warps
  const int c = (int)(unit / a.n_win), w = (int)(unit - (long long)c * a.n_win);
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  const int done = a.ms_done ? a.ms_done[c] : a.ms;
  if ((long long)(w + 1) * a.W > done) {
    if (lane == 0) { a.cn0[unit] = nan; a.pll[unit] = nan; a.locked[unit] = 0; }
    return;
  }
  const double* ip = a.ip + (long long)c * a.stride + (long long)w * a.W;
  const double* qp = a.qp + (long long)c * a.stride + (long long)w * a.W;
  const int W = a.W;
  // pass 1: sum(Z) and sum(I^2 - Q^2)
  double sz = 0.0, sd = 0.0;
  for (int k0 = 0; k0 < W; k0 += 32 * Q_UNROLL) {
    double iv[Q_UNROLL], qv[Q_UNROLL];
#pragma unroll
    for (int u = 0; u < Q_UNROLL; ++u) {
      const int k = k0 + 32 * u + lane;
      iv[u] = k < W ? ip[k] : 0.0;
      qv[u] = k < W ? qp[k] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < Q_UNROLL; ++u) {
      const double ii = iv[u] * iv[u], qq = qv[u] * qv[u];
      sz += ii + qq;
      sd += ii - qq;
    }
  }
  sz = warp_sum_f64(sz);
  sd = warp_sum_f64(sd);
  const double zm = sz / (double)W;
  // pass 2: sum((Z - Zm)^2) over the W periods of the window
  double sv = 0.0;
  for (int k0 = 0; k0 < W; k0 += 32 * Q_UNROLL) {
    double iv[Q_UNROLL], qv[Q_UNROLL];
#pragma unroll
    for (int u = 0; u < Q_UNROLL; ++u) {
      const int k = k0 + 32 * u + lane;
      iv[u] = k < W ? ip[k] : 0.0;
      qv[u] = k < W ? qp[k] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < Q_UNROLL; ++u) {
      const int k = k0 + 32 * u + lane;
      const double d = (iv[u] * iv[u] + qv[u] * qv[u]) - zm;
      if (k < W) sv += d * d;
    }
  }
  sv = warp_sum_f64(sv);
  if (lane != 0) return;
  const double zv = sv / (double)(W - 1);
  const double p2 = zm * zm - zv;
  double cn0 = nan;
  if (p2 > 0.0) {
    const double pav = sqrt(p2);
    const double nv = 0.5 * (zm - pav);
    if (nv > 0.0) cn0 = 10.0 * log10(pav / (2.0 * nv * a.acc_time));
  }
  const double pll = sz != 0.0 ? sd / sz : nan;
  a.cn0[unit] = cn0;
  a.pll[unit] = pll;
  a.locked[unit] = (cn0 >= a.cn0_min && pll >= a.pll_min) ? 1 : 0;
}

struct QualityScratch {
  DevBuf ip, qp, done, cn0, pll, locked;
};
static QualityScratch g_q;

}  // namespace sgx

using namespace sgx;

extern "C" int sgx_track_quality(const double* i_p, const double* q_p, int64_t stride, int32_t n_channels, int32_t ms,
                                 const int32_t* ms_done, const sgx_quality_settings* qs, double* cn0,
                                 double* pll_lock, uint8_t* locked, void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_track_quality", "no CUDA device");
  SGX_API_GUARD();
  if (!i_p || !q_p || !qs || !cn0 || !pll_lock || !locked || n_channels < 0 || ms < 0 || stride < ms)
    return fail(SGX_ERR_ARG, "sgx_track_quality", "bad argument (NULL pointer, n_channels < 0 or stride < ms)");
  if (qs->window_ms < 2 || !isfinite(qs->acc_time) || !(qs->acc_time > 0.0))
    return fail(SGX_ERR_ARG, "sgx_track_quality", "window_ms must be >= 2 and acc_time finite and > 0");
  if (ms_done)
    for (int32_t c = 0; c < n_channels; ++c)
      if (ms_done[c] < 0 || ms_done[c] > ms) return fail(SGX_ERR_ARG, "sgx_track_quality", "ms_done outside [0, ms]");
  const bool in_dev = is_device_ptr(i_p);
  const bool out_dev = is_device_ptr(cn0);
  if (is_device_ptr(q_p) != in_dev)
    return fail(SGX_ERR_ARG, "sgx_track_quality", "i_p and q_p must both be host or both be device memory");
  if (is_device_ptr(pll_lock) != out_dev || is_device_ptr(locked) != out_dev)
    return fail(SGX_ERR_ARG, "sgx_track_quality", "cn0, pll_lock and locked must all be host or all be device memory");
  const int n_win = ms / qs->window_ms;
  const long long n_units = (long long)n_channels * n_win;
  if (n_units == 0) return SGX_OK;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const size_t n = (size_t)n_channels;
  QualityArgs a;
  StagedOutputs out;
  long long q_stride;                       // equals a.stride: i_p and q_p are of one kind (checked above)
  int r;
  if ((r = stage_rows_in(i_p, stride, ms, n, g_q.ip, a.ip, a.stride, s)) ||
      (r = stage_rows_in(q_p, stride, ms, n, g_q.qp, a.qp, q_stride, s)) ||
      (r = stage_in(ms_done, n, g_q.done, a.ms_done, s)) ||      // NULL: all ms
      (r = out.add(cn0, (size_t)n_units, g_q.cn0, a.cn0)) || (r = out.add(pll_lock, (size_t)n_units, g_q.pll, a.pll)) ||
      (r = out.add(locked, (size_t)n_units, g_q.locked, a.locked)))
    return r;
  a.n_units = n_units;
  a.n_win = n_win;
  a.W = qs->window_ms;
  a.ms = ms;
  a.acc_time = qs->acc_time;
  a.cn0_min = qs->cn0_min;
  a.pll_min = qs->pll_lock_min;
  const long long blocks = (n_units * 32 + Q_THREADS - 1) / Q_THREADS;
  SGX_COUNTED_LAUNCH(quality_kernel, dim3((unsigned)blocks), dim3(Q_THREADS), 0, s, a);
  SGX_CUDA(cudaGetLastError());
  return out.finish(s);
}
