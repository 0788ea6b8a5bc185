// Preamble search / bit synchronisation and 20 ms bit summation on the device (SURVEY.md section 8(f) row 3).
//
// Replaces NavigationResult.findPreambles (postNavigation.py:524-631) and the bit summation of its caller
// (postNavigation.py:125-134) for a batch of tracked channels.  Everything is integer / bit work except the
// 20-sample float64 sums, which are added in numpy's pairwise order so that the sign of a sum is the
// reference's even when the sum cancels to (almost) zero.
//
// One CTA per channel:
//   1. sign bits of I_P (I_P > 0 -> 1; 0, negatives and NaN -> 0, postNavigation.py:567-569) packed into
//      shared memory with warp ballots;
//   2. correlation with the 160 ms preamble pattern at every lag k (the reference's M x M np.correlate has
//      only 160 non-zero taps): 5 funnel-shifted words XOR the pattern, popcount; candidate iff |c| > 153;
//   3. candidates with a partner 6000 ms later are verified in ascending order, one warp per candidate:
//      62 sums of 20 ms -> hard bits -> the two parity checks of navPartyChk (postNavigation.py:441-521)
//      as popcount parities; the smallest passing k wins (atomicMin);
//   4. the 1501 navigation bits that postNavigate hands to ephemeris() are produced for the winner.
#include "sgx_common.cuh"

namespace sgx {

constexpr int BS_THREADS = 256;
constexpr int PRE_LEN = 160;          // 8 preamble bits x 20 ms
constexpr int PRE_THRESHOLD = 153;    // postNavigation.py:584
constexpr int SUBFRAME_MS = 6000;     // :593
constexpr int NAV_BITS = 1501;        // 1 + 5 subframes x 300 (postNavigation.py:125)

// preamble 1 -1 -1 -1 1 -1 1 1 (postNavigation.py:554), each bit 20 times, LSB first: bit j = PRE[j / 20]
__device__ __forceinline__ unsigned pattern_word(int q) {
  unsigned w = 0;
#pragma unroll
  for (int b = 0; b < 32; ++b) {
    const int j = 32 * q + b;
    const int bit = j / 20;
    const bool one = bit == 0 || bit == 4 || bit == 6 || bit == 7;
    w |= (one ? 1u : 0u) << b;
  }
  return w;
}

// numpy's pairwise float64 sum of 20 contiguous values (DOUBLE_pairwise_sum for 8 <= n <= 128: eight running
// sums, a balanced tree over them, then the tail in order) -- what `x.reshape(20, -1, order='F').sum(0)` does
__device__ __forceinline__ double sum20(const double* a) {
  double r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = a[j];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = r[j] + a[8 + j];
  double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
#pragma unroll
  for (int j = 16; j < 20; ++j) res = res + a[j];
  return res;
}

// navPartyChk (postNavigation.py:441-521) on 32 hard bits, bit j of v = (ndat[j] == +1).  A product of +-1
// values is +1 iff the number of -1 factors is even.  Returns true when the function's status is non-zero.
__device__ __forceinline__ bool parity_ok(unsigned v) {
  if (!((v >> 1) & 1u)) v ^= 0x03FFFFFCu;          // ndat[2:26] *= -1 when D30* is not +1 (:469)
  const unsigned taps[6] = {
      // indices into ndat of the factors of parity[0..5] (:480-504)
      (1u << 0) | (1u << 2) | (1u << 3) | (1u << 4) | (1u << 6) | (1u << 7) | (1u << 11) | (1u << 12) | (1u << 13) |
          (1u << 14) | (1u << 15) | (1u << 18) | (1u << 19) | (1u << 21) | (1u << 24),
      (1u << 1) | (1u << 3) | (1u << 4) | (1u << 5) | (1u << 7) | (1u << 8) | (1u << 12) | (1u << 13) | (1u << 14) |
          (1u << 15) | (1u << 16) | (1u << 19) | (1u << 20) | (1u << 22) | (1u << 25),
      (1u << 0) | (1u << 2) | (1u << 4) | (1u << 5) | (1u << 6) | (1u << 8) | (1u << 9) | (1u << 13) | (1u << 14) |
          (1u << 15) | (1u << 16) | (1u << 17) | (1u << 20) | (1u << 21) | (1u << 23),
      (1u << 1) | (1u << 3) | (1u << 5) | (1u << 6) | (1u << 7) | (1u << 9) | (1u << 10) | (1u << 14) | (1u << 15) |
          (1u << 16) | (1u << 17) | (1u << 18) | (1u << 21) | (1u << 22) | (1u << 24),
      (1u << 1) | (1u << 2) | (1u << 4) | (1u << 6) | (1u << 7) | (1u << 8) | (1u << 10) | (1u << 11) | (1u << 15) |
          (1u << 16) | (1u << 17) | (1u << 18) | (1u << 19) | (1u << 22) | (1u << 23) | (1u << 25),
      (1u << 0) | (1u << 4) | (1u << 6) | (1u << 7) | (1u << 9) | (1u << 10) | (1u << 11) | (1u << 12) | (1u << 14) |
          (1u << 16) | (1u << 20) | (1u << 23) | (1u << 24) | (1u << 25)};
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    const unsigned minus = __popc(~v & taps[i]);             // factors equal to -1
    const unsigned plus_one = (minus & 1u) ^ 1u;             // product == +1
    ok = ok && (plus_one == ((v >> (26 + i)) & 1u));         // parity[i] == ndat[26 + i] (:507)
  }
  return ok;
}

struct BitsyncArgs {
  const double* ip;      // [n_ch][stride]
  long long stride;
  int ms;
  int n_words;           // ceil(ms / 32)
  int* first;            // [n_ch]
  unsigned char* bits;   // [n_ch][NAV_BITS] or null
  int* bits_valid;       // [n_ch] or null
};

__global__ void __launch_bounds__(BS_THREADS) bitsync_kernel(BitsyncArgs a) {
  SGX_DYN_SMEM(smem);
  unsigned* sgn = reinterpret_cast<unsigned*>(smem);           // n_words + 8 (zero padded)
  unsigned* cand = sgn + a.n_words + 8;                         // n_words
  __shared__ int best;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int NWARPS = BS_THREADS / 32;
  const double* ip = a.ip + (long long)blockIdx.x * a.stride;
  const int ms = a.ms;
  if (tid == 0) best = 0x7fffffff;
  for (int w = a.n_words + tid; w < a.n_words + 8; w += BS_THREADS) sgn[w] = 0u;

  // 1. sign bits: eight independent 256-byte row segments in flight per warp before the ballots (a single load
  //    per trip left the CTA waiting one DRAM latency per 32 samples)
  constexpr int UNR = 8;
  for (int w0 = warp * UNR; w0 < a.n_words; w0 += NWARPS * UNR) {
    double v[UNR];
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const int i = 32 * (w0 + u) + lane;
      v[u] = i < ms ? ip[i] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < UNR; ++u) {
      const unsigned m = __ballot_sync(0xffffffffu, v[u] > 0.0);
      if (lane == 0 && w0 + u < a.n_words) sgn[w0 + u] = m;
    }
  }
  __syncthreads();

  // 2. candidates: |sum_j s[k+j] p[j]| > 153 over the taps that exist (j < ms - k)
  unsigned pat[5];
#pragma unroll
  for (int q = 0; q < 5; ++q) pat[q] = pattern_word(q);
  for (int w = tid; w < a.n_words; w += BS_THREADS) {
    unsigned out = 0;
    unsigned x[7];
#pragma unroll
    for (int q = 0; q < 7; ++q) x[q] = sgn[w + q];
    if (32 * w + 31 + PRE_LEN <= ms) {
      // all 160 taps exist for the 32 lags of this word (every word but the last five of a record)
#pragma unroll 4
      for (int b = 0; b < 32; ++b) {
        int differ = 0;
#pragma unroll
        for (int q = 0; q < 5; ++q) differ += __popc(__funnelshift_r(x[q], x[q + 1], b) ^ pat[q]);
        const int c = PRE_LEN - 2 * differ;
        if (c > PRE_THRESHOLD || -c > PRE_THRESHOLD) out |= 1u << b;
      }
    } else {
      for (int b = 0; b < 32; ++b) {
        const int k = 32 * w + b;
        if (k >= ms) break;
        const int n = min(PRE_LEN, ms - k);
        int agree = 0;
#pragma unroll
        for (int q = 0; q < 5; ++q) {
          unsigned s = __funnelshift_r(x[q], x[q + 1], b);
          unsigned eq = ~(s ^ pat[q]);
          const int keep = n - 32 * q;                         // taps of this word that exist
          if (keep < 32) eq &= keep <= 0 ? 0u : (0xFFFFFFFFu >> (32 - keep));
          agree += __popc(eq);
        }
        const int c = 2 * agree - n;
        if (c > PRE_THRESHOLD || -c > PRE_THRESHOLD) out |= 1u << b;
      }
    }
    cand[w] = out;
  }
  __syncthreads();

  // 3. verification, ascending k, one warp per candidate
  for (int w = warp; w < a.n_words; w += NWARPS) {
    // a smaller k already passed?  (read by one lane and broadcast: the exit has to be warp-uniform)
    const int seen = __shfl_sync(0xffffffffu, lane == 0 ? *(volatile int*)&best : 0, 0);
    if (32 * w >= seen) break;
    const int k = 32 * w + lane;
    bool q = (cand[w] >> lane) & 1u;
    if (q) {
      const int k2 = k + SUBFRAME_MS;                           // another candidate exactly one subframe later (:593)
      q = k2 < ms && ((cand[k2 >> 5] >> (k2 & 31)) & 1u);
      // the reference reads I_P[k-40 : k+1200]; k < 40 makes that slice empty and crashes it -- passed over
      q = q && k >= 40 && k + 1200 <= ms;
    }
    unsigned todo = __ballot_sync(0xffffffffu, q);
    while (todo) {
      const int b = __ffs(todo) - 1;
      todo &= todo - 1;
      const int kc = 32 * w + b;
      // 62 bits: 2 of the previous word + TLM + HOW (:594-602); lane l sums bits l and l + 32
      const double* base = ip + (kc - 40);
      const bool b0 = sum20(base + 20 * lane) > 0.0;
      const bool b1 = lane < 30 ? sum20(base + 20 * (lane + 32)) > 0.0 : false;
      const unsigned lo = __ballot_sync(0xffffffffu, b0);       // bits 0..31
      const unsigned hi = __ballot_sync(0xffffffffu, b1);       // bits 32..61
      if (lane == 0) {
        const unsigned w1 = lo;                                  // bits[0:32]
        const unsigned w2 = (lo >> 30) | (hi << 2);              // bits[30:62]
        if (parity_ok(w1) && parity_ok(w2)) atomicMin(&best, kc);
      }
    }
  }
  __syncthreads();
  const int f = best == 0x7fffffff ? 0 : best;
  if (tid == 0) a.first[blockIdx.x] = f;

  // 4. navigation bits of the five subframes from the winner on (postNavigation.py:125-134)
  if (a.bits) {
    const bool ok = f != 0 && f - 20 >= 0 && (long long)f + 20 * (NAV_BITS - 1) <= ms;
    if (tid == 0 && a.bits_valid) a.bits_valid[blockIdx.x] = ok ? 1 : 0;
    unsigned char* o = a.bits + (long long)blockIdx.x * NAV_BITS;
    for (int j = tid; j < NAV_BITS; j += BS_THREADS) o[j] = ok ? (sum20(ip + (f - 20) + 20 * j) > 0.0 ? 1 : 0) : 0;
  }
}

struct BitsyncScratch {
  DevBuf ip, first, bits, valid;
};
static BitsyncScratch g_bs;

}  // namespace sgx

using namespace sgx;

extern "C" int sgx_find_preambles(const double* i_p, int64_t stride, int32_t n_channels, int32_t ms,
                                  int32_t* first_subframe, uint8_t* nav_bits, int32_t* nav_bits_valid,
                                  void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_find_preambles", "no CUDA device");
  SGX_API_GUARD();
  if (!i_p || !first_subframe || n_channels < 0 || ms <= 0 || stride < ms)
    return fail(SGX_ERR_ARG, "sgx_find_preambles", "bad argument");
  if (n_channels == 0) return SGX_OK;
  BitsyncArgs a;
  a.ms = ms;
  a.n_words = (ms + 31) / 32;
  const size_t smem = sizeof(unsigned) * (2 * (size_t)a.n_words + 8);
  if (smem > 200 * 1024) return fail(SGX_ERR_RANGE, "sgx_find_preambles", "record longer than 800 000 ms");
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const size_t n = (size_t)n_channels;
  int32_t* valid = nav_bits ? nav_bits_valid : nullptr;   // written only together with nav_bits
  StagedOutputs out;
  int r;
  if ((r = stage_rows_in(i_p, stride, ms, n, g_bs.ip, a.ip, a.stride, s)) ||
      (r = out.add(first_subframe, n, g_bs.first, a.first)) ||
      (r = out.add(nav_bits, (size_t)NAV_BITS * n, g_bs.bits, a.bits)) ||
      (r = out.add(valid, n, g_bs.valid, a.bits_valid)))
    return r;
  if (smem > 48 * 1024)
    SGX_CUDA(cudaFuncSetAttribute(bitsync_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  SGX_COUNTED_LAUNCH(bitsync_kernel, dim3(n_channels), dim3(BS_THREADS), smem, s, a);
  SGX_CUDA(cudaGetLastError());
  return out.finish(s);
}

// ---- relative pseudoranges (postNavigation.py:27-72), batched over recordings x measurement epochs ---------
namespace sgx {
struct PseudoArgs {
  const double* abs_sample;   // row (r, c) = abs_sample + (r*n_ch + c)*stride, ms values
  long long stride;
  const int* ms_index;    // [n_rec][n_epochs][n_ch]
  const unsigned char* active;   // [n_rec][n_epochs][n_ch]
  double* pr;             // [n_rec][n_epochs][n_ch]
  int n_rec, n_ch, n_epochs, ms;
  double samples_per_code, start_offset, c;
};

// one warp per (recording, epoch); lane = channel (n_ch <= 32)
__global__ void pseudorange_kernel(PseudoArgs a) {
  const int unit = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (unit >= a.n_rec * a.n_epochs) return;
  const int r = unit / a.n_epochs;
  const long long o = (long long)unit * a.n_ch + lane;
  double t = __longlong_as_double(0x7ff0000000000000LL);                    // +inf: not in the list (:52)
  if (lane < a.n_ch && a.active[o]) {
    const int i = a.ms_index[o];
    if (i >= 0 && i < a.ms)
      t = a.abs_sample[((long long)r * a.n_ch + lane) * a.stride + i] / a.samples_per_code;   // :60
  }
  double m = t;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, d));
  if (lane < a.n_ch) a.pr[o] = ((t - floor(m)) + a.start_offset) * a.c / 1000.0;   // :64-71, same operation order
}
}  // namespace sgx

extern "C" int sgx_pseudoranges(const double* track_out, int32_t n_recordings, int32_t n_channels, int32_t ms,
                                const int32_t* ms_index, const uint8_t* active, int32_t n_epochs,
                                double samples_per_code, double start_offset, double c, double* pseudoranges,
                                void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_pseudoranges", "no CUDA device");
  SGX_API_GUARD();
  if (!track_out || !ms_index || !active || !pseudoranges || n_channels < 1 || n_channels > 32 || ms <= 0 ||
      n_recordings < 0 || n_epochs < 0)
    return fail(SGX_ERR_ARG, "sgx_pseudoranges", "bad argument (1..32 channels)");
  const long long units = (long long)n_recordings * n_epochs;
  if (units == 0) return SGX_OK;
  cudaStream_t s = (cudaStream_t)cuda_stream;
  static DevBuf d_abs, d_idx, d_act, d_pr;
  const size_t n = (size_t)units * n_channels;
  PseudoArgs a;
  StagedOutputs out;
  int r;
  if ((r = stage_rows_in(track_out, (int64_t)SGX_TRACK_FIELDS * ms, ms, (size_t)n_recordings * n_channels, d_abs,
                         a.abs_sample, a.stride, s)) ||
      (r = stage_in(ms_index, n, d_idx, a.ms_index, s)) || (r = stage_in(active, n, d_act, a.active, s)) ||
      (r = out.add(pseudoranges, n, d_pr, a.pr)))
    return r;
  a.n_rec = n_recordings; a.n_ch = n_channels; a.n_epochs = n_epochs; a.ms = ms;
  a.samples_per_code = samples_per_code; a.start_offset = start_offset; a.c = c;
  const int threads = 256;
  const long long blocks = (units * 32 + threads - 1) / threads;
  SGX_COUNTED_LAUNCH(pseudorange_kernel, dim3((unsigned)blocks), dim3(threads), 0, s, a);
  SGX_CUDA(cudaGetLastError());
  return out.finish(s);
}
