// Tracking hot path: one CTA per (recording, channel), the whole millisecond loop on the device.
//
// Replaces reference tracking.py:59-283.  Per code period ("ms") the reference
//   T3  sizes the block from the code NCO            tracking.py:148-151
//   T4  builds early/late/prompt replicas            tracking.py:166-188   (float64 ceil of a linspace)
//   T5  carries the code phase                       tracking.py:190
//   T6  builds sin/cos of the carrier NCO            tracking.py:193-201
//   T7  mixes and forms six correlator sums          tracking.py:205-219
//   T8  Costas PLL discriminator + loop filter       tracking.py:223-235
//   T9  normalised early-late DLL + loop filter      tracking.py:238-251
//   T10 records 13 values                            tracking.py:255-275
//
// Device formulation (DESIGN.md section "K5"):
//  * the block of int8 samples is staged in shared memory one period ahead (TMA 1-D bulk copy
//    completing on an mbarrier, or 16-byte cp.async), double buffered;
//  * the replicas are piecewise constant and, with E/L at +-0.5 chip, change only at the 2 046 half-chip
//    thresholds of a period: every thread owns 8 consecutive half-chip segments (~18.7 samples each).  A
//    boundary is predicted in Q40 fixed point from the reference's own linspace parameters and, when the
//    prediction is within 1e-6 of a sample instant, settled by evaluating the reference's expression
//    fl(fl(i*step)+start) exactly (settle_boundary), so the sample->chip assignment equals ceil(tcode) of the
//    reference for every sample;
//  * default (exact) variant: the carrier twiddles w^k of a segment are quantised once per period to Q38
//    (five signed base-256 digits, built by the carrier thread's warp in float64), a segment sum is 10 dp4a per
//    four samples with exact int32 accumulation, the digits are recombined exactly and rotated by the segment's
//    start rotor in float64; the three code values enter as sign-bit flips.  Agreement with the reference's
//    float64 loop: ~2e-11 of full scale, which keeps absoluteSample identical over 37 000 ms (DESIGN.md section 5).
//    `SGX_TRK_KERNEL=segments` selects a float32 version of the same segmentation, `groups` the aligned
//    16-sample-group formulation (any correlator spacing; used automatically when dllCorrelatorSpacing != 0.5);
//  * six float64 sums per thread -> warp shuffle -> one shared-memory exchange;
//  * thread 0 (code loop: T9, T5, T3/T4 of the next period) and thread 32 (carrier loop: T6 carry, T8, T6 of the
//    next period) then run the loop filters in float64 with separately rounded operations (compiled with
//    -fmad=false) exactly in the reference's order, and the carrier thread's warp rebuilds the twiddle tables.
//  * host recordings are streamed in chunks (pause/resume through TrackState); files through two pinned staging
//    buffers (sgx_track_file).
#include <vector>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include "sgx_common.cuh"

namespace sgx {

constexpr int TRK_THREADS = 256;
constexpr int TRK_WARPS = TRK_THREADS / 32;
constexpr int TRK_MARGIN = 256;  // extra samples staged beyond samplesPerCode
// SGX_TRK_PROF phases, stamped by lane 0 of every warp: window wait + prefetch issue, correlate, reduce + barrier,
// bookkeeping (loop filters, next period's parameters and tables), end-of-period barrier
constexpr int TRK_PROF_N = 5;

struct TrackArgs {
  const int8_t* rec;
  long long rec_stride;
  const long long* rec_len;
  const sgx_channel* ch;
  const int8_t* chips;  // [32][1023] +-1
  double* out;          // [R*C][13][ms]
  int* ms_done;         // [R*C]
  int* status;          // [R*C] sgx_status of the channel
  int n_channels;
  int ms;
  int resume;           // continue every channel from `state` (streaming ingest: the recording arrives in chunks)
  long long avail;      // bytes of every recording that are resident so far (>= rec_len when complete)
  struct TrackState* state;  // [R*C]
  long long* prof;      // optional [R*C][warp][TRK_PROF_N] cycle counters per period phase (SGX_TRK_PROF=1)
  int win;              // bytes per staging buffer, multiple of 16
  long long skip;
  long long abs_base;   // sample index of rec[0] in the file (streamed windows start at the first byte that is needed)
  double fs, codeFreqBasis, codeLength, spc;
  double c1code, c2code, c1carr, c2carr;  // tau2/tau1 and PDI/tau1 (tracking.py:225-227, 241-243)
};

struct MsParams {
  double startE, stepE, startL, stepL, startP, stepP;  // np.linspace(start, ., blk, endpoint=False)
  double inv_step;  // 1/codePhaseStep, used only to *predict* event indices
  long long q0_fix, h_fix;   // Q40 fixed point: predicted sample index of threshold n is (q0 + n*h) / 2^40
  double cps;       // carrier cycles per sample
  double rem_cyc;   // remCarrPhase in cycles
  double w;         // carrFreq * 2.0 * pi (tracking.py:195), rad/s
  double rem_rad;   // remCarrPhase, rad
  double fs;
  long long pos;    // byte offset (within the recording) of sample 0 of this block
  int blk;
  int stop;         // 0 = run this period, else sgx_status / 1 = finished
};

__device__ __forceinline__ double lin_y(int i, double step, double start) {
  // element i of np.linspace: two roundings, multiply then add (no FMA)
  return __dadd_rn(__dmul_rn((double)i, step), start);
}

// First sample index whose replica index exceeds c, i.e. first i with fl(fl(i*step)+start) > c.
__device__ __forceinline__ int next_event(int c, double start, double step, double inv) {
  double q = ((double)c - start) * inv;
  double fl = floor(q);
  int i = (int)fl + 1;
  double fr = q - fl;
  if (fr < 1e-6 || fr > 1.0 - 1e-6) {
    while (i > 0 && lin_y(i - 1, step, start) > (double)c) --i;
    while (!(lin_y(i, step, start) > (double)c)) ++i;
  }
  return i;
}

struct CodeVar {
  double start, step;
  int c;    // index into the padded code (tracking.py:111) for the current sample
  int e;    // first sample index at which the index becomes c+1
  float s;  // code value +-1 at c
  __device__ __forceinline__ void init(int i0, double st, double sp, double inv, const float* code) {
    start = st;
    step = sp;
    c = (int)ceil(lin_y(i0, step, start));
    s = code[c];
    e = next_event(c, start, step, inv);
  }
  __device__ __forceinline__ void advance(double inv, const float* code) {
    c += 1;
    s = code[c];
    e = next_event(c, start, step, inv);
  }
};

__device__ __forceinline__ float byte_to_float(unsigned u_offset_binary, int k) {
  // u = x ^ 0x80 per byte; 0x4B0000uu is the float 2^23 + uu
  unsigned r = __byte_perm(u_offset_binary, 0x4B000000u, 0x7540u + (unsigned)k);
  return __uint_as_float(r) - 8388736.0f;
}

// e^{j 2 pi cyc} in float32 from a float64 phase in cycles.  The phase is reduced in float64 and split
// into a float32 head and tail; the tail enters to first order, so the result carries only the
// rounding of its two components (6e-8) instead of the 3e-8-cycle rounding of the argument -- which
// would otherwise be multiplied by k in every power w^k built from it.
__device__ __forceinline__ void cis_cycles(double cyc, float& c, float& s) {
  cyc -= rint(cyc);
  const float hi = (float)cyc;
  const float lo = (float)(cyc - (double)hi) * 6.2831853071795865f;
  float s0, c0;
  sincospif(2.0f * hi, &s0, &c0);
  c = fmaf(-s0, lo, c0);
  s = fmaf(c0, lo, s0);
}

__device__ __forceinline__ void cmul(float& r, float& i, float ar, float ai, float br, float bi) {
  r = fmaf(ar, br, -(ai * bi));
  i = fmaf(ar, bi, ai * br);
}

// The per-period float64 bookkeeping is split over two threads of different warps so that the two
// dependent chains run concurrently: thread 0 owns the code loop (T3, T4 parameters, T5, T9), thread 32
// the carrier loop (T6, T8).  Neither needs the other's result within a period.
struct CodeState {   // tracking.py:114-116, :124-126
  double codeFreq, remCodePhase, oldCodeNco, oldCodeError, nextRemCode;
  long long pos;
};
struct CarrState {   // tracking.py:118-122, :128-130
  double carrFreq, carrFreqBasis, remCarrPhase, oldCarrNco, oldCarrError, w;
};

constexpr int SGX_PAUSED = 1;   // MsParams.stop: the next block is not resident yet (streaming ingest)

struct TrackState {   // loop state of one channel between two launches of a streamed recording
  CodeState c;
  CarrState r;
  int k;        // periods completed
  int status;   // SGX_OK (finished), SGX_PAUSED, or an error
};

// T3 + T4 parameters + T5 carry for the next period.  Run by all 32 lanes of one warp with the same state, so that
// the independent float64 divisions of the chain go to different lanes of one instruction instead of running one
// after another; lane 0 writes p.
__device__ void prepare_code(const TrackArgs& a, CodeState& st, long long rec_len, MsParams& p, int lane) {
  const double step = st.codeFreq / a.fs;                             // :148
  // lane 0: the block size quotient (:150), lane 1: 1/step (used only to predict event indices)
  const double q = (lane == 1 ? 1.0 : a.codeLength - st.remCodePhase) / step;
  const int blk = (int)ceil(__shfl_sync(0xffffffffu, q, 0));
  const double inv_step = __shfl_sync(0xffffffffu, q, 1);
  const long long aligned = st.pos & ~15LL;
  int stop = 0;
  if (st.pos + blk > rec_len) stop = SGX_ERR_SHORT;                   // :159
  else if (st.pos + blk > a.avail) stop = SGX_PAUSED;                  // wait for the next chunk of the file
  else if (blk <= 0 || (st.pos - aligned) + blk > a.win) stop = SGX_ERR_RANGE;
  if (lane == 0) { p.blk = blk; p.pos = st.pos; p.stop = stop; }
  if (stop) return;
  const double rem = st.remCodePhase, spc = a.spc, bs = (double)blk * step;
  const double startE = rem - spc, startL = rem + spc, startP = rem;  // :166, :174, :182
  // lanes 0, 1, 2: the E, L, P slopes of np.linspace
  const double num = lane == 0 ? ((bs + rem) - spc) - startE : lane == 1 ? ((bs + rem) + spc) - startL : (bs + rem) - startP;
  const double d = num / (double)blk;
  const double stepE = __shfl_sync(0xffffffffu, d, 0), stepL = __shfl_sync(0xffffffffu, d, 1),
               stepP = __shfl_sync(0xffffffffu, d, 2);
  if (lane == 0) {
    p.startE = startE; p.stepE = stepE;
    p.startL = startL; p.stepL = stepL;
    p.startP = startP; p.stepP = stepP;
    p.inv_step = inv_step;
    p.h_fix = __double2ll_rn(0.5 * inv_step * 1099511627776.0);
    p.q0_fix = __double2ll_rn(-rem * inv_step * 1099511627776.0);
  }
  st.nextRemCode = (lin_y(blk - 1, stepP, startP) + step) - 1023.0;  // :190
}

// T6: carrier NCO parameters of the next period; returns cps (written to p when `write`)
__device__ double prepare_carr(const TrackArgs& a, CarrState& st, MsParams& p, bool write) {
  st.w = st.carrFreq * 2.0 * 3.141592653589793;                       // :195
  const double cps = (st.w / a.fs) * 0.15915494309189535;
  if (write) {
    p.cps = cps;
    p.w = st.w;
    p.fs = a.fs;
  }
  return cps;
}

// T6 phase of the next period (remCarrPhase); p.rem_rad is the loop's copy of it
__device__ __forceinline__ void set_carr_phase(MsParams& p, double rem) {
  p.rem_cyc = rem * 0.15915494309189535;
  p.rem_rad = rem;
}

// T6 carry (tracking.py:197): remCarrPhase after a block of `blk` samples, from the period's own w and remCarrPhase
__device__ double carry_carr_phase(double w, double rem, int blk, double fs) {
  const double TWO_PI = 6.283185307179586;  // == 2*np.pi
  double arg_end = w * ((double)blk / fs) + rem;
  double m;
  if (arg_end >= 0.0) {
    // exact remainder without the iterative fmod: with the right integer quotient the fused
    // multiply-add returns x - q*y exactly (the result of fmod is always representable)
    double q = floor(arg_end * 0.15915494309189535);
    m = __fma_rn(-q, TWO_PI, arg_end);
    if (m < 0.0) { q -= 1.0; m = __fma_rn(-q, TWO_PI, arg_end); }
    else if (m >= TWO_PI) { q += 1.0; m = __fma_rn(-q, TWO_PI, arg_end); }
  } else {
    m = fmod(arg_end, TWO_PI);
    if (m != 0.0 && m < 0.0) m += TWO_PI;
  }
  return m;
}

// ---- correlate, variant A: contiguous run of aligned 16-sample groups per thread (any sampling rate)
__device__ __forceinline__ void correlate_groups(const MsParams& P, const int8_t* cur, const float* codeS, int tid,
                                                 double& tEr, double& tEi, double& tPr, double& tPi, double& tLr,
                                                 double& tLi) {
    const int off = (int)(P.pos - (P.pos & ~15LL));
    const int ng = (off + P.blk + 15) >> 4;
    const int gpt = (ng + TRK_THREADS - 1) / TRK_THREADS;
    const int g0 = tid * gpt;
    const int g1 = min(g0 + gpt, ng);
    if (g0 < g1) {
      int ib = 16 * g0 - off;
      const int i0 = max(ib, 0);
      CodeVar E, Pm, L;
      E.init(i0, P.startE, P.stepE, P.inv_step, codeS);
      Pm.init(i0, P.startP, P.stepP, P.inv_step, codeS);
      L.init(i0, P.startL, P.stepL, P.inv_step, codeS);
      // carrier: rot = e^{j theta(ib)}, w[k] = e^{j k dtheta}
      float wr[16], wi[16], w16r, w16i, rotr, roti;
      {
        cis_cycles((double)ib * P.cps + P.rem_cyc, rotr, roti);
        float s1, c1;
        cis_cycles(P.cps, c1, s1);
        wr[0] = 1.f; wi[0] = 0.f; wr[1] = c1; wi[1] = s1;
#pragma unroll
        for (int q = 2; q < 16; ++q) {
          // w^q from the two closest already-known powers keeps the error at a few ulp
          cmul(wr[q], wi[q], wr[q >> 1], wi[q >> 1], wr[q - (q >> 1)], wi[q - (q >> 1)]);
        }
        cis_cycles(16.0 * P.cps, w16r, w16i);
      }
      for (int g = g0; g < g1; ++g, ib += 16) {
        uint4 q4 = *reinterpret_cast<const uint4*>(cur + 16 * g);
        unsigned wq[4] = {q4.x, q4.y, q4.z, q4.w};
        if (ib < 0 || ib + 16 > P.blk) {  // head / tail of the block: zero the foreign samples
#pragma unroll
          for (int b = 0; b < 16; ++b) {
            int i = ib + b;
            if (i < 0 || i >= P.blk) wq[b >> 2] &= ~(0xFFu << (8 * (b & 3)));
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) wq[j] ^= 0x80808080u;
        const int kE = E.e - ib, kP = Pm.e - ib, kL = L.e - ib;
        const int kb = min(min(kE, kP), min(kL, 16));
        // tentative state after the event(s) at kb
        CodeVar E2 = E, P2 = Pm, L2 = L;
        if (kE == kb) E2.advance(P.inv_step, codeS);
        if (kP == kb) P2.advance(P.inv_step, codeS);
        if (kL == kb) L2.advance(P.inv_step, codeS);
        const bool single = (E2.e - ib >= 16) && (P2.e - ib >= 16) && (L2.e - ib >= 16);
        if (single) {
          float Ar = 0.f, Ai = 0.f, Br = 0.f, Bi = 0.f;
#pragma unroll
          for (int b = 0; b < 16; ++b) {
            float x = byte_to_float(wq[b >> 2], b & 3);
            if (b < kb) { Ar = fmaf(x, wr[b], Ar); Ai = fmaf(x, wi[b], Ai); }
            else        { Br = fmaf(x, wr[b], Br); Bi = fmaf(x, wi[b], Bi); }
          }
          float RAr, RAi, RBr, RBi;
          cmul(RAr, RAi, rotr, roti, Ar, Ai);
          cmul(RBr, RBi, rotr, roti, Br, Bi);
          // group halves are float32 (<= 16 exact-int x float products each); totals run in float64
          tEr += (double)(E.s * RAr + E2.s * RBr); tEi += (double)(E.s * RAi + E2.s * RBi);
          tPr += (double)(Pm.s * RAr + P2.s * RBr); tPi += (double)(Pm.s * RAi + P2.s * RBi);
          tLr += (double)(L.s * RAr + L2.s * RBr); tLi += (double)(L.s * RAi + L2.s * RBi);
          E = E2; Pm = P2; L = L2;
        } else {
          // several chip boundaries inside one group (low sampling rates, or E/L boundaries that
          // round to neighbouring samples): sample-by-sample walk
          float rr = rotr, ri = roti;
#pragma unroll
          for (int b = 0; b < 16; ++b) {
            const int i = ib + b;
            while (E.e <= i) E.advance(P.inv_step, codeS);
            while (Pm.e <= i) Pm.advance(P.inv_step, codeS);
            while (L.e <= i) L.advance(P.inv_step, codeS);
            float x = byte_to_float(wq[b >> 2], b & 3);
            float pr = x * rr, pi = x * ri;
            tEr += (double)(E.s * pr); tEi += (double)(E.s * pi);
            tPr += (double)(Pm.s * pr); tPi += (double)(Pm.s * pi);
            tLr += (double)(L.s * pr); tLi += (double)(L.s * pi);
            float nr, ni;
            cmul(nr, ni, rr, ri, wr[1], wi[1]);
            rr = nr; ri = ni;
          }
          // bring the state to the first sample of the next group
          while (E.e <= ib + 15) E.advance(P.inv_step, codeS);
          while (Pm.e <= ib + 15) Pm.advance(P.inv_step, codeS);
          while (L.e <= ib + 15) L.advance(P.inv_step, codeS);
        }
        float nr, ni;
        cmul(nr, ni, rotr, roti, w16r, w16i);
        rotr = nr; roti = ni;
      }
    }
}

// ---- correlate, variant B: every thread owns 8 half-chip segments --------------------------------
// Threshold n (n = -1 .. 2046) is the value n/2 of the prompt code phase; beta(n) is the first sample
// whose phase exceeds it: for even n the boundary of P (chip n/2), for odd n the common boundary of E
// (chip (n-1)/2) and L (chip (n+1)/2).  Samples in [beta(n), beta(n+1)) therefore all have replica
// indices P = floor(n/2)+1, E = floor((n+1)/2), L = E+1 (see DESIGN.md, K5), so a segment is summed
// without any per-sample decision: sum_k x[a+k] w^k with 4*NW fixed twiddles, bytes fetched with
// unaligned 32-bit shared loads + funnel shifts, then one rotation and three signed accumulations.
// If an E boundary and its L twin fall on different samples (phase within 1e-6 of a sample instant)
// the thread falls back to the exact per-sample evaluation for its whole range.
template <int NW>
__device__ __forceinline__ void correlate_segments(const MsParams& P, const int8_t* cur, const float* codeS,
                                                   int tid, double& tEr, double& tEi, double& tPr, double& tPi,
                                                   double& tLr, double& tLi) {
  constexpr int SEGS = 8;          // 2046 half chips / 256 threads
  constexpr int LMAX = 4 * NW;     // longest segment the unrolled path takes
  const int off = (int)(P.pos - (P.pos & ~15LL));
  const int n0 = SEGS * tid - 1;
  int beta[SEGS + 1];
  bool irregular = false;
#pragma unroll
  for (int s = 0; s <= SEGS; ++s) {
    const int n = n0 + s;
    int b;
    if (n < 0) b = 0;
    else if (n > 2046) b = P.blk;
    else if ((n & 1) == 0) b = next_event(n >> 1, P.startP, P.stepP, P.inv_step);
    else {
      const int c = (n - 1) >> 1;
      const double q = ((double)c - P.startE) * P.inv_step;
      const double fl = floor(q);
      b = (int)fl + 1;
      const double fr = q - fl;
      if (fr < 1e-6 || fr > 1.0 - 1e-6) {   // too close to a sample instant: settle E and L exactly
        b = next_event(c, P.startE, P.stepE, P.inv_step);
        const int bl = next_event(c + 1, P.startL, P.stepL, P.inv_step);
        if (bl != b) irregular = true;
      }
    }
    beta[s] = max(0, min(b, P.blk));   // (a prediction of -1 occurs when rem is within rounding of one step)
  }
  if (beta[0] >= P.blk) return;
  if (irregular) {
    // exact per-sample evaluation of the three replica indices (tracking.py:166-188 verbatim)
    for (int i = beta[0]; i < beta[SEGS]; ++i) {
      const int ie = (int)ceil(lin_y(i, P.stepE, P.startE));
      const int ip = (int)ceil(lin_y(i, P.stepP, P.startP));
      const int il = (int)ceil(lin_y(i, P.stepL, P.startL));
      float sn, cs;
      cis_cycles((double)i * P.cps + P.rem_cyc, cs, sn);
      const float x = (float)cur[off + i];
      const float pr = x * cs, pi = x * sn;
      tEr += (double)(codeS[ie] * pr); tEi += (double)(codeS[ie] * pi);
      tPr += (double)(codeS[ip] * pr); tPi += (double)(codeS[ip] * pi);
      tLr += (double)(codeS[il] * pr); tLi += (double)(codeS[il] * pi);
    }
    return;
  }
  // twiddles w^k, k = 0 .. LMAX-1 for the samples of a chunk, and the five rotor steps
  // w^(LMAX-4) .. w^LMAX (segment lengths that occur), anchored on a freshly evaluated w^(LMAX-2)
  float wr[LMAX], wi[LMAX], zr[5], zi[5];
  {
    float s1, c1;
    cis_cycles(P.cps, c1, s1);
    wr[0] = 1.f; wi[0] = 0.f;
    if (LMAX > 1) { wr[1] = c1; wi[1] = s1; }
#pragma unroll
    for (int q = 2; q < LMAX; ++q)
      cmul(wr[q], wi[q], wr[q >> 1], wi[q >> 1], wr[q - (q >> 1)], wi[q - (q >> 1)]);
    cis_cycles((double)(LMAX - 2) * P.cps, zr[2], zi[2]);
    float c2, s2;
    cmul(c2, s2, c1, s1, c1, s1);
    cmul(zr[3], zi[3], zr[2], zi[2], c1, s1);
    cmul(zr[4], zi[4], zr[2], zi[2], c2, s2);
    cmul(zr[1], zi[1], zr[2], zi[2], c1, -s1);
    cmul(zr[0], zi[0], zr[2], zi[2], c2, -s2);
  }
  float rotr = 1.f, roti = 0.f;
  float fEr = 0.f, fEi = 0.f, fPr = 0.f, fPi = 0.f, fLr = 0.f, fLi = 0.f;
  bool fresh = true;
#pragma unroll
  for (int s = 0; s < SEGS; ++s) {
    int a = beta[s];
    const int b = beta[s + 1];
    if (b <= a) continue;
    const int n = n0 + s;
    const float sP = codeS[(n >> 1) + 1];
    const int ie = (n + 1) >> 1;
    const float sE = codeS[ie], sL = codeS[ie + 1];
    float Sr = 0.f, Si = 0.f;   // sum of this segment, referred to the carrier phase of sample `a0`
    const int a0 = a;
    if (fresh) {
      cis_cycles((double)a * P.cps + P.rem_cyc, rotr, roti);
      fresh = false;
    }
    float cr = 1.f, ci = 0.f;   // rotor of the current chunk relative to a0
    bool first_chunk = true;
    while (a < b) {             // one chunk unless the segment is longer than LMAX (other sampling rates)
      const int len = min(b - a, LMAX);
      const int addr = off + a;
      const unsigned* wp = reinterpret_cast<const unsigned*>(cur + (addr & ~3));
      const int sh = (addr & 3) * 8;
      unsigned raw[NW + 1];
#pragma unroll
      for (int q = 0; q <= NW; ++q) raw[q] = wp[q];
      unsigned wq[NW];
#pragma unroll
      for (int q = 0; q < NW; ++q) wq[q] = __funnelshift_r(raw[q], raw[q + 1], sh);
      if (len > LMAX - 4) {     // the usual case: only the last word is partial
        wq[NW - 1] &= 0xFFFFFFFFu >> (8 * (LMAX - len));
      } else {
#pragma unroll
        for (int q = 0; q < NW; ++q) {
          const int keep = len - 4 * q;
          if (keep < 4) wq[q] &= keep <= 0 ? 0u : (0xFFFFFFFFu >> (8 * (4 - keep)));
        }
      }
      float pr = 0.f, pi = 0.f;
#pragma unroll
      for (int q = 0; q < NW; ++q) {
        const unsigned w = wq[q] ^ 0x80808080u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float x = byte_to_float(w, k);
          pr = fmaf(x, wr[4 * q + k], pr);
          pi = fmaf(x, wi[4 * q + k], pi);
        }
      }
      a += len;
      if (first_chunk) {
        Sr = pr; Si = pi;
        first_chunk = false;
      } else {
        float tr, ti;
        cmul(tr, ti, cr, ci, pr, pi);
        Sr += tr; Si += ti;
      }
      if (a < b) {   // multi-chunk segment: advance the chunk rotor by w^LMAX
        float tr, ti;
        cmul(tr, ti, cr, ci, zr[4], zi[4]);
        cr = tr; ci = ti;
      }
    }
    float Rr, Ri;
    cmul(Rr, Ri, rotr, roti, Sr, Si);
    // eight segment sums per thread stay float32 (rounding 6e-8 of a 1/256 share of the total,
    // independent between threads); everything across threads is added in float64
    fEr = fmaf(sE, Rr, fEr); fEi = fmaf(sE, Ri, fEi);
    fPr = fmaf(sP, Rr, fPr); fPi = fmaf(sP, Ri, fPi);
    fLr = fmaf(sL, Rr, fLr); fLi = fmaf(sL, Ri, fLi);
    // rotor for the next segment
    const int len = b - a0;
    const int j = len - (LMAX - 4);
    if (j >= 0 && j <= 4) {
      float sr = zr[0], si = zi[0];
      if (j == 1) { sr = zr[1]; si = zi[1]; }
      if (j == 2) { sr = zr[2]; si = zi[2]; }
      if (j == 3) { sr = zr[3]; si = zi[3]; }
      if (j == 4) { sr = zr[4]; si = zi[4]; }
      float nr, ni;
      cmul(nr, ni, rotr, roti, sr, si);
      rotr = nr; roti = ni;
    } else {
      fresh = true;
    }
  }
  tEr += (double)fEr; tEi += (double)fEi; tPr += (double)fPr; tPi += (double)fPi; tLr += (double)fLr; tLi += (double)fLi;
}

// ---- correlate, variant C: half-chip segments with exact integer segment sums --------------------
// Same segmentation as variant B.  The per-sample twiddles w^k are quantised once per period to Q38
// (Q30 for the widest segments) fixed point and split into five (four) signed base-256 digits, so a segment sum is 10 (8) dot products per four
// samples (dp4a, int32 accumulation is exact); rotors, code signs and all accumulation are float64.
// The only approximation left is the 2^-31 twiddle quantisation (relative error of a correlator
// output ~5e-11), which keeps the carried code phase within ~1e-11 chips of the reference's and makes
// chip reassignments (DESIGN.md section 5) a once-per-many-minutes event instead of a per-second one.
template <int NW> struct ExactDigits { static constexpr int value = NW <= 5 ? 5 : 4; };   // Q38 twiddles when registers allow, else Q30
struct __align__(16) ExactTables {
  signed char tw[2][5][32];   // [re/im][digit][k], read as packed words
  double z[5][2];             // rotor steps e^{j 2 pi (LMAX-4+j) cps}
};

// Branch-free float64 sin/cos for |th| < 5e5 rad: three-term Cody-Waite reduction by pi/2 (33-bit
// pieces, k < 2^19 so every k*piece is exact) and Taylor polynomials on [-pi/4, pi/4]; max error
// 2.3e-16 over [0, 7e4] (checked against libm).  Straight-line code, so it overlaps with the integer
// work around it instead of stalling the warp like the library routine's branches do.
__device__ __forceinline__ void sincos_reduced(double th, double& sn, double& cs) {
  const double k = rint(th * 0.6366197723675814);
  double r = fma(-k, 1.5707963267341256, th);
  r = fma(-k, 6.077100506303966e-11, r);
  r = fma(-k, 2.0222662487959506e-21, r);
  const double r2 = r * r;
  double ps = -7.647163731819816e-13;                 // -1/15!
  ps = fma(ps, r2, 1.6059043836821613e-10);           //  1/13!
  ps = fma(ps, r2, -2.505210838544172e-08);           // -1/11!
  ps = fma(ps, r2, 2.7557319223985893e-06);           //  1/9!
  ps = fma(ps, r2, -1.984126984126984e-04);           // -1/7!
  ps = fma(ps, r2, 8.333333333333333e-03);            //  1/5!
  ps = fma(ps, r2, -1.6666666666666666e-01);          // -1/3!
  const double s0 = fma(ps * r2, r, r);
  double pc = 4.779477332387385e-14;                  //  1/16!
  pc = fma(pc, r2, -1.1470745597729725e-11);          // -1/14!
  pc = fma(pc, r2, 2.08767569878681e-09);             //  1/12!
  pc = fma(pc, r2, -2.755731922398589e-07);           // -1/10!
  pc = fma(pc, r2, 2.48015873015873e-05);             //  1/8!
  pc = fma(pc, r2, -1.388888888888889e-03);           // -1/6!
  pc = fma(pc, r2, 4.1666666666666664e-02);           //  1/4!
  pc = fma(pc, r2, -0.5);
  const double c0 = fma(pc, r2, 1.0);
  const int q = (int)(long long)k & 3;
  const double sa = (q & 1) ? c0 : s0, ca = (q & 1) ? s0 : c0;
  sn = (q & 2) ? -sa : sa;
  cs = ((q + 1) & 2) ? -ca : ca;
}

__device__ __forceinline__ void cis_cycles_f64(double cyc, double& c, double& s) {
  cyc -= rint(cyc);
  sincospi(2.0 * cyc, &s, &c);
}

// executed by the 32 lanes of the carrier warp once the next period's cps is known
template <int NW>
__device__ __forceinline__ void build_exact_tables(ExactTables& T, double cps, int lane) {
  constexpr int LMAX = 4 * NW;
  constexpr int ND = ExactDigits<NW>::value;
  // twiddle w^lane on lanes 0 .. LMAX-1, rotor step j (power LMAX-4+j) on lane Z0+j: on the spare lanes next to the
  // twiddle lanes in the same sincospi when there are enough of them, else in a second pass
  constexpr int Z0 = (LMAX + 5 <= 32) ? LMAX : 0;
  const bool tw = lane < LMAX, zs = lane >= Z0 && lane < Z0 + 5;
  if (tw || (Z0 > 0 && zs)) {
    double c, s;
    cis_cycles_f64((double)(tw ? lane : LMAX - 4 + (lane - Z0)) * cps, c, s);
    if (!tw) {
      T.z[lane - Z0][0] = c;
      T.z[lane - Z0][1] = s;
      return;
    }
    const double one = (double)(1LL << (8 * ND - 2));      // Q30 (4 digits) or Q38 (5 digits)
    long long w[2] = {__double2ll_rn(c * one), __double2ll_rn(s * one)};
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      long long v = w[q];
#pragma unroll
      for (int d = 0; d < ND - 1; ++d) {
        const long long b = ((v + 128) & 0xFF) - 128;   // signed digit in [-128, 127]
        T.tw[q][d][lane] = (signed char)b;
        v = (v - b) >> 8;
      }
      T.tw[q][ND - 1][lane] = (signed char)v;           // |v| <= 65
    }
  }
  if (Z0 == 0 && zs) cis_cycles_f64((double)(LMAX - 4 + lane) * cps, T.z[lane][0], T.z[lane][1]);
}

// ---- cold paths of the exact correlator, kept out of line: the unrolled segment loop has to stay inside the SM's
// instruction cache (with these inlined eight times the kernel was 115 KB of SASS and instruction fetch from the
// GPC-level cache ran at 88 % of its peak -- profiles/ncu_summary_r1_v3.md)
// (results come back by value: an output reference would pin the caller's loop-carried state in local memory)
constexpr int IRREGULAR = 1 << 30;   // flag on a settled boundary: E and L switch at different samples there
__device__ __noinline__ int settle_boundary(int n, const MsParams& P) {
  if ((n & 1) == 0) return max(0, min(next_event(n >> 1, P.startP, P.stepP, P.inv_step), P.blk));
  const int c = (n - 1) >> 1;
  const int b = next_event(c, P.startE, P.stepE, P.inv_step);
  const int bl = next_event(c + 1, P.startL, P.stepL, P.inv_step);
  return max(0, min(b, P.blk)) | (bl != b ? IRREGULAR : 0);
}

__device__ __noinline__ double2 start_rotor(int a, const MsParams& P) {   // (cos, sin)
  // the reference's own phase expression for sample a (tracking.py:193-195), evaluated in radians so that no
  // rounded 1/(2 pi) scales a 6e4 rad argument (that error would be common to all threads)
  const double th = P.w * ((double)a / P.fs) + P.rem_rad;
  double sn, cs;
  if (fabs(th) < 5.0e5) sincos_reduced(th, sn, cs);
  else sincos(th, &sn, &cs);
  return make_double2(cs, sn);
}

__device__ __noinline__ void correlate_per_sample(const MsParams& P, const int8_t* cur, const unsigned char* codeB, int off,
                                                  int i0, int i1, double* acc) {
  // exact per-sample evaluation (tracking.py:166-219 verbatim, float64)
  for (int i = i0; i < i1; ++i) {
    const int ie = (int)ceil(lin_y(i, P.stepE, P.startE));
    const int ip = (int)ceil(lin_y(i, P.stepP, P.startP));
    const int il = (int)ceil(lin_y(i, P.stepL, P.startL));
    double cs, sn;
    cis_cycles_f64((double)i * P.cps + P.rem_cyc, cs, sn);
    const double x = (double)cur[off + i];
    const double pr = x * cs, pi = x * sn;
    const double ce = codeB[ie] ? -1.0 : 1.0, cp = codeB[ip] ? -1.0 : 1.0, cl = codeB[il] ? -1.0 : 1.0;
    acc[0] += ce * pr; acc[1] += ce * pi;
    acc[2] += cp * pr; acc[3] += cp * pi;
    acc[4] += cl * pr; acc[5] += cl * pi;
  }
}

// +-x without a multiply: the code value's sign bit (0 / 0x80000000) is XORed into the high word
__device__ __forceinline__ double flip_sign(double x, unsigned m) {
  return __hiloint2double(__double2hiint(x) ^ (int)m, __double2loint(x));
}

// exact double of the 46-bit integer lo + mid*2^16 + hi*2^32 (|value| < 2^51) without an int->double conversion
// instruction: the integer, offset by 2^51, is written straight into the mantissa of 2^52 and the offset removed by
// one exact subtraction
__device__ __forceinline__ double digits_to_double(int lo, int mid, int hi) {
  long long v = (long long)mid * 65536 + (long long)lo;
  v += (long long)hi << 32;
  v += 0x4338000000000000LL;            // 2^52 exponent pattern, plus the 2^51 offset inside the mantissa
  return __longlong_as_double(v) - 6755399441055744.0;   // 2^52 + 2^51
}

// Exact correlator.  Thread tid walks the SEGS half-chip segments n = SEGS*tid - 1 ... in a ROLLED loop: one copy
// of the segment body (about 170 instructions) instead of eight keeps the whole period loop inside the SM's
// instruction cache (the unrolled kernel fetched instructions from the GPC-level cache at 88 % of that cache's
// peak and stalled on it -- profiles/ncu_summary_r1_v3.md).
template <int NW, int SEGS>
__device__ __forceinline__ void correlate_exact(const MsParams& P, const MsParams& Pcold, const int8_t* cur,
                                                const unsigned char* codeB, const ExactTables& T, int tid,
                                                double& tEr, double& tEi, double& tPr, double& tPi, double& tLr,
                                                double& tLi) {
  constexpr int LMAX = 4 * NW;
  constexpr int ND = ExactDigits<NW>::value;
  static_assert(SEGS == 8, "sign bytes are fetched for 8 half-chip segments per thread");
  const int off = (int)(P.pos - (P.pos & ~15LL));
  const int n0 = SEGS * tid - 1;
  // boundaries are equally spaced in the predicted (real-valued) sample index q_n = (n/2 - rem) / step;
  // the prediction runs in Q40 fixed point (error < 1e-9 samples over the 2046 thresholds)
  const long long FR_ONE = 1LL << 40, FR_EPS = 1099512;   // 1e-6 in Q40
  long long qf = P.q0_fix + (long long)n0 * P.h_fix;
  // boundary of threshold n -> first sample of segment n, with IRREGULAR possibly set
  auto boundary = [&](int n, long long q) -> int {
    if (n < 0) return 0;
    if (n > 2046) return P.blk;
    const long long fr = q & (FR_ONE - 1);
    // too close to a sample instant: settle with the exact expressions (Pcold: the shared-memory copy of the
    // parameters, so that P can stay in registers)
    if (fr < FR_EPS || fr > FR_ONE - FR_EPS) return settle_boundary(n, Pcold);
    return max(0, min((int)(q >> 40) + 1, P.blk));   // (a prediction of -1 occurs when rem is within rounding of one step)
  };
  int a = boundary(n0, qf);
  if ((a & ~IRREGULAR) >= P.blk) return;
  // Thread 0's first segment (n = -1: the samples before the first prompt threshold) is empty unless the block starts
  // at or before a threshold.  Skipping it makes that thread's first rotor evaluation (start_rotor, below) fall in
  // the same iteration as its warp's other lanes: one evaluation per warp instead of two (measured at 32 recordings:
  // warp 0's correlation ended ~820 cycles after the other warps' with the second evaluation, ~460 without).
  int s0 = 0;
  if (n0 < 0) {
    const int b0 = boundary(0, qf + P.h_fix);
    if ((b0 & ~IRREGULAR) == (a & ~IRREGULAR)) { s0 = 1; qf += P.h_fix; a = b0; }
  }
  // packed twiddle digits: tw[c][d] word q holds samples 4q .. 4q+3
  int twr[ND][NW], twi[ND][NW];
#pragma unroll
  for (int d = 0; d < ND; ++d)
#pragma unroll
    for (int q = 0; q < NW; ++q) {
      twr[d][q] = reinterpret_cast<const int*>(T.tw[0][d])[q];
      twi[d][q] = reinterpret_cast<const int*>(T.tw[1][d])[q];
    }
  // code signs of the 5 chips this thread's segments touch (chip 4*tid onwards), one byte each (0 = +1, 0x80 = -1):
  // two conflict-free aligned words per period instead of three float64 table reads per segment
  unsigned sg_lo = reinterpret_cast<const unsigned*>(codeB)[tid];       // chips 4 tid .. 4 tid + 3
  unsigned sg_hi = reinterpret_cast<const unsigned*>(codeB)[tid + 1];   // chip 4 tid + 4 in its low byte
  double rotr = 1.0, roti = 0.0;
  double aEr = 0, aEi = 0, aPr = 0, aPi = 0, aLr = 0, aLi = 0;
  bool fresh = true;
  const unsigned cur_s = smem_addr(cur), z_s = smem_addr(&T.z[0][0]);
#pragma unroll 1
  for (int s = s0; s < SEGS; ++s) {
    qf += P.h_fix;
    const int b = boundary(n0 + s + 1, qf);
    const int len = (b & ~IRREGULAR) - (a & ~IRREGULAR);
    if (len > 0) {
      if (len > LMAX || ((a | b) & IRREGULAR)) {
        // rare: a segment longer than the twiddle table, or one whose boundary is not shared by E, P and L.
        // Per-sample evaluation; its sums join the scaled accumulators through an exact power of two.
        double acc[6] = {0, 0, 0, 0, 0, 0};
        correlate_per_sample(Pcold, cur, codeB, off, a & ~IRREGULAR, b & ~IRREGULAR, acc);
        const double up = (double)(1LL << (8 * ND - 2));
        aEr += acc[0] * up; aEi += acc[1] * up; aPr += acc[2] * up; aPi += acc[3] * up; aLr += acc[4] * up; aLi += acc[5] * up;
        fresh = true;
      } else {
        // chips relative to 4 tid: E = floor(s/2), L = E + 1, P = floor((s+1)/2) = E (s even) or L (s odd)
        // (n = 8 tid - 1 + s); the sign bytes are shifted down by one chip after every odd s
        const unsigned mE = sg_lo << 24, mL = __byte_perm(sg_lo, 0u, 0x1444), mP = (s & 1) ? mL : mE;
        if (fresh) {
          const double2 r0 = start_rotor(a, Pcold);
          rotr = r0.x; roti = r0.y;
          fresh = false;
        }
        const int sh = ((off + a) & 3) * 8;
        unsigned raw[NW + 1];   // the NW + 1 words from the one holding sample a onwards
        {
          // 16-byte loads from the aligned base: lanes sit ~150 bytes apart, which put the 32-bit loads of a warp
          // on ~6 distinct banks (6 wavefronts per load); a 16-byte load spreads a quarter warp over 8 bank quads
          // (2 wavefronts per quarter).  The last quad is fetched only by the lanes that need a word of it.
          constexpr int NQ = (NW + 7) / 4;          // quads covering words j .. j + NW for every j in 0 .. 3
          const int ab = (off + a) & ~15, j = ((off + a) >> 2) & 3;
          unsigned wd[4 * NQ];
#pragma unroll
          for (int q = 0; q < NQ; ++q) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (q < NQ - 1 || j + NW >= 4 * (NQ - 1)) v = lds_u32x4(cur, cur_s, ab + 16 * q);
            wd[4 * q] = v.x; wd[4 * q + 1] = v.y; wd[4 * q + 2] = v.z; wd[4 * q + 3] = v.w;
          }
          unsigned t[NW + 2];
#pragma unroll
          for (int q = 0; q < NW + 2; ++q) t[q] = (j & 2) ? wd[q + 2] : wd[q];
#pragma unroll
          for (int q = 0; q <= NW; ++q) raw[q] = (j & 1) ? t[q + 1] : t[q];
        }
        // bytes at and beyond len are not part of this segment: the last word is always masked, the others only
        // in a short segment (fewer than LMAX - 4 samples: block edges)
        unsigned w[NW];
#pragma unroll
        for (int q = 0; q < NW; ++q) w[q] = __funnelshift_r(raw[q], raw[q + 1], sh);
        w[NW - 1] &= __funnelshift_lc(0xFFFFFFFFu, 0u, max(8 * (len - 4 * (NW - 1)), 0));
        if (len < LMAX - 4) {
#pragma unroll
          for (int q = 0; q < NW - 1; ++q) w[q] &= __funnelshift_lc(0xFFFFFFFFu, 0u, max(8 * (len - 4 * q), 0));
        }
        int xr[ND], xi[ND];
#pragma unroll
        for (int d = 0; d < ND; ++d) { xr[d] = 0; xi[d] = 0; }
#pragma unroll
        for (int q = 0; q < NW; ++q) {
#pragma unroll
          for (int d = 0; d < ND; ++d) {
            xr[d] = __dp4a((int)w[q], twr[d][q], xr[d]);
            xi[d] = __dp4a((int)w[q], twi[d][q], xi[d]);
          }
        }
        // exact recombination of the base-256 digits (|value| < 2^51): digit pairs merge in int32
        // (|x1*256 + x0| < 2^28), the rest in int64, and the result goes straight into a float64 mantissa
        const double Sr = digits_to_double(xr[1] * 256 + xr[0], xr[3] * 256 + xr[2], ND == 5 ? xr[ND - 1] : 0);
        const double Si = digits_to_double(xi[1] * 256 + xi[0], xi[3] * 256 + xi[2], ND == 5 ? xi[ND - 1] : 0);
        const double Rr = fma(rotr, Sr, -(roti * Si)), Ri = fma(rotr, Si, roti * Sr);
        aEr += flip_sign(Rr, mE); aEi += flip_sign(Ri, mE);
        aPr += flip_sign(Rr, mP); aPi += flip_sign(Ri, mP);
        aLr += flip_sign(Rr, mL); aLi += flip_sign(Ri, mL);
        const int j = len - (LMAX - 4);
        if (j >= 0) {
          const double2 z = lds_f64x2(&T.z[0][0], z_s, 16 * j);
          const double zr = z.x, zi = z.y;
          const double nr = fma(rotr, zr, -(roti * zi)), ni = fma(rotr, zi, roti * zr);
          rotr = nr; roti = ni;
        } else {
          fresh = true;
        }
      }
    }
    a = b;
    if (s & 1) { sg_lo = __funnelshift_r(sg_lo, sg_hi, 8); sg_hi >>= 8; }
  }
  const double sc = 1.0 / (double)(1LL << (8 * ND - 2));   // 2^-30 or 2^-38
  tEr += aEr * sc; tEi += aEi * sc; tPr += aPr * sc; tPi += aPi * sc; tLr += aLr * sc; tLi += aLi * sc;
}

template <bool BULK, int NW, bool EXACT, int NT>
__global__ void __launch_bounds__(NT, 2) track_kernel(TrackArgs a) {
  SGX_DYN_SMEM(smem);
  int8_t* buf0 = (int8_t*)smem;
  int8_t* buf1 = buf0 + a.win;
  __shared__ MsParams prm;
  constexpr int NWARPS = NT / 32;
  __shared__ double red[NWARPS][6];
  __shared__ float codeS[1040];  // 1025 used; the tail absorbs indices reached only by masked samples
  __shared__ unsigned long long mbar[2];
  __shared__ ExactTables xt;
  __shared__ CodeState cstS;   // loop state lives in shared memory: only warps 0 / 1 touch it, and keeping it
  __shared__ CarrState rstS;   // out of the register file leaves the correlator loop the registers
  __shared__ __align__(4) unsigned char codeB[EXACT ? 1040 : 4];   // code sign bytes: 0 = +1, 0x80 = -1
  __shared__ long long stampS[NWARPS][TRK_PROF_N + 1];   // SGX_TRK_PROF phase stamps of the current period
  __shared__ double remNextS;  // remCarrPhase of the next period (thread 64)

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int cid = blockIdx.x;  // recording * n_channels + channel
  const int rid = cid / a.n_channels;
  const sgx_channel chn = a.ch[cid];
  if (chn.prn == 0) {  // tracking.py:99 -- idle channel, no record
    if (tid == 0) {
      a.ms_done[cid] = 0;
      a.status[cid] = SGX_OK;
      if (a.state) { a.state[cid].k = 0; a.state[cid].status = SGX_OK; }
    }
    return;
  }
  const int8_t* rec = a.rec + (long long)rid * a.rec_stride;
  const long long rec_len = a.rec_len[rid];
  const long long rec_alloc = (rec_len + 15) & ~15LL;
  {  // padded code [c1022, c0..c1022, c0] (tracking.py:109-111)
    const int8_t* c = a.chips + (chn.prn - 1) * 1023;
    for (int i = tid; i < 1040; i += NT) {
      codeS[i] = i < 1025 ? (float)c[(i + 1022) % 1023] : 0.f;
      if (EXACT) codeB[i] = codeS[i] < 0.f ? 0x80 : 0;
    }
  }
  int k_start = 0;
  if (a.resume) {
    const TrackState* ts = a.state + cid;
    if (ts->status != SGX_PAUSED) return;   // finished (or failed) in an earlier launch
    k_start = ts->k;
    if (tid < 32) { CodeState c = ts->c; prepare_code(a, c, rec_len, prm, lane); if (lane == 0) cstS = c; }
    if (tid == 32) { CarrState r = ts->r; prepare_carr(a, r, prm, true); set_carr_phase(prm, r.remCarrPhase); rstS = r; }
    if (tid == 0 && BULK) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); }
  } else {
    if (tid < 32) {
      CodeState c;
      c.codeFreq = a.codeFreqBasis;          // :114
      c.remCodePhase = 0.0;
      c.oldCodeNco = c.oldCodeError = 0.0;
      c.nextRemCode = 0.0;
      c.pos = a.skip + (long long)chn.codePhase;  // :107
      prepare_code(a, c, rec_len, prm, lane);
      if (lane == 0) cstS = c;
    }
    if (tid == 0 && BULK) { mbar_init(&mbar[0], 1); mbar_init(&mbar[1], 1); }
    if (tid == 32) {
      CarrState r;
      r.carrFreq = chn.acquiredFreq;         // :118
      r.carrFreqBasis = chn.acquiredFreq;
      r.remCarrPhase = 0.0;
      r.oldCarrNco = r.oldCarrError = 0.0;
      prepare_carr(a, r, prm, true);
      set_carr_phase(prm, r.remCarrPhase);
      rstS = r;
    }
  }
  if (EXACT && (tid >> 5) == 1) {   // the carrier thread's warp builds the twiddle / rotor tables
    const double cps = __shfl_sync(0xffffffffu, tid == 32 ? prm.cps : 0.0, 0);
    build_exact_tables<(NW > 0 ? NW : 1)>(xt, cps, tid & 31);
  }
  __syncthreads();

  // stage the window of period 0
  auto stage = [&](int8_t* dst, long long pos) {
    long long al = pos & ~15LL;
    long long nb = rec_alloc - al;
    if (nb > a.win) nb = a.win;
    if (nb <= 0) return 0;
    if (BULK) {
      return (int)nb;
    } else {
      const int8_t* src = rec + al;
      for (int o = tid * 16; o < (int)nb; o += NT * 16) cp_async16(dst + o, src + o);
      cp_async_commit();
      return (int)nb;
    }
  };
  unsigned phase0 = 0, phase1 = 0;  // mbarrier phase parity per buffer
  bool pending0 = false, pending1 = false;
  if (prm.stop == 0) {   // window of the first period of this launch, into the buffer of its parity
    const int par = k_start & 1;
    int nb = stage(par ? buf1 : buf0, prm.pos);
    if (BULK) {
      if (nb > 0) {
        if (tid == 0) bulk_load(par ? buf1 : buf0, rec + (prm.pos & ~15LL), (unsigned)nb, &mbar[par]);
        if (par) pending1 = true; else pending0 = true;
      }
      // and the window of the second period (later windows are issued at the end of the bookkeeping); the loop
      // records it as pending at the start of the first period
      const long long npos = prm.pos + prm.blk;
      const int nb1 = stage(par ? buf0 : buf1, npos);
      if (tid == 0 && nb1 > 0 && k_start < a.ms) bulk_load(par ? buf0 : buf1, rec + (npos & ~15LL), (unsigned)nb1, &mbar[par ^ 1]);
    }
  }

  int k = k_start;
  for (; k < a.ms; ++k) {
    const MsParams P = prm;
    if (P.stop != 0) break;
    const bool stamp = a.prof && (tid & 31) == 0;
    // (stamps go to shared memory: a register array would hold registers across the whole period, and the compiler
    // kept it in local memory, with a load on every period's path even with profiling off)
    long long* ts = stampS[tid >> 5];
    if (stamp) ts[0] = clock64();
    int8_t* cur = (k & 1) ? buf1 : buf0;
    int8_t* nxt = (k & 1) ? buf0 : buf1;
    // ---- make this period's samples visible ------------------------------------------------
    if (BULK) {
      if (k & 1) { if (pending1) { mbar_wait(&mbar[1], phase1); phase1 ^= 1; pending1 = false; } }
      else       { if (pending0) { mbar_wait(&mbar[0], phase0); phase0 ^= 1; pending0 = false; } }
    } else {
      if (k == k_start) { cp_async_wait_all(); __syncthreads(); }
    }
    // ---- prefetch the next period's window -------------------------------------------------
    // (bulk copy: issued by thread 0 at the end of the previous period's bookkeeping, or before the loop -- issued
    // here it delayed warp 0's correlation by ~200 cycles every period)
    {
      long long npos = P.pos + P.blk;
      int nb = stage(nxt, npos);
      if (BULK && nb > 0) {
        if (k & 1) pending0 = true; else pending1 = true;
      }
    }
    // T6 carry (tracking.py:197): remCarrPhase after this period's block needs only this period's parameters; computed
    // here, on a warp that is not the last to finish its correlation, it is off the bookkeeping's path
    if (tid == 64) remNextS = carry_carr_phase(P.w, P.rem_rad, P.blk, P.fs);
    if (stamp) ts[1] = clock64();

    double tEr = 0.0, tEi = 0.0, tPr = 0.0, tPi = 0.0, tLr = 0.0, tLi = 0.0;
    if (EXACT)       correlate_exact<(NW > 0 ? NW : 1), 2048 / NT>(P, prm, cur, codeB, xt, tid, tEr, tEi, tPr, tPi, tLr, tLi);
    else if (NW > 0) correlate_segments<(NW > 0 ? NW : 1)>(P, cur, codeS, tid, tEr, tEi, tPr, tPi, tLr, tLi);
    else             correlate_groups(P, cur, codeS, tid, tEr, tEi, tPr, tPi, tLr, tLi);
    // I arm = sin (imaginary part), Q arm = cos (real part): tracking.py:205-207
    if (stamp) ts[2] = clock64();
    double v0 = warp_sum_f64(tEi), v1 = warp_sum_f64(tEr), v2 = warp_sum_f64(tPi), v3 = warp_sum_f64(tPr),
           v4 = warp_sum_f64(tLi), v5 = warp_sum_f64(tLr);
    if ((tid & 31) == 0) {
      double* r = red[tid >> 5];
      r[0] = v0; r[1] = v1; r[2] = v2; r[3] = v3; r[4] = v4; r[5] = v5;
    }
    if (!BULK) cp_async_wait_all();
    __syncthreads();
    if (stamp) ts[3] = clock64();
    // Bookkeeping: every lane of warp 0 runs the code loop and every lane of warp 1 the carrier loop (same values on
    // all lanes, so that independent operations of a chain can be spread over lanes); lane 0 writes the results.
    if (tid < 32) {          // ---- code loop: DLL (tracking.py:238-251), T5, T3/T4 of the next period
      CodeState cst = cstS;
      const int blk = prm.blk;   // (P.blk would stay live in a register across the correlation)
      __syncwarp();   // every lane has read the state before lane 0 writes it back
      double I_E = 0.0, Q_E = 0.0, I_L = 0.0, Q_L = 0.0;
      for (int w = 0; w < NWARPS; ++w) { I_E += red[w][0]; Q_E += red[w][1]; I_L += red[w][4]; Q_L += red[w][5]; }
      cst.remCodePhase = cst.nextRemCode;
      cst.pos = cst.pos + blk;   // cst.pos is this period's P.pos
      const double mag = sqrt(lane == 1 ? I_L * I_L + Q_L * Q_L : I_E * I_E + Q_E * Q_E);   // lane 0: early, 1: late
      const double em = __shfl_sync(0xffffffffu, mag, 0), lm = __shfl_sync(0xffffffffu, mag, 1);
      double codeError = (em - lm) / (em + lm);
      double codeNco = cst.oldCodeNco + a.c1code * (codeError - cst.oldCodeError) + codeError * a.c2code;
      cst.oldCodeNco = codeNco;
      cst.oldCodeError = codeError;
      cst.codeFreq = a.codeFreqBasis - codeNco;
      if (k + 1 < a.ms) prepare_code(a, cst, rec_len, prm, lane);
      if (lane == 0) {
        cstS = cst;
        // window of the period after next, into this period's buffer (all warps are done with it)
        if (BULK && k + 1 < a.ms && prm.stop == 0) {
          const long long npos = prm.pos + prm.blk;
          const int nb = stage(cur, npos);
          if (nb > 0) bulk_load(cur, rec + (npos & ~15LL), (unsigned)nb, &mbar[k & 1]);
        }
        double* o = a.out + (long long)cid * SGX_TRACK_FIELDS * a.ms + k;   // record (tracking.py:255-275)
        const long long m = a.ms;
        o[0 * m] = (double)(cst.pos + a.abs_base);  // fid.tell() after the read
        o[1 * m] = cst.codeFreq;
        o[4 * m] = I_E; o[5 * m] = I_L; o[6 * m] = Q_E; o[8 * m] = Q_L;
        o[9 * m] = codeError; o[10 * m] = codeNco;
      }
    } else if (tid < 64) {   // ---- carrier loop: PLL (tracking.py:223-235), T6 of the next period, twiddle tables
      CarrState rst = rstS;
      __syncwarp();   // every lane has read the state before lane 0 writes it back
      double I_P = 0.0, Q_P = 0.0;
      for (int w = 0; w < NWARPS; ++w) { I_P += red[w][2]; Q_P += red[w][3]; }
      double carrError = atan(Q_P / I_P) * 0.5 / 3.141592653589793;   // x/2.0 == x*0.5 exactly
      double carrNco = rst.oldCarrNco + a.c1carr * (carrError - rst.oldCarrError) + carrError * a.c2carr;
      rst.oldCarrNco = carrNco;
      rst.oldCarrError = carrError;
      rst.carrFreq = rst.carrFreqBasis + carrNco;
      if (k + 1 < a.ms) {
        const double cps = prepare_carr(a, rst, prm, lane == 0);
        if (EXACT) build_exact_tables<(NW > 0 ? NW : 1)>(xt, cps, lane);
      }
      if (lane == 0) {
        double* o = a.out + (long long)cid * SGX_TRACK_FIELDS * a.ms + k;
        const long long m = a.ms;
        o[2 * m] = rst.carrFreq;
        o[3 * m] = I_P; o[7 * m] = Q_P;
        o[11 * m] = carrError; o[12 * m] = carrNco;
        rstS = rst;
      }
    } else if (tid == 64) {  // ---- T6 carry, computed at the start of the period
      set_carr_phase(prm, remNextS);
    }
    if (stamp) ts[4] = clock64();
    __syncthreads();
    if (stamp) {
      ts[5] = clock64();
      long long* pr = a.prof + ((long long)cid * NWARPS + (tid >> 5)) * TRK_PROF_N;
#pragma unroll
      for (int i = 0; i < TRK_PROF_N; ++i) pr[i] += ts[i + 1] - ts[i];
    }
  }
  if (BULK) {  // never exit with a bulk copy in flight
    if (pending0) mbar_wait(&mbar[0], phase0);
    if (pending1) mbar_wait(&mbar[1], phase1);
  } else {
    cp_async_wait_all();
  }
  if (tid == 0) {
    const int status = (k == a.ms) ? SGX_OK : prm.stop;
    a.ms_done[cid] = k;
    a.status[cid] = status;
    if (a.state) { a.state[cid].c = cstS; a.state[cid].k = k; a.state[cid].status = status; }
  }
  if (tid == 32 && a.state) {
    CarrState r = rstS;
    r.remCarrPhase = prm.rem_rad;
    a.state[cid].r = r;
  }
}

// --------------------------------------------------------------------------- host entry
struct TrackScratch {
  DevBuf rec, len, ch, chips, out, done, status, state, prof;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  // file ingest: two pinned staging buffers, filled by pread() while the other one is on its way to the device
  int8_t* pin[2] = {nullptr, nullptr};
  size_t pin_cap = 0;
  cudaEvent_t pin_ev[2] = {nullptr, nullptr};
};

// A recording that lives in a file (sgx_track_file): samples [base, base + len) are what tracking can touch.
struct FileSrc {
  int fd;
  int sample_bytes;      // 1: int8 (the reference's format), 2: int16 little endian, values must fit int8
  long long base;        // first sample of the window, multiple of 16
  long long len;         // samples in the window
  long long chunk;       // samples per staging buffer
  int bad_value;         // set when an int16 sample does not fit int8
};
static TrackScratch g_trk;

static bool use_bulk() {
  const char* e = getenv("SGX_TRK_STAGE");
  return !(e && strcmp(e, "cpasync") == 0);
}

}  // namespace sgx

using namespace sgx;

static int track_core(const int8_t* rec, int64_t rec_stride, const int64_t* rec_len,
                      int32_t n_recordings, const sgx_channel* ch, int32_t n_channels,
                      const sgx_settings* st, const int8_t* ca_chips, double* out,
                      int32_t* ms_done, void* cuda_stream, sgx::FileSrc* file) {
  if ((!rec && !file) || !rec_len || !ch || !st || !ca_chips || !out || !ms_done || n_recordings <= 0 ||
      n_channels <= 0 || st->msToProcess <= 0)
    return fail(SGX_ERR_ARG, "sgx_track", "null pointer or empty problem");
  const int nch = n_recordings * n_channels;
  for (int i = 0; i < nch; ++i)
    if (ch[i].prn < 0 || ch[i].prn > SGX_NUM_PRN) return fail(SGX_ERR_ARG, "sgx_track", "PRN outside 0..32");
  cudaStream_t s = (cudaStream_t)cuda_stream;
  const int ms = st->msToProcess;
  const int win = ((st->samplesPerCode + TRK_MARGIN + 15) & ~15) + 16;

  const int8_t* d_rec = rec;
  long long stride = rec_stride;
  long long max_len = 0;
  for (int r = 0; r < n_recordings; ++r) max_len = rec_len[r] > max_len ? rec_len[r] : max_len;
  const bool host_input = file || !is_device_ptr(rec);
  if (host_input) {  // host recording: it is streamed into HBM in chunks while tracking runs (np.fromfile replacement)
    stride = (max_len + 15) & ~15LL;
    if (g_trk.rec.reserve((size_t)stride * n_recordings + 16)) return fail(SGX_ERR_CUDA, "cudaMalloc", "recording");
    d_rec = g_trk.rec.as<int8_t>();
  } else if (((rec_stride & 15) && n_recordings > 1) || ((uintptr_t)rec & 15)) {   // (one recording: the stride is not used)
    return fail(SGX_ERR_ARG, "sgx_track", "device recordings must be 16-byte aligned with a stride multiple of 16");
  }
  if (g_trk.len.reserve(sizeof(long long) * n_recordings) || g_trk.ch.reserve(sizeof(sgx_channel) * nch) ||
      g_trk.chips.reserve(32 * 1023) || g_trk.done.reserve(sizeof(int) * nch) ||
      g_trk.status.reserve(sizeof(int) * nch) || g_trk.state.reserve(sizeof(TrackState) * nch))
    return fail(SGX_ERR_CUDA, "cudaMalloc", "tracking scratch");
  SGX_CUDA(cudaMemcpyAsync(g_trk.len.p, rec_len, sizeof(long long) * n_recordings, cudaMemcpyHostToDevice, s));
  SGX_CUDA(cudaMemcpyAsync(g_trk.ch.p, ch, sizeof(sgx_channel) * nch, cudaMemcpyHostToDevice, s));
  SGX_CUDA(cudaMemcpyAsync(g_trk.chips.p, ca_chips, 32 * 1023, cudaMemcpyHostToDevice, s));
  const size_t out_bytes = sizeof(double) * (size_t)nch * SGX_TRACK_FIELDS * ms;
  double* d_out = out;
  const bool out_on_host = !is_device_ptr(out);
  if (out_on_host) {
    if (g_trk.out.reserve(out_bytes)) return fail(SGX_ERR_CUDA, "cudaMalloc", "tracking output");
    d_out = g_trk.out.as<double>();
  }

  TrackArgs a;
  a.rec = d_rec;
  a.rec_stride = stride;
  a.rec_len = g_trk.len.as<long long>();
  a.ch = g_trk.ch.as<sgx_channel>();
  a.chips = g_trk.chips.as<int8_t>();
  a.out = d_out;
  a.ms_done = g_trk.done.as<int>();
  a.status = g_trk.status.as<int>();
  a.n_channels = n_channels;
  a.ms = ms;
  a.resume = 0;
  a.avail = 0x7fffffffffffffffLL;
  a.state = g_trk.state.as<TrackState>();
  a.prof = nullptr;
  const size_t prof_n = (size_t)nch * TRK_WARPS * TRK_PROF_N;
  if (getenv("SGX_TRK_PROF")) {
    if (g_trk.prof.reserve(sizeof(long long) * prof_n)) return fail(SGX_ERR_CUDA, "cudaMalloc", "prof");
    SGX_CUDA(cudaMemsetAsync(g_trk.prof.p, 0, sizeof(long long) * prof_n, s));
    a.prof = g_trk.prof.as<long long>();
  }
  a.win = win;
  a.skip = file ? st->skipNumberOfBytes / file->sample_bytes - file->base : st->skipNumberOfBytes;
  a.abs_base = file ? file->base : 0;
  a.fs = st->samplingFreq;
  a.codeFreqBasis = st->codeFreqBasis;
  a.codeLength = (double)st->codeLength;
  a.spc = st->dllCorrelatorSpacing;
  a.c1code = st->tau2code / st->tau1code;
  a.c2code = st->PDIcode / st->tau1code;
  a.c1carr = st->tau2carr / st->tau1carr;
  a.c2carr = st->PDIcarr / st->tau1carr;

  const size_t smem = 2 * (size_t)win;
  auto launch = [&]() -> int {
  // correlate variant: half-chip segments when a segment fits the unrolled path, else aligned groups
  const double half_chip = st->samplingFreq / (2.0 * st->codeFreqBasis);   // samples per half chip
  int nw = ((int)ceil(half_chip + 0.25) + 3) / 4;
  bool exact = true;   // exact integer segment sums by default; "segments" = float32 variant, "groups" = any spacing
  if (const char* e = getenv("SGX_TRK_KERNEL")) {
    if (strcmp(e, "groups") == 0) nw = 0;
    if (strcmp(e, "segments") == 0) exact = false;
  }
  if (fabs(st->dllCorrelatorSpacing - 0.5) > 1e-12) nw = 0;                 // segment scheme assumes E/L at +-0.5 chip
  const bool bulk = use_bulk();
#define SGX_TRK_GO_NT(B, W, X, NTHR)                                                               \
  {                                                                                                \
    auto kfn = track_kernel<B, W, X, NTHR>;                                                        \
    SGX_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));   \
    SGX_COUNTED_LAUNCH(kfn, dim3(nch), dim3(NTHR), smem, s, a);                                    \
  }
#define SGX_TRK_GO(B, W, X) SGX_TRK_GO_NT(B, W, X, TRK_THREADS)
#define SGX_TRK_EXACT(W) { if (bulk) SGX_TRK_GO(true, W, true) else SGX_TRK_GO(false, W, true) }
  if (nw >= 1 && nw <= 8 && exact) {
    switch (nw) {
      case 1: SGX_TRK_EXACT(1) break;
      case 2: SGX_TRK_EXACT(2) break;
      case 3: SGX_TRK_EXACT(3) break;
      case 4: SGX_TRK_EXACT(4) break;
      case 5: SGX_TRK_EXACT(5) break;
      case 6: SGX_TRK_EXACT(6) break;
      case 7: SGX_TRK_EXACT(7) break;
      default: SGX_TRK_EXACT(8) break;
    }
  } else if (nw == 5) {
    if (bulk) SGX_TRK_GO(true, 5, false) else SGX_TRK_GO(false, 5, false)     // float32 segment variant (comparison)
  } else {
    if (bulk) SGX_TRK_GO(true, 0, false) else SGX_TRK_GO(false, 0, false)     // aligned groups: any rate / spacing
  }
#undef SGX_TRK_EXACT
#undef SGX_TRK_GO
#undef SGX_TRK_GO_NT
    return SGX_OK;
  };
  if (!host_input) {
    int rc0 = launch();
    if (rc0) return rc0;
  } else {
    // Streamed ingest: chunk c of every recording is copied on a second stream while the kernel works on
    // the periods whose samples are already resident; channels pause at the end of the resident data and
    // are resumed by the next launch (TrackState).  With pageable host memory the copies simply serialise.
    if (!g_trk.copy_stream) {
      SGX_CUDA(cudaStreamCreateWithFlags(&g_trk.copy_stream, cudaStreamNonBlocking));
      SGX_CUDA(cudaEventCreateWithFlags(&g_trk.ev[0], cudaEventDisableTiming));
      SGX_CUDA(cudaEventCreateWithFlags(&g_trk.ev[1], cudaEventDisableTiming));
    }
    long long chunk = 1024LL * st->samplesPerCode;
    if (const char* e = getenv("SGX_TRK_CHUNK_MS")) { if (atoll(e) > 0) chunk = atoll(e) * st->samplesPerCode; }
    chunk = (chunk + 15) & ~15LL;
    SGX_CUDA(cudaEventRecord(g_trk.ev[1], s));                     // the copy stream starts after earlier work on s
    SGX_CUDA(cudaStreamWaitEvent(g_trk.copy_stream, g_trk.ev[1], 0));
    int c = 0;
    if (file) chunk = file->chunk;
    for (long long off = 0; off < max_len; off += chunk, ++c) {
      const long long width = (max_len - off) < chunk ? (max_len - off) : chunk;
      if (file) {
        // pread into the pinned buffer that is free (its previous copy has completed), convert if needed, copy
        int8_t* hb = g_trk.pin[c & 1];
        if (c >= 2) SGX_CUDA(cudaEventSynchronize(g_trk.pin_ev[c & 1]));
        const size_t bytes = (size_t)width * file->sample_bytes;
        size_t got = 0;
        while (got < bytes) {
          const ssize_t r = pread(file->fd, (char*)hb + got, bytes - got, (off_t)((file->base + off) * file->sample_bytes + (long long)got));
          if (r <= 0) return fail(SGX_ERR_ARG, "sgx_track_file", "short read from the recording file");
          got += (size_t)r;
        }
        if (file->sample_bytes == 2) {   // in place, front to back: sample i lands in byte i
          const int16_t* src = (const int16_t*)hb;
          for (long long i = 0; i < width; ++i) {
            const int v = src[i];
            if (v < -128 || v > 127) file->bad_value = 1;
            hb[i] = (int8_t)v;
          }
          if (file->bad_value) return fail(SGX_ERR_ARG, "sgx_track_file", "int16 sample outside the int8 range of the correlators");
        }
        SGX_CUDA(cudaMemcpyAsync(g_trk.rec.as<int8_t>() + off, hb, (size_t)width, cudaMemcpyHostToDevice, g_trk.copy_stream));
        SGX_CUDA(cudaEventRecord(g_trk.pin_ev[c & 1], g_trk.copy_stream));
      } else
      SGX_CUDA(cudaMemcpy2DAsync(g_trk.rec.as<int8_t>() + off, (size_t)stride, rec + off, (size_t)rec_stride, (size_t)width,
                                 (size_t)n_recordings, cudaMemcpyHostToDevice, g_trk.copy_stream));
      SGX_CUDA(cudaEventRecord(g_trk.ev[0], g_trk.copy_stream));
      SGX_CUDA(cudaStreamWaitEvent(s, g_trk.ev[0], 0));
      a.avail = off + width;
      a.resume = c > 0;
      int rc0 = launch();
      if (rc0) return rc0;
    }
  }
  SGX_CUDA(cudaGetLastError());
  if (out_on_host) SGX_CUDA(cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, s));
  std::vector<int> h_status_v(nch);   // RAII: the checks below return early on errors
  int* h_status = h_status_v.data();
  SGX_CUDA(cudaMemcpyAsync(ms_done, a.ms_done, sizeof(int) * nch, cudaMemcpyDeviceToHost, s));
  SGX_CUDA(cudaMemcpyAsync(h_status, a.status, sizeof(int) * nch, cudaMemcpyDeviceToHost, s));
  SGX_CUDA(cudaStreamSynchronize(s));
  if (a.prof) {   // mean cycles per period of every warp over all channels and periods of the last launch
    std::vector<long long> hp(prof_n);
    cudaMemcpy(hp.data(), a.prof, sizeof(long long) * prof_n, cudaMemcpyDeviceToHost);
    const double per = (double)nch * ms;
    fprintf(stderr, "[sgx prof] cycles/period  warp:  wait+prefetch  correlate  reduce+bar  bookkeeping  bar  | period\n");
    for (int w = 0; w < TRK_WARPS; ++w) {
      double acc[TRK_PROF_N] = {}, tot = 0.0;
      for (int i = 0; i < nch; ++i)
        for (int j = 0; j < TRK_PROF_N; ++j) acc[j] += (double)hp[((size_t)i * TRK_WARPS + w) * TRK_PROF_N + j];
      for (int j = 0; j < TRK_PROF_N; ++j) tot += acc[j];
      fprintf(stderr, "[sgx prof] %d: %8.0f %8.0f %8.0f %8.0f %8.0f | %8.0f\n", w, acc[0] / per, acc[1] / per, acc[2] / per,
              acc[3] / per, acc[4] / per, tot / per);
    }
  }
  int rc = SGX_OK;
  for (int i = 0; i < nch; ++i)
    if (h_status[i] != SGX_OK && rc == SGX_OK) rc = h_status[i];
  if (rc == SGX_ERR_SHORT) return fail(rc, "sgx_track", "Not able to read the specified number of samples for tracking");
  if (rc != SGX_OK) return fail(rc, "sgx_track", "loop state left the supported range");
  return SGX_OK;
}

extern "C" int sgx_track(const int8_t* rec, int64_t rec_stride, const int64_t* rec_len,
                         int32_t n_recordings, const sgx_channel* ch, int32_t n_channels,
                         const sgx_settings* st, const int8_t* ca_chips, double* out,
                         int32_t* ms_done, void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_track", "no CUDA device");
  SGX_API_GUARD();
  return track_core(rec, rec_stride, rec_len, n_recordings, ch, n_channels, st, ca_chips, out, ms_done, cuda_stream,
                    nullptr);
}

// File ingest (SURVEY.md section 8(f) row 2; replaces fid.seek / np.fromfile of tracking.py:107, :154 and the
// dataType / skipNumberOfBytes handling of initialize.py:102, :466-481): the recording is read with pread() in chunks
// into two pinned staging buffers and copied to HBM on the copy stream while the kernel tracks the periods that are
// already resident.  Only the window tracking can touch is read: from the first sample any channel starts at to
// msToProcess code periods (+ margin) after the last one -- never the whole file, never a pageable copy.
extern "C" int sgx_track_file(const char* path, int32_t sample_bytes, const sgx_channel* ch, int32_t n_channels,
                              const sgx_settings* st, const int8_t* ca_chips, double* out, int32_t* ms_done,
                              int64_t chunk_samples, int64_t* window /* [2]: first sample, samples read; may be NULL */,
                              void* cuda_stream) {
  if (sgx_device_count() <= 0) return fail(SGX_ERR_NODEV, "sgx_track_file", "no CUDA device");
  SGX_API_GUARD();
  if (!path || !ch || !st || n_channels <= 0 || (sample_bytes != 1 && sample_bytes != 2))
    return fail(SGX_ERR_ARG, "sgx_track_file", "null pointer, or dataType other than int8 / int16");
  const int fd = open(path, O_RDONLY);
  if (fd < 0) return fail(SGX_ERR_ARG, "sgx_track_file", "cannot open the recording file");
  struct stat sb;
  if (fstat(fd, &sb) != 0) { close(fd); return fail(SGX_ERR_ARG, "sgx_track_file", "cannot stat the recording file"); }
  const long long file_samples = (long long)sb.st_size / sample_bytes;
  double cp_min = 1e300, cp_max = -1e300;
  for (int i = 0; i < n_channels; ++i)
    if (ch[i].prn > 0) { cp_min = ch[i].codePhase < cp_min ? ch[i].codePhase : cp_min; cp_max = ch[i].codePhase > cp_max ? ch[i].codePhase : cp_max; }
  if (cp_max < cp_min) { cp_min = cp_max = 0.0; }
  const long long skip = st->skipNumberOfBytes / sample_bytes;
  FileSrc fs;
  fs.fd = fd;
  fs.sample_bytes = sample_bytes;
  fs.bad_value = 0;
  fs.base = (skip + (long long)cp_min) & ~15LL;
  // msToProcess code periods per channel; the period length follows the code Doppler (<= 1e-5 relative): 1e-4 + 2 periods
  const double need = (double)(skip + (long long)cp_max - fs.base) + ((double)st->msToProcess * (1.0 + 1e-4) + 2.0) * st->samplesPerCode + 64.0;
  fs.len = file_samples - fs.base;
  if (fs.len > (long long)need) fs.len = (long long)need;
  if (fs.len <= 0) { close(fd); return fail(SGX_ERR_SHORT, "sgx_track_file", "Not able to read the specified number of samples for tracking"); }
  fs.chunk = chunk_samples > 0 ? chunk_samples : 1024LL * st->samplesPerCode;
  fs.chunk = (fs.chunk + 15) & ~15LL;
  const size_t pin_bytes = (size_t)fs.chunk * sample_bytes;
  if (g_trk.pin_cap < pin_bytes) {
    for (int i = 0; i < 2; ++i) {
      if (g_trk.pin[i]) cudaFreeHost(g_trk.pin[i]);
      g_trk.pin[i] = nullptr;
      if (cudaHostAlloc((void**)&g_trk.pin[i], pin_bytes, cudaHostAllocDefault) != cudaSuccess) {
        g_trk.pin_cap = 0;
        close(fd);
        return fail(SGX_ERR_CUDA, "cudaHostAlloc", "pinned staging buffers");
      }
      if (!g_trk.pin_ev[i]) cudaEventCreateWithFlags(&g_trk.pin_ev[i], cudaEventDisableTiming);
    }
    g_trk.pin_cap = pin_bytes;
  }
  if (window) { window[0] = fs.base; window[1] = fs.len; }
  const int64_t rec_len = fs.len;
  const int rc = track_core(nullptr, 0, &rec_len, 1, ch, n_channels, st, ca_chips, out, ms_done, cuda_stream, &fs);
  close(fd);
  return rc;
}
