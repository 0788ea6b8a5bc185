/* softgnss_b200.h -- C ABI of the B200-native acquisition / tracking hot paths.
 *
 * The reference (perrysou/SoftGNSS-python) is pure Python + numpy and has no FFI of its
 * own; its stage boundary is the pair of methods
 *     AcquisitionResult.acquire(longSignal)      reference acquisition.py:27-204
 *     TrackingResult.track(fid)                  reference tracking.py:13-295
 * and the recarrays they exchange.  These entry points are what a ctypes binding placed
 * inside those two methods calls instead of the numpy loops (see INTEGRATION.md for the
 * stub).  Plain pointers and sizes only; every data pointer may be a host pointer or a CUDA
 * device pointer (detected with cudaPointerGetAttributes) unless stated otherwise; the caller
 * owns all buffers.  Return value: 0 or a negative sgx_status; sgx_last_error() gives text.
 * There is no CPU fallback: without a CUDA device every compute call fails with
 * SGX_ERR_NODEV.
 *
 * Operands of the stages after tracking (sgx_find_preambles, sgx_pseudoranges, sgx_track_quality,
 * sgx_nav_solve, sgx_nav_velocity):
 *   - device operands are read and written in place, in the order of cuda_stream;
 *   - host inputs are copied to device scratch first.  An input that holds one series of ms values per
 *     channel, `stride` elements apart, is read in exactly those rows: nothing between or after them;
 *   - host outputs are written from device scratch, and then the call synchronises the stream before it
 *     returns.  A call whose outputs are all device memory (NULL optional outputs do not count) does not
 *     synchronise: its results are complete in stream order.
 */
#ifndef SOFTGNSS_B200_H
#define SOFTGNSS_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SGX_ABI_VERSION 1
#define SGX_NUM_PRN 32
#define SGX_CODE_LEN 1023
#define SGX_TRACK_FIELDS 13 /* order: absoluteSample codeFreq carrFreq I_P I_E I_L Q_E Q_P Q_L
                               dllDiscr dllDiscrFilt pllDiscr pllDiscrFilt (tracking.py:286-293) */
#define SGX_SYNTH_MAX_SATS 12

typedef enum sgx_status {
  SGX_OK = 0,
  SGX_ERR_CUDA = -1,   /* a CUDA runtime call failed                                        */
  SGX_ERR_ARG = -2,    /* bad argument (PRN outside 1..32, sizes, alignment)                 */
  SGX_ERR_SHORT = -3,  /* recording too short: tracking.py:159-163 "Not able to read ..."   */
  SGX_ERR_NODEV = -4,  /* no CUDA device                                                     */
  SGX_ERR_RANGE = -5   /* loop state left the supported range (block size vs staged window)  */
} sgx_status;

/* Receiver settings, marshalled from the reference's Settings object (initialize.py:80-173).
 * Derived integers are computed by the host with the reference's float64 expressions. */
typedef struct sgx_settings {
  double samplingFreq;         /* initialize.py:107 */
  double IF;                   /* initialize.py:105 */
  double codeFreqBasis;        /* initialize.py:109 */
  double acqSearchBand;        /* kHz, initialize.py:123 */
  double acqThreshold;         /* initialize.py:126 */
  double acqDopplerStep;       /* Hz; 500.0 = the literal at acquisition.py:101 */
  double dllCorrelatorSpacing; /* chips, initialize.py:134 */
  double tau1code, tau2code;   /* calcLoopCoef(dllNoiseBandwidth, dllDampingRatio, 1.0), tracking.py:45 */
  double tau1carr, tau2carr;   /* calcLoopCoef(pllNoiseBandwidth, pllDampingRatio, 0.25), tracking.py:52 */
  double PDIcode, PDIcarr;     /* 0.001, tracking.py:42,49 */
  int64_t skipNumberOfBytes;   /* initialize.py:94 */
  int32_t codeLength;          /* 1023 */
  int32_t samplesPerCode;      /* initialize.py:183-185 */
  int32_t numAcqSatellites;    /* len(acqSatelliteList): PRN 1..n are searched (acquisition.py:92) */
  int32_t numFrqBins;          /* acquisition.py:68 */
  int32_t acqCoherentMs;       /* 1 in the reference */
  int32_t acqNonCoherentBlocks;/* 2 in the reference (pick-max of two blocks, acquisition.py:129-133) */
  int32_t samplesPerCodeChip;  /* round(fs/codeFreqBasis), acquisition.py:145 */
  int32_t fineMs;              /* 10, acquisition.py:172-177 */
  int32_t msToProcess;         /* initialize.py:85 */
  int32_t numberOfChannels;    /* initialize.py:88 */
} sgx_settings;

/* One tracking channel as produced by preRun (acquisition.py:278-304). prn == 0: idle. */
typedef struct sgx_channel {
  int32_t prn;
  int32_t reserved;
  double acquiredFreq;
  double codePhase;
} sgx_channel;

/* Integer parameter block of the synthetic recording generator (softgnss_python_b200/synth.py). */
typedef struct sgx_synth_spec {
  uint64_t seed;
  int32_t n_sats;
  int32_t noise_k;
  int32_t n_bits;
  int32_t reserved;
  int32_t prn[SGX_SYNTH_MAX_SATS];
  int32_t amp[SGX_SYNTH_MAX_SATS];
  int32_t per0[SGX_SYNTH_MAX_SATS];
  uint64_t phi0[SGX_SYNTH_MAX_SATS];
  uint64_t dphi[SGX_SYNTH_MAX_SATS];
  uint64_t cp0[SGX_SYNTH_MAX_SATS];
  uint64_t dcp[SGX_SYNTH_MAX_SATS];
} sgx_synth_spec;

int sgx_abi_version(void);
const char* sgx_last_error(void);
/* Number of CUDA devices (0 if none / driver missing). */
int sgx_device_count(void);
/* Selects the device of this process.  The library keeps its plan caches and scratch buffers process-wide on ONE
 * device (one process per GPU, as torch.distributed launches them): once a compute entry point has run, selecting a
 * different device -- or calling a compute entry point while another device is current -- returns SGX_ERR_ARG.
 * Compute entry points are serialised by a process-wide mutex (safe, not concurrent, from several host threads). */
int sgx_set_device(int device);
/* Measured FP32 FMA throughput of the current device (FFMA burn, 16 independent chains per thread), TFLOP/s: the
 * denominator of the acquisition roofline in bench.py (SURVEY.md section 8(d): "must measure an FMA-burn peak"). */
int sgx_fp32_peak(double* tflops, void* cuda_stream);
/* Kernels launched by this library in this process since load (bench.py's gpu_launches). */
int64_t sgx_kernel_launch_count(void);

/* Replaces the body of AcquisitionResult.acquire (acquisition.py:49-204) for `n_recordings`
 * independent recordings and the PRN shard [prn_first, prn_first+prn_count) (0-based).
 *   sig        int8 [n_recordings][rec_stride]; each needs >= (blocks*coh + fineMs... ) i.e. 11 ms
 *   n_samples  valid samples per recording (the reference passes 11*samplesPerCode)
 *   ca_table   host int8 [32][samplesPerCode]   = makeCaTable()            (initialize.py:188-231)
 *   ca_chips   host int8 [32][1023]             = generateCAcode(prn)      (initialize.py:234-302)
 *   fine_idx   host uint16 [fineMs*samplesPerCode] chip index of acquisition.py:172-174
 * Outputs (host, [n_recordings][prn_count]): carrFreq/codePhase (0 when not detected),
 * peakMetric (always), and optional diagnostics (may be NULL): frqBin, finePeakIndex.
 */
int sgx_acquire(const int8_t* sig, int64_t rec_stride, int64_t n_samples, int32_t n_recordings,
                const sgx_settings* st, const int8_t* ca_table, const int8_t* ca_chips,
                const uint16_t* fine_idx, int32_t prn_first, int32_t prn_count,
                double* carrFreq, double* codePhase, double* peakMetric,
                int32_t* frqBin, int32_t* finePeakIndex, void* cuda_stream);

/* Replaces the channel/ms loops of TrackingResult.track (tracking.py:59-283) for
 * n_recordings x n_channels independent channels.
 *   rec      int8 [n_recordings][rec_stride], rec_stride % 16 == 0 and the buffer readable up to
 *            the next multiple of 16 past rec_len[r]
 *   rec_len  host int64 [n_recordings] valid bytes (the file size)
 *   ch       host [n_recordings][n_channels]
 *   out      double [n_recordings][n_channels][SGX_TRACK_FIELDS][ms] (host or device)
 *   ms_done  host int32 [n_recordings][n_channels] code periods completed
 * Returns SGX_ERR_SHORT if any active channel ran out of samples (results then cover ms_done).
 */
int sgx_track(const int8_t* rec, int64_t rec_stride, const int64_t* rec_len, int32_t n_recordings,
              const sgx_channel* ch, int32_t n_channels, const sgx_settings* st,
              const int8_t* ca_chips, double* out, int32_t* ms_done, void* cuda_stream);

/* The same for ONE recording that lives in a file: replaces fid.seek / np.fromfile(fid, dataType, blksize) of
 * tracking.py:107, :154 and the dataType / skipNumberOfBytes handling of initialize.py:102, :466-481 (SURVEY.md
 * section 8(f) row 2).  The file is read with pread() in chunks of `chunk_samples` (0: 1024 code periods) into two
 * pinned staging buffers and copied to HBM while the kernel tracks the periods already resident; only the window
 * tracking can touch is read (first sample of the earliest channel ... msToProcess code periods after the latest),
 * reported in window[0..1] when non-NULL.
 *   sample_bytes  1: int8 (the reference's format), 2: little-endian int16 whose values fit int8 (SGX_ERR_ARG
 *                 otherwise).  For int16 positions count SAMPLES: the start is skipNumberOfBytes/2 + codePhase and
 *                 absoluteSample is a sample index (the reference mixes bytes and samples for multi-byte types).
 * Results as sgx_track with n_recordings = 1; a file that ends early gives SGX_ERR_SHORT. */
int sgx_track_file(const char* path, int32_t sample_bytes, const sgx_channel* ch, int32_t n_channels,
                   const sgx_settings* st, const int8_t* ca_chips, double* out, int32_t* ms_done,
                   int64_t chunk_samples, int64_t* window, void* cuda_stream);

/* Synthetic int8 IF recordings, bit-identical to synth.generate_cpu.
 *   out   int8 [n_recordings][rec_stride] (host or device), samples start .. start+n_samples-1
 *   bits  host int8 [n_recordings][SGX_SYNTH_MAX_SATS][n_bits] nav bits (+-1)
 *   lut   host int16 [4096] cosine table, ca_chips host int8 [32][1023]
 */
int sgx_synth_generate(int8_t* out, int64_t rec_stride, int64_t n_samples, int64_t start,
                       int32_t n_recordings, const sgx_synth_spec* specs, const int8_t* bits,
                       const int16_t* lut, const int8_t* ca_chips, void* cuda_stream);

/* Test hook: unnormalised complex FFT (inverse bit 0: conjugate twiddles; bit 1: passes after the first run through
 * the persistent pass kernels, as in sgx_acquire) of `batch` rows of length n
 * through the acquisition path's FFT engine; host pointers, interleaved float32 re/im.  n must factor
 * over {2,3,5,7,11,31}.  The counterpart of np.fft.fft / n*np.fft.ifft at acquisition.py:95-126,182. */
int sgx_fft_c2c(const float* in, float* out, int32_t n, int32_t batch, int32_t inverse, void* cuda_stream);

#define SGX_NAV_BITS 1501

/* Replaces NavigationResult.findPreambles (postNavigation.py:524-631) and the 20 ms bit summation of
 * postNavigate (postNavigation.py:125-134) for n_channels tracked channels (the downstream consumer of
 * the tracking result; SURVEY.md section 8(f) row 3).
 *   i_p             double [n_channels][stride] prompt in-phase series (e.g. field 3 of sgx_track's
 *                   output with stride = SGX_TRACK_FIELDS * ms), ms values used per row
 *   first_subframe  int32 [n_channels]: ms index of the first preamble that has a
 *                   preamble-like pattern 6000 ms later and whose TLM and HOW words pass the parity
 *                   check; 0 when there is none (the reference's convention)
 *   nav_bits        optional uint8 [n_channels][SGX_NAV_BITS]: hard bits 0/1 of
 *                   I_P[first-20 : first+30000] summed over 20 ms (bit 0 = last bit of the previous
 *                   subframe), what the caller hands to ephemeris()
 *   nav_bits_valid  optional int32 [n_channels]: 1 when that window lies inside the record; written only
 *                   when nav_bits is given
 * Candidates nearer than 40 ms to the start of the record are passed over (the reference reads
 * I_P[k-40:...] with a negative start there and raises). */
int sgx_find_preambles(const double* i_p, int64_t stride, int32_t n_channels, int32_t ms,
                       int32_t* first_subframe, uint8_t* nav_bits, int32_t* nav_bits_valid,
                       void* cuda_stream);

/* Replaces NavigationResult.calculatePseudoranges (postNavigation.py:27-72), batched over recordings and
 * measurement epochs (SURVEY.md section 8(f) row 4, first half; satellite positions and the least-squares
 * fix stay with the reference's host code).
 *   track_out     double [n_recordings][n_channels][SGX_TRACK_FIELDS][ms] as written by sgx_track; only
 *                 field 0 (absoluteSample) is read
 *   ms_index      int32 [n_recordings][n_epochs][n_channels]: msOfTheSignal per channel
 *   active        uint8 [n_recordings][n_epochs][n_channels]: 1 = channel is in channelList (others get +inf
 *                 travel time, i.e. an infinite pseudorange, as in the reference)
 *   pseudoranges  double [n_recordings][n_epochs][n_channels], metres:
 *                 (absoluteSample[ms_index]/samples_per_code - floor(min over the list) + start_offset) * c / 1000
 * n_channels <= 32.  Bit-identical to the reference (same float64 operations in the same order). */
int sgx_pseudoranges(const double* track_out, int32_t n_recordings, int32_t n_channels, int32_t ms,
                     const int32_t* ms_index, const uint8_t* active, int32_t n_epochs,
                     double samples_per_code, double start_offset, double c, double* pseudoranges,
                     void* cuda_stream);

/* ---- tracking quality: C/N0 and carrier lock per window (extension; no reference behaviour) ---------------- */
/* Settings of sgx_track_quality.  The Matlab SoftGNSS line computes the same estimator in CNoVSM.m with
 * settings.CNo.VSMinterval = 40 and settings.CNo.accTime = 0.001. */
typedef struct sgx_quality_settings {
  double acc_time;      /* s per I/Q sample: 0.001 */
  double cn0_min;       /* dB-Hz: a window is locked only if cn0 >= cn0_min */
  double pll_lock_min;  /* cos 2dphi: ... and pll_lock >= pll_lock_min */
  int32_t window_ms;    /* W >= 2 code periods per estimate */
  int32_t reserved;
} sgx_quality_settings;

/* Variance-summing-method C/N0 and the narrow-band carrier-lock indicator of n_channels tracked channels, one value
 * per window of W = window_ms code periods, n_win = ms / W (windows w = 0 .. n_win-1 hold periods w*W .. w*W+W-1).
 * With I_k, Q_k the prompt samples of the window and all arithmetic in float64:
 *   Z_k = I_k^2 + Q_k^2,  Zm = mean(Z),  Zv = sum((Z_k - Zm)^2) / (W - 1)
 *   Pav = sqrt(Zm^2 - Zv),  Nv = 0.5 * (Zm - Pav),  cn0 = 10 * log10(Pav / (2 * Nv * acc_time))   [dB-Hz]
 *   pll_lock = sum(I_k^2 - Q_k^2) / sum(I_k^2 + Q_k^2)        (cos 2dphi; independent of the nav-bit signs)
 *   locked = cn0 >= cn0_min && pll_lock >= pll_lock_min       (NaN compares false)
 * cn0 is NaN unless Zm^2 - Zv > 0 and Nv > 0 (CNoVSM.m instead takes abs() of the complex value it gets there);
 * pll_lock is NaN when its denominator is 0.  A window is valid iff (w+1)*W <= ms_done[c]; invalid windows get NaN,
 * NaN, 0 (idle channels of sgx_track have ms_done = 0).  Deterministic: fixed reduction order, no atomics.
 *   i_p, q_p  double [n_channels][stride], ms values used per row; both host or both device memory.  Reads
 *             sgx_track's output in place: i_p = out + 3*ms, q_p = out + 7*ms, stride = SGX_TRACK_FIELDS*ms,
 *             n_channels = n_recordings * channels.
 *   ms_done   host int32 [n_channels] periods completed per channel, each in [0, ms]; NULL: all ms
 *   cn0, pll_lock (double), locked (uint8)  [n_channels][n_win], all three host or all three device memory.
 * SGX_ERR_ARG for window_ms < 2, acc_time not finite and > 0, stride < ms, ms_done outside [0, ms], a NULL pointer
 * or mixed host/device operands.  n_win == 0 succeeds without work. */
int sgx_track_quality(const double* i_p, const double* q_p, int64_t stride, int32_t n_channels, int32_t ms,
                      const int32_t* ms_done, const sgx_quality_settings* qs, double* cn0, double* pll_lock,
                      uint8_t* locked, void* cuda_stream);

/* ---- navigation solution (SURVEY.md section 8(f) row 4, second half) -------------------------------------- */
/* Broadcast-ephemeris terms read by geoFunctions.satpos (geoFunctions/__init__.py:779-885), one per channel,
 * in the units ephemeris.py decodes them to (seconds, radians, metres). */
typedef struct sgx_eph {
  double t_oc, a_f2, a_f1, a_f0, T_GD;
  double sqrtA, t_oe, deltan, M_0, e, omega;
  double C_uc, C_us, C_rc, C_rs;
  double i_0, iDot, C_ic, C_is, omega_0, omegaDot;
} sgx_eph;

/* Settings read by the measurement loop: settings.samplesPerCode, .startOffset, .c, .navSolPeriod,
 * .elevationMask, .useTropCorr (initialize.py:144-181). */
typedef struct sgx_nav_settings {
  double samples_per_code, start_offset, c, nav_sol_period, elevation_mask;
  int32_t use_trop_corr, reserved;
} sgx_nav_settings;

#define SGX_NAV_SOL_FIELDS 12   /* X Y Z dt GDOP PDOP HDOP VDOP TDOP latitude longitude height */

/* Replaces the measurement loop of NavigationResult.postNavigate (postNavigation.py:159-301) with the
 * functions it calls -- calculatePseudoranges (:27-72), geoFunctions.satpos (geoFunctions/__init__.py:779-885),
 * leastSquarePos (:636-739; e_r_corr :491, topocent :1003, togeod :892, tropo :1071) and cart2geo (:7-77) --
 * batched over independent recordings (one warp per recording, lane = channel; epochs are sequential because
 * the elevation mask of an epoch uses the elevations of the epoch before, :201/:241).  UTM conversion
 * (findUtmZone, cart2utm) and ephemeris decoding stay with the caller.
 *   abs_sample       double: the absoluteSample series of channel (r, c) starts at abs_sample + (r*n_channels + c)*stride
 *                    and holds ms values (sgx_track's output: pointer to its first element, stride = SGX_TRACK_FIELDS*ms)
 *   sub_frame_start  int32 [R][C]   subFrameStart of findPreambles (0: none)
 *   ready            uint8 [R][C]   1 = channel is in readyChnList (preamble found and ephemeris decoded, :166)
 *   eph              sgx_eph [R][C] ephemeris of the channel's PRN (read for ready channels only)
 *   tow              double [R]     transmitTime of the first measurement (:168)
 *   n_epochs         int32 [R]      int(fix(msToProcess - max(subFrameStart)) / navSolPeriod) (:199); epochs beyond
 *                                   it keep the reference's initial values (NaN, DOP 0)
 * Outputs (the same kind as `sol`), E = max_epochs:
 *   raw_p, corrected_p, el, az  double [R][E][C]  channel[0].rawP / .correctedP / .el / .az (:212, :243, :227)
 *   sat_pos   double [R][E][C][3], sat_clk double [R][E][C]: satpos outputs per listed channel (optional, may be NULL)
 *   active    uint8 [R][E][C]   1 = channel was in activeChnList of that epoch (channel[0].PRN != 0)
 *   sol       double [R][E][SGX_NAV_SOL_FIELDS]: X Y Z dt (NaN without a fix), DOP[5] (0 without a fix), latitude,
 *             longitude (degrees), height
 * Float64 throughout; agrees with the reference to 1e-5 m on the fix (pseudoranges are bit-identical). */
int sgx_nav_solve(const double* abs_sample, int64_t stride, int32_t n_recordings, int32_t n_channels, int32_t ms,
                  const int32_t* sub_frame_start, const uint8_t* ready, const sgx_eph* eph, const double* tow,
                  const int32_t* n_epochs, int32_t max_epochs, const sgx_nav_settings* st, double* raw_p,
                  double* corrected_p, double* el, double* az, double* sat_pos, double* sat_clk, uint8_t* active,
                  double* sol, void* cuda_stream);

/* ---- velocity and clock drift from Doppler (extension; no reference behaviour) -------------------------------- */
typedef struct sgx_vel_settings {
  double IF;               /* Hz: settings.IF, subtracted from the PLL's carrier frequency */
  double c;                /* m/s: settings.c */
  double f_L1;             /* Hz: 1575.42e6 */
  double nav_sol_period;   /* ms between epochs: settings.navSolPeriod, as in sgx_nav_settings */
  int32_t doppler_avg_ms;  /* N >= 1 code periods averaged per Doppler (default 100) */
  int32_t reserved;
} sgx_vel_settings;

#define SGX_NAV_VEL_FIELDS 8   /* VX VY VZ (ECEF, m/s) clock drift (m/s) VE VN VU (m/s) channels used */

/* Receiver velocity and clock drift at the measurement epochs of sgx_nav_solve, from the carrier frequency the PLL
 * tracked (field 2 of sgx_track's output).  Float64 throughout.  For recording r, epoch e < n_epochs[r], channel c:
 *   m = sub_frame_start[c] + (int)nav_sol_period * e (K8's msOfTheSignal); transmit time t = tow[r] advanced by e
 *   repeated additions of nav_sol_period / 1000 (as sgx_nav_solve)
 *   D = sum(carr_freq[m-N+1 .. m], increasing index) / N - IF   with N = doppler_avg_ms; D = NaN (channel excluded)
 *       when m-N+1 < 0 or m >= ms_done[c].  The window trails the epoch by (N-1)/2 ms.
 *   measured range rate rr = -(c / f_L1) * D
 *   satellite position, clock and their analytic time derivatives from the ephemeris at t (the arithmetic of
 *   satpos, geoFunctions/__init__.py:779-885): Edot = n / (1 - e cosE), nudot = Edot sqrt(1-e^2) / (1 - e cosE),
 *   udot = nudot (1 + 2 (C_us cos2phi - C_uc sin2phi)), rdot = a e sinE Edot + 2 nudot (C_rs cos2phi - C_rc sin2phi),
 *   idot = iDot + 2 nudot (C_is cos2phi - C_ic sin2phi), Omegadot = omegaDot - 7.2921151467e-5;
 *   satellite clock drift = a_f1 + 2 a_f2 dt + F e sqrtA cosE Edot
 *   Earth rotation: tau = |x_s - x_r| / c once, x_r the epoch's fix (sol X Y Z); x_s and v_s rotated about z by
 *   7.292115147e-5 * tau (e_r_corr's constant).  The rate of that rotation angle (< 1 cm/s) is ignored.
 *   channels used: active[r][e][c] == 1 and D finite.  With u_c = (x_s,rot - x_r) / |x_s,rot - x_r| the row is
 *   [-u_c, 1] and y_c = rr_c - u_c . v_s,rot + c * satellite clock drift; the 4x4 normal equations are solved by
 *   Cholesky for (vx, vy, vz, c * receiver clock drift).  The epoch is NaN when its fix is NaN, when fewer than 4
 *   channels are used, or when a Cholesky pivot is not above 1e-13 of the trace.
 *   carr_freq        double: the carrFreq series of channel (r, c) starts at carr_freq + (r*n_channels + c)*stride and
 *                    holds ms values (sgx_track's output + 2*ms, stride = SGX_TRACK_FIELDS*ms)
 *   ms_done          host int32 [R][C] periods completed, each in [0, ms]; NULL: all ms
 *   sub_frame_start, eph, tow, n_epochs, max_epochs  as given to sgx_nav_solve
 *   active           uint8 [R][E][C], sol double [R][E][SGX_NAV_SOL_FIELDS]: sgx_nav_solve's outputs
 * Outputs, E = max_epochs:
 *   vel       double [R][E][SGX_NAV_VEL_FIELDS]: VX VY VZ, clock drift, VE VN VU (rotated at sol's latitude and
 *             longitude), channels used (the count of the rule above, also when the epoch is NaN)
 *   doppler   double [R][E][C] D in Hz of the channels used, NaN elsewhere
 *   rr_resid  double [R][E][C] post-fit range-rate residual y_c - row_c . x (m/s), NaN unless used in a solution
 *   sat_vel   double [R][E][C][3], sat_clk_drift double [R][E][C] (s/s): unrotated satellite velocity and clock drift
 *             of the active channels, NaN elsewhere (optional, may be NULL)
 * Epochs >= n_epochs[r] are NaN with 0 channels used.  Deterministic: fixed summation order, no atomics.
 * SGX_ERR_ARG for NULL required pointers, 1..32 channels, ms <= 0, stride < ms, ms_done outside [0, ms],
 * doppler_avg_ms < 1, nav_sol_period < 1, c, f_L1 not finite and > 0 or IF not finite. */
int sgx_nav_velocity(const double* carr_freq, int64_t stride, int32_t n_recordings, int32_t n_channels, int32_t ms,
                     const int32_t* ms_done, const int32_t* sub_frame_start, const sgx_eph* eph, const double* tow,
                     const int32_t* n_epochs, int32_t max_epochs, const uint8_t* active, const double* sol,
                     const sgx_vel_settings* vs, double* vel, double* doppler, double* rr_resid, double* sat_vel,
                     double* sat_clk_drift, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* SOFTGNSS_B200_H */
