// world_analysis.cu -- WORLD analysis on the B200: DIO + StoneMask (f0), CheapTrick (spectral
// envelope, fused with SPTK sp2mc), D4C (aperiodicity).  Replaces the CPU pyworld/pysptk calls
// reached from realtime_voice_conversion/yukarin_wrapper/vocoder.py:26-48 ->
// acoustic_feature_wrapper.py:28-33 -> yukarin.AcousticFeature.extract (SURVEY rows a6, A-E).
//
// Mapping to the hardware (all FP64, no tensor cores: this is FFT / scan / sort work):
//   * DIO's whole-chunk FFTs (16k-64k points) go through cuFFT (D2Z once, batched Z2D for the bands);
//   * everything per-frame is ONE CTA per frame with the frame resident in shared memory:
//     window -> FFT -> smoothing (block scan) -> cepstral lifter -> FFT -> exp, so a frame's
//     intermediate spectra never reach HBM;
//   * zero-crossing extraction is an ordered block compaction (warp-shuffle scans);
//   * the sequential f0-contour repair (<= a few hundred frames) runs on a single thread.
#include <cufft.h>
#include <math.h>
#include <vector>

#include "analysis_shared.cuh"
#include "engine.h"
#include "fft.cuh"

namespace ryk {

// ------------------------------------------------------------------------------------ DIO
__global__ void k_dio_prepare(const float* __restrict__ x, int n, int y_length, int fft_size, double* __restrict__ y) {
  __shared__ double scratch[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += (double)x[i];
  double mean = block_sum(s, scratch) / y_length;
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double v = 0.0;
    if (i < n) v = (double)x[i] - mean;
    else if (i < y_length) v = -mean;
    y[i] = v;
  }
}

// time-domain filters whose spectra are cached per plan: index 0 = low-cut, 1+b = band b Nuttall LPF
__global__ void k_dio_design_filters(double* __restrict__ filt, int fft_size, int cutoff_N, const int* __restrict__ half_avg) {
  int which = blockIdx.x;
  double* f = filt + (size_t)which * fft_size;
  if (which == 0) {
    __shared__ double scratch[32];
    int N = cutoff_N;
    double s = 0.0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) s += 0.5 - 0.5 * cos((i + 1) * 2.0 * kPi / (N + 1));
    double sum = block_sum(s, scratch);
    int sh = (N - 1) / 2;
    // circularly centred: tap j of the normalised negated Hanning lands at (j - sh) mod fft_size
    for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
      int j;   // source tap
      if (i <= N - 1 - sh) j = i + sh; else if (i >= fft_size - sh) j = i - (fft_size - sh); else j = -1;
      double v = 0.0;
      if (j >= 0 && j < N) v = -(0.5 - 0.5 * cos((j + 1) * 2.0 * kPi / (N + 1))) / sum;
      if (i == 0) v += 1.0;
      f[i] = v;
    }
  } else {
    int len = half_avg[which - 1] * 4;
    for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
      double v = 0.0;
      if (i < len) {
        double tmp = i / (len - 1.0);
        v = 0.355768 - 0.487396 * cos(2.0 * kPi * tmp) + 0.144232 * cos(4.0 * kPi * tmp) - 0.012604 * cos(6.0 * kPi * tmp);
      }
      f[i] = v;
    }
  }
}

// Y *= F (low-cut), in place
__global__ void k_cmul_inplace(cufftDoubleComplex* __restrict__ y, const cufftDoubleComplex* __restrict__ f, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    cufftDoubleComplex a = y[i], b = f[i];
    y[i] = make_double2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
  }
}

__global__ void k_dio_candidates(const double* __restrict__ loc, const double* __restrict__ itv, const int* __restrict__ counts,
                                 int y_length, int f0_length, int nbands, double frame_period, double f0_floor, double f0_ceil,
                                 const double* __restrict__ boundary, double* __restrict__ cand, double* __restrict__ score) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int b = blockIdx.y;
  if (i >= f0_length) return;
  const int* c = counts + b * 4;
  double cv = 0.0, sv = kMaxValue;
  if (c[0] > 2 && c[1] > 2 && c[2] > 2 && c[3] > 2) {
    double t = i * frame_period / 1000.0;
    double v[4];
    for (int e = 0; e < 4; ++e) {
      size_t slot = ((size_t)b * 4 + e) * y_length;
      v[e] = interp1_at(loc + slot, itv + slot, c[e], t);
    }
    cv = (v[0] + v[1] + v[2] + v[3]) / 4.0;
    sv = sqrt(((v[0] - cv) * (v[0] - cv) + (v[1] - cv) * (v[1] - cv) + (v[2] - cv) * (v[2] - cv) + (v[3] - cv) * (v[3] - cv)) / 3.0);
    double bf = boundary[b];
    if (cv > bf || cv < bf / 2.0 || cv > f0_ceil || cv < f0_floor) { cv = 0.0; sv = kMaxValue; }
  }
  cand[(size_t)b * f0_length + i] = cv;
  score[(size_t)b * f0_length + i] = sv / (cv + kSafeMin);
}

__device__ inline double dio_select_best(double cur, double past, const double* cand, int nbands, int f0_length, int target, double allowed) {
  double ref = (cur * 3.0 - past) / 2.0;
  double minerr = fabs(ref - cand[target]), best = cand[target];
  for (int b = 1; b < nbands; ++b) {
    double err = fabs(ref - cand[(size_t)b * f0_length + target]);
    if (err < minerr) { minerr = err; best = cand[(size_t)b * f0_length + target]; }
  }
  if (fabs(1.0 - best / ref) > allowed) return 0.0;
  return best;
}

// best-band selection (parallel) + FixF0Contour steps 1-4 (sequential, thread 0). scratch: 3*f0_length doubles + 2*f0_length ints
__global__ void k_dio_fix(const double* __restrict__ cand, const double* __restrict__ score, int nbands, int f0_length,
                          double frame_period, double f0_floor, double* __restrict__ scratch, int* __restrict__ iscratch,
                          double* __restrict__ f0) {
  const double allowed = 0.1;
  double* best = scratch;
  double* t1 = scratch + f0_length;
  double* t2 = scratch + 2 * (size_t)f0_length;
  for (int i = threadIdx.x; i < f0_length; i += blockDim.x) {
    double tmp = score[i], bv = cand[i];
    for (int b = 1; b < nbands; ++b) {
      double s = score[(size_t)b * f0_length + i];
      if (tmp > s) { tmp = s; bv = cand[(size_t)b * f0_length + i]; }
    }
    best[i] = bv;
    f0[i] = 0.0;
  }
  __syncthreads();
  int vrm = (int)(0.5 + 1000.0 / frame_period / f0_floor) * 2 + 1;
  if (f0_length <= vrm) return;
  // step 1 (parallel)
  for (int i = threadIdx.x; i < f0_length; i += blockDim.x) {
    double v = 0.0;
    if (i >= vrm) {
      double bi = (i < vrm || i >= f0_length - vrm) ? 0.0 : best[i];
      double bp = (i - 1 < vrm || i - 1 >= f0_length - vrm) ? 0.0 : best[i - 1];
      v = fabs((bi - bp) / (kSafeMin + bi)) < allowed ? bi : 0.0;
    }
    t1[i] = v;
  }
  __syncthreads();
  // step 2 (parallel)
  int center = (vrm - 1) / 2;
  for (int i = threadIdx.x; i < f0_length; i += blockDim.x) {
    double v = t1[i];
    if (i >= center && i < f0_length - center) {
      for (int j = -center; j <= center; ++j) if (t1[i + j] == 0) { v = 0.0; break; }
    }
    t2[i] = v;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  int* pos = iscratch; int* neg = iscratch + f0_length;
  int pc = 0, nc = 0;
  for (int i = 1; i < f0_length; ++i) {
    if (t2[i] == 0 && t2[i - 1] != 0) neg[nc++] = i - 1;
    else if (t2[i - 1] == 0 && t2[i] != 0) pos[pc++] = i;
  }
  // step 3: forward extension (t1 <- t2)
  for (int i = 0; i < f0_length; ++i) t1[i] = t2[i];
  for (int i = 0; i < nc; ++i) {
    int limit = i == nc - 1 ? f0_length - 1 : neg[i + 1];
    for (int j = neg[i]; j < limit; ++j) {
      double v = dio_select_best(t1[j], t1[j - 1], cand, nbands, f0_length, j + 1, allowed);
      t1[j + 1] = v;
      if (v == 0) break;
    }
  }
  // step 4: backward extension
  for (int i = 0; i < f0_length; ++i) f0[i] = t1[i];
  for (int i = pc - 1; i >= 0; --i) {
    int limit = i == 0 ? 1 : pos[i - 1];
    for (int j = pos[i]; j > limit; --j) {
      double v = dio_select_best(f0[j], f0[j + 1], cand, nbands, f0_length, j - 1, allowed);
      f0[j - 1] = v;
      if (v == 0) break;
    }
  }
}

// ------------------------------------------------------------------------------------ StoneMask
__device__ inline double stonemask_fix(const double* power, const double* numer, int fft_size, int fs, double f0i, int nh) {
  double num = 0.0, den = 0.0;
  for (int i = 0; i < nh; ++i) {
    int index = matlab_round(f0i * fft_size / fs * (i + 1));
    double p = power[index];
    double inst = p == 0.0 ? 0.0 : (double)index * fs / fft_size + numer[index] / p * fs / 2.0 / kPi;
    double amp = sqrt(p);
    num += amp * inst;
    den += amp * (i + 1);
  }
  return num / (den + kSafeMin);
}

// StoneMask's FFT size for an f0 estimate of f0i (> 0)
__host__ __device__ inline int stonemask_fft_size(int fs, double f0i) {
  int half = (int)(1.5 * fs / f0i + 1.0);
  // NB: device pow() is not exact for integer powers (2 ulp): a truncated 2047 would wreck the FFT. Shift instead.
  return 1 << (2 + (int)(log(half * 2.0 + 1.0) / kLog2));
}

// one CTA per frame; smem: 2 * fft_cap double2 (main / diff spectra) + 64 bytes, which keeps stonemask_fix's reads of bins up to
// fft_size (a harmonic of the tentative f0 above Nyquist) inside the allocation, as the former separate arrays did.  fft_cap is the FFT size of the plan's lowest f0 (2048 at
// 24 kHz / 71 Hz); a frame whose f0 would need a larger transform keeps its unrefined estimate.
__global__ void __launch_bounds__(256) k_stonemask(const float* __restrict__ x, int x_length, int fs, double frame_period,
                                                  const double* __restrict__ f0_in, double* __restrict__ f0_out,
                                                  const double2* __restrict__ tw, int fft_cap) {
  extern __shared__ double2 sm2[];
  int frame = blockIdx.x;
  double f0i = f0_in[frame];
  if (f0i <= 40.0 || f0i > fs / 12.0) { if (threadIdx.x == 0) f0_out[frame] = 0.0; return; }
  int fft_size = stonemask_fft_size(fs, f0i);
  if (fft_size > fft_cap) { if (threadIdx.x == 0) f0_out[frame] = f0i; return; }
  double pos = frame * frame_period / 1000.0;
  int half = (int)(1.5 * fs / f0i + 1.0);
  double wlen_time = (2.0 * half + 1.0) / fs;
  int blen = half * 2 + 1;
  int lg = ilog2(fft_size);
  double2* A = sm2;                 // main
  double2* B = sm2 + fft_cap;       // diff
  // only bins 0..fft/2 of each spectrum are read: power and numer go to the upper halves (fft/2 - 1 double2 >= fft/2 + 1 doubles)
  double* power = (double*)(A + fft_size / 2 + 1);
  double* numer = (double*)(B + fft_size / 2 + 1);
  int basic_index = matlab_round((pos + (double)(-half) / fs) * fs + 0.001);
  auto mainw = [&](int i) {
    double tmp = ((basic_index + i) - 1.0) / fs - pos;
    return 0.42 + 0.5 * cos(2.0 * kPi * tmp / wlen_time) + 0.08 * cos(4.0 * kPi * tmp / wlen_time);
  };
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double a = 0.0, b = 0.0;
    if (i < blen) {
      double xv = (double)x[imax(0, imin(x_length - 1, basic_index + i - 1))];
      double mw = mainw(i), dw;
      if (i == 0) dw = -mainw(1) / 2.0;
      else if (i == blen - 1) dw = mainw(blen - 2) / 2.0;
      else dw = -(mainw(i + 1) - mainw(i - 1)) / 2.0;
      a = xv * mw; b = xv * dw;
    }
    A[i] = make_double2(a, 0.0);
    B[i] = make_double2(b, 0.0);
  }
  fft_smem(A, fft_size, lg, -1, tw);
  fft_smem(B, fft_size, lg, -1, tw);
  for (int j = threadIdx.x; j <= fft_size / 2; j += blockDim.x) {
    double2 m = A[j], d = B[j];
    numer[j] = m.x * d.y - m.y * d.x;
    power[j] = m.x * m.x + m.y * m.y;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tentative = stonemask_fix(power, numer, fft_size, fs, f0i, 2);
    double mean_f0;
    if (tentative <= 0.0 || tentative > f0i * 2) mean_f0 = 0.0;
    else mean_f0 = stonemask_fix(power, numer, fft_size, fs, tentative, 6);
    if (fabs(mean_f0 - f0i) > f0i * 0.2) mean_f0 = f0i;
    f0_out[frame] = mean_f0;
  }
}

// ------------------------------------------------------------------------------------ shared smoothing helpers
// DCCorrection, in place on a[] (smem). All threads call.
__device__ inline void dc_correction_smem(double* a, double f0, int fs, int fft_size) {
  int upper_limit = 2 + (int)(f0 * fft_size / fs);
  int nrep = upper_limit - 1;
  double dx = -(double)fs / fft_size;
  double rep[2] = {0.0, 0.0};
  int c = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < nrep; i += blockDim.x, ++c)
    rep[c] = interp1q(f0, dx, a, upper_limit + 1, (double)i * fs / fft_size);
  __syncthreads();
  c = 0;
  for (int i = threadIdx.x; i < nrep; i += blockDim.x, ++c) a[i] = a[i] + rep[c];
  __syncthreads();
}

// LinearSmoothing: in[0..half] -> out[0..half] (may alias). seg: scratch >= half + 2*boundary + 1, scan scratch >= blockDim.x
__device__ inline void linear_smoothing_smem(const double* in, double* out, double width, int fs, int fft_size,
                                             double* seg, double* scan_scratch) {
  int half = fft_size / 2;
  int boundary = (int)(width * fft_size / fs) + 1;
  int mlen = half + boundary * 2 + 1;
  __syncthreads();
  for (int i = threadIdx.x; i < mlen; i += blockDim.x) {
    double v;
    if (i < boundary) v = in[boundary - i];
    else if (i < half + boundary) v = in[i - boundary];
    else v = in[half - (i - (half + boundary))];
    seg[i] = v * fs / fft_size;
  }
  __syncthreads();
  block_inclusive_scan(seg, mlen, scan_scratch);
  double origin = -(boundary - 0.5) * fs / fft_size;
  double interval = (double)fs / fft_size;
  for (int i = threadIdx.x; i <= half; i += blockDim.x) {
    double axis = (double)i / fft_size * fs - width / 2.0;
    double low = interp1q(origin, interval, seg, mlen, axis);
    double high = interp1q(origin, interval, seg, mlen, axis + width);
    out[i] = (high - low) / width;
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------ CheapTrick (+ sp2mc)
// one CTA (256 threads) per frame. DECIDE (matches oracle): randn dither dropped, +eps constant.
constexpr int kCtMaxFft = 2048;
constexpr double kMaxF0Smem = 2000.0;   // StoneMask caps refined f0 at fs/12; scratch is sized for this
__host__ __device__ inline int ct_seg_len(int fft_size, int fs) { return fft_size / 2 + 1 + 2 * ((int)(kMaxF0Smem * 2.0 / 3.0 * fft_size / fs) + 2) + 2; }
__host__ __device__ inline int d4c_seg_len(int fft_d4c, int fs) { return fft_d4c / 2 + 1 + 2 * ((int)(kMaxF0Smem * fft_d4c / fs) + 2) + 2; }
__global__ void __launch_bounds__(256) k_cheaptrick(const float* __restrict__ x, int x_length, int fs, double frame_period,
                                                   const double* __restrict__ f0, int fft_size, double q1,
                                                   const double* __restrict__ G /*[ (order+1) ][nb]*/, int order,
                                                   int n_out, float* __restrict__ sp_out, float* __restrict__ mc_out,
                                                   double* __restrict__ sp_f64 /*nullable*/, const double2* __restrict__ tw) {
  extern __shared__ double2 sm2[];
  int frame = blockIdx.x;
  int half_fft = fft_size / 2, nb = half_fft + 1, lg = ilog2(fft_size);
  double2* A = sm2;                                   // fft_size
  double* ps = (double*)(sm2 + fft_size);             // nb (+1)
  double* seg = ps + nb + 1;                          // nb + 2*boundary + 1  (boundary <= ~ 0.67*f0*fft/fs + 1)
  double* scratch = seg + ct_seg_len(fft_size, fs);   // blockDim.x + 32
  double f0_floor = 3.0 * fs / (fft_size - 3.0);
  double cf0 = f0[frame] <= f0_floor ? kDefaultF0 : f0[frame];
  double pos = frame * frame_period / 1000.0;
  int half = matlab_round(1.5 * fs / cf0);
  int origin = matlab_round(pos * fs + 0.001);
  // window energy
  double acc = 0.0;
  for (int i = threadIdx.x; i <= half * 2; i += blockDim.x) {
    double p = (i - half) / 1.5 / fs;
    double w = 0.5 * cos(kPi * p * cf0) + 0.5;
    acc += w * w;
  }
  double average = sqrt(block_sum(acc, scratch));
  double w1 = 0.0, w2 = 0.0;
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double wv = 0.0, v = 0.0;
    if (i <= half * 2) {
      double p = (i - half) / 1.5 / fs;
      wv = (0.5 * cos(kPi * p * cf0) + 0.5) / average;
      int idx = imin(x_length - 1, imax(0, origin + i - half));
      v = (double)x[idx] * wv;
      w1 += v; w2 += wv;
    }
    A[i] = make_double2(v, wv);      // stash the window in .y until the DC removal
  }
  double s1 = block_sum(w1, scratch);
  double s2 = block_sum(w2, scratch);
  double coef = s1 / s2;
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double2 v = A[i];
    A[i] = make_double2(i <= half * 2 ? v.x - v.y * coef : 0.0, 0.0);
  }
  fft_smem(A, fft_size, lg, -1, tw);
  for (int i = threadIdx.x; i < nb; i += blockDim.x) { double2 v = A[i]; ps[i] = v.x * v.x + v.y * v.y; }
  if (threadIdx.x == 0) ps[nb] = 0.0;
  dc_correction_smem(ps, cf0, fs, fft_size);
  linear_smoothing_smem(ps, ps, cf0 * 2.0 / 3.0, fs, fft_size, seg, scratch);
  // SmoothingWithRecovery
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    int k = i <= half_fft ? i : fft_size - i;
    A[i] = make_double2(log(ps[k] + kEps), 0.0);
  }
  fft_smem(A, fft_size, lg, -1, tw);
  for (int i = threadIdx.x; i <= half_fft; i += blockDim.x) {
    double sl, cl;
    if (i == 0) { sl = 1.0; cl = (1.0 - 2.0 * q1) + 2.0 * q1; }
    else {
      double quef = (double)i / fs;
      sl = sin(kPi * cf0 * quef) / (kPi * cf0 * quef);
      cl = (1.0 - 2.0 * q1) + 2.0 * q1 * cos(2.0 * kPi * quef * cf0);
    }
    A[i] = make_double2(A[i].x * sl * cl / fft_size, 0.0);
  }
  irfft_smem(A, fft_size, lg, tw);
  // envelope + fused sp2mc (mc = G . log(sp))
  for (int i = threadIdx.x; i < nb; i += blockDim.x) {
    double spv = exp(A[i].x);
    ps[i] = log(spv);
    if (frame < n_out) {
      sp_out[(size_t)frame * nb + i] = (float)spv;
      if (sp_f64) sp_f64[(size_t)frame * nb + i] = spv;
    }
  }
  __syncthreads();
  for (int j = 0; j <= order; ++j) {
    double a = 0.0;
    for (int i = threadIdx.x; i < nb; i += blockDim.x) a += G[(size_t)j * nb + i] * ps[i];
    double m = block_sum(a, scratch);
    if (threadIdx.x == 0 && frame < n_out) mc_out[(size_t)frame * (order + 1) + j] = (float)m;
  }
}

// ------------------------------------------------------------------------------------ D4C
// block_sum of two values at once: the same warp trees and the same fixed-order pass over the warp totals as two block_sum() calls
// (bit-identical results), at the barriers of one.
__device__ inline double2 d4c_block_sum2(double a, double b, double* scratch) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  a = warp_sum(a);
  b = warp_sum(b);
  __syncthreads();
  if (lane == 0) { scratch[w] = a; scratch[32 + w] = b; }
  __syncthreads();
  if (w == 0) {
    double ra = warp_sum(lane < nw ? scratch[lane] : 0.0);
    double rb = warp_sum(lane < nw ? scratch[32 + lane] : 0.0);
    if (lane == 0) { scratch[0] = ra; scratch[1] = rb; }
  }
  __syncthreads();
  const double2 r = make_double2(scratch[0], scratch[1]);
  __syncthreads();
  return r;
}

// windowed waveform into A[i].x (i < fft), zero elsewhere; returns after DC-weight removal.
__device__ inline void d4c_window_smem(double2* A, int fft_size, const float* __restrict__ x, int x_length, int fs,
                                       double cf0, double pos, bool blackman, double ratio, double* scratch) {
  int half = matlab_round(ratio * fs / cf0 / 2.0);
  int origin = matlab_round(pos * fs + 0.001);
  double w1 = 0.0, w2 = 0.0;
  __syncthreads();
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double v = 0.0, wv = 0.0;
    if (i <= half * 2) {
      double p = (2.0 * (i - half) / ratio) / fs;
      wv = blackman ? 0.42 + 0.5 * cos(kPi * p * cf0) + 0.08 * cos(kPi * p * cf0 * 2) : 0.5 * cos(kPi * p * cf0) + 0.5;
      int idx = imin(x_length - 1, imax(0, origin + i - half));
      v = (double)x[idx] * wv;
      w1 += v; w2 += wv;
    }
    A[i] = make_double2(v, wv);
  }
  const double2 s12 = d4c_block_sum2(w1, w2, scratch);
  double coef = s12.x / s12.y;
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double2 v = A[i];
    A[i] = make_double2(i <= half * 2 ? v.x - v.y * coef : 0.0, 0.0);
  }
  __syncthreads();
}

// centroid of the frame at `pos` accumulated into cen[] (+=). tmp: nb doubles x2
__device__ inline void d4c_centroid_smem(double2* A, int fft_size, int lg, const float* __restrict__ x, int x_length, int fs,
                                         double cf0, double pos, double* tr, double* ti, double* cen, bool accumulate,
                                         double* scratch, const double2* __restrict__ tw) {
  int nb = fft_size / 2 + 1;
  d4c_window_smem(A, fft_size, x, x_length, fs, cf0, pos, true, 4.0, scratch);
  int lim = matlab_round(2.0 * fs / cf0) * 2;
  double p = 0.0;
  for (int i = threadIdx.x; i <= lim; i += blockDim.x) p += A[i].x * A[i].x;
  double power = block_sum(p, scratch);
  double sq = sqrt(power);
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double v = A[i].x;
    if (i <= lim) v = v / sq;
    A[i] = make_double2(v, 0.0);
  }
  __syncthreads();
  // WORLD needs FFT(v) and FFT((n+1) v): one complex FFT of v + i (n+1) v yields both by Hermitian symmetry.
  for (int i = threadIdx.x; i < fft_size; i += blockDim.x) {
    double v = A[i].x;
    A[i] = make_double2(v, v * (i + 1.0));
  }
  fft_smem(A, fft_size, lg, -1, tw);
  // Z[k] = X[k] + i Y[k];  X[k] = (Z[k] + conj(Z[N-k]))/2,  Y[k] = (Z[k] - conj(Z[N-k]))/(2i)
  for (int k = threadIdx.x; k < nb; k += blockDim.x) {
    double2 z = A[k];
    double2 zc = A[(fft_size - k) & (fft_size - 1)];
    double xr = 0.5 * (z.x + zc.x), xi = 0.5 * (z.y - zc.y);
    double yr = 0.5 * (z.y + zc.y), yi = -0.5 * (z.x - zc.x);
    tr[k] = xr; ti[k] = xi;
    double c = yr * xr + xi * yi;
    cen[k] = accumulate ? cen[k] + c : c;
  }
  __syncthreads();
}

// Coarse aperiodicity needs, per band, the sum of the m smallest of its n band powers and the sum of all n.  No sort: an 8-bit radix
// select over the IEEE-754 bit patterns (non-negative doubles order like their uint64 patterns) finds the m-th smallest value t of
// each band, and then sum_m = sum(v < t) + (m - #{v < t}) * t, which counts ties with t exactly.  The nb <= kD4cMaxBands bands are
// selected together, one block barrier per digit for all of them; every warp scans the histograms itself, so no second barrier.
// hist: 3 * nb * 256 ints (a histogram is zeroed two digits after it was read).  red: >= 16 * (blockDim.x / 32) doubles.
// Sums are taken in a fixed order (per-thread index order, warp trees, warps in order): the result does not depend on timing.
constexpr int kD4cMaxBands = 5;     // fmin(15000, fs/2 - 3000) / 3000
__device__ inline void d4c_select_sums(double* const* p, int nb, int n, int m, int* hist, double* red, double* sum_m, double* sum_all) {
  const int T = blockDim.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = T >> 5;
  unsigned long long prefix[kD4cMaxBands];
  int rank[kD4cMaxBands];                 // rank of the wanted value among the values that still match prefix
#pragma unroll
  for (int b = 0; b < kD4cMaxBands; ++b) { prefix[b] = 0ull; rank[b] = m - 1; }
  for (int i = threadIdx.x; i < nb * 256; i += T) hist[i] = 0;
  __syncthreads();
  for (int pass = 0; pass < 8; ++pass) {
    const int shift = 56 - 8 * pass;
    int* H = hist + (pass % 3) * nb * 256;
    int* Hn = hist + ((pass + 1) % 3) * nb * 256;
    for (int i = threadIdx.x; i < nb * 256; i += T) Hn[i] = 0;
#pragma unroll
    for (int b = 0; b < kD4cMaxBands; ++b) {
      if (b >= nb) break;
      for (int i0 = 0; i0 < n; i0 += T) {          // warp-uniform trip count: __match_any_sync needs the whole warp
        const int i = i0 + threadIdx.x;
        int bin = -1;
        if (i < n) {
          const unsigned long long key = (unsigned long long)__double_as_longlong(p[b][i]);
          if (pass == 0 || (key >> (shift + 8)) == (prefix[b] >> (shift + 8))) bin = (int)((key >> shift) & 255ull);
        }
        const unsigned same = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && lane == __ffs(same) - 1) atomicAdd(&H[b * 256 + bin], __popc(same));
      }
    }
    __syncthreads();
#pragma unroll
    for (int b = 0; b < kD4cMaxBands; ++b) {
      if (b >= nb) break;
      const int4 c0 = *(const int4*)&H[b * 256 + lane * 8];
      const int4 c1 = *(const int4*)&H[b * 256 + lane * 8 + 4];
      const int c[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
      const int tot = c[0] + c[1] + c[2] + c[3] + c[4] + c[5] + c[6] + c[7];
      int incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
      const int L = __ffs(__ballot_sync(0xffffffffu, incl > rank[b])) - 1;   // the lane whose 8 bins hold the wanted rank
      int digit = 0, below = incl - tot;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (rank[b] < below + c[j]) { digit = lane * 8 + j; break; }
        below += c[j];
      }
      digit = __shfl_sync(0xffffffffu, digit, L);
      below = __shfl_sync(0xffffffffu, below, L);
      prefix[b] |= (unsigned long long)digit << shift;
      rank[b] -= below;
    }
  }
  // prefix[b] is now the bit pattern of the m-th smallest value of band b
#pragma unroll
  for (int b = 0; b < kD4cMaxBands; ++b) {
    if (b >= nb) break;
    double s_lt = 0.0, s_all = 0.0, c_lt = 0.0;
    for (int i = threadIdx.x; i < n; i += T) {
      const double v = p[b][i];
      s_all += v;
      if ((unsigned long long)__double_as_longlong(v) < prefix[b]) { s_lt += v; c_lt += 1.0; }
    }
    s_lt = warp_sum(s_lt); s_all = warp_sum(s_all); c_lt = warp_sum(c_lt);
    if (lane == 0) { red[w * 16 + 3 * b] = s_lt; red[w * 16 + 3 * b + 1] = s_all; red[w * 16 + 3 * b + 2] = c_lt; }
  }
  __syncthreads();
#pragma unroll
  for (int b = 0; b < kD4cMaxBands; ++b) {
    if (b < nb && threadIdx.x == 32 * b) {          // one thread per band, each in its own warp
      double s_lt = 0.0, s_all = 0.0, c_lt = 0.0;
      for (int k = 0; k < nw; ++k) { s_lt += red[k * 16 + 3 * b]; s_all += red[k * 16 + 3 * b + 1]; c_lt += red[k * 16 + 3 * b + 2]; }
      sum_m[b] = s_lt + (m - c_lt) * __longlong_as_double((long long)prefix[b]);
      sum_all[b] = s_all;
    }
  }
  __syncthreads();
}

#ifdef RYK_D4C_TIMELINE
// diagnostics build only (RYK_NVCC_EXTRA=-DRYK_D4C_TIMELINE): %globaltimer stamps of k_d4c's phases, thread 0 of each CTA,
// dumped to RYK_D4C_TIMELINE_FILE after each launch outside a graph capture.  A frame that stops early leaves its later slots 0.
constexpr int kD4cTlMaxCtas = 1024, kD4cTlSlots = 16;
__device__ unsigned long long g_d4c_tl[kD4cTlMaxCtas * kD4cTlSlots];
#define D4C_TL(slot) do { if (threadIdx.x == 0 && blockIdx.x < kD4cTlMaxCtas) { unsigned long long t_; \
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); g_d4c_tl[blockIdx.x * kD4cTlSlots + (slot)] = t_; } } while (0)
#else
#define D4C_TL(slot) do {} while (0)
#endif

// one CTA (512 threads) per frame
__global__ void __launch_bounds__(512) k_d4c(const float* __restrict__ x, int x_length, int fs, double frame_period,
                                            const double* __restrict__ f0, int fft_size_out, double threshold,
                                            int n_out, float* __restrict__ ap_out, const double2* __restrict__ tw,
                                            int fft_d4c, int lt_fft) {
  extern __shared__ double2 sm2[];
  int frame = blockIdx.x;
  if (frame >= n_out) return;
  const int nb_out = fft_size_out / 2 + 1;
  float* out = ap_out + (size_t)frame * nb_out;
  const int maxfft = fft_d4c > lt_fft ? fft_d4c : lt_fft;
  double2* A = sm2;
  double* base = (double*)(sm2 + maxfft);
  const int hb = fft_d4c / 2 + 1;
  const int alen = hb + 8;
  double* sc = base;                  // static centroid
  double* sps = sc + alen;            // smoothed power spectrum
  double* gd = sps + alen;            // group delay
  double* t1 = gd + alen;             // temp
  double* t2 = t1 + alen;             // temp
  double* seg = t2 + alen;            // smoothing scratch (hb + 2*boundary + 1)
  double* nwin = seg + d4c_seg_len(fft_d4c, fs);      // Nuttall band window (window_length <= hb values)
  double* coarse = nwin + alen;       // coarse aperiodicity (nap + 2) and the per-band sums (2 kD4cMaxBands)
  double* scratch = coarse + 24;      // blockDim.x + 32
  int* hist = (int*)(((uintptr_t)(scratch + 512 + 64) + 15) & ~(uintptr_t)15);   // radix-select histograms, 3 * nap * 256 (int4 reads)
  double f0v = f0[frame];
  double pos = frame * frame_period / 1000.0;
  const float unvoiced = (float)(1.0 - kSafeMin);
  bool skip = f0v == 0.0;
  D4C_TL(0);
  if (!skip) {
    // D4C LoveTrain
    int lg = ilog2(lt_fft);
    double cf0 = f0v > 40.0 ? f0v : 40.0;
    d4c_window_smem(A, lt_fft, x, x_length, fs, cf0, pos, true, 3.0, scratch);
    fft_smem(A, lt_fft, lg, -1, tw);
    int b0 = (int)ceil(100.0 * lt_fft / fs), b1 = (int)ceil(4000.0 * lt_fft / fs), b2 = (int)ceil(7900.0 * lt_fft / fs);
    double p1 = 0.0, p2 = 0.0;
    for (int i = b0 + 1 + threadIdx.x; i <= b2; i += blockDim.x) {
      double2 v = A[i];
      double pw = v.x * v.x + v.y * v.y;
      p2 += pw;
      if (i <= b1) p1 += pw;
    }
    const double2 s12 = d4c_block_sum2(p1, p2, scratch);
    double ap0 = s12.x / s12.y;
    skip = ap0 <= threshold;     // NaN compares false, exactly like the CPU code path
  }
  D4C_TL(1);
  if (skip) {
    for (int i = threadIdx.x; i < nb_out; i += blockDim.x) out[i] = unvoiced;
    return;
  }
  int lg = ilog2(fft_d4c);
  double cf0 = f0v > 47.0 ? f0v : 47.0;
  d4c_centroid_smem(A, fft_d4c, lg, x, x_length, fs, cf0, pos - 0.25 / cf0, t1, t2, sc, false, scratch, tw);
  D4C_TL(2);
  d4c_centroid_smem(A, fft_d4c, lg, x, x_length, fs, cf0, pos + 0.25 / cf0, t1, t2, sc, true, scratch, tw);
  if (threadIdx.x == 0) sc[hb] = 0.0;
  dc_correction_smem(sc, cf0, fs, fft_d4c);
  D4C_TL(3);
  // smoothed power spectrum
  d4c_window_smem(A, fft_d4c, x, x_length, fs, cf0, pos, false, 4.0, scratch);
  fft_smem(A, fft_d4c, lg, -1, tw);
  for (int i = threadIdx.x; i < hb; i += blockDim.x) { double2 v = A[i]; sps[i] = v.x * v.x + v.y * v.y; }
  if (threadIdx.x == 0) sps[hb] = 0.0;
  dc_correction_smem(sps, cf0, fs, fft_d4c);
  linear_smoothing_smem(sps, sps, cf0, fs, fft_d4c, seg, scratch);
  D4C_TL(4);
  // static group delay
  for (int i = threadIdx.x; i < hb; i += blockDim.x) gd[i] = sc[i] / sps[i];
  linear_smoothing_smem(gd, gd, cf0 / 2.0, fs, fft_d4c, seg, scratch);
  linear_smoothing_smem(gd, t1, cf0, fs, fft_d4c, seg, scratch);
  for (int i = threadIdx.x; i < hb; i += blockDim.x) gd[i] -= t1[i];
  __syncthreads();
  D4C_TL(5);
  // coarse aperiodicity: per band, the power spectrum of a Nuttall-windowed slice of gd; two bands share one complex FFT
  // (band b in the real part, band b + 1 in the imaginary part, split by Hermitian symmetry as in d4c_centroid_smem)
  const int nap = (int)(fmin(15000.0, fs / 2.0 - 3000.0) / 3000.0);
  const int window_length = (int)(3000.0 * fft_d4c / fs) * 2 + 1;
  const int half_wl = window_length / 2;
  const int boundary = matlab_round(fft_d4c * 8.0 / window_length);
  for (int i = threadIdx.x; i < window_length; i += blockDim.x) {
    double tmp = i / (window_length - 1.0);
    nwin[i] = 0.355768 - 0.487396 * cos(2.0 * kPi * tmp) + 0.144232 * cos(4.0 * kPi * tmp) - 0.012604 * cos(6.0 * kPi * tmp);
  }
  double* const bp[kD4cMaxBands] = {sc, sps, t1, t2, seg};   // band power spectra (hb values each); sc / sps / t1 / t2 / seg are free now
  for (int b = 0; b < nap; b += 2) {
    const bool pair = b + 1 < nap;
    const int c0 = (int)(3000.0 * (b + 1) * fft_d4c / fs) - half_wl;
    const int c1 = (int)(3000.0 * (b + 2) * fft_d4c / fs) - half_wl;
    __syncthreads();
    for (int i = threadIdx.x; i < fft_d4c; i += blockDim.x) {
      double v0 = 0.0, v1 = 0.0;
      if (i < window_length) {
        v0 = gd[c0 + i] * nwin[i];
        if (pair) v1 = gd[c1 + i] * nwin[i];
      }
      A[i] = make_double2(v0, v1);
    }
    fft_smem(A, fft_d4c, lg, -1, tw);
    D4C_TL(6 + b / 2);
    double* p0 = b == 0 ? sc : b == 2 ? t1 : seg;
    double* p1 = b == 0 ? sps : t2;
    for (int k = threadIdx.x; k < hb; k += blockDim.x) {
      const double2 z = A[k];
      if (pair) {
        const double2 zc = A[(fft_d4c - k) & (fft_d4c - 1)];
        const double xr = 0.5 * (z.x + zc.x), xi = 0.5 * (z.y - zc.y);
        const double yr = 0.5 * (z.y + zc.y), yi = -0.5 * (z.x - zc.x);
        p0[k] = xr * xr + xi * xi;
        p1[k] = yr * yr + yi * yi;
      } else {
        p0[k] = z.x * z.x + z.y * z.y;
      }
    }
  }
  __syncthreads();
  D4C_TL(9);
  // pa: the fft/2 - boundary smallest of the hb band powers, pb: all of them (the CPU code sorts and takes two cumulative sums)
  double* sum_m = coarse + kD4cMaxBands + 2;
  double* sum_all = sum_m + kD4cMaxBands;
  d4c_select_sums(bp, nap, hb, fft_d4c / 2 - boundary, hist, scratch, sum_m, sum_all);
  D4C_TL(10);
  if (threadIdx.x == 0) {
    coarse[0] = -60.0;
    coarse[nap + 1] = -kSafeMin;
    for (int b = 0; b < nap; ++b) coarse[1 + b] = fmin(0.0, 10 * log10(sum_m[b] / sum_all[b]) + (cf0 - 100) / 50.0);
  }
  D4C_TL(11);
  __syncthreads();
  for (int i = threadIdx.x; i < nb_out; i += blockDim.x) {
    double fx = (double)i * fs / fft_size_out;
    // coarse axis: k*3000 for k<=nap, fs/2 at nap+1
    int n = nap + 2;
    int lo = 0, hi = n;
    while (lo < hi) {
      int mid = (lo + hi) >> 1;
      double xm = mid <= nap ? mid * 3000.0 : fs / 2.0;
      if (xm <= fx) lo = mid + 1; else hi = mid;
    }
    int k = lo < 1 ? 1 : (lo > n - 1 ? n - 1 : lo);
    double x0 = (k - 1) <= nap ? (k - 1) * 3000.0 : fs / 2.0;
    double x1 = k <= nap ? k * 3000.0 : fs / 2.0;
    double s = (fx - x0) / (x1 - x0);
    double v = coarse[k - 1] + s * (coarse[k] - coarse[k - 1]);
    out[i] = (float)pow(10.0, v / 20.0);
  }
  D4C_TL(15);
}

// f0 / voiced outputs (float32 / uint8), trimmed to n_out frames
__global__ void k_f0_out(const double* __restrict__ f0, int n_out, float* __restrict__ f0_out, uint8_t* __restrict__ voiced) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_out) { double v = f0[i]; f0_out[i] = (float)v; voiced[i] = v != 0.0 ? 1 : 0; }
}

// ------------------------------------------------------------------------------------ host side
struct DioPlan {
  int n = 0, fs = 0, fft_size = 0, y_length = 0, f0_length = 0, nbands = 0;
  double frame_period = 0, f0_floor = 0, f0_ceil = 0;
  cufftHandle fwd = 0, inv = 0, fwd_filters = 0;
  double* d_y = nullptr; cufftDoubleComplex* d_Y = nullptr; cufftDoubleComplex* d_filt_spec = nullptr;   // [1+nbands][nbins]
  cufftDoubleComplex* d_Z = nullptr; double* d_filtered = nullptr;
  int* d_half_avg = nullptr; double* d_boundary = nullptr;
  int* d_edges = nullptr; double* d_loc = nullptr; double* d_itv = nullptr; int* d_counts = nullptr;
  double* d_cand = nullptr; double* d_score = nullptr; double* d_scratch = nullptr; int* d_iscratch = nullptr;
  double* d_f0 = nullptr; double* d_f0r = nullptr;
  HarvestPlan* harvest = nullptr;          // f0 method 1: Harvest writes d_f0 instead of DIO
};


void dio_plan_free(DioPlan* p) {
  if (!p) return;
  harvest_plan_free(p->harvest);
  if (p->fwd) cufftDestroy(p->fwd);
  if (p->inv) cufftDestroy(p->inv);
  if (p->fwd_filters) cufftDestroy(p->fwd_filters);
  void* ptrs[] = {p->d_y, p->d_Y, p->d_filt_spec, p->d_Z, p->d_filtered, p->d_half_avg, p->d_boundary, p->d_edges, p->d_loc,
                  p->d_itv, p->d_counts, p->d_cand, p->d_score, p->d_scratch, p->d_iscratch, p->d_f0, p->d_f0r};
  for (void* q : ptrs) if (q) cudaFree(q);
  delete p;
}

int dio_plan_create(Engine* e, int n, int fs, double frame_period, double f0_floor, double f0_ceil, DioPlan** out, int f0_method) {
  DioPlan* p = new DioPlan();
  if (f0_method == 1 && harvest_plan_create(e, n, fs, frame_period, f0_floor, f0_ceil, &p->harvest)) { delete p; return -1; }
  p->n = n; p->fs = fs; p->frame_period = frame_period; p->f0_floor = f0_floor; p->f0_ceil = f0_ceil;
  p->nbands = 1 + (int)(log(f0_ceil / f0_floor) / kLog2 * 2.0);
  std::vector<double> boundary(p->nbands);
  std::vector<int> half_avg(p->nbands);
  for (int i = 0; i < p->nbands; ++i) {
    boundary[i] = f0_floor * pow(2.0, (i + 1) / 2.0);
    half_avg[i] = matlab_round((double)fs / boundary[i] / 2.0);
  }
  p->y_length = n + 1;
  p->fft_size = suitable_fft_size(p->y_length + matlab_round((double)fs / 50.0) * 2 + 1 + (4 * (int)(1.0 + (double)fs / boundary[0] / 2.0)));
  p->f0_length = (int)(1000.0 * n / fs / frame_period) + 1;
  int nbins = p->fft_size / 2 + 1;
  size_t ev = (size_t)p->nbands * 4 * p->y_length;
  RYK_CUDA(cudaMalloc(&p->d_y, sizeof(double) * p->fft_size));
  RYK_CUDA(cudaMalloc(&p->d_Y, sizeof(cufftDoubleComplex) * nbins));
  RYK_CUDA(cudaMalloc(&p->d_filt_spec, sizeof(cufftDoubleComplex) * nbins * (1 + p->nbands)));
  RYK_CUDA(cudaMalloc(&p->d_Z, sizeof(cufftDoubleComplex) * nbins * p->nbands));
  RYK_CUDA(cudaMalloc(&p->d_filtered, sizeof(double) * (size_t)p->fft_size * (1 + p->nbands)));
  RYK_CUDA(cudaMalloc(&p->d_half_avg, sizeof(int) * p->nbands));
  RYK_CUDA(cudaMalloc(&p->d_boundary, sizeof(double) * p->nbands));
  RYK_CUDA(cudaMalloc(&p->d_edges, sizeof(int) * ev));
  RYK_CUDA(cudaMalloc(&p->d_loc, sizeof(double) * ev));
  RYK_CUDA(cudaMalloc(&p->d_itv, sizeof(double) * ev));
  RYK_CUDA(cudaMalloc(&p->d_counts, sizeof(int) * p->nbands * 4));
  RYK_CUDA(cudaMalloc(&p->d_cand, sizeof(double) * p->nbands * p->f0_length));
  RYK_CUDA(cudaMalloc(&p->d_score, sizeof(double) * p->nbands * p->f0_length));
  RYK_CUDA(cudaMalloc(&p->d_scratch, sizeof(double) * 3 * p->f0_length));
  RYK_CUDA(cudaMalloc(&p->d_iscratch, sizeof(int) * 2 * p->f0_length));
  RYK_CUDA(cudaMalloc(&p->d_f0, sizeof(double) * p->f0_length));
  RYK_CUDA(cudaMalloc(&p->d_f0r, sizeof(double) * p->f0_length));
  RYK_CUDA(cudaMemcpyAsync(p->d_half_avg, half_avg.data(), sizeof(int) * p->nbands, cudaMemcpyHostToDevice, e->stream));
  RYK_CUDA(cudaMemcpyAsync(p->d_boundary, boundary.data(), sizeof(double) * p->nbands, cudaMemcpyHostToDevice, e->stream));
  if (cufft_ok(cufftPlan1d(&p->fwd, p->fft_size, CUFFT_D2Z, 1), "plan D2Z")) return -1;
  if (cufft_ok(cufftPlan1d(&p->inv, p->fft_size, CUFFT_Z2D, p->nbands), "plan Z2D")) return -1;
  if (cufft_ok(cufftPlan1d(&p->fwd_filters, p->fft_size, CUFFT_D2Z, 1 + p->nbands), "plan D2Z filters")) return -1;
  // filter spectra, computed once (d_filtered doubles as the time-domain staging area)
  if (cufft_ok(cufftSetStream(p->fwd_filters, e->stream), "set stream")) return -1;
  k_dio_design_filters<<<1 + p->nbands, 256, 0, e->stream>>>(p->d_filtered, p->fft_size, matlab_round((double)fs / 50.0) * 2 + 1, p->d_half_avg);
  if (cufft_ok(cufftExecD2Z(p->fwd_filters, p->d_filtered, p->d_filt_spec), "exec filters")) return -1;
  RYK_CUDA(cudaStreamSynchronize(e->stream));
  RYK_CUDA(cudaGetLastError());
  cufftDestroy(p->fwd_filters); p->fwd_filters = 0;
  *out = p;
  return 0;
}

// StoneMask refinement of `frames` f0 estimates.  Shared memory is sized for the largest FFT an f0 >= f0_floor can need (DIO and
// Harvest return no nonzero f0 below f0_floor), capped at the twiddle table's size.
int stonemask_run(Engine* e, const float* d_x, int n, int fs, double frame_period, double f0_floor, const double* d_f0_in,
                  double* d_f0_out, int frames, cudaStream_t st) {
  int fft_cap = stonemask_fft_size(fs, fmax(f0_floor, 40.0));
  if (fft_cap > kTwiddleN) fft_cap = kTwiddleN;
  k_stonemask<<<frames, 256, sizeof(double2) * 2 * fft_cap + 64, st>>>(d_x, n, fs, frame_period, d_f0_in, d_f0_out, e->d_twiddle, fft_cap);
  RYK_CUDA(cudaGetLastError());
  return 0;
}

// DIO + StoneMask: x (device float32, n samples) -> plan->d_f0r (double, f0_length frames). Stream-ordered, no sync.
int dio_stonemask_run(Engine* e, DioPlan* p, const float* d_x, cudaStream_t st) {
  if (p->harvest) {                                  // Harvest replaces DIO as the contour StoneMask refines
    if (harvest_run(e, p->harvest, d_x, p->d_f0, st)) return -1;
    return stonemask_run(e, d_x, p->n, p->fs, p->frame_period, p->f0_floor, p->d_f0, p->d_f0r, p->f0_length, st);
  }
  int nbins = p->fft_size / 2 + 1;
  if (cufft_ok(cufftSetStream(p->fwd, st), "set stream")) return -1;
  if (cufft_ok(cufftSetStream(p->inv, st), "set stream")) return -1;
  k_dio_prepare<<<1, 1024, 0, st>>>(d_x, p->n, p->y_length, p->fft_size, p->d_y);
  if (cufft_ok(cufftExecD2Z(p->fwd, p->d_y, p->d_Y), "exec D2Z")) return -1;
  k_cmul_inplace<<<(nbins + 255) / 256, 256, 0, st>>>(p->d_Y, p->d_filt_spec, nbins);
  k_band_mul<<<dim3((nbins + 255) / 256, p->nbands), 256, 0, st>>>(p->d_Y, p->d_filt_spec + nbins, p->d_Z, nbins);
  if (cufft_ok(cufftExecZ2D(p->inv, p->d_Z, p->d_filtered), "exec Z2D")) return -1;
  k_dio_zero_cross<<<dim3(4, p->nbands), 1024, 0, st>>>(p->d_filtered, p->fft_size, p->y_length, p->d_half_avg, 2, 0, (double)p->fs,
                                                      p->d_edges, p->d_loc, p->d_itv, p->d_counts);
  k_dio_candidates<<<dim3((p->f0_length + 127) / 128, p->nbands), 128, 0, st>>>(
      p->d_loc, p->d_itv, p->d_counts, p->y_length, p->f0_length, p->nbands, p->frame_period, p->f0_floor, p->f0_ceil,
      p->d_boundary, p->d_cand, p->d_score);
  k_dio_fix<<<1, 256, 0, st>>>(p->d_cand, p->d_score, p->nbands, p->f0_length, p->frame_period, p->f0_floor, p->d_scratch,
                               p->d_iscratch, p->d_f0);
  return stonemask_run(e, d_x, p->n, p->fs, p->frame_period, p->f0_floor, p->d_f0, p->d_f0r, p->f0_length, st);
}

const double* dio_plan_f0(DioPlan* p) { return p->d_f0r; }
int dio_plan_debug_copy(DioPlan* p, double* f0_raw, double* cand, double* score, int* counts, cudaStream_t st) {
  RYK_CUDA(cudaMemcpyAsync(f0_raw, p->d_f0, sizeof(double) * p->f0_length, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaMemcpyAsync(cand, p->d_cand, sizeof(double) * p->f0_length * p->nbands, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaMemcpyAsync(score, p->d_score, sizeof(double) * p->f0_length * p->nbands, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaMemcpyAsync(counts, p->d_counts, sizeof(int) * 4 * p->nbands, cudaMemcpyDeviceToHost, st));
  RYK_CUDA(cudaStreamSynchronize(st));
  return 0;
}
double* dio_plan_f0_mut(DioPlan* p) { return p->d_f0r; }
int dio_plan_frames(DioPlan* p) { return p->f0_length; }
HarvestPlan* dio_plan_harvest(DioPlan* p) { return p->harvest; }
const double* dio_plan_f0_raw(DioPlan* p) { return p->d_f0; }

size_t cheaptrick_smem_bytes(int fft_size, int fs) {
  int nb = fft_size / 2 + 1;
  return sizeof(double2) * fft_size + sizeof(double) * ((nb + 1) + ct_seg_len(fft_size, fs) + 256 + 64);
}

size_t d4c_smem_bytes(int fs) {
  int fft_d4c = (int)pow(2.0, 1.0 + (int)(log(4.0 * fs / 47.0 + 1) / kLog2));
  int lt_fft = (int)pow(2.0, 1.0 + (int)(log(3.0 * fs / 40.0 + 1) / kLog2));
  int maxfft = fft_d4c > lt_fft ? fft_d4c : lt_fft;
  int hb = fft_d4c / 2 + 1;
  int nap = (int)(fmin(15000.0, fs / 2.0 - 3000.0) / 3000.0);
  return sizeof(double2) * maxfft + sizeof(double) * (6 * (hb + 8) + d4c_seg_len(fft_d4c, fs) + 24 + 512 + 64) +
         16 + sizeof(int) * 3 * nap * 256;
}

int analysis_kernels_init() {
  RYK_CUDA(cudaFuncSetAttribute(k_stonemask, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * kTwiddleN * (int)sizeof(double2) + 64));
  RYK_CUDA(cudaFuncSetAttribute(k_cheaptrick, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  RYK_CUDA(cudaFuncSetAttribute(k_d4c, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  return 0;
}

// CheapTrick(+sp2mc) and D4C on the refined f0 in d_f0 (double, >= n_out frames). Stream-ordered.
int spectral_analysis_run(Engine* e, const float* d_x, int n, int fs, double frame_period, const double* d_f0, int n_out,
                          int fft_size, int order, float* d_sp, float* d_ap, float* d_mc, float* d_f0_out, uint8_t* d_voiced,
                          cudaStream_t st) {
  RYK_CHECK(fft_size <= kCtMaxFft && fft_size >= 64, "unsupported CheapTrick fft size");
  RYK_CHECK(e->d_G != nullptr && e->G_order == order && e->G_fft == fft_size, "sp2mc matrix not prepared for this (order, fft)");
  if (n_out <= 0) return 0;
  k_cheaptrick<<<n_out, 256, cheaptrick_smem_bytes(fft_size, fs), st>>>(d_x, n, fs, frame_period, d_f0, fft_size, -0.15, e->d_G, order,
                                                                      n_out, d_sp, d_mc, nullptr, e->d_twiddle);
  const int fft_d4c = (int)pow(2.0, 1.0 + (int)(log(4.0 * fs / 47.0 + 1) / kLog2));   // host pow: exact
  const int lt_fft = (int)pow(2.0, 1.0 + (int)(log(3.0 * fs / 40.0 + 1) / kLog2));
#ifdef RYK_D4C_TIMELINE
  { unsigned long long* tl_ = nullptr; cudaGetSymbolAddress((void**)&tl_, g_d4c_tl); cudaMemsetAsync(tl_, 0, sizeof(g_d4c_tl), st); }
#endif
  k_d4c<<<n_out, 512, d4c_smem_bytes(fs), st>>>(d_x, n, fs, frame_period, d_f0, fft_size, 0.85, n_out, d_ap, e->d_twiddle, fft_d4c, lt_fft);
#ifdef RYK_D4C_TIMELINE
  cudaStreamCaptureStatus cap_ = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(st, &cap_);
  if (const char* path = cap_ == cudaStreamCaptureStatusNone ? getenv("RYK_D4C_TIMELINE_FILE") : nullptr) {
    cudaStreamSynchronize(st);
    static std::vector<unsigned long long> h(kD4cTlMaxCtas * kD4cTlSlots);
    cudaMemcpyFromSymbol(h.data(), g_d4c_tl, sizeof(unsigned long long) * h.size());
    if (FILE* f = fopen(path, "a")) {
      fprintf(f, "# launch: %d frames, slots 0..%d\n", n_out, kD4cTlSlots - 1);
      for (int c = 0; c < n_out && c < kD4cTlMaxCtas; ++c) { for (int k = 0; k < kD4cTlSlots; ++k) fprintf(f, "%llu ", h[c * kD4cTlSlots + k]); fprintf(f, "\n"); }
      fclose(f);
    }
  }
#endif
  k_f0_out<<<(n_out + 127) / 128, 128, 0, st>>>(d_f0, n_out, d_f0_out, d_voiced);
  RYK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ryk
