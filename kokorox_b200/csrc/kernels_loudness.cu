// kernels_loudness.cu -- loudness normalisation (K14): ITU-R BS.1770 integrated loudness of each utterance's 24 kHz
// waveform, its true peak, and the static gain that brings it to the session's target under a true-peak ceiling
// (kkx.h "loudness_target" / "true_peak_max"), the lookahead true-peak limiter (kkx.h "limiter") and the EBU R128
// loudness range and maxima (kkx.h "loudness_report", at the end of this file).  The gains themselves are applied by
// resample_kernel (kernels_signal.cu).
//
// Per item (n samples x at 24 kHz):
//   loud_energy  one thread per 2400-sample segment s (the 100 ms hop): the K-weighting cascade (shelf, then
//                high-pass) runs from zero state over x[max(0, 2400 s - 4800), 2400 (s + 1)) and the sum of squares of
//                its last 2400 outputs is the segment's energy.  The slowest pole has radius 0.99007, so after 4800
//                samples the dropped history weighs 0.99007^4800 ~ 1e-21: the value is the one the filter would have
//                run serially from the item's first sample, to fp32 rounding.  A serial filter over a 510-token item
//                (~7e5 samples) would be one long dependency chain; here it is n / 2400 chains of 7200 steps.
//   loud_peak    the 4x polyphase FIR of resample_poly(x, 4, 1) (scipy's default Kaiser filter, zeros outside the
//                item), one input position (4 outputs) per thread; max |y| of the item through an integer atomicMax on
//                the float's bits (non-negative floats order like their bit patterns: exact and order-independent).
//   loud_gain    one CTA per item: block j (400 ms = segments j .. j + 3) has z_j = sum of its 4 energies / 9600,
//                l_j = -0.691 + 10 log10 z_j; the absolute gate (l_j > -70) and the relative gate (l_j > Gamma_r)
//                follow BS.1770-4; sums in double in a fixed order; L, dBTP and the gain are written per item.
// Every value is a function of the item's samples alone: an item gets the same bits in any batch, frame group or pass.
#include "kernels.h"
#include <math.h>
#include <cmath>
#include <vector>

namespace kkx {

// K-weighting as libebur128 designs it (analog prototypes through the bilinear transform, K = tan(pi f0 / fs)); at
// fs = 48000 these are the BS.1770-4 table's coefficients.
void loudness_design(double fs, double kw[10], std::vector<float>* tp_taps) {
  {   // stage 1: high shelf
    const double f0 = 1681.974450955533, G = 3.999843853973347, Q = 0.7071752369554196;
    const double K = std::tan(M_PI * f0 / fs);
    const double Vh = std::pow(10.0, G / 20.0), Vb = std::pow(Vh, 0.4996667741545416);
    const double a0 = 1.0 + K / Q + K * K;
    kw[0] = (Vh + Vb * K / Q + K * K) / a0;
    kw[1] = 2.0 * (K * K - Vh) / a0;
    kw[2] = (Vh - Vb * K / Q + K * K) / a0;
    kw[3] = 2.0 * (K * K - 1.0) / a0;
    kw[4] = (1.0 - K / Q + K * K) / a0;
  }
  {   // stage 2: high-pass (RLB); numerator 1, -2, 1 as in the standard's table
    const double f0 = 38.13547087602444, Q = 0.5003270373238773;
    const double K = std::tan(M_PI * f0 / fs);
    const double a0 = 1.0 + K / Q + K * K;
    kw[5] = 1.0; kw[6] = -2.0; kw[7] = 1.0;
    kw[8] = 2.0 * (K * K - 1.0) / a0;
    kw[9] = (1.0 - K / Q + K * K) / a0;
  }
  if (tp_taps) poly_design(4, 1, tp_taps);   // 4 * firwin(81, 1/4, ("kaiser", 5.0))
}

LoudParams loudness_params(double target_lufs, double ceiling_dbtp, bool limiter, bool report) {
  LoudParams P{};
  double kw[10];
  std::vector<float> taps;
  loudness_design(24000.0, kw, &taps);
  if ((int)taps.size() != kTpTaps) throw ArgError("loudness: unexpected true-peak filter length");
  for (int i = 0; i < 10; i++) P.kw[i] = (float)kw[i];
  for (int i = 0; i < kTpTaps; i++) P.tp[i] = taps[i];
  P.target_lufs = target_lufs;
  P.ceiling_dbtp = ceiling_dbtp;
  // a limiter or report session may run without a loudness target (report alone: measure-only, g = 1, no cap)
  P.normalise = limiter || report ? target_lufs != 0.0 : 1;
  P.limiter = limiter ? 1 : 0;
  return P;
}

// ------------------------------------------------------------------------------------------ segment energies
constexpr int kLeThreads = 128;

// one K-weighting step (transposed direct form II, fp32 FMA in a fixed order); returns the high-pass output
__device__ __forceinline__ float kweight_step(const LoudParams& P, float x, float& s1, float& s2, float& t1, float& t2) {
  const float u = fmaf(P.kw[0], x, s1);
  s1 = fmaf(P.kw[1], x, fmaf(-P.kw[3], u, s2));
  s2 = fmaf(P.kw[2], x, -P.kw[4] * u);
  const float y = fmaf(P.kw[5], u, t1);
  t1 = fmaf(P.kw[6], u, fmaf(-P.kw[8], y, t2));
  t2 = fmaf(P.kw[7], u, -P.kw[9] * y);
  return y;
}

__global__ void __launch_bounds__(kLeThreads) loud_energy_kernel(const float* __restrict__ x,
                                                                 const long long* __restrict__ in_off,
                                                                 const long long* __restrict__ in_len,
                                                                 const long long* __restrict__ seg_off, LoudParams P,
                                                                 float* __restrict__ energy, unsigned* __restrict__ peak) {
  const int b = blockIdx.y;
  if (blockIdx.x == 0 && threadIdx.x == 0) peak[b] = 0u;   // loud_peak (the next launch) accumulates into it
  const long long nseg = in_len[b] / kLoudSeg;
  const long long s = (long long)blockIdx.x * kLeThreads + threadIdx.x;
  if (s >= nseg) return;
  const float* xb = x + in_off[b];
  const long long e0 = s * kLoudSeg;
  const long long start = e0 > kLoudWarm ? e0 - kLoudWarm : 0;
  float s1 = 0.f, s2 = 0.f, t1 = 0.f, t2 = 0.f;
  for (long long i = start; i < e0; i += 8) {   // warm-up: state only (lengths are multiples of 2400)
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = __ldg(xb + i + k);
#pragma unroll
    for (int k = 0; k < 8; k++) kweight_step(P, v[k], s1, s2, t1, t2);
  }
  float acc = 0.f;
  for (long long i = e0; i < e0 + kLoudSeg; i += 8) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = __ldg(xb + i + k);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const float y = kweight_step(P, v[k], s1, s2, t1, t2);
      acc = fmaf(y, y, acc);
    }
  }
  energy[seg_off[b] + s] = acc;
}

// ------------------------------------------------------------------------------------------ true peak
// y[4q + p] = sum over k of x[k] h[4 (q - k) + p + 40], 0 <= 4 (q - k) + p + 40 <= 80: inputs q - 10 .. q + 10.
constexpr int kTpThreads = 256, kTpPer = 4, kTpTile = kTpThreads * kTpPer, kTpHalo = 10;

__global__ void __launch_bounds__(kTpThreads) loud_peak_kernel(const float* __restrict__ x,
                                                               const long long* __restrict__ in_off,
                                                               const long long* __restrict__ in_len, LoudParams P,
                                                               unsigned* __restrict__ peak, float* __restrict__ pmax) {
  __shared__ float s_x[kTpTile + 2 * kTpHalo];
  const int b = blockIdx.y, t = threadIdx.x;
  const long long n = in_len[b];
  const long long q0 = (long long)blockIdx.x * kTpTile;
  if (q0 >= n) return;
  const float* xb = x + in_off[b];
  for (int i = t; i < kTpTile + 2 * kTpHalo; i += kTpThreads) {
    const long long k = q0 - kTpHalo + i;
    s_x[i] = (k >= 0 && k < n) ? __ldg(xb + k) : 0.f;
  }
  __syncthreads();
  float m = 0.f;
#pragma unroll
  for (int i = 0; i < kTpPer; i++) {
    const int r = t + i * kTpThreads;
    if (q0 + r >= n) break;
    const float* w = s_x + r + kTpHalo;   // w[d] = x[q + d]
    float mq = 0.f;
#pragma unroll
    for (int p = 0; p < 4; p++) {
      float acc = 0.f;
#pragma unroll
      for (int d = -kTpHalo; d <= kTpHalo; d++) {   // k = q + d ascending: tap 40 + p - 4 d
        const int j = 40 + p - 4 * d;
        if (j >= 0 && j < kTpTaps) acc = fmaf(w[d], P.tp[j], acc);
      }
      mq = fmaxf(mq, fabsf(acc));
    }
    if (pmax) pmax[in_off[b] + q0 + r] = mq;   // the limiter's detector p[q]
    m = fmaxf(m, mq);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((t & 31) == 0 && m > 0.f) atomicMax(peak + b, __float_as_uint(m));
}

// ------------------------------------------------------------------------------------------ gating and gain
constexpr int kLgThreads = 256;

template <class T>
__device__ T block_sum(T v, T* red) {   // fixed-shape tree: the result depends on the thread values alone
  const int t = threadIdx.x;
  __syncthreads();
  red[t] = v;
  __syncthreads();
  for (int h = kLgThreads / 2; h > 0; h >>= 1) {
    if (t < h) red[t] += red[t + h];
    __syncthreads();
  }
  return red[0];
}

__global__ void __launch_bounds__(kLgThreads) loud_gain_kernel(const long long* __restrict__ in_len,
                                                               const long long* __restrict__ seg_off,
                                                               const float* __restrict__ energy,
                                                               const unsigned* __restrict__ peak, LoudParams P,
                                                               float* __restrict__ lufs, float* __restrict__ tp_db,
                                                               float* __restrict__ gain) {
  __shared__ double red_d[kLgThreads];
  __shared__ long long red_n[kLgThreads];
  const int b = blockIdx.x, t = threadIdx.x;
  const long long nblk = in_len[b] / kLoudSeg - 3;          // whole 400 ms blocks (<= 0: none)
  const float* e = energy + seg_off[b];
  auto level = [&](long long j, double* z) {
    *z = ((double)e[j] + (double)e[j + 1] + (double)e[j + 2] + (double)e[j + 3]) / (4.0 * kLoudSeg);
    return -0.691 + 10.0 * log10(*z);                       // z = 0: -inf, gated out
  };
  double s = 0.0;
  long long c = 0;
  for (long long j = t; j < nblk; j += kLgThreads) {
    double z;
    if (level(j, &z) > -70.0) { s += z; c++; }
  }
  const double s1 = block_sum(s, red_d);
  const long long c1 = block_sum(c, red_n);
  double L = NAN;
  if (c1 > 0) {
    const double rel = -0.691 + 10.0 * log10(s1 / (double)c1) - 10.0;
    s = 0.0; c = 0;
    for (long long j = t; j < nblk; j += kLgThreads) {
      double z;
      const double l = level(j, &z);
      if (l > -70.0 && l > rel) { s += z; c++; }
    }
    const double s2 = block_sum(s, red_d);
    const long long c2 = block_sum(c, red_n);
    if (c2 > 0) L = -0.691 + 10.0 * log10(s2 / (double)c2);
  }
  if (t != 0) return;
  const float tp = __uint_as_float(peak[b]);
  double g = 1.0;
  if (P.normalise && !isnan(L)) g = pow(10.0, (P.target_lufs - L) / 20.0);
  // rule 5's cap (not when measuring only); the limiter's sits Rmax higher and always applies (kkx.h "limiter")
  if (P.limiter || (P.normalise && !isnan(L))) {
    const double cap = pow(10.0, (P.ceiling_dbtp + (P.limiter ? kLimRmax : 0.0)) / 20.0);
    if ((double)tp * g > cap) g = cap / (double)tp;
  }
  lufs[b] = (float)L;
  tp_db[b] = (float)(20.0 * log10((double)tp));
  gain[b] = (float)g;
}

void launch_loudness(const float* x, const long long* in_off, const long long* in_len, const long long* seg_off,
                     const LoudParams& P, float* energy, unsigned* peak, float* lufs, float* tp_db, float* gain, int B,
                     long long max_len, cudaStream_t st, float* pmax) {
  if (g_dry_run) return;
  if (B < 1 || B > 65535) throw ArgError("launch_loudness: batch out of range");
  const long long max_seg = max_len / kLoudSeg;
  const long long ge = std::max(1LL, (max_seg + kLeThreads - 1) / kLeThreads);
  const long long gp = std::max(1LL, (max_len + kTpTile - 1) / kTpTile);
  if (gp > 0x7FFFFFFFLL) throw ArgError("launch_loudness: grid too large");
  loud_energy_kernel<<<dim3((unsigned)ge, B), kLeThreads, 0, st>>>(x, in_off, in_len, seg_off, P, energy, peak);
  post_launch("loud_energy", st);
  loud_peak_kernel<<<dim3((unsigned)gp, B), kTpThreads, 0, st>>>(x, in_off, in_len, P, peak, pmax);
  post_launch("loud_peak", st);
  loud_gain_kernel<<<B, kLgThreads, 0, st>>>(in_len, seg_off, energy, peak, P, lufs, tp_db, gain);
  post_launch("loud_gain", st);
}

// ------------------------------------------------------------------------------------------ lookahead limiter
// kkx.h "limiter", steps 2-7.  lim_envelope: one CTA per tile of kLimTile output samples of one item, anchored at the
// item's sample 0; it stages the detector p (loud_peak's pmax) over the tile plus the reach of the rule -- Ha + W + Hb
// samples to the left (box, release, hold), Ha + Hb to the right -- and computes in shared memory
//   q  the required reduction (dB) per sample, 0 outside the item;
//   h  the hold, a sliding minimum of q over Ha + 2 Hb + 1 samples, by doubling (min over 2, 4, .., 128, then two
//      overlapping 128-windows);
//   e  the release, min(0, r s + prefix-min over m <= r of (h[m] - m s)) with tile-relative r: terms older than W
//      are >= 0 (h >= -Rmax), so the prefix from the tile's left edge gives the windowed minimum of the rule;
//   G  the mean of 10^(e / 20) over Ha + 1 samples, as 1 - (window sum of the deficits 1 - 10^(e / 20)) / (Ha + 1);
//      the deficits are summed as 2^25-scaled integers (a prefix sum modulo 2^32; the window sum is < 121 * 2^25 <
//      2^32), so the sum is exact and independent of the scan's order, and a window of zero deficits gives G = 1.0.
// Every value is a function of the item and the tile's position in it: an item's bits do not depend on its batch.
// v = fp32(x fp32(g G)); the largest window deficit of the item (i.e. its smallest G) goes through an integer
// atomicMax.  loud_peak then measures v, and lim_trim turns that into t and the report.
constexpr int kLimThreads = 512, kLimTile = 8192;
constexpr int kLimL = kLimHa + kLimW + kLimHb;                  // q starts L samples left of the tile
constexpr int kLimSq = kLimTile + kLimL + kLimHa + kLimHb;      // q over [-L, T + Ha + Hb)
constexpr int kLimSh = kLimTile + kLimHa + kLimW;               // h over [-Ha - W, T)
constexpr int kLimSd = kLimTile + kLimHa;                       // deficits over [-Ha, T)
constexpr int kLimHold = kLimHa + 2 * kLimHb + 1;               // 141-sample hold window
constexpr float kLimS = (float)kLimSlope;
constexpr float kLimDefScale = 33554432.f;                      // 2^25
constexpr float kLimBoxScale = 1.f / ((kLimHa + 1) * 33554432.f);
static_assert(kLimHold > 128 && kLimHold <= 256, "the hold combines two 128-sample windows");
static_assert((double)(kLimHa + 1) * 33554432.0 < 4294967296.0, "window sum of the scaled deficits must fit 32 bits");

__device__ __forceinline__ float lim_gain_of(unsigned w) {   // G of a window sum of scaled deficits
  return __fsub_rn(1.f, __fmul_rn(__uint2float_rn(w), kLimBoxScale));
}

// inclusive scan of a[0 .. S) in shared memory with an exact, associative and commutative op (min, modular add);
// contiguous runs per thread, then the run totals across the block
template <class T, class Op>
__device__ void lim_scan(T* a, int S, T id, Op op, T* wt) {
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int c = (S + kLimThreads - 1) / kLimThreads;
  const int lo = min(t * c, S), hi = min(lo + c, S);
  T acc = id;
  for (int j = lo; j < hi; j++) { acc = op(acc, a[j]); a[j] = acc; }
  T v = acc;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const T u = __shfl_up_sync(0xffffffffu, v, o);
    if (lane >= o) v = op(u, v);
  }
  if (lane == 31) wt[wid] = v;
  __syncthreads();
  if (wid == 0) {
    T w = lane < kLimThreads / 32 ? wt[lane] : id;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const T u = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w = op(u, w);
    }
    if (lane < kLimThreads / 32) wt[lane] = w;
  }
  __syncthreads();
  T ex = __shfl_up_sync(0xffffffffu, v, 1);
  if (lane == 0) ex = id;
  const T carry = wid > 0 ? op(wt[wid - 1], ex) : ex;
  for (int j = lo; j < hi; j++) a[j] = op(carry, a[j]);
  __syncthreads();
}

struct LimMin { __device__ float operator()(float a, float b) const { return fminf(a, b); } };
struct LimAdd { __device__ unsigned operator()(unsigned a, unsigned b) const { return a + b; } };

__global__ void __launch_bounds__(kLimThreads) lim_envelope_kernel(const float* __restrict__ x,
                                                                   const float* __restrict__ pmax,
                                                                   const long long* __restrict__ in_off,
                                                                   const long long* __restrict__ in_len, float C,
                                                                   const float* __restrict__ gain,
                                                                   float* __restrict__ v, float* __restrict__ G,
                                                                   unsigned* __restrict__ acc) {
  extern __shared__ float lim_smem[];
  __shared__ float wtf[kLimThreads / 32];
  __shared__ unsigned wtu[kLimThreads / 32];
  float* fa = lim_smem;
  float* fb = lim_smem + kLimSq;
  const int b = blockIdx.y, t = threadIdx.x;
  const long long n = in_len[b];
  const long long i0 = (long long)blockIdx.x * kLimTile;
  if (i0 >= n) return;
  const long long off = in_off[b];
  const float g = gain[b];
  // step 2: q[j] at sample i0 - L + j
  for (int j = t; j < kLimSq; j += kLimThreads) {
    const long long i = i0 - kLimL + j;
    const float p = (i >= 0 && i < n) ? __ldg(pmax + off + i) : 0.f;
    fa[j] = p > 0.f ? fminf(0.f, C - 20.f * log10f(g * p)) : 0.f;
  }
  __syncthreads();
  // step 3: after the doubling passes src[j] = min of q over [j, j + 127]; h[j] (sample i0 - Ha - W + j) = min of q
  // over [j, j + Ha + 2 Hb], i.e. over samples [i - Hb, i + Ha + Hb]
  float* src = fa;
  float* dst = fb;
  for (int d = 1; d < 128; d <<= 1) {
    for (int j = t; j < kLimSq; j += kLimThreads) dst[j] = j + d < kLimSq ? fminf(src[j], src[j + d]) : src[j];
    __syncthreads();
    float* tmp = src; src = dst; dst = tmp;
  }
  float* h = dst;
  for (int j = t; j < kLimSh; j += kLimThreads)
    h[j] = __fsub_rn(fminf(src[j], src[j + kLimHold - 128]), __fmul_rn((float)(j - kLimHa - kLimW), kLimS));
  __syncthreads();
  // step 4: prefix minimum of h[m] - m s (tile-relative m), then e[r] = min(0, r s + that)
  lim_scan(h, kLimSh, INFINITY, LimMin(), wtf);
  unsigned* du = reinterpret_cast<unsigned*>(src);   // src is free now
  for (int j = t; j < kLimSd; j += kLimThreads) {
    const int r = j - kLimHa;
    float e = fminf(0.f, __fadd_rn(__fmul_rn((float)r, kLimS), h[r + kLimHa + kLimW]));
    if (i0 + r < 0) e = 0.f;   // e = 0 before the item's first sample
    du[j] = __float2uint_rn(__fmul_rn(__fsub_rn(1.f, exp10f(0.05f * e)), kLimDefScale));
  }
  __syncthreads();
  // step 5: window sums of the deficits over [r - Ha, r] (exact modulo 2^32); step 6: v
  lim_scan(du, kLimSd, 0u, LimAdd(), wtu);
  unsigned wmax = 0u;
  for (int r = t; r < kLimTile; r += kLimThreads) {
    const long long i = i0 + r;
    if (i >= n) break;
    const unsigned w = du[r + kLimHa] - (r > 0 ? du[r - 1] : 0u);
    const float Gi = lim_gain_of(w);
    v[off + i] = __fmul_rn(__ldg(x + off + i), __fmul_rn(g, Gi));
    if (G) G[off + i] = Gi;
    wmax = max(wmax, w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  if ((t & 31) == 0 && wmax > 0u) atomicMax(acc + gridDim.y + b, wmax);
}

// step 7 and the report, one thread per item: acc[b] = bits of v's true peak, acc[B + b] = largest window deficit
__global__ void lim_trim_kernel(const unsigned* __restrict__ acc, double ceiling_dbtp, int B, float* __restrict__ t,
                                float* __restrict__ red_db, float* __restrict__ out_db) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const double c = pow(10.0, ceiling_dbtp / 20.0);
  const float tpv = __uint_as_float(acc[b]);
  const float tb = (double)tpv > c ? (float)(c / (double)tpv) : 1.f;
  const float gmin = lim_gain_of(acc[B + b]);
  t[b] = tb;
  red_db[b] = (float)(0.0 - 20.0 * log10((double)tb * (double)gmin));
  out_db[b] = (float)(20.0 * log10((double)tb * (double)tpv));
}

size_t lim_smem_bytes() { return (size_t)2 * kLimSq * sizeof(float); }

void launch_limiter(const float* x, const float* pmax, const long long* in_off, const long long* in_len,
                    const LoudParams& P, const float* gain, float* v, float* G, unsigned* acc, float* t, float* red_db,
                    float* out_db, int B, long long max_len, cudaStream_t st) {
  if (g_dry_run) return;
  if (B < 1 || B > 65535) throw ArgError("launch_limiter: batch out of range");
  const long long tiles = std::max(1LL, (max_len + kLimTile - 1) / kLimTile);
  const long long gp = std::max(1LL, (max_len + kTpTile - 1) / kTpTile);
  if (gp > 0x7FFFFFFFLL) throw ArgError("launch_limiter: grid too large");
  const int smem = (int)lim_smem_bytes();
  prepare_smem_launch<lim_envelope_kernel>(smem);
  KKX_CUDA(cudaMemsetAsync(acc, 0, (size_t)2 * B * sizeof(unsigned), st));
  lim_envelope_kernel<<<dim3((unsigned)tiles, B), kLimThreads, smem, st>>>(x, pmax, in_off, in_len,
                                                                            (float)P.ceiling_dbtp, gain, v, G, acc);
  post_launch("lim_envelope", st);
  loud_peak_kernel<<<dim3((unsigned)gp, B), kTpThreads, 0, st>>>(v, in_off, in_len, P, acc, nullptr);
  post_launch("loud_peak", st);
  lim_trim_kernel<<<(B + 127) / 128, 128, 0, st>>>(acc, P.ceiling_dbtp, B, t, red_db, out_db);
  post_launch("lim_trim", st);
}

// ------------------------------------------------------------------------------------------ loudness range, maxima
// kkx.h "loudness_report" / kkx_last_loudness_range (EBU Tech 3341 / 3342), on loud_energy's segment energies e_i.
//   loud_short  one thread per 3 s window j (segments j .. j + 29 on the 100 ms hop): s_j = the 30 energies summed in
//               double in ascending i, / 72000; written to st at the item's seg_off, like the energies.
//   loud_range  one CTA per item: max z_j (z as loud_gain forms it) and max s_j by fixed-shape reductions (max is
//               exact); the absolute and relative gates with block_sum; then the order statistics a_lo and a_hi of the
//               gated s_j by an MSD radix select on their 64-bit patterns (non-negative doubles order like their
//               bits): 8 passes of 8-bit digits, each counting the candidates of both ranks into two 256-bin shared
//               histograms, after which one warp per rank picks the digit.  Counts are exact, so the result does not
//               depend on the order in which windows are visited, and the shared memory is fixed whatever the number
//               of windows (tens of thousands for a long program).
constexpr int kStSegs = 30;   // segments per 3 s window

__global__ void __launch_bounds__(kLeThreads) loud_short_kernel(const long long* __restrict__ in_len,
                                                                const long long* __restrict__ seg_off,
                                                                const float* __restrict__ energy,
                                                                double* __restrict__ st) {
  const int b = blockIdx.y;
  const long long nwin = in_len[b] / kLoudSeg - (kStSegs - 1);
  const long long j = (long long)blockIdx.x * kLeThreads + threadIdx.x;
  if (j >= nwin) return;
  const float* e = energy + seg_off[b] + j;
  double s = (double)__ldg(e);
#pragma unroll
  for (int i = 1; i < kStSegs; i++) s += (double)__ldg(e + i);
  st[seg_off[b] + j] = s / (double)(kStSegs * kLoudSeg);
}

__device__ double block_max(double v, double* red) {   // fixed-shape tree, like block_sum
  const int t = threadIdx.x;
  __syncthreads();
  red[t] = v;
  __syncthreads();
  for (int h = kLgThreads / 2; h > 0; h >>= 1) {
    if (t < h) red[t] = fmax(red[t], red[t + h]);
    __syncthreads();
  }
  return red[0];
}

__global__ void __launch_bounds__(kLgThreads) loud_range_kernel(const long long* __restrict__ in_len,
                                                                const long long* __restrict__ seg_off,
                                                                const float* __restrict__ energy,
                                                                const double* __restrict__ st,
                                                                float* __restrict__ lra, float* __restrict__ m_max,
                                                                float* __restrict__ s_max) {
  __shared__ double red_d[kLgThreads];
  __shared__ long long red_n[kLgThreads];
  __shared__ unsigned hist[2][256];
  __shared__ unsigned long long pre[2];   // the decided high bits of a_lo, a_hi
  __shared__ unsigned rank[2];            // their ranks among the candidates that share those bits
  const int b = blockIdx.x, t = threadIdx.x;
  const long long nseg = in_len[b] / kLoudSeg;
  const long long nblk = nseg - 3, nwin = nseg - (kStSegs - 1);   // whole 400 ms blocks, whole 3 s windows
  const float* e = energy + seg_off[b];
  const double* s = st + seg_off[b];
  // maxima: z, s >= 0, so 0 is the identity; an all-silent item gives 0 and -inf LUFS
  double zm = 0.0, sm = 0.0;
  for (long long j = t; j < nblk; j += kLgThreads)
    zm = fmax(zm, ((double)e[j] + (double)e[j + 1] + (double)e[j + 2] + (double)e[j + 3]) / (4.0 * kLoudSeg));
  for (long long j = t; j < nwin; j += kLgThreads) sm = fmax(sm, s[j]);
  zm = block_max(zm, red_d);
  sm = block_max(sm, red_d);
  double range = NAN;
  if (nwin > 0) {
    // EBU Tech 3342 gates: absolute l_s > -70, relative l_s > -0.691 + 10 log10(mean s) - 20 (strict)
    auto level = [](double v) { return -0.691 + 10.0 * log10(v); };   // v = 0: -inf, gated out
    double sa = 0.0;
    long long ca = 0;
    for (long long j = t; j < nwin; j += kLgThreads)
      if (level(s[j]) > -70.0) { sa += s[j]; ca++; }
    const double s1 = block_sum(sa, red_d);
    const long long c1 = block_sum(ca, red_n);
    if (c1 > 0) {
      const double rel = level(s1 / (double)c1) - 20.0;
      auto gated = [&](double v) { const double l = level(v); return l > -70.0 && l > rel; };
      long long cm = 0;
      for (long long j = t; j < nwin; j += kLgThreads) cm += gated(s[j]) ? 1 : 0;
      const long long m = block_sum(cm, red_n);
      if (m > 0) {
        // nearest rank of the 10 % and 95 % points, halves rounded up
        if (t < 2) {
          pre[t] = 0ull;
          rank[t] = (unsigned)(((t == 0 ? 10 : 95) * (m - 1) + 50) / 100);
        }
        for (int pass = 0; pass < 8; pass++) {
          const int shift = 56 - 8 * pass;
          const unsigned long long mask = pass == 0 ? 0ull : ~0ull << (shift + 8);
          for (int i = t; i < 2 * 256; i += kLgThreads) (&hist[0][0])[i] = 0u;
          __syncthreads();
          const unsigned long long p0 = pre[0], p1 = pre[1];
          for (long long j = t; j < nwin; j += kLgThreads) {
            const double v = s[j];
            if (!gated(v)) continue;
            const unsigned long long u = (unsigned long long)__double_as_longlong(v);
            const unsigned d = (unsigned)(u >> shift) & 255u;
            if ((u & mask) == p0) atomicAdd(&hist[0][d], 1u);
            if ((u & mask) == p1) atomicAdd(&hist[1][d], 1u);
          }
          __syncthreads();
          if (t < 64) {   // warp w: the bin in which rank[w] falls, 8 bins per lane, a warp scan of the lane totals
            const int w = t >> 5, lane = t & 31;
            unsigned c[8], tot = 0u;
#pragma unroll
            for (int k = 0; k < 8; k++) { c[k] = hist[w][lane * 8 + k]; tot += c[k]; }
            unsigned inc = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
              const unsigned u = __shfl_up_sync(0xffffffffu, inc, o);
              if (lane >= o) inc += u;
            }
            const unsigned r = rank[w];
            unsigned below = inc - tot;
            if (r >= below && r < inc) {   // exactly one lane
#pragma unroll
              for (int k = 0; k < 8; k++) {
                if (r < below + c[k]) {
                  rank[w] = r - below;
                  pre[w] |= (unsigned long long)(lane * 8 + k) << shift;
                  break;
                }
                below += c[k];
              }
            }
          }
          __syncthreads();
        }
        range = 10.0 * log10(__longlong_as_double((long long)pre[1]) / __longlong_as_double((long long)pre[0]));
      }
    }
  }
  if (t != 0) return;
  lra[b] = (float)range;
  m_max[b] = nblk > 0 ? (float)(-0.691 + 10.0 * log10(zm)) : NAN;
  s_max[b] = nwin > 0 ? (float)(-0.691 + 10.0 * log10(sm)) : NAN;
}

void launch_loudness_range(const long long* in_len, const long long* seg_off, const float* energy, double* st,
                           float* lra, float* m_max, float* s_max, int B, long long max_len, cudaStream_t stream) {
  if (g_dry_run) return;
  if (B < 1 || B > 65535) throw ArgError("launch_loudness_range: batch out of range");
  const long long max_seg = max_len / kLoudSeg;
  const long long ge = std::max(1LL, (max_seg + kLeThreads - 1) / kLeThreads);
  loud_short_kernel<<<dim3((unsigned)ge, B), kLeThreads, 0, stream>>>(in_len, seg_off, energy, st);
  post_launch("loud_short", stream);
  loud_range_kernel<<<B, kLgThreads, 0, stream>>>(in_len, seg_off, energy, st, lra, m_max, s_max);
  post_launch("loud_range", stream);
}

}  // namespace kkx
