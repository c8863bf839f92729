// kernels_signal.cu -- HBM-bound kernels: instance-norm statistics, duration head + exact
// integer length regulation (K4/K5), harmonic source (K9), STFT (K10), iSTFT head (K11), output resampling.
#include "kernels.h"
#include <cuda_bf16.h>
#include <math.h>
#include <algorithm>
#include <cmath>
#include <numeric>
#include <vector>

namespace kkx {

// ------------------------------------------------------------------------------------------
// InstanceNorm statistics: per (item, chunk of kStatRows rows) column sums and sums of squares.
// part layout: [B][nchunk][2][C] with nchunk = ceil(max_len / kStatRows).
// Block = 256 threads = XT column-quads x YT row slices (float4 loads when C % 4 == 0); the row
// slices are combined through shared memory in a fixed order (deterministic).
// ADD: the statistics are those of x + y, and the sum is also stored to `out` (same row pitch): the generator's
// `x = ups(x) + x_source` add and the first AdaIN's statistics pass in one sweep.
template <int VEC, bool ADD>
__global__ void __launch_bounds__(256) colstats_kernel(const float* __restrict__ x, int ldx, int C,
                                                       float* __restrict__ part, int nchunk,
                                                       const int* off, const int* len,
                                                       const float* __restrict__ y, float* __restrict__ out,
                                                       __nv_bfloat16* __restrict__ out_b) {
  __shared__ float red[2][256 * VEC];
  const int b = blockIdx.y, ch = blockIdx.x;
  const int L = len[b];
  const int r0 = ch * kStatRows;
  if (r0 >= L) return;
  const int r1 = min(L, r0 + kStatRows);
  const int CV = (C + VEC - 1) / VEC;           // column groups
  const int XT = CV < 256 ? CV : 256;           // threads along columns (CV is 32 / 64 / 128+ here)
  const int YT = 256 / XT;                      // row slices
  const int tx = threadIdx.x % XT, ty = threadIdx.x / XT;
  float* pp = part + ((size_t)b * nchunk + ch) * 2 * C;
  for (int cg0 = 0; cg0 < CV; cg0 += XT) {
    const int cg = cg0 + tx;
    float s[VEC], q[VEC];
#pragma unroll
    for (int v = 0; v < VEC; v++) { s[v] = 0.f; q[v] = 0.f; }
    if (cg < CV && ty < YT) {
      const float* p = x + (size_t)(off[b] + r0 + ty) * ldx + cg * VEC;
      for (int r = r0 + ty; r < r1; r += YT, p += (size_t)YT * ldx) {
        if (VEC == 4) {
          float4 v4 = *reinterpret_cast<const float4*>(p);
          if (ADD) {
            const size_t o = (size_t)(p - x);
            const float4 w4 = *reinterpret_cast<const float4*>(y + o);
            v4.x += w4.x; v4.y += w4.y; v4.z += w4.z; v4.w += w4.w;
            if (!out_b) *reinterpret_cast<float4*>(out + o) = v4;
          }
          if (out_b) {     // bf16 copy of the tensor the statistics describe (start of a bf16 residual stream); ldx == C
            const __nv_bfloat162 lo2 = __floats2bfloat162_rn(v4.x, v4.y), hi2 = __floats2bfloat162_rn(v4.z, v4.w);
            *reinterpret_cast<uint2*>(out_b + (size_t)(p - x)) =
                make_uint2(*reinterpret_cast<const uint32_t*>(&lo2), *reinterpret_cast<const uint32_t*>(&hi2));
          }
          s[0] += v4.x; q[0] = fmaf(v4.x, v4.x, q[0]);
          s[1 % VEC] += v4.y; q[1 % VEC] = fmaf(v4.y, v4.y, q[1 % VEC]);
          s[2 % VEC] += v4.z; q[2 % VEC] = fmaf(v4.z, v4.z, q[2 % VEC]);
          s[3 % VEC] += v4.w; q[3 % VEC] = fmaf(v4.w, v4.w, q[3 % VEC]);
        } else {
          const float v1 = *p;
          s[0] += v1; q[0] = fmaf(v1, v1, q[0]);
        }
      }
    }
    __syncthreads();
#pragma unroll
    for (int v = 0; v < VEC; v++) { red[0][threadIdx.x * VEC + v] = s[v]; red[1][threadIdx.x * VEC + v] = q[v]; }
    __syncthreads();
    if (ty == 0 && cg < CV) {
#pragma unroll
      for (int v = 0; v < VEC; v++) {
        float ss = 0.f, qq = 0.f;
        for (int y = 0; y < YT; y++) { ss += red[0][(y * XT + tx) * VEC + v]; qq += red[1][(y * XT + tx) * VEC + v]; }
        const int c = cg * VEC + v;
        if (c < C) { pp[c] = ss; pp[C + c] = qq; }
      }
    }
  }
}
void launch_colstats(const float* x, int ldx, int C, float* part, const int* off, const int* len,
                     int B, int max_len, cudaStream_t st, void* out_bf16) {
  if (g_dry_run) return;
  const int nchunk = (max_len + kStatRows - 1) / kStatRows;
  dim3 g(nchunk, B);
  const bool vec = (C % 4 == 0) && (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  if (out_bf16 && (!vec || ldx != C || (reinterpret_cast<uintptr_t>(out_bf16) & 7)))
    throw ArgError("launch_colstats: the bf16 copy needs ldx == C, C % 4 == 0 and aligned tensors");
  if (vec)
    colstats_kernel<4, false><<<g, 256, 0, st>>>(x, ldx, C, part, nchunk, off, len, nullptr, nullptr, static_cast<__nv_bfloat16*>(out_bf16));
  else
    colstats_kernel<1, false><<<g, 256, 0, st>>>(x, ldx, C, part, nchunk, off, len, nullptr, nullptr, nullptr);
  post_launch("colstats", st);
}
void launch_add_rows_stats(const float* a, const float* b, float* out, int C, float* part, const int* off,
                           const int* len, int B, int max_len, cudaStream_t st, void* out_bf16) {
  if (g_dry_run) return;
  if (C % 4 != 0 || ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(out)) & 15) ||
      (reinterpret_cast<uintptr_t>(out_bf16) & 7))
    throw ArgError("launch_add_rows_stats: needs C % 4 == 0 and 16-byte aligned tensors");
  const int nchunk = (max_len + kStatRows - 1) / kStatRows;
  dim3 g(nchunk, B);
  colstats_kernel<4, true><<<g, 256, 0, st>>>(a, C, C, part, nchunk, off, len, b, out, static_cast<__nv_bfloat16*>(out_bf16));
  post_launch("add_rows_stats", st);
}

// Pointwise conv with few input channels, fused with the statistics of its output (generator stage 1: noise_convs[1]
// = Conv1d(22, 128, k = 1) over the 120T+1 STFT frames, followed by the first AdaIN of noise_res[1]).
//   out[r, co] = bias[co] + sum_ci x[r, ci] * w[ci][co],   part[b][chunk][2][128] = column sums / sums of squares
// The op writes 512 B per row for 88 B read and 22 FMA per output: it is a store stream, not a GEMM.  On the tensor-core
// path it was three passes (x -> bf16 plane padded to 64 channels, a one-k-step implicit GEMM whose single-tile CTAs
// stored at 2.2 TB/s, and a colstats pass reading the 2.9 GB result back); here one CTA owns one statistics chunk
// (128 rows): the x rows are staged in shared memory, a warp shares a row (broadcast reads), a thread owns 4 output
// channels with its 4 x Ci weights in registers, stores are 512 contiguous bytes per warp, and the chunk statistics
// leave from the same registers in a fixed order.  fp32 FMA in ascending ci: exact operands, no bf16 rounding.
template <int CI>
__global__ void __launch_bounds__(256) pointwise_conv_stats_kernel(const float* __restrict__ x, int ldx,
                                                                   const float* __restrict__ w /*[CI][128]*/,
                                                                   const float* __restrict__ bias,
                                                                   float* __restrict__ out, float* __restrict__ part,
                                                                   int nchunk, const int* off, const int* len) {
  constexpr int LDS_ = 24;                         // staged row pitch (CI <= 24)
  static_assert(CI <= LDS_, "pointwise_conv_stats: at most 24 input channels");
  __shared__ __align__(16) float xs[kStatRows * LDS_];
  __shared__ float red[2][8][128];
  const int b = blockIdx.y, ch = blockIdx.x;
  const int L = len[b];
  const int r0 = ch * kStatRows;
  if (r0 >= L) return;
  const int nrows = min(kStatRows, L - r0);
  const size_t row0 = (size_t)off[b] + r0;
  const int t = threadIdx.x;
  if (ldx == LDS_) {                               // contiguous block: 128-bit loads
    const float4* src = reinterpret_cast<const float4*>(x + row0 * LDS_);
    for (int i = t; i < kStatRows * LDS_ / 4; i += 256)
      reinterpret_cast<float4*>(xs)[i] = (i * 4) / LDS_ < nrows ? src[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  } else {
    for (int i = t; i < kStatRows * LDS_; i += 256) {
      const int r = i / LDS_, c = i % LDS_;
      xs[i] = (r < nrows && c < CI) ? x[(row0 + r) * ldx + c] : 0.f;
    }
  }
  const int cq = t & 31, rl = t >> 5;              // channel quad, row lane (= warp)
  float4 wr[CI];
#pragma unroll
  for (int ci = 0; ci < CI; ci++) wr[ci] = *reinterpret_cast<const float4*>(w + ci * 128 + 4 * cq);
  const float4 b4 = *reinterpret_cast<const float4*>(bias + 4 * cq);
  float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), q4 = s4;
  __syncthreads();
  float* op = out + (row0 + rl) * 128 + 4 * cq;
#pragma unroll 4
  for (int r = rl; r < nrows; r += 8, op += 8 * 128) {
    const float* xr = xs + r * LDS_;
    float4 a = b4;
#pragma unroll
    for (int ci = 0; ci < CI; ci++) {
      const float h = xr[ci];
      a.x = fmaf(h, wr[ci].x, a.x); a.y = fmaf(h, wr[ci].y, a.y); a.z = fmaf(h, wr[ci].z, a.z); a.w = fmaf(h, wr[ci].w, a.w);
    }
    *reinterpret_cast<float4*>(op) = a;
    s4.x += a.x; s4.y += a.y; s4.z += a.z; s4.w += a.w;
    q4.x = fmaf(a.x, a.x, q4.x); q4.y = fmaf(a.y, a.y, q4.y); q4.z = fmaf(a.z, a.z, q4.z); q4.w = fmaf(a.w, a.w, q4.w);
  }
  *reinterpret_cast<float4*>(&red[0][rl][4 * cq]) = s4;
  *reinterpret_cast<float4*>(&red[1][rl][4 * cq]) = q4;
  __syncthreads();
  {
    const int which = t >> 7, c = t & 127;         // threads 0..127: sums, 128..255: sums of squares
    float acc = 0.f;
#pragma unroll
    for (int y = 0; y < 8; y++) acc += red[which][y][c];
    part[((size_t)b * nchunk + ch) * 2 * 128 + which * 128 + c] = acc;
  }
}
void launch_pointwise_conv_stats(const float* x, int ldx, int Ci, const float* w, const float* bias, float* out, int Co,
                                 float* part, const int* off, const int* len, int B, int max_len, long long sum_m,
                                 cudaStream_t st) {
  if (g_dry_run) return;
  if (Ci != 22 || Co != 128 || ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(w) |
                                 reinterpret_cast<uintptr_t>(bias)) & 15))
    throw ArgError("launch_pointwise_conv_stats: built for Conv1d(22, 128, k = 1) on 16-byte aligned tensors");
  const int nchunk = (max_len + kStatRows - 1) / kStatRows;
  dim3 g(nchunk, B);
  pointwise_conv_stats_kernel<22><<<g, 256, 0, st>>>(x, ldx, w, bias, out, part, nchunk, off, len);
  if (g_launch_stats) g_launch_stats->conv_flops += 2.0 * (double)sum_m * Co * Ci;   // counted like the GEMM path it replaces
  post_launch("pointwise_conv_stats", st);
}

// Combine the chunk partials (fp64, fixed order) -> AdaIN coefficients.  Block = 32 channels x 32 chunk
// slices (1024 threads): the grid is tiny (C/32 x B blocks), so the kernel is pure load latency -- every thread
// keeps 4 chunks (8 independent loads) in flight; the additions keep a fixed order, so the result depends only
// on the data, not on how a batch was composed.
constexpr int kCoefSlices = 32;
__global__ void __launch_bounds__(32 * kCoefSlices) adain_coef_kernel(const float* __restrict__ part, int C,
                                                                      int nchunk, const int* len,
                                                                      const float* __restrict__ sty, int sld,
                                                                      int soff, float eps, float* scale,
                                                                      float* shift) {
  __shared__ double rs[kCoefSlices][32], rq[kCoefSlices][32];
  const int b = blockIdx.y;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int L = len[b];
  const int nc = (L + kStatRows - 1) / kStatRows;
  double S = 0.0, Q = 0.0;
  if (c < C) {
    const float* pp = part + (size_t)b * nchunk * 2 * C + c;
    int k = ty;
    for (; k + 3 * kCoefSlices < nc; k += 4 * kCoefSlices) {
      float sv[4], qv[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        sv[u] = pp[(size_t)(k + kCoefSlices * u) * 2 * C];
        qv[u] = pp[(size_t)(k + kCoefSlices * u) * 2 * C + C];
      }
#pragma unroll
      for (int u = 0; u < 4; u++) { S += (double)sv[u]; Q += (double)qv[u]; }
    }
    for (; k < nc; k += kCoefSlices) {
      S += (double)pp[(size_t)k * 2 * C];
      Q += (double)pp[(size_t)k * 2 * C + C];
    }
  }
  rs[ty][tx] = S; rq[ty][tx] = Q;
  __syncthreads();
  if (ty == 0 && c < C) {
    S = 0.0; Q = 0.0;
#pragma unroll
    for (int y = 0; y < kCoefSlices; y++) { S += rs[y][tx]; Q += rq[y][tx]; }
    const double mean = S / (double)L;
    double var = Q / (double)L - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = 1.0f / sqrtf((float)var + eps);
    const float gamma = sty[(size_t)b * sld + soff + c];
    const float beta = sty[(size_t)b * sld + soff + C + c];
    const float sc = rstd * (1.0f + gamma);
    scale[(size_t)b * C + c] = sc;
    shift[(size_t)b * C + c] = beta - (float)mean * sc;
  }
}
void launch_adain_coef(const float* part, int C, int max_len, const int* len, const float* sty,
                       int sld, int soff, float eps, float* scale, float* shift, int B,
                       cudaStream_t st) {
  if (g_dry_run) return;
  const int nchunk = (max_len + kStatRows - 1) / kStatRows;
  dim3 g((C + 31) / 32, B);
  adain_coef_kernel<<<g, 32 * kCoefSlices, 0, st>>>(part, C, nchunk, len, sty, sld, soff, eps, scale, shift);
  post_launch("adain_coef", st);
}

// ------------------------------------------------------------------------------------------
// Depthwise ConvTranspose1d(k3, s2, p1, op1) applied to lrelu(x*scale+shift):
//   y[2t]   = w[1]*a[t] + bias
//   y[2t+1] = w[2]*a[t] + w[0]*a[t+1] + bias           (a[T] = 0)
__global__ void __launch_bounds__(256) pool_up_kernel(const float* __restrict__ in, int ldi,
                                                      const float* scale, const float* shift,
                                                      float slope, const float* w, const float* bias,
                                                      int C, float* out, int ldo, const int* in_off,
                                                      const int* in_len, const int* out_off) {
  const int b = blockIdx.z;
  const int T = in_len[b];
  const int t = blockIdx.x;
  if (t >= T) return;
  const float* sc = scale + (size_t)b * C;
  const float* sh = shift + (size_t)b * C;
  const float* x0 = in + (size_t)(in_off[b] + t) * ldi;
  float* y0 = out + (size_t)(out_off[b] + 2 * t) * ldo;
  for (int c = blockIdx.y * 256 + threadIdx.x; c < C; c += gridDim.y * 256) {
    float a0 = x0[c] * sc[c] + sh[c];
    a0 = a0 > 0.f ? a0 : a0 * slope;
    float a1 = 0.f;
    if (t + 1 < T) {
      a1 = x0[ldi + c] * sc[c] + sh[c];
      a1 = a1 > 0.f ? a1 : a1 * slope;
    }
    const float w0 = w[c * 3 + 0], w1 = w[c * 3 + 1], w2 = w[c * 3 + 2], bb = bias[c];
    y0[c] = w1 * a0 + bb;
    y0[ldo + c] = w2 * a0 + w0 * a1 + bb;
  }
}
void launch_pool_up(const float* in, int ldi, const float* scale, const float* shift, float slope,
                    const float* w, const float* bias, int C, float* out, int ldo,
                    const int* in_off, const int* in_len, const int* out_off, int B, int max_len,
                    cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g(max_len, (C + 255) / 256, B);
  pool_up_kernel<<<g, 256, 0, st>>>(in, ldi, scale, shift, slope, w, bias, C, out, ldo, in_off,
                                    in_len, out_off);
  post_launch("pool_up", st);
}

// ------------------------------------------------------------------------------------------
// K4 duration head.  sigmoid in fp32, 50-way sum accumulated in fp64 and rounded once, divide
// by speed, round-half-even (rintf), clamp >= 1.
__global__ void __launch_bounds__(128) duration_kernel(const float* __restrict__ logits, int K,
                                                       const float* speeds, int* pred_dur,
                                                       float* dur_float, const int* off,
                                                       const int* len) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * 128 + threadIdx.x;
  if (t >= len[b]) return;
  const size_t row = (size_t)off[b] + t;
  double s = 0.0;
  for (int k = 0; k < K; k++) {
    const float sg = 1.0f / (1.0f + expf(-logits[row * K + k]));
    s += (double)sg;
  }
  const float d = __fdiv_rn((float)s, speeds[b]);
  dur_float[row] = d;
  float r = rintf(d);
  if (!(r >= 1.0f)) r = 1.0f;       // (also catches NaN logits)
  // sum of K sigmoids <= K = 50 and speed >= 0.1 (validated on the host) bound this by 500; the explicit cap keeps the
  // float -> int conversion and the int32 prefix sum safe whatever the logits hold
  pred_dur[row] = (int)fminf(r, 1000.0f);
}
void launch_duration(const float* logits, int K, const float* speeds, int* pred_dur,
                     float* dur_float, const int* off, const int* len, int B, int max_len,
                     cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 127) / 128, B);
  duration_kernel<<<g, 128, 0, st>>>(logits, K, speeds, pred_dur, dur_float, off, len);
  post_launch("duration", st);
}

// Exclusive integer prefix sum over one item's tokens (N <= 512): one CTA of 512 threads.
__global__ void __launch_bounds__(512) dur_scan_kernel(const int* __restrict__ pred_dur, int* cum,
                                                       int cum_ld, int* total, const int* off,
                                                       const int* len) {
  __shared__ int wsum[16];
  const int b = blockIdx.x;
  const int N = len[b];
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int v = t < N ? pred_dur[off[b] + t] : 0;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) wsum[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = lane < 16 ? wsum[lane] : 0;
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < 16) wsum[lane] = w;
  }
  __syncthreads();
  const int incl = x + (warp ? wsum[warp - 1] : 0);
  if (t < N) cum[(size_t)b * cum_ld + t] = incl - v;
  if (t == N - 1) total[b] = incl;
}
void launch_dur_scan(const int* pred_dur, int* cum, int cum_ld, int* total, const int* off,
                     const int* len, int B, cudaStream_t st) {
  if (g_dry_run) return;
  dur_scan_kernel<<<B, 512, 0, st>>>(pred_dur, cum, cum_ld, total, off, len);
  post_launch("dur_scan", st);
}

// idx[j] = the token n whose frame interval [cum[n], cum[n+1]) contains j (binary search).
__global__ void __launch_bounds__(256) expand_idx_kernel(const int* __restrict__ cum, int cum_ld,
                                                         const int* tok_len, int* idx,
                                                         const int* fr_off, const int* fr_len) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= fr_len[b]) return;
  const int* c = cum + (size_t)b * cum_ld;
  int lo = 0, hi = tok_len[b] - 1;  // largest n with c[n] <= j
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (c[mid] <= j) lo = mid; else hi = mid - 1;
  }
  idx[fr_off[b] + j] = lo;
}
void launch_expand_idx(const int* cum, int cum_ld, const int* tok_len, int* idx, const int* fr_off,
                       const int* fr_len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 255) / 256, B);
  expand_idx_kernel<<<g, 256, 0, st>>>(cum, cum_ld, tok_len, idx, fr_off, fr_len);
  post_launch("expand_idx", st);
}

// K5 length regulation: exact row gather.
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ in, int ldi,
                                                          const int* in_off, const int* idx,
                                                          const int* fr_off, const int* fr_len,
                                                          int C, float* out, int ldo, int ocol) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (j >= fr_len[b]) return;
  const int n = idx[fr_off[b] + j];
  const float* src = in + (size_t)(in_off[b] + n) * ldi;
  float* dst = out + (size_t)(fr_off[b] + j) * ldo + ocol;
  for (int c = threadIdx.x & 31; c < C; c += 32) dst[c] = src[c];
}
void launch_gather_rows(const float* in, int ldi, const int* in_off, const int* idx,
                        const int* fr_off, const int* fr_len, int C, float* out, int ldo, int ocol,
                        int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 7) / 8, B);
  gather_rows_kernel<<<g, 256, 0, st>>>(in, ldi, in_off, idx, fr_off, fr_len, C, out, ldo, ocol);
  post_launch("gather_rows", st);
}

// Conv1d(1,1,k3,s2,p1) on the F0 / N curves.
__global__ void __launch_bounds__(256) curve_conv_kernel(const float* __restrict__ x,
                                                         const int* x_off, const int* x_len,
                                                         const float* w3, const float* bias,
                                                         float* out, int ldo, int ocol,
                                                         const int* out_off, const int* out_len) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * 256 + threadIdx.x;
  if (t >= out_len[b]) return;
  const int L = x_len[b];
  const float* xp = x + x_off[b];
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const int r = 2 * t - 1 + k;
    if (r >= 0 && r < L) acc = fmaf(w3[k], xp[r], acc);
  }
  out[(size_t)(out_off[b] + t) * ldo + ocol] = acc + bias[0];
}
void launch_curve_conv(const float* x, const int* x_off, const int* x_len, const float* w3,
                       const float* bias, float* out, int ldo, int ocol, const int* out_off,
                       const int* out_len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 255) / 256, B);
  curve_conv_kernel<<<g, 256, 0, st>>>(x, x_off, x_len, w3, bias, out, ldo, ocol, out_off, out_len);
  post_launch("curve_conv", st);
}

// ------------------------------------------------------------------------------------------
// K9 harmonic source.
// Coarse phase: rad_h[i] = frac(f0[i]*h/24000) (the x1/300 linear down-sampling of the
// nearest-upsampled curve reads two taps of the same 300-sample plateau, so it reproduces the
// plateau value), inclusive cumsum in fp64 rounded to fp32 per element (matches the CPU
// reference's cumsum, which accumulates in double), then ((c*2)*pi)*300 in fp32.
__global__ void __launch_bounds__(256) sine_phase_kernel(const float* __restrict__ f0,
                                                         const int* f0_off, const int* f0_len,
                                                         float* phase, const int* ph_off) {
  __shared__ double wsum[8];
  __shared__ double carry_s;
  const int b = blockIdx.x, hm = blockIdx.y;  // harmonic index 0..8
  const int L = f0_len[b];
  const float* fp = f0 + f0_off[b];
  float* pp = phase + ph_off[b] + (size_t)hm * L;
  const float mult = (float)(hm + 1);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  if (t == 0) carry_s = 0.0;
  __syncthreads();
  for (int base = 0; base < L; base += 256) {
    const int i = base + t;
    double v = 0.0;
    if (i < L) {
      const float fn = __fmul_rn(fp[i], mult);
      const float q = __fdiv_rn(fn, 24000.0f);
      const float r = q - floorf(q);          // python-style % 1
      v = (double)r;
    }
    double x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    double pre = carry_s;
    for (int w = 0; w < warp; w++) pre += wsum[w];
    const double incl = pre + x;
    if (i < L) {
      const float c = (float)incl;
      pp[i] = __fmul_rn(__fmul_rn(__fmul_rn(c, 2.0f), 3.14159265358979323846f), 300.0f);
    }
    __syncthreads();
    if (t == 255) carry_s = incl;
    __syncthreads();
  }
}
void launch_sine_phase(const float* f0, const int* f0_off, const int* f0_len, float* phase,
                       const int* ph_off, int B, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g(B, 9);
  sine_phase_kernel<<<g, 256, 0, st>>>(f0, f0_off, f0_len, phase, ph_off);
  post_launch("sine_phase", st);
}

// Philox4x32-10 counter RNG + Box-Muller for the production noise path (tests inject noise).
__device__ __forceinline__ void philox4x32_10(unsigned c0, unsigned c1, unsigned c2, unsigned c3,
                                              unsigned k0, unsigned k1, unsigned* out) {
#pragma unroll
  for (int i = 0; i < 10; i++) {
    const unsigned long long p0 = (unsigned long long)0xD2511F53u * c0;
    const unsigned long long p1 = (unsigned long long)0xCD9E8D57u * c2;
    const unsigned n0 = (unsigned)(p1 >> 32) ^ c1 ^ k0;
    const unsigned n1 = (unsigned)p1;
    const unsigned n2 = (unsigned)(p0 >> 32) ^ c3 ^ k1;
    const unsigned n3 = (unsigned)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ float u01(unsigned x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }

// Per sample: x300 linear interpolation (align_corners=False) of the coarse phase exactly as the
// CPU reference evaluates it -- src = fma(1/300, n+0.5, -0.5) clamped at 0, lambda = src - i0,
// value = fma(p[i0], 1-lambda, p[i1]*lambda) -- then sin, *0.1, uv gating, noise, Linear(9->1),
// tanh.
// sin of a harmonic phase that reaches 1e5..1e6 rad late in an utterance.  libm's sinf leaves its fast path
// above ~1e5 rad (Payne-Hanek reduction, divergent: most of this kernel's time); here the argument is reduced in
// fp64 (turns = ph / 2pi, exact to ~1e-11 of a turn) and sinpif evaluates the reduced angle.  Error vs the exact
// sin(ph): <= 2e-7 absolute (the fp32 rounding of the reduced angle).
__device__ __forceinline__ float sin_reduced(float ph) {
  const double t = (double)ph * 0.15915494309189535;
  const double fr = t - rint(t);
  return sinpif((float)(2.0 * fr));
}

__global__ void __launch_bounds__(256) sine_source_kernel(
    const float* __restrict__ f0, const int* f0_off, const int* f0_len,
    const float* __restrict__ phase, const int* ph_off, const float* __restrict__ noise,
    unsigned long long seed, const float* lin_w, const float* lin_b, float* out,
    const long long* s_off) {
  const int b = blockIdx.y;
  const int L = f0_len[b];
  const long long S = (long long)L * 300;
  const long long n = (long long)blockIdx.x * 256 + threadIdx.x;
  if (n >= S) return;
  const float f = f0[f0_off[b] + (int)(n / 300)];
  const float uv = f > 10.0f ? 1.0f : 0.0f;
  const float scale = 0.0033333334f;  // (float)(1.0/300.0)
  float src = __fmaf_rn(scale, (float)n + 0.5f, -0.5f);
  if (src < 0.f) src = 0.f;
  const int i0 = (int)src;
  const int i1 = i0 + (i0 < L - 1 ? 1 : 0);
  float lam = src - (float)i0;
  lam = fminf(fmaxf(lam, 0.f), 1.f);
  const float w0 = 1.0f - lam;
  const float namp = __fadd_rn(__fmul_rn(uv, 0.003f), __fdiv_rn(__fmul_rn(1.0f - uv, 0.1f), 3.0f));
  float nz[9];
  if (noise) {
#pragma unroll
    for (int h = 0; h < 9; h++) nz[h] = noise[n * 9 + h];
  } else {
    unsigned r[12];
    // keyed by (seed, sample index) only, NOT by the batch slot: an utterance gets the same noise
    // whether it runs alone or inside a batch (kkx_infer_batch == per-item kkx_infer)
    philox4x32_10((unsigned)n, (unsigned)(n >> 32), 0u, 0u, (unsigned)seed, (unsigned)(seed >> 32), r);
    philox4x32_10((unsigned)n, (unsigned)(n >> 32), 0u, 1u, (unsigned)seed, (unsigned)(seed >> 32), r + 4);
    philox4x32_10((unsigned)n, (unsigned)(n >> 32), 0u, 2u, (unsigned)seed, (unsigned)(seed >> 32), r + 8);
#pragma unroll
    for (int h = 0; h < 5; h++) {
      const float u1 = u01(r[2 * h]), u2 = u01(r[2 * h + 1]);
      // Box-Muller with the fast intrinsics: this is the library's own N(0,1) generator (never compared with
      // the oracle, which gets its noise injected), and libm-accurate logf / sincosf were a third of the kernel
      const float rad = sqrtf(-2.0f * __logf(u1));
      float sn, cs;
      __sincosf(6.283185307179586f * u2, &sn, &cs);
      nz[2 * h] = rad * cs;
      if (2 * h + 1 < 9) nz[2 * h + 1] = rad * sn;
    }
  }
  const float* pp = phase + ph_off[b];
  float acc = lin_b[0];
#pragma unroll
  for (int h = 0; h < 9; h++) {
    const float p0 = pp[(size_t)h * L + i0], p1 = pp[(size_t)h * L + i1];
    const float ph = __fmaf_rn(p0, w0, __fmul_rn(p1, lam));
    const float sw = __fmul_rn(sin_reduced(ph), 0.1f);
    const float v = __fadd_rn(__fmul_rn(sw, uv), __fmul_rn(namp, nz[h]));
    acc = fmaf(lin_w[h], v, acc);
  }
  out[s_off[b] + n] = tanhf(acc);
}
void launch_sine_source(const float* f0, const int* f0_off, const int* f0_len, const float* phase,
                        const int* ph_off, const float* noise, unsigned long long seed,
                        const float* lin_w, const float* lin_b, float* out, const long long* s_off,
                        int B, long long max_samples, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((unsigned)((max_samples + 255) / 256), B);
  sine_source_kernel<<<g, 256, 0, st>>>(f0, f0_off, f0_len, phase, ph_off, noise, seed, lin_w,
                                        lin_b, out, s_off);
  post_launch("sine_source", st);
}

// ------------------------------------------------------------------------------------------
// K10 STFT of the source: n_fft 20, hop 5, periodic hann, center=True.  One thread per frame.
__constant__ float c_cos20[20];
__constant__ float c_sin20[20];
__constant__ float c_hann20[20];
static void ensure_tables() {
  // once per device, and safe when two sessions on two threads reach their first STFT together
  static DevOnce once;
  int dev = 0;
  cudaGetDevice(&dev);
  once.run(dev, [] {
  float cs[20], sn[20], hw[20];
  for (int j = 0; j < 20; j++) {
    cs[j] = (float)cos(2.0 * M_PI * j / 20.0);
    sn[j] = (float)sin(2.0 * M_PI * j / 20.0);
    hw[j] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * j / 20.0));
  }
  sn[0] = 0.f; sn[10] = 0.f; cs[5] = 0.f; cs[15] = 0.f;
  KKX_CUDA(cudaMemcpyToSymbol(c_cos20, cs, sizeof cs));
  KKX_CUDA(cudaMemcpyToSymbol(c_sin20, sn, sizeof sn));
  KKX_CUDA(cudaMemcpyToSymbol(c_hann20, hw, sizeof hw));
  });
}

__global__ void __launch_bounds__(128) stft_kernel(const float* __restrict__ x,
                                                   const long long* s_off, float* har, int ldh,
                                                   const int* h_off, const int* h_len,
                                                   int replicate_pad) {
  const int b = blockIdx.y;
  const int f = blockIdx.x * 128 + threadIdx.x;
  const int F = h_len[b];
  if (f >= F) return;
  const long long S = (long long)(F - 1) * 5;
  const float* xp = x + s_off[b];
  float xw[20];
#pragma unroll
  for (int j = 0; j < 20; j++) {
    long long i = (long long)f * 5 - 10 + j;
    if (replicate_pad) {
      i = i < 0 ? 0 : (i >= S ? S - 1 : i);
    } else {
      if (i < 0) i = -i;
      if (i >= S) i = 2 * (S - 1) - i;
    }
    xw[j] = xp[i] * c_hann20[j];
  }
  float l1 = 0.f;
#pragma unroll
  for (int j = 0; j < 20; j++) l1 += fabsf(xw[j]);
  const float cut_tol = 4e-6f * l1;  // fp32 rounding floor of the 20-term sums
  float* o = har + (size_t)(h_off[b] + f) * ldh;
#pragma unroll
  for (int k = 0; k <= 10; k++) {
    float re = 0.f, im = 0.f;
#pragma unroll
    for (int j = 0; j < 20; j++) {
      const int m = (j * k) % 20;
      re = fmaf(xw[j], c_cos20[m], re);
      im = fmaf(-xw[j], c_sin20[m], im);
    }
    if (k == 0 || k == 10) im = 0.f;   // real input: DC / Nyquist are exactly real (+0)
    o[k] = hypotf(re, im);
    // branch-cut canonicalisation shared with the oracle: (re<0, |im| inside the rounding floor) -> +pi
    const bool cut = re < 0.f && fabsf(im) <= cut_tol;
    o[11 + k] = cut ? 3.14159265358979323846f : atan2f(im, re);
  }
}
void launch_stft(const float* x, const long long* s_off, float* har, int ldh, const int* h_off,
                 const int* h_len, int replicate_pad, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  ensure_tables();
  dim3 g((max_len + 127) / 128, B);
  stft_kernel<<<g, 128, 0, st>>>(x, s_off, har, ldh, h_off, h_len, replicate_pad);
  post_launch("stft", st);
}

// K11 head + iSTFT, one thread per STFT frame.
//
// Output sample n (after the n_fft/2 = 10 trim) sits at untrimmed position p = n + 10; the five samples p = 5q .. 5q+4
// ("group q", q = 2 .. F) are the overlap-add of frames q, q-1, q-2, q-3 at in-frame positions j0 + 5d.  A CTA of 128
// threads owns kIstftGroups = 124 consecutive groups (620 samples = 155 float4) and the 127 frames they touch:
//   1. the [127, 24] fp32 block of conv_post rows is staged in shared memory with coalesced 128-bit loads
//      (row pitch 24 floats -> 25 in smem, conflict-free for the per-thread row reads);
//   2. thread t turns its frame's 22 logits into the spectrum (mag = exp(x), phase = sin(x') -> mag*(cos, sin)) and
//      runs the real inverse DFT of size 20 entirely in registers: x[j] = C[j] - S[j], x[20-j] = C[j] + S[j] with
//      C[j] = sum_k Re_k cos(2 pi j k / 20), S[j] = sum_k Im_k sin(2 pi j k / 20) for j = 0..10 (the twiddles are
//      compile-time constants, ~200 FFMA per frame instead of ~360 shared-memory complex products), applies the
//      synthesis window and writes the 20 samples to shared memory (pitch 21);
//   3. thread t >= 3 adds the four overlapping frames of its group, divides by the window envelope and puts the five
//      samples into a staging row, from which the CTA stores 128-bit vectors (fp32) / 64-bit vectors (pcm16).
// FAST (tensor-core configuration, 3e-2 waveform tolerance): ex2 / sin / cos via the SFU intrinsics and a reciprocal
// multiply for the envelope; the fp32 verification configuration keeps libm expf / sinf / sincosf and a true division.
constexpr int kIstftGroups = 124;
constexpr int kIstftFrames = kIstftGroups + 3;   // 127
__host__ __device__ constexpr float tw_cos(int m) {   // cos(2 pi m / 20), m taken mod 20
  constexpr float c[20] = {1.0f, 0.95105651629515357f, 0.80901699437494742f, 0.58778525229247313f, 0.30901699437494742f,
                           0.0f, -0.30901699437494742f, -0.58778525229247313f, -0.80901699437494742f, -0.95105651629515357f,
                           -1.0f, -0.95105651629515357f, -0.80901699437494742f, -0.58778525229247313f, -0.30901699437494742f,
                           0.0f, 0.30901699437494742f, 0.58778525229247313f, 0.80901699437494742f, 0.95105651629515357f};
  return c[m % 20];
}
__host__ __device__ constexpr float tw_sin(int m) { return tw_cos(m + 15); }   // sin(x) = cos(x - pi/2)
// 16-bit PCM of an output sample: trunc(clamp(s, -1, 1) * 32767), the f32 -> i16 conversion of the reference's WebSocket
// server (kokorox-websocket/src/lib.rs:699-703; Rust `as i16` truncates toward zero, NaN -> 0)
__device__ __forceinline__ short pcm16_of(float s) {
  return (short)__float2int_rz(fminf(fmaxf(s, -1.0f), 1.0f) * 32767.0f);
}

template <bool FAST>
__global__ void __launch_bounds__(128) istft_kernel(const float* __restrict__ cp, int ldc,
                                                    const int* __restrict__ h_off, const int* __restrict__ h_len,
                                                    float* __restrict__ audio, const long long* __restrict__ s_off,
                                                    short* __restrict__ pcm) {
  __shared__ __align__(16) float s_in[kIstftFrames * 25];    // staged conv_post rows (22 used of 24, pitch 25)
  __shared__ float s_fr[kIstftFrames * 21];                  // windowed time frames, pitch 21
  __shared__ __align__(16) float s_out[kIstftGroups * 5];    // 620 output samples
  __shared__ float s_win[20];
  const int b = blockIdx.y;
  const int F = h_len[b];
  const int q0 = 2 + kIstftGroups * blockIdx.x;              // first output group of this CTA
  if (q0 > F) return;
  const int fbase = q0 - 3;                                  // frame of thread 0
  const int t = threadIdx.x;
  if (t < 20) s_win[t] = c_hann20[t];
  // ---- 1. stage the rows [fbase, fbase + 127) x 24 floats (contiguous in global memory when ldc == 24)
  {
    const int lo = max(fbase, 0), hi = min(fbase + kIstftFrames, F);   // existing frames
    const float* src = cp + (size_t)(h_off[b] + lo) * ldc;
    const int nvec = (hi - lo) * 6;                                    // float4 per row: 24 / 4 (ldc == 24, 16-byte aligned rows)
    for (int v = t; v < nvec; v += 128) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(src) + v);
      const int row = v / 6 + (lo - fbase), c4 = (v % 6) * 4;
      float* d = s_in + row * 25 + c4;
      d[0] = x.x; d[1] = x.y; d[2] = x.z; d[3] = x.w;
    }
  }
  __syncthreads();
  // ---- 2. spectrum + inverse DFT of this thread's frame
  const int f = fbase + t;
  if (t < kIstftFrames) {
    float xr[20];
    if (f >= 0 && f < F) {
      const float* c = s_in + t * 25;
      float re[11], im[11];
#pragma unroll
      for (int k = 0; k < 11; k++) {
        float mag, sn, cs;
        if (FAST) {
          mag = __expf(c[k]);
          __sincosf(__sinf(c[11 + k]), &sn, &cs);
        } else {
          mag = expf(c[k]);
          sincosf(sinf(c[11 + k]), &sn, &cs);
        }
        re[k] = mag * cs;
        im[k] = mag * sn;
      }
      // bins 0 and 10 contribute their real part only (one-sided inverse of a real signal)
#pragma unroll
      for (int j = 0; j <= 10; j++) {
        float C = 0.f, S = 0.f;
#pragma unroll
        for (int k = 1; k < 10; k++) {
          C = fmaf(re[k], tw_cos(j * k), C);
          S = fmaf(im[k], tw_sin(j * k), S);
        }
        const float base = re[0] + ((j & 1) ? -re[10] : re[10]);
        xr[j] = fmaf(2.0f, C - S, base);
        if (j >= 1 && j <= 9) xr[20 - j] = fmaf(2.0f, C + S, base);
      }
#pragma unroll
      for (int j = 0; j < 20; j++) xr[j] = xr[j] * (1.0f / 20.0f) * s_win[j];
    } else {
#pragma unroll
      for (int j = 0; j < 20; j++) xr[j] = 0.f;
    }
#pragma unroll
    for (int j = 0; j < 20; j++) s_fr[t * 21 + j] = xr[j];
  }
  __syncthreads();
  // ---- 3. overlap-add of group q = q0 + (t - 3): frames t, t-1, t-2, t-3 of this CTA
  const long long S_total = (long long)(F - 1) * 5;
  if (t >= 3 && t < kIstftFrames) {
    const int q = q0 + (t - 3);
    if (q <= F) {
#pragma unroll
      for (int j0 = 0; j0 < 5; j0++) {
        float acc = 0.f, env = 0.f;
#pragma unroll
        for (int d = 0; d < 4; d++) {
          const int ff = q - d;
          if (ff < 0 || ff >= F) continue;
          const int j = j0 + 5 * d;
          acc += s_fr[(t - d) * 21 + j];
          env = fmaf(s_win[j], s_win[j], env);
        }
        s_out[(t - 3) * 5 + j0] = FAST ? acc * __frcp_rn(env) : acc / env;
      }
    }
  }
  __syncthreads();
  // ---- 4. vector stores: sample n = 5 (q - 2) + j0 -> CTA base n0 = 620 * blockIdx.x (16-byte aligned: item offsets
  // are multiples of 600 samples)
  const long long n0 = (long long)kIstftGroups * 5 * blockIdx.x;
  const long long remain = S_total - n0;
  const int count = remain < kIstftGroups * 5 ? (int)remain : kIstftGroups * 5;
  float* dst = audio + s_off[b] + n0;
  for (int v = t; v * 4 < count; v += 128) {
    const float4 x = *reinterpret_cast<const float4*>(s_out + v * 4);
    if (v * 4 + 4 <= count) {
      *reinterpret_cast<float4*>(dst + v * 4) = x;
    } else {
      for (int e = 0; v * 4 + e < count; e++) dst[v * 4 + e] = s_out[v * 4 + e];
    }
  }
  if (pcm) {
    short* pd = pcm + s_off[b] + n0;   // optional 16-bit PCM (pcm16_of)
    for (int v = t; v * 4 < count; v += 128) {
      if (v * 4 + 4 <= count) {
        *reinterpret_cast<short4*>(pd + v * 4) = make_short4(pcm16_of(s_out[v * 4]), pcm16_of(s_out[v * 4 + 1]),
                                                             pcm16_of(s_out[v * 4 + 2]), pcm16_of(s_out[v * 4 + 3]));
      } else {
        for (int e = 0; v * 4 + e < count; e++) pd[v * 4 + e] = pcm16_of(s_out[v * 4 + e]);
      }
    }
  }
}
void launch_istft(const float* cp, int ldc, const int* h_off, const int* h_len, float* audio, short* pcm,
                  const long long* s_off, int fast, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  if (ldc != 24 || (reinterpret_cast<uintptr_t>(cp) & 15)) throw ArgError("launch_istft: conv_post rows must have pitch 24 and 16-byte alignment");
  ensure_tables();
  // groups q = 2 .. F of an item with F = max_len frames -> F - 1 groups
  dim3 g((max_len - 1 + kIstftGroups - 1) / kIstftGroups > 0 ? (max_len - 1 + kIstftGroups - 1) / kIstftGroups : 1, B);
  if (fast) istft_kernel<true><<<g, 128, 0, st>>>(cp, ldc, h_off, h_len, audio, s_off, pcm);
  else istft_kernel<false><<<g, 128, 0, st>>>(cp, ldc, h_off, h_len, audio, s_off, pcm);
  post_launch("istft", st);
}

// ------------------------------------------------------------------------------------------
// Output sample-rate conversion: 24 kHz -> out_rate by the polyphase FIR of scipy.signal.resample_poly (its defaults:
// Kaiser beta 5, half length 10 * max(U, D)), each utterance on its own with zeros outside it.
bool resample_ratio(int out_rate, int* U, int* D) {
  if (out_rate < 8000 || out_rate > 48000) return false;
  const int g = std::gcd(out_rate, 24000);
  *U = out_rate / g;
  *D = 24000 / g;
  return std::max(*U, *D) <= 320;
}

static double bessel_i0(double x) {   // power series of the modified Bessel function I0 (x <= 5 here: ~25 terms)
  double sum = 1.0, term = 1.0;
  const double q = 0.25 * x * x;
  for (int k = 1; k < 200; k++) {
    term *= q / ((double)k * k);
    sum += term;
    if (term < 1e-17 * sum) break;
  }
  return sum;
}

int resample_design(int out_rate, std::vector<float>* taps, int* U, int* D, int* H) {
  int u = 0, d = 0;
  if (!resample_ratio(out_rate, &u, &d)) return -1;
  if (u == 1 && d == 1) {   // 24 kHz: the identity (resample_poly returns its input), the pass-through mode's H = 0
    if (taps) taps->assign(1, 1.0f);
    if (U) *U = 1;
    if (D) *D = 1;
    if (H) *H = 0;
    return 1;
  }
  if (U) *U = u;
  if (D) *D = d;
  if (H) *H = 10 * std::max(u, d);
  return poly_design(u, d, taps);
}

int poly_design(int u, int d, std::vector<float>* taps) {
  const int half = 10 * std::max(u, d), n = 2 * half + 1;
  // U * firwin(2H + 1, 1 / max(U, D), window = ("kaiser", 5.0)), in double: windowed sinc, normalised to unit DC gain
  const double fc = 1.0 / std::max(u, d), beta = 5.0, i0b = bessel_i0(beta);
  std::vector<double> h(n);
  double sum = 0.0;
  for (int i = 0; i < n; i++) {
    const double m = i - half, a = fc * m;
    const double sinc = m == 0 ? 1.0 : std::sin(M_PI * a) / (M_PI * a);
    const double r = m / half;
    h[i] = fc * sinc * bessel_i0(beta * std::sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
    sum += h[i];
  }
  if (taps) {
    taps->resize(n);
    for (int i = 0; i < n; i++) (*taps)[i] = (float)(u * (h[i] / sum));
  }
  return n;
}

// ITU-T G.711 of a 16-bit sample, Sun reference g711.c (what audioop.lin2ulaw / lin2alaw(..., 2) return):
// mu-law from the 14-bit value p >> 2 (bias 33, clip 8159), A-law from the 13-bit value p >> 3.
__device__ __forceinline__ unsigned char g711_ulaw(int p) {
  int v = p >> 2;
  const int mask = v < 0 ? 0x7F : 0xFF;
  v = min(abs(v), 8159) + 33;                       // 34 .. 8192: segment = position of the top bit above bit 5
  const int seg = max(0, 31 - __clz(v) - 5);        // first seg with v <= 0x3F << seg (v <= 8192 -> seg <= 7)
  if (seg >= 8) return (unsigned char)(0x7F ^ mask);
  return (unsigned char)(((seg << 4) | ((v >> (seg + 1)) & 0xF)) ^ mask);
}
__device__ __forceinline__ unsigned char g711_alaw(int p) {
  int v = p >> 3;
  const int mask = v >= 0 ? 0xD5 : 0x55;
  if (v < 0) v = -v - 1;                            // 0 .. 4095
  const int seg = max(0, 31 - __clz(v | 1) - 4);    // first seg with v <= 0x1F << seg
  const int q = (seg < 2 ? v >> 1 : v >> seg) & 0xF;
  return (unsigned char)(((seg << 4) | q) ^ mask);
}

// y_b[m] = sum over k ascending (0 <= k < n_b, 0 <= m D - k U + H <= 2H) of x_b[k] * taps[m D - k U + H], fp32 FMA.
// Grid (output tiles of kRsTile = 2048 samples, items), 256 threads, 8 outputs per thread.  The CTA stages the
// input span its tile reads (zero outside the item) and all 2H + 1 taps in shared memory with coalesced loads.  Each
// output sample is a function of its item alone, so results do not depend on the batch around it.  Output offsets
// need not be multiples of 4 (at 11025 / 22050 / 44100 Hz they are not): every store is a scalar, coalesced across
// the warp.  PASS: U = D = 1 without a filter (the G.711 codes of the 24 kHz waveform itself).  gain (nullable): y of
// item b becomes fp32(y * gain[b]) before any output is written; without it the arithmetic is the plain filter's.
constexpr int kRsThreads = 256, kRsPer = 8, kRsTile = kRsThreads * kRsPer;
__host__ __device__ inline long long floor_div(long long a, long long b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

template <bool PASS>
__global__ void __launch_bounds__(kRsThreads) resample_kernel(const float* __restrict__ x, const long long* __restrict__ in_off,
                                                              const long long* __restrict__ in_len,
                                                              const long long* __restrict__ out_off,
                                                              const float* __restrict__ taps, int U, int D, int H,
                                                              const float* __restrict__ gain,
                                                              float* __restrict__ out, short* __restrict__ pcm,
                                                              unsigned char* __restrict__ codes, int law) {
  extern __shared__ float rs_smem[];
  const int b = blockIdx.y, t = threadIdx.x;
  const long long n = in_len[b];
  const long long n_out = (n * U + D - 1) / D;
  const long long m0 = (long long)blockIdx.x * kRsTile;
  if (m0 >= n_out) return;
  const float* xb = x + in_off[b];
  const long long ob = out_off[b];
  float y[kRsPer];
  if (PASS) {
#pragma unroll
    for (int i = 0; i < kRsPer; i++) {
      const long long m = m0 + t + i * kRsThreads;
      y[i] = m < n_out ? xb[m] : 0.f;
    }
  } else {
    const int ntap = 2 * H + 1;
    float* s_h = rs_smem;
    float* s_x = rs_smem + ((ntap + 3) & ~3);
    const long long m1 = min(m0 + kRsTile, n_out) - 1;
    const long long k0 = floor_div(m0 * D - H + U - 1, U);   // ceil((m0 D - H) / U): first input any output reads
    const long long k1 = floor_div(m1 * D + H, U);
    const int span = (int)(k1 - k0 + 1);
    for (int i = t; i < ntap; i += kRsThreads) s_h[i] = __ldg(taps + i);
    for (int i = t; i < span; i += kRsThreads) {
      const long long k = k0 + i;
      s_x[i] = (k >= 0 && k < n) ? __ldg(xb + k) : 0.f;
    }
    __syncthreads();
    // tile-relative 32-bit index math: a = m D - k0 U lies in (H - U, H + (kRsTile - 1) D]; k counts from k0
    const int a0 = (int)(m0 * D - k0 * U);
    const int kfirst = (int)max(-k0, 0LL);                       // input index >= 0
    const int klast = (int)(min(n - 1, k1) - k0);                // input index < n
#pragma unroll
    for (int i = 0; i < kRsPer; i++) {
      const int r = t + i * kRsThreads;
      float acc = 0.f;
      if (m0 + r < n_out) {
        const int a = a0 + r * D;
        int k = a > H ? (int)((unsigned)(a - H + U - 1) / (unsigned)U) : 0;   // ceil((a - H) / U): first tap <= 2H
        k = max(k, kfirst);
        // tap of input k is j = a - k U + H; the filter ends where j < 0
        for (int j = a - k * U + H; k <= klast && j >= 0; k++, j -= U) acc = fmaf(s_x[k], s_h[j], acc);
      }
      y[i] = acc;
    }
  }
  if (gain) {   // loudness normalisation: fp32(y * g), one gain per item (kernels_loudness.cu)
    const float g = gain[b];
#pragma unroll
    for (int i = 0; i < kRsPer; i++) y[i] = __fmul_rn(y[i], g);
  }
#pragma unroll
  for (int i = 0; i < kRsPer; i++) {
    const long long m = m0 + t + i * kRsThreads;
    if (m >= n_out) break;
    out[ob + m] = y[i];
    if (pcm || codes) {
      const short p = pcm16_of(y[i]);
      if (pcm) pcm[ob + m] = p;
      if (codes) codes[ob + m] = law ? g711_alaw(p) : g711_ulaw(p);
    }
  }
}

size_t resample_smem_bytes(int U, int D, int H) {
  if (U == 1 && D == 1 && H == 0) return 0;
  const long long span = ((long long)(kRsTile - 1) * D + 2 * H) / U + 2;
  return (size_t)(((2 * H + 1 + 3) & ~3) + span) * sizeof(float);
}

void launch_resample(const float* x, const long long* in_off, const long long* in_len, const long long* out_off,
                     const float* taps, int U, int D, int H, const float* gain, float* out, short* pcm,
                     unsigned char* codes, int law, int B, long long max_out, cudaStream_t st) {
  if (g_dry_run) return;
  const bool pass = U == 1 && D == 1 && H == 0;
  if (!pass && !taps) throw ArgError("launch_resample: filter taps missing");
  if (max_out <= 0) return;
  const long long tiles = (max_out + kRsTile - 1) / kRsTile;
  if (tiles > 0x7FFFFFFFLL || B > 65535) throw ArgError("launch_resample: grid too large");
  // at most 42.6 KB (11 025 Hz: 6404 taps + a 4501-sample span), inside the default 48 KB of dynamic shared memory
  const size_t smem = resample_smem_bytes(U, D, H);
  if (smem > 48 * 1024) throw ArgError("launch_resample: filter too long for one CTA");
  dim3 g((unsigned)tiles, B);
  if (pass)
    resample_kernel<true><<<g, kRsThreads, 0, st>>>(x, in_off, in_len, out_off, nullptr, 1, 1, 0, gain, out, pcm, codes,
                                                    law);
  else
    resample_kernel<false><<<g, kRsThreads, smem, st>>>(x, in_off, in_len, out_off, taps, U, D, H, gain, out, pcm, codes,
                                                        law);
  post_launch("resample", st);
}

// ------------------------------------------------------------------------------------------
// TTSKoko::mix_styles on the device (koko.rs:1255-1306): style_b[j] = sum_i table[voice_i][row_b][j] * portion_i,
// accumulated in the reference's order with separate multiply and add (no FMA contraction), so the result is
// bit-identical to the Rust loop; a single voice is portion 1.0 and therefore an exact copy.
__global__ void __launch_bounds__(256) mix_styles_kernel(const float* __restrict__ table, const int* mix_off,
                                                         const int* voice_ids, const float* portions,
                                                         const int* rows, float* styles) {
  const int b = blockIdx.x, j = threadIdx.x;
  float acc = 0.0f;
  for (int i = mix_off[b]; i < mix_off[b + 1]; i++)
    acc = __fadd_rn(acc, __fmul_rn(table[((size_t)voice_ids[i] * 511 + rows[b]) * 256 + j], portions[i]));
  styles[(size_t)b * 256 + j] = acc;
}
void launch_mix_styles(const float* table, const int* mix_off, const int* voice_ids, const float* portions,
                       const int* rows, float* styles, int B, cudaStream_t st) {
  if (g_dry_run) return;
  mix_styles_kernel<<<B, 256, 0, st>>>(table, mix_off, voice_ids, portions, rows, styles);
  post_launch("mix_styles", st);
}

}  // namespace kkx
