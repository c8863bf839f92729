// kernels_dense.cu -- fp32 SIMT shifted-GEMM (Conv1d / Linear), LayerNorm, attention, LSTM.
// These carry the precision-critical predictor path (ALBERT -> durations -> F0/N), where the
// integer frame durations must match the oracle bit for bit, and serve as the fp32 reference
// configuration ("precision"=0) for the decoder/generator.
#include "kernels.h"
#include <cuda_fp16.h>
#include <math.h>
#include "tc_ptx.cuh"

namespace kkx {

thread_local LaunchStats* g_launch_stats = nullptr;

__device__ __forceinline__ float act_apply(float v, int act, float slope, float alpha) {
  if (act == ACT_LRELU) return v > 0.f ? v : v * slope;
  if (act == ACT_SNAKE) {
    float s = sinf(alpha * v);
    return v + (1.0f / alpha) * (s * s);
  }
  if (act == ACT_GELU_NEW) {
    // 0.5*x*(1+tanh(sqrt(2/pi)*(x+0.044715*x^3)))
    float u = 0.7978845608028654f * (v + 0.044715f * v * v * v);
    return 0.5f * v * (1.0f + tanhf(u));
  }
  return v;
}

// ------------------------------------------------------------------------------------------
// Shifted GEMM.  256 threads, BMxBN output tile, BK=16; thread (ty,tx) owns rows ty+16*i and
// columns tx+16*j so that smem reads are conflict-free/broadcast and global stores coalesce.
template <int BM, int BN>
__global__ void __launch_bounds__(256) conv_f32_kernel(ConvArgs a) {
  constexpr int BK = 16, TM = BM / 16, TN = BN / 16;
  __shared__ float As[BK][BM + 1];
  __shared__ float Bs[BK][BN];
  const int b = blockIdx.z;
  const int mlen = a.m_len[b];
  const int m0 = blockIdx.x * BM;
  if (m0 >= mlen) return;
  const int n0 = blockIdx.y * BN;
  const int in_off = a.in_off[b], in_len = a.in_len[b];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const float* psc = a.pscale ? a.pscale + (size_t)b * a.pld : nullptr;
  const float* psh = a.pshift ? a.pshift + (size_t)b * a.pld : nullptr;
  const bool prologue = (psc != nullptr) || (a.pact != ACT_NONE);

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; i++)
#pragma unroll
    for (int j = 0; j < TN; j++) acc[i][j] = 0.f;

  for (int tap = 0; tap < a.ks; tap++) {
    const int shift = tap * a.dil - a.pad;
    for (int c0 = 0; c0 < a.Ci; c0 += BK) {
      // A tile: BM x BK, channel index fastest across threads
      for (int i = tid; i < BM * BK; i += 256) {
        const int kk = i & (BK - 1), m = i >> 4;
        const int c = c0 + kk, mm = m0 + m;
        float v = 0.f;
        if (c < a.Ci && mm < mlen) {
          const int r = mm * a.stride + shift;
          if (r >= 0 && r < in_len) {
            v = a.in[(size_t)(in_off + r) * a.ldi + c];
            if (prologue) {
              if (psc) v = v * psc[c] + psh[c];
              v = act_apply(v, a.pact, a.pslope, a.palpha ? a.palpha[c] : 1.f);
            }
          }
        }
        As[kk][m] = v;
      }
      // B tile: BK x BN, output channel fastest
      for (int i = tid; i < BK * BN; i += 256) {
        const int nn = i % BN, kk = i / BN;
        const int c = c0 + kk, n = n0 + nn;
        Bs[kk][nn] = (c < a.Ci && n < a.Co) ? a.w[((size_t)tap * a.Ci + c) * a.Co + n] : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < BK; kk++) {
        float ar[TM], br[TN];
#pragma unroll
        for (int i = 0; i < TM; i++) ar[i] = As[kk][ty + 16 * i];
#pragma unroll
        for (int j = 0; j < TN; j++) br[j] = Bs[kk][tx + 16 * j];
#pragma unroll
        for (int i = 0; i < TM; i++)
#pragma unroll
          for (int j = 0; j < TN; j++) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
      }
      __syncthreads();
    }
  }

  const int out_off = a.out_off[b];
  const int res_off = a.res ? a.res_off[b] : 0;
#pragma unroll
  for (int i = 0; i < TM; i++) {
    const int mm = m0 + ty + 16 * i;
    if (mm >= mlen) continue;
    const int orow = mm * a.ors + a.oro;
    float* op = a.out + (size_t)(out_off + orow) * a.ldo + a.ocol;
    const float* rp = a.res ? a.res + (size_t)(res_off + (orow >> a.res_shift)) * a.ldr + a.rcol : nullptr;
#pragma unroll
    for (int j = 0; j < TN; j++) {
      const int n = n0 + tx + 16 * j;
      if (n >= a.Co) continue;
      float v = acc[i][j] + (a.bias ? a.bias[n] : 0.f);
      v = act_apply(v, a.eact, 0.f, 1.f);
      if (rp) v += rp[n];
      v *= a.oscale;
      if (a.accumulate) v += op[n];
      op[n] = v;
    }
  }
}

void launch_conv_f32(const ConvArgs& a, cudaStream_t st) {
  if (g_dry_run) return;
  if (a.max_m <= 0 || a.B <= 0) return;
  if (g_launch_stats) g_launch_stats->conv_flops += 2.0 * (double)a.sum_m * a.Co * a.Ci * a.ks;
  // tile choice: big tiles when there is enough work to fill 148 SMs, small ones otherwise
  const long long tiles128 = (long long)((a.max_m + 127) / 128) * ((a.Co + 127) / 128) * a.B;
  if (a.Co >= 128 && tiles128 >= 148) {
    dim3 g((a.max_m + 127) / 128, (a.Co + 127) / 128, a.B);
    conv_f32_kernel<128, 128><<<g, 256, 0, st>>>(a);
  } else if (a.Co > 32) {
    dim3 g((a.max_m + 63) / 64, (a.Co + 63) / 64, a.B);
    conv_f32_kernel<64, 64><<<g, 256, 0, st>>>(a);
  } else {
    dim3 g((a.max_m + 127) / 128, (a.Co + 31) / 32, a.B);
    conv_f32_kernel<128, 32><<<g, 256, 0, st>>>(a);
  }
  if (g_launch_stats && g_launch_stats->profile && g_launch_stats->detail) {
    char nm[96]; snprintf(nm, sizeof nm, "conv_f32[ci%d co%d k%d s%d m%lld]", a.Ci, a.Co, a.ks, a.stride, a.sum_m);
    post_launch(nm, st);
  } else post_launch("conv_f32", st);
}

// ------------------------------------------------------------------------------------------
// LayerNorm over the channel axis: one warp per row, two-pass (mean, then centred variance).
__global__ void __launch_bounds__(256) layernorm_kernel(LnArgs a) {
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * 8 + warp;
  if (t >= a.len[b]) return;
  const size_t row = (size_t)a.off[b] + t;
  const float* x = a.x + row * a.ldx;
  const float* r = a.res ? a.res + row * a.ldr : nullptr;
  const int C = a.C;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) s += x[c] + (r ? r[c] : 0.f);
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)C;
  float q = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float d = x[c] + (r ? r[c] : 0.f) - mean;
    q = fmaf(d, d, q);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = 1.0f / sqrtf(q / (float)C + a.eps);
  const float* ada = a.ada ? a.ada + (size_t)b * a.ada_ld + a.ada_off : nullptr;
  float* o = a.out + row * a.ldo + a.ocol;
  for (int c = lane; c < C; c += 32) {
    float v = (x[c] + (r ? r[c] : 0.f) - mean) * rstd;
    if (a.w) v = v * a.w[c] + a.b[c];
    if (ada) v = (1.0f + ada[c]) * v + ada[C + c];
    if (a.slope != 1.f) v = v > 0.f ? v : v * a.slope;
    o[c] = v;
    if (a.pl_hi) {   // operand planes for the next split-FP16 GEMM
      uint32_t hi, lo;
      split_f16_operand(v, hi, lo);
      static_cast<uint16_t*>(a.pl_hi)[row * a.pl_ld + c] = (uint16_t)hi;
      static_cast<uint16_t*>(a.pl_lo)[row * a.pl_ld + c] = (uint16_t)lo;
    }
  }
}

// The same row normalisation with the row held in registers: one 128-bit load per 4 channels (x and the residual are
// read ONCE instead of three times), 128-bit stores of the fp32 result and 64-bit stores of the operand planes.  A lane
// owns channels 4 (lane + 32 i) .. + 3, i < NV = C / 128.  (The scalar kernel above made three passes of 4-byte
// accesses and 2-byte plane stores: ~3 TB/s on the 32 768 x 768 ALBERT rows.)
template <int NV>
__global__ void __launch_bounds__(256) layernorm_vec_kernel(LnArgs a) {
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * 8 + warp;
  if (t >= a.len[b]) return;
  const size_t row = (size_t)a.off[b] + t;
  const float4* x4 = reinterpret_cast<const float4*>(a.x + row * a.ldx);
  const float4* r4 = a.res ? reinterpret_cast<const float4*>(a.res + row * a.ldr) : nullptr;
  constexpr int C = NV * 128;
  float4 v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; i++) {
    v[i] = x4[lane + 32 * i];
    if (r4) { const float4 rr = r4[lane + 32 * i]; v[i].x += rr.x; v[i].y += rr.y; v[i].z += rr.z; v[i].w += rr.w; }
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; i++) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    q = fmaf(v[i].x, v[i].x, q); q = fmaf(v[i].y, v[i].y, q); q = fmaf(v[i].z, v[i].z, q); q = fmaf(v[i].w, v[i].w, q);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = 1.0f / sqrtf(q / (float)C + a.eps);
  const float* ada = a.ada ? a.ada + (size_t)b * a.ada_ld + a.ada_off : nullptr;
  float* o = a.out + row * a.ldo + a.ocol;
#pragma unroll
  for (int i = 0; i < NV; i++) {
    const int c = 4 * (lane + 32 * i);
    float e[4] = {v[i].x * rstd, v[i].y * rstd, v[i].z * rstd, v[i].w * rstd};
    if (a.w) {
      const float4 w4 = *reinterpret_cast<const float4*>(a.w + c), b4 = *reinterpret_cast<const float4*>(a.b + c);
      e[0] = e[0] * w4.x + b4.x; e[1] = e[1] * w4.y + b4.y; e[2] = e[2] * w4.z + b4.z; e[3] = e[3] * w4.w + b4.w;
    }
    if (ada) {
      const float4 g4 = *reinterpret_cast<const float4*>(ada + c), h4 = *reinterpret_cast<const float4*>(ada + C + c);
      e[0] = (1.0f + g4.x) * e[0] + h4.x; e[1] = (1.0f + g4.y) * e[1] + h4.y;
      e[2] = (1.0f + g4.z) * e[2] + h4.z; e[3] = (1.0f + g4.w) * e[3] + h4.w;
    }
    if (a.slope != 1.f) {
#pragma unroll
      for (int k = 0; k < 4; k++) e[k] = e[k] > 0.f ? e[k] : e[k] * a.slope;
    }
    *reinterpret_cast<float4*>(o + c) = make_float4(e[0], e[1], e[2], e[3]);
    if (a.pl_hi) {   // operand planes for the next split-FP16 GEMM
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int k = 0; k < 4; k++) split_f16_operand(e[k], hi[k], lo[k]);
      *reinterpret_cast<uint2*>(static_cast<uint16_t*>(a.pl_hi) + row * a.pl_ld + c) = make_uint2(hi[0] | (hi[1] << 16), hi[2] | (hi[3] << 16));
      *reinterpret_cast<uint2*>(static_cast<uint16_t*>(a.pl_lo) + row * a.pl_ld + c) = make_uint2(lo[0] | (lo[1] << 16), lo[2] | (lo[3] << 16));
    }
  }
}

void launch_layernorm(const LnArgs& a, cudaStream_t st) {
  if (g_dry_run) return;
  if (a.max_len <= 0) return;
  dim3 g((a.max_len + 7) / 8, a.B);
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool vec = a.C % 128 == 0 && a.C <= 1024 && a.ldx % 4 == 0 && a.ldo % 4 == 0 && a.ocol % 4 == 0 && al16(a.x) && al16(a.out) &&
                   (!a.res || (a.ldr % 4 == 0 && al16(a.res))) && (!a.w || (al16(a.w) && al16(a.b))) &&
                   (!a.ada || (a.ada_ld % 4 == 0 && a.ada_off % 4 == 0 && al16(a.ada))) &&
                   (!a.pl_hi || (a.pl_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(a.pl_hi) & 7) == 0 && (reinterpret_cast<uintptr_t>(a.pl_lo) & 7) == 0));
  // one choice per shape, never per batch: a batch and its single calls take the same kernel
  if (vec && a.C == 768) layernorm_vec_kernel<6><<<g, 256, 0, st>>>(a);
  else if (vec && a.C == 512) layernorm_vec_kernel<4><<<g, 256, 0, st>>>(a);
  else if (vec && a.C == 1024) layernorm_vec_kernel<8><<<g, 256, 0, st>>>(a);
  else if (vec && a.C == 256) layernorm_vec_kernel<2><<<g, 256, 0, st>>>(a);
  else if (vec && a.C == 128) layernorm_vec_kernel<1><<<g, 256, 0, st>>>(a);
  else layernorm_kernel<<<g, 256, 0, st>>>(a);
  post_launch("layernorm", st);
}

// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) albert_embed_kernel(const int* ids, const float* word,
                                                           const float* pos, const float* type,
                                                           const float* lnw, const float* lnb,
                                                           float* out, const int* off,
                                                           const int* len) {
  const int b = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int t = blockIdx.x * 8 + warp;
  if (t >= len[b]) return;
  const size_t row = (size_t)off[b] + t;
  const int id = ids[row];
  float v[4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int c = lane + 32 * i;
    v[i] = word[id * 128 + c] + type[c] + pos[t * 128 + c];
    s += v[i];
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * (1.0f / 128.f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 4; i++) { const float d = v[i] - mean; q = fmaf(d, d, q); }
#pragma unroll
  for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = 1.0f / sqrtf(q * (1.0f / 128.f) + 1e-12f);
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int c = lane + 32 * i;
    out[row * 128 + c] = (v[i] - mean) * rstd * lnw[c] + lnb[c];
  }
}

void launch_albert_embed(const int* ids, const float* word, const float* pos, const float* type,
                         const float* lnw, const float* lnb, float* out, const int* off,
                         const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 7) / 8, B);
  albert_embed_kernel<<<g, 256, 0, st>>>(ids, word, pos, type, lnw, lnb, out, off, len);
  post_launch("albert_embed", st);
}

__global__ void __launch_bounds__(256) embed_rows_kernel(const int* ids, const float* table, int C,
                                                         float* out, int ldo, const int* off,
                                                         const int* len) {
  const int b = blockIdx.y, t = blockIdx.x;
  if (t >= len[b]) return;
  const size_t row = (size_t)off[b] + t;
  const int id = ids[row];
  for (int c = threadIdx.x; c < C; c += blockDim.x) out[row * ldo + c] = table[(size_t)id * C + c];
}
void launch_embed_rows(const int* ids, const float* table, int C, float* out, int ldo,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g(max_len, B);
  embed_rows_kernel<<<g, 256, 0, st>>>(ids, table, C, out, ldo, off, len);
  post_launch("embed_rows", st);
}

__global__ void __launch_bounds__(256) bcast_cols_kernel(const float* vec, int ldv, int voff, int C,
                                                         float* out, int ldo, int ocol,
                                                         const int* off, const int* len) {
  const int b = blockIdx.y;
  const int rows_per_block = 256 / 32;
  const int t = blockIdx.x * rows_per_block + (threadIdx.x >> 5);
  if (t >= len[b]) return;
  const size_t row = (size_t)off[b] + t;
  for (int c = threadIdx.x & 31; c < C; c += 32) out[row * ldo + ocol + c] = vec[(size_t)b * ldv + voff + c];
}
void launch_bcast_cols(const float* vec, int ldv, int voff, int C, float* out, int ldo, int ocol,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 7) / 8, B);
  bcast_cols_kernel<<<g, 256, 0, st>>>(vec, ldv, voff, C, out, ldo, ocol, off, len);
  post_launch("bcast_cols", st);
}

__global__ void __launch_bounds__(256) copy_cols_kernel(const float* src, int lds, int scol,
                                                        float* dst, int ldd, int dcol, int C,
                                                        const int* off, const int* len) {
  const int b = blockIdx.y;
  const int t = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (t >= len[b]) return;
  const size_t row = (size_t)off[b] + t;
  for (int c = threadIdx.x & 31; c < C; c += 32) dst[row * ldd + dcol + c] = src[row * lds + scol + c];
}
void launch_copy_cols(const float* src, int lds, int scol, float* dst, int ldd, int dcol, int C,
                      const int* off, const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  dim3 g((max_len + 7) / 8, B);
  copy_cols_kernel<<<g, 256, 0, st>>>(src, lds, scol, dst, ldd, dcol, C, off, len);
  post_launch("copy_cols", st);
}

__global__ void __launch_bounds__(256) add_rows_kernel(const float* a, const float* b2, float* out,
                                                       int C, const int* off, const int* len) {
  const int b = blockIdx.y;
  const size_t n = (size_t)len[b] * C;
  const size_t base = (size_t)off[b] * C;
  for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256)
    out[base + i] = a[base + i] + b2[base + i];
}
void launch_add_rows(const float* a, const float* b, float* out, int C, const int* off,
                     const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  long long blocks = ((long long)max_len * C + 256 * 8 - 1) / (256 * 8);
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 16) blocks = 148 * 16;
  dim3 g((unsigned)blocks, B);
  add_rows_kernel<<<g, 256, 0, st>>>(a, b, out, C, off, len);
  post_launch("add_rows", st);
}

__global__ void copy_row_kernel(float* u, int C, int dst_row, int src_row, const int* off) {
  const int b = blockIdx.x;
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    u[(size_t)(off[b] + dst_row) * C + c] = u[(size_t)(off[b] + src_row) * C + c];
}
void launch_copy_row(float* u, int C, int dst_row, int src_row, const int* off, int B,
                     cudaStream_t st) {
  if (g_dry_run) return;
  copy_row_kernel<<<B, 128, 0, st>>>(u, C, dst_row, src_row, off);
  post_launch("copy_row", st);
}

// ------------------------------------------------------------------------------------------
// ALBERT self-attention (12 heads x 64), flash-style online softmax in fp32, with split-TF32 ("3xTF32") products on
// mma.sync m16n8k8, which
// keeps fp32-grade accuracy (this path feeds the duration predictor, whose integer durations must match
// the fp32 oracle bit-exactly) at several times the fp32 SIMT rate.  Attention is ~0.5 % of the model's
// FLOPs, with d = 64 and N <= 512: the warp-level MMA with register fragments fits it better than a
// TMEM pipeline.  CTA = 4 warps x 16 query rows; keys/values stream through smem in tiles of 64 as
// tf32 hi/lo planes; every product is hi*hi + hi*lo + lo*hi.
//   S = (Q/8) K^T : A = Q fragments (registers, split once), B[k=d][n=key] = K[key][d]
//   O += P V      : A = P in the accumulator layout with the key order (2t, 2t+1) taken as k = (t, t+4),
//                   so no shuffles are needed; B[k=key][n=d] = V[key][d] with the same key permutation.
__device__ __forceinline__ uint32_t att_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return r;
}
__device__ __forceinline__ void att_mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
constexpr int kAttLd = 68;   // smem row stride (floats): conflict-free B-fragment loads for both products

template <int NW>   // warps per CTA: NW*16 query rows share every staged K/V tile
__global__ void __launch_bounds__(NW * 32) attention_tc_kernel(const float* __restrict__ qkv, float* __restrict__ ctx,
                                                               const int* off, const int* len) {
  extern __shared__ uint32_t att_sm[];
  uint32_t* Kh = att_sm;                       // [64][68] tf32 hi
  uint32_t* Kl = Kh + 64 * kAttLd;
  uint32_t* Vh = Kl + 64 * kAttLd;
  uint32_t* Vl = Vh + 64 * kAttLd;
  const int b = blockIdx.z, h = blockIdx.y;
  const int N = len[b];
  const int q0 = blockIdx.x * (NW * 16);
  if (q0 >= N) return;
  const size_t base = (size_t)off[b];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;       // the two query rows of this thread's fragments

  // Q fragments (scaled by 1/8, exact), split into tf32 hi / lo once
  uint32_t qh[8][4], ql[8][4];
#pragma unroll
  for (int kk = 0; kk < 8; kk++) {
    const int d = kk * 8 + t;
    const float* p0 = qkv + (base + r0) * 2304 + h * 64 + d;
    const float* p1 = qkv + (base + r1) * 2304 + h * 64 + d;
    float v[4];
    v[0] = r0 < N ? p0[0] * 0.125f : 0.f;
    v[1] = r1 < N ? p1[0] * 0.125f : 0.f;
    v[2] = r0 < N ? p0[4] * 0.125f : 0.f;
    v[3] = r1 < N ? p1[4] * 0.125f : 0.f;
#pragma unroll
    for (int e = 0; e < 4; e++) {
      qh[kk][e] = att_tf32(v[e]);
      ql[kk][e] = att_tf32(v[e] - __uint_as_float(qh[kk][e]));
    }
  }
  float o[8][4];
#pragma unroll
  for (int n = 0; n < 8; n++) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

  // K/V tiles are fetched one tile ahead into registers (the loads fly during the MMAs of the current tile),
  // then split into tf32 hi/lo planes and stored to smem
  constexpr int NLD = 1024 / (NW * 32);        // float4 per thread, matrix and tile
  float4 kreg[NLD], vreg[NLD];
  auto prefetch = [&](int k0) {
#pragma unroll
    for (int u = 0; u < NLD; u++) {
      const int i = tid + u * (NW * 32);
      const int j = i >> 4, c4 = (i & 15) << 2;
      kreg[u] = make_float4(0.f, 0.f, 0.f, 0.f); vreg[u] = kreg[u];
      if (k0 + j < N) {
        const float* rp = qkv + (base + k0 + j) * 2304 + h * 64 + c4;
        kreg[u] = *reinterpret_cast<const float4*>(rp + 768);
        vreg[u] = *reinterpret_cast<const float4*>(rp + 1536);
      }
    }
  };
  prefetch(0);
  for (int k0 = 0; k0 < N; k0 += 64) {
    __syncthreads();
#pragma unroll
    for (int u = 0; u < NLD; u++) {
      const int i = tid + u * (NW * 32);
      const int j = i >> 4, c4 = (i & 15) << 2;
      const float kx[4] = {kreg[u].x, kreg[u].y, kreg[u].z, kreg[u].w}, vx[4] = {vreg[u].x, vreg[u].y, vreg[u].z, vreg[u].w};
      uint32_t a[4], bq[4], c[4], dq[4];
#pragma unroll
      for (int e = 0; e < 4; e++) {
        a[e] = att_tf32(kx[e]); bq[e] = att_tf32(kx[e] - __uint_as_float(a[e]));
        c[e] = att_tf32(vx[e]); dq[e] = att_tf32(vx[e] - __uint_as_float(c[e]));
      }
      *reinterpret_cast<uint4*>(Kh + j * kAttLd + c4) = make_uint4(a[0], a[1], a[2], a[3]);
      *reinterpret_cast<uint4*>(Kl + j * kAttLd + c4) = make_uint4(bq[0], bq[1], bq[2], bq[3]);
      *reinterpret_cast<uint4*>(Vh + j * kAttLd + c4) = make_uint4(c[0], c[1], c[2], c[3]);
      *reinterpret_cast<uint4*>(Vl + j * kAttLd + c4) = make_uint4(dq[0], dq[1], dq[2], dq[3]);
    }
    __syncthreads();
    if (k0 + 64 < N) prefetch(k0 + 64);

    // S = Q K^T for 16 rows x 64 keys
    float sc[8][4];
#pragma unroll
    for (int n = 0; n < 8; n++) {
      sc[n][0] = sc[n][1] = sc[n][2] = sc[n][3] = 0.f;
      const uint32_t* kh = Kh + (n * 8 + g) * kAttLd + t;
      const uint32_t* kl = Kl + (n * 8 + g) * kAttLd + t;
#pragma unroll
      for (int kk = 0; kk < 8; kk++) {
        const uint32_t bh0 = kh[kk * 8], bh1 = kh[kk * 8 + 4], bl0 = kl[kk * 8], bl1 = kl[kk * 8 + 4];
        att_mma(sc[n], ql[kk], bh0, bh1);     // small terms first
        att_mma(sc[n], qh[kk], bl0, bl1);
        att_mma(sc[n], qh[kk], bh0, bh1);
      }
    }
    // online softmax (rows r0: elements 0,1; rows r1: elements 2,3); keys beyond N masked out
    float cm0 = -INFINITY, cm1 = -INFINITY;
#pragma unroll
    for (int n = 0; n < 8; n++) {
      const int key = k0 + n * 8 + 2 * t;
      if (key >= N) { sc[n][0] = -INFINITY; sc[n][2] = -INFINITY; }
      if (key + 1 >= N) { sc[n][1] = -INFINITY; sc[n][3] = -INFINITY; }
      cm0 = fmaxf(cm0, fmaxf(sc[n][0], sc[n][1]));
      cm1 = fmaxf(cm1, fmaxf(sc[n][2], sc[n][3]));
    }
    cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 1)); cm0 = fmaxf(cm0, __shfl_xor_sync(0xffffffffu, cm0, 2));
    cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 1)); cm1 = fmaxf(cm1, __shfl_xor_sync(0xffffffffu, cm1, 2));
    const float mn0 = fmaxf(m0, cm0), mn1 = fmaxf(m1, cm1);   // finite: every tile holds at least one valid key
    const float corr0 = expf(m0 - mn0), corr1 = expf(m1 - mn1);
    float ps0 = 0.f, ps1 = 0.f;
#pragma unroll
    for (int n = 0; n < 8; n++) {
      sc[n][0] = expf(sc[n][0] - mn0); sc[n][1] = expf(sc[n][1] - mn0);
      sc[n][2] = expf(sc[n][2] - mn1); sc[n][3] = expf(sc[n][3] - mn1);
      ps0 += sc[n][0] + sc[n][1];
      ps1 += sc[n][2] + sc[n][3];
    }
    ps0 += __shfl_xor_sync(0xffffffffu, ps0, 1); ps0 += __shfl_xor_sync(0xffffffffu, ps0, 2);
    ps1 += __shfl_xor_sync(0xffffffffu, ps1, 1); ps1 += __shfl_xor_sync(0xffffffffu, ps1, 2);
    l0 = l0 * corr0 + ps0; l1 = l1 * corr1 + ps1;
    m0 = mn0; m1 = mn1;
#pragma unroll
    for (int n = 0; n < 8; n++) { o[n][0] *= corr0; o[n][1] *= corr0; o[n][2] *= corr1; o[n][3] *= corr1; }

    // O += P V: k-step kk covers keys kk*8 .. +7; fragment column t <-> key 2t, column t+4 <-> key 2t+1
#pragma unroll
    for (int kk = 0; kk < 8; kk++) {
      uint32_t ph[4], pl[4];
      const float pv[4] = {sc[kk][0], sc[kk][2], sc[kk][1], sc[kk][3]};   // a0 (g,t) a1 (g+8,t) a2 (g,t+4) a3 (g+8,t+4)
#pragma unroll
      for (int e = 0; e < 4; e++) {
        ph[e] = att_tf32(pv[e]);
        pl[e] = att_tf32(pv[e] - __uint_as_float(ph[e]));
      }
      const uint32_t* vh = Vh + (kk * 8 + 2 * t) * kAttLd + g;
      const uint32_t* vl = Vl + (kk * 8 + 2 * t) * kAttLd + g;
#pragma unroll
      for (int n = 0; n < 8; n++) {
        const uint32_t bh0 = vh[n * 8], bh1 = vh[kAttLd + n * 8], bl0 = vl[n * 8], bl1 = vl[kAttLd + n * 8];
        att_mma(o[n], pl, bh0, bh1);
        att_mma(o[n], ph, bl0, bl1);
        att_mma(o[n], ph, bh0, bh1);
      }
    }
  }
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
#pragma unroll
  for (int n = 0; n < 8; n++) {
    const int d = n * 8 + 2 * t;
    if (r0 < N) *reinterpret_cast<float2*>(ctx + (base + r0) * 768 + h * 64 + d) = make_float2(o[n][0] * i0, o[n][1] * i0);
    if (r1 < N) *reinterpret_cast<float2*>(ctx + (base + r1) * 768 + h * 64 + d) = make_float2(o[n][2] * i1, o[n][3] * i1);
  }
}

void launch_attention(const float* qkv, float* ctx, const int* off, const int* len, int B,
                      int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  constexpr int smem = 4 * 64 * kAttLd * 4;
  if (max_len > 64) {   // 128 query rows per CTA: the K/V staging (load + tf32 split) is amortised over twice the MMAs
    prepare_smem_launch<attention_tc_kernel<8>>(smem);
    dim3 g((max_len + 127) / 128, 12, B);
    attention_tc_kernel<8><<<g, 256, smem, st>>>(qkv, ctx, off, len);
  } else {
    prepare_smem_launch<attention_tc_kernel<4>>(smem);
    dim3 g((max_len + 63) / 64, 12, B);
    attention_tc_kernel<4><<<g, 128, smem, st>>>(qkv, ctx, off, len);
  }
  post_launch("attention", st);
}

// ------------------------------------------------------------------------------------------
// Bidirectional LSTM recurrence (H = 256).  One CTA per (item, direction); thread r owns gate
// row r (i,f,g,o blocks of 256).  W_hh^T is k-major so each k step is one coalesced 4 KB read
// that stays L2-resident (1 MB per direction); h lives in shared memory, c in registers.
__global__ void __launch_bounds__(1024) lstm_kernel(const float* __restrict__ xproj,
                                                    const float* __restrict__ whhT,
                                                    float* __restrict__ out, int ldo, int ocol,
                                                    const int* off, const int* len) {
  __shared__ float h[256];
  __shared__ float g[1024];
  const int b = blockIdx.x, dir = blockIdx.y;
  const int N = len[b];
  const size_t base = (size_t)off[b];
  const int r = threadIdx.x;
  const float* W = whhT + (size_t)dir * 256 * 1024 + r;
  if (r < 256) h[r] = 0.f;
  float c = 0.f;
  __syncthreads();
  for (int s = 0; s < N; s++) {
    const int t = dir == 0 ? s : N - 1 - s;
    float acc0 = xproj[(base + t) * 2048 + dir * 1024 + r];
    float acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll 8
    for (int k = 0; k < 256; k += 4) {
      acc0 = fmaf(W[(size_t)(k + 0) * 1024], h[k + 0], acc0);
      acc1 = fmaf(W[(size_t)(k + 1) * 1024], h[k + 1], acc1);
      acc2 = fmaf(W[(size_t)(k + 2) * 1024], h[k + 2], acc2);
      acc3 = fmaf(W[(size_t)(k + 3) * 1024], h[k + 3], acc3);
    }
    g[r] = (acc0 + acc1) + (acc2 + acc3);
    __syncthreads();
    if (r < 256) {
      const float ig = 1.0f / (1.0f + expf(-g[r]));
      const float fg = 1.0f / (1.0f + expf(-g[256 + r]));
      const float gg = tanhf(g[512 + r]);
      const float og = 1.0f / (1.0f + expf(-g[768 + r]));
      c = fg * c + ig * gg;
      const float hv = og * tanhf(c);
      h[r] = hv;
      out[(base + t) * ldo + ocol + dir * 256 + r] = hv;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Persistent weight-stationary bi-LSTM (K3).  One thread-block CLUSTER of 8 CTAs per (direction,
// group of G items).  CTA r of the cluster keeps the W_hh rows of hidden units [32r, 32r+32) (all
// four gates: 128 rows x 256 k fp32 = 128 KB) resident in shared memory for the whole sequence;
// every step it computes those 128 gate pre-activations for the G items of its group (weights read
// once per step and reused across items), updates its 32 cell/hidden values per item, and
// broadcasts the new h slice into the next-step h buffer of all 8 CTAs through distributed shared
// memory, followed by one cluster barrier.  Gate dot products are split over two half-warps and
// combined with a warp shuffle.
}  // namespace kkx
#include <cooperative_groups.h>
namespace kkx {
namespace cg = cooperative_groups;

// Step hand-off without a cluster barrier: every CTA pushes its new h slice (vectorised, 16 bytes per
// store) into the next-step h buffer of all 8 CTAs with st.async, which completes transaction bytes on the
// DESTINATION CTA's mbarrier; a CTA starts step s+1 as soon as its own barrier has seen all 8 slices.
// Two h buffers / two barriers (step parity) make the scheme race-free: a CTA can only be one step ahead
// of the slowest one, because it needs that CTA's slice to proceed.
__device__ __forceinline__ uint32_t lstm_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lstm_mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void lstm_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "LW_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra LD_%=;\n\t"
      "bra LW_%=;\n\t"
      "LD_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}

// Register-stationary weights: a thread owns TWO gate rows and one QUARTER of the k range for all G items and
// keeps those 2 x 64 weights in registers for the whole sequence (the 8 CTAs x 256 threads of a cluster hold
// the full 1 MB W_hh of one direction), so the per-step dot products read only h from shared memory: one
// broadcast LDS.128 feeds 8 FMAs, issued as packed FFMA2 over consecutive k.  h layout [item][quarter]
// [64 + 4 pad]: the 4 quarters of a warp hit 4 different bank groups, lanes of a quarter broadcast.
constexpr int kHQ = 68;                 // floats per h quarter (64 + 4 pad)
constexpr int kHItem = 4 * kHQ;         // floats per item in an h buffer

#ifdef KKX_LSTM_TIMING
#define LT_DECL long long lt_acc[4] = {0, 0, 0, 0}; long long lt_t = clock64();
#define LT(i) { const long long n_ = clock64(); lt_acc[i] += n_ - lt_t; lt_t = n_; }
#define LT_DUMP if (blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 && (warp == 0 || warp == 4) && maxN > 100) \
    printf("lstm G=%d warp %d steps %d: wait %lld dot %lld sync %lld gate+rest %lld (cycles per step)\n", G, warp, maxN, \
           lt_acc[0] / maxN, lt_acc[1] / maxN, lt_acc[2] / maxN, lt_acc[3] / maxN);
#else
#define LT_DECL
#define LT(i)
#define LT_DUMP
#endif
// G items per cluster.  Lane quarter q finishes (adds the input projection, writes the gate pre-activations of)
// the items g = 4i + q; warp w runs the gate non-linearities of the items g = w + 8i.  G = 10 and 12 exist because
// only 15 clusters of 8 CTAs are co-resident on a B200 (cudaOccupancyMaxActiveClusters): 64 items at G = 8 need
// 16 clusters, and the one left over used to run as a second wave, doubling the kernel's time.
// FAST (the tensor-core configuration): gate non-linearities on the SFU (ex2.approx / rcp.approx, |error| ~ 1e-7) instead
// of libm's expf / tanhf / IEEE division.  Measured with the phase counters (KKX_LSTM_TIMING): a gate slot -- one warp,
// one dependent chain through libm's expf, a division, the two-branch tanhf, twice -- took ~ 850 cycles, i.e. 1 940 of
// the 6 280 cycles of a step at G = 10 (two slots on warps 0 and 1) and 845 of 1 500 at G = 1.
__device__ __forceinline__ float lstm_sigmoid_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float lstm_tanh_fast(float x) {
  const float ax = fabsf(x), x2 = x * x;
  const float t = 1.0f - __fdividef(2.0f, __expf(2.0f * ax) + 1.0f);                 // |x| >= 0.15: abs error ~ 1e-7
  const float p = ax * fmaf(x2, fmaf(x2, fmaf(x2, -17.0f / 315.0f, 2.0f / 15.0f), -1.0f / 3.0f), 1.0f);   // next term 8e-10
  return copysignf(ax < 0.15f ? p : t, x);
}
template <int G, bool FAST>
__global__ void __launch_bounds__(256, 1) lstm_cluster_kernel(const float* __restrict__ xproj,
                                                              const float* __restrict__ whhT,
                                                              float* __restrict__ out, int ldo, int ocol,
                                                              const int* off, const int* len, int B) {
  constexpr int NQ = (G + 3) / 4;                      // item slots of a lane quarter
  constexpr int NW = (G + 7) / 8;                      // item slots of a warp (gate phase)
  extern __shared__ float4 lsm4[];
  float* hbuf = reinterpret_cast<float*>(lsm4);        // [2][G][4][68]
  float* gates2 = hbuf + 2 * G * kHItem;               // [2][G][128], by step parity: ONE block barrier per step --
  // the dot loop of step s + 1 writes the other buffer, and the buffer of step s is rewritten only behind the barrier
  // of step s + 1, which every warp reaches after its gate phase of step s
  uint64_t* bars = reinterpret_cast<uint64_t*>(gates2 + 2 * G * 128);   // [2] h-buffer "full" barriers
  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();             // 0..7: hidden-unit slice
  const int group = blockIdx.x >> 3, dir = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = lane >> 3;                             // k quarter [64q, 64q+64)
  const int rp = warp * 8 + (lane & 7);                // row pair: local gate rows 2rp, 2rp+1
  constexpr uint32_t kStepBytes = G * 256 * 4;         // bytes every CTA receives per step

  for (int i = tid; i < 2 * G * kHItem; i += 256) hbuf[i] = 0.f;
  const uint32_t bar0 = lstm_smem_u32(bars), bar1 = bar0 + 8;
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0));
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar1));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // buffer 1 receives h_1 during step 0
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar1), "r"(kStepBytes) : "memory");
  }

  int maxN = 0;
  for (int g = 0; g < G; g++) {
    const int item = group * G + g;
    maxN = max(maxN, item < B ? len[item] : 0);
  }
  int qoff[NQ], qlen[NQ];                              // the items this lane quarter finishes
#pragma unroll
  for (int i = 0; i < NQ; i++) {
    const int g = 4 * i + q, item = group * G + g;
    const bool ok = g < G && item < B;
    qoff[i] = ok ? off[item] : 0;
    qlen[i] = ok ? len[item] : 0;
  }
  int woff[NW], wlen[NW];                              // the items this warp runs the gate phase for
#pragma unroll
  for (int i = 0; i < NW; i++) {
    const int g = warp + 8 * i, item = group * G + g;
    const bool ok = g < G && item < B;
    woff[i] = ok ? off[item] : 0;
    wlen[i] = ok ? len[item] : 0;
  }
  // global gate rows of this thread's row pair (same gate block: 2rp and 2rp+1 never straddle 32);
  // local row rl = gate*32 + j  <->  W_hh row gate*256 + r*32 + j
  const int grow0 = ((2 * rp) >> 5) * 256 + r * 32 + ((2 * rp) & 31);
  // this thread's weights, k in [64q, 64q+64), as pairs over consecutive k (FFMA2 operands)
  float2 w0[32], w1[32];
  {
    const float* Wg = whhT + (size_t)dir * 256 * 1024 + (size_t)(64 * q) * 1024 + grow0;
#pragma unroll
    for (int kk = 0; kk < 32; kk++) {
      const float2 a = *reinterpret_cast<const float2*>(Wg + (size_t)(2 * kk) * 1024);       // rows (2rp, 2rp+1) at k
      const float2 b2 = *reinterpret_cast<const float2*>(Wg + (size_t)(2 * kk + 1) * 1024);  // ... at k+1
      w0[kk] = make_float2(a.x, b2.x);
      w1[kk] = make_float2(a.y, b2.y);
    }
  }
  float c[NW];                                           // cell state of (item warp + 8i, unit lane)
#pragma unroll
  for (int i = 0; i < NW; i++) c[i] = 0.f;
  const float* const xrow = xproj + dir * 1024 + grow0;
  float2 xpn[NQ];
#pragma unroll
  for (int i = 0; i < NQ; i++) {
    xpn[i] = make_float2(0.f, 0.f);
    if (qlen[i] > 0) {
      const int t = dir == 0 ? 0 : qlen[i] - 1;
      xpn[i] = *reinterpret_cast<const float2*>(xrow + (size_t)(qoff[i] + t) * 2048);
    }
  }
  cluster.sync();
  LT_DECL
  for (int s = 0; s < maxN; s++) {
    const uint32_t bcur = (s & 1) ? bar1 : bar0;
    LT(3)
    if (s > 0) lstm_mbar_wait(bcur, (uint32_t)((s - 1) >> 1) & 1u);   // h_s complete in hbuf[s&1]
    LT(0)
    // re-arm this buffer's barrier for its next use (h_{s+2}); no slice of h_{s+2} can be complete before
    // this CTA has sent h_{s+1}, and early bytes only drive the (signed) tx-count of the new phase
    if (tid == 0 && s + 2 < maxN)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bcur), "r"(kStepBytes) : "memory");
    const float* hc = hbuf + (s & 1) * G * kHItem;
    float* hn_local = hbuf + ((s + 1) & 1) * G * kHItem;
    float* gates = gates2 + (s & 1) * G * 128;
    // input projections were fetched one step ahead (xpn); fetch the next step's now so that the global
    // latency hides behind a whole step
    float2 xp[NQ];
#pragma unroll
    for (int i = 0; i < NQ; i++) {
      xp[i] = xpn[i];
      if (s + 1 < qlen[i]) {
        const int t = dir == 0 ? s + 1 : qlen[i] - 2 - s;
        xpn[i] = *reinterpret_cast<const float2*>(xrow + (size_t)(qoff[i] + t) * 2048);
      }
    }
    float2 acc0[G], acc1[G];               // (even-k, odd-k) partial sums of the two rows
#pragma unroll
    for (int g = 0; g < G; g++) { acc0[g] = make_float2(0.f, 0.f); acc1[g] = make_float2(0.f, 0.f); }
    const float4* h4 = reinterpret_cast<const float4*>(hc + q * kHQ);
#pragma unroll
    for (int kk = 0; kk < 16; kk++) {
#pragma unroll
      for (int g = 0; g < G; g++) {
        const float4 h = h4[g * (kHItem / 4) + kk];
        const float2 h01 = make_float2(h.x, h.y), h23 = make_float2(h.z, h.w);
        acc0[g] = __ffma2_rn(w0[2 * kk], h01, acc0[g]); acc1[g] = __ffma2_rn(w1[2 * kk], h01, acc1[g]);
        acc0[g] = __ffma2_rn(w0[2 * kk + 1], h23, acc0[g]); acc1[g] = __ffma2_rn(w1[2 * kk + 1], h23, acc1[g]);
      }
    }
#pragma unroll
    for (int g = 0; g < G; g++) {
      float a0 = acc0[g].x + acc0[g].y, a1 = acc1[g].x + acc1[g].y;
      a0 += __shfl_xor_sync(0xffffffffu, a0, 8);  a1 += __shfl_xor_sync(0xffffffffu, a1, 8);
      a0 += __shfl_xor_sync(0xffffffffu, a0, 16); a1 += __shfl_xor_sync(0xffffffffu, a1, 16);
      if ((g & 3) == q)
        *reinterpret_cast<float2*>(gates + g * 128 + 2 * rp) = make_float2(a0 + xp[g >> 2].x, a1 + xp[g >> 2].y);
    }
    LT(1)
    __syncthreads();
    LT(2)
    // both slots' arithmetic first, branch-free (a warp without a second item recomputes the last one and drops the
    // result), so that the two dependent chains interleave; then the stores and the hand-off
    float hv_[NW];
#pragma unroll
    for (int i = 0; i < NW; i++) {
      const int g = min(warp + 8 * i, G - 1), j = lane;
      const float* gp = gates + g * 128;
      float ig, fg, gg, og;
      if (FAST) {
        ig = lstm_sigmoid_fast(gp[j]); fg = lstm_sigmoid_fast(gp[32 + j]);
        gg = lstm_tanh_fast(gp[64 + j]); og = lstm_sigmoid_fast(gp[96 + j]);
      } else {
        ig = 1.0f / (1.0f + expf(-gp[j])); fg = 1.0f / (1.0f + expf(-gp[32 + j]));
        gg = tanhf(gp[64 + j]); og = 1.0f / (1.0f + expf(-gp[96 + j]));
      }
      c[i] = fg * c[i] + ig * gg;
      hv_[i] = og * (FAST ? lstm_tanh_fast(c[i]) : tanhf(c[i]));
    }
#pragma unroll
    for (int i = 0; i < NW; i++) {
      const int g = warp + 8 * i, j = lane;
      const float hv = hv_[i];
      if (g < G && s < wlen[i]) {
        const int t = dir == 0 ? s : wlen[i] - 1 - s;
        out[(size_t)(woff[i] + t) * ldo + ocol + dir * 256 + r * 32 + j] = hv;
      }
      // gather 4 consecutive hidden units into one lane, push 16 bytes to every CTA of the cluster (spreading the 64
      // stores of an item over all 32 lanes -- two per lane, eight shuffles -- measured 8 % slower per step)
      const float h1 = __shfl_down_sync(0xffffffffu, hv, 1);
      const float h2 = __shfl_down_sync(0xffffffffu, hv, 2);
      const float h3 = __shfl_down_sync(0xffffffffu, hv, 3);
      if (g < G && (j & 3) == 0 && s + 1 < maxN) {
        const int u = r * 32 + j;                        // hidden unit -> padded quarter layout
        const uint32_t dst = lstm_smem_u32(hn_local + g * kHItem + (u >> 6) * kHQ + (u & 63));
        const uint32_t bnext = (s & 1) ? bar0 : bar1;
#pragma unroll
        for (int d = 0; d < 8; d++) {
          const uint32_t ra = lstm_mapa(dst, (uint32_t)d), rb = lstm_mapa(bnext, (uint32_t)d);
          asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
                       ::"r"(ra), "f"(hv), "f"(h1), "f"(h2), "f"(h3), "r"(rb) : "memory");
        }
      }
    }
  }
  LT_DUMP
  cluster.sync();      // no CTA may exit while a peer can still write into its shared memory
}

template <int G>
static void launch_lstm_cluster(const float* xproj, const float* whhT, float* out, int ldo, int ocol,
                                const int* off, const int* len, int B, cudaStream_t st, int fast) {
  const size_t smem = (size_t)(2 * G * kHItem + 2 * G * 128) * sizeof(float) + 16;
  auto kern = fast ? lstm_cluster_kernel<G, true> : lstm_cluster_kernel<G, false>;
  if (fast) prepare_smem_launch<lstm_cluster_kernel<G, true>>((int)smem);
  else prepare_smem_launch<lstm_cluster_kernel<G, false>>((int)smem);
  const int groups = (B + G - 1) / G;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(8 * groups, 2, 1);
  cfg.blockDim = dim3(256, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 8; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  KKX_CUDA(cudaLaunchKernelEx(&cfg, kern, xproj, whhT, out, ldo, ocol, off, len, B));
}

void launch_lstm(const float* xproj, const float* whhT, float* out, int ldo, int ocol,
                 const int* off, const int* len, int B, cudaStream_t st, int variant) {
  if (g_dry_run) return;
  if (variant < 0) {                    // one CTA per (item, direction): the plain reference kernel (tests only)
    dim3 g(B, 2);
    lstm_kernel<<<g, 1024, 0, st>>>(xproj, whhT, out, ldo, ocol, off, len);
  } else {
    const int pp = variant;               // 1 = SFU gate functions, 0 = libm
    // smallest group size whose clusters are all co-resident: 15 clusters of 8 CTAs fit a B200
    // (cudaOccupancyMaxActiveClusters); one cluster too many runs as a second wave and doubles the time
    static std::atomic<int> max_clusters[64];      // 0 = not asked yet (two threads may both ask: same answer)
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 64) dev = 63;
    if (max_clusters[dev].load(std::memory_order_relaxed) == 0) {       // depends on how the part's GPCs are populated: ask, do not assume
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(8 * 64, 2, 1);
      cfg.blockDim = dim3(256, 1, 1);
      cfg.dynamicSmemBytes = (size_t)(2 * 8 * kHItem + 2 * 8 * 128) * sizeof(float) + 16;
      cudaLaunchAttribute at[1];
      at[0].id = cudaLaunchAttributeClusterDimension;
      at[0].val.clusterDim.x = 8; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
      cfg.attrs = at; cfg.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, lstm_cluster_kernel<8, true>, &cfg) != cudaSuccess || n <= 0) { n = 15; cudaGetLastError(); }
      max_clusters[dev].store(n, std::memory_order_relaxed);
    }
    const int kMaxClusters = max_clusters[dev].load(std::memory_order_relaxed);
    auto fits = [&](int G) { return 2 * ((B + G - 1) / G) <= kMaxClusters; };
    if (fits(1)) launch_lstm_cluster<1>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);
    else if (fits(2)) launch_lstm_cluster<2>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);
    else if (fits(4)) launch_lstm_cluster<4>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);
    else if (fits(6)) launch_lstm_cluster<6>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);     // 40 items (first frame group of B = 64) -> 14 clusters
    else if (fits(8)) launch_lstm_cluster<8>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);
    else if (fits(10)) launch_lstm_cluster<10>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);   // 64 items -> 14 clusters
    else if (fits(12)) launch_lstm_cluster<12>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);
    else launch_lstm_cluster<8>(xproj, whhT, out, ldo, ocol, off, len, B, st, pp);                  // several waves anyway
  }
  post_launch("lstm", st);
}

}  // namespace kkx
