// kernels_tc.cu -- Blackwell tensor-core path: bf16 implicit-GEMM Conv1d / ConvTranspose1d-phase /
// Linear on tcgen05.mma with TMEM accumulators, operands staged by TMA (cp.async.bulk.tensor,
// 128B swizzle) through an mbarrier ring; plus the HBM-bound "apply" kernels that produce the
// bf16 operand (AdaIN scale/shift + LeakyReLU/Snake fused, zero halo rows maintained).
//
// A conv is a sum of row-shifted GEMMs over the time-major activation matrix:
//   D[t, co] = sum_tap sum_c A[t + tap*dil - pad, c] * W[co, tap, c]
// so the A tile of tap `tap` is the same 2-D TMA box shifted by tap*dil - pad rows; rows outside
// the tensor are zero-filled by TMA and rows between ragged items are zero gap rows (kGapRows).
#include "kernels.h"
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <mutex>
#include "tc_ptx.cuh"

// perf-experiment switches (skip MMAs / loads / stores: wrong results, timing only) exist only in -DKKX_TC_DEBUG builds
#ifdef KKX_TC_DEBUG
#define TC_DBG(a, bit) ((a).debug & (bit))
#else
#define TC_DBG(a, bit) (0)
#endif

namespace kkx {

#ifdef KKX_TC_TIMING
#define TCT_DECL(n) long long tct_acc[n] = {0}; long long tct_last = clock64(); const bool tct_on = a.timing && blockIdx.x == gridDim.x - 2 && blockIdx.y == gridDim.y - 1 && blockIdx.z == gridDim.z - 1
#define TCT(slot) do { if (tct_on) { const long long now_ = clock64(); tct_acc[slot] += now_ - tct_last; tct_last = now_; } } while (0)
#define TCT_FLUSH(base, n) do { if (tct_on) for (int i_ = 0; i_ < (n); i_++) atomicAdd(reinterpret_cast<unsigned long long*>(a.timing) + (base) + i_, (unsigned long long)tct_acc[i_]); } while (0)
#else
#define TCT_DECL(n)
#define TCT(slot)
#define TCT_FLUSH(base, n)
#endif

// ------------------------------------------------------------------------------------------
// host: tensor-map encoding through the driver entry point (no libcuda link dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  if (!fn) throw CudaError("cuTensorMapEncodeTiled entry point not available");
  return fn;
}

// bf16 row-major [outer, inner] with row pitch `pitch_elems`; box = [box_outer, 64] elements,
// 128-byte swizzle (one box row = 128 B = one swizzle span).
static void make_tmap(void* out_map, const void* ptr, long long inner, long long outer,
                      long long pitch_elems, int box_outer, bool f32, bool f16 = false) {
  const int esz = f32 ? 4 : 2;
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)pitch_elems * esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode()((CUtensorMap*)out_map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : (f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16), 2, const_cast<void*>(ptr),
                            dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char b[160];
    snprintf(b, sizeof b, "cuTensorMapEncodeTiled failed (%d) inner=%lld outer=%lld pitch=%lld", (int)r, inner, outer, pitch_elems);
    throw CudaError(b);
  }
}
void make_tmap_bf16(void* out_map, const void* ptr, long long inner, long long outer,
                    long long pitch_elems, int box_outer) {
  make_tmap(out_map, ptr, inner, outer, pitch_elems, box_outer, false);
}
// fp32 container (tf32 operands): box = [box_outer, 32] elements = 128 B rows
void make_tmap_f32(void* out_map, const void* ptr, long long inner, long long outer,
                   long long pitch_elems, int box_outer) {
  make_tmap(out_map, ptr, inner, outer, pitch_elems, box_outer, true);
}

// fp16 planes: box = [box_outer, 64] elements = 128 B rows
void make_tmap_f16(void* out_map, const void* ptr, long long inner, long long outer,
                   long long pitch_elems, int box_outer) {
  make_tmap(out_map, ptr, inner, outer, pitch_elems, box_outer, false, true);
}

__device__ __forceinline__ float gelu_new_f(float v) {
  const float u = 0.7978845608028654f * (v + 0.044715f * v * v * v);
  return 0.5f * v * (1.0f + tanhf(u));
}

// ---- fp32 output epilogue of every kernel below.  Which kernel runs depends on the batch, so all of them finish an
// accumulator with these helpers: the same inputs give the same bits whatever the batch composition.  A thread handles
// columns n .. n+3 of one output row; `vec` (a.vec4 && n + 3 < Co) makes that one 16-byte access, otherwise only the
// columns below Co are touched.
// bias / residual / accumulate operand; columns >= Co read as 0
__device__ __forceinline__ float4 epi_load4(const float* p, int n, int Co, bool vec) {
  if (vec) return *reinterpret_cast<const float4*>(p);
  float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
  r.x = p[0]; if (n + 1 < Co) r.y = p[1]; if (n + 2 < Co) r.z = p[2]; if (n + 3 < Co) r.w = p[3];
  return r;
}
// (acc * wscale + bias), GELU if eact says so, then (+ res) * oscale.  Without a residual res is 0: the + 0.f stays,
// it turns -0 into +0.
__device__ __forceinline__ float4 epi_math4(float4 o, float wscale, float4 bias, int eact, float4 res, float oscale) {
  o.x = fmaf(o.x, wscale, bias.x); o.y = fmaf(o.y, wscale, bias.y); o.z = fmaf(o.z, wscale, bias.z); o.w = fmaf(o.w, wscale, bias.w);
  if (eact == ACT_GELU_NEW) { o.x = gelu_new_f(o.x); o.y = gelu_new_f(o.y); o.z = gelu_new_f(o.z); o.w = gelu_new_f(o.w); }
  o.x = (o.x + res.x) * oscale; o.y = (o.y + res.y) * oscale; o.z = (o.z + res.z) * oscale; o.w = (o.w + res.w) * oscale;
  return o;
}
// adds what is already stored when `accumulate`, then stores
__device__ __forceinline__ void epi_store4(float* p, float4 o, int n, int Co, bool vec, bool accumulate) {
  if (accumulate) { const float4 pv = epi_load4(p, n, Co, vec); o.x += pv.x; o.y += pv.y; o.z += pv.z; o.w += pv.w; }
  if (vec) {
    *reinterpret_cast<float4*>(p) = o;
  } else {
    p[0] = o.x; if (n + 1 < Co) p[1] = o.y; if (n + 2 < Co) p[2] = o.z; if (n + 3 < Co) p[3] = o.w;
  }
}

// ------------------------------------------------------------------------------------------
// The kernel.  One 128 x BN output tile per CTA.  6 warps:
//   warp 0  TMA producer (one elected lane)        warp 1  TMEM alloc + MMA issuer (one lane)
//   warps 2..5  epilogue: tcgen05.ld of the warp's 32-lane TMEM quadrant -> bias / residual /
//               scale / accumulate -> global
// MODE 0: bf16 operands, one product.  MODE 1: split-TF32 ("3xTF32"/"4xTF32"): every operand is a
// pair of tf32-exact fp32 planes (hi, lo = a - hi), D += Ahi*Bhi + Alo*Bhi + Ahi*Blo [+ Alo*Blo] on
// kind::tf32, which recovers ~fp32 accuracy on the tensor cores for the precision-critical
// predictor path (ALBERT -> durations, F0/N).
// Clusters of 2 CTAs along M sharing each weight tile by TMA multicast were measured not faster for the
// split-TF32 GEMMs (13.9 vs 12.4 ms for the 12 QKV GEMMs).
template <int BN, int STAGES, int MODE>
__global__ void __launch_bounds__(192) conv_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                      const __grid_constant__ CUtensorMap tmB,
                                                      const __grid_constant__ CUtensorMap tmA2,
                                                      const __grid_constant__ CUtensorMap tmB2,
                                                      TcConvArgs a) {
  constexpr uint32_t PLANES = MODE ? 2 : 1;
  const int KE = (MODE && !a.f16) ? 32 : 64;   // K elements per pipeline stage (one 128-byte swizzle span)
  const bool f16 = MODE && a.f16;              // split-FP16 planes instead of split-TF32
  const int cs = f16 ? 0 : 1;                  // log2(stages per hi*hi chain): a chain is 64 K-elements either way
  constexpr uint32_t A_BYTES = 128 * 128, B_BYTES = BN * 128, STAGE_BYTES = PLANES * (A_BYTES + B_BYTES);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  // MODE 1 keeps 4 accumulators in TMEM: [0] all small cross terms, [1..3] a ring for the hi*hi
  // term, which is accumulated in chains of only 64 K-elements: the tensor core adds with
  // round-toward-zero once per MMA (measured: error grows linearly, ~0.5 ulp per K=8 step), so long
  // chains would lose fp32-grade accuracy; the epilogue warps drain each finished chain and add it
  // into registers with IEEE round-to-nearest while the next chain runs.
  constexpr uint32_t TMEM_COLS = MODE ? 4 * BN : BN;
  const uint32_t bar_base = base + STAGES * STAGE_BYTES;        // full[S], empty[S], tmem_full, bfull[3], bempty[3]
  const uint32_t tmem_slot = bar_base + (2 * STAGES + 1 + 6) * 8;
  auto full_bar = [&](int s) { return bar_base + s * 8; };
  auto empty_bar = [&](int s) { return bar_base + (STAGES + s) * 8; };
  const uint32_t tfull_bar = bar_base + 2 * STAGES * 8;
  auto bfull_bar = [&](int j) { return bar_base + (2 * STAGES + 1 + j) * 8; };
  auto bempty_bar = [&](int j) { return bar_base + (2 * STAGES + 4 + j) * 8; };

  const int b = blockIdx.z;
  const int mlen = a.m_len[b];
  // phase-fused launches put (phase, n-tile) on grid.x and the m-tile on grid.y
  const bool fused = MODE == 0 && a.nphase > 1;
  const int bx = fused ? blockIdx.y : blockIdx.x, by = fused ? blockIdx.x : blockIdx.y;
  const int m0 = bx * 128;
  if (m0 >= mlen) return;  // CTA-uniform
  const int ntn = (a.Co + BN - 1) / BN;
  const int ph = fused ? by / ntn : 0;
  const int c_pad = fused ? a.phase_pad[ph] : a.pad;
  const int c_oro = fused ? a.phase_oro[ph] : a.oro;
  const int n0 = (fused ? by - ph * ntn : by) * BN;
  const int wrow0 = ph * a.Co + n0;          // row of this tile in the (phase-stacked) weight map
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.Cpad / KE;
  const int num_k = a.ks * kchunks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (MODE) {
      prefetch_tmap(&tmA2);
      prefetch_tmap(&tmB2);
    }
    for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(tfull_bar, 1);
    if (MODE) for (int j = 0; j < 3; j++) { mbar_init(bfull_bar(j), 1); mbar_init(bempty_bar(j), 4); }
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      const int row0 = a.in_off[b] + m0 - c_pad;
      TCT_DECL(2);
      for (int it = 0; it < num_k; it++) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(empty_bar(s), ph ^ 1u);
        TCT(0);
        const int tap = it / kchunks, c0 = (it - tap * kchunks) * KE;
        const uint32_t sa = base + s * STAGE_BYTES;
        const bool skipA2 = MODE && TC_DBG(a, 8);     // perf experiment: pretend the A lo plane needs no L2 traffic
        const bool skipB2 = MODE && TC_DBG(a, 16);
        mbar_expect_tx(full_bar(s), STAGE_BYTES - (skipA2 ? A_BYTES : 0) - (skipB2 ? B_BYTES : 0));
        tma_load_2d(sa, &tmA, c0, row0 + tap * a.dil, full_bar(s));
        if (MODE && !skipA2) tma_load_2d(sa + A_BYTES, &tmA2, c0, row0 + tap * a.dil, full_bar(s));
        tma_load_2d(sa + PLANES * A_BYTES, &tmB, tap * a.Cpad + c0, wrow0, full_bar(s));
        if (MODE && !skipB2) tma_load_2d(sa + 2 * A_BYTES + B_BYTES, &tmB2, tap * a.Cpad + c0, wrow0, full_bar(s));
        TCT(1);
      }
      TCT_FLUSH(0, 2);
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = MODE ? (f16 ? umma_idesc_f16(128, BN) : umma_idesc_tf32(128, BN)) : umma_idesc_bf16(128, BN);
      TCT_DECL(3);
      for (int it = 0; it < num_k; it++) {
        const int s = it % STAGES;
        const uint32_t ph = (uint32_t)(it / STAGES) & 1u;
        mbar_wait(full_bar(s), ph);
        tc_fence_after();
        TCT(0);
        const uint32_t sa = base + s * STAGE_BYTES;
        if (MODE == 0) {
          const uint64_t ad = umma_desc_sw128(sa), bd = umma_desc_sw128(sa + A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; k++)  // 4 x (K=16 bf16 = 32 B) inside the 128-byte swizzle span
            if (!TC_DBG(a, 2)) umma_bf16(tmem_base, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (it | k) ? 1u : 0u);
        } else {
          const int chain = it >> cs, j = chain % 3;
          const bool chain_start = (it & cs) == 0;
          if (chain_start && chain >= 3) {       // ring slot j must have been drained by the epilogue
            mbar_wait(bempty_bar(j), (uint32_t)(chain / 3 - 1) & 1u);
            tc_fence_after();
            TCT(1);
          }
          const uint64_t ah = umma_desc_sw128(sa), al = umma_desc_sw128(sa + A_BYTES);
          const uint64_t bh = umma_desc_sw128(sa + 2 * A_BYTES), bl = umma_desc_sw128(sa + 2 * A_BYTES + B_BYTES);
          const uint32_t t_small = tmem_base, t_big = tmem_base + (uint32_t)(BN * (1 + j));
#pragma unroll
          for (int k = 0; k < 4; k++) {  // 4 x (32 B of K: 8 tf32 or 16 fp16)
            const uint64_t o = (uint64_t)(2 * k);
            if (TC_DBG(a, 2)) continue;                 // perf experiment: no MMAs
            if (a.nprod >= 4) umma_split(t_small, al + o, bl + o, idesc, (it | k) ? 1u : 0u, f16);
            if (!TC_DBG(a, 32)) {                     // perf experiment: hi*hi only
              umma_split(t_small, al + o, bh + o, idesc, (a.nprod >= 4 || (it | k)) ? 1u : 0u, f16);
              umma_split(t_small, ah + o, bl + o, idesc, 1u, f16);
            }
            umma_split(t_big, ah + o, bh + o, idesc, (chain_start && k == 0) ? 0u : 1u, f16);
          }
          if ((it & cs) == cs || it == num_k - 1) umma_commit(bfull_bar(j));  // chain complete
        }
        umma_commit(empty_bar(s));  // frees the smem stage when these MMAs have read it
        TCT(2);
      }
      umma_commit(tfull_bar);       // accumulator complete
      TCT_FLUSH(4, 3);
    }
  } else {
    // ---- epilogue (4 warps).  All MMAs have completed when tfull_bar flips, so the pipeline
    // stages are idle and stage memory is reused as a transpose buffer: each thread drops its
    // 32-column strip of one accumulator row into padded smem (conflict-free), then the 128
    // threads write whole 128-byte row segments to global (8 lanes per row -> full-line stores,
    // coalesced residual / accumulate reads).
    const int q = warp & 3;                 // TMEM lane quadrant this warp may access
    const int et = q * 32 + lane;           // accumulator row held by this thread
    float racc[MODE ? BN : 1];              // MODE 1: fp32 (round-to-nearest) sum of the drained hi*hi chains
#ifdef KKX_TC_TIMING
    long long tct_acc[4] = {0}; long long tct_last = clock64();
    const bool tct_on = a.timing && blockIdx.x == gridDim.x - 2 && blockIdx.y == gridDim.y - 1 && blockIdx.z == gridDim.z - 1 && threadIdx.x == 64;
#endif
    if (MODE) {
#pragma unroll
      for (int e = 0; e < (MODE ? BN : 1); e++) racc[e] = 0.f;
      const int nchains = (num_k + cs) >> cs;
      for (int ch = 0; ch < nchains; ch++) {
        const int j = ch % 3;
        mbar_wait(bfull_bar(j), (uint32_t)(ch / 3) & 1u);
        tc_fence_after();
        TCT(0);
        if (BN == 64) {      // one TMEM round trip per chain (the latency path: small problems run 64-wide tiles)
          uint32_t v[64];
          tmem_ld64(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(BN * (1 + j)), v);
#pragma unroll
          for (int e = 0; e < 64; e++) racc[MODE ? (e < BN ? e : 0) : 0] += __uint_as_float(v[e]);
        } else {
#pragma unroll
          for (int c = 0; c < BN; c += 32) {
            if (TC_DBG(a, 4)) continue;                   // perf experiment: chains are not drained
            uint32_t v[32];
            tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(BN * (1 + j) + c), v);
#pragma unroll
            for (int e = 0; e < 32; e++) racc[(MODE ? c : 0) + (MODE ? e : 0)] += __uint_as_float(v[e]);
          }
        }
        tc_fence_before();
        if (lane == 0) mbar_arrive(bempty_bar(j));
        TCT(1);
      }
    }
    constexpr int PITCH = 36;               // floats per staged row (32 + 4 pad)
    float* stage_f = reinterpret_cast<float*>(smem_raw + (base - smem_u32(smem_raw)));
    const int out_off = a.out_off[b];
    const int res_off = a.res ? a.res_off[b] : 0;
    // thread t writes columns c4..c4+3 (c4 = 4*(t&7), fixed) of rows (t>>3) + 16*i, i = 0..7, of
    // every 32-column chunk.  Residual / accumulate operands of chunk c+1 are fetched while chunk c
    // is processed, and those of chunk 0 before the accumulator is even complete, so their HBM
    // latency hides behind the MMA main loop.
    const int t = threadIdx.x - 64;
    const int c4 = (t & 7) << 2;
    auto fetch = [&](int c, float4* rv) {   // residual operand of chunk c for this thread's 8 rows
      const int n = n0 + c + c4;
      const bool vec = a.vec4 && (n + 3 < a.Co);
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int mm = m0 + (t >> 3) + 16 * i;
        rv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.res && n < a.Co && mm < mlen)
          rv[i] = epi_load4(a.res + ((size_t)(res_off + ((mm * a.ors + c_oro) >> a.res_shift)) * a.ldr + a.rcol + n), n, a.Co, vec);
      }
    };
    float4 rv[8];
    if (MODE == 0) fetch(0, rv);            // overlaps the whole MMA main loop
    mbar_wait(tfull_bar, 0);
    tc_fence_after();
    TCT(2);
#pragma unroll
    for (int c = 0; c < BN; c += 32) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c, v);
      if (MODE) {
#pragma unroll
        for (int e = 0; e < 32; e++) v[e] = __float_as_uint(__uint_as_float(v[e]) + racc[(MODE ? c : 0) + (MODE ? e : 0)]);
      }
      float* buf = stage_f + ((c >> 5) & 1) * (128 * PITCH);
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<uint4*>(buf + et * PITCH + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      if (MODE) fetch(c, rv);               // MODE 1 has no registers to spare for an early fetch
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const int n = n0 + c + c4;
      if (n < a.Co) {
        const bool vec = a.vec4 && (n + 3 < a.Co);
        const float4 bb = a.bias ? epi_load4(a.bias + n, n, a.Co, vec) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int row = (t >> 3) + 16 * i;
          const int mm = m0 + row;
          if (mm >= mlen || TC_DBG(a, 1)) continue;
          const float4 o = epi_math4(*reinterpret_cast<const float4*>(buf + row * PITCH + c4), a.wscale, bb, a.eact, rv[i], a.oscale);
          epi_store4(a.out + ((size_t)(out_off + mm * a.ors + c_oro) * a.ldo + a.ocol + n), o, n, a.Co, vec, a.accumulate);
        }
      }
      if (MODE == 0 && c + 32 < BN) fetch(c + 32, rv);   // in flight during the next chunk's TMEM->smem hop
    }
    TCT(3);
    TCT_FLUSH(8, 4);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------
// Phase-loop variant (bf16, phase-fused ConvTranspose1d with a.nphase two-tap phase convs): one CTA walks the PHASES of
// ONE 128-row m-tile as consecutive tiles (same activation rows, phase p's weights at rows [p*Co, (p+1)*Co) of the
// stacked map, output rows m*ors + phase_oro[p]).  The TMA/MMA pipeline runs straight across the phases and alternates
// between two TMEM accumulators, so the epilogue of one phase (TMEM -> smem transpose -> global) runs under the next
// phase's loads and MMAs, barrier init / TMEM allocation / descriptor prefetch are paid once per a.nphase tiles, and the
// activation tile of the later phases comes out of L2.
template <int BN, int STAGES>
__global__ void __launch_bounds__(192) conv_tc_multi_kernel(const __grid_constant__ CUtensorMap tmA,
                                                            const __grid_constant__ CUtensorMap tmB,
                                                            TcConvArgs a) {
  constexpr uint32_t A_BYTES = 128 * 128, B_BYTES = BN * 128, STAGE_BYTES = A_BYTES + B_BYTES;
  constexpr int PITCH = 36;
  constexpr uint32_t STG_BYTES = 2 * 128 * PITCH * 4;  // two transpose buffers
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t stg_base = base + STAGES * STAGE_BYTES;
  const uint32_t bar_base = stg_base + STG_BYTES;       // full[S], empty[S], tfull[2], tempty[2]
  const uint32_t tmem_slot = bar_base + (2 * STAGES + 4) * 8;
  auto full_bar = [&](int s) { return bar_base + s * 8; };
  auto empty_bar = [&](int s) { return bar_base + (STAGES + s) * 8; };
  auto tfull_bar = [&](int j) { return bar_base + (2 * STAGES + j) * 8; };
  auto tempty_bar = [&](int j) { return bar_base + (2 * STAGES + 2 + j) * 8; };

  const int b = blockIdx.z;
  const int mlen = a.m_len[b];
  const int m0 = blockIdx.x * 128;
  if (m0 >= mlen) return;  // CTA-uniform
  const int ntiles = a.nphase;
  const int n0 = blockIdx.y * BN;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.Cpad >> 6;
  const int num_k = a.ks * kchunks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int j = 0; j < 2; j++) { mbar_init(tfull_bar(j), 1); mbar_init(tempty_bar(j), 4); }
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, (uint32_t)(2 * BN));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      int g = 0;
      for (int ti = 0; ti < ntiles; ti++) {
        const int row0 = a.in_off[b] + m0 - a.phase_pad[ti];
        const int wrow = ti * a.Co + n0;
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          const uint32_t ph = (uint32_t)(g / STAGES) & 1u;
          mbar_wait(empty_bar(s), ph ^ 1u);
          const int tap = it / kchunks, c0 = (it - tap * kchunks) << 6;
          const uint32_t sa = base + s * STAGE_BYTES;
          mbar_expect_tx(full_bar(s), STAGE_BYTES);
          tma_load_2d(sa, &tmA, c0, row0 + tap * a.dil, full_bar(s));
          tma_load_2d(sa + A_BYTES, &tmB, tap * a.Cpad + c0, wrow, full_bar(s));
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
      int g = 0;
      for (int ti = 0; ti < ntiles; ti++) {
        const int acc = ti & 1;
        mbar_wait(tempty_bar(acc), ((uint32_t)(ti >> 1) & 1u) ^ 1u);   // accumulator drained?
        tc_fence_after();
        const uint32_t td = tmem_base + (uint32_t)(acc * BN);
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          const uint32_t ph = (uint32_t)(g / STAGES) & 1u;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t sa = base + s * STAGE_BYTES;
          const uint64_t ad = umma_desc_sw128(sa), bd = umma_desc_sw128(sa + A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; k++)
            if (!TC_DBG(a, 2)) umma_bf16(td, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (it | k) ? 1u : 0u);
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else {
    const int q = warp & 3;
    const int et = q * 32 + lane;
    float* stage_f = reinterpret_cast<float*>(smem_raw + (stg_base - smem_u32(smem_raw)));
    const int out_off = a.out_off[b];
    const int res_off = a.res ? a.res_off[b] : 0;
    const int t = threadIdx.x - 64;
    const int c4 = (t & 7) << 2;
    int chunk_ctr = 0;
    for (int ti = 0; ti < ntiles; ti++) {
      const int oro = a.phase_oro[ti];
      const int acc = ti & 1;
      auto fetch = [&](int c, float4* rv) {
        const int n = n0 + c + c4;
        const bool vec = a.vec4 && (n + 3 < a.Co);
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int mm = m0 + (t >> 3) + 16 * i;
          rv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (a.res && n < a.Co && mm < mlen)
            rv[i] = epi_load4(a.res + ((size_t)(res_off + ((mm * a.ors + oro) >> a.res_shift)) * a.ldr + a.rcol + n), n, a.Co, vec);
        }
      };
      float4 rv[8];
      fetch(0, rv);
      mbar_wait(tfull_bar(acc), (uint32_t)(ti >> 1) & 1u);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < BN; c += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + c), v);
        if (c + 32 >= BN) {   // last TMEM read of this tile: hand the accumulator back to the MMA warp
          tc_fence_before();
          if (lane == 0) mbar_arrive(tempty_bar(acc));
        }
        float* buf = stage_f + (chunk_ctr & 1) * (128 * PITCH);
        chunk_ctr++;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<uint4*>(buf + et * PITCH + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int n = n0 + c + c4;
        if (n < a.Co) {
          const bool vec = a.vec4 && (n + 3 < a.Co);
          const float4 bb = a.bias ? epi_load4(a.bias + n, n, a.Co, vec) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 8; i++) {
            const int row = (t >> 3) + 16 * i;
            const int mm = m0 + row;
            if (mm >= mlen || TC_DBG(a, 1)) continue;
            const float4 o = epi_math4(*reinterpret_cast<const float4*>(buf + row * PITCH + c4), a.wscale, bb, a.eact, rv[i], a.oscale);
            epi_store4(a.out + ((size_t)(out_off + mm * a.ors + oro) * a.ldo + a.ocol + n), o, n, a.Co, vec, a.accumulate);
          }
        }
        if (c + 32 < BN) fetch(c + 32, rv);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, (uint32_t)(2 * BN));
  }
}

// Weight-resident phase conv (generator stage-1 up-sampling, ConvTranspose1d(256, 128, k = 12, s = 6) as 6 two-tap phase
// convs).  The kernels above stream the weight tiles with the activations: 8 k-steps x 32 KB per (m-tile, phase), i.e. the
// whole 768 KB weight set once per 128 input rows -- 11.5 GB through L2 per launch at 5.75 M output rows, which is what
// the launch took (7 TB/s out of L2; its 2.9 GB of output would stream in 0.5 ms).  Here a persistent CTA owns ONE phase:
// the phase's weights (2 taps x 4 chunks x 16 KB = 128 KB) are loaded once and stay in shared memory, the CTA walks a
// contiguous range of the batch's m-tiles, and only activation tiles go through the TMA ring (3 stages of 16 KB).  Two
// TMEM accumulators alternate, so the epilogue of a tile runs under the MMAs of the next.  Same MMAs in the same order per
// output element as conv_tc_kernel -> identical bits.  grid = (CTAs per phase, nphase).
constexpr int kUpsStages = 3;     // 128 KB of weights + 3 x 16 KB activation stages + 36 KB epilogue staging = 212 KB
__global__ void __launch_bounds__(192) conv_phase_resident_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                  const __grid_constant__ CUtensorMap tmB,
                                                                  TcConvArgs a) {
  constexpr int BN = 128, STAGES = kUpsStages;
  constexpr uint32_t A_BYTES = 128 * 128, B_BYTES = BN * 128;
  constexpr int PITCH = 36;
  constexpr uint32_t STG_BYTES = 2 * 128 * PITCH * 4;
  constexpr int MAXK = 8;                               // resident weight tiles (ks * Cpad / 64)
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = base;                         // [num_k][B_BYTES]
  const uint32_t a_base = w_base + MAXK * B_BYTES;      // [STAGES][A_BYTES]
  const uint32_t stg_base = a_base + STAGES * A_BYTES;
  const uint32_t bar_base = stg_base + STG_BYTES;       // full[S], empty[S], tfull[2], tempty[2], wfull
  const uint32_t tmem_slot = bar_base + (2 * STAGES + 5) * 8;
  auto full_bar = [&](int s) { return bar_base + s * 8; };
  auto empty_bar = [&](int s) { return bar_base + (STAGES + s) * 8; };
  auto tfull_bar = [&](int j) { return bar_base + (2 * STAGES + j) * 8; };
  auto tempty_bar = [&](int j) { return bar_base + (2 * STAGES + 2 + j) * 8; };
  const uint32_t wfull_bar = bar_base + (2 * STAGES + 4) * 8;

  const int ph = blockIdx.y;
  const int t_begin = (int)(((long long)a.ntiles_m * blockIdx.x) / gridDim.x);
  const int t_end = (int)(((long long)a.ntiles_m * (blockIdx.x + 1)) / gridDim.x);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.Cpad >> 6;
  const int num_k = a.ks * kchunks;
  auto locate = [&](int tile, int& b, int& m0) {        // tile -> (item, first row); tile_start = prefix sum of ceil(len/128)
    int lo = 0, hi = a.B;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (a.tile_start[mid] <= tile) lo = mid; else hi = mid;
    }
    b = lo; m0 = (tile - a.tile_start[lo]) * 128;
  };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int j = 0; j < 2; j++) { mbar_init(tfull_bar(j), 1); mbar_init(tempty_bar(j), 4); }
    mbar_init(wfull_bar, 1);
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, (uint32_t)(2 * BN));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  if (warp == 0) {
    if (lane == 0 && t_begin < t_end) {
      mbar_expect_tx(wfull_bar, (uint32_t)num_k * B_BYTES);
      for (int it = 0; it < num_k; it++) {
        const int tap = it / kchunks, c0 = (it - tap * kchunks) << 6;
        tma_load_2d(w_base + it * B_BYTES, &tmB, tap * a.Cpad + c0, ph * a.Co, wfull_bar);
      }
      int g = 0;
      for (int tile = t_begin; tile < t_end; tile++) {
        int b, m0;
        locate(tile, b, m0);
        const int row0 = a.in_off[b] + m0 - a.phase_pad[ph];
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          const uint32_t par = (uint32_t)(g / STAGES) & 1u;
          mbar_wait(empty_bar(s), par ^ 1u);
          const int tap = it / kchunks, c0 = (it - tap * kchunks) << 6;
          mbar_expect_tx(full_bar(s), A_BYTES);
          tma_load_2d(a_base + s * A_BYTES, &tmA, c0, row0 + tap * a.dil, full_bar(s));
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && t_begin < t_end) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
      mbar_wait(wfull_bar, 0);
      int g = 0, ti = 0;
      for (int tile = t_begin; tile < t_end; tile++, ti++) {
        const int acc = ti & 1;
        mbar_wait(tempty_bar(acc), ((uint32_t)(ti >> 1) & 1u) ^ 1u);   // accumulator drained?
        tc_fence_after();
        const uint32_t td = tmem_base + (uint32_t)(acc * BN);
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          const uint32_t par = (uint32_t)(g / STAGES) & 1u;
          mbar_wait(full_bar(s), par);
          tc_fence_after();
          const uint64_t ad = umma_desc_sw128(a_base + s * A_BYTES), bd = umma_desc_sw128(w_base + it * B_BYTES);
#pragma unroll
          for (int k = 0; k < 4; k++)
            umma_bf16(td, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (it | k) ? 1u : 0u);
          umma_commit(empty_bar(s));
        }
        umma_commit(tfull_bar(acc));
      }
    }
  } else {
    const int q = warp & 3;
    const int et = q * 32 + lane;
    float* stage_f = reinterpret_cast<float*>(smem_raw + (stg_base - smem_u32(smem_raw)));
    const int t = threadIdx.x - 64;
    const int c4 = (t & 7) << 2;
    const int oro = a.phase_oro[ph];
    int chunk_ctr = 0, ti = 0;
    for (int tile = t_begin; tile < t_end; tile++, ti++) {
      int b, m0;
      locate(tile, b, m0);
      const int mlen = a.m_len[b];
      const int out_off = a.out_off[b];
      const int acc = ti & 1;
      mbar_wait(tfull_bar(acc), (uint32_t)(ti >> 1) & 1u);
      tc_fence_after();
#pragma unroll
      for (int c = 0; c < BN; c += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BN + c), v);
        if (c + 32 >= BN) {   // last TMEM read of this tile: hand the accumulator back to the MMA warp
          tc_fence_before();
          if (lane == 0) mbar_arrive(tempty_bar(acc));
        }
        float* buf = stage_f + (chunk_ctr & 1) * (128 * PITCH);
        chunk_ctr++;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *reinterpret_cast<uint4*>(buf + et * PITCH + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int n = c + c4;       // Co == BN, vec4, no residual, activation or accumulate (conv_phase_resident_ok)
        const float4 bb = a.bias ? epi_load4(a.bias + n, n, BN, true) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const int row = (t >> 3) + 16 * i;
          const int mm = m0 + row;
          if (mm >= mlen) continue;
          const float4 o = epi_math4(*reinterpret_cast<const float4*>(buf + row * PITCH + c4), a.wscale, bb, ACT_NONE,
                                     make_float4(0.f, 0.f, 0.f, 0.f), a.oscale);
          epi_store4(a.out + ((size_t)(out_off + mm * a.ors + oro) * a.ldo + a.ocol + n), o, n, BN, true, false);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, (uint32_t)(2 * BN));
  }
}
static bool conv_phase_resident_ok(const TcConvArgs& a) {
  return a.nphase > 1 && a.Co == 128 && !a.tf32 && !a.res && !a.accumulate && a.eact == ACT_NONE && a.tile_start && a.ntiles_m > 0 &&
         a.ks * (a.Cpad >> 6) <= 8 && a.vec4 && a.ldo % 4 == 0 && a.ocol % 4 == 0;
}
static void launch_conv_phase_resident(const TcConvArgs& a, cudaStream_t st) {
  constexpr int smem = 8 * 128 * 128 + kUpsStages * 128 * 128 + 2 * 128 * 36 * 4 + (2 * kUpsStages + 5) * 8 + 16 + 1024;
  const int dev = prepare_smem_launch<conv_phase_resident_kernel>(smem);
  const int per_phase = std::max(1, std::min(device_sm_count(dev) / a.nphase, a.ntiles_m));
  dim3 g(per_phase, a.nphase, 1);
  conv_phase_resident_kernel<<<g, 192, smem, st>>>(*reinterpret_cast<const CUtensorMap*>(a.tmA),
                                                   *reinterpret_cast<const CUtensorMap*>(a.tmB), a);
}

// Final phase of the persistent split-precision GEMMs (bias, activation, residual, scale, stores) for one epilogue warp:
// a thread holds one accumulator ROW (64 columns); storing that directly makes every warp-wide store touch 32
// different rows (32 x 16 B) and kept the drain warps away from the accumulator ring for ~12 k cycles per tile (the MMA
// warp then waits on the ring).  The warp transposes its 32 x 32 blocks through a private 4 KB smem scratch (16-byte
// chunks XOR-swizzled by row: conflict-free both ways, __syncwarp only): afterwards 8 lanes cover one 128-byte row
// segment, so residual loads and stores are full-line and the bias is one float4 per block.
__device__ __forceinline__ void gemm32_final(const TcConvArgs& a, float* scr, const float (&racc)[64], int b, int m0, int n0,
                                       int hh, int q, int lane, int mlen, int oro, const float* bias) {
  const int rq = lane >> 3, cq = lane & 7;
  const int out_row0 = a.out_off[b];
  const int res_row0 = a.res ? a.res_off[b] : 0;
#pragma unroll
  for (int blk = 0; blk < 2; blk++) {
#pragma unroll
    for (int j = 0; j < 8; j++)
      *reinterpret_cast<float4*>(scr + lane * 32 + ((j ^ (lane & 7)) << 2)) =
          make_float4(racc[blk * 32 + 4 * j], racc[blk * 32 + 4 * j + 1], racc[blk * 32 + 4 * j + 2], racc[blk * 32 + 4 * j + 3]);
    __syncwarp();
    const int n = n0 + hh * 64 + blk * 32 + cq * 4;
    if (n < a.Co) {
      const bool vec = a.vec4 && (n + 3 < a.Co);
      const float4 bb = bias ? epi_load4(bias + n, n, a.Co, vec) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 rv[8];
#pragma unroll
      for (int i = 0; i < 8; i++) {
        rv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int mm = m0 + q * 32 + rq + 4 * i;
        if (a.res && mm < mlen)
          rv[i] = epi_load4(a.res + ((size_t)(res_row0 + ((mm * a.ors + oro) >> a.res_shift)) * a.ldr + a.rcol) + n, n, a.Co, vec);
      }
#pragma unroll
      for (int i = 0; i < 8; i++) {
        const int r = rq + 4 * i;
        const int mm = m0 + q * 32 + r;
        if (mm >= mlen) continue;
        const float4 o = epi_math4(*reinterpret_cast<const float4*>(scr + r * 32 + ((cq ^ (r & 7)) << 2)), a.wscale, bb, a.eact, rv[i], a.oscale);
        epi_store4(a.out + ((size_t)(out_row0 + mm * a.ors + oro) * a.ldo + a.ocol) + n, o, n, a.Co, vec, a.accumulate);
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------------------
// Persistent split-TF32 GEMM / conv (BN = 128, 3 stages of 4 x 16 KB operand planes).  One CTA per SM
// walks tiles t = blockIdx.x + i*gridDim.x of the (n-tile, item, m-tile) space, m fastest.  Same arithmetic
// and chain-split accumulation as conv_tc_kernel<128,3,1> (bit-identical results), but the TMA / MMA pipeline
// runs straight across tile boundaries: measured on the single-tile kernel, only ~46 % of a tile's time was
// MMA work -- the rest was launch + TMEM allocation + pipeline ramp (~14 %) and the final epilogue (~20 %),
// neither overlapped with anything at one CTA per SM.  Here the epilogue pulls the small-terms accumulator
// into registers right after the last chain, hands all of TMEM back, and finishes (smem transpose, bias,
// activation, residual, stores) from registers while the next tile's operands stream in and its MMAs run.
constexpr int kGemm32pThreads = 320;   // TMA warp, MMA warp, 8 epilogue warps
__global__ void __launch_bounds__(kGemm32pThreads, 1) gemm32p_kernel(const __grid_constant__ CUtensorMap tmA,
                                                         const __grid_constant__ CUtensorMap tmB,
                                                         const __grid_constant__ CUtensorMap tmA2,
                                                         const __grid_constant__ CUtensorMap tmB2,
                                                         TcConvArgs a) {
  constexpr int BN = 128, STAGES = 3;
  const bool f16 = a.f16 != 0;                 // split-FP16 planes instead of split-TF32
  const int KE = f16 ? 64 : 32;                // K elements per 128-byte span
  const int cs = f16 ? 0 : 1;                  // log2(stages per hi*hi chain): a chain is 64 K-elements either way
  constexpr uint32_t A_BYTES = 128 * 128, B_BYTES = BN * 128, STAGE_BYTES = 2 * (A_BYTES + B_BYTES);
  constexpr int NEPI = (kGemm32pThreads - 64) / 32;     // epilogue warps: 8 = two column halves x four TMEM lane quadrants
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t scr_base = base + STAGES * STAGE_BYTES;       // 8 epilogue warps x 4 KB transpose scratch
  float* const scr_f = reinterpret_cast<float*>(smem_raw + (scr_base - smem_u32(smem_raw)));
  const uint32_t bar_base = scr_base + 8 * 4096;               // full[3], empty[3], bfull[3], bempty[3], sfull, sfree
  const uint32_t tmem_slot = bar_base + 14 * 8;
  auto full_bar = [&](int s) { return bar_base + s * 8; };
  auto empty_bar = [&](int s) { return bar_base + (3 + s) * 8; };
  auto bfull_bar = [&](int j) { return bar_base + (6 + j) * 8; };
  auto bempty_bar = [&](int j) { return bar_base + (9 + j) * 8; };
  const uint32_t sfull_bar = bar_base + 12 * 8, sfree_bar = bar_base + 13 * 8;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kchunks = a.Cpad / KE;
  const int num_k = a.ks * kchunks;
  const int nchains = (num_k + cs) >> cs;
  const int ntm = a.ntiles_m;
  const int total = ntm * ((a.Co + BN - 1) / BN);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmA2);
    prefetch_tmap(&tmB2);
    for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int j = 0; j < 3; j++) { mbar_init(bfull_bar(j), 1); mbar_init(bempty_bar(j), NEPI); }
    mbar_init(sfull_bar, 1); mbar_init(sfree_bar, NEPI);
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, 512u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  // tile -> (n-tile, item, m-tile); tile_start is the prefix sum of ceil(m_len / 128) over the items
  // Order: groups of `gm` consecutive m-tiles whose operand planes (~48 MB) stay L2-resident while all the
  // n-tiles of the group are computed (n outer, m inner inside a group) -- the activation planes of a whole
  // GEMM (200 MB at M = 32768, K = 768) do not fit the 126 MB L2.
  const int NT = (a.Co + BN - 1) / BN;
  const int gm = a.group_m;
  auto decode = [&](int t, int& b, int& m0, int& n0) {
    const int g = t / (gm * NT), r = t - g * gm * NT;
    const int gsz = min(gm, ntm - g * gm);
    const int nt = r / gsz, mg = g * gm + (r - nt * gsz);
    int lo = 0, hi = a.B;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (a.tile_start[mid] <= mg) lo = mid; else hi = mid;
    }
    b = lo; m0 = (mg - a.tile_start[lo]) * 128; n0 = nt * BN;
  };

  if (warp == 0) {
    if (lane == 0) {
      int g = 0;
      TCT_DECL(2);
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        int b, m0, n0;
        decode(t, b, m0, n0);
        const int row0 = a.in_off[b] + m0 - a.pad;
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          TCT(1);
          mbar_wait(empty_bar(s), (((uint32_t)(g / STAGES)) & 1u) ^ 1u);
          TCT(0);
          const int tap = it / kchunks, c0 = (it - tap * kchunks) * KE;
          const uint32_t sa = base + s * STAGE_BYTES;
          mbar_expect_tx(full_bar(s), STAGE_BYTES);
          tma_load_2d(sa, &tmA, c0, row0 + tap * a.dil, full_bar(s));
          tma_load_2d(sa + A_BYTES, &tmA2, c0, row0 + tap * a.dil, full_bar(s));
          tma_load_2d(sa + 2 * A_BYTES, &tmB, tap * a.Cpad + c0, n0, full_bar(s));
          tma_load_2d(sa + 2 * A_BYTES + B_BYTES, &tmB2, tap * a.Cpad + c0, n0, full_bar(s));
        }
      }
      TCT_FLUSH(0, 2);
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = f16 ? umma_idesc_f16(128, BN) : umma_idesc_tf32(128, BN);
      int g = 0, gc = 0, ti = 0;
      TCT_DECL(4);
      for (int t = blockIdx.x; t < total; t += gridDim.x, ti++) {
        // the small-terms accumulator of the previous tile must have been pulled into registers
        TCT(2);
        if (ti > 0) { mbar_wait(sfree_bar, (uint32_t)(ti - 1) & 1u); tc_fence_after(); }
        TCT(3);
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          mbar_wait(full_bar(s), ((uint32_t)(g / STAGES)) & 1u);
          tc_fence_after();
          TCT(0);
          const uint32_t sa = base + s * STAGE_BYTES;
          const int G = gc + (it >> cs), j = G % 3;
          const bool chain_start = (it & cs) == 0;
          if (chain_start && G >= 3) {           // ring slot j must have been drained by the epilogue
            mbar_wait(bempty_bar(j), (uint32_t)(G / 3 - 1) & 1u);
            tc_fence_after();
          }
          TCT(1);
          const uint64_t ah = umma_desc_sw128(sa), al = umma_desc_sw128(sa + A_BYTES);
          const uint64_t bh = umma_desc_sw128(sa + 2 * A_BYTES), bl = umma_desc_sw128(sa + 2 * A_BYTES + B_BYTES);
          const uint32_t t_small = tmem_base, t_big = tmem_base + (uint32_t)(BN * (1 + j));
#pragma unroll
          for (int k = 0; k < 4; k++) {  // 4 x (32 B of K: 8 tf32 or 16 fp16)
            const uint64_t o = (uint64_t)(2 * k);
            if (a.nprod >= 4) umma_split(t_small, al + o, bl + o, idesc, (it | k) ? 1u : 0u, f16);
            umma_split(t_small, al + o, bh + o, idesc, (a.nprod >= 4 || (it | k)) ? 1u : 0u, f16);
            umma_split(t_small, ah + o, bl + o, idesc, 1u, f16);
            umma_split(t_big, ah + o, bh + o, idesc, (chain_start && k == 0) ? 0u : 1u, f16);
          }
          if ((it & cs) == cs || it == num_k - 1) umma_commit(bfull_bar(j));  // chain complete
          umma_commit(empty_bar(s));
          TCT(2);
        }
        umma_commit(sfull_bar);
        gc += nchains;
      }
      TCT_FLUSH(4, 4);
    }
  } else {
    // ---- epilogue: 8 warps.  Warp w owns TMEM lane quadrant q = w & 3 (its 32 accumulator rows) and column half
    // hh = (w - 2) >> 2 (64 of the tile's 128 columns); a thread holds ONE row x 64 columns in registers.
    // Round 1 ran this with 4 warps x 128 columns and four sequential 32-column tcgen05.ld + wait round trips per
    // chain: at ~3 000 cycles per drained chain the epilogue warps -- not the tensor pipe, not L2 -- set the pace of
    // every large split-precision GEMM (the per-chain time was the same for K = 768 and K = 2048, for tf32 and for
    // fp16 planes).  Two column halves and one 64-column load per chain cut the drain to one TMEM round trip.
    const int q = warp & 3;
    const int hh = (warp - 2) >> 2;
    const int et = q * 32 + lane;           // accumulator row held by this thread
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(hh * 64);
    int gc = 0, ti = 0;
#ifdef KKX_TC_TIMING
    long long tct_acc[4] = {0}; long long tct_last = clock64();
    const bool tct_on = a.timing && blockIdx.x == gridDim.x - 2 && threadIdx.x == 64;
#endif
    for (int t = blockIdx.x; t < total; t += gridDim.x, ti++) {
      int b, m0, n0;
      decode(t, b, m0, n0);
      const int mlen = a.m_len[b];
      float racc[64];
#pragma unroll
      for (int e = 0; e < 64; e++) racc[e] = 0.f;
      for (int ch = 0; ch < nchains; ch++) {
        const int G = gc + ch, j = G % 3;
        mbar_wait(bfull_bar(j), (uint32_t)(G / 3) & 1u);
        tc_fence_after();
        TCT(0);
        {
          uint32_t v[64];
          tmem_ld64(tq + (uint32_t)(BN * (1 + j)), v);
#pragma unroll
          for (int e = 0; e < 64; e++) racc[e] += __uint_as_float(v[e]);
        }
        tc_fence_before();
        if (lane == 0) mbar_arrive(bempty_bar(j));
        TCT(1);
      }
      gc += nchains;
      mbar_wait(sfull_bar, (uint32_t)ti & 1u);
      tc_fence_after();
      TCT(2);
      {
        uint32_t v[64];
        tmem_ld64(tq, v);
#pragma unroll
        for (int e = 0; e < 64; e++) racc[e] = __uint_as_float(v[e]) + racc[e];   // same order as the single-tile kernel
      }
      tc_fence_before();
      if (lane == 0) mbar_arrive(sfree_bar);   // TMEM is free again

      // ---- the rest runs while the next tile's pipeline is already going (see gemm32_final)
      gemm32_final(a, scr_f + (warp - 2) * 1024, racc, b, m0, n0, hh, q, lane, mlen, a.oro, a.bias);
      TCT(3);
    }
    TCT_FLUSH(8, 4);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512u);
  }
}

static void launch_gemm32p(const TcConvArgs& a, cudaStream_t st) {
  constexpr int smem = 3 * 4 * 128 * 128 + 8 * 4096 + 14 * 8 + 16 + 1024;
  const int dev = prepare_smem_launch<gemm32p_kernel>(smem);
  const int nsm = device_sm_count(dev);
  const int total = a.ntiles_m * ((a.Co + 127) / 128);
  const int grid = total < nsm ? total : nsm;
  TcConvArgs b = a;
  const long long per_tile = 128LL * a.Cpad * (a.f16 ? 4 : 8);       // bytes of hi+lo planes of one m-tile
  long long gm = 24LL * 1000000LL / (per_tile > 0 ? per_tile : 1);
  if (gm < 8) gm = 8;
  if (gm > a.ntiles_m) gm = a.ntiles_m;
  b.group_m = (int)gm;
  gemm32p_kernel<<<grid, kGemm32pThreads, smem, st>>>(*reinterpret_cast<const CUtensorMap*>(a.tmA), *reinterpret_cast<const CUtensorMap*>(a.tmB),
                                          *reinterpret_cast<const CUtensorMap*>(a.tmA2), *reinterpret_cast<const CUtensorMap*>(a.tmB2), b);
}

// ------------------------------------------------------------------------------------------
// CTA-pair version of the persistent split-FP16 GEMM (cta_group::2, clusters of two CTAs along M).
// Role counters of gemm32p_kernel showed the MMA warp's issue time at ~1270 cycles per 64-K stage against a tensor-pipe
// floor of 768: a stage moves 64 KB of TMA writes plus 12 x 8 KB of operand reads through the SM's 128 B/clk shared-
// memory port (160 KB -> 1250 cycles), and the 148 CTAs together pull ~7.5 KB/clk out of L2 -- both above what the
// hardware gives.  A pair computes a 256 x 128 tile with ONE tcgen05.mma.cta_group::2 per K step: each CTA supplies its
// own 128 rows of A (hi and lo planes) and only HALF of the weight tile (64 of the 128 rows of B); the tensor cores read
// the other half from the peer's shared memory.  Per CTA and stage: 48 KB of TMA writes + 12 x 6 KB of operand reads
// (120 KB, -25 %) and 48 instead of 64 KB from L2.
//   * both CTAs run a TMA warp; all loads of a stage count their bytes on the LEADER's full barrier (cta_group::2 TMA);
//   * only the leader issues MMAs; its commits arrive on the barriers of both CTAs (multicast);
//   * each CTA drains / finishes its own 128 accumulator rows exactly like gemm32p_kernel (same arithmetic, same order:
//     bit-identical results); "ring slot drained" / "small accumulator pulled" arrivals of both CTAs go to the leader.
// The two m-tiles of a pair are consecutive entries of the m-tile list (they may belong to different items); an odd
// list ends with a pair whose second CTA recomputes the last tile and stores nothing.
//   * the finished tile leaves through shared memory: the 8 drain warps only accumulate chains (registers) and drop the
//     128 x 128 fp32 result into a 64 KB staging tile; 6 "final" warps apply bias / activation / residual / scale and
//     store whole 512-byte rows while the drain warps are already on the next tile.  (With the final phase on the drain
//     warps the accumulator ring was not drained for ~8 k cycles per tile and the MMA warp spent 13 of its 36 Mcycles
//     per step waiting for a ring slot.)
constexpr int kG2Stages = 3;
// final warps: 16 warps x 128 registers fill the register file (registers are granted in steps of 32 per thread, so 18
// warps would get 96).  4 final warps measured slower: the GELU + plane split of the FFN GEMM (128 tanh per lane and
// tile) and the transposed V pass of the QKV GEMM took longer than the tile's MMAs (ncu: tensor pipe 29 % / 38 % active
// against 52 % for the plain GEMMs); the 89 split-precision GEMMs of a B = 64 step 25.7-25.8 ms against 23.3-23.9 ms
// with 6 (profiles/r2_gemm_final_warps_ab_v29.txt).
constexpr int kG2Fin = 6;
constexpr int kG2Threads = (2 + 8 + kG2Fin) * 32;   // TMA warp, MMA warp, 8 drain warps, the final warps
constexpr uint32_t kG2A = 128 * 128, kG2Bh = 64 * 128, kG2Stage = 2 * (kG2A + kG2Bh);
constexpr uint32_t kG2Stg = 128 * 128 * 4;
constexpr int kG2Smem = kG2Stages * (int)kG2Stage + (int)kG2Stg + 20 * 8 + 16 + 1024;
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kG2Threads, 1)
gemm32p2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh,
                const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2h, TcConvArgs a) {
  constexpr int BN = 128, STAGES = kG2Stages, NFIN = kG2Fin;
  constexpr int KE = 64;                                   // K elements per 128-byte span (fp16 planes); one chain per stage
  constexpr int NEPI = 8;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t stg_base = base + STAGES * kG2Stage;      // finished tile, fp32 [128][128], 16-byte chunks XOR-swizzled by row
  float* const stg_f = reinterpret_cast<float*>(smem_raw + (stg_base - smem_u32(smem_raw)));
  const uint32_t bar_base = stg_base + kG2Stg;             // full[4], empty[4], bfull[3], bempty[3], sfull, sfree, gfull, gfree
  const uint32_t tmem_slot = bar_base + 20 * 8;
  auto full_bar = [&](int s) { return bar_base + s * 8; };
  auto empty_bar = [&](int s) { return bar_base + (4 + s) * 8; };
  auto bfull_bar = [&](int j) { return bar_base + (8 + j) * 8; };
  auto bempty_bar = [&](int j) { return bar_base + (11 + j) * 8; };
  const uint32_t sfull_bar = bar_base + 14 * 8, sfree_bar = bar_base + 15 * 8;
  const uint32_t gfull_bar = bar_base + 16 * 8, gfree_bar = bar_base + 17 * 8;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int kchunks = a.Cpad / KE;
  const int num_k = a.ks * kchunks;                        // stages = chains per tile
  const int ntm = a.ntiles_m, ntm2 = (ntm + 1) >> 1;
  const int NT = (a.Co + BN - 1) / BN;
  const int total = ntm2 * NT;
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmBh);
    prefetch_tmap(&tmA2);
    prefetch_tmap(&tmB2h);
    for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int j = 0; j < 3; j++) { mbar_init(bfull_bar(j), 1); mbar_init(bempty_bar(j), 2 * NEPI); }
    mbar_init(sfull_bar, 1); mbar_init(sfree_bar, 2 * NEPI);
    mbar_init(gfull_bar, NEPI); mbar_init(gfree_bar, NFIN);
    mbar_init_fence();
  }
  if (warp == 1) {   // the same warp of both CTAs
    tmem_alloc<2>(tmem_slot, 512u);
  }
  tc_fence_before();
  cluster_sync_all();      // barriers of both CTAs initialised, TMEM of both allocated, before any cross-CTA traffic
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  // pair-tile -> (n-tile, this CTA's m-tile); groups of gm2 consecutive m-tile PAIRS stay L2-resident while all their
  // n-tiles are computed (same idea as gemm32p_kernel)
  const int gm2 = a.group_m > 1 ? (a.group_m >> 1) : 1;
  auto decode = [&](int t, int& b, int& m0, int& n0, bool& valid) {
    const int g = t / (gm2 * NT), r = t - g * gm2 * NT;
    const int gsz = min(gm2, ntm2 - g * gm2);
    const int nt = r / gsz;
    int mg = 2 * (g * gm2 + (r - nt * gsz)) + (int)rank;
    valid = mg < ntm;
    if (!valid) mg = ntm - 1;
    int lo = 0, hi = a.B;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (a.tile_start[mid] <= mg) lo = mid; else hi = mid;
    }
    b = lo; m0 = (mg - a.tile_start[lo]) * 128; n0 = nt * BN;
  };

  if (warp == 0) {
    if (lane == 0) {
      int g = 0;
      TCT_DECL(2);
      for (int t = pair; t < total; t += npairs) {
        int b, m0, n0; bool valid;
        decode(t, b, m0, n0, valid);
        const int row0 = a.in_off[b] + m0 - a.pad;
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          TCT(1);
          mbar_wait(empty_bar(s), (((uint32_t)(g / STAGES)) & 1u) ^ 1u);
          TCT(0);
          const int tap = it / kchunks, c0 = (it - tap * kchunks) * KE;
          const uint32_t sa = base + s * kG2Stage;
          const uint32_t lead_full = mapa_u32(full_bar(s), 0);
          if (rank == 0) mbar_expect_tx(full_bar(s), 2 * kG2Stage);      // the bytes of both CTAs
          tma_load_2d_pair(sa, &tmA, c0, row0 + tap * a.dil, lead_full);
          tma_load_2d_pair(sa + kG2A, &tmA2, c0, row0 + tap * a.dil, lead_full);
          tma_load_2d_pair(sa + 2 * kG2A, &tmBh, tap * a.Cpad + c0, n0 + (int)rank * 64, lead_full);
          tma_load_2d_pair(sa + 2 * kG2A + kG2Bh, &tmB2h, tap * a.Cpad + c0, n0 + (int)rank * 64, lead_full);
        }
      }
      TCT_FLUSH(0, 2);
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      const uint32_t idesc = umma_idesc_f16(256, BN);
      int g = 0, gc = 0, ti = 0;
      TCT_DECL(4);
      for (int t = pair; t < total; t += npairs, ti++) {
        TCT(2);
        if (ti > 0) { mbar_wait(sfree_bar, (uint32_t)(ti - 1) & 1u); tc_fence_after(); }
        TCT(3);
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          mbar_wait(full_bar(s), ((uint32_t)(g / STAGES)) & 1u);
          tc_fence_after();
          TCT(0);
          const uint32_t sa = base + s * kG2Stage;
          const int G = gc + it, j = G % 3;
          if (G >= 3) {                          // ring slot j must have been drained by the epilogues of both CTAs
            mbar_wait(bempty_bar(j), (uint32_t)(G / 3 - 1) & 1u);
            tc_fence_after();
          }
          TCT(1);
          const uint64_t ah = umma_desc_sw128(sa), al = umma_desc_sw128(sa + kG2A);
          const uint64_t bh = umma_desc_sw128(sa + 2 * kG2A), bl = umma_desc_sw128(sa + 2 * kG2A + kG2Bh);
          const uint32_t t_small = tmem_base, t_big = tmem_base + (uint32_t)(BN * (1 + j));
#pragma unroll
          for (int k = 0; k < 4; k++) {          // 4 x 16 fp16 of K; same products, same order as gemm32p_kernel
            const uint64_t o = (uint64_t)(2 * k);
            umma_f16_pair(t_small, al + o, bh + o, idesc, (it | k) ? 1u : 0u);
            umma_f16_pair(t_small, ah + o, bl + o, idesc, 1u);
            umma_f16_pair(t_big, ah + o, bh + o, idesc, k == 0 ? 0u : 1u);
          }
          umma_commit_pair(bfull_bar(j));        // chain complete (both CTAs)
          umma_commit_pair(empty_bar(s));        // stage free (both CTAs)
          TCT(2);
        }
        umma_commit_pair(sfull_bar);
        gc += num_k;
      }
      TCT_FLUSH(4, 4);
    }
  } else if (warp < 2 + NEPI) {
    // ---- drain warps: warp w owns TMEM lane quadrant q = w & 3 and column half hh; a thread accumulates one row x 64
    // columns over the tile's chains (two 32-column loads per chain keep this role inside its register budget)
    const int q = warp & 3;
    const int hh = (warp - 2) >> 2;
    const int et = q * 32 + lane;
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(hh * 64);
    const uint32_t lead_bars = mapa_u32(bar_base, 0);          // the leader's barrier block (same offsets)
    const uint32_t lead_sfree = lead_bars + 15 * 8;
    int gc = 0, ti = 0;
#ifdef KKX_TC_TIMING
    long long tct_acc[4] = {0}; long long tct_last = clock64();
    const bool tct_on = a.timing && blockIdx.x == gridDim.x - 2 && threadIdx.x == 64;
#endif
    for (int t = pair; t < total; t += npairs, ti++) {
      float racc[64];
#pragma unroll
      for (int e = 0; e < 64; e++) racc[e] = 0.f;
      for (int ch = 0; ch < num_k; ch++) {
        const int G = gc + ch, j = G % 3;
        mbar_wait(bfull_bar(j), (uint32_t)(G / 3) & 1u);
        tc_fence_after();
        TCT(0);
#pragma unroll
        for (int h2 = 0; h2 < 2; h2++) {
          uint32_t v[32];
          tmem_ld32(tq + (uint32_t)(BN * (1 + j) + h2 * 32), v);
#pragma unroll
          for (int e = 0; e < 32; e++) racc[h2 * 32 + e] += __uint_as_float(v[e]);
        }
        tc_fence_before();
        if (lane == 0) mbar_arrive_cluster(lead_bars + (uint32_t)(11 + j) * 8);
        TCT(1);
      }
      gc += num_k;
      mbar_wait(sfull_bar, (uint32_t)ti & 1u);
      tc_fence_after();
      TCT(2);
#pragma unroll
      for (int h2 = 0; h2 < 2; h2++) {
        uint32_t v[32];
        tmem_ld32(tq + (uint32_t)(h2 * 32), v);
#pragma unroll
        for (int e = 0; e < 32; e++) racc[h2 * 32 + e] = __uint_as_float(v[e]) + racc[h2 * 32 + e];   // same order as the single-tile kernel
      }
      tc_fence_before();
      if (lane == 0) mbar_arrive_cluster(lead_sfree);        // TMEM is free again
      // hand the finished rows to the final warps
      if (ti > 0) mbar_wait(gfree_bar, (uint32_t)(ti - 1) & 1u);
      float* const srow = stg_f + et * 128;
#pragma unroll
      for (int c = 0; c < 16; c++) {
        const int chunk = hh * 16 + c;                         // 16-byte chunk of the row; swizzle inside groups of 8 chunks
        *reinterpret_cast<float4*>(srow + (((chunk & ~7) | ((chunk ^ et) & 7)) << 2)) =
            make_float4(racc[4 * c], racc[4 * c + 1], racc[4 * c + 2], racc[4 * c + 3]);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(gfull_bar);
      TCT(3);
    }
    TCT_FLUSH(8, 4);
  } else {
    // ---- final warps: bias, activation, residual, scale and the stores, one 512-byte row per warp instruction (lane l
    // owns columns 4l .. 4l+3), rows fw, fw + NFIN, ... of the staged tile
    const int fw = warp - (2 + NEPI);
    int ti = 0;
    for (int t = pair; t < total; t += npairs, ti++) {
      int b, m0, n0; bool valid;
      decode(t, b, m0, n0, valid);
      const int mlen = valid ? a.m_len[b] : 0;                 // the duplicate tile of an odd list stores nothing
      const int n = n0 + lane * 4;
      const bool ncol = n < a.Co;
      const bool vec = a.vec4 && (n + 3 < a.Co);
      const float4 bb = a.bias && ncol ? epi_load4(a.bias + n, n, a.Co, vec) : make_float4(0.f, 0.f, 0.f, 0.f);
      const int out_row0 = a.out_off[b];
      const int res_row0 = a.res ? a.res_off[b] : 0;
      constexpr int RB = 4;                                    // rows per batch: residual loads of a batch are issued together
      auto res_ptr = [&](int mm) { return a.res + ((size_t)(res_row0 + ((mm * a.ors + a.oro) >> a.res_shift)) * a.ldr + a.rcol) + n; };
      auto load_res = [&](int i0, float4 (&rv)[RB]) {
#pragma unroll
        for (int i = 0; i < RB; i++) {
          rv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          const int mm = m0 + fw + NFIN * (i0 + i);
          if (a.res && ncol && mm < mlen && fw + NFIN * (i0 + i) < 128) rv[i] = epi_load4(res_ptr(mm), n, a.Co, vec);
        }
      };
      float4 rv[RB];
      load_res(0, rv);                                         // overlaps the wait for the tile
      mbar_wait(gfull_bar, (uint32_t)ti & 1u);
      if (a.attn_pl[0] && n0 >= 1536) {
        // QKV projection, V columns: the attention kernel wants V TRANSPOSED per head ([(item, head, d), key], pitch 512,
        // fp16 hi / lo of 16 v, zero-filled to a multiple of 64 keys).  The staged tile is read by columns instead: warp fw
        // takes every NFIN-th dim of the tile, a lane one token, so every store covers 32 consecutive keys (64 bytes).
        const int NR = (mlen + 63) & ~63;
        uint16_t* const vth = static_cast<uint16_t*>(a.attn_pl[4]);
        uint16_t* const vtl = static_cast<uint16_t*>(a.attn_pl[5]);
#pragma unroll 1
        for (int cl = fw; cl < 128; cl += NFIN) {                // column inside the tile
          const int cv = n0 - 1536 + cl;                       // V column: head * 64 + d
          const float bias_c = a.bias ? a.bias[n0 + cl] : 0.f;
          uint16_t* const vh = vth + ((size_t)b * 768 + cv) * 512 + m0;
          uint16_t* const vl = vtl + ((size_t)b * 768 + cv) * 512 + m0;
          const int chunk = cl >> 2, e4 = cl & 3;
#pragma unroll
          for (int tg = 0; tg < 4; tg++) {
            const int r = tg * 32 + lane;                      // token inside the tile
            if (m0 + r < NR) {
              const float raw = stg_f[r * 128 + (((chunk & ~7) | ((chunk ^ r) & 7)) << 2) + e4];
              uint32_t hi, lo;
              split_f16((m0 + r < mlen ? fmaf(raw, a.wscale, bias_c) : 0.f) * 16.0f, hi, lo);
              vh[r] = (uint16_t)hi;
              vl[r] = (uint16_t)lo;
            }
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(gfree_bar);
        continue;
      }
#pragma unroll 1
      for (int i0 = 0; i0 < (128 + NFIN - 1) / NFIN; i0 += RB) {
        float4 v[RB];
#pragma unroll
        for (int i = 0; i < RB; i++) {
          const int r = min(fw + NFIN * (i0 + i), 127);        // (rows past the tile are skipped below)
          v[i] = *reinterpret_cast<const float4*>(stg_f + r * 128 + (((lane & ~7) | ((lane ^ r) & 7)) << 2));
        }
        if (i0 + RB >= (128 + NFIN - 1) / NFIN) {             // last read of the staged tile
          __syncwarp();
          if (lane == 0) mbar_arrive(gfree_bar);
        }
#pragma unroll
        for (int i = 0; i < RB; i++) {
          const int mm = m0 + fw + NFIN * (i0 + i);
          if (mm >= mlen || !ncol || fw + NFIN * (i0 + i) >= 128) continue;
          const float4 o = epi_math4(v[i], a.wscale, bb, a.eact, rv[i], a.oscale);
          const size_t orow = (size_t)(out_row0 + mm * a.ors + a.oro);
          if (a.attn_pl[0]) {   // QKV projection, Q and K columns: fp16 hi / lo planes of 2 q (= 16 q / sqrt(64)) and 16 k
            const bool isq = n0 < 768;
            const float sc_ = isq ? 2.0f : 16.0f;
            const float e4[4] = {o.x, o.y, o.z, o.w};
            uint32_t hw[4], lw[4];
#pragma unroll
            for (int e = 0; e < 4; e++) split_f16(e4[e] * sc_, hw[e], lw[e]);
            const size_t pidx = orow * 768 + (size_t)(isq ? n : n - 768);
            *reinterpret_cast<uint2*>(static_cast<__half*>(a.attn_pl[isq ? 0 : 2]) + pidx) = make_uint2(hw[0] | (hw[1] << 16), hw[2] | (hw[3] << 16));
            *reinterpret_cast<uint2*>(static_cast<__half*>(a.attn_pl[isq ? 1 : 3]) + pidx) = make_uint2(lw[0] | (lw[1] << 16), lw[2] | (lw[3] << 16));
            continue;
          }
          if (a.out_hi) {      // operand planes for the next GEMM (host guarantees Co % 4 == 0, no accumulate)
            const float e4[4] = {o.x, o.y, o.z, o.w};
            uint32_t hw[4], lw[4];
#pragma unroll
            for (int e = 0; e < 4; e++) split_f16_operand(e4[e], hw[e], lw[e]);
            *reinterpret_cast<uint2*>(static_cast<__half*>(a.out_hi) + orow * a.out_pl_ld + n) = make_uint2(hw[0] | (hw[1] << 16), hw[2] | (hw[3] << 16));
            *reinterpret_cast<uint2*>(static_cast<__half*>(a.out_lo) + orow * a.out_pl_ld + n) = make_uint2(lw[0] | (lw[1] << 16), lw[2] | (lw[3] << 16));
            if (!a.out) continue;
          }
          epi_store4(a.out + (orow * a.ldo + a.ocol) + n, o, n, a.Co, vec, a.accumulate);
        }
        if (i0 + RB < (128 + NFIN - 1) / NFIN) load_res(i0 + RB, rv);
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();      // nobody leaves (or frees TMEM) while the peer may still signal it or the pair-MMAs read its smem
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<2>(tmem_base, 512u);
  }
}

static void launch_gemm32p2(const TcConvArgs& a, cudaStream_t st) {
  const int dev = prepare_smem_launch<gemm32p2_kernel>(kG2Smem);
  const int nsm = device_sm_count(dev);
  const int total = ((a.ntiles_m + 1) / 2) * ((a.Co + 127) / 128);
  int npairs = nsm / 2;
  if (npairs > total) npairs = total;
  TcConvArgs b = a;
  const long long per_tile = 128LL * a.Cpad * 4;                      // bytes of the hi + lo planes of one m-tile
  long long gm = 24LL * 1000000LL / (per_tile > 0 ? per_tile : 1);
  if (gm < 8) gm = 8;
  if (gm > a.ntiles_m) gm = a.ntiles_m;
  b.group_m = (int)gm;
  gemm32p2_kernel<<<2 * npairs, kG2Threads, kG2Smem, st>>>(*reinterpret_cast<const CUtensorMap*>(a.tmA), *reinterpret_cast<const CUtensorMap*>(a.tmB_c),
                                                         *reinterpret_cast<const CUtensorMap*>(a.tmA2), *reinterpret_cast<const CUtensorMap*>(a.tmB2_c), b);
}

// ------------------------------------------------------------------------------------------
// CTA-pair version of the bf16 implicit-GEMM conv (MODE 0) for the decoder's wide convs (Co a multiple of 256).
// The single-tile kernel pulls 48 KB per 64-channel K step and CTA out of L2 (A 16 KB, B 32 KB at BN = 256), two CTAs
// per SM: ~190 B/clk/SM against the ~42 B/clk/SM the L2 delivers chip-wide -- measured 30-45 % of the tensor floor.
// Here a pair of CTAs computes a 256 x 256 tile with tcgen05.mma.cta_group::2: each CTA loads its own 128 activation
// rows and HALF of the weight tile (32 KB per K step for twice the rows: a third of the L2 traffic per output row), the
// kernel is persistent (5-stage ring running across tiles, the same m-tile-pair scheduling as gemm32p2_kernel) and the
// two 256-column accumulators in TMEM alternate, so a tile's epilogue (per-warp smem transposes, full-line residual
// loads and stores: gemm32_final) runs under the next tile's MMAs.  Same accumulation order per output element as the
// single-tile kernel: identical bits.
// Phase-fused ConvTranspose1d launches (nphase > 1) are n-tiles like any other: tile (phase, n-tile, m-tile pair) reads
// the stacked weight rows of its phase, with the phase's tap shift and output row offset.
// BN is a template parameter, but only 256 is used: 128-wide pair tiles (Co = 128: the noise convs, the stage-1
// up-sampling) were measured SLOWER than the single-tile kernel (2.40 vs 1.72 ms and 2.06 vs 1.29 ms at 5.75 M output
// rows, profiles/r2_conv_pair_bn128_v30.txt) -- those convs have K = 64 ... 512 and are bound by the epilogue's stores,
// where three co-resident single-tile CTAs bring 12 epilogue warps per SM against 8 here.
template <int BN> struct CpCfg {
  static constexpr int STAGES = BN == 256 ? 5 : 7;
  static constexpr uint32_t A = 128 * 128, Bh = (BN / 2) * 128, STAGE = A + Bh;
  static constexpr int SMEM = STAGES * (int)STAGE + 8 * 4096 + 20 * 8 + 16 + 1024;
};
constexpr int kCpThreads = 320;    // TMA warp, MMA warp, 8 epilogue warps
template <int BN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kCpThreads, 1)
conv_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh, TcConvArgs a) {
  using Cfg = CpCfg<BN>;
  constexpr int STAGES = Cfg::STAGES, NEPI = 8;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t scr_base = base + STAGES * Cfg::STAGE;     // 8 epilogue warps x 4 KB transpose scratch
  float* const scr_f = reinterpret_cast<float*>(smem_raw + (scr_base - smem_u32(smem_raw)));
  const uint32_t bar_base = scr_base + 8 * 4096;            // full[S], empty[S], tfull[2], tempty[2]
  const uint32_t tmem_slot = bar_base + 20 * 8;
  auto full_bar = [&](int s) { return bar_base + s * 8; };
  auto empty_bar = [&](int s) { return bar_base + (STAGES + s) * 8; };
  auto tfull_bar = [&](int j) { return bar_base + (2 * STAGES + j) * 8; };
  auto tempty_bar = [&](int j) { return bar_base + (2 * STAGES + 2 + j) * 8; };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int kchunks = a.Cpad >> 6;
  const int num_k = a.ks * kchunks;
  const int ntm = a.ntiles_m, ntm2 = (ntm + 1) >> 1;
  const int ntn = a.Co / BN;                                // n-tiles per phase
  const int NT = ntn * (a.nphase > 1 ? a.nphase : 1);
  const int total = ntm2 * NT;
  const int npairs = gridDim.x >> 1, pair = blockIdx.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmBh);
    for (int s = 0; s < STAGES; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int j = 0; j < 2; j++) { mbar_init(tfull_bar(j), 1); mbar_init(tempty_bar(j), 2 * NEPI); }
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<2>(tmem_slot, 512u);
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  const int gm2 = a.group_m > 1 ? (a.group_m >> 1) : 1;
  // tile -> (item, m-tile of this CTA, phase, first output channel); n-tiles (all phases) are the outer loop inside a
  // group of m-tile pairs, so a group's activation tiles are served from L2 for every phase and n-tile
  auto decode = [&](int t, int& b, int& m0, int& ph, int& n0, bool& valid) {
    const int g = t / (gm2 * NT), r = t - g * gm2 * NT;
    const int gsz = min(gm2, ntm2 - g * gm2);
    const int nt = r / gsz;
    int mg = 2 * (g * gm2 + (r - nt * gsz)) + (int)rank;
    valid = mg < ntm;
    if (!valid) mg = ntm - 1;
    int lo = 0, hi = a.B;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (a.tile_start[mid] <= mg) lo = mid; else hi = mid;
    }
    b = lo; m0 = (mg - a.tile_start[lo]) * 128;
    ph = nt / ntn; n0 = (nt - ph * ntn) * BN;
  };

  if (warp == 0) {
    if (lane == 0) {
      int g = 0;
      for (int t = pair; t < total; t += npairs) {
        int b, m0, ph, n0; bool valid;
        decode(t, b, m0, ph, n0, valid);
        const int c_pad = a.nphase > 1 ? a.phase_pad[ph] : a.pad;
        const int row0 = a.in_off[b] + m0 - c_pad;
        const int wrow = ph * a.Co + n0 + (int)rank * (BN / 2);         // this CTA's half of the (phase-stacked) weight tile
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          mbar_wait(empty_bar(s), (((uint32_t)(g / STAGES)) & 1u) ^ 1u);
          const int tap = it / kchunks, c0 = (it - tap * kchunks) << 6;
          const uint32_t sa = base + s * Cfg::STAGE;
          const uint32_t lead_full = mapa_u32(full_bar(s), 0);
          if (rank == 0) mbar_expect_tx(full_bar(s), 2 * Cfg::STAGE);
          tma_load_2d_pair(sa, &tmA, c0, row0 + tap * a.dil, lead_full);
          tma_load_2d_pair(sa + Cfg::A, &tmBh, tap * a.Cpad + c0, wrow, lead_full);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BN);
      int g = 0, ti = 0;
      for (int t = pair; t < total; t += npairs, ti++) {
        const int buf = ti & 1;
        mbar_wait(tempty_bar(buf), (((uint32_t)(ti >> 1)) & 1u) ^ 1u);   // both CTAs' epilogues are done with this accumulator
        tc_fence_after();
        const uint32_t td = tmem_base + (uint32_t)(buf * BN);
        for (int it = 0; it < num_k; it++, g++) {
          const int s = g % STAGES;
          mbar_wait(full_bar(s), ((uint32_t)(g / STAGES)) & 1u);
          tc_fence_after();
          const uint32_t sa = base + s * Cfg::STAGE;
          const uint64_t ad = umma_desc_sw128(sa), bd = umma_desc_sw128(sa + Cfg::A);
#pragma unroll
          for (int k = 0; k < 4; k++) umma_f16_pair(td, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (it | k) ? 1u : 0u);
          umma_commit_pair(empty_bar(s));
        }
        umma_commit_pair(tfull_bar(buf));
      }
    }
  } else {
    // epilogue: warp w owns TMEM lane quadrant q = w & 3 (32 rows) and column half hh (BN / 2 columns)
    const int q = warp & 3;
    const int hh = (warp - 2) >> 2;
    const uint32_t lead_bars = mapa_u32(bar_base, 0);
    int ti = 0;
    for (int t = pair; t < total; t += npairs, ti++) {
      int b, m0, ph, n0; bool valid;
      decode(t, b, m0, ph, n0, valid);
      const int mlen = valid ? a.m_len[b] : 0;
      const int c_oro = a.nphase > 1 ? a.phase_oro[ph] : a.oro;
      const int buf = ti & 1;
      mbar_wait(tfull_bar(buf), ((uint32_t)(ti >> 1)) & 1u);
      tc_fence_after();
      const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + hh * (BN / 2));
#pragma unroll 1
      for (int h2 = 0; h2 < BN / 128; h2++) {
        float racc[64];
#pragma unroll
        for (int c = 0; c < 2; c++) {
          uint32_t v[32];
          tmem_ld32(tq + (uint32_t)(h2 * 64 + c * 32), v);
#pragma unroll
          for (int e = 0; e < 32; e++) racc[c * 32 + e] = __uint_as_float(v[e]);
        }
        if (h2 == BN / 128 - 1) {      // last TMEM read of this tile by this warp: hand the accumulator back
          tc_fence_before();
          if (lane == 0) mbar_arrive_cluster(lead_bars + (uint32_t)(2 * STAGES + 2 + buf) * 8);
        }
        gemm32_final(a, scr_f + (warp - 2) * 1024, racc, b, m0, n0 + hh * (BN / 2) + h2 * 64, 0, q, lane, mlen, c_oro, a.bias);
      }
    }
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<2>(tmem_base, 512u);
  }
}

// true when launch_conv_tc runs the bf16 CTA-pair kernel for these arguments (tmB_c: the weight map with 128-row boxes)
static bool conv_tc_takes_pair_bf16(const TcConvArgs& a, int nsm) {
  if (a.tf32 || !a.pair || !a.tmB_c) return false;
  if (a.Co < 256 || a.Co % 256 != 0 || !a.tile_start || a.ntiles_m < 2) return false;
  return (long long)((a.ntiles_m + 1) / 2) * (a.Co / 256) * (a.nphase > 1 ? a.nphase : 1) >= nsm / 2;     // at least one tile per pair
}

template <int BN>
static void launch_conv_pair_t(const TcConvArgs& a, cudaStream_t st) {
  const int dev = prepare_smem_launch<conv_pair_kernel<BN>>(CpCfg<BN>::SMEM);
  const int nsm = device_sm_count(dev);
  const int total = ((a.ntiles_m + 1) / 2) * (a.Co / BN) * (a.nphase > 1 ? a.nphase : 1);
  int npairs = nsm / 2;
  if (npairs > total) npairs = total;
  TcConvArgs b = a;
  const long long per_tile = 128LL * a.Cpad * 2;                      // activation bytes of one m-tile
  long long gm = 24LL * 1000000LL / (per_tile > 0 ? per_tile : 1);
  if (gm < 8) gm = 8;
  if (gm > a.ntiles_m) gm = a.ntiles_m;
  b.group_m = (int)gm;
  conv_pair_kernel<BN><<<2 * npairs, kCpThreads, CpCfg<BN>::SMEM, st>>>(*reinterpret_cast<const CUtensorMap*>(a.tmA), *reinterpret_cast<const CUtensorMap*>(a.tmB_c), b);
}
static void launch_conv_pair(const TcConvArgs& a, cudaStream_t st) { launch_conv_pair_t<256>(a, st); }

template <int BN, int STAGES>
static void launch_tc_multi(const TcConvArgs& a, cudaStream_t st) {
  constexpr int smem = STAGES * (128 * 128 + BN * 128) + 2 * 128 * 36 * 4 + (2 * STAGES + 4) * 8 + 16 + 1024;
  prepare_smem_launch<conv_tc_multi_kernel<BN, STAGES>>(smem);
  dim3 g((a.max_m + 127) / 128, (a.Co + BN - 1) / BN, a.B);
  conv_tc_multi_kernel<BN, STAGES><<<g, 192, smem, st>>>(*reinterpret_cast<const CUtensorMap*>(a.tmA),
                                                         *reinterpret_cast<const CUtensorMap*>(a.tmB), a);
}

template <int BN, int STAGES, int MODE>
static void launch_tc(const TcConvArgs& a, cudaStream_t st) {
  constexpr int PLANES = MODE ? 2 : 1;
  constexpr int smem = STAGES * PLANES * (128 * 128 + BN * 128) + (2 * STAGES + 7) * 8 + 16 + 1024;
  prepare_smem_launch<conv_tc_kernel<BN, STAGES, MODE>>(smem);
  const unsigned gx = (unsigned)((a.max_m + 127) / 128);
  dim3 g(gx, (a.Co + BN - 1) / BN, a.B);
  if (MODE == 0 && a.nphase > 1) g = dim3((unsigned)(a.nphase * ((a.Co + BN - 1) / BN)), gx, a.B);
  const CUtensorMap* mA = reinterpret_cast<const CUtensorMap*>(a.tmA);
  const CUtensorMap* mB = reinterpret_cast<const CUtensorMap*>(a.tmB);
  const CUtensorMap* mA2 = reinterpret_cast<const CUtensorMap*>(a.tmA2 ? a.tmA2 : a.tmA);
  const CUtensorMap* mB2 = reinterpret_cast<const CUtensorMap*>(a.tmB2 ? a.tmB2 : a.tmB);
  conv_tc_kernel<BN, STAGES, MODE><<<g, 192, smem, st>>>(*mA, *mB, *mA2, *mB2, a);
}

bool conv_tc_takes_pair(const TcConvArgs& a) {
  if (!(a.tf32 && a.f16 && a.pair && a.nprod == 3 && a.tmA2 && a.tmB2 && a.tmB_c && a.tmB2_c)) return false;
  if (!(a.Co > 64 && a.tile_start && a.ntiles_m >= 2)) return false;
  if (a.force_kernel == 0) {   // small problems take the 64-wide single-tile kernel (see launch_conv_tc)
    int dev = 0;
    cudaGetDevice(&dev);
    const long long tiles128 = (long long)a.ntiles_m * ((a.Co + 127) / 128);
    if (tiles128 < device_sm_count(dev)) return false;
  }
  return true;
}

void launch_conv_tc(const TcConvArgs& a0, cudaStream_t st) {
  if (g_dry_run) return;
  if (a0.max_m <= 0 || a0.B <= 0) return;
  TcConvArgs a = a0;
#ifdef KKX_TC_DEBUG
  static const int dbg = [] { const char* e = getenv("KKX_TC_DEBUG"); return e ? atoi(e) : 0; }();
  a.debug = dbg;
#else
  a.debug = 0;
#endif
  a.vec4 = ((a.ldo | a.ocol) % 4 == 0) && (!a.res || ((a.ldr | a.rcol) % 4 == 0)) ? 1 : 0;
  if (g_launch_stats) g_launch_stats->conv_flops += 2.0 * (double)a.sum_m * a.Co * a.Ci * a.ks * (a.nphase > 1 ? a.nphase : 1);
  if (a.nphase > 1 && (a.tf32 || a.nphase > 10 || a.Co % tc_box_n(a.Co) != 0)) throw ArgError("launch_conv_tc: unsupported phase-fused shape");
  if (a.tf32) {
    // split-TF32: 4 operand planes per stage (64 KB at BN=128) -> 3 stages, one CTA per SM
    // Small problems (one utterance): fewer 128-wide tiles than SMs -> 64-wide single-tile CTAs fill twice as many
    // SMs and shorten the latency-bound launch (B=1, 510 tokens: 3.4 -> 2.8 ms over the 74 GEMMs of a step).  The
    // per-element accumulation order is the same in both kernels, so results do not depend on the choice.
    int cur_dev = 0;
    cudaGetDevice(&cur_dev);
    const int nsm = device_sm_count(cur_dev);
    const long long tiles128 = (long long)(a.ntiles_m > 0 ? a.ntiles_m : (a.sum_m + 127) / 128) * ((a.Co + 127) / 128);
    const bool small = tiles128 < nsm && a.tmB_c && a.tmB2_c && a.force_kernel == 0;
    if (a.Co > 64 && small) {
      TcConvArgs b = a; b.tmB = a.tmB_c; b.tmB2 = a.tmB2_c;
      launch_tc<64, 4, 1>(b, st);
    } else if (a.Co > 64 && a.tile_start && a.ntiles_m > 0 && a.tmA2 && a.tmB2) {
      // CTA pairs (cta_group::2) for the split-FP16 planes when the weight maps with 64-row boxes exist
      if (conv_tc_takes_pair(a)) launch_gemm32p2(a, st);
      else launch_gemm32p(a, st);
    }
    else if (a.Co > 64) launch_tc<128, 3, 1>(a, st);
    else launch_tc<64, 4, 1>(a, st);
    if (g_launch_stats && g_launch_stats->profile && g_launch_stats->detail) {
      char nm[96]; snprintf(nm, sizeof nm, "conv_tc_tf32x3[ci%d co%d k%d m%lld]", a.Ci, a.Co, a.ks, a.sum_m);
      post_launch(nm, st);
    } else post_launch("conv_tc_tf32x3", st);
    return;
  }
  // smem per CTA ~97 KB in every configuration -> two CTAs per SM, so one tile's epilogue overlaps
  // the other's TMA/MMA main loop (TMEM: 2 x 256 columns = the whole 512-column file)
  // Multi-tile CTAs (4 tiles per CTA, pipeline across tiles, double-buffered TMEM accumulators) measured slower than
  // 2-3 co-resident single-tile CTAs: 202 vs 182 ms per B=64 step.  The kernel is bound by L2->SM operand traffic
  // (A re-fetched per tap, B per tile), not by prologue / epilogue serialisation (profiles/r1_conv_tc_experiments.txt).
  int pdev = 0;
  cudaGetDevice(&pdev);
  if (a.phase_loop == 3 && conv_phase_resident_ok(a)) {
    launch_conv_phase_resident(a, st);     // stage-1 up-sampling of a batch: persistent CTAs with one phase's weights resident
  } else if (a.nphase > 1 && a.Co == 128 && a.phase_loop && !a.res && !a.accumulate) {
    // one CTA loops over the phases of its m-tile (2 stages: two CTAs per SM; 3: one)
    if (a.phase_loop == 2) launch_tc_multi<128, 3>(a, st);
    else launch_tc_multi<128, 2>(a, st);
  }
  else if (conv_tc_takes_pair_bf16(a, device_sm_count(pdev))) launch_conv_pair(a, st);   // wide convs of big batches: CTA pairs
  else if (a.Co > 128) launch_tc<256, 2, 0>(a, st);
  else if (a.Co > 64) launch_tc<128, 2, 0>(a, st);   // 65 KB smem -> three CTAs per SM
  else launch_tc<64, 4, 0>(a, st);
  if (g_launch_stats && g_launch_stats->profile && g_launch_stats->detail) {
    char nm[96]; snprintf(nm, sizeof nm, "conv_tc[ci%d co%d k%d%s m%lld]", a.Ci, a.Co, a.ks, a.nphase > 1 ? " phases" : "", a.sum_m);
    post_launch(nm, st);
  } else post_launch("conv_tc", st);
}

// ------------------------------------------------------------------------------------------
// Operand producer: out_bf16[r, c] = act(x[r, c] * scale[b, c] + shift[b, c]) for rows of item b,
// 0 for halo/gap rows and for pad columns c >= C.  Covers rows [off-gap, off+len+gap_after).
// Each thread produces 4 consecutive channels (float4 load when aligned, one 8-byte store); the
// bf16 result absorbs the error of the fast sin / division intrinsics used for Snake.
__device__ __forceinline__ float apply_act(float v, int act, float slope, float al) {
  if (act == ACT_LRELU) return v > 0.f ? v : v * slope;
  if (act == ACT_SNAKE) { const float s = __sinf(al * v); return v + __fdividef(s * s, al); }
  return v;
}
constexpr int kApplyRows = 16;  // rows per CTA (tf32 producer)
constexpr int kApplyRowsB = 64; // rows per CTA (bf16 producer)
__global__ void __launch_bounds__(256) apply_bf16_kernel(const float* __restrict__ x, int ldx, int C,
                                                         const float* scale, const float* shift,
                                                         int act, float slope, const float* alpha,
                                                         __nv_bfloat16* __restrict__ out, int Cpad, int rows_total,
                                                         const int* off, const int* len, int vec_ok) {
  const int b = blockIdx.y;
  const int L = len[b], o = off[b];
  // item b zeroes its leading gap and kGapRows rows after its end (never reaching the next item,
  // whose own leading gap covers the alignment slack); the last item zeroes up to rows_total
  const int r_begin = o - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : o + L + kGapRows;
  const int rb = r_begin + blockIdx.x * kApplyRowsB;
  if (rb >= r_end) return;
  const int re = min(r_end, rb + kApplyRowsB);
  const int cq = Cpad >> 2;                 // column quads per row
  // thread -> (column quad, row lane); a thread keeps its quad's coefficients in registers
  const int lanes = cq >= 256 ? 1 : 256 / cq;
  for (int q0 = 0; q0 < cq; q0 += 256) {
    const int qi = q0 + (cq >= 256 ? threadIdx.x : threadIdx.x % cq);
    const int rl = cq >= 256 ? 0 : threadIdx.x / cq;
    if (qi >= cq || rl >= lanes) continue;
    const int c = qi << 2;
    float sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f}, al[4] = {1.f, 1.f, 1.f, 1.f};
#pragma unroll
    for (int e = 0; e < 4; e++) {
      if (c + e < C) {
        if (scale) { sc[e] = scale[(size_t)b * C + c + e]; sh[e] = shift[(size_t)b * C + c + e]; }
        if (alpha) al[e] = alpha[c + e];
      }
    }
    for (int r = rb + rl; r < re; r += lanes) {
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (r >= o && r < o + L && c < C) {
        const float* xp = x + (size_t)r * ldx + c;
        if (vec_ok && c + 3 < C) {
          const float4 t = *reinterpret_cast<const float4*>(xp);
          v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
        } else {
#pragma unroll
          for (int e = 0; e < 4; e++) if (c + e < C) v[e] = xp[e];
        }
#pragma unroll
        for (int e = 0; e < 4; e++)
          v[e] = (c + e < C) ? apply_act(fmaf(v[e], sc[e], sh[e]), act, slope, al[e]) : 0.f;
      }
      __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
      uint2 pk;
      pk.x = *reinterpret_cast<uint32_t*>(&lo);
      pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(out + (size_t)r * Cpad + c) = pk;
    }
  }
}

// The same producer for the common case (128-bit loads possible, activation known at compile time): a thread owns one
// column quad and walks its rows FOUR at a time -- the four 128-bit loads are issued before any of the math, so a
// thread keeps 64 bytes in flight instead of 16 (the generic kernel above branches on the activation per element and
// ran the 77 k x 1024 decoder tensors at ~2.4 TB/s).  Same arithmetic per element -> the same bits.
template <int ACT>
__global__ void __launch_bounds__(256) apply_bf16_fast_kernel(const float* __restrict__ x, int ldx, int C,
                                                              const float* __restrict__ scale, const float* __restrict__ shift,
                                                              float slope, const float* __restrict__ alpha,
                                                              __nv_bfloat16* __restrict__ out, int Cpad, int rows_total,
                                                              const int* off, const int* len) {
  const int b = blockIdx.y;
  const int L = len[b], o = off[b];
  const int r_begin = o - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : o + L + kGapRows;
  const int rb = r_begin + blockIdx.x * kApplyRowsB;
  if (rb >= r_end) return;
  const int re = min(r_end, rb + kApplyRowsB);
  const int cq = Cpad >> 2;
  const int lanes = cq >= 256 ? 1 : 256 / cq;
  for (int q0 = 0; q0 < cq; q0 += 256) {
    const int qi = q0 + (cq >= 256 ? threadIdx.x : threadIdx.x % cq);
    const int rl = cq >= 256 ? 0 : threadIdx.x / cq;
    if (qi >= cq || rl >= lanes) continue;
    const int c = qi << 2;
    const bool full = c + 3 < C;              // quads straddling C (e.g. C = 1090) take scalar loads, pad quads store zeros
    float sc[4] = {1.f, 1.f, 1.f, 1.f}, sh[4] = {0.f, 0.f, 0.f, 0.f}, al[4] = {1.f, 1.f, 1.f, 1.f};
#pragma unroll
    for (int e = 0; e < 4; e++) {
      if (c + e < C) {
        if (scale) { sc[e] = scale[(size_t)b * C + c + e]; sh[e] = shift[(size_t)b * C + c + e]; }
        if (alpha) al[e] = alpha[c + e];
      }
    }
    for (int r = rb + rl; r < re; r += 4 * lanes) {
      float4 t[4];
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int rr = r + u * lanes;
        t[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rr < re && rr >= o && rr < o + L && c < C) {
          const float* xp = x + (size_t)rr * ldx + c;
          if (full) t[u] = *reinterpret_cast<const float4*>(xp);
          else { t[u].x = xp[0]; if (c + 1 < C) t[u].y = xp[1]; if (c + 2 < C) t[u].z = xp[2]; }
        }
      }
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const int rr = r + u * lanes;
        if (rr >= re) break;
        float v[4] = {t[u].x, t[u].y, t[u].z, t[u].w};
        const bool in = rr >= o && rr < o + L;
#pragma unroll
        for (int e = 0; e < 4; e++)
          v[e] = (in && c + e < C) ? apply_act(fmaf(v[e], sc[e], sh[e]), ACT, slope, al[e]) : 0.f;
        __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t*>(&lo);
        pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(out + (size_t)rr * Cpad + c) = pk;
      }
    }
  }
}

void launch_apply_bf16(const float* x, int ldx, int C, const float* scale, const float* shift, int act,
                       float slope, const float* alpha, void* out, int Cpad, int rows_total,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  const int rows = max_len + 2 * kGapRows + 8;
  dim3 g((rows + kApplyRowsB - 1) / kApplyRowsB, B);
  const int vec_ok = (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) ? 1 : 0;
  // one choice per shape (never per batch); both kernels compute the same bits
  if (vec_ok && C >= 64 && act == ACT_NONE)
    apply_bf16_fast_kernel<ACT_NONE><<<g, 256, 0, st>>>(x, ldx, C, scale, shift, slope, alpha, (__nv_bfloat16*)out, Cpad, rows_total, off, len);
  else if (vec_ok && C >= 64 && act == ACT_LRELU)
    apply_bf16_fast_kernel<ACT_LRELU><<<g, 256, 0, st>>>(x, ldx, C, scale, shift, slope, alpha, (__nv_bfloat16*)out, Cpad, rows_total, off, len);
  else if (vec_ok && C >= 64 && act == ACT_SNAKE)
    apply_bf16_fast_kernel<ACT_SNAKE><<<g, 256, 0, st>>>(x, ldx, C, scale, shift, slope, alpha, (__nv_bfloat16*)out, Cpad, rows_total, off, len);
  else
    apply_bf16_kernel<<<g, 256, 0, st>>>(x, ldx, C, scale, shift, act, slope, alpha, (__nv_bfloat16*)out, Cpad,
                                         rows_total, off, len, vec_ok);
  post_launch("apply_bf16", st);
}

// im2col operand producer for strided convs with few channels (noise_convs[0]: 22 ch, k12, s6, p3):
// out[m, tap*C + c] = in[m*stride + tap - pad, c] (0 outside the item), bf16 [rows_out_total, Cpad].
__global__ void __launch_bounds__(256) im2col_bf16_kernel(const float* __restrict__ in, int ldi, int C, int ks,
                                                          int stride, int pad, __nv_bfloat16* out, int Cpad,
                                                          int rows_total, const int* in_off, const int* in_len,
                                                          const int* out_off, const int* out_len) {
  const int b = blockIdx.y;
  const int Lo = out_len[b], oo = out_off[b], Li = in_len[b], io = in_off[b];
  const int r_begin = oo - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : oo + Lo + kGapRows;
  const int rb = r_begin + blockIdx.x * 8;
  if (rb >= r_end) return;
  const int re = min(r_end, rb + 8);
  const int total = (re - rb) * Cpad;
  for (int i = threadIdx.x; i < total; i += 256) {
    const int r = rb + i / Cpad, k = i % Cpad;
    float v = 0.f;
    const int m = r - oo;
    if (m >= 0 && m < Lo && k < ks * C) {
      const int tap = k / C, c = k - tap * C;
      const int ir = m * stride + tap - pad;
      if (ir >= 0 && ir < Li) v = in[(size_t)(io + ir) * ldi + c];
    }
    out[(size_t)r * Cpad + k] = __float2bfloat16_rn(v);
  }
}
// The same gather for noise_convs[0] (C = 22 of ldi = 24, k = 12, stride 6, pad 3) with compile-time geometry: the KS input
// rows of an output row are ONE contiguous window of KS * 24 floats (output column tap * 22 + c <- window index tap * 24 + c),
// and consecutive output rows' windows overlap by half.  A CTA stages the input rows of its RPB output rows in shared memory
// with 128-bit loads and every thread writes 8 consecutive bf16 (one 16-byte store).  The generic kernel above did one
// 4-byte load, two integer divisions and one 2-byte store per element (1.2 TB/s).
template <int C, int LDI, int KS, int STRIDE, int PAD, int RPB>
__global__ void __launch_bounds__(256) im2col_bf16_fast_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out,
                                                               int Cpad, int rows_total, const int* in_off, const int* in_len,
                                                               const int* out_off, const int* out_len) {
  constexpr int WROWS = (RPB - 1) * STRIDE + KS;        // input rows a CTA touches
  __shared__ __align__(16) float win[WROWS * LDI];
  const int b = blockIdx.y;
  const int Lo = out_len[b], oo = out_off[b], Li = in_len[b], io = in_off[b];
  const int r_begin = oo - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : oo + Lo + kGapRows;
  const int rb = r_begin + blockIdx.x * RPB;
  if (rb >= r_end) return;
  const int re = min(r_end, rb + RPB);
  const int m0 = rb - oo;                               // first output row of the CTA relative to the item (may be < 0)
  const int ir0 = m0 * STRIDE - PAD;                    // first input row of the window
  for (int i = threadIdx.x; i < WROWS * LDI / 4; i += 256) {
    const int ir = ir0 + (i * 4) / LDI;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ir >= 0 && ir < Li) v = *reinterpret_cast<const float4*>(in + (size_t)(io + ir) * LDI + (i * 4) % LDI);
    reinterpret_cast<float4*>(win)[i] = v;
  }
  __syncthreads();
  const int chunks = Cpad >> 3;                         // 16-byte output chunks per row
  for (int i = threadIdx.x; i < (re - rb) * chunks; i += 256) {
    const int rl = i / chunks, k0 = (i - rl * chunks) << 3;
    const int m = m0 + rl;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if (m >= 0 && m < Lo) {
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; e++) {
        const int k = k0 + e;
        const int tap = k / C, c = k - tap * C;
        v[e] = k < KS * C ? win[(rl * STRIDE + tap) * LDI + c] : 0.f;
      }
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const __nv_bfloat162 p = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
        w[e] = *reinterpret_cast<const uint32_t*>(&p);
      }
    }
    *reinterpret_cast<uint4*>(out + (size_t)(rb + rl) * Cpad + k0) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

void launch_im2col_bf16(const float* in, int ldi, int C, int ks, int stride, int pad, void* out, int Cpad,
                        int rows_total, const int* in_off, const int* in_len, const int* out_off,
                        const int* out_len, int B, int max_out_len, cudaStream_t st, int force_generic) {
  if (g_dry_run) return;
  const int rows = max_out_len + 2 * kGapRows + 8;
  if (!force_generic && C == 22 && ldi == 24 && ks == 12 && stride == 6 && pad == 3 && Cpad % 8 == 0 &&
      ((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0) {
    constexpr int RPB = 32;
    dim3 g((rows + RPB - 1) / RPB, B);
    im2col_bf16_fast_kernel<22, 24, 12, 6, 3, RPB><<<g, 256, 0, st>>>(in, (__nv_bfloat16*)out, Cpad, rows_total, in_off, in_len,
                                                                      out_off, out_len);
  } else {
    dim3 g((rows + 7) / 8, B);
    im2col_bf16_kernel<<<g, 256, 0, st>>>(in, ldi, C, ks, stride, pad, (__nv_bfloat16*)out, Cpad, rows_total,
                                          in_off, in_len, out_off, out_len);
  }
  post_launch("im2col_bf16", st);
}

// Split-TF32 operand producer: hi = rna_tf32(v), lo = rna_tf32(v - hi), two fp32 planes
// [rows_total, Cpad]; same prologue fusion and halo zeroing as apply_bf16.
__device__ __forceinline__ float to_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__global__ void __launch_bounds__(256) apply_tf32_kernel(const float* __restrict__ x, int ldx, int C,
                                                         const float* scale, const float* shift,
                                                         int act, float slope, float* out_hi, float* out_lo,
                                                         int Cpad, int rows_total, const int* off,
                                                         const int* len, int vec_ok) {
  const int b = blockIdx.y;
  const int L = len[b], o = off[b];
  const int r_begin = o - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : o + L + kGapRows;
  const int rb = r_begin + blockIdx.x * kApplyRows;
  if (rb >= r_end) return;
  const int re = min(r_end, rb + kApplyRows);
  const float* sc = scale ? scale + (size_t)b * C : nullptr;
  const float* sh = shift ? shift + (size_t)b * C : nullptr;
  // one column quad per thread: float4 load, two float4 stores (the kernel is a pure HBM stream:
  // 4 B read + 8 B written per element)
  const int cq = Cpad >> 2;
  const int total = (re - rb) * cq;
  for (int i = threadIdx.x; i < total; i += 256) {
    const int r = rb + i / cq;
    const int c = (i % cq) << 2;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r >= o && r < o + L && c < C) {
      const float* xp = x + (size_t)r * ldx + c;
      if (vec_ok && c + 3 < C) {
        const float4 t = *reinterpret_cast<const float4*>(xp);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; e++) if (c + e < C) v[e] = xp[e];
      }
#pragma unroll
      for (int e = 0; e < 4; e++) {
        if (c + e < C) {
          if (sc) v[e] = v[e] * sc[c + e] + sh[c + e];            // same arithmetic as the fp32 SIMT prologue
          if (act == ACT_LRELU) v[e] = v[e] > 0.f ? v[e] : v[e] * slope;
        } else v[e] = 0.f;
      }
    }
    float hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; e++) { hi[e] = to_tf32(v[e]); lo[e] = to_tf32(v[e] - hi[e]); }
    *reinterpret_cast<float4*>(out_hi + (size_t)r * Cpad + c) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4*>(out_lo + (size_t)r * Cpad + c) = make_float4(lo[0], lo[1], lo[2], lo[3]);
  }
}
void launch_apply_tf32(const float* x, int ldx, int C, const float* scale, const float* shift, int act,
                       float slope, float* out_hi, float* out_lo, int Cpad, int rows_total,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  const int rows = max_len + 2 * kGapRows + 8;
  dim3 g((rows + kApplyRows - 1) / kApplyRows, B);
  const int vec_ok = (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) ? 1 : 0;
  apply_tf32_kernel<<<g, 256, 0, st>>>(x, ldx, C, scale, shift, act, slope, out_hi, out_lo, Cpad, rows_total, off, len, vec_ok);
  post_launch("apply_tf32", st);
}

// Split-FP16 operand producer: the same prologue arithmetic, then v * 16 as two fp16 planes hi = rn(v), lo = rn(v - hi).
// fp16 and tf32 carry the same 11-bit significand, so hi + lo holds 22 bits exactly like the tf32 pair; the factor 16
// (undone, exactly, in the GEMM epilogue) keeps lo out of the fp16 subnormal range for |v| >= 2^-7, below which the
// absolute error is <= 2^-29.  Values beyond +-4094 would saturate (Kokoro's activations are O(1) .. O(10^2)).
__global__ void __launch_bounds__(256) apply_f16x2_kernel(const float* __restrict__ x, int ldx, int C,
                                                          const float* scale, const float* shift,
                                                          int act, float slope, __half* out_hi, __half* out_lo,
                                                          int Cpad, int rows_total, const int* off,
                                                          const int* len, int vec_ok) {
  const int b = blockIdx.y;
  const int L = len[b], o = off[b];
  const int r_begin = o - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : o + L + kGapRows;
  const int rb = r_begin + blockIdx.x * kApplyRows;
  if (rb >= r_end) return;
  const int re = min(r_end, rb + kApplyRows);
  const float* sc = scale ? scale + (size_t)b * C : nullptr;
  const float* sh = shift ? shift + (size_t)b * C : nullptr;
  const int cq = Cpad >> 2;
  const int total = (re - rb) * cq;
  for (int i = threadIdx.x; i < total; i += 256) {
    const int r = rb + i / cq;
    const int c = (i % cq) << 2;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r >= o && r < o + L && c < C) {
      const float* xp = x + (size_t)r * ldx + c;
      if (vec_ok && c + 3 < C) {
        const float4 t = *reinterpret_cast<const float4*>(xp);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
#pragma unroll
        for (int e = 0; e < 4; e++) if (c + e < C) v[e] = xp[e];
      }
#pragma unroll
      for (int e = 0; e < 4; e++) {
        if (c + e < C) {
          if (sc) v[e] = v[e] * sc[c + e] + sh[c + e];            // same arithmetic as the fp32 SIMT prologue
          if (act == ACT_LRELU) v[e] = v[e] > 0.f ? v[e] : v[e] * slope;
        } else v[e] = 0.f;
      }
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; e++) split_f16_operand(v[e], hi[e], lo[e]);
    *reinterpret_cast<uint2*>(out_hi + (size_t)r * Cpad + c) = make_uint2(hi[0] | (hi[1] << 16), hi[2] | (hi[3] << 16));
    *reinterpret_cast<uint2*>(out_lo + (size_t)r * Cpad + c) = make_uint2(lo[0] | (lo[1] << 16), lo[2] | (lo[3] << 16));
  }
}
float split_f16_host(const float* w, size_t n, unsigned short* hi, unsigned short* lo) {
  float mx = 0.f;
  for (size_t i = 0; i < n; i++) mx = fmaxf(mx, fabsf(w[i]));
  int s = 0;
  if (mx > 0.f && isfinite(mx)) {
    int e;
    frexpf(mx, &e);                    // mx = m * 2^e, m in [0.5, 1)
    s = 14 - e;                        // mx * 2^s in [2^13, 2^14)
  }
  if (s > 60) s = 60;
  if (s < -60) s = -60;
  const float up = ldexpf(1.f, s);
  for (size_t i = 0; i < n; i++) {
    uint32_t h, l;
    split_f16(w[i] * up, h, l);        // the scaling is exact (power of two)
    hi[i] = (unsigned short)h;
    lo[i] = (unsigned short)l;
  }
  return ldexpf(1.f, -s);
}

void launch_apply_f16x2(const float* x, int ldx, int C, const float* scale, const float* shift, int act,
                        float slope, void* out_hi, void* out_lo, int Cpad, int rows_total,
                        const int* off, const int* len, int B, int max_len, cudaStream_t st) {
  if (g_dry_run) return;
  const int rows = max_len + 2 * kGapRows + 8;
  dim3 g((rows + kApplyRows - 1) / kApplyRows, B);
  const int vec_ok = (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) ? 1 : 0;
  apply_f16x2_kernel<<<g, 256, 0, st>>>(x, ldx, C, scale, shift, act, slope, static_cast<__half*>(out_hi),
                                        static_cast<__half*>(out_lo), Cpad, rows_total, off, len, vec_ok);
  post_launch("apply_f16x2", st);
}

// Depthwise ConvTranspose1d(k3,s2,p1,op1) on lrelu(x*scale+shift) -> bf16 operand [2T rows, Cpad]
__global__ void __launch_bounds__(256) pool_up_bf16_kernel(const float* __restrict__ in, int ldi,
                                                           const float* scale, const float* shift,
                                                           float slope, const float* w, const float* bias,
                                                           int C, __nv_bfloat16* out, int Cpad,
                                                           int rows_total, const int* in_off,
                                                           const int* in_len, const int* out_off) {
  const int b = blockIdx.y;
  const int T = in_len[b], oo = out_off[b];
  const int r_begin = oo - kGapRows;
  const int r_end = (b == (int)gridDim.y - 1) ? rows_total : oo + 2 * T + kGapRows;
  const float* sc = scale + (size_t)b * C;
  const float* sh = shift + (size_t)b * C;
  const long long total = (long long)(r_end - r_begin) * Cpad;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int r = r_begin + (int)(i / Cpad);
    const int c = (int)(i % Cpad);
    float v = 0.f;
    const int j = r - oo;
    if (j >= 0 && j < 2 * T && c < C) {
      const int t = j >> 1;
      const float* x0 = in + (size_t)(in_off[b] + t) * ldi;
      float a0 = x0[c] * sc[c] + sh[c];
      a0 = a0 > 0.f ? a0 : a0 * slope;
      if ((j & 1) == 0) {
        v = w[c * 3 + 1] * a0 + bias[c];
      } else {
        float a1 = 0.f;
        if (t + 1 < T) { a1 = x0[ldi + c] * sc[c] + sh[c]; a1 = a1 > 0.f ? a1 : a1 * slope; }
        v = w[c * 3 + 2] * a0 + w[c * 3 + 0] * a1 + bias[c];
      }
    }
    out[(size_t)r * Cpad + c] = __float2bfloat16_rn(v);
  }
}

void launch_pool_up_bf16(const float* in, int ldi, const float* scale, const float* shift, float slope,
                         const float* w, const float* bias, int C, void* out, int Cpad, int rows_total,
                         const int* in_off, const int* in_len, const int* out_off, int B, int max_len,
                         cudaStream_t st) {
  if (g_dry_run) return;
  long long work = (long long)(2 * max_len + 2 * kGapRows + 8) * Cpad;
  long long blocks = (work + 256 * 4 - 1) / (256 * 4);
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 8) blocks = 148 * 8;
  dim3 g((unsigned)blocks, B);
  pool_up_bf16_kernel<<<g, 256, 0, st>>>(in, ldi, scale, shift, slope, w, bias, C, (__nv_bfloat16*)out, Cpad,
                                         rows_total, in_off, in_len, out_off);
  post_launch("pool_up_bf16", st);
}

}  // namespace kkx
