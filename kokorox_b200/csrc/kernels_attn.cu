// kernels_attn.cu -- ALBERT self-attention (12 heads x 64, N <= 512, key-padding mask) on tcgen05 / TMEM, fed by TMA.
//
// north_star: "the ALBERT/PL-BERT encoder ... use tcgen05/TMEM tiles fed by TMA".  Round 1 ran attention on legacy
// mma.sync fragments (kernels_dense.cu attention_tc_kernel, kept as the fallback); this is the Blackwell-native form.
// The path feeds the duration predictor, whose integer durations must match the fp32 oracle bit for bit, so every
// product is split-precision (hi*hi + hi*lo + lo*hi with 11-bit significands, fp32 accumulation) like the mma.sync
// kernel.  The planes are FP16 ("3xFP16", the same 22 significand bits as the tf32 pair of the first version): role
// counters showed the MMA thread issuing for 63 % of a CTA's life at ~66 cycles per 128 x 64 x 8 tf32 MMA -- twice the
// tensor-pipe floor, a per-instruction cost -- and kind::f16 covers K = 16 per instruction, so the same work is half the
// instructions (and half the operand bytes).  Exact power-of-two scaling keeps the fp16 low parts normal:
//   Q planes hold 2 q (= 16 * q/8), K planes 16 k  ->  S' = 256 S;   P planes hold 4096 p, V planes 16 v  ->  O' = 65536 O.
//
// Two kernels per layer:
//   attn_prep_kernel   qkv [rows, 2304] fp32 -> fp16 hi/lo planes  Q [rows, 768], K [rows, 768] and the TRANSPOSED
//                      V^T [(item, head, d), key] (pitch 512), so that both MMAs take K-major operands straight from
//                      128B-swizzled TMA boxes (keys beyond the item's length are zero-filled up to a multiple of 64).
//                      (Big batches skip it: the QKV GEMM's final warps write the planes, kernels_tc.cu.)
//   attn_umma_kernel   persistent CTAs over the (item, head, 128 query rows) work items, 10 warps:
//       warp 0     TMA producer: the Q planes per work item (prefetched), a 4-stage ring of K and V^T tiles of 64 keys
//       warp 1     MMA issuer:  S_j = Q K_j^T (M 128, N 64 keys, K 64: 12 UMMAs) into one of two TMEM S buffers,
//                               O_j = P_j V_j  (A = P from TENSOR MEMORY, B = V^T tile: 12 UMMAs) into a TMEM O tile
//       warps 2-9  softmax, two warps per block of 32 query rows (each takes 32 of a tile's 64 keys and 32 of the 64 output
//                  dims; row maxima exchanged through smem): thread = query row = TMEM lane: tcgen05.ld
//                  of S_j, mask, online max, exp, split P into fp16 hi/lo and tcgen05.st them back to TMEM as the A
//                  operand of the second MMA; then the O tile is drained and folded into the fp32 running output with
//                  the flash rescaling (each 64-key chain is added in fp32 RN -- the tensor core truncates per
//                  accumulate, the same chain splitting the split-precision GEMMs use).
//   S, P and O are all double-buffered in TMEM: S_{j+1} is issued before the softmax of tile j starts and O_j = P_j V_j
//   runs while the softmax warps are already on tile j+1 (they fold O_j in after writing P_{j+1}; the order of the
//   floating-point operations is unchanged), so the tensor pipe works under the exponentials.
// TMEM columns: S0 0..63, S1 64..127, P buffer pb at 128 + 64 pb (hi 32 columns = 64 keys, then lo), O0 256..319, O1 320..383.
#include "kernels.h"
#include <cstdio>
#include <cuda.h>
#include "tc_ptx.cuh"

namespace kkx {

// Optional per-role phase timing (-DKKX_TC_TIMING, diagnostics only): the MMA thread and one softmax thread of CTA
// (0, 0, 0) of every launch attribute the cycles between consecutive ticks to a slot of g_attn_tim.
#ifdef KKX_TC_TIMING
__device__ unsigned long long g_attn_tim[24];
#define ATT_DECL(cond) long long att_acc[8] = {0}; long long att_last = clock64(); const bool att_on = (cond) && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0
#define ATT(slot) do { if (att_on) { const long long now_ = clock64(); att_acc[slot] += now_ - att_last; att_last = now_; } } while (0)
#define ATT_FLUSH(base) do { if (att_on) for (int i_ = 0; i_ < 8; i_++) atomicAdd(g_attn_tim + (base) + i_, (unsigned long long)att_acc[i_]); } while (0)
#else
#define ATT_DECL(cond)
#define ATT(slot)
#define ATT_FLUSH(base)
#endif

namespace {
__device__ __forceinline__ uint32_t to_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return r;
}
// D[tmem] (+)= A[tmem] * B[smem desc], kind::f16 (fp16 operands, fp32 accumulate)
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
}
constexpr float kQScale = 2.0f;          // 16 * (1/8): the 1/sqrt(64) of the scores folded in, exact
constexpr float kKVScale = 16.0f;
constexpr float kPScale = 4096.0f;
constexpr float kSInv = 1.0f / 256.0f;    // S = q.k / 8 = S' / (kQScale * kKVScale * 8)
constexpr float kOInv = 1.0f / 65536.0f;  // O = O' / (kPScale * kKVScale)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr int kVtPitch = 512;          // keys per V^T row (ALBERT max_position_embeddings)

// ------------------------------------------------------------------------------------------ operand planes
__global__ void __launch_bounds__(256) attn_prep_kernel(const float* __restrict__ qkv, __half* __restrict__ qh,
                                                        __half* __restrict__ ql, __half* __restrict__ kh,
                                                        __half* __restrict__ kl, __half* __restrict__ vth,
                                                        __half* __restrict__ vtl, const int* __restrict__ off,
                                                        const int* __restrict__ len) {
  __shared__ unsigned short s_h[64][34], s_l[64][34];
  const int b = blockIdx.z, h = blockIdx.y, t0 = blockIdx.x * 32;
  const int N = len[b];
  const int NR = (N + 63) & ~63;                       // V^T is consumed in tiles of 64 keys: zero-fill up to there
  if (t0 >= NR) return;
  const int tid = threadIdx.x, r = tid >> 3, c8 = (tid & 7) << 3;
  const int token = t0 + r;
  const bool valid = token < N;
  const size_t row = (size_t)off[b] + token;
  float q[8], k[8], v[8];
#pragma unroll
  for (int e = 0; e < 8; e++) { q[e] = 0.f; k[e] = 0.f; v[e] = 0.f; }
  if (valid) {
    const float* src = qkv + row * 2304 + h * 64 + c8;
    const float4 a0 = *reinterpret_cast<const float4*>(src), a1 = *reinterpret_cast<const float4*>(src + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(src + 768), b1 = *reinterpret_cast<const float4*>(src + 772);
    const float4 c0 = *reinterpret_cast<const float4*>(src + 1536), c1 = *reinterpret_cast<const float4*>(src + 1540);
    q[0] = a0.x; q[1] = a0.y; q[2] = a0.z; q[3] = a0.w; q[4] = a1.x; q[5] = a1.y; q[6] = a1.z; q[7] = a1.w;
    k[0] = b0.x; k[1] = b0.y; k[2] = b0.z; k[3] = b0.w; k[4] = b1.x; k[5] = b1.y; k[6] = b1.z; k[7] = b1.w;
    v[0] = c0.x; v[1] = c0.y; v[2] = c0.z; v[3] = c0.w; v[4] = c1.x; v[5] = c1.y; v[6] = c1.z; v[7] = c1.w;
    uint32_t w[4][8];   // qh ql kh kl
#pragma unroll
    for (int e = 0; e < 8; e++) {
      split_f16(q[e] * kQScale, w[0][e], w[1][e]);
      split_f16(k[e] * kKVScale, w[2][e], w[3][e]);
    }
    __half* dst[4] = {qh, ql, kh, kl};
#pragma unroll
    for (int p = 0; p < 4; p++)
      *reinterpret_cast<uint4*>(dst[p] + row * 768 + h * 64 + c8) =
          make_uint4(w[p][0] | (w[p][1] << 16), w[p][2] | (w[p][3] << 16), w[p][4] | (w[p][5] << 16), w[p][6] | (w[p][7] << 16));
  }
#pragma unroll
  for (int e = 0; e < 8; e++) {
    uint32_t hi, lo;
    split_f16(v[e] * kKVScale, hi, lo);
    s_h[c8 + e][r] = (unsigned short)hi;
    s_l[c8 + e][r] = (unsigned short)lo;
  }
  __syncthreads();
  // V^T rows: (item, head, d), 32 keys of this block contiguous (64 bytes): 4 threads x 8 keys per d
  const int d = tid >> 2, seg = (tid & 3) << 3;
  const size_t vrow = ((size_t)(b * 12 + h) * 64 + d) * kVtPitch + t0 + seg;
  *reinterpret_cast<uint4*>(vth + vrow) =
      make_uint4(s_h[d][seg] | ((uint32_t)s_h[d][seg + 1] << 16), s_h[d][seg + 2] | ((uint32_t)s_h[d][seg + 3] << 16),
                 s_h[d][seg + 4] | ((uint32_t)s_h[d][seg + 5] << 16), s_h[d][seg + 6] | ((uint32_t)s_h[d][seg + 7] << 16));
  *reinterpret_cast<uint4*>(vtl + vrow) =
      make_uint4(s_l[d][seg] | ((uint32_t)s_l[d][seg + 1] << 16), s_l[d][seg + 2] | ((uint32_t)s_l[d][seg + 3] << 16),
                 s_l[d][seg + 4] | ((uint32_t)s_l[d][seg + 5] << 16), s_l[d][seg + 6] | ((uint32_t)s_l[d][seg + 7] << 16));
}

// ------------------------------------------------------------------------------------------ the attention kernel
constexpr uint32_t kQPlane = 128 * 128;                // one Q plane: [128 rows x 64 fp16] = 16 KB
constexpr uint32_t kTilePlane = 64 * 128;              // one K / V^T plane of a 64-key tile: [64 x 64 fp16] = 8 KB
constexpr uint32_t kStage = 4 * kTilePlane;            // Kh | Kl | VTh | VTl = 32 KB
constexpr int kAttnStages = 4;
constexpr int kAttnThreads = 320;                      // TMA warp, MMA warp, 8 softmax warps
constexpr int kAttnSmem = 4 * kQPlane + kAttnStages * kStage + 32 * 8 + 16 + 3072 + 1024;   // 2 Q buffers, K/V ring, barriers, exchange buffers
constexpr uint32_t kColS0 = 0, kColP = 128, kColO = 256;   // P buffer pb: hi at kColP + 64 pb (32 columns = 64 keys), lo 32 columns further

// Persistent: a CTA walks the work items w = blockIdx.x, blockIdx.x + gridDim.x, ... of the (item, head, query block)
// space, query block fastest (the CTAs that run together share K / V^T tiles in L2).  With one CTA per work item the
// start-up (TMEM allocation, Q load: ~4 k cycles) and the tear-down (output rows, ~5 k) were exposed 21 times per SM and
// launch -- 30 % of a CTA's life; here the TMA warp prefetches the next item's Q into a second buffer, the MMA thread
// issues the next item's S_0 under the last softmax of the current one, and all barrier phases follow running counters
// (`g` = key tiles processed so far by this CTA, `it` = work items so far).
struct AttnItem {
  int b, h, q0, N, nt;
};
__device__ __forceinline__ bool attn_item(int w, int QB, const int* __restrict__ len, AttnItem& a) {
  const int qb = w % QB, bh = w / QB;
  a.h = bh % 12; a.b = bh / 12;
  a.q0 = qb * 128;
  a.N = len[a.b];
  a.nt = (a.N + 63) >> 6;
  return a.q0 < a.N;
}

__global__ void __launch_bounds__(kAttnThreads, 1) attn_umma_kernel(const __grid_constant__ CUtensorMap tmQh,
                                                           const __grid_constant__ CUtensorMap tmQl,
                                                           const __grid_constant__ CUtensorMap tmKh,
                                                           const __grid_constant__ CUtensorMap tmKl,
                                                           const __grid_constant__ CUtensorMap tmVh,
                                                           const __grid_constant__ CUtensorMap tmVl,
                                                           const int* __restrict__ off, const int* __restrict__ len,
                                                           float* __restrict__ ctx, int QB, int W) {
  constexpr int NST = kAttnStages;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  auto q_h = [&](int qi) { return base + (uint32_t)qi * 2u * kQPlane; };      // Q buffer qi: hi plane, lo plane
  auto q_l = [&](int qi) { return base + (uint32_t)qi * 2u * kQPlane + kQPlane; };
  const uint32_t st0 = base + 4 * kQPlane;
  const uint32_t bar_base = st0 + NST * kStage;
  // K and V^T of a stage have their own full / empty barriers: K_j is free again as soon as S_j has been computed,
  // V^T_j only after P_j V_j; the stage ring (4 deep) is independent of the double-buffered S / P / O in TMEM
  auto fullk_bar = [&](int s) { return bar_base + s * 8; };
  auto emptyk_bar = [&](int s) { return bar_base + (NST + s) * 8; };
  auto fullv_bar = [&](int s) { return bar_base + (2 * NST + s) * 8; };
  auto emptyv_bar = [&](int s) { return bar_base + (3 * NST + s) * 8; };
  auto sfull_bar = [&](int i) { return bar_base + (4 * NST + i) * 8; };
  auto sfree_bar = [&](int i) { return bar_base + (4 * NST + 2 + i) * 8; };
  auto pfull_bar = [&](int i) { return bar_base + (4 * NST + 4 + i) * 8; };
  auto ofull_bar = [&](int i) { return bar_base + (4 * NST + 6 + i) * 8; };
  auto ofree_bar = [&](int i) { return bar_base + (4 * NST + 8 + i) * 8; };
  auto qfull_bar = [&](int i) { return bar_base + (4 * NST + 10 + i) * 8; };
  auto qfree_bar = [&](int i) { return bar_base + (4 * NST + 12 + i) * 8; };
  const uint32_t tmem_slot = bar_base + 32 * 8;
  const uint32_t xch_base = tmem_slot + 16;             // row maxima [2][2][128] + row sums [2][128] (floats)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmQh);
    prefetch_tmap(&tmKh);
    prefetch_tmap(&tmVh);
    for (int s = 0; s < NST; s++) {
      mbar_init(fullk_bar(s), 1); mbar_init(emptyk_bar(s), 1); mbar_init(fullv_bar(s), 1); mbar_init(emptyv_bar(s), 1);
    }
    for (int s = 0; s < 2; s++) {
      mbar_init(sfull_bar(s), 1); mbar_init(sfree_bar(s), 8);
      mbar_init(pfull_bar(s), 8); mbar_init(ofull_bar(s), 1); mbar_init(ofree_bar(s), 8);
      mbar_init(qfull_bar(s), 1); mbar_init(qfree_bar(s), 1);
    }
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, 512u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  if (warp == 0) {
    if (lane == 0) {
      int g = 0, it = 0;                                // key tiles / work items issued so far
      for (int w = blockIdx.x; w < W; w += gridDim.x) {
        AttnItem a;
        if (!attn_item(w, QB, len, a)) continue;
        const int qi = it & 1;
        const int qrow = off[a.b] + a.q0, krow0 = off[a.b], vrow = (a.b * 12 + a.h) * 64;
        mbar_wait(qfree_bar(qi), (((uint32_t)(it >> 1)) & 1u) ^ 1u);     // the S MMAs of item it - 2 are done with this Q buffer
        mbar_expect_tx(qfull_bar(qi), 2 * kQPlane);
        tma_load_2d(q_h(qi), &tmQh, a.h * 64, qrow, qfull_bar(qi));
        tma_load_2d(q_l(qi), &tmQl, a.h * 64, qrow, qfull_bar(qi));
        auto load_k = [&](int j) {
          const int s = (g + j) % NST;
          mbar_wait(emptyk_bar(s), (((uint32_t)((g + j) / NST)) & 1u) ^ 1u);
          const uint32_t sa = st0 + s * kStage;
          mbar_expect_tx(fullk_bar(s), 2 * kTilePlane);
          tma_load_2d(sa, &tmKh, a.h * 64, krow0 + j * 64, fullk_bar(s));
          tma_load_2d(sa + kTilePlane, &tmKl, a.h * 64, krow0 + j * 64, fullk_bar(s));
        };
        auto load_v = [&](int j) {
          const int s = (g + j) % NST;
          mbar_wait(emptyv_bar(s), (((uint32_t)((g + j) / NST)) & 1u) ^ 1u);
          const uint32_t sa = st0 + s * kStage;
          mbar_expect_tx(fullv_bar(s), 2 * kTilePlane);
          tma_load_2d(sa + 2 * kTilePlane, &tmVh, j * 64, vrow, fullv_bar(s));
          tma_load_2d(sa + 3 * kTilePlane, &tmVl, j * 64, vrow, fullv_bar(s));
        };
        // issue order = the order in which the MMA warp needs (and frees) the buffers: K_0, K_1, V_0, K_2, V_1, ...
        load_k(0);
        for (int j = 0; j < a.nt; j++) {
          if (j + 1 < a.nt) load_k(j + 1);
          load_v(j);
        }
        g += a.nt; it++;
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(128, 64);
      ATT_DECL(true);
      // S'_j = Q' K'_j^T of key tile j of item `a` (global tile index gt, item counter it_), small terms first
      auto issue_s = [&](const AttnItem& a, int j, int gt, int it_) {
        const int s = gt & 1, st = gt % NST, qi = it_ & 1;
        if (j == 0) {
          mbar_wait(qfull_bar(qi), ((uint32_t)(it_ >> 1)) & 1u);
          tc_fence_after();
        }
        ATT(0);
        mbar_wait(fullk_bar(st), ((uint32_t)(gt / NST)) & 1u);
        tc_fence_after();
        ATT(1);
        if (gt >= 2) {                                 // the softmax warps have read the S tile that used this buffer
          mbar_wait(sfree_bar(s), ((uint32_t)((gt >> 1) - 1)) & 1u);
          tc_fence_after();
        }
        ATT(2);
        const uint32_t sa = st0 + st * kStage;
        const uint32_t t_s = tmem_base + kColS0 + 64u * (uint32_t)s;
        const uint64_t ah = umma_desc_sw128(q_h(qi)), al = umma_desc_sw128(q_l(qi));
        const uint64_t bh = umma_desc_sw128(sa), bl = umma_desc_sw128(sa + kTilePlane);
#pragma unroll
        for (int k = 0; k < 4; k++) {                  // 4 x (K = 16 fp16 = 32 B) = the 64 dims of a head
          const uint64_t o = (uint64_t)(2 * k);
          umma_bf16(t_s, al + o, bh + o, idesc, k ? 1u : 0u);      // (kind::f16; the descriptor selects fp16)
          umma_bf16(t_s, ah + o, bl + o, idesc, 1u);
          umma_bf16(t_s, ah + o, bh + o, idesc, 1u);
        }
        umma_commit(sfull_bar(s));
        umma_commit(emptyk_bar(st));                   // K_j is consumed
        if (j == a.nt - 1) umma_commit(qfree_bar(qi)); // the item's last S: its Q buffer is free
        ATT(3);
      };
      // first valid work item
      int w = blockIdx.x;
      AttnItem cur;
      bool have = false;
      for (; w < W; w += gridDim.x) if (attn_item(w, QB, len, cur)) { have = true; break; }
      int g = 0, it = 0;
      if (have) issue_s(cur, 0, 0, 0);
      while (have) {
        // look ahead: the next valid work item (its S_0 is issued under the last softmax of the current item)
        AttnItem nxt;
        bool have_n = false;
        int wn = w + gridDim.x;
        for (; wn < W; wn += gridDim.x) if (attn_item(wn, QB, len, nxt)) { have_n = true; break; }
        for (int j = 0; j < cur.nt; j++) {
          const int gt = g + j;
          if (j + 1 < cur.nt) issue_s(cur, j + 1, gt + 1, it);      // runs under the softmax of tile j
          else if (have_n) issue_s(nxt, 0, gt + 1, it + 1);
          const int s = gt & 1, st = gt % NST;           // P / O buffer and stage of this tile
          mbar_wait(fullv_bar(st), ((uint32_t)(gt / NST)) & 1u);   // V^T_j has landed
          ATT(4);
          mbar_wait(pfull_bar(s), ((uint32_t)(gt >> 1)) & 1u);     // P_j is in TMEM
          tc_fence_after();
          ATT(5);
          if (gt >= 2) {                                 // the O tile that used this buffer has been read out
            mbar_wait(ofree_bar(s), ((uint32_t)((gt >> 1) - 1)) & 1u);
            tc_fence_after();
          }
          ATT(6);
          const uint32_t sa = st0 + st * kStage;
          const uint32_t t_o = tmem_base + kColO + 64u * (uint32_t)s;
          const uint32_t t_ph = tmem_base + kColP + 64u * (uint32_t)s, t_pl = t_ph + 32u;
          const uint64_t vh = umma_desc_sw128(sa + 2 * kTilePlane), vl = umma_desc_sw128(sa + 3 * kTilePlane);
#pragma unroll
          for (int kk = 0; kk < 4; kk++) {               // 16 keys (8 TMEM columns of packed fp16 pairs) per UMMA
            const uint64_t o = (uint64_t)(2 * kk);
            umma_f16_ts(t_o, t_pl + 8u * kk, vh + o, idesc, kk ? 1u : 0u);
            umma_f16_ts(t_o, t_ph + 8u * kk, vl + o, idesc, 1u);
            umma_f16_ts(t_o, t_ph + 8u * kk, vh + o, idesc, 1u);
          }
          umma_commit(ofull_bar(s));
          umma_commit(emptyv_bar(st));                   // V^T_j is consumed
          ATT(7);
        }
        g += cur.nt; it++;
        cur = nxt; have = have_n; w = wn;
      }
      ATT_FLUSH(0);
    }
  } else {
    // ---- softmax: 8 warps.  Warp w owns TMEM lane quadrant q = w & 3 (32 query rows, one per thread) and key half
    // kh = (w - 2) >> 2: the 32 keys [32 kh, 32 kh + 32) of every tile and, for the output, the 32 dims [32 kh, 32 kh + 32).
    // With fp16 planes the MMA thread needs ~14 k cycles per work item and one warp per row block needed ~39 k for its
    // exp / split / fold chain (role counters); two warps per row block halve that chain.  The two warps of a row
    // exchange their partial row maxima through shared memory once per tile; their partial sums stay separate until
    // the end (both are scaled to the same running maximum).
    const int q = warp & 3;
    const int kh = (warp - 2) >> 2;
    const int row = q * 32 + lane;                     // query row of this thread
    const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16);
    float* const xmax = reinterpret_cast<float*>(smem_raw + (xch_base - smem_u32(smem_raw)));   // [2 buffers][2 halves][128 rows]
    float* const xl = xmax + 512;                                                               // [2 halves][128 rows]
    const int pair_bar = 1 + q;                        // named barrier of the two warps of this quadrant
    ATT_DECL(warp == 2 && lane == 0);
    int g = 0;
    for (int w = blockIdx.x; w < W; w += gridDim.x) {
      AttnItem a;
      if (!attn_item(w, QB, len, a)) continue;
      const int N = a.N, nt = a.nt;
      float m = -INFINITY, l = 0.f;
      float o[32];
#pragma unroll
      for (int e = 0; e < 32; e++) o[e] = 0.f;
      for (int j = 0; j < nt; j++) {
        const int gt = g + j, s = gt & 1;
        ATT(7);
        mbar_wait(sfull_bar(s), ((uint32_t)(gt >> 1)) & 1u);
        tc_fence_after();
        ATT(0);
        float sc[32];
        {
          uint32_t v[32];
          tmem_ld32(tq + kColS0 + 64u * (uint32_t)s + 32u * (uint32_t)kh, v);
#pragma unroll
          for (int e = 0; e < 32; e++) sc[e] = __uint_as_float(v[e]) * kSInv;     // exact: the planes' power-of-two scaling
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(sfree_bar(s));
        ATT(1);
        // key-padding mask + online softmax; the row maximum is the maximum over both halves
        const int kbase = j * 64 + kh * 32;
        float cm = -INFINITY;
#pragma unroll
        for (int e = 0; e < 32; e++) {
          if (kbase + e >= N) sc[e] = -INFINITY;
          cm = fmaxf(cm, sc[e]);
        }
        xmax[(s * 2 + kh) * 128 + row] = cm;
        asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
        cm = fmaxf(cm, xmax[(s * 2 + (kh ^ 1)) * 128 + row]);
        const float mn = fmaxf(m, cm);                   // finite: every tile holds at least one valid key
        const float corr = expf(m - mn);
        float ps = 0.f;
#pragma unroll
        for (int e = 0; e < 32; e++) { sc[e] = expf(sc[e] - mn); ps += sc[e]; }
        l = l * corr + ps;
        m = mn;
        ATT(2);
        // P_j -> TMEM as fp16 hi / lo planes of 4096 p, two keys per 32-bit column (A operand of the second MMA): this
        // warp's 32 keys are 16 columns of each plane.  The MMAs that read this P buffer two tiles ago are complete: this
        // thread waited for that O tile before it got here.
        {
          uint32_t ph[16], pl[16];
#pragma unroll
          for (int e = 0; e < 16; e++) {                 // two keys per packed conversion (cvt.rn.f16x2.f32): same rounding
            const float p0 = sc[2 * e] * kPScale, p1 = sc[2 * e + 1] * kPScale;
            const __half2 hi = __floats2half2_rn(p0, p1);
            const float2 hf = __half22float2(hi);
            const __half2 lo = __floats2half2_rn(p0 - hf.x, p1 - hf.y);
            ph[e] = *reinterpret_cast<const uint32_t*>(&hi);
            pl[e] = *reinterpret_cast<const uint32_t*>(&lo);
          }
          tmem_st16(tq + kColP + 64u * (uint32_t)s + 16u * (uint32_t)kh, ph);
          tmem_st16(tq + kColP + 64u * (uint32_t)s + 32u + 16u * (uint32_t)kh, pl);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pfull_bar(s));
        ATT(3);
        // fold in this warp's 32 dims of O_{j-1} (its MMAs ran under this tile's softmax), then rescale to the new
        // running maximum: the same operations in the same order as add-after-rescale inside one iteration
        if (j >= 1) {
          const int go = gt - 1, so = go & 1;
          mbar_wait(ofull_bar(so), ((uint32_t)(go >> 1)) & 1u);
          tc_fence_after();
          ATT(4);
          uint32_t v[32];
          tmem_ld32(tq + kColO + 64u * (uint32_t)so + 32u * (uint32_t)kh, v);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(ofree_bar(so));
#pragma unroll
          for (int e = 0; e < 32; e++) o[e] += __uint_as_float(v[e]) * kOInv;
        }
#pragma unroll
        for (int e = 0; e < 32; e++) o[e] *= corr;
        ATT(5);
      }
      {
        const int go = g + nt - 1, so = go & 1;
        mbar_wait(ofull_bar(so), ((uint32_t)(go >> 1)) & 1u);
        tc_fence_after();
        uint32_t v[32];
        tmem_ld32(tq + kColO + 64u * (uint32_t)so + 32u * (uint32_t)kh, v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ofree_bar(so));       // (the next work item reuses the buffer)
#pragma unroll
        for (int e = 0; e < 32; e++) o[e] += __uint_as_float(v[e]) * kOInv;
      }
      // the row sum is the sum of the two halves' sums, added in a fixed order
      xl[kh * 128 + row] = l;
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");
      if (a.q0 + row < N) {
        const float inv = 1.0f / (xl[row] + xl[128 + row]);
        float* dst = ctx + ((size_t)off[a.b] + a.q0 + row) * 768 + a.h * 64 + kh * 32;
#pragma unroll
        for (int e = 0; e < 32; e += 4)
          *reinterpret_cast<float4*>(dst + e) = make_float4(o[e] * inv, o[e + 1] * inv, o[e + 2] * inv, o[e + 3] * inv);
      }
      asm volatile("bar.sync %0, 64;" ::"r"(pair_bar) : "memory");     // xl is rewritten by the next work item
      ATT(6);
      g += nt;
    }
    ATT_FLUSH(8);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512u);
  }
}
}  // namespace

void attention_timing_dump() {
#ifdef KKX_TC_TIMING
  unsigned long long h[24] = {0};
  cudaMemcpyFromSymbol(h, g_attn_tim, sizeof h);
  unsigned long long z[24] = {0};
  cudaMemcpyToSymbol(g_attn_tim, z, sizeof z);
  fprintf(stderr, "[attention timing, CTA (0,0,0) of every launch] (kcycles) MMA wait_q %.1f wait_K %.1f wait_sfree %.1f issue_S %.1f wait_V %.1f wait_P %.1f wait_ofree %.1f issue_PV %.1f |"
          " SOFTMAX wait_S %.1f ld+arrive %.1f mask+exp %.1f split+st_P %.1f wait_O %.1f fold %.1f final %.1f loop %.1f\n",
          h[0] / 1e3, h[1] / 1e3, h[2] / 1e3, h[3] / 1e3, h[4] / 1e3, h[5] / 1e3, h[6] / 1e3, h[7] / 1e3,
          h[8] / 1e3, h[9] / 1e3, h[10] / 1e3, h[11] / 1e3, h[12] / 1e3, h[13] / 1e3, h[14] / 1e3, h[15] / 1e3);
#endif
}

// scratch size in floats: six fp16 planes (Q, K: hi / lo [rows, 768]; V^T: hi / lo [B * 768, 512])
size_t attention_umma_scratch_floats(int rows_total, int B) {
  return ((size_t)4 * rows_total * 768 + (size_t)2 * B * 768 * kVtPitch) / 2 + 64;
}

void attention_umma_planes(float* scratch, int rows_total, int B, void* (&pl)[6]) {
  const size_t plane = (size_t)rows_total * 768;
  __half* p0 = reinterpret_cast<__half*>(scratch);
  pl[0] = p0; pl[1] = p0 + plane; pl[2] = p0 + 2 * plane; pl[3] = p0 + 3 * plane;
  pl[4] = p0 + 4 * plane; pl[5] = p0 + 4 * plane + (size_t)B * 768 * kVtPitch;
}

void launch_attention_umma(const float* qkv, float* scratch, float* ctx, const int* off, const int* len, int B,
                           int max_len, int rows_total, cudaStream_t st, bool planes_ready) {
  if (g_dry_run) return;
  if (max_len > kVtPitch) throw ArgError("launch_attention_umma: more than 512 tokens");
  void* pl[6];
  attention_umma_planes(scratch, rows_total, B, pl);
  __half* qh = static_cast<__half*>(pl[0]); __half* ql = static_cast<__half*>(pl[1]);
  __half* kh = static_cast<__half*>(pl[2]); __half* kl = static_cast<__half*>(pl[3]);
  __half* vth = static_cast<__half*>(pl[4]); __half* vtl = static_cast<__half*>(pl[5]);
  const int dev = prepare_smem_launch<attn_umma_kernel>(kAttnSmem);
  if (!planes_ready) {
    dim3 gp((((max_len + 63) & ~63) + 31) / 32, 12, B);
    attn_prep_kernel<<<gp, 256, 0, st>>>(qkv, qh, ql, kh, kl, vth, vtl, off, len);
    post_launch("attn_prep", st);
  }
  alignas(64) CUtensorMap mQh, mQl, mKh, mKl, mVh, mVl;
  make_tmap_f16(&mQh, qh, 768, rows_total, 768, 128);
  make_tmap_f16(&mQl, ql, 768, rows_total, 768, 128);
  make_tmap_f16(&mKh, kh, 768, rows_total, 768, 64);
  make_tmap_f16(&mKl, kl, 768, rows_total, 768, 64);
  make_tmap_f16(&mVh, vth, kVtPitch, (long long)B * 768, kVtPitch, 64);
  make_tmap_f16(&mVl, vtl, kVtPitch, (long long)B * 768, kVtPitch, 64);
  const int QB = (max_len + 127) / 128, W = B * 12 * QB;
  const int nsm = device_sm_count(dev);
  attn_umma_kernel<<<W < nsm ? W : nsm, kAttnThreads, kAttnSmem, st>>>(mQh, mQl, mKh, mKl, mVh, mVl, off, len, ctx, QB, W);
  post_launch("attention", st);
}

}  // namespace kkx
