// kernels_arb.cu -- fused generator res-block convolution (SURVEY A.9 AdaINResBlock1, K6/K7/K8):
//
//   y[t, co] = bias[co] + sum_tap sum_c  snake( x[t + tap*dil - pad, c] * scale[b,c] + shift[b,c] ) * W[co, tap, c]
//
// as ONE persistent tcgen05 kernel per conv.  Compared with the generic conv_tc path (colstats ->
// adain_coef -> apply_bf16 -> conv_tc) it removes three HBM passes and most of the L2->SM operand
// traffic:
//   * the AdaIN scale/shift + Snake operand transform runs inside the kernel: 6 producer warps read the
//     raw activations (fp32 residual stream or bf16 intermediate) once per tile -- a halo tile of
//     128*MSUB + 2*pad rows per 64-channel chunk -- and write the bf16 operand straight into the
//     128B-swizzled smem layout the tensor core reads;
//   * every tap of the conv reads a ROW-SHIFTED VIEW of that one halo tile (UMMA descriptor start
//     address + tap*dil*128 B), so the activations are fetched once per tile instead of once per tap, and
//     each weight tile (TMA ring; resident when the whole set fits) is shared by all rows of the tile;
//   * the epilogue adds bias / residual, writes bf16 (conv1) or fp32 (conv2), and emits the per-128-row
//     column sums (sum x, sum x^2) the next AdaIN needs, so no separate statistics pass reads the tensor
//     again.  Two accumulator layouts: rows as M with a smem-transposed epilogue (C = 256), or the
//     transposed accumulator described at ArbCfg (C = 128) whose epilogue needs no transpose at all.
// TMEM holds two accumulator sets (512 columns): the epilogue of tile i overlaps the MMAs of tile i+1;
// the operand producers run one channel chunk (or more, with three slots) ahead of the MMA warp.
//
// Warp roles (512 threads, 1 CTA/SM, persistent over a contiguous range of tiles):
//   warp 0      weight-tile TMA producer          warp 1        TMEM alloc + tcgen05.mma issuer
//   warps 2-9   epilogue (two groups of 4)        warps 10-15   operand producers (transform)
#include "kernels.h"
#include "tc_ptx.cuh"
#include <type_traits>
#include <cstdlib>

namespace kkx {

namespace {

// Optional per-role phase timing (-DKKX_ARB_TIMING, diagnostics only): designated threads of CTA 0 attribute
// the cycles between consecutive TICKs to a slot and add their totals to a.timing[] at kernel end.
#ifdef KKX_ARB_TIMING
#define TIM_DECL(n) long long tim_acc[n] = {0}; long long tim_last = clock64(); const bool tim_on = a.timing && blockIdx.x == 0
#define TICK(slot) do { if (tim_on) { const long long now_ = clock64(); tim_acc[slot] += now_ - tim_last; tim_last = now_; } } while (0)
#define TIM_FLUSH(base, n) do { if (tim_on) for (int i_ = 0; i_ < (n); i_++) atomicAdd(reinterpret_cast<unsigned long long*>(a.timing) + (base) + i_, (unsigned long long)tim_acc[i_]); } while (0)
#else
#define TIM_DECL(n)
#define TICK(slot)
#define TIM_FLUSH(base, n)
#endif

// perf-experiment switches (skip loads / stores / math: wrong results, timing only) exist only in -DKKX_EXPERIMENTS builds
#ifdef KKX_EXPERIMENTS
#define ARB_DBG(a, bit) ((a).debug & (bit))
#else
#define ARB_DBG(a, bit) (0)
#endif

constexpr int kArbThreads = 512;   // 16 warps: TMA, MMA, 8 epilogue, 6 operand producers (128 regs/thread)
constexpr int kArbMaxB = 512;

// T ("transposed", C = 128 only): the WEIGHT tile is the M operand (128 output channels) and the 256
// activation rows are the N operand of one 128x256 MMA, so the accumulator is [channel][row]:
//   * a weight tile is read from smem once per 256 rows instead of once per 128 (the tensor pipe's own
//     operand reads saturate the 128 B/clk smem port at M = N = 128; 75 % with N = 256);
//   * after tcgen05.ld a thread owns ONE channel and 32 consecutive rows: global accesses are already
//     coalesced across the warp (32 channels = 128 contiguous bytes per row), so the epilogue needs no smem
//     transpose and no barrier, the bias is a per-thread scalar, and the AdaIN statistics are plain
//     per-thread sums (no shuffles); the freed smem holds a third operand slot.
// C = 256 keeps rows as M: 128-row tiles with a smem-transposed epilogue.  At C = 128 the transposed accumulator and the
// branch-free operand transform together took arb_conv from 104 to 93 ms per B = 64 step against rows as M
// (profiles/r1_step_b64_fused_v9_detail.txt).  512-row tiles at C = 128 (two 128x256 MMAs per weight tile, halving the
// weight re-streaming; the two accumulators fill TMEM, so the epilogue no longer overlaps the next tile's MMAs) were no
// net win on 5.7 M rows: conv1 k7 1.40 -> 1.25 ms, conv1 k11 unchanged, conv2 k7 / k11 1.65 -> 1.81 / 1.81 -> 2.19 ms.
template <int BN>
struct ArbCfg {
  static constexpr bool T = BN == 128;                      // transposed accumulator
  static constexpr int MSUB = T ? 2 : 1;                    // 128-row sub-tiles per tile
  static constexpr int KCH = BN / 64;                       // 64-channel chunks
  static constexpr int RA = MSUB * 128 + 56;                // rows per A slot (halo <= 2*25, 8-row granule)
  static constexpr uint32_t A_SLOT = RA * 128;              // bytes (multiple of 1024)
  static constexpr int NA = 3;                              // A slots
  static constexpr uint32_t B_STAGE = BN * 128;             // bytes
  static constexpr int NB = T ? 6 : 3;                      // B stages
  static constexpr int PITCH = 36;                          // floats per staged epilogue row
  static constexpr uint32_t STG = T ? 0 : 2 * 128 * PITCH * 4;   // one transpose buffer per epilogue group
  static constexpr uint32_t STAT = 4 * BN * 2 * 4;          // per-quadrant column sums
  static constexpr uint32_t COEF = 3 * BN * 4;              // per-item operand-transform coefficients
  static constexpr int NBAR = 2 * NA + 2 * NB + 4;
  static constexpr uint32_t SMEM = NA * A_SLOT + NB * B_STAGE + STG + STAT + COEF + NBAR * 8 + 16 + (3 * kArbMaxB + 2) * 4 + 1024;
  static_assert(A_SLOT % 1024 == 0, "A slot must keep the 1024-byte swizzle alignment");
};

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

// tile cursor: walks the (item, tile-in-item) pairs in item-major order
struct TileCur {
  int b, mt;
  __device__ __forceinline__ void init(const int* ts, int B, int tile) {
    int lo = 0, hi = B;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (ts[mid] <= tile) lo = mid; else hi = mid;
    }
    b = lo; mt = tile - ts[lo];
  }
  __device__ __forceinline__ void next(const int* ts) {
    mt++;
    while (ts[b] + mt >= ts[b + 1]) { b++; mt = 0; if (ts[b] < 0) break; }   // ts[B+1] = -1 sentinel
  }
};

// CONV2 = false: "conv1" of a res-block iteration -- fp32 input (residual stream), bf16 output, statistics.
// CONV2 = true : "conv2" -- bf16 input, fp32 output = (y + residual) * oscale (stored, or added to the
//                previous value with one reduction per element), optional statistics.
// The two roles are separate instantiations so that each carries only its own epilogue / producer code:
// with 16 warps in four different roles the hot code of all roles has to stay inside the instruction cache
// (an earlier, more generic version of this kernel lost ~40 % of its time to instruction-fetch stalls).
// POST (generator conv_post, 128 -> 22 channels, k = 7): the same pipeline with LeakyReLU as the operand transform,
// the weight set zero-padded to 128 output channels and an fp32 [rows, ldo] store of the first `cout` channels.
// The generic path re-fetched the activation tile for each of the 7 taps and needed a separate LeakyReLU -> bf16
// pass over the 4.7 GB stage output.
// SB ("stream in bf16"): the res-block's residual stream x is stored as bf16 between iterations instead of fp32.  The
// k = 3 / k = 7 convs are HBM-bound (16 B per row-channel and iteration with an fp32 stream); with a bf16 stream an
// iteration moves 10 B: conv1 reads bf16 x (SB = 1), conv2 reads the bf16 residual and writes either the next bf16 x
// (SB = 1) or -- last iteration -- the fp32 block output (SB = 2).  The AdaIN statistics still come from the fp32
// accumulator, before any rounding.
template <int BN, bool CONV2, bool POST = false, int SB = 0, bool PB = false>
__global__ void __launch_bounds__(kArbThreads, 1) arb_conv_kernel(const __grid_constant__ CUtensorMap tmB, ArbConvArgs a) {
  using Cfg = ArbCfg<BN>;
  constexpr bool T = Cfg::T;
  constexpr int MSUB = Cfg::MSUB;
  static_assert(SB == 0 || (!POST && (CONV2 || SB == 1)), "stream-bf16 variants: conv1 SB=1, conv2 SB=1 (bf16 out) / SB=2 (fp32 out)");
  static_assert(!PB || (T && !CONV2 && !POST && SB == 0), "balanced-producer variant: conv1, transposed accumulator, fp32 input");
  constexpr bool XIN_BF = CONV2 || SB != 0;          // element type of the operand the producers read
  constexpr bool OUT_BF = !CONV2 || SB == 1;         // epilogue writes bf16 (conv1 always; conv2 when the stream stays bf16)
  static_assert(!POST || (T && !CONV2), "post variant: transposed accumulator, fp32 input");
  // Warp split between epilogue and operand producers (14 warps besides TMA and MMA): 8 + 6.  A 4 + 10 split for
  // conv1 in transposed mode (trivial epilogue, producer-bound) was measured: no gain (1.14 / 1.35 / 1.61 ms vs
  // 1.20 / 1.29 / 1.63 ms at k = 3 / 7 / 11) -- the producers are limited by the shared-memory port they share
  // with the tensor pipe's operand reads, not by their thread count.
  // conv1 in transposed mode (trivial epilogue, producer-bound) can run 4 epilogue + 8 producer warps (+ 2 idle) so that
  // every scheduler carries two producer warps (with 8 + 6, schedulers 2 and 3 carry two producer warps each and a third
  // of the Snake sines: MUFU-bound).  Selected per launch by the PB template flag.
  constexpr int NEW = PB ? 4 : 8;                           // epilogue warps (4 is supported by the transposed epilogue)
  constexpr int NPW = PB ? 8 : 14 - NEW;                    // producer warps
  constexpr int kProdThreads = NPW * 32;
  constexpr int kProdRows = kProdThreads / 8;               // rows per producer pass (24 or 32: multiples of 8)
  constexpr int KCH = Cfg::KCH, NA = Cfg::NA, NB = Cfg::NB, PITCH = Cfg::PITCH;
  constexpr int MT = MSUB * 128;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const gbase = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t a_base = base;
  const uint32_t b_base = a_base + NA * Cfg::A_SLOT;
  const uint32_t stg_base = b_base + NB * Cfg::B_STAGE;
  const uint32_t stat_base = stg_base + Cfg::STG;
  const uint32_t coef_base = stat_base + Cfg::STAT;
  const uint32_t bar_base = coef_base + Cfg::COEF;
  const uint32_t tmem_slot = bar_base + Cfg::NBAR * 8;
  const uint32_t ts_base = tmem_slot + 16;
  auto fullA = [&](int s) { return bar_base + s * 8; };
  auto emptyA = [&](int s) { return bar_base + (NA + s) * 8; };
  auto fullB = [&](int s) { return bar_base + (2 * NA + s) * 8; };
  auto emptyB = [&](int s) { return bar_base + (2 * NA + NB + s) * 8; };
  auto tfull = [&](int j) { return bar_base + (2 * NA + 2 * NB + j) * 8; };
  auto tempty = [&](int j) { return bar_base + (2 * NA + 2 * NB + 2 + j) * 8; };
  int* const s_ts = reinterpret_cast<int*>(gbase + (ts_base - base));
  int* const s_len = s_ts + (kArbMaxB + 2);
  int* const s_off = s_len + kArbMaxB;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = a.B;
#pragma unroll 1
  for (int i = threadIdx.x; i <= B + 1; i += kArbThreads) s_ts[i] = i <= B ? a.tile_start[i] : -1;
#pragma unroll 1
  for (int i = threadIdx.x; i < B; i += kArbThreads) { s_len[i] = a.len[i]; s_off[i] = a.off[i]; }

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmB);
    for (int s = 0; s < NA; s++) { mbar_init(fullA(s), kProdThreads / 32); mbar_init(emptyA(s), 1); }
    for (int s = 0; s < NB; s++) { mbar_init(fullB(s), 1); mbar_init(emptyB(s), 1); }
    for (int j = 0; j < 2; j++) { mbar_init(tfull(j), 1); mbar_init(tempty(j), NEW); }
    mbar_init_fence();
  }
  if (warp == 1) {
    tmem_alloc<1>(tmem_slot, 512u);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_of(tmem_slot);

  // contiguous tile range of this CTA (neighbouring tiles share halo rows and, mostly, the item)
  const int t_begin = (int)(((long long)a.total_tiles * blockIdx.x) / gridDim.x);
  const int t_end = (int)(((long long)a.total_tiles * (blockIdx.x + 1)) / gridDim.x);
  const int ks = a.ks, dil = a.dil, pad = a.pad;

  if (warp == 0) {
    // ------------------------------------------------------------------ weight tiles (TMA)
    if (lane == 0 && t_begin < t_end) {
      int g = 0;
      TIM_DECL(2);
      // k=3 at C=128: the whole weight set (KCH*ks tiles) fits the ring -> load it once, keep it resident
      const bool resident = KCH * ks <= NB;
#pragma unroll 1
      for (int tile = t_begin; tile < (resident ? t_begin + 1 : t_end); tile++) {
#pragma unroll 1
        for (int c = 0; c < KCH; c++)
#pragma unroll 1
          for (int tap = 0; tap < ks; tap++, g++) {
            const int s = g % NB;
            mbar_wait(emptyB(s), (((uint32_t)(g / NB)) & 1u) ^ 1u);
            TICK(0);
            mbar_expect_tx(fullB(s), Cfg::B_STAGE);
            tma_load_2d(b_base + s * Cfg::B_STAGE, &tmB, tap * BN + c * 64, 0, fullB(s));
            TICK(1);
          }
      }
      TIM_FLUSH(0, 2);
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issue
    if (lane == 0 && t_begin < t_end) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN);
      int gA = 0, gB = 0, ti = 0;
      TileCur cur;
      cur.init(s_ts, B, t_begin);
      const bool resident = KCH * ks <= NB;
      TIM_DECL(4);
#pragma unroll 1
      for (int tile = t_begin; tile < t_end; tile++, ti++) {
        const int rem = s_len[cur.b] - cur.mt * MT;         // rows of this item left from the tile start
        (void)rem;
        const int buf = ti & 1;
        mbar_wait(tempty(buf), (((uint32_t)(ti >> 1)) & 1u) ^ 1u);
        tc_fence_after();
        TICK(0);
#pragma unroll 1
        for (int c = 0; c < KCH; c++, gA++) {
          const int sa = gA % NA;
          mbar_wait(fullA(sa), ((uint32_t)(gA / NA)) & 1u);
          tc_fence_after();
          TICK(1);
          const uint32_t slot = a_base + sa * Cfg::A_SLOT;
#pragma unroll 1
          for (int tap = 0; tap < ks; tap++, gB++) {
            const int sb = resident ? c * ks + tap : gB % NB;
            if (!resident || ti == 0) {
              mbar_wait(fullB(sb), resident ? 0u : ((uint32_t)(gB / NB)) & 1u);
              tc_fence_after();
            }
            TICK(2);
            const uint64_t bd = umma_desc_sw128(b_base + sb * Cfg::B_STAGE);
            if (T) {
              // D[co, row] += W[co, k] * Act[row + tap*dil, k]: weights = M operand, 256 rows = N operand
              constexpr uint32_t idescT = umma_idesc_bf16(128, 256);
              const uint64_t xd = umma_desc_sw128(slot + (uint32_t)(tap * dil) * 128u);
              const uint32_t td = tmem_base + (uint32_t)(buf * 256);
#pragma unroll
              for (int k = 0; k < 4; k++)
                if (!ARB_DBG(a, 8)) umma_bf16(td, bd + (uint64_t)(2 * k), xd + (uint64_t)(2 * k), idescT, (c | tap | k) ? 1u : 0u);
            } else {
#pragma unroll
              for (int sub = 0; sub < MSUB; sub++) {
                if (sub * 128 >= rem) continue;
                // row-shifted view of the halo tile: start address moves by whole 128-byte rows; the
                // 128B swizzle is a function of the absolute smem address, so the view stays consistent
                // with how the producers (and TMA) lay rows out (verified on B200, tools/arb_probe.py)
                const uint64_t ad = umma_desc_sw128(slot + (uint32_t)(sub * 128 + tap * dil) * 128u);
                const uint32_t td = tmem_base + (uint32_t)((buf * MSUB + sub) * BN);
#pragma unroll
                for (int k = 0; k < 4; k++)
                  umma_bf16(td, ad + (uint64_t)(2 * k), bd + (uint64_t)(2 * k), idesc, (c | tap | k) ? 1u : 0u);
              }
            }
            if (!resident) umma_commit(emptyB(sb));
            TICK(3);
          }
          umma_commit(emptyA(sa));
        }
        umma_commit(tfull(buf));
        cur.next(s_ts);
      }
      TIM_FLUSH(4, 4);
    }
  } else if (T && warp < 2 + NEW) {
    // ------------------------------------------------------------------ epilogue, transposed accumulator
    // warp: 32 channels (TMEM lane quadrant q) x 128 rows (row half eg); thread: one channel.  Register j of
    // a 32-column tcgen05.ld is row j of the chunk, so a warp-wide access to row j covers 32 consecutive
    // channels = 128 contiguous bytes.  No smem, no barrier; statistics are per-thread sums.
    const int eg = (warp - 2) >> 2;          // row group (NEW / 4 groups share the tile's rows)
    const int q = warp & 3;
    const int co = q * 32 + lane;
    const float bias_c = a.bias[co];
    const float2 bias2 = make_float2(bias_c, bias_c);
    const float2 os2 = make_float2(a.oscale, a.oscale);
    const bool accum = a.accumulate != 0;
    // residual rows are prefetched two 32-row chunks ahead (two register buffers), across tile boundaries
    constexpr int RW = MSUB * 128 / (NEW / 4);   // rows per epilogue warp (row group eg of the tile)
    constexpr int NCHK = RW / 32;            // 32-row chunks per warp and tile (4 or 8)
    auto fetchT = [&](int L, int off, int m0, int ch, float (&rv)[32]) {
      if (!CONV2 || ARB_DBG(a, 2)) return;
      const int row = m0 + eg * RW + ch * 32;
      const int left = L - row;
      if (SB) {
        const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(a.res) + (size_t)(off + row) * 128 + co;
#pragma unroll
        for (int j = 0; j < 32; j++)
          if (j < left) rv[j] = __bfloat162float(rp[j * 128]);
      } else {
        const float* rp = a.res + (size_t)(off + row) * 128 + co;
#pragma unroll
        for (int j = 0; j < 32; j++)
          if (j < left) {
            if (ARB_DBG(a, 32)) asm volatile("ld.global.L1::no_allocate.f32 %0, [%1];" : "=f"(rv[j]) : "l"(rp + j * 128));
            else rv[j] = rp[j * 128];
          }
      }
    };
    int ti = 0;
    TileCur cur;
    float rv0[32], rv1[32];
    if (t_begin < t_end) {
      cur.init(s_ts, B, t_begin);
      fetchT(s_len[cur.b], s_off[cur.b], cur.mt * MT, 0, rv0);
      fetchT(s_len[cur.b], s_off[cur.b], cur.mt * MT, 1, rv1);
    }
#ifdef KKX_ARB_TIMING
    long long tim_acc[9] = {0}; long long tim_last = clock64();
    const bool tim_on = a.timing && blockIdx.x == 0 && warp == 2 && lane == 0;
#endif
#pragma unroll 1
    for (int tile = t_begin; tile < t_end; tile++, ti++) {
      const int b = cur.b;
      const int L = s_len[b], off = s_off[b];
      const int m0 = cur.mt * MT;
      const int buf = ti & 1;
      cur.next(s_ts);                       // cur now names the NEXT tile (prefetch target)
      const bool has_next = tile + 1 < t_end;
      const int nL = has_next ? s_len[cur.b] : 0, noff = has_next ? s_off[cur.b] : 0, nm0 = cur.mt * MT;
      TICK(8);
      mbar_wait(tfull(buf), ((uint32_t)(ti >> 1)) & 1u);
      tc_fence_after();
      TICK(0);
      float2 s2 = make_float2(0.f, 0.f), q2 = s2;
      auto bodyT = [&](int ch, float (&rv)[32], auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        const int row = m0 + eg * RW + ch * 32;
        const int left = ARB_DBG(a, 2) ? 0 : L - row;
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 256 + eg * RW + ch * 32), v);
        if (ch == NCHK - 1) {      // last TMEM read of this tile by this warp
          tc_fence_before();
          if (lane == 0) mbar_arrive(tempty(buf));
        }
        TICK(1);
        if (CONV2 && !OUT_BF) {
          float* op = a.out_f32 + (size_t)(off + row) * 128 + co;
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            float2 o = make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
            o = __fadd2_rn(__fadd2_rn(o, make_float2(rv[j], rv[j + 1])), bias2);
            if (!FULL) { o.x = j < left ? o.x : 0.f; o.y = j + 1 < left ? o.y : 0.f; }
            s2 = __fadd2_rn(s2, o);
            q2 = __ffma2_rn(o, o, q2);
            o = __fmul2_rn(o, os2);
            if (accum) {      // exactly one add per element and launch -> order-independent
              if (FULL || j < left) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(op + j * 128), "f"(o.x) : "memory");
              if (FULL || j + 1 < left) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(op + (j + 1) * 128), "f"(o.y) : "memory");
            } else {
              if (FULL || j < left) op[j * 128] = o.x;
              if (FULL || j + 1 < left) op[(j + 1) * 128] = o.y;
            }
          }
        } else if (POST) {
          // fp32 [rows, ldo] store of the real output channels (co < cout: 88 contiguous bytes per row for 22)
          if (co < a.cout) {
            float* op = a.out_f32 + (size_t)(off + row) * a.ldo + co;
#pragma unroll
            for (int j = 0; j < 32; j++)
              if (FULL || j < left) op[(size_t)j * a.ldo] = __uint_as_float(v[j]) + bias_c;
          }
        } else {
          // bf16 output: lanes 2i / 2i+1 exchange so that each lane stores one 4-byte word (two channels):
          // even lanes the word of row j, odd lanes the word of row j+1
          const int odd = lane & 1;
          __nv_bfloat16* op = a.out_bf16 + (size_t)(off + row + odd) * 128 + (co & ~1);
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            float2 o = make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
            if (CONV2) o = __fadd2_rn(o, make_float2(rv[j], rv[j + 1]));      // bf16 stream: x_next = y + x (+ bias below)
            o = __fadd2_rn(o, bias2);
            if (!FULL) { o.x = j < left ? o.x : 0.f; o.y = j + 1 < left ? o.y : 0.f; }
            s2 = __fadd2_rn(s2, o);
            q2 = __ffma2_rn(o, o, q2);
            const float send = odd ? o.x : o.y;
            const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
            const uint32_t w = odd ? pack_bf16(recv, o.y) : pack_bf16(o.x, recv);
            if (FULL || j + odd < left) *reinterpret_cast<uint32_t*>(op + j * 128) = w;
          }
        }
        TICK(5);
        // refill this register buffer with the rows of chunk ch+2 (possibly of the next tile)
        if (ch + 2 < NCHK) fetchT(L, off, m0, ch + 2, rv);
        else if (has_next) fetchT(nL, noff, nm0, ch + 2 - NCHK, rv);
        TICK(6);
        if ((ch & 3) == 3) {   // 128 rows done: one thread per channel and statistics chunk
          if (a.part && row - 96 < L) {
            float* pp = a.part + ((size_t)b * a.nchunk + (size_t)((row - 96) >> 7)) * 2 * 128 + co;
            pp[0] = s2.x + s2.y;
            pp[128] = q2.x + q2.y;
          }
          s2 = make_float2(0.f, 0.f); q2 = s2;
        }
      };
      if (L - m0 >= MT && !ARB_DBG(a, 2)) {
#pragma unroll
        for (int ch = 0; ch < NCHK; ch += 2) { bodyT(ch, rv0, std::true_type{}); bodyT(ch + 1, rv1, std::true_type{}); }
      } else {
#pragma unroll
        for (int ch = 0; ch < NCHK; ch += 2) { bodyT(ch, rv0, std::false_type{}); bodyT(ch + 1, rv1, std::false_type{}); }
      }
      TICK(7);
    }
    TIM_FLUSH(8, 9);
  } else if (!T && warp < 10) {
    // ------------------------------------------------------------------ epilogue (2 groups of 4 warps)
    // group eg owns the 32-column chunks of parity eg; inside a group, thread `et` drops its accumulator
    // row into padded smem, then thread t handles columns c4..c4+3 of rows (t>>3) + 16*i (full 128-byte
    // row segments per 8 lanes -> coalesced residual reads and stores).
    const int eg = (warp - 2) >> 2;
    const int q = warp & 3;                 // TMEM lane quadrant of this warp
    const int et = q * 32 + lane;           // accumulator row held by this thread
    const int t = (threadIdx.x - 64) & 127; // 0..127 inside the group
    const int tr = t >> 3;                  // first row handled after the transpose
    const int c4 = (t & 7) << 2;
    const int bar_id = 1 + eg;
    float* const buf_f = reinterpret_cast<float*>(gbase + (stg_base - base)) + eg * (128 * PITCH);
    float* const stat_f = reinterpret_cast<float*>(gbase + (stat_base - base));   // [4][BN][2]
    const float* const st_rd = buf_f + tr * PITCH + c4;
    float* const st_wr = buf_f + et * PITCH;
    constexpr int NCH = BN / 64;            // 32-column chunks per group and sub-tile (2 or 4)
    constexpr int RS = 16 * BN;             // elements between the rows one thread handles
    const float2 os2 = make_float2(a.oscale, a.oscale);
    const bool accum = a.accumulate != 0;
    // Residual operands are prefetched TWO chunk iterations ahead (two register buffers), across sub-tile
    // and tile boundaries: with ~2 us of HBM latency under load, one iteration of lead is not enough.
    auto fetch = [&](int L, int off, int m0, int e, float4 (&rv)[8]) {   // iteration e of a tile: (sub, chunk)
      if (!CONV2) return;
      const int sub = e / NCH, ci = e & (NCH - 1);
      const int row = m0 + sub * 128 + tr;
      const int left = L - row;            // row i valid iff 16*i < left
      if (SB) {
        const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(a.res) + (size_t)(off + row) * BN + ((2 * ci + eg) * 32 + c4);
#pragma unroll
        for (int i = 0; i < 8; i++)
          if (16 * i < left) {
            const uint2 w = *reinterpret_cast<const uint2*>(rp + i * RS);
            rv[i] = make_float4(__uint_as_float(w.x << 16), __uint_as_float(w.x & 0xFFFF0000u),
                                __uint_as_float(w.y << 16), __uint_as_float(w.y & 0xFFFF0000u));
          }
      } else {
        const float* rp = a.res + (size_t)(off + row) * BN + ((2 * ci + eg) * 32 + c4);
#pragma unroll
        for (int i = 0; i < 8; i++)
          if (16 * i < left) rv[i] = *reinterpret_cast<const float4*>(rp + i * RS);
      }
    };
    int ti = 0;
    TileCur cur;
    float4 rv0[8], rv1[8];
#ifdef KKX_ARB_TIMING
    long long tim_acc[9] = {0}; long long tim_last = clock64();
    const bool tim_on = a.timing && blockIdx.x == 0 && warp == 2 && lane == 0;
#endif
    if (t_begin < t_end) {
      cur.init(s_ts, B, t_begin);
      fetch(s_len[cur.b], s_off[cur.b], cur.mt * MT, 0, rv0);
      fetch(s_len[cur.b], s_off[cur.b], cur.mt * MT, 1, rv1);
    }
#pragma unroll 1
    for (int tile = t_begin; tile < t_end; tile++, ti++) {
      const int b = cur.b;
      const int L = s_len[b], off = s_off[b];
      const int m0 = cur.mt * MT;
      const int nsub = min(MSUB, (L - m0 + 127) >> 7);
      const int E = nsub * NCH;
      const int buf = ti & 1;
      cur.next(s_ts);                       // cur now names the NEXT tile (prefetch target)
      const bool has_next = tile + 1 < t_end;
      const int nL = has_next ? s_len[cur.b] : 0, noff = has_next ? s_off[cur.b] : 0, nm0 = cur.mt * MT;
      TICK(8);
      mbar_wait(tfull(buf), ((uint32_t)(ti >> 1)) & 1u);
      tc_fence_after();
      TICK(0);
      auto body = [&](int e, float4 (&rv)[8], auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;   // every row of the sub-tile is inside the item
        const int sub = e / NCH, ci = e & (NCH - 1);
        const int row = m0 + sub * 128 + tr;
        const int n = (2 * ci + eg) * 32 + c4;
        {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * MSUB + sub) * BN + n - c4), v);
          if (e == E - 1) {   // last TMEM read of this tile: hand the accumulators back
            tc_fence_before();
            if (lane == 0) mbar_arrive(tempty(buf));
          }
          TICK(1);
          asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");   // staging buffer drained by the previous iteration
          TICK(2);
#pragma unroll
          for (int j = 0; j < 32; j += 4)
            *reinterpret_cast<uint4*>(st_wr + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          TICK(3);
        }
        asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
        TICK(4);
        const float4 bb = *reinterpret_cast<const float4*>(a.bias + n);
        const float2 b01 = make_float2(bb.x, bb.y), b23 = make_float2(bb.z, bb.w);
        const int left = L - row;
        const size_t g0 = (size_t)(off + row) * BN + n;
        float2 s01 = make_float2(0.f, 0.f), s23 = s01, q01 = s01, q23 = s01;
        // packed fp32 (FADD2 / FFMA2 / FMUL2): the epilogue is issue-bound, this halves its math instructions
#pragma unroll
        for (int i = 0; i < 8; i++) {
          const bool ok = FULL || 16 * i < left;
          const float4 ov = *reinterpret_cast<const float4*>(st_rd + i * 16 * PITCH);
          float2 o01 = make_float2(ov.x, ov.y), o23 = make_float2(ov.z, ov.w);
          if (CONV2) { o01 = __fadd2_rn(o01, make_float2(rv[i].x, rv[i].y)); o23 = __fadd2_rn(o23, make_float2(rv[i].z, rv[i].w)); }
          o01 = __fadd2_rn(o01, b01); o23 = __fadd2_rn(o23, b23);
          if (!FULL) { o01.x = ok ? o01.x : 0.f; o01.y = ok ? o01.y : 0.f; o23.x = ok ? o23.x : 0.f; o23.y = ok ? o23.y : 0.f; }
          s01 = __fadd2_rn(s01, o01); s23 = __fadd2_rn(s23, o23);
          q01 = __ffma2_rn(o01, o01, q01); q23 = __ffma2_rn(o23, o23, q23);
          if (OUT_BF) {
            uint2 pk;
            pk.x = pack_bf16(o01.x, o01.y); pk.y = pack_bf16(o23.x, o23.y);
            if (ok) *reinterpret_cast<uint2*>(a.out_bf16 + g0 + i * RS) = pk;
          } else {
            o01 = __fmul2_rn(o01, os2); o23 = __fmul2_rn(o23, os2);
            float* op = a.out_f32 + g0 + i * RS;
            if (ok) {
              if (accum)   // exactly one add per element and launch -> order-independent, no load round trip
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(op), "f"(o01.x), "f"(o01.y), "f"(o23.x), "f"(o23.y) : "memory");
              else
                *reinterpret_cast<float4*>(op) = make_float4(o01.x, o01.y, o23.x, o23.y);
            }
          }
        }
        TICK(5);
        // refill this register buffer with the operand of iteration e+2 (possibly of the next tile)
        if (e + 2 < E) fetch(L, off, m0, e + 2, rv);
        else if (has_next) fetch(nL, noff, nm0, e + 2 - E, rv);
        TICK(6);
        if (a.part) {
          // rows of one column quad live in lanes l, l+8, l+16, l+24
#pragma unroll
          for (int d = 8; d <= 16; d <<= 1) {
            float2 t0, t1, t2, t3;
            t0.x = __shfl_xor_sync(0xffffffffu, s01.x, d); t0.y = __shfl_xor_sync(0xffffffffu, s01.y, d);
            t1.x = __shfl_xor_sync(0xffffffffu, s23.x, d); t1.y = __shfl_xor_sync(0xffffffffu, s23.y, d);
            t2.x = __shfl_xor_sync(0xffffffffu, q01.x, d); t2.y = __shfl_xor_sync(0xffffffffu, q01.y, d);
            t3.x = __shfl_xor_sync(0xffffffffu, q23.x, d); t3.y = __shfl_xor_sync(0xffffffffu, q23.y, d);
            s01 = __fadd2_rn(s01, t0); s23 = __fadd2_rn(s23, t1); q01 = __fadd2_rn(q01, t2); q23 = __fadd2_rn(q23, t3);
          }
          if (lane < 8) {
            // warp w of the group covers rows 2w, 2w+1 (+16i) of the transposed tile: slot (t >> 5)
            float* sp = stat_f + ((size_t)(t >> 5) * BN + n) * 2;
            *reinterpret_cast<float4*>(sp) = make_float4(s01.x, q01.x, s01.y, q01.y);
            *reinterpret_cast<float4*>(sp + 4) = make_float4(s23.x, q23.x, s23.y, q23.y);
          }
          if (ci == NCH - 1) {   // sub-tile complete: combine the four warps' sums in a fixed order
            asm volatile("bar.sync %0, 128;" ::"r"(bar_id) : "memory");
            if (t < BN / 2) {
              const int nn = ((t >> 5) * 2 + eg) * 32 + (t & 31);
              float* pp = a.part + ((size_t)b * a.nchunk + (size_t)((m0 >> 7) + sub)) * 2 * BN + nn;
              const float* sf = stat_f + 2 * nn;
              pp[0] = (sf[0] + sf[2 * BN]) + (sf[4 * BN] + sf[6 * BN]);
              pp[BN] = (sf[1] + sf[2 * BN + 1]) + (sf[4 * BN + 1] + sf[6 * BN + 1]);
            }
            // the next statistic write happens after two more group barriers
          }
        }
        TICK(7);
      };
      if (L - m0 >= MT) {   // hot path: full tile, no row predicates
#pragma unroll 1
        for (int e = 0; e < E; e += 2) {
          body(e, rv0, std::true_type{});
          body(e + 1, rv1, std::true_type{});
        }
        continue;
      }
#pragma unroll 1
      for (int e = 0; e < E; e += 2) {   // last tile of an item
        body(e, rv0, std::false_type{});
        body(e + 1, rv1, std::false_type{});
      }
    }
    TIM_FLUSH(8, 9);
  } else if (warp < 2 + NEW + NPW) {
    // ------------------------------------------------------------------ operand producers
    // y = snake(x*sc + sh) = ial * (u + sin(u)^2), u = x*(al*sc) + al*sh: three per-channel coefficients,
    // cached in smem per item.  Loads run one group (4 passes of 24 rows) ahead of the transform through
    // two register buffers, across chunk and tile boundaries, so HBM/L2 latency stays hidden.
    const int pt = threadIdx.x - (2 + NEW) * 32;   // 0..kProdThreads-1
    const int cg = pt & 7;                  // 8-channel group inside the 64-channel chunk
    const int rl = pt >> 3;                 // row lane 0..23
    constexpr int GP = PB ? 3 : 4;         // (bf16-input producers with 6 passes per group, 18 instead of 12 KB in flight: no change, v34)
    constexpr int GR = GP * kProdRows;      // rows per load group (96: a multiple of 8 -> constant swizzle phase)
    const int ra_used = MT + 2 * pad;       // <= Cfg::RA
    const int ngc = (ra_used + GR - 1) / GR;                 // load groups per chunk
    float* const coef = reinterpret_cast<float*>(gbase + (coef_base - base));   // [3][BN]: al*sc, al*sh, 1/al
    const int F = (t_end - t_begin) * KCH * ngc;
    using Raw = typename std::conditional<XIN_BF, uint4, float4>::type;
    constexpr int RPP = XIN_BF ? 1 : 2;     // raw vectors per pass (8 channels)
    constexpr int XE = XIN_BF ? 2 : 4;      // bytes per input element
    // this thread's byte offset inside an A slot, minus the row part: 16-byte chunk cg of row r sits at
    // chunk position cg ^ (r & 7); all rows this thread writes have r = rl (mod 8)
    const uint32_t sw = (uint32_t)rl * 128u + (uint32_t)((cg ^ (rl & 7)) << 4);

    TileCur lc; int l_c = 0, l_g = 0;                                  // load stream
    TileCur sc_; int s_c = 0, s_g = 0, gA = 0, coef_b = -1;             // transform stream
    if (F > 0) { lc.init(s_ts, B, t_begin); sc_ = lc; }
    float2 cA[4], cB[4], cI[4];
#ifdef KKX_ARB_TIMING
    long long tim_acc[5] = {0}; long long tim_last = clock64();
    const bool tim_on = a.timing && blockIdx.x == 0 && warp == 10 && lane == 0;
#endif

    auto issue = [&](Raw (&rb)[GP][RPP]) {
      const int L = s_len[lc.b];
      const int row = lc.mt * MT - pad + l_g * GR + rl;     // item-relative row of pass 0
      const int rloc = l_g * GR + rl;
      const char* xp = reinterpret_cast<const char*>(a.x) + ((size_t)(s_off[lc.b] + row) * BN + (l_c * 64 + cg * 8)) * XE;
#pragma unroll
      for (int p = 0; p < GP; p++) {
        if ((unsigned)(row + p * kProdRows) < (unsigned)L && rloc + p * kProdRows < ra_used && !ARB_DBG(a, 1)) {
#pragma unroll
          for (int v = 0; v < RPP; v++) {
            const char* gp = xp + (size_t)p * kProdRows * BN * XE + v * 16;
            if (ARB_DBG(a, 16)) {
              uint4 t;
              asm volatile("ld.global.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(t.x), "=r"(t.y), "=r"(t.z), "=r"(t.w) : "l"(gp));
              rb[p][v] = *reinterpret_cast<Raw*>(&t);
            } else rb[p][v] = *reinterpret_cast<const Raw*>(gp);
          }
        }
      }
      if (++l_g == ngc) { l_g = 0; if (++l_c == KCH) { l_c = 0; lc.next(s_ts); } }
    };
    auto process = [&](Raw (&rb)[GP][RPP]) {
      const int b = sc_.b;
      const int sa = gA % NA;
      if (s_g == 0) {
        if (!POST && b != coef_b) {   // new item: rebuild the coefficient table (all producer threads take this branch together)
          asm volatile("bar.sync 3, %0;" ::"n"(kProdThreads) : "memory");
          for (int ch = pt; ch < BN; ch += kProdThreads) {
            const float al = a.alpha[ch], s = a.scale[(size_t)b * BN + ch], h = a.shift[(size_t)b * BN + ch];
            coef[ch] = al * s; coef[BN + ch] = al * h; coef[2 * BN + ch] = 1.0f / al;
          }
          asm volatile("bar.sync 3, %0;" ::"n"(kProdThreads) : "memory");
          coef_b = b;
        }
        const float* cp = coef + s_c * 64 + cg * 8;
#pragma unroll
        for (int e = 0; !POST && e < 4; e += 2) {
          const float4 t0 = *reinterpret_cast<const float4*>(cp + 2 * e);
          const float4 t1 = *reinterpret_cast<const float4*>(cp + BN + 2 * e);
          const float4 t2 = *reinterpret_cast<const float4*>(cp + 2 * BN + 2 * e);
          cA[e] = make_float2(t0.x, t0.y); cA[e + 1] = make_float2(t0.z, t0.w);
          cB[e] = make_float2(t1.x, t1.y); cB[e + 1] = make_float2(t1.z, t1.w);
          cI[e] = make_float2(t2.x, t2.y); cI[e + 1] = make_float2(t2.z, t2.w);
        }
        TICK(1);
        mbar_wait(emptyA(sa), (((uint32_t)(gA / NA)) & 1u) ^ 1u);
        TICK(2);
      }
      const int L = s_len[b];
      const int row = sc_.mt * MT - pad + s_g * GR + rl;
      const int rloc = s_g * GR + rl;
      uint8_t* const sp = gbase + (a_base - base) + (size_t)sa * Cfg::A_SLOT + (size_t)(s_g * GR) * 128 + sw;
#pragma unroll
      for (int p = 0; p < GP; p++) {
        // straight-line: rows outside the item produce zeros through a select, only the store is predicated
        const uint32_t inmask = (unsigned)(row + p * kProdRows) < (unsigned)L ? 0xFFFFFFFFu : 0u;
        float2 xv[4];
        if (XIN_BF) {
          const uint4 raw = *reinterpret_cast<const uint4*>(&rb[p][0]);
          xv[0] = make_float2(__uint_as_float(raw.x << 16), __uint_as_float(raw.x & 0xFFFF0000u));
          xv[1] = make_float2(__uint_as_float(raw.y << 16), __uint_as_float(raw.y & 0xFFFF0000u));
          xv[2] = make_float2(__uint_as_float(raw.z << 16), __uint_as_float(raw.z & 0xFFFF0000u));
          xv[3] = make_float2(__uint_as_float(raw.w << 16), __uint_as_float(raw.w & 0xFFFF0000u));
        } else {
          const float4 f0 = *reinterpret_cast<const float4*>(&rb[p][0]);
          const float4 f1 = *reinterpret_cast<const float4*>(&rb[p][RPP - 1]);
          xv[0] = make_float2(f0.x, f0.y); xv[1] = make_float2(f0.z, f0.w);
          xv[2] = make_float2(f1.x, f1.y); xv[3] = make_float2(f1.z, f1.w);
        }
        uint32_t pw[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {   // packed fp32 math around the two scalar MUFU.SIN
          if (POST) {      // LeakyReLU: max(x, slope * x) for 0 < slope < 1
            const float2 lx = __fmul2_rn(xv[e], make_float2(a.slope, a.slope));
            pw[e] = pack_bf16(fmaxf(xv[e].x, lx.x), fmaxf(xv[e].y, lx.y)) & inmask;
            continue;
          }
          if (ARB_DBG(a, 4)) { pw[e] = pack_bf16(xv[e].x, xv[e].y) & inmask; continue; }
          const float2 u = __ffma2_rn(xv[e], cA[e], cB[e]);
          const float2 sn = make_float2(__sinf(u.x), __sinf(u.y));
          const float2 y = __fmul2_rn(__ffma2_rn(sn, sn, u), cI[e]);
          pw[e] = pack_bf16(y.x, y.y) & inmask;   // mask, not select: keeps the 16 chains of a group branch-free
        }
        const uint4 pk = make_uint4(pw[0], pw[1], pw[2], pw[3]);
        if (rloc + p * kProdRows < ra_used) *reinterpret_cast<uint4*>(sp + p * kProdRows * 128) = pk;
      }
      TICK(3);
      if (++s_g == ngc) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(fullA(sa));
        s_g = 0; gA++;
        if (++s_c == KCH) { s_c = 0; sc_.next(s_ts); }
      }
    };

    Raw bufA[GP][RPP], bufB[GP][RPP];
#pragma unroll
    for (int p = 0; p < GP; p++)
#pragma unroll
      for (int v = 0; v < RPP; v++) { bufA[p][v] = Raw(); bufB[p][v] = Raw(); }
    if (F > 0) issue(bufA);
#pragma unroll 1
    for (int f = 0; f < F; f += 2) {
      if (f + 1 < F) issue(bufB);
      TICK(0);
      process(bufA);
      if (f + 1 >= F) break;
      if (f + 2 < F) issue(bufA);
      TICK(0);
      process(bufB);
    }
    TIM_FLUSH(20, 5);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512u);
  }
}

template <int BN, bool CONV2, bool POST = false, int SB = 0, bool PB = false>
void launch_arb_t(const ArbConvArgs& a, cudaStream_t st) {
  using Cfg = ArbCfg<BN>;
  const int dev = prepare_smem_launch<arb_conv_kernel<BN, CONV2, POST, SB, PB>>((int)Cfg::SMEM);
  const int nsm = device_sm_count(dev);
  const int grid = a.total_tiles < nsm ? a.total_tiles : nsm;
  arb_conv_kernel<BN, CONV2, POST, SB, PB><<<grid, kArbThreads, Cfg::SMEM, st>>>(*reinterpret_cast<const CUtensorMap*>(a.tmB), a);
}

}  // namespace

int arb_tile_rows(int C) { return (C == 128 ? ArbCfg<128>::MSUB : ArbCfg<256>::MSUB) * 128; }

bool arb_conv_supported(int C, int ks, int dil, int B) {
  return (C == 128 || C == 256) && ks >= 1 && dil >= 1 && dil * (ks - 1) <= 50 && (ks & 1) && B <= kArbMaxB;
}

void launch_arb_conv(const ArbConvArgs& a, cudaStream_t st) {
  if (g_dry_run) return;
  if (a.total_tiles <= 0 || a.B <= 0) return;
  if (!arb_conv_supported(a.C, a.ks, a.dil, a.B)) throw ArgError("launch_arb_conv: unsupported shape");
  if (a.post) {
    if (a.C != 128 || a.in_bf16 || !a.out_f32 || a.out_bf16 || a.res || a.accumulate || a.part || a.cout < 1 || a.cout > 128 ||
        a.ldo < a.cout || !(a.slope > 0.f && a.slope < 1.f))
      throw ArgError("launch_arb_conv: unsupported post-conv arguments");
    if (g_launch_stats) g_launch_stats->conv_flops += 2.0 * (double)a.sum_m * a.C * a.cout * a.ks;
    launch_arb_t<128, false, true>(a, st);
    post_launch("post_conv", st);
    return;
  }
  // roles: conv1 = (fp32 | bf16 stream) in -> bf16 out (+statistics); conv2 = bf16 in + (fp32 | bf16) residual ->
  // fp32 out (block output / fp32 stream) or bf16 out (next x of a bf16 stream)
  const bool conv2 = a.res != nullptr;
  if (conv2 ? (!a.in_bf16 || (a.out_f32 != nullptr) == (a.out_bf16 != nullptr) || (a.out_bf16 && (!a.res_bf16 || a.accumulate)))
            : (!a.out_bf16 || a.out_f32 || a.accumulate || a.res_bf16))
    throw ArgError("launch_arb_conv: unsupported input/output combination");
#ifdef KKX_EXPERIMENTS
  static const int dbg = env_int("KKX_ARB_DBG", 0);
  if (dbg && !a.debug) { ArbConvArgs d = a; d.debug = dbg; launch_arb_conv(d, st); return; }
#endif
  const bool stream_bf = conv2 ? a.res_bf16 != 0 : a.in_bf16 != 0;
  if (g_launch_stats) {
    const double fl = 2.0 * (double)a.sum_m * a.C * a.C * a.ks;
    g_launch_stats->conv_flops += fl;
    g_launch_stats->arb_flops += fl;
    // every tensor once: conv1 reads x (4 / 2 B), writes bf16; conv2 reads bf16 + the residual (4 / 2 B), writes 4 / 2 B
    const double bytes = conv2 ? 2.0 + (a.res_bf16 ? 2.0 : 4.0) + (a.out_bf16 ? 2.0 : 4.0) : (a.in_bf16 ? 2.0 : 4.0) + 2.0;
    g_launch_stats->arb_bytes += (double)a.sum_m * a.C * bytes;
  }
  if (stream_bf) {
    if (a.C == 128) {
      if (!conv2) launch_arb_t<128, false, false, 1>(a, st);
      else if (a.out_bf16) launch_arb_t<128, true, false, 1>(a, st);
      else launch_arb_t<128, true, false, 2>(a, st);
    } else {
      if (!conv2) launch_arb_t<256, false, false, 1>(a, st);
      else if (a.out_bf16) launch_arb_t<256, true, false, 1>(a, st);
      else launch_arb_t<256, true, false, 2>(a, st);
    }
  } else if (a.C == 128) {
    // conv1: 4 epilogue + 8 producer warps, two producer warps on every scheduler -- measured against 8 + 6 on one box
    // (profiles/r2_arb_balanced_producers_v32.txt): k = 3 1.45 -> 1.15 ms, k = 7 1.50 -> 1.25 ms, k = 11 unchanged
    if (a.in_bf16) launch_arb_t<128, true>(a, st); else launch_arb_t<128, false, false, 0, true>(a, st);
  } else {
    if (a.in_bf16) launch_arb_t<256, true>(a, st); else launch_arb_t<256, false>(a, st);
  }
  if (g_launch_stats && g_launch_stats->profile && g_launch_stats->detail) {
    char nm[96]; snprintf(nm, sizeof nm, "arb_conv[c%d k%d d%d %s%s m%lld]", a.C, a.ks, a.dil, conv2 ? "conv2" : "conv1", stream_bf ? " sb" : "", a.sum_m);
    post_launch(nm, st);
  } else post_launch("arb_conv", st);
}

}  // namespace kkx
