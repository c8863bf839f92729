// kernels_flac.cu -- lossless FLAC encoding of 16-bit mono PCM on the device (kkx_infer_batch_flac, kkx.h).
//
// Every item becomes one FLAC stream (RFC 9639, streamable subset): a 42-byte head (fLaC + STREAMINFO), then frames
// of 4096 samples, each with one CONSTANT, FIXED (order 0..4, Rice partitions), LPC (order p = "flac_lpc_order", when
// that is on) or VERBATIM subframe.  The choice and every byte are a pure function of the item's samples (integer
// arithmetic, plus the LPC coefficient design in IEEE binary64 with one rounding per operation in a fixed order; ties
// broken by a fixed rule), so an item encodes to the same bytes whatever batch it is in.  Three launches:
//   flac_analyze  one CTA per frame: cost of every (order, partition order, Rice parameter) -> choice + frame size;
//                 its LPC variant first designs the frame's order-p predictor (window, autocorrelation, Levinson-
//                 Durbin, quantisation) on the block it already holds in shared memory
//   flac_scan     one CTA: byte offset of every frame and every item
//   flac_pack     one CTA per frame: bit positions by a block scan, codes OR-ed into a shared bit buffer, CRC-8 of
//                 the header and CRC-16 of the frame, then the frame's bytes; the CTA of an item's first frame also
//                 writes the item's 42-byte head (STREAMINFO needs the item's smallest and largest frame).
#include "kernels.h"
#include "bitpack.cuh"
#include <cmath>

namespace kkx {

namespace {
constexpr int kBlock = 4096;          // samples per frame (STREAMINFO min = max block size)
constexpr int kThreads = 256;         // one CTA per frame, 16 samples per thread
constexpr int kPer = kBlock / kThreads;
constexpr int kMaxPorder = 8;         // 256 partitions at most
constexpr int kParts = 1 << kMaxPorder;
constexpr int kOrders = 5, kRice = 15;
constexpr int kHead = 42;             // "fLaC" + metadata block header + 34-byte STREAMINFO
constexpr int kLpcPrec = 12;          // quantised coefficient precision (bits)
constexpr int kLpcWin = 1024;         // entries of the window's taper table M

enum : int { SUB_CONSTANT = 0, SUB_FIXED = 1, SUB_VERBATIM = 2, SUB_LPC = 3 };

struct FlacFrame {        // analysis result of one frame
  int bytes;              // whole frame, header and CRC-16 included
  int kind, order, porder;
  unsigned char k[kParts];  // Rice parameter of each partition (FIXED, LPC)
  int shift;                // LPC: quantisation shift and coefficients q_1..q_order
  short q[kMaxLpcOrder];
};

// M[k] = nint(2^15 * 0.5 * (1 - cos(pi (k + 0.5) / 1024))), designed in double on the host, uploaded once per device
__device__ int g_lpc_window[kLpcWin];

__host__ __device__ inline int utf8_len(unsigned v) {
  return v < 0x80 ? 1 : v < 0x800 ? 2 : v < 0x10000 ? 3 : v < 0x200000 ? 4 : v < 0x4000000 ? 5 : 6;
}
__device__ __forceinline__ int bs_code(int bs) {
  switch (bs) {
    case 4096: return 12;
    case 192: return 1;
    case 576: return 2;
    case 1152: return 3;
    case 2304: return 4;
    case 256: return 8;
    case 512: return 9;
    case 1024: return 10;
    case 2048: return 11;
    default: return bs <= 256 ? 6 : 7;
  }
}
__host__ __device__ inline int rate_code(int rate) {
  switch (rate) {
    case 8000: return 4;
    case 16000: return 5;
    case 22050: return 6;
    case 24000: return 7;
    case 32000: return 8;
    case 44100: return 9;
    case 48000: return 10;
    case 12000: return 12;   // + 8-bit rate in kHz
    case 11025: return 13;   // + 16-bit rate in Hz
    default: return -1;
  }
}
__device__ __forceinline__ int header_bytes(int fi, int bs, int rate) {
  const int bc = bs_code(bs), rc = rate_code(rate);
  return 4 + utf8_len((unsigned)fi) + (bc == 6 ? 1 : bc == 7 ? 2 : 0) + (rc == 12 ? 1 : rc == 13 ? 2 : 0) + 1;
}

// residual of fixed order o at sample s >= o of the block x, folded to u = e >= 0 ? 2e : -2e - 1 (< 2^20)
template <class T>
__device__ __forceinline__ unsigned fold_residual(const T* x, int s, int o) {
  int e;
  switch (o) {
    case 0: e = x[s]; break;
    case 1: e = x[s] - x[s - 1]; break;
    case 2: e = x[s] - 2 * x[s - 1] + x[s - 2]; break;
    case 3: e = x[s] - 3 * x[s - 1] + 3 * x[s - 2] - x[s - 3]; break;
    default: e = x[s] - 4 * x[s - 1] + 6 * x[s - 2] - 4 * x[s - 3] + x[s - 4]; break;
  }
  return e >= 0 ? 2u * (unsigned)e : 2u * (unsigned)(-e) - 1u;
}

__device__ __forceinline__ unsigned fold(int e) { return e >= 0 ? 2u * (unsigned)e : 2u * (unsigned)(-e) - 1u; }

// LPC residual at sample s >= p: x[s] - ((sum_j q_j x[s - j]) >> shift), the sum exact in int32 (< 2^30)
__device__ __forceinline__ int lpc_residual(const short* x, int s, int p, const int* q, int shift) {
  int acc = 0;
  for (int j = 0; j < p; j++) acc += q[j] * (int)x[s - 1 - j];
  return (int)x[s] - (acc >> shift);
}

__device__ __forceinline__ int finest_porder(int bs) { return min(kMaxPorder, __ffs(bs) - 1); }

struct LpcDesign { int valid, shift, q[kMaxLpcOrder]; };

// Levinson-Durbin and quantisation of kkx.h's "flac_lpc_order" rules 4-5 on one thread: binary64 with one rounding
// per operation (the _rn intrinsics are never contracted into a fused multiply-add), in the order the rules give.
// Every loop has compile-time bounds (guarded by p), so the arrays live in registers.
__device__ __forceinline__ LpcDesign lpc_design(const long long (&Rl)[kMaxLpcOrder + 1], int p) {
  LpcDesign out{};
  double R[kMaxLpcOrder + 1], a[kMaxLpcOrder + 1] = {};
#pragma unroll
  for (int l = 0; l <= kMaxLpcOrder; l++) R[l] = (double)Rl[l];   // |R| < 2^42: exact
  if (R[0] == 0.0) return out;
  double err = R[0];
#pragma unroll
  for (int i = 1; i <= kMaxLpcOrder; i++) {
    if (i > p) break;
    double acc = R[i];
#pragma unroll
    for (int j = 1; j < i; j++) acc = __dsub_rn(acc, __dmul_rn(a[j], R[i - j]));
    const double k = __ddiv_rn(acc, err);
    double na[kMaxLpcOrder + 1];
#pragma unroll
    for (int j = 1; j < i; j++) na[j] = __dsub_rn(a[j], __dmul_rn(k, a[i - j]));
#pragma unroll
    for (int j = 1; j < i; j++) a[j] = na[j];
    a[i] = k;
    err = __dmul_rn(err, __dsub_rn(1.0, __dmul_rn(k, k)));
    if (!(err > 0.0)) return out;
  }
  double cmax = 0.0;
#pragma unroll
  for (int j = 1; j <= kMaxLpcOrder; j++)
    if (j <= p) cmax = fmax(cmax, fabs(a[j]));
  if (cmax == 0.0) return out;
  int e;
  frexp(cmax, &e);
  const int shift = min(15, kLpcPrec - 1 - e);
  if (shift < 0) return out;
  const double scale = ldexp(1.0, shift);
  double ef = 0.0;
#pragma unroll
  for (int j = 1; j <= kMaxLpcOrder; j++) {
    if (j > p) break;
    ef = __dadd_rn(ef, __dmul_rn(a[j], scale));
    const double qd = fmin(fmax(floor(__dadd_rn(ef, 0.5)), -2048.0), 2047.0);
    out.q[j - 1] = (int)qd;
    ef = __dsub_rn(ef, qd);
  }
  out.shift = shift;
  out.valid = 1;
  return out;
}
}  // namespace

// ---------------------------------------------------------------------------------------------- analysis
// Shared: the block, then the Rice sums S[r][k][p] = sum over residual samples of finest partition p of (u >> k), one
// row r per candidate predictor: FIXED orders 0..4, and (kLpc) the frame's LPC predictor of order p as row 5.  A row
// with w warm-up samples (w = o, or p) leaves those out, so the first partition holds (bs >> q) - w residuals at every
// level.  Sums of neighbours give the coarser partition orders; all fit in 32 bits (at most 4096 samples of u < 2^20).
// kLpc = false is the encoder without "flac_lpc_order"; p is ignored there.
template <bool kLpc>
__global__ void __launch_bounds__(kThreads) flac_analyze_kernel(const short* __restrict__ pcm,
                                                                const long long* __restrict__ soff,
                                                                const int* __restrict__ foff, int B, int rate, int p,
                                                                FlacFrame* __restrict__ frames) {
  constexpr int kRows = kLpc ? kOrders + 1 : kOrders;
  extern __shared__ unsigned char fa_smem[];
  short* xs = reinterpret_cast<short*>(fa_smem);
  unsigned* S = reinterpret_cast<unsigned*>(fa_smem + kBlock * sizeof(short));          // [kRows * kRice][kParts]
  unsigned* cost = S + kRows * kRice * kParts;                                          // [r][q]
  unsigned char* kbest = reinterpret_cast<unsigned char*>(cost + kRows * (kMaxPorder + 1));  // [r][2^q - 1 + j]
  __shared__ int s_choice[3];
  __shared__ __align__(16) long long s_R[kLpc ? kThreads / 32 : 1][16];   // [warp][lag], 16-byte rows
  __shared__ LpcDesign s_lpc;

  const int f = blockIdx.x, t = threadIdx.x;
  const int b = frame_item(foff, B, f);
  const int fi = f - foff[b];
  const long long n = soff[b + 1] - soff[b];
  const long long s0 = (long long)fi * kBlock;
  const int bs = (int)min((long long)kBlock, n - s0);
  const short* xg = pcm + soff[b] + s0;
  for (int i = t; i < bs; i += kThreads) xs[i] = xg[i];
  if (!kLpc)   // (the LPC variant first uses S as the windowed block)
    for (int i = t; i < kRows * kRice * kParts; i += kThreads) S[i] = 0u;
  for (int i = t; i < kRows * (kMaxPorder + 1); i += kThreads) cost[i] = 0u;
  __syncthreads();
  const int first = xs[0];
  bool same = true;
  for (int i = t; i < bs; i += kThreads) same &= xs[i] == first;
  if (__syncthreads_and(same)) {
    if (t == 0) {
      FlacFrame& fr = frames[f];
      fr.kind = SUB_CONSTANT; fr.order = 0; fr.porder = 0;
      fr.bytes = header_bytes(fi, bs, rate) + 3 + 2;
    }
    return;
  }

  bool lpc = false;   // the frame has an LPC candidate (uniform over the CTA)
  if constexpr (kLpc) {
    if (t == 0) s_lpc.valid = 0;
    if (p < bs) {
      // window (integers only), then R[l] = sum_i xw[i] xw[i - l], exact in int64 whatever the order of the sums
      int* xw = reinterpret_cast<int*>(S);
      const int L = bs >> 2;
      for (int i = t; i < bs; i += kThreads) {
        int w = 1 << 15;
        if (i < L) w = g_lpc_window[(i * kLpcWin) / L];
        else if (i >= bs - L) w = g_lpc_window[((bs - 1 - i) * kLpcWin) / L];
        xw[i] = ((int)xs[i] * w + (1 << 14)) >> 15;
      }
      __syncthreads();
      long long r[kMaxLpcOrder + 1];
#pragma unroll
      for (int l = 0; l <= kMaxLpcOrder; l++) r[l] = 0;
      for (int i = t; i < bs; i += kThreads) {
        const int v = xw[i];
#pragma unroll
        for (int l = 0; l <= kMaxLpcOrder; l++)
          if (l <= p && i >= l) r[l] += (long long)(v * xw[i - l]);   // |xw| <= 2^15: the product fits in int32
      }
#pragma unroll
      for (int l = 0; l <= kMaxLpcOrder; l++) {
#pragma unroll
        for (int d = 16; d; d >>= 1) r[l] += __shfl_xor_sync(0xffffffffu, r[l], d);
        if ((t & 31) == 0) s_R[t >> 5][l] = r[l];
      }
      __syncthreads();
      if (t == 0) {
        long long R[kMaxLpcOrder + 1];
#pragma unroll
        for (int l = 0; l <= kMaxLpcOrder; l++) {
          R[l] = 0;
#pragma unroll
          for (int w = 0; w < kThreads / 32; w++) R[l] += s_R[w][l];
        }
        s_lpc = lpc_design(R, p);
      }
    }
    for (int i = t; i < kRows * kRice * kParts; i += kThreads) S[i] = 0u;
    __syncthreads();
    lpc = s_lpc.valid != 0;
  }

  const int qmax = finest_porder(bs);
  const int pf = bs >> qmax;                 // finest partition size
  bool wide = false;                         // an LPC residual folds to u >= 2^20: no LPC candidate
  {
    int lq[kLpc ? kMaxLpcOrder : 1];
    int lshift = 0;
    if constexpr (kLpc) {
#pragma unroll
      for (int j = 0; j < kMaxLpcOrder; j++) lq[j] = j < p ? s_lpc.q[j] : 0;
      lshift = s_lpc.shift;
    }
    unsigned acc[kRows][kRice];
#pragma unroll
    for (int o = 0; o < kRows; o++)
#pragma unroll
      for (int k = 0; k < kRice; k++) acc[o][k] = 0u;
    const int c0 = t * kPer, c1 = min(c0 + kPer, bs);
    int pt = c0 / pf;
    for (int s = c0; s < c1; s++) {
      const int ps = s / pf;
      if (ps != pt) {   // flush the previous partition's share (integer adds: the order of arrival does not matter)
#pragma unroll
        for (int o = 0; o < kRows; o++)
#pragma unroll
          for (int k = 0; k < kRice; k++) {
            if (acc[o][k]) atomicAdd(&S[(o * kRice + k) * kParts + pt], acc[o][k]);
            acc[o][k] = 0u;
          }
        pt = ps;
      }
#pragma unroll
      for (int o = 0; o < kOrders; o++) {
        if (s >= o) {
          const unsigned u = fold_residual(xs, s, o);
#pragma unroll
          for (int k = 0; k < kRice; k++) acc[o][k] += u >> k;
        }
      }
      if constexpr (kLpc) {
        if (lpc && s >= p) {
          int a = 0;
#pragma unroll
          for (int j = 0; j < kMaxLpcOrder; j++)
            if (j < p) a += lq[j] * (int)xs[s - 1 - j];
          const unsigned u = fold((int)xs[s] - (a >> lshift));
          wide |= u >= (1u << 20);
#pragma unroll
          for (int k = 0; k < kRice; k++) acc[kOrders][k] += u >> k;
        }
      }
    }
    if (c0 < c1) {
#pragma unroll
      for (int o = 0; o < kRows; o++)
#pragma unroll
        for (int k = 0; k < kRice; k++)
          if (acc[o][k]) atomicAdd(&S[(o * kRice + k) * kParts + pt], acc[o][k]);
    }
  }
  if constexpr (kLpc) {
    if (__syncthreads_or(wide)) lpc = false;
  } else {
    __syncthreads();
  }

  // from the finest level up: per partition the cheapest k (ties: smaller k), then merge neighbours in place.  The
  // sum of level q's partition j sits at index j << (qmax - q).
  for (int q = qmax; q >= 0; q--) {
    const int np = 1 << q, psize = bs >> q, sh = qmax - q;
#pragma unroll
    for (int o = 0; o < kRows; o++) {
      const int warm = o < kOrders ? o : p;
      // the cheapest k of a partition costs at most n_part (2^20 >> 14) + 15 n_part bits, so a level's total fits in
      // 32 bits; one atomic per warp (the 64-bit shared atomic is a compare-and-swap loop)
      unsigned part = 0u;
      if (psize > warm && (o < kOrders || lpc)) {
        for (int j = t; j < np; j += kThreads) {
          const long long cnt = psize - (j == 0 ? warm : 0);
          unsigned long long best = ~0ull;
          int kb = 0;
          for (int k = 0; k < kRice; k++) {
            const unsigned long long c = (unsigned long long)S[(o * kRice + k) * kParts + (j << sh)] + cnt * (k + 1);
            if (c < best) { best = c; kb = k; }
          }
          kbest[o * (2 * kParts - 1) + (np - 1) + j] = (unsigned char)kb;
          part += 4u + (unsigned)best;
        }
      }
      part = __reduce_add_sync(0xffffffffu, part);
      if ((t & 31) == 0 && part) atomicAdd(&cost[o * (kMaxPorder + 1) + q], part);
    }
    __syncthreads();
    if (q > 0) {
      const int nh = np >> 1;
      for (int w = t; w < kRows * kRice * nh; w += kThreads) {
        const int ok = w / nh, j = w - ok * nh;
        S[ok * kParts + ((2 * j) << sh)] += S[ok * kParts + ((2 * j + 1) << sh)];
      }
      __syncthreads();
    }
  }

  if (t == 0) {
    unsigned long long best = ~0ull;
    int bo = 0, bq = 0;
    for (int o = 0; o < kOrders; o++)
      for (int q = 0; q <= qmax; q++) {
        if ((bs >> q) <= o) continue;
        const unsigned long long c = 8ull + 16ull * o + 6ull + cost[o * (kMaxPorder + 1) + q];
        if (c < best) { best = c; bo = o; bq = q; }
      }
    int kind = SUB_FIXED;
    if (kLpc && lpc) {   // the cheapest partition order of the LPC predictor; it replaces FIXED only when cheaper
      unsigned long long lbest = ~0ull;
      int lq = 0;
      for (int q = 0; q <= qmax; q++) {
        if ((bs >> q) <= p) continue;
        const unsigned long long c = 8ull + 16ull * p + 4 + 5 + 12ull * p + 6 + cost[kOrders * (kMaxPorder + 1) + q];
        if (c < lbest) { lbest = c; lq = q; }
      }
      if (lbest < best) { best = lbest; kind = SUB_LPC; bo = p; bq = lq; }
    }
    const unsigned long long verbatim = 8ull + 16ull * bs;
    if (verbatim < best) kind = SUB_VERBATIM;
    const unsigned long long bits = kind == SUB_VERBATIM ? verbatim : best;
    FlacFrame& fr = frames[f];
    fr.kind = kind; fr.order = bo; fr.porder = bq;
    fr.bytes = header_bytes(fi, bs, rate) + (int)((bits + 7) / 8) + 2;
    if (kLpc && kind == SUB_LPC) fr.shift = s_lpc.shift;
    s_choice[0] = kind; s_choice[1] = bo; s_choice[2] = bq;
  }
  __syncthreads();
  if (s_choice[0] == SUB_FIXED || s_choice[0] == SUB_LPC) {
    const int row = s_choice[0] == SUB_LPC ? kOrders : s_choice[1], np = 1 << s_choice[2];
    for (int j = t; j < np; j += kThreads) frames[f].k[j] = kbest[row * (2 * kParts - 1) + (np - 1) + j];
  }
  // one coefficient per thread, plain 16-bit stores.  (A thread-0 loop over j < p was compiled, CUDA 12.9 for
  // sm_100a, into paired 32-bit stores whose upper half came from the wrong register: flac_pack then rebuilt other
  // residuals than the ones costed here.)
  if (kLpc && s_choice[0] == SUB_LPC && t < p) frames[f].q[t] = (short)s_lpc.q[t];
}

// ---------------------------------------------------------------------------------------------- offsets
// Frame f of item b starts at 42 (b + 1) + (bytes of all frames before f); item b at that of its first frame - 42.
__global__ void __launch_bounds__(1024) flac_scan_kernel(const FlacFrame* __restrict__ frames,
                                                         const int* __restrict__ foff, int B, int F,
                                                         long long* __restrict__ frame_off,
                                                         long long* __restrict__ item_off) {
  __shared__ long long warp_sum[32];
  __shared__ long long carry;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  if (t == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < F; base += 1024) {
    const int f = base + t;
    const long long v = f < F ? frames[f].bytes : 0;
    long long x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const long long y = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warp_sum[wid] = x;
    __syncthreads();
    if (wid == 0) {
      long long w = warp_sum[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += y;
      }
      warp_sum[lane] = w;
    }
    __syncthreads();
    const long long excl = carry + (wid ? warp_sum[wid - 1] : 0) + x - v;
    if (f < F) {
      const int b = frame_item(foff, B, f);
      frame_off[f] = excl + (long long)kHead * (b + 1);
      if (f == foff[b]) item_off[b] = excl + (long long)kHead * b;
    }
    __syncthreads();
    if (t == 1023) carry = excl + v;
    __syncthreads();
  }
  if (t == 0) item_off[B] = carry + (long long)kHead * B;
}

// ---------------------------------------------------------------------------------------------- packing
// CRC-16 (poly 0x8005, init 0, unreflected, no final xor) is linear: crc(A || B) = crc(A) * x^(8 |B|) ^ crc(B).
__device__ __forceinline__ unsigned crc16_mulmod(unsigned a, unsigned b) {   // a * b mod (x^16 + 0x8005)
  unsigned r = 0;
  for (int i = 15; i >= 0; i--) {
    r = (r << 1) ^ ((r & 0x8000u) ? 0x18005u : 0u);
    if ((b >> i) & 1u) r ^= a;
  }
  return r & 0xFFFFu;
}
struct Crc16Pow { unsigned v[15]; };   // v[i] = x^(8 * 2^i) mod P: frames are shorter than 2^15 bytes
constexpr Crc16Pow crc16_pows() {
  Crc16Pow t{};
  unsigned p = 0x100u;   // x^8
  for (int i = 0; i < 15; i++) {
    t.v[i] = p;
    unsigned r = 0;      // p * p mod P
    for (int b = 15; b >= 0; b--) {
      r = ((r << 1) ^ ((r & 0x8000u) ? 0x18005u : 0u)) & 0x1FFFFu;
      if ((p >> b) & 1u) r ^= p;
    }
    p = r & 0xFFFFu;
  }
  return t;
}
__constant__ Crc16Pow kCrc16Pow = crc16_pows();
__device__ __forceinline__ unsigned crc16_shift(unsigned c, int nbytes) {    // c * x^(8 nbytes) mod P
  for (int i = 0; nbytes; i++, nbytes >>= 1)
    if (nbytes & 1) c = crc16_mulmod(c, kCrc16Pow.v[i]);
  return c;
}

__global__ void __launch_bounds__(kThreads) flac_pack_kernel(const short* __restrict__ pcm,
                                                             const long long* __restrict__ soff,
                                                             const int* __restrict__ foff, int B, int rate,
                                                             const FlacFrame* __restrict__ frames,
                                                             const long long* __restrict__ frame_off,
                                                             unsigned char* __restrict__ out) {
  constexpr int kWords = (16 + 1 + 2 * kBlock + 2) / 4 + 2;
  __shared__ short xs[kBlock];
  __shared__ unsigned bits[kWords];
  __shared__ unsigned short crc_tab[256];
  __shared__ unsigned char ks[kParts];
  __shared__ int lq[kMaxLpcOrder];
  __shared__ int warp_sum[kThreads / 32];
  __shared__ unsigned s_crc;
  __shared__ int s_hdr;

  const int f = blockIdx.x, t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int b = frame_item(foff, B, f);
  const int fi = f - foff[b];
  const long long n = soff[b + 1] - soff[b];
  const long long s0 = (long long)fi * kBlock;
  const int bs = (int)min((long long)kBlock, n - s0);
  const FlacFrame& fr = frames[f];
  const int nbytes = fr.bytes, kind = fr.kind, o = fr.order, q = fr.porder;
  const bool lpc = kind == SUB_LPC;
  const int shift = lpc ? fr.shift : 0;
  const short* xg = pcm + soff[b] + s0;
  for (int i = t; i < bs; i += kThreads) xs[i] = xg[i];
  for (int i = t; i < kWords; i += kThreads) bits[i] = 0u;
  for (int i = t; i < kParts; i += kThreads) ks[i] = (kind == SUB_FIXED || lpc) && i < (1 << q) ? fr.k[i] : 0;
  if (lpc && t < o) lq[t] = fr.q[t];
  {
    unsigned c = (unsigned)t << 8;
    for (int i = 0; i < 8; i++) c = (c << 1) ^ ((c & 0x8000u) ? 0x8005u : 0u);
    crc_tab[t] = (unsigned short)c;
  }
  if (t == 0) s_crc = 0u;
  __syncthreads();

  if (t == 0) {   // frame header + its CRC-8 (poly 0x07, init 0)
    unsigned char h[16];
    int m = 0;
    const int bc = bs_code(bs), rc = rate_code(rate);
    h[m++] = 0xFF; h[m++] = 0xF8;
    h[m++] = (unsigned char)((bc << 4) | rc);
    h[m++] = 0x08;                                    // mono, 16 bits
    const unsigned v = (unsigned)fi;
    const int ul = utf8_len(v);
    if (ul == 1) {
      h[m++] = (unsigned char)v;
    } else {
      h[m++] = (unsigned char)((0xFF00u >> ul) | (v >> (6 * (ul - 1))));
      for (int i = ul - 2; i >= 0; i--) h[m++] = (unsigned char)(0x80u | ((v >> (6 * i)) & 0x3Fu));
    }
    if (bc == 6) h[m++] = (unsigned char)(bs - 1);
    if (bc == 7) { h[m++] = (unsigned char)((bs - 1) >> 8); h[m++] = (unsigned char)(bs - 1); }
    if (rc == 12) h[m++] = (unsigned char)(rate / 1000);
    if (rc == 13) { h[m++] = (unsigned char)(rate >> 8); h[m++] = (unsigned char)rate; }
    unsigned crc = 0;
    for (int i = 0; i < m; i++) {
      crc ^= h[i];
      for (int j = 0; j < 8; j++) crc = ((crc << 1) ^ ((crc & 0x80u) ? 0x07u : 0u)) & 0xFFu;
    }
    h[m++] = (unsigned char)crc;
    for (int i = 0; i < m; i++) put_bits(bits, 8 * i, h[i], 8);
    s_hdr = m;
  }
  __syncthreads();
  const int sub = 8 * s_hdr;   // first bit of the subframe

  if (kind == SUB_CONSTANT) {
    if (t == 0) { put_bits(bits, sub, 0x00u, 8); put_bits(bits, sub + 8, (unsigned short)xs[0], 16); }
  } else if (kind == SUB_VERBATIM) {
    if (t == 0) put_bits(bits, sub, 0x02u, 8);
    for (int s = t; s < bs; s += kThreads) put_bits(bits, sub + 8 + 16 * s, (unsigned short)xs[s], 16);
  } else {
    // element s: a warm-up sample (16 bits) for s < o; else [if s == o: (LPC: precision - 1 (4 bits), shift
    // (5 bits), o coefficients (12 bits each)) method + partition order (6 bits)] [Rice parameter (4 bits) if s starts
    // a partition] then the code: (u >> k) zeros, a one, the low k bits
    const int psize = bs >> q;
    const int c0 = t * kPer, c1 = min(c0 + kPer, bs);
    const int head = lpc ? 4 + 5 + kLpcPrec * o : 0;
    auto residual = [&](int s) { return lpc ? fold(lpc_residual(xs, s, o, lq, shift)) : fold_residual(xs, s, o); };
    int len = 0;
    for (int s = c0; s < c1; s++) {
      if (s < o) { len += 16; continue; }
      const int k = ks[s / psize];
      len += (int)(residual(s) >> k) + 1 + k + (s == o ? head + 10 : (s % psize == 0 ? 4 : 0));
    }
    int x = len;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, d);
      if (lane >= d) x += y;
    }
    if (lane == 31) warp_sum[wid] = x;
    __syncthreads();
    if (wid == 0) {
      int w = lane < kThreads / 32 ? warp_sum[lane] : 0;
#pragma unroll
      for (int d = 1; d < kThreads / 32; d <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, w, d);
        if (lane >= d) w += y;
      }
      if (lane < kThreads / 32) warp_sum[lane] = w;
    }
    __syncthreads();
    int pos = sub + 8 + (wid ? warp_sum[wid - 1] : 0) + x - len;
    if (t == 0) put_bits(bits, sub, lpc ? 0x40u | (unsigned)((o - 1) << 1) : 0x10u | (unsigned)(o << 1), 8);
    for (int s = c0; s < c1; s++) {
      if (s < o) { put_bits(bits, pos, (unsigned short)xs[s], 16); pos += 16; continue; }
      const int k = ks[s / psize];
      if (s == o && lpc) {
        put_bits(bits, pos, kLpcPrec - 1, 4);
        put_bits(bits, pos + 4, (unsigned)shift, 5);
        pos += 9;
        for (int j = 0; j < o; j++, pos += kLpcPrec) put_bits(bits, pos, (unsigned)lq[j] & 0xFFFu, kLpcPrec);
      }
      if (s == o) { put_bits(bits, pos, (unsigned)q, 6); pos += 6; }
      if (s == o || s % psize == 0) { put_bits(bits, pos, (unsigned)k, 4); pos += 4; }
      const unsigned u = residual(s);
      pos += (int)(u >> k);
      put_bits(bits, pos, (1u << k) | (u & ((1u << k) - 1u)), k + 1);
      pos += k + 1;
    }
  }
  __syncthreads();

  // CRC-16 of bytes [0, nbytes - 2): per-thread chunks with the table, shifted past the bytes after them and XOR-ed
  {
    const int m = nbytes - 2, chunk = (m + kThreads - 1) / kThreads;
    const int i0 = min(m, t * chunk), i1 = min(m, i0 + chunk);
    unsigned c = 0;
    for (int i = i0; i < i1; i++) c = ((c << 8) ^ crc_tab[((c >> 8) ^ get_byte(bits, i)) & 0xFFu]) & 0xFFFFu;
    if (i1 > i0) c = crc16_shift(c, m - i1);
#pragma unroll
    for (int d = 16; d; d >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, d);
    if (lane == 0 && c) atomicXor(&s_crc, c);
    __syncthreads();
    if (t == 0) put_bits(bits, 8 * m, s_crc, 16);
    __syncthreads();
  }
  unsigned char* dst = out + frame_off[f];
  for (int i = t; i < nbytes; i += kThreads) dst[i] = (unsigned char)get_byte(bits, i);

  if (fi == 0) {   // the item's head: fLaC, last-block flag + STREAMINFO (type 0, 34 bytes)
    int mn = 0x7FFFFFFF, mx = 0;
    for (int g = foff[b] + t; g < foff[b + 1]; g += kThreads) { mn = min(mn, frames[g].bytes); mx = max(mx, frames[g].bytes); }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
      mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, d));
      mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    }
    __syncthreads();
    if (lane == 0) { warp_sum[wid] = mn; }
    __syncthreads();
    if (t == 0) for (int w = 1; w < kThreads / 32; w++) mn = min(mn, warp_sum[w]);
    __syncthreads();
    if (lane == 0) { warp_sum[wid] = mx; }
    __syncthreads();
    if (t == 0) {
      for (int w = 1; w < kThreads / 32; w++) mx = max(mx, warp_sum[w]);
      unsigned char* h = out + frame_off[f] - kHead;
      const unsigned char lead[8] = {'f', 'L', 'a', 'C', 0x80, 0, 0, 34};
      for (int i = 0; i < 8; i++) h[i] = lead[i];
      h[8] = kBlock >> 8; h[9] = kBlock & 0xFF; h[10] = kBlock >> 8; h[11] = kBlock & 0xFF;
      h[12] = (unsigned char)(mn >> 16); h[13] = (unsigned char)(mn >> 8); h[14] = (unsigned char)mn;
      h[15] = (unsigned char)(mx >> 16); h[16] = (unsigned char)(mx >> 8); h[17] = (unsigned char)mx;
      // 20-bit rate, 3-bit channels - 1 (0), 5-bit bits per sample - 1 (15), 36-bit total samples
      const unsigned long long v = ((unsigned long long)rate << 44) | (15ull << 36) | ((unsigned long long)n & 0xFFFFFFFFFull);
      for (int i = 0; i < 8; i++) h[18 + i] = (unsigned char)(v >> (56 - 8 * i));
      for (int i = 0; i < 16; i++) h[26 + i] = 0;   // MD5 zero: "not computed"
    }
  }
}

// ---------------------------------------------------------------------------------------------- host side
long long flac_frames(long long n) { return (n + kBlock - 1) / kBlock; }

long long flac_bound(long long n_items, long long n_frames, long long n_samples) {
  return kHead * n_items + (16 + 1 + 2) * n_frames + 2 * n_samples;
}

size_t flac_work_bytes(long long n_frames) {
  return (size_t)n_frames * (sizeof(FlacFrame) + sizeof(long long)) + 256;
}

bool flac_rate_ok(int rate) { return rate_code(rate) >= 0; }

void flac_lpc_window(int* m) {
  const double pi = 3.14159265358979323846;
  for (int k = 0; k < kLpcWin; k++)
    m[k] = (int)std::floor(32768.0 * (0.5 * (1.0 - std::cos(pi * (k + 0.5) / kLpcWin))) + 0.5);
}

static size_t analyze_smem(int rows) {
  return kBlock * sizeof(short) + (size_t)rows * kRice * kParts * sizeof(unsigned) +
         rows * (kMaxPorder + 1) * sizeof(unsigned) + rows * (2 * kParts - 1);
}

void launch_flac(const short* pcm, const long long* soff, const int* foff, int B, int F, int rate, int lpc_order,
                 void* work, unsigned char* out, long long* item_off, cudaStream_t st) {
  if (g_dry_run) return;
  if (!flac_rate_ok(rate)) throw ArgError("launch_flac: no FLAC sample-rate code for " + std::to_string(rate) + " Hz");
  if (B < 1 || F < B) throw ArgError("launch_flac: every item needs at least one sample");
  if (lpc_order < 0 || lpc_order > kMaxLpcOrder) throw ArgError("launch_flac: LPC order outside 0..12");
  FlacFrame* frames = static_cast<FlacFrame*>(work);
  long long* frame_off = reinterpret_cast<long long*>(reinterpret_cast<char*>(work) +
                                                      (((size_t)F * sizeof(FlacFrame) + 255) & ~size_t(255)));
  if (lpc_order == 0) {
    const size_t smem = analyze_smem(kOrders);
    prepare_smem_launch<flac_analyze_kernel<false>>((int)smem);
    flac_analyze_kernel<false><<<F, kThreads, smem, st>>>(pcm, soff, foff, B, rate, 0, frames);
  } else {
    static DevOnce once;
    const int dev = prepare_smem_launch<flac_analyze_kernel<true>>((int)analyze_smem(kOrders + 1));
    once.run(dev, [] {
      int m[kLpcWin];
      flac_lpc_window(m);
      KKX_CUDA(cudaMemcpyToSymbol(g_lpc_window, m, sizeof m));
    });
    const size_t smem = analyze_smem(kOrders + 1);
    flac_analyze_kernel<true><<<F, kThreads, smem, st>>>(pcm, soff, foff, B, rate, lpc_order, frames);
  }
  post_launch("flac_analyze", st);
  flac_scan_kernel<<<1, 1024, 0, st>>>(frames, foff, B, F, frame_off, item_off);
  post_launch("flac_scan", st);
  flac_pack_kernel<<<F, kThreads, 0, st>>>(pcm, soff, foff, B, rate, frames, frame_off, out);
  post_launch("flac_pack", st);
}

}  // namespace kkx
