// kernels_mp3.cu -- constant-bitrate MPEG audio Layer III of 16-bit mono PCM on the device (kkx_infer_batch_mp3,
// kkx.h).
//
// There is no bit reservoir, so every frame stands alone and its byte offset follows from its index in closed form
// (kernels.h Mp3Format).  One launch, one CTA per frame and 128 threads per granule (one or two granules a frame):
//   1. stage the frame's input plus its halo -- the previous granule (the MDCT overlap) and 480 samples before it
//      (the reach of the 512-tap window) -- so a frame shares no state with its neighbours;
//   2. polyphase analysis (ISO 11172-3 window C[i], 64 x 32 matrixing), the 18-point MDCT of block type 0 with the
//      sine window, the eight alias-reduction butterflies per subband boundary;
//   3. per granule, the global gain by the binary search of kkx.h: quantise, split into big_values / count1 / zero
//      regions, cost every Huffman table that covers the largest value (integer sums), fit against the bit budget;
//   4. per granule, code lengths -> a block prefix sum -> codes OR-ed into the frame's shared bit buffer, which the
//      CTA then stores at the frame's offset together with its header and side information.
// Nothing depends on the launch shape or the batch: the frame's bytes are a function of its item's samples.
#include "kernels.h"
#include "bitpack.cuh"
#include "mp3_tables.h"
#include <cmath>

namespace kkx {

namespace {
constexpr int kGr = 576;                       // samples per granule
constexpr int kGroup = 128;                    // threads per granule
constexpr int kIxMax = 15 + (1 << 13) - 1;     // 8206: the largest value linbits = 13 can carry
constexpr int kRegion0 = 7, kRegion1 = 7;      // region0_count / region1_count: every region uses one table, so the
                                               // split is immaterial
constexpr int kMaxFrame = 1441;                // bytes: 144000 * 320 / 32000 + 1 = 72000 * 160 / 8000 + 1
constexpr int kBitWords = (kMaxFrame + 3) / 4 + 2;
constexpr int kMaxSlots = 18 * 3;              // subband slots of a two-granule frame and its halo granule
constexpr int kMaxIn = kGr * 3 + 480;          // input samples of the same
// analysis constants (mp3_consts): window C [512], matrixing M [64][32] (k fastest), windowed MDCT W [18][36],
// butterflies cs [8], ca [8]
constexpr int kOffC = 0, kOffM = 512, kOffW = kOffM + 64 * 32, kOffCs = kOffW + 18 * 36, kOffCa = kOffCs + 8;
constexpr int kConsts = kOffCa + 8;
constexpr int kCand = 15;                      // candidate big_values tables: 1 2 3 5 .. 13 15, one of 16..23, one of 24..31
constexpr int kCounters = kCand + 3;           // + count1 A, count1 B, sign bits

__device__ const mp3tab::Tables kTab = mp3tab::kTables;

struct Granule {
  int gg, big, end, table, c1, bits, fits;     // big / end: first element of count1 / of the zero region
};

__device__ __forceinline__ int cand_table(int c, int t16, int t24) {
  constexpr int fixed[13] = {1, 2, 3, 5, 6, 7, 8, 9, 10, 11, 12, 13, 15};
  return c < 13 ? fixed[c] : c == 13 ? t16 : t24;
}

// the smallest linbits table of 16..23 / 24..31 whose range covers m (the last one when none does)
__device__ __forceinline__ int escape_table(int first, int m) {
  for (int t = first; t < first + 7; t++)
    if (15 + (1 << kTab.info[t].linbits) - 1 >= m) return t;
  return first + 7;
}

__device__ __forceinline__ int pair_bits(const unsigned char* hlen, int table, int x, int y) {
  if (table == 0) return 0;
  const mp3tab::HuffInfo in = kTab.info[table];
  const int lin = in.linbits;
  const int xc = min(x, 15), yc = min(y, 15);
  return hlen[in.base + xc * in.xlen + yc] + (lin && x >= 15 ? lin : 0) + (lin && y >= 15 ? lin : 0) + (x != 0) +
         (y != 0);
}

// One evaluation of global gain gg for the granule of this thread's group (lt = thread in the group).  Every thread
// of the CTA calls it in lockstep (three __syncthreads); the result is in *g.
__device__ void evaluate(int gg, const float* xa, int* ix, int lt, int* red, int* cnt, Granule* g, int budget,
                         const unsigned char* hlen) {
  const int lane = lt & 31, w = lt >> 5;
  const float q = exp2f(-0.1875f * (float)(gg - 210));
  int mx = 0, lastnz = -1, lastbig = -1, firstnz = kGr;
  for (int i = lt; i < kGr; i += kGroup) {
    const float v = fminf(xa[i] * q, 1e6f);
    const int v_ix = (int)floorf(v - 0.0946f + 0.5f);
    ix[i] = v_ix;
    mx = max(mx, v_ix);
    if (v_ix) { lastnz = i; firstnz = min(firstnz, i); }
    if (v_ix > 1) lastbig = i;
  }
  mx = __reduce_max_sync(0xffffffffu, mx);
  lastnz = __reduce_max_sync(0xffffffffu, lastnz);
  lastbig = __reduce_max_sync(0xffffffffu, lastbig);
  firstnz = __reduce_min_sync(0xffffffffu, firstnz);
  if (lane == 0) { red[4 * w] = mx; red[4 * w + 1] = lastnz; red[4 * w + 2] = lastbig; red[4 * w + 3] = firstnz; }
  if (lt < kCounters) cnt[lt] = 0;
  __syncthreads();
  mx = red[0]; lastnz = red[1]; lastbig = red[2]; firstnz = red[3];
  for (int k = 1; k < kGroup / 32; k++) {
    mx = max(mx, red[4 * k]); lastnz = max(lastnz, red[4 * k + 1]);
    lastbig = max(lastbig, red[4 * k + 2]); firstnz = min(firstnz, red[4 * k + 3]);
  }
  const int end = (lastnz + 2) & ~1;                        // trailing zero pairs stripped
  const int big = end - 4 * ((end - lastbig - 1) >> 2);     // quadruples of values <= 1 from the top down
  const int mbig = mx > 1 ? mx : (firstnz < big ? 1 : 0);   // the largest value below `big`
  const int t16 = escape_table(16, mbig), t24 = escape_table(24, mbig);
  int c[kCounters];
#pragma unroll
  for (int k = 0; k < kCounters; k++) c[k] = 0;
  for (int p = lt; 2 * p < big; p += kGroup) {
    const int x = ix[2 * p], y = ix[2 * p + 1];
    const int xc = min(x, 15), yc = min(y, 15);
    c[kCand + 2] += (x != 0) + (y != 0);
#pragma unroll
    for (int k = 0; k < kCand; k++) {
      const mp3tab::HuffInfo in = kTab.info[cand_table(k, t16, t24)];
      if (in.linbits)
        c[k] += hlen[in.base + xc * 16 + yc] + (x >= 15 ? in.linbits : 0) + (y >= 15 ? in.linbits : 0);
      else if (in.xlen > mbig)
        c[k] += hlen[in.base + x * in.xlen + y];
    }
  }
  for (int e = big + 4 * lt; e < end; e += 4 * kGroup) {
    const int v = ix[e], x1 = ix[e + 1], x2 = ix[e + 2], x3 = ix[e + 3];
    c[kCand] += kTab.qlen[0][8 * v + 4 * x1 + 2 * x2 + x3];
    c[kCand + 1] += 4;
    c[kCand + 2] += v + x1 + x2 + x3;
  }
#pragma unroll
  for (int k = 0; k < kCounters; k++) {
    const int s = __reduce_add_sync(0xffffffffu, c[k]);
    if (lane == 0 && s) atomicAdd(cnt + k, s);          // integer sums: the order of arrival does not matter
  }
  __syncthreads();
  if (lt == 0) {
    int table = 0, best = 0;
    if (mbig > 0) {
      best = 0x7FFFFFFF;
      for (int k = 0; k < kCand; k++) {                   // ascending table numbers: ties keep the lowest
        const int t = cand_table(k, t16, t24);
        const mp3tab::HuffInfo in = kTab.info[t];
        const bool covers = in.linbits ? 15 + (1 << in.linbits) - 1 >= mbig : in.xlen > mbig;
        if (covers && cnt[k] < best) { best = cnt[k]; table = t; }
      }
    }
    if (best == 0x7FFFFFFF) best = 0;   // no table covers the largest value: ix > 8206, which does not fit anyway
    const int c1 = cnt[kCand + 1] < cnt[kCand] ? 1 : 0;
    const int bits = best + min(cnt[kCand], cnt[kCand + 1]) + cnt[kCand + 2];
    *g = Granule{gg, big, end, table, c1, bits, mx <= kIxMax && bits <= budget ? 1 : 0};
  }
  __syncthreads();
}

__global__ void __launch_bounds__(2 * kGroup) mp3_encode_kernel(const short* __restrict__ pcm,
                                                                const long long* __restrict__ soff,
                                                                const int* __restrict__ foff,
                                                                const long long* __restrict__ boff, int B,
                                                                Mp3Format fmt, const float* __restrict__ consts,
                                                                unsigned char* __restrict__ out) {
  extern __shared__ float mp3_smem[];
  float* xin = mp3_smem;                 // [kMaxIn] input of the frame and its halo
  float* Y = xin + kMaxIn;               // [slots][64] windowed sums; then xr, |xr|^(3/4), ix of each granule
  float* S = Y + kMaxSlots * 64;         // [slots][32] subband samples
  float* cst = S + kMaxSlots * 32;       // [kConsts]
  unsigned* bits = reinterpret_cast<unsigned*>(cst + kConsts);                  // [kBitWords]
  unsigned char* hlen = reinterpret_cast<unsigned char*>(bits + kBitWords);     // [kHuffEntries]
  __shared__ int red[2][4 * (kGroup / 32)];
  __shared__ int cnt[2][kCounters];
  __shared__ int scan[2][kGroup / 32];
  __shared__ Granule gs[2];

  const int ngr = fmt.ngr, nthr = ngr * kGroup, t = threadIdx.x;
  const int nslot = 18 * (ngr + 1), nin = kGr * (ngr + 1) + 480;
  const int f = blockIdx.x;
  const int b = frame_item(foff, B, f);
  const long long fl = f - foff[b];
  const long long n = soff[b + 1] - soff[b];
  const short* x = pcm + soff[b];
  const long long t0 = (long long)kGr * (fl * ngr - 1) - 480;   // sample of xin[0]
  for (int i = t; i < nin; i += nthr) {
    const long long s = t0 + i;
    xin[i] = s >= 0 && s < n ? (float)x[s] * (1.f / 32768.f) : 0.f;
  }
  for (int i = t; i < kConsts; i += nthr) cst[i] = consts[i];
  for (int i = t; i < kBitWords; i += nthr) bits[i] = 0u;
  for (int i = t; i < mp3tab::kHuffEntries; i += nthr) hlen[i] = kTab.len[i];
  __syncthreads();

  // polyphase analysis: slot s sees the 512 samples ending at xin[32 s + 511]
  for (int idx = t; idx < nslot * 64; idx += nthr) {
    const int s = idx >> 6, i = idx & 63;
    const float* xs = xin + 32 * s + 511 - i;
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < 8; j++) acc = fmaf(cst[kOffC + i + 64 * j], xs[-64 * j], acc);
    Y[idx] = acc;
  }
  __syncthreads();
  for (int idx = t; idx < nslot * 32; idx += nthr) {
    const int s = idx >> 5, k = idx & 31;
    const float* ys = Y + 64 * s;
    float acc = 0.f;
#pragma unroll 16
    for (int i = 0; i < 64; i++) acc = fmaf(cst[kOffM + 32 * i + k], ys[i], acc);
    S[idx] = (s & 1) && (k & 1) ? -acc : acc;        // frequency inversion of the odd subbands
  }
  __syncthreads();
  float* xr = Y;                         // [ngr][576]
  float* xa = Y + 2 * kGr;               // [ngr][576]
  int* ix = reinterpret_cast<int*>(Y + 4 * kGr);   // [ngr][576]
  for (int idx = t; idx < ngr * kGr; idx += nthr) {  // MDCT of granule j over slots 18 j .. 18 j + 35
    const int k = idx & 31, r = idx >> 5, m = r % 18, j = r / 18;
    const float* ss = S + 18 * j * 32 + k;
    const float* wm = cst + kOffW + 36 * m;
    float acc = 0.f;
#pragma unroll 12
    for (int i = 0; i < 36; i++) acc = fmaf(wm[i], ss[32 * i], acc);
    xr[j * kGr + 18 * k + m] = acc;
  }
  __syncthreads();
  for (int idx = t; idx < ngr * 31 * 8; idx += nthr) {
    const int j = idx / 248, r = idx - 248 * j, sb = 1 + (r >> 3), i = r & 7;
    float* g = xr + j * kGr;
    const float bu = g[18 * sb - 1 - i], bd = g[18 * sb + i];
    const float cs = cst[kOffCs + i], ca = cst[kOffCa + i];
    g[18 * sb - 1 - i] = fmaf(bu, cs, bd * ca);
    g[18 * sb + i] = fmaf(bd, cs, -bu * ca);
  }
  __syncthreads();
  for (int idx = t; idx < ngr * kGr; idx += nthr) xa[idx] = powf(fabsf(xr[idx]), 0.75f);

  // the frame's length and each granule's bit budget
  const long long fb0 = fl * fmt.anum / fmt.rate, fb1 = (fl + 1) * fmt.anum / fmt.rate;
  const int len = (int)(fb1 - fb0), pad = (int)(len - fmt.anum / fmt.rate);
  const int main_bits = 8 * (len - 4 - fmt.side);
  const int grp = t / kGroup, lt = t - grp * kGroup;
  const int share = ngr == 2 ? (grp == 0 ? main_bits / 2 : main_bits - main_bits / 2) : main_bits;
  const int budget = min(4095, share);
  const float* gxa = xa + grp * kGr;
  int* gix = ix + grp * kGr;
  __syncthreads();
  int lo = 0, hi = 255;
  while (lo < hi) {          // always eight steps, so the two granules of a frame stay in lockstep
    const int mid = (lo + hi) >> 1;
    evaluate(mid, gxa, gix, lt, red[grp], cnt[grp], &gs[grp], budget, hlen);
    if (gs[grp].fits) hi = mid; else lo = mid + 1;
  }
  evaluate(lo, gxa, gix, lt, red[grp], cnt[grp], &gs[grp], budget, hlen);

  if (t == 0) {   // header and side information
    const unsigned h = 0xFFE00000u | (unsigned)fmt.version << 19 | 1u << 17 | 1u << 16 | (unsigned)fmt.br_index << 12 |
                       (unsigned)fmt.sr_index << 10 | (unsigned)pad << 9 | 3u << 6;
    put_bits(bits, 0, h, 32);
    int pos = 32;
    auto put = [&](unsigned v, int nb) { put_bits(bits, pos, v, nb); pos += nb; };
    put(0, ngr == 2 ? 9 + 5 + 4 : 8 + 1);     // main_data_begin, private bits, scfsi
    for (int j = 0; j < ngr; j++) {
      const Granule& g = gs[j];
      put((unsigned)g.bits, 12);
      put((unsigned)(g.big >> 1), 9);
      put((unsigned)g.gg, 8);
      put(0, ngr == 2 ? 4 : 9);               // scalefac_compress
      put(0, 1);                              // window_switching_flag
      for (int r = 0; r < 3; r++) put((unsigned)g.table, 5);
      put(kRegion0, 4);
      put(kRegion1, 3);
      put(0, ngr == 2 ? 2 : 1);               // (preflag,) scalefac_scale
      put((unsigned)g.c1, 1);
    }
  }

  // the granule's codes: elements 0..287 are the big_values pairs, 288.. the count1 quadruples; thread lt owns
  // elements [4 lt, 4 lt + 4)
  const Granule g = gs[grp];
  const float* gxr = xr + grp * kGr;
  const int npair = g.big >> 1, nquad = (g.end - g.big) >> 2;
  auto elem_bits = [&](int e) {
    if (e < 288) {
      if (e >= npair) return 0;
      return pair_bits(hlen, g.table, gix[2 * e], gix[2 * e + 1]);
    }
    const int qd = e - 288;
    if (qd >= nquad) return 0;
    const int* v = gix + g.big + 4 * qd;
    const int idx = 8 * v[0] + 4 * v[1] + 2 * v[2] + v[3];
    return (int)kTab.qlen[g.c1][idx] + v[0] + v[1] + v[2] + v[3];
  };
  int mine = 0;
  for (int e = 4 * lt; e < 4 * lt + 4; e++) mine += elem_bits(e);
  const int lane = lt & 31, w = lt >> 5;
  int incl = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += y;
  }
  if (lane == 31) scan[grp][w] = incl;
  __syncthreads();
  int pos = 8 * (4 + fmt.side) + (grp == 1 ? gs[0].bits : 0) + incl - mine;
  for (int k = 0; k < w; k++) pos += scan[grp][k];
  for (int e = 4 * lt; e < 4 * lt + 4; e++) {
    if (e < 288) {
      if (e >= npair || g.table == 0) continue;
      const mp3tab::HuffInfo in = kTab.info[g.table];
      const int xv[2] = {gix[2 * e], gix[2 * e + 1]};
      const int code = in.base + min(xv[0], 15) * in.xlen + min(xv[1], 15);
      put_bits(bits, pos, kTab.code[code], hlen[code]);
      pos += hlen[code];
      for (int u = 0; u < 2; u++) {
        if (in.linbits && xv[u] >= 15) { put_bits(bits, pos, (unsigned)(xv[u] - 15), in.linbits); pos += in.linbits; }
        if (xv[u]) { put_bits(bits, pos, gxr[2 * e + u] < 0.f ? 1u : 0u, 1); pos += 1; }
      }
    } else {
      const int qd = e - 288;
      if (qd >= nquad) continue;
      const int* v = gix + g.big + 4 * qd;
      const int idx = 8 * v[0] + 4 * v[1] + 2 * v[2] + v[3];
      put_bits(bits, pos, kTab.qcode[g.c1][idx], kTab.qlen[g.c1][idx]);
      pos += kTab.qlen[g.c1][idx];
      for (int u = 0; u < 4; u++)
        if (v[u]) { put_bits(bits, pos, gxr[g.big + 4 * qd + u] < 0.f ? 1u : 0u, 1); pos += 1; }
    }
  }
  __syncthreads();
  unsigned char* dst = out + boff[b] + fb0;
  for (int i = t; i < len; i += nthr) dst[i] = (unsigned char)get_byte(bits, i);
}

size_t encode_smem() {
  return (size_t)(kMaxIn + kMaxSlots * 64 + kMaxSlots * 32 + kConsts) * sizeof(float) + kBitWords * sizeof(unsigned) +
         mp3tab::kHuffEntries;
}

double window_c(int i) {   // Table C.1 from Table B.3: C[i] = D[i] / 32
  const int j = i <= 256 ? i : 512 - i;
  double d = mp3tab::kWindowD16[j];
  if (i > 256 && (j & 63) != 0) d = -d;
  return d / 65536.0 / 32.0;
}
}  // namespace

// ---------------------------------------------------------------------------------------------- host side
Mp3Format mp3_format(int rate, int kbps) {
  static const int mpeg1[14] = {32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320};
  static const int lsf[14] = {8, 16, 24, 32, 40, 48, 56, 64, 80, 96, 112, 128, 144, 160};
  Mp3Format m;
  m.rate = rate;
  switch (rate) {
    case 44100: m.version = 3; m.sr_index = 0; break;
    case 48000: m.version = 3; m.sr_index = 1; break;
    case 32000: m.version = 3; m.sr_index = 2; break;
    case 22050: m.version = 2; m.sr_index = 0; break;
    case 24000: m.version = 2; m.sr_index = 1; break;
    case 16000: m.version = 2; m.sr_index = 2; break;
    case 11025: m.version = 0; m.sr_index = 0; break;
    case 12000: m.version = 0; m.sr_index = 1; break;
    case 8000: m.version = 0; m.sr_index = 2; break;
    default: throw ArgError("MP3: no MPEG audio version has the sample rate " + std::to_string(rate) + " Hz");
  }
  const bool v1 = m.version == 3;
  const int* tab = v1 ? mpeg1 : lsf;
  m.kbps = kbps == 0 ? (v1 ? 192 : 160) : kbps;
  for (int i = 0; i < 14; i++)
    if (tab[i] == m.kbps) m.br_index = i + 1;
  if (!m.br_index) {
    std::string list;
    for (int i = 0; i < 14; i++) list += (i ? ", " : "") + std::to_string(tab[i]);
    const char* name = v1 ? "MPEG-1" : m.version == 2 ? "MPEG-2" : "MPEG-2.5";
    throw ArgError(std::string("MP3 bitrate ") + std::to_string(kbps) + " kbps is not in the " + name +
                   " Layer III table at " + std::to_string(rate) + " Hz (0 = default, or one of " + list + ")");
  }
  m.ngr = v1 ? 2 : 1;
  m.spf = kGr * m.ngr;
  m.side = v1 ? 17 : 9;
  m.anum = (v1 ? 144000LL : 72000LL) * m.kbps;
  return m;
}

long long mp3_frames(const Mp3Format& fmt, long long n) { return (n + kMp3Delay + fmt.spf - 1) / fmt.spf; }

long long mp3_bytes(const Mp3Format& fmt, long long frames) { return frames * fmt.anum / fmt.rate; }

size_t mp3_const_bytes() { return kConsts * sizeof(float); }

void mp3_consts(void* host_dst) {
  float* c = static_cast<float*>(host_dst);
  const double pi = 3.14159265358979323846;
  for (int i = 0; i < 512; i++) c[kOffC + i] = (float)window_c(i);
  for (int i = 0; i < 64; i++)
    for (int k = 0; k < 32; k++) c[kOffM + 32 * i + k] = (float)std::cos((2 * k + 1) * (i - 16) * pi / 64.0);
  // forward MDCT of block type 0 with the sine window, scaled by 1/9 so that the standard inverse, windowed and
  // overlap-added, returns the subband samples
  for (int m = 0; m < 18; m++)
    for (int i = 0; i < 36; i++)
      c[kOffW + 36 * m + i] = (float)(std::sin(pi / 36.0 * (i + 0.5)) *
                                      std::cos(pi / 72.0 * (2 * i + 19) * (2 * m + 1)) / 9.0);
  static const double ci[8] = {-0.6, -0.535, -0.33, -0.185, -0.095, -0.041, -0.0142, -0.0037};
  for (int i = 0; i < 8; i++) {
    const double r = std::sqrt(1.0 + ci[i] * ci[i]);
    c[kOffCs + i] = (float)(1.0 / r);
    c[kOffCa + i] = (float)(ci[i] / r);
  }
}

void mp3_tables(uint32_t* codes, uint8_t* lens, int32_t* xlen, int32_t* linbits, uint32_t* c1_codes, uint8_t* c1_lens,
                double* window) {
  const mp3tab::Tables& T = mp3tab::kTables;
  for (int t = 0; t < 32; t++) {
    const mp3tab::HuffInfo in = T.info[t];
    if (xlen) xlen[t] = in.xlen;
    if (linbits) linbits[t] = in.linbits;
    for (int e = 0; e < 256; e++) {
      const bool has = t > 0 && e < in.xlen * in.xlen;
      if (codes) codes[t * 256 + e] = has ? T.code[in.base + e] : 0u;
      if (lens) lens[t * 256 + e] = has ? T.len[in.base + e] : 0;
    }
  }
  for (int k = 0; k < 2; k++)
    for (int e = 0; e < 16; e++) {
      if (c1_codes) c1_codes[k * 16 + e] = T.qcode[k][e];
      if (c1_lens) c1_lens[k * 16 + e] = T.qlen[k][e];
    }
  if (window)
    for (int i = 0; i < 512; i++) window[i] = window_c(i);
}

void launch_mp3(const short* pcm, const long long* soff, const int* foff, const long long* boff, int B, int F,
                const Mp3Format& fmt, const void* consts, unsigned char* out, cudaStream_t st) {
  if (g_dry_run) return;
  if (B < 1 || F < B) throw ArgError("launch_mp3: every item needs at least one frame");
  const size_t smem = encode_smem();
  prepare_smem_launch<mp3_encode_kernel>((int)smem);
  mp3_encode_kernel<<<F, fmt.ngr * kGroup, smem, st>>>(pcm, soff, foff, boff, B, fmt, static_cast<const float*>(consts),
                                                       out);
  post_launch("mp3_encode", st);
}

}  // namespace kkx
