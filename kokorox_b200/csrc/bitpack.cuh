// bitpack.cuh -- device helpers shared by the stream encoders (kernels_flac.cu, kernels_mp3.cu): an MSB-first bit
// buffer in shared memory and the item that owns a frame.
#pragma once

namespace kkx {
namespace {

// item b owns frames [foff[b], foff[b + 1]); the last b with foff[b] <= f
__device__ __forceinline__ int frame_item(const int* foff, int B, int f) {
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(foff + mid) <= f) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// MSB-first bit buffer in 32-bit words: stream bit i is bit 31 - (i & 31) of word i >> 5.  nbits <= 32.  Fields OR
// into a zeroed buffer, so threads may write disjoint fields in any order.
__device__ __forceinline__ void put_bits(unsigned* buf, int pos, unsigned v, int nbits) {
  if (nbits <= 0) return;
  const unsigned long long w = (unsigned long long)v << (64 - nbits - (pos & 31));
  const unsigned hi = (unsigned)(w >> 32), lo = (unsigned)w;
  if (hi) atomicOr(buf + (pos >> 5), hi);
  if (lo) atomicOr(buf + (pos >> 5) + 1, lo);
}
__device__ __forceinline__ unsigned get_byte(const unsigned* buf, int i) {
  return (buf[i >> 2] >> (24 - 8 * (i & 3))) & 0xFFu;
}

}  // namespace
}  // namespace kkx
