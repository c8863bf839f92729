// testapi.cu -- op-level test hooks (include/kkx_test.h).  Parity harness only.
#include "../../include/kkx_test.h"
#include "kernels.h"
#include "model.h"
#include <algorithm>
#include <cstring>
#include <limits>
#include <string>
#include <vector>

using namespace kkx;
static thread_local std::string t_err;

namespace {
struct DevBuf {
  void* p = nullptr;
  DevBuf(const void* host, size_t bytes) {
    KKX_CUDA(cudaMalloc(&p, bytes ? bytes : 4));
    if (host && bytes) KKX_CUDA(cudaMemcpy(p, host, bytes, cudaMemcpyHostToDevice));
  }
  ~DevBuf() { if (p) cudaFree(p); }
  template <class T> T* as() { return static_cast<T*>(p); }
};
template <class F> int run(int device, F&& f) {
  try {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) throw CudaError("no CUDA device (no CPU fallback)");
    KKX_CUDA(cudaSetDevice(device));
    f();
    KKX_CUDA(cudaDeviceSynchronize());
    return KKX_OK;
  } catch (const std::exception& e) {
    t_err = e.what();
    cudaGetLastError();
    return KKX_ERR_CUDA;
  }
}
}  // namespace

extern "C" {

KKX_API const char* kkx_test_last_error(void) { return t_err.c_str(); }

KKX_API int64_t kkx_test_tensor_specs(char* buf, int64_t capacity) {
  std::string s;
  for (auto& sp : kokoro_tensor_specs()) {
    s += sp.first;
    for (int d : sp.second) s += " " + std::to_string(d);
    s += "\n";
  }
  if (buf && capacity > 0) {
    const size_t n = std::min<size_t>(s.size(), (size_t)capacity - 1);
    memcpy(buf, s.data(), n);
    buf[n] = 0;
  }
  return (int64_t)s.size();
}

KKX_API int64_t kkx_test_resample_taps(int32_t out_rate, float* dst, int64_t capacity) {
  std::vector<float> taps;
  const int n = resample_design(out_rate, &taps, nullptr, nullptr, nullptr);
  if (n < 0) return KKX_ERR_ARG;
  if (dst && capacity > 0) memcpy(dst, taps.data(), (size_t)std::min<int64_t>(capacity, n) * sizeof(float));
  return n;
}

KKX_API int kkx_test_resample(int device, const float* x, int32_t B, const int64_t* lens, int32_t out_rate, int32_t law,
                              float* out, int16_t* pcm, uint8_t* codes) {
  return run(device, [&] {
    if (!x || !lens || !out || B < 1 || law < -1 || law > 1) throw ArgError("kkx_test_resample: bad argument");
    std::vector<float> taps;
    int U = 1, D = 1, H = 0;
    if (out_rate != 24000 && resample_design(out_rate, &taps, &U, &D, &H) < 0) throw ArgError("rejected out_rate");
    std::vector<long long> in_off(B), in_len(B), out_off(B);
    long long ni = 0, no = 0, max_out = 0;
    for (int b = 0; b < B; b++) {
      if (lens[b] < 1) throw ArgError("kkx_test_resample: every item needs >= 1 sample");
      const long long m = (lens[b] * U + D - 1) / D;
      in_off[b] = ni; in_len[b] = lens[b]; out_off[b] = no;
      ni += lens[b]; no += m; max_out = std::max(max_out, m);
    }
    DevBuf dx(x, (size_t)ni * 4), dt(taps.data(), taps.size() * 4), dio(in_off.data(), B * 8), dil(in_len.data(), B * 8);
    DevBuf doo(out_off.data(), B * 8), dout(nullptr, (size_t)no * 4), dpcm(nullptr, pcm ? (size_t)no * 2 : 0);
    DevBuf dcode(nullptr, codes && law >= 0 ? (size_t)no : 0);
    launch_resample(dx.as<float>(), dio.as<long long>(), dil.as<long long>(), doo.as<long long>(),
                    taps.empty() ? nullptr : dt.as<float>(), U, D, H, nullptr, dout.as<float>(), pcm ? dpcm.as<short>() : nullptr,
                    codes && law >= 0 ? dcode.as<unsigned char>() : nullptr, law > 0 ? 1 : 0, B, max_out, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)no * 4, cudaMemcpyDeviceToHost));
    if (pcm) KKX_CUDA(cudaMemcpy(pcm, dpcm.p, (size_t)no * 2, cudaMemcpyDeviceToHost));
    if (codes && law >= 0) KKX_CUDA(cudaMemcpy(codes, dcode.p, (size_t)no, cudaMemcpyDeviceToHost));
  });
}

KKX_API int64_t kkx_test_loudness_design(double fs, double* kweight, float* tp_taps, int64_t capacity) {
  if (!(fs > 0)) return KKX_ERR_ARG;
  double kw[10];
  std::vector<float> taps;
  loudness_design(fs, kw, &taps);
  if (kweight) memcpy(kweight, kw, sizeof kw);
  if (tp_taps && capacity > 0) memcpy(tp_taps, taps.data(), (size_t)std::min<int64_t>(capacity, taps.size()) * sizeof(float));
  return (int64_t)taps.size();
}

KKX_API int kkx_test_loudness(int device, const float* x, int32_t B, const int64_t* lens, int32_t target_centi_lufs,
                              int32_t ceiling_centi_dbtp, float* lufs, float* true_peak_dbtp, float* gain) {
  return run(device, [&] {
    if (!x || !lens || B < 1) throw ArgError("kkx_test_loudness: bad argument");
    std::vector<long long> in_off(B), in_len(B), seg_off(B);
    long long ni = 0, nseg = 0, max_len = 0;
    for (int b = 0; b < B; b++) {
      if (lens[b] < 1) throw ArgError("kkx_test_loudness: every item needs >= 1 sample");
      in_off[b] = ni; in_len[b] = lens[b]; seg_off[b] = nseg;
      ni += lens[b]; nseg += lens[b] / kLoudSeg; max_len = std::max<long long>(max_len, lens[b]);
    }
    const LoudParams P = loudness_params(target_centi_lufs / 100.0, ceiling_centi_dbtp / 100.0);
    DevBuf dx(x, (size_t)ni * 4), dio(in_off.data(), B * 8), dil(in_len.data(), B * 8), dso(seg_off.data(), B * 8);
    DevBuf de(nullptr, (size_t)std::max(nseg, 1LL) * 4), dp(nullptr, B * 4), dr(nullptr, (size_t)B * 3 * 4);
    float* r = dr.as<float>();
    launch_loudness(dx.as<float>(), dio.as<long long>(), dil.as<long long>(), dso.as<long long>(), P, de.as<float>(),
                    dp.as<unsigned>(), r, r + B, r + 2 * B, B, max_len, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    if (lufs) KKX_CUDA(cudaMemcpy(lufs, r, B * 4, cudaMemcpyDeviceToHost));
    if (true_peak_dbtp) KKX_CUDA(cudaMemcpy(true_peak_dbtp, r + B, B * 4, cudaMemcpyDeviceToHost));
    if (gain) KKX_CUDA(cudaMemcpy(gain, r + 2 * B, B * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int64_t kkx_test_flac(int device, const int16_t* pcm, int32_t B, const int64_t* lens, int32_t rate,
                              uint8_t* dst, int64_t capacity, int64_t* byte_offsets) {
  long long total = 0;
  const int rc = run(device, [&] {
    if (!pcm || !lens || !byte_offsets || B < 1) throw ArgError("kkx_test_flac: bad argument");
    if (!flac_rate_ok(rate)) throw ArgError("kkx_test_flac: rejected rate");
    std::vector<long long> soff(B + 1, 0);
    std::vector<int> foff(B + 1, 0);
    for (int b = 0; b < B; b++) {
      if (lens[b] < 1) throw ArgError("kkx_test_flac: every item needs >= 1 sample");
      soff[b + 1] = soff[b] + lens[b];
      foff[b + 1] = foff[b] + (int)flac_frames(lens[b]);
    }
    const int F = foff[B];
    DevBuf dp(pcm, (size_t)soff[B] * 2), ds(soff.data(), (B + 1) * 8), df(foff.data(), (B + 1) * 4);
    DevBuf dio(nullptr, (B + 1) * 8), dw(nullptr, flac_work_bytes(F)), dout(nullptr, (size_t)flac_bound(B, F, soff[B]));
    launch_flac(dp.as<short>(), ds.as<long long>(), df.as<int>(), B, F, rate, dw.p, dout.as<unsigned char>(),
                dio.as<long long>(), 0);
    KKX_CUDA(cudaDeviceSynchronize());
    std::vector<long long> io(B + 1);
    KKX_CUDA(cudaMemcpy(io.data(), dio.p, (B + 1) * 8, cudaMemcpyDeviceToHost));
    for (int b = 0; b <= B; b++) byte_offsets[b] = io[b];
    total = io[B];
    if (dst) {
      if (capacity < total) throw ArgError("kkx_test_flac: dst too small");
      KKX_CUDA(cudaMemcpy(dst, dout.p, (size_t)total, cudaMemcpyDeviceToHost));
    }
  });
  return rc == KKX_OK ? (int64_t)total : (int64_t)rc;
}

KKX_API int kkx_test_conv(int device, const float* in, int rows_in, int ldi, int Ci, const float* w,
                          const float* bias, int Co, int ks, int dil, int pad, int stride,
                          const float* pscale, const float* pshift, int pact, float pslope,
                          const float* palpha, int m_len, int ors, int oro, int out_rows,
                          const float* res, int res_rows, int res_shift, float oscale, int eact,
                          int accumulate, float* out) {
  return run(device, [&] {
    DevBuf din(in, (size_t)rows_in * ldi * 4), dw(w, (size_t)ks * Ci * Co * 4), db(bias, bias ? Co * 4 : 0);
    DevBuf dps(pscale, pscale ? Ci * 4 : 0), dph(pshift, pshift ? Ci * 4 : 0), dal(palpha, palpha ? Ci * 4 : 0);
    DevBuf dres(res, res ? (size_t)res_rows * Co * 4 : 0), dout(out, (size_t)out_rows * Co * 4);
    int meta[4] = {0, rows_in, m_len, 0};
    DevBuf dm(meta, sizeof meta);
    ConvArgs a;
    a.in = din.as<float>(); a.ldi = ldi; a.in_off = dm.as<int>(); a.in_len = dm.as<int>() + 1;
    a.m_len = dm.as<int>() + 2; a.max_m = m_len; a.B = 1;
    a.w = dw.as<float>(); a.bias = bias ? db.as<float>() : nullptr;
    a.Ci = Ci; a.Co = Co; a.ks = ks; a.dil = dil; a.pad = pad; a.stride = stride;
    a.pscale = pscale ? dps.as<float>() : nullptr; a.pshift = pshift ? dph.as<float>() : nullptr; a.pld = Ci;
    a.pact = pact; a.pslope = pslope; a.palpha = palpha ? dal.as<float>() : nullptr;
    a.out = dout.as<float>(); a.ldo = Co; a.ocol = 0; a.out_off = dm.as<int>(); a.ors = ors; a.oro = oro;
    a.eact = eact;
    a.res = res ? dres.as<float>() : nullptr; a.ldr = Co; a.rcol = 0; a.res_off = dm.as<int>() + 3;
    a.res_shift = res_shift; a.oscale = oscale; a.accumulate = accumulate;
    launch_conv_f32(a, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)out_rows * Co * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_conv_tc(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                             int Co, int ks, int dil, int pad, const float* pscale, const float* pshift,
                             int pact, float pslope, const float* palpha, int m_len, int ors, int oro,
                             int out_rows, const float* res, int res_rows, int res_shift, float oscale,
                             int accumulate, float* out) {
  return run(device, [&] {
    const int Cpad = (Ci + 63) & ~63;
    const int off = kGapRows, rows_total = (off + L + kGapRows + 7) & ~7;
    std::vector<uint16_t> hw((size_t)Co * ks * Cpad, 0);
    for (int o = 0; o < Co; o++)
      for (int k = 0; k < ks; k++)
        for (int c = 0; c < Ci; c++) {
          float f = w[((size_t)o * ks + k) * Ci + c];
          uint32_t u; memcpy(&u, &f, 4);
          hw[((size_t)o * ks + k) * Cpad + c] = (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
        }
    std::vector<float> xin((size_t)rows_total * Ci, 0.f);
    memcpy(xin.data() + (size_t)off * Ci, x, (size_t)L * Ci * 4);
    DevBuf dx(xin.data(), xin.size() * 4), dw(hw.data(), hw.size() * 2), db(bias, bias ? Co * 4 : 0);
    DevBuf dps(pscale, pscale ? Ci * 4 : 0), dph(pshift, pshift ? Ci * 4 : 0), dal(palpha, palpha ? Ci * 4 : 0);
    DevBuf dres(res, res ? (size_t)res_rows * Co * 4 : 0), dout(out, (size_t)out_rows * Co * 4);
    DevBuf dab(nullptr, (size_t)rows_total * Cpad * 2);
    KKX_CUDA(cudaMemset(dab.p, 0xFF, (size_t)rows_total * Cpad * 2));  // NaN-fill: the producer must zero halos
    int meta[5] = {off, L, m_len, 0, 0};
    DevBuf dm(meta, sizeof meta);
    launch_apply_bf16(dx.as<float>(), Ci, Ci, pscale ? dps.as<float>() : nullptr, pshift ? dph.as<float>() : nullptr,
                      pact, pslope, palpha ? dal.as<float>() : nullptr, dab.p, Cpad, rows_total, dm.as<int>(),
                      dm.as<int>() + 1, 1, L, 0);
    alignas(64) unsigned char tmA[128], tmB[128];
    make_tmap_bf16(tmA, dab.p, Cpad, rows_total, Cpad, 128);
    make_tmap_bf16(tmB, dw.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, tc_box_n(Co));
    TcConvArgs a;
    a.tmA = tmA; a.tmB = tmB; a.Cpad = Cpad; a.Ci = Ci; a.Co = Co; a.ks = ks; a.dil = dil; a.pad = pad;
    a.in_off = dm.as<int>(); a.m_len = dm.as<int>() + 2; a.max_m = m_len; a.B = 1; a.sum_m = m_len;
    a.bias = bias ? db.as<float>() : nullptr;
    a.out = dout.as<float>(); a.ldo = Co; a.ocol = 0; a.out_off = dm.as<int>() + 3; a.ors = ors; a.oro = oro;
    a.res = res ? dres.as<float>() : nullptr; a.ldr = Co; a.rcol = 0; a.res_off = dm.as<int>() + 4;
    a.res_shift = res_shift; a.oscale = oscale; a.accumulate = accumulate;
    launch_conv_tc(a, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)out_rows * Co * 4, cudaMemcpyDeviceToHost));
  });
}

static inline float host_tf32(float f) {   // cvt.rna.tf32.f32
  uint32_t u; memcpy(&u, &f, 4);
  u = (u + 0x1000u) & ~0x1FFFu;
  float r; memcpy(&r, &u, 4);
  return r;
}

KKX_API int kkx_test_conv_tf32(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                               int Co, int ks, int dil, int pad, int nprod, int eact, float* out) {
  return run(device, [&] {
    const int Cpad = (Ci + 63) & ~63;
    const int off = kGapRows, rows_total = (off + L + kGapRows + 7) & ~7;
    std::vector<float> whi((size_t)Co * ks * Cpad, 0.f), wlo((size_t)Co * ks * Cpad, 0.f);
    for (int o = 0; o < Co; o++)
      for (int k = 0; k < ks; k++)
        for (int c = 0; c < Ci; c++) {
          const float f = w[((size_t)o * ks + k) * Ci + c];
          const float hi = host_tf32(f);
          whi[((size_t)o * ks + k) * Cpad + c] = hi;
          wlo[((size_t)o * ks + k) * Cpad + c] = host_tf32(f - hi);
        }
    std::vector<float> xin((size_t)rows_total * Ci, 0.f);
    memcpy(xin.data() + (size_t)off * Ci, x, (size_t)L * Ci * 4);
    DevBuf dx(xin.data(), xin.size() * 4), dwh(whi.data(), whi.size() * 4), dwl(wlo.data(), wlo.size() * 4);
    DevBuf db(bias, bias ? Co * 4 : 0), dout(nullptr, (size_t)L * Co * 4);
    DevBuf dah(nullptr, (size_t)rows_total * Cpad * 4), dal(nullptr, (size_t)rows_total * Cpad * 4);
    KKX_CUDA(cudaMemset(dah.p, 0xFF, (size_t)rows_total * Cpad * 4));
    KKX_CUDA(cudaMemset(dal.p, 0xFF, (size_t)rows_total * Cpad * 4));
    int meta[4] = {off, L, 0, 0};
    DevBuf dm(meta, sizeof meta);
    launch_apply_tf32(dx.as<float>(), Ci, Ci, nullptr, nullptr, ACT_NONE, 0.f, dah.as<float>(), dal.as<float>(), Cpad,
                      rows_total, dm.as<int>(), dm.as<int>() + 1, 1, L, 0);
    alignas(64) unsigned char tA[128], tA2[128], tB[128], tB2[128];
    make_tmap_f32(tA, dah.p, Cpad, rows_total, Cpad, 128);
    make_tmap_f32(tA2, dal.p, Cpad, rows_total, Cpad, 128);
    make_tmap_f32(tB, dwh.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, tc_box_n_tf32(Co));
    make_tmap_f32(tB2, dwl.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, tc_box_n_tf32(Co));
    TcConvArgs a;
    a.tmA = tA; a.tmA2 = tA2; a.tmB = tB; a.tmB2 = tB2; a.tf32 = 1; a.nprod = nprod; a.eact = eact;
    a.Cpad = Cpad; a.Ci = Ci; a.Co = Co; a.ks = ks; a.dil = dil; a.pad = pad;
    a.in_off = dm.as<int>(); a.m_len = dm.as<int>() + 1; a.max_m = L; a.B = 1; a.sum_m = L;
    a.bias = bias ? db.as<float>() : nullptr;
    a.out = dout.as<float>(); a.ldo = Co; a.ocol = 0; a.out_off = dm.as<int>() + 2; a.ors = 1; a.oro = 0;
    launch_conv_tc(a, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)L * Co * 4, cudaMemcpyDeviceToHost));
  });
}

// kernel: 0 = the launcher's own choice, 1 = single-tile kernel, 2 = persistent kernel, 3 = persistent CTA-pair kernel
static int conv_f16x3_impl(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                           int Co, int ks, int dil, int pad, int eact, int kernel, const float* res, float oscale, float* out) {
  return run(device, [&] {
    const int Cpad = (Ci + 63) & ~63;
    const int off = kGapRows, rows_total = (off + L + kGapRows + 7) & ~7;
    std::vector<float> wp((size_t)Co * ks * Cpad, 0.f);
    for (int o = 0; o < Co; o++)
      for (int k = 0; k < ks; k++)
        for (int c = 0; c < Ci; c++) wp[((size_t)o * ks + k) * Cpad + c] = w[((size_t)o * ks + k) * Ci + c];
    std::vector<unsigned short> whi(wp.size()), wlo(wp.size());
    const float wscale = split_f16_host(wp.data(), wp.size(), whi.data(), wlo.data());
    std::vector<float> xin((size_t)rows_total * Ci, 0.f);
    memcpy(xin.data() + (size_t)off * Ci, x, (size_t)L * Ci * 4);
    DevBuf dx(xin.data(), xin.size() * 4), dwh(whi.data(), whi.size() * 2), dwl(wlo.data(), wlo.size() * 2);
    DevBuf db(bias, bias ? Co * 4 : 0), dout(nullptr, (size_t)L * Co * 4);
    DevBuf dah(nullptr, (size_t)rows_total * Cpad * 2), dal(nullptr, (size_t)rows_total * Cpad * 2);
    KKX_CUDA(cudaMemset(dah.p, 0xFF, (size_t)rows_total * Cpad * 2));
    KKX_CUDA(cudaMemset(dal.p, 0xFF, (size_t)rows_total * Cpad * 2));
    int meta[4] = {off, L, 0, 0};
    DevBuf dm(meta, sizeof meta);
    launch_apply_f16x2(dx.as<float>(), Ci, Ci, nullptr, nullptr, ACT_NONE, 0.f, dah.p, dal.p, Cpad,
                       rows_total, dm.as<int>(), dm.as<int>() + 1, 1, L, 0);
    alignas(64) unsigned char tA[128], tA2[128], tB[128], tB2[128], tBc[128], tB2c[128];
    make_tmap_f16(tA, dah.p, Cpad, rows_total, Cpad, 128);
    make_tmap_f16(tA2, dal.p, Cpad, rows_total, Cpad, 128);
    make_tmap_f16(tB, dwh.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, tc_box_n_tf32(Co));
    make_tmap_f16(tB2, dwl.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, tc_box_n_tf32(Co));
    // tile table of the one item, so that large problems take the persistent kernel like the model does
    const int nt = (L + 127) / 128;
    int tiles[2] = {0, nt};
    DevBuf dt(tiles, sizeof tiles);
    TcConvArgs a;
    a.tmA = tA; a.tmA2 = tA2; a.tmB = tB; a.tmB2 = tB2; a.tf32 = 1; a.nprod = 3; a.eact = eact;
    a.f16 = 1; a.wscale = wscale / kSplitF16Scale;
    if (tc_box_n_tf32(Co) == 128) {
      make_tmap_f16(tBc, dwh.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, 64);
      make_tmap_f16(tB2c, dwl.p, (long long)ks * Cpad, Co, (long long)ks * Cpad, 64);
      a.tmB_c = tBc; a.tmB2_c = tB2c;
    }
    a.Cpad = Cpad; a.Ci = Ci; a.Co = Co; a.ks = ks; a.dil = dil; a.pad = pad;
    a.in_off = dm.as<int>(); a.m_len = dm.as<int>() + 1; a.max_m = L; a.B = 1; a.sum_m = L;
    a.bias = bias ? db.as<float>() : nullptr;
    a.out = dout.as<float>(); a.ldo = Co; a.ocol = 0; a.out_off = dm.as<int>() + 2; a.ors = 1; a.oro = 0;
    a.tile_start = dt.as<int>(); a.ntiles_m = nt;
    DevBuf dres(res, res ? (size_t)L * Co * 4 : 0);
    if (res) { a.res = dres.as<float>(); a.ldr = Co; a.rcol = 0; a.res_off = dm.as<int>() + 2; a.res_shift = 0; }
    a.oscale = oscale;
    if (kernel) a.force_kernel = 1;
    if (kernel == 1) { a.tile_start = nullptr; a.ntiles_m = 0; }
    a.pair = (kernel == 0 || kernel == 3) ? 1 : 0;
    launch_conv_tc(a, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)L * Co * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_conv_f16x3(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                                int Co, int ks, int dil, int pad, int eact, float* out) {
  return conv_f16x3_impl(device, x, L, Ci, w, bias, Co, ks, dil, pad, eact, 0, nullptr, 1.f, out);
}

KKX_API int kkx_test_conv_f16x3_k(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                                  int Co, int ks, int dil, int pad, int eact, int kernel, const float* res, float oscale,
                                  float* out) {
  return conv_f16x3_impl(device, x, L, Ci, w, bias, Co, ks, dil, pad, eact, kernel, res, oscale, out);
}

KKX_API int kkx_test_lstm(int device, const float* xproj, const float* whhT, int N, float* out) {
  return run(device, [&] {
    DevBuf dx(xproj, (size_t)N * 2048 * 4), dw(whhT, (size_t)2 * 256 * 1024 * 4), dout(nullptr, (size_t)N * 512 * 4);
    int meta[2] = {0, N};
    DevBuf dm(meta, sizeof meta);
    launch_lstm(dx.as<float>(), dw.as<float>(), dout.as<float>(), 512, 0, dm.as<int>(), dm.as<int>() + 1, 1, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)N * 512 * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_lstm_batch(int device, const float* xproj, const float* whhT, int B, const int* off,
                                const int* len, int rows, float* out) {
  return run(device, [&] {
    DevBuf dx(xproj, (size_t)rows * 2048 * 4), dw(whhT, (size_t)2 * 256 * 1024 * 4), dout(out, (size_t)rows * 512 * 4);
    DevBuf doff(off, B * 4), dlen(len, B * 4);
    launch_lstm(dx.as<float>(), dw.as<float>(), dout.as<float>(), 512, 0, doff.as<int>(), dlen.as<int>(), B, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)rows * 512 * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_lstm_batch_v(int device, const float* xproj, const float* whhT, int B, const int* off,
                                  const int* len, int rows, int variant, int reps, float* out, float* ms) {
  return run(device, [&] {
    DevBuf dx(xproj, (size_t)rows * 2048 * 4), dw(whhT, (size_t)2 * 256 * 1024 * 4), dout(out, (size_t)rows * 512 * 4);
    DevBuf doff(off, B * 4), dlen(len, B * 4);
    cudaEvent_t e0, e1;
    KKX_CUDA(cudaEventCreate(&e0)); KKX_CUDA(cudaEventCreate(&e1));
    launch_lstm(dx.as<float>(), dw.as<float>(), dout.as<float>(), 512, 0, doff.as<int>(), dlen.as<int>(), B, 0, variant);
    KKX_CUDA(cudaEventRecord(e0, 0));
    for (int i = 0; i < reps; i++)
      launch_lstm(dx.as<float>(), dw.as<float>(), dout.as<float>(), 512, 0, doff.as<int>(), dlen.as<int>(), B, 0, variant);
    KKX_CUDA(cudaEventRecord(e1, 0));
    KKX_CUDA(cudaDeviceSynchronize());
    float t = 0.f;
    KKX_CUDA(cudaEventElapsedTime(&t, e0, e1));
    if (ms) *ms = reps > 0 ? t / reps : 0.f;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)rows * 512 * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_pointwise_conv_stats(int device, const float* x, const float* w, const float* bias, int B,
                                          const int* off, const int* len, int rows, int max_len, float* out, float* part,
                                          float* part_ref) {
  return run(device, [&] {
    const int nchunk = (max_len + kStatRows - 1) / kStatRows;
    const size_t np = (size_t)B * nchunk * 2 * 128;
    DevBuf dx(x, (size_t)rows * 24 * 4), dw(w, (size_t)22 * 128 * 4), db(bias, 128 * 4), dout(out, (size_t)rows * 128 * 4);
    DevBuf dp(part, np * 4), dpr(part_ref, np * 4), doff(off, B * 4), dlen(len, B * 4);
    long long sum_m = 0;
    for (int b = 0; b < B; b++) sum_m += len[b];
    launch_pointwise_conv_stats(dx.as<float>(), 24, 22, dw.as<float>(), db.as<float>(), dout.as<float>(), 128, dp.as<float>(),
                                doff.as<int>(), dlen.as<int>(), B, max_len, sum_m, 0);
    // the statistics pass it replaces, over the tensor just written
    launch_colstats(dout.as<float>(), 128, 128, dpr.as<float>(), doff.as<int>(), dlen.as<int>(), B, max_len, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)rows * 128 * 4, cudaMemcpyDeviceToHost));
    KKX_CUDA(cudaMemcpy(part, dp.p, np * 4, cudaMemcpyDeviceToHost));
    KKX_CUDA(cudaMemcpy(part_ref, dpr.p, np * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_layernorm(int device, const float* x, const float* res, const float* w, const float* b,
                               const float* ada, int rows, int C, float eps, float slope, float* out,
                               unsigned short* pl_hi, unsigned short* pl_lo) {
  return run(device, [&] {
    const size_t n = (size_t)rows * C;
    DevBuf dx(x, n * 4), dr(res, res ? n * 4 : 0), dw(w, w ? (size_t)C * 4 : 0), db(b, b ? (size_t)C * 4 : 0);
    DevBuf da(ada, ada ? (size_t)2 * C * 4 : 0), dout(nullptr, n * 4), dhi(nullptr, pl_hi ? n * 2 : 0), dlo(nullptr, pl_lo ? n * 2 : 0);
    int meta[2] = {0, rows};
    DevBuf dm(meta, sizeof meta);
    LnArgs a;
    a.x = dx.as<float>(); a.ldx = C;
    if (res) { a.res = dr.as<float>(); a.ldr = C; }
    if (w) { a.w = dw.as<float>(); a.b = db.as<float>(); }
    if (ada) { a.ada = da.as<float>(); a.ada_ld = 2 * C; a.ada_off = 0; }
    a.eps = eps; a.slope = slope; a.out = dout.as<float>(); a.ldo = C; a.ocol = 0;
    a.off = dm.as<int>(); a.len = dm.as<int>() + 1; a.B = 1; a.max_len = rows; a.C = C;
    if (pl_hi) { a.pl_hi = dhi.p; a.pl_lo = dlo.p; a.pl_ld = C; }
    launch_layernorm(a, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, n * 4, cudaMemcpyDeviceToHost));
    if (pl_hi) {
      KKX_CUDA(cudaMemcpy(pl_hi, dhi.p, n * 2, cudaMemcpyDeviceToHost));
      KKX_CUDA(cudaMemcpy(pl_lo, dlo.p, n * 2, cudaMemcpyDeviceToHost));
    }
  });
}

KKX_API int kkx_test_im2col(int device, const float* in, int rows_in, int B, const int* in_off, const int* in_len,
                            const int* out_off, const int* out_len, int rows_out, int max_out_len, int Cpad, int generic,
                            unsigned short* out) {
  return run(device, [&] {
    DevBuf di(in, (size_t)rows_in * 24 * 4), dout(out, (size_t)rows_out * Cpad * 2);
    DevBuf dio(in_off, B * 4), dil(in_len, B * 4), doo(out_off, B * 4), dol(out_len, B * 4);
    launch_im2col_bf16(di.as<float>(), 24, 22, 12, 6, 3, dout.p, Cpad, rows_out, dio.as<int>(), dil.as<int>(), doo.as<int>(),
                       dol.as<int>(), B, max_out_len, 0, generic);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(out, dout.p, (size_t)rows_out * Cpad * 2, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_attention(int device, const float* qkv, int N, float* ctx) {
  return run(device, [&] {
    DevBuf dq(qkv, (size_t)N * 2304 * 4), dout(nullptr, (size_t)N * 768 * 4);
    int meta[2] = {0, N};
    DevBuf dm(meta, sizeof meta);
    launch_attention(dq.as<float>(), dout.as<float>(), dm.as<int>(), dm.as<int>() + 1, 1, N, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(ctx, dout.p, (size_t)N * 768 * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_attention_batch(int device, const float* qkv, int B, const int* off, const int* len, int rows,
                                     int umma, float* ctx) {
  return run(device, [&] {
    int max_len = 0;
    for (int b = 0; b < B; b++) max_len = std::max(max_len, len[b]);
    DevBuf dq(qkv, (size_t)rows * 2304 * 4), dout(ctx, (size_t)rows * 768 * 4);
    DevBuf doff(off, (size_t)B * 4), dlen(len, (size_t)B * 4);
    if (umma) {
      // scratch deliberately filled with NaN patterns: stale gap rows must never reach a valid result
      const size_t nf = attention_umma_scratch_floats(rows, B);
      DevBuf ds(nullptr, nf * 4);
      KKX_CUDA(cudaMemset(ds.p, 0xFF, nf * 4));
      launch_attention_umma(dq.as<float>(), ds.as<float>(), dout.as<float>(), doff.as<int>(), dlen.as<int>(), B, max_len, rows, 0);
      KKX_CUDA(cudaDeviceSynchronize());
    } else {
      launch_attention(dq.as<float>(), dout.as<float>(), doff.as<int>(), dlen.as<int>(), B, max_len, 0);
      KKX_CUDA(cudaDeviceSynchronize());
    }
    KKX_CUDA(cudaMemcpy(ctx, dout.p, (size_t)rows * 768 * 4, cudaMemcpyDeviceToHost));
  });
}

KKX_API int kkx_test_adain_coef(int device, const float* x, int L, int C, const float* gamma_beta,
                                float* scale, float* shift) {
  return run(device, [&] {
    const int nch = (L + kStatRows - 1) / kStatRows;
    DevBuf dx(x, (size_t)L * C * 4), dgb(gamma_beta, (size_t)2 * C * 4), dpart(nullptr, (size_t)nch * 2 * C * 4);
    DevBuf dsc(nullptr, C * 4), dsh(nullptr, C * 4);
    int meta[2] = {0, L};
    DevBuf dm(meta, sizeof meta);
    launch_colstats(dx.as<float>(), C, C, dpart.as<float>(), dm.as<int>(), dm.as<int>() + 1, 1, L, 0);
    launch_adain_coef(dpart.as<float>(), C, L, dm.as<int>() + 1, dgb.as<float>(), 2 * C, 0, 1e-5f,
                      dsc.as<float>(), dsh.as<float>(), 1, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    KKX_CUDA(cudaMemcpy(scale, dsc.p, C * 4, cudaMemcpyDeviceToHost));
    KKX_CUDA(cudaMemcpy(shift, dsh.p, C * 4, cudaMemcpyDeviceToHost));
  });
}

static inline uint16_t host_bf16(float f) {
  uint32_t u; memcpy(&u, &f, 4);
  return (uint16_t)((u + 0x7FFFu + ((u >> 16) & 1u)) >> 16);
}

}  // extern "C"

static int arb_conv_test(int device, const float* x, int B, const int* lens, int C, int in_bf16,
                         const float* scale, const float* shift, const float* alpha, const float* w,
                         const float* bias, int ks, int dil, const float* res, int res_bf16, float oscale,
                         int accumulate, int want_bf16, float* out, float* sums, int desc_mode) {
  return run(device, [&] {
    if (!arb_conv_supported(C, ks, dil, B)) throw ArgError("kkx_test_arb_conv: unsupported shape");
    // ragged Level layout with NaN-filled gap rows: the kernel must never consume a gap row
    std::vector<int> off(B), tiles(B + 1, 0);
    const int MT = arb_tile_rows(C);
    int o = kGapRows, maxL = 0; long long sumL = 0;
    for (int b = 0; b < B; b++) {
      off[b] = o; o = (o + lens[b] + kGapRows + 7) & ~7;
      tiles[b + 1] = tiles[b] + (lens[b] + MT - 1) / MT;
      maxL = std::max(maxL, lens[b]); sumL += lens[b];
    }
    const int rows = o;
    const float qnan = std::numeric_limits<float>::quiet_NaN();
    std::vector<float> hx((size_t)rows * C, qnan), hres((size_t)rows * C, qnan), hout((size_t)rows * C, qnan);
    size_t src = 0;
    for (int b = 0; b < B; b++) {
      memcpy(hx.data() + (size_t)off[b] * C, x + src * C, (size_t)lens[b] * C * 4);
      if (res) memcpy(hres.data() + (size_t)off[b] * C, res + src * C, (size_t)lens[b] * C * 4);
      memcpy(hout.data() + (size_t)off[b] * C, out + src * C, (size_t)lens[b] * C * 4);
      src += lens[b];
    }
    std::vector<uint16_t> hxb;
    if (in_bf16) { hxb.resize(hx.size()); for (size_t i = 0; i < hx.size(); i++) hxb[i] = host_bf16(hx[i]); }
    std::vector<uint16_t> hw((size_t)C * ks * C);
    for (size_t i = 0; i < hw.size(); i++) hw[i] = host_bf16(w[i]);
    DevBuf dx(in_bf16 ? (const void*)hxb.data() : (const void*)hx.data(), hx.size() * (in_bf16 ? 2 : 4));
    DevBuf dw(hw.data(), hw.size() * 2), db(bias, C * 4), dsc(scale, (size_t)B * C * 4), dsh(shift, (size_t)B * C * 4);
    std::vector<uint16_t> hresb;
    if (res && res_bf16) { hresb.resize(hres.size()); for (size_t i = 0; i < hres.size(); i++) hresb[i] = host_bf16(hres[i]); }
    DevBuf dal(alpha, C * 4), dres(res ? (res_bf16 ? (const void*)hresb.data() : (const void*)hres.data()) : nullptr,
                                   res ? hres.size() * (res_bf16 ? 2 : 4) : 0);
    DevBuf dout(hout.data(), hout.size() * 4), doutb(nullptr, hout.size() * 2);
    KKX_CUDA(cudaMemset(doutb.p, 0xFF, hout.size() * 2));
    const int nchunk = (maxL + 127) / 128;
    DevBuf dpart(nullptr, (size_t)B * nchunk * 2 * C * 4);
    KKX_CUDA(cudaMemset(dpart.p, 0, (size_t)B * nchunk * 2 * C * 4));
    DevBuf doff(off.data(), B * 4), dlen(lens, B * 4), dts(tiles.data(), (B + 1) * 4);
    alignas(64) unsigned char tmB[128];
    make_tmap_bf16(tmB, dw.p, (long long)ks * C, C, (long long)ks * C, tc_box_n(C));
    ArbConvArgs a;
    a.x = dx.p; a.in_bf16 = in_bf16; a.scale = dsc.as<float>(); a.shift = dsh.as<float>(); a.alpha = dal.as<float>();
    a.tmB = tmB; a.C = C; a.ks = ks; a.dil = dil; a.pad = dil * (ks - 1) / 2;
    a.off = doff.as<int>(); a.len = dlen.as<int>(); a.tile_start = dts.as<int>(); a.B = B; a.total_tiles = tiles[B];
    a.sum_m = sumL; a.bias = db.as<float>();
    a.out_bf16 = want_bf16 ? doutb.as<__nv_bfloat16>() : nullptr;
    a.out_f32 = want_bf16 ? nullptr : dout.as<float>();
    a.res = res ? dres.as<float>() : nullptr; a.res_bf16 = res ? res_bf16 : 0; a.oscale = oscale; a.accumulate = accumulate;
    a.part = sums ? dpart.as<float>() : nullptr; a.nchunk = nchunk; (void)desc_mode;
    launch_arb_conv(a, 0);
    KKX_CUDA(cudaDeviceSynchronize());
    if (want_bf16) {
      std::vector<uint16_t> hb(hout.size());
      KKX_CUDA(cudaMemcpy(hb.data(), doutb.p, hb.size() * 2, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < hb.size(); i++) { uint32_t u = (uint32_t)hb[i] << 16; memcpy(&hout[i], &u, 4); }
    } else {
      KKX_CUDA(cudaMemcpy(hout.data(), dout.p, hout.size() * 4, cudaMemcpyDeviceToHost));
    }
    src = 0;
    for (int b = 0; b < B; b++) {
      memcpy(out + src * C, hout.data() + (size_t)off[b] * C, (size_t)lens[b] * C * 4);
      src += lens[b];
    }
    if (sums) {
      std::vector<float> hp((size_t)B * nchunk * 2 * C);
      KKX_CUDA(cudaMemcpy(hp.data(), dpart.p, hp.size() * 4, cudaMemcpyDeviceToHost));
      for (int b = 0; b < B; b++)
        for (int k = 0; k < 2; k++)
          for (int c = 0; c < C; c++) {
            double acc = 0.0;
            for (int ch = 0; ch < (lens[b] + 127) / 128; ch++) acc += hp[(((size_t)b * nchunk + ch) * 2 + k) * C + c];
            sums[((size_t)b * 2 + k) * C + c] = (float)acc;
          }
    }
  });
}

extern "C" {

KKX_API int kkx_test_arb_conv(int device, const float* x, int B, const int* lens, int C, int in_bf16,
                              const float* scale, const float* shift, const float* alpha, const float* w,
                              const float* bias, int ks, int dil, const float* res, float oscale,
                              int accumulate, int want_bf16, float* out, float* sums, int desc_mode) {
  return arb_conv_test(device, x, B, lens, C, in_bf16, scale, shift, alpha, w, bias, ks, dil, res, 0, oscale, accumulate,
                       want_bf16, out, sums, desc_mode);
}

KKX_API int kkx_test_arb_conv_stream(int device, const float* x, int B, const int* lens, int C, const float* scale,
                                     const float* shift, const float* alpha, const float* w, const float* bias, int ks,
                                     int dil, const float* res, float oscale, int accumulate, int want_bf16, float* out,
                                     float* sums) {
  return arb_conv_test(device, x, B, lens, C, 1, scale, shift, alpha, w, bias, ks, dil, res, 1, oscale, accumulate,
                       want_bf16, out, sums, 0);
}

}  // extern "C"
