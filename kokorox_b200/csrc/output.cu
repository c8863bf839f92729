// output.cu -- the output stage of a run (output.h): everything between the iSTFT's waveform and what the caller
// fetches.  Host-side orchestration only; the kernels are in kernels_signal.cu, kernels_loudness.cu, kernels_flac.cu
// and kernels_mp3.cu.
#include "output.h"
#include "model.h"
#include <algorithm>
#include <cstring>
#include <string>

namespace kkx {

namespace {
size_t round256(size_t b) { return (b + 255) & ~size_t(255); }

// A grow-only arena, reset for the run; when it is too small the stream must be done with the old one.
void grow(Arena& a, size_t bytes, cudaStream_t st) {
  a.reset();
  if (bytes <= a.capacity()) return;
  KKX_CUDA(cudaStreamSynchronize(st));
  a.reserve(bytes + bytes / 4);
}

// Offsets in the encoder's table block: soff [P + 1] | boff [P + 1] | foff [P + 1] | work, each 256-byte aligned.
struct TableLayout {
  size_t boff, foff, work;
  explicit TableLayout(int P)
      : boff(round256((size_t)(P + 1) * sizeof(long long))), foff(2 * boff),
        work(foff + round256((size_t)(P + 1) * sizeof(int))) {}
};
}  // namespace

// The post-processing pass runs unless the output is the plain 24 kHz waveform or its PCM: G.711 codes, loudness
// normalisation, the limiter and the loudness report want it (at 24 kHz as a pass-through, U = D = 1, which applies
// the gain, or none when only measuring).  The taps live on the device per Model and are rebuilt only when the rate
// changes.
OutputPlan output_plan(const Options& opt, Encoding enc, int kbps, OutputBuffers& buf, cudaStream_t st) {
  OutputPlan p;
  p.enc = enc;
  p.rate = opt.out_rate;
  if (enc == Encoding::MP3) p.mp3 = mp3_format(opt.out_rate, kbps);
  if (enc == Encoding::FLAC) p.flac_lpc = opt.flac_lpc_order;
  p.loud = opt.loudness_target != 0;
  p.limit = opt.limiter != 0;
  p.report = opt.loudness_report != 0;
  p.measure = p.loud || p.limit || p.report;
  if (p.measure) p.par = loudness_params(opt.loudness_target / 100.0, opt.true_peak_max / 100.0, p.limit, p.report);
  p.post = opt.out_rate != 24000 || p.law() || p.measure;
  if (opt.out_rate == 24000) return p;
  std::vector<float> taps;
  if (resample_design(opt.out_rate, &taps, &p.U, &p.D, &p.H) < 0)
    throw ArgError("out_rate " + std::to_string(opt.out_rate) + " is not supported");
  if (buf.taps_rate != opt.out_rate) {
    KKX_CUDA(cudaStreamSynchronize(st));
    if (buf.d_taps) cudaFree(buf.d_taps);
    buf.d_taps = nullptr; buf.taps_rate = 0;
    KKX_CUDA(cudaMalloc(&buf.d_taps, taps.size() * sizeof(float)));
    KKX_CUDA(cudaMemcpy(buf.d_taps, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
    buf.taps_rate = opt.out_rate;
  }
  p.taps = buf.d_taps;
  return p;
}

Spans make_spans(const std::vector<long long>& len24, long long in0, long long out0, int U, int D) {
  Spans s;
  const int n = s.n = (int)len24.size();
  s.host.assign((size_t)4 * n, 0);
  long long* in_off = s.host.data();
  long long* in_len = in_off + n;
  long long* out_off = in_off + 2 * n;
  long long* seg_off = in_off + 3 * n;
  for (int k = 0; k < n; k++) {
    const long long m = (len24[k] * U + D - 1) / D;
    in_off[k] = in0; in_len[k] = len24[k]; out_off[k] = out0; seg_off[k] = s.nseg;
    in0 += len24[k]; out0 += m; s.nseg += len24[k] / kLoudSeg;
    s.max_len = std::max(s.max_len, len24[k]);
    s.max_out = std::max(s.max_out, m);
  }
  s.in_end = in0; s.out_end = out0;
  return s;
}

void post_programs(const OutputPlan& p, const Spans& s, const OutputBuffers& o, int k0, int P, Arena& scratch,
                   cudaStream_t st) {
  const int K = s.n;
  auto row = [&](int i) { return o.report + (size_t)i * P + k0; };
  const float* wav = o.wav24;
  float* gain = nullptr;
  if (p.measure) {   // per-program 2400-sample segment energies and true peaks of the 24 kHz waveform
    float* energy = scratch.alloc<float>((size_t)std::max(s.nseg, 1LL));
    unsigned* peak = scratch.alloc<unsigned>(K);
    gain = row(2);
    launch_loudness(o.wav24, s.in_off, s.in_len, s.seg_off, p.par, energy, peak, row(0), row(1), gain, K, s.max_len,
                    st, p.limit ? o.lim_p : nullptr);
    if (p.report) {   // on the same energies, before the limiter
      double* short_e = scratch.alloc<double>((size_t)std::max(s.nseg, 1LL));
      launch_loudness_range(s.in_len, s.seg_off, energy, short_e, row(3), row(4), row(5), K, s.max_len, st);
      if (!p.loud && !p.limit) gain = nullptr;   // measure-only: the resampling pass is the plain output's arithmetic
    }
    if (p.limit) {    // the limited waveform v is resampled instead, with the static trim t as its gain
      unsigned* acc = scratch.alloc<unsigned>((size_t)2 * K);
      launch_limiter(o.wav24, o.lim_p, s.in_off, s.in_len, p.par, gain, o.lim_v, nullptr, acc, row(6), row(7), row(8),
                     K, s.max_len, st);
      wav = o.lim_v;
      gain = row(6);
    }
  }
  // grids span the longest program (64-bit sample indices); CTAs past a shorter program's end return at once
  launch_resample(wav, s.in_off, s.in_len, s.out_off, p.taps, p.U, p.D, p.H, gain, o.audio,
                  p.pcm() ? static_cast<short*>(o.twin) : nullptr,
                  p.law() ? static_cast<unsigned char*>(o.twin) : nullptr, p.enc == Encoding::ALAW ? 1 : 0, K,
                  s.max_out, st);
}

// FLAC: 4096 samples a frame, byte offsets found by the encoder; MP3: frame counts and bytes in closed form.
StreamTables stream_tables(const OutputPlan& p, const std::vector<long long>& soff) {
  const bool flac = p.enc == Encoding::FLAC;
  StreamTables t;
  const int P = t.P = (int)soff.size() - 1;
  std::vector<int> foff(P + 1, 0);
  t.boff.assign(P + 1, 0);
  for (int k = 0; k < P; k++) {
    const long long n = soff[k + 1] - soff[k];
    if (flac && n > kMaxFlacSamples) throw ArgError("program too long for one FLAC stream (2^36 - 1 samples at most)");
    const long long nf = flac ? flac_frames(n) : mp3_frames(p.mp3, n);
    if (foff[k] + nf > 0x7FFFFFFFLL) throw ArgError(flac ? "batch too long for one FLAC encode" : "batch too long for one MP3 encode");
    foff[k + 1] = foff[k] + (int)nf;
    if (!flac) t.boff[k + 1] = t.boff[k] + mp3_bytes(p.mp3, nf);
  }
  t.F = foff[P];
  t.bound = flac ? (size_t)flac_bound(P, t.F, soff[P]) : (size_t)t.boff[P];
  const TableLayout L(P);
  const size_t consts = flac ? 0 : mp3_const_bytes();
  t.dev_bytes = L.work + (flac ? flac_work_bytes(t.F) : consts);
  t.host.assign(L.work + consts, 0);
  memcpy(t.host.data(), soff.data(), (size_t)(P + 1) * sizeof(long long));
  memcpy(t.host.data() + L.boff, t.boff.data(), (size_t)(P + 1) * sizeof(long long));
  memcpy(t.host.data() + L.foff, foff.data(), (size_t)(P + 1) * sizeof(int));
  if (!flac) mp3_consts(t.host.data() + L.work);
  return t;
}

void encode_streams(const OutputPlan& p, StreamTables& t, const short* pcm, void* tables, unsigned char* out,
                    cudaStream_t st) {
  const TableLayout L(t.P);
  char* base = static_cast<char*>(tables);
  const long long* soff = reinterpret_cast<const long long*>(base);
  long long* boff = reinterpret_cast<long long*>(base + L.boff);
  const int* foff = reinterpret_cast<const int*>(base + L.foff);
  if (p.enc == Encoding::FLAC) {
    launch_flac(pcm, soff, foff, t.P, t.F, p.rate, p.flac_lpc, base + L.work, out, boff, st);
    KKX_CUDA(cudaMemcpyAsync(t.boff.data(), boff, (size_t)(t.P + 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
  } else {
    launch_mp3(pcm, soff, foff, boff, t.P, t.F, p.mp3, base + L.work, out, st);
  }
}

void OutputBuffers::reserve(const OutputPlan& p, long long samples, long long n24, int P, const StreamTables& t,
                            cudaStream_t st) {
  const size_t twin_bytes = p.enc == Encoding::F32 ? 0 : (size_t)samples * bytes_per_sample(p.enc);
  const size_t rep_floats = p.measure ? (size_t)kReportRows * P : 0;
  grow(wave, round256((size_t)samples * sizeof(float)) + round256(twin_bytes) + rep_floats * sizeof(float), st);
  audio = wave.alloc<float>(samples);
  twin = twin_bytes ? wave.alloc_bytes(twin_bytes) : nullptr;
  report = rep_floats ? wave.alloc<float>(rep_floats) : nullptr;
  const size_t w24 = p.post ? round256((size_t)n24 * sizeof(float)) : 0;
  const size_t table_bytes = is_stream(p.enc) ? t.dev_bytes : 0;
  grow(work, w24 + (p.limit ? 2 * w24 : 0) + table_bytes, st);
  wav24 = p.post ? work.alloc<float>(n24) : nullptr;
  lim_p = p.limit ? work.alloc<float>(n24) : nullptr;
  lim_v = p.limit ? work.alloc<float>(n24) : nullptr;
  tables = table_bytes ? work.alloc_bytes(table_bytes) : nullptr;
  bytes = nullptr;
  if (is_stream(p.enc)) {
    grow(streams, t.bound, st);
    bytes = streams.alloc<unsigned char>(t.bound);
  }
}

}  // namespace kkx
