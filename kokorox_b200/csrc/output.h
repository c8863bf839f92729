// output.h -- what a run does with its waveform after the iSTFT (output.cu): the plan of the run, the per-program span
// tables, the output buffers, the loudness / limiter / resampling pass and the FLAC / MP3 encoder.
#pragma once
#include "common.h"
#include "kernels.h"
#include <vector>

namespace kkx {

struct Options;

// What a run returns besides the f32 waveform, which every run writes: its 16-bit PCM twin, the G.711 codes of that
// PCM (mu-law / A-law), or one FLAC or MP3 stream per item encoded from it (kkx.h).
enum class Encoding { F32, PCM16, ULAW, ALAW, FLAC, MP3 };
inline bool is_stream(Encoding e) { return e == Encoding::FLAC || e == Encoding::MP3; }
inline long long bytes_per_sample(Encoding e) {
  return e == Encoding::F32 ? sizeof(float) : e == Encoding::ULAW || e == Encoding::ALAW ? 1 : sizeof(short);
}

// The per-program report of a run: one [kReportRows][P] float table on the device, rows
//   0 lufs, 1 dBTP, 2 gain | 3 LRA, 4 max momentary, 5 max short-term | 6 t, 7 max reduction (dB), 8 output dBTP
// (the gain and the limiter's static trim t feed the resampling pass).  A run produces some of the row groups:
constexpr int kReportRows = 9;
enum : unsigned { kRepLoudness = 1, kRepRange = 2, kRepLimiter = 4 };

// Everything after the iSTFT that a run's options, encoding and bitrate decide.
struct OutputPlan {
  Encoding enc = Encoding::F32;
  int rate = 24000;                     // the output rate
  int flac_lpc = 0;                     // FLAC: the LPC order (kkx.h "flac_lpc_order"), 0 = off
  bool loud = false;                    // normalise to a loudness target
  bool limit = false;                   // the lookahead limiter
  bool report = false;                  // the loudness report
  bool measure = false;                 // the loudness kernels run (any of the three)
  // The post-processing pass runs: the iSTFT writes a 24 kHz waveform that is measured, limited and resampled
  // (U = D = 1: a pass-through that applies the gain and the encoding).  Otherwise the iSTFT writes the output.
  bool post = false;
  int U = 1, D = 1, H = 0;              // resampling ratio U / D, filter half length H
  const float* taps = nullptr;          // device, 2H + 1 (none at 24 kHz)
  LoudParams par{};
  Mp3Format mp3{};
  bool law() const { return enc == Encoding::ULAW || enc == Encoding::ALAW; }
  bool pcm() const { return enc == Encoding::PCM16 || is_stream(enc); }
  unsigned groups() const {
    return (loud || report ? kRepLoudness : 0) | (report ? kRepRange : 0) | (limit ? kRepLimiter : 0);
  }
  long long out_len(long long n24) const { return (n24 * U + D - 1) / D; }   // samples of a program of n24
};

// Consecutive programs of a 24 kHz waveform and where their output goes.  `host` holds the table [4][n] (in_off |
// in_len | out_off | seg_off) to be uploaded as one block; place() points the device rows into that block.
struct Spans {
  int n = 0;
  long long nseg = 0, max_len = 0, max_out = 0;   // loudness segments in all, the longest input and output
  long long in_end = 0, out_end = 0;              // one past the last program's input and output
  std::vector<long long> host;
  const long long *in_off = nullptr, *in_len = nullptr, *out_off = nullptr, *seg_off = nullptr;
  size_t bytes() const { return host.size() * sizeof(long long); }
  void place(const long long* dev) {
    in_off = dev; in_len = dev + n; out_off = dev + 2 * n; seg_off = dev + 3 * n;
  }
};
// len24: the programs' 24 kHz lengths; they lie back to back from in0 and write back to back from out0, each
// ceil(len U / D) samples.
Spans make_spans(const std::vector<long long>& len24, long long in0, long long out0, int U, int D);

// The FLAC / MP3 encoder's tables of a run: frames per program as a prefix (foff), the programs' byte offsets (MP3:
// known from the frame counts; FLAC: found by the encoder, valid once encode_streams' stream is done).  `host` is the
// device table block's upload: soff | boff | foff, and MP3's analysis constants.
struct StreamTables {
  int P = 0, F = 0;
  std::vector<long long> boff;
  size_t bound = 0;                 // bytes of encoded output
  size_t dev_bytes = 0;             // the device block (the FLAC encoder's work area after the uploaded part)
  std::vector<unsigned char> host;
};
// soff [P + 1]: sample offsets of the programs.  Throws ArgError when a program or the batch is too long.
StreamTables stream_tables(const OutputPlan& p, const std::vector<long long>& soff);
// Launches the encoder on pcm (laid out as soff) into out; `tables` = the device copy of t.host (t.dev_bytes).
void encode_streams(const OutputPlan& p, StreamTables& t, const short* pcm, void* tables, unsigned char* out,
                    cudaStream_t st);

// A Model's output memory, grow-only: what the caller fetches (waveform, its encoding, the report), the encoded
// streams, and the run's 24 kHz waveform, limiter and encoder-table scratch.  An arena is re-reserved only after the
// stream is done with it.
struct OutputBuffers {
  Arena wave, streams, work;
  float* audio = nullptr;            // [samples] the f32 waveform at the output rate
  void* twin = nullptr;              // its 16-bit PCM or G.711 twin
  float* report = nullptr;           // [kReportRows][P]
  unsigned char* bytes = nullptr;    // FLAC / MP3 streams
  float* wav24 = nullptr;            // the 24 kHz waveform, item b at its run-wide offset
  float* lim_p = nullptr;            // limiter: the detector and the limited waveform, indexed like wav24
  float* lim_v = nullptr;
  void* tables = nullptr;            // the encoder's table block
  float* d_taps = nullptr; int taps_rate = 0;   // the resampling filter of taps_rate
  ~OutputBuffers() { if (d_taps) cudaFree(d_taps); }
  // samples at the output rate, n24 at 24 kHz, P programs; t: the encoder's tables (streams only)
  void reserve(const OutputPlan& p, long long samples, long long n24, int P, const StreamTables& t, cudaStream_t st);
};

// The plan of a run; uploads the resampling filter into `buf` when the rate changed.  Throws ArgError for an
// unsupported out_rate or MP3 bitrate.
OutputPlan output_plan(const Options& opt, Encoding enc, int kbps, OutputBuffers& buf, cudaStream_t st);

// The post-processing pass over programs [k0, k0 + s.n) of P, whose 24 kHz waveform o.wav24 is complete: loudness,
// the report, the limiter, then resampling into o.audio / o.twin.  Scratch comes from `scratch`.
void post_programs(const OutputPlan& p, const Spans& s, const OutputBuffers& o, int k0, int P, Arena& scratch,
                   cudaStream_t st);

}  // namespace kkx
