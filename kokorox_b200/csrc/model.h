// model.h -- weight set + forward pass orchestration of Kokoro-82M on one B200.
#pragma once
#include "common.h"
#include "kernels.h"
#include "output.h"
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

namespace kkx {

struct HostTensor {
  std::vector<int> shape;
  const float* data = nullptr;
  size_t numel = 0;
};

// The checkpoint as named fp32 host tensors (upstream state-dict names, weight-norm folded).  Two sources,
// dispatched on the file's magic -- OrtKoko::new receives the path of the downloaded model file
// (ort_koko.rs:31-35, ort_base.rs:27-33, hf_cache.rs:135-144), so kkx_create accepts that file as it is:
//   * "KKXW0001": the flat file kokorox_b200/weightfile.py writes (random-init recipe, .pth converter);
//   * an ONNX ModelProto (kokoro-v1.0.onnx / onnx/model*.onnx): onnx_loader.cu reads the protobuf wire format,
//     names the anonymised initialisers through the node graph and dequantises fp16 / int8 / 4-bit variants.
class WeightFile {
 public:
  explicit WeightFile(const std::string& path);
  const HostTensor& get(const std::string& name) const;
  bool has(const std::string& name) const { return t_.count(name) != 0; }
  // takes ownership of `data` (used by the ONNX reader); an existing entry of that name is replaced
  void put(const std::string& name, const std::vector<int>& shape, std::vector<float>&& data);
  void erase(const std::string& name) { t_.erase(name); }
  std::vector<std::string> names() const;
  const std::string& format() const { return format_; }   // "kkxw" or "onnx"

 private:
  void load_kkxw(const std::string& path);
  std::vector<char> buf_;
  std::deque<std::vector<float>> owned_;
  std::map<std::string, HostTensor> t_;
  std::string format_;
};
// onnx_loader.cu: fills `out` with the Kokoro-82M state dict recovered from an ONNX file image; throws IoError
// listing every tensor it could not resolve.
void load_onnx_weights(const std::string& path, const std::vector<char>& bytes, WeightFile& out);
// (name, shape) of every tensor of Kokoro-82M that WeightSet::load reads (onnx_loader.cu)
std::vector<std::pair<std::string, std::vector<int>>> kokoro_tensor_specs();

// bf16 weight [Co][ks][Cpad] + its TMA descriptor (tensor-core path)
struct TcW {
  void* w = nullptr;
  alignas(64) unsigned char tmap[128];
  // one CTA's half (128-row boxes) of a 256-wide weight tile for the CTA-pair conv; exists when the map's row count
  // (phase-stacked weights: all phases) is a multiple of 128
  alignas(64) unsigned char tmap_h[128];
  bool has_h = false;
  const void* pair_map(int co_tile) const { return co_tile >= 256 && co_tile % 256 == 0 && has_h ? tmap_h : nullptr; }
  int Cpad = 0, Ci = 0, Co = 0, ks = 0;
};
// split-TF32 weight: tf32-exact hi / lo fp32 planes [Co][ks][Cpad] + TMA descriptors
struct TcW32 {
  float* hi = nullptr; float* lo = nullptr;
  alignas(64) unsigned char tm_hi[128];
  alignas(64) unsigned char tm_lo[128];
  alignas(64) unsigned char tm_hi_c[128];   // half-height boxes (64 rows) for the 64-wide small-problem tiles (Co > 64 only)
  alignas(64) unsigned char tm_lo_c[128];
  bool has_c = false;
  int Cpad = 0, Ci = 0, Co = 0, ks = 0;
  // split-FP16 planes of w * 2^s (same layout, 2-byte elements) + their TMA descriptors; wscale16 = 2^-s
  void* h_hi = nullptr; void* h_lo = nullptr;
  alignas(64) unsigned char tm16_hi[128];
  alignas(64) unsigned char tm16_lo[128];
  alignas(64) unsigned char tm16_hi_c[128];
  alignas(64) unsigned char tm16_lo_c[128];
  float wscale16 = 1.f;
};
struct LstmW { float* wih = nullptr; float* bias = nullptr; float* whhT = nullptr; int in = 0; TcW32 t_ih; };
struct AdaBlkW {  // AdainResBlk1d (SURVEY A.6)
  int ci = 0, co = 0; bool up = false;
  float *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr, *w1x1 = nullptr;
  float *poolw = nullptr, *poolb = nullptr;
  int sty1 = 0, sty2 = 0;  // offsets into the per-item style-parameter table
  TcW t1, t2, t1x1;
  TcW32 s1, s2, s1x1;   // split-TF32 variants (predictor F0/N blocks)
};
struct ArbW {  // AdaINResBlock1 (SURVEY A.9)
  int c = 0, k = 0;
  float *w1[3], *b1[3], *w2[3], *b2[3], *a1[3], *a2[3];
  int s1[3], s2[3];
  TcW t1[3], t2[3];
};

struct Weights {
  // ALBERT
  float *word, *pos, *type, *emb_lnw, *emb_lnb, *map_w, *map_b;
  float *qkv_w, *qkv_b, *dense_w, *dense_b, *attn_lnw, *attn_lnb;
  float *ffn_w, *ffn_b, *ffo_w, *ffo_b, *full_lnw, *full_lnb;
  float *benc_w, *benc_b;
  TcW32 t_map, t_qkv, t_dense, t_ffn, t_ffo, t_benc, t_durp, t_tcnn[3];
  // predictor
  LstmW dur_lstm[3]; int dur_ada[3];
  LstmW pred_lstm, shared_lstm;
  float *durp_w, *durp_b;
  AdaBlkW f0blk[3], nblk[3];
  float *f0proj_w, *f0proj_b, *nproj_w, *nproj_b;
  // text encoder
  float* temb; float *tcnn_w[3], *tcnn_b[3], *tln_g[3], *tln_b[3]; LstmW te_lstm;
  // decoder
  AdaBlkW enc, dec[4];
  float *f0conv_w, *f0conv_b, *nconv_w, *nconv_b, *asr_w, *asr_b;
  // generator
  float *lin_w, *lin_b, *nc0_w, *nc0_b, *nc1_w, *nc1_b;
  ArbW nres[2], res[6];
  std::vector<float*> ups0, ups1;  // per-phase [2][Ci][Co]
  std::vector<TcW> tups0, tups1;   // per-phase bf16 [Co][2][Ci]
  TcW tups0_all, tups1_all;        // the phases stacked along Co (phase-fused launch): [s*Co][2][Ci]
  TcW t_nc0, t_nc1, t_asr;         // noise_convs (nc0 as an im2col GEMM, K = 12*22), asr_res
  float *ups0_b, *ups1_b, *post_w, *post_b;
  TcW t_post_arb; float* post_b128 = nullptr;   // conv_post zero-padded to 128 output channels for the fused kernel
  // style FC tables (all AdaIN / AdaLN fcs of one style half concatenated)
  float *sty_pro_w, *sty_pro_b, *sty_dec_w, *sty_dec_b;
  int sty_pro_n = 0, sty_dec_n = 0;
};

void arb_timing_dump();  // diagnostics (model_forward.cu); no-op unless KKX_ARB_TIMING=1

struct DebugStage { std::vector<float> data; long long rows = 0, cols = 0; };

struct Options {
  // 1 (default) = the benchmarked configuration: decoder + generator convs on tcgen05 with bf16 operands, predictor
  // on split-TF32 tensor cores; 0 = fp32 SIMT everywhere (verification mode, tightest parity, ~6x slower)
  int precision = 1;
  unsigned long long noise_seed = 0x5eed;
  int max_frames = 49152;
  int stft_replicate = 0;
  // latency path (calls of one utterance): replay the token phase from a CUDA graph keyed by the token count, and
  // run independent branches (text encoder | ALBERT + durations, F0 | N, harmonic source + noise blocks | decoder)
  // on two streams for batches of at most fork_max_batch utterances (their kernels do not fill the GPU)
  int latency_graphs = 1;
  int fork_max_batch = 4;
  // ALBERT attention kernel: 1 = tcgen05 / TMEM / TMA (kernels_attn.cu), 0 = the mma.sync kernel of round 1
  int attention_umma = 1;
  // split-precision GEMMs of the predictor path: 1 = fp16 hi/lo planes ("3xFP16": the same 22 significand bits as
  // 3xTF32 at half the operand bytes and twice the MMA rate), 0 = tf32 hi/lo planes
  int split_f16 = 1;
  // generator res-blocks: keep the residual stream between the three iterations of a block in bf16 (10 instead of
  // 16 bytes per row-channel and iteration; the k = 3 / k = 7 convs are HBM-bound)
  int stream_bf16 = 0;
  // ConvTranspose1d up-sampling: all phases in one launch (L2 serves the re-reads of the input) instead of s launches
  int fuse_phases = 1;
  // persistent split-FP16 GEMMs: CTA pairs (tcgen05 cta_group::2, 256 x 128 tiles, half the weight tile per CTA)
  int gemm_pair = 1;
  // ALBERT: LayerNorm and the FFN GEMM leave their results as split-FP16 operand planes for the next GEMM (no separate
  // fp32 -> planes pass; the FFN activation never exists in fp32)
  int fuse_planes = 1;
  // bf16 decoder convs with Co % 256 == 0: CTA pairs (256 x 256 tiles, half the weight tile per CTA, persistent)
  int conv_pair = 1;
  // generator stage 1: noise_convs[1] (22 -> 128, k = 1) as one fp32 store-stream pass that also emits the statistics of its
  // output (kernels_signal.cu pointwise_conv_stats_kernel) instead of bf16 plane + implicit GEMM + statistics pass
  int fuse_noise_stats = 1;
  // stage-1 up-sampling conv (256 -> 128, 6 phases): one CTA per 128-row m-tile loops over the phases with a pipeline that
  // runs across them (1 = two-stage ring, two CTAs per SM; 2 = three stages, one CTA per SM; 0 = one CTA per (tile, phase));
  // 3 = persistent CTAs that keep ONE phase's weights resident in shared memory and stream only activation tiles
  int ups_phase_loop = 3;
  // LSTM gate non-linearities on the SFU (ex2 / rcp approximations, |error| ~ 1e-7) in the tensor-core configuration;
  // precision = 0 always uses libm's expf / tanhf and IEEE division
  int lstm_fast_gates = 1;
  // sample rate of every waveform a run returns (kkx.h "out_rate"); 24000 = the model's own rate, no resampling
  int out_rate = 24000;
  // loudness normalisation (kkx.h): integrated-loudness target in 1/100 LUFS (0 = off) and true-peak ceiling in
  // 1/100 dBTP
  int loudness_target = 0;
  int true_peak_max = -100;
  // lookahead true-peak limiter (kkx.h "limiter"): 0 = off, 1 = on
  int limiter = 0;
  // EBU R128 loudness report (kkx.h "loudness_report"): 0 = off, 1 = measure every program (without a target or the
  // limiter: measure only, the output is unchanged)
  int loudness_report = 0;
  // FLAC linear prediction (kkx.h "flac_lpc_order"): 0 = off, 1..12 = one LPC candidate of that order per frame
  int flac_lpc_order = 0;
};

// Device-resident weights of one checkpoint on one GPU: every layout the kernels read (fp32 SIMT, bf16 / split-TF32
// tensor-core copies with their TMA descriptors).  Immutable after construction and shared by every session created
// from the same (file, device): the reference's servers build two or three sessions of one model (koko main.rs:1477,
// 1596; TTSManager koko.rs:129-142) and each OrtKoko::new re-loads the file; here the second kkx_create is free.
class WeightSet {
 public:
  static std::shared_ptr<const WeightSet> acquire(const std::string& path, int device);
  ~WeightSet();
  WeightSet(const WeightSet&) = delete;
  WeightSet& operator=(const WeightSet&) = delete;
  Weights W;
  int device = 0;
  size_t device_bytes = 0;
  std::string format;          // "kkxw" / "onnx"

 private:
  WeightSet() = default;
  void load(const WeightFile& wf);
  float* up(const std::vector<float>& v);
  TcW make_tc(const std::vector<float>& w_co_ks_ci, int Co, int ks, int Ci);
  TcW32 make_tc32(const std::vector<float>& w_co_ks_ci, int Co, int ks, int Ci);
  std::vector<void*> owned_;
};

// Hard limits that keep every row / sample index inside int32 and the frame arena inside one GPU (ADVICE r1):
constexpr float kMinSpeed = 0.1f, kMaxSpeed = 10.f;   // dur per token <= 50 / speed <= 500 frames
constexpr int kMaxItemFrames = 65536;                  // one utterance: <= 27 min of audio (120*T+1 rows fit int32;
                                                       // at out_rate 48000: 1 200 samples per frame, 7.9e7 per utterance)
// A program (kkx_infer_programs) has no frame cap of its own: its sample offsets, lengths and segment indices are 64-bit
// in every kernel that reads them.  Its FLAC stream counts samples in STREAMINFO's 36-bit field.
constexpr long long kMaxFlacSamples = (1LL << 36) - 1;

// A program table: item offsets p[0 .. P] of P runs of consecutive items, p[0] = 0, p[P] = B, strictly increasing.
// Throws ArgError otherwise.
void check_programs(int B, int P, const int32_t* p);

// Optional parts of a Model::gemm / Model::tc_conv launch, set by name; the defaults are a plain Linear (a k = 1 conv).
// The fields mean what they mean in ConvArgs (kernels.h): taps ks at input rows m + tap * dil - pad, output row
// m * ors + oro, epilogue activation eact, residual res (rows of Lres, shifted right by res_shift), scale oscale.
// tc_conv takes its taps from the weight and has neither the prologue nor the operand planes.
struct ConvOpt {
  int eact = ACT_NONE;
  int ks = 1, dil = 1, pad = 0;
  int ors = 1, oro = 0;
  // prologue on the input operand: pact(x * pscale[b, c] + pshift[b, c]), LeakyReLU slope pslope
  const float* pscale = nullptr; const float* pshift = nullptr; int pact = ACT_NONE; float pslope = 0.f;
  const float* res = nullptr; int ldr = 0; const Level* Lres = nullptr; int res_shift = 0;
  float oscale = 1.f;
  // Operand planes handed from producer to consumer without the fp32 round trip (gemm, split-FP16 path only):
  //   in_hi / in_lo   the input already exists as fp16 hi / lo planes [Lin.rows, Cpad of the weight] (written by the
  //                   LayerNorm before, or by the GEMM before): no apply pass;
  //   out_hi / out_lo ask the GEMM to leave its result as planes [rows, out_ld] for the next GEMM INSTEAD of the fp32
  //                   output; honoured only by the CTA-pair kernel -- gemm returns whether it happened (otherwise the
  //                   fp32 output was written as usual);
  //   attn_scratch    the same for the QKV projection and the planes of launch_attention_umma.
  const void* in_hi = nullptr; const void* in_lo = nullptr;
  void* out_hi = nullptr; void* out_lo = nullptr; int out_ld = 0;
  float* attn_scratch = nullptr;
};

class Model {
 public:
  Model(const std::string& weights_path, int device);
  ~Model();

  // Stage inputs on the device (H2D), run the forward pass, fetch results (D2H).  stage() validates everything
  // before it touches the session state, so a rejected batch leaves the previous one intact; run() needs a staged
  // batch and fetch() a completed run (StateError otherwise).
  void stage(int B, const int64_t* tokens, const int32_t* tok_offsets, const float* styles,
             const float* speeds);
  // styles taken from the device-resident voice table (load_voices) instead of host vectors
  void load_voices(const float* table, int n_voices);
  void stage_voices(int B, const int64_t* tokens, const int32_t* tok_offsets, const int32_t* mix_offsets,
                    const int32_t* voice_ids, const float* portions, const int32_t* style_rows, const float* speeds);
  // Optional host sink for the waveform: called once the total sample count is known (after the token phase);
  // returns a pinned buffer of >= n floats.  Each frame group's audio is then copied to it on a second stream as
  // soon as the group's iSTFT is done, overlapping the device->host copy with the next group's kernels.
  std::function<float*(long long)> host_sink;
  bool sink_filled() const { return sink_filled_; }
  // A FLAC or MP3 run launches the encoder (kernels_flac.cu, kernels_mp3.cu) after the forward pass: gpu_us does not
  // include it.  kbps: the MP3 bitrate (mp3_format; 0 = the default), ignored by the other encodings.
  // programs: the run's program table (check_programs, P + 1 item offsets); every output -- sample offsets, the
  // encoded bytes, FLAC streams, loudness -- is per program, a program being one utterance whose 24 kHz waveform is
  // the concatenation of its items' (kkx.h, kkx_infer_programs).  Empty = one item per program.
  void run(Encoding enc = Encoding::F32, const std::vector<int>& programs = {}, int kbps = 0);
  long long total_samples() const { return total_samples_; }
  // The f32 waveform of the last run, whatever its encoding; sample_offsets [P + 1] per program.
  void fetch(float* dst, long long capacity, int64_t* sample_offsets, int32_t* pred_dur);
  // The output of the last run in its encoding: 4 bytes per sample for F32, 2 for PCM16, 1 for G.711, the FLAC or
  // MP3 streams back to back.  byte_offsets [P + 1] locate each program's bytes.
  long long encoded_bytes() const;
  void fetch_encoded(void* dst, long long capacity_bytes, int64_t* byte_offsets, int64_t* sample_offsets,
                     int32_t* pred_dur);
  // The report of the last run's programs (output.h): the row groups it produced (kRepLoudness | kRepRange |
  // kRepLimiter; 0 = none), and then last_report() holds kReportRows floats per program k at kReportRows k, in the
  // device table's row order.
  unsigned report_groups() const { return ran_ ? plan_.groups() : 0; }
  const std::vector<float>& last_report() const { return report_; }

  void set_noise(const float* noise, long long n);
  void set_inject(const std::string& name, int item, const void* data, long long count);
  void set_debug(bool on, int item = -1) { debug_ = on; debug_item_ = item; }
  const DebugStage* debug_stage(const std::string& name, int item) const;
  const std::vector<int>& group_first() const { return group_first_; }   // first item of each frame group of the last run

  Options opt;
  LaunchStats stats;
  long long last_frames = 0;
  double last_gpu_us = 0;
  std::map<std::string, std::pair<long long, double>> prof_;  // kernel -> (launches, total us)
  int device() const { return device_; }
  cudaStream_t stream() const { return stream_; }
  const WeightSet& weight_set() const { return *ws_; }
  long weight_sessions() const { return ws_.use_count(); }   // sessions sharing this device weight set

 private:
  struct Run {  // per-call state
    float* d = nullptr;        // [R,640]  DurationEncoder output (A.3)
    float* t_en = nullptr;     // [R,512]  TextEncoder output (A.4)
    float* sty_pro = nullptr;  // [B, sty_pro_n] predictor-side AdaIN/AdaLN parameters
    float* sty_dec = nullptr;  // [B, sty_dec_n] decoder-side AdaIN parameters
    int* pred_dur = nullptr;   // [R]
    int* cum = nullptr;        // [B,512] exclusive prefix sums of pred_dur
    int* total = nullptr;      // [B]     T_b
    std::vector<int> T;        // frames per item (host)
    Level styL;                // one item of B rows (style FC GEMMs)
  };
  // Linear / Conv1d on the precision-critical path: split-TF32 tensor cores when precision==1 and
  // the weight has a TcW32, fp32 SIMT otherwise.  Returns true when the result went to the operand planes of `o`
  // instead of `out`.
  bool gemm(const Level& Lin, const Level& Lm, const float* in, int ldi, int K, const float* w, const TcW32* w32,
            const float* bias, int N, float* out, int ldo, int ocol, const ConvOpt& o = ConvOpt());
  bool planes_ok() const { return opt.precision == 1 && opt.split_f16 && opt.fuse_planes; }
  float* split_hi_ = nullptr; float* split_lo_ = nullptr; size_t split_cap_ = 0;  // scratch planes (floats) of the current lane
  // Two execution lanes: lane 0 = stream_, lane 1 = stream2_ (forked branches of small batches).  cur_ is the stream
  // every launcher of the forward pass uses; each lane has its own split-TF32 scratch planes.
  struct Lane { float* hi = nullptr; float* lo = nullptr; size_t cap = 0; };
  Lane lane_[2];
  int lane_id_ = 0;
  void set_lane_scratch(int i, float* hi, float* lo, size_t cap) { lane_[i].hi = hi; lane_[i].lo = lo; lane_[i].cap = cap; if (i == lane_id_) use_lane(i); }
  void use_lane(int i) {
    lane_id_ = i; cur_ = i ? stream2_ : stream_;
    split_hi_ = lane_[i].hi; split_lo_ = lane_[i].lo; split_cap_ = lane_[i].cap;
  }
  void fork_lane1();   // lane 1 starts after everything issued so far on lane 0
  void join_lane1();   // lane 0 continues after everything issued so far on lane 1
  bool can_fork(int B) const { return B <= opt.fork_max_batch && !debug_ && !stats.profile && !stats.check_each; }
  // bf16 tensor-core conv of the operand buffer `abuf` [rows_total, w.Cpad]
  void tc_conv(const void* abuf, int rows_total, const TcW& w, const Level& Lin, const Level& Lm, const float* bias,
               float* out, int ldo, int ocol, const Level& Lout, const ConvOpt& o = ConvOpt());
  void token_phase(Run& r);          // graph replay or eager issue, then the one host sync of the call
  void token_issue(Run& r);          // every token-rate launch + the D2H of frame counts / durations (no sync)
  void token_finish(Run& r);         // sync, read T_b, validate
  size_t token_arena_bytes() const;
  // items [b0, b1); programs [k0, k1) are those whose last item is in the group (post-processed after it)
  void frame_phase(Run& r, int b0, int b1, int k0, int k1, bool dry);
  void adain_blk(Arena& A, const AdaBlkW& w, const float* x, int ldx, const Level& Lin, const Level& Lout,
                 const float* sty, int sld, float* out, int ldo, int ocol);
  void arb(Arena& A, const ArbW& w, const float* x, const Level& L, const float* sty, int sld, float* xw, float* t1,
           float* out, float oscale, bool accumulate, const float* part_x = nullptr, const void* x_bf16 = nullptr);
  bool use_stream_bf16(int C, int k, int B) const;
  // generator up-sampling: ConvTranspose1d(Ci, Co, k = 2s, stride s, padding s/2) of LeakyReLU(0.1)(x), x [Lin rows,
  // Ci] -> out [Lout rows, Co], as s two-tap phase convs whose output rows are shifted by `shift`.  w_all: the phases
  // stacked (one launch for all); w_tc / w32: one bf16 / fp32 weight per phase.  No phase-fused launch when `dry`.
  void upsample(Arena& A, const float* x, const Level& Lin, float* out, const Level& Lout, int s, int shift,
                const TcW& w_all, const std::vector<TcW>& w_tc, const std::vector<float*>& w32, const float* bias,
                bool dry);
  // generator stage after its up-sampling: x += x_source xs, then acc = the mean of the three res-blocks w[0..2] of x
  // (sty: the items' decoder-side style parameters; xw / t: the res-blocks' work buffers)
  void res_stage(Arena& A, const ArbW* w, float* x, const float* xs, const Level& L, const float* sty, float* xw,
                 float* t, float* acc);
  // first_off: row offset of item 0 (kGapRows for activations; 0 for the per-item style tables)
  Level make_level(const std::vector<int>& lens, Arena& A, int first_off = kGapRows);
  // copy `bytes` of host data to device memory through the pinned staging arena (true async copy on stream_)
  void upload(void* dst, const void* src, size_t bytes);
  void capture(const char* name, const float* p, int ld, int col, int cols, const Level& L,
               int item0);
  bool want_debug(int item) const { return debug_ && (debug_item_ < 0 || debug_item_ == item); }

  int device_ = 0;
  std::shared_ptr<const WeightSet> ws_;
  const Weights& W;
  cudaStream_t stream_ = nullptr;
  cudaStream_t stream2_ = nullptr;   // lane 1
  cudaStream_t cur_ = nullptr;       // stream of the current lane
  cudaEvent_t ev_fork_ = nullptr, ev_join_ = nullptr;
  // token-phase CUDA graphs of single-utterance calls: key = token count + every address the captured nodes embed
  struct GraphKey {
    int n_tokens, precision; const void *tok_base, *io_ids, *io_level, *h_T, *h_dur;
    bool operator<(const GraphKey& o) const {
      return std::tie(n_tokens, precision, tok_base, io_ids, io_level, h_T, h_dur) <
             std::tie(o.n_tokens, o.precision, o.tok_base, o.io_ids, o.io_level, o.h_T, o.h_dur);
    }
  };
  struct GraphEntry { cudaGraphExec_t exec = nullptr; Run run; long long launches = 0; };
  std::map<GraphKey, GraphEntry> graphs_;
  PinnedArena graph_pin_;            // staging of uploads captured into graphs: must outlive the call, never reset
  bool capturing_ = false;
  void clear_graphs();
 public:
  long long graph_replays = 0;
 private:
  Arena tokA_, frA_, ioA_;
  PinnedArena pin_;
  bool debug_ = false; int debug_item_ = -1;
  std::map<std::string, DebugStage> dbg_;
  // staged inputs
  int B_ = 0;
  bool staged_ = false, ran_ = false;
  std::vector<int> tok_len_;
  int* d_ids_ = nullptr; float* d_styles_ = nullptr; float* d_speeds_ = nullptr;
  Level tokL_;
  // the output stage of the current run: its plan, buffers, encoder tables (FLAC / MP3: the programs' byte offsets)
  // and the host copy of its report (program-major)
  OutputPlan plan_;
  OutputBuffers out_;
  StreamTables streams_;
  std::vector<float> report_;
  // program table of the current run (P + 1 item offsets); s24_off_ [B + 1]: each item's offset in the run's 24 kHz
  // waveform, where a program is contiguous
  std::vector<int> prog_;
  std::vector<long long> s24_off_;
  int n_prog() const { return (int)prog_.size() - 1; }
  float* d_voices_ = nullptr; int n_voices_ = 0;                           // [V][511][256] voice table
  std::vector<long long> sample_off_;                                      // [P + 1] at the output rate
  int* h_pred_dur_ = nullptr; size_t h_pred_dur_cap_ = 0;                  // pinned: per-row integer durations of the last run
  int* h_T_ = nullptr; size_t h_T_cap_ = 0;                                // pinned: frames per item
  long long total_samples_ = 0;
  std::vector<int> group_first_;
  // test hooks
  float* d_noise_ = nullptr; long long noise_n_ = 0;
  std::map<int, std::vector<int>> inj_dur_;
  std::map<int, std::vector<float>> inj_f0_, inj_n_;
  cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
  cudaStream_t copy_stream_ = nullptr; cudaEvent_t ev_grp_ = nullptr; bool sink_filled_ = false;
};

}  // namespace kkx
