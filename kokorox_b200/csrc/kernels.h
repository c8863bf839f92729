// kernels.h -- launchers for the hand-written sm_100a kernels of the Kokoro-82M forward pass.
// Activations are time-major [rows, C] fp32 ("NLC"), ragged items packed along rows (Level).
#pragma once
#include "common.h"
#include <cuda_bf16.h>

namespace kkx {

enum Act : int { ACT_NONE = 0, ACT_LRELU = 1, ACT_SNAKE = 2, ACT_GELU_NEW = 3 };

// Generic fp32 "shifted GEMM": Conv1d / ConvTranspose1d phase / Linear, with a fused
// normalise+activate prologue on the input operand and a fused bias/activation/residual/scale
// epilogue.  For item b and m in [0, m_len[b]):
//   out[out_off[b] + m*ors + oro, ocol + n] (+)= oscale * ( eact( bias[n] +
//        sum_{tap<ks} sum_{c<Ci} A(in_off[b] + m*stride + tap*dil - pad, c) * w[tap][c][n] )
//        + res[res_off[b] + ((m*ors+oro) >> res_shift), rcol + n] )
//   A(r, c) = pact( in[r, c] * pscale[b, c] + pshift[b, c] ) for 0 <= r - in_off[b] < in_len[b], else 0
struct ConvArgs {
  const float* in = nullptr; int ldi = 0;
  const int* in_off = nullptr; const int* in_len = nullptr;
  const int* m_len = nullptr; int max_m = 0; int B = 1;
  long long sum_m = 0;  // sum of m_len over items (host copy; FLOP accounting only)
  const float* w = nullptr; const float* bias = nullptr;
  int Ci = 0, Co = 0, ks = 1, dil = 1, pad = 0, stride = 1;
  const float* pscale = nullptr; const float* pshift = nullptr; int pld = 0;
  int pact = ACT_NONE; float pslope = 0.f; const float* palpha = nullptr;
  float* out = nullptr; int ldo = 0; int ocol = 0; const int* out_off = nullptr;
  int ors = 1, oro = 0;
  int eact = ACT_NONE;
  const float* res = nullptr; int ldr = 0; int rcol = 0; const int* res_off = nullptr;
  int res_shift = 0;
  float oscale = 1.f; int accumulate = 0;
};
void launch_conv_f32(const ConvArgs& a, cudaStream_t st);

// Tensor-core (tcgen05) variant of the shifted GEMM, stride 1 only: bf16 operands fetched by TMA
// (A = activations [rows_total, Cpad] with zero gap rows / pad columns, B = weights
// [Co, ks*Cpad]), fp32 accumulation in TMEM, fp32 epilogue (bias, residual, scale, accumulate).
struct TcConvArgs {
  const void* tmA = nullptr;  // host pointers to CUtensorMap objects (copied into kernel params)
  const void* tmB = nullptr;
  const void* tmA2 = nullptr; // split-TF32 mode: the "lo" planes
  const void* tmB2 = nullptr;
  const void* tmB_c = nullptr;   // weight maps with half-height boxes: a CTA's half of the weight tile in the CTA-pair
  const void* tmB2_c = nullptr;  // kernels, and the 64-wide tiles of the small-problem split-precision kernel
  int debug = 0;  // KKX_TC_DEBUG bit mask (perf experiments): 1 skip global stores, 2 skip MMA issue, 4 skip TMEM loads
                  // (placed here, it keeps wscale / eact 8-byte aligned: the epilogue reads them with one 64-bit load)
  int tf32 = 0;               // 1 = split-precision operands (hi / lo planes), nprod products (3 or 4)
  int nprod = 3;
  int f16 = 0;                // split planes are fp16 (2 B, 64 K-elements per 128-byte span) instead of tf32-in-fp32:
                              // the same 11-bit significands, half the operand bytes and twice the MMA rate
  float wscale = 1.f;         // the accumulator is multiplied by this before the bias (undoes the power-of-two
                              // scaling of fp16 weight / activation planes; 1 for tf32)
  int eact = ACT_NONE;
  int Cpad = 0, Ci = 0, Co = 0, ks = 1, dil = 1, pad = 0;
  const int* in_off = nullptr; const int* m_len = nullptr; int max_m = 0; int B = 1; long long sum_m = 0;
  const float* bias = nullptr;
  float* out = nullptr; int ldo = 0; int ocol = 0; const int* out_off = nullptr; int ors = 1, oro = 0;
  const float* res = nullptr; int ldr = 0; int rcol = 0; const int* res_off = nullptr; int res_shift = 0;
  float oscale = 1.f; int accumulate = 0; int vec4 = 0;
  long long* timing = nullptr;   // diagnostics (-DKKX_TC_TIMING builds)
  const int* tile_start = nullptr; int ntiles_m = 0;   // persistent split-TF32 GEMM: prefix sum of ceil(m_len/128) per item
  int group_m = 1;               // (set by the launcher) m-tiles per L2-resident group
  // persistent CTA-pair kernel only: also (or, with out == nullptr, only) write the result as split-FP16 operand planes
  // [rows, out_pl_ld] (hi / lo halves of 16 * value, like launch_apply_f16x2) for the GEMM that consumes it next
  void* out_hi = nullptr; void* out_lo = nullptr; int out_pl_ld = 0;
  // persistent CTA-pair kernel only, QKV projection of ALBERT (Co = 2304): write the result directly as the attention
  // kernel's operand planes (kernels_attn.cu: fp16 hi / lo of 2 q and 16 k, row-major [rows, 768], and of 16 v
  // transposed per head, [(item, head, d), key] with pitch 512 and zero-filled to a multiple of 64 keys) instead of fp32:
  // attn_pl = {qh, ql, kh, kl, vth, vtl}
  void* attn_pl[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int pair = 0;                  // persistent split-FP16 GEMM: CTA pairs (cta_group::2, 256 x 128 tiles) when tmB_c / tmB2_c exist
  int force_kernel = 0;          // tests: 1 = never take the small-problem (64-wide single-tile) kernel
  // Phase-fused ConvTranspose1d (bf16 path, MODE 0): `nphase` two-tap phase convs in ONE launch.  The weights of the
  // phases are stacked along the weight map's rows (phase p at rows [p*Co, (p+1)*Co)), each phase has its own tap shift
  // and output row offset, and the phase is the FASTEST grid dimension, so the CTAs that read one activation tile run
  // together and the re-reads are served from L2 instead of HBM (the phases used to be 10 + 6 separate launches).
  int nphase = 1;
  int phase_pad[10] = {0};
  int phase_oro[10] = {0};
  int phase_loop = 0;            // Co = 128 only: one CTA per m-tile loops over the phases (conv_tc_multi_kernel)
};
void launch_conv_tc(const TcConvArgs& a, cudaStream_t st);
// true when launch_conv_tc will run the CTA-pair kernel for these arguments (the only kernel that honours out_hi / out_lo)
bool conv_tc_takes_pair(const TcConvArgs& a);
// out_map: 128-byte CUtensorMap storage (64-byte aligned).  bf16 [outer, inner], box [box_outer, 64].
void make_tmap_bf16(void* out_map, const void* ptr, long long inner, long long outer,
                    long long pitch_elems, int box_outer);
void make_tmap_f32(void* out_map, const void* ptr, long long inner, long long outer,
                   long long pitch_elems, int box_outer);
void make_tmap_f16(void* out_map, const void* ptr, long long inner, long long outer,
                   long long pitch_elems, int box_outer);
inline int tc_box_n(int Co) { return Co > 128 ? 256 : (Co > 64 ? 128 : 64); }
inline int tc_box_n_tf32(int Co) { return Co > 64 ? 128 : 64; }
void launch_apply_tf32(const float* x, int ldx, int C, const float* scale, const float* shift, int act,
                       float slope, float* out_hi, float* out_lo, int Cpad, int rows_total,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st);
// fp16 hi / lo planes of kSplitF16Scale * act(x * scale + shift) (saturating at the fp16 range), [rows, Cpad] halves
constexpr float kSplitF16Scale = 16.f;
// host: fp16 hi / lo planes of w * 2^s, s chosen so that max|w| * 2^s lies in [2^13, 2^14) (the lo plane of every
// weight down to 2^-14 of the largest then stays a normal fp16); returns 2^-s
float split_f16_host(const float* w, size_t n, unsigned short* hi, unsigned short* lo);
void launch_apply_f16x2(const float* x, int ldx, int C, const float* scale, const float* shift, int act,
                        float slope, void* out_hi, void* out_lo, int Cpad, int rows_total,
                        const int* off, const int* len, int B, int max_len, cudaStream_t st);
// bf16 operand producers (AdaIN scale/shift + activation fused; zero halo rows and pad columns)
void launch_apply_bf16(const float* x, int ldx, int C, const float* scale, const float* shift, int act,
                       float slope, const float* alpha, void* out, int Cpad, int rows_total,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st);
void launch_im2col_bf16(const float* in, int ldi, int C, int ks, int stride, int pad, void* out, int Cpad,
                        int rows_total, const int* in_off, const int* in_len, const int* out_off,
                        const int* out_len, int B, int max_out_len, cudaStream_t st, int force_generic = 0);
void launch_pool_up_bf16(const float* in, int ldi, const float* scale, const float* shift, float slope,
                         const float* w, const float* bias, int C, void* out, int Cpad, int rows_total,
                         const int* in_off, const int* in_len, const int* out_off, int B, int max_len,
                         cudaStream_t st);

// Fused generator res-block conv (kernels_arb.cu): AdaIN scale/shift + Snake applied to the raw
// activations inside the kernel, every tap a row-shifted view of one smem halo tile, epilogue with
// bias / residual / scale / accumulate, fp32 and/or bf16 outputs and per-128-row column sums for
// the next AdaIN.  C = Ci = Co in {128, 256}; all tensors [rows, C] with the Level's row offsets.
struct ArbConvArgs {
  const void* x = nullptr; int in_bf16 = 0;           // raw input: fp32 or bf16 [rows, C]
  const float* scale = nullptr; const float* shift = nullptr;  // AdaIN coefficients [B][C]
  const float* alpha = nullptr;                        // Snake alpha [C]
  const void* tmB = nullptr;                           // host pointer to the weight CUtensorMap (bf16 [C][ks*C], box [C,64])
  int C = 0, ks = 1, dil = 1, pad = 0;
  const int* off = nullptr; const int* len = nullptr;  // Level (device)
  const int* tile_start = nullptr;                     // [B+1] prefix sum of ceil(len/arb_tile_rows(C))
  int B = 1; int total_tiles = 0; long long sum_m = 0;
  const float* bias = nullptr;
  __nv_bfloat16* out_bf16 = nullptr;                   // y (+res) as bf16, unscaled (nullable)
  float* out_f32 = nullptr;                            // (y + res) * oscale (+ previous value) (nullable)
  const float* res = nullptr; float oscale = 1.f; int accumulate = 0;
  int res_bf16 = 0;                                    // `res` points at bf16 data (bf16 residual stream); conv1 of such a
                                                       // stream has in_bf16 = 1, conv2 writes out_bf16 (next x) or out_f32
  float* part = nullptr; int nchunk = 0;               // column sums of (y + res): [B][nchunk][2][C], 128-row chunks
  long long* timing = nullptr;                         // diagnostics (-DKKX_ARB_TIMING builds): per-role phase cycle counters
  int debug = 0;                                       // diagnostics (-DKKX_EXPERIMENTS builds, wrong results): 1 = producers skip
                                                       // the global loads, 2 = epilogue skips the global stores / residual loads,
                                                       // 4 = producers skip the transform, 8 = MMA warp issues nothing but commits
  // "post" variant (generator conv_post): operand transform = LeakyReLU(slope) instead of AdaIN + Snake, weights
  // zero-padded to C output channels, fp32 output [rows, ldo] of the first `cout` channels, no statistics
  int post = 0, cout = 0, ldo = 0; float slope = 0.f;
};
int arb_tile_rows(int C);   // rows per persistent-kernel tile: 256 at C = 128 (transposed accumulator), 128 at C = 256
bool arb_conv_supported(int C, int ks, int dil, int B);
void launch_arb_conv(const ArbConvArgs& a, cudaStream_t st);

// y = act( LN(x (+res)) [* w + b] [(1+gamma_b) * . + beta_b] ), one row at a time.
struct LnArgs {
  const float* x = nullptr; int ldx = 0;
  const float* res = nullptr; int ldr = 0;
  const float* w = nullptr; const float* b = nullptr;         // affine [C] (nullable)
  const float* ada = nullptr; int ada_ld = 0; int ada_off = 0; // per-item gamma at ada_off, beta at ada_off+C
  float eps = 1e-5f; float slope = 1.f;                        // slope != 1 -> LeakyReLU
  float* out = nullptr; int ldo = 0; int ocol = 0;
  const int* off = nullptr; const int* len = nullptr; int B = 1; int max_len = 0; int C = 0;
  // optional second output: the result as split-FP16 operand planes [rows, pl_ld] (hi / lo halves of 16 * value, the
  // arithmetic of launch_apply_f16x2) for the GEMM that reads it next
  void* pl_hi = nullptr; void* pl_lo = nullptr; int pl_ld = 0;
};
void launch_layernorm(const LnArgs& a, cudaStream_t st);

// ALBERT embeddings: word[id] + pos[t] + type[0] -> LayerNorm(128, eps 1e-12).  out [rows,128]
void launch_albert_embed(const int* ids, const float* word, const float* pos, const float* type,
                         const float* lnw, const float* lnb, float* out, const int* off,
                         const int* len, int B, int max_len, cudaStream_t st);
// out[row, 0:C] = table[ids[row], :]
void launch_embed_rows(const int* ids, const float* table, int C, float* out, int ldo,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st);
// out[row, ocol + c] = vec[b*ldv + voff + c]  (broadcast a per-item vector over the item's rows)
void launch_bcast_cols(const float* vec, int ldv, int voff, int C, float* out, int ldo, int ocol,
                       const int* off, const int* len, int B, int max_len, cudaStream_t st);
// dst[row, dcol + c] = src[row, scol + c]
void launch_copy_cols(const float* src, int lds, int scol, float* dst, int ldd, int dcol, int C,
                      const int* off, const int* len, int B, int max_len, cudaStream_t st);
// out = a + b over the items' rows, C columns (all ld = C)
void launch_add_rows(const float* a, const float* b, float* out, int C, const int* off,
                     const int* len, int B, int max_len, cudaStream_t st);
// u[off[b] + dst_row] = u[off[b] + src_row] (ReflectionPad1d((1,0)) fix-up)
void launch_copy_row(float* u, int C, int dst_row, int src_row, const int* off, int B,
                     cudaStream_t st);

// softmax(QK^T/8)V per item and head; qkv [rows, 2304] (q|k|v, head h at h*64); ctx [rows,768]
void launch_attention(const float* qkv, float* ctx, const int* off, const int* len, int B,
                      int max_len, cudaStream_t st);

// The same on tcgen05 / TMEM fed by TMA (kernels_attn.cu): split-TF32 products, P kept in tensor memory as the A
// operand of the second MMA.  scratch: attention_umma_scratch_floats(rows_total, B) floats (tf32 hi/lo planes of
// Q/8, K and the transposed V); rows_total = rows of the packed qkv / ctx matrices (Level.rows).
size_t attention_umma_scratch_floats(int rows_total, int B);
void attention_timing_dump();   // diagnostics (-DKKX_TC_TIMING builds): role cycle counters of attn_umma_kernel; no-op otherwise
// planes_ready: the QKV GEMM already wrote the operand planes into `scratch` (TcConvArgs::attn_pl); qkv is not read.
void launch_attention_umma(const float* qkv, float* scratch, float* ctx, const int* off, const int* len, int B,
                           int max_len, int rows_total, cudaStream_t st, bool planes_ready = false);
// the six plane pointers inside an attention scratch buffer: qh, ql, kh, kl, vth, vtl
void attention_umma_planes(float* scratch, int rows_total, int B, void* (&pl)[6]);

// Bidirectional LSTM recurrence, H=256.  xproj [rows, 2048] = x W_ih^T + b_ih + b_hh for
// (fwd i,f,g,o | bwd i,f,g,o); whhT [2][256][1024] (k-major); out [rows, ldo] cols ocol..+512.
// variant: 1 = cluster kernel with SFU gate functions (the tensor-core configuration), 0 = cluster kernel with libm
// gate functions (fp32 configuration), -1 = one CTA per (item, direction) (plain kernel, tests only).
void launch_lstm(const float* xproj, const float* whhT, float* out, int ldo, int ocol,
                 const int* off, const int* len, int B, cudaStream_t st, int variant = 1);

// InstanceNorm statistics -> AdaIN coefficients.
//   partial sums over row chunks, then scale[b,c] = rstd*(1+gamma), shift[b,c] = beta - mean*scale
//   with gamma = sty[b*sld + soff + c], beta = sty[b*sld + soff + C + c].
constexpr int kStatRows = 128;
// out_bf16 (nullable, needs ldx == C): also write a bf16 copy [rows, C] of x -- the start of a bf16 residual stream
void launch_colstats(const float* x, int ldx, int C, float* part, const int* off, const int* len,
                     int B, int max_len, cudaStream_t st, void* out_bf16 = nullptr);  // part [B][nchunk_max][2][C]
// out = a + b (all [rows, C], row pitch C) and the chunk statistics of the sum, in one pass; with out_bf16 the sum is
// written ONLY as bf16 [rows, C] (statistics still from the fp32 sum) and `out` is left untouched
void launch_add_rows_stats(const float* a, const float* b, float* out, int C, float* part, const int* off,
                           const int* len, int B, int max_len, cudaStream_t st, void* out_bf16 = nullptr);
// out[r, co] = bias[co] + sum_ci x[r, ci] * w[ci][co] for Conv1d(22, 128, k = 1) (generator noise_convs[1]) and the chunk
// statistics of the result (same `part` layout as launch_colstats) in one pass; fp32 SIMT, store-bound
void launch_pointwise_conv_stats(const float* x, int ldx, int Ci, const float* w, const float* bias, float* out, int Co,
                                 float* part, const int* off, const int* len, int B, int max_len, long long sum_m,
                                 cudaStream_t st);
void launch_adain_coef(const float* part, int C, int max_len, const int* len, const float* sty,
                       int sld, int soff, float eps, float* scale, float* shift, int B,
                       cudaStream_t st);

// Depthwise ConvTranspose1d(k3,s2,p1,op1) on lrelu(x*scale+shift): in [T,C] -> out [2T,C]
void launch_pool_up(const float* in, int ldi, const float* scale, const float* shift, float slope,
                    const float* w /*[C][3]*/, const float* bias, int C, float* out, int ldo,
                    const int* in_off, const int* in_len, const int* out_off, int B, int max_len,
                    cudaStream_t st);

// Duration head (K4): dur = sum_k sigmoid(logits[row,k]) / speed_b -> rintf -> max(.,1)
void launch_duration(const float* logits, int K, const float* speeds, int* pred_dur,
                     float* dur_float, const int* off, const int* len, int B, int max_len,
                     cudaStream_t st);
// cum[b, n] = exclusive prefix sum of pred_dur over the item's tokens; total[b] = T_b
void launch_dur_scan(const int* pred_dur, int* cum, int cum_ld, int* total, const int* off,
                     const int* len, int B, cudaStream_t st);
// idx[fr_off[b] + j] = token n with cum[b,n] <= j < cum[b,n] + dur[n]
void launch_expand_idx(const int* cum, int cum_ld, const int* tok_len, int* idx, const int* fr_off,
                       const int* fr_len, int B, int max_len, cudaStream_t st);
// K5: out[out_off[b] + j, ocol + c] = in[in_off[b] + idx[idx_off[b] + j], c]
void launch_gather_rows(const float* in, int ldi, const int* in_off, const int* idx,
                        const int* fr_off, const int* fr_len, int C, float* out, int ldo, int ocol,
                        int B, int max_len, cudaStream_t st);

// Conv1d(1,1,k3,s2,p1) on a curve: x [2T] -> out[t, ocol] (ld ldo), t < T
void launch_curve_conv(const float* x, const int* x_off, const int* x_len, const float* w3,
                       const float* bias, float* out, int ldo, int ocol, const int* out_off,
                       const int* out_len, int B, int max_len, cudaStream_t st);

// K9 SineGen + SourceModuleHnNSF.
//   phase: per (item, harmonic) fp64 inclusive scan of frac(f0*h/24000) over 2T coarse steps,
//          stored as fp32 ((c*2)*pi)*300
//   source: per sample linear x300 interpolation of the coarse phase, sin, uv gating, noise,
//          Linear(9->1), tanh -> har_source [samples]
void launch_sine_phase(const float* f0, const int* f0_off, const int* f0_len, float* phase,
                       const int* ph_off /*per item, in floats*/, int B, cudaStream_t st);
void launch_sine_source(const float* f0, const int* f0_off, const int* f0_len, const float* phase,
                        const int* ph_off, const float* noise /*nullable, [t*9+h]*/,
                        unsigned long long seed, const float* lin_w, const float* lin_b,
                        float* out, const long long* s_off, int B, long long max_samples,
                        cudaStream_t st);
// K10 STFT (n_fft 20, hop 5, periodic hann, center): x [600T] -> har[row, 0:11]=|X|, [11:22]=angle
void launch_stft(const float* x, const long long* s_off, float* har, int ldh, const int* h_off,
                 const int* h_len, int replicate_pad, int B, int max_len, cudaStream_t st);
// K11 head: mag = exp(cp[:, :11]), ph = sin(cp[:, 11:]) -> iSTFT -> audio [600T]
//   fast != 0: SFU exp / sin / cos and a reciprocal envelope (tensor-core configuration); 0: libm + true division
void launch_istft(const float* cp, int ldc, const int* h_off, const int* h_len, float* audio, short* pcm /*nullable*/,
                  const long long* s_off, int fast, int B, int max_len, cudaStream_t st);

// Output sample-rate conversion 24 kHz -> out_rate (scipy.signal.resample_poly with its defaults), per utterance.
//   resample_ratio: U / D = out_rate / 24000 reduced; false unless 8000 <= out_rate <= 48000 and max(U, D) <= 320.
//   resample_design: the 2H + 1 fp32 taps U * firwin(2H + 1, 1 / max(U, D), ("kaiser", 5.0)), H = 10 max(U, D),
//                    designed in double on the host; returns the tap count, or -1 for a rejected rate.  24000 is the
//                    identity: one tap 1.0, H = 0 (firwin has no filter with cutoff 1; resample_poly copies its input).
//   launch_resample: item b reads x[in_off[b] .. + in_len[b]) and writes ceil(in_len[b] U / D) samples at out_off[b]
//                    as f32 and optionally as 16-bit PCM (trunc(clamp(y, -1, 1) * 32767)) and / or G.711 codes of that
//                    PCM value (law 0 = mu-law, 1 = A-law); U = D = 1 with H = 0 is a pass-through (no taps).
//                    max_out = largest per-item output length.  gain (nullable): every output y of item b is
//                    fp32(y * gain[b]) (loudness normalisation); null leaves the arithmetic as it is.
//                    Profile name "resample".
//   poly_design:     the taps of resample_poly(x, u, d) for any u / d (the true-peak filter uses 4 / 1).
bool resample_ratio(int out_rate, int* U, int* D);
int resample_design(int out_rate, std::vector<float>* taps, int* U, int* D, int* H);
int poly_design(int u, int d, std::vector<float>* taps);
void launch_resample(const float* x, const long long* in_off, const long long* in_len, const long long* out_off,
                     const float* taps, int U, int D, int H, const float* gain /*nullable*/, float* out,
                     short* pcm /*nullable*/, unsigned char* codes /*nullable*/, int law, int B, long long max_out,
                     cudaStream_t st);

// Loudness normalisation (kernels_loudness.cu, K14): ITU-R BS.1770 integrated loudness of each item's 24 kHz waveform
// with a true-peak ceiling (kkx.h "loudness_target").
//   loudness_design: the K-weighting biquads at fs in double (shelf b0 b1 b2 a1 a2, then high-pass b0 b1 b2 a1 a2)
//                    and, if tp_taps is given, the 81 taps of resample_poly(x, 4, 1).
//   LoudParams:      everything the kernels read, passed by value (fp32 biquads, the 4x taps, target and ceiling).
//   launch_loudness: item b = x[in_off[b] .. + in_len[b]); writes lufs[b] (NaN = undefined), tp_db[b] (dBTP) and
//                    gain[b].  energy: scratch of in_len[b] / 2400 floats per item at seg_off[b]; peak: [B] scratch.
//                    Three launches: "loud_energy", "loud_peak", "loud_gain".
constexpr int kLoudSeg = 2400, kLoudWarm = 4800, kTpTaps = 81;
struct LoudParams {
  float kw[10];
  float tp[kTpTaps];
  double target_lufs, ceiling_dbtp;
};
void loudness_design(double fs, double kw[10], std::vector<float>* tp_taps);
LoudParams loudness_params(double target_lufs, double ceiling_dbtp);
void launch_loudness(const float* x, const long long* in_off, const long long* in_len, const long long* seg_off,
                     const LoudParams& P, float* energy, unsigned* peak, float* lufs, float* tp_db, float* gain, int B,
                     long long max_len, cudaStream_t st);

// Lossless FLAC of 16-bit mono PCM (kernels_flac.cu; the bitstream rules are in kkx.h, kkx_infer_batch_flac).
//   Item b is pcm[soff[b] .. soff[b + 1]) (>= 1 sample) and has flac_frames(n_b) frames of 4096 samples; foff[b + 1]
//   is the prefix sum of those counts (F = foff[B] frames).  launch_flac writes item b's stream to
//   out[item_off[b] .. item_off[b + 1]) (item_off [B + 1], device); out must hold flac_bound(B, F, samples) bytes and
//   work flac_work_bytes(F).  rate: one of the nine "out_rate" values.  Three launches, profile names
//   "flac_analyze", "flac_scan", "flac_pack".
long long flac_frames(long long n);
long long flac_bound(long long n_items, long long n_frames, long long n_samples);
size_t flac_work_bytes(long long n_frames);
bool flac_rate_ok(int rate);
void launch_flac(const short* pcm, const long long* soff, const int* foff, int B, int F, int rate, void* work,
                 unsigned char* out, long long* item_off, cudaStream_t st);

// mix_styles (koko.rs:1255-1306) on a device-resident voice table [V][511][256]
void launch_mix_styles(const float* table, const int* mix_off, const int* voice_ids, const float* portions,
                       const int* rows, float* styles, int B, cudaStream_t st);

}  // namespace kkx
