/*
 * kkx_test.h -- test hooks of libkkx.so (parity harness only; the Rust shim binds nothing from
 * this header): whole-model hooks (noise / teacher forcing / stage dumps) and op-level entry
 * points.  The op-level calls take host pointers in and out, one ragged item; each allocates
 * device scratch, runs ONE hand-written kernel and copies the result back, so that tests/ can
 * compare a kernel against the matching torch op in isolation.
 */
#ifndef KKX_TEST_H_
#define KKX_TEST_H_
#include "kkx.h"
#ifdef __cplusplus
extern "C" {
#endif

/* ---- whole-model hooks (moved here from kkx.h: the parity harness is their only user) -------------------
 * kkx_set_noise: explicit SineGen noise, element (sample t, harmonic h) at noise[t*9+h]; n = number of floats;
 *   n == 0 returns to the on-device generator.  With a batch every item reads the same buffer from offset 0.
 * kkx_set_inject_item: teacher-force an intermediate of batch item `item` (any frame group) in every following
 *   call: name is "pred_dur" (int32 data, n_tokens entries in 1..500), "F0" or "N" (f32 data, 2T entries);
 *   count == 0 clears that item's entry.  kkx_set_inject is the item-0 form.
 * kkx_debug_enable / kkx_debug_select: keep stage tensors alive for kkx_debug_stage -- of every item, or of one
 *   item only (a B = 64 x 510 batch would otherwise hold tens of GB of host copies).
 * kkx_debug_stage: after a call, copy a named stage tensor of item `item` to host.  Returns the number of floats the
 *   stage holds (rows*cols) or <0; rows/cols are written if non-NULL; at most `capacity` floats are copied (dst may
 *   be NULL to query the size).  Stage names match oracle/kokoro_ref.py (`bert`, `d`, `dur_logits`, `F0`, ...). */
KKX_API int kkx_set_noise(kkx_ctx* ctx, const float* noise, int64_t n);
KKX_API int kkx_set_inject(kkx_ctx* ctx, const char* name, const void* data, int64_t count);
KKX_API int kkx_set_inject_item(kkx_ctx* ctx, int32_t item, const char* name, const void* data, int64_t count);
KKX_API int kkx_debug_enable(kkx_ctx* ctx, int enable);
KKX_API int kkx_debug_select(kkx_ctx* ctx, int enable, int32_t item);
KKX_API int64_t kkx_debug_stage(kkx_ctx* ctx, const char* name, int32_t item, float* dst, int64_t capacity,
                        int64_t* rows, int64_t* cols);

/* Generic shifted-GEMM kernel (Conv1d / ConvTranspose1d phase / Linear), see kernels.h ConvArgs.
 * in [rows_in, ldi]; w [ks][Ci][Co]; out [out_rows, Co] (pre-filled by the caller; rows not
 * written keep their value); res [ceil(out_rows >> res_shift), Co] or NULL. */
KKX_API int kkx_test_conv(int device, const float* in, int rows_in, int ldi, int Ci, const float* w,
                          const float* bias, int Co, int ks, int dil, int pad, int stride,
                          const float* pscale, const float* pshift, int pact, float pslope,
                          const float* palpha, int m_len, int ors, int oro, int out_rows,
                          const float* res, int res_rows, int res_shift, float oscale, int eact,
                          int accumulate, float* out);
/* xproj [N,2048], whhT [2][256][1024] -> out [N,512] */
KKX_API int kkx_test_lstm(int device, const float* xproj, const float* whhT, int N, float* out);
/* ragged batch: xproj [rows,2048], items at off[b] with len[b] rows -> out [rows,512] (pre-zeroed) */
KKX_API int kkx_test_lstm_batch(int device, const float* xproj, const float* whhT, int B, const int* off,
                                const int* len, int rows, float* out);
/* the same with an explicit kernel variant (1 = cluster kernel, SFU gate functions; 0 = cluster kernel, libm gate
   functions; -1 = plain one-CTA-per-item kernel) and the average device time of `reps` further launches */
KKX_API int kkx_test_lstm_batch_v(int device, const float* xproj, const float* whhT, int B, const int* off,
                                  const int* len, int rows, int variant, int reps, float* out, float* ms);
/* Conv1d(22, 128, k = 1) fused with the chunk statistics of its output (kernels_signal.cu): x [rows,24] (22 used),
   w [22][128], items at off[b] (len[b] rows) -> out [rows,128] (pre-filled by the caller), part [B][nchunk][2][128] with
   nchunk = ceil(max_len / 128); part_ref receives what launch_colstats computes from `out` */
KKX_API int kkx_test_pointwise_conv_stats(int device, const float* x, const float* w, const float* bias, int B,
                                          const int* off, const int* len, int rows, int max_len, float* out, float* part,
                                          float* part_ref);
/* row LayerNorm of x (+ res) [rows,C] with optional affine w / b [C], per-item AdaLN (ada = gamma [C] then beta [C]),
   LeakyReLU slope (1 = none); optional fp16 hi / lo operand planes of 16 * result (raw half bits) */
KKX_API int kkx_test_layernorm(int device, const float* x, const float* res, const float* w, const float* b,
                               const float* ada, int rows, int C, float eps, float slope, float* out,
                               unsigned short* pl_hi, unsigned short* pl_lo);
/* im2col operand producer of noise_convs[0] (22 of 24 input columns, k = 12, stride 6, pad 3): in [rows_in,24] fp32 with
   items at in_off[b] (in_len[b] rows) -> out [rows_out,Cpad] bf16 bits (pre-filled by the caller) with items at out_off[b]
   (out_len[b] rows) and 32 zeroed gap rows around each; generic = 1 forces the element-wise kernel */
KKX_API int kkx_test_im2col(int device, const float* in, int rows_in, int B, const int* in_off, const int* in_len,
                            const int* out_off, const int* out_len, int rows_out, int max_out_len, int Cpad, int generic,
                            unsigned short* out);
/* qkv [N,2304] -> ctx [N,768] */
KKX_API int kkx_test_attention(int device, const float* qkv, int N, float* ctx);
/* ragged batch through the tcgen05 / TMEM attention kernel (kernels_attn.cu), or the mma.sync kernel (umma = 0):
 * qkv [rows,2304] with items at off[b] (len[b] rows) -> ctx [rows,768] (rows outside the items are left untouched) */
KKX_API int kkx_test_attention_batch(int device, const float* qkv, int B, const int* off, const int* len, int rows,
                                     int umma, float* ctx);
/* x [L,C] + style row (gamma|beta, 2C) -> scale [C], shift [C] (InstanceNorm stats + AdaIN) */
KKX_API int kkx_test_adain_coef(int device, const float* x, int L, int C, const float* gamma_beta,
                                float* scale, float* shift);
/* Tensor-core (tcgen05/TMEM/TMA) shifted GEMM, stride 1: x [L, Ci] fp32 is rounded to bf16 by the
 * operand-producer kernel (optional per-channel scale/shift + activation), w [Co][ks][Ci] fp32 is
 * rounded to bf16 on the host; fp32 accumulation and epilogue.  out [out_rows, Co] pre-filled. */
KKX_API int kkx_test_conv_tc(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                             int Co, int ks, int dil, int pad, const float* pscale, const float* pshift,
                             int pact, float pslope, const float* palpha, int m_len, int ors, int oro,
                             int out_rows, const float* res, int res_rows, int res_shift, float oscale,
                             int accumulate, float* out);
/* Split-TF32 tensor-core GEMM/conv (fp32-grade accuracy on tcgen05 kind::tf32): x [L,Ci], w [Co][ks][Ci]
 * fp32, nprod = 3 or 4 partial products, eact 0 / 3 (gelu_new).  out [L, Co]. */
KKX_API int kkx_test_conv_tf32(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                               int Co, int ks, int dil, int pad, int nprod, int eact, float* out);
/* The same with split-FP16 operand planes ("3xFP16": fp16 hi/lo planes, kind::f16 MMAs, power-of-two scaling undone in
 * the epilogue); problems with >= 148 output tiles take the persistent kernel, smaller ones the single-tile kernel. */
KKX_API int kkx_test_conv_f16x3(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                                int Co, int ks, int dil, int pad, int eact, float* out);
/* The same with the kernel chosen by the caller -- 1 = single-tile, 2 = persistent, 3 = persistent CTA-pair
 * (tcgen05 cta_group::2) -- plus an optional residual [L, Co] and output scale: out = (conv + bias (+act) + res) * oscale.
 * The three kernels accumulate every output element in the same order; tests compare them bit for bit. */
KKX_API int kkx_test_conv_f16x3_k(int device, const float* x, int L, int Ci, const float* w, const float* bias,
                                  int Co, int ks, int dil, int pad, int eact, int kernel, const float* res, float oscale,
                                  float* out);
/* Fused generator res-block conv (kernels_arb.cu): out = (conv1d(snake(x*scale_b+shift_b), w, dilation) + bias + res)
 * * oscale (+ out when accumulate); B ragged items packed along rows (x, res, out: [sum lens, C]); C in
 * {128, 256}; w [C][ks][C]; x optionally rounded to bf16 first (in_bf16); result as fp32 or, want_bf16, the
 * unscaled bf16 output widened to fp32.  sums (nullable) [B][2][C] = column sums of (conv+bias+res) and of
 * its square.  desc_mode selects the UMMA base-offset convention for row-shifted operand views. */
KKX_API int kkx_test_arb_conv(int device, const float* x, int B, const int* lens, int C, int in_bf16,
                              const float* scale, const float* shift, const float* alpha, const float* w,
                              const float* bias, int ks, int dil, const float* res, float oscale,
                              int accumulate, int want_bf16, float* out, float* sums, int desc_mode);
/* Host-only: the library's tensor spec table (onnx_loader.cu kokoro_tensor_specs) as text lines "name d0 d1 ...\n";
 * returns the full length, writes at most capacity-1 characters + NUL. */
KKX_API int64_t kkx_test_tensor_specs(char* buf, int64_t capacity);
/* The same kernel on a bf16 residual stream: x and res are rounded to bf16 first; res == NULL is conv1 (bf16 x -> bf16
 * out), res != NULL is conv2 (bf16 residual -> the next bf16 x when want_bf16, else the fp32 block output). */
KKX_API int kkx_test_arb_conv_stream(int device, const float* x, int B, const int* lens, int C, const float* scale,
                                     const float* shift, const float* alpha, const float* w, const float* bias, int ks,
                                     int dil, const float* res, float oscale, int accumulate, int want_bf16, float* out,
                                     float* sums);
/* Output resampling (kernels_signal.cu resample_kernel).
 * kkx_test_resample_taps: host only -- the fp32 filter the library designs for out_rate (U * firwin(2H + 1,
 *   1 / max(U, D), ("kaiser", 5.0)), H = 10 max(U, D)); copies at most `capacity` taps to dst (nullable) and returns
 *   the tap count, or < 0 for a rate "out_rate" rejects; at 24000 the filter is the identity (one tap 1.0).
 * kkx_test_resample: B items packed back to back in x (item b has lens[b] >= 1 samples, any length) -> out (packed, item
 *   b has ceil(lens[b] U / D) samples); pcm (nullable) the 16-bit twin, codes (nullable) the G.711 twin of law 0 / 1
 *   (law -1 = none).  At 24000 the kernel runs its pass-through mode (U = D = 1, no filter). */
KKX_API int64_t kkx_test_resample_taps(int32_t out_rate, float* dst, int64_t capacity);
KKX_API int kkx_test_resample(int device, const float* x, int32_t B, const int64_t* lens, int32_t out_rate, int32_t law,
                              float* out, int16_t* pcm, uint8_t* codes);
/* FLAC encoder (kernels_flac.cu) on caller-supplied PCM: B items packed back to back (item b has lens[b] >= 1
 * samples), rate = any accepted "out_rate".  Writes the B FLAC files back to back into dst (nullable: size query)
 * and their offsets into byte_offsets [B + 1]; returns the total byte count or < 0. */
KKX_API int64_t kkx_test_flac(int device, const int16_t* pcm, int32_t B, const int64_t* lens, int32_t rate,
                              uint8_t* dst, int64_t capacity, int64_t* byte_offsets);
/* The same with "flac_lpc_order" = order (0..12; 0 gives kkx_test_flac's bytes). */
KKX_API int64_t kkx_test_flac_lpc(int device, const int16_t* pcm, int32_t B, const int64_t* lens, int32_t rate,
                                  int32_t order, uint8_t* dst, int64_t capacity, int64_t* byte_offsets);
/* Host only: the LPC window's taper table M [1024] of "flac_lpc_order" rule 2 (kkx.h), as the encoder uploads it.
 * Returns 0, or < 0 for a null m1024. */
KKX_API int kkx_test_flac_lpc_window(int32_t* m1024);
/* MP3 encoder (kernels_mp3.cu) on caller-supplied PCM, like kkx_test_flac: kbps as in kkx_infer_batch_mp3 (0 = the
 * default of the rate's version).  Returns the total byte count or < 0. */
KKX_API int64_t kkx_test_mp3(int device, const int16_t* pcm, int32_t B, const int64_t* lens, int32_t rate, int32_t kbps,
                             uint8_t* dst, int64_t capacity, int64_t* byte_offsets);
/* Host only: the MP3 encoder's tables.  Huffman table t (0..31): the pair (x, y) at codes / lens
 * [t * 256 + x * xlen[t] + y] (len 0: no entry), xlen [32] (0: no such table), linbits [32], the count1 tables A and B at c1_codes / c1_lens
 * [k * 16 + 8v + 4w + 2x + y], and the 512-tap analysis window C[i] of ISO 11172-3 Table C.1.  Any pointer may be
 * null.  Returns 0. */
KKX_API int kkx_test_mp3_tables(uint32_t* codes, uint8_t* lens, int32_t* xlen, int32_t* linbits, uint32_t* c1_codes,
                                uint8_t* c1_lens, double* window);
/* Loudness normalisation (kernels_loudness.cu, kkx.h "loudness_target").
 * kkx_test_loudness_design: host only -- the K-weighting biquads the library designs in double for sample rate fs
 *   (kweight[10], nullable: shelf b0 b1 b2 a1 a2, then high-pass b0 b1 b2 a1 a2; a0 = 1) and the fp32 taps of the
 *   true-peak filter (4 * firwin(81, 1/4, ("kaiser", 5.0)), at most `capacity` to tp_taps, nullable); returns the tap
 *   count.  The library itself measures at 24 kHz only.
 * kkx_test_loudness: B items packed back to back in x (item b has lens[b] >= 1 samples at 24 kHz) -> per item the
 *   integrated loudness (LUFS, NaN = undefined), the true peak (dBTP) and the gain for the given target (1/100 LUFS)
 *   and ceiling (1/100 dBTP); each output nullable.  The same three launches the model runs per frame group. */
KKX_API int64_t kkx_test_loudness_design(double fs, double* kweight, float* tp_taps, int64_t capacity);
KKX_API int kkx_test_loudness(int device, const float* x, int32_t B, const int64_t* lens, int32_t target_centi_lufs,
                              int32_t ceiling_centi_dbtp, float* lufs, float* true_peak_dbtp, float* gain);
/* Lookahead true-peak limiter (kernels_loudness.cu, kkx.h "limiter"), on B items packed as for kkx_test_loudness, with
 * the given target (1/100 LUFS, 0 = no normalisation) and ceiling (1/100 dBTP).  Per item: gain = the static g of
 * step 1, t = the trim of step 7, max_reduction_db and true_peak_dbtp = the kkx_last_limiter report; per sample
 * (packed like x): G = the smoothed gain of step 5 and v = the limited waveform of step 6.  Every pointer is nullable. */
KKX_API int kkx_test_limiter(int device, const float* x, int32_t B, const int64_t* lens, int32_t target_centi_lufs,
                             int32_t ceiling_centi_dbtp, float* gain, float* G, float* v, float* t,
                             float* max_reduction_db, float* true_peak_dbtp);
/* EBU R128 loudness range and maxima (kernels_loudness.cu, kkx.h kkx_last_loudness_range), on B items packed as for
 * kkx_test_loudness: the launches a "loudness_report" run makes (loud_energy, loud_peak, loud_gain, then loud_short
 * and loud_range).  Per item: lra (LU), m_max and s_max (LUFS); NaN = undefined.  Every output pointer is nullable. */
KKX_API int kkx_test_loudness_range(int device, const float* x, int32_t B, const int64_t* lens, float* lra,
                                    float* m_max, float* s_max);
/* Signal-path kernels.  These hooks take the caller's row layout: items at offsets into host buffers that already hold
 * the gap rows between them (the model's Level layout), and every output buffer is pre-filled by the caller and copied
 * back whole, so that anything a kernel writes outside its items shows.
 * kkx_test_sine_source: harmonic source (kernels_signal.cu sine_phase, then sine_source).  f0 [rows_f0], item b at
 *   f0_off[b] with L_b = f0_len[b] = 2T_b coarse steps; noise (nullable: the on-device Philox generator keyed by `seed`)
 *   [t * 9 + h] of item-local sample t, one buffer every item reads from offset 0 like kkx_set_noise, noise_n >=
 *   300 * max L_b * 9 floats; lin_w [9], lin_b [1] (m_source.l_linear).  phase (nullable) receives the coarse phase, items
 *   back to back as [9][L_b]; har the source, items back to back (300 L_b samples each). */
KKX_API int kkx_test_sine_source(int device, const float* f0, int rows_f0, int B, const int* f0_off, const int* f0_len,
                                 const float* noise, int64_t noise_n, uint64_t seed, const float* lin_w, const float* lin_b,
                                 float* phase, float* har);
/* kkx_test_stft: STFT (n_fft 20, hop 5) of B items of x (n_x samples; item b has 5 (F_b - 1) samples at s_off[b]) ->
 *   har [rows_h, 24] (magnitudes in columns 0..10, phases in 11..21), item b at h_off[b] with F_b = h_len[b] frames;
 *   replicate_pad 0 = reflect padding. */
KKX_API int kkx_test_stft(int device, const float* x, int64_t n_x, int B, const int64_t* s_off, const int* h_off,
                          const int* h_len, int rows_h, int replicate_pad, float* har);
/* kkx_test_istft: head + iSTFT of conv_post rows cp [rows, 24] (item b at h_off[b], F_b = h_len[b] frames) -> audio
 *   [n_audio], item b's 5 (F_b - 1) samples at s_off[b] (a multiple of 4); pcm (nullable) the 16-bit twin at the same
 *   offsets.  fast = 1 is the tensor-core configuration's SFU variant, 0 the libm variant. */
KKX_API int kkx_test_istft(int device, const float* cp, int rows, int B, const int* h_off, const int* h_len, int fast,
                           int64_t n_audio, const int64_t* s_off, float* audio, int16_t* pcm);
/* kkx_test_durations: duration head and length regulator (duration, dur_scan, then expand_idx and gather_rows).
 *   logits [rows_tok, 50] with item b at tok_off[b] (1 <= N_b = tok_len[b] <= 512), speeds [B] -> dur_float and pred_dur
 *   [rows_tok], cum [B][512] (exclusive prefix sums), total [B] (frames T_b) and fr_off [B]: the frame level the model
 *   builds (32 gap rows, 8-row alignment), whose row count the call returns (or < 0).  Every output pointer is
 *   nullable; idx [rows_fr] and out [rows_fr, ldo] are written only when both are given and capacity_rows >= rows_fr
 *   (otherwise the call is a size query): out[fr_off[b] + j, ocol + c] = feat[tok_off[b] + idx[fr_off[b] + j], c],
 *   feat [rows_tok, C]. */
KKX_API int64_t kkx_test_durations(int device, const float* logits, const float* speeds, const float* feat, int C, int ldo,
                                   int ocol, int B, const int* tok_off, const int* tok_len, int rows_tok, float* dur_float,
                                   int32_t* pred_dur, int32_t* cum, int32_t* total, int32_t* fr_off, int32_t* idx,
                                   float* out, int64_t capacity_rows);
/* kkx_test_pool_up: depthwise ConvTranspose1d(k3, s2, p1, op1) on lrelu(x * scale_b + shift_b, slope): x [rows_in, C]
 *   with item b at in_off[b] (T_b = in_len[b] rows), scale / shift [B][C], w [C][3], bias [C]; item b's 2T_b output rows
 *   at out_off[b].  Cpad == 0: the fp32 kernel, out float [rows_out, C]; Cpad >= C: the bf16 operand kernel, out bf16
 *   bits [rows_out, Cpad], which also zeroes the gap rows and pad columns. */
KKX_API int kkx_test_pool_up(int device, const float* x, int rows_in, int C, int B, const int* in_off, const int* in_len,
                             const float* scale, const float* shift, float slope, const float* w, const float* bias,
                             const int* out_off, int rows_out, int Cpad, void* out);
/* kkx_test_post_conv: generator conv_post in the tensor-core configuration (kernels_arb.cu, post variant): x
 *   [rows, 128] fp32 with item b at off[b] (len[b] rows, >= 32 gap rows around each), w [22][7][128] (out channel, tap,
 *   in channel; rounded to bf16 here), bias [22] -> out [rows, 24] = Conv1d(128, 22, 7, pad 3) of bf16(lrelu(x, slope))
 *   in columns 0..21 of the item rows. */
KKX_API int kkx_test_post_conv(int device, const float* x, int rows, int B, const int* off, const int* len, const float* w,
                               const float* bias, float slope, float* out);
/* kkx_test_curve_conv: Conv1d(1, 1, k3, s2, p1) of the F0 / N curves: x [rows_x], item b at x_off[b] (x_len[b] values)
 *   -> out[out_off[b] + t, ocol] of out [rows_out, ldo], t < out_len[b]. */
KKX_API int kkx_test_curve_conv(int device, const float* x, int rows_x, int B, const int* x_off, const int* x_len,
                                const float* w3, const float* bias, float* out, int rows_out, int ldo, int ocol,
                                const int* out_off, const int* out_len);
/* kkx_test_add_rows_stats: a += b in place on the item rows (a, b [rows, C], item b at off[b]) and the chunk statistics
 *   part [B][ceil(max len / 128)][2][C] of the sum; with out_bf16 (bf16 bits [rows, C], nullable) the sum goes there
 *   only and `a` is left as it was. */
KKX_API int kkx_test_add_rows_stats(int device, float* a, const float* b, int rows, int C, int B, const int* off,
                                    const int* len, uint16_t* out_bf16, float* part);
KKX_API const char* kkx_test_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
