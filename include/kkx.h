/*
 * kkx.h -- C ABI of the B200-native Kokoro-82M inference backend.
 *
 * Drop-in boundary for the ONNX-Runtime session wrapper of byteowlz/kokorox
 * (/root/reference/kokorox/src/onn/).  Each entry point names the reference interface it
 * replaces.  Plain pointers and sizes only; every function is callable from Rust FFI
 * (`extern "C"`), cgo, or ctypes.  No function aborts or throws across the ABI: all failures
 * are a negative return code plus a message retrievable with kkx_last_error().
 *
 * Thread safety: a kkx_ctx may be shared between threads (the reference shares one
 * `Arc<OrtKoko>` between tokio workers, ort_koko.rs:13-18, koko.rs:36-45); calls on one ctx
 * are serialised internally, exactly like the reference's `Mutex<Session>` (ort_koko.rs:77-78).
 * Use one ctx per GPU for multi-GPU request sharding.
 */
#ifndef KKX_H_
#define KKX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct kkx_ctx kkx_ctx;

#if defined(__GNUC__)
#define KKX_API __attribute__((visibility("default")))
#else
#define KKX_API
#endif

#define KKX_OK 0
#define KKX_ERR_ARG (-1)      /* bad argument (null pointer, token id out of 0..177, n_tokens > 512, speed outside [0.1, 10]) */
#define KKX_ERR_IO (-2)       /* model file missing / malformed / tensor missing or unresolved  */
#define KKX_ERR_CUDA (-3)     /* CUDA runtime error (message has the cudaError string)          */
#define KKX_ERR_NO_DEVICE (-4)/* no CUDA device / device ordinal out of range -- there is NO CPU fallback */
#define KKX_ERR_STATE (-5)    /* ctx not initialised ("Session is not initialized.", ort_koko.rs:88-90), or a call
                               * out of sequence (run before stage, fetch before run, ticket of a destroyed ctx) */

#define KKX_STYLE_DIM 256     /* ort_koko.rs:61-65: style tensor [B,256]                        */
#define KKX_MAX_TOKENS 512    /* ALBERT max_position_embeddings; koko.rs:781-783 chunks to <=500 */
#define KKX_SAMPLE_RATE 24000 /* koko.rs:59                                                     */

/* Replaces kokorox::onn::init_ort(dylib_path) (onn/mod.rs:19-49): process-wide one-time init.
 * Checks that a CUDA driver and at least one sm_100 device are present.  Optional: kkx_create
 * performs the same check.  Returns KKX_OK or KKX_ERR_NO_DEVICE. */
KKX_API int kkx_init(void);

/* Replaces OrtKoko::new(model_path) -> OrtBase::load_model (ort_koko.rs:31-35,
 * ort_base.rs:14-39, `commit_from_file(model_path)`): loads the model file onto GPU `device_ordinal` and builds
 * every derived weight layout.  `weights_path` is what the reference passes -- the downloaded ONNX file
 * (kokoro-v1.0.onnx, onnx/model.onnx or one of the fp16 / q8 / uint8 / q4 variants of hf_cache.rs:135-144; the
 * initialisers are read straight from the protobuf, named through the node graph and dequantised at load) -- or a
 * KKXW file written by kokorox_b200/weightfile.py / convert.py.  The format is detected from the file's magic.
 * Sessions created from the same (file, device) share one device-resident weight set (the reference's servers hold
 * two or three sessions of one model, koko main.rs:1477,1596).  A new session runs the benchmarked configuration
 * ("precision" = 1, see kkx_set_option).  On failure *out is NULL and kkx_last_error(NULL) has the reason; for an
 * ONNX file that does not resolve it lists the tensors that could not be found. */
KKX_API int kkx_create(const char* weights_path, int device_ordinal, kkx_ctx** out);

/* Host-only helper (no GPU needed): reads `src_path` exactly as kkx_create would (ONNX or KKXW) and writes the
 * recovered Kokoro-82M state dict as a KKXW file, e.g. to convert a downloaded model_q8f16.onnx once.
 * *out_tensors (nullable) receives the tensor count. */
KKX_API int kkx_convert_model_file(const char* src_path, const char* dst_kkxw_path, int32_t* out_tensors);

/* Drop of OrtKoko (koko.rs:1338-1375 `cleanup`): frees all device and pinned host memory. */
KKX_API void kkx_destroy(kkx_ctx* ctx);

/* Error string of the CALLING THREAD's last failed call (the ctx argument is accepted for symmetry and may be
 * NULL): thread-local, so threads sharing one ctx never see -- or race with -- each other's messages; read it
 * on the thread that got the error code.  The Rust shim turns rc<0 into Err(kkx_last_error()), matching
 * the Result<_, String> / Box<dyn Error> returns of ort_koko.rs:31,42. */
KKX_API const char* kkx_last_error(const kkx_ctx* ctx);

/* Replaces OrtKoko::infer(tokens, styles, speed) at B=1 (ort_koko.rs:37-91; call site
 * koko.rs:1168-1177).
 *   tokens     [n_tokens] i64, INCLUDING the leading and trailing 0 pad (koko.rs:1168-1173);
 *              2 <= n_tokens <= 512, ids in 0..177 (tts/vocab.rs:5-20)   -- "input_ids"
 *   style256   [256] f32 (koko.rs:1255-1306 mix_styles row)             -- "style"
 *   speed      in [0.1, 10] (durations are 50/speed frames per token at most) -- "speed"
 *   out_audio  receives a library-owned pinned host buffer of *out_samples f32 mono at the session's "out_rate"
 *              (default 24 kHz: 600 * sum(pred_dur) samples; at rate r: ceil(600 * sum(pred_dur) * U / D), see
 *              "out_rate"); valid until kkx_release(ctx, ptr) -- outputs[0]
 *   out_pred_dur  nullable; [n_tokens] predicted integer frame durations (not observable
 *              through the reference graph; exposed for parity tests).
 * Thread-safe.  By default concurrent callers run one after another, like the reference's
 * Mutex<Session> (ort_koko.rs:14,77).  With option "coalesce" = K > 1 the callers that are waiting while a
 * step runs are merged into ONE ragged batch of up to K utterances (the batching queue SURVEY 8f row 4 asks the
 * servers for, openai lib.rs:400-412): each caller still gets exactly the waveform it would get alone (batched
 * and single results are bit-identical), as a view into a shared pinned buffer that is recycled once every
 * caller of that batch has called kkx_release.  A request that fails validation fails alone. */
KKX_API int kkx_infer(kkx_ctx* ctx, const int64_t* tokens, int32_t n_tokens, const float* style256,
              float speed, float** out_audio, int64_t* out_samples, int32_t* out_pred_dur);

/* Ragged batch of independent utterances (new capability; the reference only ever calls infer
 * with B=1, koko.rs:1175, and serialises callers on a mutex).  Item b uses
 * tokens[tok_offsets[b] .. tok_offsets[b+1]), styles[b*256 ..], speeds[b]; result b is
 * (*out_audio)[out_sample_offsets[b] .. out_sample_offsets[b+1]) and equals what kkx_infer
 * returns for that item alone.  out_pred_dur (nullable) is indexed like tokens. */
KKX_API int kkx_infer_batch(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                    const float* styles, const float* speeds, float** out_audio,
                    int64_t* out_sample_offsets, int32_t* out_pred_dur);

/* Returns an audio buffer obtained from kkx_infer / kkx_infer_batch / kkx_wait to the library. */
KKX_API void kkx_release(kkx_ctx* ctx, float* audio);

/* ---- asynchronous form of kkx_infer (SURVEY 8f row 4).  The reference's WebSocket server synthesises and sends
 * sentence by sentence, `for sentence ... { synthesize_and_send_chunk(...).await }` (kokorox-websocket/src/lib.rs:
 * 371-376), so sentence k+1 cannot start while k is on the wire, and its servers block one thread per request on
 * Mutex<Session> (openai lib.rs:400-412, ort_koko.rs:77).
 *   kkx_submit  copies the request (the caller's buffers are free again on return), queues it and returns a
 *               ticket at once; a worker thread owned by the ctx runs whatever is queued as ragged batches of up
 *               to "async_batch" utterances (each result is bit-identical to the caller's own kkx_infer).
 *   kkx_poll    1 = finished (kkx_wait will not block), 0 = still queued / running, <0 = unknown ticket.
 *   kkx_wait    blocks until the request has finished and redeems the ticket (once): same outputs as kkx_infer;
 *               out_pred_dur (nullable) must hold n_tokens entries.  A failed request returns its own error code
 *               and message here.  Release the audio with kkx_release. */
typedef int64_t kkx_ticket;
KKX_API int kkx_submit(kkx_ctx* ctx, const int64_t* tokens, int32_t n_tokens, const float* style256, float speed,
                       kkx_ticket* out_ticket);
KKX_API int kkx_poll(kkx_ctx* ctx, kkx_ticket ticket);
KKX_API int kkx_wait(kkx_ctx* ctx, kkx_ticket ticket, float** out_audio, int64_t* out_samples,
                     int32_t* out_pred_dur);

/* ---- "next" rows of the hot-path scope (SURVEY 8f): the host work either side of the call.
 *
 * kkx_load_voices replaces TTSKoko::load_voices (koko.rs:1308-1334): uploads the voice table once,
 *   table [n_voices][511][256] f32 (row = un-padded token count, koko.rs:1262).
 * kkx_infer_batch_voices replaces TTSKoko::mix_styles + OrtKoko::infer (koko.rs:1161-1180, 1255-1306): like
 *   kkx_infer_batch, but the style of item b is mixed ON THE DEVICE from the table:
 *     style_b[j] = sum over i in [mix_offsets[b], mix_offsets[b+1]) of table[voice_ids[i]][style_rows[b]][j] * voice_portions[i]
 *   in that order with separate multiply and add, i.e. bit-identical to the reference loop (koko.rs:1296-1302).
 *   A single voice ("af_sky") is one entry with portion 1.0; a mix "af_sky.4+af_nicole.5" is two entries with
 *   portions 0.4, 0.5 (portion = weight * 0.1, NOT renormalised, koko.rs:1283). */
KKX_API int kkx_load_voices(kkx_ctx* ctx, const float* table, int32_t n_voices);
KKX_API int kkx_infer_batch_voices(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                           const int32_t* mix_offsets, const int32_t* voice_ids, const float* voice_portions,
                           const int32_t* style_rows, const float* speeds, float** out_audio,
                           int64_t* out_sample_offsets, int32_t* out_pred_dur);

/* kkx_infer_batch_pcm16: like kkx_infer_batch, but the waveform comes back as 16-bit PCM,
 *   pcm = trunc(clamp(s, -1, 1) * 32767) -- the f32 -> i16 conversion of the reference's WebSocket server
 *   (kokorox-websocket/src/lib.rs:699-703) fused into the iSTFT kernel; half the device->host bytes.  At an
 *   "out_rate" other than 24000 the same conversion is applied to the resampled value, inside the resampling kernel.
 *   Release the buffer with kkx_release_pcm16. */
KKX_API int kkx_infer_batch_pcm16(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                          const float* styles, const float* speeds, int16_t** out_pcm,
                          int64_t* out_sample_offsets, int32_t* out_pred_dur);
KKX_API void kkx_release_pcm16(kkx_ctx* ctx, int16_t* pcm);

/* kkx_infer_batch_g711: like kkx_infer_batch_pcm16, but every sample comes back as one ITU-T G.711 byte, for
 *   telephony (SIP / PSTN, PCMU / PCMA media streams): law 0 = mu-law (PCMU), 1 = A-law (PCMA); any other value is
 *   KKX_ERR_ARG.  The code of a sample is the G.711 encoding of the same 16-bit value p that kkx_infer_batch_pcm16
 *   returns -- mu-law of the 14-bit p >> 2 (bias 33, clip 8159), A-law of the 13-bit p >> 3 -- i.e. the Sun reference
 *   g711.c, equal to Python's audioop.lin2ulaw / lin2alaw(..., 2).  Works at every "out_rate" (8000 is the G.711 rate;
 *   at 24000 the codes are those of the model's own waveform).  Offsets count codes (= samples).  One pass (no
 *   "max_tokens" split); release the buffer with kkx_release_g711.  No WAV container: telephony transports carry
 *   raw codes. */
KKX_API int kkx_infer_batch_g711(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                 const float* styles, const float* speeds, int32_t law /* 0 = mu-law, 1 = A-law */,
                                 uint8_t** out_codes, int64_t* out_sample_offsets, int32_t* out_pred_dur);
KKX_API void kkx_release_g711(kkx_ctx* ctx, uint8_t* codes);

/* kkx_infer_batch_flac: like kkx_infer_batch_pcm16, but item b comes back as one complete FLAC file (RFC 9639,
 *   streamable subset): bytes [out_byte_offsets[b], out_byte_offsets[b+1]) of *out_bytes.  Decoding it yields exactly
 *   the int16 samples kkx_infer_batch_pcm16 returns for that item, at the session's "out_rate".
 *   out_sample_offsets (nullable) as in kkx_infer_batch_pcm16.  One pass (no "max_tokens" split).  Encoded on the
 *   device; the bytes are a function of the item's samples alone (same bytes in any batch).  For n samples p[0..n)
 *   at rate r:
 *   head     "fLaC", metadata block header (last 1, type 0 STREAMINFO, length 34), STREAMINFO: min = max block size
 *            4096, min / max frame size = this stream's smallest / largest frame in bytes, rate r, 1 channel,
 *            16 bits, n total samples, MD5 all zero ("not computed").
 *   frames   frame i holds p[4096 i, min(n, 4096 (i + 1))) (bs samples); no prediction crosses a frame.  Header:
 *            FF F8, block-size code (4096: 1100; a short last block: its table code 192 / 576 / 1152 / 2304 /
 *            256 / 512 / 1024 / 2048, else 0110 + 8-bit bs - 1 if bs <= 256, else 0111 + 16-bit bs - 1),
 *            sample-rate code (8000 0100, 16000 0101, 22050 0110, 24000 0111, 32000 1000, 44100 1001,
 *            48000 1010, 12000 1100 + byte 12, 11025 1101 + 16-bit 11025), byte 08 (mono, 16 bits), frame number
 *            i in FLAC's UTF-8 coding, CRC-8 (poly 0x07, init 0).  Footer: zero bits to a byte boundary, CRC-16
 *            of the frame (poly 0x8005, init 0, big-endian).
 *   subframe one per frame, wasted-bits flag 0:
 *            CONSTANT (00, 16-bit value) if all bs samples are equal (bs = 1 included); else the cheapest FIXED
 *            (10 | o << 1): order o in 0..4 (o < bs), warm-up = first o samples (16 bits each), Rice method 0,
 *            partition order q in 0..8 (bs % 2^q == 0, (bs >> q) > o; the first partition holds (bs >> q) - o
 *            residuals), per partition the k in 0..14 minimising sum (u >> k) + n_part (k + 1), residual
 *            e folded to u = e >= 0 ? 2e : -2e - 1 and coded as (u >> k) zeros, a one, the low k bits.  Cost
 *            8 + 16 o + 6 + sum over partitions (4 + sum (u >> k) + n_part (k + 1)) bits; ties go to the smaller
 *            o, then q, then k.  VERBATIM (02, bs x 16 bits) only if strictly cheaper (8 + 16 bs bits), so no
 *            frame is larger than verbatim.  No Rice escapes.  LPC subframes only with "flac_lpc_order" (below).
 *   Release the buffer with kkx_release_flac.  KKX_ERR_ARG for a null out_bytes or out_byte_offsets. */
KKX_API int kkx_infer_batch_flac(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                 const float* styles, const float* speeds, uint8_t** out_bytes,
                                 int64_t* out_byte_offsets /* [batch + 1], required */,
                                 int64_t* out_sample_offsets /* [batch + 1], nullable */, int32_t* out_pred_dur);
KKX_API void kkx_release_flac(kkx_ctx* ctx, uint8_t* bytes);

/* kkx_infer_programs: one output per PROGRAM instead of one per item, for a request that was split into chunks (the
 *   reference splits text into chunks of at most 500 tokens, koko.rs:781-783, runs one infer per chunk and joins the
 *   audio with extend_from_slice, koko.rs:947-1191; its OpenAI server and `file --merge` return one file per request).
 *   Program k is the run of consecutive items [program_offsets[k], program_offsets[k+1]).  Items take their inputs
 *   as in kkx_infer_batch.  Let x_k be the concatenation, in item order, of the 24 kHz model waveforms of program k's
 *   items -- each exactly what kkx_infer_batch returns for the item at "out_rate" 24000 with loudness off -- so x_k
 *   has n_k = sum of 600 T_b samples.  The program is then treated as one utterance of waveform x_k:
 *   1. Loudness (when "loudness_target" != 0): rules 1-5 of "loudness_target" below apply to x_k as one signal: the
 *      K-weighting starts from zero state at x_k's first sample and runs across the joins, the 400 ms blocks start
 *      at x_k's sample 0, gating is over all of x_k's blocks, the true peak is that of resample_poly(x_k, 4, 1);
 *      one gain g_k for the whole program.
 *   2. Rate: y_k = resample_poly(x_k, U, D) under the "out_rate" rule, with zeros outside x_k, ceil(n_k U / D)
 *      samples (at 24000, y_k = x_k).
 *   3. Samples: each returned sample is fp32(y * g_k); PCM16, G.711 and FLAC follow from that value by their rules
 *      above.  FLAC is one file per program under the kkx_infer_batch_flac rules, with n = the program's sample count.
 *   4. Purity: a program's output depends on its own items only -- not on its position in the call, on the other
 *      programs, or on how "max_frames" splits the items into frame groups (a program may span several groups).
 *   5. Identity: a program of one item returns exactly what the entry point of that encoding returns for that item
 *      (bits, FLAC bytes and the loudness report).  At 24000 with loudness off, an F32 or PCM16 program is the
 *      bit-exact concatenation of its items' outputs (the reference's extend_from_slice).
 *   encoding: KKX_ENC_F32 (4 bytes per sample), _PCM16 (2), _ULAW / _ALAW (1, G.711 as kkx_infer_batch_g711), _FLAC.
 *   Program k's output is bytes [out_byte_offsets[k], out_byte_offsets[k+1]) of *out_bytes (offsets in bytes for every
 *   encoding); out_sample_offsets (nullable, [n_programs + 1]) in output-rate samples; out_pred_dur (nullable) is
 *   indexed like tokens.  One pass (no "max_tokens" split).  Afterwards kkx_last_loudness, kkx_last_loudness_range
 *   and the "loudness_items" stat report per program (their batch is n_programs).  A FLAC program holds at most
 *   2^36 - 1 samples (the STREAMINFO field; longer is KKX_ERR_ARG).  Release the buffer with kkx_release_programs.
 *   KKX_ERR_ARG, with the session left as it was, for: a null out_bytes or out_byte_offsets; n_programs outside
 *   1..batch; program_offsets null, not starting at 0, not ending at batch, or not strictly increasing (no empty
 *   program); encoding outside 0..4.
 *   Not provided: pauses, cross-fades or silence trimming at the joins (the reference joins chunks as they are);
 *   programs through kkx_infer, coalescing, kkx_submit, kkx_infer_batch_voices or kkx_run_staged; a "max_tokens" split
 *   of a program call; streaming a program before its last item is done; Opus.  MP3 programs: kkx_infer_programs_mp3
 *   (the bitrate does not fit in the encoding code). */
#define KKX_ENC_F32 0   /* f32 samples, 4 bytes each */
#define KKX_ENC_PCM16 1
#define KKX_ENC_ULAW 2
#define KKX_ENC_ALAW 3
#define KKX_ENC_FLAC 4
KKX_API int kkx_infer_programs(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                               const float* styles, const float* speeds,
                               int32_t n_programs, const int32_t* program_offsets /* [n_programs + 1] */,
                               int32_t encoding, void** out_bytes,
                               int64_t* out_byte_offsets /* [n_programs + 1], required */,
                               int64_t* out_sample_offsets /* [n_programs + 1], nullable */,
                               int32_t* out_pred_dur /* nullable, indexed like tokens */);
KKX_API void kkx_release_programs(kkx_ctx* ctx, void* bytes);

/* kkx_infer_batch_mp3: like kkx_infer_batch_flac, but item b comes back as one MP3 file (MPEG audio Layer III,
 *   constant bitrate): bytes [out_byte_offsets[b], out_byte_offsets[b+1]) of *out_bytes (out_byte_offsets required,
 *   out_sample_offsets nullable).  kkx_infer_programs_mp3: kkx_infer_programs' arguments and rules with kbps in place
 *   of encoding, one MP3 file per program.  Release either buffer with kkx_release_mp3.  Encoded on the device after
 *   the forward pass; kkx_last_loudness, kkx_last_limiter and kkx_last_loudness_range report as after a PCM16 call.
 *   Input: the int16 samples p[0..n) that kkx_infer_batch_pcm16 returns for the item (program) at the session's
 *   "out_rate", taken as p / 32768; samples outside [0, n) are zero.
 *   Format: mono (mode 11), no CRC (protection bit 1), private / copyright / original / emphasis 0, no bit reservoir
 *   (main_data_begin 0), long blocks only (window_switching_flag 0, block type 0), no scalefactors
 *   (scalefac_compress 0, so every slen is 0 in MPEG-1 and LSF coding; scfsi 0, preflag 0, scalefac_scale 0), no
 *   ID3 tag, no Xing / Info / LAME frame.  Version by "out_rate": MPEG-1 at 32000, 44100, 48000 (two granules of
 *   576 samples a frame); MPEG-2 LSF at 16000, 22050, 24000 and MPEG-2.5 at 8000, 11025, 12000 (one granule a
 *   frame).  MPEG-2.5 is not part of ISO/IEC 13818-3, but common decoders play it.
 *   kbps: MPEG-1 32, 40, 48, 56, 64, 80, 96, 112, 128, 160, 192, 224, 256, 320; MPEG-2 / 2.5 8, 16, 24, 32, 40, 48,
 *   56, 64, 80, 96, 112, 128, 144, 160; 0 = 192 at the MPEG-1 rates and 160 at the others (at the model's 24000 the
 *   format allows at most 160).  Any other value is KKX_ERR_ARG (the message names the version and its table) with
 *   the session left as it was, as is a null out_bytes or out_byte_offsets and, for programs, any program-table
 *   error of kkx_infer_programs.
 *   Frames: with A = 144000 kbps / rate (MPEG-1) or 72000 kbps / rate, frame f of a file takes bytes
 *   [floor(f A), floor((f + 1) A)) (64-bit integers); its padding bit is its length minus floor(A).  The decoded
 *   signal is the input delayed by D = 1057 samples (one granule of MDCT overlap, 576, plus the analysis / synthesis
 *   filterbank, 481).  A file has F = ceil((n + D) / samples per frame) frames, so a standard decoder emits every
 *   input sample, and floor(F A) bytes.  Granule g of a file (frame g / 2 of MPEG-1, frame g otherwise) codes the
 *   MDCT of subband slots 18 (g - 1) .. 18 g + 17, slot s being the filterbank output over input samples
 *   32 s - 480 .. 32 s + 31.  A granule's bit budget is min(4095, its share of the frame's main-data bits); in an
 *   MPEG-1 frame granule 0 takes floor(half) and granule 1 the rest (granule 1's data follows granule 0's directly).
 *   Unused bits are zero.
 *   Analysis: the ISO 11172-3 polyphase filterbank (window C[i] of Table C.1, matrixing cos((2k + 1)(i - 16) pi / 64)),
 *   odd samples of odd subbands negated, the 18-point MDCT of block type 0 with the sine window (scaled by 1/9, the
 *   inverse of the standard IMDCT), the eight alias-reduction butterflies with c_i = -0.6, -0.535, -0.33, -0.185,
 *   -0.095, -0.041, -0.0142, -0.0037.
 *   Quantisation: ix = nint((|xr| / 2^((gg - 210) / 4))^0.75 - 0.0946), nint(v) = floor(v + 0.5).  A gg fits when
 *   no ix exceeds 8206 (15 + 2^13 - 1) and the granule's part2_3_length (below) is within its budget.  gg is found by
 *   lo = 0, hi = 255; while lo < hi { mid = (lo + hi) / 2; if fits(mid) hi = mid else lo = mid + 1 } -- written
 *   down so that every implementation takes the same steps where the bit count is not monotone.  There is no
 *   psychoacoustic model: the quantisation noise is white across the spectrum; the tests pin the signal-to-noise
 *   ratio of decoded speech per rate.
 *   Regions: strip trailing zero pairs; then take quadruples whose values are all <= 1 into count1, from the top
 *   down; big_values is what remains (in pairs).  One Huffman table for all three big_values regions: among the
 *   tables whose range covers the largest value there (table 0 when it is 0; for tables 16..31 the linbits decide),
 *   the one with the fewest bits, ties to the lowest number.  region0_count 7, region1_count 7.  Count1 uses the
 *   cheaper of tables A and B, ties to A.  part2_3_length = the bits of the codes, linbits and sign bits.
 *   Purity and identity as for FLAC programs: a file's bytes are a function of its samples alone (batch, position,
 *   frame groups and other programs do not matter), a one-item program returns exactly the kkx_infer_batch_mp3 bytes
 *   of that item, and no floating-point atomics or launch-shape-dependent results enter.
 *   Not provided: VBR or ABR, the bit reservoir, a psychoacoustic model, short blocks, scalefactors, per-region
 *   Huffman tables, the Xing / LAME tag (encoder delay for gapless playback), ID3, CRC, Opus, a "max_tokens" split. */
KKX_API int kkx_infer_batch_mp3(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                const float* styles, const float* speeds, int32_t kbps, uint8_t** out_bytes,
                                int64_t* out_byte_offsets /* [batch + 1], required */,
                                int64_t* out_sample_offsets /* [batch + 1], nullable */, int32_t* out_pred_dur);
KKX_API int kkx_infer_programs_mp3(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                   const float* styles, const float* speeds,
                                   int32_t n_programs, const int32_t* program_offsets /* [n_programs + 1] */,
                                   int32_t kbps, uint8_t** out_bytes,
                                   int64_t* out_byte_offsets /* [n_programs + 1], required */,
                                   int64_t* out_sample_offsets /* [n_programs + 1], nullable */,
                                   int32_t* out_pred_dur /* nullable, indexed like tokens */);
KKX_API void kkx_release_mp3(kkx_ctx* ctx, uint8_t* bytes);

/* ---- output containers (host-side byte work after the pcm16 / f32 result; no GPU involved, no ctx needed).
 * kkx_wav_header_pcm16: the 44-byte RIFF/WAVE header of the WebSocket server's `encode_audio`
 *   (kokorox-websocket/src/lib.rs:707-731): PCM format 1, mono, 16 bit, sizes filled in from n_samples.
 * kkx_wav_header_f32_stream: the streaming header of utils/wav.rs:19-43: IEEE-float format 3, both size fields
 *   0xFFFFFFFF placeholders; f32 samples follow as little-endian bytes (wav.rs:45-50), i.e. the result buffer as is.
 * kkx_encode_wav16_base64: `encode_audio` end to end for a pcm16 result: base64 (standard alphabet, '=' padded)
 *   of header + samples.  Returns the number of characters (without the terminating NUL, which is written when
 *   capacity allows); writes nothing if capacity is too small, so call with dst = NULL to size the buffer. */
KKX_API int32_t kkx_wav_header_pcm16(uint8_t* dst44, int64_t n_samples, int32_t sample_rate);
KKX_API int32_t kkx_wav_header_f32_stream(uint8_t* dst44, int32_t channels, int32_t sample_rate);
KKX_API int64_t kkx_encode_wav16_base64(const int16_t* pcm, int64_t n_samples, int32_t sample_rate, char* dst,
                                int64_t capacity);

/* ---- device-resident variant (bench.py `value`: inputs already in HBM, output stays in HBM).
 * Stages the batch on the device once; kkx_run_staged() then runs the whole forward with no
 * host<->device payload traffic (only the per-item frame counts cross, 4 bytes per item).
 * Returns total samples (at "out_rate") in *out_total_samples and kernel launches in *out_launches
 * (either may be NULL). */
KKX_API int kkx_stage_batch(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                    const float* styles, const float* speeds);
KKX_API int kkx_run_staged(kkx_ctx* ctx, int64_t* out_total_samples, int64_t* out_launches);
/* Copies the result of the last kkx_run_staged to host memory. */
KKX_API int kkx_fetch_staged(kkx_ctx* ctx, float* dst_audio, int64_t capacity, int64_t* out_sample_offsets,
                     int32_t* out_pred_dur);

/* ---- options.  Known keys:
 *   "precision"   1 (DEFAULT, the benchmarked configuration) = tcgen05 tensor cores: bf16 decoder + generator,
 *                 split-TF32 predictor; 0 = fp32 SIMT everywhere (verification mode: tightest parity, several
 *                 times slower)
 *   "noise_seed"  seed of the on-device Philox N(0,1) generator for the SineGen noise
 *   "max_frames"  frame budget per frame-phase group (memory control for large batches)
 *   "max_tokens"  token budget per pass of one kkx_infer_batch call (default 40960): larger batches are run in
 *                 several passes and concatenated, so a call may carry any number of utterances
 *   "stft_replicate" 0 = reflect edge padding (upstream STFT), 1 = replicate (conv-STFT export)
 *   "coalesce"    0/1 = off; K > 1 (<= 512) = merge up to K concurrent kkx_infer callers per step
 *   "coalesce_wait_us"  how long the caller that found the queue idle waits for company (default 0: no
 *                 added latency -- batches form from whatever queued up behind the running step)
 *   "async_batch" most kkx_submit requests the worker merges into one ragged batch (default 64)
 *   "latency_graphs" 0/1: replay the token phase of single-utterance calls from a CUDA graph keyed by the token
 *                 count (default 1; captured on the second call with a given count)
 *   "fork_max_batch" largest batch whose independent branches (text encoder | ALBERT, F0 | N, harmonic source |
 *                 decoder) run on two streams (default 4; 0 = never).  Results do not depend on either option.
 *   kernel selection, all default 1 and none of them changes a bit of the result (each names the round-2 kernel it
 *   switches on; 0 selects the kernel it replaced -- for A/B measurements and the bit-identity tests):
 *   "attention_umma" (tcgen05 attention), "split_f16" (fp16 instead of tf32 operand planes; fp32-grade either way, but
 *   not the same bits), "gemm_pair" (split-precision GEMMs on CTA pairs, tcgen05 cta_group::2), "conv_pair" (the
 *   decoder's wide bf16 convs on CTA pairs), "fuse_planes" (LayerNorm / FFN / QKV GEMM write the next kernel's operand
 *   planes directly), "fuse_phases" (ConvTranspose1d phases in one launch), "ups_phase_loop" (default 3: the stage-1
 *   up-sampling conv on persistent CTAs with resident weights; 1 / 2 = one CTA per row tile looping over the phases,
 *   0 = one CTA per (tile, phase); same bits); "lstm_fast_gates" (SFU gate functions in the LSTM recurrence of the
 *   tensor-core configuration; fp32-grade, not the same bits as libm) and "fuse_noise_stats" (the generator's 22 -> 128
 *   noise conv in fp32 together with the statistics of its output instead of bf16 operands on the tensor cores);
 *   "stream_bf16" (default 0) keeps the res-block residual stream in bf16.
 *   "out_rate"    sample rate of every waveform the session returns (default 24000, the model's rate; nothing is
 *                 resampled then).  Accepted: r in 8000..48000 with U = r/g, D = 24000/g (g = gcd(r, 24000)) and
 *                 max(U, D) <= 320 -- 8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000; anything else is
 *                 KKX_ERR_ARG naming the reduced ratio, and the session keeps its rate.  Applies to every waveform entry
 *                 point (kkx_infer, _batch, _batch_voices, _batch_pcm16, _batch_g711, kkx_wait and coalesced / async
 *                 batches, kkx_run_staged / kkx_fetch_staged) for runs that start after the call; every sample count
 *                 and offset is then in output-rate samples.  One rate per session (sessions of one file share the
 *                 device weights, so a server holds one session per rate).  Each utterance (item, or program of
 *                 kkx_infer_programs) is resampled on its own, with zeros outside it, exactly as
 *                 scipy.signal.resample_poly(x, U, D) with its defaults:
 *                   H = 10 max(U, D),  h = U * firwin(2H + 1, 1 / max(U, D), window = ("kaiser", 5.0))
 *                   y[m] = sum over k ascending, 0 <= k < n, 0 <= mD - kU + H <= 2H, of x[k] * h[mD - kU + H],
 *                   0 <= m < ceil(n U / D)   (n = 600 T input samples)
 *                 accumulated in fp32 (taps designed in double, stored as fp32), one output per thread on the GPU, so
 *                 results stay bit-identical to the item's own B = 1 call.  16-bit PCM and G.711 are converted from y.
 *   "loudness_target"  integrated-loudness target in 1/100 LUFS (e.g. -2300 = EBU R128's -23 LUFS, -1600 podcast,
 *                 -1400 streaming); 0 (DEFAULT) = off: no kernel is added and every bit and launch is as before.
 *                 Accepted: 0 or -7000..-500.
 *   "true_peak_max"  true-peak ceiling in 1/100 dBTP (default -100, EBU R128's -1 dBTP); accepted -2000..0.
 *                 For both, any other value is KKX_ERR_ARG and the session keeps its setting.  Like "out_rate", one
 *                 setting per session, followed by every waveform entry point (kkx_infer, _batch, _batch_voices,
 *                 _batch_pcm16, _batch_g711, _batch_flac, coalesced and kkx_submit batches, kkx_run_staged /
 *                 kkx_fetch_staged, kkx_infer_programs) for runs that start after the call.  Each item (utterance), or
 *                 program of kkx_infer_programs, is measured and scaled on its own, on its 24 kHz model waveform x
 *                 (n samples), before resampling and integer conversion, so it gets the same gain at every "out_rate":
 *                 1. K-weighting (ITU-R BS.1770-4): two biquads designed in double at fs = 24000 with libebur128's
 *                    analog parameters and the bilinear transform, K = tan(pi f0 / fs) -- shelf f0 =
 *                    1681.974450955533 Hz, G = 3.999843853973347 dB, Q = 0.7071752369554196, Vb = Vh^0.4996667741545416;
 *                    high-pass f0 = 38.13547087602444 Hz, Q = 0.5003270373238773, numerator 1, -2, 1 (at fs = 48000
 *                    these are the standard's coefficient table); zero state at the item's first sample.
 *                 2. Blocks of 400 ms (9600 samples) on a 100 ms hop (2400), from sample 0, whole blocks only:
 *                    z_j = mean square of the K-weighted block, l_j = -0.691 + 10 log10 z_j.
 *                 3. Gating: absolute gate l_j > -70; relative gate Gamma_r = -0.691 + 10 log10(mean z over the
 *                    absolute-gated blocks) - 10; L = -0.691 + 10 log10(mean z over blocks with l_j > -70 and
 *                    l_j > Gamma_r) (strict comparisons).  L is undefined when no block passes: items shorter than
 *                    400 ms (fewer than 16 frames) and silence.
 *                 4. True peak tp = max |resample_poly(x, 4, 1)| over the item, with scipy's default filter
 *                    h = 4 firwin(81, 1/4, ("kaiser", 5.0)) and zeros outside the item; dBTP = 20 log10 tp.  (A
 *                    deliberate deviation from the 48-tap example filter of the BS.1770 annex: the same design rule
 *                    as "out_rate", so the measurement is reproducible with scipy alone.)
 *                 5. Gain g = 10^((target - L) / 20); if tp g > 10^(ceiling / 20) then g = 10^(ceiling / 20) / tp
 *                    (a static gain: no limiter, no compressor).  Undefined L: g = 1 exactly.
 *                 6. Each returned sample is fp32(y * g), y being the sample the same run returns with the option off
 *                    (the iSTFT sample at 24 kHz, the resampling FIR's output at other rates); PCM16, G.711 and FLAC
 *                    follow from that value by their rules above, so an item with undefined L comes back bit-identical
 *                    to normalisation off.  The measurement runs in fp32 on the device (the filter restarted from zero
 *                    state 4800 samples before each 2400-sample segment, sums in double); values and bits of an item
 *                    do not depend on its batch, frame group or pass.  One loudness across several items (program
 *                    loudness of a request split into chunks) is kkx_infer_programs.  Rule 5 caps the gain, so an
 *                    item whose peak-to-loudness ratio exceeds ceiling - target comes back quieter than the target;
 *                    "limiter" reaches it.  Measurement without normalisation, loudness range and maximum momentary /
 *                    short-term loudness: "loudness_report".  Not provided: compression, measurement at the output rate.
 *   "limiter"     lookahead true-peak limiter: 0 (DEFAULT) = off, every bit, byte and launch as without it; 1 = on.
 *                 Any other value is KKX_ERR_ARG and the session keeps its setting.  One setting per session, followed
 *                 by the same entry points as "loudness_target" for runs that start after the call.  It works on each
 *                 item's (program's) 24 kHz model waveform x (n samples), before resampling and integer conversion,
 *                 with or without "loudness_target".  c = 10^(C / 20), C = "true_peak_max" / 100.  Fixed constants:
 *                 lookahead Ha = 120 samples (5 ms), FIR guard Hb = 10 (the half-support of the 4x true-peak filter),
 *                 largest reduction Rmax = 12 dB, release slope s = 0.0025 dB per sample (60 dB/s), release window
 *                 W = Rmax / s = 4800 samples.
 *                 1. Static gain: g = 10^((T - L) / 20) when "loudness_target" T != 0 and L is defined, else g = 1;
 *                    instead of rule 5's cap, if tp g > c 10^(Rmax / 20) then g = c 10^(Rmax / 20) / tp (tp of rule 4;
 *                    this cap applies also when L is undefined or T = 0).
 *                 2. Detector: p[i] = max over j = 0..3 of |u[4 i + j]|, u = resample_poly(x, 4, 1) with rule 4's
 *                    filter and zeros outside the item; q[i] = min(0, C - 20 log10(g p[i])), q = 0 where p = 0 and
 *                    outside [0, n).
 *                 3. Hold: h[i] = min over k in [-Hb, Ha + Hb] of q[i + k].
 *                 4. Release: e[i] = min(0, min over m in [i - W, i] of (h[m] + (i - m) s)) -- a linear-in-dB recovery
 *                    without a recurrence (h >= -Rmax makes older terms >= 0), so tiles of an item are computed
 *                    independently.
 *                 5. Attack: G[i] = mean over k = 0..Ha of 10^(e[i - k] / 20), e = 0 before the first sample; G = 1.0
 *                    exactly where e is 0 throughout the window.  Every gain within Hb of a detected peak is at most
 *                    that peak's required gain.
 *                 6. v[i] = fp32(x[i] fp32(g G[i])).
 *                 7. Trim: tp_v = max |resample_poly(v, 4, 1)|, t = min(1, c / tp_v).
 *                 8. y = v resampled under the "out_rate" rule; each returned sample is fp32(y t).  PCM16, G.711 and
 *                    FLAC follow from that value by their rules.
 *                 Consequences: the 24 kHz-domain output has true peak <= c to fp32 rounding, so PCM16, G.711 and FLAC
 *                 never clip; an item the limiter does not touch (G = 1, t = 1) is bit-identical at 24000 to the
 *                 limiter-off run with the same g (with loudness off: a silent item, or one whose true peak is under the
 *                 ceiling, is bit-identical to the plain output); an item's (program's) bits do not depend on its
 *                 batch, frame group, "max_tokens" pass, coalescing or kkx_submit.  kkx_last_loudness keeps reporting
 *                 L and dBTP of the input and gain = g of step 1.  Device work: the loudness launches (three, also
 *                 when "loudness_target" is 0; loud_peak writes p), then "lim_envelope", "loud_peak" on v and
 *                 "lim_trim" -- 3 launches more than loudness alone per frame group that completes a program (6 more
 *                 than plain output when "loudness_target" is 0; a resampling pass runs also at 24000).
 *                 Not provided: compression, a limiter at the output rate, user-set lookahead / release / Rmax.
 *   "loudness_report"  the EBU R128 / Tech 3341 report of every item (program): 0 (DEFAULT) = off, every bit, byte and
 *                 launch as without it; 1 = on.  Any other value is KKX_ERR_ARG and the session keeps its setting.  One
 *                 setting per session, followed by the same entry points as "loudness_target" for runs that start
 *                 after the call.  Each item (program of kkx_infer_programs) is measured on its 24 kHz model waveform x,
 *                 the x that rules 1-4 of "loudness_target" measure.
 *                 Measure-only: with "loudness_target" = 0 and "limiter" = 0, every returned sample, byte and FLAC file
 *                 is bit-identical to the same run with the option off, at every "out_rate" and in every encoding; the
 *                 applied gain is exactly 1 (rule 5's ceiling does not apply: measuring never rescales).  With
 *                 "loudness_target" or "limiter" on, the option adds the statistics alone: gains, samples and
 *                 kkx_last_loudness are as without it.
 *                 After a synchronous call that ran with it, kkx_last_loudness succeeds also when "loudness_target"
 *                 was 0 (gain = the applied g: 1 in measure-only, step 1's g under the limiter), and
 *                 kkx_last_loudness_range reports, on the segment energies e_i of rule 2 (K-weighted sum of squares of
 *                 segment i, 2400 samples; n_seg = floor(n / 2400)):
 *                 1. Momentary: z_j = (e_j + e_{j+1} + e_{j+2} + e_{j+3}) / 9600 for every whole 400 ms block (rule 2's
 *                    z_j), summed in double in ascending order; M = -0.691 + 10 log10(max_j z_j).
 *                 2. Short-term: s_j = (sum over i = j .. j + 29 of e_i) / 72000 for every whole 3 s window on the
 *                    100 ms hop from sample 0 (j = 0 .. n_seg - 30), summed in double in ascending i;
 *                    l_s = -0.691 + 10 log10 s_j; S = -0.691 + 10 log10(max_j s_j).
 *                 3. Gates (EBU Tech 3342): absolute l_s > -70; relative Gamma = -0.691 + 10 log10(mean s over the
 *                    absolute-gated windows) - 20, l_s > Gamma (strict comparisons, as in rule 3).
 *                 4. Range: the m windows that pass, their s sorted a_0 <= .. <= a_{m-1}; lo = floor((10 (m - 1) +
 *                    50) / 100), hi = floor((95 (m - 1) + 50) / 100) (nearest rank, halves up, in integers);
 *                    LRA = 10 log10(a_hi / a_lo) LU (0 for m = 1).
 *                 5. Undefined: M is NaN without a whole 400 ms block (n < 9600); S and LRA are NaN without a whole 3 s
 *                    window (n < 72000); LRA is NaN when no window passes the gates.  M and S are -inf for silence.
 *                 6. The values describe x, unscaled (as kkx_last_loudness does): under a static gain g the output's M
 *                    and S are these plus 20 log10 g and its LRA is the same; with the limiter on they are not the
 *                    output's values.
 *                 Every value is a function of the program's samples alone: not of its batch, position, frame group,
 *                 "max_tokens" pass, coalescing or kkx_submit.  Device work: the three loudness launches (also when
 *                 "loudness_target" is 0), then "loud_short" (one thread per 3 s window) and "loud_range" (one CTA per
 *                 program: maxima, gates, and the 10 % / 95 % points by an exact radix select) -- 2 launches more than
 *                 loudness alone per frame group that completes a program; measure-only at 24000 adds 3 + 2 + 1 (the
 *                 resampling pass-through, without a gain) to plain output.
 *                 Not provided: measurement at the output rate or of the limiter's output, a momentary / short-term
 *                 time series (a loudness curve), reports of coalesced and kkx_submit batches.
 *   "flac_lpc_order"  linear prediction in FLAC output: 0 (DEFAULT) = off, every byte and launch as without it, for
 *                 every entry point; p in 1..12 (12: the streamable-subset limit up to 48 kHz, RFC 9639 section 7) adds
 *                 one LPC candidate of order p per frame.  Any other value is KKX_ERR_ARG and the session keeps its
 *                 setting.  One setting per session, followed by kkx_infer_batch_flac and by KKX_ENC_FLAC
 *                 kkx_infer_programs runs that start after the call; no other encoding is affected.  Frame i's
 *                 subframe (x = its bs int16 samples), in addition to the kkx_infer_batch_flac rules:
 *                 1. Eligibility: CONSTANT frames stay CONSTANT; a frame has an LPC candidate only if p < bs.
 *                 2. Window (integers only): M[k] = nint(2^15 0.5 (1 - cos(pi (k + 0.5) / 1024))), k = 0..1023,
 *                    nint(v) = floor(v + 0.5), designed in double on the host.  L = bs >> 2; W[i] = 2^15 for
 *                    L <= i < bs - L; for i < L, W[i] = W[bs - 1 - i] = M[(i 1024) / L] (integer division; L = 0:
 *                    no taper).  xw[i] = (x[i] W[i] + 2^14) >> 15 (arithmetic shift).
 *                 3. Autocorrelation: R[l] = sum over i = l..bs-1 of xw[i] xw[i - l], l = 0..p, exact in int64
 *                    (|R| < 2^42), then converted to double (exact).
 *                 4. Levinson-Durbin in IEEE binary64, one rounding per operation, no fused multiply-add, in this
 *                    order: err = R[0]; for i = 1..p: acc = R[i]; for j = 1..i-1 ascending acc = acc - a[j] R[i - j];
 *                    k = acc / err; a'[j] = a[j] - k a[i - j] for j = 1..i-1 (the old a), a'[i] = k;
 *                    err = err (1 - k k).  No candidate if R[0] = 0 or err <= 0 after any step.
 *                 5. Quantisation, precision 12: cmax = max |a_j|, no candidate if 0; e = the exponent of
 *                    frexp(cmax) (cmax = m 2^e, 0.5 <= m < 1); shift = min(15, 11 - e), no candidate if < 0; ef = 0,
 *                    for j = 1..p: ef = ef + a_j 2^shift, q_j = clamp(floor(ef + 0.5), -2048, 2047), ef = ef - q_j.
 *                 6. Residual: e[s] = x[s] - ((sum over j = 1..p of q_j x[s - j]) >> shift), s = p..bs-1 (the sum
 *                    exact in int32); no candidate if any folded u >= 2^20.
 *                 7. Cost 8 + 16 p + 4 + 5 + 12 p + 6 + the partition / Rice cost of FIXED with o = p (partition
 *                    order q with (bs >> q) > p, ties to the smaller q, then k).  The cheaper of the best FIXED and
 *                    the LPC candidate is picked, ties going to FIXED; VERBATIM only if strictly cheaper than that
 *                    pick.  So no frame is larger than with the option off, and a stream where LPC never wins is
 *                    byte-identical to it.
 *                 8. Bitstream: subframe header 0, type 32 + p - 1, wasted bits 0; p warm-up samples (16 bits each);
 *                    precision - 1 = 11 (4 bits); shift (5-bit two's complement, 0..15); q_1..q_p (12 bits each, q_1
 *                    multiplies x[s - 1]); the residual as for FIXED (method 00, 4-bit partition order, 4-bit k per
 *                    partition, the first partition holding (bs >> q) - p residuals).
 *                 Frame headers, CRCs, STREAMINFO and MD5 = 0 as without the option.  Purity and identity as for FLAC
 *                 programs: a file's bytes are a function of its samples alone.  Device work: the same three
 *                 launches; flac_analyze runs its LPC variant, which designs the predictor on the block it holds.
 * kkx_get_stat keys: "launches", "last_frames", "gpu_us", "precision", "coalesced_batches",
 * "coalesced_requests", "coalesced_largest", "async_batches", "async_requests", "frame_groups",
 * "group_first:<g>" (first item of frame group g of the last run), "weights_sessions" (sessions sharing this
 * ctx's device weight set), "weights_bytes", "weights_from_onnx", "graph_replays", "out_rate", "loudness_target",
 * "true_peak_max", "loudness_items" (items -- programs after kkx_infer_programs -- kkx_last_loudness reports now; 0
 * if it would fail with KKX_ERR_STATE), "limiter", "limiter_items" (the same for kkx_last_limiter), "loudness_report"
 * (the option's value), "flac_lpc_order" (the option's value). */
KKX_API int kkx_set_option(kkx_ctx* ctx, const char* key, int64_t value);
KKX_API int64_t kkx_get_stat(kkx_ctx* ctx, const char* key); /* "launches", "last_frames", "gpu_us" ... */

/* What loudness normalisation (or "loudness_report") measured and applied in the last SYNCHRONOUS call on the ctx
 * (kkx_infer without "coalesce", kkx_infer_batch and its _voices / _pcm16 / _g711 / _flac forms, kkx_run_staged), in
 * item order, over every pass of a "max_tokens" split; after kkx_infer_programs, in program order (one entry per
 * program).  Per item: lufs = integrated loudness L (NaN when undefined), true_peak_dbtp = 20 log10 tp of the unscaled
 * item (-inf for silence), gain = the applied g.  Each pointer is nullable and receives `batch` floats.
 * KKX_ERR_STATE if no synchronous call has completed or that call ran with "loudness_target" = 0 and
 * "loudness_report" = 0; KKX_ERR_ARG if `batch` is not that call's item count.  Coalesced callers and kkx_submit
 * batches are normalised but not reported here (a batch of several callers has no per-caller report). */
KKX_API int kkx_last_loudness(kkx_ctx* ctx, int32_t batch, float* lufs, float* true_peak_dbtp, float* gain);

/* What the limiter ("limiter" = 1) did in the last SYNCHRONOUS call, with kkx_last_loudness's scope, order and errors
 * (KKX_ERR_STATE when that call ran with the limiter off).  Per item (program): max_reduction_db =
 * -20 log10(t min over i of G[i]) (>= 0; 0 = untouched), true_peak_dbtp = 20 log10(t tp_v), the output's true peak.
 * Each pointer is nullable and receives `batch` floats. */
KKX_API int kkx_last_limiter(kkx_ctx* ctx, int32_t batch, float* max_reduction_db, float* true_peak_dbtp);

/* The EBU R128 statistics of "loudness_report" (rules 1-6 there) for the last SYNCHRONOUS call, with kkx_last_loudness's
 * scope, order and errors (KKX_ERR_STATE when that call ran with "loudness_report" = 0; KKX_ERR_ARG when `batch` is
 * not its item or program count).  Per item (program): loudness_range_lu = LRA (EBU Tech 3342), max_momentary_lufs =
 * M, max_short_term_lufs = S; NaN where undefined.  They describe the unscaled 24 kHz waveform: under the applied gain
 * g the output's M and S are 20 log10 g higher and its LRA is the same.  Each pointer is nullable and receives `batch`
 * floats. */
KKX_API int kkx_last_loudness_range(kkx_ctx* ctx, int32_t batch, float* loudness_range_lu, float* max_momentary_lufs,
                                    float* max_short_term_lufs);

/* Per-kernel device timing of the last run (CUDA events on the library's stream, one after every
 * launch).  kkx_profile_json writes {"conv_flops": F, "gpu_us": T, "kernels": {name: [launches,
 * total_us]}} and returns the full length of the text. */
KKX_API int kkx_profile_enable(kkx_ctx* ctx, int enable);
KKX_API int64_t kkx_profile_json(kkx_ctx* ctx, char* buf, int64_t capacity);

/* Library / build identification, e.g. "kkx 0.1 sm_100a". */
KKX_API const char* kkx_version(void);

#ifdef __cplusplus
}
#endif
#endif /* KKX_H_ */
