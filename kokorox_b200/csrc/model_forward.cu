// model_forward.cu -- the forward pass proper: token phase (ALBERT, DurationEncoder, duration
// head, TextEncoder) and frame phase (length regulation, F0/N predictor, Decoder, Generator,
// iSTFT).  SURVEY.md Appendix A.1 - A.10; replaces ort_koko.rs:79 `sess.run`.
#include "model.h"
#include <algorithm>
#include <cmath>
#include <cstdlib>

namespace kkx {

namespace {
// diagnostics: per-role phase cycle counters of the fused res-block conv (KKX_ARB_TIMING=1 on a
// -DKKX_ARB_TIMING build); 4 variants (conv1/conv2 x C128/C256) x 32 slots
long long* g_arb_timing = nullptr;
long long* arb_timing_buf() {
  static const bool on = env_flag("KKX_ARB_TIMING", false);
  if (!on) return nullptr;
  if (!g_arb_timing) {
    KKX_CUDA(cudaMalloc(&g_arb_timing, 128 * sizeof(long long)));
    KKX_CUDA(cudaMemset(g_arb_timing, 0, 128 * sizeof(long long)));
  }
  return g_arb_timing;
}
ConvArgs gemm_args(const Level& L, const float* in, int ldi, int K, const float* w, const float* bias,
                   int N, float* out, int ldo, int ocol) {
  ConvArgs a;
  a.in = in; a.ldi = ldi; a.in_off = L.d_off; a.in_len = L.d_len;
  a.m_len = L.d_len; a.max_m = L.max_len; a.B = L.B; a.sum_m = L.sum_len;
  a.w = w; a.bias = bias; a.Ci = K; a.Co = N;
  a.out = out; a.ldo = ldo; a.ocol = ocol; a.out_off = L.d_off;
  return a;
}
// what every tensor-core launch fills alike: input rows of item b from Lin, output rows m of Lm stored at the rows of
// Lout, epilogue and residual
TcConvArgs tc_args(const Level& Lin, const Level& Lm, const Level& Lout, const float* bias, float* out, int ldo, int ocol,
                   const ConvOpt& o) {
  TcConvArgs a;
  a.eact = o.eact; a.dil = o.dil; a.pad = o.pad;
  a.in_off = Lin.d_off; a.m_len = Lm.d_len; a.max_m = Lm.max_len; a.B = Lm.B; a.sum_m = Lm.sum_len;
  a.tile_start = Lm.d_tiles128; a.ntiles_m = Lm.ntiles128;
  a.bias = bias; a.out = out; a.ldo = ldo; a.ocol = ocol; a.out_off = Lout.d_off; a.ors = o.ors; a.oro = o.oro;
  a.res = o.res; a.ldr = o.ldr; a.res_off = o.Lres ? o.Lres->d_off : nullptr; a.res_shift = o.res_shift;
  a.oscale = o.oscale;
  return a;
}
}  // namespace

void arb_timing_dump() {
  if (!g_arb_timing) return;
  attention_timing_dump();
  long long h[128];
  cudaDeviceSynchronize();
  cudaMemcpy(h, g_arb_timing, sizeof h, cudaMemcpyDeviceToHost);
  cudaMemset(g_arb_timing, 0, sizeof h);
  fprintf(stderr, "[tf32x3 timing, CTA 0 of every launch] (Mcycles) TMA wait_empty %.2f issue %.2f | MMA wait_full %.2f wait_ring %.2f issue %.2f |"
          " EPI wait_chain %.2f drain %.2f wait_final %.2f final %.2f\n", h[100] / 1e6, h[101] / 1e6, h[104] / 1e6, h[105] / 1e6, h[106] / 1e6,
          h[108] / 1e6, h[109] / 1e6, h[110] / 1e6, h[111] / 1e6);
  const char* nm[4] = {"conv1 C128", "conv2 C128", "conv1 C256", "conv2 C256"};
  for (int v = 0; v < 3; v++) {
    const long long* t = h + v * 32;
    fprintf(stderr, "[arb timing %s] (Mcycles)  TMA wait %.2f issue %.2f | MMA wait_tempty %.2f wait_fullA %.2f wait_fullB %.2f issue %.2f |"
            " EPI wait_tfull %.2f tmem_ld %.2f barA %.2f sts %.2f barB %.2f compute+store %.2f fetch %.2f stats %.2f tile %.2f |"
            " PROD issue %.2f coef %.2f wait_emptyA %.2f transform %.2f mov+arrive %.2f\n", nm[v],
            t[0] / 1e6, t[1] / 1e6, t[4] / 1e6, t[5] / 1e6, t[6] / 1e6, t[7] / 1e6, t[8] / 1e6, t[9] / 1e6, t[10] / 1e6, t[11] / 1e6,
            t[12] / 1e6, t[13] / 1e6, t[14] / 1e6, t[15] / 1e6, t[16] / 1e6, t[20] / 1e6, t[21] / 1e6, t[22] / 1e6, t[23] / 1e6, t[24] / 1e6);
  }
}

void Model::tc_conv(const void* abuf, int rows_total, const TcW& w, const Level& Lin, const Level& Lm, const float* bias,
                    float* out, int ldo, int ocol, const Level& Lout, const ConvOpt& o) {
  alignas(64) unsigned char tmA[128];
  if (g_dry_run) return;
  make_tmap_bf16(tmA, abuf, w.Cpad, rows_total, w.Cpad, 128);
  TcConvArgs a = tc_args(Lin, Lm, Lout, bias, out, ldo, ocol, o);
  a.tmA = tmA; a.tmB = w.tmap;
  a.Cpad = w.Cpad; a.Ci = w.Ci; a.Co = w.Co; a.ks = w.ks;
  if (opt.conv_pair && w.pair_map(w.Co)) {      // CTA-pair kernel (taken when the batch gives every pair a tile)
    a.tmB_c = w.pair_map(w.Co); a.pair = 1;
  }
  launch_conv_tc(a, cur_);
}

bool Model::gemm(const Level& Lin, const Level& Lm, const float* in, int ldi, int K, const float* w, const TcW32* w32,
                 const float* bias, int N, float* out, int ldo, int ocol, const ConvOpt& o) {
  cudaStream_t st = cur_;
  if (opt.precision == 1 && w32 && w32->hi && split_hi_ && (size_t)Lin.rows * w32->Cpad <= split_cap_) {
    if (g_dry_run) return false;
    const bool f16 = opt.split_f16 && w32->h_hi;
    alignas(64) unsigned char tA[128], tA2[128];
    TcConvArgs a = tc_args(Lin, Lm, Lm, bias, out, ldo, ocol, o);
    if (f16) {
      const bool planes_in = o.in_hi && o.in_lo && !o.pscale && o.pact == ACT_NONE && o.ks == 1;
      // the scratch planes hold 2-byte elements in this mode (half of the fp32-sized buffers is used)
      if (!planes_in)
        launch_apply_f16x2(in, ldi, K, o.pscale, o.pshift, o.pact, o.pslope, split_hi_, split_lo_, w32->Cpad, Lin.rows,
                           Lin.d_off, Lin.d_len, Lin.B, Lin.max_len, st);
      make_tmap_f16(tA, planes_in ? o.in_hi : split_hi_, w32->Cpad, Lin.rows, w32->Cpad, 128);
      make_tmap_f16(tA2, planes_in ? o.in_lo : split_lo_, w32->Cpad, Lin.rows, w32->Cpad, 128);
      a.tmB = w32->tm16_hi; a.tmB2 = w32->tm16_lo; a.f16 = 1;
      a.wscale = w32->wscale16 / kSplitF16Scale;
      if (w32->has_c) { a.tmB_c = w32->tm16_hi_c; a.tmB2_c = w32->tm16_lo_c; a.pair = opt.gemm_pair; }
    } else {
      launch_apply_tf32(in, ldi, K, o.pscale, o.pshift, o.pact, o.pslope, split_hi_, split_lo_, w32->Cpad, Lin.rows,
                        Lin.d_off, Lin.d_len, Lin.B, Lin.max_len, st);
      make_tmap_f32(tA, split_hi_, w32->Cpad, Lin.rows, w32->Cpad, 128);
      make_tmap_f32(tA2, split_lo_, w32->Cpad, Lin.rows, w32->Cpad, 128);
      a.tmB = w32->tm_hi; a.tmB2 = w32->tm_lo;
      if (w32->has_c) { a.tmB_c = w32->tm_hi_c; a.tmB2_c = w32->tm_lo_c; }
    }
    a.tmA = tA; a.tmA2 = tA2; a.tf32 = 1; a.nprod = 3;
    a.Cpad = w32->Cpad; a.Ci = K; a.Co = N; a.ks = o.ks;
    if (long long* tim = arb_timing_buf()) a.timing = tim + 100;   // diagnostics: slots 100..111
    bool planes_out = false;
    if (o.out_hi && o.out_lo && f16 && N % 4 == 0 && o.out_ld >= N && ocol == 0 && conv_tc_takes_pair(a)) {
      a.out_hi = o.out_hi; a.out_lo = o.out_lo; a.out_pl_ld = o.out_ld; a.out = nullptr;
      planes_out = true;
    } else if (o.attn_scratch && f16 && N == 2304 && o.eact == ACT_NONE && !o.res && o.oscale == 1.f && conv_tc_takes_pair(a)) {
      attention_umma_planes(o.attn_scratch, Lm.rows, Lm.B, a.attn_pl);
      a.out = nullptr;
      planes_out = true;
    }
    launch_conv_tc(a, st);
    return planes_out;
  }
  ConvArgs c = gemm_args(Lm, in, ldi, K, w, bias, N, out, ldo, ocol);
  c.in_off = Lin.d_off; c.in_len = Lin.d_len;
  c.ks = o.ks; c.dil = o.dil; c.pad = o.pad; c.ors = o.ors; c.oro = o.oro; c.eact = o.eact;
  c.pscale = o.pscale; c.pshift = o.pshift; c.pld = K; c.pact = o.pact; c.pslope = o.pslope;
  c.res = o.res; c.ldr = o.ldr; c.res_off = o.Lres ? o.Lres->d_off : nullptr; c.res_shift = o.res_shift;
  c.oscale = o.oscale;
  launch_conv_f32(c, st);
  return false;
}

// ------------------------------------------------------------------------------------------
// Token phase: everything at phoneme-token rate, for the whole batch.
size_t Model::token_arena_bytes() const {
  const size_t R = (size_t)tokL_.rows;
  return R * (128 + 768 * 4 + 2304 + 2048 + 2048 + 640 * 2 + 512 * 6 + 64 + 16 + 2 * 2048 + 2048 + 2 * 512 + (768 + 2048)) * sizeof(float) +
         (size_t)B_ * (W.sty_pro_n + W.sty_dec_n + 1024) * sizeof(float) + (4 << 20) +
         (opt.attention_umma ? attention_umma_scratch_floats((int)R, B_) * sizeof(float) + 1024 : 0);
}

void Model::token_phase(Run& r) {
  // host buffers the D2H at the end of the phase lands in (pinned; sized before any capture)
  const size_t R = (size_t)tokL_.rows;
  if (R > h_pred_dur_cap_) {
    KKX_CUDA(cudaStreamSynchronize(stream_));
    if (h_pred_dur_) cudaFreeHost(h_pred_dur_);
    h_pred_dur_ = nullptr; h_pred_dur_cap_ = 0;
    KKX_CUDA(cudaMallocHost(&h_pred_dur_, (R + R / 4) * sizeof(int)));
    h_pred_dur_cap_ = R + R / 4;
  }
  if ((size_t)B_ > h_T_cap_) {
    KKX_CUDA(cudaStreamSynchronize(stream_));
    if (h_T_) cudaFreeHost(h_T_);
    h_T_ = nullptr; h_T_cap_ = 0;
    KKX_CUDA(cudaMallocHost(&h_T_, ((size_t)B_ + 64) * sizeof(int)));
    h_T_cap_ = (size_t)B_ + 64;
  }
  const size_t need = token_arena_bytes();
  if (need > tokA_.capacity()) {
    KKX_CUDA(cudaStreamSynchronize(stream_));
    clear_graphs();                      // captured nodes embed addresses of the old arena
    tokA_.reserve(need);
  }
  // Single-utterance calls: the launch sequence of the token phase depends only on the token count, so it is
  // captured once (on the second call with that count) and replayed afterwards -- ~190 launches become one.
  const bool graph_ok = opt.latency_graphs && B_ == 1 && !debug_ && !stats.profile && !stats.check_each && inj_dur_.empty();
  if (graph_ok) {
    const GraphKey key{tok_len_[0], opt.lstm_fast_gates * 32 + opt.precision * 16 + opt.attention_umma * 8 + opt.split_f16 * 4 + opt.gemm_pair * 2 + opt.fuse_planes, tokA_.base(), d_ids_, tokL_.d_off, h_T_, h_pred_dur_};
    auto it = graphs_.find(key);
    if (it != graphs_.end() && it->second.exec) {
      r = it->second.run;
      if (cudaGraphLaunch(it->second.exec, stream_) == cudaSuccess) {
        stats.launches += it->second.launches;
        graph_replays++;
        token_finish(r);
        return;
      }
      cudaGetLastError();
      cudaGraphExecDestroy(it->second.exec);
      graphs_.erase(it);
    } else if (it != graphs_.end()) {
      if (graphs_.size() > 64) clear_graphs();          // bound the cache; entries are cheap to rebuild
      GraphEntry e;
      const long long l0 = stats.launches;
      cudaGraph_t g = nullptr;
      KKX_CUDA(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
      capturing_ = true;
      token_issue(r);                                   // (throws -> Model::run ends the capture)
      capturing_ = false;
      KKX_CUDA(cudaStreamEndCapture(stream_, &g));
      const cudaError_t ie = cudaGraphInstantiate(&e.exec, g, 0);
      cudaGraphDestroy(g);
      if (ie != cudaSuccess) { cudaGetLastError(); e.exec = nullptr; }
      e.run = r;
      e.launches = stats.launches - l0;
      if (e.exec && cudaGraphLaunch(e.exec, stream_) == cudaSuccess) {
        graphs_[key] = e;
        graph_replays++;
        token_finish(r);
        return;
      }
      cudaGetLastError();
      if (e.exec) cudaGraphExecDestroy(e.exec);
      graphs_.erase(key);
      stats.launches = l0;                              // fall through to an eager run
    } else {
      graphs_[key] = GraphEntry();                      // first sighting: run eagerly (also warms kernel attributes)
    }
  }
  token_issue(r);
  token_finish(r);
}

void Model::token_issue(Run& r) {
  use_lane(0);
  cudaStream_t st = stream_;
  const Level& L = tokL_;
  const size_t R = (size_t)L.rows;
  const int B = B_;
  tokA_.reset();
  Arena& A = tokA_;
  const bool fork = can_fork(B);

  // style-parameter tables for every AdaIN / AdaLN of the model: two GEMMs over the batch
  r.styL = make_level(std::vector<int>{B}, A, 0);   // one "item" of B rows at row 0
  r.sty_pro = A.alloc<float>((size_t)B * W.sty_pro_n);
  r.sty_dec = A.alloc<float>((size_t)B * W.sty_dec_n);
  launch_conv_f32(gemm_args(r.styL, d_styles_ + 128, 256, 128, W.sty_pro_w, W.sty_pro_b, W.sty_pro_n,
                            r.sty_pro, W.sty_pro_n, 0), st);
  launch_conv_f32(gemm_args(r.styL, d_styles_, 256, 128, W.sty_dec_w, W.sty_dec_b, W.sty_dec_n,
                            r.sty_dec, W.sty_dec_n, 0), st);

  // scratch planes for the split-TF32 operand producer (largest K on this path: 2048; the text encoder's lane: 512)
  {
    float* hi = A.alloc<float>(R * 2048); float* lo = A.alloc<float>(R * 2048);
    set_lane_scratch(0, hi, lo, R * 2048);
    float* hi1 = A.alloc<float>(R * 512); float* lo1 = A.alloc<float>(R * 512);
    set_lane_scratch(1, hi1, lo1, R * 512);
  }

  // ---- TextEncoder (A.4) -- independent of the duration path: on lane 1 for small batches, so that its CNN and
  // LSTM run beside ALBERT instead of after it
  float* ta = A.alloc<float>(R * 512);
  float* tb = A.alloc<float>(R * 512);
  float* xp_te = A.alloc<float>(R * 2048);
  r.t_en = A.alloc<float>(R * 512);
  auto text_encoder = [&] {
    cudaStream_t ts = cur_;
    launch_embed_rows(d_ids_, W.temb, 512, ta, 512, L.d_off, L.d_len, B, L.max_len, ts);
    ConvOpt k5;
    k5.ks = 5; k5.pad = 2;
    for (int i = 0; i < 3; i++) {
      gemm(L, L, ta, 512, 512, W.tcnn_w[i], &W.t_tcnn[i], W.tcnn_b[i], 512, tb, 512, 0, k5);
      LnArgs ln;
      ln.x = tb; ln.ldx = 512; ln.w = W.tln_g[i]; ln.b = W.tln_b[i]; ln.eps = 1e-5f; ln.slope = 0.2f;
      ln.out = ta; ln.ldo = 512; ln.off = L.d_off; ln.len = L.d_len; ln.B = B; ln.max_len = L.max_len;
      ln.C = 512;
      launch_layernorm(ln, ts);
    }
    gemm(L, L, ta, 512, 512, W.te_lstm.wih, &W.te_lstm.t_ih, W.te_lstm.bias, 2048, xp_te, 2048, 0);
    launch_lstm(xp_te, W.te_lstm.whhT, r.t_en, 512, 0, L.d_off, L.d_len, B, ts, opt.precision != 0 && opt.lstm_fast_gates);
  };
  if (fork) {
    fork_lane1();
    use_lane(1);
    text_encoder();
    use_lane(0);
  }

  // ---- ALBERT (A.2)
  float* e = A.alloc<float>(R * 128);
  float* h = A.alloc<float>(R * 768);
  float* h1 = A.alloc<float>(R * 768);
  float* ctx = A.alloc<float>(R * 768);
  float* tmp = A.alloc<float>(R * 768);
  float* qkv = A.alloc<float>(R * 2304);
  float* ff = A.alloc<float>(R * 2048);
  float* att_scratch = opt.attention_umma ? A.alloc<float>(attention_umma_scratch_floats((int)R, B)) : nullptr;
  // operand planes passed between LayerNorm / FFN and the next GEMM (fp16 hi + lo: R x C x 2 x 2 bytes = one float each)
  const bool pl_ok = planes_ok();
  void* p768h = pl_ok ? A.alloc_bytes(R * 768 * 2) : nullptr;
  void* p768l = pl_ok ? A.alloc_bytes(R * 768 * 2) : nullptr;
  void* p2048h = pl_ok ? A.alloc_bytes(R * 2048 * 2) : nullptr;
  void* p2048l = pl_ok ? A.alloc_bytes(R * 2048 * 2) : nullptr;
  bool h_planes = false;      // p768 holds the planes of h
  launch_albert_embed(d_ids_, W.word, W.pos, W.type, W.emb_lnw, W.emb_lnb, e, L.d_off, L.d_len, B,
                      L.max_len, st);
  gemm(L, L, e, 128, 128, W.map_w, &W.t_map, W.map_b, 768, h, 768, 0);
  for (int layer = 0; layer < 12; layer++) {
    ConvOpt oq;
    if (h_planes) { oq.in_hi = p768h; oq.in_lo = p768l; }
    if (pl_ok && att_scratch) oq.attn_scratch = att_scratch;   // Q/8, K, V^T planes straight from the GEMM's final warps
    const bool qkv_planes = gemm(L, L, h, 768, 768, W.qkv_w, &W.t_qkv, W.qkv_b, 2304, qkv, 2304, 0, oq);
    if (att_scratch) launch_attention_umma(qkv, att_scratch, ctx, L.d_off, L.d_len, B, L.max_len, L.rows, st, qkv_planes);
    else launch_attention(qkv, ctx, L.d_off, L.d_len, B, L.max_len, st);
    gemm(L, L, ctx, 768, 768, W.dense_w, &W.t_dense, W.dense_b, 768, tmp, 768, 0);
    LnArgs ln;
    ln.x = h; ln.ldx = 768; ln.res = tmp; ln.ldr = 768; ln.w = W.attn_lnw; ln.b = W.attn_lnb;
    ln.eps = 1e-12f; ln.out = h1; ln.ldo = 768; ln.off = L.d_off; ln.len = L.d_len; ln.B = B;
    ln.max_len = L.max_len; ln.C = 768;
    if (pl_ok) { ln.pl_hi = p768h; ln.pl_lo = p768l; ln.pl_ld = 768; }      // h1 as planes for the FFN GEMM
    launch_layernorm(ln, st);
    ConvOpt of;
    of.eact = ACT_GELU_NEW;
    if (pl_ok) { of.in_hi = p768h; of.in_lo = p768l; of.out_hi = p2048h; of.out_lo = p2048l; of.out_ld = 2048; }
    const bool ff_planes = gemm(L, L, h1, 768, 768, W.ffn_w, &W.t_ffn, W.ffn_b, 2048, ff, 2048, 0, of);
    ConvOpt oo;
    if (ff_planes) { oo.in_hi = p2048h; oo.in_lo = p2048l; }                // gelu(ffn) exists only as planes
    gemm(L, L, ff, 2048, 2048, W.ffo_w, &W.t_ffo, W.ffo_b, 768, tmp, 768, 0, oo);
    ln.x = tmp; ln.res = h1; ln.w = W.full_lnw; ln.b = W.full_lnb; ln.out = h;
    launch_layernorm(ln, st);                                                 // h (+ its planes for the next QKV / bert_encoder)
    h_planes = pl_ok;
  }
  capture("bert", h, 768, 0, 768, L, 0);

  // ---- bert_encoder + DurationEncoder (A.3)
  float* xa = A.alloc<float>(R * 640);
  float* xb = A.alloc<float>(R * 640);
  float* xp = A.alloc<float>(R * 2048);
  float* lo = A.alloc<float>(R * 512);
  {
    ConvOpt ob;
    if (h_planes) { ob.in_hi = p768h; ob.in_lo = p768l; }
    gemm(L, L, h, 768, 768, W.benc_w, &W.t_benc, W.benc_b, 512, xa, 640, 0, ob);
  }
  capture("d_en", xa, 640, 0, 512, L, 0);
  launch_bcast_cols(d_styles_, 256, 128, 128, xa, 640, 512, L.d_off, L.d_len, B, L.max_len, st);
  launch_bcast_cols(d_styles_, 256, 128, 128, xb, 640, 512, L.d_off, L.d_len, B, L.max_len, st);
  float* cur = xa; float* nxt = xb;
  for (int i = 0; i < 3; i++) {
    gemm(L, L, cur, 640, 640, W.dur_lstm[i].wih, &W.dur_lstm[i].t_ih, W.dur_lstm[i].bias, 2048, xp, 2048, 0);
    launch_lstm(xp, W.dur_lstm[i].whhT, lo, 512, 0, L.d_off, L.d_len, B, st, opt.precision != 0 && opt.lstm_fast_gates);
    LnArgs ln;
    ln.x = lo; ln.ldx = 512; ln.ada = r.sty_pro; ln.ada_ld = W.sty_pro_n; ln.ada_off = W.dur_ada[i];
    ln.eps = 1e-5f; ln.out = nxt; ln.ldo = 640; ln.ocol = 0; ln.off = L.d_off; ln.len = L.d_len;
    ln.B = B; ln.max_len = L.max_len; ln.C = 512;
    launch_layernorm(ln, st);
    std::swap(cur, nxt);
  }
  r.d = cur;
  capture("d", r.d, 640, 0, 640, L, 0);

  // ---- duration head (A.1, K4)
  gemm(L, L, r.d, 640, 640, W.pred_lstm.wih, &W.pred_lstm.t_ih, W.pred_lstm.bias, 2048, xp, 2048, 0);
  launch_lstm(xp, W.pred_lstm.whhT, lo, 512, 0, L.d_off, L.d_len, B, st, opt.precision != 0 && opt.lstm_fast_gates);
  capture("dur_lstm", lo, 512, 0, 512, L, 0);
  float* logits = A.alloc<float>(R * 50);
  gemm(L, L, lo, 512, 512, W.durp_w, &W.t_durp, W.durp_b, 50, logits, 50, 0);
  capture("dur_logits", logits, 50, 0, 50, L, 0);
  r.pred_dur = A.alloc<int>(R);
  float* durf = A.alloc<float>(R);
  r.cum = A.alloc<int>((size_t)B * 512);
  r.total = A.alloc<int>(B);
  launch_duration(logits, 50, d_speeds_, r.pred_dur, durf, L.d_off, L.d_len, B, L.max_len, st);
  capture("dur_float", durf, 1, 0, 1, L, 0);
  for (auto& kv : inj_dur_) {   // test hook: teacher-forced durations of single items
    const int b = kv.first;
    if (b >= B) throw ArgError("inject pred_dur: item index out of range");
    if ((int)kv.second.size() != L.len[b]) throw ArgError("inject pred_dur: length != n_tokens of the item");
    upload(r.pred_dur + L.off[b], kv.second.data(), kv.second.size() * sizeof(int));
  }
  launch_dur_scan(r.pred_dur, r.cum, 512, r.total, L.d_off, L.d_len, B, st);

  if (fork) join_lane1();
  else text_encoder();               // large batches: same stream, after the duration path
  capture("t_en", r.t_en, 512, 0, 512, L, 0);

  set_lane_scratch(0, nullptr, nullptr, 0);
  set_lane_scratch(1, nullptr, nullptr, 0);
  // ---- frame counts decide every later launch shape: they go to the host, and token_finish() waits for them
  KKX_CUDA(cudaMemcpyAsync(h_T_, r.total, B * sizeof(int), cudaMemcpyDeviceToHost, st));
  KKX_CUDA(cudaMemcpyAsync(h_pred_dur_, r.pred_dur, R * sizeof(int), cudaMemcpyDeviceToHost, st));
}

void Model::token_finish(Run& r) {
  const int B = B_;
  KKX_CUDA(cudaStreamSynchronize(stream_));   // the one mid-pipeline host sync
  r.T.resize(B);
  for (int b = 0; b < B; b++) {
    r.T[b] = h_T_[b];
    // 1 <= dur <= 50 / speed per token by construction; the cap bounds every later row / sample index (ADVICE r1)
    if (r.T[b] < 1 || r.T[b] > kMaxItemFrames)
      throw ArgError("item " + std::to_string(b) + ": " + std::to_string(r.T[b]) + " frames is outside 1.." +
                     std::to_string(kMaxItemFrames) + " (utterance too long for one call at this speed)");
  }
}

// ------------------------------------------------------------------------------------------
// AdainResBlk1d (A.6).  x [Lin rows, ci] -> out [Lout rows, co] (Lout = 2*Lin when upsampling).
void Model::adain_blk(Arena& A, const AdaBlkW& w, const float* x, int ldx, const Level& Lin, const Level& Lout,
                      const float* sty, int sld, float* out, int ldo, int ocol) {
  cudaStream_t st = cur_;
  const int B = Lin.B;
  const int nch_in = (Lin.max_len + kStatRows - 1) / kStatRows;
  const int nch_out = (Lout.max_len + kStatRows - 1) / kStatRows;
  float* part = A.alloc<float>((size_t)B * std::max(nch_in, nch_out) * 2 * std::max(w.ci, w.co));
  float* sc1 = A.alloc<float>((size_t)B * w.ci);
  float* sh1 = A.alloc<float>((size_t)B * w.ci);
  float* sc2 = A.alloc<float>((size_t)B * w.co);
  float* sh2 = A.alloc<float>((size_t)B * w.co);
  float* t = A.alloc<float>((size_t)Lout.rows * w.co);

  launch_colstats(x, ldx, w.ci, part, Lin.d_off, Lin.d_len, B, Lin.max_len, st);
  launch_adain_coef(part, w.ci, Lin.max_len, Lin.d_len, sty, sld, w.sty1, 1e-5f, sc1, sh1, B, st);
  ConvOpt k3;   // conv1 and conv2
  k3.ks = 3; k3.pad = 1;
  ConvOpt o2 = k3;   // conv2 adds the shortcut (x or its 1x1 conv) and scales the sum by 1/sqrt(2)
  o2.res = x; o2.ldr = ldx; o2.Lres = &Lin; o2.res_shift = w.up ? 1 : 0; o2.oscale = 0.70710678118654752440f;
  if (opt.precision == 1 && w.t1.w) {
    // tensor-core path: bf16 operands produced by the apply kernels, tcgen05 convs, fp32 results
    const int cpi = w.t1.Cpad, cpo = w.t2.Cpad;
    void* a1 = A.alloc_bytes((size_t)Lout.rows * cpi * 2);
    if (w.up)
      launch_pool_up_bf16(x, ldx, sc1, sh1, 0.2f, w.poolw, w.poolb, w.ci, a1, cpi, Lout.rows, Lin.d_off,
                          Lin.d_len, Lout.d_off, B, Lin.max_len, st);
    else
      launch_apply_bf16(x, ldx, w.ci, sc1, sh1, ACT_LRELU, 0.2f, nullptr, a1, cpi, Lin.rows, Lin.d_off,
                        Lin.d_len, B, Lin.max_len, st);
    tc_conv(a1, Lout.rows, w.t1, Lout, Lout, w.b1, t, w.co, 0, Lout, k3);
    launch_colstats(t, w.co, w.co, part, Lout.d_off, Lout.d_len, B, Lout.max_len, st);
    launch_adain_coef(part, w.co, Lout.max_len, Lout.d_len, sty, sld, w.sty2, 1e-5f, sc2, sh2, B, st);
    void* a2 = A.alloc_bytes((size_t)Lout.rows * cpo * 2);
    launch_apply_bf16(t, w.co, w.co, sc2, sh2, ACT_LRELU, 0.2f, nullptr, a2, cpo, Lout.rows, Lout.d_off,
                      Lout.d_len, B, Lout.max_len, st);
    if (w.w1x1) {
      void* a3 = A.alloc_bytes((size_t)Lin.rows * cpi * 2);
      float* s = A.alloc<float>((size_t)Lin.rows * w.co);
      launch_apply_bf16(x, ldx, w.ci, nullptr, nullptr, ACT_NONE, 0.f, nullptr, a3, cpi, Lin.rows, Lin.d_off,
                        Lin.d_len, B, Lin.max_len, st);
      tc_conv(a3, Lin.rows, w.t1x1, Lin, Lin, nullptr, s, w.co, 0, Lin);
      o2.res = s; o2.ldr = w.co;
    }
    tc_conv(a2, Lout.rows, w.t2, Lout, Lout, w.b2, out, ldo, ocol, Lout, o2);
    return;
  }
  // fp32-grade path (SIMT fp32, or split-TF32 tensor cores for the F0/N predictor blocks)
  if (w.up) {
    float* p = A.alloc<float>((size_t)Lout.rows * w.ci);
    launch_pool_up(x, ldx, sc1, sh1, 0.2f, w.poolw, w.poolb, w.ci, p, w.ci, Lin.d_off, Lin.d_len,
                   Lout.d_off, B, Lin.max_len, st);
    gemm(Lout, Lout, p, w.ci, w.ci, w.w1, &w.s1, w.b1, w.co, t, w.co, 0, k3);
  } else {
    ConvOpt o1 = k3;
    o1.pscale = sc1; o1.pshift = sh1; o1.pact = ACT_LRELU; o1.pslope = 0.2f;
    gemm(Lin, Lin, x, ldx, w.ci, w.w1, &w.s1, w.b1, w.co, t, w.co, 0, o1);
  }
  launch_colstats(t, w.co, w.co, part, Lout.d_off, Lout.d_len, B, Lout.max_len, st);
  launch_adain_coef(part, w.co, Lout.max_len, Lout.d_len, sty, sld, w.sty2, 1e-5f, sc2, sh2, B, st);

  if (w.w1x1) {
    float* s = A.alloc<float>((size_t)Lin.rows * w.co);
    gemm(Lin, Lin, x, ldx, w.ci, w.w1x1, &w.s1x1, nullptr, w.co, s, w.co, 0);
    o2.res = s; o2.ldr = w.co;
  }
  o2.pscale = sc2; o2.pshift = sh2; o2.pact = ACT_LRELU; o2.pslope = 0.2f;
  gemm(Lout, Lout, t, w.co, w.co, w.w2, &w.s2, w.b2, w.co, out, ldo, ocol, o2);
}

// AdaINResBlock1 (A.9): three (AdaIN -> Snake -> dilated conv -> AdaIN -> Snake -> conv) + residual
// iterations.  Reads x, uses xw/t1 as work buffers, writes (or accumulates) oscale * result to out.
bool Model::use_stream_bf16(int C, int k, int B) const {
  return opt.precision == 1 && opt.stream_bf16 && arb_conv_supported(C, k, 5, B);
}

void Model::arb(Arena& A, const ArbW& w, const float* x, const Level& L, const float* sty, int sld, float* xw,
                float* t1, float* out, float oscale, bool accumulate, const float* part_x, const void* x_bf16) {
  cudaStream_t st = cur_;
  const int B = L.B, C = w.c, k = w.k;
  const int nch = (L.max_len + kStatRows - 1) / kStatRows;
  float* part = A.alloc<float>((size_t)B * nch * 2 * C);
  float* sc = A.alloc<float>((size_t)B * C);
  float* sh = A.alloc<float>((size_t)B * C);
  const int dil[3] = {1, 3, 5};
  const float* cur = x;
  const bool tc = opt.precision == 1;
  void* abuf = tc ? A.alloc_bytes((size_t)L.rows * w.t1[0].Cpad * 2) : nullptr;
  if (tc) {
    // fused path (kernels_arb.cu): AdaIN + Snake inside the conv kernel, bf16 intermediate, column
    // statistics for the next AdaIN from the conv epilogues -- one colstats pass per res-block
    ArbConvArgs base;
    base.C = C; base.ks = k; base.off = L.d_off; base.len = L.d_len; base.B = B; base.sum_m = L.sum_len;
    const bool t256 = arb_tile_rows(C) == 256;
    base.tile_start = t256 ? L.d_tiles256 : L.d_tiles128;
    base.total_tiles = t256 ? L.ntiles256 : L.ntiles128;
    base.scale = sc; base.shift = sh; base.nchunk = nch;
    // bf16 residual stream: x0 arrives as bf16 (from the caller's add_rows_stats, or copied by the statistics pass
    // below), x1 / x2 live in `xw` as bf16 and the block output leaves in fp32
    const bool sb = use_stream_bf16(C, k, B);
    void* xb0 = nullptr;
    if (sb && !x_bf16) xb0 = A.alloc_bytes((size_t)L.rows * C * 2);
    // statistics of the block input: shared by the three res-blocks of a stage (computed once by the caller)
    if (!part_x) launch_colstats(cur, C, C, part, L.d_off, L.d_len, B, L.max_len, st, xb0);
    else if (sb && !x_bf16) throw ArgError("arb: a bf16 stream with caller-provided statistics needs the bf16 input too");
    const void* curb = sb ? (x_bf16 ? x_bf16 : xb0) : nullptr;
    long long* tim = arb_timing_buf();
    static const int tim_ks = env_int("KKX_ARB_TIMING_KS", 0);   // diagnostics: restrict the role counters to one kernel size
    if (tim_ks && tim_ks != k) tim = nullptr;
    for (int j = 0; j < 3; j++) {
      launch_adain_coef(j == 0 && part_x ? part_x : part, C, L.max_len, L.d_len, sty, sld, w.s1[j], 1e-5f, sc, sh, B, st);
      ArbConvArgs c1 = base;
      if (tim) c1.timing = tim + (C == 128 ? 0 : 64);
      c1.x = sb ? curb : (const void*)cur; c1.in_bf16 = sb ? 1 : 0; c1.alpha = w.a1[j]; c1.tmB = w.t1[j].tmap; c1.dil = dil[j];
      c1.pad = dil[j] * (k - 1) / 2; c1.bias = w.b1[j];
      c1.out_bf16 = static_cast<__nv_bfloat16*>(abuf); c1.part = part;
      launch_arb_conv(c1, st);
      launch_adain_coef(part, C, L.max_len, L.d_len, sty, sld, w.s2[j], 1e-5f, sc, sh, B, st);
      float* dst = (j == 2) ? out : xw;
      ArbConvArgs c2 = base;
      if (tim) c2.timing = tim + (C == 128 ? 32 : 96);
      c2.x = abuf; c2.in_bf16 = 1; c2.alpha = w.a2[j]; c2.tmB = w.t2[j].tmap; c2.dil = 1; c2.pad = (k - 1) / 2;
      c2.bias = w.b2[j];
      if (sb) {
        c2.res = static_cast<const float*>(curb); c2.res_bf16 = 1;
        if (j == 2) { c2.out_f32 = out; c2.oscale = oscale; c2.accumulate = accumulate ? 1 : 0; }
        else { c2.out_bf16 = reinterpret_cast<__nv_bfloat16*>(xw); c2.part = part; curb = xw; }
      } else {
        c2.out_f32 = dst; c2.res = cur;
        if (j == 2) { c2.oscale = oscale; c2.accumulate = accumulate ? 1 : 0; } else c2.part = part;
      }
      launch_arb_conv(c2, st);
      cur = dst;
    }
    return;
  }
  for (int j = 0; j < 3; j++) {
    launch_colstats(cur, C, C, part, L.d_off, L.d_len, B, L.max_len, st);
    launch_adain_coef(part, C, L.max_len, L.d_len, sty, sld, w.s1[j], 1e-5f, sc, sh, B, st);
    ConvArgs c1 = gemm_args(L, cur, C, C, w.w1[j], w.b1[j], C, t1, C, 0);
    c1.ks = k; c1.dil = dil[j]; c1.pad = dil[j] * (k - 1) / 2;
    c1.pscale = sc; c1.pshift = sh; c1.pld = C; c1.pact = ACT_SNAKE; c1.palpha = w.a1[j];
    launch_conv_f32(c1, st);
    launch_colstats(t1, C, C, part, L.d_off, L.d_len, B, L.max_len, st);
    launch_adain_coef(part, C, L.max_len, L.d_len, sty, sld, w.s2[j], 1e-5f, sc, sh, B, st);
    float* dst = (j == 2) ? out : xw;
    ConvArgs c2 = gemm_args(L, t1, C, C, w.w2[j], w.b2[j], C, dst, C, 0);
    c2.ks = k; c2.dil = 1; c2.pad = (k - 1) / 2;
    c2.pscale = sc; c2.pshift = sh; c2.pld = C; c2.pact = ACT_SNAKE; c2.palpha = w.a2[j];
    c2.res = cur; c2.ldr = C; c2.res_off = L.d_off;
    if (j == 2) { c2.oscale = oscale; c2.accumulate = accumulate ? 1 : 0; }
    launch_conv_f32(c2, st);
    cur = dst;
  }
}

// Phase ph of the up-sampling conv reads input rows m + q0 - tap (q0 = ph < s/2) and writes output row
// s*m + q0*s + ph - s/2 + shift.
void Model::upsample(Arena& A, const float* x, const Level& Lin, float* out, const Level& Lout, int s, int shift,
                     const TcW& w_all, const std::vector<TcW>& w_tc, const std::vector<float*>& w32, const float* bias,
                     bool dry) {
  cudaStream_t st = cur_;
  const int Ci = w_all.Ci, Co = w_all.Co;
  void* xbf = nullptr;
  if (opt.precision == 1) {
    xbf = A.alloc_bytes((size_t)Lin.rows * w_all.Cpad * 2);
    launch_apply_bf16(x, Ci, Ci, nullptr, nullptr, ACT_LRELU, 0.1f, nullptr, xbf, w_all.Cpad, Lin.rows, Lin.d_off,
                      Lin.d_len, Lin.B, Lin.max_len, st);
  }
  ConvOpt o;
  o.dil = -1; o.ors = s;
  if (opt.precision == 1 && opt.fuse_phases && !dry) {   // all s phases in one launch
    alignas(64) unsigned char tmA[128];
    make_tmap_bf16(tmA, xbf, w_all.Cpad, Lin.rows, w_all.Cpad, 128);
    TcConvArgs a = tc_args(Lin, Lin, Lout, bias, out, Co, 0, o);
    a.tmA = tmA; a.tmB = w_all.tmap;
    a.Cpad = w_all.Cpad; a.Ci = Ci; a.Co = Co; a.ks = 2;
    a.nphase = s; a.phase_loop = opt.ups_phase_loop;
    for (int ph = 0; ph < s; ph++) {
      const int q0 = ph < s / 2 ? 1 : 0;
      a.phase_pad[ph] = -q0; a.phase_oro[ph] = q0 * s + ph - s / 2 + shift;
    }
    if (opt.conv_pair && w_all.pair_map(Co)) { a.tmB_c = w_all.pair_map(Co); a.pair = 1; }
    launch_conv_tc(a, st);
    return;
  }
  for (int ph = 0; ph < s; ph++) {
    const int q0 = ph < s / 2 ? 1 : 0;
    o.pad = -q0; o.oro = q0 * s + ph - s / 2 + shift;
    if (opt.precision == 1) {
      tc_conv(xbf, Lin.rows, w_tc[ph], Lin, Lin, bias, out, Co, 0, Lout, o);
      continue;
    }
    ConvArgs c = gemm_args(Lin, x, Ci, Ci, w32[ph], bias, Co, out, Co, 0);
    c.out_off = Lout.d_off;
    c.ks = 2; c.dil = o.dil; c.pad = o.pad; c.ors = o.ors; c.oro = o.oro;
    c.pact = ACT_LRELU; c.pslope = 0.1f;
    launch_conv_f32(c, st);
  }
}

void Model::res_stage(Arena& A, const ArbW* w, float* x, const float* xs, const Level& L, const float* sty, float* xw,
                      float* t, float* acc) {
  cudaStream_t st = cur_;
  const int C = w[0].c;
  float* px = nullptr;
  void* xb = nullptr;
  if (opt.precision == 1) {   // x += x_source and the statistics of the sum (input of three res-blocks) in one pass
    px = A.alloc<float>((size_t)L.B * ((L.max_len + kStatRows - 1) / kStatRows) * 2 * C);
    // (bf16 residual stream: the sum is written once, as the bf16 x all three res-blocks read)
    bool sb = true;
    for (int j = 0; j < 3; j++) sb = sb && use_stream_bf16(C, w[j].k, L.B);
    xb = sb ? A.alloc_bytes((size_t)L.rows * C * 2) : nullptr;
    launch_add_rows_stats(x, xs, x, C, px, L.d_off, L.d_len, L.B, L.max_len, st, xb);
  } else {
    launch_add_rows(x, xs, x, C, L.d_off, L.d_len, L.B, L.max_len, st);
  }
  for (int j = 0; j < 3; j++) arb(A, w[j], x, L, sty, W.sty_dec_n, xw, t, acc, 1.0f / 3.0f, j > 0, px, xb);
}

// ------------------------------------------------------------------------------------------
// Frame phase for items [b0, b1): length regulation, F0/N, decoder, generator, iSTFT.
void Model::frame_phase(Run& r, int b0, int b1, int k0, int k1, bool dry) {
  use_lane(0);
  cudaStream_t st = stream_;
  Arena& A = frA_;
  const int B = b1 - b0;
  // small batches: independent branches run on two streams (N | F0, harmonic source + noise blocks | decoder)
  const bool fork = !dry && can_fork(B);
  cudaStream_t st1 = fork ? stream2_ : stream_;
  std::vector<int> T(r.T.begin() + b0, r.T.begin() + b1), T2(B), T20(B), T120(B), one(B, 1);
  long long maxS = 0;
  for (int b = 0; b < B; b++) {
    T2[b] = 2 * T[b]; T20[b] = 20 * T[b]; T120[b] = 120 * T[b] + 1;
    maxS = std::max(maxS, 600LL * T[b]);
  }
  Level FR = make_level(T, A), FR2 = make_level(T2, A), G20 = make_level(T20, A), G120 = make_level(T120, A);
  // per-item views into batch-level (token-phase) arrays
  const int* tok_off = tokL_.d_off + b0;
  const int* tok_len = tokL_.d_len + b0;
  const int* cum = r.cum + (size_t)b0 * 512;
  const float* sty_pro = r.sty_pro + (size_t)b0 * W.sty_pro_n;
  const float* sty_dec = r.sty_dec + (size_t)b0 * W.sty_dec_n;
  // curve (F0 / N) offsets: element offsets == FR2 row offsets (ld 1); phase offsets; group-local sample offsets of
  // the harmonic source (s_loc); each item's offset in the run's 24 kHz waveform (s24)
  std::vector<int> ph_off(B);
  std::vector<long long> s_loc(B);
  {
    int po = 0; long long so = 0;
    for (int b = 0; b < B; b++) {
      ph_off[b] = po; po += 9 * T2[b];
      s_loc[b] = so; so += 600LL * T[b];
    }
  }
  int* d_ph_off = A.alloc<int>(B);
  long long* d_s_loc = A.alloc<long long>(B);
  long long* d_s24 = A.alloc<long long>(B);
  upload(d_ph_off, ph_off.data(), B * sizeof(int));
  upload(d_s_loc, s_loc.data(), B * sizeof(long long));
  upload(d_s24, s24_off_.data() + b0, B * sizeof(long long));
  // output resampling: the iSTFT writes each item into r.wav24 at its run-wide offset, so that a program is one
  // contiguous span there; once a program's last item is done (programs [k0, k1) here) the resampling pass reads
  // the span (p_in, p_len) and writes r.audio at the program's output-rate offset (p_out)
  const int K = k1 - k0;
  long long *d_p_in = nullptr, *d_p_len = nullptr, *d_p_out = nullptr;
  long long max_out = 0, max_len24 = 0;
  // loudness normalisation, the limiter and the loudness report: per-program 2400-sample segment energies (offsets
  // seg_off), true-peak, limiter and short-term energy scratch
  long long* d_seg_off = nullptr;
  float* energy = nullptr;
  double* short_e = nullptr;
  unsigned* peak = nullptr;
  unsigned* lim_acc = nullptr;
  if (resample_ && K > 0) {
    std::vector<long long> p_in(K), p_len(K), p_out(K), seg_off(K);
    long long nseg = 0;
    for (int k = 0; k < K; k++) {
      p_in[k] = s24_off_[prog_[k0 + k]];
      p_len[k] = s24_off_[prog_[k0 + k + 1]] - p_in[k];
      p_out[k] = sample_off_[k0 + k];
      max_out = std::max(max_out, sample_off_[k0 + k + 1] - p_out[k]);
      max_len24 = std::max(max_len24, p_len[k]);
      seg_off[k] = nseg;
      nseg += p_len[k] / kLoudSeg;
    }
    d_p_in = A.alloc<long long>(K);
    d_p_len = A.alloc<long long>(K);
    d_p_out = A.alloc<long long>(K);
    upload(d_p_in, p_in.data(), K * sizeof(long long));
    upload(d_p_len, p_len.data(), K * sizeof(long long));
    upload(d_p_out, p_out.data(), K * sizeof(long long));
    if (loud_ || lim_ || rep_) {
      d_seg_off = A.alloc<long long>(K);
      energy = A.alloc<float>((size_t)std::max(nseg, 1LL));
      peak = A.alloc<unsigned>(K);
      upload(d_seg_off, seg_off.data(), K * sizeof(long long));
    }
    if (lim_) lim_acc = A.alloc<unsigned>((size_t)2 * K);
    if (rep_) short_e = A.alloc<double>((size_t)std::max(nseg, 1LL));
  }

  // ---- length regulation (K4/K5)
  int* idx = A.alloc<int>(FR.rows);
  float* en = A.alloc<float>((size_t)FR.rows * 640);
  float* x514 = A.alloc<float>((size_t)FR.rows * 520);
  launch_expand_idx(cum, 512, tok_len, idx, FR.d_off, FR.d_len, B, FR.max_len, st);
  launch_gather_rows(r.d, 640, tok_off, idx, FR.d_off, FR.d_len, 640, en, 640, 0, B, FR.max_len, st);
  launch_gather_rows(r.t_en, 512, tok_off, idx, FR.d_off, FR.d_len, 512, x514, 520, 0, B, FR.max_len, st);
  if (debug_ && !dry) {
    // idx as float for the debug channel
    bool any = false;
    for (int b = 0; b < B; b++) any = any || want_debug(b0 + b);
    if (any) {
      KKX_CUDA(cudaStreamSynchronize(st));
      std::vector<int> hi(FR.rows);
      KKX_CUDA(cudaMemcpy(hi.data(), idx, FR.rows * sizeof(int), cudaMemcpyDeviceToHost));
      for (int b = 0; b < B; b++) {
        if (!want_debug(b0 + b)) continue;
        DebugStage s; s.rows = FR.len[b]; s.cols = 1; s.data.resize(FR.len[b]);
        for (int j = 0; j < FR.len[b]; j++) s.data[j] = (float)hi[FR.off[b] + j];
        dbg_["idx#" + std::to_string(b0 + b)] = std::move(s);
      }
    }
  }
  capture("en", en, 640, 0, 640, FR, b0);
  capture("asr", x514, 520, 0, 512, FR, b0);

  // ---- F0 / N predictor (A.7)
  float* xp = A.alloc<float>((size_t)FR.rows * 2048);
  float* shd = A.alloc<float>((size_t)FR.rows * 512);
  {
    const size_t cap = std::max((size_t)FR.rows * 640, (size_t)FR2.rows * 512);
    float* hi = A.alloc<float>(cap); float* lo = A.alloc<float>(cap);
    set_lane_scratch(0, hi, lo, cap);
    float* hi1 = A.alloc<float>(cap); float* lo1 = A.alloc<float>(cap);
    set_lane_scratch(1, hi1, lo1, cap);
  }
  gemm(FR, FR, en, 640, 640, W.shared_lstm.wih, &W.shared_lstm.t_ih, W.shared_lstm.bias, 2048, xp, 2048, 0);
  launch_lstm(xp, W.shared_lstm.whhT, shd, 512, 0, FR.d_off, FR.d_len, B, st, opt.precision != 0 && opt.lstm_fast_gates);
  capture("shared_lstm", shd, 512, 0, 512, FR, b0);
  float* curves[2];
  if (fork) fork_lane1();
  for (int k = 0; k < 2; k++) {
    const AdaBlkW* blk = k == 0 ? W.f0blk : W.nblk;
    if (fork) use_lane(k);                       // F0 stack on lane 0, N stack on lane 1
    float* y0 = A.alloc<float>((size_t)FR.rows * 512);
    float* y1 = A.alloc<float>((size_t)FR2.rows * 256);
    float* y2 = A.alloc<float>((size_t)FR2.rows * 256);
    adain_blk(A, blk[0], shd, 512, FR, FR, sty_pro, W.sty_pro_n, y0, 512, 0);
    adain_blk(A, blk[1], y0, 512, FR, FR2, sty_pro, W.sty_pro_n, y1, 256, 0);
    adain_blk(A, blk[2], y1, 256, FR2, FR2, sty_pro, W.sty_pro_n, y2, 256, 0);
    curves[k] = A.alloc<float>(FR2.rows);
    launch_conv_f32(gemm_args(FR2, y2, 256, 256, k == 0 ? W.f0proj_w : W.nproj_w,
                              k == 0 ? W.f0proj_b : W.nproj_b, 1, curves[k], 1, 0), cur_);
  }
  use_lane(0);
  if (fork) join_lane1();
  float* f0 = curves[0]; float* nc = curves[1];
  set_lane_scratch(0, nullptr, nullptr, 0);          // decoder / generator use the bf16 operand path
  set_lane_scratch(1, nullptr, nullptr, 0);
  if (!dry) {   // test hook: teacher-forced F0 / N curves of single items (any frame group)
    for (int k = 0; k < 2; k++) {
      for (auto& kv : (k == 0 ? inj_f0_ : inj_n_)) {
        const int b = kv.first - b0;
        if (kv.first >= B_) throw ArgError("inject F0/N: item index out of range");
        if (b < 0 || b >= B) continue;
        if ((int)kv.second.size() != FR2.len[b]) throw ArgError("inject F0/N: length != 2T of the item");
        upload((k == 0 ? f0 : nc) + FR2.off[b], kv.second.data(), kv.second.size() * sizeof(float));
      }
    }
  }
  capture("F0", f0, 1, 0, 1, FR2, b0);
  capture("N", nc, 1, 0, 1, FR2, b0);

  // ---- harmonic source, STFT and both noise res-blocks (A.9, K9/K10): they need only F0, so for small batches
  // they run on lane 1 beside the decoder (lane 0) and join before the first `x += x_source`
  if (fork) { fork_lane1(); use_lane(1); }
  float* phase = A.alloc<float>((size_t)9 * FR2.sum_len + 16);
  float* src = A.alloc<float>((size_t)600 * FR.sum_len + 16);
  float* har = A.alloc<float>((size_t)G120.rows * 24);
  launch_sine_phase(f0, FR2.d_off, FR2.d_len, phase, d_ph_off, B, st1);
  if (!dry && d_noise_) {
    for (int b = 0; b < B; b++)
      if (600LL * T[b] * 9 > noise_n_) throw ArgError("noise buffer smaller than 600*T*9");
  }
  launch_sine_source(f0, FR2.d_off, FR2.d_len, phase, d_ph_off, d_noise_, opt.noise_seed, W.lin_w,
                     W.lin_b, src, d_s_loc, B, maxS, st1);
  if (debug_ && !dry) {
    bool any = false;
    for (int b = 0; b < B; b++) any = any || want_debug(b0 + b);
    if (any) KKX_CUDA(cudaStreamSynchronize(st1));
    for (int b = 0; b < B; b++) {
      if (!want_debug(b0 + b)) continue;
      DebugStage s; s.rows = 600LL * T[b]; s.cols = 1; s.data.resize(s.rows);
      KKX_CUDA(cudaMemcpy(s.data.data(), src + s_loc[b], s.rows * sizeof(float), cudaMemcpyDeviceToHost));
      dbg_["har_source#" + std::to_string(b0 + b)] = std::move(s);
    }
  }
  launch_stft(src, d_s_loc, har, 24, G120.d_off, G120.d_len, opt.stft_replicate, B, G120.max_len, st1);
  capture("har", har, 24, 0, 22, G120, b0);

  // ---- generator stage 0 (20T rows, 256 ch)
  const size_t n20 = (size_t)G20.rows * 256, n120 = (size_t)G120.rows * 128;
  float* xs0 = A.alloc<float>(n20);
  float* x0 = A.alloc<float>(n20);
  float* w0 = A.alloc<float>(n20);
  float* t0 = A.alloc<float>(n20);
  float* acc0 = A.alloc<float>(n20);
  if (opt.precision == 1) {
    void* col = A.alloc_bytes((size_t)G20.rows * W.t_nc0.Cpad * 2);
    launch_im2col_bf16(har, 24, 22, 12, 6, 3, col, W.t_nc0.Cpad, G20.rows, G120.d_off, G120.d_len, G20.d_off,
                       G20.d_len, B, G20.max_len, st1);
    tc_conv(col, G20.rows, W.t_nc0, G20, G20, W.nc0_b, xs0, 256, 0, G20);
  } else {
    ConvArgs c = gemm_args(G20, har, 24, 22, W.nc0_w, W.nc0_b, 256, xs0, 256, 0);
    c.in_off = G120.d_off; c.in_len = G120.d_len;
    c.ks = 12; c.stride = 6; c.pad = 3;
    launch_conv_f32(c, st1);
  }
  arb(A, W.nres[0], xs0, G20, sty_dec, W.sty_dec_n, w0, t0, xs0, 1.f, false);
  capture("gen.x_source.0", xs0, 256, 0, 256, G20, b0);
  // (stage-1 buffers; the stage-1 noise branch is part of the same lane)
  float* xs1 = A.alloc<float>(n120);
  float* x1 = A.alloc<float>(n120);
  float* w1 = A.alloc<float>(n120);
  float* t1 = A.alloc<float>(n120);
  float* acc1 = A.alloc<float>(n120);
  float* pxs1 = nullptr;      // chunk statistics of xs1 when the conv below produced them
  if (opt.precision == 1 && opt.fuse_noise_stats && !use_stream_bf16(128, W.nres[1].k, B)) {
    // Conv1d(22, 128, k = 1) is a store stream (22 FMA per output): one fp32 pass that also emits the statistics the
    // first AdaIN of noise_res[1] needs, instead of bf16 plane + one-k-step implicit GEMM + colstats
    pxs1 = A.alloc<float>((size_t)B * ((G120.max_len + kStatRows - 1) / kStatRows) * 2 * 128);
    launch_pointwise_conv_stats(har, 24, 22, W.nc1_w, W.nc1_b, xs1, 128, pxs1, G120.d_off, G120.d_len, B, G120.max_len,
                                G120.sum_len, st1);
  } else if (opt.precision == 1) {
    void* hb = A.alloc_bytes((size_t)G120.rows * W.t_nc1.Cpad * 2);
    launch_apply_bf16(har, 24, 22, nullptr, nullptr, ACT_NONE, 0.f, nullptr, hb, W.t_nc1.Cpad, G120.rows, G120.d_off,
                      G120.d_len, B, G120.max_len, st1);
    tc_conv(hb, G120.rows, W.t_nc1, G120, G120, W.nc1_b, xs1, 128, 0, G120);
  } else {
    launch_conv_f32(gemm_args(G120, har, 24, 22, W.nc1_w, W.nc1_b, 128, xs1, 128, 0), st1);
  }
  arb(A, W.nres[1], xs1, G120, sty_dec, W.sty_dec_n, w1, t1, xs1, 1.f, false, pxs1);
  capture("gen.x_source.1", xs1, 128, 0, 128, G120, b0);
  use_lane(0);

  // ---- decoder (A.8)
  float* xA = A.alloc<float>((size_t)FR.rows * 1096);
  float* xB = A.alloc<float>((size_t)FR.rows * 1096);
  launch_curve_conv(f0, FR2.d_off, FR2.d_len, W.f0conv_w, W.f0conv_b, x514, 520, 512, FR.d_off, FR.d_len, B, FR.max_len, st);
  launch_curve_conv(nc, FR2.d_off, FR2.d_len, W.nconv_w, W.nconv_b, x514, 520, 513, FR.d_off, FR.d_len, B, FR.max_len, st);
  adain_blk(A, W.enc, x514, 520, FR, FR, sty_dec, W.sty_dec_n, xA, 1096, 0);
  capture("dec.encode", xA, 1096, 0, 1024, FR, b0);
  launch_conv_f32(gemm_args(FR, x514, 520, 512, W.asr_w, W.asr_b, 64, xA, 1096, 1024), st);
  launch_copy_cols(x514, 520, 512, xA, 1096, 1088, 2, FR.d_off, FR.d_len, B, FR.max_len, st);
  launch_copy_cols(xA, 1096, 1024, xB, 1096, 1024, 66, FR.d_off, FR.d_len, B, FR.max_len, st);
  float* dcur = xA; float* dnxt = xB;
  for (int i = 0; i < 3; i++) {
    adain_blk(A, W.dec[i], dcur, 1096, FR, FR, sty_dec, W.sty_dec_n, dnxt, 1096, 0);
    std::swap(dcur, dnxt);
    capture(("dec.decode." + std::to_string(i)).c_str(), dcur, 1096, 0, 1024, FR, b0);
  }
  float* y = A.alloc<float>((size_t)FR2.rows * 512);
  adain_blk(A, W.dec[3], dcur, 1096, FR, FR2, sty_dec, W.sty_dec_n, y, 512, 0);
  capture("dec.decode.3", y, 512, 0, 512, FR2, b0);

  // ---- generator stage 0: ConvTranspose1d(512, 256, k20, s10, p5), res-blocks
  upsample(A, y, FR2, x0, G20, 10, 0, W.tups0_all, W.tups0, W.ups0, W.ups0_b, dry);
  if (fork) join_lane1();
  capture("gen.ups.0", x0, 256, 0, 256, G20, b0);
  res_stage(A, W.res, x0, xs0, G20, sty_dec, w0, t0, acc0);
  capture("gen.stage.0", acc0, 256, 0, 256, G20, b0);

  // ---- generator stage 1 (120T+1 rows, 128 ch): ConvTranspose1d(256, 128, k12, s6, p3) + ReflectionPad1d((1, 0)),
  // res-blocks
  upsample(A, acc0, G20, x1, G120, 6, 1, W.tups1_all, W.tups1, W.ups1, W.ups1_b, dry);
  launch_copy_row(x1, 128, 0, 2, G120.d_off, B, st);
  capture("gen.ups.1", x1, 128, 0, 128, G120, b0);
  res_stage(A, W.res + 3, x1, xs1, G120, sty_dec, w1, t1, acc1);
  capture("gen.stage.1", acc1, 128, 0, 128, G120, b0);

  // ---- head (K11)
  float* cp = A.alloc<float>((size_t)G120.rows * 24);
  if (opt.precision == 1) {
    // fused: LeakyReLU in the operand producer, all 7 taps from one activation tile (kernels_arb.cu, POST)
    ArbConvArgs pc;
    pc.C = 128; pc.ks = 7; pc.dil = 1; pc.pad = 3; pc.off = G120.d_off; pc.len = G120.d_len; pc.B = B;
    pc.sum_m = G120.sum_len; pc.tile_start = G120.d_tiles256; pc.total_tiles = G120.ntiles256;
    pc.x = acc1; pc.in_bf16 = 0; pc.tmB = W.t_post_arb.tmap; pc.bias = W.post_b128;
    pc.out_f32 = cp; pc.post = 1; pc.cout = 22; pc.ldo = 24; pc.slope = 0.01f;
    launch_arb_conv(pc, st);
  } else {
    ConvArgs c = gemm_args(G120, acc1, 128, 128, W.post_w, W.post_b, 22, cp, 24, 0);
    c.ks = 7; c.pad = 3; c.pact = ACT_LRELU; c.pslope = 0.01f;
    launch_conv_f32(c, st);
  }
  capture("conv_post", cp, 24, 0, 22, G120, b0);
  const bool law = enc_ == Encoding::ULAW || enc_ == Encoding::ALAW;
  short* pcm = enc_ == Encoding::PCM16 || is_stream(enc_) ? static_cast<short*>(r.twin) : nullptr;
  if (!resample_) {   // the output is the 24 kHz waveform: program layout == item layout
    launch_istft(cp, 24, G120.d_off, G120.d_len, r.audio, pcm, d_s24, opt.precision == 1, B, G120.max_len, st);
    return;
  }
  launch_istft(cp, 24, G120.d_off, G120.d_len, r.wav24, nullptr, d_s24, opt.precision == 1, B, G120.max_len, st);
  if (K == 0) return;   // every program of this group goes on into the next
  const int P = n_prog();
  float* gain = nullptr;
  const float* wav = r.wav24;
  // measured on the 24 kHz waveform; the gain rides on the resampling pass (r.loud = lufs | dBTP | gain)
  if (loud_ || lim_ || rep_) {
    gain = r.loud + 2 * (size_t)P + k0;
    launch_loudness(r.wav24, d_p_in, d_p_len, d_seg_off, loud_par_, energy, peak, r.loud + k0, r.loud + P + k0, gain,
                    K, max_len24, st, lim_ ? r.lim_p : nullptr);
  }
  if (rep_) {   // the report on the same energies, before the limiter (r.rng = LRA | max momentary | max short-term)
    launch_loudness_range(d_p_len, d_seg_off, energy, short_e, r.rng + k0, r.rng + P + k0, r.rng + 2 * (size_t)P + k0,
                          K, max_len24, st);
    if (!loud_ && !lim_) gain = nullptr;   // measure-only: the resampling pass is the plain output's arithmetic
  }
  if (lim_) {   // the limited waveform v is resampled instead, with the static trim t as its gain (r.lim = t | report)
    launch_limiter(r.wav24, r.lim_p, d_p_in, d_p_len, loud_par_, gain, r.lim_v, nullptr, lim_acc, r.lim + k0,
                   r.lim + P + k0, r.lim + 2 * (size_t)P + k0, K, max_len24, st);
    wav = r.lim_v;
    gain = r.lim + k0;
  }
  // grids span the longest program (64-bit sample indices); CTAs past a shorter program's end return at once
  launch_resample(wav, d_p_in, d_p_len, d_p_out, d_taps_, rs_U_, rs_D_, rs_H_, gain, r.audio, pcm,
                  law ? static_cast<unsigned char*>(r.twin) : nullptr, enc_ == Encoding::ALAW ? 1 : 0, K, max_out, st);
}

}  // namespace kkx
