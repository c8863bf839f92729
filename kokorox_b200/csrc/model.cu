// model.cu -- Kokoro-82M forward pass on one B200: weight preparation + kernel orchestration.
// Replaces `sess.run` of /root/reference/kokorox/src/onn/ort_koko.rs:79 (the ONNX graph
// kokoro-v1.0.onnx); the architecture follows SURVEY.md Appendix A (A.1 - A.10).
#include "model.h"
#include <algorithm>
#include <cmath>
#include <cstring>
#include <fstream>
#include <stdlib.h>
#include <sys/stat.h>

namespace kkx {

thread_local bool g_dry_run = false;

// ============================================================================ weight file
namespace {
// a + b with overflow detection (extents come from a file)
bool add_ok(size_t a, size_t b, size_t* out) { *out = a + b; return *out >= a; }
}  // namespace

WeightFile::WeightFile(const std::string& path) {
  std::ifstream f(path, std::ios::binary | std::ios::ate);
  if (!f) throw IoError("cannot open weight file: " + path);
  const std::streamsize sz = f.tellg();
  if (sz < 16) throw IoError(path + ": not a model file (shorter than 16 bytes)");
  f.seekg(0);
  buf_.resize((size_t)sz);
  if (!f.read(buf_.data(), sz)) throw IoError("short read: " + path);
  if (memcmp(buf_.data(), "KKXW0001", 8) == 0) {
    format_ = "kkxw";
    load_kkxw(path);
    return;
  }
  // anything else must be an ONNX ModelProto -- the file OrtKoko::new is given (ort_base.rs:27-33)
  format_ = "onnx";
  load_onnx_weights(path, buf_, *this);
  std::vector<char>().swap(buf_);   // every tensor was converted into owned_ storage
}

void WeightFile::load_kkxw(const std::string& path) {
  const size_t sz = buf_.size();
  uint32_t n, hb;
  memcpy(&n, buf_.data() + 8, 4);
  memcpy(&hb, buf_.data() + 12, 4);
  size_t p = 16;
  auto need = [&](size_t k) { if (k > sz || p > sz - k) throw IoError(path + ": truncated header"); };
  for (uint32_t i = 0; i < n; i++) {
    need(2);
    uint16_t ln; memcpy(&ln, buf_.data() + p, 2); p += 2;
    need(ln);
    std::string name(buf_.data() + p, ln); p += ln;
    need(8);
    uint32_t dtype, ndim; memcpy(&dtype, buf_.data() + p, 4); memcpy(&ndim, buf_.data() + p + 4, 4); p += 8;
    if (dtype != 0 || ndim > 8) throw IoError(name + ": unsupported dtype/rank");
    HostTensor t;
    need(4 * (size_t)ndim + 16);
    size_t numel = 1;
    for (uint32_t d = 0; d < ndim; d++) {
      uint32_t v; memcpy(&v, buf_.data() + p, 4); p += 4;
      if (v > 0x7fffffffu || (v != 0 && numel > (size_t(1) << 40) / v)) throw IoError(name + ": bad dims");
      t.shape.push_back((int)v); numel *= v;
    }
    uint64_t off, nb; memcpy(&off, buf_.data() + p, 8); memcpy(&nb, buf_.data() + p + 8, 8); p += 16;
    // overflow-checked extent: hb + off + nb <= sz, 4-byte aligned payload
    size_t start, end;
    if (nb != (uint64_t)numel * 4 || off > sz || nb > sz || !add_ok((size_t)hb, (size_t)off, &start) ||
        !add_ok(start, (size_t)nb, &end) || end > sz || (start & 3) != 0)
      throw IoError(name + ": bad extent");
    t.data = reinterpret_cast<const float*>(buf_.data() + start);
    t.numel = numel;
    t_[name] = t;
  }
}

void WeightFile::put(const std::string& name, const std::vector<int>& shape, std::vector<float>&& data) {
  size_t numel = 1;
  for (int d : shape) numel *= (size_t)d;
  if (numel != data.size()) throw IoError(name + ": shape does not match the element count");
  owned_.push_back(std::move(data));
  HostTensor t;
  t.shape = shape; t.data = owned_.back().data(); t.numel = numel;
  t_[name] = t;
}

std::vector<std::string> WeightFile::names() const {
  std::vector<std::string> v;
  for (auto& kv : t_) v.push_back(kv.first);
  return v;
}

const HostTensor& WeightFile::get(const std::string& name) const {
  auto it = t_.find(name);
  if (it == t_.end()) throw IoError("weight tensor missing: " + name);
  return it->second;
}

// ============================================================================ construction
namespace {
int check_device(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    throw CudaError("no CUDA device available (this backend has no CPU fallback)");
  if (device < 0 || device >= ndev) throw CudaError("device ordinal out of range");
  KKX_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  KKX_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    char b[160];
    snprintf(b, sizeof b, "device %d is sm_%d%d; this library is built for sm_100a only", device,
             prop.major, prop.minor);
    throw CudaError(b);
  }
  return device;
}
std::mutex g_ws_mu;
std::map<std::string, std::weak_ptr<const WeightSet>> g_ws_cache;
}  // namespace

std::shared_ptr<const WeightSet> WeightSet::acquire(const std::string& path, int device) {
  // key: canonical path + size + mtime + device, so a replaced file is re-read
  std::string key = path;
  if (char* rp = realpath(path.c_str(), nullptr)) { key = rp; free(rp); }
  struct stat stt;
  if (stat(path.c_str(), &stt) != 0) throw IoError("cannot open weight file: " + path);
  key += "|" + std::to_string((long long)stt.st_size) + "|" + std::to_string((long long)stt.st_mtime) + "." +
         std::to_string((long long)stt.st_mtim.tv_nsec) + "|" + std::to_string(device);
  std::lock_guard<std::mutex> lk(g_ws_mu);   // held across the load: a second session of the same file waits and shares
  auto it = g_ws_cache.find(key);
  if (it != g_ws_cache.end())
    if (auto sp = it->second.lock()) return sp;
  KKX_CUDA(cudaSetDevice(device));
  std::shared_ptr<WeightSet> ws(new WeightSet());
  ws->device = device;
  WeightFile wf(path);
  ws->format = wf.format();
  ws->load(wf);
  g_ws_cache[key] = ws;
  for (auto i = g_ws_cache.begin(); i != g_ws_cache.end();)   // drop entries whose sets are gone
    i = i->second.expired() ? g_ws_cache.erase(i) : std::next(i);
  return ws;
}

WeightSet::~WeightSet() {
  cudaSetDevice(device);
  for (void* p : owned_) cudaFree(p);
}

Model::Model(const std::string& weights_path, int device)
    : device_(check_device(device)), ws_(WeightSet::acquire(weights_path, device_)), W(ws_->W) {
  KKX_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  KKX_CUDA(cudaStreamCreateWithFlags(&stream2_, cudaStreamNonBlocking));
  KKX_CUDA(cudaEventCreateWithFlags(&ev_fork_, cudaEventDisableTiming));
  KKX_CUDA(cudaEventCreateWithFlags(&ev_join_, cudaEventDisableTiming));
  cur_ = stream_;
  KKX_CUDA(cudaEventCreate(&ev0_));
  KKX_CUDA(cudaEventCreate(&ev1_));
  KKX_CUDA(cudaStreamCreateWithFlags(&copy_stream_, cudaStreamNonBlocking));
  KKX_CUDA(cudaEventCreateWithFlags(&ev_grp_, cudaEventDisableTiming));
  pin_.reserve(size_t(4) << 20);
  graph_pin_.reserve(size_t(1) << 20);
  const char* dbg = getenv("KKX_DEBUG_SYNC");
  stats.check_each = dbg && dbg[0] == '1';
  const char* det = getenv("KKX_PROFILE_DETAIL");
  stats.detail = det && det[0] == '1';
}

Model::~Model() {
  cudaSetDevice(device_);
  if (stream_) cudaStreamSynchronize(stream_);
  if (stream2_) cudaStreamSynchronize(stream2_);
  clear_graphs();
  if (d_taps_) cudaFree(d_taps_);
  if (d_voices_) cudaFree(d_voices_);
  if (d_noise_) cudaFree(d_noise_);
  if (h_pred_dur_) cudaFreeHost(h_pred_dur_);
  if (h_T_) cudaFreeHost(h_T_);
  if (ev0_) cudaEventDestroy(ev0_);
  if (ev1_) cudaEventDestroy(ev1_);
  if (copy_stream_) cudaStreamDestroy(copy_stream_);
  if (ev_grp_) cudaEventDestroy(ev_grp_);
  if (ev_fork_) cudaEventDestroy(ev_fork_);
  if (ev_join_) cudaEventDestroy(ev_join_);
  if (stream2_) cudaStreamDestroy(stream2_);
  if (stream_) cudaStreamDestroy(stream_);
}

void Model::clear_graphs() {
  for (auto& kv : graphs_)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  graphs_.clear();
  graph_pin_.reset();
}

void Model::fork_lane1() {
  KKX_CUDA(cudaEventRecord(ev_fork_, stream_));
  KKX_CUDA(cudaStreamWaitEvent(stream2_, ev_fork_, 0));
}

void Model::join_lane1() {
  KKX_CUDA(cudaEventRecord(ev_join_, stream2_));
  KKX_CUDA(cudaStreamWaitEvent(stream_, ev_join_, 0));
}

float* WeightSet::up(const std::vector<float>& v) {
  float* d = nullptr;
  const size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(float);
  KKX_CUDA(cudaMalloc(&d, bytes));
  owned_.push_back(d);
  device_bytes += bytes;
  KKX_CUDA(cudaMemcpy(d, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return d;
}

namespace {
std::vector<float> raw(const WeightFile& wf, const std::string& n) {
  const HostTensor& t = wf.get(n);
  return std::vector<float>(t.data, t.data + t.numel);
}
void expect(const HostTensor& t, std::initializer_list<int> shp, const std::string& n) {
  if (t.shape != std::vector<int>(shp)) throw IoError("unexpected shape for " + n);
}
// torch Linear [N][K] -> [K][N]
std::vector<float> linT(const WeightFile& wf, const std::string& n, int N, int K) {
  const HostTensor& t = wf.get(n);
  if ((int)t.numel != N * K) throw IoError("unexpected size for " + n);
  std::vector<float> o((size_t)N * K);
  for (int i = 0; i < N; i++)
    for (int k = 0; k < K; k++) o[(size_t)k * N + i] = t.data[(size_t)i * K + k];
  return o;
}
// Conv1d [Co][Ci][k] -> [k][Ci][Co]
std::vector<float> convW(const WeightFile& wf, const std::string& n, int Co, int Ci, int k) {
  const HostTensor& t = wf.get(n);
  expect(t, {Co, Ci, k}, n);
  std::vector<float> o((size_t)Co * Ci * k);
  for (int oc = 0; oc < Co; oc++)
    for (int c = 0; c < Ci; c++)
      for (int tt = 0; tt < k; tt++)
        o[((size_t)tt * Ci + c) * Co + oc] = t.data[((size_t)oc * Ci + c) * k + tt];
  return o;
}
// Conv1d [Co][Ci][k] -> [Co][k][Ci] (tensor-core weight layout before padding / bf16 rounding)
std::vector<float> convCoKsCi(const WeightFile& wf, const std::string& n, int Co, int Ci, int k) {
  const HostTensor& t = wf.get(n);
  expect(t, {Co, Ci, k}, n);
  std::vector<float> o((size_t)Co * Ci * k);
  for (int oc = 0; oc < Co; oc++)
    for (int c = 0; c < Ci; c++)
      for (int tt = 0; tt < k; tt++)
        o[((size_t)oc * k + tt) * Ci + c] = t.data[((size_t)oc * Ci + c) * k + tt];
  return o;
}
uint16_t f2bf(float f) {  // round-to-nearest-even fp32 -> bf16
  uint32_t u;
  memcpy(&u, &f, 4);
  const uint32_t r = u + 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(r >> 16);
}
}  // namespace

TcW WeightSet::make_tc(const std::vector<float>& w, int Co, int ks, int Ci) {
  TcW t;
  t.Ci = Ci; t.Co = Co; t.ks = ks; t.Cpad = (Ci + 63) & ~63;
  std::vector<uint16_t> h((size_t)Co * ks * t.Cpad, 0);
  for (int o = 0; o < Co; o++)
    for (int k = 0; k < ks; k++)
      for (int c = 0; c < Ci; c++)
        h[((size_t)o * ks + k) * t.Cpad + c] = f2bf(w[((size_t)o * ks + k) * Ci + c]);
  KKX_CUDA(cudaMalloc(&t.w, h.size() * 2));
  owned_.push_back(t.w);
  device_bytes += h.size() * 2;
  KKX_CUDA(cudaMemcpy(t.w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  make_tmap_bf16(t.tmap, t.w, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, tc_box_n(Co));
  if (Co >= 128 && Co % 128 == 0) {
    make_tmap_bf16(t.tmap_h, t.w, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, 128);
    t.has_h = true;
  }
  return t;
}

namespace {
float host_tf32(float f) {  // cvt.rna.tf32.f32
  uint32_t u;
  memcpy(&u, &f, 4);
  u = (u + 0x1000u) & ~0x1FFFu;
  float r;
  memcpy(&r, &u, 4);
  return r;
}
std::vector<float> concat(std::initializer_list<const HostTensor*> ts) {
  std::vector<float> o;
  for (auto t : ts) o.insert(o.end(), t->data, t->data + t->numel);
  return o;
}
}  // namespace

TcW32 WeightSet::make_tc32(const std::vector<float>& w, int Co, int ks, int Ci) {
  TcW32 t;
  t.Ci = Ci; t.Co = Co; t.ks = ks; t.Cpad = (Ci + 63) & ~63;
  std::vector<float> hi((size_t)Co * ks * t.Cpad, 0.f), lo((size_t)Co * ks * t.Cpad, 0.f);
  for (int o = 0; o < Co; o++)
    for (int k = 0; k < ks; k++)
      for (int c = 0; c < Ci; c++) {
        const float f = w[((size_t)o * ks + k) * Ci + c];
        const float h = host_tf32(f);
        hi[((size_t)o * ks + k) * t.Cpad + c] = h;
        lo[((size_t)o * ks + k) * t.Cpad + c] = host_tf32(f - h);
      }
  t.hi = up(hi); t.lo = up(lo);
  make_tmap_f32(t.tm_hi, t.hi, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, tc_box_n_tf32(Co));
  make_tmap_f32(t.tm_lo, t.lo, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, tc_box_n_tf32(Co));
  if (tc_box_n_tf32(Co) == 128) {
    make_tmap_f32(t.tm_hi_c, t.hi, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, 64);
    make_tmap_f32(t.tm_lo_c, t.lo, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, 64);
    t.has_c = true;
  }
  // split-FP16 planes of the same (zero-padded) matrix
  {
    std::vector<float> wp((size_t)Co * ks * t.Cpad, 0.f);
    for (int o = 0; o < Co; o++)
      for (int k = 0; k < ks; k++)
        for (int c = 0; c < Ci; c++) wp[((size_t)o * ks + k) * t.Cpad + c] = w[((size_t)o * ks + k) * Ci + c];
    std::vector<unsigned short> h16(wp.size()), l16(wp.size());
    t.wscale16 = split_f16_host(wp.data(), wp.size(), h16.data(), l16.data());
    KKX_CUDA(cudaMalloc(&t.h_hi, h16.size() * 2)); owned_.push_back(t.h_hi);
    KKX_CUDA(cudaMalloc(&t.h_lo, l16.size() * 2)); owned_.push_back(t.h_lo);
    device_bytes += h16.size() * 4;
    KKX_CUDA(cudaMemcpy(t.h_hi, h16.data(), h16.size() * 2, cudaMemcpyHostToDevice));
    KKX_CUDA(cudaMemcpy(t.h_lo, l16.data(), l16.size() * 2, cudaMemcpyHostToDevice));
    make_tmap_f16(t.tm16_hi, t.h_hi, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, tc_box_n_tf32(Co));
    make_tmap_f16(t.tm16_lo, t.h_lo, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, tc_box_n_tf32(Co));
    if (t.has_c) {
      make_tmap_f16(t.tm16_hi_c, t.h_hi, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, 64);
      make_tmap_f16(t.tm16_lo_c, t.h_lo, (long long)ks * t.Cpad, Co, (long long)ks * t.Cpad, 64);
    }
  }
  return t;
}

void WeightSet::load(const WeightFile& wf) {
  auto U = [&](const std::string& n) { return up(raw(wf, n)); };
  auto LT = [&](const std::string& n, int N, int K) { return up(linT(wf, n, N, K)); };
  auto CW = [&](const std::string& n, int Co, int Ci, int k) { return up(convW(wf, n, Co, Ci, k)); };

  // ---- ALBERT (A.2)
  const std::string E = "bert.embeddings.", L = "bert.encoder.albert_layer_groups.0.albert_layers.0.";
  W.word = U(E + "word_embeddings.weight");
  W.pos = U(E + "position_embeddings.weight");
  W.type = U(E + "token_type_embeddings.weight");
  W.emb_lnw = U(E + "LayerNorm.weight"); W.emb_lnb = U(E + "LayerNorm.bias");
  W.map_w = LT("bert.encoder.embedding_hidden_mapping_in.weight", 768, 128);
  W.map_b = U("bert.encoder.embedding_hidden_mapping_in.bias");
  {
    std::vector<float> qkv((size_t)768 * 2304), qb(2304);
    const char* nm[3] = {"query", "key", "value"};
    for (int j = 0; j < 3; j++) {
      const HostTensor& t = wf.get(L + "attention." + nm[j] + ".weight");
      const HostTensor& bb = wf.get(L + "attention." + nm[j] + ".bias");
      expect(t, {768, 768}, nm[j]);
      for (int n = 0; n < 768; n++) {
        qb[j * 768 + n] = bb.data[n];
        for (int k = 0; k < 768; k++) qkv[(size_t)k * 2304 + j * 768 + n] = t.data[(size_t)n * 768 + k];
      }
    }
    W.qkv_w = up(qkv); W.qkv_b = up(qb);
  }
  W.dense_w = LT(L + "attention.dense.weight", 768, 768); W.dense_b = U(L + "attention.dense.bias");
  W.attn_lnw = U(L + "attention.LayerNorm.weight"); W.attn_lnb = U(L + "attention.LayerNorm.bias");
  W.ffn_w = LT(L + "ffn.weight", 2048, 768); W.ffn_b = U(L + "ffn.bias");
  W.ffo_w = LT(L + "ffn_output.weight", 768, 2048); W.ffo_b = U(L + "ffn_output.bias");
  W.full_lnw = U(L + "full_layer_layer_norm.weight"); W.full_lnb = U(L + "full_layer_layer_norm.bias");
  W.benc_w = LT("bert_encoder.weight", 512, 768); W.benc_b = U("bert_encoder.bias");
  // split-TF32 copies (torch Linear [N][K] is already [Co][1][Ci])
  W.t_map = make_tc32(raw(wf, "bert.encoder.embedding_hidden_mapping_in.weight"), 768, 1, 128);
  W.t_qkv = make_tc32(concat({&wf.get(L + "attention.query.weight"), &wf.get(L + "attention.key.weight"),
                              &wf.get(L + "attention.value.weight")}), 2304, 1, 768);
  W.t_dense = make_tc32(raw(wf, L + "attention.dense.weight"), 768, 1, 768);
  W.t_ffn = make_tc32(raw(wf, L + "ffn.weight"), 2048, 1, 768);
  W.t_ffo = make_tc32(raw(wf, L + "ffn_output.weight"), 768, 1, 2048);
  W.t_benc = make_tc32(raw(wf, "bert_encoder.weight"), 512, 1, 768);

  // ---- LSTMs (A.11 gate order i,f,g,o)
  auto LSTM = [&](const std::string& p, int in) {
    LstmW l; l.in = in;
    std::vector<float> wih((size_t)in * 2048), bias(2048), whh((size_t)2 * 256 * 1024);
    const char* sfx[2] = {"", "_reverse"};
    for (int d = 0; d < 2; d++) {
      const HostTensor& a = wf.get(p + ".weight_ih_l0" + sfx[d]);
      const HostTensor& h = wf.get(p + ".weight_hh_l0" + sfx[d]);
      const HostTensor& bi = wf.get(p + ".bias_ih_l0" + sfx[d]);
      const HostTensor& bh = wf.get(p + ".bias_hh_l0" + sfx[d]);
      expect(a, {1024, in}, p); expect(h, {1024, 256}, p);
      for (int g = 0; g < 1024; g++) {
        bias[d * 1024 + g] = bi.data[g] + bh.data[g];
        for (int k = 0; k < in; k++) wih[(size_t)k * 2048 + d * 1024 + g] = a.data[(size_t)g * in + k];
        for (int k = 0; k < 256; k++) whh[((size_t)d * 256 + k) * 1024 + g] = h.data[(size_t)g * 256 + k];
      }
    }
    l.wih = up(wih); l.bias = up(bias); l.whhT = up(whh);
    l.t_ih = make_tc32(concat({&wf.get(p + ".weight_ih_l0"), &wf.get(p + ".weight_ih_l0_reverse")}), 2048, 1, in);
    return l;
  };

  // ---- style FC tables
  std::vector<float> pro_w, pro_b, dec_w, dec_b;
  std::vector<std::pair<std::string, int>> pro_list, dec_list;  // (fc prefix, outputs)
  auto add_sty = [&](std::vector<std::pair<std::string, int>>& lst, int& total, const std::string& fc, int nout) {
    const int off = total;
    lst.push_back({fc, nout});
    total += nout;
    return off;
  };
  int npro = 0, ndec = 0;

  for (int i = 0; i < 3; i++) {
    W.dur_lstm[i] = LSTM("predictor.text_encoder.lstms." + std::to_string(2 * i), 640);
    W.dur_ada[i] = add_sty(pro_list, npro, "predictor.text_encoder.lstms." + std::to_string(2 * i + 1) + ".fc", 1024);
  }
  W.pred_lstm = LSTM("predictor.lstm", 640);
  W.shared_lstm = LSTM("predictor.shared", 640);
  W.te_lstm = LSTM("text_encoder.lstm", 512);
  W.durp_w = LT("predictor.duration_proj.linear_layer.weight", 50, 512);
  W.durp_b = U("predictor.duration_proj.linear_layer.bias");
  W.t_durp = make_tc32(raw(wf, "predictor.duration_proj.linear_layer.weight"), 50, 1, 512);

  auto BLK = [&](const std::string& p, int ci, int co, bool upf, bool pro) {
    AdaBlkW b; b.ci = ci; b.co = co; b.up = upf;
    b.w1 = CW(p + ".conv1.weight", co, ci, 3); b.b1 = U(p + ".conv1.bias");
    b.w2 = CW(p + ".conv2.weight", co, co, 3); b.b2 = U(p + ".conv2.bias");
    if (ci != co) b.w1x1 = CW(p + ".conv1x1.weight", co, ci, 1);
    if (upf) { b.poolw = U(p + ".pool.weight"); b.poolb = U(p + ".pool.bias"); }
    if (pro) {   // F0/N predictor blocks: split-TF32 (fp32-grade) tensor-core weights
      b.s1 = make_tc32(convCoKsCi(wf, p + ".conv1.weight", co, ci, 3), co, 3, ci);
      b.s2 = make_tc32(convCoKsCi(wf, p + ".conv2.weight", co, co, 3), co, 3, co);
      if (ci != co) b.s1x1 = make_tc32(convCoKsCi(wf, p + ".conv1x1.weight", co, ci, 1), co, 1, ci);
    }
    if (!pro) {  // decoder blocks: bf16 tensor-core weights
      b.t1 = make_tc(convCoKsCi(wf, p + ".conv1.weight", co, ci, 3), co, 3, ci);
      b.t2 = make_tc(convCoKsCi(wf, p + ".conv2.weight", co, co, 3), co, 3, co);
      if (ci != co) b.t1x1 = make_tc(convCoKsCi(wf, p + ".conv1x1.weight", co, ci, 1), co, 1, ci);
    }
    auto& lst = pro ? pro_list : dec_list; int& tot = pro ? npro : ndec;
    b.sty1 = add_sty(lst, tot, p + ".norm1.fc", 2 * ci);
    b.sty2 = add_sty(lst, tot, p + ".norm2.fc", 2 * co);
    return b;
  };
  const char* br[2] = {"F0", "N"};
  for (int k = 0; k < 2; k++) {
    AdaBlkW* dst = k == 0 ? W.f0blk : W.nblk;
    const std::string p = std::string("predictor.") + br[k];
    dst[0] = BLK(p + ".0", 512, 512, false, true);
    dst[1] = BLK(p + ".1", 512, 256, true, true);
    dst[2] = BLK(p + ".2", 256, 256, false, true);
  }
  W.f0proj_w = LT("predictor.F0_proj.weight", 1, 256); W.f0proj_b = U("predictor.F0_proj.bias");
  W.nproj_w = LT("predictor.N_proj.weight", 1, 256); W.nproj_b = U("predictor.N_proj.bias");

  // ---- text encoder (A.4)
  W.temb = U("text_encoder.embedding.weight");
  for (int i = 0; i < 3; i++) {
    const std::string p = "text_encoder.cnn." + std::to_string(i);
    W.tcnn_w[i] = CW(p + ".0.weight", 512, 512, 5); W.tcnn_b[i] = U(p + ".0.bias");
    W.t_tcnn[i] = make_tc32(convCoKsCi(wf, p + ".0.weight", 512, 512, 5), 512, 5, 512);
    W.tln_g[i] = U(p + ".1.gamma"); W.tln_b[i] = U(p + ".1.beta");
  }

  // ---- decoder (A.8)
  W.enc = BLK("decoder.encode", 514, 1024, false, false);
  for (int i = 0; i < 3; i++) W.dec[i] = BLK("decoder.decode." + std::to_string(i), 1090, 1024, false, false);
  W.dec[3] = BLK("decoder.decode.3", 1090, 512, true, false);
  W.f0conv_w = U("decoder.F0_conv.weight"); W.f0conv_b = U("decoder.F0_conv.bias");
  W.nconv_w = U("decoder.N_conv.weight"); W.nconv_b = U("decoder.N_conv.bias");
  W.asr_w = CW("decoder.asr_res.0.weight", 64, 512, 1); W.asr_b = U("decoder.asr_res.0.bias");

  // ---- generator (A.9)
  const std::string G = "decoder.generator.";
  W.lin_w = U(G + "m_source.l_linear.weight"); W.lin_b = U(G + "m_source.l_linear.bias");
  W.nc0_w = CW(G + "noise_convs.0.weight", 256, 22, 12); W.nc0_b = U(G + "noise_convs.0.bias");
  W.nc1_w = CW(G + "noise_convs.1.weight", 128, 22, 1); W.nc1_b = U(G + "noise_convs.1.bias");
  auto ARB = [&](const std::string& p, int c, int k) {
    ArbW a; a.c = c; a.k = k;
    for (int j = 0; j < 3; j++) {
      const std::string sj = std::to_string(j);
      a.w1[j] = CW(p + ".convs1." + sj + ".weight", c, c, k); a.b1[j] = U(p + ".convs1." + sj + ".bias");
      a.w2[j] = CW(p + ".convs2." + sj + ".weight", c, c, k); a.b2[j] = U(p + ".convs2." + sj + ".bias");
      a.a1[j] = U(p + ".alpha1." + sj); a.a2[j] = U(p + ".alpha2." + sj);
      a.t1[j] = make_tc(convCoKsCi(wf, p + ".convs1." + sj + ".weight", c, c, k), c, k, c);
      a.t2[j] = make_tc(convCoKsCi(wf, p + ".convs2." + sj + ".weight", c, c, k), c, k, c);
      a.s1[j] = add_sty(dec_list, ndec, p + ".adain1." + sj + ".fc", 2 * c);
      a.s2[j] = add_sty(dec_list, ndec, p + ".adain2." + sj + ".fc", 2 * c);
    }
    return a;
  };
  W.nres[0] = ARB(G + "noise_res.0", 256, 7);
  W.nres[1] = ARB(G + "noise_res.1", 128, 11);
  const int rk[3] = {3, 7, 11};
  for (int i = 0; i < 2; i++)
    for (int j = 0; j < 3; j++) W.res[i * 3 + j] = ARB(G + "resblocks." + std::to_string(i * 3 + j), i == 0 ? 256 : 128, rk[j]);
  auto UPS = [&](const std::string& n, int Ci, int Co, int k, int s, std::vector<float*>& out, std::vector<TcW>& tout,
                 TcW& tall) {
    const HostTensor& t = wf.get(n);
    expect(t, {Ci, Co, k}, n);
    {   // all phases stacked along the output-channel axis: row p*Co + o = phase p, channel o
      std::vector<float> tw((size_t)s * Co * 2 * Ci);
      for (int r = 0; r < s; r++)
        for (int o = 0; o < Co; o++)
          for (int j = 0; j < 2; j++)
            for (int c = 0; c < Ci; c++)
              tw[(((size_t)r * Co + o) * 2 + j) * Ci + c] = t.data[((size_t)c * Co + o) * k + r + j * s];
      tall = make_tc(tw, s * Co, 2, Ci);
      tall.Co = Co;                                                    // per-phase output channels
      make_tmap_bf16(tall.tmap, tall.w, (long long)2 * tall.Cpad, (long long)s * Co, (long long)2 * tall.Cpad, tc_box_n(Co));
    }
    for (int r = 0; r < s; r++) {
      std::vector<float> tw((size_t)Co * 2 * Ci);
      for (int o = 0; o < Co; o++)
        for (int j = 0; j < 2; j++)
          for (int c = 0; c < Ci; c++)
            tw[((size_t)o * 2 + j) * Ci + c] = t.data[((size_t)c * Co + o) * k + r + j * s];
      tout.push_back(make_tc(tw, Co, 2, Ci));
      std::vector<float> ph((size_t)2 * Ci * Co);
      for (int j = 0; j < 2; j++)
        for (int c = 0; c < Ci; c++)
          for (int o = 0; o < Co; o++)
            ph[((size_t)j * Ci + c) * Co + o] = t.data[((size_t)c * Co + o) * k + r + j * s];
      out.push_back(up(ph));
    }
  };
  UPS(G + "ups.0.weight", 512, 256, 20, 10, W.ups0, W.tups0, W.tups0_all); W.ups0_b = U(G + "ups.0.bias");
  UPS(G + "ups.1.weight", 256, 128, 12, 6, W.ups1, W.tups1, W.tups1_all); W.ups1_b = U(G + "ups.1.bias");
  W.post_w = CW(G + "conv_post.weight", 22, 128, 7); W.post_b = U(G + "conv_post.bias");
  {
    std::vector<float> wp = convCoKsCi(wf, G + "conv_post.weight", 22, 128, 7);
    wp.resize((size_t)128 * 7 * 128, 0.f);                 // rows 22..127 are zero
    W.t_post_arb = make_tc(wp, 128, 7, 128);
    std::vector<float> b128 = raw(wf, G + "conv_post.bias");
    b128.resize(128, 0.f);
    W.post_b128 = up(b128);
  }
  W.t_nc1 = make_tc(convCoKsCi(wf, G + "noise_convs.1.weight", 128, 22, 1), 128, 1, 22);
  // noise_convs[0] as a 1-tap GEMM over the im2col operand: K index = tap*22 + c
  W.t_nc0 = make_tc(convCoKsCi(wf, G + "noise_convs.0.weight", 256, 22, 12), 256, 1, 12 * 22);
  W.t_asr = make_tc(convCoKsCi(wf, "decoder.asr_res.0.weight", 64, 512, 1), 64, 1, 512);

  // ---- build the two style FC tables: W^T [128][n], bias [n]
  auto build = [&](const std::vector<std::pair<std::string, int>>& lst, int total, float*& dw, float*& db) {
    std::vector<float> w((size_t)128 * total), b(total);
    int off = 0;
    for (auto& e : lst) {
      const HostTensor& t = wf.get(e.first + ".weight");
      const HostTensor& bb = wf.get(e.first + ".bias");
      expect(t, {e.second, 128}, e.first);
      for (int o = 0; o < e.second; o++) {
        b[off + o] = bb.data[o];
        for (int k = 0; k < 128; k++) w[(size_t)k * total + off + o] = t.data[(size_t)o * 128 + k];
      }
      off += e.second;
    }
    dw = up(w); db = up(b);
  };
  build(pro_list, npro, W.sty_pro_w, W.sty_pro_b);
  build(dec_list, ndec, W.sty_dec_w, W.sty_dec_b);
  W.sty_pro_n = npro; W.sty_dec_n = ndec;
}

// ============================================================================ helpers
void Model::upload(void* dst, const void* src, size_t bytes) {
  if (bytes == 0 || g_dry_run) return;
  if (capturing_) {
    // the memcpy node keeps this staging address: it has to stay valid (and unchanged) for every replay
    void* stg = graph_pin_.alloc_bytes(bytes);
    if (!stg) throw CudaError("graph staging arena exhausted");
    memcpy(stg, src, bytes);
    KKX_CUDA(cudaMemcpyAsync(dst, stg, bytes, cudaMemcpyHostToDevice, cur_));
    return;
  }
  void* stg = pin_.alloc_bytes(bytes);
  if (!stg) {   // staging full: everything issued so far has to land before the arena can be reused
    KKX_CUDA(cudaStreamSynchronize(stream_));
    KKX_CUDA(cudaStreamSynchronize(stream2_));
    pin_.reset();
    pin_.reserve(std::max<size_t>(bytes * 2, size_t(4) << 20));
    stg = pin_.alloc_bytes(bytes);
    if (!stg) throw CudaError("pinned staging arena exhausted");
  }
  memcpy(stg, src, bytes);
  KKX_CUDA(cudaMemcpyAsync(dst, stg, bytes, cudaMemcpyHostToDevice, cur_));
}

Level Model::make_level(const std::vector<int>& lens, Arena& A, int first_off) {
  Level L;
  L.B = (int)lens.size();
  L.len = lens;
  L.off.resize(L.B);
  long long o = first_off;
  for (int b = 0; b < L.B; b++) {
    L.off[b] = (int)o;
    o = (o + lens[b] + kGapRows + 7) & ~7LL;
    if (o > 0x7fffff00LL) throw ArgError("batch too large: packed row offsets exceed int32");
    L.max_len = std::max(L.max_len, lens[b]);
    L.sum_len += lens[b];
  }
  L.rows = (int)o;
  // one device block, one upload: off[B] len[B] tiles128[B+1] tiles256[B+1]
  const size_t n = (size_t)4 * L.B + 2;
  int* d = A.alloc<int>(n);
  L.d_off = d; L.d_len = d + L.B;
  L.d_tiles128 = d + 2 * L.B; L.d_tiles256 = L.d_tiles128 + L.B + 1;
  std::vector<int> h(n, 0);
  int* t128 = h.data() + 2 * L.B; int* t256 = t128 + L.B + 1;
  for (int b = 0; b < L.B; b++) {
    h[b] = L.off[b]; h[L.B + b] = lens[b];
    t128[b + 1] = t128[b] + (lens[b] + 127) / 128;
    t256[b + 1] = t256[b] + (lens[b] + 255) / 256;
  }
  L.ntiles128 = t128[L.B]; L.ntiles256 = t256[L.B];
  upload(d, h.data(), n * sizeof(int));
  return L;
}

void Model::capture(const char* name, const float* p, int ld, int col, int cols, const Level& L,
                    int item0) {
  if (!debug_ || g_dry_run) return;
  bool any = false;
  for (int b = 0; b < L.B; b++) any = any || want_debug(item0 + b);
  if (!any) return;
  KKX_CUDA(cudaStreamSynchronize(stream_));
  for (int b = 0; b < L.B; b++) {
    if (!want_debug(item0 + b)) continue;
    DebugStage s;
    s.rows = L.len[b]; s.cols = cols;
    s.data.resize((size_t)s.rows * cols);
    if (s.rows > 0)
      KKX_CUDA(cudaMemcpy2D(s.data.data(), cols * sizeof(float), p + (size_t)L.off[b] * ld + col,
                            ld * sizeof(float), cols * sizeof(float), s.rows, cudaMemcpyDeviceToHost));
    dbg_[std::string(name) + "#" + std::to_string(item0 + b)] = std::move(s);
  }
}

const DebugStage* Model::debug_stage(const std::string& name, int item) const {
  auto it = dbg_.find(name + "#" + std::to_string(item));
  return it == dbg_.end() ? nullptr : &it->second;
}

void Model::set_noise(const float* noise, long long n) {
  KKX_CUDA(cudaSetDevice(device_));
  KKX_CUDA(cudaStreamSynchronize(stream_));
  if (d_noise_) { cudaFree(d_noise_); d_noise_ = nullptr; }
  noise_n_ = 0;
  if (noise && n > 0) {
    KKX_CUDA(cudaMalloc(&d_noise_, n * sizeof(float)));
    KKX_CUDA(cudaMemcpy(d_noise_, noise, n * sizeof(float), cudaMemcpyHostToDevice));
    noise_n_ = n;
  }
}

void Model::set_inject(const std::string& name, int item, const void* data, long long count) {
  if (item < 0) throw ArgError("inject: item index must be >= 0");
  const bool clear = !data || count <= 0;
  if (name == "pred_dur") {
    if (clear) { inj_dur_.erase(item); return; }
    const int* d = static_cast<const int*>(data);
    long long sum = 0;
    for (long long i = 0; i < count; i++) {
      if (d[i] < 1 || d[i] > 500) throw ArgError("inject pred_dur: every duration must be in 1..500");
      sum += d[i];
    }
    if (sum > kMaxItemFrames) throw ArgError("inject pred_dur: more than " + std::to_string(kMaxItemFrames) + " frames");
    inj_dur_[item].assign(d, d + count);
  } else if (name == "F0" || name == "N") {
    auto& m = name == "F0" ? inj_f0_ : inj_n_;
    if (clear) { m.erase(item); return; }
    m[item].assign(static_cast<const float*>(data), static_cast<const float*>(data) + count);
  } else {
    throw ArgError("unknown inject name: " + name);
  }
}


// ============================================================================ staging / IO
void Model::stage(int B, const int64_t* tokens, const int32_t* tok_offsets, const float* styles,
                  const float* speeds) {
  // ---- validate everything first: a rejected batch must leave the session exactly as it was (ADVICE r1)
  if (B <= 0) throw ArgError("batch must be >= 1");
  if (!tokens || !tok_offsets || !speeds) throw ArgError("null input pointer");   // styles == nullptr: filled by stage_voices
  if (tok_offsets[0] < 0) throw ArgError("tok_offsets[0] must be >= 0");
  std::vector<int> lens(B);
  for (int b = 0; b < B; b++) {
    const long long n = (long long)tok_offsets[b + 1] - tok_offsets[b];
    if (n < 1 || n > 512) throw ArgError("n_tokens must be in 1..512 (got " + std::to_string(n) + ")");
    if (!(speeds[b] >= kMinSpeed && speeds[b] <= kMaxSpeed))
      throw ArgError("speed must be in [0.1, 10] (got " + std::to_string(speeds[b]) + ")");
    lens[b] = (int)n;
    for (int t = 0; t < lens[b]; t++) {
      const int64_t id = tokens[tok_offsets[b] + t];
      if (id < 0 || id > 177) throw ArgError("token id out of range 0..177: " + std::to_string(id));
    }
  }
  // ---- commit
  KKX_CUDA(cudaSetDevice(device_));
  staged_ = false; ran_ = false; B_ = 0;
  use_lane(0);
  pin_.reset();                                  // the stream is idle here: run() drains it before returning
  ioA_.reserve((size_t)B * (560 * 4 + 1024 + 64) + (1 << 20));
  ioA_.reset();
  g_dry_run = false;
  tokL_ = make_level(lens, ioA_);
  std::vector<int> ids((size_t)tokL_.rows, 0);
  for (int b = 0; b < B; b++)
    for (int t = 0; t < lens[b]; t++) ids[tokL_.off[b] + t] = (int)tokens[tok_offsets[b] + t];
  d_ids_ = ioA_.alloc<int>(tokL_.rows);
  d_styles_ = ioA_.alloc<float>((size_t)B * 256);
  d_speeds_ = ioA_.alloc<float>(B);
  upload(d_ids_, ids.data(), ids.size() * sizeof(int));
  if (styles) upload(d_styles_, styles, (size_t)B * 256 * sizeof(float));
  upload(d_speeds_, speeds, B * sizeof(float));
  B_ = B;
  tok_len_ = lens;
  staged_ = true;
}

void Model::load_voices(const float* table, int n_voices) {
  if (!table || n_voices < 1) throw ArgError("load_voices: null table or n_voices < 1");
  KKX_CUDA(cudaSetDevice(device_));
  KKX_CUDA(cudaStreamSynchronize(stream_));
  if (d_voices_) { cudaFree(d_voices_); d_voices_ = nullptr; n_voices_ = 0; }
  const size_t bytes = (size_t)n_voices * 511 * 256 * sizeof(float);
  KKX_CUDA(cudaMalloc(&d_voices_, bytes));
  KKX_CUDA(cudaMemcpy(d_voices_, table, bytes, cudaMemcpyHostToDevice));
  n_voices_ = n_voices;
}

void Model::stage_voices(int B, const int64_t* tokens, const int32_t* tok_offsets, const int32_t* mix_offsets,
                         const int32_t* voice_ids, const float* portions, const int32_t* style_rows,
                         const float* speeds) {
  if (!d_voices_) throw ArgError("no voice table loaded (kkx_load_voices)");
  if (B <= 0 || !mix_offsets || !voice_ids || !portions || !style_rows) throw ArgError("null input pointer");
  if (mix_offsets[0] < 0) throw ArgError("mix_offsets[0] must be >= 0");
  for (int b = 0; b < B; b++) {
    if (mix_offsets[b + 1] <= mix_offsets[b]) throw ArgError("every item needs at least one voice");
    if (style_rows[b] < 0 || style_rows[b] > 510) throw ArgError("style row must be in 0..510 (koko.rs:1262 indexes a 511-row table)");
    for (int i = mix_offsets[b]; i < mix_offsets[b + 1]; i++)
      if (voice_ids[i] < 0 || voice_ids[i] >= n_voices_) throw ArgError("voice id out of range");
  }
  stage(B, tokens, tok_offsets, nullptr, speeds);
  staged_ = false;                               // not runnable until the styles are mixed
  const int nmix = mix_offsets[B];
  int* d_mo = ioA_.alloc<int>(B + 1);
  int* d_vi = ioA_.alloc<int>(nmix);
  float* d_po = ioA_.alloc<float>(nmix);
  int* d_rows = ioA_.alloc<int>(B);
  upload(d_mo, mix_offsets, (B + 1) * sizeof(int));
  upload(d_vi, voice_ids, nmix * sizeof(int));
  upload(d_po, portions, nmix * sizeof(float));
  upload(d_rows, style_rows, B * sizeof(int));
  g_launch_stats = nullptr;
  launch_mix_styles(d_voices_, d_mo, d_vi, d_po, d_rows, d_styles_, B, stream_);
  // (host-mixed and device-mixed styles live at the same address, so token-phase graphs serve both entry points)
  staged_ = true;
}

void check_programs(int B, int P, const int32_t* p) {
  if (P < 1 || P > B) throw ArgError("n_programs must be in 1.." + std::to_string(B) + " (got " + std::to_string(P) + ")");
  if (!p) throw ArgError("program_offsets is null");
  if (p[0] != 0 || p[P] != B) throw ArgError("program_offsets must start at 0 and end at the batch size");
  for (int k = 0; k < P; k++)
    if (p[k + 1] <= p[k]) throw ArgError("program_offsets must be strictly increasing (no empty program)");
}

namespace {
long long bytes_per_sample(Encoding e) {
  return e == Encoding::F32 ? sizeof(float) : e == Encoding::ULAW || e == Encoding::ALAW ? 1 : sizeof(short);
}
}  // namespace

long long Model::encoded_bytes() const {
  if (!ran_) return 0;
  return enc_ == Encoding::FLAC ? flac_off_[n_prog()] : total_samples_ * bytes_per_sample(enc_);
}

void Model::fetch_encoded(void* dst, long long capacity_bytes, int64_t* byte_offsets, int64_t* sample_offsets,
                          int32_t* pred_dur) {
  if (!ran_) throw StateError("no completed run to fetch from");
  fetch(nullptr, 0, sample_offsets, pred_dur);
  if (byte_offsets)
    for (int k = 0; k <= n_prog(); k++)
      byte_offsets[k] = enc_ == Encoding::FLAC ? flac_off_[k] : sample_off_[k] * bytes_per_sample(enc_);
  if (dst) {
    const long long n = encoded_bytes();
    if (capacity_bytes < n) throw ArgError("output buffer too small");
    const void* src = enc_ == Encoding::FLAC ? flacA_.base() : enc_ == Encoding::F32 ? audioA_.base() : twinA_.base();
    KKX_CUDA(cudaMemcpyAsync(dst, src, (size_t)n, cudaMemcpyDeviceToHost, stream_));
    KKX_CUDA(cudaStreamSynchronize(stream_));
  }
}

// The resampling pass of this run: off at 24 kHz unless G.711 codes or loudness normalisation are wanted (then a
// pass-through, U = D = 1, which applies the gain).  The taps live on the device per Model and are rebuilt only when
// the rate changes.
void Model::prepare_resample() {
  loud_ = opt.loudness_target != 0;
  if (loud_) loud_par_ = loudness_params(opt.loudness_target / 100.0, opt.true_peak_max / 100.0);
  resample_ = opt.out_rate != 24000 || enc_ == Encoding::ULAW || enc_ == Encoding::ALAW || loud_;
  rs_U_ = 1; rs_D_ = 1; rs_H_ = 0;
  if (opt.out_rate == 24000) return;
  std::vector<float> taps;
  if (resample_design(opt.out_rate, &taps, &rs_U_, &rs_D_, &rs_H_) < 0)
    throw ArgError("out_rate " + std::to_string(opt.out_rate) + " is not supported");
  if (taps_rate_ != opt.out_rate) {
    KKX_CUDA(cudaStreamSynchronize(stream_));
    if (d_taps_) cudaFree(d_taps_);
    d_taps_ = nullptr; taps_rate_ = 0;
    KKX_CUDA(cudaMalloc(&d_taps_, taps.size() * sizeof(float)));
    KKX_CUDA(cudaMemcpy(d_taps_, taps.data(), taps.size() * sizeof(float), cudaMemcpyHostToDevice));
    taps_rate_ = opt.out_rate;
  }
}

void Model::fetch(float* dst, long long capacity, int64_t* sample_offsets, int32_t* pred_dur) {
  if (!ran_ || B_ <= 0 || n_prog() < 1 || (int)sample_off_.size() != n_prog() + 1)
    throw StateError("no completed run to fetch from");
  KKX_CUDA(cudaSetDevice(device_));
  if (sample_offsets)
    for (int k = 0; k <= n_prog(); k++) sample_offsets[k] = sample_off_[k];
  if (pred_dur) {
    size_t k = 0;
    for (int b = 0; b < B_; b++)
      for (int t = 0; t < tok_len_[b]; t++) pred_dur[k++] = h_pred_dur_[tokL_.off[b] + t];
  }
  if (dst) {
    if (capacity < total_samples_) throw ArgError("audio buffer too small");
    KKX_CUDA(cudaMemcpyAsync(dst, audioA_.base(), total_samples_ * sizeof(float), cudaMemcpyDeviceToHost, stream_));
    KKX_CUDA(cudaStreamSynchronize(stream_));
  }
}

// A grow-only output buffer, reset for the run; when it is too small the stream must be done with the old one.
void Model::grow(Arena& a, size_t bytes) {
  a.reset();
  if (bytes <= a.capacity()) return;
  KKX_CUDA(cudaStreamSynchronize(stream_));
  a.reserve(bytes + bytes / 4);
}

// ============================================================================ forward
void Model::run(Encoding enc, const std::vector<int>& programs) {
  if (!staged_ || B_ <= 0) throw StateError("no batch staged");
  if (!programs.empty()) check_programs(B_, (int)programs.size() - 1, programs.data());
  KKX_CUDA(cudaSetDevice(device_));
  ran_ = false;
  enc_ = enc;
  if (programs.empty()) {
    prog_.resize(B_ + 1);
    for (int b = 0; b <= B_; b++) prog_[b] = b;
  } else {
    prog_ = programs;
  }
  const int P = n_prog();
  use_lane(0);
  prepare_resample();
  g_launch_stats = &stats;
  stats.launches = 0;
  stats.conv_flops = 0;
  stats.arb_flops = 0; stats.arb_bytes = 0;
  stats.n_events = 0;
  stats.names.clear();
  dbg_.clear();
  group_first_.clear();
  KKX_CUDA(cudaEventRecord(ev0_, stream_));
  if (stats.profile) cudaEventRecord(stats.next_event(), stream_);
  Run r;
  try {
    token_phase(r);
  } catch (...) {
    if (capturing_) {                 // a failed capture must be ended before the stream is usable again
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(stream_, &g);
      if (g) cudaGraphDestroy(g);
      capturing_ = false;
    }
    cudaStreamSynchronize(stream_);   // nothing may still be reading the staging / arenas when the caller retries
    cudaStreamSynchronize(stream2_);
    cudaGetLastError();
    use_lane(0);
    throw;
  }

  // Items lie back to back in the run's 24 kHz waveform (600 T_b samples each), so a program is contiguous there.
  // Sample counts at the output rate are per program: program k of n_k samples at 24 kHz has ceil(n_k U / D).
  s24_off_.assign(B_ + 1, 0);
  long long tot = 0;
  for (int b = 0; b < B_; b++) {
    tot += r.T[b];
    s24_off_[b + 1] = s24_off_[b] + 600LL * r.T[b];
  }
  sample_off_.assign(P + 1, 0);
  for (int k = 0; k < P; k++) {
    const long long n24 = s24_off_[prog_[k + 1]] - s24_off_[prog_[k]];
    sample_off_[k + 1] = sample_off_[k] + (n24 * rs_U_ + rs_D_ - 1) / rs_D_;
  }
  total_samples_ = sample_off_[P];
  last_frames = tot;
  grow(audioA_, (size_t)total_samples_ * sizeof(float));
  r.audio = audioA_.alloc<float>(total_samples_);
  if (enc != Encoding::F32) {
    const size_t bytes = (size_t)total_samples_ * bytes_per_sample(enc);
    grow(twinA_, bytes);
    r.twin = twinA_.alloc_bytes(bytes);
  }
  if (resample_) {
    grow(wav24A_, (size_t)s24_off_[B_] * sizeof(float));
    r.wav24 = wav24A_.alloc<float>(s24_off_[B_]);
  }
  if (loud_) {
    grow(loudA_, (size_t)P * 3 * sizeof(float));
    r.loud = loudA_.alloc<float>((size_t)P * 3);
  }
  // FLAC: the encoder's tables -- sample offsets, frames per program (4096 samples each) as a prefix, program byte
  // offsets -- and its output, ready before the forward pass so that the encoder follows it without a host round trip
  struct { int F = 0; long long *soff = nullptr, *ioff = nullptr; int* foff = nullptr; void* work = nullptr;
           unsigned char* out = nullptr; } fl;
  if (enc == Encoding::FLAC) {
    std::vector<int> foff(P + 1, 0);
    for (int k = 0; k < P; k++) {
      const long long n = sample_off_[k + 1] - sample_off_[k];
      if (n > kMaxFlacSamples) throw ArgError("program too long for one FLAC stream (2^36 - 1 samples at most)");
      const long long nf = flac_frames(n);
      if (foff[k] + nf > 0x7FFFFFFFLL) throw ArgError("batch too long for one FLAC encode");
      foff[k + 1] = foff[k] + (int)nf;
    }
    fl.F = foff[P];
    const size_t bound = (size_t)flac_bound(P, fl.F, total_samples_);
    grow(flacA_, bound);
    fl.out = flacA_.alloc<unsigned char>(bound);
    grow(flacTabA_, 3 * ((size_t)(P + 1) * sizeof(long long) + 256) + flac_work_bytes(fl.F));
    fl.soff = flacTabA_.alloc<long long>(P + 1);
    fl.foff = flacTabA_.alloc<int>(P + 1);
    fl.ioff = flacTabA_.alloc<long long>(P + 1);
    fl.work = flacTabA_.alloc_bytes(flac_work_bytes(fl.F));
    upload(fl.soff, sample_off_.data(), (size_t)(P + 1) * sizeof(long long));
    upload(fl.foff, foff.data(), (size_t)(P + 1) * sizeof(int));
  }
  h_loud_.clear();
  sink_filled_ = false;
  float* sink = (host_sink && !debug_) ? host_sink(total_samples_) : nullptr;
  // (both streams are idle here: the previous run synchronised them, and the outputs were sized above)
  try {
    int b0 = 0, k0 = 0;
    while (b0 < B_) {
      int b1 = b0; long long fr = 0;
      // at most 512 items per group: the fused generator kernels keep per-item tables in shared memory, and a
      // batch must take the same code path as a single call (results are bit-identical either way)
      while (b1 < B_ && b1 - b0 < 512 && (b1 == b0 || fr + r.T[b1] <= opt.max_frames)) { fr += r.T[b1]; b1++; }
      group_first_.push_back(b0);
      int k1 = k0;   // programs [k0, k1) end in this group
      while (k1 < P && prog_[k1 + 1] <= b1) k1++;
      // size the arena with a dry run of the same allocation sequence (no launches, no copies)
      frA_.reset();
      frA_.set_virtual(true);
      g_dry_run = true;
      try {
        frame_phase(r, b0, b1, k0, k1, true);
      } catch (...) {
        g_dry_run = false; frA_.set_virtual(false);
        throw;
      }
      g_dry_run = false;
      frA_.set_virtual(false);
      const size_t need = frA_.used();
      if (need + (1 << 20) > frA_.capacity()) {
        KKX_CUDA(cudaStreamSynchronize(stream_));
        frA_.reserve(need + need / 8 + (1 << 20));
      }
      frA_.reset();
      frame_phase(r, b0, b1, k0, k1, false);
      if (sink && k1 > k0) {   // the programs this group completed go to the host while the next group computes
        const long long s0 = sample_off_[k0], s1 = sample_off_[k1];
        KKX_CUDA(cudaEventRecord(ev_grp_, stream_));
        KKX_CUDA(cudaStreamWaitEvent(copy_stream_, ev_grp_, 0));
        if (s1 > s0)
          KKX_CUDA(cudaMemcpyAsync(sink + s0, r.audio + s0, (size_t)(s1 - s0) * sizeof(float), cudaMemcpyDeviceToHost, copy_stream_));
      }
      b0 = b1;
      k0 = k1;
    }
    KKX_CUDA(cudaEventRecord(ev1_, stream_));
    if (enc == Encoding::FLAC) {
      launch_flac(static_cast<const short*>(r.twin), fl.soff, fl.foff, P, fl.F, opt.out_rate, fl.work, fl.out, fl.ioff,
                  stream_);
      flac_off_.assign(P + 1, 0);
      KKX_CUDA(cudaMemcpyAsync(flac_off_.data(), fl.ioff, (size_t)(P + 1) * sizeof(long long),
                               cudaMemcpyDeviceToHost, stream_));
    }
    KKX_CUDA(cudaStreamSynchronize(stream_));
    if (sink) { KKX_CUDA(cudaStreamSynchronize(copy_stream_)); sink_filled_ = true; }
    if (loud_) {   // [3][P] on the device -> program-major on the host
      std::vector<float> rows((size_t)P * 3);
      KKX_CUDA(cudaMemcpy(rows.data(), r.loud, rows.size() * sizeof(float), cudaMemcpyDeviceToHost));
      h_loud_.resize(rows.size());
      for (int k = 0; k < P; k++)
        for (int j = 0; j < 3; j++) h_loud_[(size_t)k * 3 + j] = rows[(size_t)j * P + k];
    }
  } catch (...) {
    cudaStreamSynchronize(stream_);
    cudaStreamSynchronize(stream2_);
    cudaStreamSynchronize(copy_stream_);
    use_lane(0);
    throw;
  }
  arb_timing_dump();
  float ms = 0.f;
  cudaEventElapsedTime(&ms, ev0_, ev1_);
  last_gpu_us = ms * 1e3;
  if (stats.profile) {
    prof_.clear();
    for (size_t i = 0; i + 1 < stats.n_events && i < stats.names.size(); i++) {
      float dt = 0.f;
      cudaEventElapsedTime(&dt, stats.events[i], stats.events[i + 1]);
      auto& e = prof_[stats.names[i]];
      e.first += 1; e.second += dt * 1e3;
    }
  }
  g_launch_stats = nullptr;
  ran_ = true;
}

}  // namespace kkx
