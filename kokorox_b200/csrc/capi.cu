// capi.cu -- the extern "C" boundary (include/kkx.h).  Every entry point catches all C++
// exceptions and converts them to a negative return code + message: nothing unwinds or aborts
// across the ABI (the reference `expect`s on bad outputs, ort_koko.rs:82,86, and its CLI turns a
// panic into abort(); a library must not).  The entry points take their C linkage from the declarations in the headers.
#include "../../include/kkx.h"
#include "../../include/kkx_test.h"
#include "model.h"
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <initializer_list>
#include <mutex>
#include <map>
#include <numeric>
#include <functional>
#include <sstream>
#include <atomic>
#include <thread>

using namespace kkx;

struct kkx_ctx {
  std::unique_ptr<Model> model;
  std::mutex mu;  // single-flight like the reference's Mutex<Session> (ort_koko.rs:14,77-78)
  // pinned result buffers; their own lock, so that kkx_release never waits for the step `mu` is held across
  std::mutex pool_mu;
  // One result buffer (cap in bytes), referenced once by every pointer handed out into it: a plain result is a block
  // with one reference, a coalesced batch one block with a reference per caller's view.
  struct Block { void* base; size_t cap; int refs; };
  std::map<void*, Block*> handed;        // every pointer handed to a caller -> its block
  std::vector<std::pair<void*, size_t>> pinned_free;  // returned buffers kept for reuse
  size_t pinned_free_bytes = 0;
  size_t pinned_hi = 0;                  // largest request so far: big buffers are sized alike so they recycle

  // Request coalescing (SURVEY 8f row 4): concurrent kkx_infer callers queue here; one of them becomes the
  // leader, runs everything queued as ONE ragged batch and hands each caller a view into the shared result
  // buffer.  The reference queues the same callers on Mutex<Session> and runs them one by one (ort_koko.rs:77).
  struct Waiter {
    const int64_t* tokens; int32_t n; const float* style; float speed; int32_t* pred_dur;
    float* audio = nullptr; int64_t samples = 0; int rc = 0; std::string err; bool done = false;
  };
  std::mutex qmu;
  std::condition_variable qcv;
  std::deque<Waiter*> queue;
  bool leader = false;
  long long max_tokens = 40960;  // tokens per pass of one call (64 x 512-token utterances + slack)
  std::atomic<int> coalesce_max{0};      // 0/1 = off (reference behaviour); >1 = largest batch a leader gathers
  std::atomic<int> coalesce_wait_us{0};  // how long a leader waits for company before it runs
  int64_t coalesced_batches = 0, coalesced_requests = 0, coalesced_largest = 0;   // guarded by qmu

  // Asynchronous requests (kkx_submit / kkx_poll / kkx_wait): a worker thread owned by the ctx drains the queue in
  // FIFO batches, so a caller can hand in sentence k+1 and go on sending sentence k (websocket lib.rs:371-376).
  struct AsyncReq {
    std::vector<int64_t> tokens; float style[256]; std::vector<int32_t> dur;
    Waiter w{};
    bool taken = false;
  };
  std::mutex amu;
  std::condition_variable acv_work, acv_done;
  std::map<int64_t, std::unique_ptr<AsyncReq>> tickets;
  std::deque<Waiter*> aqueue;
  std::thread worker;
  bool worker_started = false, astop = false;
  int64_t next_ticket = 1;
  std::atomic<int> async_batch{64};      // most requests the worker merges into one ragged batch
  int64_t async_batches = 0, async_requests = 0;                                 // guarded by amu

  // Per-item report of the last synchronous call (kkx_last_loudness / _limiter / _loudness_range), guarded by `mu`:
  // kReportRows floats per item (output.h), appended pass by pass; `groups` = the row groups its runs produced, valid
  // once the call has succeeded.
  std::vector<float> report;
  unsigned report_groups = 0;
  bool report_valid = false;
};

static thread_local std::string g_err;
static constexpr int kMaxCoalesce = 512;
// Most tokens in one batch the coalescing leader or the async worker gathers: the 64 x 512-token working set the
// step is sized for.
static constexpr long long kBatchTokens = 64 * 512;

template <class F>
static int guarded(F&& f) {
  std::string msg;
  int rc = KKX_OK;
  try {
    f();
    return KKX_OK;
  } catch (const ArgError& e) { rc = KKX_ERR_ARG; msg = e.what();
  } catch (const IoError& e) { rc = KKX_ERR_IO; msg = e.what();
  } catch (const StateError& e) { rc = KKX_ERR_STATE; msg = e.what();
  } catch (const CudaError& e) { rc = KKX_ERR_CUDA; msg = e.what();
  } catch (const std::exception& e) { rc = KKX_ERR_CUDA; msg = e.what();
  } catch (...) { rc = KKX_ERR_CUDA; msg = "unknown error"; }
  g_launch_stats = nullptr;
  g_dry_run = false;
  g_err = msg;
  return rc;
}

static int check_ctx(kkx_ctx* ctx) {
  if (!ctx) { g_err = "null ctx"; return KKX_ERR_ARG; }
  if (!ctx->model) { g_err = "Session is not initialized."; return KKX_ERR_STATE; }
  return KKX_OK;
}

// Every entry point that works on the session: `f` runs single-flight under ctx->mu, its exception becomes the
// return code and kkx_last_error's message.
template <class F>
static int session_call(kkx_ctx* ctx, F&& f) {
  const int rc = check_ctx(ctx);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(ctx->mu);
  return guarded(f);
}

KKX_API const char* kkx_version(void) { return "kkx 0.1 sm_100a"; }

KKX_API int kkx_init(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0) {
    g_err = std::string("no CUDA device available: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
            " (the B200 backend has no CPU fallback)";
    cudaGetLastError();
    return KKX_ERR_NO_DEVICE;
  }
  return KKX_OK;
}

KKX_API int kkx_create(const char* weights_path, int device_ordinal, kkx_ctx** out) {
  if (out) *out = nullptr;
  if (!weights_path || !out) { g_err = "kkx_create: null argument"; return KKX_ERR_ARG; }
  int rc = kkx_init();
  if (rc != KKX_OK) return rc;
  kkx_ctx* ctx = new (std::nothrow) kkx_ctx();
  if (!ctx) { g_err = "out of memory"; return KKX_ERR_CUDA; }
  rc = guarded([&] { ctx->model.reset(new Model(weights_path, device_ordinal)); });
  if (rc != KKX_OK) { delete ctx; return rc; }
  *out = ctx;
  return KKX_OK;
}

// Host-only: read a model file the way kkx_create does (KKXW or ONNX, see kkx.h) and write the recovered state dict
// as a KKXW file.  Lets a deployment convert once and lets the CPU test-suite check the ONNX reader without a GPU.
KKX_API int kkx_convert_model_file(const char* src_path, const char* dst_kkxw_path, int32_t* out_tensors) {
  if (!src_path || !dst_kkxw_path) { g_err = "kkx_convert_model_file: null argument"; return KKX_ERR_ARG; }
  return guarded([&] {
    WeightFile wf(src_path);
    std::vector<std::string> names;
    for (auto& sp : kokoro_tensor_specs()) names.push_back(sp.first);
    std::vector<char> hdr;
    auto put = [&](const void* p, size_t n) { hdr.insert(hdr.end(), (const char*)p, (const char*)p + n); };
    std::vector<uint64_t> offs;
    uint64_t off = 0;
    for (auto& n : names) {
      const HostTensor& t = wf.get(n);
      const uint16_t ln = (uint16_t)n.size();
      put(&ln, 2); put(n.data(), n.size());
      const uint32_t dtype = 0, ndim = (uint32_t)t.shape.size();
      put(&dtype, 4); put(&ndim, 4);
      for (int d : t.shape) { const uint32_t v = (uint32_t)d; put(&v, 4); }
      const uint64_t nb = (uint64_t)t.numel * 4;
      put(&off, 8); put(&nb, 8);
      offs.push_back(off);
      off += (nb + 63) / 64 * 64;
    }
    const uint32_t n = (uint32_t)names.size();
    const uint32_t header_bytes = (uint32_t)((16 + hdr.size() + 255) / 256 * 256);
    FILE* f = fopen(dst_kkxw_path, "wb");
    if (!f) throw IoError(std::string("cannot write ") + dst_kkxw_path);
    bool ok = fwrite("KKXW0001", 1, 8, f) == 8 && fwrite(&n, 4, 1, f) == 1 && fwrite(&header_bytes, 4, 1, f) == 1 &&
              fwrite(hdr.data(), 1, hdr.size(), f) == hdr.size();
    std::vector<char> zeros(256, 0);
    ok = ok && fwrite(zeros.data(), 1, header_bytes - 16 - hdr.size(), f) == header_bytes - 16 - hdr.size();
    for (size_t i = 0; ok && i < names.size(); i++) {
      const HostTensor& t = wf.get(names[i]);
      const size_t nb = t.numel * 4, pad = (nb + 63) / 64 * 64 - nb;
      ok = fwrite(t.data, 1, nb, f) == nb && fwrite(zeros.data(), 1, pad, f) == pad;
    }
    ok = (fclose(f) == 0) && ok;
    if (!ok) throw IoError(std::string("short write: ") + dst_kkxw_path);
    if (out_tensors) *out_tensors = (int32_t)names.size();
  });
}

KKX_API void kkx_destroy(kkx_ctx* ctx) {
  if (!ctx) return;
  if (ctx->worker_started) {   // stop the async worker; requests still queued fail with KKX_ERR_STATE
    {
      std::lock_guard<std::mutex> al(ctx->amu);
      ctx->astop = true;
    }
    ctx->acv_work.notify_all();
    if (ctx->worker.joinable()) ctx->worker.join();
  }
  try {
    if (ctx->model) cudaSetDevice(ctx->model->device());
    for (auto& h : ctx->handed)
      if (--h.second->refs == 0) { cudaFreeHost(h.second->base); delete h.second; }
    for (auto& p : ctx->pinned_free) cudaFreeHost(p.first);
    ctx->model.reset();
  } catch (...) {}
  delete ctx;
}

// The message of the calling thread's last failed call (any ctx).  Thread-local on purpose: with many threads
// sharing one ctx (the reference's Arc<OrtKoko>), a per-ctx string could be rewritten by another thread while the
// caller still reads it.
KKX_API const char* kkx_last_error(const kkx_ctx* ctx) { (void)ctx; return g_err.c_str(); }

// A pooled pinned result buffer of at least `need` bytes
static void* take_pinned(kkx_ctx* ctx, size_t need, size_t* cap_out) {
  void* host = nullptr;
  size_t cap = 0, hi = 0;
  {
    std::lock_guard<std::mutex> pl(ctx->pool_mu);
    hi = ctx->pinned_hi = std::max(ctx->pinned_hi, need);
    size_t best = ctx->pinned_free.size();   // smallest buffer that fits
    for (size_t i = 0; i < ctx->pinned_free.size(); i++)
      if (ctx->pinned_free[i].second >= need &&
          (best == ctx->pinned_free.size() || ctx->pinned_free[i].second < ctx->pinned_free[best].second))
        best = i;
    if (best < ctx->pinned_free.size()) {
      host = ctx->pinned_free[best].first; cap = ctx->pinned_free[best].second;
      ctx->pinned_free.erase(ctx->pinned_free.begin() + best);
      ctx->pinned_free_bytes -= cap;
    }
  }
  if (!host) {
    // pinned allocation costs ~1 ms per MB and synchronises the device: give every request in the top size class
    // the same capacity, so a stream of similar batches reuses the pooled buffers instead of outgrowing them
    const size_t base = need >= hi / 2 ? hi : need;
    cap = std::max<size_t>(base + base / 8, 4096);
    KKX_CUDA(cudaMallocHost(&host, cap));
  }
  *cap_out = cap;
  return host;
}
// Result buffer `base` handed out at the addresses `at`, one reference each; kkx_release recycles it with the last.
static void hand_out(kkx_ctx* ctx, void* base, size_t cap, const std::vector<void*>& at) {
  std::lock_guard<std::mutex> pl(ctx->pool_mu);
  auto* b = new kkx_ctx::Block{base, cap, (int)at.size()};
  for (void* p : at) ctx->handed[p] = b;
}

KKX_API void kkx_release(kkx_ctx* ctx, float* audio);

// The report of a synchronous call (kkx_last_loudness / _limiter / _loudness_range; caller holds ctx->mu; throws):
// `runs(note)` runs the model one or more times and calls note() after each run, which appends that run's rows; the
// report restarts before `runs` and is valid once it has returned.  Coalesced and asynchronous batches do not come
// through here, so they leave the report alone (kkx.h).
template <class F>
static void record_report(kkx_ctx* ctx, F&& runs) {
  const Model& m = *ctx->model;
  ctx->report.clear(); ctx->report_groups = 0; ctx->report_valid = false;
  runs([&] {
    if (!m.report_groups()) return;
    ctx->report_groups |= m.report_groups();
    ctx->report.insert(ctx->report.end(), m.last_report().begin(), m.last_report().end());
  });
  ctx->report_valid = true;
}
// items of the last synchronous call's report with row group `group`, 0 without one
static int64_t report_items(const kkx_ctx* ctx, unsigned group) {
  return ctx->report_valid && (ctx->report_groups & group) ? (int64_t)(ctx->report.size() / kReportRows) : 0;
}

// The argument contract of one utterance (kkx.h): checked before a request is queued anywhere.
static int validate_request(const int64_t* tokens, int32_t n_tokens, const float* style256, float speed) {
  if (!tokens || !style256) { g_err = "null argument"; return KKX_ERR_ARG; }
  if (n_tokens < 1 || n_tokens > KKX_MAX_TOKENS) { g_err = "n_tokens must be in 1..512 (got " + std::to_string(n_tokens) + ")"; return KKX_ERR_ARG; }
  if (!(speed >= kMinSpeed && speed <= kMaxSpeed)) { g_err = "speed must be in [0.1, 10] (got " + std::to_string(speed) + ")"; return KKX_ERR_ARG; }
  for (int32_t i = 0; i < n_tokens; i++)
    if (tokens[i] < 0 || tokens[i] > 177) { g_err = "token id out of range 0..177: " + std::to_string(tokens[i]); return KKX_ERR_ARG; }
  return KKX_OK;
}

// One ragged batch through the model into a pooled pinned buffer (caller holds ctx->mu; throws).  The buffer is
// handed to the model as a sink: every frame group's audio is copied out on a second stream while the next
// group computes.  `note` follows the run (record_report).
static void run_staged_locked(kkx_ctx* ctx, float** host_out, size_t* cap_out, int64_t* out_sample_offsets,
                              int32_t* out_pred_dur, const std::function<void()>& note) {
  Model& m = *ctx->model;
  float* host = nullptr;
  size_t cap = 0;
  m.host_sink = [&](long long n) { host = static_cast<float*>(take_pinned(ctx, n * sizeof(float), &cap)); return host; };
  try {
    m.run();
    m.host_sink = nullptr;
    note();
    const long long n = m.total_samples();
    if (!host) host = static_cast<float*>(take_pinned(ctx, n * sizeof(float), &cap));
    m.fetch(m.sink_filled() ? nullptr : host, n, out_sample_offsets, out_pred_dur);
  } catch (...) { m.host_sink = nullptr; if (host) cudaFreeHost(host); throw; }
  *host_out = host;
  *cap_out = cap;
}
// A result buffer that came back: kept for reuse (pinned allocation costs milliseconds and synchronises the device)
// up to 64 buffers and 1 GiB, freed otherwise.
static void recycle_pinned(kkx_ctx* ctx, void* host, size_t cap) {
  {
    std::lock_guard<std::mutex> pl(ctx->pool_mu);
    if (ctx->pinned_free.size() < 64 && ctx->pinned_free_bytes + cap <= (size_t(1) << 30)) {
      ctx->pinned_free.push_back({host, cap});
      ctx->pinned_free_bytes += cap;
      return;
    }
  }
  if (ctx->model) cudaSetDevice(ctx->model->device());
  cudaFreeHost(host);
}

// A call may carry any number of utterances; the device working set is bounded by running at most `max_tokens`
// tokens per pass (the token phase keeps ~75 KB per token row; the frame phase has its own budget, max_frames).
// Utterances are independent and a batch's results do not depend on its composition, so the split is invisible
// apart from one host-side concatenation.
static void run_batch_locked(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                             const float* styles, const float* speeds, float** host_out, size_t* cap_out,
                             int64_t* out_sample_offsets, int32_t* out_pred_dur, const std::function<void()>& note) {
  if (batch <= 0 || !tok_offsets) throw ArgError("batch must be >= 1");
  const long long budget = ctx->max_tokens;
  if (batch == 1 || (long long)tok_offsets[batch] - tok_offsets[0] <= budget) {
    ctx->model->stage(batch, tokens, tok_offsets, styles, speeds);
    run_staged_locked(ctx, host_out, cap_out, out_sample_offsets, out_pred_dur, note);
    return;
  }
  if (!styles) throw ArgError("null input pointer");
  struct Part { float* host; size_t cap; int b0, b1; };
  std::vector<Part> parts;
  std::vector<int64_t> soff((size_t)batch + 1, 0);
  try {
    for (int b0 = 0; b0 < batch;) {
      int b1 = b0 + 1;
      while (b1 < batch && (long long)tok_offsets[b1 + 1] - tok_offsets[b0] <= budget) b1++;
      std::vector<int64_t> so((size_t)(b1 - b0) + 1, 0);
      Part p{nullptr, 0, b0, b1};
      ctx->model->stage(b1 - b0, tokens, tok_offsets + b0, styles + (size_t)b0 * 256, speeds + b0);
      run_staged_locked(ctx, &p.host, &p.cap, so.data(),
                        out_pred_dur ? out_pred_dur + (tok_offsets[b0] - tok_offsets[0]) : nullptr, note);
      parts.push_back(p);
      for (int i = 0; i < b1 - b0; i++) soff[b0 + i + 1] = soff[b0] + so[i + 1];
      b0 = b1;
    }
    size_t cap = 0;
    float* host = static_cast<float*>(take_pinned(ctx, soff[batch] * sizeof(float), &cap));
    for (const Part& p : parts)
      memcpy(host + soff[p.b0], p.host, (size_t)(soff[p.b1] - soff[p.b0]) * sizeof(float));
    for (const Part& p : parts) recycle_pinned(ctx, p.host, p.cap);
    if (out_sample_offsets) memcpy(out_sample_offsets, soff.data(), soff.size() * sizeof(int64_t));
    *host_out = host;
    *cap_out = cap;
  } catch (...) {
    for (const Part& p : parts) cudaFreeHost(p.host);
    throw;
  }
}

KKX_API int kkx_infer_batch(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                    const float* styles, const float* speeds, float** out_audio,
                    int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return session_call(ctx, [&] {
    if (!out_audio) throw ArgError("out_audio is null");
    *out_audio = nullptr;
    float* host = nullptr;
    size_t cap = 0;
    record_report(ctx, [&](const std::function<void()>& note) {
      run_batch_locked(ctx, batch, tokens, tok_offsets, styles, speeds, &host, &cap, out_sample_offsets, out_pred_dur,
                       note);
    });
    hand_out(ctx, host, cap, {host});
    *out_audio = host;
  });
}

// Leader side of the coalescer and of the async worker: run `batch` as one ragged batch; on failure re-run the
// requests one by one so that only the offending caller sees the error.  True when the batch ran as one.
static bool serve_coalesced(kkx_ctx* ctx, const std::vector<kkx_ctx::Waiter*>& batch) {
  const int B = (int)batch.size();
  std::vector<int32_t> offs(B + 1, 0);
  for (int i = 0; i < B; i++) offs[i + 1] = offs[i] + std::max(batch[i]->n, 0);
  std::vector<int64_t> toks((size_t)std::max(offs[B], 1));
  std::vector<float> styles((size_t)B * 256), speeds(B);
  std::vector<int64_t> soff(B + 1, 0);
  std::vector<int32_t> dur((size_t)std::max(offs[B], 1));
  bool args_ok = true;
  for (int i = 0; i < B; i++) {
    kkx_ctx::Waiter& w = *batch[i];
    if (!w.tokens || !w.style || w.n <= 0) { args_ok = false; continue; }
    memcpy(&toks[offs[i]], w.tokens, (size_t)w.n * sizeof(int64_t));
    memcpy(&styles[(size_t)i * 256], w.style, 256 * sizeof(float));
    speeds[i] = w.speed;
  }
  const std::function<void()> no_report = [] {};
  std::lock_guard<std::mutex> lk(ctx->mu);
  float* host = nullptr;
  size_t cap = 0;
  int rc = KKX_ERR_ARG;
  if (args_ok)
    rc = guarded([&] {
      run_batch_locked(ctx, B, toks.data(), offs.data(), styles.data(), speeds.data(), &host, &cap, soff.data(),
                       dur.data(), no_report);
    });
  if (rc == KKX_OK) {
    std::vector<void*> views(B);
    for (int i = 0; i < B; i++) {
      kkx_ctx::Waiter& w = *batch[i];
      w.audio = host + soff[i];
      w.samples = soff[i + 1] - soff[i];   // >= 200: every token lasts at least one frame, so view addresses are distinct
      if (w.pred_dur) memcpy(w.pred_dur, &dur[offs[i]], (size_t)w.n * sizeof(int32_t));
      w.rc = KKX_OK;
      views[i] = w.audio;
    }
    hand_out(ctx, host, cap, views);
    return true;
  }
  for (int i = 0; i < B; i++) {   // isolate the failure
    kkx_ctx::Waiter& w = *batch[i];
    const int32_t o1[2] = {0, w.n};
    int64_t s1[2] = {0, 0};
    float* h1 = nullptr;
    size_t c1 = 0;
    w.rc = guarded([&] {
      if (!w.tokens || !w.style) throw ArgError("null argument");
      run_batch_locked(ctx, 1, w.tokens, o1, w.style, &w.speed, &h1, &c1, s1, w.pred_dur, no_report);
    });
    if (w.rc == KKX_OK) {
      hand_out(ctx, h1, c1, {h1});
      w.audio = h1;
      w.samples = s1[1];
    } else {
      w.err = g_err;      // guarded() left the message in this (the leader's) thread
    }
  }
  return false;
}

// The request batcher of the coalescing leader and of the async worker (caller holds `lk` on `queue`'s mutex, which
// is released while the batch runs): takes a FIFO batch of at most `want` requests and kBatchTokens tokens off
// `queue` and serves it.  `together` says whether it ran as one batch.
static std::vector<kkx_ctx::Waiter*> serve_queue(kkx_ctx* ctx, std::deque<kkx_ctx::Waiter*>& queue,
                                                 std::unique_lock<std::mutex>& lk, size_t want, const char* what,
                                                 bool* together) {
  std::vector<kkx_ctx::Waiter*> batch;
  long long tok = 0;
  while (!queue.empty() && batch.size() < want) {
    kkx_ctx::Waiter* q = queue.front();
    if (!batch.empty() && tok + q->n > kBatchTokens) break;
    tok += std::max(q->n, 0);
    batch.push_back(q);
    queue.pop_front();
  }
  lk.unlock();
  *together = false;
  try {
    *together = serve_coalesced(ctx, batch);
  } catch (...) {   // (allocation failure outside guarded()): fail the batch, never leave the queue without a server
    for (auto* w : batch) { w->rc = KKX_ERR_CUDA; w->err = std::string("internal error while serving ") + what; w->audio = nullptr; }
  }
  lk.lock();
  for (auto* w : batch) w->done = true;
  return batch;
}

static int infer_coalesced(kkx_ctx* ctx, kkx_ctx::Waiter& w) {
  std::unique_lock<std::mutex> ql(ctx->qmu);
  ctx->queue.push_back(&w);
  if (ctx->leader) ctx->qcv.notify_all();   // a leader may be waiting for company
  while (!w.done) {
    if (ctx->leader) { ctx->qcv.wait(ql); continue; }
    ctx->leader = true;
    const size_t want = (size_t)std::max(ctx->coalesce_max.load(), 1);
    const int wait_us = ctx->coalesce_wait_us.load();
    if (wait_us > 0 && ctx->queue.size() < want)
      ctx->qcv.wait_for(ql, std::chrono::microseconds(wait_us), [&] { return ctx->queue.size() >= want; });
    bool together = false;
    const auto batch = serve_queue(ctx, ctx->queue, ql, want, "a coalesced batch", &together);
    if (together) {
      ctx->coalesced_batches++;
      ctx->coalesced_requests += (int64_t)batch.size();
      ctx->coalesced_largest = std::max<int64_t>(ctx->coalesced_largest, (int64_t)batch.size());
    } else {
      for (auto* b : batch)
        if (b->rc == KKX_OK) { ctx->coalesced_batches++; ctx->coalesced_requests++; }
    }
    ctx->leader = false;
    ctx->qcv.notify_all();
  }
  if (w.rc != KKX_OK) g_err = w.err;
  return w.rc;
}

KKX_API int kkx_load_voices(kkx_ctx* ctx, const float* table, int32_t n_voices) {
  return session_call(ctx, [&] { ctx->model->load_voices(table, n_voices); });
}

KKX_API int kkx_infer_batch_voices(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                           const int32_t* mix_offsets, const int32_t* voice_ids, const float* voice_portions,
                           const int32_t* style_rows, const float* speeds, float** out_audio,
                           int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return session_call(ctx, [&] {
    if (!out_audio) throw ArgError("out_audio is null");
    *out_audio = nullptr;
    ctx->model->stage_voices(batch, tokens, tok_offsets, mix_offsets, voice_ids, voice_portions, style_rows, speeds);
    float* host = nullptr;
    size_t cap = 0;
    record_report(ctx, [&](const std::function<void()>& note) {
      run_staged_locked(ctx, &host, &cap, out_sample_offsets, out_pred_dur, note);
    });
    hand_out(ctx, host, cap, {host});
    *out_audio = host;
  });
}

// The encoded entry points (kkx_infer_batch_pcm16 / _g711 / _flac / _mp3, kkx_infer_programs / _mp3): one pass of
// the batch with `enc` (kbps: the MP3 bitrate), its bytes in a pooled pinned buffer.  `out_name`: the out-pointer's
// name in the messages; `byte_offsets`: whether the entry point takes out_byte_offsets (then it must not be null);
// `bad_enc`: why the requested encoding is refused ("" = it is not); `programs`: whether the call takes a program
// table (n_programs, program_offsets), one item per program otherwise.  Every check runs before the batch is staged,
// so a rejected call leaves the session as it was.
template <class T>
static int infer_encoded(kkx_ctx* ctx, const char* out_name, T** out, bool byte_offsets, int64_t* out_byte_offsets,
                         Encoding enc, const std::string& bad_enc, int32_t kbps, bool programs, int32_t n_programs,
                         const int32_t* program_offsets, int32_t batch, const int64_t* tokens,
                         const int32_t* tok_offsets, const float* styles, const float* speeds,
                         int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return session_call(ctx, [&] {
    if (!out) throw ArgError(std::string(out_name) + " is null");
    *out = nullptr;
    if (byte_offsets && !out_byte_offsets) throw ArgError("out_byte_offsets is null");
    if (!bad_enc.empty()) throw ArgError(bad_enc);
    if (enc == Encoding::MP3) mp3_format(ctx->model->opt.out_rate, kbps);
    std::vector<int> table;
    if (programs) {
      if (batch < 1) throw ArgError("batch must be >= 1");
      check_programs(batch, n_programs, program_offsets);
      table.assign(program_offsets, program_offsets + n_programs + 1);
    }
    Model& m = *ctx->model;
    m.stage(batch, tokens, tok_offsets, styles, speeds);
    void* host = nullptr;
    size_t cap = 0;
    record_report(ctx, [&](const std::function<void()>& note) {
      m.run(enc, table, kbps);
      note();
      const long long n = m.encoded_bytes();
      host = take_pinned(ctx, (size_t)n, &cap);
      try {
        m.fetch_encoded(host, n, out_byte_offsets, out_sample_offsets, out_pred_dur);
      } catch (...) { cudaFreeHost(host); throw; }
    });
    hand_out(ctx, host, cap, {host});
    *out = static_cast<T*>(host);
  });
}

KKX_API int kkx_infer_batch_pcm16(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                          const float* styles, const float* speeds, int16_t** out_pcm,
                          int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return infer_encoded(ctx, "out_pcm", out_pcm, false, nullptr, Encoding::PCM16, "", 0, false, 0, nullptr, batch,
                       tokens, tok_offsets, styles, speeds, out_sample_offsets, out_pred_dur);
}

KKX_API void kkx_release_pcm16(kkx_ctx* ctx, int16_t* pcm) { kkx_release(ctx, reinterpret_cast<float*>(pcm)); }

KKX_API int kkx_infer_batch_g711(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                 const float* styles, const float* speeds, int32_t law, uint8_t** out_codes,
                                 int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  const std::string bad = law == 0 || law == 1 ? "" : "law must be 0 (mu-law) or 1 (A-law), got " + std::to_string(law);
  return infer_encoded(ctx, "out_codes", out_codes, false, nullptr, law ? Encoding::ALAW : Encoding::ULAW, bad, 0,
                       false, 0, nullptr, batch, tokens, tok_offsets, styles, speeds, out_sample_offsets, out_pred_dur);
}

KKX_API void kkx_release_g711(kkx_ctx* ctx, uint8_t* codes) { kkx_release(ctx, reinterpret_cast<float*>(codes)); }

KKX_API int kkx_infer_batch_flac(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                 const float* styles, const float* speeds, uint8_t** out_bytes,
                                 int64_t* out_byte_offsets, int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return infer_encoded(ctx, "out_bytes", out_bytes, true, out_byte_offsets, Encoding::FLAC, "", 0, false, 0, nullptr,
                       batch, tokens, tok_offsets, styles, speeds, out_sample_offsets, out_pred_dur);
}

KKX_API void kkx_release_flac(kkx_ctx* ctx, uint8_t* bytes) { kkx_release(ctx, reinterpret_cast<float*>(bytes)); }

KKX_API int kkx_infer_programs(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                               const float* styles, const float* speeds, int32_t n_programs,
                               const int32_t* program_offsets, int32_t encoding, void** out_bytes,
                               int64_t* out_byte_offsets, int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  static const Encoding enc[] = {Encoding::F32, Encoding::PCM16, Encoding::ULAW, Encoding::ALAW, Encoding::FLAC};
  const bool ok = encoding >= KKX_ENC_F32 && encoding <= KKX_ENC_FLAC;
  const std::string bad = ok ? "" : "encoding must be in 0..4 (KKX_ENC_F32 .. KKX_ENC_FLAC), got " +
                                    std::to_string(encoding) + " (MP3: kkx_infer_programs_mp3)";
  return infer_encoded(ctx, "out_bytes", out_bytes, true, out_byte_offsets, ok ? enc[encoding] : Encoding::F32, bad, 0,
                       true, n_programs, program_offsets, batch, tokens, tok_offsets, styles, speeds,
                       out_sample_offsets, out_pred_dur);
}

KKX_API void kkx_release_programs(kkx_ctx* ctx, void* bytes) { kkx_release(ctx, static_cast<float*>(bytes)); }

KKX_API int kkx_infer_batch_mp3(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                const float* styles, const float* speeds, int32_t kbps, uint8_t** out_bytes,
                                int64_t* out_byte_offsets, int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return infer_encoded(ctx, "out_bytes", out_bytes, true, out_byte_offsets, Encoding::MP3, "", kbps, false, 0, nullptr,
                       batch, tokens, tok_offsets, styles, speeds, out_sample_offsets, out_pred_dur);
}

KKX_API int kkx_infer_programs_mp3(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                                   const float* styles, const float* speeds, int32_t n_programs,
                                   const int32_t* program_offsets, int32_t kbps, uint8_t** out_bytes,
                                   int64_t* out_byte_offsets, int64_t* out_sample_offsets, int32_t* out_pred_dur) {
  return infer_encoded(ctx, "out_bytes", out_bytes, true, out_byte_offsets, Encoding::MP3, "", kbps, true, n_programs,
                       program_offsets, batch, tokens, tok_offsets, styles, speeds, out_sample_offsets, out_pred_dur);
}

KKX_API void kkx_release_mp3(kkx_ctx* ctx, uint8_t* bytes) { kkx_release(ctx, reinterpret_cast<float*>(bytes)); }

// ---- output containers: host-side byte work (little-endian host assumed, as everywhere in this library)
static void put_u16(uint8_t* p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
static void put_u32(uint8_t* p, uint32_t v) { put_u16(p, v & 0xFFFF); put_u16(p + 2, v >> 16); }
static void wav_header(uint8_t* h, uint32_t riff_size, uint32_t data_size, uint32_t format, uint32_t channels,
                       uint32_t rate, uint32_t bits) {
  memcpy(h, "RIFF", 4); put_u32(h + 4, riff_size); memcpy(h + 8, "WAVEfmt ", 8);
  put_u32(h + 16, 16); put_u16(h + 20, format); put_u16(h + 22, channels); put_u32(h + 24, rate);
  put_u32(h + 28, rate * channels * bits / 8); put_u16(h + 32, channels * bits / 8); put_u16(h + 34, bits);
  memcpy(h + 36, "data", 4); put_u32(h + 40, data_size);
}

KKX_API int32_t kkx_wav_header_pcm16(uint8_t* dst44, int64_t n_samples, int32_t sample_rate) {
  if (!dst44 || n_samples < 0 || sample_rate <= 0) return KKX_ERR_ARG;
  const uint32_t bytes = (uint32_t)(n_samples * 2);     // u32 arithmetic like the reference (`as u32`)
  wav_header(dst44, 36u + bytes, bytes, 1, 1, (uint32_t)sample_rate, 16);
  return 44;
}

KKX_API int32_t kkx_wav_header_f32_stream(uint8_t* dst44, int32_t channels, int32_t sample_rate) {
  if (!dst44 || channels <= 0 || sample_rate <= 0) return KKX_ERR_ARG;
  wav_header(dst44, 0xFFFFFFFFu, 0xFFFFFFFFu, 3, (uint32_t)channels, (uint32_t)sample_rate, 32);
  return 44;
}

KKX_API int64_t kkx_encode_wav16_base64(const int16_t* pcm, int64_t n_samples, int32_t sample_rate, char* dst,
                                int64_t capacity) {
  if (n_samples < 0 || sample_rate <= 0 || (!pcm && n_samples > 0)) return KKX_ERR_ARG;
  const int64_t nbytes = 44 + n_samples * 2;
  const int64_t nchars = (nbytes + 2) / 3 * 4;
  if (!dst || capacity < nchars) return nchars;
  static const char T[] = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
  uint8_t head[48];
  kkx_wav_header_pcm16(head, n_samples, sample_rate);
  const uint8_t* body = reinterpret_cast<const uint8_t*>(pcm);
  const int64_t nbody = n_samples * 2;
  // the header is 44 = 14 * 3 + 2 bytes: borrow up to 4 body bytes so that it ends on a 3-byte group
  const int borrow = (int)std::min<int64_t>(4, nbody);
  for (int i = 0; i < borrow; i++) head[44 + i] = body[i];
  const int hbytes = 44 + borrow;                        // 48 when there is a body: 16 whole groups
  char* o = dst;
  auto group = [&](const uint8_t* p, int n) {            // n in 1..3 input bytes -> 4 chars
    const uint32_t v = ((uint32_t)p[0] << 16) | ((n > 1 ? (uint32_t)p[1] : 0u) << 8) | (n > 2 ? (uint32_t)p[2] : 0u);
    o[0] = T[v >> 18]; o[1] = T[(v >> 12) & 63];
    o[2] = n > 1 ? T[(v >> 6) & 63] : '=';
    o[3] = n > 2 ? T[v & 63] : '=';
    o += 4;
  };
  int hp = 0;
  for (; hp + 3 <= hbytes; hp += 3) group(head + hp, 3);
  if (hp < hbytes) {                                     // only when the body has < 4 bytes (0 or 2): tail of the stream
    group(head + hp, hbytes - hp);
  } else {
    int64_t bp = borrow;
    for (; bp + 3 <= nbody; bp += 3) group(body + bp, 3);
    if (bp < nbody) group(body + bp, (int)(nbody - bp));
  }
  if (capacity > nchars) *o = 0;
  return nchars;
}

KKX_API int kkx_infer(kkx_ctx* ctx, const int64_t* tokens, int32_t n_tokens, const float* style256,
              float speed, float** out_audio, int64_t* out_samples, int32_t* out_pred_dur) {
  if (out_samples) *out_samples = 0;
  if (ctx && ctx->model && ctx->coalesce_max.load() > 1) {
    if (out_audio) *out_audio = nullptr; else { g_err = "out_audio is null"; return KKX_ERR_ARG; }
    // validate BEFORE queueing: a bad request must fail here, alone and at once, not inside somebody's batch
    const int vrc = validate_request(tokens, n_tokens, style256, speed);
    if (vrc != KKX_OK) return vrc;
    kkx_ctx::Waiter w{tokens, n_tokens, style256, speed, out_pred_dur};
    const int rc = infer_coalesced(ctx, w);
    if (rc == KKX_OK) { *out_audio = w.audio; if (out_samples) *out_samples = w.samples; }
    return rc;
  }
  const int32_t offs[2] = {0, n_tokens};
  int64_t soff[2] = {0, 0};
  const int rc = kkx_infer_batch(ctx, 1, tokens, offs, style256, &speed, out_audio, soff, out_pred_dur);
  if (rc == KKX_OK && out_samples) *out_samples = soff[1];
  return rc;
}

// ---- asynchronous entry points --------------------------------------------------------------------------------
static void async_worker(kkx_ctx* ctx) {
  std::unique_lock<std::mutex> al(ctx->amu);
  for (;;) {
    ctx->acv_work.wait(al, [&] { return ctx->astop || !ctx->aqueue.empty(); });
    if (ctx->astop) {
      for (auto* w : ctx->aqueue) { w->rc = KKX_ERR_STATE; w->err = "session destroyed before the request ran"; w->done = true; }
      ctx->aqueue.clear();
      ctx->acv_done.notify_all();
      return;
    }
    bool together = false;
    const auto batch = serve_queue(ctx, ctx->aqueue, al, (size_t)std::max(ctx->async_batch.load(), 1),
                                   "an asynchronous batch", &together);
    ctx->async_batches++;
    ctx->async_requests += (int64_t)batch.size();
    ctx->acv_done.notify_all();
  }
}

KKX_API int kkx_submit(kkx_ctx* ctx, const int64_t* tokens, int32_t n_tokens, const float* style256, float speed,
                       kkx_ticket* out_ticket) {
  int rc = check_ctx(ctx);
  if (rc) return rc;
  if (!out_ticket) { g_err = "out_ticket is null"; return KKX_ERR_ARG; }
  *out_ticket = 0;
  rc = validate_request(tokens, n_tokens, style256, speed);
  if (rc) return rc;
  try {
    std::unique_ptr<kkx_ctx::AsyncReq> r(new kkx_ctx::AsyncReq());
    r->tokens.assign(tokens, tokens + n_tokens);      // the caller's buffers are free again when this call returns
    memcpy(r->style, style256, sizeof r->style);
    r->dur.assign((size_t)n_tokens, 0);
    r->w.tokens = r->tokens.data(); r->w.n = n_tokens; r->w.style = r->style; r->w.speed = speed;
    r->w.pred_dur = r->dur.data();
    std::lock_guard<std::mutex> al(ctx->amu);
    if (ctx->astop) { g_err = "Session is not initialized."; return KKX_ERR_STATE; }
    if (!ctx->worker_started) {
      ctx->worker = std::thread(async_worker, ctx);
      ctx->worker_started = true;
    }
    const int64_t t = ctx->next_ticket++;
    ctx->aqueue.push_back(&r->w);
    ctx->tickets[t] = std::move(r);
    *out_ticket = t;
  } catch (const std::exception& e) { g_err = e.what(); return KKX_ERR_CUDA; }
  ctx->acv_work.notify_one();
  return KKX_OK;
}

KKX_API int kkx_poll(kkx_ctx* ctx, kkx_ticket ticket) {
  int rc = check_ctx(ctx);
  if (rc) return rc;
  std::lock_guard<std::mutex> al(ctx->amu);
  auto it = ctx->tickets.find(ticket);
  if (it == ctx->tickets.end() || it->second->taken) { g_err = "unknown ticket"; return KKX_ERR_ARG; }
  return it->second->w.done ? 1 : 0;
}

KKX_API int kkx_wait(kkx_ctx* ctx, kkx_ticket ticket, float** out_audio, int64_t* out_samples, int32_t* out_pred_dur) {
  int rc = check_ctx(ctx);
  if (rc) return rc;
  if (out_audio) *out_audio = nullptr;
  if (out_samples) *out_samples = 0;
  std::unique_ptr<kkx_ctx::AsyncReq> r;
  {
    std::unique_lock<std::mutex> al(ctx->amu);
    auto it = ctx->tickets.find(ticket);
    if (it == ctx->tickets.end() || it->second->taken) { g_err = "unknown ticket"; return KKX_ERR_ARG; }
    it->second->taken = true;                         // a ticket is redeemed once
    kkx_ctx::AsyncReq* p = it->second.get();
    ctx->acv_done.wait(al, [&] { return p->w.done; });
    r = std::move(it->second);
    ctx->tickets.erase(it);
  }
  if (r->w.rc != KKX_OK) { g_err = r->w.err; return r->w.rc; }
  if (out_pred_dur) memcpy(out_pred_dur, r->dur.data(), r->dur.size() * sizeof(int32_t));
  if (out_samples) *out_samples = r->w.samples;
  if (out_audio) *out_audio = r->w.audio; else kkx_release(ctx, r->w.audio);
  return KKX_OK;
}

KKX_API void kkx_release(kkx_ctx* ctx, float* audio) {
  if (!ctx || !audio) return;
  kkx_ctx::Block* b = nullptr;
  {
    std::lock_guard<std::mutex> pl(ctx->pool_mu);
    auto it = ctx->handed.find(audio);
    if (it == ctx->handed.end()) return;
    b = it->second;
    ctx->handed.erase(it);
    if (--b->refs > 0) return;
  }
  recycle_pinned(ctx, b->base, b->cap);
  delete b;
}

KKX_API int kkx_stage_batch(kkx_ctx* ctx, int32_t batch, const int64_t* tokens, const int32_t* tok_offsets,
                    const float* styles, const float* speeds) {
  return session_call(ctx, [&] { ctx->model->stage(batch, tokens, tok_offsets, styles, speeds); });
}

KKX_API int kkx_run_staged(kkx_ctx* ctx, int64_t* out_total_samples, int64_t* out_launches) {
  return session_call(ctx, [&] {
    record_report(ctx, [&](const std::function<void()>& note) {
      ctx->model->run();
      note();
    });
    if (out_total_samples) *out_total_samples = ctx->model->total_samples();
    if (out_launches) *out_launches = ctx->model->stats.launches;
  });
}

KKX_API int kkx_fetch_staged(kkx_ctx* ctx, float* dst_audio, int64_t capacity, int64_t* out_sample_offsets,
                     int32_t* out_pred_dur) {
  return session_call(ctx, [&] { ctx->model->fetch(dst_audio, capacity, out_sample_offsets, out_pred_dur); });
}

// kkx_get_stat's value of `k` (caller holds ctx->mu), -1 for an unknown key
static int64_t session_stat(kkx_ctx* ctx, const std::string& k) {
  if (k == "launches") return ctx->model->stats.launches;
  if (k == "last_frames") return ctx->model->last_frames;
  if (k == "gpu_us") return (int64_t)ctx->model->last_gpu_us;
  if (k == "precision") return ctx->model->opt.precision;
  if (k == "out_rate") return ctx->model->opt.out_rate;
  if (k == "loudness_target") return ctx->model->opt.loudness_target;
  if (k == "true_peak_max") return ctx->model->opt.true_peak_max;
  if (k == "loudness_items") return report_items(ctx, kRepLoudness);
  if (k == "limiter") return ctx->model->opt.limiter;
  if (k == "loudness_report") return ctx->model->opt.loudness_report;
  if (k == "flac_lpc_order") return ctx->model->opt.flac_lpc_order;
  if (k == "limiter_items") return report_items(ctx, kRepLimiter);
  if (k == "graph_replays") return ctx->model->graph_replays;
  if (k == "frame_groups") return (int64_t)ctx->model->group_first().size();
  if (k.rfind("group_first:", 0) == 0) {     // first item of frame group g of the last run
    const long g = atol(k.c_str() + 12);
    const auto& gf = ctx->model->group_first();
    return g >= 0 && g < (long)gf.size() ? gf[g] : -1;
  }
  if (k == "weights_sessions") return (int64_t)ctx->model->weight_sessions();
  if (k == "weights_bytes") return (int64_t)ctx->model->weight_set().device_bytes;
  if (k == "weights_from_onnx") return ctx->model->weight_set().format == "onnx" ? 1 : 0;
  {
    std::lock_guard<std::mutex> ql(ctx->qmu);
    if (k == "coalesced_batches") return ctx->coalesced_batches;
    if (k == "coalesced_requests") return ctx->coalesced_requests;
    if (k == "coalesced_largest") return ctx->coalesced_largest;
  }
  {
    std::lock_guard<std::mutex> al(ctx->amu);
    if (k == "async_batches") return ctx->async_batches;
    if (k == "async_requests") return ctx->async_requests;
  }
  return -1;
}

KKX_API int64_t kkx_get_stat(kkx_ctx* ctx, const char* key) {
  int64_t v = -1;
  session_call(ctx, [&] { if (key) v = session_stat(ctx, key); });
  return v;
}

KKX_API int kkx_set_option(kkx_ctx* ctx, const char* key, int64_t value) {
  return session_call(ctx, [&] {
    if (!key) throw ArgError("null key");
    Options& o = ctx->model->opt;
    const std::string k(key);
    if (k == "precision") { if (value < 0 || value > 1) throw ArgError("precision must be 0 or 1"); o.precision = (int)value; }
    else if (k == "noise_seed") o.noise_seed = (unsigned long long)value;
    else if (k == "max_frames") { if (value < 1) throw ArgError("max_frames must be >= 1"); o.max_frames = (int)value; }
    else if (k == "stft_replicate") o.stft_replicate = value ? 1 : 0;
    else if (k == "latency_graphs") o.latency_graphs = value ? 1 : 0;
    else if (k == "attention_umma") o.attention_umma = value ? 1 : 0;
    else if (k == "lstm_fast_gates") o.lstm_fast_gates = value ? 1 : 0;
    else if (k == "fuse_noise_stats") o.fuse_noise_stats = value ? 1 : 0;
    else if (k == "ups_phase_loop") o.ups_phase_loop = value < 0 ? 0 : value > 3 ? 3 : (int)value;
    else if (k == "split_f16") o.split_f16 = value ? 1 : 0;
    else if (k == "stream_bf16") o.stream_bf16 = value ? 1 : 0;
    else if (k == "fuse_phases") o.fuse_phases = value ? 1 : 0;
    else if (k == "gemm_pair") o.gemm_pair = value ? 1 : 0;
    else if (k == "fuse_planes") o.fuse_planes = value ? 1 : 0;
    else if (k == "conv_pair") o.conv_pair = value ? 1 : 0;
    else if (k == "fork_max_batch") { if (value < 0 || value > 512) throw ArgError("fork_max_batch must be in 0..512"); o.fork_max_batch = (int)value; }
    else if (k == "max_tokens") { if (value < 512) throw ArgError("max_tokens must be >= 512"); ctx->max_tokens = value; }
    else if (k == "coalesce") {
      if (value < 0 || value > kMaxCoalesce) throw ArgError("coalesce must be in 0..512");
      ctx->coalesce_max.store((int)value);
    } else if (k == "coalesce_wait_us") {
      if (value < 0 || value > 1000000) throw ArgError("coalesce_wait_us must be in 0..1000000");
      ctx->coalesce_wait_us.store((int)value);
    } else if (k == "async_batch") {
      if (value < 1 || value > kMaxCoalesce) throw ArgError("async_batch must be in 1..512");
      ctx->async_batch.store((int)value);
    } else if (k == "out_rate") {
      int U = 0, D = 0;
      if (value < 8000 || value > 48000 || !resample_ratio((int)value, &U, &D)) {
        const long long g = value > 0 ? std::gcd<long long>(value, 24000) : 1;
        throw ArgError("out_rate " + std::to_string(value) + " Hz is not supported: out_rate / 24000 reduces to U/D = " +
                       std::to_string(value / g) + "/" + std::to_string(24000 / g) +
                       "; accepted are 8000..48000 Hz with max(U, D) <= 320 (8000, 11025, 12000, 16000, 22050, 24000, "
                       "32000, 44100, 48000)");
      }
      o.out_rate = (int)value;
    } else if (k == "loudness_target") {
      if (value != 0 && (value < -7000 || value > -500))
        throw ArgError("loudness_target " + std::to_string(value) +
                       " is not supported: give 1/100 LUFS in -7000..-500 (e.g. -2300 for -23 LUFS), or 0 for off");
      o.loudness_target = (int)value;
    } else if (k == "true_peak_max") {
      if (value < -2000 || value > 0)
        throw ArgError("true_peak_max " + std::to_string(value) + " is not supported: give 1/100 dBTP in -2000..0");
      o.true_peak_max = (int)value;
    } else if (k == "limiter") {
      if (value != 0 && value != 1)
        throw ArgError("limiter " + std::to_string(value) + " is not supported: give 0 (off) or 1 (on)");
      o.limiter = (int)value;
    } else if (k == "loudness_report") {
      if (value != 0 && value != 1)
        throw ArgError("loudness_report " + std::to_string(value) + " is not supported: give 0 (off) or 1 (on)");
      o.loudness_report = (int)value;
    } else if (k == "flac_lpc_order") {
      if (value < 0 || value > kMaxLpcOrder)
        throw ArgError("flac_lpc_order " + std::to_string(value) +
                       " is not supported: give 0 (off) or an LPC order in 1..12");
      o.flac_lpc_order = (int)value;
    }
    else throw ArgError("unknown option: " + k);
  });
}

// Row group `group` of the last synchronous call's report: per item b, rows row0, row0 + 1, ... into cols[0], cols[1],
// ... (null columns are skipped).  `off`: the error when that call did not produce the group.
static int last_report(kkx_ctx* ctx, int32_t batch, unsigned group, const char* off, int row0,
                       std::initializer_list<float*> cols) {
  return session_call(ctx, [&] {
    if (!ctx->report_valid) throw StateError("no synchronous call has completed on this session");
    if (!(ctx->report_groups & group)) throw StateError(off);
    const int64_t n = (int64_t)(ctx->report.size() / kReportRows);
    if (batch != n)
      throw ArgError("batch " + std::to_string(batch) + " does not match the last call's " + std::to_string(n) + " items");
    int row = row0;
    for (float* c : cols) {
      if (c)
        for (int64_t b = 0; b < n; b++) c[b] = ctx->report[b * kReportRows + row];
      row++;
    }
  });
}

KKX_API int kkx_last_loudness(kkx_ctx* ctx, int32_t batch, float* lufs, float* true_peak_dbtp, float* gain) {
  return last_report(ctx, batch, kRepLoudness,
                     "the last synchronous call ran with loudness normalisation and the loudness report off", 0,
                     {lufs, true_peak_dbtp, gain});
}

KKX_API int kkx_last_limiter(kkx_ctx* ctx, int32_t batch, float* max_reduction_db, float* true_peak_dbtp) {
  return last_report(ctx, batch, kRepLimiter, "the last synchronous call ran with the limiter off", 7,
                     {max_reduction_db, true_peak_dbtp});
}

KKX_API int kkx_last_loudness_range(kkx_ctx* ctx, int32_t batch, float* loudness_range_lu, float* max_momentary_lufs,
                                    float* max_short_term_lufs) {
  return last_report(ctx, batch, kRepRange, "the last synchronous call ran with the loudness report off", 3,
                     {loudness_range_lu, max_momentary_lufs, max_short_term_lufs});
}

KKX_API int kkx_profile_enable(kkx_ctx* ctx, int enable) {
  return session_call(ctx, [&] { ctx->model->stats.profile = enable != 0; });
}

KKX_API int64_t kkx_profile_json(kkx_ctx* ctx, char* buf, int64_t capacity) {
  int64_t len = -1;
  session_call(ctx, [&] {
    std::ostringstream os;
    os << "{\"conv_flops\": " << ctx->model->stats.conv_flops << ", \"arb_flops\": " << ctx->model->stats.arb_flops
       << ", \"arb_bytes\": " << ctx->model->stats.arb_bytes << ", \"gpu_us\": " << ctx->model->last_gpu_us
       << ", \"kernels\": {";
    bool first = true;
    for (auto& kv : ctx->model->prof_) {
      if (!first) os << ", ";
      first = false;
      os << "\"" << kv.first << "\": [" << kv.second.first << ", " << kv.second.second << "]";
    }
    os << "}}";
    const std::string s = os.str();
    if (buf && capacity > 0) {
      const size_t n = std::min<size_t>(s.size(), (size_t)capacity - 1);
      memcpy(buf, s.data(), n);
      buf[n] = 0;
    }
    len = (int64_t)s.size();
  });
  return len;
}

KKX_API int kkx_set_noise(kkx_ctx* ctx, const float* noise, int64_t n) {
  return session_call(ctx, [&] { ctx->model->set_noise(noise, n); });
}

KKX_API int kkx_set_inject_item(kkx_ctx* ctx, int32_t item, const char* name, const void* data, int64_t count) {
  return session_call(ctx, [&] {
    if (!name) throw ArgError("null name");
    ctx->model->set_inject(name, item, count > 0 ? data : nullptr, count);
  });
}

KKX_API int kkx_set_inject(kkx_ctx* ctx, const char* name, const void* data, int64_t count) {
  return kkx_set_inject_item(ctx, 0, name, data, count);
}

KKX_API int kkx_debug_enable(kkx_ctx* ctx, int enable) {
  return session_call(ctx, [&] { ctx->model->set_debug(enable != 0, -1); });
}

KKX_API int kkx_debug_select(kkx_ctx* ctx, int enable, int32_t item) {
  return session_call(ctx, [&] { ctx->model->set_debug(enable != 0, item); });
}

KKX_API int64_t kkx_debug_stage(kkx_ctx* ctx, const char* name, int32_t item, float* dst, int64_t capacity,
                        int64_t* rows, int64_t* cols) {
  int64_t n = -1;
  session_call(ctx, [&] {
    if (!name) return;
    const DebugStage* s = ctx->model->debug_stage(name, item);
    if (!s) { g_err = std::string("no such debug stage: ") + name; return; }
    if (rows) *rows = s->rows;
    if (cols) *cols = s->cols;
    n = (int64_t)s->data.size();
    if (dst && capacity > 0) memcpy(dst, s->data.data(), (size_t)std::min(n, capacity) * sizeof(float));
  });
  return n;
}
