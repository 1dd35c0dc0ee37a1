// Side-door C ABI (include/sr_b200.h): model lifecycle, host-buffer and device-resident entry points,
// unit-op hooks for the parity tests.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/sr_b200_testhooks.h"
#include "common.cuh"
#include "engine.h"
#include "gemm.h"

using namespace srb;

namespace srb {   // cache_api.cu
std::mutex& cache_mutex(sr_cache* c);
int cache_topk_dev_locked(sr_cache* c, const void* d_queries_f16, int b, int k, void* cuda_stream);
}

// A captured forward (+ sequence head) for one launch geometry.  Small calls -- one prompt, the reference's operating
// mode -- are launch-bound (~140 kernels of a few microseconds each); replaying them as a CUDA graph removes the
// per-launch host cost and most of the gaps between kernels.
struct ForwardGraph {
  cudaGraphExec_t exec = nullptr;
  uint64_t ws_gen = 0;            // workspace generation the pointers inside were captured against
  uint64_t last_use = 0;
};
struct sr_model {
  Model* m = nullptr;
  cudaStream_t private_stream = nullptr;
  std::map<uint64_t, ForwardGraph> graphs;   // key: (batch, tokens, max_len, head, pooler_mode, flavour)
  uint64_t tick = 0;
  __half* q16 = nullptr;                     // fp16 copy of the last embeddings for sr_cache_lookup_ids
  size_t q16_elems = 0;
  ~sr_model() {
    for (auto& kv : graphs)
      if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
    if (q16) cudaFree(q16);
  }
};

namespace {
thread_local std::string g_err;
int fail(const std::string& e) {
  g_err = e;
  fprintf(stderr, "[srb200] %s\n", e.c_str());
  return -1;
}
struct DeviceGuard {
  explicit DeviceGuard(int dev) { cudaSetDevice(dev); }
};

// host ids/cu -> pinned -> device; returns T and max_len
int stage_inputs(Model& m, const int32_t* ids, const int32_t* cu, int batch, size_t out_elems_per_row_seq,
                 size_t out_elems_per_row_tok, int* T_out, int* max_len_out) {
  if (batch <= 0 || !ids || !cu) return fail("bad arguments");
  if (cu[0] != 0) return fail("cu_seqlens[0] must be 0");
  int max_len = 0;
  for (int b = 0; b < batch; ++b) {
    const int len = cu[b + 1] - cu[b];
    if (len <= 0) return fail("empty or negative-length sequence in batch");
    max_len = len > max_len ? len : max_len;
  }
  const int T = cu[batch];
  const size_t out_elems = std::max(out_elems_per_row_seq * static_cast<size_t>(batch),
                                    out_elems_per_row_tok * static_cast<size_t>(T));
  if (workspace_reserve(m, T, batch, out_elems)) return fail("workspace allocation failed");
  Workspace& w = m.ws;
  memcpy(w.h_ids, ids, sizeof(int32_t) * T);
  memcpy(w.h_cu, cu, sizeof(int32_t) * (batch + 1));
  if (cudaMemcpyAsync(w.ids, w.h_ids, sizeof(int32_t) * T, cudaMemcpyHostToDevice, m.stream) != cudaSuccess ||
      cudaMemcpyAsync(w.cu, w.h_cu, sizeof(int32_t) * (batch + 1), cudaMemcpyHostToDevice, m.stream) != cudaSuccess)
    return fail("H2D copy failed");
  *T_out = T;
  *max_len_out = max_len;
  return 0;
}

// SRB_GRAPHS=0 disables the replay (A/B measurements)
bool graphs_enabled() {
  static const bool on = [] {
    const char* e = getenv("SRB_GRAPHS");
    return !(e && e[0] == '0');
  }();
  return on;
}
constexpr int kGraphMaxTokens = 2048;   // beyond this the kernels are long enough to hide their launches
constexpr size_t kGraphCacheCap = 96;

// Runs `eager` (a fixed launch sequence on m.stream for the geometry `key` names) through the graph cache.  Anything
// that goes wrong while capturing falls back to plain launches.
template <typename Fn>
int run_graphed(sr_model* h, uint64_t key, bool eligible, Fn&& eager) {
  Model& m = *h->m;
  Workspace& w = m.ws;
  if (!eligible || !graphs_enabled() || m.prof.on || m.precise.on || m.stream != h->private_stream) return eager();
  auto it = h->graphs.find(key);
  if (it != h->graphs.end() && it->second.ws_gen != w.generation) {   // a workspace buffer was reallocated
    cudaGraphExecDestroy(it->second.exec);
    h->graphs.erase(it);
    it = h->graphs.end();
  }
  if (it == h->graphs.end()) {
    if (h->graphs.size() >= kGraphCacheCap) {   // evict the least recently used geometry
      auto old = h->graphs.begin();
      for (auto j = h->graphs.begin(); j != h->graphs.end(); ++j)
        if (j->second.last_use < old->second.last_use) old = j;
      cudaGraphExecDestroy(old->second.exec);
      h->graphs.erase(old);
    }
    // run once eagerly first: lazy one-time setup (function attributes, entry points) must not happen under capture
    if (eager()) return -1;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    if (cudaStreamBeginCapture(m.stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return 0; }
    const int rc = eager();
    const cudaError_t ce = cudaStreamEndCapture(m.stream, &graph);
    if (rc != 0 || ce != cudaSuccess || !graph || cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
      cudaGetLastError();
      if (graph) cudaGraphDestroy(graph);
      return 0;   // the eager pass above already produced this call's results
    }
    cudaGraphDestroy(graph);
    ForwardGraph fg;
    fg.exec = exec;
    fg.ws_gen = w.generation;
    fg.last_use = ++h->tick;
    h->graphs[key] = fg;
    return 0;       // results of the eager pass stand
  }
  it->second.last_use = ++h->tick;
  if (cudaGraphLaunch(it->second.exec, m.stream) != cudaSuccess) {
    cudaGetLastError();
    return eager();
  }
  return 0;
}

// encoder_forward + head_sequence for a small call
int forward_and_head(sr_model* h, int head, int batch, int T, int max_len, int pooler_mode) {
  Model& m = *h->m;
  Workspace& w = m.ws;
  auto eager = [&]() {
    if (encoder_forward(m, w.ids, w.cu, batch, T, max_len, 0)) return fail("encoder_forward failed");
    if (head_sequence(m, head, w.cu, batch, pooler_mode)) return fail("head_sequence failed");
    return 0;
  };
  const uint64_t key = (static_cast<uint64_t>(batch) << 48) ^ (static_cast<uint64_t>(T) << 28) ^
                       (static_cast<uint64_t>(max_len) << 12) ^ (static_cast<uint64_t>(head) << 4) ^
                       (static_cast<uint64_t>(pooler_mode) << 1) ^ static_cast<uint64_t>(m.head_flavor);
  return run_graphed(h, key, T <= kGraphMaxTokens && batch <= 64, eager);
}

int finish(Model& m) {
  const cudaError_t e = cudaStreamSynchronize(m.stream);
  if (e != cudaSuccess) return fail(std::string("CUDA failure: ") + cudaGetErrorString(e));
  return 0;
}
}  // namespace

extern "C" {

const char* sr_last_error(void) { return g_err.c_str(); }

int sr_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int sr_model_load(const char* model_dir, int device, sr_model** out) {
  if (!model_dir || !out) return fail("bad arguments");
  std::string err;
  Model* m = model_load(model_dir, device, &err);
  if (!m) return fail("sr_model_load(" + std::string(model_dir) + "): " + err);
  sr_model* h = new sr_model();
  h->m = m;
  h->private_stream = m->stream;
  *out = h;
  return 0;
}

int sr_model_add_head(sr_model* h, const char* model_dir, int token_level) {
  if (!h || !model_dir) return fail("bad arguments");
  std::lock_guard<std::mutex> lk(h->m->mu);
  std::string err;
  const int id = model_add_head(h->m, model_dir, token_level, &err);
  if (id < 0) return fail("sr_model_add_head: " + err);
  return id;
}

void sr_model_free(sr_model* h) {
  if (!h) return;
  h->m->stream = h->private_stream;
  model_free(h->m);
  delete h;
}

int sr_model_info(const sr_model* h, sr_model_info_t* out) {
  if (!h || !out) return -1;
  const EncoderConfig& c = h->m->cfg;
  out->arch = c.arch; out->hidden = c.H; out->layers = c.L; out->heads = c.heads; out->intermediate = c.I;
  out->vocab = c.vocab; out->max_pos = c.max_pos; out->num_heads_loaded = static_cast<int>(h->m->heads.size());
  out->device = h->m->device;
  return 0;
}

int sr_head_num_classes(const sr_model* h, int head) {
  if (!h || head < 0 || head >= static_cast<int>(h->m->heads.size())) return -1;
  return h->m->heads[head].num_classes;
}

int sr_classify_ids(sr_model* h, int head, const int32_t* ids, const int32_t* cu, int batch, int pooler_mode,
                    float* probs, float* logits, int32_t* cls, float* conf) {
  if (!h) return fail("null model");
  Model& m = *h->m;
  if (head < 0 || head >= static_cast<int>(m.heads.size())) return fail("no such head");
  std::lock_guard<std::mutex> lk(m.mu);
  DeviceGuard dg(m.device);
  const int C = m.heads[head].num_classes;
  int T, max_len;
  if (stage_inputs(m, ids, cu, batch, C, 0, &T, &max_len)) return -1;
  Workspace& w = m.ws;
  if (forward_and_head(h, head, batch, T, max_len, pooler_mode)) return -1;
  const size_t n = static_cast<size_t>(batch) * C;
  if (probs) cudaMemcpyAsync(w.h_out, w.probs, n * 4, cudaMemcpyDeviceToHost, m.stream);
  if (logits) cudaMemcpyAsync(w.h_out + w.h_out_elems, w.logits, n * 4, cudaMemcpyDeviceToHost, m.stream);
  cudaMemcpyAsync(w.h_cls, w.cls, sizeof(int) * batch, cudaMemcpyDeviceToHost, m.stream);
  cudaMemcpyAsync(w.h_conf, w.conf, sizeof(float) * batch, cudaMemcpyDeviceToHost, m.stream);
  if (finish(m)) return -1;
  if (probs) memcpy(probs, w.h_out, n * 4);
  if (logits) memcpy(logits, w.h_out + w.h_out_elems, n * 4);
  if (cls) memcpy(cls, w.h_cls, sizeof(int) * batch);
  if (conf) memcpy(conf, w.h_conf, sizeof(float) * batch);
  return 0;
}

int sr_classify_tokens_ids(sr_model* h, int head, const int32_t* ids, const int32_t* cu, int batch, float* probs,
                           float* logits, int32_t* pred, float* conf) {
  if (!h) return fail("null model");
  Model& m = *h->m;
  if (head < 0 || head >= static_cast<int>(m.heads.size())) return fail("no such head");
  std::lock_guard<std::mutex> lk(m.mu);
  DeviceGuard dg(m.device);
  const int C = m.heads[head].num_classes;
  int T, max_len;
  if (stage_inputs(m, ids, cu, batch, 0, C, &T, &max_len)) return -1;
  Workspace& w = m.ws;
  if (encoder_forward(m, w.ids, w.cu, batch, T, max_len, 0)) return fail("encoder_forward failed");
  if (head_tokens(m, head, batch, T)) return fail("head_tokens failed");
  const size_t n = static_cast<size_t>(T) * C;
  if (probs) cudaMemcpyAsync(w.h_out, w.probs, n * 4, cudaMemcpyDeviceToHost, m.stream);
  if (logits) cudaMemcpyAsync(w.h_out + w.h_out_elems, w.logits, n * 4, cudaMemcpyDeviceToHost, m.stream);
  cudaMemcpyAsync(w.h_cls, w.cls, sizeof(int) * T, cudaMemcpyDeviceToHost, m.stream);
  cudaMemcpyAsync(w.h_conf, w.conf, sizeof(float) * T, cudaMemcpyDeviceToHost, m.stream);
  if (finish(m)) return -1;
  if (probs) memcpy(probs, w.h_out, n * 4);
  if (logits) memcpy(logits, w.h_out + w.h_out_elems, n * 4);
  if (pred) memcpy(pred, w.h_cls, sizeof(int) * T);
  if (conf) memcpy(conf, w.h_conf, sizeof(float) * T);
  return 0;
}

int sr_embed_ids(sr_model* h, const int32_t* ids, const int32_t* cu, int batch, int target_layer, int target_dim,
                 float* emb) {
  if (!h || !emb) return fail("bad arguments");
  Model& m = *h->m;
  std::lock_guard<std::mutex> lk(m.mu);
  DeviceGuard dg(m.device);
  const int H = m.cfg.H;
  if (target_layer > m.cfg.L) return fail("target_layer exceeds num_hidden_layers");
  if (target_dim > H) return fail("target_dim exceeds hidden_size");
  const int dim = target_dim <= 0 ? H : target_dim;
  int T, max_len;
  if (stage_inputs(m, ids, cu, batch, 0, 0, &T, &max_len)) return -1;
  Workspace& w = m.ws;
  if (encoder_forward(m, w.ids, w.cu, batch, T, max_len, target_layer)) return fail("encoder_forward failed");
  // mmBERT: +1e-12 on the norm (mmbert_embedding.rs:781-796); BERT similarity: none (similarity.rs:338-341)
  if (head_embedding(m, w.cu, batch, dim, m.cfg.arch == ARCH_MODERNBERT ? 1e-12f : 0.f)) return fail("embedding head failed");
  const size_t n = static_cast<size_t>(batch) * dim;
  cudaMemcpyAsync(w.h_out, w.emb, n * 4, cudaMemcpyDeviceToHost, m.stream);
  if (finish(m)) return -1;
  memcpy(emb, w.h_out, n * 4);
  return 0;
}

int sr_embed_ids_padded(sr_model* h, const int32_t* ids, const int32_t* cu, const int32_t* real_lens, int batch, float* emb) {
  if (!h || !emb || !real_lens) return fail("bad arguments");
  Model& m = *h->m;
  if (m.cfg.arch != ARCH_BERT) return fail("sr_embed_ids_padded: BERT-family similarity models only");
  std::lock_guard<std::mutex> lk(m.mu);
  DeviceGuard dg(m.device);
  int T, max_len;
  if (stage_inputs(m, ids, cu, batch, 0, 0, &T, &max_len)) return -1;
  for (int b = 0; b < batch; ++b)
    if (real_lens[b] <= 0 || real_lens[b] > cu[b + 1] - cu[b]) return fail("real_lens[b] must be in 1..len(b)");
  Workspace& w = m.ws;
  if (cudaMemcpyAsync(w.kv_lens, real_lens, sizeof(int32_t) * batch, cudaMemcpyHostToDevice, m.stream) != cudaSuccess)
    return fail("H2D copy failed");
  m.cur_kv_lens = w.kv_lens;
  const int rc_f = encoder_forward(m, w.ids, w.cu, batch, T, max_len, 0);
  const int rc_h = rc_f ? -1 : head_embedding(m, w.cu, batch, m.cfg.H, 0.f);
  m.cur_kv_lens = nullptr;
  if (rc_f) return fail("encoder_forward failed");
  if (rc_h) return fail("embedding head failed");
  const size_t n = static_cast<size_t>(batch) * m.cfg.H;
  cudaMemcpyAsync(w.h_out, w.emb, n * 4, cudaMemcpyDeviceToHost, m.stream);
  if (finish(m)) return -1;
  memcpy(emb, w.h_out, n * 4);
  return 0;
}

int sr_cache_lookup_ids(sr_model* h, sr_cache* c, const int32_t* ids, const int32_t* cu, int batch, int target_layer, int k,
                        int32_t* out_idx, float* out_score) {
  if (!h || !c || !out_idx || !out_score || k <= 0) return fail("bad arguments");
  Model& m = *h->m;
  std::lock_guard<std::mutex> lk(m.mu);
  // lock order: model, then cache.  Held until the result copies have landed: d_idx / d_score / the scan workspace belong
  // to the cache and another thread's sr_cache_topk / sr_cache_add on it must not touch them meanwhile.
  std::lock_guard<std::mutex> lkc(cache_mutex(c));
  DeviceGuard dg(m.device);
  const int dim = sr_cache_dim(c);
  if (dim <= 0 || dim > m.cfg.H) return fail("cache dimension exceeds hidden_size");
  if (target_layer > m.cfg.L) return fail("target_layer exceeds num_hidden_layers");
  int T, max_len;
  if (stage_inputs(m, ids, cu, batch, 0, 0, &T, &max_len)) return -1;
  Workspace& w = m.ws;
  if (encoder_forward(m, w.ids, w.cu, batch, T, max_len, target_layer)) return fail("encoder_forward failed");
  if (head_embedding(m, w.cu, batch, dim, m.cfg.arch == ARCH_MODERNBERT ? 1e-12f : 0.f)) return fail("embedding head failed");
  const size_t n = static_cast<size_t>(batch) * dim;
  if (n > h->q16_elems) {
    if (h->q16) cudaFree(h->q16);
    h->q16 = nullptr; h->q16_elems = 0;
    if (cudaMalloc(reinterpret_cast<void**>(&h->q16), n * 2) != cudaSuccess) return fail("allocation failed");
    h->q16_elems = n;
  }
  if (cast_rows_f16(m.stream, w.emb, n, h->q16)) return fail("cast failed");
  if (cache_topk_dev_locked(c, h->q16, batch, k, m.stream)) return fail("cache scan failed");
  cudaMemcpyAsync(out_idx, sr_cache_dev_idx(c), static_cast<size_t>(batch) * k * 4, cudaMemcpyDeviceToHost, m.stream);
  cudaMemcpyAsync(out_score, sr_cache_dev_score(c), static_cast<size_t>(batch) * k * 4, cudaMemcpyDeviceToHost, m.stream);
  return finish(m);
}

int sr_classify_multi_ids(sr_model* h, const int* heads, int n_heads, const int32_t* ids, const int32_t* cu,
                          int batch, float** probs_out, int32_t** cls_out) {
  if (!h || !heads || n_heads <= 0) return fail("bad arguments");
  Model& m = *h->m;
  std::lock_guard<std::mutex> lk(m.mu);
  DeviceGuard dg(m.device);
  size_t cseq = 0, ctok = 0;
  for (int i = 0; i < n_heads; ++i) {
    if (heads[i] < 0 || heads[i] >= static_cast<int>(m.heads.size())) return fail("no such head");
    const Head& hd = m.heads[heads[i]];
    if (hd.token_level) ctok = std::max<size_t>(ctok, hd.num_classes);
    else cseq = std::max<size_t>(cseq, hd.num_classes);
  }
  int T, max_len;
  if (stage_inputs(m, ids, cu, batch, cseq, ctok, &T, &max_len)) return -1;
  Workspace& w = m.ws;
  if (encoder_forward(m, w.ids, w.cu, batch, T, max_len, 0)) return fail("encoder_forward failed");
  for (int i = 0; i < n_heads; ++i) {
    const Head& hd = m.heads[heads[i]];
    const size_t rows = hd.token_level ? T : batch;
    if (hd.token_level ? head_tokens(m, heads[i], batch, T) : head_sequence(m, heads[i], w.cu, batch, 0))
      return fail("head failed");
    const size_t n = rows * hd.num_classes;
    if (probs_out && probs_out[i]) cudaMemcpyAsync(w.h_out, w.probs, n * 4, cudaMemcpyDeviceToHost, m.stream);
    cudaMemcpyAsync(w.h_cls, w.cls, sizeof(int) * rows, cudaMemcpyDeviceToHost, m.stream);
    if (finish(m)) return -1;
    if (probs_out && probs_out[i]) memcpy(probs_out[i], w.h_out, n * 4);
    if (cls_out && cls_out[i]) memcpy(cls_out[i], w.h_cls, sizeof(int) * rows);
  }
  return 0;
}

// ---- shared-base multi-task pass over unmerged LoRA checkpoints (engine.h: LoraShared) --------------------------------
int sr_model_load_lora_shared(const char* const* task_dirs, const int* token_level, int n_tasks, int mode, int device, sr_model** out) {
  if (!task_dirs || n_tasks <= 0 || n_tasks > 8 || !out || mode < 0 || mode > 1) return fail("bad arguments");
  std::vector<std::string> dirs;
  std::vector<int> tl;
  for (int t = 0; t < n_tasks; ++t) {
    if (!task_dirs[t]) return fail("bad arguments");
    dirs.push_back(task_dirs[t]);
    tl.push_back(token_level ? token_level[t] : -1);
  }
  std::string err;
  Model* m = model_load_lora_shared(dirs, tl, device, mode == SR_LORA_GROUPED, &err);
  if (!m) return fail("sr_model_load_lora_shared: " + err);
  sr_model* h = new sr_model();
  h->m = m;
  h->private_stream = m->stream;
  *out = h;
  return 0;
}

int sr_checkpoint_has_adapters(const char* model_dir) { return model_dir ? checkpoint_has_adapters(model_dir) : -1; }

int sr_lora_shared_tasks(const sr_model* h) { return h ? h->m->lora.tasks : -1; }
int sr_lora_shared_mode(const sr_model* h) { return h && h->m->lora.tasks > 0 ? (h->m->lora.grouped ? SR_LORA_GROUPED : SR_LORA_LOWRANK) : -1; }

int sr_classify_lora_shared_ids(sr_model* h, const int32_t* ids, const int32_t* cu, int batch, int pooler_mode,
                                float** probs_out, int32_t** cls_out, float** conf_out) {
  if (!h) return fail("null model");
  Model& m = *h->m;
  const int nt = m.lora.tasks;
  if (nt <= 0) return fail("not a shared-LoRA model");
  if (batch <= 0 || !ids || !cu || cu[0] != 0) return fail("bad arguments");
  std::lock_guard<std::mutex> lk(m.mu);
  DeviceGuard dg(m.device);
  if (m.precise.on) return fail("the precise path serves merged weights only");
  const int T1 = cu[batch];
  if (T1 <= 0 || static_cast<long long>(T1) * nt > (1ll << 30)) return fail("bad arguments");
  // the batch once per task, task-major: rows [t * T1p, t * T1p + T1) run with task t's adapters.  The grouped form pads every
  // copy to whole 256-row GEMM blocks (a block multiplies ONE task's matrices); the pad rows form one extra sequence per copy
  // that runs through the encoder and is read by nobody.
  const bool grouped = m.lora.grouped;
  const int T1p = grouped ? (T1 + 255) / 256 * 256 : T1;
  const int pad = T1p - T1;
  const int Bp = batch + (pad > 0 ? 1 : 0);
  std::vector<int32_t> rids(static_cast<size_t>(T1p) * nt, 0), rcu(static_cast<size_t>(Bp) * nt + 1);
  for (int t = 0; t < nt; ++t) {
    memcpy(rids.data() + static_cast<size_t>(t) * T1p, ids, sizeof(int32_t) * T1);
    for (int b = 0; b <= batch; ++b) rcu[static_cast<size_t>(t) * Bp + b] = t * T1p + cu[b];
  }
  rcu[static_cast<size_t>(Bp) * nt] = nt * T1p;
  size_t cseq = 0, ctok = 0;
  for (int t = 0; t < nt; ++t) {
    const Head& hd = m.heads[m.lora.head_of_task[t]];
    if (hd.token_level) ctok = std::max<size_t>(ctok, hd.num_classes);
    else cseq = std::max<size_t>(cseq, hd.num_classes);
  }
  int T, max_len;
  if (stage_inputs(m, rids.data(), rcu.data(), Bp * nt, cseq, ctok, &T, &max_len)) return -1;
  Workspace& w = m.ws;
  m.lora.rows_per_task = T1p;
  const uint64_t key = (1ull << 63) ^ (static_cast<uint64_t>(batch) << 48) ^ (static_cast<uint64_t>(T1) << 28) ^
                       (static_cast<uint64_t>(max_len) << 12);
  const int rc = run_graphed(h, key, T <= kGraphMaxTokens && Bp * nt <= 64, [&]() {
    return encoder_forward(m, w.ids, w.cu, Bp * nt, T, max_len, 0) ? fail("encoder_forward failed") : 0;
  });
  m.lora.rows_per_task = 0;
  if (rc) return -1;
  for (int t = 0; t < nt; ++t) {
    const int head = m.lora.head_of_task[t];
    const Head& hd = m.heads[head];
    const size_t rows = hd.token_level ? T1 : batch;
    if (hd.token_level ? head_tokens(m, head, batch, T1, t * T1p) : head_sequence(m, head, w.cu + static_cast<size_t>(t) * Bp, batch, pooler_mode))
      return fail("head failed");
    const size_t n = rows * hd.num_classes;
    if (probs_out && probs_out[t]) cudaMemcpyAsync(w.h_out, w.probs, n * 4, cudaMemcpyDeviceToHost, m.stream);
    cudaMemcpyAsync(w.h_cls, w.cls, sizeof(int) * rows, cudaMemcpyDeviceToHost, m.stream);
    cudaMemcpyAsync(w.h_conf, w.conf, sizeof(float) * rows, cudaMemcpyDeviceToHost, m.stream);
    if (finish(m)) return -1;
    if (probs_out && probs_out[t]) memcpy(probs_out[t], w.h_out, n * 4);
    if (cls_out && cls_out[t]) memcpy(cls_out[t], w.h_cls, sizeof(int) * rows);
    if (conf_out && conf_out[t]) memcpy(conf_out[t], w.h_conf, sizeof(float) * rows);
  }
  return 0;
}

int sr_model_set_precise(sr_model* h, int on) {
  if (!h) return fail("null model");
  std::lock_guard<std::mutex> lk(h->m->mu);
  DeviceGuard dg(h->m->device);
  if (on && h->m->lora.tasks > 0) return fail("sr_model_set_precise: shared-LoRA models have no precise form (load the tasks as separate slots)");
  if (on) {
    std::string err;
    if (precise_prepare(*h->m, &err)) return fail("sr_model_set_precise: " + err);
  }
  cudaStreamSynchronize(h->m->stream);
  h->m->precise.on = on != 0;
  return 0;
}

int sr_model_set_head_flavor(sr_model* h, int flavor) {
  if (!h || flavor < 0 || flavor > 1) return -1;
  std::lock_guard<std::mutex> lk(h->m->mu);
  h->m->head_flavor = flavor;
  return 0;
}

// ---- device-resident entries -------------------------------------------------------------------------
int sr_model_set_stream(sr_model* h, void* stream) {
  if (!h) return -1;
  std::lock_guard<std::mutex> lk(h->m->mu);
  cudaStreamSynchronize(h->m->stream);
  h->m->stream = stream ? static_cast<cudaStream_t>(stream) : h->private_stream;
  return 0;
}
int sr_reserve(sr_model* h, int total_tokens, int batch, int max_classes_rows) {
  if (!h) return -1;
  DeviceGuard dg(h->m->device);
  return workspace_reserve(*h->m, total_tokens, batch, static_cast<size_t>(max_classes_rows));
}
int sr_forward_dev(sr_model* h, const int32_t* d_ids, const int32_t* d_cu, int batch, int total_tokens, int max_len,
                   int num_layers) {
  if (!h) return -1;
  DeviceGuard dg(h->m->device);
  return encoder_forward(*h->m, d_ids, d_cu, batch, total_tokens, max_len, num_layers);
}
int sr_head_seq_dev(sr_model* h, int head, const int32_t* d_cu, int batch, int pooler_mode) {
  if (!h) return -1;
  return head_sequence(*h->m, head, d_cu, batch, pooler_mode);
}
int sr_head_tokens_dev(sr_model* h, int head, int batch, int total_tokens) {
  if (!h) return -1;
  return head_tokens(*h->m, head, batch, total_tokens);
}
int sr_head_embed_dev(sr_model* h, const int32_t* d_cu, int batch, int dim) {
  if (!h) return -1;
  return head_embedding(*h->m, d_cu, batch, dim, h->m->cfg.arch == ARCH_MODERNBERT ? 1e-12f : 0.f);
}
int sr_sync(sr_model* h) {
  if (!h) return -1;
  return finish(*h->m);
}
int sr_profile_enable(sr_model* h, int on) {
  if (!h) return -1;
  cudaStreamSynchronize(h->m->stream);
  profile_enable(*h->m, on != 0);
  return 0;
}
int sr_profile_read(sr_model* h, float* ms8, int* count8) {
  if (!h || !ms8 || !count8) return -1;
  if (profile_collect(*h->m)) return -1;
  for (int i = 0; i < PC_COUNT; ++i) { ms8[i] = h->m->prof.ms[i]; count8[i] = h->m->prof.count[i]; }
  return 0;
}
long long sr_launch_count(void) { return launches_total(); }
const float* sr_dev_probs(const sr_model* h) { return h ? h->m->ws.probs : nullptr; }
const float* sr_dev_logits(const sr_model* h) { return h ? h->m->ws.logits : nullptr; }
const int32_t* sr_dev_cls(const sr_model* h) { return h ? h->m->ws.cls : nullptr; }
const float* sr_dev_conf(const sr_model* h) { return h ? h->m->ws.conf : nullptr; }
const float* sr_dev_emb(const sr_model* h) { return h ? h->m->ws.emb : nullptr; }
const float* sr_dev_hidden(const sr_model* h) { return h ? h->m->ws.x : nullptr; }

#ifdef SRB_TEST_HOOKS
// ---- unit-op hooks ---------------------------------------------------------------------------------------
int sr_test_gemm(const void* a, const void* w, void* out, int m, int n, int k, int epi, int ldo, const float* bias,
                 const float* resid, const int32_t* pos, const float* rope_cos, const float* rope_sin, int rope_cols) {
  GemmDesc g;
  g.M = m; g.N = n; g.K = k; g.A = a; g.W = w; g.out = out; g.ldo = ldo;
  g.epi = static_cast<GemmEpilogue>(epi);
  g.bias = bias; g.resid = resid; g.ldr = ldo; g.pos = pos; g.rope_cos = rope_cos; g.rope_sin = rope_sin;
  g.rope_cols = rope_cols;
  return gemm_f16(nullptr, g);
}
int sr_test_gemm_fold(const void* a, const void* w, void* out, int m, int n, int k, int epi, int ldo, const float* bias,
                      const float* resid, const int32_t* pos, const float* rope_cos, const float* rope_sin, int rope_cols,
                      float* row_stats, void* raw16, const float* fold_stats, float fold_eps, int fold_h, float* pivot_out,
                      const float* pivot_in, const float* pivot_in_stats) {
  GemmDesc g;
  g.M = m; g.N = n; g.K = k; g.A = a; g.W = w; g.out = out; g.ldo = ldo;
  g.epi = static_cast<GemmEpilogue>(epi);
  g.bias = bias; g.resid = resid; g.ldr = ldo; g.pos = pos; g.rope_cos = rope_cos; g.rope_sin = rope_sin;
  g.rope_cols = rope_cols;
  g.row_stats = row_stats; g.raw16 = raw16;
  g.fold_stats = fold_stats; g.fold_eps = fold_eps; g.fold_h = fold_h;
  g.pivot_out = pivot_out; g.pivot_in = pivot_in; g.pivot_in_stats = pivot_in_stats;
  return gemm_f16(nullptr, g);
}
int sr_test_gemm_resid_hl(const void* a, const void* w, void* hi, void* lo, int m, int n, int k, const float* bias, float* row_stats,
                          float* pivot_out, const float* pivot_in, const float* pivot_in_stats) {
  GemmDesc g;
  g.M = m; g.N = n; g.K = k; g.A = a; g.W = w; g.out = hi; g.lo16 = lo; g.ldo = n;
  g.epi = EPI_RESID_HL;
  g.bias = bias; g.row_stats = row_stats;
  g.pivot_out = pivot_out; g.pivot_in = pivot_in; g.pivot_in_stats = pivot_in_stats;
  return gemm_f16(nullptr, g);
}
int sr_test_hl_to_f32(const void* hi, const void* lo, const float* pivot, int t, int hdim, float* x) {
  return hl_to_f32(nullptr, static_cast<const __half*>(hi), static_cast<const __half*>(lo), pivot, t, hdim, x);
}
int sr_test_attention(const void* qkv, void* out, const int32_t* cu, int batch, int max_len, int num_heads, int window) {
  return attention_fwd(nullptr, static_cast<const __half*>(qkv), static_cast<__half*>(out), cu, batch, max_len,
                       num_heads, 64, window);
}
int sr_test_attention_tc(const void* qkv, void* out, const int32_t* cu, int batch, int total_tokens, int max_len,
                         int num_heads, int window) {
  return attention_tc_fwd(nullptr, static_cast<const __half*>(qkv), static_cast<__half*>(out), cu, batch, total_tokens,
                          max_len, num_heads, 64, window);
}
int sr_test_attention_win(const void* qkv, void* out, const int32_t* cu, int batch, int total_tokens, int max_len,
                          int num_heads, int window) {
  return attention_win_fwd(nullptr, static_cast<const __half*>(qkv), static_cast<__half*>(out), cu, batch, total_tokens,
                           max_len, num_heads, 64, window);
}
int sr_test_attention_trace(void* dev_buf_3x4096_i64) {
  attention_tc_set_trace(static_cast<long long*>(dev_buf_3x4096_i64));
  attention_win_set_trace(static_cast<long long*>(dev_buf_3x4096_i64));
  return 0;
}
int sr_test_layernorm(const float* x, int t, int hdim, const float* w, const float* b, float eps, float* y32, void* y16) {
  return layernorm_rows(nullptr, x, t, hdim, w, b, eps, y32, static_cast<__half*>(y16));
}
int sr_test_cache_topk_plan(int b, int n, int d, int k, int32_t* route, int32_t* chunks, int32_t* chunk_rows,
                            int64_t* stage2_smem) {
  if (!route || !chunks || !chunk_rows || !stage2_smem) return -1;
  const CacheTopkPlan p = cache_topk_plan(b, n, d, k);
  *route = p.route;
  *chunks = p.chunks;
  *chunk_rows = p.chunk_rows;
  *stage2_smem = static_cast<int64_t>(p.stage2_smem);
  return 0;
}

#endif  // SRB_TEST_HOOKS

}  // extern "C"
