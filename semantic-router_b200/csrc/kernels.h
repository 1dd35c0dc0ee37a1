// Host-callable launchers of the HBM-bound kernels (elementwise.cu), attention (attention.cu) and the
// cache scan (cache_scan.cu).  All pointers are device pointers; all launches are asynchronous on `stream`.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace srb {

// kernel-launch accounting (engine.cu): every launcher below bumps it; bench.py reports it as gpu_launches
void note_launch(int n = 1);
// SRB_PDL=1 turns programmatic dependent launch on for the tcgen05 kernels (measured neutral: default off)
bool pdl_enabled();
long long launches_total();

// ---- attention.cu (mma.sync flash attention: v1 kernel, kept as the comparator for the tcgen05 kernel's tests)
int attention_fwd(cudaStream_t stream, const __half* qkv, __half* out, const int* cu_seqlens, int batch,
                  int max_len, int num_heads, int head_dim, int window);

// ---- attention_tc.cu (tcgen05 / TMEM / TMA flash attention; the production path)
// kv_lens [batch] (optional, global attention only): keys >= kv_lens[b] of sequence b are masked for EVERY query row while
// all rows stay queries -- right-padded sequences whose pads are queries, as candle's BertModel sees them under a
// fixed-padding tokenizer (core/similarity.rs:189-222)
int attention_tc_fwd(cudaStream_t stream, const __half* qkv, __half* out, const int* cu_seqlens, int batch,
                     int total_tokens, int max_len, int num_heads, int head_dim, int window, const int* kv_lens = nullptr);
// One-shot tcgen05 attention for sliding-window layers (window <= 64): a 128-row query tile sees <= 256 keys, so the
// tile is a single score block (no online softmax).  attention_win.cu.
int attention_win_fwd(cudaStream_t stream, const __half* qkv, __half* out, const int* cu_seqlens, int batch,
                      int total_tokens, int max_len, int num_heads, int head_dim, int window);

// debug: device buffer of 3 x 4096 int64 receiving CTA 0's event timeline (nullptr disables)
void attention_tc_set_trace(long long* dev_buf);
void attention_win_set_trace(long long* dev_buf);

// ---- elementwise.cu
// pos[t] = t - cu_seqlens[seq(t)]
int compute_positions(cudaStream_t stream, const int* cu_seqlens, int batch, int* pos);
// ModernBERT embeddings: x = LN_nobias(E[ids]); writes fp32 residual stream and its fp16 copy.
// lo (optional): fp16(x - fp16(x)), the low half of the fp16-pair form of the residual stream; x may be null then
int embed_ln_modernbert(cudaStream_t stream, const int* ids, int T, int H, int vocab, const float* table,
                        const float* ln_w, float eps, float* x, __half* h, __half* lo = nullptr);
// x[r, :] = pivot[r] + hi[r, :] + lo[r, :]  (pivot null: 0)
int hl_to_f32(cudaStream_t stream, const __half* hi, const __half* lo, const float* pivot, int T, int H, float* x);
// BERT embeddings: x = LN(word[id] + pos[p] + type[0]).
int embed_ln_bert(cudaStream_t stream, const int* ids, const int* pos, int T, int H, int vocab, int max_pos,
                  const float* word, const float* pos_emb, const float* type0, const float* ln_w,
                  const float* ln_b, float eps, float* x, __half* h);
// Row LayerNorm of fp32 x[T,H]; optional outputs: y32 (may alias x) and y16.
int layernorm_rows(cudaStream_t stream, const float* x, int T, int H, const float* w, const float* b, float eps,
                   float* y32, __half* y16);
// fp32 -> fp16 row copy
int cast_rows_f16(cudaStream_t stream, const float* x, size_t n, __half* y);

enum PoolMode { POOL_MEAN = 0, POOL_CLS = 1 };
// pooled[b,:] = mean_t / first-token of (optionally LayerNorm'ed) x rows of sequence b.
// `part` [batch, kPoolParts, H] and `arrived` [batch] (zero on entry, zero again on exit) are scratch.
constexpr int kPoolParts = 8;
int pool_rows(cudaStream_t stream, const float* x, const int* cu_seqlens, int batch, int H, PoolMode mode,
              const float* ln_w, const float* ln_b, float eps, float* pooled, float* part, int* arrived,
              const int* div_lens = nullptr);   // div_lens [batch]: divide the sums by these instead of the row counts
// emb[b, :dim] = pooled[b, :dim] / (||pooled[b,:dim]||_2 + norm_eps)
int l2_normalize_rows(cudaStream_t stream, const float* pooled, int batch, int H, int dim, float norm_eps,
                      float* emb);

struct SeqHeadWeights {
  // ModernBERT: dense [H,H] (no bias) -> gelu_tanh -> LN(norm_w, 0, 1e-12); BERT: pooler [H,H]+bias -> tanh
  const float* dense_w = nullptr;
  const float* dense_b = nullptr;
  const float* norm_w = nullptr;
  int dense_mode = 0;  // 0 none, 1 ModernBERT head, 2 BERT pooler y = x @ P^T (+b), 3 BERT pooler y = x @ P (+b)
  const float* cls_w = nullptr;  // [C,H]
  const float* cls_b = nullptr;  // [C]
  int num_classes = 0;
  int argmax_last = 0;  // 0: first max wins (strict > from 0.0), 1: last max wins (max_by)
  // HF/ONNX-export flavour of the ModernBERT head (onnx-binding twin): erf GELU and eps = config.norm_eps
  int gelu_erf = 0;
  float head_eps = 1e-12f;
};
// logits/probs [B,C], cls int32 [B], conf fp32 [B]
int seq_head(cudaStream_t stream, const float* pooled, int batch, int H, const SeqHeadWeights& w, float* logits,
             float* probs, int* cls, float* conf);

// Token head tail: (optional: gelu_tanh + LN(norm_w, 0, 1e-12) of the fp16 dense output) -> classifier ->
// logits/probs [T,C], pred int32 [T] (argmax over logits; first max unless argmax_last), conf [T].
// hidden32 path: optional LayerNorm(pre_ln_w, no bias, pre_ln_eps) first (ModernBERT final_norm).
int token_head(cudaStream_t stream, const float* hidden32, const __half* dense16, int T, int H,
               const float* norm_w, const float* pre_ln_w, float pre_ln_eps, const float* cls_w,
               const float* cls_b, int C, int argmax_last, float* logits, float* probs, int* pred, float* conf,
               int gelu_erf = 0, float head_eps = 1e-12f);

// ---- cache_scan.cu
// scores = Q[B,D] . C[N,D]^T (fp16 operands, fp32 accumulate); per query top-k (descending score, lower
// index wins ties); rows with valid[i]==0 are skipped.  out_idx int32 [B,k] (global id = row + id_offset,
// -1 when fewer than k valid rows), out_score fp32 [B,k].
int cache_topk(cudaStream_t stream, const __half* queries, int B, const __half* cache, const uint8_t* valid,
               int N, int D, int k, int id_offset, int* out_idx, float* out_score, void* workspace,
               size_t workspace_bytes);
size_t cache_topk_workspace_bytes(int B, int N, int k);
// Which pipeline cache_topk runs for (B, N, D, k); cache_topk branches on this and nothing else.
enum CacheTopkRoute {
  CACHE_ROUTE_REFUSED = -1,  // k > 64, or more stage-2 candidates than shared memory holds: error before any launch
  CACHE_ROUTE_NONE = 0,      // B <= 0 or k <= 0: nothing to do
  CACHE_ROUTE_EMPTY = 1,     // N == 0: every slot (-1, -inf)
  CACHE_ROUTE_GEMV = 2,      // B <= 4: scores_small_kernel per chunk, select_stage1, select_stage2
  CACHE_ROUTE_FUSED = 3,     // B > 4, k <= 8: EPI_TOPK GEMM lists, select_stage2
  CACHE_ROUTE_GEMM = 4,      // otherwise: EPI_RESID GEMM scores per chunk, select_stage1, select_stage2
};
struct CacheTopkPlan {
  int route = CACHE_ROUTE_NONE;
  int chunks = 0;          // score chunks of the GEMV / GEMM routes
  int chunk_rows = 0;      // stored rows per chunk (a multiple of the 8192-row stage-1 segment)
  size_t stage2_smem = 0;  // dynamic shared memory of the final select_stage2 (FUSED: its upper bound)
};
CacheTopkPlan cache_topk_plan(int B, int N, int D, int k);
// k-way merge of G per-shard lists [G][B,k] -> [B,k]
int cache_merge_topk(cudaStream_t stream, const int* idx_parts, const float* score_parts, int G, int B, int k,
                     int* out_idx, float* out_score);

// sharded-cache exchange format: 8-byte entries {fp32 score, int32 global id}
int cache_pack_pairs(cudaStream_t stream, const int* idx, const float* score, int n, void* pairs_out);
// merge of G gathered lists in that format, pairs [G][B][k] -> [B,k]
int cache_merge_packed(cudaStream_t stream, const void* pairs, int G, int B, int k, int* out_idx, float* out_score);

}  // namespace srb
