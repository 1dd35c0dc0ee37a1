/* sr_b200_testhooks.h -- hooks for the parity tests and profiling tools.  NOT exported by the product libraries
 * (lib/libcandle_semantic_router.so, lib/libonnx_semantic_router.so): the same objects plus these entry points are linked
 * into lib/lib{candle,onnx}_semantic_router_testhooks.so (built with -DSRB_TEST_HOOKS), which only tests/ and tools/ load.
 */
#ifndef SR_B200_TESTHOOKS_H
#define SR_B200_TESTHOOKS_H
#include "sr_b200.h"
#ifdef __cplusplus
extern "C" {
#endif

/* ---- host-logic test hooks (no GPU): the span logic the text ABI runs after the token classifiers ------------ */
/* BIO decoding of per-token predictions (offsets [n,2] = byte spans, (0,0) = special token).  In
 * libcandle_semantic_router: traditional/modernbert.rs:1478-1567; in libonnx_semantic_router:
 * mmbert_classifier.rs:952-1050 (other I- handling, spans clipped at text_len).  labels[i] = name of class i.
 * Writes up to cap entities and their types as "TYPE\n..." into types_out; returns the entity count. */
SR_API int sr_test_bio_decode(const int32_t* pred, const float* conf, const int32_t* offsets, int n, const char* const* labels,
                       int n_labels, int text_len, int32_t* ent_start, int32_t* ent_end, float* ent_conf, char* types_out,
                       int types_cap, int cap);
/* detect_hallucinations after the token classifier (ffi/classify.rs:1536-1660); -1 in the ONNX library. */
SR_API int sr_test_hallucination_spans(const int32_t* pred, const float* conf, const int32_t* offsets, int n, int answer_start,
                                int answer_len, float threshold, int32_t* span_start, int32_t* span_end, float* span_conf,
                                int cap, int* has_hallucination, float* overall_confidence);

/* ---- unit-op hooks for the parity tests (device pointers, legacy default stream) --------------------- */
SR_API int sr_test_gemm(const void* a_f16, const void* w_f16, void* out, int m, int n, int k, int epi, int ldo,
                 const float* bias, const float* resid, const int32_t* pos, const float* rope_cos,
                 const float* rope_sin, int rope_cols);
/* sr_test_gemm plus the LayerNorm-fold operands (gemm.h): EPI_RESID may emit per-row (sum, sum of squares) partials
 * row_stats [n/128][m][2] and raw16 = fp16(out); EPI_ROPE / EPI_GEGLU (weights: W diag(gamma) with zero-sum rows) scale
 * the accumulator rows by the rstd computed from fold_stats over rows of length fold_h.  pivot_*: row pivots (gemm.h). */
SR_API int sr_test_gemm_fold(const void* a_f16, const void* w_f16, void* out, int m, int n, int k, int epi, int ldo,
                             const float* bias, const float* resid, const int32_t* pos, const float* rope_cos,
                             const float* rope_sin, int rope_cols, float* row_stats, void* raw16_f16,
                             const float* fold_stats, float fold_eps, int fold_h, float* pivot_out, const float* pivot_in,
                             const float* pivot_in_stats);
/* EPI_RESID_HL (gemm.h): the residual stream as an fp16 pair, in place.  (hi + lo) holds x - pivot_in; after the call it holds
 * x + a w^T (+bias) - pivot_out with pivot_out = pivot_in + (row mean of the old pair, from pivot_in_stats; 0 without), and
 * row_stats [n/128][m][2] the (sum, sum of squares) partials of the new pair. */
SR_API int sr_test_gemm_resid_hl(const void* a_f16, const void* w_f16, void* hi_f16, void* lo_f16, int m, int n, int k,
                                 const float* bias, float* row_stats, float* pivot_out, const float* pivot_in,
                                 const float* pivot_in_stats);
SR_API int sr_test_hl_to_f32(const void* hi_f16, const void* lo_f16, const float* pivot, int t, int hdim, float* x);
SR_API int sr_test_attention(const void* qkv_f16, void* out_f16, const int32_t* cu_seqlens, int batch, int max_len,
                      int num_heads, int window);
SR_API int sr_test_attention_tc(const void* qkv_f16, void* out_f16, const int32_t* cu_seqlens, int batch, int total_tokens,
                                int max_len, int num_heads, int window);
SR_API int sr_test_attention_win(const void* qkv_f16, void* out_f16, const int32_t* d_cu_seqlens, int batch, int total_tokens,
                                 int max_len, int num_heads, int window);
/* debug: CTA-0 event timeline of the next tcgen05 attention launches into a device buffer of 3 x 4096 int64 (NULL = off) */
SR_API int sr_test_attention_trace(void* dev_buf_3x4096_i64);
SR_API int sr_test_layernorm(const float* x, int t, int h, const float* w, const float* b, float eps, float* y32,
                      void* y16);
/* The pipeline sr_cache_topk takes for b queries over n stored rows of dim d and top-k (host only, no GPU needed):
 * route -1 refused, 0 nothing to do (b or k <= 0), 1 empty store, 2 GEMV scores + two-stage selection (b <= 4),
 * 3 GEMM with the fused top-8 epilogue (b > 4, k <= 8), 4 GEMM scores + two-stage selection; chunks / chunk_rows: the
 * score chunks of routes 2 and 4; stage2_smem: shared memory of the final selection (route 3: its upper bound). */
SR_API int sr_test_cache_topk_plan(int b, int n, int d, int k, int32_t* route, int32_t* chunks, int32_t* chunk_rows,
                                   int64_t* stage2_smem);

#ifdef __cplusplus
}
#endif
#endif
