// Semantic-cache lookup: cosine scores of a query batch against a device-resident fp16 matrix of unit
// vectors, then per-query top-k with the reference tie rule.
//
// Replaces the Go scalar loop `embeddingDotProduct` + `scanLinearForSimilarity`
// (/root/reference/src/semantic-router/pkg/cache/inmemory_cache_search.go:14-20,65-89; first max wins) and
// the stable-sort top-k of `calculate_similarity_batch`
// (/root/reference/candle-binding/src/ffi/embedding.rs:1640-1681; lower index first on ties).
//
// v1 pipeline: scores[B, chunk] = Q . C^T on the tcgen05 GEMM (fp16 operands, fp32 accumulate, fp32 store;
// HBM-bound for small B, tensor-bound for B >= ~256), then a two-stage selection:
//   stage 1: one CTA per (query, 8192-score segment): each warp takes the top-k of its 1024 register-resident scores with
//            warp shuffles, warp 0 merges the eight lists
//   stage 2: one CTA per query: same selection over the segment winners.
#include "kernels.h"

#include "common.cuh"
#include "gemm.h"

namespace srb {
namespace {

constexpr int kSelThreads = 256;
constexpr int kPerThread = 32;
constexpr int kSegment = kSelThreads * kPerThread;  // 8192 scores per stage-1 CTA

struct Cand {
  float v;
  int i;
};
__device__ __forceinline__ bool better(float v, int i, float bv, int bi) {
  // larger score wins; equal score: lower (non-negative) index wins; index -1 = nothing
  if (i < 0) return false;
  if (bi < 0) return true;
  return v > bv || (v == bv && i < bi);
}
__device__ __forceinline__ Cand block_argmax(Cand c, Cand* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, c.v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, c.i, o);
    if (better(ov, oi, c.v, c.i)) { c.v = ov; c.i = oi; }
  }
  const int warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane_id() == 0) red[warp] = c;
  __syncthreads();
  Cand b = red[0];
#pragma unroll
  for (int k = 1; k < kSelThreads / 32; ++k)
    if (better(red[k].v, red[k].i, b.v, b.i)) b = red[k];
  return b;
}

__device__ __forceinline__ Cand warp_argmax(Cand c) {   // every lane ends up with the winner
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, c.v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, c.i, o);
    if (better(ov, oi, c.v, c.i)) { c.v = ov; c.i = oi; }
  }
  return c;
}

// scores: [B, ld] fp32 for local rows [row0, row0 + n); out: cand_idx/cand_score [B, total_segments, k]
// One CTA per (query, 8192-score segment); each of its eight warps owns 1024 scores in registers (32 per lane).
// Exact top-k of a warp's 1024 scores without k full passes: the k-th largest of the 32 LANE MAXIMA is a lower bound L of
// the k-th largest score (at least k scores are >= L), so only scores >= L can be winners -- typically k..2k of them.
// They are compacted into a per-warp list (ballot + popc) and the k rounds of warp argmax run over that short list.
// A warp whose list would overflow (hundreds of tied scores) falls back to k passes over its registers.  Warp 0 then
// merges the eight lists.  (The first version -- k block-wide argmax rounds over all 8192 scores -- took 3.4x the time
// of the score GEMM it follows.)
constexpr int kListCap = 128;   // candidates per warp

__global__ void __launch_bounds__(kSelThreads)
select_stage1(const float* __restrict__ scores, int ld, int n, int row0, const uint8_t* __restrict__ valid,
              int k, int seg0, int total_segments, int* __restrict__ cand_idx, float* __restrict__ cand_score) {
  constexpr int kWarps = kSelThreads / 32;
  __shared__ float lv[kWarps][kListCap];
  __shared__ int li[kWarps][kListCap];
  __shared__ float wv[kWarps * 64];
  __shared__ int wi[kWarps * 64];
  const int q = blockIdx.y, seg = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = lane_id();
  const int base = seg * kSegment + warp * (kSegment / kWarps);   // first local row of this warp's 1024 scores
  const float* s = scores + static_cast<size_t>(q) * ld + base;
  float v[kPerThread];
  float lm = -INFINITY;
#pragma unroll
  for (int j = 0; j < kPerThread; ++j) {
    const int c = base + j * 32 + lane;  // coalesced
    const bool ok = c < n && (!valid || valid[row0 + c]);
    v[j] = ok ? s[j * 32 + lane] : -INFINITY;
    lm = fmaxf(lm, v[j]);
  }
  // rank of this lane's maximum among the 32 (ties by lane): the lane of rank min(k,32)-1 holds the bound L
  int rank = 0;
#pragma unroll
  for (int o = 0; o < 32; ++o) {
    const float ov = __shfl_sync(0xffffffffu, lm, o);
    rank += (ov > lm || (ov == lm && o < lane)) ? 1 : 0;
  }
  const int want = (k < 32 ? k : 32) - 1;
  const unsigned who = __ballot_sync(0xffffffffu, rank == want);
  float L = __shfl_sync(0xffffffffu, lm, __ffs(who) - 1);
  if (k > 32) L = -INFINITY;   // more winners than lanes: every finite score is a candidate
  // compact the candidates (score >= L, finite) into this warp's list
  int count = 0;
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int j = 0; j < kPerThread; ++j) {
    const bool cand = v[j] >= L && v[j] != -INFINITY;
    const unsigned m = __ballot_sync(0xffffffffu, cand);
    const int at = count + __popc(m & lt);
    if (cand && at < kListCap) { lv[warp][at] = v[j]; li[warp][at] = row0 + base + j * 32 + lane; }
    count += __popc(m);
  }
  __syncwarp();
  if (count <= kListCap) {
    for (int r = 0; r < k; ++r) {
      Cand c{-INFINITY, -1};
      int where = -1;
      for (int t = lane; t < count; t += 32)
        if (better(lv[warp][t], li[warp][t], c.v, c.i)) { c.v = lv[warp][t]; c.i = li[warp][t]; where = t; }
      const Cand b = warp_argmax(c);
      if (where >= 0 && b.i >= 0 && c.i == b.i) li[warp][where] = -1;   // indices are unique: exactly one owner
      __syncwarp();
      if (lane == 0) { wv[warp * 64 + r] = b.i >= 0 ? b.v : -INFINITY; wi[warp * 64 + r] = b.i; }
    }
  } else {   // pathological ties: k passes over the registers
    uint32_t removed = 0;
    for (int r = 0; r < k; ++r) {
      Cand c{-INFINITY, -1};
      int cj = -1;
#pragma unroll
      for (int j = 0; j < kPerThread; ++j) {
        const bool live = !((removed >> j) & 1u) && v[j] != -INFINITY;
        const int idx = row0 + base + j * 32 + lane;
        if (live && better(v[j], idx, c.v, c.i)) { c.v = v[j]; c.i = idx; cj = j; }
      }
      const Cand b = warp_argmax(c);
      if (b.i >= 0 && b.i == c.i) removed |= 1u << cj;
      if (lane == 0) { wv[warp * 64 + r] = b.i >= 0 ? b.v : -INFINITY; wi[warp * 64 + r] = b.i; }
    }
  }
  __syncthreads();
  if (warp != 0) return;
  int* oi = cand_idx + (static_cast<size_t>(q) * total_segments + seg0 + seg) * k;
  float* os = cand_score + (static_cast<size_t>(q) * total_segments + seg0 + seg) * k;
  for (int r = 0; r < k; ++r) {
    Cand c{-INFINITY, -1};
    int where = -1;
    for (int w = 0; w < kWarps; ++w)
      for (int t = lane; t < k; t += 32) {
        const int at = w * 64 + t;
        if (better(wv[at], wi[at], c.v, c.i)) { c.v = wv[at]; c.i = wi[at]; where = at; }
      }
    const Cand b = warp_argmax(c);
    if (where >= 0 && b.i >= 0 && c.i == b.i) wi[where] = -1;
    __syncwarp();
    if (lane == 0) { oi[r] = b.i; os[r] = b.i >= 0 ? b.v : -INFINITY; }
  }
}

// ---- scores for a handful of queries (the reference's operating mode is ONE query per lookup): a GEMV, not a GEMM.
// HBM-bound by construction: every stored row is read once (D * 2 bytes), one warp per row, the queries sit in shared
// memory as fp32.  fp16 x fp16 products are exact in fp32, accumulation is fp32 in a fixed order (lane-strided chunks,
// then an xor-shuffle tree): deterministic.  The 128-row MMA tile would spend 127/128 of its work on padding here.
template <int NB>
__global__ void __launch_bounds__(256)
scores_small_kernel(const __half* __restrict__ queries, const __half* __restrict__ cache, int n, int D, int ld,
                    float* __restrict__ scores) {
  extern __shared__ float qs[];   // [NB][D]
  for (int i = threadIdx.x; i < NB * D; i += blockDim.x) qs[i] = __half2float(queries[i]);
  __syncthreads();
  const int lane = lane_id();
  const int warps = gridDim.x * (blockDim.x >> 5);
  const int chunks = D >> 3;   // 16-byte units per row
  for (int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n; row += warps) {
    const uint4* r4 = reinterpret_cast<const uint4*>(cache + static_cast<size_t>(row) * D);
    float acc[NB];
#pragma unroll
    for (int b = 0; b < NB; ++b) acc[b] = 0.f;
    for (int c = lane; c < chunks; c += 32) {
      const uint4 u = __ldg(r4 + c);
      const float2 x0 = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
      const float2 x1 = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      const float2 x2 = __half22float2(*reinterpret_cast<const __half2*>(&u.z));
      const float2 x3 = __half22float2(*reinterpret_cast<const __half2*>(&u.w));
#pragma unroll
      for (int b = 0; b < NB; ++b) {
        const float4 qa = *reinterpret_cast<const float4*>(qs + b * D + 8 * c);
        const float4 qb = *reinterpret_cast<const float4*>(qs + b * D + 8 * c + 4);
        float t = acc[b];
        t = fmaf(x0.x, qa.x, t); t = fmaf(x0.y, qa.y, t); t = fmaf(x1.x, qa.z, t); t = fmaf(x1.y, qa.w, t);
        t = fmaf(x2.x, qb.x, t); t = fmaf(x2.y, qb.y, t); t = fmaf(x3.x, qb.z, t); t = fmaf(x3.y, qb.w, t);
        acc[b] = t;
      }
    }
#pragma unroll
    for (int b = 0; b < NB; ++b) {
      const float t = warp_sum(acc[b]);
      if (lane == 0) scores[static_cast<size_t>(b) * ld + row] = t;
    }
  }
}

// per query: top-k over `ncand` candidates; writes global ids (local + id_offset)
__global__ void __launch_bounds__(kSelThreads)
select_stage2(const int* __restrict__ cand_idx, const float* __restrict__ cand_score, int ncand, int k, int id_offset,
              int* __restrict__ out_idx, float* __restrict__ out_score) {
  __shared__ Cand red[kSelThreads / 32];
  extern __shared__ uint8_t dyn[];
  float* sv = reinterpret_cast<float*>(dyn);
  int* si = reinterpret_cast<int*>(sv + ncand);
  const int q = blockIdx.x;
  for (int c = threadIdx.x; c < ncand; c += kSelThreads) {
    sv[c] = cand_score[static_cast<size_t>(q) * ncand + c];
    si[c] = cand_idx[static_cast<size_t>(q) * ncand + c];
  }
  __syncthreads();
  for (int r = 0; r < k; ++r) {
    Cand c{-INFINITY, -1};
    int where = -1;
    for (int j = threadIdx.x; j < ncand; j += kSelThreads)
      if (better(sv[j], si[j], c.v, c.i)) { c.v = sv[j]; c.i = si[j]; where = j; }
    const Cand b = block_argmax(c, red);
    if (where >= 0 && c.i == b.i && b.i >= 0) si[where] = -1;  // unique local ids: exactly one owner
    if (threadIdx.x == 0) {
      out_idx[static_cast<size_t>(q) * k + r] = b.i >= 0 ? b.i + id_offset : -1;
      out_score[static_cast<size_t>(q) * k + r] = b.i >= 0 ? b.v : -INFINITY;
    }
    __syncthreads();
  }
}

// merge of G per-shard lists holding GLOBAL ids
__global__ void __launch_bounds__(kSelThreads)
merge_kernel(const int* __restrict__ idx_parts, const float* __restrict__ score_parts, int G, int B, int k,
             int* __restrict__ out_idx, float* __restrict__ out_score) {
  __shared__ Cand red[kSelThreads / 32];
  extern __shared__ uint8_t dyn[];
  float* sv = reinterpret_cast<float*>(dyn);
  int* si = reinterpret_cast<int*>(sv + G * k);
  const int q = blockIdx.x;
  for (int c = threadIdx.x; c < G * k; c += kSelThreads) {
    const int g = c / k, j = c % k;
    sv[c] = score_parts[(static_cast<size_t>(g) * B + q) * k + j];
    si[c] = idx_parts[(static_cast<size_t>(g) * B + q) * k + j];
  }
  __syncthreads();
  for (int r = 0; r < k; ++r) {
    Cand c{-INFINITY, -1};
    int where = -1;
    for (int j = threadIdx.x; j < G * k; j += kSelThreads)
      if (better(sv[j], si[j], c.v, c.i)) { c.v = sv[j]; c.i = si[j]; where = j; }
    const Cand b = block_argmax(c, red);
    if (where >= 0 && c.i == b.i && b.i >= 0) si[where] = -1;
    if (threadIdx.x == 0) {
      out_idx[static_cast<size_t>(q) * k + r] = b.i;
      out_score[static_cast<size_t>(q) * k + r] = b.i >= 0 ? b.v : -INFINITY;
    }
    __syncthreads();
  }
}

// Exchange format of a sharded cache (SURVEY 8e): one 8-byte entry per (query, rank) = {fp32 score, int32 GLOBAL id}.
// Each rank packs its [B,k] result into this form, ONE all-gather moves B * k * 8 bytes per rank, and the merge below
// reads the G gathered lists directly.
__global__ void pack_pairs_kernel(const int* __restrict__ idx, const float* __restrict__ score, int n, int2* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = make_int2(__float_as_int(score[i]), idx[i]);
}
// merge of G per-shard lists in the packed form: pairs [G][B][k]
__global__ void __launch_bounds__(kSelThreads)
merge_packed_kernel(const int2* __restrict__ pairs, int G, int B, int k, int* __restrict__ out_idx,
                    float* __restrict__ out_score) {
  __shared__ Cand red[kSelThreads / 32];
  extern __shared__ uint8_t dyn[];
  float* sv = reinterpret_cast<float*>(dyn);
  int* si = reinterpret_cast<int*>(sv + G * k);
  const int q = blockIdx.x;
  for (int c = threadIdx.x; c < G * k; c += kSelThreads) {
    const int g = c / k, j = c % k;
    const int2 e = pairs[(static_cast<size_t>(g) * B + q) * k + j];
    sv[c] = __int_as_float(e.x);
    si[c] = e.y;
  }
  __syncthreads();
  for (int r = 0; r < k; ++r) {
    Cand c{-INFINITY, -1};
    int where = -1;
    for (int j = threadIdx.x; j < G * k; j += kSelThreads)
      if (better(sv[j], si[j], c.v, c.i)) { c.v = sv[j]; c.i = si[j]; where = j; }
    const Cand b = block_argmax(c, red);
    if (where >= 0 && c.i == b.i && b.i >= 0) si[where] = -1;   // global ids are unique across shards
    if (threadIdx.x == 0) {
      out_idx[static_cast<size_t>(q) * k + r] = b.i;
      out_score[static_cast<size_t>(q) * k + r] = b.i >= 0 ? b.v : -INFINITY;
    }
    __syncthreads();
  }
}

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
inline int chunk_rows(int B, int N) {
  // keep the score buffer <= 1 GiB; multiple of the stage-1 segment
  size_t rows = (static_cast<size_t>(1) << 30) / (static_cast<size_t>(B > 0 ? B : 1) * 4);
  rows = rows / kSegment * kSegment;
  if (rows < static_cast<size_t>(kSegment)) rows = kSegment;
  const size_t need = align_up(static_cast<size_t>(N), kSegment);
  return static_cast<int>(rows < need ? rows : need);
}

}  // namespace

constexpr int kFusedK = 8;        // list length of the GEMM's top-k epilogue (gemm.h EPI_TOPK)
constexpr int kFusedLists = 320;  // upper bound of the lists per query (= 2 x CTAs launched <= 2 x SMs)
constexpr size_t kStage2SmemMax = 200 * 1024;   // candidates select_stage2 holds in shared memory
// A launch gets 48 KB of shared memory without the per-kernel opt-in, the static `red` array of select_stage2 /
// merge_packed_kernel included: at exactly 48 KB of candidates the launch fails without the opt-in
// (tests/test_cache_topk_exact_gpu.py: gemv-k64-stage2-48k, test_sharded_packed_merge_exact[96-8-64]).
constexpr size_t kSmemDefault = 48 * 1024 - sizeof(Cand) * (kSelThreads / 32);

CacheTopkPlan cache_topk_plan(int B, int N, int D, int k) {
  CacheTopkPlan p;
  if (B <= 0 || k <= 0) { p.route = CACHE_ROUTE_NONE; return p; }
  if (k > 64) { p.route = CACHE_ROUTE_REFUSED; return p; }
  if (N <= 0) { p.route = CACHE_ROUTE_EMPTY; return p; }
  if (B > 4 && k <= kFusedK && D % 8 == 0) {
    p.route = CACHE_ROUTE_FUSED;
    p.stage2_smem = static_cast<size_t>(kFusedLists) * kFusedK * 8;   // bound: the GEMM reports the lists it launched
    return p;
  }
  p.route = (B <= 4 && D % 8 == 0 && static_cast<size_t>(B) * D * 4 <= 48 * 1024) ? CACHE_ROUTE_GEMV : CACHE_ROUTE_GEMM;
  p.chunk_rows = chunk_rows(B, N);
  p.chunks = (N + p.chunk_rows - 1) / p.chunk_rows;
  p.stage2_smem = static_cast<size_t>((N + kSegment - 1) / kSegment) * k * 8;
  if (p.stage2_smem > kStage2SmemMax) p.route = CACHE_ROUTE_REFUSED;
  return p;
}

size_t cache_topk_workspace_bytes(int B, int N, int k) {
  const int chunk = chunk_rows(B, N);
  const size_t segs = (static_cast<size_t>(N) + kSegment - 1) / kSegment;
  const size_t two_pass = align_up(static_cast<size_t>(B) * chunk * 4, 256) + 2 * align_up(static_cast<size_t>(B) * segs * k * 4, 256);
  const size_t fused = 2 * align_up(static_cast<size_t>(B) * kFusedLists * kFusedK * 4, 256);
  return two_pass > fused ? two_pass : fused;
}

int cache_topk(cudaStream_t stream, const __half* queries, int B, const __half* cache, const uint8_t* valid, int N,
               int D, int k, int id_offset, int* out_idx, float* out_score, void* workspace, size_t workspace_bytes) {
  const CacheTopkPlan plan = cache_topk_plan(B, N, D, k);
  if (plan.route == CACHE_ROUTE_NONE) return 0;
  if (plan.route == CACHE_ROUTE_REFUSED) {
    // before any launch: nothing is queued for a request that cannot be served
    if (k > 64) fprintf(stderr, "[srb200] cache_topk: k=%d unsupported (<= 64)\n", k);
    else fprintf(stderr, "[srb200] cache_topk: too many candidates (%zu bytes of stage-2 shared memory)\n", plan.stage2_smem);
    return -1;
  }
  if (workspace_bytes < cache_topk_workspace_bytes(B, N, k)) {
    fprintf(stderr, "[srb200] cache_topk: workspace too small\n");
    return -1;
  }
  const int chunk = chunk_rows(B, N);
  const int segs = (N + kSegment - 1) / kSegment;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  float* scores = reinterpret_cast<float*>(ws);
  int* cand_idx = reinterpret_cast<int*>(ws + align_up(static_cast<size_t>(B) * chunk * 4, 256));
  float* cand_score = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(cand_idx) +
                                               align_up(static_cast<size_t>(B) * segs * k * 4, 256));
  if (plan.route == CACHE_ROUTE_EMPTY) {
    select_stage2<<<B, kSelThreads, 0, stream>>>(cand_idx, cand_score, 0, k, id_offset, out_idx, out_score);
    SRB_CUDA_CHECK(cudaGetLastError());
  note_launch();
    return 0;
  }
  if (plan.route == CACHE_ROUTE_FUSED) {
    // Scores never leave the SM: the GEMM's epilogue keeps a running top-8 per (query, CTA) and only those short lists
    // are written (B x <= 148 x 8 pairs); no 1 GiB score chunks, no selection pass over them.
    int* l_idx = reinterpret_cast<int*>(ws);
    float* l_score = reinterpret_cast<float*>(ws + align_up(static_cast<size_t>(B) * kFusedLists * kFusedK * 4, 256));
    int lists = 0;
    GemmDesc g;
    g.M = B; g.N = static_cast<int>(align_up(N, 256)); g.K = D; g.A = queries; g.W = cache;   // the store is padded to 256 rows
    g.epi = EPI_TOPK; g.topk_idx = l_idx; g.topk_score = l_score; g.topk_valid = valid; g.topk_n = N; g.topk_lists = &lists;
    // a CTA only writes the lists of the query rows it walked: every other slot must read "nothing" (idx -1)
    SRB_CUDA_CHECK(cudaMemsetAsync(l_idx, 0xFF, static_cast<size_t>(B) * kFusedLists * kFusedK * 4, stream));
    if (gemm_f16(stream, g)) return -1;
    if (lists <= 0 || lists > kFusedLists) { fprintf(stderr, "[srb200] cache_topk: %d lists\n", lists); return -1; }
    const int ncand = lists * kFusedK;
    select_stage2<<<B, kSelThreads, static_cast<size_t>(ncand) * 8, stream>>>(l_idx, l_score, ncand, k, id_offset, out_idx, out_score);
    SRB_CUDA_CHECK(cudaGetLastError());
    note_launch();
    return 0;
  }
  for (int row0 = 0; row0 < N; row0 += chunk) {
    const int n = (N - row0) < chunk ? (N - row0) : chunk;
    const int n_pad = static_cast<int>(align_up(n, 64));  // cache allocation is padded to 256 rows
    if (plan.route == CACHE_ROUTE_GEMV) {
      static int num_sms = 0;
      if (!num_sms) {
        int dev = 0;
        SRB_CUDA_CHECK(cudaGetDevice(&dev));
        SRB_CUDA_CHECK(cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev));
      }
      const int grid = num_sms * 8;   // 8 CTAs x 8 warps per SM: enough loads in flight to cover the HBM latency
      const size_t smem = static_cast<size_t>(B) * D * 4;
      const __half* cw = cache + static_cast<size_t>(row0) * D;
      switch (B) {
        case 1: scores_small_kernel<1><<<grid, 256, smem, stream>>>(queries, cw, n, D, chunk, scores); break;
        case 2: scores_small_kernel<2><<<grid, 256, smem, stream>>>(queries, cw, n, D, chunk, scores); break;
        case 3: scores_small_kernel<3><<<grid, 256, smem, stream>>>(queries, cw, n, D, chunk, scores); break;
        default: scores_small_kernel<4><<<grid, 256, smem, stream>>>(queries, cw, n, D, chunk, scores); break;
      }
      SRB_CUDA_CHECK(cudaGetLastError());
      note_launch();
    } else {
      GemmDesc g;
      g.M = B; g.N = n_pad; g.K = D; g.A = queries; g.W = cache + static_cast<size_t>(row0) * D;
      g.out = scores; g.ldo = chunk; g.epi = EPI_RESID; g.resid = nullptr; g.ldr = chunk;
      if (gemm_f16(stream, g)) return -1;
    }
    const dim3 grid((n + kSegment - 1) / kSegment, B);
    select_stage1<<<grid, kSelThreads, 0, stream>>>(scores, chunk, n, row0, valid, k, row0 / kSegment, segs, cand_idx,
                                                    cand_score);
    SRB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  }
  const int ncand = segs * k;
  const size_t smem = plan.stage2_smem;
  if (smem > kSmemDefault)
    SRB_CUDA_CHECK(cudaFuncSetAttribute(select_stage2, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  select_stage2<<<B, kSelThreads, smem, stream>>>(cand_idx, cand_score, ncand, k, id_offset, out_idx, out_score);
  SRB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  return 0;
}

int cache_merge_topk(cudaStream_t stream, const int* idx_parts, const float* score_parts, int G, int B, int k,
                     int* out_idx, float* out_score) {
  if (B <= 0) return 0;
  merge_kernel<<<B, kSelThreads, static_cast<size_t>(G) * k * 8, stream>>>(idx_parts, score_parts, G, B, k, out_idx,
                                                                          out_score);
  SRB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  return 0;
}

int cache_pack_pairs(cudaStream_t stream, const int* idx, const float* score, int n, void* pairs_out) {
  if (n <= 0) return 0;
  pack_pairs_kernel<<<(n + 255) / 256, 256, 0, stream>>>(idx, score, n, static_cast<int2*>(pairs_out));
  SRB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  return 0;
}

int cache_merge_packed(cudaStream_t stream, const void* pairs, int G, int B, int k, int* out_idx, float* out_score) {
  if (B <= 0) return 0;
  const size_t smem = static_cast<size_t>(G) * k * 8;
  if (smem > 48 * 1024) { fprintf(stderr, "[srb200] cache_merge_packed: G * k = %d too large\n", G * k); return -1; }
  if (smem > kSmemDefault)
    SRB_CUDA_CHECK(cudaFuncSetAttribute(merge_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  merge_packed_kernel<<<B, kSelThreads, smem, stream>>>(static_cast<const int2*>(pairs), G, B, k, out_idx, out_score);
  SRB_CUDA_CHECK(cudaGetLastError());
  note_launch();
  return 0;
}

}  // namespace srb
