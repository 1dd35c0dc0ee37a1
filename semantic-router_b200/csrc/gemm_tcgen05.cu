// Persistent, warp-specialised tcgen05 GEMM for sm_100a with fused epilogues.
//
//   C[M,N] = A[M,K] (fp16, K-major)  x  W[N,K]^T (fp16, K-major == nn.Linear layout), fp32 accumulate in TMEM.
//
// Replaces the dense f32 `gemm`+rayon matmuls behind candle's Linear on the reference's hot loop
// (/root/reference/candle-binding/src/model_architectures/traditional/candle_models/modernbert.rs
//  :123 Wqkv, :196 Wo, :236-238 Wi/GeGLU/Wo) with one kernel family:
//   * warp 0      : TMA producer  (cp.async.bulk.tensor 2D, 128B swizzle, mbarrier complete_tx)
//   * warp 1      : TMEM allocator + single-thread tcgen05.mma issuer (UMMA 128 x BN x 16)
//   * warps 2..5  : epilogue (tcgen05.ld 32x32b -> registers -> fused math -> global)
//   * TMEM holds two BN-column fp32 accumulator stages so the epilogue of tile i overlaps the MMAs of tile i+1.
// Fused epilogues: bias, RoPE (rotate-half, modernbert.rs:61-85), fp32 residual add (:300-303),
// GeGLU = gelu_erf(a)*b (:238), erf-GELU (BERT intermediate).
#include "gemm.h"

#include <cstdlib>
#include <mutex>

#include "common.cuh"
#include "kernels.h"

namespace srb {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 fp16 = 128 B = one swizzle-128B row
constexpr int kGemmThreads = 192;
// EPI_TOPK runs EIGHT epilogue warps (two per scheduler, each half of the tile's columns): its epilogue is a chain of
// dependent scalar work per score (one warp per scheduler issued one instruction every ~6 cycles and the scan ran at a
// tenth of the tensor rate); the other flavours keep four.
// EW = epilogue warps: 4 (one per TMEM lane quadrant) or 8 (two per quadrant, each takes every other chunk of a tile).
__host__ __device__ constexpr int gemm_threads(int ew) { return 64 + 32 * ew; }
__host__ __device__ constexpr int default_ew(int epi) { return epi == EPI_TOPK ? 8 : 4; }
constexpr int kStageBufBytes = 4096;   // one epilogue staging box: 32 rows x 128 B
constexpr int kBarrierBytes = 512;
constexpr int kSmemLimit = 232448;     // 227 KB opt-in limit per CTA
// staging boxes per epilogue warp.  The fp32-residual epilogue is the HBM-bound one (it reads and writes 4 B per
// output element): it keeps two residual loads and two stores in flight per warp, the others only need two boxes.
// The fp16-pair residual epilogue keeps three (hi, lo) box pairs per warp: one pair loading, one computing, one storing --
// two pairs per warp when it runs eight warps (the second warp of a scheduler covers the first one's store drain).
__host__ __device__ constexpr int stage_bufs(int epi, int ew = 4) {
  return epi == EPI_RESID ? 4 : (epi == EPI_RESID_HL ? (ew == 8 ? 4 : 6) : 2);
}

// kPair: a cluster of two CTAs (one TPC) computes a 256 x BN tile with cta_group::2 UMMAs; each CTA stages its own
// 128 rows of A and half of the B tile, and holds its 128 rows of the accumulator in its own TMEM.
template <int BN, int EPI, bool kPair = false, int EW = 4, int XB = 0>
struct GemmCfg {
  static constexpr int kBufs = stage_bufs(EPI, EW) + XB;   // XB: extra staging boxes per epilogue warp (A/B: SRB_EPI_XB)
  static constexpr int kEpiWarps = EW;
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = (kPair ? BN / 2 : BN) * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = 2 * BN;  // two accumulator stages
  static constexpr int kRawBufs = EPI == EPI_RESID ? 2 : 0;   // fp16 copy of the residual stream (LayerNorm fold)
  static constexpr int kEpiBytes = EW * (kBufs + kRawBufs) * kStageBufBytes;
  static constexpr int kFit = (kSmemLimit - kEpiBytes - 1024 /*align slack*/ - kBarrierBytes) / kStageBytes;
  static constexpr int kStages = kFit < 6 ? kFit : 6;   // as deep as shared memory allows, 6 at most
  static constexpr int kSmemBytes = kStages * kStageBytes + kEpiBytes + 1024 + kBarrierBytes;
  static_assert(kStages >= 3, "mainloop ring too shallow");
};

struct KArgs {
  int M, N, K;
  const float* bias;
  int has_resid;
  const int* pos;
  const float* rope_cos;
  const float* rope_sin;
  int rope_cols;
  float* row_stats;          // EPI_RESID: accumulate (sum, sumsq) per row
  int has_raw16;             // EPI_RESID: tmap_aux is the fp16 copy of the output
  const float* fold_stats;   // EPI_ROPE / EPI_GEGLU: per-row (sum, sumsq) of the A rows (null: no fold)
  float fold_eps;
  float fold_inv_h;
  int fold_parts;            // 128-column slices the row statistics come in
  float* pivot_out;          // EPI_RESID: row pivots (see gemm.h)
  const float* pivot_in;
  const float* pivot_in_stats;
  int* topk_idx;             // EPI_TOPK
  float* topk_score;
  const uint8_t* topk_valid;
  int topk_n;
  int grouped;               // EPI_TOPK: grouped tile schedule (see the kernel)
  int interleave;            // tiles w, w + W, ... per worker instead of a contiguous range
  int K2;                    // K extension: k-blocks beyond K come from (tmap_a2, tmap_b2) -- low-rank adapters (gemm.h)
  int mask_block, mask_rows; // EPI_F16: keep column c of row r only when c / mask_block == r / mask_rows (0: off)
  int grp_rows;              // > 0: W is a stack of [N, K] matrices, rows [g * grp_rows, (g + 1) * grp_rows) of A multiply matrix g
  int dbg;                   // timing experiments only (SRB_GEMM_DBG): 1 = EPI_RESID_HL without its arithmetic, 2 = without its residual traffic,
                             // 4 = RoPE / GeGLU epilogues without their arithmetic, 8 = without their output stores
};
constexpr int kTopK = 8;
constexpr bool kEpi8Default = false;

// LayerNorm fold, consumer side.  W'' = (W diag(gamma)) with every row re-centred to sum zero, so that
// sum_k x[r,k] W''[n,k] = sum_k (x[r,k] - mean_r) W'[n,k]: the mean subtraction of the LayerNorm happens inside the GEMM
// (the centring matrix I - 11^T/H commutes into the weights) and the epilogue is left with the per-row rstd factor --
// which the RoPE epilogue folds into the row's cos / sin registers (the rotation is linear), so q and k cost nothing.
__device__ __forceinline__ void fold_scale(float rstd, uint32_t* a, uint32_t* b) {
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    a[i] = __float_as_uint(__uint_as_float(a[i]) * rstd);
    b[i] = __float_as_uint(__uint_as_float(b[i]) * rstd);
  }
}

template <int BN, int EPI, bool kPair, int EW = 4, int XB = 0>
__global__ void __launch_bounds__(gemm_threads(EW), 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
            const __grid_constant__ CUtensorMap tmap_out, const __grid_constant__ CUtensorMap tmap_aux,
            const __grid_constant__ CUtensorMap tmap_a2, const __grid_constant__ CUtensorMap tmap_b2, const KArgs p) {
  using Cfg = GemmCfg<BN, EPI, kPair, EW, XB>;
  static_assert(Cfg::kSmemBytes <= kSmemLimit, "over the 227 KB shared-memory opt-in limit");
  static_assert(EW == 4 || EW == 8, "four or eight epilogue warps");
  static_assert(EW == 4 || EPI == EPI_TOPK || EPI == EPI_ROPE || EPI == EPI_GEGLU || EPI == EPI_RESID_HL,
                "eight epilogue warps: TOPK / ROPE / GEGLU / RESID_HL");
  constexpr bool kHL = EPI == EPI_RESID_HL;
  constexpr int kCtas = kPair ? 2 : 1;
  constexpr int kStageBufs = Cfg::kBufs;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + Cfg::kStages * Cfg::kABytes;
  uint8_t* smem_epi = smem + Cfg::kStages * Cfg::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_epi + Cfg::kEpiBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + Cfg::kStages;
  uint64_t* tfull_bar = bars + 2 * Cfg::kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* resid_bar = tempty_bar + 2;  // [EW warps][kStageBufs]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(resid_bar + EW * kStageBufs);
  static_assert((2 * Cfg::kStages + 4 + EW * kStageBufs) * 8 + 4 <= kBarrierBytes, "barrier block too small");

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = kPair ? cluster_ctarank() : 0u;
  const int m_blocks = (p.M + BM * kCtas - 1) / (BM * kCtas);  // (pair: 256-row blocks, this CTA owns one half)
  const int n_blocks = (p.N + BN - 1) / BN;
  const int k1_blocks = (p.K + BK - 1) / BK;
  // K extension: the accumulator also takes A2[M, K2] x W2[N, K2]^T -- same stages, same MMAs, other tensor maps
  const int k_blocks = k1_blocks + (p.K2 + BK - 1) / BK;
  const int num_tiles = m_blocks * n_blocks;
  auto row_base = [&](int m_blk) { return (m_blk * kCtas + static_cast<int>(cta_rank)) * BM; };
  // contiguous tile range per CTA (n fastest): one CTA walks all N tiles of an M block back to back, so the
  // A row-block stays hot in L2 and per-row epilogue state (RoPE cos/sin) is reused across tiles
  const int num_workers = gridDim.x / kCtas;
  const int base = num_tiles / num_workers, rem = num_tiles % num_workers;
  const int bid = blockIdx.x / kCtas;
  int t_begin = bid * base + (bid < rem ? bid : rem);
  int t_end = t_begin + base + (bid < rem ? 1 : 0);
  // EPI_TOPK, grouped schedule (p.grouped): worker w owns query block w % m_blocks for its whole life (its running
  // top-8 lists live in registers) and walks the stored-row tiles g, g + G, g + 2G, ... with g = w / m_blocks,
  // G = workers / m_blocks.  The m_blocks workers of a group therefore ask for the SAME stored-row tile at about the
  // same time: one HBM read, the rest L2 hits -- the store streams once per batch instead of once per query block
  // (ncu, B = 1024 over 1 M x 768: 11.2 GB read with the contiguous schedule against 1.54 GB algorithmic).
  // Tiles are numbered t = m_blk * n_blocks + n_blk as everywhere else; `t_step` is the distance between two tiles of
  // this worker (1 for the contiguous ranges).
  int t_step = 1;
  // Interleaved schedule (p.interleave; the fp32-residual GEMMs): worker w takes tiles w, w + W, w + 2W, ...  With
  // n fastest in the tile numbering the N / BN tiles of one row block run AT THE SAME TIME on neighbouring workers, so
  // each A k-block is pulled from HBM once and hit in L2 by the others.  The contiguous ranges re-read A from HBM for
  // every column tile here (ncu inside a step: MLP-out 986 MB read against 705 MB algorithmic) because the residual
  // stream that passes through L2 between two tiles of one worker (~60 MB) evicts the row block.
  if (p.interleave) {
    t_begin = bid;
    t_end = num_tiles;
    t_step = num_workers;
  }
  if constexpr (EPI == EPI_TOPK) {
    if (p.grouped) {
      const int groups = num_workers / m_blocks;
      const int m_own = bid % m_blocks, g_own = bid / m_blocks;
      t_begin = m_own * n_blocks + g_own;
      t_end = (m_own + 1) * n_blocks;
      t_step = groups;
      if (g_own >= groups) t_end = t_begin;   // workers beyond the last full group stay idle
    }
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    tma_prefetch_desc(&tmap_out);
#pragma unroll
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tfull_bar[0], 1);
    mbar_init(&tfull_bar[1], 1);
    mbar_init(&tempty_bar[0], EW * kCtas);  // the leader's MMA waits for the epilogue warps of both CTAs
    mbar_init(&tempty_bar[1], EW * kCtas);
    for (int i = 0; i < EW * kStageBufs; ++i) mbar_init(&resid_bar[i], 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    if constexpr (kPair) tmem_alloc_pair<Cfg::kTmemCols>(tmem_slot);
    else tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();                           // tmem_slot / barrier init visible inside this CTA ...
  if constexpr (kPair) cluster_sync_all();   // ... and the peer's barriers initialised before anything targets them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // PDL: everything above overlapped the previous kernel's tail; nothing below may start before its writes are visible
  griddep_launch_dependents();
  griddep_wait();

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int t = t_begin; t < t_end; t += t_step) {
        const int m_blk = t / n_blocks, n_blk = t % n_blocks;
        // grouped weights (one matrix per task, stacked along N): the row block picks its matrix; blocks never straddle
        // two groups (grp_rows is a multiple of the block height, checked on the host)
        const int w_row0 = p.grp_rows > 0 ? ((m_blk * BM * kCtas) / p.grp_rows) * p.N : 0;
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1);
          const bool ext = kb >= k1_blocks;
          const CUtensorMap* ma = ext ? &tmap_a2 : &tmap_a;
          const CUtensorMap* mb = ext ? &tmap_b2 : &tmap_b;
          const int kc = (ext ? kb - k1_blocks : kb) * BK;
          if constexpr (kPair) {
            // both CTAs' loads are credited to the leader's barrier, which expects the bytes of the whole pair
            const uint32_t lead_full = mapa_u32(smem_u32(&full_bar[s]), 0);
            if (cta_rank == 0) mbar_expect_tx(&full_bar[s], 2 * Cfg::kStageBytes);
            tma_load_2d_pair(smem_a + s * Cfg::kABytes, ma, lead_full, kc, row_base(m_blk));
            tma_load_2d_pair(smem_b + s * Cfg::kBBytes, mb, lead_full, kc,
                             (ext ? 0 : w_row0) + n_blk * BN + static_cast<int>(cta_rank) * (BN / 2));
          } else {
            mbar_expect_tx(&full_bar[s], Cfg::kStageBytes);
            tma_load_2d(smem_a + s * Cfg::kABytes, ma, &full_bar[s], kc, m_blk * BM);
            tma_load_2d(smem_b + s * Cfg::kBBytes, mb, &full_bar[s], kc, (ext ? 0 : w_row0) + n_blk * BN);
          }
          if (++s == Cfg::kStages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (one thread) =================
    if (lane == 0 && cta_rank == 0) {
      constexpr uint32_t idesc = umma_idesc_f16(BM * kCtas, BN);
      int s = 0;
      uint32_t ph = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int t = t_begin; t < t_end; t += t_step) {
        mbar_wait(&tempty_bar[as], aph ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(as * BN);
        for (int kb = 0; kb < k_blocks; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint64_t da = umma_desc_sw128(smem_u32(smem_a + s * Cfg::kABytes));
          const uint64_t db = umma_desc_sw128(smem_u32(smem_b + s * Cfg::kBBytes));
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // advance 16 fp16 = 32 B along K inside the swizzle atom: +2 in (addr >> 4) units
            if constexpr (kPair)
              umma_f16_pair(d_tmem, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                            (kb > 0 || k > 0) ? 1u : 0u);
            else
              umma_f16(d_tmem, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                       (kb > 0 || k > 0) ? 1u : 0u);
          }
          // frees this smem stage (in both CTAs of a pair) when the MMAs have read it
          if constexpr (kPair) umma_commit_pair(&empty_bar[s], 3);
          else umma_commit(&empty_bar[s]);
          if (++s == Cfg::kStages) { s = 0; ph ^= 1; }
        }
        if constexpr (kPair) umma_commit_pair(&tfull_bar[as], 3);  // accumulator stage complete
        else umma_commit(&tfull_bar[as]);
        if (++as == 2) { as = 0; aph ^= 1; }
      }
    }
  } else {
    // ================= epilogue warps: TMEM -> registers -> swizzled smem box -> TMA store =================
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;   // EW == 8: which of the two warps of this quadrant (takes chunks half, half + 2, ...)
    uint8_t* my_bufs = smem_epi + (warp - 2) * ((kStageBufs + Cfg::kRawBufs) * kStageBufBytes);
    uint8_t* my_raw = my_bufs + kStageBufs * kStageBufBytes;   // [kRawBufs] fp16 boxes (32 rows x 64 columns)
    const bool want_raw = (EPI == EPI_RESID) && p.has_raw16;
    const bool want_stats = (EPI == EPI_RESID || kHL) && p.row_stats != nullptr;
    const bool fold = (EPI == EPI_ROPE || EPI == EPI_GEGLU) && p.fold_stats != nullptr;
    float f_rstd = 1.f;   // fold: rstd of this thread's row
    float pv = 0.f;       // fold producer: this thread's row pivot (EPI_RESID_HL: the pivot SHIFT of this GEMM)
    float pv_prev = 0.f;  // EPI_RESID_HL: the pivot the stored pair is relative to
    int pv_mblk = -1;
    int fold_mblk = -1;
    uint64_t* my_rbar = resid_bar + (warp - 2) * kStageBufs;
    int as = 0;
    uint32_t aph = 0;
    int cb = 0;                 // staging buffer to use next
    uint32_t rph = 0;           // phase bit per staging buffer (residual loads)
    // chunk geometry: a chunk is one 32-row x 128-byte output box of this warp
    constexpr int kAccPerChunk = (EPI == EPI_RESID || EPI == EPI_TOPK) ? 32 : (EPI == EPI_GEGLU ? 128 : 64);  // accumulator columns
    constexpr int kOutPerChunk = (EPI == EPI_RESID || EPI == EPI_TOPK) ? 32 : 64;                                // output columns
    constexpr int kChunks = BN / kAccPerChunk;
    constexpr int kPairs = kStageBufs / 2;   // EPI_RESID_HL: (hi, lo) box pairs of this warp
    // EPI_RESID_HL with eight warps: the two warps of a TMEM lane quadrant take the two 128-column halves of a tile (whole
    // statistics slices each); with four warps a warp walks all chunks
    constexpr int kWarpChunks = (kHL && EW == 8) ? kChunks / 2 : kChunks;
    const int c_base = (kHL && EW == 8) ? half * kWarpChunks : 0;
    const int n_out = (EPI == EPI_GEGLU) ? p.N / 2 : p.N;
    const bool use_resid = (EPI == EPI_RESID) && p.has_resid;

    // EPI_RESID: residual boxes are TMA-loaded one chunk ahead (flat over (tile, chunk) of this CTA)
    auto out_col = [&](int t, int c) { return (t % n_blocks) * (BN / kAccPerChunk * kOutPerChunk) + c * kOutPerChunk; };
    auto chunk_valid = [&](int t, int c) { return t < t_end && out_col(t, c) < n_out; };
    auto issue_resid = [&](int t, int c, int buf) {  // lane 0 only
      if constexpr (kHL) {   // buf = pair index: hi box, then lo box, one barrier for both
        uint8_t* pb = my_bufs + buf * 2 * kStageBufBytes;
        mbar_expect_tx(&my_rbar[buf], 2 * kStageBufBytes);
        tma_load_2d(pb, &tmap_out, &my_rbar[buf], out_col(t, c), row_base(t / n_blocks) + quad * 32);
        tma_load_2d(pb + kStageBufBytes, &tmap_aux, &my_rbar[buf], out_col(t, c), row_base(t / n_blocks) + quad * 32);
      } else {
        mbar_expect_tx(&my_rbar[buf], kStageBufBytes);
        tma_load_2d(my_bufs + buf * kStageBufBytes, &tmap_out, &my_rbar[buf], out_col(t, c),
                    row_base(t / n_blocks) + quad * 32);
      }
    };
    // residual prefetch cursor: runs kAhead chunks in front of the chunk being processed (flat over this CTA's
    // (tile, chunk) sequence); with 4 boxes that keeps two loads and two stores of this warp in flight
    constexpr int kRing = kHL ? kPairs : kStageBufs;   // residual-load ring: boxes, or box pairs
    constexpr int kAhead = kHL ? 1 : (kStageBufs - 2 > 0 ? kStageBufs - 2 : 1);
    int pf_t = t_begin, pf_c = 0, pf_buf = 0;
    auto pf_issue = [&]() {  // lane 0 only
      if (!chunk_valid(pf_t, c_base + pf_c)) return;
      issue_resid(pf_t, c_base + pf_c, pf_buf);
      if (++pf_buf == kRing) pf_buf = 0;
      if (++pf_c >= kWarpChunks || !chunk_valid(pf_t, c_base + pf_c)) { pf_t += t_step; pf_c = 0; }
    };
    if ((use_resid || (kHL && !(p.dbg & 2))) && lane == 0) {
#pragma unroll
      for (int i = 0; i < kAhead; ++i) pf_issue();
    }

    // EPI_ROPE: this thread's cos/sin row, reloaded only when the M block changes
    float cs[EPI == EPI_ROPE ? 32 : 1], sn[EPI == EPI_ROPE ? 32 : 1];
    int rope_mblk = -1;

    // EPI_TOPK: this thread's running top-8 (descending) over the columns this CTA walks for its current row
    float tk_v[EPI == EPI_TOPK ? kTopK : 1];
    int tk_i[EPI == EPI_TOPK ? kTopK : 1];
    int tk_mblk = -1;
    auto tk_reset = [&]() {
#pragma unroll
      for (int i = 0; i < (EPI == EPI_TOPK ? kTopK : 1); ++i) { tk_v[i] = -INFINITY; tk_i[i] = -1; }
    };
    auto tk_flush = [&](int m_blk_done) {   // this CTA's list for the row it has just left
      const int row = row_base(m_blk_done) + quad * 32 + lane;
      if (row < p.M) {
        const size_t at = (static_cast<size_t>(row) * (2 * (gridDim.x / kCtas)) + 2 * bid + half) * kTopK;
#pragma unroll
        for (int i = 0; i < (EPI == EPI_TOPK ? kTopK : 1); ++i) { p.topk_idx[at + i] = tk_i[i]; p.topk_score[at + i] = tk_v[i]; }
      }
    };
    for (int t = t_begin; t < t_end; t += t_step) {
      const int m_blk = t / n_blocks, n_blk = t % n_blocks;
      const int row0 = row_base(m_blk) + quad * 32;
      if constexpr (EPI == EPI_TOPK) {
        if (m_blk != tk_mblk) {
          if (tk_mblk >= 0) tk_flush(tk_mblk);
          tk_reset();
          tk_mblk = m_blk;
        }
      }
      if constexpr (EPI == EPI_ROPE || EPI == EPI_GEGLU) {
        if (fold && m_blk != fold_mblk) {
          const int row = row0 + lane < p.M ? row0 + lane : p.M - 1;
          float s1 = 0.f, s2 = 0.f;
          for (int k = 0; k < p.fold_parts; ++k) {   // fixed slice order: reproducible
            const float2 st = __ldg(reinterpret_cast<const float2*>(p.fold_stats) + static_cast<size_t>(k) * p.M + row);
            s1 += st.x;
            s2 += st.y;
          }
          const float mean = s1 * p.fold_inv_h;
          const float var = fmaxf(s2 * p.fold_inv_h - mean * mean, 0.f);
          f_rstd = rsqrtf(var + p.fold_eps);
          fold_mblk = m_blk;
          rope_mblk = -1;   // the row's cos / sin registers carry rstd: reload them for this M block
        }
      }
      if constexpr (EPI == EPI_ROPE) {
        if (m_blk != rope_mblk && n_blk * BN < p.rope_cols) {
          const int row = row0 + lane;
          const int pos = __ldg(p.pos + (row < p.M ? row : p.M - 1));   // rows past M: any valid table row (never stored)
          const float4* c4 = reinterpret_cast<const float4*>(p.rope_cos + static_cast<size_t>(pos) * 32);
          const float4* s4 = reinterpret_cast<const float4*>(p.rope_sin + static_cast<size_t>(pos) * 32);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 a = __ldg(c4 + i), b = __ldg(s4 + i);
            cs[4 * i] = a.x; cs[4 * i + 1] = a.y; cs[4 * i + 2] = a.z; cs[4 * i + 3] = a.w;
            sn[4 * i] = b.x; sn[4 * i + 1] = b.y; sn[4 * i + 2] = b.z; sn[4 * i + 3] = b.w;
          }
          if (fold) {   // LayerNorm fold: the rstd factor of the row rides on the (linear) rotation
#pragma unroll
            for (int i = 0; i < 32; ++i) { cs[i] *= f_rstd; sn[i] *= f_rstd; }
          }
          rope_mblk = m_blk;
        }
      }
      float st1 = 0.f, st2 = 0.f;   // EPI_RESID: this row's (sum, sum of squares) over the current 128-column slice
      if constexpr (kHL) {
        // pivot shift of this row: the stored pair is x - pivot_in; the new pivot is pivot_in + (mean of x - pivot_in),
        // read from the previous residual GEMM's statistics (0 for the first one: the embedding's pair is x itself)
        if (m_blk != pv_mblk) {
          pv = 0.f;
          pv_prev = 0.f;
          if (p.pivot_in_stats) {
            const int row = row0 + lane < p.M ? row0 + lane : p.M - 1;
            float s1 = 0.f;
            const int parts = p.N >> 7;
            for (int k = 0; k < parts; ++k)
              s1 += __ldg(reinterpret_cast<const float2*>(p.pivot_in_stats) + static_cast<size_t>(k) * p.M + row).x;
            pv = s1 / static_cast<float>(p.N);
            pv_prev = __ldg(p.pivot_in + row);
          }
          pv_mblk = m_blk;
        }
      }
      if constexpr (EPI == EPI_RESID) {
        if (want_stats && m_blk != pv_mblk) {   // the row's pivot: its mean after the previous residual GEMM
          pv = 0.f;
          if (p.pivot_in_stats) {
            const int row = row0 + lane < p.M ? row0 + lane : p.M - 1;
            float s1 = 0.f;
            const int parts = p.N >> 7;
            for (int k = 0; k < parts; ++k)
              s1 += __ldg(reinterpret_cast<const float2*>(p.pivot_in_stats) + static_cast<size_t>(k) * p.M + row).x;
            pv = __ldg(p.pivot_in + row) + s1 / static_cast<float>(p.N);
          }
          pv_mblk = m_blk;
        }
      }
      mbar_wait(&tfull_bar[as], aph);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + static_cast<uint32_t>(as * BN);

      if constexpr (EPI == EPI_TOPK) {
        // This warp scans columns [half * BN/2, (half+1) * BN/2) of the tile, 32 at a time, the TMEM load of the next
        // chunk in flight while the current one is reduced.  The common path per chunk is the maximum of 32 scores and
        // one compare against the list's tail; validity (invalidated rows, padding rows >= topk_n) is only looked up
        // for a score that would enter the list -- after the first tiles that is rare, and the byte loads of a `valid`
        // sweep were most of the old epilogue.
        auto topk_chunk = [&](uint32_t* r, int ocol0) {
          float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            m0 = fmax3(m0, __uint_as_float(r[i]), __uint_as_float(r[i + 1]));
            m1 = fmax3(m1, __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
            m2 = fmax3(m2, __uint_as_float(r[i + 4]), __uint_as_float(r[i + 5]));
            m3 = fmax3(m3, __uint_as_float(r[i + 6]), __uint_as_float(r[i + 7]));
          }
          // Take the chunk's maximum while it beats the list's tail (usually zero or one round): a round is ~150
          // instructions, against ~1300 for trying all 32 scores in turn -- and with 32 rows per warp some lane
          // triggers in most chunks, so the round's length is what the epilogue costs.
          float cm = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
          while (cm > tk_v[kTopK - 1]) {   // strict: an equal score at a higher column never displaces
            int ci = 31;
#pragma unroll
            for (int i = 30; i >= 0; --i)
              if (__uint_as_float(r[i]) == cm) ci = i;          // lowest column holding the maximum
            ci = __uint_as_float(r[31]) == cm && ci == 31 ? 31 : ci;
            float cv = cm;
            int cidx = ocol0 + ci;
            const bool ok = cidx < p.topk_n && (!p.topk_valid || __ldg(p.topk_valid + (cidx < p.topk_n ? cidx : 0)));
            if (ok) {
              // Insertion into the list, ordered by score and then by column.  The entries it displaces move down one
              // place each: one that equals the next entry has the lower column and must shift past it, not fall off
              // the end.  (With a plain `cv > tk_v[j]` a list of eight equal scores that then took a higher one lost
              // its LOWEST column: tests/test_cache_topk_exact_gpu.py, fused-b128-same and fused-grouped-b1000-same.)
#pragma unroll
              for (int j = 0; j < kTopK; ++j) {
                if (cv > tk_v[j] || (cv == tk_v[j] && cidx < tk_i[j])) {
                  const float tv = tk_v[j]; const int ti = tk_i[j];
                  tk_v[j] = cv; tk_i[j] = cidx;
                  cv = tv; cidx = ti;
                }
              }
            }
            float n0 = -INFINITY, n1 = -INFINITY;
#pragma unroll
            for (int i = 0; i < 32; i += 2) {   // drop it and find the next maximum
              if (i == ci) r[i] = 0xff800000u;
              if (i + 1 == ci) r[i + 1] = 0xff800000u;
              n0 = fmaxf(n0, __uint_as_float(r[i]));
              n1 = fmaxf(n1, __uint_as_float(r[i + 1]));
            }
            cm = fmaxf(n0, n1);
          }
        };
        constexpr int kPer = kChunks / 2;
        static_assert(EPI != EPI_TOPK || kPer % 2 == 0, "chunk pairs");
        const int cbeg = half * kPer;
        uint32_t ra[32], rb[32];
        tmem_ld32(t_row + cbeg * 32, ra);
#pragma unroll 1
        for (int cc = 0; cc < kPer; cc += 2) {
          tmem_ld_wait();
          tmem_ld32(t_row + (cbeg + cc + 1) * 32, rb);
          topk_chunk(ra, out_col(t, cbeg + cc));
          tmem_ld_wait();
          if (cc + 2 < kPer) tmem_ld32(t_row + (cbeg + cc + 2) * 32, ra);
          topk_chunk(rb, out_col(t, cbeg + cc + 1));
        }
      }
      if constexpr (kHL) {
        // 64-column chunks: the (hi, lo) boxes of the chunk arrive by TMA one chunk ahead, are updated in place in
        // shared memory and leave by TMA; statistics per 128-column slice as in EPI_RESID
#pragma unroll 1
        for (int cc = 0; cc < kWarpChunks; ++cc) {
          const int c = c_base + cc;
          const int ocol0 = out_col(t, c);
          if (ocol0 >= n_out) break;
          uint8_t* hb = my_bufs + cb * 2 * kStageBufBytes;
          uint8_t* lb = hb + kStageBufBytes;
          if (!(p.dbg & 2)) {
          if (lane == 0) {
            // the pair the prefetch cursor points at was stored kPairs - 1 chunks ago: all but the newest store group read out
            bulk_wait_read<kPairs - kAhead - 1>();
            pf_issue();
          }
          mbar_wait(&my_rbar[cb], (rph >> cb) & 1u);
          rph ^= 1u << cb;
          }
#pragma unroll
          for (int hf = 0; hf < ((p.dbg & 1) ? 0 : 2); ++hf) {
            uint32_t r[32];
            tmem_ld32(t_row + c * 64 + hf * 32, r);
            tmem_ld_wait();
#pragma unroll
            for (int u = 0; u < 4; ++u) {   // 16-byte units: 8 columns each
              const uint32_t off = box_off(lane, hf * 4 + u);
              uint4 hv = *reinterpret_cast<const uint4*>(hb + off);
              uint4 lv = *reinterpret_cast<const uint4*>(lb + off);
              uint32_t hw[4] = {hv.x, hv.y, hv.z, hv.w}, lw[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&hw[k]));
                const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&lw[k]));
                float x0 = (fh.x + fl.x) + (__uint_as_float(r[8 * u + 2 * k]) - pv);
                float x1 = (fh.y + fl.y) + (__uint_as_float(r[8 * u + 2 * k + 1]) - pv);
                if (p.bias) {
                  const float2 b = __ldg(reinterpret_cast<const float2*>(p.bias + ocol0 + hf * 32 + 8 * u) + k);
                  x0 += b.x; x1 += b.y;
                }
                st1 += x0 + x1;
                st2 += x0 * x0 + x1 * x1;
                const __half2 nh = __floats2half2_rn(x0, x1);
                const float2 fb = __half22float2(nh);
                hw[k] = *reinterpret_cast<const uint32_t*>(&nh);
                lw[k] = pack_half2(x0 - fb.x, x1 - fb.y);
              }
              sts16(hb + off, hw[0], hw[1], hw[2], hw[3]);
              sts16(lb + off, lw[0], lw[1], lw[2], lw[3]);
            }
          }
          if (c & 1) {   // a 128-column slice is complete: its partial goes out, once
            if (row0 + lane < p.M) {
              const size_t part = static_cast<size_t>((ocol0 - 64) >> 7);
              *reinterpret_cast<float2*>(p.row_stats + 2 * (part * p.M + row0 + lane)) = make_float2(st1, st2);
              if (part == 0) p.pivot_out[row0 + lane] = pv_prev + pv;
            }
            st1 = 0.f;
            st2 = 0.f;
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && !(p.dbg & 2)) {
            tma_store_2d(&tmap_out, hb, ocol0, row0);
            tma_store_2d(&tmap_aux, lb, ocol0, row0);
            bulk_commit();
          }
          if (++cb == kPairs) cb = 0;
        }
      }
#pragma unroll 1
      for (int c = (EW == 8 ? half : 0); c < ((EPI == EPI_TOPK || kHL) ? 0 : kChunks); c += EW / 4) {
        const int ocol0 = out_col(t, c);
        if (ocol0 >= n_out) break;
        uint8_t* buf = my_bufs + cb * kStageBufBytes;
        uint8_t* my_row = buf;  // + box_off(lane, chunk16)
        if (use_resid) {
          // the box the prefetch cursor points at was last used kStageBufs - kAhead chunks ago: its store must have
          // been read out (all but the newest kStageBufs - kAhead - 1 store groups complete)
          if (lane == 0) {
            bulk_wait_read<(kStageBufs - kAhead - 1 > 0 ? kStageBufs - kAhead - 1 : 0)>();
            pf_issue();
          }
          mbar_wait(&my_rbar[cb], (rph >> cb) & 1u);
          rph ^= 1u << cb;
        } else {
          if (lane == 0) bulk_wait_read<kStageBufs - 1>();  // this buffer's previous store has been read out
          __syncwarp();
        }

        if constexpr (EPI == EPI_RESID) {
          uint32_t r[32];
          tmem_ld32(t_row + c * 32, r);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            float4* q = reinterpret_cast<float4*>(my_row + box_off(lane, i));
            float4 x = use_resid ? *q : make_float4(0.f, 0.f, 0.f, 0.f);
            x.x += __uint_as_float(r[4 * i]);
            x.y += __uint_as_float(r[4 * i + 1]);
            x.z += __uint_as_float(r[4 * i + 2]);
            x.w += __uint_as_float(r[4 * i + 3]);
            if (p.bias) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + ocol0) + i);
              x.x += b.x; x.y += b.y; x.z += b.z; x.w += b.w;
            }
            *q = x;
            x.x -= pv; x.y -= pv; x.z -= pv; x.w -= pv;   // statistics and the fp16 copy are taken of x - pivot
            st1 += (x.x + x.y) + (x.z + x.w);
            st2 += (x.x * x.x + x.y * x.y) + (x.z * x.z + x.w * x.w);
            if (want_raw) {   // fp16 copy: chunk c fills 16-byte units (c & 1) * 4 + i / 2 of the 64-column box
              r[2 * i] = pack_half2(x.x, x.y);
              r[2 * i + 1] = pack_half2(x.z, x.w);
            }
          }
          if (want_stats && (c & 3) == 3) {   // a 128-column slice is complete: its partial goes out, once
            if (row0 + lane < p.M) {
              const size_t part = static_cast<size_t>((ocol0 - 96) >> 7);
              *reinterpret_cast<float2*>(p.row_stats + 2 * (part * p.M + row0 + lane)) = make_float2(st1, st2);
              if (part == 0 && p.pivot_out) p.pivot_out[row0 + lane] = pv;
            }
            st1 = 0.f;
            st2 = 0.f;
          }
          if (want_raw) {
            uint8_t* rb = my_raw + ((c >> 1) & 1) * kStageBufBytes;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              sts16(rb + box_off(lane, (c & 1) * 4 + i), r[4 * i], r[4 * i + 1], r[4 * i + 2], r[4 * i + 3]);
          }
        } else if constexpr (EPI == EPI_F16 || EPI == EPI_GELU) {
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            uint32_t r[32];
            tmem_ld32(t_row + c * 64 + hf * 32, r);
            tmem_ld_wait();
            uint32_t h[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              float v0 = __uint_as_float(r[2 * i]), v1 = __uint_as_float(r[2 * i + 1]);
              if (p.bias) {
                const float2 b = __ldg(reinterpret_cast<const float2*>(p.bias + ocol0 + hf * 32) + i);
                v0 += b.x; v1 += b.y;
              }
              if constexpr (EPI == EPI_GELU) { v0 = gelu_erf_fast_f(v0); v1 = gelu_erf_fast_f(v1); }
              if constexpr (EPI == EPI_F16) {
                if (p.mask_block > 0) {   // adapter projections: a row keeps the column block of its own task only
                  const int own = (row0 + lane) / p.mask_rows, col = ocol0 + hf * 32 + 2 * i;
                  if (col / p.mask_block != own) v0 = 0.f;
                  if ((col + 1) / p.mask_block != own) v1 = 0.f;
                }
              }
              h[i] = pack_half2(v0, v1);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
              sts16(my_row + box_off(lane, hf * 4 + i), h[4 * i], h[4 * i + 1], h[4 * i + 2], h[4 * i + 3]);
          }
        } else if constexpr (EPI == EPI_ROPE) {
          uint32_t r1[32], r2[32];
          tmem_ld32(t_row + c * 64, r1);
          tmem_ld32(t_row + c * 64 + 32, r2);
          tmem_ld_wait();
          if (fold && ocol0 >= p.rope_cols) fold_scale(f_rstd, r1, r2);   // v columns: no rotation to carry rstd
          if (ocol0 < p.rope_cols && !(p.dbg & 4)) {  // q and k heads: rotate-half over the 64-wide head (in place, packed)
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float a0 = __uint_as_float(r1[2 * i]), a1 = __uint_as_float(r1[2 * i + 1]);
              const float b0 = __uint_as_float(r2[2 * i]), b1 = __uint_as_float(r2[2 * i + 1]);
              r1[i] = pack_half2(a0 * cs[2 * i] - b0 * sn[2 * i], a1 * cs[2 * i + 1] - b1 * sn[2 * i + 1]);
              r2[i] = pack_half2(a0 * sn[2 * i] + b0 * cs[2 * i], a1 * sn[2 * i + 1] + b1 * cs[2 * i + 1]);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              r1[i] = pack_half2(__uint_as_float(r1[2 * i]), __uint_as_float(r1[2 * i + 1]));
              r2[i] = pack_half2(__uint_as_float(r2[2 * i]), __uint_as_float(r2[2 * i + 1]));
            }
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            sts16(my_row + box_off(lane, i), r1[4 * i], r1[4 * i + 1], r1[4 * i + 2], r1[4 * i + 3]);
            sts16(my_row + box_off(lane, 4 + i), r2[4 * i], r2[4 * i + 1], r2[4 * i + 2], r2[4 * i + 3]);
          }
        } else if constexpr (EPI == EPI_GEGLU) {
          // W rows are pre-interleaved in 32-row groups [a(32j..32j+31) | b(32j..32j+31)]: accumulator columns
          // [64j, 64j+32) hold `a`, [64j+32, 64j+64) the matching `b`; one output chunk = two such groups
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            uint32_t ra[32], rb[32];
            tmem_ld32(t_row + c * 128 + hf * 64, ra);
            tmem_ld32(t_row + c * 128 + hf * 64 + 32, rb);
            tmem_ld_wait();
            if (p.dbg & 4) {   // timing experiment: no GeGLU arithmetic
#pragma unroll
              for (int i = 0; i < 16; ++i) ra[i] = pack_half2(__uint_as_float(ra[2 * i]), __uint_as_float(rb[2 * i + 1]));
            } else if (p.dbg & 16) {   // A/B: the round-1 form (separate rstd multiplies, degree-6 erf)
            if (fold) fold_scale(f_rstd, ra, rb);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float g0 = gelu_erf_fast_f(__uint_as_float(ra[2 * i])) * __uint_as_float(rb[2 * i]);
              const float g1 = gelu_erf_fast_f(__uint_as_float(ra[2 * i + 1])) * __uint_as_float(rb[2 * i + 1]);
              ra[i] = pack_half2(g0, g1);
            }
            } else {
              const float rs = fold ? f_rstd : 1.0f;
              const float kz = rs * 0.70710678118654752440f, kh = 0.5f * rs * rs;
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float g0 = geglu_fold_f(__uint_as_float(ra[2 * i]), __uint_as_float(rb[2 * i]), kz, kh);
                const float g1 = geglu_fold_f(__uint_as_float(ra[2 * i + 1]), __uint_as_float(rb[2 * i + 1]), kz, kh);
                ra[i] = pack_half2(g0, g1);
              }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
              sts16(my_row + box_off(lane, hf * 4 + i), ra[4 * i], ra[4 * i + 1], ra[4 * i + 2], ra[4 * i + 3]);
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0 && !(p.dbg & 8)) {
          tma_store_2d(&tmap_out, buf, ocol0, row0);  // rows >= M / cols >= N are clipped by the TMA unit
          if constexpr (EPI == EPI_RESID) {
            // the fp16 box completes every second chunk and rides in the same bulk group as that chunk's fp32 store
            // (its staging box is reused four chunks later, far behind the wait_group.read above)
            if (want_raw && (c & 1)) tma_store_2d(&tmap_aux, my_raw + ((c >> 1) & 1) * kStageBufBytes, ocol0 - 32, row0);
          }
          bulk_commit();
        }
        if (++cb == kStageBufs) cb = 0;
      }
      // release this accumulator stage back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (kPair) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[as]), 0));
        else mbar_arrive(&tempty_bar[as]);
      }
      if (++as == 2) { as = 0; aph ^= 1; }
    }
    if constexpr (EPI == EPI_TOPK) {
      if (tk_mblk >= 0) tk_flush(tk_mblk);
    }
    if (lane == 0) bulk_wait_read<0>();  // smem must outlive the last stores' reads
    __syncwarp();
  }

  tc_fence_before();
  if constexpr (kPair) cluster_sync_all();  // neither CTA may retire while the other still targets its smem/TMEM
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if constexpr (kPair) tmem_dealloc_pair<Cfg::kTmemCols>(tmem_base);
    else tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  });
  return fn;
}

template <int BN, int EPI, bool kPair, int EW = 4, int XB = 0>
int launch(cudaStream_t stream, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc,
           const CUtensorMap& tx, const CUtensorMap& ta2, const CUtensorMap& tb2, const KArgs& ka, int num_sms,
           int grid_override = 0) {
  using Cfg = GemmCfg<BN, EPI, kPair, EW, XB>;
  constexpr int kCtas = kPair ? 2 : 1;
  // per-device attribute; cheap enough to set on every launch (multi-GPU processes switch devices)
  SRB_CUDA_CHECK(cudaFuncSetAttribute(gemm_kernel<BN, EPI, kPair, EW, XB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      Cfg::kSmemBytes));
  const int m_blocks = (ka.M + BM * kCtas - 1) / (BM * kCtas), n_blocks = (ka.N + BN - 1) / BN;
  const int tiles = m_blocks * n_blocks;
  const int workers = num_sms / kCtas;
  const int grid = grid_override > 0 ? grid_override : (tiles < workers ? tiles : workers) * kCtas;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(gemm_threads(EW));
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCtas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
  SRB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, gemm_kernel<BN, EPI, kPair, EW, XB>, ta, tb, tc, tx, ta2, tb2, ka));
  note_launch();
  return 0;
}

// SRB_GEMM_PAIR=0 forces the 1-CTA tiles (A/B measurements); default: pairs whenever they apply
bool pair_enabled() {
  static const bool on = [] {
    const char* e = getenv("SRB_GEMM_PAIR");
    return !(e && e[0] == '0');
  }();
  return on;
}

}  // namespace

static int make_tmap_2d(CUtensorMap* out, CUtensorMapDataType dt, int elem_bytes, const void* ptr, uint64_t cols,
                        uint64_t rows, uint64_t ld_elems, uint32_t box_cols, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    fprintf(stderr, "[srb200] cuTensorMapEncodeTiled entry point unavailable\n");
    return -1;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld_elems * elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, dt, 2, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    fprintf(stderr, "[srb200] cuTensorMapEncodeTiled failed: %d (cols=%llu rows=%llu ld=%llu box=%ux%u)\n", (int)r,
            (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)ld_elems, box_cols, box_rows);
    return -1;
  }
  return 0;
}

int make_tmap_2d_f16(CUtensorMap* out, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld_elems,
                     uint32_t box_cols, uint32_t box_rows) {
  return make_tmap_2d(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ptr, cols, rows, ld_elems, box_cols, box_rows);
}

int make_tmap_f16_kmajor(CUtensorMap* out, const void* ptr, uint64_t rows, uint64_t k, uint32_t box_rows) {
  return make_tmap_2d(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, ptr, k, rows, k, BK, box_rows);
}

int gemm_f16(cudaStream_t stream, const GemmDesc& g) {
  if (g.M <= 0) return 0;
  if (g.K % 8 != 0 || g.N % 64 != 0 || g.ldo % 8 != 0) {
    fprintf(stderr, "[srb200] gemm_f16: unsupported shape M=%d N=%d K=%d ldo=%d\n", g.M, g.N, g.K, g.ldo);
    return -1;
  }
  if (g.epi == EPI_RESID && g.resid && (g.resid != g.out || g.ldr != g.ldo)) {
    fprintf(stderr, "[srb200] gemm_f16: EPI_RESID runs in place (resid must alias out) or without residual\n");
    return -1;
  }
  const bool is_hl = g.epi == EPI_RESID_HL;
  if (is_hl && (!g.lo16 || !g.row_stats || !g.pivot_out || g.N % 128 != 0 || g.ldo != g.N || g.raw16 || g.resid)) {
    fprintf(stderr, "[srb200] gemm_f16: EPI_RESID_HL needs out (hi) + lo16 with ld = N, row_stats, pivot_out, N %% 128 == 0\n");
    return -1;
  }
  if (g.epi == EPI_GEGLU && g.N % 128 != 0) {
    fprintf(stderr, "[srb200] gemm_f16: EPI_GEGLU needs N %% 128 == 0\n");
    return -1;
  }
  static int num_sms = 0;  // all devices of one box are the same part
  if (!num_sms) {
    int dev = 0, n = 0;
    SRB_CUDA_CHECK(cudaGetDevice(&dev));
    SRB_CUDA_CHECK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    num_sms = n;
  }
  // BN = 256 when N tiles evenly (768, 2304, 3072, ...), else 128 (e.g. MiniLM 384).
  // the fp32-residual epilogue carries 96 KB of staging boxes: its 1-CTA form uses 128-column tiles (32 KB stages)
  // Small problems (a single prompt: 4 row blocks) would put a 256-column grid on a fraction of the SMs; with
  // 128-column tiles twice as many CTAs each do half the mainloop and half the epilogue (SRB_SMALL_BN128=0: off).
  static const bool small_bn128 = [] { const char* e = getenv("SRB_SMALL_BN128"); return !(e && e[0] == '0'); }();
  const long long tiles256 = static_cast<long long>((g.M + BM - 1) / BM) * (g.N / 256);
  const bool small = small_bn128 && g.epi != EPI_TOPK && g.N % 128 == 0 && tiles256 * 2 <= num_sms;
  const bool resid_like = g.epi == EPI_RESID || is_hl;   // 96 KB of staging boxes
  const bool bn256 = (g.N % 256 == 0) && !small && !(resid_like && !(g.M >= 2048 && pair_enabled()));
  // CTA pairs (256 x 256 tiles, cta_group::2) once there are enough rows to fill the machine with them
  const bool pair = bn256 && g.M >= 2048 && pair_enabled() && g.epi != EPI_TOPK;
  CUtensorMap ta, tb, tc;
  if (make_tmap_f16_kmajor(&ta, g.A, static_cast<uint64_t>(g.a_rows > 0 ? g.a_rows : g.M), g.K, BM)) return -1;
  const int w_groups = g.w_groups > 1 ? g.w_groups : 1;
  if (w_groups > 1 && (g.w_group_rows <= 0 || g.w_group_rows % (pair ? 256 : 128) != 0 || g.N % (bn256 ? 256 : 128) != 0 || g.epi == EPI_TOPK)) {
    fprintf(stderr, "[srb200] gemm_f16: grouped weights need w_group_rows %% %d == 0 and whole column tiles\n", pair ? 256 : 128);
    return -1;
  }
  if (make_tmap_f16_kmajor(&tb, g.W, static_cast<uint64_t>(g.N) * w_groups, g.K, (bn256 && !pair) ? 256 : 128)) return -1;
  // output boxes: 32 rows x 128 bytes (64 fp16 or 32 fp32 columns), clipped at M rows / n_out columns
  if (g.epi == EPI_TOPK) {
    tc = ta;   // no matrix output
  } else if (g.epi == EPI_RESID) {
    if (make_tmap_2d(&tc, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, g.out, g.N, g.M, g.ldo, 32, 32)) return -1;
  } else if (is_hl) {
    if (make_tmap_2d(&tc, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, g.out, g.N, g.M, g.N, 64, 32)) return -1;
  } else {
    const uint64_t n_out = g.epi == EPI_GEGLU ? g.N / 2 : g.N;
    if (make_tmap_2d(&tc, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, g.out, n_out, g.M, g.ldo, 64, 32)) return -1;
  }
  KArgs ka;
  ka.M = g.M; ka.N = g.N; ka.K = g.K;
  ka.bias = g.bias; ka.has_resid = g.resid != nullptr;
  ka.pos = g.pos; ka.rope_cos = g.rope_cos; ka.rope_sin = g.rope_sin; ka.rope_cols = g.rope_cols;
  ka.row_stats = nullptr; ka.has_raw16 = 0;
  ka.pivot_out = g.pivot_out; ka.pivot_in = g.pivot_in; ka.pivot_in_stats = g.pivot_in_stats;
  ka.topk_idx = g.topk_idx; ka.topk_score = g.topk_score; ka.topk_valid = g.topk_valid; ka.topk_n = g.topk_n;
  ka.grouped = 0;
  // SRB_RESID_INTERLEAVE=0 restores the contiguous ranges for the residual GEMMs (A/B measurements)
  static const bool resid_interleave = [] { const char* e = getenv("SRB_RESID_INTERLEAVE"); return !(e && e[0] == '0'); }();
  static const int interleave_min_k = [] { const char* e = getenv("SRB_RESID_INTERLEAVE"); return (e && e[0] == '2') ? 0 : 768; }();
  // fp16-pair form: interleaved for every K (attn-out 5.36 -> 5.28 ms / 22 launches, same box)
  // measured on the headline step (same box, tools/gpu_r2_ab2.sh): MLP-out (K = 1152) 7.0 -> 6.77 ms / 22 launches, attn-out
  // (K = 768: its row block is two thirds the size and mostly survived in L2 already) 6.42 -> 6.52 ms -- so only K > 768
  ka.interleave = (((g.epi == EPI_RESID && g.resid != nullptr) || is_hl) && resid_interleave && (is_hl || g.K > interleave_min_k) &&
                   g.N / (bn256 ? 256 : 128) > 1) ? 1 : 0;
  if ((g.pivot_in != nullptr) != (g.pivot_in_stats != nullptr) || ((g.pivot_out || g.pivot_in) && !g.row_stats)) {
    fprintf(stderr, "[srb200] gemm_f16: pivots come with row_stats, pivot_in with pivot_in_stats\n");
    return -1;
  }
  ka.fold_stats = nullptr; ka.fold_eps = 0.f; ka.fold_inv_h = 0.f; ka.fold_parts = 0;
  ka.K2 = 0; ka.mask_block = 0; ka.mask_rows = 0;
  ka.grp_rows = w_groups > 1 ? g.w_group_rows : 0;
  static const int hl_dbg = [] { const char* e = getenv("SRB_GEMM_DBG"); return e ? atoi(e) : 0; }();
  ka.dbg = hl_dbg;
  CUtensorMap ta2 = ta, tb2 = tb;   // K extension (low-rank adapters): unused copies otherwise
  if (g.K2 > 0) {
    if (!g.A2 || !g.W2 || g.K2 % 8 != 0 || g.epi == EPI_TOPK) {
      fprintf(stderr, "[srb200] gemm_f16: K extension needs A2, W2 and K2 %% 8 == 0\n");
      return -1;
    }
    if (make_tmap_f16_kmajor(&ta2, g.A2, static_cast<uint64_t>(g.a_rows > 0 ? g.a_rows : g.M), g.K2, BM)) return -1;
    if (make_tmap_f16_kmajor(&tb2, g.W2, g.N, g.K2, (bn256 && !pair) ? 256 : 128)) return -1;
    ka.K2 = g.K2;
  }
  if (g.mask_block > 0) {
    if (g.epi != EPI_F16 || g.mask_rows <= 0) {
      fprintf(stderr, "[srb200] gemm_f16: the column-block mask belongs to EPI_F16\n");
      return -1;
    }
    ka.mask_block = g.mask_block; ka.mask_rows = g.mask_rows;
  }
  CUtensorMap tx = tc;   // auxiliary output map (fp16 copy of the residual stream); unused otherwise
  if (is_hl) {
    if (make_tmap_2d(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, g.lo16, g.N, g.M, g.N, 64, 32)) return -1;
    ka.row_stats = g.row_stats;
  } else if (g.row_stats || g.raw16) {
    if (g.epi != EPI_RESID || g.N % 128 != 0) {
      fprintf(stderr, "[srb200] gemm_f16: row_stats / raw16 belong to EPI_RESID with N %% 128 == 0\n");
      return -1;
    }
    ka.row_stats = g.row_stats;
    if (g.raw16) {
      if (make_tmap_2d(&tx, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, g.raw16, g.N, g.M, g.N, 64, 32)) return -1;
      ka.has_raw16 = 1;
    }
  }
  if (g.fold_stats) {
    if ((g.epi != EPI_ROPE && g.epi != EPI_GEGLU) || g.fold_h <= 0 || g.fold_h % 128 != 0) {
      fprintf(stderr, "[srb200] gemm_f16: LayerNorm fold belongs to EPI_ROPE / EPI_GEGLU with the row length\n");
      return -1;
    }
    ka.fold_stats = g.fold_stats; ka.fold_eps = g.fold_eps;
    ka.fold_inv_h = 1.0f / static_cast<float>(g.fold_h);
    ka.fold_parts = g.fold_h / 128;
  }
#define SRB_LAUNCH(E)                                                               \
  return pair    ? launch<256, E, true>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms)        \
         : bn256 ? launch<256, E, false>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms)       \
                 : launch<128, E, false>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms)
  // SRB_EPI8=1: eight epilogue warps for the two compute-heavy epilogues of the CTA-pair kernels (A/B measurements)
  static const bool epi8 = [] { const char* e = getenv("SRB_EPI8"); return e ? e[0] == '1' : kEpi8Default; }();
  // SRB_EPI_XB=1: four staging boxes per epilogue warp instead of two for the RoPE / GeGLU pair kernels (A/B measurements)
  static const bool epi_xb = [] { const char* e = getenv("SRB_EPI_XB"); return e && e[0] == '1'; }();
  switch (g.epi) {
    case EPI_F16: SRB_LAUNCH(EPI_F16);
    case EPI_ROPE:
      if (pair && epi8) return launch<256, EPI_ROPE, true, 8>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
      if (pair && epi_xb) return launch<256, EPI_ROPE, true, 4, 2>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
      SRB_LAUNCH(EPI_ROPE);
    case EPI_RESID:
      return pair ? launch<256, EPI_RESID, true>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms)
                  : launch<128, EPI_RESID, false>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
    case EPI_RESID_HL: {
      // SRB_HL_EW8=1: eight epilogue warps (two box pairs each, three mainloop stages).  Measured slower on the headline
      // step (profiles/r2_hl_experiments.txt): the arithmetic hides better (attn-out without its traffic 3.66 -> 3.31 ms)
      // but the data path with two pairs per warp and the shallower mainloop lose more (5.43 -> 5.58, MLP-out 5.90 -> 6.66)
      static const bool hl8 = [] { const char* e = getenv("SRB_HL_EW8"); return e && e[0] == '1'; }();
      if (pair && hl8) return launch<256, EPI_RESID_HL, true, 8>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
      return pair ? launch<256, EPI_RESID_HL, true>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms)
                  : launch<128, EPI_RESID_HL, false>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
    }
    case EPI_GEGLU:
      if (pair && epi8) return launch<256, EPI_GEGLU, true, 8>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
      if (pair && epi_xb) return launch<256, EPI_GEGLU, true, 4, 2>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
      SRB_LAUNCH(EPI_GEGLU);
    case EPI_GELU: SRB_LAUNCH(EPI_GELU);
    case EPI_TOPK: {
      if (!g.topk_idx || !g.topk_score || !g.topk_lists || g.N % 256 != 0) {
        fprintf(stderr, "[srb200] gemm_f16: EPI_TOPK needs list buffers and N %% 256 == 0\n");
        return -1;
      }
      // 1-CTA 128 x 256 tiles: the query batch is the short dimension here, the stored rows stream as N
      const int m_blocks = (g.M + BM - 1) / BM, n_blocks = g.N / 256;
      const long long tiles = static_cast<long long>(m_blocks) * n_blocks;
      // grouped schedule (kernel comment at t_step): whole groups of m_blocks workers, each group at least one tile.
      // SRB_TOPK_GROUPED=0 restores the contiguous ranges (A/B measurements).
      static const bool grouped_on = [] { const char* e = getenv("SRB_TOPK_GROUPED"); return !(e && e[0] == '0'); }();
      const int groups = m_blocks > 0 ? num_sms / m_blocks : 0;
      if (grouped_on && m_blocks > 1 && groups >= 1 && n_blocks >= groups) {
        ka.grouped = 1;
        *g.topk_lists = 2 * groups * m_blocks;   // two lists per worker: one per column half (eight epilogue warps)
        return launch<256, EPI_TOPK, false, 8>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms, groups * m_blocks);
      }
      *g.topk_lists = 2 * static_cast<int>(tiles < num_sms ? tiles : num_sms);
      return launch<256, EPI_TOPK, false, 8>(stream, ta, tb, tc, tx, ta2, tb2, ka, num_sms);
    }
  }
#undef SRB_LAUNCH
  return -1;
}

}  // namespace srb
