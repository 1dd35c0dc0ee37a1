"""Semantic-cache top-k (cache_scan.cu: cache_topk) against an exact float64 oracle on every selection route.

Grid data: every component of a stored row or a query is j/16 with an integer j in [-3, 3].  Such values are exact in
fp16, every product is a multiple of 2^-8, and for D <= 1024 every partial sum stays below 2^6 in magnitude, so every
score is exact in fp32 whatever the accumulation order, with or without FMA.  The kernels' scores must therefore EQUAL
the oracle's and the ids must match exactly: there is no tolerance on grid data.

The stores are tie-heavy.  Grid queries have positive components, so the HOT vector (every component 3/16) scores
strictly above every other grid vector; HOT rows are planted at tile (255/256), stage-1 segment (8191/8192), score-chunk
and shard boundaries and tie with each other.  Below them lie either copies of a few pool vectors (ties every few rows,
across every tile, segment and chunk) or one vector repeated on every row (every stage-1 warp sees 1024 equal scores
and takes its overflow path; the fused epilogue's lists fill with equal scores before a HOT row displaces one).

Routes are asserted through the sr_test_cache_topk_plan hook, the function cache_topk itself branches on, so a case
cannot silently move to another route when a threshold changes.  The CPU-only tests (no `gpu` mark) check the oracle
and the route table.
"""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import cache_oracle as co, synth

ROUTE_REFUSED, ROUTE_NONE, ROUTE_EMPTY, ROUTE_GEMV, ROUTE_FUSED, ROUTE_GEMM = -1, 0, 1, 2, 3, 4
SEGMENT = 8192            # scores per stage-1 CTA
SMEM_DEFAULT = 48 * 1024  # dynamic shared memory a launch gets without opting in
HOT = 3.0 / 16


# ---- exact oracle -------------------------------------------------------------------------------------------------
def exact_topk(q, rows, k, valid=None, id_offset=0, block=64):
    """Top-k of q [B, D] against rows [N, D] (torch tensors, any float dtype, any device) with the reference tie rule.

    Scores in float64; rows with valid == False score -inf; a stable descending sort puts the lower index first on
    equal scores.  Slots past the number of valid rows are (-1, -inf).  Returns (ids int32 [B, k] with id_offset added,
    scores float64 [B, k]) on q's device."""
    import torch
    B, N = q.shape[0], rows.shape[0]
    out_i = torch.full((B, k), -1, dtype=torch.int32, device=q.device)
    out_s = torch.full((B, k), float("-inf"), dtype=torch.float64, device=q.device)
    if N == 0:
        return out_i, out_s
    r64 = rows.to(torch.float64)
    kk = min(k, N)
    for b0 in range(0, B, block):
        s = q[b0:b0 + block].to(torch.float64) @ r64.T
        if valid is not None:
            s[:, ~valid] = float("-inf")
        order = torch.sort(-s, dim=1, stable=True).indices[:, :kk]   # ascending in -s: equal scores keep index order
        sc = torch.gather(s, 1, order)
        out_i[b0:b0 + block, :kk] = torch.where(torch.isneginf(sc), -1, order + id_offset).to(torch.int32)
        out_s[b0:b0 + block, :kk] = sc
    return out_i, out_s


def check_exact(idx, sc, oi, os_, what=""):
    """Kernel (ids, fp32 scores) == oracle (ids, float64 scores) exactly, -1 / -inf padding included."""
    oi, os_ = np.asarray(oi), np.asarray(os_)
    bad = np.argwhere((idx != oi) | (sc.astype(np.float64) != os_))
    if bad.size:
        b, r = bad[0]
        raise AssertionError(f"{what}: {len(bad)} of {idx.size} slots differ; first at query {b} rank {r}: kernel "
                             f"({idx[b, r]}, {sc[b, r]!r}) oracle ({oi[b, r]}, {os_[b, r]!r}); kernel row "
                             f"{idx[b, :12].tolist()} oracle row {oi[b, :12].tolist()}")


# ---- route plan (test-hook library; host code, no GPU) --------------------------------------------------------------
def plan(srlib, b, n, d, k):
    f = srlib.hooks().sr_test_cache_topk_plan
    i32p = C.POINTER(C.c_int32)
    f.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, i32p, i32p, i32p, C.POINTER(C.c_int64)]
    route, chunks, rows, smem = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int64()
    assert f(b, n, d, k, C.byref(route), C.byref(chunks), C.byref(rows), C.byref(smem)) == 0
    return {"route": route.value, "chunks": chunks.value, "chunk_rows": rows.value, "stage2_smem": smem.value}


def fused_grouped(b, n, sms):
    """gemm_f16's choice of the grouped EPI_TOPK schedule (gemm_tcgen05.cu, case EPI_TOPK): 128-row query blocks,
    256-row store tiles, whole groups of m_blocks workers with at least one tile each."""
    m_blocks, n_blocks = -(-b // 128), -(-n // 256)
    groups = sms // m_blocks
    return m_blocks > 1 and groups >= 1 and n_blocks >= groups


# (id, B, N, D, k, store kind, id_offset, route, chunks, fused schedule: None / "contiguous" / "grouped")
CASES = [
    ("gemv-k1", 1, 20000, 72, 1, "pool", 0, ROUTE_GEMV, 1, None),
    ("gemv-k33-same", 1, 20000, 136, 33, "same", 5000, ROUTE_GEMV, 1, None),
    ("gemv-k8", 4, 10000, 768, 8, "pool", 77, ROUTE_GEMV, 1, None),
    ("gemv-k16-same", 3, 20000, 256, 16, "same", 0, ROUTE_GEMV, 1, None),
    ("gemv-k64", 4, 9000, 1024, 64, "pool", 0, ROUTE_GEMV, 1, None),
    ("gemv-k64-big-stage2", 1, 800000, 64, 64, "pool", 123, ROUTE_GEMV, 1, None),
    ("gemv-k64-stage2-48k", 1, 786000, 64, 64, "same", 0, ROUTE_GEMV, 1, None),
    ("fused-b5-k1", 5, 3000, 136, 1, "pool", 0, ROUTE_FUSED, 0, "contiguous"),
    ("fused-b128-same", 128, 20000, 768, 8, "same", 9, ROUTE_FUSED, 0, "contiguous"),
    ("fused-b129", 129, 5000, 72, 8, "pool", 0, ROUTE_FUSED, 0, "contiguous"),
    ("fused-grouped-b300", 300, 20000, 256, 8, "pool", 40000, ROUTE_FUSED, 0, "grouped"),
    ("fused-grouped-b1000-same", 1000, 4608, 1024, 8, "same", 0, ROUTE_FUSED, 0, "grouped"),
    ("gemm-b5-k9", 5, 1050, 72, 9, "pool", 3, ROUTE_GEMM, 1, None),
    ("gemm-b130-k32-same", 130, 1050, 136, 32, "same", 0, ROUTE_GEMM, 1, None),
    ("gemm-b5-k33-same", 5, 1050, 768, 33, "same", 0, ROUTE_GEMM, 1, None),
    ("gemm-b130-k64", 130, 1050, 1024, 64, "pool", 1 << 20, ROUTE_GEMM, 1, None),
    ("gemm-b16-k10", 16, 20000, 256, 10, "pool", 0, ROUTE_GEMM, 1, None),
    ("gemm-two-chunks", 1024, 300000, 64, 16, "pool", 11, ROUTE_GEMM, 2, None),
]
CASE_IDS = [c[0] for c in CASES]


def hot_rows(n, chunk_rows=0, early=True):
    """Where HOT rows go: across a 256-row tile and its column halves, an 8192-row segment and a score chunk.  Row 100
    (early) sits behind at least eight equal scores in the first column half of tile 0."""
    rows = ([100] if early else []) + [255, 256, SEGMENT - 1, SEGMENT]
    if chunk_rows and n > chunk_rows:
        rows += [chunk_rows - 1, chunk_rows]
    return sorted(r for r in rows if r < n)


def grid_store(torch, kind, n, d, seed, hot=(), pool=16, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed)
    if kind == "pool":
        p = torch.randint(-3, 4, (pool, d), generator=g, device=device)
        rows = p[torch.randint(0, pool, (n,), generator=g, device=device)]
    else:   # "same": one vector on every row
        rows = torch.randint(-3, 4, (1, d), generator=g, device=device).expand(n, d).clone()
    rows = rows.to(torch.float32) / 16
    if len(hot):
        rows[list(hot)] = HOT
    return rows


def grid_queries(torch, b, d, seed, device="cuda"):
    g = torch.Generator(device=device).manual_seed(seed + 1)
    return torch.randint(1, 4, (b, d), generator=g, device=device).to(torch.float32) / 16


def make_cache(srlib, rows_t, d, id_offset=0):
    n = rows_t.shape[0]
    c = srlib.Cache(max(n, 1), d, id_offset=id_offset)
    if n:
        c.add(rows_t.cpu().numpy())
    return c


# ---- CPU: the oracle itself -----------------------------------------------------------------------------------------
def test_oracle_tie_rule_and_padding():
    import torch
    rows = torch.tensor([[1.0, 0], [0, 1], [1, 0], [0.5, 0], [1, 0]])
    q = torch.tensor([[1.0, 0], [0, 1]])
    i, s = exact_topk(q, rows, 4, id_offset=10)
    assert i.tolist() == [[10, 12, 14, 13], [11, 10, 12, 13]]            # equal scores: lower index first
    assert s.tolist() == [[1, 1, 1, 0.5], [1, 0, 0, 0]]
    valid = torch.tensor([True, True, False, True, True])
    i, s = exact_topk(q[:1], rows, 7, valid=valid)
    assert i.tolist() == [[0, 4, 3, 1, -1, -1, -1]]                         # invalid row skipped, -1 past the valid rows
    assert s[0, :4].tolist() == [1, 1, 0.5, 0] and torch.isneginf(s[0, 4:]).all()
    i, s = exact_topk(q, rows, 3, valid=torch.zeros(5, dtype=torch.bool))
    assert (i == -1).all() and torch.isneginf(s).all()
    i, s = exact_topk(q, rows[:0], 2)
    assert (i == -1).all() and torch.isneginf(s).all()


def test_oracle_matches_numpy_oracle_on_tie_free_data():
    import torch
    rng = np.random.default_rng(3)
    rows = rng.standard_normal((500, 32)).astype(np.float32)
    q = rng.standard_normal((7, 32)).astype(np.float32)
    valid = rng.random(500) > 0.3
    for k, v in ((10, None), (10, valid), (600, None)):
        oi, os_ = co.topk_batch(q, rows, k, valid=v)
        i, s = exact_topk(torch.from_numpy(q), torch.from_numpy(rows), k, valid=None if v is None else torch.from_numpy(v))
        kk = oi.shape[1]
        assert np.array_equal(i.numpy()[:, :kk], oi)
        assert np.allclose(s.numpy()[:, :kk], os_, rtol=1e-5, atol=1e-5)
        assert (i.numpy()[:, kk:] == -1).all()


def test_grid_scores_are_exact_in_fp32():
    """The premise of the exact checks: grid scores at D = 1024 survive fp32 accumulation in any order unchanged."""
    import torch
    rows = grid_store(torch, "pool", 64, 1024, 0, pool=64, device="cpu")
    rows[:8] = HOT
    q = grid_queries(torch, 8, 1024, 0, device="cpu")
    exact = q.double() @ rows.double().T
    assert (exact.abs() < 64).all() and (exact * 256 == (exact * 256).round()).all()
    perm = torch.randperm(1024)
    assert torch.equal((q @ rows.T).double(), exact)
    assert torch.equal((q[:, perm] @ rows[:, perm].T).double(), exact)
    acc = torch.zeros(8, 64)
    for j in torch.randperm(1024).tolist():                                  # one term at a time, random order
        acc += q[:, j:j + 1] * rows[:, j]
    assert torch.equal(acc.double(), exact)


# ---- CPU: the route table -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_case_route(srlib, case):
    _, b, n, d, k, _, _, route, chunks, _ = case
    p = plan(srlib, b, n, d, k)
    assert (p["route"], p["chunks"]) == (route, chunks), p


def test_route_table(srlib):
    """Every route and sub-route the exact cases rely on, and the thresholds between them."""
    routes = {c[7] for c in CASES}
    assert routes == {ROUTE_GEMV, ROUTE_FUSED, ROUTE_GEMM}
    assert plan(srlib, 0, 100, 64, 8)["route"] == ROUTE_NONE
    assert plan(srlib, 3, 100, 64, 0)["route"] == ROUTE_NONE
    assert plan(srlib, 3, 0, 64, 8)["route"] == ROUTE_EMPTY
    assert plan(srlib, 4, 100, 64, 8)["route"] == ROUTE_GEMV
    assert plan(srlib, 5, 100, 64, 8)["route"] == ROUTE_FUSED
    assert plan(srlib, 5, 100, 64, 9)["route"] == ROUTE_GEMM
    assert plan(srlib, 4, 100, 3072, 8)["route"] == ROUTE_GEMV           # 4 x 3072 x 4 bytes of fp32 queries: 48 KB
    assert plan(srlib, 4, 100, 3080, 8)["route"] == ROUTE_GEMM           # beyond: the GEMV's shared memory is full
    assert plan(srlib, 4, 100, 64, 64)["route"] == ROUTE_GEMV
    assert plan(srlib, 4, 100, 64, 65)["route"] == ROUTE_REFUSED
    # score chunks: 1 GiB of fp32 scores at most, in whole 8192-row segments
    assert plan(srlib, 1024, 300000, 64, 16)["chunk_rows"] == 262144
    assert plan(srlib, 1024, 262144, 64, 16)["chunks"] == 1
    assert plan(srlib, 1024, 262145, 64, 16)["chunks"] == 2
    # stage 2 holds segs * k (score, id) pairs: > 48 KB needs the opt-in, > 200 KB is refused before any launch
    p = plan(srlib, 1, 800000, 64, 64)
    assert p["stage2_smem"] == 98 * 64 * 8 and p["stage2_smem"] > SMEM_DEFAULT
    assert plan(srlib, 1, 786000, 64, 64)["stage2_smem"] == SMEM_DEFAULT   # exactly 48 KB: needs the opt-in as well
    assert plan(srlib, 1, 400 * SEGMENT, 8, 64)["route"] == ROUTE_GEMV    # 400 segments x 64 x 8 bytes = 200 KB
    assert plan(srlib, 1, 400 * SEGMENT + 1, 8, 64)["route"] == ROUTE_REFUSED
    assert plan(srlib, 1, 400 * SEGMENT + 1, 8, 8)["route"] == ROUTE_GEMV
    # the fused schedule of the cases, for the B200's 148 SMs (the GPU tests re-check it with the device's count)
    assert {c[9] for c in CASES if c[7] == ROUTE_FUSED} == {"contiguous", "grouped"}
    for c in CASES:
        if c[7] == ROUTE_FUSED:
            assert fused_grouped(c[1], c[2], 148) == (c[9] == "grouped"), c[0]


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sms(cuda):
    import torch
    assert os.environ.get("SRB_TOPK_GROUPED", "1") != "0"
    return torch.cuda.get_device_properties(cuda).multi_processor_count


def _assert_route(srlib, sms, case):
    _, b, n, d, k, _, _, route, chunks, sched = case
    p = plan(srlib, b, n, d, k)
    assert (p["route"], p["chunks"]) == (route, chunks), p
    if route == ROUTE_FUSED:
        assert fused_grouped(b, n, sms) == (sched == "grouped"), (sms, sched)
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_route_exact(srlib, cuda, sms, case):
    import torch
    name, b, n, d, k, kind, off, route, chunks, _ = case
    p = _assert_route(srlib, sms, case)
    hot = hot_rows(n, p["chunk_rows"])
    seed = sum(map(ord, name))
    rows = grid_store(torch, kind, n, d, seed, hot)
    q = grid_queries(torch, b, d, seed)
    oi, os_ = exact_topk(q, rows, k, id_offset=off)
    oi, os_ = oi.cpu().numpy(), os_.cpu().numpy()
    # the fixture does what it claims: the HOT rows lead, in index order, then the ties below them
    lead = min(k, len(hot))
    assert (oi[:, :lead] == np.array(hot[:lead]) + off).all()
    if k > len(hot):
        assert (os_[:, len(hot)] == os_[:, k - 1]).any()
    c = make_cache(srlib, rows, d, off)
    idx, sc = c.topk(q.cpu().numpy(), k)
    c.close()
    check_exact(idx, sc, oi, os_, name)


VALIDITY_CASES = [   # (id, B, k, route)
    ("gemv", 4, 16, ROUTE_GEMV),
    ("fused", 64, 8, ROUTE_FUSED),
    ("fused-grouped", 300, 8, ROUTE_FUSED),
    ("gemm", 130, 33, ROUTE_GEMM),
]


@pytest.mark.gpu
@pytest.mark.parametrize("vcase", VALIDITY_CASES, ids=[v[0] for v in VALIDITY_CASES])
def test_validity(srlib, cuda, sms, vcase):
    """Invalidated rows on one tie-heavy store: the winners' lowest members, a whole segment and a whole tile, and all
    but fewer than k rows."""
    import torch
    name, b, k, route = vcase
    n, d, off = 20000, 136, 500
    assert plan(srlib, b, n, d, k)["route"] == route
    if name == "fused-grouped":
        assert fused_grouped(b, n, sms)
    hot = hot_rows(n)
    rows = grid_store(torch, "same", n, d, 7, hot)
    q = grid_queries(torch, b, d, 7)
    qh = q.cpu().numpy()
    valid = np.ones(n, dtype=bool)
    c = make_cache(srlib, rows, d, off)

    def invalidate_and_check(drop, what):
        for r in drop:
            c.invalidate(int(r))
        valid[list(drop)] = False
        idx, sc = c.topk(qh, k)
        oi, os_ = exact_topk(q, rows, k, valid=torch.from_numpy(valid).to(cuda), id_offset=off)
        check_exact(idx, sc, oi.cpu().numpy(), os_.cpu().numpy(), f"{name}: {what}")
        return idx

    idx = invalidate_and_check([hot[0], hot[1], 0, 1], "lowest HOT rows and lowest tied rows invalidated")
    assert idx[0, 0] == hot[2] + off
    invalidate_and_check(range(SEGMENT, 2 * SEGMENT), "segment 1 invalidated")
    invalidate_and_check(range(256, 512), "tile 1 invalidated")
    keep = [5, 7000, n - 1]                                                  # fewer than k valid rows remain
    idx = invalidate_and_check([r for r in np.flatnonzero(valid) if r not in keep], "all but three rows invalidated")
    assert (idx[:, 3:] == -1).all() and (idx[:, :3] == np.array(keep) + off).all()
    c.close()


@pytest.mark.gpu
def test_empty_store(srlib, cuda):
    c = srlib.Cache(16, 64, id_offset=100)
    for b, k in ((1, 1), (4, 64), (64, 8), (300, 9)):
        assert plan(srlib, b, 0, 64, k)["route"] == ROUTE_EMPTY
        idx, sc = c.topk(np.full((b, 64), 1.0 / 16, np.float32), k)
        assert (idx == -1).all() and np.isneginf(sc).all()
    c.close()


@pytest.mark.gpu
def test_stage2_refusal_is_clean(srlib, cuda):
    """More stage-2 candidates than 200 KB of shared memory hold (B <= 4 or k > 8 over > 3.28 M rows at k = 64): an
    error before any launch, and the cache keeps serving; the same all-tied store at k = 8 returns rows 0..7."""
    n, d = 400 * SEGMENT + 1000, 8
    assert plan(srlib, 1, n, d, 64)["route"] == ROUTE_REFUSED
    c = srlib.Cache(n, d, id_offset=1)
    c.add(np.zeros((n, d), np.float32))
    q = np.full((1, d), 1.0 / 16, np.float32)
    with pytest.raises(srlib.SrError):
        c.topk(q, 64)
    idx, sc = c.topk(q, 8)
    assert idx.tolist() == [list(range(1, 9))] and (sc == 0).all()
    c.close()


def _shards(n, bounds):
    return list(zip(bounds[:-1], bounds[1:]))


@pytest.mark.gpu
@pytest.mark.parametrize("b,k", [(3, 16), (64, 8), (130, 33)])
def test_sharded_merge_exact(srlib, cuda, b, k):
    """A tie-heavy store split into four unequal shards (the first holds fewer than k rows; HOT rows sit on a shard
    boundary): the host merge of the per-shard lists equals the unsharded top-k exactly."""
    import torch
    n, d = 30000, 128
    bounds = [0, 5, 9000, 22000, n]
    hot = hot_rows(n) + [8999, 9000]
    rows = grid_store(torch, "pool", n, d, 21, sorted(hot), pool=8)
    q = grid_queries(torch, b, d, 21)
    qh = q.cpu().numpy()
    parts_i, parts_s = [], []
    for lo, hi in _shards(n, bounds):
        c = make_cache(srlib, rows[lo:hi], d, id_offset=lo)
        i, s = c.topk(qh, k)
        parts_i.append(i); parts_s.append(s)
        c.close()
    assert (parts_i[0][:, 5:] == -1).all()
    mi, ms = srlib.merge_topk(parts_i, parts_s)
    oi, os_ = exact_topk(q, rows, k)
    check_exact(mi, ms, oi.cpu().numpy(), os_.cpu().numpy(), "host merge")


@pytest.mark.gpu
@pytest.mark.parametrize("g,b,k", [(4, 64, 8), (96, 8, 64)])
def test_sharded_packed_merge_exact(srlib, cuda, g, b, k):
    """The device exchange form: sr_cache_topk_packed_dev per shard into one [G][B][k] pair buffer, then
    sr_cache_merge_packed_dev, all on the caller's stream.  G = 96, k = 64 fills exactly the merge's 48 KB of shared
    memory; one more shard is refused."""
    import torch
    L = srlib.lib()
    d = 64
    rng = np.random.default_rng(g)
    sizes = [5] + rng.integers(20, 400 if g > 4 else 12000, g - 1).tolist()
    bounds = np.concatenate([[0], np.cumsum(sizes)]).tolist()
    n = bounds[-1]
    hot = sorted({r for r in hot_rows(n) + [bounds[1], bounds[2] - 1, bounds[2]] if r < n})
    rows = grid_store(torch, "pool", n, d, 31 + g, hot, pool=8)
    q = grid_queries(torch, b, d, 31 + g)
    q16 = q.to(torch.float16).contiguous()
    pairs = torch.empty((g + 1, b, k, 2), dtype=torch.int32, device=cuda)
    out_i = torch.empty((b, k), dtype=torch.int32, device=cuda)
    out_s = torch.empty((b, k), dtype=torch.float32, device=cuda)
    caches = [make_cache(srlib, rows[lo:hi], d, id_offset=lo) for lo, hi in _shards(n, bounds)]
    torch.cuda.synchronize()
    stream = torch.cuda.Stream(device=cuda)          # one caller stream orders the scans, the packing and the merge
    h = stream.cuda_stream
    for s, c in enumerate(caches):
        assert L.sr_cache_topk_packed_dev(c.handle, q16.data_ptr(), b, k, pairs[s].data_ptr(), h) == 0
    assert L.sr_cache_merge_packed_dev(0, pairs.data_ptr(), g, b, k, out_i.data_ptr(), out_s.data_ptr(), h) == 0
    if g * k * 8 == SMEM_DEFAULT:
        assert L.sr_cache_merge_packed_dev(0, pairs.data_ptr(), g + 1, b, k, out_i.data_ptr(), out_s.data_ptr(), h) == -1
    stream.synchronize()
    for c in caches:
        c.close()
    assert (pairs[0, :, 5:, 1] == -1).all()
    oi, os_ = exact_topk(q, rows, k)
    check_exact(out_i.cpu().numpy(), out_s.cpu().numpy(), oi.cpu().numpy(), os_.cpu().numpy(), "packed merge")


UNIT_CASES = [   # (id, B, N, D, k, route, fused schedule)
    ("gemv", 3, 70001, 384, 16, ROUTE_GEMV, None),
    ("fused", 64, 20000, 256, 8, ROUTE_FUSED, "contiguous"),
    ("fused-grouped", 300, 20000, 256, 8, ROUTE_FUSED, "grouped"),
    ("gemm", 16, 20000, 256, 10, ROUTE_GEMM, None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("ucase", UNIT_CASES, ids=[u[0] for u in UNIT_CASES])
def test_unit_vectors(srlib, cuda, sms, ucase):
    """Realistic data on each route: fp16 unit vectors, half the queries perturbed copies of stored rows.  Ids exact
    against the float64 oracle; scores to fp32 accumulation error."""
    import torch
    name, b, n, d, k, route, sched = ucase
    _assert_route(srlib, sms, (name, b, n, d, k, None, 0, route, 0 if route == ROUTE_FUSED else 1, sched))
    rng = np.random.default_rng(n + d + b)
    rows = synth.make_cache(rng, n, d).astype(np.float16).astype(np.float32)
    q, src = synth.make_queries(rng, rows, b)
    q = q.astype(np.float16).astype(np.float32)
    c = srlib.Cache(n, d, id_offset=17)
    c.add(rows)
    idx, sc = c.topk(q, k)
    c.close()
    oi, os_ = exact_topk(torch.from_numpy(q).to(cuda), torch.from_numpy(rows).to(cuda), k, id_offset=17)
    assert np.array_equal(idx, oi.cpu().numpy())
    assert np.abs(sc - os_.cpu().numpy()).max() < 1e-5
    assert (idx[:len(src), 0] == src + 17).all()
