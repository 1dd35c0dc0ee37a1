#!/usr/bin/env python
"""bench.py -- prompts/sec classified by the B200 signal-extraction path (BASELINE.json metric).

A "step" = one pass of the hot path (encoder forward + sequence head) over one batch of synthetic prompts.
Workload at every N: BASELINE.json configs[1] per GPU -- ModernBERT-base intent classifier (L22 H768 I1152
V50368, 14 classes), batch 256, seq 512, all sequences full length; weak scaling (each rank classifies its own
batch; no data-path collective: prompts are independent, SURVEY.md 8e).

  value  : kernel-only throughput, ids resident in HBM, CUDA-event timed on the launching stream
  e2e    : the same metric through the C-ABI host-buffer call (sr_classify_ids): pinned-host -> device copy of
           the ids and device -> host read of probabilities/classes inside the timed region
  roofline: dominant kernel = the tcgen05 GEMM launch with the most time; algorithmic FLOPs / CUDA-event time
  cpu_baseline / --impl reference: the oracle restatement of the reference's candle CPU path (torch fp32 CPU,
           one prompt per call = the reference's operating mode) on the box's host cores.
  text_e2e : 256 UTF-8 texts through the reference-facing TEXT call (`classify_batch` of libonnx_semantic_router: the
           host tokenizer sits inside the timed call), reported beside e2e with the host threads that tokenised.

Other workloads (`--workload`, not the headline): `cache-1m-768-b1024` / `cache-1m-768-b1` = BASELINE cfg 4, the
semantic-cache cosine top-8 over 1 M x 768 fp16 rows; under torchrun the rows are sharded over the ranks, every rank
scans its shard for the whole query batch and ONE NCCL all-gather of 8-byte {score, id} entries + a device merge give
every rank the global result (checked against the unsharded scan).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "modernbert-base-b256-s512": dict(batch=256, seq=512, layers=22, vocab=50368, classes=14),
    # smaller variants for quick checks (NOT the headline configuration)
    "modernbert-base-b32-s512": dict(batch=32, seq=512, layers=22, vocab=50368, classes=14),
    "modernbert-base-b16-s512": dict(batch=16, seq=512, layers=22, vocab=50368, classes=14),
    "modernbert-base-b64-s512": dict(batch=64, seq=512, layers=22, vocab=50368, classes=14),
    "modernbert-base-b128-s512": dict(batch=128, seq=512, layers=22, vocab=50368, classes=14),
    "modernbert-6l-b64-s128": dict(batch=64, seq=128, layers=6, vocab=4096, classes=14),
    # BASELINE cfg 4: semantic-cache scan, N stored unit vectors (fp16 in HBM), B queries per step, top-k
    "cache-1m-768-b1024": dict(kind="cache", rows=1_000_000, dim=768, batch=1024, k=8),
    "cache-1m-768-b1": dict(kind="cache", rows=1_000_000, dim=768, batch=1, k=8),
    "cache-64k-768-b256": dict(kind="cache", rows=65_536, dim=768, batch=256, k=8),   # quick check
    # BASELINE cfg 5: Poisson stream, lengths log-uniform [64, 2048], classify + cache lookup per request (tools/stream_harness.py)
    "stream-cfg5": dict(kind="stream", batch=256, seq=2048, layers=22, vocab=50368, classes=14, rows=1_000_000, k=8, embed_layers=6),
    "stream-small": dict(kind="stream", batch=256, seq=2048, layers=22, vocab=50368, classes=14, rows=65_536, k=8, embed_layers=6),
}
PC_NAMES = ["embed", "norm", "gemm_qkv", "attention", "gemm_attn_out", "gemm_mlp_in", "gemm_mlp_out", "head"]


def algorithmic_flops_per_token(cfg, seq):
    """SURVEY.md 8(d): linear layers + attention, sliding window exploited, padding excluded."""
    H, I, L = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
    lin = 2 * (3 * H * H + H * H + 2 * I * H + H * I)
    tot = 0
    for li in range(L):
        local = (li % cfg.global_attn_every_n_layers) != 0
        sk = min(seq, cfg.local_attention + 1) if local else seq
        tot += lin + 4 * H * sk
    return tot


def make_model_dir(wl, tag):
    from oracle import encoder_oracle as eo, synth
    cfg = eo.ModernBertConfig(vocab_size=wl["vocab"], num_hidden_layers=wl["layers"],
                              max_position_embeddings=max(1024, wl["seq"]), pad_token_id=0)
    d = os.path.join(tempfile.gettempdir(), f"srb_bench_{tag}")
    marker = os.path.join(d, ".complete")
    if not os.path.exists(marker):
        w = synth.make_modernbert_weights(cfg, wl["classes"], seed=1234)
        synth.write_model_dir(d, cfg, w, {i: f"cat{i}" for i in range(wl["classes"])})
        open(marker, "w").write("ok")
    return cfg, d


def make_batch(wl, seed):
    from oracle import synth
    rng = np.random.default_rng(seed)
    seqs = synth.make_ids(rng, [wl["seq"]] * wl["batch"], wl["vocab"])
    ids = np.ascontiguousarray(np.concatenate(seqs).astype(np.int32))
    cu = (np.arange(wl["batch"] + 1) * wl["seq"]).astype(np.int32)
    return ids, cu


def config_of(workload, wl, world):
    """The `config` object both arms print (same keys, same values: the driver compares them)."""
    if wl.get("kind") == "cache":
        return {"workload": workload, "rows": wl["rows"], "dim": wl["dim"], "queries_per_step": wl["batch"], "top_k": wl["k"],
                "store_dtype": "f16 (GPU arm) / f32 (CPU arm, as pkg/cache holds it)",
                "sharding": f"rows over {world} rank(s), queries replicated", "n_ranks": world}
    return {"workload": workload, "model": "ModernBERT-base (random init)", "batch_per_gpu": wl["batch"],
            "seq_len": wl["seq"], "layers": wl["layers"], "classes": wl["classes"], "global_batch": world * wl["batch"],
            "parallelism": f"dp{world} (independent prompts, no collective)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads():
    """Threads the CPU arm can really use: affinity mask, capped by the cgroup CPU quota when one is set."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return int(os.environ.get("SR_B200_CPU_THREADS", min(n, 64)))


class CpuReference:
    """Oracle (torch fp32 CPU) in the reference's operating mode: one prompt per call, seq = wl['seq']."""

    def __init__(self, cfg, wdir, wl):
        import torch
        from safetensors.numpy import load_file
        from oracle import encoder_oracle as eo
        from oracle import synth
        torch.set_num_threads(host_threads())
        self.torch, self.eo, self.cfg = torch, eo, cfg
        self.wt = {k: torch.from_numpy(v) for k, v in load_file(os.path.join(wdir, "model.safetensors")).items()}
        rng = np.random.default_rng(99)
        self.seqs = synth.make_ids(rng, [wl["seq"]] * 64, wl["vocab"])
        self.i = 0

    def one(self):
        s = self.seqs[self.i % len(self.seqs)]
        self.i += 1
        with self.torch.no_grad():
            self.eo.modernbert_classify(self.wt, self.cfg, self.torch.from_numpy(s[None].astype(np.int64)),
                                        self.torch.ones(1, len(s), dtype=self.torch.long))

    def run(self, n):
        t0 = time.perf_counter()
        for _ in range(n):
            self.one()
        return time.perf_counter() - t0


def cpu_reference_prompts_per_s(cfg, wdir, wl, budget_s):
    ref = CpuReference(cfg, wdir, wl)
    t1 = ref.run(1)                                   # warm-up + estimate
    if t1 > budget_s / 2:                             # very slow host: the estimate is the sample
        return 1.0 / t1, 1, t1
    n = int(max(1, min(64, budget_s / max(t1, 1e-3))))
    dt = ref.run(n)
    return n / dt, n, dt


def cache_data(wl, device=None):
    """Seeded synthetic cfg 4 data (SURVEY 8d): N unit vectors rounded to fp16, B queries = half perturbed copies of stored
    rows (|noise| = 0.1), half fresh.  Returns (store fp32 numpy [N,D] holding fp16-representable values, queries fp32)."""
    n, d, b = wl["rows"], wl["dim"], wl["batch"]
    rng = np.random.default_rng(1234)
    store = np.empty((n, d), dtype=np.float32)
    for i in range(0, n, 131072):
        blk = rng.standard_normal((min(131072, n - i), d), dtype=np.float32)
        blk /= np.linalg.norm(blk, axis=1, keepdims=True)
        store[i:i + blk.shape[0]] = blk.astype(np.float16).astype(np.float32)
    nb = b // 2
    q = np.empty((b, d), dtype=np.float32)
    if nb:
        noise = rng.standard_normal((nb, d), dtype=np.float32)
        noise *= 0.1 / np.linalg.norm(noise, axis=1, keepdims=True)
        q[:nb] = store[rng.integers(0, n, nb)] + noise
    q[nb:] = rng.standard_normal((b - nb, d), dtype=np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    return store, q


def cpu_cache_queries_per_s(store, q, budget_s):
    """oracle/cache_scan.c: the Go scalar scan (pkg/cache/inmemory_cache_search.go:14-20,65-89), OpenMP over queries."""
    from oracle import cache_oracle as co
    co.build_c()
    nt = host_threads()
    qs = np.ascontiguousarray(np.resize(q, (max(nt, 1), q.shape[1])))
    t0 = time.perf_counter()
    co.scan_linear_c(qs[:1], store, 1)                    # one query on one thread: the estimate
    t1 = time.perf_counter() - t0
    rounds = int(max(1, min(8, budget_s / max(t1, 1e-3))))
    qs = np.ascontiguousarray(np.resize(q, (rounds * nt, q.shape[1])))
    t0 = time.perf_counter()
    co.scan_linear_c(qs, store, nt)
    dt = time.perf_counter() - t0
    return len(qs) / dt, len(qs), dt, nt


def run_reference_cache(args, wl, rank, world):
    if rank != 0:
        return
    store, q = cache_data(wl)
    from oracle import cache_oracle as co
    co.build_c()
    nt = host_threads()
    per_step = max(nt, 1)
    qs = np.ascontiguousarray(np.resize(q, (per_step, q.shape[1])))
    for _ in range(min(args.warmup, 1)):
        co.scan_linear_c(qs, store, nt)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        co.scan_linear_c(qs, store, nt)
    t_tot = time.perf_counter() - t0
    v = per_step * args.steps / t_tot
    sample = f"{per_step} queries/step x {args.steps} steps, one Go-equivalent scalar scan of the {wl['rows']} x {wl['dim']} f32 store per query, {nt} threads"
    print(json.dumps({
        "impl": "reference", "metric": "cache lookups/sec (cosine top-k over the store)", "value": v, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, wl, world),
        "cpu_baseline": {"value": v, "unit": "queries/s", "cores": nt, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_reference(args, wl, rank, world):
    if wl.get("kind") == "cache":
        return run_reference_cache(args, wl, rank, world)
    if wl.get("kind") == "stream":
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "cfg 5 is a GPU serving harness; the CPU arm of its two stages is --workload modernbert-base-b256-s512 / cache-1m-768-b1024"}))
        return
    if rank != 0:
        return
    cfg, wdir = make_model_dir(wl, args.workload)
    per_step = max(1, args.ref_prompts_per_step)
    ref = CpuReference(cfg, wdir, wl)
    for _ in range(args.warmup):
        ref.run(1)
    t_tot = sum(ref.run(per_step) for _ in range(args.steps))
    n_tot = per_step * args.steps
    v = n_tot / t_tot
    cores = host_threads()
    sample = f"{per_step} prompts/step x {args.steps} steps, seq {wl['seq']}, one prompt per call (reference operating mode)"
    print(json.dumps({
        "impl": "reference", "metric": "prompts/sec classified", "value": v, "unit": "prompts/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, wl, world),
        "cpu_baseline": {"value": v, "unit": "prompts/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "prompts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def device_to_host(ptr, shape, typestr):
    """Host copy of a contiguous array in the library's device memory, read through the CUDA array interface."""
    import torch

    class DeviceView:
        __cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 3}
    return torch.as_tensor(DeviceView(), device="cuda").cpu().numpy()


def dump_step_outputs(out_dir, L, h, B, Cn, prefix):
    """What the last timed step left in the model's result buffers, i.e. what sr_classify_ids hands its caller:
    logits / probs [B, C], cls / conf [B]; float32, cls as float64 (exact for class ids)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"logits": device_to_host(L.sr_dev_logits(h), (B, Cn), "<f4"),
              "probs": device_to_host(L.sr_dev_probs(h), (B, Cn), "<f4"),
              "cls": device_to_host(L.sr_dev_cls(h), (B,), "<i4").astype(np.float64),
              "conf": device_to_host(L.sr_dev_conf(h), (B,), "<f4")}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def text_e2e_classify(wl, wdir, local_rank, steps):
    """256 texts -> `classify_batch` of libonnx_semantic_router (the reference's only true batch text entry,
    onnx-binding/semantic-router.go:119): tokenizer + H2D + forward + head + D2H inside the timed call."""
    import semantic_router_b200 as pkg
    from oracle import tokenizer_fixtures as tf

    class ClsRes(C.Structure):   # ClassificationResultFFI, onnx-binding/semantic-router.go:63-71
        _fields_ = [("label", C.c_char_p), ("class_id", C.c_int), ("confidence", C.c_float), ("num_classes", C.c_int),
                    ("probabilities", C.POINTER(C.c_float)), ("processing_time_ms", C.c_float), ("error", C.c_bool)]
    tok_path = os.path.join(wdir, "tokenizer.json")
    if not os.path.exists(tok_path):
        tmp = tok_path + f".{os.getpid()}.tmp"
        tf.BUILDERS["modernbert"](tmp)
        os.replace(tmp, tok_path)
    rng = np.random.default_rng(3)
    words = ["".join(chr(97 + int(c)) for c in rng.integers(0, 26, int(rng.integers(2, 10)))) for _ in range(5000)]
    n = wl["batch"]
    texts = [" ".join(words[int(j)] for j in rng.integers(0, len(words), 420)) for _ in range(n)]   # > seq tokens: truncated to 512
    os.environ["SR_B200_DEVICE"] = str(local_rank)          # one process per GPU: this rank's slot lives on its GPU
    X = C.CDLL(os.path.join(os.path.dirname(pkg.LIB_PATH), "libonnx_semantic_router.so"))
    X.init_sequence_classifier.argtypes = [C.c_char_p, C.c_char_p, C.c_bool]
    X.init_sequence_classifier.restype = C.c_bool
    X.classify_batch.argtypes = [C.c_char_p, C.POINTER(C.c_char_p), C.c_int, C.POINTER(ClsRes)]
    X.free_classification_result.argtypes = [C.POINTER(ClsRes)]
    if not X.init_sequence_classifier(b"bench_intent", wdir.encode(), True):
        return None
    arr = (C.c_char_p * n)(*[t.encode() for t in texts])
    res = (ClsRes * n)()

    def once():
        if X.classify_batch(b"bench_intent", arr, n, res) != 0:
            raise RuntimeError("classify_batch failed")
        for i in range(n):
            X.free_classification_result(C.byref(res[i]))
    for _ in range(3):
        once()
    t0 = time.perf_counter()
    for _ in range(steps):
        once()
    dt = time.perf_counter() - t0
    return {"seconds": dt, "texts": n * steps, "text_bytes": int(np.mean([len(t) for t in texts])),
            "host_threads": host_threads()}


def main_cache(args, wl, rank, world, local_rank):
    """BASELINE cfg 4: cosine top-k of B queries over N stored unit vectors; rows sharded over the ranks when world > 1."""
    import importlib
    import torch
    import torch.distributed as dist
    import semantic_router_b200 as pkg
    sh = importlib.import_module("semantic-router_b200.sharding")
    L = pkg.lib()
    L.sr_launch_count.restype = C.c_longlong
    N, D, B, K = wl["rows"], wl["dim"], wl["batch"], wl["k"]
    store, q = cache_data(wl)
    lo, hi = sh.shard_range(N, rank, world)
    shard = pkg.Cache(hi - lo, D, device=local_rank, id_offset=lo)           # results carry GLOBAL ids
    for i in range(lo, hi, 250_000):
        shard.add(store[i:min(i + 250_000, hi)])
    d_q16 = torch.from_numpy(q).cuda().half().contiguous()
    q_pinned = torch.from_numpy(q).pin_memory()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    sp = C.c_void_p(stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()

    def scan_only():        # this rank's shard, results stay in the cache's device buffers
        if L.sr_cache_topk_dev(shard.handle, C.c_void_p(d_q16.data_ptr()), B, K, sp) != 0:
            raise RuntimeError("sr_cache_topk_dev failed")

    def step_dev():         # the whole lookup on the device: scan (+ pack, all-gather, merge when sharded)
        if world > 1:
            return sh.sharded_topk_dev(shard, d_q16, K)
        scan_only()
        return None

    for _ in range(max(3, args.warmup)):
        step_dev()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.sr_launch_count()
    barrier(); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step_dev()
    ev1.record(stream)
    torch.cuda.synchronize(); barrier()
    ms = ev0.elapsed_time(ev1)
    launches = L.sr_launch_count() - launches0
    # the timed region of this workload can be shorter than one nvidia-smi period (100 ms): the same loop keeps running
    # until the sampler has seen the GPU under this load for >= 0.5 s, then it stops
    t_keep = time.perf_counter()
    while time.perf_counter() - t_keep < 0.5:
        for _ in range(args.steps):
            step_dev()
        torch.cuda.synchronize()
    clocks = dict(sampler.stop(), note="sampled while the timed loop kept repeating (>= 0.5 s)")
    # the scan alone (the dominant kernel: fused top-k GEMM at B > 4, GEMV at B <= 4; + the short list merge)
    ka, kb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ka.record(stream)
    for _ in range(args.steps):
        scan_only()
    kb.record(stream)
    torch.cuda.synchronize()
    scan_ms = ka.elapsed_time(kb) / args.steps
    t = torch.tensor([ms, scan_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, scan_ms_max = float(t[0].item()), float(t[1].item())
    value = B * args.steps / (ms_max / 1e3)

    # ---- e2e: queries in pinned host memory -> device, lookup, merged ids / scores back on the host
    def step_e2e():
        if world == 1:
            return shard.topk(q, K)                                       # the C-ABI host-buffer call (sr_cache_topk)
        dq = q_pinned.to("cuda", non_blocking=True).half()
        oi, os_ = sh.sharded_topk_dev(shard, dq, K)
        return oi.cpu().numpy(), os_.cpu().numpy()
    for _ in range(2):
        out = step_e2e()
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step_e2e()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = B * args.steps / float(t.item())

    # ---- parity inside the bench: the sharded result equals the unsharded scan (rank 0 holds a full copy for the check)
    check = None
    if rank == 0:
        from oracle import cache_oracle as co
        mi, msc = out
        if world > 1:
            full = pkg.Cache(N, D, device=local_rank)
            for i in range(0, N, 250_000):
                full.add(store[i:i + 250_000])
            fi, fs = full.topk(q, K)
            full.close()
            check = {"ids_equal_unsharded": bool((mi == fi).all()), "max_score_delta": float(np.abs(msc - fs).max())}
        nchk = min(B, 4)
        oi, osc = co.topk_batch(q[:nchk], store, K)
        check = dict(check or {}, ids_equal_oracle_first_rows=bool((mi[:nchk] == oi).all()),
                     max_score_delta_oracle=float(np.abs(msc[:nchk] - osc).max()))
    if rank == 0:
        pk = peaks()
        rows_local = hi - lo
        if B > 4:
            peak = pk.get("bf16_tflops") or 1600.0
            src = "measured (MEASURED_PEAKS.json bf16_tflops: kernel timed alone)" if pk.get("bf16_tflops") else "fallback (B200_PROFILING.md)"
            ach = 2.0 * B * rows_local * D / (scan_ms_max * 1e-3) / 1e12
            roof = {"bound": "tensor", "kernel": "gemm_kernel<256,EPI_TOPK> (+ select_stage2)", "achieved": ach, "peak": peak,
                    "unit": "TFLOP/s", "frac": ach / peak, "traffic": None, "peak_source": src,
                    "flops_per_launch": 2.0 * B * rows_local * D, "ms_per_launch": scan_ms_max,
                    "algorithmic_bytes_per_launch": rows_local * D * 2 + B * D * 2 + B * K * 8}
        else:
            peak = pk.get("hbm_gbs") or 6400.0
            src = "measured (MEASURED_PEAKS.json hbm_gbs)" if pk.get("hbm_gbs") else "fallback (B200_PROFILING.md)"
            ach = (rows_local * D * 2 + B * D * 2 + B * K * 8) / (scan_ms_max * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": "scores_small_kernel (+ select_stage1/2)", "achieved": ach, "peak": peak,
                    "unit": "GB/s", "frac": ach / peak, "traffic": None, "peak_source": src,
                    "bytes_per_launch": rows_local * D * 2 + B * D * 2 + B * K * 8, "ms_per_launch": scan_ms_max}
        try:   # the committed ncu capture is of the UNSHARDED store (1 M rows on one GPU): no figure for a shard
            if world == 1 and wl["rows"] == 1_000_000:
                roof["traffic"] = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["dram_bytes_per_launch"].get(
                    "cache_topk_b1024" if B > 4 else "cache_scores_b1")
        except Exception:
            pass
        line = {
            "metric": "cache lookups/sec (cosine top-k over the store)", "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": dict(config_of(args.workload, wl, world),
                           l2_policy=f"the store shard ({rows_local * D * 2 / 1e6:.0f} MB) is streamed every step and exceeds the 126 MB L2" if rows_local * D * 2 > 126e6 else "store shard fits L2 (quick-check workload)"),
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": int(B * D * 4), "d2h_bytes_per_step": int(B * K * 8)},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
            "exchange": {"collective": "all_gather_into_tensor (NCCL)" if world > 1 else None, "bytes_per_rank": B * K * 8 if world > 1 else 0,
                         "scan_ms": scan_ms_max, "step_ms": ms_max / args.steps},
            "check": check,
        }
        if world == 1 and not args.no_cpu_baseline:
            v, n, dt, nt = cpu_cache_queries_per_s(store, q, args.cpu_budget_s)
            line["cpu_baseline"] = {"value": v, "unit": "queries/s", "cores": nt, "kind": "port",
                                    "sample": f"{n} queries, one Go-equivalent scalar scan of the {N} x {D} f32 store each (oracle/cache_scan.c), {dt:.1f} s"}
        print(json.dumps(line))
    shard.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="modernbert-base-b256-s512", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-budget-s", type=float, default=20.0)
    ap.add_argument("--ref-prompts-per-step", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-text-e2e", action="store_true")
    ap.add_argument("--qps", type=float, default=100000.0, help="stream workloads: offered load of the whole job (BASELINE cfg 5: 100 k)")
    ap.add_argument("--duration", type=float, default=3.0, help="stream workloads: seconds of arrivals per phase")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (logits, probs, cls, conf) as DIR/<name>.npy; the inputs "
                         "are seeded, so two builds run with the same arguments can be compared array for array "
                         "(under torchrun each rank writes DIR/rank<r>_<name>.npy)")
    args = ap.parse_args()
    wl = WORKLOADS[args.workload]
    if args.dump_outputs and (args.impl != "b200" or wl.get("kind")):
        ap.error("--dump-outputs covers the encoder workloads of the b200 arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU path; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    # NCCL's own log level is whatever the caller set (NCCL_DEBUG=INFO shows the rings / NVLS); its lines go to stderr so
    # that stdout stays the one JSON line
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()

    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB) or not os.path.exists(ge.LIB_ONNX):
        if local_rank == 0:
            ge.build()
        barrier()
    if wl.get("kind") == "cache":
        main_cache(args, wl, rank, world, local_rank)
        if world > 1:
            dist.destroy_process_group()
        return
    if wl.get("kind") == "stream":
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import stream_harness
        stream_harness.run(args, wl, rank, world, local_rank, sys.modules[__name__])
        if world > 1:
            dist.destroy_process_group()
        return
    if local_rank == 0:
        cfg, wdir = make_model_dir(wl, args.workload)
    barrier()
    cfg, wdir = make_model_dir(wl, args.workload)

    import semantic_router_b200 as pkg
    L = pkg.lib()
    L.sr_profile_enable.argtypes = [C.c_void_p, C.c_int]
    L.sr_profile_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.sr_launch_count.restype = C.c_longlong
    model = pkg.Model(wdir, device=local_rank)
    h = model.handle
    B, S, Cn = wl["batch"], wl["seq"], wl["classes"]
    T = B * S
    ids, cu = make_batch(wl, 1000 + rank)
    d_ids = torch.from_numpy(ids).cuda()
    d_cu = torch.from_numpy(cu).cuda()
    stream = torch.cuda.Stream()          # explicit non-default stream: kernels AND timing events live on it
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    L.sr_model_set_stream(h, C.c_void_p(stream.cuda_stream))
    assert L.sr_reserve(h, T, B, B * Cn) == 0

    def step_dev():
        rc = L.sr_forward_dev(h, d_ids.data_ptr(), d_cu.data_ptr(), B, T, S, 0)
        rc |= L.sr_head_seq_dev(h, 0, d_cu.data_ptr(), B, 0)
        if rc:
            raise RuntimeError("device step failed: " + L.sr_last_error().decode())

    for _ in range(max(3, args.warmup)):
        step_dev()
    torch.cuda.synchronize()

    # ---------------- timed region (kernel-only; inputs resident in HBM; activations >> L2 between steps).
    # Nothing but the step's own launches sits between the two events: the per-category profile runs in a second loop.
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = L.sr_launch_count()
    barrier(); torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step_dev()
    ev1.record(stream)
    torch.cuda.synchronize(); barrier()
    ms = ev0.elapsed_time(ev1)
    launches = L.sr_launch_count() - launches0
    clocks = sampler.stop()
    if args.dump_outputs:   # before anything else runs on the model: its result buffers still hold the last timed step
        dump_step_outputs(args.dump_outputs, L, h, B, Cn, "" if world == 1 else f"rank{rank}_")
    t = torch.tensor([ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * args.steps / (ms_max / 1e3)

    # ---------------- per-category device times (CUDA event pairs around each launch, same stream), OUTSIDE `value`
    prof_steps = max(2, min(args.steps, 5))
    L.sr_profile_enable(h, 1)
    for _ in range(prof_steps):
        step_dev()
    prof_ms = (C.c_float * 8)(); prof_n = (C.c_int * 8)()
    L.sr_profile_read(h, prof_ms, prof_n)
    L.sr_profile_enable(h, 0)

    # ---------------- e2e through the C-ABI host-buffer call
    L.sr_model_set_stream(h, None)
    out = model.classify_packed(ids, cu, want_logits=False)      # warm-up (allocates pinned staging)
    model.classify_packed(ids, cu, want_logits=False)
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = model.classify_packed(ids, cu, want_logits=False)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(t.item())
    h2d = ids.nbytes + cu.nbytes
    d2h = B * Cn * 4 + B * 4 + B * 4

    # ---------------- text in, labels out: the reference-facing batch call with the tokenizer inside
    text = None
    if not args.no_text_e2e:
        try:
            barrier()
            tr = text_e2e_classify(wl, wdir, local_rank, max(2, min(args.steps, 5)))
            if tr:
                t = torch.tensor([tr["seconds"]], device="cuda", dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                text = {"value": world * tr["texts"] / float(t.item()), "unit": "prompts/s",
                        "call": "classify_batch (libonnx_semantic_router), 256 texts/call truncated to 512 tokens",
                        "text_bytes_per_prompt": tr["text_bytes"], "host_threads": tr["host_threads"]}
        except Exception as e:   # the headline line must survive a failure of the secondary measurement
            text = {"error": str(e)[:200]}

    if rank == 0:
        pk = peaks()
        peak_tf = pk.get("bf16_tflops_sustained")
        peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)"
        if not peak_tf:
            peak_tf, peak_src = 1400.0, "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"
        H, I = cfg.hidden_size, cfg.intermediate_size
        gemm_flops = {2: 2 * T * 3 * H * H, 4: 2 * T * H * H, 5: 2 * T * 2 * I * H, 6: 2 * T * H * I}
        per_launch = {k: (prof_ms[k] / prof_n[k]) if prof_n[k] else None for k in gemm_flops}
        dom = max((k for k in gemm_flops if per_launch[k]), key=lambda k: prof_ms[k])
        achieved = gemm_flops[dom] / (per_launch[dom] * 1e-3) / 1e12
        traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of that kernel from the committed ncu capture
        for tf_name in ("r2_traffic.json", "r1_traffic.json"):
            try:
                traffic = json.load(open(os.path.join(ROOT, "profiles", tf_name)))["dram_bytes_per_launch"].get(PC_NAMES[dom])
                if traffic:
                    break
            except Exception:
                pass
        step_flops = algorithmic_flops_per_token(cfg, S) * T
        breakdown = {PC_NAMES[i]: {"ms_per_step": prof_ms[i] / prof_steps, "launches": prof_n[i] // max(1, prof_steps)}
                     for i in range(8)}
        line = {
            "metric": "prompts/sec classified", "value": value, "unit": "prompts/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": dict(config_of(args.workload, wl, world),
                           l2_policy="activations per step (>1 GB) exceed the 126 MB L2; no explicit flush"),
            "e2e": {"value": e2e_value, "unit": "prompts/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h)},
            "text_e2e": text,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "gemm_kernel<256," + PC_NAMES[dom] + ">", "achieved": achieved,
                         "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                         "peak_source": peak_src, "flops_per_launch": gemm_flops[dom],
                         "ms_per_launch": per_launch[dom]},
            "step_tflops": step_flops / (ms_max / args.steps * 1e-3) / 1e12,
            "step_frac_of_peak": step_flops / (ms_max / args.steps * 1e-3) / 1e12 / peak_tf,
            "breakdown": breakdown,
            "breakdown_note": f"per-category CUDA-event times from a separate profiled loop of {prof_steps} steps (not inside `value`)",
        }
        if world == 1 and not args.no_cpu_baseline:
            v, n, dt = cpu_reference_prompts_per_s(cfg, wdir, wl, args.cpu_budget_s)
            line["cpu_baseline"] = {"value": v, "unit": "prompts/s", "cores": host_threads(), "kind": "port",
                                    "sample": f"{n} prompts, seq {S}, one prompt per call, torch fp32 CPU oracle, {dt:.1f} s"}
        print(json.dumps(line))
    model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
