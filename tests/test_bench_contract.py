"""bench.py's line contract, on the CPU: the reference arm (`--impl reference`, the oracle port timed on the host cores)
prints ONE JSON line with the keys the driver reads; without a GPU the own arm refuses instead of falling back."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=ROOT,
                          env=e, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--workload", "modernbert-6l-b64-s128", "--steps", "2", "--warmup", "1",
              "--ref-prompts-per-step", "2"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    for key in ("metric", "value", "unit", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "e2e", "cpu_baseline"):
        assert key in d, key
    assert d["value"] > 0 and d["higher_is_better"] is True and d["config"]["workload"] == "modernbert-6l-b64-s128"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert abs(d["e2e"]["value"] - d["value"]) < 1e-9 and d["e2e"]["unit"] == d["unit"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"] and abs(cb["value"] - d["value"]) < 1e-9


def test_reference_arm_cache_workload_same_config_keys():
    """The cache workloads (BASELINE cfg 4) go through the same contract: the CPU arm times the C restatement of the Go
    scalar scan; `config` is built by one function for both arms (bench.config_of), so their keys cannot drift apart."""
    sys.path.insert(0, ROOT)
    import bench
    r = _run(["--impl", "reference", "--workload", "cache-64k-768-b256", "--steps", "1", "--warmup", "0"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert d["config"] == bench.config_of("cache-64k-768-b256", bench.WORKLOADS["cache-64k-768-b256"], 1)
    want = bench.config_of("modernbert-base-b256-s512", bench.WORKLOADS["modernbert-base-b256-s512"], 8)
    assert want["batch_per_gpu"] == 256 and want["seq_len"] == 512 and want["global_batch"] == 2048


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--workload", "modernbert-6l-b64-s128", "--gpus", "2", "--steps", "1", "--warmup", "0"],
             env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(srlib, cuda, tmp_path):
    """--dump-outputs: two runs with the same arguments write identical arrays, `steps` in the line is the --steps
    asked for, and the arrays are what the host-buffer call returns to its caller for the same seeded batch."""
    sys.path.insert(0, ROOT)
    import bench
    workload = "modernbert-6l-b64-s128"
    names = ("logits", "probs", "cls", "conf")
    runs = []
    for i, steps in enumerate((2, 3)):
        d = tmp_path / f"run{i}"
        r = _run(["--workload", workload, "--steps", str(steps), "--warmup", "1", "--no-cpu-baseline", "--no-text-e2e",
                  "--dump-outputs", str(d)])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in names)
        runs.append({n: np.load(d / (n + ".npy")) for n in names})
    for n in names:
        assert runs[0][n].dtype in (np.float32, np.float64) and np.array_equal(runs[0][n], runs[1][n]), n
    wl = bench.WORKLOADS[workload]
    _, wdir = bench.make_model_dir(wl, workload)
    ids, cu = bench.make_batch(wl, 1000)
    m = srlib.Model(wdir, device=0)
    want = m.classify_packed(ids, cu)
    m.close()
    assert runs[0]["logits"].shape == (wl["batch"], wl["classes"])
    for n in names:
        assert np.array_equal(runs[0][n], want[n].astype(runs[0][n].dtype)), n


def test_dump_outputs_refused_where_it_has_no_meaning(tmp_path):
    r = _run(["--impl", "reference", "--workload", "modernbert-6l-b64-s128", "--steps", "1", "--warmup", "0",
              "--dump-outputs", str(tmp_path / "d")])
    assert r.returncode == 2 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


def test_own_arm_refuses_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = _run(["--workload", "modernbert-6l-b64-s128", "--steps", "1", "--warmup", "1"])
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)
