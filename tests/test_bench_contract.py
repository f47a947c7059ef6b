"""CPU: the driver contract of bench.py that can be checked without a GPU -- the reference arm (`--impl reference`,
which times the CPU oracle port because the reference has no implementation of this path: SURVEY.md §0) prints one
JSON line with the keys the driver reads, and the GPU arm refuses to run without the CUDA library / a GPU instead of
falling back to the CPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def test_reference_arm_line():
    # a small corpus / slice keeps the CPU suite short; the driver runs the defaults (50M docs, 1M-document slice)
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--docs", "400000", "--cpu-slice", "20000"])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    assert "hybrid" in d["metric"] and "hybrid BM25+cosine+RRF" in d["config"]["workload"] and "model" not in d["config"]
    assert d["dtype"] == "bf16" and d["config"]["n_docs"] == 400000
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["sample"]
    # every host core, also under torch.distributed.run (which exports OMP_NUM_THREADS=1: VERDICT r1)
    assert cb["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_ignores_omp_num_threads():
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", LOCAL_RANK="0", WORLD_SIZE="2")
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--docs", "400000", "--cpu-slice", "20000"], env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0)) and d["n_gpus"] == 2


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_reference_arm_dumps_the_last_timed_step(tmp_path):
    # step i scores query batch i % 4: 1 and 5 steps end on the same batch, 2 steps on another
    import numpy as np
    dumps = {}
    for steps in (1, 5, 2):
        d = tmp_path / str(steps)
        r = _run(["--impl", "reference", "--steps", str(steps), "--warmup", "1", "--docs", "400000", "--cpu-slice", "20000",
                  "--dump-outputs", str(d)])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps[steps] = {n: np.load(d / (n + ".npy")) for n in ("hybrid_ids", "hybrid_rrf", "hybrid_rank_cosine", "hybrid_rank_bm25")}
    for steps in (1, 5, 2):
        a = dumps[steps]
        assert a["hybrid_rrf"].dtype == np.float32 and a["hybrid_ids"].dtype == np.float64
        assert all(v.shape == (256, 100) for v in a.values())
        assert np.all(a["hybrid_ids"] < 20000) and np.all(np.diff(a["hybrid_rrf"], axis=1) <= 0)
        assert np.all((a["hybrid_rank_cosine"] >= 0) & (a["hybrid_rank_cosine"] <= 100))
    assert all(np.array_equal(dumps[1][n], dumps[5][n]) for n in dumps[1])
    assert not np.array_equal(dumps[1]["hybrid_ids"], dumps[2]["hybrid_ids"])


def test_steps_must_be_positive():
    r = _run(["--impl", "reference", "--steps", "0"])
    assert r.returncode != 0 and "--steps" in r.stderr


def test_gpu_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the arm would simply run")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0
    assert "value" not in r.stdout
