"""GPU: bench.py --dump-outputs writes what the last timed hybrid step returned -- the same lists the host-buffer call
gives for that step's query batch on an index built the way the benchmark builds it."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_DOCS = 300_000


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_is_the_last_timed_step(tmp_path):
    # 3 warmup + 2 timed steps: the last timed step is step 4, which runs query batch 4 % 4 = 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--repeats", "1",
                        "--docs", str(N_DOCS), "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    got = [np.load(tmp_path / (n + ".npy")) for n in ("hybrid_ids", "hybrid_rrf", "hybrid_rank_cosine", "hybrid_rank_bm25")]

    import torch
    import openintel_b200 as oi
    B = _bench_module()
    ix, _, _, cdf, _, _, _ = B.build_hybrid_index(oi, N_DOCS, 0, 1, 0, None, torch.device("cuda", 0))
    try:
        q = B._unit_queries(4, B.BATCH, B.DIM, 1234)[0].numpy()
        qt = B._zipf_queries(B.BATCH, B.QTERMS, cdf, 100)
        want = ix.search_hybrid(q, qt, B.TOPK, B.RRF_K)
    finally:
        ix.close()
    assert np.array_equal(got[0], want[0].astype(np.float64))
    assert np.array_equal(got[1].view(np.uint32), want[1].view(np.uint32))
    assert np.array_equal(got[2], want[2].astype(np.float64)) and np.array_equal(got[3], want[3].astype(np.float64))
