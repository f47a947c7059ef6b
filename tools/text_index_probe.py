#!/usr/bin/env python3
"""Throughput of oi_index_build_bm25_text (post text -> vocabulary + BM25 CSR on the device) next to the host
IndexBuilder on the same posts, with CSR equality checked.

Corpus: seeded, about 2M posts / 300 MB, words drawn from a Zipf vocabulary of about 1M distinct [0-9a-z] words of 2..14
characters (so the sort sees many distinct keys and many keys shared by long words), every fifth word capitalised and
some posts ending in punctuation.  Prints one JSON line:
  * host_builder_s: hostlib.IndexBuilder add + finish (one CPU thread),
  * gpu_call_s: the blocking C call, host clock (includes the host -> device copy of the text from pageable memory),
  * h2d_ms / kernels_ms: device time of the copies and of the kernels of one call (torch.profiler, a separate call),
  * gpu_text_MBps / gpu_tokens_per_s: over the kernel time alone, and over the whole call,
  * top_kernels_ms: the kernels that dominate,
  * csr_equal / vocab_equal: against the host builder.
The card name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def corpus(n_posts, n_words, seed):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789", dtype=np.uint8)
    lens = rng.integers(2, 15, size=n_words)
    chars = rng.choice(alpha, size=int(lens.sum()))
    cut = np.concatenate([[0], np.cumsum(lens)])
    words = [chars[cut[i]:cut[i + 1]].tobytes().decode() for i in range(n_words)]
    caps = [w.capitalize() for w in words]
    p = 1.0 / np.arange(1, n_words + 1) ** 1.05
    ntok = np.clip(rng.lognormal(2.75, 0.6, size=n_posts).astype(np.int64), 2, 200)
    ids = rng.choice(n_words, size=int(ntok.sum()), p=p / p.sum())
    texts, at = [], 0
    for k in ntok.tolist():
        seg = ids[at:at + k].tolist()
        at += k
        texts.append(" ".join(caps[w] if j % 5 == 0 else words[w] for j, w in enumerate(seg)) + ("!" if k % 3 == 0 else ""))
    return texts, int(ntok.sum())


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # the card is named in the output either way
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--posts", type=int, default=2_000_000)
    ap.add_argument("--words", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch
    import openintel_b200 as oi
    from openintel_b200 import capi, hostlib
    t0 = time.perf_counter()
    texts, n_tokens = corpus(a.posts, a.words, 11)
    gen_s = time.perf_counter() - t0
    blob, offs = capi.pack_texts(texts)
    n_bytes = int(offs[-1])

    b = hostlib.IndexBuilder()
    t0 = time.perf_counter()
    for i in range(0, len(texts), 65536):
        b.add(texts[i:i + 65536])
    csr = b.finish()
    host_s = time.perf_counter() - t0

    ix = oi.GpuIndex(n_docs=len(texts), dim=16, max_k=10, max_batch=1)
    L = ix.L
    nt, nb = C.c_uint32(), C.c_uint64()

    def call():
        ix._ck(L.oi_index_build_bm25_text(ix.h, blob.ctypes.data, offs.ctypes.data, len(texts), C.byref(nt), C.byref(nb)))

    call()  # warm-up: module load, cub's first calls
    times = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        call()
        times.append(time.perf_counter() - t0)
    gpu_s = min(times)

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        call()
    h2d_us = kern_us = 0.0
    per = {}
    for e in prof.key_averages():
        dt = getattr(e, "self_device_time_total", None)
        if dt is None:
            dt = getattr(e, "self_cuda_time_total", 0.0)
        if "Memcpy HtoD" in e.key:
            h2d_us += dt
        elif dt and "Memcpy" not in e.key and "Memset" not in e.key:
            kern_us += dt
            per[e.key[:80]] = per.get(e.key[:80], 0.0) + dt
    top = dict(sorted(((k, round(v / 1e3, 3)) for k, v in per.items()), key=lambda kv: -kv[1])[:8])

    ix.n_terms = nt.value
    vb = np.empty(max(nb.value, 1), dtype=np.uint8)
    vo = np.empty(nt.value + 1, dtype=np.uint64)
    ix._ck(L.oi_index_read_vocabulary(ix.h, vb.ctypes.data, vo.ctypes.data))
    to = np.empty(nt.value + 1, dtype=np.uint64)
    P = int(csr["term_offsets"][-1]) if nt.value == csr["n_terms"] else 0
    di, tf, dl = np.empty(P, np.uint32), np.empty(P, np.uint32), np.empty(len(texts), np.uint32)
    csr_equal = False
    if nt.value == csr["n_terms"]:
        ix._ck(L.oi_index_read_bm25(ix.h, to.ctypes.data, di.ctypes.data, tf.ctypes.data, dl.ctypes.data, None))
        csr_equal = all(np.array_equal(x, csr[f]) for x, f in ((to, "term_offsets"), (di, "doc_ids"), (tf, "tfs"), (dl, "doc_len")))
    raw = vb.tobytes()
    vocab_equal = nt.value == csr["n_terms"] and all(raw[vo[t]:vo[t + 1]].decode() == b.term(t) for t in range(nt.value))
    ix.close()
    b.close()
    torch.cuda.synchronize()
    print(json.dumps({
        "workload": "oi_index_build_bm25_text: %d posts, %.1f MB of text, %d tokens, %d terms, %d postings" % (
            len(texts), n_bytes / 1e6, n_tokens, csr["n_terms"], len(csr["doc_ids"])),
        "gpu": gpu_info(), "corpus_gen_s": round(gen_s, 2),
        "host_builder_s": round(host_s, 3), "host_builder_MBps": round(n_bytes / host_s / 1e6, 1),
        "gpu_call_s": round(gpu_s, 4), "gpu_call_reps_s": [round(t, 4) for t in times],
        "h2d_ms": round(h2d_us / 1e3, 3), "h2d_share_of_call": round(h2d_us / 1e6 / gpu_s, 3),
        "kernels_ms": round(kern_us / 1e3, 3),
        "gpu_text_MBps_kernels": round(n_bytes / (kern_us / 1e6) / 1e6, 1) if kern_us else None,
        "gpu_tokens_per_s_kernels": round(n_tokens / (kern_us / 1e6)) if kern_us else None,
        "gpu_text_MBps_call": round(n_bytes / gpu_s / 1e6, 1), "speedup_call_vs_host": round(host_s / gpu_s, 1),
        "top_kernels_ms": top, "csr_equal": bool(csr_equal), "vocab_equal": bool(vocab_equal),
        "n_terms": nt.value}), flush=True)


if __name__ == "__main__":
    main()
