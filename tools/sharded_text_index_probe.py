#!/usr/bin/env python3
"""The document-sharded lift on the device next to the host path, for the corpus of tools/text_index_probe.py (about 2M
posts / 300 MB, seeded) split into G contiguous shards that all live on one GPU.

Per G, one JSON line:
  * build_s: oi_index_build_bm25_text per shard, blocking call, host clock (min over reps),
  * union_s: oi_index_bm25_union_vocabulary per shard over the G gathered vocabularies, blocking call, host clock,
  * build_kernels_ms / union_kernels_ms / union_top_kernels_ms: device time of the kernels of one build and one union of
    shard 0 (torch.profiler, separate calls),
  * host_builder_s per slice, host_union_s (sorted(set().union(...))) and host_remap_s (dict re-index, every shard):
    what store.lift_shard does on the host,
  * arrays_equal: every shard's vocabulary and CSR against the host path's.
The card name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def kernel_ms(prof):
    tot, per = 0.0, {}
    for e in prof.key_averages():
        dt = getattr(e, "self_device_time_total", None)
        if dt is None:
            dt = getattr(e, "self_cuda_time_total", 0.0)
        if dt and "Memcpy" not in e.key and "Memset" not in e.key:
            tot += dt
            per[e.key[:80]] = per.get(e.key[:80], 0.0) + dt
    top = dict(sorted(((k, round(v / 1e3, 3)) for k, v in per.items()), key=lambda kv: -kv[1])[:5])
    return round(tot / 1e3, 3), top


def host_path(texts, world):
    """store.lift_shard's work for every slice: IndexBuilder, Python union, dict remap"""
    from openintel_b200 import hostlib, sharding
    build_s, local = [], []
    for r in range(world):
        base, n = sharding.shard_range(len(texts), world, r)
        b = hostlib.IndexBuilder()
        t0 = time.perf_counter()
        for i in range(base, base + n, 65536):
            b.add(texts[i:min(i + 65536, base + n)])
        csr = b.finish()
        build_s.append(time.perf_counter() - t0)
        local.append((csr, [b.term(i) for i in range(csr["n_terms"])]))
        b.close()
    t0 = time.perf_counter()
    vocab = sorted(set().union(*(v for _, v in local)))
    union_s = time.perf_counter() - t0
    t0 = time.perf_counter()
    pos = {w: i for i, w in enumerate(vocab)}
    offs = []
    for csr, lv in local:
        gid = np.array([pos[w] for w in lv], dtype=np.int64)
        lens = np.zeros(len(vocab), dtype=np.uint64)
        lens[gid] = np.diff(csr["term_offsets"])
        off = np.zeros(len(vocab) + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        offs.append(off)
    remap_s = time.perf_counter() - t0
    return dict(build_s=build_s, union_s=union_s, remap_s=remap_s, vocab=vocab, offs=offs, local=[c for c, _ in local])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--posts", type=int, default=2_000_000)
    ap.add_argument("--words", type=int, default=1_000_000)
    ap.add_argument("--shards", default="2,8")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    import openintel_b200 as oi
    from openintel_b200 import capi, sharding
    from text_index_probe import corpus, gpu_info
    texts, n_tokens = corpus(a.posts, a.words, 11)
    info = gpu_info()
    for world in [int(x) for x in a.shards.split(",")]:
        spans = [sharding.shard_range(len(texts), world, r) for r in range(world)]
        slices = [capi.pack_texts(texts[base:base + n]) for base, n in spans]
        shards = [oi.GpuIndex(n_docs=n, dim=16, doc_base=base, max_k=10, max_batch=1) for base, n in spans]
        nt, nb = C.c_uint32(), C.c_uint64()

        def build(r):
            ix, (blob, offs) = shards[r], slices[r]
            ix._ck(ix.L.oi_index_build_bm25_text(ix.h, blob.ctypes.data, offs.ctypes.data, len(offs) - 1, C.byref(nt), C.byref(nb)))
            ix.n_terms, ix.vocab_bytes = nt.value, nb.value

        def gather():
            vp = [ix.read_vocabulary_packed() for ix in shards]
            blob = np.concatenate([b for b, _ in vp])
            lens = np.concatenate([np.diff(o.astype(np.int64)) for _, o in vp])
            return blob, np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)

        def union(r, blob, offs):
            ix = shards[r]
            ix._ck(ix.L.oi_index_bm25_union_vocabulary(ix.h, blob.ctypes.data, offs.ctypes.data, len(offs) - 1, C.byref(nt), C.byref(nb)))
            ix.n_terms, ix.vocab_bytes = nt.value, nb.value

        for r in range(world):  # warm-up: module load, cub's first calls
            build(r)
        union(0, *gather())
        build_t = [[] for _ in range(world)]
        union_t = [[] for _ in range(world)]
        for _ in range(a.reps):
            for r in range(world):
                t0 = time.perf_counter()
                build(r)
                build_t[r].append(time.perf_counter() - t0)
            blob, offs = gather()
            for r in range(world):
                t0 = time.perf_counter()
                union(r, blob, offs)
                union_t[r].append(time.perf_counter() - t0)
        n_entries, entry_bytes = len(offs) - 1, int(offs[-1])
        # kernel time of one build and one union of shard 0, profiled in calls of their own
        for r in range(world):
            build(r)
        blob, offs = gather()
        build(0)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            build(0)
        build_k, _ = kernel_ms(prof)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            union(0, blob, offs)
        union_k, union_top = kernel_ms(prof)
        for r in range(1, world):
            union(r, blob, offs)

        hp = host_path(texts, world)
        ok = True
        want_bytes = "".join(hp["vocab"]).encode()
        for r, ix in enumerate(shards):
            vb, vo = ix.read_vocabulary_packed()
            ok = ok and ix.n_terms == len(hp["vocab"]) and vb.tobytes() == want_bytes
            P = int(hp["offs"][r][-1])
            to, di, tf = np.empty(ix.n_terms + 1, np.uint64), np.empty(max(P, 1), np.uint32), np.empty(max(P, 1), np.uint32)
            dl = np.empty(ix.n_docs, np.uint32)
            ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, di.ctypes.data, tf.ctypes.data, dl.ctypes.data, None))
            c = hp["local"][r]
            ok = ok and np.array_equal(to, hp["offs"][r]) and np.array_equal(di[:P], c["doc_ids"]) \
                and np.array_equal(tf[:P], c["tfs"]) and np.array_equal(dl, c["doc_len"])
            ix.close()
        torch.cuda.synchronize()
        print(json.dumps({
            "workload": "sharded text lift: %d posts, %.1f MB of text, %d tokens, G = %d shards on one GPU, %d terms in the "
                        "union, %d gathered entries (%.1f MB)" % (len(texts), sum(int(s[1][-1]) for s in slices) / 1e6, n_tokens,
                                                                  world, len(hp["vocab"]), n_entries, entry_bytes / 1e6),
            "gpu": info,
            "build_s": [round(min(t), 4) for t in build_t], "union_s": [round(min(t), 4) for t in union_t],
            "union_reps_s": [round(t, 4) for t in union_t[0]],
            "build_kernels_ms": build_k, "union_kernels_ms": union_k, "union_top_kernels_ms": union_top,
            "host_builder_s": [round(t, 3) for t in hp["build_s"]], "host_union_s": round(hp["union_s"], 3),
            "host_remap_s": round(hp["remap_s"], 3),
            "arrays_equal": bool(ok)}), flush=True)


if __name__ == "__main__":
    main()
