"""ctypes view of libopenintel_host.so — the C++ host layer's tokenizer and index builder
(openintel_b200/host/openintel_host.hpp), for tests and for Python callers that want to build a
BM25 index from post texts.  CPU only; scoring still happens in libopenintel_gpu.so."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib_path():
    return os.path.join(_HERE, "host", "libopenintel_host.so")


def load():
    global _lib
    if _lib is None:
        p = lib_path()
        if not os.path.exists(p):
            raise OSError("libopenintel_host.so is missing (%s): run `python openintel_b200/host/build.py`" % p)
        L = C.CDLL(p)
        vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
        L.oih_builder_create.restype = vp
        L.oih_builder_destroy.argtypes = [vp]
        L.oih_builder_add.argtypes = [vp, vp, vp, u64]
        L.oih_builder_finish.argtypes = [vp, C.POINTER(u32), C.POINTER(u32), C.POINTER(u64)]
        L.oih_builder_export.argtypes = [vp, vp, vp, vp, vp]
        L.oih_builder_term_id.restype = u32
        L.oih_builder_term_id.argtypes = [vp, C.c_char_p, u32]
        L.oih_builder_query_terms.restype = u32
        L.oih_builder_query_terms.argtypes = [vp, C.c_char_p, u32, vp, u32]
        L.oih_builder_term.restype = u32
        L.oih_builder_term.argtypes = [vp, u32, C.c_char_p, u32]
        L.oih_tokenize.restype = u64
        L.oih_last_error.restype = C.c_char_p
        L.oih_store_open.restype = vp
        L.oih_store_open.argtypes = [C.c_char_p]
        L.oih_store_close.argtypes = [vp]
        L.oih_store_info.argtypes = [vp, C.POINTER(u64), C.POINTER(u32)]
        L.oih_store_lift_posts.restype = C.c_int64
        L.oih_store_lift_posts.argtypes = [vp, vp]
        L.oih_store_embeddings.restype = C.c_int
        L.oih_store_embeddings.argtypes = [vp, vp]
        L.oih_builder_post_id.restype = u32
        L.oih_builder_post_id.argtypes = [vp, u32, C.c_char_p, u32]
        L.oih_tokenize.argtypes = [C.c_char_p, u64, C.c_char_p, u64]
        _lib = L
    return _lib


def tokenize(text):
    raw = text.encode("utf-8") if isinstance(text, str) else bytes(text)
    out = C.create_string_buffer(len(raw) + 1)
    n = load().oih_tokenize(raw, len(raw), out, len(raw) + 1)
    s = out.raw[:n].decode("ascii")
    return s.split("\n") if s else []


class IndexBuilder:
    """posts -> vocabulary + CSR (term_offsets u64, doc_ids u32, tfs u32, doc_len u32)"""

    def __init__(self):
        self.L = load()
        self.b = C.c_void_p(self.L.oih_builder_create())

    def close(self):
        if getattr(self, "b", None):
            self.L.oih_builder_destroy(self.b)
            self.b = None

    __del__ = close

    def add(self, texts):
        raw = [t.encode("utf-8") if isinstance(t, str) else bytes(t) for t in texts]
        offs = np.zeros(len(raw) + 1, dtype=np.uint64)
        offs[1:] = np.cumsum([len(r) for r in raw])
        blob = b"".join(raw) or b"\0"
        self.L.oih_builder_add(self.b, C.c_char_p(blob), offs.ctypes.data, len(raw))

    def finish(self):
        nd, nt, npost = C.c_uint32(), C.c_uint32(), C.c_uint64()
        self.L.oih_builder_finish(self.b, C.byref(nd), C.byref(nt), C.byref(npost))
        to = np.empty(nt.value + 1, dtype=np.uint64)
        di = np.empty(npost.value, dtype=np.uint32)
        tf = np.empty(npost.value, dtype=np.uint32)
        dl = np.empty(nd.value, dtype=np.uint32)
        self.L.oih_builder_export(self.b, to.ctypes.data, di.ctypes.data, tf.ctypes.data, dl.ctypes.data)
        return dict(term_offsets=to, doc_ids=di, tfs=tf, doc_len=dl, n_docs=nd.value, n_terms=nt.value)

    def term_id(self, token):
        raw = token.encode("utf-8")
        return int(self.L.oih_builder_term_id(self.b, raw, len(raw)))

    def term(self, term_id):
        n = self.L.oih_builder_term(self.b, term_id, None, 0)
        buf = C.create_string_buffer(n + 1)
        self.L.oih_builder_term(self.b, term_id, buf, n)
        return buf.raw[:n].decode("ascii")

    def post_id(self, doc):
        n = self.L.oih_builder_post_id(self.b, doc, None, 0)
        buf = C.create_string_buffer(n + 1)
        self.L.oih_builder_post_id(self.b, doc, buf, n)
        return buf.raw[:n].decode("utf-8")

    def query_terms(self, text):
        raw = text.encode("utf-8")
        out = np.empty(max(len(raw), 1), dtype=np.uint32)
        n = self.L.oih_builder_query_terms(self.b, raw, len(raw), out.ctypes.data, len(out))
        return out[:n].copy()


class CppPostStore:
    """The C++ reader of the SQLite post store (host/openintel_store.hpp), for tests: the compiled host layer must
    lift the same CSR and the same normalised rows out of a store as openintel_b200.store does."""

    def __init__(self, path):
        self.L = load()
        self.s = self.L.oih_store_open(path.encode("utf-8"))
        if not self.s:
            raise OSError(self.L.oih_last_error().decode("utf-8", "replace"))
        n, d = C.c_uint64(), C.c_uint32()
        self.L.oih_store_info(self.s, C.byref(n), C.byref(d))
        self.n_posts, self.dim = n.value, d.value

    def close(self):
        if getattr(self, "s", None):
            self.L.oih_store_close(self.s)
            self.s = None

    __del__ = close

    def lift_posts(self, builder):
        n = self.L.oih_store_lift_posts(self.s, builder.b)
        if n < 0:
            raise ValueError(self.L.oih_last_error().decode("utf-8", "replace"))
        return n

    def embeddings(self):
        out = np.empty((self.n_posts, self.dim), dtype=np.float32)
        if self.L.oih_store_embeddings(self.s, out.ctypes.data) != 0:
            raise ValueError(self.L.oih_last_error().decode("utf-8", "replace"))
        return out
