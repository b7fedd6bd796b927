"""ctypes wrapper over corpus/libindexgen.so (test/bench infrastructure, see indexgen.h)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DB_NAMES = [
    "word_docids", "exact_word_docids", "word_prefix_docids", "exact_word_prefix_docids",
    "word_pair_proximity_docids", "word_position_docids", "word_fid_docids",
    "word_prefix_position_docids", "word_prefix_fid_docids", "field_id_word_count_docids",
]


class _DbView(C.Structure):
    _fields_ = [("n_keys", C.c_uint64), ("key_bytes", C.c_void_p), ("key_offsets", C.c_void_p),
                ("val_bytes", C.c_void_p), ("val_offsets", C.c_void_p)]


def build_lib():
    so = os.path.join(_HERE, "libindexgen.so")
    src = os.path.join(_HERE, "indexgen.cpp")
    if not os.path.exists(so) or (os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(so)):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


_lib = None


def lib():
    global _lib
    if _lib is None:
        l = C.CDLL(build_lib())
        l.ig_new.restype = C.c_void_p
        l.ig_new.argtypes = [C.c_uint32, C.c_uint32]
        l.ig_free.argtypes = [C.c_void_p]
        l.ig_set_stop_words.argtypes = [C.c_void_p, C.c_char_p]
        l.ig_add_text.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_char_p]
        l.ig_add_synthetic.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_double, C.c_uint32, C.c_uint32, C.c_uint64]
        l.ig_synthetic_queries.restype = C.c_void_p
        l.ig_synthetic_queries.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_int]
        l.ig_free_str.argtypes = [C.c_void_p]
        l.ig_build.argtypes = [C.c_void_p]
        l.ig_n_docs.restype = C.c_uint32
        l.ig_n_docs.argtypes = [C.c_void_p]
        l.ig_n_words.restype = C.c_uint64
        l.ig_n_words.argtypes = [C.c_void_p]
        l.ig_dictionary.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
        l.ig_db.argtypes = [C.c_void_p, C.c_int, C.POINTER(_DbView)]
        l.ig_documents_ids.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        l.ig_queries_from_arrays.restype = C.c_void_p
        l.ig_queries_from_arrays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint32, C.c_uint64, C.c_int]
        l.ig_query_source.argtypes = [C.c_void_p] + [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)] + \
                                     [C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]
        l.ig_fill_embeddings_f16.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64]
        _lib = l
    return _lib


def _arr(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_uint8 * (n * np.dtype(dtype).itemsize)).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype).copy()


class DbImage:
    """One LMDB-format database: sorted byte keys + CBO values as flat numpy arrays."""

    def __init__(self, key_bytes, key_offsets, val_bytes, val_offsets):
        self.key_bytes, self.key_offsets, self.val_bytes, self.val_offsets = key_bytes, key_offsets, val_bytes, val_offsets

    @property
    def n_keys(self):
        return len(self.key_offsets) - 1

    def key(self, i):
        return bytes(self.key_bytes[self.key_offsets[i]:self.key_offsets[i + 1]])

    def val(self, i):
        return bytes(self.val_bytes[self.val_offsets[i]:self.val_offsets[i + 1]])


class IndexImage:
    """Everything the query path reads from the LMDB environment, as byte images."""

    def __init__(self, n_fields=1, exact_mask=0, stop_words=()):
        self._l = lib()
        self._h = self._l.ig_new(n_fields, exact_mask)
        self.n_fields = n_fields
        self.exact_mask = exact_mask
        self.stop_words = frozenset(stop_words)
        if stop_words:
            self._l.ig_set_stop_words(self._h, " ".join(stop_words).encode())
        self.built = False

    def add_text(self, docid, fid, text):
        self._l.ig_add_text(self._h, docid, fid, text.encode())

    def add_synthetic(self, n_docs, vocab, zipf_s=1.07, len_lo=3, len_hi=15, seed=0xB200):
        self._l.ig_add_synthetic(self._h, n_docs, vocab, zipf_s, len_lo, len_hi, seed)

    def synthetic_queries(self, n, seed=1, with_typos=True):
        p = self._l.ig_synthetic_queries(self._h, n, seed, 1 if with_typos else 0)
        s = C.string_at(p).decode()
        self._l.ig_free_str(p)
        return [q for q in s.split("\n") if q]

    def build(self):
        self._l.ig_build(self._h)
        self.built = True
        self.n_docs = self._l.ig_n_docs(self._h)
        nw = self._l.ig_n_words(self._h)
        pb, po = C.c_void_p(), C.c_void_p()
        self._l.ig_dictionary(self._h, C.byref(pb), C.byref(po))
        self.dict_offsets = _arr(po.value, nw + 1, np.uint64)
        self.dict_bytes = _arr(pb.value, int(self.dict_offsets[-1]) if nw else 0, np.uint8)
        self.n_words = int(nw)
        self.dbs = []
        for i in range(len(DB_NAMES)):
            v = _DbView()
            self._l.ig_db(self._h, i, C.byref(v))
            ko = _arr(v.key_offsets, v.n_keys + 1, np.uint64)
            vo = _arr(v.val_offsets, v.n_keys + 1, np.uint64)
            kb = _arr(v.key_bytes, int(ko[-1]), np.uint8)
            vb = _arr(v.val_bytes, int(vo[-1]), np.uint8)
            self.dbs.append(DbImage(kb, ko, vb, vo))
        p, n = C.c_void_p(), C.c_uint64()
        self._l.ig_documents_ids(self._h, C.byref(p), C.byref(n))
        self.documents_ids_cbo = _arr(p.value, n.value, np.uint8)
        return self

    def word(self, i):
        return bytes(self.dict_bytes[self.dict_offsets[i]:self.dict_offsets[i + 1]]).decode()

    def db(self, name):
        return self.dbs[DB_NAMES.index(name)]

    def __del__(self):
        try:
            self._l.ig_free(self._h)
        except Exception:
            pass


def synthetic_embeddings_f16(n, d=768, seed=0xE5BED, first_row=0):
    """SURVEY §8(d) cfg 4: n x d i.i.d. N(0,1) rows, L2-normalised, as IEEE binary16 (numpy float16); deterministic per (seed, row)."""
    out = np.empty((n, d), np.float16)
    lib().ig_fill_embeddings_f16(out.ctypes.data_as(C.c_void_p), first_row, n, d, seed)
    return out


class CachedImage:
    """An IndexImage restored from the on-disk cache (same attributes; queries come from the persisted word/document arrays)."""

    def __init__(self, path):
        import json

        meta = json.load(open(os.path.join(path, "meta.json")))
        self.n_docs, self.n_words, self.n_fields = meta["n_docs"], meta["n_words"], meta["n_fields"]
        self.exact_mask, self.stop_words, self.built = 0, frozenset(), True
        ld = lambda name: np.load(os.path.join(path, name + ".npy"), mmap_mode="r")
        self.dict_bytes, self.dict_offsets = np.ascontiguousarray(ld("dict_bytes")), np.ascontiguousarray(ld("dict_offsets"))
        self.dbs = [DbImage(*(np.ascontiguousarray(ld(f"db{i}_{part}")) for part in ("kb", "ko", "vb", "vo"))) for i in range(len(DB_NAMES))]
        self.documents_ids_cbo = np.ascontiguousarray(ld("documents_ids"))
        self._qs = [np.ascontiguousarray(ld(n)) for n in ("q_word_bytes", "q_word_off", "q_doc_off", "q_doc_words")]

    def synthetic_queries(self, n, seed=1, with_typos=True):
        wb, wo, do, dw = self._qs
        l = lib()
        p = l.ig_queries_from_arrays(wb.ctypes.data_as(C.c_void_p), wo.ctypes.data_as(C.c_void_p), do.ctypes.data_as(C.c_void_p), len(do) - 1,
                                     dw.ctypes.data_as(C.c_void_p), n, seed, 1 if with_typos else 0)
        s = C.string_at(p).decode()
        l.ig_free_str(p)
        return [q for q in s.split("\n") if q]

    def word(self, i):
        return bytes(self.dict_bytes[self.dict_offsets[i]:self.dict_offsets[i + 1]]).decode()

    def db(self, name):
        return self.dbs[DB_NAMES.index(name)]


def synthetic_image(n_docs, vocab, seed=0xB200, n_fields=1, cache_min_docs=2_000_000, log=None):
    """The synthetic corpus of SURVEY §8(d), built (multi-threaded) or restored from B200_CORPUS_CACHE (default
    b200_corpus_cache_<uid> in the temporary directory: users sharing a host do not share it).  Only corpora of at least
    cache_min_docs documents are cached; concurrent processes (the ranks of a torchrun launch, the two arms of the bench) build once:
    the first takes a lock directory, the others wait for its `done` file.  Without a writable cache directory the corpus is built."""
    import json
    import tempfile
    import time

    def build():
        img = IndexImage(n_fields)
        img.add_synthetic(n_docs, vocab, seed=seed)
        return img.build()

    if n_docs < cache_min_docs or os.environ.get("B200_CORPUS_CACHE") == "off":
        return build()
    root = os.environ.get("B200_CORPUS_CACHE", os.path.join(tempfile.gettempdir(), f"b200_corpus_cache_{os.getuid()}"))
    path = os.path.join(root, f"syn_v3_{n_docs}_{vocab}_{seed:x}_{n_fields}")
    done = os.path.join(path, "done")
    if not os.path.exists(done):
        try:
            os.makedirs(root, exist_ok=True)
            os.mkdir(path)
            owner = True
        except FileExistsError:
            owner = False
        except OSError:
            return build()
        if not owner:
            t0 = time.time()
            while not os.path.exists(done) and time.time() - t0 < 1800:
                time.sleep(1.0)
            if not os.path.exists(done):
                return build()
        else:
            img = build()
            try:
                sv = lambda name, a: np.save(os.path.join(path, name + ".npy"), a)
                sv("dict_bytes", img.dict_bytes)
                sv("dict_offsets", img.dict_offsets)
                for i, db in enumerate(img.dbs):
                    for part, a in zip(("kb", "ko", "vb", "vo"), (db.key_bytes, db.key_offsets, db.val_bytes, db.val_offsets)):
                        sv(f"db{i}_{part}", a)
                sv("documents_ids", img.documents_ids_cbo)
                l = img._l
                wb, wo, do, dw = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
                nw, nd, ndw = C.c_uint64(), C.c_uint64(), C.c_uint64()
                l.ig_query_source(img._h, C.byref(wb), C.byref(wo), C.byref(nw), C.byref(do), C.byref(nd), C.byref(dw), C.byref(ndw))
                word_off = _arr(wo.value, nw.value + 1, np.uint64)
                sv("q_word_off", word_off)
                sv("q_word_bytes", _arr(wb.value, int(word_off[-1]) + 1, np.uint8))
                sv("q_doc_off", _arr(do.value, nd.value + 1, np.uint32))
                sv("q_doc_words", _arr(dw.value, ndw.value, np.uint32))
                l.ig_free_str(C.cast(wb, C.c_char_p))
                l.ig_free_str(C.cast(wo, C.c_char_p))
                json.dump({"n_docs": int(img.n_docs), "n_words": int(img.n_words), "n_fields": n_fields}, open(os.path.join(path, "meta.json"), "w"))
                open(done, "w").write("ok")
            except OSError as e:  # no room for the cache: go on without it
                if log:
                    log(f"corpus cache not written: {e}")
            return img
    return CachedImage(path)
