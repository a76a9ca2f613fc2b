"""ctypes wrapper of oracle/_ref/libtrinity_ref.so (the reference's own hot path compiled in place by
oracle/build_ref.sh), and its recorded stand-in for machines without it.  TEST INFRASTRUCTURE ONLY — never imported by the product
package.

The tests compare against `load_golden_ref()`: every reference call made through it is keyed by a hash of its inputs.  Recording
(TRN_GOLDEN_RECORD=<dir>, needs oracle/_ref) runs the reference and writes per call a fingerprint of its output; replaying (the default)
recomputes the output with this repository's own plain-C oracle (oracle/trinity_oracle.c) and host encoders and accepts it only if it
matches the fingerprint: the exact bytes for docIDs, postings and index bytes (with a sparse patch where the reference's bytes differ,
e.g. its uninitialised padding), a weighted checksum within the recorded oracle-vs-reference tolerance for scores.  Small outputs that
nothing here can recompute (segment directories, full-size batch checksums) are stored whole.  tests/golden/reference_calls.json.gz
holds the records: `python tests/refharness.py merge <dir>` builds it from a recording."""
from __future__ import annotations

import base64
import ctypes as C
import gzip
import hashlib
import json
import os
import sys
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
REF_SO = ROOT / "oracle" / "_ref" / "libtrinity_ref.so"
REF_GPU_SO = ROOT / "oracle" / "_ref" / "libtrinity_ref_gpu.so"  # the same reference objects + the reference-side binding of libtrinity_b200.so


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class RefLib:
    def __init__(self, L):
        self.L = L
        vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
        L.tref_new.restype = vp
        L.tref_new.argtypes = [C.c_int]
        L.tref_free.argtypes = [vp]
        L.tref_add_term.argtypes = [vp, C.c_char_p, vp, vp, u32, vp]
        L.tref_finish.argtypes = [vp, u64]
        L.tref_from_bytes.restype = vp
        L.tref_from_bytes.argtypes = [C.c_int, vp, u64, vp, u64, vp, vp, vp, vp, u32, u64, u64]
        L.tref_index_size.restype = u64
        L.tref_index_size.argtypes = [vp]
        L.tref_index_data.restype = vp
        L.tref_index_data.argtypes = [vp]
        L.tref_hits_size.restype = u64
        L.tref_hits_size.argtypes = [vp]
        L.tref_hits_data.restype = vp
        L.tref_hits_data.argtypes = [vp]
        L.tref_num_terms.restype = u32
        L.tref_num_terms.argtypes = [vp]
        L.tref_term.argtypes = [vp, u32, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32)]
        L.tref_decode.restype = C.c_int64
        L.tref_decode.argtypes = [vp, u32, vp, vp, u64]
        L.tref_advance.argtypes = [vp, u32, vp, u32, vp]
        L.tref_positions.restype = C.c_int64
        L.tref_positions.argtypes = [vp, u32, vp, u64]
        L.tref_bm25.restype = C.c_double
        L.tref_bm25.argtypes = [vp, u32, u32]
        L.tref_exec.restype = C.c_int64
        L.tref_exec.argtypes = [vp, C.c_char_p, C.c_int, vp, vp, u64]
        L.tref_exec2.restype = C.c_int64
        L.tref_exec2.argtypes = [vp, C.c_char_p, C.c_int, u32, vp, vp, u64]
        L.tref_exec3.restype = C.c_int64
        L.tref_exec3.argtypes = [vp, C.c_char_p, C.c_int, u32, u32, vp, vp, u64]
        L.tref_exec_masked.restype = C.c_int64
        L.tref_exec_masked.argtypes = [vp, C.c_char_p, C.c_int, vp, u32, vp, vp, u64]
        L.tref_exec_batch.restype = C.c_double
        L.tref_exec_batch.argtypes = [vp, vp, u32, C.c_int, u32, C.c_int, vp, vp, vp, vp]
        L.tref_synth_build.restype = vp
        L.tref_synth_build.argtypes = [C.c_int, u32, u32, u32, u64, C.c_int, C.c_int]
        L.tref_last_error.restype = C.c_char_p
        L.tref_segment_write.argtypes = [C.c_int, C.c_char_p, u32, vp, vp, vp, vp, vp, u32, u32]
        L.tref_segment_open.restype = vp
        L.tref_segment_open.argtypes = [C.c_char_p]
        L.tref_collection_open.restype = vp
        L.tref_collection_open.argtypes = [vp, u32]
        L.tref_collection_exec.restype = C.c_int64
        L.tref_collection_exec.argtypes = [vp, C.c_char_p, C.c_int, vp, vp, u64, vp]
        L.tref_resolve.argtypes = [vp, C.c_char_p, C.POINTER(u32), C.POINTER(u32), C.POINTER(u32)]
        L.tref_field_stats.argtypes = [vp, C.POINTER(u64), C.POINTER(u32), C.POINTER(u64), C.POINTER(u32)]

    def collection_open(self, paths):
        """IndexSourcesCollection over several segment directories (scanned newest generation first)"""
        enc = [str(p).encode() for p in paths]
        arr = (C.c_char_p * len(enc))(*enc)
        h = self.L.tref_collection_open(C.cast(arr, C.c_void_p), len(enc))
        if not h:
            raise RuntimeError(self.err())
        x = RefIndex(self, -1, C.c_void_p(h))
        x.nsources = len(enc)
        return x

    def segment_write(self, codec: int, path: str, lists: dict, erased=(), replace_below: int = 0):
        """Index `lists` ({term: (docids, freqs)}) with the reference's SegmentIndexSession and commit() the segment to `path`
        (the last path component must be a number: the segment's generation).  Documents with id < replace_below are committed with
        replace() — updates of documents an older segment holds — and, like `erased`, land in updated_documents.ids."""
        names = list(lists)
        enc = [n.encode() for n in names]
        arr = (C.c_char_p * len(enc))(*enc)
        counts = np.array([len(lists[n][0]) for n in names], np.uint32)
        d = np.ascontiguousarray(np.concatenate([np.asarray(lists[n][0], np.uint32) for n in names]) if names else np.zeros(0, np.uint32))
        f = np.ascontiguousarray(np.concatenate([np.asarray(lists[n][1], np.uint32) for n in names]) if names else np.zeros(0, np.uint32))
        er = np.ascontiguousarray(erased, np.uint32)
        if self.L.tref_segment_write(codec, str(path).encode(), len(enc), C.cast(arr, C.c_void_p), _p(counts), _p(d), _p(f), _p(er), len(er), replace_below) != 0:
            raise RuntimeError(self.err())

    def segment_open(self, path: str):
        """The reference's SegmentIndexSource over `path`, wrapped for exec()"""
        h = self.L.tref_segment_open(str(path).encode())
        if not h:
            raise RuntimeError(self.err())
        return RefIndex(self, -1, C.c_void_p(h))

    def err(self):
        return self.L.tref_last_error().decode()


class RefIndex:
    """An in-memory index authored by the reference Encoders (or wrapping foreign bytes) + reference exec."""

    def __new__(cls, rl, codec: int, handle=None):
        if isinstance(rl, GoldenRef):
            return GoldenIndex(rl, codec)
        return super().__new__(cls)

    def __init__(self, rl: RefLib, codec: int, handle=None):
        self.rl, self.codec = rl, codec
        self.h = C.c_void_p(rl.L.tref_new(codec)) if handle is None else handle
        self.names = []

    @classmethod
    def from_bytes(cls, rl, codec, index, hits, names, terms, docs_cnt, sum_hits=0):
        if isinstance(rl, GoldenRef):
            return GoldenIndex.from_bytes(rl, codec, index, hits, names, terms, docs_cnt, sum_hits)
        index = np.ascontiguousarray(index, np.uint8)
        hits = np.ascontiguousarray(hits, np.uint8) if hits is not None and len(hits) else None
        enc = [n.encode() for n in names]
        arr = (C.c_char_p * len(enc))(*enc)
        docs = np.ascontiguousarray(terms["documents"], np.uint32)
        off = np.ascontiguousarray(terms["chunk_off"], np.uint32)
        ln = np.ascontiguousarray(terms["chunk_len"], np.uint32)
        h = rl.L.tref_from_bytes(codec, _p(index), index.size, _p(hits), 0 if hits is None else hits.size,
                                 C.cast(arr, C.c_void_p), _p(docs), _p(off), _p(ln), len(enc), docs_cnt, sum_hits)
        if not h:
            raise RuntimeError(rl.err())
        x = cls(rl, codec, C.c_void_p(h))
        x.names = list(names)
        return x

    @classmethod
    def synth_build(cls, rl, codec, ndocs, nterms, min_df=1000, seed=0x5EED, with_hits=True, threads=1):
        """the BASELINE.md synthetic index authored by the reference's own Encoders (no product code involved)"""
        if isinstance(rl, GoldenRef):
            return GoldenIndex.synth_build(rl, codec, ndocs, nterms, min_df, seed, with_hits, threads)
        h = rl.L.tref_synth_build(codec, ndocs, nterms, min_df, seed, int(with_hits), threads)
        if not h:
            raise RuntimeError(rl.err())
        x = cls(rl, codec, C.c_void_p(h))
        x.names = [f"t{r:04d}" for r in range(1, nterms + 1)]
        return x

    def add_term(self, name, docids, freqs, positions=None):
        d = np.ascontiguousarray(docids, np.uint32)
        f = np.ascontiguousarray(freqs, np.uint32)
        p = None if positions is None else np.ascontiguousarray(positions, np.uint32)
        r = self.rl.L.tref_add_term(self.h, name.encode(), _p(d), _p(f), len(d), _p(p))
        if r < 0:
            raise RuntimeError(self.rl.err())
        self.names.append(name)
        return r

    def finish(self, docs_cnt):
        if self.rl.L.tref_finish(self.h, docs_cnt) != 0:
            raise RuntimeError(self.rl.err())

    def index(self):
        n = self.rl.L.tref_index_size(self.h)
        return np.ctypeslib.as_array(C.cast(self.rl.L.tref_index_data(self.h), C.POINTER(C.c_uint8)), shape=(n,)).copy()

    def hits(self):
        n = self.rl.L.tref_hits_size(self.h)
        if not n:
            return np.zeros(0, np.uint8)
        return np.ctypeslib.as_array(C.cast(self.rl.L.tref_hits_data(self.h), C.POINTER(C.c_uint8)), shape=(n,)).copy()

    def terms(self):
        from trinity_b200._ffi import TERM_DTYPE
        n = self.rl.L.tref_num_terms(self.h)
        out = np.zeros(n, TERM_DTYPE)
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        for i in range(n):
            self.rl.L.tref_term(self.h, i, C.byref(a), C.byref(b), C.byref(c))
            out[i] = (a.value, b.value, c.value)
        return out

    def decode(self, term_idx, cap):
        d, f = np.zeros(cap, np.uint32), np.zeros(cap, np.uint32)
        n = self.rl.L.tref_decode(self.h, term_idx, _p(d), _p(f), cap)
        if n < 0:
            raise RuntimeError(self.rl.err())
        return d[:n], f[:n]

    def positions(self, term_idx, cap):
        """flat positions of every document of the term (freq entries per document), via the reference's materialize_hits"""
        p = np.zeros(max(cap, 1), np.uint32)
        n = self.rl.L.tref_positions(self.h, term_idx, _p(p), cap)
        if n < 0:
            raise RuntimeError(self.rl.err())
        return p[:n]

    def advance(self, term_idx, targets):
        t = np.ascontiguousarray(targets, np.uint32)
        o = np.zeros(len(t), np.uint32)
        if self.rl.L.tref_advance(self.h, term_idx, _p(t), len(t), _p(o)) != 0:
            raise RuntimeError(self.rl.err())
        return o

    def collection_exec(self, q: str, scored: bool, cap: int):
        """per-source exec_query over the collection -> [(ids, scores)] in collection order"""
        ids = np.zeros(max(cap, 1), np.uint32)
        sc = np.zeros(max(cap, 1), np.float64)
        cnt = np.zeros(self.nsources, np.uint64)
        n = self.rl.L.tref_collection_exec(self.h, q.encode(), 1 if scored else 0, _p(ids), _p(sc), cap, _p(cnt))
        if n < 0:
            raise RuntimeError(self.rl.err())
        out, at = [], 0
        for c in cnt:
            c = int(c)
            out.append((ids[at:at + c], sc[at:at + c] if scored else None))
            at += c
        return out

    def resolve(self, term: str):
        a, b, c = C.c_uint32(), C.c_uint32(), C.c_uint32()
        if self.rl.L.tref_resolve(self.h, term.encode(), C.byref(a), C.byref(b), C.byref(c)) != 0:
            raise RuntimeError(self.rl.err())
        return a.value, b.value, c.value

    def field_stats(self):
        a, b, c, d = C.c_uint64(), C.c_uint32(), C.c_uint64(), C.c_uint32()
        if self.rl.L.tref_field_stats(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)) != 0:
            raise RuntimeError(self.rl.err())
        return {"sumTermHits": a.value, "totalTerms": b.value, "sumTermsDocs": c.value, "docsCnt": d.value}

    def bm25(self, term_idx, freq):
        return self.rl.L.tref_bm25(self.h, term_idx, freq)

    def exec(self, q: str, scored: bool, cap: int, parser_flags: int = 0, min_match: int = 0):
        """parser_flags: ast_parser::Flags; 8 = ParseConstTrueExpr (the <expr> syntax -> Optional), 16 = ParseMatchSomeExpr ([a, b, c]);
        min_match: match_some.min of every MatchSome group (the parser leaves it at 1)"""
        ids = np.zeros(max(cap, 1), np.uint32)
        sc = np.zeros(max(cap, 1), np.float64)
        n = self.rl.L.tref_exec3(self.h, q.encode(), 1 if scored else 0, parser_flags, min_match, _p(ids), _p(sc), cap)
        if n < 0:
            raise RuntimeError(self.rl.err())
        assert n <= cap, "reference produced more matches than the capacity given"
        return ids[:n], (sc[:n] if scored else None)

    def exec_masked(self, q: str, scored: bool, masked, cap: int):
        """exec_query with the reference's masked_documents_registry holding `masked` docIDs"""
        mk = np.ascontiguousarray(masked, np.uint32)
        ids = np.zeros(max(cap, 1), np.uint32)
        sc = np.zeros(max(cap, 1), np.float64)
        n = self.rl.L.tref_exec_masked(self.h, q.encode(), 1 if scored else 0, _p(mk), len(mk), _p(ids), _p(sc), cap)
        if n < 0:
            raise RuntimeError(self.rl.err())
        return ids[:n], (sc[:n] if scored else None)

    def exec_batch(self, queries, scored: bool, k: int, threads: int):
        enc = [q.encode() for q in queries]
        arr = (C.c_char_p * len(enc))(*enc)
        nq = len(enc)
        counts = np.zeros(nq, np.uint64)
        sums = np.zeros(nq, np.uint64)
        tid = np.zeros((nq, k), np.uint32)
        tsc = np.zeros((nq, k), np.float64)
        el = self.rl.L.tref_exec_batch(self.h, C.cast(arr, C.c_void_p), nq, 1 if scored else 0, k, threads, _p(counts), _p(sums), _p(tid), _p(tsc))
        if el < 0:
            raise RuntimeError(self.rl.err())
        return el, counts, sums, tid, tsc

    def __del__(self):
        try:
            self.rl.L.tref_free(self.h)
        except Exception:
            pass


_ref = None
_ref_gpu = None


def reference_built() -> bool:
    """oracle/_ref exists only where build() could read the reference sources"""
    return REF_SO.exists()


def load_ref_gpu() -> RefLib:
    """the reference compiled with its exec_query() span site going through integration/gpu_exec.cpp (needs a CUDA device at run time)"""
    global _ref_gpu
    if _ref_gpu is None:
        if not REF_GPU_SO.exists():
            raise FileNotFoundError(f"{REF_GPU_SO} not built (build() builds it where the reference sources are readable)")
        rl = RefLib(C.CDLL(str(REF_GPU_SO)))
        rl.L.tref_gpu_attach.argtypes = [C.c_void_p, C.c_int, C.c_uint64]
        rl.L.tref_gpu_detach.argtypes = [C.c_void_p]
        rl.L.tref_gpu_spans_executed.restype = C.c_uint64
        rl.L.tref_gpu_spans_executed.argtypes = [C.c_void_p]
        _ref_gpu = rl
    return _ref_gpu


def load_ref() -> RefLib:
    global _ref
    if _ref is None:
        if not REF_SO.exists():
            raise FileNotFoundError(f"{REF_SO} not built (build() builds it where the reference sources are readable)")
        _ref = RefLib(C.CDLL(str(REF_SO)))
    return _ref


# ============================================================================================ recorded reference (see module docstring)
GOLDEN_CALLS = ROOT / "tests" / "golden" / "reference_calls.json.gz"
RECORD_DIR = os.environ.get("TRN_GOLDEN_RECORD")
_calls = None


def _feed(h, p):
    if isinstance(p, np.generic):
        p = p.item()
    if isinstance(p, np.ndarray):
        a = np.ascontiguousarray(p)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    elif isinstance(p, (list, tuple)):
        h.update(b"[")
        for x in p:
            _feed(h, x)
        h.update(b"]")
    else:
        h.update(repr(p).encode())
    h.update(b"|")


def _key(*parts) -> str:
    h = hashlib.sha1()
    _feed(h, parts)
    return h.hexdigest()[:16]


def _pack(b: bytes) -> str:
    return base64.b64encode(zlib.compress(b, 9)).decode()


def _unpack(s: str) -> bytes:
    return zlib.decompress(base64.b64decode(s))


def _put(key, rec):
    with open(Path(RECORD_DIR) / f"calls_{os.getpid()}.jsonl", "a") as f:
        f.write(json.dumps([key, rec]) + "\n")


def _get(key, what):
    global _calls
    if _calls is None:
        _calls = json.loads(gzip.decompress(GOLDEN_CALLS.read_bytes())) if GOLDEN_CALLS.exists() else {}
    if key not in _calls:
        raise AssertionError(f"{what}: no recorded reference output for this call (its inputs changed since the recording)")
    return _calls[key]


def _exact(key, what, real, pred):
    """an output that must equal the reference's byte for byte; `pred` = the same output computed by this repository"""
    if RECORD_DIR:
        real = np.ascontiguousarray(real)
        rec = {"h": _key(real)}
        if pred is None or pred.shape != real.shape or pred.dtype != real.dtype:
            rec["full"] = _pack(real.tobytes())
            print(f"refharness: {what}: stored whole ({real.nbytes} bytes)", file=sys.stderr)
        else:
            ru, pu = real.reshape(-1).view(np.uint8), np.ascontiguousarray(pred).reshape(-1).view(np.uint8)
            d = np.flatnonzero(ru != pu)
            if d.size:
                rec["p"] = [np.diff(d, prepend=0).tolist(), ru[d].tolist()]
        _put(key, rec)
        return real
    rec = _get(key, what)
    if "full" in rec:
        out = np.frombuffer(_unpack(rec["full"]), np.uint8).view(pred.dtype).copy()
    else:
        out = np.array(pred, copy=True)
        if "p" in rec:
            out.reshape(-1).view(np.uint8)[np.cumsum(rec["p"][0])] = rec["p"][1]
    if _key(out) != rec["h"]:
        raise AssertionError(f"{what}: this repository's oracle no longer reproduces the reference's recorded output")
    return out


def _fingerprint(s):
    w = 0.5 + np.random.default_rng(len(s)).random(len(s))
    return [float(np.sum(s)), float(np.dot(s, w)), float(np.max(np.abs(s))) if len(s) else 0.0]


def _scores(key, what, real, pred):
    """scores: the oracle's own, accepted within the oracle-vs-reference difference seen at recording time"""
    pred = np.asarray(pred, np.float64)
    if RECORD_DIR:
        real = np.asarray(real, np.float64)
        assert real.shape == pred.shape, what
        err = float(np.max(np.abs(real - pred) / np.maximum(np.abs(real), 1e-30))) if len(real) else 0.0
        assert err <= 1e-6, f"{what}: the oracle's scores differ from the reference's by {err:.2e}"
        _put(key, {"n": len(real), "f": _fingerprint(real), "t": max(1e-12, 4 * err)})
        return real
    rec = _get(key, what)
    got, want = _fingerprint(pred), rec["f"]
    tol = rec["t"] * len(pred) * max(want[2], 1e-30)
    if len(pred) != rec["n"] or any(abs(a - b) > tol for a, b in zip(got, want)):
        raise AssertionError(f"{what}: this repository's oracle no longer reproduces the reference's recorded scores")
    return pred


def _stored(key, what, compute):
    """a small JSON-able output kept as is (bm25 values, term lookups, field statistics)"""
    if RECORD_DIR:
        v = compute()
        _put(key, {"v": v})
        return v
    return _get(key, what)["v"]


def _u32(a):
    return np.ascontiguousarray(a, np.uint32)


class GoldenRef:
    """stand-in for RefLib: the real library while recording, the recorded outputs otherwise"""

    def __init__(self, real=None):
        self.real = real

    def segment_write(self, codec: int, path, lists: dict, erased=(), replace_below: int = 0):
        key = _key("segment_write", codec, Path(path).name, [(n, _u32(d), _u32(f)) for n, (d, f) in lists.items()], _u32(erased), replace_below)
        if RECORD_DIR:
            self.real.segment_write(codec, path, lists, erased, replace_below)
            _put(key, {"files": {f.name: _pack(f.read_bytes()) for f in sorted(Path(path).iterdir())}})
            return
        for name, b in _get(key, f"segment_write {path}")["files"].items():
            (Path(path) / name).write_bytes(_unpack(b))

    def segment_open(self, path):
        files = sorted(Path(path).iterdir())
        x = GoldenIndex(self, -1, ident=_key("segment", [(f.name, np.frombuffer(f.read_bytes(), np.uint8)) for f in files]))
        x.real = self.real.segment_open(path) if RECORD_DIR else None
        return x


class GoldenIndex:
    """stand-in for RefIndex (see module docstring); the index itself is rebuilt by this repository's encoders (add_term), taken as
    given (from_bytes) or generated (synth_build), and executed by the plain-C oracle"""

    def __init__(self, rl: GoldenRef, codec: int, ident=None):
        self.rl, self.codec, self.ident = rl, codec, ident
        self.names, self._lists, self._built = [], [], None
        self.real = RefIndex(rl.real, codec) if RECORD_DIR and ident is None else None

    @classmethod
    def from_bytes(cls, rl, codec, index, hits, names, terms, docs_cnt, sum_hits=0):
        index = np.ascontiguousarray(index, np.uint8)
        hits = np.ascontiguousarray(hits, np.uint8) if hits is not None and len(hits) else np.zeros(0, np.uint8)
        terms = np.ascontiguousarray(terms)
        x = cls(rl, codec, ident=_key("from_bytes", codec, index, hits, list(names), terms, docs_cnt, sum_hits))
        x.names, x.ndocs, x._built = list(names), docs_cnt, (index, hits, terms)
        if RECORD_DIR:
            x.real = RefIndex.from_bytes(rl.real, codec, index, hits, names, terms, docs_cnt, sum_hits)
        return x

    @classmethod
    def synth_build(cls, rl, codec, ndocs, nterms, min_df=1000, seed=0x5EED, with_hits=True, threads=1):
        import trinity_b200 as tb
        x = cls(rl, codec, ident=_key("synth_build", codec, ndocs, nterms, min_df, seed, with_hits))
        s = tb.SynthIndex(codec, ndocs, nterms, min_df=min_df, seed=seed, with_hits=with_hits, threads=threads)
        x.names, x.ndocs = list(s.names), ndocs
        x._built = (np.array(s.index), np.array(s.hits), np.array(s.terms))
        if RECORD_DIR:
            x.real = RefIndex.synth_build(rl.real, codec, ndocs, nterms, min_df, seed, with_hits, threads)
        return x

    def add_term(self, name, docids, freqs, positions=None):
        d, f = _u32(docids), _u32(freqs)
        p = None if positions is None else _u32(positions)
        self._lists.append((name, d, f, p))
        self.names.append(name)
        if self.real is not None:
            assert self.real.add_term(name, d, f, p) == len(self.names) - 1
        return len(self.names) - 1

    def finish(self, docs_cnt):
        self.ndocs = docs_cnt
        self.ident = _key("add_term", self.codec, [(n, d, f, p) for n, d, f, p in self._lists], docs_cnt)
        if self.real is not None:
            self.real.finish(docs_cnt)

    # ---- this repository's view of the same index
    def _index(self):
        if self._built is None:
            import trinity_b200 as tb
            b = tb.IndexBuilder(self.codec)
            for _, d, f, p in self._lists:
                b.add_term(d, f, p)
            self._built = (b.index(), b.hits(), b.terms_array())
        return self._built

    def _oracle(self):
        import oracle_c
        return oracle_c.load()

    def _call(self, *args):
        return _key(self.ident, *args), f"reference {args[0]} {args[1:]!r}"[:200]

    def index(self):
        return _exact(*self._call("index"), self.real.index() if RECORD_DIR else None, self._index()[0])

    def hits(self):
        return _exact(*self._call("hits"), self.real.hits() if RECORD_DIR else None, self._index()[1])

    def terms(self):
        return _exact(*self._call("terms"), self.real.terms() if RECORD_DIR else None, self._index()[2])

    def decode(self, term_idx, cap):
        import oracle_c
        index, _, terms = self._index()
        d, f = oracle_c.decode(self._oracle(), self.codec, index, terms[term_idx])
        real = self.real.decode(term_idx, cap) if RECORD_DIR else (None, None)
        return (_exact(*self._call("decode.d", term_idx, cap), real[0], d[:cap]),
                _exact(*self._call("decode.f", term_idx, cap), real[1], f[:cap]))

    def positions(self, term_idx, cap):
        import oracle_c
        index, hits, terms = self._index()
        p = oracle_c.positions(self._oracle(), self.codec, index, hits, terms[term_idx])
        return _exact(*self._call("positions", term_idx, cap), self.real.positions(term_idx, cap) if RECORD_DIR else None, p[:cap])

    def advance(self, term_idx, targets):
        t = _u32(targets)
        d, _ = self.decode(term_idx, int(self._index()[2][term_idx]["documents"]))
        out, cur = np.zeros(len(t), np.uint32), 0
        for i, x in enumerate(t.tolist()):   # PostingsListIterator::advance: never moves backwards
            if cur < x or cur == 0:
                j = int(np.searchsorted(d, x))
                cur = int(d[j]) if j < len(d) else 0xFFFFFFFF
            out[i] = cur
        return _exact(*self._call("advance", term_idx, t), self.real.advance(term_idx, t) if RECORD_DIR else None, out)

    def bm25(self, term_idx, freq):
        return _stored(*self._call("bm25", term_idx, freq), lambda: self.real.bm25(term_idx, freq))

    def resolve(self, term: str):
        return tuple(_stored(*self._call("resolve", term), lambda: list(self.real.resolve(term))))

    def field_stats(self):
        return _stored(*self._call("field_stats"), lambda: self.real.field_stats())

    def _oracle_exec(self, q, scored, parser_flags, min_match):
        import oracle_c
        import trinity_b200 as tb
        index, hits, terms = self._index()
        nodes = tb.parse_query(q, tb.TermDictionary(self.names), min_match=min_match or None)
        for x in nodes:
            if x["kind"] == tb.NODE_TERM and x["term"] != tb.EMPTY_TERM:
                x["weight"] = tb.bm25_idf(int(terms["documents"][x["term"]]), self.ndocs)
        return oracle_c.exec_query(self._oracle(), self.codec, index, terms, nodes, self.ndocs, scored, hits=hits)

    def exec(self, q: str, scored: bool, cap: int, parser_flags: int = 0, min_match: int = 0):
        ids, sc = self._oracle_exec(q, scored, parser_flags, min_match)
        real = self.real.exec(q, scored, cap, parser_flags, min_match) if RECORD_DIR else (None, None)
        what = self._call("exec", q, scored, cap, parser_flags, min_match)
        ids = _exact(what[0] + ".ids", what[1], real[0], ids[:cap])
        return ids, (_scores(what[0] + ".scores", what[1], real[1], sc[:cap]) if scored else None)

    def exec_masked(self, q: str, scored: bool, masked, cap: int):
        mk = _u32(masked)
        ids, sc = self._oracle_exec(q, scored, 0, 0)
        keep = ~np.isin(ids, mk)
        real = self.real.exec_masked(q, scored, mk, cap) if RECORD_DIR else (None, None)
        what = self._call("exec_masked", q, scored, mk, cap)
        ids = _exact(what[0] + ".ids", what[1], real[0], ids[keep][:cap])
        return ids, (_scores(what[0] + ".scores", what[1], real[1], sc[keep][:cap]) if scored else None)

    def exec_batch(self, queries, scored: bool, k: int, threads: int):
        """full-size batches: the per-query match counts, docID sums and top-k are stored whole (the elapsed time is not)"""
        key, what = self._call("exec_batch", list(queries), scored, k)
        if RECORD_DIR:
            el, *out = self.real.exec_batch(queries, scored, k, threads)
            _put(key, {"out": [_pack(np.ascontiguousarray(a).tobytes()) for a in out]})
            return (el, *out)
        rec = _get(key, what)
        nq = len(queries)
        shapes = ((np.uint64, (nq,)), (np.uint64, (nq,)), (np.uint32, (nq, k)), (np.float64, (nq, k)))
        return (0.0, *(np.frombuffer(_unpack(b), dt).reshape(sh).copy() for b, (dt, sh) in zip(rec["out"], shapes)))


def load_golden_ref() -> GoldenRef:
    """what the tests compare against: the reference itself while recording, its recorded outputs otherwise"""
    if RECORD_DIR:
        Path(RECORD_DIR).mkdir(parents=True, exist_ok=True)
        return GoldenRef(load_ref())
    return GoldenRef()


def merge_recording(src: str, dst: Path = GOLDEN_CALLS):
    calls = json.loads(gzip.decompress(dst.read_bytes())) if dst.exists() else {}
    for f in sorted(Path(src).glob("calls_*.jsonl")):
        for line in f.read_text().splitlines():
            k, v = json.loads(line)
            calls[k] = v
    dst.write_bytes(gzip.compress(json.dumps(calls, sort_keys=True, separators=(",", ":")).encode(), 9, mtime=0))
    print(f"{dst}: {len(calls)} calls, {dst.stat().st_size} bytes")


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "merge":
        merge_recording(sys.argv[2])
    else:
        sys.exit("usage: python tests/refharness.py merge <recording dir>")
