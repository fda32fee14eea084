"""ctypes binding of the CPU oracle (oracle/_build/liboracle.so).

TEST INFRASTRUCTURE. Only tests/, __graft_entry__.smoke() and bench.py's CPU legs import this.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
LIB_PATH = os.path.join(ORACLE_DIR, "_build", "liboracle.so")
REF_SIMDCOMP = os.path.join(ORACLE_DIR, "_ref", "libsimdcomp_ref.so")
_tmp_lib = None   # a library built outside a read-only tree, reused for the rest of the process


def build(force=False):
    """Compiles the oracle when its sources are newer than the library; returns the library's path."""
    global _tmp_lib
    if _tmp_lib is not None and not force:
        return _tmp_lib
    src = [os.path.join(ORACLE_DIR, f) for f in ("oracle.cpp", "oracle.h", "Makefile")]
    stale = (not os.path.exists(LIB_PATH)) or any(
        os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in src)
    path = LIB_PATH
    if force or stale:
        make = ["make", "-C", ORACLE_DIR, "-s"]
        out_dir = os.path.dirname(LIB_PATH)
        if not os.access(out_dir if os.path.isdir(out_dir) else ORACLE_DIR, os.W_OK):
            # read-only tree: build into a private temporary directory, never into the tree
            out_dir = tempfile.mkdtemp(prefix="oracle-")
            atexit.register(shutil.rmtree, out_dir, True)
            make.append("BUILD=" + out_dir)
            path = os.path.join(out_dir, "liboracle.so")
        subprocess.check_call(make, stdout=subprocess.DEVNULL)
        if path != LIB_PATH:
            _tmp_lib = path
    if os.path.isdir("/root/reference/third_party/simdcomp/src") and not os.path.exists(REF_SIMDCOMP):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "-s", "ref"], stdout=subprocess.DEVNULL)
    return path


class BM25Stats(C.Structure):
    _fields_ = [("idf", C.c_float), ("norm_const", C.c_float), ("norm_length", C.c_float)]


class Hit(C.Structure):
    _fields_ = [("score", C.c_float), ("doc", C.c_uint32), ("seg", C.c_uint32)]


class TermMeta(C.Structure):
    _fields_ = [("docs_count", C.c_uint32), ("freq", C.c_uint32), ("doc_start", C.c_uint64),
                ("e_skip_start", C.c_uint64)]


class Pred(C.Structure):
    _fields_ = [("field", C.c_uint64), ("op", C.c_int32), ("is_float", C.c_int32),
                ("lo_i", C.c_int64), ("hi_i", C.c_int64), ("lo_f", C.c_double), ("hi_f", C.c_double)]


class BM25Term(C.Structure):
    _fields_ = [("idf", C.c_float), ("norm_const", C.c_float), ("norm_length", C.c_float),
                ("boost", C.c_float), ("term", C.c_uint32)]


class GroupRow(C.Structure):
    _fields_ = [("key", C.c_int64), ("count", C.c_uint64), ("sum_i128", C.c_int64 * 2),
                ("sum_f64", C.c_double), ("cnt_f64", C.c_uint64)]


OP = dict(LT=0, LE=1, GT=2, GE=3, EQ=4, NE=5, BETWEEN=6, IS_NULL=7, IS_NOT_NULL=8)
HIT_DTYPE = np.dtype([("score", "<f4"), ("doc", "<u4"), ("seg", "<u4")])
GROUP_DTYPE = np.dtype([("key", "<i8"), ("count", "<u8"), ("sum_lo", "<i8"), ("sum_hi", "<i8"),
                        ("sum_f64", "<f8"), ("cnt_f64", "<u8")])

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    L = C.CDLL(build())
    u32p, u8p, u64p, f32p = (C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.POINTER(C.c_uint64),
                             C.POINTER(C.c_float))
    vp = C.c_void_p
    L.orc_pack128.argtypes = [vp, vp, C.c_uint32]
    L.orc_unpack128.argtypes = [vp, vp, C.c_uint32]
    L.orc_pack128_d1.argtypes = [C.c_uint32, vp, vp, C.c_uint32]
    L.orc_unpack128_d1.argtypes = [C.c_uint32, vp, vp, C.c_uint32]
    L.orc_use_simdcomp_ref.argtypes = [C.c_char_p]
    for n in ("orc_svb_encode",):
        getattr(L, n).argtypes = [vp, C.c_uint32, vp]
        getattr(L, n).restype = C.c_size_t
    L.orc_svb_decode.argtypes = [vp, vp, C.c_uint32]
    L.orc_svb_decode.restype = C.c_size_t
    L.orc_svb_delta_encode.argtypes = [vp, C.c_uint32, vp, C.c_uint32]
    L.orc_svb_delta_encode.restype = C.c_size_t
    L.orc_svb_delta_decode.argtypes = [vp, vp, C.c_uint32, C.c_uint32]
    L.orc_svb_delta_decode.restype = C.c_size_t
    L.orc_encode_doc_block.argtypes = [vp, C.c_uint32, C.c_uint32, vp]
    L.orc_encode_doc_block.restype = C.c_size_t
    L.orc_decode_doc_block.argtypes = [vp, C.c_uint32, C.c_uint32, vp]
    L.orc_decode_doc_block.restype = C.c_size_t
    L.orc_encode_freq_block.argtypes = [vp, C.c_uint32, vp]
    L.orc_encode_freq_block.restype = C.c_size_t
    L.orc_decode_freq_block.argtypes = [vp, C.c_uint32, vp]
    L.orc_decode_freq_block.restype = C.c_size_t
    L.orc_bm25_collect.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_float, C.c_float,
                                   C.POINTER(BM25Stats)]
    L.orc_bm25_num.argtypes = [C.c_float, C.c_float, C.c_float]
    L.orc_bm25_num.restype = C.c_float
    L.orc_bm25_score.argtypes = [vp, vp, C.c_uint32, C.c_float, C.c_float, C.c_float, vp]
    L.orc_collect_nth.argtypes = [vp, vp, C.c_uint64, C.c_uint32, C.c_float, vp, u32p, f32p]
    L.orc_collect_nth.restype = C.c_uint64
    L.orc_segment_new.argtypes = [C.c_uint32, C.c_int, C.c_float]
    L.orc_segment_new.restype = vp
    L.orc_segment_free.argtypes = [vp]
    L.orc_segment_set_norms.argtypes = [vp, vp]
    L.orc_segment_add_term.argtypes = [vp, vp, vp, C.c_uint32]
    L.orc_segment_add_term.restype = C.c_int64
    L.orc_segment_doc_bytes.argtypes = [vp, u64p]
    L.orc_segment_doc_bytes.restype = vp
    L.orc_segment_num_terms.argtypes = [vp]
    L.orc_segment_num_terms.restype = C.c_uint32
    L.orc_segment_term_meta.argtypes = [vp, C.c_uint32, C.POINTER(TermMeta)]
    L.orc_segment_docs.argtypes = [vp]
    L.orc_segment_docs.restype = C.c_uint32
    L.orc_segment_norm_sum.argtypes = [vp]
    L.orc_segment_norm_sum.restype = C.c_uint64
    L.orc_segment_norm_bytes.argtypes = [vp, u32p]
    L.orc_segment_norm_bytes.restype = vp
    L.orc_segment_decode_term.argtypes = [vp, C.c_uint32, vp, vp]
    L.orc_segment_decode_term.restype = C.c_uint32
    L.orc_segment_skip_level0.argtypes = [vp, C.c_uint32, vp, vp, vp, vp, u32p, u32p, u32p]
    L.orc_segment_skip_level0.restype = C.c_uint32
    L.orc_segment_add_column.argtypes = [vp, C.c_uint64, C.c_int, vp, vp, C.c_uint64]
    L.orc_segment_set_docs_mask.argtypes = [vp, vp, C.c_size_t]
    L.orc_bm25_topk.argtypes = [vp, C.c_size_t, C.c_int, vp, C.c_size_t, C.c_float, C.c_float, vp, C.c_uint32,
                                C.c_float, C.c_int, vp, u32p, u64p, u64p]
    L.orc_bm25_topk_batch.argtypes = [vp, C.c_size_t, C.c_int, vp, vp, C.c_size_t, C.c_float, C.c_float, vp, C.c_uint32,
                                      C.c_float, C.c_int, C.c_int, vp, vp, vp, u64p]
    L.orc_synth_segment.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, vp, u64p]
    L.orc_synth_segment.restype = vp
    L.orc_filter_bitmap.argtypes = [vp, vp, C.c_size_t, vp]
    L.orc_filter_count_sum.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_uint64, C.c_int, u64p, vp,
                                       C.POINTER(C.c_double)]
    L.orc_filter_groupby.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_uint64, C.c_uint64, C.c_uint64,
                                     C.c_int, vp, C.c_uint64, u64p]
    L.orc_tfidf_idf.argtypes = [C.c_uint64, C.c_uint64]
    L.orc_tfidf_idf.restype = C.c_float
    L.orc_set_contract.argtypes = [C.c_int]
    L.orc_set_contract.restype = None
    L.orc_count_max_levels.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64]
    L.orc_count_max_levels.restype = C.c_uint32
    L.orc_synth_hash.argtypes = [C.c_uint64, C.c_uint64]
    L.orc_synth_hash.restype = C.c_uint64
    L.orc_synth_column.argtypes = [C.c_uint64, C.c_int, C.c_uint64, C.c_uint64, vp]
    L.orc_synth_doc_lengths.argtypes = [C.c_uint64, C.c_uint32, vp]
    L.orc_synth_term.argtypes = [C.c_uint32, C.c_uint64, C.c_uint32, vp, vp, vp]
    L.orc_synth_term.restype = C.c_uint32
    _lib = L
    return L


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def use_simdcomp_ref(on=True):
    """Route the oracle's 128-value unpack through the reference's own simdcomp."""
    if on:
        if not os.path.exists(REF_SIMDCOMP):
            return False
        return lib().orc_use_simdcomp_ref(REF_SIMDCOMP.encode()) == 0
    lib().orc_use_simdcomp_ref(None)
    return True


# ---------------------------------------------------------------- codec helpers
def encode_doc_block(docs, prev):
    docs = np.ascontiguousarray(docs, dtype=np.uint32)
    out = np.zeros(4 * 128 + 64, dtype=np.uint8)
    n = lib().orc_encode_doc_block(ptr(docs), len(docs), prev, ptr(out))
    return out[:n].copy()


def decode_doc_block(buf, length, prev):
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    pad = np.concatenate([buf, np.zeros(64, np.uint8)])
    out = np.zeros(128, dtype=np.uint32)
    n = lib().orc_decode_doc_block(ptr(pad), length, prev, ptr(out))
    return out[:length].copy(), n


def encode_freq_block(freqs):
    freqs = np.ascontiguousarray(freqs, dtype=np.uint32)
    out = np.zeros(4 * 128 + 64, dtype=np.uint8)
    n = lib().orc_encode_freq_block(ptr(freqs), len(freqs), ptr(out))
    return out[:n].copy()


def decode_freq_block(buf, length):
    buf = np.ascontiguousarray(buf, dtype=np.uint8)
    pad = np.concatenate([buf, np.zeros(64, np.uint8)])
    out = np.zeros(128, dtype=np.uint32)
    n = lib().orc_decode_freq_block(ptr(pad), length, ptr(out))
    return out[:length].copy(), n


def bm25_stats(docs_with_field, total_term_freq, docs_with_term, k=1.2, b=0.75):
    st = BM25Stats()
    lib().orc_bm25_collect(docs_with_field, total_term_freq, docs_with_term, k, b, C.byref(st))
    return st


def tfidf_idf(docs_with_field, docs_with_term):
    return float(lib().orc_tfidf_idf(int(docs_with_field), int(docs_with_term)))


def set_contract(on):
    """1: c1 of the BM25 form as one fused multiply-add (a clang -mfma build of bm25.cpp:105); 0: source order."""
    lib().orc_set_contract(1 if on else 0)


def bm25_score(freq, norm, stats, k=1.2, boost=1.0):
    freq = np.ascontiguousarray(freq, dtype=np.uint32)
    out = np.zeros(len(freq), dtype=np.float32)
    num = lib().orc_bm25_num(k, boost, stats.idf)
    nptr = None
    if norm is not None:
        norm = np.ascontiguousarray(norm, dtype=np.uint32)
        nptr = ptr(norm)
    lib().orc_bm25_score(ptr(freq), nptr, len(freq), num, stats.norm_const, stats.norm_length, ptr(out))
    return out


def collect_nth(scores, docs, k, threshold_in=np.finfo(np.float32).tiny):
    scores = np.ascontiguousarray(scores, dtype=np.float32)
    docs = np.ascontiguousarray(docs, dtype=np.uint32)
    hits = np.zeros(2 * k, dtype=HIT_DTYPE)
    acc = C.c_uint32()
    thr = C.c_float()
    total = lib().orc_collect_nth(ptr(scores), ptr(docs), len(scores), k, threshold_in, ptr(hits),
                                  C.byref(acc), C.byref(thr))
    return hits[:acc.value].copy(), total, thr.value


def make_pred(field, op, lo=0, hi=0, is_float=False):
    p = Pred()
    p.field = field
    p.op = OP[op] if isinstance(op, str) else op
    p.is_float = 1 if is_float else 0
    if is_float:
        p.lo_f, p.hi_f = float(lo), float(hi)
    else:
        p.lo_i, p.hi_i = int(lo), int(hi)
    return p


def pred_array(preds):
    arr = (Pred * max(len(preds), 1))()
    for i, p in enumerate(preds):
        arr[i] = p
    return arr


COLTYPE = {np.dtype("int64"): 0, np.dtype("float64"): 1, np.dtype("int32"): 2}


class Segment:
    """One index segment held by the oracle: postings (.doc stream), norms, table columns."""

    def __init__(self, n_docs, has_wand=True, wand_b=0.75):
        self.n_docs = int(n_docs)
        self.h = lib().orc_segment_new(self.n_docs, 1 if has_wand else 0, wand_b)
        self.has_wand = has_wand
        self.has_norms = False

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_segment_free(self.h)
            self.h = None

    def set_norms(self, norms):
        norms = np.ascontiguousarray(norms, dtype=np.uint32)
        assert len(norms) == self.n_docs
        lib().orc_segment_set_norms(self.h, ptr(norms))
        self.has_norms = True

    def add_term(self, docs, freqs):
        docs = np.ascontiguousarray(docs, dtype=np.uint32)
        freqs = np.ascontiguousarray(freqs, dtype=np.uint32)
        assert len(docs) == len(freqs)
        return int(lib().orc_segment_add_term(self.h, ptr(docs), ptr(freqs), len(docs)))

    def doc_bytes(self):
        size = C.c_uint64()
        p = lib().orc_segment_doc_bytes(self.h, C.byref(size))
        if size.value == 0:
            return np.zeros(0, np.uint8)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(size.value,)).copy()

    def num_terms(self):
        return int(lib().orc_segment_num_terms(self.h))

    def term_meta(self, t):
        m = TermMeta()
        lib().orc_segment_term_meta(self.h, t, C.byref(m))
        return m

    def term_metas(self):
        return [self.term_meta(t) for t in range(self.num_terms())]

    def norm_sum(self):
        return int(lib().orc_segment_norm_sum(self.h))

    def norm_bytes(self):
        w = C.c_uint32()
        p = lib().orc_segment_norm_bytes(self.h, C.byref(w))
        n = self.n_docs * w.value
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n,)).copy(), w.value

    def decode_term(self, t):
        m = self.term_meta(t)
        docs = np.zeros(max(m.docs_count, 1), np.uint32)
        freqs = np.zeros(max(m.docs_count, 1), np.uint32)
        n = lib().orc_segment_decode_term(self.h, t, ptr(docs), ptr(freqs))
        return docs[:n], freqs[:n]

    def skip_level0(self, t):
        m = self.term_meta(t)
        cap = max((m.docs_count - 1) // 128, 1) if m.docs_count else 1
        last = np.zeros(cap, np.uint32)
        dptr = np.zeros(cap, np.uint64)
        wf = np.zeros(cap, np.uint32)
        wn = np.zeros(cap, np.uint32)
        rf, rn, nl = C.c_uint32(), C.c_uint32(), C.c_uint32()
        n = lib().orc_segment_skip_level0(self.h, t, ptr(last), ptr(dptr), ptr(wf), ptr(wn), C.byref(rf),
                                          C.byref(rn), C.byref(nl))
        return dict(last_doc=last[:n], doc_ptr=dptr[:n], wand_freq=wf[:n], wand_norm=wn[:n],
                    root=(rf.value, rn.value), num_levels=nl.value)

    def set_docs_mask(self, deleted_docs):
        d = np.ascontiguousarray(deleted_docs, dtype=np.uint32)
        rc = lib().orc_segment_set_docs_mask(self.h, ptr(d) if len(d) else None, len(d))
        assert rc == 0

    def add_column(self, field, values, validity=None):
        values = np.ascontiguousarray(values)
        t = COLTYPE[values.dtype]
        vptr = None
        if validity is not None:
            validity = np.ascontiguousarray(validity, dtype=np.uint64)
            vptr = ptr(validity)
        rc = lib().orc_segment_add_column(self.h, field, t, ptr(values), vptr, len(values))
        assert rc == 0


def _seg_array(segs):
    arr = (C.c_void_p * len(segs))()
    for i, s in enumerate(segs):
        arr[i] = s.h
    return arr


def term_array(terms):
    arr = (BM25Term * max(len(terms), 1))()
    for i, t in enumerate(terms):
        arr[i] = t
    return arr


def bm25_topk(segs, kind, terms, k, k1=1.2, filt=None, threshold_in=np.finfo(np.float32).tiny, mode=0, b=0.75):
    """terms: list of BM25Term. Returns (hits ndarray, total_matches, postings_scored)."""
    hits = np.zeros(max(k, 1), dtype=HIT_DTYPE)
    n_out, total, scored = C.c_uint32(), C.c_uint64(), C.c_uint64()
    fp = C.byref(filt) if filt is not None else None
    rc = lib().orc_bm25_topk(_seg_array(segs), len(segs), 1 if kind in (1, "AND") else 0, term_array(terms),
                             len(terms), k1, b, fp, k, threshold_in, mode, ptr(hits), C.byref(n_out),
                             C.byref(total), C.byref(scored))
    assert rc == 0
    return hits[:n_out.value].copy(), total.value, scored.value


def bm25_topk_batch(segs, kind, queries_terms, k, k1=1.2, filt=None, threshold_in=np.finfo(np.float32).tiny,
                    mode=2, threads=1, b=0.75):
    """queries_terms: list of lists of BM25Term. Returns (hits [Q,k], n_out, total, postings_scored)."""
    nq = len(queries_terms)
    flat = [t for q in queries_terms for t in q]
    off = np.zeros(nq + 1, np.uint32)
    off[1:] = np.cumsum([len(q) for q in queries_terms])
    hits = np.zeros((nq, k), dtype=HIT_DTYPE)
    n_out = np.zeros(nq, np.uint32)
    total = np.zeros(nq, np.uint64)
    scored = C.c_uint64()
    fp = C.byref(filt) if filt is not None else None
    rc = lib().orc_bm25_topk_batch(_seg_array(segs), len(segs), 1 if kind in (1, "AND") else 0, term_array(flat),
                                   ptr(off), nq, k1, b, fp, k, threshold_in, mode, threads, ptr(hits), ptr(n_out),
                                   ptr(total), C.byref(scored))
    assert rc == 0
    return hits, n_out, total, scored.value


def synth_segment_mt(n_docs, t0, nt, doc0=0, threads=8):
    """Multi-threaded oracle builder for a synthetic shard: returns (Segment, docs_count[nt], sum_dl)."""
    dc = np.zeros(nt, np.uint32)
    sdl = C.c_uint64()
    seg = Segment.__new__(Segment)
    seg.n_docs = int(n_docs)
    seg.h = lib().orc_synth_segment(doc0, n_docs, t0, nt, threads, ptr(dc), C.byref(sdl))
    seg.has_wand = True
    seg.has_norms = True
    return seg, dc, sdl.value


def filter_bitmap(seg, preds, rows):
    mask = np.zeros((rows + 63) // 64, dtype=np.uint64)
    rc = lib().orc_filter_bitmap(seg.h, pred_array(preds), len(preds), ptr(mask))
    assert rc == 0
    return mask


def filter_count_sum(segs, preds, sum_field, threads=1):
    cnt = C.c_uint64()
    s128 = (C.c_int64 * 2)()
    sf = C.c_double()
    rc = lib().orc_filter_count_sum(_seg_array(segs), len(segs), pred_array(preds), len(preds), sum_field,
                                    threads, C.byref(cnt), s128, C.byref(sf))
    assert rc == 0
    si = (int(s128[1]) << 64) | (int(s128[0]) & 0xFFFFFFFFFFFFFFFF)
    return cnt.value, si, sf.value


def filter_groupby(segs, preds, key_field, sum_int_field, avg_f64_field, cap, threads=1):
    out = np.zeros(cap, dtype=GROUP_DTYPE)
    n = C.c_uint64()
    rc = lib().orc_filter_groupby(_seg_array(segs), len(segs), pred_array(preds), len(preds), key_field,
                                  sum_int_field, avg_f64_field, threads, ptr(out), cap, C.byref(n))
    assert rc == 0, rc
    return out[:n.value].copy()


# ---------------------------------------------------------------- synthetic inputs
def synth_column(stream, kind, row0, rows):
    out = np.zeros(rows, dtype=np.float64 if kind in (2, 4) else np.int64)
    lib().orc_synth_column(stream, kind, row0, rows, ptr(out))
    return out


def synth_doc_lengths(doc0, n):
    out = np.zeros(n, np.uint32)
    lib().orc_synth_doc_lengths(doc0, n, ptr(out))
    return out


def synth_term(t, doc0, n, dl):
    docs = np.zeros(n, np.uint32)
    freqs = np.zeros(n, np.uint32)
    c = lib().orc_synth_term(t, doc0, n, ptr(dl), ptr(docs), ptr(freqs))
    return docs[:c].copy(), freqs[:c].copy()


def synth_segment(n_docs, terms, doc0=0, has_wand=True):
    """Oracle-built synthetic segment: norms + the given synthetic term ids."""
    seg = Segment(n_docs, has_wand=has_wand)
    dl = synth_doc_lengths(doc0, n_docs)
    seg.set_norms(dl)
    lists = []
    for t in terms:
        d, f = synth_term(t, doc0, n_docs, dl)
        seg.add_term(d, f)
        lists.append((d, f))
    return seg, dl, lists
