"""CPU-side checks of the product's host code (no GPU): the C ABI library loads and exports every
declared symbol, the PostingsWriter mirror is byte-identical to the oracle's writer restatement, and
the staging parser's block table agrees with the oracle's reading of the same ".doc" stream."""
import os
import re

import numpy as np
import pytest

import orc
import serenedb_b200 as sdb
from serenedb_b200 import _native


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(orc.ROOT, "include", "sdbg.h")).read()
    declared = set(re.findall(r"\b(sdbg_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = _native.lib()
    for name in sorted(declared):
        assert hasattr(L, name), f"libsdbg.so does not export {name}"
    assert declared == set(_native.SIGNATURES), declared ^ set(_native.SIGNATURES)


def test_no_device_is_a_loud_error_not_a_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(_native.SdbgError, match="ENODEVICE"):
        sdb.Context(0)


def _random_lists(rng, n):
    cases = [1, 2, 5, 127, 128, 129, 255, 256, 257, 1000, 4096, 4097, n]
    out = []
    for c in cases:
        docs = np.sort(rng.choice(np.arange(1, n + 1), size=c, replace=False)).astype(np.uint32)
        out.append(docs)
    # dense / regular shapes that hit all-same and bitset encodings
    out.append(np.arange(1, n + 1, dtype=np.uint32))
    out.append(np.arange(3, n + 1, 7, dtype=np.uint32))
    out.append(np.sort(rng.choice(np.arange(1, 2000), size=900, replace=False)).astype(np.uint32))
    return out


@pytest.mark.parametrize("has_wand", [True, False])
def test_writer_mirror_is_byte_identical_to_oracle(has_wand):
    rng = np.random.default_rng(11)
    n = 20000
    dl = rng.integers(1, 400, size=n).astype(np.uint32)
    oseg = orc.Segment(n, has_wand=has_wand)
    oseg.set_norms(dl)
    w = sdb.PostingsWriter(n, norms=dl, has_wand=has_wand)
    for docs in _random_lists(rng, n):
        freqs = np.minimum(rng.geometric(0.4, size=len(docs)), dl[docs - 1]).astype(np.uint32)
        oseg.add_term(docs, freqs)
        w.add_term(docs, freqs)
    doc, metas = w.finish()
    assert np.array_equal(doc, oseg.doc_bytes())
    for t, m in enumerate(oseg.term_metas()):
        assert (m.docs_count, m.freq, m.doc_start, m.e_skip_start) == tuple(int(x) for x in metas[t])


def test_writer_matches_oracle_on_synthetic_corpus():
    n = 300_000
    terms = [0, 2, 17, 100, 255]
    oseg, dl, lists = orc.synth_segment(n, terms)
    w = sdb.PostingsWriter(n, norms=dl)
    for d, f in lists:
        w.add_term(d, f)
    doc, metas = w.finish()
    assert np.array_equal(doc, oseg.doc_bytes())
    assert _native.lib().sdbg_synth_hash(100, 12345) == orc.lib().orc_synth_hash(100, 12345)


def test_stage_parser_block_table_matches_oracle():
    rng = np.random.default_rng(5)
    n = 50000
    dl = rng.integers(1, 300, size=n).astype(np.uint32)
    oseg = orc.Segment(n, has_wand=True)
    oseg.set_norms(dl)
    lists = []
    for docs in _random_lists(rng, n):
        freqs = np.minimum(rng.geometric(0.5, size=len(docs)), dl[docs - 1]).astype(np.uint32)
        oseg.add_term(docs, freqs)
        lists.append((docs, freqs))
    metas = np.array([(m.docs_count, m.freq, m.doc_start, m.e_skip_start) for m in oseg.term_metas()],
                     dtype=sdb.engine.TERM_META_DTYPE)
    st = sdb.stage_parse_host(oseg.doc_bytes(), metas, has_wand=True)
    for t, (docs, freqs) in enumerate(lists):
        b0, b1 = st["term_blk_begin"][t], st["term_blk_begin"][t + 1]
        nblk = (len(docs) + 127) // 128
        assert b1 - b0 == nblk
        last = docs[127::128].tolist()
        if len(docs) % 128:
            last.append(int(docs[-1]))
        assert st["last_doc"][b0:b1].tolist() == last
        assert st["prev_last"][b0:b1].tolist() == [0] + last[:-1]
        lens = ((st["packed"][b0:b1] >> 12) & 127) + 1
        assert lens.tolist() == [128] * (len(docs) // 128) + ([len(docs) % 128] if len(docs) % 128 else [])
        if len(docs) > 1:
            sk = oseg.skip_level0(t)
            ne = len(sk["last_doc"])
            assert st["max_freq"][b0:b0 + ne].tolist() == sk["wand_freq"].tolist()
            assert st["max_norm"][b0:b0 + ne].tolist() == sk["wand_norm"].tolist()
            # blocks without a level-0 entry fall back to the list maximum
            assert (st["max_freq"][b1 - 1], st["max_norm"][b1 - 1]) == sk["root"] or ne == nblk


def test_stage_parser_rejects_corrupt_streams():
    n = 5000
    oseg, dl, lists = orc.synth_segment(n, [0, 5])
    metas = np.array([(m.docs_count, m.freq, m.doc_start, m.e_skip_start) for m in oseg.term_metas()],
                     dtype=sdb.engine.TERM_META_DTYPE)
    doc = oseg.doc_bytes()
    bad = doc.copy()
    bad[int(metas[0]["doc_start"])] = 6  # reserved de_for_streamvbyte1234 header
    with pytest.raises(_native.SdbgError, match="EFORMAT"):
        sdb.stage_parse_host(bad, metas)
    with pytest.raises(_native.SdbgError, match="EFORMAT"):
        sdb.stage_parse_host(doc[: len(doc) // 2], metas)


def test_bm25_collect_matches_oracle():
    s = sdb.BM25(1.2, 0.75)
    for dwf, ttf, dwt in [(4, 80, 1), (7, 7, 1), (7, 7, 3), (10_000_000, 1_355_000_000, 1_000_000), (5, 0, 2)]:
        t = s.collect(dwf, ttf, dwt)
        o = orc.bm25_stats(dwf, ttf, dwt)
        assert (t.idf, t.norm_const, t.norm_length) == (o.idf, o.norm_const, o.norm_length)
        assert float(s.num(t)) == orc.lib().orc_bm25_num(1.2, 1.0, o.idf)


def test_cpp_adapters_build_and_fail_loudly_without_gpu():
    """GpuTopKIterator / GpuAggScan compile against the mock reference headers and link with the C ABI;
    without a device the self-test reports SDBG_ENODEVICE instead of computing anything on the CPU."""
    import subprocess
    import torch
    from serenedb_b200 import build as b
    exe = b.build_adapters()
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by tests/test_gpu_adapters.py")
    res = subprocess.run([exe, "1000"], capture_output=True, text=True)
    assert res.returncode == 3 and '"error": -2' in res.stdout


def _for_decode(headers, words, rows):
    """Independent (pure Python) decoder of the bit-packed column format described in include/sdbg.h."""
    out = np.zeros(rows, np.int64)
    for g, hd in enumerate(headers):
        r0 = g * 2048
        bits, base = int(hd["bits"]), int(hd["base"])
        for i in range(min(2048, rows - r0)):
            v = 0
            if bits:
                bit = i * bits
                wi, sh = int(hd["off8"]) + (bit >> 6), bit & 63
                x = (int(words[wi]) >> sh) | ((int(words[wi + 1]) << (64 - sh)) if sh and sh + bits > 64 else 0)
                v = x & ((1 << bits) - 1)
            u = (base + v) & 0xFFFFFFFFFFFFFFFF
            out[r0 + i] = u - (1 << 64) if u >= (1 << 63) else u
    return out


def test_for_bitpacked_column_writer_round_trips():
    """sdbg_pack_for (host-side writer, no GPU needed): frame-of-reference bit-packing in 2048-row groups; widths 0 (constant
    group) .. 64, negative bases, the int64 extremes, ragged last group; capacity errors report the room needed."""
    import ctypes as C
    import serenedb_b200 as sdb
    from serenedb_b200 import _native as N
    rng = np.random.default_rng(1)
    i64 = np.iinfo(np.int64)
    cases = [rng.integers(0, 100000, 5000), rng.integers(-2**62, 2**62, 4097), np.full(3000, -7), np.array([i64.min, i64.max, 0]),
             rng.integers(-1000, 1001, 2048), np.arange(10_000) // 100, np.array([5]), rng.integers(0, 2, 6000)]
    for vals in cases:
        vals = vals.astype(np.int64)
        h, w, rows = sdb.pack_for(vals)
        assert rows == len(vals) and len(h) == (rows + 2047) // 2048
        assert np.array_equal(_for_decode(h, w, rows), vals)
        span = [int(vals[g * 2048:(g + 1) * 2048].max()) - int(vals[g * 2048:(g + 1) * 2048].min()) for g in range(len(h))]
        assert [int(b) for b in h["bits"]] == [s.bit_length() for s in span]          # the narrowest width that holds max - min
    vals = cases[0].astype(np.int64)
    n = C.c_uint64(0)
    hdr = np.zeros(3, sdb.engine.FOR_BLOCK_DTYPE)
    small = np.zeros(4, np.uint64)
    rc = N.lib().sdbg_pack_for(vals.ctypes.data_as(C.c_void_p), len(vals), hdr.ctypes.data_as(C.c_void_p), small.ctypes.data_as(C.c_void_p), 4, C.byref(n))
    assert rc == -6 and n.value == 1330                                                # ECAPACITY, room needed
