"""Oracle codec: block encoder choice + round trips (format_block_128.hpp), StreamVByte round trips."""
import numpy as np
import pytest

import orc

RNG = np.random.default_rng(0x5EDB2026)


def _sorted_docs(n, prev, mean_gap):
    gaps = RNG.geometric(1.0 / mean_gap, size=n).astype(np.uint64)
    return (prev + np.cumsum(gaps)).astype(np.uint32)


DE = dict(values=0, same08=1, same16=2, same32=3, bitset=4, svb=5, dsvb=7, bitpack02=8)
E = dict(values=0, same08=1, same16=2, same32=3, svb=4, bitpack01=5)


def test_doc_block_encoder_choices():
    """Encoder picks the smallest candidate in the reference's order (format_block_128.hpp:57-154)."""
    # all deltas equal -> all_same (1 byte payload), also for a single-doc tail
    d = np.arange(1, 129, dtype=np.uint32) * 3 + 10
    buf = orc.encode_doc_block(d, 10)
    assert buf[0] == DE["same08"] and len(buf) == 2 and buf[1] == 3
    buf = orc.encode_doc_block(np.array([1000], np.uint32), 0)
    assert buf[0] == DE["same16"] and len(buf) == 3
    buf = orc.encode_doc_block(np.array([70000], np.uint32), 0)
    assert buf[0] == DE["same32"] and len(buf) == 5
    # dense block (p = 0.5): bitset wins over bit packing when 1+8*words-2 < 16*bits
    d = _sorted_docs(128, 77, 2.0)
    buf = orc.encode_doc_block(d, 77)
    words = (int(d[-1]) - 77 + 1 + 63) // 64
    bits = int(np.max(np.diff(np.concatenate([[77], d]))).item()).bit_length()
    if 1 + 8 * words - 2 < 16 * bits:
        assert buf[0] == DE["bitset"] and buf[1] == words and len(buf) == 2 + 8 * words
    else:
        assert buf[0] == DE["bitpack02"] + bits - 2
    # sparse full block -> delta bit packing, 16*b bytes
    d = _sorted_docs(128, 5, 1000.0)
    buf = orc.encode_doc_block(d, 5)
    bits = int(np.max(np.diff(np.concatenate([[5], d]))).item()).bit_length()
    assert buf[0] == DE["bitpack02"] + bits - 2 and len(buf) == 1 + 16 * bits
    # sparse tail -> (delta) streamvbyte with u16 size prefix; never bit packing
    d = _sorted_docs(50, 5, 1000.0)
    buf = orc.encode_doc_block(d, 5)
    assert buf[0] in (DE["svb"], DE["dsvb"], DE["bitset"])
    assert int(buf[1]) | (int(buf[2]) << 8) == len(buf) - 3 or buf[0] == DE["bitset"]


@pytest.mark.parametrize("length", [1, 2, 3, 4, 5, 31, 32, 33, 64, 100, 127, 128])
@pytest.mark.parametrize("gap", [1.0, 1.5, 2.0, 3.0, 10.0, 100.0, 5000.0, 3.0e6])
def test_doc_block_roundtrip(length, gap):
    for _ in range(3):
        prev = int(RNG.integers(0, 5000))
        if gap == 1.0:
            d = (prev + 1 + np.arange(length)).astype(np.uint32)
        else:
            d = _sorted_docs(length, prev, gap)
        buf = orc.encode_doc_block(d, prev)
        back, used = orc.decode_doc_block(buf, length, prev)
        assert used == len(buf)
        assert np.array_equal(back, d)


@pytest.mark.parametrize("length", [1, 3, 4, 17, 127, 128])
@pytest.mark.parametrize("maxf", [1, 2, 3, 9, 300, 70000, 2 ** 31 - 1])
def test_freq_block_roundtrip(length, maxf):
    for same in (False, True):
        f = RNG.integers(1, maxf + 1, size=length, dtype=np.uint64).astype(np.uint32)
        if same:
            f[:] = maxf
        buf = orc.encode_freq_block(f)
        back, used = orc.decode_freq_block(buf, length)
        assert used == len(buf)
        assert np.array_equal(back, f)
        if bool(np.all(f == f[0])):
            assert buf[0] in (E["same08"], E["same16"], E["same32"])
        elif length == 128:
            assert buf[0] >= E["bitpack01"] or buf[0] == E["values"]
        else:
            assert buf[0] in (E["svb"], E["values"])


def test_streamvbyte_layout_and_roundtrip():
    """Public StreamVByte 1234 layout: ceil(n/4) key bytes, 2 bits/value LSB-first = len-1."""
    L = orc.lib()
    v = np.array([1, 256, 65536, 1 << 24, 7], np.uint32)
    out = np.zeros(64, np.uint8)
    n = L.orc_svb_encode(orc.ptr(v), len(v), orc.ptr(out))
    assert n == 2 + 1 + 2 + 3 + 4 + 1
    assert out[0] == (0 | (1 << 2) | (2 << 4) | (3 << 6)) and out[1] == 0
    assert list(out[2:6]) == [1, 0, 1, 0]
    back = np.zeros(len(v), np.uint32)
    assert L.orc_svb_decode(orc.ptr(out), orc.ptr(back), len(v)) == n
    assert np.array_equal(back, v)
    for length in (1, 5, 64, 127):
        d = _sorted_docs(length, 9, 70000.0)
        buf = np.zeros(5 * 128, np.uint8)
        n = L.orc_svb_delta_encode(orc.ptr(d), length, orc.ptr(buf), 9)
        back = np.zeros(length, np.uint32)
        assert L.orc_svb_delta_decode(orc.ptr(buf), orc.ptr(back), length, 9) == n
        assert np.array_equal(back, d)
