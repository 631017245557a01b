"""CPU tests: pin the oracle (oracle/*.c) against the golden vectors of SURVEY.md Appendix A
(captured from the real reference build) and against streams of the real reference itself
(liblz4 1.9.4 / libzstd 1.5.5 behind the unmodified lib/*-mt_*.c), re-made through the same
library calls and checked against digests of the reference's output (tests/golden/reference_streams.json)."""
import os

import numpy as np
import pytest

import _oracle as o
import zstdmt_b200 as z

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def hexb(s):
    return np.frombuffer(bytes.fromhex(s.replace(" ", "")), dtype=np.uint8)


# ---- Appendix A vectors -------------------------------------------------------------
LZ4_EMPTY = "502a4d18 04000000 0f000000 04224d18 64 40 a7 00000000 055dcc02"
LZ4_A = "502a4d18 04000000 1c000000 04224d18 6c 40 0100000000000000 49 01000080 41 00000000 4d9a6510"
ZSTD_EMPTY = "502a4d18 04000000 09000000 28b52ffd 20 00 010000"


def test_xxh32_known_answers():
    assert o.xxh32(b"") == 0x02CC5D05                         # checksum bytes 05 5d cc 02 of the empty frame
    assert o.xxh32(np.zeros(1 << 20, np.uint8)) == 0x9430F97F  # frame ends 7f f9 30 94 (Appendix A)
    assert o.xxh32(b"A") == 0x10659A4D                        # "A" frame ends 4d 9a 65 10


def test_golden_lz4_empty_and_A():
    rc, out = o.orc_decode(o.CODEC_LZ4, hexb(LZ4_EMPTY), 16)
    assert rc == 0 and out.size == 0
    rc, out = o.orc_decode(o.CODEC_LZ4, hexb(LZ4_A), 16)
    assert rc == 0 and out.tobytes() == b"A"
    # our encoder restatement must emit exactly the reference's bytes for these two
    assert o.orc_encode_lz4(b"").tobytes() == hexb(LZ4_EMPTY).tobytes()
    assert o.orc_encode_lz4(b"A").tobytes() == hexb(LZ4_A).tobytes()


def test_golden_zstd_empty():
    rc, out = o.orc_decode(o.CODEC_ZSTD, hexb(ZSTD_EMPTY), 16)
    assert rc == 0 and out.size == 0


def test_golden_header_checksums():
    # HC bytes 0xA7 (empty), 0x49 ("A"), 0x88 (1 MiB) from Appendix A
    assert (o.xxh32(bytes([0x64, 0x40])) >> 8) & 0xFF == 0xA7
    assert (o.xxh32(bytes([0x6C, 0x40]) + (1).to_bytes(8, "little")) >> 8) & 0xFF == 0x49
    assert (o.xxh32(bytes([0x4C, 0x40]) + (1 << 20).to_bytes(8, "little")) >> 8) & 0xFF == 0x88


def test_golden_fixture_files():
    """tests/golden/*.bin were produced by the real reference (tests/golden/make_golden.py)."""
    import json
    with open(os.path.join(GOLD, "manifest.json")) as f:
        man = json.load(f)
    assert man["cases"]
    for case in man["cases"]:
        framed = np.fromfile(os.path.join(GOLD, case["file"]), dtype=np.uint8)
        src = z.gen_stream(case["kind"], case["n"], case["chunk"], first=case["first"])
        codec = o.CODEC_LZ4 if case["codec"] == "lz4" else o.CODEC_ZSTD
        rc, out = o.orc_decode(codec, framed, case["n"])
        assert rc == 0, case
        assert out.size == case["n"] and np.array_equal(out, src), case
        assert o.xxh32(framed) == case["xxh32_framed"], case


def test_ref_lz4_zeros_1mib_matches_appendix_a():
    f, _ = o.reference_stream(o.CODEC_LZ4, np.zeros(1 << 20, np.uint8), 1, 1 << 20)
    assert f.size == 4356
    assert f[:28].tobytes().hex() == "502a4d1804000000f810000004224d184c400000100000000000880b010000"[:56]
    assert f[-8:].tobytes().hex() == "000000007ff93094"
    rc, out = o.orc_decode(o.CODEC_LZ4, f, 1 << 20)
    assert rc == 0 and out.size == 1 << 20 and not out.any()


@pytest.mark.parametrize("codec,level", [(1, 1), (1, 3), (2, 1), (2, 3), (2, 9)])
@pytest.mark.parametrize("kind", [z.GEN_MIX, z.GEN_TEXT, z.GEN_RANDOM, z.GEN_ZEROS])
def test_oracle_decodes_reference_streams(codec, level, kind):
    n = (5 << 20) + 12345 if kind == z.GEN_MIX else (1 << 20) + 77
    src = z.gen_stream(kind, n, 1 << 20)
    f, _ = o.reference_stream(codec, src, level, 1 << 20)
    rc, out = o.orc_decode(codec, f, n)
    assert rc == 0 and out.size == n and np.array_equal(out, src)


@pytest.mark.parametrize("n", [0, 1, 11, 12, 13, 39, 40, 65535, 65536, 65537, (1 << 20) - 1, (1 << 20) + 1])
def test_b200_encoder_twin_roundtrips_through_reference(n):
    src = z.gen_stream(z.GEN_MIX, n, 1 << 20, first=1)
    f = o.orc_encode_lz4(src)
    rc, out, frames = o.lib_decompress(o.CODEC_LZ4, f, n)           # liblz4, the reference's decoder
    assert rc == 0 and out.size == n and np.array_equal(out, src) and frames == max(1, -(-n // (1 << 20)))
    rc, out = o.orc_decode(o.CODEC_LZ4, f, n)
    assert rc == 0 and np.array_equal(out, src)


def test_oracle_rejects_corruption():
    src = z.gen_stream(z.GEN_TEXT, 200000, 1 << 20)
    f = o.orc_encode_lz4(src)
    bad = f.copy(); bad[-1] ^= 1                    # content checksum
    assert o.orc_decode(o.CODEC_LZ4, bad, src.size)[0] == -7
    bad = f.copy(); bad[0] ^= 1                     # skippable magic
    assert o.orc_decode(o.CODEC_LZ4, bad, src.size)[0] == -2
    bad = f.copy(); bad[12 + 4 + 2 + 8] ^= 1        # header checksum byte
    assert o.orc_decode(o.CODEC_LZ4, bad, src.size)[0] == -4
    assert o.orc_decode(o.CODEC_LZ4, f[:-3], src.size)[0] == -1


@pytest.mark.parametrize("chunk", [65536, 200000, 1 << 20])
def test_b200_encoder_twin_length_field_corner_cases(chunk):
    """The CPU twin of the GPU LZ4 encoder on the stream that exercises every length-field form (15 / 270 / 1290 ...
    boundaries, 255-runs, block-ending literals): the real liblz4 behind the reference wrapper must restore it."""
    from _data import long_runs_stream
    src = long_runs_stream(1)
    framed = o.orc_encode_lz4(src, chunk)
    rc, back = o.orc_decode(o.CODEC_LZ4, framed, src.size)
    assert rc == 0 and np.array_equal(back, src)
    rc, back, _ = o.lib_decompress(o.CODEC_LZ4, framed, src.size)
    assert rc == 0 and np.array_equal(back, src)
