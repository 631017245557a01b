"""Write tests/golden/reference_streams.json: digests of what the ORIGINAL project (oracle/_ref: unmodified
lib/{lz4,zstd}-mt_*.c + liblz4 / libzstd) computes for every input the suite compares it on.

  streams : {LZ4MT,ZSTDCB}_compressCCtx output per (codec, level, chunk, input): length, SHA-256, the counters of
            the compress call and of the reference's decoder on that stream.  The tests re-make each stream with
            _oracle.lib_compress and require the same bytes, so they run without oracle/_ref.
  decoded : the reference decoder's result on streams the tests build otherwise (rc, output length, SHA-256).
  libraries: the liblz4 / libzstd versions the streams were re-made with.

It also checks that _oracle.lib_decompress, which the tests use in place of the reference's decoder, accepts the
streams that decoder accepts with one thread and with four (restoring the same bytes), and refuses the others.

Needs oracle/_ref, i.e. a build() where the original project's sources are at hand (oracle/Makefile REF=...).
Run from the repository root:  python tests/golden/make_reference_digests.py"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, os.path.dirname(TESTS)); sys.path.insert(0, TESTS)
import _oracle as o
import zstdmt_b200 as z

LZ4, ZSTD = o.CODEC_LZ4, o.CODEC_ZSTD
KINDS = [z.GEN_MIX, z.GEN_TEXT, z.GEN_RANDOM, z.GEN_ZEROS]
MIB = 1 << 20


def stream_cases():
    """(codec, level, compress chunk, source) for every reference_stream() call of the suite and of smoke()."""
    yield LZ4, 1, MIB, np.zeros(MIB, np.uint8)                                        # test_oracle: Appendix A zeros
    for codec, level in [(LZ4, 1), (LZ4, 3), (ZSTD, 1), (ZSTD, 3), (ZSTD, 9)]:         # test_oracle_decodes_reference_streams
        for kind in KINDS:
            n = (5 << 20) + 12345 if kind == z.GEN_MIX else MIB + 77
            yield codec, level, MIB, z.gen_stream(kind, n, MIB)
    for level in (1, 3, 19):                                                          # test_cabi: host block scan
        for kind in KINDS:
            yield ZSTD, level, 1 << 19, z.gen_stream(kind, MIB + 12345, MIB)
    for level in (1, 3, 9):                                                           # test_gpu_lz4: decode bit-exact
        for kind in KINDS:
            yield LZ4, level, MIB, z.gen_stream(kind, (10 << 20) + 999, MIB)
    for n, chunk, level in [(0, MIB, 1), (1, MIB, 1), ((6 << 20) + 3, MIB, 1), ((70 << 20) + 1, MIB, 3), (9 << 20, 4 << 20, 1)]:
        yield LZ4, level, chunk, z.gen_stream(z.GEN_MIX, n, chunk)                    # test_gpu_lz4: LZ4MT_decompressDCtx
    for chunk in (65536, 100000, MIB, 4 << 20):                                       # test_gpu_lz4_decode: callbacks
        yield LZ4, 1, chunk, z.gen_stream(z.GEN_MIX, (21 << 20) + 12345, chunk)
    for level in (1, 3, 9, 19):                                                       # test_gpu_zstd: decode bit-exact
        for kind in KINDS:
            yield ZSTD, level, MIB, z.gen_stream(kind, (6 << 20) + 999, MIB)
    big = z.gen_stream(z.GEN_MIX, (300 << 20) + 7, MIB)                               # test_gpu_multigpu
    yield LZ4, 1, MIB, big
    yield ZSTD, 3, MIB, big
    yield LZ4, 1, MIB, z.gen_stream(z.GEN_MIX, (2 << 20) + (1 << 19) + 123, MIB)     # smoke()


def decoded_cases():
    """(codec, stream) for every reference_decoded() call of the suite."""
    import test_gpu_plain_streams as t
    n, chunk = (3 << 20) + 77, MIB
    yield ZSTD, t.zstdmt_style_stream(z.gen_stream(z.GEN_MIX, n, chunk), chunk)


def lz4_frame_without_content_size(data):
    p = o.LZ4FPrefs(compressionLevel=1, blockMode=0, contentSize=0, contentChecksumFlag=1)
    L = o.lz4_lib()
    cap = L.LZ4F_compressFrameBound(data.size, o.ctypes.byref(p))
    out = np.empty(cap, np.uint8)
    n = L.LZ4F_compressFrame(out.ctypes.data, cap, data.ctypes.data, data.size, o.ctypes.byref(p))
    assert not L.LZ4F_isError(n)
    return out[:n]


def wrap(payloads):
    return np.concatenate([np.concatenate([np.array([o.SKIPPABLE_MAGIC, 4, p.size], "<u4").view(np.uint8), p]) for p in payloads])


def decoder_cases():
    """(codec, stream, output room) on which lib_decompress must agree with the reference's decoder."""
    for n in (0, 1, 11, 12, 13, 39, 40, 65535, 65536, 65537, MIB - 1, MIB + 1, (3 << 20) + 5):
        src = z.gen_stream(z.GEN_MIX, n, MIB, first=1)
        yield LZ4, o.orc_encode_lz4(src), n                                           # the GPU encoder's CPU twin
        yield LZ4, o.lib_compress(LZ4, src, 1, MIB), n
        yield ZSTD, o.lib_compress(ZSTD, src, 3, MIB), n
    src = z.gen_stream(z.GEN_TEXT, (2 << 20) + 99, MIB)
    good = o.lib_compress(LZ4, src, 1, 1 << 19)
    yield LZ4, good, src.size - 2                                                     # output room one byte short
    yield LZ4, wrap([lz4_frame_without_content_size(src[a:a + (1 << 19)]) for a in range(0, src.size, 1 << 19)]), src.size
    yield LZ4, wrap([lz4_frame_without_content_size(src[:30])]), 30                   # tiny first frame, no content size
    yield LZ4, wrap([lz4_frame_without_content_size(src[:30]), lz4_frame_without_content_size(src[30:5000])]), 5000
    bad = good.copy(); bad[-1] ^= 1                                                   # content checksum
    yield LZ4, bad, src.size
    f = o.lib_compress(LZ4, src[:100000], 1, MIB)[12:]
    yield LZ4, wrap([f[:-9]]), 100000                                                 # frame cut short
    yield LZ4, wrap([np.concatenate([f, np.arange(5, dtype=np.uint8)])]), 100000      # bytes after the frame's end
    zf = o.lib_compress(ZSTD, src[:100000], 3, MIB)[12:]
    yield ZSTD, wrap([np.concatenate([zf, zf])]), 200000                              # two zstd frames in one payload
    yield ZSTD, wrap([np.concatenate([zf, np.arange(5, dtype=np.uint8)])]), 100000    # bytes after the frame's end


def check_decoder_agreement():
    for codec, stream, room in decoder_cases():
        rc1, back1, _ = o.ref_decompress(codec, stream, room, threads=1)
        rc4, back4, _ = o.ref_decompress(codec, stream, room, threads=4)
        ref_ok = rc1 == 0 and rc4 == 0 and np.array_equal(back1, back4)
        if codec == LZ4:                                # one decode path (pt_decompress) on every thread count
            assert (rc1 == 0) == (rc4 == 0), (stream.size, room, rc1, rc4)
        lrc, lback, _ = o.lib_decompress(codec, stream, room)
        assert ref_ok == (lrc == 0), (codec, stream.size, room, rc1, rc4, lrc)
        assert not ref_ok or np.array_equal(back1, lback), (codec, stream.size, room)


def main():
    assert o.have_ref(), "oracle/_ref not built: build() with the original project's sources at hand"
    T = min(os.cpu_count() or 1, 16)
    check_decoder_agreement()
    out = {"generator": "tests/golden/make_reference_digests.py", "libraries": o.library_versions(), "streams": {}, "decoded": {}}
    for codec, level, chunk, src in stream_cases():
        rc, framed, st = o.ref_compress(codec, src, threads=T, level=level, chunk=chunk)
        assert rc == 0
        assert np.array_equal(framed, o.lib_compress(codec, src, level, chunk)), "lib_compress no longer frames like the reference"
        rc, back, dst = o.ref_decompress(codec, framed, src.size, threads=T)
        assert rc == 0 and np.array_equal(back, src)
        out["streams"][o.stream_key(codec, level, chunk, src)] = {
            "n": int(src.size), "framed_bytes": int(framed.size), "sha256": o.sha256(framed),
            "compress_stats": [int(x) for x in st[:4]], "decompress_stats": [int(x) for x in dst[:4]]}
    for codec, stream in decoded_cases():
        rc, back, _ = o.ref_decompress(codec, stream, 1 << 30, threads=T)
        out["decoded"]["%s:%s" % ("lz4" if codec == LZ4 else "zstd", o.sha256(stream))] = {
            "rc": int(rc), "out_bytes": int(back.size), "sha256": o.sha256(back)}
    with open(os.path.join(HERE, "reference_streams.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote %d stream and %d decode digests" % (len(out["streams"]), len(out["decoded"])))


if __name__ == "__main__":
    main()
