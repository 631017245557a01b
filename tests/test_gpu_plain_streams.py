"""Plain (unframed) .lz4 / .zst streams — what the reference routes to st_decompress (lz4-mt_decompress.c:391-483,
zstd-mt_decompress.c:552-687; SURVEY §8(f) row 2).  Inputs are produced by the codec libraries the reference links
(liblz4 1.9.4 / libzstd of the image, called directly through ctypes), decoded through LZ4MT_/ZSTDCB_decompressDCtx."""
import ctypes

import numpy as np
import pytest

import _oracle as o
import zstdmt_b200 as z
from _oracle import LZ4FPrefs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def lz4f(data, **kw):
    try:
        L = ctypes.CDLL("liblz4.so.1")
    except OSError:
        pytest.skip("liblz4.so.1 not present")
    L.LZ4F_compressFrameBound.restype = ctypes.c_size_t; L.LZ4F_compressFrameBound.argtypes = [ctypes.c_size_t, ctypes.c_void_p]
    L.LZ4F_compressFrame.restype = ctypes.c_size_t
    L.LZ4F_compressFrame.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    p = LZ4FPrefs()
    for k, v in kw.items():
        setattr(p, k, v)
    cap = L.LZ4F_compressFrameBound(data.size, ctypes.byref(p))
    out = np.empty(cap, np.uint8)
    n = L.LZ4F_compressFrame(out.ctypes.data, cap, data.ctypes.data, data.size, ctypes.byref(p))
    assert n < (1 << 62)
    return out[:n].copy()


def zstd1(data, level):
    try:
        L = ctypes.CDLL("libzstd.so.1")
    except OSError:
        pytest.skip("libzstd.so.1 not present")
    L.ZSTD_compressBound.restype = ctypes.c_size_t; L.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    L.ZSTD_compress.restype = ctypes.c_size_t; L.ZSTD_compress.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    cap = L.ZSTD_compressBound(data.size)
    out = np.empty(cap, np.uint8)
    n = L.ZSTD_compress(out.ctypes.data, cap, data.ctypes.data, data.size, level)
    assert n < (1 << 62)
    return out[:n].copy()


@pytest.mark.parametrize("prefs", [dict(), dict(blockMode=1, contentSize=1, contentChecksumFlag=1), dict(blockSizeID=7, blockMode=1),
                                   dict(blockSizeID=5, contentChecksumFlag=1, blockChecksumFlag=1), dict(compressionLevel=9, blockSizeID=6)])
def test_plain_lz4_frame(gpu, prefs):
    src = z.gen_stream(z.GEN_MIX, (5 << 20) + 321, 1 << 20)
    if prefs.get("contentSize"):
        prefs = dict(prefs, contentSize=int(src.size))
    frame = lz4f(src, **prefs)
    rc, back, st = z.decompress_mem(z.CODEC_LZ4, frame, src.size + 16, threads=4)
    assert rc == 0, z.lib().LZ4MT_getErrorString(rc)
    assert back.size == src.size and np.array_equal(back, src)
    assert st["insize"] == frame.size and st["outsize"] == src.size


def test_plain_lz4_concatenated_frames_and_skippable(gpu):
    a = z.gen_stream(z.GEN_TEXT, 700000, 1 << 20)
    b = z.gen_stream(z.GEN_MIX, 300000, 1 << 20, first=5)
    skip = np.frombuffer(bytes.fromhex("512a4d18") + (5).to_bytes(4, "little") + b"hello", np.uint8)     # user skippable frame
    stream = np.concatenate([lz4f(a), skip, lz4f(b, blockMode=1, contentChecksumFlag=1), lz4f(np.zeros(0, np.uint8))])
    rc, back, st = z.decompress_mem(z.CODEC_LZ4, stream, a.size + b.size + 16, threads=2)
    assert rc == 0 and np.array_equal(back, np.concatenate([a, b]))
    bad = stream.copy(); bad[-1] ^= 0xFF; bad = np.concatenate([stream, np.frombuffer(b"\x01\x02\x03\x04\x05", np.uint8)])
    rc, _, _ = z.decompress_mem(z.CODEC_LZ4, bad, a.size + b.size + 16)
    assert z.lib().LZ4MT_isError(rc)                                        # trailing garbage is not silently accepted


@pytest.mark.parametrize("level", [1, 3, 12, 19])
def test_plain_zstd_frames(gpu, level):
    a = z.gen_stream(z.GEN_MIX, (6 << 20) + 17, 1 << 20)           # one frame, window > 1 MiB, 128 KiB blocks
    b = z.gen_stream(z.GEN_TEXT, 1 << 20, 1 << 20)
    stream = np.concatenate([zstd1(a, level), zstd1(b, level), zstd1(np.zeros(0, np.uint8), level)])
    rc, back, st = z.decompress_mem(z.CODEC_ZSTD, stream, a.size + b.size + 16, threads=4)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    assert np.array_equal(back, np.concatenate([a, b]))
    assert st["outsize"] == a.size + b.size


def test_plain_zstd_small_and_empty(gpu):
    for n in (0, 1, 5, 200):
        src = z.gen_stream(z.GEN_TEXT, n, 1 << 20)
        fr = zstd1(src, 3)
        rc, back, st = z.decompress_mem(z.CODEC_ZSTD, fr, n + 16)
        assert rc == 0 and np.array_equal(back, src), n


# ---------------------------------------------------------------- stock .zst frames: content checksum, no content size
def zstd_adv(data, level=3, checksum=1, content_size=1, pieces=None):
    """ZSTD_compressStream2 with ZSTD_c_checksumFlag / ZSTD_c_contentSizeFlag; `pieces`: stream the input in pieces without
    a pledged size (the frame header then carries no content size, as for `zstd < pipe`)."""
    try:
        L = ctypes.CDLL("libzstd.so.1")
    except OSError:
        pytest.skip("libzstd.so.1 not present")

    class Buf(ctypes.Structure):
        _fields_ = [("p", ctypes.c_void_p), ("size", ctypes.c_size_t), ("pos", ctypes.c_size_t)]

    L.ZSTD_createCCtx.restype = ctypes.c_void_p
    L.ZSTD_CCtx_setParameter.restype = ctypes.c_size_t; L.ZSTD_CCtx_setParameter.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    L.ZSTD_compressStream2.restype = ctypes.c_size_t
    L.ZSTD_compressStream2.argtypes = [ctypes.c_void_p, ctypes.POINTER(Buf), ctypes.POINTER(Buf), ctypes.c_int]
    L.ZSTD_freeCCtx.argtypes = [ctypes.c_void_p]
    L.ZSTD_compressBound.restype = ctypes.c_size_t; L.ZSTD_compressBound.argtypes = [ctypes.c_size_t]
    cctx = L.ZSTD_createCCtx()
    assert L.ZSTD_CCtx_setParameter(cctx, 100, level) < (1 << 62)           # ZSTD_c_compressionLevel
    assert L.ZSTD_CCtx_setParameter(cctx, 200, content_size) < (1 << 62)    # ZSTD_c_contentSizeFlag
    assert L.ZSTD_CCtx_setParameter(cctx, 201, checksum) < (1 << 62)        # ZSTD_c_checksumFlag
    cap = L.ZSTD_compressBound(data.size) + 1024
    out = np.empty(cap, np.uint8)
    ob = Buf(out.ctypes.data, cap, 0)
    cuts = [data.size] if not pieces else pieces
    at = 0
    for i, n in enumerate(cuts):
        ib = Buf(data.ctypes.data + at, n, 0)
        last = i == len(cuts) - 1
        while True:
            r = L.ZSTD_compressStream2(cctx, ctypes.byref(ob), ctypes.byref(ib), 2 if last else 0)     # ZSTD_e_end / ZSTD_e_continue
            assert r < (1 << 62)
            if (last and r == 0) or (not last and ib.pos == ib.size):
                break
        at += n
    assert at == data.size
    L.ZSTD_freeCCtx(cctx)
    return out[: ob.pos].copy()


@pytest.mark.parametrize("level", [1, 3, 9])
def test_plain_zstd_with_content_checksum(gpu, level):
    """What the stock `zstd` CLI writes by default: frame content checksum = low 32 bits of XXH64 (verified on the GPU)."""
    a = z.gen_stream(z.GEN_MIX, (3 << 20) + 11, 1 << 20)
    b = z.gen_stream(z.GEN_TEXT, 70000, 1 << 20)
    fa, fb, fe = zstd_adv(a, level, checksum=1), zstd_adv(b, level, checksum=1), zstd_adv(np.zeros(0, np.uint8), level, checksum=1)
    assert fa[4] & 4 and fb[4] & 4                                      # Content_Checksum_flag set in the frame header descriptor
    stream = np.concatenate([fa, fb, fe])
    rc, back, st = z.decompress_mem(z.CODEC_ZSTD, stream, a.size + b.size + 16, threads=4)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    assert np.array_equal(back, np.concatenate([a, b]))
    bad = stream.copy(); bad[fa.size - 1] ^= 0x40                       # frame a's stored checksum
    rc, _, _ = z.decompress_mem(z.CODEC_ZSTD, bad, a.size + b.size + 16)
    assert z.lib().ZSTDCB_isError(rc) and b"contentChecksum" in z.lib().ZSTDCB_getErrorString(rc)
    bad = stream.copy(); bad[fa.size // 2] ^= 0x01                       # payload damage: either the block decode or the checksum must notice
    rc, _, _ = z.decompress_mem(z.CODEC_ZSTD, bad, a.size + b.size + 16)
    assert z.lib().ZSTDCB_isError(rc)


@pytest.mark.parametrize("checksum", [0, 1])
def test_plain_zstd_streamed_frames_without_content_size(gpu, checksum):
    """Frames written by a streaming producer carry no Frame_Content_Size (zstd-mt_decompress.c:463-522 grows its
    buffer by doubling there); here the output room is bounded from the block headers."""
    a = z.gen_stream(z.GEN_MIX, (2 << 20) + 12345, 1 << 20, first=2)
    fr = zstd_adv(a, 3, checksum=checksum, pieces=[100000, 1 << 20, a.size - 100000 - (1 << 20)])
    assert (fr[4] >> 6) == 0 and not (fr[4] & 0x20)                      # no FCS field, not single-segment
    b = z.gen_stream(z.GEN_TEXT, 300000, 1 << 20)
    stream = np.concatenate([fr, zstd1(b, 3)])
    rc, back, st = z.decompress_mem(z.CODEC_ZSTD, stream, a.size + b.size + 16, threads=4)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    assert np.array_equal(back, np.concatenate([a, b]))
    # the same frames behind the 12-byte MT headers (pzstd-style framed stream)
    def wrap(f): return np.concatenate([np.frombuffer((0x184D2A50).to_bytes(4, "little") + (4).to_bytes(4, "little") + int(f.size).to_bytes(4, "little"), np.uint8), f])
    framed = np.concatenate([wrap(fr), wrap(zstd_adv(b, 3, checksum=1))])
    rc, back, st = z.decompress_mem(z.CODEC_ZSTD, framed, a.size + b.size + 16, threads=4)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    assert np.array_equal(back, np.concatenate([a, b]))


def zstdmt_style_stream(src, chunk):
    """A 9-byte empty zstd frame, then [12-byte skippable header][zstd frame of one chunk]*."""
    parts = [np.frombuffer(bytes.fromhex("28b52ffd2000010000"), np.uint8)]
    for a in range(0, src.size, chunk):
        f = zstd1(src[a:a + chunk], 3)
        parts += [np.frombuffer((0x184D2A50).to_bytes(4, "little") + (4).to_bytes(4, "little") + int(f.size).to_bytes(4, "little"), np.uint8), f]
    return np.concatenate(parts)


def test_zstdmt_style_stream(gpu):
    """zstdmt-style framing: a 9-byte empty zstd frame, then [12-byte skippable header][zstd frame]* — the second branch of
    the stream sniffing (zstd-mt_decompress.c:745-749, first-frame fix-up :231-263)."""
    n, chunk = (3 << 20) + 77, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    stream = zstdmt_style_stream(src, chunk)
    rc, back, st = z.decompress_mem(z.CODEC_ZSTD, stream, n + 16, threads=4)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    assert np.array_equal(back, src) and st["frames"] == -(-n // chunk)
    ref = o.reference_decoded(o.CODEC_ZSTD, stream)                     # the reference accepted the very same bytes
    assert ref["rc"] == 0 and ref["out_bytes"] == n and ref["sha256"] == o.sha256(src)


@pytest.mark.parametrize("codec", ["lz4", "zstd"])
def test_plain_streams_decode_in_bounded_batches(gpu, codec, monkeypatch):
    """Many frames, batches of 1 MiB of input (ZSTDMT_B200_PLAIN_MB): the host drops decoded input before it reads on;
    one frame larger than a batch still decodes."""
    monkeypatch.setenv("ZSTDMT_B200_PLAIN_MB", "1")
    rng = np.random.default_rng(11)
    sizes = [int(x) for x in rng.integers(1, 900000, 30)] + [6 << 20] + [int(x) for x in rng.integers(1, 200000, 10)]
    srcs = [z.gen_stream(z.GEN_MIX if i % 2 else z.GEN_TEXT, s, 1 << 20, first=i) for i, s in enumerate(sizes)]
    if codec == "lz4":
        frames = [lz4f(s, blockMode=i & 1, contentChecksumFlag=1, contentSize=int(s.size) if i % 3 else 0) for i, s in enumerate(srcs)]
        cid = z.CODEC_LZ4
    else:
        frames = [zstd_adv(s, 3, checksum=i & 1) if i % 3 else zstd_adv(s, 3, checksum=1, pieces=[s.size // 2, s.size - s.size // 2]) for i, s in enumerate(srcs)]
        cid = z.CODEC_ZSTD
    stream = np.concatenate(frames)
    total = sum(sizes)
    rc, back, st = z.decompress_mem(cid, stream, total + 16, threads=4, inputsize=1 << 16)
    assert rc == 0
    assert back.size == total and np.array_equal(back, np.concatenate(srcs))
    assert st["insize"] == stream.size and st["outsize"] == total
    rc, _, _ = z.decompress_mem(cid, stream[:-3], total + 16, inputsize=1 << 16)     # truncated last frame
    assert rc != 0
