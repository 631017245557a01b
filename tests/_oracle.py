"""ctypes bindings to the TEST-ONLY oracle: oracle/liboracle.so (CPU restatement),
oracle/_ref/libzstdmt_ref.so (the unmodified reference wrapper + liblz4/libzstd, only where the
original project's sources were at hand), and the codec libraries the reference links (liblz4.so.1,
libzstd.so.1) called directly.

The suite does not need oracle/_ref: streams the reference writes are re-made here frame by frame
with the same library calls and checked against digests of the reference's own output
(tests/golden/reference_streams.json, written by tests/golden/make_reference_digests.py)."""
import concurrent.futures
import ctypes
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "reference_streams.json")
c_sz = ctypes.c_size_t
c_vp = ctypes.c_void_p

CODEC_LZ4, CODEC_ZSTD = 1, 2
SKIPPABLE_MAGIC = 0x184D2A50
_orc = None
_ref = None
_lz4 = None
_zstd = None
_golden_data = None


def orc():
    global _orc
    if _orc is None:
        L = ctypes.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
        L.orc_xxh32.restype = ctypes.c_uint32; L.orc_xxh32.argtypes = [c_vp, c_sz, ctypes.c_uint32]
        L.orc_mt_decode.restype = ctypes.c_int; L.orc_mt_decode.argtypes = [ctypes.c_int, c_vp, c_sz, c_vp, c_sz, ctypes.POINTER(c_sz)]
        L.orc_mt_encode_lz4_b200.restype = c_sz; L.orc_mt_encode_lz4_b200.argtypes = [c_vp, c_sz, c_sz, c_vp, c_sz]
        L.orc_lz4f_decode.restype = ctypes.c_int; L.orc_lz4f_decode.argtypes = [c_vp, c_sz, c_vp, c_sz, ctypes.POINTER(c_sz), ctypes.POINTER(c_sz)]
        L.orc_zstd_decode.restype = ctypes.c_int; L.orc_zstd_decode.argtypes = [c_vp, c_sz, c_vp, c_sz, ctypes.POINTER(c_sz), ctypes.POINTER(c_sz)]
        L.orc_lz4_block_compress_b200.restype = c_sz; L.orc_lz4_block_compress_b200.argtypes = [c_vp, c_sz, c_vp, c_sz]
        L.orc_lz4_block_bound.restype = c_sz; L.orc_lz4_block_bound.argtypes = [c_sz]
        L.orc_lz4_block_decode.restype = ctypes.c_long; L.orc_lz4_block_decode.argtypes = [c_vp, c_sz, c_vp, c_sz, c_sz]
        L.orc_mt_scan.restype = ctypes.c_long; L.orc_mt_scan.argtypes = [c_vp, c_sz, c_vp, c_vp, c_sz]
        _orc = L
    return _orc


def have_ref():
    return os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libzstdmt_ref.so"))


def ref():
    global _ref
    if _ref is None:
        L = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libzstdmt_ref.so"))
        for f in ("ref_lz4_compress_mem", "ref_zstd_compress_mem"):
            getattr(L, f).restype = c_sz
            getattr(L, f).argtypes = [ctypes.c_int] * 3 + [c_vp, c_sz, c_vp, c_sz, ctypes.POINTER(c_sz)]
        for f in ("ref_lz4_decompress_mem", "ref_zstd_decompress_mem"):
            getattr(L, f).restype = c_sz
            getattr(L, f).argtypes = [ctypes.c_int] * 2 + [c_vp, c_sz, c_vp, c_sz, ctypes.POINTER(c_sz)]
        _ref = L
    return _ref


def _arr(data):
    return np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data, dtype=np.uint8)


def ref_compress(codec, data, threads=1, level=1, chunk=1 << 20):
    """The real reference: {LZ4MT,ZSTDCB}_compressCCtx -> liblz4 / libzstd."""
    data = _arr(data)
    cap = data.size + data.size // 64 + 65536 + 64 * (data.size // chunk + 2)
    out = np.empty(cap, np.uint8); st = (c_sz * 5)()
    fn = ref().ref_lz4_compress_mem if codec == CODEC_LZ4 else ref().ref_zstd_compress_mem
    rc = fn(threads, level, chunk, data.ctypes.data, data.size, out.ctypes.data, cap, st)
    return rc, out[: st[0]].copy(), list(st)


def ref_decompress(codec, data, out_cap, threads=1):
    data = _arr(data)
    out = np.empty(out_cap + 1, np.uint8); st = (c_sz * 5)()
    fn = ref().ref_lz4_decompress_mem if codec == CODEC_LZ4 else ref().ref_zstd_decompress_mem
    rc = fn(threads, 0, data.ctypes.data, data.size, out.ctypes.data, out_cap + 1, st)
    return rc, out[: st[0]].copy(), list(st)


def orc_decode(codec, data, out_cap):
    data = _arr(data)
    out = np.empty(out_cap + 1, np.uint8); got = c_sz(0)
    rc = orc().orc_mt_decode(codec, data.ctypes.data, data.size, out.ctypes.data, out_cap + 1, ctypes.byref(got))
    return rc, out[: got.value]


def orc_encode_lz4(data, chunk=1 << 20):
    data = _arr(data)
    cap = data.size + data.size // 100 + 4096 + 64 * (data.size // chunk + 2)
    out = np.empty(cap, np.uint8)
    n = orc().orc_mt_encode_lz4_b200(data.ctypes.data, data.size, chunk, out.ctypes.data, cap)
    return out[:n].copy()


def xxh32(data, seed=0):
    data = _arr(data)
    return orc().orc_xxh32(data.ctypes.data, data.size, seed)


# ---- the codec libraries the reference links, called directly ---------------------------------
class LZ4FPrefs(ctypes.Structure):
    _fields_ = [("blockSizeID", ctypes.c_int), ("blockMode", ctypes.c_int), ("contentChecksumFlag", ctypes.c_int), ("frameType", ctypes.c_int),
                ("contentSize", ctypes.c_ulonglong), ("dictID", ctypes.c_uint), ("blockChecksumFlag", ctypes.c_int),
                ("compressionLevel", ctypes.c_int), ("autoFlush", ctypes.c_uint), ("favorDecSpeed", ctypes.c_uint), ("reserved", ctypes.c_uint * 3)]


def lz4_lib():
    global _lz4
    if _lz4 is None:
        L = ctypes.CDLL("liblz4.so.1")
        for f in ("LZ4F_compressFrameBound", "LZ4F_compressFrame", "LZ4F_createDecompressionContext", "LZ4F_decompress",
                  "LZ4F_freeDecompressionContext"):
            getattr(L, f).restype = c_sz
        L.LZ4F_isError.restype = ctypes.c_uint; L.LZ4F_isError.argtypes = [c_sz]
        L.LZ4_versionNumber.restype = ctypes.c_int
        L.LZ4F_compressFrameBound.argtypes = [c_sz, c_vp]
        L.LZ4F_compressFrame.argtypes = [c_vp, c_sz, c_vp, c_sz, c_vp]
        L.LZ4F_createDecompressionContext.argtypes = [ctypes.POINTER(c_vp), ctypes.c_uint]
        L.LZ4F_decompress.argtypes = [c_vp, c_vp, ctypes.POINTER(c_sz), c_vp, ctypes.POINTER(c_sz), c_vp]
        L.LZ4F_freeDecompressionContext.argtypes = [c_vp]
        _lz4 = L
    return _lz4


def zstd_lib():
    global _zstd
    if _zstd is None:
        L = ctypes.CDLL("libzstd.so.1")
        for f in ("ZSTD_compressBound", "ZSTD_compress", "ZSTD_decompress", "ZSTD_findFrameCompressedSize"):
            getattr(L, f).restype = c_sz
        L.ZSTD_findFrameCompressedSize.argtypes = [c_vp, c_sz]
        L.ZSTD_versionNumber.restype = ctypes.c_uint
        L.ZSTD_isError.restype = ctypes.c_uint; L.ZSTD_isError.argtypes = [c_sz]
        L.ZSTD_compressBound.argtypes = [c_sz]
        L.ZSTD_compress.argtypes = [c_vp, c_sz, c_vp, c_sz, ctypes.c_int]
        L.ZSTD_decompress.argtypes = [c_vp, c_sz, c_vp, c_sz]
        _zstd = L
    return _zstd


def _frame_one(codec, data, level):
    """One chunk as the reference frames it: LZ4F_compressFrame (linked blocks, content size, content checksum) or
    ZSTD_compress at `level`, behind the 12-byte skippable header that carries the frame's size."""
    if codec == CODEC_LZ4:
        L = lz4_lib()
        p = LZ4FPrefs(compressionLevel=level, blockMode=0, contentSize=1, contentChecksumFlag=1)
        cap = L.LZ4F_compressFrameBound(data.size, ctypes.byref(p))
        out = np.empty(12 + cap, np.uint8)
        n = L.LZ4F_compressFrame(out[12:].ctypes.data, cap, data.ctypes.data, data.size, ctypes.byref(p))
        assert not L.LZ4F_isError(n)
    else:
        L = zstd_lib()
        cap = L.ZSTD_compressBound(data.size)
        out = np.empty(12 + cap, np.uint8)
        n = L.ZSTD_compress(out[12:].ctypes.data, cap, data.ctypes.data, data.size, level)
        assert not L.ZSTD_isError(n)
    out[:12] = np.array([SKIPPABLE_MAGIC, 4, n], dtype="<u4").view(np.uint8)
    return out[: 12 + n]


def lib_compress(codec, data, level, chunk):
    """The framed stream {LZ4MT,ZSTDCB}_compressCCtx writes: one frame per `chunk` bytes (one empty frame for empty
    input), in order.  Chunks are independent, so they are compressed on a thread pool (ctypes drops the GIL)."""
    data = _arr(data)
    cuts = list(range(0, data.size, chunk)) or [0]
    with concurrent.futures.ThreadPoolExecutor(min(32, os.cpu_count() or 1)) as ex:
        frames = list(ex.map(lambda a: _frame_one(codec, data[a: a + chunk], level), cuts))
    return np.concatenate(frames)


def lib_decompress(codec, framed, out_cap):
    """Decode a framed stream as the reference's decoder does, with the library calls it makes, frame by frame behind
    the 12-byte skippable headers; a stream is accepted only if the reference accepts it with one thread and with
    several, and restores the same bytes:
      LZ4  (lz4-mt_decompress.c pt_decompress): the output room is the LE64 content-size field at payload offset 6
           (64 KiB for a first frame under 40 bytes); ONE LZ4F_decompress call into that room must end the frame.
           A frame without a content-size field is refused: the 8 bytes there are then header checksum, block size
           and data, and the room they name is not allocatable or too small.  Bytes after the frame's end are
           ignored, as there.
      zstd: the payload must hold exactly one zstd frame, decoded to its end.  The reference's multi-threaded path
           (zstd-mt_decompress.c pt_decompress) decodes the first frame of a payload and ignores what follows; with
           one thread it streams the whole input through libzstd and decodes what follows as further frames.  So a
           payload with bytes after its first frame is refused here, as the two paths would not agree on it, and so
           is a payload whose first frame is cut short.
    Like ref_decompress, it has out_cap + 1 bytes of output room; more output fails, as the reference's fn_write
    does.  Returns (rc, output, frames); rc != 0 when the stream is refused."""
    framed = _arr(framed)
    out = np.empty(out_cap + 1, np.uint8)
    pos, at, frames = 0, 0, 0
    while at < framed.size:
        if framed.size - at < 12:
            return -1, out[:pos], frames
        magic, four, size = (int(x) for x in framed[at: at + 12].view("<u4"))
        if magic != SKIPPABLE_MAGIC or four != 4 or at + 12 + size > framed.size:
            return -2, out[:pos], frames
        payload = framed[at + 12: at + 12 + size]
        left = out.size - pos
        if codec == CODEC_LZ4:
            L = lz4_lib()
            if frames == 0 and size < 40:
                room = min(1 << 16, left)
            elif size >= 14 and int(payload[6:14].view("<u8")[0]) <= left:
                room = int(payload[6:14].view("<u8")[0])
            else:
                return -5, out[:pos], frames
            ctx = c_vp()
            assert not L.LZ4F_isError(L.LZ4F_createDecompressionContext(ctypes.byref(ctx), 100))
            dst = c_sz(room); srcn = c_sz(size)
            hint = L.LZ4F_decompress(ctx, out[pos:].ctypes.data, ctypes.byref(dst), payload.ctypes.data, ctypes.byref(srcn), None)
            L.LZ4F_freeDecompressionContext(ctx)
            if L.LZ4F_isError(hint) or hint != 0:
                return -3, out[:pos], frames
            pos += dst.value
        else:
            L = zstd_lib()
            first = L.ZSTD_findFrameCompressedSize(payload.ctypes.data, size)
            if L.ZSTD_isError(first) or first != size:
                return -4, out[:pos], frames
            r = L.ZSTD_decompress(out[pos:].ctypes.data, left, payload.ctypes.data, size)
            if L.ZSTD_isError(r):
                return -3, out[:pos], frames
            pos += r
        at += 12 + size
        frames += 1
    return 0, out[:pos], frames


# ---- what the reference computed, kept as digests --------------------------------------------
def sha256(data):
    return hashlib.sha256(_arr(data).data).hexdigest()


def _golden():
    global _golden_data
    if _golden_data is None:
        with open(GOLDEN_REF) as f:
            _golden_data = json.load(f)
    return _golden_data


def library_versions():
    """The liblz4 / libzstd versions lib_compress frames with, e.g. {"liblz4": "1.9.4", "libzstd": "1.5.5"}."""
    def dotted(v):
        return "%d.%d.%d" % (v // 10000, v // 100 % 100, v % 100)
    return {"liblz4": dotted(lz4_lib().LZ4_versionNumber()), "libzstd": dotted(zstd_lib().ZSTD_versionNumber())}


def stream_key(codec, level, chunk, src):
    return "%s:l%d:c%d:%s" % ("lz4" if codec == CODEC_LZ4 else "zstd", level, chunk, sha256(src))


def reference_stream(codec, src, level, chunk):
    """The stream {LZ4MT,ZSTDCB}_compressCCtx of the original project writes for `src`, re-made with lib_compress and
    checked byte for byte (length + SHA-256) against the reference's own output.  Returns (framed, record): the
    record holds the reference's counters, compress_stats = [out bytes, frames, insize, outsize] and
    decompress_stats = [out bytes, frames, insize, outsize] of its decoder on that stream."""
    src = _arr(src)
    rec = _golden()["streams"].get(stream_key(codec, level, chunk, src))
    assert rec is not None, "no digest of the reference's stream for this input: add the case to tests/golden/make_reference_digests.py"
    framed = lib_compress(codec, src, level, chunk)
    assert framed.size == rec["framed_bytes"] and sha256(framed) == rec["sha256"], \
        "stream differs from the reference's: digests were made with %s, this machine has %s" % (_golden()["libraries"], library_versions())
    return framed, rec


def reference_decoded(codec, stream):
    """What the reference's decoder made of `stream` when the golden data was written: {"rc", "out_bytes", "sha256"}."""
    key = "%s:%s" % ("lz4" if codec == CODEC_LZ4 else "zstd", sha256(stream))
    rec = _golden()["decoded"].get(key)
    assert rec is not None, "the reference never decoded this stream: add the case to tests/golden/make_reference_digests.py"
    return rec
