"""GPU parity tests of the block-parallel LZ4F decoder (lz4_decode.cuh): frames with linked blocks (what the reference
produces, lib/lz4-mt_compress.c:141-146), every blockMaxSize, streaming frames with partial blocks (sequential fallback),
length-field corner cases.  Inputs come from the real liblz4 (through ctypes); the bar is bit-exact output."""
import ctypes

import numpy as np
import pytest

import _oracle as o
import zstdmt_b200 as z
from _data import long_runs_stream
from test_gpu_plain_streams import LZ4FPrefs, lz4f

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def wrap(frames):
    """12-byte skippable header in front of every LZ4F frame (lz4-mt_compress.c:293-298)."""
    parts = []
    for f in frames:
        parts.append(np.frombuffer((0x184D2A50).to_bytes(4, "little") + (4).to_bytes(4, "little") + int(f.size).to_bytes(4, "little"), np.uint8))
        parts.append(f)
    return np.concatenate(parts)


def gpu_decode(torch, framed, out_sizes):
    offs, sizes = z.scan_frames(framed)
    dec = z.Lz4DeviceDecompressor(offs, sizes, out_sizes)
    d = torch.from_numpy(np.ascontiguousarray(framed)).cuda()
    out, status = dec.run(d)
    torch.cuda.synchronize()
    return out[: dec.out_total].cpu().numpy(), status.cpu().numpy(), dec.out_size.cpu().numpy()


@pytest.mark.parametrize("bsid", [4, 5, 6, 7])
@pytest.mark.parametrize("linked", [0, 1])
@pytest.mark.parametrize("kind", [z.GEN_MIX, z.GEN_TEXT])
def test_every_block_size_linked_and_independent(torch, bsid, linked, kind):
    n = (9 << 20) + 4567
    src = z.gen_stream(kind, n, 1 << 20, first=3)
    cuts = [0, 5 << 20, n]                                             # two frames: 5 MiB and the rest
    frames = [lz4f(src[a:b], blockSizeID=bsid, blockMode=0 if linked else 1, contentSize=b - a, contentChecksumFlag=1) for a, b in zip(cuts, cuts[1:])]
    back, status, osz = gpu_decode(torch, wrap(frames), [b - a for a, b in zip(cuts, cuts[1:])])
    assert not status.any(), status
    assert osz.tolist() == [b - a for a, b in zip(cuts, cuts[1:])]
    assert np.array_equal(back, src)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("level", [1, 9])
def test_length_field_corner_cases_linked(torch, seed, level):
    src = long_runs_stream(seed)
    frames = [lz4f(src, blockMode=0, contentSize=int(src.size), contentChecksumFlag=1, compressionLevel=level)]
    back, status, osz = gpu_decode(torch, wrap(frames), [src.size])
    assert not status.any(), status
    assert np.array_equal(back, src)


def lz4f_streaming(data, pieces, flush=True, **kw):
    """LZ4F_compressBegin / Update / (Flush) / End: blocks end wherever the caller flushes -> partial, linked blocks."""
    L = ctypes.CDLL("liblz4.so.1")
    L.LZ4F_createCompressionContext.restype = ctypes.c_size_t
    L.LZ4F_createCompressionContext.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_uint]
    for f in ("LZ4F_compressBegin", "LZ4F_compressUpdate", "LZ4F_flush", "LZ4F_compressEnd", "LZ4F_compressBound", "LZ4F_freeCompressionContext"):
        getattr(L, f).restype = ctypes.c_size_t
    L.LZ4F_compressBegin.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    L.LZ4F_compressUpdate.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    L.LZ4F_flush.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    L.LZ4F_compressEnd.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
    L.LZ4F_compressBound.argtypes = [ctypes.c_size_t, ctypes.c_void_p]
    L.LZ4F_freeCompressionContext.argtypes = [ctypes.c_void_p]
    p = LZ4FPrefs()
    for k, v in kw.items():
        setattr(p, k, v)
    ctx = ctypes.c_void_p()
    assert L.LZ4F_createCompressionContext(ctypes.byref(ctx), 100) == 0
    cap = data.size + data.size // 100 + 65536 * 2 + 64 * (len(pieces) + 2) + 1024
    out = np.empty(cap, np.uint8)
    pos = L.LZ4F_compressBegin(ctx, out.ctypes.data, cap, ctypes.byref(p))
    assert pos < (1 << 62)
    at = 0
    for n in pieces:
        r = L.LZ4F_compressUpdate(ctx, out.ctypes.data + pos, cap - pos, data.ctypes.data + at, n, None)
        assert r < (1 << 62); pos += r; at += n
        if flush:
            r = L.LZ4F_flush(ctx, out.ctypes.data + pos, cap - pos, None)
            assert r < (1 << 62); pos += r
    assert at == data.size
    r = L.LZ4F_compressEnd(ctx, out.ctypes.data + pos, cap - pos, None)
    assert r < (1 << 62); pos += r
    L.LZ4F_freeCompressionContext(ctx)
    return out[:pos].copy()


@pytest.mark.parametrize("linked", [0, 1])
def test_streaming_frames_with_partial_blocks_take_the_sequential_pass(torch, linked):
    n = 700000
    src = z.gen_stream(z.GEN_TEXT, n, 1 << 20, first=7)
    pieces = [1000, 65536, 30000, 65535, 1, 100000, 65537]
    pieces.append(n - sum(pieces))
    fr = lz4f_streaming(src, pieces, blockMode=0 if linked else 1, contentChecksumFlag=1)
    # a second, ordinary frame in the same batch keeps the fast path busy next to the fallback
    src2 = z.gen_stream(z.GEN_MIX, 300000, 1 << 20)
    fr2 = lz4f(src2, blockMode=0, contentSize=int(src2.size), contentChecksumFlag=1)
    back, status, osz = gpu_decode(torch, wrap([fr, fr2]), [n, src2.size])
    assert not status.any(), status
    assert osz.tolist() == [n, src2.size]
    assert np.array_equal(back[:n], src) and np.array_equal(back[n:], src2)
    # the same frame through the callback API as a plain .lz4 stream
    rc, back2, st = z.decompress_mem(z.CODEC_LZ4, fr, n + 16)
    assert rc == 0 and np.array_equal(back2, src)


def test_corrupt_linked_frame_is_reported_not_hung(torch):
    """A damaged block in the middle of a linked frame: the blocks behind it must not wait forever."""
    n = 1 << 20
    src = z.gen_stream(z.GEN_TEXT, n, 1 << 20)
    fr = lz4f(src, blockMode=0, contentSize=n, contentChecksumFlag=1)
    good = wrap([fr, fr])
    bad = good.copy(); bad[12 + fr.size // 2] ^= 0x5A; bad[12 + fr.size // 2 + 1] ^= 0xA5
    back, status, osz = gpu_decode(torch, bad, [n, n])
    assert status[0] != 0 and status[1] == 0
    assert np.array_equal(back[n:], src)


def test_many_small_and_ragged_frames(torch):
    """Frames of every size class in one batch: empty, tiny, one block, just over a block, several blocks."""
    rng = np.random.default_rng(5)
    sizes = [0, 1, 5, 13, 64, 65535, 65536, 65537, 131072, 131073, 200000, 1 << 20, (1 << 20) + 1] + [int(x) for x in rng.integers(1, 300000, 40)]
    srcs = [z.gen_stream(z.GEN_MIX if i % 3 else z.GEN_TEXT, s, 1 << 20, first=i) for i, s in enumerate(sizes)]
    frames = [lz4f(s, blockMode=i & 1, contentSize=int(s.size), contentChecksumFlag=1) for i, s in enumerate(srcs)]
    back, status, osz = gpu_decode(torch, wrap(frames), sizes)
    assert not status.any(), status
    assert osz.tolist() == sizes
    assert np.array_equal(back, np.concatenate(srcs))


@pytest.mark.parametrize("chunk", [65536, 100000, 1 << 20, 4 << 20])
def test_reference_framed_stream_through_callbacks(torch, chunk):
    """BASELINE config 3 in small: a stream framed by the unmodified reference decodes through LZ4MT_decompressDCtx."""
    n = (21 << 20) + 12345
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    framed, _ = o.reference_stream(o.CODEC_LZ4, src, 1, chunk)
    rc, back, st = z.decompress_mem(z.CODEC_LZ4, framed, n + 16, threads=4)
    assert rc == 0, z.lib().LZ4MT_getErrorString(rc)
    assert np.array_equal(back, src)
