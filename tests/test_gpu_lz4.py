"""GPU parity tests for the LZ4 path (run on the B200 box: pytest -m gpu).

Bars (BASELINE.json north_star):
  * decode: bit-exact with the original for reference-produced streams;
  * container bytes: 12-byte headers byte-equal to the reference layout;
  * encode: the GPU stream is restored exactly by the reference's own decoder (both its
    single-thread and multi-thread paths) and is bit-identical to the oracle's CPU twin.
All calls go through the C-ABI (zmt_* device entry points or LZ4MT_* callbacks)."""
import numpy as np
import pytest

import _oracle as o
import zstdmt_b200 as z

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def gpu_compress(torch, src, chunk):
    n = int(src.size)
    d_in = torch.from_numpy(src).cuda() if n else torch.empty(1, dtype=torch.uint8, device="cuda")
    comp = z.Lz4DeviceCompressor(n, chunk)
    out, foff = comp.run(d_in)
    torch.cuda.synchronize()
    foff_h = foff.cpu().numpy()
    return out[: int(foff_h[-1])].cpu().numpy(), foff_h


def gpu_decompress(torch, framed, out_sizes):
    offs, sizes = z.scan_frames(framed)
    assert len(offs) == len(out_sizes)
    dec = z.Lz4DeviceDecompressor(offs, sizes, out_sizes)
    d = torch.from_numpy(np.ascontiguousarray(framed)).cuda()
    out, status = dec.run(d)
    torch.cuda.synchronize()
    return out[: dec.out_total].cpu().numpy(), status.cpu().numpy(), dec.out_size.cpu().numpy()


def chunk_sizes(n, chunk):
    return [min(chunk, n - i * chunk) for i in range(max(1, -(-n // chunk)))]


@pytest.mark.parametrize("n", [0, 1, 11, 12, 13, 39, 40, 4095, 4096, 4097, 65535, 65536, 65537, (1 << 20) - 1, 1 << 20, (1 << 20) + 1])
def test_compress_matches_oracle_twin_edge_sizes(torch, n):
    src = z.gen_stream(z.GEN_MIX, n, 1 << 20, first=1)
    framed, foff = gpu_compress(torch, src, 1 << 20)
    expect = o.orc_encode_lz4(src, 1 << 20)
    assert framed.size == expect.size and np.array_equal(framed, expect)


from _data import long_runs_stream as _long_runs_stream


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("chunk", [1 << 20, 65536, 200000])
def test_compress_length_field_corner_cases(torch, seed, chunk):
    src = _long_runs_stream(seed)
    framed, foff = gpu_compress(torch, src, chunk)
    expect = o.orc_encode_lz4(src, chunk)
    assert framed.size == expect.size and np.array_equal(framed, expect)
    rc, back, _ = o.lib_decompress(o.CODEC_LZ4, framed, src.size)      # the reference's decoder (liblz4) restores it
    assert rc == 0 and np.array_equal(back, src)
    rc, back = o.orc_decode(o.CODEC_LZ4, framed, src.size)
    assert rc == 0 and np.array_equal(back, src)
    back, status, sizes = gpu_decompress(torch, framed, chunk_sizes(src.size, chunk))
    assert (status == 0).all() and np.array_equal(back, src)


@pytest.mark.parametrize("kind", [z.GEN_MIX, z.GEN_TEXT, z.GEN_RANDOM, z.GEN_ZEROS])
@pytest.mark.parametrize("chunk", [1 << 20, 4 << 20, 100000])
def test_compress_roundtrip_through_reference(torch, kind, chunk):
    n = (9 << 20) + 4321
    src = z.gen_stream(kind, n, chunk)
    framed, foff = gpu_compress(torch, src, chunk)
    # bit-exact with the CPU twin of the kernel
    expect = o.orc_encode_lz4(src, chunk)
    assert framed.size == expect.size and np.array_equal(framed, expect)
    # container: every 12-byte header is [0x184D2A50][4][payload size] (lz4-mt_compress.c:293-298)
    for i in range(len(foff) - 1):
        h = framed[int(foff[i]): int(foff[i]) + 12].view("<u4")
        assert h[0] == 0x184D2A50 and h[1] == 4 and h[2] == foff[i + 1] - foff[i] - 12
    # the reference's decoder (liblz4, frame by frame) restores the input
    rc, back, frames = o.lib_decompress(o.CODEC_LZ4, framed, n)
    assert rc == 0 and back.size == n and np.array_equal(back, src)
    assert frames == len(foff) - 1
    rc, back = o.orc_decode(o.CODEC_LZ4, framed, n)
    assert rc == 0 and np.array_equal(back, src)


def test_zeros_config1_container(torch):
    """BASELINE config 1: 64 MiB of zeros in 1 MiB chunks -> 64 identical frames."""
    n = 64 << 20
    src = np.zeros(n, np.uint8)
    framed, foff = gpu_compress(torch, src, 1 << 20)
    sizes = np.diff(foff)
    assert len(sizes) == 64 and len(set(sizes.tolist())) == 1
    f0 = framed[: int(sizes[0])]
    for i in range(1, 64):
        assert np.array_equal(framed[int(foff[i]): int(foff[i + 1])], f0)
    # LZ4F header fields equal the reference's except FLG.indep (0x6C vs 0x4C): same content size, checksum
    assert f0[12:16].tobytes().hex() == "04224d18" and f0[16] == 0x6C and f0[17] == 0x40
    assert f0[-8:].tobytes().hex() == "000000007ff93094"      # end mark + XXH32(1 MiB zeros), Appendix A
    rc, back, _ = o.lib_decompress(o.CODEC_LZ4, framed, n)
    assert rc == 0 and back.size == n and not back.any()


@pytest.mark.parametrize("level", [1, 3, 9])
@pytest.mark.parametrize("kind", [z.GEN_MIX, z.GEN_TEXT, z.GEN_RANDOM, z.GEN_ZEROS])
def test_decode_reference_streams_bit_exact(torch, level, kind):
    n, chunk = (10 << 20) + 999, 1 << 20
    src = z.gen_stream(kind, n, chunk)
    framed, _ = o.reference_stream(o.CODEC_LZ4, src, level, chunk)   # linked blocks, FLG 0x4C
    back, status, osz = gpu_decompress(torch, framed, chunk_sizes(n, chunk))
    assert not status.any(), status
    assert back.size == n and np.array_equal(back, src)
    assert osz.tolist() == chunk_sizes(n, chunk)


def test_decode_golden_fixtures(torch):
    import json, os
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    man = json.load(open(os.path.join(gold, "manifest.json")))
    for case in man["cases"]:
        if case["codec"] != "lz4":
            continue
        framed = np.fromfile(os.path.join(gold, case["file"]), dtype=np.uint8)
        src = z.gen_stream(case["kind"], case["n"], case["chunk"], first=case["first"])
        back, status, osz = gpu_decompress(torch, framed, chunk_sizes(case["n"], case["chunk"]))
        assert not status.any(), (case, status)
        assert np.array_equal(back[: case["n"]], src), case


def test_decode_detects_corruption(torch):
    n, chunk = 3 << 20, 1 << 20
    src = z.gen_stream(z.GEN_TEXT, n, chunk)
    framed = o.orc_encode_lz4(src, chunk)
    offs, sizes = z.scan_frames(framed)
    bad = framed.copy(); bad[int(offs[1]) - 1] ^= 1                 # frame 0 content checksum
    _, status, _ = gpu_decompress(torch, bad, chunk_sizes(n, chunk))
    assert status.tolist() == [7, 0, 0]
    bad = framed.copy(); bad[int(offs[1]) + 12 + 4 + 2 + 8] ^= 1    # frame 1 header checksum
    _, status, _ = gpu_decompress(torch, bad, chunk_sizes(n, chunk))
    assert status.tolist() == [0, 4, 0]
    bad = framed.copy(); bad[int(offs[2]) + 12] ^= 1                # frame 2 LZ4F magic
    _, status, _ = gpu_decompress(torch, bad, chunk_sizes(n, chunk))
    assert status.tolist() == [0, 0, 2]
    bad = framed.copy(); bad[int(offs[0]) + 12 + 40] ^= 0x55        # inside frame 0's first block
    _, status, _ = gpu_decompress(torch, bad, chunk_sizes(n, chunk))
    assert status[0] != 0 and status[1] == 0 and status[2] == 0


# ---------------------------------------------------------------- callback API (host buffers)
@pytest.mark.parametrize("n,chunk", [(0, 1 << 20), (1, 1 << 20), ((5 << 20) + 77, 1 << 20), ((3 << 20) + 5, 300000), (70 << 20, 1 << 20)])
def test_LZ4MT_compressCCtx_callbacks(torch, n, chunk):
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    rc, framed, st = z.compress_mem(z.CODEC_LZ4, src, threads=4, level=1, chunk=chunk)
    assert rc == 0
    nframes = max(1, -(-n // chunk))
    # statistics semantics (lz4-mt_compress.c:356-380): frames written, raw bytes read, bytes incl. headers
    assert st["frames"] == nframes and st["insize"] == n and st["outsize"] == framed.size == st["out_bytes"]
    assert st["writes"] == nframes                         # exactly one fn_write per frame, in order
    assert np.array_equal(framed, o.orc_encode_lz4(src, chunk))
    rc, back, _ = o.lib_decompress(o.CODEC_LZ4, framed, n)
    assert rc == 0 and np.array_equal(back, src)


@pytest.mark.parametrize("n,chunk,level", [(0, 1 << 20, 1), (1, 1 << 20, 1), ((6 << 20) + 3, 1 << 20, 1), ((70 << 20) + 1, 1 << 20, 3), (9 << 20, 4 << 20, 1)])
def test_LZ4MT_decompressDCtx_callbacks(torch, n, chunk, level):
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    framed, ref = o.reference_stream(o.CODEC_LZ4, src, level, chunk)
    rst, st_r = ref["compress_stats"], ref["decompress_stats"]
    rc, back, st = z.decompress_mem(z.CODEC_LZ4, framed, n + 16, threads=4)
    assert rc == 0, z.lib().LZ4MT_getErrorString(rc)
    assert back.size == n and np.array_equal(back, src)
    # decompress statistics: Insize counts payload + 12 per frame (lz4-mt_decompress.c:238,264)
    assert st["frames"] == rst[1] and st["insize"] == framed.size and st["outsize"] == n
    # same counters as the reference's own decoder on the same stream
    assert [st["frames"], st["insize"], st["outsize"]] == [st_r[1], st_r[2], st_r[3]]


def test_callback_error_paths(torch):
    L = z.lib()
    smax = (1 << 64) - 1
    src = z.gen_stream(z.GEN_TEXT, 1 << 20, 1 << 20)
    framed = o.orc_encode_lz4(src, 1 << 20)
    # bad first magic -> data_error (lz4-mt_decompress.c:515-516)
    bad = framed.copy(); bad[0] ^= 1
    rc, _, _ = z.decompress_mem(z.CODEC_LZ4, bad, 2 << 20)
    assert rc == smax - 4 + 1
    # skippable size field != 4 -> data_error (:235)
    bad = framed.copy(); bad[4] = 5
    rc, _, _ = z.decompress_mem(z.CODEC_LZ4, bad, 2 << 20)
    assert rc == smax - 4 + 1
    # truncated payload -> data_error (:261-262)
    rc, _, _ = z.decompress_mem(z.CODEC_LZ4, framed[:-100], 2 << 20)
    assert rc == smax - 4 + 1
    # corrupt content checksum -> compression_library, message names the checksum (SURVEY §8b [probe])
    bad = framed.copy(); bad[-1] ^= 1
    rc, _, _ = z.decompress_mem(z.CODEC_LZ4, bad, 2 << 20)
    assert rc == smax - 8 + 1 and L.LZ4MT_isError(rc)
    assert b"contentChecksum" in L.LZ4MT_getErrorString(rc)
    # write callback failing (output too small) is reported as read_fail (shared mt_error, lz4-mt_compress.c:161-173,195-196)
    rc, _, _ = z.decompress_mem(z.CODEC_LZ4, framed, 1000)
    assert rc == smax - 2 + 1


def test_python_callbacks_observe_reference_call_pattern(torch):
    """Compress: reads of exactly `inputsize` until a 0-byte read; writes one per frame, in order."""
    import ctypes
    L = z.lib()
    n, chunk = (2 << 20) + 100, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    pos = [0]; reads = []; writes = []

    def rd(arg, b):
        want = b.contents.size; reads.append(want)
        take = min(want, n - pos[0])
        ctypes.memmove(b.contents.buf, src[pos[0]:].ctypes.data, take) if take else None
        pos[0] += take; b.contents.size = take
        return 0

    def wr(arg, b):
        writes.append(ctypes.string_at(b.contents.buf, b.contents.size))
        return 0

    rw = z.RdWr(z.RW_FN(rd), None, z.RW_FN(wr), None)
    ctx = L.LZ4MT_createCCtx(2, 1, chunk)
    rc = L.LZ4MT_compressCCtx(ctx, ctypes.byref(rw))
    assert rc == 0
    assert reads == [chunk] * 4                     # 3 data reads + the 0-byte EOF read
    assert len(writes) == 3 and L.LZ4MT_GetFramesCCtx(ctx) == 3
    assert L.LZ4MT_GetInsizeCCtx(ctx) == n and L.LZ4MT_GetOutsizeCCtx(ctx) == sum(map(len, writes))
    L.LZ4MT_freeCCtx(ctx)
    assert b"".join(writes) == o.orc_encode_lz4(src, chunk).tobytes()


@pytest.mark.parametrize("spec", ["0,0,0,0,0,0", "0,0,0,0,0,0,0,0"])
def test_more_device_slots_than_host_buffers_share_the_pinned_ring(torch, spec, monkeypatch):
    """A call over more devices than it keeps batches in flight: the device-side slots beyond the fourth borrow the pinned
    staging buffers of slot i % 4 and the reader holds batch q + 4 back until batch q is written.  One GPU named several times
    stands in for several GPUs; the stream must be byte-identical, the counters too."""
    monkeypatch.setenv("ZSTDMT_GPUS", spec)
    n, chunk = (150 << 20) + 4321, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    rc, framed, st = z.compress_mem(z.CODEC_LZ4, src, threads=4, level=1, chunk=chunk)
    assert rc == 0 and st["frames"] == -(-n // chunk) and st["insize"] == n and st["outsize"] == framed.size
    assert np.array_equal(framed, o.orc_encode_lz4(src, chunk))
    rc, zf, zst = z.compress_mem(z.CODEC_ZSTD, src[: 40 << 20], threads=4, level=3, chunk=chunk)
    assert rc == 0
    rc, back, _ = z.decompress_mem(z.CODEC_ZSTD, zf, (40 << 20) + 16, threads=4)
    assert rc == 0 and np.array_equal(back, src[: 40 << 20])
    rc, back, _ = z.decompress_mem(z.CODEC_LZ4, framed, n + 16, threads=4)
    assert rc == 0 and np.array_equal(back, src)
