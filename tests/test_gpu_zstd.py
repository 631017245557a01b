"""GPU parity tests for the Zstandard path (pytest -m gpu), through the C-ABI.

Bars (BASELINE.json north_star): compression "produces a stream the reference CPU path decompresses to the
identical input" — checked with libzstd, the library the reference decodes with, frame by frame behind the 12-byte
headers, and with the oracle's RFC 8878 restatement; container bytes byte-checked; decode of the reference's own
streams (re-made through libzstd, checked against digests of its output) bit-exact with the original."""
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
    comp = z.ZstdDeviceCompressor(n, chunk)
    out, foff = comp.run(d_in)
    torch.cuda.synchronize()
    foff_h = foff.cpu().numpy()
    return out[: int(foff_h[-1])].cpu().numpy(), foff_h


def gpu_decompress(torch, framed):
    dec = z.ZstdDeviceDecompressor(framed)
    d = torch.from_numpy(np.ascontiguousarray(framed)).cuda()
    out, status = dec.run(d)
    torch.cuda.synchronize()
    return out[: dec.out_total].cpu().numpy(), status.cpu().numpy()[: dec.n], dec


ZSTD_EMPTY = bytes.fromhex("502a4d18040000000900000028b52ffd2000010000")     # SURVEY.md Appendix A


def test_empty_input_equals_reference_bytes(torch):
    framed, foff = gpu_compress(torch, np.zeros(0, np.uint8), 1 << 20)
    assert framed.tobytes() == ZSTD_EMPTY


@pytest.mark.parametrize("n", [1, 2, 63, 64, 255, 256, 257, 4095, 4096, 4097, 16384, 65535, 65536, 65537, 65791, 65792, (1 << 20) - 1, 1 << 20, (1 << 20) + 1])
def test_compress_edge_sizes_roundtrip(torch, n):
    src = z.gen_stream(z.GEN_MIX, n, 1 << 20, first=1)
    framed, foff = gpu_compress(torch, src, 1 << 20)
    rc, back = o.orc_decode(o.CODEC_ZSTD, framed, n)
    assert rc == 0 and back.size == n and np.array_equal(back, src)
    rc, back, _ = o.lib_decompress(o.CODEC_ZSTD, framed, n)
    assert rc == 0 and np.array_equal(back, src)
    back, status, dec = gpu_decompress(torch, framed)
    assert not status.any() and np.array_equal(back, src)


@pytest.mark.parametrize("kind", [z.GEN_MIX, z.GEN_TEXT, z.GEN_RANDOM, z.GEN_ZEROS])
@pytest.mark.parametrize("chunk", [1 << 20, 4 << 20, 100000])
def test_compress_roundtrip_through_reference(torch, kind, chunk):
    n = (9 << 20) + 4321
    src = z.gen_stream(kind, n, chunk)
    framed, foff = gpu_compress(torch, src, chunk)
    # container + zstd frame header per chunk: [0x184D2A50][4][size] 28 B5 2F FD <FHD> <FCS>
    for i in range(len(foff) - 1):
        f = framed[int(foff[i]): int(foff[i + 1])]
        h = f[:12].view("<u4")
        assert h[0] == 0x184D2A50 and h[1] == 4 and h[2] == f.size - 12
        assert f[12:16].tobytes().hex() == "28b52ffd"
        cn = min(chunk, n - i * chunk)
        if cn > 65791:
            assert f[16] == 0xA0 and int(f[17:21].view("<u4")[0]) == cn         # same FHD / FCS as the reference (Appendix A)
    rc, back, frames = o.lib_decompress(o.CODEC_ZSTD, framed, n)
    assert rc == 0 and back.size == n and np.array_equal(back, src) and frames == len(foff) - 1
    rc, back = o.orc_decode(o.CODEC_ZSTD, framed, n)
    assert rc == 0 and np.array_equal(back, src)
    back, status, dec = gpu_decompress(torch, framed)
    assert not status.any() and back.size == n and np.array_equal(back, src)


@pytest.mark.parametrize("first", [2, 3, 4, 5, 6, 7])
def test_every_data_class_roundtrips(torch, first):
    """One chunk of every Silesia-mix class.  Class 6 (random) regression: a single stray 4-byte match inside an
    otherwise incompressible window used to claim the whole window as its literal run."""
    n = 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, 1 << 20, first=first)
    framed, foff = gpu_compress(torch, src, 1 << 20)
    rc, back = o.orc_decode(o.CODEC_ZSTD, framed, n)
    assert rc == 0 and np.array_equal(back, src)
    back, status, dec = gpu_decompress(torch, framed)
    assert not status.any() and np.array_equal(back, src)


@pytest.mark.parametrize("run_len,seed", [(7196, 1), (5, 2), (30000, 3)])
def test_pending_match_then_incompressible_tail(torch, run_len, seed):
    """Regression (found by tools/stress_gpu.py): a window that starts with one long match and continues with
    incompressible bytes keeps that match pending until the window ends, so no sub-block is closed on the way and the
    final block carries up to 64 KiB of literals — more than the literal scratch used to hold (40 KiB)."""
    rng = np.random.default_rng(seed)
    win = []
    for w in range(6):
        head = rng.integers(0, 256, 1 + w, dtype=np.uint8)
        run = np.full(run_len, int(head[-1]), np.uint8)
        win.append(np.concatenate([head, run, rng.integers(0, 256, 65536 - head.size - run_len, dtype=np.uint8)]))
    src = np.concatenate(win)
    framed, foff = gpu_compress(torch, src, 1 << 20)
    rc, back = o.orc_decode(o.CODEC_ZSTD, framed, src.size)
    assert rc == 0 and np.array_equal(back, src)
    rc, b2, _ = o.lib_decompress(o.CODEC_ZSTD, framed, src.size)
    assert rc == 0 and np.array_equal(b2, src)
    back, status, dec = gpu_decompress(torch, framed)
    assert not status.any() and np.array_equal(back, src)


def test_ratio_between_lz4_path_and_libzstd(torch):
    """Sanity: the entropy stage must buy something over the LZ4 container on text."""
    n = 8 << 20
    src = z.gen_stream(z.GEN_TEXT, n, 1 << 20)
    framed, _ = gpu_compress(torch, src, 1 << 20)
    lz4 = o.orc_encode_lz4(src, 1 << 20)
    assert framed.size < 0.9 * lz4.size


@pytest.mark.parametrize("level", [1, 3, 9, 19])
@pytest.mark.parametrize("kind", [z.GEN_MIX, z.GEN_TEXT, z.GEN_RANDOM, z.GEN_ZEROS])
def test_decode_reference_streams_bit_exact(torch, level, kind):
    """libzstd's own frames (what zstd-mt / the reference CLI writes): FSE-described tables, FSE-coded Huffman weights,
    treeless literals, repeat modes and repeat offsets (SURVEY fact 0.6) — decoded by the frame-sequential entropy pass."""
    n, chunk = (6 << 20) + 999, 1 << 20
    src = z.gen_stream(kind, n, chunk)
    framed, _ = o.reference_stream(o.CODEC_ZSTD, src, level, chunk)
    back, status, dec = gpu_decompress(torch, framed)
    assert dec.scan_ok
    assert not status.any(), status
    assert back.size == n and np.array_equal(back, src)
    # and through ZSTDCB_decompressDCtx with host buffers
    rc, back2, st2 = z.decompress_mem(z.CODEC_ZSTD, framed, n + 16, threads=4)
    assert rc == 0 and np.array_equal(back2, src)


def test_decode_golden_fixtures(torch):
    import json, os
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    man = json.load(open(os.path.join(gold, "manifest.json")))
    seen = 0
    for case in man["cases"]:
        if case["codec"] != "zstd":
            continue
        framed = np.fromfile(os.path.join(gold, case["file"]), dtype=np.uint8)
        src = z.gen_stream(case["kind"], case["n"], case["chunk"], first=case["first"])
        back, status, dec = gpu_decompress(torch, framed)
        assert not status.any(), (case, status)
        assert np.array_equal(back[: case["n"]], src), case
        seen += 1
    assert seen >= 3


def test_decode_detects_corruption(torch):
    """zstd frames of this path carry no checksum (like the reference's), so only structural damage is detectable:
    a wrong content size, a broken block header, a sequence bitstream that does not end where it must."""
    n = 3 << 20
    src = z.gen_stream(z.GEN_TEXT, n, 1 << 20)
    framed, foff = gpu_compress(torch, src, 1 << 20)
    bad = framed.copy(); bad[int(foff[1]) + 12 + 5] ^= 0x01               # frame 1: content size field
    back, status, dec = gpu_decompress(torch, bad)
    assert status[1] != 0 and status[0] == 0 and status[2] == 0
    assert np.array_equal(back[: 1 << 20], src[: 1 << 20])
    bad = framed.copy(); bad[int(foff[2]) - 1] = 0                          # frame 1: last byte of the last block's bitstream (end marker gone)
    back, status, dec = gpu_decompress(torch, bad)
    assert status[1] != 0 and status[0] == 0 and status[2] == 0
    bad = framed.copy(); bad[int(foff[0]) + 12 + 9] |= 0x06                 # frame 0: first block header -> reserved block type 3
    dec = z.ZstdDeviceDecompressor(bad)
    assert not dec.scan_ok                                                  # the host scan already refuses it


@pytest.mark.parametrize("n,chunk,level", [(0, 1 << 20, 3), (1, 1 << 20, 3), ((5 << 20) + 77, 1 << 20, 3), ((3 << 20) + 5, 300000, 1), (40 << 20, 4 << 20, 3)])
def test_ZSTDCB_callbacks_roundtrip(torch, n, chunk, level):
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    rc, framed, st = z.compress_mem(z.CODEC_ZSTD, src, threads=4, level=level, chunk=chunk)
    assert rc == 0
    nframes = max(1, -(-n // chunk))
    assert st["frames"] == nframes and st["insize"] == n and st["outsize"] == framed.size and st["writes"] == nframes
    rc, back, _ = o.lib_decompress(o.CODEC_ZSTD, framed, n)
    assert rc == 0 and np.array_equal(back, src)
    rc, back, st = z.decompress_mem(z.CODEC_ZSTD, framed, n + 16, threads=4)
    assert rc == 0 and back.size == n and np.array_equal(back, src)
    assert st["frames"] == nframes and st["outsize"] == n


def test_ZSTDMT_aliases(torch):
    L = z.lib()
    c = L.ZSTDMT_createCCtx(2, 3, 1 << 20); assert c
    assert L.ZSTDMT_GetInsizeCCtx(c) == 0
    L.ZSTDMT_freeCCtx(c)


def test_zstd_bad_stream_errors(torch):
    smax = (1 << 64) - 1
    src = z.gen_stream(z.GEN_TEXT, 1 << 20, 1 << 20)
    rc, framed, st = z.compress_mem(z.CODEC_ZSTD, src, threads=2, level=3, chunk=1 << 20)
    assert rc == 0
    bad = framed.copy(); bad[0] ^= 1                                  # neither skippable nor zstd magic -> data_error (zstd-mt_decompress.c:755-758)
    rc, _, _ = z.decompress_mem(z.CODEC_ZSTD, bad, 2 << 20)
    assert rc == smax - 5 + 1
    rc, _, _ = z.decompress_mem(z.CODEC_ZSTD, framed[:-50], 2 << 20)  # truncated payload -> data_error (:352-353)
    assert rc == smax - 5 + 1


def test_default_chunk_at_level_22_roundtrips(torch):
    """inputsize = 0 at level 22 means 256 MiB chunks (zstd-mt_compress.c:118-127): one frame larger than every default
    staging slot — compress and decompress slots must grow (input, output, block table, entropy scratch) instead of failing."""
    import ctypes
    M = z.memio_lib()
    n = (300 << 20) + 1234
    src = z.gen_stream(z.GEN_TEXT, n, 1 << 20)
    cap = n + n // 64 + (1 << 20)
    out = np.empty(cap, np.uint8); st = (ctypes.c_size_t * 5)()
    rc = M.zmt_zstd_compress_mem(4, 22, 0, src.ctypes.data, n, out.ctypes.data, cap, st)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    framed = out[: int(st[0])]
    offs, sizes = z.scan_frames(framed)
    assert len(offs) == 2 and st[1] == 2                   # 256 MiB + the rest
    back = np.empty(n + 16, np.uint8)
    rc = M.zmt_zstd_decompress_mem(4, 0, framed.ctypes.data, framed.size, back.ctypes.data, n + 16, st)
    assert rc == 0, z.lib().ZSTDCB_getErrorString(rc)
    assert int(st[0]) == n and np.array_equal(back[:n], src)
