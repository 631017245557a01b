"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol the
headers in include/ declare; argument validation and error plumbing behave like the
reference (no compute calls — those need a GPU)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import zstdmt_b200 as z

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for h in ("zstdmt_b200_lz4.h", "zstdmt_b200_zstd.h", "zstdmt_b200_dev.h"):
        p = os.path.join(ROOT, "include", h)
        if not os.path.exists(p):
            continue
        txt = open(p).read()
        txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
        for m in re.finditer(r"\b((?:LZ4MT|ZSTDCB|ZSTDMT|zmt)_\w+)\s*\(", txt):
            names.add(m.group(1))
    names.discard("ZSTDCB_PREFIX"); names.discard("ZSTDCB_ERROR")
    return sorted(names)


def test_library_exports_every_declared_symbol():
    L = z.lib()
    syms = declared_symbols()
    assert len(syms) >= 44
    for s in syms:
        assert hasattr(L, s), "missing export: " + s
    out = subprocess.run(["nm", "-D", z.LIB_PATH], capture_output=True, text=True).stdout
    assert " B lz4mt_errcode" in out or " D lz4mt_errcode" in out
    assert " B zstdmt_errcode" in out or " D zstdmt_errcode" in out


def test_harness_libraries_export_their_header_and_product_does_not():
    """include/zstdmt_b200_harness.h: generator and in-memory callback drivers live outside the product library."""
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "zstdmt_b200_harness.h")).read(), flags=re.S)
    names = sorted(set(m.group(1) for m in re.finditer(r"\b(zmt_\w+)\s*\(", txt)))
    assert len(names) >= 7
    G, M, L = z.gen_lib(), z.memio_lib(), z.lib()
    for s in names:
        assert hasattr(G, s) or hasattr(M, s), "missing harness export: " + s
        assert not hasattr(L, s), "harness symbol leaked into the product library: " + s


def test_create_validates_like_reference():
    L = z.lib()
    # lz4-mt_compress.c:103-108 / lz4-mt_decompress.c:101-102
    assert not L.LZ4MT_createCCtx(0, 1, 0) and not L.LZ4MT_createCCtx(129, 1, 0)
    assert not L.LZ4MT_createCCtx(1, 0, 0) and not L.LZ4MT_createCCtx(1, 13, 0)
    assert not L.LZ4MT_createDCtx(0, 0) and not L.LZ4MT_createDCtx(129, 0)
    # zstd-mt_compress.c:105-110
    assert not L.ZSTDCB_createCCtx(0, 3, 0) and not L.ZSTDCB_createCCtx(1, 23, 0) and not L.ZSTDCB_createCCtx(1, 0, 0)
    c = L.LZ4MT_createCCtx(4, 1, 1 << 20); assert c
    assert L.LZ4MT_GetFramesCCtx(c) == 0 and L.LZ4MT_GetInsizeCCtx(c) == 0 and L.LZ4MT_GetOutsizeCCtx(c) == 0
    L.LZ4MT_freeCCtx(c); L.LZ4MT_freeCCtx(None)
    d = L.ZSTDMT_createDCtx(2, 0); assert d
    L.ZSTDMT_freeDCtx(d)


def test_error_convention():
    L = z.lib()
    size_t_max = ctypes.c_size_t(-1).value
    # isError(c) <=> c > (size_t)-maxCode   (lz4 maxCode 10, zstd 11)
    assert L.LZ4MT_isError(size_t_max - 8 + 1)      # (size_t)-8 compression_library
    assert not L.LZ4MT_isError(0) and not L.LZ4MT_isError(size_t_max - 10 + 1)
    assert L.ZSTDCB_isError(size_t_max - 10 + 1) and not L.ZSTDCB_isError(size_t_max - 11 + 1)
    assert L.LZ4MT_getErrorString(size_t_max - 4 + 1) == b"Malformed input"
    assert L.ZSTDCB_getErrorString(size_t_max - 5 + 1) == b"Malformed input"
    assert L.LZ4MT_getErrorString(size_t_max - 9 + 1) == b"Unspecified lz4mt error code"   # canceled has no entry (lz4-mt_common.c:40-62)
    # NULL contexts: lz4 -> compressionParameter_unsupported (lz4-mt_compress.c:317), zstd -> init_missing (zstd-mt_compress.c:327)
    assert L.LZ4MT_compressCCtx(None, None) == size_t_max - 7 + 1
    assert L.ZSTDCB_compressCCtx(None, None) == size_t_max - 2 + 1
    assert L.LZ4MT_GetInsizeCCtx(None) == 0
    assert L.ZSTDCB_GetInsizeCCtx(None) == size_t_max - 2 + 1


def test_no_gpu_fails_loudly():
    """Without a CUDA device the product must return an error — never fall back to a CPU codec."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import numpy as np
    rc, out, st = z.compress_mem(z.CODEC_LZ4, np.zeros(1000, np.uint8), chunk=1 << 16)
    assert z.lib().LZ4MT_isError(rc) and out.size == 0


def test_chunk_count_and_bounds():
    L = z.lib()
    assert L.zmt_chunk_count(0, 1 << 20) == 1            # empty input still yields one frame (lz4-mt_compress.c:265)
    assert L.zmt_chunk_count(1, 1 << 20) == 1
    assert L.zmt_chunk_count((1 << 20) + 1, 1 << 20) == 2
    assert L.zmt_lz4c_out_bound(1, 1 << 20) >= 1048679   # LZ4F_compressFrameBound(1 MiB)+12 (Appendix A)


@pytest.mark.parametrize("level", [1, 3, 19])
@pytest.mark.parametrize("kind", [z.GEN_TEXT, z.GEN_MIX, z.GEN_RANDOM, z.GEN_ZEROS])
def test_zstd_host_block_scan_on_reference_frames(level, kind):
    """zmt_zstd_scan_frame_host is host logic (the reader thread runs it per frame): on frames made by the real
    reference it must account for every byte of the frame, report the frame's content size and reject truncation /
    trailing bytes.  No GPU involved."""
    import _oracle as o
    import ctypes
    L = z.lib()
    n = (1 << 20) + 12345
    src = z.gen_stream(kind, n, 1 << 20)
    framed, _ = o.reference_stream(o.CODEC_ZSTD, src, level, 1 << 19)
    offs, sizes = z.scan_frames(framed)
    assert len(offs) == 3
    dsz = L.zmt_zstd_blk_desc_bytes()
    total = 0
    for i in range(len(offs)):
        fr = np.ascontiguousarray(framed[int(offs[i]) + 12: int(offs[i]) + 12 + int(sizes[i])])
        cap = fr.size // 3 + 16
        blocks = np.zeros(cap * dsz, np.uint8)
        nblk = ctypes.c_uint32(0); scr = ctypes.c_uint64(0); cs = ctypes.c_uint64(0); nsq = ctypes.c_uint32(0)
        rc = L.zmt_zstd_scan_frame_host(fr.ctypes.data, fr.size, 0, i, blocks.ctypes.data, ctypes.byref(nblk), cap, ctypes.byref(scr), ctypes.byref(cs), ctypes.byref(nsq))
        assert rc == 0 and nblk.value >= 1
        total += cs.value
        # descriptors: comp_off (u64) + comp_size (u32) lead every record; blocks tile the frame after its header
        rec = blocks[: nblk.value * dsz].reshape(nblk.value, dsz)
        comp_off = rec[:, :8].copy().view("<u8")[:, 0]; comp_size = rec[:, 8:12].copy().view("<u4")[:, 0]
        assert (np.diff(comp_off.astype(np.int64)) > 0).all() and int(comp_off[-1]) + int(comp_size[-1]) <= fr.size
        # truncated frame / trailing byte
        nb2 = ctypes.c_uint32(0); s2 = ctypes.c_uint64(0)
        rc = L.zmt_zstd_scan_frame_host(fr.ctypes.data, fr.size - 1, 0, i, blocks.ctypes.data, ctypes.byref(nb2), cap, ctypes.byref(s2), ctypes.byref(cs), ctypes.byref(nsq))
        assert rc != 0
        fr2 = np.concatenate([fr, np.zeros(1, np.uint8)])
        nb2 = ctypes.c_uint32(0); s2 = ctypes.c_uint64(0)
        rc = L.zmt_zstd_scan_frame_host(fr2.ctypes.data, fr2.size, 0, i, blocks.ctypes.data, ctypes.byref(nb2), cap, ctypes.byref(s2), ctypes.byref(cs), ctypes.byref(nsq))
        assert rc != 0
    assert total == n


def test_zstd_host_scan_flags_checksum_and_missing_content_size():
    """Frames as the stock zstd CLI / a streaming producer writes them: the host scan accounts for the 4 checksum bytes,
    reports flag 2 (checksum) / 4 (no content size) and, without a content size, an upper bound of the output."""
    import ctypes
    import test_gpu_plain_streams as t
    L = z.lib()
    src = z.gen_stream(z.GEN_MIX, 700000, 1 << 20)
    dsz = L.zmt_zstd_blk_desc_bytes()
    for fr, want_flags, exact in ((t.zstd_adv(src, 3, checksum=1), 2, True), (t.zstd_adv(src, 3, checksum=0, pieces=[300000, 400000]), 4, False),
                                  (t.zstd_adv(src, 3, checksum=1, pieces=[1, 699999]), 6, False)):
        cap = fr.size // 3 + 16
        blocks = np.zeros(cap * dsz, np.uint8)
        nblk = ctypes.c_uint32(0); scr = ctypes.c_uint64(0); cs = ctypes.c_uint64(0); fl = ctypes.c_uint32(0)
        rc = L.zmt_zstd_scan_frame_host(fr.ctypes.data, fr.size, 0, 0, blocks.ctypes.data, ctypes.byref(nblk), cap, ctypes.byref(scr), ctypes.byref(cs), ctypes.byref(fl))
        assert rc == 0 and (fl.value & 6) == want_flags
        assert cs.value == src.size if exact else cs.value >= src.size
        nb2 = ctypes.c_uint32(0); s2 = ctypes.c_uint64(0)
        assert L.zmt_zstd_scan_frame_host(fr.ctypes.data, fr.size - 1, 0, 0, blocks.ctypes.data, ctypes.byref(nb2), cap, ctypes.byref(s2), ctypes.byref(cs), ctypes.byref(fl)) != 0


def test_levels_above_the_implemented_class_are_announced_or_refused(monkeypatch, capfd):
    """Levels the device encoder does not implement are accepted with a one-time notice (the CLI default for lz4 is 3),
    or refused like any bad parameter under ZSTDMT_B200_STRICT_LEVEL=1 — never silently mapped."""
    L = z.lib()
    c = L.LZ4MT_createCCtx(2, 9, 1 << 20)
    assert c
    L.LZ4MT_freeCCtx(c)
    err = capfd.readouterr().err
    assert "level 9" in err and "level-2" in err
    c = L.LZ4MT_createCCtx(2, 12, 1 << 20); assert c; L.LZ4MT_freeCCtx(c)
    assert "level" not in capfd.readouterr().err                     # said once per codec
    monkeypatch.setenv("ZSTDMT_B200_STRICT_LEVEL", "1")
    assert not L.LZ4MT_createCCtx(2, 3, 1 << 20) and not L.ZSTDCB_createCCtx(2, 5, 0)
    c = L.LZ4MT_createCCtx(2, 1, 1 << 20); assert c; L.LZ4MT_freeCCtx(c)
    c = L.ZSTDCB_createCCtx(2, 3, 0); assert c; L.ZSTDCB_freeCCtx(c)
