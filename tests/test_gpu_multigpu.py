"""The north_star multi-GPU path: ONE {LZ4MT,ZSTDCB}_{compress,decompress} call deals its batches round-robin over the
GPUs named by ZSTDMT_GPUS and re-serialises the frames on the host in frame order (the pt_write rule,
lib/lz4-mt_compress.c:178-205).  Chunks are independent and the encoder is deterministic (SURVEY fact 0.7), so the
stream must be byte-identical to the one-GPU stream.  Skipped on a box with a single GPU."""
import os

import numpy as np
import pytest

import _oracle as o
import zstdmt_b200 as z

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ngpu():
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 CUDA devices")
    return torch.cuda.device_count()


def with_gpus(spec, fn):
    old = os.environ.get("ZSTDMT_GPUS")
    os.environ["ZSTDMT_GPUS"] = spec
    try:
        return fn()
    finally:
        if old is None:
            os.environ.pop("ZSTDMT_GPUS", None)
        else:
            os.environ["ZSTDMT_GPUS"] = old


def batches(n):
    L = z.lib()
    L.zmt_device_batches.restype = z.c_u64; L.zmt_device_batches.argtypes = [z.ctypes.c_int]
    return [int(L.zmt_device_batches(d)) for d in range(n)]


@pytest.mark.parametrize("codec,chunk", [(z.CODEC_LZ4, 1 << 20), (z.CODEC_ZSTD, 1 << 20), (z.CODEC_ZSTD, 4 << 20), (z.CODEC_LZ4, 300000)])
def test_one_call_over_all_gpus_is_byte_identical_and_in_order(ngpu, codec, chunk):
    n = (200 << 20) + 12345
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    rc, one, st1 = with_gpus("0", lambda: z.compress_mem(codec, src, threads=4, level=1 if codec == z.CODEC_LZ4 else 3, chunk=chunk))
    assert rc == 0
    before = batches(ngpu)
    rc, allg, st = with_gpus("all", lambda: z.compress_mem(codec, src, threads=4, level=1 if codec == z.CODEC_LZ4 else 3, chunk=chunk))
    assert rc == 0
    after = batches(ngpu)
    assert all(a > b for a, b in zip(after, before)), (before, after)          # every GPU took batches
    assert allg.size == one.size and np.array_equal(allg, one)                 # same bytes, same order
    assert st["frames"] == st1["frames"] and st["insize"] == n and st["outsize"] == allg.size
    # the reference's decoder (liblz4 / libzstd, frame by frame) restores the multi-GPU stream
    rc, back, _ = o.lib_decompress(codec, allg, n)
    assert rc == 0 and np.array_equal(back, src)
    # decompression dealt over all GPUs: frames come back in order
    before = batches(ngpu)
    rc, back, dst = with_gpus("all", lambda: z.decompress_mem(codec, allg, n + 16, threads=4))
    after = batches(ngpu)
    assert rc == 0 and back.size == n and np.array_equal(back, src)
    assert sum(a > b for a, b in zip(after, before)) >= 2
    assert dst["frames"] == st["frames"]


def test_reference_framed_stream_decodes_over_all_gpus(ngpu):
    n, chunk = (300 << 20) + 7, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    for codec, level in ((z.CODEC_LZ4, 1), (z.CODEC_ZSTD, 3)):
        framed, _ = o.reference_stream(codec, src, level, chunk)
        rc, back, st = with_gpus("all", lambda: z.decompress_mem(codec, framed, n + 16, threads=4))
        assert rc == 0 and np.array_equal(back, src)


def test_explicit_device_list(ngpu):
    n, chunk = 64 << 20, 1 << 20
    src = z.gen_stream(z.GEN_TEXT, n, chunk)
    before = batches(ngpu)
    rc, out, st = with_gpus("1", lambda: z.compress_mem(z.CODEC_LZ4, src, threads=2, level=1, chunk=chunk))
    after = batches(ngpu)
    assert rc == 0 and np.array_equal(out, o.orc_encode_lz4(src, chunk))
    assert after[1] > before[1] and after[0] == before[0]


def test_calling_thread_gets_its_cuda_device_back(ngpu):
    """The pipeline switches the calling thread between the GPUs it deals to; on return the thread's current device must be
    the one it came with (a CUDA / torch caller keeps its own notion of it).  Checked at the driver level."""
    import ctypes
    import torch
    cu = ctypes.CDLL("libcuda.so.1")
    def cur():
        d = ctypes.c_int(-1)
        assert cu.cuCtxGetDevice(ctypes.byref(d)) == 0
        return d.value
    torch.cuda.set_device(0)
    torch.zeros(1, device="cuda")                       # make device 0's context current on this thread
    assert cur() == 0
    src = z.gen_stream(z.GEN_TEXT, 64 << 20, 1 << 20)
    rc, framed, _ = with_gpus("all", lambda: z.compress_mem(z.CODEC_LZ4, src, threads=4, level=1, chunk=1 << 20))
    assert rc == 0 and cur() == 0
    rc, back, _ = with_gpus("all", lambda: z.decompress_mem(z.CODEC_LZ4, framed, src.size + 16, threads=4))
    assert rc == 0 and cur() == 0 and np.array_equal(back, src)
    assert float(torch.ones(4, device="cuda").sum().item()) == 4.0 and torch.cuda.current_device() == 0
