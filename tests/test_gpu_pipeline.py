"""GPU tests of the host pipeline's less travelled branches (run on the B200 box: pytest -m gpu).

The main paths are covered elsewhere; these pin batch boundaries that close on the frame count, the whole-slot
D2H, carried frames and slots that grow for one frame, the slot pool (device-only borrowers included), repeated
calls on one context, ring sharing, and errors raised inside Python callbacks.  Every call checks the bytes, the
frame / insize / outsize counters and how often fn_read and fn_write were called."""
import ctypes
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

import _oracle as o
import zstdmt_b200 as z

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CODECS = [z.CODEC_LZ4, z.CODEC_ZSTD]
SMAX = (1 << 64) - 1


@pytest.fixture(scope="module")
def torch():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    torch.cuda.set_device(0)
    return torch


def level_of(codec):
    return 1 if codec == z.CODEC_LZ4 else 3


def err(codec, name):
    """Library error codes (include/lz4-mt.h, include/zstd-mt.h)."""
    neg = {"read_fail": (2, 3), "canceled": (9, 10)}[name][codec == z.CODEC_ZSTD]
    return SMAX - neg + 1


def check_compressed(codec, src, chunk, rc, framed, st):
    """The result of a successful compress call: bytes, counters and call counts."""
    assert rc == 0
    nframes = max(1, -(-src.size // chunk))
    assert st["frames"] == nframes and st["insize"] == src.size and st["outsize"] == framed.size == st["out_bytes"]
    assert st["reads"] == nframes + 1 and st["writes"] == nframes            # one read per chunk + the 0-byte EOF read
    if codec == z.CODEC_LZ4:
        assert np.array_equal(framed, o.orc_encode_lz4(src, chunk))
    else:
        rc, back, frames = o.lib_decompress(o.CODEC_ZSTD, framed, src.size)
        assert rc == 0 and frames == nframes and np.array_equal(back, src)


def compress_checked(codec, src, chunk, threads=4):
    rc, framed, st = z.compress_mem(codec, src, threads=threads, level=level_of(codec), chunk=chunk)
    check_compressed(codec, src, chunk, rc, framed, st)
    return framed.copy(), st


def in_fresh_process(tmp_path, env, script, **arrays):
    """Runs `script` in a new process, so that the process-wide slot pool starts empty and a call gets the slots its own
    knobs ask for.  `z` and `np` are imported, `arrays` are bound to their names, and the dict `out` comes back."""
    np.savez(tmp_path / "in.npz", **arrays)
    prog = ("import sys, pickle, numpy as np\nsys.path.insert(0, %r)\nimport zstdmt_b200 as z\n"
            "globals().update(dict(np.load(%r)))\nout = {}\n%s\npickle.dump(out, open(%r, 'wb'))\n"
            % (ROOT, str(tmp_path / "in.npz"), script, str(tmp_path / "out.pkl")))
    r = subprocess.run([sys.executable, "-c", prog], env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    with open(tmp_path / "out.pkl", "rb") as f:
        return pickle.load(f)


def decompress_reads(codec, nframes):
    """fn_read calls of a framed decode: LZ4 sniffs magic (4) + rest of the header (8), zstd reads 16 bytes at once;
    then the first payload, a header + payload per further frame, and the 0-byte read at the end."""
    return 2 * nframes + 2 if codec == z.CODEC_LZ4 else 2 * nframes + 1


def check_decompressed(codec, framed, src, nframes, rc, back, st):
    assert rc == 0, z.lib().LZ4MT_getErrorString(rc) if codec == z.CODEC_LZ4 else z.lib().ZSTDCB_getErrorString(rc)
    assert back.size == src.size and np.array_equal(back, src)
    assert st["frames"] == nframes and st["insize"] == framed.size and st["outsize"] == src.size
    assert st["reads"] == decompress_reads(codec, nframes) and st["writes"] == nframes


def decompress_checked(codec, framed, src, nframes):
    rc, back, st = z.decompress_mem(codec, framed, src.size + 16, threads=4)
    check_decompressed(codec, framed, src, nframes, rc, back, st)
    return st


# ---------------------------------------------------------------- batches that close on the frame count
@pytest.mark.parametrize("codec", CODECS)
def test_more_frames_than_a_decompress_table_holds(torch, codec):
    """10 000 frames of 1 KiB: a decompress batch closes at 8192 frames long before its 32 MiB of input."""
    chunk, nframes = 1024, 10000
    src = z.gen_stream(z.GEN_MIX, chunk * nframes - 100, chunk)
    framed, _ = compress_checked(codec, src, chunk)
    decompress_checked(codec, framed, src, nframes)


# ---------------------------------------------------------------- whole-slot D2H
@pytest.mark.parametrize("codec", CODECS)
def test_whole_slot_d2h_matches_piecewise(torch, codec, monkeypatch):
    n, chunk = (70 << 20) + 4321, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    framed, _ = compress_checked(codec, src, chunk)
    nframes = -(-n // chunk)
    st_pieces = decompress_checked(codec, framed, src, nframes)
    monkeypatch.setenv("ZSTDMT_B200_D2H_PIECE_MB", "0")
    st_whole = decompress_checked(codec, framed, src, nframes)
    assert st_whole == st_pieces


# ---------------------------------------------------------------- carried frames, slots grown for one frame
def mixed_stream(codec):
    """Frames smaller and larger than 1 MiB of payload, and small frames that decode to more than 2 MiB."""
    parts = [(z.GEN_MIX, 700 << 10, 64 << 10), (z.GEN_RANDOM, (3 << 20) + 5, 3 << 20), (z.GEN_ZEROS, 4 << 20, 4 << 20),
             (z.GEN_MIX, 2 << 20, 200000), (z.GEN_TEXT, 3 << 20, 3 << 19), (z.GEN_RANDOM, 900 << 10, 900 << 10),
             (z.GEN_MIX, 1 << 20, 1 << 16)]
    srcs, frames, outs = [], [], []
    for i, (kind, n, chunk) in enumerate(parts):
        s = z.gen_stream(kind, n, chunk, first=i)
        f, _ = compress_checked(codec, s, chunk)
        srcs.append(s); frames.append(f); outs += [min(chunk, n - k) for k in range(0, n, chunk)]
    framed = np.concatenate(frames)
    _, payloads = z.scan_frames(framed)
    assert payloads.max() > 1 << 20 and max(outs) > 2 << 20
    return framed, np.concatenate(srcs), len(outs)


@pytest.mark.parametrize("codec", CODECS)
def test_small_decode_batches_carry_and_grow(torch, codec, tmp_path):
    """ZSTDMT_B200_DBATCH_MB=1 gives 1 MiB / 2 MiB decode slots: frames that do not fit behind the others start the next
    batch, and the empty slot grows for a single frame of more than 1 MiB of payload or 2 MiB of output.  Both calls run
    in a fresh process: pooled slots of earlier calls are larger and would hold the whole stream in one batch."""
    framed, src, nframes = mixed_stream(codec)
    script = "rc, back, st = z.decompress_mem(%d, framed, %d, threads=4)\nout.update(rc=rc, back=back.copy(), st=st)" % (codec, src.size + 16)
    runs = [in_fresh_process(tmp_path, env, script, framed=framed) for env in ({}, {"ZSTDMT_B200_DBATCH_MB": "1"})]
    for r in runs:
        check_decompressed(codec, framed, src, nframes, r["rc"], r["back"], r["st"])
    assert runs[1]["st"] == runs[0]["st"]


# ---------------------------------------------------------------- slot pool
@pytest.mark.parametrize("codec", CODECS)
def test_pool_off_and_pooled_slots_agree(torch, codec, tmp_path):
    """Two contexts in a row over six device slots on one GPU, in a fresh process so that the pool starts empty.  The
    first compress context's eight slots (four owning the pinned buffers, four device-only borrowers) and the first
    decode context's six slots all fit the 16-entry pool, so the second contexts take every slot back from it,
    borrowers included.  With ZSTDMT_B200_NO_POOL=1 every context allocates its own.  All give the same results."""
    n, chunk = (40 << 20) + 77, 1 << 20
    src = z.gen_stream(z.GEN_TEXT, n, chunk)
    nframes = -(-n // chunk)
    script = ("out['res'] = []\nfor _ in range(2):\n"
              "    rc, f, st = z.compress_mem(%d, src, threads=4, level=%d, chunk=%d)\n"
              "    rc2, back, dst = z.decompress_mem(%d, f, %d, threads=4)\n"
              "    out['res'].append((rc, f.copy(), st, rc2, back.copy(), dst))\n" % (codec, level_of(codec), chunk, codec, n + 16))
    results = []
    for env in ({}, {"ZSTDMT_B200_NO_POOL": "1"}):
        results += in_fresh_process(tmp_path, dict(env, ZSTDMT_GPUS="0,0,0,0,0,0"), script, src=src)["res"]
    for rc, framed, st, rc2, back, dst in results:
        check_compressed(codec, src, chunk, rc, framed, st)
        check_decompressed(codec, framed, src, nframes, rc2, back, dst)
        assert np.array_equal(framed, results[0][1]) and st == results[0][2] and dst == results[0][5]


# ---------------------------------------------------------------- Python callbacks
class CbIO:
    """fn_read / fn_write over host memory, recording every call.  fail_read_at / fail_write_at: the 1-based call that
    returns an error code instead of moving bytes."""

    def __init__(self, data, fail_read_at=None, read_rv=-2, fail_write_at=None, write_rv=-1):
        self.data = np.ascontiguousarray(data, dtype=np.uint8)
        self.pos, self.reads, self.writes = 0, [], []
        self.fail_read_at, self.read_rv, self.fail_write_at, self.write_rv = fail_read_at, read_rv, fail_write_at, write_rv
        self.failed, self.writes_after_failure = False, 0
        self.rdwr = z.RdWr(z.RW_FN(self._rd), None, z.RW_FN(self._wr), None)

    def _rd(self, arg, b):
        want = b.contents.size
        self.reads.append(want)
        if len(self.reads) == self.fail_read_at:
            return self.read_rv
        take = min(want, self.data.size - self.pos)
        if take:
            ctypes.memmove(b.contents.buf, self.data[self.pos:].ctypes.data, take)
        self.pos += take
        b.contents.size = take
        return 0

    def _wr(self, arg, b):
        if self.fail_write_at is not None and len(self.writes) + 1 >= self.fail_write_at:
            if self.failed:
                self.writes_after_failure += 1
            self.failed = True
            return self.write_rv
        self.writes.append(ctypes.string_at(b.contents.buf, b.contents.size))
        return 0

    def written(self):
        return b"".join(self.writes)


def api(codec):
    L = z.lib()
    pre = "LZ4MT_" if codec == z.CODEC_LZ4 else "ZSTDCB_"
    return lambda name: getattr(L, pre + name)


def counters(f, ctx, kind):
    return f("GetFrames" + kind)(ctx), f("GetInsize" + kind)(ctx), f("GetOutsize" + kind)(ctx)


@pytest.mark.parametrize("codec", CODECS)
def test_compress_context_called_twice(torch, codec):
    """Slots persist across calls on one context and the stream is the same.  zstd resets its counters per call, LZ4
    keeps counting, as the reference does."""
    f = api(codec)
    n, chunk = (20 << 20) + 12345, 1 << 20
    nframes = -(-n // chunk)
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    expect, _ = compress_checked(codec, src, chunk)
    ctx = f("createCCtx")(4, level_of(codec), chunk)
    assert ctx
    try:
        for call in (1, 2):
            io = CbIO(src)
            assert f("compressCCtx")(ctx, ctypes.byref(io.rdwr)) == 0
            assert io.reads == [chunk] * (nframes + 1) and len(io.writes) == nframes
            assert io.written() == expect.tobytes()
            k = call if codec == z.CODEC_LZ4 else 1
            assert counters(f, ctx, "CCtx") == (k * nframes, k * n, k * expect.size)
    finally:
        f("freeCCtx")(ctx)


@pytest.mark.parametrize("env", [{"ZSTDMT_B200_SLOTS": "2"},
                                 {"ZSTDMT_B200_SLOTS": "2", "ZSTDMT_GPUS": "0,0,0,0,0,0"},
                                 {"ZSTDMT_B200_NO_RING_SHARE": "1", "ZSTDMT_GPUS": "0,0,0,0,0,0"}],
                         ids=["slots2", "slots2-gpus6", "no-ring-share-gpus6"])
@pytest.mark.parametrize("codec", CODECS)
def test_slot_count_and_ring_share_knobs_keep_the_stream(torch, codec, env, monkeypatch):
    n, chunk = (60 << 20) + 999, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    framed, st = compress_checked(codec, src, chunk)
    dst = decompress_checked(codec, framed, src, -(-n // chunk))
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    framed2, st2 = compress_checked(codec, src, chunk)
    assert np.array_equal(framed2, framed) and st2 == st
    assert decompress_checked(codec, framed, src, -(-n // chunk)) == dst


@pytest.mark.parametrize("codec", CODECS)
def test_read_canceled_mid_stream(torch, codec):
    f = api(codec)
    n, chunk = 20 << 20, 1 << 20
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    expect, _ = compress_checked(codec, src, chunk)
    # compress: batches of 8 chunks; read 11 cancels inside the second batch, so only the first batch counts as read
    ctx = f("createCCtx")(4, level_of(codec), chunk)
    io = CbIO(src, fail_read_at=11)
    try:
        assert f("compressCCtx")(ctx, ctypes.byref(io.rdwr)) == err(codec, "canceled")
        assert len(io.reads) == 11
        frames, insize, outsize = counters(f, ctx, "CCtx")
        assert insize == 8 * chunk and frames == len(io.writes) <= 8 and outsize == len(io.written())
        assert expect.tobytes().startswith(io.written())
    finally:
        f("freeCCtx")(ctx)
    # decompress: cancel on the header read of the fourth frame
    ctx = f("createDCtx")(4, 0)
    io = CbIO(expect, fail_read_at=decompress_reads(codec, 3))
    try:
        assert f("decompressDCtx")(ctx, ctypes.byref(io.rdwr)) == err(codec, "canceled")
        assert len(io.reads) == decompress_reads(codec, 3)
        frames, insize, outsize = counters(f, ctx, "DCtx")
        assert frames == len(io.writes) == 0 and outsize == 0 and insize <= expect.size
    finally:
        f("freeDCtx")(ctx)


@pytest.mark.parametrize("codec", CODECS)
def test_write_failure_stops_the_call(torch, codec):
    """fn_write failing at frame k is reported as read_fail; the call returns and no fn_write follows the failure."""
    f = api(codec)
    n, chunk, k = 20 << 20, 1 << 20, 5
    src = z.gen_stream(z.GEN_MIX, n, chunk)
    expect, _ = compress_checked(codec, src, chunk)
    offs, _ = z.scan_frames(expect)
    ctx = f("createCCtx")(4, level_of(codec), chunk)
    io = CbIO(src, fail_write_at=k + 1)
    try:
        assert f("compressCCtx")(ctx, ctypes.byref(io.rdwr)) == err(codec, "read_fail")
        assert len(io.writes) == k and io.writes_after_failure == 0
        assert io.written() == expect[: int(offs[k])].tobytes()
        frames, insize, outsize = counters(f, ctx, "CCtx")
        assert frames == k and outsize == int(offs[k]) and k * chunk <= insize <= n
    finally:
        f("freeCCtx")(ctx)
    ctx = f("createDCtx")(4, 0)
    io = CbIO(expect, fail_write_at=k + 1)
    try:
        assert f("decompressDCtx")(ctx, ctypes.byref(io.rdwr)) == err(codec, "read_fail")
        assert len(io.writes) == k and io.writes_after_failure == 0
        assert io.written() == src[: k * chunk].tobytes()
        frames, insize, outsize = counters(f, ctx, "DCtx")
        assert frames == k and outsize == k * chunk and insize <= expect.size
    finally:
        f("freeDCtx")(ctx)
