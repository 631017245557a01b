"""The reference's own integration test (programs/Makefile:252-260: random data -> ./$m-mt -z -> ./$m-mt -d -> cmp), run with
the reference's UNMODIFIED CLI (programs/main.c via programs/{lz4,zstd}-mt.c) linked against libzstdmt_b200.so
(oracle/Makefile target `cli`; binaries live in oracle/_ref/, built where /root/reference exists).  Also crosses the
two implementations: files written by the B200-backed tool are read by the reference-backed tool and vice versa."""
import os
import subprocess

import numpy as np
import pytest

import zstdmt_b200 as z

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFDIR = os.path.join(ROOT, "oracle", "_ref")


def tool(name):
    p = os.path.join(REFDIR, name)
    if not os.path.exists(p):
        pytest.skip(name + " not built (needs the original project's sources at build time)")
    return p


def run(cmd, stdout=None):
    r = subprocess.run(cmd, stdout=stdout if stdout is not None else subprocess.PIPE, stderr=subprocess.PIPE, timeout=300)
    assert r.returncode == 0, (cmd, r.stderr[-500:])
    return r


@pytest.fixture(scope="module")
def gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.mark.parametrize("codec", ["lz4", "zstd"])
def test_reference_make_tests_roundtrip(gpu, tmp_path, codec):
    """`make tests`: 10 MiB of random bytes, default level / threads / chunk size."""
    src = tmp_path / "test.bin"
    src.write_bytes(os.urandom(10 << 20))
    b200 = tool("%s-mt-b200" % codec)
    run([b200, "-z", "-k", "-f", str(src)])
    comp = str(src) + (".lz4" if codec == "lz4" else ".zst")
    assert os.path.exists(comp)
    out = tmp_path / "back.bin"
    with open(out, "wb") as f:
        run([b200, "-d", "-c", comp], stdout=f)
    assert out.read_bytes() == src.read_bytes()


@pytest.mark.parametrize("codec,level", [("lz4", "-1"), ("zstd", "-3")])
def test_cross_with_reference_cli(gpu, tmp_path, codec, level):
    """B200-written file -> reference tool decodes; reference-written file -> B200 tool decodes (compressible data)."""
    data = z.gen_stream(z.GEN_MIX, (9 << 20) + 12345, 1 << 20)
    src = tmp_path / "mix.bin"
    src.write_bytes(data.tobytes())
    b200, ref = tool("%s-mt-b200" % codec), tool("%s-mt-ref" % codec)
    ext = ".lz4" if codec == "lz4" else ".zst"
    a = tmp_path / ("a" + ext); b = tmp_path / ("b" + ext)
    with open(a, "wb") as f:
        run([b200, level, "-T", "4", "-b", "1", "-c", str(src)], stdout=f)
    with open(b, "wb") as f:
        run([ref, level, "-T", "4", "-b", "1", "-c", str(src)], stdout=f)
    for tool_, file_, threads in ((ref, a, "1"), (ref, a, "4"), (b200, b, "4"), (b200, a, "2")):
        r = run([tool_, "-d", "-T", threads, "-c", str(file_)])
        assert r.stdout == data.tobytes(), (tool_, file_)
    # -B statistics line "Level;Threads;InSize;OutSize;Frames" (main.c:238-243) has the reference's shape
    r = run([b200, level, "-T", "4", "-b", "1", "-B", "-c", str(src)])
    line = [l for l in r.stderr.decode().splitlines() if l.count(";") == 4 and l[0].isdigit()]
    assert line, r.stderr[-300:]
    f = line[-1].split(";")
    assert int(f[2]) == data.size and int(f[4]) == 10 and int(f[3]) == a.stat().st_size
