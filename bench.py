#!/usr/bin/env python
"""bench.py — benchmarks of the zstdmt hot path on B200 (one JSON line per run, the driver's contract).

    python bench.py --gpus N --steps K --warmup W [--mode M]        (N>1: under torchrun, one rank per GPU)
    python bench.py --impl reference [--mode M] ...                  (the reference's own pthread + liblz4/libzstd path on the host cores)

Modes = the BASELINE.json configs (default: lz4-compress, the config the headline metric is quoted on):
    lz4-compress    configs[1]  lz4-mt level 1, 8 GiB Silesia-mix per GPU, 1 MiB chunks                 (weak scaling)
    lz4-decompress  configs[2]  lz4-mt decompress-only, 32 GiB stream framed by the REFERENCE, 1->8 GPUs  (strong scaling)
    zstd-compress   configs[3]  zstd-mt level 3, 8 GiB synthetic text per GPU, 1 MiB chunks              (weak scaling)
    zstd-mix        configs[4]  zstd-mt level 3, Silesia-mix, 4 MiB chunks, 8 GiB per GPU (64 GiB at 8)  (weak scaling)
The default run also carries short device-timed legs of the other configs in `extra` (so a 1->8 GPU sweep records
them at every N); `--no-extra` drops them.  `--steps K` is the number of timed steps of every device-timed leg.

--dump-outputs DIR writes what the timed path computed in its last step, as float32 / float64 .npy files (rank 0's
share under N>1), so that two builds can be compared output for output on identical inputs:
    compress modes  : frame_offsets (the frame_off array, all of it), framed_sample_positions + framed_sample (a fixed,
                      seeded sample of the framed bytes)
    lz4-decompress  : status and out_size (per frame, all of them), decoded_sample_positions + decoded_sample

A step = one pass of the per-chunk hot path over the whole batch:
  value    : GB/s of (bytes in + bytes out), device-timed with CUDA events, inputs resident in HBM, max over ranks
  e2e      : the same metric through the reference-shaped callback API with HOST buffers — ONE call on rank 0 that deals
             its batches over all N GPUs (ZSTDMT_GPUS=0..N-1) and reassembles the frames in order; H2D/D2H inside
  roofline : the dominant kernel of the mode against the measured HBM copy peak
  cpu_baseline : the unmodified reference (oracle/_ref) on this box's cores, bounded sample (N=1 only)
Multi-GPU: chunks are dealt round-robin in batches of 8 (the product's granularity), no collective on the data path.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np

GIB = 1 << 30
DEAL_BATCH = 8            # chunks per dealt batch (host_api.cpp: compress slots hold 8 MiB = 8 chunks of 1 MiB)
DUMP_SAMPLES = 1 << 21    # sampled bytes per --dump-outputs buffer: 8 B position + 4 B value each, 24 MiB
DUMP_SEED = 20240601

MODES = {
    "lz4-compress": dict(codec="lz4", op="c", kind="mix", chunk_mib=1, gib=8.0, level=1, scaling="weak",
                         metric="lz4-mt level-1 compress throughput, bytes in + framed bytes out",
                         workload="lz4-mt level 1, 8 GiB synthetic Silesia-mix generator, 1 MiB chunks, per GPU (BASELINE configs[1])"),
    "lz4-decompress": dict(codec="lz4", op="d", kind="mix", chunk_mib=1, gib=32.0, level=1, scaling="strong",
                           metric="lz4-mt decompress throughput, framed bytes in + bytes out",
                           workload="lz4-mt decompress-only, 32 GiB stream pre-framed by the reference (LZ4MT_compressCCtx level 1, 1 MiB chunks, "
                                    "linked blocks; a 2 GiB framed Silesia-mix segment tiled 16x), split over the GPUs (BASELINE configs[2])"),
    "zstd-compress": dict(codec="zstd", op="c", kind="text", chunk_mib=1, gib=8.0, level=3, scaling="weak",
                          metric="zstd-mt level-3 compress throughput, bytes in + framed bytes out",
                          workload="zstd-mt level 3, 8 GiB synthetic text, 1 MiB chunks, per GPU (BASELINE configs[3])"),
    "zstd-mix": dict(codec="zstd", op="c", kind="mix", chunk_mib=4, gib=8.0, level=3, scaling="weak",
                     metric="zstd-mt level-3 compress throughput, bytes in + framed bytes out",
                     workload="zstd-mt level 3, synthetic Silesia-mix, 4 MiB chunks, round-robin over the GPUs, 8 GiB per GPU = 64 GiB at 8 GPUs (BASELINE configs[4])"),
}

KERNEL_NAMES = ["lz4_blocks_pipe_kernel", "xxh32_kernel", "lz4_frame_sizes_kernel", "scan_u64_kernel", "lz4_frame_pack_kernel",
                "lz4_parse_blocks_kernel", "xxh32_kernel(decode)", "lz77_blocks_kernel<zstd>", "zstd_frame_pack_kernel", "zstd_decode(3 kernels)",
                "lz4_exec_blocks_kernel"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="lz4-compress", choices=sorted(MODES))
    ap.add_argument("--size-gib", type=float, default=float(os.environ.get("ZMT_BENCH_GIB", "0")), help="override the mode's size (per GPU; total for lz4-decompress)")
    ap.add_argument("--ref-sample-gib", type=float, default=float(os.environ.get("ZMT_BENCH_REF_GIB", "2")))
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the end-to-end leg (default min(steps, 8))")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="device-timed leg only (profiling runs under ncu)")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the rank's process to the CPUs next to its GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's outputs to DIR/<name>.npy")
    return ap.parse_args()


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.p, self.lines = index, None, []

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True); self.t.start()
        except Exception:
            self.p = None
        return self

    def _pump(self):
        for ln in self.p.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def traffic_per_launch(kernel_key, algorithmic_bytes):
    """DRAM bytes per launch of a kernel: dram__bytes_read.sum + dram__bytes_write.sum of ONE ncu --set full capture
    (profiles/r2_traffic.json, else r1; made at a smaller size), scaled by algorithmic bytes to this launch."""
    for name in ("r2_traffic.json", "r1_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))[kernel_key]
            return float(t["dram_bytes"]) / float(t["algorithmic_bytes"]) * algorithmic_bytes
        except Exception:
            continue
    return None


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def gpu_local_cpus(index):
    """CPUs next to GPU `index` (its PCIe root's NUMA node), from sysfs; None if unknown."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("00000000:"):
            bus = bus[4:]
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bus).read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        return cpus or None
    except Exception:
        return None


def kind_id(z, name):
    return {"mix": z.GEN_MIX, "text": z.GEN_TEXT, "zeros": z.GEN_ZEROS, "random": z.GEN_RANDOM}[name]


def ref_fn(o, codec, op):
    return getattr(o.ref(), "ref_%s_%s_mem" % (codec, "compress" if op == "c" else "decompress"))


def ref_framed_segment(z, o, M, seg_bytes):
    """A Silesia-mix segment framed as the UNMODIFIED reference frames it (LZ4MT/ZSTDCB_compressCCtx): the same
    liblz4 / libzstd call per chunk behind the same 12-byte headers, byte for byte (tests/_oracle.py lib_compress,
    checked against digests of the reference's output by the test suite)."""
    chunk = M["chunk_mib"] << 20
    src = z.gen_stream(kind_id(z, M["kind"]), seg_bytes, chunk)
    return src, o.lib_compress(o.CODEC_LZ4 if M["codec"] == "lz4" else o.CODEC_ZSTD, src, M["level"], chunk)


# =============================================================================== reference arm
def run_reference(args):
    """The reference's own CPU implementation of the path (oracle/_ref: unmodified lib/*-mt_*.c + liblz4 / libzstd),
    all host threads, bounded sample per step.  Loads the generator library only — never the product library."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import _oracle as o
    import zstdmt_b200 as z
    M = MODES[args.mode]
    chunk = M["chunk_mib"] << 20
    cores = os.cpu_count() or 1
    threads = min(cores, 128)                      # *_THREAD_MAX
    size = args.size_gib if args.size_gib > 0 else M["gib"]
    n = int(min(args.ref_sample_gib, size) * GIB) // chunk * chunk
    st = (ctypes.c_size_t * 5)()
    if M["op"] == "c":
        src = z.gen_stream(kind_id(z, M["kind"]), n, chunk)
        cap = n + n // 64 + (1 << 20)
        out = np.empty(cap, np.uint8)
        fn = ref_fn(o, M["codec"], "c")
        def step():
            t = time.perf_counter()
            rc = fn(threads, M["level"], chunk, src.ctypes.data, n, out.ctypes.data, cap, st)
            dt = time.perf_counter() - t
            assert rc == 0
            return dt, n + int(st[0]), int(st[0])
        sample = "first %d MiB of the workload per step, %s_compressCCtx(T=%d, level %d, %d MiB chunks), memory-to-memory callbacks" % (
            n >> 20, "LZ4MT" if M["codec"] == "lz4" else "ZSTDCB", threads, M["level"], M["chunk_mib"])
    else:
        src, framed = ref_framed_segment(z, o, M, n)
        back = np.empty(n + 16, np.uint8)
        fn = ref_fn(o, M["codec"], "d")
        def step():
            t = time.perf_counter()
            rc = fn(threads, 0, framed.ctypes.data, framed.size, back.ctypes.data, n + 16, st)
            dt = time.perf_counter() - t
            assert rc == 0 and int(st[0]) == n
            return dt, n + framed.size, framed.size
        sample = "one %d MiB reference-framed segment of the workload per step, LZ4MT_decompressDCtx(T=%d), memory-to-memory callbacks" % (n >> 20, threads)
    for _ in range(args.warmup):
        step()
    tot, alg, comp = 0.0, 0, 0
    for _ in range(args.steps):
        dt, a, comp = step(); tot += dt; alg += a
    gbs = alg / tot / 1e9
    line = {
        "impl": "reference", "metric": M["metric"], "value": gbs, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot / args.steps * 1e3,
        "higher_is_better": True, "scaling": M["scaling"], "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": M["workload"] + " — this arm: a %d MiB sample of it per step (a throughput; the B200 arm runs the full size)" % (n >> 20),
                   "mode": args.mode, "chunk_bytes": chunk, "sample_bytes_per_step": n, "threads": threads},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "reference", "sample": sample, "cpu_model": cpu_model()},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ratio": n / comp,
    }
    print(json.dumps(line))


# =============================================================================== B200 arm
class Job:
    """torch.distributed plumbing: NCCL for the timing all-reduces, a gloo group for host-side barriers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if args.gpus > 1 and self.world != args.gpus:
            raise SystemExit("--gpus %d needs torchrun --nproc-per-node %d (WORLD_SIZE=%d)" % (args.gpus, args.gpus, self.world))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device (no CPU fallback in the product path)")
        torch.cuda.set_device(self.local)
        self.cpu_group = None
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.cpu_group = dist.new_group(backend="gloo")
        self.stream = torch.cuda.current_stream()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def host_barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.cpu_group)

    def reduce(self, v, op):
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op={"max": self.dist.ReduceOp.MAX, "sum": self.dist.ReduceOp.SUM}[op])
        return float(t.item())

    def gather(self, v):
        if self.world == 1:
            return [float(v)]
        t = self.torch.tensor([float(v)], dtype=self.torch.float64, device="cuda")
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(x.item()) for x in out]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def to_device(torch, host, d=None):
    n = host.size
    if d is None:
        d = torch.empty(n, dtype=torch.uint8, device="cuda")
    step = 256 << 20
    for o in range(0, n, step):
        d[o:o + step].copy_(torch.from_numpy(host[o:o + step]))
    return d


def timed_steps(job, L, fn, steps, warmup):
    """W untimed + K timed calls of fn() on job.stream, bracketed by barrier + synchronize; per-kernel CUDA-event times
    from zmt_prof_*.  Returns (max-over-ranks ms total, this rank's ms total, kernel ms per launch[], launches[], clocks)."""
    torch = job.torch
    for _ in range(max(warmup, 3)):
        fn()
    job.barrier()
    sampler = ClockSampler(job.local).start()
    L.zmt_prof_begin.restype = None
    L.zmt_prof_end.restype = ctypes.c_int
    L.zmt_prof_begin()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    job.barrier()
    ev0.record(job.stream)
    for _ in range(steps):
        fn()
    ev1.record(job.stream)
    job.barrier()
    ms = (ctypes.c_double * 16)(); cnt = (ctypes.c_int * 16)()
    L.zmt_prof_end(ms, cnt, 16)
    clocks = sampler.stop()
    mine = ev0.elapsed_time(ev1)
    return job.reduce(mine, "max"), mine, [ms[i] / max(cnt[i], 1) for i in range(16)], [int(cnt[i]) for i in range(16)], clocks


def sample_device_bytes(torch, buf, nbytes, prefix):
    """A fixed, seeded sample of the first `nbytes` of a device byte buffer: {prefix_positions: float64, prefix: float32}.
    The positions depend on nbytes and DUMP_SEED only, so equal-length outputs are sampled at the same places."""
    if nbytes <= DUMP_SAMPLES:
        pos = np.arange(nbytes, dtype=np.int64)
    else:
        pos = np.sort(np.random.default_rng(DUMP_SEED).integers(0, nbytes, DUMP_SAMPLES, dtype=np.int64))
    vals = buf[torch.from_numpy(pos).to(buf.device)].cpu().numpy()
    return {prefix + "_positions": pos.astype(np.float64), prefix: vals.astype(np.float32)}


def roofline(kms, algorithmic_bytes, ids):
    """The dominant kernel among `ids` (largest mean launch time) against the measured HBM peak."""
    peak, peak_src = measured_peaks()
    k = max(ids, key=lambda i: kms[i])
    if kms[k] <= 0:
        return None
    achieved = algorithmic_bytes / (kms[k] * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic_per_launch(KERNEL_NAMES[k], algorithmic_bytes), "kernel": KERNEL_NAMES[k], "kernel_ms": kms[k],
            "peak_source": peak_src, "algorithmic_bytes_per_launch": algorithmic_bytes}


def gpus_env(spec):
    class _E:
        def __enter__(self):
            self.old = os.environ.get("ZSTDMT_GPUS"); os.environ["ZSTDMT_GPUS"] = spec
        def __exit__(self, *a):
            if self.old is None:
                os.environ.pop("ZSTDMT_GPUS", None)
            else:
                os.environ["ZSTDMT_GPUS"] = self.old
    return _E()


def e2e_calls(job, fn, alg_bytes, steps, spec, everyone):
    """Wall-clock GB/s of `steps` calls of fn() (after one warm-up call that allocates the pinned rings).
    everyone=False: rank 0 alone calls (the other ranks wait at a host barrier), devices from `spec`."""
    val, ms = None, None
    job.barrier()
    if everyone or job.rank == 0:
        with gpus_env(spec):
            fn()
            t = time.perf_counter()
            for _ in range(steps):
                fn()
            dt = time.perf_counter() - t
        val, ms = alg_bytes * steps / dt / 1e9, dt / steps * 1e3
    job.host_barrier()
    return val, ms


# ------------------------------------------------------------------------------- compress legs (configs[1], [3], [4])
def leg_compress(job, args, M, gib, steps, warmup, full):
    """Device-timed compress of this rank's share; full=True adds the parity gates, e2e and cpu_baseline material."""
    import zstdmt_b200 as z
    torch = job.torch
    L = z.lib()
    lz4 = M["codec"] == "lz4"
    chunk = M["chunk_mib"] << 20
    n = int(gib * GIB) // chunk * chunk
    nchunks = n // chunk
    t0 = time.time()
    src = z.gen_stream(kind_id(z, M["kind"]), n, chunk, deal=(job.rank, job.world, DEAL_BATCH))
    gen_s = time.time() - t0
    d_in = to_device(torch, src)
    comp = (z.Lz4DeviceCompressor if lz4 else z.ZstdDeviceCompressor)(n, chunk)
    dev_ms, my_ms, kms, cnt, clocks = timed_steps(job, L, lambda: comp.run(d_in, job.stream), steps, warmup)
    framed = int(comp.frame_off[-1].item())
    outputs = None
    if full and args.dump_outputs:                      # (out, frame_off) of the last timed step
        outputs = {"frame_offsets": comp.frame_off.cpu().numpy().astype(np.float64)}
        outputs.update(sample_device_bytes(torch, comp.out, framed, "framed_sample"))
    alg_mine = n + framed
    total_alg = job.reduce(alg_mine, "sum")
    ids = [0, 1, 2, 3, 4] if lz4 else [7, 8]
    res = {"value": total_alg * steps / (dev_ms * 1e-3) / 1e9, "ms_per_step": dev_ms / steps, "ratio": n / framed,
           "per_rank_ms": [x / steps for x in job.gather(my_ms)], "per_rank_kernel_ms": job.gather(kms[ids[0]]),
           "kernel_ms": {KERNEL_NAMES[i]: kms[i] for i in ids}, "launches": int(job.reduce((5 if lz4 else 4) * steps, "sum")),      # kernels per step: lz4 5 (all event-timed), zstd 4
           "roofline": roofline(kms, alg_mine, ids[:1]), "clocks": clocks, "gen_seconds": gen_s,
           "n": n, "chunk": chunk, "nchunks": nchunks, "framed": framed, "alg_mine": alg_mine, "outputs": outputs}
    # ---- parity gate at full size (not timed): GPU decode of the GPU stream == the input, on the device
    out, foff = comp.out, comp.frame_off
    if lz4:
        foff_h = foff.cpu().numpy().astype(np.uint64)
        sizes = (np.diff(foff_h) - 12).astype(np.uint32)
        dec = z.Lz4DeviceDecompressor(foff_h[:-1], sizes, [chunk] * nchunks)
    else:
        dec = z.ZstdDeviceDecompressor(out[:framed].cpu().numpy())
    dout, status = dec.run(out, job.stream)
    torch.cuda.synchronize()
    assert int(status.abs().sum().item()) == 0, "GPU decode of the GPU stream reported errors"
    assert torch.equal(dout[:n], d_in), "round trip mismatch at full size"
    if full or not args.no_extra:
        # device-timed decode of our own stream (LZ4: independent blocks)
        dms, _, dk, dc, _ = timed_steps(job, L, lambda: dec.run(out, job.stream), steps, 3)
        res["decompress_own_stream"] = {"device_gbs": total_alg * steps / (dms * 1e-3) / 1e9, "ms_per_step": dms / steps,
                                        "kernel_ms": {KERNEL_NAMES[i]: dk[i] for i in ([5, 10, 6] if lz4 else [9])}}
    res["_keep"] = (src, d_in, comp, dec)
    # ---- the reference's decoder restores a slice of this very stream (rank 0)
    if full and job.rank == 0:
        try:
            import _oracle as o
            if o.have_ref():
                k = min(nchunks, max(1, (256 << 20) // chunk))
                cut = int(comp.frame_off[k].item())
                sl = out[:cut].cpu().numpy()
                rc, back, _ = o.ref_decompress(o.CODEC_LZ4 if lz4 else o.CODEC_ZSTD, sl, k * chunk, threads=min(os.cpu_count() or 1, 64))
                assert rc == 0 and np.array_equal(back, src[: k * chunk]), "the reference decoder did not restore the GPU stream"
                res["reference_decoder_gate"] = "%d MiB of the GPU stream restored bit-exact by the reference's decoder" % ((k * chunk) >> 20)
        except AssertionError:
            raise
        except Exception as e:
            res["reference_decoder_gate"] = "skipped: %r" % (e,)
    return res


def e2e_compress(job, args, M, leg, steps):
    """ONE {LZ4MT,ZSTDCB}_compressCCtx call on rank 0 over its host stream, batches dealt over all the job's GPUs."""
    import zstdmt_b200 as z
    Mi = z.memio_lib()
    src, d_in, comp, dec = leg["_keep"]
    n, chunk = leg["n"], leg["chunk"]
    fn = Mi.zmt_lz4_compress_mem if M["codec"] == "lz4" else Mi.zmt_zstd_compress_mem
    cap = z.mt_bound(n, chunk)
    h_out = np.empty(cap, np.uint8)
    st = (ctypes.c_size_t * 5)()
    threads = 4
    outb = [0]
    def call():
        rc = fn(threads, M["level"], chunk, src.ctypes.data, n, h_out.ctypes.data, cap, st)
        assert rc == 0, rc
        outb[0] = int(st[0])
    spec_all = ",".join(str(i) for i in range(job.world))
    val, ms = e2e_calls(job, call, leg["alg_mine"], steps, spec_all, everyone=False)
    e2e = None
    if job.rank == 0:
        assert outb[0] == leg["framed"], "e2e stream size differs from the device path"
        assert np.array_equal(h_out[: 1 << 20], comp.out[: 1 << 20].cpu().numpy())       # same bytes as the device path
        e2e = {"value": val, "unit": "GB/s", "h2d_bytes_per_step": n + 4 * leg["nchunks"], "d2h_bytes_per_step": outb[0] + 8 * (leg["nchunks"] + leg["nchunks"] // DEAL_BATCH + 1),
               "api": "%s_compressCCtx, one call on rank 0, in-memory fn_read/fn_write (harness/memio_glue.c), threads=%d, ZSTDMT_GPUS=%s: batches dealt over %d GPU(s), frames reassembled in order"
                      % ("LZ4MT" if M["codec"] == "lz4" else "ZSTDCB", threads, spec_all, job.world),
               "ms_per_step": ms, "steps": steps, "bytes_per_step": leg["alg_mine"]}
    extra = {}
    if job.world > 1:
        # for comparison: every rank its own call on its own GPU at the same time (N independent streams)
        v, _ = e2e_calls(job, call, leg["alg_mine"], min(steps, 3), str(job.local), everyone=True)
        extra["e2e_n_independent_calls_gbs"] = job.reduce(v, "sum")
    return e2e, extra, h_out, outb[0]


def e2e_decompress_own(job, M, leg, h_out, outb, steps):
    """{LZ4MT,ZSTDCB}_decompressDCtx end to end on the stream just produced (rank 0, all GPUs)."""
    import zstdmt_b200 as z
    Mi = z.memio_lib()
    n = leg["n"]
    fn = Mi.zmt_lz4_decompress_mem if M["codec"] == "lz4" else Mi.zmt_zstd_decompress_mem
    st = (ctypes.c_size_t * 5)()
    back = np.empty(n + 16, np.uint8) if job.rank == 0 else None
    def call():
        rc = fn(4, 0, h_out.ctypes.data, outb, back.ctypes.data, n + 16, st)
        assert rc == 0 and int(st[0]) == n, (rc, int(st[0]))
    val, ms = e2e_calls(job, call, n + outb, steps, ",".join(str(i) for i in range(job.world)), everyone=False)
    if job.rank == 0:
        src = leg["_keep"][0]
        assert np.array_equal(back[: 1 << 22], src[: 1 << 22]) and np.array_equal(back[n - (1 << 20): n], src[n - (1 << 20):])
    return val


def cpu_baseline(args, M, src, n, chunk, codec_fn_c, codec_fn_d, with_decode):
    """The unmodified reference on this box's cores, bounded sample (rank 0, N=1)."""
    cores = os.cpu_count() or 1
    T = min(cores, 128)
    ns = min(n, int(args.ref_sample_gib * GIB)) // chunk * chunk
    capr = ns + ns // 64 + (1 << 20)
    outr = np.empty(capr, np.uint8); st = (ctypes.c_size_t * 5)()
    best = None
    for _ in range(3):
        tt = time.perf_counter()
        rc = codec_fn_c(T, M["level"], chunk, src.ctypes.data, ns, outr.ctypes.data, capr, st)
        dt = time.perf_counter() - tt
        assert rc == 0
        best = dt if best is None else min(best, dt)
    fr = int(st[0])
    ns1 = min(ns, 256 << 20)
    tt = time.perf_counter()
    rc = codec_fn_c(1, M["level"], chunk, src.ctypes.data, ns1, outr.ctypes.data, capr, st)
    dt1 = time.perf_counter() - tt
    fr1 = int(st[0])
    base = {"value": (ns + fr) / best / 1e9, "unit": "GB/s", "cores": T, "kind": "reference", "ratio": ns / fr, "cpu_model": cpu_model(),
            "sample": "first %d MiB of the same workload, %s_compressCCtx(T=%d, level %d) best of 3; T=1 on %d MiB: %.3f GB/s"
                      % (ns >> 20, "LZ4MT" if M["codec"] == "lz4" else "ZSTDCB", T, M["level"], ns1 >> 20, (ns1 + fr1) / dt1 / 1e9)}
    if with_decode:
        rc = codec_fn_c(T, M["level"], chunk, src.ctypes.data, ns, outr.ctypes.data, capr, st)
        frs = outr[: int(st[0])].copy(); backr = np.empty(ns + 16, np.uint8); bestd = None
        for _ in range(3):
            tt = time.perf_counter()
            rc = codec_fn_d(T, 0, frs.ctypes.data, frs.size, backr.ctypes.data, ns + 16, st)
            dt = time.perf_counter() - tt
            assert rc == 0
            bestd = dt if bestd is None else min(bestd, dt)
        base["decompress_gbs"] = (ns + frs.size) / bestd / 1e9
    return base


# ------------------------------------------------------------------------------- decompress leg (configs[2])
def leg_lz4_decompress(job, args, M, total_gib, steps, warmup, seg_gib=2.0, dump=False):
    """Device-timed decode of a stream framed by the reference: a `seg_gib` framed segment tiled to `total_gib`, tiles
    dealt round-robin over the ranks (strong scaling)."""
    import zstdmt_b200 as z
    torch = job.torch
    L = z.lib()
    chunk = M["chunk_mib"] << 20
    total = int(total_gib * GIB) // chunk * chunk
    seg = min(int(seg_gib * GIB), total) // chunk * chunk
    tiles = max(1, total // seg)
    mine = [t for t in range(tiles) if t % job.world == job.rank]
    import _oracle as o
    src, framed = ref_framed_segment(z, o, M, seg)
    framer = "reference framing (LZ4MT_compressCCtx level 1 layout, liblz4 %s, linked blocks)" % o.library_versions()["liblz4"]
    offs, sizes = z.scan_frames(framed)
    nf = len(offs)
    k = max(1, len(mine))
    d_seg = to_device(torch, framed)
    d_src = to_device(torch, src)
    d_in = torch.empty(framed.size * k, dtype=torch.uint8, device="cuda")
    for i in range(k):
        d_in[i * framed.size:(i + 1) * framed.size].copy_(d_seg)
    del d_seg
    all_offs = np.concatenate([offs + np.uint64(i * framed.size) for i in range(k)])
    all_sizes = np.tile(sizes, k)
    outs = [chunk] * (seg // chunk)
    dec = z.Lz4DeviceDecompressor(all_offs, all_sizes, outs * k)
    run = (lambda: dec.run(d_in, job.stream)) if mine else (lambda: None)
    dout, status = dec.run(d_in, job.stream)
    torch.cuda.synchronize()
    assert int(status.abs().sum().item()) == 0, "GPU decode of the reference-framed stream reported errors"
    for i in range(k):
        assert torch.equal(dout[i * seg:(i + 1) * seg], d_src), "decode of the reference-framed stream differs from the source (tile %d)" % i
    dev_ms, my_ms, kms, cnt, clocks = timed_steps(job, L, run, steps, warmup)
    outputs = None
    if dump and mine:                                   # (out, status) of the last timed step, and the per-frame sizes
        outputs = {"status": dec.status.cpu().numpy().astype(np.float64), "out_size": dec.out_size.cpu().numpy().astype(np.float64)}
        outputs.update(sample_device_bytes(torch, dec.out, dec.out_total, "decoded_sample"))
    alg_mine = (framed.size + seg) * len(mine)
    total_alg = job.reduce(alg_mine, "sum")
    ids = [5, 10, 6]
    res = {"value": total_alg * steps / (dev_ms * 1e-3) / 1e9, "ms_per_step": dev_ms / steps, "ratio": seg / framed.size,
           "per_rank_ms": [x / steps for x in job.gather(my_ms if mine else 0.0)], "kernel_ms": {KERNEL_NAMES[i]: kms[i] for i in ids},
           "launches": int(job.reduce(8 * steps if mine else 0, "sum")),        # 8 kernels per decode step (3 of them event-timed)
           "roofline": roofline(kms, alg_mine, [5, 10]) if mine else None, "clocks": clocks, "framed_by": framer,
           "total_out_bytes": seg * tiles, "tiles": tiles, "segment_bytes": seg, "segment_framed_bytes": int(framed.size), "frames_per_segment": nf,
           "tiles_per_rank": [len([t for t in range(tiles) if t % job.world == r]) for r in range(job.world)], "alg_mine": alg_mine,
           "outputs": outputs, "_keep": (src, framed)}
    del dec, dout, d_in, d_src
    torch.cuda.empty_cache()
    return res


def e2e_lz4_decompress(job, leg, steps, tiles=4):
    """ONE LZ4MT_decompressDCtx call on rank 0 over `tiles` copies of the reference-framed segment in host memory."""
    import zstdmt_b200 as z
    Mi = z.memio_lib()
    src, framed = leg["_keep"]
    seg = src.size
    st = (ctypes.c_size_t * 5)()
    if job.rank == 0:
        h_in = np.tile(framed, tiles)
        back = np.empty(seg * tiles + 16, np.uint8)
    def call():
        rc = Mi.zmt_lz4_decompress_mem(4, 0, h_in.ctypes.data, h_in.size, back.ctypes.data, back.size, st)
        assert rc == 0 and int(st[0]) == seg * tiles, (rc, int(st[0]))
    spec_all = ",".join(str(i) for i in range(job.world))
    alg = (framed.size + seg) * tiles
    val, ms = e2e_calls(job, call, alg, steps, spec_all, everyone=False)
    if job.rank != 0:
        return None
    for i in (0, tiles - 1):
        assert np.array_equal(back[i * seg: i * seg + (1 << 22)], src[: 1 << 22]) and np.array_equal(back[(i + 1) * seg - (1 << 20):(i + 1) * seg], src[seg - (1 << 20):])
    return {"value": val, "unit": "GB/s", "h2d_bytes_per_step": int(h_in.size), "d2h_bytes_per_step": seg * tiles + 12 * (seg >> 20) * tiles,
            "api": "LZ4MT_decompressDCtx, one call on rank 0 over %d tiles of the reference-framed segment (%d MiB out), in-memory fn_read/fn_write, threads=4, ZSTDMT_GPUS=%s"
                   % (tiles, (seg * tiles) >> 20, spec_all), "ms_per_step": ms, "steps": steps, "bytes_per_step": alg}


# ------------------------------------------------------------------------------- driver
def run_b200(args):
    job = Job(args)
    import zstdmt_b200 as z
    M = MODES[args.mode]
    bound = None
    if not args.no_bind:
        cpus = gpu_local_cpus(job.local)
        if cpus:
            full_aff = os.sched_getaffinity(0)
            os.sched_setaffinity(0, cpus)
            bound = "rank process bound to the %d CPUs next to GPU %d" % (len(cpus), job.local)
    steps, warmup = args.steps, max(args.warmup, 3)
    e2e_steps = args.e2e_steps if args.e2e_steps > 0 else min(steps, 8)
    size = args.size_gib if args.size_gib > 0 else M["gib"]
    extra = {}
    if M["op"] == "c":
        leg = leg_compress(job, args, M, size, steps, warmup, full=True)
        e2e, h_out = None, None
        if not args.no_e2e:
            e2e, e2x, h_out, outb = e2e_compress(job, args, M, leg, e2e_steps)
            extra.update(e2x)
        if not args.no_extra and not args.no_e2e:
            extra["decompress_own_stream"] = leg.get("decompress_own_stream")
            v = e2e_decompress_own(job, M, leg, h_out, outb, min(e2e_steps, 3))
            if job.rank == 0:
                extra["decompress_own_stream"]["e2e_gbs"] = v
        cfg_par = "chunks dealt round-robin in batches of %d over %d GPU(s), no collective" % (DEAL_BATCH, job.world)
        l2 = "inputs (%.1f GiB per GPU) larger than L2" % (leg["n"] / GIB)
    else:
        leg = leg_lz4_decompress(job, args, M, size, steps, warmup, dump=bool(args.dump_outputs))
        e2e = None if args.no_e2e else e2e_lz4_decompress(job, leg, min(e2e_steps, 5))
        cfg_par = "tiles of the framed stream dealt round-robin over %d GPU(s), no collective" % job.world
        l2 = "inputs (%.1f GiB framed per GPU) larger than L2" % (leg["alg_mine"] / GIB / 2)
    line = {
        "metric": M["metric"], "value": leg["value"], "unit": "GB/s", "n_gpus": job.world, "steps": steps, "warmup": warmup,
        "ms_per_step": leg["ms_per_step"], "higher_is_better": True, "scaling": M["scaling"], "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": M["workload"], "mode": args.mode, "chunk_bytes": M["chunk_mib"] << 20, "parallelism": cfg_par, "l2_policy": l2, "placement": bound},
        "clocks": leg["clocks"], "e2e": e2e, "gpu_launches": leg["launches"], "roofline": leg["roofline"],
        "per_rank_ms": leg["per_rank_ms"], "kernel_ms": leg["kernel_ms"], "ratio": leg["ratio"],
    }
    for k in ("per_rank_kernel_ms", "reference_decoder_gate", "framed_by", "tiles_per_rank", "total_out_bytes", "gen_seconds"):
        if k in leg:
            line[k] = leg[k]
    # ---- CPU baseline beside it (rank 0, N=1 only)
    if job.world == 1:
        try:
            import _oracle as o
            if not o.have_ref():
                line["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": 0, "kind": "reference", "sample": "oracle/_ref not built"}
            else:
                if bound:
                    os.sched_setaffinity(0, full_aff)                   # the reference gets every host thread
                if M["op"] == "c":
                    line["cpu_baseline"] = cpu_baseline(args, M, leg["_keep"][0], leg["n"], leg["chunk"], ref_fn(o, M["codec"], "c"), ref_fn(o, M["codec"], "d"), not args.no_extra)
                else:
                    src, framed = leg["_keep"]
                    T = min(os.cpu_count() or 1, 128); st = (ctypes.c_size_t * 5)(); back = np.empty(src.size + 16, np.uint8); best = None
                    for _ in range(3):
                        tt = time.perf_counter()
                        rc = ref_fn(o, "lz4", "d")(T, 0, framed.ctypes.data, framed.size, back.ctypes.data, src.size + 16, st)
                        dt = time.perf_counter() - tt
                        assert rc == 0
                        best = dt if best is None else min(best, dt)
                    line["cpu_baseline"] = {"value": (src.size + framed.size) / best / 1e9, "unit": "GB/s", "cores": T, "kind": "reference", "cpu_model": cpu_model(),
                                            "sample": "one %d MiB reference-framed segment, LZ4MT_decompressDCtx(T=%d) best of 3" % (src.size >> 20, T)}
                if bound:
                    os.sched_setaffinity(0, cpus)
        except Exception as e:  # the baseline must never take the GPU result down with it
            line["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": 0, "kind": "reference", "sample": "failed: %r" % (e,)}
    # ---- short legs of the other configs (device-timed; recorded at every N by the driver's sweep)
    if not args.no_extra and args.mode == "lz4-compress":
        leg.pop("_keep", None)
        del h_out
        job.torch.cuda.empty_cache()
        xs = steps
        for name, gib in (("lz4-decompress", MODES["lz4-decompress"]["gib"]), ("zstd-compress", 2.0), ("zstd-mix", 2.0)):
            try:
                Mx = MODES[name]
                if Mx["op"] == "d":
                    lx = leg_lz4_decompress(job, args, Mx, gib, xs, 3)
                else:
                    lx = leg_compress(job, args, Mx, gib, xs, 3, full=False)
                lx.pop("_keep", None)
                extra[name] = {"workload": Mx["workload"] + (" — short leg: %.0f GiB per GPU" % gib if Mx["op"] == "c" else ""), "scaling": Mx["scaling"],
                               "device_gbs": lx["value"], "ms_per_step": lx["ms_per_step"], "ratio": lx["ratio"], "per_rank_ms": lx["per_rank_ms"],
                               "kernel_ms": lx["kernel_ms"], "roofline": lx["roofline"], "steps": xs}
                for k in ("framed_by", "tiles_per_rank", "total_out_bytes", "decompress_own_stream"):
                    if k in lx:
                        extra[name][k] = lx[k]
                del lx
                job.torch.cuda.empty_cache()
            except AssertionError:
                raise
            except Exception as e:
                if job.world > 1:
                    raise                                   # a rank that skips the rest of a leg would leave the others in its collectives
                extra[name] = {"error": repr(e)}
    line["extra"] = extra
    if job.rank == 0 and args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in leg["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    if job.rank == 0:
        print(json.dumps(line))
    job.close()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
