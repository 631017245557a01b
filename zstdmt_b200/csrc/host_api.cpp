// host_api.cpp — the drop-in boundary: LZ4MT_* / ZSTDCB_* (+ ZSTDMT_* aliases) on top of the CUDA kernels.
//
// Replaces the pthread worker pools of
//   /root/reference/lib/lz4-mt_compress.c:207-353   (pt_compress, pt_write, LZ4MT_compressCCtx)
//   /root/reference/lib/lz4-mt_decompress.c:165-567 (pt_read, pt_decompress, pt_write, LZ4MT_decompressDCtx)
//   /root/reference/lib/zstd-mt_compress.c:177-392  and  lib/zstd-mt_decompress.c:209-843
// with one software pipeline per call:
//
//   reader thread  : fn_read -> pinned staging slot (B chunks / frames per slot)
//   submit (caller): H2D -> kernels -> D2H of the size table, one CUDA stream per slot,
//                    slots dealt round-robin over the GPUs named by ZSTDMT_GPUS
//   writer thread  : waits for the slot's event, D2H of the used bytes, fn_write strictly in
//                    frame order (the pt_write rule, lz4-mt_compress.c:186-202)
//
// Callback contract kept: reads never overlap reads, writes never overlap writes, a read and a
// write may overlap (as with the reference's read_mutex / write_mutex).  No CPU codec fallback:
// if the CUDA runtime or a kernel fails the call returns *_error_compression_library.
#ifndef _GNU_SOURCE
#define _GNU_SOURCE
#endif
#include <cuda_runtime.h>
#include <sched.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>
#include "zmt_dev.h"

namespace {

// ------------------------------------------------------------------ generic boundary types
struct GenBuffer { void* buf; size_t size; size_t allocated; };     // == LZ4MT_Buffer == ZSTDCB_Buffer
typedef int (gen_rw_fn)(void* arg, GenBuffer* b);
struct GenRdWr { gen_rw_fn* fn_read; void* arg_read; gen_rw_fn* fn_write; void* arg_write; };

enum { CODEC_LZ4 = 1, CODEC_ZSTD = 2 };
#define MT_MAGIC_SKIPPABLE 0x184D2A50u
#define LZ4F_MAGIC         0x184D2204u
#define ZSTD_MAGIC         0xFD2FB528u

// error numbering differs between the codecs (lz4-mt.h:41-53 vs zstd-mt.h:41-54)
struct ErrCodes { size_t mem, read_fail, write_fail, data_error, frame_compress, frame_decompress, param, library, canceled, init_missing; };
const ErrCodes kErrLz4  = { (size_t)-1, (size_t)-2, (size_t)-3, (size_t)-4, (size_t)-5, (size_t)-6, (size_t)-7, (size_t)-8, (size_t)-9, (size_t)-7 };
const ErrCodes kErrZstd = { (size_t)-1, (size_t)-3, (size_t)-4, (size_t)-5, (size_t)-6, (size_t)-7, (size_t)-8, (size_t)-9, (size_t)-10, (size_t)-2 };

inline uint32_t rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
inline uint64_t rd64(const uint8_t* p) { return (uint64_t)rd32(p) | ((uint64_t)rd32(p + 4) << 32); }

// callback return -> library error (mt_error, lz4-mt_compress.c:161-173: write failures also map to read_fail)
inline size_t mt_error(const ErrCodes& E, int rv)
{
    switch (rv) { case -1: return E.read_fail; case -2: return E.canceled; case -3: return E.mem; }
    return E.read_fail;
}

size_t env_size(const char* name, size_t dflt)
{
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    char* end = nullptr; unsigned long long x = strtoull(v, &end, 10);
    return (end && end != v) ? (size_t)x : dflt;
}

std::vector<int> env_devices()
{
    std::vector<int> devs;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return devs;
    const char* v = getenv("ZSTDMT_GPUS");
    if (v && *v) {
        if (!strcmp(v, "all")) { for (int i = 0; i < ndev; i++) devs.push_back(i); return devs; }
        const char* p = v;
        while (*p) {
            char* end = nullptr; long d = strtol(p, &end, 10);
            if (end == p) break;
            if (d >= 0 && d < ndev) devs.push_back((int)d);
            p = (*end == ',') ? end + 1 : end;
            if (*end != ',' && *end != 0) break;
        }
        if (!devs.empty()) return devs;
    }
    int cur = 0;
    if (cudaGetDevice(&cur) != cudaSuccess) cur = 0;
    devs.push_back(cur);
    return devs;
}

// batches submitted per device since the library was loaded (zmt_device_batches: lets a caller / test see the round-robin deal)
std::atomic<uint64_t> g_dev_batches[64];

// ------------------------------------------------------------------ NUMA placement
// The staging rings are the memcpy targets / sources of the (serialised) fn_read / fn_write callbacks and the DMA
// sources / targets of the GPU: both want them on the GPU's own NUMA node.  Linux places pages on the node of the
// thread that first touches them, so the pinned buffers are allocated with the calling thread temporarily bound to
// the CPUs of the GPU's PCIe root (/sys/bus/pci/devices/<id>/local_cpulist), and the reader / writer threads of a
// call run there too.  ZSTDMT_B200_NUMA=0 turns both off.
struct CpuSet { cpu_set_t set; bool ok = false; };

bool numa_enabled() { static int on = -1; if (on < 0) { const char* v = getenv("ZSTDMT_B200_NUMA"); on = (v && *v == '0') ? 0 : 1; } return on == 1; }

CpuSet device_local_cpus(int dev)
{
    CpuSet r; CPU_ZERO(&r.set);
    if (!numa_enabled()) return r;
    char id[32] = {0};
    if (cudaDeviceGetPCIBusId(id, (int)sizeof(id), dev) != cudaSuccess) { cudaGetLastError(); return r; }
    for (char* q = id; *q; q++) if (*q >= 'A' && *q <= 'Z') *q = (char)(*q - 'A' + 'a');
    char path[128]; snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", id);
    FILE* f = fopen(path, "r");
    if (!f) return r;
    char buf[1024] = {0};
    const bool got = fgets(buf, sizeof(buf), f) != nullptr;
    fclose(f);
    if (!got) return r;
    int n = 0;
    for (const char* q = buf; *q && *q != '\n';) {          // "0-31,64-95"
        char* end = nullptr; long a = strtol(q, &end, 10); if (end == q) break;
        long b = a; q = end;
        if (*q == '-') { b = strtol(q + 1, &end, 10); if (end == q + 1) break; q = end; }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) { if (c >= 0) { CPU_SET((int)c, &r.set); n++; } }
        if (*q == ',') q++;
    }
    // stay inside the affinity the process was given (containers, numactl)
    cpu_set_t cur; CPU_ZERO(&cur);
    if (sched_getaffinity(0, sizeof(cur), &cur) == 0) {
        cpu_set_t both; CPU_AND(&both, &cur, &r.set);
        if (CPU_COUNT(&both) == 0) return r;
        r.set = both;
    }
    r.ok = n > 0;
    return r;
}

// binds the calling thread for the lifetime of the object (or for good with keep())
struct ScopedAffinity {
    cpu_set_t old; bool active = false;
    explicit ScopedAffinity(const CpuSet& c) {
        if (!c.ok) return;
        CPU_ZERO(&old);
        if (sched_getaffinity(0, sizeof(old), &old) != 0) return;
        active = sched_setaffinity(0, sizeof(c.set), &c.set) == 0;
    }
    ~ScopedAffinity() { if (active) sched_setaffinity(0, sizeof(old), &old); }
};

// all devices of a call on one node -> that node's CPUs, else nothing (the staging rings then live on several nodes)
CpuSet common_local_cpus(const std::vector<int>& devs)
{
    CpuSet r; CPU_ZERO(&r.set);
    for (size_t i = 0; i < devs.size(); i++) {
        const CpuSet c = device_local_cpus(devs[i]);
        if (!c.ok) return CpuSet();
        if (i == 0) r = c; else if (!CPU_EQUAL(&r.set, &c.set)) return CpuSet();
    }
    return r;
}

// The pipeline switches the calling thread's current CUDA device while it deals batches over ZSTDMT_GPUS; a drop-in
// library must hand the thread back as it found it (a torch / CUDA caller keeps its own notion of the current device).
struct DeviceRestore {
    int prev = -1;
    DeviceRestore() { if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; } }
    ~DeviceRestore() { if (prev >= 0) cudaSetDevice(prev); }
};

// ------------------------------------------------------------------ optional stage timing (ZSTDMT_B200_TRACE=1)
inline bool trace_on() { static int on = -1; if (on < 0) on = getenv("ZSTDMT_B200_TRACE") ? 1 : 0; return on == 1; }
inline double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// seconds per stage of one call: inside callbacks / waiting for a slot / the zstd host block scan / waiting for the device
struct Clocks { double rd_total = 0, rd_cb = 0, rd_scan = 0, rd_wait = 0, sub_enqueue = 0, sub_wait = 0, wr_gpu = 0, wr_cb = 0, wr_wait = 0; };

// adds its own lifetime to `acc`; the clock is only read under ZSTDMT_B200_TRACE=1
struct Timed {
    double* acc; double t0;
    explicit Timed(double& a) : acc(trace_on() ? &a : nullptr), t0(acc ? now() : 0) {}
    ~Timed() { if (acc) *acc += now() - t0; }
};

// ------------------------------------------------------------------ device codec table
struct CodecOps {
    size_t   (*c_work)(uint32_t nchunks, uint32_t chunk);
    uint64_t (*c_bound)(uint32_t nchunks, uint32_t chunk);
    int      (*compress)(const void*, uint64_t, uint32_t, const uint32_t*, uint32_t, void*, void*, uint64_t*, void*);
};

const CodecOps* codec_ops(int codec)
{
    static const CodecOps lz4 = { zmt_lz4c_workspace_bytes, zmt_lz4c_out_bound, zmt_lz4_compress_device };
    static const CodecOps zstd = { zmt_zstdc_workspace_bytes, zmt_zstdc_out_bound, zmt_zstd_compress_device };
    return codec == CODEC_LZ4 ? &lz4 : &zstd;
}

// ------------------------------------------------------------------ batch tables
// One entry per chunk (compress) or frame (decompress); every field means the same in both directions and codecs.
// Layout (cap entries): u64 frame_off, out_off, out_size, expect [cap+1] | u32 frame_len, frame_flags, status [cap] | u32 first_blk [cap+1]
struct Tables {
    uint64_t *frame_off, *out_off;    // the frame's 12-byte header in the slot's input (decompress) / its output; out_off[n] = total
    uint64_t *out_size, *expect;      // bytes the device decoded / zstd: header content size, ~0 when that is only a bound
    uint32_t *frame_len, *frame_flags;// input bytes (chunk / frame payload) / zstd: scan flags (sequential pass, checksum, no size)
    uint32_t *status, *first_blk;     // ZMT_ST_* of the frame / zstd: its first block descriptor; first_blk[n] = total
};
inline size_t tables_bytes(size_t cap) { return 4 * (cap + 1) * 8 + 3 * cap * 4 + (cap + 1) * 4 + 64; }
inline Tables tables_at(uint8_t* base, size_t cap)
{
    Tables t;
    t.frame_off = (uint64_t*)base; t.out_off = t.frame_off + cap + 1; t.out_size = t.out_off + cap + 1; t.expect = t.out_size + cap + 1;
    t.frame_len = (uint32_t*)(t.expect + cap + 1); t.frame_flags = t.frame_len + cap; t.status = t.frame_flags + cap; t.first_blk = t.status + cap;
    return t;
}

// lz4 decode block table: every frame owns max(1, ceil(out / 64 KiB)) slots
inline uint32_t lz4_block_slots(uint64_t out_bytes) { const uint64_t nb = (out_bytes + 65535) / 65536; return nb ? (uint32_t)nb : 1; }
inline uint32_t lz4_slot_cap(size_t out_cap, size_t tab_cap) { return (uint32_t)(out_cap / 65536 + tab_cap + 1); }

// ------------------------------------------------------------------ staging slots
struct SlotCaps {
    size_t in = 0, out = 0, work = 0, tab = 0;   // bytes of input, output and workspace; entries of the batch tables
    uint32_t blk = 0;                            // zstd decompress: block descriptors
    uint64_t scr = 0;                            // zstd decompress: entropy scratch bytes the workspace was sized for
};

struct Slot {
    int dev = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev = nullptr, evp[2] = { nullptr, nullptr };       // evp: decompress writer, output pieces in flight
    uint8_t *h_in = nullptr, *h_out = nullptr, *d_in = nullptr, *d_out = nullptr, *d_work = nullptr;
    uint8_t *h_tab = nullptr, *d_tab = nullptr; size_t tab_bytes = 0;      // batch tables: pinned host mirror + device copy
    uint8_t *h_blk = nullptr, *d_blk = nullptr;                             // zstd block descriptors built by the reader
    SlotCaps cap;
    bool ok = false;
    bool host_alias = false;     // h_in / h_out are borrowed from another slot of the same context (never freed here)
    // batch contents
    uint32_t n = 0;              // chunks / frames in this batch
    uint32_t nslots = 1;         // lz4 decompress: block-table slots of this batch (sum of lz4_block_slots over frames)
    uint32_t nblk = 0;           // zstd decompress: block descriptors of this batch
    size_t in_used = 0, out_used = 0;
    int state = 0;               // 0 free, 1 filled, 2 submitted
};

void slot_free_raw(Slot& s)
{
    cudaSetDevice(s.dev);
    if (s.stream) cudaStreamSynchronize(s.stream);
    for (uint8_t* p : { s.h_in, s.h_out, s.h_tab, s.h_blk }) if (p) cudaFreeHost(p);
    for (uint8_t* p : { s.d_in, s.d_out, s.d_work, s.d_tab, s.d_blk }) if (p) cudaFree(p);
    for (cudaEvent_t e : { s.ev, s.evp[0], s.evp[1] }) if (e) cudaEventDestroy(e);
    if (s.stream) cudaStreamDestroy(s.stream);
    s = Slot();
}

// Process-wide pool of staging slots: pinned allocations cost ~0.1 s per context otherwise (the reference's
// malloc'd buffers are free by comparison).  Slots go back to the pool when a context is freed and are
// reused by the next context that needs the same device and no larger capacities.
std::mutex g_pool_mu;
std::vector<Slot> g_pool;
const size_t kPoolMax = 16;

// Takes a slot of at least `want` (the same table capacity) on `dev` from the pool, or allocates one.  With a
// `host_owner` the slot borrows that slot's pinned staging buffers and has only its device side (a call over more
// devices than it keeps batches in flight: the host ring stays 4 x 8 MiB — cache-resident for the callbacks' memcpy —
// while every device has its own device-side buffers).
bool slot_acquire(Slot& s, int dev, const SlotCaps& want, const Slot* host_owner)
{
    const bool own_host = host_owner == nullptr;
    bool found = false;
    {
        std::lock_guard<std::mutex> g(g_pool_mu);
        for (size_t i = 0; i < g_pool.size() && !found; i++) {
            const Slot& c = g_pool[i];
            if (c.dev == dev && (c.h_in != nullptr) == own_host && c.cap.in >= want.in && c.cap.out >= want.out && c.cap.work >= want.work &&
                c.cap.blk >= want.blk && c.cap.tab == want.tab) {
                s = c; g_pool.erase(g_pool.begin() + (long)i); found = true;
            }
        }
    }
    if (!found) {
        s = Slot(); s.dev = dev;
        if (cudaSetDevice(dev) != cudaSuccess) return false;
        const ScopedAffinity bind(own_host ? device_local_cpus(dev) : CpuSet());     // first touch of the pinned rings happens on the GPU's node
        const size_t blk_bytes = (size_t)want.blk * zmt_zstd_blk_desc_bytes();
        s.tab_bytes = tables_bytes(want.tab);
        bool ok = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming) == cudaSuccess;
        for (int k = 0; k < 2; k++) ok = ok && cudaEventCreateWithFlags(&s.evp[k], cudaEventDisableTiming) == cudaSuccess;
        if (own_host) {
            ok = ok && cudaHostAlloc((void**)&s.h_in, want.in + 64, cudaHostAllocPortable) == cudaSuccess;
            ok = ok && cudaHostAlloc((void**)&s.h_out, want.out + 64, cudaHostAllocPortable) == cudaSuccess;
        }
        ok = ok && cudaMalloc((void**)&s.d_in, want.in + 256) == cudaSuccess;
        ok = ok && cudaMalloc((void**)&s.d_out, want.out + 256) == cudaSuccess;
        ok = ok && cudaMalloc((void**)&s.d_work, want.work + 256) == cudaSuccess;
        ok = ok && cudaHostAlloc((void**)&s.h_tab, s.tab_bytes, cudaHostAllocPortable) == cudaSuccess;
        ok = ok && cudaMalloc((void**)&s.d_tab, s.tab_bytes) == cudaSuccess;
        if (want.blk) {
            ok = ok && cudaHostAlloc((void**)&s.h_blk, blk_bytes, cudaHostAllocPortable) == cudaSuccess;
            ok = ok && cudaMalloc((void**)&s.d_blk, blk_bytes) == cudaSuccess;
        }
        s.cap = want; s.ok = ok;
        if (!ok) { cudaGetLastError(); slot_free_raw(s); return false; }
    }
    s.cap.scr = want.scr;              // what the caller sized the workspace for
    s.state = 0; s.n = 0; s.in_used = s.out_used = 0;
    if (!own_host) { s.h_in = host_owner->h_in; s.h_out = host_owner->h_out; s.host_alias = true; }
    return true;
}

// Back to the pool (a borrower without the owner's buffers, as a device-only slot), or freed.
void slot_release(Slot& s)
{
    if (s.host_alias) { s.h_in = nullptr; s.h_out = nullptr; s.host_alias = false; }
    if (s.ok) {
        cudaSetDevice(s.dev);
        if (s.stream) cudaStreamSynchronize(s.stream);
        std::lock_guard<std::mutex> g(g_pool_mu);
        if (g_pool.size() < kPoolMax && !getenv("ZSTDMT_B200_NO_POOL")) { g_pool.push_back(s); s = Slot(); return; }
    }
    slot_free_raw(s);
}

// ------------------------------------------------------------------ pipeline state shared by the 3 threads
struct Pipe {
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Slot> slots;
    size_t fill_seq = 0, submit_seq = 0, write_seq = 0;
    bool reader_done = false;
    size_t error = 0;                 // first error wins
    Clocks clk;
    void fail(size_t e) { std::lock_guard<std::mutex> g(mu); if (!error) error = e; cv.notify_all(); }
};

struct Ctx {
    int codec = 0, level = 0, threads = 0;
    size_t inputsize = 0;
    size_t insize = 0, outsize = 0, frames = 0, curframe = 0;
    bool is_comp = false;
    std::vector<int> devs;
    Pipe pipe;
    size_t lib_errcode = 0;
    const ErrCodes* E = nullptr;
};

void ctx_release_slots(Ctx* c)
{
    for (auto& s : c->pipe.slots) if (s.ok && s.host_alias) slot_release(s);      // borrowers before the owners of the host buffers
    for (auto& s : c->pipe.slots) if (s.ok) slot_release(s);
    c->pipe.slots.clear();
}

// the devices of a context, chosen on its first call (ZSTDMT_GPUS)
bool ctx_devices(Ctx* c)
{
    if (c->pipe.slots.empty()) c->devs = env_devices();
    if (c->devs.empty()) { c->lib_errcode = ZMT_ST_CUDA; return false; }
    return true;
}

// pinned staging slots (batches in flight) of a call: one per host thread asked for, 2..4
size_t host_slots(const Ctx* c) { return c->threads >= 4 ? 4 : c->threads >= 3 ? 3 : 2; }

// a frame status as the call's error: a frame cut short is "could not decompress frame", anything else the library's
size_t status_error(Ctx* c, uint32_t st)
{
    c->lib_errcode = st;
    return (st == ZMT_ST_TRUNCATED || st == ZMT_ST_TRAILING) ? c->E->frame_decompress : c->E->library;
}

// reads exactly `want` bytes unless EOF; returns 0 ok / error; *got = delivered
size_t read_some(Ctx* c, GenRdWr* rw, void* dst, size_t want, size_t* got)
{
    GenBuffer b; b.buf = dst; b.size = want; b.allocated = want;
    int rv;
    { const Timed t(c->pipe.clk.rd_cb); rv = rw->fn_read(rw->arg_read, &b); }
    if (rv != 0) return mt_error(*c->E, rv);
    if (b.size > want) return c->E->read_fail;
    *got = b.size; return 0;
}

size_t write_all(Ctx* c, GenRdWr* rw, void* src, size_t n)
{
    GenBuffer b; b.buf = src; b.size = n; b.allocated = n;
    int rv;
    { const Timed t(c->pipe.clk.wr_cb); rv = rw->fn_write(rw->arg_write, &b); }
    if (rv != 0) return mt_error(*c->E, rv);
    c->outsize += b.size;
    return 0;
}

// ------------------------------------------------------------------ the pipeline
// One call over c->pipe.slots, batch q in slot q % N:
//   fill(slot, last)  reader thread, every fn_read call; puts slot.n > 0 items into the slot, or 0 at the end of the
//                     input; sets `last` when the input ended behind this batch
//   submit(slot)      calling thread: H2D, kernels, D2H of the tables, event slot.ev recorded
//   drain(slot)       writer thread, after slot.ev: every fn_write call, strictly in order
// Each returns 0 or the call's error; the first error stops all three.  Batch q + in_flight is not filled before batch
// q is written (slots that share their host buffers).  Reads never overlap reads, writes never overlap writes.
template <class Fill, class Submit, class Drain>
size_t run_pipeline(Ctx* c, size_t in_flight, Fill fill, Submit submit, Drain drain)
{
    Pipe& P = c->pipe;
    const size_t N = P.slots.size();
    const double slot_mib = (double)P.slots[0].cap.in / (1 << 20);
    P.fill_seq = P.submit_seq = P.write_seq = 0; P.reader_done = false; P.error = 0; P.clk = Clocks();
    for (auto& s : P.slots) s.state = 0;

    // the slot of sequence number `seq` once it is in `state`; nullptr on an error or when the reader has ended before it
    auto await = [&](const size_t& seq, int state, double& clk) -> Slot* {
        const Timed t(clk);
        std::unique_lock<std::mutex> lk(P.mu);
        Slot* s = &P.slots[seq % N];
        P.cv.wait(lk, [&] {
            if (P.error) return true;
            if (state == 0) return s->state == 0 && P.fill_seq - P.write_seq < in_flight;
            return s->state == state || (P.reader_done && seq == P.fill_seq);
        });
        return (P.error || s->state != state) ? nullptr : s;
    };
    auto advance = [&](Slot* s, int state, size_t& seq) {
        { std::lock_guard<std::mutex> g(P.mu); s->state = state; seq++; }
        P.cv.notify_all();
    };

    const CpuSet host_cpus = common_local_cpus(c->devs);
    std::thread reader([&]() {
        const ScopedAffinity bind(host_cpus);
        {
            const Timed t(P.clk.rd_total);
            for (bool last = false; !last;) {
                Slot* s = await(P.fill_seq, 0, P.clk.rd_wait);
                if (!s) break;
                const size_t e = fill(*s, last);
                if (e) { P.fail(e); break; }
                if (s->n == 0) break;
                advance(s, 1, P.fill_seq);
            }
        }
        { std::lock_guard<std::mutex> g(P.mu); P.reader_done = true; }
        P.cv.notify_all();
    });
    std::thread writer([&]() {
        const ScopedAffinity bind(host_cpus);
        for (;;) {
            Slot* s = await(P.write_seq, 2, P.clk.wr_wait);
            if (!s) break;
            cudaSetDevice(s->dev);
            cudaError_t ce;
            { const Timed t(P.clk.wr_gpu); ce = cudaEventSynchronize(s->ev); }
            const size_t e = ce == cudaSuccess ? drain(*s) : (c->lib_errcode = ZMT_ST_CUDA, c->E->library);
            if (e) { P.fail(e); break; }
            advance(s, 0, P.write_seq);
        }
    });
    for (;;) {
        Slot* s = await(P.submit_seq, 1, P.clk.sub_wait);
        if (!s) break;
        size_t e;
        { const Timed t(P.clk.sub_enqueue); cudaSetDevice(s->dev); e = submit(*s); }
        if (s->dev >= 0 && s->dev < 64) g_dev_batches[s->dev]++;
        if (e) { P.fail(e); break; }
        advance(s, 2, P.submit_seq);
    }
    reader.join(); writer.join();
    for (auto& s : P.slots) if (s.ok) { cudaSetDevice(s.dev); cudaStreamSynchronize(s.stream); }
    if (trace_on()) {
        const Clocks& k = P.clk;
        fprintf(stderr, "[zstdmt_b200] %s: reader total %.3fs cb %.3fs scan %.3fs wait %.3fs | submit enqueue %.3fs wait %.3fs | "
                        "writer gpu-wait %.3fs cb %.3fs wait %.3fs | slots %zu x %.1f MiB\n", c->is_comp ? "compress" : "decompress",
                k.rd_total, k.rd_cb, k.rd_scan, k.rd_wait, k.sub_enqueue, k.sub_wait, k.wr_gpu, k.wr_cb, k.wr_wait, N, slot_mib);
    }
    return P.error;
}

// ------------------------------------------------------------------ compression
size_t compress_run(Ctx* c, GenRdWr* rw)
{
    const DeviceRestore restore_device;
    const ErrCodes& E = *c->E;
    const CodecOps* ops = codec_ops(c->codec);
    Pipe& P = c->pipe;
    const size_t chunk = c->inputsize;
    // Slots in flight: the call is bound by the serialised callbacks (one memcpy stream); a GPU turns a batch around in a
    // fraction of the time the reader needs to fill the next one, so more devices do not need more batches in flight.
    // Measured on the 2-socket Xeon hosts of the B200 pool (one GPU, 4 GiB, GB/s end to end): 4 slots x 8 MiB 18.2
    // (the default), 4 x 4 MiB 15.8, 4 x 16 MiB 14.4, 8 x 8 MiB 13.7, 8 x 4 MiB 9.9, 16 x 2 MiB 5.2: a ring that outgrows the
    // last-level cache slows the callbacks' memcpy, and small batches pay the per-batch launch + copy latency.  A call over
    // more devices than host slots therefore shares the host ring: every device gets device-side slots, and those beyond
    // the first `base_slots` borrow the pinned buffers of slot i % base_slots (ZSTDMT_B200_NO_RING_SHARE=1: every slot its
    // own, 8 x 8 MiB over 8 devices, 14.3 GB/s).
    if (!ctx_devices(c)) return E.library;
    const size_t base_slots = host_slots(c);
    size_t nsl = env_size("ZSTDMT_B200_SLOTS", base_slots > c->devs.size() ? base_slots : c->devs.size());
    if (nsl < 2) nsl = 2;
    if (nsl < c->devs.size()) nsl = c->devs.size();
    if (nsl > 64) nsl = 64;
    const bool no_alias = getenv("ZSTDMT_B200_NO_RING_SHARE") != nullptr;
    if (!no_alias && nsl > base_slots) nsl = (nsl + base_slots - 1) / base_slots * base_slots;   // batch q uses host buffer q % base_slots: needs base_slots | slots
    size_t B = (env_size("ZSTDMT_B200_BATCH_MB", 8) << 20) / chunk;
    if (B < 1) B = 1;
    if (B > 65536) B = 65536;

    if (P.slots.empty()) {
        P.slots.resize(nsl);
        SlotCaps caps;
        caps.in = B * chunk; caps.out = (size_t)ops->c_bound((uint32_t)B, (uint32_t)chunk); caps.work = ops->c_work((uint32_t)B, (uint32_t)chunk); caps.tab = B;
        for (size_t i = 0; i < P.slots.size(); i++) {
            const Slot* owner = (i < base_slots || no_alias) ? nullptr : &P.slots[i % base_slots];
            if (!slot_acquire(P.slots[i], c->devs[i % c->devs.size()], caps, owner)) { ctx_release_slots(c); return E.mem; }
        }
    }
    const size_t N = P.slots.size();
    const size_t in_flight = (N > base_slots && !no_alias) ? base_slots : N;

    // reader: B chunks per slot (pt_compress read section, lz4-mt_compress.c:255-277)
    size_t frames_read = 0;
    auto fill = [&](Slot& s, bool& last) -> size_t {
        const Tables T = tables_at(s.h_tab, s.cap.tab);
        uint32_t n = 0; size_t got_bytes = 0;
        while (n < B) {
            size_t got = 0;
            const size_t e = read_some(c, rw, s.h_in + (size_t)n * chunk, chunk, &got);
            if (e) return e;
            if (got == 0 && frames_read > 0) { last = true; break; }
            T.frame_len[n] = (uint32_t)got; got_bytes += got; frames_read++; n++;
        }
        s.n = n; s.in_used = got_bytes;
        c->insize += got_bytes; c->frames += n;
        return 0;
    };
    auto submit = [&](Slot& s) -> size_t {
        const Tables Th = tables_at(s.h_tab, s.cap.tab), Td = tables_at(s.d_tab, s.cap.tab);
        bool full = true;
        for (uint32_t i = 0; i < s.n; i++) if (Th.frame_len[i] != chunk) { full = false; break; }
        cudaError_t ce = cudaSuccess;
        if (full) ce = cudaMemcpyAsync(s.d_in, s.h_in, (size_t)s.n * chunk, cudaMemcpyHostToDevice, s.stream);
        else for (uint32_t i = 0; i < s.n && ce == cudaSuccess; i++)
            if (Th.frame_len[i]) ce = cudaMemcpyAsync(s.d_in + (size_t)i * chunk, s.h_in + (size_t)i * chunk, Th.frame_len[i], cudaMemcpyHostToDevice, s.stream);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(Td.frame_len, Th.frame_len, (size_t)s.n * 4, cudaMemcpyHostToDevice, s.stream);
        int st = ZMT_ST_CUDA;
        if (ce == cudaSuccess) st = ops->compress(s.d_in, 0, (uint32_t)chunk, Td.frame_len, s.n, s.d_work, s.d_out, Td.out_off, s.stream);
        if (st == ZMT_ST_OK) {
            ce = cudaMemcpyAsync(Th.out_off, Td.out_off, ((size_t)s.n + 1) * 8, cudaMemcpyDeviceToHost, s.stream);
            if (ce == cudaSuccess) ce = cudaEventRecord(s.ev, s.stream);
            if (ce != cudaSuccess) st = ZMT_ST_CUDA;
        }
        if (st != ZMT_ST_OK) { c->lib_errcode = (size_t)st; return E.library; }
        return 0;
    };
    // writer: one fn_write per frame, in order (pt_write, lz4-mt_compress.c:178-205)
    auto drain = [&](Slot& s) -> size_t {
        const Tables T = tables_at(s.h_tab, s.cap.tab);
        const uint64_t total = T.out_off[s.n];
        if (total > s.cap.out) { c->lib_errcode = ZMT_ST_DST_SMALL; return E.library; }
        cudaError_t ce;
        {
            const Timed t(P.clk.wr_gpu);
            ce = cudaMemcpyAsync(s.h_out, s.d_out, total, cudaMemcpyDeviceToHost, s.stream);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(s.stream);
        }
        if (ce != cudaSuccess) { c->lib_errcode = ZMT_ST_CUDA; return E.library; }
        for (uint32_t i = 0; i < s.n; i++) {
            const size_t e = write_all(c, rw, s.h_out + T.out_off[i], (size_t)(T.out_off[i + 1] - T.out_off[i]));
            if (e) return e;
            c->curframe++;
        }
        return 0;
    };
    return run_pipeline(c, in_flight, fill, submit, drain);
}

// ------------------------------------------------------------------ decompression
// Walks the block headers of the LZ4 frame p[0..n) (magic, FLG and BD already read): *bound = the sum of the blocks'
// output bounds (each block <= blockMaxSize).  Returns the offset just past the end mark, 0 if the frame runs past n.
size_t lz4f_walk_blocks(const uint8_t* p, size_t n, uint64_t* bound)
{
    const uint32_t flg = p[4], id = (p[5] >> 4) & 7;
    const uint64_t blkmax = 1ull << (8 + 2 * id);
    size_t q = 4 + 2 + ((flg & 8) ? 8 : 0) + ((flg & 1) ? 4 : 0) + 1;
    *bound = 0;
    for (;;) {
        if (q + 4 > n) return 0;
        const uint32_t bh = rd32(p + q); q += 4;
        if (bh == 0) return q;
        const uint32_t bs = bh & 0x7FFFFFFFu;
        *bound += (bh & 0x80000000u) ? bs : blkmax;
        q += (size_t)bs + ((flg & 0x10) ? 4 : 0);
    }
}

// Output size of one payload, from its own header (pt_decompress sizes the buffer from
// LE64 @ payload+6, lz4-mt_decompress.c:329-335).  Returns false if the header is unusable.
bool lz4f_out_size(const uint8_t* p, size_t n, uint64_t* out)
{
    if (n < 7 || rd32(p) != LZ4F_MAGIC) { *out = 0; return true; }     // the device decoder reports the precise status
    const uint32_t flg = p[4], bd = p[5];
    if (flg & 0x08) {
        if (n < 15) return false;
        // untrusted field: LZ4 cannot expand by more than 255x, anything larger is a corrupt header (the reference
        // fails its malloc there); without this bound a huge value would wrap the running output offsets
        const uint64_t v = rd64(p + 6);
        if (v > (uint64_t)n * 255 + 65536) return false;
        *out = v; return true;
    }
    if (((bd >> 4) & 7) < 4) return false;
    lz4f_walk_blocks(p, n, out);                                         // no content-size field: the block walk bounds it
    return true;
}

// zstd / lz4 decode of one batch whose tables are on the device
int launch_decode(bool is_zstd, const void* d_in, uint64_t in_bytes, const void* d_blk, uint32_t nblk, const Tables& Td, uint32_t n,
                  uint32_t nslots, void* d_out, void* d_work, cudaStream_t st)
{
    return is_zstd ? zmt_zstd_decompress_device(d_in, d_blk, nblk, Td.first_blk, Td.expect, Td.frame_flags, n, d_out, Td.out_off, Td.out_size, Td.status, d_work, st)
                   : zmt_lz4_decompress_device(d_in, in_bytes, Td.frame_off, Td.frame_len, n, nslots, d_out, Td.out_off, Td.out_size, Td.status, d_work, st);
}

size_t decode_work_bytes(bool is_zstd, const SlotCaps& k)
{
    return is_zstd ? zmt_zstdd_workspace_bytes((uint32_t)k.tab, k.blk, k.scr) : zmt_lz4d_workspace_bytes((uint32_t)k.tab, lz4_slot_cap(k.out, k.tab), k.in);
}

// ------------------------------------------------------------------ plain (unframed) single streams
// What the reference routes to st_decompress (lz4-mt_decompress.c:391-483, zstd-mt_decompress.c:552-687): an ordinary
// .lz4 / .zst file, i.e. codec frames back to back without the 12-byte size headers.  Frame lengths are only known after
// walking the block headers, so the host reads ahead, cuts the bytes it holds into complete frames, and decodes them in
// batches of at most ~kPlainBatch input bytes with the same GPU kernels; the consumed bytes are dropped before the next
// read, so memory is bounded by the batch size or by the largest single frame, whichever is larger (the reference streams
// through two fixed buffers; a frame here must fit in host and device memory as a whole).  `first`/`have` = the bytes
// already consumed by the stream-type sniffing.
struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    bool need(size_t n) {                                   // grow-only
        if (n <= cap && p) return true;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        const size_t want = n + n / 4 + 4096;
        if (cudaMalloc(&p, want) != cudaSuccess) { cudaGetLastError(); if (cudaMalloc(&p, n ? n : 1) != cudaSuccess) { cudaGetLastError(); p = nullptr; return false; } cap = n; return true; }
        cap = want; return true;
    }
};

size_t decompress_single_stream(Ctx* c, GenRdWr* rw, const uint8_t* first, size_t have)
{
    const ErrCodes& E = *c->E;
    const bool is_zstd = c->codec == CODEC_ZSTD;
    const size_t kPlainBatch = env_size("ZSTDMT_B200_PLAIN_MB", 64) << 20;
    const size_t piece = c->inputsize < (64u << 10) ? (size_t)1 << 20 : c->inputsize;
    const size_t dsz = zmt_zstd_blk_desc_bytes();
    std::vector<uint8_t> in(12, 0);                         // 12 pad bytes: the LZ4 kernel addresses a frame as base + off + 12
    in.insert(in.end(), first, first + have);
    bool eof = false;
    size_t pos = 0;                                         // parse position inside in[12..]
    const std::vector<int> devs = env_devices();
    if (devs.empty() || cudaSetDevice(devs[0]) != cudaSuccess) { c->lib_errcode = ZMT_ST_CUDA; return E.library; }
    DevBuf d_in, d_out, d_tab, d_blk, d_work;
    cudaStream_t st = nullptr;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) != cudaSuccess) { c->lib_errcode = ZMT_ST_CUDA; return E.library; }
    struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } guard{st};
    std::vector<uint8_t> out, blocks, h_tab;
    std::vector<uint64_t> foff, ooff, expect; std::vector<uint32_t> fcs, first_blk, fflags;
    c->insize = have;

    for (;;) {
        // ---- cut complete frames out of what we hold, up to one batch
        foff.clear(); ooff.assign(1, 0); expect.clear(); fcs.clear(); first_blk.assign(1, 0); fflags.clear();
        uint32_t nblk = 0, nslots = 0; uint64_t scratch = 0;
        const size_t batch_start = pos;
        bool need_more = false;
        while (!need_more) {
            const uint8_t* s = in.data() + 12; const size_t n = in.size() - 12;
            if (pos >= n) { need_more = !eof; break; }
            if (!foff.empty() && pos - batch_start >= kPlainBatch) break;
            if (n - pos < 4) { if (eof) return E.data_error; need_more = true; break; }
            const uint32_t magic = rd32(s + pos);
            if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {          // skippable frame: magic, LE32 size, payload
                if (n - pos < 8 || n - pos - 8 < rd32(s + pos + 4)) { if (eof) return E.data_error; need_more = true; break; }
                pos += 8 + (size_t)rd32(s + pos + 4); continue;
            }
            if (!is_zstd) {
                if (magic != LZ4F_MAGIC) return E.data_error;
                if (n - pos < 7) { if (eof) return E.data_error; need_more = true; break; }
                const uint32_t flg = s[pos + 4], id = (s[pos + 5] >> 4) & 7;
                if ((flg >> 6) != 1 || id < 4) { c->lib_errcode = ZMT_ST_BAD_HEADER; return E.library; }
                uint64_t bound = 0;
                size_t q = lz4f_walk_blocks(s + pos, n - pos, &bound);
                if (q && (flg & 4)) q += 4;
                if (!q || q > n - pos) { if (eof) return status_error(c, ZMT_ST_TRUNCATED); need_more = true; break; }
                uint64_t osz = bound;
                if (flg & 8) { osz = rd64(s + pos + 6); if (osz > bound) { c->lib_errcode = ZMT_ST_CONTENT_SIZE; return E.library; } }    // untrusted field, bounded by the block walk
                foff.push_back(pos); fcs.push_back((uint32_t)q); ooff.push_back(ooff.back() + osz);
                nslots += lz4_block_slots(osz);
                pos += q;
            } else {
                if (magic < 0xFD2FB522u || magic > 0xFD2FB528u) return E.data_error;
                uint64_t cs = 0; uint32_t fl = 0; size_t used = 0;
                const uint32_t nblk0 = nblk; const uint64_t scr0 = scratch;
                int zr;
                for (;;) {
                    nblk = nblk0; scratch = scr0;
                    zr = zmt_zstd_scan_frame_host2(s + pos, n - pos, 12 + pos, (uint32_t)foff.size(), blocks.data(), &nblk, (uint32_t)(blocks.size() / dsz), &scratch, &cs, &fl, &used);
                    if (zr != ZMT_ST_DST_SMALL) break;
                    blocks.resize(blocks.size() * 2 + 4096 * dsz);            // block table full: grow and rescan this frame
                }
                if (zr == ZMT_ST_TRUNCATED && !eof) { nblk = nblk0; scratch = scr0; need_more = true; break; }
                if (zr != ZMT_ST_OK) return status_error(c, zr);
                foff.push_back(pos); expect.push_back((fl & 4u) ? ~0ull : cs); fflags.push_back(fl); first_blk.push_back(nblk); ooff.push_back(ooff.back() + cs);
                pos += used;
            }
        }
        const uint32_t nf = (uint32_t)foff.size();
        if (nf == 0) {
            if (!need_more) break;                                            // EOF, everything consumed
        } else {
            // ---- decode this batch
            const uint64_t total = ooff.back();
            const size_t in_bytes = pos + 12;                                   // frames address the buffer from its 12-byte pad
            const size_t tab_bytes = tables_bytes(nf);
            h_tab.resize(tab_bytes);
            const Tables T = tables_at(h_tab.data(), nf);
            for (uint32_t i = 0; i < nf; i++) {
                T.frame_off[i] = foff[i]; T.out_off[i] = ooff[i];
                if (is_zstd) { T.expect[i] = expect[i]; T.frame_flags[i] = fflags[i]; T.first_blk[i] = first_blk[i]; } else T.frame_len[i] = fcs[i];
            }
            T.out_off[nf] = total; if (is_zstd) T.first_blk[nf] = nblk;
            const size_t wk = is_zstd ? zmt_zstdd_workspace_bytes(nf, nblk, scratch) : zmt_lz4d_workspace_bytes(nf, nslots, in_bytes);
            if (!d_in.need(in_bytes + 256) || !d_out.need(total + 256) || !d_tab.need(tab_bytes) || !d_work.need(wk) || (is_zstd && !d_blk.need((size_t)nblk * dsz + 16))) return E.mem;
            const Tables Td = tables_at((uint8_t*)d_tab.p, nf);
            // only the bytes of this batch travel (the device addresses them at their buffer offsets)
            const size_t lo = 12 + batch_start, hi = in_bytes;
            cudaMemcpyAsync((uint8_t*)d_in.p + lo, in.data() + lo, hi - lo, cudaMemcpyHostToDevice, st);
            cudaMemcpyAsync(d_tab.p, h_tab.data(), tab_bytes, cudaMemcpyHostToDevice, st);
            if (is_zstd && nblk) cudaMemcpyAsync(d_blk.p, blocks.data(), (size_t)nblk * dsz, cudaMemcpyHostToDevice, st);
            const int rc = launch_decode(is_zstd, d_in.p, in_bytes, d_blk.p, nblk, Td, nf, nslots, d_out.p, d_work.p, st);
            out.resize(total ? total : 1);
            std::vector<uint32_t> status(nf); std::vector<uint64_t> osz(nf);
            cudaError_t ce = cudaSuccess;
            if (rc == ZMT_ST_OK) {
                if (total) ce = cudaMemcpyAsync(out.data(), d_out.p, total, cudaMemcpyDeviceToHost, st);
                if (ce == cudaSuccess) ce = cudaMemcpyAsync(status.data(), Td.status, (size_t)nf * 4, cudaMemcpyDeviceToHost, st);
                if (ce == cudaSuccess) ce = cudaMemcpyAsync(osz.data(), Td.out_size, (size_t)nf * 8, cudaMemcpyDeviceToHost, st);
                if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);
            }
            if (rc != ZMT_ST_OK || ce != cudaSuccess) { cudaGetLastError(); c->lib_errcode = ZMT_ST_CUDA; return E.library; }
            for (uint32_t i = 0; i < nf; i++) {
                if (status[i] != ZMT_ST_OK) return status_error(c, status[i]);
                // frame by frame, in pieces of at most `piece` bytes (st_decompress writes as it goes)
                for (uint64_t o = 0; o < osz[i];) {
                    const size_t len = (size_t)((osz[i] - o) < piece ? (osz[i] - o) : piece);
                    const size_t e = write_all(c, rw, out.data() + ooff[i] + o, len);
                    if (e) return e;
                    o += len;
                }
            }
            // drop what has been decoded
            in.erase(in.begin() + 12, in.begin() + 12 + (long)pos);
            pos = 0;
        }
        if (need_more) {
            // ---- read ahead: at least one more piece, up to a batch beyond the parse position
            size_t goal = in.size() + piece;
            if (goal < 12 + pos + kPlainBatch) goal = 12 + pos + kPlainBatch;
            if (in.size() - 12 - pos >= kPlainBatch) goal = in.size() + (in.size() - 12 - pos) / 2;     // one frame larger than a batch: read ahead geometrically
            while (!eof && in.size() < goal) {
                const size_t old = in.size();
                in.resize(old + piece);
                size_t got = 0;
                const size_t e = read_some(c, rw, in.data() + old, piece, &got);
                in.resize(old + got);
                if (e) return e;
                c->insize += got;
                if (got == 0) eof = true;
            }
        } else if (eof && pos >= in.size() - 12) break;
    }
    return 0;
}

// ---- framed streams: the pipeline
// What the reader has put into one decompress slot so far.
struct BatchFill {
    uint32_t n = 0, nblk = 0, nslots = 0;
    size_t in_used = 0;
    uint64_t out_used = 0, scr = 0;
    SlotCaps need;                      // after ADMIT_MOVE: what a slot holding this frame alone needs
};
enum Admit { ADMIT_APPEND, ADMIT_MOVE, ADMIT_ERROR };

// Sizes the frame (12-byte header + `len` payload bytes) at s.h_in + bf.in_used — LZ4 from its header, zstd by the host
// block scan — and appends it to the batch tables, or reports that it does not fit behind the frames already in the
// slot (ADMIT_MOVE) or that it is broken (ADMIT_ERROR, *err = the call's error).
Admit admit_frame(Ctx* c, Slot& s, BatchFill& bf, uint32_t len, size_t* err)
{
    const bool is_zstd = c->codec == CODEC_ZSTD;
    const uint8_t* p = s.h_in + bf.in_used + 12;
    uint64_t osz = 0, scr = bf.scr;
    uint32_t flags = 0, nblk = bf.nblk;
    bool fits = true;
    bf.need = SlotCaps();
    if (!is_zstd) {
        if (!lz4f_out_size(p, len, &osz)) { c->lib_errcode = ZMT_ST_BAD_HEADER; *err = c->E->library; return ADMIT_ERROR; }
    } else {
        int zr;
        { const Timed t(c->pipe.clk.rd_scan); zr = zmt_zstd_scan_frame_host(p, len, bf.in_used + 12, bf.n, s.h_blk, &nblk, s.cap.blk, &scr, &osz, &flags); }
        if (zr == ZMT_ST_DST_SMALL) { fits = false; bf.need.blk = len / 3 + 16; }       // more blocks than descriptors: every block costs >= 3 bytes
        else if (zr != ZMT_ST_OK) { *err = status_error(c, zr); return ADMIT_ERROR; }
        else if (scr > s.cap.scr) fits = false;
    }
    if (fits && osz > s.cap.out - bf.out_used) fits = false;
    if (!fits) { bf.need.in = 12 + (size_t)len; bf.need.out = osz; bf.need.scr = scr; return ADMIT_MOVE; }
    const Tables T = tables_at(s.h_tab, s.cap.tab);
    T.frame_off[bf.n] = bf.in_used; T.frame_len[bf.n] = len; T.out_off[bf.n] = bf.out_used;
    if (is_zstd) { T.first_blk[bf.n] = bf.nblk; T.expect[bf.n] = (flags & 4u) ? ~0ull : osz; T.frame_flags[bf.n] = flags; bf.nblk = nblk; bf.scr = scr; }   // flag 4: no content size in the header, osz is a bound
    else bf.nslots += lz4_block_slots(osz);
    bf.in_used += 12 + (size_t)len; bf.out_used += osz; bf.n++;
    return ADMIT_APPEND;
}

// The reader of a framed decode (pt_read, lz4-mt_decompress.c:192-281 / zstd-mt_decompress.c:209-369): frames behind
// 12-byte skippable headers, read on the reader thread into the slot of each batch.
struct FramedReader {
    Ctx* c; GenRdWr* rw; bool is_zstd;
    uint8_t first[16];                   // what the stream-type sniffing read
    bool hdr_pending = false;            // first 12-byte header already (partly) read into `first`
    size_t first_payload_have = 0;       // zstd pzstd-style: 4 payload bytes already read
    std::vector<uint8_t> carry;          // a whole frame that did not fit where it was read: it starts a batch
    size_t stat_in = 0;                  // input bytes of the batch being filled (insize counts committed batches)

    FramedReader(Ctx* c_, GenRdWr* rw_) : c(c_), rw(rw_), is_zstd(c_->codec == CODEC_ZSTD) {}
    size_t sniff(bool* framed);
    size_t fill(Slot& s, bool& last);
    size_t read_frame(Slot& s, const BatchFill& bf, uint32_t* len, bool* eof);
    size_t place(Slot& s, BatchFill& bf, uint32_t len, bool* moved);
    bool grow(Slot& s, const SlotCaps& need);
};

// Stream-type sniffing on the calling thread (LZ4MT_decompressDCtx, lz4-mt_decompress.c:503-520; ZSTDCB_decompressDCtx,
// zstd-mt_decompress.c:721-759).  A plain stream is decoded right here (*framed = false, the call's result returned).
size_t FramedReader::sniff(bool* framed)
{
    const ErrCodes& E = *c->E;
    size_t got = 0;
    *framed = false;
    if (!is_zstd) {
        size_t e = read_some(c, rw, first, 4, &got); if (e) return e;
        if (got != 4) return E.data_error;
        if (rd32(first) != MT_MAGIC_SKIPPABLE) {
            if (rd32(first) != LZ4F_MAGIC) return E.data_error;
            return decompress_single_stream(c, rw, first, 4);          // plain .lz4 stream (st_decompress, lz4-mt_decompress.c:512-520)
        }
        e = read_some(c, rw, first + 4, 8, &got); if (e) return e;
        if (got != 8) return E.read_fail;
    } else {
        size_t e = read_some(c, rw, first, 16, &got); if (e) return e;
        auto is_zstd_magic = [](const uint8_t* p) { uint32_t m = rd32(p); return m >= 0xFD2FB522u && m <= 0xFD2FB528u; };
        auto is_skip = [](const uint8_t* p) { return rd32(p) == MT_MAGIC_SKIPPABLE && rd32(p + 4) == 4; };
        if (got < 16) {
            if (got < 4 || !is_zstd_magic(first)) return E.data_error;
            if (got == 9) return 0;                                    // empty file (zstd-mt_decompress.c:735-740)
            return decompress_single_stream(c, rw, first, got);        // short plain zstd stream
        }
        c->insize += 16;
        if (is_skip(first) && is_zstd_magic(first + 12)) first_payload_have = 4;                                // pzstd style
        else if (is_zstd_magic(first) && rd32(first + 9) == MT_MAGIC_SKIPPABLE) {                                  // zstdmt style: 9-byte empty frame + 12-byte header
            // (only the magic can be tested here, as IsZstd_Skippable does, zstd-mt_decompress.c:156-159: 7 of the header's 12
            //  bytes are in hand; the size field is checked with the assembled header.  Round 1 read its 4 bytes past the buffer.)
            uint8_t tmp[12]; memcpy(tmp, first + 9, 7);
            e = read_some(c, rw, tmp + 7, 5, &got); if (e) return e;
            if (got != 5) return E.data_error;
            c->insize += 5; memcpy(first, tmp, 12);
        } else if (is_zstd_magic(first)) return decompress_single_stream(c, rw, first, 16);    // plain .zst (zstd-mt_decompress.c:747-752)
        else return E.data_error;
    }
    hdr_pending = true; *framed = true;
    return 0;
}

// One batch: frames until the slot's table is full, a frame does not fit (it starts the next batch) or the input ends.
size_t FramedReader::fill(Slot& s, bool& last)
{
    BatchFill bf;
    bool moved = false;
    stat_in = 0;
    while (bf.n < s.cap.tab && !moved) {
        uint32_t len = 0;
        if (carry.empty()) {
            const size_t e = read_frame(s, bf, &len, &last);
            if (e) return e;
            if (last) break;
        } else len = (uint32_t)(carry.size() - 12);
        const size_t e = place(s, bf, len, &moved);
        if (e) return e;
    }
    s.n = bf.n;
    if (bf.n == 0) return 0;
    const Tables T = tables_at(s.h_tab, s.cap.tab);
    T.out_off[bf.n] = bf.out_used;
    if (is_zstd) T.first_blk[bf.n] = bf.nblk;
    s.nblk = bf.nblk; s.nslots = bf.nslots; s.in_used = bf.in_used; s.out_used = (size_t)bf.out_used;
    c->insize += stat_in; c->frames += bf.n;
    return 0;
}

// The next frame of the input: read behind the frames already in the slot if it fits there, else into `carry`.
// *eof at the end of the input.
size_t FramedReader::read_frame(Slot& s, const BatchFill& bf, uint32_t* len, bool* eof)
{
    const ErrCodes& E = *c->E;
    uint8_t hdr[12]; size_t pre = 0, g = 0;
    if (hdr_pending) { memcpy(hdr, first, 12); hdr_pending = false; pre = first_payload_have; }
    else {
        const size_t e = read_some(c, rw, hdr, 12, &g);
        if (e) return e;
        if (g == 0) { *eof = true; return 0; }
        if (g != 12) return E.read_fail;
        if (rd32(hdr) != MT_MAGIC_SKIPPABLE) return E.data_error;
        if (is_zstd) stat_in += 12;
    }
    if (rd32(hdr + 4) != 4) return E.data_error;
    if (!is_zstd) stat_in += 12;
    *len = rd32(hdr + 8);
    if (*len < pre) return E.data_error;
    uint8_t* dst = s.h_in + bf.in_used;
    if (bf.in_used + 12 + *len > s.cap.in) { carry.resize(12 + (size_t)*len); dst = carry.data(); }
    memcpy(dst, hdr, 12);
    if (pre) memcpy(dst + 12, first + 12, pre);
    const size_t e = read_some(c, rw, dst + 12 + pre, *len - pre, &g);
    if (e) return e;
    if (g != *len - pre) return E.data_error;
    stat_in += g;
    return 0;
}

// Appends the frame held in `carry` (or already at s.h_in + bf.in_used when `carry` is empty) to the batch.  A frame
// that does not fit behind the others stays in `carry` for the next batch (*moved); a single frame larger than the
// slot grows the empty slot (input, output, zstd block table and entropy scratch) until it fits.
size_t FramedReader::place(Slot& s, BatchFill& bf, uint32_t len, bool* moved)
{
    const size_t flen = 12 + (size_t)len;
    for (int tries = 0;; tries++) {
        if (!carry.empty()) {
            if (bf.in_used + flen > s.cap.in) {
                if (bf.n > 0) { *moved = true; return 0; }
                SlotCaps need; need.in = flen;
                if (!grow(s, need)) return c->E->mem;
            }
            memcpy(s.h_in + bf.in_used, carry.data(), flen);
        }
        size_t e = 0;
        const Admit a = admit_frame(c, s, bf, len, &e);
        if (a == ADMIT_ERROR) return e;
        if (a == ADMIT_APPEND) { carry.clear(); return 0; }
        if (carry.empty()) carry.assign(s.h_in + bf.in_used, s.h_in + bf.in_used + flen);
        if (bf.n > 0) { *moved = true; return 0; }
        if (tries == 2 || !grow(s, bf.need)) return c->E->mem;
    }
}

// (Re)allocates the still empty slot with at least the capacities in `need`; under the pipeline's mutex because the
// writer's wait reads s.state.
bool FramedReader::grow(Slot& s, const SlotCaps& need)
{
    SlotCaps k = s.cap;
    if (need.in > k.in) k.in = need.in;
    if (need.out > k.out) k.out = need.out;
    if (need.blk > k.blk) k.blk = need.blk;
    k.scr = is_zstd ? (need.scr > 3 * (uint64_t)k.out ? need.scr : 3 * (uint64_t)k.out) : 0;
    k.work = decode_work_bytes(is_zstd, k);
    std::lock_guard<std::mutex> g(c->pipe.mu);
    const int dev = s.dev;
    slot_release(s);
    return slot_acquire(s, dev, k, nullptr);
}

// Submit of a decode batch: H2D of the frames and tables, the decoder, D2H of sizes and status (and of the whole output
// when piece_bytes is 0).
size_t decode_submit(Ctx* c, Slot& s, uint64_t piece_bytes)
{
    const bool is_zstd = c->codec == CODEC_ZSTD;
    const Tables Th = tables_at(s.h_tab, s.cap.tab), Td = tables_at(s.d_tab, s.cap.tab);
    cudaError_t ce = cudaMemcpyAsync(s.d_in, s.h_in, s.in_used, cudaMemcpyHostToDevice, s.stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(s.d_tab, s.h_tab, s.tab_bytes, cudaMemcpyHostToDevice, s.stream);
    if (ce == cudaSuccess && is_zstd && s.nblk) ce = cudaMemcpyAsync(s.d_blk, s.h_blk, (size_t)s.nblk * zmt_zstd_blk_desc_bytes(), cudaMemcpyHostToDevice, s.stream);
    int st = ZMT_ST_CUDA;
    if (ce == cudaSuccess) st = launch_decode(is_zstd, s.d_in, s.in_used, s.d_blk, s.nblk, Td, s.n, s.nslots, s.d_out, s.d_work, s.stream);
    if (st == ZMT_ST_OK) {
        if (s.out_used && piece_bytes == 0) ce = cudaMemcpyAsync(s.h_out, s.d_out, s.out_used, cudaMemcpyDeviceToHost, s.stream);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(Th.out_size, Td.out_size, (size_t)s.n * 8, cudaMemcpyDeviceToHost, s.stream);
        if (ce == cudaSuccess) ce = cudaMemcpyAsync(Th.status, Td.status, (size_t)s.n * 4, cudaMemcpyDeviceToHost, s.stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(s.ev, s.stream);
        if (ce != cudaSuccess) st = ZMT_ST_CUDA;
    }
    if (st != ZMT_ST_OK) { c->lib_errcode = (size_t)st; return c->E->library; }
    return 0;
}

// Writer of a decode batch (pt_write, lz4-mt_decompress.c:165-187): one fn_write per frame.  The decoded bytes come over
// in pieces of piece_bytes, one piece ahead of the one being written: what fn_write's memcpy reads was DMA-written
// moments ago and is still in the last-level cache, instead of a whole 64 MiB slot that was copied long before its
// first byte is used.
size_t decode_drain(Ctx* c, GenRdWr* rw, Slot& s, uint64_t piece_bytes)
{
    const Tables T = tables_at(s.h_tab, s.cap.tab);
    uint32_t issued = 0, ready = 0, piece_end[2] = { 0, 0 };     // frames [0, issued) requested, [0, ready) landed
    int np_issued = 0, np_ready = 0;                               // piece k: event evp[k & 1], frames up to piece_end[k & 1]
    auto issue_piece = [&]() -> bool {
        uint32_t j = issued; const uint64_t lo = T.out_off[j]; uint64_t hi = lo;
        while (j < s.n && hi - lo < piece_bytes) { hi = T.out_off[j] + T.out_size[j]; j++; }
        if (hi > s.cap.out) hi = s.cap.out;
        if (hi > lo && cudaMemcpyAsync(s.h_out + lo, s.d_out + lo, (size_t)(hi - lo), cudaMemcpyDeviceToHost, s.stream) != cudaSuccess) return false;
        if (cudaEventRecord(s.evp[np_issued & 1], s.stream) != cudaSuccess) return false;
        piece_end[np_issued++ & 1] = issued = j;
        return true;
    };
    for (uint32_t i = 0; i < s.n; i++) {
        if (T.status[i] != ZMT_ST_OK) return status_error(c, T.status[i]);
        if (piece_bytes && i >= ready) {
            bool ok = np_issued > np_ready || issue_piece();                                // the piece holding frame i
            if (ok && issued < s.n && np_issued == np_ready + 1) ok = issue_piece();        // and one ahead
            ok = ok && cudaEventSynchronize(s.evp[np_ready & 1]) == cudaSuccess;
            if (!ok) { c->lib_errcode = ZMT_ST_CUDA; return c->E->library; }
            ready = piece_end[np_ready++ & 1];
        }
        const size_t e = write_all(c, rw, s.h_out + T.out_off[i], (size_t)T.out_size[i]);
        if (e) return e;
        c->curframe++;
    }
    return 0;
}

size_t decompress_run(Ctx* c, GenRdWr* rw)
{
    const DeviceRestore restore_device;
    Pipe& P = c->pipe;
    const bool is_zstd = c->codec == CODEC_ZSTD;
    FramedReader reader(c, rw);
    bool framed = false;
    const size_t r = reader.sniff(&framed);
    if (!framed) return r;
    if (!ctx_devices(c)) return c->E->library;
    if (P.slots.empty()) {
        const size_t base_slots = host_slots(c);
        P.slots.resize(base_slots > c->devs.size() ? base_slots : c->devs.size());
        // decode batches must hold enough frames to fill the GPU (one warp per 64 KiB block): 32 MiB of frames measured best
        SlotCaps caps;
        caps.in = env_size("ZSTDMT_B200_DBATCH_MB", 32) << 20; caps.out = 2 * caps.in; caps.tab = 8192;
        // zstd scratch: 16 B per sequence + the literals: ~2x the output on text, bounded at 3x + tables (the reader closes a batch early otherwise)
        if (is_zstd) { caps.blk = 32768; caps.scr = 3 * (uint64_t)caps.out; }
        caps.work = decode_work_bytes(is_zstd, caps);
        for (size_t i = 0; i < P.slots.size(); i++)
            if (!slot_acquire(P.slots[i], c->devs[i % c->devs.size()], caps, nullptr)) { ctx_release_slots(c); return c->E->mem; }
    }
    const uint64_t piece_bytes = (uint64_t)env_size("ZSTDMT_B200_D2H_PIECE_MB", 2) << 20;      // 0: whole slot right after the kernels (measured 0 / 2 / 4 / 8 MiB: 12.8 / 15.1 / 14.3 / 12.8 GB/s)
    return run_pipeline(c, P.slots.size(), [&](Slot& s, bool& last) { return reader.fill(s, last); },
                        [&](Slot& s) { return decode_submit(c, s, piece_bytes); }, [&](Slot& s) { return decode_drain(c, rw, s, piece_bytes); });
}

// ------------------------------------------------------------------ context helpers
Ctx* ctx_new(int codec, bool comp, int threads, int level, size_t inputsize)
{
    Ctx* c = new (std::nothrow) Ctx();
    if (!c) return nullptr;
    c->codec = codec; c->is_comp = comp; c->threads = threads; c->level = level; c->inputsize = inputsize;
    c->E = codec == CODEC_LZ4 ? &kErrLz4 : &kErrZstd;
    return c;
}
void ctx_delete(Ctx* c) { if (!c) return; const DeviceRestore restore_device; ctx_release_slots(c); delete c; }

// Levels.  The device encoders implement one search class per codec (LZ4: the greedy single-probe parse of level 1-2;
// zstd: the same parse + Huffman / predefined-FSE entropy stage, "level 3 (predefined FSE tables)" in BASELINE terms).
// Higher levels are accepted — the CLI default for lz4 is 3 (programs/lz4-mt.c:19) and must keep working — and produce
// the same stream; that is said once on stderr (ZSTDMT_B200_QUIET=1 silences it) instead of silently, and
// ZSTDMT_B200_STRICT_LEVEL=1 turns it into the reference's own answer for a bad parameter (create returns NULL,
// lib/lz4-mt_compress.c:103-108).
bool level_ok(int codec, int level)
{
    const int implemented = codec == CODEC_LZ4 ? 2 : 3;
    if (level <= implemented) return true;
    if (getenv("ZSTDMT_B200_STRICT_LEVEL")) return false;
    static std::atomic<int> told[3];
    if (!getenv("ZSTDMT_B200_QUIET") && told[codec].exchange(1) == 0)
        fprintf(stderr, "[zstdmt_b200] %s level %d requested: the device encoder implements the level-%d search class, the stream is valid but its ratio is that class's\n",
                codec == CODEC_LZ4 ? "lz4" : "zstd", level, implemented);
    return true;
}

const char* status_string(size_t st)
{
    switch (st) {
    case ZMT_ST_TRUNCATED: return "frame truncated";
    case ZMT_ST_BAD_MAGIC: return "ERROR_frameType_unknown";
    case ZMT_ST_BAD_HEADER: return "ERROR_frameHeader_incomplete";
    case ZMT_ST_HDR_CHECKSUM: return "ERROR_headerChecksum_invalid";
    case ZMT_ST_BLOCK: return "ERROR_decompressionFailed";
    case ZMT_ST_DST_SMALL: return "ERROR_dstMaxSize_tooSmall";
    case ZMT_ST_CONTENT_CHECKSUM: return "ERROR_contentChecksum_invalid";
    case ZMT_ST_CONTENT_SIZE: return "ERROR_frameSize_wrong";
    case ZMT_ST_TRAILING: return "trailing bytes after frame";
    case ZMT_ST_UNSUPPORTED: return "stream type not supported by the B200 path";
    case ZMT_ST_CUDA: return "CUDA runtime / kernel failure";
    case ZMT_ST_BAD_ARG: return "bad argument";
    }
    return nullptr;
}

const char* error_string(bool lz4, size_t code, size_t lib_errcode)
{
    const size_t neg = 0 - code;
    // the reference returns the codec library's own message whenever its global errcode is set
    // (lz4-mt_common.c:37-38); we own the status table instead of liblz4 / libzstd
    if (lib_errcode && status_string(lib_errcode) && neg == (lz4 ? 8u : 9u)) return status_string(lib_errcode);
    static const char* lz4s[] = { "No error detected", "Allocation error : not enough memory", "Read failure", "Write failure", "Malformed input",
                                  "Could not compress frame at once", "Could not decompress frame at once", "Compression parameter is out of bound",
                                  "Compression library reports failure" };
    static const char* zs[] = { "No error detected", "Allocation error : not enough memory", nullptr, "Read failure", "Write failure", "Malformed input",
                                "Could not compress frame at once", "Could not decompress frame at once", "Compression parameter is out of bound",
                                "Compression library reports failure" };
    if (lz4) { if (neg < 9) return lz4s[neg]; return "Unspecified lz4mt error code"; }
    if (neg < 10 && zs[neg]) return zs[neg];
    return "Unspecified zstmt error code";
}

}  // namespace

// =================================================================== exported C ABI
extern "C" {

uint64_t zmt_device_batches(int dev) { return (dev >= 0 && dev < 64) ? g_dev_batches[dev].load() : 0; }

size_t lz4mt_errcode = 0;      // lib/lz4-mt_common.c:16
size_t zstdmt_errcode = 0;     // lib/zstd-mt_common.c:19

// ---------------- LZ4MT_*
unsigned LZ4MT_isError(size_t code) { return code > (size_t)-10; }                     // lz4-mt_common.c:25-28 (maxCode = 10)
const char* LZ4MT_getErrorString(size_t code) { return error_string(true, code, lz4mt_errcode); }

void* LZ4MT_createCCtx(int threads, int level, int inputsize)                          // lz4-mt_compress.c:92-156
{
    if (threads < 1 || threads > 128) return nullptr;
    if (level < 1 || level > 12) return nullptr;
    if (inputsize < 0) return nullptr;
    if (!level_ok(CODEC_LZ4, level)) return nullptr;
    return ctx_new(CODEC_LZ4, true, threads, level, inputsize ? (size_t)inputsize : (size_t)4 << 20);
}
size_t LZ4MT_compressCCtx(void* ctx, void* rdwr)                                       // lz4-mt_compress.c:312-353
{
    Ctx* c = (Ctx*)ctx;
    if (!c) return kErrLz4.param;
    if (!rdwr) return kErrLz4.param;
    size_t r = compress_run(c, (GenRdWr*)rdwr);
    if (c->lib_errcode) lz4mt_errcode = c->lib_errcode;
    return r;
}
size_t LZ4MT_GetFramesCCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->curframe : 0; }     // lz4-mt_compress.c:374-380
size_t LZ4MT_GetInsizeCCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->insize : 0; }
size_t LZ4MT_GetOutsizeCCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->outsize : 0; }
void LZ4MT_freeCCtx(void* ctx) { ctx_delete((Ctx*)ctx); }

void* LZ4MT_createDCtx(int threads, int inputsize)                                     // lz4-mt_decompress.c:90-142
{
    if (threads < 1 || threads > 128) return nullptr;
    if (inputsize < 0) return nullptr;
    return ctx_new(CODEC_LZ4, false, threads, 0, inputsize ? (size_t)inputsize : (size_t)64 << 10);
}
size_t LZ4MT_decompressDCtx(void* ctx, void* rdwr)                                     // lz4-mt_decompress.c:485-567
{
    Ctx* c = (Ctx*)ctx;
    if (!c || !rdwr) return kErrLz4.param;
    size_t r = decompress_run(c, (GenRdWr*)rdwr);
    if (c->lib_errcode) lz4mt_errcode = c->lib_errcode;
    return r;
}
size_t LZ4MT_GetFramesDCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->curframe : 0; }
size_t LZ4MT_GetInsizeDCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->insize : 0; }
size_t LZ4MT_GetOutsizeDCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->outsize : 0; }
void LZ4MT_freeDCtx(void* ctx) { ctx_delete((Ctx*)ctx); }

// ---------------- ZSTDCB_*
unsigned ZSTDCB_isError(size_t code) { return code > (size_t)-11; }                    // zstd-mt_common.c:26-29 (maxCode = 11)
const char* ZSTDCB_getErrorString(size_t code) { return error_string(false, code, zstdmt_errcode); }

void* ZSTDCB_createCCtx(int threads, int level, int inputsize)                         // zstd-mt_compress.c:94-155
{
    if (threads < 1 || threads > 128) return nullptr;
    if (level < 1 || level > 22) return nullptr;
    if (inputsize < 0) return nullptr;
    if (!level_ok(CODEC_ZSTD, level)) return nullptr;
    size_t chunk = (size_t)inputsize;
    if (!chunk) {
        // the reference indexes its table by `level`, not level-1 (zstd-mt_compress.c:119-127); level 22 reads past
        // the end there — we clamp to the last entry instead of replicating the overrun
        static const int windowLog[] = { 19, 19, 20, 20, 20, 21, 21, 21, 21, 21, 22, 22, 22, 22, 22, 23, 23, 23, 23, 25, 26, 27 };
        int idx = level > 21 ? 21 : level;
        chunk = (size_t)1 << (windowLog[idx] + 1);
        if (chunk > ((size_t)1 << 30)) chunk = (size_t)1 << 30;     // keep int-sized like the reference's int inputsize
    }
    return ctx_new(CODEC_ZSTD, true, threads, level, chunk);
}
size_t ZSTDCB_compressCCtx(void* ctx, void* rdwr)                                      // zstd-mt_compress.c:322-392
{
    Ctx* c = (Ctx*)ctx;
    if (!c) return kErrZstd.init_missing;
    if (!rdwr) return kErrZstd.param;
    c->insize = c->outsize = c->frames = c->curframe = 0;                               // counters reset per call (:337-341)
    c->lib_errcode = 0;
    size_t r = compress_run(c, (GenRdWr*)rdwr);
    if (c->lib_errcode) zstdmt_errcode = c->lib_errcode;
    return r;
}
size_t ZSTDCB_GetFramesCCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->curframe : kErrZstd.init_missing; }  // :395-420
size_t ZSTDCB_GetInsizeCCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->insize : kErrZstd.init_missing; }
size_t ZSTDCB_GetOutsizeCCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->outsize : kErrZstd.init_missing; }
void ZSTDCB_freeCCtx(void* ctx) { ctx_delete((Ctx*)ctx); }

void* ZSTDCB_createDCtx(int threads, int inputsize)                                    // zstd-mt_decompress.c:105-139
{
    if (threads < 1 || threads > 128) return nullptr;
    if (inputsize < 0) return nullptr;
    return ctx_new(CODEC_ZSTD, false, threads, 0, inputsize ? (size_t)inputsize : (size_t)512 << 10);
}
size_t ZSTDCB_decompressDCtx(void* ctx, void* rdwr)                                    // zstd-mt_decompress.c:693-843
{
    Ctx* c = (Ctx*)ctx;
    if (!c || !rdwr) return kErrZstd.param;
    size_t r = decompress_run(c, (GenRdWr*)rdwr);
    if (c->lib_errcode) zstdmt_errcode = c->lib_errcode;
    return r;
}
size_t ZSTDCB_GetFramesDCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->curframe : 0; }    // :845-869
size_t ZSTDCB_GetInsizeDCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->insize : 0; }
size_t ZSTDCB_GetOutsizeDCtx(void* ctx) { return ctx ? ((Ctx*)ctx)->outsize : 0; }
void ZSTDCB_freeDCtx(void* ctx) { ctx_delete((Ctx*)ctx); }

// ---------------- ZSTDMT_* spellings (lib/README.md:43-76)
unsigned ZSTDMT_isError(size_t code) { return ZSTDCB_isError(code); }
const char* ZSTDMT_getErrorString(size_t code) { return ZSTDCB_getErrorString(code); }
void* ZSTDMT_createCCtx(int t, int l, int i) { return ZSTDCB_createCCtx(t, l, i); }
size_t ZSTDMT_compressCCtx(void* c, void* r) { return ZSTDCB_compressCCtx(c, r); }
size_t ZSTDMT_GetFramesCCtx(void* c) { return ZSTDCB_GetFramesCCtx(c); }
size_t ZSTDMT_GetInsizeCCtx(void* c) { return ZSTDCB_GetInsizeCCtx(c); }
size_t ZSTDMT_GetOutsizeCCtx(void* c) { return ZSTDCB_GetOutsizeCCtx(c); }
void ZSTDMT_freeCCtx(void* c) { ZSTDCB_freeCCtx(c); }
void* ZSTDMT_createDCtx(int t, int i) { return ZSTDCB_createDCtx(t, i); }
size_t ZSTDMT_decompressDCtx(void* c, void* r) { return ZSTDCB_decompressDCtx(c, r); }
size_t ZSTDMT_GetFramesDCtx(void* c) { return ZSTDCB_GetFramesDCtx(c); }
size_t ZSTDMT_GetInsizeDCtx(void* c) { return ZSTDCB_GetInsizeDCtx(c); }
size_t ZSTDMT_GetOutsizeDCtx(void* c) { return ZSTDCB_GetOutsizeDCtx(c); }
void ZSTDMT_freeDCtx(void* c) { ZSTDCB_freeDCtx(c); }

}  // extern "C"
