// zstd_decode.cu — Zstandard frame decoding on sm_100a (the ZSTD_decompressStream step of
// /root/reference/lib/zstd-mt_decompress.c:442-527, one frame per 12-byte container header).
//
// Kernels per batch, all block-parallel (a zstd frame of a 1 MiB chunk has ~64 blocks of ours, 8 of libzstd's):
//   zstd_seq_predef_kernel   one LANE per block: the sequences of blocks on the predefined FSE tables (everything our encoder
//                            writes) — 32 serial state chains per warp instruction
//   zstd_literals_kernel     8 blocks per warp: lane 4g + j decodes Huffman stream j of block g (table per group in SMEM; weights
//                            direct or FSE-coded; treeless literals take the tree from the block the host scan named)
//   zstd_entropy_kernel      one warp per block: whatever the two above left (raw / RLE literals, described tables)
//   zstd_entropy_dep_kernel  one warp per block of a frame with inter-block state (treeless literals, Repeat_Mode tables, repeat
//                            offsets — what libzstd emits for the reference): inherited tables are rebuilt from the describing
//                            block's header, offsets stay as coded; zstd_resolve_offsets_kernel (one warp per frame) then
//                            applies the repeat-offset rule over the frame's records in order
//   zstd_entropy_seq_kernel  one warp per FRAME, blocks in order, state carried: only frames a block-parallel decoder flags at
//                            run time (a repeat offset where the headers showed no state)
//   zstd_offsets_kernel      one thread per frame: exclusive scan of the regenerated sizes -> output offset per block,
//                            content-size check against the frame header
//   zstd_execute_kernel      one warp per block, blocks by ticket (block-index-major): up to 32 sequences per step, written to
//                            global memory and to a window in SMEM; a match that reaches below the block's own output waits for
//                            the `done` flags of the blocks it reads from
//   zstd_checksum_kernel     one warp per frame with a content checksum: XXH64 of the regenerated frame
// Host side (zmt_zstd_scan_frame_host): walks frame + block headers (3 bytes per block + the two section headers), sizes the
// scratch, names per block the block whose header describes each table it uses, flags per frame (state, checksum, no size).
//
// Scope (DESIGN.md §7): the full block format of RFC 8878 — raw / RLE / compressed blocks, Huffman literals with direct
// or FSE-coded weights, 1 or 4 streams, treeless reuse, sequence tables predefined / RLE / FSE-described / repeat,
// repeat offsets, content checksum, frames without a content size — i.e. what libzstd and the zstd CLI emit (SURVEY.md
// fact 0.6).  Not handled (reported per frame as ZMT_ST_UNSUPPORTED, never decoded on the CPU): dictionaries.
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <vector>
#include "common.cuh"
#include "zmt_dev.h"

extern "C" void zmt_prof_mark(int id, void* stream, int end);     // lz4_kernels.cu: record a begin / end event when profiling is armed

// ---------------------------------------------------------------- block descriptors (host-built)
#define ZB_RAW 0u
#define ZB_RLE 1u
#define ZB_CMP 2u
struct ZBlk {
    uint64_t comp_off;      // offset of the block CONTENT (after its 3-byte header) in the input buffer
    uint32_t comp_size;     // content bytes (1 for RLE)
    uint32_t frame;         // frame index in the batch
    uint32_t type;          // ZB_*
    uint32_t regen_hint;    // raw / RLE: regenerated size; compressed: literal bytes (regenerated)
    uint32_t nseq;          // compressed: number of sequences
    uint32_t first;         // 1 if first block of its frame
    uint64_t seq_off;       // scratch offsets (bytes) for this block's sequence records / literals
    uint64_t lit_off;
    // blocks whose tables come from an earlier block of the frame (treeless literals, Repeat_Mode sequence tables): index of
    // the block whose section header DESCRIBES the table in use (ZB_SELF / ZB_PREDEF / ZB_NONE otherwise) — found by the
    // host scan, so that every block can be entropy-decoded on its own
    uint32_t huf_src, ll_src, of_src, ml_src;
};
#define ZB_SELF   0xFFFFFFFFu
#define ZB_PREDEF 0xFFFFFFFEu
#define ZB_NONE   0xFFFFFFFDu
struct ZDSeq { uint32_t ll; uint32_t off; uint32_t ml; uint32_t pad; };

// per-frame flags (the d_frame_seq[] argument; produced by zmt_zstd_scan_frame_host)
#define ZF_NEEDS_SEQ 1u     // blocks depend on earlier blocks: frame-sequential entropy pass
#define ZF_CHECKSUM  2u     // 4-byte content checksum (low 32 bits of XXH64) follows the last block
#define ZF_NO_SIZE   4u     // no Frame_Content_Size: the reported size is an upper bound (128 KiB per compressed block)

// ---------------------------------------------------------------- predefined FSE decode tables
struct ZFseDTable { uint8_t sym[64]; uint8_t nb[64]; uint16_t base[64]; uint32_t log; };
__constant__ ZFseDTable d_fse_ll, d_fse_of, d_fse_ml;
__constant__ uint32_t d_ll_base[36], d_ml_base[53];
__constant__ uint8_t  d_ll_bits[36], d_ml_bits[53];

// ---------------------------------------------------------------- backward bit reader over global memory
// bit `off` = number of unread bits; reads below the stream start return zeros (off goes negative = exhausted).
// A 64-bit window of the stream (bits [wbit, wbit + 64)) lives in registers and is refilled with eight byte loads
// when a read would fall below it — about once per 56 bits instead of four byte loads per read.
struct BackBits {
    const uint8_t* p; int32_t off; int32_t wbit; int32_t nbytes; uint64_t win;
    __device__ __forceinline__ bool init(const uint8_t* s, uint32_t n)
    {
        nbytes = (int32_t)n;
        if (n == 0) return false;
        const uint32_t lastb = s[n - 1];
        if (lastb == 0) return false;
        p = s; off = (int32_t)(n * 8) - (int32_t)(__clz(lastb) - 24 + 1);
        wbit = 0x7FFFFFFF; win = 0;                      // empty window: the first read refills
        return true;
    }
    // up to 32 bits
    __device__ __forceinline__ uint32_t read(uint32_t nb)
    {
        if (nb == 0) return 0;
        const int32_t top = off;                         // bits [top - nb, top); may reach below 0
        off -= (int32_t)nb;
        if (off < wbit) {
            const int32_t tb = (top + 7) >> 3;           // window = the 8 bytes ending with the byte that holds bit top-1 (floor for negatives)
            const int32_t b0 = tb - 8;
            uint64_t w = 0;
            if (b0 >= 0 && tb + 8 <= nbytes) {
                // two aligned 8-byte loads + a funnel shift (the second word stays inside the stream: tb + 8 <= n)
                const uint8_t* a = p + b0;
                const uint64_t* A = reinterpret_cast<const uint64_t*>((uintptr_t)a & ~(uintptr_t)7);
                const uint32_t sh = (uint32_t)((uintptr_t)a & 7) * 8;
                const uint64_t x = A[0];
                w = sh ? (x >> sh) | (A[1] << (64 - sh)) : x;
            } else {
#pragma unroll
                for (int k = 0; k < 8; k++) { const int32_t b = b0 + k; if (b >= 0) w |= (uint64_t)p[b] << (8 * k); }
            }
            win = w; wbit = b0 * 8;
        }
        // bits above the stream end never matter: callers only ask for bits that exist or pad below the start
        return (uint32_t)(win >> (off - wbit)) & (nb >= 32 ? 0xFFFFFFFFu : ((1u << nb) - 1));
    }
};

// Bit reader for the lane-per-block sequence decoder: one refill per sequence (64 bits ending at the byte that holds the
// next unread bit: >= 57 valid bits), reads are a shift and a mask.  bitpos = unread bits of the stream; reading below bit 0
// yields zeros and drives bitpos negative (the caller checks it once per sequence).
struct FastBits {
    const uint8_t* p; int32_t bitpos, base, nbytes; uint64_t win;
    __device__ __forceinline__ bool init(const uint8_t* s, uint32_t n)
    {
        nbytes = (int32_t)n; p = s; base = 0; win = 0;
        if (n == 0) return false;
        const uint32_t lastb = s[n - 1];
        if (lastb == 0) return false;
        bitpos = (int32_t)(n * 8) - (int32_t)(__clz(lastb) - 24 + 1);
        return true;
    }
    __device__ __forceinline__ void refill()
    {
        const int32_t tb = bitpos > 0 ? (bitpos + 7) >> 3 : 0;            // bytes [tb - 8, tb) hold the next bits
        const int32_t b0 = tb - 8;
        uint64_t w = 0;
        if (b0 >= 0 && tb + 8 <= nbytes) {
            const uint8_t* a = p + b0;
            const uint64_t* A = reinterpret_cast<const uint64_t*>((uintptr_t)a & ~(uintptr_t)7);
            const uint32_t sh = (uint32_t)((uintptr_t)a & 7) * 8;
            const uint64_t x = A[0];
            w = sh ? (x >> sh) | (A[1] << (64 - sh)) : x;
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) { const int32_t b = b0 + k; if (b >= 0 && b < nbytes) w |= (uint64_t)p[b] << (8 * k); }
        }
        win = w; base = b0 * 8;
    }
    // nb <= 32, and at most 57 bits between two refills
    __device__ __forceinline__ uint32_t read(uint32_t nb)
    {
        bitpos -= (int32_t)nb;
        const int32_t sh = bitpos - base;                                   // >= 0 while the refill discipline holds; negative only past the stream start
        const uint64_t v = sh >= 0 ? (win >> sh) : (win << (-sh & 63));
        return (uint32_t)v & (nb >= 32 ? 0xFFFFFFFFu : ((1u << nb) - 1));
    }
};

__device__ __forceinline__ void zd_fail(uint32_t* status, uint32_t f, uint32_t code) { atomicCAS(&status[f], 0u, code); }

// literals section header of a compressed block -> header bytes, compressed size, type, size format; false if malformed
__device__ __forceinline__ bool zd_lit_header(const uint8_t* src, uint32_t n, uint32_t* lhdr, uint32_t* lcomp, uint32_t* lregen, uint32_t* ltype, uint32_t* sf_out)
{
    if (n < 1) return false;
    const uint32_t b0 = src[0], lt = b0 & 3, sf = (b0 >> 2) & 3;
    *ltype = lt; *sf_out = sf;
    if (lt < 2) {
        if (sf == 0 || sf == 2) { *lregen = b0 >> 3; *lhdr = 1; }
        else if (sf == 1) { if (n < 2) return false; *lregen = (b0 >> 4) | ((uint32_t)src[1] << 4); *lhdr = 2; }
        else { if (n < 3) return false; *lregen = (b0 >> 4) | ((uint32_t)src[1] << 4) | ((uint32_t)src[2] << 12); *lhdr = 3; }
        *lcomp = lt == 0 ? *lregen : 1;
    } else {
        if (n < 5) return false;
        if (sf < 2) { const uint32_t v = src[0] | (src[1] << 8) | ((uint32_t)src[2] << 16); *lregen = (v >> 4) & 0x3FF; *lcomp = (v >> 14) & 0x3FF; *lhdr = 3; }
        else if (sf == 2) { const uint32_t v = ldg_le32(src); *lregen = (v >> 4) & 0x3FFF; *lcomp = (v >> 18) & 0x3FFF; *lhdr = 4; }
        else { const uint64_t v = (uint64_t)ldg_le32(src) | ((uint64_t)src[4] << 32); *lregen = (uint32_t)((v >> 4) & 0x3FFFF); *lcomp = (uint32_t)((v >> 22) & 0x3FFFF); *lhdr = 5; }
    }
    return (uint64_t)*lhdr + *lcomp <= n;
}

// ---------------------------------------------------------------- per-warp decoding tables (shared memory)
// FSE decode entry: base (16) | nbBits (8) << 16 | symbol << 24
struct ZWarpTabs {
    uint16_t huf[2048];            // (nbBits << 8) | symbol
    uint32_t ll[512], of[256], ml[512];          // tables described in the stream (or RLE: 1 entry)
    uint32_t pll[64], pof[32], pml[64];          // predefined tables
    uint32_t wtab[64];             // FSE table of the Huffman weights (log <= 6)
    uint8_t  wts[256];
    int16_t  norm[64];
    uint32_t hufbits;              // maxbits of the current Huffman table (0 = none yet)
};
#define ZD_NEEDS_SEQ 0x7Fu         // internal status: the frame needs the frame-sequential pass

// Build an FSE decode table from normalized counts (RFC 8878 §4.1.1), one lane.
__device__ bool zd_fse_build(uint32_t* tab, const int16_t* norm, int nsym, int log)
{
    const int size = 1 << log, step = (size >> 1) + (size >> 3) + 3;
    int high = size - 1, pos = 0;
    uint16_t next[64];
    for (int s = 0; s < nsym; s++) { if (norm[s] == -1) { tab[high--] = (uint32_t)s << 24; next[s] = 1; } else next[s] = (uint16_t)norm[s]; }
    for (int s = 0; s < nsym; s++)
        for (int i = 0; i < norm[s]; i++) { tab[pos] = (uint32_t)s << 24; do { pos = (pos + step) & (size - 1); } while (pos > high); }
    if (pos != 0) return false;
    for (int i = 0; i < size; i++) {
        const uint32_t sy = tab[i] >> 24;
        const uint32_t x = next[sy]++;
        const uint32_t nb = (uint32_t)log - (31 - __clz(x));
        tab[i] = (sy << 24) | (nb << 16) | (((x << nb) - (uint32_t)size) & 0xFFFF);
    }
    return true;
}

// Normalized-count header, forward bit order (FSE_readNCount).  Returns bytes consumed or -1.
__device__ int zd_read_ncount(const uint8_t* src, uint32_t n, int16_t* norm, int* nsym, int* log, int maxlog, int maxsym)
{
    uint32_t bitpos = 0;
    auto peek = [&](uint32_t k) -> uint32_t {
        const uint32_t b = bitpos >> 3; uint64_t v = 0;
        for (uint32_t q = 0; q < 5; q++) if (b + q < n) v |= (uint64_t)src[b + q] << (8 * q);
        return (uint32_t)(v >> (bitpos & 7)) & ((1u << k) - 1);
    };
    if (n < 1) return -1;
    const int al = (int)peek(4) + 5; bitpos += 4;
    if (al > maxlog) return -1;
    int remaining = (1 << al) + 1, threshold = 1 << al, nbits = al + 1, sym = 0; bool prev0 = false;
    for (int i = 0; i <= maxsym; i++) norm[i] = 0;
    while (remaining > 1 && sym <= maxsym) {
        if (prev0) {
            for (;;) { const uint32_t rep = peek(2); bitpos += 2; sym += (int)rep; if (rep != 3) break; }
            if (sym > maxsym + 1) return -1;
            prev0 = false;
            if (sym > maxsym) break;
        }
        const int max = (2 * threshold - 1) - remaining;
        int count;
        const uint32_t lo = peek((uint32_t)nbits - 1);
        if ((int)lo < max) { count = (int)lo; bitpos += (uint32_t)nbits - 1; }
        else { count = (int)peek((uint32_t)nbits); if (count >= threshold) count -= max; bitpos += (uint32_t)nbits; }
        count--;
        remaining -= count < 0 ? -count : count;
        norm[sym++] = (int16_t)count;
        prev0 = (count == 0);
        while (remaining < threshold) { nbits--; threshold >>= 1; }
    }
    if (remaining != 1 || sym > maxsym + 1) return -1;
    if (((bitpos + 7) >> 3) > n) return -1;
    *nsym = sym; *log = al;
    return (int)((bitpos + 7) >> 3);
}

// one of the three sequence tables for this block: mode 0 predefined, 1 RLE, 2 FSE-described, 3 repeat
// cur = {table pointer, log}; returns false on error, sets *need_state when mode 3 cannot be honoured
struct ZTabRef { const uint32_t* t; uint32_t log; };
__device__ bool zd_seq_table(ZTabRef& cur, uint32_t mode, uint32_t* custom, const uint32_t* predef, uint32_t predef_log, int16_t* norm,
                             const uint8_t*& qp, uint32_t& qn, int maxlog, int maxsym, bool have_prev, bool* need_state)
{
    if (mode == 0) { cur.t = predef; cur.log = predef_log; return true; }
    if (mode == 1) { if (qn < 1 || qp[0] > maxsym) return false; custom[0] = (uint32_t)qp[0] << 24; cur.t = custom; cur.log = 0; qp++; qn--; return true; }
    if (mode == 2) {
        int nsym = 0, log = 0;
        const int used = zd_read_ncount(qp, qn, norm, &nsym, &log, maxlog, maxsym);
        if (used < 0) return false;
        if (!zd_fse_build(custom, norm, nsym, log)) return false;
        cur.t = custom; cur.log = (uint32_t)log; qp += used; qn -= (uint32_t)used; return true;
    }
    if (!have_prev) { *need_state = true; return false; }
    return true;                                           // repeat: keep cur
}

// Huffman decoding table from a tree description at lp (at most `avail` bytes): direct 4-bit weights, or weights coded
// with a small FSE table.  Whole warp; returns 0 / ZMT_ST_BLOCK, *tbytes_out = bytes of the description.
__device__ uint32_t zd_huf_build(ZWarpTabs& W, const uint8_t* __restrict__ lp, uint32_t lcomp, uint32_t lane, uint32_t* tbytes_out)
{
    uint32_t tbytes = 0;
    {
            // ---- Huffman tree description: direct 4-bit weights, or weights coded with a small FSE table
            const uint32_t hb = lp[0];
            uint32_t nw;
            if (hb >= 128) {
                nw = hb - 127; tbytes = 1 + (nw + 1) / 2;
                if (tbytes > lcomp) return ZMT_ST_BLOCK;
                for (uint32_t i = lane; i < 256; i += 32) {
                    uint32_t w = 0;
                    if (i < nw) { const uint32_t by = lp[1 + i / 2]; w = (i & 1) ? (by & 15) : (by >> 4); }
                    W.wts[i] = (uint8_t)w;
                }
            } else {
                if (hb == 0 || 1 + hb > lcomp) return ZMT_ST_BLOCK;
                tbytes = 1 + hb;
                uint32_t cnt = 0;
                if (lane == 0) {                                // serial: at most 255 weights
                    int nsym = 0, log = 0; bool ok = true;
                    const int hl = zd_read_ncount(lp + 1, hb, W.norm, &nsym, &log, 6, 15);
                    BackBits R;
                    if (hl < 0 || !zd_fse_build(W.wtab, W.norm, nsym, log) || !R.init(lp + 1 + hl, hb - (uint32_t)hl)) ok = false;
                    if (ok) {
                        uint32_t s1 = R.read((uint32_t)log), s2 = R.read((uint32_t)log);
                        if (R.off < 0) ok = false;
                        while (ok) {
                            if (cnt >= 254) { ok = false; break; }
                            uint32_t e = W.wtab[s1]; W.wts[cnt++] = (uint8_t)(e >> 24); s1 = (e & 0xFFFF) + R.read((e >> 16) & 0xFF);
                            if (R.off < 0) { W.wts[cnt++] = (uint8_t)(W.wtab[s2] >> 24); break; }
                            if (cnt >= 254) { ok = false; break; }
                            e = W.wtab[s2]; W.wts[cnt++] = (uint8_t)(e >> 24); s2 = (e & 0xFFFF) + R.read((e >> 16) & 0xFF);
                            if (R.off < 0) { W.wts[cnt++] = (uint8_t)(W.wtab[s1] >> 24); break; }
                        }
                    }
                    if (!ok) cnt = 0xFFFFFFFFu;
                }
                cnt = __shfl_sync(ZMT_FULL_MASK, cnt, 0);
                if (cnt == 0xFFFFFFFFu) return ZMT_ST_BLOCK;
                nw = cnt;
                __syncwarp();
                for (uint32_t i = nw + lane; i < 256; i += 32) W.wts[i] = 0;
            }
            __syncwarp();
            uint32_t total = 0;
            for (uint32_t i = lane; i < nw; i += 32) { const uint32_t w = W.wts[i]; if (w > 11) total += 1u << 20; else if (w) total += 1u << (w - 1); }
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) total += __shfl_xor_sync(ZMT_FULL_MASK, total, d);
            if (total == 0 || total >= 2048) return ZMT_ST_BLOCK;
            const uint32_t maxbits = 32 - __clz(total);
            const uint32_t left = (1u << maxbits) - total;
            if (left == 0 || (left & (left - 1)) || maxbits > 11) return ZMT_ST_BLOCK;
            if (lane == 0) W.wts[nw] = (uint8_t)(32 - __clz(left));
            __syncwarp();
            uint32_t cntw[12];
#pragma unroll
            for (int w = 0; w < 12; w++) cntw[w] = 0;
            for (uint32_t s = 0; s <= nw; s++) { const uint32_t w = W.wts[s]; cntw[w < 12 ? w : 0]++; }
            for (uint32_t s = lane; s <= nw; s += 32) {
                const uint32_t w = W.wts[s];
                if (!w || w > 11) continue;
                uint32_t start = 0;
                for (uint32_t ww = 1; ww < w; ww++) start += cntw[ww] << (ww - 1);
                uint32_t r = 0;
                for (uint32_t t = 0; t < s; t++) r += W.wts[t] == w ? 1u : 0u;
                start += r << (w - 1);
                const uint16_t e = (uint16_t)(((maxbits + 1 - w) << 8) | s);
                for (uint32_t k = 0; k < (1u << (w - 1)); k++) W.huf[start + k] = e;
            }
            if (lane == 0) W.hufbits = maxbits;
            __syncwarp();
    }
    *tbytes_out = tbytes;
    return 0;
}

// Decode one compressed block with one warp.  `fs` (frame state) carries tables + repeat offsets across blocks in the
// frame-sequential pass; in the block-parallel pass fs == nullptr and anything that needs earlier blocks returns
// ZD_NEEDS_SEQ.  Returns 0 ok / ZMT_ST_* / ZD_NEEDS_SEQ; *regen_out = regenerated bytes.
struct ZFrameState { ZTabRef ll, of, ml; uint32_t rep[3]; bool have_tabs; bool raw_offsets; bool huf_ready; };
__device__ uint32_t zd_block(ZWarpTabs& W, const uint8_t* __restrict__ src, uint32_t n, const ZBlk& B, uint8_t* __restrict__ lit,
                             ZDSeq* __restrict__ seqs, ZFrameState* fs, uint32_t* regen_out, uint32_t lane, uint32_t seq_done = 0, uint32_t seq_ml = 0,
                             uint32_t lit_done = 0)
{
    // ---- literals section
    if (n < 1) return ZMT_ST_BLOCK;
    const uint32_t b0 = src[0], ltype = b0 & 3, sf = (b0 >> 2) & 3;
    uint32_t lregen, lcomp = 0, lhdr, streams = 1;
    if (ltype < 2) {
        if (sf == 0 || sf == 2) { lregen = b0 >> 3; lhdr = 1; }
        else if (sf == 1) { lregen = (b0 >> 4) | ((uint32_t)src[1] << 4); lhdr = 2; }
        else { lregen = (b0 >> 4) | ((uint32_t)src[1] << 4) | ((uint32_t)src[2] << 12); lhdr = 3; }
        lcomp = ltype == 0 ? lregen : 1;
    } else {
        if (sf < 2) { const uint32_t v = src[0] | (src[1] << 8) | ((uint32_t)src[2] << 16); lregen = (v >> 4) & 0x3FF; lcomp = (v >> 14) & 0x3FF; lhdr = 3; streams = sf == 0 ? 1 : 4; }
        else if (sf == 2) { const uint32_t v = ldg_le32(src); lregen = (v >> 4) & 0x3FFF; lcomp = (v >> 18) & 0x3FFF; lhdr = 4; streams = 4; }
        else { const uint64_t v = (uint64_t)ldg_le32(src) | ((uint64_t)src[4] << 32); lregen = (uint32_t)((v >> 4) & 0x3FFFF); lcomp = (uint32_t)((v >> 22) & 0x3FFFF); lhdr = 5; streams = 4; }
    }
    if (lhdr + lcomp > n || lregen != B.regen_hint) return ZMT_ST_BLOCK;
    const uint8_t* lp = src + lhdr;
    if (lit_done) { }                                              // literals already decoded by zstd_literals_kernel
    else if (ltype == 0) { for (uint32_t i = lane; i < lregen; i += 32) lit[i] = lp[i]; }
    else if (ltype == 1) { const uint8_t v = lp[0]; for (uint32_t i = lane; i < lregen; i += 32) lit[i] = v; }
    else {
        uint32_t tbytes = 0;
        if (ltype == 2) {
            { const uint32_t hr = zd_huf_build(W, lp, lcomp, lane, &tbytes); if (hr) return hr; }
        } else {
            // treeless: reuse the previous block's table (frame-sequential pass, or rebuilt from the source block's description)
            if (!fs) return ZD_NEEDS_SEQ;
            if (W.hufbits == 0) return ZMT_ST_BLOCK;
        }
        const uint32_t maxbits = W.hufbits;
        if (tbytes + (streams == 4 ? 6u : 0u) > lcomp) return ZMT_ST_BLOCK;
        const uint8_t* sp = lp + tbytes;
        uint32_t ssz[4], spos[4], per = lregen, nsym[4];
        if (streams == 4) {
            const uint32_t s1 = sp[0] | (sp[1] << 8), s2 = sp[2] | (sp[3] << 8), s3 = sp[4] | (sp[5] << 8);
            const uint32_t body = lcomp - tbytes - 6;
            if (s1 + s2 + s3 > body) return ZMT_ST_BLOCK;
            ssz[0] = s1; ssz[1] = s2; ssz[2] = s3; ssz[3] = body - s1 - s2 - s3;
            spos[0] = 0; spos[1] = s1; spos[2] = s1 + s2; spos[3] = s1 + s2 + s3;
            per = (lregen + 3) / 4;
            if (per * 3 > lregen) return ZMT_ST_BLOCK;
            nsym[0] = nsym[1] = nsym[2] = per; nsym[3] = lregen - 3 * per;
            sp += 6;
        } else { ssz[0] = lcomp - tbytes; spos[0] = 0; nsym[0] = lregen; ssz[1] = ssz[2] = ssz[3] = 0; spos[1] = spos[2] = spos[3] = 0; nsym[1] = nsym[2] = nsym[3] = 0; }
        bool okh = true;
        if (lane < streams) {
            BackBits R;
            const uint32_t cnt = nsym[lane];
            uint8_t* o = lit + lane * per;
            if (!R.init(sp + spos[lane], ssz[lane])) okh = false;
            else {
                uint32_t st = R.read(maxbits);
                for (uint32_t i = 0; i < cnt; i++) {
                    const uint32_t e = W.huf[st], nb = e >> 8;
                    o[i] = (uint8_t)e;
                    st = ((st << nb) & ((1u << maxbits) - 1)) | R.read(nb);
                }
                if (R.off != -(int32_t)maxbits) okh = false;
            }
        }
        if (!__all_sync(ZMT_FULL_MASK, okh)) return ZMT_ST_BLOCK;
    }

    // ---- sequences section: lane 0 walks the three interleaved FSE states
    const uint8_t* qp = src + lhdr + lcomp;
    uint32_t qn = n - lhdr - lcomp;
    uint32_t rc = 0, total_ml = 0;
    if (seq_done) { *regen_out = lregen + seq_ml; return 0; }      // sequences already decoded by zstd_seq_predef_kernel
    if (lane == 0) {
        do {
            if (qn < 1) { rc = ZMT_ST_BLOCK; break; }
            uint32_t nseq; const uint32_t q0 = qp[0];
            uint32_t used = 1;
            if (q0 == 0) nseq = 0;
            else if (q0 < 128) nseq = q0;
            else if (q0 < 255) { if (qn < 2) { rc = ZMT_ST_BLOCK; break; } nseq = ((q0 - 128) << 8) + qp[1]; used = 2; }
            else { if (qn < 3) { rc = ZMT_ST_BLOCK; break; } nseq = qp[1] + (qp[2] << 8) + 0x7F00; used = 3; }
            if (nseq != B.nseq) { rc = ZMT_ST_BLOCK; break; }
            if (nseq == 0) { if (used != qn) rc = ZMT_ST_BLOCK; break; }
            if (qn < used + 1) { rc = ZMT_ST_BLOCK; break; }
            const uint32_t modes = qp[used];
            if (modes & 3) { rc = ZMT_ST_BLOCK; break; }
            qp += used + 1; qn -= used + 1;
            ZTabRef tl, to, tm; bool need = false;
            if (fs) { tl = fs->ll; to = fs->of; tm = fs->ml; } else { tl.t = to.t = tm.t = nullptr; tl.log = to.log = tm.log = 0; }
            const bool hp = fs && fs->have_tabs;
            if (!zd_seq_table(tl, (modes >> 6) & 3, W.ll, W.pll, 6, W.norm, qp, qn, 9, 35, hp, &need) ||
                !zd_seq_table(to, (modes >> 4) & 3, W.of, W.pof, 5, W.norm, qp, qn, 8, 31, hp, &need) ||
                !zd_seq_table(tm, (modes >> 2) & 3, W.ml, W.pml, 6, W.norm, qp, qn, 9, 52, hp, &need)) { rc = need ? ZD_NEEDS_SEQ : ZMT_ST_BLOCK; break; }
            if (fs) { fs->ll = tl; fs->of = to; fs->ml = tm; fs->have_tabs = true; }
            BackBits R;                                           // (the one-refill-per-sequence reader of the lane-per-block kernel needs two
            if (!R.init(qp, qn)) { rc = ZMT_ST_BLOCK; break; }    //  refills here — described tables, offsets to 31 bits — and measured slower: 6.9 -> 8.5 ms)
            uint32_t sLL = R.read(tl.log), sOF = R.read(to.log), sML = R.read(tm.log);
            uint32_t r0 = fs ? fs->rep[0] : 1, r1 = fs ? fs->rep[1] : 4, r2 = fs ? fs->rep[2] : 8;
            for (uint32_t i = 0; i < nseq; i++) {
                const uint32_t eo = to.t[sOF], em = tm.t[sML], el = tl.t[sLL];
                const uint32_t ofc = eo >> 24, mlc = em >> 24, llc = el >> 24;
                if (ofc > 31 || mlc > 52 || llc > 35) { rc = ZMT_ST_BLOCK; break; }
                uint32_t ofv = 1u << ofc;                         // offset codes above 25 do not occur below 32 MiB windows
                if (ofc > 24) { ofv += R.read(ofc - 16) << 16; ofv += R.read(16); } else ofv += R.read(ofc);
                const uint32_t ml = d_ml_base[mlc] + R.read(d_ml_bits[mlc]);
                const uint32_t ll = d_ll_base[llc] + R.read(d_ll_bits[llc]);
                uint32_t off;
                if (fs && fs->raw_offsets) off = ofv;             // block-parallel pass: zstd_resolve_offsets_kernel applies the repeat-offset rule
                else if (ofv > 3) { off = ofv - 3; r2 = r1; r1 = r0; r0 = off; }
                else {
                    if (!fs) { rc = ZD_NEEDS_SEQ; break; }        // repeat offsets need the frame's history
                    const uint32_t idx = ofv + (ll == 0 ? 1u : 0u);
                    if (idx == 1) off = r0;
                    else {
                        off = idx == 4 ? r0 - 1 : (idx == 2 ? r1 : r2);
                        if (off == 0) { rc = ZMT_ST_BLOCK; break; }
                        if (idx > 2) r2 = r1;
                        r1 = r0; r0 = off;
                    }
                }
                if (i + 1 < nseq) {
                    sLL = (el & 0xFFFF) + R.read((el >> 16) & 0xFF);
                    sML = (em & 0xFFFF) + R.read((em >> 16) & 0xFF);
                    sOF = (eo & 0xFFFF) + R.read((eo >> 16) & 0xFF);
                }
                if (R.off < 0) { rc = ZMT_ST_BLOCK; break; }
                ZDSeq q; q.ll = ll; q.off = off; q.ml = ml; q.pad = (fs && fs->raw_offsets) ? 1u : 0u;
                seqs[i] = q;
                total_ml += ml;
            }
            if (rc == 0 && R.off != 0) rc = ZMT_ST_BLOCK;
            if (rc == 0 && fs) { fs->rep[0] = r0; fs->rep[1] = r1; fs->rep[2] = r2; }
        } while (0);
    }
    rc = __shfl_sync(ZMT_FULL_MASK, rc, 0);
    total_ml = __shfl_sync(ZMT_FULL_MASK, total_ml, 0);
    *regen_out = lregen + total_ml;
    return rc;
}

__device__ __forceinline__ void zd_load_predef(ZWarpTabs& W, uint32_t lane)
{
    for (uint32_t i = lane; i < 64; i += 32) {
        W.pll[i] = ((uint32_t)d_fse_ll.sym[i] << 24) | ((uint32_t)d_fse_ll.nb[i] << 16) | d_fse_ll.base[i];
        W.pml[i] = ((uint32_t)d_fse_ml.sym[i] << 24) | ((uint32_t)d_fse_ml.nb[i] << 16) | d_fse_ml.base[i];
    }
    W.pof[lane] = ((uint32_t)d_fse_of.sym[lane] << 24) | ((uint32_t)d_fse_of.nb[lane] << 16) | d_fse_of.base[lane];
    if (lane == 0) W.hufbits = 0;
    __syncwarp();
}

// ---------------------------------------------------------------- kernel 0: sequences of predefined-table blocks, one LANE per block
// The three interleaved FSE states of a block are one serial chain; a warp that walks one chain on one lane wastes 31
// issue slots of every instruction (round 1: 1.56 active lanes per instruction, the kernel issue-bound at 71 %).  Blocks
// whose three tables are the predefined ones (every block our encoder writes; `Compression_Modes` = 0) need no per-block
// table memory, so here every lane walks the chain of its own block: 32 chains per warp instruction.  Blocks with
// described / RLE / repeated tables are left to the warp-per-block kernel below (seq_done stays 0).
#define ZS_THREADS 128
__global__ void __launch_bounds__(ZS_THREADS)
zstd_seq_predef_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, uint32_t nblocks, const uint32_t* __restrict__ frame_seq,
                       uint8_t* __restrict__ scratch, uint32_t* __restrict__ seq_done, uint32_t* __restrict__ seq_ml, uint32_t* __restrict__ status)
{
    __shared__ uint32_t pll[64], pof[32], pml[64], llx[36], mlx[53];      // FSE entries; base | bits << 24
    for (uint32_t i = threadIdx.x; i < 64; i += ZS_THREADS) {
        pll[i] = ((uint32_t)d_fse_ll.sym[i] << 24) | ((uint32_t)d_fse_ll.nb[i] << 16) | d_fse_ll.base[i];
        pml[i] = ((uint32_t)d_fse_ml.sym[i] << 24) | ((uint32_t)d_fse_ml.nb[i] << 16) | d_fse_ml.base[i];
        if (i < 32) pof[i] = ((uint32_t)d_fse_of.sym[i] << 24) | ((uint32_t)d_fse_of.nb[i] << 16) | d_fse_of.base[i];
        if (i < 36) llx[i] = d_ll_base[i] | ((uint32_t)d_ll_bits[i] << 24);
        if (i < 53) mlx[i] = d_ml_base[i] | ((uint32_t)d_ml_bits[i] << 24);
    }
    __syncthreads();
    const uint32_t b = blockIdx.x * ZS_THREADS + threadIdx.x;
    if (b >= nblocks) return;
    const ZBlk B = blocks[b];
    if (B.type != ZB_CMP || (frame_seq[B.frame] & ZF_NEEDS_SEQ)) return;
    const uint8_t* src = in + B.comp_off;
    const uint32_t n = B.comp_size;
    // literals section header -> start of the sequences section (validated again by the literal decoder)
    if (n < 1) return;
    const uint32_t b0 = src[0], ltype = b0 & 3, sf = (b0 >> 2) & 3;
    uint32_t lcomp, lhdr;
    if (ltype < 2) {
        uint32_t lregen;
        if (sf == 0 || sf == 2) { lregen = b0 >> 3; lhdr = 1; }
        else if (sf == 1) { if (n < 2) return; lregen = (b0 >> 4) | ((uint32_t)src[1] << 4); lhdr = 2; }
        else { if (n < 3) return; lregen = (b0 >> 4) | ((uint32_t)src[1] << 4) | ((uint32_t)src[2] << 12); lhdr = 3; }
        lcomp = ltype == 0 ? lregen : 1;
    } else {
        if (n < 5) return;
        if (sf < 2) { const uint32_t v = src[0] | (src[1] << 8) | ((uint32_t)src[2] << 16); lcomp = (v >> 14) & 0x3FF; lhdr = 3; }
        else if (sf == 2) { const uint32_t v = ldg_le32(src); lcomp = (v >> 18) & 0x3FFF; lhdr = 4; }
        else { const uint64_t v = (uint64_t)ldg_le32(src) | ((uint64_t)src[4] << 32); lcomp = (uint32_t)((v >> 22) & 0x3FFFF); lhdr = 5; }
    }
    if ((uint64_t)lhdr + lcomp + 1 > n) return;
    const uint8_t* qp = src + lhdr + lcomp;
    uint32_t qn = n - lhdr - lcomp;
    uint32_t nseq; const uint32_t q0 = qp[0];
    uint32_t used = 1;
    if (q0 == 0) nseq = 0;
    else if (q0 < 128) nseq = q0;
    else if (q0 < 255) { if (qn < 2) return; nseq = ((q0 - 128) << 8) + qp[1]; used = 2; }
    else { if (qn < 3) return; nseq = qp[1] + (qp[2] << 8) + 0x7F00; used = 3; }
    if (nseq != B.nseq) return;                               // the general path reports it
    if (nseq == 0) { if (used == qn) { seq_ml[b] = 0; seq_done[b] = 1; } return; }
    if (qn < used + 1 || qp[used] != 0) return;               // not all-predefined: general path
    qp += used + 1; qn -= used + 1;
    FastBits R;
    if (!R.init(qp, qn)) return;
    ZDSeq* seqs = reinterpret_cast<ZDSeq*>(scratch + B.seq_off);
    R.refill();
    uint32_t sLL = R.read(6), sOF = R.read(5), sML = R.read(6);
    uint32_t total_ml = 0;
    for (uint32_t i = 0; i < nseq; i++) {
        R.refill();                                            // >= 57 bits: offset (<= 24) + match extra (<= 16) + literal extra (<= 16)
        const uint32_t eo = pof[sOF], em = pml[sML], el = pll[sLL];
        const uint32_t ofc = eo >> 24, mlc = em >> 24, llc = el >> 24;
        if (ofc > 24) return;                                  // windows above 16 MiB: the general path
        const uint32_t ofv = (1u << ofc) + R.read(ofc);
        const uint32_t mx = mlx[mlc], lx = llx[llc];
        const uint32_t ml = (mx & 0xFFFFFF) + R.read(mx >> 24);
        const uint32_t ll = (lx & 0xFFFFFF) + R.read(lx >> 24);
        if (ofv <= 3) {                                        // repeat offset: needs the frame's history -> frame-sequential pass
            atomicMax(&status[B.frame], ZD_NEEDS_SEQ | 0x8000u);
            return;
        }
        if (i + 1 < nseq) {
            if (ofc + (mx >> 24) + (lx >> 24) > 40) R.refill();             // rare: keep 17 bits for the three state updates
            sLL = (el & 0xFFFF) + R.read((el >> 16) & 0xFF);
            sML = (em & 0xFFFF) + R.read((em >> 16) & 0xFF);
            sOF = (eo & 0xFFFF) + R.read((eo >> 16) & 0xFF);
        }
        if (R.bitpos < 0) return;                              // malformed: the general path redoes the block and reports it
        ZDSeq q; q.ll = ll; q.off = ofv - 3; q.ml = ml; q.pad = 0;
        seqs[i] = q;
        total_ml += ml;
    }
    if (R.bitpos != 0) return;
    seq_ml[b] = total_ml; seq_done[b] = 1;
}

// ---------------------------------------------------------------- kernel 0b: Huffman literals, 8 blocks per warp
// A block's literals are 4 independent Huffman streams: one warp per block keeps 4 lanes busy.  Here a warp takes 8
// blocks: lane 4g + j decodes stream j of block g, every group of 4 lanes builds its block's decoding table in its own
// 4 KiB of shared memory (weights direct or FSE-coded, counting sort by weight, fill).  Handles 4-stream
// Huffman-compressed literals with their own tree (what our encoder and libzstd emit for all but tiny blocks); raw / RLE /
// single-stream / treeless literals stay with the warp-per-block kernel (lit_done stays 0), and so does any block this
// kernel finds malformed, so that errors are reported in one place.  Treeless literals take the tree from the block
// the host scan named (ZBlk::huf_src).
#define ZL_WARPS 2
#define ZL_GROUPS 8
struct ZLitGroup {
    uint16_t huf[2048];            // (nbBits << 8) | symbol
    uint8_t  wts[256];
    uint16_t start[256];           // first table index of every symbol
    uint32_t wtab[64];             // FSE table of the weights
    int16_t  norm[64];
    uint32_t next[16];             // counting sort cursors per weight
};

__global__ void __launch_bounds__(32 * ZL_WARPS)
zstd_literals_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, uint32_t nblocks, const uint32_t* __restrict__ frame_seq,
                     uint8_t* __restrict__ scratch, uint32_t* __restrict__ lit_done)
{
    extern __shared__ __align__(16) uint8_t zl_smem[];
    ZLitGroup* G = reinterpret_cast<ZLitGroup*>(zl_smem) + ((threadIdx.x >> 5) * ZL_GROUPS + ((threadIdx.x & 31) >> 2));
    const uint32_t lane = threadIdx.x & 31, j = lane & 3;
    const uint32_t gmask = 0xFu << (lane & ~3u);                       // the 4 lanes of this group
    const uint32_t b = (blockIdx.x * ZL_WARPS + (threadIdx.x >> 5)) * ZL_GROUPS + (lane >> 2);
    bool ok = b < nblocks;
    ZBlk B; B.type = ZB_RAW; B.comp_size = 0; B.comp_off = 0; B.frame = 0; B.regen_hint = 0; B.lit_off = 0; B.huf_src = ZB_SELF;
    if (ok) { B = blocks[b]; ok = B.type == ZB_CMP && B.comp_size >= 3; }
    const uint8_t* src = in + B.comp_off;
    const uint32_t n = B.comp_size;
    uint32_t lregen = 0, lcomp = 0, lhdr = 0, ltype = 0, sf = 0;
    if (ok) {
        ok = zd_lit_header(src, n, &lhdr, &lcomp, &lregen, &ltype, &sf) && ltype >= 2 && lregen == B.regen_hint && lcomp >= 1;
        if (ok && ltype == 3 && (!(frame_seq[B.frame] & ZF_NEEDS_SEQ) || B.huf_src >= nblocks)) ok = false;     // treeless needs the host-named source block
    }
    const uint32_t nstreams = sf == 0 ? 1u : 4u;
    // the tree description: in this block's own literals section, or (treeless) in the block that last described one
    const uint8_t* lp = src + lhdr;                                     // own literals section content
    const uint8_t* dlp = lp; uint32_t dcomp = lcomp;
    if (ok && ltype == 3) {
        const ZBlk S = blocks[B.huf_src];
        uint32_t sh, sc, sr, st, ssf;
        if (S.type != ZB_CMP || !zd_lit_header(in + S.comp_off, S.comp_size, &sh, &sc, &sr, &st, &ssf) || st != 2 || sc < 1) ok = false;
        else { dlp = in + S.comp_off + sh; dcomp = sc; }
    }
    // ---- weights
    uint32_t nw = 0, tbytes = 0;
    if (ok) {
        const uint32_t hb = dlp[0];
        if (hb >= 128) {
            nw = hb - 127; tbytes = 1 + (nw + 1) / 2;
            if (tbytes > dcomp) ok = false;
            else for (uint32_t i = j; i < 256; i += 4) {
                uint32_t w = 0;
                if (i < nw) { const uint32_t by = dlp[1 + i / 2]; w = (i & 1) ? (by & 15) : (by >> 4); }
                G->wts[i] = (uint8_t)w;
            }
        } else {
            if (hb == 0 || 1 + hb > dcomp) ok = false;
            else {
                tbytes = 1 + hb;
                uint32_t cnt = 0;
                if (j == 0) {                                           // serial: at most 255 weights
                    int nsym = 0, log = 0; bool good = true;
                    const int hl = zd_read_ncount(dlp + 1, hb, G->norm, &nsym, &log, 6, 15);
                    BackBits R;
                    if (hl < 0 || !zd_fse_build(G->wtab, G->norm, nsym, log) || !R.init(dlp + 1 + hl, hb - (uint32_t)hl)) good = false;
                    if (good) {
                        uint32_t s1 = R.read((uint32_t)log), s2 = R.read((uint32_t)log);
                        if (R.off < 0) good = false;
                        while (good) {
                            if (cnt >= 254) { good = false; break; }
                            uint32_t e = G->wtab[s1]; G->wts[cnt++] = (uint8_t)(e >> 24); s1 = (e & 0xFFFF) + R.read((e >> 16) & 0xFF);
                            if (R.off < 0) { G->wts[cnt++] = (uint8_t)(G->wtab[s2] >> 24); break; }
                            if (cnt >= 254) { good = false; break; }
                            e = G->wtab[s2]; G->wts[cnt++] = (uint8_t)(e >> 24); s2 = (e & 0xFFFF) + R.read((e >> 16) & 0xFF);
                            if (R.off < 0) { G->wts[cnt++] = (uint8_t)(G->wtab[s1] >> 24); break; }
                        }
                    }
                    if (!good) cnt = 0xFFFFFFFFu;
                }
                cnt = __shfl_sync(gmask, cnt, lane & ~3u);
                if (cnt == 0xFFFFFFFFu) ok = false; else nw = cnt;
            }
        }
    }
    __syncwarp();
    if (ok && dlp[0] < 128) for (uint32_t i = nw + j; i < 256; i += 4) G->wts[i] = 0;
    __syncwarp();
    // ---- table: total weight -> maxbits and the implied last weight; counting sort by weight; fill
    uint32_t maxbits = 0;
    {
        uint32_t total = 0;
        if (ok) for (uint32_t i = j; i < nw; i += 4) { const uint32_t w = G->wts[i]; if (w > 11) total += 1u << 20; else if (w) total += 1u << (w - 1); }
        total += __shfl_xor_sync(ZMT_FULL_MASK, total, 1);
        total += __shfl_xor_sync(ZMT_FULL_MASK, total, 2);
        if (ok) {
            if (total == 0 || total >= 2048) ok = false;
            else {
                maxbits = 32 - __clz(total);
                const uint32_t left = (1u << maxbits) - total;
                if (left == 0 || (left & (left - 1)) || maxbits > 11) ok = false;
                else if (j == 0) G->wts[nw] = (uint8_t)(32 - __clz(left));
            }
        }
    }
    __syncwarp();
    if (ok && j == 0) {
        uint32_t cntw[12];
#pragma unroll
        for (int w = 0; w < 12; w++) cntw[w] = 0;
        for (uint32_t s2 = 0; s2 <= nw; s2++) {
            const uint32_t w = G->wts[s2];
#pragma unroll
            for (int k = 1; k < 12; k++) cntw[k] += (w == (uint32_t)k) ? 1u : 0u;
        }
        uint32_t acc = 0;
#pragma unroll
        for (int k = 1; k < 12; k++) { G->next[k] = acc; acc += cntw[k] << (k - 1); }
        for (uint32_t s2 = 0; s2 <= nw; s2++) {
            const uint32_t w = G->wts[s2];
            if (w && w < 12) { const uint32_t p0 = G->next[w]; G->start[s2] = (uint16_t)p0; G->next[w] = p0 + (1u << (w - 1)); }
        }
    }
    __syncwarp();
    if (ok) for (uint32_t s2 = j; s2 <= nw; s2 += 4) {
        const uint32_t w = G->wts[s2];
        if (!w || w > 11) continue;
        const uint16_t e = (uint16_t)(((maxbits + 1 - w) << 8) | s2);
        const uint32_t p0 = G->start[s2], cnt = 1u << (w - 1);
        for (uint32_t k = 0; k < cnt; k++) G->huf[p0 + k] = e;
    }
    __syncwarp();
    // ---- the streams (4 with a 6-byte jump table, or 1)
    const uint32_t tb_own = ltype == 2 ? tbytes : 0u;                    // description bytes inside this block's own section
    if (ok && tb_own + (nstreams == 4 ? 6u : 0u) > lcomp) ok = false;
    bool fine = true;
    if (ok && j < nstreams) {
        const uint8_t* sp = lp + tb_own;
        uint32_t ssz, spos, cnt, per = lregen;
        if (nstreams == 4) {
            const uint32_t s1 = sp[0] | (sp[1] << 8), s2 = sp[2] | (sp[3] << 8), s3 = sp[4] | (sp[5] << 8);
            const uint32_t body = lcomp - tb_own - 6;
            per = (lregen + 3) / 4;
            if (s1 + s2 + s3 > body || per * 3 > lregen) fine = false;
            ssz = j == 0 ? s1 : j == 1 ? s2 : j == 2 ? s3 : body - s1 - s2 - s3;
            spos = j == 0 ? 0 : j == 1 ? s1 : j == 2 ? s1 + s2 : s1 + s2 + s3;
            cnt = j < 3 ? per : lregen - 3 * per;
            sp += 6;
        } else { ssz = lcomp - tb_own; spos = 0; cnt = lregen; }
        if (fine) {
            uint8_t* o = scratch + B.lit_off + j * per;
            BackBits R;
            if (!R.init(sp + spos, ssz)) fine = false;
            else {
                const uint32_t msk = (1u << maxbits) - 1;
                uint32_t st = R.read(maxbits);
                for (uint32_t i = 0; i < cnt; i++) {
                    const uint32_t e = G->huf[st], nb = e >> 8;
                    o[i] = (uint8_t)e;
                    st = ((st << nb) & msk) | R.read(nb);
                }
                if (R.off != -(int32_t)maxbits) fine = false;
            }
        }
    }
    // all 4 streams of the block must agree
    const uint32_t good = __ballot_sync(ZMT_FULL_MASK, ok && fine);
    if (ok && j == 0 && ((good >> (lane & ~3u)) & 0xFu) == 0xFu) lit_done[b] = 1;
}

// ---------------------------------------------------------------- kernel 1a: block-parallel entropy decode (self-contained blocks)
#define ZD_WARPS 4
__global__ void __launch_bounds__(32 * ZD_WARPS)
zstd_entropy_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, uint32_t nblocks, const uint32_t* __restrict__ frame_seq,
                    uint8_t* __restrict__ scratch, uint32_t* __restrict__ regen, uint32_t* __restrict__ status,
                    const uint32_t* __restrict__ seq_done, const uint32_t* __restrict__ seq_ml, const uint32_t* __restrict__ lit_done)
{
    __shared__ ZWarpTabs tabs[ZD_WARPS];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * ZD_WARPS + wid;
    if (b >= nblocks) return;
    const ZBlk B = blocks[b];
    if (B.type != ZB_CMP) { if (lane == 0) regen[b] = B.regen_hint; return; }
    if (frame_seq[B.frame] & ZF_NEEDS_SEQ) return;           // this frame goes through the frame-sequential pass
    if (seq_done[b] && lit_done[b]) { if (lane == 0) regen[b] = B.regen_hint + seq_ml[b]; return; }    // nothing left for this block
    ZWarpTabs& W = tabs[wid];
    zd_load_predef(W, lane);
    uint32_t rg = 0;
    const uint32_t rc = zd_block(W, in + B.comp_off, B.comp_size, B, scratch + B.lit_off, reinterpret_cast<ZDSeq*>(scratch + B.seq_off), nullptr, &rg, lane,
                                 seq_done[b], seq_ml[b], lit_done[b]);
    if (lane == 0) {
        if (rc == 0) regen[b] = rg;
        else if (rc == ZD_NEEDS_SEQ) atomicMax(&status[B.frame], ZD_NEEDS_SEQ | 0x8000u);      // flag (cleared by the sequential pass)
        else zd_fail(status, B.frame, rc);
    }
}

// ---------------------------------------------------------------- kernel 1c: block-parallel entropy decode of frames with inter-block state
// What libzstd emits for the reference (SURVEY fact 0.6): treeless literals, Repeat_Mode sequence tables and repeat
// offsets tie the blocks of a frame together.  None of it needs the earlier blocks' DATA, only their section headers:
// the host scan names, per block, the block whose header describes each table in use (ZBlk::*_src), this kernel rebuilds
// those tables from there, decodes the block on its own warp like any other, and leaves the offsets as coded; the
// repeat-offset rule is applied afterwards by one lane per frame (zstd_resolve_offsets_kernel).

// Build sequence table `which` (0 LL, 1 OF, 2 ML) as block S describes it (mode 1 or 2 there).  One lane.
__device__ bool zd_inherit_table(ZTabRef& cur, uint32_t which, const uint8_t* src, uint32_t n, ZWarpTabs& W)
{
    uint32_t lhdr, lcomp, lregen, lt, sf;
    if (!zd_lit_header(src, n, &lhdr, &lcomp, &lregen, &lt, &sf)) return false;
    const uint8_t* qp = src + lhdr + lcomp;
    uint32_t qn = n - lhdr - lcomp;
    if (qn < 1) return false;
    const uint32_t q0 = qp[0];
    const uint32_t used = q0 < 128 ? 1u : q0 < 255 ? 2u : 3u;
    if (q0 == 0 || qn < used + 1) return false;
    const uint32_t modes = qp[used];
    qp += used + 1; qn -= used + 1;
    uint32_t* const custom[3] = { W.ll, W.of, W.ml };
    const uint32_t* const predef[3] = { W.pll, W.pof, W.pml };
    const uint32_t plog[3] = { 6, 5, 6 };
    const int maxlog[3] = { 9, 8, 9 }, maxsym[3] = { 35, 31, 52 };
    for (uint32_t t = 0; t <= which; t++) {
        const uint32_t mode = (modes >> (6 - 2 * t)) & 3;
        if (t == which) {
            if (mode != 1 && mode != 2) return false;              // the host scan only names blocks that describe the table
            bool need = false;
            return zd_seq_table(cur, mode, custom[t], predef[t], plog[t], W.norm, qp, qn, maxlog[t], maxsym[t], false, &need);
        }
        // skip the description of an earlier table
        if (mode == 1) { if (qn < 1) return false; qp++; qn--; }
        else if (mode == 2) {
            int ns = 0, lg = 0;
            const int u = zd_read_ncount(qp, qn, W.norm, &ns, &lg, maxlog[t], maxsym[t]);
            if (u < 0) return false;
            qp += u; qn -= (uint32_t)u;
        }
    }
    return false;
}

__global__ void __launch_bounds__(32 * ZD_WARPS)
zstd_entropy_dep_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, uint32_t nblocks, const uint32_t* __restrict__ frame_seq,
                        uint8_t* __restrict__ scratch, uint32_t* __restrict__ regen, uint32_t* __restrict__ status, const uint32_t* __restrict__ lit_done)
{
    __shared__ ZWarpTabs tabs[ZD_WARPS];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * ZD_WARPS + wid;
    if (b >= nblocks) return;
    const ZBlk B = blocks[b];
    if (B.type != ZB_CMP || !(frame_seq[B.frame] & ZF_NEEDS_SEQ)) return;
    ZWarpTabs& W = tabs[wid];
    zd_load_predef(W, lane);
    ZFrameState fs; fs.rep[0] = 1; fs.rep[1] = 4; fs.rep[2] = 8; fs.have_tabs = true; fs.raw_offsets = true; fs.huf_ready = false;
    fs.ll.t = W.pll; fs.ll.log = 6; fs.of.t = W.pof; fs.of.log = 5; fs.ml.t = W.pml; fs.ml.log = 6;
    uint32_t bad = 0;
    // ---- treeless literals: the tree of the block that last described one
    if (!lit_done[b] && B.huf_src != ZB_SELF) {
        if (B.huf_src >= nblocks) bad = 1;
        else {
            const ZBlk S = blocks[B.huf_src];
            uint32_t lhdr, lcomp, lregen, lt, sf, tb;
            if (S.type != ZB_CMP || !zd_lit_header(in + S.comp_off, S.comp_size, &lhdr, &lcomp, &lregen, &lt, &sf) || lt != 2 || lcomp < 1) bad = 1;
            else if (zd_huf_build(W, in + S.comp_off + lhdr, lcomp, lane, &tb)) bad = 1;
        }
    }
    // ---- repeated sequence tables: rebuilt from the describing block (lane 0), predefined ones are already in place
    if (!bad && B.nseq) {
        uint32_t r = 0;
        if (lane == 0) {
            const uint32_t srcs[3] = { B.ll_src, B.of_src, B.ml_src };
            ZTabRef* const refs[3] = { &fs.ll, &fs.of, &fs.ml };
            for (uint32_t t = 0; t < 3 && !r; t++) {
                if (srcs[t] == ZB_SELF || srcs[t] == ZB_PREDEF) continue;
                if (srcs[t] >= nblocks) { r = 1; break; }
                const ZBlk S = blocks[srcs[t]];
                if (S.type != ZB_CMP || !zd_inherit_table(*refs[t], t, in + S.comp_off, S.comp_size, W)) r = 1;
            }
        }
        bad = __shfl_sync(ZMT_FULL_MASK, r, 0);
        // the table references live in lane 0's registers: broadcast (pointers into this warp's shared tables)
        fs.ll.t = (const uint32_t*)__shfl_sync(ZMT_FULL_MASK, (unsigned long long)fs.ll.t, 0); fs.ll.log = __shfl_sync(ZMT_FULL_MASK, fs.ll.log, 0);
        fs.of.t = (const uint32_t*)__shfl_sync(ZMT_FULL_MASK, (unsigned long long)fs.of.t, 0); fs.of.log = __shfl_sync(ZMT_FULL_MASK, fs.of.log, 0);
        fs.ml.t = (const uint32_t*)__shfl_sync(ZMT_FULL_MASK, (unsigned long long)fs.ml.t, 0); fs.ml.log = __shfl_sync(ZMT_FULL_MASK, fs.ml.log, 0);
    }
    __syncwarp();
    if (bad) { if (lane == 0) zd_fail(status, B.frame, ZMT_ST_BLOCK); return; }
    uint32_t rg = 0;
    const uint32_t rc = zd_block(W, in + B.comp_off, B.comp_size, B, scratch + B.lit_off, reinterpret_cast<ZDSeq*>(scratch + B.seq_off), &fs, &rg, lane, 0, 0, lit_done[b]);
    if (lane == 0) {
        if (rc == 0) regen[b] = rg;
        else zd_fail(status, B.frame, rc == ZD_NEEDS_SEQ ? ZMT_ST_BLOCK : rc);
    }
}

// One WARP per frame: the repeat-offset rule (RFC 8878 3.1.1.5) over the frame's sequences in order.  Records written by the
// block-parallel pass carry the coded offset value and pad = 1.  32 records are loaded at once (coalesced); the rule itself
// is a serial state machine over (r0, r1, r2), walked by all lanes in lockstep with the records passed by shuffle; lane j
// keeps the resolved offset of record j and stores it.
__global__ void __launch_bounds__(32 * ZD_WARPS)
zstd_resolve_offsets_kernel(const ZBlk* __restrict__ blocks, const uint32_t* __restrict__ frame_first_blk, const uint32_t* __restrict__ frame_seq,
                            uint8_t* __restrict__ scratch, uint32_t* __restrict__ status, uint32_t nframes)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t f = blockIdx.x * ZD_WARPS + (threadIdx.x >> 5);
    if (f >= nframes || !(frame_seq[f] & ZF_NEEDS_SEQ) || (status[f] & 0xFF) != 0) return;
    uint32_t r0 = 1, r1 = 4, r2 = 8;
    for (uint32_t b = frame_first_blk[f]; b < frame_first_blk[f + 1]; b++) {
        const ZBlk B = blocks[b];
        if (B.type != ZB_CMP || B.nseq == 0) continue;
        uint4* seqs = reinterpret_cast<uint4*>(scratch + B.seq_off);        // ZDSeq = {ll, off, ml, pad}
        for (uint32_t base = 0; base < B.nseq; base += 32) {
            const uint32_t cnt = B.nseq - base < 32 ? B.nseq - base : 32;
            uint4 q = make_uint4(1, 4, 0, 0);
            if (lane < cnt) q = seqs[base + lane];
            uint32_t mine = q.y;
            const uint32_t raw = __ballot_sync(0xFFFFFFFFu, lane < cnt && q.w == 1);
            if (raw == 0) continue;                                         // block failed or already resolved: leave it
            const uint32_t reps = __ballot_sync(0xFFFFFFFFu, lane < cnt && q.y <= 3);
            if (reps == 0) {
                // no repeat code in these 32: the history is simply the last three offsets
                mine = q.y - 3;
                const uint32_t a0 = __shfl_sync(0xFFFFFFFFu, mine, (cnt - 1) & 31);
                const uint32_t a1 = cnt >= 2 ? __shfl_sync(0xFFFFFFFFu, mine, (cnt - 2) & 31) : r0;
                const uint32_t a2 = cnt >= 3 ? __shfl_sync(0xFFFFFFFFu, mine, (cnt - 3) & 31) : (cnt == 2 ? r0 : r1);
                r0 = a0; r1 = a1; r2 = a2;
            } else {
                bool bad = false;
                for (uint32_t j = 0; j < cnt; j++) {
                    const uint32_t ofv = __shfl_sync(0xFFFFFFFFu, q.y, j), ll = __shfl_sync(0xFFFFFFFFu, q.x, j);
                    uint32_t off;
                    if (ofv > 3) { off = ofv - 3; r2 = r1; r1 = r0; r0 = off; }
                    else {
                        const uint32_t idx = ofv + (ll == 0 ? 1u : 0u);
                        if (idx == 1) off = r0;
                        else {
                            off = idx == 4 ? r0 - 1 : (idx == 2 ? r1 : r2);
                            if (off == 0) { bad = true; break; }
                            if (idx > 2) r2 = r1;
                            r1 = r0; r0 = off;
                        }
                    }
                    if (lane == j) mine = off;
                }
                if (bad) { if (lane == 0) zd_fail(status, f, ZMT_ST_BLOCK); return; }
            }
            if (lane < cnt) { uint32_t* w = reinterpret_cast<uint32_t*>(seqs + base + lane); w[1] = mine; w[3] = 0; }
        }
    }
}

// ---------------------------------------------------------------- kernel 1b: frame-sequential entropy decode
// One warp per frame that needs state across blocks: Huffman table reuse (treeless literals), Repeat_Mode sequence
// tables, repeat offsets.  Same per-block routine, blocks in order, state in registers / this warp's shared tables.
__global__ void __launch_bounds__(32 * ZD_WARPS)
zstd_entropy_seq_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, const uint32_t* __restrict__ frame_first_blk,
                        const uint32_t* __restrict__ frame_seq, uint8_t* __restrict__ scratch, uint32_t* __restrict__ regen,
                        uint32_t* __restrict__ status, uint32_t nframes, uint32_t flagged_only)
{
    __shared__ ZWarpTabs tabs[ZD_WARPS];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const uint32_t f = blockIdx.x * ZD_WARPS + wid;
    if (f >= nframes) return;
    const uint32_t st0 = status[f];
    const bool flagged = (st0 & 0x8000u) != 0;
    // flagged_only: frames the host scan marked were decoded block-parallel (kernel 1c); this pass then only takes the
    // frames a block-parallel decoder flagged at run time (a repeat offset in a frame whose headers showed no state)
    if (!flagged && (flagged_only || !(frame_seq[f] & ZF_NEEDS_SEQ))) return;
    __syncwarp();
    if (lane == 0 && flagged) status[f] = 0;
    ZWarpTabs& W = tabs[wid];
    zd_load_predef(W, lane);
    ZFrameState fs; fs.rep[0] = 1; fs.rep[1] = 4; fs.rep[2] = 8; fs.have_tabs = false; fs.raw_offsets = false; fs.huf_ready = false;
    fs.ll.t = fs.of.t = fs.ml.t = nullptr; fs.ll.log = fs.of.log = fs.ml.log = 0;
    for (uint32_t b = frame_first_blk[f]; b < frame_first_blk[f + 1]; b++) {
        const ZBlk B = blocks[b];
        if (B.type != ZB_CMP) continue;                      // raw / RLE blocks: regen already set by kernel 1a
        uint32_t rg = 0;
        const uint32_t rc = zd_block(W, in + B.comp_off, B.comp_size, B, scratch + B.lit_off, reinterpret_cast<ZDSeq*>(scratch + B.seq_off), &fs, &rg, lane);
        if (rc != 0) { if (lane == 0) zd_fail(status, f, rc == ZD_NEEDS_SEQ ? ZMT_ST_BLOCK : rc); return; }
        if (lane == 0) regen[b] = rg;
        __syncwarp();
    }
}

// ---------------------------------------------------------------- kernel 2: output offsets per block
__global__ void zstd_offsets_kernel(const ZBlk* __restrict__ blocks, uint32_t nblocks, const uint32_t* __restrict__ frame_first_blk,
                                    const uint32_t* __restrict__ regen, uint64_t* __restrict__ blk_out, const uint64_t* __restrict__ out_off,
                                    const uint64_t* __restrict__ expect, unsigned long long* __restrict__ out_size, uint32_t* __restrict__ status,
                                    uint32_t nframes)
{
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes) return;
    const uint32_t b0 = frame_first_blk[f], b1 = frame_first_blk[f + 1];
    uint64_t pos = 0;
    const uint64_t cap = out_off[f + 1] - out_off[f];
    for (uint32_t b = b0; b < b1; b++) { blk_out[b] = out_off[f] + pos; pos += regen[b]; }
    out_size[f] = pos;
    // expect = ~0: the frame header carries no content size (streamed frames); the room then is only a bound
    if ((status[f] & 0xFF) == 0 && ((expect[f] != ~0ull && pos != expect[f]) || pos > cap)) status[f] = pos > cap ? ZMT_ST_DST_SMALL : ZMT_ST_CONTENT_SIZE;
}

// ---------------------------------------------------------------- kernel 3: sequence execution
#define ZX_WARPS 8
#define ZX_SPAN 2048u          // bytes a step of the execute pass may regenerate: staged in shared memory
// One block, one warp.  Blocks are handed out by a ticket counter (see the kernel below), so every block this one may wait
// for — lower indices of the same frame — is held by a warp that is already running: the wait cannot deadlock whatever
// order the hardware schedules CTAs in.
__device__ void zx_block(uint32_t b, uint32_t lane, const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, const uint8_t* __restrict__ scratch,
                         const uint32_t* __restrict__ regen, const uint64_t* __restrict__ blk_out, const uint64_t* __restrict__ out_off,
                         uint8_t* __restrict__ out, uint32_t* __restrict__ done, uint32_t* __restrict__ status, uint8_t* S)
{
    const ZBlk B = blocks[b];
    volatile uint32_t* vdone = done;
    // a frame that already failed: do not touch memory, just release the waiters
    if ((status[B.frame] & 0xFF) != 0) { __syncwarp(); if (lane == 0) { __threadfence(); vdone[b] = 1; } return; }
    uint8_t* dst = out + blk_out[b];
    const uint64_t frame_base = out_off[B.frame];
    const uint32_t rg = regen[b];
    if (B.type == ZB_RAW) { const uint8_t* s = in + B.comp_off; for (uint32_t i = lane; i < rg; i += 32) dst[i] = s[i]; }
    else if (B.type == ZB_RLE) { const uint8_t v = in[B.comp_off]; for (uint32_t i = lane; i < rg; i += 32) dst[i] = v; }
    else {
        const uint8_t* lit = scratch + B.lit_off;
        const ZDSeq* seqs = reinterpret_cast<const ZDSeq*>(scratch + B.seq_off);
        uint32_t op = 0, lp = 0;
        bool bad = false;
        uint32_t waited_to = b;                              // blocks [waited_to, b) are known complete
        const uint64_t blk_abs = blk_out[b];                 // absolute output address of this block
        const uint64_t blk_in_frame = blk_abs - frame_base;
        // Up to 32 sequences per step: one coalesced load of the records, positions from two warp scans.  Everything the step
        // regenerates — at most ZX_SPAN bytes, else the step is cut shorter — is written to global memory AND to a window in
        // shared memory: every lane copies its own literal run (literals come from the scratch, no ordering among them), then
        // the matches run; a source byte at or above the step's first output byte is read from the window, so a chain of
        // matches feeding each other runs at shared-memory latency instead of one L2 round trip per link.
        for (uint32_t base = 0; base < B.nseq;) {
            uint32_t cnt = B.nseq - base < 32 ? B.nseq - base : 32;
            uint32_t ll = 0, off = 0, ml = 0;
            if (lane < cnt) { const ZDSeq q = seqs[base + lane]; ll = q.ll; off = q.off; ml = q.ml; }
            uint32_t it = ll + ml, il = ll;                  // inclusive scans: output bytes, literal bytes
            if (lane < cnt && (ll > rg || ml > rg)) { it = 0x40000000u; }    // absurd lengths: caught below, keep the scan from wrapping
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t a = __shfl_up_sync(0xFFFFFFFFu, it, d), c = __shfl_up_sync(0xFFFFFFFFu, il, d);
                if (lane >= (uint32_t)d) { it = (it + a) | ((it | a) & 0x40000000u); il += c; }
            }
            const uint32_t nfit = __popc(__ballot_sync(0xFFFFFFFFu, lane < cnt && it <= ZX_SPAN));      // sorted: a prefix
            if (nfit == 0) {
                // the first sequence alone is larger than the window: straight in global memory, by the whole warp
                const uint32_t qll = __shfl_sync(0xFFFFFFFFu, ll, 0), qoff = __shfl_sync(0xFFFFFFFFu, off, 0), qml = __shfl_sync(0xFFFFFFFFu, ml, 0);
                const uint32_t mp = op + qll;
                if ((uint64_t)op + qll + qml > rg || (uint64_t)lp + qll > B.regen_hint || qoff == 0 || (uint64_t)qoff > blk_in_frame + mp) { bad = true; break; }
                for (uint32_t k = lane; k < qll; k += 32) dst[op + k] = lit[lp + k];
                if (qoff > mp) {
                    const unsigned long long need = blk_abs + mp - qoff;
                    bool waited = false;
                    while (waited_to > 0 && blocks[waited_to - 1].frame == B.frame && blk_out[waited_to - 1] + regen[waited_to - 1] > need) {
                        waited_to--; waited = true;
                        if (lane == 0) { while (vdone[waited_to] == 0) __nanosleep(64); }
                    }
                    __syncwarp();
                    if (waited) __threadfence();
                }
                __syncwarp();
                uint8_t* d = dst + mp;
                const uint8_t* m = d - qoff;
                if (qoff >= qml) { for (uint32_t k = lane; k < qml; k += 32) d[k] = m[k]; }
                else if (qoff >= 32) { for (uint32_t k = 0; k < qml; k += 32) { if (k + lane < qml) d[k + lane] = m[k + lane]; __syncwarp(); } }
                else { for (uint32_t k = lane; k < qml; k += 32) d[k] = m[k % qoff]; }
                __syncwarp();
                op += qll + qml; lp += qll; base += 1;
                continue;
            }
            cnt = nfit;
            if (lane >= cnt) { ll = 0; ml = 0; }
            const uint32_t my_op = op + it - (ll + ml), my_lp = lp + il - ll, my_mp = my_op + ll;
            const bool mybad = lane < cnt && ((uint64_t)my_op + ll + ml > rg || (uint64_t)my_lp + ll > B.regen_hint || off == 0 || (uint64_t)off > blk_in_frame + my_mp);
            const uint32_t badmask = __ballot_sync(0xFFFFFFFFu, mybad);
            const uint32_t lim = badmask ? (uint32_t)(__ffs(badmask) - 1) : cnt;      // sequences of this step that are executed
            const int32_t wb = -(int32_t)op;                                           // S[wb + p] = window byte of block position p (op <= p < op + ZX_SPAN)
            if (lane < lim && ll <= 32) {
                // loads first, stores after, 8 bytes at a time: a byte-wise load -> store loop pays one L2 latency per byte
                const uint8_t* ls = lit + my_lp; uint8_t* d = dst + my_op; uint8_t* dw = S + (wb + (int32_t)my_op);
                for (uint32_t k = 0; k < ll; k += 8) {
                    uint8_t x[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) x[j] = (k + j < ll) ? ls[k + j] : (uint8_t)0;
#pragma unroll
                    for (int j = 0; j < 8; j++) if (k + j < ll) { d[k + j] = x[j]; dw[k + j] = x[j]; }
                }
            }
            uint32_t longmask = __ballot_sync(0xFFFFFFFFu, lane < lim && ll > 32);
            while (longmask) {                                // long literal runs: the whole warp copies
                const int jl = __ffs(longmask) - 1; longmask &= longmask - 1;
                const uint32_t o = __shfl_sync(0xFFFFFFFFu, my_op, jl), l0 = __shfl_sync(0xFFFFFFFFu, my_lp, jl), n = __shfl_sync(0xFFFFFFFFu, ll, jl);
                for (uint32_t k = lane; k < n; k += 32) { const uint8_t x = lit[l0 + k]; dst[o + k] = x; S[wb + (int32_t)(o + k)] = x; }
            }
            // ---- matches.  Any source below this block: wait (once per step) for the earlier blocks it touches.
            {
                unsigned long long need = ~0ull;                            // lowest absolute output address read by this step
                if (lane < lim && ml && off > my_mp) need = blk_abs + my_mp - off;
#pragma unroll
                for (int x = 16; x > 0; x >>= 1) { const unsigned long long y = __shfl_xor_sync(0xFFFFFFFFu, need, x); need = y < need ? y : need; }
                if (need != ~0ull) {
                    bool waited = false;
                    while (waited_to > 0 && blocks[waited_to - 1].frame == B.frame && blk_out[waited_to - 1] + regen[waited_to - 1] > need) {
                        waited_to--; waited = true;
                        if (lane == 0) { while (vdone[waited_to] == 0) __nanosleep(64); }
                    }
                    __syncwarp();
                    if (waited) __threadfence();
                }
            }
            __syncwarp();                                                   // this step's literals are in place (global and window)
            // (the destinations [my_mp, my_mp + ml) of a step are sorted and disjoint: a match is independent iff its source
            //  touches no destination of an earlier match of the step — binary search over the lanes by shuffle, as in
            //  lz4_exec_blocks_kernel — and does not overlap its own destination; independent matches run lane-parallel)
            const bool act = lane < lim && ml != 0;
            const int32_t sp = (int32_t)my_mp - (int32_t)off;               // block-relative source start (negative: earlier blocks)
            const int32_t e_end = act ? (int32_t)(my_mp + ml) : 0x7FFFFFFF, d_beg = act ? (int32_t)my_mp : 0x7FFFFFFF;
            uint32_t a = 0;
#pragma unroll
            for (uint32_t stp = 16; stp > 0; stp >>= 1) {
                const int32_t v = __shfl_sync(0xFFFFFFFFu, e_end, (a + stp - 1) & 31);
                if (v <= sp) a += stp;
            }
            const int32_t da = __shfl_sync(0xFFFFFFFFu, d_beg, a & 31);
            const bool indep = act && off >= ml && !(a < lane && da < sp + (int32_t)ml);
            if (indep && ml <= 32) {
                uint8_t* d = dst + my_mp; uint8_t* dw = S + (wb + (int32_t)my_mp);
                const int32_t nlow = sp >= (int32_t)op ? 0 : ((int32_t)op - sp < (int32_t)ml ? (int32_t)op - sp : (int32_t)ml);
                const uint8_t* m = dst + sp;
                int32_t k = 0;
                for (; k < nlow; k += 8) {
                    uint8_t x[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) x[j] = (k + j < nlow) ? m[k + j] : (uint8_t)0;
#pragma unroll
                    for (int j = 0; j < 8; j++) if (k + j < nlow) { d[k + j] = x[j]; dw[k + j] = x[j]; }
                }
                k = nlow;
                for (; k < (int32_t)ml; k++) { const uint8_t x = S[wb + sp + k]; d[k] = x; dw[k] = x; }
            }
            uint32_t dm = __ballot_sync(0xFFFFFFFFu, act && !(indep && ml <= 32));       // long independent ones and the dependent ones: in order, whole warp
            if (dm) __syncwarp();
            while (dm) {
                const int jq = __ffs(dm) - 1; dm &= dm - 1;
                const uint32_t qoff = __shfl_sync(0xFFFFFFFFu, off, jq), qml = __shfl_sync(0xFFFFFFFFu, ml, jq), mp = __shfl_sync(0xFFFFFFFFu, my_mp, jq);
                const int32_t qs = (int32_t)mp - (int32_t)qoff;
                uint8_t* d = dst + mp; uint8_t* dw = S + (wb + (int32_t)mp);
                if (qoff >= qml) { for (uint32_t k = lane; k < qml; k += 32) { const int32_t q = qs + (int32_t)k; const uint8_t x = q >= (int32_t)op ? S[wb + q] : dst[q]; d[k] = x; dw[k] = x; } }
                else if (qoff >= 32) {
                    for (uint32_t k = 0; k < qml; k += 32) {
                        if (k + lane < qml) { const int32_t q = qs + (int32_t)(k + lane); const uint8_t x = q >= (int32_t)op ? S[wb + q] : dst[q]; d[k + lane] = x; dw[k + lane] = x; }
                        __syncwarp();
                    }
                } else { for (uint32_t k = lane; k < qml; k += 32) { const int32_t q = qs + (int32_t)(k % qoff); const uint8_t x = q >= (int32_t)op ? S[wb + q] : dst[q]; d[k] = x; dw[k] = x; } }
                __syncwarp();
            }
            __syncwarp();
            if (badmask) { bad = true; break; }
            op += __shfl_sync(0xFFFFFFFFu, it, cnt - 1);
            lp += __shfl_sync(0xFFFFFFFFu, il, cnt - 1);
            base += cnt;
        }
        if (!bad) {
            const uint32_t rest = B.regen_hint - lp;
            if (op + rest != rg) bad = true;
            else for (uint32_t k = lane; k < rest; k += 32) dst[op + k] = lit[lp + k];
        }
        if (bad && lane == 0) zd_fail(status, B.frame, ZMT_ST_BLOCK);
    }
    __syncwarp();
    if (lane == 0) { __threadfence(); vdone[b] = 1; }
}

// Ticket order, as in lz4_exec_blocks_kernel: within a window of ZX_WIN frames block-index-major (block 0 of every frame,
// then block 1, ...), so that the blocks of one frame — a dependency chain wherever matches reach below their block — are
// not handed to neighbouring warps, and as many independent chains are in flight as there are frames.  Block (f, b-1)
// always holds a lower ticket than (f, b).  Windows with very ragged block counts fall back to frame-major order.
#define ZX_WIN 16384u
__global__ void __launch_bounds__(256)
zstd_ticket_windows_kernel(const uint32_t* __restrict__ frame_first_blk, uint32_t nframes, unsigned long long* __restrict__ wbase)
{
    __shared__ uint32_t red[256];
    const uint32_t nwin = (nframes + ZX_WIN - 1) / ZX_WIN;
    unsigned long long base = 0;
    for (uint32_t w = 0; w < nwin; w++) {
        const uint32_t f0 = w * ZX_WIN, f1 = f0 + ZX_WIN < nframes ? f0 + ZX_WIN : nframes;
        uint32_t mx = 0;
        for (uint32_t f = f0 + threadIdx.x; f < f1; f += 256) { const uint32_t c = frame_first_blk[f + 1] - frame_first_blk[f]; mx = c > mx ? c : mx; }
        red[threadIdx.x] = mx;
        __syncthreads();
        for (uint32_t d = 128; d > 0; d >>= 1) { if (threadIdx.x < d && red[threadIdx.x + d] > red[threadIdx.x]) red[threadIdx.x] = red[threadIdx.x + d]; __syncthreads(); }
        mx = red[0];
        __syncthreads();
        const unsigned long long real = frame_first_blk[f1] - frame_first_blk[f0], grid = (unsigned long long)(f1 - f0) * mx;
        const bool frame_major = grid > 8 * real + 65536;
        if (threadIdx.x == 0) wbase[w] = base | (frame_major ? (1ull << 63) : 0ull);
        base += frame_major ? real : grid;
    }
    if (threadIdx.x == 0) wbase[nwin] = base;
}

__global__ void __launch_bounds__(32 * ZX_WARPS)
zstd_execute_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, uint32_t nblocks, const uint8_t* __restrict__ scratch,
                    const uint32_t* __restrict__ regen, const uint64_t* __restrict__ blk_out, const uint64_t* __restrict__ out_off,
                    uint8_t* __restrict__ out, uint32_t* __restrict__ done, uint32_t* __restrict__ status, unsigned long long* __restrict__ ticket,
                    const uint32_t* __restrict__ frame_first_blk, const unsigned long long* __restrict__ wbase, uint32_t nframes)
{
    __shared__ __align__(16) uint8_t stage[ZX_WARPS][ZX_SPAN];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t nwin = (nframes + ZX_WIN - 1) / ZX_WIN;
    const unsigned long long ntickets = wbase[nwin] & ~(1ull << 63);
    for (;;) {
        unsigned long long tk = 0;
        if (lane == 0) tk = atomicAdd(ticket, 1ull);
        tk = __shfl_sync(0xFFFFFFFFu, tk, 0);
        if (tk >= ntickets) return;
        uint32_t lo = 0, hi = nwin;
        while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if ((wbase[mid] & ~(1ull << 63)) <= tk) lo = mid; else hi = mid; }
        const unsigned long long wb = wbase[lo];
        const unsigned long long tl = tk - (wb & ~(1ull << 63));
        const uint32_t f0 = lo * ZX_WIN, wn = (f0 + ZX_WIN < nframes ? ZX_WIN : nframes - f0);
        uint32_t b;
        if (wb >> 63) b = frame_first_blk[f0] + (uint32_t)tl;
        else {
            const uint32_t fb = (uint32_t)(tl / wn), ff = f0 + (uint32_t)(tl % wn);
            const uint32_t s0 = frame_first_blk[ff];
            if (fb >= frame_first_blk[ff + 1] - s0) continue;
            b = s0 + fb;
        }
        if (b >= nblocks) continue;
        zx_block(b, lane, in, blocks, scratch, regen, blk_out, out_off, out, done, status, stage[threadIdx.x >> 5]);
        __syncwarp();
    }
}

// ---------------------------------------------------------------- kernel 4: frame content checksum (XXH64, seed 0; RFC 8878 3.1.1)
// One warp per frame that carries a checksum (what the stock zstd CLI writes by default; the reference path —
// ZSTD_compress, zstd-mt_compress.c:284-286 — never does).  Lanes 0..3 run the four accumulator chains, each over its
// 8-byte word of every 32-byte stripe; eight stripes are loaded ahead of their use.
#define XP64_1 0x9E3779B185EBCA87ull
#define XP64_2 0xC2B2AE3D27D4EB4Full
#define XP64_3 0x165667B19E3779F9ull
#define XP64_4 0x85EBCA77C2B2AE63ull
#define XP64_5 0x27D4EB2F165667C5ull
__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
__device__ __forceinline__ uint64_t xxh64_round(uint64_t acc, uint64_t v) { return rotl64(acc + v * XP64_2, 31) * XP64_1; }
__device__ __forceinline__ uint64_t xxh64_merge(uint64_t h, uint64_t v) { return (h ^ xxh64_round(0, v)) * XP64_1 + XP64_4; }
__device__ __forceinline__ uint64_t ldg_le64u(const uint8_t* p)
{
    if (((uintptr_t)p & 7) == 0) return *reinterpret_cast<const uint64_t*>(p);
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) v |= (uint64_t)p[i] << (8 * i);
    return v;
}

__global__ void __launch_bounds__(32 * ZD_WARPS)
zstd_checksum_kernel(const uint8_t* __restrict__ in, const ZBlk* __restrict__ blocks, const uint32_t* __restrict__ frame_first_blk,
                     const uint32_t* __restrict__ frame_seq, const uint8_t* __restrict__ out, const uint64_t* __restrict__ out_off,
                     const unsigned long long* __restrict__ out_size, uint32_t* __restrict__ status, uint32_t nframes)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t f = blockIdx.x * ZD_WARPS + (threadIdx.x >> 5);
    if (f >= nframes || !(frame_seq[f] & ZF_CHECKSUM) || (status[f] & 0xFF) != 0) return;
    const uint32_t b1 = frame_first_blk[f + 1];
    if (b1 == frame_first_blk[f]) return;
    const ZBlk BL = blocks[b1 - 1];
    const uint8_t* p = out + out_off[f];
    const uint64_t n = out_size[f];
    uint64_t h;
    if (n >= 32) {
        const uint32_t j = lane & 3;
        uint64_t acc = j == 0 ? XP64_1 + XP64_2 : j == 1 ? XP64_2 : j == 2 ? 0ull : 0ull - XP64_1;
        const uint64_t ns = n >> 5;
        uint64_t s = 0;
        if (lane < 4) {
            for (; s + 8 <= ns; s += 8) {
                uint64_t v[8];
#pragma unroll
                for (int k = 0; k < 8; k++) v[k] = ldg_le64u(p + ((s + k) << 5) + 8 * j);
#pragma unroll
                for (int k = 0; k < 8; k++) acc = xxh64_round(acc, v[k]);
            }
            for (; s < ns; s++) acc = xxh64_round(acc, ldg_le64u(p + (s << 5) + 8 * j));
        }
        const uint64_t a1 = __shfl_sync(0xFFFFFFFFu, acc, 0), a2 = __shfl_sync(0xFFFFFFFFu, acc, 1), a3 = __shfl_sync(0xFFFFFFFFu, acc, 2), a4 = __shfl_sync(0xFFFFFFFFu, acc, 3);
        h = rotl64(a1, 1) + rotl64(a2, 7) + rotl64(a3, 12) + rotl64(a4, 18);
        h = xxh64_merge(h, a1); h = xxh64_merge(h, a2); h = xxh64_merge(h, a3); h = xxh64_merge(h, a4);
    } else h = XP64_5;
    if (lane == 0) {
        h += n;
        const uint8_t* q = p + (n & ~31ull); const uint8_t* end = p + n;
        while (q + 8 <= end) { h ^= xxh64_round(0, ldg_le64u(q)); h = rotl64(h, 27) * XP64_1 + XP64_4; q += 8; }
        if (q + 4 <= end) { h ^= (uint64_t)((uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24)) * XP64_1; h = rotl64(h, 23) * XP64_2 + XP64_3; q += 4; }
        while (q < end) { h ^= (*q) * XP64_5; h = rotl64(h, 11) * XP64_1; q++; }
        h ^= h >> 33; h *= XP64_2; h ^= h >> 29; h *= XP64_3; h ^= h >> 32;
        const uint8_t* c = in + BL.comp_off + BL.comp_size;
        const uint32_t stored = (uint32_t)c[0] | ((uint32_t)c[1] << 8) | ((uint32_t)c[2] << 16) | ((uint32_t)c[3] << 24);
        if (stored != (uint32_t)h) zd_fail(status, f, ZMT_ST_CONTENT_CHECKSUM);
    }
}

// ================================================================ host side
static void zd_build_dtable(ZFseDTable& T, const int16_t* norm, int nsym, int log)
{
    const int size = 1 << log, step = (size >> 1) + (size >> 3) + 3;
    int high = size - 1, pos = 0; uint16_t next[64];
    memset(&T, 0, sizeof(T)); T.log = (uint32_t)log;
    for (int s = 0; s < nsym; s++) { if (norm[s] == -1) { T.sym[high--] = (uint8_t)s; next[s] = 1; } else next[s] = (uint16_t)norm[s]; }
    for (int s = 0; s < nsym; s++)
        for (int i = 0; i < norm[s]; i++) { T.sym[pos] = (uint8_t)s; do { pos = (pos + step) & (size - 1); } while (pos > high); }
    for (int i = 0; i < size; i++) {
        const uint16_t x = next[T.sym[i]]++;
        int hb = 0; while ((1 << (hb + 1)) <= x) hb++;
        T.nb[i] = (uint8_t)(log - hb);
        T.base[i] = (uint16_t)(((uint32_t)x << T.nb[i]) - size);
    }
}

static int zd_sm_count()
{
    static std::mutex mu; static int n[64];
    int dev = 0; cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    std::lock_guard<std::mutex> g(mu);
    if (!n[dev]) { cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev); if (n[dev] <= 0) n[dev] = 148; }
    return n[dev];
}

static int zd_tables_init()
{
    static std::mutex mu; static bool done[64];   // devices whose __constant__ copies are loaded (contexts may run on several host threads)
    int dev = 0; if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return ZMT_ST_CUDA;
    std::lock_guard<std::mutex> guard(mu);
    if (done[dev]) return ZMT_ST_OK;
    static const int16_t LLn[36] = { 4,3,2,2,2,2,2,2,2,2,2,2,2,1,1,1,2,2,2,2,2,2,2,2,2,3,2,1,1,1,1,1,-1,-1,-1,-1 };
    static const int16_t MLn[53] = { 1,4,3,2,2,2,2,2,2,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,-1,-1,-1,-1,-1,-1,-1 };
    static const int16_t OFn[29] = { 1,1,1,1,1,1,2,2,2,1,1,1,1,1,1,1,1,1,1,1,1,1,1,1,-1,-1,-1,-1,-1 };
    static const uint32_t LLb[36] = { 0,1,2,3,4,5,6,7,8,9,10,11,12,13,14,15,16,18,20,22,24,28,32,40,48,64,128,256,512,1024,2048,4096,8192,16384,32768,65536 };
    static const uint8_t  LLx[36] = { 0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,6,7,8,9,10,11,12,13,14,15,16 };
    static const uint32_t MLb[53] = { 3,4,5,6,7,8,9,10,11,12,13,14,15,16,17,18,19,20,21,22,23,24,25,26,27,28,29,30,31,32,33,34,35,37,39,41,43,47,51,59,67,83,99,131,259,515,1027,2051,4099,8195,16387,32771,65539 };
    static const uint8_t  MLx[53] = { 0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,1,1,1,1,2,2,3,3,4,4,5,7,8,9,10,11,12,13,14,15,16 };
    ZFseDTable t;
    zd_build_dtable(t, LLn, 36, 6); if (cudaMemcpyToSymbol(d_fse_ll, &t, sizeof(t)) != cudaSuccess) return ZMT_ST_CUDA;
    zd_build_dtable(t, OFn, 29, 5); if (cudaMemcpyToSymbol(d_fse_of, &t, sizeof(t)) != cudaSuccess) return ZMT_ST_CUDA;
    zd_build_dtable(t, MLn, 53, 6); if (cudaMemcpyToSymbol(d_fse_ml, &t, sizeof(t)) != cudaSuccess) return ZMT_ST_CUDA;
    cudaMemcpyToSymbol(d_ll_base, LLb, sizeof(LLb)); cudaMemcpyToSymbol(d_ml_base, MLb, sizeof(MLb));
    cudaMemcpyToSymbol(d_ll_bits, LLx, sizeof(LLx)); cudaMemcpyToSymbol(d_ml_bits, MLx, sizeof(MLx));
    if (cudaGetLastError() != cudaSuccess) return ZMT_ST_CUDA;
    if (cudaDeviceSynchronize() != cudaSuccess) return ZMT_ST_CUDA;    // the kernels run on non-blocking streams: nothing else orders the table copies before them
    done[dev] = true;
    return ZMT_ST_OK;
}

static inline uint32_t h_rd32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }

// Walk one zstd frame on the host (frame header + 3-byte block headers + the two section headers of every
// compressed block).  `base_off` = offset of the frame's first byte inside the batch input buffer.
// Appends block descriptors (scratch offsets assigned from *scratch_used).  Returns ZMT_ST_*.
extern "C" int zmt_zstd_scan_frame_host(const uint8_t* frame, size_t n, uint64_t base_off, uint32_t frame_idx,
                                        void* blocks_out, uint32_t* nblocks_io, uint32_t max_blocks,
                                        uint64_t* scratch_used, uint64_t* content_size, uint32_t* needs_seq)
{
    return zmt_zstd_scan_frame_host2(frame, n, base_off, frame_idx, blocks_out, nblocks_io, max_blocks, scratch_used, content_size, needs_seq, nullptr);
}

// same, for frames whose length is not known in advance (plain .zst streams): *consumed receives the frame length
extern "C" int zmt_zstd_scan_frame_host2(const uint8_t* frame, size_t n, uint64_t base_off, uint32_t frame_idx,
                                         void* blocks_out, uint32_t* nblocks_io, uint32_t max_blocks,
                                         uint64_t* scratch_used, uint64_t* content_size, uint32_t* needs_seq, size_t* consumed)
{
    *needs_seq = 0;
    ZBlk* out = (ZBlk*)blocks_out;
    if (n < 6 || h_rd32(frame) != 0xFD2FB528u) return n < 6 ? ZMT_ST_TRUNCATED : ZMT_ST_BAD_MAGIC;
    const uint32_t fhd = frame[4], fcs = fhd >> 6, single = (fhd >> 5) & 1, did = fhd & 3;
    if (fhd & 0x08) return ZMT_ST_BAD_HEADER;
    const bool has_chk = (fhd & 0x04) != 0;                          // XXH64 content checksum after the last block (verified on the device)
    if (did) return ZMT_ST_UNSUPPORTED;                               // dictionaries: not on the reference path
    size_t pos = 5 + (single ? 0 : 1);
    const size_t fl = fcs == 0 ? (single ? 1 : 0) : fcs == 1 ? 2 : fcs == 2 ? 4 : 8;
    if (n < pos + fl) return ZMT_ST_TRUNCATED;
    uint64_t cs = 0;
    if (fl == 1) cs = frame[pos]; else if (fl == 2) cs = (uint64_t)(frame[pos] | (frame[pos + 1] << 8)) + 256;
    else if (fl == 4) cs = h_rd32(frame + pos); else if (fl == 8) cs = (uint64_t)h_rd32(frame + pos) | ((uint64_t)h_rd32(frame + pos + 4) << 32);
    pos += fl;
    const bool no_size = fl == 0;                                     // streamed frame: size from the blocks (bound: 128 KiB per compressed block)
    uint64_t bound = 0;
    if (has_chk) *needs_seq |= ZF_CHECKSUM;
    if (no_size) *needs_seq |= ZF_NO_SIZE;
    bool first = true;
    uint32_t last_huf = ZB_NONE, cur_src[3] = { ZB_NONE, ZB_NONE, ZB_NONE };     // block that last described the Huffman tree / each sequence table
    for (;;) {
        if (n - pos < 3) return ZMT_ST_TRUNCATED;
        const uint32_t bh = frame[pos] | (frame[pos + 1] << 8) | ((uint32_t)frame[pos + 2] << 16); pos += 3;
        const uint32_t last = bh & 1, type = (bh >> 1) & 3, bs = bh >> 3;
        if (type == 3 || bs > 128 * 1024) return ZMT_ST_BLOCK;
        if (*nblocks_io >= max_blocks) return ZMT_ST_DST_SMALL;
        ZBlk& B = out[*nblocks_io];
        memset(&B, 0, sizeof(B));
        B.frame = frame_idx; B.type = type; B.first = first ? 1 : 0; B.comp_off = base_off + pos;
        bound += type == ZB_CMP ? 128 * 1024 : bs;
        if (type == ZB_RAW) { if (n - pos < bs) return ZMT_ST_TRUNCATED; B.comp_size = bs; B.regen_hint = bs; pos += bs; }
        else if (type == ZB_RLE) { if (n - pos < 1) return ZMT_ST_TRUNCATED; B.comp_size = 1; B.regen_hint = bs; pos += 1; }
        else {
            if (n - pos < bs || bs < 2) return ZMT_ST_TRUNCATED;
            const uint8_t* s = frame + pos;
            const uint32_t b0 = s[0], lt = b0 & 3, sf = (b0 >> 2) & 3;
            uint32_t lregen, lcomp, lhdr;
            if (lt < 2) {
                if (sf == 0 || sf == 2) { lregen = b0 >> 3; lhdr = 1; }
                else if (sf == 1) { if (bs < 2) return ZMT_ST_BLOCK; lregen = (b0 >> 4) | ((uint32_t)s[1] << 4); lhdr = 2; }
                else { if (bs < 3) return ZMT_ST_BLOCK; lregen = (b0 >> 4) | ((uint32_t)s[1] << 4) | ((uint32_t)s[2] << 12); lhdr = 3; }
                lcomp = lt == 0 ? lregen : 1;
            } else {
                if (bs < 5) return ZMT_ST_BLOCK;
                if (sf < 2) { const uint32_t v = s[0] | (s[1] << 8) | ((uint32_t)s[2] << 16); lregen = (v >> 4) & 0x3FF; lcomp = (v >> 14) & 0x3FF; lhdr = 3; }
                else if (sf == 2) { const uint32_t v = h_rd32(s); lregen = (v >> 4) & 0x3FFF; lcomp = (v >> 18) & 0x3FFF; lhdr = 4; }
                else { const uint64_t v = (uint64_t)h_rd32(s) | ((uint64_t)s[4] << 32); lregen = (uint32_t)((v >> 4) & 0x3FFFF); lcomp = (uint32_t)((v >> 22) & 0x3FFFF); lhdr = 5; }
            }
            if ((uint64_t)lhdr + lcomp + 1 > bs) return ZMT_ST_BLOCK;
            const uint8_t* q = s + lhdr + lcomp; const uint32_t qn = bs - lhdr - lcomp;
            uint32_t nseq; const uint32_t q0 = q[0];
            if (q0 == 0) nseq = 0; else if (q0 < 128) nseq = q0;
            else if (q0 < 255) { if (qn < 2) return ZMT_ST_BLOCK; nseq = ((q0 - 128) << 8) + q[1]; }
            else { if (qn < 3) return ZMT_ST_BLOCK; nseq = q[1] + (q[2] << 8) + 0x7F00; }
            // state across blocks visible in the headers: treeless literals, FSE-coded weights are fine block-parallel,
            // any non-predefined sequence table mode may be followed by Repeat_Mode -> frame-sequential pass
            {
                const uint32_t used = q0 == 0 ? 1u : q0 < 128 ? 1u : q0 < 255 ? 2u : 3u;
                if (lt == 3) *needs_seq |= ZF_NEEDS_SEQ;
                if (nseq && qn > used && q[used] != 0) *needs_seq |= ZF_NEEDS_SEQ;
                const uint32_t me = *nblocks_io;
                B.huf_src = ZB_SELF;
                if (lt == 2) last_huf = me; else if (lt == 3) B.huf_src = last_huf;
                B.ll_src = B.of_src = B.ml_src = ZB_SELF;
                if (nseq && qn > used) {
                    uint32_t* const dst3[3] = { &B.ll_src, &B.of_src, &B.ml_src };
                    for (uint32_t t = 0; t < 3; t++) {
                        const uint32_t mode = (q[used] >> (6 - 2 * t)) & 3;
                        if (mode == 0) cur_src[t] = ZB_PREDEF; else if (mode != 3) cur_src[t] = me;
                        *dst3[t] = (mode == 3) ? cur_src[t] : (mode == 0 ? ZB_PREDEF : ZB_SELF);
                    }
                }
            }
            B.comp_size = bs; B.regen_hint = lregen; B.nseq = nseq;
            B.seq_off = *scratch_used; *scratch_used += (((uint64_t)nseq * sizeof(ZDSeq)) + 15) & ~15ull;
            B.lit_off = *scratch_used; *scratch_used += ((uint64_t)lregen + 15) & ~15ull;
            pos += bs;
        }
        (*nblocks_io)++;
        first = false;
        if (last) break;
    }
    if (has_chk) { if (n - pos < 4) return ZMT_ST_TRUNCATED; pos += 4; }
    *content_size = no_size ? bound : cs;
    if (consumed) { *consumed = pos; return ZMT_ST_OK; }
    return pos == n ? ZMT_ST_OK : ZMT_ST_TRAILING;
}

extern "C" size_t zmt_zstd_blk_desc_bytes(void) { return sizeof(ZBlk); }

// workspace: [regen u32 x nblocks][done u32 x nblocks][blk_out u64 x nblocks][expect u64 x nframes][scratch ...]
extern "C" size_t zmt_zstdd_workspace_bytes(uint32_t nframes, uint32_t nblocks, uint64_t scratch_bytes)
{
    return (size_t)(((uint64_t)nblocks * 4 + 255) & ~255ull) * 2 + (((uint64_t)nblocks * 8 + 255) & ~255ull) + (((uint64_t)nframes * 8 + 255) & ~255ull)
           + 256 + (size_t)((((uint64_t)nframes / ZX_WIN + 2) * 8 + 255) & ~255ull) + 3 * (size_t)(((uint64_t)nblocks * 4 + 255) & ~255ull) + scratch_bytes + 1024;
}

// d_blocks: nblocks descriptors (device copy of what zmt_zstd_scan_frame_host produced); d_frame_first_blk: nframes+1;
// d_expect: content size per frame (from the frame headers)
extern "C" int zmt_zstd_decompress_device(const void* d_in, const void* d_blocks, uint32_t nblocks, const uint32_t* d_frame_first_blk,
                                          const uint64_t* d_expect, const uint32_t* d_frame_seq, uint32_t nframes, void* d_out, const uint64_t* d_out_off,
                                          uint64_t* d_out_size, uint32_t* d_status, void* d_work, void* stream_)
{
    cudaStream_t stream = (cudaStream_t)stream_;
    if (nframes == 0) return ZMT_ST_OK;
    const int ti = zd_tables_init(); if (ti != ZMT_ST_OK) return ti;
    uint8_t* w = (uint8_t*)d_work;
    uint32_t* regen = (uint32_t*)w; w += (((uint64_t)nblocks * 4 + 255) & ~255ull);
    uint32_t* done = (uint32_t*)w; w += (((uint64_t)nblocks * 4 + 255) & ~255ull);
    uint64_t* blk_out = (uint64_t*)w; w += (((uint64_t)nblocks * 8 + 255) & ~255ull);
    w += (((uint64_t)nframes * 8 + 255) & ~255ull);
    unsigned long long* xticket = (unsigned long long*)w; w += 256;
    unsigned long long* xwbase = (unsigned long long*)w; w += (((uint64_t)nframes / ZX_WIN + 2) * 8 + 255) & ~255ull;
    uint32_t* seq_done = (uint32_t*)w; w += (((uint64_t)nblocks * 4 + 255) & ~255ull);
    uint32_t* seq_ml = (uint32_t*)w; w += (((uint64_t)nblocks * 4 + 255) & ~255ull);
    uint32_t* lit_done = (uint32_t*)w; w += (((uint64_t)nblocks * 4 + 255) & ~255ull);
    uint8_t* scratch = w;
    cudaMemsetAsync(d_status, 0, (size_t)nframes * 4, stream);
    cudaMemsetAsync(regen, 0, (size_t)nblocks * 4, stream);
    cudaMemsetAsync(done, 0, (size_t)nblocks * 4, stream);
    zmt_prof_mark(ZMT_K_ZSTD_DECODE, stream, 0);
    if (nblocks) {
        cudaMemsetAsync(seq_done, 0, (size_t)nblocks * 4, stream);
        cudaMemsetAsync(lit_done, 0, (size_t)nblocks * 4, stream);
        static const bool no_fast = getenv("ZSTDMT_B200_NO_FAST_ENTROPY") != nullptr;      // A/B knob: warp-per-block entropy decode only
        if (!no_fast) {
            const size_t lsm = sizeof(ZLitGroup) * ZL_GROUPS * ZL_WARPS;
            cudaFuncSetAttribute(zstd_literals_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm);
            const uint32_t per = ZL_GROUPS * ZL_WARPS;
            zstd_literals_kernel<<<(nblocks + per - 1) / per, 32 * ZL_WARPS, lsm, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, nblocks, d_frame_seq, scratch, lit_done);
        }
        if (!no_fast)
        zstd_seq_predef_kernel<<<(nblocks + ZS_THREADS - 1) / ZS_THREADS, ZS_THREADS, 0, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, nblocks, d_frame_seq, scratch,
                                                                                           seq_done, seq_ml, d_status);
        zstd_entropy_kernel<<<(nblocks + ZD_WARPS - 1) / ZD_WARPS, 32 * ZD_WARPS, 0, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, nblocks, d_frame_seq, scratch, regen, d_status,
                                                                                           seq_done, seq_ml, lit_done);
        if (!no_fast) {
            zstd_entropy_dep_kernel<<<(nblocks + ZD_WARPS - 1) / ZD_WARPS, 32 * ZD_WARPS, 0, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, nblocks, d_frame_seq, scratch, regen,
                                                                                               d_status, lit_done);
            zstd_resolve_offsets_kernel<<<(nframes + ZD_WARPS - 1) / ZD_WARPS, 32 * ZD_WARPS, 0, stream>>>((const ZBlk*)d_blocks, d_frame_first_blk, d_frame_seq, scratch, d_status, nframes);
        }
        zstd_entropy_seq_kernel<<<(nframes + ZD_WARPS - 1) / ZD_WARPS, 32 * ZD_WARPS, 0, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, d_frame_first_blk, d_frame_seq,
                                                                                           scratch, regen, d_status, nframes, no_fast ? 0u : 1u);
    }
    zstd_offsets_kernel<<<(nframes + 127) / 128, 128, 0, stream>>>((const ZBlk*)d_blocks, nblocks, d_frame_first_blk, regen, blk_out, d_out_off, d_expect,
                                                                   (unsigned long long*)d_out_size, d_status, nframes);
    if (nblocks) {
        const uint32_t gmax = (uint32_t)(zd_sm_count() * (2048 / (32 * ZX_WARPS)));
        const uint32_t gneed = (nblocks + ZX_WARPS - 1) / ZX_WARPS;
        cudaMemsetAsync(xticket, 0, 8, stream);
        zstd_ticket_windows_kernel<<<1, 256, 0, stream>>>(d_frame_first_blk, nframes, xwbase);
        zstd_execute_kernel<<<gneed < gmax ? gneed : gmax, 32 * ZX_WARPS, 0, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, nblocks, scratch, regen, blk_out,
                                                                                     d_out_off, (uint8_t*)d_out, done, d_status, xticket, d_frame_first_blk, xwbase, nframes);
        zstd_checksum_kernel<<<(nframes + ZD_WARPS - 1) / ZD_WARPS, 32 * ZD_WARPS, 0, stream>>>((const uint8_t*)d_in, (const ZBlk*)d_blocks, d_frame_first_blk, d_frame_seq,
                                                                                           (const uint8_t*)d_out, d_out_off, (const unsigned long long*)d_out_size, d_status, nframes);
    }
    zmt_prof_mark(ZMT_K_ZSTD_DECODE, stream, 1);
    return cudaGetLastError() == cudaSuccess ? ZMT_ST_OK : ZMT_ST_CUDA;
}
