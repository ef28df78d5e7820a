// compress_b200/csrc/b2c_zstd_enc.cuh -- zstd chunk encoder for sm_100a: entropy stages, framing, work records.
//
// Turns N independent chunks (<= 64 KiB at level 1, <= 128 KiB at levels 2-3) into N complete zstd frames (what one zstd.Encoder.EncodeAll call does
// per chunk, zstd/encoder.go:722-839) or bare blocks.  Replaces, for the GPU path, the reference's
//   zstd/enc_fast.go:294-531  fastEncoder.EncodeNoHist      (match finding)
//   zstd/blockenc.go:481-826  blockEnc.encode               (entropy stage, byte-identical here)
//   zstd/frameenc.go:25-92    frameHeader.appendTo
//   zstd/internal/xxhash      XXH64 frame checksum
//
// B200-first design: a pipeline of four kernels on one stream, each shaped after the parallelism its stage really has, with
// a per-chunk work record (ChunkWork header + a slab of the work pool) in HBM/L2 between them:
//   K1 parse    b2c_lz.cuh: the tile-ordered match finder (levels 1-3; also the S2 / Snappy block encoders), with the
//               literal and sequence-code histograms counted as the literals and codes are written
//   K2 tables   one 4-warp CTA per chunk: the Huffman table (reference tie-breaking) and the three FSE
//               tables are tiny serial problems -- thousands of them run side by side.
//   K3 chains   one LANE per (chunk, tANS chain): the reference's serial state walk, 32 chunks per warp.
//   K4 pack     one CTA per chunk: code-length / bit-count prefix sums, every thread packs its own bit
//               range of the 4 Huffman streams and of the sequence bitstream into a staging buffer,
//               headers, one coalesced write-back (raw / RLE block fallbacks included).
//   K5 xxh64    four lanes per chunk (the four XXH64 accumulators).
// The parse differs from the reference's serial greedy parse; the entropy stage is byte-identical to
// blockEnc.encode for the same (literals, sequences) -- tests/check_util.py verifies both properties.
// This file: work record and pool layout, S2 tag emitters, K2..K5.
#pragma once
#include "b2c_common.cuh"
#include "b2c_fse.cuh"
#include "b2c_huff.cuh"
#include "b2c_seq.cuh"

namespace b2c {

constexpr uint32_t ENC_MAX_CHUNK = 1u << 16;   // block size of zstd level 1 and of the S2 block encoders
#ifndef PACK_THREADS
#define PACK_THREADS 512
#endif
#ifndef PACK_SEQ_UNROLL
#define PACK_SEQ_UNROLL 1
#endif
#ifndef PACK_SEQ_COMBINE
#define PACK_SEQ_COMBINE 1   // 1: state bits of the three chains in one append, LL+ML extra bits in one
#endif
#ifndef PACK_BITS_LUT
#define PACK_BITS_LUT 1      // extra-bit counts from a 2 x 64 byte shared-memory table instead of compare chains
#endif
#ifndef PACK_MIN_CTAS
#define PACK_MIN_CTAS 2   // two CTAs per SM: caps the kernel at 64 registers per thread
#endif
constexpr int PACK_UNROLL = PACK_SEQ_UNROLL;   // unroll factor of the two per-sequence loops
constexpr int PACK_NT = PACK_THREADS;     // K4 threads per CTA (a multiple of 128: four Huffman streams)

enum { ENC_FLAG_CRC = 1, ENC_FLAG_FRAME = 2 };

// Per-chunk work record handed from kernel to kernel (global memory, L2 resident for the active chunks): a small
// header (this struct) plus one slab of the work pool holding the arrays whose size depends on the block size
// (literals, per-sequence values, codes, state bits; layout below, sized by the host per level).
struct alignas(16) ChunkWork {
    uint32_t n, nseq, nlit, kind;          // kind: 0 compressed candidate, 1 raw block, 2 RLE block, 3 too big
    uint32_t rleLen, hufStatus, hufTableLog, tableDescLen;
    uint32_t maxSym[3], pad0;
    uint32_t mode[3], pad1;                // 0 predefined, 1 RLE, 2 FSE
    uint32_t ncountLen[3], pad2;
    uint32_t finalState[3], pad3;
    unsigned long long xxh;
    uint32_t litHist[256];
    uint32_t seqHist[3][64];
    uint16_t ctVal[256];
    uint8_t ctBits[256];
    uint8_t tableDesc[320];
    uint8_t ncount[3][96];
    FseCTable tbl[3];                      // the table each chain uses (new, predefined copy, or RLE)
};

// Frame mode (b2c_zstd_encode_frames_*): chunk i is block `i` of the batch's block list -- `len` bytes at src_base + off,
// preceded (in the same frame, contiguous in memory) by `hist` bytes the match finder may refer to (fastBase.hist /
// addBlock, zstd/enc_base.go:57-199).  Bit 0 of flags: last block of its frame (blockHeader.setLast, blockenc.go:120).
struct EncBlockDesc {
    uint64_t off;
    uint32_t len, hist, frame, flags;
};

struct ZstdEncParams {
    const EncBlockDesc *desc;     // frame mode: block descriptors (then src_stride / src_sizes are unused); else nullptr
    const uint8_t *src_base;      // chunk i at src_base + i * src_stride
    uint64_t src_stride;
    const uint32_t *src_sizes;    // per-chunk sizes (<= 65536); nullptr => all chunks are src_size_all
    uint32_t src_size_all;
    uint8_t *dst_base;
    uint64_t dst_stride;
    uint32_t dst_cap;             // capacity of every destination slot
    int64_t *out_sizes;           // bytes written per chunk, negative = error
    uint32_t nchunks;
    uint32_t flags;
    uint8_t *scratch;             // per-CTA parse scratch: gridDim.x(K1) * LzLayout<..>::SCRATCH_BYTES
    ChunkWork *work;              // [nchunks]
    uint8_t *pool;                // [nchunks] slabs of pool_stride bytes: lit | seqOF | seqLL | seqML | codes[3] | stb[3]
    uint64_t pool_stride;
    uint32_t maxseq;              // capacity of the per-sequence arrays (multiple of 16)
    uint32_t blockmax;            // largest block this launch accepts (65536 or 131072)
    uint32_t big;                 // 1: litLen / matchLen arrays are u32 (blocks > 64 KiB), 0: u16
    uint32_t level;               // 1 fastest, 2 default
    uint64_t src_total;           // non-zero: the chunks tile one buffer of src_total bytes (the last chunk is shorter)
    uint32_t *counter;            // persistent parse kernels: next chunk to hand out (zeroed before the launch)
    uint32_t chunk0;              // sub-batch offset: kernels work on chunks [chunk0, chunk0 + nchunks) of the call
    // optional debug dump (tests): per chunk {nseq, nlit, kind, litMode} + seq triples + literals
    uint32_t *dbg_hdr;            // [nchunks][4]
    uint32_t *dbg_seqs;           // [nchunks][dbg_seq_cap][3]
    uint8_t *dbg_lits;            // [nchunks][65536]
    uint32_t dbg_seq_cap;
    unsigned long long *dbg_cycles;  // optional [nchunks][16][32] per-warp stamps inside K1 (clock64)
};

#ifdef B2C_EMU
#define B2C_PHASE(k) do { } while (0)
#else
// Every warp's lane 0 stamps clock64 right after each barrier.  BAR.SYNC does not block at issue, so the stamp
// captures the warp's ARRIVAL time at the preceding barrier; the release time is the maximum over warps.
#define B2C_PHASE(k)                                                                                   \
    do {                                                                                               \
        if (P.dbg_cycles && (threadIdx.x & 31) == 0)                                                   \
            P.dbg_cycles[((uint64_t)chunk * 16 + (k)) * 32 + (threadIdx.x >> 5)] = (unsigned long long)clock64(); \
    } while (0)
#endif

B2C_DEV uint32_t chunk_size(const ZstdEncParams &P, uint32_t c) {
    if (P.desc) return P.desc[c].len;
    if (P.src_sizes) return P.src_sizes[c];
    if (P.src_total) {
        const uint64_t off = (uint64_t)c * P.src_stride;
        return (uint32_t)(P.src_total - off < P.src_size_all ? P.src_total - off : P.src_size_all);
    }
    return P.src_size_all;
}
B2C_DEV const uint8_t *chunk_src(const ZstdEncParams &P, uint32_t c) {
    return P.desc ? P.src_base + P.desc[c].off : P.src_base + (uint64_t)c * P.src_stride;
}
B2C_DEV uint32_t chunk_hist(const ZstdEncParams &P, uint32_t c) { return P.desc ? P.desc[c].hist : 0u; }
B2C_DEV uint32_t chunk_last(const ZstdEncParams &P, uint32_t c) { return P.desc ? (P.desc[c].flags & 1u) : 1u; }

// ---- work pool layout (one slab per chunk) ----
B2C_DEV uint32_t wk_off_lit() { return 0; }
B2C_DEV uint32_t wk_off_of(const ZstdEncParams &P) { return (P.blockmax + 64 + 15) & ~15u; }
B2C_DEV uint32_t wk_off_ll(const ZstdEncParams &P) { return wk_off_of(P) + 4 * P.maxseq; }
B2C_DEV uint32_t wk_off_ml(const ZstdEncParams &P) { return wk_off_ll(P) + (P.big ? 4u : 2u) * P.maxseq; }
B2C_DEV uint32_t wk_off_codes(const ZstdEncParams &P) { return wk_off_ml(P) + (P.big ? 4u : 2u) * P.maxseq; }
B2C_DEV uint32_t wk_off_stb(const ZstdEncParams &P) { return wk_off_codes(P) + 3 * P.maxseq; }
B2C_DEV uint8_t *wk_slab(const ZstdEncParams &P, uint32_t chunk) { return P.pool + (uint64_t)chunk * P.pool_stride; }
B2C_DEV uint8_t *wk_lit(const ZstdEncParams &P, uint32_t chunk) { return wk_slab(P, chunk); }
B2C_DEV uint32_t *wk_of(const ZstdEncParams &P, uint32_t chunk) { return reinterpret_cast<uint32_t *>(wk_slab(P, chunk) + wk_off_of(P)); }
B2C_DEV uint8_t *wk_codes(const ZstdEncParams &P, uint32_t chunk, int c) { return wk_slab(P, chunk) + wk_off_codes(P) + (uint32_t)c * P.maxseq; }
B2C_DEV uint16_t *wk_stb(const ZstdEncParams &P, uint32_t chunk, int c) {
    return reinterpret_cast<uint16_t *>(wk_slab(P, chunk) + wk_off_stb(P)) + (uint32_t)c * P.maxseq;
}
// host side of the layout: slab bytes for a block size (maxseq = blockmax / 4 + 64: a match is at least 4 bytes)
static inline uint32_t wk_maxseq(uint32_t blockmax) { return blockmax / 4 + 64; }
static inline uint64_t wk_pool_stride(uint32_t blockmax) {
    const uint64_t ms = wk_maxseq(blockmax), lenb = blockmax > 65536 ? 4 : 2;
    return (((uint64_t)blockmax + 64 + 15) & ~15ull) + 4 * ms + 2 * lenb * ms + 3 * ms + 6 * ms;
}
// litLen / matchLen-3 of sequence i (u16 arrays for blocks <= 64 KiB, u32 above)
struct WkLens {
    uint8_t *ll, *ml;
    uint32_t big;
    B2C_DEV void put(uint32_t i, uint32_t vll, uint32_t vml) const {
        if (big) { reinterpret_cast<uint32_t *>(ll)[i] = vll; reinterpret_cast<uint32_t *>(ml)[i] = vml; }
        else { reinterpret_cast<uint16_t *>(ll)[i] = (uint16_t)vll; reinterpret_cast<uint16_t *>(ml)[i] = (uint16_t)vml; }
    }
    // plain loads: for values written earlier in the SAME kernel (the read-only path is not coherent with them)
    B2C_DEV uint32_t peek_ll(uint32_t i) const { return big ? reinterpret_cast<const uint32_t *>(ll)[i] : (uint32_t)reinterpret_cast<const uint16_t *>(ll)[i]; }
    B2C_DEV uint32_t peek_ml(uint32_t i) const { return big ? reinterpret_cast<const uint32_t *>(ml)[i] : (uint32_t)reinterpret_cast<const uint16_t *>(ml)[i]; }
    B2C_DEV uint32_t get_ll(uint32_t i) const {
        return big ? B2C_LDG(reinterpret_cast<const uint32_t *>(ll) + i) : (uint32_t)B2C_LDG(reinterpret_cast<const uint16_t *>(ll) + i);
    }
    B2C_DEV uint32_t get_ml(uint32_t i) const {
        return big ? B2C_LDG(reinterpret_cast<const uint32_t *>(ml) + i) : (uint32_t)B2C_LDG(reinterpret_cast<const uint16_t *>(ml) + i);
    }
};
B2C_DEV WkLens wk_lens(const ZstdEncParams &P, uint32_t chunk) {
    WkLens w; w.ll = wk_slab(P, chunk) + wk_off_ll(P); w.ml = wk_slab(P, chunk) + wk_off_ml(P); w.big = P.big; return w;
}

// 6-byte multiplicative hash: two 32-bit multiply-adds (the reference's hashLen(u, bits, 6), zstd/hash.go:27,
// is a 64-bit multiply = ~8 integer instructions per position on the SM; table contents are an
// implementation detail, only the verified matches reach the output).
B2C_DEV uint32_t enc_hash6(uint32_t lo, uint32_t hi) {
    return lo * 0x9E3779B1u + (hi & 0xffffu) * 0x85EBCA6Bu;
}

// length of the common prefix of src[a..limitA) and src[b..], cooperative over the warp
B2C_DEV uint32_t warp_match_len(const uint8_t *src, uint32_t a, uint32_t b, uint32_t limitA) {
    unsigned lane = lane_id();
    uint32_t rem = limitA - a;
    uint32_t k = 0;
    for (;;) {
        uint32_t pos = k + 4 * lane;
        uint32_t eq = 0;
        if (pos < rem) {
            uint32_t x = ld32u(src, a + pos) ^ ld32u(src, b + pos);
            eq = x ? (uint32_t)(__ffs((int)x) - 1) >> 3 : 4u;
            uint32_t nv = rem - pos;
            if (eq > nv) eq = nv;
        }
        unsigned stop = __ballot_sync(FULLMASK, eq < 4);
        if (stop) {
            int fl = __ffs((int)stop) - 1;
            uint32_t e = __shfl_sync(FULLMASK, eq, fl);
            return k + 4 * (uint32_t)fl + e;
        }
        k += 128;
    }
}

struct ParseShared {
    uint32_t ws[40];        // block scan scratch
    uint32_t nextChunk, pad0, kind, rleLen;   // nextChunk: the chunk this CTA takes next (dynamic schedule of the persistent kernels)
    uint64_t mbar;
};
// ------------------------------------------------------------------------------------------------ K1
// ---- S2 / Snappy byte-tag emitters for offsets < 65536 (s2/encode_go.go:80-289; byte layouts pinned by the KATs of
// s2/s2_test.go:827-942).  *_size give the bytes the matching put would write.
enum { LZ_MODE_ZSTD = 0, LZ_MODE_S2 = 1, LZ_MODE_SNAPPY = 2 };

B2C_DEV uint32_t s2_lit_hdr_size(uint32_t ll) { return ll == 0 ? 0u : (ll <= 60 ? 1u : (ll <= 256 ? 2u : 3u)); }
B2C_DEV uint32_t s2_put_lit_hdr(uint8_t *d, uint32_t ll) {   // emitLiteral's tag bytes (ll <= 65536)
    if (ll == 0) return 0;
    const uint32_t n = ll - 1;
    if (n < 60) { d[0] = (uint8_t)(n << 2); return 1; }
    if (n < 256) { d[0] = 60 << 2; d[1] = (uint8_t)n; return 2; }
    d[0] = 61 << 2; d[1] = (uint8_t)n; d[2] = (uint8_t)(n >> 8);
    return 3;
}
B2C_DEV uint32_t s2_repeat_size(uint32_t off, uint32_t len) {
    len -= 4;
    if (len <= 4) return 2;
    if (len < 8 && off < 2048) return 2;
    if (len < (1 << 8) + 4) return 3;
    if (len < (1 << 16) + (1 << 8)) return 4;
    return 5;
}
B2C_DEV uint32_t s2_put_repeat(uint8_t *d, uint32_t off, uint32_t len) {   // emitRepeat, len < 2^16 + 2^8 + 4 here
    len -= 4;
    if (len <= 4) { d[0] = (uint8_t)(len << 2 | 1); d[1] = 0; return 2; }
    if (len < 8 && off < 2048) { d[1] = (uint8_t)off; d[0] = (uint8_t)((off >> 8) << 5 | len << 2 | 1); return 2; }
    if (len < (1 << 8) + 4) { len -= 4; d[2] = (uint8_t)len; d[1] = 0; d[0] = 5 << 2 | 1; return 3; }
    if (len < (1 << 16) + (1 << 8)) { len -= 1 << 8; d[3] = (uint8_t)(len >> 8); d[2] = (uint8_t)len; d[1] = 0; d[0] = 6 << 2 | 1; return 4; }
    len -= 1 << 16;
    d[4] = (uint8_t)(len >> 16); d[3] = (uint8_t)(len >> 8); d[2] = (uint8_t)len; d[1] = 0; d[0] = 7 << 2 | 1;
    return 5;
}
B2C_DEV uint32_t s2_copy_size(uint32_t off, uint32_t len) {
    if (len > 64) return (off < 2048) ? 2 + s2_repeat_size(off, len - 8) : 3 + s2_repeat_size(off, len - 60);
    return (len >= 12 || off >= 2048) ? 3u : 2u;
}
B2C_DEV uint32_t s2_put_copy(uint8_t *d, uint32_t off, uint32_t len) {   // emitCopy, offset < 65536
    if (len > 64) {
        uint32_t o;
        if (off < 2048) { d[1] = (uint8_t)off; d[0] = (uint8_t)((off >> 8) << 5 | (8 - 4) << 2 | 1); len -= 8; o = 2; }
        else { d[2] = (uint8_t)(off >> 8); d[1] = (uint8_t)off; d[0] = 59 << 2 | 2; len -= 60; o = 3; }
        return o + s2_put_repeat(d + o, off, len);
    }
    if (len >= 12 || off >= 2048) { d[2] = (uint8_t)(off >> 8); d[1] = (uint8_t)off; d[0] = (uint8_t)((len - 1) << 2 | 2); return 3; }
    d[1] = (uint8_t)off; d[0] = (uint8_t)((off >> 8) << 5 | (len - 4) << 2 | 1);
    return 2;
}
B2C_DEV uint32_t snappy_copy_size(uint32_t off, uint32_t len) {
    uint32_t sz = 0;
    while (len > 64) { sz += 3; len -= 60; }
    return sz + ((len >= 12 || off >= 2048) ? 3u : 2u);
}
B2C_DEV uint32_t snappy_put_copy(uint8_t *d, uint32_t off, uint32_t len) {   // emitCopyNoRepeat, offset < 65536
    uint32_t o = 0;
    while (len > 64) { d[o + 2] = (uint8_t)(off >> 8); d[o + 1] = (uint8_t)off; d[o] = 59 << 2 | 2; len -= 60; o += 3; }
    if (len >= 12 || off >= 2048) { d[o + 2] = (uint8_t)(off >> 8); d[o + 1] = (uint8_t)off; d[o] = (uint8_t)((len - 1) << 2 | 2); return o + 3; }
    d[o + 1] = (uint8_t)off; d[o] = (uint8_t)((off >> 8) << 5 | (len - 4) << 2 | 1);
    return o + 2;
}

// ------------------------------------------------------------------------------------------------ K2
// One 128-thread CTA per chunk.  Warp 0 builds the Huffman table cooperatively (rank sort with 32 lanes, the
// serial tree / setMaxHeight / table serialisation on lane 0); lane 0 of warps 1..3 builds one FSE table each.
#ifndef TABLES_MIN_CTAS
#define TABLES_MIN_CTAS 8      // resident K2 CTAs per SM the register allocation is held to
#endif
constexpr int TABLES_NT = 128;
struct TablesShared {
    HufWork hw;
    SeqWork sw;
};
B2C_DEV void zstd_tables_chunk(TablesShared *ts, const ZstdEncParams &P, uint32_t chunk) {
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    ChunkWork *W = P.work + chunk;
    const uint32_t nseq = W->nseq, nlit = W->nlit;
    if (P.dbg_hdr && W->kind != 3) {
        // debug dump of the parse (tests): the sequences (of raw blocks too) and the literals of compressed candidates
        const WkLens wlen = wk_lens(P, chunk);
        const uint32_t *wof = wk_of(P, chunk);
        for (uint32_t i = tid; i < nseq && i < P.dbg_seq_cap && i < P.maxseq; i += TABLES_NT) {
            uint32_t *d = P.dbg_seqs + ((uint64_t)chunk * P.dbg_seq_cap + i) * 3;
            d[0] = wlen.get_ll(i); d[1] = wlen.get_ml(i); d[2] = wof[i];
        }
        if (W->kind == 0) {
            const uint8_t *lit = wk_lit(P, chunk);
            for (uint32_t i = tid; i < nlit; i += TABLES_NT) P.dbg_lits[(uint64_t)chunk * P.blockmax + i] = lit[i];
        }
    }
    if (P.dbg_hdr) __syncthreads();      // every warp has read the parse's kind before a table error may change it
    if (W->kind != 0) return;
    if (w == 0) {
        HufWork *hw = &ts->hw;
        for (uint32_t s = lane; s < 256; s += 32) hw->count[s] = W->litHist[s];
        if (lane == 0) { hw->status = HUF_INCOMPRESSIBLE; hw->tableDescLen = 0; hw->tableLog = 0; }
        __syncwarp();
        if (nlit > 16) huf_build_table(hw, nlit, lane, 32, -1);
        __syncwarp();
        if (hw->status == HUF_OK) {
            for (uint32_t s = lane; s < 256; s += 32) { W->ctVal[s] = hw->ctVal[s]; W->ctBits[s] = hw->ctBits[s]; }
            for (uint32_t i = lane; i < hw->tableDescLen; i += 32) W->tableDesc[i] = hw->tableDesc[i];
        }
        if (lane == 0) { W->hufStatus = (uint32_t)hw->status; W->hufTableLog = hw->tableLog; W->tableDescLen = hw->tableDescLen; }
    } else {
        const int which = (int)w - 1;
        SeqWork *sw = &ts->sw;
        for (uint32_t s = lane; s < 64; s += 32) sw->hist[which][s] = W->seqHist[which][s];
        if (lane == 0) sw->maxSym[which] = W->maxSym[which];
        __syncwarp();
        seq_build_table(sw, which, nseq, wk_codes(P, chunk, which)[0], lane);
        __syncwarp();
        // publish the table this chain will use
        const FseCTable *t = seq_table(sw, which);
        const uint32_t *s32 = reinterpret_cast<const uint32_t *>(t);
        uint32_t *d32 = reinterpret_cast<uint32_t *>(&W->tbl[which]);
        for (uint32_t i = lane; i < sizeof(FseCTable) / 4; i += 32) d32[i] = s32[i];
        for (uint32_t i = lane; i < sw->ncountLen[which] && i < 96; i += 32) W->ncount[which][i] = sw->ncount[which][i];
        if (lane == 0) {
            W->mode[which] = sw->mode[which]; W->ncountLen[which] = sw->ncountLen[which];
            if (sw->ncountLen[which] == SEQ_TABLE_ERR) { W->ncountLen[which] = 0; W->kind = 1; }  // internal error: store raw
        }
    }
}

// The chunk loop of a K2 CTA (chunks first, first + stride, ...).  K2 is bound by instruction issue, not by latency:
// its serial stretches run with one active lane, and at 8 CTAs per SM the schedulers are about half busy.  Splitting
// the Huffman work over two warps (codes / table description, pipelined over consecutive chunks) was measured and
// changed nothing; what helps is fewer warp instructions (e.g. the sort over 2^ceil(log2(symbolLen)) keys).
B2C_DEV void zstd_tables_loop(TablesShared *ts, const ZstdEncParams &P, uint32_t first, uint32_t stride) {
    for (uint32_t c = first; c < P.nchunks; c += stride) {
        zstd_tables_chunk(ts, P, c);
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ K3
// One lane per (chunk, chain): CTA = 96 threads = 3 warps; warp c walks chain c of 32 consecutive chunks.
// Per-lane tables live in shared memory, interleaved so that lane l only ever touches bank l:
// 128 words of packed u16 next-states + 64 words of (deltaNbBits | (deltaFindState + 512) << 21).
constexpr int CHAIN_NT = 96;
constexpr int CHAIN_XXH_NT = 128;   // optional extra warps of a chains CTA: XXH64 of its 32 chunks, four lanes per chunk
constexpr uint32_t CHAIN_SMEM_WORDS_PER_LANE = 64 + 56;   // 256 x u8 next-state offsets + 56 x u32 symbol transforms
constexpr uint32_t CHAIN_SMEM_BYTES = CHAIN_NT * CHAIN_SMEM_WORDS_PER_LANE * 4;
// K3: one lane per (chunk, table) walks the tANS state chain from the last sequence to the first
// (blockenc.go:757-803 restated as three independent recurrences) and stores, per sequence, the bits it emits:
// stb[i] = value | nbBits << 12.  The recurrence is latency-bound, so the loop keeps the dependent path to
// add/shift/add + one shared-memory load per step: codes arrive eight at a time (one 8-byte load, requested two
// blocks ahead), their symbol transforms are fetched up front, results leave as one 16-byte store per 8 steps.
// Per-lane tables are interleaved so lane l only touches bank l: next states are kept as u8 offsets from tableSize
// (4 per word), 45 KB per CTA, so five CTAs fit an SM and a 16 384-chunk batch is a single wave.
B2C_DEV void zstd_chains_block(uint32_t *smem32, const ZstdEncParams &P, uint32_t chunk0) {
    const unsigned tid = threadIdx.x, lane = tid & 31, which = tid >> 5;
    const uint32_t chunk = chunk0 + lane;
    const bool live = chunk < P.nchunks && P.work[chunk < P.nchunks ? chunk : 0].kind == 0;
    ChunkWork *W = P.work + (live ? chunk : 0);
    uint32_t *st32 = smem32 + which * 32 * CHAIN_SMEM_WORDS_PER_LANE;  // this warp's region
    uint8_t *tState = reinterpret_cast<uint8_t *>(st32 + lane);        // element i at byte (i >> 2) * 128 + (i & 3)
    uint32_t *tSym = st32 + 64 * 32 + lane;                            // element i of lane l at word i * 32 + l
#define TSTATE(i) tState[(((uint32_t)(i)) >> 2) * 128 + (((uint32_t)(i)) & 3)]
    uint32_t nseq = 0, useRLE = 1, tableLog = 0, tableSize = 1;
    if (live) {
        const FseCTable *t = &W->tbl[which];
        nseq = W->nseq; useRLE = t->useRLE; tableLog = t->tableLog; tableSize = 1u << tableLog;
        if (!useRLE) {
            const uint32_t *sw = reinterpret_cast<const uint32_t *>(t->stateTable);
            const uint32_t ts2 = tableSize / 2;
            for (uint32_t i = 0; i < ts2; i += 2) {      // tableSize >= 32: four states per word
                const uint32_t v0 = sw[i], v1 = sw[i + 1];
                st32[(i >> 1) * 32 + lane] = ((v0 & 0xffff) - tableSize) | (((v0 >> 16) - tableSize) << 8) |
                                             (((v1 & 0xffff) - tableSize) << 16) | (((v1 >> 16) - tableSize) << 24);
            }
            const uint32_t sl = t->symbolLen;
            for (uint32_t i = 0; i < 56; i++)
                tSym[i * 32] = (i < sl) ? (t->deltaNbBits[i] | ((uint32_t)((int32_t)t->deltaFindState[i] + 512) << 21)) : 0u;
        }
    }
    __syncwarp();
    const uint8_t *codes = wk_codes(P, live ? chunk : 0, (int)which);
    uint16_t *stb = wk_stb(P, live ? chunk : 0, (int)which);
    uint32_t state = 0;
    const bool run = live && !useRLE && nseq >= 1;
    if (run) {
        const uint32_t e = tSym[(codes[nseq - 1] < 56u ? codes[nseq - 1] : 0u) * 32];
        const uint32_t dnb = e & 0x1fffffu;
        const int32_t dfs = (int32_t)(e >> 21) - 512;
        const uint32_t nbBitsOut = (dnb + (1u << 15)) >> 16;
        const int32_t im = (int32_t)((nbBitsOut << 16) - dnb);
        state = tableSize + TSTATE((im >> nbBitsOut) + dfs);
    }
    // sequences nseq-2 .. 0 in blocks of eight (block k = sequences 8k .. 8k+7), top block first
    const int32_t top = run ? (int32_t)nseq - 2 : -1;
    const int32_t blk = top >> 3;                                  // -1 when there is nothing to do
    const uint32_t nblk = warp_max((uint32_t)(blk + 1));
    const uint2 *c8 = reinterpret_cast<const uint2 *>(codes);
    uint2 cwA = make_uint2(0, 0), cwB = make_uint2(0, 0);
    if (blk >= 0) cwA = c8[blk];
    if (blk >= 1) cwB = c8[blk - 1];
    for (uint32_t it = 0; it < nblk; it++) {
        const int32_t k = blk - (int32_t)it;
        if (k >= 0) {
            uint2 cwC = make_uint2(0, 0);
            if (k >= 2) cwC = c8[k - 2];
            uint32_t e[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                uint32_t code = (((j < 4) ? cwA.x : cwA.y) >> (8 * (j & 3))) & 63u;
                if (code >= 56u) code = 0;     // bytes past the last sequence are not codes
                e[j] = tSym[code * 32];
            }
            uint32_t o[4] = {0, 0, 0, 0};
#pragma unroll
            for (int pos = 7; pos >= 0; pos--) {
                if (8 * k + pos <= top) {
                    const uint32_t nb = (state + (e[pos] & 0x1fffffu)) >> 16;
                    o[pos >> 1] |= ((state & ((1u << nb) - 1)) | (nb << 12)) << (16 * (pos & 1));
                    state = tableSize + TSTATE((int32_t)(state >> nb) + (int32_t)(e[pos] >> 21) - 512);
                }
            }
            *reinterpret_cast<uint4 *>(stb + 8 * k) = make_uint4(o[0], o[1], o[2], o[3]);
            cwA = cwB; cwB = cwC;
        }
    }
    if (live) {
        if (useRLE) { for (uint32_t i = 0; i + 1 < nseq; i++) stb[i] = 0; state = 0; }
        W->finalState[which] = state;
    }
#undef TSTATE
}

// ------------------------------------------------------------------------------------------------ K4
struct PackShared {
    HufWork hw;               // only ctVal/ctBits/tableDesc*/scan/stream* hold their usual content here; two unused
                              // members are reused (two CTAs must fit an SM, there is no kilobyte to spare):
                              //   hw.count[256] = Huffman codes as (code | nbits << 16)               (PACK_PK)
                              //   hw.nsym[0..127] = extra-bit counts per LL / ML code, seqenc.go:61-97  (PACK_LLB / PACK_MLB)
    uint32_t scan[40];
    uint32_t litMode, lhSize, litPayload, pos;
};
#if PACK_BITS_LUT
#define PACK_LLB(c) ((uint32_t)ps->hw.nsym[(c) & 63])
#define PACK_MLB(c) ((uint32_t)ps->hw.nsym[64 + ((c) & 63)])
#else
#define PACK_LLB(c) seq_ll_bits(c)
#define PACK_MLB(c) seq_ml_bits(c)
#endif
#ifndef PACK_LIT_SMEM_BYTES
#define PACK_LIT_SMEM_BYTES (40 * 1024)
#endif
// K4 shared-memory plan per block size: the staging buffer holds the whole output, literals are staged when they fit.
// 64 KiB blocks: 64 K + 40 K -> two CTAs per SM; 128 KiB blocks (level 2): 128 K + 64 K -> one CTA per SM.
template <uint32_t BLOCK> struct PackCfg {
    static constexpr uint32_t STAGE_BYTES = BLOCK + 128;
    static constexpr uint32_t LIT_SMEM = (BLOCK <= 65536) ? (uint32_t)PACK_LIT_SMEM_BYTES : 64u * 1024u;
    static constexpr uint32_t SMEM_SH = STAGE_BYTES + LIT_SMEM;
    static constexpr uint32_t SMEM_BYTES = SMEM_SH + ((sizeof(PackShared) + 15) / 16) * 16;
};
constexpr uint32_t PACK_SMEM_BYTES = PackCfg<65536>::SMEM_BYTES;
static_assert(PACK_LIT_SMEM_BYTES != 40 * 1024 || 2 * (PACK_SMEM_BYTES + 1024) <= 228 * 1024, "two K4 CTAs must fit one SM");
static_assert(PackCfg<131072>::SMEM_BYTES <= 227 * 1024, "the 128 KiB K4 CTA must fit one SM");

B2C_DEV uint32_t frame_header_bytes(uint32_t n) {
    if (n == 0) return 6;
    bool single = n > 1024;
    uint32_t fh = 4 + 1 + (single ? 0 : 1);
    if (n >= 256) fh += (n >= 65536 + 256) ? 4 : 2; else if (single) fh += 1;
    return fh;
}
// frameHeader.appendTo (frameenc.go:25-92), single chunk, no dictionary
B2C_DEV uint32_t write_frame_header(uint8_t *o8, uint32_t n, bool crc) {
    uint32_t o = 0;
    o8[o++] = 0x28; o8[o++] = 0xB5; o8[o++] = 0x2F; o8[o++] = 0xFD;
    if (n == 0) { o8[o++] = 32; o8[o++] = 0; return o; }  // WithZeroFrames (encoder.go:732-751)
    bool single = n > 1024;
    uint32_t fcs = (n >= 256) ? ((n >= 65536 + 256) ? 2u : 1u) : 0u;
    o8[o++] = (uint8_t)((crc ? 4u : 0u) | (single ? 32u : 0u) | (fcs << 6));
    if (!single) {
        uint32_t ws = 1u << (32 - (uint32_t)__clz((int)n));  // WindowSize(n) (enc_base.go:42-50)
        if (ws < 1024) ws = 1024;
        o8[o++] = (uint8_t)(((32 - (uint32_t)__clz((int)(ws - 1))) - 10) << 3);
    }
    if (fcs == 0) { if (single) o8[o++] = (uint8_t)n; }
    else if (fcs == 1) { uint32_t v = n - 256; o8[o++] = (uint8_t)v; o8[o++] = (uint8_t)(v >> 8); }
    else { o8[o++] = (uint8_t)n; o8[o++] = (uint8_t)(n >> 8); o8[o++] = (uint8_t)(n >> 16); o8[o++] = (uint8_t)(n >> 24); }
    return o;
}

template <uint32_t BLOCK>
B2C_DEV void zstd_pack_chunk(uint8_t *smem, const ZstdEncParams &P, uint32_t chunk) {
    constexpr uint32_t PACK_STAGE_BYTES = PackCfg<BLOCK>::STAGE_BYTES;
    constexpr uint32_t PACK_LIT_SMEM = PackCfg<BLOCK>::LIT_SMEM;
    const unsigned tid = threadIdx.x;
    uint8_t *stage = smem;
    PackShared *ps = reinterpret_cast<PackShared *>(smem + PackCfg<BLOCK>::SMEM_SH);
    ChunkWork *W = P.work + chunk;
    const uint8_t *gsrc = chunk_src(P, chunk);
    uint8_t *gdst = P.dst_base + (uint64_t)chunk * P.dst_stride;
    const uint32_t n = W->n;
    const uint32_t lastBit = chunk_last(P, chunk);
    const bool frame = (P.flags & ENC_FLAG_FRAME) != 0;
    const bool crc = frame && (P.flags & ENC_FLAG_CRC) != 0;
    uint32_t kind = W->kind;
    if (kind == 3) { if (tid == 0) P.out_sizes[chunk] = -3; return; }
    const uint32_t nseq = W->nseq, nlit = W->nlit;
    const uint32_t fh = frame ? frame_header_bytes(n) : 0;

    if (kind == 0) {
        const uint8_t *lit = wk_lit(P, chunk);
        if (nlit <= PACK_LIT_SMEM) {
            uint8_t *ls = smem + PACK_STAGE_BYTES;
            const uint4 *g4 = reinterpret_cast<const uint4 *>(lit);
            uint4 *s4 = reinterpret_cast<uint4 *>(ls);
            for (uint32_t i = tid; i < (nlit + 15) / 16; i += PACK_NT) s4[i] = g4[i];
            lit = ls;
        }
        HufWork *hw = &ps->hw;
        // Huffman table into shared memory
        if (tid < 64) { ps->hw.nsym[tid] = (uint8_t)seq_ll_bits(tid); ps->hw.nsym[64 + tid] = (uint8_t)seq_ml_bits(tid); }
        for (uint32_t s = tid; s < 256; s += PACK_NT) { hw->ctVal[s] = W->ctVal[s]; hw->ctBits[s] = W->ctBits[s]; }
        for (uint32_t i = tid; i < W->tableDescLen; i += PACK_NT) hw->tableDesc[i] = W->tableDesc[i];
        if (tid == 0) { hw->tableDescLen = W->tableDescLen; hw->status = (int32_t)W->hufStatus; }
        __syncthreads();
        // ------------------------------------------------------------ literals section sizes
        const bool four = nlit >= 1024;
        HufEncState hst;
        uint32_t payload = 0;
        const bool hufOK = hw->status == HUF_OK;
        if (hufOK) payload = huf_enc_sizes(hw, ps->hw.count, lit, nlit, four ? 1 : 0, tid, PACK_NT, 0, &hst);
        if (tid == 0) {
            // huff0 compress(): out >= wantSize => ErrIncompressible (compress.go:155-158, WantLogLess 4)
            uint32_t mode = 2;
            if (!hufOK) mode = (hw->status == HUF_USE_RLE) ? 1u : 0u;
            else {
                uint32_t wantSize = nlit - (nlit >> 4);
                if (payload >= wantSize) mode = 0;
                else if (payload + 5 > nlit) {
                    // blockenc.go:534-544: compare with the raw representation
                    uint32_t inBits = 32 - (uint32_t)__clz((int)nlit);
                    uint32_t szRaw = inBits < 5 ? 1 : (inBits < 12 ? 2 : 3);
                    uint32_t compBits = payload ? 32 - (uint32_t)__clz((int)payload) : 0;
                    uint32_t szComp = (compBits <= 10 && inBits <= 10) ? 3 : ((compBits <= 14 && inBits <= 14) ? 4 : 5);
                    if (payload + szComp >= nlit + szRaw) mode = 0;
                }
            }
            uint32_t lh;
            if (mode == 2) {
                uint32_t inBits = 32 - (uint32_t)__clz((int)nlit);
                uint32_t compBits = payload ? 32 - (uint32_t)__clz((int)payload) : 0;
                lh = (compBits <= 10 && inBits <= 10) ? 3 : ((compBits <= 14 && inBits <= 14) ? 4 : 5);
            } else {
                uint32_t inBits = nlit ? 32 - (uint32_t)__clz((int)nlit) : 0;
                lh = inBits < 5 ? 1 : (inBits < 12 ? 2 : 3);
            }
            ps->litMode = mode; ps->lhSize = lh; ps->litPayload = payload;
        }
        __syncthreads();
        const uint32_t litMode = ps->litMode, lhSize = ps->lhSize;
        const uint32_t litOff = fh + 3 + lhSize;  // staging offset of the literal payload
        const uint32_t litBytes = (litMode == 2) ? ps->litPayload : (litMode == 1 ? 1u : nlit);
        const uint32_t nsHdr = (nseq < 128) ? 1u : (nseq < 0x7f00 ? 2u : 3u);
        const uint32_t seqOff = litOff + litBytes;
        const uint32_t tblOff = seqOff + nsHdr + 1;
        const uint32_t bsOff = tblOff + W->ncountLen[0] + W->ncountLen[1] + W->ncountLen[2];

        // ------------------------------------------------------------ sequence bitstream sizes
        const uint8_t *cLL = wk_codes(P, chunk, TBL_LL), *cOF = wk_codes(P, chunk, TBL_OF), *cML = wk_codes(P, chunk, TBL_ML);
        const uint16_t *stbLL = wk_stb(P, chunk, TBL_LL), *stbOF = wk_stb(P, chunk, TBL_OF), *stbML = wk_stb(P, chunk, TBL_ML);
        const WkLens wlen = wk_lens(P, chunk);
        const uint32_t *wof = wk_of(P, chunk);
        const uint32_t per = (nseq + PACK_NT - 1) / PACK_NT;
        uint32_t tA = tid * per, tB = tA + per;
        if (tA > nseq) tA = nseq;
        if (tB > nseq) tB = nseq;
        uint32_t mybits = 0;
#pragma unroll PACK_UNROLL
        for (uint32_t t = tA; t < tB; t++) {
            uint32_t idx = nseq - 1 - t;
            uint32_t cl = B2C_LDG(cLL + idx), co = B2C_LDG(cOF + idx), cm = B2C_LDG(cML + idx);
            mybits += PACK_LLB(cl) + PACK_MLB(cm) + co;
            if (t) mybits += (uint32_t)(B2C_LDG(stbLL + idx) >> 12) + (uint32_t)(B2C_LDG(stbOF + idx) >> 12) + (uint32_t)(B2C_LDG(stbML + idx) >> 12);
        }
        uint32_t totalBits;
        uint32_t exBits = group_scan_excl(mybits, ps->scan, 0, PACK_NT, tid, &totalBits);
        const uint32_t tlLL = W->tbl[TBL_LL].tableLog, tlOF = W->tbl[TBL_OF].tableLog, tlML = W->tbl[TBL_ML].tableLog;
        const uint32_t flushBits = tlML + tlOF + tlLL;
        const uint32_t bsBytes = (totalBits + flushBits + 1 + 7) >> 3;
        const uint32_t blockBytes = (bsOff - fh - 3) + bsBytes;  // block content size
        const uint32_t total = fh + 3 + blockBytes + (crc ? 4u : 0u);
        // blockenc.go:811-817: not smaller than the input => raw block.  Also covers staging overflow.
        const bool useRaw = (blockBytes >= n) || (total + 8 > PACK_STAGE_BYTES);
        if (!useRaw) {
            uint32_t zw = (total + 8 + 3) / 4;
            for (uint32_t i = tid; i < zw; i += PACK_NT) reinterpret_cast<uint32_t *>(stage)[i] = 0;
            __syncthreads();
            if (litMode == 2) {
                huf_enc_pack(hw, ps->hw.count, lit, four ? 1 : 0, stage, litOff, tid, PACK_NT, 0, &hst);
            } else if (litMode == 0) {
                for (uint32_t i = tid; i < nlit; i += PACK_NT) stage[litOff + i] = lit[i];
            } else if (tid == 0) {
                stage[litOff] = lit[0];
            }
            __syncthreads();  // byte stores above must not race the word atomics below
            {
                BitRun br;
                br.init(reinterpret_cast<uint32_t *>(stage), bsOff * 8 + exBits);
#pragma unroll PACK_UNROLL
                for (uint32_t t = tA; t < tB; t++) {
                    uint32_t idx = nseq - 1 - t;
                    uint32_t cl = B2C_LDG(cLL + idx), co = B2C_LDG(cOF + idx), cm = B2C_LDG(cML + idx);
                    const uint32_t vLL = wlen.get_ll(idx), vML = wlen.get_ml(idx), vOF = B2C_LDG(wof + idx);
#if PACK_SEQ_COMBINE
                    if (t) {
                        // three state flushes (<= 9 bits each) in one append: OF, ML, LL (blockenc.go:757-790)
                        uint32_t so = B2C_LDG(stbOF + idx), sm = B2C_LDG(stbML + idx), sl = B2C_LDG(stbLL + idx);
                        const uint32_t no = so >> 12, nm = sm >> 12;
                        br.add((so & 0xfff) | ((sm & 0xfff) << no) | ((sl & 0xfff) << (no + nm)), no + nm + (sl >> 12));
                    }
                    // extra bits: LL and ML (<= 16 bits each) together, then OF
                    uint32_t lb = PACK_LLB(cl), mb = PACK_MLB(cm);
                    br.add((vLL & ((1u << lb) - 1)) | ((vML & ((1u << mb) - 1)) << lb), lb + mb);
                    br.add(vOF & ((1u << co) - 1), co);
#else
                    if (t) {
                        uint32_t so = B2C_LDG(stbOF + idx), sm = B2C_LDG(stbML + idx), sl = B2C_LDG(stbLL + idx);
                        br.add(so & 0xfff, so >> 12);
                        br.add(sm & 0xfff, sm >> 12);
                        br.add(sl & 0xfff, sl >> 12);
                    }
                    uint32_t lb = PACK_LLB(cl), mb = PACK_MLB(cm);
                    br.add(vLL & ((1u << lb) - 1), lb);
                    br.add(vML & ((1u << mb) - 1), mb);
                    br.add(vOF & ((1u << co) - 1), co);
#endif
                }
                if (tB == nseq && tA < tB) {
                    // final states: ml, of, ll (blockenc.go:804-806) + end mark
                    br.add(W->finalState[TBL_ML] & ((1u << tlML) - 1), tlML);
                    br.add(W->finalState[TBL_OF] & ((1u << tlOF) - 1), tlOF);
                    br.add(W->finalState[TBL_LL] & ((1u << tlLL) - 1), tlLL);
                    br.add(1u, 1);
                }
                br.finish();
            }
            __syncthreads();
            // byte-granular headers (after all word-granular atomics)
            if (tid == 0) {
                uint32_t o = 0;
                if (frame) o = write_frame_header(stage, n, crc);
                uint32_t bh = lastBit | (2u << 1) | (blockBytes << 3);  // compressed block
                stage[o++] = (uint8_t)bh; stage[o++] = (uint8_t)(bh >> 8); stage[o++] = (uint8_t)(bh >> 16);
                // literals header (blockenc.go:153-238)
                uint64_t lh;
                if (litMode == 2) {
                    uint64_t comp = ps->litPayload;
                    if (lhSize == 3) lh = 2u | ((four ? 1u : 0u) << 2) | ((uint64_t)nlit << 4) | (comp << 14);
                    else if (lhSize == 4) lh = 2u | (2u << 2) | ((uint64_t)nlit << 4) | (comp << 18);
                    else lh = 2u | (3u << 2) | ((uint64_t)nlit << 4) | (comp << 22);
                } else {
                    uint64_t ty = (litMode == 1) ? 1u : 0u;
                    if (lhSize == 1) lh = ty | ((uint64_t)nlit << 3);
                    else if (lhSize == 2) lh = ty | (1u << 2) | ((uint64_t)nlit << 4);
                    else lh = ty | (3u << 2) | ((uint64_t)nlit << 4);
                }
                for (uint32_t k = 0; k < lhSize; k++) stage[o++] = (uint8_t)(lh >> (8 * k));
                o = seqOff;
                if (nseq < 128) stage[o++] = (uint8_t)nseq;
                else if (nseq < 0x7f00) { stage[o++] = (uint8_t)(128 + (nseq >> 8)); stage[o++] = (uint8_t)nseq; }
                else { uint32_t v = nseq - 0x7f00; stage[o++] = 255; stage[o++] = (uint8_t)v; stage[o++] = (uint8_t)(v >> 8); }
                stage[o++] = (uint8_t)((W->mode[TBL_LL] << 6) | (W->mode[TBL_OF] << 4) | (W->mode[TBL_ML] << 2));
                for (int c = 0; c < 3; c++)
                    for (uint32_t k = 0; k < W->ncountLen[c]; k++) stage[o++] = W->ncount[c][k];
                if (crc) {
                    uint32_t c32 = (uint32_t)W->xxh;
                    uint32_t e = total - 4;
                    stage[e] = (uint8_t)c32; stage[e + 1] = (uint8_t)(c32 >> 8); stage[e + 2] = (uint8_t)(c32 >> 16); stage[e + 3] = (uint8_t)(c32 >> 24);
                }
            }
            __syncthreads();
            // one coalesced write-back
            if (total <= P.dst_cap) {
                if ((reinterpret_cast<uintptr_t>(gdst) & 15) == 0) {
                    const uint4 *s4 = reinterpret_cast<const uint4 *>(stage);
                    uint4 *d4 = reinterpret_cast<uint4 *>(gdst);
                    uint32_t n16 = total / 16;
                    for (uint32_t i = tid; i < n16; i += PACK_NT) d4[i] = s4[i];
                    for (uint32_t i = n16 * 16 + tid; i < total; i += PACK_NT) gdst[i] = stage[i];
                } else {
                    for (uint32_t i = tid; i < total; i += PACK_NT) gdst[i] = stage[i];
                }
                if (tid == 0) P.out_sizes[chunk] = (int64_t)total;
            } else if (tid == 0) P.out_sizes[chunk] = -4;  // destination too small
            if (P.dbg_hdr && tid == 0) {
                uint32_t *d = P.dbg_hdr + (uint64_t)chunk * 4;
                d[0] = nseq; d[1] = nlit; d[2] = 0; d[3] = litMode;
            }
            return;
        }
        kind = 1;  // fall through to the raw block
    }

    // ---------------------------------------------------------------- raw / RLE block (+ frame)
    {
        __syncthreads();
        uint8_t *hdr = stage;
        if (tid == 0) {
            uint32_t o = 0;
            if (frame) o = write_frame_header(hdr, n, crc);
            uint32_t bh = (kind == 2) ? (lastBit | (1u << 1) | (W->rleLen << 3)) : (lastBit | (0u << 1) | (n << 3));
            hdr[o++] = (uint8_t)bh; hdr[o++] = (uint8_t)(bh >> 8); hdr[o++] = (uint8_t)(bh >> 16);
            ps->pos = o;
        }
        __syncthreads();
        const uint32_t hlen = ps->pos;
        const uint32_t body = (kind == 2) ? 1u : n;
        const bool crcHere = crc && n > 0;
        const uint32_t total = hlen + body + (crcHere ? 4u : 0u);
        if (total <= P.dst_cap) {
            for (uint32_t i = tid; i < hlen; i += PACK_NT) gdst[i] = hdr[i];
            for (uint32_t i = tid; i < body; i += PACK_NT) gdst[hlen + i] = gsrc[i];
            if (crcHere && tid < 4) gdst[hlen + body + tid] = (uint8_t)((uint32_t)W->xxh >> (8 * tid));
            if (tid == 0) P.out_sizes[chunk] = (int64_t)total;
        } else if (tid == 0) P.out_sizes[chunk] = -4;
        if (P.dbg_hdr && tid == 0) {
            uint32_t *d = P.dbg_hdr + (uint64_t)chunk * 4;
            d[0] = nseq; d[1] = nlit; d[2] = kind; d[3] = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------------ K5
// XXH64 of every chunk (xxh64_quad, b2c_common.cuh): four lanes per chunk hold the four accumulators.
B2C_DEV void zstd_xxh_quad(const ZstdEncParams &P, uint32_t chunk, unsigned q /*0..3*/, unsigned quadBaseLane) {
    const bool live = chunk < P.nchunks;
    const uint8_t *src = chunk_src(P, live ? chunk : 0);
    uint32_t n = live ? chunk_size(P, chunk) : 0;
    const bool ok = n <= P.blockmax;
    if (!ok) n = 0;
    const uint64_t h = xxh64_quad(src, n, q, quadBaseLane);
    if (q == 0 && live && ok) P.work[chunk].xxh = h;
}

#ifndef B2C_EMU
extern "C" __global__ void __launch_bounds__(TABLES_NT, TABLES_MIN_CTAS) b2c_zstd_tables_kernel(ZstdEncParams P) {
    __shared__ TablesShared ts;
    if (threadIdx.x < 3) seq_build_predef(&ts.sw, (int)threadIdx.x);
    __syncthreads();
    zstd_tables_loop(&ts, P, blockIdx.x, gridDim.x);
}
// K3 + K5 in one launch: the three chain warps of a CTA walk the tANS chains of 32 chunks; when the launch has
// CHAIN_NT + CHAIN_XXH_NT threads, four more warps compute the XXH64 of the same 32 chunks (four lanes per chunk).  Both
// are latency-bound serial recurrences that need few registers, so they hide behind each other (as its own kernel XXH64
// cost 0.44 ms per GiB; a side stream beside the parse kernel did not overlap with it on the device).
extern "C" __global__ void __launch_bounds__(CHAIN_NT + CHAIN_XXH_NT) b2c_zstd_chains_kernel(ZstdEncParams P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    if (threadIdx.x < CHAIN_NT) zstd_chains_block(reinterpret_cast<uint32_t *>(smem), P, blockIdx.x * 32);
    else {
        const unsigned t = threadIdx.x - CHAIN_NT;
        zstd_xxh_quad(P, blockIdx.x * 32 + (t >> 2), t & 3, (t & 31) & ~3u);
    }
}
extern "C" __global__ void __launch_bounds__(PACK_NT, PACK_MIN_CTAS) b2c_zstd_pack_kernel(ZstdEncParams P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    zstd_pack_chunk<65536>(smem, P, blockIdx.x);
}
extern "C" __global__ void __launch_bounds__(PACK_NT, 1) b2c_zstd_pack128_kernel(ZstdEncParams P) {
    extern __shared__ __align__(1024) uint8_t smem[];
    zstd_pack_chunk<131072>(smem, P, blockIdx.x);
}
extern "C" __global__ void __launch_bounds__(128) b2c_zstd_xxh_kernel(ZstdEncParams P) {
    unsigned gt = blockIdx.x * blockDim.x + threadIdx.x;
    zstd_xxh_quad(P, gt >> 2, gt & 3, (threadIdx.x & 31) & ~3u);
}
#endif

}  // namespace b2c
