// compress_b200/csrc/b2c_lz.cuh -- the round-2 match finder for the zstd block encoders (levels 1 and 2), sm_100a.
//
// Replaces, for the GPU path, the reference's serial match finders
//   zstd/enc_fast.go:294-531   fastEncoder.EncodeNoHist        (level 1: one table, 6-byte hash, 64 KiB blocks)
//   zstd/enc_dfast.go:372-675  doubleFastEncoder.EncodeNoHist  (level 2: long 8-byte + short 5-byte table, long match
//                                                               preferred, lazy long check at s+1, 128 KiB blocks)
// with one parallel parse whose output (literals + sequences) feeds the unchanged entropy stages K2..K4.
//
// Why a new table discipline.  Round 1 kept the EARLIEST position of every hash in a static table so that 1024 threads
// could probe it at once; scoring parse variants with the oracle's entropy stage (tests/model/) showed that recency is
// what the reference's "latest position" table buys: on 64 KiB text chunks a latest-position candidate is worth -6 %
// output, on HTML -12 %.  A fully dynamic table is serial; what is built here is the parallel form that keeps most of
// it: positions are inserted in TILES (4 per thread, in position order); a slot holds the earliest position of the
// latest tile that touched it.  A position therefore sees (a) "far": the slot as the earlier tiles left it and (b) "near":
// the earliest equal-hash position of its own tile, when that lies before it.  Per tile: probe (far) | barrier | plain
// stores | barrier | losers of a store race fix the slot with atomicMin (exact minimum, so the result never depends
// on scheduling) | barrier | probe (near).  Slots are 32-bit: position << 14 | 14 hash bits, so a candidate is
// accepted by its tag and the dense pass never reads the input at the candidate (random shared-memory reads are what
// bounded the round-1 kernel: about 3.4 bank-conflict cycles per warp access, five accesses per position there, four
// here for a much better parse).  The chunk itself is streamed from global memory during the dense pass (coalesced,
// prefetched one tile ahead) and only afterwards staged into the dead table's shared memory by one TMA bulk copy for
// the random accesses of the walk.
//
// After the dense pass every thread runs the greedy scan over its own 128-byte range (set bit -> candidate distance
// from a per-CTA scratch array -> extend forwards/backwards -> emit -> skip), neighbours are merged by a prefix
// maximum of match ends (as in round 1), sequences and codes are written, and the literals are produced by a
// warp-cooperative stream compaction of the staged chunk under a one-bit-per-position literal mask (coalesced byte
// stores; no 64 KiB literal staging buffer, which is what lets two CTAs share an SM).  The literal and sequence-code
// histograms are counted on the way, with shared-memory atomics into 1.8 KB of the per-thread arrays that are dead by
// then (see LZ_HIST_WORDS), so no later pass has to read the literals and codes back.
#pragma once
#include "b2c_zstd_enc.cuh"

namespace b2c {

constexpr uint32_t LZ_RANGE = 128;          // bytes walked by one thread
constexpr uint32_t LZ_MAXREC = LZ_RANGE / 4;   // matches a thread can start inside its range (min match 4)
constexpr uint32_t LZ_TAGBITS = 14;
constexpr uint32_t LZ_TAGMASK = (1u << LZ_TAGBITS) - 1;
constexpr uint32_t LZ_EMPTY = 0xffffffffu;
#ifndef LZ_PPT1
#define LZ_PPT1 8           // positions per thread and tile of the single-table configurations (4 or 8)
#endif
#ifndef LZ_INS_FAST
#define LZ_INS_FAST 2       // insertion stride of the "fastest" classes (zstd level 1, S2 fast): 2 = only even positions enter
#endif                      // the table (every position is still probed): one random access per position less, about +2 % output
constexpr uint32_t LZ_EXT_CAP = 256;        // per-thread forward extension limit; longer matches are finished by warp 0

template <int LV> struct LzCfg;
enum { LZ_ZSTD1 = 1, LZ_ZSTD2 = 2, LZ_S2FAST = 3, LZ_S2BETTER = 4, LZ_ZSTD3 = 5 };
template <> struct LzCfg<1> {
    static constexpr int NT = 512;
    static constexpr uint32_t BLOCK = 65536;
    static constexpr bool LONG = false;
    static constexpr int SMLS = 6, LMLS = 8;   // bytes hashed for the short / long table
    static constexpr int PPT = LZ_PPT1;        // positions per thread and tile (tile = NT * PPT positions)
    static constexpr int INS = LZ_INS_FAST;    // insertion stride
    static constexpr uint32_t TBITS = 14;
    static constexpr uint32_t KREC = 16;      // match records (4 bytes each) per thread kept in shared memory
    static constexpr int MIN_CTAS = 2;
};
template <> struct LzCfg<2> {
    static constexpr int NT = 1024;
    static constexpr uint32_t BLOCK = 131072;
    static constexpr bool LONG = true;
    static constexpr int SMLS = 5, LMLS = 8;
    static constexpr int PPT = 4;
    static constexpr int INS = 1;
    static constexpr uint32_t TBITS = 14;
    static constexpr uint32_t KREC = 8;
    static constexpr int MIN_CTAS = 1;
};

// zstd level 3 (SpeedBetterCompression, zstd/enc_better.go:56-568): the level-2 shape with the finest tile order this
// kernel offers -- one position per thread and tile, so a position's "near" candidate comes from the previous 1024
// positions at most and its "far" candidate from everything before: the closest this parse gets to the reference's
// always-current tables (its chained long table, :298-347, is replaced by the near / far pair of every slot).
template <> struct LzCfg<5> {
    static constexpr int NT = 1024;
    static constexpr uint32_t BLOCK = 131072;
    static constexpr bool LONG = true;
    static constexpr int SMLS = 5, LMLS = 8;
    static constexpr int PPT = 1;
    static constexpr int INS = 1;
    static constexpr uint32_t TBITS = 14;
    static constexpr uint32_t KREC = 8;
    static constexpr int MIN_CTAS = 1;
};

// S2 block encoders (s2/encode_all.go:72 encodeBlockGo: one table, 4-byte minimum match; s2/encode_better.go:485
// encodeBlockBetterGo64K: long 7-byte + short 4-byte table, long preferred, lazy step): 64 KiB blocks, two CTAs per SM
template <> struct LzCfg<3> {
    static constexpr int NT = 512;
    static constexpr uint32_t BLOCK = 65536;
    static constexpr bool LONG = false;
    static constexpr int SMLS = 4, LMLS = 8;
    static constexpr int PPT = LZ_PPT1;
    static constexpr int INS = LZ_INS_FAST;
    static constexpr uint32_t TBITS = 14;
    static constexpr uint32_t KREC = 16;
    static constexpr int MIN_CTAS = 2;
};
template <> struct LzCfg<4> {
    static constexpr int NT = 512;
    static constexpr uint32_t BLOCK = 65536;
    static constexpr bool LONG = true;
    static constexpr int SMLS = 4, LMLS = 7;
    static constexpr int PPT = 4;
    static constexpr int INS = 1;
    static constexpr uint32_t TBITS = 13;
    static constexpr uint32_t KREC = 12;      // (the second bitmap takes the room of four records per thread)
    static constexpr int MIN_CTAS = 2;
};

template <int LV> struct LzLayout {
    using C = LzCfg<LV>;
    static constexpr uint32_t NTAB = C::LONG ? 2 : 1;
    static constexpr uint32_t TAB_BYTES = NTAB * (4u << C::TBITS);
    static constexpr uint32_t SRC_BYTES = C::BLOCK + 128;
    static constexpr uint32_t A_BYTES = TAB_BYTES > SRC_BYTES ? TAB_BYTES : SRC_BYTES;
    static constexpr uint32_t BM_BYTES = C::BLOCK / 8 + 16;
    static constexpr uint32_t SM_A = 0;
    static constexpr uint32_t SM_BM = SM_A + A_BYTES;
    static constexpr uint32_t SM_BML = SM_BM + BM_BYTES;
    static constexpr uint32_t SM_REC = SM_BML + (C::LONG ? BM_BYTES : 0);
    static constexpr uint32_t REC_BYTES = C::KREC * C::NT * 4;
    static constexpr uint32_t SM_ARR = SM_REC + REC_BYTES;                      // keptEnd u32 | lastOff u32 | longLen u32 | cnt u8 | cap u8
    // S2 modes: per-warp output windows in the candidate bitmaps (dead after the walk); a thread's piece is < 400 bytes
    static constexpr uint32_t SM_STG = SM_BM;
    static constexpr uint32_t STG_S2 = ((BM_BYTES * (C::LONG ? 2u : 1u)) / (C::NT / 32)) & ~15u;
    static constexpr uint32_t SM_SH = SM_ARR + C::NT * 14;
    static constexpr uint32_t SMEM_BYTES = SM_SH + ((sizeof(ParseShared) + 2 * 80 * 4 + 15) / 16) * 16;
    // per-CTA global scratch: candidate distances (u16 per position) + spilled match records [k][thread]
    static constexpr uint32_t DIST_BYTES = C::BLOCK * 2;
    static constexpr uint32_t SCRATCH_BYTES = DIST_BYTES + (LZ_MAXREC - C::KREC) * C::NT * 4;
};
static_assert(2 * (LzLayout<1>::SMEM_BYTES + 1024) <= 228 * 1024, "two level-1 parse CTAs must fit one SM");
static_assert(LzLayout<2>::SMEM_BYTES <= 227 * 1024 && LzLayout<5>::SMEM_BYTES <= 227 * 1024, "the level-2 / level-3 parse CTA must fit one SM");
static_assert(2 * (LzLayout<3>::SMEM_BYTES + 1024) <= 228 * 1024 && 2 * (LzLayout<4>::SMEM_BYTES + 1024) <= 228 * 1024, "two S2 parse CTAs must fit one SM");
// zstd histograms of a chunk: 256 literal counters + 3 x 64 sequence-code counters, u32, in the longLen array
// of SM_ARR (NT words; last read before the merge scan, see lz_parse_chunk)
constexpr uint32_t LZ_HIST_WORDS = 256 + 3 * 64;
static_assert(LzCfg<1>::NT >= (int)LZ_HIST_WORDS && LzCfg<2>::NT >= (int)LZ_HIST_WORDS && LzCfg<5>::NT >= (int)LZ_HIST_WORDS,
              "the zstd histograms must fit the longLen array");

// hashes: two 32-bit multiply-adds (the reference's hashLen is a 64-bit multiply, zstd/hash.go:27-33; table contents
// are an implementation detail, only verified matches reach the output)
template <int MLS> B2C_DEV uint32_t lz_hash_short(uint32_t lo, uint32_t hi) {
    if constexpr (MLS == 4) return lo * 0x9E3779B1u;
    else if constexpr (MLS == 5) return lo * 0x9E3779B1u + (hi & 0xffu) * 0x85EBCA6Bu;
    else return lo * 0x9E3779B1u + (hi & 0xffffu) * 0x85EBCA6Bu;
}
template <int MLS> B2C_DEV uint32_t lz_hash_long(uint32_t lo, uint32_t hi) {
    if constexpr (MLS == 7) return lo * 0xC2B2AE3Du + (hi & 0xffffffu) * 0x27D4EB2Fu;
    else return lo * 0xC2B2AE3Du + hi * 0x27D4EB2Fu;
}

// exclusive scan of two values per thread (same conventions as group_scan_excl; ws: >= 80 words)
B2C_DEV void group_scan_excl_pair(uint32_t a, uint32_t b, uint32_t *ws, int nthreads, unsigned tid, uint32_t *exA,
                                  uint32_t *exB, uint32_t *totA, uint32_t *totB) {
    const unsigned lane = tid & 31, w = tid >> 5;
    const uint32_t ia = warp_scan_incl(a), ib = warp_scan_incl(b);
    if (lane == 31) { ws[w] = ia; ws[40 + w] = ib; }
    __syncthreads();
    if (w == 0) {
        const int nw = nthreads >> 5;
        const uint32_t xa = (lane < (unsigned)nw) ? ws[lane] : 0, xb = (lane < (unsigned)nw) ? ws[40 + lane] : 0;
        const uint32_t sa = warp_scan_incl(xa), sb = warp_scan_incl(xb);
        ws[lane] = sa - xa; ws[40 + lane] = sb - xb;
        if (lane == 31) { ws[32] = sa; ws[72] = sb; }
    }
    __syncthreads();
    *exA = ws[w] + ia - a; *exB = ws[40 + w] + ib - b;
    *totA = ws[32]; *totB = ws[72];
}

// match record of a thread (4 bytes, never rewritten): start - range start (7 bits) | length << 7 (9 bits: the walk caps
// a match at 256 bytes forwards and 127 backwards) | distance << 16.  A match that warp 0 finished keeps its walked
// length here and its full length in longLen[thread].  Trimming against earlier threads is applied when a record is
// read (it only needs the thread's R), so the records are written once.
B2C_DEV uint32_t lz_rec(uint32_t rel, uint32_t len, uint32_t d) { return rel | (len << 7) | (d << 16); }
B2C_DEV uint32_t lz_rec_rel(uint32_t r) { return r & 127u; }
B2C_DEV uint32_t lz_rec_len(uint32_t r) { return (r >> 7) & 511u; }
B2C_DEV uint32_t lz_rec_d(uint32_t r) { return r >> 16; }

// One tile of the dense pass for the four positions 4g .. 4g+3 of this thread (words w0..w2 hold their 11 bytes).
// GUARD: the tile reaches past the last hashable position (only the last tile of a chunk).
// A slot is position << 14 | tag, so for a slot r and this position's entry e the difference t = e - r is
// (distance << 14) exactly when the tags agree and r lies before e: "t & (sign | tag bits) == 0" is the whole
// acceptance test and t >> 14 the candidate's distance (an empty slot, all ones, can only pass with a distance beyond
// the position, which the walk rejects).
template <int LV, bool GUARD>
B2C_DEV void lz_dense_tile(uint32_t *TS, uint32_t *TL, uint32_t *bm, uint32_t *bml, uint16_t *cd, uint32_t g, uint32_t npos,
                           const uint32_t (&wv)[LzCfg<LV>::PPT < 4 ? 3 : LzCfg<LV>::PPT / 4 + 2], unsigned lane) {
    using C = LzCfg<LV>;
    constexpr int PPT = C::PPT;
    constexpr uint32_t BAD = 0x80000000u | LZ_TAGMASK | (C::BLOCK > 65536 ? 0x40000000u : 0u);   // wrong tag, not earlier, or >= 64 KiB away
    const uint32_t p0 = PPT * g;
    uint32_t hs[PPT], fs[PPT];                  // short table: hash (index = high bits, tag = low bits) and far slot content
    uint32_t hl[C::LONG ? PPT : 1], fl[C::LONG ? PPT : 1];
#define LZ_IDX(h) ((h) >> (32 - C::TBITS))
#define LZ_ENT(h, j) (((p0 + (j)) << LZ_TAGBITS) | ((h) & LZ_TAGMASK))
#pragma unroll
    for (int j = 0; j < PPT; j++) {
        uint32_t lo, hi;
        if constexpr (PPT < 4) {        // the thread's first position is not word aligned: byte offset (PPT * g) & 3, + j
            const uint32_t bo = ((PPT * g) & 3u) + j;          // 0 .. 4
            const uint32_t sh = (bo & 3u) * 8;
            const uint32_t a = bo >= 4 ? wv[1] : wv[0], bb = bo >= 4 ? wv[2] : wv[1], c = bo >= 4 ? 0u : wv[2];
            lo = __funnelshift_r(a, bb, sh); hi = __funnelshift_r(bb, c, sh);
        } else {
            const uint32_t a = wv[j >> 2], bb = wv[(j >> 2) + 1], c = wv[(j >> 2) + 2];
            lo = (j & 3) ? __funnelshift_r(a, bb, 8 * (j & 3)) : a;
            hi = (j & 3) ? __funnelshift_r(bb, c, 8 * (j & 3)) : bb;
        }
        hs[j] = lz_hash_short<C::SMLS>(lo, hi);
        fs[j] = TS[LZ_IDX(hs[j])];                                     // far candidate: the slot as earlier tiles left it
        if constexpr (C::LONG) {
            hl[j] = lz_hash_long<C::LMLS>(lo, hi);
            fl[j] = TL[LZ_IDX(hl[j])];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = PPT - 1; j >= 0; j--)                                 // the thread's lowest position lands last
        if ((C::INS == 1 || (j & 1) == 0) && (!GUARD || p0 + j < npos)) {
            TS[LZ_IDX(hs[j])] = LZ_ENT(hs[j], j);
            if constexpr (C::LONG) TL[LZ_IDX(hl[j])] = LZ_ENT(hl[j], j);
        }
    __syncthreads();
    {
        // all slots are read before the first fix: the loads overlap (an atomic between two loads would order them), and a
        // stale value can only cause a redundant atomicMin
        uint32_t cs[PPT], cl[C::LONG ? PPT : 1];
#pragma unroll
        for (int j = 0; j < PPT; j++)
            if (C::INS == 1 || (j & 1) == 0) {
                cs[j] = TS[LZ_IDX(hs[j])];
                if constexpr (C::LONG) cl[j] = TL[LZ_IDX(hl[j])];
            }
#pragma unroll
        for (int j = 0; j < PPT; j++)
            if ((C::INS == 1 || (j & 1) == 0) && (!GUARD || p0 + j < npos)) {
                if (cs[j] > LZ_ENT(hs[j], j)) atomicMin(&TS[LZ_IDX(hs[j])], LZ_ENT(hs[j], j));   // lost a store race: exact minimum of the tile
                if constexpr (C::LONG) { if (cl[j] > LZ_ENT(hl[j], j)) atomicMin(&TL[LZ_IDX(hl[j])], LZ_ENT(hl[j], j)); }
            }
    }
    __syncthreads();
    uint32_t bitsA = 0, bitsL = 0, dist[PPT];
#pragma unroll
    for (int j = 0; j < PPT; j++) {
        uint32_t d = 0;
        bool ok = false, okL = false;
        if (!GUARD || p0 + j < npos) {
            if constexpr (C::LONG) {
                const uint32_t e = LZ_ENT(hl[j], j);
                const uint32_t tn = e - TL[LZ_IDX(hl[j])], tf = e - fl[j];
                const bool nearOk = (tn & BAD) == 0 && tn != 0;           // near: the tile's earliest equal-hash position, if before this one
                okL = nearOk || (tf & BAD) == 0;
                if (okL) d = (nearOk ? tn : tf) >> LZ_TAGBITS;
            }
            if (!okL) {
                const uint32_t e = LZ_ENT(hs[j], j);
                const uint32_t tn = e - TS[LZ_IDX(hs[j])], tf = e - fs[j];
                const bool nearOk = (tn & BAD) == 0 && tn != 0;
                ok = nearOk || (tf & BAD) == 0;
                if (ok) d = (nearOk ? tn : tf) >> LZ_TAGBITS;
            }
        }
        dist[j] = d;
        if (ok || okL) bitsA |= 1u << j;
        if (okL) bitsL |= 1u << j;
    }
#undef LZ_IDX
#undef LZ_ENT
    if constexpr (PPT == 8) {
        *reinterpret_cast<uint4 *>(cd + p0) = make_uint4(dist[0] | (dist[1] << 16), dist[2] | (dist[3] << 16),
                                                          dist[4] | (dist[5] << 16), dist[6] | (dist[7] << 16));
        // one byte per thread, one bitmap word per four threads
        uint32_t word = bitsA << (8 * (lane & 3));
        word |= __shfl_xor_sync(FULLMASK, word, 1);
        word |= __shfl_xor_sync(FULLMASK, word, 2);
        if ((lane & 3) == 0) bm[g >> 2] = word;
    } else if constexpr (PPT == 1) {
        cd[p0] = (uint16_t)dist[0];
        const unsigned wa = __ballot_sync(FULLMASK, bitsA & 1u);
        if (lane == 0) bm[g >> 5] = wa;
        if constexpr (C::LONG) {
            const unsigned wl = __ballot_sync(FULLMASK, bitsL & 1u);
            if (lane == 0) bml[g >> 5] = wl;
        }
    } else if constexpr (PPT == 2) {
        *reinterpret_cast<uint32_t *>(cd + p0) = dist[0] | (dist[1] << 16);
        uint32_t word = bitsA << (2 * (lane & 15)), wl = bitsL << (2 * (lane & 15));
#pragma unroll
        for (int x = 1; x < 16; x <<= 1) { word |= __shfl_xor_sync(FULLMASK, word, x); wl |= __shfl_xor_sync(FULLMASK, wl, x); }
        if ((lane & 15) == 0) { bm[g >> 4] = word; if constexpr (C::LONG) bml[g >> 4] = wl; }
    } else {
        *reinterpret_cast<uint2 *>(cd + p0) = make_uint2(dist[0] | (dist[1] << 16), dist[2] | (dist[3] << 16));
        uint32_t word = bitsA << (4 * (lane & 7));
        word |= __shfl_xor_sync(FULLMASK, word, 1);
        word |= __shfl_xor_sync(FULLMASK, word, 2);
        word |= __shfl_xor_sync(FULLMASK, word, 4);
        if ((lane & 7) == 0) bm[g >> 3] = word;
        if constexpr (C::LONG) {
            uint32_t wl = bitsL << (4 * (lane & 7));
            wl |= __shfl_xor_sync(FULLMASK, wl, 1);
            wl |= __shfl_xor_sync(FULLMASK, wl, 2);
            wl |= __shfl_xor_sync(FULLMASK, wl, 4);
            if ((lane & 7) == 0) bml[g >> 3] = wl;
        }
    }
}

// One warp writes staging bytes [ph, ph + fill) to gd[0, fill): the staging offset has the destination's 16-byte phase, so
// the middle leaves as 16-byte vectors and only the ragged ends use byte stores.
B2C_DEV void lz_warp_flush(const uint8_t *stg, uint32_t ph, uint32_t fill, uint8_t *gd, unsigned lane) {
    __syncwarp();
    const uint32_t head = fill < ((16 - ph) & 15) ? fill : ((16 - ph) & 15);
    if (lane < head) gd[lane] = stg[ph + lane];
    const uint32_t nvec = (fill - head) / 16;
    const uint4 *sv = reinterpret_cast<const uint4 *>(stg + ph + head);
    uint4 *gv = reinterpret_cast<uint4 *>(gd + head);
    for (uint32_t v = lane; v < nvec; v += 32) gv[v] = sv[v];
    const uint32_t done = head + nvec * 16;
    if (lane < fill - done) gd[done + lane] = stg[ph + done + lane];
    __syncwarp();
}

template <int LV, int MODE>
B2C_DEV void lz_parse_chunk(uint8_t *smem, const ZstdEncParams &P, uint32_t chunk, uint8_t *scratch) {
    using C = LzCfg<LV>;
    using L = LzLayout<LV>;
    constexpr int NT = C::NT;
    constexpr uint32_t TSIZE = 1u << C::TBITS;
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    uint32_t *TS = reinterpret_cast<uint32_t *>(smem + L::SM_A);
    uint32_t *TL = TS + TSIZE;                                   // level 2 only
    uint8_t *src = smem + L::SM_A;                               // after the dense pass
    uint32_t *bm = reinterpret_cast<uint32_t *>(smem + L::SM_BM);   // any candidate; later the literal mask
    uint32_t *bml = reinterpret_cast<uint32_t *>(smem + L::SM_BML); // long candidate (level 2)
    ParseShared *sh = reinterpret_cast<ParseShared *>(smem + L::SM_SH);
    uint32_t *ws2 = reinterpret_cast<uint32_t *>(smem + L::SM_SH + ((sizeof(ParseShared) + 15) / 16) * 16);
    uint16_t *plut = reinterpret_cast<uint16_t *>(ws2 + 96);   // byte-permute selector per 4-bit mask: the set bytes, in order
    constexpr bool ZSTD = (MODE == LZ_MODE_ZSTD);
    ChunkWork *W = ZSTD ? P.work + chunk : nullptr;
    const WkLens wlen = ZSTD ? wk_lens(P, chunk) : WkLens{nullptr, nullptr, 0};
    uint32_t *const wof = ZSTD ? wk_of(P, chunk) : nullptr;
    uint8_t *const wcodes = ZSTD ? wk_codes(P, chunk, 0) : nullptr;
    const uint32_t mseq = ZSTD ? P.maxseq : 0xffffffffu;
    uint16_t *cd = reinterpret_cast<uint16_t *>(scratch);

    // Frame mode: the block is parsed as the tail of a "virtual chunk" that starts `hist` bytes earlier (the end of the
    // previous block(s) of the same frame, contiguous in memory).  The dense pass covers the whole virtual chunk, so the
    // tables hold the history's positions when the block's own tiles are probed; the walk, the literals and the sequences
    // cover only [hist, n).  This is fastBase.hist / addBlock (zstd/enc_base.go:57-199) without a table that survives
    // between blocks: every block of a frame is parsed independently of the others.
    const uint32_t hist = ZSTD ? chunk_hist(P, chunk) : 0u;
    const uint8_t *gsrc = chunk_src(P, chunk) - hist;
    const uint32_t n = chunk_size(P, chunk) + hist;
    if (n > C::BLOCK || (ZSTD && n > P.blockmax)) {
        if (tid == 0) {
            if constexpr (ZSTD) { W->n = n - hist; W->kind = 3; }   // reported as B2C_ERR_TOO_BIG by the pack kernel
            else P.out_sizes[chunk] = -3;
        }
        return;
    }
    B2C_PHASE(0);
    // ---------------------------------------------------------------- P0: empty tables
    for (uint32_t i = tid; i < L::NTAB * TSIZE; i += NT) TS[i] = LZ_EMPTY;
    if (tid < 16) {
        uint32_t sel = 0, k = 0;
        for (uint32_t bb = 0; bb < 4; bb++)
            if ((tid >> bb) & 1) { sel |= bb << (4 * k); k++; }
        plut[tid] = (uint16_t)sel;
    }
    __syncthreads();

    // ---------------------------------------------------------------- P1: dense pass, tile by tile
    // aligned word k of the chunk's address range holds chunk bytes [4k - mis, 4k - mis + 4)
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(gsrc) & 3), msh = mis * 8;
    const uint32_t *gw = reinterpret_cast<const uint32_t *>(gsrc - mis);
    const uint32_t nraw = (n + mis + 3) >> 2;      // aligned words that contain chunk bytes
#define LZ_RAW(k) (((k) < nraw) ? B2C_LDG(gw + (k)) : 0u)
#define LZ_WORD(dst, wi)                                                                         \
    do {                                                                                         \
        const uint32_t k_ = (wi);                                                                \
        const uint32_t a_ = LZ_RAW(k_);                                                          \
        if (mis) { const uint32_t b_ = LZ_RAW(k_ + 1); (dst) = __funnelshift_r(a_, b_, msh); }   \
        else (dst) = a_;                                                                         \
    } while (0)
    const uint32_t npos = (n >= 8) ? n - 7 : 0;    // positions with 8 readable bytes
    constexpr int PPT = C::PPT, NWRD = PPT < 4 ? 3 : PPT / 4 + 2;      // a thread's PPT positions read NWRD words from word (PPT * g) / 4 on
    static_assert(!C::LONG || PPT <= 4, "the two-table configurations keep at most four positions per thread");
#define LZ_WI(gg) ((uint32_t)(PPT * (gg)) >> 2)
    const uint32_t ngroups = (npos + PPT - 1) / PPT;
    const uint32_t ntiles = (ngroups + NT - 1) / NT;
    {
        uint32_t wv[NWRD], nwv[NWRD];
#pragma unroll
        for (int q = 0; q < NWRD; q++) { wv[q] = 0; nwv[q] = 0; }
        if (ntiles) {
#pragma unroll
            for (int q = 0; q < NWRD; q++) LZ_WORD(wv[q], LZ_WI(tid) + q);
        }
        for (uint32_t k = 0; k < ntiles; k++) {
            const uint32_t g = k * NT + tid;
            // the next tile's words are requested before this tile's barriers; whole tiles of an aligned chunk take the
            // unguarded forms (block-uniform tests)
            if (k + 1 < ntiles) {
                if (mis == 0 && LZ_WI((k + 2) * NT) + 3 < nraw) {
#pragma unroll
                    for (int q = 0; q < NWRD; q++) nwv[q] = B2C_LDG(gw + LZ_WI(g + NT) + q);
                } else {
#pragma unroll
                    for (int q = 0; q < NWRD; q++) LZ_WORD(nwv[q], LZ_WI(g + NT) + q);
                }
            }
            if (PPT * (k + 1) * NT <= npos) lz_dense_tile<LV, false>(TS, TL, bm, bml, cd, g, npos, wv, lane);
            else lz_dense_tile<LV, true>(TS, TL, bm, bml, cd, g, npos, wv, lane);
#pragma unroll
            for (int q = 0; q < NWRD; q++) wv[q] = nwv[q];
        }
    }
    __syncthreads();      // the tables are dead: their memory takes the chunk
    B2C_PHASE(1);

    // ---------------------------------------------------------------- P2: stage the chunk (TMA bulk copy when aligned)
    {
#ifndef B2C_EMU
        const bool bulk = ((reinterpret_cast<uintptr_t>(gsrc) & 15) == 0) && ((n & 15) == 0) && n > 0;
        if (bulk) {
            if (tid == 0) {
                mbar_init(&sh->mbar, 1);
                mbar_fence_init();
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy table accesses before the async write
                mbar_expect_tx(&sh->mbar, n);
                tma_load_1d(src, gsrc, n, &sh->mbar);
            }
            __syncthreads();
            mbar_wait(&sh->mbar, 0);
        } else
#endif
        {
            uint32_t *sw = reinterpret_cast<uint32_t *>(src);
            for (uint32_t i = tid; i < (n + 3) / 4; i += NT) { uint32_t v; LZ_WORD(v, i); sw[i] = v; }
        }
        // bytes behind the chunk are read (never used) by unaligned 8-byte loads: keep them defined
        for (uint32_t i = ((n + 3) & ~3u) / 4 + tid; i < ((n + 3) & ~3u) / 4 + 8; i += NT) reinterpret_cast<uint32_t *>(src)[i] = 0;
        __syncthreads();
#ifndef B2C_EMU
        if (bulk && tid == 0) { asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(&sh->mbar))); }
#endif
    }
#undef LZ_WORD
#undef LZ_RAW
#undef LZ_WI
    B2C_PHASE(2);

    // ---------------------------------------------------------------- P3: walk, one thread per 128-byte range
    // Every thread runs the greedy scan over its own range: next marked position, candidate = position - stored distance,
    // extend forwards / backwards, emit, skip past the match.  Threads never communicate (bitmaps, distances and the
    // chunk are read-only here), so the parse does not depend on scheduling.  A match may run past the end of the
    // range; the merge step trims whatever a later thread found inside it.
    // record k of thread t (k < KREC in shared memory, the rest in the per-CTA scratch): see lz_rec()
    uint32_t *recS = reinterpret_cast<uint32_t *>(smem + L::SM_REC);
    uint32_t *recG = reinterpret_cast<uint32_t *>(scratch + L::DIST_BYTES);
#define REC(k, t) (*(((k) < C::KREC) ? &recS[(k) * NT + (t)] : &recG[((k) - C::KREC) * NT + (t)]))
    uint32_t *keptEndA = reinterpret_cast<uint32_t *>(smem + L::SM_ARR);
    uint32_t *lastOffA = keptEndA + NT;
    uint32_t *longLen = lastOffA + NT;          // full length of a thread's last record when warp 0 finished it, else 0
    uint8_t *cntA = reinterpret_cast<uint8_t *>(longLen + NT);
    uint8_t *capA = cntA + NT;
    const uint32_t nlanes = (n + LZ_RANGE - 1) / LZ_RANGE;
    const uint32_t *srcw = reinterpret_cast<const uint32_t *>(src);
    const uint32_t b = tid * LZ_RANGE;                                   // this thread's range [b, e)
    const uint32_t e = (b + LZ_RANGE < n) ? b + LZ_RANGE : n;
    uint32_t cnt = 0, lastE = 0;
    bool capped = false;
    {
        const uint32_t pend = (tid < nlanes) ? (e < npos ? e : npos) : 0u;
        uint32_t p = b > hist ? b : hist, nextEmit = p;            // (history is never walked, nor extended into backwards)
        while (p < pend) {
            // next set bit in [p, pend)
            uint32_t wi = p >> 5;
            uint32_t wv = bm[wi] & (0xffffffffu << (p & 31));
            while (wv == 0 && (wi + 1) * 32 < pend) wv = bm[++wi];
            if (wv == 0) break;
            p = wi * 32 + (uint32_t)(__ffs((int)wv) - 1);
            if (p >= pend) break;
            if constexpr (C::LONG) {
                // doubleFastEncoder's preference (enc_dfast.go:202-239): a long match wins; a short match yields to a
                // long match that starts one byte later
                const bool isL = (bml[p >> 5] >> (p & 31)) & 1;
                if (!isL && p + 1 < pend && ((bml[(p + 1) >> 5] >> ((p + 1) & 31)) & 1)) p = p + 1;
            }
            const uint32_t d = cd[p];
            if (d == 0 || d > p) { p++; continue; }
            const uint32_t cand = p - d;
            const uint32_t lim = (p + LZ_EXT_CAP < n) ? p + LZ_EXT_CAP : n;
            // forward: 4 bytes per step from two unaligned streams (aligned word loads + funnel shifts); the tag that
            // accepted the candidate is a hash, so the comparison starts at the first byte
            uint32_t len = 0;
            {
                uint32_t ia = p >> 2, ib = cand >> 2;
                const uint32_t sha = (p & 3) * 8, shb = (cand & 3) * 8;
                uint32_t wa0 = srcw[ia], wb0 = srcw[ib];
                while (p + len < lim) {
                    const uint32_t wa1 = srcw[++ia], wb1 = srcw[++ib];
                    const uint32_t x = __funnelshift_r(wa0, wa1, sha) ^ __funnelshift_r(wb0, wb1, shb);
                    if (x) { len += (uint32_t)(__ffs((int)x) - 1) >> 3; break; }
                    len += 4; wa0 = wa1; wb0 = wb1;
                }
            }
            bool cp = false;
            if (p + len >= lim) { len = lim - p; cp = lim < n; }
            if (len < 4) { p++; continue; }
            capped = cp;
            uint32_t s = p, t = cand;
            while (s > nextEmit && t > 0 && src[s - 1] == src[t - 1]) { s--; t--; len++; }
            REC(cnt, tid) = lz_rec(s - b, len, d);
            cnt++;
            p = s + len;
            nextEmit = p;
        }
        if (cnt) lastE = nextEmit;
    }
    B2C_PHASE(6);
    cntA[tid] = (uint8_t)cnt;
    capA[tid] = (uint8_t)((cnt != 0) && capped);
    longLen[tid] = 0;
    __syncthreads();
    // long matches: warp 0 walks the capped records in order and finishes them cooperatively (128 bytes per step);
    // a capped record that already lies inside an earlier finished one is skipped, so a chunk of zeros costs one pass
    if (w == 0) {
        uint32_t covered = 0;
        for (uint32_t base = 0; base < nlanes; base += 32) {
            const uint32_t t = base + lane;
            unsigned m = __ballot_sync(FULLMASK, t < nlanes && capA[t]);
            while (m) {
                const uint32_t tt = base + (uint32_t)(__ffs((int)m) - 1);
                m &= m - 1;
                const uint32_t r = REC((uint32_t)cntA[tt] - 1, tt);
                const uint32_t s0 = tt * LZ_RANGE + lz_rec_rel(r), l0 = lz_rec_len(r), d0 = lz_rec_d(r);
                const uint32_t e0 = s0 + l0;
                if (e0 > covered) {
                    const uint32_t ext = warp_match_len(src, e0, e0 - d0, n);
                    if (lane == 0) longLen[tt] = l0 + ext;
                    covered = e0 + ext;
                }
            }
        }
    }
    __syncthreads();
    const uint32_t myLong = longLen[tid];
    if (myLong) lastE = b + lz_rec_rel(REC(cnt - 1, tid)) + myLong;
    B2C_PHASE(3);

    // ---------------------------------------------------------------- P4: merge (trim overlaps), global layout
    uint32_t dummyTotal;
    const uint32_t R = group_scan_excl_max(lastE, sh->ws, 0, NT, tid, &dummyTotal);   // everything before R is taken
    // the zstd histograms live in longLen, whose last read (myLong) precedes the barriers of the scan above;
    // the barrier before the next scan orders this zeroing before the counting in P5 / P6
    uint32_t *const hcnt = longLen;             // [0, 256) literal bytes | 256 + 64 * table + code
    if constexpr (ZSTD) { if (tid < LZ_HIST_WORDS) hcnt[tid] = 0; }
    B2C_PHASE(8);
    // A record survives when at least 4 of its bytes lie behind R; the dropped ones are a prefix of the thread's records
    // (records are ordered and disjoint), so the kept ones are firstKept .. cnt-1, the first of them possibly trimmed.
    uint32_t kept = 0, firstKept = cnt, sumLen = 0, keptE = 0, lastOff = 0;
    for (uint32_t j = 0; j < cnt; j++) {
        const uint32_t r = REC(j, tid);
        const uint32_t s0 = b + lz_rec_rel(r), e0 = s0 + ((j + 1 == cnt && myLong) ? myLong : lz_rec_len(r));
        if (e0 <= R) continue;
        const uint32_t s2 = s0 > R ? s0 : R, l2 = e0 - s2;
        if (l2 < 4) continue;
        if (kept == 0) firstKept = j;
        kept++; sumLen += l2; keptE = e0; lastOff = lz_rec_d(r);
    }
    B2C_PHASE(9);
    keptEndA[tid] = keptE;
    lastOffA[tid] = lastOff;
    uint32_t seqEx, lenEx, nseq, sumAll, keyTotal;
    __syncthreads();   // sh->ws is reused by the next scan
    group_scan_excl_pair(kept, sumLen, ws2, NT, tid, &seqEx, &lenEx, &nseq, &sumAll);
    (void)lenEx;
    // nearest earlier thread that kept something: gives the end of the previous sequence and its offset
    const uint32_t keyEx = group_scan_excl_max(kept ? tid + 1 : 0u, sh->ws, 0, NT, tid, &keyTotal);
    B2C_PHASE(10);
    const uint32_t nlit = n - hist - sumAll;
    const uint32_t prevE0 = keyEx ? keptEndA[keyEx - 1] : hist;        // end of the sequence before this thread's first
    const uint32_t pOff0 = keyEx ? lastOffA[keyEx - 1] : 0u;

    if constexpr (!ZSTD) {
        // -------------------------------------------------------------- S2 / Snappy emission (s2/encode_go.go:80-289)
        // Sizes per thread -> block scan -> every thread writes its literal runs and copy / repeat tags into its warp's
        // staging window (the lanes of a warp produce one contiguous piece of the block, in lane order), windows leave
        // as 16-byte vectors.  A repeat tag is used whenever the offset equals the previous copy's.
        constexpr bool SNAPPY = (MODE == LZ_MODE_SNAPPY);
        const uint32_t hdrLen = n < 128 ? 1u : (n < 16384 ? 2u : 3u);       // uvarint(n), n <= 65536
        const bool firstThread = (seqEx == 0);                               // no sequence before this thread's
        uint32_t mySize = 0;
        {
            uint32_t pe = prevE0, po = pOff0;
            bool fst = firstThread;
            for (uint32_t j = firstKept; j < cnt; j++) {
                const uint32_t r = REC(j, tid);
                const uint32_t s0 = b + lz_rec_rel(r), e0 = s0 + ((j + 1 == cnt && myLong) ? myLong : lz_rec_len(r));
                const uint32_t s2 = s0 > R ? s0 : R, l2 = e0 - s2, d0 = lz_rec_d(r), ll = s2 - pe;
                mySize += s2_lit_hdr_size(ll) + ll;
                if (SNAPPY) mySize += snappy_copy_size(d0, l2);
                else mySize += (!fst && d0 == po) ? s2_repeat_size(d0, l2) : s2_copy_size(d0, l2);
                pe = e0; po = d0; fst = false;
            }
        }
        uint32_t bodyNoTail;
        __syncthreads();
        const uint32_t myOff = group_scan_excl(mySize, sh->ws, 0, NT, tid, &bodyNoTail);
        const uint32_t lastEnd = keyTotal ? keptEndA[keyTotal - 1] : 0u;      // end of the last sequence of the block
        const uint32_t tl = n - lastEnd;
        const uint32_t body = bodyNoTail + s2_lit_hdr_size(tl) + tl;
        uint8_t *gdst = P.dst_base + (uint64_t)chunk * P.dst_stride;
        // encodeBlock's "not compressible" rule (s2/encode_all.go:88: dstLimit), blocks below minNonLiteralBlockSize
        // (s2/encode.go:375) and the empty input are stored as one literal
        const bool store = (n < 32) || (nseq == 0) || (body > n - (n >> 5) - 5);
        const uint32_t total = hdrLen + (store ? s2_lit_hdr_size(n) + n : body);
        if (total > P.dst_cap) {
            if (tid == 0) P.out_sizes[chunk] = -4;
        } else {
            if (tid == 0) {
                uint32_t o = 0, v = n;
                while (v >= 0x80) { gdst[o++] = (uint8_t)(v | 0x80); v >>= 7; }
                gdst[o++] = (uint8_t)v;
                if (store) s2_put_lit_hdr(gdst + o, n);
                else s2_put_lit_hdr(gdst + hdrLen + bodyNoTail, tl);
                P.out_sizes[chunk] = (int64_t)total;
            }
            if (store) {
                const uint32_t o0 = hdrLen + s2_lit_hdr_size(n);
                for (uint32_t i = tid; i < n; i += NT) gdst[o0 + i] = src[i];
            } else {
                // (the match records are still being read, so the windows live in the candidate bitmaps, which are dead)
                static_assert(L::STG_S2 >= 96 + 128 + 32 * 6 + 16, "a thread's piece (without a long leading run) must fit a window");
                uint8_t *stg = smem + L::SM_STG + w * L::STG_S2;
                uint8_t *gbody = gdst + hdrLen;
                // A thread's piece starts with the literals since the previous sequence, which may be long (everything the
                // earlier threads left unmatched).  A leading run of more than 96 bytes does not go through the window:
                // when its thread is next, the warp copies it from the staged chunk straight to the destination.
                uint32_t bigLL = 0;
                if (kept) {
                    const uint32_t r = REC(firstKept, tid);
                    const uint32_t s0 = b + lz_rec_rel(r);
                    const uint32_t ll0 = (s0 > R ? s0 : R) - prevE0;
                    if (ll0 > 96) bigLL = ll0;
                }
                uint32_t curOff = myOff, curSize = mySize;     // what is left of this thread's piece
                bool bigPending = bigLL != 0;
                uint32_t doneLanes = 0;
                while (doneLanes < 32) {
                    if (__shfl_sync(FULLMASK, (int)bigPending, (int)doneLanes)) {
                        const uint32_t ll = __shfl_sync(FULLMASK, bigLL, (int)doneLanes);
                        const uint32_t from = __shfl_sync(FULLMASK, prevE0, (int)doneLanes);
                        const uint32_t at = __shfl_sync(FULLMASK, curOff, (int)doneLanes);
                        const uint32_t hb = s2_lit_hdr_size(ll);
                        if (lane == doneLanes) { s2_put_lit_hdr(gbody + at, ll); bigPending = false; curOff += hb + ll; curSize -= hb + ll; }
                        for (uint32_t k = lane; k < ll; k += 32) gbody[at + hb + k] = src[from + k];
                        continue;
                    }
                    const uint32_t winStart = __shfl_sync(FULLMASK, curOff, (int)doneLanes);
                    const uint32_t ph = (uint32_t)((reinterpret_cast<uintptr_t>(gbody) + winStart) & 15);
                    const bool fits = lane >= doneLanes && !bigPending && (curOff + curSize - winStart + ph <= L::STG_S2);
                    const unsigned fm = __ballot_sync(FULLMASK, fits) >> doneLanes;
                    uint32_t take = (fm == 0xffffffffu >> doneLanes) ? 32 - doneLanes : (uint32_t)(__ffs((int)~fm) - 1);
                    // (without its leading run an S2 piece is at most 96 + 128 literal bytes and 32 x (1 + 5) tag bytes: it fits.
                    // A Snappy piece with a very long match -- 3 bytes per 60 -- may not: that thread writes to the
                    // destination directly)
                    const bool direct = (take == 0);
                    if (direct) take = 1;
                    if (lane >= doneLanes && lane < doneLanes + take && curSize) {
                        uint8_t *d = direct ? gbody + curOff : stg + ph + (curOff - winStart);
                        uint32_t pe = prevE0, po = pOff0;
                        bool fst = firstThread;
                        for (uint32_t j = firstKept; j < cnt; j++) {
                            const uint32_t r = REC(j, tid);
                            const uint32_t s0 = b + lz_rec_rel(r), e0 = s0 + ((j + 1 == cnt && myLong) ? myLong : lz_rec_len(r));
                            const uint32_t s2 = s0 > R ? s0 : R, l2 = e0 - s2, d0 = lz_rec_d(r), ll = s2 - pe;
                            if (!(j == firstKept && bigLL)) {          // (a long leading run has been written already)
                                d += s2_put_lit_hdr(d, ll);
                                for (uint32_t k = 0; k < ll; k++) d[k] = src[pe + k];
                                d += ll;
                            }
                            if (SNAPPY) d += snappy_put_copy(d, d0, l2);
                            else d += (!fst && d0 == po) ? s2_put_repeat(d, d0, l2) : s2_put_copy(d, d0, l2);
                            pe = e0; po = d0; fst = false;
                        }
                    }
                    const uint32_t lastLane = doneLanes + take - 1;
                    const uint32_t winEnd = __shfl_sync(FULLMASK, curOff + curSize, (int)lastLane);
                    if (!direct) lz_warp_flush(stg, ph, winEnd - winStart, gbody + winStart, lane);
                    doneLanes += take;
                }
                // trailing literals: straight from the staged chunk
                const uint32_t th = s2_lit_hdr_size(tl);
                uint8_t *dt = gbody + bodyNoTail + th;
                for (uint32_t k = tid; k < tl; k += NT) dt[k] = src[lastEnd + k];
            }
        }
        __syncthreads();
        B2C_PHASE(4);
        B2C_PHASE(5);
        return;
    } else {
    // blockEnc.encode early decisions (blockenc.go:481-503): no sequences => literals-only (raw) block; then the
    // single-sequence RLE test; then `saved < 16` => raw
    uint32_t kind = 0;
    const uint32_t nblk = n - hist;                                    // the block itself
    const int saved = (int)nblk - (int)nlit - (int)(nblk >> 6);
    if (nseq == 0) kind = 1;
    else if (nseq != 1 && saved < 16) kind = 1;
    if (nseq > mseq) kind = 1;      // cannot happen (mseq >= BLOCK / 4); keeps the arrays safe

    // ---------------------------------------------------------------- P5: literal mask, sequences, codes
    uint32_t *mask = bm;     // one bit per position: 1 = literal.  Thread t owns the four words of its own range.
    uint32_t myLit = 0;
    if (kind == 0 || (P.dbg_hdr && nseq <= mseq)) {      // (the parity tests also want the sequences of blocks stored raw)
        // -- per thread: the four mask words of the own range
        uint32_t m4[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const uint32_t lo = b + 32 * k;
            m4[k] = (lo >= n) ? 0u : (n - lo >= 32 ? 0xffffffffu : ((1u << (n - lo)) - 1));
        }
        // clear [x, y) (absolute positions, clipped to this thread's range) in m4
#define LZ_CLEAR(x, y)                                                                                   \
    do {                                                                                                 \
        const uint32_t x_ = (x) > b ? (x) - b : 0u, y_ = ((y) < e ? (y) : e);                             \
        if (y_ > b && x_ < y_ - b) {                                                                      \
            const uint32_t yy_ = y_ - b;                                                                  \
            _Pragma("unroll") for (int k_ = 0; k_ < 4; k_++) {                                            \
                const uint32_t lo_ = 32u * k_;                                                            \
                const uint32_t a_ = x_ > lo_ ? x_ - lo_ : 0u, c_ = yy_ > lo_ ? yy_ - lo_ : 0u;            \
                if (a_ < 32 && c_ > a_) {                                                                 \
                    const uint32_t hi_ = c_ >= 32 ? 0xffffffffu : ((1u << c_) - 1);                       \
                    m4[k_] &= ~(hi_ & (0xffffffffu << a_));                                               \
                }                                                                                         \
            }                                                                                             \
        }                                                                                                 \
    } while (0)
        LZ_CLEAR(b, prevE0);              // the part of this range covered by the last kept match of the earlier threads
        for (uint32_t j = firstKept; j < cnt; j++) {
            const uint32_t r = REC(j, tid);
            const uint32_t s0 = b + lz_rec_rel(r), e0 = s0 + ((j + 1 == cnt && myLong) ? myLong : lz_rec_len(r));
            LZ_CLEAR(s0 > R ? s0 : R, e0);
        }
#undef LZ_CLEAR
#pragma unroll
        for (int k = 0; k < 4; k++) { mask[4 * tid + k] = m4[k]; myLit += (uint32_t)__popc(m4[k]); }

        // -- per warp: the kept records of the 32 lanes, flattened, 32 sequences per step, so that every store of the
        //    step is one coalesced access (lane l handles flat index f + l; its owner lane is found by a binary search
        //    over the lanes' exclusive counts; the previous sequence's end and offset come from the neighbouring lane)
        {
            const uint32_t incl = warp_scan_incl(kept), excl = incl - kept;
            const uint32_t total = __shfl_sync(FULLMASK, incl, 31);
            const uint32_t gbase = __shfl_sync(FULLMASK, seqEx, 0);
            uint32_t carryE = __shfl_sync(FULLMASK, prevE0, 0), carryD = __shfl_sync(FULLMASK, pOff0, 0);
            for (uint32_t f0 = 0; f0 < total; f0 += 32) {
                const uint32_t f = f0 + lane;
                const bool live = f < total;
                uint32_t o = 0;                        // owner: the largest lane whose exclusive count is <= f
#pragma unroll
                for (int st = 16; st > 0; st >>= 1) {
                    const uint32_t c = o + st;
                    const uint32_t v = __shfl_sync(FULLMASK, excl, (int)(c & 31));
                    if (c < 32 && v <= f) o = c;
                }
                const uint32_t oExcl = __shfl_sync(FULLMASK, excl, (int)o), oFirst = __shfl_sync(FULLMASK, firstKept, (int)o);
                const uint32_t oCnt = __shfl_sync(FULLMASK, cnt, (int)o), oLong = __shfl_sync(FULLMASK, myLong, (int)o);
                const uint32_t oR = __shfl_sync(FULLMASK, R, (int)o);
                uint32_t s2 = 0, e0 = 0, d0 = 0;
                if (live) {
                    const uint32_t ot = (tid & ~31u) + o, j = oFirst + (f - oExcl);
                    const uint32_t r = REC(j, ot);
                    const uint32_t s0 = ot * LZ_RANGE + lz_rec_rel(r);
                    e0 = s0 + ((j + 1 == oCnt && oLong) ? oLong : lz_rec_len(r));
                    s2 = s0 > oR ? s0 : oR;
                    d0 = lz_rec_d(r);
                }
                uint32_t pe = __shfl_up_sync(FULLMASK, e0, 1), pd = __shfl_up_sync(FULLMASK, d0, 1);
                if (lane == 0) { pe = carryE; pd = carryD; }
                if (live) {
                    const uint32_t gi = gbase + f, ll = s2 - pe, l2 = e0 - s2;
                    // repeat code 1 (= offset of the previous sequence, valid with litLen > 0; seqdec.go:463-500)
                    const bool isrep = (gi > 0) && (d0 == pd) && (ll > 0);
                    const uint32_t ofv = isrep ? 1u : d0 + 3;
                    wlen.put(gi, ll, l2 - 3); wof[gi] = ofv;
                    const uint32_t cll = seq_ll_code(ll), cof = highbit32(ofv), cml = seq_ml_code(l2 - 3);
                    wcodes[TBL_LL * mseq + gi] = (uint8_t)cll;
                    wcodes[TBL_OF * mseq + gi] = (uint8_t)cof;
                    wcodes[TBL_ML * mseq + gi] = (uint8_t)cml;
                    if (kind == 0) {      // (only compressed candidates use the histograms)
                        atomicAdd(&hcnt[256 + 64 * TBL_LL + cll], 1u);
                        atomicAdd(&hcnt[256 + 64 * TBL_OF + cof], 1u);
                        atomicAdd(&hcnt[256 + 64 * TBL_ML + cml], 1u);
                    }
                }
                carryE = __shfl_sync(FULLMASK, e0, 31); carryD = __shfl_sync(FULLMASK, d0, 31);
            }
        }
    }
    B2C_PHASE(11);
    if (tid == 0) { sh->kind = kind; sh->rleLen = 0; }
    __syncthreads();
    // single-sequence RLE block test (blockenc.go:484-493); nlit <= 1
    if (kind == 0 && nseq == 1 && nlit <= 1 && tid == 0) {
        const uint32_t ll0 = wlen.peek_ll(0), of0 = wof[0];
        if (ll0 == nlit && of0 - 3 == 1) { sh->kind = 2; sh->rleLen = wlen.peek_ml(0) + 3 + ll0; }
        else if (saved < 16) sh->kind = 1;
    } else if (kind == 0 && nseq == 1 && saved < 16 && tid == 0) sh->kind = 1;
    uint32_t litEx, litTotal;
    litEx = group_scan_excl(myLit, sh->ws, 0, NT, tid, &litTotal);   // literal index of this thread's first literal
    __syncthreads();
    kind = sh->kind;
    B2C_PHASE(4);

    // ---------------------------------------------------------------- P6: literals by stream compaction
    // Warp w compacts the 4 KiB its own lanes walked: per step the 128 bytes of one range (lane j: word j), the four mask
    // bits of the word select the literal bytes, a warp scan gives their places, byte stores go out in order (a step
    // writes at most 128 consecutive bytes).  The literal index of a byte is its rank under the mask, which is exactly
    // the order blockEnc.literals has (every sequence's literals precede its match).
    if (kind == 0) {
        // per-warp staging (the match records are dead): literal bytes are collected in shared memory at the same
        // 16-byte phase as their destination and leave as 16-byte vectors; only the ragged ends use byte stores
        constexpr uint32_t STG = L::REC_BYTES / (NT / 32);               // bytes of staging per warp
        uint8_t *stg = smem + L::SM_REC + w * STG;
        uint8_t *glit = wk_lit(P, chunk);
        uint32_t gpos = __shfl_sync(FULLMASK, litEx, 0);                // literal index of staging byte `ph`
        uint32_t ph = (uint32_t)((reinterpret_cast<uintptr_t>(glit) + gpos) & 15), fill = 0;
        const uint32_t nr = (w * 32 * LZ_RANGE >= n) ? 0u : ((n - w * 32 * LZ_RANGE + LZ_RANGE - 1) / LZ_RANGE < 32 ? (n - w * 32 * LZ_RANGE + LZ_RANGE - 1) / LZ_RANGE : 32u);
        // four ranges (512 bytes) per step: one warp scan serves all four (the four counts travel in the bytes of one word,
        // each at most 128); the literal bytes of a word are gathered with one byte permute (selector table by mask nibble)
        for (uint32_t i0 = 0;; i0 += 4) {
            const bool last = i0 >= nr;
            if (last || ph + fill + 512 > STG) {
                lz_warp_flush(stg, ph, fill, glit + gpos, lane);
                gpos += fill; fill = 0;
                ph = (uint32_t)((reinterpret_cast<uintptr_t>(glit) + gpos) & 15);
            }
            if (last) break;
            uint32_t nib[4], pc = 0;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t t = w * 32 + i0 + q;
                const uint32_t mw = (i0 + q < nr) ? mask[4 * t + (lane >> 3)] : 0u;
                nib[q] = (mw >> (4 * (lane & 7))) & 15u;
                pc |= (uint32_t)__popc(nib[q]) << (8 * q);
            }
            const uint32_t incl = warp_scan_incl(pc);
            const uint32_t tots = __shfl_sync(FULLMASK, incl, 31);
            if (tots == 0) continue;
            uint32_t rbase = ph + fill;
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const uint32_t c = (pc >> (8 * q)) & 0xffu;
                if (c) {
                    const uint32_t v = srcw[32 * (w * 32 + i0 + q) + lane];
                    const uint32_t packed = __byte_perm(v, 0u, (uint32_t)plut[nib[q]]);
                    uint8_t *o = stg + rbase + ((incl >> (8 * q)) & 0xffu) - c;
                    o[0] = (uint8_t)packed;
                    atomicAdd(&hcnt[packed & 0xffu], 1u);
                    if (c > 1) { o[1] = (uint8_t)(packed >> 8); atomicAdd(&hcnt[(packed >> 8) & 0xffu], 1u); }
                    if (c > 2) { o[2] = (uint8_t)(packed >> 16); atomicAdd(&hcnt[(packed >> 16) & 0xffu], 1u); }
                    if (c > 3) { o[3] = (uint8_t)(packed >> 24); atomicAdd(&hcnt[packed >> 24], 1u); }
                }
                rbase += (tots >> (8 * q)) & 0xffu;
            }
            fill = rbase - ph;
        }
    }
#undef REC
    if (tid == 0) { W->n = nblk; W->nseq = nseq; W->nlit = nlit; W->kind = kind; W->rleLen = sh->rleLen; }
    __syncthreads();
    if (kind == 0) {
        // histograms of a compressed candidate (zstd_tables_chunk reads them for no other kind); warp t < 3 publishes code
        // table t and its highest used code
        for (uint32_t i = tid; i < 256; i += NT) W->litHist[i] = hcnt[i];
        if (w < 3) {
            const uint32_t lo = hcnt[256 + 64 * w + lane], hi = hcnt[256 + 64 * w + 32 + lane];
            W->seqHist[w][lane] = lo; W->seqHist[w][32 + lane] = hi;
            const unsigned nzLo = __ballot_sync(FULLMASK, lo != 0), nzHi = __ballot_sync(FULLMASK, hi != 0);
            if (lane == 0)
                W->maxSym[w] = nzHi ? 32 + (31 - (uint32_t)__clz((int)nzHi)) : (nzLo ? 31 - (uint32_t)__clz((int)nzLo) : 0u);
        }
    }
    B2C_PHASE(5);
    }   // zstd mode
}

#ifdef B2C_EMU
// CPU emulator only (tests/emu runs it between the parse and the tables): recounts the histograms of every compressed
// candidate from the literals and codes in the work pool and compares them, and the highest used codes, with what the
// parse counted.  A difference turns the chunk into an error (kind 3: its output size is negative), so every test of
// the emulated encoder fails on it.  The device pipeline has no such pass.
constexpr int HIST_NT = 128;
constexpr uint32_t HIST_SMEM_BYTES = LZ_HIST_WORDS * 4 + 16;
B2C_DEV void zstd_hist_chunk(uint8_t *smem, const ZstdEncParams &P, uint32_t chunk) {
    const unsigned tid = threadIdx.x;
    ChunkWork *W = P.work + chunk;
    uint32_t *h = reinterpret_cast<uint32_t *>(smem);       // [0, 256) literal bytes | 256 + 64 * table + code
    uint32_t *bad = h + LZ_HIST_WORDS;
    for (uint32_t i = tid; i < LZ_HIST_WORDS; i += HIST_NT) h[i] = 0;
    if (tid == 0) *bad = 0;
    __syncthreads();
    const bool cand = W->kind == 0;
    if (cand) {
        const uint8_t *lit = wk_lit(P, chunk);
        for (uint32_t i = tid; i < W->nlit; i += HIST_NT) atomicAdd(&h[lit[i]], 1u);
        for (int t = 0; t < 3; t++) {
            const uint8_t *codes = wk_codes(P, chunk, t);
            for (uint32_t i = tid; i < W->nseq; i += HIST_NT) atomicAdd(&h[256 + 64 * t + (codes[i] & 63u)], 1u);
        }
    }
    __syncthreads();
    if (cand) {
        for (uint32_t i = tid; i < 256; i += HIST_NT)
            if (h[i] != W->litHist[i]) *bad = 1;
        for (uint32_t i = tid; i < 192; i += HIST_NT)
            if (h[256 + i] != W->seqHist[i / 64][i % 64]) *bad = 1;
        if (tid < 3) {
            uint32_t mx = 0;
            for (uint32_t c = 0; c < 64; c++)
                if (h[256 + 64 * tid + c]) mx = c;
            if (mx != W->maxSym[tid]) *bad = 1;
        }
    }
    __syncthreads();
    if (tid == 0 && *bad) W->kind = 3;
    __syncthreads();
}
#endif

#ifndef B2C_EMU
// The parse kernels are persistent (one CTA per resident slot); chunks are handed out through a global counter, so a CTA
// that starts late (its SM was busy with another stream's kernel) or meets slow chunks simply takes fewer of them.  The
// output of a chunk does not depend on the CTA that parses it (the per-CTA scratch holds nothing across chunks).
template <int LV, int MODE> B2C_DEV void lz_parse_loop(uint8_t *smem, const ZstdEncParams &P) {
    uint8_t *scratch = P.scratch + (uint64_t)blockIdx.x * LzLayout<LV>::SCRATCH_BYTES;
    ParseShared *sh = reinterpret_cast<ParseShared *>(smem + LzLayout<LV>::SM_SH);
    for (;;) {
        __syncthreads();                                     // the previous chunk's last reads of the shared record
        if (threadIdx.x == 0) sh->nextChunk = atomicAdd(P.counter, 1u);
        __syncthreads();
        const uint32_t c = sh->nextChunk;
        if (c >= P.nchunks) break;
        lz_parse_chunk<LV, MODE>(smem, P, c, scratch);
    }
}
#define B2C_LZ_KERNEL(name, LV, MODE)                                                                                      \
    extern "C" __global__ void __launch_bounds__(LzCfg<LV>::NT, LzCfg<LV>::MIN_CTAS) name(ZstdEncParams P) {               \
        extern __shared__ __align__(1024) uint8_t smem[];                                                                  \
        lz_parse_loop<LV, MODE>(smem, P);                                                                                  \
    }
B2C_LZ_KERNEL(b2c_lz_parse1_kernel, 1, LZ_MODE_ZSTD)
B2C_LZ_KERNEL(b2c_lz_parse2_kernel, 2, LZ_MODE_ZSTD)
B2C_LZ_KERNEL(b2c_lz_parse3_kernel, 5, LZ_MODE_ZSTD)
// S2 / Snappy block encoders: the same parse, tag-stream emission instead of the entropy stages (one kernel per block batch)
B2C_LZ_KERNEL(b2c_lz_s2_fast_kernel, 3, LZ_MODE_S2)
B2C_LZ_KERNEL(b2c_lz_snappy_fast_kernel, 3, LZ_MODE_SNAPPY)
B2C_LZ_KERNEL(b2c_lz_s2_better_kernel, 4, LZ_MODE_S2)
B2C_LZ_KERNEL(b2c_lz_snappy_better_kernel, 4, LZ_MODE_SNAPPY)
#undef B2C_LZ_KERNEL
#endif

}  // namespace b2c
