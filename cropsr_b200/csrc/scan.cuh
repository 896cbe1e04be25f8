// Device side of libcropsr_b200: pack, scan + score, segment counts, rescore (sm_100a).
//
// HBM layout of a packed genome shard: an array of TILE RECORDS (plus, per tile, a PAM record and a
// header, below), one per 16384 token
// positions of a segment, each record self-contained so that ONE bulk (TMA) copy stages
// everything a CTA needs for the tile:
//     word 0            descriptor {t_start, token length L, owned positions n, segment}
//     word 1            halo: the 32 positions before the tile
//     words 2 .. 513    the tile: 512 words of 32 positions
//     word 514          halo: the 32 positions after the tile
// A word is a uint4 of four 32-position bit planes {code low bit, code high bit (A0 T1 C2
// G3, CROPSR.py:300-302), lower-case, other byte}: 0.5 byte per base.
//
// k_scan_score is one cooperative, persistent launch:
//   count phase   every CTA takes the PAM hit counts of a contiguous range of tiles from their 48-byte
//                 headers (k_pack counted every 2,048-position chunk; only the tiles at the ends of a
//                 token, where the bounds depend on the guide length, are counted again from their PAM
//                 records) and publishes the range total and the range-local exclusive prefix of every
//                 chunk (ranges of any length are walked in batches of 256 tiles with a running prefix:
//                 one count phase, one grid barrier, one tail for a genome of any size);
//   grid barrier, every CTA scans the range totals into shared memory;
//   emit phase    tiles are handed out dynamically; the global output offset of a tile is
//                 range prefix + tile prefix (one load), so there is no ordering between
//                 CTAs and no spinning.  Hits are compacted through shared memory and one
//                 thread per candidate extracts the 30-base window from the staged words,
//                 scores it (fp64, canonical OpenBLAS lane order) and stores
//                 (pos, packed 30-mer, x) coalesced into the two ordered strand streams.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "npexp.cuh"
#include "rs1.cuh"

namespace cg = cooperative_groups;

// ------------------------------------------------------------------ geometry
#ifndef CRP_CTAS_PER_SM
#define CRP_CTAS_PER_SM 4                                   // resident CTAs per SM the scan kernel is compiled for (64 registers)
#endif
static constexpr int kThreads = 256;
static constexpr int kWarps = kThreads / 32;
static constexpr int kTileWords = 2 * kThreads;            // every thread owns word tid and word tid + 256
static constexpr int kTile = kTileWords * 32;              // 16384 positions
static constexpr int kRecWords = kTileWords + 3;           // descriptor + halo + tile + halo
static constexpr uint32_t kRecBytes = kRecWords * 16;      // 8240, one bulk copy
static constexpr int kStages = 2;                          // staged tiles per CTA
static constexpr int kListCap = 1024;                      // hits per strand of a tile compacted in one go
static constexpr int kPrefWords = 10;                      // per tile: 8 warp prefixes, tile total, pad (80 B, one bulk copy)
static constexpr uint32_t kNoTile = 0xFFFFFFFFu;
static constexpr int kMaxPeers = 8;                        // GPUs of one box
static constexpr uint32_t kAlign = 128;                    // positions; segment placement granularity

// PAM record of a tile, read by the count phase instead of the full record: descriptor, then for
// the 512 tile words and the right halo word the two planes the PAM tests need (upper-case G,
// upper-case C) -- 0.25 byte per base
static constexpr int kPamWords = kTileWords + 1;           // uint2 {upper G, upper C} each
static constexpr uint32_t kPamBytes = (16 + kPamWords * 8 + 15) / 16 * 16;   // 4128, one bulk copy
static constexpr int kCountStages = 6;                     // slots of the ring control block: sized for the PAM-record ring the count phase
                                                           // ran until it moved to tile headers; it now uses mbarrier 0, the emit phase kStages
// Tile header, read by the count phase: the descriptor and the PAM hits of the tile's eight 2,048-position
// chunks (plus | minus << 16) counted by k_pack under every bound that does not depend on the guide
// length -- ownership, t <= L - 3, '-' t >= 2.  Only a tile that reaches into the first l + 5 or the last
// l - 7 positions of its token (CROPSR.py:419 / :430) is counted again at scan time, from its PAM record.
struct __align__(16) TileHdr {
    uint4 desc;
    uint32_t cnt[8];
};
static_assert(sizeof(TileHdr) == 48, "bulk copies move multiples of 16 bytes");
static constexpr uint32_t kPackItems = 544;                // k_pack: threads per tile (17 warps; 515 of them write a record word)
static_assert(kPackItems % 32 == 0 && kPackItems >= (uint32_t)kRecWords, "whole warps per tile");
static constexpr int kHdrBatch = 256;                      // tile headers of a CTA's count range staged and scanned at once (12 KB)
static_assert(kRecBytes % 16 == 0, "bulk copies move multiples of 16 bytes");

// record word 0
struct TileDesc {
    uint32_t t_start;   // token-relative position of the tile's first position
    uint32_t L;         // token length
    uint32_t n;         // positions of this tile owned by the segment (<= kTile)
    uint32_t segment;   // index of the segment in the genome
};

// what k_pack needs to build one record
struct PackDesc {
    uint64_t ascii_off;  // offset in the ASCII staging buffer of token position stage_begin
    uint32_t stage_begin, stage_end;   // token positions present in the staging buffer
    TileDesc td;
};

// ------------------------------------------------------------------ k_pack
// bits b of a 32-position word starting at token position t0 with lo <= t0+b <= hi
CRP_HD uint32_t range_mask(int32_t t0, int32_t lo, int32_t hi) {
    int32_t a = lo - t0, b = hi - t0;
    if (a < 0) a = 0;
    if (b > 31) b = 31;
    if (a > b) return 0u;
    return (0xFFFFFFFFu >> (31 - b)) & (0xFFFFFFFFu << a);
}

// PAM hits of one tile word under the bounds that hold for every guide length (what a tile header counts):
// g / c = upper-case G / C of the word's 32 positions, gn / cn = of the two positions after it, tw = token
// position of bit 0.  '+' t <= min(L - 3, last owned position); '-' 2 <= t <= the same.  -> plus | minus << 16
CRP_HD uint32_t pack_word_hits(uint32_t g, uint32_t c, uint32_t gn, uint32_t cn, int32_t tw, const TileDesc td) {
    uint32_t hp = crp_funnel_r(g, gn, 1) & crp_funnel_r(g, gn, 2), hm = c & crp_funnel_r(c, cn, 1);
    const int32_t hi_p = min((int32_t)td.L - 3, (int32_t)td.t_start + (int32_t)td.n - 1);
    if (tw < 2 || tw + 31 > hi_p) {                    // first word of a token, last words of a token or of a segment
        hp &= range_mask(tw, 0, hi_p);
        hm &= range_mask(tw, 2, hi_p);
    }
    return (uint32_t)crp_popc(hp) | ((uint32_t)crp_popc(hm) << 16);
}

// byte -> nibble: bit0 code low, bit1 code high (A0 T1 C2 G3), bit2 lower-case, bit3 other.
// 'U' and 'Z' are "other" bytes that still score (reference replace chains,
// CROPSR.py:120,128,458): they carry the code of T resp. G.
__host__ __device__ inline uint32_t classify(uint32_t c) {
    uint32_t up = c & 0xDFu;
    uint32_t r = 8u;
    if (up == 'A') r = 0u;
    else if (up == 'T') r = 1u;
    else if (up == 'C') r = 2u;
    else if (up == 'G') r = 3u;
    if (r < 8u) return r | ((c & 0x20u) >> 3);
    if (c == 'U') return 8u | 1u;
    if (c == 'Z') return 8u | 3u;
    return 8u;
}

// One thread per record word.  Positions outside the staged part of the token become
// "other" bytes (they never match a PAM and never score).
// descs == NULL: the shard is ONE segment, described by `one` (descriptor of its first tile,
// td.n = positions of the whole segment); tile j then follows by arithmetic, so that a
// pipelined ingest needs no descriptor upload.
// The byte classes come from a 256-entry table whose entries hold the four plane bits one per
// BYTE lane (code low | code high << 8 | lower << 16 | other << 24): eight consecutive bases
// accumulate as  acc += entry << k  (one IMAD each, no bit twiddling), which leaves 8 positions
// of every plane in one byte of acc, and byte permutes assemble the 32-position planes.
// hdr (zeroed before the launch): the descriptor again and the chunk counts of TileHdr -- the 16 warps that
// pack the 512 tile words of a tile add the hits of their 32 words with one atomic each.
// n_items = tiles * kPackItems.
__global__ void __launch_bounds__(256, 8)
k_pack(const uint8_t *__restrict__ ascii, const PackDesc *__restrict__ descs, const PackDesc one, uint64_t n_items,
       uint4 *__restrict__ records, unsigned char *__restrict__ pam, TileHdr *__restrict__ hdr) {
    __shared__ uint32_t lut[256];
    {
        const uint32_t nib = classify(threadIdx.x);
        lut[threadIdx.x] = (nib & 1u) | ((nib >> 1) & 1u) << 8 | ((nib >> 2) & 1u) << 16 | ((nib >> 3) & 1u) << 24;
    }
    __syncthreads();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t item = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; item < n_items; item += stride) {
        // items of a tile: its 512 tile words (16 warps: every warp sits inside ONE chunk of one tile), then the
        // descriptor, the two halo words and 29 idle slots (the 17th warp)
        const uint64_t tile = item / kPackItems;
        const uint32_t i = (uint32_t)(item - tile * kPackItems);
        const uint32_t k = i < (uint32_t)kTileWords ? i + 2u : i == (uint32_t)kTileWords ? 0u : i == (uint32_t)kTileWords + 1u ? 1u : (uint32_t)kTileWords + 2u;
        const uint64_t it = tile * kRecWords + k;              // record word
        uint32_t hits = 0;                                     // (plus | minus << 16) of a tile word
        uint32_t pg = 0, pc = 0;                               // upper-case G / C planes of my word
        TileDesc td = {0u, 0u, 0u, 0u};
        uint64_t ascii_off = 0;
        uint32_t stage_lo = 0, stage_hi = 0;
        if (i < (uint32_t)kTileWords + 3u) {
            PackDesc pd;
            if (descs) {
                pd = descs[tile];
            } else {
                pd = one;
                const uint32_t done = (uint32_t)tile * (uint32_t)kTile;
                pd.td.t_start = one.td.t_start + done;
                pd.td.n = one.td.n - done < (uint32_t)kTile ? one.td.n - done : (uint32_t)kTile;
            }
            td = pd.td, ascii_off = pd.ascii_off, stage_lo = pd.stage_begin, stage_hi = pd.stage_end;
            if (k == 0) {
                const uint4 d = make_uint4(pd.td.t_start, pd.td.L, pd.td.n, pd.td.segment);
                records[it] = d;
                *reinterpret_cast<uint4 *>(pam + tile * kPamBytes) = d;
                hdr[tile].desc = d;
            } else {
                const int64_t p0 = (int64_t)pd.td.t_start + ((int64_t)k - 2) * 32;   // token position of bit 0
                const int64_t lo = pd.stage_begin, hi = pd.stage_end;
                uint32_t o0 = 0, o1 = 0, ol = 0, oo = 0;
                if (p0 >= lo && p0 + 32 <= hi) {
                    const uint4 *src = reinterpret_cast<const uint4 *>(ascii + pd.ascii_off + (uint64_t)(p0 - lo));
                    const uint4 a = __ldg(src), b = __ldg(src + 1);
                    const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                    uint32_t acc[4];
#pragma unroll
                    for (int g = 0; g < 4; ++g) {                  // 8 bases -> one byte of every plane
                        uint32_t s = 0;
#pragma unroll
                        for (int j = 0; j < 8; ++j) s += lut[(v[2 * g + (j >> 2)] >> (8 * (j & 3))) & 0xFFu] << j;
                        acc[g] = s;
                    }
                    const uint32_t t01 = __byte_perm(acc[0], acc[1], 0x5140), t23 = __byte_perm(acc[2], acc[3], 0x5140);
                    const uint32_t u01 = __byte_perm(acc[0], acc[1], 0x7362), u23 = __byte_perm(acc[2], acc[3], 0x7362);
                    o0 = __byte_perm(t01, t23, 0x5410);
                    o1 = __byte_perm(t01, t23, 0x7632);
                    ol = __byte_perm(u01, u23, 0x5410);
                    oo = __byte_perm(u01, u23, 0x7632);
                } else {
                    for (int bit = 0; bit < 32; ++bit) {
                        const int64_t p = p0 + bit;
                        uint32_t e = 1u << 24;
                        if (p >= lo && p < hi) e = lut[ascii[pd.ascii_off + (uint64_t)(p - lo)]];
                        o0 |= (e & 1u) << bit;
                        o1 |= ((e >> 8) & 1u) << bit;
                        ol |= ((e >> 16) & 1u) << bit;
                        oo |= ((e >> 24) & 1u) << bit;
                    }
                }
                records[it] = make_uint4(o0, o1, ol, oo);
                if (k >= 2) {                       // tile words and the right halo: the planes of the PAM tests
                    const uint32_t up = ~(ol | oo);
                    const uint32_t g = o0 & o1 & up, c = ~o0 & o1 & up;
                    reinterpret_cast<uint2 *>(pam + tile * kPamBytes + 16)[k - 2] = make_uint2(g, c);
                    pg = g, pc = c;
                }
            }
        }
        // ---- hits of the tile words under the guide-independent bounds.  The warp is whole here (n_items is a
        // multiple of 32), its lanes hold 32 consecutive words of ONE chunk: the two positions after a word are
        // the next lane's, the last lane reads its two bytes.
        if (i < (uint32_t)kTileWords) {
            uint32_t gn = __shfl_down_sync(0xFFFFFFFFu, pg, 1), cn = __shfl_down_sync(0xFFFFFFFFu, pc, 1);
            const int64_t p0 = (int64_t)td.t_start + (int64_t)i * 32;
            if ((threadIdx.x & 31) == 31) {
                gn = 0, cn = 0;
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int64_t q = p0 + 32 + j;
                    if (q >= (int64_t)stage_lo && q < (int64_t)stage_hi) {
                        const uint32_t ch = ascii[ascii_off + (uint64_t)(q - stage_lo)];
                        gn |= (uint32_t)(ch == 'G') << j;
                        cn |= (uint32_t)(ch == 'C') << j;
                    }
                }
            }
            hits = pack_word_hits(pg, pc, gn, cn, (int32_t)p0, td);
        }
        // the warp is whole here (n_items is a multiple of 32) and inside one chunk: one add per warp
        const uint32_t sum = __reduce_add_sync(0xFFFFFFFFu, hits);
        if ((threadIdx.x & 31) == 0 && sum) atomicAdd(&hdr[tile].cnt[i / 64u], sum);
    }
}

// ------------------------------------------------------------------ k_fasta_strip
// Device side of the formatted-path ingest (CROPSR.py:54-74 with cropsr_functions.py:221-229):
// the sequence lines of one FASTA record, exactly as they sit in the file, become the token
// the reference scans:  ' + bases + ') + (, or ] for the last record).  The record must be
// "plain": every line `width` bases long except the last one, '\n' line ends, printable
// non-blank ASCII without quotes or backslashes -- then str(list_of_tuples) changes nothing
// but the decoration.  Anything else sets *bad (the host then falls back to the literal
// Python ingest); so does a base where a line end is due or the other way round.  The host
// derives n_bases from the byte count of the record and `width`, so every byte is accounted for.
struct FastaRec {
    uint64_t raw_off;     // first sequence byte of the record in the raw buffer
    uint64_t ascii_off;   // token position 0 in the ASCII staging buffer (16-byte aligned)
    uint64_t first_item;  // 16-byte output groups before this record
    uint32_t n_bases, width;
    uint32_t last, pad;   // last: last record of the file (its token ends in ')]', not '),')
};

// Bases of a record of n_bytes > 0 sequence bytes ending in last_byte, in lines of width > 0 bases: one line end per
// full line, the last one optional.  0 when no such lines give that byte count (a whole number of width + 1 byte lines).
inline uint64_t fasta_record_bases(uint64_t n_bytes, uint8_t last_byte, uint32_t width) {
    const uint64_t body = last_byte == '\n' ? n_bytes - 1 : n_bytes;
    const uint64_t k = body / ((uint64_t)width + 1), r = body % ((uint64_t)width + 1);
    return r ? k * width + r : 0;
}

// the byte loads of k_fasta_strip, with a host twin: tests/fasta_strip_emu.cu runs fasta_strip_group on the CPU
CRP_HD uint32_t crp_ldg_u8(const uint8_t *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}

// One item of k_fasta_strip: the 16 token bytes of record r from token position p0 (a multiple of 16) into w[4],
// four per word, little-endian.  Returns 1 if a byte it reads breaks the record's plainness.
CRP_HD unsigned int fasta_strip_group(const uint8_t *__restrict__ raw, const FastaRec &r, uint64_t p0, uint32_t w[4]) {
    const uint64_t n = r.n_bases, L = n + 4;
    uint64_t b = p0 ? p0 - 1 : 0;                  // base index of the first base byte of the group
    uint64_t line = b / r.width;
    uint32_t col = (uint32_t)(b - line * r.width);
    const uint8_t *src = raw + r.raw_off + b + line;
    if (b && !col) {                               // the group starts a line: the line end before it is this group's
        col = r.width;                             // to check (the group before stops at the last base of the line)
        --src;
    }
    unsigned int err = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const uint64_t p = p0 + i;
        uint32_t c = 0;
        if (p == 0 || p == n + 1) c = '\'';
        else if (p == n + 2) c = ')';
        else if (p == n + 3) c = r.last ? ']' : ',';
        else if (p < L) {
            if (col == r.width) {                  // a line end is due here
                if (crp_ldg_u8(src) != '\n') err = 1;
                ++src;
                col = 0;
            }
            c = crp_ldg_u8(src++);
            ++col;
            if (c <= 0x20 || c >= 0x7F || c == '\'' || c == '"' || c == '\\' || c == '>') err = 1;
        }
        w[i >> 2] |= c << (8 * (i & 3));
    }
    return err;
}

__global__ void __launch_bounds__(256)
k_fasta_strip(const uint8_t *__restrict__ raw, const FastaRec *__restrict__ recs, uint32_t n_recs, uint64_t n_items,
              uint8_t *__restrict__ ascii, unsigned int *__restrict__ bad) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; it < n_items; it += stride) {
        uint32_t lo = 0, hi = n_recs;                  // last record with first_item <= it
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (recs[mid].first_item <= it) lo = mid;
            else hi = mid;
        }
        const FastaRec r = recs[lo];
        const uint64_t p0 = (it - r.first_item) * 16;  // token position of output byte 0
        uint32_t w[4] = {0, 0, 0, 0};
        const unsigned int err = fasta_strip_group(raw, r, p0, w);
        *reinterpret_cast<uint4 *>(ascii + r.ascii_off + p0) = make_uint4(w[0], w[1], w[2], w[3]);
        if (err) atomicOr(bad, 1u);
    }
}

// ------------------------------------------------------------------ small device helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
    const uint32_t b = smem_u32(bar);
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(b),
        "r"(parity)
        : "memory");
}

struct Hits {
    uint32_t pA, mA, pB, mB;   // '+' / '-' hit masks of the lane's two words (A: first half of the warp chunk, B: second)
};

// PAM tests and bounds of this lane's two words of a staged tile.  Warp w owns the 64 words
// [64w, 64w + 64) of the tile (2048 positions); lane l owns words 64w + l (A) and 64w + 32 + l (B).
//   '+': (?=.GG) at t  <=>  tok[t+1]==tok[t+2]=='G'            (CROPSR.py:415)
//   '-': (?=CC.) at t  <=>  tok[t]==tok[t+1]=='C' and t+2 < L  (CROPSR.py:426)
//   bounds (CROPSR.py:419 / :430): '+' t >= l+5;  '-' 2 <= t <= L-l+7
//   plus ownership: t inside the n positions of the tile that the segment owns.
// All positions fit int32: L < 2^31 - 2^15 (crp_genome_add_segment), 1 <= l <= 10^6.
CRP_HD Hits hits_from_planes(uint32_t gA, uint32_t gAn, uint32_t cA, uint32_t cAn, uint32_t gB, uint32_t gBn, uint32_t cB,
                             uint32_t cBn, const TileDesc td, int l, int wordA) {
    Hits h;
    h.pA = crp_funnel_r(gA, gAn, 1) & crp_funnel_r(gA, gAn, 2);
    h.pB = crp_funnel_r(gB, gBn, 1) & crp_funnel_r(gB, gBn, 2);
    h.mA = cA & crp_funnel_r(cA, cAn, 1);
    h.mB = cB & crp_funnel_r(cB, cBn, 1);
    const int32_t t0 = (int32_t)td.t_start, L = (int32_t)td.L;
    const int32_t last_owned = t0 + (int32_t)td.n - 1;
    const int32_t hi_p = min(L - 3, last_owned);
    const int32_t hi_m = min(L - l + 7, hi_p);
    if (t0 < l + 5 || t0 + kTile - 1 > hi_m) {   // edge tiles only
        const int32_t tA = t0 + 32 * wordA, tB = tA + 32 * 32;
        h.pA &= range_mask(tA, l + 5, hi_p);
        h.pB &= range_mask(tB, l + 5, hi_p);
        h.mA &= range_mask(tA, 2, hi_m);
        h.mB &= range_mask(tB, 2, hi_m);
    }
    return h;
}

CRP_HD Hits tile_hits(const uint4 *__restrict__ rec, const TileDesc td, int l, int wordA) {
    const uint4 a = rec[2 + wordA], an = rec[3 + wordA], b = rec[34 + wordA], bn = rec[35 + wordA];
    const uint32_t uA = ~(a.z | a.w), uAn = ~(an.z | an.w), uB = ~(b.z | b.w), uBn = ~(bn.z | bn.w);   // upper-case ACGT
    return hits_from_planes(a.x & a.y & uA, an.x & an.y & uAn, ~a.x & a.y & uA, ~an.x & an.y & uAn, b.x & b.y & uB,
                            bn.x & bn.y & uBn, ~b.x & b.y & uB, ~bn.x & bn.y & uBn, td, l, wordA);
}

// Count phase, tiles at the ends of a token: ONE warp counts a whole PAM record straight from global memory.
// Lane l owns the words 32 i + l (i = 0 .. 15); warp chunk c of the tile (what a warp of the emit phase
// compacts) is the words [64 c, 64 c + 64), i.e. iterations 2 c and 2 c + 1.  cnt[c] = (plus | minus << 16)
// of chunk c.  The loads of eight iterations are issued together: two round trips to memory per tile.
__device__ __forceinline__ void warp_count_tile(const unsigned char *__restrict__ rec, int l, int lane,
                                                uint32_t *__restrict__ cnt) {
    const uint4 d = __ldg(reinterpret_cast<const uint4 *>(rec));
    const uint2 *w = reinterpret_cast<const uint2 *>(rec + 16);
    const int32_t t0 = (int32_t)d.x, L = (int32_t)d.y;
    const int32_t last_owned = t0 + (int32_t)d.z - 1;
    const int32_t hi_p = min(L - 3, last_owned);
    const int32_t hi_m = min(L - l + 7, hi_p);
    const bool edge = t0 < l + 5 || t0 + kTile - 1 > hi_m;         // warp-uniform
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        uint2 a[8], an[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int word = 32 * (8 * half + i) + lane;
            a[i] = __ldg(w + word);
            an[i] = __ldg(w + word + 1);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t n = 0;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int i = 2 * c + h, word = 32 * (8 * half + i) + lane;
                uint32_t p = __funnelshift_r(a[i].x, an[i].x, 1) & __funnelshift_r(a[i].x, an[i].x, 2);
                uint32_t m = a[i].y & __funnelshift_r(a[i].y, an[i].y, 1);
                if (edge) {
                    const int32_t tw = t0 + 32 * word;
                    p &= range_mask(tw, l + 5, hi_p);
                    m &= range_mask(tw, 2, hi_m);
                }
                n += __popc(p) | (__popc(m) << 16);
            }
            n = __reduce_add_sync(0xFFFFFFFFu, n);
            if (lane == 0) cnt[4 * half + c] = n;
        }
    }
}

struct ScanArgs {
    const uint4 *records;            // n_tiles records of kRecWords words
    const unsigned char *pam;        // n_tiles PAM records of kPamBytes bytes (count phase, tiles at the ends of a token)
    const TileHdr *hdr;              // n_tiles tile headers (count phase)
    uint32_t n_tiles;
    uint32_t static_eighths;         // share of the tiles dealt round-robin, in 1/8 (the rest are ticketed)
    int guide_len;
    uint32_t flags;
    const double *tables;            // RS1 lane tables (RS1_TABLE_DOUBLES doubles)
    uint64_t capacity;               // entries per strand stream
    uint32_t *pos_plus, *pos_minus;
    unsigned long long *packed_plus, *packed_minus;
    double *x_plus, *x_minus;
    // scan state; nothing needs initialising before the launch.  Counts are (plus << 32) | minus.
    unsigned long long *warp_pref;   // [n_tiles][kPrefWords] exclusive prefix of every warp chunk inside its count range, then the tile total
    unsigned long long *cta_tot;     // [gridDim.x] range totals
    unsigned int *tickets;           // [0] emit-phase dispenser of the dynamic tiles, [1] CTAs done with the segment counts
    unsigned long long *seg_counts;  // [2 * seg_stride] out: plus[0..n_seg) then, from seg_stride on, minus[0..n_seg);
                                     // slots n_seg .. seg_stride-1 are zeroed (fixed-size block of a sharded scan's all-gather)
    unsigned long long *seg_counts_host;   // the same block again in mapped pinned host memory (or NULL): the host reads its
                                           // counts when the kernel's event has fired, without a copy that would queue behind
                                           // the row copies of earlier segments on the device-to-host engine
    unsigned int *fault;                   // CRP_CHECKED builds: first violated invariant (code | line << 8), else untouched
    const uint32_t *seg_first_tile, *seg_tile_count;   // [n_seg]
    uint32_t n_seg, seg_stride;
    // Sharded scan, fused exchange (world > 1): the segment counts also go -- plain stores over NVLink --
    // into every rank's gather buffer, followed by a flag; the kernel returns once the blocks of all ranks
    // have landed in its own buffer.  The all-gather of the counts hides behind the emit phase.
    uint32_t world, rank, epoch;     // world <= 1: no exchange
    unsigned long long *peer_gather[kMaxPeers];   // rank p's buffer of this epoch's parity: [world][2 * seg_stride]
    unsigned int *peer_flags[kMaxPeers];          // rank p's flags of this epoch's parity: [world], flag[r] = epoch once r's block is in
    unsigned int *xchg_error;        // set if a peer's block did not arrive in time
    unsigned long long xchg_timeout_ns;
};

// CRP_CHECKED builds (make checked): the kernel verifies its own invariants -- indices into the hit
// lists, the staged record, the count ring and the output streams, and that the emit phase finds in
// every warp chunk exactly the hits the count phase counted there -- and records the first violation
// in *fault instead of trapping (the context stays usable; the host turns it into CRP_ERR_STATE).
// This pool's compute-sanitizer is closed, so this is how out-of-bounds and ordering bugs are hunted.
#ifdef CRP_CHECKED
#define CRP_CHECK(a, cond, code)                                                            \
    do {                                                                                    \
        if (!(cond) && (a).fault) atomicCAS((a).fault, 0u, (unsigned)(code) | ((unsigned)__LINE__ << 8)); \
    } while (0)
#else
#define CRP_CHECK(a, cond, code) \
    do {                         \
    } while (0)
#endif

// every rank's block is in my gather buffer (or the timeout struck): spun by the first `world` threads of one CTA
__device__ __forceinline__ void xchg_wait(const ScanArgs &a) {
    if (threadIdx.x < a.world) {
        volatile unsigned int *flag = a.peer_flags[a.rank] + threadIdx.x;
        unsigned long long t0, t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        while (*flag != a.epoch) {
            __nanosleep(200);
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > a.xchg_timeout_ns) {
                atomicExch(a.xchg_error, 1u + threadIdx.x);
                break;
            }
        }
        __threadfence_system();
    }
}

// this rank's block is complete in every peer's buffer: raise the flags (one thread)
__device__ __forceinline__ void xchg_publish(const ScanArgs &a) {
    __threadfence_system();
    for (uint32_t p = 0; p < a.world; ++p) *reinterpret_cast<volatile unsigned int *>(a.peer_flags[p] + a.rank) = a.epoch;
}

// A rank whose shard has no tile still takes part in the exchange.
__global__ void k_exchange_empty(const ScanArgs a) {
    for (uint32_t sg = threadIdx.x; sg < 2 * a.seg_stride; sg += blockDim.x) {
        a.seg_counts[sg] = 0ull;
        if (a.seg_counts_host) a.seg_counts_host[sg] = 0ull;
        for (uint32_t p = 0; p < a.world; ++p) a.peer_gather[p][(size_t)a.rank * 2 * a.seg_stride + sg] = 0ull;
    }
    __syncthreads();
    if (threadIdx.x == 0 && a.world > 1) xchg_publish(a);
    if (a.world > 1) xchg_wait(a);
}

// optional phase timeline (tools/phase_timeline.py): 8 x u64 per CTA, or NULL
__device__ unsigned long long *g_dbg_times = nullptr;
__device__ __forceinline__ void dbg_stamp(int slot) {
    unsigned long long *p = g_dbg_times;
    if (p && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p[8ull * blockIdx.x + slot] = t;
    }
}

struct Window {
    uint32_t s0, s1, valid;              // planar codes / scoring mask of the 30-mer, output order
    unsigned long long packed;
};

// 30-base window of one hit out of the staged record.
// '+': tok[t-25, t+5) read backwards (output base q = tok[t+4-q]), upper-case bases complemented;
// '-': tok[t-2, t+28) read forwards.   ws = position inside the tile + kWinBias: the window start
// relative to the first halo position (the hit lists hold this biased value).
static constexpr uint32_t kWinBiasPlus = 7u, kWinBiasMinus = 30u;
template <bool kMinus>
CRP_HD Window extract_window(const uint4 *__restrict__ rec, uint32_t ws, uint32_t t, uint32_t L) {
    const uint32_t wi = 1u + (ws >> 5), sh = ws;            // shf.r.wrap uses the low 5 bits of the amount
    const uint4 lo = rec[wi], hi = rec[wi + 1];
    const uint32_t p0 = crp_funnel_r(lo.x, hi.x, sh), p1 = crp_funnel_r(lo.y, hi.y, sh);
    const uint32_t lw = crp_funnel_r(lo.z, hi.z, sh), ot = crp_funnel_r(lo.w, hi.w, sh);
    const uint32_t special = ot & p0;       // 'U' / 'Z': "other" bytes that still score
    const uint32_t valid = ~ot | special;
    Window w;
    if (kMinus) {
        w.s0 = (p0 ^ special) & 0x3FFFFFFFu;                 // U scores as A, Z as C
        w.s1 = p1 & 0x3FFFFFFFu;
        w.valid = valid & 0x3FFFFFFFu;
    } else {
        w.s0 = crp_brev(p0 ^ ~(lw | ot)) >> 2;               // A<->T, C<->G of upper-case bases flips the low code bit
        w.s1 = crp_brev(p1) >> 2;
        w.valid = crp_brev(valid) >> 2;
    }
    // flags without predicates: valid <= 0x3FFFFFFF, so bit 30 of valid + 1 is set iff all 30 bases
    // score; x <= 0x3FFFFFFF, so bit 30 of x + 0x3FFFFFFF is set iff x != 0
    const uint32_t hi32 = w.s1 | (~(w.valid + 1u) & (uint32_t)(CRP_PACKED_UNSCORED >> 32));
    const uint32_t irr = (lw | ot) & 0x3FFFFFFFu;
    uint32_t lo32 = w.s0 | ((irr + 0x3FFFFFFFu) & (uint32_t)CRP_PACKED_IRREGULAR);
    if (t + (kMinus ? 28u : 5u) > L) lo32 |= (uint32_t)CRP_PACKED_TRUNCATED;
    w.packed = ((unsigned long long)hi32 << 32) | lo32;
    return w;
}

__device__ __forceinline__ unsigned long long unpack_counts(uint32_t c) {   // (plus | minus << 16) -> plus << 32 | minus
    return ((unsigned long long)(c & 0xFFFFu) << 32) | (c >> 16);
}

// The emit phase's twin of extract_window + rs1_canonical: the same packed word and the same x from the same
// staged record, arranged for the instruction mix of the candidate loop, whose bound is the integer-ALU pipe
// (LOP3 / SHF / IADD3 issue every other cycle; multiplies run beside them on the FMA pipe):
//   * the class masks come straight from the shifted planes (one LOP3 each) and may carry junk in bits 30 / 31;
//   * '+' windows are shifted by ws - 2 (the hit list holds that: kWinBiasPlusHot), so that BREV alone aligns them;
//   * the word index, the truncation flag and the flag merges are multiplies / multiply-highs;
//   * flags are selected into the words (bit 31 of either flag source is provably clear).
// xt = L - (28 | 5) - (token position of list value 0): list value ws is truncated iff xt - ws < 0 (all < 2^31).
static constexpr uint32_t kWinBiasPlusHot = kWinBiasPlus - 2u;
template <bool kMinus>
CRP_HD double score_hit(const double *__restrict__ tab, const uint4 *__restrict__ rec, uint32_t ws, uint32_t xt,
                        unsigned long long &packed) {
    const uint32_t wbyte = crp_umulhi(ws, 1u << 27) * 16u;  // 16 * (ws >> 5)
    const uint4 lo = *reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(rec) + 16 + wbyte);
    const uint4 hi = *reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(rec) + 32 + wbyte);
    const uint32_t p0 = crp_funnel_r(lo.x, hi.x, ws), p1 = crp_funnel_r(lo.y, hi.y, ws);
    const uint32_t lw = crp_funnel_r(lo.z, hi.z, ws), ot = crp_funnel_r(lo.w, hi.w, ws);
    uint32_t xs;                                            // xt - ws, on the FMA pipe
#ifdef __CUDA_ARCH__
    asm("mad.lo.u32 %0, %1, 0xFFFFFFFF, %2;" : "=r"(xs) : "r"(ws), "r"(xt));
#else
    xs = xt - ws;
#endif
    const uint32_t trunc = crp_umulhi(xs, 2u);              // its sign bit
    constexpr uint32_t kWin = kMinus ? 0x3FFFFFFFu : 0xFFFFFFFCu;    // the window's 30 bits in the shifted planes
    uint32_t mA, mT, mC, mG, w0, w1;
    if (kMinus) {
        const uint32_t s0 = p0 & ~ot;                       // U scores as A, Z as C: "other" bytes lose the low code bit
        const uint32_t e = ~(p0 ^ ot);                      // low code bit clear AND the base scores (valid = ~ot | p0)
        mA = e & ~p1, mC = e & p1, mT = s0 & ~p1, mG = s0 & p1;
        w0 = s0, w1 = p1;
    } else {
        uint32_t q0;                                        // p0 ^ ~(lw | ot): A<->T, C<->G of upper-case bases flips the low code bit
#ifdef __CUDA_ARCH__
        asm("lop3.b32 %0, %1, %2, %3, 0xE1;" : "=r"(q0) : "r"(p0), "r"(lw), "r"(ot));   // one LOP3, not one shared with irr + one
#else
        q0 = p0 ^ ~(lw | ot);
#endif
        const uint32_t s0 = crp_brev(q0), s1 = crp_brev(p1), valid = crp_brev(~ot | p0);
        mA = ~s1 & ~s0 & valid, mT = ~s1 & s0 & valid, mC = s1 & ~s0 & valid, mG = s1 & s0 & valid;
        w0 = s0, w1 = s1;
    }
    // flag sources: a value <= 0x3FFFFFFF plus 0x3FFFFFFF has bit 30 set iff it is not zero, and bit 31 clear
    const uint32_t irr = (lw | ot) & kWin, uns = ot & ~p0 & kWin;
    const uint32_t y0 = (kMinus ? irr : crp_umulhi(irr, 1u << 30)) + 0x3FFFFFFFu;
    const uint32_t f1 = (kMinus ? uns : crp_umulhi(uns, 1u << 30)) + 0x3FFFFFFFu;
    static_assert(CRP_PACKED_IRREGULAR == (1ull << 30) && CRP_PACKED_TRUNCATED == (1ull << 31) && CRP_PACKED_UNSCORED == (1ull << 62),
                  "flag bits of the packed word");
    uint32_t f0, lo32, hi32;
#ifdef __CUDA_ARCH__
    asm("mad.lo.u32 %0, %1, 0x80000000, %2;" : "=r"(f0) : "r"(trunc), "r"(y0));         // bit 31 of y0 is clear: the add is an OR
    // (w & 0x3FFFFFFF) | (f & 0xC0000000) as ONE bit select each
    asm("lop3.b32 %0, %1, 0x3FFFFFFF, %2, 0xE2;" : "=r"(lo32) : "r"(w0), "r"(f0));
    asm("lop3.b32 %0, %1, 0x3FFFFFFF, %2, 0xE2;" : "=r"(hi32) : "r"(w1), "r"(f1));
#else
    f0 = trunc * 0x80000000u + y0;
    lo32 = (w0 & 0x3FFFFFFFu) | (f0 & 0xC0000000u);
    hi32 = (w1 & 0x3FFFFFFFu) | (f1 & 0xC0000000u);
#endif
    packed = ((unsigned long long)hi32 << 32) | lo32;
    return rs1_canonical_masks(tab, mA, mT, mC, mG);
}

// store v at p iff cond != 0, as a predicated store (no branch, no divergence)
__device__ __forceinline__ void st_list_if(uint16_t *p, uint32_t cond, uint32_t v) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "setp.ne.u32 q, %0, 0;\n"
        "@q st.shared.u16 [%1], %2;\n"
        "}\n" ::"r"(cond),
        "r"(smem_u32(p)), "h"((unsigned short)v)
        : "memory");
}
// hits of one word into the compacted list, ascending; first = slot of the word's first hit.
// The first three hits are straight-line predicated code (a 32-position word holds more than
// three hits of a strand in ~1 % of the words at 36 % GC), the rest loop.
__device__ __forceinline__ void list_hits(uint16_t *__restrict__ first, uint32_t m, uint32_t pos0) {
    const uint32_t l0 = m & (0u - m);
    st_list_if(first, l0, pos0 + 31u - (uint32_t)__clz(l0));
    m ^= l0;
    const uint32_t l1 = m & (0u - m);
    st_list_if(first + 1, l1, pos0 + 31u - (uint32_t)__clz(l1));
    m ^= l1;
    const uint32_t l2 = m & (0u - m);
    st_list_if(first + 2, l2, pos0 + 31u - (uint32_t)__clz(l2));
    m ^= l2;
    first += 3;
    while (m) {
        const uint32_t lb = m & (0u - m);
        *first++ = (uint16_t)(pos0 + 31u - (uint32_t)__clz(lb));
        m ^= lb;
    }
}
// same, for a tile with more than kListCap hits on a strand: only ranks [lo, lo + kListCap)
__device__ __forceinline__ void list_hits_window(uint16_t *__restrict__ list, uint32_t m, uint32_t rank_first,
                                                 uint32_t pos0, uint32_t lo) {
    uint32_t r = rank_first;
    while (m) {
        const uint32_t lb = m & (0u - m);
        if (r - lo < (uint32_t)kListCap) list[r - lo] = (uint16_t)(pos0 + 31u - (uint32_t)__clz(lb));
        m ^= lb;
        ++r;
    }
}

// listed hit i of one strand of a tile: window, score, stores (coalesced across the lanes of a warp)
template <bool kScore, bool kMinus>
__device__ __forceinline__ void emit_one(const ScanArgs &a, const double *__restrict__ tab, const uint4 *__restrict__ rec,
                                         const uint16_t *__restrict__ list, uint32_t i, uint32_t row0, uint32_t t_start,
                                         uint32_t L) {
    uint32_t *const pos = kMinus ? a.pos_minus : a.pos_plus;
    unsigned long long *const packed = kMinus ? a.packed_minus : a.packed_plus;
    double *const xs = kMinus ? a.x_minus : a.x_plus;
    constexpr uint32_t kBias = kMinus ? kWinBiasMinus : kWinBiasPlusHot;
    const uint32_t xt = L - (kMinus ? 28u : 5u) - (t_start - kBias);
    const uint32_t ws = list[i], t = t_start - kBias + ws;
    const uint32_t row = row0 + i;
    CRP_CHECK(a, i < (uint32_t)kListCap, 1);                                 // inside the hit list
    CRP_CHECK(a, ws >= kBias && 2u + (ws >> 5) < (uint32_t)kRecWords, 2);   // window inside the record
    CRP_CHECK(a, row < (uint32_t)a.capacity && t < L, 3);                    // inside the stream, inside the token
    CRP_CHECK(a, i == 0 || list[i - 1] < ws, 4);                             // positions ascend
    __stcs(pos + row, t);
    if (kScore) {
        unsigned long long word;
        const double x = score_hit<kMinus>(tab, rec, ws, xt, word);
#ifdef CRP_CHECKED
        {   // the generic path (extras, rescore) must agree bit for bit
            const Window w = extract_window<kMinus>(rec, ws + (kMinus ? 0u : 2u), t, L);
            CRP_CHECK(a, w.packed == word, 14);
            CRP_CHECK(a, __double_as_longlong(rs1_canonical(tab, w.s0, w.s1, w.valid)) == __double_as_longlong(x), 15);
            // and the lane tables must agree with the column-by-column replay, which reads no table
            CRP_CHECK(a, __double_as_longlong(rs1_dense(w.s0, w.s1, w.valid, CRP_CLASS_CANONICAL, CRP_CLASS_CANONICAL)) ==
                             __double_as_longlong(x), 16);
        }
#endif
        __stcs(packed + row, word);
        __stcs(xs + row, x);
    }
}

// rows of a strand stream fit 32 bits: the scan state packs the two strand counts of a shard into one
// 64-bit word (plus << 32 | minus), and launch_scan clamps the capacity.  -> hits of the list that have a row
__device__ __forceinline__ uint32_t rows_left(const ScanArgs &a, uint32_t count, uint32_t row0) {
    const uint32_t cap = (uint32_t)a.capacity;
    return row0 >= cap ? 0u : min(count, cap - row0);
}

// one thread per listed hit of one strand (dense tiles: a window of kListCap ranks at a time)
template <bool kScore, bool kMinus>
__device__ __forceinline__ void emit_strand(const ScanArgs &a, const double *__restrict__ tab,
                                            const uint4 *__restrict__ rec, const uint16_t *__restrict__ list,
                                            uint32_t count, uint32_t row0, uint32_t t_start, uint32_t L, uint32_t slot) {
    count = rows_left(a, count, row0);
    for (uint32_t i = slot; i < count; i += kThreads) emit_one<kScore, kMinus>(a, tab, rec, list, i, row0, t_start, L);
}

// Ring of staged tiles of a CTA.  full[s] completes when the bulk copies of slot s (the tile
// record and, in the emit phase, the tile's prefix block) have landed.
struct __align__(16) Ring {
    unsigned long long pref[kStages][kPrefWords];   // bulk-copy destination (emit phase)
    unsigned long long full[kCountStages];          // mbarriers (count phase: [0], the header copies; emit phase: the first kStages)
    unsigned long long pre;                         // first emit tile, fetched before the grid barrier
    unsigned long long rbase[kStages];              // global prefix of the count range of the staged tile (emit phase)
    uint32_t tile[kCountStages];                    // staged tile, or kNoTile: the sequence has ended
    uint32_t done[kCountStages];                    // (reset, not read: left from the PAM-record ring)
};
static_assert(kCountStages >= kStages, "the ring control block holds the emit phase's slots");

__device__ __forceinline__ void mbar_inval(unsigned long long *bar) {
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect(unsigned long long *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_copy(void *dst, const void *src, uint32_t bytes, unsigned long long *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// (re)arm the ring at the start of a phase; every thread of the CTA calls it
__device__ __forceinline__ void ring_reset(Ring &ring, bool first, bool wave_start) {
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kCountStages; ++s) {
            if (!first) mbar_inval(&ring.full[s]);
            mbar_init(&ring.full[s], 1);
            ring.done[s] = 0;
            ring.tile[s] = kNoTile;
        }
        if (wave_start) {
            if (!first) mbar_inval(&ring.pre);
            mbar_init(&ring.pre, 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
}

template <bool kScore>
__global__ void __launch_bounds__(kThreads, CRP_CTAS_PER_SM)
k_scan_score(const ScanArgs a) {
    // dynamic shared memory: [stages][hit lists][range prefixes]
    extern __shared__ __align__(128) unsigned char s_dyn[];
    auto stage = [&](int s) { return reinterpret_cast<uint4 *>(s_dyn + (size_t)s * kRecBytes); };
    uint16_t *const s_list = reinterpret_cast<uint16_t *>(s_dyn + kStages * kRecBytes);
    unsigned long long *const s_rangepref =
        reinterpret_cast<unsigned long long *>(s_dyn + kStages * kRecBytes + 2 * (size_t)kListCap * sizeof(uint16_t));
    __shared__ __align__(16) double s_tab[kScore ? RS1_TABLE_DOUBLES : 1];   // static: LDS takes the table offset as an immediate
    __shared__ Ring ring;
    __shared__ unsigned long long s_scan[kWarps];

    cg::grid_group grid = cg::this_grid();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int l = a.guide_len;
    const uint32_t G = gridDim.x, cta = blockIdx.x;

    dbg_stamp(0);
    // the lane tables arrive by bulk copy while the first count phase runs
    __shared__ __align__(8) unsigned long long s_tabbar;
    if (tid == 0) {
        mbar_init(&s_tabbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (kScore) {
            mbar_expect(&s_tabbar, (uint32_t)kRs1TableBytes);
            bulk_copy(s_tab, a.tables, (uint32_t)kRs1TableBytes, &s_tabbar);
        }
    }

    auto record = [&](uint32_t tile) { return a.records + (size_t)tile * kRecWords; };
    const uint32_t nt = a.n_tiles;
    const uint32_t k = (nt + G - 1) / G;                           // tiles per count range

    // ================================================= count phase: tiles [r_lo, r_lo + n_mine)
    const uint32_t r_lo = min(nt, cta * k), n_mine = min(nt, r_lo + k) - r_lo;
    if (cta == 0 && tid == 0) {                                    // read after the grid barrier
        a.tickets[0] = 0;
        a.tickets[1] = 0;
    }
    ring_reset(ring, true, true);
    dbg_stamp(1);
    // The headers of the range arrive by ONE bulk copy per kHdrBatch tiles (48 bytes per tile instead of the
    // 4 KB PAM record the count phase used to stream: k_pack has already counted every chunk under the bounds
    // that do not depend on the guide length).  A tile that reaches into the first l + 5 or the last l - 7
    // positions of its token -- two per token for any sensible l -- is counted here, by one warp, straight from
    // its PAM record in global memory, and its counts replace those of the staged header.  Then thread j owns
    // tile j of the batch: its eight chunk counts, one CTA-wide scan of the tile totals, one prefix block.
    TileHdr *const s_hdr = reinterpret_cast<TileHdr *>(s_dyn);
    static_assert(kHdrBatch == kThreads, "one tile header per thread");
    unsigned long long range_run = 0;
    for (uint32_t h_lo = 0, hb = 0; h_lo < n_mine; h_lo += kHdrBatch, ++hb) {
        const uint32_t h_n = min(n_mine - h_lo, (uint32_t)kHdrBatch);
        if (tid == 0) {
            mbar_expect(&ring.full[0], h_n * (uint32_t)sizeof(TileHdr));
            bulk_copy(s_dyn, a.hdr + (size_t)(r_lo + h_lo), h_n * (uint32_t)sizeof(TileHdr), &ring.full[0]);
        }
        mbar_wait(&ring.full[0], hb & 1u);
        for (uint32_t j = warp; j < h_n; j += kWarps) {
            const uint4 d = s_hdr[j].desc;
            const int32_t t0 = (int32_t)d.x, L = (int32_t)d.y;
            if (t0 < l + 5 || t0 + kTile - 1 > L - l + 7) {            // warp-uniform
                CRP_CHECK(a, r_lo + h_lo + j < nt, 5);
                CRP_CHECK(a, reinterpret_cast<const uint32_t *>(a.pam + (size_t)(r_lo + h_lo + j) * kPamBytes)[0] == d.x, 6);   // the same tile
                warp_count_tile(a.pam + (size_t)(r_lo + h_lo + j) * kPamBytes, l, lane, s_hdr[j].cnt);
            }
        }
        __syncthreads();
        {
            unsigned long long c[kWarps], mine = 0ull;
#pragma unroll
            for (int q = 0; q < kWarps; ++q) {
                c[q] = (uint32_t)tid < h_n ? unpack_counts(s_hdr[tid].cnt[q]) : 0ull;
                mine += c[q];
            }
            unsigned long long incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                if (lane >= o) incl += v;
            }
            if (lane == 31) s_scan[warp] = incl;
            __syncthreads();
            unsigned long long before = range_run, total = 0;
#pragma unroll
            for (int q = 0; q < kWarps; ++q) {
                const unsigned long long x = s_scan[q];
                if (q < warp) before += x;
                total += x;
            }
            if ((uint32_t)tid < h_n) {
                unsigned long long *pf = a.warp_pref + (size_t)(r_lo + h_lo + tid) * kPrefWords;
                unsigned long long run = before + incl - mine;             // prefix at the start of my tile
#pragma unroll
                for (int q = 0; q < kWarps; ++q) {
                    pf[q] = run;
                    run += c[q];
                }
                pf[kWarps] = run;                                          // prefix at the end of the tile
                asm volatile("fence.proxy.async.global;" ::: "memory");   // read back by bulk copies after the grid barrier
            }
            range_run += total;
            __syncthreads();                                       // s_scan and the staged headers are free
        }
    }
    if (tid == 0) a.cta_tot[cta] = range_run;
    // The first emit tile of this CTA is known (static share): its record is fetched across the
    // grid barrier -- the count ring is idle now -- and its prefix block, which another CTA may
    // have written, right after the barrier.
    const uint32_t ns = (uint32_t)((unsigned long long)nt * a.static_eighths / 8 / G);
    const bool pre = ns > 0;
    const uint32_t t_pre = cta;
    if (pre && tid == 0) {
        mbar_expect(&ring.pre, kRecBytes + kPrefWords * 8);
        bulk_copy(stage(0), record(t_pre), kRecBytes, &ring.pre);
    }
    dbg_stamp(2);
    grid.sync();
    dbg_stamp(3);
    if (pre && tid == 0) bulk_copy(ring.pref[0], a.warp_pref + (size_t)t_pre * kPrefWords, kPrefWords * 8, &ring.pre);

    // ================================================= exclusive scan of the range totals
    {
        unsigned long long v[4] = {0, 0, 0, 0}, mine = 0;     // thread owns ranges 4*tid .. 4*tid+3
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t i = 4u * tid + q;
            if (i < G) v[q] = a.cta_tot[i];
            mine += v[q];
        }
        unsigned long long incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long x = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += x;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        unsigned long long before = 0;
#pragma unroll
        for (int q = 0; q < kWarps; ++q) {
            const unsigned long long x = s_scan[q];
            if (q < warp) before += x;
        }
        unsigned long long run = before + incl - mine;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const uint32_t i = 4u * tid + q;
            if (i < G) s_rangepref[i] = run;
            run += v[q];
        }
    }

    // ================================================= emit phase
    // The first ns * G tiles are dealt round-robin (tile known without a round trip); the rest go
    // through the ticket counter, which evens out what the data-dependent emit work left unbalanced.
    const uint32_t dyn_lo = ns * G, n_dyn = nt - dyn_lo;
    unsigned int *const ticket = a.tickets;
    auto produce_emit = [&](uint32_t n, int s) {     // one thread: stage tile number n of this CTA into slot s
        uint32_t t;
        if (n < ns) {
            t = n * G + cta;
        } else {
            const uint32_t q = atomicAdd(ticket, 1u);
            t = q < n_dyn ? dyn_lo + q : kNoTile;
        }
        ring.tile[s] = t;
        if (t != kNoTile) {
            CRP_CHECK(a, t < nt && t / k < G, 11);
            ring.rbase[s] = s_rangepref[t / k];
            mbar_expect(&ring.full[s], kRecBytes + kPrefWords * 8);
            bulk_copy(stage(s), record(t), kRecBytes, &ring.full[s]);
            bulk_copy(ring.pref[s], a.warp_pref + (size_t)t * kPrefWords, kPrefWords * 8, &ring.full[s]);
        } else {
            mbar_arrive(&ring.full[s]);
        }
    };
    ring_reset(ring, false, false);                            // also publishes s_rangepref
    dbg_stamp(4);
    if (kScore) mbar_wait(&s_tabbar, 0);
    // per-segment candidate counts: prefix at the end of the segment's last tile minus prefix at the
    // start of its first one (segments are dealt to threads).  In a sharded scan the counts go to
    // every rank's gather buffer as well, and the last CTA through raises this rank's flags there.
    {
        const bool xchg = a.world > 1;
        for (uint32_t sg = cta * kThreads + tid; sg < a.seg_stride; sg += G * kThreads) {
            unsigned long long plus = 0, minus = 0;
            if (sg < a.n_seg) {                                                         // beyond: padding of the all-gather block
                const uint32_t f = a.seg_first_tile ? a.seg_first_tile[sg] : 0u;        // NULL: one segment = all tiles
                const uint32_t c = a.seg_tile_count ? a.seg_tile_count[sg] : a.n_tiles;
                if (c) {
                    const unsigned long long cnt = s_rangepref[(f + c - 1) / k] + a.warp_pref[(size_t)(f + c - 1) * kPrefWords + kWarps] -
                                                   (s_rangepref[f / k] + a.warp_pref[(size_t)f * kPrefWords]);
                    plus = cnt >> 32;
                    minus = cnt & 0xFFFFFFFFull;
                }
            }
            a.seg_counts[sg] = plus;
            a.seg_counts[a.seg_stride + sg] = minus;
            if (a.seg_counts_host) {
                a.seg_counts_host[sg] = plus;
                a.seg_counts_host[a.seg_stride + sg] = minus;
            }
            if (xchg) {
                CRP_CHECK(a, (size_t)(a.rank + 1) * 2 * a.seg_stride <= (size_t)kMaxPeers * 2 * 32768, 12);
                const size_t at = (size_t)a.rank * 2 * a.seg_stride + sg;
                for (uint32_t p = 0; p < a.world; ++p) {
                    a.peer_gather[p][at] = plus;
                    a.peer_gather[p][at + a.seg_stride] = minus;
                }
            }
        }
        if (xchg && cta * kThreads < a.seg_stride) {           // this CTA wrote counts
            __threadfence_system();
            __syncthreads();
            if (tid == 0) {
                const uint32_t writers = min(G, (a.seg_stride + kThreads - 1) / kThreads);
                __threadfence_system();                        // cumulative: the CTA's stores, observed through the barrier
                if (atomicAdd(a.tickets + 1, 1u) == writers - 1) xchg_publish(a);
            }
        }
    }
    if (tid == 0) {
        if (pre) mbar_arrive(&ring.full[0]);                   // tile 0 came through ring.pre: skip that phase of slot 0
        else produce_emit(0, 0);
    }
    uint16_t *const list_p = s_list, *const list_m = s_list + kListCap;
    for (uint32_t n = 0;; ++n) {
        const int s = n % kStages;
        // next tile of this CTA: its copies land while this tile is emitted (slot s^1 was
        // released by the barrier that ended tile n - 1)
        if (tid == 0) produce_emit(n + 1, s ^ 1);
        const bool first_pre = pre && n == 0;
        if (first_pre) mbar_wait(&ring.pre, 0u);
        else mbar_wait(&ring.full[s], (n / kStages) & 1u);
        if (!first_pre && ring.tile[s] == kNoTile) break;
        const uint4 *rec = stage(s);
        const uint4 d = rec[0];
        const TileDesc td = {d.x, d.y, d.z, d.w};
        const unsigned long long tile_pref = ring.pref[s][0];
        const unsigned long long base = (first_pre ? s_rangepref[t_pre / k] : ring.rbase[s]) + tile_pref;
        const unsigned long long off = ring.pref[s][warp] - tile_pref;          // hits of the tile before my warp chunk
        const unsigned long long tot = ring.pref[s][kWarps] - tile_pref;
        const uint32_t np = (uint32_t)(tot >> 32), nm = (uint32_t)tot;
        const uint32_t base_p = (uint32_t)(base >> 32), base_m = (uint32_t)base;
        const uint32_t wordA = 64 * warp + lane;
        // A warp whose 2,048-position chunk holds no hit on either strand -- a soft-masked block, an N run:
        // half of all chunks on the 50-60 % lower-case configs -- skips its whole front end; the count
        // phase has already said so (prefix block).  Warp-uniform.
        const bool busy = ring.pref[s][warp + 1] != ring.pref[s][warp];
        Hits h = {0u, 0u, 0u, 0u};
        uint32_t epA = 0, emA = 0, epB = 0, emB = 0;
        if (busy) {
            h = tile_hits(rec, td, l, wordA);
            // ---- warp scan of the per-word counts: the A words of the chunk precede its B words
            const uint32_t cA = __popc(h.pA) | (__popc(h.mA) << 16), cB = __popc(h.pB) | (__popc(h.mB) << 16);
            uint32_t iA = cA, iB = cB;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t vA = __shfl_up_sync(0xFFFFFFFFu, iA, o), vB = __shfl_up_sync(0xFFFFFFFFu, iB, o);
                if (lane >= o) {
                    iA += vA;
                    iB += vB;
                }
            }
            const uint32_t totA = __shfl_sync(0xFFFFFFFFu, iA, 31);
            // rank (inside the tile, per strand) of the first hit of my words
            const uint32_t xA = iA - cA, xB = totA + iB - cB;
            const uint32_t op = (uint32_t)(off >> 32), om = (uint32_t)off;
            epA = op + (xA & 0xFFFFu), emA = om + (xA >> 16), epB = op + (xB & 0xFFFFu), emB = om + (xB >> 16);
#ifdef CRP_CHECKED
            {
                const uint32_t mine = totA + __shfl_sync(0xFFFFFFFFu, iB, 31);       // hits of my warp chunk, (plus | minus << 16)
                const unsigned long long nxt = ring.pref[s][warp + 1] - ring.pref[s][warp];
                CRP_CHECK(a, (uint32_t)(nxt >> 32) == (mine & 0xFFFFu) && (uint32_t)nxt == (mine >> 16), 7);   // count phase == emit phase
                if (np <= (uint32_t)kListCap && nm <= (uint32_t)kListCap)
                    CRP_CHECK(a, epA + __popc(h.pA) <= np && epB + __popc(h.pB) <= np && emA + __popc(h.mA) <= nm && emB + __popc(h.mB) <= nm, 10);
            }
#endif
        }
#ifdef CRP_CHECKED
        else {                                                 // the count phase said "no hit here": verify
            const Hits hh = tile_hits(rec, td, l, wordA);
            CRP_CHECK(a, (hh.pA | hh.pB | hh.mA | hh.mB) == 0u, 13);
        }
        CRP_CHECK(a, ring.tile[s] == kNoTile || first_pre || ring.tile[s] < nt, 8);
        CRP_CHECK(a, (unsigned long long)base_p + np <= 0xFFFFFFFFull && (unsigned long long)base_m + nm <= 0xFFFFFFFFull, 9);
#endif
        if (np <= (uint32_t)kListCap && nm <= (uint32_t)kListCap) {
            if (busy) {
                list_hits(list_p + epA, h.pA, 32u * wordA + kWinBiasPlusHot);
                list_hits(list_p + epB, h.pB, 32u * (wordA + 32) + kWinBiasPlusHot);
                list_hits(list_m + emA, h.mA, 32u * wordA + kWinBiasMinus);
                list_hits(list_m + emB, h.mB, 32u * (wordA + 32) + kWinBiasMinus);
            }
            __syncthreads();
            emit_strand<kScore, false>(a, s_tab, rec, list_p, np, base_p, td.t_start, td.L, tid);
            emit_strand<kScore, true>(a, s_tab, rec, list_m, nm, base_m, td.t_start, td.L, tid ^ (kThreads / 2));
        } else {                                               // dense tile: windows of kListCap ranks
            for (uint32_t lo = 0; lo < np || lo < nm; lo += kListCap) {
                const uint32_t cp = np > lo ? min(np - lo, (uint32_t)kListCap) : 0u;
                const uint32_t cm = nm > lo ? min(nm - lo, (uint32_t)kListCap) : 0u;
                if (lo) __syncthreads();
                if (busy) {
                    list_hits_window(list_p, h.pA, epA, 32u * wordA + kWinBiasPlusHot, lo);
                    list_hits_window(list_p, h.pB, epB, 32u * (wordA + 32) + kWinBiasPlusHot, lo);
                    list_hits_window(list_m, h.mA, emA, 32u * wordA + kWinBiasMinus, lo);
                    list_hits_window(list_m, h.mB, emB, 32u * (wordA + 32) + kWinBiasMinus, lo);
                }
                __syncthreads();
                emit_strand<kScore, false>(a, s_tab, rec, list_p, cp, base_p + lo, td.t_start, td.L, tid);
                emit_strand<kScore, true>(a, s_tab, rec, list_m, cm, base_m + lo, td.t_start, td.L, tid);
            }
        }
        __syncthreads();                                       // slot s and the lists are free again
    }
    dbg_stamp(5);
    // sharded scan: the counts of every rank are in this rank's buffer before the kernel -- and the
    // copy to the host behind it -- ends (they were sent a whole emit phase ago)
    if (a.world > 1 && cta == 0) xchg_wait(a);
}

// CRP_SCAN_LOGISTIC: x -> 1 / (1 + np.exp(x)) over a finished stream, numpy's digits (npexp.cuh)
__global__ void k_logistic(double *__restrict__ x, uint64_t n) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) x[i] = np_logistic_f64(x[i]);
}

// rs1_score(sequences) of the reference (CROPSR.py:285-313) on its own input: n rows of 30
// ASCII bytes (only 'A' 'T' 'C' 'G' score, CROPSR.py:300-302), row i summed in the BLAS class
// cls[i] (first-order matmul | second-order matmul << 4), then the reference's logistic.
__global__ void k_rs1_rows(const uint8_t *__restrict__ rows, const uint8_t *__restrict__ cls, uint64_t n,
                           double *__restrict__ score, int logistic) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *r = rows + 30 * i;
    uint32_t s0 = 0, s1 = 0, valid = 0;
    for (int q = 0; q < 30; ++q) {
        const uint32_t c = r[q];
        const uint32_t code = c == 'A' ? 0u : c == 'T' ? 1u : c == 'C' ? 2u : c == 'G' ? 3u : 4u;
        if (code < 4u) {
            valid |= 1u << q;
            s0 |= (code & 1u) << q;
            s1 |= (code >> 1) << q;
        }
    }
    const double x = rs1_dense(s0, s1, valid, (int)(cls[i] & 15u), (int)(cls[i] >> 4));
    score[i] = logistic ? np_logistic_f64(x) : x;
}

struct RescoreItem {
    uint32_t tile;     // record holding token position t
    uint32_t pl;       // position of t inside the tile
    uint32_t strand;   // '+' or '-'
    uint32_t cls;
};

__global__ void k_rescore(const uint4 *__restrict__ records, const RescoreItem *__restrict__ items, uint64_t n,
                          double *__restrict__ x_out) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RescoreItem it = items[i];
    const uint4 *rec = records + (size_t)it.tile * kRecWords;
    const Window w = it.strand == '-' ? extract_window<true>(rec, it.pl + kWinBiasMinus, 0u, 0xFFFFFFFFu)
                                      : extract_window<false>(rec, it.pl + kWinBiasPlus, 0u, 0xFFFFFFFFu);
    x_out[i] = rs1_dense(w.s0, w.s1, w.valid, (int)(it.cls & 15u), (int)(it.cls >> 4));
}
