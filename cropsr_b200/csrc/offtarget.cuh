// Off-target counts (opt-in; the reference leaves specificity to an external aligner: the nearest thing
// in it is the bowtie2 call of /root/reference/prmrdsgn2.py:139-160, which aligns primers, not guides).
//
// Semantics (oracle/offtarget_oracle.py states the same, byte by byte).  Coordinates are token
// coordinates (decoration bytes of the formatted path included).  A BASE is a byte of ACGTacgt, case
// folded to the code A0 T1 C2 G3; its complement is code ^ 1.  U, Z, N, IUPAC codes, quotes and parens
// are not bases.
//   site '+' at t   tok[t+1], tok[t+2] in {G, g}, t >= 20, tok[t-20 .. t) all bases;  P = tok[t-20 .. t)
//   site '-' at t   tok[t], tok[t+1] in {C, c}, t + 23 <= L, tok[t+3 .. t+23) all bases;
//                   P = reverse complement of tok[t+3 .. t+23)
//   (the PAM's N is any byte, as in the reference's .GG / CC. regexes; a site belongs to the segment
//   that owns t; every token of every genome handle added to an index is searched)
//   key             P[i] in bits 2i, 2i+1 of a uint64 (P[0] = the PAM-distal 5' base): 40 bits
//   mismatches      popc((x | x >> 1) & 0x5555555555), x = a ^ b
//   query           a scan candidate (uppercase PAM, guide length 20): P from the same formulas at its t
//                   and strand.  A candidate whose protospacer is cut off by the token end or holds a
//                   non-base has no counts (all 0xFFFFFFFF); a valid one is always a site itself, and
//                   that site is not counted.  User guides: 20 bases in the protospacer orientation,
//                   nothing subtracted.
//   output          mm_d = number of (other) sites at exactly d mismatches, d = 0 .. k, k <= 3.
//
// Other PAMs (crp_offtarget_new_pam, oracle/offtarget_pam_oracle.py): an index holds the sites of one pattern N S2 S3,
// S2 and S3 sets of codes given by the IUPAC letters A C G T R Y S W K M B D H V (N refused).  With comp(S) =
// {c ^ 1 : c in S}:
//   site '+' at t   tok[t+1] a base in S2, tok[t+2] a base in S3, t >= 20, tok[t-20 .. t) all bases
//   site '-' at t   tok[t] a base in comp(S3), tok[t+1] a base in comp(S2), t + 23 <= L, tok[t+3 .. t+23) all bases
// NGG is the definition above.  Key, mismatches and loci are unchanged.  A candidate's own site is a site of the index
// exactly when G is in S2 and in S3; only then is it subtracted (counts, scores) -- otherwise a candidate row starts at
// 0, as a guide's does.  The listing leaves out a site at the candidate's own locus in either case.
//
// Algorithm: exact pigeonhole filtering.  P is cut into 5 parts of 4 nt; with <= 3 mismatches at least
// two parts match exactly.  For each of the 10 part pairs (i, j) sites and queries are bucketed by the
// 16-bit key of those 8 nt (a counting sort: histogram, scan, scatter) and compared within buckets on the
// 24 bits of the other three parts.  A (query, site) pair is counted only at the pair (i, j) formed by
// its two LOWEST exactly matching parts, so every pair with d <= k is counted exactly once; that test
// runs only on the rare path d <= k.  The hot loop is XOR / SHF / LOP3 / POPC / compare.  One join kernel,
// k_ot_join<Op>, serves counts, listings and scores: the mode's Op (OtCount, OtList, OtScore) decides what a pair
// with d <= k does.
//
// Listing (an index built with loci): every site also has a 64-bit locus (ot_locus) at the slot of its key, and
// k_ot_join<OtList> stores the index of every site with d <= k in the query row's slice of the output (sized by
// the caller from the counts) instead of counting it.
//
// Scores (oracle/offtarget_score_oracle.py states the same): the pairs are exactly those the counts count.  The
// mismatch positions of a pair (0 = P[0], PAM-distal, .. 19) form a set of size d <= 3, ranked colexicographically:
//   rank({})        = 0
//   rank({a})       = 1 + a
//   rank({a<b})     = 21 + a + C(b,2)
//   rank({a<b<c})   = 211 + a + C(b,2) + C(c,3)                       (1,351 sets, ranks 0 .. 1350)
// A caller-given table w[1351] (uint32, < 2^31) gives each set a weight; the score of a query is the uint64 sum of
// w[rank] over its pairs (the candidate's own site, rank 0, subtracted; nothing subtracted for guides).  With the
// table of the MIT specificity score (Hsu et al. 2013, as CRISPOR's calcHitScore computes it: score1 * score2 *
// score3 * 100 in IEEE double, stored as round(hit * 2^24)) the sum over a candidate's NGG sites within k <= 3
// mismatches is H * 2^24, and its specificity 100 / (100 + H) * 100.  CRISPOR sums over 4 mismatches as well, so its
// numbers are not these.  Integer atomics make the sum independent of the order of the pairs.
#pragma once
#include "scan.cuh"

static constexpr uint32_t kOtBuckets = 1u << 16;           // 8 nt of a part pair
static constexpr int kOtPairs = 10;
static constexpr int kOtThreads = 128;                      // k_ot_join: CTA size = queries per work item
static constexpr uint32_t kOtSiteTile = 2048;               // sites of a work item, staged in shared memory (8 KB)
static constexpr uint32_t kOtNoCount = 0xFFFFFFFFu;         // counts of a candidate without a protospacer
static constexpr unsigned long long kOtInvalid = 1ull << 63;   // query key: no protospacer
static constexpr int kOtScanThreads = 1024;                 // k_ot_scan: 64 buckets per thread
static constexpr uint32_t kOtMaxSegments = 1u << 24;        // segments of a genome handle an index with loci takes
static constexpr uint32_t kOtMaxGenomes = 127;              // genome handles of an index with loci
static constexpr unsigned long long kOtNoLocus = ~0ull;     // genome ordinal 127: never a site's locus
static constexpr uint32_t kOtScoreSets = 1351;              // mismatch-position sets of size <= 3 (ot_mask_rank)
static constexpr unsigned long long kOtNoScore = ~0ull;     // score of a candidate without a protospacer

// Locus of a site: t (token coordinates, as in the key's definition) in bits 0-31, the segment index in its genome
// handle in bits 32-55, the ordinal of the add_genome call that added the handle in bits 56-62, strand in bit 63
// (1 = '-').
CRP_HD unsigned long long ot_locus(uint32_t t, uint32_t segment, uint32_t genome, bool minus) {
    return (unsigned long long)t | (unsigned long long)(segment & 0xFFFFFFu) << 32 |
           (unsigned long long)(genome & 0x7Fu) << 56 | (unsigned long long)minus << 63;
}
// the locus of the site at bit b of tile word kw of a record whose descriptor word is desc ({t_start, L, n, segment})
CRP_HD unsigned long long ot_site_locus(uint4 desc, uint32_t kw, uint32_t b, uint32_t genome, bool minus) {
    return ot_locus(desc.x + 32u * kw + b, desc.w, genome, minus);
}

// ------------------------------------------------------------------ keys (host and device: tests/offtarget_emu.cu)
CRP_HD unsigned long long ot_spread20(uint32_t v) {         // bit i -> bit 2i
    unsigned long long x = v & 0xFFFFFu;
    x = (x | x << 16) & 0x0000FFFF0000FFFFull;
    x = (x | x << 8) & 0x00FF00FF00FF00FFull;
    x = (x | x << 4) & 0x0F0F0F0F0F0F0F0Full;
    x = (x | x << 2) & 0x3333333333333333ull;
    x = (x | x << 1) & 0x5555555555555555ull;
    return x;
}

// PAM tests of the 32 positions of record word `cur` (bit b = position p0 + b; `next` is the word after it):
// '+' G/g at p0+b+1 and p0+b+2, '-' C/c at p0+b and p0+b+1.  Bases only: U / Z carry the code of T / G but are
// "other" bytes, and so is every position outside the token.
CRP_HD uint32_t ot_pam_plus(uint4 cur, uint4 next) {
    const uint32_t g = cur.x & cur.y & ~cur.w, gn = next.x & next.y & ~next.w;
    return crp_funnel_r(g, gn, 1) & crp_funnel_r(g, gn, 2);
}
CRP_HD uint32_t ot_pam_minus(uint4 cur, uint4 next) {
    const uint32_t c = ~cur.x & cur.y & ~cur.w, cn = ~next.x & next.y & ~next.w;
    return c & crp_funnel_r(c, cn, 1);
}

// The same for a PAM pattern N S2 S3 (crp_offtarget_new_pam): s2, s3 are the code sets of letters 2 and 3, bit c set
// for code c (A0 T1 C2 G3; {G} = 8 is NGG).  A letter matches a base of its set; never a non-base.
CRP_HD uint32_t ot_pam_letter(uint4 w, uint32_t set) {
    const uint32_t m = ((~w.x & ~w.y) & (0u - (set & 1u))) | ((w.x & ~w.y) & (0u - (set >> 1 & 1u))) |
                       ((~w.x & w.y) & (0u - (set >> 2 & 1u))) | ((w.x & w.y) & (0u - (set >> 3 & 1u)));
    return m & ~w.w;
}
// {c ^ 1 : c in set}: the letters of the '-' strand
CRP_HD uint32_t ot_pam_comp(uint32_t set) { return (set & 5u) << 1 | (set >> 1 & 5u); }
// '+' a letter of s2 at p0+b+1 and of s3 at p0+b+2; '-' a letter of comp(s3) at p0+b and of comp(s2) at p0+b+1
CRP_HD uint32_t ot_pam_plus_sets(uint4 cur, uint4 next, uint32_t s2, uint32_t s3) {
    return crp_funnel_r(ot_pam_letter(cur, s2), ot_pam_letter(next, s2), 1) &
           crp_funnel_r(ot_pam_letter(cur, s3), ot_pam_letter(next, s3), 2);
}
CRP_HD uint32_t ot_pam_minus_sets(uint4 cur, uint4 next, uint32_t s2, uint32_t s3) {
    const uint32_t c2 = ot_pam_comp(s2), c3 = ot_pam_comp(s3);
    return ot_pam_letter(cur, c3) & crp_funnel_r(ot_pam_letter(cur, c2), ot_pam_letter(next, c2), 1);
}

// Key of the site at bit b of word `cur` from the three words around it (positions p0-32 .. p0+63):
// '+' reads tok[t-20 .. t), '-' tok[t+3 .. t+23) reversed and complemented.  false: the protospacer holds a
// byte that is not a base (t < 20 and t + 23 > L fall out here too: outside the token every byte is "other").
template <bool kMinus>
CRP_HD bool ot_key(uint4 prev, uint4 cur, uint4 next, uint32_t b, unsigned long long &key) {
    const uint4 lo = kMinus ? cur : prev, hi = kMinus ? next : cur;
    const uint32_t sh = kMinus ? b + 3u : b + 12u;
    const uint32_t c0 = (uint32_t)((((unsigned long long)hi.x << 32) | lo.x) >> sh) & 0xFFFFFu;
    const uint32_t c1 = (uint32_t)((((unsigned long long)hi.y << 32) | lo.y) >> sh) & 0xFFFFFu;
    const uint32_t ot = (uint32_t)((((unsigned long long)hi.w << 32) | lo.w) >> sh) & 0xFFFFFu;
    if (ot) return false;
    const uint32_t k0 = kMinus ? (crp_brev(c0) >> 12) ^ 0xFFFFFu : c0, k1 = kMinus ? crp_brev(c1) >> 12 : c1;
    key = ot_spread20(k0) | ot_spread20(k1) << 1;
    return true;
}

// part pair p = 0 .. 9 -> (i, j), i < j, in the order (0,1) (0,2) .. (3,4)
CRP_HD void ot_pair(int p, int &i, int &j) {
    int n = 0;
    for (i = 0; i < 5; ++i)
        for (j = i + 1; j < 5; ++j)
            if (n++ == p) return;
}
CRP_HD uint32_t ot_bucket(unsigned long long key, int i, int j) {
    return ((uint32_t)(key >> (8 * i)) & 0xFFu) | ((uint32_t)(key >> (8 * j)) & 0xFFu) << 8;
}
// the other three parts, ascending, in bytes 0 .. 2
CRP_HD uint32_t ot_rest(unsigned long long key, int i, int j) {
    uint32_t r = 0, m = 0;
    for (int p = 0; p < 5; ++p)
        if (p != i && p != j) r |= ((uint32_t)(key >> (8 * p)) & 0xFFu) << (8 * m++);
    return r;
}
// Mismatches of a (query, site) pair of one bucket of part pair (i, j), from the rest keys; -1 when the
// pair is not counted here: more than k mismatches, or a part below j other than i also matches exactly --
// then the pair belongs to a lower part pair.  The parts below j other than i are rest bytes 0 .. j-2.
CRP_HD int ot_rest_mismatches(uint32_t q, uint32_t s, uint32_t k, uint32_t jm1) {
    const uint32_t x = q ^ s, y = (x | x >> 1) & 0x555555u;
    const uint32_t d = (uint32_t)crp_popc(y);
    if (d > k) return -1;
    for (uint32_t m = 0; m < jm1; ++m)
        if (!((y >> (8 * m)) & 0xFFu)) return -1;
    return (int)d;
}
// Colex rank (see the head of this file) of the protospacer positions of the mismatches of a pair of part pair
// (i, j), from y = (x | x >> 1) & 0x555555 of the rest keys' XOR x: rest nucleotide m (bit 2m) is position 4p + m % 4
// of the part p that rest byte m / 4 holds (the parts other than i and j, ascending).  At most 3 bits of y are set.
CRP_HD uint32_t ot_mask_rank(uint32_t y, int i, int j) {
    uint32_t rank = 0, n = 0;
    for (; y; y &= y - 1) {
        const uint32_t m = (uint32_t)crp_popc((y & (0u - y)) - 1u) >> 1;   // the lowest set bit, 2m
        uint32_t p = m >> 2;
        p += p >= (uint32_t)i;
        p += p >= (uint32_t)j;
        const uint32_t x = 4u * p + (m & 3u);
        ++n;
        rank += n == 1 ? x : n == 2 ? x * (x - 1u) / 2u : x * (x - 1u) * (x - 2u) / 6u;
    }
    return rank + (n == 0 ? 0u : n == 1 ? 1u : n == 2 ? 21u : 211u);
}

// ------------------------------------------------------------------ kernels
__device__ __forceinline__ uint32_t ot_lanemask_lt() {
    uint32_t m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

// Sites of a genome handle: one thread per tile word, reading the tile records as k_other_runs does (the halo
// words cover the 20 positions to the left and the 23 to the right of every owned position).  keys == NULL:
// count only.  Otherwise keys[base + slot] for an unordered slot per site, and with kLoci its locus at
// loci[base + slot] (ot_site_locus: t and segment from the tile's descriptor word); the instantiation without loci reads
// neither field.  kSets: the sites of the PAM pattern N s2 s3 (ot_pam_plus_sets); without it NGG (ot_pam_plus), and
// s2 / s3 are not read.
struct OtSiteArgs {
    const uint4 *records;
    uint32_t n_tiles;
    unsigned long long *keys;
    unsigned long long base;
    unsigned long long *n;              // counter
    unsigned long long *loci;           // kLoci only
    uint32_t genome;                    // kLoci only: ordinal of the genome handle in the index
    uint32_t s2, s3;                    // kSets only: code sets of PAM letters 2 and 3
};

template <bool kLoci, bool kSets>
__global__ void __launch_bounds__(256) k_ot_sites(const OtSiteArgs a) {
    const uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31;
    uint32_t plus = 0, minus = 0;
    uint4 desc = make_uint4(0, 0, 0, 0);   // kLoci: the tile's descriptor word
    uint32_t kw = 0;                    // kLoci: the tile word
    uint4 prev = make_uint4(0, 0, 0, 0), cur = prev, next = prev;
    if (it < (uint64_t)a.n_tiles * kTileWords) {
        const uint32_t tile = (uint32_t)(it / kTileWords), k = (uint32_t)(it % kTileWords);
        const uint4 *rec = a.records + (size_t)tile * kRecWords;
        const uint32_t n_owned = rec[0].z, p0 = 32u * k;
        if (p0 < n_owned) {
            const uint32_t own = n_owned - p0 >= 32u ? 0xFFFFFFFFu : (1u << (n_owned - p0)) - 1u;
            prev = rec[1 + k], cur = rec[2 + k], next = rec[3 + k];
            if constexpr (kSets) {
                plus = ot_pam_plus_sets(cur, next, a.s2, a.s3) & own;
                minus = ot_pam_minus_sets(cur, next, a.s2, a.s3) & own;
            } else {
                plus = ot_pam_plus(cur, next) & own;
                minus = ot_pam_minus(cur, next) & own;
            }
            if constexpr (kLoci) {
                desc = rec[0];
                kw = k;
            }
        }
    }
    unsigned long long key;
    uint32_t mine = 0;                  // valid sites of this word
    for (uint32_t m = plus; m; m &= m - 1) mine += ot_key<false>(prev, cur, next, __ffs(m) - 1, key);
    for (uint32_t m = minus; m; m &= m - 1) mine += ot_key<true>(prev, cur, next, __ffs(m) - 1, key);
    uint32_t incl = mine;               // warp-inclusive prefix, one atomic per warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= (uint32_t)d) incl += v;
    }
    unsigned long long slot = 0;
    if (lane == 31 && incl) slot = atomicAdd(a.n, (unsigned long long)incl);
    slot = __shfl_sync(0xFFFFFFFFu, slot, 31) + incl - mine;
    if (!a.keys || !mine) return;
    unsigned long long *out = a.keys + a.base + slot, *lout = kLoci ? a.loci + a.base + slot : nullptr;
    for (uint32_t m = plus; m; m &= m - 1)
        if (ot_key<false>(prev, cur, next, __ffs(m) - 1, key)) {
            *out++ = key;
            if constexpr (kLoci) *lout++ = ot_site_locus(desc, kw, __ffs(m) - 1, a.genome, false);
        }
    for (uint32_t m = minus; m; m &= m - 1)
        if (ot_key<true>(prev, cur, next, __ffs(m) - 1, key)) {
            *out++ = key;
            if constexpr (kLoci) *lout++ = ot_site_locus(desc, kw, __ffs(m) - 1, a.genome, true);
        }
}

// Query keys of one strand stream of a scan (rows in segment order): the protospacer is read from the tile
// records at the candidate's (segment, t) -- not from the packed 30-mer, whose '+' windows hold the bases of
// lower-case positions uncomplemented.  With counts, the counts row is primed: valid [own, 0, ..], invalid all
// kOtNoCount.  own is 0xFFFFFFFF (-1) when the query's own site is a site of the index (it brings mm0 to 0), else 0.
struct OtQueryArgs {
    const uint4 *records;
    const uint32_t *pos;
    uint64_t n;
    const uint32_t *seg_row;            // [n_seg + 1] first row of every segment in the stream
    const uint32_t *seg_tile, *seg_begin;   // [n_seg] first tile record / first owned position
    uint32_t n_seg, k1;                 // k1 = max_mm + 1 counts per query
    int minus;
    unsigned long long *keys;
    uint32_t *counts;                   // [n][k1], or NULL
    uint32_t own;                       // mm0 of a valid row before the join
};

__global__ void k_ot_queries(const OtQueryArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    uint32_t lo = 0, hi = a.n_seg;      // last segment whose first row is <= i
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a.seg_row + mid) <= i) lo = mid;
        else hi = mid;
    }
    const uint32_t t = a.pos[i], rel = t - __ldg(a.seg_begin + lo), p = rel % kTile, k = p >> 5, b = p & 31u;
    const uint4 *rec = a.records + (size_t)(__ldg(a.seg_tile + lo) + rel / kTile) * kRecWords;
    unsigned long long key = 0;
    const bool ok = a.minus ? ot_key<true>(rec[1 + k], rec[2 + k], rec[3 + k], b, key)
                            : ot_key<false>(rec[1 + k], rec[2 + k], rec[3 + k], b, key);
    a.keys[i] = ok ? key : kOtInvalid;
    if (!a.counts) return;
    uint32_t *c = a.counts + i * a.k1;
    c[0] = ok ? a.own : kOtNoCount;
    for (uint32_t d = 1; d < a.k1; ++d) c[d] = ok ? 0u : kOtNoCount;
}

// Selected rows of a strand stream for listing (rows ascending): the query key k_ot_queries wrote for the row and
// the locus of the row's own site, which the listing leaves out.  A selected row without a protospacer sets
// `invalid`.
struct OtGatherArgs {
    const unsigned long long *keys;     // [stream rows], k_ot_queries
    const uint32_t *pos, *rows;
    const uint32_t *seg_row;            // [n_seg + 1] first row of every segment in the stream
    uint64_t n;                         // selected rows
    uint32_t n_seg, genome;
    int minus;
    unsigned long long *sel_keys, *own; // [n]
    unsigned int *invalid;
};

__global__ void k_ot_gather(const OtGatherArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const uint32_t r = a.rows[i];
    uint32_t lo = 0, hi = a.n_seg;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(a.seg_row + mid) <= r) lo = mid;
        else hi = mid;
    }
    const unsigned long long key = a.keys[r];
    if (key & kOtInvalid) atomicOr(a.invalid, 1u);
    a.sel_keys[i] = key;
    a.own[i] = ot_locus(a.pos[r], lo, a.genome, a.minus != 0);
}

// ---- geometry of a work item of k_ot_join (host and device: tests/offtarget_join_emu.cu checks it exhaustively)
// Sites allocated past the last one of a part pair's site array: the bulk copy of a tile rounds its source down to 16
// bytes and its length up to 16, so it reads up to 12 bytes (3 uint32 sites, 1.5 uint2 sites) past the last site.
static constexpr uint32_t kOtSitePad = 8;

CRP_HD uint32_t crp_ldg_u32(const uint32_t *p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}
// work items of a bucket of ns sites and nq queries (k_ot_scan): query tiles x site tiles, 0 unless both are present.
// 64-bit: one bucket of 2^32 - 1 queries and sites has 2^46 items, which k_ot_scan's check of the part pair's total
// (< 2^32) then catches; in 32 bits the product, and the tile counts near 2^32, would wrap unseen.
CRP_HD unsigned long long ot_bucket_items(uint32_t ns, uint32_t nq) {
    return ns && nq ? ((unsigned long long)nq + kOtThreads - 1) / kOtThreads *
                          (((unsigned long long)ns + kOtSiteTile - 1) / kOtSiteTile)
                    : 0ull;
}
// the bucket of work item `item` (< item_off[kOtBuckets]): the last b with item_off[b] <= item.  Empty buckets repeat
// the offset of the bucket after them, so the last such b is the one with items.
CRP_HD uint32_t ot_item_bucket(const uint32_t *item_off, uint32_t item) {
    uint32_t lo = 0, hi = kOtBuckets;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (crp_ldg_u32(item_off + mid) <= item) lo = mid;
        else hi = mid;
    }
    return lo;
}
// the tiles of work item `item` of bucket b: queries [q0, q0 + nq_t) and sites [s0, s0 + ns_t) of the bucket-ordered
// arrays; item - item_off[b] = qt * n_st + st over the bucket's n_st site tiles
struct OtItem {
    uint32_t q0, nq_t, s0, ns_t;
};
CRP_HD OtItem ot_item(const uint32_t *soff, const uint32_t *qoff, const uint32_t *item_off, uint32_t b, uint32_t item) {
    const uint32_t sb = crp_ldg_u32(soff + b), ns = crp_ldg_u32(soff + b + 1) - sb;
    const uint32_t qb = crp_ldg_u32(qoff + b), nq = crp_ldg_u32(qoff + b + 1) - qb;
    const uint32_t n_st = (ns + kOtSiteTile - 1) / kOtSiteTile, local = item - crp_ldg_u32(item_off + b);
    const uint32_t qt = local / n_st, st = local % n_st;
    OtItem it;
    it.s0 = sb + st * kOtSiteTile;
    it.ns_t = min(kOtSiteTile, ns - st * kOtSiteTile);
    it.q0 = qb + qt * kOtThreads;
    it.nq_t = min((uint32_t)kOtThreads, nq - qt * kOtThreads);
    return it;
}
// The bulk copy of the tile [s0, s0 + ns_t) of site elements of kSize bytes: from element ot_copy_first (16-byte
// aligned), ot_copy_bytes (a multiple of 16, at most (kOtSiteTile + 16 / kSize) elements) into the shared tile, where
// site s0 is element s0 - a0.
template <uint32_t kSize>
CRP_HD uint32_t ot_copy_first(uint32_t s0) { return s0 & ~(16u / kSize - 1u); }
template <uint32_t kSize>
CRP_HD uint32_t ot_copy_bytes(uint32_t s0, uint32_t ns_t, uint32_t a0) { return ((s0 + ns_t - a0) * kSize + 15u) & ~15u; }
CRP_HD uint32_t ot_copy_offset(uint32_t s0, uint32_t a0) { return s0 - a0; }
// The split of a tile's queries over the CTA: g threads per query; thread tid < nq_t * g holds query tid % nq_t and
// visits the sites tid / nq_t, + g, ...; the others are idle.
CRP_HD uint32_t ot_threads_per_query(uint32_t nq_t) { return kOtThreads / nq_t; }
CRP_HD bool ot_thread_active(uint32_t tid, uint32_t nq_t, uint32_t g) { return tid < nq_t * g; }

// ---- counting sort by the bucket of part pair (i, j): histogram, scan, scatter.  Warps aggregate their
// atomics per bucket (__match_any_sync): a repeat family puts whole warps into one bucket.
__global__ void k_ot_hist(const unsigned long long *__restrict__ keys, uint64_t n, int pi, int pj, uint32_t *hist) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {
        const uint64_t i = base + lane;
        const unsigned long long key = i < n ? keys[i] : kOtInvalid;
        const bool ok = !(key & kOtInvalid);
        const uint32_t b = ok ? ot_bucket(key, pi, pj) : 0xFFFFFFFFu;
        const uint32_t grp = __match_any_sync(0xFFFFFFFFu, b);
        if (ok && (grp & ot_lanemask_lt()) == 0) atomicAdd(hist + b, (uint32_t)__popc(grp));
    }
}

// one CTA per array: 0 sites, 1 queries (exclusive offsets and scatter cursors), 2 work items per bucket
// (query tiles x site tiles) and the comparisons of this part pair
struct OtScanArgs {
    const uint32_t *hist[2];
    uint32_t *off[2], *cursor[2];
    uint32_t *item_off;
    unsigned long long *comparisons;
    unsigned int *overflow;             // set if a part pair has 2^32 work items or more
};

__global__ void __launch_bounds__(kOtScanThreads) k_ot_scan(const OtScanArgs a) {
    constexpr uint32_t per = kOtBuckets / kOtScanThreads;
    __shared__ unsigned long long s_warp[kOtScanThreads / 32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, which = blockIdx.x;
    auto value = [&](uint32_t b) -> unsigned long long {
        if (which < 2) return a.hist[which][b];
        return ot_bucket_items(a.hist[0][b], a.hist[1][b]);
    };
    unsigned long long sum = 0, cmp = 0;
    for (uint32_t e = 0; e < per; ++e) {
        const uint32_t b = tid * per + e;
        sum += value(b);
        if (which == 2) cmp += (unsigned long long)a.hist[0][b] * a.hist[1][b];
    }
    unsigned long long incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned long long o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= (uint32_t)d) incl += o;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long w = s_warp[lane], wi = w;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned long long o = __shfl_up_sync(0xFFFFFFFFu, wi, d);
            if (lane >= (uint32_t)d) wi += o;
        }
        s_warp[lane] = wi - w;
    }
    __syncthreads();
    unsigned long long run = s_warp[warp] + incl - sum;   // totals stay below 2^32: < 2^32 sites / queries
    uint32_t *off = which < 2 ? a.off[which] : a.item_off;
    for (uint32_t e = 0; e < per; ++e) {
        const uint32_t b = tid * per + e;
        off[b] = (uint32_t)run;
        if (which < 2) a.cursor[which][b] = (uint32_t)run;
        run += value(b);
    }
    if (tid == kOtScanThreads - 1) {
        off[kOtBuckets] = (uint32_t)run;
        if (run >> 32) atomicOr(a.overflow, 1u);
    }
    if (which == 2) {
        for (int d = 16; d; d >>= 1) cmp += __shfl_down_sync(0xFFFFFFFFu, cmp, d);
        if (lane == 0 && cmp) atomicAdd(a.comparisons, cmp);
    }
}

// sites -> rest key at its bucket slot; queries (idx != NULL) -> {rest key, row}
__global__ void k_ot_scatter(const unsigned long long *__restrict__ keys, uint64_t n, int pi, int pj, uint32_t *cursor,
                             uint32_t *out_sites, uint2 *out_queries) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < n; base += stride) {
        const uint64_t i = base + lane;
        const unsigned long long key = i < n ? keys[i] : kOtInvalid;
        const bool ok = !(key & kOtInvalid);
        const uint32_t b = ok ? ot_bucket(key, pi, pj) : 0xFFFFFFFFu;
        const uint32_t grp = __match_any_sync(0xFFFFFFFFu, b);
        const uint32_t leader = __ffs(grp) - 1;
        uint32_t slot = 0;
        if (ok && lane == leader) slot = atomicAdd(cursor + b, (uint32_t)__popc(grp));
        slot = __shfl_sync(0xFFFFFFFFu, slot, leader) + __popc(grp & ot_lanemask_lt());
        if (!ok) continue;
        const uint32_t r = ot_rest(key, pi, pj);
        if (out_queries) out_queries[slot] = make_uint2(r, (uint32_t)i);
        else out_sites[slot] = r;
    }
}

// The join of one part pair.  Work item = (query tile of <= 128 queries) x (site tile of <= 2048 sites) of one
// bucket, so that a bucket of a repeat family (10^5 sites and more) spreads over many CTAs and an average bucket
// (~130 sites, configs[1]) is one item.  A persistent grid walks the items of the part pair; the site tile arrives by
// one bulk copy, every thread holds one query and a slice of the tile (a tile with few queries gives each query
// several threads).  What a pair with d <= k does is the mode's Op (OtCount, OtList, OtScore below):
//   Op::Site                      the element of the site array: the rest key, or {rest key, site index}
//   Op::Shared sh                 per CTA in shared memory, filled by op.setup(sh, tid) before the first item
//   Op::Acc acc{}                 per thread and item
//   op.visit(acc, sh, a, q, s, d) on the rare path d <= k
//   op.flush(acc, a, q)           after the thread's slice of the tile
struct OtJoin {
    const void *sites;                  // Op::Site in bucket order
    const uint2 *queries;               // {rest key, row} in bucket order
    const uint32_t *soff, *qoff, *item_off;   // [kOtBuckets + 1]
    uint32_t k, jm1;
    int pi, pj;                         // the part pair
};

CRP_HD uint32_t ot_site_rest(uint32_t s) { return s; }
CRP_HD uint32_t ot_site_rest(uint2 s) { return s.x; }

template <class Op>
__global__ void __launch_bounds__(kOtThreads) k_ot_join(const OtJoin a, const Op op) {
    using Site = typename Op::Site;
    __shared__ __align__(16) Site s_sites[kOtSiteTile + 16 / sizeof(Site)];   // the copy starts up to 16 bytes early
    __shared__ typename Op::Shared sh;
    __shared__ __align__(8) unsigned long long bar;
    const uint32_t tid = threadIdx.x;
    const uint32_t total = a.item_off[kOtBuckets];
    op.setup(sh, tid);
    if (tid == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t phase = 0;
    for (uint32_t item = blockIdx.x; item < total; item += gridDim.x) {
        const OtItem it = ot_item(a.soff, a.qoff, a.item_off, ot_item_bucket(a.item_off, item), item);
        const uint32_t s0 = it.s0, ns_t = it.ns_t, nq_t = it.nq_t;
        const uint32_t a0 = ot_copy_first<sizeof(Site)>(s0);
        if (tid == 0) {
            const uint32_t bytes = ot_copy_bytes<sizeof(Site)>(s0, ns_t, a0);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // earlier generic reads of the tile come first
            mbar_expect(&bar, bytes);
            bulk_copy(s_sites, static_cast<const Site *>(a.sites) + a0, bytes, &bar);
        }
        const uint32_t g = ot_threads_per_query(nq_t);
        const bool active = ot_thread_active(tid, nq_t, g);
        const uint2 q = active ? a.queries[it.q0 + tid % nq_t] : make_uint2(0, 0);
        mbar_wait(&bar, phase);
        phase ^= 1u;
        if (active) {
            const Site *S = s_sites + ot_copy_offset(s0, a0);
            typename Op::Acc acc{};
            for (uint32_t s = tid / nq_t; s < ns_t; s += g) {
                const Site site = S[s];
                const int d = ot_rest_mismatches(q.x, ot_site_rest(site), a.k, a.jm1);
                if (d < 0) continue;
                op.visit(acc, sh, a, q, site, d);
            }
            op.flush(acc, a, q);
        }
        __syncthreads();                                                     // the tile is read before the next copy
    }
}

// Counts: per thread and item four register counts, flushed with one atomic per non-zero count.
struct OtCount {
    using Site = uint32_t;
    struct Shared {};
    struct Acc {
        uint32_t c0, c1, c2, c3;
    };
    uint32_t *counts;                   // [rows][k + 1], primed by the caller
    __device__ void setup(Shared &, uint32_t) const {}
    __device__ void visit(Acc &acc, const Shared &, const OtJoin &, uint2, Site, int d) const {
        acc.c0 += d == 0;
        acc.c1 += d == 1;
        acc.c2 += d == 2;
        acc.c3 += d == 3;
    }
    __device__ void flush(const Acc &acc, const OtJoin &a, uint2 q) const {
        uint32_t *c = counts + (size_t)q.y * (a.k + 1);
        if (acc.c0) atomicAdd(c, acc.c0);
        if (acc.c1) atomicAdd(c + 1, acc.c1);
        if (acc.c2) atomicAdd(c + 2, acc.c2);
        if (acc.c3) atomicAdd(c + 3, acc.c3);
    }
};

// Listing: the sites carry their index (a 16 KB tile).  A pair takes a slot of the query row's slice with one atomic
// on the row's cursor and stores the site index; a slot beyond the slice is never written -- the overflow flag is
// raised instead.  The query's own site (d = 0, same locus) is left out.
struct OtList {
    using Site = uint2;                 // {rest key, site index}
    struct Shared {};
    struct Acc {};
    const unsigned long long *loci;     // [sites]
    const unsigned long long *own;      // [rows] locus of the row's own site, kOtNoLocus for none; NULL: no row has one
    const unsigned long long *first;    // [rows + 1] slice of every row in out
    uint32_t *cursor;                   // [rows] zeroed: sites found per row
    uint32_t *out;                      // [first[rows]] site indices
    unsigned int *overflow;
    __device__ void setup(Shared &, uint32_t) const {}
    __device__ void visit(Acc &, const Shared &, const OtJoin &, uint2 q, Site site, int d) const {
        if (d == 0 && own && __ldg(loci + site.y) == __ldg(own + q.y)) return;
        const unsigned long long b = __ldg(first + q.y), len = __ldg(first + q.y + 1) - b;
        const uint32_t slot = atomicAdd(cursor + q.y, 1u);
        if (slot < len) out[b + slot] = site.y;
        else atomicOr(overflow, 1u);
    }
    __device__ void flush(const Acc &, const OtJoin &, uint2) const {}
};

// Scores: a copy of the weight table (5.4 KB) in shared memory.  A pair adds w[rank] of its mismatch-position set to
// a uint64 in a register; a non-zero sum is flushed with one 64-bit atomic per thread and item.  Rows are primed by
// the caller: a candidate with -w[0] (its own site adds w[0]), a candidate without a protospacer with kOtNoScore (it
// joins no bucket), a guide with 0.
struct OtScore {
    using Site = uint32_t;
    struct Shared {
        uint32_t w[kOtScoreSets];
    };
    struct Acc {
        unsigned long long sum;
    };
    const uint32_t *weights;            // [kOtScoreSets], by ot_mask_rank
    unsigned long long *sums;           // [rows]
    __device__ void setup(Shared &sh, uint32_t tid) const {
        for (uint32_t r = tid; r < kOtScoreSets; r += kOtThreads) sh.w[r] = __ldg(weights + r);
    }
    __device__ void visit(Acc &acc, const Shared &sh, const OtJoin &a, uint2 q, Site site, int) const {
        const uint32_t x = q.x ^ site;
        acc.sum += sh.w[ot_mask_rank((x | x >> 1) & 0x555555u, a.pi, a.pj)];
    }
    __device__ void flush(const Acc &acc, const OtJoin &, uint2 q) const {
        if (acc.sum) atomicAdd(sums + q.y, acc.sum);
    }
};

// The score rows of a candidate stream from the query keys k_ot_queries wrote: `own` (= -w[0]) or kOtNoScore.
__global__ void k_ot_score_prime(const unsigned long long *__restrict__ keys, uint64_t n, unsigned long long own,
                                 unsigned long long *sums) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) sums[i] = keys[i] & kOtInvalid ? kOtNoScore : own;
}
