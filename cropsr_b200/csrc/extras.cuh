// Opt-in per-candidate side outputs (north_star subsystems 3 and 4).  None of this exists in
// the reference at this commit (SURVEY.md "five facts" 2): the reference parses -L / -g and
// never uses them, so these outputs NEVER enter the parity CSV.  Semantics are pinned by
// oracle/extras_oracle.py instead:
//   gc        G+C count of the 20-base protospacer = scored 30-mer[5:25]; the one hint the
//             reference gives is cropsr_functions.py:174-179 (`sequence[5:-5]`, "< 10 -> low")
//   flags     bit0 poly-T (TTTT inside the protospacer: Pol III terminator)
//             bit1 homopolymer run >= 5      bit2 low GC (gc < 10)
//             bit3 the protospacer holds a base that does not score (N, IUPAC, quote, ...)
//   run       longest homopolymer run in the protospacer
//   cut       cut site = end_pos - 3 of the CSV row (CROPSR.py:155-158)
//   flank     [cut - L, cut + L) clipped to the token: the window handed to primer design
//   feature   index of the innermost annotated interval containing the cut site, or -1
#pragma once
#include "scan.cuh"

static constexpr uint32_t kProto = 0x01FFFFE0u;     // bits 5..24 of the 30-mer

struct ExtrasArgs {
    const uint4 *records;
    const uint32_t *pos;          // t of the candidates of one segment, one strand
    uint64_t n;
    uint32_t first_tile, seg_begin, L, flank;
    int minus;
    uint8_t *gc, *flags, *run;
    uint32_t *cut, *flank_lo, *flank_hi;
};

__global__ void k_extras(const ExtrasArgs a) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const uint32_t t = a.pos[i], rel = t - a.seg_begin;
    const uint4 *rec = a.records + (size_t)(a.first_tile + rel / kTile) * kRecWords;
    const Window w = a.minus ? extract_window<true>(rec, rel % kTile + kWinBiasMinus, t, a.L)
                             : extract_window<false>(rec, rel % kTile + kWinBiasPlus, t, a.L);
    const uint32_t v = w.valid & kProto, s0 = w.s0, s1 = w.s1;
    const uint32_t gc = __popc(s1 & v);                                    // C = 2, G = 3: high code bit
    const uint32_t isT = ~s1 & s0 & v;
    const uint32_t t4 = isT & (isT >> 1) & (isT >> 2) & (isT >> 3);        // bit q: T at q..q+3 (all inside the mask)
    // same[q]: bases q and q+1 both score and are equal
    uint32_t same = ~(s0 ^ (s0 >> 1)) & ~(s1 ^ (s1 >> 1)) & v & (v >> 1);
    uint32_t run = v ? 1u : 0u;
    while (same) {
        same &= same >> 1;
        ++run;
    }
    uint32_t f = 0;
    if (t4) f |= 1u;
    if (run >= 5) f |= 2u;
    if (gc < 10) f |= 4u;
    if (v != kProto) f |= 8u;
    const uint32_t cut = a.minus ? t : t - 3u;
    if (a.gc) a.gc[i] = (uint8_t)gc;
    if (a.flags) a.flags[i] = (uint8_t)f;
    if (a.run) a.run[i] = (uint8_t)run;
    if (a.cut) a.cut[i] = cut;
    if (a.flank_lo) a.flank_lo[i] = cut > a.flank ? cut - a.flank : 0u;
    if (a.flank_hi) a.flank_hi[i] = a.flank >= a.L - cut ? a.L : cut + a.flank;     // cut < L: no 32-bit wrap
}

// Intervals sorted by start, inclusive [start, end]; maxend[j] = max(end[0..j]).  One thread
// per candidate: binary search of the last start <= cut, then walk back while an earlier
// interval can still contain the cut site (nested / overlapping features).
__global__ void k_annotate(const uint32_t *__restrict__ pos, uint64_t n, int minus, const uint32_t *__restrict__ start,
                           const uint32_t *__restrict__ end, const uint32_t *__restrict__ maxend, uint32_t n_iv,
                           int32_t *__restrict__ feature) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t cut = minus ? pos[i] : pos[i] - 3u;
    uint32_t lo = 0, hi = n_iv;                       // first interval with start > cut
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(start + mid) <= cut) lo = mid + 1;
        else hi = mid;
    }
    int32_t found = -1;
    for (int64_t j = (int64_t)lo - 1; j >= 0 && __ldg(maxend + j) >= cut; --j)
        if (__ldg(end + j) >= cut) {
            found = (int32_t)j;
            break;
        }
    feature[i] = found;
}


// ------------------------------------------------------------------ runs of bytes that are not A C G T a c g t
// SURVEY.md 8f.2 ("N-run side table"): the gaps of an assembly -- runs of N, IUPAC codes or any other byte --
// as (start, length) in token coordinates, read off the `other` plane of the tile records.  One thread per
// tile word: a set bit whose predecessor is clear starts a run, one whose successor is clear ends it; the
// boundaries go to two unordered lists (runs are disjoint, so the i-th smallest start pairs with the i-th
// smallest end on the host).  Positions outside the segment never count, and runs are clipped to it.
struct RunArgs {
    const uint4 *records;
    uint32_t first_tile, n_tiles;
    uint32_t seg_begin, seg_end;        // token positions the segment owns
    uint32_t *starts, *ends;            // token positions (end = last position of the run)
    unsigned int *n_starts, *n_ends;    // counters (the lists hold at most `capacity` entries each; the counters keep counting)
    uint32_t capacity;
};

__global__ void k_other_runs(const RunArgs a) {
    const uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= (uint64_t)a.n_tiles * kTileWords) return;
    const uint32_t tile = (uint32_t)(it / kTileWords), k = (uint32_t)(it % kTileWords);
    const uint4 *rec = a.records + (size_t)(a.first_tile + tile) * kRecWords;
    const uint4 d = rec[0];
    const uint32_t t_start = d.x, n_owned = d.z;                  // owned positions of this tile: [0, n_owned)
    const uint32_t p0 = 32u * k;                                  // first position of my word inside the tile
    if (p0 >= n_owned) return;
    const uint32_t own = n_owned - p0 >= 32u ? 0xFFFFFFFFu : (1u << (n_owned - p0)) - 1u;
    const uint32_t o = rec[2 + k].w & own;
    if (!o) return;
    // neighbours: the bit before my word and the bit after it (halo words at the tile edges), 0 where the
    // segment starts / ends
    const uint32_t first = t_start + p0;
    const uint32_t prev = first > a.seg_begin ? rec[1 + k].w >> 31 : 0u;
    const uint32_t next = first + 32u < a.seg_end ? rec[3 + k].w & 1u : 0u;
    uint32_t st = o & ~((o << 1) | prev);
    uint32_t en = o & ~((o >> 1) | (next << 31));
    while (st) {
        const uint32_t b = __ffs(st) - 1;
        st &= st - 1;
        const unsigned int slot = atomicAdd(a.n_starts, 1u);
        if (slot < a.capacity) a.starts[slot] = t_start + p0 + b;
    }
    while (en) {
        const uint32_t b = __ffs(en) - 1;
        en &= en - 1;
        const unsigned int slot = atomicAdd(a.n_ends, 1u);
        if (slot < a.capacity) a.ends[slot] = t_start + p0 + b;
    }
}
