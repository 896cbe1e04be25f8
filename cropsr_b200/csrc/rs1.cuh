// Rule-Set-1 scoring on the device (reference: /root/reference/CROPSR.py:285-313).
//
// The reference evaluates  matrix @ weights  with OpenBLAS; which fp64 additions happen in
// which order depends on the row's position inside the np.matmul call (SURVEY.md 8c):
//   canonical  4 sequential accumulators by column mod 4, combined (p0+p2)+(p1+p3)
//   pair       2 accumulators by column mod 2, q0+q1
//   single     ddot (AVX-512) lane order
// rs1_canonical() is the fused-scan fast path (table driven, exact); rs1_dense() replays any
// of the three classes column by column for the few rows that need it (k_rescore).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <vector>

#include "../../include/cropsr_b200.h"
#ifndef RS1_WEIGHTS_INC
#define RS1_WEIGHTS_INC "rs1_weights.inc"      // kernel experiments build against other table sets (tools/variants.sh)
#endif
#include RS1_WEIGHTS_INC

static constexpr size_t kRs1TableBytes = (size_t)RS1_TABLE_DOUBLES * sizeof(double);

// Canonical lane order: one sequential accumulator per column-mod-4 lane, i.e. per base
// class for the first-order term and per SECOND base for the dinucleotide term, columns in
// ascending order; lanes combined (p0+p2)+(p1+p3) = (A+C)+(T+G).  A lane's value is a
// function of which of its entries match, so the leading entries of every lane come from a
// table of exact sequential fp64 sums (built on the host at crp_init, staged in shared
// memory; rs1_weights.inc).  s0/s1: planar code bits of the scored 30-mer (bit q = base q),
// valid: bases that score.
__constant__ double c_rs1_k[] = RS1_K_VALUES;

// ---- the few intrinsics the scoring path uses, with host twins: the device functions below are
// __host__ __device__ so that tests/host_emu.cu can run the SAME source on the CPU (table-driven lanes
// against the dense replay, score_hit against extract_window) -- test infrastructure, nothing in the
// library calls the host side.
#include <math.h>
#include <string.h>
static const double h_rs1_k[] = RS1_K_VALUES;
#ifdef __CUDA_ARCH__
#define RS1_K(i) c_rs1_k[i]
#else
#define RS1_K(i) h_rs1_k[i]
#endif
#define CRP_HD __host__ __device__ __forceinline__
CRP_HD uint32_t crp_umulhi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((unsigned long long)a * b) >> 32);
#endif
}
CRP_HD uint32_t crp_brev(uint32_t a) {
#ifdef __CUDA_ARCH__
    return __brev(a);
#else
    uint32_t r = 0;
    for (int i = 0; i < 32; ++i) r |= ((a >> i) & 1u) << (31 - i);
    return r;
#endif
}
CRP_HD uint32_t crp_funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) {   // shf.r.wrap: the low 5 bits of sh
#ifdef __CUDA_ARCH__
    return __funnelshift_r(lo, hi, sh);
#else
    return (uint32_t)(((((unsigned long long)hi) << 32) | lo) >> (sh & 31u));
#endif
}
CRP_HD int crp_popc(uint32_t a) {
#ifdef __CUDA_ARCH__
    return __popc(a);
#else
    return __builtin_popcount(a);
#endif
}
CRP_HD double crp_dadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    volatile double r = a + b;          // one IEEE add, never contracted
    return r;
#endif
}
CRP_HD double crp_fma(double a, double b, double c) {
#ifdef __CUDA_ARCH__
    return __fma_rn(a, b, c);
#else
    return fma(a, b, c);
#endif
}
CRP_HD double crp_hi2double(uint32_t hi) {                               // hi = high word of the double, low word 0
#ifdef __CUDA_ARCH__
    return __hiloint2double((int)hi, 0);
#else
    const unsigned long long u = (unsigned long long)hi << 32;
    double d;
    memcpy(&d, &u, 8);
    return d;
#endif
}

// lane table entry: `off` doubles into the tables, byte index idx8
#define RS1_LD(T, off, idx8) (*reinterpret_cast<const double *>(reinterpret_cast<const char *>(T) + 8u * (off) + (idx8)))
// top `bits` bits of the hash, scaled to bytes, as multiplies (FMA pipe; shifts would go to the ALU pipe)
#define RS1_TOP(h, bits) (crp_umulhi((h), 1u << (bits)) * 8u)
// the same with the top few hash bits added to the slot (spreads the probable states over the banks), as ONE
// multiply-high by mul = 2^bits + spare: top bits + top few bits + the carry out of the low part, and the
// perfect hashes are searched under exactly this function (gen_rs1_inc.py slot_of).  Written as two multiply-highs and an
// add, ptxas turns one of them into LEA.HI -- an integer-ALU instruction per lane, the pipe the scan is bound by.
#define RS1_SWZ(h, mul) (crp_umulhi((h), (mul)) * 8u)
// bit select: a where the mask is set, b elsewhere (one LOP3)
#define RS1_SEL(mask, a, b) (((a) & (mask)) | ((b) & ~(mask)))
#define RS1_SHL1(m) ((m) << 1)
#define RS1_SHL(m, k) ((m) << (k))
// acc + w iff the match bit is set, as ONE DFMA: bit (a single bit p >= 20 of a class mask)
// read as the high word of a double is a power of two, w_scaled = w / that power.
#define RS1_FMA_BIT(bit, w_scaled, acc) crp_fma(crp_hi2double(bit), (w_scaled), (acc))

// m*: class masks of the scored 30-mer (bit q = base q has that code and scores).  Bits 30 and 31
// may hold anything: every use below is ANDed with a constant below 2^30 (gen_rs1_inc.py asserts it).
CRP_HD double rs1_canonical_masks(const double *__restrict__ T, uint32_t mA, uint32_t mT, uint32_t mC,
                                                      uint32_t mG) {
    RS1_LANE_SUMS(T, mA, mT, mC, mG)
    const double first = crp_dadd(crp_dadd(fA, fC), crp_dadd(fT, fG));
    const double second = crp_dadd(crp_dadd(dA, dC), crp_dadd(dT, dG));
    // (score_first + score_second + intersect + low_gc) * -1, CROPSR.py:312
    // -(t + k) == (-t) + (-k) in IEEE arithmetic: the final negation rides on the operands
    return crp_dadd(-crp_dadd(crp_dadd(first, second), RS1_K(RS1_K_INTERCEPT)), -RS1_K(RS1_K_LOW_GC));
}
CRP_HD double rs1_canonical(const double *__restrict__ T, uint32_t s0, uint32_t s1,
                                                uint32_t valid) {
    return rs1_canonical_masks(T, ~s1 & ~s0 & valid, ~s1 & s0 & valid, s1 & ~s0 & valid, s1 & s0 & valid);
}

// Host side: the table slot (relative to ln.offset) of lane ln when exactly the table entries in `on`
// match (bit i = entries[i]; forced entries carry no match bit and are ignored).  *outside is set if a
// match bit falls outside its group's mask, which the lane's select masks would drop.  The hash that
// RS1_LANE_SUMS computes on the device; build_rs1_tables and tests/rs1_lanes_emu.cu share it.
static uint32_t rs1_table_slot(const Rs1Lane &ln, uint32_t on, bool *outside) {
    uint32_t h = 0;
    for (int g = 0; g < ln.n_groups; ++g) {
        uint32_t x = 0;                           // match bits of this first-base group
        for (int i = 0; i < ln.n_table; ++i) {
            const Rs1Entry &e = ln.entries[i];
            if (!e.forced && (on >> i & 1) && ln.groups[g].first_base == e.first_base) x |= 1u << e.bit;
        }
        if (outside && (x & ~ln.groups[g].mask)) *outside = true;
        h += x * ln.groups[g].magic;
    }
    uint32_t slot = ln.bits ? h >> (32 - ln.bits) : 0u;
    if (ln.swizzle) slot = (uint32_t)(((unsigned long long)h * (unsigned)ln.swizzle) >> 32);   // RS1_SWZ
    return slot;
}

// Host side: exact sequential sums of every valid subset of each lane's table entries
// (forced entries -- the PAM bases -- are part of every sum).
static int build_rs1_tables(std::vector<double> &tab, char *err, size_t errlen) {
    tab.assign(RS1_TABLE_DOUBLES, 0.0);
    std::vector<char> used(RS1_TABLE_DOUBLES, 0);
    for (const Rs1Lane &ln : kRs1Lanes) {
        if (ln.bits < 0) continue;                // no table: the lane is summed entry by entry
        int free_idx[16], n_free = 0;
        for (int i = 0; i < ln.n_table; ++i)
            if (!ln.entries[i].forced) free_idx[n_free++] = i;
        for (uint32_t sub = 0; sub < (1u << n_free); ++sub) {
            bool ok = true;                       // two entries at one position are mutually exclusive
            for (int i = 0; i < n_free && ok; ++i)
                for (int j = i + 1; j < n_free; ++j)
                    if ((sub >> i & 1) && (sub >> j & 1) && ln.entries[free_idx[i]].pos == ln.entries[free_idx[j]].pos)
                        ok = false;
            if (!ok) continue;
            uint32_t on = 0;                      // the subset as entry bits
            for (int i = 0; i < n_free; ++i)
                if (sub >> i & 1) on |= 1u << free_idx[i];
            bool outside = false;
            const uint32_t slot = rs1_table_slot(ln, on, &outside);
            if (outside) {
                snprintf(err, errlen, "rs1 lane %s: entry outside its group mask", ln.name);
                return -1;
            }
            volatile double sum = 0.0;            // one IEEE add per entry, in ascending column order
            for (int i = 0, f = 0; i < ln.n_table; ++i) {
                const bool on_i = ln.entries[i].forced ? true : ((sub >> f++) & 1);
                if (on_i) sum = sum + ln.entries[i].weight;
            }
            const uint32_t idx = ln.offset + slot;
            if (idx >= RS1_TABLE_DOUBLES || used[idx]) {
                snprintf(err, errlen, "rs1 table hash of lane %s is not injective", ln.name);
                return -1;
            }
            used[idx] = 1;
            tab[idx] = sum;
        }
    }
    return 0;
}

__constant__ double c_w1[120] = RS1_DENSE_FIRST;
__constant__ double c_w2[464] = RS1_DENSE_SECOND;
#ifndef __CUDA_ARCH__
static const double h_w1[120] = RS1_DENSE_FIRST;
static const double h_w2[464] = RS1_DENSE_SECOND;
#endif

// Dense emulation of one row of np.matmul(matrix, weights) for a given lane class.
// ind(j) is the 0/1 matrix entry of column j.
template <typename Ind>
__host__ __device__ double blas_row(const double *w, int d, int cls, Ind ind) {
    if (cls == CRP_CLASS_CANONICAL) {
        double p[4] = {0.0, 0.0, 0.0, 0.0};
        for (int j = 0; j < d; ++j)
            if (ind(j)) p[j & 3] = crp_dadd(p[j & 3], w[j]);
        return crp_dadd(crp_dadd(p[0], p[2]), crp_dadd(p[1], p[3]));
    }
    if (cls == CRP_CLASS_PAIR) {
        double q[2] = {0.0, 0.0};
        for (int j = 0; j < d; ++j)
            if (ind(j)) q[j & 1] = crp_dadd(q[j & 1], w[j]);
        return crp_dadd(q[0], q[1]);
    }
    // CRP_CLASS_SINGLE: OpenBLAS ddot (AVX-512): 4 accumulators x 8 lanes over
    // the 32-column blocks, folded to 4 lanes, one 16-column pass, lane-wise
    // ((a0+a1)+a2)+a3, (l0+l2)+(l1+l3), then a sequential tail.
    double acc[4][8];
    for (int a = 0; a < 4; ++a)
        for (int l = 0; l < 8; ++l) acc[a][l] = 0.0;
    const int n32 = d & ~31;
    for (int j = 0; j < n32; ++j)
        if (ind(j)) {
            int a = (j & 31) >> 3, l = j & 7;
            acc[a][l] = crp_dadd(acc[a][l], w[j]);
        }
    double f[4][4];
    for (int a = 0; a < 4; ++a)
        for (int i = 0; i < 4; ++i) f[a][i] = crp_dadd(acc[a][i], acc[a][i + 4]);
    int pos = n32;
    if (d & 16) {
        for (int a = 0; a < 4; ++a)
            for (int i = 0; i < 4; ++i) {
                int j = pos + 4 * a + i;
                if (ind(j)) f[a][i] = crp_dadd(f[a][i], w[j]);
            }
        pos += 16;
    }
    double t[4];
    for (int i = 0; i < 4; ++i)
        t[i] = crp_dadd(crp_dadd(crp_dadd(f[0][i], f[1][i]), f[2][i]), f[3][i]);
    double dot = crp_dadd(crp_dadd(t[0], t[2]), crp_dadd(t[1], t[3]));
    for (int j = pos; j < d; ++j)
        if (ind(j)) dot = crp_dadd(dot, w[j]);
    return dot;
}

__host__ __device__ inline double rs1_dense(uint32_t s0, uint32_t s1, uint32_t valid, int cls1, int cls2) {
#ifdef __CUDA_ARCH__
    const double *w1 = c_w1, *w2 = c_w2;
#else
    const double *w1 = h_w1, *w2 = h_w2;
#endif
    auto code = [&](int p) -> int { return (int)(((s1 >> p) & 1u) << 1 | ((s0 >> p) & 1u)); };
    auto ok = [&](int p) -> bool { return (valid >> p) & 1u; };
    double first = blas_row(w1, 120, cls1, [&](int j) { int p = j >> 2; return ok(p) && code(p) == (j & 3); });
    double second = blas_row(w2, 464, cls2, [&](int j) {
        int p = j >> 4;
        return ok(p) && ok(p + 1) && code(p) == ((j >> 2) & 3) && code(p + 1) == (j & 3);
    });
    return -crp_dadd(crp_dadd(crp_dadd(first, second), RS1_INTERCEPT), RS1_LOW_GC);
}
