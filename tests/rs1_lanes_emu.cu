// TEST INFRASTRUCTURE: every Rule Set 1 lane state through the table path, on the CPU, from the SAME source as
// the scan kernel (rs1.cuh / scan.cuh are __host__ __device__ with host twins of their intrinsics).
//
// Input: a file of 30-mers, one per line, over A T C G and N (a byte that does not score), written by
// tests/test_rs1_lanes.py so that together they realise every set of matching entries a scanned 30-mer can
// give each of the eight lanes.  For every row this program asserts, bit for bit:
//   A  rs1_canonical (tables from build_rs1_tables) == rs1_dense (column-by-column replay of OpenBLAS'
//      canonical lane order, which reads no table);
//   S  every table load of RS1_LANE_SUMS reads the slot rs1_table_slot gives the row's matching table entries;
//   B  score_hit == rs1_dense with the row planted on either strand of a staged record, at tile positions
//      0, 1, 30, 31, 32 and 16383 (windows in the halo words and across word edges), with the bytes written
//      plain, lower case, or as U / Z where those score as the intended base.
// It then asserts coverage: the table slots the rows visit are exactly the slots build_rs1_tables fills for
// the table states some 30-mer can reach (a per-position walk over A T C G N with bases 2 and 3 'C').
// It prints, per lane, the number of distinct sets of matching entries (over all the lane's entries) the rows
// realise; the Python test compares them with its own enumeration from cropsr_b200/rs1.py.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <set>
#include <string>
#include <vector>

#include "../cropsr_b200/csrc/scan.cuh"

static unsigned long long rng_state = 0x2545F4914F6CDD1Dull;
static inline unsigned long long rnd() {   // xorshift64*
    rng_state ^= rng_state >> 12;
    rng_state ^= rng_state << 25;
    rng_state ^= rng_state >> 27;
    return rng_state * 0x2545F4914F6CDD1Dull;
}

static unsigned long long bits_of(double d) {
    unsigned long long u;
    memcpy(&u, &d, 8);
    return u;
}

static int code_of(char c) { return c == 'A' ? 0 : c == 'T' ? 1 : c == 'C' ? 2 : c == 'G' ? 3 : 4; }

// ---- RS1_LANE_SUMS with every table load recorded (the library's rs1_canonical_masks is already compiled
// with the plain load; the macro body expands again here)
struct Load { uint32_t off, idx8; };
static Load g_loads[8];
static int g_n_loads;
static double probe_ld(const double *T, uint32_t off, uint32_t idx8) {
    if (g_n_loads < 8) g_loads[g_n_loads] = {off, idx8};
    ++g_n_loads;
    return RS1_LD(T, off, idx8);
}
#define RS1_PROBE_LD(T, off, idx8) probe_ld((T), (off), (idx8))
#undef RS1_LD
#define RS1_LD RS1_PROBE_LD
static void probe_lanes(const double *T, uint32_t mA, uint32_t mT, uint32_t mC, uint32_t mG) {
    g_n_loads = 0;
    RS1_LANE_SUMS(T, mA, mT, mC, mG)
    (void)fA, (void)fT, (void)fC, (void)fG, (void)dA, (void)dT, (void)dC, (void)dG;
}
#undef RS1_LD

// entry i of lane ln matches the row (codes c[30], 4 = does not score)
static bool entry_matches(const Rs1Lane &ln, const Rs1Entry &e, const int *c) {
    if (e.first_base < 0) return c[e.pos] == ln.lane_base;
    return c[e.pos] == e.first_base && c[e.pos + 1] == ln.lane_base;
}

// Can some 30-mer over A T C G N, bases 2 and 3 'C', make exactly the table entries in `on` match?
// Every entry ties at most two adjacent positions, so a walk over the positions with the base of the
// current one as state decides it.
static bool table_state_reachable(const Rs1Lane &ln, uint32_t on) {
    auto unary_ok = [&](int p, int b) {
        for (int i = 0; i < ln.n_table; ++i) {
            const Rs1Entry &e = ln.entries[i];
            if (e.forced || e.first_base >= 0 || e.pos != p) continue;
            if ((b == ln.lane_base) != (bool)(on >> i & 1)) return false;
        }
        return p < 2 || p > 3 || b == 2;
    };
    auto pair_ok = [&](int p, int a, int b) {       // bases a at p, b at p + 1
        for (int i = 0; i < ln.n_table; ++i) {
            const Rs1Entry &e = ln.entries[i];
            if (e.forced || e.first_base < 0 || e.pos != p) continue;
            if ((a == e.first_base && b == ln.lane_base) != (bool)(on >> i & 1)) return false;
        }
        return true;
    };
    bool can[5];
    for (int b = 0; b < 5; ++b) can[b] = unary_ok(0, b);
    for (int p = 1; p < 30; ++p) {
        bool nx[5];
        for (int b = 0; b < 5; ++b) {
            nx[b] = false;
            if (!unary_ok(p, b)) continue;
            for (int a = 0; a < 5 && !nx[b]; ++a) nx[b] = can[a] && pair_ok(p - 1, a, b);
        }
        memcpy(can, nx, sizeof can);
    }
    return can[0] || can[1] || can[2] || can[3] || can[4];
}

// ---- staged records: one tile of a token, the row planted into it
struct Stage {
    std::vector<unsigned char> tok;
    std::vector<uint4> rec;
    uint32_t t_start, L;
    void set(uint32_t q, unsigned char ch) {             // token byte q and its record bits
        tok[q] = ch;
        const int64_t rel = (int64_t)q - t_start + 64;    // record word 1 holds t_start - 32 ..
        if (rel < 32 || rel >= 32 * (int64_t)kRecWords) return;
        const int k = (int)(rel / 32), b = (int)(rel % 32);
        const uint32_t nib = classify(ch), m = 1u << b;
        uint4 &w = rec[k];
        w.x = (w.x & ~m) | ((nib & 1u) << b), w.y = (w.y & ~m) | (((nib >> 1) & 1u) << b);
        w.z = (w.z & ~m) | (((nib >> 2) & 1u) << b), w.w = (w.w & ~m) | (((nib >> 3) & 1u) << b);
    }
};

// token byte that scores as `scored` (a row letter) in a window of the given strand; deco 0: plain
// upper case, 1: lower case, 2: U / Z where they score as this base (else plain)
static unsigned char token_byte(char scored, bool minus, int deco) {
    if (scored == 'N') return deco == 1 ? 'n' : 'N';
    if (deco == 1) return (unsigned char)(scored | 0x20);          // lower case is neither complemented nor dropped
    if (minus) {
        if (deco == 2 && scored == 'A') return 'U';
        if (deco == 2 && scored == 'C') return 'Z';
        return (unsigned char)scored;
    }
    if (deco == 2 && scored == 'T') return 'U';                     // '+' windows are read complemented
    if (deco == 2 && scored == 'G') return 'Z';
    return (unsigned char)(scored == 'A' ? 'T' : scored == 'T' ? 'A' : scored == 'C' ? 'G' : 'C');
}

int main(int argc, char **argv) {
    if (argc < 2) {
        printf("usage: rs1_lanes_emu ROWS_FILE\n");
        return 2;
    }
    std::vector<double> tab;
    char err[256];
    if (build_rs1_tables(tab, err, sizeof err)) {
        printf("FAIL build_rs1_tables: %s\n", err);
        return 1;
    }
    std::vector<std::string> rows;
    {
        FILE *f = fopen(argv[1], "r");
        if (!f) {
            printf("FAIL cannot open %s\n", argv[1]);
            return 1;
        }
        char line[128];
        while (fgets(line, sizeof line, f)) {
            size_t n = strcspn(line, "\r\n");
            line[n] = 0;
            if (n == 0) continue;
            if (n != 30 || strspn(line, "ATCGN") != 30 || line[2] != 'C' || line[3] != 'C') {
                printf("FAIL bad row '%s'\n", line);
                return 1;
            }
            rows.emplace_back(line);
        }
        fclose(f);
    }
    // the stage: a token of three tiles of random upper-case bases, its middle tile staged
    Stage st;
    st.t_start = kTile, st.L = 3u * kTile;
    st.tok.resize(st.L);
    for (auto &ch : st.tok) ch = (unsigned char)"ACGT"[rnd() & 3];
    st.rec.assign(kRecWords, make_uint4(0, 0, 0, 0));
    for (int k = 1; k < kRecWords; ++k)
        for (int b = 0; b < 32; ++b) st.set(st.t_start + (uint32_t)(k - 2) * 32u + (uint32_t)b, st.tok[st.t_start + (k - 2) * 32 + b]);
    static const uint32_t kPlaces[] = {0u, 1u, 30u, 31u, 32u, (uint32_t)kTile - 1u};

    std::set<uint32_t> states[8], table_states[8], visited[8];
    long bad = 0, n_placed = 0, deco_n[3] = {0, 0, 0};
    for (size_t r = 0; r < rows.size() && bad < 10; ++r) {
        const std::string &row = rows[r];
        int c[31];
        uint32_t s0 = 0, s1 = 0, valid = 0;
        for (int q = 0; q < 30; ++q) {
            c[q] = code_of(row[q]);
            if (c[q] < 4) valid |= 1u << q, s0 |= (uint32_t)(c[q] & 1) << q, s1 |= (uint32_t)(c[q] >> 1) << q;
        }
        c[30] = 4;
        const double dense = rs1_dense(s0, s1, valid, CRP_CLASS_CANONICAL, CRP_CLASS_CANONICAL);
        // A
        const double x = rs1_canonical(tab.data(), s0, s1, valid);
        if (bits_of(x) != bits_of(dense)) {
            printf("FAIL A: %s table %a dense %a\n", row.c_str(), x, dense);
            ++bad;
        }
        // S, and the states
        probe_lanes(tab.data(), ~s1 & ~s0 & valid, ~s1 & s0 & valid, s1 & ~s0 & valid, s1 & s0 & valid);
        int n_tabled = 0;
        for (int l = 0; l < 8; ++l) {
            const Rs1Lane &ln = kRs1Lanes[l];
            uint32_t on = 0;
            for (int i = 0; i < ln.n_entries; ++i)
                if (entry_matches(ln, ln.entries[i], c)) on |= 1u << i;
            states[l].insert(on);
            if (ln.bits < 0) continue;
            ++n_tabled;
            const uint32_t ton = on & ((1u << ln.n_table) - 1u);
            table_states[l].insert(ton);
            const uint32_t slot = rs1_table_slot(ln, ton, nullptr);
            int hits = 0;
            for (int k = 0; k < g_n_loads && k < 8; ++k)
                if (g_loads[k].off == (uint32_t)ln.offset) {
                    ++hits;
                    if (g_loads[k].idx8 != 8u * slot) {
                        printf("FAIL S: %s lane %s reads slot %u.%u, its entries %#x have slot %u\n", row.c_str(), ln.name,
                               g_loads[k].idx8 / 8u, g_loads[k].idx8 % 8u, ton, slot);
                        ++bad;
                    }
                }
            if (hits != 1) {
                printf("FAIL S: lane %s loaded %d times\n", ln.name, hits);
                ++bad;
            }
            visited[l].insert(slot);
        }
        if (g_n_loads != n_tabled) {
            printf("FAIL S: %d table loads for %d tabled lanes\n", g_n_loads, n_tabled);
            ++bad;
        }
        // B
        for (uint32_t p : kPlaces)
            for (int minus = 0; minus < 2; ++minus) {
                const int deco = (int)(rnd() % 3);
                ++deco_n[deco], ++n_placed;
                const uint32_t t = st.t_start + p;
                const uint32_t first = minus ? t - 2u : t - 25u;        // token position of the window's first byte
                unsigned char saved[30];
                for (int q = 0; q < 30; ++q) {
                    // output base q is tok[t - 2 + q] ('-') or tok[t + 4 - q] ('+'); bases 2 and 3 (the PAM) stay plain
                    const uint32_t at = minus ? t - 2u + (uint32_t)q : t + 4u - (uint32_t)q;
                    saved[at - first] = st.tok[at];
                    st.set(at, token_byte(row[q], minus, q == 2 || q == 3 ? 0 : deco));
                }
                unsigned long long word = 0;
                double xs;
                Window w;
                if (minus) {
                    const uint32_t ws = p + kWinBiasMinus, xt = st.L - 28u - (st.t_start - kWinBiasMinus);
                    xs = score_hit<true>(tab.data(), st.rec.data(), ws, xt, word);
                    w = extract_window<true>(st.rec.data(), ws, t, st.L);
                } else {
                    const uint32_t ws = p + kWinBiasPlusHot, xt = st.L - 5u - (st.t_start - kWinBiasPlusHot);
                    xs = score_hit<false>(tab.data(), st.rec.data(), ws, xt, word);
                    w = extract_window<false>(st.rec.data(), p + kWinBiasPlus, t, st.L);
                }
                if (w.valid != valid || (w.s0 & valid) != s0 || (w.s1 & valid) != s1) {
                    printf("FAIL B: %s planted at %u %c (deco %d) reads as s0 %08x s1 %08x valid %08x\n", row.c_str(), p,
                           minus ? '-' : '+', deco, w.s0, w.s1, w.valid);
                    ++bad;
                }
                if (bits_of(xs) != bits_of(dense) || word != w.packed) {
                    printf("FAIL B: %s at %u %c (deco %d): score_hit %a dense %a, packed %016llx / %016llx\n", row.c_str(), p,
                           minus ? '-' : '+', deco, xs, dense, word, w.packed);
                    ++bad;
                }
                for (int i = 0; i < 30; ++i) st.set(first + (uint32_t)i, saved[i]);
            }
    }
    if (bad) return 1;
    // coverage
    for (int l = 0; l < 8; ++l) {
        const Rs1Lane &ln = kRs1Lanes[l];
        if (ln.bits < 0) {
            printf("LANE %s states %zu table - slots -\n", ln.name, states[l].size());
            continue;
        }
        int free_idx[16], n_free = 0;
        for (int i = 0; i < ln.n_table; ++i)
            if (!ln.entries[i].forced) free_idx[n_free++] = i;
        std::set<uint32_t> want;
        long filled = 0;
        for (uint32_t sub = 0; sub < (1u << n_free); ++sub) {      // the subsets build_rs1_tables fills
            bool ok = true;
            for (int i = 0; i < n_free && ok; ++i)
                for (int j = i + 1; j < n_free; ++j)
                    if ((sub >> i & 1) && (sub >> j & 1) && ln.entries[free_idx[i]].pos == ln.entries[free_idx[j]].pos) ok = false;
            if (!ok) continue;
            ++filled;
            uint32_t on = 0;
            for (int i = 0; i < n_free; ++i)
                if (sub >> i & 1) on |= 1u << free_idx[i];
            if (table_state_reachable(ln, on)) want.insert(rs1_table_slot(ln, on, nullptr));
        }
        if (visited[l] != want) {
            long miss = 0, extra = 0;
            for (uint32_t s : want) miss += !visited[l].count(s);
            for (uint32_t s : visited[l]) extra += !want.count(s);
            printf("FAIL coverage: lane %s: %ld reachable slots not visited, %ld visited slots not reachable\n", ln.name, miss, extra);
            return 1;
        }
        printf("LANE %s states %zu table %zu slots %zu of %zu reachable, %ld filled\n", ln.name, states[l].size(),
               table_states[l].size(), visited[l].size(), want.size(), filled);
    }
    if (!deco_n[0] || !deco_n[1] || !deco_n[2]) {
        printf("FAIL B: not every byte flavour was planted\n");
        return 1;
    }
    printf("OK %zu rows, %ld plantings, every reachable table slot visited\n", rows.size(), n_placed);
    return 0;
}
