// TEST INFRASTRUCTURE: the per-site functions of the off-target kernels (csrc/offtarget.cuh), run on the CPU from the
// SAME source, so that without a GPU
//   A  the site tests and the key builder of k_ot_sites / k_ot_queries (ot_pam_plus, ot_pam_minus, ot_key on the three
//      record words around a position) equal a byte-by-byte reading of random tokens: every byte class, both strands,
//      lower-case PAMs, sites straddling tile edges and token ends, segments that start or end inside a token;
//   B  the pair rule of k_ot_join (ot_bucket, ot_rest, ot_rest_mismatches) counts a (query, site) pair with d <= 3
//      mismatches at exactly one of the 10 part pairs and a pair with d >= 4 at none: exhaustively over all 1,351
//      mismatch-position sets of size <= 3 (random substitutions at those positions, random keys), for every k, and
//      on a sample of larger sets.
// Built and run by tests/test_offtarget.py (nvcc, no GPU needed).  Nothing here is part of the library.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <tuple>
#include <vector>

#include "../cropsr_b200/csrc/offtarget.cuh"

static unsigned long long rng_state = 0x2545F4914F6CDD1Dull;
static inline unsigned long long rnd() {   // xorshift64*
    rng_state ^= rng_state >> 12;
    rng_state ^= rng_state << 25;
    rng_state ^= rng_state >> 27;
    return rng_state * 0x2545F4914F6CDD1Dull;
}

static int code_of(unsigned char c) {      // A0 T1 C2 G3 of ACGTacgt, else -1
    switch (c) {
    case 'A': case 'a': return 0;
    case 'T': case 't': return 1;
    case 'C': case 'c': return 2;
    case 'G': case 'g': return 3;
    default: return -1;
    }
}

typedef std::tuple<uint32_t, int, unsigned long long> Site;   // t, strand (0 '+', 1 '-'), key

// the definition, byte by byte
static void sites_by_bytes(const std::vector<unsigned char> &tok, uint32_t lo, uint32_t hi, std::vector<Site> &out) {
    const int64_t L = (int64_t)tok.size();
    for (int64_t t = lo; t < hi; ++t) {
        if (t + 2 < L && code_of(tok[t + 1]) == 3 && code_of(tok[t + 2]) == 3 && t >= 20) {
            unsigned long long key = 0;
            bool ok = true;
            for (int i = 0; i < 20 && ok; ++i) {
                const int c = code_of(tok[t - 20 + i]);
                ok = c >= 0;
                key |= (unsigned long long)(c & 3) << (2 * i);
            }
            if (ok) out.emplace_back((uint32_t)t, 0, key);
        }
        if (t + 1 < L && code_of(tok[t]) == 2 && code_of(tok[t + 1]) == 2 && t + 23 <= L) {
            unsigned long long key = 0;
            bool ok = true;
            for (int i = 0; i < 20 && ok; ++i) {
                const int c = code_of(tok[t + 22 - i]);
                ok = c >= 0;
                key |= (unsigned long long)((c ^ 1) & 3) << (2 * i);
            }
            if (ok) out.emplace_back((uint32_t)t, 1, key);
        }
    }
}

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 120;
    long bad = 0, n_sites = 0, n_edge = 0, n_minus = 0, n_lower_pam = 0;
    // ---------------------------------------------------------------- A
    static const char alphabet[] = "GGGGCCCCggccAATTatNnUZ'()*RY";
    std::vector<uint4> rec(kRecWords);
    for (int round = 0; round < rounds && bad < 10; ++round) {
        const uint32_t L = 1u + (uint32_t)(rnd() % (round % 4 == 0 ? 200u : 40000u));
        std::vector<unsigned char> tok(L);
        const int flavour = round % 3;     // 0 every byte class, 1 bases only (many sites), 2 bases with rare others
        for (auto &ch : tok) {
            const unsigned long long r = rnd();
            ch = flavour == 1 ? (unsigned char)"GCgcATat"[r & 7]
                 : flavour == 2 && r % 50 ? (unsigned char)"GGCCgcAT"[r & 7]
                                          : (unsigned char)alphabet[r % (sizeof alphabet - 1)];
        }
        uint32_t seg_b = 0, seg_e = L;     // a 128-aligned part of the token (a shard boundary), or the whole token
        if (round % 3 == 1 && L > 512) {
            seg_b = (uint32_t)(rnd() % (L / 2)) / kAlign * kAlign;
            seg_e = seg_b + (uint32_t)(1 + rnd() % (L - seg_b));
            if (seg_e < L) seg_e = (seg_e + kAlign - 1) / kAlign * kAlign;
            if (seg_e > L) seg_e = L;
        }
        const int64_t st_lo = seg_b >= 32 ? seg_b - 32 : 0, st_hi = seg_e + 32 < L ? seg_e + 32 : L;   // staged bytes
        std::vector<Site> want, got;
        sites_by_bytes(tok, seg_b, seg_e, want);
        for (uint32_t t_start = seg_b; t_start < seg_e; t_start += kTile) {
            const uint32_t n_owned = seg_e - t_start < (uint32_t)kTile ? seg_e - t_start : (uint32_t)kTile;
            for (int k = 1; k < kRecWords; ++k) {                  // the planes k_pack writes
                uint32_t o0 = 0, o1 = 0, ol = 0, oo = 0;
                for (int b = 0; b < 32; ++b) {
                    const int64_t q = (int64_t)t_start + ((int64_t)k - 2) * 32 + b;
                    const uint32_t nib = q >= st_lo && q < st_hi ? classify(tok[(size_t)q]) : 8u;
                    o0 |= (nib & 1u) << b, o1 |= ((nib >> 1) & 1u) << b, ol |= ((nib >> 2) & 1u) << b, oo |= ((nib >> 3) & 1u) << b;
                }
                rec[k] = make_uint4(o0, o1, ol, oo);
            }
            for (const Site &s : want) {                           // k_ot_queries: the words around a candidate's t
                const uint32_t t = std::get<0>(s);
                if (t < t_start || t >= t_start + n_owned) continue;
                const uint32_t p = t - t_start, k = p >> 5, b = p & 31u;
                unsigned long long key = 0;
                const bool ok = std::get<1>(s) ? ot_key<true>(rec[1 + k], rec[2 + k], rec[3 + k], b, key)
                                               : ot_key<false>(rec[1 + k], rec[2 + k], rec[3 + k], b, key);
                if (!ok || key != std::get<2>(s)) {
                    printf("FAIL A: query key at t=%u strand %d: %016llx, want %016llx\n", t, std::get<1>(s), key, std::get<2>(s));
                    ++bad;
                }
            }
            for (uint32_t k = 0; k < (uint32_t)kTileWords; ++k) {  // k_ot_sites: one thread per tile word
                const uint32_t p0 = 32u * k;
                if (p0 >= n_owned) break;
                const uint32_t own = n_owned - p0 >= 32u ? 0xFFFFFFFFu : (1u << (n_owned - p0)) - 1u;
                const uint4 prev = rec[1 + k], cur = rec[2 + k], next = rec[3 + k];
                unsigned long long key;
                for (uint32_t m = ot_pam_plus(cur, next) & own; m; m &= m - 1) {
                    const uint32_t b = __builtin_ctz(m);
                    if (ot_key<false>(prev, cur, next, b, key)) got.emplace_back(t_start + p0 + b, 0, key);
                }
                for (uint32_t m = ot_pam_minus(cur, next) & own; m; m &= m - 1) {
                    const uint32_t b = __builtin_ctz(m);
                    if (ot_key<true>(prev, cur, next, b, key)) got.emplace_back(t_start + p0 + b, 1, key);
                }
            }
        }
        std::sort(want.begin(), want.end());
        std::sort(got.begin(), got.end());
        if (want != got) {
            printf("FAIL A: L=%u segment [%u, %u) flavour %d: %zu sites by bytes, %zu from the records\n", L, seg_b, seg_e, flavour,
                   want.size(), got.size());
            ++bad;
        }
        for (const Site &s : want) {
            const uint32_t t = std::get<0>(s), p = (t - seg_b) % kTile;
            n_sites++;
            n_minus += std::get<1>(s);
            n_edge += p < 23 || p + 23 >= (uint32_t)kTile || t < 25 || t + 26 > L;
            n_lower_pam += std::get<1>(s) ? tok[t] == 'c' || tok[t + 1] == 'c' : tok[t + 1] == 'g' || tok[t + 2] == 'g';
        }
    }
    if (!bad && (n_sites < 1000 || n_edge == 0 || n_minus == 0 || n_minus == n_sites || n_lower_pam == 0)) {
        printf("FAIL A: the sample does not exercise both strands, tile edges and lower-case PAMs (%ld sites)\n", n_sites);
        return 1;
    }
    // ---------------------------------------------------------------- B
    long n_sets = 0, n_large = 0;
    std::vector<int> S;
    auto check = [&](const std::vector<int> &pos) {
        for (int rep = 0; rep < 4; ++rep) {
            const unsigned long long q = rnd() & ((1ull << 40) - 1);
            unsigned long long s = q;
            for (int p : pos) s ^= (unsigned long long)(1 + rnd() % 3) << (2 * p);   // a different base at p
            for (uint32_t k = 0; k <= 3; ++k) {
                int counted = 0, d_seen = -1;
                for (int pp = 0; pp < kOtPairs; ++pp) {
                    int i, j;
                    ot_pair(pp, i, j);
                    if (ot_bucket(q, i, j) != ot_bucket(s, i, j)) continue;       // not in the same bucket
                    const int d = ot_rest_mismatches(ot_rest(q, i, j), ot_rest(s, i, j), k, (uint32_t)(j - 1));
                    if (d >= 0) ++counted, d_seen = d;
                }
                const int want_n = (int)pos.size() <= (int)k ? 1 : 0;
                if (counted != want_n || (want_n && d_seen != (int)pos.size())) {
                    printf("FAIL B: %zu mismatches, k=%u: counted %d times (d=%d)\n", pos.size(), k, counted, d_seen);
                    ++bad;
                    return;
                }
            }
        }
    };
    // all subsets of size <= 3 of the 20 positions, enumerated as bit sets
    for (uint32_t m = 0; m < (1u << 20) && bad < 10; ++m) {
        const int n = __builtin_popcount(m);
        if (n > 3) continue;
        S.clear();
        for (int p = 0; p < 20; ++p)
            if (m >> p & 1u) S.push_back(p);
        check(S);
        ++n_sets;
    }
    for (int r = 0; r < 20000 && bad < 10; ++r, ++n_large) {            // 4 .. 20 mismatches
        const int n = 4 + (int)(rnd() % 17);
        std::vector<int> all(20);
        for (int p = 0; p < 20; ++p) all[p] = p;
        for (int p = 0; p < n; ++p) std::swap(all[p], all[p + rnd() % (20 - p)]);
        S.assign(all.begin(), all.begin() + n);
        std::sort(S.begin(), S.end());
        check(S);
    }
    if (bad) return 1;
    if (n_sets != 1351) {
        printf("FAIL B: %ld mismatch-position sets of size <= 3, not 1351\n", n_sets);
        return 1;
    }
    printf("OK %ld sites (%ld '-', %ld at tile edges or token ends, %ld with a lower-case PAM), %ld + %ld mismatch sets\n",
           n_sites, n_minus, n_edge, n_lower_pam, n_sets, n_large);
    return 0;
}
