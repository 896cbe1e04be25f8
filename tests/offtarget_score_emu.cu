// TEST INFRASTRUCTURE: the rank of k_ot_join<OtScore> (csrc/offtarget.cuh: ot_mask_rank behind the pair rule
// ot_bucket / ot_rest / ot_rest_mismatches of k_ot_join), run on the CPU from the SAME source.  For every part pair
// (i, j) and every one of the 1,351 mismatch-position sets of size <= 3, query and site keys are built with
// substitutions at exactly those positions (random keys and random substitute bases, several draws):
//   - where the pair rule keeps the set at (i, j) -- parts i and j match and no part below j other than i does --
//     the bucket keys agree, ot_rest_mismatches returns |set| and ot_mask_rank returns the set's colex rank,
//     computed here from binomials: {1, 21, 211}[|set| - 1] + C(a,1) + C(b,2) + C(c,3);
//   - everywhere else ot_rest_mismatches rejects the pair, or the bucket keys differ;
//   - each set is kept at exactly one part pair, and a smaller k rejects sets larger than k.
// Built and run by tests/test_offtarget_score.py (nvcc, no GPU needed).  Nothing here is part of the library.
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "../cropsr_b200/csrc/offtarget.cuh"

static unsigned long long rng_state = 0x853C49E6748FEA9Bull;
static inline unsigned long long rnd() {   // xorshift64*
    rng_state ^= rng_state >> 12;
    rng_state ^= rng_state << 25;
    rng_state ^= rng_state >> 27;
    return rng_state * 0x2545F4914F6CDD1Dull;
}

static uint32_t binom(uint32_t n, uint32_t r) {
    uint64_t v = 1;
    for (uint32_t t = 0; t < r; ++t) v = v * (n - t) / (t + 1);
    return n < r ? 0u : (uint32_t)v;
}

int main() {
    // the sets in rank order: size, then colex (largest element first)
    std::vector<std::vector<int>> sets = {{}};
    for (int a = 0; a < 20; ++a) sets.push_back({a});
    for (int b = 1; b < 20; ++b)
        for (int a = 0; a < b; ++a) sets.push_back({a, b});
    for (int c = 2; c < 20; ++c)
        for (int b = 1; b < c; ++b)
            for (int a = 0; a < b; ++a) sets.push_back({a, b, c});
    if (sets.size() != kOtScoreSets) {
        printf("FAIL %zu sets\n", sets.size());
        return 1;
    }
    long bad = 0, kept = 0, rejected = 0;
    for (size_t r = 0; r < sets.size() && bad < 20; ++r) {
        const std::vector<int> &set = sets[r];
        static const uint32_t offset[4] = {0, 1, 21, 211};
        uint32_t want_rank = offset[set.size()];
        for (size_t e = 0; e < set.size(); ++e) want_rank += binom((uint32_t)set[e], (uint32_t)e + 1);
        if (want_rank != r) {
            printf("FAIL binomial rank of set %zu is %u\n", r, want_rank);
            ++bad;
        }
        bool part_hit[5] = {false, false, false, false, false};
        for (int p : set) part_hit[p / 4] = true;
        int lo0 = -1, lo1 = -1;                    // the two lowest exactly matching parts
        for (int p = 0; p < 5; ++p)
            if (!part_hit[p]) {
                if (lo0 < 0) lo0 = p;
                else if (lo1 < 0) lo1 = p;
            }
        for (int draw = 0; draw < 8; ++draw) {
            const unsigned long long q = rnd() & 0xFFFFFFFFFFull;
            unsigned long long s = q;
            for (int p : set) s ^= (1ull + rnd() % 3ull) << (2 * p);   // another base at p
            int n_kept = 0;
            for (int pp = 0; pp < kOtPairs; ++pp) {
                int i = 0, j = 0;
                ot_pair(pp, i, j);
                const bool want = i == lo0 && j == lo1;
                const bool same_bucket = ot_bucket(q, i, j) == ot_bucket(s, i, j);
                const uint32_t rq = ot_rest(q, i, j), rs = ot_rest(s, i, j);
                const int d = ot_rest_mismatches(rq, rs, 3u, (uint32_t)(j - 1));
                const bool got = same_bucket && d >= 0;
                if (got != want) {
                    printf("FAIL set %zu pair (%d,%d): kept %d, want %d\n", r, i, j, (int)got, (int)want);
                    ++bad;
                    continue;
                }
                if (!got) {
                    ++rejected;
                    continue;
                }
                ++n_kept;
                ++kept;
                const uint32_t x = rq ^ rs, rank = ot_mask_rank((x | x >> 1) & 0x555555u, i, j);
                if (d != (int)set.size() || rank != r) {
                    printf("FAIL set %zu pair (%d,%d): d %d rank %u\n", r, i, j, d, rank);
                    ++bad;
                }
                for (uint32_t k = 0; k < set.size(); ++k)            // a smaller k rejects it
                    if (ot_rest_mismatches(rq, rs, k, (uint32_t)(j - 1)) >= 0) {
                        printf("FAIL set %zu pair (%d,%d): kept at k = %u\n", r, i, j, k);
                        ++bad;
                    }
            }
            if (n_kept != 1) {
                printf("FAIL set %zu kept at %d part pairs\n", r, n_kept);
                ++bad;
            }
        }
    }
    if (bad) return 1;
    printf("OK %zu sets, %ld kept, %ld rejected\n", sets.size(), kept, rejected);
    return 0;
}
