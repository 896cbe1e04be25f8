// TEST INFRASTRUCTURE: the PAM tests of k_ot_sites<*, true> (csrc/offtarget.cuh ot_pam_plus_sets / ot_pam_minus_sets),
// run on the CPU from the SAME source, so that without a GPU
//   A  for all 14 x 14 pairs of IUPAC letters (A C G T R Y S W K M B D H V) as letters 2 and 3, every bit of the two
//      masks of every tile word equals a byte-by-byte reading of random tokens of every byte class (upper, lower, N,
//      IUPAC, U / Z, decoration): '+' tok[t+1] a base in S2 and tok[t+2] a base in S3, '-' tok[t] a base in comp(S3)
//      and tok[t+1] a base in comp(S2), with the PAM letters straddling word edges, tile edges (the halo word) and
//      token ends;
//   B  the sets {G}, {G} give ot_pam_plus and ot_pam_minus bit for bit, on random record words of any content.
// The letter sets are written out here as strings of bases, not taken from the library.
// Built and run by tests/test_offtarget_pams.py (nvcc, no GPU needed).  Nothing here is part of the library.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../cropsr_b200/csrc/offtarget.cuh"

static unsigned long long rng_state = 0xD1B54A32D192ED03ull;
static inline unsigned long long rnd() {   // xorshift64*
    rng_state ^= rng_state >> 12;
    rng_state ^= rng_state << 25;
    rng_state ^= rng_state >> 27;
    return rng_state * 0x2545F4914F6CDD1Dull;
}

static const char kLetters[] = "ACGTRYSWKMBDHV";
static const char *kBases[] = {"A", "C", "G", "T", "AG", "CT", "CG", "AT", "GT", "AC", "CGT", "AGT", "ACT", "ACG"};

static int code_of(unsigned char c) {      // A0 T1 C2 G3 of ACGTacgt, else -1
    switch (c) {
    case 'A': case 'a': return 0;
    case 'T': case 't': return 1;
    case 'C': case 'c': return 2;
    case 'G': case 'g': return 3;
    default: return -1;
    }
}
static uint32_t set_of(const char *bases) {   // bit c for code c
    uint32_t s = 0;
    for (; *bases; ++bases) s |= 1u << code_of((unsigned char)*bases);
    return s;
}
static const char kComp[] = "TAGC";           // complement by code: A0 -> T, T1 -> A, C2 -> G, G3 -> C
// does byte c read as a base of `bases` (complemented when comp)?
static bool in_letter(int c, const char *bases, bool comp) {
    if (c < 0) return false;
    const int code = code_of((unsigned char)c);
    if (code < 0) return false;
    const char b = comp ? kComp[code] : "ATCG"[code];
    return strchr(bases, b) != nullptr;
}

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 40;
    long bad = 0, n_plus = 0, n_minus = 0, n_edge = 0, n_lower = 0;
    // ---------------------------------------------------------------- A
    static const char alphabet[] = "ACGTACGTacgtacgtGGAAGCNnRYSWKMBDHVryUZ'()*,.";
    std::vector<uint4> rec(kRecWords);
    for (int round = 0; round < rounds && bad < 10; ++round) {
        const uint32_t L = 1u + (uint32_t)(rnd() % (round % 4 == 0 ? 300u : 2u * kTile + 500u));
        std::vector<int> tok(L);
        for (auto &ch : tok) {
            const unsigned long long r = rnd();
            ch = round % 2 ? (unsigned char)"ACGTacgtAG"[r % 10] : (unsigned char)alphabet[r % (sizeof alphabet - 1)];
        }
        auto at = [&](int64_t q) { return q >= 0 && q < (int64_t)L ? tok[(size_t)q] : -1; };
        for (uint32_t t_start = 0; t_start < L; t_start += kTile) {
            for (int k = 1; k < kRecWords; ++k) {                  // the planes k_pack writes; outside the token "other"
                uint32_t o0 = 0, o1 = 0, ol = 0, oo = 0;
                for (int b = 0; b < 32; ++b) {
                    const int64_t q = (int64_t)t_start + ((int64_t)k - 2) * 32 + b;
                    const uint32_t nib = at(q) >= 0 ? classify((uint32_t)at(q)) : 8u;
                    o0 |= (nib & 1u) << b, o1 |= ((nib >> 1) & 1u) << b, ol |= ((nib >> 2) & 1u) << b, oo |= ((nib >> 3) & 1u) << b;
                }
                rec[k] = make_uint4(o0, o1, ol, oo);
            }
            for (int i2 = 0; i2 < 14; ++i2)
                for (int i3 = 0; i3 < 14; ++i3) {
                    const uint32_t s2 = set_of(kBases[i2]), s3 = set_of(kBases[i3]);
                    for (int k = 0; k < kTileWords && bad < 10; ++k) {
                        const uint32_t plus = ot_pam_plus_sets(rec[2 + k], rec[3 + k], s2, s3);
                        const uint32_t minus = ot_pam_minus_sets(rec[2 + k], rec[3 + k], s2, s3);
                        for (int b = 0; b < 32; ++b) {
                            const int64_t t = (int64_t)t_start + 32 * k + b;
                            const bool wp = in_letter(at(t + 1), kBases[i2], false) && in_letter(at(t + 2), kBases[i3], false);
                            const bool wm = in_letter(at(t), kBases[i3], true) && in_letter(at(t + 1), kBases[i2], true);
                            if (wp != (bool)(plus >> b & 1u) || wm != (bool)(minus >> b & 1u)) {
                                if (bad < 10)
                                    printf("N%c%c t=%lld: plus %d/%d minus %d/%d\n", kLetters[i2], kLetters[i3], (long long)t,
                                           (int)(plus >> b & 1u), wp, (int)(minus >> b & 1u), wm);
                                ++bad;
                            }
                            n_plus += wp, n_minus += wm;
                            n_edge += (wp || wm) && (b >= 30 || k == kTileWords - 1 || t + 3 >= (int64_t)L);
                            n_lower += wp && at(t + 2) >= 'a';
                        }
                    }
                }
        }
    }
    // ---------------------------------------------------------------- B
    for (int i = 0; i < 200000 && bad < 10; ++i) {
        const uint4 cur = make_uint4((uint32_t)rnd(), (uint32_t)rnd(), (uint32_t)rnd(), (uint32_t)rnd() & (uint32_t)rnd());
        const uint4 next = make_uint4((uint32_t)rnd(), (uint32_t)rnd(), (uint32_t)rnd(), (uint32_t)rnd() & (uint32_t)rnd());
        if (ot_pam_plus_sets(cur, next, 8u, 8u) != ot_pam_plus(cur, next) ||
            ot_pam_minus_sets(cur, next, 8u, 8u) != ot_pam_minus(cur, next)) {
            printf("NGG words differ at %d\n", i);
            ++bad;
        }
    }
    if (bad || !n_plus || !n_minus || !n_edge || !n_lower) {
        printf("FAIL: %ld mismatches (plus %ld minus %ld edge %ld lower %ld)\n", bad, n_plus, n_minus, n_edge, n_lower);
        return 1;
    }
    printf("OK: %ld '+' and %ld '-' pattern sites over 196 patterns, %ld at word / tile / token edges, %ld lower case\n",
           n_plus, n_minus, n_edge, n_lower);
    return 0;
}
