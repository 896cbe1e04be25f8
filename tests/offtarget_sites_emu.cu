// TEST INFRASTRUCTURE: the locus packing of k_ot_sites<true> (csrc/offtarget.cuh: ot_site_locus on the descriptor
// word of a tile record, as the kernel stores it next to the key), run on the CPU from the SAME source and compared
// with a byte-by-byte reading of random tokens: every byte class, both strands, lower-case PAMs, sites in the halo
// and at tile edges and token ends, several segments per token (128-aligned shard boundaries) and several tokens per
// genome handle, and genome ordinals up to 126.  The locus is decoded here by its documented bit fields (t 0-31,
// segment 32-55, genome 56-62, strand 63), not by the library's helper.
// Built and run by tests/test_offtarget_sites.py (nvcc, no GPU needed).  Nothing here is part of the library.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <tuple>
#include <vector>

#include "../cropsr_b200/csrc/offtarget.cuh"

static unsigned long long rng_state = 0x9E3779B97F4A7C15ull;
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

// t, strand (0 '+', 1 '-'), key, segment, genome
typedef std::tuple<uint32_t, int, unsigned long long, uint32_t, uint32_t> Site;

// the definition, byte by byte, for the positions [lo, hi) a segment owns
static void sites_by_bytes(const std::vector<unsigned char> &tok, uint32_t lo, uint32_t hi, uint32_t seg, uint32_t genome,
                           std::vector<Site> &out) {
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
            if (ok) out.emplace_back((uint32_t)t, 0, key, seg, genome);
        }
        if (t + 1 < L && code_of(tok[t]) == 2 && code_of(tok[t + 1]) == 2 && t + 23 <= L) {
            unsigned long long key = 0;
            bool ok = true;
            for (int i = 0; i < 20 && ok; ++i) {
                const int c = code_of(tok[t + 22 - i]);
                ok = c >= 0;
                key |= (unsigned long long)((c ^ 1) & 3) << (2 * i);
            }
            if (ok) out.emplace_back((uint32_t)t, 1, key, seg, genome);
        }
    }
}

int main(int argc, char **argv) {
    const int rounds = argc > 1 ? atoi(argv[1]) : 60;
    long bad = 0, n_sites = 0, n_minus = 0, n_edge = 0, n_halo = 0, n_lower_pam = 0, n_multi_seg = 0;
    static const char alphabet[] = "GGGGCCCCggccAATTatNnUZ'()*RY";
    std::vector<uint4> rec(kRecWords);
    for (int round = 0; round < rounds && bad < 10; ++round) {
        const uint32_t genome = (uint32_t)(rnd() % kOtMaxGenomes);
        const int n_tok = 1 + (int)(rnd() % 3);
        uint32_t seg = 0;                  // segment index in the handle: running over the handle's tokens
        std::vector<Site> want, got;
        for (int ti = 0; ti < n_tok; ++ti) {
            const uint32_t L = 1u + (uint32_t)(rnd() % (round % 4 == 0 ? 300u : 50000u));
            std::vector<unsigned char> tok(L);
            const int flavour = round % 3;     // 0 every byte class, 1 bases only (many sites), 2 bases with rare others
            for (auto &ch : tok) {
                const unsigned long long r = rnd();
                ch = flavour == 1 ? (unsigned char)"GCgcATat"[r & 7]
                     : flavour == 2 && r % 50 ? (unsigned char)"GGCCgcAT"[r & 7]
                                              : (unsigned char)alphabet[r % (sizeof alphabet - 1)];
            }
            // the token cut into 1 .. 4 segments at 128-aligned boundaries
            std::vector<uint32_t> cuts = {0u};
            const int n_cut = L > 4 * kAlign ? (int)(rnd() % 4) : 0;
            for (int c = 0; c < n_cut; ++c) cuts.push_back((uint32_t)(rnd() % L) / kAlign * kAlign);
            cuts.push_back(L);
            std::sort(cuts.begin(), cuts.end());
            cuts.erase(std::unique(cuts.begin(), cuts.end()), cuts.end());
            n_multi_seg += cuts.size() > 2;
            for (size_t c = 0; c + 1 < cuts.size(); ++c, ++seg) {
                const uint32_t seg_b = cuts[c], seg_e = cuts[c + 1];
                sites_by_bytes(tok, seg_b, seg_e, seg, genome, want);
                const int64_t st_lo = seg_b >= 32 ? seg_b - 32 : 0, st_hi = seg_e + 32 < L ? seg_e + 32 : L;   // staged bytes
                for (uint32_t t_start = seg_b; t_start < seg_e; t_start += kTile) {
                    const uint32_t n_owned = seg_e - t_start < (uint32_t)kTile ? seg_e - t_start : (uint32_t)kTile;
                    rec[0] = make_uint4(t_start, L, n_owned, seg);                  // the descriptor word k_pack writes
                    for (int k = 1; k < kRecWords; ++k) {
                        uint32_t o0 = 0, o1 = 0, ol = 0, oo = 0;
                        for (int b = 0; b < 32; ++b) {
                            const int64_t q = (int64_t)t_start + ((int64_t)k - 2) * 32 + b;
                            const uint32_t nib = q >= st_lo && q < st_hi ? classify(tok[(size_t)q]) : 8u;
                            o0 |= (nib & 1u) << b, o1 |= ((nib >> 1) & 1u) << b, ol |= ((nib >> 2) & 1u) << b, oo |= ((nib >> 3) & 1u) << b;
                        }
                        rec[k] = make_uint4(o0, o1, ol, oo);
                    }
                    for (uint32_t k = 0; k < (uint32_t)kTileWords; ++k) {      // k_ot_sites<true>: one thread per tile word
                        const uint32_t p0 = 32u * k;
                        if (p0 >= rec[0].z) break;
                        const uint32_t own = rec[0].z - p0 >= 32u ? 0xFFFFFFFFu : (1u << (rec[0].z - p0)) - 1u;
                        const uint4 prev = rec[1 + k], cur = rec[2 + k], next = rec[3 + k];
                        unsigned long long key;
                        for (int minus = 0; minus < 2; ++minus) {
                            const uint32_t hits = (minus ? ot_pam_minus(cur, next) : ot_pam_plus(cur, next)) & own;
                            for (uint32_t m = hits; m; m &= m - 1) {
                                const uint32_t b = __builtin_ctz(m);
                                const bool ok = minus ? ot_key<true>(prev, cur, next, b, key) : ot_key<false>(prev, cur, next, b, key);
                                if (!ok) continue;
                                const unsigned long long loc = ot_site_locus(rec[0], k, b, genome, minus != 0);
                                got.emplace_back((uint32_t)(loc & 0xFFFFFFFFull), (int)(loc >> 63), key,
                                                 (uint32_t)((loc >> 32) & 0xFFFFFFull), (uint32_t)((loc >> 56) & 0x7Full));
                            }
                        }
                    }
                }
            }
            for (const Site &s : want) {
                if (std::get<3>(s) >= seg - (uint32_t)(cuts.size() - 1) && std::get<0>(s) < L) {
                    const uint32_t t = std::get<0>(s);
                    n_lower_pam += std::get<1>(s) ? t + 1 < L && (tok[t] == 'c' || tok[t + 1] == 'c')
                                                  : t + 2 < L && (tok[t + 1] == 'g' || tok[t + 2] == 'g');
                }
            }
        }
        std::sort(want.begin(), want.end());
        std::sort(got.begin(), got.end());
        if (want != got) {
            printf("FAIL: round %d (genome %u, %d tokens): %zu sites by bytes, %zu from the records\n", round, genome, n_tok,
                   want.size(), got.size());
            for (size_t i = 0; i < std::min(want.size(), got.size()); ++i)
                if (want[i] != got[i]) {
                    printf("  first difference: want t=%u s=%d seg=%u g=%u, got t=%u s=%d seg=%u g=%u\n", std::get<0>(want[i]),
                           std::get<1>(want[i]), std::get<3>(want[i]), std::get<4>(want[i]), std::get<0>(got[i]),
                           std::get<1>(got[i]), std::get<3>(got[i]), std::get<4>(got[i]));
                    break;
                }
            ++bad;
        }
        for (const Site &s : want) {
            const uint32_t p = std::get<0>(s) % kTile;
            n_sites++;
            n_minus += std::get<1>(s);
            n_edge += p < 23 || p + 23 >= (uint32_t)kTile;
            n_halo += (std::get<0>(s) % kAlign) < 23 || (std::get<0>(s) % kAlign) + 23 >= kAlign;
        }
    }
    if (bad) return 1;
    if (n_sites < 1000 || n_minus == 0 || n_minus == n_sites || n_edge == 0 || n_halo == 0 || n_lower_pam == 0 ||
        n_multi_seg == 0) {
        printf("FAIL: the sample does not exercise both strands, tile and segment edges, lower-case PAMs and several "
               "segments (%ld sites)\n", n_sites);
        return 1;
    }
    printf("OK %ld sites (%ld '-', %ld at tile edges, %ld near 128-aligned boundaries, %ld with a lower-case PAM), %ld "
           "tokens cut into several segments\n", n_sites, n_minus, n_edge, n_halo, n_lower_pam, n_multi_seg);
    return 0;
}
