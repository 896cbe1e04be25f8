// TEST INFRASTRUCTURE: the work-item geometry of k_ot_join (csrc/offtarget.cuh: ot_bucket_items, ot_item_bucket,
// ot_item, ot_copy_first / ot_copy_bytes / ot_copy_offset, ot_threads_per_query, ot_thread_active), run on the CPU from
// the SAME source, so that without a GPU
//   A  over bucket tables built as k_ot_scan builds them (soff, qoff, item_off), for every nq in 1 .. 300 and ns in
//      {1, 2, 3, 2047, 2048, 2049, 4095, 4096, 4097, 6145}, at buckets 0 and 65535 and at middle buckets whose first
//      site has every residue mod 4, next to empty buckets, buckets with sites only and buckets with queries only:
//      every work item maps to its own bucket, and the items of a bucket tile [0, nq) x [0, ns) exactly once;
//   B  for every item and both site sizes (4: counts and scores, 8: listings) the bulk copy starts 16-byte aligned, is
//      a multiple of 16 bytes, covers the tile, fits the shared tile of kOtSiteTile + 16 / size elements, puts site s0
//      at the tile's offset and reads nothing past the site array's padding (kOtSitePad);
//   C  for every nq_t in 1 .. 128 and a dense sample of ns_t in 1 .. 2048 the active threads of the split visit every
//      (query, site) pair of the tile exactly once (the kernel's loop: site tid / nq_t, step g), and every thread that
//      holds no query is inactive.
// Built and run by tests/test_offtarget_join_edges.py (nvcc, no GPU needed).  Nothing here is part of the library.
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "../cropsr_b200/csrc/offtarget.cuh"

static long bad = 0;
#define FAIL(...)                                                                                                      \
    do {                                                                                                               \
        if (bad++ < 20) printf("FAIL " __VA_ARGS__);                                                                   \
    } while (0)

struct Tables {
    std::vector<uint32_t> ns, nq;                       // per bucket
    std::vector<uint32_t> soff, qoff, item_off;         // [kOtBuckets + 1], exclusive prefixes as k_ot_scan writes them
};

static void prefix(Tables &t) {
    unsigned long long s = 0, q = 0, it = 0;
    for (uint32_t b = 0; b < kOtBuckets; ++b) {
        t.soff[b] = (uint32_t)s, t.qoff[b] = (uint32_t)q, t.item_off[b] = (uint32_t)it;
        s += t.ns[b], q += t.nq[b], it += ot_bucket_items(t.ns[b], t.nq[b]);
    }
    t.soff[kOtBuckets] = (uint32_t)s, t.qoff[kOtBuckets] = (uint32_t)q, t.item_off[kOtBuckets] = (uint32_t)it;
    if (it >> 32) FAIL("test tables with 2^32 items\n");
}

// B for one site size: the copy of the tile [s0, s0 + ns_t) of an array of n_sites sites (+ kOtSitePad allocated)
template <uint32_t kSize>
static void check_copy(uint32_t s0, uint32_t ns_t, uint32_t n_sites, long &n_copies) {
    const uint32_t a0 = ot_copy_first<kSize>(s0), bytes = ot_copy_bytes<kSize>(s0, ns_t, a0), off = ot_copy_offset(s0, a0);
    const unsigned long long src = (unsigned long long)a0 * kSize, alloc = (unsigned long long)(n_sites + kOtSitePad) * kSize;
    ++n_copies;
    if (src % 16 || bytes % 16 || !bytes)
        FAIL("copy of size %u at s0=%u: source byte %llu, %u bytes: not whole 16-byte units\n", kSize, s0, src, bytes);
    else if (src + bytes > alloc)
        FAIL("copy of size %u at s0=%u ns_t=%u: reads to byte %llu of an allocation of %llu (%u sites)\n", kSize, s0, ns_t,
             src + bytes, alloc, n_sites);
    else if (bytes > (kOtSiteTile + 16 / kSize) * kSize)
        FAIL("copy of size %u at s0=%u ns_t=%u: %u bytes overflow the shared tile\n", kSize, s0, ns_t, bytes);
    else if ((unsigned long long)off + ns_t > bytes / kSize || a0 + off != s0)   // shared element e holds site a0 + e
        FAIL("copy of size %u at s0=%u ns_t=%u: tile offset %u does not put sites [s0, s0 + ns_t) in the %u copied\n", kSize,
             s0, ns_t, off, bytes / kSize);
}

int main() {
    static const uint32_t kNs[] = {1, 2, 3, 2047, 2048, 2049, 4095, 4096, 4097, 6145};
    Tables t;
    t.ns.assign(kOtBuckets, 0), t.nq.assign(kOtBuckets, 0);
    t.soff.resize(kOtBuckets + 1), t.qoff.resize(kOtBuckets + 1), t.item_off.resize(kOtBuckets + 1);
    long n_tables = 0, n_items = 0, n_copies = 0, n_targets = 0;
    bool residue[4] = {false, false, false, false}, first_bucket = false, last_bucket = false;
    std::vector<uint32_t> touched;
    // ---------------------------------------------------------------- A, B
    for (uint32_t nq = 1; nq <= 300 && bad < 20; ++nq)
        for (uint32_t ns : kNs) {
            for (uint32_t b : touched) t.ns[b] = t.nq[b] = 0;
            touched.clear();
            auto put = [&](uint32_t b, uint32_t s, uint32_t q) {
                t.ns[b] = s, t.nq[b] = q;
                touched.push_back(b);
            };
            // targets at buckets 0 and 65535 and at four middle buckets, each behind a bucket of sites only that gives
            // its first site residue r mod 4 and before a bucket of queries only; empty buckets between them
            const uint32_t mid = 2 + (uint32_t)(n_tables * 40503u) % 60000u;
            put(0, ns, nq);
            put(kOtBuckets - 1, ns, nq);
            uint32_t before = ns;                        // sites in buckets below the next filler
            for (uint32_t r = 0; r < 4; ++r) {
                const uint32_t m = mid + 1000 * r;
                const uint32_t fill = 4 + (r + 4 - before % 4) % 4;
                put(m - 1, fill, 0);
                put(m, ns, nq);
                put(m + 1, 0, 1 + (uint32_t)(n_tables % 200));
                before += fill + ns;
            }
            prefix(t);
            ++n_tables;
            const uint32_t n_sites = t.soff[kOtBuckets];
            for (uint32_t b : touched) {
                const unsigned long long items = ot_bucket_items(t.ns[b], t.nq[b]);
                if (items != (t.ns[b] && t.nq[b] ? (unsigned long long)((t.nq[b] + 127) / 128) * ((t.ns[b] + 2047) / 2048) : 0))
                    FAIL("bucket %u: %llu items for %u queries x %u sites\n", b, items, t.nq[b], t.ns[b]);
                if (!items) continue;
                ++n_targets;
                residue[t.soff[b] % 4] |= b != 0 && b != kOtBuckets - 1 && t.ns[b] > kOtSiteTile;
                first_bucket |= b == 0;
                last_bucket |= b == kOtBuckets - 1;
                const uint32_t n_qt = (t.nq[b] + 127) / 128, n_st = (t.ns[b] + 2047) / 2048;
                std::vector<char> seen((size_t)n_qt * n_st, 0);
                for (uint32_t item = t.item_off[b]; item < t.item_off[b + 1]; ++item, ++n_items) {
                    const uint32_t got = ot_item_bucket(t.item_off.data(), item);
                    if (got != b) {
                        FAIL("item %u of bucket %u (nq %u, ns %u) maps to bucket %u\n", item, b, t.nq[b], t.ns[b], got);
                        continue;
                    }
                    const OtItem it = ot_item(t.soff.data(), t.qoff.data(), t.item_off.data(), b, item);
                    const uint32_t q = it.q0 - t.qoff[b], s = it.s0 - t.soff[b];
                    if (q % kOtThreads || s % kOtSiteTile || q >= t.nq[b] || s >= t.ns[b] ||
                        it.nq_t != std::min<uint32_t>(kOtThreads, t.nq[b] - q) || it.ns_t != std::min<uint32_t>(kOtSiteTile, t.ns[b] - s)) {
                        FAIL("item %u of bucket %u (nq %u, ns %u): queries %u + %u, sites %u + %u are no tile of the bucket\n", item,
                             b, t.nq[b], t.ns[b], q, it.nq_t, s, it.ns_t);
                        continue;
                    }
                    char &mark = seen[(size_t)(q / kOtThreads) * n_st + s / kOtSiteTile];
                    if (mark) FAIL("bucket %u (nq %u, ns %u): tile (%u, %u) twice\n", b, t.nq[b], t.ns[b], q, s);
                    mark = 1;
                    check_copy<4>(it.s0, it.ns_t, n_sites, n_copies);
                    check_copy<8>(it.s0, it.ns_t, n_sites, n_copies);
                }
                for (char m : seen)
                    if (!m) {
                        FAIL("bucket %u (nq %u, ns %u): a tile is not covered\n", b, t.nq[b], t.ns[b]);
                        break;
                    }
            }
        }
    if (!bad && !(residue[0] && residue[1] && residue[2] && residue[3] && first_bucket && last_bucket))
        FAIL("the tables do not reach every residue of a multi-tile bucket and buckets 0 and 65535\n");
    // a bucket of 2^32 - 1 queries and sites: 2^25 x 2^21 items, not a wrapped 32-bit product
    if (ot_bucket_items(0xFFFFFFFFu, 0xFFFFFFFFu) != 1ull << 46 || ot_bucket_items(1, 0xFFFFFFFFu) != 1ull << 25)
        FAIL("ot_bucket_items wraps near 2^32\n");
    // ---------------------------------------------------------------- C
    long n_splits = 0;
    std::vector<uint32_t> visits;
    for (uint32_t nq_t = 1; nq_t <= kOtThreads && bad < 20; ++nq_t)
        for (uint32_t ns_t = 1; ns_t <= kOtSiteTile; ns_t += ns_t < 70 || ns_t > kOtSiteTile - 70 ? 1 : 97) {
            visits.assign((size_t)nq_t * ns_t, 0);
            const uint32_t g = ot_threads_per_query(nq_t);
            for (uint32_t tid = 0; tid < kOtThreads; ++tid) {
                if (!ot_thread_active(tid, nq_t, g)) continue;
                const uint32_t qi = tid % nq_t;
                for (uint32_t s = tid / nq_t; s < ns_t; s += g) ++visits[(size_t)qi * ns_t + s];
            }
            if (g < 1 || nq_t * g > kOtThreads) FAIL("nq_t %u: %u threads per query\n", nq_t, g);
            for (size_t i = 0; i < visits.size(); ++i)
                if (visits[i] != 1) {
                    FAIL("nq_t %u ns_t %u: query %zu, site %zu visited %u times\n", nq_t, ns_t, i / ns_t, i % ns_t, visits[i]);
                    break;
                }
            ++n_splits;
        }
    if (bad) return 1;
    printf("OK %ld tables, %ld buckets with items, %ld items, %ld copies, %ld thread splits\n", n_tables, n_targets, n_items,
           n_copies, n_splits);
    return 0;
}
