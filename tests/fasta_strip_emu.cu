// TEST INFRASTRUCTURE: the device FASTA ingest (k_fasta_strip) run on the CPU from the SAME source.
//
// scan.cuh gives the body of one k_fasta_strip item (fasta_strip_group, __host__ __device__) and the host's
// base count of a record (fasta_record_bases, what crp_genome_add_fasta_record derives n_bases from).  This
// program lays records out as commit_enqueue does (raw_off and ascii_off rounded to 16 bytes, first_item the
// 16-byte groups before the record), finds each item's record with the kernel's binary search, runs the group
// function on every item and compares with a byte-by-byte reading written without the kernel's arithmetic:
//   a record is PLAIN for a width w when it splits on '\n' into lines of exactly w bytes, then a last line of
//   1 .. w bytes and an optional final '\n', and every other byte is in 0x21 .. 0x7E and is none of ' " \ >;
//   its token is ' + the bases + ') -- then , or, for the file's last record, ].
// Asserted: accepted <=> every record plain, and accepted => every token equal to the reading, over
//   A  clean records: widths 1 .. 130 and 4095 .. 4097, every token length mod 16, last line full or partial,
//      with and without the final '\n';
//   B  every line end replaced by A N a, blank, tab, ' " \, 0x7F, 0x80, and moved one byte left or right;
//   C  base slots -- the first and last base of the record and of every 16-byte group -- replaced by bad bytes
//      (blank, tab, ' " \ >, 0x7F, 0x80, 0xFF, 0x00, '\n') and by the printable edges ! and ~;
//   D  buffers of 1 to 300 records of mixed widths and lengths, 1-base records among them, clean and with
//      one defect in one record.
// Raw padding between records is 0x00: a read outside its record makes a plain record refused.
// Built and run by tests/test_fasta_ingest.py (nvcc, no GPU needed).  Nothing here is part of the library.
// Usage: fasta_strip_emu [-a]     -a: report every failing case, not only the first
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

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

struct Rec {
    std::vector<uint8_t> bytes;   // the sequence bytes of the record, as in the file
    uint32_t width;
    bool last;
};

// ---------------------------------------------------------------- the reading
static bool bad_byte(uint8_t c) { return c < 0x21 || c > 0x7E || c == '\'' || c == '"' || c == '\\' || c == '>'; }

static bool reading(const Rec &r, std::string &tok) {
    const std::vector<uint8_t> &s = r.bytes;
    std::vector<size_t> starts, ends;             // lines, split on '\n'
    size_t at = 0;
    for (size_t i = 0; i < s.size(); ++i)
        if (s[i] == '\n') starts.push_back(at), ends.push_back(i), at = i + 1;
    if (at < s.size()) starts.push_back(at), ends.push_back(s.size());   // a last line without its '\n'
    if (starts.empty()) return false;
    tok = "'";
    for (size_t j = 0; j < starts.size(); ++j) {
        const size_t len = ends[j] - starts[j];
        if (j + 1 < starts.size() ? len != r.width : (len < 1 || len > r.width)) return false;
        for (size_t i = starts[j]; i < ends[j]; ++i) {
            if (bad_byte(s[i])) return false;
            tok += (char)s[i];
        }
    }
    tok += r.last ? "')]" : "'),";
    return true;
}

// ---------------------------------------------------------------- the device path, on the CPU
// crp_genome_add_fasta_record's checks, commit_enqueue's layout, then every item of k_fasta_strip.
static bool device(const std::vector<Rec> &recs, std::vector<std::string> &toks) {
    std::vector<FastaRec> fr;
    uint64_t raw_total = 0, ascii_total = 0, items = 0;
    for (const Rec &r : recs) {
        if (r.bytes.empty() || !r.width) return false;
        const uint64_t n_bases = fasta_record_bases(r.bytes.size(), r.bytes.back(), r.width);
        if (!n_bases) return false;
        FastaRec f{};
        f.raw_off = raw_total;
        f.ascii_off = ascii_total;
        f.first_item = items;
        f.n_bases = (uint32_t)n_bases;
        f.width = r.width;
        f.last = r.last ? 1u : 0u;
        fr.push_back(f);
        const uint64_t L = n_bases + 4;
        raw_total += (r.bytes.size() + 15) / 16 * 16;
        ascii_total += (L + 15) / 16 * 16;
        items += (L + 15) / 16;
    }
    std::vector<uint8_t> raw(raw_total + 64, 0), ascii(ascii_total + 64, 0xEE);
    for (size_t i = 0; i < recs.size(); ++i) memcpy(raw.data() + fr[i].raw_off, recs[i].bytes.data(), recs[i].bytes.size());
    const uint32_t n_recs = (uint32_t)fr.size();
    unsigned int bad = 0;
    for (uint64_t it = 0; it < items; ++it) {
        uint32_t lo = 0, hi = n_recs;             // the kernel's search: last record with first_item <= it
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (fr[mid].first_item <= it) lo = mid;
            else hi = mid;
        }
        const FastaRec r = fr[lo];
        const uint64_t p0 = (it - r.first_item) * 16;
        uint32_t w[4] = {0, 0, 0, 0};
        bad |= fasta_strip_group(raw.data(), r, p0, w);
        for (int i = 0; i < 16; ++i) ascii[r.ascii_off + p0 + i] = (uint8_t)(w[i >> 2] >> (8 * (i & 3)));
    }
    toks.clear();
    for (const FastaRec &f : fr) toks.emplace_back((const char *)ascii.data() + f.ascii_off, (size_t)f.n_bases + 4);
    return !bad;
}

// ---------------------------------------------------------------- cases
static bool all_failures = false;
static long n_cases = 0, n_accepted = 0, n_failed = 0;

// false on a mismatch (and then the case is printed)
static bool check(const std::vector<Rec> &recs, const char *what) {
    ++n_cases;
    bool plain = true;
    std::vector<std::string> want(recs.size()), got;
    for (size_t i = 0; i < recs.size() && plain; ++i) plain = reading(recs[i], want[i]);
    const bool accepted = device(recs, got);
    n_accepted += accepted;
    size_t diff = recs.size();
    if (accepted && plain)
        for (size_t i = 0; i < recs.size() && diff == recs.size(); ++i)
            if (got[i] != want[i]) diff = i;
    if (accepted == plain && diff == recs.size()) return true;
    ++n_failed;
    printf("FAIL %s: %zu record(s), plain %d, accepted %d", what, recs.size(), (int)plain, (int)accepted);
    if (diff < recs.size()) {
        size_t k = 0;
        while (k < got[diff].size() && k < want[diff].size() && got[diff][k] == want[diff][k]) ++k;
        printf(", record %zu (width %u): token of %zu bytes, reading %zu, first difference at %zu", diff, recs[diff].width,
               got[diff].size(), want[diff].size(), k);
    }
    printf("\n");
    return all_failures;
}

static uint8_t base() {                            // mostly bases, sometimes any byte a plain record may hold
    static const char acgt[] = "ACGTACGTACGTacgtNn";
    const unsigned long long r = rnd();
    if (r % 16) return (uint8_t)acgt[(r >> 8) % (sizeof acgt - 1)];
    uint8_t c;
    do c = (uint8_t)(0x21 + (rnd() % 94)); while (bad_byte(c));
    return c;
}

// a plain record of n bases in lines of width w
static Rec plain_record(uint64_t n, uint32_t w, bool final_nl, bool last) {
    Rec r;
    r.width = w, r.last = last;
    for (uint64_t i = 0; i < n; ++i) {
        if (i && i % w == 0) r.bytes.push_back('\n');
        r.bytes.push_back(base());
    }
    if (final_nl) r.bytes.push_back('\n');
    return r;
}

static size_t slot_of_base(uint64_t i, uint32_t w) { return (size_t)(i + i / w); }   // byte offset of base i

int main(int argc, char **argv) {
    all_failures = argc > 1 && !strcmp(argv[1], "-a");
    std::vector<uint32_t> widths;
    for (uint32_t w = 1; w <= 130; ++w) widths.push_back(w);
    for (uint32_t w = 4095; w <= 4097; ++w) widths.push_back(w);
    static const uint8_t slot_bytes[] = {'A', 'N', 'a', ' ', '\t', '\'', '"', '\\', 0x7F, 0x80};
    static const uint8_t base_bytes[] = {' ', '\t', '\'', '"', '\\', '>', 0x7F, 0x80, 0xFF, 0x00, '\n', '!', '~'};
    char what[160];
    long n_a = 0, n_b = 0, n_c = 0, n_d = 0;
    for (uint32_t w : widths) {
        // enough lines that the line ends fall on every residue mod 16 of the base index (33 line ends at
        // most widths, 17 at the widest)
        const uint64_t lines = w > 1000 ? 18 : 34;
        // ---- A: every token length mod 16 (n = lines * w - d), last line full or partial, final '\n' or not
        for (uint64_t d = 0; d < 16; ++d)
            for (int nl = 0; nl < 2; ++nl) {
                const uint64_t n = lines * w > d ? lines * w - d : 1;
                snprintf(what, sizeof what, "A width %u bases %llu final newline %d", w, (unsigned long long)n, nl);
                if (!check({plain_record(n, w, nl, nl)}, what)) return 1;
                ++n_a;
            }
        // ---- B: every line end, the final one included, replaced or moved
        const uint64_t n = lines * w + (w + 1) / 2;     // last line partial (full for width 1)
        const Rec clean = plain_record(n, w, true, true);
        for (uint64_t j = 1; j <= (n - 1) / w + 1; ++j) {             // the line end after line j
            const size_t slot = j * w <= n - 1 ? slot_of_base(j * w, w) - 1 : clean.bytes.size() - 1;
            for (uint8_t c : slot_bytes) {
                Rec r = clean;
                r.bytes[slot] = c;
                snprintf(what, sizeof what, "B width %u line end before base %llu replaced by 0x%02x", w, (unsigned long long)(j * w), c);
                if (!check({r}, what)) return 1;
                ++n_b;
            }
            for (int dir = -1; dir <= 1; dir += 2) {
                if (slot + dir >= clean.bytes.size()) continue;
                Rec r = clean;
                std::swap(r.bytes[slot], r.bytes[slot + dir]);
                snprintf(what, sizeof what, "B width %u line end before base %llu moved %+d", w, (unsigned long long)(j * w), dir);
                if (!check({r}, what)) return 1;
                ++n_b;
            }
        }
        // ---- C: the first and last base of the record and of every group (bases 16 g - 1 and 16 g + 14), on
        // the record of B without its final '\n'; every group at widths up to 64, else the groups at the
        // record's ends and those that hold or follow a line end
        Rec bare = clean;
        bare.bytes.pop_back();
        std::vector<uint64_t> slots = {0, n - 1};
        for (uint64_t g = 0; 16 * g <= n; ++g) {
            const uint64_t first = g ? 16 * g - 1 : 0, end = 16 * g + 15 < n ? 16 * g + 15 : n;   // bases [first, end)
            const bool edge = w <= 64 || g < 2 || end + 32 > n || first / w != (end - 1) / w || first % w == 0;
            if (!edge) continue;
            slots.push_back(first);
            slots.push_back(end - 1);
        }
        for (uint64_t i : slots)
            for (uint8_t c : base_bytes) {
                Rec r = bare;
                r.bytes[slot_of_base(i, w)] = c;
                snprintf(what, sizeof what, "C width %u base %llu of %llu replaced by 0x%02x", w, (unsigned long long)i, (unsigned long long)n, c);
                if (!check({r}, what)) return 1;
                ++n_c;
            }
    }
    // ---- D: buffers of several records, clean and with one defect
    long n_records_d = 0;
    static const int first_sizes[] = {1, 2, 300};
    for (int round = 0; round < 160; ++round) {
        const int n_recs = round < 3 ? first_sizes[round] : 1 + (int)(rnd() % 300);
        std::vector<Rec> recs;
        for (int k = 0; k < n_recs; ++k) {
            const unsigned long long r = rnd();
            const uint32_t w = r % 7 == 0 ? 1 + (uint32_t)(rnd() % 3) : r % 11 == 0 ? 4095 + (uint32_t)(rnd() % 3) : 1 + (uint32_t)(rnd() % 130);
            const uint64_t n = r % 5 == 0 ? 1 : 1 + rnd() % (r % 3 == 0 ? 40ull : 4ull * w + 40);
            recs.push_back(plain_record(n, w, (r >> 20) & 1, k == n_recs - 1));
        }
        n_records_d += n_recs;
        snprintf(what, sizeof what, "D round %d: %d clean records", round, n_recs);
        if (!check(recs, what)) return 1;
        const int k = (int)(rnd() % n_recs);
        Rec &r = recs[k];
        const size_t slot = (size_t)(rnd() % r.bytes.size());
        const uint8_t was = r.bytes[slot];
        r.bytes[slot] = was == '\n' ? slot_bytes[rnd() % sizeof slot_bytes] : base_bytes[rnd() % 11];
        snprintf(what, sizeof what, "D round %d: %d records, record %d (width %u) byte %zu 0x%02x -> 0x%02x", round, n_recs, k, r.width,
                 slot, was, r.bytes[slot]);
        if (!check(recs, what)) return 1;
        n_d += 2;
    }
    if (n_failed) {
        printf("%ld of %ld cases failed\n", n_failed, n_cases);
        return 1;
    }
    if (n_accepted == 0 || n_accepted == n_cases) {
        printf("FAIL: the cases do not hold both accepted and refused buffers\n");
        return 1;
    }
    printf("OK %ld cases (%ld accepted): %ld clean records at %zu widths, %ld line-end defects, %ld base defects, %ld buffers of %ld records\n",
           n_cases, n_accepted, n_a, widths.size(), n_b, n_c, n_d, n_records_d);
    return 0;
}
