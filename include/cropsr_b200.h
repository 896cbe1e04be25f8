/*
 * cropsr_b200.h -- C ABI of libcropsr_b200.so: the B200 (sm_100a) implementation
 * of CROPSR's genome-wide Cas9 gRNA candidate scan + Rule-Set-1 scoring.
 *
 * The reference (H2muller/CROPSR) has no FFI: its hot path is Python inside
 * CROPSR.py main().  Each entry point below names the reference code it
 * replaces (paths relative to /root/reference).  The Python host
 * (cropsr_b200/) binds these with ctypes; INTEGRATION.md shows the binding a
 * maintainer would add to the reference's own CROPSR.py.
 *
 * Conventions: every function returns 0 on success or a negative crp_status;
 * crp_last_error() gives the message for the calling thread.  Device memory is
 * owned by the opaque handles; host output buffers are caller-allocated.  All
 * calls are synchronous with respect to the host unless stated.  One process
 * drives one GPU (crp_init picks it); multi-GPU runs use one process per GPU.
 * There is no CPU fallback: without a usable CUDA device every compute entry
 * point fails with CRP_ERR_CUDA.
 */
#ifndef CROPSR_B200_H
#define CROPSR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum crp_status {
    CRP_OK = 0,
    CRP_ERR_CUDA = -1,      /* CUDA runtime/driver error (message has the detail) */
    CRP_ERR_ARG = -2,       /* bad argument                                        */
    CRP_ERR_STATE = -3,     /* call out of order (e.g. scan before commit)         */
    CRP_ERR_NOMEM = -4,     /* host or device allocation failed                    */
    CRP_ERR_RANGE = -5,     /* token/segment too large for the 31-bit position     */
    CRP_ERR_FORMAT = -6     /* FASTA bytes are not plain fixed-width records: use the host ingest */
} crp_status;

typedef struct crp_genome crp_genome;   /* packed genome shard resident in HBM     */
typedef struct crp_result crp_result;   /* compacted candidate streams in HBM      */

/* ---- scan flags --------------------------------------------------------- */
#define CRP_SCAN_DEFAULT     0u
#define CRP_SCAN_NO_SCORE    1u   /* positions only (forced when guide_len != 20)  */
#define CRP_SCAN_LOGISTIC    2u   /* store 1/(1+np.exp(x)) instead of x (see below) */
#define CRP_SCAN_EXTRAS      4u   /* also compute the opt-in per-candidate extras  */

/* ---- summation classes for crp_rescore (SURVEY.md 8c) -------------------- */
#define CRP_CLASS_CANONICAL  0    /* 4 lanes by column mod 4, (p0+p2)+(p1+p3)      */
#define CRP_CLASS_PAIR       1    /* 2 lanes by column mod 2, q0+q1                */
#define CRP_CLASS_SINGLE     2    /* n==1 np.matmul -> ddot lane order             */

/* ---- packed 30-mer layout (one uint64 per candidate) --------------------
 * The scored 30-mer in output order q = 0..29 (the order of the CSV
 * long_sequence column), 2 bits per base, PLANAR, code A0 T1 C2 G3
 * (reference CROPSR.py:300-302):
 *   bits  0..29  low  code bit of base q        bit 30  window has a byte that is
 *   bits 32..61  high code bit of base q                not uppercase ACGT
 *   bit 31  window truncated at the token end (reference emits an 11-field
 *           "error row" with score -1, CROPSR.py:466-468)
 *   bit 62  some base contributes nothing to the score (N, IUPAC, quote, ...)
 *   bit 63  reserved (0)
 */
#define CRP_PACKED_IRREGULAR  (1ull << 30)
#define CRP_PACKED_TRUNCATED  (1ull << 31)
#define CRP_PACKED_UNSCORED   (1ull << 62)

/* ---- library / device ---------------------------------------------------- */

/* Select the CUDA device this process drives and create the library's stream. */
int crp_init(int device);
int crp_shutdown(void);
const char *crp_last_error(void);
int crp_device_count(int *count);
/* ABI version of this header (bumped on any signature change). */
int crp_abi_version(void);
/* Positions per scan tile: segment boundaries chosen by the host should be
 * multiples of this (any multiple of 128 is accepted). */
int crp_tile_size(void);
/* 1 for the self-checking build (make -C cropsr_b200/csrc checked: libcropsr_b200_checked.so):
 * k_scan_score verifies its own index and ordering invariants and a violated one fails the scan
 * with CRP_ERR_STATE naming it.  Slower; for tests (compute-sanitizer is not available everywhere). */
int crp_checked_build(void);

/* Wait for everything this library has queued on the device. */
int crp_device_synchronize(void);
/* Evict the L2 cache (a 512 MiB memset on the library stream, waited for): benchmarks call it
 * between timed scans so that no scan finds its tile records in L2. */
int crp_flush_l2(void);

/* ---- several GPUs: one process per GPU, one NCCL communicator ---------------
 * The reference scans its chromosomes one after the other in one Python loop
 * (CROPSR.py:409); here the genome is cut into contiguous, tile-aligned shards
 * (cropsr_b200/shard.py), every process scans its own shard, and the only exchange is an
 * all-gather of the per-segment candidate counts, from which every rank derives where its rows
 * sit in the reference's order (token by token, '+' then '-').  The launcher creates the id on
 * rank 0 (crp_comm_unique_id), hands the 128 bytes to every rank by whatever channel it has
 * (cropsr_b200/launch.py: a TCP rendezvous on MASTER_ADDR:MASTER_PORT), and every rank calls
 * crp_comm_init after crp_init.  NCCL is loaded with dlopen("libnccl.so.2") on first use: a
 * single-GPU process never needs it. */
#define CRP_COMM_ID_BYTES 128
int crp_comm_unique_id(uint8_t *id /* [CRP_COMM_ID_BYTES] */);
int crp_comm_init(int rank, int world, const uint8_t *id);
int crp_comm_info(int *rank, int *world);           /* 0 / 1 without a communicator */
/* Exchange of crp_scan_score_sharded: 0 = fused into the kernel when possible (default), 1 = NCCL
 * all-gather.  Set it on every rank.  crp_comm_exchange_info says what a sharded scan will do. */
int crp_comm_set_exchange(int mode);
int crp_comm_exchange_info(int *fused, const char **why);
/* Device-wide synchronize, then an all-reduce of one word over all ranks, waited for. */
int crp_comm_barrier(void);
/* Element-wise max / sum of n host doubles over all ranks, in place (timings, totals). */
int crp_comm_max_f64(double *v, uint32_t n);
int crp_comm_sum_f64(double *v, uint32_t n);
/* All-gather of n host words per rank, host in / host out: out[rank * n + i]. */
int crp_comm_allgather_u64(const uint64_t *in, uint32_t n, uint64_t *out);
int crp_comm_shutdown(void);
/* Link probe (benchmarks): h2d_bytes up and d2h_bytes down, pinned, both directions at once,
 * `reps` rounds; *ms = mean wall time of a round. */
int crp_link_probe(uint64_t h2d_bytes, uint64_t d2h_bytes, uint32_t reps, float *ms);

/* Pinned host memory for staging (FASTA bytes in, candidate arrays out). */
int crp_host_alloc(void **ptr, uint64_t bytes);
int crp_host_free(void *ptr);

/* ---- ingest: replaces the per-token Python strings of the ingest dict -----
 * (CROPSR.py:54-74 import_fasta_file; the values of the dict built by
 * cropsr_functions.py:190-196 generate_dictionary).  A *token* is one dict
 * value, decoration bytes of the formatted path included.  A *segment* is the
 * part [seg_begin, seg_end) of a token whose PAM positions this GPU owns; the
 * library stages the halo it needs from the token itself.
 */
int crp_genome_new(crp_genome **g);
/* token_ascii points at position 0 of the whole token in host memory and must
 * stay valid until crp_genome_commit returns.  seg_begin must be a multiple of
 * 128 (0 for a whole token).  Segments are scanned in the order added. */
int crp_genome_add_segment(crp_genome *g, uint32_t token_id,
                           const uint8_t *token_ascii, uint64_t token_len,
                           uint64_t seg_begin, uint64_t seg_end);
/* Device-side ingest of one record of a multi-line FASTA file -- replaces, for that record,
 * the text pipeline of CROPSR.py:54-74 (import_fasta_file) and cropsr_functions.py:221-229
 * (formatted: split on '>', drop the line ends, str() of the list of tuples): the file's own
 * bytes go to the device, a kernel drops the line ends and adds the decoration that the
 * reference's repr round trip leaves around every sequence ("'" + bases + "')," -- "')]" for
 * the last record of the file), and the pack kernel reads the result.  seq_bytes points at the
 * first byte after the header line, n_bytes runs to the next '>' or the end of the file, and
 * line_width is the length of the first sequence line.  Only "plain" records qualify: every
 * line line_width bases long except the last, '\n' line ends, printable non-blank ASCII, no
 * quotes, backslashes or '>' -- text that str()/split() leave untouched.  Anything else makes
 * this call or crp_genome_commit return CRP_ERR_FORMAT, and the caller ingests the file the
 * literal way (cropsr_b200/ingest.py).  The bytes must stay valid until crp_genome_commit
 * returns.  The whole token is one segment. */
int crp_genome_add_fasta_record(crp_genome *g, uint32_t token_id, const uint8_t *seq_bytes, uint64_t n_bytes,
                                uint32_t line_width, int last_record);
/* Length of the token of a segment, and -- for records ingested by the call above -- its
 * bytes (the rows of the CSV are formatted from them on the host; CROPSR.py:463-469).  The
 * device copy of the tokens is dropped by crp_genome_release_tokens / crp_genome_free. */
int crp_genome_token_length(const crp_genome *g, uint32_t segment, uint64_t *token_len);
int crp_genome_fetch_token(const crp_genome *g, uint32_t segment, uint8_t *dst, uint64_t capacity);
int crp_genome_release_tokens(crp_genome *g);
/* H2D copy + pack kernel: ASCII -> 2-bit code planes + lower-case plane +
 * other-byte plane (0.5 byte per base resident in HBM). */
int crp_genome_commit(crp_genome *g);
int crp_genome_num_segments(const crp_genome *g, uint32_t *n);
int crp_genome_num_positions(const crp_genome *g, uint64_t *n);   /* sum of segment lengths */
int crp_genome_free(crp_genome *g);

/* ---- scan + score: replaces CROPSR.py:413-434 (regex PAM scan, bounds,
 * window slicing, gRNA / reverse-complement transforms) and CROPSR.py:285-313
 * (rs1_score) for every segment of the genome in one launch sequence.
 * Output per strand is ONE ordered stream over (segment order, ascending t):
 *   pos     uint32  t, the regex match position inside the token
 *   packed  uint64  see layout above               (guide_len == 20 only)
 *   x       float64 pre-activation -(((A+B)+0.59763615)+(-0.2026259)) summed
 *                   in the canonical lane order; the reference's score is
 *                   1/(1+np.exp(x)) (CROPSR.py:312-313).  With
 *                   CRP_SCAN_LOGISTIC the stored value is that score itself, with
 *                   numpy's digits (see crp_logistic).
 * Reference order of a token's candidates = its '+' stream then its '-' stream
 * (CROPSR.py:417-434).
 */
int crp_scan_score(crp_genome *g, int guide_len, uint32_t flags, crp_result **res);
/* The same scan on one shard of a genome that is spread over the ranks of crp_comm_init: the
 * kernel writes this shard's per-segment counts as a block of 2 * slots words
 * {plus[0..slots), minus[0..slots)} (slots >= the segments of every rank; unused slots are 0),
 * and every rank ends up with the blocks of all ranks -- the one exchange step of the path.
 *   fused exchange (default when every rank could map its peers' buffers through CUDA IPC):
 *     the kernel itself stores its block into every rank's gather buffer over NVLink as soon as
 *     its count phase is through, raises a flag there, and returns once all blocks have landed
 *     in its own buffer: the all-gather rides behind the emit phase and costs no launch;
 *   NCCL exchange (crp_comm_set_exchange(1), CRP_COMM_EXCHANGE=nccl, or no peer mapping):
 *     an ncclAllGather on the same stream, right behind the kernel.
 * crp_result_timing reports kernel + exchange either way, crp_result_timing_detail the kernel
 * alone as well.  Collective: every rank must call it, with the same slots. */
int crp_scan_score_sharded(crp_genome *g, int guide_len, uint32_t flags, uint32_t slots, crp_result **res);
/* counts[(rank * 2 + strand) * slots + segment] of the scan above, strand 0 = '+'. */
int crp_result_gathered_counts(const crp_result *res, uint64_t *counts /* [world][2][slots] */);
int crp_result_totals(const crp_result *res, uint64_t *n_plus, uint64_t *n_minus);
/* Per-segment candidate counts, arrays of crp_genome_num_segments() entries. */
int crp_result_segment_counts(const crp_result *res, uint64_t *n_plus, uint64_t *n_minus);
/* Device pointer to uint64[2*num_segments] {plus[0..n), minus[0..n)} for the
 * NCCL all-gather of per-shard counts (global offsets across GPUs). */
int crp_result_device_counts(const crp_result *res, void **dev_ptr);
/* Copy candidates [first, first+count) of one strand stream ('+' or '-') to
 * caller-allocated host arrays; any output pointer may be NULL. */
int crp_result_fetch(const crp_result *res, char strand, uint64_t first, uint64_t count,
                     uint32_t *pos, uint64_t *packed, double *x);
int crp_result_free(crp_result *res);

/* ---- whole call from host memory, pipelined -------------------------------
 * The same work as add_segment/commit/scan_score/fetch, one segment after the
 * other, but overlapped: segment k+1 is copied in and packed while segment k is
 * scanned and segment k-1 is copied out (three streams; PCIe in both directions
 * at once).  Tokens and arenas should be pinned (crp_host_alloc).  Rows of a
 * strand land in its arena in segment order; n_plus / n_minus [n_segments]
 * receive the per-segment counts.  Returns CRP_ERR_RANGE if an arena of
 * `capacity` rows per strand is too small (the counts are still filled in).
 * packed / x arenas may be NULL (and are ignored when guide_len != 20).
 * ms_device (optional) receives the summed device time of the scan kernels.
 * [begin, end) is taken as given, exactly as by crp_genome_add_segment: there is
 * no sentinel, so end = 0 (or end = begin) owns no position.  Every descriptor is
 * checked before any device work: begin <= end <= token_len, begin % 128 == 0,
 * token non-NULL when token_len > 0, token_len below 2^31 - 2^15.  A violation
 * returns CRP_ERR_ARG with n_plus / n_minus zeroed. */
typedef struct crp_segment_desc {
    uint32_t token_id;
    const uint8_t *token;       /* position 0 of the whole token */
    uint64_t token_len;
    uint64_t begin, end;        /* positions [begin, end) of the token this call owns */
} crp_segment_desc;
int crp_scan_segments(uint32_t n_segments, const crp_segment_desc *segments, int guide_len, uint32_t flags,
                      uint64_t capacity, uint32_t *pos_plus, uint64_t *packed_plus, double *x_plus,
                      uint32_t *pos_minus, uint64_t *packed_minus, double *x_minus,
                      uint64_t *n_plus, uint64_t *n_minus, float *ms_device);

/* Re-evaluate x for selected candidates in a given BLAS summation class
 * (rows of an np.matmul call that OpenBLAS sums in a different lane order:
 * the tail rows of each emitted slice, SURVEY.md 8c).  Items are identified by
 * (segment index, t, strand).  cls[i] = class of the first-order product
 * (matrix1 @ first_matrix, CROPSR.py:305) | class of the dinucleotide product
 * (matrix2 @ second_matrix, CROPSR.py:311) << 4. */
int crp_rescore(const crp_genome *g, uint64_t n, const uint32_t *segment, const uint32_t *t,
                const char *strand, const uint8_t *cls, double *x_out);

/* ---- opt-in side outputs (never part of the reference CSV: the reference parses
 * -L and -g and does not use them, CROPSR.py:41,375) -------------------------
 * Per candidate of one segment and strand, in stream order; any pointer may be
 * NULL.  guide_len 20 only.
 *   gc        G+C count of the 20-base protospacer (scored 30-mer[5:25]; the
 *             reference's only hint: cropsr_functions.py:174-179)
 *   flags     bit0 TTTT in the protospacer, bit1 homopolymer run >= 5,
 *             bit2 gc < 10, bit3 protospacer holds a base that does not score
 *   run       longest homopolymer run in the protospacer
 *   cut       cut site = end_pos - 3 of the CSV row (CROPSR.py:155-158)
 *   flank_lo/hi  [cut - flank, cut + flank) clipped to the token (the -L window
 *             meant for prmrdsgn2 primer design) */
int crp_result_extras(const crp_result *res, uint32_t segment, char strand, uint32_t flank,
                      uint8_t *gc, uint8_t *flags, uint8_t *run,
                      uint32_t *cut, uint32_t *flank_lo, uint32_t *flank_hi);
/* The same for every segment of one strand stream in one call (arrays of crp_result_totals()
 * entries, stream order): one launch per segment queued back to back, one copy per array, one wait. */
int crp_result_extras_strand(const crp_result *res, char strand, uint32_t flank,
                             uint8_t *gc, uint8_t *flags, uint8_t *run,
                             uint32_t *cut, uint32_t *flank_lo, uint32_t *flank_hi);
/* Gap table of one segment (SURVEY.md 8f.2, opt-in; the reference has nothing like it): maximal runs of
 * bytes that are not A C G T a c g t -- N, IUPAC codes, anything else; the quote / paren decoration of a
 * formatted-path token is such a run too -- at least min_len long, read off the packed records on the
 * device: start[i] (token coordinate) and length[i], ascending.  *n_runs receives the number of runs;
 * CRP_ERR_RANGE if it exceeds `capacity` (call again with more room). */
int crp_genome_other_runs(const crp_genome *g, uint32_t segment, uint32_t min_len, uint64_t capacity,
                          uint32_t *start, uint32_t *length, uint64_t *n_runs);
/* feature[i] = index of the innermost interval [start, end] (inclusive, token
 * coordinates, sorted by start) that contains candidate i's cut site, or -1:
 * a binary search per candidate in device memory. */
int crp_result_annotate(const crp_result *res, uint32_t segment, char strand, uint32_t n_intervals,
                        const uint32_t *start, const uint32_t *end, int32_t *feature);

/* The same for a whole strand stream: the intervals of segment s are [iv_offset[s], iv_offset[s+1])
 * of start / end (iv_offset has num_segments + 1 entries); feature[i] indexes its segment's run. */
int crp_result_annotate_strand(const crp_result *res, char strand, const uint64_t *iv_offset,
                               const uint32_t *start, const uint32_t *end, int32_t *feature);

/* crispr_id characters: replaces get_id() (CROPSR.py:316-318: np.random.choice of 36 characters,
 * [n, 7]) value for value on numpy's legacy MT19937 generator -- the caller passes the state of
 * np.random.get_state() (key[624], pos) and stores the advanced state back, so that a seeded run
 * reproduces the reference's ids and every later draw.  out receives 7 ASCII bytes per id.
 * Host only, no GPU involved. */
int crp_legacy_ids(uint32_t *mt_key, int32_t *mt_pos, uint64_t n_ids, uint8_t *out);

/* ---- primer enumeration over windows of a packed genome (opt-in; SURVEY.md 8f.4).
 * Replaces the part of /root/reference/prmrdsgn2.py that needs no aligner, for many fragments at
 * once: get_primers (:115-124) on the fragment and on its reverse complement (:104-112), the
 * Primer GC % / Tm (:76-95), filter_primers (:127-137) and the Tm pairing of main() (:260-266).
 * The fields of crp_primer_params are the reference's CLI flags -e -s -l -m -x -M -X -D (:26-54).
 * Window i is token positions [lo[i], hi[i]) of segment[i] (inside the positions that segment
 * owns), e.g. the flank_lo / flank_hi of crp_result_extras.  Per window:
 *   n_fwd / n_rev   primers that pass the GC / Tm filter, forward and reverse-complement side
 *   n_pairs         pairs of itertools.product(forward, reverse) with math.isclose(Tm, Tm, abs_tol=D)
 *   first[4 i ..]   the first such pair in the reference's order: forward (start, length),
 *                   reverse (start on the reverse complement, length); 0xFFFF x 4 if there is none
 *   status          0, or 1 if the window is shorter than e + l bases (the reference would slice
 *                   short or empty primers there; such windows are reported, not designed)
 * Limits: 12 <= s < l <= 32 (so every primer has >= 13 bases: one Tm formula), e + l <= 1024.
 * Any output pointer may be NULL. */
typedef struct crp_primer_params {
    uint32_t e, s, l;           /* -e extension, -s shortest, -l longest                   */
    double m, x;                /* -m / -x  min / max Tm                                   */
    double M, X;                /* -M / -X  min / max GC percentage                        */
    double D;                   /* -D accepted Tm difference of a pair                     */
} crp_primer_params;
int crp_primer_windows(const crp_genome *g, uint64_t n, const uint32_t *segment, const uint32_t *lo,
                       const uint32_t *hi, const crp_primer_params *params, uint32_t *n_fwd, uint32_t *n_rev,
                       uint64_t *n_pairs, uint16_t *first, uint8_t *status);

/* ---- host-side row formatter: replaces the per-row tuple + csv.writer path of
 * CROPSR.py:463-474.  Writes n_rows CSV rows (excel dialect, "\r\n", repr() floats,
 * the 11-field error-row variant where scored[i] == 0) into `out`, byte-identical
 * to the reference's writer; multi-threaded, no GPU involved.  Row i is the
 * candidate (token_of[i], t[i], minus[i]) with id ids[7 * id_index[i] .. +7).
 * Returns CRP_ERR_RANGE (and the size needed in *out_bytes) if out is too small.
 * Rows are formatted into a scratch buffer the library keeps between calls (sized for the worst
 * row of the largest call so far): one call at a time per process. */
int crp_format_rows(uint64_t n_rows, const char *ids, const uint64_t *id_index, const uint32_t *token_of,
                    const uint32_t *t, const uint8_t *minus, const uint8_t *scored, const double *score,
                    uint32_t n_tokens, const uint8_t *const *tokens, const uint64_t *token_len,
                    const char *const *chrom, const uint32_t *chrom_len, int guide_len, int n_threads,
                    char *out, uint64_t out_capacity, uint64_t *out_bytes);

/* ---- the reference's logistic, CROPSR.py:313: score = 1 / (1 + np.exp(x)).  numpy's float64
 * exp on an AVX-512 host is the vendored SVML routine __svml_exp8_ha; the device evaluates a
 * restatement of it (csrc/npexp.cuh), so for |x| < 707.7 the result has numpy's digits, not
 * libm's.  Host arrays in and out.  The same function is applied in place to the x streams of a
 * scan started with CRP_SCAN_LOGISTIC. */
int crp_logistic(uint64_t n, const double *x, double *score);

/* rs1_score(sequences) itself (CROPSR.py:285-313) on the reference's own argument: n rows of 30
 * ASCII bytes, row-major (only 'A' 'T' 'C' 'G' score, everything else contributes 0,
 * CROPSR.py:300-302).  cls[i] = BLAS lane class of row i in the two np.matmul calls
 * (CRP_CLASS_* of the first-order call | class of the second-order call << 4; which rows of an
 * n-row call are not canonical is index logic, cropsr_b200/blas_order.py).  score[i] is the
 * reference's return value, logistic included. */
int crp_rs1_score(uint64_t n, const uint8_t *rows, const uint8_t *cls, double *score);
/* The same without the logistic: x[i] = -(((A+B)+0.59763615)+(-0.2026259)) of row i in class cls[i]
 * (a host that holds the tokens re-sums the few non-canonical rows of a slice without a genome handle). */
int crp_rs1_preactivation(uint64_t n, const uint8_t *rows, const uint8_t *cls, double *x);

/* ---- off-target counts (opt-in; the reference has none: its nearest relative is the bowtie2 call of
 * /root/reference/prmrdsgn2.py:139-160, which aligns primers with an external aligner).  An index holds the
 * 40-bit protospacer keys of every NGG site, both strands, case-insensitive, of every genome handle added
 * to it; the counts of a query are the numbers of sites at exactly d = 0 .. max_mm mismatches (max_mm <= 3),
 * found by exact pigeonhole filtering on the device.  Semantics in csrc/offtarget.cuh and
 * oracle/offtarget_oracle.py:
 *   site '+' at t   tok[t+1], tok[t+2] in {G, g}, tok[t-20 .. t) all of ACGTacgt; P = tok[t-20 .. t)
 *   site '-' at t   tok[t], tok[t+1] in {C, c}, tok[t+3 .. t+23) all of ACGTacgt; P = revcomp(tok[t+3 .. t+23))
 *   key             base P[i] (code A0 T1 C2 G3, case folded) in bits 2i, 2i+1; P[0] is the PAM-distal base
 * Positions are token coordinates; the index is built on its own stream, ordered behind each genome's. */
typedef struct crp_offtarget crp_offtarget;
int crp_offtarget_new(crp_offtarget **ix);
/* The genome must be committed; its site keys are copied (the genome may be freed afterwards, but a
 * result of it can only be counted while both live).  CRP_ERR_RANGE beyond 2^32 - 1 sites in all. */
int crp_offtarget_add_genome(crp_offtarget *ix, const crp_genome *g);
int crp_offtarget_num_sites(const crp_offtarget *ix, uint64_t *n);
/* All site keys, in no particular order; CRP_ERR_RANGE (and *n) if capacity is too small. */
int crp_offtarget_fetch_sites(const crp_offtarget *ix, uint64_t capacity, uint64_t *keys, uint64_t *n);
/* Counts of every candidate of one strand stream of a scan whose genome was added (CRP_ERR_STATE otherwise,
 * and for guide_len != 20): counts[i * (max_mm + 1) + d], stream order, the candidate's own site not counted.
 * A candidate whose protospacer is cut off by the token end or holds a byte outside ACGTacgt has no
 * counts: max_mm + 1 times 0xFFFFFFFF. */
int crp_offtarget_count_candidates(crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm,
                                   uint32_t *counts /* [n_strand][max_mm + 1] */);
/* The same for arbitrary protospacer keys (< 2^40; user guides in the orientation followed by NGG in the
 * genome); nothing is subtracted. */
int crp_offtarget_count_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, uint32_t max_mm, uint32_t *counts);
/* ---- off-target loci.  An index made by crp_offtarget_new_with_loci also keeps one uint64 LOCUS per site, at
 * the slot of its key (8 more bytes per site of device memory):
 *   bits 0-31   t, token coordinates (the t of the definition above and of a candidate's pam_pos)
 *   bits 32-55  the segment index in its genome handle
 *   bits 56-62  the ordinal of the add_genome call that added the handle (0, 1, ...)
 *   bit 63      strand, 1 = '-'
 * add_genome of such an index answers CRP_ERR_RANGE for a handle of 2^24 segments or more and for a 128th
 * handle.  An index made by crp_offtarget_new behaves as before and keeps no loci. */
int crp_offtarget_new_with_loci(crp_offtarget **ix);
/* ---- other PAMs.  An index made by crp_offtarget_new_pam holds the sites of the PAM pattern `pam` instead of NGG
 * (with loci when with_loci is non-zero): three characters, any case, N followed by two IUPAC letters for one to three
 * bases, A C G T R Y S W K M B D H V (N is refused there).  With S2, S3 the code sets of letters 2 and 3 and
 * comp(S) = {c ^ 1 : c in S}:
 *   site '+' at t   tok[t+1] a base in S2, tok[t+2] a base in S3, tok[t-20 .. t) all of ACGTacgt; P = tok[t-20 .. t)
 *   site '-' at t   tok[t] a base in comp(S3), tok[t+1] a base in comp(S2), tok[t+3 .. t+23) all of ACGTacgt;
 *                   P = revcomp(tok[t+3 .. t+23))
 * Keys, loci and every count, list and score call work on such an index as on an NGG one (crp_offtarget_new and
 * crp_offtarget_new_with_loci are "NGG"), with one rule for scan candidates: their own site is a site of the index
 * exactly when G is in S2 and in S3 (NGG, NRG, NKG, ...), and only then is it subtracted from the counts and the
 * score.  Otherwise a candidate's row starts at 0, as a key's does.  A listing leaves out a site at the candidate's
 * own locus either way.  CRP_ERR_ARG for NULL or a pattern outside this definition. */
int crp_offtarget_new_pam(crp_offtarget **ix, const char *pam, int with_loci);
/* The loci in crp_offtarget_fetch_sites order; CRP_ERR_STATE on an index without loci, CRP_ERR_RANGE (and *n)
 * if capacity is too small. */
int crp_offtarget_fetch_loci(const crp_offtarget *ix, uint64_t capacity, uint64_t *loci, uint64_t *n);
/* LISTING: the sites that the counts of a row count, as site indices (positions in fetch_sites / fetch_loci
 * order).  The caller sizes row i's slice from its counts: first[i + 1] - first[i] = sum of mm_d, d <= max_mm,
 * first[0] = 0; the library writes the row's sites into sites[first[i] .. first[i + 1]) in no particular
 * order and never outside the slice.  If a row finds another number of sites than its slice holds, the call
 * answers CRP_ERR_STATE and nothing is copied to `sites`.  A candidate's own site (same locus) is left out.
 * CRP_ERR_ARG: max_mm > 3, first not starting at 0 or decreasing, rows not ascending and distinct or beyond the
 * stream, a selected row without a protospacer, a key >= 2^40.  CRP_ERR_STATE: an index without loci, a genome
 * not added, guide_len != 20. */
int crp_offtarget_list_candidates(crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm,
                                  uint64_t n_rows, const uint32_t *rows,   /* stream rows, ascending, distinct */
                                  const uint64_t *first,                   /* [n_rows + 1], first[0] = 0 */
                                  uint32_t *sites);                        /* [first[n_rows]] site indices */
int crp_offtarget_list_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, uint32_t max_mm,
                            const uint64_t *first, uint32_t *sites);
/* ---- off-target SCORES: per query the uint64 sum, over the pairs its counts count (NGG sites within d <= max_mm
 * mismatches, the candidate's own site subtracted, nothing subtracted for keys), of weights[rank of the pair's
 * mismatch-position set].  The positions are 0 .. 19 of P (0 = PAM-distal), and the sets of size <= 3 are ranked
 * colexicographically:
 *   rank({}) = 0   rank({a}) = 1 + a   rank({a<b}) = 21 + a + C(b,2)   rank({a<b<c}) = 211 + a + C(b,2) + C(c,3)
 * Entries for sets larger than max_mm are not read; an entry >= 2^31 among the others is CRP_ERR_ARG, so that no sum
 * can overflow.  A candidate without a protospacer gets CRP_OT_NO_SCORE.  The sum does not depend on the order in
 * which pairs are found.  With round(hit * 2^24) of the MIT hit score (Hsu et al. 2013, CRISPOR's calcHitScore) as
 * weights, sum / 2^24 is the MIT hit-score sum over the index's sites (NGG, or its PAM pattern) within max_mm <= 3
 * mismatches -- CRISPOR also sums 4-mismatch sites, so its score is not this one.  Other refusals as for the count
 * calls. */
#define CRP_OT_SCORE_SETS 1351
#define CRP_OT_NO_SCORE 0xFFFFFFFFFFFFFFFFull
int crp_offtarget_score_candidates(crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm,
                                   const uint32_t *weights /* [CRP_OT_SCORE_SETS] */, uint64_t *sums /* [n_strand] */);
int crp_offtarget_score_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, uint32_t max_mm,
                             const uint32_t *weights, uint64_t *sums);
/* ms_sites: device time of every add_genome; ms_count and comparisons (sum over the 10 part pairs and the
 * 65,536 buckets of queries x sites) of the last count, list or score call. */
int crp_offtarget_timing(const crp_offtarget *ix, float *ms_sites, float *ms_count, uint64_t *comparisons);
int crp_offtarget_free(crp_offtarget *ix);

/* Kernel timings (CUDA events on the library stream) of the last commit /
 * scan: milliseconds. */
int crp_genome_timing(const crp_genome *g, float *ms_h2d, float *ms_pack);
/* ms_scan: every launch of the scan (a rerun after a capacity overflow included) and, for a
 * sharded scan, the all-gather behind it. */
int crp_result_timing(const crp_result *res, float *ms_scan);
/* ms_kernels: the scan kernels alone; ms_total = ms_scan above; n_launches: 1, or 2 if the first
 * capacity guess (1/8 candidate per position and strand) was too small and the scan ran again. */
int crp_result_timing_detail(const crp_result *res, float *ms_kernels, float *ms_total, uint32_t *n_launches);
/* The library's counters since crp_init as one JSON object (launches, commits, scans, sharded scans,
 * fused exchanges, capacity reruns, positions, candidates, bytes over the link, summed event times,
 * communicator, block cache).  CRP_ERR_RANGE (and *needed) if buf is too small. */
int crp_perf_report(char *buf, uint64_t capacity, uint64_t *needed);
/* Number of kernel launches issued by this library since crp_init. */
int crp_launch_count(uint64_t *n);
/* Profiling hook (tools/phase_timeline.py): device buffer of 8 x uint64 per CTA that k_scan_score
 * stamps with %globaltimer at its phase boundaries, or NULL to switch the stamps off. */
int crp_debug_set_times(void *dev_ptr);

#ifdef __cplusplus
}
#endif
#endif /* CROPSR_B200_H */
