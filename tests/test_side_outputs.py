"""The four kernels behind --side-output (csrc/extras.cuh k_extras / k_annotate / k_other_runs, csrc/primers.cuh
k_primers) and the two tables they feed (pipeline.write_side_output, write_gap_table), at their edges.

CPU: the whole-table oracle (oracle/side_output_oracle.py) pinned on a hand-written two-record genome and GFF; the
refusal of a flanking length outside 32 bits before any device work.
GPU: both tables through run_cas9 byte for byte against the oracle (both ingest paths, several genome handles,
nested / equal-start / absent-chromosome features, flanks from 0 to 2**32 - 1); k_primers over a grid of
(e, s, l), filters and D against primer_oracle.design_fast; the gap runs past both retry sizes; gc / flags / run of
every candidate, truncated ones included; feature lookup on deep nesting and equal starts."""
import multiprocessing
import os

import numpy as np
import pytest

import cropsr_oracle as oracle
import extras_oracle
import primer_oracle as po
import side_output_oracle as so
from helpers import fixture_path, fixture_text, synthetic_fasta

TILE = 16384                    # positions per scan tile (kTile)

# ---------------------------------------------------------------- a hand-written genome (clean path: two lines per record)
HAND_A = "GATC" * 7 + "GA" + "GATTACAGCTTCAGTCATCA" + "AGG" + "T" + "GATC" * 10 + "N" * 12 + "GATC" * 6   # 130 bases
HAND_B = "T" * 8 + "CCA" + "GTNcRTTTTT"          # one '-' candidate whose protospacer runs 10 bases past the end
HAND_FASTA = f">chrA\n{HAND_A}\n>chrB\n{HAND_B}"
HAND_GFF = "##gff-version 3\n" + "".join("\t".join(r) + "\n" for r in [
    ("chrA", "t", "gene", "1", "130", ".", "+", ".", "ID=geneA"),
    ("chrA", "t", "exon", "40", "50", ".", "+", ".", "ID=exonA"),              # not gene / CDS: ignored
    ("chrA", "t", "gene", "48", "100", ".", "+", ".", "ID=geneA2"),            # same start as cdsA, longer: loses
    ("chrA", "t", "CDS", "48", "60", ".", "+", ".", "ID=cdsA;Parent=geneA"),   # starts on the cut site (token 47)
    ("chrB", "t", "gene", "1", "9", ".", "-", ".", "ID=geneB"),                # ends on the cut site (token 8)
    ("chrZ", "t", "gene", "1", "1000", ".", "-", ".", "ID=geneZ")])            # no such record
HAND_INFO = "#pacId\tlocusName\ttranscriptName\tpeptideName\tPfam\n1\tcdsA\t\t\tPF00001\n"
HAND_ROWS = [
    "chromosome\tstrand\tpam_pos\tcutsite\tgc\tpoly_t\thomopolymer\tlow_gc\tunscored_base\tlongest_run\tflank_start\t"
    "flank_end\tfeature_type\tfeature_attributes\tfwd_primers\trev_primers\tprimer_pairs\tfirst_pair\tannotation_info",
    # protospacer GATTACAGCTTCAGTCATCA: 8 G/C, longest run 2; the flank is the whole 130-base token = e + l
    "chrA\t+\t50\t47\t8\t0\t0\t1\t0\t2\t0\t130\tCDS\tID=cdsA;Parent=geneA\t770\t767\t58049\t0+21/0+21\tPfam=PF00001",
    # protospacer GTNCRTTTTT + 10 positions past the end: G and C, TTTTT, unscored bytes; flank of 21 < 130: no primers
    "chrB\t-\t8\t8\t2\t1\t1\t1\t1\t5\t0\t21\tgene\tID=geneB\t\t\t\t\t",
]


def _write(path, text):
    with open(path, "w", newline="") as f:
        f.write(text)
    return str(path)


def test_oracle_composition_on_a_hand_written_genome(tmp_path):
    from cropsr_b200 import ingest
    tokens = oracle.import_fasta_text(HAND_FASTA)
    assert not oracle.needs_formatting(HAND_FASTA)
    frame = ingest.import_gff_file(_write(tmp_path / "a.gff", HAND_GFF))
    info = _write(tmp_path / "info.txt", HAND_INFO)
    assert so.side_output_text(tokens, frame, 200, False, info) == "".join(r + "\r\n" for r in HAND_ROWS)
    assert so.gaps_text(tokens) == "chromosome\tstart\tlength\r\nchrA\t94\t12\r\n"
    # flank 64: windows of 128 and 21 bases, both short of e + l; no -p table: the column stays blank
    rows = so.side_output_text(tokens, frame, 64, False).split("\r\n")
    assert rows[1].split("\t")[10:] == ["0", "111", "CDS", "ID=cdsA;Parent=geneA", "", "", "", "", ""]
    # the formatted path: the same features one position later (GFF coordinates shift by 0, not -1)
    assert so.feature_at(so.features_by_chromosome(frame, True)["chrA"], 48)[4] == "ID=cdsA;Parent=geneA"
    assert so.feature_at(so.features_by_chromosome(frame, False)["chrA"], 48)[4] == "ID=cdsA;Parent=geneA"
    assert so.feature_at(so.features_by_chromosome(frame, True)["chrA"], 46)[4] == "ID=geneA"
    assert so.token_chromosome("[('chrA',", True) == so.token_chromosome("('chrA',", True) == "chrA"
    # the rows the truncation rule adds agree with extras_oracle wherever the window is complete
    for key, tok in oracle.import_fasta_text(synthetic_fasta(3, [3000, 700], n_frac=0.01)).items():
        for c, e in zip(oracle.candidates_for_token(key, tok), extras_oracle.extras_for_token(key, tok)):
            if e["full"]:
                assert so.protospacer_stats(so.protospacer(c[4], c[6])) == (e["gc"], e["flags"], e["run"])


@pytest.mark.parametrize("flank", ["-1", "4294967296", "4294967496"])
def test_cli_refuses_flank_outside_32_bits_before_any_device_work(built_lib, flank):
    from cropsr_b200 import cli, engine
    with pytest.raises(SystemExit) as e:
        cli.main(["-f", "missing.fa", "--cas9", "--side-output", "side.tsv", "-L", flank])
    assert "--side-output" in str(e.value.code) and f"-L {flank}" in str(e.value.code)
    assert engine._device is None                                         # refused before engine.init


def test_run_cas9_refuses_flank_outside_32_bits_before_reading_anything(built_lib, tmp_path):
    from cropsr_b200 import engine, pipeline
    for flank in (-1, 1 << 32):
        with pytest.raises(ValueError, match="-L"):
            pipeline.run_cas9(str(tmp_path / "missing.fa"), None, str(tmp_path / "o.csv"), side_output=str(tmp_path / "s.tsv"),
                              flank=flank, time_path=str(tmp_path / "time.txt"))
    assert engine._device is None and not os.path.exists(tmp_path / "o.csv")


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def _test_gff(tokens, formatted_path):
    """A GFF made for the tokens: per record a feature per cut site sample (ending / starting exactly on it),
    two features with equal starts, twelve nested genes, other feature types, and records that do not exist"""
    shift = 0 if formatted_path else 1          # token coordinate -> GFF coordinate
    rows, n = [], 0

    def add(chrom, ftype, a, b):
        nonlocal n
        n += 1
        rows.append((chrom, "test", ftype, str(a + shift), str(b + shift), ".", "+", ".", f"ID={ftype}{n};Name=f{n}"))

    for key, tok in tokens.items():
        chrom = so.token_chromosome(key, formatted_path)
        L = len(tok)
        cuts = [e["cut"] for e in extras_oracle.extras_for_token(key, tok, 0)]
        for i in range(12):                                               # nested, over the middle half
            add(chrom, "gene", L // 4 + 3 * i, max(3 * L // 4 - 5 * i, L // 4 + 3 * i))
        for c in cuts[::max(7, len(cuts) // 100)]:
            add(chrom, "CDS", max(c - 40, 0), c)                          # ends on the cut site
            add(chrom, "CDS", c, c + 9)                                   # starts on it
            add(chrom, "gene", c, c + 30)                                 # equal start, longer: loses to the CDS
            add(chrom, "exon", c - 1, c + 1)                              # not a selected type
        for c in cuts[3::max(11, len(cuts) // 50)]:
            add(chrom, "gene", max(c - 5, 0), c + 5)                      # identical intervals: the later row wins
            add(chrom, "CDS", max(c - 5, 0), c + 5)
        add("absent_" + chrom, "gene", 1, 10 ** 6)
    return "##gff-version 3\n" + "".join("\t".join(r) + "\n" for r in rows)


# name, device_ingest, flank, handle_limit, gff ("sample" or "test"), -p file
TABLE_CASES = [
    ("sample_genome.fa", True, 200, None, "sample", True),
    ("sample_genome.fa", False, 64, None, "test", False),
    ("edge_fmt.fa", True, 200, None, "test", False),
    ("edge_fmt.fa", True, 65, 1, "test", False),
    ("edge_fmt.fa", False, 200, 300, "test", True),
    ("clean3.fa", True, 0, None, "test", False),
    ("clean3.fa", True, 64, None, "test", False),
    ("clean3.fa", True, 65, 1, "test", False),
    ("clean3.fa", True, 200, None, "test", False),
    ("clean3.fa", True, 5000, None, "test", True),
    ("clean3.fa", False, (1 << 32) - 1, None, "test", False),
    ("edge_clean.fa", True, 200, 1, "test", False),
    ("edge_clean.fa", True, 5000, 250, "sample", False),
]


@pytest.mark.gpu
@pytest.mark.parametrize("fasta, device_ingest, flank, handle_limit, gff, info", TABLE_CASES)
def test_side_output_tables_match_oracle(eng, tmp_path, fasta, device_ingest, flank, handle_limit, gff, info):
    """--side-output and its .gaps.tsv byte for byte.  flank 64 leaves every primer window 1 base short of e + l,
    65 makes interior ones exactly 130 bases, 5000 clips at both token ends, 2**32 - 1 must not wrap in 32 bits;
    handle_limit puts the tokens into several genome handles (scan.parts)."""
    from cropsr_b200 import ingest, pipeline
    text = fixture_text(fasta)
    tokens = oracle.import_fasta_text(text)
    formatted_path = oracle.needs_formatting(text)
    gff_path = fixture_path("sample_genome.gff") if gff == "sample" else _write(tmp_path / "t.gff", _test_gff(tokens, formatted_path))
    info_path = None
    if info:
        info_path = _write(tmp_path / "info.txt", "#pacId\tlocusName\ttranscriptName\tpeptideName\tPfam\tPanther\n"
                           "1\tPAU8\tNP_009332.1\tNP_009332.1.p\tPF00660\t\n2\tf3\t\t\tPF1\tPTHR2\n")
    side = tmp_path / "side.tsv"
    stats = pipeline.run_cas9(fixture_path(fasta), gff_path, str(tmp_path / "out.csv"), 20, False, 1, str(tmp_path / "time.txt"),
                              out=lambda *a: None, side_output=str(side), flank=flank, device_ingest=device_ingest,
                              annotation_info=info_path, handle_limit=handle_limit)
    n_windows = sum(1 for tok in tokens.values() for e in extras_oracle.extras_for_token("k", tok, flank)
                    if e["flank_hi"] - e["flank_lo"] >= so.PRIMER_REGION)
    if n_windows > 2000:
        with multiprocessing.get_context("spawn").Pool(min(os.cpu_count() or 1, 32)) as pool:      # design_fast is Python
            want = so.side_output_text(tokens, ingest.import_gff_file(gff_path), flank, formatted_path, info_path,
                                       pool_map=lambda f, xs: pool.map(f, xs, chunksize=64))
    else:
        want = so.side_output_text(tokens, ingest.import_gff_file(gff_path), flank, formatted_path, info_path)
    got = side.read_bytes().decode()
    if got != want:
        g, w = got.split("\r\n"), want.split("\r\n")
        bad = next(i for i in range(min(len(g), len(w))) if g[i] != w[i]) if len(g) == len(w) else None
        pytest.fail(f"{len(g)} vs {len(w)} lines; first difference: {g[bad] if bad is not None else ''!r} vs "
                    f"{w[bad] if bad is not None else ''!r}")
    assert len(want.split("\r\n")) == stats["candidates"] + 2
    assert (tmp_path / "side.tsv.gaps.tsv").read_bytes().decode() == so.gaps_text(tokens)


def test_test_gff_reaches_the_feature_rules(tmp_path):
    """The GFF the table tests write puts CDS, gene and no feature under clean3's candidates"""
    from cropsr_b200 import ingest
    text = fixture_text("clean3.fa")
    tokens = oracle.import_fasta_text(text)
    frame = ingest.import_gff_file(_write(tmp_path / "t.gff", _test_gff(tokens, False)))
    rows = so.side_output_rows(tokens, frame, 64, False)
    kinds = {r[13].split(";")[0][3:].rstrip("0123456789") for r in rows}
    assert {"CDS", "gene", ""} <= kinds


# ---------------------------------------------------------------- the flank window in 32 bits
@pytest.mark.gpu
def test_extras_flank_window_does_not_wrap_at_32_bits(eng):
    """flank_hi = min(cut + flank, L) must not be computed as a wrapping 32-bit sum; a flank outside
    0 <= flank < 2**32 is refused instead of being wrapped by the uint32 argument."""
    from cropsr_b200 import pipeline
    tokens = oracle.import_fasta_text(synthetic_fasta(41, [5000, 900]))
    genome, result, _ = pipeline.scan_tokens(tokens, 20)
    try:
        for flank in ((1 << 32) - 1, (1 << 32) - 10, 1 << 31, 4000, 0):
            for strand in "+-":
                whole = result.extras_strand(strand, flank)
                off = result.off_plus if strand == "+" else result.off_minus
                for seg, (key, tok) in enumerate(tokens.items()):
                    rows = [e for e in extras_oracle.extras_for_token(key, tok, flank) if e["strand"] == strand]
                    a, b = int(off[seg]), int(off[seg + 1])
                    one = result.extras(seg, strand, flank)
                    for name in ("cut", "flank_lo", "flank_hi"):
                        want = [e[name] for e in rows]
                        assert whole[name][a:b].tolist() == want and one[name].tolist() == want, (flank, strand, name)
        for bad in (-1, 1 << 32, (1 << 32) + 200):
            with pytest.raises(ValueError):
                result.extras(0, "+", bad)
            with pytest.raises(ValueError):
                result.extras_strand("-", bad)
    finally:
        result.free()
        genome.free()


# ---------------------------------------------------------------- k_extras: every row
def _iupac_token(rng, n, p_other=0.08):
    alphabet = np.frombuffer(b"ACGTacgtNnRYSWKMU", dtype=np.uint8)
    p = np.array([20, 20, 24, 24, 4, 4, 5, 5] + [p_other * 100 / 9] * 9)
    return rng.choice(alphabet, size=n, p=p / p.sum()).tobytes().decode()


def _oracle_stats(key, tok):
    """{(strand, t): (gc, flags, run)} of every candidate of a token"""
    return {(c[6], c[1] if c[6] == "+" else c[1] - 3): so.protospacer_stats(so.protospacer(c[4], c[6]))
            for c in oracle.candidates_for_token(key, tok)}


@pytest.mark.gpu
def test_extras_of_every_row_including_truncated_ones(eng):
    """gc, flags and run of every candidate -- '-' rows whose protospacer runs up to 10 bases past the token end
    included -- on tokens with lower case, N, IUPAC and U, and on tokens that end just after a CC"""
    from cropsr_b200 import engine
    rng = np.random.default_rng(11)
    toks = [_iupac_token(rng, int(n)) for n in rng.integers(30, 3000, size=12)]
    toks += ["ACGT" * 3 + "CC" + "A" * m for m in range(10, 22)]          # a '-' hit 12 .. 23 bases from the end
    toks += ["TTTTTCCAGGGGGGGGGG", "CCCCCCCCCCCCCCCCCCCCCCCCC", "ccgttttaaaacc" * 3]
    g = engine.Genome()
    for t in toks:
        g.add_token(t)
    r = g.commit().scan(20)
    try:
        truncated = 0
        for strand in "+-":
            ex = r.extras_strand(strand, 200)
            pos = r.fetch(strand, want=("pos",))["pos"]
            off = r.off_plus if strand == "+" else r.off_minus
            for seg, tok in enumerate(toks):
                want = _oracle_stats(">k", tok)
                for i in range(int(off[seg]), int(off[seg + 1])):
                    t = int(pos[i])
                    assert (int(ex["gc"][i]), int(ex["flags"][i]), int(ex["run"][i])) == want[(strand, t)], (seg, strand, t)
                    truncated += strand == "-" and t + 23 > len(tok)
                assert sorted(t for s, t in want if s == strand) == pos[int(off[seg]):int(off[seg + 1])].tolist()
        assert truncated >= 6
    finally:
        r.free()
        g.free()


@pytest.mark.gpu
def test_extras_and_annotation_of_segments_that_start_inside_their_token(eng):
    """add_segment pieces with a tile-aligned begin > 0: each piece's candidates get the extras and features of
    the whole token (the records are addressed relative to seg_begin)"""
    from cropsr_b200 import engine
    rng = np.random.default_rng(12)
    tok = _iupac_token(rng, 3 * TILE + 5000, p_other=0.01)
    cuts = [0, TILE, 2 * TILE + 128 * 3, len(tok)]
    want = _oracle_stats(">k", tok)
    ex_want = {(e["strand"], e["t"]): e for e in extras_oracle.extras_for_token(">k", tok, 300)}
    start = np.sort(rng.integers(0, len(tok), size=300)).astype(np.uint32)
    end = (start + rng.integers(0, 4000, size=300)).astype(np.uint32)
    g = engine.Genome()
    for a, b in zip(cuts, cuts[1:]):
        g.add_segment(0, tok, a, b)
    r = g.commit().scan(20)
    try:
        seen = set()
        iv_off = np.array([0, 0, 300, 300], dtype=np.uint64)             # only the middle piece has intervals
        for strand in "+-":
            feat = r.annotate_strand(strand, iv_off, start, end)
            off = r.off_plus if strand == "+" else r.off_minus
            for seg in range(3):
                got = r.extras(seg, strand, 300)
                pos = r.fetch_segment(seg, strand, want=("pos",))["pos"].tolist()
                for i, t in enumerate(pos):
                    seen.add((strand, t))
                    assert (int(got["gc"][i]), int(got["flags"][i]), int(got["run"][i])) == want[(strand, t)]
                    e = ex_want[(strand, t)]
                    assert (int(got["cut"][i]), int(got["flank_lo"][i]), int(got["flank_hi"][i])) == \
                        (e["cut"], e["flank_lo"], e["flank_hi"])
                f = feat[int(off[seg]):int(off[seg + 1])]
                if seg == 1:
                    assert np.array_equal(f, extras_oracle.annotate(got["cut"].tolist(), start, end))
                else:
                    assert (f == -1).all()
        assert seen == set(want)
    finally:
        r.free()
        g.free()


# ---------------------------------------------------------------- k_annotate
@pytest.mark.gpu
def test_annotation_interval_shapes(eng):
    """Deep nesting (the maxend walk-back goes back over hundreds of intervals), equal starts (sorted longer first,
    so the shorter wins), cut sites exactly on a start or an end, and annotate_strand with segments that have no
    intervals next to ones that have"""
    from cropsr_b200 import engine
    rng = np.random.default_rng(13)
    toks = [_iupac_token(rng, n, p_other=0.0) for n in (20000, 900, 15000, 4000, 700)]
    g = engine.Genome()
    for t in toks:
        g.add_token(t)
    r = g.commit().scan(20)
    try:
        ivs = []
        for k, tok in enumerate(toks):
            L = len(tok)
            if k in (1, 4):                                              # no intervals
                ivs.append((np.empty(0, np.int64), np.empty(0, np.int64)))
                continue
            cuts = sorted({e["cut"] for e in extras_oracle.extras_for_token(">k", tok, 0)})
            iv = [(0, L - 1)]                                            # one outer feature ...
            iv += [(x, x + 1) for x in range(10, L - 10, 13)]            # ... then hundreds of short ones after it
            iv += [(5 + i, L - 6 - i) for i in range(40)]                # deep nesting
            for c in cuts[::5]:
                iv += [(c, c + 20), (c, c), (c - 20, c), (c, c + 3)]     # equal starts; cut on a start, on an end
            for c in cuts[2::9]:
                iv += [(c - 4, c + 4), (c - 4, c + 4)]                   # identical
            iv = [(a, b) for a, b in iv if 0 <= a <= b]
            a = np.array([x for x, _ in iv], dtype=np.int64)
            b = np.array([y for _, y in iv], dtype=np.int64)
            order = np.lexsort((-b, a))                                  # annotate.intervals_for_tokens' order
            ivs.append((a[order], b[order]))
        iv_off = np.concatenate(([0], np.cumsum([len(a) for a, _ in ivs]))).astype(np.uint64)
        start = np.concatenate([a for a, _ in ivs]).astype(np.uint32)
        end = np.concatenate([b for _, b in ivs]).astype(np.uint32)
        deep = 0
        for strand in "+-":
            feat = r.annotate_strand(strand, iv_off, start, end)
            pos = r.fetch(strand, want=("pos",))["pos"].astype(np.int64)
            off = r.off_plus if strand == "+" else r.off_minus
            for seg, (a, b) in enumerate(ivs):
                lo, hi = int(off[seg]), int(off[seg + 1])
                cut = pos[lo:hi] - (3 if strand == "+" else 0)
                want = extras_oracle.annotate(cut.tolist(), a, b)
                assert np.array_equal(feat[lo:hi], want), (seg, strand)
                assert np.array_equal(r.annotate(seg, strand, a, b), want)
                walk = np.searchsorted(a, cut, side="right") - 1 - want          # intervals the walk-back passes
                deep += int(((want >= 0) & (walk > 50)).sum())
        assert deep > 50
        assert (r.annotate_strand("+", np.zeros(len(toks) + 1, np.uint64), start[:0], end[:0]) == -1).all()
    finally:
        r.free()
        g.free()


# ---------------------------------------------------------------- k_other_runs
@pytest.mark.gpu
def test_gap_runs_past_both_retry_sizes(eng):
    """more than 65,536 runs in one segment (the library's first boundary list), more than 4,096 kept runs
    (Genome.other_runs' first capacity) but fewer at a larger min_len, an all-N token, runs across every tile edge
    of a multi-tile segment, and runs touching both ends of add_segment pieces"""
    from cropsr_b200 import engine
    rng = np.random.default_rng(14)
    singles = "".join("A" + "NRYSWKM"[i % 7] for i in range(70000))                      # 70,000 runs of one byte
    pairs = "".join(("ACGT" if i % 50 else "ACGTNNNNNNNN"[:9]) + "NN" for i in range(5000))  # 5,000 runs >= 2, 100 >= 7
    all_n = "N" * 40000
    edges = bytearray(_iupac_token(rng, 5 * TILE + 77, p_other=0.0).encode())
    for k in range(1, 6):
        edges[k * TILE - 3:k * TILE + 4] = b"N" * 7                                      # across every tile edge
    edges[TILE + 31:TILE + 33] = b"nR"                                                   # across a word edge
    edges[0:3] = b"RRR"
    edges[-5:] = b"NNNNN"
    edges = edges.decode()
    toks = [singles, pairs, all_n, edges, "ACGT", "N"]
    g = engine.Genome()
    for t in toks:
        g.add_token(t)
    pieces = [0, TILE, 3 * TILE, len(edges)]                                             # the same token in pieces
    for a, b in zip(pieces, pieces[1:]):
        g.add_segment(len(toks), edges, a, b)
    g.commit()
    try:
        for seg, tok in enumerate(toks):
            for min_len in (1, 2, 7, 10):
                start, length = g.other_runs(seg, min_len)
                assert list(zip(start.tolist(), length.tolist())) == extras_oracle.other_runs(tok, min_len), (seg, min_len)
        assert len(g.other_runs(0, 1)[0]) == 70000 and len(g.other_runs(1, 2)[0]) == 5000 and len(g.other_runs(1, 7)[0]) == 100
        for p, (a, b) in enumerate(zip(pieces, pieces[1:])):                            # clipped to the piece
            for min_len in (1, 3):
                start, length = g.other_runs(len(toks) + p, min_len)
                want = [(s + a, n) for s, n in extras_oracle.other_runs(edges[a:b], min_len)]
                assert list(zip(start.tolist(), length.tolist())) == want, (p, min_len)
    finally:
        g.free()


# ---------------------------------------------------------------- k_primers
def _primer_genome(eng, rng):
    """Tokens whose lengths are multiples of 16,384 plus tile-aligned pieces with begin > 0; lower case, N, IUPAC"""
    from cropsr_b200 import engine
    def frag(n):
        return _iupac_token(rng, n, p_other=0.03)
    toks = [frag(2 * TILE), frag(TILE + 3000), frag(TILE)]
    g = engine.Genome()
    segs = []                                                  # (segment, token, begin, end)
    for k, t in enumerate(toks[:2]):
        segs.append((g.add_token(t), t, 0, len(t)))
    segs.append((g.add_segment(2, toks[1], TILE, len(toks[1])), toks[1], TILE, len(toks[1])))
    segs.append((g.add_segment(3, toks[2], 0, TILE), toks[2], 0, TILE))
    g.commit()
    return g, segs


def _windows(rng, segs, region, n_random, max_extra=300):
    """(segment, lo, hi): exactly `region` bases, from the segment's first position, to the last position of a token
    whose length is a multiple of 16,384, over tile edges, and random ones"""
    out = []
    for s, tok, a, b in segs:
        out += [(s, a, a + region), (s, b - region, b), (s, a, min(b, a + region + 1))]
        for edge in range((a // TILE + 1) * TILE, b, TILE):
            out.append((s, max(a, edge - region // 2), min(b, edge - region // 2 + region + 7)))
    for _ in range(n_random):
        s, tok, a, b = segs[int(rng.integers(len(segs)))]
        n = int(rng.integers(region, region + max_extra))
        lo = int(rng.integers(a, b - n + 1))
        out.append((s, lo, lo + n))
    out.append((segs[0][0], segs[0][2], segs[0][2] + region - 1))          # one base short: status 1
    return out


def _check_primers(eng, g, segs, windows, params):
    from cropsr_b200 import primers
    tok_of = {s: tok for s, tok, _, _ in segs}
    seg = np.array([w[0] for w in windows], np.uint32)
    lo = np.array([w[1] for w in windows], np.uint32)
    hi = np.array([w[2] for w in windows], np.uint32)
    out = primers.design_windows(g, seg, lo, hi, **params)
    p = dict(primers.DEFAULTS, **params)
    region = p["e"] + p["l"]
    cache = {}
    for k, (s, a, b) in enumerate(windows):
        if b - a < region:
            assert out["status"][k] == 1 and out["n_pairs"][k] == 0 and out["first"][k].tolist() == [0xFFFF] * 4
            continue
        frag = tok_of[s][a:b]
        if frag not in cache:
            cache[frag] = po.design_fast(frag, **p)
        want = cache[frag]
        got = (int(out["status"][k]), int(out["n_fwd"][k]), int(out["n_rev"][k]), int(out["n_pairs"][k]), out["first"][k].tolist())
        assert got == (0, want["n_fwd"], want["n_rev"], want["n_pairs"], list(want["first"]) if want["first"] else [0xFFFF] * 4), \
            (params, s, a, b)
    return out


PASS_ALL = dict(m=-1e9, x=1e9, M=-1.0, X=101.0)
PASS_NONE = dict(m=1e9)
PRIMER_GRID = [
    (dict(e=1, s=12, l=13), 60),
    (dict(e=1, s=12, l=31), 60),
    (dict(e=1, s=12, l=31, **PASS_ALL), 60),
    (dict(e=1, s=12, l=31, D=0.0, **PASS_ALL), 60),
    (dict(e=7, s=12, l=31, D=1000.0, **PASS_ALL), 60),          # every pair Tm-close
    (dict(e=40, s=13, l=32, D=0.0, **PASS_ALL), 30),                # l = 32, 627 classes
    (dict(e=100), 40),
    (dict(e=100, D=0.0), 40),
    (dict(e=100, **PASS_NONE), 20),
    (dict(e=100, D=1000.0), 20),
    (dict(e=500, s=12, l=30), 6),
    (dict(e=992, s=20, l=32), 4),
    (dict(e=994, s=29, l=30), 4),
    (dict(e=994, s=29, l=30, **PASS_ALL, D=1000.0), 2),
]


@pytest.mark.gpu
@pytest.mark.parametrize("params, n_random", PRIMER_GRID, ids=lambda v: ",".join(f"{k}={v[k]}" for k in v) if isinstance(v, dict) else str(v))
def test_primer_windows_parameter_grid(eng, params, n_random):
    """k_primers against design_fast: 1 to 32 mask words per end, 13-base primers with up to 608 classes, l = 32,
    filters that pass nothing or everything, D = 0 and D that makes every pair close; windows of exactly e + l
    bases, from a segment's first position, up to the last position of a 2 x 16,384-base token, over tile edges,
    in pieces whose begin is a tile edge"""
    from cropsr_b200 import primers
    rng = np.random.default_rng(15 + params["e"])
    g, segs = _primer_genome(eng, rng)
    try:
        region = params["e"] + params.get("l", primers.DEFAULTS["l"])
        _check_primers(eng, g, segs, _windows(rng, segs, region, n_random), params)
    finally:
        g.free()


@pytest.mark.gpu
def test_primer_windows_beyond_one_grid_sweep(eng):
    """More windows than the launch grid x 8 warps (the grid-stride loop: a warp reuses its histogram), with 608
    classes of which every one passes -- a histogram bin a warp leaves uncleared shows up here"""
    rng = np.random.default_rng(16)
    g, segs = _primer_genome(eng, rng)
    try:
        sm = eng.perf_report()["sm_count"]
        n = sm * 8 * 8 + 3000
        windows = _windows(rng, segs, 32, n, max_extra=40)
        for params in (dict(e=1, s=12, l=31, **PASS_ALL), dict(e=1, s=12, l=31, D=0.0, **PASS_ALL)):
            _check_primers(eng, g, segs, windows, params)
    finally:
        g.free()


@pytest.mark.gpu
def test_primer_parameter_refusals(eng):
    """e + l = 1024 is the largest region (one mask word per lane); s >= 12; at most 640 (N, gc) classes"""
    from cropsr_b200 import engine, primers, _native
    g = engine.Genome()
    g.add_token(_iupac_token(np.random.default_rng(17), 3000, p_other=0.0))
    g.commit()
    try:
        for ok in (dict(e=992, s=20, l=32), dict(e=994, s=29, l=30), dict(e=1, s=12, l=31)):
            assert primers.design_windows(g, [0], [0], [2000], **ok)["status"][0] == 0
        for bad in (dict(e=993, s=20, l=32), dict(e=996, s=29, l=30), dict(s=11, l=20), dict(e=1, s=12, l=32),
                    dict(e=0), dict(s=20, l=20), dict(s=20, l=33)):
            with pytest.raises(_native.CropsrError):
                primers.design_windows(g, [0], [0], [2000], **bad)
    finally:
        g.free()
