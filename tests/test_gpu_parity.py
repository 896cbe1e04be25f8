"""Parity of the CUDA path (through the C ABI) with the oracle and with the
golden CSVs of the unmodified reference.  Everything here needs a B200."""
import csv
import io
import os

import numpy as np
import pytest

import cropsr_oracle as oracle
from helpers import fixture_path, fixture_text, golden_csv, normalised_digest, synthetic_fasta

pytestmark = pytest.mark.gpu

ALL_CASES = ["sample", "sample_t6", "multi3", "multi3_l18", "multi3_l23", "clean3", "clean3_trailing_nl",
             "edge_clean", "edge_fmt", "single_candidate", "ws_header", "dup_keys", "empty_records",
             "mid50k", "mid50k_t5", "mid50k_c1000", "mid50k_c1557", "multi3_c20", "sample_c5000_t4"]


@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


@pytest.mark.parametrize("name", ALL_CASES)
def test_cli_csv_is_byte_identical_to_reference(name, manifest, eng, tmp_path, capsys):
    """Full drop-in run: FASTA -> CSV, ids seeded like the golden run."""
    from cropsr_b200 import pipeline
    case = manifest["cases"][name]
    out = tmp_path / "out.csv"
    np.random.seed(case["seed"])
    lines = []
    pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out),
                      case["guide_len"], False, case["blas_threads"], str(tmp_path / "time.txt"),
                      out=lambda *a: lines.append(" ".join(a)), chunk_rows=case.get("chunk"))
    got = out.read_bytes().decode()
    assert got == golden_csv(name)
    want_stdout = open(os.path.join(os.path.dirname(fixture_path("x")), "..", "cases", name + ".stdout")).read()
    assert "\n".join(lines) + ("\n" if lines else "") == want_stdout
    assert (tmp_path / "time.txt").read_text().count("Total runtime of the program is ") == case["time_txt_records"]


def _check_against_oracle(eng, text, guide_len):
    from cropsr_b200 import ingest, pipeline, _native as N
    tokens = ingest.fasta_text_to_tokens(text)
    genome, result, _ = pipeline.scan_tokens(tokens, guide_len)
    try:
        for seg, (key, tok) in enumerate(tokens.items()):
            plus, minus = oracle.pam_hits(tok, guide_len)
            gp = result.fetch_segment(seg, "+")
            gm = result.fetch_segment(seg, "-")
            assert gp["pos"].tolist() == plus
            assert gm["pos"].tolist() == minus
            if guide_len != 20:
                assert gp["x"] is None
                continue
            cands = oracle.candidates_for_token(key, tok, guide_len)
            x = np.concatenate((gp["x"], gm["x"]))
            packed = np.concatenate((gp["packed"], gm["packed"]))
            full = np.array([len(c[4]) == 30 for c in cands], dtype=bool)
            assert np.array_equal((packed & np.uint64(N.PACKED_TRUNCATED)) != 0, ~full)
            if full.any():
                seqs = np.array([oracle.scored_bytes(c[4]) for c, f in zip(cands, full) if f])
                want = oracle.preactivation_model(seqs, classes=np.zeros(len(seqs), dtype=np.int8))
                assert np.array_equal(x[full], want)
                # packed 30-mer: planar A0 T1 C2 G3 codes of the scored bases
                code = np.full(seqs.shape, -1)
                for c, b in enumerate(b"ATCG"):
                    code[seqs == b] = c
                lo = np.array([sum(((int(v) & 1) << q) for q, v in enumerate(row) if v >= 0) for row in code], dtype=np.uint64)
                hi = np.array([sum((((int(v) >> 1) & 1) << q) for q, v in enumerate(row) if v >= 0) for row in code], dtype=np.uint64)
                scoring = code >= 0
                pk = packed[full]
                got_lo = pk & np.uint64(0x3FFFFFFF)
                got_hi = (pk >> np.uint64(32)) & np.uint64(0x3FFFFFFF)
                mask = np.array([sum((1 << q) for q, v in enumerate(row) if v) for row in scoring], dtype=np.uint64)
                assert np.array_equal(got_lo & mask, lo) and np.array_equal(got_hi & mask, hi)
                assert np.array_equal((pk & np.uint64(N.PACKED_UNSCORED)) != 0, ~scoring.all(axis=1))
                # irregular = the token window holds a byte that is not upper-case ACGT
                def window(c):
                    return tok[c[1] - 25:c[1] + 5] if c[6] == "+" else tok[c[1] - 5:c[1] + 25]
                irregular = np.array([any(ch not in "ACGT" for ch in window(c)) for c, f in zip(cands, full) if f])
                assert np.array_equal((pk & np.uint64(N.PACKED_IRREGULAR)) != 0, irregular)
    finally:
        result.free()
        genome.free()


@pytest.mark.parametrize("fasta", ["multi3.fa", "clean3.fa", "edge_clean.fa", "edge_fmt.fa", "ws_header.fa",
                                   "dup_keys.fa", "empty_records.fa", "single_candidate.fa", "mid50k.fa",
                                   "sample_genome.fa"])
@pytest.mark.parametrize("guide_len", [20, 18, 23])
def test_candidate_streams_match_oracle(eng, fasta, guide_len):
    _check_against_oracle(eng, fixture_text(fasta), guide_len)


@pytest.mark.parametrize("seed", range(12))
def test_random_fastas_match_oracle(eng, seed):
    rng = np.random.default_rng(1000 + seed)
    n_rec = int(rng.integers(1, 6))
    alphabet = np.frombuffer(b"ACGTacgtNRYUZ", dtype=np.uint8)
    p = np.array([20, 20, 20, 20, 3, 3, 3, 3, 1, .3, .3, .2, .2])
    recs = []
    for k in range(n_rec):
        n = int(rng.integers(0, 30000)) if seed % 3 else int(rng.integers(0, 200))
        recs.append((f"r{k}", rng.choice(alphabet, size=n, p=p / p.sum()).tobytes().decode()))
    if seed % 2:
        text = "".join(f">{h}\n" + "\n".join(s[i:i + 70] for i in range(0, len(s), 70)) + "\n" for h, s in recs)
    else:
        text = "\n".join(f">{h}\n{s}" for h, s in recs if s)
    _check_against_oracle(eng, text, 20)


@pytest.mark.parametrize("guide_len", [1, 1000, 20000, 40000, 70000, 200000])
def test_guide_lengths_that_span_tiles(eng, guide_len):
    """The bounds of CROPSR.py:419 / :430 reach guide_len + 5 positions into a token and guide_len - 7 back
    from its end.  With a long guide several tiles at either end of a token are counted from their PAM
    records at scan time; all the others take the counts k_pack wrote into their tile headers, which hold
    for every guide length.  Positions only (the reference scores 20-mers)."""
    rng = np.random.default_rng(77)
    alphabet = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)
    p = np.array([15, 15, 30, 30, 2, 2, 2, 2, 2], dtype=float)
    recs = [(f"long{k}", rng.choice(alphabet, size=n, p=p / p.sum()).tobytes().decode())
            for k, n in enumerate((70001, 40000, 16380, 300))]
    text = "".join(f">{h}\n{s}\n" for h, s in recs)
    _check_against_oracle(eng, text, guide_len)


def test_tile_boundaries_and_dense_hits(eng):
    # PAMs straddling every 8192-position tile edge; poly-G / poly-C worst-case density
    body = bytearray(b"AT" * 20000)
    for edge in (8192, 16384, 24576, 32768):
        for off in range(-3, 3):
            body[edge + off] = ord("G")
        body[edge - 40:edge - 36] = b"CCCC"
    text = ">t\n" + body.decode() + "\n>g\n" + "G" * 20000 + "\n>c\n" + "C" * 20000 + "\n"
    _check_against_oracle(eng, text, 20)


def test_rescore_classes_match_oracle(eng):
    from cropsr_b200 import ingest, pipeline
    text = fixture_text("mid50k.fa")
    tokens = ingest.fasta_text_to_tokens(text)
    genome, result, _ = pipeline.scan_tokens(tokens, 20)
    (key, tok), = tokens.items()
    cands = [c for c in oracle.candidates_for_token(key, tok, 20) if len(c[4]) == 30][:600]
    seqs = np.array([oracle.scored_bytes(c[4]) for c in cands])
    t = np.array([c[1] - 3 if c[6] == "-" else c[1] for c in cands], dtype=np.uint32)
    strand = np.array([c[6].encode() for c in cands], dtype="S1")
    seg = np.zeros(len(cands), dtype=np.uint32)
    for c1 in (0, 1, 2):
        for c2 in (0, 1, 2):
            m1, m2 = oracle.indicator_matrices(seqs)
            a = oracle.lane_sums(m1, oracle.W1, np.full(len(seqs), c1, dtype=np.int8))
            b = oracle.lane_sums(m2, oracle.W2, np.full(len(seqs), c2, dtype=np.int8))
            want = (a + b + oracle.INTERCEPT + oracle.LOW_GC) * -1
            got = genome.rescore(seg, t, strand, np.full(len(seqs), c1 | (c2 << 4), dtype=np.uint8))
            assert np.array_equal(got, want), (c1, c2)
    result.free()
    genome.free()


def test_sharded_scan_equals_whole_scan(eng):
    """N logical shards on one GPU: segments with halos + offset arithmetic give
    exactly the single-shard streams (the multi-GPU data path minus NCCL)."""
    from cropsr_b200 import engine, ingest, shard
    text = synthetic_fasta(7, [70000, 30000, 90000], gc=0.5)
    tokens = ingest.fasta_text_to_tokens(text)
    toks = [v.encode() for v in tokens.values()]
    whole = engine.Genome()
    for b in toks:
        whole.add_token(b)
    ref = whole.commit().scan(20)
    ref_tab = []
    for s in range(len(toks)):
        for strand in "+-":
            f = ref.fetch_segment(s, strand)
            ref_tab += list(zip([s] * len(f["pos"]), [strand] * len(f["pos"]), f["pos"].tolist(), f["x"].tolist(), f["packed"].tolist()))
    for ws in (2, 3, 4, 7):
        plans = shard.plan([len(b) for b in toks], ws)
        counts, rows = [], {}
        for r, segs in enumerate(plans):
            g = engine.Genome()
            for k, a, b in segs:
                g.add_segment(k, toks[k], a, b)
            res = g.commit().scan(20)
            counts.append((res.seg_plus.tolist(), res.seg_minus.tolist()))
            rows[r] = [(res.fetch_segment(s, "+"), res.fetch_segment(s, "-")) for s in range(len(segs))]
            res.free()
            g.free()
        offs, total = shard.global_offsets(plans, counts)
        assert total == len(ref_tab)
        table = [None] * total
        for r, segs in enumerate(plans):
            for s, (k, a, b) in enumerate(segs):
                for si, strand in enumerate("+-"):
                    f = rows[r][s][si]
                    for i in range(len(f["pos"])):
                        table[offs[r][s][si] + i] = (k, strand, int(f["pos"][i]), float(f["x"][i]), int(f["packed"][i]))
        assert table == ref_tab, ws
    ref.free()
    whole.free()


def test_full_size_properties(eng):
    """At a BASELINE-scale chromosome (34 Mbp) the oracle is too slow for the
    whole thing, so check size-independent properties: sorted, unique positions;
    every reported hit is a PAM in the text; a sampled window re-scored through
    the dense crp_rescore path equals the fused kernel's x; counts equal a
    vectorised numpy PAM count."""
    from cropsr_b200 import engine, ingest
    text = synthetic_fasta(2, [34000000], gc=0.36, lower_frac=0.15)
    tokens = ingest.fasta_text_to_tokens(text)
    (key, tok), = tokens.items()
    b = tok.encode()
    arr = np.frombuffer(b, dtype=np.uint8)
    g = engine.Genome()
    g.add_token(b)
    res = g.commit().scan(20)
    L = len(arr)
    isg, isc = arr == ord("G"), arr == ord("C")
    plus = np.nonzero(isg[1:-1] & isg[2:])[0]
    plus = plus[plus >= 25]
    minus = np.nonzero(isc[:-2] & isc[1:-1])[0]
    minus = minus[(minus >= 2) & (minus <= L - 13)]
    gp, gm = res.fetch("+"), res.fetch("-")
    assert np.array_equal(gp["pos"], plus.astype(np.uint32))
    assert np.array_equal(gm["pos"], minus.astype(np.uint32))
    rng = np.random.default_rng(0)
    for strand, f in (("+", gp), ("-", gm)):
        pick = rng.choice(len(f["pos"]), size=20000, replace=False)
        x2 = g.rescore(np.zeros(len(pick), np.uint32), f["pos"][pick], np.full(len(pick), strand.encode(), "S1"),
                       np.zeros(len(pick), np.uint8))
        assert np.array_equal(x2, f["x"][pick])
        # and a smaller sample against the oracle's literal string path
        for i in pick[:300]:
            t = int(f["pos"][i])
            if strand == "+":
                long_ = oracle.grna(tok[t - 25:t + 5])
            else:
                long_ = oracle.grna(oracle.reverse_complement(tok[t - 2:t + 28]))
            if len(long_) == 30:
                want = oracle.preactivation_model(np.array([oracle.scored_bytes(long_)]), classes=np.zeros(1, np.int8))
                assert f["x"][i] == want[0]
    res.free()
    g.free()


def test_static_and_ticketed_tile_dealing_match_oracle(eng, monkeypatch):
    """The emit phase deals part of the tiles round-robin and the rest through a ticket counter: all
    static, all ticketed, and the default split give the same streams."""
    for eighths in ("8", "0", "4"):
        monkeypatch.setenv("CRP_STATIC_EIGHTHS", eighths)
        _check_against_oracle(eng, synthetic_fasta(23, [90000, 40000], gc=0.5, lower_frac=0.2), 20)


def test_long_count_ranges_and_prefetched_first_tile(eng, monkeypatch):
    """With few CTAs every CTA counts a long range of tiles: the 6-slot ring of PAM records is
    refilled many times, by different warps, and ranges longer than 32 tiles are walked in batches
    with a running prefix (on a multi-Gbp genome that is the normal case: 237 tiles per CTA on the
    maize-scale config); the first emit tile is fetched across the grid barrier.  3, 7 and 1 CTAs
    force it on ~100 tiles (1 CTA: four batches, the ring goes round sixteen times)."""
    text = synthetic_fasta(31, [900000, 650000, 37], gc=0.45, lower_frac=0.15, n_frac=0.001)
    monkeypatch.setenv("CRP_SCAN_GRID", "3")
    _check_against_oracle(eng, text, 20)
    monkeypatch.setenv("CRP_SCAN_GRID", "7")
    _check_against_oracle(eng, text, 20)
    monkeypatch.setenv("CRP_STATIC_EIGHTHS", "8")
    _check_against_oracle(eng, text, 20)
    monkeypatch.setenv("CRP_SCAN_GRID", "1")
    monkeypatch.setenv("CRP_STATIC_EIGHTHS", "4")
    _check_against_oracle(eng, text, 20)
    monkeypatch.setenv("CRP_SCAN_GRID", "2")
    monkeypatch.setenv("CRP_STATIC_EIGHTHS", "0")
    _check_against_oracle(eng, synthetic_fasta(32, [1100000], gc=0.5, lower_frac=0.1), 20)     # 68 tiles: 34 per CTA, 32 + 2


def test_pipelined_call_equals_plain_scan(eng):
    """crp_scan_segments (overlapped H2D / pack / scan / D2H, one segment at a time) returns
    exactly the rows of the plain add_segment/commit/scan/fetch path, in segment order."""
    from cropsr_b200 import engine, ingest
    text = synthetic_fasta(31, [70000, 1500, 45000], gc=0.5)
    toks = [v.encode() for v in ingest.fasta_text_to_tokens(text).values()]
    cut = 2 * engine.TILE
    segs = [(0, toks[0], 0, cut), (0, toks[0], cut, len(toks[0])), (1, toks[1], 0, None), (2, toks[2], 0, None)]
    for guide_len in (20, 18):
        g = engine.Genome()
        for k, tok, a, b in segs:
            g.add_segment(k, tok, a, b)
        res = g.commit().scan(guide_len)
        arena, n_plus, n_minus, ms = engine.scan_segments(segs, guide_len)
        assert n_plus.tolist() == res.seg_plus.tolist() and n_minus.tolist() == res.seg_minus.tolist()
        for strand, n in (("+", res.n_plus), ("-", res.n_minus)):
            want = res.fetch(strand)
            got = arena.arrays[strand]
            assert np.array_equal(got["pos"][:n], want["pos"])
            if guide_len == 20:
                assert np.array_equal(got["packed"][:n], want["packed"])
                assert np.array_equal(got["x"][:n], want["x"])
        # an arena that is too small is replaced by one of the right size
        small = engine.Arena(16, guide_len == 20)
        arena2, p2, m2, _ = engine.scan_segments(segs, guide_len, arena=small)
        assert p2.tolist() == n_plus.tolist() and arena2.capacity >= max(res.n_plus, res.n_minus)
        assert np.array_equal(arena2.arrays["-"]["pos"][:res.n_minus], res.fetch("-")["pos"])
        arena.free()
        arena2.free()
        res.free()
        g.free()


@pytest.mark.parametrize("seed", range(4))
def test_extras_and_annotation_match_oracle(eng, seed):
    """Opt-in side outputs (GC / poly-T / homopolymer / cut / flank / feature index): device
    kernels vs the independent string oracle, on FASTAs with lower-case, N and IUPAC."""
    import extras_oracle
    from cropsr_b200 import ingest, pipeline
    rng = np.random.default_rng(500 + seed)
    alphabet = np.frombuffer(b"ACGTacgtNRU", dtype=np.uint8)
    p = np.array([20, 20, 20, 20, 3, 3, 3, 3, 1, .3, .2])
    recs = [(f"r{k}", rng.choice(alphabet, size=int(rng.integers(100, 40000)), p=p / p.sum()).tobytes().decode())
            for k in range(3)]
    recs.append(("polyT", "ACGT" * 10 + "TTTTTTTTGG" * 30 + "CCAAAAAAAA" * 30))
    text = "".join(f">{h}\n" + "\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + "\n" for h, s in recs)
    tokens = ingest.fasta_text_to_tokens(text)
    genome, result, _ = pipeline.scan_tokens(tokens, 20)
    try:
        for seg, (key, tok) in enumerate(tokens.items()):
            want = extras_oracle.extras_for_token(key, tok, flank=150)
            n_iv = int(rng.integers(0, 40))
            a = np.sort(rng.integers(0, max(len(tok), 1), size=n_iv)).astype(np.uint32)
            b = (a + rng.integers(0, 3000, size=n_iv)).astype(np.uint32)
            for strand in "+-":
                rows = [r for r in want if r["strand"] == strand]
                got = result.extras(seg, strand, flank=150)
                assert got["cut"].tolist() == [r["cut"] for r in rows]
                assert got["flank_lo"].tolist() == [r["flank_lo"] for r in rows]
                assert got["flank_hi"].tolist() == [r["flank_hi"] for r in rows]
                full = np.array([r["full"] for r in rows], dtype=bool)
                for name in ("gc", "flags", "run"):
                    assert got[name][full].tolist() == [r[name] for r in rows if r["full"]], (name, strand)
                feat = result.annotate(seg, strand, a, b)
                assert np.array_equal(feat, extras_oracle.annotate([r["cut"] for r in rows], a, b))
    finally:
        result.free()
        genome.free()


def test_cli_side_output_leaves_csv_untouched(manifest, eng, tmp_path):
    """--side-output writes its own table; the parity CSV stays byte-identical to the reference's."""
    from cropsr_b200 import pipeline
    case = manifest["cases"]["sample"]
    out, side = tmp_path / "out.csv", tmp_path / "side.tsv"
    np.random.seed(case["seed"])
    info = tmp_path / "annotation_info.txt"       # -p: rows keyed by names the sample GFF uses (Name= of a gene and of a CDS)
    info.write_text("#pacId\tlocusName\ttranscriptName\tpeptideName\tPfam\tPanther\tKOG\tec\tKO\tGO\n"
                    "1\tPAU8\tNP_009332.1\tNP_009332.1.p\tPF00660\t\t\t\t\tGO:0030437\n")
    stats = pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out), 20, False,
                              case["blas_threads"], str(tmp_path / "time.txt"), out=lambda *a: None,
                              side_output=str(side), flank=200, annotation_info=str(info))
    assert out.read_bytes().decode() == golden_csv("sample")
    rows = list(csv.reader(open(side), delimiter="\t"))
    assert len(rows) == stats["candidates"] + 1
    assert rows[0][:5] == ["chromosome", "strand", "pam_pos", "cutsite", "gc"]
    assert any(r[12] == "CDS" for r in rows[1:]) and any(r[12] == "" for r in rows[1:])
    assert all(0 <= int(r[4]) <= 20 for r in rows[1:])
    # primer columns: filled wherever the flank holds e + l = 130 bases, and consistent
    assert rows[0][14:] == ["fwd_primers", "rev_primers", "primer_pairs", "first_pair", "annotation_info"]
    filled = [r for r in rows[1:] if r[14] != ""]
    assert len(filled) > 0.99 * stats["candidates"]
    assert all(int(r[16]) <= int(r[14]) * int(r[15]) and (r[17] != "") == (int(r[16]) > 0) for r in filled)
    hit = [r for r in rows[1:] if r[18]]
    assert hit and all(r[18] == "Pfam=PF00660;GO=GO:0030437" and ("PAU8" in r[13] or "NP_009332.1" in r[13]) for r in hit)


def test_device_fasta_ingest_equals_text_ingest(manifest, eng, tmp_path):
    """crp_genome_add_fasta_record + k_fasta_strip: tokens rebuilt on the device from the file's own
    bytes equal the tokens of the literal text pipeline, candidates and scores included."""
    from cropsr_b200 import ingest, pipeline
    texts = [open(fixture_path(n), "rb").read() for n in ("sample_genome.fa", "multi3.fa", "edge_fmt.fa", "mid50k.fa")]
    texts.append(synthetic_fasta(11, [70000, 16385, 59, 60, 61, 1], gc=0.45, lower_frac=0.3).encode())
    texts.append(b">one_line\n" + b"ACGGTCCA" * 40 + b"\n>no_final_newline\n" + b"GGCCAATT" * 9 + b"\nGGC")
    for k, data in enumerate(texts):
        path = tmp_path / f"in{k}.fa"
        path.write_bytes(data)
        fast = pipeline.scan_fasta_file(str(path), 20)
        assert fast is not None, k
        keys, scan = fast
        (genome, result, _, _), token_bytes = scan.parts[0], scan.token_bytes
        assert len(scan.parts) == 1
        tokens = ingest.fasta_text_to_tokens(data.decode())
        g2, r2, tb2 = pipeline.scan_tokens(tokens, 20)
        try:
            assert keys == list(tokens.keys())
            assert token_bytes == tb2
            for seg in range(len(keys)):
                for strand in "+-":
                    a, b = result.fetch_segment(seg, strand), r2.fetch_segment(seg, strand)
                    assert np.array_equal(a["pos"], b["pos"]) and np.array_equal(a["packed"], b["packed"])
                    assert np.array_equal(a["x"], b["x"])
        finally:
            for h in (result, genome, r2, g2):
                h.free()


def test_device_fasta_ingest_refuses_text_that_is_not_plain(eng, tmp_path):
    """Ragged lines, blanks or quotes inside the sequence: the device validation answers
    CRP_ERR_FORMAT and the pipeline falls back to the literal host ingest."""
    from cropsr_b200 import pipeline
    # width 61, the line end after line 11 replaced by a base: line 12 starts at base 671, the first base of the
    # 16-byte group of k_fasta_strip at token position 672
    rows = [(b"ACGGTCCATTGA" * 6)[k % 12:k % 12 + 61] for k in range(20)]
    merged = b">a\n" + b"\n".join(rows[:10]) + b"\n" + rows[10] + b"A" + rows[11] + b"\n" + b"\n".join(rows[12:]) + b"\n"
    for k, data in enumerate((b">a\nACGTACGT\nACGT\nACGTACGT\n", b">a\nACGTACGT\nAC GTACG\nAC\n", b">a\nACGTACGT\nAC'TACGT\nAC\n",
                              b">a\nACGTACGT\nACGTACGT\n\n", b">a\nACGTACGT\n\nACGTACGT\n", merged)):
        path = tmp_path / f"bad{k}.fa"
        path.write_bytes(data)
        assert pipeline.scan_fasta_file(str(path), 20) is None, data


def test_cli_csv_same_with_and_without_device_ingest(manifest, eng, tmp_path):
    from cropsr_b200 import pipeline
    case = manifest["cases"]["sample"]
    outs = []
    for dev in (True, False):
        out = tmp_path / f"out{int(dev)}.csv"
        np.random.seed(case["seed"])
        pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out), 20, False,
                          case["blas_threads"], str(tmp_path / "time.txt"), out=lambda *a: None, device_ingest=dev)
        outs.append(out.read_bytes())
    assert outs[0] == outs[1] == golden_csv("sample").encode()


def test_device_logistic_has_numpys_digits(eng):
    """csrc/npexp.cuh: 1 / (1 + np.exp(x)) on the device equals the golden vectors of the reference
    environment's numpy and the CPU oracle bit for bit -- and np.exp on this host if it is an AVX-512 one."""
    from test_oracle_golden import oracle_np_exp
    v = np.load(os.path.join(os.path.dirname(__file__), "golden", "np_exp_vectors.npz"))
    keep = np.abs(v["x"]) < 700
    assert np.array_equal(eng.logistic(v["x"][keep]), v["score"][keep])
    rng = np.random.default_rng(9)
    x = np.concatenate([rng.uniform(-18, 9, 2_000_000), rng.uniform(-700, 700, 200_000), rng.normal(0, 1, 200_000)])
    with np.errstate(all="ignore"):
        want = 1.0 / (1.0 + oracle_np_exp(x))
    got = eng.logistic(x)
    assert np.array_equal(got, want)
    feats = getattr(np._core._multiarray_umath, "__cpu_features__", {})
    if feats.get("AVX512_SKX"):
        assert np.array_equal(got, 1.0 / (1.0 + np.exp(x)))


def test_logistic_flag_stores_the_reference_score(eng):
    """CRP_SCAN_LOGISTIC: the x stream holds 1 / (1 + np.exp(x)) with numpy's digits."""
    from cropsr_b200 import ingest, pipeline, _native as N
    from test_oracle_golden import oracle_np_exp
    tokens = ingest.fasta_text_to_tokens(synthetic_fasta(31, [50000], gc=0.5, lower_frac=0.1))
    g1, r1, _ = pipeline.scan_tokens(tokens, 20)
    g2, r2, _ = pipeline.scan_tokens(tokens, 20, flags=N.CRP_SCAN_LOGISTIC)
    try:
        for strand in "+-":
            x = r1.fetch_segment(0, strand)["x"]
            y = r2.fetch_segment(0, strand)["x"]
            assert len(x) > 100
            assert np.array_equal(y, 1.0 / (1.0 + oracle_np_exp(x)))
    finally:
        for h in (r1, g1, r2, g2):
            h.free()


def test_scan_segments_logistic_equals_scan_score_plus_logistic(eng):
    """crp_scan_segments with CRP_SCAN_LOGISTIC: the rows leave on their own stream, and must be the
    rows AFTER the logistic pass the lane queued (ADVICE r1: the copy used to race the pass)."""
    from cropsr_b200 import engine, ingest, _native as N
    toks = [np.frombuffer(v.encode(), np.uint8) for v in
            ingest.fasta_text_to_tokens(synthetic_fasta(41, [300000, 70000, 120000], gc=0.5, lower_frac=0.1)).values()]
    segs = [(k, t, 0, None) for k, t in enumerate(toks)]
    for _ in range(3):
        a_plain, np_, nm_, _ms = engine.scan_segments(segs, 20)
        a_log, lp, lm, _ms = engine.scan_segments(segs, 20, flags=N.CRP_SCAN_LOGISTIC)
        assert np.array_equal(np_, lp) and np.array_equal(nm_, lm)
        for strand, n in (("+", int(np_.sum())), ("-", int(nm_.sum()))):
            x = a_plain.arrays[strand]["x"][:n]
            y = a_log.arrays[strand]["x"][:n]
            assert n > 1000 and np.array_equal(y, engine.logistic(x))
            assert np.array_equal(a_plain.arrays[strand]["pos"][:n], a_log.arrays[strand]["pos"][:n])
        a_plain.free()
        a_log.free()


def test_many_scaffolds_match_oracle(eng):
    """configs[4] shape in small: hundreds of scaffolds, some shorter than one window, some a
    few tiles long -- per-segment counts, order and scores against the oracle."""
    rng = np.random.default_rng(77)
    lengths = [int(x) for x in rng.integers(1, 3000, size=300)] + [40000, 16384, 16385, 1, 29, 30, 31, 52, 53]
    _check_against_oracle(eng, synthetic_fasta(78, lengths, gc=0.5, lower_frac=0.2, n_frac=0.002, width=60), 20)


def test_reference_callables_on_the_device(eng):
    """CROPSR.find_PAM_site and CROPSR.rs1_score (SURVEY 8b) against the regex and against the
    oracle's np.matmul / np.exp port of the reference function, for every row-count class."""
    import re
    import CROPSR
    rng = np.random.default_rng(21)
    for n in (0, 1, 2, 3, 5, 7, 40, 3000, 70001):
        tok = "".join(rng.choice(list("ACGTacgtN"), size=n, p=[.2, .2, .22, .22, .04, .04, .03, .03, .02]))
        for pat in ("(?=.GG)", "(?=CC.)"):
            assert CROPSR.find_PAM_site(pat, tok) == [m.span() for m in re.finditer(pat, tok)], (n, pat)
    tok = "GGGGGGGGCCCCCCCC" + "'),"
    for pat in ("(?=.GG)", "(?=CC.)"):
        assert CROPSR.find_PAM_site(pat, tok) == [m.span() for m in re.finditer(pat, tok)]
    alphabet = np.frombuffer(b"ATCGNatcg'", dtype=np.uint8)
    for n in (1, 2, 3, 4, 5, 6, 7, 8, 9, 4098, 4099):
        seqs = rng.choice(alphabet, size=(n, 30), p=[.23, .23, .23, .23, .02, .01, .01, .01, .01, .02])
        got = CROPSR.rs1_score(seqs)
        assert np.array_equal(got, oracle.score_model(seqs, threads=1)), n
        feats = getattr(np._core._multiarray_umath, "__cpu_features__", {})
        if feats.get("AVX512_SKX") and os.environ.get("OPENBLAS_NUM_THREADS") == "1":
            assert np.array_equal(got, oracle.score_blas(seqs)), n       # the reference function itself
    # a placeholder row (CROPSR.py:459, np.empty(30,)) turns the reference's matrix into float64
    ph = np.array([np.frombuffer(b"ACGT" * 7 + b"AC", np.uint8), np.full(30, 1e-310)])
    conv = np.array([np.frombuffer(b"ACGT" * 7 + b"AC", np.uint8), np.zeros(30, np.uint8)])
    assert ph.dtype == np.float64
    assert np.array_equal(CROPSR.rs1_score(ph), oracle.score_model(conv, threads=1))


@pytest.mark.parametrize("name", ["big1", "big2"])
def test_cli_over_one_million_candidates_equals_reference_digest(name, eng, tmp_path):
    """SURVEY 8a row 10 end to end: more than 1,000,000 candidates through the reference's chunk
    plan (misplaced last slice, ids[start-k-1] with start > 0; big2: cumulative re-emission across
    the 1e6 boundary and 8-thread BLAS row classes of a 1e6-row matmul).  The golden is the sha256
    of the CSV the UNMODIFIED reference wrote for the same seeded FASTA
    (tests/golden/make_big_golden.py -> cases/big_manifest.json)."""
    import hashlib, importlib.util, json
    from cropsr_b200 import pipeline
    here = os.path.dirname(fixture_path("x"))
    spec = importlib.util.spec_from_file_location("make_big_golden", os.path.join(here, "..", "make_big_golden.py"))
    mbg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mbg)
    with open(os.path.join(here, "..", "cases", "big_manifest.json")) as f:
        case = json.load(f)["cases"][name]
    text = mbg.big_fasta(name)
    assert hashlib.sha256(text.encode()).hexdigest() == case["fasta_sha256"]
    fa = tmp_path / (name + ".fa")
    with open(fa, "w", newline="") as f:
        f.write(text)
    out = tmp_path / "out.csv"
    np.random.seed(case["seed"])
    stats = pipeline.run_cas9(str(fa), fixture_path("sample_genome.gff"), str(out), 20, False, case["blas_threads"],
                              str(tmp_path / "time.txt"), out=lambda *a: None)
    data = out.read_bytes()
    assert data.count(b"\r\n") - 1 == case["rows"] == stats["rows"]
    if hashlib.sha256(data).hexdigest() != case["csv_sha256"]:
        # say which layer differs before failing: structure, then scores to 12 digits, then raw bytes
        text = data.decode()
        assert normalised_digest(text) == case["digest_no_id_no_score"], "rows / sequences / coordinates differ"
        assert normalised_digest(text, "%.12g") == case["digest_no_id_score_12g"], "scores differ beyond 1e-12"
        raise AssertionError("ids or last score digits differ from the reference's CSV")


def test_several_genome_handles_give_the_same_csv(manifest, eng, tmp_path):
    """Genomes beyond the 32-bit limits of one handle (ADVICE r1: the 10 Gbp config) are spread
    over several handles: with the per-handle limit shrunk, tokens of multi3 / sample land in
    different handles, rows come from the host rescorer, and the CSV stays byte-identical --
    through both ingests."""
    from cropsr_b200 import pipeline
    for name, limit in (("multi3", 1), ("multi3_c20", 3000), ("mid50k_t5", 100), ("sample_c5000_t4", 1000)):
        case = manifest["cases"][name]
        for dev in (True, False):
            out = tmp_path / f"{name}_{dev}.csv"
            np.random.seed(case["seed"])
            pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out), case["guide_len"],
                              False, case["blas_threads"], str(tmp_path / "time.txt"), out=lambda *a: None,
                              device_ingest=dev, chunk_rows=case.get("chunk"), handle_limit=limit)
            assert out.read_bytes().decode() == golden_csv(name), (name, dev)


def test_host_rescorer_equals_crp_rescore(eng):
    """HostRescorer (30 scored bytes from the host token through crp_rs1_preactivation) against
    crp_rescore (packed records) for every class pair, both strands, tile-edge candidates included."""
    from cropsr_b200 import ingest, pipeline
    tokens = ingest.fasta_text_to_tokens(synthetic_fasta(52, [40000, 17000], gc=0.5, lower_frac=0.2, n_frac=0.003))
    genome, result, token_bytes = pipeline.scan_tokens(tokens, 20)
    host = pipeline.HostRescorer(token_bytes)
    try:
        for seg in range(2):
            for strand in "+-":
                pos = result.fetch_segment(seg, strand, want=("pos",))["pos"][:600]
                for cls in (0x00, 0x01, 0x10, 0x11, 0x02, 0x20, 0x22, 0x12, 0x21):
                    c = np.full(len(pos), cls, np.uint8)
                    st = np.full(len(pos), strand.encode(), "S1")
                    sg = np.full(len(pos), seg, np.uint32)
                    assert np.array_equal(genome.rescore(sg, pos, st, c), host.rescore(sg, pos, st, c)), (seg, strand, cls)
    finally:
        result.free()
        genome.free()


@pytest.mark.parametrize("exchange", ["fused", "nccl"])
@pytest.mark.parametrize("n_dev", [2, 3, 8])
def test_multi_gpu_cli_writes_the_reference_csv(n_dev, exchange, manifest, eng, tmp_path, monkeypatch):
    """CROPSR.py --devices 0-(n-1): one process per GPU, contiguous shards, the NCCL all-gather of the
    per-segment counts inside the library, rows placed in reference order -- the CSV must be the
    unmodified reference's, byte for byte.  Needs n GPUs on the box (gpurun --gpus n)."""
    from cropsr_b200 import pipeline
    if eng.device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    monkeypatch.setenv("CRP_COMM_EXCHANGE", exchange)      # read by crp_comm_init in every rank (workers inherit it)
    names = ("multi3", "sample", "mid50k_t5", "multi3_c20", "edge_fmt", "empty_records", "single_candidate")
    if n_dev > 2:           # every case spawns n_dev processes (CUDA context + NCCL init each, 10-30 s per case on a
        names = ("multi3", "sample", "empty_records")        # 4- or 8-GPU box): keep the big boxes short
    for name in names:
        case = manifest["cases"][name]
        out = tmp_path / f"{name}.csv"
        np.random.seed(case["seed"])
        stats = pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out), case["guide_len"],
                                  False, case["blas_threads"], str(tmp_path / "time.txt"), out=lambda *a: None,
                                  chunk_rows=case.get("chunk"), devices=list(range(n_dev)))
        assert out.read_bytes().decode() == golden_csv(name), name
        assert len(stats["ranks"]) == n_dev
        if exchange == "nccl":
            assert not any(r["fused_exchange"] for r in stats["ranks"])
        else:       # fused wherever the peers could be mapped; the note says why not otherwise
            assert all(r["fused_exchange"] or r["exchange_note"] for r in stats["ranks"]), stats["ranks"]


def _gpu_table_digest(eng, workload, limit=None):
    """digest of the device's unique-candidate table of a whole synthetic config (oracle/vector_oracle.TableDigest)"""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
    import vector_oracle as vo
    import workloads as W
    from cropsr_b200 import pipeline
    lengths = W.token_lengths(workload)
    d = vo.TableDigest()
    for first, cnt in pipeline._groups(lengths, limit):
        g = eng.Genome()
        for k in range(first, first + cnt):
            g.add_token(W.token(workload, k))
        g.commit()
        r = g.scan(20)
        plus, minus = r.fetch("+"), r.fetch("-")
        for s in range(cnt):
            a, b = int(r.off_plus[s]), int(r.off_plus[s + 1])
            c, e = int(r.off_minus[s]), int(r.off_minus[s + 1])
            d.add_token(first + s, (plus["pos"][a:b], plus["packed"][a:b], plus["x"][a:b]),
                        (minus["pos"][c:e], minus["packed"][c:e], minus["x"][c:e]))
        r.free()
        g.free()
    return d


def _table_digests():
    import json
    with open(os.path.join(os.path.dirname(fixture_path("x")), "..", "table_digests.json")) as f:
        return json.load(f)


def test_whole_candidate_table_of_configs1_equals_oracle_digest(eng):
    """configs[1], all 5 chromosomes, 135 Mbp / 7.37 M candidates: pos, packed 30-mer and fp64 x of EVERY
    candidate against the vectorised oracle's committed digest (tests/golden/make_table_digests.py)."""
    want = _table_digests()["arabidopsis"]
    d = _gpu_table_digest(eng, "arabidopsis")
    assert (d.tokens, d.candidates) == (want["tokens"], want["candidates"])
    assert d.hexdigest() == want["sha256"]


@pytest.mark.slow
@pytest.mark.parametrize("workload", ["sorghum", "maize", "sugarcane"])
def test_whole_candidate_table_of_larger_configs_equals_oracle_digest(eng, workload):
    """configs[2..4] (60 % lower-case; repeats + N runs; 20,100 records / 10.5 Gbp over several genome handles):
    the same whole-table digest.  Minutes of host-side generation and hashing, so CROPSR_SLOW=1."""
    want = _table_digests().get(workload)
    if want is None:
        pytest.skip("digest not generated yet")
    d = _gpu_table_digest(eng, workload)
    assert (d.tokens, d.candidates) == (want["tokens"], want["candidates"])
    assert d.hexdigest() == want["sha256"]


def test_many_scaffolds_cli_and_batched_side_outputs(eng, tmp_path):
    """configs[4] shape in small through the whole CLI: 1,500 records, most of them shorter than one
    window, a few with candidates -- the cumulative re-emission (CROPSR.py:407,442) then writes ~10^5 rows.
    Byte-identical to the oracle; and the whole-strand side-output calls (one per strand instead of one
    per segment) return what the per-segment calls return."""
    import io
    from cropsr_b200 import ingest, pipeline
    rng = np.random.default_rng(91)
    lengths = [int(x) for x in rng.integers(5, 29, size=1500)]
    for k in rng.choice(1500, size=30, replace=False):
        lengths[int(k)] = int(rng.integers(150, 400))
    text = synthetic_fasta(92, lengths, gc=0.5, lower_frac=0.2, n_frac=0.0, width=60)
    fa = tmp_path / "scaffolds.fa"
    with open(fa, "w", newline="") as f:
        f.write(text)
    out = tmp_path / "out.csv"
    np.random.seed(5)
    stats = pipeline.run_cas9(str(fa), fixture_path("sample_genome.gff"), str(out), 20, False, 1, str(tmp_path / "time.txt"),
                              out=lambda *a: None)
    np.random.seed(5)
    want = oracle.run_to_string(text, 20, "model", 1)
    assert out.read_bytes().decode() == want
    assert stats["tokens"] == 1500 and stats["rows"] > 20 * stats["candidates"]
    # whole-strand calls == per-segment calls
    tokens = ingest.fasta_text_to_tokens(text)
    genome, result, _ = pipeline.scan_tokens(tokens, 20)
    try:
        n_seg = len(tokens)
        ivs = [(np.sort(rng.integers(0, max(len(t), 1), size=3)).astype(np.uint32)) for t in tokens.values()]
        iv_off = np.arange(0, 3 * n_seg + 1, 3, dtype=np.uint64)
        start = np.concatenate(ivs)
        end = start + np.uint32(40)
        for strand in "+-":
            whole = result.extras_strand(strand, 200)
            feat = result.annotate_strand(strand, iv_off, start, end)
            off = result.off_plus if strand == "+" else result.off_minus
            for seg in range(n_seg):
                a, b = int(off[seg]), int(off[seg + 1])
                if a == b:
                    continue
                one = result.extras(seg, strand, 200)
                for key in one:
                    assert np.array_equal(whole[key][a:b], one[key]), (seg, strand, key)
                assert np.array_equal(feat[a:b], result.annotate(seg, strand, start[3 * seg:3 * seg + 3], end[3 * seg:3 * seg + 3]))
    finally:
        result.free()
        genome.free()


def test_pipelined_call_groups_small_segments(eng):
    """crp_scan_segments puts consecutive small segments into one genome handle (one commit + one scan
    per group): 5,000 short records and two long ones, counts per segment and rows in segment order
    equal the plain scan's."""
    from cropsr_b200 import engine, ingest
    rng = np.random.default_rng(17)
    lengths = [int(x) for x in rng.integers(1, 700, size=5000)]
    lengths[777] = 400000
    lengths[3100] = 18 << 20          # a group of its own (>= 16 MiB)
    text = synthetic_fasta(18, lengths, gc=0.5, lower_frac=0.1, n_frac=0.0)
    toks = [np.frombuffer(v.encode(), np.uint8) for v in ingest.fasta_text_to_tokens(text).values()]
    arena, n_plus, n_minus, _ = engine.scan_segments([(k, t, 0, None) for k, t in enumerate(toks)], 20)
    g = engine.Genome()
    for t in toks:
        g.add_token(t)
    r = g.commit().scan(20)
    try:
        assert np.array_equal(n_plus, r.seg_plus) and np.array_equal(n_minus, r.seg_minus)
        for strand, n in (("+", r.n_plus), ("-", r.n_minus)):
            want = r.fetch(strand)
            for name in ("pos", "packed", "x"):
                assert np.array_equal(arena.arrays[strand][name][:n], want[name]), (strand, name)
    finally:
        arena.free()
        r.free()
        g.free()


def test_checked_build_sees_no_violated_invariant(eng):
    """libcropsr_b200_checked.so (make checked, -DCRP_CHECKED): k_scan_score verifies its own invariants --
    hit-list, record, ring and stream indices, ascending positions, and that the emit phase finds in every
    warp chunk exactly the hits the count phase counted -- and a violated one fails the scan.  The small
    cases with the most edges (tile borders, dense tiles, long count ranges with 1-7 CTAs, static / ticketed
    dealing, the edge fixtures, many scaffolds) run under it in a subprocess.  (compute-sanitizer is closed
    on the GPU pool this was developed on: profiles/README.md.)"""
    import subprocess, sys
    root = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
    lib = os.path.join(root, "cropsr_b200", "libcropsr_b200_checked.so")
    if not os.path.exists(lib):
        pytest.skip("checked library not built (make -C cropsr_b200/csrc checked)")
    if os.environ.get("CROPSR_B200_LIB"):
        return                      # already inside such a subprocess
    env = dict(os.environ, CROPSR_B200_LIB=lib)
    probe = subprocess.run([sys.executable, "-c", "from cropsr_b200 import _native as N; print(N.lib.crp_checked_build())"],
                           cwd=root, env=env, capture_output=True, text=True, timeout=120)
    assert probe.stdout.strip() == "1", probe.stderr[-1000:]
    sel = ("test_tile_boundaries or test_long_count_ranges or test_static_and_ticketed or test_many_scaffolds_match or "
           "test_random_fastas or test_sharded_scan or test_pipelined or (test_candidate_streams and (edge or multi3 or mid50k))")
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "tests/test_gpu_parity.py", "-k", sel],
                         cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]


def test_perf_report_counts_what_ran(eng):
    from cropsr_b200 import ingest, pipeline
    before = eng.perf_report()
    tokens = ingest.fasta_text_to_tokens(synthetic_fasta(61, [50000, 20000], gc=0.5))
    genome, result, _ = pipeline.scan_tokens(tokens, 20)
    n = result.n_plus + result.n_minus
    result.fetch("+")
    result.free()
    genome.free()
    after = eng.perf_report()
    assert after["commits"] == before["commits"] + 1 and after["scans"] == before["scans"] + 1
    assert after["candidates"] == before["candidates"] + n
    assert after["positions_packed"] == before["positions_packed"] + sum(len(t) for t in tokens.values())
    assert after["kernel_launches"] >= before["kernel_launches"] + 2 and after["d2h_row_bytes"] > before["d2h_row_bytes"]


def test_gap_table_matches_oracle(eng, tmp_path):
    """Genome.other_runs (k_other_runs: runs of bytes that are not ACGTacgt, read off the `other` plane of the
    packed records) against the string oracle: N runs across tile edges, at the token ends, IUPAC singletons,
    the decoration of formatted-path tokens, several segments of one token."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
    import extras_oracle
    from cropsr_b200 import engine, ingest
    rng = np.random.default_rng(5)
    body = bytearray(synthetic_fasta(6, [70000], gc=0.5, lower_frac=0.3, n_frac=0.0005, width=10**9).split("\n")[1].encode())
    for lo, n in ((0, 7), (16380, 9), (16384 * 2 - 3, 40), (32768, 1), (40000, 5000), (69990, 10)):
        body[lo:lo + n] = b"N" * n
    text = ">g\n" + "\n".join(body.decode()[i:i + 80] for i in range(0, len(body), 80)) + "\n>h\nNNACGTNN\n>i\nACGT\n"
    tokens = ingest.fasta_text_to_tokens(text)
    g = engine.Genome()
    for tok in tokens.values():
        g.add_token(tok)
    g.commit()
    try:
        for seg, tok in enumerate(tokens.values()):
            for min_len in (1, 4, 10):
                start, length = g.other_runs(seg, min_len)
                assert list(zip(start.tolist(), length.tolist())) == extras_oracle.other_runs(tok, min_len), (seg, min_len)
    finally:
        g.free()
    # one token cut into tile-aligned segments: the runs of the pieces, clipped at the cuts, tile the token's runs
    tok = list(tokens.values())[0]
    g = engine.Genome()
    cuts = [0, 16384, 49152, len(tok)]
    for a, b in zip(cuts, cuts[1:]):
        g.add_segment(0, tok, a, b)
    g.commit()
    try:
        covered = np.zeros(len(tok), bool)
        for seg in range(3):
            for a, n in zip(*[x.tolist() for x in g.other_runs(seg, 1)]):
                assert cuts[seg] <= a and a + n <= cuts[seg + 1] and not covered[a:a + n].any()
                covered[a:a + n] = True
        want = np.zeros(len(tok), bool)
        for a, n in extras_oracle.other_runs(tok, 1):
            want[a:a + n] = True
        assert np.array_equal(covered, want)
    finally:
        g.free()
