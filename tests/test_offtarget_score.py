"""Off-target scores (csrc/offtarget.cuh k_ot_join<OtScore> / ot_mask_rank, crp_offtarget_score_candidates / score_keys,
engine.mit_weights / mit_specificity / OffTargetIndex.score_candidates / score_guides, pipeline.write_offtarget_scores,
--offtarget-scores).

CPU: the MIT transcription pinned by checkpoints and digests, the oracle pinned by hand on the hand-built genome, the
rank and pair rule of the kernel emulated on the host (tests/offtarget_score_emu.cu), the CLI refusals.
GPU: sums against the string oracle (fixtures, several genome handles, MIT and random weight tables, guides), indicator
tables against the counts at configs[1] size, the table through run_cas9 and the CLI, the error codes."""
import hashlib
import os
import shutil
import subprocess
from math import comb

import numpy as np
import pytest

import cropsr_oracle as oracle
import offtarget_score_oracle as sco
from helpers import ROOT, fixture_path, fixture_text, golden_csv

# ---------------------------------------------------------------- the hand-built genome of test_offtarget.py
GUIDE = "GATTACAGCTTCAGTCATCA"
FILL = "T" * 30


def _sub(guide, positions):
    g = list(guide)
    for p in positions:
        g[p] = "T" if g[p] == "A" else "A"
    return "".join(g)


def _rc(s):
    return s[::-1].translate(str.maketrans("ACGTacgt", "TGCAtgca"))


def hand_tokens():
    """chrA: d0 (a quote in the window: no site) at 20, c0 exact '+' AGG at 73, c1 1 substitution (position 3) at
    126, c2 2 substitutions (7, 11) on '-' at 159, c3 3 substitutions (0, 15, 19) lower case with tgg at 232, c4 exact
    with a lower-case gg (a site, not a candidate) at 285, c5 4 substitutions at 338, c6 an N inside at 391.
    chrB: e0 exact CGG at 50, then a '-' copy cut off by the token end."""
    t1 = ("'" + GUIDE[1:] + "AGG" + FILL
          + GUIDE + "AGG" + FILL
          + _sub(GUIDE, [3]) + "AGG" + FILL
          + "CCT" + _rc(_sub(GUIDE, [7, 11])) + FILL
          + _sub(GUIDE, [0, 15, 19]).lower() + "tgg" + FILL
          + GUIDE + "Agg" + FILL
          + _sub(GUIDE, [1, 5, 9, 13]) + "AGG" + FILL
          + GUIDE[:10] + "N" + GUIDE[11:] + "AGG" + FILL
          + "'),")
    t2 = FILL + GUIDE + "CGG" + FILL + "CCA" + _rc(GUIDE)[:18]
    return {">chrA": t1, ">chrB": t2}


M_SHA256 = "7a741c30e0a5fe15b0b1466a55be32fa9ed8dad25fa7a9a722b7a4a7499071a2"
TABLE_SHA256 = "d96f7a465e290649529bfb8b3711cddf62572dc83f1311bc059fa69d7670a407"


def rank(positions):
    """colex rank of an ascending position set of size <= 3 (include/cropsr_b200.h)"""
    return [0, 1, 21, 211][len(positions)] + sum(comb(p, e + 1) for e, p in enumerate(positions))


def all_sets():
    from itertools import combinations
    return sorted((c for d in range(4) for c in combinations(range(20), d)), key=rank)


def test_mit_transcription_checkpoints(built_lib):
    from cropsr_b200 import engine
    assert hashlib.sha256(np.array(sco.M, dtype="<f8").tobytes()).hexdigest() == M_SHA256
    assert hashlib.sha256(np.array(engine.MIT_M, dtype="<f8").tobytes()).hexdigest() == M_SHA256
    sets = all_sets()
    assert len(sets) == 1351 and [rank(s) for s in sets] == list(range(1351))
    assert engine.score_sets() == sets
    oracle_table = np.array([sco.mit_weight(s) for s in sets], dtype="<u4")
    table = engine.mit_weights()
    assert table.dtype == np.uint32 and np.array_equal(table, oracle_table)
    assert hashlib.sha256(table.astype("<u4").tobytes()).hexdigest() == TABLE_SHA256
    assert len(np.unique(table)) == 1216 and int(table.max()) == 1677721600 == 100 << 24
    for positions, value in [((), 100.0), ((0,), 100.0), ((19,), 41.7), ((0, 19), 10.425), ((12, 13), 0.3009881868131869),
                             ((5, 6, 7), 0.9586184371184372), ((2, 9, 17), 0.578083204102564)]:
        assert sco.hit(positions) == value == engine.mit_hit(positions), positions
    assert table[rank((19,))] == 699609907 == sco.mit_weight((19,))


def test_mit_specificity_rounds_and_passes_no_score_through(built_lib):
    from cropsr_b200 import engine
    no = engine.OffTargetIndex.NO_SCORE
    sums = np.array([0, 100 << 24, 300 << 24, no, 1 << 24, 303 * (1 << 24) + 3756], dtype=np.uint64)
    assert engine.mit_specificity(sums).tolist() == [100, 50, 25, no, 99, 25]
    assert engine.mit_specificity(sums).tolist()[:3] == [sco.specificity(int(s)) for s in sums[:3]]


def test_hand_built_score_rows_are_what_the_definition_says():
    """c0 (and e0, its copy on chrB) is hit by two exact copies (100 each), c1 at {3} (M[3] = 0: 100), c2 at {7, 11}
    (0.492 * 19/79 / 4 * 100) and c3 at {0, 15, 19} (0.172 * 0.417 / 3 / 9 * 100); c5 (4 substitutions) has no pair."""
    h711, h3711, h01519 = 0.492 * 19 / 79 / 4 * 100, 0.492 * 19 / 79 / 9 * 100, 0.172 * 0.417 / 3 / 9 * 100
    assert sco.hit((7, 11)) == pytest.approx(h711, rel=1e-12)
    assert sco.hit((3, 7, 11)) == pytest.approx(h3711, rel=1e-12)
    assert sco.hit((0, 15, 19)) == pytest.approx(h01519, rel=1e-12)
    # the table sums the fixed-point weights (2**-24 each), so its last digit may differ from these float sums
    assert 300 + h711 + h01519 == pytest.approx(303.223872, abs=1e-6)
    assert 300 + h3711 == pytest.approx(301.314768, abs=1e-6)
    assert 3 * h711 + h3711 == pytest.approx(10.189452, abs=1e-6)
    assert sco.scores_table(hand_tokens(), 3).split("\r\n") == [
        "chromosome\tstrand\tpam_pos\tprotospacer\tmit_hit_sum\tmit_specificity",
        "chrA\t+\t73\tGATTACAGCTTCAGTCATCA\t303.223872\t25",       # c0: c4, e0, c1, c2, c3
        "chrA\t+\t126\tGATAACAGCTTCAGTCATCA\t301.314768\t25",      # c1: c0, c4, e0 at {3}, c2 at {3, 7, 11}
        "chrA\t+\t338\tGTTTAAAGCATCAATCATCA\t0.000000\t100",       # c5: nothing within 3
        "chrA\t+\t391\t\t\t",                                      # c6: N in the protospacer
        "chrA\t-\t159\tGATTACAACTTAAGTCATCA\t10.189452\t91",       # c2: three copies at {7, 11}, c1 at {3, 7, 11}
        "chrB\t+\t50\tGATTACAGCTTCAGTCATCA\t303.223872\t25",       # e0 mirrors c0
        "chrB\t-\t83\t\t\t",                                       # cut off by the token end
        ""]
    assert sco.scores_table(hand_tokens(), 1).split("\r\n")[1:3] == [
        "chrA\t+\t73\tGATTACAGCTTCAGTCATCA\t300.000000\t25", "chrA\t+\t126\tGATAACAGCTTCAGTCATCA\t300.000000\t25"]
    # random weights: the oracle sums the table entry of each pair's set, the own site (rank 0) left out
    w = np.arange(1351, dtype=np.int64) * 7 + 5
    row = sco.candidate_sums(list(hand_tokens().values()), 3, lambda s: int(w[rank(s)]))[0]
    assert row[4] == 2 * w[0] + w[rank((3,))] + w[rank((7, 11))] + w[rank((0, 15, 19))]


def test_score_rank_and_pair_rule_on_the_cpu(tmp_path):
    """tests/offtarget_score_emu.cu compiles ot_mask_rank and the pair rule of k_ot_join -- the SAME
    source -- for the host and checks every part pair against all 1,351 mismatch-position sets of size <= 3."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "offtarget_score_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "offtarget_score_emu.cu")], check=True, capture_output=True, timeout=600)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


@pytest.mark.parametrize("argv, why", [(["-l", "18"], "20-base guides"), (["--devices", "0-1"], "one GPU"),
                                       (["--mismatches", "4"], "0 to 3"), (["--mismatches", "-1"], "0 to 3")])
def test_cli_refuses_offtarget_scores_before_any_device_work(built_lib, argv, why):
    from cropsr_b200 import cli, engine
    with pytest.raises(SystemExit) as e:
        cli.main(["-f", "missing.fa", "--cas9", "--offtarget-scores", "out.tsv"] + argv)
    assert "--offtarget-scores" in str(e.value.code) and why in str(e.value.code)
    assert engine._device is None


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def _scan(tokens, limit=None):
    from cropsr_b200 import pipeline
    return pipeline.scan_token_bytes([v.encode("ascii") for v in tokens.values()], 20, limit=limit)


def _device_sums(eng, scan, k, weights):
    """(token, strand, t, sum or None) in reference order, from one index over all handles"""
    index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts])
    rows = []
    try:
        for g, r, first, cnt in scan.parts:
            per = {}
            for strand in "+-":
                pos = r.fetch(strand, want=("pos",))["pos"]
                per[strand] = (pos, index.score_candidates(r, strand, k, weights), r.off_plus if strand == "+" else r.off_minus)
            for s in range(cnt):
                for strand in "+-":
                    pos, c, off = per[strand]
                    for i in range(int(off[s]), int(off[s + 1])):
                        rows.append((first + s, strand, int(pos[i]), None if c[i] == index.NO_SCORE else int(c[i])))
    finally:
        index.free()
    return rows


def _same(got, want):
    """True, or (rows that differ, the first of them as (got, want)): a short message when nearly every row differs"""
    if got == want:
        return True
    bad = [i for i, (x, y) in enumerate(zip(got, want)) if x != y]
    return len(got), len(want), len(bad), (got[bad[0]], want[bad[0]]) if bad else None


def _tables():
    """(name, uint32 table): MIT and two seeded random tables below 2**31"""
    from cropsr_b200 import engine
    rng = np.random.default_rng(41)
    return [("mit", engine.mit_weights()),
            ("random", rng.integers(0, 1 << 31, size=1351, dtype=np.uint32)),
            ("random_small", rng.integers(0, 1000, size=1351, dtype=np.uint32))]


def _oracle_sums(pairs, k, table):
    return [(a, b, c, e) for a, b, c, _, e in sco.candidate_sums(None, k, lambda s: int(table[rank(s)]), pairs)]


@pytest.mark.gpu
@pytest.mark.parametrize("fasta", ["hand", "multi3.fa", "clean3.fa", "edge_fmt.fa", "edge_clean.fa", "sample_genome.fa"])
def test_candidate_scores_equal_oracle(eng, fasta):
    tokens = hand_tokens() if fasta == "hand" else oracle.import_fasta_text(fixture_text(fasta))
    scans = [_scan(tokens)] + ([_scan(tokens, limit=1)] if len(tokens) > 1 else [])
    try:
        if len(scans) > 1:
            assert len(scans[1].parts) > 1
        pairs = sco.candidate_pairs(list(tokens.values()), 3)
        for k in range(4):
            for name, table in _tables():
                want = _oracle_sums(pairs, k, table)
                for scan in scans:
                    assert _same(_device_sums(eng, scan, k, table), want) is True, (k, name, len(scan.parts))
        if fasta == "hand":                                    # NO_SCORE rows: the N and the cut-off copy
            assert sum(1 for *_, s in want if s is None) == 2
    finally:
        for scan in scans:
            scan.free()


@pytest.mark.gpu
def test_score_guides_equal_oracle(eng):
    tokens = oracle.import_fasta_text(fixture_text("sample_genome.fa"))
    scan = _scan(tokens)
    try:
        index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts])
        import offtarget_oracle as ot
        present = [ot.protospacer(tok, t, s) for tok in tokens.values() for t, s, _ in ot.sites(tok)[:25]]
        rng = np.random.default_rng(5)
        absent = ["".join(rng.choice(list("ACGT"), 20)) for _ in range(10)]
        guides = present + [p.lower() for p in present[:8]] + absent
        for k in range(4):
            for name, table in _tables():
                got = index.score_guides(guides, k, table)
                want = sco.guide_sums(list(tokens.values()), guides, k, lambda s: int(table[rank(s)]))
                assert got.tolist() == want, (k, name)
        assert index.score_guides([], 3).shape == (0,)
        assert index.score_guides(absent, 0).tolist() == [0] * len(absent)
        index.free()
    finally:
        scan.free()


def _check_indicator_tables(index, results):
    """weight 1 for the sets of size d and 0 for the rest gives mm_d of count_candidates, for every d <= k; all ones
    gives their sum; NO_SCORE exactly where NO_COUNT.  -> total pairs per d at k = 3"""
    sizes = np.array([len(s) for s in all_sets()])
    totals = np.zeros(4, np.int64)
    for r in results:
        for strand in "+-":
            for k in (1, 3):
                counts = index.count_candidates(r, strand, k)
                ok = counts[:, 0] != index.NO_COUNT
                for d in range(k + 1):
                    got = index.score_candidates(r, strand, k, (sizes == d).astype(np.uint32))
                    assert np.array_equal(got[~ok], np.full((~ok).sum(), index.NO_SCORE, np.uint64))
                    assert np.array_equal(got[ok], counts[ok, d].astype(np.uint64)), (strand, k, d)
                got = index.score_candidates(r, strand, k, np.ones(1351, np.uint32))
                assert np.array_equal(got[ok], counts[ok].astype(np.uint64).sum(axis=1)), (strand, k)
            totals += counts[ok].astype(np.int64).sum(axis=0)
    return totals


@pytest.mark.gpu
def test_configs1_indicator_tables_reproduce_the_counts(eng):
    """configs[1] (arabidopsis, 135 Mbp): the indicator tables against the counts on every candidate of both strands."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import workloads as W
    genomes, results = [], []
    index = eng.OffTargetIndex()
    try:
        for t in range(len(W.token_lengths("arabidopsis"))):
            g = eng.Genome()
            g.add_token(W.token("arabidopsis", t))
            g.commit()
            genomes.append(g)
            results.append(g.scan(20))
            index.add_genome(g)
        assert (_check_indicator_tables(index, results) > 0).all()
    finally:
        index.free()
        for x in results + genomes:
            x.free()


@pytest.mark.gpu
def test_indicator_tables_in_a_bucket_with_more_than_100k_sites(eng):
    """The tandem genome of test_offtarget.py: one bucket of every part pair holds > 10^5 sites, so a query's pairs
    come from many site tiles and every thread of a work item flushes many hits."""
    from cropsr_b200 import pipeline
    n_units = 120_000
    unit = "atcgatcagg"
    rng = np.random.default_rng(7)
    units = [unit] * n_units
    for i in rng.choice(n_units, size=200, replace=False):
        units[i] = unit.upper()
    for i in rng.choice(n_units, size=100, replace=False):
        u = list(units[i])
        u[int(rng.integers(0, 7))] = "t" if u[0].islower() else "T"
        units[i] = "".join(u)
    tok = "ACGTTGCA" + "".join(units) + "TTGCA"
    scan = pipeline.scan_token_bytes([tok.encode()], 20)
    try:
        index = eng.OffTargetIndex([scan.parts[0][0]])
        assert index.num_sites() > 100_000
        totals = _check_indicator_tables(index, [scan.parts[0][1]])
        assert totals[0] > 150 * 100_000 and totals[1] > 0
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_errors(eng):
    from cropsr_b200 import _native as N
    from cropsr_b200.engine import lib
    tokens = hand_tokens()
    scan = _scan(tokens)
    g, r, _, _ = scan.parts[0]
    index = eng.OffTargetIndex([g])
    try:
        w = eng.mit_weights()
        for k, at in ((3, 1350), (1, 20), (0, 0)):
            bad = w.copy()
            bad[at] = 1 << 31
            for call in (lambda: index.score_candidates(r, "+", k, bad), lambda: index.score_guides([GUIDE], k, bad)):
                with pytest.raises(N.CropsrError) as e:
                    call()
                assert e.value.code == -2
        ignored = w.copy()
        ignored[21:] = 0xFFFFFFFF                                  # sets of size 2 and 3 are not read at k = 1
        assert np.array_equal(index.score_candidates(r, "+", 1, ignored), index.score_candidates(r, "+", 1, w))
        for call in (lambda: index.score_candidates(r, "+", 4), lambda: index.score_guides([GUIDE], 4)):
            with pytest.raises(N.CropsrError) as e:
                call()
            assert e.value.code == -2
        out = np.zeros(8, np.uint64)
        assert lib.crp_offtarget_score_candidates(index._h, r._h, b"+", 3, None, out.ctypes.data) == -2
        with pytest.raises(ValueError):
            index.score_candidates(r, "+", 3, w[:100])
    finally:
        index.free()
        scan.free()


def _run(case_fasta, d, k, device_ingest, seed, blas, scores=True, counts=True, sites=True):
    from cropsr_b200 import pipeline
    d.mkdir()
    np.random.seed(seed)
    pipeline.run_cas9(fixture_path(case_fasta), fixture_path("sample_genome.gff"), str(d / "out.csv"), 20, False, blas,
                      str(d / "time.txt"), out=lambda *a: None, device_ingest=device_ingest,
                      offtargets=str(d / "ot.tsv") if counts else None, max_mismatches=k,
                      offtarget_sites=str(d / "sites.tsv") if sites else None, max_sites=50,
                      offtarget_scores=str(d / "scores.tsv") if scores else None)
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["sample", "edge_fmt"])
def test_run_cas9_scores_table_equals_oracle_and_leaves_the_other_tables_untouched(manifest, eng, tmp_path, case):
    c = manifest["cases"][case]
    tokens = oracle.import_fasta_text(fixture_text(c["fasta"]))
    for k in (3, 1):
        want = sco.scores_table(tokens, k)
        for dev in (True, False):
            base = _run(c["fasta"], tmp_path / f"base{k}{dev}", k, dev, c["seed"], c["blas_threads"], scores=False)
            new = _run(c["fasta"], tmp_path / f"new{k}{dev}", k, dev, c["seed"], c["blas_threads"])
            alone = _run(c["fasta"], tmp_path / f"alone{k}{dev}", k, dev, c["seed"], c["blas_threads"], counts=False,
                         sites=False)
            for name in ("out.csv", "ot.tsv", "sites.tsv"):
                assert (new / name).read_bytes() == (base / name).read_bytes(), name
            assert (alone / "out.csv").read_bytes() == (base / "out.csv").read_bytes()
            assert (new / "out.csv").read_bytes().decode() == golden_csv(case)
            for d in (new, alone):
                got = (d / "scores.tsv").read_bytes().decode()
                assert _same(got.split("\r\n"), want.split("\r\n")) is True, (k, dev, d.name)
            assert not (alone / "ot.tsv").exists() and not (alone / "sites.tsv").exists()


@pytest.mark.gpu
def test_cli_scores_table_equals_oracle(eng, tmp_path):
    from cropsr_b200 import cli
    path = tmp_path / "g.fa"
    path.write_text(fixture_text("clean3.fa"))
    tokens = oracle.import_fasta_text(fixture_text("clean3.fa"))
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        assert cli.main(["-f", str(path), "-g", fixture_path("sample_genome.gff"), "--cas9", "-o", str(tmp_path / "o.csv"),
                         "--offtarget-scores",
                         str(tmp_path / "s.tsv"), "--mismatches", "2"]) == 0
    finally:
        os.chdir(cwd)
    got = (tmp_path / "s.tsv").read_bytes().decode()
    assert _same(got.split("\r\n"), sco.scores_table(tokens, 2).split("\r\n")) is True
