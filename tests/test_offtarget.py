"""Off-target counts (csrc/offtarget.cuh, crp_offtarget_*, engine.OffTargetIndex, --offtargets).

CPU: the semantics pinned by hand, the vectorised oracle pinned to the string oracle, the per-site functions and
the pair rule of the kernels emulated on the host (tests/offtarget_emu.cu), the CLI refusals.
GPU: site multisets and per-candidate counts against the brute-force oracle, guides, several genome handles, the CLI
table, and configs[1] at size."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import cropsr_oracle as oracle
import offtarget_oracle as ot
from helpers import ROOT, fixture_path, fixture_text, golden_csv, synthetic_fasta

# ---------------------------------------------------------------- a hand-built genome
GUIDE = "GATTACAGCTTCAGTCATCA"         # no GG / CC in it or in its reverse complement: it makes no sites of its own
FILL = "T" * 30


def _sub(guide, positions):
    """the guide with a different base (A, or T for an A) at each position"""
    g = list(guide)
    for p in positions:
        g[p] = "T" if g[p] == "A" else "A"
    return "".join(g)


def _rc(s):
    return s[::-1].translate(str.maketrans("ACGTacgt", "TGCAtgca"))


def hand_tokens():
    """Two tokens: a formatted-path token (quote / paren decoration) and a clean one.  Copies of GUIDE:
      c0  exact, '+', upper-case AGG (a candidate)            c1  1 substitution, '+', AGG
      c2  2 substitutions, reverse orientation ('-' site)    c3  3 substitutions, lower-case, tgg
      c4  exact, lower-case gg PAM (a site, not a candidate)  c5  4 substitutions, AGG
      c6  exact with an N inside                             d0  exact right after the decoration quote (its window
                                                                 holds the quote: no site, not a candidate either)
      token 2: e0 exact copy with CGG, and at the token end a '-' copy cut short (a candidate with no counts)."""
    t1 = ("'" + GUIDE[1:] + "AGG" + FILL                                  # d0: t = 20, tok[0] = "'"
          + GUIDE + "AGG" + FILL                                          # c0
          + _sub(GUIDE, [3]) + "AGG" + FILL                               # c1
          + "CCT" + _rc(_sub(GUIDE, [7, 11])) + FILL                      # c2
          + _sub(GUIDE, [0, 15, 19]).lower() + "tgg" + FILL               # c3
          + GUIDE + "Agg" + FILL                                          # c4
          + _sub(GUIDE, [1, 5, 9, 13]) + "AGG" + FILL                     # c5
          + GUIDE[:10] + "N" + GUIDE[11:] + "AGG" + FILL                  # c6
          + "'),")
    t2 = FILL + GUIDE + "CGG" + FILL + "CCA" + _rc(GUIDE)[:18]             # e0, then the cut-off '-' copy
    return {">chrA": t1, ">chrB": t2}


def test_hand_built_counts_are_what_the_definition_says():
    toks = list(hand_tokens().values())
    keys = np.array([k for tok in toks for _, _, k in ot.sites(tok)], dtype=np.uint64)
    # the guide itself: c0, c4, e0 exact; c1 at 1; c2 at 2; c3 at 3 (c5 has 4, c6 and d0 are no sites)
    assert ot.counts_for_key(ot.key_of(GUIDE), keys, 3).tolist() == [3, 1, 1, 1]
    assert ot.counts_for_key(ot.key_of(GUIDE.lower()), keys, 1).tolist() == [3, 1]
    # every candidate (upper-case PAM), reference order; written out by hand from the layout above
    assert ot.candidate_rows(toks, 3) == [
        (0, "+", 73, GUIDE, [2, 1, 1, 1]),                      # c0: c4 and e0 exact (itself not counted), c1, c2, c3
        (0, "+", 126, _sub(GUIDE, [3]), [0, 3, 0, 1]),          # c1: the three exact copies at 1, c2 at 1 + 2
        (0, "+", 338, _sub(GUIDE, [1, 5, 9, 13]), [0, 0, 0, 0]),   # c5: 4 from everything
        (0, "+", 391, None, None),                              # c6: N in the protospacer
        (0, "-", 159, _sub(GUIDE, [7, 11]), [0, 0, 3, 1]),      # c2, read in the guide's orientation
        (1, "+", 50, GUIDE, [2, 1, 1, 1]),                      # e0: sites of the other record count too
        (1, "-", 83, None, None),                               # cut off by the token end
    ]
    # d0 (t = 20, the quote in its window) is no site and no candidate; c3 and c4 (lower-case PAM) are sites only
    assert not any(t == 20 for t, _, _ in ot.sites(toks[0]))
    assert {t for t, s, _ in ot.sites(toks[0]) if s == "+"} >= {232, 285}


@pytest.mark.parametrize("fasta", ["multi3.fa", "clean3.fa", "edge_clean.fa", "edge_fmt.fa", "sample_genome.fa"])
def test_vectorised_site_keys_equal_the_string_oracle(fasta):
    for tok in oracle.import_fasta_text(fixture_text(fasta)).values():
        t, s, k = ot.site_keys_np(tok.encode("ascii"))
        assert sorted(zip(t.tolist(), ["+-"[x] for x in s.tolist()], k.tolist())) == sorted(ot.sites(tok))
    for tok in hand_tokens().values():
        t, s, k = ot.site_keys_np(tok.encode("ascii"))
        assert sorted(zip(t.tolist(), ["+-"[x] for x in s.tolist()], k.tolist())) == sorted(ot.sites(tok))


def test_offtarget_site_functions_and_pair_rule_on_the_cpu(tmp_path):
    """tests/offtarget_emu.cu compiles the per-site functions of k_ot_sites / k_ot_queries and the pair rule of
    k_ot_join -- the SAME source -- for the host and checks them against byte-by-byte readings and all 1,351
    mismatch-position sets of size <= 3."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "offtarget_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "offtarget_emu.cu")], check=True, capture_output=True, timeout=600)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


@pytest.mark.parametrize("argv, why", [(["-l", "18"], "20-base guides"), (["--devices", "0-1"], "one GPU"),
                                       (["--mismatches", "4"], "0 to 3"), (["--mismatches", "-1"], "0 to 3")])
def test_cli_refuses_offtargets_before_any_device_work(built_lib, argv, why, capsys):
    from cropsr_b200 import cli, engine
    with pytest.raises(SystemExit) as e:
        cli.main(["-f", "missing.fa", "--cas9", "--offtargets", "out.tsv"] + argv)
    assert "--offtargets" in str(e.value.code) and why in str(e.value.code)
    assert engine._device is None                                         # refused before engine.init


def test_guide_keys_validate_their_input(built_lib):
    from cropsr_b200 import engine
    assert engine.guide_keys([GUIDE, GUIDE.lower()]).tolist() == [ot.key_of(GUIDE)] * 2
    for bad in (GUIDE[:19], GUIDE + "A", GUIDE[:19] + "N", GUIDE[:19] + "U"):
        with pytest.raises(ValueError):
            engine.guide_keys([bad])


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def planted_fasta(seed, n_copies=300, length=60_000):
    """Random bases with many copies of a few 23-mers (protospacer + NGG) at 0-4 substitutions, in mixed case
    and orientation: many (query, site) pairs at every d <= 3, and the d = 4 pairs that must not count."""
    rng = np.random.default_rng(seed)
    seq = bytearray(rng.choice(np.frombuffer(b"ACGT", np.uint8), size=length).tobytes())
    protos = ["".join(rng.choice(list("ACGT"), 20)) for _ in range(4)]
    for _ in range(n_copies):
        p = list(protos[rng.integers(len(protos))])
        for q in rng.choice(20, size=int(rng.integers(0, 5)), replace=False):
            p[q] = rng.choice([b for b in "ACGT" if b != p[q]])
        site = "".join(p) + rng.choice(list("ACGT")) + "GG"
        if rng.random() < 0.3:
            site = site.lower()
        elif rng.random() < 0.2:
            site = site[:20] + site[20:].lower()
        if rng.random() < 0.5:
            site = _rc(site)
        at = int(rng.integers(0, length - 23))
        seq[at:at + 23] = site.encode()
    body = seq.decode()
    return ">r1\n" + "\n".join(body[i:i + 80] for i in range(0, 30_000, 80)) + "\n>r2\n" + \
        "\n".join(body[i:i + 80] for i in range(30_000, length, 80)) + "\n"


def _scan(text, device_ingest=False, tmp_path=None, limit=None):
    """(tokens, ScanOutput) through the host ingest, or the device ingest (None where the file is not plain)"""
    from cropsr_b200 import ingest, pipeline
    if device_ingest:
        path = tmp_path / "g.fa"
        path.write_text(text)
        fast = pipeline.scan_fasta_file(str(path), 20)
        if fast is None:
            return None
        keys, scan = fast
        return dict(zip(keys, [b.decode("ascii") for b in scan.token_bytes])), scan
    tokens = ingest.fasta_text_to_tokens(text)
    return tokens, pipeline.scan_token_bytes([v.encode("ascii") for v in tokens.values()], 20, limit=limit)


def _device_rows(eng, scan, k):
    """(token, strand, t, counts or None) in reference order, from one index over all handles"""
    index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts])
    rows = []
    try:
        for g, r, first, cnt in scan.parts:
            per = {}
            for strand in "+-":
                pos = r.fetch(strand, want=("pos",))["pos"]
                c = index.count_candidates(r, strand, k)
                off = r.off_plus if strand == "+" else r.off_minus
                per[strand] = (pos, c, off)
            for s in range(cnt):
                for strand in "+-":
                    pos, c, off = per[strand]
                    for i in range(int(off[s]), int(off[s + 1])):
                        rows.append((first + s, strand, int(pos[i]),
                                     None if c[i, 0] == eng.OffTargetIndex.NO_COUNT else c[i].tolist()))
    finally:
        index.free()
    return rows


def _oracle_rows(tokens, k):
    return [(a, b, c, e) for a, b, c, _, e in ot.candidate_rows(list(tokens.values()), k)]


@pytest.mark.gpu
@pytest.mark.parametrize("fasta", ["multi3.fa", "clean3.fa", "edge_clean.fa", "edge_fmt.fa", "ws_header.fa", "dup_keys.fa",
                                   "single_candidate.fa", "empty_records.fa", "mid50k.fa", "sample_genome.fa"])
def test_site_multiset_equals_oracle_on_fixtures(eng, fasta, tmp_path):
    text = fixture_text(fasta)
    for dev in (False, True):
        got = _scan(text, dev, tmp_path)
        if got is None:                        # not a plain FASTA file: the host ingest only
            continue
        tokens, scan = got
        try:
            index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts])
            want = sorted(k for tok in tokens.values() for _, _, k in ot.sites(tok))
            assert index.num_sites() == len(want)
            assert sorted(index.sites().tolist()) == want, (fasta, dev)
            index.free()
        finally:
            scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
def test_site_multiset_on_random_fastas_with_iupac(eng, seed, tmp_path):
    rng = np.random.default_rng(100 + seed)
    text = synthetic_fasta(200 + seed, [int(x) for x in rng.integers(100, 40_000, size=3)], gc=0.55, lower_frac=0.4, n_frac=0.01)
    iupac = np.frombuffer(b"RYKMSWBDHVN", np.uint8)
    b = bytearray(text.encode())
    for i in rng.choice(len(b), size=len(b) // 200, replace=False):
        if chr(b[i]) in "ACGTacgt":
            b[i] = int(rng.choice(iupac))
    text = b.decode()
    for dev in (False, True):
        tokens, scan = _scan(text, dev, tmp_path)
        try:
            index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts])
            assert sorted(index.sites().tolist()) == sorted(k for tok in tokens.values() for _, _, k in ot.sites(tok))
            index.free()
        finally:
            scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_candidate_counts_equal_brute_force_on_random_fastas(eng, seed):
    text = synthetic_fasta(300 + seed, [20_000, 9_000], gc=0.5, lower_frac=0.3, n_frac=0.005)
    tokens, scan = _scan(text)
    try:
        for k in range(4):
            assert _device_rows(eng, scan, k) == _oracle_rows(tokens, k), k
    finally:
        scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_candidate_counts_equal_brute_force_on_planted_repeats(eng, seed):
    tokens, scan = _scan(planted_fasta(seed))
    try:
        for k in range(4):
            got = _device_rows(eng, scan, k)
            assert got == _oracle_rows(tokens, k), k
        assert sum(1 for r in got if r[3] and sum(r[3]) >= 10) > 50    # the repeats are there
    finally:
        scan.free()


@pytest.mark.gpu
def test_one_bucket_with_more_than_100k_sites(eng):
    """Tandem copies of a 10-base unit with one gg: every copy is a site with the same key, so one bucket of
    every part pair holds > 10^5 sites (the work is split into site tiles x query tiles).  A few copies are
    upper case (candidates); a few are mutated."""
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
    tokens = {">tandem": tok}
    from cropsr_b200 import pipeline
    scan = pipeline.scan_token_bytes([tok.encode()], 20)
    try:
        index = eng.OffTargetIndex([scan.parts[0][0]])
        t, s, keys = ot.site_keys_np(tok.encode())
        assert index.num_sites() == len(keys) > 100_000
        assert sorted(index.sites().tolist()) == sorted(keys.tolist())
        g, r, _, _ = scan.parts[0]
        for k in (0, 3):
            pos = r.fetch("+", want=("pos",))["pos"]
            c = index.count_candidates(r, "+", k)
            assert len(pos) >= 150
            assert index.timing()["comparisons"] > 10 * len(pos) * 100_000 // 2
            for i in range(len(pos)):
                codes = ot.protospacer_codes(tok, int(pos[i]), "+")
                want = ot.counts_for_key(ot._key(codes), keys, k)
                want[0] -= 1
                assert c[i].tolist() == want.tolist(), (k, i)
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_count_guides_equals_oracle(eng):
    tokens, scan = _scan(planted_fasta(11))
    try:
        index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts])
        keys = np.array([k for tok in tokens.values() for _, _, k in ot.sites(tok)], dtype=np.uint64)
        present = [ot.protospacer(tok, t, s) for tok in tokens.values() for t, s, _ in ot.sites(tok)[:40]]
        rng = np.random.default_rng(3)
        absent = ["".join(rng.choice(list("ACGT"), 20)) for _ in range(30)]
        guides = present + [p.lower() for p in present[:10]] + present[:5] + absent
        for k in range(4):
            got = index.count_guides(guides, k)
            want = np.array([ot.counts_for_key(ot.key_of(g.upper()), keys, k) for g in guides])
            assert np.array_equal(got.astype(np.int64), want), k
        assert index.count_guides([], 3).shape == (0, 4)
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_several_handles_count_like_one(eng):
    """Tokens spread over several genome handles (handle_limit shrunk): one index over all handles gives the
    counts of a single-handle run, candidate for candidate."""
    text = planted_fasta(5)
    tokens, one = _scan(text)
    _, many = _scan(text, limit=1)
    try:
        assert len(one.parts) == 1 and len(many.parts) == 2
        for k in (0, 3):
            assert _device_rows(eng, many, k) == _device_rows(eng, one, k)
    finally:
        one.free()
        many.free()


@pytest.mark.gpu
def test_errors(eng):
    from cropsr_b200 import _native as N, ingest, pipeline
    tokens = ingest.fasta_text_to_tokens(fixture_text("multi3.fa"))
    g, r, _ = pipeline.scan_tokens(tokens, 20)
    g18, r18, _ = pipeline.scan_tokens(tokens, 18)
    index = eng.OffTargetIndex()
    try:
        with pytest.raises(N.CropsrError) as e:
            index.count_candidates(r, "+", 3)                     # genome not added
        assert e.value.code == -3
        index.add_genome(g)
        with pytest.raises(N.CropsrError) as e:
            index.add_genome(g)                                   # twice
        assert e.value.code == -3
        with pytest.raises(N.CropsrError) as e:
            index.count_candidates(r, "+", 4)
        assert e.value.code == -2
        index.add_genome(g18)
        with pytest.raises(N.CropsrError) as e:
            index.count_candidates(r18, "+", 3)                   # guide length 18
        assert e.value.code == -3
    finally:
        index.free()
        for x in (r, g, r18, g18):
            x.free()


def _table_from_oracle(tokens, k):
    keys = list(tokens.keys())
    lines = ["\t".join(["chromosome", "strand", "pam_pos", "protospacer"] + [f"mm{d}" for d in range(k + 1)])]
    for ti, strand, t, proto, counts in ot.candidate_rows(list(tokens.values()), k):
        lines.append("\t".join([keys[ti][1:], strand, str(t), proto or ""] +
                               ([str(c) for c in counts] if counts else [""] * (k + 1))))
    return "\r\n".join(lines) + "\r\n"


@pytest.mark.gpu
def test_cli_offtarget_table_equals_oracle_and_leaves_csv_untouched(manifest, eng, tmp_path):
    from cropsr_b200 import pipeline
    case = manifest["cases"]["sample"]
    tokens = oracle.import_fasta_text(fixture_text(case["fasta"]))
    for k, side in ((3, True), (1, False)):
        out, table = tmp_path / f"out{k}.csv", tmp_path / f"ot{k}.tsv"
        np.random.seed(case["seed"])
        pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out), 20, False,
                          case["blas_threads"], str(tmp_path / "time.txt"), out=lambda *a: None,
                          side_output=str(tmp_path / "side.tsv") if side else None, offtargets=str(table), max_mismatches=k)
        assert out.read_bytes().decode() == golden_csv("sample")
        assert table.read_bytes().decode() == _table_from_oracle(tokens, k)


@pytest.mark.gpu
def test_configs1_mm0_of_every_candidate_and_sampled_histograms(eng):
    """configs[1] (arabidopsis, 135 Mbp): mm0 of every candidate of both strands against an np.unique count over the
    oracle's site keys, and the full k = 3 histograms of 64 sampled candidates against brute force over all sites."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import workloads as W
    lengths = W.token_lengths("arabidopsis")
    genomes, results, site_tables = [], [], []
    index = eng.OffTargetIndex()
    try:
        for k in range(len(lengths)):
            tok = W.token("arabidopsis", k)
            g = eng.Genome()
            g.add_token(tok)
            g.commit()
            genomes.append(g)
            results.append(g.scan(20))
            index.add_genome(g)
            site_tables.append(ot.site_keys_np(tok))
        all_keys = np.concatenate([s[2] for s in site_tables])
        assert index.num_sites() == len(all_keys)
        uniq, cnt = np.unique(all_keys, return_counts=True)
        rng = np.random.default_rng(1)
        sample = []
        for k, (g, r) in enumerate(zip(genomes, results)):
            t_all, s_all, k_all = site_tables[k]
            for si, strand in enumerate("+-"):
                pos = r.fetch(strand, want=("pos",))["pos"].astype(np.int64)
                c = index.count_candidates(r, strand, 0)[:, 0]
                sel = s_all == si
                order = np.argsort(t_all[sel])
                ts, ks = t_all[sel][order], k_all[sel][order]
                at = np.minimum(np.searchsorted(ts, pos), max(len(ts) - 1, 0))
                valid = (ts[at] == pos) if len(ts) else np.zeros(len(pos), bool)
                want = np.full(len(pos), eng.OffTargetIndex.NO_COUNT, dtype=np.int64)
                qk = ks[at[valid]]
                want[valid] = cnt[np.searchsorted(uniq, qk)] - 1
                assert np.array_equal(c.astype(np.int64), want), (k, strand)
                for i in rng.choice(np.nonzero(valid)[0], size=7, replace=False):
                    sample.append((k, strand, int(i), int(ks[at[i]])))
        sample = sample[:64]
        # full histograms: one k = 3 call per (chromosome, strand), rows picked out
        full = {}
        for k, strand, i, key in sample:
            if (k, strand) not in full:
                full[(k, strand)] = index.count_candidates(results[k], strand, 3)
            want = ot.counts_for_key(key, all_keys, 3)
            want[0] -= 1
            assert full[(k, strand)][i].tolist() == want.tolist(), (k, strand, i)
        assert len(sample) == 64
    finally:
        index.free()
        for x in results + genomes:
            x.free()
