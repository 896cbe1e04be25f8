"""Off-target sites at other PAM patterns (csrc/offtarget.cuh ot_pam_plus_sets / ot_pam_minus_sets, k_ot_sites<*, true>,
crp_offtarget_new_pam, engine.OffTargetIndex(pam=), --offtarget-pams).

CPU: the pattern oracle pinned by hand, NGG through the pattern oracle equal to offtarget_oracle, the vectorised keys
equal to the string oracle, the PAM tests of the kernel emulated on the host (tests/offtarget_pam_emu.cu), the pattern
parser, and the CLI refusals.
GPU: site multisets per pattern, counts / listings / scores against brute force, a > 10^5-site NAG bucket,
new_pam("NGG") against new, configs[1] cross-checks between NGG, NAG and NRG, the three tables through run_cas9 and the
CLI, and the error codes."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import cropsr_oracle as oracle
import offtarget_oracle as ot
import offtarget_pam_oracle as po
import offtarget_score_oracle as sco
import offtarget_sites_oracle as so
from helpers import ROOT, fixture_path, fixture_text, golden_csv, synthetic_fasta

GUIDE = "GATTACAGCTTCAGTCATCA"         # no GG / CC in it or in its reverse complement
FILL = "T" * 30


def _rc(s):
    return s[::-1].translate(str.maketrans("ACGTacgt", "TGCAtgca"))


def hand_tokens():
    """chrA: NGG candidate GUIDE+AGG at 50; NAG '+' copies of GUIDE at 103 (CAG) and 156 (lower-case tag); NGA '+' at 209
    (CGA); no site at 262 (CAN: N in letter 3) or 315 (CUG: U in letter 2); a NAG '-' copy at 348 (CTA + revcomp) and an
    NGA '-' copy at 401 (TCA + revcomp).  chrB: a NAG '+' copy at t = L - 3.  chrC: GUIDE + TA: an NTA site at t = L - 3,
    and t = L - 2 is no site.
    chrD: a NAG '-' copy with t + 23 = L.  chrE: the same one base short, t + 23 = L + 1: no site."""
    t1 = (FILL + GUIDE + "AGG" + FILL + GUIDE + "CAG" + FILL + GUIDE + "tag" + FILL + GUIDE + "CGA" + FILL
          + GUIDE + "CAN" + FILL + GUIDE + "CUG" + FILL + "CTA" + _rc(GUIDE) + FILL + "TCA" + _rc(GUIDE) + FILL)
    return {">chrA": t1, ">chrB": FILL + GUIDE + "CAG", ">chrC": FILL + GUIDE + "TA", ">chrD": FILL + "CTA" + _rc(GUIDE),
            ">chrE": FILL + "CTA" + _rc(GUIDE)[:-1]}


def _guide_sites(tok, pam):
    key = ot.key_of(GUIDE)
    return [(t, s) for t, s, k in po.sites(tok, pam) if k == key]


def test_hand_built_pattern_sites_are_what_the_definition_says():
    tk = hand_tokens()
    a, b, c, d, e = tk.values()
    assert _guide_sites(a, "NAG") == [(103, "+"), (156, "+"), (348, "-")]
    assert _guide_sites(a, "NGA") == [(209, "+"), (401, "-")]
    assert _guide_sites(a, "NGG") == [(50, "+")]
    assert _guide_sites(a, "NRG") == [(50, "+"), (103, "+"), (156, "+"), (348, "-")]
    assert _guide_sites(a, "nar") == [(103, "+"), (156, "+"), (348, "-")]        # CGA and TCA are not NAR
    assert a[263:265] == "AN" and a[316:318] == "UG"
    for pam in ("NAG", "NAD", "NAV", "NTG", "NKG", "NBG", "NHG"):
        assert not [t for t, st, _ in po.sites(a, pam) if st == "+" and t in (262, 315)], pam
    assert (len(b) - 3, "+") in _guide_sites(b, "NAG")
    assert c.endswith("TA") and (len(c) - 3, "+") in [(t, st) for t, st, _ in po.sites(c, "NTA")]
    for pam in ("NAG", "NAD", "NAV", "NTA"):
        assert not [t for t, st, _ in po.sites(c, pam) if st == "+" and t >= len(c) - 2], pam
    assert _guide_sites(d, "NAG") == [(30, "-")] and 30 + 23 == len(d)
    assert _guide_sites(e, "NAG") == [] and 30 + 23 == len(e) + 1
    # the candidate GUIDE+AGG at 50: NAG holds 5 exact copies and not its own site; NRG holds its own site as well
    rows = {pam: [r for r in po.candidate_rows(list(tk.values()), 3, pam) if r[:3] == (0, "+", 50)][0]
            for pam in ("NGG", "NAG", "NGA", "NRG")}
    assert rows["NGG"][4][0] == 0 and rows["NAG"][4][0] == 5 and rows["NGA"][4][0] == 2 and rows["NRG"][4][0] == 5
    assert rows["NGG"][3] == GUIDE
    # both ingest paths give the same tokens (their coordinates include the formatted path's decoration), and the
    # protospacers of their sites are those of the plain tokens
    text = "".join(f"{k}\n{v}\n" for k, v in tk.items())
    from cropsr_b200 import ingest
    host, ref = ingest.fasta_text_to_tokens(text), oracle.import_fasta_text(text)
    assert host == ref
    for pam in ("NAG", "NGA", "NRG"):
        assert [sorted(k for _, _, k in po.sites(t, pam)) for t in host.values()] == \
            [sorted(k for _, _, k in po.sites(t, pam)) for t in tk.values()]


@pytest.mark.parametrize("seed", range(3))
def test_ngg_pattern_is_the_ngg_oracle_and_vectorised_keys_equal_strings(seed):
    from cropsr_b200 import ingest
    text = synthetic_fasta(700 + seed, [4_000, 1_200], gc=0.5, lower_frac=0.3, n_frac=0.01)
    b = bytearray(text.encode())
    rng = np.random.default_rng(seed)
    for i in rng.choice(len(b), size=len(b) // 100, replace=False):
        if chr(b[i]) in "ACGTacgt":
            b[i] = int(rng.choice(np.frombuffer(b"RYKMSWBDHVNUZ", np.uint8)))
    tokens = list(ingest.fasta_text_to_tokens(b.decode()).values())
    for tok in tokens:
        assert po.sites(tok, "NGG") == po.sites(tok) == ot.sites(tok)
        for pam in ("NGG", "NAG", "NGA", "NRG", "NKH", "NBV", "NTA", "NCC"):
            t, s, k = po.site_keys_np(tok.encode(), pam)
            assert sorted(zip(t.tolist(), ["+-"[x] for x in s.tolist()], k.tolist())) == sorted(po.sites(tok, pam)), pam
    assert po.candidate_rows(tokens, 3, "NGG") == ot.candidate_rows(tokens, 3)


def test_table_oracles_without_extra_patterns_are_the_ngg_tables_and_add_up_with_them():
    from cropsr_b200 import ingest
    tokens = ingest.fasta_text_to_tokens(synthetic_fasta(811, [3_000, 900], gc=0.55, lower_frac=0.3, n_frac=0.01))
    tokens[">hand"] = hand_tokens()[">chrA"]
    toks = list(tokens.values())
    for k in (1, 3):
        assert po.sites_table(tokens, k, 4) == so.sites_table(tokens, k, 4)
        assert po.scores_table(tokens, k) == sco.scores_table(tokens, k)
        want = ["\t".join(["chromosome", "strand", "pam_pos", "protospacer"] + [f"mm{d}" for d in range(k + 1)])]
        for ti, strand, t, proto, counts in ot.candidate_rows(toks, k):
            want.append("\t".join([list(tokens)[ti][1:], strand, str(t), proto or ""] +
                                  ([str(c) for c in counts] if counts else [""] * (k + 1))))
        assert po.counts_table(tokens, k) == "\r\n".join(want) + "\r\n"
        # with NAG and NGA: the extra columns, the site_pam column, and the rows of the three patterns merged
        counts = po.counts_table(tokens, k, ["NAG", "NGA"]).split("\r\n")
        assert counts[0].endswith("\t".join([f"NAG_mm{d}" for d in range(k + 1)] + [f"NGA_mm{d}" for d in range(k + 1)]))
        sites = po.sites_table(tokens, k, 1000, ["NAG", "NGA"]).split("\r\n")[1:-1]
        assert "NAG" in {r.split("\t")[-1] for r in sites} <= {"NGG", "NAG", "NGA"}
        assert sorted(r.rsplit("\t", 1)[0] for r in sites if r.endswith("NGG")) == \
            sorted(so.sites_table(tokens, k, 1000).split("\r\n")[1:-1])
        nrg = po.candidate_rows(toks, k, "NRG")
        for row, ngg, nag in zip(nrg, po.candidate_rows(toks, k), po.candidate_rows(toks, k, "NAG")):
            assert row[4] == (None if ngg[4] is None else [x + y for x, y in zip(ngg[4], nag[4])])
        scores = po.scores_table(tokens, k, ["NAG"]).split("\r\n")
        assert scores[0].endswith("mit_specificity\tNAG_mit_hit_sum\tall_mit_specificity")


def test_pattern_parser_disjointness_and_own_site_rule(built_lib):
    from cropsr_b200 import engine
    assert engine.parse_pam("nag") == "NAG" and engine.parse_pam("NkH") == "NKH"
    for bad in ("", "NA", "NAGG", "AGG", "NNG", "NGN", "NXG", "N G", "NAU", 5):
        with pytest.raises(ValueError):
            engine.parse_pam(bad)
    letters = "ACGTRYSWKMBDHV"
    for x in letters:
        for y in letters:
            pam = "N" + x + y
            assert engine.pam_has_own_site(pam) == po.own_site(pam), pam
            for other in ("NGG", "NAG", "NRA", "NHV"):
                assert engine.pams_overlap(pam, other) == po.overlap(pam, other), (pam, other)
    assert engine.pams_overlap("NRG", "NGG") and engine.pams_overlap("NAG", "NAR")
    assert not engine.pams_overlap("NAG", "NGA") and not engine.pams_overlap("NAG", "NGG")
    assert engine.pam_has_own_site("NKG") and not engine.pam_has_own_site("NAG") and not engine.pam_has_own_site("NGH")


def test_pattern_site_tests_on_the_cpu(tmp_path):
    """tests/offtarget_pam_emu.cu compiles ot_pam_plus_sets / ot_pam_minus_sets -- the SAME source as the kernel -- for
    the host and checks them against a byte-by-byte reading for all 196 letter pairs, and {G}, {G} against NGG."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "offtarget_pam_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "offtarget_pam_emu.cu")], check=True, capture_output=True, timeout=600)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


@pytest.mark.parametrize("argv, why", [
    (["--offtargets", "o.tsv", "--offtarget-pams", "NXG"], "N followed by two"),
    (["--offtargets", "o.tsv", "--offtarget-pams", "NAG,"], "N followed by two"),
    (["--offtarget-scores", "o.tsv", "--offtarget-pams", "NNG"], "N followed by two"),
    (["--offtargets", "o.tsv", "--offtarget-pams", "NGG"], "always counted"),
    (["--offtarget-sites", "o.tsv", "--offtarget-pams", "NRG"], "NAG instead of NRG"),
    (["--offtargets", "o.tsv", "--offtarget-pams", "NAG,NAR"], "overlap"),
    (["--offtargets", "o.tsv", "--offtarget-pams", "NAG,nag"], "twice"),
    (["--offtarget-pams", "NAG"], "no off-target table"),
    (["--offtargets", "o.tsv", "--offtarget-pams", "NAG", "-l", "18"], "20-base guides"),
    (["--offtargets", "o.tsv", "--offtarget-pams", "NAG", "--devices", "0-1"], "one GPU"),
])
def test_cli_refuses_offtarget_pams_before_any_device_work(built_lib, argv, why):
    from cropsr_b200 import cli, engine
    with pytest.raises(SystemExit) as e:
        cli.main(["-f", "missing.fa", "--cas9"] + argv)
    msg = str(e.value.code)
    assert why in msg, msg
    assert "--offtarget-pams" in msg or why in ("20-base guides", "one GPU")
    assert engine._device is None


# ================================================================ GPU
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


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


def _iupac_fasta(seed, lengths):
    rng = np.random.default_rng(seed)
    text = synthetic_fasta(seed, lengths, gc=0.5, lower_frac=0.4, n_frac=0.01)
    b = bytearray(text.encode())
    for i in rng.choice(len(b), size=len(b) // 200, replace=False):
        if chr(b[i]) in "ACGTacgt":
            b[i] = int(rng.choice(np.frombuffer(b"RYKMSWBDHVNU", np.uint8)))
    return b.decode()


def planted_fasta(seed, pam="NAG", n_copies=300, length=60_000):
    """Random bases with many copies of a few protospacers at 0-4 substitutions, each followed by a PAM of `pam` or by
    NGG, in mixed case and orientation, several of them across the 16,384-position tile edges"""
    rng = np.random.default_rng(seed)
    seq = bytearray(rng.choice(np.frombuffer(b"ACGT", np.uint8), size=length).tobytes())
    protos = ["".join(rng.choice(list("ACGT"), 20)) for _ in range(4)]
    s2, s3 = po.letter_sets(pam)
    for n in range(n_copies):
        p = list(protos[rng.integers(len(protos))])
        for q in rng.choice(20, size=int(rng.integers(0, 5)), replace=False):
            p[q] = rng.choice([b for b in "ACGT" if b != p[q]])
        tail = "GG" if rng.random() < 0.3 else rng.choice(sorted(s2)) + rng.choice(sorted(s3))
        site = "".join(p) + rng.choice(list("ACGT")) + tail
        if rng.random() < 0.3:
            site = site.lower()
        if rng.random() < 0.5:
            site = _rc(site)
        at = int(rng.integers(0, length - 23)) if n % 10 else max(0, 16_384 * (1 + n % 3) - int(rng.integers(0, 23)))
        seq[at:at + 23] = site.encode()
    body = seq.decode()
    return ">r1\n" + "\n".join(body[i:i + 80] for i in range(0, 40_000, 80)) + "\n>r2\n" + \
        "\n".join(body[i:i + 80] for i in range(40_000, length, 80)) + "\n"


def _rows(scan):
    """(token, strand, t, stream row) of every candidate in reference order, and its part"""
    out = []
    for part, (g, r, first, cnt) in enumerate(scan.parts):
        for s in range(cnt):
            for strand in "+-":
                off = r.off_plus if strand == "+" else r.off_minus
                pos = r.fetch(strand, want=("pos",))["pos"]
                out += [(first + s, strand, int(pos[i]), part, i) for i in range(int(off[s]), int(off[s + 1]))]
    return out


def _check_index_against_oracle(eng, tokens, scan, pam, ks=range(4), lists=True, scores=True):
    """counts, listings (as loci) and scores of every candidate of one pattern's index against the pattern oracle"""
    toks = list(tokens.values())
    index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], loci=lists, pam=pam)
    try:
        where = _rows(scan)
        if lists:
            gen, seg, t, strand = index.site_loci()
            firsts = [first for _, _, first, _ in scan.parts]
            locus = [(firsts[gi] + si, int(ti), "+-"[st]) for gi, si, ti, st in zip(gen, seg, t, strand)]
        rng = np.random.default_rng(5)
        wts = rng.integers(0, 1 << 31, size=eng.SCORE_SETS, dtype=np.uint32)
        rank = {x: i for i, x in enumerate(eng.score_sets())}
        for k in ks:
            want = po.listing(toks, k, pam)
            assert [w[:3] for w in want] == [w[:3] for w in where]
            got = {(p, s): index.count_candidates(r, s, k) for p, (_, r, _, _) in enumerate(scan.parts) for s in "+-"}
            for (ti, s, t, part, i), (_, _, _, proto, counts, found) in zip(where, want):
                c = got[(part, s)][i]
                assert (None if c[0] == index.NO_COUNT else c.tolist()) == counts, (pam, k, ti, s, t)
            if lists:
                for part, (_, r, _, _) in enumerate(scan.parts):
                    for s in "+-":
                        rows, first, sites = index.list_candidates(r, s, k, counts=got[(part, s)])
                        sel = {(ti, st, t): w[5] for (ti, st, t, p, i), w in zip(where, want) if p == part and st == s}
                        by_row = {i: (ti, st, t) for ti, st, t, p, i in where if p == part and st == s}
                        for j, row in enumerate(rows.tolist()):
                            have = sorted(locus[x] for x in sites[int(first[j]):int(first[j + 1])].tolist())
                            assert have == sorted(f[1:4] for f in sel[by_row[row]]), (pam, k, row)
            if scores:
                for weights, wfun in ((None, sco.mit_weight), (wts, lambda x: int(wts[rank[tuple(x)]]))):
                    want_s = po.sums(toks, k, pam, wfun)
                    got_s = {(p, s): index.score_candidates(r, s, k, weights)
                             for p, (_, r, _, _) in enumerate(scan.parts) for s in "+-"}
                    for (ti, s, t, part, i), w in zip(where, want_s):
                        v = int(got_s[(part, s)][i])
                        assert (None if v == index.NO_SCORE else v) == w, (pam, k, ti, s, t)
        guides = [w[3] for w in po.listing(toks, 0, pam) if w[3]][:30] + ["".join(x) for x in
                                                                            rng.choice(list("ACGT"), (10, 20))]
        for k in ks:
            assert index.count_guides(guides, k).astype(np.int64).tolist() == po.guide_counts(toks, guides, k, pam)
    finally:
        index.free()


@pytest.mark.gpu
@pytest.mark.parametrize("fasta", ["multi3.fa", "edge_clean.fa", "edge_fmt.fa", "mid50k.fa", "sample_genome.fa"])
def test_site_multisets_per_pattern_on_fixtures(eng, fasta, tmp_path):
    text = fixture_text(fasta)
    for dev in (False, True):
        got = _scan(text, dev, tmp_path)
        if got is None:
            continue
        tokens, scan = got
        try:
            for pam in ("NAG", "NGA", "NRG", "NKH", "NGG"):
                for loci in (False, True):
                    index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], loci=loci, pam=pam)
                    want = sorted((ti, t, s, k) for ti, tok in enumerate(tokens.values()) for t, s, k in po.sites(tok, pam))
                    assert index.pam == pam and index.num_sites() == len(want)
                    if loci:
                        g, seg, t, st = index.site_loci()
                        firsts = [first for _, _, first, _ in scan.parts]
                        have = sorted((firsts[a] + b, int(c), "+-"[d], int(k)) for a, b, c, d, k in
                                      zip(g, seg, t, st, index.sites()))
                        assert have == want, (fasta, dev, pam)
                    else:
                        assert sorted(index.sites().tolist()) == sorted(w[3] for w in want), (fasta, dev, pam)
                    index.free()
        finally:
            scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_site_multisets_on_random_fastas_with_iupac_and_planted_tile_edges(eng, seed, tmp_path):
    for text in (_iupac_fasta(900 + seed, [40_000, 17_000, 300]), planted_fasta(seed, ["NAG", "NGA", "NKH"][seed])):
        for dev in (False, True):
            tokens, scan = _scan(text, dev, tmp_path)
            try:
                for pam in ("NAG", "NGA", "NRG", "NKH", "NBV"):
                    index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], pam=pam)
                    want = sorted(k for tok in tokens.values() for _, _, k in po.sites(tok, pam))
                    assert sorted(index.sites().tolist()) == want, (seed, dev, pam)
                    index.free()
            finally:
                scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("seed, pam", [(0, "NAG"), (1, "NGA"), (2, "NRG"), (3, "NKH")])
def test_counts_listings_scores_against_brute_force_on_planted_repeats(eng, seed, pam):
    tokens, scan = _scan(planted_fasta(seed, pam, n_copies=200, length=40_000))
    try:
        _check_index_against_oracle(eng, tokens, scan, pam)
    finally:
        scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("pam", ["NAG", "NRG"])
def test_counts_listings_scores_with_several_handles_and_random_fastas(eng, pam):
    text = _iupac_fasta(77, [12_000, 7_000, 2_000])
    tokens, scan = _scan(text, limit=1)
    try:
        assert len(scan.parts) == 3
        _check_index_against_oracle(eng, tokens, scan, pam, ks=(0, 3))
    finally:
        scan.free()


@pytest.mark.gpu
def test_one_nag_bucket_with_more_than_100k_sites(eng):
    rng = np.random.default_rng(9)
    unit = "".join(rng.choice(list("ACGT"), 20)) + "CAG"
    tok = (unit * 110_000) + "".join(rng.choice(list("ACGT"), 5_000))
    from cropsr_b200 import pipeline
    scan = pipeline.scan_token_bytes([tok.encode()], 20)
    try:
        index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], pam="NAG")
        t, s, keys = po.site_keys_np(tok.encode(), "NAG")
        assert index.num_sites() == len(keys) > 100_000
        assert sorted(index.sites().tolist()) == sorted(keys.tolist())
        guides = [unit[:20], unit[:19] + ("A" if unit[19] != "A" else "C")]
        for k in (0, 3):
            got = index.count_guides(guides, k).astype(np.int64)
            want = np.array([ot.counts_for_key(ot.key_of(g), keys, k) for g in guides])
            assert np.array_equal(got, want)
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_new_pam_ngg_equals_new(eng):
    from cropsr_b200 import _native as N
    tokens, scan = _scan(planted_fasta(4, "NGG", n_copies=200, length=40_000))
    handles = [g for g, _, _, _ in scan.parts]
    try:
        a = eng.OffTargetIndex(handles, loci=True)
        b = eng.OffTargetIndex.__new__(eng.OffTargetIndex)
        b.pam, b.loci, b._h = "NGG", True, C.c_void_p()
        N.check(N.lib.crp_offtarget_new_pam(C.byref(b._h), b"ngg", 1))
        for g in handles:
            b.add_genome(g)
        def table(ix):                                  # (key, genome, segment, t, strand) per site index
            return list(zip(ix.sites().tolist(), *[x.tolist() for x in ix.site_loci()]))
        ta, tb = table(a), table(b)
        assert sorted(ta) == sorted(tb)
        for _, r, _, _ in scan.parts:
            for s in "+-":
                for k in (0, 3):
                    ca, cb = a.count_candidates(r, s, k), b.count_candidates(r, s, k)
                    assert np.array_equal(ca, cb)
                    ra, fa, sa = a.list_candidates(r, s, k, counts=ca)
                    rb, fb, sb = b.list_candidates(r, s, k, counts=cb)
                    assert np.array_equal(ra, rb) and np.array_equal(fa, fb)
                    for j in range(len(ra)):
                        assert sorted(ta[x] for x in sa[fa[j]:fa[j + 1]].tolist()) == \
                            sorted(tb[x] for x in sb[fb[j]:fb[j + 1]].tolist())
                    assert np.array_equal(a.score_candidates(r, s, k), b.score_candidates(r, s, k))
        a.free()
        b.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_error_codes_of_new_pam(eng):
    from cropsr_b200 import _native as N
    h = C.c_void_p()
    for pam in (b"", b"N", b"NA", b"NAGG", b"AGG", b"NNG", b"NGN", b"NXG", b"N\x00G", b"NA\x00"):
        assert N.lib.crp_offtarget_new_pam(C.byref(h), pam, 0) == -2, pam
    assert N.lib.crp_offtarget_new_pam(None, b"NAG", 0) == -2
    assert N.lib.crp_offtarget_new_pam(C.byref(h), None, 0) == -2
    for pam in (b"NAG", b"nag", b"NvH", b"NGG"):
        assert N.lib.crp_offtarget_new_pam(C.byref(h), pam, 1) == 0
        assert N.lib.crp_offtarget_free(h) == 0
    with pytest.raises(ValueError):
        eng.OffTargetIndex(pam="NNG")


@pytest.mark.gpu
def test_configs1_ngg_nag_and_nrg_agree(eng):
    """configs[1] (arabidopsis, 135 Mbp): NAG site keys against site_keys_np; per candidate and every k the NRG counts
    equal NGG + NAG, the NRG MIT sums equal S_NGG + S_NAG exactly, and on sampled rows the NRG listing is the union of
    the NGG and NAG listings, compared as loci."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import workloads as W
    genomes, results, nag_keys = [], [], []
    for k in range(len(W.token_lengths("arabidopsis"))):
        tok = W.token("arabidopsis", k)
        g = eng.Genome()
        g.add_token(tok)
        g.commit()
        genomes.append(g)
        results.append(g.scan(20))
        nag_keys.append(po.site_keys_np(tok, "NAG")[2])
    idx = {pam: eng.OffTargetIndex(genomes, loci=True, pam=pam) for pam in ("NGG", "NAG", "NRG")}
    try:
        want = np.sort(np.concatenate(nag_keys))
        assert np.array_equal(np.sort(idx["NAG"].sites()), want)
        assert idx["NRG"].num_sites() == idx["NGG"].num_sites() + idx["NAG"].num_sites()
        loci = {pam: ix.site_loci() for pam, ix in idx.items()}
        rng = np.random.default_rng(2)
        for r in results:
            for s in "+-":
                for k in range(4):
                    c = {pam: ix.count_candidates(r, s, k).astype(np.int64) for pam, ix in idx.items()}
                    ok = c["NGG"][:, 0] != eng.OffTargetIndex.NO_COUNT
                    assert np.array_equal(c["NRG"][ok], c["NGG"][ok] + c["NAG"][ok]), (s, k)
                    sums = {pam: ix.score_candidates(r, s, k) for pam, ix in idx.items()}
                    assert np.array_equal(sums["NRG"][ok], sums["NGG"][ok] + sums["NAG"][ok]), (s, k)
                    if k in (1, 3):
                        rows = np.sort(rng.choice(np.nonzero(ok)[0], size=20, replace=False))
                        lists = {}
                        for pam, ix in idx.items():
                            rr, f, st = ix.list_candidates(r, s, k, rows=rows, counts=c[pam].astype(np.uint32))
                            lists[pam] = [sorted(tuple(int(a[x]) for a in loci[pam]) for x in st[f[j]:f[j + 1]].tolist())
                                          for j in range(len(rr))]
                        for j in range(len(rows)):
                            assert lists["NRG"][j] == sorted(lists["NGG"][j] + lists["NAG"][j]), (s, k, j)
    finally:
        for ix in idx.values():
            ix.free()
        for x in results + genomes:
            x.free()


@pytest.mark.gpu
def test_run_cas9_and_cli_tables_with_extra_pams(manifest, eng, tmp_path):
    from cropsr_b200 import cli, pipeline
    case = manifest["cases"]["sample"]
    tokens = oracle.import_fasta_text(fixture_text(case["fasta"]))
    pams = ["NAG", "NGA"]
    for k, pp in ((3, pams), (1, ["NGA"]), (2, [])):
        out, c, s, sc = (tmp_path / f"{n}{k}" for n in ("out.csv", "c.tsv", "s.tsv", "sc.tsv"))
        np.random.seed(case["seed"])
        stats = pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(out), 20, False,
                                  case["blas_threads"], str(tmp_path / "time.txt"), out=lambda *a: None,
                                  offtargets=str(c), offtarget_sites=str(s), offtarget_scores=str(sc),
                                  max_mismatches=k, max_sites=40, offtarget_pams=pp)
        assert out.read_bytes().decode() == golden_csv("sample")
        assert c.read_bytes().decode() == po.counts_table(tokens, k, pp), k
        assert s.read_bytes().decode() == po.sites_table(tokens, k, 40, pp), k
        assert sc.read_bytes().decode() == po.scores_table(tokens, k, pp), k
        if not pp:
            assert s.read_bytes().decode() == so.sites_table(tokens, k, 40)
            assert sc.read_bytes().decode() == sco.scores_table(tokens, k)
        assert stats["offtarget_pairs"] == s.read_bytes().decode().count("\r\n") - 1
    # the CLI, with a lower-case pattern
    d = tmp_path / "cli"
    d.mkdir()
    np.random.seed(case["seed"])
    cwd = os.getcwd()
    try:
        os.chdir(d)
        cli.main(["-f", fixture_path(case["fasta"]), "-g", fixture_path("sample_genome.gff"), "-o", "out.csv", "--cas9",
                  "--offtargets", "ot.tsv",
                  "--offtarget-sites", "s.tsv", "--offtarget-scores", "sc.tsv", "--offtarget-pams", "nag,NGA"])
    finally:
        os.chdir(cwd)
    assert (d / "ot.tsv").read_bytes().decode() == po.counts_table(tokens, 3, pams)
    assert (d / "s.tsv").read_bytes().decode() == po.sites_table(tokens, 3, 1000, pams)
    assert (d / "sc.tsv").read_bytes().decode() == po.scores_table(tokens, 3, pams)
