"""Off-target loci and listing (csrc/offtarget.cuh k_ot_sites<true> / k_ot_join<OtList>, crp_offtarget_new_with_loci /
fetch_loci / list_candidates / list_keys, engine.OffTargetIndex(loci=True), pipeline.write_offtarget_sites,
--offtarget-sites).

CPU: the sites oracle pinned by hand on planted sites, listing lengths against the counts oracle, the locus packing
of the kernel emulated on the host (tests/offtarget_sites_emu.cu), the batching of the Python listing, the CLI
refusals.
GPU: listings against brute force (random FASTAs with IUPAC bytes, planted repeats, a > 10^5-site bucket, several
genome handles, guides), the cap, the error codes, the table through run_cas9, and configs[1] at size."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import offtarget_oracle as ot
import offtarget_sites_oracle as so
from helpers import ROOT, fixture_path, fixture_text, golden_csv, synthetic_fasta

# ---------------------------------------------------------------- a hand-built genome (the layout of test_offtarget.py)
GUIDE = "GATTACAGCTTCAGTCATCA"         # no GG / CC in it or in its reverse complement: it makes no sites of its own
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


HEADER = "chromosome\tstrand\tpam_pos\tprotospacer\tsite_chromosome\tsite_strand\tsite_pam_pos\tsite_protospacer\tmismatches"
# c0 and c2, written out from the layout: mismatches first, then token, position, strand; differing bases lower case
C0_ROWS = ["chrA\t+\t73\tGATTACAGCTTCAGTCATCA\tchrA\t+\t285\tGATTACAGCTTCAGTCATCA\t0",
           "chrA\t+\t73\tGATTACAGCTTCAGTCATCA\tchrB\t+\t50\tGATTACAGCTTCAGTCATCA\t0",
           "chrA\t+\t73\tGATTACAGCTTCAGTCATCA\tchrA\t+\t126\tGATaACAGCTTCAGTCATCA\t1",
           "chrA\t+\t73\tGATTACAGCTTCAGTCATCA\tchrA\t-\t159\tGATTACAaCTTaAGTCATCA\t2",
           "chrA\t+\t73\tGATTACAGCTTCAGTCATCA\tchrA\t+\t232\taATTACAGCTTCAGTaATCt\t3"]
C2_ROWS = ["chrA\t-\t159\tGATTACAACTTAAGTCATCA\tchrA\t+\t73\tGATTACAgCTTcAGTCATCA\t2",
           "chrA\t-\t159\tGATTACAACTTAAGTCATCA\tchrA\t+\t285\tGATTACAgCTTcAGTCATCA\t2",
           "chrA\t-\t159\tGATTACAACTTAAGTCATCA\tchrB\t+\t50\tGATTACAgCTTcAGTCATCA\t2",
           "chrA\t-\t159\tGATTACAACTTAAGTCATCA\tchrA\t+\t126\tGATaACAgCTTcAGTCATCA\t3"]


def test_hand_built_site_rows_are_what_the_definition_says():
    lines = so.sites_table(hand_tokens(), 3).split("\r\n")
    assert lines[0] == HEADER and lines[-1] == ""
    rows = lines[1:-1]
    assert [r for r in rows if r.startswith("chrA\t+\t73\t")] == C0_ROWS
    assert [r for r in rows if r.startswith("chrA\t-\t159\t")] == C2_ROWS
    # c1 lists the three exact copies at 1 and c2 at 3; e0 mirrors c0 (c0 at 73 in its place); c5, c6 and the cut-off
    # '-' copy list nothing
    assert [r.split("\t")[2] for r in rows] == ["73"] * 5 + ["126"] * 4 + ["159"] * 4 + ["50"] * 5
    assert rows[13] == "chrB\t+\t50\tGATTACAGCTTCAGTCATCA\tchrA\t+\t73\tGATTACAGCTTCAGTCATCA\t0"
    # k = 1 keeps the rows with at most one mismatch; the cap leaves out whole candidates
    assert so.sites_table(hand_tokens(), 1).split("\r\n")[1:4] == C0_ROWS[:3]
    capped = so.sites_table(hand_tokens(), 3, max_sites=4).split("\r\n")[1:-1]
    assert capped == [r for r in rows if r.split("\t")[2] in ("126", "159")]
    # a guide lists every site, nothing subtracted
    assert [(d, ti, t, s) for d, ti, t, s, _ in so.guide_listing(list(hand_tokens().values()), [GUIDE], 3)[0]] == \
        [(0, 0, 73, "+"), (0, 0, 285, "+"), (0, 1, 50, "+"), (1, 0, 126, "+"), (2, 0, 159, "-"), (3, 0, 232, "+")]


@pytest.mark.parametrize("seed", range(3))
def test_listing_length_equals_the_counts_oracle_on_small_random_fastas(seed):
    from cropsr_b200 import ingest
    tokens = list(ingest.fasta_text_to_tokens(synthetic_fasta(500 + seed, [3_000, 1_500], gc=0.55, lower_frac=0.3,
                                                             n_frac=0.01)).values())
    for k in (1, 3):
        rows = so.listing(tokens, k)
        assert [r[:5] for r in rows] == ot.candidate_rows(tokens, k)
        for ti, strand, t, proto, counts, found in rows:
            assert len(found) == (sum(counts) if counts else 0)
            assert [d for d, *_ in found] == sorted(d for d, *_ in found)


def test_vectorised_neighbours_equal_the_string_oracle():
    tokens = list(hand_tokens().values())
    tabs = [ot.site_keys_np(tok.encode()) for tok in tokens]
    keys = np.concatenate([t[2] for t in tabs])
    where = [(ti, int(t), "+-"[int(s)]) for ti, tab in enumerate(tabs) for t, s in zip(tab[0], tab[1])]
    for k in range(4):
        idx, d = so.neighbours_np(ot.key_of(GUIDE), keys, k)
        want = so.guide_listing(tokens, [GUIDE], k)[0]
        assert sorted((int(x), *where[i]) for i, x in zip(idx.tolist(), d.tolist())) == sorted(w[:4] for w in want)


def test_locus_packing_on_the_cpu(tmp_path):
    """tests/offtarget_sites_emu.cu compiles the locus packing of k_ot_sites<true> -- the SAME source -- for the host
    and checks it against a byte-by-byte reading of random records."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "offtarget_sites_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "offtarget_sites_emu.cu")], check=True, capture_output=True, timeout=600)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


def test_listing_batches_bound_every_call(built_lib, monkeypatch):
    from cropsr_b200 import engine
    monkeypatch.setattr(engine, "LIST_BATCH_SITES", 10)
    index = engine.OffTargetIndex.__new__(engine.OffTargetIndex)        # no device: only the batching runs
    totals = [3, 4, 3, 0, 25, 1, 9, 1, 0, 0, 2]
    calls = []

    def call(lo, hi, f, out):
        calls.append((lo, hi, f.tolist(), len(out)))
        out[:] = lo
    first, sites = index._list(len(totals), totals, call)
    assert first.tolist() == [0] + np.cumsum(totals).tolist() and len(sites) == sum(totals)
    assert [c[:2] for c in calls] == [(0, 4), (4, 5), (5, 7), (7, 11)]
    for lo, hi, f, n in calls:
        assert f[0] == 0 and f[-1] == n and (n <= 10 or hi - lo == 1)
    index._h = None


@pytest.mark.parametrize("argv, why", [(["-l", "18"], "20-base guides"), (["--devices", "0-1"], "one GPU"),
                                       (["--mismatches", "4"], "0 to 3"), (["--max-sites", "0"], "at least 1"),
                                       (["--offtargets", "c.tsv", "--max-sites", "-3"], "at least 1")])
def test_cli_refuses_offtarget_sites_before_any_device_work(built_lib, argv, why):
    from cropsr_b200 import cli, engine
    with pytest.raises(SystemExit) as e:
        cli.main(["-f", "missing.fa", "--cas9", "--offtarget-sites", "out.tsv"] + argv)
    assert "--offtarget-sites" in str(e.value.code) and why in str(e.value.code)
    assert engine._device is None


# ---------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def planted_fasta(seed, n_copies=300, length=60_000):
    """Random bases with many copies of a few 23-mers (protospacer + NGG) at 0-4 substitutions, in mixed case
    and orientation: many (query, site) pairs at every d <= 3, and the d = 4 pairs that must not be listed."""
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


def _iupac_fasta(seed):
    rng = np.random.default_rng(700 + seed)
    text = synthetic_fasta(800 + seed, [int(x) for x in rng.integers(5_000, 25_000, size=3)], gc=0.55, lower_frac=0.4,
                           n_frac=0.01)
    iupac = np.frombuffer(b"RYKMSWBDHVN", np.uint8)
    b = bytearray(text.encode())
    for i in rng.choice(len(b), size=len(b) // 200, replace=False):
        if chr(b[i]) in "ACGTacgt":
            b[i] = int(rng.choice(iupac))
    return b.decode()


def _scan(text, limit=None):
    from cropsr_b200 import ingest, pipeline
    tokens = ingest.fasta_text_to_tokens(text)
    return tokens, pipeline.scan_token_bytes([v.encode("ascii") for v in tokens.values()], 20, limit=limit)


def _site_table(index, scan):
    """(token, t, strand, key) of every site, in sites() order"""
    keys = index.sites()
    gen, seg, t, strand = index.site_loci()
    first = np.array([f for _, _, f, _ in scan.parts], dtype=np.int64)
    tok = first[gen.astype(np.int64)] + seg.astype(np.int64)
    return list(zip(tok.tolist(), t.tolist(), ["+-"[x] for x in strand.tolist()], keys.tolist()))


def _device_listing(eng, scan, k, index=None):
    """{(token, strand, t): sorted [(site token, site t, site strand, site key)]} of every candidate with a protospacer,
    and {(token, strand, t): sum of counts}"""
    own = index is None
    if own:
        index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], loci=True)
    try:
        where = _site_table(index, scan)
        got, totals = {}, {}
        for g, r, first, cnt in scan.parts:
            for strand in "+-":
                pos = r.fetch(strand, want=("pos",))["pos"]
                off = r.off_plus if strand == "+" else r.off_minus
                seg_of = np.repeat(np.arange(cnt), np.diff(off).astype(np.int64))
                counts = index.count_candidates(r, strand, k)
                rows, fst, sites = index.list_candidates(r, strand, k, counts=counts)
                for i, row in enumerate(rows.tolist()):
                    key = (first + int(seg_of[row]), strand, int(pos[row]))
                    got[key] = sorted(where[s] for s in sites[fst[i]:fst[i + 1]].tolist())
                    totals[key] = int(counts[row].astype(np.int64).sum())
    finally:
        if own:
            index.free()
    return got, totals


def _oracle_listing(tokens, k):
    return {(ti, strand, t): sorted((si, st, ss, sk) for _, si, st, ss, sk in found)
            for ti, strand, t, proto, _, found in so.listing(list(tokens.values()), k) if proto is not None}


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(2))
def test_listing_equals_brute_force_on_random_fastas_with_iupac(eng, seed):
    tokens, scan = _scan(_iupac_fasta(seed))
    try:
        for k in range(4):
            got, totals = _device_listing(eng, scan, k)
            assert got == _oracle_listing(tokens, k), k
            assert all(len(v) == totals[key] for key, v in got.items())
    finally:
        scan.free()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(2))
def test_listing_equals_brute_force_on_planted_repeats(eng, seed):
    tokens, scan = _scan(planted_fasta(seed))
    try:
        for k in range(4):
            got, totals = _device_listing(eng, scan, k)
            assert got == _oracle_listing(tokens, k), k
            assert all(len(v) == totals[key] for key, v in got.items())
        assert sum(1 for v in got.values() if len(v) >= 10) > 50         # the repeats are there
    finally:
        scan.free()


@pytest.mark.gpu
def test_site_loci_equal_the_oracle_sites(eng):
    tokens, scan = _scan(_iupac_fasta(5), limit=1)
    try:
        assert len(scan.parts) > 1
        index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], loci=True)
        want = sorted((ti, t, s, key) for ti, tok in enumerate(tokens.values()) for t, s, key in ot.sites(tok))
        assert sorted(_site_table(index, scan)) == want
        gen = index.site_loci()[0]
        assert set(gen.tolist()) == set(range(len(scan.parts)))
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_cap_keeps_candidates_at_n_and_leaves_out_those_above(eng, tmp_path):
    from cropsr_b200 import pipeline
    tokens, scan = _scan(planted_fasta(21))
    try:
        rows = so.listing(list(tokens.values()), 3)
        totals = sorted({len(f) for *_, f in rows if len(f) > 1})
        n = totals[len(totals) // 2]
        at_n = [(ti, s, t) for ti, s, t, _, _, f in rows if len(f) == n]
        above = [(ti, s, t) for ti, s, t, _, _, f in rows if len(f) == n + 1]
        assert at_n and above
        for cap in (n, n + 1):
            path = tmp_path / f"sites{cap}.tsv"
            pairs, capped = pipeline.write_offtarget_sites(str(path), tokens, scan, 3, max_sites=cap)
            text = path.read_bytes().decode()
            assert text == so.sites_table(tokens, 3, max_sites=cap)
            assert pairs == text.count("\r\n") - 1
            assert capped == sum(1 for *_, f in rows if len(f) > cap)
            names = [key[1:] for key in tokens]
            listed = {(names.index(r.split("\t")[0]), r.split("\t")[1], int(r.split("\t")[2]))
                      for r in text.split("\r\n")[1:-1]}
            assert set(at_n) <= listed
            assert set(above) <= listed if cap == n + 1 else not set(above) & listed
    finally:
        scan.free()


@pytest.mark.gpu
def test_one_bucket_with_more_than_100k_sites_lists_every_copy(eng):
    """Tandem copies of a 10-base unit with one gg: every copy is a site with the same key, so one bucket of every
    part pair holds > 10^5 sites.  A few copies are upper case (candidates); a few are mutated."""
    from cropsr_b200 import pipeline
    n_units = 120_000
    unit = "atcgatcagg"
    rng = np.random.default_rng(7)
    units = [unit] * n_units
    for i in rng.choice(n_units, size=40, replace=False):
        units[i] = unit.upper()
    for i in rng.choice(n_units, size=100, replace=False):
        u = list(units[i])
        u[int(rng.integers(0, 7))] = "t" if u[0].islower() else "T"
        units[i] = "".join(u)
    tok = "ACGTTGCA" + "".join(units) + "TTGCA"
    scan = pipeline.scan_token_bytes([tok.encode()], 20)
    try:
        index = eng.OffTargetIndex([scan.parts[0][0]], loci=True)
        t_all, s_all, k_all = ot.site_keys_np(tok.encode())
        assert len(k_all) > 100_000
        _, r, _, _ = scan.parts[0]
        pos = r.fetch("+", want=("pos",))["pos"].astype(np.int64)
        where = _site_table(index, scan)
        for k in (0, 3):
            rows, first, sites = index.list_candidates(r, "+", k)
            assert len(rows) >= 30
            for i, row in enumerate(rows.tolist()):
                key = ot._key(ot.protospacer_codes(tok, int(pos[row]), "+"))
                idx, _ = so.neighbours_np(key, k_all, k)
                want = sorted((0, int(t_all[j]), "+-"[int(s_all[j])], int(k_all[j])) for j in idx.tolist()
                              if not (t_all[j] == pos[row] and s_all[j] == 0))
                assert sorted(where[s] for s in sites[first[i]:first[i + 1]].tolist()) == want, (k, i)
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_several_handles_list_like_one(eng):
    text = planted_fasta(5)
    tokens, one = _scan(text)
    _, many = _scan(text, limit=1)
    try:
        assert len(one.parts) == 1 and len(many.parts) == 2
        for k in (0, 3):
            assert _device_listing(eng, many, k)[0] == _device_listing(eng, one, k)[0]
    finally:
        one.free()
        many.free()


@pytest.mark.gpu
def test_list_guides_equals_oracle(eng):
    tokens, scan = _scan(planted_fasta(11))
    try:
        index = eng.OffTargetIndex([g for g, _, _, _ in scan.parts], loci=True)
        where = _site_table(index, scan)
        present = [ot.protospacer(tok, t, s) for tok in tokens.values() for t, s, _ in ot.sites(tok)[:30]]
        rng = np.random.default_rng(3)
        guides = present + [p.lower() for p in present[:5]] + ["".join(rng.choice(list("ACGT"), 20)) for _ in range(10)]
        for k in range(4):
            first, sites = index.list_guides(guides, k)
            want = so.guide_listing(list(tokens.values()), [g.upper() for g in guides], k)
            for i in range(len(guides)):
                got = sorted(where[s] for s in sites[first[i]:first[i + 1]].tolist())
                assert got == sorted((ti, t, s, key) for _, ti, t, s, key in want[i]), (k, i)
        first, sites = index.list_guides([], 3)
        assert first.tolist() == [0] and len(sites) == 0
        index.free()
    finally:
        scan.free()


@pytest.mark.gpu
def test_errors(eng):
    import ctypes as C
    from cropsr_b200 import _native as N
    from cropsr_b200.engine import lib
    tokens, scan = _scan(planted_fasta(3))
    g, r, _, _ = scan.parts[0]
    plain = eng.OffTargetIndex([g])
    index = eng.OffTargetIndex([g], loci=True)
    try:
        for call in (lambda: plain.list_candidates(r, "+", 3), lambda: plain.list_guides([GUIDE], 3), plain.site_loci):
            with pytest.raises(N.CropsrError) as e:
                call()
            assert e.value.code == -3
        counts = index.count_candidates(r, "+", 3)
        valid = np.nonzero(counts[:, 0] != index.NO_COUNT)[0]
        busy = valid[counts[valid].astype(np.int64).sum(axis=1) > 0][:4]
        assert len(busy) == 4
        for bad_rows in (busy[::-1], np.array([busy[0], busy[0]])):
            with pytest.raises(N.CropsrError) as e:
                index.list_candidates(r, "+", 3, rows=bad_rows, counts=counts)
            assert e.value.code == -2
        beyond, f0 = np.array([len(counts)], dtype=np.uint32), np.zeros(2, dtype=np.uint64)
        assert lib.crp_offtarget_list_candidates(index._h, r._h, b"+", 3, 1, beyond.ctypes.data, f0.ctypes.data, None) == -2
        with pytest.raises(N.CropsrError) as e:
            index.list_candidates(r, "+", 4, rows=busy, counts=np.zeros((len(counts), 5), np.uint32))
        assert e.value.code == -2
        with pytest.raises(N.CropsrError) as e:
            index.list_guides([GUIDE], 4)
        assert e.value.code == -2
        # a slice one short: CRP_ERR_STATE, nothing written, the guard values after first[n] untouched
        rows = np.ascontiguousarray(busy, dtype=np.uint32)
        first = np.zeros(len(rows) + 1, dtype=np.uint64)
        first[1:] = np.cumsum(counts[busy].astype(np.uint64).sum(axis=1))
        first[2:] -= np.uint64(1)
        out = np.full(int(first[-1]) + 8, 0xDEADBEEF, dtype=np.uint32)
        rc = lib.crp_offtarget_list_candidates(index._h, r._h, b"+", 3, len(rows), rows.ctypes.data, first.ctypes.data,
                                               out.ctypes.data)
        assert rc == -3
        assert (out == 0xDEADBEEF).all()
        # the right slices list the same rows as the Python face
        first[2:] += np.uint64(1)
        out = np.full(int(first[-1]) + 8, 0xDEADBEEF, dtype=np.uint32)
        assert lib.crp_offtarget_list_candidates(index._h, r._h, b"+", 3, len(rows), rows.ctypes.data, first.ctypes.data,
                                                 out.ctypes.data) == 0
        assert (out[int(first[-1]):] == 0xDEADBEEF).all()
        _, f2, s2 = index.list_candidates(r, "+", 3, rows=busy, counts=counts)
        assert f2.tolist() == first.tolist()
        assert [sorted(s2[f2[i]:f2[i + 1]]) for i in range(4)] == [sorted(out[first[i]:first[i + 1]]) for i in range(4)]
        # a row without a protospacer, a key of 41 bits
        invalid = np.nonzero(counts[:, 0] == index.NO_COUNT)[0]
        if len(invalid):
            with pytest.raises(N.CropsrError) as e:
                index.list_candidates(r, "+", 3, rows=invalid[:1], counts=np.zeros_like(counts))
            assert e.value.code == -2
        key = np.array([1 << 40], dtype=np.uint64)
        f1 = np.array([0, 0], dtype=np.uint64)
        assert lib.crp_offtarget_list_keys(index._h, 1, key.ctypes.data, 3, f1.ctypes.data, None) == -2
        n = C.c_uint64(0)
        assert lib.crp_offtarget_fetch_loci(index._h, 0, None, C.byref(n)) == -5 and n.value == index.num_sites()
    finally:
        plain.free()
        index.free()
        scan.free()


@pytest.mark.gpu
def test_run_cas9_sites_table_equals_oracle_and_leaves_the_other_outputs_untouched(manifest, eng, tmp_path):
    import cropsr_oracle as oracle
    from cropsr_b200 import pipeline
    case = manifest["cases"]["sample"]
    tokens = oracle.import_fasta_text(fixture_text(case["fasta"]))

    def run(tag, k, sites):
        d = tmp_path / tag
        d.mkdir()
        np.random.seed(case["seed"])
        lines = []
        stats = pipeline.run_cas9(fixture_path(case["fasta"]), fixture_path("sample_genome.gff"), str(d / "out.csv"), 20,
                                  True, case["blas_threads"], str(d / "time.txt"),
                                  out=lambda *a: lines.append(tuple(str(x).replace(str(d), "D") for x in a)),
                                  side_output=str(d / "side.tsv"), offtargets=str(d / "ot.tsv"), max_mismatches=k,
                                  offtarget_sites=str(d / "sites.tsv") if sites else None, max_sites=50)
        return d, stats, lines

    for k in (3, 1):
        base, s0, l0 = run(f"base{k}", k, False)
        new, s1, l1 = run(f"new{k}", k, True)
        for name in ("out.csv", "ot.tsv", "side.tsv", "side.tsv.gaps.tsv"):
            assert (new / name).read_bytes() == (base / name).read_bytes(), name
        assert (new / "out.csv").read_bytes().decode() == golden_csv("sample")
        text = (new / "sites.tsv").read_bytes().decode()
        assert text == so.sites_table(tokens, k, max_sites=50)
        assert s1["offtarget_pairs"] == text.count("\r\n") - 1 > 0
        assert s1["offtarget_capped"] == sum(1 for *_, f in so.listing(list(tokens.values()), k) if len(f) > 50)
        assert "offtarget_pairs" not in s0
        extra = [a for a in l1 if a not in l0]
        assert len(l1) == len(l0) + 1 and len(extra) == 1 and "off-target sites listed" in extra[0][0]


@pytest.mark.gpu
@pytest.mark.parametrize("n_sample", [250, pytest.param(2000, marks=pytest.mark.slow)])
def test_configs1_listing_at_size(eng, n_sample):
    """configs[1] (arabidopsis, 135 Mbp): every candidate with at most 1,000 sites within 3 mismatches is listed;
    the listing sums to the counts over all candidates, and sampled candidates equal vectorised brute force over
    site_keys_np (8.75 M sites each: ~40 ms per candidate on the CPU, so the 2,000-candidate sample is CROPSR_SLOW)."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import workloads as W
    lengths = W.token_lengths("arabidopsis")
    genomes, results, tabs = [], [], []
    index = eng.OffTargetIndex(loci=True)
    try:
        for k in range(len(lengths)):
            tok = W.token("arabidopsis", k)
            g = eng.Genome()
            g.add_token(tok)
            g.commit()
            genomes.append(g)
            results.append(g.scan(20))
            index.add_genome(g)
            tabs.append(ot.site_keys_np(tok))
        all_keys = np.concatenate([t[2] for t in tabs])
        all_tok = np.concatenate([np.full(len(t[2]), i, np.int64) for i, t in enumerate(tabs)])
        all_t = np.concatenate([t[0] for t in tabs]).astype(np.int64)
        all_s = np.concatenate([t[1] for t in tabs]).astype(np.int64)
        where = (all_tok << 34) | (all_t << 1) | all_s              # the own site of a sampled candidate by search
        where_order = np.argsort(where)
        site_keys = index.sites()
        gen, seg, s_t, s_strand = index.site_loci()
        assert (seg == 0).all()                       # one token per handle
        rng = np.random.default_rng(2)
        listed = total = 0
        sample = []
        for ti, r in enumerate(results):
            for strand in "+-":
                counts = index.count_candidates(r, strand, 3)
                ok = counts[:, 0] != index.NO_COUNT
                tot = np.where(ok, counts.astype(np.int64).sum(axis=1), 0)
                rows = np.nonzero(ok & (tot <= 1000))[0]
                rows, first, sites = index.list_candidates(r, strand, 3, rows=rows, counts=counts)
                assert np.array_equal(np.diff(first).astype(np.int64), tot[rows])
                listed += len(sites)
                total += int(tot[rows].sum())
                pos = r.fetch(strand, want=("pos",))["pos"].astype(np.int64)
                for i in rng.choice(len(rows), size=min(len(rows), n_sample // (2 * len(results)) + 1), replace=False):
                    sample.append((ti, strand, int(pos[rows[i]]), sites[first[i]:first[i + 1]]))
        assert listed == total > 0
        for ti, strand, t, got in sample:
            si = 0 if strand == "+" else 1
            w = (ti << 34) | (t << 1) | si
            j = np.searchsorted(where, w, sorter=where_order)
            at = where_order[j:j + 1]
            assert len(at) == 1 and where[at[0]] == w
            idx, _ = so.neighbours_np(int(all_keys[at[0]]), all_keys, 3)
            idx = idx[idx != at[0]]
            want = sorted(zip(all_tok[idx].tolist(), all_t[idx].tolist(), all_s[idx].tolist(), all_keys[idx].tolist()))
            have = sorted(zip(gen[got].astype(np.int64).tolist(), s_t[got].astype(np.int64).tolist(),
                              s_strand[got].astype(np.int64).tolist(), site_keys[got].tolist()))
            assert have == want, (ti, strand, t)
        assert len(sample) >= n_sample
    finally:
        index.free()
        for x in results + genomes:
            x.free()
