"""Every Rule Set 1 lane state against the dense BLAS-order replay, on the CPU and through the scan,
rescore and row-score kernels.

The canonical score sums eight lanes, one per base class: first-order fA fT fC fG and dinucleotide
dA dT dC dG (csrc/rs1.cuh).  A lane's value depends only on which of its entries match the 30-mer, and
most of it is one load from a perfect-hash table.  Random rows reach few of the large states: a dG state
with six or seven matching entries fixes 12 - 14 bases.  So the states are enumerated here, from
cropsr_b200/rs1.py alone (not from the generated rs1_weights.inc):

  * lane f<B> holds the FIRST entries of base B, by position;
  * lane d<B> holds the SECOND entries whose second base is B, in column order 16p + 4c1 + B.

Bases 2 and 3 of every scanned 30-mer are the PAM's upper-case C.  Positions tied together by the lane's
dinucleotide entries form small groups; every assignment of a group's positions is tried, and a lane's
states are the products of its groups' sets of matching entries.  A fifth letter stands for a byte that
does not score (N, or any byte but a base, U or Z).  It adds no state: in every group, the set of
matching entries an assignment with an N gives, some assignment of bases gives too (the counts are compared
below).  Rows with N still go through the kernels, for the scoring mask.

tests/rs1_lanes_emu.cu runs the scan kernel's own source on the CPU with a few 30-mers per state, and the
GPU tests plant them into a genome and compare every kernel that scores them with the oracle."""
import itertools
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

import cropsr_oracle as oracle
from cropsr_b200 import rs1

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LANES = ["fA", "fT", "fC", "fG", "dA", "dT", "dC", "dG"]
ROWS_PER_STATE = 3          # two over A T C G, one with N outside (and, where it can, inside) the lane's groups


def lane_entries(name):
    """[(positions, bases)] of a lane in column order"""
    b = "ATCG".index(name[1])
    if name[0] == "f":
        return [((p,), (c,)) for p, c in sorted(rs1.FIRST) if c == b]
    return [((p, p + 1), (c1, c2)) for p, c1, c2 in sorted(rs1.SECOND) if c2 == b]


def lane_groups(entries):
    """[(positions, entry indices)]: positions linked by one entry, with the entries on them"""
    parent = {}

    def find(p):
        while parent.setdefault(p, p) != p:
            p = parent[p]
        return p

    for pos, _ in entries:
        for p in pos:
            parent[find(p)] = find(pos[0])
    groups = {}
    for i, (pos, _) in enumerate(entries):
        groups.setdefault(find(pos[0]), []).append(i)
    out = []
    for idx in groups.values():
        out.append((sorted({p for i in idx for p in entries[i][0]}), idx))
    return sorted(out)


def group_states(entries, positions, idx, letters):
    """{bitmask of matching entries: [assignments (position -> code, 4 = does not score)]} of one group"""
    out = {}
    choices = [[2] if p in (2, 3) else letters for p in positions]
    for bases in itertools.product(*choices):
        at = dict(zip(positions, bases))
        m = 0
        for i in idx:
            pos, want = entries[i]
            if all(at[p] == c for p, c in zip(pos, want)):
                m |= 1 << i
        out.setdefault(m, []).append(at)
    return out


def lane_states(name, letters=(0, 1, 2, 3)):
    """(entries, groups, per-group state dicts, number of reachable states)"""
    entries = lane_entries(name)
    groups = lane_groups(entries)
    per = [group_states(entries, pos, idx, letters) for pos, idx in groups]
    return entries, groups, per, int(np.prod([len(g) for g in per]))


def lane_rows(name, rng):
    """ROWS_PER_STATE 30-mers for every reachable state of one lane (state order, 'N' for a byte that does not score)"""
    entries, groups, per4, _ = lane_states(name)
    _, _, per5, _ = lane_states(name, (0, 1, 2, 3, 4))
    fixed = {p for pos, _ in groups for p in pos}
    rows = []
    for combo in itertools.product(*[sorted(g) for g in per4]):
        for k in range(ROWS_PER_STATE):
            codes = rng.integers(0, 4, 30)
            if k == 2:                                     # N elsewhere, and an N realisation where there is one
                codes[rng.random(30) < 0.3] = 4
            for g4, g5, m in zip(per4, per5, combo):
                ways = g5[m] if k == 2 else g4[m]
                for p, c in ways[int(rng.integers(len(ways)))].items():
                    codes[p] = c
            codes[[2, 3]] = 2
            assert all(codes[p] != 4 or p in fixed or k == 2 for p in range(30))
            rows.append("".join("ATCGN"[c] for c in codes))
    return rows


def all_rows(seed=11):
    rng = np.random.default_rng(seed)
    return {name: lane_rows(name, rng) for name in LANES}


def test_lane_states_do_not_depend_on_a_non_scoring_byte():
    """The counts over A T C G equal the counts with a fifth, non-scoring letter (module docstring), and the
    states of a lane are at most all subsets of its entries that can match together."""
    for name in LANES:
        entries, _, _, n4 = lane_states(name)
        _, _, _, n5 = lane_states(name, (0, 1, 2, 3, 4))
        assert n4 == n5, name
        assert 0 < n4 <= 2 ** len(entries)


def _emulator(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "rs1_lanes_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O1", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "rs1_lanes_emu.cu")], check=True, capture_output=True, timeout=600)
    return exe


def test_every_lane_state_on_the_cpu(tmp_path):
    """tests/rs1_lanes_emu.cu on ROWS_PER_STATE rows of every reachable state of every lane: the table path
    (rs1_canonical, and score_hit on both strands at the tile's edge positions) equals the dense replay bit for
    bit, every table load reads the slot of the row's matching entries, the rows visit every table slot a
    30-mer can reach, and the states the emulator tells apart from the .inc entries are the ones counted here."""
    exe = _emulator(tmp_path)
    rows = all_rows()
    path = tmp_path / "rows.txt"
    path.write_text("".join(r + "\n" for name in LANES for r in rows[name]))
    r = subprocess.run([exe, str(path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.rstrip().splitlines()[-1].startswith("OK"), r.stdout[-3000:] + r.stderr
    got = {}
    for line in r.stdout.splitlines():
        if line.startswith("LANE "):
            f = line.split()
            got[f[1]] = int(f[3])
            if f[5] != "-":
                assert f[7] == f[9], line                 # slots visited == reachable slots
    want = {name: lane_states(name)[3] for name in LANES}
    print("reachable lane states:", want, "total", sum(want.values()))
    assert got == want


# ------------------------------------------------------------------------------------------------ GPU
def _plant(rows_by_lane, n_tokens, seed, one_strand=False):
    """FASTA text of tokens holding every row as a '+' and a '-' candidate (or one of them), with the planted
    (token index, t, strand, row) list.  Windows are 30 bytes apart plus a gap of 1 - 7 filler bytes, so they
    fall on every phase of the 32-position words and some cross tile edges.  Filler is A / T: no extra PAM.
    Every other window is written in lower case, or with U or Z where they score as the intended base."""
    rng = np.random.default_rng(seed)
    comp = {"A": "T", "T": "A", "C": "G", "G": "C"}
    items = [(r, st) for name in LANES for k, r in enumerate(rows_by_lane[name])
             for st in (("+-"[k % 2],) if one_strand else "+-")]
    per_tok = -(-len(items) // n_tokens)
    toks, planted = [], []
    for ti in range(n_tokens):
        buf = ["".join(rng.choice(list("AT"), 64))]
        pos = 64
        for j, (row, st) in enumerate(items[ti * per_tok:(ti + 1) * per_tok]):
            deco = int(rng.integers(1, 4)) if j % 2 else 0
            w = []
            for q, ch in enumerate(row):
                if ch == "N":
                    b = "n" if deco == 1 else "N"
                elif deco == 1 and q not in (2, 3):
                    b = ch.lower()                         # lower case scores uncomplemented on both strands
                elif deco == 2 and q not in (2, 3) and ch == ("A" if st == "-" else "T"):
                    b = "U"
                elif deco == 3 and q not in (2, 3) and ch == ("C" if st == "-" else "G"):
                    b = "Z"
                else:
                    b = ch if st == "-" else comp[ch]
                w.append(b)
            if st == "+":                                  # output base q = tok[t + 4 - q], window tok[t-25, t+5)
                buf.append("".join(reversed(w)))
                planted.append((ti, pos + 25, "+", row))
            else:                                          # output base q = tok[t - 2 + q]
                buf.append("".join(w))
                planted.append((ti, pos + 2, "-", row))
            gap = int(rng.integers(1, 8))
            buf.append("".join(rng.choice(list("AT"), gap)))
            pos += 30 + gap
        buf.append("A" * 64)
        toks.append("".join(buf))
    # one line per record and no final line end: the reference reads this layout without its repr() quirk,
    # so token positions are the positions above
    text = "\n".join(f">planted{ti}\n{tok}" for ti, tok in enumerate(toks))
    return text, planted


def _row_bytes(rows):
    return np.array([np.frombuffer(r.encode(), np.uint8) for r in rows])


def _want(seqs, c1, c2):
    m1, m2 = oracle.indicator_matrices(seqs)
    a = oracle.lane_sums(m1, oracle.W1, np.full(len(seqs), c1, dtype=np.int8))
    b = oracle.lane_sums(m2, oracle.W2, np.full(len(seqs), c2, dtype=np.int8))
    return (a + b + oracle.INTERCEPT + oracle.LOW_GC) * -1


def _chunked_canonical(seqs, step=20000):
    return np.concatenate([oracle.preactivation_model(seqs[i:i + step], classes=np.zeros(len(seqs[i:i + step]), np.int8))
                           for i in range(0, len(seqs), step)] or [np.empty(0)])


CLASS_PAIRS = [(c1, c2) for c1 in (0, 1, 2) for c2 in (0, 1, 2)]


@pytest.fixture(scope="module")
def planted():
    """The planted genome (two tokens), its oracle candidates, and the check that every planted candidate
    scores the intended row through the oracle's own window functions."""
    from cropsr_b200 import ingest
    rows = all_rows()
    text, plant = _plant(rows, 2, 5)
    tokens = ingest.fasta_text_to_tokens(text)
    keys = list(tokens)
    cands = [oracle.candidates_for_token(k, tokens[k], 20) for k in keys]
    index = [{(c[1] - 3 if c[6] == "-" else c[1], c[6]): c for c in cs} for cs in cands]
    for ti, t, st, row in plant:
        c = index[ti][(t, st)]
        got = oracle.scored_bytes(c[4])
        want = np.frombuffer(row.encode(), np.uint8)
        ok = np.isin(got, np.frombuffer(b"ATCG", np.uint8))
        assert len(c[4]) == 30 and np.array_equal(ok, want != ord("N")) and np.array_equal(got[ok], want[ok]), (ti, t, st, row, c[4])
    return tokens, cands, plant


@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def _check_scan(tokens, cands, flags=0):
    from cropsr_b200 import pipeline, _native as N
    from test_oracle_golden import oracle_np_exp
    genome, result, _ = pipeline.scan_tokens(tokens, 20, flags=flags)
    try:
        for seg, (key, tok) in enumerate(tokens.items()):
            cs = cands[seg]
            plus, minus = oracle.pam_hits(tok, 20)
            gp, gm = result.fetch_segment(seg, "+"), result.fetch_segment(seg, "-")
            assert gp["pos"].tolist() == plus and gm["pos"].tolist() == minus
            full = np.array([len(c[4]) == 30 for c in cs])
            assert full.all()
            seqs = np.array([oracle.scored_bytes(c[4]) for c in cs])
            want = _chunked_canonical(seqs)
            x = np.concatenate((gp["x"], gm["x"]))
            if flags & N.CRP_SCAN_LOGISTIC:
                with np.errstate(all="ignore"):
                    want = 1.0 / (1.0 + oracle_np_exp(want))
            assert np.array_equal(x, want), int(np.sum(x != want))
            packed = np.concatenate((gp["packed"], gm["packed"]))
            code = np.full(seqs.shape, 4, np.uint64)
            for c, b in enumerate(b"ATCG"):
                code[seqs == b] = c
            scoring = code < 4
            q = np.uint64(1) << np.arange(30, dtype=np.uint64)
            lo = ((code & np.uint64(1)) * q * scoring).sum(axis=1, dtype=np.uint64)
            hi = ((code >> np.uint64(1)) * q * scoring).sum(axis=1, dtype=np.uint64)
            mask = (q * scoring).sum(axis=1, dtype=np.uint64)
            assert np.array_equal(packed & np.uint64(0x3FFFFFFF) & mask, lo)
            assert np.array_equal((packed >> np.uint64(32)) & np.uint64(0x3FFFFFFF) & mask, hi)
            assert np.array_equal((packed & np.uint64(N.PACKED_UNSCORED)) != 0, ~scoring.all(axis=1))
            assert not np.any(packed & np.uint64(N.PACKED_TRUNCATED))
            windows = [tok[c[1] - 25:c[1] + 5] if c[6] == "+" else tok[c[1] - 5:c[1] + 25] for c in cs]
            irregular = np.array([any(ch not in "ACGT" for ch in w) for w in windows])
            assert np.array_equal((packed & np.uint64(N.PACKED_IRREGULAR)) != 0, irregular)
    finally:
        result.free()
        genome.free()


@pytest.mark.gpu
def test_planted_states_through_the_scan(eng, planted):
    """k_scan_score on the planted genome: pos, packed and x of every candidate (planted or not) against the
    oracle, bit for bit -- and x again as 1 / (1 + np.exp(x)) under CRP_SCAN_LOGISTIC."""
    from cropsr_b200 import _native as N
    tokens, cands, _ = planted
    _check_scan(tokens, cands)
    _check_scan(tokens, cands, N.CRP_SCAN_LOGISTIC)


@pytest.mark.gpu
def test_planted_states_through_rescore_and_row_scores(eng, planted):
    """Every class pair, for every planted candidate: Genome.rescore (k_rescore on the packed records) and
    HostRescorer (the host token through k_rs1_rows) against indicator_matrices + lane_sums; and the rows
    themselves through engine.rs1_preactivation / rs1_score."""
    from cropsr_b200 import pipeline
    from test_oracle_golden import oracle_np_exp
    tokens, cands, plant = planted
    genome, result, token_bytes = pipeline.scan_tokens(tokens, 20)
    host = pipeline.HostRescorer(token_bytes)
    try:
        seg = np.array([p[0] for p in plant], np.uint32)
        t = np.array([p[1] for p in plant], np.uint32)
        st = np.array([p[2].encode() for p in plant], "S1")
        seqs = _row_bytes([p[3] for p in plant])
        seqs = np.where(seqs == ord("N"), 0, seqs).astype(np.uint8)
        rows = _row_bytes([r for name in LANES for r in all_rows()[name]])
        for c1, c2 in CLASS_PAIRS:
            cls = c1 | (c2 << 4)
            want = _want(seqs, c1, c2)
            c = np.full(len(plant), cls, np.uint8)
            assert np.array_equal(genome.rescore(seg, t, st, c), want), (c1, c2)
            assert np.array_equal(host.rescore(seg, t, st, c), want), (c1, c2)
            want_rows = _want(rows, c1, c2)
            cr = np.full(len(rows), cls, np.uint8)
            assert np.array_equal(eng.rs1_preactivation(rows, cr), want_rows), (c1, c2)
            with np.errstate(all="ignore"):
                assert np.array_equal(eng.rs1_score(rows, cr), 1.0 / (1.0 + oracle_np_exp(want_rows))), (c1, c2)
    finally:
        result.free()
        genome.free()


@pytest.mark.gpu
def test_planted_states_in_the_csv(eng, tmp_path):
    """run_cas9 on a planted FASTA (every lane state once, on alternating strands, in one record) writes the
    oracle's CSV byte for byte at one and at eight BLAS threads.  The slices are cut so that rows take the
    pair class (a 1-thread slice of 4k + 2 rows) and the ddot class (the reference's one-row last slice)."""
    from cropsr_b200 import ingest, pipeline
    rng = np.random.default_rng(3)
    one = {name: lane_rows(name, rng)[::ROWS_PER_STATE] for name in LANES}
    text, _ = _plant(one, 1, 9, one_strand=True)
    (key, tok), = ingest.fasta_text_to_tokens(text).items()
    n = len(oracle.candidates_for_token(key, tok, 20))
    fa = tmp_path / "planted.fa"
    fa.write_text(text)
    classes = set()
    for threads, chunk in ((1, 4 * (n // 12) + 2), (8, n - 1)):
        for start, count in oracle.emission_slices(n, chunk):
            classes |= set(oracle.row_classes(count, 464, threads).tolist())
        out = tmp_path / f"out{threads}.csv"
        np.random.seed(17)
        pipeline.run_cas9(str(fa), os.path.join(ROOT, "tests", "golden", "fixtures", "sample_genome.gff"), str(out), 20,
                          False, threads, str(tmp_path / "time.txt"), out=lambda *a: None, chunk_rows=chunk)
        np.random.seed(17)
        want = oracle.run_to_string(text, 20, "model", threads, chunk=chunk)
        assert out.read_bytes().decode() == want, threads
    assert classes == {oracle.CANONICAL, oracle.PAIR, oracle.SINGLE}


@pytest.mark.gpu
def test_planted_states_under_the_checked_build(eng):
    """libcropsr_b200_checked.so: k_scan_score checks every x against rs1_dense (code 16) besides its other
    invariants; the planted scan runs under it in a subprocess and must pass."""
    lib = os.path.join(ROOT, "cropsr_b200", "libcropsr_b200_checked.so")
    if not os.path.exists(lib):
        pytest.skip("checked library not built (make -C cropsr_b200/csrc checked)")
    if os.environ.get("CROPSR_B200_LIB"):
        return                      # already inside such a subprocess
    env = dict(os.environ, CROPSR_B200_LIB=lib)
    probe = subprocess.run([sys.executable, "-c", "from cropsr_b200 import _native as N; print(N.lib.crp_checked_build())"],
                           cwd=ROOT, env=env, capture_output=True, text=True, timeout=120)
    assert probe.stdout.strip() == "1", probe.stderr[-1000:]
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "tests/test_rs1_lanes.py", "-k",
                          "test_planted_states_through_the_scan"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "1 passed" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]
