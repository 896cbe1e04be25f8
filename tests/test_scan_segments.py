"""crp_scan_segments (engine.scan_segments), the pipelined whole call behind every end-to-end number:
host tokens in, candidate rows out, H2D / pack / scan / D2H overlapped over three lanes.  Its rows are
compared with the string oracle at the edges of the call's own planning -- segments cut into pieces
(the crumb rule, per-segment counts summed back), pieces grouped under a byte cap, segments that start
inside their token, the capacity rerun of a group while later groups are queued, column subsets, arena
capacities -- and on the exact inputs of bench.py's e2e leg (shard.plan segments, CRP_SCAN_LOGISTIC,
want=("pos", "x"), one arena reused from call to call)."""
import os

import numpy as np
import pytest

import cropsr_oracle as oracle

TILE = 16384                 # crp_tile_size(); test_tile_constant checks it on the device
DEFAULT_PIECE = 32 << 20     # positions per piece without CRP_PIECE_POSITIONS
MAX_PIECES_PER_GROUP = 4096
SENTINEL = 0xA5
CRP_ERR_ARG = -2            # include/cropsr_b200.h


# ---------------------------------------------------------------- the planning, restated
def piece_size(env):
    """CRP_PIECE_POSITIONS: below one tile it is ignored, otherwise rounded down to a tile multiple."""
    if env is None:
        return DEFAULT_PIECE
    v = int(env)
    return v // TILE * TILE if v >= TILE else DEFAULT_PIECE


def plan_pieces(segments, P):
    """(segment index, begin, end) of every piece: P positions each, and a last piece of at most P / 4
    positions is merged into the one before it (no crumb).  An empty segment is one empty piece."""
    out = []
    for k, (b, e) in enumerate(segments):
        if e <= b:
            out.append((k, b, e))
            continue
        b0 = b
        while b0 < e:
            e0 = b0 + P
            if e0 + P // 4 >= e:
                e0 = e
            out.append((k, b0, e0))
            b0 = e0
    return out


def plan_groups(segments, P):
    """Number of groups (one commit and one scan each): a new group starts when the next piece would
    take the group past P + P / 4 positions, or the group already holds 4,096 pieces."""
    groups, nbytes, count = 0, 0, 0
    for _, b, e in plan_pieces(segments, P):
        nb = e - b
        if groups == 0 or nbytes + nb > P + P // 4 or count >= MAX_PIECES_PER_GROUP:
            groups, nbytes, count = groups + 1, 0, 0
        count += 1
        nbytes += nb
    return groups


def plan_h2d_bytes(segments, P):
    """Token bytes the call copies in for (token_len, begin, end) segments: every piece stages its
    positions plus 32 bytes of context on each side, clipped to the token, in 16-byte units."""
    total = 0
    for k, b, e in plan_pieces([(b, e) for _, b, e in segments], P):
        L = segments[k][0]
        total += (min(e + 32, L) - max(b - 32, 0) + 15) // 16 * 16
    return total


def planned(eng, before, segments, P, calls=1):
    """The library's counters moved by exactly what the model plans for `calls` calls of (token_len,
    begin, end) segments: one commit per group, and the staged bytes of every piece (a piece more or
    less, e.g. a crumb, moves the second)."""
    after = eng.perf_report()
    assert after["commits"] - before["commits"] == calls * plan_groups([(b, e) for _, b, e in segments], P)
    assert after["h2d_token_bytes"] - before["h2d_token_bytes"] == calls * plan_h2d_bytes(segments, P)


def test_planning_model_cuts_where_the_rules_say():
    """The model above on the token lengths the GPU cases are built around (CPU only)."""
    P = 16384
    lens = lambda n: [e - b for _, b, e in plan_pieces([(0, n)], P)]
    assert lens(P) == [P] and lens(P + 1) == [P + 1]
    assert lens(P + P // 4 - 1) == [P + P // 4 - 1] and lens(P + P // 4) == [P + P // 4]
    assert lens(P + P // 4 + 1) == [P, P // 4 + 1]
    assert lens(3 * P + P // 4 + 1) == [P, P, P, P // 4 + 1]
    assert lens(5 * P - 1) == [P, P, P, P, P - 1]
    assert lens(0) == [0] and plan_pieces([(128, 128)], P) == [(0, 128, 128)]
    assert plan_pieces([(2 * TILE + 384, 5 * P)], P)[1] == (0, 2 * TILE + 384 + P, 2 * TILE + 384 + 2 * P)
    assert plan_groups([(0, P + P // 4)], P) == 1 and plan_groups([(0, P)] * 2, P) == 2
    assert plan_groups([(0, 1)] * 5000, P) == 2 and plan_groups([(0, 300)] * 68 + [(0, 1)], P) == 1
    assert plan_groups([(0, 300)] * 69, P) == 2
    assert piece_size(None) == piece_size("100") == DEFAULT_PIECE
    assert piece_size("20000") == 16384 and piece_size("49152") == 49152 and piece_size("16383") == DEFAULT_PIECE
    # a crumb merged into the piece before it stages 64 bytes less than a piece of its own would
    assert plan_h2d_bytes([(P + P // 4 + 40, 0, P + P // 4)], P) == P + P // 4 + 32
    assert plan_h2d_bytes([(P + P // 4 + 40, 0, P + P // 4 + 1)], P) == (P + 32) + (P // 4 + 1 + 64 + 15) // 16 * 16
    assert plan_h2d_bytes([(100, 0, 0)], P) == 32 and plan_h2d_bytes([(0, 0, 0)], P) == 0


# ---------------------------------------------------------------- the oracle, segment by segment
_ROWS = {}


def _token_rows(tok, l):
    """Expected rows of a whole token, per strand: pos, and at l = 20 whether the 30-mer is whole,
    and for the whole ones x, the scored 2-bit code planes with their mask, and the unscored /
    irregular flags (built as _check_against_oracle in test_gpu_parity.py builds them)."""
    key = (tok, l)
    if key in _ROWS:
        return _ROWS[key]
    plus, minus = oracle.pam_hits(tok, l)
    out = {"+": {"pos": np.array(plus, np.int64)}, "-": {"pos": np.array(minus, np.int64)}}
    if l == 20:
        cands = oracle.candidates_for_token(">k", tok, l)
        arr = np.frombuffer(tok.encode(), np.uint8)
        weights = np.uint64(1) << np.arange(30, dtype=np.uint64)
        for strand, lo_c, hi_c in (("+", 0, len(plus)), ("-", len(plus), len(cands))):
            rows = out[strand]
            cs = cands[lo_c:hi_c]
            full = np.array([len(c[4]) == 30 for c in cs], dtype=bool)
            seqs = np.array([oracle.scored_bytes(c[4]) for c, f in zip(cs, full) if f], dtype=np.uint8).reshape(-1, 30)
            rows["full"] = full
            rows["x"] = oracle.preactivation_model(seqs, classes=np.zeros(len(seqs), dtype=np.int8))
            code = np.full(seqs.shape, -1, np.int64)
            for c, b in enumerate(b"ATCG"):
                code[seqs == b] = c
            scoring = code >= 0
            rows["lo"] = (((code & 1) * scoring).astype(np.uint64) * weights).sum(axis=1, dtype=np.uint64)
            rows["hi"] = ((((code >> 1) & 1) * scoring).astype(np.uint64) * weights).sum(axis=1, dtype=np.uint64)
            rows["mask"] = (scoring.astype(np.uint64) * weights).sum(axis=1, dtype=np.uint64)
            rows["unscored"] = ~scoring.all(axis=1)
            # irregular: the token window holds a byte that is not upper-case ACGT
            t = rows["pos"][full]
            first = t - 25 if strand == "+" else t - 2
            win = arr[first[:, None] + np.arange(30)] if len(t) else np.zeros((0, 30), np.uint8)
            rows["irregular"] = ~np.isin(win, np.frombuffer(b"ACGT", np.uint8)).all(axis=1)
    _ROWS[key] = out
    return out


def expected(segments, l):
    """Per-segment counts and the rows of each strand in segment order, for (token_id, token str,
    begin, end) descriptors: the token's oracle rows with begin <= t < end."""
    counts = {"+": [], "-": []}
    rows = {}
    for strand in "+-":
        parts = []
        for _, tok, b, e in segments:
            whole = _token_rows(tok, l)[strand]
            sel = (whole["pos"] >= b) & (whole["pos"] < e)
            counts[strand].append(int(sel.sum()))
            part = {"pos": whole["pos"][sel]}
            if l == 20:
                full = whole["full"]
                fsel = sel[full]
                part["full"] = full[sel]
                for name in ("x", "lo", "hi", "mask", "unscored", "irregular"):
                    part[name] = whole[name][fsel]
            parts.append(part)
        rows[strand] = {name: np.concatenate([p[name] for p in parts]) if parts else np.zeros(0)
                        for name in (parts[0] if parts else {"pos": 0})}
    return counts, rows


def check_rows(want, strand, pos=None, packed=None, x=None, logistic=False):
    """Compare one strand's columns (each already cut to its row count) with expected()'s rows."""
    from cropsr_b200 import _native as N
    from test_oracle_golden import oracle_np_exp
    w = want[strand]
    if pos is not None:
        assert np.array_equal(pos.astype(np.int64), w["pos"]), strand
    if "full" not in w:
        return
    full = w["full"]
    if x is not None:
        want_x = 1.0 / (1.0 + oracle_np_exp(w["x"])) if logistic else w["x"]
        assert np.array_equal(x[full], want_x), strand
    if packed is not None:
        assert np.array_equal((packed & np.uint64(N.PACKED_TRUNCATED)) != 0, ~full), strand
        pk = packed[full]
        lo, hi = pk & np.uint64(0x3FFFFFFF), (pk >> np.uint64(32)) & np.uint64(0x3FFFFFFF)
        assert np.array_equal(lo & w["mask"], w["lo"]) and np.array_equal(hi & w["mask"], w["hi"]), strand
        assert np.array_equal((pk & np.uint64(N.PACKED_UNSCORED)) != 0, w["unscored"]), strand
        assert np.array_equal((pk & np.uint64(N.PACKED_IRREGULAR)) != 0, w["irregular"]), strand


@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def full_arena(eng, capacity):
    a = eng.Arena(capacity, True)
    for strand in "+-":
        for v in a.arrays[strand].values():
            v.view(np.uint8)[:] = SENTINEL
    return a


def run_and_check(eng, segments, l, P_env=None, flags=0, want=("pos", "packed", "x"), arena=None, monkeypatch=None):
    """One scan_segments call on str-token descriptors, checked against the oracle; the call must
    commit exactly the groups the planning model predicts.  Returns (arena, n_plus, n_minus)."""
    from cropsr_b200 import _native as N
    if monkeypatch is not None:
        if P_env is None:
            monkeypatch.delenv("CRP_PIECE_POSITIONS", raising=False)
        else:
            monkeypatch.setenv("CRP_PIECE_POSITIONS", str(P_env))
    counts, rows = expected(segments, l)
    need = max(sum(counts["+"]), sum(counts["-"]), 1)
    if arena is None:
        arena = eng.Arena(need + 100, True, want)
    assert arena.capacity >= need
    before = eng.perf_report()
    arena, n_plus, n_minus, ms = eng.scan_segments([(k, tok, b, e) for k, tok, b, e in segments], l,
                                                   flags=flags, arena=arena, want=want)
    planned(eng, before, [(len(tok), b, e) for _, tok, b, e in segments], piece_size(P_env))
    assert n_plus.tolist() == counts["+"] and n_minus.tolist() == counts["-"]
    scored = l == 20 and not (flags & N.CRP_SCAN_NO_SCORE)
    for strand, n in (("+", sum(counts["+"])), ("-", sum(counts["-"]))):
        a = arena.arrays[strand]
        cut = lambda name: a[name][:n] if a.get(name) is not None and scored else None
        check_rows(rows, strand, pos=a["pos"][:n] if a.get("pos") is not None else None,
                   packed=cut("packed"), x=cut("x"), logistic=bool(flags & N.CRP_SCAN_LOGISTIC))
    return arena, n_plus, n_minus


# ---------------------------------------------------------------- synthetic tokens
def random_token(seed, n, plant_every=TILE):
    """Upper / lower case, N and IUPAC codes; a '+' and a '-' PAM within 3 positions of every multiple
    of plant_every (CCGGCCGG over [c-4, c+4): '-' at c-4 and c, '+' at c-3 and c+1)."""
    rng = np.random.default_rng(seed)
    alphabet = np.frombuffer(b"ACGTacgtNRYKM", dtype=np.uint8)
    p = np.array([20, 20, 22, 22, 4, 4, 4, 4, 1, .3, .3, .2, .2])
    s = rng.choice(alphabet, size=n, p=p / p.sum())
    for c in range(plant_every, n - 4, plant_every):
        s[c - 4:c + 4] = np.frombuffer(b"CCGGCCGG", np.uint8)
    return s.tobytes().decode()


def edge_lengths(P):
    q = P // 4
    return [P, 1, P + 1, 29, P + q - 1, 37, P + q, 300, P + q + 1, 3 * P + q + 1, 1, 5 * P - 1, 29]


# ---------------------------------------------------------------- 1. piece edges
@pytest.mark.gpu
@pytest.mark.parametrize("P_env", [16384, 32768, 49152, 20000, 100])
def test_piece_edges_match_oracle(eng, monkeypatch, P_env):
    P = piece_size(P_env) if P_env != 100 else 16384       # token lengths of the 16,384 case when the value is ignored
    toks = [random_token(100 + k, n) for k, n in enumerate(edge_lengths(P))]
    segs = [(k, t, 0, len(t)) for k, t in enumerate(toks)]
    arena, _, _ = run_and_check(eng, segs, 20, P_env, monkeypatch=monkeypatch)
    arena.free()


# ---------------------------------------------------------------- 2. guide lengths across pieces
def spanning_tokens():
    """The tokens of test_guide_lengths_that_span_tiles (test_gpu_parity.py)."""
    rng = np.random.default_rng(77)
    alphabet = np.frombuffer(b"ACGTacgtN", dtype=np.uint8)
    p = np.array([15, 15, 30, 30, 2, 2, 2, 2, 2], dtype=float)
    return [rng.choice(alphabet, size=n, p=p / p.sum()).tobytes().decode() for n in (70001, 40000, 16380, 300)]


@pytest.mark.gpu
@pytest.mark.parametrize("l", [20, 18, 23, 1, 1000, 40000, 70000])
def test_guide_lengths_across_pieces_match_oracle(eng, monkeypatch, l):
    """With P = 16,384 the 70,001-position token is four pieces; at l = 70,000 every one of them lies
    inside both bound regions, so each is counted from PAM records."""
    segs = [(k, t, 0, len(t)) for k, t in enumerate(spanning_tokens())]
    arena, _, _ = run_and_check(eng, segs, l, 16384, monkeypatch=monkeypatch)
    arena.free()


# ---------------------------------------------------------------- 3. segments that start inside their token
BEGINS = (0, 128, 384, TILE - 128, TILE, TILE + 128, 2 * TILE + 384)


def inside_segment_sets():
    a, b = random_token(7, 90001), random_token(8, 52345)
    L = len(a)
    sets = [[(0, a, s, min(L, s + 20011 + s % 1000)) for s in BEGINS],            # one per begin, ends off the tile grid
            [(0, a, s, e) for s, e in zip((0, 384, TILE - 128, TILE + 128, 2 * TILE + 384, 40064),
                                          (384, TILE - 128, TILE + 128, 2 * TILE + 384, 40064, L))],  # adjacent
            [(0, a, 128, 5001), (0, a, TILE, TILE + 3001), (0, a, 2 * TILE + 384, L - 17), (1, b, 384, 50001)]]  # gaps
    return a, sets


@pytest.mark.gpu
@pytest.mark.parametrize("l", [20, 18, 23, 40000])
def test_segments_that_start_inside_their_token_match_oracle(eng, monkeypatch, l):
    a, sets = inside_segment_sets()
    for segs in sets:
        counts, rows = expected(segs, l)
        g = eng.Genome()
        for k, tok, s, e in segs:
            g.add_segment(k, tok, s, e)
        res = g.commit().scan(l)
        try:
            assert res.seg_plus.tolist() == counts["+"] and res.seg_minus.tolist() == counts["-"]
            for strand in "+-":
                f = res.fetch(strand)
                check_rows(rows, strand, f["pos"], f["packed"], f["x"])
        finally:
            res.free()
            g.free()
        for P_env in (None, 16384):
            arena, _, _ = run_and_check(eng, segs, l, P_env, monkeypatch=monkeypatch)
            arena.free()
    # the adjacent segments tile the token: together they return the whole token's rows
    assert sets[1][0][2] == 0 and sets[1][-1][3] == len(a) and all(p[3] == q[2] for p, q in zip(sets[1], sets[1][1:]))
    monkeypatch.setenv("CRP_PIECE_POSITIONS", "16384")
    whole, wp, wm, _ = eng.scan_segments([(0, a, 0, len(a))], l)
    parts, pp, pm, _ = eng.scan_segments(sets[1], l)
    assert int(pp.sum()) == int(wp[0]) and int(pm.sum()) == int(wm[0])
    for strand, n in (("+", int(wp[0])), ("-", int(wm[0]))):
        for name, v in whole.arrays[strand].items():
            if v is not None:
                assert np.array_equal(parts.arrays[strand][name][:n], v[:n]), (strand, name)
    whole.free()
    parts.free()


# ---------------------------------------------------------------- 4. bench's e2e call
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
def test_bench_e2e_inputs_place_the_whole_table(eng, monkeypatch, world):
    """Every rank's shard.plan segments (tile-aligned begins, ends inside a token, (k, 0, 0) for the
    empty token) through scan_segments with bench's flags and columns and one arena reused from rank to
    rank; the rows placed with shard.global_offsets are the oracle's whole-genome table."""
    from cropsr_b200 import shard, _native as N
    from test_oracle_golden import oracle_np_exp
    monkeypatch.setenv("CRP_PIECE_POSITIONS", "16384")
    toks = [random_token(40 + k, n) for k, n in enumerate((70001, 0, 130001, 300, 45000, 1))]
    plans = shard.plan([len(t) for t in toks], world)
    assert any(seg == (1, 0, 0) for segs in plans for seg in segs)
    want_pos, want_x, want_full = [], [], []
    for t in toks:
        r = _token_rows(t, 20)
        for strand in "+-":
            want_pos.append(r[strand]["pos"])
            x = np.zeros(len(r[strand]["pos"]))
            x[r[strand]["full"]] = 1.0 / (1.0 + oracle_np_exp(r[strand]["x"]))
            want_x.append(x)
            want_full.append(r[strand]["full"])
    want_pos, want_x, want_full = (np.concatenate(v) for v in (want_pos, want_x, want_full))
    arena = eng.Arena(len(want_pos), True, ("pos", "x"))
    counts, placed = [], []
    for segs in plans:
        descs = [(k, toks[k], a, b) for k, a, b in segs]
        before = eng.perf_report()
        arena2, n_plus, n_minus, _ = eng.scan_segments(descs, 20, flags=N.CRP_SCAN_LOGISTIC, arena=arena, want=("pos", "x"))
        assert arena2 is arena
        planned(eng, before, [(len(toks[k]), a, b) for k, a, b in segs], 16384)
        counts.append((n_plus.copy(), n_minus.copy()))
        rows = {}
        for strand, n in (("+", int(n_plus.sum())), ("-", int(n_minus.sum()))):
            rows[strand] = (arena.arrays[strand]["pos"][:n].copy(), arena.arrays[strand]["x"][:n].copy())
        placed.append(rows)
    offs, total = shard.global_offsets(plans, counts)
    assert total == len(want_pos)
    pos = np.full(total, -1, np.int64)
    x = np.zeros(total)
    for r, segs in enumerate(plans):
        for si, strand in enumerate("+-"):
            first = 0
            for s in range(len(segs)):
                n = int(counts[r][si][s])
                o = offs[r][s][si]
                pos[o:o + n] = placed[r][strand][0][first:first + n]
                x[o:o + n] = placed[r][strand][1][first:first + n]
                first += n
    assert np.array_equal(pos, want_pos)
    assert np.array_equal(x[want_full], want_x[want_full])
    arena.free()


# ---------------------------------------------------------------- 5. capacity rerun inside the pipeline
@pytest.mark.gpu
@pytest.mark.parametrize("logistic", [False, True])
def test_capacity_rerun_inside_the_pipeline_matches_oracle(eng, monkeypatch, logistic):
    """Poly-G and poly-C pieces hold a candidate at nearly every position, far above the first guess of
    positions / 8 + 4096: their groups are launched again from scan_finish while the groups after them
    are already queued on the lanes, and with CRP_SCAN_LOGISTIC the pass then runs on the row-copy stream."""
    from cropsr_b200 import _native as N
    normal = [random_token(60 + k, 20000) for k in range(3)]
    segs = [(0, normal[0], 0, 20000), (1, "G" * 100000, 0, 100000), (2, normal[1], 0, 20000),
            (3, "C" * 100000, 0, 100000), (4, normal[2], 0, 20000)]
    before = eng.perf_report()["capacity_reruns"]
    arena, _, _ = run_and_check(eng, segs, 20, 16384, flags=N.CRP_SCAN_LOGISTIC if logistic else 0,
                                monkeypatch=monkeypatch)
    assert eng.perf_report()["capacity_reruns"] - before >= 2
    arena.free()


# ---------------------------------------------------------------- 6. columns and flags
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["pos", "pos+x", "pos+packed", "packed+x", "no_score", "l18"])
def test_columns_and_flags_leave_the_rest_of_the_arena_alone(eng, monkeypatch, case):
    """Only the requested, scored columns are written, and only rows [0, n): every other byte of an arena
    pre-filled with a sentinel keeps it."""
    from cropsr_b200 import _native as N
    monkeypatch.setenv("CRP_PIECE_POSITIONS", "16384")
    want = {"pos": ("pos",), "pos+x": ("pos", "x"), "pos+packed": ("pos", "packed"), "packed+x": ("packed", "x"),
            "no_score": ("pos", "packed", "x"), "l18": ("pos", "packed", "x")}[case]
    l = 18 if case == "l18" else 20
    flags = N.CRP_SCAN_NO_SCORE if case == "no_score" else 0
    toks = [random_token(80 + k, n) for k, n in enumerate((50001, 300, 29, 21000))]
    segs = [(k, t, 0, len(t)) for k, t in enumerate(toks)]
    counts, rows = expected(segs, l)
    arena = full_arena(eng, max(sum(counts["+"]), sum(counts["-"])) + 333)
    cols = {s: dict(arena.arrays[s]) for s in "+-"}
    for s in "+-":                     # hide what was not asked for: the library gets NULL there
        for name in cols[s]:
            if name not in want:
                arena.arrays[s][name] = None
    got, n_plus, n_minus, _ = eng.scan_segments(segs, l, flags=flags, arena=arena, want=want)
    assert got is arena
    assert n_plus.tolist() == counts["+"] and n_minus.tolist() == counts["-"]
    scored = l == 20 and not flags
    for s, n in (("+", sum(counts["+"])), ("-", sum(counts["-"]))):
        for name, v in cols[s].items():
            written = name in want and (name == "pos" or scored)
            b = v.view(np.uint8)
            head = b[:n * v.itemsize]
            assert (b[n * v.itemsize:] == SENTINEL).all(), (s, name)
            if not written:
                assert (head == SENTINEL).all(), (s, name)
        c = {name: cols[s][name][:n] if name in want and (name == "pos" or scored) else None for name in cols[s]}
        check_rows(rows, s, c["pos"], c["packed"], c["x"])
    arena.free()


# ---------------------------------------------------------------- 7. arena edges
@pytest.mark.gpu
def test_arena_edges(eng, monkeypatch):
    monkeypatch.setenv("CRP_PIECE_POSITIONS", "16384")
    toks = [random_token(90 + k, n) for k, n in enumerate((60001, 300, 20481))]
    segs = [(k, t, 0, len(t)) for k, t in enumerate(toks)]
    counts, rows = expected(segs, 20)
    exact = max(sum(counts["+"]), sum(counts["-"]))
    # capacity exactly the larger strand: one library call, the arena comes back
    arena = eng.Arena(exact, True)
    got, _, _ = run_and_check(eng, segs, 20, 16384, arena=arena)
    assert got is arena
    # one row short: the call answers CRP_ERR_RANGE with the counts, and engine.scan_segments repeats it
    small = eng.Arena(exact - 1, True)
    before = eng.perf_report()
    got2, n_plus, n_minus, ms = eng.scan_segments(segs, 20, arena=small)
    planned(eng, before, [(len(t), 0, len(t)) for t in toks], 16384, calls=2)
    assert got2 is not small and got2.capacity >= exact and ms > 0
    assert n_plus.tolist() == counts["+"] and n_minus.tolist() == counts["-"]
    for s, n in (("+", sum(counts["+"])), ("-", sum(counts["-"]))):
        a = got2.arrays[s]
        check_rows(rows, s, a["pos"][:n], a["packed"][:n], a["x"][:n])
    got2.free()
    # an arena reused from a larger call: only rows [0, n) are the new call's
    short = [(0, toks[1], 0, len(toks[1])), (1, toks[0], 16384, 20000)]
    got3, _, _ = run_and_check(eng, short, 20, 16384, arena=arena)
    assert got3 is arena
    arena.free()
    # no segment at all
    before = eng.perf_report()["commits"]
    a0, p0, m0, ms0 = eng.scan_segments([], 20)
    assert len(p0) == 0 and len(m0) == 0 and eng.perf_report()["commits"] == before
    a0.free()


# ---------------------------------------------------------------- 8. the end of a segment is taken literally
@pytest.mark.gpu
def test_segment_end_is_taken_literally(eng, monkeypatch):
    """[begin, end) is what the descriptor says: end = 0 owns nothing, as it does for add_segment, and a
    descriptor add_segment would refuse is refused before any group is copied, packed or scanned."""
    from cropsr_b200 import _native as N
    from cropsr_b200._native import CropsrError
    monkeypatch.setenv("CRP_PIECE_POSITIONS", "16384")
    tok = random_token(5, 60000)
    other = random_token(6, 40000)
    for b, e in ((0, 0), (128, 128), (TILE, TILE)):
        g = eng.Genome()
        g.add_segment(0, tok, b, e)
        res = g.commit().scan(20)
        assert res.n_plus == res.n_minus == 0
        res.free()
        g.free()
        arena, n_plus, n_minus, _ = eng.scan_segments([(0, tok, b, e)], 20)
        assert n_plus.tolist() == [0] and n_minus.tolist() == [0]
        arena.free()
    # an empty segment between two others: the others' rows, nothing from it
    arena, n_plus, n_minus = run_and_check(eng, [(0, other, 0, 40000), (1, tok, 0, 0), (0, other, 0, 16384)], 20, 16384)
    assert n_plus[1] == n_minus[1] == 0
    arena.free()
    good = [(0, other, 0, 40000), (1, tok, 0, 60000), (0, other, 128, 30000)]
    bad = [(1, tok, 4096, 0), (1, tok, 256, 128), (1, tok, 0, 60001), (1, tok, 100, 200), (1, tok, 16384 + 64, 30000)]
    for d in bad:
        for where in (0, 1, len(good)):
            segs = good[:where] + [d] + good[where:]
            before = eng.perf_report()
            with pytest.raises(CropsrError) as e:
                eng.scan_segments(segs, 20, arena=eng.Arena(100000, True))
            assert e.value.code == CRP_ERR_ARG, (d, where)
            after = eng.perf_report()
            assert after["commits"] == before["commits"] and after["scans"] == before["scans"], (d, where)
    # through the C ABI directly: a NULL token of positive length, a token past the 31-bit range
    import ctypes as C
    buf = np.frombuffer(tok.encode(), np.uint8)
    for desc in (N.SegmentDesc(0, None, 100, 0, 0), N.SegmentDesc(0, buf.ctypes.data, (1 << 31) - (1 << 15), 0, 16)):
        descs = (N.SegmentDesc * 2)(N.SegmentDesc(1, buf.ctypes.data, len(buf), 0, len(buf)), desc)
        n_plus = np.full(2, 7, np.uint64)
        n_minus = np.full(2, 7, np.uint64)
        before = eng.perf_report()["commits"]
        rc = N.lib.crp_scan_segments(2, descs, 20, 0, 0, None, None, None, None, None, None,
                                     n_plus.ctypes.data, n_minus.ctypes.data, None)
        assert rc == CRP_ERR_ARG and eng.perf_report()["commits"] == before
        assert n_plus.tolist() == [0, 0] and n_minus.tolist() == [0, 0]


# ---------------------------------------------------------------- 9. at size
def _arabidopsis():
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
    import workloads as W
    return [W.token("arabidopsis", k) for k in range(len(W.token_lengths("arabidopsis")))]


def _digest_token(d, k, arena, first, n_p, n_m, cols=("pos", "packed", "x")):
    p, m = arena.arrays["+"], arena.arrays["-"]
    d.add_token(k, tuple(p[c][first[0]:first[0] + n_p] for c in cols), tuple(m[c][first[1]:first[1] + n_m] for c in cols))


@pytest.mark.gpu
def test_configs1_through_the_pipelined_call_equals_oracle_digest(eng, monkeypatch):
    """configs[1] (5 chromosomes of 21-34 Mbp) with the default 32 Mi pieces and with 4 Mi pieces (5-8
    pieces per chromosome): the whole-table digest of the committed oracle; then bench's flags and columns
    give the same positions and the logistic of the same x."""
    import json
    import vector_oracle as vo
    from cropsr_b200 import _native as N
    from helpers import GOLDEN
    with open(os.path.join(GOLDEN, "table_digests.json")) as f:
        want = json.load(f)["arabidopsis"]
    toks = _arabidopsis()
    segs = [(k, t, 0, len(t)) for k, t in enumerate(toks)]
    arena = None
    for P_env in (None, 4194304):
        if P_env is None:
            monkeypatch.delenv("CRP_PIECE_POSITIONS", raising=False)
        else:
            monkeypatch.setenv("CRP_PIECE_POSITIONS", str(P_env))
        before = eng.perf_report()
        arena, n_plus, n_minus, _ = eng.scan_segments(segs, 20, arena=arena)
        planned(eng, before, [(len(t), 0, len(t)) for t in toks], piece_size(P_env))
        d = vo.TableDigest()
        first = [0, 0]
        for k in range(len(toks)):
            _digest_token(d, k, arena, first, int(n_plus[k]), int(n_minus[k]))
            first[0] += int(n_plus[k])
            first[1] += int(n_minus[k])
        assert (d.tokens, d.candidates) == (want["tokens"], want["candidates"]), P_env
        assert d.hexdigest() == want["sha256"], P_env
    n = {"+": int(n_plus.sum()), "-": int(n_minus.sum())}
    log, lp, lm, _ = eng.scan_segments(segs, 20, flags=N.CRP_SCAN_LOGISTIC, want=("pos", "x"))
    assert np.array_equal(lp, n_plus) and np.array_equal(lm, n_minus)
    for s in "+-":
        assert np.array_equal(log.arrays[s]["pos"][:n[s]], arena.arrays[s]["pos"][:n[s]])
        assert np.array_equal(log.arrays[s]["x"][:n[s]], eng.logistic(arena.arrays[s]["x"][:n[s]]))
    log.free()
    arena.free()


# ---------------------------------------------------------------- 10. maize through bench's e2e inputs
@pytest.mark.gpu
@pytest.mark.slow
def test_maize_shard_plans_through_the_pipelined_call_equal_oracle_digest(eng, monkeypatch):
    """configs[3] (10 chromosomes of 150-307 Mbp, 2.29 Gbp) as bench's e2e leg feeds it at 2 and 8 GPUs:
    every rank's shard.plan segments with the default 32 Mi pieces, so every chromosome is cut; the rows,
    taken in the order shard.global_offsets places them, hash to the committed digest."""
    import json
    import sys
    import vector_oracle as vo
    from cropsr_b200 import shard
    from helpers import GOLDEN
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tools"))
    import workloads as W
    monkeypatch.delenv("CRP_PIECE_POSITIONS", raising=False)
    with open(os.path.join(GOLDEN, "table_digests.json")) as f:
        want = json.load(f)["maize"]
    lengths = W.token_lengths("maize")
    toks = [W.token("maize", k) for k in range(len(lengths))]
    arena = eng.Arena(max(want["plus"], want["minus"]), True)
    for world in (2, 8):
        plans = shard.plan(lengths, world)
        counts = []
        d = vo.TableDigest()
        pending = {}            # token -> rows of its pieces so far, per strand (a token ends on a later rank)
        placed = {"+": 0, "-": 0}
        rank_rows = []
        for segs in plans:
            arena, n_plus, n_minus, _ = eng.scan_segments([(k, toks[k], a, b) for k, a, b in segs], 20, arena=arena)
            counts.append((n_plus.copy(), n_minus.copy()))
            first = [0, 0]
            for s, (k, a, b) in enumerate(segs):
                parts = pending.setdefault(k, {"+": [], "-": []})
                for si, strand in enumerate("+-"):
                    n = int((n_plus, n_minus)[si][s])
                    cols = arena.arrays[strand]
                    parts[strand].append(tuple(cols[c][first[si]:first[si] + n].copy() for c in ("pos", "packed", "x")))
                    rank_rows.append((len(counts) - 1, s, si, n))
                    first[si] += n
                if b == lengths[k]:
                    rows = {st: tuple(np.concatenate([p[i] for p in parts[st]]) for i in range(3)) for st in "+-"}
                    d.add_token(k, rows["+"], rows["-"])
                    del pending[k]
        assert not pending
        # the placement bench derives from the counts: each token's '+' rows, then its '-' rows, pieces in rank order
        offs, total = shard.global_offsets(plans, counts)
        assert total == want["candidates"]
        run = 0
        token_start = {}
        for k in range(len(lengths)):
            token_start[k] = run
            run += sum(int(counts[r][si][s]) for r, segs in enumerate(plans) for s, seg in enumerate(segs)
                       if seg[0] == k for si in (0, 1))
        seen = {}
        for r, s, si, n in rank_rows:
            k = plans[r][s][0]
            key = (k, si)
            if key not in seen:
                plus_total = sum(int(counts[rr][0][ss]) for rr, sg in enumerate(plans) for ss, g in enumerate(sg) if g[0] == k)
                seen[key] = token_start[k] + (plus_total if si else 0)
            assert offs[r][s][si] == seen[key], (world, r, s, si)
            seen[key] += n
        assert (d.tokens, d.candidates) == (want["tokens"], want["candidates"]), world
        assert d.hexdigest() == want["sha256"], world
    arena.free()


# ---------------------------------------------------------------- 11. checked build
@pytest.mark.gpu
def test_checked_build_sees_no_violated_invariant_in_the_pipelined_call(eng):
    """Cases 1-5 again under libcropsr_b200_checked.so (make checked), in a subprocess: k_scan_score
    verifies its own invariants on every group, rerun and piece of them."""
    import subprocess
    import sys
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
    sel = ("test_piece_edges or test_guide_lengths_across_pieces or test_segments_that_start_inside or "
           "test_bench_e2e_inputs or test_capacity_rerun")
    out = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "tests/test_scan_segments.py", "-k", sel],
                         cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]


@pytest.mark.gpu
def test_tile_constant(eng):
    assert eng.TILE == TILE
