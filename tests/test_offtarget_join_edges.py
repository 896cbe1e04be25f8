"""The off-target join at its edges (csrc/offtarget.cuh: k_ot_join<OtCount | OtList | OtScore> and the geometry of its
work items).

CPU: the geometry (bucket search, tiles, bulk-copy window, thread split) run on the host from the same source
(tests/offtarget_join_emu.cu); the numpy model of the join's buckets against a direct pairwise count.
GPU: genomes built from site families so that chosen bucket shapes occur -- queries x sites across tile edges, every
first-site residue of a bucket of several site tiles, buckets 0 and 65535, a part pair with more work items than the
persistent grid has CTAs.  Every shape is asserted through the model, and the model's comparisons must equal the
device's after every call.  At those shapes counts, listings and scores (random, 2^31 - 1 and one-hot weights) equal
brute force for k = 0 .. 3, at NGG and at NAG; candidates inside a bucket of three site tiles leave their own site out
exactly once."""
import functools
import os
import shutil
import subprocess
from math import comb

import numpy as np
import pytest

import offtarget_oracle as ot
import offtarget_pam_oracle as pam_oracle
import offtarget_sites_oracle as sites_oracle
from helpers import ROOT

THREADS, SITE_TILE, BUCKETS = 128, 2048, 1 << 16      # kOtThreads, kOtSiteTile, kOtBuckets
PAIRS = [(i, j) for i in range(5) for j in range(i + 1, 5)]   # ot_pair order


# ---------------------------------------------------------------- the model of the join's buckets
def bucket_of(keys, i, j):
    """ot_bucket: the 8 nt of parts i and j"""
    keys = np.asarray(keys, dtype=np.uint64)
    lo = (keys >> np.uint64(8 * i)) & np.uint64(0xFF)
    hi = (keys >> np.uint64(8 * j)) & np.uint64(0xFF)
    return (lo | hi << np.uint64(8)).astype(np.int64)


def join_model(site_keys, query_keys):
    """Per part pair, in ot_pair order, what k_ot_hist / k_ot_scan build for these keys (queries with a protospacer
    only): per bucket ns, nq, soff (first site, so soff % 4 and % 2 are the residues of the uint32 and uint2 copies),
    items; item_off and the pair's total items."""
    model = []
    for i, j in PAIRS:
        ns = np.bincount(bucket_of(site_keys, i, j), minlength=BUCKETS).astype(np.int64)
        nq = np.bincount(bucket_of(query_keys, i, j), minlength=BUCKETS).astype(np.int64)
        items = np.where((ns > 0) & (nq > 0), -(-nq // THREADS) * -(-ns // SITE_TILE), 0)
        model.append(dict(pair=(i, j), ns=ns, nq=nq, soff=np.concatenate(([0], np.cumsum(ns)))[:-1], items=items,
                          item_off=np.concatenate(([0], np.cumsum(items))), total=int(items.sum())))
    return model


def model_comparisons(model):
    """sum over the ten pairs and every bucket of nq * ns: what the device reports as comparisons"""
    return sum(int((m["ns"] * m["nq"]).sum()) for m in model)


def model_buckets(model):
    """(pair, bucket, nq, ns, soff) of every bucket with work items"""
    return [(p, int(b), int(m["nq"][b]), int(m["ns"][b]), int(m["soff"][b]))
            for p, m in enumerate(model) for b in np.nonzero(m["items"])[0]]


def test_model_equals_a_direct_pairwise_count():
    rng = np.random.default_rng(5)
    base = rng.integers(0, 1 << 40, size=6, dtype=np.uint64)

    def mutate(n):                                  # copies of a few keys with a few random bases changed
        keys = base[rng.integers(0, len(base), size=n)].copy()
        for _ in range(3):
            pos = rng.integers(0, 20, size=n).astype(np.uint64) * np.uint64(2)
            keys ^= rng.integers(0, 4, size=n).astype(np.uint64) << pos
        return keys
    sites, queries = mutate(400), np.concatenate((mutate(150), [0, (1 << 40) - 1]))
    sites = np.concatenate((sites, [0, 0, (1 << 40) - 1]))
    model = join_model(sites, queries)
    direct = 0
    for p, (i, j) in enumerate(PAIRS):
        part = lambda k, n: (int(k) >> (8 * n)) & 0xFF
        same = [(part(q, i), part(q, j)) == (part(s, i), part(s, j)) for q in queries for s in sites]
        direct += sum(same)
        for b in {part(q, i) | part(q, j) << 8 for q in queries}:
            assert model[p]["nq"][b] == sum(part(q, i) | part(q, j) << 8 == b for q in queries)
            assert model[p]["ns"][b] == sum(part(s, i) | part(s, j) << 8 == b for s in sites)
        m = model[p]
        assert m["item_off"][-1] == m["total"] == sum(-(-int(m["nq"][b]) // 128) * -(-int(m["ns"][b]) // 2048)
                                                      for b in range(BUCKETS) if m["nq"][b] and m["ns"][b])
    assert model_comparisons(model) == direct > 0
    assert {(p, b) for p, b, _, _, _ in model_buckets(model)} >= {(p, 0) for p in range(10)} | {(p, BUCKETS - 1) for p in range(10)}


def test_join_geometry_on_the_cpu(tmp_path):
    """tests/offtarget_join_emu.cu compiles the work-item geometry of k_ot_join -- the SAME source -- for the host and
    checks bucket search, tiling, copy window and thread split exhaustively over bucket tables built as k_ot_scan builds
    them."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "offtarget_join_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "offtarget_join_emu.cu")], check=True, capture_output=True, timeout=600)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


# ---------------------------------------------------------------- site families
def _rc(s):
    return s[::-1].translate(str.maketrans("ACGTacgt", "TGCAtgca"))


def _key(p):
    return ot.key_of(p)


def _substitute(rng, p, positions):
    """p with a different base at each position (never C at position 0, see _unit)"""
    q = list(p)
    for x in positions:
        q[x] = rng.choice([b for b in "ACGT" if b != p[x] and not (x == 0 and b == "C")])
    return "".join(q)


def _positions(rng, parts, n_extra, avoid):
    """one position in each of `parts`, then n_extra more in parts not in `avoid` (a second one in a part if need be)"""
    pos = [4 * m + int(rng.integers(0, 4)) for m in parts]
    free = [4 * m + r for m in range(5) if m not in avoid for r in range(4) if 4 * m + r not in pos]
    rng.shuffle(free)
    free.sort(key=lambda x: x // 4 in parts)        # untouched parts first
    return pos + free[:n_extra]


def variants(rng, p):
    """Copies of p at d = 1, 2, 3 such that every part pair (i, j) is the counting pair (the two lowest exact parts) of
    some copy at every d it admits (d >= j - 1), and copies at d = 4 that must not count: [(protospacer, d, (i, j))]"""
    out = []
    for i, j in PAIRS:
        below = [m for m in range(j) if m != i]
        for d in range(max(len(below), 1), 4):
            out.append((_substitute(rng, p, _positions(rng, below, d - len(below), {i, j})), d, (i, j)))
    for _ in range(6):
        out.append((_substitute(rng, p, rng.choice(20, size=4, replace=False)), 4, None))
    return out


def decoy(rng, p):
    """p's parts 0 and 1 with >= 4 substitutions in parts 2 .. 4: in p's bucket of pair (0, 1), within k of nothing there"""
    return _substitute(rng, p, 8 + rng.choice(12, size=int(rng.integers(4, 8)), replace=False))


def _unit(p, pam, rng, lower=None):
    """NN + protospacer + PAM in a random orientation and case.  The NN keeps units from lending each other bases or a
    PAM; a protospacer that does not start with C makes the unit hold no other site of NGG or NAG."""
    s = p + pam
    if (rng.random() < 0.3) if lower is None else lower:
        s = s.lower()
    return "NN" + (_rc(s) if rng.random() < 0.5 else s)


def _base(rng, used):
    """a protospacer whose five parts differ from those of every base chosen before (and not C at position 0)"""
    while True:
        p = "".join(rng.choice(list("ACGT"), 20))
        parts = {(m, p[4 * m:4 * m + 4]) for m in range(5)}
        if p[0] != "C" and not parts & used:
            used |= parts
            return p


# ---------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def _genome(eng, tok):
    g = eng.Genome()
    g.add_token(tok)
    g.commit()
    return g


def _count(index, keys, k):
    from cropsr_b200._native import check, lib
    out = np.empty((len(keys), k + 1), dtype=np.uint32)
    check(lib.crp_offtarget_count_keys(index._h, len(keys), keys.ctypes.data, k, out.ctypes.data))
    return out


def _list(index, keys, k, counts):
    from cropsr_b200._native import check, lib
    first = np.zeros(len(keys) + 1, dtype=np.uint64)
    np.cumsum(counts.astype(np.uint64).sum(axis=1), out=first[1:])
    out = np.empty(int(first[-1]), dtype=np.uint32)
    check(lib.crp_offtarget_list_keys(index._h, len(keys), keys.ctypes.data, k, first.ctypes.data,
                                      out.ctypes.data if len(out) else None))
    return first, out


def _score(index, keys, k, w):
    from cropsr_b200._native import check, lib
    out = np.empty(len(keys), dtype=np.uint64)
    check(lib.crp_offtarget_score_keys(index._h, len(keys), keys.ctypes.data, k, w.ctypes.data, out.ctypes.data))
    return out


_COMB = np.array([[comb(p, e) for e in range(4)] for p in range(20)], dtype=np.int64)


def ranks(key, site_keys):
    """(mismatches, colex rank of the mismatch-position set) of key against every site (rank meaningful for d <= 3)"""
    d = ot.mismatches(np.uint64(key), site_keys)
    near = np.nonzero(d <= 3)[0]
    x = np.bitwise_xor(np.uint64(key), np.asarray(site_keys, dtype=np.uint64)[near])
    y = (x | x >> np.uint64(1)) & np.uint64(0x5555555555)
    bits = ((y[:, None] >> (np.uint64(2) * np.arange(20, dtype=np.uint64))) & np.uint64(1)).astype(np.int64)
    e = np.cumsum(bits, axis=1)                       # position p is element e of the set (1 = the lowest)
    r = np.zeros(len(d), dtype=np.int64)
    r[near] = np.array([0, 1, 21, 211])[d[near]] + (bits * _COMB[np.arange(20), np.minimum(e, 3)]).sum(axis=1)
    return d, r


def _check_index(index, tok, pam):
    """the index holds the oracle's sites of tok: returns the oracle's (key, t, strand) as the device orders them"""
    t, s, keys = pam_oracle.site_keys_np(tok.encode(), pam)
    dev = index.sites()
    _, _, lt, ls = index.site_loci()
    assert sorted(zip(dev.tolist(), lt.tolist(), ls.tolist())) == sorted(zip(keys.tolist(), t.tolist(), s.tolist()))
    return dev, lt, ls


def _weight_tables(rng, one_hot_ranks):
    tables = {"random": rng.integers(0, 1 << 31, size=1351, dtype=np.uint32),
              "max": np.full(1351, (1 << 31) - 1, dtype=np.uint32)}
    for d, r in one_hot_ranks.items():
        w = np.zeros(1351, dtype=np.uint32)
        w[r] = (1 << 31) - 1
        tables[f"one-hot d={d}"] = w
    return tables


# ---------------------------------------------------------------- shapes on purpose, against brute force
NQ = (1, 2, 3, 43, 64, 65, 127, 128, 129, 255, 256, 257)
NS = (1, 2047, 2048, 2049, 4096, 4097)
BIG_NQ, BIG_NS = 65536, 4097            # 512 query tiles x 3 site tiles at pair (0, 1): 1,536 work items


@functools.lru_cache(maxsize=1)
def grid_genome(seed):
    """One token of site families: for every (nq, ns) of NQ x NS a base protospacer whose bucket of pair (0, 1) holds
    exactly ns sites (exact copies, the variants of `variants` that keep parts 0 and 1, decoys), queried by nq copies
    of its key; a family of BIG_NS sites for BIG_NQ queries; all-A and all-G protospacers (buckets 0 and 65535 of every
    pair) with a few queries; random guides that find no bucket.  Every unit once with AGG (an NGG site) and once with
    AAG (a NAG site), so both indexes have the same keys.  -> (token, query keys, {key: (nq, ns)})"""
    rng = np.random.default_rng(seed)
    used = {(m, x * 4) for m in range(5) for x in "AG"}
    units, queries, targets = [], [], {}

    def family(nq, ns):
        p = _base(rng, used)
        sites = [p]
        if ns >= SITE_TILE - 1:                    # exact copies, the rich variants, decoys up to ns in the bucket
            sites += [p] * 63
            sites += [v for v, _, _ in variants(rng, p)]
            in_bucket = sum(v[:8] == p[:8] for v in sites)
            sites += [decoy(rng, p) for _ in range(ns - in_bucket)]
        assert sum(v[:8] == p[:8] for v in sites) == ns
        units.extend((v, p[:8]) for v in sites)
        queries.extend([_key(p)] * nq)
        targets[_key(p)] = (nq, ns)

    for nq in NQ:
        for ns in NS:
            family(nq, ns)
    family(BIG_NQ, BIG_NS)
    # a variant whose changed parts 0 and 1 happen to be those of another family would add a site to its bucket
    prefixes = {q for _, q in units}
    units = [v for v, q in units if v[:8] == q or v[:8] not in prefixes]
    units += ["A" * 20] * 3 + ["G" * 20] * 5
    queries += [0] * 2 + [(1 << 40) - 1]
    queries += [_key(_base(rng, used)) for _ in range(20)]
    order = rng.permutation(len(units))
    tok = "".join(_unit(units[i], pam, rng) for i in order for pam in ("AGG", "AAG")) + "NN"
    return tok, np.array(queries, dtype=np.uint64), targets


def _assert_shapes(model, queries, targets, sm_count):
    buckets = model_buckets(model)
    pair01 = {(nq, ns) for p, _, nq, ns, _ in buckets if p == 0}
    assert pair01 >= {(nq, ns) for nq in NQ for ns in NS} | {(BIG_NQ, BIG_NS)}
    multi = [s0 for _, _, _, ns, s0 in buckets if ns > SITE_TILE]
    assert {s0 % 4 for s0 in multi} == {0, 1, 2, 3}            # uint32 sites: every residue of the copy's start
    assert {s0 % 2 for s0 in multi} == {0, 1}                  # uint2 sites
    assert {b for p, b, _, _, _ in buckets} >= {0, BUCKETS - 1}
    assert max(m["total"] for m in model) > 8 * sm_count       # more items than the persistent grid has CTAs
    assert any(((m["ns"] > 0) & (m["nq"] == 0)).any() for m in model)   # buckets with sites and no queries
    assert any(((m["ns"] == 0) & (m["nq"] > 0)).any() for m in model)   # and with queries and no sites


@pytest.mark.gpu
@pytest.mark.parametrize("pam", ["NGG", "NAG"])
def test_counts_listings_and_scores_at_chosen_bucket_shapes(eng, pam):
    tok, queries, targets = grid_genome(17)
    sm_count = eng.perf_report()["sm_count"]
    g = _genome(eng, tok)
    index = eng.OffTargetIndex([g], loci=True, pam=pam)
    try:
        dev_keys, _, _ = _check_index(index, tok, pam)
        model = join_model(dev_keys, queries)
        _assert_shapes(model, queries, targets, sm_count)
        want_cmp = model_comparisons(model)
        uniq, row_of = np.unique(queries, return_inverse=True)
        per_key = [ranks(q, dev_keys) for q in uniq]            # brute force over the index's sites, per distinct key
        rng = np.random.default_rng(3)
        big = next(key for key, shape in targets.items() if shape == (BIG_NQ, BIG_NS))
        d0, r0 = ranks(big, dev_keys)
        one_hot = {d: int(r0[d0 == d][0]) for d in range(4)}    # a set of every size that occurs
        tables = _weight_tables(rng, one_hot)
        for k in range(4):
            want_counts = np.array([np.bincount(d[d <= k], minlength=k + 1) for d, _ in per_key])
            got = _count(index, queries, k)
            assert index.timing()["comparisons"] == want_cmp
            assert np.array_equal(got.astype(np.int64), want_counts[row_of]), k
            # listings: every row lists exactly its brute-force sites, each once
            first, listed = _list(index, queries, k, got)
            assert index.timing()["comparisons"] == want_cmp
            rows = np.repeat(np.arange(len(queries)), np.diff(first).astype(np.int64))
            got_sorted = listed[np.lexsort((listed, rows))]
            want_sites = [np.nonzero(d <= k)[0] for d, _ in per_key]
            want_sorted = np.concatenate([want_sites[u] for u in row_of]) if len(listed) else listed
            assert np.array_equal(got_sorted.astype(np.int64), want_sorted), k
            for name, w in tables.items():
                got_s = _score(index, queries, k, w)
                assert index.timing()["comparisons"] == want_cmp
                want_s = np.array([int(w[r[d <= k]].astype(np.uint64).sum()) for d, r in per_key], dtype=np.uint64)
                assert np.array_equal(got_s, want_s[row_of]), (k, name)
                if name == "max" and k == 3:
                    assert want_s.max() > 1 << 32                      # rows pass 2^32
    finally:
        index.free()
        g.free()


# ---------------------------------------------------------------- candidates in a dense bucket
def dense_genome(seed, n_copies=4100):
    """n_copies lower-case copies (sites, not candidates) of one protospacer in both orientations and its variants; one
    upper-case '+' copy (a candidate) in front of them and two '+' and two '-' behind them, so that their own sites
    need not fall in the first of the bucket's three site tiles.  Every unit with agg and again with aag (NAG sites of
    the same keys).  A strand stream has 2 or 3 candidate rows: nq_t = 2 or 3, 64 or 42 threads per query."""
    rng = np.random.default_rng(seed)
    p = _base(rng, set())
    while "GG" in p or "CC" in p:                   # no scan candidates inside the upper-case copies
        p = _base(rng, set())
    low = [_unit(p, "agg", rng, lower=True) + _unit(p, "aag", rng, lower=True) for _ in range(n_copies)]
    var = [_unit(v, "agg", rng, lower=True) + _unit(v, "aag", rng, lower=True) for v, _, _ in variants(rng, p)]
    plus, minus = "NN" + p + "AGG", "NN" + _rc(p + "AGG")
    tok = plus + "".join(low[:2000]) + "".join(var) + "".join(low[2000:]) + plus * 2 + minus * 2 + "NN"
    return tok, p


@pytest.mark.gpu
@pytest.mark.parametrize("pam", ["NGG", "NAG"])
def test_candidates_in_a_bucket_of_three_site_tiles_leave_their_own_site_out_once(eng, pam):
    tok, p = dense_genome(23)
    g = _genome(eng, tok)
    r = g.scan(20)
    index = eng.OffTargetIndex([g], loci=True, pam=pam)
    own = pam == "NGG"
    try:
        dev_keys, lt, ls = _check_index(index, tok, pam)
        ot_t, ot_s, ot_k = pam_oracle.site_keys_np(tok.encode(), pam)
        d_all, r_all = ranks(_key(p), dev_keys)
        tables = _weight_tables(np.random.default_rng(4), {d: int(r_all[d_all == d][0]) for d in range(1, 4)} | {0: 0})
        for si, strand in enumerate("+-"):
            pos = r.fetch(strand, want=("pos",))["pos"].astype(np.int64)
            assert len(pos) in (2, 3)                                   # g = 64 or 42 threads per query
            model = join_model(dev_keys, np.array([_key(p)] * len(pos), dtype=np.uint64))
            assert any(nq == len(pos) and ns > 2 * SITE_TILE for _, _, nq, ns, _ in model_buckets(model))
            for k in range(4):
                want = np.bincount(d_all[d_all <= k], minlength=k + 1)
                want[0] -= own                                         # the own site, only where it is a site
                c = index.count_candidates(r, strand, k)
                assert index.timing()["comparisons"] == model_comparisons(model)
                assert np.array_equal(c.astype(np.int64), np.tile(want, (len(pos), 1))), (strand, k)
                rows, first, listed = index.list_candidates(r, strand, k, counts=c)
                assert index.timing()["comparisons"] == model_comparisons(model)
                for i, t in enumerate(pos):
                    got = listed[int(first[i]):int(first[i + 1])].astype(np.int64)
                    assert len(np.unique(got)) == len(got)
                    sel, _ = sites_oracle.neighbours_np(_key(p), ot_k, k)
                    keep = ~((ot_t[sel] == t) & (ot_s[sel] == si))       # the listing leaves out the own locus
                    assert own == (not keep.all())
                    want_l = sorted(zip(ot_k[sel][keep].tolist(), ot_t[sel][keep].tolist(), ot_s[sel][keep].tolist()))
                    assert sorted(zip(dev_keys[got].tolist(), lt[got].tolist(), ls[got].tolist())) == want_l, (strand, k, i)
                for name, w in tables.items():
                    s = index.score_candidates(r, strand, k, weights=w)
                    assert index.timing()["comparisons"] == model_comparisons(model)
                    want_s = int(w[r_all[d_all <= k]].astype(np.uint64).sum()) - (int(w[0]) if own else 0)
                    assert s.tolist() == [want_s] * len(pos), (strand, k, name)
                    if name == "max":
                        assert want_s > 1 << 36                            # one thread's slice of a tile passes 2^32
    finally:
        index.free()
        r.free()
        g.free()
