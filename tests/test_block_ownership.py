"""Every device and pinned block a library call takes from the block cache goes back to it (csrc/cropsr_b200.cu
DevBuf, PinnedBuf): perf_report()["block_cache"]'s live_blocks and pinned_live_blocks are the same after each call
below as before it -- successful calls, whole object lifetimes, and error returns after device work.  No call here
provokes a CUDA error or runs out of memory."""
import ctypes as C

import numpy as np
import pytest

from helpers import synthetic_fasta


@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


def _live(eng):
    c = eng.perf_report()["block_cache"]
    return c["live_blocks"], c["pinned_live_blocks"]


def _gives_back(eng, call, code=None):
    """call() leaves as many blocks handed out as it found; code: the CropsrError code it must fail with"""
    from cropsr_b200._native import CropsrError
    before = _live(eng)
    if code is None:
        call()
    else:
        with pytest.raises(CropsrError) as e:
            call()
        assert e.value.code == code
    assert _live(eng) == before


def _tokens():
    """two tokens; N bytes give other runs and candidates without a protospacer (NO_COUNT rows), and a copy of 5 kbp of
    the first at the end of the second gives candidates with off-target sites"""
    from cropsr_b200 import ingest
    a, b = ingest.fasta_text_to_tokens(synthetic_fasta(7, [60000, 30000], gc=0.5, n_frac=0.005)).values()
    return [a, b + a[10000:15000]]


def _genome(eng, tokens):
    g = eng.Genome()
    for t in tokens:
        g.add_token(t)
    return g.commit()


@pytest.mark.gpu
def test_successful_calls_give_back_every_block(eng):
    from cropsr_b200 import primers
    tokens = _tokens()
    g = _genome(eng, tokens)
    r = g.scan(20)
    index = eng.OffTargetIndex([g], loci=True)
    try:
        rng = np.random.default_rng(1)
        rows = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=(300, 30))
        _gives_back(eng, lambda: eng.rs1_score(rows, np.zeros(300, np.uint8)))
        _gives_back(eng, lambda: eng.logistic(rng.normal(size=1000)))
        pos = r.fetch_segment(0, "+")["pos"][:50]
        assert len(pos) == 50
        _gives_back(eng, lambda: g.rescore(np.zeros(50, np.uint32), pos, np.full(50, b"+", "S1"), np.zeros(50, np.uint8)))
        _gives_back(eng, lambda: r.extras(1, "-"))
        _gives_back(eng, lambda: r.extras_strand("+"))
        start, end = np.array([100, 5000], np.uint32), np.array([2000, 9000], np.uint32)
        _gives_back(eng, lambda: r.annotate(0, "+", start, end))
        _gives_back(eng, lambda: r.annotate_strand("-", np.array([0, 2, 2], np.uint64), start, end))
        _gives_back(eng, lambda: g.other_runs(0))
        _gives_back(eng, lambda: primers.design_windows(g, [0, 1], [1000, 2000], [1600, 2700]))
        _gives_back(eng, lambda: eng.scan_segments([(k, t, 0, None) for k, t in enumerate(tokens)], 20)[0].free())
        _gives_back(eng, eng.flush_l2)
        _gives_back(eng, lambda: eng.link_probe(1 << 20, 1 << 20, 2))
        guides = ["GATTACAGCTTCAGTCATCA", "acgtacgtacgtacgtacgt"]
        for s in "+-":
            _gives_back(eng, lambda: index.count_candidates(r, s, 3))
            _gives_back(eng, lambda: index.list_candidates(r, s, 2))
            _gives_back(eng, lambda: index.score_candidates(r, s, 3))
        _gives_back(eng, lambda: index.count_guides(guides, 3))
        _gives_back(eng, lambda: index.list_guides(guides, 3))
        _gives_back(eng, lambda: index.score_guides(guides, 3))
    finally:
        index.free()
        r.free()
        g.free()


@pytest.mark.gpu
def test_object_lifetimes_give_back_every_block(eng):
    tokens = _tokens()
    before = _live(eng)
    g = _genome(eng, tokens)
    held = _live(eng)
    assert held[0] > before[0]
    r = g.scan(20)
    assert _live(eng)[0] > held[0] and _live(eng)[1] > held[1]          # streams, state and pinned counts
    r.free()
    assert _live(eng) == held
    for loci, pam in ((False, "NGG"), (True, "NGG"), (True, "NAG"), (False, "NRG")):
        index = eng.OffTargetIndex([g], loci=loci, pam=pam)
        g2 = _genome(eng, tokens[1:])
        index.add_genome(g2)                       # the growth step: the site arrays are replaced
        assert index.num_sites() > 0
        g2.free()
        index.free()
        assert _live(eng) == held, (loci, pam)
    g.free()
    assert _live(eng) == before


@pytest.mark.gpu
def test_device_fasta_genome_gives_back_every_block(eng):
    from cropsr_b200 import ingest
    text = synthetic_fasta(8, [20000, 9000], width=60).encode()
    arr = np.frombuffer(text, np.uint8)
    before = _live(eng)
    g = eng.Genome()
    for _, off, nbytes, width, last in ingest.plain_fasta_layout(text):
        g.add_fasta_record(arr, off, nbytes, width, last)
    g.commit()
    assert len(g.fetch_token(0)) == 20004
    g.release_tokens()
    g.free()
    assert _live(eng) == before


@pytest.mark.gpu
def test_error_returns_give_back_every_block(eng):
    from cropsr_b200 import _native as N
    from cropsr_b200.engine import lib
    tokens = _tokens()
    g = _genome(eng, tokens)
    r = g.scan(20)
    index = eng.OffTargetIndex([g], loci=True)
    try:
        counts = index.count_candidates(r, "+", 3)
        valid = np.nonzero(counts[:, 0] != index.NO_COUNT)[0]
        busy = np.ascontiguousarray(valid[counts[valid].astype(np.int64).sum(axis=1) > 0][:4], dtype=np.uint32)
        assert len(busy) == 4
        first = np.zeros(len(busy) + 1, dtype=np.uint64)
        first[1:] = np.cumsum(counts[busy].astype(np.uint64).sum(axis=1))
        first[2:] -= np.uint64(1)                  # a slice one short: CRP_ERR_STATE after the join
        out = np.empty(int(first[-1]) + 1, dtype=np.uint32)

        def short():
            N.check(lib.crp_offtarget_list_candidates(index._h, r._h, b"+", 3, len(busy), busy.ctypes.data,
                                                      first.ctypes.data, out.ctypes.data))
        _gives_back(eng, short, code=-3)
        # a row without a protospacer: CRP_ERR_ARG after k_ot_gather
        invalid = np.nonzero(counts[:, 0] == index.NO_COUNT)[0]
        assert len(invalid)
        _gives_back(eng, lambda: index.list_candidates(r, "+", 3, rows=invalid[:1], counts=np.zeros_like(counts)),
                    code=-2)
        # more runs than the capacity: CRP_ERR_RANGE after the run kernel
        start, length, n = np.empty(1, np.uint32), np.empty(1, np.uint32), C.c_uint64(0)

        def runs():
            N.check(lib.crp_genome_other_runs(g._h, 0, 1, 1, start.ctypes.data, length.ctypes.data, C.byref(n)))
        _gives_back(eng, runs, code=-5)
        assert n.value > 1
    finally:
        index.free()
        r.free()
        g.free()
    # an arena too small for the rows: CRP_ERR_RANGE after every group was scanned
    descs = (N.SegmentDesc * len(tokens))()
    keep = [np.frombuffer(t.encode(), np.uint8) for t in tokens]
    for k, a in enumerate(keep):
        descs[k] = N.SegmentDesc(k, a.ctypes.data, len(a), 0, len(a))
    arena = eng.Arena(16, True)
    n_plus, n_minus, ms = np.zeros(len(tokens), np.uint64), np.zeros(len(tokens), np.uint64), C.c_float(0)
    p, m = arena.arrays["+"], arena.arrays["-"]

    def small():
        N.check(lib.crp_scan_segments(len(tokens), descs, 20, N.CRP_SCAN_DEFAULT, arena.capacity, p["pos"].ctypes.data,
                                      p["packed"].ctypes.data, p["x"].ctypes.data, m["pos"].ctypes.data,
                                      m["packed"].ctypes.data, m["x"].ctypes.data, n_plus.ctypes.data,
                                      n_minus.ctypes.data, C.byref(ms)))
    _gives_back(eng, small, code=-5)
    assert n_plus.sum() > 16
    arena.free()
    # a device FASTA record that is not plain: CRP_ERR_FORMAT from the commit, then the genome's free
    seq = bytearray(b"\n".join([b"ACGT" * 15] * 40) + b"\n")
    seq[130] = ord(" ")
    arr = np.frombuffer(bytes(seq), np.uint8)

    def not_plain():
        g2 = eng.Genome()
        try:
            g2.add_fasta_record(arr, 0, len(arr), 60, True)
            g2.commit()
        finally:
            g2.free()
    _gives_back(eng, not_plain, code=-6)
