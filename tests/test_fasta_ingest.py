"""The device FASTA ingest (crp_genome_add_fasta_record + k_fasta_strip) against the text ingest.

The reference is ingest.fasta_text_to_tokens (keys and token strings) and, where rows are compared,
pipeline.scan_tokens on those tokens.  k_fasta_strip hands every thread 16 token bytes; a record
must be refused (CRP_ERR_FORMAT, -6) whenever a line end is not where the fixed width puts it --
the line end just before a group's first base included -- so that the pipeline falls back to the
literal host ingest instead of scanning a token the reference would not build."""
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_BASES = np.frombuffer(b"ACGTACGTACGTacgtNn", dtype=np.uint8)
_OTHER = np.array([c for c in range(0x21, 0x7F) if c not in b"'\"\\>"], dtype=np.uint8)   # printable, plain


def _bases(rng, n):
    """n bytes a plain record may hold: mostly bases, one in 16 any other printable plain byte"""
    s = rng.choice(_BASES, n)
    odd = rng.random(n) < 1 / 16
    s[odd] = rng.choice(_OTHER, int(odd.sum()))
    return s


def _lines(seq, w, final_nl):
    """bases -> sequence lines of width w (uint8), the last line partial or full, with or without its '\\n'"""
    n = len(seq)
    k = -(-n // w)
    buf = np.full((k, w + 1), ord("\n"), dtype=np.uint8)
    pad = np.zeros(k * w, dtype=np.uint8)
    pad[:n] = seq
    buf[:, :w] = pad.reshape(k, w)
    r = n - (k - 1) * w
    if final_nl and r < w:
        buf[k - 1, r] = ord("\n")
    return buf.reshape(-1)[:n + k - 1 + int(final_nl)]


def _fasta(records, final_nl=True):
    """records: [(bases uint8, width)] -> file bytes (every record but the last ends in '\\n')"""
    parts = []
    for i, (seq, w) in enumerate(records):
        parts.append(b">chr%d\n" % (i + 1) + _lines(seq, w, final_nl or i + 1 < len(records)).tobytes())
    return b"".join(parts)


def _base_slot(i, w):
    """byte offset of base i in a record's sequence lines"""
    return i + i // w


def _line_end_slot(b, w):
    """byte offset of the line end just before base b (b a positive multiple of w)"""
    return b + b // w - 1


def _group_edge_bases(w, first, count):
    """the first `count` bases b >= first that start a line (b % w == 0) and a 16-byte group of k_fasta_strip
    (token position b + 1 a multiple of 16, i.e. b % 16 == 15); odd widths only"""
    inv = pow(16, -1, w)
    it = -(-(first + 1) // 16)
    it += (inv - it) % w
    return [16 * (it + k * w) - 1 for k in range(count)]


def _device_tokens(data):
    """plain_fasta_layout + one genome handle: (keys, [token bytes]); CropsrError when refused"""
    from cropsr_b200 import engine, ingest
    layout = ingest.plain_fasta_layout(data)
    assert layout is not None
    arr = np.frombuffer(data, dtype=np.uint8)
    g = engine.Genome()
    try:
        for key, off, nbytes, width, last in layout:
            g.add_fasta_record(arr, off, nbytes, width, last)
        g.commit()
        return [rec[0] for rec in layout], [g.fetch_token(s).tobytes() for s in range(len(layout))]
    finally:
        g.free()


def _reference(data):
    from cropsr_b200 import ingest
    tokens = ingest.fasta_text_to_tokens(data.decode("ascii"))
    return list(tokens.keys()), [v.encode("ascii") for v in tokens.values()], tokens


# ---------------------------------------------------------------------------------------------- CPU
def test_fasta_strip_source_on_the_cpu(tmp_path):
    """tests/fasta_strip_emu.cu runs k_fasta_strip's group function and the host's base count -- the SAME
    source, __host__ __device__ -- on every item of records laid out as commit_enqueue lays them, against a
    byte-by-byte reading: accepted <=> plain, accepted => token equal, at widths 1-130 and 4095-4097, every
    token length mod 16, every line end replaced or moved, bad bytes at group and record edges, and
    buffers of 1-300 records."""
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    exe = str(tmp_path / "fasta_strip_emu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "-o", exe,
                    os.path.join(ROOT, "tests", "fasta_strip_emu.cu")], check=True, capture_output=True, timeout=600)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def eng(built_lib):
    from cropsr_b200 import engine
    engine.init(0)
    return engine


CLEAN_WIDTHS = [1, 2, 3, 7, 15, 16, 17, 31, 33, 59, 60, 61, 63, 65, 79, 80, 81, 127, 129, 4097]
ROW_WIDTHS = {1, 17, 61, 80, 4097}


def _rows_equal(scan_result, ref_result, seg_a, seg_b):
    for strand in "+-":
        a, b = scan_result.fetch_segment(seg_a, strand), ref_result.fetch_segment(seg_b, strand)
        assert np.array_equal(a["pos"], b["pos"]) and np.array_equal(a["packed"], b["packed"]), (seg_a, strand)
        assert np.array_equal(a["x"], b["x"]), (seg_a, strand)


@pytest.mark.gpu
def test_device_ingest_equals_text_ingest_at_every_width(eng, tmp_path):
    """At each width: 16 records whose token lengths take every value mod 16 (last line full or partial), a
    one-line record, and the file with and without its final '\\n'.  fetch_token of every segment and the
    keys equal the text ingest; at a few widths the rows of both strands equal scan_tokens."""
    from cropsr_b200 import pipeline
    rng = np.random.default_rng(5)
    for w in CLEAN_WIDTHS:
        lines = 18 if w > 1000 else 40
        recs = [(_bases(rng, max(1, lines * w - d)), w) for d in range(16)]
        recs.append((_bases(rng, 3 * w + 5), 3 * w + 5))                # one line
        for final_nl in (True, False):
            data = _fasta(recs[::-1] if final_nl else recs, final_nl)
            keys, toks, tokens = _reference(data)
            assert len({len(t) % 16 for t in toks}) == 16
            got_keys, got = _device_tokens(data)
            assert got_keys == keys, w
            assert [i for i, (a, b) in enumerate(zip(got, toks)) if a != b] == [], (w, final_nl)
            if w in ROW_WIDTHS and final_nl:
                path = tmp_path / f"w{w}.fa"
                path.write_bytes(data)
                keys2, scan = pipeline.scan_fasta_file(str(path), 20)
                g2, r2, tb2 = pipeline.scan_tokens(tokens, 20)
                try:
                    assert keys2 == keys and scan.token_bytes == tb2 and len(scan.parts) == 1
                    for seg in range(len(keys)):
                        _rows_equal(scan.parts[0][1], r2, seg, seg)
                finally:
                    scan.free()
                    r2.free()
                    g2.free()


@pytest.mark.gpu
def test_device_ingest_refuses_every_misplaced_line_end(eng):
    """Commit only: in a record of 40 lines, each of the first 33 line ends (every residue mod 16 of the
    base after it, at odd widths) replaced by A, blank, tab or a quote, and the first and last base of the
    16-byte group holding the base after it replaced by a blank or '>': every one answers CRP_ERR_FORMAT."""
    from cropsr_b200 import engine
    from cropsr_b200._native import CropsrError
    rng = np.random.default_rng(6)
    missed, n = [], 0
    for w in (1, 3, 61, 63, 129, 60, 64):
        nb = 40 * w - w // 2
        clean = _lines(_bases(rng, nb), w, True)
        cases = []
        for j in range(1, 34):
            b = j * w                                          # the base after line end j
            for c in b"A \t'":
                cases.append((f"line end before base {b} -> {chr(c)!r}", _line_end_slot(b, w), c))
            g = (b + 1) // 16                                  # its 16-byte group: bases 16 g - 1 .. 16 g + 14
            for i in (max(16 * g - 1, 0), min(16 * g + 14, nb - 1)):
                for c in b" >":
                    cases.append((f"base {i} (group of base {b}) -> {chr(c)!r}", _base_slot(i, w), c))
        for what, slot, c in cases:
            arr = clean.copy()
            arr[slot] = c
            g = engine.Genome()
            n += 1
            try:
                g.add_fasta_record(arr, 0, len(arr), w, True)
                g.commit()
                missed.append((w, what))
            except CropsrError as e:
                assert e.code == -6, (w, what, e)
            finally:
                g.free()
    assert n > 1000
    assert missed == [], f"{len(missed)} of {n} defects accepted: {missed}"


def _repro(lines, w=61, at=10, byte=b"A"):
    """one record of `lines` lines of width w whose line end after line `at` (0-based) is replaced by `byte`:
    line at + 1 starts at base 61 * 11 = 671, the first base of the group at token position 672"""
    rng = np.random.default_rng(7)
    rows = [_bases(rng, w).tobytes() for _ in range(lines)]
    return b">chr1\n" + b"\n".join(rows[:at]) + b"\n" + rows[at] + byte + rows[at + 1] + b"\n" + b"\n".join(rows[at + 2:]) + b"\n"


@pytest.mark.gpu
def test_line_end_at_a_group_edge_falls_back_to_the_host_ingest(eng, tmp_path):
    """Two lines merged through the line end just before a group's first base: run_cas9 writes the CSV of the
    host ingest either way, because the device ingest refuses the file (scan_fasta_file -> None)."""
    from cropsr_b200 import pipeline
    from helpers import fixture_path
    data = _repro(2000)
    path = tmp_path / "merged.fa"
    path.write_bytes(data)
    outs = []
    for dev in (True, False):
        out = tmp_path / f"out{int(dev)}.csv"
        np.random.seed(3)
        pipeline.run_cas9(str(path), fixture_path("sample_genome.gff"), str(out), 20, False, 1,
                          str(tmp_path / "time.txt"), out=lambda *a: None, device_ingest=dev)
        outs.append(out.read_bytes())
    assert outs[0].count(b"\n") > 1000
    assert outs[0] == outs[1]
    assert pipeline.scan_fasta_file(str(path), 20) is None


@pytest.mark.gpu
def test_grid_stride_passes(eng):
    """A record of more than three times the token bytes one launch of k_fasta_strip covers (sm_count * 16
    CTAs of 256 threads, 16 bytes each) at an odd width: its token equals the text ingest's.  The same
    record with a blank in the line end before a group's first base in the last pass is refused."""
    from cropsr_b200._native import CropsrError
    sm = int(eng.perf_report()["sm_count"])
    stride = sm * 16 * 256                                   # items of one pass
    w = 61
    n = 16 * (3 * stride + stride // 4)
    rng = np.random.default_rng(8)
    seq = _bases(rng, n)
    data = _fasta([(seq, w)])
    keys, toks, _ = _reference(data)
    assert len(toks[0]) > 3 * 16 * stride
    got_keys, got = _device_tokens(data)
    assert got_keys == keys and got[0] == toks[0]
    b = _group_edge_bases(w, 16 * 3 * stride, 1)[0]          # item (b + 1) / 16 lies in the fourth pass
    assert 3 * stride <= (b + 1) // 16 < -(-(n + 4) // 16) and b < n - w
    arr = bytearray(data)
    arr[len(b">chr1\n") + _line_end_slot(b, w)] = ord(" ")
    with pytest.raises(CropsrError) as e:
        _device_tokens(bytes(arr))
    assert e.value.code == -6


@pytest.mark.gpu
def test_device_ingest_over_several_handles(eng, tmp_path):
    """scan_fasta_file with a small per-handle limit: eight records over four genome handles give the tokens
    of the text ingest (')]' on the last record only) and its rows; a misplaced line end in a record of the
    third handle sends the file to the host ingest."""
    from cropsr_b200 import pipeline
    rng = np.random.default_rng(9)
    widths = [61, 63, 33, 17, 61, 129, 15, 81]
    recs = [(_bases(rng, 3000 + 37 * i), w) for i, w in enumerate(widths)]
    data = _fasta(recs)
    keys, toks, tokens = _reference(data)
    path = tmp_path / "several.fa"
    path.write_bytes(data)
    got_keys, scan = pipeline.scan_fasta_file(str(path), 20, limit=7000)
    g2, r2, _ = pipeline.scan_tokens(tokens, 20)
    try:
        assert len(scan.parts) == 4 and got_keys == keys
        assert scan.token_bytes == toks
        assert [t.endswith(b"')]") for t in scan.token_bytes] == [False] * 7 + [True]
        for k in range(len(keys)):
            tp, xp, tm, xm = scan.token_rows(k)
            p, m = r2.fetch_segment(k, "+"), r2.fetch_segment(k, "-")
            assert np.array_equal(tp, p["pos"]) and np.array_equal(xp, p["x"]), k
            assert np.array_equal(tm, m["pos"]) and np.array_equal(xm, m["x"]), k
    finally:
        scan.free()
        r2.free()
        g2.free()
    # record 6 (width 129) sits in the third handle; blank the line end before one of its group-edge bases
    off = data.index(b">chr6\n") + len(b">chr6\n")
    b = _group_edge_bases(129, 0, 1)[0]
    assert b < 3000 - 129
    bad = bytearray(data)
    bad[off + _line_end_slot(b, 129)] = ord(" ")
    path.write_bytes(bytes(bad))
    assert pipeline.scan_fasta_file(str(path), 20, limit=7000) is None


@pytest.mark.gpu
def test_mixed_segments_and_error_codes(eng):
    """One handle with add_token and add_fasta_record segments interleaved: every segment's rows equal an
    all-add_token handle, and fetch_token gives the FASTA segments' tokens.  Then the documented codes:
    fetch_token of an add_token segment, after release_tokens (CRP_ERR_STATE) or into a short buffer
    (CRP_ERR_RANGE); add_fasta_record of a whole number of width + 1 byte lines, of zero bytes (CRP_ERR_FORMAT)
    or after the commit (CRP_ERR_STATE); a token at the 31-bit limit (CRP_ERR_RANGE, before any device work)."""
    from cropsr_b200 import engine, ingest, pipeline
    from cropsr_b200._native import CropsrError, lib
    rng = np.random.default_rng(10)
    recs = [(_bases(rng, n), w) for n, w in ((4000, 61), (2500, 80), (1, 7), (3333, 33), (5000, 63))]
    data = _fasta(recs)
    keys, toks, tokens = _reference(data)
    layout = ingest.plain_fasta_layout(data)
    arr = np.frombuffer(data, dtype=np.uint8)
    from_tokens = (1, 4)
    g = engine.Genome()
    g2, r2, _ = pipeline.scan_tokens(tokens, 20)
    res = None

    def code(fn, *a):
        with pytest.raises(CropsrError) as e:
            fn(*a)
        return e.value.code

    try:
        for s, (key, off, nbytes, width, last) in enumerate(layout):
            if s in from_tokens:
                g.add_token(toks[s])
            else:
                g.add_fasta_record(arr, off, nbytes, width, last)
        g.commit()
        res = g.scan(20)
        for s in range(len(layout)):
            _rows_equal(res, r2, s, s)
            if s not in from_tokens:
                assert g.fetch_token(s).tobytes() == toks[s], s
        assert code(g.fetch_token, 1) == -3
        short = np.empty(len(toks[0]), dtype=np.uint8)
        assert lib.crp_genome_fetch_token(g._h, 0, short.ctypes.data, len(toks[0]) - 1) == -5
        assert lib.crp_genome_fetch_token(g._h, 0, short.ctypes.data, len(toks[0])) == 0
        assert short.tobytes() == toks[0]
        assert code(g.add_fasta_record, arr, layout[0][1], layout[0][2], layout[0][3], False) == -3
        g.release_tokens()
        assert code(g.fetch_token, 0) == -3
    finally:
        for h in (res, g, r2, g2):
            if h is not None:
                h.free()
    g = engine.Genome()
    try:
        lines = np.frombuffer(b"ACGT\nACGT\n\n", dtype=np.uint8)                  # two 5-byte lines, then '\n'
        assert code(g.add_fasta_record, lines, 0, len(lines), 4, True) == -6
        assert code(g.add_fasta_record, lines, 0, 0, 4, True) == -6
        assert code(g.add_fasta_record, lines, 0, 9, 0, True) == -6
        # one line of 2^31 - 2^15 - 4 bases is a token of 2^31 - 2^15 positions: one too many.  Only the last
        # byte is read, so the untouched pages of np.zeros are never materialised.
        limit = (1 << 31) - (1 << 15) - 4
        big = np.zeros(limit, dtype=np.uint8)
        launches = eng.launch_count()
        assert code(g.add_fasta_record, big, 0, limit, (1 << 31) - 1, True) == -5
        assert g.add_fasta_record(big, 0, limit - 1, (1 << 31) - 1, True) == 0
        assert eng.launch_count() == launches
    finally:
        g.free()
