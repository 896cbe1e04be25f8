"""End-to-end --cas9 run: ingest -> GPU scan+score -> reference-order emission.

Mirror of /root/reference/CROPSR.py:333-486 main().  Differences that are
deliberate and documented in DESIGN.md: the whole genome is scanned on the GPU
in one launch sequence before the per-token emission loop starts, and the
reference's 5-second sleep per token (CROPSR.py:478) is not performed.
"""
import time

import numpy as np

from . import emit, engine, ingest


# A genome handle addresses its positions and its candidate rows with 32 bits (crp_genome_commit
# answers CRP_ERR_RANGE beyond that); a run keeps every handle well below, so that a 10 Gbp genome
# -- which the reference handles given enough RAM -- is simply several handles scanned in turn.
MAX_POSITIONS_PER_GENOME = 1 << 31


class HostRescorer:
    """x of a few candidates re-summed in another BLAS class from the HOST copy of the tokens:
    the 30 scored bytes of the window (CROPSR.py:458, long.replace('U','T').upper()) go through
    crp_rs1_preactivation.  Same values as crp_rescore (which reads the packed records of one
    genome handle); used where the rows of a slice span several handles or several GPUs."""

    def __init__(self, token_bytes):
        self.token_bytes = token_bytes

    def rescore(self, tok_index, t, strand, cls):
        rows = np.zeros((len(t), 30), dtype=np.uint8)
        for i, (k, ti, st) in enumerate(zip(np.asarray(tok_index).tolist(), np.asarray(t).tolist(),
                                            np.asarray(strand).tolist())):
            long_ = emit.guide_strings(self.token_bytes[k], int(ti), st in (b"-", "-"), 20)[1]
            b = long_.replace("U", "T").upper().encode("ascii")
            rows[i, :len(b)] = np.frombuffer(b, dtype=np.uint8)[:30]
        return engine.rs1_preactivation(rows, cls)


class ScanOutput:
    """Everything the emission loop needs from a finished scan, whichever way it ran (one
    handle, several handles on one GPU, several GPUs): per-token candidate rows in reference
    order, the counts, a rescorer, timings."""

    def __init__(self, token_bytes, parts, guide_len):
        self.token_bytes = token_bytes
        self.parts = parts                      # [(genome, result, first token, n tokens)]
        self.guide_len = guide_len
        n = len(token_bytes)
        self.seg_plus = np.zeros(n, dtype=np.uint64)
        self.seg_minus = np.zeros(n, dtype=np.uint64)
        self._rows = [None] * len(parts)
        for g, r, first, cnt in parts:
            self.seg_plus[first:first + cnt] = r.seg_plus
            self.seg_minus[first:first + cnt] = r.seg_minus
        self._part_of = np.zeros(n, dtype=np.int64)
        for i, (_, _, first, cnt) in enumerate(parts):
            self._part_of[first:first + cnt] = i
        self._host = HostRescorer(token_bytes)

    def locate(self, k):
        """(genome, result, segment index) of token k"""
        g, r, first, _ = self.parts[self._part_of[k]]
        return g, r, k - first

    def token_rows(self, k):
        """(t_plus, x_plus, t_minus, x_minus) of token k; the strands of a handle come over in one
        device-to-host copy each the first time one of its tokens is asked for."""
        i = int(self._part_of[k])
        g, r, first, _ = self.parts[i]
        if self._rows[i] is None:
            want = ("pos", "x")
            self._rows[i] = (r.fetch("+", want=want), r.fetch("-", want=want))
        plus, minus = self._rows[i]
        s = k - first
        a, b = int(r.off_plus[s]), int(r.off_plus[s + 1])
        c, d = int(r.off_minus[s]), int(r.off_minus[s + 1])
        sl = lambda col, lo, hi: None if col is None else col[lo:hi]
        return plus["pos"][a:b], sl(plus["x"], a, b), minus["pos"][c:d], sl(minus["x"], c, d)

    def rescore(self, tok_index, t, strand, cls):
        if len(self.parts) == 1:                # one handle: token index == segment index
            return self.parts[0][0].rescore(tok_index, t, strand, cls)
        return self._host.rescore(tok_index, t, strand, cls)

    def scan_ms(self):
        return float(sum(r.scan_ms() for _, r, _, _ in self.parts))

    def timing(self):
        t = {"h2d_ms": 0.0, "pack_ms": 0.0}
        for g, _, _, _ in self.parts:
            for k, v in g.timing().items():
                t[k] += v
        return t

    def free(self):
        for g, r, _, _ in self.parts:
            r.free()
            g.free()
        self.parts = []
        self._rows = []


def _groups(lengths, limit=None):
    """consecutive runs of tokens whose summed length stays below the per-handle limit"""
    limit = MAX_POSITIONS_PER_GENOME if limit is None else limit
    out, first, acc = [], 0, 0
    for k, n in enumerate(lengths):
        if k > first and acc + n > limit:
            out.append((first, k - first))
            first, acc = k, 0
        acc += n
    out.append((first, len(lengths) - first))
    return [g for g in out if g[1] > 0] or [(0, 0)]


def scan_tokens(tokens, guide_len=20, flags=0):
    """Pack every token of the ingest dict into HBM and scan it.
    Returns (genome, result, token_bytes) for callers that want the raw handles of a
    single-handle scan (tests, smoke); run_cas9 goes through scan_token_bytes."""
    genome = engine.Genome()
    token_bytes = []
    for value in tokens.values():
        b = value.encode("ascii") if isinstance(value, str) else bytes(value)
        token_bytes.append(b)
        genome.add_token(b)
    genome.commit()
    result = genome.scan(guide_len, flags)
    return genome, result, token_bytes


def scan_token_bytes(token_bytes, guide_len=20, flags=0, limit=None):
    """-> ScanOutput; tokens are spread over as many genome handles as the 32-bit limits ask for."""
    parts = []
    for first, cnt in _groups([len(b) for b in token_bytes], limit):
        genome = engine.Genome()
        for b in token_bytes[first:first + cnt]:
            genome.add_token(b)
        genome.commit()
        parts.append((genome, genome.scan(guide_len, flags), first, cnt))
    return ScanOutput(token_bytes, parts, guide_len)


def scan_fasta_file(fasta, guide_len=20, flags=0, limit=None):
    """Device-side ingest of a plain multi-line FASTA file: the file's bytes go to the GPU as they
    are, k_fasta_strip builds the tokens there, and the host gets them back for row formatting.
    Returns (keys, ScanOutput), or None when the file needs the literal host
    ingest (clean path, blanks in headers, duplicate names, ragged lines, ...)."""
    from ._native import CropsrError
    with open(fasta, "rb") as f:
        data = f.read()
    layout = ingest.plain_fasta_layout(data)
    if layout is None:
        return None
    arr = np.frombuffer(data, dtype=np.uint8)
    parts, token_bytes = [], []
    try:
        for first, cnt in _groups([rec[2] for rec in layout], limit):
            genome = engine.Genome()
            parts.append((genome, None, first, cnt))
            for key, off, nbytes, width, last in layout[first:first + cnt]:
                genome.add_fasta_record(arr, off, nbytes, width, last)
            genome.commit()
            parts[-1] = (genome, genome.scan(guide_len, flags), first, cnt)
            token_bytes += [genome.fetch_token(seg).tobytes() for seg in range(cnt)]
            genome.release_tokens()
    except CropsrError as e:
        for g, r, _, _ in parts:
            if r is not None:
                r.free()
            g.free()
        if e.code == -6:            # CRP_ERR_FORMAT: not plain after all
            return None
        raise
    return [rec[0] for rec in layout], ScanOutput(token_bytes, parts, guide_len)


def write_side_output(path, tokens, scan, gff_frame, flank, formatted_path, annotation_info=None):
    """Opt-in table of the per-candidate side outputs (one row per unique candidate, reference
    order).  NOT part of the reference's CSV: GC, poly-T / homopolymer flags, cut site, the
    +-L flank window, the GFF feature under the cut site (device kernels k_extras / k_annotate;
    semantics in oracle/extras_oracle.py) and the prmrdsgn2-style primer enumeration on the flank
    (k_primers, cropsr_b200/primers.py: primers passing the GC / Tm filter on either side, Tm-compatible
    pairs, the first pair; empty where the flank is shorter than e + l = 130 bases)."""
    import csv
    import pandas as pd
    from . import annotate, primers
    ivs = annotate.intervals_for_tokens(gff_frame, list(tokens.keys()), formatted_path)
    info = annotate.read_annotation_info(annotation_info) if annotation_info else {}    # -p: Phytozome annotation_info.txt
    columns = ["chromosome", "strand", "pam_pos", "cutsite", "gc", "poly_t", "homopolymer", "low_gc",
               "unscored_base", "longest_run", "flank_start", "flank_end", "feature_type", "feature_attributes",
               "fwd_primers", "rev_primers", "primer_pairs", "first_pair", "annotation_info"]
    with open(path, "w", newline="") as f:
        csv.writer(f, delimiter="\t").writerow(columns)
    # GFF rows are looked up per DISTINCT feature, then spread over the candidates: whole columns,
    # no Python work per candidate.  The device is asked once per strand of a genome handle -- every
    # segment's extras / annotation / primer windows in one call each -- so 20,000 scaffolds cost a
    # handful of host round trips; the rows are then put back into the reference's order
    # (token by token, '+' then '-').
    gff_feature = gff_frame["feature"].to_numpy(dtype=object)
    gff_attr = gff_frame["attributes"].to_numpy(dtype=object)
    keys = list(tokens.keys())
    for genome, result, first, cnt in scan.parts:
        part_ivs = ivs[first:first + cnt]
        iv_off = np.concatenate(([0], np.cumsum([len(iv["start"]) for iv in part_ivs]))).astype(np.uint64)
        iv_start = np.concatenate([iv["start"] for iv in part_ivs]) if cnt else np.empty(0, np.uint32)
        iv_end = np.concatenate([iv["end"] for iv in part_ivs]) if cnt else np.empty(0, np.uint32)
        iv_row = np.concatenate([np.asarray(iv["row"], dtype=np.int64) for iv in part_ivs]) if cnt else np.empty(0, np.int64)
        cols = {}
        for strand, seg_cnt in (("+", result.seg_plus), ("-", result.seg_minus)):
            seg_cnt = seg_cnt.astype(np.int64)
            n = int(seg_cnt.sum())
            seg_of = np.repeat(np.arange(cnt, dtype=np.int64), seg_cnt)
            pos = result.fetch(strand, want=("pos",))["pos"]
            ex = result.extras_strand(strand, flank)
            feat = result.annotate_strand(strand, iv_off, iv_start, iv_end)
            pr = primers.design_windows(genome, seg_of.astype(np.uint32), ex["flank_lo"], ex["flank_hi"])
            if n and len(iv_row):
                at = np.minimum(np.maximum(feat, 0) + iv_off[seg_of].astype(np.int64), len(iv_row) - 1)
                rows = np.where(feat >= 0, iv_row[at], -1)
            else:
                rows = np.full(n, -1, dtype=np.int64)
            ft = np.full(n, "", dtype=object)
            fa = np.full(n, "", dtype=object)
            ai = np.full(n, "", dtype=object)
            hit = rows >= 0
            if hit.any():
                uniq, inv = np.unique(rows[hit], return_inverse=True)
                ft[hit] = gff_feature[uniq][inv]
                fa[hit] = gff_attr[uniq][inv]
                ai[hit] = np.array([annotate.lookup_annotation_info(info, a) for a in gff_attr[uniq]], dtype=object)[inv]
            fl = ex["flags"].astype(np.int64)
            ok = pr["status"] == 0
            firstp = pr["first"].astype(np.int64)
            has_pair = ok & (firstp[:, 0] != 0xFFFF) if n else np.zeros(0, bool)
            pair = np.full(n, "", dtype=object)
            if has_pair.any():
                pair[has_pair] = [f"{a}+{b}/{c}+{d}" for a, b, c, d in firstp[has_pair].tolist()]
            blank_unless_ok = lambda a: np.where(ok, a.astype(np.int64).astype(str).astype(object), "")
            chrom = np.array([k[1:] for k in keys[first:first + cnt]], dtype=object)[seg_of] if n else np.empty(0, object)
            cols[strand] = (seg_of, pd.DataFrame({
                "chromosome": chrom, "strand": strand, "pam_pos": pos.astype(np.int64), "cutsite": ex["cut"].astype(np.int64),
                "gc": ex["gc"].astype(np.int64), "poly_t": fl & 1, "homopolymer": (fl >> 1) & 1, "low_gc": (fl >> 2) & 1,
                "unscored_base": (fl >> 3) & 1, "longest_run": ex["run"].astype(np.int64),
                "flank_start": ex["flank_lo"].astype(np.int64), "flank_end": ex["flank_hi"].astype(np.int64),
                "feature_type": ft, "feature_attributes": fa, "fwd_primers": blank_unless_ok(pr["n_fwd"]),
                "rev_primers": blank_unless_ok(pr["n_rev"]), "primer_pairs": blank_unless_ok(pr["n_pairs"]),
                "first_pair": pair, "annotation_info": ai}, columns=columns))
        # reference order: per token its '+' rows, then its '-' rows -- a stable sort on (token, strand)
        frame = pd.concat([cols["+"][1], cols["-"][1]], ignore_index=True)
        order = np.argsort(np.concatenate((2 * cols["+"][0], 2 * cols["-"][0] + 1)), kind="stable")
        frame.iloc[order].to_csv(path, sep="\t", mode="a", header=False, index=False, lineterminator="\r\n")


def write_gap_table(path, tokens, scan, min_len=10):
    """Opt-in companion of the side output (SURVEY.md 8f.2): the gaps of the assembly -- runs of at least
    min_len bytes that are not ACGTacgt (N, IUPAC) -- one row per run, token coordinates, read off the packed
    records on the device (Genome.other_runs / k_other_runs).  Not part of the reference's output."""
    import csv
    with open(path, "w", newline="") as f:
        w = csv.writer(f, delimiter="\t")
        w.writerow(["chromosome", "start", "length"])
        for k, key in enumerate(tokens.keys()):
            genome, _, seg = scan.locate(k)
            start, length = genome.other_runs(seg, min_len)
            w.writerows((key[1:], int(a), int(b)) for a, b in zip(start.tolist(), length.tolist()))


_UPPER_DNA = np.frombuffer(b"ATCG", dtype=np.uint8)
_COMPLEMENT = np.arange(256, dtype=np.uint8)
_COMPLEMENT[list(b"ATCG")] = list(b"TAGC")


def _protospacers(scan, first, seg, pos, strand):
    """The protospacers of candidates with one, read from the host tokens: uint8 [n, 20], upper case, in the
    orientation followed by the PAM -- '+' tok[t-20:t], '-' the reverse complement of tok[t+3:t+23].  seg: each
    candidate's token within the part that starts at token `first`; pos: its pam_pos t."""
    rows = []
    for s, t in zip(seg.tolist(), pos.tolist()):
        tok = scan.token_bytes[first + s]
        rows.append(tok[t - 20:t] if strand == "+" else tok[t + 3:t + 23][::-1])
    b = np.frombuffer(b"".join(rows), dtype=np.uint8).reshape(-1, 20) & 0xDF
    return _COMPLEMENT[b] if strand == "-" else b


def write_offtarget_table(path, tokens, scan, k=3, index=None, counts=None, extra=()):
    """Opt-in off-target table (not part of the reference's output): one row per unique candidate in
    reference order (token by token, '+' then '-', ascending t) with its protospacer as upper-case DNA
    in the orientation followed by the PAM, and the numbers of OTHER NGG sites of the whole genome at
    exactly 0 .. k mismatches (k_ot_* kernels; semantics in oracle/offtarget_oracle.py).  Protospacer
    and counts are blank where the candidate has none (cut off by the token end, or a byte outside
    ACGTacgt).  One index is built from every genome handle of the scan before anything is counted:
    handles split at MAX_POSITIONS_PER_GENOME see each other's sites.  index: such an index, built by the
    caller (and not freed here); counts: offtarget_counts(index, scan, k), computed here when not given.
    extra: (pam, index, counts or None) of further PAM patterns (--offtarget-pams), each adding the columns
    {pam}_mm0 .. {pam}_mmk of the sites of its index after mm0 .. mmk, in the order given."""
    groups = [("", index, counts)] + [(f"{pam}_", ix, c) for pam, ix, c in extra]

    def values(index, part, result, strand):
        out = {}
        for prefix, ix, cnt in groups:
            ix = index if ix is None else ix
            c = ix.count_candidates(result, strand, k) if cnt is None else cnt[(part, strand)]
            if not prefix:
                ok = c[:, 0] != index.NO_COUNT
            out.update({f"{prefix}mm{d}": c[:, d].astype(np.int64).astype(str).astype(object) for d in range(k + 1)})
        return ok, out
    _write_candidate_table(path, tokens, scan, [f"{prefix}mm{d}" for prefix, _, _ in groups for d in range(k + 1)],
                           values, index)


def write_offtarget_scores(path, tokens, scan, k=3, index=None, extra=()):
    """Opt-in off-target score table (not part of the reference's output): the rows of write_offtarget_table, in
    its order, with mit_hit_sum, the sum of the MIT hit scores (Hsu et al. 2013, CRISPOR's calcHitScore) of the
    candidate's OTHER NGG sites within k mismatches (.6f), and mit_specificity, 100 / (100 + mit_hit_sum) * 100
    rounded to an integer (CRISPOR's calcMitGuideScore); both blank where the candidate has no protospacer
    (k_ot_join<OtScore>; semantics in oracle/offtarget_score_oracle.py).  CRISPOR also sums 4-mismatch sites, so its
    numbers differ.  index: an index over the scan's genome handles, built by the caller (and not freed here), else
    built here.  extra: (pam, index) of further PAM patterns (--offtarget-pams): one {pam}_mit_hit_sum column each, in
    the order given, then all_mit_specificity from the exact sum of the integer sums of all patterns."""
    weights = engine.mit_weights()

    def hit_sum(sums, ok):
        hit = np.zeros(len(sums), dtype=object)
        hit[ok] = np.char.mod("%.6f", sums[ok].astype(np.float64) / engine.SCORE_ONE).astype(object)
        return hit

    def values(index, part, result, strand):
        sums = index.score_candidates(result, strand, k, weights)
        ok = sums != np.uint64(index.NO_SCORE)
        out = {"mit_hit_sum": hit_sum(sums, ok), "mit_specificity": engine.mit_specificity(sums).astype(str).astype(object)}
        if extra:
            total = sums.copy()
            for pam, ix in extra:
                s = ix.score_candidates(result, strand, k, weights)
                out[f"{pam}_mit_hit_sum"] = hit_sum(s, ok)
                total[ok] += s[ok]
            out["all_mit_specificity"] = engine.mit_specificity(total).astype(str).astype(object)
        return ok, out
    columns = ["mit_hit_sum", "mit_specificity"]
    if extra:
        columns += [f"{pam}_mit_hit_sum" for pam, _ in extra] + ["all_mit_specificity"]
    _write_candidate_table(path, tokens, scan, columns, values, index)


def _write_candidate_table(path, tokens, scan, value_columns, values, index=None):
    """The per-candidate off-target tables: chromosome strand pam_pos protospacer, then value_columns from
    values(index, part, result, strand) -> (ok, {column: object array}) per strand stream; protospacer and values
    blank where not ok.  index None: one is built over every genome handle of the scan and freed here."""
    import csv
    import pandas as pd
    keys = list(tokens.keys())
    columns = ["chromosome", "strand", "pam_pos", "protospacer"] + value_columns
    with open(path, "w", newline="") as f:
        csv.writer(f, delimiter="\t").writerow(columns)
    own_index = index is None
    if own_index:
        index = engine.OffTargetIndex([g for g, _, _, _ in scan.parts])
    try:
        for part, (genome, result, first, cnt) in enumerate(scan.parts):
            cols = {}
            for strand, seg_cnt in (("+", result.seg_plus), ("-", result.seg_minus)):
                seg_of = np.repeat(np.arange(cnt, dtype=np.int64), seg_cnt.astype(np.int64))
                n = len(seg_of)
                pos = result.fetch(strand, want=("pos",))["pos"]
                ok, vals = values(index, part, result, strand)
                if not n:
                    ok = np.zeros(0, bool)
                proto = np.full(n, "", dtype=object)
                if ok.any():
                    b = _protospacers(scan, first, seg_of[ok], pos[ok], strand)
                    proto[ok] = b.view("S20").ravel().astype("U20").astype(object)
                frame = {"chromosome": np.array([key[1:] for key in keys[first:first + cnt]], dtype=object)[seg_of]
                         if n else np.empty(0, object),
                         "strand": strand, "pam_pos": pos.astype(np.int64), "protospacer": proto}
                for c in value_columns:
                    frame[c] = np.where(ok, vals[c], "") if n else np.empty(0, object)
                cols[strand] = (seg_of, pd.DataFrame(frame, columns=columns))
            frame = pd.concat([cols["+"][1], cols["-"][1]], ignore_index=True)
            order = np.argsort(np.concatenate((2 * cols["+"][0], 2 * cols["-"][0] + 1)), kind="stable")
            frame.iloc[order].to_csv(path, sep="\t", mode="a", header=False, index=False, lineterminator="\r\n")
    finally:
        if own_index:
            index.free()


def offtarget_counts(index, scan, k=3):
    """{(part, strand): index.count_candidates} of every genome handle of the scan: both off-target tables
    from one count per strand"""
    return {(part, strand): index.count_candidates(result, strand, k)
            for part, (_, result, _, _) in enumerate(scan.parts) for strand in "+-"}


def write_offtarget_sites(path, tokens, scan, k=3, max_sites=1000, index=None, counts=None, extra=()):
    """Opt-in off-target sites table (not part of the reference's output): one row per (candidate, other NGG
    site of the genome within k mismatches), candidates in the order of write_offtarget_table, and within a
    candidate by mismatches, then the site's token (file order), site_pam_pos, '+' before '-'.  site_protospacer
    is the site's 20 bases in the orientation followed by NGG, upper case, with the bases that differ from the
    candidate's protospacer in lower case (semantics in oracle/offtarget_sites_oracle.py).  A candidate with no
    other site, or with more than max_sites, writes no rows: its counts are in the --offtargets table.
    index: an index with loci over the scan's genome handles in scan.parts order, built by the caller (and not
    freed here); counts: offtarget_counts(index, scan, k).  extra: (pam, index with loci, counts or None) of further PAM
    patterns (--offtarget-pams), disjoint from NGG and from each other: their sites join the listing, a last column
    site_pam names the pattern of each row's site, and max_sites caps a candidate's total over all patterns.  Returns
    (pairs written, candidates left out by the cap)."""
    import csv
    import pandas as pd
    keys = list(tokens.keys())
    names = np.array([key[1:] for key in keys], dtype=object)
    columns = ["chromosome", "strand", "pam_pos", "protospacer", "site_chromosome", "site_strand", "site_pam_pos",
               "site_protospacer", "mismatches"] + (["site_pam"] if extra else [])
    with open(path, "w", newline="") as f:
        csv.writer(f, delimiter="\t").writerow(columns)
    own_index = index is None
    if own_index:
        index = engine.OffTargetIndex([g for g, _, _, _ in scan.parts], loci=True)
    pairs = capped = 0
    try:
        part_first = np.array([first for _, _, first, _ in scan.parts], dtype=np.int64)
        groups = []                                     # (pam, index, counts, site keys, site token, t, strand)
        for pam, ix, cnt in [("NGG", index, counts)] + list(extra):
            site_keys = ix.sites()
            s_gen, s_seg, s_t, s_strand = ix.site_loci()
            s_tok = part_first[s_gen.astype(np.int64)] + s_seg.astype(np.int64) if len(site_keys) else np.zeros(0, np.int64)
            groups.append((pam, ix, cnt, site_keys, s_tok, s_t.astype(np.int64), s_strand.astype(np.int64)))
        for part, (genome, result, first, cnt) in enumerate(scan.parts):
            chunks = []
            for si, (strand, seg_cnt) in enumerate((("+", result.seg_plus), ("-", result.seg_minus))):
                seg_of = np.repeat(np.arange(cnt, dtype=np.int64), seg_cnt.astype(np.int64))
                if not len(seg_of):
                    continue
                cs = [ix.count_candidates(result, strand, k) if c is None else c[(part, strand)]
                      for _, ix, c, *_ in groups]
                ok = cs[0][:, 0] != index.NO_COUNT
                total = np.where(ok, sum(c[:, :k + 1].astype(np.int64).sum(axis=1) for c in cs), 0)
                capped += int((total > max_sites).sum())
                rows = np.nonzero((total > 0) & (total <= max_sites))[0]
                if not len(rows):
                    continue
                pos = result.fetch(strand, want=("pos",))["pos"].astype(np.int64)
                for (pam, ix, _, site_keys, s_tok, s_t, s_strand), c in zip(groups, cs):
                    lrows, lfirst, sites = ix.list_candidates(result, strand, k, rows=rows, counts=c)
                    lrows = lrows.astype(np.int64)
                    cb = _protospacers(scan, first, seg_of[lrows], pos[lrows], strand)
                    per = np.diff(lfirst).astype(np.int64)
                    cand = np.repeat(np.arange(len(lrows)), per)
                    sk = site_keys[sites]
                    sb = _UPPER_DNA[((sk[:, None] >> (2 * np.arange(20, dtype=np.uint64))) & np.uint64(3)).astype(np.intp)]
                    differ = sb != cb[cand]
                    sb = sb | (differ.astype(np.uint8) << 5)              # lower case where the bases differ
                    mm = differ.sum(axis=1)
                    row = lrows[cand]
                    site = sites.astype(np.int64)
                    chunks.append((seg_of[row], np.full(len(row), si), row, mm, s_tok[site], s_t[site], s_strand[site],
                                   pos, cb[cand], sb, strand, pam))
            if not chunks:
                continue
            frames, sort_keys = [], []
            for seg, sidx, row, mm, tok_i, site_t, site_s, pos, cb, sb, strand, pam in chunks:
                frame = {
                    "chromosome": names[first + seg], "strand": strand, "pam_pos": pos[row],
                    "protospacer": cb.view("S20").ravel().astype("U20").astype(object),
                    "site_chromosome": names[tok_i], "site_strand": np.array(["+", "-"], dtype=object)[site_s],
                    "site_pam_pos": site_t, "site_protospacer": sb.view("S20").ravel().astype("U20").astype(object),
                    "mismatches": mm}
                if extra:
                    frame["site_pam"] = pam
                frames.append(pd.DataFrame(frame, columns=columns))
                sort_keys.append(np.stack((seg, sidx, row, mm, tok_i, site_t, site_s)))
            frame = pd.concat(frames, ignore_index=True)
            key = np.concatenate(sort_keys, axis=1)
            order = np.lexsort(key[::-1])
            frame.iloc[order].to_csv(path, sep="\t", mode="a", header=False, index=False, lineterminator="\r\n")
            pairs += len(frame)
    finally:
        if own_index:
            index.free()
    return pairs, capped


def check_offtarget_args(guide_len, devices, max_mismatches, max_sites=None, pams=()):
    """The off-target tables' limits, checked before any device work: ValueError with the reason.
    max_sites: the cap of the sites table (write_offtarget_sites), at least 1.  pams: PAM patterns whose sites are
    counted besides NGG (--offtarget-pams): each a pattern of engine.parse_pam, none of them overlapping NGG or
    another (a base triple matches at most one pattern, so no site is found twice).  Returns them upper case."""
    if int(guide_len) != 20:
        raise ValueError(f"off-target counts are defined for 20-base guides, not -l {guide_len}")
    if devices is not None and len(devices) > 1:
        raise ValueError("off-target counts run on one GPU: the index needs every site of the genome on one device; "
                         "run without --devices, or with one device")
    if int(max_mismatches) not in (0, 1, 2, 3):
        raise ValueError(f"--mismatches {max_mismatches}: 0 to 3 mismatches are supported")
    if max_sites is not None and int(max_sites) < 1:
        raise ValueError(f"--max-sites {max_sites}: at least 1")
    out = []
    for text in pams:
        try:
            pam = engine.parse_pam(text)
        except ValueError as e:
            raise ValueError(f"--offtarget-pams: {e}") from None
        if pam == "NGG":
            raise ValueError("--offtarget-pams: NGG sites are always counted; list the other patterns only")
        if engine.pams_overlap(pam, "NGG"):
            raise ValueError(f"--offtarget-pams {pam}: it overlaps NGG, whose sites are always counted; list the bases "
                             f"outside NGG instead (NAG instead of NRG)")
        for other in out:
            if other == pam:
                raise ValueError(f"--offtarget-pams: {pam} is listed twice")
            if engine.pams_overlap(pam, other):
                raise ValueError(f"--offtarget-pams: {other} and {pam} overlap; the patterns must be disjoint")
        out.append(pam)
    return out


def check_side_output_args(flank):
    """The side output's limit, checked before any device work: ValueError unless 0 <= flank < 2**32 (the flank
    window [cut - flank, cut + flank) is computed in 32-bit token coordinates)."""
    if not 0 <= int(flank) < 1 << 32:
        raise ValueError(f"-L {flank}: the flanking length must be 0 to 2**32 - 1")


def run_cas9(fasta, gff, output="data.csv", guide_len=20, verbose=False, blas_threads=1,
             time_path="time.txt", out=print, side_output=None, flank=200, device_ingest=True, annotation_info=None,
             chunk_rows=None, devices=None, handle_limit=None, offtargets=None, max_mismatches=3,
             offtarget_sites=None, max_sites=1000, offtarget_scores=None, offtarget_pams=()):
    """devices: CUDA ordinals; more than one shards the genome over one process per GPU
    (cropsr_b200/multi.py) and writes the same CSV.  handle_limit: positions per genome handle
    (tests shrink it to walk the several-handles path on small inputs).  offtargets: path of the opt-in
    off-target table (write_offtarget_table, guide length 20 on one GPU), written after the CSV with
    counts at 0 .. max_mismatches.  offtarget_sites: path of the opt-in off-target sites table
    (write_offtarget_sites: every other site within max_mismatches of every candidate with at most max_sites
    of them); with both tables one index serves both and every strand is counted once.  offtarget_scores: path of
    the opt-in off-target score table (write_offtarget_scores: MIT hit-score sum and specificity over the NGG sites
    within max_mismatches); one index, with loci only when the sites table needs them, serves every table.
    offtarget_pams: PAM patterns whose sites every off-target table also reads (NAG, NGA, ...: disjoint from NGG and
    from each other, check_offtarget_args), one index each after the NGG index; without them every table is as
    before."""
    pams = []
    if offtarget_pams and offtargets is None and offtarget_sites is None and offtarget_scores is None:
        raise ValueError("--offtarget-pams: no off-target table asked for (--offtargets, --offtarget-sites, "
                         "--offtarget-scores)")
    if offtargets is not None or offtarget_sites is not None or offtarget_scores is not None:
        pams = check_offtarget_args(guide_len, devices, max_mismatches, max_sites if offtarget_sites is not None else None,
                                    offtarget_pams)
    if side_output:
        check_side_output_args(flank)
    begin = time.time()
    timing = open(time_path, "w")                       # CROPSR.py:371
    multi_gpu = devices is not None and len(devices) > 1
    fast = scan_fasta_file(fasta, guide_len, limit=handle_limit) if device_ingest and not multi_gpu else None
    if fast is not None:                                # :374, on the device
        keys, scan = fast
        tokens = {k: b[:25].decode("ascii") for k, b in zip(keys, scan.token_bytes)}   # stdout only
        if verbose:
            out(f"Genome file {fasta} successfully imported")
            out("formatting genome")
            out(f"Genome file {fasta} successfully formatted")
            out("The genome was successfully converted to a dictionary")
    else:
        tokens = ingest.import_fasta_file(fasta, verbose)   # :374
    gff_frame = ingest.import_gff_file(gff, verbose)    # :375 (parsed, never used by the reference)
    if verbose:
        out("\n            Initiating PAM site detection.\n            \n"
            "            Please wait, this may take a while...\n            ")
    emit.write_header(output)                           # :402-405

    if fast is None:
        token_bytes = [v.encode("ascii") if isinstance(v, str) else bytes(v) for v in tokens.values()]
        if multi_gpu:
            from . import multi
            scan = multi.scan_on_devices(token_bytes, devices, guide_len)
        else:
            scan = scan_token_bytes(token_bytes, guide_len, limit=handle_limit)
    per_token = scan.seg_plus.astype(np.int64) + scan.seg_minus.astype(np.int64)
    table = emit.CandidateTable(guide_len, capacity=int(per_token.sum()))
    rows_written = 0
    # the cumulative list sizes of every emission are known once the scan is through: their ids
    # (CROPSR.py:448) are drawn ahead, in the reference's order, while rows are being written
    id_stream = emit.IdStream(np.cumsum(per_token))
    for k, (key, value) in enumerate(tokens.items()):
        out("Searching on Chromosome: ", key[:25])       # :410-411
        out("With start of sequence: ", value[:25])
        t_plus, x_plus, t_minus, x_minus = scan.token_rows(k)
        table.append_token(key, scan.token_bytes[k], k, t_plus, x_plus, t_minus, x_minus)
        if verbose:
            n = len(t_plus) + len(t_minus)
            out(f"\n                {n:n} Cas9 PAM sites were found on {key[1:]}\n                ")
        rows_written += emit.emit_cumulative(output, table, scan, blas_threads, id_stream, chunk_rows)
        timing.write("Total runtime of the program is " + str(time.time() - begin))   # :476-477
    id_stream.close()
    timing.close()
    if side_output and guide_len == 20:
        if multi_gpu:
            raise NotImplementedError("--side-output needs the packed genome on one device: run it without --devices")
        with open(fasta, "r") as f:
            formatted_path = ingest.needs_formatting(f.read())
        write_side_output(side_output, tokens, scan, gff_frame, flank, formatted_path, annotation_info)
        write_gap_table(side_output + ".gaps.tsv", tokens, scan)
    ot_stats = {}
    if offtargets is not None or offtarget_sites is not None or offtarget_scores is not None:
        handles = [g for g, _, _, _ in scan.parts]
        indexes = []                                    # NGG first, then the extra patterns in the order given
        try:
            for pam in ["NGG"] + pams:
                indexes.append(engine.OffTargetIndex(handles, loci=offtarget_sites is not None, pam=pam))
            index = indexes[0]
            # with the sites table, each strand is counted once for both count-driven tables
            counts = [offtarget_counts(ix, scan, max_mismatches) if offtarget_sites is not None else None
                      for ix in indexes]
            extra = [(pam, ix, c) for pam, ix, c in zip(pams, indexes[1:], counts[1:])]
            if offtargets is not None:
                write_offtarget_table(offtargets, tokens, scan, max_mismatches, index=index, counts=counts[0],
                                      extra=extra)
            if offtarget_sites is not None:
                pairs, capped = write_offtarget_sites(offtarget_sites, tokens, scan, max_mismatches, max_sites,
                                                      index=index, counts=counts[0], extra=extra)
                ot_stats = {"offtarget_pairs": pairs, "offtarget_capped": capped}
            if offtarget_scores is not None:
                write_offtarget_scores(offtarget_scores, tokens, scan, max_mismatches, index=index,
                                       extra=[(pam, ix) for pam, ix, _ in extra])
        finally:
            for ix in indexes:
                ix.free()
        if verbose and offtarget_sites is not None:
            at = f" at {', '.join(['NGG'] + pams)} PAMs" if pams else ""
            out(f"{pairs:n} off-target sites{at} listed in {offtarget_sites}; {capped:n} candidates with more than "
                f"{max_sites:n} left out")
    stats = {"tokens": len(tokens), "candidates": len(table), "rows": rows_written,
             "scan_ms": scan.scan_ms(), **scan.timing(), **ot_stats}
    t_plus = x_plus = t_minus = x_minus = None          # views into the scan's row arrays
    scan.free()
    if verbose:
        out(f"The output file has been generated at {output}")
    return stats
