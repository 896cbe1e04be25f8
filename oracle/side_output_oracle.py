"""CPU ORACLE for the whole --side-output table and its .gaps.tsv companion, byte for byte.  TEST
INFRASTRUCTURE ONLY: only tests/ may import it.

Built from the tokens with Python strings, extras_oracle (candidates, cut site, flank window, gap runs) and
primer_oracle.design_fast (primer columns).  The only library code it calls is the GFF and annotation-info
parsing that tests/test_host_logic.py already pins (ingest.import_gff_file, which the caller uses to make the
frame, and annotate.read_annotation_info / lookup_annotation_info).  UNPINNED BY THE REFERENCE, like
extras_oracle: the reference writes no such table.  The rules:

- Rows: one per unique candidate, token by token (ingest-dict order), '+' rows then '-' rows, each by
  ascending pam_pos; CRLF line ends, tab separated, csv quoting (QUOTE_MINIMAL) where a cell needs it.
- Protospacer (gc, poly_t, homopolymer, low_gc, unscored_base, longest_run): the 20 bases [5:25] of the
  scored 30-mer.  Positions past the token end are unscored bytes: they set unscored_base (flag 8), are never
  G/C and break runs.  That is what the packed records hold there, and it gives every row, truncated '-'
  rows within 23 bases of the token end included, a defined gc / flags / run.
- cutsite = pam_pos - 3 on '+', pam_pos on '-'; flank = [max(cut - flank, 0), min(cut + flank, len(token))).
- Features: GFF rows whose type is gene or CDS, with finite start and end, on the record the token holds.
  GFF coordinates (1-based) shift by -1 on the clean ingest path and by 0 on the formatted path (whose tokens
  carry a leading quote).  A feature holds the cut site when start <= cut <= end (inclusive).  Among the
  holding features the one with the latest start wins; among equal starts the shorter one (smaller end); among
  identical intervals the later GFF row.
- Primer columns (fwd_primers, rev_primers, primer_pairs, first_pair) are blank where
  flank_end - flank_start < e + l (130 with the defaults); otherwise design_fast of token[flank_start:flank_end]
  with the defaults, and first_pair printed as "fi+fN/ri+rN" (blank when no pair is Tm-close).
- annotation_info: lookup_annotation_info of the feature's attributes in the -p table ('' without one).
- chromosome is the ingest key without its first character (formatted path: "('name',").
- .gaps.tsv: header chromosome / start / length, then per token its maximal runs of bytes that are not
  ACGTacgt of at least 10 bytes, ascending, in token coordinates; CRLF line ends.
"""
import csv
import io
import math

import cropsr_oracle as oracle
import extras_oracle
import primer_oracle

COLUMNS = ["chromosome", "strand", "pam_pos", "cutsite", "gc", "poly_t", "homopolymer", "low_gc", "unscored_base",
           "longest_run", "flank_start", "flank_end", "feature_type", "feature_attributes", "fwd_primers",
           "rev_primers", "primer_pairs", "first_pair", "annotation_info"]
FEATURES = ("gene", "CDS")
PRIMER_REGION = 100 + 30          # e + l of primer_oracle's defaults
GAP_MIN_LEN = 10


def protospacer(long_, strand):
    """The 20 scored bytes [5:25] of a candidate's 30-mer as a string, '-' for a position past the token end.
    long_ is the reference's long sequence (cropsr_oracle.candidates_for_token): a '+' window is read
    backwards, so what the token end cuts off is its head; a '-' window loses its tail."""
    pad = "-" * (30 - len(long_))
    full = pad + long_ if strand == "+" else long_ + pad
    return full.replace("U", "T").upper()[5:25]          # cropsr_oracle.scored_bytes


def protospacer_stats(proto):
    """-> (gc, flags, run) of a 20-byte scored protospacer (extras_oracle's rules; non-ACGT bytes unscored)"""
    gc = proto.count("G") + proto.count("C")
    run = best = 0
    prev = None
    for ch in proto:
        if ch in "ACGT":
            run = run + 1 if ch == prev else 1
            prev = ch
        else:
            run, prev = 0, None
        best = max(best, run)
    flags = (1 if "TTTT" in proto else 0) | (2 if best >= 5 else 0) | (4 if gc < 10 else 0) | \
            (8 if any(ch not in "ACGT" for ch in proto) else 0)
    return gc, flags, best


def token_chromosome(key, formatted_path):
    """The GFF seqid a token's ingest key stands for: '>chr1' (clean), "[('chr1'," / "('chr2'," (formatted)"""
    return key.strip("[](),").strip("'\"") if formatted_path else key[1:]


def features_by_chromosome(gff_frame, formatted_path):
    """{seqid: [(start, end, frame row, type, attributes)]} in token coordinates, GFF row order"""
    shift = 0 if formatted_path else -1
    out = {}
    for row, (chrom, ftype, start, end, attr) in enumerate(zip(gff_frame["chromosome"].tolist(), gff_frame["feature"].tolist(),
                                                                gff_frame["start"].tolist(), gff_frame["end"].tolist(),
                                                                gff_frame["attributes"].tolist())):
        if ftype not in FEATURES:
            continue
        try:
            start, end = float(start), float(end)
        except (TypeError, ValueError):
            continue
        if not (math.isfinite(start) and math.isfinite(end)):
            continue
        out.setdefault(chrom, []).append((int(start) + shift, int(end) + shift, row, ftype, attr))
    return out


def feature_at(features, cut):
    """The winning feature holding the cut site, or None"""
    return max((f for f in features if f[0] <= cut <= f[1]), key=lambda f: (f[0], -f[1], f[2]), default=None)


def _text(v):
    return v if isinstance(v, str) else ""            # a missing GFF cell (NaN) prints empty


def side_output_rows(tokens, gff_frame, flank, formatted_path, info=None, design=primer_oracle.design_fast, pool_map=map):
    """-> list of rows (lists of str) in table order.  tokens: the ingest dict {key: token}; info: the dict of
    annotate.read_annotation_info, or None; pool_map: a map function for the primer designs (a process pool's,
    to spread design_fast over CPUs)."""
    from cropsr_b200 import annotate
    feats = features_by_chromosome(gff_frame, formatted_path)
    rows, frags, where = [], [], []
    for key, tok in tokens.items():
        fl = feats.get(token_chromosome(key, formatted_path), [])
        ex = extras_oracle.extras_for_token(key, tok, flank)
        for c, e in zip(oracle.candidates_for_token(key, tok, 20), ex):
            strand = c[6]
            gc, flags, run = protospacer_stats(protospacer(c[4], strand))
            f = feature_at(fl, e["cut"])
            ftype, attr = (_text(f[3]), _text(f[4])) if f else ("", "")
            ai = annotate.lookup_annotation_info(info, f[4]) if (f and info) else ""
            rows.append([key[1:], strand, str(e["t"]), str(e["cut"]), str(gc), str(flags & 1), str(flags >> 1 & 1),
                         str(flags >> 2 & 1), str(flags >> 3 & 1), str(run), str(e["flank_lo"]), str(e["flank_hi"]),
                         ftype, attr, "", "", "", "", ai])
            if e["flank_hi"] - e["flank_lo"] >= PRIMER_REGION:
                frags.append(tok[e["flank_lo"]:e["flank_hi"]])
                where.append(len(rows) - 1)
    for i, d in zip(where, pool_map(design, frags)):
        first = d["first"]
        rows[i][14:18] = [str(d["n_fwd"]), str(d["n_rev"]), str(d["n_pairs"]),
                          "{}+{}/{}+{}".format(*first) if first else ""]
    return rows


def side_output_text(tokens, gff_frame, flank, formatted_path, annotation_info=None, pool_map=map):
    """The whole --side-output file as a str (annotation_info: path of the -p file, or None)"""
    from cropsr_b200 import annotate
    info = annotate.read_annotation_info(annotation_info) if annotation_info else None
    buf = io.StringIO(newline="")
    w = csv.writer(buf, delimiter="\t", lineterminator="\r\n")
    w.writerow(COLUMNS)
    w.writerows(side_output_rows(tokens, gff_frame, flank, formatted_path, info, pool_map=pool_map))
    return buf.getvalue()


def gaps_text(tokens, min_len=GAP_MIN_LEN):
    """The whole .gaps.tsv file as a str"""
    buf = io.StringIO(newline="")
    w = csv.writer(buf, delimiter="\t", lineterminator="\r\n")
    w.writerow(["chromosome", "start", "length"])
    for key, tok in tokens.items():
        w.writerows((key[1:], a, n) for a, n in extras_oracle.other_runs(tok, min_len))
    return buf.getvalue()
