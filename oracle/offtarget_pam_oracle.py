"""CPU ORACLE for off-target sites at other PAM patterns (csrc/offtarget.cuh k_ot_sites<*, true>,
crp_offtarget_new_pam, engine.OffTargetIndex(pam=), --offtarget-pams).  TEST INFRASTRUCTURE ONLY.

Parity status: UNPINNED BY THE REFERENCE (it has no off-target search).  Written from the definition with Python
strings, on top of offtarget_oracle (whose NGG functions it leaves as they are); it keeps its own IUPAC table:

  pattern     three characters, any case: N, then two of A C G T R Y S W K M B D H V (N refused there); S2, S3 the
              bases of letters 2 and 3
  site '+' t  tok[t+1] a base in S2, tok[t+2] a base in S3, t >= 20, tok[t-20:t] all bases;     P = tok[t-20:t]
  site '-' t  tok[t] a base in comp(S3), tok[t+1] a base in comp(S2), t + 23 <= L, tok[t+3:t+23] all bases;
              P = revcomp(tok[t+3:t+23])
  own site    a candidate's own site is a site of the pattern exactly when G is in S2 and in S3; only then is it
              subtracted from its counts and score.  A listing leaves out a site at the candidate's own locus.
  tables      with extra patterns (--offtarget-pams, disjoint from NGG and from each other):
                counts   after mm0 .. mmK one group {PAM}_mm0 .. {PAM}_mmK per extra pattern, in the order given,
                         blank where the candidate has no protospacer
                sites    a last column site_pam; the rows of all patterns merged in the order mismatches, site token,
                         site_pam_pos, '+' before '-'; max_sites caps a candidate's total over all patterns
                scores   after mit_hit_sum and mit_specificity (NGG) one {PAM}_mit_hit_sum per extra pattern, then
                         all_mit_specificity = int(round(100 / (100 + H) * 100)), H = (S_NGG + sum of S_PAM) / 2**24
              Without extra patterns every table is offtarget_oracle's / offtarget_sites_oracle's /
              offtarget_score_oracle's, byte for byte.
"""
import numpy as np

import cropsr_oracle as oracle
import offtarget_oracle as ot
import offtarget_score_oracle as sco
import offtarget_sites_oracle as so

LETTERS = {"A": "A", "C": "C", "G": "G", "T": "T", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT", "M": "AC",
           "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG"}
_COMP = {"A": "T", "T": "A", "C": "G", "G": "C"}


def parse(pam):
    """the pattern upper case, or ValueError"""
    p = str(pam).upper()
    if len(p) != 3 or p[0] != "N" or p[1] not in LETTERS or p[2] not in LETTERS:
        raise ValueError(f"bad PAM pattern {pam!r}")
    return p


def letter_sets(pam):
    """(S2, S3) as sets of upper-case bases"""
    p = parse(pam)
    return set(LETTERS[p[1]]), set(LETTERS[p[2]])


def own_site(pam):
    s2, s3 = letter_sets(pam)
    return "G" in s2 and "G" in s3


def overlap(a, b):
    (a2, a3), (b2, b3) = letter_sets(a), letter_sets(b)
    return bool(a2 & b2) and bool(a3 & b3)


def _in(ch, bases):
    return ch in "ACGTacgt" and ch.upper() in bases


def sites(tok, pam="NGG"):
    """[(t, strand, key)] of one token, '+' then '-' by ascending t"""
    s2, s3 = letter_sets(pam)
    c2, c3 = {_COMP[b] for b in s2}, {_COMP[b] for b in s3}
    L = len(tok)
    out = []
    for strand in "+-":
        for t in range(L):
            if strand == "+":
                ok = t + 2 < L and _in(tok[t + 1], s2) and _in(tok[t + 2], s3)
            else:
                ok = t + 1 < L and _in(tok[t], c3) and _in(tok[t + 1], c2)
            if not ok:
                continue
            codes = ot.protospacer_codes(tok, t, strand)
            if codes is not None:
                out.append((t, strand, ot._key(codes)))
    return out


def site_keys_np(tok, pam="NGG"):
    """(t, strand 0 '+' / 1 '-', key) arrays of one token (bytes / uint8 array), any order"""
    s2, s3 = letter_sets(pam)
    b = np.frombuffer(tok, dtype=np.uint8) if isinstance(tok, (bytes, bytearray)) else np.asarray(tok, dtype=np.uint8)
    code = ot._LUT[b].astype(np.int64)
    L = len(b)
    bad = np.concatenate(([0], np.cumsum(code < 0)))

    def member(bases):                                  # bytes of ACGTacgt whose base is in `bases`
        m = np.zeros(256, bool)
        for x in bases:
            m[ord(x)] = m[ord(x.lower())] = True
        return m[b]
    out_t, out_s, out_k = [], [], []
    if L >= 23:
        t = np.nonzero(member(s2)[1:L - 1] & member(s3)[2:L])[0]
        t = t[t >= 20]
        t = t[bad[t] - bad[t - 20] == 0]
        key = np.zeros(len(t), dtype=np.uint64)
        for i in range(20):
            key |= code[t - 20 + i].astype(np.uint64) << np.uint64(2 * i)
        out_t.append(t), out_s.append(np.zeros(len(t), np.int8)), out_k.append(key)
        t = np.nonzero(member({_COMP[x] for x in s3})[:L - 1] & member({_COMP[x] for x in s2})[1:L])[0]
        t = t[t + 23 <= L]
        t = t[bad[t + 23] - bad[t + 3] == 0]
        key = np.zeros(len(t), dtype=np.uint64)
        for i in range(20):
            key |= (code[t + 22 - i] ^ 1).astype(np.uint64) << np.uint64(2 * i)
        out_t.append(t), out_s.append(np.ones(len(t), np.int8)), out_k.append(key)
    if not out_t:
        return np.zeros(0, np.int64), np.zeros(0, np.int8), np.zeros(0, np.uint64)
    return np.concatenate(out_t), np.concatenate(out_s), np.concatenate(out_k)


def all_sites(tokens, pam="NGG"):
    """[(token index, t, strand, key)] of every token: token by token, '+' then '-' by ascending t"""
    return [(ti, t, s, key) for ti, tok in enumerate(tokens) for t, s, key in sites(tok, pam)]


def candidate_rows(tokens, k, pam="NGG"):
    """offtarget_oracle.candidate_rows against the sites of `pam`: (token index, strand, t, protospacer or None,
    [mm_0 .. mm_k] or None), the own site subtracted only where own_site(pam)"""
    keys = np.array([key for _, _, _, key in all_sites(tokens, pam)], dtype=np.uint64)
    rows = []
    for ti, tok in enumerate(tokens):
        plus, minus = oracle.pam_hits(tok, 20)
        for strand, ts in (("+", plus), ("-", minus)):
            for t in ts:
                codes = ot.protospacer_codes(tok, t, strand)
                if codes is None:
                    rows.append((ti, strand, t, None, None))
                    continue
                c = ot.counts_for_key(ot._key(codes), keys, k)
                c[0] -= own_site(pam)
                rows.append((ti, strand, t, "".join(ot.DNA[x] for x in codes), c.tolist()))
    return rows


def listing(tokens, k, pam="NGG"):
    """candidate_rows with the sites of each row: [(d, site token, site t, site strand, site key)] in the sites
    table's order, the site at the candidate's own locus left out"""
    every = all_sites(tokens, pam)
    keys = np.array([key for _, _, _, key in every], dtype=np.uint64)
    rows = []
    for ti, strand, t, proto, counts in candidate_rows(tokens, k, pam):
        found = []
        if proto is not None and len(keys):
            d = ot.mismatches(np.uint64(ot.key_of(proto)), keys)
            found = sorted((int(d[i]),) + every[i] for i in np.nonzero(d <= k)[0].tolist()
                           if every[i][:3] != (ti, t, strand))
            found.sort(key=lambda e: (e[0], e[1], e[2], e[3] == "-"))
        rows.append((ti, strand, t, proto, counts, found))
    return rows


def sums(tokens, k, pam="NGG", weight=sco.mit_weight):
    """per candidate_rows row: S = sum of weight(mismatch set) over the row's listing, or None"""
    out = []
    for ti, strand, t, proto, _, found in listing(tokens, k, pam):
        out.append(None if proto is None else
                   sum(weight(sco.mismatch_positions(proto, so.key_bases(sk))) for *_, sk in found))
    return out


def guide_counts(tokens, guides, k, pam="NGG"):
    keys = np.array([key for _, _, _, key in all_sites(tokens, pam)], dtype=np.uint64)
    return [ot.counts_for_key(ot.key_of(g), keys, k).tolist() for g in guides]


# ---- the tables of run_cas9 / the CLI, byte for byte, of a {'>name': token} dict
def counts_table(tokens, k, pams=()):
    names = [key[1:] for key in tokens]
    toks = list(tokens.values())
    groups = [candidate_rows(toks, k, "NGG")] + [candidate_rows(toks, k, p) for p in pams]
    cols = [f"mm{d}" for d in range(k + 1)] + [f"{p}_mm{d}" for p in pams for d in range(k + 1)]
    lines = ["\t".join(["chromosome", "strand", "pam_pos", "protospacer"] + cols)]
    for rows in zip(*groups):
        ti, strand, t, proto, _ = rows[0]
        vals = [str(c) for r in rows for c in r[4]] if proto else [""] * len(cols)
        lines.append("\t".join([names[ti], strand, str(t), proto or ""] + vals))
    return "\r\n".join(lines) + "\r\n"


def sites_table(tokens, k, max_sites=1000, pams=()):
    names = [key[1:] for key in tokens]
    toks = list(tokens.values())
    patterns = ["NGG"] + list(pams)
    groups = [listing(toks, k, p) for p in patterns]
    lines = ["\t".join(so.COLUMNS + (["site_pam"] if pams else []))]
    for rows in zip(*groups):
        ti, strand, t, proto, _, _ = rows[0]
        found = sorted(((d, si, st, ss, sk, p) for p, r in zip(patterns, rows) for d, si, st, ss, sk in r[5]),
                       key=lambda e: (e[0], e[1], e[2], e[3] == "-"))
        if not found or len(found) > max_sites:
            continue
        for d, si, st, ss, sk, p in found:
            lines.append("\t".join([names[ti], strand, str(t), proto, names[si], ss, str(st),
                                    so.site_protospacer(sk, proto), str(d)] + ([p] if pams else [])))
    return "\r\n".join(lines) + "\r\n"


def scores_table(tokens, k, pams=()):
    names = [key[1:] for key in tokens]
    toks = list(tokens.values())
    base = candidate_rows(toks, 0, "NGG")
    groups = [sums(toks, k, p) for p in ["NGG"] + list(pams)]
    cols = sco.COLUMNS + ([f"{p}_mit_hit_sum" for p in pams] + ["all_mit_specificity"] if pams else [])
    lines = ["\t".join(cols)]
    for i, (ti, strand, t, proto, _) in enumerate(base):
        S = [g[i] for g in groups]
        if proto is None:
            vals = [""] * (len(cols) - 3)
        else:
            vals = [proto, f"{S[0] / sco.ONE:.6f}", str(sco.specificity(S[0]))]
            if pams:
                vals += [f"{s / sco.ONE:.6f}" for s in S[1:]] + [str(sco.specificity(sum(S)))]
        lines.append("\t".join([names[ti], strand, str(t)] + vals))
    return "\r\n".join(lines) + "\r\n"
