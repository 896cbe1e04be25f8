"""CPU ORACLE for the opt-in off-target listing and sites table (k_ot_join<OtList>, crp_offtarget_list_*,
engine.OffTargetIndex.list_candidates / list_guides, pipeline.write_offtarget_sites).  TEST INFRASTRUCTURE ONLY.

Parity status: UNPINNED BY THE REFERENCE (it has no off-target search).  Written from the definition with Python
strings, brute force over offtarget_oracle.sites:

  listing of a candidate   every site of every token within k mismatches of the candidate's protospacer, its own
                           site (same token, t and strand) left out: as many sites as its counts sum to
  listing of a guide       every site within k mismatches; nothing left out
  sites table              tab-separated, a header row, '\\r\\n' line ends; one row per (candidate, listed site):
                             chromosome strand pam_pos protospacer site_chromosome site_strand site_pam_pos
                             site_protospacer mismatches
                           candidates in offtarget_oracle.candidate_rows order, and within a candidate by mismatches,
                           the site's token (file order), site_pam_pos, '+' before '-'; site_protospacer is the
                           site's 20 bases, upper case, in the orientation followed by NGG, with the bases that differ
                           from the candidate's protospacer in lower case; a candidate with no listed site or with
                           more than max_sites writes no rows

`neighbours_np` is the vectorised helper for sampled genome-scale checks, over the arrays of
offtarget_oracle.site_keys_np.
"""
import numpy as np

import offtarget_oracle as ot

COLUMNS = ["chromosome", "strand", "pam_pos", "protospacer", "site_chromosome", "site_strand", "site_pam_pos",
           "site_protospacer", "mismatches"]


def all_sites(tokens):
    """[(token index, t, strand, key)] of every token: token by token, '+' then '-' by ascending t"""
    return [(ti, t, s, key) for ti, tok in enumerate(tokens) for t, s, key in ot.sites(tok)]


def _sort_key(entry):
    d, ti, t, strand, _ = entry
    return d, ti, t, strand == "-"


def listing(tokens, k):
    """One row per unique candidate in candidate_rows order: (token index, strand, t, protospacer or None,
    counts or None, sites), sites = [(d, site token, site t, site strand, site key)] in the table's order
    (empty for a candidate without a protospacer)."""
    every = all_sites(tokens)
    keys = np.array([key for _, _, _, key in every], dtype=np.uint64)
    rows = []
    for ti, strand, t, proto, counts in ot.candidate_rows(tokens, k):
        found = []
        if proto is not None:
            d = ot.mismatches(np.uint64(ot.key_of(proto)), keys) if len(keys) else np.zeros(0, np.int64)
            for i in np.nonzero(d <= k)[0].tolist():
                si, st, ss, sk = every[i]
                if (si, st, ss) != (ti, t, strand):
                    found.append((int(d[i]), si, st, ss, sk))
            found.sort(key=_sort_key)
        rows.append((ti, strand, t, proto, counts, found))
    return rows


def guide_listing(tokens, guides, k):
    """[[(d, site token, site t, site strand, site key)] in the table's order] of 20-base guides"""
    every = all_sites(tokens)
    keys = np.array([key for _, _, _, key in every], dtype=np.uint64)
    out = []
    for g in guides:
        d = ot.mismatches(np.uint64(ot.key_of(g)), keys) if len(keys) else np.zeros(0, np.int64)
        out.append(sorted(((int(d[i]),) + every[i][:3] + (every[i][3],) for i in np.nonzero(d <= k)[0].tolist()),
                          key=_sort_key))
    return out


def key_bases(key):
    """the 20 bases of a key, upper case, P[0] first"""
    return "".join(ot.DNA[(int(key) >> (2 * i)) & 3] for i in range(20))


def site_protospacer(key, protospacer):
    """the site's bases, lower case where they differ from the candidate's protospacer"""
    return "".join(b if b == p else b.lower() for b, p in zip(key_bases(key), protospacer))


def sites_table(tokens, k, max_sites=1000):
    """The sites table, byte by byte, of a {'>name': token} dict"""
    names = [key[1:] for key in tokens]
    lines = ["\t".join(COLUMNS)]
    for ti, strand, t, proto, counts, found in listing(list(tokens.values()), k):
        if not found or len(found) > max_sites:
            continue
        for d, si, st, ss, sk in found:
            lines.append("\t".join([names[ti], strand, str(t), proto, names[si], ss, str(st),
                                    site_protospacer(sk, proto), str(d)]))
    return "\r\n".join(lines) + "\r\n"


def neighbours_np(key, site_keys, k):
    """(indices, mismatches) of the sites of site_keys (uint64, e.g. site_keys_np's keys concatenated) within k
    mismatches of key, brute force; the caller leaves a candidate's own site out"""
    d = ot.mismatches(np.uint64(key), site_keys)
    idx = np.nonzero(d <= k)[0]
    return idx, d[idx]
