"""CPU ORACLE for the opt-in off-target scores (csrc/offtarget.cuh k_ot_join<OtScore>, crp_offtarget_score_*,
engine.OffTargetIndex.score_candidates / score_guides, pipeline.write_offtarget_scores).  TEST INFRASTRUCTURE ONLY.

Parity status: UNPINNED BY THE REFERENCE (it has no off-target search).  Written from the definition with Python
strings, brute force over offtarget_oracle.sites; it keeps its own copy of the MIT constants and reads nothing of
the engine's weight table:

  pairs             exactly those the counts of offtarget_oracle count: every NGG site of every token within
                    d <= k <= 3 mismatches of the candidate's protospacer, the candidate's own site left out
  mismatch set      the positions (0 = P[0], PAM-distal, .. 19) where the two protospacer strings differ
  hit               CRISPOR's calcHitScore of the set, in this IEEE double order:
                      score1 = 1.0; for p ascending: score1 *= 1 - M[p]
                      score2 = 1.0 if n < 2 else 1.0 / (((19 - mean(consecutive distances)) / 19.0) * 4 + 1)
                      score3 = 1.0 if n == 0 else 1.0 / (n ** 2)
                      hit = score1 * score2 * score3 * 100
                    (the mean of CONSECUTIVE distances, as CRISPOR computes it, not the paper's all-pairs mean)
  weight            round(hit * 2**24), half to even
  sum S             the integer sum of the weights of a candidate's pairs; a candidate without a protospacer has none
  mit_hit_sum       S / 2**24 as a float, formatted .6f
  mit_specificity   int(round(100 / (100 + S / 2**24) * 100))  (CRISPOR's calcMitGuideScore)
  scores table      tab-separated, a header row, '\\r\\n' line ends; one row per candidate in
                    offtarget_oracle.candidate_rows order: chromosome strand pam_pos protospacer mit_hit_sum
                    mit_specificity; protospacer and both scores blank where the candidate has no protospacer

CRISPOR sums over 4 mismatches and NAG / NGA sites too; these numbers cover NGG sites within k <= 3 only.
"""
import numpy as np

import offtarget_oracle as ot

M = [0, 0, 0.014, 0, 0, 0.395, 0.317, 0, 0.389, 0.079, 0.445, 0.508, 0.613, 0.851, 0.732, 0.828, 0.615, 0.804,
     0.685, 0.583]
ONE = 1 << 24
COLUMNS = ["chromosome", "strand", "pam_pos", "protospacer", "mit_hit_sum", "mit_specificity"]


def hit(positions):
    positions = sorted(positions)
    score1 = 1.0
    for p in positions:
        score1 *= 1 - M[p]
    n = len(positions)
    if n < 2:
        score2 = 1.0
    else:
        dists = [positions[i + 1] - positions[i] for i in range(n - 1)]
        score2 = 1.0 / (((19 - sum(dists) / len(dists)) / 19.0) * 4 + 1)
    score3 = 1.0 if n == 0 else 1.0 / (n ** 2)
    return score1 * score2 * score3 * 100


def mit_weight(positions):
    return round(hit(positions) * ONE)


def mismatch_positions(a, b):
    """positions where two 20-base protospacer strings differ, case-insensitive"""
    return tuple(i for i, (x, y) in enumerate(zip(a.upper(), b.upper())) if x != y)


def _site_strings(tokens):
    """(keys array, protospacer strings) of every site of every token"""
    found = [(key, ot.protospacer(tok, t, s)) for tok in tokens for t, s, key in ot.sites(tok)]
    return np.array([k for k, _ in found], dtype=np.uint64), [p for _, p in found]


def _pairs(proto, keys, strings, k):
    """mismatch sets of every site within k mismatches of a protospacer string"""
    near = np.nonzero(ot.mismatches(np.uint64(ot.key_of(proto)), keys) <= k)[0] if len(keys) else []
    return [mismatch_positions(proto, strings[i]) for i in near]


def candidate_pairs(tokens, k):
    """One row per candidate in offtarget_oracle.candidate_rows order: (token index, strand, t, protospacer or None,
    [mismatch set of every OTHER site within k mismatches] or None)"""
    keys, strings = _site_strings(tokens)
    rows = []
    for ti, strand, t, proto, _ in ot.candidate_rows(tokens, 0):
        if proto is None:
            rows.append((ti, strand, t, None, None))
            continue
        sets = _pairs(proto, keys, strings, k)
        sets.remove(())                                 # the candidate's own site
        rows.append((ti, strand, t, proto, sets))
    return rows


def candidate_sums(tokens, k, weight=mit_weight, pairs=None):
    """candidate_pairs rows with S = sum of weight(mismatch set) in place of the sets (None without a protospacer).
    pairs: candidate_pairs(tokens, K) for some K >= k, to reuse"""
    pairs = candidate_pairs(tokens, k) if pairs is None else pairs
    return [(ti, strand, t, proto, None if sets is None else sum(weight(x) for x in sets if len(x) <= k))
            for ti, strand, t, proto, sets in pairs]


def guide_sums(tokens, guides, k, weight=mit_weight):
    """S of 20-base guides (protospacer orientation, any case) over every site; nothing left out"""
    keys, strings = _site_strings(tokens)
    return [sum(weight(s) for s in _pairs(g, keys, strings, k)) for g in guides]


def specificity(S):
    return int(round(100 / (100 + S / ONE) * 100))


def scores_table(tokens, k):
    """the --offtarget-scores table of a token dict ({'>name': sequence}), byte for byte"""
    names = [key[1:] for key in tokens]
    lines = ["\t".join(COLUMNS)]
    for ti, strand, t, proto, S in candidate_sums(list(tokens.values()), k):
        lines.append("\t".join([names[ti], strand, str(t)] +
                               ([proto, f"{S / ONE:.6f}", str(specificity(S))] if proto else ["", "", ""])))
    return "\r\n".join(lines) + "\r\n"
