"""CPU ORACLE for the opt-in off-target counts (csrc/offtarget.cuh).  TEST INFRASTRUCTURE ONLY.

Parity status: UNPINNED BY THE REFERENCE.  The reference leaves specificity to an external aligner
(the bowtie2 call of /root/reference/prmrdsgn2.py:139-160), so this module is the specification the
CUDA kernels are tested against, written from the definition with Python strings:

  base        a byte of ACGTacgt, case folded to the code A0 T1 C2 G3; complement = code ^ 1
  site '+' t  tok[t+1], tok[t+2] in "Gg", t >= 20, tok[t-20:t] all bases;     P = tok[t-20:t]
  site '-' t  tok[t], tok[t+1] in "Cc", t + 23 <= L, tok[t+3:t+23] all bases;  P = revcomp(tok[t+3:t+23])
  key         P[i] in bits 2i, 2i+1 (P[0] = the PAM-distal 5' base)
  query       a scan candidate (cropsr_oracle.pam_hits, l = 20) with the P of the same formulas, or None
              when P is cut off or holds a non-base; its own site is not counted
  counts      mm_d = sites at exactly d mismatches, d = 0 .. k

`site_keys_np` is a vectorised builder for genome-scale checks, pinned to `sites` by the tests.
"""
import numpy as np

import cropsr_oracle as oracle

CODE = {c: i for i, c in enumerate("ATCG")}
CODE.update({c.lower(): i for c, i in list(CODE.items())})
DNA = "ATCG"


def _key(codes):
    k = 0
    for i, c in enumerate(codes):
        k |= c << (2 * i)
    return k


def protospacer_codes(tok, t, strand):
    """codes of P for a site / candidate at t, or None (cut off by the token end or a non-base)"""
    if strand == "+":
        if t < 20:
            return None
        win = tok[t - 20:t]
        codes = [CODE.get(ch) for ch in win]
    else:
        if t + 23 > len(tok):
            return None
        win = tok[t + 3:t + 23]
        codes = [None if CODE.get(ch) is None else CODE[ch] ^ 1 for ch in reversed(win)]
    if len(codes) != 20 or any(c is None for c in codes):
        return None
    return codes


def protospacer(tok, t, strand):
    """P as upper-case DNA, or None"""
    codes = protospacer_codes(tok, t, strand)
    return None if codes is None else "".join(DNA[c] for c in codes)


def key_of(guide):
    """key of a 20-base guide string in the protospacer orientation (case-insensitive)"""
    codes = [CODE[ch] for ch in guide]
    assert len(codes) == 20
    return _key(codes)


def sites(tok):
    """[(t, strand, key)] of one token, '+' then '-' by ascending t"""
    L = len(tok)
    out = []
    for strand in "+-":
        for t in range(L):
            if strand == "+":
                ok = t + 2 < L and tok[t + 1] in "Gg" and tok[t + 2] in "Gg"
            else:
                ok = t + 1 < L and tok[t] in "Cc" and tok[t + 1] in "Cc"
            if not ok:
                continue
            codes = protospacer_codes(tok, t, strand)
            if codes is not None:
                out.append((t, strand, _key(codes)))
    return out


def mismatches(a, b):
    """number of differing bases of two keys (numpy arrays or ints)"""
    x = np.bitwise_xor(np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64))
    y = (x | (x >> np.uint64(1))) & np.uint64(0x5555555555)
    return np.bitwise_count(y).astype(np.int64)


def counts_for_key(key, site_keys, k):
    """[mm_0 .. mm_k] of one key against all sites, brute force"""
    d = mismatches(np.uint64(key), site_keys)
    return np.bincount(d[d <= k], minlength=k + 1)[:k + 1].astype(np.int64)


def candidate_rows(tokens, k):
    """One row per unique scan candidate in reference order (token by token, '+' then '-', ascending t):
    (token index, strand, t, protospacer or None, [mm_0 .. mm_k] or None), against the sites of ALL tokens."""
    all_keys = np.array([key for tok in tokens for _, _, key in sites(tok)], dtype=np.uint64)
    rows = []
    for ti, tok in enumerate(tokens):
        plus, minus = oracle.pam_hits(tok, 20)
        for strand, ts in (("+", plus), ("-", minus)):
            for t in ts:
                codes = protospacer_codes(tok, t, strand)
                if codes is None:
                    rows.append((ti, strand, t, None, None))
                    continue
                c = counts_for_key(_key(codes), all_keys, k)
                c[0] -= 1                               # the candidate's own site
                rows.append((ti, strand, t, "".join(DNA[x] for x in codes), c.tolist()))
    return rows


# ---- vectorised site keys (genome-scale checks)
_LUT = np.full(256, -1, dtype=np.int8)
for _c, _v in CODE.items():
    _LUT[ord(_c)] = _v


def site_keys_np(tok):
    """(t, strand 0 '+' / 1 '-', key) arrays of one token (bytes / uint8 array), any order"""
    b = np.frombuffer(tok, dtype=np.uint8) if isinstance(tok, (bytes, bytearray)) else np.asarray(tok, dtype=np.uint8)
    code = _LUT[b].astype(np.int64)
    L = len(b)
    bad = np.concatenate(([0], np.cumsum(code < 0)))          # non-bases in [0, i) = bad[i]
    g = (b == ord("G")) | (b == ord("g"))
    c = (b == ord("C")) | (b == ord("c"))
    out_t, out_s, out_k = [], [], []
    if L >= 23:
        t = np.nonzero(g[1:L - 1] & g[2:L])[0]                # tok[t+1], tok[t+2]
        t = t[t >= 20]
        t = t[bad[t] - bad[t - 20] == 0]
        key = np.zeros(len(t), dtype=np.uint64)
        for i in range(20):
            key |= code[t - 20 + i].astype(np.uint64) << np.uint64(2 * i)
        out_t.append(t), out_s.append(np.zeros(len(t), np.int8)), out_k.append(key)
        t = np.nonzero(c[:L - 1] & c[1:L])[0]
        t = t[t + 23 <= L]
        t = t[bad[t + 23] - bad[t + 3] == 0]
        key = np.zeros(len(t), dtype=np.uint64)
        for i in range(20):
            key |= (code[t + 22 - i] ^ 1).astype(np.uint64) << np.uint64(2 * i)
        out_t.append(t), out_s.append(np.ones(len(t), np.int8)), out_k.append(key)
    if not out_t:
        return np.zeros(0, np.int64), np.zeros(0, np.int8), np.zeros(0, np.uint64)
    return np.concatenate(out_t), np.concatenate(out_s), np.concatenate(out_k)
