"""numpy restatement of the in-frame indel rule (restatement choice U19, DESIGN.md "In-frame indels").

Input: unpacked column states [R, L] (bits 0-2: 0-3 A/C/G/T, 4 '-', 5 N, 7 not spanned) and the insertion events
(read, col, off, len, pool) as ms_expand_cigar appends them.  The hypergeometric tail is scipy's."""
import math

import numpy as np
from scipy.stats import hypergeom

AA = None


def _aa_table():
    global AA
    if AA is None:
        ncbi = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG"
        AA = "".join(ncbi[16 * "TCAG".index(a) + 4 * "TCAG".index(b) + "TCAG".index(c)] for a in "ACGT" for b in "ACGT" for c in "ACGT")
    return AA


def codon_starts(L, genes, region=None):
    """per gene: the tested codons [(codon index, start column)], as K2 enumerates them"""
    lo, hi = 0, L
    if region:
        lo, hi = max(0, region[0] - 1), min(L, region[1] - 1)
    out = []
    for (b, e) in genes:
        gb, ge = b - 1, min(e - 1, L)
        cods, s, ci = [], gb, 0
        while s + 3 <= ge:
            if s >= lo and s + 3 <= hi and s >= 0:
                cods.append((ci, s))
            s += 3
            ci += 1
        out.append(cods)
    return out


def start_bits(L, genes, region=None):
    m = np.zeros(L, dtype=bool)
    for cods in codon_starts(L, genes, region):
        for _, s in cods:
            m[s] = True
    return m


def counts(states, events, start, read0=0):
    """-> cnt [L, 2] (k_del, n_ins of every column), strings [(col, x)] in id order, tally [nsid] over reads
    [read0, read0 + R) of the events' numbering"""
    st = np.asarray(states) & 7
    R, L = st.shape
    gap, clean = st == 4, st < 4
    cnt = np.zeros((L, 2), dtype=np.int64)
    if L >= 3:
        cnt[: L - 2, 0] = (gap[:, :-2] & gap[:, 1:-1] & gap[:, 2:]).sum(axis=0)
    cnt[: L - 1, 1] = (clean[:, :-1] & clean[:, 1:]).sum(axis=0)
    read, col, off, ln, pool = events if events is not None else ([], [], [], [], b"")
    first = {}
    for i in range(len(read)):
        c = int(col[i])
        if c - 2 < 0 or c + 1 >= L or not (start[c - 2] and start[c + 1]):
            continue
        first.setdefault((int(read[i]), c), i)
    kept = []
    for (r, c), i in first.items():
        n = int(ln[i])
        x = bytes(pool[int(off[i]): int(off[i]) + n]).decode("latin-1")
        if n < 3 or n % 3 or any(ch not in "ACGTacgt" for ch in x):
            continue
        kept.append((r, c, x.upper()))
    strings = sorted({(c, x) for _, c, x in kept})
    sid = {k: i for i, k in enumerate(strings)}
    tally = np.zeros(len(strings), dtype=np.int64)
    for r, c, x in kept:
        lr = r - read0
        if 0 <= lr < R and clean[lr, c] and clean[lr, c + 1]:
            tally[sid[(c, x)]] += 1
    return cnt, strings, tally


def fisher_p(k, n, e):
    """P(X >= k) of [[k, n-k], [e, n-e]]"""
    return float(hypergeom.sf(k - 1, 2 * n, k + e, n))


def expected(n, P):
    ex = math.ceil(n * P)
    return n if ex >= n else int(ex)


def _codon_hist(st, s):
    c = st[:, s: s + 3]
    ok = (c < 4).all(axis=1)
    idx = 16 * c[ok, 0].astype(np.int64) + 4 * c[ok, 1] + c[ok, 2]
    return np.bincount(idx, minlength=64)


def _ref_codon(refseq, s, hist):
    if refseq is not None and s + 3 <= len(refseq):
        t = refseq[s: s + 3]
        if all(ch in "ACGTacgt" for ch in t):
            return 16 * "ACGT".index(t[0].upper()) + 4 * "ACGT".index(t[1].upper()) + "ACGT".index(t[2].upper())
    return int(np.argmax(hist)) if hist.sum() else -1


def call(states, cnt, strings, tally, genes, refseq=None, region=None, deletion_rate=3e-3, insertion_rate=3e-3, alpha=0.01,
         min_perc=-1.0, max_perc=-1.0):
    """-> list of dicts sorted by (gene, codon, deletion first, string); states are all the reads (K2's coverage)"""
    st = np.asarray(states) & 7
    L = st.shape[1]
    Pdel = 1.0
    for _ in range(3):
        Pdel *= deletion_rate
    by_col = {}
    for i, (c, x) in enumerate(strings):
        by_col.setdefault(c, []).append(i)
    out = []
    hist_cache = {}

    def hist(s):
        if s not in hist_cache:
            hist_cache[s] = _codon_hist(st, s)
        return hist_cache[s]

    def test(k, n, P, m):
        if k == 0 or n == 0:
            return None
        e = expected(n, P)
        if k <= e and 0.5 * m >= alpha:
            return None
        p = fisher_p(k, n, e)
        if not (p * m < alpha):
            return None
        perc = 100.0 * k / n
        if min_perc >= 0 and not perc > min_perc:
            return None
        if max_perc >= 0 and not perc < max_perc:
            return None
        return e, p

    for g, cods in enumerate(codon_starts(L, genes, region)):
        m = len(cods)
        starts = {s for _, s in cods}
        for ci, s in cods:
            k = int(cnt[s, 0])
            n = k + int(hist(s).sum())
            r = test(k, n, Pdel, m)
            if r:
                out.append(dict(gene=g, codon_index=ci, col=s, kind=0, inserted="", count=k, coverage=n, expected=r[0], pvalue=r[1],
                                ntests=m, ref_codon=_ref_codon(refseq, s, hist(s)), next_codon=-1))
            c = s + 2
            if s + 3 not in starts:
                continue
            for i in by_col.get(c, []):
                x = strings[i][1]
                P = 1.0
                for _ in range(len(x)):
                    P *= insertion_rate
                k, n = int(tally[i]), int(cnt[c, 1])
                r = test(k, n, P, m)
                if r:
                    out.append(dict(gene=g, codon_index=ci, col=c, kind=1, inserted=x, count=k, coverage=n, expected=r[0], pvalue=r[1],
                                    ntests=m, ref_codon=_ref_codon(refseq, s, hist(s)), next_codon=_ref_codon(refseq, s + 3, hist(s + 3))))
    return out


def translate(x):
    """amino acids of an in-frame string, '*' for a stop"""
    aa = _aa_table()
    return "".join(aa[16 * "ACGT".index(x[i]) + 4 * "ACGT".index(x[i + 1]) + "ACGT".index(x[i + 2])] for i in range(0, len(x) - 2, 3))


def label(kind, ref_codon, next_codon, aa_pos, inserted=""):
    """D67del; T69_S70insSS (stop codons of the reference read 'X', as K2's labels; inserted stops '*')"""
    aa = _aa_table()
    a = lambda c: aa[c].replace("*", "X") if c >= 0 else "?"
    if kind == 0:
        return f"{a(ref_codon)}{aa_pos}del"
    return f"{a(ref_codon)}{aa_pos}_{a(next_codon)}{aa_pos + 1}ins{translate(inserted)}"
