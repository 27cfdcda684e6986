"""Pairwise variant linkage restated from the column states (restatement choice U14), for the tests.

Independent of the library's bit matrices and Gram contraction: B (read carries the variant's codon) and M (the three
columns of the variant's codon are all A/C/G/T) are read straight off the [R, L] state array, the 2x2 tables are dense
products of those, and the Fisher tails come from the C oracle's long-double mso_fisher_greater (full tails, no early stop).
"""
import numpy as np

MIN_SPACING = 3          # pairs whose codons share a column are not tested
MIN_READS = 10           # default informative reads of a tested pair
LINKED, EXCLUSIVE = 1, 2


def carry_and_clean(states, keys):
    """-> B, M: [R, V] bool.  keys: (start column, codon 16*b0+4*b1+b2) pairs."""
    st = np.asarray(states) & 7
    R, L = st.shape
    B = np.zeros((R, len(keys)), dtype=bool)
    M = np.zeros((R, len(keys)), dtype=bool)
    for i, (col, codon) in enumerate(keys):
        if col + 2 >= L:
            continue                                   # outside the reference: no read spans it
        s = st[:, col: col + 3]
        M[:, i] = (s < 4).all(axis=1)
        B[:, i] = (s == np.array([(codon >> 4) & 3, (codon >> 2) & 3, codon & 3])).all(axis=1)
    return B, M


def tables(states, keys):
    """dense [V, V] int64 n, a, b, c over the informative reads of each pair"""
    B, M = carry_and_clean(states, keys)
    Bf, Mf = B.astype(np.float64), M.astype(np.float64)     # exact: counts stay far below 2^53
    n = np.rint(Mf.T @ Mf).astype(np.int64)
    a = np.rint(Bf.T @ Bf).astype(np.int64)
    bm = np.rint(Bf.T @ Mf).astype(np.int64)                  # bm[v, w] = B_v . M_w
    return n, a, bm - a, bm.T - a


def tails(a, b, c, d, fisher_greater):
    """p_together = P(X >= a), p_apart = P(X <= a) for the top-left cell.  The tail on a's side of the mean, the one that
    can be small, comes from the long-double oracle; the other one (about 1/2 or more) from scipy, because a direct sum
    starting that far on the other side of the mode underflows to 0 even in long double."""
    from scipy.stats import hypergeom
    n, r, k = a + b + c + d, a + b, a + c
    if a * n >= r * k:
        return fisher_greater(a, b, c, d), float(hypergeom.cdf(a, n, r, k))
    return float(hypergeom.sf(a - 1, n, r, k)), fisher_greater(b, a, d, c)


def measures(a, b, c, n):
    """D' and r^2 of one table (0 when a margin is empty or full)"""
    mv, mw = a + b, a + c
    if mv == 0 or mv == n or mw == 0 or mw == n:
        return 0.0, 0.0
    nn = float(n)
    fv, fw = mv / nn, mw / nn
    D = a / nn - fv * fw
    r2 = (D * D) / (fv * (1.0 - fv) * (fw * (1.0 - fw)))
    if D > 0:
        dp = D / min(fv * (1.0 - fw), (1.0 - fv) * fw)
    elif D < 0:
        dp = D / min(fv * fw, (1.0 - fv) * (1.0 - fw))
    else:
        dp = 0.0
    return dp, r2


def linkage(states, keys, fisher_greater, alpha=0.01, min_reads=MIN_READS):
    """-> dict(pairs=[(v, w, both, v_only, w_only, neither, d_prime, r2, pvalue, relation)], ntested, n, a, b, c)"""
    n, a, b, c = tables(states, keys)
    V = len(keys)
    cols = np.array([k[0] for k in keys], dtype=np.int64)
    tested = [(v, w) for v in range(V) for w in range(v + 1, V)
              if abs(cols[v] - cols[w]) >= MIN_SPACING and n[v, w] >= min_reads]
    m = len(tested)
    pairs = []
    for v, w in tested:
        A, Bq, Cq, N = int(a[v, w]), int(b[v, w]), int(c[v, w]), int(n[v, w])
        D = N - A - Bq - Cq
        pt, pa = tails(A, Bq, Cq, D, fisher_greater)
        if pt * m < alpha:
            rel, p = LINKED, pt
        elif pa * m < alpha:
            rel, p = EXCLUSIVE, pa
        else:
            continue
        dp, r2 = measures(A, Bq, Cq, N)
        pairs.append((v, w, A, Bq, Cq, D, dp, r2, p, rel))
    return dict(pairs=pairs, ntested=m, n=n, a=a, b=b, c=c)
