"""numpy restatement of in-frame indels in phasing (restatement choice U20, DESIGN.md "Phasing indels"), for the tests.

From the column states [R, L] (bits 0-2: 0-3 A/C/G/T, 4 '-', 5 N, 6-7 not spanned), the insertion events (read, col, off,
len, pool) and the three key lists it gives B and M for every key, the damage flags, and the haplotypes (patterns, juliet's
order, counts, hap_id, the six read categories).  Independent of the library: no bit-slicing, no stream, no exclusion mask --
each read's columns are judged one key at a time.  Linkage and abundance are linkage_oracle's and haplotype_abundance_oracle's
rules fed with these B and M.
"""
import numpy as np

import haplotype_abundance_oracle as hao
import linkage_oracle as lo

GAP, HET, PARTIAL = 1, 2, 4


def first_events(events, R, read0=0):
    """{(local read, c): upper-cased string, or None when the read's first event at c is not in frame or not all A/C/G/T}"""
    out = {}
    if events is None:
        return out
    read, col, off, ln, pool = events
    for i in range(len(read)):
        key = (int(read[i]) - read0, int(col[i]))
        if key in out or not 0 <= key[0] < R:
            continue
        x = bytes(pool[int(off[i]): int(off[i]) + int(ln[i])]).decode("latin-1")
        ok = len(x) >= 3 and len(x) % 3 == 0 and all(ch in "ACGTacgt" for ch in x)
        out[key] = x.upper() if ok else None
    return out


def _category(s):
    """[..] states -> flags of the non-clean ones"""
    return np.where(s == 4, GAP, np.where(s == 5, HET, np.where(s > 5, PARTIAL, 0))).astype(np.uint8)


def bits(states, sub_keys, del_cols, ins_keys, events=None, read0=0):
    """-> B, M [R, K] bool and flags [R] uint8 (GAP | HET | PARTIAL) for the keys sub_keys [(col, codon)], then the deletion
    start columns, then the insertion keys [(c, x)]"""
    st = np.asarray(states) & 7
    R, L = st.shape
    V, nd, ni = len(sub_keys), len(del_cols), len(ins_keys)
    B = np.zeros((R, V + nd + ni), dtype=bool)
    M = np.zeros((R, V + nd + ni), dtype=bool)
    flags = np.zeros(R, dtype=np.uint8)
    pad = np.concatenate([st, np.full((R, 3), 7, dtype=st.dtype)], axis=1)     # past the reference: not spanned
    # columns of a deletion key the read carries in full: never damage
    exempt = np.zeros((R, L + 3), dtype=bool)
    for k, s in enumerate(del_cols):
        w = pad[:, s: s + 3]
        B[:, V + k] = (w == 4).all(axis=1)
        M[:, V + k] = B[:, V + k] | (w < 4).all(axis=1)
        exempt[:, s: s + 3] |= B[:, V + k][:, None]
        bad = ~M[:, V + k]
        if bad.any():
            flags[bad] |= np.bitwise_or.reduce(_category(w[bad]), axis=1)
    sB, sM = lo.carry_and_clean(st, sub_keys)
    B[:, :V], M[:, :V] = sB, sM
    for v, (col, _) in enumerate(sub_keys):
        w = pad[:, col: col + 3]
        cat = np.where(exempt[:, col: col + 3], 0, _category(w))
        flags |= np.bitwise_or.reduce(cat, axis=1)
    ev = first_events(events, R, read0)
    for i, (c, x) in enumerate(ins_keys):
        w = pad[:, c: c + 2]
        k = V + nd + i
        M[:, k] = (w < 4).all(axis=1)
        B[:, k] = M[:, k] & np.array([ev.get((r, c)) == x for r in range(R)], dtype=bool)
        bad = ~M[:, k]
        if bad.any():
            flags[bad] |= np.bitwise_or.reduce(_category(w[bad]), axis=1)
    return B, M, flags


def words(B):
    """[R, K] bool -> [R, max(1, ceil(K/32))] uint32 patterns, bit k of word k // 32"""
    R, K = B.shape
    out = np.zeros((R, max(1, (K + 31) // 32)), dtype=np.uint32)
    for k in range(K):
        out[:, k >> 5] |= B[:, k].astype(np.uint32) << np.uint32(k & 31)
    return out


def phase(B, flags, min_reads=10):
    """juliet's haplotypes of the undamaged reads: patterns [H, nw] in order (count desc, then ascending words), counts,
    nreported, hap_id (position in the order, -1 damaged) and the six read categories"""
    W = words(B)
    R, nw = W.shape
    ok = flags == 0
    groups = {}
    for r in np.flatnonzero(ok):
        groups.setdefault(tuple(int(x) for x in W[r]), []).append(r)
    order = sorted(groups, key=lambda p: (-len(groups[p]), p))
    hap = np.full(R, -1, dtype=np.int32)
    for h, p in enumerate(order):
        hap[groups[p]] = h
    counts = np.array([len(groups[p]) for p in order], dtype=np.uint64)
    nrep = int((counts >= min_reads).sum())
    ctr = dict(reported=int(counts[:nrep].sum()), insufficient=int(counts[nrep:].sum()), damaged=int((~ok).sum()),
               gaps=int(((flags & GAP) != 0).sum()), heteroduplex=int(((flags & HET) != 0).sum()), partial=int(((flags & PARTIAL) != 0).sum()))
    pats = np.array(order, dtype=np.uint32).reshape(len(order), nw)
    return dict(patterns=pats, counts=counts, nreported=nrep, hap_id=hap, counters=ctr)


def key_columns(sub_keys, del_cols, ins_keys):
    """linkage's column of each key: the codon's start, s for a deletion, c for an insertion"""
    return [k[0] for k in sub_keys] + list(del_cols) + [c for c, _ in ins_keys]


def linkage(B, M, cols, fisher_greater, alpha=0.01, min_reads=lo.MIN_READS):
    """linkage_oracle.linkage's rule on given B and M"""
    Bf, Mf = B.astype(np.float64), M.astype(np.float64)
    n = np.rint(Mf.T @ Mf).astype(np.int64)
    a = np.rint(Bf.T @ Bf).astype(np.int64)
    bm = np.rint(Bf.T @ Mf).astype(np.int64)
    b, c = bm - a, bm.T - a
    K = B.shape[1]
    tested = [(v, w) for v in range(K) for w in range(v + 1, K) if abs(cols[v] - cols[w]) >= lo.MIN_SPACING and n[v, w] >= min_reads]
    m = len(tested)
    pairs = []
    for v, w in tested:
        A, Bq, Cq, N = int(a[v, w]), int(b[v, w]), int(c[v, w]), int(n[v, w])
        D = N - A - Bq - Cq
        pt, pa = lo.tails(A, Bq, Cq, D, fisher_greater)
        if pt * m < alpha:
            rel, p = lo.LINKED, pt
        elif pa * m < alpha:
            rel, p = lo.EXCLUSIVE, pa
        else:
            continue
        dp, r2 = lo.measures(A, Bq, Cq, N)
        pairs.append((v, w, A, Bq, Cq, D, dp, r2, p, rel))
    return dict(pairs=pairs, ntested=m, n=n, a=a, b=b, c=c)


def abundance(B, M, patterns, tol=hao.TOL, max_iter=hao.MAX_ITER):
    """haplotype_abundance_oracle's rule on given B and M"""
    return hao.abundance_from_sets(hao.compat_sets(B, M, hao.pattern_bits(patterns, B.shape[1])), tol, max_iter)
