"""Sub-threshold variant linkage (restatement choice U21) restated in numpy, for the tests.

From a codon histogram [L, 64] and the per-read column states: K2's positions and expected counts as test_gpu_call_edges
restates them, the tails from hypergeom_reference (mpmath), B and M straight off the states (linkage_oracle.carry_and_clean),
the pair tables as dense products, the groups by a plain graph search.  Tails far from every threshold are screened with
scipy first: only the decision matters there, and mpmath would take minutes on a 200 000-read histogram.
"""
import numpy as np
from scipy.stats import hypergeom

import hypergeom_reference as ref
import linkage_oracle as lo

MAX_CANDIDATES = 2048
SCREEN = 4.0        # a scipy tail above SCREEN x the bound cannot be below it


def _codon_of(s):
    return 16 * "ACGT".index(s[0].upper()) + 4 * "ACGT".index(s[1].upper()) + "ACGT".index(s[2].upper())


def _upper_scipy(a, b, c, d):
    return float(hypergeom.sf(a - 1, a + b + c + d, a + c, a + b))


def positions(L, genes, refseq=None, region=None):
    """K2's tested codon starts: (gene, codon_index, col, ref_codon or -1, ntests)"""
    lo_, hi = 0, L
    if region and region[1] > region[0]:
        lo_, hi = max(0, region[0] - 1), min(L, region[1] - 1)
    reflen = min(len(refseq), L) if refseq else 0
    out = []
    for g, (gb1, ge1) in enumerate(genes):
        gb, ge = gb1 - 1, min(ge1 - 1, L)
        pos = [(ci, s) for ci, s in enumerate(range(gb, ge - 2, 3)) if s >= lo_ and s + 3 <= hi and s >= 0]
        for ci, s in pos:
            rc = -1
            if s + 3 <= reflen and all(ch in "ACGTacgt" for ch in refseq[s:s + 3]):
                rc = _codon_of(refseq[s:s + 3])
            out.append((g, ci, s, rc, len(pos)))
    return out


def candidates(codon, L, genes, refseq=None, sub=5e-4, dele=3e-3, alpha=0.01, min_reads=5, candidate_alpha=0.1, region=None,
               max_candidates=MAX_CANDIDATES):
    """-> (candidates ordered by (col, codon), dropped): dicts with gene, codon_index, col, ref_codon, codon, count, coverage,
    expected, ntests, pvalue (mpf)"""
    P = ref.codon_error_table(sub, dele)
    recs = {}
    for g, ci, s, rc, ntests in positions(L, genes, refseq, region):
        h = [int(x) for x in codon[s]]
        n = sum(h)
        if n == 0:
            continue
        if rc < 0:
            rc = max(range(64), key=lambda c: (h[c], -c))
        bound = max(alpha / ntests, candidate_alpha)
        for c in range(64):
            k = h[c]
            if c == rc or k < min_reads:
                continue
            e = ref.expected_count(n, P[ref.mismatches(rc, c)])
            if _upper_scipy(k, n - k, e, n - e) > SCREEN * bound:
                continue
            p = ref.k2_pvalue(k, n, e)
            called = p * ntests < alpha
            if not called and not p < candidate_alpha:
                continue
            recs.setdefault((s, c), []).append((dict(gene=g, codon_index=ci, col=s, ref_codon=rc, codon=c, count=k, coverage=n,
                                                     expected=e, ntests=ntests, pvalue=p), called))
    out = []
    for key in sorted(recs):
        rs = recs[key]
        if any(called for _, called in rs):
            continue
        out.append(min((r for r, _ in rs), key=lambda r: (r["pvalue"], r["gene"])))
    dropped = 0
    if len(out) > max_candidates:
        out.sort(key=lambda r: (r["pvalue"], r["col"], r["codon"]))
        dropped = len(out) - max_candidates
        out = sorted(out[:max_candidates], key=lambda r: (r["col"], r["codon"]))
    return out, dropped


def pairs(B, M, cols, fc, alpha=0.01, min_reads=lo.MIN_READS):
    """linked pairs (v, w, a, b, c, d, d_prime, r2, p) with w >= fc, and m_r"""
    Bf, Mf = B.astype(np.float64), M.astype(np.float64)
    V = B.shape[1]
    if V < 2 or fc >= V:
        return [], 0
    n = np.rint(Mf.T @ Mf[:, fc:]).astype(np.int64)
    a = np.rint(Bf.T @ Bf[:, fc:]).astype(np.int64)
    bm = np.rint(Bf.T @ Mf[:, fc:]).astype(np.int64)           # B_v . M_w
    mb = np.rint(Mf.T @ Bf[:, fc:]).astype(np.int64)           # M_v . B_w
    cols = np.asarray(cols, dtype=np.int64)
    tested = [(v, w) for w in range(fc, V) for v in range(w)
              if abs(cols[v] - cols[w]) >= lo.MIN_SPACING and n[v, w - fc] >= min_reads]
    m = len(tested)
    out = []
    for v, w in sorted(tested):
        A, N = int(a[v, w - fc]), int(n[v, w - fc])
        Bq, Cq = int(bm[v, w - fc]) - A, int(mb[v, w - fc]) - A
        D = N - A - Bq - Cq
        if _upper_scipy(A, Bq, Cq, D) * m > SCREEN * alpha:
            continue
        p = ref.fisher_greater(A, Bq, Cq, D)
        if not p * m < alpha:
            continue
        dp, r2 = ref.linkage_measures(A, Bq, Cq, N)
        out.append((v, w, A, Bq, Cq, D, float(dp), float(r2), p))
    return out, m


def groups(pair_list, fc, V):
    """connected components (>= 2 members) of the candidate-candidate pairs, ordered by their smallest key"""
    adj = {k: set() for k in range(fc, V)}
    for p in pair_list:
        if p[0] >= fc:
            adj[p[0]].add(p[1])
            adj[p[1]].add(p[0])
    seen, out = set(), []
    for k in range(fc, V):
        if k in seen or not adj[k]:
            continue
        comp, stack = set(), [k]
        while stack:
            x = stack.pop()
            if x in comp:
                continue
            comp.add(x)
            stack.extend(adj[x] - comp)
        seen |= comp
        out.append(sorted(comp))
    return out


def support(B, M, group_list):
    """(carriers, informative) per group"""
    car = [int(B[:, g].all(axis=1).sum()) for g in group_list]
    inf = [int(M[:, g].all(axis=1).sum()) for g in group_list]
    return car, inf


def rare_linkage(states, codon, L, genes, called_keys, refseq=None, sub=5e-4, dele=3e-3, alpha=0.01, min_reads=5,
                 candidate_alpha=0.1, link_min_reads=lo.MIN_READS, region=None, max_candidates=MAX_CANDIDATES):
    """The whole of U21 from the histogram and the states; called_keys: the reported (col, codon) calls."""
    cands, dropped = candidates(codon, L, genes, refseq, sub, dele, alpha, min_reads, candidate_alpha, region, max_candidates)
    called = sorted(set(called_keys))
    keys = called + [(c["col"], c["codon"]) for c in cands]
    fc = len(called)
    B, M = lo.carry_and_clean(states, keys)
    pl, m = pairs(B, M, [k[0] for k in keys], fc, alpha, link_min_reads)
    gl = groups(pl, fc, len(keys))
    car, inf = support(B, M, gl)
    return dict(candidates=cands, dropped=dropped, keys=keys, first_candidate=fc, pairs=pl, tested=m, groups=gl, carriers=car,
                informative=inf, B=B, M=M)
