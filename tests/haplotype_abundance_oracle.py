"""Haplotype abundance restated in numpy (restatement choice U18), for the tests.

Independent of the library's masks, class table and EM kernels: B and M come from linkage_oracle.carry_and_clean on the
[R, L] state array, the compatibility sets are dense boolean products, and the EM is the textbook update over the distinct
sets (classes) with numpy sums.
"""
import numpy as np

import linkage_oracle as lo

TOL = 1e-10
MAX_ITER = 10000


def pattern_bits(patterns, V):
    """[H, ceil(V/32)] uint32 phasing patterns -> [H, V] bool (bits >= V ignored)"""
    P = np.asarray(patterns, dtype=np.uint32)
    H = P.shape[0]
    out = np.zeros((H, V), dtype=bool)
    for v in range(V):
        out[:, v] = (P[:, v >> 5] >> np.uint32(v & 31)) & 1
    return out


def compat_sets(B, M, P):
    """S[r, h]: read r agrees with pattern h at every key where it is clean.  B, M: [R, V] bool; P: [H, V] bool."""
    R, H = B.shape[0], P.shape[0]
    if H == 0:
        return np.zeros((R, 0), dtype=bool)
    if B.shape[1] == 0:
        return np.ones((R, H), dtype=bool)
    Pf = P.astype(np.float32)
    S = np.empty((R, H), dtype=bool)
    for r0 in range(0, R, 65536):                      # mismatches = (M & B) . (1 - P) + (M & ~B) . P, exact in float32
        b, m = B[r0: r0 + 65536], M[r0: r0 + 65536]
        mis = (m & b).astype(np.float32) @ (1.0 - Pf).T + (m & ~b).astype(np.float32) @ Pf.T
        S[r0: r0 + 65536] = mis == 0
    return S


def em(classes, counts, tol=TOL, max_iter=MAX_ITER):
    """EM over the classes ([C, H] bool sets, [C] read counts) -> (pi, iterations, converged, log-likelihood)"""
    classes = np.asarray(classes, dtype=bool)
    n = np.asarray(counts, dtype=np.float64)
    H = classes.shape[1]
    N = n.sum()
    pi = np.full(H, 1.0 / H) if H else np.zeros(0)
    if H == 0 or N == 0:
        return pi, 0, True, 0.0
    Sf = classes.astype(np.float64)
    it, conv = 0, False
    while it < max_iter:
        d = Sf @ pi
        nxt = pi * ((n / d) @ Sf) / N
        it += 1
        diff = np.abs(nxt - pi).max()
        pi = nxt
        if diff < tol:
            conv = True
            break
    return pi, it, conv, float((n * np.log(Sf @ pi)).sum())


def kkt_gradient(classes, counts, pi):
    """(1/N) sum_c n_c [h in S_c] / sum_{S_c} pi: <= 1 for every h at the MLE, = 1 where pi_h > 0"""
    Sf = np.asarray(classes, dtype=np.float64)
    n = np.asarray(counts, dtype=np.float64)
    return ((n / (Sf @ pi)) @ Sf) / n.sum()


def abundance_from_sets(S, tol=TOL, max_iter=MAX_ITER):
    """All of U18 from the per-read sets S [R, H] bool."""
    S = np.asarray(S, dtype=bool)
    R, H = S.shape
    k = S.sum(axis=1)
    incompatible = k == 0
    uninformative = (k == H) & (H >= 2) & ~incompatible
    used = ~incompatible & ~uninformative
    unique = used & (k == 1)
    if used.any():
        classes, counts = np.unique(S[used], axis=0, return_counts=True)
    else:
        classes, counts = np.zeros((0, H), dtype=bool), np.zeros(0, dtype=np.int64)
    pi, it, conv, ll = em(classes, counts, tol, max_iter)
    return dict(
        unique_reads=S[unique].sum(axis=0).astype(np.int64),
        compatible_reads=S.sum(axis=0).astype(np.int64),
        em_frequency=pi,
        counters=dict(unique=int(unique.sum()), ambiguous=int((used & (k > 1)).sum()), uninformative=int(uninformative.sum()),
                      incompatible=int(incompatible.sum())),
        reads_used=int(used.sum()), iterations=it, converged=conv, log_likelihood=ll, used=used, S=S,
        classes=classes, class_counts=counts)


def abundance(states, keys, patterns, tol=TOL, max_iter=MAX_ITER):
    """U18 for the reads [R, L] (states), the pooled phasing keys and the [H, ceil(V/32)] uint32 patterns"""
    B, M = lo.carry_and_clean(states, keys)
    return abundance_from_sets(compat_sets(B, M, pattern_bits(patterns, len(keys))), tol, max_iter)
