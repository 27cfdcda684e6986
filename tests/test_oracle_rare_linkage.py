"""The restatement of sub-threshold variant linkage (rare_linkage_oracle.py, restatement choice U21) at its edges, on hand-built
histograms and read matrices, and its known answer: a 0.25 % minor strain in 6000 reads that K2 does not call is found as one
linked group."""
import numpy as np

import hypergeom_reference as ref
import rare_linkage_oracle as ro
from minorseq_b200.synth import SynthConfig, make_tables, synth_states

AAA, CAA, GAA, TAA, ACA = 0, 16, 32, 48, 4
N = 1000


def hist(L, cols):
    h = np.zeros((L, 64), dtype=np.uint32)
    for s, bins in cols.items():
        for c, k in bins.items():
            h[s, c] = k
    return h


def column(k, codon=CAA):
    return {AAA: N - k, codon: k}


def p_of(k):
    P = ref.codon_error_table(5e-4, 3e-3)
    return ref.k2_pvalue(k, N, ref.expected_count(N, P[1]))


def keys_of(cands):
    return [(c["col"], c["codon"]) for c in cands]


def test_min_reads_is_inclusive():
    h = hist(9, {0: column(8)})
    for mr, want in ((8, [(0, CAA)]), (9, [])):
        got, _ = ro.candidates(h, 9, [(1, 10)], min_reads=mr)
        assert keys_of(got) == want, mr


def test_candidate_bound_is_strict():
    """p(8 of 1000, e = 1) = 0.0193: a candidate just above the bound, not just below it; called at p * ntests < alpha"""
    h = hist(9, {0: column(8)})
    p = float(p_of(8))
    for ca, want in ((p * (1 + 1e-9), [(0, CAA)]), (p * (1 - 1e-9), [])):
        got, _ = ro.candidates(h, 9, [(1, 10)], candidate_alpha=ca)
        assert keys_of(got) == want, ca
    # 3 positions: p * 3 = 0.058 >= alpha = 0.05, not called: a candidate; alpha 0.06: called, so no candidate
    assert keys_of(ro.candidates(h, 9, [(1, 10)], alpha=0.05)[0]) == [(0, CAA)]
    assert ro.candidates(h, 9, [(1, 10)], alpha=0.06)[0] == []


def test_called_in_one_gene_is_no_candidate_in_another():
    """the same column in a one-codon gene (ntests 1: called at alpha 0.05) and in a 3-codon gene (not called there)"""
    h = hist(9, {3: column(8)})
    assert keys_of(ro.candidates(h, 9, [(1, 10)], alpha=0.05)[0]) == [(3, CAA)]
    assert ro.candidates(h, 9, [(1, 10), (4, 7)], alpha=0.05)[0] == []
    # two genes that both leave it uncalled: one record, the gene with the smallest p, the lowest index on ties
    got, _ = ro.candidates(h, 9, [(1, 10), (4, 10)], alpha=0.01)
    assert keys_of(got) == [(3, CAA)] and got[0]["gene"] == 0


def test_truncation_at_the_cap():
    cols = {0: column(5), 3: column(9), 6: column(6), 9: column(8), 12: column(7)}
    h = hist(15, cols)
    got, dropped = ro.candidates(h, 15, [(1, 16)], max_candidates=3)
    assert dropped == 1 and keys_of(got) == [(3, CAA), (9, CAA), (12, CAA)]       # the 3 smallest p of 4, by column
    got, dropped = ro.candidates(h, 15, [(1, 16)])
    assert dropped == 0 and len(got) == 4                                          # k = 5: p = 0.109 >= 0.1


def test_truncation_ties_by_column_and_codon():
    h = hist(9, {0: {AAA: N - 16, CAA: 8, GAA: 8}, 3: column(8)})
    got, dropped = ro.candidates(h, 9, [(1, 10)], max_candidates=2, alpha=1e-9)
    assert dropped == 1 and keys_of(got) == [(0, CAA), (0, GAA)]


def _reads(tables, spacing, L=60):
    """B, M, cols: key 2i at column 6i, key 2i+1 `spacing` columns on; the pair's reads (a both, b v only, c w only, d neither)
    are clean at its two keys only"""
    rowsB, rowsM = [], []
    V = 2 * len(tables)
    for i, (a, b, c, d) in enumerate(tables):
        for cv, cw, k in ((1, 1, a), (1, 0, b), (0, 1, c), (0, 0, d)):
            for _ in range(k):
                rb, rm = np.zeros(V, bool), np.zeros(V, bool)
                rm[2 * i] = rm[2 * i + 1] = True
                rb[2 * i], rb[2 * i + 1] = bool(cv), bool(cw)
                rowsB.append(rb)
                rowsM.append(rm)
    cols = []
    for i in range(len(tables)):
        cols += [6 * i, 6 * i + spacing]
    return np.array(rowsB), np.array(rowsM), cols


def test_spacing_and_min_reads_of_a_pair():
    t = (5, 0, 0, 5)                            # n = 10, p = 1 / C(10, 5)
    for spacing, tested in ((3, 1), (2, 0)):
        B, M, cols = _reads([t], spacing)
        got, m = ro.pairs(B, M, cols, fc=1)
        assert m == tested and len(got) == tested, spacing
    B, M, cols = _reads([(5, 0, 0, 4)], 3)       # n = 9
    assert ro.pairs(B, M, cols, fc=1) == ([], 0)
    B, M, cols = _reads([(5, 0, 0, 4)], 3)
    assert ro.pairs(B, M, cols, fc=1, min_reads=9)[1] == 1


def test_only_pairs_with_a_candidate_are_tested():
    B, M, cols = _reads([(5, 0, 0, 5), (5, 0, 0, 5)], 3)     # keys 0..3; the pairs (0, 1) and (2, 3) have informative reads
    assert ro.pairs(B, M, cols, fc=4)[1] == 0                  # no candidate
    assert ro.pairs(B, M, cols, fc=2)[1] == 1                  # (2, 3) only: (0, 1) is a pair of called keys
    got, m = ro.pairs(B, M, cols, fc=0)
    assert m == 2 and [p[:2] for p in got] == [(0, 1), (2, 3)]


def test_groups_ignore_called_edges():
    pairs = [(0, 2), (0, 3), (2, 4), (5, 6), (4, 7)]
    assert ro.groups([p + (0,) * 7 for p in pairs], fc=2, V=8) == [[2, 4, 7], [5, 6]]


def test_detects_a_quarter_percent_strain():
    """SynthConfig seed 3: K2 calls none of the minor strain's four codons in 6000 reads; they form the one linked group"""
    L = 3000
    t = make_tables(SynthConfig(L=L, seed=3, minor_fracs=(0.0025,), variants_per_minor=(4, 4)))
    st = synth_states(t, 0, 6000)
    codon = np.zeros((L, 64), dtype=np.uint32)
    s3 = st[:, :L - L % 3].reshape(6000, -1, 3) & 7
    clean = (s3 < 4).all(axis=2)
    code = (16 * s3[:, :, 0].astype(np.int64) + 4 * s3[:, :, 1] + s3[:, :, 2])
    for j in range(s3.shape[1]):
        codon[3 * j] = np.bincount(code[clean[:, j], j], minlength=64)
    truth = sorted((c, k) for (_, c, k) in t.truth)
    res = ro.rare_linkage(st, codon, L, [(1, L + 1)], [])
    assert set(truth) <= set(res["keys"])             # candidates: every planted codon is left uncalled by K2
    assert [[res["keys"][i] for i in g] for g in res["groups"]] == [truth]
    assert res["carriers"][0] > 0 and res["informative"][0] > res["carriers"][0]
