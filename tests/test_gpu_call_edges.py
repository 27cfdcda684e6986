"""K2 (call_kernel) at its edges, against the mpmath reference in hypergeom_reference.py rather than the oracle.

Codon histograms are written straight into the handle's count tensor, so every column is exactly the one a case needs:
alpha straddling p * ntests by 1e-10, codons at or below their expected count, coverage 1 and 2, k = n, e = 0, a bin of
2^31, ties for the major codon, reference sequences with N, lowercase or shorter than L, the strict percentage filters,
1024 / 1025 / 63-per-column calls, repeated calls, and genes that are short, run past L or overlap.  Every field of every
call is compared; p-values to 1e-12 relative (both below 1e-290 when the reference is below 1e-300).

Limit: K2 sums a column's 64 bins in uint32; columns of 2^32 reads or more are out of range and not tested.
"""
import mpmath as mp
import numpy as np
import pytest

import hypergeom_reference as ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from minorseq_b200 import Handle, Juliet  # noqa: E402

RTOL = 1e-12
MARGIN = 5e-11          # no codon of a case may sit closer than this (relative) to its threshold, bar the straddled ones
DEFAULTS = dict(substitution_rate=5e-4, deletion_rate=3e-3, alpha=0.01, min_perc=None, max_perc=None, region=None)


def codon_of(s):
    return 16 * "ACGT".index(s[0].upper()) + 4 * "ACGT".index(s[1].upper()) + "ACGT".index(s[2].upper())


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def histogram(L, cols):
    """cols: {start column: {codon: count}} -> [L, 64] uint32"""
    h = np.zeros((L, 64), dtype=np.uint32)
    for s, bins in cols.items():
        for c, k in bins.items():
            h[s, c] = k
    return h


_PCACHE = {}


def pvalue(k, n, e):
    if (k, n, e) not in _PCACHE:
        _PCACHE[(k, n, e)] = ref.k2_pvalue(k, n, e)
    return _PCACHE[(k, n, e)]


def decide(p, ntests, alpha):
    """called iff p * ntests < alpha, from the reference p; refuses a case that sits too close to its threshold to be decided
    by a 1e-12 p-value, except p within 1e-17 of 1 (the kernel's 1 - tail is then exactly 1.0)"""
    with mp.workdps(ref.DPS):
        x = p * ntests
        if 1 - p < mp.mpf("1e-17"):
            return 1.0 * ntests < alpha
        assert abs(x / alpha - 1) > MARGIN, ("case too close to its threshold", mp.nstr(p, 20), ntests, alpha)
        return x < alpha


def k2_reference(codon, L, genes, refseq=None, substitution_rate=5e-4, deletion_rate=3e-3, alpha=0.01, min_perc=None,
                 max_perc=None, region=None):
    """juliet's codon test restated: genes in order, codons of a gene in order, Bonferroni over the gene's tested codons"""
    P = ref.codon_error_table(substitution_rate, deletion_rate)
    lo, hi = 0, L
    if region and region[1] > region[0]:
        lo, hi = max(0, region[0] - 1), min(L, region[1] - 1)
    reflen = min(len(refseq), L) if refseq else 0
    out = []
    for g, (gb1, ge1) in enumerate(genes):
        gb, ge = gb1 - 1, min(ge1 - 1, L)
        pos = [(ci, s) for ci, s in enumerate(range(gb, ge - 2, 3)) if s >= lo and s + 3 <= hi and s >= 0]
        ntests = len(pos)
        for ci, s in pos:
            h = [int(x) for x in codon[s]]
            n = sum(h)
            if n == 0:
                continue
            rc = -1
            if s + 3 <= reflen and all(ch in "ACGTacgt" for ch in refseq[s:s + 3]):
                rc = codon_of(refseq[s:s + 3])
            if rc < 0:
                rc = max(range(64), key=lambda c: (h[c], -c))
            for c in range(64):
                k = h[c]
                if c == rc or k == 0:
                    continue
                e = ref.expected_count(n, P[ref.mismatches(rc, c)])
                if k <= e and 0.5 * ntests >= alpha:
                    continue
                p = pvalue(k, n, e)
                if not decide(p, ntests, alpha):
                    continue
                perc = 100.0 * k / n
                if min_perc is not None and not perc > min_perc:
                    continue
                if max_perc is not None and not perc < max_perc:
                    continue
                out.append(dict(gene=g, codon_index=ci, col=s, ref_codon=rc, codon=c, count=k, coverage=n, expected=e, ntests=ntests,
                                pvalue=p))
    out.sort(key=lambda v: (v["gene"], v["col"], v["codon"]))
    return out


def gpu_call(hd, codon, L, genes, refseq=None, **kw):
    prm = dict(DEFAULTS, **kw)
    j = Juliet(L, genes, refseq=refseq, handle=hd, **prm)
    j.counts_tensor()[L * 8:] = torch.from_numpy(codon.reshape(-1).view(np.int32)).cuda()
    torch.cuda.synchronize()
    return j, j.call()


def assert_calls(got, want, what=""):
    key = lambda v: (v["gene"], v["col"], v["codon"])
    got_keys = [(v.gene, v.col, v.codon) for v in got]
    assert got_keys == [key(v) for v in want], (what, sorted(set(got_keys) ^ set(map(key, want)))[:10])
    for g, w in zip(got, want):
        for f in ("gene", "codon_index", "col", "ref_codon", "codon", "count", "coverage", "expected", "ntests"):
            assert getattr(g, f) == w[f], (what, f, getattr(g, f), w[f], key(w))
        if w["pvalue"] > mp.mpf("1e-300"):
            assert ref.rel_err(g.pvalue, w["pvalue"]) <= RTOL, (what, key(w), g.pvalue, mp.nstr(w["pvalue"], 20))
        else:
            assert g.pvalue < 1e-290, (what, key(w), g.pvalue)


def check(hd, codon, L, genes, refseq=None, **kw):
    _, got = gpu_call(hd, codon, L, genes, refseq=refseq, **kw)
    want = k2_reference(codon, L, genes, refseq=refseq, **dict(DEFAULTS, **kw))
    assert_calls(got, want, kw)
    return got


# codons as 16 * b0 + 4 * b1 + b2 over ACGT; from AAA: 1 mismatch AAC AAG AAT ACA AGA CAA TAA, 2 CCA ACC AGG, 3 CCC TTT
AAA, AAC, AAG, AAT, ACA, AGA, CAA, TAA, CCA, ACC, AGG, CCC, TTT = 0, 1, 2, 3, 4, 8, 16, 48, 20, 5, 10, 21, 63


# ----------------------------------------------------------------------------------------------------- threshold straddle
def straddle_columns():
    """(n, k, nm) -> one column each: major AAA at n - k, the minor codon k times with nm mismatches.  p = 1/2 exactly at
    k = e + 1 (the tail stops early there), p ~ 1e-2 .. 1e-12, and deep tails near 1e-200."""
    return [(10_000, 3, 1), (10_000, 10, 1), (1_000_000, 316, 1), (100_000, 130, 2), (10_000_000, 3880, 1), (3000, 2, 3)]


MINOR = {1: AAC, 2: CCA, 3: CCC}


@pytest.mark.parametrize("case", range(6))
def test_threshold_straddle(hd, case):
    n, k, nm = straddle_columns()[case]
    L, genes = 30, [(1, 31)]                                  # 10 codons: ntests = 10
    minor = MINOR[nm]
    assert ref.mismatches(AAA, minor) == nm
    codon = histogram(L, {9: {AAA: n - k, minor: k}, 0: {AAA: 500}})
    P = ref.codon_error_table(5e-4, 3e-3)
    e = ref.expected_count(n, P[nm])
    p = pvalue(k, n, e)
    if case == 0:
        assert k == e + 1 and abs(p - 0.5) < mp.mpf("1e-50")
    if case == 4:
        assert mp.mpf("1e-260") < p < mp.mpf("1e-150")
    for side, f in (("above", 1 + 1e-10), ("below", 1 - 1e-10)):
        alpha = float(p * 10 * f)
        got = check(hd, codon, L, genes, alpha=alpha)
        assert ((9, minor) in {(v.col, v.codon) for v in got}) == (side == "above"), (side, alpha, mp.nstr(p, 17))


# ---------------------------------------------------------------------------------------------------------- lower side
@pytest.mark.parametrize("alpha", [0.6, 1.0])
def test_codons_at_or_below_expected_with_large_alpha(hd, alpha):
    """A region of one codon (ntests = 1) with alpha above ntests / 2 makes K2 test codons seen no more often than expected.
    Their tail holds the mode; summed from k = 1 its first term underflowed and p came out 0, so a codon seen once in 100 000
    reads with 2 683 expected was called.  Now such codons get p ~ 1 and only the reference's calls come back."""
    L, genes, n = 30, [(1, 31)], 100_000
    minors = {AAC: 1, AAG: 2, ACA: 1000, CAA: 2600, TAA: 2682, AAT: 2683, AGA: 2684, CCA: 1, ACC: 50, AGG: 99, CCC: 1, TTT: 2}
    codon = histogram(L, {6: {AAA: n - sum(minors.values()), **minors}})
    kw = dict(substitution_rate=0.1, alpha=alpha, region=(7, 10))
    got = check(hd, codon, L, genes, **kw)
    P = ref.codon_error_table(0.1, 3e-3)
    called = {v.codon for v in got}
    assert all(v.ntests == 1 for v in got)
    assert {AAC, AAG, ACA, CCA} & called == set()           # 1, 2, 1000 seen with 2683 expected; 1 seen with 100 expected
    for c in (AAC, AAG, ACA, CCA):
        e = ref.expected_count(n, P[ref.mismatches(AAA, c)])
        assert 1 - pvalue(minors[c], n, e) < mp.mpf("1e-17")


# ------------------------------------------------------------------------------------------------------ coverage extremes
def test_coverage_extremes(hd):
    L, genes = 36, [(1, 37)]
    cols = {0: {CCC: 1},                                     # n = 1, the reference codon absent: k = n
            3: {CCC: 1, TTT: 1},                             # n = 2, one each
            6: {AAA: 1, AAC: 1},
            9: {CCC: 30},                                    # k = n = 30
            12: {CCC: 1000},                                 # k = n = 1000: p below 1e-300
            15: {AAA: 2, ACA: 2, TTT: 1},
            18: {CCC: 2 ** 31},                              # one bin of 2^31, reference absent
            21: {AAA: 2 ** 31, TTT: 2 ** 30},                # n = 3 * 2^30
            24: {AAA: 2 ** 31}}                              # one bin of 2^31, the reference itself
    refseq = "AAA" * 12
    codon = histogram(L, cols)
    for alpha in (0.01, 6.5, 11.9):                         # above ntests / 2 = 6: codons at their expectation are tested
        check(hd, codon, L, genes, refseq=refseq, alpha=alpha)
        check(hd, codon, L, genes, alpha=alpha)
    # e = 0: both error rates 0, every non-reference codon is unexpected
    got = check(hd, codon, L, genes, refseq=refseq, substitution_rate=0.0, deletion_rate=0.0, alpha=6.5)
    assert got and all(v.expected == 0 for v in got)
    got = check(hd, codon, L, genes, refseq=refseq, substitution_rate=0.0, deletion_rate=0.0)
    assert (0, CCC) not in {(v.col, v.codon) for v in got}      # p = 1/2 for a single read


# ----------------------------------------------------------------------------------------------------------- major codon
def test_major_codon_ties_and_reference_sequences(hd):
    L, genes = 45, [(1, 46)]
    cols = {0: {c: 1000 for c in range(64)},                 # all 64 tied: codon 0 is the reference, the other 63 called
            3: {5: 1000, 37: 1000, 2: 10},                   # c vs c + 32: the lane / half split of the reduction
            6: {37: 1000, 5: 999, 60: 1000},                 # the tie is in the upper half only
            9: {35: 700, 52: 700, 63: 700},                  # three-way tie across lanes of the upper half
            12: {17: 500, 18: 500},
            15: {40: 900, 41: 10},
            18: {CCC: 900, AAA: 300},
            21: {TTT: 400, AAA: 400}}
    codon = histogram(L, cols)
    got = check(hd, codon, L, genes)
    assert sum(1 for v in got if v.col == 0) == 63 and all(v.ref_codon == 0 for v in got if v.col == 0)
    assert {v.ref_codon for v in got if v.col == 3} == {5} and {v.ref_codon for v in got if v.col == 6} == {37}
    assert {v.ref_codon for v in got if v.col == 9} == {35}
    for refseq in ("AAANNNAAAcccaaaAAAaaaTTTAAAAAAAAAAAAAAAAAAAAA",   # N: the major codon; lowercase is a base
                   "ACGTACGTACGTACGTACG",                            # shorter than L: past its end, the major codon
                   "AAA" * 15 + "TTTTTT",                            # longer than L
                   "aCgNNNtTtAAAGGGTGTCCCAAAAAA"):
        check(hd, codon, L, genes, refseq=refseq)


# ----------------------------------------------------------------------------------------------------- percentage filters
def test_percentage_filters_are_strict(hd):
    L, genes = 30, [(1, 31)]
    codon = histogram(L, {0: {AAA: 980, CCC: 20}, 3: {AAA: 2, CCC: 1}, 6: {AAA: 900, TTT: 100}, 9: {AAA: 500, CCC: 500}})
    for mn, mx in ((2.0, None), (1.9999999999999998, None), (None, 2.0), (None, 2.0000000000000004), (2.0, 10.0), (None, 100.0 / 3),
                   (100.0 / 3, None), (10.0, 50.0), (None, 50.0000000001), (0.0, 100.0)):
        got = check(hd, codon, L, genes, min_perc=mn, max_perc=mx)
        calls = {(v.col, v.codon) for v in got}
        if mn == 2.0:
            assert (0, CCC) not in calls
        if mx == 2.0:
            assert (0, CCC) not in calls
        if mn == 1.9999999999999998 or mx == 2.0000000000000004:
            assert (0, CCC) in calls


# ---------------------------------------------------------------------------------------------------------- call counts
@pytest.mark.parametrize("ncalls", [1023, 1024, 1025, 1260])
def test_call_counts_around_the_pinned_stage(hd, ncalls):
    """The first 1024 calls come back with the count in one pinned copy; more take a second download."""
    full, rest = divmod(ncalls, 63)
    L = 3 * (full + 1)
    cols = {3 * i: {c: 1000 for c in range(64)} for i in range(full)}
    cols[3 * full] = {AAA: 1000, **{c: 1000 for c in range(1, rest + 1)}}
    codon = histogram(L, cols)
    got = check(hd, codon, L, [(1, L + 1)])
    assert len(got) == ncalls


# ------------------------------------------------------------------------------------------------------- repeated calls
def test_repeated_calls_with_positions_of_equal_size(hd):
    """The position table is uploaded only when it changed; two calls whose tables have the same byte size but different
    contents (another reference codon, another gene frame) must each use their own."""
    L = 30
    codon = histogram(L, {s: {AAA: 900, CCC: 100, TTT: 50} for s in range(0, 28)})
    j, _ = gpu_call(hd, codon, L, [(1, 31)])
    for refseq in (None, "CCC" * 10, "TTT" * 10, None):
        j.refseq = refseq
        assert_calls(j.call(), k2_reference(codon, L, [(1, 31)], refseq=refseq), refseq)
    for genes in ([(1, 28)], [(2, 29)], [(3, 30)], [(1, 28)]):       # 9 codons each, shifted frames
        check(hd, codon, L, genes)


# ------------------------------------------------------------------------------------------------------------------ genes
def test_genes_short_past_the_end_and_overlapping(hd):
    L = 30
    codon = histogram(L, {s: {AAA: 5000, CCC: 8 + s, TTT: 3} for s in range(0, 28)})
    got = check(hd, codon, L, [(5, 7), (10, 11), (1, 100), (4, 19), (2, 30)])
    assert {v.gene for v in got} <= {2, 3, 4} and {v.ntests for v in got if v.gene == 3} == {5}
    assert check(hd, codon, L, [(5, 7)]) == []                       # a gene shorter than a codon: nothing tested
    # the same column under two overlapping genes with 10 and 5 tests, alpha between p * 5 and p * 10: called in the second only
    n, k = 5020, 17
    e = ref.expected_count(n, ref.codon_error_table(5e-4, 3e-3)[3])
    alpha = float(pvalue(k, n, e) * 7.5)
    got = check(hd, codon, L, [(1, 31), (10, 25)], alpha=alpha)
    assert {(v.gene, v.codon_index, v.ntests) for v in got if v.col == 9 and v.codon == CCC} == {(1, 0, 5)}
