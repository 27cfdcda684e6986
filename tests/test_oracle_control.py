"""control_oracle (restatement choice U22) on the CPU: its tails against scipy's two-sample Fisher test on small tables, the
edges of the rule (no control coverage, k0 = 0, equal frequencies), and the row rules: the union of control calls and listed
variants, model_call, --drm-only and the order."""
import itertools

import numpy as np
import pytest
from scipy.stats import fisher_exact

import control_oracle as co
import hypergeom_reference as ref

AAA, AAC, CCC, TTT = 0, 1, 21, 63


def _hist(L, cols):
    h = np.zeros((L, 64), dtype=np.uint32)
    for s, bins in cols.items():
        for c, k in bins.items():
            h[s, c] = k
    return h


@pytest.mark.parametrize("k,n,k0,n0", [t for t in itertools.product((1, 2, 5), (5, 9), (0, 1, 4), (4, 7, 30)) if t[0] <= t[1] and t[2] <= t[3]])
def test_tail_against_scipy(k, n, k0, n0):
    want = fisher_exact([[k, n - k], [k0, n0 - k0]], alternative="greater")[1]
    assert abs(float(co.pvalue(k, n, k0, n0)) - want) <= 1e-12 * max(want, 1e-300)


def test_no_control_coverage_gives_one_and_is_counted():
    L, genes = 9, [(1, 10)]
    smp = _hist(L, {0: {AAA: 900, CCC: 100}, 3: {AAA: 900, CCC: 100}})
    ctl = _hist(L, {0: {AAA: 1000}})
    recs, unc = co.control(smp, ctl, L, genes, listed=[(0, 3, CCC)])
    assert unc == 1                                          # column 3 is covered by the sample only; column 6 by neither
    by_col = {r["col"]: r for r in recs}
    assert by_col[3]["pvalue"] == 1 and by_col[3]["called"] == 0 and by_col[3]["listed"] == 1
    assert by_col[0]["called"] == 1 and by_col[0]["listed"] == 0 and by_col[0]["control_count"] == 0


def test_equal_frequencies_are_not_enriched():
    for k, n in ((10, 1000), (1, 7), (250, 500), (3, 3)):
        assert co.pvalue(k, n, k, n) >= 0.5
        assert co.pvalue(k, n, 2 * k, 2 * n) >= 0.5


def test_k0_zero_against_scipy():
    for k, n, n0 in ((3, 100, 100), (12, 6000, 6000), (1, 2, 1)):
        want = fisher_exact([[k, n - k], [0, n0]], alternative="greater")[1]
        assert abs(float(co.pvalue(k, n, 0, n0)) - want) <= 1e-12 * want


def test_reference_codon_is_the_samples_major():
    """the control's own major codon does not matter: a control dominated by CCC still tests the sample's CCC minority"""
    L, genes = 3, [(1, 4)]
    smp = _hist(L, {0: {AAA: 600, CCC: 400}})
    ctl = _hist(L, {0: {CCC: 900, AAA: 100}})
    recs, _ = co.control(smp, ctl, L, genes, listed=[(0, 0, CCC)])
    assert [(r["ref_codon"], r["codon"], r["called"]) for r in recs] == [(AAA, CCC, 0)]
    assert recs[0]["pvalue"] > 0.5
    recs, _ = co.control(smp, ctl, L, genes, refseq="CCC", listed=[(0, 0, AAA)])
    assert [(r["ref_codon"], r["codon"], r["called"]) for r in recs] == [(CCC, AAA, 1)]


def test_row_rules():
    """union of the control calls and the listed variants, model_call from the list, --drm-only, (gene, col, codon) order"""
    L, genes = 12, [(1, 13), (4, 10)]
    smp = _hist(L, {0: {AAA: 900, CCC: 100}, 3: {AAA: 990, AAC: 10, TTT: 60}, 6: {AAA: 950, CCC: 50}})
    ctl = _hist(L, {0: {AAA: 900, CCC: 100}, 3: {AAA: 1000}, 6: {AAA: 990, CCC: 10}})
    listed = [(0, 0, CCC), (0, 3, AAC), (1, 3, AAC)]
    recs, _ = co.control(smp, ctl, L, genes, listed=listed)
    keys = [(r["gene"], r["col"], r["codon"]) for r in recs]
    assert keys == sorted(keys)
    assert set(listed) <= set(keys)
    got = {(r["gene"], r["col"], r["codon"]): (r["called"], r["listed"]) for r in recs}
    assert got[(0, 0, CCC)] == (0, 1)                        # the hot spot: as frequent in the control
    assert got[(0, 3, TTT)] == (1, 0) and got[(1, 3, TTT)] == (1, 0)   # a control call that K2 did not list
    assert got[(0, 6, CCC)] == (1, 0)
    rows = co.report_rows(recs)
    assert [(r["control_call"], r["model_call"]) for r in rows] == [(bool(r["called"]), bool(r["listed"])) for r in recs]
    drm = lambda r: ["drugX"] if r["col"] == 3 else []
    rows = co.report_rows(recs, drm, drm_only=True)
    assert {r["col"] for r in rows} == {3} and all(r["known_drm"] == "drugX" for r in rows)


def test_percentage_filters_apply_to_control_calls_only():
    L, genes = 3, [(1, 4)]
    smp = _hist(L, {0: {AAA: 900, CCC: 100}})
    ctl = _hist(L, {0: {AAA: 1000}})
    assert [r["called"] for r in co.control(smp, ctl, L, genes)[0]] == [1]
    assert co.control(smp, ctl, L, genes, min_perc=10.0)[0] == []        # strict: 10 % is not above 10 %
    assert co.control(smp, ctl, L, genes, max_perc=10.0)[0] == []
    recs, _ = co.control(smp, ctl, L, genes, min_perc=10.0, listed=[(0, 0, CCC)])
    assert [(r["called"], r["listed"]) for r in recs] == [(0, 1)]


def test_histogram_counts_clean_codons_at_starts():
    st = np.array([[0, 0, 1, 2, 3, 0], [0, 5, 1, 2, 3, 0], [7, 7, 7, 2, 3, 8 | 0], [0, 0, 1, 2, 3, 0]], dtype=np.uint8)
    h = co.histogram(st, 6, [(1, 7)])
    assert h[0, 1] == 2 and h[0].sum() == 2                  # 'N' and uncovered reads do not count
    assert h[3].sum() == 4 and h[3, 16 * 2 + 4 * 3] == 4     # the insertion-follows bit is not part of the state
    assert h[1].sum() == 0 and h[2].sum() == 0


def test_reference_module_agrees_with_its_own_tails():
    """p is the upper tail of the hypergeometric with the table's margins"""
    k, n, k0, n0 = 7, 40, 3, 60
    assert abs(co.pvalue(k, n, k0, n0) - ref.upper(k, k + k0, n - k + n0 - k0, n)) < ref.mp.mpf("1e-50")
