"""ms_control_capture / ms_control_call (Juliet.capture_control, Juliet.control_call) against control_oracle.py: records
exactly, p-values to 1e-9 relative (both below 1e-290 where the reference is below 1e-300).  Generator reads at L = 3000 and
9719 (genes in three frames), crafted histograms at the edges of the rule, and the state rules of the capture."""
import mpmath as mp
import numpy as np
import pytest

import control_oracle as co
import hypergeom_reference as ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from minorseq_b200 import Handle, Juliet, _lib, host_rows, synth_device  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

PVAL_RTOL = 1e-9
AAA, AAC, CAA, CCC, TTT = 0, 1, 16, 21, 63
FIELDS = ("gene", "codon_index", "col", "ref_codon", "codon", "count", "coverage", "control_count", "control_coverage", "ntests",
          "called", "listed")


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def _hist(L, cols):
    h = np.zeros((L, 64), dtype=np.uint32)
    for s, bins in cols.items():
        for c, k in bins.items():
            h[s, c] = k
    return h


def _sync(hd):
    _lib.check(hd.lib.ms_synchronize(hd.h), hd.h)
    torch.cuda.synchronize()


def _write(j, hd, codon):
    _sync(hd)
    j.counts_tensor()[j.L * 8:] = torch.from_numpy(codon.reshape(-1).view(np.int32)).cuda()
    torch.cuda.synchronize()


def _crafted(hd, smp, ctl, L, genes, **kw):
    """a Juliet whose capture holds `ctl` and whose counts hold `smp`"""
    j = Juliet(L, genes, handle=hd, **kw)
    _write(j, hd, ctl)
    j.capture_control()
    _write(j, hd, smp)
    return j


def _listed(j, triples):
    """Variant records for (gene, col, codon) triples, at the gene's codon index"""
    out = []
    for g, s, c in triples:
        v = _lib.Variant()
        v.gene, v.col, v.codon, v.codon_index = g, s, c, (s - (j.genes[g][0] - 1)) // 3
        out.append(v)
    return out


def _check(got, want):
    rows, unc = got.rows, got.uncovered_positions
    want_rows, want_unc = want
    assert unc == want_unc
    assert [(r.gene, r.col, r.codon) for r in rows] == [(w["gene"], w["col"], w["codon"]) for w in want_rows]
    for r, w in zip(rows, want_rows):
        for f in FIELDS:
            assert getattr(r, f) == w[f], (f, getattr(r, f), w)
        if w["pvalue"] > mp.mpf("1e-300"):
            assert ref.rel_err(r.pvalue, w["pvalue"]) <= PVAL_RTOL, (r.pvalue, mp.nstr(w["pvalue"], 17), w)
        else:
            assert r.pvalue < 1e-290, (r.pvalue, w)


def _kw(params):
    return dict(alpha=params.get("alpha", 0.01), min_perc=params.get("min_perc"), max_perc=params.get("max_perc"),
                region=params.get("region"))


# ------------------------------------------------------------------------------------------------------------ generator reads
GENES_9719 = [(1, 9719), (2, 3001), (3, 6002), (4000, 9700)]      # three frames, overlapping


@pytest.mark.parametrize("L,genes,R,refseq,region", [
    (3000, [(1, 3001)], 6001, True, None),
    (3000, [(1, 3001)], 6001, False, None),
    (3000, [(1, 3001), (302, 2999)], 4003, True, (450, 2400)),
    (9719, GENES_9719, 3005, True, None),
    (9719, GENES_9719, 3005, False, (1000, 8000)),
])
def test_generator_reads_against_the_oracle(hd, oracle, L, genes, R, refseq, region):
    t = make_tables(SynthConfig(L=L, seed=41, minor_fracs=(0.05, 0.01), trunc=0.2))
    tc = make_tables(SynthConfig(L=L, seed=41, minor_fracs=(0.05,), trunc=0.2))     # the same reference, one strain fewer
    R0 = R + 1234
    d0 = synth_device(hd, tc, 10 ** 6, R0)          # other reads: noise is a function of (seed, read, column)
    d = synth_device(hd, t, 0, R)
    rs = t.refseq if refseq else None
    j = Juliet(L, genes, refseq=rs, handle=hd, region=region)
    j.pileup_device(d0.data_ptr(), R0)
    j.capture_control()
    j.reset()
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    got = j.control_call(variants)
    st = oracle.unpack(host_rows(d, R, L), L, nthreads=8)
    st0 = oracle.unpack(host_rows(d0, R0, L), L, nthreads=8)
    smp, ctl = co.histogram(st, L, genes, region), co.histogram(st0, L, genes, region)
    _, codon = j.get_counts()
    assert np.array_equal(codon, smp)
    listed = [(v.gene, v.col, v.codon) for v in variants]
    want = co.control(smp, ctl, L, genes, refseq=rs, region=region, listed=listed)
    _check(got, want)
    assert len(variants) > 0 and sum(r.listed for r in got.rows) == len(variants)
    # the strain that the control lacks is called against it; the shared one is not
    private = {(c, k) for (s, c, k) in t.truth if s == 2}
    shared = {(c, k) for (s, c, k) in t.truth if s == 1}
    calls = {(r.col, r.codon) for r in got.rows if r.called}
    in_genes = {(r.col, r.codon) for r in got.rows}
    assert private & in_genes <= calls and not (shared & calls)


# ---------------------------------------------------------------------------------------------------------- crafted edges
def test_edges_of_the_rule(hd):
    """n0 = 0, k0 = 0, k0 > k n0 / n (listed: p near 1), the reference codon from the sample, coverage 1, k = n"""
    L, genes = 30, [(1, 31)]
    smp = _hist(L, {0: {AAA: 900, CCC: 100}, 3: {AAA: 990, CCC: 10}, 6: {AAA: 950, CCC: 50}, 9: {AAA: 1000, TTT: 3},
                    12: {CCC: 1}, 15: {TTT: 40}, 18: {AAA: 10, CCC: 30}, 21: {c: 100 for c in range(64)}})
    ctl = _hist(L, {3: {AAA: 1000}, 6: {AAA: 900, CCC: 100}, 9: {AAA: 1000}, 12: {AAA: 5}, 15: {AAA: 40}, 18: {AAA: 30, CCC: 10},
                    21: {AAA: 6400}, 24: {AAA: 1}})
    listed = [(0, 6, CCC), (0, 0, CCC), (0, 9, TTT)]
    for refseq in (None, "AAA" * 10):
        j = _crafted(hd, smp, ctl, L, genes, refseq=refseq)
        got = j.control_call(_listed(j, listed))
        want = co.control(smp, ctl, L, genes, refseq=refseq, listed=listed)
        _check(got, want)
        by = {(r.col, r.codon): r for r in got.rows}
        assert by[(0, CCC)].pvalue == 1.0 and by[(0, CCC)].control_coverage == 0 and not by[(0, CCC)].called
        assert by[(6, CCC)].listed and not by[(6, CCC)].called and by[(6, CCC)].pvalue > 0.99
        assert by[(3, CCC)].called and by[(3, CCC)].control_count == 0
        assert got.uncovered_positions == 1


@pytest.mark.parametrize("case", range(4))
def test_decision_straddles_alpha(hd, case):
    """alpha = p * ntests * (1 +- 1e-10): called above, not below; a codon that is not listed only comes back when called"""
    n, k, n0, k0 = [(6000, 40, 6000, 12), (10_000, 9, 100_000, 20), (1_000_000, 1200, 500_000, 450), (300, 299, 280, 270)][case]
    L, genes = 30, [(1, 31)]                                  # ntests = 10
    smp = _hist(L, {9: {AAA: n - k, CCC: k}, 0: {AAA: 500}})
    ctl = _hist(L, {9: {AAA: n0 - k0, CCC: k0}, 0: {AAA: 500}})
    p = ref.fisher_greater(k, n - k, k0, n0 - k0)
    refseq = "AAA" * 10                                       # k close to n: CCC would be the sample's major codon
    for side, f in (("above", 1 + 1e-10), ("below", 1 - 1e-10)):
        alpha = float(p * 10 * f)
        j = _crafted(hd, smp, ctl, L, genes, alpha=alpha, refseq=refseq)
        for listed in ([], [(0, 9, CCC)]):
            got = j.control_call(_listed(j, listed))
            _check(got, co.control(smp, ctl, L, genes, refseq=refseq, alpha=alpha, listed=listed))
            rows = [r for r in got.rows if (r.col, r.codon) == (9, CCC)]
            assert [r.called for r in rows] == ([1] if side == "above" else ([0] if listed else [])), (side, rows)


def test_coverages_near_two_to_the_31(hd):
    L, genes = 15, [(1, 16)]
    big = 2 ** 31
    smp = _hist(L, {0: {AAA: big - 3000, CCC: 3000}, 3: {AAA: big, CCC: 2 ** 30}, 6: {AAA: big - 10, TTT: 10}, 9: {AAA: 1000, CCC: 10}})
    ctl = _hist(L, {0: {AAA: big - 1000, CCC: 1000}, 3: {AAA: big, CCC: 1000}, 6: {AAA: 2 ** 30, TTT: 2 ** 30}, 9: {AAA: big, CCC: 100}})
    listed = [(0, 6, TTT), (0, 9, CCC)]
    j = _crafted(hd, smp, ctl, L, genes)
    got = j.control_call(_listed(j, listed))
    _check(got, co.control(smp, ctl, L, genes, listed=listed))
    by = {(r.col, r.codon): r for r in got.rows}
    assert by[(0, CCC)].called and by[(3, CCC)].called and by[(6, TTT)].pvalue == 1.0 and by[(9, CCC)].called


def test_percentage_filters_and_overlapping_genes(hd):
    L = 30
    smp = _hist(L, {s: {AAA: 900, CCC: 100, TTT: 30} for s in range(0, 28)})
    ctl = _hist(L, {s: {AAA: 1000, TTT: 30} for s in range(0, 28)})
    genes = [(1, 31), (2, 29), (10, 25)]
    for kw in (dict(), dict(min_perc=10.0), dict(max_perc=10.0), dict(min_perc=9.0, max_perc=11.0), dict(region=(4, 20))):
        j = _crafted(hd, smp, ctl, L, genes, **kw)
        listed = [(v.gene, v.col, v.codon) for v in j.call()]
        _check(j.control_call(), co.control(smp, ctl, L, genes, listed=listed, **_kw(kw)))


def test_output_regrows(hd):
    """more records than the first device buffer (4096): every position with 63 control calls"""
    L = 3 * 80
    smp = _hist(L, {s: {c: 100 for c in range(64)} for s in range(0, L, 3)})
    ctl = _hist(L, {s: {AAA: 6400} for s in range(0, L, 3)})
    j = _crafted(hd, smp, ctl, L, [(1, L + 1)])
    got = j.control_call([], cap=16)
    assert len(got.rows) == 80 * 63 and all(r.called and not r.listed for r in got.rows)
    want = co.control(smp, ctl, L, [(1, L + 1)])
    _check(got, want)


# ------------------------------------------------------------------------------------------------------------ state rules
def test_capture_state_rules(hd):
    L, genes = 30, [(1, 31)]
    smp = _hist(L, {0: {AAA: 900, CCC: 100}, 3: {AAA: 990, CCC: 10}, 6: {AAA: 950, CCC: 50}})
    ctl = _hist(L, {0: {AAA: 900, CCC: 100}, 3: {AAA: 1000}, 6: {AAA: 990, CCC: 10}})
    j = Juliet(L, genes, handle=hd)
    _write(j, hd, smp)
    fields = lambda vs: [tuple(getattr(v, f) for f, _ in _lib.Variant._fields_) for v in vs]
    before = fields(j.call())
    with pytest.raises(_lib.MsError, match="no control captured"):
        j.control_call()
    _write(j, hd, ctl)
    j.capture_control()
    j.reset()                                                # the capture survives a reset of the counts
    _write(j, hd, smp)
    assert fields(j.call()) == before                        # capturing does not change K2
    first = j.control_call()
    second = j.control_call()
    assert [bytes(r) for r in first.rows] == [bytes(r) for r in second.rows] and first.uncovered_positions == second.uncovered_positions
    listed = [(v.gene, v.col, v.codon) for v in j.call()]
    _check(first, co.control(smp, ctl, L, genes, listed=listed))
    Juliet(L, genes, handle=hd)                              # a new layout drops the capture
    with pytest.raises(_lib.MsError, match="no control captured"):
        j.control_call()


def test_listed_variant_outside_the_positions_is_refused(hd):
    L, genes = 30, [(1, 31)]
    smp = _hist(L, {0: {AAA: 900, CCC: 100}})
    j = _crafted(hd, smp, smp, L, genes, region=(1, 10))
    with pytest.raises(_lib.MsError, match="tested positions"):
        j.control_call(_listed(j, [(0, 12, CCC)]))
