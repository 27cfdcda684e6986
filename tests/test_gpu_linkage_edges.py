"""Pairwise linkage (ms_linkage / Juliet.linkage) at its edges, against the mpmath / Fraction reference in
hypergeom_reference.py.

Reads are made so that every pair of keys has a chosen 2x2 table: pair i owns two codons, v at column 6 i (CAA against an
all-A reference) and w 2 or 3 columns on (AAG), and four read types that cover only those two codons (both, v only, w only,
neither).  Reads of other pairs leave a pair's codons uncovered, so pairs across groups have no informative reads and are
not tested.  Tables: margins empty or full, the cell at the bounds of its range and at mode - 1 / mode / mode + 1, zero cells,
n = min_reads - 1 and min_reads, codons 2 and 3 columns apart, n up to 2 000 000; alpha straddling p * m by 1e-10 on
either tail.  Relation, counts and the number of tested pairs exactly, p to 1e-12 relative, D' and r^2 to 1e-14 absolute.
"""
from fractions import Fraction

import mpmath as mp
import numpy as np
import pytest

import hypergeom_reference as ref

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from minorseq_b200 import Handle, Juliet, device_rows  # noqa: E402
from minorseq_b200.synth import pack_states  # noqa: E402

RTOL = 1e-12
MARGIN = 5e-11
LINKED, EXCLUSIVE = 1, 2
V_CODON, W_CODON = 16 * 1, 2          # CAA, AAG (the reference is all A)
GROUP = 6                             # columns per pair


class _Var:
    def __init__(self, col, codon):
        self.col, self.codon = col, codon


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def phased(hd, tables, spacing=None):
    """tables: (a, b, c, d) per pair -> (Juliet phased with linkage on, keys, per-pair spacing)"""
    spacing = spacing or [3] * len(tables)
    G = len(tables)
    L = GROUP * G
    proto, counts = [], []
    for i, ((a, b, c, d), sp) in enumerate(zip(tables, spacing)):
        v, w = GROUP * i, GROUP * i + sp
        for carry_v, carry_w, k in ((1, 1, a), (1, 0, b), (0, 1, c), (0, 0, d)):
            st = np.full(L, 7, dtype=np.uint8)          # uncovered
            st[v:v + 3] = 0
            st[w:w + 3] = 0
            if carry_v:
                st[v] = 1                                # C at the first base of v's codon
            if carry_w:
                st[w + 2] = 2                            # G at the last base of w's codon
            proto.append(st)
            counts.append(k)
    rows = np.repeat(pack_states(np.array(proto)), counts, axis=0)
    d = device_rows(rows)
    j = Juliet(L, [(1, L + 1)], handle=hd)
    keys = [_Var(GROUP * i, V_CODON) for i in range(G)] + [_Var(GROUP * i + sp, W_CODON) for i, sp in enumerate(spacing)]
    _, sorted_keys = j.phase_device(keys, d.data_ptr(), rows.shape[0], want_hap_id=False, linkage=True)
    assert sorted_keys == sorted((k.col, k.codon) for k in keys)
    return j, sorted_keys, spacing


_TAILS = {}


def tails(t):
    if t not in _TAILS:
        _TAILS[t] = (ref.fisher_greater(*t), ref.fisher_less(*t))
    return _TAILS[t]


def decide(p, m, alpha):
    with mp.workdps(ref.DPS):
        if 1 - p < mp.mpf("1e-17"):
            return 1.0 * m < alpha
        assert abs(p * m / alpha - 1) > MARGIN, ("case too close to its threshold", mp.nstr(p, 20), m, alpha)
        return p * m < alpha


def expected(tables, spacing, alpha, min_reads):
    tested = [i for i, (t, sp) in enumerate(zip(tables, spacing)) if sp >= 3 and sum(t) >= min_reads]
    m = len(tested)
    pairs = []
    for i in tested:
        pt, pa = tails(tables[i])
        if decide(pt, m, alpha):
            pairs.append((i, LINKED, pt))
        elif decide(pa, m, alpha):
            pairs.append((i, EXCLUSIVE, pa))
    return m, pairs


def check(j, keys, tables, spacing, alpha, min_reads=10):
    lk = j.linkage(alpha=alpha, min_reads=min_reads)
    index = {k: n for n, k in enumerate(keys)}
    vw = [(index[(GROUP * i, V_CODON)], index[(GROUP * i + sp, W_CODON)]) for i, sp in enumerate(spacing)]
    for i, (v, w) in enumerate(vw):                      # the counts behind every pair, tested or not
        a, b, c, d = tables[i]
        assert (lk.n[v, w], lk.a[v, w], lk.b[v, w], lk.c[v, w]) == (a + b + c + d, a, b, c), (i, tables[i])
    m, want = expected(tables, spacing, alpha, min_reads)
    assert lk.ntested == m
    got = list(zip(lk.v.tolist(), lk.w.tolist()))
    assert got == [vw[i] for i, _, _ in want], (alpha, min_reads)
    for k, (i, rel, p) in enumerate(want):
        a, b, c, d = tables[i]
        assert (lk.both[k], lk.v_only[k], lk.w_only[k], lk.neither[k], lk.relation[k]) == (a, b, c, d, rel), tables[i]
        if p > mp.mpf("1e-300"):
            assert ref.rel_err(lk.pvalue[k], p) <= RTOL, (tables[i], lk.pvalue[k], mp.nstr(p, 20))
        else:
            assert lk.pvalue[k] < 1e-290, tables[i]
        wdp, wr2 = ref.linkage_measures(a, b, c, a + b + c + d)
        assert abs(Fraction(float(lk.d_prime[k])) - wdp) <= Fraction(1, 10 ** 14), (tables[i], lk.d_prime[k], float(wdp))
        assert abs(Fraction(float(lk.r2[k])) - wr2) <= Fraction(1, 10 ** 14), (tables[i], lk.r2[k], float(wr2))
    return lk


def around_mode(n, mv, mw):
    lo, hi = max(0, mv + mw - n), min(mv, mw)
    mode = (mv + 1) * (mw + 1) // (n + 2)
    return [(a, mv - a, mw - a, n - mv - mw + a) for a in sorted({lo, lo + 1, mode - 1, mode, mode + 1, hi - 1, hi}) if lo <= a <= hi]


SMALL = ([(0, 0, 5, 5), (5, 5, 0, 0), (0, 5, 0, 5), (5, 0, 5, 0), (10, 0, 0, 0), (0, 0, 0, 10), (0, 10, 0, 0), (0, 0, 10, 0),
          (30, 0, 5, 965), (30, 5, 0, 965), (0, 40, 60, 900), (900, 40, 60, 0), (998, 1, 1, 0), (0, 1, 1, 998), (1, 0, 0, 999),
          (999, 0, 0, 1), (20, 5, 5, 70), (2, 30, 30, 38), (3, 2, 2, 2), (3, 2, 2, 3)]
         + around_mode(1000, 300, 400) + around_mode(101, 50, 50) + around_mode(10_007, 5003, 1429))


def test_linkage_table_shapes(hd):
    tables = SMALL + [(20, 5, 5, 70), (2, 30, 30, 38)]
    spacing = [3] * len(SMALL) + [2, 2]                  # the last two share a column: never tested
    j, keys, spacing = phased(hd, tables, spacing)
    for alpha in (0.01, 0.5, 1.0):
        check(j, keys, tables, spacing, alpha)
    for min_reads in (9, 10, 11, 1):                     # (3, 2, 2, 2) has n = 9, (3, 2, 2, 3) n = 10
        lk = check(j, keys, tables, spacing, 0.05, min_reads)
        assert lk.ntested == sum(1 for t, sp in zip(tables, spacing) if sp >= 3 and sum(t) >= min_reads)


@pytest.mark.parametrize("which", ["together", "apart"])
def test_linkage_alpha_straddle(hd, which):
    """alpha = p * m * (1 +- 1e-10) on a linked pair's P(X >= a) and on an exclusive pair's P(X <= a)"""
    tables = SMALL
    j, keys, spacing = phased(hd, tables)
    m, _ = expected(tables, spacing, 0.01, 10)
    t = (20, 5, 5, 70) if which == "together" else (2, 30, 30, 38)
    p = tails(t)[0 if which == "together" else 1]
    i = tables.index(t)
    for side, f in (("above", 1 + 1e-10), ("below", 1 - 1e-10)):
        lk = check(j, keys, tables, spacing, float(p * m * f))
        v = keys.index((GROUP * i, V_CODON))
        assert (v in lk.v.tolist()) == (side == "above"), (which, side)


def test_linkage_large_tables(hd):
    """n = 200 000 and 2 000 000: the mode of a balanced table, single reads against the rest, and the exclusive pair
    [[n - 10^4, 5000], [5000, 0]], whose D' is exactly -1 (a / n - f_v f_w in doubles was off by ~2e-11)"""
    n, n2 = 2_000_000, 200_000
    tables = ([around_mode(n, n // 2, n // 2)[3], (n - 10_000, 5000, 5000, 0)] + around_mode(n2, n2 // 2, n2 // 2)[2:5]
              + [(1, 0, 0, n2 - 1), (0, 1, 1, n2 - 2), (n2 - 2, 1, 0, 1)] + around_mode(n2, 1, n2 // 7))
    j, keys, spacing = phased(hd, tables)
    for alpha in (0.01, 1.0):
        lk = check(j, keys, tables, spacing, alpha)
    k = [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(lk.both, lk.v_only, lk.w_only, lk.neither)].index((n - 10_000, 5000, 5000, 0))
    assert lk.d_prime[k] == -1.0 and lk.relation[k] == EXCLUSIVE
