"""The library's statistics core (fisher_core.h, linkage_core.h: the code K2 and the linkage kernels run on the GPU) compiled
for the host and compared with the mpmath / Fraction reference in hypergeom_reference.py at the tables where it can go wrong:
coverage 1 and 2, e = 0 or n, k = n, codons at or below their expected count, linkage margins that are empty or full, cells
at the bounds of their range and around the mode, and counts up to 10^7.

Bar: p-values to 1e-12 relative wherever the reference is above 1e-300 (both below 1e-290 otherwise); D' and r^2 to 1e-14
absolute.  Limit: K2 sums a column's 64 bins in uint32, so columns of 2^32 reads or more are out of range and not tested.
"""
import ctypes as C
import itertools
import math
import os
import subprocess
from fractions import Fraction

import mpmath as mp
import pytest

import hypergeom_reference as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "minorseq_b200", "csrc")
RTOL = 1e-12
TINY_REF, TINY_GOT = mp.mpf("1e-300"), 1e-290

SHIM = (
    '#include "linkage_core.h"\n'
    'extern "C" double upper(uint32_t a, uint32_t b, uint32_t c, uint32_t d, double enough) { return ms::fisher_upper(a, b, c, d, enough); }\n'
    'extern "C" void linkage(uint32_t a, uint32_t b, uint32_t c, uint32_t d, double enough, double* o) '
    '{ ms::linkage_tails(a, b, c, d, enough, o, o + 1); ms::linkage_measures(a, b, c, a + b + c + d, o + 2, o + 3); }\n')


@pytest.fixture(scope="module")
def core(tmp_path_factory):
    d = tmp_path_factory.mktemp("fisher_core")
    (d / "shim.cpp").write_text(SHIM)
    so = d / "core.so"
    res = subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-Wall", "-Werror", f"-I{CSRC}",
                          str(d / "shim.cpp"), "-o", str(so)], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lib = C.CDLL(str(so))
    lib.upper.restype = C.c_double
    lib.upper.argtypes = [C.c_uint32] * 4 + [C.c_double]
    lib.linkage.restype = None
    lib.linkage.argtypes = [C.c_uint32] * 4 + [C.c_double, C.POINTER(C.c_double)]
    return lib


def linkage(core, a, b, c, d, enough=2.0):
    o = (C.c_double * 4)()
    core.linkage(a, b, c, d, enough, o)
    return tuple(o)


def assert_close(got, want, what):
    if want > TINY_REF:
        assert ref.rel_err(got, want) <= RTOL, (what, got, mp.nstr(want, 20))
    else:
        assert got < TINY_GOT, (what, got, mp.nstr(want, 20))


def assert_enough(got, want, enough, what):
    """a result below `enough` is the whole tail; one at or above it only promises that the tail is not below `enough`"""
    if got < enough:
        assert_close(got, want, what)
    else:
        assert want >= enough * (1 - 1e-9), (what, got, mp.nstr(want, 20), enough)


# ---------------------------------------------------------------------------------------------------- the reference itself
def test_reference_against_exact_sums():
    """The mpmath tails against exact rational sums of binomial products on every table of a small grid, and the two tails
    of each table add up to 1 + P(X = a)."""
    for white, black, draws in itertools.product((0, 1, 2, 5, 13), (0, 1, 3, 7, 20), (0, 1, 4, 9)):
        if draws > white + black:
            continue
        tot = math.comb(white + black, draws)
        lo, hi = ref._support(white, black, draws)
        for a in range(lo - 1, hi + 2):
            up = Fraction(sum(math.comb(white, x) * math.comb(black, draws - x) for x in range(max(a, lo), hi + 1)), tot)
            dn = Fraction(sum(math.comb(white, x) * math.comb(black, draws - x) for x in range(lo, min(a, hi) + 1)), tot)
            for got, want in ((ref.upper(a, white, black, draws), up), (ref.lower(a, white, black, draws), dn)):
                with mp.workdps(ref.DPS):
                    assert abs(got - mp.mpf(want.numerator) / want.denominator) <= mp.mpf("1e-50"), (a, white, black, draws)


def test_reference_large_tables_are_consistent():
    """At 10^5 - 10^7 reads: P(X >= a) + P(X <= a - 1) = 1 from the two summation directions (to 1e-30: a sum stops once its
    terms fall below 1e-40 of it, and the slowly falling tails here leave up to ~1e-38 behind)."""
    for white, black, draws in ((5_000_000, 5_000_000, 5_000_000), (2683, 197317, 100000), (1_000_000, 1_000_000, 999_999)):
        mode = ref._mode(white, black, draws)
        for a in (mode - 40, mode, mode + 1, mode + 300):
            with mp.workdps(ref.DPS):
                s = ref.upper(a, white, black, draws) + ref.lower(a - 1, white, black, draws)
                assert abs(s - 1) < mp.mpf("1e-30"), (a, white, black, draws)


# ------------------------------------------------------------------------------------------------------------------ K2
def k2_tables():
    """(k, n, e) in the shape K2 tests: [[k, n - k], [e, n - e]]"""
    out = set()
    for n in (1, 2, 3, 7, 10, 100, 1000, 10_000, 100_000, 1_000_000, 10_000_000):
        for e in {0, 1, n - 1, n}:
            if not 0 <= e <= n:
                continue
            for k in {n, e + 1, max(1, e)}:
                if 1 <= k <= n:
                    out.add((k, n, e))
    # codons at or below their expected count (tested by K2 only when alpha > ntests / 2): k down to 1, e in the thousands
    for n, e in ((100_000, 2683), (1_000_000, 2683), (1_000_000, 70_000), (10_000_000, 9_000)):
        for k in (1, 2, 3, 10, e // 10, e // 2, e - 100, e - 1, e, e + 1, e + 2, e + 100):
            out.add((k, n, e))
    # the default error table at real coverages: e from codon_error_table, k around and far above it
    P = ref.codon_error_table(5e-4, 3e-3)
    for n in (1, 2, 3, 10, 2907, 100_000, 3_000_000, 10_000_000):
        for nm in (1, 2, 3):
            e = ref.expected_count(n, P[nm])
            for k in (1, e, e + 1, e + 3, 2 * e + 10, n // 100, n // 3, n):
                if 1 <= k <= n:
                    out.add((k, n, e))
    return sorted(out)


def test_k2_upper_tail_matches_reference(core):
    tables = k2_tables()
    assert len(tables) > 150
    for k, n, e in tables:
        want = ref.k2_pvalue(k, n, e)
        assert_close(core.upper(k, n - k, e, n - e, 2.0), want, (k, n, e))


def test_k2_codons_below_expected_are_not_significant(core):
    """The codon from the issue that motivated fisher_upper: seen once in 100 000 reads with 2 683 expected.  Its tail was
    summed from k = 1, whose point mass underflows, and came out 0 (significant at any alpha) instead of 1."""
    assert core.upper(1, 99_999, 2683, 97_317, 2.0) == 1.0
    assert core.upper(1, 999_999, 70_000, 930_000, 2.0) == 1.0
    for k, n, e in k2_tables():
        if k <= e:
            assert core.upper(k, n - k, e, n - e, 2.0) >= 0.5, (k, n, e)


def test_k2_expected_count():
    """e = min(n, ceil(n P)) with P in doubles: the default rates, a substitution rate of 0.1, e = 0 and e = n"""
    P = ref.codon_error_table(5e-4, 3e-3)
    assert [ref.expected_count(n, P[1]) for n in (1, 2, 1000, 2907, 10_000)] == [1, 1, 1, 1, 2]
    assert ref.expected_count(100_000, ref.codon_error_table(0.1, 3e-3)[1]) == 2683
    assert ref.codon_error_table(0.0, 0.0) == [1.0, 0.0, 0.0, 0.0]
    assert ref.expected_count(5, ref.codon_error_table(0.0, 0.0)[1]) == 0
    assert ref.expected_count(5, 1.0) == 5 and ref.expected_count(5, 1.5) == 5


@pytest.mark.parametrize("k,n,e", [(2, 100, 0), (5, 1000, 1), (60, 5940, 1), (30, 2907, 1), (101, 100_000, 84), (51, 100, 50),
                                   (10_001, 10_000_000, 10_000), (2000, 1_000_000, 1000), (1, 99_999, 2683)])
def test_k2_enough_contract(core, k, n, e):
    want = ref.k2_pvalue(k, n, e)
    wf = float(want)
    for enough in (2.0, 1.0, wf * 4, wf * 1.0001, wf * (1 + 1e-9), wf, wf * (1 - 1e-9), wf / 4, 1e-300, 1e-12, 0.5, 0.25):
        if enough <= 0.0:
            continue
        assert_enough(core.upper(k, n - k, e, n - e, enough), want, enough, (k, n, e, enough))


# -------------------------------------------------------------------------------------------------------------- linkage
def linkage_tables():
    """(a, b, c, d): margins empty or full, the cell at both bounds of its range, next to them and at mode - 1, mode, mode + 1"""
    out = {(0, 0, 0, 0), (0, 0, 0, 10), (10, 0, 0, 0), (0, 10, 0, 0), (0, 0, 10, 0), (5, 5, 0, 0), (0, 0, 5, 5), (5, 0, 5, 0),
           (0, 5, 0, 5), (0, 5, 5, 0), (5, 0, 0, 5), (1, 0, 0, 0), (0, 1, 0, 0), (1, 1, 1, 1), (3, 0, 0, 7)}
    for n in (10, 11, 101, 1000, 10_007, 200_000, 2_000_000):
        for mv, mw in itertools.product({1, 2, n // 3, n // 2, n - 1}, {1, n // 7, n // 2, n - 2, n - 1}):
            if not (0 < mv < n and 0 < mw < n):
                continue
            lo, hi = max(0, mv + mw - n), min(mv, mw)
            mode = (mv + 1) * (mw + 1) // (n + 2)
            for a in {lo, lo + 1, mode - 1, mode, mode + 1, hi - 1, hi}:
                if lo <= a <= hi:
                    out.add((a, mv - a, mw - a, n - mv - mw + a))
    return sorted(out)


def test_linkage_tails_and_measures_match_reference(core):
    tables = linkage_tables()
    assert len(tables) > 400
    for a, b, c, d in tables:
        pt, pa, dp, r2 = linkage(core, a, b, c, d)
        assert_close(pt, ref.fisher_greater(a, b, c, d), ("together", a, b, c, d))
        assert_close(pa, ref.fisher_less(a, b, c, d), ("apart", a, b, c, d))
        wdp, wr2 = ref.linkage_measures(a, b, c, a + b + c + d)
        assert abs(Fraction(dp) - wdp) <= Fraction(1, 10 ** 14), ("D'", a, b, c, d, dp, float(wdp))
        assert abs(Fraction(r2) - wr2) <= Fraction(1, 10 ** 14), ("r2", a, b, c, d, r2, float(wr2))
        assert -1.0 <= dp <= 1.0 and 0.0 <= r2 <= 1.0


@pytest.mark.parametrize("n", [4, 1000, 2_000_000, 2 ** 31])
def test_linkage_measures_cancellation(core, n):
    """Tables where a / n and f_v f_w nearly cancel.  D' is exactly -1 or 1 when the cell behind the smaller D_max is empty
    (in doubles a / n - f_v f_w gave -1.0005 for [[n-2, 1], [1, 0]] at n = 2 000 000), and r^2 keeps its 1e-14."""
    for t, want_dp in (((n - 2, 1, 1, 0), -1.0), ((0, 1, 1, n - 2), -1.0), ((1, 0, 0, n - 1), 1.0), ((n - 1, 0, 0, 1), 1.0),
                       ((n - 3, 1, 1, 1), None), ((1, 1, 0, n - 2), 1.0), ((n - 2, 0, 1, 1), 1.0)):
        _, _, dp, r2 = linkage(core, *t)
        wdp, wr2 = ref.linkage_measures(t[0], t[1], t[2], n)
        if want_dp is not None:
            assert wdp == want_dp and dp == want_dp, (t, dp)
        assert abs(Fraction(dp) - wdp) <= Fraction(1, 10 ** 14), (t, dp, float(wdp))
        assert abs(Fraction(r2) - wr2) <= Fraction(1, 10 ** 14), (t, r2, float(wr2))


def test_linkage_enough_contract(core):
    """Only the small tail is stopped early; a stopped tail is never below `enough`, an unstopped one is exact."""
    tables = [t for t in linkage_tables() if sum(t) >= 1000][::9]
    assert len(tables) > 20
    for a, b, c, d in tables:
        want_t, want_a = ref.fisher_greater(a, b, c, d), ref.fisher_less(a, b, c, d)
        for w in (want_t, want_a):
            wf = float(w)
            for enough in (wf * 2, wf * (1 + 1e-9), wf * (1 - 1e-9), wf / 2, 1e-300, 0.5):
                if enough <= 0.0:
                    continue
                pt, pa, _, _ = linkage(core, a, b, c, d, enough)
                assert_enough(pt, want_t, enough, ("together", a, b, c, d, enough))
                assert_enough(pa, want_a, enough, ("apart", a, b, c, d, enough))
