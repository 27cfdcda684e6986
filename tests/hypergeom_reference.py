"""High-precision reference for the project's statistics: hypergeometric tails in mpmath, linkage measures in exact
fractions, and K2's expected error count.  Plain restatements of the definitions, written for the tests; nothing here
shares code with the library or with the long-double oracle under oracle/.

Tails.  X ~ Hypergeometric(white, black, draws), P(X = x) = C(white, x) C(black, draws - x) / C(white + black, draws).  One
point mass comes from loggamma, the rest of a tail from the exact term ratio, summed outward from the starting point until
a falling term is below 1e-40 of the sum.  A tail that holds the mode is taken as 1 minus the other tail, which is then
short; at 60 significant digits that subtraction costs nothing that matters at a 1e-12 bar.
"""
import math
from fractions import Fraction

import mpmath as mp

DPS = 60            # significant digits of every returned value
_STOP = mp.mpf("1e-40")


def _support(white, black, draws):
    return max(0, draws - black), min(white, draws)


def _pmf(x, white, black, draws):
    """P(X = x) from log-gammas; the working precision grows with the size of the logs so that DPS digits survive exp"""
    lg = mp.loggamma
    with mp.workdps(DPS + 15 + len(str(white + black + 1))):
        lp = (lg(white + 1) - lg(x + 1) - lg(white - x + 1) + lg(black + 1) - lg(draws - x + 1) - lg(black - draws + x + 1)
              - lg(white + black + 1) + lg(draws + 1) + lg(white + black - draws + 1))
        return mp.exp(lp)


def _sum_up(a, white, black, draws):
    """sum of P(X = x) for x = a, a + 1, ... (a inside the support)"""
    hi = _support(white, black, draws)[1]
    with mp.workdps(DPS + 10):
        term = _pmf(a, white, black, draws)
        s = +term
        x = a
        while x < hi:
            num, den = (white - x) * (draws - x), (x + 1) * (black - draws + x + 1)
            term = term * num / den
            s += term
            x += 1
            if num < den and term < s * _STOP:
                break
        return s


def _sum_down(a, white, black, draws):
    """sum of P(X = x) for x = a, a - 1, ... (a inside the support)"""
    lo = _support(white, black, draws)[0]
    with mp.workdps(DPS + 10):
        term = _pmf(a, white, black, draws)
        s = +term
        x = a
        while x > lo:
            num, den = x * (black - draws + x), (white - x + 1) * (draws - x + 1)
            term = term * num / den
            s += term
            x -= 1
            if num < den and term < s * _STOP:
                break
        return s


def _mode(white, black, draws):
    return (white + 1) * (draws + 1) // (white + black + 2)


def upper(a, white, black, draws):
    """P(X >= a) as an mpf"""
    lo, hi = _support(white, black, draws)
    if a <= lo:
        return mp.mpf(1)
    if a > hi:
        return mp.mpf(0)
    if a >= _mode(white, black, draws):
        return _sum_up(a, white, black, draws)
    with mp.workdps(DPS + 10):
        return 1 - _sum_down(a - 1, white, black, draws)


def lower(a, white, black, draws):
    """P(X <= a) as an mpf: the upper tail of draws - X ~ Hypergeometric(black, white, draws)"""
    return upper(draws - a, black, white, draws)


def fisher_greater(a, b, c, d):
    """one-sided "greater" p-value of the 2x2 table [[a, b], [c, d]]: P(X >= a) for the top-left cell"""
    return upper(a, a + c, b + d, a + b)


def fisher_less(a, b, c, d):
    """P(X <= a) for the top-left cell of the tables with the margins of [[a, b], [c, d]]"""
    return lower(a, a + c, b + d, a + b)


def linkage_measures(a, b, c, n):
    """(D', r^2) as Fractions; both 0 when a margin is empty or full (restatement choice U14)"""
    mv, mw = a + b, a + c
    if mv in (0, n) or mw in (0, n):
        return Fraction(0), Fraction(0)
    fv, fw = Fraction(mv, n), Fraction(mw, n)
    D = Fraction(a, n) - fv * fw
    r2 = D * D / (fv * (1 - fv) * fw * (1 - fw))
    if D > 0:
        dp = D / min(fv * (1 - fw), (1 - fv) * fw)
    elif D < 0:
        dp = D / min(fv * fw, (1 - fv) * (1 - fw))
    else:
        dp = Fraction(0)
    return dp, r2


def codon_error_table(sub_rate, del_rate):
    """P(ref codon -> a codon with nm mismatching bases), nm = 0..3.  Restatement choice U1 defines it in doubles, so it is
    built here with the same float operations in the same order (Python floats are IEEE doubles)."""
    match, mis = 1.0 - sub_rate - del_rate, sub_rate / 3.0
    out = []
    for nm in range(4):
        p = 1.0
        for _ in range(3 - nm):
            p *= match
        for _ in range(nm):
            p *= mis
        out.append(p)
    return out


def mismatches(ref_codon, codon):
    return sum(((ref_codon >> (2 * i)) & 3) != ((codon >> (2 * i)) & 3) for i in range(3))


def expected_count(n, P):
    """K2's expected error count e = min(n, ceil(n * P)), the product in doubles"""
    return min(n, math.ceil(float(n) * P))


def k2_pvalue(k, n, e):
    """K2's p-value of a codon seen k times in n with expected count e: the table [[k, n - k], [e, n - e]]"""
    return fisher_greater(k, n - k, e, n - e)


def rel_err(got, want):
    """|got - want| / want, evaluated in mpmath (want > 0)"""
    with mp.workdps(DPS):
        return abs(mp.mpf(got) - want) / want
