"""Pairwise linkage without a GPU: the test oracle's tails and measures against scipy and an independent formulation, and the
library's host/device core (linkage_core.h + fisher_core.h, compiled here as plain C++) against the oracle."""
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import linkage_oracle as lo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "minorseq_b200", "csrc")


def _random_tables(seed, k=200):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(k):
        n = int(rng.integers(10, 20000))
        p = rng.dirichlet([1.0, 0.3, 0.3, 1.0])
        a, b, c, d = (int(x) for x in rng.multinomial(n, p))
        out.append((a, b, c, d))
    out += [(0, 0, 0, 10), (10, 0, 0, 0), (5, 5, 0, 0), (0, 5, 5, 0), (3, 0, 0, 7), (1, 2, 3, 4)]
    return out


def test_oracle_tails_match_scipy(oracle):
    for a, b, c, d in _random_tables(1):
        want_t = stats.fisher_exact([[a, b], [c, d]], alternative="greater")[1]
        want_a = stats.fisher_exact([[a, b], [c, d]], alternative="less")[1]
        got_t, got_a = lo.tails(a, b, c, d, oracle.fisher)
        assert got_t == pytest.approx(want_t, rel=1e-9, abs=1e-300), (a, b, c, d)
        assert got_a == pytest.approx(want_a, rel=1e-9, abs=1e-300), (a, b, c, d)


def test_oracle_measures_match_haplotype_formulation():
    """D' and r^2 against D = (ad - bc) / n^2 and r^2 = (ad - bc)^2 / ((a+b)(c+d)(a+c)(b+d)) in exact integers."""
    for a, b, c, d in _random_tables(2):
        n = a + b + c + d
        dp, r2 = lo.measures(a, b, c, n)
        den = (a + b) * (c + d) * (a + c) * (b + d)
        if den == 0:
            assert (dp, r2) == (0.0, 0.0)
            continue
        cross = a * d - b * c
        assert r2 == pytest.approx(cross * cross / den, rel=1e-12, abs=1e-15)
        fv, fw = (a + b) / n, (a + c) / n
        dmax = min(fv * (1 - fw), (1 - fv) * fw) if cross > 0 else min(fv * fw, (1 - fv) * (1 - fw))
        want = 0.0 if cross == 0 else (cross / (n * n)) / dmax
        assert dp == pytest.approx(want, rel=1e-9, abs=1e-12)
        assert -1.0 - 1e-12 <= dp <= 1.0 + 1e-12 and 0.0 <= r2 <= 1.0 + 1e-12


def test_oracle_counts_from_states():
    """A hand-made read set: a read with an 'N' elsewhere still counts; a damaged codon removes the read from its pairs only."""
    L = 12
    st = np.zeros((5, L), dtype=np.uint8)                   # all A
    keys = [(0, 16 * 1 + 4 * 1 + 1), (6, 16 * 2 + 4 * 2 + 2)]    # CCC at 0, GGG at 6
    st[0, 0:3] = 1; st[0, 6:9] = 2                           # both
    st[1, 0:3] = 1                                           # v only
    st[2, 6:9] = 2; st[2, 11] = 5                            # w only, an N outside both codons
    st[3, 1] = 4                                             # deletion in v's codon: not informative
    n, a, b, c = lo.tables(st, keys)
    assert (n[0, 1], a[0, 1], b[0, 1], c[0, 1]) == (4, 1, 1, 1)
    assert (n[0, 0], n[1, 1]) == (4, 5)
    assert (a[0, 0], a[1, 1]) == (2, 2)


def _core_driver(tmp_path):
    src = tmp_path / "core.cpp"
    src.write_text(
        '#include <cstdio>\n#include "linkage_core.h"\n'
        "int main() {\n"
        "  unsigned a, b, c, d; double enough;\n"
        "  while (std::scanf(\"%u %u %u %u %lf\", &a, &b, &c, &d, &enough) == 5) {\n"
        "    double dp, r2; ms::linkage_measures(a, b, c, a + b + c + d, &dp, &r2);\n"
        "    double pt, pa; ms::linkage_tails(a, b, c, d, enough, &pt, &pa);\n"
        "    std::printf(\"%.17g %.17g %.17g %.17g\\n\", dp, r2, pt, pa);\n"
        "  }\n  return 0;\n}\n")
    exe = tmp_path / "core"
    res = subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-Wall", "-Werror", f"-I{CSRC}", str(src), "-o", str(exe)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return str(exe)


def test_library_core_matches_oracle(oracle, tmp_path):
    """The library's statistics core (host build of linkage_core.h / fisher_core.h): D', r^2 to 1e-12, both tails to 1e-9
    relative, and an early-stopped tail is still exact whenever it is below the threshold it was given."""
    exe = _core_driver(tmp_path)
    tabs = _random_tables(3)
    enough = [2.0 if i % 2 == 0 else 1e-6 for i in range(len(tabs))]
    inp = "".join(f"{a} {b} {c} {d} {e!r}\n" for (a, b, c, d), e in zip(tabs, enough))
    res = subprocess.run([exe], input=inp, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    for (a, b, c, d), e, line in zip(tabs, enough, res.stdout.splitlines()):
        dp, r2, pt, pa = (float(x) for x in line.split())
        wdp, wr2 = lo.measures(a, b, c, a + b + c + d)
        assert dp == pytest.approx(wdp, abs=1e-12) and r2 == pytest.approx(wr2, abs=1e-12)
        for got, want in zip((pt, pa), lo.tails(a, b, c, d, oracle.fisher)):
            if want < e:
                assert got == pytest.approx(want, rel=1e-9, abs=1e-300), (a, b, c, d)
            else:                                  # stopped early: only "not below the threshold" is promised
                assert got >= e * (1 - 1e-12) or got == pytest.approx(want, rel=1e-9, abs=1e-15), (a, b, c, d)
