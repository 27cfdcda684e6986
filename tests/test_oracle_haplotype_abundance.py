"""The haplotype-abundance restatement (haplotype_abundance_oracle.py, restatement choice U18) on known answers and the
maximum-likelihood conditions, and the compile check of its CUDA kernels (CPU only)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import haplotype_abundance_oracle as ha

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sets(*groups):
    """rows of S from (set of haplotype indices, read count) pairs over H = 1 + the largest index"""
    H = 1 + max((max(s) for s, _ in groups if s), default=-1)
    rows = []
    for s, n in groups:
        rows += [[h in s for h in range(H)]] * n
    return np.array(rows, dtype=bool).reshape(-1, H)


def test_only_unique_reads():
    S = _sets(({0}, 70), ({1}, 20), ({2}, 10))
    a = ha.abundance_from_sets(S)
    assert np.allclose(a["em_frequency"], [0.7, 0.2, 0.1], rtol=0, atol=1e-15)
    assert a["counters"] == dict(unique=100, ambiguous=0, uninformative=0, incompatible=0)
    assert a["unique_reads"].tolist() == [70, 20, 10] and a["compatible_reads"].tolist() == [70, 20, 10]
    assert a["converged"] and a["iterations"] == 2          # the first step lands on the answer, the second sees no change


def test_shared_reads_split_in_proportion():
    """{A}:a, {B}:b, {A,B}:x, {C}:c -> pi_C = c/N, pi_A = a/(a+b) (a+b+x)/N"""
    a_, b_, x, c = 300, 100, 200, 400
    S = _sets(({0}, a_), ({1}, b_), ({0, 1}, x), ({2}, c))
    r = ha.abundance_from_sets(S)
    N = a_ + b_ + x + c
    want = [a_ / (a_ + b_) * (a_ + b_ + x) / N, b_ / (a_ + b_) * (a_ + b_ + x) / N, c / N]
    assert np.allclose(r["em_frequency"], want, rtol=0, atol=1e-9)
    assert r["counters"] == dict(unique=a_ + b_ + c, ambiguous=x, uninformative=0, incompatible=0)
    assert r["unique_reads"].tolist() == [a_, b_, c] and r["compatible_reads"].tolist() == [a_ + x, b_ + x, c]
    assert r["reads_used"] == N and r["converged"]


def test_incompatible_and_uninformative_reads_change_nothing():
    base = _sets(({0}, 30), ({1}, 50), ({0, 1}, 40), ({2}, 5))
    more = np.vstack([base, np.zeros((17, 3), dtype=bool), np.ones((23, 3), dtype=bool)])
    a, b = ha.abundance_from_sets(base), ha.abundance_from_sets(more)
    assert np.array_equal(a["em_frequency"], b["em_frequency"])
    assert a["iterations"] == b["iterations"] and a["log_likelihood"] == b["log_likelihood"]
    assert b["counters"] == dict(a["counters"], uninformative=23, incompatible=17)
    assert (b["compatible_reads"] - a["compatible_reads"]).tolist() == [23, 23, 23]
    assert np.array_equal(a["unique_reads"], b["unique_reads"])


def test_one_iteration_does_not_converge():
    S = _sets(({0}, 30), ({1}, 50), ({0, 1}, 40))
    r = ha.abundance_from_sets(S, max_iter=1)
    assert r["iterations"] == 1 and not r["converged"]


def test_edge_cases():
    r = ha.abundance_from_sets(np.zeros((12, 0), dtype=bool))              # H = 0: every read incompatible
    assert r["counters"]["incompatible"] == 12 and r["iterations"] == 0 and r["converged"]
    r = ha.abundance_from_sets(np.ones((12, 4), dtype=bool))               # N = 0: pi stays 1/H
    assert np.array_equal(r["em_frequency"], np.full(4, 0.25)) and r["iterations"] == 0 and r["converged"]
    assert r["counters"]["uninformative"] == 12
    r = ha.abundance_from_sets(np.ones((12, 1), dtype=bool))               # H = 1: a compatible read is unique
    assert r["counters"]["unique"] == 12 and r["em_frequency"].tolist() == [1.0]


def test_compatibility_rule():
    """agreement is required only where the read is clean"""
    B = np.array([[1, 0, 1], [1, 0, 1], [0, 0, 0]], dtype=bool)
    M = np.array([[1, 1, 1], [1, 0, 0], [0, 0, 0]], dtype=bool)
    P = np.array([[1, 0, 1], [1, 1, 0], [0, 1, 1]], dtype=bool)
    S = ha.compat_sets(B, M, P)
    assert S.tolist() == [[True, False, False], [True, True, False], [True, True, True]]
    pat = np.array([[0b101], [0b011 | (1 << 7)]], dtype=np.uint32)           # bit 7 >= V is ignored
    assert ha.pattern_bits(pat, 3).tolist() == [[1, 0, 1], [1, 1, 0]]


@pytest.mark.parametrize("seed", range(8))
def test_mle_conditions_on_random_class_tables(seed):
    rng = np.random.default_rng(seed)
    H = int(rng.integers(2, 40))
    C = int(rng.integers(1, 300))
    classes = rng.random((C, H)) < rng.uniform(0.05, 0.5)
    classes[classes.sum(axis=1) == 0, 0] = True
    counts = rng.integers(1, 1000, size=C)
    pi, it, conv, _ = ha.em(classes, counts, max_iter=200000)
    assert conv
    assert abs(pi.sum() - 1.0) < 1e-12
    g = ha.kkt_gradient(classes, counts, pi)
    assert (g <= 1.0 + 1e-6).all()
    assert np.allclose(g[pi > 1e-3], 1.0, rtol=0, atol=1e-6)


def test_abundance_kernels_do_not_spill():
    """The compatibility and EM kernels compile for sm_100a without spills."""
    nvcc = shutil.which("nvcc", path="/usr/local/cuda/bin") or shutil.which("nvcc")
    if not nvcc:
        pytest.skip("nvcc not found")
    src = os.path.join(ROOT, "minorseq_b200", "csrc", "abundance.cu")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                          "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out.stderr)
    assert len(spills) == 6 and all(s == ("0", "0") for s in spills), out.stderr
    assert "abundance_compat_kernel" in out.stderr and "abundance_sum_kernel" in out.stderr
