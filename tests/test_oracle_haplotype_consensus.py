"""CPU checks of the test-side U15 oracle (tests/haplotype_consensus_oracle.py) and of the grouped pile-up's build."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import haplotype_consensus_oracle as hco
from minorseq_b200.synth import SynthConfig, make_tables, synth_states

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def col_of(rows):
    """[L, 8] counts from per-column lists of (state, count)"""
    col = np.zeros((len(rows), 8), dtype=np.uint32)
    for j, cells in enumerate(rows):
        for s, n in cells:
            col[j, s] += n
        col[j, 7] = col[j, :6].sum()
    return col


def insertion_events(rng, R, L, nsites=6, per_site=(650, 850)):
    """random events: a few columns, each with a frequent in-frame string, a rarer one and some out-of-frame noise"""
    read, col, off, ln, pool = [], [], [], [], bytearray()
    for c in rng.choice(L - 1, size=nsites, replace=False):
        for s, k in ((b"ACG", rng.integers(*per_site)), (b"TTTAAA", rng.integers(1, 8)), (b"GA", rng.integers(1, 8))):
            for r in rng.choice(R, size=int(k), replace=False):
                read.append(int(r)); col.append(int(c)); off.append(len(pool)); ln.append(len(s))
                pool += s
    return (np.array(read), np.array(col), np.array(off), np.array(ln), bytes(pool))


@pytest.fixture(scope="module")
def mixture():
    t = make_tables(SynthConfig(L=600, seed=7, minor_fracs=(0.3, 0.2), trunc=0.0))
    states = synth_states(t, 0, 900)
    labels = np.random.default_rng(1).integers(-1, 4, size=900)
    return t, states, labels


def test_group_counts_equal_k1_oracle_per_group(oracle, mixture):
    _, states, labels = mixture
    counts = hco.group_counts(states, labels, 3)
    for g in range(3):
        col, _ = oracle.pileup(np.ascontiguousarray(states[labels == g]), codons=False)
        np.testing.assert_array_equal(counts[g], col)


def test_reduces_to_fuse_when_every_column_is_covered(oracle, mixture):
    """With votes >= min_coverage everywhere U15 is U6-U8: every group's sequence is oracle.fuse's on that group's reads."""
    _, states, labels = mixture
    rng = np.random.default_rng(2)
    read, col, off, ln, pool = insertion_events(rng, len(labels), states.shape[1])
    counts = hco.group_counts(states, labels, 3)
    for g in range(3):
        votes = counts[g, :, :5].sum(axis=1)
        min_cov = int(votes.min())
        assert min_cov > 0
        mine = labels[read] == g
        seq = hco.consensus(counts[g], [(c, pool[o: o + n]) for c, o, n in zip(col[mine], off[mine], ln[mine])], min_coverage=min_cov)
        ref = oracle.fuse(counts[g], col[mine], off[mine], ln[mine], pool, min_coverage=min_cov)
        assert seq == ref
        assert "ACG" in seq or not mine.any()


def test_interior_thin_columns_become_n_and_ends_are_trimmed():
    A, C, G, T, D = 0, 1, 2, 3, 4
    col = col_of([[(A, 3)],              # thin: leading run, trimmed
                  [(C, 2), (G, 1)],      # thin
                  [(G, 12)],
                  [(T, 5)],              # thin inside: N
                  [(D, 11), (A, 1)],     # deletion wins: removed
                  [(A, 10), (C, 10)],    # tie: first maximum, A
                  [(C, 9), (T, 1)],      # exactly min_coverage
                  [],                    # no votes: thin inside
                  [(G, 10)],
                  [(T, 4)],              # thin: trailing run, trimmed
                  []])
    assert hco.consensus(col, min_coverage=10) == "GNACNG"
    # min_coverage 0 counts as 1: only the empty columns are thin, and they are trimmed at the end
    assert hco.consensus(col, min_coverage=0) == "ACGTACNGT"
    assert hco.consensus(col, min_coverage=100) == ""


def test_insertions_only_after_kept_columns():
    col = col_of([[(1, 2)], [(0, 20)], [(2, 20)], [(3, 4)], [(0, 20)], [(1, 3)]])
    ins = [(0, b"TTT")] * 3 + [(1, b"GGG")] * 15 + [(3, b"CCC")] * 4 + [(4, b"AAA")] * 11 + [(5, b"ACG")] * 3
    # after column 0 (trimmed) and column 5 (trimmed): dropped; after 1, 3 (thin but inside) and 4: spliced
    assert hco.consensus(col, ins, min_coverage=10, ins_distance=1) == "AGGGGNCCCAAAA"
    # spacing: 1 accepted, 3 too close, 4 is 3 away from 1
    assert hco.consensus(col, ins, min_coverage=10, ins_distance=3) == "AGGGGNAAAA"
    # support is judged against the column's own votes: 4 of 4 at column 3 passes, 11 of 20 passes, 10 of 20 would not
    assert hco.consensus(col, ins[:-3 - 1], min_coverage=10, ins_distance=1) == "AGGGGNCCCA"


def test_insertions_stay_in_their_group(mixture):
    _, states, labels = mixture
    target = np.nonzero(labels == 1)[0]
    read = np.concatenate([target, target])
    col = np.full(len(read), 250)
    pool = b"GATTAC"
    off = np.zeros(len(read), dtype=np.int64)
    ln = np.concatenate([np.full(len(target), 6), np.full(len(target), 3)])
    seqs = hco.haplotype_consensus(states, labels, 3, (read, col, off, ln, pool), min_coverage=1)
    plain = hco.haplotype_consensus(states, labels, 3, None, min_coverage=1)
    assert seqs[0] == plain[0] and seqs[2] == plain[2]
    assert seqs[1] != plain[1] and len(seqs[1]) == len(plain[1]) + 3        # GAT ties GATTAC on count, shorter first


def test_group_kernels_do_not_spill():
    """The grouped pile-up and consensus kernels compile for sm_100a without spills."""
    nvcc = shutil.which("nvcc", path="/usr/local/cuda/bin") or shutil.which("nvcc")
    if not nvcc:
        pytest.skip("nvcc not found")
    src = os.path.join(ROOT, "minorseq_b200", "csrc", "group.cu")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                          "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out.stderr)
    assert spills and all(s == ("0", "0") for s in spills), out.stderr
    assert "group_pileup_kernel" in out.stderr
