"""Read alignment's restatement (U16, tests/align_oracle.c) on hand-made known answers, and against a full-matrix overlap DP."""
import os
import random
import re
import shutil
import subprocess

import pytest

from align_oracle import AlignOracle, revcomp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rand_seq(rng, n):
    return "".join(rng.choice("ACGT") for _ in range(n))


@pytest.fixture(scope="module")
def ao():
    return AlignOracle()


@pytest.fixture(scope="module")
def ref():
    return rand_seq(random.Random(7), 2000)


def one(ao, ref, read, min_seeds=10):
    ao.set_reference(ref)
    return ao.align([read], min_seeds)[0]


def test_read_equal_to_reference(ao, ref):
    assert one(ao, ref, ref) == (True, 0, 0, 2 * len(ref), f"{len(ref)}=")
    assert one(ao, ref, ref[300:1300]) == (True, 0, 300, 2000, "1000=")


def test_one_substitution_is_one_x(ao, ref):
    r = list(ref[300:1300])
    r[400] = "A" if r[400] != "A" else "C"
    assert one(ao, ref, "".join(r)) == (True, 0, 300, 2 * 999 - 3, "400=1X599=")


def test_homopolymer_indels_land_leftmost(ao, ref):
    ref2 = ref[:1000] + "CAAAAAAG" + ref[1000:]
    dele = ref2[500:1001] + "AAAAA" + ref2[1007:1500]        # one A fewer
    ins = ref2[500:1001] + "AAAAAAA" + ref2[1007:1500]       # one A more
    assert one(ao, ref2, dele) == (True, 0, 500, 2 * 999 - 4, "501=1D498=")
    assert one(ao, ref2, ins) == (True, 0, 500, 2 * 1000 - 4, "501=1I499=")


def test_reverse_complement_same_cigar(ao, ref):
    r = list(ref[300:1300])
    r[10] = "G" if r[10] != "G" else "T"
    del r[600]
    r = "".join(r)
    fwd = one(ao, ref, r)
    rev = one(ao, ref, revcomp(r))
    assert fwd[0] and rev[0] and fwd[1] == 0 and rev[1] == 1
    assert fwd[2:] == rev[2:]


def test_overhangs_are_soft_clips(ao, ref):
    rng = random.Random(3)
    sub = ref[:1200]
    head, tail = rand_seq(rng, 70), rand_seq(rng, 45)
    assert one(ao, sub, head + sub + tail) == (True, 0, 0, 2400, f"70S1200=45S")   # longer than the reference: S on both sides
    assert one(ao, ref, head + ref[:500]) == (True, 0, 0, 1000, "70S500=")
    assert one(ao, ref, ref[1700:] + tail) == (True, 0, 1700, 600, "300=45S")


def test_unmapped_reads(ao, ref):
    rng = random.Random(5)
    ao.set_reference(ref)
    res = ao.align([ref[100:114], rand_seq(rng, 3000), ""])
    assert all(r == (False, 0, -1, 0, "") for r in res)


def test_min_seeds_boundary(ao, ref):
    # a read of 15 + 4 (n - 1) bases has n strided k-mers, all unique in a random 2 kb reference
    at, under = ref[600:600 + 15 + 4 * 9], ref[600:600 + 15 + 4 * 8]
    ao.set_reference(ref)
    assert ao.align([at], 10)[0][0] and not ao.align([under], 10)[0][0]
    assert ao.align([under], 9)[0][0]
    assert ao.align([at], 11)[0] == (False, 0, -1, 0, "")


def ops_of(cigar):
    return [(int(n), op) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", cigar)]


def test_long_indels_are_followed_by_the_band(ao, ref):
    """A 40-base deletion and a 30-base insertion: the band follows the path across them (the optimum of the full
    matrix); with linear gaps a long gap may be split by chance matches, so only its total is fixed."""
    rng = random.Random(11)
    dele = ref[200:800] + ref[840:1500]
    ins = ref[200:800] + rand_seq(rng, 30) + ref[800:1500]
    for read, span, gap_op, gap in ((dele, 1300, "D", 40), (ins, 1300, "I", 30)):
        res = one(ao, ref, read)
        ops = ops_of(res[4])
        assert res[0] and res[2] == 200 and res[3] == ao.overlap_score(read, ref), res
        assert "S" not in res[4] and sum(n for n, op in ops if op in "=XD") == span
        assert sum(n for n, op in ops if op == gap_op) >= gap


def mutate(rng, s, sub=0.03, indel=0.01):
    out = []
    for c in s:
        x = rng.random()
        if x < sub:
            out.append(rng.choice([b for b in "ACGT" if b != c]))
        elif x < sub + indel:
            continue
        elif x < sub + 2 * indel:
            out.append(c + rng.choice("ACGT"))
        else:
            out.append(c)
    return "".join(out)


@pytest.mark.parametrize("seed", range(12))
def test_band_score_equals_full_matrix(ao, seed):
    """On reads whose optimal path stays well inside the band, the banded score is the full-matrix optimum.  The read's
    first 20 bases are exact, so the first seed sits on the path's start diagonal (a path cannot start before k0)."""
    rng = random.Random(100 + seed)
    ref = rand_seq(rng, rng.randint(200, 700))
    a = rng.randint(0, len(ref) // 3)
    b = rng.randint(2 * len(ref) // 3, len(ref))
    read = ref[a:a + 20] + mutate(rng, ref[a + 20:b - 20]) + ref[b - 20:b]
    ao.set_reference(ref)
    res = ao.align([read], 1)[0]
    assert res[0] and res[1] == 0
    assert res[3] == ao.overlap_score(read, ref)


def test_align_kernels_do_not_spill():
    """The seed, band and compaction kernels compile for sm_100a without spills."""
    nvcc = shutil.which("nvcc", path="/usr/local/cuda/bin") or shutil.which("nvcc")
    if not nvcc:
        pytest.skip("nvcc not found")
    src = os.path.join(ROOT, "minorseq_b200", "csrc", "align.cu")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                          "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out.stderr)
    assert len(spills) == 3 and all(s == ("0", "0") for s in spills), out.stderr
    assert "align_band_kernel" in out.stderr and "align_seed_kernel" in out.stderr
