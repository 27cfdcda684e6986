"""CPU: the restatement of in-frame indels in phasing (phase_indel_oracle.py, U20) on hand-built known answers, its agreement
with the C restatement of phasing when there are no indel keys, and that phase_indel.cu compiles for sm_100a without spills
while phase_bits_kernel keeps its registers."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import phase_indel_oracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = 30


def base_states(R):
    return np.tile(np.array([i % 4 for i in range(L)], dtype=np.uint8), (R, 1))


def codon(st_row, s):
    return 16 * int(st_row[s]) + 4 * int(st_row[s + 1]) + int(st_row[s + 2])


def events(evs):
    pool, off = b"", []
    for _, _, x in evs:
        off.append(len(pool))
        pool += x.encode()
    return ([e[0] for e in evs], [e[1] for e in evs], off, [len(e[2]) for e in evs], pool)


def test_full_deletion_at_a_substitution_codon_is_phased():
    st = base_states(3)
    sub = [(6, codon(st[0], 6)), (12, codon(st[0], 12))]
    st[1, 6:9] = 4                                   # carries the deletion in full
    B, M, f = po.bits(st, sub, [6], [])
    assert list(f) == [0, 0, 0]
    assert B[1].tolist() == [False, True, True] and M[1].tolist() == [False, True, True]
    assert B[0].tolist() == [True, True, False] and M[0].tolist() == [True, True, True]
    # without the deletion key the same read is a gap (the rule of phasing today)
    _, _, f0 = po.bits(st, sub, [], [])
    assert list(f0) == [0, po.GAP, 0]


@pytest.mark.parametrize("cols", [[6], [7], [6, 7], [7, 8]])
def test_partial_gap_in_a_deletion_codon_is_a_gap(cols):
    st = base_states(2)
    st[1, cols] = 4
    B, M, f = po.bits(st, [(6, codon(st[0], 6))], [6], [])
    assert list(f) == [0, po.GAP] and not B[1].any() and not M[1].any()
    # the deletion key alone judges its columns the same way
    _, _, f2 = po.bits(st, [], [6], [])
    assert list(f2) == [0, po.GAP]


def test_n_at_an_insertion_boundary_is_heteroduplex():
    st = base_states(3)
    st[1, 9] = 5
    st[2, 8] = 5                                     # not a column of the key
    B, M, f = po.bits(st, [], [], [(8 + 1, "AAA")])
    assert list(f) == [0, po.HET, 0]
    B, M, f = po.bits(st, [], [], [(8, "AAA")])
    assert list(f) == [0, po.HET, po.HET] and M[:, 0].tolist() == [True, False, False]


def test_unspanned_c_plus_1_is_partial():
    st = base_states(2)
    st[1, 12:] = 7
    B, M, f = po.bits(st, [], [], [(11, "AAA")])
    assert list(f) == [0, po.PARTIAL] and M[:, 0].tolist() == [True, False]


def test_first_event_decides():
    st = base_states(5)
    evs = [(0, 11, "AAA"), (1, 11, "CCC"), (1, 11, "AAA"),       # read 1: the second event does not count
           (2, 11, "aaa"), (3, 11, "AA"), (3, 11, "AAA"),        # lower case counts; an out-of-frame first event hides the rest
           (4, 14, "AAA")]                                        # another column
    B, M, f = po.bits(st, [], [], [(11, "AAA"), (11, "CCC")], events(evs))
    assert B[:, 0].tolist() == [True, False, True, False, False]
    assert B[:, 1].tolist() == [False, True, False, False, False]
    assert M.all() and not f.any()
    st[0, 12] = 4                                                 # no longer clean at c+1: B = 0 and damaged
    B, M, f = po.bits(st, [], [], [(11, "AAA")], events(evs))
    assert not B[0, 0] and f[0] == po.GAP


def test_other_frame_codon_over_a_deletion():
    st = base_states(4)
    sub = [(7, codon(st[0], 7)), (4, codon(st[0], 4))]           # codons 7-9 and 4-6 overlap the deletion 6-8 partly
    st[1, 6:9] = 4                                                # full deletion: neither codon is damage
    st[2, 6:8] = 4                                                # partial gap: a gap
    st[3, 6:9] = 4
    st[3, 9] = 5                                                  # full deletion, but column 9 of codon 7 is an N
    B, M, f = po.bits(st, sub, [6], [])
    assert list(f) == [0, 0, po.GAP, po.HET]
    assert B[1].tolist() == [False, False, True] and M[1].tolist() == [False, False, True]


def test_keys_across_a_word():
    rng = np.random.default_rng(1)
    Ls = 120
    st = np.tile(rng.integers(0, 4, Ls).astype(np.uint8), (4, 1))
    sub = [(3 * i, codon(st[0], 3 * i)) for i in range(31)]      # bits 0-30
    dels = [93, 96]                                               # bits 31, 32
    ins = [(101, "GGG"), (104, "TTT")]                            # bits 33, 34
    st[1, 93:96] = 4
    st[2, 96:99] = 4
    evs = [(1, 101, "GGG"), (2, 104, "TTT"), (3, 101, "GGG"), (3, 104, "TTT")]
    B, M, f = po.bits(st, sub, dels, ins, events(evs))
    assert not f.any()
    W = po.words(B)
    assert W.shape == (4, 2)
    full = (1 << 31) - 1                                          # every read carries the 31 substitution keys
    assert W.tolist() == [[full, 0], [full | 1 << 31, 0b10], [full, 0b101], [full, 0b110]]
    ph = po.phase(B, f, min_reads=1)
    assert sorted(ph["counts"].tolist()) == [1, 1, 1, 1] and ph["counters"]["reported"] == 4


def test_no_indel_keys_equals_phasing(oracle):
    from minorseq_b200.synth import SynthConfig, make_tables, synth_states
    t = make_tables(SynthConfig(L=600, seed=77, n_rate=2e-2, trunc=0.3))
    st = synth_states(t, 0, 3000)
    rng = np.random.default_rng(3)
    for r in rng.choice(3000, 200, replace=False):
        s = int(rng.integers(0, 590))
        st[r, s: s + int(rng.integers(1, 4))] = 4
    sub = sorted({(int(c), int(k)) for c, k in zip(rng.integers(0, 598, 40), rng.integers(0, 64, 40))})
    sub += [(3, codon(st[0], 3)) if (st[0, 3:6] < 4).all() else (3, 0)]
    sub = sorted(set(sub))
    B, M, f = po.bits(st, sub, [], [])
    bits, flags = oracle.phase_bits(st, [k[0] for k in sub], [k[1] for k in sub])
    assert np.array_equal(po.words(B), bits) and np.array_equal(f, flags)
    g = oracle.phase_group(bits, flags, len(sub))
    ph = po.phase(B, f)
    assert np.array_equal(ph["counts"], g["counts"]) and np.array_equal(ph["patterns"], g["patterns"])
    assert np.array_equal(ph["hap_id"], g["hap_id"]) and ph["counters"] == g["counters"] and ph["nreported"] == g["nreported"]


def test_linkage_and_abundance_take_the_indel_keys(oracle):
    R = 400
    st = np.tile(np.array([i % 4 for i in range(60)], dtype=np.uint8), (R, 1))
    sub = [(30, 16 * 3 + 4 * 0 + 1)]                  # a minor codon at 30
    carriers = np.arange(0, R, 4)
    st[carriers, 30:33] = [3, 0, 1]
    st[carriers, 9:12] = 4                            # travels with a deletion at 9 ...
    evs = [(int(r), 44, "AAC") for r in carriers]     # ... and an insertion at 44
    B, M, f = po.bits(st, sub, [9], [(44, "AAC")], events(evs))
    assert not f.any() and B[carriers].all() and not B[np.setdiff1d(np.arange(R), carriers)].any()
    cols = po.key_columns(sub, [9], [(44, "AAC")])
    assert cols == [30, 9, 44]
    lk = po.linkage(B, M, cols, oracle.fisher)
    assert [(p[0], p[1], p[2], p[9]) for p in lk["pairs"]] == [(0, 1, 100, 1), (0, 2, 100, 1), (1, 2, 100, 1)]
    ph = po.phase(B, f)
    ab = po.abundance(B, M, ph["patterns"][: ph["nreported"]])
    assert ab["unique_reads"].tolist() == [300, 100]


def _ptxas(src):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                          "-c", "-o", os.devnull, os.path.join(ROOT, "minorseq_b200", "csrc", src)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return out.stderr


def _kernel_lines(log, name):
    """{mangled name: (stack / spill line, registers line)} of the kernels whose name contains `name`"""
    res, cur = {}, None
    for line in log.splitlines():
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1) if name in m.group(1) else None
            if cur:
                res[cur] = []
        elif cur and ("stack frame" in line or "registers" in line):
            res[cur].append(line.split(":", 1)[-1].strip())
    return res


def test_phase_indel_kernels_do_not_spill():
    log = _ptxas("phase_indel.cu")
    k = _kernel_lines(log, "phase_indel")
    assert len(k) == 3
    for lines in k.values():
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in lines[0]


def test_phase_bits_kernel_unchanged():
    """the indel keys leave phase_bits_kernel as it was: same registers, no stack (sm_100a, CUDA 12.9)"""
    k = _kernel_lines(_ptxas("phase.cu"), "phase_bits_kernel")
    got = {("ILb1E" in n): lines for n, lines in k.items()}
    assert got[False] == ["0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", "Used 56 registers, used 0 barriers"]
    assert got[True] == ["0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", "Used 64 registers, used 0 barriers"]
