"""CPU: the in-frame indel restatement (indel_oracle.py, U19) on hand-built known answers, its p-values against mpmath, the
labels, the DRM grammar's new tokens (target_config.hpp), and that indel.cu compiles for sm_100a without spills."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import hypergeom_reference as ref
import indel_oracle as io

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
L = 30
GENES = [(1, 31)]            # ten codons, starts 0, 3, ..., 27; boundaries 2, 5, ..., 26


def base_states(R):
    return np.tile(np.array([i % 4 for i in range(L)], dtype=np.uint8), (R, 1))


def events(evs):
    """[(read, col, string)] -> (read, col, off, len, pool)"""
    pool, off = b"", []
    for _, _, x in evs:
        off.append(len(pool))
        pool += x.encode()
    return ([e[0] for e in evs], [e[1] for e in evs], off, [len(e[2]) for e in evs], pool)


def run(st, evs=None, **kw):
    start = io.start_bits(L, GENES)
    cnt, strings, tally = io.counts(st, events(evs or []), start)
    return cnt, strings, tally


def test_codon_deletion_counts():
    st = base_states(10)
    st[0, 6:9] = 4                       # codon 2 deleted
    st[1, 6:8] = 4                       # partial gap: not a deletion, not clean
    st[2, 7] = 5                         # N in the codon
    st[3, :4] = 7                        # does not span codon 0 or 1
    cnt, _, _ = run(st)
    assert cnt[6, 0] == 1 and cnt[7, 0] == 0 and cnt[3, 0] == 0
    hist = io._codon_hist(st, 6)
    assert hist.sum() == 7               # n_del = 1 + 7: the partial gap and the N are in neither term
    assert cnt[0, 1] == 9                # clean at columns 0 and 1: read 3 does not span them


def test_insertions_at_boundaries():
    st = base_states(12)
    evs = [(0, 5, "AAA"), (1, 5, "AAA"), (2, 5, "ccgGGT"), (3, 4, "AAA"),   # 3 and 6 bases at boundary 5; col 4 is inside a codon
           (4, 8, "AA"), (5, 8, "AAAA"), (6, 8, "ANA"), (7, 8, "AAX"),        # none counted
           (8, 11, "TTT"), (8, 11, "GGG"),                                   # two I ops on one column: the first decides
           (9, 14, "AA"), (9, 14, "CCC")]                                    # ... even when it is not counted
    st[1, 6] = 5                                                             # read 1 is not clean at c+1
    cnt, strings, tally = run(st, evs)
    assert strings == [(5, "AAA"), (5, "CCGGGT"), (11, "TTT")]
    assert list(tally) == [1, 1, 1]
    assert cnt[5, 1] == 11 and cnt[8, 1] == 12


def test_reads_outside_the_rank_are_not_tallied():
    st = base_states(4)
    evs = [(0, 5, "AAA"), (5, 5, "AAA"), (6, 5, "CCC")]
    start = io.start_bits(L, GENES)
    cnt, strings, tally = io.counts(st, events(evs), start, read0=3)     # this rank holds reads 3..6
    assert strings == [(5, "AAA"), (5, "CCC")] and list(tally) == [1, 1]


def test_known_answer_calls():
    R = 2000
    st = base_states(R)
    st[:40, 9:12] = 4                                    # 2 % codon-3 deletion
    evs = [(r, 14, "GGCGGC") for r in range(100, 140)]   # 2 % six-base insertion after codon 5
    cnt, strings, tally = run(st, evs)
    calls = io.call(st, cnt, strings, tally, GENES)
    assert [(c["kind"], c["col"], c["count"], c["coverage"]) for c in calls] == [(0, 9, 40, 2000), (1, 14, 40, 2000)]
    for c in calls:
        e = c["expected"]
        assert float(ref.rel_err(c["pvalue"], ref.k2_pvalue(c["count"], c["coverage"], e))) < 1e-9
    d, i = calls
    assert io.label(0, d["ref_codon"], -1, d["codon_index"] + 1) == "R4del"                       # CGT
    assert io.label(1, i["ref_codon"], i["next_codon"], i["codon_index"] + 1, i["inserted"]) == "T5_Y6insGG"   # ACG | TAC
    assert i["codon_index"] == 4 and i["inserted"] == "GGCGGC"


def test_no_call_at_the_error_rate():
    R = 2000
    st = base_states(R)
    st[:1, 9:12] = 4
    evs = [(0, 14, "GGC")]
    cnt, strings, tally = run(st, evs)
    assert io.call(st, cnt, strings, tally, GENES) == []


def test_percentage_filters_and_region():
    R = 1000
    st = base_states(R)
    st[:50, 9:12] = 4
    cnt, strings, tally = run(st)
    assert len(io.call(st, cnt, strings, tally, GENES)) == 1
    assert io.call(st, cnt, strings, tally, GENES, min_perc=5.0) == []          # 50 / 1000 = 5 %: not above
    assert io.call(st, cnt, strings, tally, GENES, max_perc=5.0) == []
    assert io.call(st, cnt, strings, tally, GENES, region=(13, 31)) == []       # codon 3 (columns 9-11) outside


def test_insertion_needs_both_codons_tested():
    R = 1000
    st = base_states(R)
    evs = [(r, 14, "GGC") for r in range(50)]
    cnt, strings, tally = run(st, evs)
    assert [c["col"] for c in io.call(st, cnt, strings, tally, GENES)] == [14]
    assert io.call(st, cnt, strings, tally, GENES, region=(1, 16)) == []        # the codon at 15 is outside the region


@pytest.mark.parametrize("k,n,e", [(1, 1, 0), (2, 2, 1), (40, 2000, 1), (40, 6000, 1), (120, 6000, 1), (3, 10 ** 6, 1),
                                   (200, 10 ** 6, 27), (5, 7, 5), (160, 10 ** 5, 100)])
def test_pvalues_against_mpmath(k, n, e):
    assert float(ref.rel_err(io.fisher_p(k, n, e), ref.k2_pvalue(k, n, e))) < 1e-9


def test_expected_counts():
    assert io.expected(6000, 3e-3 ** 3) == 1
    assert io.expected(6000, 3e-3 ** 6) == 1
    assert io.expected(10, 1.0) == 10 and io.expected(0, 0.5) == 0


def test_translation_of_inserted_strings():
    assert io.translate("TCTTCT") == "SS"
    assert io.translate("TAATGA") == "**"
    act, agt = 16 * 0 + 4 * 1 + 3, 16 * 0 + 4 * 2 + 3                # ACT = T, AGT = S
    assert io.label(1, act, agt, 69, "TCTTCT") == "T69_S70insSS"
    assert io.label(1, act, agt, 69, "TAA") == "T69_S70ins*"
    assert io.label(0, 16 * 2 + 4 * 0 + 1, -1, 67) == "D67del"       # GAC = D
    assert io.label(1, -1, agt, 69, "TCT") == "?69_S70insS"


HOST_TEST = r"""
#include <cstdio>
#include "target_config.hpp"
int main() {
    using namespace mscfg;
    auto t = [](const char* tok, int pos, char ref, int kind, char aa) {   // kind 0 substitution to aa, 1 insertion, 2 deletion
        const DrmPosition p = parse_drm_position(tok);
        return kind == 0 ? drm_matches(p, pos, ref, aa) : drm_matches_indel(p, pos, ref, kind == 1);
    };
    int bad = 0;
    auto expect = [&](bool got, bool want, const char* what) { if (got != want) { puts(what); ++bad; } };
    expect(t("69ins", 69, 'T', 1, 0), true, "69ins insertion");
    expect(t("T69ins", 69, 'T', 1, 0), true, "T69ins insertion");
    expect(t("T69ins", 69, 'S', 1, 0), false, "T69ins wrong ref");
    expect(t("T69ins", 70, 'T', 1, 0), false, "T69ins wrong position");
    expect(t("69ins", 69, 'T', 2, 0), false, "69ins deletion");
    expect(t("67del", 67, 'D', 2, 0), true, "67del deletion");
    expect(t("D67del", 67, 'D', 2, 0), true, "D67del deletion");
    expect(t("D67del", 67, 'D', 1, 0), false, "D67del insertion");
    expect(t("D67del", 67, 'N', 2, 0), false, "D67del wrong ref");
    expect(t("69", 69, 'T', 1, 0), true, "bare position insertion");
    expect(t("69", 69, 'T', 2, 0), true, "bare position deletion");
    expect(t("T69", 69, 'T', 1, 0), true, "T69 insertion");
    expect(t("T69D", 69, 'T', 1, 0), false, "T69D insertion");
    expect(t("T69D", 69, 'T', 0, 'D'), true, "T69D substitution");
    expect(t("T69D", 69, 'T', 0, 'N'), false, "T69D other substitution");
    expect(t("69", 69, 'T', 0, 'N'), true, "bare position substitution");
    expect(t("T69ins", 69, 'T', 0, 'N'), false, "T69ins substitution");
    expect(t("D67del", 67, 'D', 0, 'N'), false, "D67del substitution");
    expect(t("D67del", 67, 'D', 0, 'd'), false, "D67del substitution d");
    expect(t("M184VI", 184, 'M', 0, 'V'), true, "M184VI");
    expect(t("M184VI", 184, 'M', 0, 'I'), true, "M184VI I");
    expect(t("M184VI", 184, 'M', 2, 0), false, "M184VI deletion");
    const DrmPosition p = parse_drm_position("M184VI");
    expect(p.mut_aas == "VI" && p.ref_aa == 'M' && p.pos == 184 && p.kind == kDrmSubstitution, true, "M184VI parse");
    const DrmPosition q = parse_drm_position("69ins");
    expect(q.mut_aas.empty() && q.ref_aa == '*' && q.pos == 69 && q.kind == kDrmInsertion && q.text == "69ins", true, "69ins parse");
    return bad;
}
"""


def test_drm_grammar_indel_tokens(tmp_path):
    gxx = shutil.which("g++", path="/usr/bin") or shutil.which("g++")
    if not gxx:
        pytest.skip("g++ not found")
    src = tmp_path / "drm.cpp"
    src.write_text(HOST_TEST)
    exe = tmp_path / "drm"
    out = subprocess.run([gxx, "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "minorseq_b200", "host"), "-o", str(exe), str(src)],
                         capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    run = subprocess.run([str(exe)], capture_output=True, text=True)
    assert run.returncode == 0, run.stdout


def test_indel_kernels_do_not_spill():
    """The count, event and test kernels compile for sm_100a without spills."""
    nvcc = shutil.which("nvcc", path="/usr/local/cuda/bin") or shutil.which("nvcc")
    if not nvcc:
        pytest.skip("nvcc not found")
    src = os.path.join(ROOT, "minorseq_b200", "csrc", "indel.cu")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false", "-Xptxas", "-v",
                          "-c", src, "-o", os.devnull], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", out.stderr)
    assert spills and all(s == ("0", "0") for s in spills), out.stderr
    for k in ("indel_count_kernel", "indel_ins_kernel", "indel_test_kernel"):
        assert k in out.stderr
