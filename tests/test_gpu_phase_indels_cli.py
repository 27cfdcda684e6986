"""`juliet --mode-phasing --indels --phase-indels` (U20) on a BAM written with I / D CIGARs: the haplotypes, their `indels`, the
calls' `haplotype_hit` and the linkage rows against the numpy restatement (phase_indel_oracle.py), --drm-only, the missing-option
errors, the report without --phase-indels, and --gpus 2 equal to one GPU."""
import subprocess

import pytest

import phase_indel_oracle as po
from minorseq_b200.api import CODONS
from test_gpu_indels_cli import _run, juliet, sample  # noqa: F401  (fixtures)
from test_host_cpp import _gpu_count

pytestmark = pytest.mark.gpu


def events(evs):
    pool, off = b"", []
    for _, _, x in evs:
        off.append(len(pool))
        pool += x.encode()
    return ([e[0] for e in evs], [e[1] for e in evs], off, [len(e[2]) for e in evs], pool)


def restated(rep, conf, st, evs):
    begin = {g["name"]: g["begin"] for g in conf["genes"]}
    sub = sorted({(begin[g["name"]] - 1 + 3 * (vp["ref_position"] - 1), CODONS.index(vc["codon"]))
                  for g in rep["genes"] for vp in g.get("variant_positions", []) for va in vp["variant_amino_acids"] for vc in va["variant_codons"]})
    calls = rep["indels"]["calls"]
    dels = sorted({c["abs_pos"] - 1 for c in calls if c["type"] == "deletion"})
    ins = sorted({(c["abs_pos"] - 1, c["inserted"]) for c in calls if c["type"] == "insertion"})
    B, M, f = po.bits(st, sub, dels, ins, events(evs))
    return sub, dels, ins, B, M, f


@pytest.mark.parametrize("drm_only", [False, True])
def test_phase_indels_report(juliet, sample, tmp_path, drm_only, oracle):
    t, st, evs, bam, cpath, conf = sample
    extra = ["--drm-only"] if drm_only else []
    rep0, js0, _ = _run(juliet, ["--config", cpath, "--mode-phasing", "--indels", "--linkage"] + extra + [bam], tmp_path, "base")
    rep, js, html = _run(juliet, ["--config", cpath, "--mode-phasing", "--indels", "--linkage", "--phase-indels"] + extra + [bam], tmp_path, "pi")
    assert '"haplotype_hit": [' in js and all("indels" not in h for h in rep0["haplotypes"])
    assert all("haplotype_hit" not in c for c in rep0["indels"]["calls"])
    calls, haps = rep["indels"]["calls"], rep["haplotypes"]
    assert [{k: v for k, v in c.items() if k != "haplotype_hit"} for c in calls] == rep0["indels"]["calls"]
    assert len(calls) >= 2 and (not drm_only or all(c["known_drm"] for c in calls))
    sub, dels, ins, B, M, f = restated(rep, conf, st, evs)
    ph = po.phase(B, f)
    nrep = ph["nreported"]
    assert [h["reads"] for h in haps] == ph["counts"][:nrep].tolist()
    cats = rep["haplotype_read_categories"]
    c = ph["counters"]
    assert (cats["reported"], cats["insufficient_coverage"], cats["unsuitable"], cats["unsuitable_gaps"], cats["unsuitable_heteroduplex"],
            cats["unsuitable_partial"]) == (c["reported"], c["insufficient"], c["damaged"], c["gaps"], c["heteroduplex"], c["partial"])
    V = len(sub)
    for k, h in enumerate(haps):
        assert len(h["codons"]) == V
        bit = lambda v: bool((int(ph["patterns"][k][v >> 5]) >> (v & 31)) & 1)
        want = []
        for key in range(V, V + len(dels) + len(ins)):
            if bit(key):
                for cc in calls:
                    kk = V + dels.index(cc["abs_pos"] - 1) if cc["type"] == "deletion" else V + len(dels) + ins.index((cc["abs_pos"] - 1, cc["inserted"]))
                    if kk == key:
                        want.append(cc["gene"] + " " + cc["label"])
        assert h["indels"] == want
        for cc in calls:
            assert cc["haplotype_hit"][k] == (cc["gene"] + " " + cc["label"] in h["indels"])
    assert any(any(cc["haplotype_hit"]) for cc in calls)
    lk = po.linkage(B, M, po.key_columns(sub, dels, ins), oracle.fisher)
    pairs = rep["linkage"]["pairs"]
    assert len(pairs) == len(lk["pairs"]) and rep["linkage"]["tested_pairs"] == lk["ntested"]
    for p, w in zip(pairs, lk["pairs"]):
        assert (p["both"], p["a_only"], p["b_only"], p["neither"]) == w[2:6]
        for side, key in (("a", w[0]), ("b", w[1])):
            if key >= V + len(dels):
                assert p[side]["codon"] == "+" + ins[key - V - len(dels)][1]
            elif key >= V:
                assert p[side]["codon"] == "---" and p[side]["abs_pos"] == dels[key - V] + 1
    assert "In-frame Insertions and Deletions" in html


def test_fasta_of_the_deletion_haplotype(juliet, sample, tmp_path):
    t, st, evs, bam, cpath, conf = sample
    out = tmp_path / "h.fasta"
    rep, _, _ = _run(juliet, ["--config", cpath, "--mode-phasing", "--indels", "--phase-indels", bam, str(out)], tmp_path, "fa")
    seqs = {}
    for block in out.read_text().split(">")[1:]:
        head, *lines = block.strip().split("\n")
        seqs[head.split("|")[1]] = "".join(lines)
    dels = [c for c in rep["indels"]["calls"] if c["type"] == "deletion"]
    assert dels
    d = dels[0]
    name = d["gene"] + " " + d["label"]
    carriers = [h["name"] for h in rep["haplotypes"] if name in h["indels"]]
    others = [h["name"] for h in rep["haplotypes"] if name not in h["indels"]]
    assert carriers and others
    s = d["abs_pos"] - 1
    flank = t.refseq[s - 12: s] + t.refseq[s + 3: s + 15]
    assert flank in seqs["haplotype_" + carriers[0]]
    assert flank not in seqs["haplotype_" + others[0]]


def test_missing_options(juliet, sample, tmp_path):
    _, _, _, bam, cpath, _ = sample
    for args in (["--phase-indels"], ["--phase-indels", "--mode-phasing"], ["--phase-indels", "--indels"]):
        res = subprocess.run([juliet, "--config", cpath] + args + [bam, str(tmp_path / "x.json")], capture_output=True, text=True)
        assert res.returncode != 0 and "--phase-indels" in res.stderr


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_phase_indels_two_gpus(juliet, sample, tmp_path):
    _, _, _, bam, cpath, _ = sample
    args = ["--config", cpath, "--mode-phasing", "--indels", "--linkage", "--haplotype-abundance", "--phase-indels"]
    _, js1, h1 = _run(juliet, args + [bam], tmp_path, "one")
    _, js2, h2 = _run(juliet, args + ["--gpus", "2", bam], tmp_path, "two")
    assert js1.replace(" --gpus 2", "") == js2.replace(" --gpus 2", "") and h1.replace(" --gpus 2", "") == h2.replace(" --gpus 2", "")
