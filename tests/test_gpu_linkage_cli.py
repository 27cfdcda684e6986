"""`juliet --linkage`: the report's "linkage" block against the column-state restatement (linkage_oracle.py), the report
without --linkage unchanged, and --gpus 2 equal to one GPU."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

import linkage_oracle as lo
from minorseq_b200 import build as msbuild
from minorseq_b200.api import translate
from minorseq_b200.synth import SynthConfig, make_tables, synth_states
from test_host_cpp import _gpu_count, _make_bam

pytestmark = pytest.mark.gpu

BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minorseq_b200", "bin")
FIXED = "2026-01-01T00:00:00.000Z"


@pytest.fixture(scope="module")
def juliet():
    msbuild.build_library()
    msbuild.build_host()
    return os.path.join(BIN, "juliet")


def _codon(k):
    return "".join("ACGT"[(k >> s) & 3] for s in (4, 2, 0))


def _run(juliet, args, tmp_path, tag):
    oj, oh = str(tmp_path / f"{tag}.json"), str(tmp_path / f"{tag}.html")
    env = dict(os.environ, MS_FIXED_TIMESTAMP=FIXED)
    res = subprocess.run([juliet] + args + [oj, oh], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr
    rep = json.load(open(oj))
    cmd = rep["input"]["command_line"]
    return rep, open(oj).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X"), \
        open(oh).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X")


def test_juliet_cli_linkage_matches_oracle(juliet, oracle, tmp_path):
    cfg = SynthConfig(L=900, seed=79, n_rate=2e-2, trunc=0.05, ins=0.0)
    t = make_tables(cfg)
    st = synth_states(t, 0, 20000)
    bam = str(tmp_path / "in.bam")
    _make_bam(bam, t, st)
    conf = {"genes": [{"name": "geneA", "begin": 1, "end": 451}, {"name": "geneB", "begin": 452, "end": 899}],
            "referenceName": "synthetic_ref", "referenceSequence": t.refseq, "version": "test"}
    cpath = tmp_path / "cfg.json"
    cpath.write_text(json.dumps(conf))
    rep, js, html = _run(juliet, ["--config", str(cpath), "--linkage", bam], tmp_path, "lk")
    # the same run without --linkage: the same report minus the block, and no HTML section
    rep0, js0, html0 = _run(juliet, ["--config", str(cpath), bam], tmp_path, "plain")
    lk = rep.pop("linkage")
    rep["input"]["command_line"] = rep0["input"]["command_line"] = ""
    assert rep == rep0
    assert '"linkage"' not in js0 and "Variant Linkage" not in html0
    section = re.compile(r'<details open><summary>Variant Linkage</summary>.*?</details>\n', re.S)
    assert len(section.findall(html)) == 1 and section.sub("", html) == html0

    keep = (st & 7 != 7).any(axis=1)
    sto = st[keep]
    genes = [(1, 451), (452, 899)]
    mask = np.zeros(900, dtype=np.uint8)
    for (b, e) in genes:
        mask[b - 1: e - 3: 3] = 1
    _, codon = oracle.pileup(sto, mask)
    ov = oracle.call(codon, genes, refseq=t.refseq)
    keys = sorted({(v.col, v.codon) for v in ov})
    want = lo.linkage(sto, keys, oracle.fisher, alpha=0.01)
    assert (lk["min_reads"], lk["alpha"], lk["tested_pairs"]) == (10, 0.01, want["ntested"])
    assert len(want["pairs"]) > 0 and len(lk["pairs"]) == len(want["pairs"])
    labels = {}
    for ov_ in ov:
        labels.setdefault((ov_.col, ov_.codon), []).append(
            f"{('geneA', 'geneB')[ov_.gene]} {translate(ov_.ref_codon)}{ov_.codon_index + 1}{translate(ov_.codon)}")
    for got, p in zip(lk["pairs"], want["pairs"]):
        v, w = p[0], p[1]
        assert got["a"] == {"abs_pos": keys[v][0] + 1, "codon": _codon(keys[v][1]), "labels": labels[keys[v]]}
        assert got["b"] == {"abs_pos": keys[w][0] + 1, "codon": _codon(keys[w][1]), "labels": labels[keys[w]]}
        assert (got["both"], got["a_only"], got["b_only"], got["neither"]) == p[2:6]
        assert got["reads"] == sum(p[2:6])
        assert got["relation"] == ("linked" if p[9] == lo.LINKED else "exclusive")
        assert abs(got["d_prime"] - p[6]) <= 1e-12 and abs(got["r2"] - p[7]) <= 1e-12
        assert abs(got["pValue"] - p[8]) <= 1e-9 * p[8] + 1e-300
        assert got["pValueCorrected"] == pytest.approx(min(1.0, p[8] * want["ntested"]), rel=1e-9, abs=1e-300)


def test_juliet_cli_linkage_with_phasing_two_gpus_equal_one(juliet, tmp_path):
    """`--mode-phasing --linkage --gpus 2`: the linkage counts are summed over the ranks inside the library; the report is
    byte-identical to one GPU's."""
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    t = make_tables(SynthConfig(L=900, seed=78, n_rate=2e-3, trunc=0.05, ins=2e-3))
    st = synth_states(t, 0, 20001)
    bam = str(tmp_path / "in.bam")
    _make_bam(bam, t, st)
    outs = {}
    for n in (1, 2):
        rep, js, html = _run(juliet, ["--mode-phasing", "--linkage", "--gpus", str(n), bam], tmp_path, f"g{n}")
        assert len(rep["linkage"]["pairs"]) > 0 and len(rep["haplotypes"]) >= 2
        outs[n] = (js, html)
    assert outs[1] == outs[2]
