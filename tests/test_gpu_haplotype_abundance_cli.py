"""`juliet --mode-phasing --haplotype-abundance`: the report's "haplotype_abundance" block against the numpy restatement
(haplotype_abundance_oracle.py) run on the BAM's reads, the rest of the report unchanged, the HTML section only with the
option, the option refused without --mode-phasing, and --gpus 2 equal to one GPU."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

import haplotype_abundance_oracle as ha
from minorseq_b200 import build as msbuild
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


def _run(juliet, args, tmp_path, tag):
    oj, oh = str(tmp_path / f"{tag}.json"), str(tmp_path / f"{tag}.html")
    env = dict(os.environ, MS_FIXED_TIMESTAMP=FIXED)
    res = subprocess.run([juliet] + args + [oj, oh], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr
    rep = json.load(open(oj))
    cmd = rep["input"]["command_line"]
    return rep, open(oj).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X"), \
        open(oh).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X")


def test_juliet_cli_abundance_matches_oracle(juliet, oracle, tmp_path):
    cfg = SynthConfig(L=900, seed=81, n_rate=2e-2, trunc=0.05, ins=0.0)
    t = make_tables(cfg)
    st = synth_states(t, 0, 20000)
    bam = str(tmp_path / "in.bam")
    _make_bam(bam, t, st)
    conf = {"genes": [{"name": "geneA", "begin": 1, "end": 451}, {"name": "geneB", "begin": 452, "end": 899}],
            "referenceName": "synthetic_ref", "referenceSequence": t.refseq, "version": "test"}
    cpath = tmp_path / "cfg.json"
    cpath.write_text(json.dumps(conf))
    rep, js, html = _run(juliet, ["--config", str(cpath), "--mode-phasing", "--haplotype-abundance", bam], tmp_path, "ab")
    rep0, js0, html0 = _run(juliet, ["--config", str(cpath), "--mode-phasing", bam], tmp_path, "plain")
    ab = rep.pop("haplotype_abundance")
    rep["input"]["command_line"] = rep0["input"]["command_line"] = ""
    assert rep == rep0
    assert '"haplotype_abundance"' not in js0 and "Haplotype Abundance" not in html0
    section = re.compile(r'<details open><summary>Haplotype Abundance</summary>.*?</details>\n', re.S)
    assert len(section.findall(html)) == 1 and section.sub("", html) == html0

    keep = (st & 7 != 7).any(axis=1)
    sto = st[keep]
    genes = [(1, 451), (452, 899)]
    mask = np.zeros(900, dtype=np.uint8)
    for (b, e) in genes:
        mask[b - 1: e - 3: 3] = 1
    _, codon = oracle.pileup(sto, mask)
    keys = sorted({(v.col, v.codon) for v in oracle.call(codon, genes, refseq=t.refseq)})
    haps = rep["haplotypes"]
    assert len(haps) >= 2
    nw = max(1, (len(keys) + 31) // 32)
    pat = np.zeros((len(haps), nw), dtype=np.uint32)
    for k, hp in enumerate(haps):
        assert len(hp["codons"]) == len(keys)
        for v, c in enumerate(hp["codons"]):
            if c:
                pat[k, v >> 5] |= np.uint32(1 << (v & 31))
    want = ha.abundance(sto, keys, pat)
    assert (ab["tolerance"], ab["max_iterations"]) == (1e-10, 10000)
    assert ab["read_categories"] == want["counters"] and ab["reads_used"] == want["reads_used"]
    assert sum(ab["read_categories"].values()) == len(sto)
    assert ab["converged"] == want["converged"] and abs(ab["iterations"] - want["iterations"]) <= 1
    assert abs(ab["log_likelihood"] - want["log_likelihood"]) <= 1e-9 * abs(want["log_likelihood"])
    assert [h["name"] for h in ab["haplotypes"]] == [h["name"] for h in haps]
    for k, h in enumerate(ab["haplotypes"]):
        assert h["reads"] == haps[k]["reads"]
        assert h["unique_reads"] == want["unique_reads"][k] >= h["reads"]
        assert h["compatible_reads"] == want["compatible_reads"][k]
        assert abs(h["em_frequency"] - want["em_frequency"][k]) <= 1e-9
        assert abs(h["em_reads"] - want["em_frequency"][k] * want["reads_used"]) <= 1e-9 * want["reads_used"]
        assert h["em_percentage"] == f"{100 * h['em_frequency']:.1f}"


def test_juliet_cli_abundance_needs_phasing(juliet, tmp_path):
    t = make_tables(SynthConfig(L=900, seed=82))
    bam = str(tmp_path / "in.bam")
    _make_bam(bam, t, synth_states(t, 0, 500))
    res = subprocess.run([juliet, "--haplotype-abundance", bam, str(tmp_path / "o.json")], capture_output=True, text=True)
    assert res.returncode != 0 and "--mode-phasing" in res.stderr
    assert not os.path.exists(tmp_path / "o.json")


def test_juliet_cli_abundance_two_gpus_equal_one(juliet, tmp_path):
    """`--gpus 2`: the ranks' classes are merged inside the library; the report is byte-identical to one GPU's."""
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    t = make_tables(SynthConfig(L=900, seed=83, n_rate=2e-2, trunc=0.05, ins=2e-3))
    st = synth_states(t, 0, 20001)
    bam = str(tmp_path / "in.bam")
    _make_bam(bam, t, st)
    outs = {}
    for n in (1, 2):
        rep, js, html = _run(juliet, ["--mode-phasing", "--haplotype-abundance", "--gpus", str(n), bam], tmp_path, f"g{n}")
        assert rep["haplotype_abundance"]["read_categories"]["ambiguous"] > 0
        outs[n] = (js, html)
    assert outs[1] == outs[2]
