"""`juliet --rare-linkage`: the report's "rare_linkage" block and HTML section for a 0.25 % strain that K2 does not call, the
report without the option unchanged, and --gpus 2 equal to one GPU."""
import json
import os
import subprocess

import pytest

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


@pytest.fixture(scope="module")
def sample(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("rare")
    t = make_tables(SynthConfig(L=3000, seed=3, minor_fracs=(0.0025,), variants_per_minor=(4, 4)))
    st = synth_states(t, 0, 6000)
    bam = str(tmp / "in.bam")
    _make_bam(bam, t, st)
    conf = {"genes": [{"name": "geneA", "begin": 1, "end": 3001}], "referenceName": "synthetic_ref", "referenceSequence": t.refseq,
            "version": "test"}
    cpath = tmp / "cfg.json"
    cpath.write_text(json.dumps(conf))
    return t, bam, str(cpath)


def _run(juliet, args, tmp_path, tag):
    oj, oh = str(tmp_path / f"{tag}.json"), str(tmp_path / f"{tag}.html")
    env = dict(os.environ, MS_FIXED_TIMESTAMP=FIXED)
    res = subprocess.run([juliet] + args + [oj, oh], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr
    rep = json.load(open(oj))
    cmd = rep["input"]["command_line"]
    return rep, open(oj).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X"), \
        open(oh).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X")


def _codon(k):
    return "".join("ACGT"[(k >> s) & 3] for s in (4, 2, 0))


def test_rare_linkage_reports_the_strain(juliet, sample, tmp_path):
    t, bam, cpath = sample
    rep, _, html = _run(juliet, ["--config", cpath, "--rare-linkage", bam], tmp_path, "rare")
    rl = rep["rare_linkage"]
    assert rl["min_reads"] == 5 and rl["candidate_alpha"] == 0.1 and rl["max_candidates"] == 2048 and rl["dropped_candidates"] == 0
    truth = sorted((c + 1, _codon(k)) for (_, c, k) in t.truth)
    assert len(rl["groups"]) == 1
    g = rl["groups"][0]
    members = sorted((c["abs_pos"], c["codon"]) for c in rl["candidates"] if c["group"] == 0)
    assert members == truth and len(g["members"]) == 4
    assert 0 < g["carriers"] < g["informative"] and abs(g["frequency"] - g["carriers"] / g["informative"]) < 1e-15
    assert rl["tested_pairs"] > 0 and len(rl["pairs"]) >= 3
    assert all(p["pValueCorrected"] < 0.01 for p in rl["pairs"])
    assert "Linked sub-threshold variants" in html
    for c in rl["candidates"]:
        if c["group"] == 0:
            assert c["label"] in html


def test_report_without_the_option_is_unchanged(juliet, sample, tmp_path):
    _, bam, cpath = sample
    rep, _, html = _run(juliet, ["--config", cpath, "--mode-phasing", "--linkage", "--rare-linkage", "--rare-min-reads", "4", bam], tmp_path, "with")
    rep0, _, html0 = _run(juliet, ["--config", cpath, "--mode-phasing", "--linkage", bam], tmp_path, "without")
    rl = rep.pop("rare_linkage")
    assert rl["min_reads"] == 4
    rep["input"]["command_line"] = rep0["input"]["command_line"] = ""
    assert rep == rep0
    assert "Linked sub-threshold variants" not in html0


def test_bad_options(juliet, sample, tmp_path):
    _, bam, cpath = sample
    for args in (["--rare-min-reads", "0"], ["--rare-candidate-alpha", "0"], ["--rare-candidate-alpha", "2"]):
        res = subprocess.run([juliet, "--config", cpath, "--rare-linkage"] + args + [bam, str(tmp_path / "x.json")], capture_output=True,
                             text=True)
        assert res.returncode != 0 and "--rare-" in res.stderr


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_rare_linkage_two_gpus(juliet, sample, tmp_path):
    _, bam, cpath = sample
    args = ["--config", cpath, "--mode-phasing", "--linkage", "--haplotype-abundance", "--rare-linkage"]
    _, js1, h1 = _run(juliet, args + [bam], tmp_path, "one")
    _, js2, h2 = _run(juliet, args + ["--gpus", "2", bam], tmp_path, "two")
    assert js1.replace(" --gpus 2", "") == js2.replace(" --gpus 2", "") and h1.replace(" --gpus 2", "") == h2.replace(" --gpus 2", "")
