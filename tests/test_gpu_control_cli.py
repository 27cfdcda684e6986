"""`juliet --control`: a systematic 1 % substitution present in sample and control is called by K2 but explained by the
control, a true 1 % minor in the sample only is called by both; the "control" block against control_oracle.py; the report
without the block equal to the run without the option; --drm-only; a control on another reference; --gpus 2."""
import json
import os
import re
import subprocess

import mpmath as mp
import numpy as np
import pytest

import bam_util
import control_oracle as co
import hypergeom_reference as ref
from minorseq_b200 import build as msbuild
from minorseq_b200.synth import SynthConfig, make_tables, synth_states
from test_host_cpp import _gpu_count, _make_bam

pytestmark = pytest.mark.gpu

BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minorseq_b200", "bin")
FIXED = "2026-01-01T00:00:00.000Z"
L, R = 3000, 6000
HOT, MINOR = 300, 1500          # codon starts: the systematic error, the sample's private minor
GENES = [(1, 3001)]


@pytest.fixture(scope="module")
def juliet():
    msbuild.build_library()
    msbuild.build_host()
    return os.path.join(BIN, "juliet")


def _substitute(st, refseq, col, every, phase):
    """1 % of the reads (r % every == phase) that are clean at the codon get base col changed to the next one"""
    base = "ACGT".index(refseq[col])
    for r in range(phase, st.shape[0], every):
        if ((st[r, col - (col % 3): col - (col % 3) + 3] & 7) < 4).all():
            st[r, col] = (st[r, col] & 8) | ((base + 1) & 3)


@pytest.fixture(scope="module")
def pair(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("control")
    t = make_tables(SynthConfig(L=L, seed=9, minor_fracs=()))
    st = synth_states(t, 0, R)
    st0 = synth_states(t, 10 ** 6, R)
    _substitute(st, t.refseq, HOT + 1, 100, 3)
    _substitute(st0, t.refseq, HOT + 1, 100, 5)
    _substitute(st, t.refseq, MINOR + 2, 100, 11)
    bam, cbam = str(tmp / "sample.bam"), str(tmp / "control.bam")
    _make_bam(bam, t, st)
    _make_bam(cbam, t, st0)
    conf = {"genes": [{"name": "geneA", "begin": 1, "end": 3001,
                       "drms": [{"name": "drugX", "positions": [str(MINOR // 3 + 1), str(700)]}]}],
            "referenceName": "synthetic_ref", "referenceSequence": t.refseq, "version": "test"}
    cpath = tmp / "cfg.json"
    cpath.write_text(json.dumps(conf))
    return t, st, st0, bam, cbam, str(cpath)


def _run(juliet, args, tmp_path, tag):
    oj, oh = str(tmp_path / f"{tag}.json"), str(tmp_path / f"{tag}.html")
    env = dict(os.environ, MS_FIXED_TIMESTAMP=FIXED)
    res = subprocess.run([juliet] + args + [oj, oh], capture_output=True, text=True, env=env)
    assert res.returncode == 0, res.stderr
    rep = json.load(open(oj))
    cmd = rep["input"]["command_line"]
    html = open(oh).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X")
    return rep, open(oj).read().replace(cmd, "CMD").replace(f"{tag}.json", "X").replace(f"{tag}.html", "X"), html


def _codon(k):
    return "".join("ACGT"[(k >> s) & 3] for s in (4, 2, 0))


def _called(rep):
    out = set()
    for g in rep["genes"]:
        for vp in g["variant_positions"]:
            for va in vp["variant_amino_acids"]:
                for vc in va["variant_codons"]:
                    out.add((vp["ref_position"], vc["codon"]))
    return out


def test_known_answer(juliet, pair, tmp_path):
    t, _, _, bam, cbam, cpath = pair
    rep, _, html = _run(juliet, ["--config", cpath, "--control", cbam, bam], tmp_path, "ka")
    cb = rep["control"]
    assert cb["input_file"] == cbam and cb["reads"] == R and cb["alpha"] == 0.01 and cb["uncovered_positions"] == 0
    rows = {(r["abs_pos"], r["codon"]): r for r in cb["rows"]}
    hot = [r for r in cb["rows"] if r["abs_pos"] == HOT + 1]
    minor = [r for r in cb["rows"] if r["abs_pos"] == MINOR + 1]
    assert len(hot) == 1 and len(minor) == 1, cb["rows"]
    assert hot[0]["model_call"] and not hot[0]["control_call"] and hot[0]["pValueCorrected"] > 0.01
    assert minor[0]["model_call"] and minor[0]["control_call"] and minor[0]["pValueCorrected"] < 1e-6
    assert minor[0]["known_drm"] == "drugX" and minor[0]["position"] == MINOR // 3 + 1
    assert 50 <= minor[0]["count"] <= 62 and minor[0]["control_count"] == 0
    assert {(hot[0]["position"], hot[0]["codon"]), (minor[0]["position"], minor[0]["codon"])} <= _called(rep)
    assert all(r["model_call"] or r["control_call"] for r in rows.values())
    assert "Control Comparison" in html and minor[0]["label"] in html


def test_block_equals_the_oracle(juliet, pair, oracle, tmp_path):
    t, st, st0, bam, cbam, cpath = pair
    rep, _, _ = _run(juliet, ["--config", cpath, "--control", cbam, bam], tmp_path, "or")
    smp, ctl = co.histogram(st, L, GENES), co.histogram(st0, L, GENES)
    listed = [(v.gene, v.col, v.codon) for v in oracle.call(smp, GENES, refseq=t.refseq)]
    recs, unc = co.control(smp, ctl, L, GENES, refseq=t.refseq, listed=listed)
    drugs = lambda r: ["drugX"] if r["codon_index"] + 1 in (MINOR // 3 + 1, 700) else []
    want = co.report_rows(recs, drugs)
    got = rep["control"]["rows"]
    assert rep["control"]["uncovered_positions"] == unc
    assert [(r["abs_pos"], r["codon"]) for r in got] == [(w["col"] + 1, _codon(w["codon"])) for w in want]
    for g, w in zip(got, want):
        assert g["gene"] == "geneA" and g["position"] == w["codon_index"] + 1 and g["ref_codon"] == _codon(w["ref_codon"])
        for f in ("count", "coverage", "control_count", "control_coverage", "control_call", "model_call", "known_drm"):
            assert g[f] == w[f], (f, g, w)
        assert ref.rel_err(g["pValue"], w["pvalue"]) <= 1e-9 or (w["pvalue"] < mp.mpf("1e-300") and g["pValue"] < 1e-290)
        assert abs(g["pValueCorrected"] - min(1.0, float(w["pvalue"]) * w["ntests"])) <= 1e-9 * max(g["pValueCorrected"], 1e-300)


def _strip_section(html):
    return re.sub(r"<details open><summary>Control Comparison</summary>.*?</details>\n", "", html, flags=re.S)


@pytest.mark.parametrize("extra", [[], ["--mode-phasing", "--linkage"]])
def test_report_without_the_block_is_unchanged(juliet, pair, tmp_path, extra):
    _, _, _, bam, cbam, cpath = pair
    rep, _, html = _run(juliet, ["--config", cpath] + extra + ["--control", cbam, bam], tmp_path, "with")
    rep0, _, html0 = _run(juliet, ["--config", cpath] + extra + [bam], tmp_path, "without")
    assert "control" in rep and "control" not in rep0 and "Control Comparison" not in html0
    rep.pop("control")
    rep["input"]["command_line"] = rep0["input"]["command_line"] = ""
    assert rep == rep0
    assert _strip_section(html).replace("CMD", "") == html0.replace("CMD", "")


def test_drm_only(juliet, pair, tmp_path):
    _, _, _, bam, cbam, cpath = pair
    rep, _, _ = _run(juliet, ["--config", cpath, "--control", cbam, bam], tmp_path, "all")
    rep_d, _, _ = _run(juliet, ["--config", cpath, "--control", cbam, "--drm-only", bam], tmp_path, "drm")
    want = [r for r in rep["control"]["rows"] if r["known_drm"]]
    assert want and rep_d["control"]["rows"] == want


def test_control_on_another_reference_is_refused(juliet, pair, tmp_path):
    t, _, st0, bam, _, cpath = pair
    for name, length in (("other_ref", L), ("synthetic_ref", L + 3)):
        recs = [bam_util.states_to_record(f"c/{r}", st0[r], t.strain_base[0], None, 0, False) for r in range(200)]
        other = str(tmp_path / f"{name}_{length}.bam")
        bam_util.write_bam(other, name, length, [x for x in recs if x is not None])
        oj = tmp_path / f"refused_{length}.json"
        res = subprocess.run([juliet, "--config", cpath, "--control", other, bam, str(oj)], capture_output=True, text=True)
        assert res.returncode == 1 and "--control needs the same reference" in res.stderr, res.stderr
        assert not oj.exists()


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_two_gpus(juliet, pair, tmp_path):
    _, _, _, bam, cbam, cpath = pair
    args = ["--config", cpath, "--mode-phasing", "--control", cbam]
    _, js1, h1 = _run(juliet, args + [bam], tmp_path, "one")
    _, js2, h2 = _run(juliet, args + ["--gpus", "2", bam], tmp_path, "two")
    assert js1.replace(" --gpus 2", "") == js2.replace(" --gpus 2", "") and h1.replace(" --gpus 2", "") == h2.replace(" --gpus 2", "")
    assert np.isfinite(json.loads(js1)["control"]["rows"][0]["pValue"])
