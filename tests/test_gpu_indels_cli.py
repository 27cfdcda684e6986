"""`juliet --indels`: the report's "indels" block against the numpy restatement (indel_oracle.py) on a BAM written with I / D
CIGARs, DRM tokens such as T69ins / D67del in known_drm and the drug summary (a token with another reference amino acid does not
match), the rest of the report unchanged by the option, --drm-only, and --gpus 2 equal to one GPU."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

import indel_oracle as io
from minorseq_b200 import build as msbuild
from minorseq_b200.synth import SynthConfig, make_tables, synth_states
from test_host_cpp import _gpu_count, _make_bam

pytestmark = pytest.mark.gpu

BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minorseq_b200", "bin")
FIXED = "2026-01-01T00:00:00.000Z"
L, R = 900, 6000
DEL_COL, INS_COL = 198, 206          # codon 67 of the gene (columns 198-200); the boundary after codon 69 (204-206)


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
    return rep, open(oj).read(), open(oh).read()


@pytest.fixture(scope="module")
def sample(tmp_path_factory):
    tmp = tmp_path_factory.mktemp("indels")
    t = make_tables(SynthConfig(L=L, seed=97, n_rate=2e-2, trunc=0.05, ins=0.0))
    st = synth_states(t, 0, R)
    ins = {}
    for r in range(0, R, 100):                               # 1 % codon-67 deletion
        if (st[r, DEL_COL: DEL_COL + 3] != 7).all():
            st[r, DEL_COL: DEL_COL + 3] = 4
    for r in range(1, R, 50):                                # 2 % six-base insertion after codon 69
        if st[r, INS_COL] != 7:
            st[r, INS_COL] |= 8
            ins[r] = {INS_COL: "TCTTCT"}
    for r in range(7, R, 500):                               # an out-of-frame insertion: never counted
        if st[r, 300] != 7:
            st[r, 300] |= 8
            ins[r] = {300: "AC"}
    bam = str(tmp / "in.bam")
    _make_bam(bam, t, st, insertions=ins)
    aa = lambda c: io.label(0, 16 * "ACGT".index(t.refseq[c]) + 4 * "ACGT".index(t.refseq[c + 1]) + "ACGT".index(t.refseq[c + 2]), -1, 0)[0]
    other = next(x for x in "ACDEFGHIKLMNPQRSTVWY" if x != aa(204))
    conf = {"genes": [{"name": "RT", "begin": 1, "end": 601,     # the reference amino acids of codons 69 and 67 (and a wrong one)
                       "drms": [{"name": "NRTI", "positions": [f"{aa(204)}69ins", f"{aa(DEL_COL)}67del", "M184V"]},
                                {"name": "wrong_ref", "positions": [f"{other}69ins"]}]},
                      {"name": "other", "begin": 602, "end": 899}],
            "referenceName": "synthetic_ref", "referenceSequence": t.refseq, "version": "test"}
    cpath = tmp / "cfg.json"
    cpath.write_text(json.dumps(conf))
    # the reads as the reader admits them, and their insertion events in its order
    keep = np.nonzero((st & 7 != 7).any(axis=1))[0]
    evs = []
    for k, r in enumerate(keep):
        for c, x in sorted(ins.get(int(r), {}).items()):
            evs.append((k, c, x))
    return t, st[keep], evs, bam, str(cpath), conf


def test_juliet_cli_indels_match_oracle(juliet, sample, tmp_path):
    t, st, evs, bam, cpath, conf = sample
    rep, js, html = _run(juliet, ["--config", cpath, "--indels", bam], tmp_path, "ind")
    rep0, js0, html0 = _run(juliet, ["--config", cpath, bam], tmp_path, "plain")
    block = rep.pop("indels")
    # everything outside the block, the section and the drug summaries is unchanged
    ds, ds0 = rep.pop("drug_summaries"), rep0.pop("drug_summaries")
    rep["input"]["command_line"] = rep0["input"]["command_line"] = ""
    assert rep == rep0
    assert '"indels"' not in js0 and "In-frame Insertions and Deletions" not in html0
    assert len(re.findall(r"<details open><summary>In-frame Insertions and Deletions</summary>", html)) == 1

    genes = [(g["begin"], g["end"]) for g in conf["genes"]]
    pool, off = b"", []
    for _, _, x in evs:
        off.append(len(pool))
        pool += x.encode()
    ev = ([e[0] for e in evs], [e[1] for e in evs], off, [len(e[2]) for e in evs], pool)
    cnt, strings, tally = io.counts(st, ev, io.start_bits(L, genes))
    want = io.call(st, cnt, strings, tally, genes, refseq=t.refseq)
    assert block["deletion_rate"] == 3e-3 and block["insertion_rate"] == 3e-3
    calls = block["calls"]
    assert len(calls) == len(want)
    for c, w in zip(calls, want):
        assert c["gene"] == conf["genes"][w["gene"]]["name"]
        assert c["type"] == ("deletion" if w["kind"] == 0 else "insertion")
        assert c["label"] == io.label(w["kind"], w["ref_codon"], w["next_codon"], w["codon_index"] + 1, w["inserted"])
        assert c["ref_position"] == w["codon_index"] + 1 and c["abs_pos"] == w["col"] + 1 and c["inserted"] == w["inserted"]
        assert (c["count"], c["coverage"], c["expected"]) == (w["count"], w["coverage"], w["expected"])
        assert abs(c["pValue"] - w["pvalue"]) <= 1e-9 * w["pvalue"]
    d67 = [c for c in calls if c["type"] == "deletion" and c["ref_position"] == 67]
    i69 = [c for c in calls if c["type"] == "insertion" and c["ref_position"] == 69 and c["inserted"] == "TCTTCT"]
    assert len(d67) == 1 and len(i69) == 1 and i69[0]["label"].endswith("insSS")
    assert d67[0]["known_drm"] == "NRTI" and i69[0]["known_drm"] == "NRTI"
    nrti = [d for d in ds if d["drug"] == "NRTI"]
    assert nrti and any(v.startswith(i69[0]["label"] + " (RT, ") for v in nrti[0]["variants"])
    assert any(v.startswith(d67[0]["label"] + " (RT, ") for v in nrti[0]["variants"])
    assert i69[0]["label"] in html
    # --drm-only keeps the DRM indels
    rep_d, _, _ = _run(juliet, ["--config", cpath, "--indels", "--drm-only", bam], tmp_path, "drm")
    assert all(c["known_drm"] for c in rep_d["indels"]["calls"]) and len(rep_d["indels"]["calls"]) >= 2


@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_juliet_cli_indels_two_gpus(juliet, sample, tmp_path):
    _, _, _, bam, cpath, _ = sample
    rep1, _, _ = _run(juliet, ["--config", cpath, "--indels", bam], tmp_path, "one")
    rep2, _, _ = _run(juliet, ["--config", cpath, "--indels", "--gpus", "2", bam], tmp_path, "two")
    assert rep1["indels"] == rep2["indels"]
