"""`juliet --mode-phasing in.bam out.json out.fasta`: every FASTA record against the test-side U15 oracle on the reads the
report lists for that haplotype, the JSON and HTML unchanged by the FASTA, the option checks, and --gpus 2 equal to one GPU."""
import json
import os
import subprocess

import numpy as np
import pytest

import haplotype_consensus_oracle as hco
from minorseq_b200 import build as msbuild
from minorseq_b200.synth import SynthConfig, make_tables, read_strains, synth_states
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
    """a mixture whose strain-1 reads carry an in-frame insertion after column 450; other insertion flags insert one base"""
    t = make_tables(SynthConfig(L=900, seed=81, n_rate=2e-3, trunc=0.05, ins=1e-3))
    R = 20001
    st = synth_states(t, 0, R)
    strains, _, _ = read_strains(t, 0, R)
    ins = {}
    for r in np.nonzero(strains == 1)[0]:
        if st[r, 450] & 7 != 7:
            st[r, 450] |= 8
            ins[int(r)] = {450: "GGC"}
    bam = str(tmp_path_factory.mktemp("hapcons") / "in.bam")
    _make_bam(bam, t, st, insertions=ins)
    return t, st, ins, bam


def _run(juliet, args, outs, env_extra=None):
    env = dict(os.environ, MS_FIXED_TIMESTAMP=FIXED, **(env_extra or {}))
    return subprocess.run([juliet] + args + outs, capture_output=True, text=True, env=env)


def _fasta(path):
    recs, name = [], None
    for line in open(path).read().splitlines():
        if line.startswith(">"):
            recs.append([line[1:], ""])
        else:
            assert len(line) <= 70
            recs[-1][1] += line
    return recs


def test_fasta_records_equal_oracle_on_listed_reads(juliet, sample, tmp_path):
    t, st, ins, bam = sample
    oj, oh, of = (str(tmp_path / f"o.{x}") for x in ("json", "html", "fasta"))
    res = _run(juliet, ["--mode-phasing", "--hap-min-coverage", "12", bam], [oj, oh, of])
    assert res.returncode == 0, res.stderr
    rep = json.load(open(oj))
    haps = rep["haplotypes"]
    recs = _fasta(of)
    assert len(haps) >= 2 and len(recs) == len(haps)
    labels = np.full(st.shape[0], -1, dtype=np.int64)
    for k, h in enumerate(haps):
        for n in h["read_names"]:
            labels[int(n.split("/")[1])] = k
    read, col, off, ln, pool = [], [], [], [], bytearray()
    for r, c in zip(*np.nonzero(st & 8)):
        s = ins.get(int(r), {}).get(int(c), "A").encode()
        read.append(r); col.append(c); off.append(len(pool)); ln.append(len(s))
        pool += s
    want = hco.haplotype_consensus(st, labels, len(haps), (read, col, off, ln, bytes(pool)), min_coverage=12)
    for k, ((head, seq), h) in enumerate(zip(recs, haps)):
        assert head == f"in.bam|haplotype_{h['name']}|synthetic_ref reads={h['reads']}"
        assert seq == want[k], k
    assert sum("GGC" in s for s in want) >= 1


def test_json_and_html_unchanged_by_fasta(juliet, sample, tmp_path):
    _, _, _, bam = sample
    texts = []
    for tag, extra in (("a", [str(tmp_path / "a.fasta")]), ("b", [])):
        oj, oh = str(tmp_path / f"{tag}.json"), str(tmp_path / f"{tag}.html")
        res = _run(juliet, ["--mode-phasing", bam], [oj, oh] + extra)
        assert res.returncode == 0, res.stderr
        cmd = json.load(open(oj))["input"]["command_line"]      # the call itself is recorded: it names the outputs
        texts.append(tuple(open(p).read().replace(cmd, "CMD") for p in (oj, oh)))
    assert texts[0] == texts[1]


def test_fasta_needs_mode_phasing(juliet, sample, tmp_path):
    _, _, _, bam = sample
    res = _run(juliet, [bam], [str(tmp_path / "o.json"), str(tmp_path / "o.fasta")])
    assert res.returncode != 0 and "--mode-phasing" in res.stderr
    assert not os.path.exists(tmp_path / "o.json")


def test_fasta_two_gpus_equal_one(juliet, sample, tmp_path):
    if _gpu_count() < 2:
        pytest.skip("needs two GPUs")
    _, _, _, bam = sample
    out = []
    for n in (1, 2):
        of = str(tmp_path / f"g{n}.fasta")
        res = _run(juliet, ["--mode-phasing", "--gpus", str(n), bam], [of])
        assert res.returncode == 0, res.stderr
        out.append(open(of).read())
    assert out[0] == out[1] and out[0].count(">") >= 2
