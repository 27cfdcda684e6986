"""`align reads.bam reference.fasta out.bam`: record handling, and juliet / fuse from its output against the generator's own
alignment on a mixture where the overlap alignment's answer is known exactly."""
import json
import os
import subprocess

import numpy as np
import pytest

import bam_util
from align_oracle import revcomp
from minorseq_b200 import build as msbuild
from minorseq_b200.synth import SynthConfig, make_tables, synth_states

pytestmark = pytest.mark.gpu

BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minorseq_b200", "bin")
FIXED = "2026-01-01T00:00:00.000Z"


@pytest.fixture(scope="module")
def binaries():
    msbuild.build_library()
    msbuild.build_host()
    return BIN


def run(binaries, prog, *args):
    res = subprocess.run([os.path.join(binaries, prog)] + [str(a) for a in args], capture_output=True, text=True,
                         env=dict(os.environ, MS_FIXED_TIMESTAMP=FIXED))
    assert res.returncode == 0, res.stderr
    return res


def write_fasta(path, name, seq):
    with open(path, "w") as f:
        f.write(f">{name} a description\n")
        for i in range(0, len(seq), 60):
            f.write(seq[i:i + 60] + "\n")


def write_generator_bam(path, t, st):
    """The generator's own alignment of the reads (every fifth one stored reverse), as the other CLI tests build it."""
    recs = []
    for r in range(st.shape[0]):
        rec = bam_util.states_to_record(f"m/{r}/ccs", st[r], t.strain_base[0], None, 0x10 if r % 5 == 0 else 0)
        if rec is not None:
            recs.append(rec)
    bam_util.write_bam(path, "synthetic_ref", t.cfg.L, recs)
    return bam_util.read_bam(path)[2]


def unaligned(recs):
    """The generator's records as an unaligned ccs.bam holds them: native SEQ, flag 0x4, no position or CIGAR."""
    out = []
    for r in recs:
        seq = revcomp(r["seq"]) if r["flag"] & 0x10 else r["seq"]
        out.append(bam_util.record(r["name"], 0x4, -1, [], seq, r["aux"], ref_id=-1, mapq=0))
    return out


@pytest.fixture(scope="module")
def exact(tmp_path_factory, binaries):
    """No insertions, deletions or truncation; the first and last 8 columns of every read are the reference's base (an
    overlap alignment soft-clips a mismatch at the reference's ends by design)."""
    d = tmp_path_factory.mktemp("align_exact")
    t = make_tables(SynthConfig(L=900, seed=31, dele=0.0, ins=0.0, trunc=0.0, n_rate=2e-3))
    st = synth_states(t, 0, 6000)
    ref = t.strain_base[0]
    for cols in (slice(0, 8), slice(892, 900)):
        st[:, cols] = ref[cols]
    gen = str(d / "gen.bam")
    keep = write_generator_bam(gen, t, st)
    ccs = str(d / "sample.ccs.bam")
    bam_util.write_bam(ccs, "none", 1, unaligned(keep))
    fa = str(d / "ref.fasta")
    write_fasta(fa, "synthetic_ref", t.refseq)
    out = str(d / "aligned.bam")
    res = run(binaries, "align", ccs, fa, out)
    return t, d, gen, out, keep, res


def test_align_records(exact):
    t, d, gen, out, keep, res = exact
    text, refs, recs = bam_util.read_bam(out)
    assert refs == [("synthetic_ref", 900)]
    assert "@PG\tID:align" in text and "SO:unknown" in text and "SN:synthetic_ref\tLN:900" in text
    assert [r["name"] for r in recs] == [r["name"] for r in keep]
    for a, g in zip(recs, keep):
        assert a["seq"] == g["seq"] and a["flag"] & 0x10 == g["flag"] & 0x10 and a["pos"] == g["pos"] == 0
        assert all(op in "=X" for _, op in a["cigar"]), a["cigar"]
        assert a["cigar"] == g["cigar"] and a["mapq"] == 60 and b"ASi" in a["aux"]
    assert "0 unmapped" in res.stderr


def test_juliet_and_fuse_equal_from_align_output(exact, binaries):
    t, d, gen, out, keep, _ = exact
    conf = {"genes": [{"name": "geneA", "begin": 1, "end": 451}, {"name": "geneB", "begin": 452, "end": 898}],
            "referenceName": "synthetic_ref", "referenceSequence": t.refseq, "version": "test"}
    cpath = d / "cfg.json"
    cpath.write_text(json.dumps(conf))
    for name, bam in (("gen", gen), ("aln", out)):
        run(binaries, "juliet", "--mode-phasing", "-c", cpath, bam, d / f"{name}.json")
        run(binaries, "juliet", "--mode-phasing", "-c", cpath, bam, d / f"{name}.html")
        run(binaries, "fuse", bam, d / f"{name}.fasta")

    def strip(p):
        j = json.loads(open(p).read())
        j.pop("input")           # the input file and the command line
        return j
    a, g = strip(d / "aln.json"), strip(d / "gen.json")
    assert a == g
    assert a.get("haplotypes") or a.get("genes")
    html = [open(d / f"{n}.html").read().replace(str(d / f"{n}.html"), "Y").replace(str(gen), "X").replace(str(out), "X")
            for n in ("gen", "aln")]
    assert html[0] == html[1]
    fasta = [open(d / f"{n}.fasta").read().split("\n", 1) for n in ("gen", "aln")]
    assert fasta[0][0] == ">gen.bam|fuse|synthetic_ref" and fasta[1][0] == ">aligned.bam|fuse|synthetic_ref"   # the input's name
    assert fasta[0][1] == fasta[1][1]


def juliet_reports(binaries, d, conf, bams, phasing=True):
    cpath = d / "cfg.json"
    cpath.write_text(json.dumps(conf))
    out = {}
    for name, bam in bams.items():
        run(binaries, "juliet", *(["--mode-phasing"] if phasing else []), "-c", cpath, bam, d / f"{name}.json", d / f"{name}.html")
        run(binaries, "fuse", bam, d / f"{name}.fasta")
        out[name] = (json.loads(open(d / f"{name}.json").read()), open(d / f"{name}.fasta").read().split("\n", 1)[1])
    return out


def called(report):
    return [(g["name"], vp["ref_position"], vc["codon"]) for g in report["genes"] for vp in g["variant_positions"]
            for va in vp["variant_amino_acids"] for vc in va["variant_codons"]]


def test_indel_mixture_gives_the_same_calls(binaries, tmp_path):
    """bench.py's C3 mixture (deletions, homopolymer deletions, insertions, truncation, N): fuse's consensus is identical and
    every variant juliet calls from the generator's alignment is called from align's.  align's output is not the generator's
    alignment (a deletion inside a homopolymer is placed leftmost, an adjacent insertion and deletion become a mismatch,
    indels next to a read's end are scored, not known), so codon counts move slightly; the extra calls, the haplotype
    patterns and their read counts of both runs are printed (DESIGN.md "K6 read alignment" records one run)."""
    t = make_tables(SynthConfig(L=3000, seed=20240003))
    st = synth_states(t, 0, 20000)
    gen = str(tmp_path / "gen.bam")
    recs = write_generator_bam(gen, t, st)
    ccs = str(tmp_path / "c3.ccs.bam")
    bam_util.write_bam(ccs, "none", 1, unaligned(recs))
    fa = tmp_path / "ref.fasta"
    write_fasta(fa, "synthetic_ref", t.refseq)
    aln = str(tmp_path / "aln.bam")
    res = run(binaries, "align", ccs, fa, aln)
    print(res.stderr.strip())
    conf = {"genes": [{"name": "pol", "begin": 1, "end": 3001}], "referenceName": "synthetic_ref", "referenceSequence": t.refseq,
            "version": "test"}
    rep = juliet_reports(binaries, tmp_path, conf, {"gen": gen, "aln": aln})
    (jg, fg), (ja, fa_) = rep["gen"], rep["aln"]
    assert fa_ == fg
    cg, ca = called(jg), called(ja)
    assert cg and set(cg) <= set(ca)
    planted = {(c // 3 + 1, "".join("ACGT"[(codon >> s) & 3] for s in (4, 2, 0))) for _, c, codon in t.truth}
    assert planted <= {(p, c) for _, p, c in ca}
    freq = {(g["name"], vp["ref_position"], vc["codon"]): (vc["count"], vp["coverage"]) for g in ja["genes"] for vp in g["variant_positions"]
            for va in vp["variant_amino_acids"] for vc in va["variant_codons"]}
    print("calls only from align (count, coverage):", [(k, freq[k]) for k in ca if k not in set(cg)])
    print("haplotypes, generator:", [(h["name"], h["reads"], "".join(h["codons"])) for h in jg["haplotypes"]])
    print("haplotypes, align:", [(h["name"], h["reads"], "".join(h["codons"])) for h in ja["haplotypes"]])
    print("read categories (generator, align):", jg["haplotype_read_categories"], ja["haplotype_read_categories"])


def test_records_kept_and_dropped(binaries, tmp_path):
    rng = np.random.default_rng(3)
    ref = "".join("ACGT"[x] for x in rng.integers(0, 4, 1500))
    fa = tmp_path / "r.fasta"
    write_fasta(fa, "amp", ref)
    qv = "".join(chr(33 + (i % 40)) for i in range(600))
    recs = [
        bam_util.record("fwd", 0x4, -1, [], ref[100:700], bam_util.aux_z("dq", qv) + b"NMi\x05\x00\x00\x00", ref_id=-1, mapq=0),
        bam_util.record("rev", 0x4, -1, [], revcomp(ref[300:900]), bam_util.aux_z("dq", qv), ref_id=-1, mapq=0),
        bam_util.record("sec", 0x104, -1, [], ref[:300], ref_id=-1, mapq=0),
        bam_util.record("sup", 0x804, -1, [], ref[:300], ref_id=-1, mapq=0),
        bam_util.record("junk", 0x4, -1, [], "ACGT" * 100, ref_id=-1, mapq=0),
        bam_util.record("rev-stored", 0x10, 5, [(600, "=")], ref[200:800], ref_id=0),
    ]
    inp = tmp_path / "in.bam"
    bam_util.write_bam(str(inp), "old", 5000, recs)
    out = tmp_path / "out.bam"
    res = run(binaries, "align", inp, fa, out)
    assert "2 secondary/supplementary dropped" in res.stderr and "1 unmapped" in res.stderr
    _, refs, got = bam_util.read_bam(str(out))
    assert refs == [("amp", 1500)]
    assert [r["name"] for r in got] == ["fwd", "rev", "junk", "rev-stored"]
    f, r, j, s = got
    assert (f["flag"], f["pos"], f["cigar"], f["seq"]) == (0, 100, [(600, "=")], ref[100:700])
    assert (r["flag"], r["pos"], r["cigar"], r["seq"]) == (0x10, 300, [(600, "=")], ref[300:900])
    assert (j["flag"], j["pos"], j["ref_id"], j["cigar"], j["seq"]) == (0x4, -1, -1, [], "ACGT" * 100)
    assert (s["flag"], s["pos"], s["cigar"], s["seq"]) == (0x10, 200, [(600, "=")], ref[200:800])
    assert b"NMi" not in f["aux"] and b"ASi" + (1200).to_bytes(4, "little") in f["aux"]
    assert bam_util.aux_z("dq", qv) in f["aux"] and bam_util.aux_z("dq", qv) in r["aux"]    # per-base tracks stay native


def test_pg_id_stays_unique(binaries, tmp_path):
    rng = np.random.default_rng(4)
    ref = "".join("ACGT"[x] for x in rng.integers(0, 4, 800))
    fa = tmp_path / "r.fasta"
    write_fasta(fa, "amp", ref)
    bam_util.write_bam(str(tmp_path / "a.bam"), "old", 5000, [bam_util.record("r", 0x4, -1, [], ref[100:600], ref_id=-1, mapq=0)])
    run(binaries, "align", tmp_path / "a.bam", fa, tmp_path / "b.bam")
    run(binaries, "align", tmp_path / "b.bam", fa, tmp_path / "c.bam")
    text = bam_util.read_bam(str(tmp_path / "c.bam"))[0]
    assert "@PG\tID:align\t" in text and "@PG\tID:align.1\tPN:align\tVN:minorseq_b200-0.1.0\tPP:align\n" in text


def test_missing_input_fails(binaries, tmp_path):
    fa = tmp_path / "r.fasta"
    write_fasta(fa, "amp", "ACGT" * 100)
    res = subprocess.run([os.path.join(binaries, "align"), str(tmp_path / "nope.bam"), str(fa), str(tmp_path / "o.bam")],
                         capture_output=True, text=True)
    assert res.returncode != 0 and not os.path.exists(tmp_path / "o.bam")


def diverged_reference(t, rng):
    """The major strain with 2 % substitutions and two in-frame 3-base indels, none of them near a planted variant.  Returns
    the sequence and the map from a major-strain column to its column in it."""
    major = list(t.refseq)
    L = len(major)
    planted = {c for _, col, _ in t.truth for c in range(col - 6, col + 9)}
    free = [j for j in range(L) if j not in planted]
    for j in rng.choice(free, size=int(0.02 * L), replace=False):
        major[j] = "ACGT"[("ACGT".index(major[j]) + int(rng.integers(1, 4))) % 4]
    cut = next(c for c in range(900, L, 3) if all(x not in planted for x in range(c, c + 3)))
    put = next(c for c in range(2100, L, 3) if c not in planted and c - 1 not in planted)
    seq = major[:cut] + major[cut + 3:put] + list("GCA") + major[put:]
    # a major column c maps to c (before the deletion), c - 3 (between), c (after the insertion)
    col = {c: c if c < cut else c - 3 if c < put else c for c in range(L) if not cut <= c < cut + 3}
    return "".join(seq), col


@pytest.fixture(scope="module")
def flow(tmp_path_factory, binaries):
    """Reads of bench.py's C3 mixture as an unaligned ccs.bam, a diverged reference, and a config over its whole length."""
    d = tmp_path_factory.mktemp("julietflow")
    t = make_tables(SynthConfig(L=3000, seed=20240003))
    st = synth_states(t, 0, 20000)
    recs = write_generator_bam(str(d / "gen.bam"), t, st)
    bam_util.write_bam(str(d / "m64001_sample.ccs.bam"), "none", 1, unaligned(recs))
    ref, col = diverged_reference(t, np.random.default_rng(8))
    write_fasta(d / "ref.fasta", "diverged_ref", ref)
    conf = {"genes": [{"name": "pol", "begin": 1, "end": len(ref) + 1}], "referenceName": "diverged_ref", "referenceSequence": ref,
            "version": "test"}
    (d / "cfg.json").write_text(json.dumps(conf))
    return t, d, ref, col


def _in(d, *cmd):
    res = subprocess.run([str(c) for c in cmd], cwd=d, capture_output=True, text=True, env=dict(os.environ, MS_FIXED_TIMESTAMP=FIXED))
    assert res.returncode == 0, res.stderr
    return res


def _without_command_line(html):
    import re
    return re.sub(r"Command Line Call:</td><td style=\"text-align:left\"><tt>[^<]*</tt>", "", html)


def test_julietflow_equals_the_steps_by_hand(flow, binaries):
    t, d, ref, col = flow
    a, b = d / "flow", d / "hand"
    a.mkdir()
    b.mkdir()
    for x in (a, b):
        for f in ("m64001_sample.ccs.bam", "ref.fasta", "cfg.json"):
            os.symlink(d / f, x / f)
    _in(a, os.path.join(binaries, "julietflow"), "-i", "m64001_sample.ccs.bam", "-r", "ref.fasta", "-c", "cfg.json", "-k")
    stem = "tmp/m64001_sample/m64001_sample"
    (b / "tmp" / "m64001_sample").mkdir(parents=True)
    bn = lambda p: os.path.join(binaries, p)   # noqa: E731
    _in(b, bn("align"), "m64001_sample.ccs.bam", "ref.fasta", f"{stem}.ref.bam")
    _in(b, bn("fuse"), f"{stem}.ref.bam", f"{stem}.consensus.fasta")
    _in(b, bn("align"), "m64001_sample.ccs.bam", f"{stem}.consensus.fasta", f"{stem}.consensus.bam")
    _in(b, bn("cleric"), f"{stem}.consensus.bam", f"{stem}.consensus.fasta", "ref.fasta", f"{stem}.cleric.bam")
    _in(b, bn("juliet"), "-c", "cfg.json", f"{stem}.cleric.bam", "m64001_sample.json", "m64001_sample.html")
    ja, jb = (json.loads(open(x / "m64001_sample.json").read()) for x in (a, b))
    assert ja["input"].pop("command_line") != jb["input"].pop("command_line")
    assert ja == jb
    assert _without_command_line(open(a / "m64001_sample.html").read()) == _without_command_line(open(b / "m64001_sample.html").read())
    for f in ("ref.bam", "consensus.fasta", "consensus.bam", "cleric.bam"):      # -k keeps the intermediates
        assert open(a / f"{stem}.{f}", "rb").read() == open(b / f"{stem}.{f}", "rb").read()
    # every planted minor codon is called, at its column in the diverged reference
    calls = {(vp["ref_position"], vc["codon"]) for g in ja["genes"] for vp in g["variant_positions"]
             for va in vp["variant_amino_acids"] for vc in va["variant_codons"]}
    planted = {(col[c] // 3 + 1, "".join("ACGT"[(codon >> s) & 3] for s in (4, 2, 0))) for _, c, codon in t.truth}
    assert planted and planted <= calls, sorted(planted - calls)


def test_julietflow_removes_intermediates_and_fails_loudly(flow, binaries):
    t, d, ref, col = flow
    x = d / "plain"
    x.mkdir()
    for f in ("m64001_sample.ccs.bam", "ref.fasta", "cfg.json"):
        os.symlink(d / f, x / f)
    _in(x, os.path.join(binaries, "julietflow"), "-i", "m64001_sample.ccs.bam", "-r", "ref.fasta", "-c", "cfg.json")
    assert sorted(os.listdir(x)) == ["cfg.json", "m64001_sample.ccs.bam", "m64001_sample.html", "m64001_sample.json", "ref.fasta"]
    res = subprocess.run([os.path.join(binaries, "julietflow"), "-i", "missing.ccs.bam", "-r", "ref.fasta"], cwd=x,
                         capture_output=True, text=True)
    assert res.returncode != 0 and "missing.ccs.bam" in res.stderr
    bad = x / "bad.fasta"
    bad.write_text(">a\nACGT\n>b\nACGT\n")                 # align refuses a reference with two records: the flow stops there
    res = subprocess.run([os.path.join(binaries, "julietflow"), "-i", "m64001_sample.ccs.bam", "-r", str(bad)], cwd=x,
                         capture_output=True, text=True)
    assert res.returncode != 0 and "step 1/5 (align) failed" in res.stderr and "exactly one sequence" in res.stderr
    assert not os.path.exists(x / "bad.json")
