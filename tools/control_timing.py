"""Cost of the control comparison (restatement choice U22) on one GPU.

Kernel: CUDA events on the handle's stream (ms_timer_start / ms_timer_stop) around ms_control_call and, on the same counts,
around ms_call (K2) and ms_pileup_dev (K1).  Each call ends in a host synchronise.  Shapes: T (1 M reads x 3 kb, one gene,
the default 10 / 5 / 1 % mixture) and C4 (1 M reads x 9719 columns, HIV's 15 genes).  The control is a clean sample of
the same reference with the generator's error process: other reads of the same seed without the minor strains, so its
histogram holds the error background a real control holds.  The listed codons are K2's calls.  Medians over N repetitions
after one warm-up.

juliet: the binary's stage laps (--timing-json) with and without --control on a 200 k-read sample and a 200 k-read control,
3 kb, written to a temporary directory with packed2bam.  Medians of the laps and of the whole run over N runs after one
warm-up run.

The GPU's name and power limit are read in the same run.
    python tools/control_timing.py [--reps N] [--out FILE.json] [--shapes T,C4] [--cli-reads 200000]"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from minorseq_b200 import Handle, Juliet, _lib, build, synth_device  # noqa: E402
from minorseq_b200._lib import ControlVariant, Gene, Variant  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables, pack_states, synth_states  # noqa: E402

HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240003), 1_000_000, None),
    "C4": (SynthConfig(L=9719, seed=20240004), 1_000_000, HIV_GENES),
}
CONTROL_READ0 = 10 ** 8      # the control's reads: other reads of the same generator, no overlap with the sample's


def control_config(cfg):
    return SynthConfig(**dict(cfg.__dict__, minor_fracs=()))


def measure(name, reps):
    cfg, R, genes = SHAPES[name]
    genes = genes or [(1, cfg.L + 1)]
    hd = Handle(0)
    lib = hd.lib
    j = Juliet(cfg.L, genes, handle=hd)
    dc = synth_device(hd, make_tables(control_config(cfg)), CONTROL_READ0, R)
    j.pileup_device(dc.data_ptr(), R)
    j.capture_control()
    del dc
    d = synth_device(hd, make_tables(cfg), 0, R)
    g = (Gene * len(genes))(*[Gene(b, e) for (b, e) in genes])
    calls = (Variant * 65536)()
    out = (ControlVariant * 65536)()
    n, unc = C.c_int64(), C.c_int64()

    def timed(fn):
        _lib.check(lib.ms_timer_start(hd.h), hd.h)
        fn()
        ms = C.c_double()
        _lib.check(lib.ms_timer_stop(hd.h, C.byref(ms)), hd.h)
        return ms.value

    def pileup():
        j.reset()
        j.pileup_device(d.data_ptr(), R)
        _lib.check(lib.ms_synchronize(hd.h), hd.h)

    stages = {k: [] for k in ("pileup", "k2_call", "control_call")}
    info = {}
    for i in range(reps + 1):
        st = dict(pileup=timed(pileup))
        st["k2_call"] = timed(lambda: _lib.check(lib.ms_call(hd.h, g, len(genes), None, C.byref(j.params), calls, 65536, C.byref(n)), hd.h))
        nl = min(int(n.value), 65536)
        st["control_call"] = timed(lambda: _lib.check(lib.ms_control_call(hd.h, g, len(genes), None, C.byref(j.params), calls, nl, out, 65536,
                                                                          C.byref(n), C.byref(unc)), hd.h))
        rows = [out[k] for k in range(min(int(n.value), 65536))]
        info = dict(k2_calls=nl, control_rows=int(n.value), control_calls=sum(r.called for r in rows),
                    k2_calls_explained_by_control=sum(1 for r in rows if r.listed and not r.called), uncovered_positions=int(unc.value))
        if i:
            for k, v in st.items():
                stages[k].append(v)
    res = dict(shape=name, reads=R, control_reads=R, L=cfg.L, genes=len(genes), **info)
    for k, v in stages.items():
        res[f"{k}_ms"] = statistics.median(v)
    hd.close()
    return res


def write_bam(d, tag, t, read0, R):
    parts = []
    for r0 in range(0, R, 20_000):
        parts.append(pack_states(synth_states(t, read0 + r0, min(20_000, R - r0))))
    p = os.path.join(d, f"{tag}.bin")
    np.concatenate(parts).tofile(p)
    bam = os.path.join(d, f"{tag}.bam")
    subprocess.check_call([os.path.join(build.BIN, "packed2bam"), p, str(t.cfg.L), str(R), os.path.join(d, "ref.txt"), bam])
    os.remove(p)
    return bam


def juliet_laps(R, reps):
    build.build_library()
    build.build_host()
    cfg = SynthConfig(L=3000, seed=20240003)
    t = make_tables(cfg)
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "ref.txt"), "w").write(t.refseq + "\n")
        bam = write_bam(d, "sample", t, 0, R)
        cbam = write_bam(d, "control", make_tables(control_config(cfg)), CONTROL_READ0, R)
        conf = os.path.join(d, "cfg.json")
        json.dump({"genes": [{"name": "pol", "begin": 1, "end": 3001}], "referenceName": "synthetic_ref", "referenceSequence": t.refseq},
                  open(conf, "w"))
        res = {}
        for tag, extra in (("without_control", []), ("with_control", ["--control", cbam])):
            laps, totals = {}, []
            for i in range(reps + 1):
                tj = os.path.join(d, "t.json")
                subprocess.check_call([os.path.join(build.BIN, "juliet"), "-c", conf] + extra + ["--timing-json", tj, bam, os.path.join(d, "o.json")])
                tim = json.load(open(tj))
                if i:
                    totals.append(tim["total_ms"])
                    for s in tim["stages"]:
                        laps.setdefault(s["stage"], []).append(s["ms"])
            res[tag] = dict(total_ms=statistics.median(totals), stages={k: statistics.median(v) for k, v in laps.items()})
        return dict(reads=R, control_reads=R, L=3000, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--cli-reps", type=int, default=3)
    ap.add_argument("--cli-reads", type=int, default=200_000)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default="T,C4")
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res = dict(gpu=gpu, kernel=[measure(s, a.reps) for s in a.shapes.split(",") if s])
    if a.cli_reads > 0:
        res["juliet"] = juliet_laps(a.cli_reads, a.cli_reps)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
