"""Device time of the per-haplotype consensus (restatement choice U15): the counting sort of the read labels, the grouped
pile-up kernel (CUDA events, MS_STAGE_GROUP_PILEUP) and the consensus call, with K1 on the same reads for comparison.
    python tools/haplotype_consensus_timing.py [--reps N] [--out FILE.json]
Shapes: T (1 M reads x 3 kb, 4 strains), C4 (1 M reads x 9719 columns, HIV's 15 genes) and C5 (500 k reads x 6144 columns,
2048 dense sites): each labelled by its own phasing; C5 also with 4096 random labels (~120 reads per group: one flush per
work item, the worst case of the kernel) and T with every read in one group (the same reads without the grouping).
Medians over N repetitions after one warm-up.  Achieved bandwidth = 16 B x blocks per read x labelled reads over the
pile-up kernel's time (the kernel reads every 16-byte block of every labelled read once).  The GPU's name and power limit
are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from minorseq_b200 import Handle, Juliet, _lib, synth_device  # noqa: E402
from minorseq_b200._lib import FuseParams  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

STAGE_GROUP_PILEUP = 10
HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240003), 1_000_000, None),
    "C4": (SynthConfig(L=9719, seed=20240004), 1_000_000, HIV_GENES),
    "C5": (SynthConfig(L=6144, seed=20240005, dense_sites=2048, dense_strains=64, n_rate=2e-5, dele=2e-5, trunc=0.0), 500_000, None),
}


def timed_group_pileup(j, d, lab_ptr, R, ngroups, reps):
    """medians of: the whole ms_group_pileup_dev (sort + pile-up, device events around it) and the pile-up kernel alone"""
    lib, h = j.lib, j.hd.h
    tot, ker = [], []
    for i in range(reps + 1):
        _lib.check(lib.ms_set_groups(h, ngroups), h)
        _lib.check(lib.ms_timer_start(h), h)
        _lib.check(lib.ms_group_pileup_dev(h, C.c_void_p(d.data_ptr()), C.c_void_p(lab_ptr), R), h)
        ms = C.c_double()
        _lib.check(lib.ms_timer_stop(h, C.byref(ms)), h)
        k = C.c_double()
        _lib.check(lib.ms_stage_kernel_ms(h, STAGE_GROUP_PILEUP, C.byref(k)), h)
        if i:
            tot.append(ms.value)
            ker.append(k.value)
    return statistics.median(tot), statistics.median(ker)


def timed_consensus(j, ngroups, reps):
    lib, h = j.lib, j.hd.h
    prm = FuseParams(10, 0.5, 20)
    off = np.zeros(ngroups + 1, dtype=np.int64)
    cap = ngroups * (j.L + 16)
    seq = np.empty(max(1, cap), dtype=np.uint8)
    wall = []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        _lib.check(lib.ms_group_consensus(h, C.byref(prm), None, None, None, None, 0, None, 0, seq.ctypes.data, cap, off.ctypes.data), h)
        if i:
            wall.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(wall)


def row(name, j, d, lab, R, ngroups, reps):
    labelled = int(((lab >= 0) & (lab < ngroups)).sum().item())   # (a synchronising read: the labels are in place)
    tot, ker = timed_group_pileup(j, d, lab.data_ptr(), R, ngroups, reps)
    nblk = (j.L + 31) // 32
    alg = 16 * nblk * labelled
    return dict(case=name, reads=R, L=j.L, groups=ngroups, labelled_reads=labelled, sort_plus_pileup_ms=tot, pileup_kernel_ms=ker,
                sort_ms_by_difference=tot - ker, algorithmic_bytes=alg, pileup_GBps=alg / ker / 1e6,
                consensus_ms_wall=timed_consensus(j, ngroups, reps))


def measure(name, reps):
    cfg, R, genes = SHAPES[name]
    t = make_tables(cfg)
    hd = Handle(0)
    L = cfg.L
    j = Juliet(L, genes or [(1, L + 1)], refseq=None if genes else t.refseq, handle=hd, mode_phasing=True)
    d = synth_device(hd, t, 0, R)
    _lib.check(hd.lib.ms_set_timing(hd.h, 1), hd.h)
    k1 = []
    for i in range(reps + 1):
        j.reset()
        j.pileup_device(d.data_ptr(), R)
        ms, n = C.c_double(), C.c_int64()
        _lib.check(hd.lib.ms_pileup_kernel_ms(hd.h, C.byref(ms), C.byref(n)), hd.h)
        if i:
            k1.append(ms.value)
    if cfg.dense_sites:
        class V:
            def __init__(self, c, k):
                self.col, self.codon = c, k
        variants = [V(c, k) for (c, k) in sorted({(c, k) for (_, c, k) in t.truth})]
    else:
        variants = j.call()
    haps, keys = j.phase_device(variants, d.data_ptr(), R, cap=1 << 16)
    nrep = haps.nreported
    out = dict(shape=name, reads=R, L=L, variants=len(keys), reported_haplotypes=nrep, k1_kernel_ms=statistics.median(k1), rows=[])
    d_hap, Rh = C.c_void_p(), C.c_int64()
    _lib.check(hd.lib.ms_phase_hap_device(hd.h, C.byref(d_hap), C.byref(Rh)), hd.h)
    _lib.check(hd.lib.ms_synchronize(hd.h), hd.h)
    from minorseq_b200.api import _as_tensor
    lab = _as_tensor(d_hap.value, (R,), torch.int32, 0).clone()
    out["rows"].append(row("haplotypes", j, d, lab, R, nrep, reps))
    if name == "T":
        out["rows"].append(row("one group", j, d, torch.zeros(R, dtype=torch.int32, device="cuda:0"), R, 1, reps))
    if name == "C5":
        g = torch.from_numpy(np.random.default_rng(5).integers(0, 4096, size=R).astype(np.int32)).cuda()
        out["rows"].append(row("4096 random groups", j, d, g, R, 4096, reps))
    hd.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("haplotype_consensus_timing.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = dict(gpu=gpu.splitlines(), results=[])
    for name in a.shapes.split(","):
        r = measure(name, a.reps)
        print(json.dumps(r), flush=True)
        report["results"].append(r)
    print(json.dumps(dict(gpu=report["gpu"])), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
