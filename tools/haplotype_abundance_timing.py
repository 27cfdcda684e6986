"""Device time of haplotype abundance's stages (restatement choice U18), CUDA events on the handle's stream
(ms_set_timing / ms_stage_kernel_ms): abundance_compat_kernel, the EM (all iterations with the host's checks between batches),
and the whole ms_haplotype_abundance call on a host clock; class grouping and ordering is the rest of the call.  Also the EM's
iteration count and time per iteration, and the reads the EM uses against the reads phasing reports.
    python tools/haplotype_abundance_timing.py [--reps N] [--out FILE.json]
Shapes: T (1 M reads x 3 kb, 4 strains), C4 (1 M reads x 9719 columns, HIV's 15 genes, the variants K2 calls) and C5
(500 k reads x 6144 columns, 2048 dense sites as the keys); the patterns are the reported haplotypes.  Medians over N
repetitions after one warm-up; one GPU, so the class all-gather is not measured.  The GPU's name and power limit are read
in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from minorseq_b200 import Handle, Juliet, _lib, synth_device  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

STAGE_COMPAT, STAGE_EM = 13, 14
HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240003), 1_000_000, None),
    "C4": (SynthConfig(L=9719, seed=20240004), 1_000_000, HIV_GENES),
    "C5": (SynthConfig(L=6144, seed=20240005, dense_sites=2048, dense_strains=64, n_rate=2e-5, dele=2e-5, trunc=0.0), 500_000, None),
}


class _V:
    def __init__(self, col, codon):
        self.col, self.codon = col, codon


def stage(hd, s):
    ms = C.c_double()
    _lib.check(hd.lib.ms_stage_kernel_ms(hd.h, s, C.byref(ms)), hd.h)
    return ms.value


def measure(name, reps):
    cfg, R, genes = SHAPES[name]
    t = make_tables(cfg)
    hd = Handle(0)
    j = Juliet(cfg.L, genes or [(1, cfg.L + 1)], handle=hd, refseq=None if genes else t.refseq)
    d = synth_device(hd, t, 0, R)
    if cfg.dense_sites:
        variants = [_V(c, k) for c, k in sorted({(c, k) for (_, c, k) in t.truth})]
    else:
        j.pileup_device(d.data_ptr(), R)
        variants = j.call(cap=8192)
    hap, keys = j.phase_device(variants, d.data_ptr(), R, want_hap_id=False, abundance=True)
    _lib.check(hd.lib.ms_set_timing(hd.h, 1), hd.h)
    compat, em, total = [], [], []
    ab = None
    for i in range(reps + 1):
        _lib.check(hd.lib.ms_synchronize(hd.h), hd.h)
        t0 = time.perf_counter()
        ab = j.haplotype_abundance()
        t1 = time.perf_counter()
        if i:
            total.append(1e3 * (t1 - t0))
            compat.append(stage(hd, STAGE_COMPAT))
            em.append(stage(hd, STAGE_EM))
    H, V = hap.nreported, len(keys)
    vwords, hw = max(1, (V + 31) // 32), max(1, (H + 31) // 32)
    c_ms, e_ms, t_ms = statistics.median(compat), statistics.median(em), statistics.median(total)
    nbytes = R * (2 * vwords + hw) * 4           # B and M rows read, one mask row written
    out = dict(shape=name, reads=R, L=cfg.L, keys=V, haplotypes=H, compat_ms=c_ms, compat_gb_per_s=nbytes / c_ms / 1e6,
               em_ms=e_ms, iterations=ab.iterations, converged=ab.converged,
               em_ms_per_iteration=e_ms / ab.iterations if ab.iterations else None,
               grouping_and_order_ms=t_ms - c_ms - e_ms, call_ms=t_ms, reads_used=ab.reads_used, reported_reads=int(hap.counters["reported"]),
               counters=ab.counters)
    hd.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default="T,C4,C5")
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res = dict(gpu=gpu, shapes=[measure(s, a.reps) for s in a.shapes.split(",")])
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
