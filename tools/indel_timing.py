"""Device time of the in-frame indel pass (restatement choice U19): indel_count_kernel from CUDA events on the handle's stream
(ms_set_timing / ms_stage_kernel_ms, MS_STAGE_INDELS), and the whole Juliet.indels call (counts, event tally, all-reduce,
test, download) on a host clock.  The kernel's algorithmic bytes are one more read of the tiles, R * ceil(L/32) * 16 bytes
(about R * L / 2); the rate printed is those bytes over the kernel time.
    python tools/indel_timing.py [--reps N] [--out FILE.json]
Shapes: T (1 M reads x 3 kb, one gene) and C4 (1 M reads x 9719 columns, HIV's 15 genes); 0.5 % of the reads carry a
six-base insertion event at one boundary (the event tally is timed with the call).  The working set (1.5 GB and 4.9 GB
of tiles) is far larger than L2.  Medians over N repetitions after one warm-up; one GPU.  The GPU's name and power limit
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

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from minorseq_b200 import Handle, Juliet, _lib, synth_device  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

STAGE_INDELS = 15
HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240003), 1_000_000, None, 302),
    "C4": (SynthConfig(L=9719, seed=20240004), 1_000_000, HIV_GENES, 2755),
}


def measure(name, reps):
    cfg, R, genes, ins_col = SHAPES[name]
    t = make_tables(cfg)
    hd = Handle(0)
    j = Juliet(cfg.L, genes or [(1, cfg.L + 1)], handle=hd, refseq=None if genes else t.refseq)
    d = synth_device(hd, t, 0, R)
    j.pileup_device(d.data_ptr(), R)
    reads = np.arange(0, R, 200, dtype=np.int64)
    ev = (reads, np.full(len(reads), ins_col, dtype=np.int32), np.zeros(len(reads), dtype=np.int64), np.full(len(reads), 6, dtype=np.int32),
          b"TCTTCT")
    _lib.check(hd.lib.ms_set_timing(hd.h, 1), hd.h)
    kern, total = [], []
    res = None
    for i in range(reps + 1):
        _lib.check(hd.lib.ms_synchronize(hd.h), hd.h)
        t0 = time.perf_counter()
        res = j.indels(d.data_ptr(), R, insertions=ev)
        t1 = time.perf_counter()
        if i:
            ms = C.c_double()
            _lib.check(hd.lib.ms_stage_kernel_ms(hd.h, STAGE_INDELS, C.byref(ms)), hd.h)
            kern.append(ms.value)
            total.append(1e3 * (t1 - t0))
    k_ms, t_ms = statistics.median(kern), statistics.median(total)
    nbytes = R * ((cfg.L + 31) // 32) * 16
    out = dict(shape=name, reads=R, L=cfg.L, events=len(reads), count_kernel_ms=k_ms, count_kernel_gb_per_s=nbytes / k_ms / 1e6,
               call_ms=t_ms, calls=len(res.count), count_kernel_ms_all=kern)
    hd.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default="T,C4")
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
