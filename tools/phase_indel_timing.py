"""Device time of phasing with in-frame indel keys (restatement choice U20): ms_phase_dev with and without two deletion and two
insertion keys after the called substitution keys (CUDA events on the handle's stream, ms_timer_start / ms_timer_stop), and
the new kernels' own times (torch.profiler, CUDA activities, in a separate pass).  The rate printed for phase_indel_kernel is
16 B x touched blocks x reads over its time.
    python tools/phase_indel_timing.py [--reps N] [--out FILE.json]
Shapes: T (1 M reads x 3 kb, one gene) and C4 (1 M reads x 9719 columns, HIV's 15 genes); 1 % of the reads carry an insertion
event (half at each insertion key's boundary).  The tiles (1.5 GB and 4.9 GB) are far larger than L2.  Medians over N
repetitions after one warm-up; one GPU.  The GPU's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
from types import SimpleNamespace

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from minorseq_b200 import Handle, Juliet, _lib, synth_device  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
# (config, reads, genes, deletion starts, insertion boundaries): codon starts and boundaries of gene 0 (T) / of Pol (C4)
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240003), 1_000_000, None, (300, 603), (302, 605)),
    "C4": (SynthConfig(L=9719, seed=20240004), 1_000_000, HIV_GENES, (2750, 3053), (2752, 3055)),
}


def measure(name, reps):
    import torch
    cfg, R, genes, dels, ins = SHAPES[name]
    t = make_tables(cfg)
    hd = Handle(0)
    j = Juliet(cfg.L, genes or [(1, cfg.L + 1)], handle=hd, refseq=None if genes else t.refseq)
    d = synth_device(hd, t, 0, R)
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    reads = np.arange(0, R, 100, dtype=np.int64)
    n = len(reads)
    ev = (np.concatenate([reads, reads + 50]), np.repeat(np.array(ins, dtype=np.int32), n), np.repeat(np.array([0, 6], dtype=np.int64), n),
          np.repeat(np.array([6, 3], dtype=np.int32), n), b"TCTTCTAAA")
    order = np.argsort(ev[0], kind="stable")
    ev = tuple(a[order] for a in ev[:4]) + (ev[4],)
    res = j.indels(d.data_ptr(), R, insertions=ev)
    sids = [s for s in range(len(res.strings)) if res.string_col[s] in ins]
    assert len(sids) == 2, res.strings
    rec = SimpleNamespace(kind=[0, 0, 1, 1], col=list(dels) + [int(res.string_col[s]) for s in sids], sid=[-1, -1] + sids,
                          string_col=res.string_col, strings=res.strings)
    V = len({(v.col, v.codon) for v in variants})

    out = dict(shape=name, reads=R, L=cfg.L, substitution_keys=V, indel_keys=4, events=2 * n)
    for tag, indels in (("without", None), ("with", rec)):
        times = []
        for i in range(reps + 1):      # ms_phase_dev alone between CUDA events; ms_phase_begin_indels outside the window
            _begin(j, variants, indels, R)
            _lib.check(hd.lib.ms_timer_start(hd.h), hd.h)
            _lib.check(hd.lib.ms_phase_dev(hd.h, C.c_void_p(d.data_ptr()), R), hd.h)
            ms = C.c_double()
            _lib.check(hd.lib.ms_timer_stop(hd.h, C.byref(ms)), hd.h)
            if i:
                times.append(ms.value)
        out[f"phase_dev_ms_{tag}"] = statistics.median(times)
        out[f"phase_dev_ms_{tag}_all"] = times
    # the kernels' own times
    from torch.profiler import ProfilerActivity, profile
    _begin(j, variants, rec, R)
    _lib.check(hd.lib.ms_phase_dev(hd.h, C.c_void_p(d.data_ptr()), R), hd.h)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            _begin(j, variants, rec, R)
            _lib.check(hd.lib.ms_phase_dev(hd.h, C.c_void_p(d.data_ptr()), R), hd.h)
        _lib.check(hd.lib.ms_synchronize(hd.h), hd.h)
    per = {}
    for e in prof.events():
        for k in ("phase_indel_kernel", "phase_indel_ins_kernel", "phase_bits_kernel"):
            if k in e.name and (k != "phase_indel_kernel" or "ins_kernel" not in e.name):
                per.setdefault(k, []).append(e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3)
    blocks = len({c >> 5 for c in dels} | {(c + 2) >> 5 for c in dels} | {c >> 5 for c in ins} | {(c + 1) >> 5 for c in ins})
    for k, v in per.items():
        out[f"{k}_ms"] = statistics.median(v)
    if "phase_indel_kernel" in per:
        out["phase_indel_kernel_touched_blocks"] = blocks
        out["phase_indel_kernel_gb_per_s"] = 16 * blocks * R / out["phase_indel_kernel_ms"] / 1e6
    hd.close()
    torch.cuda.synchronize()
    return out


def _begin(j, variants, indels, R):
    """ms_phase_begin_indels as Juliet.phase_device issues it, without the phasing that follows"""
    keys = sorted({(v.col, v.codon) for v in variants})
    vc = np.array([k[0] for k in keys], dtype=np.int32)
    vd = np.array([k[1] for k in keys], dtype=np.int32)
    dcol = np.array(sorted({int(c) for k, c in zip(indels.kind, indels.col) if k == 0}) if indels else [], dtype=np.int32)
    isid = np.array(sorted({int(s) for k, s in zip(indels.kind, indels.sid) if k == 1}) if indels else [], dtype=np.int32)
    _lib.check(j.lib.ms_phase_begin_indels(j.hd.h, vc.ctypes.data, vd.ctypes.data, len(keys), dcol.ctypes.data, len(dcol), isid.ctypes.data,
                                           len(isid), R), j.hd.h)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
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
