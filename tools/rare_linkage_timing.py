"""Device time of sub-threshold variant linkage (restatement choice U21), stage by stage, CUDA events on the handle's stream
(ms_timer_start / ms_timer_stop) around each C-ABI call, which ends in a host synchronise:
    candidates   ms_rare_candidates (rare_candidate_kernel, the download and the host merge)
    bits         ms_phase_begin + ms_phase_dev on the called keys ++ candidates, with the clean-codon matrix
    gram         ms_linkage_device (the stacked [B | M] Gram matrix; tcgen05 at >= 256 keys and >= 32768 reads)
    pairs        ms_rare_linkage (rare_count_kernel, rare_pair_kernel, the download and the sort)
    support      ms_rare_support over the groups
and the whole of Juliet.rare_linkage with a host clock.
    python tools/rare_linkage_timing.py [--reps N] [--out FILE.json] [--shapes T,C4,S6k]
Shapes: T (1 M reads x 3 kb, one gene, the default 10 / 5 / 1 % mixture), C4 (1 M reads x 9719 columns, HIV's 15 genes), S6k
(6000 reads x 3 kb with a 0.25 % strain of four codons, the detection case).  Medians over N repetitions after one warm-up;
one GPU, so no all-reduce is timed.  The GPU's name and power limit are read in the same run."""
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
from minorseq_b200._lib import Gene, LinkagePair, LinkageParams, RareParams, Variant  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240003), 1_000_000, None),
    "C4": (SynthConfig(L=9719, seed=20240004), 1_000_000, HIV_GENES),
    "S6k": (SynthConfig(L=3000, seed=3, minor_fracs=(0.0025,), variants_per_minor=(4, 4)), 6000, None),
}


def measure(name, reps):
    import torch
    cfg, R, genes = SHAPES[name]
    genes = genes or [(1, cfg.L + 1)]
    t = make_tables(cfg)
    hd = Handle(0)
    lib = hd.lib
    j = Juliet(cfg.L, genes, handle=hd)
    d = synth_device(hd, t, 0, R)
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    called = sorted({(v.col, v.codon) for v in variants})
    fc = len(called)
    g = (Gene * len(genes))(*[Gene(b, e) for (b, e) in genes])
    rp = RareParams()
    lib.ms_rare_params_default(C.byref(rp))
    lp = LinkageParams(j.params.alpha, 10)
    cand = (Variant * 4096)()
    pairs = (LinkagePair * 65536)()
    n, dropped, m = C.c_int64(), C.c_int64(), C.c_int64()

    def timed(fn):
        _lib.check(lib.ms_timer_start(hd.h), hd.h)
        fn()
        ms = C.c_double()
        _lib.check(lib.ms_timer_stop(hd.h, C.byref(ms)), hd.h)
        return ms.value

    stages = {k: [] for k in ("candidates", "bits", "gram", "pairs", "support", "whole_call")}
    info = {}
    for i in range(reps + 1):
        st = {}
        st["candidates"] = timed(lambda: _lib.check(lib.ms_rare_candidates(hd.h, g, len(genes), None, C.byref(j.params), C.byref(rp), cand, 4096,
                                                                           C.byref(n), C.byref(dropped)), hd.h))
        nc = int(n.value)
        keys = called + [(cand[k].col, cand[k].codon) for k in range(nc)]
        vc = np.array([k[0] for k in keys], dtype=np.int32)
        vd = np.array([k[1] for k in keys], dtype=np.int32)
        _lib.check(lib.ms_set_linkage(hd.h, 1), hd.h)

        def bits():
            _lib.check(lib.ms_phase_begin(hd.h, vc.ctypes.data, vd.ctypes.data, len(keys), R), hd.h)
            _lib.check(lib.ms_phase_dev(hd.h, C.c_void_p(d.data_ptr()), R), hd.h)
        st["bits"] = timed(bits)
        gp, dim = C.c_void_p(), C.c_int32()
        st["gram"] = timed(lambda: (_lib.check(lib.ms_linkage_device(hd.h, C.byref(gp), C.byref(dim)), hd.h),
                                    _lib.check(lib.ms_synchronize(hd.h), hd.h)))
        st["pairs"] = timed(lambda: _lib.check(lib.ms_rare_linkage(hd.h, fc, C.byref(lp), pairs, 65536, C.byref(n), C.byref(m)), hd.h))
        npairs = min(int(n.value), 65536)
        grp = np.full(max(1, len(keys)), -1, dtype=np.int32)
        ng = lib.ms_rare_groups(pairs, npairs, fc, len(keys), grp.ctypes.data)
        nw = max(1, (len(keys) + 31) // 32)
        masks = np.zeros((max(1, ng), nw), dtype=np.uint32)
        for k in range(len(keys)):
            if grp[k] >= 0:
                masks[grp[k], k >> 5] |= np.uint32(1 << (k & 31))
        car, inf = np.zeros(max(1, ng), np.uint64), np.zeros(max(1, ng), np.uint64)
        st["support"] = timed(lambda: _lib.check(lib.ms_rare_support(hd.h, masks.ctypes.data, ng, car.ctypes.data, inf.ctypes.data), hd.h))
        t0 = time.perf_counter()
        j.rare_linkage(d.data_ptr(), R, variants=variants)
        st["whole_call"] = 1e3 * (time.perf_counter() - t0)
        info = dict(called_keys=fc, candidates=nc, dropped=int(dropped.value), tested_pairs=int(m.value), linked_pairs=npairs, groups=int(ng),
                    gram_dim=int(dim.value))
        if i:
            for k, v in st.items():
                stages[k].append(v)
    out = dict(shape=name, reads=R, L=cfg.L, **info)
    for k, v in stages.items():
        out[f"{k}_ms"] = statistics.median(v)
    hd.close()
    torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default="T,C4,S6k")
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
