"""Device time of pairwise linkage's stages, CUDA events on the handle's stream (ms_set_timing / ms_stage_kernel_ms):
phase_bits_kernel without and with the clean-codon matrix, the stacked [B | M] Gram contraction through each kernel
(popcount-AND, tcgen05), the statistics kernels, and -- with two GPUs -- the Gram all-reduce over a communicator.
    python tools/linkage_timing.py [--reps N] [--out FILE.json]
Shapes: T (1 M reads x 3 kb, the default mixture, the variants K2 calls) and C5 (500 k reads, 2048 dense sites).
Medians over N repetitions after one warm-up; the GPU's name and power limit are read in the same run."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from minorseq_b200 import Handle, Juliet, _lib, synth_device  # noqa: E402
from minorseq_b200._lib import LinkageParams  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables  # noqa: E402

STAGE_BITS, STAGE_GRAM, STAGE_STATS, STAGE_ALLREDUCE = 1, 2, 8, 9
SHAPES = {
    "T": (SynthConfig(L=3000, seed=20240001), 1_000_000),
    "C5": (SynthConfig(L=6144, seed=20240005, dense_sites=2048, dense_strains=64, n_rate=2e-5, dele=2e-5, trunc=0.0), 500_000),
}


def stage(hd, s):
    ms = C.c_double()
    _lib.check(hd.lib.ms_stage_kernel_ms(hd.h, s, C.byref(ms)), hd.h)
    return ms.value


def keys_of(hd, t, d, R):
    if t.cfg.dense_sites:
        return sorted({(c, k) for (_, c, k) in t.truth})
    j = Juliet(t.cfg.L, [(1, t.cfg.L + 1)], handle=hd)
    j.pileup_device(d.data_ptr(), R)
    return sorted({(v.col, v.codon) for v in j.call()})


def phase(hd, keys, d, R, linkage):
    import numpy as np
    vc = np.array([k[0] for k in keys], dtype=np.int32)
    vk = np.array([k[1] for k in keys], dtype=np.int32)
    lib = hd.lib
    _lib.check(lib.ms_set_linkage(hd.h, 1 if linkage else 0), hd.h)
    _lib.check(lib.ms_phase_begin(hd.h, vc.ctypes.data, vk.ctypes.data, len(keys), R), hd.h)
    _lib.check(lib.ms_phase_dev(hd.h, C.c_void_p(d.data_ptr()), R), hd.h)


def gram(hd):
    g, dim = C.c_void_p(), C.c_int32()
    _lib.check(hd.lib.ms_linkage_device(hd.h, C.byref(g), C.byref(dim)), hd.h)
    _lib.check(hd.lib.ms_synchronize(hd.h), hd.h)
    return dim.value


def measure(name, reps):
    cfg, R = SHAPES[name]
    t = make_tables(cfg)
    hd = Handle(0)
    lib = hd.lib
    _lib.check(lib.ms_set_layout(hd.h, cfg.L, None), hd.h)
    d = synth_device(hd, t, 0, R)
    keys = keys_of(hd, t, d, R)
    _lib.check(lib.ms_set_layout(hd.h, cfg.L, None), hd.h)
    _lib.check(lib.ms_set_timing(hd.h, 1), hd.h)
    out = dict(shape=name, reads=R, L=cfg.L, variants=len(keys))
    for linkage in (False, True):
        times = []
        for i in range(reps + 1):
            phase(hd, keys, d, R, linkage)
            _lib.check(lib.ms_synchronize(hd.h), hd.h)
            if i:
                times.append(stage(hd, STAGE_BITS))
        out["phase_bits_ms_" + ("with_M" if linkage else "without_M")] = statistics.median(times)
    p = LinkageParams()
    lib.ms_linkage_params_default(C.byref(p))
    n, m = C.c_int64(), C.c_int64()
    for variant, label in ((1, "popcount"), (2, "tcgen05")):
        _lib.check(lib.ms_set_cooccurrence_variant(hd.h, variant), hd.h)
        gt, st, wall = [], [], []
        for i in range(reps + 1):
            phase(hd, keys, d, R, True)
            out["gram_dim"] = gram(hd)
            t0 = time.perf_counter()
            _lib.check(lib.ms_linkage(hd.h, C.byref(p), None, 0, C.byref(n), C.byref(m)), hd.h)   # Gram cached: statistics only
            if i:
                wall.append(1e3 * (time.perf_counter() - t0))
                gt.append(stage(hd, STAGE_GRAM))
                st.append(stage(hd, STAGE_STATS))
        out[f"gram_ms_{label}"] = statistics.median(gt)
        out[f"stats_ms_{label}_run"] = statistics.median(st)
        out[f"ms_linkage_host_ms_{label}_run"] = statistics.median(wall)
    _lib.check(lib.ms_set_cooccurrence_variant(hd.h, 0), hd.h)
    out["tested_pairs"], out["significant_pairs"] = m.value, n.value
    hd.close()
    return out


def measure_allreduce(name, reps):
    """two ranks on devices 0 and 1 (one thread each), each phasing half of the reads; the Gram all-reduce per call"""
    cfg, R = SHAPES[name]
    t = make_tables(cfg)
    hds = [Handle(0), Handle(1)]
    ident = C.create_string_buffer(128)
    _lib.check(hds[0].lib.ms_comm_unique_id(ident))
    half = [(0, R // 2 // 8 * 8), (R // 2 // 8 * 8, R)]
    rows = [synth_device(hds[r], t, half[r][0], half[r][1] - half[r][0]) for r in range(2)]
    keys = keys_of(hds[0], t, rows[0], half[0][1]) if cfg.dense_sites else None
    if keys is None:       # the T keys as one GPU calls them on all reads
        hd1 = Handle(0)
        dall = synth_device(hd1, t, 0, R)
        keys = keys_of(hd1, t, dall, R)
        del dall
        hd1.close()
    res = [[], []]
    errs = []

    def rank(r):
        try:
            hd = hds[r]
            _lib.check(hd.lib.ms_comm_init(hd.h, ident, r, 2), hd.h)
            _lib.check(hd.lib.ms_set_layout(hd.h, cfg.L, None), hd.h)
            _lib.check(hd.lib.ms_set_timing(hd.h, 1), hd.h)
            for i in range(reps + 1):
                phase(hd, keys, rows[r], half[r][1] - half[r][0], True)
                gram(hd)
                if i:
                    res[r].append(stage(hd, STAGE_ALLREDUCE))
        except Exception as e:        # reported by the main thread
            errs.append(repr(e))

    th = [threading.Thread(target=rank, args=(r,)) for r in range(2)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    for hd in hds:
        hd.close()
    if errs:
        raise RuntimeError("; ".join(errs))
    return dict(shape=name, ranks=2, allreduce_ms_rank0=statistics.median(res[0]), allreduce_ms_rank1=statistics.median(res[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("linkage_timing.py needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = dict(gpu=gpu.splitlines(), results=[])
    for name in SHAPES:
        r = measure(name, a.reps)
        print(json.dumps(r), flush=True)
        report["results"].append(r)
    if torch.cuda.device_count() >= 2:
        for name in SHAPES:
            r = measure_allreduce(name, a.reps)
            print(json.dumps(r), flush=True)
            report["results"].append(r)
    else:
        report["allreduce"] = "not measured: one GPU"
    print(json.dumps(dict(gpu=report["gpu"])), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()
