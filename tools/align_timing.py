"""K6 read alignment: 200 k and 1 M reads x 3 kb against a 3.3 kb amplicon, half of them reverse-strand.

Times the seed and band kernels (CUDA events around the last chunk's launches, MS_STAGE_ALIGN_SEED / _BAND; the band kernel
includes the traceback) and the whole ms_align_reads call from host arrays (host clock, the call ends in a synchronise),
medians after one warm-up.  GCUPS = band cells by count over band-kernel time; the count is 128 cells per anti-diagonal from
the start diagonal to the band's exit at the reference's end, la + lb - pos anti-diagonals per read (an upper bound).  Also the
CPU restatement's single-thread reads/s on a sample.  Reads carry 1 % substitutions and 1 % deletions."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from minorseq_b200 import Aligner, _lib  # noqa: E402
from align_oracle import AlignOracle  # noqa: E402



def _constants():
    """The stage ids and ms_align_reads' chunk rule, read from the headers that define them."""
    import re
    text = open(os.path.join(ROOT, "include", "minorseq_b200.h")).read() + open(os.path.join(ROOT, "minorseq_b200", "csrc", "align_rule.h")).read()
    return {k: int(v) for k, v in re.findall(r"\b(MS_STAGE_ALIGN_\w+|MS_ALN_CHUNK_\w+) = (\d+)", text)}


K = _constants()
COMP = np.zeros(256, dtype=np.uint8)
for a, b in zip(b"ACGTN", b"TGCAN"):
    COMP[a] = b


def make_reads(rng, ref, R, la=3000, block=50000):
    r = np.frombuffer(ref.encode(), dtype=np.uint8)
    parts, lens = [], []
    for r0 in range(0, R, block):
        n = min(block, R - r0)
        start = rng.integers(0, len(r) - la + 1, n)
        m = r[start[:, None] + np.arange(la)[None, :]]
        sub = rng.random(m.shape, dtype=np.float32) < 0.01
        m[sub] = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, int(sub.sum()))]
        rev = rng.random(n) < 0.5
        m[rev] = COMP[m[rev, ::-1]]
        keep = rng.random(m.shape, dtype=np.float32) >= 0.01
        parts.append(m[keep].tobytes())
        lens.append(keep.sum(1))
    off = np.zeros(R + 1, dtype=np.int64)
    off[1:] = np.cumsum(np.concatenate(lens))
    return b"".join(parts), off


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="200000,1000000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    rng = np.random.default_rng(2026)
    ref = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, 3300)].tobytes().decode()
    al = Aligner(device=0)
    al.set_reference(ref)
    lib, h = al.lib, al.hd.h
    check = _lib.check
    check(lib.ms_set_timing(h, 1), h)
    res = {"gpu": smi, "reference": len(ref), "read_length": 3000}
    for R in [int(x) for x in args.sizes.split(",")]:
        seq, off = make_reads(rng, ref, R)
        out = (_lib.ReadAlignment * R)()
        cap = int(off[-1] // 4)
        cig = np.zeros(cap, dtype=np.uint32)
        n = C.c_int64()
        walls, seeds, bands = [], [], []
        for rep in range(args.reps + 1):
            t0 = time.perf_counter()
            check(lib.ms_align_reads(h, C.byref(al.params), seq, off.ctypes.data_as(C.c_void_p), R, out, cig.ctypes.data_as(C.c_void_p),
                                     cap, C.byref(n)), h)
            wall = time.perf_counter() - t0
            s, b = C.c_double(), C.c_double()
            check(lib.ms_stage_kernel_ms(h, K["MS_STAGE_ALIGN_SEED"], C.byref(s)), h)
            check(lib.ms_stage_kernel_ms(h, K["MS_STAGE_ALIGN_BAND"], C.byref(b)), h)
            if rep:
                walls.append(wall); seeds.append(s.value); bands.append(b.value)
        r0 = 0                                # the first read of the last chunk (ms_align_reads' chunk rule), which the stage events time
        while True:
            r1 = r0 + 1
            while r1 < R and r1 - r0 < K["MS_ALN_CHUNK_READS"] and off[r1 + 1] - off[r0] <= K["MS_ALN_CHUNK_MBASES"] << 20:
                r1 += 1
            if r1 == R:
                break
            r0 = r1
        last = R - r0
        mapped = sum(out[r].mapped for r in range(R))
        rev = sum(out[r].strand for r in range(R) if out[r].mapped)
        cells = 128.0 * float(sum((off[r + 1] - off[r]) + len(ref) - out[r].pos for r in range(R - last, R) if out[r].mapped))
        row = {"reads": R, "mapped": mapped, "reverse": rev, "call_s": statistics.median(walls),
               "reads_per_s": R / statistics.median(walls), "last_chunk_reads": last,
               "seed_ms": statistics.median(seeds), "band_ms": statistics.median(bands),
               "seed_reads_per_s": last / statistics.median(seeds) * 1e3, "band_reads_per_s": last / statistics.median(bands) * 1e3,
               "band_gcups_by_count": cells / (statistics.median(bands) * 1e-3) / 1e9}
        res[f"R{R}"] = row
        print(json.dumps(row), flush=True)
    ao = AlignOracle()
    ao.set_reference(ref)
    seq, off = make_reads(rng, ref, 100)
    reads = [seq[off[r]:off[r + 1]].decode() for r in range(100)]
    t0 = time.perf_counter()
    ao.align(reads)
    res["oracle_reads_per_s_single_thread"] = 100 / (time.perf_counter() - t0)
    print(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
