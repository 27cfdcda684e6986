#!/usr/bin/env python
"""bench.py -- juliet pileup + call + phase throughput (aligned CCS reads/s) on N B200s.

A "step" is one full pass of the hot path over one batch of synthetic reads.  `--config` picks the workload:

  T  (default) juliet --mode-phasing, 1 M reads x 3 kb PER GPU (weak scaling) -- the size BASELINE.json's metric and target are quoted on
  C1 juliet, 5 k reads x 3 kb            C3 juliet --mode-phasing, 200 k reads x 3 kb, 4 strains
  C2 fuse consensus, 50 k reads x 3 kb   C4 juliet, full HIV genome: 1 M reads x 9719 columns, 15 genes in 3 frames
  C5 phasing stress: 500 k reads x 6144 columns, 2048 dense variant sites, + co-occurrence matrix
  (C1..C5 = BASELINE.json configs[0..4]; their read totals are FIXED and split over the ranks: strong scaling)

step (juliet): pivot sample -> K1 pileup -> (N>1: one NCCL all-reduce of the count tensor) -> K2 codon test -> K3 phasing
(bit-vectors, grouping, all-gather + merge of the haplotype lists, order).

  value     reads/s with the packed reads resident in HBM (CUDA events on the launching stream, max over ranks)
  e2e       the same pass through the host-buffer C-ABI entry point: pinned host EVENT ROWS (the compact form of the
            CIGAR walk, include/minorseq_b200.h) -> H2D -> expansion on the GPU -> kernels -> D2H of the results
  roofline  K1 (pileup_csa_kernel): algorithmic bytes L/2 per read / its CUDA-event time, against the measured HBM copy
            bandwidth in MEASURED_PEAKS.json; `kernels` adds the phasing gather, the expansion and (C5) the tcgen05 kernel
  cpu_baseline  the CPU restatement (oracle/, "port": the reference ships no source), single-threaded, rank 0 at N=1
  digest    results of a fixed 65536-read batch sharded over the N ranks (outside the timed region); must equal the
            committed N=1 digest (tests/golden/bench_digest.json): counts and haplotypes are bit-identical for every N

`--impl reference` times the CPU restatement with all host threads on its own C-generated reads (states resident in host
memory before the timed region: no unpacking is timed).

`--dump-outputs DIR` writes what the last timed step returned (rank 0, float64 .npy files, at most 64 MB in all) so that
two builds can be compared output for output: the inputs depend only on the arguments.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "aligned CCS reads/sec pileup+call+phase"
MIN_PERC = 0.5   # juliet --min-perc (doc/JULIET.md:342-344): keeps the called set independent of the total read count
UNIT = "reads/s"
L2_BYTES = 126 << 20
HIV_GENES = [(1, 634), (790, 1186), (1186, 1879), (1879, 1921), (1921, 2086), (2086, 2134), (2134, 2292), (2253, 2550),
             (2550, 4230), (4230, 5096), (5041, 5620), (5559, 5850), (6062, 6310), (6225, 8795), (8797, 9417)]
# img juliet_target.png gives the first eight intervals and RT's start (SURVEY App. C-9); the rest cover all three frames

CONFIGS = {
    "T": dict(kind="juliet", L=3000, reads=1_000_000, scaling="weak", seed=20240003, phasing=True,
              what="juliet --mode-phasing, synthetic HIV-like amplicon, 4 strains (major + 10/5/1 % minors), one gene in frame 0, reference-guided"),
    "C1": dict(kind="juliet", L=3000, reads=5_000, scaling="strong", seed=20240001, phasing=True,
               what="BASELINE configs[0]: juliet on one synthetic pol amplicon, 5k CCS reads x 3 kb"),
    "C2": dict(kind="fuse", L=3000, reads=50_000, scaling="strong", seed=20240002, phasing=False,
               what="BASELINE configs[1]: fuse consensus of a 50k-read x 3 kb amplicon alignment"),
    "C3": dict(kind="juliet", L=3000, reads=200_000, scaling="strong", seed=20240003, phasing=True,
               what="BASELINE configs[2]: juliet with phasing, 200k reads x 3 kb, 4 mixed strains (1-10 % minors)"),
    "C4": dict(kind="juliet", L=9719, reads=1_000_000, scaling="strong", seed=20240004, phasing=True, genes=HIV_GENES, no_refseq=True,
               what="BASELINE configs[3]: juliet full HIV genome target config, 1M reads x 9719 columns, 15 genes in 3 frames, read-sharded"),
    "C5": dict(kind="stress", L=6144, reads=500_000, scaling="strong", seed=20240005, phasing=True,
               synth=dict(dense_sites=2048, dense_strains=64, n_rate=2e-5, dele=2e-5, trunc=0.0),
               what="BASELINE configs[4]: phasing stress, 500k reads x 6144 columns, 2048 dense variant sites (pileup + phasing + co-occurrence)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="T", choices=sorted(CONFIGS))
    ap.add_argument("--reads-per-gpu", type=int, default=0, help="config T only: reads per GPU (default 1M)")
    ap.add_argument("--L", type=int, default=0, help="override the config's reference length")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the CPU sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-digest", action="store_true")
    ap.add_argument("--write-digest", action="store_true", help="N=1 only: (re)write tests/golden/bench_digest.json")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU pass's outputs: it needs --impl ours")
    return args


def resolve(args, world):
    c = dict(CONFIGS[args.config])
    c["name"] = args.config
    if args.L:
        c["L"] = args.L
    if args.seed:
        c["seed"] = args.seed
    L = c["L"]
    c.setdefault("genes", [(1, L - L % 3 + 1)])
    if c["scaling"] == "weak":
        c["reads_per_gpu"] = args.reads_per_gpu or c["reads"]
        c["total_reads"] = c["reads_per_gpu"] * world
    else:
        c["total_reads"] = c["reads"]
        c["reads_per_gpu"] = (c["reads"] + world - 1) // world
    return c


def shard(c, rank, world):
    """[lo, hi) of the global read range this rank owns (contiguous ranges, SURVEY 8e)."""
    if c["scaling"] == "weak":
        return rank * c["reads_per_gpu"], (rank + 1) * c["reads_per_gpu"]
    per = c["reads_per_gpu"]
    return min(c["total_reads"], rank * per), min(c["total_reads"], (rank + 1) * per)


def workload_config(c, world):
    row_bytes = ((c["L"] + 31) // 32) * 16
    per_gpu = c["reads_per_gpu"] * row_bytes
    return {"workload": f"{c['name']}: {c['what']}; {c['total_reads']} reads x {c['L']} columns in total, {c['reads_per_gpu']} per GPU, --min-perc {MIN_PERC}",
            "config": c["name"], "total_reads": c["total_reads"], "reads_per_gpu": c["reads_per_gpu"], "L": c["L"], "seed": c["seed"], "min_perc": MIN_PERC,
            "l2_policy": ("packed input per GPU (%.2f GB) is larger than the 126 MB L2" % (per_gpu / 1e9)) if per_gpu > 2 * L2_BYTES else
                         ("packed input per GPU (%.1f MB) fits the L2: a 256 MB buffer is overwritten between timed steps, each step timed on its own" % (per_gpu / 1e6)),
            "parallelism": f"read-sharded x{world}, one NCCL all-reduce of the count tensor"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons (B200_PROFILING.md).  The subprocess is started BEFORE CUDA / NCCL
    are initialised (forking a process that already holds NCCL state can wedge later collectives) and keeps
    sampling every 20 ms; finish(t0, t1) reports the samples that fall inside the timed window."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.proc = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def run(self):
        if not self.proc:
            return
        try:
            for line in self.proc.stdout:
                self.rows.append((time.time(), [x.strip() for x in line.split(",")]))
        except Exception:
            pass

    def finish(self, t0, t1):
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        inside = [r for (ts, r) in self.rows if t0 - 0.02 <= ts <= t1 + 0.02]
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed steps + e2e steps"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def k1_source_hash():
    hsh = hashlib.sha256()
    for f in ("pileup.cu", "pileup.cuh"):
        hsh.update(open(os.path.join(ROOT, "minorseq_b200", "csrc", f), "rb").read())
    return hsh.hexdigest()[:16]


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_pass(oracle, st, c, refseq, nthreads):
    """One pass of the CPU restatement over resident column states (one byte per column); returns seconds."""
    from minorseq_b200.synth import start_mask_words
    L = c["L"]
    genes = c["genes"]
    words = start_mask_words(L, genes)
    mask = np.array([(int(words[j >> 5]) >> (j & 31)) & 1 for j in range(L)], dtype=np.uint8)
    t0 = time.perf_counter()
    if c["kind"] == "fuse":
        col, _ = oracle.pileup(st, None, codons=False, nthreads=nthreads)
        oracle.fuse(col)
        return time.perf_counter() - t0
    col, codon = oracle.pileup(st, mask, nthreads=nthreads)
    if c["kind"] == "stress":
        keys = c["sites"]
    else:
        v = oracle.call(codon, genes, refseq=refseq, min_perc=MIN_PERC)
        keys = sorted({(x.col, x.codon) for x in v})
    bits, flags = oracle.phase_bits(st, [k[0] for k in keys], [k[1] for k in keys], nthreads=nthreads)
    oracle.phase_group(bits, flags, len(keys))
    return time.perf_counter() - t0


def tables_for(c):
    from minorseq_b200.synth import SynthConfig, make_tables
    t = make_tables(SynthConfig(L=c["L"], seed=c["seed"], **c.get("synth", {})))
    if c["kind"] == "stress":
        c["sites"] = sorted({(col, k) for (_, col, k) in t.truth})
    return t


def run_reference(args, rank, world):
    """The CPU arm: the restatement in oracle/ (the reference ships documentation only), all host threads."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_binding
    oracle = oracle_binding.load()
    c = resolve(args, world)
    t = tables_for(c)
    cores = os.cpu_count() or 1
    # a bounded sample of the workload: what ~0.5 s per step of this machine's threads can take, at most one GPU's share
    sample = args.cpu_sample or int(min(c["reads_per_gpu"], 500_000 * 3000 // c["L"]))
    if c["kind"] == "stress":
        sample = args.cpu_sample or min(sample, 20_000)      # V = 2048: the serial sort of 256-byte patterns dominates
    st = oracle.synth_states(t, 0, sample, nthreads=cores)    # resident before the timed region (no unpacking is timed)
    refseq = None if c.get("no_refseq") else t.refseq
    for _ in range(max(1, args.warmup)):
        cpu_pass(oracle, st, c, refseq, cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        cpu_pass(oracle, st, c, refseq, cores)
    dt = (time.perf_counter() - t0) / args.steps
    v = sample / dt
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": c["scaling"],
            "vs_baseline": None, "dtype": "u32 counts / f64 p-values", "data": "synthetic", "config": workload_config(c, world),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{sample} reads of the same generator per step, column states resident in host memory (pileup and phase bits "
                                       f"OpenMP x{cores}; call and grouping serial); CPU RESTATEMENT written from doc/JULIET.md, not the juliet binary"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def bind_to_gpu_numa(local_rank):
    """Pin this rank's threads to the CPUs NVML names as local to its GPU (when the container's cpuset allows), so that
    the pinned staging buffers of the e2e path are first-touched on that GPU's NUMA node.  Returns the CPU count or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        ideal = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = ideal & allowed
        if len(cpus) >= 2 and cpus != allowed:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------ digest
DIGEST_READS = 65536
DIGEST_PATH = os.path.join(ROOT, "tests", "golden", "bench_digest.json")


def result_digest(j, res, lo, world, dist, torch, device):
    """Everything a juliet pass returns, hashed: all-reduced counts, variants (p-values bit for bit), the haplotype list in
    juliet's order, the six read categories and a position-weighted checksum of the per-read haplotype ids over all ranks."""
    col, codon = j.get_counts()
    hv = hashlib.sha256()
    for v in res.variants:
        hv.update(np.array([v.gene, v.codon_index, v.col, v.ref_codon, v.codon, v.count, v.coverage, v.expected, v.ntests], dtype=np.int64).tobytes())
        hv.update(np.float64(v.pvalue).tobytes())
    hp = res.haplotypes
    hh = hashlib.sha256()
    hh.update(np.ascontiguousarray(hp.patterns[: hp.nreported]).tobytes())
    hh.update(np.ascontiguousarray(hp.counts[: hp.nreported]).tobytes())
    ids = hp.hap_id.astype(np.int64)
    w = (np.arange(lo, lo + len(ids), dtype=np.int64) % 1000003) + 1
    chk = torch.tensor([int(((ids + 2) * w).sum())], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(chk, op=dist.ReduceOp.SUM)
    return {"reads": DIGEST_READS, "counts_sha256": hashlib.sha256(col.tobytes() + codon.tobytes()).hexdigest()[:32],
            "variants": len(res.variants), "variants_sha256": hv.hexdigest()[:32], "haplotypes_reported": int(hp.nreported),
            "distinct_patterns": int(hp.ndistinct), "haplotypes_sha256": hh.hexdigest()[:32], "counters": hp.counters,
            "hap_id_checksum": int(chk.item())}


# ------------------------------------------------------------------------------------------------ --dump-outputs
DUMP_LIMIT = 64 << 20
HAP_COUNTERS = ("reported", "insufficient", "damaged", "gaps", "heteroduplex", "partial")


def step_outputs(kind, j, res, cooc):
    """What a caller of the timed pass holds after it, as float64 arrays (every count and id here is exact in float64).
    variants: one row per call, columns gene, codon_index, col, ref_codon, codon, count, coverage, expected, ntests, pvalue.
    haplotype_summary: nreported, ndistinct, then the six read categories of HAP_COUNTERS."""
    def f8(a):
        return np.asarray(a, dtype=np.float64)

    if kind == "fuse":
        return {"consensus": f8(np.frombuffer(res.encode(), dtype=np.uint8))}
    col, codon = j.get_counts()
    out = {"col_counts": f8(col), "codon_counts": f8(codon)}
    hap = res
    if kind == "juliet":
        out["variants"] = f8([[v.gene, v.codon_index, v.col, v.ref_codon, v.codon, v.count, v.coverage, v.expected, v.ntests, v.pvalue]
                              for v in res.variants]).reshape(-1, 10)
        out["keys"] = f8(res.keys).reshape(-1, 2)
        hap = res.haplotypes
    else:
        out["cooccurrence"] = f8(cooc.cpu().numpy())
    if hap is not None:
        out["haplotype_patterns"] = f8(hap.patterns)
        out["haplotype_counts"] = f8(hap.counts)
        out["haplotype_summary"] = f8([hap.nreported, hap.ndistinct] + [hap.counters[k] for k in HAP_COUNTERS])
    return out


def dump_outputs(d, out):
    """Writes out as d/<name>.npy.  When the arrays exceed DUMP_LIMIT in all, each large one is cut to a fixed, seeded
    sample of its rows and the row indices go beside it as <name>_rows.npy."""
    os.makedirs(d, exist_ok=True)
    if sum(a.nbytes for a in out.values()) > DUMP_LIMIT:
        per = DUMP_LIMIT // (2 * len(out))
        for name, a in list(out.items()):
            if a.nbytes > per:
                keep = max(1, per // max(1, a.nbytes // len(a)))
                rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
                out[name], out[name + "_rows"] = a[rows], rows.astype(np.float64)
    for name, a in out.items():
        np.save(os.path.join(d, name + ".npy"), a)


def main():
    args = parse()
    if os.environ.get("BENCH_WATCHDOG"):
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["BENCH_WATCHDOG"]), exit=True)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"      # NCCL's version banner goes to stdout, in front of the one JSON line
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    affinity = bind_to_gpu_numa(local_rank) if world > 1 else None   # pinned buffers land on the GPU's NUMA node
    sampler = ClockSampler(local_rank)   # before CUDA / NCCL come up
    sampler.start()
    import torch
    import torch.distributed as dist
    from minorseq_b200 import Fuse, Juliet, _lib, encode_rows, host_rows, synth_device

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))
    c = resolve(args, world)
    t = tables_for(c)
    L = c["L"]
    lo, hi = shard(c, rank, world)
    Rg = hi - lo
    genes = c["genes"]
    refseq = None if c.get("no_refseq") else t.refseq
    if c["kind"] == "fuse":
        j = Fuse(L, device=local_rank)
    else:
        j = Juliet(L, genes, refseq=refseq, device=local_rank, mode_phasing=c["phasing"], min_perc=MIN_PERC)
    lib = j.lib
    if world > 1:
        j.hd.attach_comm()     # native ncclAllReduce / ncclAllGather on the handle's stream
    nw = int(lib.ms_row_words(L))

    def synth(tab, read0, n):
        return synth_device(j.hd, tab, read0, n)          # device tile layout (csrc/rows.cuh)

    def rows_to_host(n):
        """the first n reads of this rank's batch as plain host rows [n, row_words]"""
        return host_rows(d_packed[: int(lib.ms_tiled_words(L, n))], n, L)

    d_packed = synth(t, lo, Rg)
    torch.cuda.synchronize()
    _lib.check(lib.ms_set_timing(j.hd.h, 1), j.hd.h)

    class V:
        def __init__(self, col, k):
            self.col, self.codon = col, k
    site_vars = [V(col, k) for col, k in c.get("sites", [])]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def tail_stress(ptr):
        _lib.check(lib.ms_allreduce_counts(j.hd.h), j.hd.h)
        hap, _ = j.phase_device(site_vars, ptr, Rg, want_hap_id=False)
        return hap, j.cooccurrence()

    def step():
        if c["kind"] == "juliet":
            return j.run_device(d_packed.data_ptr(), Rg, want_hap_id=False)
        j.reset()
        j.pileup_device(d_packed.data_ptr(), Rg)
        if c["kind"] == "fuse":
            j.allreduce_counts()
            return j.consensus()
        return tail_stress(d_packed.data_ptr())

    flush_l2 = Rg * nw * 4 <= 2 * L2_BYTES
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if flush_l2 else None
    res = None
    for _ in range(max(3, args.warmup)):
        res = step()
    # ---- timed region: device-resident inputs
    k1_ms, launches0 = [], j.hd.launches
    barrier()
    t_window0 = time.time()
    el = C.c_double()
    elapsed_ms = 0.0
    if not flush_l2:
        _lib.check(lib.ms_timer_start(j.hd.h), j.hd.h)      # CUDA events on the stream the kernels are launched on
    for _ in range(args.steps):
        if flush_l2:
            flush_buf.fill_(1)
            torch.cuda.synchronize()
            _lib.check(lib.ms_timer_start(j.hd.h), j.hd.h)
        res = step()
        if flush_l2:
            _lib.check(lib.ms_timer_stop(j.hd.h, C.byref(el)), j.hd.h)
            elapsed_ms += el.value
        ms, rd = C.c_double(), C.c_int64()
        _lib.check(lib.ms_pileup_kernel_ms(j.hd.h, C.byref(ms), C.byref(rd)), j.hd.h)
        k1_ms.append(ms.value)
    if not flush_l2:
        _lib.check(lib.ms_timer_stop(j.hd.h, C.byref(el)), j.hd.h)
        elapsed_ms = el.value
    barrier()
    launches = j.hd.launches - launches0
    cooc = None
    if c["kind"] == "stress":
        res, cooc = res
    if args.dump_outputs and rank == 0:      # before the e2e pass below reuses the handle's buffers
        dump_outputs(args.dump_outputs, step_outputs(c["kind"], j, res, cooc))

    def stage_ms(stage):
        ms = C.c_double()
        return ms.value if lib.ms_stage_kernel_ms(j.hd.h, stage, C.byref(ms)) == 0 else None
    k3_ms, cooc_ms = stage_ms(1), stage_ms(2)
    allreduce_ms, hapmerge_ms = stage_ms(4), stage_ms(5)     # N > 1: the two exchanges of the pass, device time on this rank
    tm = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_per_step = float(tm.item()) / args.steps
    value = c["total_reads"] / (ms_per_step / 1e3)

    # ---- e2e: the host-buffer entry point (pinned host event rows -> H2D -> expansion -> kernels -> D2H results)
    e2e, expand_ms, expand_full_ms = None, None, None
    if not args.no_e2e:
        base = t.refseq                 # the sequence the rows are encoded against: the configured / major-strain reference
        rows_host = rows_to_host(Rg)
        hdr, ev = encode_rows(rows_host, L, base)
        del rows_host
        th = torch.from_numpy(hdr.view(np.uint8)).pin_memory()
        te = torch.from_numpy(ev if len(ev) else np.zeros(1, np.uint8)).pin_memory()
        hdr_p, ev_p = th.numpy().view(hdr.dtype), te.numpy()
        j.set_base(base)

        def e2e_step():
            if c["kind"] == "juliet":
                r = j.run_events_host(hdr_p, ev_p)
                col, codon = j.get_counts()
                return col.nbytes + codon.nbytes + len(r.variants) * 48 + (r.haplotypes.patterns.nbytes + r.haplotypes.counts.nbytes if r.haplotypes else 0)
            j.reset()
            keep = C.c_void_p()
            _lib.check(lib.ms_pileup_events_host(j.hd.h, hdr_p.ctypes.data_as(C.c_void_p), ev_p.ctypes.data_as(C.c_void_p), Rg, C.byref(keep)), j.hd.h)
            if c["kind"] == "fuse":
                j.allreduce_counts()
                return len(j.consensus()) + L * 32
            hap, _ = tail_stress(keep.value)
            return hap.patterns.nbytes + hap.counts.nbytes + L * 288
        for _ in range(2):
            e2e_step()
        barrier()
        esteps = args.steps
        d2h = 0
        t0 = time.perf_counter()
        for _ in range(esteps):
            d2h = e2e_step()
        barrier()
        dt = torch.tensor([(time.perf_counter() - t0) / esteps], dtype=torch.float64, device=dev)
        h2d = torch.tensor([hdr.nbytes + ev.nbytes], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dist.all_reduce(h2d, op=dist.ReduceOp.SUM)
        expand_ms = stage_ms(3)
        upload_ms, pass_ms = stage_ms(6), stage_ms(7)
        # the link's share: one plain pinned -> device copy of the same bytes, timed alone (box to box the PCIe rate differs by 30 %)
        dh_, de_ = torch.empty_like(th, device=dev), torch.empty_like(te, device=dev)
        for _ in range(2):
            dh_.copy_(th, non_blocking=True); de_.copy_(te, non_blocking=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(5):
            dh_.copy_(th, non_blocking=True); de_.copy_(te, non_blocking=True)
        torch.cuda.synchronize()
        copy_ms = (time.perf_counter() - t0) / 5 * 1e3
        # expand_events_kernel on the whole batch with the event rows already in HBM (device time, most recent of 3 launches)
        scratch = torch.empty(int(lib.ms_tiled_words(L, Rg)), dtype=torch.int32, device=dev)
        for _ in range(3):
            _lib.check(lib.ms_expand_events_dev(j.hd.h, C.c_void_p(dh_.data_ptr()), C.c_void_p(de_.data_ptr()), Rg, C.c_void_p(scratch.data_ptr())), j.hd.h)
        expand_full_ms = stage_ms(3)
        del dh_, de_, scratch
        e2e = {"value": c["total_reads"] / float(dt.item()), "unit": UNIT, "h2d_bytes_per_step": int(h2d.item()),
               "d2h_bytes_per_step": int(world * d2h), "ms_per_step": float(dt.item()) * 1e3, "steps": esteps,
               "upload_ms": upload_ms, "pass_device_ms": pass_ms, "plain_h2d_copy_ms": copy_ms, "plain_h2d_copy_gbs": (hdr.nbytes + ev.nbytes) / copy_ms / 1e6,
               "host_format": "event rows (ms_read_hdr + per-read event lists against the reference sequence: 1 byte per QV-filtered base, 12 bits per other event), expanded to packed reads on the GPU",
               "h2d_bytes_per_read": float(h2d.item()) / c["total_reads"], "planar_row_bytes_per_read": nw * 4}
        # for comparison: the same pass from planar rows in pinned host memory (round 1's e2e path), config T at N=1 only
        if c["name"] == "T" and world == 1:
            host = torch.from_numpy(rows_to_host(Rg).view(np.int32)).pin_memory()
            hp_ = host.numpy().view(np.uint32)
            j.run_host(hp_)
            t0 = time.perf_counter()
            for _ in range(2):
                j.run_host(hp_)
                j.get_counts()
            e2e["planar_rows_ms_per_step"] = (time.perf_counter() - t0) / 2 * 1e3
            del host

    clocks = sampler.finish(t_window0, time.time())

    # ---- digest: a fixed global batch sharded over the ranks, outside every timed region
    digest = None
    if c["kind"] == "juliet" and not args.no_digest and L == 3000 and refseq is not None:
        from minorseq_b200.synth import SynthConfig, make_tables
        td = make_tables(SynthConfig(L=3000, seed=20240003))
        dlo, dhi = DIGEST_READS * rank // world, DIGEST_READS * (rank + 1) // world
        dd = synth(td, dlo, dhi - dlo)
        jd = Juliet(3000, [(1, 3001)], refseq=td.refseq, mode_phasing=True, min_perc=MIN_PERC, handle=j.hd)
        rd_ = jd.run_device(dd.data_ptr(), dhi - dlo, want_hap_id=True)
        digest = result_digest(jd, rd_, dlo, world, dist, torch, dev)
        if args.write_digest and world == 1 and rank == 0:
            json.dump(digest, open(DIGEST_PATH, "w"), indent=1)
        try:
            digest["equals_committed_n1_digest"] = {k: v for k, v in digest.items()} == json.load(open(DIGEST_PATH))
        except Exception:
            digest["equals_committed_n1_digest"] = None

    # ---- roofline of the dominant kernel (K1) and of the other measured kernels
    peak, peak_src = measured_peak()
    k1 = float(np.mean(k1_ms))
    alg_bytes = Rg * (L / 2.0)
    achieved = alg_bytes / (k1 / 1e3) / 1e9
    traffic = None   # dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of THIS kernel build on this workload
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_k1_traffic.json")))
        if tj["workload"] == {"reads_per_gpu": Rg, "L": L} and tj.get("k1_source_sha") == k1_source_hash():
            traffic = tj["dram_bytes_read"] + tj["dram_bytes_write"]
    except Exception:
        pass
    roof = {"kernel": "pileup_csa_kernel", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "algorithmic_bytes": alg_bytes, "peak_source": peak_src, "algorithmic_bytes_per_read": L / 2.0, "kernel_ms": k1,
            "kernel_share_of_step": k1 / ms_per_step, "kernels": []}
    if k3_ms:
        keys = res.keys if c["kind"] == "juliet" else [(v.col, v.codon) for v in site_vars]
        nk = len(keys)
        nb = len({col >> 5 for col, _ in keys} | {(col + 2) >> 5 for col, _ in keys})     # distinct 32-column blocks the variants touch
        b = Rg * (16.0 * nb + 4.0 * ((nk + 31) // 32) + 1)
        roof["kernels"].append({"kernel": "phase_bits_kernel", "bound": "hbm", "variants": nk, "blocks": nb, "algorithmic_bytes": b, "kernel_ms": k3_ms,
                                "achieved": b / (k3_ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s", "frac": b / (k3_ms / 1e3) / 1e9 / peak,
                                "note": "algorithmic = 16 B per read and distinct touched block (tile layout: whole 128 B lines serve 8 reads) + bit-vector and flag out"})
    if expand_ms:
        b = Rg * (nw * 4.0) + float(e2e["h2d_bytes_per_step"]) / world
        k = {"kernel": "expand_events_kernel", "bound": "hbm", "algorithmic_bytes": b, "kernel_ms": expand_full_ms, "kernel_ms_last_chunk": expand_ms,
             "peak": peak, "unit": "GB/s",
             "note": f"writes {nw * 4} B and reads ~{e2e['h2d_bytes_per_read']:.0f} B per read; kernel_ms = the whole batch with its event rows resident "
                     "(instruction-bound: ncu summary in profiles/), kernel_ms_last_chunk = the last chunk of the e2e upload pipeline"}
        if expand_full_ms:
            k["achieved"] = b / (expand_full_ms / 1e3) / 1e9
            k["frac"] = k["achieved"] / peak
        roof["kernels"].append(k)
    if cooc_ms and c["kind"] == "stress":
        nk = len(site_vars)
        macs = float(nk) * nk * Rg     # the tcgen05 launch computes whole 256 x 256 tiles of the upper triangle; count the useful half + diagonal
        useful = macs / 2 + nk * Rg / 2
        roof["kernels"].append({"kernel": "cooccurrence_tc_kernel", "bound": "tensor", "variants": nk, "kernel_ms": cooc_ms,
                                "achieved": 2 * useful / (cooc_ms / 1e3) / 1e12, "unit": "Top/s (u8 MAC = 2 ops, useful upper triangle)",
                                "peak": 2 * json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops", 1673.6) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 4500.0,
                                "peak_source": "2 x measured dense bf16 TFLOP/s (int8 tensor rate is nominally twice bf16)"})
        k = roof["kernels"][-1]
        k["frac"] = k["achieved"] / k["peak"]

    # ---- CPU restatement beside it (rank 0, N=1)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_binding
        oracle = oracle_binding.load()
        probe = oracle.unpack(rows_to_host(min(2000, Rg)), L)
        tp = cpu_pass(oracle, probe, c, refseq, 1)
        sample = args.cpu_sample or int(min(Rg, max(2000, 2000 * 12.0 / max(tp, 1e-3))))
        st = oracle.unpack(rows_to_host(sample), L, nthreads=os.cpu_count() or 1)   # not timed
        ts = cpu_pass(oracle, st, c, refseq, 1)
        cpu = {"value": sample / ts, "unit": UNIT, "cores": 1, "kind": "port", "host_cores": os.cpu_count(),
               "sample": f"first {sample} reads of the same device-generated batch as resident column states, one pass, {ts:.1f} s; "
                         "CPU RESTATEMENT written from doc/JULIET.md (the reference ships no source), single-threaded"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": c["scaling"], "vs_baseline": None,
                "dtype": "u32 counts / f64 p-values", "data": "synthetic", "config": workload_config(c, world),
                "clocks": clocks, "e2e": e2e, "host_affinity_cpus": affinity, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
                "digest": digest}
        if world > 1:
            line["exchanges"] = {"count_allreduce_ms": allreduce_ms, "haplotype_allgather_and_merge_ms": hapmerge_ms,
                                 "note": "device time on rank 0 of the pass's two exchanges (NCCL all-reduce of the count tensor; "
                                         "all-gather of the compact pattern lists + the replicated merge kernels)"}
        if c["kind"] == "juliet":
            hp = res.haplotypes
            line["result_check"] = {"variants": len(res.variants), "haplotypes_reported": hp.nreported if hp else None, "counters": hp.counters if hp else None}
        elif c["kind"] == "fuse":
            line["result_check"] = {"consensus_length": len(res), "consensus_equals_major_strain": res == t.refseq}
        else:
            line["result_check"] = {"sites": len(site_vars), "distinct_patterns": res.ndistinct, "haplotypes_reported": res.nreported, "counters": res.counters}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
