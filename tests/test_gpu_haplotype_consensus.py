"""Grouped pile-up and per-haplotype consensus on the GPU (restatement choice U15) against numpy and the test-side oracle
(haplotype_consensus_oracle.py), and the generator's known answer on a C3-shaped mixture."""
import ctypes as C
import os
import socket
import sys

import numpy as np
import pytest

import haplotype_consensus_oracle as hco
from minorseq_b200 import Fuse, Handle, Juliet, synth_device
from minorseq_b200._lib import FuseParams
from minorseq_b200.synth import SynthConfig, make_tables, read_strains

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C3 = SynthConfig(L=3000, seed=20240003)       # bench.py's C3 mixture: major + 10 / 5 / 1 % minors
C3_READS = 40_000                             # >= 200 reads of the 1 % strain


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def _labels(R, ngroups, rng):
    """random labels (including -1 and >= ngroups) with groups of 0, 1, 2047, 2048 and 5000 reads where ngroups allows"""
    lab = rng.integers(-1, ngroups + 2, size=R).astype(np.int32)
    perm = rng.permutation(R)
    sizes = [5000, 2047, 2048, 1, 0][:ngroups] if ngroups > 1 else [5000]
    start = 0
    for g, n in enumerate(sizes):
        lab[lab == g] = -1
        lab[perm[start: start + n]] = g
        start += n
    return lab


@pytest.mark.parametrize("L", [900, 3000, 9719])
@pytest.mark.parametrize("ngroups", [1, 3, 200])
def test_group_counts_equal_numpy(hd, oracle, L, ngroups):
    R = 12_003                                                  # not a multiple of 8
    t = make_tables(SynthConfig(L=L, seed=300 + L))
    j = Juliet(L, [(1, L + 1)], handle=hd)
    d = synth_device(hd, t, 0, R)
    states = oracle.synth_states(t, 0, R, nthreads=8)
    lab = _labels(R, ngroups, np.random.default_rng(L + ngroups))
    d_lab = torch.from_numpy(lab).cuda()
    torch.cuda.synchronize()                                    # the labels are copied on torch's stream
    j.group_pileup(d.data_ptr(), d_lab.data_ptr(), R, ngroups)
    got = j.group_counts()
    np.testing.assert_array_equal(got, hco.group_counts(states, lab, ngroups))
    if ngroups >= 5:
        assert got[4].sum() == 0 and got[3, :, 7].max() <= 1


def test_one_group_equals_k1(hd):
    """every read in group 0: the group's counts are K1's column counts (with the insertion tally on), at 200 k x 3 kb"""
    L, R = 3000, 200_000
    t = make_tables(SynthConfig(L=L, seed=20240003))
    j = Juliet(L, [(1, L + 1)], handle=hd)
    d = synth_device(hd, t, 0, R)
    j.set_count_insertions(True)
    j.pileup_device(d.data_ptr(), R)
    col, _ = j.get_counts()
    lab = torch.zeros(R, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    j.group_pileup(d.data_ptr(), lab.data_ptr(), R, 1)
    np.testing.assert_array_equal(j.group_counts()[0], col)
    assert col[:, 6].sum() > 0


def test_two_accumulating_calls_equal_one(hd):
    L, R, R1 = 3000, 20_003, 8_000                              # the second call starts at a tile (multiple of 8 reads)
    t = make_tables(SynthConfig(L=L, seed=5))
    j = Juliet(L, [(1, L + 1)], handle=hd)
    d = synth_device(hd, t, 0, R)
    lab = torch.from_numpy(_labels(R, 3, np.random.default_rng(9))).cuda()
    torch.cuda.synchronize()
    j.group_pileup(d.data_ptr(), lab.data_ptr(), R, 3)
    one = j.group_counts()
    tile_bytes = ((L + 31) // 32) * 128
    j.group_pileup(d.data_ptr(), lab.data_ptr(), R1, 3)
    j.group_pileup(d.data_ptr() + (R1 // 8) * tile_bytes, lab.data_ptr() + 4 * R1, R - R1, 3, accumulate=True)
    np.testing.assert_array_equal(j.group_counts(), one)


def _strain_insertions(t, R, strain, col, s=b"GGC"):
    st, _, _ = read_strains(t, 0, R)
    read = np.nonzero(st == strain)[0]
    return (read, np.full(len(read), col), np.zeros(len(read), dtype=np.int64), np.full(len(read), len(s)), s)


@pytest.fixture(scope="module")
def c3_run(hd):
    t = make_tables(C3)
    R = C3_READS
    d = synth_device(hd, t, 0, R)
    j = Juliet(C3.L, [(1, C3.L + 1)], refseq=t.refseq, handle=hd, mode_phasing=True)
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    haps, keys = j.phase_device(variants, d.data_ptr(), R)
    ins = _strain_insertions(t, R, 2, 1500)
    plain = j.haplotype_consensus(d.data_ptr(), R)
    counts = j.group_counts()
    with_ins = j.haplotype_consensus(d.data_ptr(), R, insertions=ins)
    return dict(t=t, R=R, d=d, j=j, haps=haps, keys=keys, plain=plain, counts=counts, with_ins=with_ins, ins=ins)


def _pattern_of(keys, cols_codons):
    nw = max(1, (len(keys) + 31) // 32)
    p = np.zeros(nw, dtype=np.uint32)
    for v, k in enumerate(keys):
        if k in cols_codons:
            p[v >> 5] |= np.uint32(1 << (v & 31))
    return p


def test_known_answer_every_strain(c3_run):
    t, haps, keys, seqs = c3_run["t"], c3_run["haps"], c3_run["keys"], c3_run["plain"]
    assert len(seqs) == haps.nreported >= 4
    strains, _, _ = read_strains(t, 0, c3_run["R"])
    for s in range(t.nstrains):
        assert (strains == s).sum() >= 200
        planted = {(c, k) for (ss, c, k) in t.truth if ss == s}
        assert planted <= set(keys)
        want = _pattern_of(keys, planted)
        ks = [k for k in range(haps.nreported) if np.array_equal(haps.patterns[k], want)]
        assert len(ks) == 1, f"strain {s}: no reported haplotype with exactly its codons"
        assert seqs[ks[0]] == "".join("ACGT"[b] for b in t.strain_base[s]), f"strain {s}"


def test_major_haplotype_equals_fuse(c3_run):
    t, d, R = c3_run["t"], c3_run["d"], c3_run["R"]
    f = Fuse(C3.L, handle=Handle(0))
    f.pileup_device(d.data_ptr(), R)
    assert c3_run["plain"][0] == f.consensus() == "".join("ACGT"[b] for b in t.strain_base[0])


def test_planted_insertion_only_in_its_strain(c3_run):
    t, haps, plain, got = c3_run["t"], c3_run["haps"], c3_run["plain"], c3_run["with_ins"]
    strains, _, _ = read_strains(t, 0, c3_run["R"])
    want = _pattern_of(c3_run["keys"], {(c, k) for (ss, c, k) in t.truth if ss == 2})
    k2 = [k for k in range(haps.nreported) if np.array_equal(haps.patterns[k], want)][0]
    assert got[k2] == plain[k2][:1501] + "GGC" + plain[k2][1501:]
    for k in range(haps.nreported):
        if got[k] != plain[k]:          # only haplotypes made of strain 2's reads
            assert np.all(strains[haps.hap_id == k] == 2)


def test_parity_with_oracle(c3_run, oracle):
    t, haps, R = c3_run["t"], c3_run["haps"], c3_run["R"]
    states = oracle.synth_states(t, 0, R, nthreads=8)
    lab = np.where(haps.hap_id < haps.nreported, haps.hap_id, -1)
    np.testing.assert_array_equal(c3_run["counts"], hco.group_counts(states, lab, haps.nreported))
    assert c3_run["plain"] == hco.haplotype_consensus(states, lab, haps.nreported)
    assert c3_run["with_ins"] == hco.haplotype_consensus(states, lab, haps.nreported, c3_run["ins"])
    assert hco.haplotype_consensus(states, lab, haps.nreported, c3_run["ins"], min_coverage=400) == \
        c3_run["j"].haplotype_consensus(c3_run["d"].data_ptr(), R, insertions=c3_run["ins"], min_coverage=400)


def test_capacity_retry_returns_the_same_sequences(c3_run):
    j, seqs = c3_run["j"], c3_run["plain"]
    lib = j.lib
    nrep = len(seqs)
    prm = FuseParams(10, 0.5, 20)
    off = np.zeros(nrep + 1, dtype=np.int64)
    small = np.zeros(16, dtype=np.uint8)
    rc = lib.ms_group_consensus(j.hd.h, C.byref(prm), None, None, None, None, 0, None, 0, small.ctypes.data, 16, off.ctypes.data)
    assert rc == -4 and off[-1] == sum(len(s) for s in seqs)
    rc = lib.ms_group_consensus(j.hd.h, C.byref(prm), None, None, None, None, 0, None, 0, None, 0, off.ctypes.data)
    assert rc == -4
    buf = np.zeros(int(off[-1]), dtype=np.uint8)
    assert lib.ms_group_consensus(j.hd.h, C.byref(prm), None, None, None, None, 0, None, 0, buf.ctypes.data, len(buf), off.ctypes.data) == 0
    assert [buf[off[k]: off[k + 1]].tobytes().decode() for k in range(nrep)] == seqs


# ---- two ranks with the library's communicator
def _rank_pass(device, read0, nreads, native):
    sys.path.insert(0, ROOT)
    from minorseq_b200 import Juliet, synth_device
    from minorseq_b200.synth import make_tables
    t = make_tables(C3)
    j = Juliet(C3.L, [(1, C3.L + 1)], refseq=t.refseq, device=device, mode_phasing=True)
    if native:
        assert j.hd.attach_comm()
    d = synth_device(j.hd, t, read0, nreads)
    j.pileup_device(d.data_ptr(), nreads)
    j.allreduce_counts()
    haps, _ = j.phase_device(j.call(), d.data_ptr(), nreads)
    seqs = j.haplotype_consensus(d.data_ptr(), nreads)
    return dict(seqs=seqs, counts=j.group_counts(), nreported=haps.nreported)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device(f"cuda:{rank}"))
    try:
        per = C3_READS // world
        q.put((rank, _rank_pass(rank, rank * per, per, True)))
    finally:
        dist.barrier()
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_gpus_equal_one():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=500) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    one = _rank_pass(0, 0, C3_READS, False)
    for r in range(world):
        assert out[r]["nreported"] == one["nreported"]
        np.testing.assert_array_equal(out[r]["counts"], one["counts"])
        assert out[r]["seqs"] == one["seqs"]
