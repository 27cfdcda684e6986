"""K6 read alignment on the GPU, bit for bit against the U16 restatement (tests/align_oracle.c): strand, position, score,
CIGAR and the set of unmapped reads."""
import ctypes as C

import numpy as np
import pytest

from align_oracle import AlignOracle, revcomp

pytestmark = pytest.mark.gpu

BASES = np.frombuffer(b"ACGT", dtype=np.uint8)


def rand_ref(rng, n):
    return BASES[rng.integers(0, 4, n)].tobytes().decode()


def simulate(rng, ref, n, min_len, max_len, sub=0.01, dele=0.01, ins=0.01, n_runs=0.3):
    """Reads from random windows of ref (truncated at both ends) with substitutions, insertions, runs of N and deletions
    (of any base, so in homopolymers too); half of them reverse-complemented."""
    r = np.frombuffer(ref.encode(), dtype=np.uint8)
    reads = []
    for _ in range(n):
        ln = int(rng.integers(min_len, max_len + 1))
        s = int(rng.integers(0, max(1, len(r) - ln + 1)))
        x = r[s:s + ln].copy()
        u = rng.random(len(x))
        x[u < sub] = BASES[rng.integers(0, 4, int((u < sub).sum()))]
        pieces = np.split(x, np.nonzero((u >= sub) & (u < sub + ins))[0] + 1)
        y = np.concatenate([np.concatenate([p, BASES[rng.integers(0, 4, 1)]]) for p in pieces[:-1]] + [pieces[-1]])
        if len(y) > 40 and rng.random() < n_runs:
            a = int(rng.integers(0, len(y) - 20))
            y[a:a + int(rng.integers(1, 12))] = ord("N")
        y = y[rng.random(len(y)) >= dele]
        seq = y.tobytes().decode()
        reads.append(revcomp(seq) if rng.random() < 0.5 else seq)
    return reads


def gpu_vs_oracle(aligner, ao, ref, reads, min_seeds=10):
    aligner.set_reference(ref)
    ao.set_reference(ref)
    got = aligner.align(reads)
    want = ao.align(reads, min_seeds)
    bad = [(k, g, w) for k, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, f"{len(bad)} of {len(reads)} differ, first: {bad[:3]}"
    return got


@pytest.fixture(scope="module")
def aligner():
    from minorseq_b200 import Aligner
    return Aligner(device=0)


@pytest.fixture(scope="module")
def ao():
    return AlignOracle()


def test_20k_synthetic_reads(aligner, ao):
    rng = np.random.default_rng(20)
    ref = rand_ref(rng, 1024)
    reads = simulate(rng, ref, 20000, 60, 1100)
    got = gpu_vs_oracle(aligner, ao, ref, reads)
    mapped = sum(g[0] for g in got)
    assert mapped > 19000 and sum(g[1] for g in got) > 9000


@pytest.mark.parametrize("L", [32, 1024, 9719, 65535])
def test_reference_lengths(aligner, ao, L):
    rng = np.random.default_rng(L)
    ref = rand_ref(rng, L)
    n = 300 if L <= 9719 else 40
    reads = simulate(rng, ref, n, min(L, 20), min(L + 40, 3000))
    reads += [ref, revcomp(ref)]
    got = gpu_vs_oracle(aligner, ao, ref, reads)
    if L >= 1024:
        assert got[-2] == (True, 0, 0, 2 * L, f"{L}=") and got[-1] == (True, 1, 0, 2 * L, f"{L}=")


def test_reference_too_long_is_refused(aligner):
    from minorseq_b200._lib import MsError
    with pytest.raises(MsError):
        aligner.set_reference("A" * 65536)


def test_batch_sizes_and_read_lengths(aligner, ao):
    rng = np.random.default_rng(5)
    ref = rand_ref(rng, 9719)
    aligner.set_reference(ref)
    assert aligner.align([]) == []
    gpu_vs_oracle(aligner, ao, ref, [ref[4000:7000]])
    reads = [ref[100:115], ref[200:216], revcomp(ref[300:316]), ref[1000:4000], revcomp(ref[2000:5000])]
    reads += [rand_ref(rng, 5000) + ref + rand_ref(rng, 5281)]     # 20 000 bases: overhangs on both sides
    reads += [revcomp(ref + ref[:281])]                            # 10 000 bases
    got = gpu_vs_oracle(aligner, ao, ref, reads)
    assert got[3] == (True, 0, 1000, 6000, "3000=") and got[4] == (True, 1, 2000, 6000, "3000=")
    assert got[5][:3] == (True, 0, 0) and got[5][4].startswith("5000S") and got[5][4].endswith("5281S")


def test_longest_read_resizes_the_slabs(aligner, ao):
    rng = np.random.default_rng(9)
    ref = rand_ref(rng, 3000)
    gpu_vs_oracle(aligner, ao, ref, simulate(rng, ref, 500, 100, 400))
    long_reads = [rand_ref(rng, 9000) + r + rand_ref(rng, 8000) for r in simulate(rng, ref, 3, 2900, 3000)]
    gpu_vs_oracle(aligner, ao, ref, simulate(rng, ref, 500, 100, 400) + long_reads)
    gpu_vs_oracle(aligner, ao, ref, simulate(rng, ref, 200, 100, 400))


def test_min_seeds_option(ao):
    from minorseq_b200 import Aligner
    rng = np.random.default_rng(13)
    ref = rand_ref(rng, 2000)
    reads = [ref[600:600 + 15 + 4 * n] for n in range(0, 14)] + simulate(rng, ref, 200, 20, 90, sub=0.05)
    for m in (1, 9, 10, 11):
        a = Aligner(device=0, min_seeds=m)
        gpu_vs_oracle(a, ao, ref, reads, min_seeds=m)


def test_cigar_capacity_retry(aligner, ao):
    from minorseq_b200 import _lib
    rng = np.random.default_rng(17)
    ref = rand_ref(rng, 2000)
    reads = simulate(rng, ref, 300, 200, 1500, sub=0.03)
    want = gpu_vs_oracle(aligner, ao, ref, reads)
    lib = aligner.lib
    seq = "".join(reads).encode()
    off = np.zeros(len(reads) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(r) for r in reads])
    out = (_lib.ReadAlignment * len(reads))()
    n = C.c_int64()
    small = np.zeros(5, dtype=np.uint32)
    rc = lib.ms_align_reads(aligner.hd.h, C.byref(aligner.params), seq, off.ctypes.data_as(C.c_void_p), len(reads), out,
                            small.ctypes.data_as(C.c_void_p), 5, C.byref(n))
    assert rc == -4 and n.value > 5
    assert [(bool(o.mapped), o.strand, o.pos, o.score) for o in out] == [w[:4] for w in want]
    cig = np.zeros(n.value, dtype=np.uint32)
    assert lib.ms_align_reads(aligner.hd.h, C.byref(aligner.params), seq, off.ctypes.data_as(C.c_void_p), len(reads), out,
                              cig.ctypes.data_as(C.c_void_p), n.value, C.byref(n)) == 0
    from align_oracle import cigar_string
    assert [cigar_string(cig[o.cigar_off:o.cigar_off + o.ncigar]) for o in out] == [w[4] for w in want]


def test_20k_generator_reads(aligner, ao, tmp_path):
    """The synthetic generator's reads (its deletions, homopolymer deletions, insertions, N and truncation) through
    bam_util.states_to_record with the alignment stripped, every other read reverse-complemented."""
    import bam_util
    from minorseq_b200.synth import SynthConfig, make_tables, synth_states
    t = make_tables(SynthConfig(L=1024, seed=71, trunc=0.2, n_rate=5e-3, dele=6e-3, ins=3e-3))
    st = synth_states(t, 0, 20000)
    recs = [bam_util.states_to_record(f"r{r}", st[r], t.strain_base[0]) for r in range(st.shape[0])]
    bam_util.write_bam(str(tmp_path / "g.bam"), "ref", 1024, [x for x in recs if x is not None])
    reads = [r["seq"] if k % 2 else revcomp(r["seq"]) for k, r in enumerate(bam_util.read_bam(str(tmp_path / "g.bam"))[2])]
    got = gpu_vs_oracle(aligner, ao, t.refseq, reads)
    assert len(reads) > 19000 and sum(g[0] for g in got) > 0.9 * len(reads)
