"""Haplotype abundance on the GPU (ms_haplotype_abundance / Juliet.haplotype_abundance) against the numpy restatement in
haplotype_abundance_oracle.py: integers exactly, pi to 1e-9, the log-likelihood to 1e-9 relative, iterations within one;
the mask-width edges, the refused inputs, invariants against phasing, and the generator's known answer."""
import collections
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import haplotype_abundance_oracle as ha  # noqa: E402
from minorseq_b200 import Handle, Juliet, _lib, device_rows, host_rows, synth_device  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables, pack_states, read_strains, synth_states  # noqa: E402

_V = collections.namedtuple("_V", "col codon")


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def _check(ab, want, R=None):
    assert ab.counters == want["counters"]
    assert ab.reads_used == want["reads_used"]
    assert ab.unique_reads.tolist() == want["unique_reads"].tolist()
    assert ab.compatible_reads.tolist() == want["compatible_reads"].tolist()
    assert np.abs(ab.em_frequency - want["em_frequency"]).max(initial=0.0) <= 1e-9
    assert abs(ab.log_likelihood - want["log_likelihood"]) <= 1e-9 * abs(want["log_likelihood"]) + 1e-300
    assert abs(ab.iterations - want["iterations"]) <= 1 and ab.converged == want["converged"]
    if R is not None:
        assert sum(ab.counters.values()) == R
    if len(ab.em_frequency) and ab.reads_used:
        assert abs(ab.em_frequency.sum() - 1.0) <= 1e-12


def _same(a, b):
    for k in ("unique_reads", "compatible_reads", "em_frequency"):
        assert np.array_equal(getattr(a, k), getattr(b, k)), k
    assert (a.counters, a.iterations, a.converged, a.log_likelihood) == (b.counters, b.iterations, b.converged, b.log_likelihood)


def _phased(hd, oracle, t, R, keys=None, from_states=False):
    """reads [0, R) of the generator phased with abundance on -> (juliet, haplotypes, keys, device reads, states)"""
    if from_states:
        st = synth_states(t, 0, R)
        d = device_rows(pack_states(st))
    else:
        d = synth_device(hd, t, 0, R)
        st = oracle.unpack(host_rows(d, R, t.cfg.L), t.cfg.L, nthreads=8)
    j = Juliet(t.cfg.L, [(1, t.cfg.L + 1)], handle=hd)
    if keys is None:
        j.pileup_device(d.data_ptr(), R)
        variants = j.call()
    else:
        variants = [_V(c, k) for c, k in keys]
    hap, keys = j.phase_device(variants, d.data_ptr(), R, abundance=True)
    return j, hap, keys, d, st


def test_abundance_parity_c1(hd, oracle):
    t = make_tables(SynthConfig(L=3000, seed=20240001))
    j, hap, keys, _, st = _phased(hd, oracle, t, 5000, from_states=True)
    assert hap.nreported >= 2
    ab = j.haplotype_abundance()
    want = ha.abundance(st, keys, hap.patterns[:hap.nreported])
    _check(ab, want, 5000)
    assert (ab.unique_reads >= hap.counts[:hap.nreported]).all()
    assert want["reads_used"] > hap.counters["reported"]                    # the point: damaged reads are used


@pytest.fixture(scope="module")
def c3(hd, oracle):
    """C3 shape (200k reads x 3 kb, the 10 / 5 / 1 % minor mixture)"""
    t = make_tables(SynthConfig(L=3000, seed=20240003))
    R = 200_000
    j, hap, keys, d, st = _phased(hd, oracle, t, R)
    ab = j.haplotype_abundance()
    return dict(t=t, R=R, j=j, hap=hap, keys=keys, d=d, st=st, ab=ab, want=ha.abundance(st, keys, hap.patterns[:hap.nreported]))


def test_abundance_parity_c3(c3):
    _check(c3["ab"], c3["want"], c3["R"])
    assert c3["ab"].counters["ambiguous"] > 0 and c3["ab"].counters["incompatible"] > 0


def test_abundance_invariants_c3(c3, hd):
    """unique >= phasing count; two calls are bit-identical; a too-small buffer is refused and the retry gives the same;
    phasing and linkage results are unchanged with abundance on"""
    j, hap, ab = c3["j"], c3["hap"], c3["ab"]
    assert (ab.unique_reads >= hap.counts[:hap.nreported]).all()
    _same(ab, j.haplotype_abundance())
    H = hap.nreported
    pat = np.ascontiguousarray(hap.patterns[:H])
    prm = _lib.AbundanceParams(1e-10, 10000)
    rows = (_lib.AbundanceRow * H)()
    it, conv, ll = C.c_int32(), C.c_int32(), C.c_double()
    rc = j.lib.ms_haplotype_abundance(hd.h, C.byref(prm), pat.ctypes.data_as(C.c_void_p), H, rows, H - 1, None, C.byref(it),
                                      C.byref(conv), C.byref(ll))
    assert rc == -4                                                          # MS_ERR_CAPACITY
    _same(ab, j.haplotype_abundance())
    # phasing (and linkage) with abundance on and off
    out = []
    for on in (False, True):
        _lib.check(j.lib.ms_set_linkage(hd.h, 1), hd.h)
        _lib.check(j.lib.ms_set_abundance(hd.h, 1 if on else 0), hd.h)
        R = c3["R"]
        _lib.check(j.lib.ms_phase_begin(hd.h, np.array([k[0] for k in c3["keys"]], dtype=np.int32).ctypes.data_as(C.c_void_p),
                                        np.array([k[1] for k in c3["keys"]], dtype=np.int32).ctypes.data_as(C.c_void_p),
                                        len(c3["keys"]), R), hd.h)
        _lib.check(j.lib.ms_phase_dev(hd.h, C.c_void_p(c3["d"].data_ptr()), R), hd.h)
        h2 = j._haplotypes_device(len(c3["keys"]), max(1, (len(c3["keys"]) + 31) // 32), R, True)
        lk = j.linkage()
        out.append((h2, lk))
    (h0, l0), (h1, l1) = out
    assert np.array_equal(h0.patterns, h1.patterns) and np.array_equal(h0.counts, h1.counts) and np.array_equal(h0.hap_id, h1.hap_id)
    assert h0.counters == h1.counters
    assert np.array_equal(h0.patterns, hap.patterns) and np.array_equal(h0.counts, hap.counts)
    for k in ("v", "w", "both", "pvalue", "n", "a"):
        assert np.array_equal(getattr(l0, k), getattr(l1, k)), k


def test_abundance_known_answer_c3(c3):
    """The generator's strains as the patterns: a strain's reads fit their own strain except for the share substitution
    noise explains, and each strain's frequency is within 5 sigma of its share of the EM's reads."""
    t, keys, st, R = c3["t"], c3["keys"], c3["st"], c3["R"]
    index = {k: i for i, k in enumerate(keys)}
    V, nw = len(keys), max(1, (len(keys) + 31) // 32)
    S = t.nstrains
    pat = np.zeros((S, nw), dtype=np.uint32)
    carried = np.zeros(S, dtype=np.int64)
    for s, c, k in t.truth:
        v = index[(c, k)]
        pat[s, v >> 5] |= np.uint32(1 << (v & 31))
        carried[s] += 1
    j = c3["j"]
    ab = j.haplotype_abundance(pat)
    want = ha.abundance(st, keys, pat)
    _check(ab, want, R)
    strain, _, _ = read_strains(t, 0, R)
    Sr = want["S"]
    sub = t.cfg.sub
    for s in range(S):
        mine = strain == s
        miss = 1.0 - Sr[mine, s].mean()
        p = 3 * carried[s] * sub + V * sub / 3      # a carried codon hit by a substitution; an uncarried one turned into the alt
        assert miss <= p + 5 * np.sqrt(max(p, 1e-6) * (1 - p) / mine.sum()), (s, miss, p)
    used = want["used"]
    N = used.sum()
    for s in range(S):
        share = (strain[used] == s).mean()
        sigma = np.sqrt(share * (1 - share) / N)
        assert abs(ab.em_frequency[s] - share) <= 5 * sigma + 1e-9, (s, ab.em_frequency[s], share)


def test_abundance_v2048_c5_mixture(hd, oracle):
    """V = 2048 keys (64 words per read row) over 40k reads of the C5 mixture with 'N' noise, its 64 strains as the patterns.
    Almost every read has an 'N' in some key's codon, so phasing reports nothing; abundance still uses the reads."""
    t = make_tables(SynthConfig(L=6144, seed=20240005, dense_sites=2048, dense_strains=64, n_rate=2e-3, dele=2e-5, trunc=0.02))
    keys = sorted({(c, k) for (_, c, k) in t.truth})
    assert len(keys) == 2048
    j, hap, keys, _, st = _phased(hd, oracle, t, 40_000, keys=keys)
    index = {k: i for i, k in enumerate(keys)}
    pat = np.zeros((t.nstrains, 64), dtype=np.uint32)
    for s, c, k in t.truth:
        v = index[(c, k)]
        pat[s, v >> 5] |= np.uint32(1 << (v & 31))
    ab = j.haplotype_abundance(pat)
    want = ha.abundance(st, keys, pat)
    _check(ab, want, 40_000)
    assert want["reads_used"] > max(5_000, hap.counters["reported"])


@pytest.fixture(scope="module")
def dense(hd, oracle):
    """reads for V = 1, 32, 33 keys (one, one full and two words of the read rows); the handle holds one phased read set at a
    time, so a test phases the one it uses again (_dense)"""
    out = {}
    for V in (1, 32, 33):
        t = make_tables(SynthConfig(L=600, seed=900 + V, dense_sites=V, dense_strains=8, n_rate=2e-2, trunc=0.05))
        keys = sorted({(c, k) for (_, c, k) in t.truth})
        j, hap, keys, d, st = _phased(hd, oracle, t, 12_000, keys=keys)
        out[V] = dict(j=j, hap=hap, keys=keys, st=st, d=d)
    return out


def _dense(dense, V):
    c = dense[V]
    c["j"].phase_device([_V(a, b) for a, b in c["keys"]], c["d"].data_ptr(), 12_000, abundance=True)
    return c


def _random_patterns(rng, H, V, first=None):
    nw = max(1, (V + 31) // 32)
    seen, rows = set(), []
    for p in (first if first is not None else []):
        if len(rows) < H and p.tobytes() not in seen:
            seen.add(p.tobytes())
            rows.append(p.copy())
    while len(rows) < H:
        p = rng.integers(0, 2 ** 32, size=nw, dtype=np.uint64).astype(np.uint32)
        if V % 32:
            p[-1] &= np.uint32((1 << (V % 32)) - 1)
        if p.tobytes() not in seen:
            seen.add(p.tobytes())
            rows.append(p)
    return np.array(rows, dtype=np.uint32).reshape(H, nw)


@pytest.mark.parametrize("V,H", [(1, 1), (1, 2)] + [(V, H) for V in (32, 33) for H in (1, 2, 31, 32, 33, 64, 65, 700)])
def test_abundance_direct_patterns(dense, V, H):
    c = _dense(dense, V)
    rng = np.random.default_rng(V * 10007 + H)
    pat = _random_patterns(rng, H, V, first=c["hap"].patterns[:c["hap"].nreported])
    rng.shuffle(pat)
    ab = c["j"].haplotype_abundance(pat)
    _check(ab, ha.abundance(c["st"], c["keys"], pat), 12_000)


def test_abundance_pattern_bits_beyond_v_ignored(dense):
    c = _dense(dense, 33)
    pat = _random_patterns(np.random.default_rng(5), 40, 33)
    high = pat.copy()
    high[:, 1] |= np.uint32(0xF0000000)
    _same(c["j"].haplotype_abundance(pat), c["j"].haplotype_abundance(high))


def test_abundance_edges_and_refusals(dense, hd):
    c = _dense(dense, 32)
    j = c["j"]
    ab = j.haplotype_abundance(np.zeros((0, 1), dtype=np.uint32))            # H = 0: every read incompatible, no EM
    assert ab.counters == dict(unique=0, ambiguous=0, uninformative=0, incompatible=12_000)
    assert ab.iterations == 0 and ab.converged and len(ab.em_frequency) == 0
    one = j.haplotype_abundance(c["hap"].patterns[:1], max_iter=1)            # H = 1: no ambiguity, one step
    _check(one, ha.abundance(c["st"], c["keys"], c["hap"].patterns[:1], max_iter=1), 12_000)
    pat = _random_patterns(np.random.default_rng(1), 8, 32)
    with pytest.raises(_lib.MsError, match="duplicate"):
        j.haplotype_abundance(np.vstack([pat, pat[3:4]]))
    with pytest.raises(_lib.MsError, match="4096"):
        j.haplotype_abundance(_random_patterns(np.random.default_rng(2), 4097, 32))
    big = j.haplotype_abundance(_random_patterns(np.random.default_rng(2), 4096, 32))
    assert sum(big.counters.values()) == 12_000
    # read set phased without the clean-codon matrix
    t = make_tables(SynthConfig(L=600, seed=932, dense_sites=32, dense_strains=8))
    d = synth_device(hd, t, 0, 1000)
    j2 = Juliet(600, [(1, 601)], handle=hd)
    j2.phase_device([_V(a, b) for a, b in c["keys"]], d.data_ptr(), 1000, abundance=False)
    with pytest.raises(_lib.MsError, match="ms_set_abundance"):
        j2.haplotype_abundance()


def test_abundance_no_reads(hd):
    """N = 0 (no phased reads): pi stays 1/H, no iteration"""
    j = Juliet(600, [(1, 601)], handle=hd)
    d = device_rows(np.zeros((0, j.row_words), dtype=np.uint32))
    j.phase_device([_V(3, 5), _V(9, 17)], d.data_ptr(), 0, abundance=True)
    ab = j.haplotype_abundance(np.array([[1], [2], [3]], dtype=np.uint32))
    assert ab.em_frequency.tolist() == [1 / 3] * 3 and ab.iterations == 0 and ab.converged and ab.reads_used == 0
    assert ab.log_likelihood == 0.0


def test_abundance_two_phase_calls_equal_one(dense, hd):
    """reads phased in two ms_phase_dev calls give the same classes and EM as one call"""
    c = _dense(dense, 33)
    j, keys, st = c["j"], c["keys"], c["st"]
    pat = np.ascontiguousarray(c["hap"].patterns[:c["hap"].nreported])
    one = j.haplotype_abundance(pat)
    vc = np.array([k[0] for k in keys], dtype=np.int32)
    vk = np.array([k[1] for k in keys], dtype=np.int32)
    R, R1 = st.shape[0], 4_999
    d1, d2 = device_rows(pack_states(st[:R1])), device_rows(pack_states(st[R1:]))
    _lib.check(j.lib.ms_set_abundance(hd.h, 1), hd.h)
    _lib.check(j.lib.ms_phase_begin(hd.h, vc.ctypes.data_as(C.c_void_p), vk.ctypes.data_as(C.c_void_p), len(keys), R), hd.h)
    _lib.check(j.lib.ms_phase_dev(hd.h, C.c_void_p(d1.data_ptr()), R1), hd.h)
    _lib.check(j.lib.ms_phase_dev(hd.h, C.c_void_p(d2.data_ptr()), R - R1), hd.h)
    _same(one, j.haplotype_abundance(pat))
