"""Pairwise variant linkage on the GPU (ms_linkage / Juliet.linkage) against the column-state restatement in
linkage_oracle.py: the significant-pair list exactly (indices, the four counts, relation), D' and r^2 to 1e-12, p-values to
1e-9 relative; the stacked Gram matrix under both contraction kernels; invariants against K2 and phasing; the generator's
known answer."""
import collections
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import linkage_oracle as lo  # noqa: E402
from minorseq_b200 import Handle, Juliet, _lib, device_rows, host_rows, synth_device  # noqa: E402
from minorseq_b200._lib import LinkageParams  # noqa: E402
from minorseq_b200.api import _as_tensor  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables, pack_states, synth_states  # noqa: E402

PVAL_RTOL = 1e-9
_V = collections.namedtuple("_V", "col codon")


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def _called(hd, L, d, R):
    j = Juliet(L, [(1, L + 1)], handle=hd)
    j.pileup_device(d.data_ptr(), R)
    return j, j.call()


def _states(hd, oracle, t, R):
    d = synth_device(hd, t, 0, R)
    return d, oracle.unpack(host_rows(d, R, t.cfg.L), t.cfg.L, nthreads=8)


def _check_pairs(lk, want):
    got = list(zip(lk.v.tolist(), lk.w.tolist(), lk.both.tolist(), lk.v_only.tolist(), lk.w_only.tolist(), lk.neither.tolist(),
                   lk.relation.tolist()))
    assert got == [(p[0], p[1], p[2], p[3], p[4], p[5], p[9]) for p in want["pairs"]]
    assert lk.ntested == want["ntested"]
    for k, p in enumerate(want["pairs"]):
        assert abs(lk.d_prime[k] - p[6]) <= 1e-12 and abs(lk.r2[k] - p[7]) <= 1e-12, p
        assert abs(lk.pvalue[k] - p[8]) <= PVAL_RTOL * p[8] + 1e-300, p
    for name in "nabc":
        assert np.array_equal(getattr(lk, name), want[name]), name


@pytest.fixture(scope="module")
def c3(hd, oracle):
    """C3 shape (200k reads x 3 kb, the default 10 / 5 / 1 % minor mixture) with the oracle's answer"""
    t = make_tables(SynthConfig(L=3000, seed=20240003))
    R = 200_000
    d, st = _states(hd, oracle, t, R)
    j, variants = _called(hd, 3000, d, R)
    hap, keys = j.phase_device(variants, d.data_ptr(), R, want_hap_id=False, linkage=True)
    lk = j.linkage()
    return dict(t=t, st=st, keys=keys, hap=hap, lk=lk, j=j, want=lo.linkage(st, keys, oracle.fisher))


def test_linkage_parity_c1(oracle, hd):
    t = make_tables(SynthConfig(L=3000, seed=20240001))
    st = synth_states(t, 0, 5000)
    d = device_rows(pack_states(st))
    j, variants = _called(hd, 3000, d, st.shape[0])
    hap, keys = j.phase_device(variants, d.data_ptr(), st.shape[0], linkage=True)
    assert len(keys) >= 8
    lk = j.linkage()
    want = lo.linkage(st, keys, oracle.fisher)
    assert len(want["pairs"]) > 0
    _check_pairs(lk, want)
    # motivation: with 2 % 'N' every tested pair has more informative reads than phasing has undamaged ones
    undamaged = hap.counters["reported"] + hap.counters["insufficient"]
    cols = np.array([k[0] for k in keys])
    tested = (np.abs(cols[:, None] - cols[None, :]) >= lo.MIN_SPACING) & (lk.n >= lo.MIN_READS)
    tested &= np.triu(np.ones_like(tested), 1).astype(bool)
    assert tested.sum() == lk.ntested > 0
    assert lk.n[tested].min() > undamaged


def test_linkage_parity_c3(c3):
    assert len(c3["want"]["pairs"]) > 0
    _check_pairs(c3["lk"], c3["want"])


def test_linkage_known_answer_c3(c3):
    """Planted variants of the same minor strain are linked (D' > 0.9); variants of different minor strains are exclusive."""
    lk, keys = c3["lk"], c3["keys"]
    index = {k: i for i, k in enumerate(keys)}
    strain = {index[(c, k)]: s for (s, c, k) in c3["t"].truth if (c, k) in index}
    assert len(strain) == len(c3["t"].truth)          # every planted variant is called at 200k reads
    rel = {(int(v), int(w)): (int(r), float(dp)) for v, w, r, dp in zip(lk.v, lk.w, lk.relation, lk.d_prime)}
    cols = np.array([k[0] for k in keys])
    same = cross = 0
    for v in strain:
        for w in strain:
            if v >= w or abs(cols[v] - cols[w]) < lo.MIN_SPACING or lk.n[v, w] < lo.MIN_READS:
                continue
            if strain[v] == strain[w]:
                assert rel[(v, w)][0] == lo.LINKED and rel[(v, w)][1] > 0.9, (v, w)
                same += 1
            else:
                assert rel[(v, w)][0] == lo.EXCLUSIVE, (v, w)
                cross += 1
    assert same > 0 and cross > 0


def test_linkage_invariants_c3(c3, hd):
    """diag(M^T M) = K2 coverage and diag(B^T B) = K2 count of every key; a capacity retry gives the same counts."""
    j, lk = c3["j"], c3["lk"]
    col, codon = j.get_counts()
    for i, (c, k) in enumerate(c3["keys"]):
        assert lk.n[i, i] == codon[c].sum() and lk.a[i, i] == codon[c, k]
    p = LinkageParams(0.01, 10)
    n, m = C.c_int64(), C.c_int64()
    _lib.check(j.lib.ms_linkage(hd.h, C.byref(p), None, 0, C.byref(n), C.byref(m)), hd.h)   # cap 0: sizes only
    assert (n.value, m.value) == (len(lk.v), lk.ntested)
    again = j.linkage(cap=1)                                                                   # grows once more
    for name in ("v", "w", "both", "v_only", "w_only", "neither", "relation", "d_prime", "r2", "pvalue", "n", "a", "b", "c"):
        assert np.array_equal(getattr(again, name), getattr(lk, name)), name


def _device_bits(j, hd, nw):
    b, f, r = C.c_void_p(), C.c_void_p(), C.c_int64()
    _lib.check(j.lib.ms_phase_device(hd.h, C.byref(b), C.byref(f), C.byref(r)), hd.h)
    _lib.check(j.lib.ms_synchronize(hd.h), hd.h)
    bits = _as_tensor(b.value, (r.value * nw,), torch.int32, hd.device).cpu().numpy().view(np.uint32).copy()
    flags = _as_tensor(f.value, (r.value,), torch.uint8, hd.device).cpu().numpy().copy()
    return bits, flags


@pytest.mark.parametrize("V", [20, 40])
def test_linkage_leaves_phasing_unchanged(hd, V):
    """With linkage on, bits, flags, haplotypes, hap_id and the co-occurrence matrix are those of a run without it
    (one-word and two-word bit-vectors)."""
    t = make_tables(SynthConfig(L=960, seed=57, dense_sites=V, dense_strains=8, n_rate=2e-2, trunc=0.05))
    R = 20_000
    d = synth_device(hd, t, 0, R)
    sites = sorted({(c, k) for (_, c, k) in t.truth})
    j = Juliet(960, [(1, 961)], handle=hd)
    out = []
    for on in (False, True):
        hap, keys = j.phase_device([_V(c, k) for c, k in sites], d.data_ptr(), R, want_hap_id=True, linkage=on)
        bits, flags = _device_bits(j, hd, (len(keys) + 31) // 32)
        out.append((bits, flags, hap, j.cooccurrence().cpu().numpy()))
    (b0, f0, h0, c0), (b1, f1, h1, c1) = out
    assert np.array_equal(b0, b1) and np.array_equal(f0, f1) and np.array_equal(c0, c1)
    assert np.array_equal(h0.patterns, h1.patterns) and np.array_equal(h0.counts, h1.counts) and np.array_equal(h0.hap_id, h1.hap_id)
    assert h0.counters == h1.counters
    # and linkage on a read set phased without it is refused rather than answered from stale bits
    j.phase_device([_V(c, k) for c, k in sites], d.data_ptr(), R, linkage=False)
    with pytest.raises(_lib.MsError):
        j.linkage()


def test_linkage_gram_kernels_agree_dense(oracle, hd):
    """V >= 256 and >= 32768 reads: the stacked Gram matrix is bit-identical under the popcount-AND and the tcgen05
    contraction and equals the oracle's n, a, b, c; the pair list (hundreds of rows, multi-chunk rows) matches too."""
    L, R = 1536, 40_000
    t = make_tables(SynthConfig(L=L, seed=20240006, dense_sites=300, dense_strains=16, n_rate=2e-3, dele=1e-3, trunc=0.02))
    d, st = _states(hd, oracle, t, R)
    sites = sorted({(c, k) for (_, c, k) in t.truth})
    assert len(sites) >= 256
    j = Juliet(L, [(1, L + 1)], handle=hd)
    _, keys = j.phase_device([_V(c, k) for c, k in sites], d.data_ptr(), R, want_hap_id=False, linkage=True)
    grams = {}
    for variant in (1, 2):
        _lib.check(j.lib.ms_set_cooccurrence_variant(hd.h, variant), hd.h)
        try:
            j.phase_device([_V(c, k) for c, k in sites], d.data_ptr(), R, want_hap_id=False, linkage=True)   # a fresh read set
            g, dim = C.c_void_p(), C.c_int32()
            _lib.check(j.lib.ms_linkage_device(hd.h, C.byref(g), C.byref(dim)), hd.h)
            _lib.check(j.lib.ms_synchronize(hd.h), hd.h)
            grams[variant] = _as_tensor(g.value, (dim.value, dim.value), torch.int32, hd.device).cpu().numpy().copy()
        finally:
            _lib.check(j.lib.ms_set_cooccurrence_variant(hd.h, 0), hd.h)
    assert np.array_equal(grams[1], grams[2])
    lk = j.linkage()
    want = lo.linkage(st, keys, oracle.fisher)
    assert len(want["pairs"]) > 300
    _check_pairs(lk, want)
