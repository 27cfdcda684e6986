"""Sub-threshold variant linkage on the GPU (ms_rare_candidates, ms_rare_linkage, ms_rare_support, Juliet.rare_linkage) against
the restatement in rare_linkage_oracle.py: candidates, tables, groups and support exactly, p-values to 1e-9 relative.  Edges
on crafted histograms and reads, the 0.25 % strain at 6000 reads, the cap of 2048 candidates, key counts on both sides of the
tcgen05 size rule, and no candidate-candidate linked pair in clean samples or in C3's 1 / 5 / 10 % mixture."""
import ctypes as C

import mpmath as mp
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import hypergeom_reference as ref  # noqa: E402
import linkage_oracle as lo  # noqa: E402
import rare_linkage_oracle as ro  # noqa: E402
from minorseq_b200 import Handle, Juliet, _lib, device_rows, host_rows, synth_device  # noqa: E402
from minorseq_b200._lib import LinkagePair, LinkageParams  # noqa: E402
from minorseq_b200.api import _ptr  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables, pack_states  # noqa: E402

PVAL_RTOL = 1e-9
AAA, CAA, GAA = 0, 16, 32
N = 1000


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


def _hist(L, cols):
    h = np.zeros((L, 64), dtype=np.uint32)
    for s, bins in cols.items():
        for c, k in bins.items():
            h[s, c] = k
    return h


def _gpu_candidates(hd, codon, L, genes, alpha=0.01, min_reads=5, candidate_alpha=0.1):
    j = Juliet(L, genes, handle=hd, alpha=alpha)
    j.counts_tensor()[L * 8:] = torch.from_numpy(codon.reshape(-1).view(np.int32)).cuda()
    torch.cuda.synchronize()
    return j.rare_candidates(min_reads=min_reads, candidate_alpha=candidate_alpha, cap=16)


def _check_p(got, want, what):
    """to PVAL_RTOL where the exact tail is a normal double; a tail below 1e-300 may underflow (dense tables reach 1e-513)"""
    if want > mp.mpf("1e-300"):
        assert ref.rel_err(got, want) <= PVAL_RTOL, (got, what)
    else:
        assert got < 1e-290, (got, what)


def _check_candidates(got, want):
    got_c, got_d = got
    want_c, want_d = want
    assert got_d == want_d
    assert [(c.col, c.codon) for c in got_c] == [(w["col"], w["codon"]) for w in want_c]
    for g, w in zip(got_c, want_c):
        for f in ("gene", "codon_index", "ref_codon", "count", "coverage", "expected", "ntests"):
            assert getattr(g, f) == w[f], (f, w)
        _check_p(g.pvalue, w["pvalue"], w)


@pytest.mark.parametrize("case", ["min_reads", "bound_above", "bound_below", "called_elsewhere", "two_genes", "none", "single",
                                  "cap_small"])
def test_candidate_edges(hd, case):
    p8 = float(ref.k2_pvalue(8, N, 1))
    L, genes, kw = 9, [(1, 10)], {}
    h = _hist(9, {0: {AAA: N - 8, CAA: 8}})
    if case == "min_reads":
        kw = dict(min_reads=9)
    elif case == "bound_above":
        kw = dict(candidate_alpha=p8 * (1 + 1e-9))
    elif case == "bound_below":
        kw = dict(candidate_alpha=p8 * (1 - 1e-9))
    elif case == "called_elsewhere":
        h, genes, kw = _hist(9, {3: {AAA: N - 8, CAA: 8}}), [(1, 10), (4, 7)], dict(alpha=0.05)
    elif case == "two_genes":
        h, genes = _hist(9, {3: {AAA: N - 8, CAA: 8}}), [(1, 10), (4, 10)]
    elif case == "none":
        h = _hist(9, {0: {AAA: N}, 3: {AAA: N}})
    elif case == "cap_small":
        L, genes = 15, [(1, 16)]
        h = _hist(15, {s: {AAA: N - k, CAA: k} for s, k in ((0, 5), (3, 9), (6, 6), (9, 8), (12, 7))})
    got = _gpu_candidates(hd, h, L, genes, **kw)
    want = ro.candidates(h, L, genes, **kw)
    _check_candidates(got, want)
    if case in ("bound_above", "single", "two_genes"):
        assert len(got[0]) == 1
    if case in ("min_reads", "bound_below", "called_elsewhere", "none"):
        assert got[0] == []


def test_candidate_cap_drops_the_largest_p(hd):
    """2400 candidates (20 codons at each of 120 positions, counts 12..15): 2048 kept by p, then (column, codon)"""
    L = 360
    ks = [12, 13, 14, 15]
    cols = {}
    for s in range(0, L, 3):
        bins = {AAA: 0}
        for i, c in enumerate(range(1, 64, 3)[:20]):
            bins[c] = ks[(s // 3 + i) % 4]
        bins[AAA] = 20 * N - sum(bins.values())
        cols[s] = bins
    h = _hist(L, cols)
    got = _gpu_candidates(hd, h, L, [(1, L + 1)], alpha=1e-12)
    want = ro.candidates(h, L, [(1, L + 1)], alpha=1e-12)
    assert want[1] == 2400 - 2048 and len(want[0]) == 2048
    _check_candidates(got, want)


# ------------------------------------------------------------------------------------------------------------ pair statistics
def _phase(hd, L, states, keys, fc, variant=0):
    """phase `keys` (called first, candidates from fc) with the clean-codon matrix -> (pairs record array, m_r)"""
    lib = hd.lib
    rows = pack_states(states)
    d = device_rows(rows)
    Juliet(L, [(1, L + 1)], handle=hd)
    vc = np.array([k[0] for k in keys], dtype=np.int32)
    vd = np.array([k[1] for k in keys], dtype=np.int32)
    _lib.check(lib.ms_set_cooccurrence_variant(hd.h, variant), hd.h)
    try:
        _lib.check(lib.ms_set_linkage(hd.h, 1), hd.h)
        _lib.check(lib.ms_phase_begin(hd.h, _ptr(vc), _ptr(vd), len(keys), rows.shape[0]), hd.h)
        _lib.check(lib.ms_phase_dev(hd.h, C.c_void_p(d.data_ptr()), rows.shape[0]), hd.h)
        p = LinkageParams(0.01, 10)
        n, m = C.c_int64(), C.c_int64()
        _lib.check(lib.ms_rare_linkage(hd.h, fc, C.byref(p), None, 0, C.byref(n), C.byref(m)), hd.h)
        out = (LinkagePair * max(1, n.value))()
        _lib.check(lib.ms_rare_linkage(hd.h, fc, C.byref(p), out, n.value, C.byref(n), C.byref(m)), hd.h)
    finally:
        _lib.check(lib.ms_set_cooccurrence_variant(hd.h, 0), hd.h)
    return np.ctypeslib.as_array(out)[: n.value].copy(), int(m.value), d


def _check_pairs(got, m, want, want_m, p_rows=None):
    assert m == want_m
    assert [tuple(int(x) for x in (r["v"], r["w"], r["both"], r["v_only"], r["w_only"], r["neither"])) for r in got] == \
        [p[:6] for p in want]
    assert all(int(r["relation"]) == lo.LINKED for r in got)
    for r, p in list(zip(got, want))[:p_rows]:
        assert abs(r["d_prime"] - p[6]) <= 1e-12 and abs(r["r2"] - p[7]) <= 1e-12, p
        _check_p(float(r["pvalue"]), p[8], p)


def _pair_states(tables, spacing):
    """each table (a, b, c, d) gets keys CAA at 6i and AAG at 6i + spacing[i] over an all-A reference; reads clean at those only"""
    G = len(tables)
    L = 6 * G + 3
    proto, counts = [], []
    for i, ((a, b, c, d), sp) in enumerate(zip(tables, spacing)):
        v, w = 6 * i, 6 * i + sp
        for cv, cw, k in ((1, 1, a), (1, 0, b), (0, 1, c), (0, 0, d)):
            st = np.full(L, 7, dtype=np.uint8)
            st[v:v + 3] = 0
            st[w:w + 3] = 0
            if cv:
                st[v] = 1
            if cw:
                st[w + 2] = 2
            proto.append(st)
            counts.append(k)
    states = np.repeat(np.array(proto), counts, axis=0)
    keys = [(6 * i, CAA) for i in range(G)] + [(6 * i + sp, 2) for i, sp in enumerate(spacing)]
    return L, states, keys


@pytest.mark.parametrize("fc", [0, 6, 12])
def test_pair_edges(hd, fc):
    """spacing 2 vs 3, n = 9 vs 10, empty and full margins, strong and weak tables; fc = 12: no candidate, nothing tested"""
    tables = [(5, 0, 0, 5), (5, 0, 0, 5), (5, 0, 0, 4), (12, 2, 2, 5484), (1, 3, 3, 100), (0, 0, 10, 10)]
    spacing = [3, 2, 3, 3, 3, 3]
    L, states, keys = _pair_states(tables, spacing)
    got, m, _ = _phase(hd, L, states, keys, fc)
    B, M = lo.carry_and_clean(states, keys)
    want, want_m = ro.pairs(B, M, [k[0] for k in keys], fc)
    _check_pairs(got, m, want, want_m)
    if fc == 0:
        assert any(p[:6] == (3, 9, 12, 2, 2, 5484) for p in want)


def test_support_against_numpy(hd, oracle):
    """overlapping key sets across words, a set over every key, bits past V ignored; counts equal the restated B / M"""
    t = make_tables(SynthConfig(L=960, seed=57, dense_sites=40, dense_strains=8, n_rate=2e-2, trunc=0.05))
    sites = sorted({(c, k) for (_, c, k) in t.truth})
    R = 20_000
    st = oracle.unpack(host_rows(synth_device(hd, t, 0, R), R, 960), 960, nthreads=8)
    _phase(hd, 960, st, sites, 0)
    V = len(sites)
    nw = (V + 31) // 32
    rng = np.random.default_rng(1)
    sets = [[0, 1], [2, 33], list(range(V)), [V - 1], rng.choice(V, 5, replace=False).tolist()]
    masks = np.zeros((len(sets), nw), dtype=np.uint32)
    for g, s in enumerate(sets):
        for k in s:
            masks[g, k >> 5] |= np.uint32(1 << (k & 31))
    masks[3, nw - 1] |= np.uint32(1 << 31) if V % 32 else 0
    car, inf = np.zeros(len(sets), np.uint64), np.zeros(len(sets), np.uint64)
    _lib.check(hd.lib.ms_rare_support(hd.h, _ptr(masks), len(sets), _ptr(car), _ptr(inf)), hd.h)
    B, M = lo.carry_and_clean(st, sites)
    want_c, want_i = ro.support(B, M, sets)
    assert car.tolist() == want_c and inf.tolist() == want_i


# ----------------------------------------------------------------------------------------------------------- whole feature
def _run(hd, oracle, cfg, R, called_from_gpu=True):
    t = make_tables(cfg)
    L = cfg.L
    d = synth_device(hd, t, 0, R)
    j = Juliet(L, [(1, L + 1)], handle=hd)
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    res = j.rare_linkage(d.data_ptr(), R, variants=variants)
    return t, d, j, variants, res


def test_detection_quarter_percent(hd, oracle):
    """the known answer of test_oracle_rare_linkage on the GPU, everything against the restatement"""
    cfg = SynthConfig(L=3000, seed=3, minor_fracs=(0.0025,), variants_per_minor=(4, 4))
    R = 6000
    t, d, j, variants, res = _run(hd, oracle, cfg, R)
    st = oracle.unpack(host_rows(d, R, 3000), 3000, nthreads=8)
    _, codon = j.get_counts()
    want = ro.rare_linkage(st, codon, 3000, [(1, 3001)], [(v.col, v.codon) for v in variants])
    _check_candidates((res.candidates, res.dropped), (want["candidates"], want["dropped"]))
    assert res.keys == want["keys"] and res.first_candidate == want["first_candidate"]
    _check_pairs(res.pairs, res.tested, want["pairs"], want["tested"])
    assert res.groups == want["groups"]
    assert res.carriers.tolist() == want["carriers"] and res.informative.tolist() == want["informative"]
    truth = sorted((c, k) for (_, c, k) in t.truth)
    assert [[res.keys[i] for i in g] for g in res.groups] == [truth]


@pytest.mark.parametrize("variant", [1, 2])
def test_tcgen05_size_rule(hd, oracle, variant):
    """>= 256 keys and >= 32768 reads (the tcgen05 Gram) and the popcount-AND kernel give the same pairs as the restatement"""
    L, R = 1536, 40_000
    t = make_tables(SynthConfig(L=L, seed=20240006, dense_sites=300, dense_strains=16, n_rate=2e-3, dele=1e-3, trunc=0.02))
    d = synth_device(hd, t, 0, R)
    st = oracle.unpack(host_rows(d, R, L), L, nthreads=8)
    sites = sorted({(c, k) for (_, c, k) in t.truth})
    assert len(sites) >= 256
    fc = 250
    got, m, _ = _phase(hd, L, st, sites, fc, variant=variant)
    B, M = lo.carry_and_clean(st, sites)
    want, want_m = _dense_pairs(B, M, [k[0] for k in sites], fc)
    _check_pairs(got, m, want, want_m, p_rows=50)


def _dense_pairs(B, M, cols, fc):
    """ro.pairs with the mpmath tail only for the first 50 linked pairs (the dense layout links tens of thousands)"""
    import scipy.stats as ss
    Bf, Mf = B.astype(np.float64), M.astype(np.float64)
    n = np.rint(Mf.T @ Mf).astype(np.int64)
    a = np.rint(Bf.T @ Bf).astype(np.int64)
    bm = np.rint(Bf.T @ Mf).astype(np.int64)
    V = B.shape[1]
    tested = [(v, w) for w in range(fc, V) for v in range(w) if abs(cols[v] - cols[w]) >= 3 and n[v, w] >= 10]
    m = len(tested)
    out = []
    for v, w in sorted(tested):
        A, Nn = int(a[v, w]), int(n[v, w])
        Bq, Cq = int(bm[v, w]) - A, int(bm[w, v]) - A
        D = Nn - A - Bq - Cq
        ps = float(ss.hypergeom.sf(A - 1, Nn, A + Cq, A + Bq))
        if ps * m > 4 * 0.01:
            continue
        if ps * m > 0.25 * 0.01 or len(out) < 50:
            p = ref.fisher_greater(A, Bq, Cq, D)
            if not p * m < 0.01:
                continue
        else:
            p = ps
        dp, r2 = ref.linkage_measures(A, Bq, Cq, Nn)
        out.append((v, w, A, Bq, Cq, D, float(dp), float(r2), p))
    return out, m


# ---------------------------------------------------------------------------------------------------------------- specificity
@pytest.mark.parametrize("R", [6000, 200_000])
@pytest.mark.parametrize("seed", [11, 12, 13, 14, 15])
def test_clean_samples_have_no_linked_candidates(hd, oracle, R, seed):
    _, _, _, _, res = _run(hd, oracle, SynthConfig(L=3000, seed=seed, minor_fracs=()), R)
    cc = [(int(v), int(w)) for v, w in zip(res.pairs["v"], res.pairs["w"]) if v >= res.first_candidate]
    assert cc == [] and res.groups == [], (len(res.candidates), res.tested)


def test_c3_mixture_has_no_linked_candidates(hd, oracle):
    _, _, _, variants, res = _run(hd, oracle, SynthConfig(L=3000, seed=20240003), 200_000)
    assert len(variants) > 0
    cc = [(int(v), int(w)) for v, w in zip(res.pairs["v"], res.pairs["w"]) if v >= res.first_candidate]
    assert cc == [] and res.groups == [], (len(res.candidates), res.tested)
