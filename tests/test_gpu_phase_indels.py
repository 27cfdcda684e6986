"""GPU: in-frame indel keys in phasing (ms_phase_begin_indels / Juliet.phase_device(..., indels=...), csrc/phase_indel.cu,
U20) against the numpy restatement (phase_indel_oracle.py): the bit matrix, the damage flags and counters, the haplotypes
(patterns, order, counts, hap_id), the linkage counts and pairs and the abundance rows, at L = 3000, 9719 and 12500, R not a
multiple of 8, ragged spans, genes in three frames, deletion starts at columns 30 and 31 of a block, an insertion boundary at
column 31, and key lists within one word and across a word.  Also: no indel keys is ms_phase_begin bit for bit, bits [0, V)
are today's for reads undamaged under both rules, the pile-up and the calls are unchanged, and a known answer at 6000x."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

import phase_indel_oracle as po
from test_gpu_indels import events, inject
from minorseq_b200 import Juliet, device_rows, pack_states
from minorseq_b200.api import _as_tensor
from minorseq_b200.synth import SynthConfig, make_tables, synth_states

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def device_matrix(j, R, K):
    """(bits [R, nw] uint32, flags [R] uint8) of the last ms_phase_dev"""
    b, f, n = C.c_void_p(), C.c_void_p(), C.c_int64()
    assert j.lib.ms_phase_device(j.hd.h, C.byref(b), C.byref(f), C.byref(n)) == 0 and n.value == R
    assert j.lib.ms_synchronize(j.hd.h) == 0
    nw = max(1, (K + 31) // 32)
    bits = _as_tensor(b.value, (R * nw,), torch.int32, j.hd.device).cpu().numpy().view(np.uint32).reshape(R, nw)
    flags = _as_tensor(f.value, (R,), torch.uint8, j.hd.device).cpu().numpy()
    return bits.copy(), flags.copy()


def key_record(res, del_cols, sids):
    """an Indels-like record whose calls are the given deletion columns and insertion string ids"""
    return SimpleNamespace(kind=[0] * len(del_cols) + [1] * len(sids), col=list(del_cols) + [int(res.string_col[s]) for s in sids],
                           sid=[-1] * len(del_cols) + list(sids), string_col=res.string_col, strings=res.strings)


def check_all(j, oracle, st, evs, keys, hap, lk=True):
    R = st.shape[0]
    sub = [k for k in keys if not isinstance(k[0], str)]
    dels = [k[1] for k in keys if k[0] == "del"]
    ins = [(k[1], k[2]) for k in keys if k[0] == "ins"]
    B, M, flags = po.bits(st, sub, dels, ins, events(evs))
    bits, f = device_matrix(j, R, len(keys))
    assert np.array_equal(bits, po.words(B))
    assert np.array_equal(f, flags)
    want = po.phase(B, flags, j.min_hap_reads)
    assert hap.counters == want["counters"]
    assert hap.nreported == want["nreported"] and hap.ndistinct == len(want["counts"])
    k = len(hap.counts)
    assert np.array_equal(hap.counts, want["counts"][:k]) and np.array_equal(hap.patterns, want["patterns"][:k])
    assert np.array_equal(hap.hap_id, want["hap_id"])
    if lk:
        got = j.linkage()
        w = po.linkage(B, M, po.key_columns(sub, dels, ins), oracle.fisher)
        for name in "nabc":
            assert np.array_equal(getattr(got, name), w[name]), name
        assert list(zip(got.v.tolist(), got.w.tolist(), got.both.tolist(), got.relation.tolist())) == [(p[0], p[1], p[2], p[9]) for p in w["pairs"]]
        assert got.ntested == w["ntested"]
        for i, p in enumerate(w["pairs"]):
            assert abs(got.pvalue[i] - p[8]) <= 1e-9 * p[8] + 1e-300
        ab = j.haplotype_abundance()
        wa = po.abundance(B, M, want["patterns"][: want["nreported"]])
        assert np.array_equal(ab.unique_reads, wa["unique_reads"]) and np.array_equal(ab.compatible_reads, wa["compatible_reads"])
        assert ab.counters == wa["counters"] and ab.iterations == wa["iterations"]
        assert np.allclose(ab.em_frequency, wa["em_frequency"], rtol=1e-9, atol=1e-12)
    return B, M, flags


# (L, R, deletion starts, insertion boundaries); gene 0 is in frame 0: starts 30 and 126 sit at column 30 of a block, 63 and
# 159 at column 31; the boundaries 95 and 191 at column 31
SHAPES = [(3000, 4003, (30, 201), (95, 302)), (9719, 3001, (63, 126), (191,)), (12500, 2005, (159, 30), (95,))]


@pytest.mark.parametrize("wide", [False, True], ids=["one_word", "two_words"])
@pytest.mark.parametrize("L,R,dels,ins", SHAPES)
def test_phase_indels_match_oracle(oracle, L, R, dels, ins, wide):
    cfg = SynthConfig(L=L, seed=9500 + L, trunc=0.3, n_rate=2e-2)
    t = make_tables(cfg)
    st = synth_states(t, 0, R)
    evs = []
    for i, s in enumerate(dels):
        st, e = inject(st, L + i, del_codon=s, ins_col=ins[i % len(ins)], del_every=17 + i, ins_every=13 + i)
        evs += e
    evs.sort(key=lambda e: e[0])
    genes = [(1, L + 1), (3, L // 2), (L // 3 + 2, L - 10)]
    d = device_rows(pack_states(st))
    j = Juliet(L, genes, refseq=t.refseq, device=0, mode_phasing=True)
    j.pileup_device(d.data_ptr(), R)
    called = j.call()
    col0, codon0 = j.get_counts()
    res = j.indels(d.data_ptr(), R, insertions=events(evs))
    sids = [s for s in range(len(res.strings)) if res.string_col[s] in ins and res.strings[s] == "TCTTCT"]
    assert len(sids) == len(ins)
    variants = called
    if wide:      # every call, and enough noise strings to pass a word
        sids = sorted(set(sids) | set(range(min(len(res.strings), 40))))
    else:
        variants = called[:6]
    rec = key_record(res, sorted(dels), sids)
    # today's phasing of the same reads, for bits [0, V)
    j.phase_device(variants, d.data_ptr(), R)
    V = j._V
    bits0, flags0 = device_matrix(j, R, V)
    hap, keys = j.phase_device(variants, d.data_ptr(), R, linkage=True, abundance=True, indels=rec)
    assert len(keys) == V + len(dels) + len(sids) and (len(keys) > 32) == wide
    B, M, flags = check_all(j, oracle, st, evs, keys, hap)
    both = (flags0 == 0) & (flags == 0)
    assert both.any() and np.array_equal(po.words(B[:, :V])[both], bits0[both])
    # the pile-up, the codon calls and the indel calls are unchanged
    col1, codon1 = j.get_counts()
    assert np.array_equal(col0, col1) and np.array_equal(codon0, codon1)
    assert [(v.col, v.codon, v.count, v.pvalue) for v in j.call()] == [(v.col, v.codon, v.count, v.pvalue) for v in called]
    res2 = j.indels(d.data_ptr(), R, insertions=events(evs))
    assert res2.label == res.label and np.array_equal(res2.count, res.count) and np.array_equal(res2.pvalue, res.pvalue)


def test_no_indel_keys_is_phase_begin(oracle):
    L, R = 3000, 4001
    t = make_tables(SynthConfig(L=L, seed=9601, trunc=0.3, n_rate=2e-2))
    st, evs = inject(synth_states(t, 0, R), 3, del_codon=300, ins_col=602)
    d = device_rows(pack_states(st))
    j = Juliet(L, [(1, L + 1)], device=0, mode_phasing=True)
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    res = j.indels(d.data_ptr(), R, insertions=events(evs))
    hap0, keys0 = j.phase_device(variants, d.data_ptr(), R)
    bits0, flags0 = device_matrix(j, R, len(keys0))
    hap1, keys1 = j.phase_device(variants, d.data_ptr(), R, indels=key_record(res, [], []))
    bits1, flags1 = device_matrix(j, R, len(keys1))
    assert keys0 == keys1 and np.array_equal(bits0, bits1) and np.array_equal(flags0, flags1)
    assert hap0.counters == hap1.counters and np.array_equal(hap0.hap_id, hap1.hap_id) and np.array_equal(hap0.patterns, hap1.patterns)
    ob, of = oracle.phase_bits(st, [k[0] for k in keys0], [k[1] for k in keys0])
    assert np.array_equal(bits0, ob) and np.array_equal(flags0, of)


def test_refusals():
    L, R = 600, 800
    t = make_tables(SynthConfig(L=L, seed=9602))
    st = synth_states(t, 0, R)
    d = device_rows(pack_states(st))
    j = Juliet(L, [(1, L + 1)], device=0, mode_phasing=True)
    j.pileup_device(d.data_ptr(), R)
    one = np.array([30], dtype=np.int32)
    h = j.hd.h
    assert j.lib.ms_phase_begin_indels(h, None, None, 0, one.ctypes.data, 1, None, 0, R) != 0     # no ms_indel_count_dev yet
    j.indels(d.data_ptr(), R)
    for bad in ([L - 2], [-1], [30, 30]):
        a = np.array(bad, dtype=np.int32)
        assert j.lib.ms_phase_begin_indels(h, None, None, 0, a.ctypes.data, len(a), None, 0, R) != 0
    sid = np.array([0], dtype=np.int32)
    assert j.lib.ms_phase_begin_indels(h, None, None, 0, None, 0, sid.ctypes.data, 1, R) != 0     # no such string id
    assert j.lib.ms_phase_begin_indels(h, None, None, 0, one.ctypes.data, 1, None, 0, R) == 0
    assert j.lib.ms_phase_dev(h, C.c_void_p(d.data_ptr()), R - 8) != 0                            # other reads than counted
    assert j.lib.ms_phase_begin_indels(h, None, None, 0, one.ctypes.data, 1, None, 0, R) == 0
    assert j.lib.ms_phase_dev(h, C.c_void_p(d.data_ptr()), R) == 0


def test_known_answer_at_6000x(oracle):
    L, R = 1200, 6000
    t = make_tables(SynthConfig(L=L, seed=9701, trunc=0.0, n_rate=2e-2))
    st = synth_states(t, 0, R)
    genes = [(1, L + 1)]
    d = device_rows(pack_states(st))
    j = Juliet(L, genes, refseq=t.refseq, device=0, mode_phasing=True)
    j.pileup_device(d.data_ptr(), R)
    variants = j.call()
    hap, keys = j.phase_device(variants, d.data_ptr(), R)
    assert hap.nreported >= 2
    Bp = hap.patterns[1]
    carried = {keys[v][0] for v in range(len(keys)) if (Bp[v >> 5] >> (v & 31)) & 1}
    # a called codon where B carries no variant: B's reads lose it; and an insertion at a boundary away from the variants
    s = next(k[0] for k in keys if k[0] not in carried and 60 <= k[0] <= L - 60)
    c = next(b for b in range(302, L - 60, 3) if all(abs(b - k[0]) >= 6 for k in keys))
    breads = np.flatnonzero(hap.hap_id == 1)
    st2 = st.copy()
    st2[breads, s: s + 3] = 4
    evs = [(int(r), c, "AGTAGC") for r in breads]
    for r in breads:
        st2[r, c] |= 8
    d2 = device_rows(pack_states(st2))
    j = Juliet(L, genes, refseq=t.refseq, device=0, mode_phasing=True)
    j.pileup_device(d2.data_ptr(), R)
    variants2 = j.call()
    base, keys0 = j.phase_device(variants2, d2.data_ptr(), R)
    _, flags0 = device_matrix(j, R, len(keys0))
    assert (flags0[breads] & po.GAP).all()                    # without the indel keys every read of B is a gap
    res = j.indels(d2.data_ptr(), R, insertions=events(evs))
    got = {(int(k), int(cc), x) for k, cc, x in zip(res.kind, res.col, res.inserted)}
    assert (0, s, "") in got and (1, c, "AGTAGC") in got
    hap2, keys2 = j.phase_device(variants2, d2.data_ptr(), R, linkage=True, abundance=True, indels=res)
    B, M, flags = check_all(j, oracle, st2, evs, keys2, hap2)
    kd, ki = keys2.index(("del", s)), keys2.index(("ins", c, "AGTAGC"))
    want = [int(b) for b in breads if flags[b] == 0]
    assert len(want) > 0.8 * len(breads)
    rows = [h for h in range(hap2.nreported) if (hap2.patterns[h][kd >> 5] >> (kd & 31)) & 1 and (hap2.patterns[h][ki >> 5] >> (ki & 31)) & 1]
    assert len(rows) == 1 and hap2.counts[rows[0]] == len(want)
    # the deletion-carrying reads are no longer gaps
    assert not (flags[want] & po.GAP).any() and base.counters["gaps"] > hap2.counters["gaps"]
    lk = j.linkage()
    sub_carried = [v for v in range(len(keys0)) if (hap2.patterns[rows[0]][v >> 5] >> (v & 31)) & 1]
    linked = {(int(v), int(w)) for v, w, rel in zip(lk.v, lk.w, lk.relation) if rel == 1}
    assert sub_carried and any((v, ki) in linked for v in sub_carried)
