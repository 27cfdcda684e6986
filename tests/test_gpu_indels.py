"""GPU: in-frame indels (Juliet.indels, csrc/indel.cu, U19) against the numpy restatement (indel_oracle.py): the counters and
string tallies bit-exact, the calls with p-values within 1e-9, on generator reads with codon deletions and insertions
injected into a minor set of reads, at L = 3000, 9719 and 12500 (column segments of the walk), R not a multiple of 8,
ragged spans and genes in three frames.  Also: n_del - k_del is K2's coverage, calling twice equals calling once, the
pile-up, the codon calls and phasing are unchanged, and the known answers at 6000x."""
import numpy as np
import pytest

import indel_oracle as io
from minorseq_b200 import Juliet, device_rows, pack_states
from minorseq_b200.synth import SynthConfig, make_tables, synth_states

pytestmark = pytest.mark.gpu


def inject(st, seed, del_codon, ins_col, del_every=100, ins_every=50, ins_str="TCTTCT"):
    """codon deletions at del_codon in every del_every-th read, ins_str after ins_col in every ins_every-th read, plus noise
    events: other lengths, letters, columns inside codons, lower case and repeated events on one column"""
    rng = np.random.default_rng(seed)
    st = st.copy()
    R, L = st.shape
    evs = []
    for r in range(0, R, del_every):
        if (st[r, del_codon: del_codon + 3] & 7 != 7).all():
            st[r, del_codon: del_codon + 3] = 4
    for r in range(1, R, ins_every):
        evs.append((r, ins_col, ins_str))
        st[r, ins_col] |= 8
    for _ in range(R // 4):
        r, c = int(rng.integers(R)), int(rng.integers(L - 1))
        n = int(rng.integers(1, 8))
        x = "".join(rng.choice(list("ACGTacgtN"), size=n))
        evs.append((r, c, x))
        if rng.random() < 0.2:
            evs.append((r, c, "GGG"))                  # a second event at the same column: never counted
        st[r, c] |= 8
    evs.sort(key=lambda e: e[0])                       # ms_expand_cigar order: by read, then column
    return st, evs


def events(evs):
    pool, off = b"", []
    for _, _, x in evs:
        off.append(len(pool))
        pool += x.encode()
    return (np.array([e[0] for e in evs], dtype=np.int64), np.array([e[1] for e in evs], dtype=np.int32), np.array(off, dtype=np.int64),
            np.array([len(e[2]) for e in evs], dtype=np.int32), pool)


def check_against_oracle(j, res, st, evs, genes, refseq=None, **kw):
    ev = events(evs)
    start = io.start_bits(st.shape[1], genes, kw.get("region"))
    cnt, strings, tally = io.counts(st, ev, start)
    assert np.array_equal(res.cnt.astype(np.int64), cnt)
    assert list(zip(res.string_col.tolist(), res.strings)) == strings
    assert np.array_equal(res.tally.astype(np.int64), tally)
    want = io.call(st, cnt, strings, tally, genes, refseq=refseq, **kw)
    got = [(int(res.gene[i]), int(res.codon_index[i]), int(res.col[i]), int(res.kind[i]), res.inserted[i], int(res.count[i]), int(res.coverage[i]),
            int(res.expected[i]), int(res.ntests[i]), int(res.ref_codon[i]), int(res.next_codon[i])) for i in range(len(res.count))]
    assert got == [(w["gene"], w["codon_index"], w["col"], w["kind"], w["inserted"], w["count"], w["coverage"], w["expected"], w["ntests"],
                    w["ref_codon"], w["next_codon"]) for w in want]
    for i, w in enumerate(want):
        assert abs(res.pvalue[i] - w["pvalue"]) <= 1e-9 * w["pvalue"]
        assert res.label[i] == io.label(w["kind"], w["ref_codon"], w["next_codon"], w["codon_index"] + 1, w["inserted"])
    return want


@pytest.mark.parametrize("L,R", [(3000, 4003), (9719, 3001), (12500, 2005)])
def test_indels_match_oracle(L, R):
    cfg = SynthConfig(L=L, seed=9100 + L, trunc=0.3, n_rate=2e-2)
    t = make_tables(cfg)
    st = synth_states(t, 0, R)
    st, evs = inject(st, L, del_codon=201, ins_col=302, del_every=25, ins_every=25)   # gene 0 in frame 0: codon 67 at 201, boundary 302
    genes = [(1, L + 1), (3, L // 2), (L // 3 + 2, L - 10)]    # frames 0, 2, and (L//3 + 1) % 3
    d = device_rows(pack_states(st))
    j = Juliet(L, genes, refseq=t.refseq, device=0, mode_phasing=True)
    res0 = j.run_device(d.data_ptr(), R, want_hap_id=True)
    col0, codon0 = j.get_counts()
    res = j.indels(d.data_ptr(), R, insertions=events(evs))
    want = check_against_oracle(j, res, st, evs, genes, refseq=t.refseq)
    assert any(w["kind"] == 0 and w["col"] == 201 for w in want) and any(w["kind"] == 1 and w["inserted"] == "TCTTCT" for w in want)
    # n_del - k_del = K2's coverage of the codon
    for i in range(len(res.count)):
        if res.kind[i] == 0:
            assert res.coverage[i] - res.count[i] == codon0[res.col[i]].sum()
    # calling twice equals calling once; the pile-up, the codon calls and the haplotypes are unchanged
    res2 = j.indels(d.data_ptr(), R, insertions=events(evs))
    assert np.array_equal(res2.cnt, res.cnt) and np.array_equal(res2.tally, res.tally) and res2.label == res.label
    assert np.array_equal(res2.pvalue, res.pvalue)
    col1, codon1 = j.get_counts()
    assert np.array_equal(col0, col1) and np.array_equal(codon0, codon1)
    res1 = j.run_device(d.data_ptr(), R, want_hap_id=True)
    assert [(v.col, v.codon, v.count, v.pvalue) for v in res1.variants] == [(v.col, v.codon, v.count, v.pvalue) for v in res0.variants]
    assert np.array_equal(res1.haplotypes.counts, res0.haplotypes.counts) and np.array_equal(res1.haplotypes.hap_id, res0.haplotypes.hap_id)


def test_region_filters_and_majority_reference():
    L, R = 3000, 2600
    t = make_tables(SynthConfig(L=L, seed=9301, n_rate=2e-2))
    st, evs = inject(synth_states(t, 0, R), 5, del_codon=600, ins_col=902, del_every=40, ins_every=30)
    genes = [(1, L + 1)]
    d = device_rows(pack_states(st))
    for kw in (dict(region=(550, 1200)), dict(min_perc=2.8), dict(max_perc=2.8)):
        j = Juliet(L, genes, device=0, region=kw.get("region"), min_perc=kw.get("min_perc"), max_perc=kw.get("max_perc"))
        j.run_device(d.data_ptr(), R)
        res = j.indels(d.data_ptr(), R, insertions=events(evs))
        check_against_oracle(j, res, st, evs, genes, **kw)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_known_answers_at_6000x(seed):
    L, R = 1200, 6000
    t = make_tables(SynthConfig(L=L, seed=9400 + seed, trunc=0.0, n_rate=2e-2, minor_fracs=(0.05,)))
    clean = synth_states(t, 0, R)
    genes = [(1, L + 1)]
    d = device_rows(pack_states(clean))
    j = Juliet(L, genes, refseq=t.refseq, device=0)
    j.run_device(d.data_ptr(), R)
    assert len(j.indels(d.data_ptr(), R).count) == 0                   # no indel call on clean reads
    st, evs = inject(clean, seed, del_codon=300, ins_col=602, del_every=100, ins_every=50)
    d = device_rows(pack_states(st))
    j.run_device(d.data_ptr(), R)
    res = j.indels(d.data_ptr(), R, insertions=events(evs))
    got = {(int(k), int(c), x) for k, c, x in zip(res.kind, res.col, res.inserted)}
    assert (0, 300, "") in got and (1, 602, "TCTTCT") in got
    check_against_oracle(j, res, st, evs, genes, refseq=t.refseq)
