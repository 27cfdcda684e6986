"""In-frame indels (csrc/indel.cu, restatement choice U19) at their edges.

Counts: indel_count_kernel and indel_ins_kernel exactly against indel_oracle.counts, on states built in numpy: a deletion
window at every column phase (s % 32 = 29..31 reach into the next block), runs of 1, 2, 4 and 6 gaps and runs that end at N,
at an unspanned column or at the end of the read; the last block for L = 3 .. 65, from packed rows and from the rows
expand_events_kernel writes; the column-segment seams of the walk; R around the 2040-read work item; a column every one of
100 000 reads deletes; a shard with read0 > 0; and the insertion events' edges (c + 1 in the next block, dropped events, the
first event of a read deciding, lower case, strings longer than L).

Calls: indel_test_kernel against the mpmath reference (hypergeom_reference.py) with test_gpu_call_edges' decision rule.
K2's codon histogram at a deletion's start is written straight into the count tensor, so a few reads make tables of any n.
Covered: alpha straddling p * ntests by 1e-10, e = 0 (rate 0, a rate^129 that underflows), e = 1 (a subnormal rate^126),
e = n (rate 1), the deletion's e stepping from 1 to 2, k <= e with alpha > ntests / 2, coverage 1 and 2, k = n without a clean
codon, the strict percentage filters, n = 2^32 - 1, regions, overlapping frames, a gene past L, reference fallbacks to the
majority codon, a too-small output, and the refused parameters.  Every field of every call is compared; p-values to 1e-12
relative (both below 1e-290 when the reference is below 1e-300).

Limit: indel_test_kernel sums a deletion's n = k + coverage in uint32; tables of 2^32 reads or more are out of range and not
tested (n = 2^32 - 1 is).
"""
import ctypes as C
import json
import math
import os
import re
import subprocess

import mpmath as mp
import numpy as np
import pytest

import hypergeom_reference as ref
import indel_oracle as io
from test_gpu_call_edges import RTOL, codon_of, decide, pvalue
from test_gpu_indels import events

gpu = pytest.mark.gpu

DEFAULTS = dict(deletion_rate=3e-3, insertion_rate=3e-3, alpha=0.01, min_perc=None, max_perc=None)
FIELDS = ("gene", "codon_index", "col", "kind", "sid", "ref_codon", "next_codon", "count", "coverage", "expected", "ntests")
FRAMES3 = lambda L: [(1, L + 1), (2, L + 1), (3, L + 1)]    # every column past 1 is a codon start and a boundary


# ------------------------------------------------------------------------------------------------------------ reference
def indel_reference(codon, cnt, strings, tally, L, genes, refseq=None, region=None, deletion_rate=3e-3, insertion_rate=3e-3,
                    alpha=0.01, min_perc=None, max_perc=None):
    """The calls from the integers: codon = K2's histogram [L, 64] (the deletions' coverage and the majority codon), cnt /
    strings / tally as indel_oracle.counts returns them; e and p from hypergeom_reference, called by decide()"""
    Pdel = 1.0
    for _ in range(3):
        Pdel *= deletion_rate
    reflen = min(len(refseq), L) if refseq else 0

    def codon_at(s):
        if s + 3 <= reflen and all(ch in "ACGTacgt" for ch in refseq[s:s + 3]):
            return codon_of(refseq[s:s + 3])
        h = [int(x) for x in codon[s]]
        return max(range(64), key=lambda c: (h[c], -c)) if sum(h) else -1

    def test(k, n, P, m):
        if k == 0 or n == 0:
            return None
        e = ref.expected_count(n, P)
        if k <= e and 0.5 * m >= alpha:
            return None
        p = pvalue(k, n, e)
        if not decide(p, m, alpha):
            return None
        perc = 100.0 * k / n
        if min_perc is not None and not perc > min_perc:
            return None
        if max_perc is not None and not perc < max_perc:
            return None
        return e, p

    by_col = {}
    for i, (c, _) in enumerate(strings):
        by_col.setdefault(c, []).append(i)
    out = []
    for g, cods in enumerate(io.codon_starts(L, genes, region)):
        m = len(cods)
        starts = {s for _, s in cods}
        for ci, s in cods:
            k = int(cnt[s, 0])
            n = k + sum(int(x) for x in codon[s])
            r = test(k, n, Pdel, m)
            if r:
                out.append(dict(gene=g, codon_index=ci, col=s, kind=0, sid=-1, ref_codon=codon_at(s), next_codon=-1, count=k, coverage=n,
                                expected=r[0], ntests=m, pvalue=r[1], inserted=""))
            if s + 3 not in starts:
                continue
            for i in by_col.get(s + 2, []):
                x = strings[i][1]
                P = 1.0
                for _ in range(len(x)):
                    P *= insertion_rate
                k, n = int(tally[i]), int(cnt[s + 2, 1])
                r = test(k, n, P, m)
                if r:
                    out.append(dict(gene=g, codon_index=ci, col=s + 2, kind=1, sid=i, ref_codon=codon_at(s), next_codon=codon_at(s + 3),
                                    count=k, coverage=n, expected=r[0], ntests=m, pvalue=r[1], inserted=x))
    return out


def codon_histogram(st):
    """K2's histogram of every column from the states (the reads with a clean codon there)"""
    st = np.asarray(st) & 7
    L = st.shape[1]
    h = np.zeros((L, 64), dtype=np.int64)
    for s in range(L - 2):
        h[s] = io._codon_hist(st, s)
    return h


def sorted_events(evs):
    """(read, col, x) in ms_expand_cigar's order: by read; a read's events at one column keep their order"""
    return sorted(evs, key=lambda e: e[0])


# ---------------------------------------------------------------------------------------------------------------- GPU glue
@pytest.fixture(scope="module")
def hd():
    from minorseq_b200 import Handle
    h = Handle(0)
    yield h
    h.close()


def assert_counts(res, st, evs, genes, region=None, read0=0):
    L = st.shape[1]
    cnt, strings, tally = io.counts(st, events(evs) if evs else None, io.start_bits(L, genes, region), read0)
    bad = np.nonzero((res.cnt.astype(np.int64) != cnt).any(axis=1))[0]
    assert len(bad) == 0, ("cnt differs at columns", bad[:10].tolist(), res.cnt[bad[:5]].tolist(), cnt[bad[:5]].tolist())
    assert list(zip(res.string_col.tolist(), res.strings)) == strings
    assert np.array_equal(res.tally.astype(np.int64), tally), (res.tally.tolist(), tally.tolist())
    return cnt, strings, tally


def count_case(hd, st, genes, evs=(), read0=0, rows=None):
    """Juliet.indels on the reads st (packed with pack_states unless rows, a device tile tensor, is given)"""
    from minorseq_b200 import Juliet, device_rows, pack_states
    R, L = st.shape
    j = Juliet(L, genes, handle=hd)
    d = device_rows(pack_states(st)) if rows is None else rows
    res = j.indels(d.data_ptr(), R, insertions=events(sorted_events(evs)) if evs else None, read0=read0)
    return j, res


def write_histogram(j, hist):
    """hist: {start column: {codon: count}} replaces K2's histogram at those columns"""
    import torch
    from minorseq_b200 import _lib
    _lib.check(j.lib.ms_synchronize(j.hd.h), j.hd.h)
    t = j.counts_tensor()
    for s, bins in hist.items():
        row = np.zeros(64, dtype=np.uint32)
        for c, k in bins.items():
            row[c] = k
        lo = j.L * 8 + 64 * s
        t[lo: lo + 64] = torch.from_numpy(row.view(np.int32)).to(t.device)
    torch.cuda.synchronize()


def assert_calls(res, want, what=""):
    key = lambda w: (w["gene"], w["col"], w["kind"], w["sid"])
    got = [(int(res.gene[i]), int(res.col[i]), int(res.kind[i]), int(res.sid[i])) for i in range(len(res.count))]
    assert got == [key(w) for w in want], (what, sorted(set(got) ^ set(map(key, want)))[:10])
    for i, w in enumerate(want):
        for f in FIELDS:
            assert int(getattr(res, f)[i]) == w[f], (what, f, int(getattr(res, f)[i]), w[f], key(w))
        assert res.inserted[i] == w["inserted"], (what, key(w))
        assert res.label[i] == io.label(w["kind"], w["ref_codon"], w["next_codon"], w["codon_index"] + 1, w["inserted"]), (what, res.label[i])
        if w["pvalue"] > mp.mpf("1e-300"):
            assert ref.rel_err(res.pvalue[i], w["pvalue"]) <= RTOL, (what, key(w), res.pvalue[i], mp.nstr(w["pvalue"], 20))
        else:
            assert res.pvalue[i] < 1e-290, (what, key(w), res.pvalue[i])


def call_case(hd, st, genes, evs=(), hist=None, refseq=None, region=None, **kw):
    """pile-up of st, K2's histogram replaced at the columns of hist, Juliet.indels; counts and calls checked -> (res, want)"""
    from minorseq_b200 import Juliet, device_rows, pack_states
    R, L = st.shape
    prm = dict(DEFAULTS, **kw)
    j = Juliet(L, genes, refseq=refseq, region=region, handle=hd)
    j.reset()
    d = device_rows(pack_states(st))
    j.pileup_device(d.data_ptr(), R)
    if hist:
        write_histogram(j, hist)
    _, codon = j.get_counts()
    evs = sorted_events(evs)
    res = j.indels(d.data_ptr(), R, insertions=events(evs) if evs else None, **prm)
    cnt, strings, tally = assert_counts(res, st, evs, genes, region)
    want = indel_reference(codon, cnt, strings, tally, L, genes, refseq=refseq, region=region, **prm)
    assert_calls(res, want, kw)
    return j, res, want


# ------------------------------------------------------------------------------------------------------ hand-built reads
def small_tables_reads():
    """L = 30, one gene (10 codons), no reference: reads that span only the columns they are about"""
    L = 30
    rows, evs = [], []

    def read(lo, hi, gaps=()):
        r = np.full(L, 7, dtype=np.uint8)
        r[lo:hi] = 0
        r[list(gaps)] = 4
        rows.append(r)
        return len(rows) - 1

    read(0, 3, (0, 1, 2))                                   # codon 0: k = n = 1
    read(3, 6, (3, 4, 5))                                   # codon 3: k = 1, n = 2
    read(3, 6)
    for _ in range(30):                                     # codon 6: k = n = 30, no clean codon there: ref_codon -1
        read(6, 9, (6, 7, 8))
    evs.append((read(11, 13), 11, "TCT"))                   # boundary 11: k = n = 1
    for _ in range(2):                                      # boundary 14: k = n = 2
        evs.append((read(14, 16), 14, "TCT"))
    evs.append((read(17, 19), 17, "GCA"))                   # boundary 17: k = 1, n = 2
    read(17, 19)
    return np.stack(rows), evs, [(1, 31)]


def expected_edge_reads():
    """L = 30, one gene: deletions of 12, 1 and 30 reads; insertions of TCT, a 129-base and a 126-base string by 20 reads, GGG
    by one, among 200 clean reads"""
    L = 30
    base = np.zeros(L, dtype=np.uint8)
    rows, evs = [base.copy() for _ in range(200)], []
    for s, k in ((0, 12), (3, 1), (6, 30)):
        for _ in range(k):
            r = base.copy()
            r[s:s + 3] = 4
            rows.append(r)
    for c, x, k in ((2, "TCT", 20), (5, "TCA" * 43, 20), (8, "ACG" * 42, 20), (11, "GGG", 1)):
        for _ in range(k):
            evs.append((len(rows), c, x))
            rows.append(base.copy())
    return np.stack(rows), evs, [(1, 31)]


def insertion_event_reads():
    """L = 120, genes in frame 0 (whole) and frame 2 (columns 3-71): the insertion events' edges"""
    L = 120
    rng = np.random.default_rng(5)
    base = rng.integers(0, 4, size=L, dtype=np.uint8)
    rows, evs = [], []

    def read(*ev, **st):
        r = base.copy()
        for c, s in st.get("at", {}).items():
            r[c] = s
        if "end" in st:
            r[st["end"]:] = 7
        rows.append(r)
        for c, x in ev:
            evs.append((len(rows) - 1, c, x))
            r[c] |= 8

    for c in (31, 95):                  # c % 32 = 31: c + 1 is in the next block, c - 31 in this one
        read((c, "TCT"), at={c - 31: 4})                # counted: c and c + 1 clean, c - 31 a gap
        read((c, "TCT"), at={c + 1: 4})                 # c + 1 a gap, c - 31 clean: not counted
        read((c, "TCT"), at={c + 1: 5})                 # c + 1 N
        read((c, "TCT"), end=c + 1)                     # c + 1 unspanned
        read((c, "TCT"), at={c: 4})                     # c itself a gap
        read((c, "TCT"), at={c - 31: 5})                # counted
    read((116, "TCT"))                                  # c = L - 4: the last boundary
    read((118, "TCT"))                                  # c = L - 2: c + 1 is no codon start
    read((119, "TCT"))
    read((1, "TCT"))                                    # c - 2 < 0 (c + 1 starts a frame-2 codon)
    read((70, "TCT"))                                   # c - 2 = 68 is frame 2's last codon, c + 1 no start
    read((2, "TCT"))                                    # c = 2: the first boundary
    read((50, "TCT"), (50, "GGG"))                      # two events at one column: the first decides
    read((50, "TC"), (50, "GGG"))                       # ... and is out of frame: the read counts for no string
    read((50, "TNT"), (50, "GGG"))                      # ... or holds an N
    read((50, "GGG"))
    read((50, "tct"))                                   # lower case: the id of TCT
    read((50, "gGaTcC"))
    for x in ("", "A", "AC", "ACGT"):                   # lengths 0, 1, 2 and 4
        read((50, x))
    read((50, "ACG" * 42))                              # 126 and 129 bases, longer than L
    read((50, "TCA" * 43))
    read((53, "TCT"), (56, "TCT"))                      # two columns of one read
    for _ in range(20):
        read()
    return np.stack(rows), evs, [(1, L + 1), (3, 72)]


# -------------------------------------------------------------------------------------------------------- CPU self-check
def test_reference_matches_the_restatement():
    """The mpmath reference of this file equals indel_oracle.call (scipy tails, to 1e-9) on the hand-built reads"""
    rng = np.random.default_rng(11)
    noisy = rng.choice(np.array([0, 1, 2, 3, 0, 1, 4, 4, 5, 7], dtype=np.uint8), size=(400, 60))
    noisy_ev = [(int(r), int(c), x) for r, c, x in zip(rng.integers(0, 400, 300), rng.integers(2, 57, 300),
                                                       rng.choice(["TCT", "tct", "GGA", "AC", "TTTAAA"], 300))]
    cases = [(small_tables_reads(), [dict(), dict(deletion_rate=0.0, insertion_rate=0.0, alpha=6.0)]),
             (expected_edge_reads(), [dict(), dict(deletion_rate=0.0, insertion_rate=0.0), dict(deletion_rate=1.0, insertion_rate=1.0, alpha=11.0)]),
             (insertion_event_reads(), [dict(), dict(alpha=1.5, insertion_rate=0.2)]),
             ((noisy, noisy_ev, FRAMES3(60)), [dict(), dict(min_perc=5.0), dict(max_perc=20.0, alpha=0.5)])]
    total = 0
    for (st, evs, genes), kws in cases:
        evs = sorted_events(evs)
        L = st.shape[1]
        for region in (None, (4, L - 5)):
            cnt, strings, tally = io.counts(st, events(evs), io.start_bits(L, genes, region))
            for kw in kws:
                prm = dict(DEFAULTS, **kw)
                want = indel_reference(codon_histogram(st), cnt, strings, tally, L, genes, region=region, **prm)
                alt = dict(prm, min_perc=-1.0 if prm["min_perc"] is None else prm["min_perc"],
                           max_perc=-1.0 if prm["max_perc"] is None else prm["max_perc"])
                other = io.call(st, cnt, strings, tally, genes, region=region, **alt)
                assert len(want) == len(other), (kw, region, len(want), len(other))
                total += len(want)
                for w, o in zip(want, other):
                    assert {f: w[f] for f in FIELDS if f != "sid"} == {f: o[f] for f in FIELDS if f != "sid"}
                    assert w["inserted"] == o["inserted"]
                    assert abs(float(w["pvalue"]) - o["pvalue"]) <= 1e-9 * float(w["pvalue"])
    assert total >= 40, total


# ------------------------------------------------------------------------------------------------------------- 1. counts
@gpu
def test_deletion_windows_at_every_column_phase(hd):
    L = 128
    rng = np.random.default_rng(1)
    base = rng.integers(0, 4, size=L, dtype=np.uint8)
    rows = []

    def read(gaps=(), at=None, end=None):
        r = base.copy()
        r[list(gaps)] = 4
        for c, s in (at or {}).items():
            r[c] = s
        if end is not None:
            r[end:] = 7
        rows.append(r)

    for s in range(96):
        read(range(s, s + 3))
    for n in (1, 2, 4, 6):                                  # a run of 6 counts at s .. s+3
        for s in (0, 28, 29, 30, 31, 60, 61, 62, 63, 93, L - n):
            read(range(s, s + n))
    for s in (27, 28, 29, 30, 31, 62, 63):                  # runs that end at N, at an unspanned column, at the read's end
        read(range(s, s + 3), at={s + 3: 5})
        read(range(s, s + 2), at={s + 2: 5})
        read(range(s, s + 2), at={s + 2: 7})
        read(range(s, s + 3), end=s + 3)
        read(range(s, s + 2), end=s + 2)
        read(range(s, s + 3), at={s - 1: 7})
    st = np.vstack([np.stack(rows), rng.choice(np.array([0, 1, 2, 3, 4, 4, 4, 4, 5, 7], dtype=np.uint8), size=(300, L))])
    _, res = count_case(hd, st, [(1, L + 1)])
    assert_counts(res, st, [], [(1, L + 1)])
    assert all(res.cnt[s, 0] >= 1 for s in range(96))


def _expand(j, st, base):
    """the rows of st as expand_events_kernel writes them from their event rows against base"""
    import torch
    from minorseq_b200 import _lib, encode_states
    R, L = st.shape
    hdr, ev = encode_states(st, base)
    j.set_base(base)
    dh = torch.from_numpy(np.ascontiguousarray(hdr).view(np.uint8)).cuda()
    de = torch.from_numpy(ev if len(ev) else np.zeros(1, np.uint8)).cuda()
    out = torch.zeros(int(j.lib.ms_tiled_words(L, R)), dtype=torch.int32, device="cuda")
    _lib.check(j.lib.ms_expand_events_dev(j.hd.h, C.c_void_p(dh.data_ptr()), C.c_void_p(de.data_ptr()), R, C.c_void_p(out.data_ptr())), j.hd.h)
    _lib.check(j.lib.ms_synchronize(j.hd.h), j.hd.h)
    return out


@gpu
@pytest.mark.parametrize("L", [3, 31, 32, 33, 63, 64, 65])
def test_last_block_from_packed_and_expanded_rows(hd, L):
    """Deletions at L - 3 and clean reads through L - 1: cnt at L - 2 and L - 1 is 0 (no window fits), and the rows from
    pack_states and from expand_events_kernel (the not-spanned padding past L) give the same counts"""
    rng = np.random.default_rng(L)
    base = rng.integers(0, 4, size=L, dtype=np.uint8)
    rows = [base.copy() for _ in range(9)]
    for lo in (L - 3, L - 2, L - 1, max(0, L - 4)):
        for _ in range(5):
            r = base.copy()
            r[lo:] = 4
            rows.append(r)
    r = base.copy()
    r[L - 3:] = 4
    r[:max(0, L - 5)] = 7
    rows.append(r)
    st = np.vstack([np.stack(rows), rng.choice(np.array([0, 1, 2, 3, 4, 4, 4, 5, 7], dtype=np.uint8), size=(37, L))])
    genes = [(1, L + 1)]
    j, res = count_case(hd, st, genes)
    cnt, _, _ = assert_counts(res, st, [], genes)
    assert res.cnt[L - 3, 0] >= 6 and res.cnt[L - 1, 1] == 0 and (L < 2 or res.cnt[L - 2, 0] == 0) and res.cnt[L - 1, 0] == 0
    _, res2 = count_case(hd, st, genes, rows=_expand(j, st, base))
    assert np.array_equal(res2.cnt, res.cnt)


def seams(L):
    """the column-segment seams of ms_indel_count_dev's walk"""
    nblk = (L + 31) // 32
    nseg = -(-nblk // 256)
    seg_len = -(-nblk // nseg)
    return [32 * seg_len * i for i in range(1, nseg)]


@gpu
@pytest.mark.parametrize("L", [8193, 9719, 12500, 20000])
def test_column_segment_seams(hd, L):
    sm = seams(L)
    assert sm and {9719: [4864], 12500: [6272]}.get(L, sm) == sm
    rng = np.random.default_rng(L)
    base = rng.integers(0, 4, size=L, dtype=np.uint8)
    rows, evs = [], []
    for c0 in sm:
        for s in range(c0 - 40, c0 + 41):
            r = base.copy()
            r[s:s + 3] = 4
            rows.append(r)
        c = c0 - 1                                          # insertion boundary: c + 1 in the next segment
        for st_next, x in ((0, "TCT"), (4, "TCT"), (5, "TCT"), (7, "GGAACC"), (0, "GGAACC")):
            r = base.copy()
            r[c0] = base[c0] if st_next == 0 else st_next
            r[c0 - 32] = 4                                  # the same bit of the segment's previous block is a gap
            evs.append((len(rows), c, x))
            rows.append(r)
    st = np.stack(rows)
    genes = FRAMES3(L)
    _, res = count_case(hd, st, genes, evs)
    _, strings, tally = assert_counts(res, st, evs, genes)
    assert {(c, x): int(t) for (c, x), t in zip(strings, tally)} == {**{(c0 - 1, "TCT"): 1 for c0 in sm}, **{(c0 - 1, "GGAACC"): 1 for c0 in sm}}


@gpu
@pytest.mark.parametrize("R", [1, 7, 8, 2039, 2040, 2041, 4081])
def test_read_counts_around_work_items(hd, R):
    L = 100
    rng = np.random.default_rng(R)
    st = rng.choice(np.array([0, 1, 2, 3, 4, 4, 4, 5, 7], dtype=np.uint8), size=(R, L))
    st[: R // 2 + 1, 40:43] = 4
    evs = [(int(r), int(c), str(x)) for r, c, x in zip(rng.integers(0, R, R), rng.integers(0, L, R),
                                                       rng.choice(["TCT", "tct", "GGAACC", "AC", "TNT", "GGG"], R))]
    _, res = count_case(hd, st, FRAMES3(L), evs)
    assert_counts(res, st, evs, FRAMES3(L))
    assert res.cnt[40, 0] >= R // 2 + 1


@gpu
def test_a_column_every_read_deletes(hd):
    """k_del = R = 100 000: the column's sum crosses 49 work items and their counter flushes"""
    R, L = 100_000, 40
    rng = np.random.default_rng(7)
    st = np.tile(rng.integers(0, 4, size=L, dtype=np.uint8), (R, 1))
    st[:, 10:13] = 4
    st[::7, 20:23] = 4
    st[::11, 31] = 5
    st[::13, 33:] = 7
    _, res = count_case(hd, st, [(1, L + 1)])
    assert_counts(res, st, [], [(1, L + 1)])
    assert int(res.cnt[10, 0]) == R and int(res.cnt[8, 1]) == R


@gpu
def test_shard_counts_its_own_reads_and_events(hd):
    """reads [read0, read0 + R) of a larger run: the string ids come from all the run's events, the tallies from the shard's"""
    Rall, L, read0, R = 5000, 96, 1703, 2411
    rng = np.random.default_rng(3)
    st = rng.choice(np.array([0, 1, 2, 3, 0, 1, 2, 3, 4, 5, 7], dtype=np.uint8), size=(Rall, L))
    evs = [(int(r), int(c), str(x)) for r, c, x in zip(rng.integers(0, Rall, 4000), rng.integers(0, L, 4000),
                                                       rng.choice(["TCT", "tct", "GGAACC", "AC", "GGG"], 4000))]
    evs += [(10, 50, "AAAAAA"), (read0 - 1, 50, "CCCCCC"), (read0 + R, 50, "TTTTTT"), (read0, 50, "GGGGGG"), (read0 + R - 1, 50, "ACGACG")]
    st[[10, read0 - 1, read0 + R, read0, read0 + R - 1], 50:52] = 0
    sh = st[read0:read0 + R]
    _, res = count_case(hd, sh, FRAMES3(L), evs, read0=read0)
    _, strings, tally = assert_counts(res, sh, evs, FRAMES3(L), read0=read0)
    t = {s: int(k) for s, k in zip(strings, tally)}
    assert t[(50, "AAAAAA")] == t[(50, "CCCCCC")] == t[(50, "TTTTTT")] == 0 and t[(50, "GGGGGG")] == t[(50, "ACGACG")] == 1


@gpu
def test_insertion_event_edges(hd):
    st, evs, genes = insertion_event_reads()
    _, res = count_case(hd, st, genes, evs)
    _, strings, tally = assert_counts(res, st, evs, genes)
    t = {s: int(k) for s, k in zip(strings, tally)}
    assert t[(31, "TCT")] == t[(95, "TCT")] == 2 and t[(50, "TCT")] == 2 and t[(50, "GGG")] == 1     # c - 31 a gap or N
    assert t[(50, "ACG" * 42)] == t[(50, "TCA" * 43)] == 1 and (116, "TCT") in t and (2, "TCT") in t
    assert {c for c, _ in strings} == {2, 31, 50, 53, 56, 95, 116}     # 1, 70, 118 and 119 are no boundaries


# -------------------------------------------------------------------------------------------------------------- 2. calls
def deletion_reads(L, cols):
    """{start column: k} -> reads of base AAA..., k of them with '-' at s, s+1, s+2"""
    rows = []
    for s, k in cols.items():
        r = np.zeros(L, dtype=np.uint8)
        r[s:s + 3] = 4
        rows += [r] * k
    return np.stack(rows)


def insertion_reads(L, n, strings):
    """n clean reads; strings: {(c, x): k} -> the first reads carry the events"""
    st = np.zeros((n, L), dtype=np.uint8)
    evs, r = [], 0
    for (c, x), k in strings.items():
        for _ in range(k):
            evs.append((r, c, x))
            r += 1
    return st, evs


@gpu
@pytest.mark.parametrize("kind,k,lo,hi", [("del", 13, 1e-4, 1e-2), ("del", 45, 1e-13, 1e-11), ("del", 673, 1e-201, 1e-199),
                                          ("ins", 32, 1e-4, 1e-2), ("ins", 74, 1e-13, 1e-11), ("ins", 715, 1e-201, 1e-199)])
def test_threshold_straddle(hd, kind, k, lo, hi):
    """alpha = (1 +- 1e-10) p * ntests: called above, not below.  Deletion: n = 10^6 (K2's histogram), e = 1; insertion: n =
    10 000 reads, insertion_rate 0.1, e = 11."""
    L, genes = 30, [(1, 31)]                                  # ntests = 10
    if kind == "del":
        st, evs, hist, kw = deletion_reads(L, {9: k}), [], {9: {0: 1_000_000 - k}}, dict()
        n, P, key = 1_000_000, 3e-3 * 3e-3 * 3e-3, (0, 9)
    else:
        (st, evs), hist, kw = insertion_reads(L, 10_000, {(8, "TCT"): k}), None, dict(insertion_rate=0.1)
        n, P, key = 10_000, 0.1 * 0.1 * 0.1, (1, 8)
    e = ref.expected_count(n, P)
    p = pvalue(k, n, e)
    assert mp.mpf(lo) < p < mp.mpf(hi), mp.nstr(p, 5)
    for side, f in (("above", 1 + 1e-10), ("below", 1 - 1e-10)):
        _, res, _ = call_case(hd, st, genes, evs, hist=hist, alpha=float(p * 10 * f), **kw)
        assert (key in set(zip(res.kind.tolist(), res.col.tolist()))) == (side == "above"), (side, mp.nstr(p, 17))


@gpu
def test_expected_count_edges(hd):
    st, evs, genes = expected_edge_reads()
    P126 = math.prod([3e-3] * 126)
    P129 = math.prod([3e-3] * 129)
    assert P129 == 0.0 and 0.0 < P126 < 2.2250738585072014e-308             # rate^129 underflows, rate^126 is subnormal
    _, res, want = call_case(hd, st, genes, evs)
    got = {(w["col"], w["inserted"][:3]): w["expected"] for w in want}
    assert got.get((5, "TCA")) == 0 and got.get((8, "ACG")) == 1            # e = 0 and e = 1 from the long strings
    _, res, want = call_case(hd, st, genes, evs, deletion_rate=0.0, insertion_rate=0.0)
    assert want and all(w["expected"] == 0 for w in want) and {w["kind"] for w in want} == {0, 1}
    for alpha in (0.01, 6.0, 11.0):                                          # e = n: p = 1, called only when ntests < alpha
        _, res, want = call_case(hd, st, genes, evs, deletion_rate=1.0, insertion_rate=1.0, alpha=alpha)
        assert all(w["expected"] == w["coverage"] for w in want) and bool(want) == (alpha > 10)


@gpu
def test_deletion_expected_steps_from_one_to_two(hd):
    """e = ceil(n * 2.7e-8) changes from 1 to 2 between n0 - 1 and n0 (found in doubles, as the kernel computes it)"""
    Pd = 1.0
    for _ in range(3):
        Pd *= 3e-3
    n0 = int(1.0 / Pd)
    while math.ceil(n0 * Pd) < 2:
        n0 += 1
    while math.ceil((n0 - 1) * Pd) >= 2:
        n0 -= 1
    assert ref.expected_count(n0 - 1, Pd) == 1 and ref.expected_count(n0, Pd) == 2
    L, genes = 30, [(1, 31)]
    k = 12
    hist = {0: {0: n0 - 1 - k}, 3: {0: n0 - k}, 6: {0: n0 - k + 1}}
    _, res, want = call_case(hd, deletion_reads(L, {0: k, 3: k, 6: k}), genes, hist=hist, alpha=0.5)
    assert [(w["col"], w["coverage"], w["expected"]) for w in want] == [(0, n0 - 1, 1), (3, n0, 2), (6, n0 + 1, 2)]


@gpu
@pytest.mark.parametrize("alpha", [0.6, 1.0, 1.5])
def test_at_or_below_expected_with_large_alpha(hd, alpha):
    """k <= e is tested once alpha > ntests / 2: one-codon genes (deletions, n = 100 000, deletion_rate 0.1, e = 101) and a
    two-codon gene (insertions, n = 2000 reads, insertion_rate 0.1, e = 3); p >= 1/2 there comes from 1 - P(X <= k - 1)"""
    L = 30
    ks = {0: 1, 3: 50, 6: 101, 9: 102, 12: 130}
    genes = [(s + 1, s + 4) for s in ks] + [(16, 22)]
    ins, evs = insertion_reads(L, 2000, {(17, "AAA"): 1, (17, "CCC"): 3, (17, "GGG"): 10})
    st = np.vstack([ins, deletion_reads(L, ks)])
    hist = {s: {0: 100_000 - k} for s, k in ks.items()}
    _, res, want = call_case(hd, st, genes, [(r, c, x) for r, c, x in evs], hist=hist, deletion_rate=0.1, insertion_rate=0.1, alpha=alpha)
    assert ref.expected_count(100_000, 0.1 * 0.1 * 0.1) == 101
    called = {(w["kind"], w["col"], w["inserted"]) for w in want}
    assert (0, 6, "") in called and (0, 9, "") in called                     # k = e and k = e + 1: p ~ 1/2
    assert ((1, 17, "CCC") in called) == (alpha > 1.4)                       # k = e in a gene of 2 tests: p ~ 0.66


@gpu
def test_small_tables(hd):
    st, evs, genes = small_tables_reads()
    _, res, want = call_case(hd, st, genes, evs)
    assert [(w["col"], w["ref_codon"]) for w in want] == [(6, -1)] and res.label == ["?3del"]
    _, res, want = call_case(hd, st, genes, evs, deletion_rate=0.0, insertion_rate=0.0, alpha=6.0)     # e = 0, everything tested
    assert {(w["col"], w["count"], w["coverage"]) for w in want} == {(0, 1, 1), (3, 1, 2), (6, 30, 30), (11, 1, 1), (14, 2, 2), (17, 1, 2)}
    for kw in (dict(alpha=6.0), dict(deletion_rate=0.0, insertion_rate=0.0)):
        call_case(hd, st, genes, evs, **kw)


@gpu
def test_percentage_filters_are_strict(hd):
    """100 k / n = 2.0 exactly for a deletion (20 of 1000) and an insertion (20 of 1000)"""
    L, genes = 30, [(1, 31)]
    ins, evs = insertion_reads(L, 1000, {(5, "TCT"): 20})
    dl = deletion_reads(L, {0: 20})
    dl[:, 3:] = 7
    st = np.vstack([ins, dl])
    for mn, mx, called in ((2.0, None, False), (None, 2.0, False), (1.9999999999999998, None, True), (None, 2.0000000000000004, True),
                           (2.0, 2.0000000000000004, False), (1.9999999999999998, 2.0, False)):
        _, res, want = call_case(hd, st, genes, evs, hist={0: {0: 980}}, min_perc=mn, max_perc=mx)
        assert {(w["kind"], w["col"]) for w in want} == ({(0, 0), (1, 5)} if called else set()), (mn, mx)


@gpu
def test_deletion_coverage_at_the_uint32_limit(hd):
    """k + coverage = 2^32 - 1 (the coverage split over two bins; e = 116), and 2^32 - 2"""
    L, genes = 30, [(1, 31)]
    top = 2 ** 32 - 1
    hist = {0: {0: 2 ** 31, 21: 2 ** 31 - 1 - 300}, 3: {63: top - 40}, 6: {0: top - 1 - 300}}
    _, res, want = call_case(hd, deletion_reads(L, {0: 300, 3: 40, 6: 300}), genes, hist=hist)
    assert [(w["col"], w["coverage"], w["ref_codon"]) for w in want] == [(0, top, 0), (6, top - 1, 0)]
    assert want[0]["expected"] == 116


@gpu
def test_regions_frames_genes_past_the_end_and_references(hd):
    L = 60
    rng = np.random.default_rng(60)
    base = rng.integers(0, 4, size=L, dtype=np.uint8)
    st = np.tile(base, (400, 1))
    evs = []
    for i, s in enumerate((9, 10, 11, 30, 54)):              # deletions in frames 0, 1, 2 and in the gene past L
        st[i * 30: i * 30 + 20 + i, s:s + 3] = 4
    for i, c in enumerate((11, 12, 13, 32, 8)):              # insertions at boundaries of the three frames
        for r in range(200 + 25 * i, 200 + 25 * i + 15 + i):
            evs.append((r, c, "TCT" if i % 2 else "GGAACC"))
    genes = [(1, 61), (2, 50), (3, 40), (31, 90)]
    hist = {9: {5: 1000, 37: 1000}, 12: {5: 700, 60: 700, 9: 699}, 3: {40: 500}}     # ties: the lowest index wins
    for refseq in (None, "".join("ACGT"[b] for b in base), "AAAAAAAAANNNcccAAAaaaTTT", "ACGTACGTACGTAC", "acgt" * 15 + "TTTTTT"):
        j, res, want = call_case(hd, st, genes, evs, hist=hist, refseq=refseq)
        if refseq is None:
            assert {(w["col"], w["ref_codon"]) for w in want if w["kind"] == 0 and w["col"] == 9} == {(9, 5)}
            assert {w["next_codon"] for w in want if w["kind"] == 1 and w["col"] == 11} == {5}
        assert {w["gene"] for w in want} == {0, 1, 2, 3}
    _, _, want = call_case(hd, st, genes, evs, hist=hist, region=(1, 13))    # codons 0..9 of gene 0: the boundary 11 is cut off
    assert {(w["gene"], w["ntests"]) for w in want} <= {(0, 4), (1, 3), (2, 3)} and (1, 11) not in {(w["kind"], w["col"]) for w in want}
    # too small an output: MS_ERR_CAPACITY with the number of calls, then the same records
    from minorseq_b200 import _lib
    j, res, want = call_case(hd, st, genes, evs, hist=hist)
    assert len(want) >= 3

    def raw(cap):
        p = _lib.IndelParams()
        j.lib.ms_indel_params_default(C.byref(p))
        g = (_lib.Gene * len(genes))(*[_lib.Gene(b, e) for b, e in genes])
        out = (_lib.Indel * max(1, cap))()
        n = C.c_int64()
        rc = j.lib.ms_indel_call(j.hd.h, g, len(genes), None, C.byref(p), out, cap, C.byref(n))
        return rc, n.value, np.ctypeslib.as_array(out)[:min(cap, n.value)].copy()

    rc, n, first = raw(1)
    assert rc == -4 and n == len(want) and len(first) == 1
    rc, n, rec = raw(n)
    assert rc == 0 and n == len(want)
    for f in FIELDS + ("pvalue",):
        assert np.array_equal(rec[f], getattr(res, f)), f
    assert all(first[0][f] == rec[0][f] for f in FIELDS + ("pvalue",))


@gpu
def test_call_parameters_are_refused(hd):
    from minorseq_b200 import _lib
    st, evs, genes = expected_edge_reads()
    nan = float("nan")
    for kw, msg in ((dict(deletion_rate=-1e-3), "deletion_rate"), (dict(deletion_rate=1.0000000000000002), "deletion_rate"),
                    (dict(deletion_rate=nan), "deletion_rate"), (dict(insertion_rate=-0.5), "insertion_rate"),
                    (dict(insertion_rate=1.5), "insertion_rate"), (dict(insertion_rate=nan), "insertion_rate"),
                    (dict(alpha=0.0), "alpha"), (dict(alpha=-0.01), "alpha"), (dict(alpha=nan), "alpha")):
        with pytest.raises(_lib.MsError, match=f"ms_indel_call: {msg}"):
            call_case(hd, st, genes, evs, **kw)
    call_case(hd, st, genes, evs, deletion_rate=0.0, insertion_rate=1.0, alpha=1e-300)      # the bounds are accepted


@gpu
def test_juliet_cli_refuses_a_bad_insertion_rate(tmp_path):
    from minorseq_b200 import build as msbuild
    from minorseq_b200.synth import SynthConfig, make_tables, synth_states
    from test_host_cpp import _make_bam
    msbuild.build_library()
    msbuild.build_host()
    juliet = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "minorseq_b200", "bin", "juliet")
    t = make_tables(SynthConfig(L=300, seed=5))
    bam = str(tmp_path / "in.bam")
    _make_bam(bam, t, synth_states(t, 0, 200))
    cfg = tmp_path / "cfg.json"
    cfg.write_text(json.dumps({"genes": [{"name": "G", "begin": 1, "end": 301}], "referenceName": "synthetic_ref",
                               "referenceSequence": t.refseq, "version": "test"}))
    for rate in ("-0.5", "nan"):
        oj, oh = tmp_path / f"{rate}.json", tmp_path / f"{rate}.html"
        res = subprocess.run([juliet, "--config", str(cfg), "--indels", "--insertion-rate", rate, bam, str(oj), str(oh)],
                             capture_output=True, text=True)
        assert res.returncode == 1 and re.search(r"ERROR: ms_indel_call failed: ms_indel_call: insertion_rate must lie in \[0, 1\]",
                                                 res.stderr), (rate, res.returncode, res.stderr)
    res = subprocess.run([juliet, "--config", str(cfg), "--indels", "--insertion-rate", "1", bam, str(tmp_path / "ok.json"),
                          str(tmp_path / "ok.html")], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
