"""Consensus parity at the edges: fuse's consensus (K4, csrc/fuse.cu) against `oracle.fuse`, and the per-haplotype consensus
(U15, csrc/group.cu) against haplotype_consensus_oracle.py, compared as exact strings.

The column rule and the insertion rule are driven from hand-built column counts written straight into the count tensor, so
that exact ties, votes equal to min_coverage, support equal to ins_fraction * votes and spacing equal to ins_distance are hit
on purpose, at lengths on both sides of consensus_kernel's per-thread column ranges (per = ceil(L / 1024)) and at insertion
counts on both sides of the hash table's size steps.  Then both consensus paths run from reads: random shapes for K4, and
random labelled groups (empty, one read, a middle window, a thin hole in a span longer than 1024 columns, stray labels) for
U15.  Last, the fuse CLI at L = 9719 with insertions written into the BAM.  Fixed seeds throughout."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import haplotype_consensus_oracle as hco
import ins_table_replica as itr

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from minorseq_b200 import Fuse, Handle, Juliet, _lib, device_rows  # noqa: E402
from minorseq_b200._lib import FuseParams  # noqa: E402
from minorseq_b200.synth import SynthConfig, make_tables, pack_states  # noqa: E402

MS_ERR_ARG, MS_ERR_CAPACITY = -1, -4
_ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


@pytest.fixture(scope="module")
def hd():
    h = Handle(0)
    yield h
    h.close()


# ---------------------------------------------------------------- helpers
def _ptr(a):
    return None if a is None else a.ctypes.data


def _events(ev):
    """[(column, bytes)] -> (col, off, len, pool), one pool entry per event"""
    ln = np.array([len(s) for _, s in ev], dtype=np.int32)
    off = np.concatenate([[0], np.cumsum(ln, dtype=np.int64)[:-1]]).astype(np.int64) if len(ev) else np.zeros(0, np.int64)
    return np.array([c for c, _ in ev], dtype=np.int32), off, ln, b"".join(s for _, s in ev)


def _fuse_on_counts(hd, col, min_coverage=50, ins_fraction=0.5, ins_distance=20):
    """a Fuse whose count tensor holds the [L, 8] counts col"""
    L = col.shape[0]
    f = Fuse(L, handle=hd, min_coverage=min_coverage, ins_fraction=ins_fraction, ins_distance=ins_distance)
    ct = f.counts_tensor()
    ct[: L * 8] = torch.from_numpy(np.ascontiguousarray(col, dtype=np.uint32).reshape(-1).view(np.int32)).cuda()
    torch.cuda.synchronize()          # torch's copy before the handle's stream reads the counts
    return f


def _both(oracle, f, col, ev=(), min_coverage=10, ins_fraction=0.5, ins_distance=20):
    """K4 on the GPU and the oracle with the same counts, events and thresholds: the strings must be equal"""
    f.params.min_coverage, f.params.ins_fraction, f.params.ins_distance = min_coverage, ins_fraction, ins_distance
    ic, io, il, pool = _events(list(ev))
    want = oracle.fuse(col, ic, io, il, pool, min_coverage=min_coverage, ins_fraction=ins_fraction, ins_distance=ins_distance)
    got = f.consensus(ic, io, il, pool)
    if got != want:
        k = next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), min(len(got), len(want)))
        pytest.fail(f"consensus differs (L={col.shape[0]}, lengths {len(got)} / {len(want)}, first at {k}: "
                    f"{got[max(0, k - 5): k + 5]!r} / {want[max(0, k - 5): k + 5]!r})")
    return want


def _majority_columns(L, rng, votes=20):
    """every column a clear majority of a random base, exactly `votes` votes"""
    col = np.zeros((L, 8), dtype=np.uint32)
    b = rng.integers(0, 4, size=L)
    col[np.arange(L), b] = votes - 4
    for s in range(5):
        col[:, s] += (b != s).astype(np.uint32)
    col[:, 7] = col[:, :6].sum(axis=1)
    return col


_PAIRS = [(a, b) for a in range(5) for b in range(a + 1, 5)]


def _columns(L, rng, min_cov):
    """random votes, exact ties between every pair of A C G T -, three- and five-way ties, N-majority columns, zero-vote
    columns, votes of min_cov - 1, min_cov and min_cov + 1, '-'-majority columns; column 0 an A and column L - 1 a T"""
    col = np.zeros((L, 8), dtype=np.uint32)
    kind = rng.integers(0, 8, size=L)
    ntie = 0
    for j in range(L):
        k = kind[j]
        if k == 0:
            col[j, :6] = rng.integers(0, 60, size=6)
        elif k in (1, 2):                                      # a tie of two, cycling through the ten pairs
            v = int(rng.integers(1, 60))
            col[j, :5] = rng.integers(0, v, size=5)
            a, b = _PAIRS[ntie % len(_PAIRS)]
            ntie += 1
            col[j, a] = col[j, b] = v
            col[j, 5] = rng.integers(0, 2 * v)
        elif k == 3:                                           # three or five equal maxima
            v = int(rng.integers(1, 40))
            col[j, :5] = rng.integers(0, v, size=5)
            col[j, rng.choice(5, size=int(rng.choice([3, 5])), replace=False)] = v
        elif k == 4:                                           # N outvotes everything, but does not vote
            col[j, :5] = rng.integers(0, 5, size=5)
            col[j, 5] = 1000
        elif k == 5:                                           # no votes at all
            col[j, 5] = rng.integers(0, 3)
        elif k == 6:                                           # votes next to the threshold
            t = max(0, min_cov + int(rng.integers(-1, 2)))
            col[j, :5] = rng.multinomial(t, rng.dirichlet(np.ones(5)))
        else:                                                  # the deletion wins
            col[j, :4] = rng.integers(0, 20, size=4)
            col[j, 4] = 25 + rng.integers(0, 20)
    col[0, :6] = (100, 0, 0, 0, 0, 0)
    col[L - 1, :6] = (0, 0, 0, 100, 0, 0)
    col[:, 6] = rng.integers(0, 3, size=L)
    col[:, 7] = col[:, :6].sum(axis=1)
    return col


def _codon(i, n=3):
    """a distinct in-frame string per i"""
    return "".join("ACGT"[(i >> (2 * k)) & 3] for k in range(n)).encode()


# ---------------------------------------------------------------- 1. K4 column rule
LENGTHS = [3, 4, 1023, 1024, 1025, 2047, 2048, 2049, 3000, 9719, 20000]


@pytest.mark.parametrize("L", LENGTHS)
def test_column_rule_on_hand_built_counts(oracle, hd, L):
    rng = np.random.default_rng(1000 + L)
    for m in (0, 1, 50):
        col = _columns(L, rng, m)
        f = _fuse_on_counts(hd, col)
        want = _both(oracle, f, col, min_coverage=m)
        assert want[0] == "A" and want[-1] == "T"
    above = int(col[:, :5].sum(axis=1).max()) + 1             # above every column's votes: nothing is written
    assert _both(oracle, f, col, min_coverage=above) == ""


# ---------------------------------------------------------------- 2. K4 insertion rule
@pytest.mark.parametrize("L", [L for L in LENGTHS if L > 1024])
def test_insertions_at_thread_range_boundaries(oracle, hd, L):
    """accepted insertions after the first and last column of several threads' column ranges, after column 0 and L - 1"""
    rng = np.random.default_rng(2000 + L)
    per = -(-L // 1024)
    used = -(-L // per)                                        # threads that own at least one column
    ks = sorted({1, 2, 3, used // 2, used - 2, used - 1})
    targets = sorted({0, L - 1} | {k * per - 1 for k in ks} | {k * per for k in ks if k * per < L})
    col = _columns(L, rng, 50)
    col[targets] = _majority_columns(len(targets), rng, votes=50)
    col[targets[1::3], :6] = (2, 2, 2, 2, 42, 0)               # some of them removed ('-' wins): the insertion stays
    ev = [(c, _codon(i, 3 * (1 + i % 2))) for i, c in enumerate(targets) for _ in range(26)]
    rng.shuffle(ev)
    f = _fuse_on_counts(hd, col)
    want = _both(oracle, f, col, ev, min_coverage=50, ins_distance=1)
    assert len(want) - len(oracle.fuse(col)) == sum(3 * (1 + i % 2) for i in range(len(targets)))   # every one accepted
    _both(oracle, f, col, ev, min_coverage=50, ins_distance=per + 1)


@pytest.mark.parametrize("nins", [0, 1, 511, 512, 513, 1024, 1025, 200_000])
def test_insertion_table_sizes(oracle, hd, nins):
    """event counts on both sides of the table's size steps (1024 slots up to 512 events, 2048 up to 1024, 4096 above), and
    200 k events over about 2 k distinct (column, string) keys"""
    L = 3000
    rng = np.random.default_rng(3000 + nins)
    nkeys = int(np.clip(nins // 4, 1, 2000))
    kcol = rng.integers(-1, L + 1, size=nkeys)                 # -1 and L: keys the rule must ignore
    kstr = [bytes(rng.choice(_ACGT, size=int(rng.choice([3, 3, 6, 4])))) for _ in range(nkeys)]
    w = rng.dirichlet(np.full(nkeys, 0.5))
    which = rng.choice(nkeys, size=nins, p=w)
    ev = [(int(kcol[k]), kstr[k]) for k in which]
    col = _columns(L, rng, 50)
    expect = np.bincount(which, minlength=nkeys)               # votes around twice a key's support: some pass, some fail
    for k in range(nkeys):
        if 0 <= kcol[k] < L:
            col[kcol[k], :5] = rng.multinomial(int(rng.integers(0, 2 * expect[k] + 2)), rng.dirichlet(np.ones(5)))
    f = _fuse_on_counts(hd, col)
    want = _both(oracle, f, col, ev, min_coverage=50)
    if nins >= 511:
        assert len(want) > len(oracle.fuse(col))              # some insertions accepted
    assert itr.table_size(nins) == {0: 1024, 1: 1024, 511: 1024, 512: 1024, 513: 2048, 1024: 2048, 1025: 4096}.get(nins, 1 << 19)


def test_long_probe_chain_wraps_past_the_table_end(oracle, hd):
    """441 distinct 9-long strings at one column and one string at each of ten other columns, every key's home slot among the last
    64 of the 1024-slot table: the probe chains are hundreds of slots long and must wrap past slot 1023.  The home slots come
    from a host replica of ins_tally_kernel's hash (ins_table_replica.py), checked against fuse.cu's source first."""
    bad = itr.source_mismatches()
    assert not bad, "ins_table_replica.py no longer matches csrc/fuse.cu, so this case may not wrap: " + "; ".join(bad)
    L, ts, c0 = 3000, 1024, 1500
    others = [100 + 250 * i for i in range(10)]
    rng = np.random.default_rng(4)

    def near_end(c, need):
        got = {}
        while len(got) < need:
            cand = [bytes(x) for x in rng.choice(_ACGT, size=(4096, 9))]
            home = itr.key_hash(c, cand) & np.uint64(ts - 1)
            got.update((s, None) for s, h in zip(cand, home) if h >= ts - 64)
        return list(got)[:need]

    chain = near_end(c0, 441)
    star = sorted(chain)[200]                                  # not the smallest: ins_fraction 0 must pick another
    ev = [(c0, s) for s in chain if s != star] + [(c0, star)] * 3
    ev += [(c, s) for c in others for s in near_end(c, 1) * 3]
    keys = sorted(set(ev))
    nins = len(ev)
    homes = np.concatenate([itr.key_hash(c, [s]) for c, s in keys]) & np.uint64(ts - 1)
    assert itr.table_size(nins) == ts and len(keys) == 451
    assert itr.forced_wrap(homes, ts), "no probe chain is forced past the table end"
    order = rng.permutation(nins)
    ev = [ev[i] for i in order]
    col = _majority_columns(L, rng)
    col[[c0] + others, :6] = (1, 1, 1, 1, 0, 0)               # 4 votes: 3 events pass at 0.5, 1 does not
    f = _fuse_on_counts(hd, col)
    want = _both(oracle, f, col, ev, min_coverage=1)
    assert star.decode() in want and len(want) == L + 9 * 11
    _both(oracle, f, col, ev, min_coverage=1, ins_fraction=0.0)   # every string passes: the smallest bytes win at c0


@pytest.mark.parametrize("frac", [0.0, 0.5, 0.99])
def test_insertion_support_boundary(oracle, hd, frac):
    """support exactly ins_fraction * votes (rejected: the test is strict) and one above; several passing strings at one column,
    ordered by (length, bytes) compared unsigned, with 'N' and multi-byte UTF-8 strings among them"""
    L = 2100
    rng = np.random.default_rng(int(frac * 100) + 5)
    col = _majority_columns(L, rng)
    ev, c = [], 10
    for v in (1, 2, 3, 10, 40, 100, 101, 200):
        lo = int(np.floor(frac * v))
        for sup in sorted({lo, lo + 1, int(np.ceil(frac * v))}):
            if sup == 0:
                continue
            col[c, :6] = 0
            col[c, :5] = rng.multinomial(v, [0.6, 0.1, 0.1, 0.1, 0.1])
            ev += [(c, _codon(c))] * sup
            c += 25
    for strings in ([("AAA", 1), ("ACN", 2), ("ACA", 1), ("éA", 5), ("€", 1), ("TTTTTT", 9), ("GG", 9)],
                    [("TTT", 3), ("éA", 3), ("€", 3)],
                    [("ACT", 4), ("ACN", 4), ("ACA", 4), ("NNN", 4)],
                    [("é€A", 6), ("€é", 6), ("NNNNNN", 6)]):
        col[c, :6] = (4, 2, 2, 2, 0, 0)
        ev += [(c, s.encode()) for s, n in strings for _ in range(n)]
        c += 25
    assert c < L
    rng.shuffle(ev)
    f = _fuse_on_counts(hd, col)
    _both(oracle, f, col, ev, ins_fraction=frac)


@pytest.mark.parametrize("dist", [0, 1, 20])
def test_insertion_spacing(oracle, hd, dist):
    """candidates ins_distance - 1, ins_distance and ins_distance + 1 columns apart, a greedy chain where a rejected candidate
    must not move the spacing origin, and two strings at one column"""
    L = 3000
    rng = np.random.default_rng(60 + dist)
    col = _majority_columns(L, rng)
    ev, c = [], 7
    for s in (dist - 1, dist, dist + 1):
        if s >= 0:
            ev += [(c, b"GGC")] * 15 + [(c + s, b"TTA")] * 15
            c += 100
    for d in (0, max(0, dist - 1), dist, 2 * dist, 2 * dist + 1, 3 * dist):
        ev += [(c + d, _codon(d))] * 12
    c += 100
    ev += [(c, b"CCG")] * 11 + [(c, b"CAG")] * 11
    rng.shuffle(ev)
    f = _fuse_on_counts(hd, col)
    _both(oracle, f, col, ev, ins_distance=dist)


def test_insertion_events_the_rule_ignores(oracle, hd):
    """columns -1 and L, lengths 0, 1, 2, 4 and 5 never count; an insertion after a '-'-majority column and after a zero-vote
    column is judged like any other"""
    L = 1500
    rng = np.random.default_rng(8)
    col = _majority_columns(L, rng, votes=10)
    ev = [(-1, b"GGG")] * 10 + [(L, b"GGG")] * 10 + [(100, b"")] * 10
    ev += [(200, b"A")] * 10 + [(300, b"GC")] * 10 + [(400, b"ACGT")] * 10 + [(500, b"ACGTA")] * 10
    ev += [(600, b"AAAA")] * 10 + [(600, b"CCC")] * 6          # the 4-long string is out of frame: CCC wins
    col[700, :6] = (1, 1, 1, 1, 20, 0)
    ev += [(700, b"GAT")] * 13
    col[800, :6] = (0, 0, 0, 0, 0, 5)
    ev += [(800, b"TAG")]
    col[900, :6] = 0
    ev += [(900, b"CAT")] * 4
    rng.shuffle(ev)
    f = _fuse_on_counts(hd, col)
    want = _both(oracle, f, col, ev)
    assert len(want) == L - 3 + 3 + 3 + 3 + 3
    _both(oracle, f, col, ev, min_coverage=0, ins_fraction=0.0, ins_distance=0)


def test_fuse_error_paths(oracle, hd):
    L = 100
    col = _majority_columns(L, np.random.default_rng(9))
    f = _fuse_on_counts(hd, col)
    lib = hd.lib
    prm = FuseParams(50, 0.5, 20)
    seq = np.zeros(L + 64, dtype=np.uint8)
    n = C.c_int64()
    pool = np.frombuffer(b"GGCAT", dtype=np.uint8)

    def call(c, o, ln, nins=None):
        ic, io, il = np.array(c, np.int32), np.array(o, np.int64), np.array(ln, np.int32)
        return lib.ms_fuse(hd.h, C.byref(prm), _ptr(ic), _ptr(io), _ptr(il), len(ic) if nins is None else nins, _ptr(pool), len(pool),
                           _ptr(seq), len(seq), C.byref(n))

    assert call([5], [3], [3]) == MS_ERR_ARG                   # past the pool's end
    assert call([5, 6], [0, -1], [3, 3]) == MS_ERR_ARG         # before its start
    assert call([5], [0], [-3]) == MS_ERR_ARG
    assert call([5], [0], [3], nins=-1) == MS_ERR_ARG
    prm.min_coverage = 10
    assert call([5] * 11, [0] * 11, [3] * 11) == 0 and n.value == L + 3       # the handle still works
    assert seq[: n.value].tobytes().decode() == oracle.fuse(col, [5] * 11, [0] * 11, [3] * 11, b"GGCAT", min_coverage=10)
    assert f.consensus([5], [0], [3], b"GGC") == oracle.fuse(col, [5], [0], [3], b"GGC")


@pytest.mark.parametrize("L", [1, 2])
def test_reference_shorter_than_a_codon_is_refused(hd, L):
    with pytest.raises(_lib.MsError, match="error -1"):
        Fuse(L, handle=hd)


# ---------------------------------------------------------------- 3. K4 from reads
_VOCAB = [b"A", b"GC", b"GGC", b"TTA", b"ACGT", b"ACGTA", b"GGCGGC", b"NNA", b"TTTAAA", b"CAG", b"CAGCAGCAG"]
_VOFF = np.concatenate([[0], np.cumsum([len(s) for s in _VOCAB])[:-1]]).astype(np.int64)
_VLEN = np.array([len(s) for s in _VOCAB], dtype=np.int32)
_VPOOL = b"".join(_VOCAB)


def _random_reads(rng, L, R, p_sub, p_del, p_n, trunc):
    """[R, L] states of noisy copies of one random sequence, a share of the reads truncated at a random end"""
    base = rng.integers(0, 4, size=L).astype(np.uint8)
    u = rng.random((R, L))
    st = np.where(u < p_n, 5, np.where(u < p_n + p_del, 4, np.where(u < p_n + p_del + p_sub, rng.integers(0, 4, size=(R, L)), base)))
    st = st.astype(np.uint8)
    for c in rng.choice(L, size=min(L, 3), replace=False):     # a few major deletions
        st[rng.random(R) < 0.7, c] = 4
    cut = rng.random(R) < trunc
    b = np.where(cut & (rng.random(R) < 0.5), rng.integers(0, L, size=R), 0)
    e = np.where(cut, np.maximum(b + 1, rng.integers(0, L + 1, size=R)), L)
    cols = np.arange(L)
    st[(cols[None, :] < b[:, None]) | (cols[None, :] >= e[:, None])] = 7
    return st


def _read_insertions(rng, st, p_ins, hot):
    """insertion events on spanned columns (bit 3 set, as the CIGAR expansion sets it): scattered ones from the vocabulary and,
    at `hot` columns, one string carried by a random share of the reads there.  -> (read, col, vocabulary index)"""
    R, L = st.shape
    spanned = (st & 7) != 7
    which = np.full((R, L), -1, dtype=np.int64)
    e = (rng.random((R, L)) < p_ins) & spanned
    which[e] = rng.integers(0, len(_VOCAB), size=int(e.sum()))
    for c in hot:
        share = rng.uniform(0.3, 0.95)
        m = spanned[:, c] & (rng.random(R) < share)
        which[m, c] = int(rng.choice([2, 3, 6, 9, 10, 4]))
    r, c = np.nonzero(which >= 0)
    st[r, c] |= 8
    return r, c, which[r, c]


@pytest.mark.parametrize("seed", list(range(500, 524)))
def test_fuse_from_reads_random(oracle, hd, seed):
    rng = np.random.default_rng(seed)
    L = int(rng.choice([rng.integers(9, 200), rng.integers(200, 3500), rng.integers(3500, 12501)]))
    R = int(rng.choice([rng.integers(0, 40), rng.integers(40, 1500), rng.integers(1500, 4001)]))
    if L > 6000:
        R = min(R, 1500)
    st = _random_reads(rng, L, R, float(rng.choice([5e-3, 5e-2])), float(rng.choice([3e-3, 3e-2, 0.2])),
                       float(rng.choice([0.0, 2e-2, 0.1])), float(rng.choice([0.0, 0.05, 0.5])))
    hot = rng.choice(L, size=max(1, L // 150), replace=False)
    r, c, k = _read_insertions(rng, st, float(rng.choice([0.0, 1e-3, 1e-2])), hot)
    ic, io, il = c.astype(np.int32), _VOFF[k], _VLEN[k]
    prm = dict(min_coverage=int(rng.choice([0, 1, 10, 50])), ins_fraction=float(rng.choice([0.0, 0.3, 0.5])),
               ins_distance=int(rng.choice([0, 1, 20])))
    f = Fuse(L, handle=hd, **prm)
    packed = pack_states(st) if R else np.zeros((0, 4 * ((L + 31) // 32)), dtype=np.uint32)
    mode = seed % 3                                            # one call, two batches, or from host rows
    if mode == 0 or R == 0:
        d = device_rows(packed)
        f.pileup_device(d.data_ptr(), R)
    elif mode == 1:
        r1 = 8 * (R // 16)
        d1, d2 = device_rows(packed[:r1]), device_rows(packed[r1:])
        f.pileup_device(d1.data_ptr(), r1)
        f.pileup_device(d2.data_ptr(), R - r1)
    else:
        f.pileup_host(np.ascontiguousarray(packed))
    ocol, _ = oracle.pileup(st, None, codons=False) if R else (np.zeros((L, 8), np.uint32), None)
    got_col = f.counts_tensor()[: L * 8].cpu().numpy().view(np.uint32).reshape(L, 8)
    np.testing.assert_array_equal(got_col[:, :6], ocol[:, :6])
    want = oracle.fuse(ocol, ic, io, il, _VPOOL, **prm)
    assert f.consensus(ic, io, il, _VPOOL) == want, (seed, L, R, prm)


# ---------------------------------------------------------------- 4. U15, randomised groups
def _group_consensus(j, ngroups, labels, ins, min_coverage, ins_fraction, ins_distance):
    """ms_group_consensus through ctypes on the counts of the last group_pileup, with the capacity retry: a first call with
    no room reports the sizes.  ins: (read, col, off, len, pool); each event carries its read's raw label."""
    read, col, off, ln, pool = ins
    nins = len(read)
    ig = np.ascontiguousarray(labels[read], dtype=np.int32) if nins else None
    ic = np.ascontiguousarray(col, dtype=np.int32) if nins else None
    io = np.ascontiguousarray(off, dtype=np.int64) if nins else None
    il = np.ascontiguousarray(ln, dtype=np.int32) if nins else None
    pl = np.frombuffer(pool, dtype=np.uint8) if nins else None
    prm = FuseParams(min_coverage, ins_fraction, ins_distance)
    so = np.zeros(ngroups + 1, dtype=np.int64)

    def call(buf, cap):
        return j.lib.ms_group_consensus(j.hd.h, C.byref(prm), _ptr(ig), _ptr(ic), _ptr(io), _ptr(il), nins, _ptr(pl), len(pool),
                                        _ptr(buf), cap, _ptr(so))

    rc = call(None, 0)
    if so[-1] == 0:
        assert rc == 0
        return [""] * ngroups
    assert rc == MS_ERR_CAPACITY
    buf = np.zeros(int(so[-1]), dtype=np.uint8)
    assert call(buf, len(buf)) == 0, j.lib.ms_last_error(j.hd.h)
    return [buf[so[g]: so[g + 1]].tobytes().decode() for g in range(ngroups)]


class _Groups:
    """reads and insertion events built group by group; labels are the group ids, shuffled with the reads at the end"""

    def __init__(self, L, rng):
        self.L, self.rng, self.rows, self.lab, self.ev = L, rng, [], [], []
        self.seq = {}

    def sequence(self, g):
        if g not in self.seq:
            self.seq[g] = self.rng.integers(0, 4, size=self.L).astype(np.uint8)
        return self.seq[g]

    def reads(self, g, n, lo=0, hi=None, noise=0.02):
        """n reads of group g's sequence covering [lo, hi), with substitutions, deletions and N"""
        hi = self.L if hi is None else hi
        st = np.full((n, self.L), 7, dtype=np.uint8)
        if n == 0:
            return st
        u = self.rng.random((n, hi - lo))
        body = np.broadcast_to(self.sequence(g)[lo:hi], (n, hi - lo)).copy()
        body[u < noise] = self.rng.integers(0, 4, size=int((u < noise).sum()))
        body[(u >= noise) & (u < 1.5 * noise)] = 4
        body[(u >= 1.5 * noise) & (u < 2 * noise)] = 5
        st[:, lo:hi] = body
        return st

    def add(self, st, g):
        first = len(self.lab)                                   # index of the first new read
        self.rows.append(st)
        self.lab += [g] * st.shape[0]
        return first

    def insert(self, reads, c, s):
        """an insertion of s after column c on each of the given reads (only where the read spans c)"""
        for r in reads:
            self.ev.append((int(r), int(c), s))

    def finish(self):
        L = self.L
        st = np.concatenate(self.rows) if self.rows else np.zeros((0, L), np.uint8)
        lab = np.array(self.lab, dtype=np.int32)
        ev = [(r, c, s) for (r, c, s) in self.ev if (st[r, c] & 7) != 7]
        for r, c, _ in ev:
            st[r, c] |= 8
        perm = self.rng.permutation(len(lab))
        inv = np.empty_like(perm)
        inv[perm] = np.arange(len(perm))
        pool = b"".join(s for _, _, s in ev)
        ln = np.array([len(s) for _, _, s in ev], dtype=np.int32)
        off = np.concatenate([[0], np.cumsum(ln, dtype=np.int64)[:-1]]).astype(np.int64) if ev else np.zeros(0, np.int64)
        read = np.array([inv[r] for r, _, _ in ev], dtype=np.int64)
        col = np.array([c for _, c, _ in ev], dtype=np.int32)
        return st[perm], lab[perm], (read, col, off, ln, pool)


def _kinds(L, G):
    """the kind of each group: the special ones first (those the shape allows), then random ones"""
    kinds = (["hole", "bound"] if L > 1100 else []) + ["leak_a", "leak_b", "tie", "exact", "del", "window", "empty", "one"]
    return (kinds + ["random"] * G)[:G]


def _build_groups(L, G, thr, rng):
    """reads and events of the groups _kinds(L, G) names, plus stray reads labelled -1 and >= G with events of their own"""
    b = _Groups(L, rng)
    kinds = _kinds(L, G)
    for g in range(G):
        kind = kinds[g]
        if kind == "hole":                                     # ~30 reads over [20, L - 20), most skip a 100-column window
            n = max(30, thr + 3)
            st = b.reads(g, n, 20, L - 20)
            w = L // 2
            st[3:, w: w + 100] = 7
            r0 = b.add(st, g)
            b.insert(range(r0, r0 + 3), w + 50, b"GAC")          # judged against the three votes of the thin column
            b.insert(range(r0, r0 + n), w - 200, b"TTG")
        elif kind == "bound":                                  # insertions at the per-thread boundaries of a span > 1024
            n = thr + 4
            x0, x1 = 7, L - 3
            r0 = b.add(b.reads(g, n, x0, x1, noise=0.004), g)
            per = -(-(x1 - x0) // 1024)
            used = -(-(x1 - x0) // per)
            for i, k in enumerate(sorted({1, 2, used // 2, used - 1})):
                b.insert(range(r0, r0 + n), x0 + k * per - 1, _codon(2 * i))
                b.insert(range(r0, r0 + n), x0 + k * per, _codon(2 * i + 1))
            b.insert(range(r0, r0 + n), x0, b"CCC")
            b.insert(range(r0, r0 + n), x1 - 1, b"AAAGGG")
        elif kind == "leak_a":                                 # an accepted insertion near the end of the group ...
            r0 = b.add(b.reads(g, thr + 2), g)
            b.insert(range(r0, r0 + thr + 2), L - 4, b"GTA")
        elif kind == "leak_b":                                 # ... and one near the start of the next: spacing is per group
            r0 = b.add(b.reads(g, thr + 2), g)
            b.insert(range(r0, r0 + thr + 2), 2, b"CTA")
        elif kind == "tie":                                    # half A half C, half a base half '-': the lowest code wins
            n = 2 * max(1, (thr + 1) // 2)
            st = b.reads(g, n, noise=0.0)
            st[: n // 2, 1::3] = 0
            st[n // 2:, 1::3] = 1
            st[: n // 2, 2::3] = 4
            st[n // 2:, 2::3] = 3
            b.add(st, g)
        elif kind == "exact":                                  # every column exactly at the threshold
            b.add(b.reads(g, thr, noise=0.0), g)
        elif kind == "del":                                    # '-'-majority columns inside the span
            n = thr + 6
            st = b.reads(g, n, 0, L)
            st[: n - 2, L // 3] = 4
            st[: n - 1, L // 2] = 4
            r0 = b.add(st, g)
            b.insert(range(r0, r0 + n), L // 3, b"GGA")
        elif kind == "window":                                 # the reads cover only a middle window, one a little more
            n = thr + 2
            r0 = b.add(b.reads(g, n, L // 4, 3 * L // 4 + 1), g)
            b.insert(range(r0, r0 + n), L // 2, b"ATG")
            r1 = b.add(b.reads(g, 1, L // 4 - 3, 3 * L // 4 + 1), g)
            b.insert([r1], L // 4 - 2, b"TTT")                   # after a trimmed column (thr > 1): ignored
        elif kind == "one":
            r0 = b.add(b.reads(g, 1, 1, L - 1), g)
            b.insert([r0], L // 2, b"CAT")
        elif kind == "random":
            n = int(rng.integers(0, 25))
            lo = rng.integers(0, L // 3 + 1, size=n)
            hi = rng.integers(2 * L // 3, L + 1, size=n)
            for i in range(n):
                b.add(b.reads(g, 1, int(lo[i]), int(max(hi[i], lo[i] + 1)), noise=0.05), g)
            if n:
                first = len(b.lab) - n
                for c in rng.choice(L, size=min(L, 3), replace=False):
                    b.insert([r for r in range(first, first + n) if rng.random() < 0.7], c, _VOCAB[int(rng.integers(0, len(_VOCAB)))])
    for stray in (-1, G, G + 7):                               # reads no group counts, and their events with them
        r0 = b.add(b.reads(0, 20), stray)
        b.insert(range(r0, r0 + 20), L // 2 + 1, b"CCCGGG")
    return b.finish()


GROUP_CASES = [  # (seed, L, ngroups, min_coverage, ins_fraction, ins_distance)
    (1, 33, 1, 10, 0.5, 20), (2, 33, 7, 0, 0.0, 0), (3, 33, 200, 1, 0.5, 20),
    (4, 1025, 2, 1, 0.5, 20), (5, 1025, 1000, 10, 0.5, 0), (6, 1025, 7, 400, 0.0, 20),
    (7, 3000, 7, 10, 0.5, 20), (8, 3000, 200, 10, 0.0, 0), (9, 3000, 2, 400, 0.5, 20),
    (10, 9719, 1, 0, 0.5, 20), (11, 9719, 2, 10, 0.0, 20), (12, 9719, 7, 1, 0.5, 0),
]


@pytest.mark.parametrize("seed,L,G,mc,frac,dist", GROUP_CASES)
def test_group_consensus_random_groups(oracle, hd, seed, L, G, mc, frac, dist):
    rng = np.random.default_rng(seed)
    st, lab, ins = _build_groups(L, G, max(1, mc), rng)
    R = st.shape[0]
    j = Juliet(L, [(1, L + 1)], handle=hd)
    d = device_rows(pack_states(st))
    d_lab = torch.from_numpy(lab).cuda()
    torch.cuda.synchronize()                                   # the labels are copied on torch's stream
    j.group_pileup(d.data_ptr(), d_lab.data_ptr(), R, G)
    np.testing.assert_array_equal(j.group_counts(), hco.group_counts(st, lab, G))
    got = _group_consensus(j, G, lab, ins, mc, frac, dist)
    want = hco.haplotype_consensus(st, lab, G, ins, min_coverage=mc, ins_fraction=frac, ins_distance=dist)
    bad = [g for g in range(G) if got[g] != want[g]]
    assert not bad, f"groups {bad[:8]} differ; first: {got[bad[0]][:80]!r} / {want[bad[0]][:80]!r}"
    kinds = _kinds(L, G)
    if "empty" in kinds:
        assert want[kinds.index("empty")] == ""
    if "hole" in kinds:                                        # the thin window is a run of N with the insertion inside it
        assert "N" * 40 + "GAC" in want[kinds.index("hole")] or mc <= 3


def test_group_consensus_without_reads(hd):
    """no reads at all: every group's sequence is empty, and the first call already succeeds"""
    L, G = 1025, 7
    j = Juliet(L, [(1, L + 1)], handle=hd)
    d = device_rows(np.zeros((0, 4 * ((L + 31) // 32)), dtype=np.uint32))
    lab = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    j.group_pileup(d.data_ptr(), lab.data_ptr(), 0, G)
    assert j.group_counts().sum() == 0
    ins = (np.array([0]), np.array([5]), np.array([0]), np.array([3]), b"GGC")
    assert _group_consensus(j, G, np.array([2], np.int32), ins, 10, 0.5, 20) == [""] * G


# ---------------------------------------------------------------- 5. the fuse CLI at L = 9719
@pytest.fixture(scope="module")
def binaries():
    from minorseq_b200 import build as msbuild
    msbuild.build_library()
    return msbuild.build_host()


def test_fuse_cli_long_reference_matches_oracle(binaries, oracle, tmp_path):
    """insertions in the BAM after column 0, after columns at K4's per-thread range boundaries (per = 10 at L = 9719) and
    after column L - 1; one too close to an accepted one and one out of frame"""
    from test_host_cpp import _make_bam
    L, R = 9719, 240
    rng = np.random.default_rng(9719)
    t = make_tables(SynthConfig(L=L, seed=9719))
    st = _random_reads(rng, L, R, 5e-3, 3e-3, 2e-3, 0.1)
    accepted = {0: "GGC", 29: "TTAGGC", 50: "CAG", 5119: "ACG", 5150: "GATTAC", 9690: "CCA", L - 1: "TGA"}
    rejected = {9700: "AAA", 3000: "GG"}
    ins = {}
    for r in range(R):
        d = {c: s for c, s in {**accepted, **rejected}.items() if (st[r, c] & 7) != 7 and rng.random() < 0.8}
        for c in d:
            st[r, c] |= 8
        ins[r] = d
    bam = str(tmp_path / "long.bam")
    _make_bam(bam, t, st, insertions=ins)
    fa = str(tmp_path / "out.fasta")
    res = subprocess.run([os.path.join(binaries, "fuse"), bam, fa], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    lines = open(fa).read().split("\n")
    assert lines[0].startswith(">long.bam|fuse|synthetic_ref")
    got = "".join(lines[1:])
    keep = (st & 7 != 7).any(axis=1)
    ocol, _ = oracle.pileup(st[keep], None, codons=False)
    ev = [(c, s) for r in range(R) if keep[r] for c, s in sorted(ins[r].items())]
    ic, io, il, pool = _events([(c, s.encode()) for c, s in ev])
    want = oracle.fuse(ocol, ic, io, il, pool)
    assert got == want
    assert len(want) - len(oracle.fuse(ocol)) == sum(len(s) for s in accepted.values())
