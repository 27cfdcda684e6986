"""Test-side restatement of restatement choice U15, the per-haplotype consensus, from column states and read labels (numpy).

Not part of `oracle/`: the product's rules for U6-U8 are checked against `oracle.fuse` there; this file restates only what
U15 adds on top of them:
  * a group's reads are the reads labelled g (for haplotypes: the rank in juliet's order, below nreported);
  * its columns are counted as K1 counts all reads (A C G T - N ins cov);
  * each column is called as fuse calls it (votes = A+C+G+T+-, the first maximum in that order, a '-' column is removed),
    except that a column with fewer than max(1, min_coverage) votes is written 'N' -- inside the span from the first to
    the last column with enough votes; the columns outside it are trimmed;
  * insertions: the group's own events tallied by (column, string), in frame and seen in more than ins_fraction * votes
    of the group's reads at that column, after a column inside the span, greedy spacing ins_distance left to right over
    the candidates in (column, length, string) order.
"""
from collections import Counter

import numpy as np


def group_counts(states: np.ndarray, labels: np.ndarray, ngroups: int) -> np.ndarray:
    """[R, L] uint8 states (bits 0-2 state, bit 3 insertion-follows), [R] labels -> [ngroups, L, 8] uint32 counts of the
    reads labelled g; other labels are skipped."""
    R, L = states.shape
    labels = np.asarray(labels)
    out = np.zeros((ngroups, L, 8), dtype=np.uint32)
    st = states & 7
    ins = (states >> 3) & 1
    for g in range(ngroups):
        m = labels == g
        s = st[m]
        for k in range(6):
            out[g, :, k] = (s == k).sum(axis=0)
        out[g, :, 6] = ins[m].sum(axis=0)
        out[g, :, 7] = (s <= 5).sum(axis=0)
    return out


def consensus(col: np.ndarray, ins=(), min_coverage=10, ins_fraction=0.5, ins_distance=20) -> str:
    """U15 for one group: col [L, 8] its counts, ins its insertion events as (column, bytes) pairs."""
    votes = col[:, :5].astype(np.int64).sum(axis=1)
    thr = max(1, int(min_coverage))
    covered = np.nonzero(votes >= thr)[0]
    if len(covered) == 0:
        return ""
    lo, hi = int(covered[0]), int(covered[-1])
    tally = Counter((int(c), bytes(s)) for c, s in ins)
    acc, last = {}, -1
    for c, s in sorted(tally, key=lambda k: (k[0], len(k[1]), k[1])):
        if c < lo or c > hi or c in acc or len(s) == 0 or len(s) % 3:
            continue
        if not tally[(c, s)] > ins_fraction * float(votes[c]):
            continue
        if last >= 0 and c - last < ins_distance:
            continue
        acc[c] = s
        last = c
    out = []
    for j in range(lo, hi + 1):
        if votes[j] < thr:
            out.append("N")
        else:
            best = int(np.argmax(col[j, :5]))          # first maximum in the order A, C, G, T, -
            if best < 4:
                out.append("ACGT"[best])
        if j in acc:
            out.append(acc[j].decode())
    return "".join(out)


def haplotype_consensus(states, labels, ngroups, insertions=None, min_coverage=10, ins_fraction=0.5, ins_distance=20):
    """Every group's sequence.  insertions: (read, col, off, len, pool) events; an event belongs to its read's group."""
    counts = group_counts(states, labels, ngroups)
    per = [[] for _ in range(ngroups)]
    if insertions is not None:
        read, col, off, ln, pool = insertions
        labels = np.asarray(labels)
        for r, c, o, n in zip(read, col, off, ln):
            g = int(labels[r])
            if 0 <= g < ngroups:
                per[g].append((int(c), pool[int(o): int(o) + int(n)]))
    return [consensus(counts[g], per[g], min_coverage, ins_fraction, ins_distance) for g in range(ngroups)]
