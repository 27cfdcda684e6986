"""The control comparison (restatement choice U22) restated in numpy, for the tests.

From the per-read column states of a sample and a control: the codon histograms (a codon counts where all three states are
A/C/G/T, at the genes' codon starts), K2's positions and reference codon (rare_linkage_oracle.positions; the sample's major
codon, lowest index on ties, where the reference sequence has none), and for every codon c != ref with sample count k >= 1
the tail p = P(X >= k) of [[k, n - k], [k0, n0 - k0]] from hypergeom_reference (mpmath); p = 1 when n0 = 0.  A codon that is
not listed and whose scipy tail is far above alpha / ntests cannot be called: only the decision matters there, so mpmath is
skipped for it.
"""
import numpy as np
from scipy.stats import hypergeom

import hypergeom_reference as ref
import rare_linkage_oracle as ro

SCREEN = 4.0        # a scipy tail above SCREEN x the bound cannot be below it


def start_mask(L, genes, region=None):
    m = np.zeros(L, dtype=bool)
    for _, _, s, _, _ in ro.positions(L, genes, region=region):
        m[s] = True
    return m


def histogram(states, L, genes, region=None):
    """[R, L] states -> [L, 64] uint32 codon histogram at the genes' codon starts"""
    st = np.asarray(states) & 7
    h = np.zeros((L, 64), dtype=np.uint32)
    for s in np.nonzero(start_mask(L, genes, region))[0]:
        a, b, c = st[:, s].astype(np.int64), st[:, s + 1].astype(np.int64), st[:, s + 2].astype(np.int64)
        ok = (a < 4) & (b < 4) & (c < 4)
        h[s] = np.bincount((16 * a + 4 * b + c)[ok], minlength=64)
    return h


def _upper_scipy(a, b, c, d):
    return float(hypergeom.sf(a - 1, a + b + c + d, a + c, a + b))


def pvalue(k, n, k0, n0):
    """U22's p: the control's 2x2 test, 1 without control coverage"""
    if n0 == 0:
        return ref.mp.mpf(1)
    return ref.fisher_greater(k, n - k, k0, n0 - k0)


def control(codon, ctl, L, genes, refseq=None, alpha=0.01, min_perc=None, max_perc=None, region=None, listed=()):
    """-> (records sorted by (gene, col, codon), uncovered positions).  listed: (gene, col, codon) triples.  A record is a dict
    with the fields of ms_control_variant (pvalue an mpf; None where the codon is neither called nor listed, never returned)."""
    listed = set(listed)
    out, uncovered = [], 0
    for g, ci, s, rc, ntests in ro.positions(L, genes, refseq, region):
        h, h0 = [int(x) for x in codon[s]], [int(x) for x in ctl[s]]
        n, n0 = sum(h), sum(h0)
        if n == 0:
            continue
        if n0 == 0:
            uncovered += 1
        if rc < 0:
            rc = max(range(64), key=lambda c: (h[c], -c))
        for c in range(64):
            k, k0 = h[c], h0[c]
            if c == rc or k == 0:
                continue
            is_listed = (g, s, c) in listed
            if not is_listed and n0 > 0 and _upper_scipy(k, n - k, k0, n0 - k0) > SCREEN * alpha / ntests:
                continue
            p = pvalue(k, n, k0, n0)
            called = bool(p * ntests < alpha)
            perc = 100.0 * k / n
            if min_perc is not None and not perc > min_perc:
                called = False
            if max_perc is not None and not perc < max_perc:
                called = False
            if not called and not is_listed:
                continue
            out.append(dict(gene=g, codon_index=ci, col=s, ref_codon=rc, codon=c, count=k, coverage=n, control_count=k0,
                            control_coverage=n0, ntests=ntests, called=int(called), listed=int(is_listed), pvalue=p))
    out.sort(key=lambda r: (r["gene"], r["col"], r["codon"]))
    return out, uncovered


def report_rows(records, drugs_of=None, drm_only=False):
    """juliet's "control" rows: every record (the control calls and the listed report variants), with control_call /
    model_call; --drm-only keeps the rows with a DRM (drugs_of(record) -> list of drug names)"""
    rows = []
    for r in records:
        drugs = drugs_of(r) if drugs_of else []
        if drm_only and not drugs:
            continue
        rows.append(dict(r, control_call=bool(r["called"]), model_call=bool(r["listed"]), known_drm=" + ".join(drugs)))
    return rows
