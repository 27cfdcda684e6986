// linkage_core.h -- pairwise variant linkage measures (restatement choice U14, SURVEY App. B), host + device.
//
// For two called variants v, w and the n reads whose codons at both are clean (all three states A/C/G/T):
//   a = reads carrying both, b = v only, c = w only, d = n - a - b - c.
// f_v = (a+b)/n, f_w = (a+c)/n, D = a/n - f_v f_w, r^2 = D^2 / (f_v(1-f_v) f_w(1-f_w)), D' = D / D_max with
// D_max = min(f_v(1-f_w), (1-f_v) f_w) for D > 0 and min(f_v f_w, (1-f_v)(1-f_w)) for D < 0.  Both are 0 when a margin
// is empty or full.  Build with -fmad=false (like fisher_core.h) so that host and device give the same doubles.
#pragma once
#include <stdint.h>
#include "fisher_core.h"

namespace ms {

// pairs whose codons share a column are determined by the bases themselves and are not tested
constexpr int32_t kLinkageMinSpacing = 3;
constexpr int32_t kLinkageMinReads = 10;     // default informative reads of a tested pair (the haplotype threshold, F21)
enum { kLinkageLinked = 1, kLinkageExclusive = 2 };

// Evaluated as n^2 D = a d - b c and the n^2-scaled margins, products of 32-bit counts that are exact in 64-bit integers: the
// difference a/n - f_v f_w in doubles cancels, and for a table like [[n-2, 1], [1, 0]] gave D' = -1.0005 instead of -1.
MS_HD void linkage_measures(uint32_t a, uint32_t b, uint32_t c, uint32_t n, double* d_prime, double* r2) {
    *d_prime = 0.0;
    *r2 = 0.0;
    const uint32_t mv = a + b, mw = a + c;
    if (mv == 0 || mv == n || mw == 0 || mw == n) return;
    const uint64_t v1 = mv, v0 = n - mv, w1 = mw, w0 = n - mw;
    const uint64_t ad = static_cast<uint64_t>(a) * (n - mv - c), bc = static_cast<uint64_t>(b) * c;
    const double cross = ad >= bc ? static_cast<double>(ad - bc) : -static_cast<double>(bc - ad);   // n^2 D
    *r2 = (cross * cross) / (static_cast<double>(v1 * v0) * static_cast<double>(w1 * w0));
    if (ad > bc) {
        const uint64_t x = v1 * w0, y = v0 * w1;
        *d_prime = cross / static_cast<double>(x < y ? x : y);
    } else if (ad < bc) {
        const uint64_t x = v1 * w1, y = v0 * w0;
        *d_prime = cross / static_cast<double>(x < y ? x : y);
    }
}

// The two one-sided Fisher tails of the top-left cell X of the tables with the margins of [[a,b],[c,d]]:
// p_together = P(X >= a) (fisher_upper), p_apart = P(X <= a) = fisher_greater of the mirrored table.  Only the tail that lies on
// a's side of the mode can be small; it is summed directly (stopped once it reaches `enough`, as in K2).  The other one holds the
// mode and is taken as 1 - its complement: summed from a, its first term can lie so far out that it underflows to 0, and a
// strongly linked pair's P(X <= a) would come out as 0 instead of 1.
MS_HD void linkage_tails(uint32_t a, uint32_t b, uint32_t c, uint32_t d, double enough, double* p_together, double* p_apart) {
    *p_together = fisher_upper<true>(a, b, c, d, enough);
    if (fisher_at_or_above_mode(a, b, c, d))
        *p_apart = (b == 0 || c == 0) ? 1.0 : 1.0 - fisher_greater<true>(a + 1, b - 1, c - 1, d + 1);   // 1 - P(X >= a + 1)
    else
        *p_apart = fisher_greater<true>(b, a, d, c, enough);
}

}  // namespace ms
