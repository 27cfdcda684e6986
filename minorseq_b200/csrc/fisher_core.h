// fisher_core.h -- fp64 one-sided Fisher exact test, host + device.
//
// juliet's test is "a Bonferroni-corrected Fisher's Exact test"
// (/root/reference/doc/JULIET.md:42).  The tail P(X >= a) of the hypergeometric
// distribution is evaluated from one saddle-point point mass (Loader's binomial
// deviance formulation: stirlerr / bd0, as published in "Fast and accurate
// computation of binomial probabilities", C. Loader 2000) followed by the exact
// term-ratio recurrence.  Unlike a difference of log-gammas this keeps ~1e-14
// relative accuracy at coverages of 1e6 reads, which the 1e-9 parity bar against
// the long-double oracle needs.  Only + - * / log exp log1p are used; build with
// FMA contraction off (-fmad=false) so host and device agree to the last ulps of
// the libm calls.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define MS_HD __host__ __device__ inline
#else
#define MS_HD inline
#endif

namespace ms {

// log(n!) - Stirling approximation, n integer valued
MS_HD double stirlerr(double n) {
    const double sfe[16] = {0.0,
                            0.08106146679532725821967026,
                            0.04134069595540929409382208,
                            0.02767792568499833914878929,
                            0.02079067210376509311152277,
                            0.01664469118982119216319487,
                            0.01387612882307074799874573,
                            0.01189670994589177009505572,
                            0.01041126526197209649747857,
                            0.009255462182712732917728637,
                            0.008330563433362871256469319,
                            0.007573675487951840794972024,
                            0.006942840107209529865664153,
                            0.006408994188004207068439631,
                            0.005951370112758847735624416,
                            0.00555473355196280137103869};
    const double S0 = 1.0 / 12.0, S1 = 1.0 / 360.0, S2 = 1.0 / 1260.0, S3 = 1.0 / 1680.0, S4 = 1.0 / 1188.0;
    if (n < 16.0) return sfe[static_cast<int>(n)];
    const double nn = n * n;
    if (n > 500.0) return (S0 - S1 / nn) / n;
    if (n > 80.0) return (S0 - (S1 - S2 / nn) / nn) / n;
    if (n > 35.0) return (S0 - (S1 - (S2 - S3 / nn) / nn) / nn) / n;
    return (S0 - (S1 - (S2 - (S3 - S4 / nn) / nn) / nn) / nn) / n;
}

// deviance term x*log(x/np) + np - x, stable when x is close to np
MS_HD double bd0(double x, double np) {
    if (fabs(x - np) < 0.1 * (x + np)) {
        double v = (x - np) / (x + np);
        double s = (x - np) * v;
        double ej = 2.0 * x * v;
        v = v * v;
        for (int j = 1; j < 1000; ++j) {
            ej *= v;
            const double s1 = s + ej / (2 * j + 1);
            if (s1 == s) return s1;
            s = s1;
        }
    }
    return x * log(x / np) + np - x;
}

// kPreciseLog: take log(1 - x/n) as log((n - x) / n) when x > n/2.  log1p(-x/n) loses the low digits of 1 - x/n when x is
// close to n: relative error ~1e-16 * x / (n - x), 4e-11 in a linkage table such as [[1999999, 0], [0, 1]].  K2 keeps the
// plain form so that its p-values stay the same bit for bit: in its tables [[k, n-k], [e, n-e]] the loss is x / (n - x) =
// k / e, and where that is large enough to matter (~1e4) the tail is far below 1e-300.
template <bool kPreciseLog = false>
MS_HD double dbinom_raw(double x, double n, double p, double q) {
    const double ln2pi = 1.83787706640934548356065947281;
    if (p == 0.0) return x == 0.0 ? 1.0 : 0.0;
    if (q == 0.0) return x == n ? 1.0 : 0.0;
    if (x == 0.0) {
        if (n == 0.0) return 1.0;
        const double lc = (p < 0.1) ? -bd0(n, n * q) - n * p : n * log(q);
        return exp(lc);
    }
    if (x == n) {
        const double lc = (q < 0.1) ? -bd0(n, n * p) - n * q : n * log(p);
        return exp(lc);
    }
    if (x < 0.0 || x > n) return 0.0;
    const double lc = stirlerr(n) - stirlerr(x) - stirlerr(n - x) - bd0(x, n * p) - bd0(n - x, n * q);
    const double lf = ln2pi + log(x) + (kPreciseLog && x > 0.5 * n ? log((n - x) / n) : log1p(-x / n));
    return exp(lc - 0.5 * lf);
}

// P(X = x), X ~ Hypergeometric(white r, black b, draws n)
template <bool kPreciseLog = false>
MS_HD double dhyper(double x, double r, double b, double n) {
    if (x < 0.0 || x > r || n - x > b || n - x < 0.0) return 0.0;
    if (n == 0.0) return x == 0.0 ? 1.0 : 0.0;
    const double p = n / (r + b), q = (r + b - n) / (r + b);
    const double p1 = dbinom_raw<kPreciseLog>(x, r, p, q);
    const double p2 = dbinom_raw<kPreciseLog>(n - x, b, p, q);
    const double p3 = dbinom_raw<kPreciseLog>(n, r + b, p, q);
    return p1 * p2 / p3;
}

// one-sided "greater" p-value of the 2x2 table [[a,b],[c,d]].  `enough`: the caller only needs to know whether
// p < enough, so the (monotone) partial sum is returned as soon as it reaches it.  Codons at their expected
// sequencing-error count have p ~ 0.5 and a tail of a few hundred slowly falling terms; their first term alone is
// orders of magnitude above a Bonferroni threshold, and they are most of what K2 would otherwise spend its time on.
template <bool kPreciseLog = false>
MS_HD double fisher_greater(uint32_t a, uint32_t b, uint32_t c, uint32_t d, double enough = 2.0) {
    const double white = static_cast<double>(a) + c, black = static_cast<double>(b) + d;
    const double draws = static_cast<double>(a) + b;
    const double xmax = white < draws ? white : draws;
    double x = a;
    double term = dhyper<kPreciseLog>(x, white, black, draws);
    double sum = term;
    while (x < xmax && term > 0.0 && sum < enough) {
        const double ratio = (white - x) * (draws - x) / ((x + 1.0) * (black - draws + x + 1.0));
        term *= ratio;
        sum += term;
        x += 1.0;
        // the pmf is unimodal: once it is falling, terms below 2^-70 of the sum cannot change the
        // double result any more (far inside the 1e-9 parity bar against the long-double oracle)
        if (ratio < 1.0 && term < sum * 8.470329472543003e-22) break;
    }
    return sum > 1.0 ? 1.0 : sum;
}

// true when the top-left cell a of [[a,b],[c,d]] is at or above the mode of its hypergeometric distribution, i.e. the upper
// tail P(X >= a) is the one that can be small
MS_HD bool fisher_at_or_above_mode(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    const double n = static_cast<double>(a) + b + c + d;
    const double mode = floor((static_cast<double>(a) + b + 1.0) * (static_cast<double>(a) + c + 1.0) / (n + 2.0));
    return static_cast<double>(a) >= mode;
}

// P(X >= a) on either side of the mode.  At or above it the tail is summed directly (stopped at `enough`, as in
// fisher_greater).  Below it the tail holds the mode and is taken as 1 - P(X <= a - 1), the upper tail of the mirrored
// table: summed from a, its first term can lie so far out that it underflows to 0, and the sum would be 0 instead of ~1.
template <bool kPreciseLog = false>
MS_HD double fisher_upper(uint32_t a, uint32_t b, uint32_t c, uint32_t d, double enough = 2.0) {
    if (fisher_at_or_above_mode(a, b, c, d)) return fisher_greater<kPreciseLog>(a, b, c, d, enough);
    return (a == 0 || d == 0) ? 1.0 : 1.0 - fisher_greater<kPreciseLog>(b + 1, a - 1, d - 1, c + 1);
}

// P(ref codon -> codon) for nm mismatching bases (restatement choice U1, SURVEY App. B)
inline void codon_error_table(double sub_rate, double del_rate, double out[4]) {
    const double match = 1.0 - sub_rate - del_rate, mis = sub_rate / 3.0;
    for (int nm = 0; nm < 4; ++nm) {
        double p = 1.0;
        for (int i = 0; i < 3 - nm; ++i) p *= match;
        for (int i = 0; i < nm; ++i) p *= mis;
        out[nm] = p;
    }
}

}  // namespace ms
