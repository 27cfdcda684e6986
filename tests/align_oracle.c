/* align_oracle.c -- CPU restatement of read alignment (restatement choice U16), the checker of align.cu.
 *
 * Written from the rule, not from the kernels: the seed window is found by sorting the diagonals and sweeping, the band
 * keeps whole anti-diagonals indexed by read position, and the traceback keeps every anti-diagonal's band start.  The
 * constants come from the header the kernels use.  mso_overlap_score is the same scoring over the full matrix, without a
 * band or seeds, for checking that the band follows the optimal path.                                                  */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include "../minorseq_b200/csrc/align_rule.h"

#define W MS_ALN_BAND
#define NEG MS_ALN_NEG

static int code(char c) { return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1; }
static int score(char x, char y) { return (code(x) >= 0 && code(x) == code(y)) ? MS_ALN_MATCH : MS_ALN_MISMATCH; }
static char comp(char c) { return c == 'A' ? 'T' : c == 'C' ? 'G' : c == 'G' ? 'C' : c == 'T' ? 'A' : 'N'; }

typedef struct { uint32_t kmer; int32_t t; } Entry;
typedef struct { const char* ref; int32_t lb; Entry* e; int64_t n; } mso_align_index;

static int cmp_entry(const void* a, const void* b) {
    const Entry *x = (const Entry*)a, *y = (const Entry*)b;
    if (x->kmer != y->kmer) return x->kmer < y->kmer ? -1 : 1;
    return x->t < y->t ? -1 : x->t > y->t;
}
static int cmp_int(const void* a, const void* b) {
    const int x = *(const int*)a, y = *(const int*)b;
    return x < y ? -1 : x > y;
}

static int kmer_at(const char* s, int32_t q, uint32_t* out) {
    uint32_t x = 0;
    for (int c = 0; c < MS_ALN_K; ++c) {
        const int v = code(s[q + c]);
        if (v < 0) return 0;
        x = (x << 2) | (uint32_t)v;
    }
    *out = x;
    return 1;
}

mso_align_index* mso_align_index_new(const char* ref, int32_t lb) {
    mso_align_index* ix = (mso_align_index*)calloc(1, sizeof(mso_align_index));
    Entry* all = (Entry*)malloc(sizeof(Entry) * (size_t)(lb + 1));
    int64_t n = 0, m = 0;
    for (int32_t t = 0; t + MS_ALN_K <= lb; ++t)
        if (kmer_at(ref, t, &all[n].kmer)) all[n++].t = t;
    qsort(all, (size_t)n, sizeof(Entry), cmp_entry);
    for (int64_t a = 0; a < n;) {
        int64_t e = a + 1;
        while (e < n && all[e].kmer == all[a].kmer) ++e;
        if (e == a + 1) all[m++] = all[a];
        a = e;
    }
    ix->ref = ref; ix->lb = lb; ix->e = all; ix->n = m;
    return ix;
}

void mso_align_index_free(mso_align_index* ix) {
    if (ix) { free(ix->e); free(ix); }
}

static int32_t find(const mso_align_index* ix, uint32_t kmer) {
    int64_t lo = 0, hi = ix->n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) / 2;
        if (ix->e[mid].kmer < kmer) lo = mid + 1; else hi = mid;
    }
    return lo < ix->n && ix->e[lo].kmer == kmer ? ix->e[lo].t : -1;
}

/* the strand's support and d0 (U16 "Seeds") */
static int32_t strand_support(const mso_align_index* ix, const char* s, int32_t la, int32_t* d0) {
    const int32_t npos = la >= MS_ALN_K ? (la - MS_ALN_K) / MS_ALN_STRIDE + 1 : 0;
    int* d = (int*)malloc(sizeof(int) * (size_t)(npos + 1));
    int* sorted = (int*)malloc(sizeof(int) * (size_t)(npos + 1));
    int n = 0;
    for (int32_t q = 0; q + MS_ALN_K <= la; q += MS_ALN_STRIDE) {
        uint32_t x;
        int32_t t;
        if (kmer_at(s, q, &x) && (t = find(ix, x)) >= 0) d[n++] = t - q;
    }
    memcpy(sorted, d, sizeof(int) * (size_t)n);
    qsort(sorted, (size_t)n, sizeof(int), cmp_int);
    int best = 0, top = 0;
    for (int hi = 0, lo = 0; hi < n; ++hi) {
        while (sorted[lo] < sorted[hi] - (MS_ALN_WINDOW - 1)) ++lo;
        if (hi - lo + 1 > best) { best = hi - lo + 1; top = sorted[hi]; }
    }
    for (int e = 0; e < n; ++e)
        if (d[e] <= top && d[e] >= top - (MS_ALN_WINDOW - 1)) { *d0 = d[e]; break; }
    free(d); free(sorted);
    return best;
}

static int32_t at(const int32_t* h, int32_t b, int32_t i) { return (i >= b && i < b + W) ? h[i - b] : NEG; }

/* One read, native orientation.  Returns 1 mapped, 0 unmapped, -1 when cap is too small (*ncigar = ops needed).
 * cigar: BAM-encoded ops of the aligned strand.                                                                      */
int mso_align_read(const mso_align_index* ix, const char* read, int32_t la, int32_t min_seeds, int32_t* strand, int32_t* pos,
                   int32_t* score_out, uint32_t* cigar, int32_t cap, int32_t* ncigar) {
    const char* ref = ix->ref;
    const int32_t lb = ix->lb;
    *strand = 0; *pos = -1; *score_out = 0; *ncigar = 0;
    char* rc = (char*)malloc((size_t)la + 1);
    for (int32_t x = 0; x < la; ++x) rc[x] = comp(read[la - 1 - x]);
    int32_t df = 0, dr = 0;
    const int32_t sf = strand_support(ix, read, la, &df), sr = strand_support(ix, rc, la, &dr);
    const int rev = sr > sf;
    if ((rev ? sr : sf) < min_seeds || (rev ? sr : sf) == 0) { free(rc); return 0; }
    const char* a = rev ? rc : read;
    const int32_t d0 = rev ? dr : df;
    const int32_t i0 = d0 >= 0 ? 0 : -d0, j0 = d0 >= 0 ? d0 : 0, k0 = i0 + j0;

    /* the band, anti-diagonal by anti-diagonal */
    const int64_t nad_max = (int64_t)la + lb + 2;
    uint8_t* mv = (uint8_t*)malloc((size_t)nad_max * W);
    int32_t* band = (int32_t*)malloc(sizeof(int32_t) * (size_t)nad_max);
    int32_t h1[W], h2[W], cur[W];
    int32_t b1 = 0, b2 = 0, b = i0 - W / 2;
    for (int p = 0; p < W; ++p) h1[p] = h2[p] = NEG;
    int32_t best = NEG, bk = 0, bi = 0;
    for (int32_t k = k0;; ++k) {
        const int64_t rel = k - k0;
        int any = 0;
        band[rel] = b;
        for (int p = 0; p < W; ++p) {
            const int32_t i = b + p, j = k - i;
            uint8_t m = 3;
            if (i < 0 || i > la || j < 0 || j > lb) cur[p] = NEG;
            else if (i == 0 || j == 0) { cur[p] = 0; any = 1; }
            else {
                any = 1;
                int32_t h = at(h2, b2, i - 1) + score(a[i - 1], ref[j - 1]);
                m = 0;
                if (at(h1, b1, i - 1) + MS_ALN_GAP > h) { h = at(h1, b1, i - 1) + MS_ALN_GAP; m = 1; }
                if (at(h1, b1, i) + MS_ALN_GAP > h) { h = at(h1, b1, i) + MS_ALN_GAP; m = 2; }
                cur[p] = h < NEG / 2 ? NEG : h;
            }
            mv[rel * W + p] = m;
            if (i >= 0 && i <= la && j >= 0 && j <= lb && (i == la || j == lb) && cur[p] > NEG / 2 && cur[p] > best) {
                best = cur[p]; bk = k; bi = i;
            }
        }
        if (!any) break;
        const int down = cur[W - 1] > cur[0];
        memcpy(h2, h1, sizeof h1); b2 = b1;
        memcpy(h1, cur, sizeof cur); b1 = b;
        b += down;
    }
    int ret = 0;
    if (best > NEG / 2) {
        /* walk back, collecting single ops from the end */
        uint8_t* ops = (uint8_t*)malloc((size_t)la + lb + 2);
        int64_t n = 0;
        int32_t i = bi, k = bk;
        while (i > 0 && k - i > 0) {
            const int32_t j = k - i;
            const uint8_t m = mv[(int64_t)(k - k0) * W + (i - band[k - k0])];
            if (m == 0) { ops[n++] = (code(a[i - 1]) >= 0 && code(a[i - 1]) == code(ref[j - 1])) ? 7 : 8; --i; k -= 2; }
            else if (m == 1) { ops[n++] = 1; --i; --k; }
            else { ops[n++] = 2; --k; }
        }
        /* run-length, forward order, with the overhangs */
        uint32_t* tmp = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)(n + 2));
        int32_t nc = 0;
        if (i > 0) tmp[nc++] = (uint32_t)i << 4 | 4u;
        for (int64_t x = n - 1; x >= 0; --x) {
            if (nc > 0 && (tmp[nc - 1] & 15u) == ops[x]) tmp[nc - 1] += 16u;
            else tmp[nc++] = 1u << 4 | ops[x];
        }
        if (la - bi > 0) tmp[nc++] = (uint32_t)(la - bi) << 4 | 4u;
        *ncigar = nc;
        *strand = rev; *pos = k - i; *score_out = best;
        if (nc <= cap) { memcpy(cigar, tmp, sizeof(uint32_t) * (size_t)nc); ret = 1; }
        else ret = -1;
        free(tmp); free(ops);
    }
    free(mv); free(band); free(rc);
    return ret;
}

/* The best overlap score over the full (la + 1) x (lb + 1) matrix: free start on row 0 and column 0, end on row la or column
 * lb, same scores.  No band, no seeds: the reference the band is checked against.                                       */
int32_t mso_overlap_score(const char* a, int32_t la, const char* ref, int32_t lb) {
    int32_t* prev = (int32_t*)calloc((size_t)lb + 1, sizeof(int32_t));
    int32_t* cur = (int32_t*)calloc((size_t)lb + 1, sizeof(int32_t));
    int32_t best = NEG;
    for (int32_t i = 0; i <= la; ++i) {
        for (int32_t j = 0; j <= lb; ++j) {
            if (i == 0 || j == 0) { cur[j] = 0; continue; }
            int32_t h = prev[j - 1] + score(a[i - 1], ref[j - 1]);
            if (prev[j] + MS_ALN_GAP > h) h = prev[j] + MS_ALN_GAP;
            if (cur[j - 1] + MS_ALN_GAP > h) h = cur[j - 1] + MS_ALN_GAP;
            cur[j] = h;
        }
        if (cur[lb] > best) best = cur[lb];
        if (i == la)
            for (int32_t j = 0; j <= lb; ++j) if (cur[j] > best) best = cur[j];
        int32_t* t = prev; prev = cur; cur = t;
    }
    free(prev); free(cur);
    return best;
}
