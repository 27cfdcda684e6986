/* align_rule.h -- the constants of read alignment (restatement choice U16, DESIGN.md "K6 read alignment"), shared by the
 * kernels (align.cu) and the CPU restatement the tests compare them with (tests/align_oracle.c).  Plain C.            */
#ifndef MS_ALIGN_RULE_H
#define MS_ALIGN_RULE_H

enum {
    MS_ALN_K = 15,            /* seed length: reference k-mers that are all ACGT and occur exactly once */
    MS_ALN_STRIDE = 4,        /* read positions q = 0 (mod 4) are looked up */
    MS_ALN_WINDOW = 65,       /* a strand's support: most hits whose diagonals fall in 65 consecutive diagonals */
    MS_ALN_BAND = 128,        /* W: band cells per anti-diagonal */
    MS_ALN_MATCH = 2,         /* U13's scores, shared with cleric */
    MS_ALN_MISMATCH = -3,
    MS_ALN_GAP = -4,
    MS_ALN_MAX_LEN = 65535,   /* longest read and longest reference */
    MS_ALN_MIN_SEEDS = 10,    /* default of --min-seeds */
    MS_ALN_CHUNK_READS = 131072,   /* ms_align_reads uploads at most this many reads ... */
    MS_ALN_CHUNK_MBASES = 256      /* ... and 2^20 times this many bases per chunk */
};

/* -infinity of the band: outside the matrix, outside the band, before the first anti-diagonal.  A cell whose best move
 * scores below MS_ALN_NEG / 2 is -infinity as well; no real score comes near it (|score| <= 3 * 2 * 65535).          */
#define MS_ALN_NEG (-(1 << 28))

#endif
