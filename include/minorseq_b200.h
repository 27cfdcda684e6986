/*
 * minorseq_b200.h -- C ABI of the B200-native juliet/fuse hot path.
 *
 * The reference (PacificBiosciences/minorseq) documents no library, plugin or
 * FFI interface: its only boundary is the process interface
 *     juliet [--config|-c X] [--region b-e] [--mode-phasing] [--min-perc p]
 *            [--max-perc p] [--drm-only] in.bam out.{json,html}
 *                                        (/root/reference/doc/JULIET.md:61-66,
 *                                         :121,:195,:270-271,:342-354,:370)
 *     fuse in.bam out.fasta              (/root/reference/doc/FUSE.md:22-32)
 * so this header IS the drop-in boundary a maintainer would bind: the juliet /
 * fuse mains (minorseq_b200/host/), bench.py and the tests all sit on top of
 * it.  Each entry point names the documented juliet/fuse behaviour it replaces.
 *
 * Conventions: plain C types only; every function returns MS_OK (0) or a
 * negative ms_status; ms_last_error(h) holds the text; no exceptions cross the
 * ABI; one handle per GPU (per rank); calls on one handle are serialised by the
 * caller; all device work is enqueued on the handle's stream.  There is NO CPU
 * fallback: ms_create fails when no sm_100 device is present.
 *
 * Packed read format ("planar 4-bit", L/2 bytes per read rounded up to 16 B):
 *   a read is ceil(L/32) blocks; block b is four consecutive u32 bit-planes
 *   P0,P1,P2,P3 (words 4b..4b+3); bit j of each plane is reference column
 *   32b+j.  (P0,P1,P2) = state bits 0,1,2:
 *       0=A 1=C 2=G 3=T 4='-' deletion 5='N' QV-filtered base 7=not spanned
 *   P3 = an insertion follows this column in this read.  Columns >= L in the
 *   last block are state 7.
 * Two arrangements of the same 16-byte blocks:
 *   plain rows (HOST side: ms_expand_cigar, ms_pack_states, ms_pileup_host, ms_encode_rows): rows are
 *     contiguous, read r starts at word r * ms_row_words(L);
 *   tiles (DEVICE side: everything that takes a device pointer to packed reads -- ms_pileup_dev, ms_phase_dev,
 *     ms_juliet_pass_dev, ms_synth_dev, ms_expand_events_dev): reads are grouped in tiles of 8 consecutive
 *     reads stored block-major; the 16-byte block b of read 8t+i is the uint4 at index
 *     (t * nblk + b) * 8 + (i ^ (b & 7)),  nblk = ceil(L/32).  A buffer holds ceil(R/8) whole tiles
 *     (ms_tiled_words); the slots of reads >= R in the last tile are never interpreted, and a pointer into the
 *     middle of a buffer must start at a tile (a multiple of 8 reads).  One 128-byte line thus serves one block
 *     of 8 reads (the phasing gather) and a column segment of a tile is contiguous (the pile-up's bulk copies).
 *     ms_pileup_host / the event expansion produce tiles themselves; ms_tile_rows(_dev) converts plain rows.
 */
#ifndef MINORSEQ_B200_H
#define MINORSEQ_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    MS_OK = 0,
    MS_ERR_ARG = -1,        /* bad argument / call order */
    MS_ERR_CUDA = -2,       /* CUDA runtime error, text in ms_last_error */
    MS_ERR_NODEVICE = -3,   /* no usable sm_100 GPU: there is no CPU fallback */
    MS_ERR_CAPACITY = -4,   /* caller buffer too small; required size reported */
    MS_ERR_FORMAT = -5      /* malformed input (e.g. CIGAR 'M', doc/JULIET.md:53) */
} ms_status;

enum { MS_A = 0, MS_C = 1, MS_G = 2, MS_T = 3, MS_DEL = 4, MS_N = 5, MS_UNCOV = 7 };
enum { MS_COL_INS = 6, MS_COL_COV = 7 };     /* col[j][6] insertion flags, col[j][7] = A+C+G+T+-+N */
enum { MS_FLAG_GAP = 1, MS_FLAG_HET = 2, MS_FLAG_PARTIAL = 4 };

typedef struct ms_handle ms_handle;

/* ---- format helpers (host only, no GPU work) -------------------------------- */
/* u32 words per packed read = 4*ceil(L/32). */
int32_t ms_row_words(int32_t L);
/* Read admission filter (doc/JULIET.md:58 "Reads that are not primary or supplementary
 * alignments, get ignored"): 1 = use the record, 0 = skip (BAM FLAG 0x4 unmapped, 0x100 secondary). */
int ms_read_admitted(uint32_t bam_flag);
/* one byte per column (bits0-2 state, bit3 insertion-follows) -> plain planar rows (host arrangement). */
int ms_pack_states(const uint8_t *states, int64_t R, int32_t L, uint32_t *packed);
int ms_unpack_states(const uint32_t *packed, int64_t R, int32_t L, uint8_t *states);
/* plain rows <-> device tiles (see the format note above).  ms_tiled_words = u32 words of a tile buffer for R reads. */
int64_t ms_tiled_words(int32_t L, int64_t R);
int ms_tile_rows(const uint32_t *rows, int64_t R, int32_t L, uint32_t *tiled /* ms_tiled_words(L,R) */);
int ms_untile_rows(const uint32_t *tiled, int64_t R, int32_t L, uint32_t *rows);
/* Replaces juliet/fuse's per-record CIGAR walk (doc/JULIET.md:49-58, doc/FUSE.md:13-15):
 * expands one aligned record into one packed row.  cigar = BAM-encoded ops
 * (len<<4|op); op 'M'(0) is rejected with MS_ERR_FORMAT ("cigar M is forbidden").
 * seq = one base per byte (ACGTN), qv_mask[i]!=0 turns base i into 'N'
 * (doc/JULIET.md:256-259), may be NULL.  Inserted strings are appended to the
 * caller's event arrays (ins_col/ins_off/ins_len/ins_pool) when non-NULL.       */
int ms_expand_cigar(const uint32_t *cigar, int32_t ncigar, int32_t pos,
                    const char *seq, const uint8_t *qv_mask, int32_t lseq,
                    int32_t L, uint32_t *row /* ms_row_words(L) */,
                    int32_t *ins_col, int64_t *ins_off, int32_t *ins_len,
                    int64_t ins_cap, int64_t *nins, char *ins_pool, int64_t pool_cap,
                    int64_t *pool_used);

/* ---- lifecycle --------------------------------------------------------------- */
int ms_create(int device, ms_handle **out);
void ms_destroy(ms_handle *h);
const char *ms_last_error(const ms_handle *h);   /* h == NULL: error of the last failed ms_create */
/* cudaStream_t to enqueue on (e.g. torch's current stream); NULL = the handle's own stream. */
int ms_set_stream(ms_handle *h, void *cuda_stream);
int ms_synchronize(ms_handle *h);
/* page-locked host memory for the packed rows handed to ms_pileup_host (NULL on failure) */
void *ms_alloc_pinned(size_t bytes);
void ms_free_pinned(void *p);
/* number of kernels this handle has launched so far (bench.py's gpu_launches) */
int64_t ms_launch_count(const ms_handle *h);
/* on: record CUDA events around each K1 launch on the handle's stream; ms_pileup_kernel_ms
 * then returns the device time of the most recent K1 kernel and the reads it processed
 * (bench.py's roofline.achieved).                                                     */
int ms_set_timing(ms_handle *h, int on);
/* CUDA-event stopwatch on the handle's stream: start records an event, stop records a second one,
 * waits for it and returns the device time between them in milliseconds.              */
int ms_timer_start(ms_handle *h);
int ms_timer_stop(ms_handle *h, double *ms);
int ms_pileup_kernel_ms(ms_handle *h, double *ms, int64_t *reads);
/* Same for the other measured kernels (most recent launch while timing was on; MS_ERR_ARG if none):
 * phase_bits_kernel, the co-occurrence kernel (popcount-AND or tcgen05), expand_events_kernel, and with a communicator
 * attached the two exchanges: the count all-reduce, and the haplotype-list all-gather + merge kernels.  Two spans of
 * the host-buffer pass (ms_juliet_pass_events_host) as well: MS_STAGE_UPLOAD = first to last host->device copy on the
 * copy stream, MS_STAGE_PASS = start of the pass to the arrival of its last result on the main stream.             */
/* Pairwise linkage adds two: MS_STAGE_LINKAGE_STATS = its statistics kernels (m, tests, row offsets), MS_STAGE_LINKAGE_ALLREDUCE
 * = the all-reduce of its Gram matrix; its contraction is timed as MS_STAGE_COOCCURRENCE.  MS_STAGE_GROUP_PILEUP = the
 * grouped pile-up kernel of ms_group_pileup_dev (without the counting sort in front of it).  Read alignment adds two:
 * MS_STAGE_ALIGN_SEED = align_seed_kernel, MS_STAGE_ALIGN_BAND = align_band_kernel (banded DP and traceback) of the last
 * chunk of ms_align_reads.  Haplotype abundance adds two: MS_STAGE_ABUNDANCE_COMPAT = abundance_compat_kernel,
 * MS_STAGE_ABUNDANCE_EM = the EM iterations (host checks included).  MS_STAGE_INDELS = indel_count_kernel of
 * ms_indel_count_dev.                                                                                                   */
enum { MS_STAGE_PHASE_BITS = 1, MS_STAGE_COOCCURRENCE = 2, MS_STAGE_EXPAND = 3, MS_STAGE_ALLREDUCE = 4, MS_STAGE_HAPMERGE = 5,
       MS_STAGE_UPLOAD = 6, MS_STAGE_PASS = 7, MS_STAGE_LINKAGE_STATS = 8, MS_STAGE_LINKAGE_ALLREDUCE = 9,
       MS_STAGE_GROUP_PILEUP = 10, MS_STAGE_ALIGN_SEED = 11, MS_STAGE_ALIGN_BAND = 12, MS_STAGE_ABUNDANCE_COMPAT = 13,
       MS_STAGE_ABUNDANCE_EM = 14, MS_STAGE_INDELS = 15 };
int ms_stage_kernel_ms(ms_handle *h, int stage, double *ms);

/* ---- K1: pileup (juliet "MSA counts", doc/JULIET.md:96-100; fuse doc/FUSE.md:17-20) -- */
/* Reference length and the columns where a codon of some configured gene starts
 * (bit j of word j/32; NULL = count no codons, i.e. fuse).  Zeroes the counts.
 * With a start mask the insertion flags are not tallied (col[j][6] stays 0: juliet
 * ignores insertions, doc/JULIET.md:26-27) unless ms_set_count_insertions(h, 1).  */
int ms_set_layout(ms_handle *h, int32_t L, const uint32_t *start_mask);
int ms_set_count_insertions(ms_handle *h, int on);
int ms_reset_counts(ms_handle *h);
/* Accumulate R device-resident packed reads (tiles) into the handle's count tensor.     */
int ms_pileup_dev(ms_handle *h, const uint32_t *d_packed, int64_t R);
/* device-resident plain rows -> tiles (d_tiled: ms_tiled_words(L,R) words; needs ms_set_layout) */
int ms_tile_rows_dev(ms_handle *h, const uint32_t *d_rows, int64_t R, uint32_t *d_tiled);
/* Same from host memory (plain rows, pinned recommended): chunked H2D copies, permuted into
 * tiles on the GPU and overlapped with the kernel.  If keep_dev != NULL it receives a device
 * pointer to the uploaded reads (tiles), owned by the handle and valid until the next
 * ms_pileup_host / ms_destroy, so ms_phase_dev can run without a second upload.          */
int ms_pileup_host(ms_handle *h, const uint32_t *h_packed, int64_t R, const uint32_t **keep_dev);
/* The count tensor [ col: L*8 u32 | codon: L*64 u32 ] in device memory, for the
 * caller's cross-GPU sum (one NCCL all-reduce; integer sums are order independent). */
int ms_counts_device(ms_handle *h, uint32_t **d_counts, int64_t *nwords);
/* Copy counts to host: col[L][8] = A,C,G,T,-,N,ins,coverage ; codon[L][64] indexed by
 * start column, codon = 16*b0+4*b1+b2, only reads whose codon is all A/C/G/T.    */
int ms_get_counts(ms_handle *h, uint32_t *col, uint32_t *codon);
/* selects the K1 implementation: 0 = bit-sliced carry-save kernel (default),
 * 1 = shared-memory-atomic histogram kernel (kept only as the ncu A/B baseline). */
int ms_set_pileup_variant(ms_handle *h, int variant);

/* ---- event rows: the compact host->device form of an aligned read ------------------------------
 * What juliet/fuse's per-record CIGAR walk (doc/JULIET.md:49-58, doc/FUSE.md:13-15) hands to the GPU when the
 * caller wants the PCIe link to carry events instead of whole rows: a CCS alignment is "the base sequence, except
 * at a few columns" (X / D / I ops and QV-filtered bases, :256-259).  Per read: its span [begin,end) and a byte string
 *   [nN: u16 little-endian] [N list: nN bytes] [rest list: 12-bit entries, entry k in bits [12k, 12k+12) of the rest]
 * (no bytes at all when the read equals the base on its whole span).  Both lists walk the columns from `begin`: an
 * entry's column = the previous entry's column + its delta.  N list, for the QV-filtered bases (two thirds of the
 * events of CCS data): one byte per entry, 0..254 = this column is 'N', 255 = move on by 255 columns.  Rest list:
 * entry = delta << 4 | nibble, delta 0..254 = this column holds nibble = state | insertion-follows << 3, delta 255 =
 * move on by 255 columns; n entries take ceil(1.5 n) bytes.  Spanned columns without an entry hold the base
 * sequence's base, columns outside the span are "not spanned"; no column appears twice.  hdr has R+1 entries: the
 * byte string of read r is events[hdr[r].ev_off .. hdr[r+1].ev_off); hdr[R] is the sentinel written by
 * ms_events_seal (total byte count + a hash of the base sequence; rows encoded against another base are rejected
 * with MS_ERR_FORMAT).  Reference length <= 65535.  The GPU rebuilds the packed reads (expand_events_kernel) and
 * K1/K3 run on them unchanged.  ~112 B per 3 kb read at CCS error rates (85 events, 60 of them 'N'), against
 * 1504 B for the plain row.                                                                                     */
typedef struct { uint32_t ev_off; uint16_t begin, end; } ms_read_hdr;
/* worst-case number of event BYTES of one read (every column in the rest list + skips + the count) */
int64_t ms_events_bound(int32_t L);
/* base: L bytes, one base (0..3) per reference column: the configured referenceSequence, or any sequence close to
 * the reads (the encoding is lossless for every base; a close one makes it short).                                */
int ms_encode_states(const uint8_t *states, int64_t R, int32_t L, const uint8_t *base,
                     ms_read_hdr *hdr /* R+1 */, uint8_t *events, int64_t cap /* bytes */, int64_t *nbytes);
int ms_encode_rows(const uint32_t *packed, int64_t R, int32_t L, const uint8_t *base,
                   ms_read_hdr *hdr /* R+1 */, uint8_t *events, int64_t cap /* bytes */, int64_t *nbytes);
/* Incremental form for a BAM loop (one ms_expand_cigar row at a time, e.g. per host thread): base_planes from
 * ms_base_planes (2*ceil(L/32) words); appends the row's event bytes at events[*nbytes...] and advances *nbytes;
 * fills *hdr (ev_off = the old *nbytes).  The caller seals the finished array with ms_events_seal.                */
int ms_base_planes(const uint8_t *base, int32_t L, uint32_t *planes);
int ms_encode_row(const uint32_t *row, int32_t L, const uint32_t *base_planes, ms_read_hdr *hdr,
                  uint8_t *events, int64_t cap /* bytes */, int64_t *nbytes);
int ms_events_seal(ms_read_hdr *hdr, int64_t R, int64_t nbytes, const uint8_t *base, int32_t L);
/* The handle's copy of the base sequence (after ms_set_layout, which forgets it). */
int ms_set_base(ms_handle *h, const uint8_t *base);
/* Device-resident event rows -> R packed reads at d_packed (tiles, ms_tiled_words(L,R) words).  */
int ms_expand_events_dev(ms_handle *h, const ms_read_hdr *d_hdr, const uint8_t *d_events, int64_t R,
                         uint32_t *d_packed);
/* ms_pileup_host for event rows: chunked H2D of the events, expansion and pile-up behind each chunk.
 * keep_dev as in ms_pileup_host (the expanded rows, for ms_phase_dev).                               */
int ms_pileup_events_host(ms_handle *h, const ms_read_hdr *hdr, const uint8_t *events, int64_t R,
                          const uint32_t **keep_dev);

/* ---- cross-GPU exchange (one process per GPU; SURVEY 8e) ---------------------------------
 * Rank 0 creates the 128-byte NCCL unique id, the caller hands it to every rank over its own
 * control channel, every rank attaches its handle.  world == 1 is a no-op.              */
int ms_comm_unique_id(char id[128]);
int ms_comm_init(ms_handle *h, const char id[128], int rank, int world);
int ms_comm_size(const ms_handle *h);
/* The path's one data-path collective: in-place integer sum of the count tensor over all
 * ranks (ncclAllReduce, uint32, sum), enqueued on the handle's stream between K1 and K2.
 * With a communicator attached, ms_phase_groups also all-gathers the ranks' compact
 * (pattern, count) lists and returns the concatenation and the summed marginals.        */
int ms_allreduce_counts(ms_handle *h);

/* ---- K2: per-codon minor-variant test (doc/JULIET.md:38-42) --------------------- */
typedef struct { int32_t begin, end; } ms_gene;   /* 1-based [begin,end), doc/JULIET.md:134-136 */
typedef struct {
    double substitution_rate, deletion_rate;   /* error model (restatement choice U1) */
    double alpha;                              /* call iff p * ntests < alpha */
    double min_perc, max_perc;                 /* --min-perc / --max-perc, < 0 = off */
    int32_t region_begin, region_end;          /* --region, 1-based [b,e); 0,0 = off */
} ms_call_params;
typedef struct {
    int32_t gene, codon_index, col, ref_codon, codon;
    uint32_t count, coverage, expected, ntests;
    double pvalue;                             /* uncorrected one-sided Fisher p (fp64) */
} ms_variant;
void ms_call_params_default(ms_call_params *p);
/* Runs on the handle's (all-reduced) counts.  refseq NULL or shorter than L =>
 * tested against the major codon (doc/JULIET.md:133-134).  Variants come back
 * sorted by (gene, col, codon).  *n receives the number found (may exceed cap). */
int ms_call(ms_handle *h, const ms_gene *genes, int32_t ngenes, const char *refseq,
            const ms_call_params *prm, ms_variant *out, int64_t cap, int64_t *n);

/* ---- K3: read-level phasing (--mode-phasing, doc/JULIET.md:192-211,:372-381) ----- */
typedef struct { uint64_t reported, insufficient, damaged, gaps, heteroduplex, partial; } ms_phase_counters;
/* Declare the pooled variant list (start column, codon) and the number of reads
 * this handle will phase; allocates the bit matrix and the grouping table.       */
int ms_phase_begin(ms_handle *h, const int32_t *var_col, const int32_t *var_codon, int32_t V,
                   int64_t max_reads);
/* Bit-vectors + damage flags for R more device-resident reads (tiles), appended.          */
int ms_phase_dev(ms_handle *h, const uint32_t *d_packed, int64_t R);
/* Distinct patterns of this handle's undamaged reads with their counts (in no particular
 * order; with a communicator attached, the concatenation over all ranks), and the damage
 * marginals.  *H may exceed cap: call again with a larger buffer (the pass is cached).  */
int ms_phase_groups(ms_handle *h, uint32_t *patterns /* cap*ceil(V/32) */, uint64_t *counts,
                    int64_t cap, int64_t *H, ms_phase_counters *ctr);
/* Host: (pattern,count) lists from all ranks -> equal patterns merged, then juliet's
 * haplotype order (count desc, then ascending words) in place; entries [0,*nreported)
 * have count >= min_reads; the unreported rest follows in the same order (left unsorted
 * when it exceeds 65536 entries); fills reported/insufficient of ctr.  Pure host logic. */
int ms_haplotype_order(uint32_t *patterns, uint64_t *counts, int64_t H, int32_t V,
                       int32_t min_reads, int64_t *Hmerged, int64_t *nreported,
                       ms_phase_counters *ctr);
void ms_haplotype_name(int64_t rank, char buf[3]);      /* [A-Z][a-z]? doc/JULIET.md:198 */
/* hap_id (host, one per phased read, in upload order): rank in ordered_patterns,
 * or -1 if damaged.                                                               */
int ms_phase_assign(ms_handle *h, const uint32_t *ordered_patterns, int64_t H, int32_t *hap_id);
/* Grouping, merge over ranks (with a communicator: one all-gather of the ranks' compact
 * lists, merged on the device), juliet's haplotype order (count desc, then ascending
 * words) and the per-read haplotype id in ONE call, without the full pattern list ever
 * leaving the GPU: patterns/counts receive the first min(cap,*H) haplotypes of the order,
 * *H the number of distinct patterns, *nreported how many have >= min_reads reads (they
 * come first), ctr all six read categories of doc/JULIET.md:372-381.  hap_id (host, one per
 * read phased on this handle, may be NULL): position in that order, -1 if damaged.
 * Same results as ms_phase_groups + ms_haplotype_order + ms_phase_assign.               */
int ms_phase_haplotypes(ms_handle *h, int32_t min_reads, uint32_t *patterns, uint64_t *counts,
                        int64_t cap, int64_t *H, int64_t *nreported, ms_phase_counters *ctr,
                        int32_t *hap_id);
/* Device pointers to the per-read results (R*ceil(V/32) words, R bytes).          */
int ms_phase_device(ms_handle *h, uint32_t **d_bits, uint8_t **d_flags, int64_t *R);
/* C[v][w] = #reads carrying both (V*V int32, device buffer owned by the handle).
 * Popcount-AND over the transposed bit matrix, or -- when the contraction is large (V >= 256 and
 * >= 32768 reads) -- u8 x u8 -> s32 tcgen05 MMA with the accumulator in tensor memory; same integers. */
int ms_cooccurrence(ms_handle *h, int32_t **d_C);
/* 0 = choose by size (default), 1 = popcount-AND kernel, 2 = tensor-core kernel (A/B measurements, tests) */
int ms_set_cooccurrence_variant(ms_handle *h, int32_t variant);

/* ---- pairwise variant linkage (restatement choice U14) ------------------------------------------
 * Do two called variants sit on the same genomes?  Unlike phasing, a read counts for a pair whenever its codons at
 * BOTH variants are clean (all three states A/C/G/T), whatever it holds elsewhere.  For the pooled phasing keys v < w
 * whose codons share no column (|col_v - col_w| >= 3) and with n >= min_reads informative reads, the 2x2 table
 *     a = both, b = v only, c = w only, d = neither   (a+b+c+d = n)
 * gives D' and r^2, and two one-sided Fisher tests: p_together = P(>= a carry both), p_apart = P(<= a carry both).
 * With m = the number of tested pairs (Bonferroni), a pair is "linked" if p_together * m < alpha and "exclusive" if
 * p_apart * m < alpha; only these significant pairs are listed.  Every rank computes the same list from the same,
 * all-reduced counts.                                                                                               */
typedef struct { double alpha; int32_t min_reads; } ms_linkage_params;
enum { MS_LINKED = 1, MS_EXCLUSIVE = 2 };
typedef struct {
    int32_t v, w;                               /* indices in the ms_phase_begin list, v < w */
    uint32_t both, v_only, w_only, neither;     /* the 2x2 table over the informative reads */
    double d_prime, r2;
    double pvalue;                              /* uncorrected one-sided Fisher p of the reported relation (fp64) */
    int32_t relation;                           /* MS_LINKED or MS_EXCLUSIVE */
} ms_linkage_pair;
/* alpha 0.01 (juliet's --alpha), min_reads 10 */
void ms_linkage_params_default(ms_linkage_params *p);
/* on: the next ms_phase_begin also allocates the clean-codon matrix and ms_phase_dev fills it (off by default). */
int ms_set_linkage(ms_handle *h, int on);
/* The significant pairs of the phased reads (with a communicator attached: of all ranks' reads), ordered by v, then w.
 * *n receives their number (may exceed cap: call again, the counts are cached until the next ms_phase_begin /
 * ms_phase_dev); *ntested the Bonferroni m.  A collective when a communicator is attached: every rank calls it.       */
int ms_linkage(ms_handle *h, const ms_linkage_params *prm, ms_linkage_pair *out, int64_t cap, int64_t *n,
               int64_t *ntested);
/* The (all-reduced) stacked Gram matrix [B | M]^T [B | M] in device memory, dim x dim int32 with dim = 64*ceil(V/32):
 * B = the phasing bits (rows 0..), M = the clean-codon bits (rows dim/2..).  So for variants v, w (h = dim/2):
 * both = G[v][w], v carried and w clean = G[v][h+w], n = G[h+v][h+w], diag(M^T M) = K2 coverage, diag(B^T B) = K2 count.
 * Owned by the handle; same caching and collective rule as ms_linkage.                                              */
int ms_linkage_device(ms_handle *h, int32_t **d_gram, int32_t *dim);

/* ---- haplotype abundance (restatement choice U18) ------------------------------------------------
 * Phasing counts a haplotype's reads among the reads that are clean at EVERY key; abundance also uses the damaged ones.
 * With B (read carries key v's codon) and M (key v's three columns are all A/C/G/T) as in linkage, read r is compatible
 * with pattern h iff B[r][v] == P[h][v] for every v with M[r][v] = 1; S_r = the patterns it is compatible with.  A read is
 * "incompatible" (S_r empty), "uninformative" (S_r = all H patterns, H >= 2), "unique" (|S_r| = 1) or "ambiguous".  The
 * unique and ambiguous reads (N of them) give the maximum-likelihood frequencies by EM: pi_h = 1/H to start, then
 *     pi'_h = (1/N) sum_r [h in S_r] pi_h / sum_{h' in S_r} pi_h'
 * until max_h |pi' - pi| < tolerance or max_iterations iterations.  Reads with the same S_r form a class; the classes are
 * merged over the ranks and totally ordered (count desc, then mask words asc), and the EM runs over them in that order with
 * fixed-order sums: the same bits on every run, rank and number of GPUs.                                                */
typedef struct { double tolerance; int32_t max_iterations; } ms_abundance_params;
typedef struct {
    uint64_t unique_reads;       /* reads with S_r = {h} */
    uint64_t compatible_reads;   /* reads with h in S_r */
    double em_frequency;         /* pi_h */
} ms_abundance_row;
typedef struct { uint64_t unique, ambiguous, uninformative, incompatible; } ms_abundance_counters;
/* tolerance 1e-10, max_iterations 10000 */
void ms_abundance_params_default(ms_abundance_params *p);
/* on: the next ms_phase_begin also allocates the clean-codon matrix and ms_phase_dev fills it (as ms_set_linkage). */
int ms_set_abundance(ms_handle *h, int on);
/* The abundance of H distinct patterns (rows of max(1, ceil(V/32)) words, as ms_phase_haplotypes returns them; bits >= V
 * are ignored; H <= 4096) over the phased reads (with a communicator attached: all ranks' reads; a collective, and every
 * rank passes the same patterns).  rows[h] in the order of the patterns; MS_ERR_CAPACITY when cap < H (nothing is
 * computed).  MS_ERR_ARG for duplicate patterns, H > 4096, or reads phased without ms_set_abundance / ms_set_linkage.
 * H = 0 or N = 0: no EM (pi = 1/H, *iterations 0, *converged 1).  *loglik = sum over the N reads of log sum_{h in S_r} pi_h. */
int ms_haplotype_abundance(ms_handle *h, const ms_abundance_params *prm, const uint32_t *patterns, int64_t H,
                           ms_abundance_row *rows, int64_t cap, ms_abundance_counters *counters, int32_t *iterations,
                           int32_t *converged, double *loglik);

/* ---- in-frame codon deletions and insertions (restatement choice U19) ------------------------------------------
 * The reads are the ones K1 piles up; codon starts are the layout's start mask, limited by the genes and the region as in
 * ms_call.  A read is "clean" at a column holding A/C/G/T.
 *   deletion of the codon at s:  k = reads with '-' at s, s+1 and s+2;  n = k + K2's coverage at s (reads with a clean codon);
 *   insertion at the boundary c = s+2 between the codons at s and s+3 of one gene (both tested):  n = reads clean at c and
 *   c+1;  k(x) = those of them whose FIRST insertion event at column c (ms_expand_cigar's ins_col) is the string x, of a
 *   length that is a multiple of 3 and >= 3, all A/C/G/T (upper-cased).  Other insertions stay in n and count for no x.
 * Test as K2: e = min(n, ceil(n P)) with P = deletion_rate^3 or insertion_rate^len(x), p = one-sided Fisher of
 * [[k, n-k], [e, n-e]], called iff p * ntests < alpha (ntests = the gene's tested codons, as K2), then min_perc / max_perc
 * on 100 k / n.  Needs the (all-reduced) K1 counts of the same reads.                                                 */
typedef struct {
    double deletion_rate, insertion_rate;      /* error model: P = deletion_rate^3, insertion_rate^len */
    double alpha;                              /* call iff p * ntests < alpha */
    double min_perc, max_perc;                 /* < 0 = off */
    int32_t region_begin, region_end;          /* 1-based [b,e); 0,0 = off */
} ms_indel_params;
enum { MS_INDEL_DELETION = 0, MS_INDEL_INSERTION = 1 };
typedef struct {
    int32_t gene, codon_index;                 /* the deleted codon / the codon before the insertion */
    int32_t col;                               /* deletion: its start column s; insertion: the column c = s+2 it follows */
    int32_t kind;                              /* MS_INDEL_DELETION or MS_INDEL_INSERTION */
    int32_t sid;                               /* insertion: string id (ms_indel_inserted); deletion: -1 */
    int32_t ref_codon;                         /* reference codon at s: referenceSequence, else the majority (-1: no clean read) */
    int32_t next_codon;                        /* insertion: the same at s+3; deletion: -1 */
    uint32_t count, coverage, expected, ntests;
    double pvalue;                             /* uncorrected one-sided Fisher p (fp64) */
} ms_indel;
/* deletion_rate 3e-3, insertion_rate 3e-3, alpha 0.01, no percentage filter, no region */
void ms_indel_params_default(ms_indel_params *p);
/* Counts R device-resident reads (tiles), which are reads [read0, read0 + R) of the caller's numbering, afresh: k_del and
 * n_ins of every column, and k(x).  The insertion events (ins_read in that numbering, ins_col, ins_off / ins_len into
 * ins_pool, in the order ms_expand_cigar appends them) are ALL the events of the run: the string ids are assigned from all of
 * them (one per (column, upper-cased x), in that order), so every rank that passes the same list gets the same ids; only the
 * events of this rank's reads are counted.                                                                              */
int ms_indel_count_dev(ms_handle *h, const uint32_t *d_packed, int64_t R, int64_t read0, const int64_t *ins_read,
                       const int32_t *ins_col, const int64_t *ins_off, const int32_t *ins_len, int64_t nins,
                       const char *ins_pool, int64_t pool_len);
/* Host copy of the counts: cnt[L][2] = k_del, n_ins; tally[sid] (the first min(cap, *nstrings)).  Summed over the ranks once
 * ms_indel_call has run.                                                                                               */
int ms_indel_counts(ms_handle *h, uint32_t *cnt, uint32_t *tally, int64_t cap, int64_t *nstrings);
/* The upper-cased string of id sid and its column (col may be NULL); MS_ERR_CAPACITY when cap < *len. */
int ms_indel_inserted(ms_handle *h, int32_t sid, int32_t *col, char *buf, int64_t cap, int64_t *len);
/* The called indels, sorted by (gene, codon, deletion before insertion, string).  *n receives their number; MS_ERR_CAPACITY
 * when it exceeds cap (out holds the first cap; call again, the counts are kept).  With a communicator attached a collective:
 * the first call after ms_indel_count_dev sums the counts over the ranks (one all-reduce), and every rank gets the same list. */
int ms_indel_call(ms_handle *h, const ms_gene *genes, int32_t ngenes, const char *refseq, const ms_indel_params *prm,
                  ms_indel *out, int64_t cap, int64_t *n);

/* ---- the whole juliet pass in one call ------------------------------------------------------
 * reset -> pileup -> (all-reduce when a communicator is attached) -> codon test -> phasing, i.e. everything
 * juliet does between BAM decode and report writing.  The caller owns the result buffers; on
 * MS_ERR_CAPACITY the n* fields hold the sizes needed.  patterns/counts receive the first
 * min(patterns_cap, npatterns) haplotypes of juliet's order, [0,nreported) being the reported ones (rows
 * ceil(nkeys/32) words apart; the buffer must hold patterns_cap * ceil(keys_cap/32) words); npatterns is the
 * number of distinct patterns, and only nreported > patterns_cap counts as too small.  key_col/key_codon is
 * the pooled variant list the bit-vectors refer to.  hap_id (host, R entries, may be NULL) as in
 * ms_phase_haplotypes.  Afterwards ms_get_counts / ms_cooccurrence can be called as usual.            */
typedef struct {
    ms_variant *variants;  int64_t variants_cap, nvariants;
    int32_t *key_col, *key_codon; int32_t keys_cap, nkeys;
    uint32_t *patterns; uint64_t *counts; int64_t patterns_cap, npatterns, nreported;
    ms_phase_counters counters;
    int32_t *hap_id;
} ms_juliet_result;
int ms_juliet_pass_dev(ms_handle *h, const uint32_t *d_packed, int64_t R, const ms_gene *genes, int32_t ngenes,
                       const char *refseq, const ms_call_params *prm, int32_t phase, int32_t min_hap_reads,
                       ms_juliet_result *out);
int ms_juliet_pass_host(ms_handle *h, const uint32_t *h_packed, int64_t R, const ms_gene *genes, int32_t ngenes,
                        const char *refseq, const ms_call_params *prm, int32_t phase, int32_t min_hap_reads,
                        ms_juliet_result *out);

/* The same pass from event rows in host memory (ms_pileup_events_host in place of ms_pileup_host): what the
 * bench.py's e2e calls -- the PCIe link carries ~112 B instead of 1504 B per 3 kb read.                       */
int ms_juliet_pass_events_host(ms_handle *h, const ms_read_hdr *hdr, const uint8_t *events, int64_t R,
                               const ms_gene *genes, int32_t ngenes, const char *refseq, const ms_call_params *prm,
                               int32_t phase, int32_t min_hap_reads, ms_juliet_result *out);

/* ---- K4: fuse consensus (doc/FUSE.md:17-24) --------------------------------------- */
typedef struct { int32_t min_coverage; double ins_fraction; int32_t ins_distance; } ms_fuse_params;
void ms_fuse_params_default(ms_fuse_params *p);
/* Consensus of the handle's (all-reduced) column counts plus the in-frame
 * insertion rule over the caller's insertion events.  *len may exceed cap.        */
int ms_fuse(ms_handle *h, const ms_fuse_params *prm,
            const int32_t *ins_col, const int64_t *ins_off, const int32_t *ins_len,
            int64_t nins, const char *ins_pool, int64_t pool_len,
            char *seq, int64_t cap, int64_t *len);

/* ---- grouped pile-up and per-group consensus (restatement choice U15) -------------------------------------------
 * What is the full sequence of each haplotype?  K1's column counts per group of reads: every read carries an int32 label
 * (device memory, one per read, in read order); a read labelled g in [0, ngroups) is counted into group g's columns, any
 * other label is skipped.  The group tensor is [ngroups][L][8] u32, each [L][8] laid out as ms_get_counts' col
 * (A,C,G,T,-,N,ins,coverage).  ms_set_groups allocates and zeroes it (after ms_set_layout; a new layout forgets it),
 * ms_group_pileup_dev accumulates R more device-resident reads (tiles) into it.                                      */
int ms_set_groups(ms_handle *h, int32_t ngroups);
int ms_group_pileup_dev(ms_handle *h, const uint32_t *d_packed, const int32_t *d_group, int64_t R);
/* In-place u32 sum of the group tensor over the ranks (ncclAllReduce); a collective, a no-op without a communicator. */
int ms_allreduce_group_counts(ms_handle *h);
int ms_get_group_counts(ms_handle *h, uint32_t *col /* ngroups*L*8 */);
/* Device pointer (owned by the handle) to the per-read position in juliet's haplotype order of the last ms_phase_haplotypes
 * (-1 = damaged; R = the reads phased on this handle), e.g. the labels of ms_group_pileup_dev.  Valid until the next phasing
 * call.  Computed here if ms_phase_haplotypes was called with hap_id == NULL.                                          */
int ms_phase_hap_device(ms_handle *h, int32_t **d_hap, int64_t *R);
/* fuse's consensus (U6-U8) of every group's (all-reduced) counts, with U15's one difference: inside the span from the first
 * to the last column with votes >= min_coverage, a column with fewer votes is written as 'N' instead of being dropped
 * (columns outside the span are trimmed).  Insertion events carry their group (ins_group; events of other groups are
 * skipped) and are tallied and judged against their own group's votes; only insertions after a column inside the span
 * are candidates.  Group g's sequence is seq[seq_off[g] .. seq_off[g+1]) (seq_off: ngroups + 1 entries, always filled);
 * MS_ERR_CAPACITY when cap < seq_off[ngroups] (seq may be NULL to query the size).                                     */
int ms_group_consensus(ms_handle *h, const ms_fuse_params *prm, const int32_t *ins_group, const int32_t *ins_col,
                       const int64_t *ins_off, const int32_t *ins_len, int64_t nins, const char *ins_pool, int64_t pool_len,
                       char *seq, int64_t cap, int64_t *seq_off);

/* ---- cleric's alignment step (doc/CLERIC.md:19-23,41-44; SURVEY 8f row 4) ------------------------
 * Global Needleman-Wunsch of the original reference a against the target reference b on the GPU
 * (tiled wavefront, N x M cells; match +2, mismatch -3, linear gap -4, ties diagonal > consume-a >
 * consume-b -- restatement choice U13).  ops receives the path in forward order: 'M' both advance,
 * 'D' only a advances (a base of a that b lacks), 'I' only b advances; cap must be >= la + lb.
 * The per-read CIGAR projection through this path is host code (minorseq_b200/host/cleric.hpp).   */
int ms_align_refs(ms_handle *h, const char *a, int32_t la, const char *b, int32_t lb,
                  char *ops, int64_t cap, int64_t *nops, int64_t *score);

/* ---- K6: read alignment (restatement choice U16; DESIGN.md "K6 read alignment") ---------------------------------
 * Overlap alignment of unaligned CCS reads to one amplicon reference: unique 15-mer seeds pick the strand and a start
 * diagonal, then a 128-cell adaptive band (Suzuki & Kasahara) with U13's scores (match +2, mismatch -3, linear gap -4)
 * finds the best path from the top or left edge to the bottom or right edge.  Reads and references are at most 65535
 * bases.  A read is its native sequence (the caller reverse-complements a BAM record with flag 0x10 first).
 * ms_align_set_reference builds the seed index (host) and uploads it with the reference; it stays until the next call. */
typedef struct { int32_t min_seeds; } ms_align_params;    /* the winning strand's seed support must reach min_seeds (>= 1) */
typedef struct {
    int32_t mapped;        /* 0: no strand reached min_seeds; the other fields are strand 0, pos -1, score 0, no CIGAR */
    int32_t strand;        /* 1: the reverse complement of the read was aligned (BAM flag 0x10) */
    int32_t pos;           /* 0-based reference position of the first aligned base */
    int32_t score;         /* the alignment's score (AS:i) */
    int64_t cigar_off;     /* first op in the caller's cigar array */
    int32_t ncigar;        /* ops: BAM-encoded len << 4 | op, only S = X I D, in the aligned strand's orientation */
} ms_read_alignment;
void ms_align_params_default(ms_align_params *p);    /* min_seeds 10 */
int ms_align_set_reference(ms_handle *h, const char *ref, int32_t L);
/* R reads, read r = seq[off[r] .. off[r+1]) (off: R + 1 entries).  out: R entries, in read order.  *ncigar receives the
 * total number of ops; MS_ERR_CAPACITY when it exceeds cap (out is filled all the same; call again with a larger cigar). */
int ms_align_reads(ms_handle *h, const ms_align_params *prm, const char *seq, const int64_t *off, int64_t R,
                   ms_read_alignment *out, uint32_t *cigar, int64_t cap, int64_t *ncigar);

/* ---- synthetic amplicon generator (bench/tests; SURVEY 8d) ------------------------- */
typedef struct {
    uint64_t seed;
    int32_t L, nstrains;
    uint32_t thr_N, thr_sub, thr_ins20, thr_trunc16;  /* integer thresholds, see synth.py */
} ms_synth_params;
/* strain_base: nstrains*L bytes (0..3); thr_del: L u32; strain_cum: nstrains u32 cumulative
 * mixture thresholds.  Writes R packed reads (tiles, ms_tiled_words(L,R) words) for reads [read0, read0+R) on the device.  */
int ms_synth_dev(ms_handle *h, const ms_synth_params *p, const uint8_t *strain_base,
                 const uint32_t *thr_del, const uint32_t *strain_cum,
                 int64_t read0, int64_t R, uint32_t *d_packed);

#ifdef __cplusplus
}
#endif
#endif
