// handle.h -- internal state behind the opaque ms_handle of include/minorseq_b200.h
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/minorseq_b200.h"
#include <nvtx3/nvToolsExt.h>

// NVTX range over a stage of the path (decode / H2D / K1-K4 / exchanges, SURVEY.md 5): shows up in Nsight timelines, costs a
// few nanoseconds when no tool is attached
struct MsRange {
    explicit MsRange(const char* name) { nvtxRangePushA(name); }
    ~MsRange() { nvtxRangePop(); }
    MsRange(const MsRange&) = delete;
    MsRange& operator=(const MsRange&) = delete;
};

// grow-only device buffer: the hot path never pays cudaMalloc/cudaFree twice for the same size
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap && p) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        const size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

struct ms_handle {
    int device = 0;
    int num_sms = 0;
    int max_smem = 0;
    cudaStream_t own_stream = nullptr, copy_stream = nullptr, stream = nullptr;
    cudaEvent_t ev_copy[2] = {nullptr, nullptr};
    cudaEvent_t ev_chunk[16] = {};              // upload pipeline: one per in-flight chunk, reused round-robin
    cudaEvent_t ev_stagefree[2] = {};           // ms_pileup_host: staging buffer k has been permuted into tiles
    cudaEvent_t ev_k1[2] = {nullptr, nullptr};  // around the last K1 launch when timing is on
    cudaEvent_t ev_timer[2] = {nullptr, nullptr};  // ms_timer_start / ms_timer_stop
    int expand_ctas = 0, expand_ctas_nblk = -1;   // expand_events_kernel: resident CTAs per SM for row length nblk
    cudaEvent_t ev_stage[16][2] = {};              // when timing is on: around the last launch of MS_STAGE_* (ms_stage_kernel_ms)
    bool stage_seen[16] = {};
    bool timing = false;
    int64_t k1_reads = 0;
    std::string err;
    int64_t launches = 0;

    // layout
    int32_t L = 0, nblk = 0;
    bool count_codons = false;
    bool count_ins = false;  // with a codon layout, also tally insertion flags (kModeBoth)
    int variant = 0;
    uint32_t* d_counts = nullptr;  // [L*8 | L*64]
    uint32_t* d_start = nullptr;   // [nblk]
    uint2* d_pivot = nullptr;      // [nblk+1]
    uint8_t* d_pivot_state = nullptr;  // [nblk*32 + 2]
    uint2* d_pivot2 = nullptr;         // [nblk+1] designated base of the DENSE kernel (runner-up of the sample where frequent)
    uint8_t* d_pivot2_state = nullptr;
    uint32_t *d_part_col = nullptr, *d_part_piv = nullptr, *d_part_piv2 = nullptr;
    int32_t groups = 1, wpg = 1, stages = 2, stages_hi = 2, stage_bytes = 0, smem_bytes = 0, smem_bytes_hi = 0;
    int32_t nseg = 1, seg_len = 0;   // column segments of K1 (abi_core.cu, ms_set_layout)
    bool have_pivot = false;
    bool log_mode = false;       // K1 logs flagged chunks for codon_exception_kernel (dense start masks)
    // DENSE variant of K1 (a second bit-sliced codon count): picked once per layout from the pivot sample
    bool dense_known = false, dense = false;
    DevBuf b_exc_list, b_exc_cnt;  // K1's per-thread exception logs
    std::vector<uint32_t> h_start;

    // event rows (events.cu): base sequence planes, staging of the uploaded headers and events
    DevBuf b_base, b_ev_hdr, b_ev;
    uint32_t base_hash = 0;
    bool have_base = false;

    // host-upload staging (ms_pileup_host keeps the rows for phasing)
    uint32_t* d_upload = nullptr;               // tiles (rows.cuh)
    size_t upload_cap = 0;
    DevBuf b_rowstage[2];                       // plain rows of one upload chunk, before the permutation into tiles

    // call
    void* d_call_buf = nullptr;
    size_t call_cap = 0;
    void* call_stage = nullptr;   // pinned
    size_t call_stage_cap = 0;
    std::vector<uint8_t> call_pos_cache;
    size_t call_npos = 0;        // codon positions of the last ms_call_launch (sizes of its device buffers)

    // phasing (all buffers grow-only, reused across ms_phase_begin calls)
    int32_t V = 0, vwords = 0;
    int64_t phase_cap = 0, phase_n = 0;
    int32_t nblocklist = 0;
    int32_t phase_nrec = 0;          // words of phase_bits_kernel's variant stream
    bool phase_ordered = true;       // the stream visits the words of the bit-vector one after the other
    bool phase_partial_all = false;  // some variant lies outside the reference: every read is partial
    int64_t tab_size = 0, tab_size_max = 0, tab_hint = 0;
    int64_t gcap_hint = 0;       // distinct-pattern capacity the last ordering pass needed
    bool table_valid = false;
    int table_attempt = 0;
    DevBuf b_plan;   // PhasePlan built on the device by the single-call pass
    void* plan_stage = nullptr;   // pinned, sizeof(PhasePlan): its download
    uint32_t* counts_stage = nullptr; size_t counts_stage_words = 0;   // pinned: ms_get_counts goes through it (pageable destinations are slow)
    DevBuf b_var, b_blocklist, b_bits, b_flags, b_slot, b_tab_key, b_tab_cnt, b_tab_rep, b_ctr, b_groups, b_gather, b_rank, b_hap,
        b_pat, b_cooc, b_bits_t;
    // device-side merge + ordering (phase_order.cu)
    DevBuf b_gslot, b_mt_key, b_mt_cnt, b_mt_rep, b_mslot, b_mindex, b_m_cnt, b_m_pat, b_m_rank, b_ord, b_keys, b_out, b_tc_tiles;
    DevBuf b_nw_seq, b_nw_hrow, b_nw_hcol, b_nw_dir;   // nw.cu (cleric's reference-to-reference alignment)
    int32_t tc_tiles_V = -1;     // variant count the uploaded tcgen05 tile list belongs to
    int cooc_variant = 0;        // 0 auto, 1 popcount-AND, 2 tcgen05 int8
    // pairwise linkage (linkage.cu): ms_set_linkage before ms_phase_begin makes phase_bits_kernel also write the clean-codon
    // matrix b_mbits; the stacked Gram matrix of [B | M] is computed (and all-reduced) once per phased read set
    bool linkage = false;        // ms_set_linkage
    bool link_ready = false;     // b_mbits belongs to the current phased read set
    bool gram_valid = false;     // b_link_gram holds the (reduced) Gram matrix of the current read set
    std::vector<int32_t> link_col;   // start column of each variant of the current ms_phase_begin
    DevBuf b_mbits, b_link_gram, b_link_col, b_link_sig, b_link_rows, b_link_out;
    // haplotype abundance (abundance.cu): ms_set_abundance before ms_phase_begin records b_mbits as linkage does.  Per call: the
    // patterns, one compatibility mask per read and its EM flag, the class table, this rank's class list (exchanged block), the
    // ordered class list and the EM's state.  The merge and sort scratch of phase_order.cu (b_gather, b_mt_*, b_mslot, b_mindex,
    // b_m_*, b_ord, b_keys) is reused: it holds nothing between calls.
    bool abundance = false;      // ms_set_abundance
    DevBuf b_ab_pat, b_ab_mask, b_ab_flag, b_ab_slot, b_ab_tab_key, b_ab_tab_cnt, b_ab_tab_rep, b_ab_ctr, b_ab_blk, b_ab_out, b_ab_em;
    std::vector<uint32_t> groups_cnt, groups_pat;   // host copy of the last grouping pass (all ranks when a comm is attached)
    bool hap_ranked = false;     // b_rank maps the table slots of the current phased reads to the last ms_phase_haplotypes order
    bool hap_assigned = false;   // ... and b_hap holds the per-read positions in it (ms_phase_hap_device)
    uint64_t groups_marg[4] = {0, 0, 0, 0};
    bool groups_valid = false;
    void* h_stage = nullptr;      // pinned host staging for small D2H reads
    size_t h_stage_cap = 0;

    // cross-GPU exchange (comm.cu): ncclComm_t, NULL = single rank
    void* comm = nullptr;
    int world = 1, rank = 0;

    // fuse
    char* d_seq = nullptr;

    // grouped pile-up (group.cu): column counts [label_groups][L][8] of the reads of each label, and the counting sort's buffers
    int32_t label_groups = -1;   // ms_set_groups; -1 = not set
    int32_t label_L = 0;         // L of the layout the group counts belong to
    DevBuf b_gcol, b_ghist, b_gtot, b_goff, b_gioff, b_glist;

    // read alignment (align.cu): the reference and its seed hash table, then per chunk of reads their bases and offsets, seeds,
    // the seed kernel's hit scratch, the band kernel's move-bit slabs and band-move bits, CIGAR slots, results, packed CIGARs
    int32_t aln_L = -1, aln_bits = 0;   // reference length (-1 = none set), log2 of the hash table's size
    // in-frame indels (indel.cu): [L][2] k_del, n_ins | tally[sid] (one buffer: one all-reduce), the events, the call's buffer
    int32_t indel_L = 0;                  // L of the layout the counts belong to; 0 = none
    bool indel_reduced = false;           // the counts have been summed over the ranks
    std::vector<int32_t> indel_col;       // per string id: its column ...
    std::vector<std::string> indel_str;   // ... and its upper-cased string
    DevBuf b_indel_cnt, b_indel_ev, b_indel_out;

    DevBuf b_aln_ref, b_aln_idx, b_aln_seq, b_aln_off, b_aln_seed, b_aln_scratch, b_aln_slab, b_aln_mbits, b_aln_cig, b_aln_res, b_aln_ctr,
        b_aln_dst, b_aln_pack;
};

#define MS_CUDA(h, call)                                                                    \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                  \
            return MS_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

// bench.py's per-kernel rooflines: CUDA events on the handle's stream around the dominant kernel of a stage
#define MS_STAGE_BEGIN(h, s) do { if ((h)->timing) cudaEventRecord((h)->ev_stage[s][0], (h)->stream); } while (0)
#define MS_STAGE_END(h, s) do { if ((h)->timing) { cudaEventRecord((h)->ev_stage[s][1], (h)->stream); (h)->stage_seen[s] = true; } } while (0)

#define MS_FAIL(h, code, msg) \
    do {                      \
        (h)->err = (msg);     \
        return (code);        \
    } while (0)
