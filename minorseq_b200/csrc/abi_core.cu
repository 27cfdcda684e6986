// abi_core.cu -- lifecycle, layout and the K1 launchers of the C ABI (include/minorseq_b200.h).
#include <algorithm>
#include <cstring>
#include <cstdlib>
#include "handle.h"
#include "pileup.cuh"
#include "rows.cuh"

static std::string g_create_error;
void ms_events_set_smem_attr(int max_smem);
void ms_cooc_tc_set_smem_attr();
void ms_phase_set_smem_attr();
void ms_group_set_smem_attr();
void ms_indel_set_smem_attr();
int ms_tile_rows_launch(ms_handle* h, const uint32_t* d_rows, int64_t R, uint32_t* d_tiled);

extern "C" {

int ms_create(int device, ms_handle** out) {
    if (!out) return MS_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0 || device < 0 || device >= ndev) {
        g_create_error = std::string("no usable CUDA device (") + (e != cudaSuccess ? cudaGetErrorString(e) : "index out of range") +
                         "); minorseq_b200 has no CPU fallback";
        return MS_ERR_NODEVICE;
    }
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        g_create_error = cudaGetErrorString(e);
        return MS_ERR_CUDA;
    }
    if (prop.major != 10) {
        g_create_error = "device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                         ", this library is built for sm_100a only";
        return MS_ERR_NODEVICE;
    }
    ms_handle* h = new ms_handle();
    h->device = device;
    h->num_sms = prop.multiProcessorCount;
    h->max_smem = static_cast<int>(prop.sharedMemPerBlockOptin);
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_copy[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_copy[1], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&h->ev_k1[0]) != cudaSuccess || cudaEventCreate(&h->ev_k1[1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_timer[0]) != cudaSuccess || cudaEventCreate(&h->ev_timer[1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[1][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[1][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[2][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[2][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[3][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[3][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[4][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[4][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[5][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[5][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[6][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[6][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[7][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[7][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[8][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[8][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[9][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[9][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[10][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[10][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[11][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[11][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[12][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[12][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[13][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[13][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[14][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[14][1]) != cudaSuccess ||
        cudaEventCreate(&h->ev_stage[15][0]) != cudaSuccess || cudaEventCreate(&h->ev_stage[15][1]) != cudaSuccess) {
        g_create_error = cudaGetErrorString(cudaGetLastError());
        delete h;
        return MS_ERR_CUDA;
    }
    for (cudaEvent_t& ev : h->ev_stagefree)
        if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
            g_create_error = cudaGetErrorString(cudaGetLastError());
            delete h;
            return MS_ERR_CUDA;
        }
    for (cudaEvent_t& ev : h->ev_chunk)
        if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
            g_create_error = cudaGetErrorString(cudaGetLastError());
            delete h;
            return MS_ERR_CUDA;
        }
    h->stream = h->own_stream;
    ms::pileup_set_smem_attr(h->max_smem);
    ms_events_set_smem_attr(h->max_smem);
    ms_cooc_tc_set_smem_attr();
    ms_phase_set_smem_attr();
    ms_group_set_smem_attr();
    ms_indel_set_smem_attr();
    *out = h;
    return MS_OK;
}

static void free_layout(ms_handle* h) {
    cudaFree(h->d_counts); cudaFree(h->d_start); cudaFree(h->d_pivot); cudaFree(h->d_pivot_state);
    cudaFree(h->d_pivot2); cudaFree(h->d_pivot2_state);
    cudaFree(h->d_part_col); cudaFree(h->d_part_piv); cudaFree(h->d_part_piv2);
    h->d_counts = nullptr; h->d_start = nullptr; h->d_pivot = nullptr; h->d_pivot_state = nullptr;
    h->d_pivot2 = nullptr; h->d_pivot2_state = nullptr;
    h->d_part_col = h->d_part_piv = h->d_part_piv2 = nullptr;
}

void ms_phase_free_internal(ms_handle* h);
void ms_comm_free_internal(ms_handle* h);

void ms_destroy(ms_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    ms_comm_free_internal(h);
    free_layout(h);
    ms_phase_free_internal(h);
    cudaFree(h->d_upload); cudaFree(h->d_call_buf); cudaFree(h->d_seq);
    h->b_exc_list.release(); h->b_exc_cnt.release();
    h->b_base.release(); h->b_ev_hdr.release(); h->b_ev.release();
    for (DevBuf* b : {&h->b_gcol, &h->b_ghist, &h->b_gtot, &h->b_goff, &h->b_gioff, &h->b_glist}) b->release();
    for (DevBuf* b : {&h->b_aln_ref, &h->b_aln_idx, &h->b_aln_seq, &h->b_aln_off, &h->b_aln_seed, &h->b_aln_scratch, &h->b_aln_slab,
                      &h->b_aln_mbits, &h->b_aln_cig, &h->b_aln_res, &h->b_aln_ctr, &h->b_aln_dst, &h->b_aln_pack})
        b->release();
    for (cudaEvent_t ev : h->ev_chunk) cudaEventDestroy(ev);
    for (cudaEvent_t ev : h->ev_stagefree) cudaEventDestroy(ev);
    h->b_rowstage[0].release(); h->b_rowstage[1].release();
    if (h->call_stage) cudaFreeHost(h->call_stage);
    if (h->counts_stage) cudaFreeHost(h->counts_stage);
    cudaEventDestroy(h->ev_copy[0]); cudaEventDestroy(h->ev_copy[1]);
    cudaEventDestroy(h->ev_k1[0]); cudaEventDestroy(h->ev_k1[1]);
    cudaEventDestroy(h->ev_timer[0]); cudaEventDestroy(h->ev_timer[1]);
    for (DevBuf* b : {&h->b_ab_pat, &h->b_ab_mask, &h->b_ab_flag, &h->b_ab_slot, &h->b_ab_tab_key, &h->b_ab_tab_cnt, &h->b_ab_tab_rep, &h->b_ab_ctr,
                      &h->b_ab_blk, &h->b_ab_out, &h->b_ab_em, &h->b_indel_cnt, &h->b_indel_ev, &h->b_indel_out,
                      &h->b_rare_pos, &h->b_rare_out, &h->b_rare_pairs, &h->b_rare_sup, &h->b_control, &h->b_control_pos, &h->b_control_out})
        b->release();
    for (int s = 1; s < 16; ++s) { cudaEventDestroy(h->ev_stage[s][0]); cudaEventDestroy(h->ev_stage[s][1]); }
    cudaStreamDestroy(h->own_stream); cudaStreamDestroy(h->copy_stream);
    delete h;
}

const char* ms_last_error(const ms_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int ms_set_stream(ms_handle* h, void* s) {
    if (!h) return MS_ERR_ARG;
    h->stream = s ? static_cast<cudaStream_t>(s) : h->own_stream;
    return MS_OK;
}

int ms_synchronize(ms_handle* h) {
    if (!h) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    return MS_OK;
}

int64_t ms_launch_count(const ms_handle* h) { return h ? h->launches : 0; }

void* ms_alloc_pinned(size_t bytes) {
    void* p = nullptr;
    return cudaMallocHost(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr;
}

void ms_free_pinned(void* p) {
    if (p) cudaFreeHost(p);
}

int ms_timer_start(ms_handle* h) {
    if (!h) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, cudaEventRecord(h->ev_timer[0], h->stream));
    return MS_OK;
}

int ms_timer_stop(ms_handle* h, double* ms) {
    if (!h || !ms) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, cudaEventRecord(h->ev_timer[1], h->stream));
    MS_CUDA(h, cudaEventSynchronize(h->ev_timer[1]));
    float f = 0.f;
    MS_CUDA(h, cudaEventElapsedTime(&f, h->ev_timer[0], h->ev_timer[1]));
    *ms = f;
    return MS_OK;
}

int ms_set_timing(ms_handle* h, int on) {
    if (!h) return MS_ERR_ARG;
    h->timing = on != 0;
    return MS_OK;
}

int ms_pileup_kernel_ms(ms_handle* h, double* ms, int64_t* reads) {
    if (!h || !ms || !h->timing) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, cudaEventSynchronize(h->ev_k1[1]));
    float f = 0.f;
    MS_CUDA(h, cudaEventElapsedTime(&f, h->ev_k1[0], h->ev_k1[1]));
    *ms = f;
    if (reads) *reads = h->k1_reads;
    return MS_OK;
}

int ms_stage_kernel_ms(ms_handle* h, int stage, double* ms) {
    if (!h || !ms || stage < 1 || stage > 15 || !h->timing || !h->stage_seen[stage]) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, cudaEventSynchronize(h->ev_stage[stage][1]));
    float f = 0.f;
    MS_CUDA(h, cudaEventElapsedTime(&f, h->ev_stage[stage][0], h->ev_stage[stage][1]));
    *ms = f;
    return MS_OK;
}

int ms_set_count_insertions(ms_handle* h, int on) {
    if (!h) return MS_ERR_ARG;
    h->count_ins = on != 0;
    return MS_OK;
}

int ms_set_pileup_variant(ms_handle* h, int variant) {
    if (!h || variant < 0 || variant > 1) return MS_ERR_ARG;
    h->variant = variant;
    return MS_OK;
}

int ms_set_layout(ms_handle* h, int32_t L, const uint32_t* start_mask) {
    if (!h || L < 3) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    h->indel_L = 0;   // the indel counts belong to the old layout
    h->control_valid = false;   // and so does a captured control
    const int32_t nblk = (L + 31) / 32;
    // CTA shape.  W warps span a row or a column segment of it (31 counting lanes per warp -- lane 31 is the codon
    // look-ahead provider -- and 32 in the last), G row-groups per CTA with W*G <= 12.  With nseg > 1 CTA c handles
    // segment c % nseg of its tiles, every segment but the last carrying one look-ahead block of the next.  In the tile
    // layout (rows.cuh) a segment of a tile is as contiguous as a whole tile -- one bulk copy per chunk either way -- so
    // the shape is picked for lane occupancy alone: counting blocks per CTA step out of the 12 x 32 lanes, discounted by
    // the imbalance when nseg does not divide the CTA count.  3 kb: whole rows (3 warps x 4 groups, 98 %); 9.7 kb: five
    // segments of 61 blocks (2 x 6, 95 %) instead of one 10-warp row (79 %); 6 kb: two of 96 (4 x 3, 75 %).
    static const int kGroups[13] = {0, 12, 6, 4, 3, 2, 2, 1, 1, 1, 1, 1, 1};
    const int budget = h->max_smem - ms::kPileupSmemHeaderHi - 16;     // shapes must fit the HI instantiation as well
    const int forced = getenv("MS_K1_NSEG") ? atoi(getenv("MS_K1_NSEG")) : 0;   // tuning knob (tools/k1_segments.py)
    auto shape = [&](int nseg, int& W, int& need) {
        const int seg_len = (nblk + nseg - 1) / nseg;
        if (nseg > 1 && seg_len * (nseg - 1) >= nblk) return false;        // an empty last segment
        need = seg_len + (nseg > 1 ? 1 : 0);
        W = need <= 32 ? 1 : 1 + (need - 32 + 30) / 31;
        return W <= 12 && budget / (kGroups[W] * need * 128) >= 3;        // the ring needs three slots per row-group
    };
    int best_nseg = 0, best_W = 0;
    {
        double best_score = 0.0;
        for (int nseg = 1; nseg <= 64; ++nseg) {
            int Wn = 0, nn = 0;
            if (forced > 0 && nseg != forced) continue;
            if (!shape(nseg, Wn, nn)) continue;
            const int ctas = std::max(h->num_sms, nseg);
            const double balance = static_cast<double>(ctas / nseg) * nseg / ctas;     // segments with one CTA fewer set the pace
            double score = static_cast<double>(kGroups[Wn]) * nblk / nseg / 384.0 * balance;
            if (nseg == 1) score *= 1.04;                                               // whole rows: no look-ahead block read twice
            if (score > best_score) { best_score = score; best_nseg = nseg; best_W = Wn; }
        }
    }
    if (best_nseg == 0) MS_FAIL(h, MS_ERR_ARG, "reference too long for this build's pile-up kernel");
    const int32_t W = best_W;
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    free_layout(h);
    h->label_groups = -1;   // group counts belong to the old layout
    h->b_gcol.release();
    h->L = L; h->nblk = nblk; h->count_codons = start_mask != nullptr; h->have_pivot = false;
    h->have_base = false;
    h->wpg = W;
    h->groups = kGroups[W];
    h->nseg = best_nseg;
    h->seg_len = (nblk + best_nseg - 1) / best_nseg;
    const int row_bytes = (h->seg_len + (best_nseg > 1 ? 1 : 0)) * 16;   // bytes of one read in a ring slot
    h->stage_bytes = h->groups * 8 * row_bytes;                          // one tile (segment) per row-group
    // Clean non-pivot codons: with one reading frame they are resolved inside K1 from the shared-memory slot; where reading
    // frames overlap every substituted base makes up to three of them, and it is cheaper to log the flagged 8-read chunks per
    // thread and resolve them afterwards in codon_exception_kernel (1M x 3 kb: 1 frame K1 0.386 vs 0.351 + 0.09 ms for the
    // exception kernel; 1M x 9.7 kb with HIV's 15 genes: K1 1.40 vs 1.14 ms and a step of 1.69 vs 1.66 ms; three full-length
    // frames: 0.59 vs 0.42 + 0.07 ms).  Logged as soon as more than 0.5 % of the columns start codons of overlapping frames
    // (HIV's genes: 1.6 %).
    int64_t nstarts = 0, noverlap = 0;
    if (start_mask) {
        auto is_start = [&](int32_t j) { return j + 2 < L && ((start_mask[j >> 5] >> (j & 31)) & 1u) != 0; };
        for (int32_t j = 0; j + 2 < L; ++j) {
            if (!is_start(j)) continue;
            ++nstarts;
            if (is_start(j + 1) || is_start(j + 2)) ++noverlap;
        }
    }
    h->log_mode = start_mask != nullptr && (nstarts * 20 > static_cast<int64_t>(L) * 9 || noverlap * 200 > static_cast<int64_t>(L));
    if (const char* e = getenv("MS_K1_LOG")) h->log_mode = start_mask != nullptr && atoi(e) != 0;   // tuning knob (A/B runs)
    const int merge_bytes = (h->groups - 1) * 9 * ms::kPlanesAll * W * 32 * 4 + 64;  // end-of-kernel group merge reuses the ring (up to 9 masks)
    h->stages = std::max(3, std::min(8, (h->max_smem - ms::kPileupSmemHeader - 16) / h->stage_bytes));
    h->stages_hi = std::max(3, std::min(8, budget / h->stage_bytes));
    h->smem_bytes = ms::kPileupSmemHeader + std::max(h->stages * h->stage_bytes + 16, merge_bytes);
    h->smem_bytes_hi = ms::kPileupSmemHeaderHi + std::max(h->stages_hi * h->stage_bytes + 16, merge_bytes);
    // DENSE variant (pileup.cu, read_masks): a second bit-sliced codon count per start column; chosen at the first pile-up
    // after this call from the pivot sample's statistics
    h->dense_known = false; h->dense = false;
    if (h->smem_bytes > h->max_smem || h->smem_bytes_hi > h->max_smem) MS_FAIL(h, MS_ERR_ARG, "row too long for the shared-memory ring");
    const size_t ncounts = static_cast<size_t>(L) * 72;
    MS_CUDA(h, cudaMalloc(&h->d_counts, ncounts * 4));
    MS_CUDA(h, cudaMemsetAsync(h->d_counts, 0, ncounts * 4, h->stream));
    MS_CUDA(h, cudaMalloc(&h->d_start, nblk * 4));
    MS_CUDA(h, cudaMalloc(&h->d_pivot, (nblk + 1) * sizeof(uint2)));
    MS_CUDA(h, cudaMalloc(&h->d_pivot_state, nblk * 32 + 16));   // + {non-pivot, all} sample statistics behind the states
    MS_CUDA(h, cudaMalloc(&h->d_pivot2, (nblk + 1) * sizeof(uint2)));
    MS_CUDA(h, cudaMalloc(&h->d_pivot2_state, nblk * 32 + 16));
    MS_CUDA(h, cudaMemsetAsync(h->d_pivot, 0, (nblk + 1) * sizeof(uint2), h->stream));
    MS_CUDA(h, cudaMemsetAsync(h->d_pivot2, 0, (nblk + 1) * sizeof(uint2), h->stream));
    MS_CUDA(h, cudaMemsetAsync(h->d_pivot2_state, 0, nblk * 32 + 16, h->stream));
    MS_CUDA(h, cudaMemsetAsync(h->d_pivot_state, 0, nblk * 32 + 16, h->stream));
    h->h_start.assign(nblk, 0u);
    if (start_mask) {
        for (int32_t b = 0; b < nblk; ++b) h->h_start[b] = start_mask[b];
        // a codon must fit inside the reference
        for (int32_t j = std::max(0, L - 2); j < nblk * 32; ++j) h->h_start[j >> 5] &= ~(1u << (j & 31));
    }
    MS_CUDA(h, cudaMemcpyAsync(h->d_start, h->h_start.data(), nblk * 4, cudaMemcpyHostToDevice, h->stream));
    const size_t slices = static_cast<size_t>(h->num_sms);
    MS_CUDA(h, cudaMalloc(&h->d_part_col, slices * nblk * 256 * 4));
    MS_CUDA(h, cudaMalloc(&h->d_part_piv, slices * nblk * 32 * 4));
    MS_CUDA(h, cudaMalloc(&h->d_part_piv2, slices * nblk * 32 * 4));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    return MS_OK;
}

int ms_reset_counts(ms_handle* h) {
    if (!h || !h->d_counts) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, cudaMemsetAsync(h->d_counts, 0, static_cast<size_t>(h->L) * 72 * 4, h->stream));
    h->have_pivot = false;
    return MS_OK;
}

int ms_pileup_dev(ms_handle* h, const uint32_t* d_packed, int64_t R) {
    MsRange nvtx_range("K1 pileup");
    if (!h || !h->d_counts || R < 0 || (R > 0 && !d_packed)) return MS_ERR_ARG;
    if (R == 0) return MS_OK;
    MS_CUDA(h, cudaSetDevice(h->device));
    uint32_t* col = h->d_counts;
    uint32_t* codon = h->d_counts + static_cast<size_t>(h->L) * 8;
    if (h->variant == 1) {
        dim3 grid(std::max(1, std::min<int>(static_cast<int>((R + 255) / 256), 4 * h->num_sms / std::max(1, h->nblk / 8 + 1) + 1)),
                  h->nblk);
        ms::pileup_atomic_kernel<<<grid, 256, 256 * 4, h->stream>>>(d_packed, R, h->L, h->nblk, h->d_start, col, codon,
                                                                   h->count_codons ? 1 : 0);
        ms::coverage_kernel<<<(h->L + 255) / 256, 256, 0, h->stream>>>(col, h->L);
        h->launches += 2;
        MS_CUDA(h, cudaGetLastError());
        return MS_OK;
    }
    if (h->count_codons && !h->have_pivot) {
        const bool want_stat = !h->dense_known;
        uint32_t* dense_stat = reinterpret_cast<uint32_t*>(h->d_pivot_state + static_cast<size_t>(h->nblk) * 32 + 8);
        if (want_stat) MS_CUDA(h, cudaMemsetAsync(dense_stat, 0, 8, h->stream));
        ms::pivot_sample_kernel<<<h->nblk, 256, 0, h->stream>>>(d_packed, R, h->nblk, h->L, h->d_pivot, h->d_pivot_state,
                                                               h->d_pivot2, h->d_pivot2_state, want_stat ? dense_stat : nullptr);
        if (want_stat) {
            // once per layout: are non-pivot bases the exception (sequencing errors, low-frequency variants) or the rule
            // (dense high-frequency variants, > 2 % of the sampled clean bases)?  One 8-byte read decides which K1 runs.
            uint32_t st[2] = {0, 0};
            MS_CUDA(h, cudaMemcpyAsync(st, dense_stat, 8, cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
            h->dense = static_cast<uint64_t>(st[0]) * 50u > st[1];
            h->dense_known = true;
        }
        h->launches++;
        h->have_pivot = true;
    }
    ms::PileupArgs a;
    a.packed = d_packed; a.R = R; a.L = h->L; a.nblk = h->nblk;
    a.warps_per_group = h->wpg; a.groups = h->groups;
    a.nseg = h->nseg; a.seg_len = h->seg_len;
    const bool dense = h->count_codons && h->dense;
    a.stages = h->stages; a.stages_hi = h->stages_hi; a.stage_bytes = h->stage_bytes;
    a.pivot = h->d_pivot; a.pivot2 = h->d_pivot2; a.start_mask = h->d_start; a.codon = codon;
    a.part_col = h->d_part_col; a.part_piv = h->d_part_piv; a.part_piv2 = h->d_part_piv2;
    const int mode = !h->count_codons ? ms::kModeFuse : (h->count_ins ? ms::kModeBoth : ms::kModeJuliet);
    const int64_t T = static_cast<int64_t>(h->groups) * 8;
    const int64_t ntiles = (R + T - 1) / T;
    const int grid = static_cast<int>(std::min<int64_t>(h->num_sms, ntiles * h->nseg));   // >= nseg: every segment has a CTA
    const int threads = h->wpg * h->groups * 32;
    if (R > (1LL << 27)) MS_FAIL(h, MS_ERR_ARG, "more than 2^27 reads in one ms_pileup_dev call: split the batch");
    // decided with the layout (ms_set_layout); the DENSE instantiation always logs (its exact trigger leaves few entries, and it
    // has no registers to spare for the in-kernel path: C5 K1 0.56 -> 0.49 ms)
    static const bool log_forced = getenv("MS_K1_LOG") != nullptr;
    const bool log_mode = mode != ms::kModeFuse && (h->log_mode || (dense && !log_forced));
    const int64_t groups_per_seg = static_cast<int64_t>(std::max(1, grid / h->nseg)) * h->groups;
    const int64_t reads_per_group = (R + groups_per_seg - 1) / groups_per_seg;
    // entries = flagged reads (~1.6 % of a thread's reads at CCS error rates, more at variant columns): room for 4 %
    const uint32_t exc_cap = log_mode ? static_cast<uint32_t>(std::min<int64_t>(8192, std::max<int64_t>(64, reads_per_group / 25))) : 0u;
    const int64_t nlists = static_cast<int64_t>(grid) * threads;
    if (mode != ms::kModeFuse) {
        MS_CUDA(h, h->b_exc_list.ensure(static_cast<size_t>(nlists) * std::max(1u, exc_cap) * 16));
        MS_CUDA(h, h->b_exc_cnt.ensure(static_cast<size_t>(nlists) * 4));
    }
    a.exc_list = h->b_exc_list.as<uint4>(); a.exc_cnt = h->b_exc_cnt.as<uint32_t>(); a.exc_cap = exc_cap; a.exc_lists = nlists;
    if (h->timing) MS_CUDA(h, cudaEventRecord(h->ev_k1[0], h->stream));
    // row-groups of more than 2047 reads: the instantiation with two more counter planes in shared memory (pileup.cu)
    const int64_t steps_max = (ntiles + std::max(1, grid / h->nseg) - 1) / std::max(1, grid / h->nseg);   // tiles of the busiest CTA
    const bool hi = steps_max * 8 > ms::kMaxReadsPerFlush;
    ms::pileup_launch(mode, dense, hi, grid, threads, hi ? h->smem_bytes_hi : h->smem_bytes, h->stream, a);
    if (h->timing) { MS_CUDA(h, cudaEventRecord(h->ev_k1[1], h->stream)); h->k1_reads = R; }
    if (log_mode) { ms::pileup_exceptions_launch(dense, grid, threads, h->stream, a); h->launches++; }
    const int64_t nfin = static_cast<int64_t>(h->L) * 9 * 4;
    ms::pileup_finalize_kernel<<<static_cast<int>((nfin + 255) / 256), 256, 0, h->stream>>>(
        h->d_part_col, h->d_part_piv, dense ? h->d_part_piv2 : nullptr, grid, h->nblk, h->L, h->d_pivot_state, h->d_pivot2_state, h->d_start, col, codon,
        h->count_codons ? 1 : 0, h->nseg, h->seg_len);
    h->launches += 2;
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

int ms_pileup_host(ms_handle* h, const uint32_t* h_packed, int64_t R, const uint32_t** keep_dev) {
    MsRange nvtx_range("H2D rows + tile + K1");
    if (!h || !h->d_counts || R < 0 || (R > 0 && !h_packed)) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    const size_t row_bytes = static_cast<size_t>(h->nblk) * 16;
    const size_t need = std::max<size_t>(16, static_cast<size_t>(ms::tiles_of(R)) * 8 * row_bytes);   // whole tiles
    // plain rows go up in chunks on the copy stream into one of two staging buffers; behind each chunk the main stream
    // permutes it into the tile layout (rows.cuh) and piles it up
    const int64_t chunk_rows = std::max<int64_t>(1024, ((static_cast<int64_t>(64) << 20) / static_cast<int64_t>(row_bytes)) & ~static_cast<int64_t>(7));
    const size_t stage_need = static_cast<size_t>(std::min<int64_t>(chunk_rows, std::max<int64_t>(R, 1))) * row_bytes;
    if (need > h->upload_cap || stage_need > h->b_rowstage[0].cap || stage_need > h->b_rowstage[1].cap) {
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->copy_stream));
        if (need > h->upload_cap) {
            cudaFree(h->d_upload);
            h->d_upload = nullptr; h->upload_cap = 0;
            MS_CUDA(h, cudaMalloc(&h->d_upload, need));
            h->upload_cap = need;
        }
        MS_CUDA(h, h->b_rowstage[0].ensure(stage_need));
        MS_CUDA(h, h->b_rowstage[1].ensure(stage_need));
    }
    // the copy stream must not start overwriting the staging buffers before earlier work on the main stream is done
    MS_CUDA(h, cudaEventRecord(h->ev_copy[1], h->stream));
    MS_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->ev_copy[1], 0));
    int k = 0;
    for (int64_t r0 = 0; r0 < R; r0 += chunk_rows, ++k) {
        const int64_t nr = std::min(chunk_rows, R - r0);
        uint32_t* stage = h->b_rowstage[k & 1].as<uint32_t>();
        uint8_t* dst = reinterpret_cast<uint8_t*>(h->d_upload) + static_cast<size_t>(r0) * row_bytes;   // r0 is a multiple of 8
        const uint8_t* src = reinterpret_cast<const uint8_t*>(h_packed) + static_cast<size_t>(r0) * row_bytes;
        if (k >= 2) MS_CUDA(h, cudaStreamWaitEvent(h->copy_stream, h->ev_stagefree[k & 1], 0));   // its previous chunk has been tiled
        MS_CUDA(h, cudaMemcpyAsync(stage, src, static_cast<size_t>(nr) * row_bytes, cudaMemcpyHostToDevice, h->copy_stream));
        cudaEvent_t ev = h->ev_chunk[k & 15];   // a wait snapshots the record it follows, so the ring can be reused at once
        MS_CUDA(h, cudaEventRecord(ev, h->copy_stream));
        MS_CUDA(h, cudaStreamWaitEvent(h->stream, ev, 0));
        int rc = ms_tile_rows_launch(h, stage, nr, reinterpret_cast<uint32_t*>(dst));
        if (rc != MS_OK) return rc;
        MS_CUDA(h, cudaEventRecord(h->ev_stagefree[k & 1], h->stream));
        rc = ms_pileup_dev(h, reinterpret_cast<const uint32_t*>(dst), nr);
        if (rc != MS_OK) return rc;
    }
    if (keep_dev) *keep_dev = h->d_upload;
    return MS_OK;
}

int ms_counts_device(ms_handle* h, uint32_t** d_counts, int64_t* nwords) {
    if (!h || !h->d_counts) return MS_ERR_ARG;
    if (d_counts) *d_counts = h->d_counts;
    if (nwords) *nwords = static_cast<int64_t>(h->L) * 72;
    return MS_OK;
}

int ms_get_counts(ms_handle* h, uint32_t* col, uint32_t* codon) {
    if (!h || !h->d_counts) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    const size_t L = h->L;
    // one device->host copy into pinned memory, then plain memcpys: a copy straight into a pageable destination is staged by the
    // driver in small pieces and takes several times as long
    if (h->counts_stage_words < L * 72) {
        if (h->counts_stage) cudaFreeHost(h->counts_stage);
        h->counts_stage = nullptr; h->counts_stage_words = 0;
        MS_CUDA(h, cudaMallocHost(&h->counts_stage, L * 72 * 4));
        h->counts_stage_words = L * 72;
    }
    const size_t first = col ? 0 : L * 8, last = codon ? L * 72 : L * 8;
    if (last > first) {
        MS_CUDA(h, cudaMemcpyAsync(h->counts_stage + first, h->d_counts + first, (last - first) * 4, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        if (col) memcpy(col, h->counts_stage, L * 8 * 4);
        if (codon) memcpy(codon, h->counts_stage + L * 8, L * 64 * 4);
    }
    return MS_OK;
}

}  // extern "C"
