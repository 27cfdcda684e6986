// call.cu -- K2: per-gene, per-codon minor-variant test on the (all-reduced) codon histogram.
//
// Replaces juliet's variant discovery: "comparing the number of observed mutated
// codons to the number of expected mutations at a given position ... a
// Bonferroni-corrected Fisher's Exact test" (/root/reference/doc/JULIET.md:38-42);
// reference codon from referenceSequence, else the major codon (:133-134); genes
// treated separately, overlaps allowed (:261-264); --region (:270-271);
// --min-perc / --max-perc (:342-354).  SURVEY.md rows a6-a9; unpinned choices U1-U3, U6.
#include <algorithm>
#include <cstring>
#include <vector>
#include "fisher_core.h"
#include "handle.h"

namespace ms {

struct CallPos {
    int32_t gene, codon_index, col, ref_codon;  // ref_codon < 0: use the major codon
    uint32_t ntests;
};

struct CallConst {
    double P[4];
    double alpha, min_perc, max_perc;
};

// the major codon of a column whose 64 bins the warp holds as (lane, lane + 32), lowest index on ties: maximise (count, -index).
// Integer-only, so every kernel that shares it picks the same codon.
__device__ __forceinline__ int major_codon(uint32_t k0, uint32_t k1, int lane) {
    uint32_t bc = k0, bi = lane;
    if (k1 > bc) { bc = k1; bi = lane + 32; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const uint32_t oc = __shfl_xor_sync(0xffffffffu, bc, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oc > bc || (oc == bc && oi < bi)) { bc = oc; bi = oi; }
    }
    return static_cast<int>(bi);
}

// one warp per codon position; lane tests codons lane and lane+32
__global__ void call_kernel(const uint32_t* __restrict__ codon, const CallPos* __restrict__ pos, int32_t npos,
                            CallConst cc, ms_variant* __restrict__ out, unsigned long long* __restrict__ nout,
                            unsigned long long cap) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= npos) return;
    const CallPos ps = pos[warp];
    const uint32_t* h = codon + static_cast<size_t>(ps.col) * 64;
    const uint32_t k0 = h[lane], k1 = h[lane + 32];
    uint32_t n = k0 + k1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if (n == 0) return;
    const int ref = ps.ref_codon >= 0 ? ps.ref_codon : major_codon(k0, k1, lane);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int c = lane + 32 * half;
        const uint32_t k = half ? k1 : k0;
        if (c == ref || k == 0) continue;
        int nm = 0;
#pragma unroll
        for (int i = 0; i < 3; ++i) nm += (((ref >> (2 * i)) & 3) != ((c >> (2 * i)) & 3)) ? 1 : 0;
        const double ex = ceil(static_cast<double>(n) * cc.P[nm]);
        const uint32_t e = ex >= static_cast<double>(n) ? n : static_cast<uint32_t>(ex);
        // Both rows of [[k,n-k],[e,n-e]] sum to n, so X is symmetric about (k+e)/2 and k <= e implies
        // p >= 1/2: such a codon can never be called when alpha <= ntests/2, skip the exact tail.
        if (k <= e && 0.5 * static_cast<double>(ps.ntests) >= cc.alpha) continue;
        // a codon is called iff p * ntests < alpha: stop summing the tail once that is out of reach (the p-value of a
        // codon that is not called is never reported).  For k > e the mode floor((k+e+1)/2) is <= k and fisher_upper is
        // fisher_greater itself; a k <= e codon (tested only when alpha > ntests/2) gets 1 - P(X <= k-1), not an underflow.
        const double p = fisher_upper(k, n - k, e, n - e, 1.000001 * cc.alpha / static_cast<double>(ps.ntests));
        if (!(p * static_cast<double>(ps.ntests) < cc.alpha)) continue;
        const double perc = 100.0 * static_cast<double>(k) / static_cast<double>(n);
        if (cc.min_perc >= 0.0 && !(perc > cc.min_perc)) continue;
        if (cc.max_perc >= 0.0 && !(perc < cc.max_perc)) continue;
        const unsigned long long slot = atomicAdd(nout, 1ULL);
        if (slot < cap) {
            ms_variant v;
            v.gene = ps.gene; v.codon_index = ps.codon_index; v.col = ps.col; v.ref_codon = ref; v.codon = c;
            v.count = k; v.coverage = n; v.expected = e; v.ntests = ps.ntests; v.pvalue = p;
            out[slot] = v;
        }
    }
}

// Sub-threshold candidates (restatement choice U21): K2's test on call_kernel's position table, one warp per position.  The tail
// only has to be exact below max(alpha / ntests, candidate_alpha): below alpha / ntests it decides K2's call exactly as K2 does,
// below candidate_alpha it is the candidate's p.  Every codon with count >= min_reads that K2 calls, or whose p is below
// candidate_alpha, is written with its call flag: a (column, codon) called in one gene is no candidate in any, which the host
// decides after all genes are in.
struct RareRec {
    ms_variant v;
    int32_t called, pad;
};

struct RareConst {
    double P[4];
    double alpha, candidate_alpha;
    uint32_t min_reads;
};

__global__ void rare_candidate_kernel(const uint32_t* __restrict__ codon, const CallPos* __restrict__ pos, int32_t npos, RareConst rc,
                                      RareRec* __restrict__ out, unsigned long long* __restrict__ nout, unsigned long long cap) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= npos) return;
    const CallPos ps = pos[warp];
    const uint32_t* h = codon + static_cast<size_t>(ps.col) * 64;
    const uint32_t k0 = h[lane], k1 = h[lane + 32];
    uint32_t n = k0 + k1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_xor_sync(0xffffffffu, n, o);
    if (n == 0) return;
    const int ref = ps.ref_codon >= 0 ? ps.ref_codon : major_codon(k0, k1, lane);
    const double nt = static_cast<double>(ps.ntests);
    const double bound = fmax(rc.alpha / nt, rc.candidate_alpha);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int c = lane + 32 * half;
        const uint32_t k = half ? k1 : k0;
        if (c == ref || k < rc.min_reads) continue;
        int nm = 0;
#pragma unroll
        for (int i = 0; i < 3; ++i) nm += (((ref >> (2 * i)) & 3) != ((c >> (2 * i)) & 3)) ? 1 : 0;
        const double ex = ceil(static_cast<double>(n) * rc.P[nm]);
        const uint32_t e = ex >= static_cast<double>(n) ? n : static_cast<uint32_t>(ex);
        if (k <= e && 0.5 >= bound) continue;    // p >= 1/2 (call_kernel): neither called nor a candidate
        const double p = fisher_upper(k, n - k, e, n - e, 1.000001 * bound);
        const bool called = p * nt < rc.alpha;
        if (!called && !(p < rc.candidate_alpha)) continue;
        const unsigned long long slot = atomicAdd(nout, 1ULL);
        if (slot < cap) {
            RareRec r;
            r.v.gene = ps.gene; r.v.codon_index = ps.codon_index; r.v.col = ps.col; r.v.ref_codon = ref; r.v.codon = c;
            r.v.count = k; r.v.coverage = n; r.v.expected = e; r.v.ntests = ps.ntests; r.v.pvalue = p;
            r.called = called ? 1 : 0; r.pad = 0;
            out[slot] = r;
        }
    }
}

// Control comparison (restatement choice U22): K2's position table and reference codon, but each codon c != ref of the sample,
// seen k times in n, is tested against the control's count k0 of c in its clean coverage n0 at the same column:
// p = P(X >= k) of [[k, n - k], [k0, n0 - k0]] (one-sided "greater"), p = 1 when n0 = 0.  Called iff p * ntests < alpha and the
// percentage filters pass, as in K2.  The rows are unequal (n != n0), so K2's k <= e shortcut has no counterpart: every codon
// with k >= 1 goes through fisher_upper, whose tail below the mode is 1 - P(X <= k - 1), summed away from the mode and short.
// Listed codons (the report's K2 calls) get the whole tail, the others stop at alpha / ntests as K2's do.  The precise log:
// the tables can have k close to n (a minor strain absent from the control).  ctr[0] = records, ctr[1] = positions that the
// sample covers and the control does not.
struct ControlConst {
    double alpha, min_perc, max_perc;
};

__global__ void control_call_kernel(const uint32_t* __restrict__ codon, const uint32_t* __restrict__ control, const CallPos* __restrict__ pos,
                                    const unsigned long long* __restrict__ listed, int32_t npos, ControlConst cc,
                                    ms_control_variant* __restrict__ out, unsigned long long* __restrict__ ctr, unsigned long long cap) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= npos) return;
    const CallPos ps = pos[warp];
    const uint32_t* h = codon + static_cast<size_t>(ps.col) * 64;
    const uint32_t* h0 = control + static_cast<size_t>(ps.col) * 64;
    const uint32_t k0 = h[lane], k1 = h[lane + 32], c0 = h0[lane], c1 = h0[lane + 32];
    uint32_t n = k0 + k1, n0 = c0 + c1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        n += __shfl_xor_sync(0xffffffffu, n, o);
        n0 += __shfl_xor_sync(0xffffffffu, n0, o);
    }
    if (n == 0) return;
    if (n0 == 0 && lane == 0) atomicAdd(ctr + 1, 1ULL);
    const int ref = ps.ref_codon >= 0 ? ps.ref_codon : major_codon(k0, k1, lane);
    const unsigned long long lmask = listed[warp];
    const double nt = static_cast<double>(ps.ntests);
    const double enough = 1.000001 * cc.alpha / nt;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const int c = lane + 32 * half;
        const uint32_t k = half ? k1 : k0, kc = half ? c1 : c0;
        if (c == ref || k == 0) continue;
        const bool is_listed = (lmask >> c) & 1ULL;
        const double p = n0 == 0 ? 1.0 : fisher_upper<true>(k, n - k, kc, n0 - kc, is_listed ? 2.0 : enough);
        bool called = p * nt < cc.alpha;
        const double perc = 100.0 * static_cast<double>(k) / static_cast<double>(n);
        if (cc.min_perc >= 0.0 && !(perc > cc.min_perc)) called = false;
        if (cc.max_perc >= 0.0 && !(perc < cc.max_perc)) called = false;
        if (!called && !is_listed) continue;
        const unsigned long long slot = atomicAdd(ctr, 1ULL);
        if (slot < cap) {
            ms_control_variant v;
            v.gene = ps.gene; v.codon_index = ps.codon_index; v.col = ps.col; v.ref_codon = ref; v.codon = c;
            v.count = k; v.coverage = n; v.control_count = kc; v.control_coverage = n0; v.ntests = ps.ntests;
            v.called = called ? 1 : 0; v.listed = is_listed ? 1 : 0; v.pvalue = p;
            out[slot] = v;
        }
    }
}

static int base_code(char ch) {
    switch (ch) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return -1;
    }
}

// K2's position table: every tested codon start of every gene (inside --region), its reference codon and the gene's ntests
int call_positions(ms_handle* h, const ms_gene* genes, int32_t ngenes, const char* refseq, const ms_call_params* prm,
                   std::vector<CallPos>& pos) {
    const int32_t L = h->L;
    const size_t reflen = refseq ? strnlen(refseq, static_cast<size_t>(L)) : 0;
    int32_t lo = 0, hi = L;
    if (prm->region_end > prm->region_begin) {
        lo = std::max(0, prm->region_begin - 1);
        hi = std::min(L, prm->region_end - 1);
    }
    pos.clear();
    for (int32_t g = 0; g < ngenes; ++g) {
        const int32_t gb = genes[g].begin - 1, ge = std::min(genes[g].end - 1, L);
        const size_t first = pos.size();
        for (int32_t s = gb, ci = 0; s + 3 <= ge; s += 3, ++ci) {
            if (!(s >= lo && s + 3 <= hi && s >= 0)) continue;
            if (!((h->h_start[s >> 5] >> (s & 31)) & 1u))
                MS_FAIL(h, MS_ERR_ARG, "gene codon start not in the layout's start mask");
            CallPos p;
            p.gene = g; p.codon_index = ci; p.col = s; p.ref_codon = -1; p.ntests = 0;
            if (static_cast<size_t>(s) + 3 <= reflen) {
                const int b0 = base_code(refseq[s]), b1 = base_code(refseq[s + 1]), b2 = base_code(refseq[s + 2]);
                if (b0 >= 0 && b1 >= 0 && b2 >= 0) p.ref_codon = 16 * b0 + 4 * b1 + b2;
            }
            pos.push_back(p);
        }
        const uint32_t nt = static_cast<uint32_t>(pos.size() - first);
        for (size_t i = first; i < pos.size(); ++i) pos[i].ntests = nt;
    }
    return MS_OK;
}

}  // namespace ms

extern "C" {

void ms_call_params_default(ms_call_params* p) {
    if (!p) return;
    p->substitution_rate = 5e-4; p->deletion_rate = 3e-3; p->alpha = 0.01;
    p->min_perc = -1.0; p->max_perc = -1.0; p->region_begin = 0; p->region_end = 0;
}

}  // extern "C"

// K2 in two halves so that the single-call pass (pass.cu) can keep the GPU busy between them: ms_call_launch enqueues the kernel
// and tells where its output lives on the device, ms_call_collect downloads, waits, sorts.  ms_call = launch + collect.
int ms_call_launch(ms_handle* h, const ms_gene* genes, int32_t ngenes, const char* refseq, const ms_call_params* prm,
                   const ms_variant** d_calls, const unsigned long long** d_ncalls, int64_t* calls_cap) {
    MsRange nvtx_range("K2 call");
    if (!h || !h->d_counts || !genes || ngenes < 0 || !prm) return MS_ERR_ARG;
    if (!h->count_codons) MS_FAIL(h, MS_ERR_ARG, "ms_set_layout was called without a codon start mask");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t L = h->L;
    std::vector<ms::CallPos> pos;
    const int prc = ms::call_positions(h, genes, ngenes, refseq, prm, pos);
    if (prc != MS_OK) return prc;
    h->call_npos = pos.size();
    if (d_calls) *d_calls = nullptr;
    if (d_ncalls) *d_ncalls = nullptr;
    if (calls_cap) *calls_cap = 0;
    if (pos.empty()) return MS_OK;
    const size_t npos = pos.size();
    const size_t dev_cap = npos * 63;
    const size_t need = 64 + dev_cap * sizeof(ms_variant) + npos * sizeof(ms::CallPos);
    if (need > h->call_cap) {
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        cudaFree(h->d_call_buf);
        h->d_call_buf = nullptr; h->call_cap = 0;
        MS_CUDA(h, cudaMalloc(&h->d_call_buf, need));
        h->call_cap = need;
        h->call_pos_cache.clear();
    }
    uint8_t* base = static_cast<uint8_t*>(h->d_call_buf);
    unsigned long long* d_n = reinterpret_cast<unsigned long long*>(base);
    ms_variant* d_out = reinterpret_cast<ms_variant*>(base + 64);
    ms::CallPos* d_pos = reinterpret_cast<ms::CallPos*>(base + 64 + dev_cap * sizeof(ms_variant));
    // small pinned stage: position table up, [count | first variants] down, one copy each way
    constexpr size_t kQuick = 1024;
    const size_t stage_need = std::max(npos * sizeof(ms::CallPos), 64 + kQuick * sizeof(ms_variant));
    if (stage_need > h->call_stage_cap) {
        if (h->call_stage) cudaFreeHost(h->call_stage);
        h->call_stage = nullptr; h->call_stage_cap = 0;
        MS_CUDA(h, cudaMallocHost(&h->call_stage, stage_need + 4096));
        h->call_stage_cap = stage_need + 4096;
    }
    const size_t pos_bytes = npos * sizeof(ms::CallPos);
    const bool same_pos = h->call_pos_cache.size() == pos_bytes && memcmp(h->call_pos_cache.data(), pos.data(), pos_bytes) == 0;
    MS_CUDA(h, cudaMemsetAsync(d_n, 0, 8, h->stream));
    if (!same_pos) {
        memcpy(h->call_stage, pos.data(), pos_bytes);
        MS_CUDA(h, cudaMemcpyAsync(d_pos, h->call_stage, pos_bytes, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));  // the stage is reused for the download below
        h->call_pos_cache.assign(reinterpret_cast<const uint8_t*>(pos.data()), reinterpret_cast<const uint8_t*>(pos.data()) + pos_bytes);
    }
    ms::CallConst cc;
    ms::codon_error_table(prm->substitution_rate, prm->deletion_rate, cc.P);
    cc.alpha = prm->alpha; cc.min_perc = prm->min_perc; cc.max_perc = prm->max_perc;
    const int threads = 128;
    const int blocks = static_cast<int>((npos * 32 + threads - 1) / threads);
    ms::call_kernel<<<blocks, threads, 0, h->stream>>>(h->d_counts + static_cast<size_t>(L) * 8, d_pos,
                                                       static_cast<int32_t>(npos), cc, d_out, d_n, dev_cap);
    h->launches++;
    MS_CUDA(h, cudaGetLastError());
    const size_t quick = std::min(kQuick, dev_cap);
    MS_CUDA(h, cudaMemcpyAsync(h->call_stage, base, 64 + quick * sizeof(ms_variant), cudaMemcpyDeviceToHost, h->stream));
    if (d_calls) *d_calls = d_out;
    if (d_ncalls) *d_ncalls = d_n;
    if (calls_cap) *calls_cap = static_cast<int64_t>(dev_cap);
    return MS_OK;
}

// waits for the stream (unless the caller already has: `synced`), sorts, hands the variants over
int ms_call_collect(ms_handle* h, bool synced, ms_variant* out, int64_t cap, int64_t* n) {
    if (!h || !n || (cap > 0 && !out)) return MS_ERR_ARG;
    *n = 0;
    if (h->call_npos == 0) return MS_OK;
    MS_CUDA(h, cudaSetDevice(h->device));
    if (!synced) MS_CUDA(h, cudaStreamSynchronize(h->stream));
    constexpr size_t kQuick = 1024;
    const size_t dev_cap = h->call_npos * 63;
    const size_t quick = std::min(kQuick, dev_cap);
    uint8_t* base = static_cast<uint8_t*>(h->d_call_buf);
    const ms_variant* d_out = reinterpret_cast<const ms_variant*>(base + 64);
    unsigned long long cnt = 0;
    memcpy(&cnt, h->call_stage, 8);
    std::vector<ms_variant> v(cnt);
    if (cnt <= quick) {
        if (cnt) memcpy(v.data(), static_cast<uint8_t*>(h->call_stage) + 64, cnt * sizeof(ms_variant));
    } else {
        MS_CUDA(h, cudaMemcpyAsync(v.data(), d_out, cnt * sizeof(ms_variant), cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    std::sort(v.begin(), v.end(), [](const ms_variant& a, const ms_variant& b) {
        if (a.gene != b.gene) return a.gene < b.gene;
        if (a.col != b.col) return a.col < b.col;
        return a.codon < b.codon;
    });
    *n = static_cast<int64_t>(cnt);
    for (int64_t i = 0; i < std::min<int64_t>(cap, static_cast<int64_t>(cnt)); ++i) out[i] = v[i];
    return MS_OK;
}

extern "C" {

int ms_call(ms_handle* h, const ms_gene* genes, int32_t ngenes, const char* refseq, const ms_call_params* prm,
            ms_variant* out, int64_t cap, int64_t* n) {
    if (!n || (cap > 0 && !out)) return MS_ERR_ARG;
    int rc = ms_call_launch(h, genes, ngenes, refseq, prm, nullptr, nullptr, nullptr);
    if (rc != MS_OK) return rc;
    return ms_call_collect(h, false, out, cap, n);
}

}  // extern "C"

extern "C" {

void ms_rare_params_default(ms_rare_params* p) {
    if (!p) return;
    p->candidate_alpha = 0.1;
    p->min_reads = 5;
}

int ms_rare_candidates(ms_handle* h, const ms_gene* genes, int32_t ngenes, const char* refseq, const ms_call_params* prm,
                       const ms_rare_params* rp, ms_variant* out, int64_t cap, int64_t* n, int64_t* dropped) {
    MsRange nvtx_range("rare candidates");
    if (!h || !h->d_counts || !genes || ngenes < 0 || !prm || !rp || !n || cap < 0 || (cap > 0 && !out)) return MS_ERR_ARG;
    if (rp->min_reads < 1 || !(rp->candidate_alpha > 0.0) || !(prm->alpha > 0.0)) MS_FAIL(h, MS_ERR_ARG, "ms_rare_candidates: bad parameters");
    if (!h->count_codons) MS_FAIL(h, MS_ERR_ARG, "ms_set_layout was called without a codon start mask");
    MS_CUDA(h, cudaSetDevice(h->device));
    *n = 0;
    if (dropped) *dropped = 0;
    std::vector<ms::CallPos> pos;
    int rc = ms::call_positions(h, genes, ngenes, refseq, prm, pos);
    if (rc != MS_OK) return rc;
    if (pos.empty()) return MS_OK;
    const size_t npos = pos.size();
    MS_CUDA(h, h->b_rare_pos.ensure(npos * sizeof(ms::CallPos)));
    MS_CUDA(h, cudaMemcpyAsync(h->b_rare_pos.p, pos.data(), npos * sizeof(ms::CallPos), cudaMemcpyHostToDevice, h->stream));
    ms::RareConst cc;
    ms::codon_error_table(prm->substitution_rate, prm->deletion_rate, cc.P);
    cc.alpha = prm->alpha; cc.candidate_alpha = rp->candidate_alpha; cc.min_reads = static_cast<uint32_t>(rp->min_reads);
    // the records are few (codons seen min_reads times with a small p); the buffer grows and the kernel runs again if not
    size_t dev_cap = std::min<size_t>(npos * 63, 1 << 16);
    unsigned long long cnt = 0;
    for (;;) {
        MS_CUDA(h, h->b_rare_out.ensure(64 + dev_cap * sizeof(ms::RareRec)));
        unsigned long long* d_n = h->b_rare_out.as<unsigned long long>();
        MS_CUDA(h, cudaMemsetAsync(d_n, 0, 8, h->stream));
        const int threads = 128;
        const int blocks = static_cast<int>((npos * 32 + threads - 1) / threads);
        ms::rare_candidate_kernel<<<blocks, threads, 0, h->stream>>>(h->d_counts + static_cast<size_t>(h->L) * 8, h->b_rare_pos.as<ms::CallPos>(),
                                                                     static_cast<int32_t>(npos), cc,
                                                                     reinterpret_cast<ms::RareRec*>(h->b_rare_out.as<uint8_t>() + 64), d_n, dev_cap);
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
        MS_CUDA(h, cudaMemcpyAsync(&cnt, d_n, 8, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        if (cnt <= dev_cap) break;
        dev_cap = static_cast<size_t>(cnt);
    }
    std::vector<ms::RareRec> rec(cnt);
    if (cnt) {
        MS_CUDA(h, cudaMemcpyAsync(rec.data(), h->b_rare_out.as<uint8_t>() + 64, cnt * sizeof(ms::RareRec), cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    std::sort(rec.begin(), rec.end(), [](const ms::RareRec& a, const ms::RareRec& b) {
        if (a.v.col != b.v.col) return a.v.col < b.v.col;
        if (a.v.codon != b.v.codon) return a.v.codon < b.v.codon;
        return a.v.gene < b.v.gene;
    });
    // one record per (column, codon) that no gene calls: the gene with the smallest p, the lowest gene index on ties
    std::vector<ms_variant> cand;
    for (size_t i = 0; i < rec.size();) {
        size_t j = i;
        bool called = false;
        size_t best = i;
        for (; j < rec.size() && rec[j].v.col == rec[i].v.col && rec[j].v.codon == rec[i].v.codon; ++j) {
            called = called || rec[j].called;
            if (rec[j].v.pvalue < rec[best].v.pvalue) best = j;
        }
        if (!called) cand.push_back(rec[best].v);
        i = j;
    }
    const auto by_col = [](const ms_variant& a, const ms_variant& b) { return a.col != b.col ? a.col < b.col : a.codon < b.codon; };
    if (cand.size() > MS_RARE_MAX_CANDIDATES) {
        std::sort(cand.begin(), cand.end(), [&](const ms_variant& a, const ms_variant& b) {
            if (a.pvalue != b.pvalue) return a.pvalue < b.pvalue;
            return by_col(a, b);
        });
        if (dropped) *dropped = static_cast<int64_t>(cand.size()) - MS_RARE_MAX_CANDIDATES;
        cand.resize(MS_RARE_MAX_CANDIDATES);
        std::sort(cand.begin(), cand.end(), by_col);
    }
    *n = static_cast<int64_t>(cand.size());
    for (int64_t i = 0; i < std::min<int64_t>(cap, *n); ++i) out[i] = cand[i];
    return MS_OK;
}

int ms_control_capture(ms_handle* h) {
    if (!h || !h->d_counts) return MS_ERR_ARG;
    if (!h->count_codons) MS_FAIL(h, MS_ERR_ARG, "ms_set_layout was called without a codon start mask");
    MS_CUDA(h, cudaSetDevice(h->device));
    const size_t bytes = static_cast<size_t>(h->L) * 64 * 4;
    MS_CUDA(h, h->b_control.ensure(bytes));
    MS_CUDA(h, cudaMemcpyAsync(h->b_control.p, h->d_counts + static_cast<size_t>(h->L) * 8, bytes, cudaMemcpyDeviceToDevice, h->stream));
    h->control_valid = true;
    return MS_OK;
}

int ms_control_call(ms_handle* h, const ms_gene* genes, int32_t ngenes, const char* refseq, const ms_call_params* prm,
                    const ms_variant* listed, int64_t nlisted, ms_control_variant* out, int64_t cap, int64_t* n,
                    int64_t* uncovered_positions) {
    MsRange nvtx_range("control call");
    if (!h || !h->d_counts || !genes || ngenes < 0 || !prm || !n || cap < 0 || (cap > 0 && !out) || nlisted < 0 || (nlisted > 0 && !listed))
        return MS_ERR_ARG;
    if (!(prm->alpha > 0.0)) MS_FAIL(h, MS_ERR_ARG, "ms_control_call: alpha must be > 0");
    if (!h->count_codons) MS_FAIL(h, MS_ERR_ARG, "ms_set_layout was called without a codon start mask");
    if (!h->control_valid) MS_FAIL(h, MS_ERR_ARG, "ms_control_call: no control captured for this layout (call ms_control_capture first)");
    MS_CUDA(h, cudaSetDevice(h->device));
    *n = 0;
    if (uncovered_positions) *uncovered_positions = 0;
    std::vector<ms::CallPos> pos;
    int rc = ms::call_positions(h, genes, ngenes, refseq, prm, pos);
    if (rc != MS_OK) return rc;
    if (pos.empty()) return MS_OK;
    const size_t npos = pos.size();
    // listed codons -> one 64-bit mask per position table entry; a gene's entries are contiguous and ordered by column
    std::vector<unsigned long long> mask(npos, 0ULL);
    std::vector<size_t> gene_first(static_cast<size_t>(ngenes) + 1, npos);
    for (size_t i = npos; i-- > 0;) gene_first[pos[i].gene] = i;
    for (int32_t g = ngenes - 1; g >= 0; --g) gene_first[g] = std::min(gene_first[g], gene_first[g + 1]);
    for (int64_t i = 0; i < nlisted; ++i) {
        const ms_variant& v = listed[i];
        if (v.gene < 0 || v.gene >= ngenes || v.codon < 0 || v.codon > 63) MS_FAIL(h, MS_ERR_ARG, "ms_control_call: a listed variant has no such gene or codon");
        const auto b = pos.begin() + static_cast<std::ptrdiff_t>(gene_first[v.gene]), e = pos.begin() + static_cast<std::ptrdiff_t>(gene_first[v.gene + 1]);
        const auto it = std::lower_bound(b, e, v.col, [](const ms::CallPos& p, int32_t col) { return p.col < col; });
        if (it == e || it->col != v.col) MS_FAIL(h, MS_ERR_ARG, "ms_control_call: a listed variant is not at one of the gene's tested positions");
        mask[static_cast<size_t>(it - pos.begin())] |= 1ULL << v.codon;
    }
    const size_t mask_bytes = npos * sizeof(unsigned long long);
    MS_CUDA(h, h->b_control_pos.ensure(mask_bytes + npos * sizeof(ms::CallPos)));
    unsigned long long* d_mask = h->b_control_pos.as<unsigned long long>();
    ms::CallPos* d_pos = reinterpret_cast<ms::CallPos*>(h->b_control_pos.as<uint8_t>() + mask_bytes);
    MS_CUDA(h, cudaMemcpyAsync(d_mask, mask.data(), mask_bytes, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(d_pos, pos.data(), npos * sizeof(ms::CallPos), cudaMemcpyHostToDevice, h->stream));
    ms::ControlConst cc;
    cc.alpha = prm->alpha; cc.min_perc = prm->min_perc; cc.max_perc = prm->max_perc;
    // the records are the listed codons and the control calls, few; the buffer grows and the kernel runs again if not
    size_t dev_cap = std::min<size_t>(npos * 63, std::max<size_t>(1 << 12, 2 * static_cast<size_t>(nlisted)));
    unsigned long long st[2] = {0, 0};
    for (;;) {
        MS_CUDA(h, h->b_control_out.ensure(64 + dev_cap * sizeof(ms_control_variant)));
        unsigned long long* d_ctr = h->b_control_out.as<unsigned long long>();
        MS_CUDA(h, cudaMemsetAsync(d_ctr, 0, 16, h->stream));
        const int threads = 128;
        const int blocks = static_cast<int>((npos * 32 + threads - 1) / threads);
        ms::control_call_kernel<<<blocks, threads, 0, h->stream>>>(h->d_counts + static_cast<size_t>(h->L) * 8, h->b_control.as<uint32_t>(), d_pos,
                                                                   d_mask, static_cast<int32_t>(npos), cc,
                                                                   reinterpret_cast<ms_control_variant*>(h->b_control_out.as<uint8_t>() + 64), d_ctr,
                                                                   dev_cap);
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
        MS_CUDA(h, cudaMemcpyAsync(st, d_ctr, 16, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        if (st[0] <= dev_cap) break;
        dev_cap = static_cast<size_t>(st[0]);
    }
    std::vector<ms_control_variant> rec(st[0]);
    if (st[0]) {
        MS_CUDA(h, cudaMemcpyAsync(rec.data(), h->b_control_out.as<uint8_t>() + 64, st[0] * sizeof(ms_control_variant), cudaMemcpyDeviceToHost,
                                   h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    std::sort(rec.begin(), rec.end(), [](const ms_control_variant& a, const ms_control_variant& b) {
        if (a.gene != b.gene) return a.gene < b.gene;
        if (a.col != b.col) return a.col < b.col;
        return a.codon < b.codon;
    });
    *n = static_cast<int64_t>(st[0]);
    if (uncovered_positions) *uncovered_positions = static_cast<int64_t>(st[1]);
    for (int64_t i = 0; i < std::min<int64_t>(cap, *n); ++i) out[i] = rec[i];
    return MS_OK;
}

}  // extern "C"
