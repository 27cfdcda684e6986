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
    int ref = ps.ref_codon;
    if (ref < 0) {
        // major codon, lowest index wins ties: maximise (count, -index)
        uint32_t bc = k0, bi = lane;
        if (k1 > bc) { bc = k1; bi = lane + 32; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const uint32_t oc = __shfl_xor_sync(0xffffffffu, bc, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (oc > bc || (oc == bc && oi < bi)) { bc = oc; bi = oi; }
        }
        ref = static_cast<int>(bi);
    }
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

static int base_code(char ch) {
    switch (ch) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return -1;
    }
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
    const size_t reflen = refseq ? strnlen(refseq, static_cast<size_t>(L)) : 0;
    int32_t lo = 0, hi = L;
    if (prm->region_end > prm->region_begin) {
        lo = std::max(0, prm->region_begin - 1);
        hi = std::min(L, prm->region_end - 1);
    }
    std::vector<ms::CallPos> pos;
    for (int32_t g = 0; g < ngenes; ++g) {
        const int32_t gb = genes[g].begin - 1, ge = std::min(genes[g].end - 1, L);
        const size_t first = pos.size();
        for (int32_t s = gb, ci = 0; s + 3 <= ge; s += 3, ++ci) {
            if (!(s >= lo && s + 3 <= hi && s >= 0)) continue;
            if (!((h->h_start[s >> 5] >> (s & 31)) & 1u))
                MS_FAIL(h, MS_ERR_ARG, "gene codon start not in the layout's start mask");
            ms::CallPos p;
            p.gene = g; p.codon_index = ci; p.col = s; p.ref_codon = -1; p.ntests = 0;
            if (static_cast<size_t>(s) + 3 <= reflen) {
                const int b0 = ms::base_code(refseq[s]), b1 = ms::base_code(refseq[s + 1]), b2 = ms::base_code(refseq[s + 2]);
                if (b0 >= 0 && b1 >= 0 && b2 >= 0) p.ref_codon = 16 * b0 + 4 * b1 + b2;
            }
            pos.push_back(p);
        }
        const uint32_t nt = static_cast<uint32_t>(pos.size() - first);
        for (size_t i = first; i < pos.size(); ++i) pos[i].ntests = nt;
    }
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
