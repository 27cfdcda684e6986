// rare.cu -- sub-threshold variant linkage (restatement choice U21; include/minorseq_b200.h "sub-threshold variant linkage").
//
// The keys are the called variants followed by K2's sub-threshold candidates (call.cu, rare_candidate_kernel), phased with the
// clean-codon matrix as for ms_linkage: the stacked Gram matrix of ms_linkage_device holds every pair's 2x2 table.  Only the
// pairs with a candidate on the right are tested, and only for the linked tail: a codon seen in a handful of reads can be
// significant through its co-carriers only.
//   rare_count_kernel    m_r = the number of tested pairs (w >= first_candidate, |col_v - col_w| >= 3, n >= min_reads)
//   rare_pair_kernel     P(X >= a) (fisher_upper<true>, stopped once it reaches alpha / m_r), the linked pairs appended with
//                        their table, D' and r^2; the host sorts them by (v, w)
//   rare_support_kernel  per key set, the reads carrying every key and the reads clean at every key: one lane per read, the
//                        sets' (word, mask) entries staged in shared memory, warp-aggregated atomics
// Every value depends on the integer counts only, so every run and rank gets the same bytes.
#include <algorithm>
#include <numeric>
#include <vector>
#include "link_table.cuh"
#include "linkage_core.h"
#include "phase_internal.cuh"

int ms_comm_allreduce_u32(ms_handle* h, uint32_t* d, size_t count);

namespace ms {

constexpr int kRareThreads = 128;
constexpr int kRareSupportEntries = 4096;   // (word, mask) entries of the key sets staged per launch
constexpr int kRareSupportSets = 1024;      // key sets per launch

__device__ __forceinline__ bool rare_tested(const int32_t* __restrict__ col, const LinkTable& t, int32_t v, int32_t w, int32_t min_reads) {
    const int32_t dc = col[v] - col[w];
    return (dc >= kLinkageMinSpacing || -dc >= kLinkageMinSpacing) && t.n >= static_cast<uint32_t>(min_reads);
}

// row v: the pairs (v, w) with w > v and w >= fc
__global__ void __launch_bounds__(kRareThreads) rare_count_kernel(const int32_t* __restrict__ G, int32_t dim, int32_t V, int32_t fc,
                                                                 const int32_t* __restrict__ col, int32_t min_reads,
                                                                 unsigned long long* __restrict__ ctr) {
    const int32_t v = blockIdx.x;
    unsigned long long k = 0;
    for (int32_t w = max(v + 1, fc) + static_cast<int32_t>(threadIdx.x); w < V; w += kRareThreads)
        k += rare_tested(col, link_table(G, dim, v, w), v, w, min_reads) ? 1 : 0;
    for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xffffffffu, k, o);
    if ((threadIdx.x & 31) == 0 && k) atomicAdd(ctr, k);
}

// ctr[0] = m_r, ctr[1] = linked pairs found (out holds the first cap of them, in no particular order)
__global__ void __launch_bounds__(kRareThreads) rare_pair_kernel(const int32_t* __restrict__ G, int32_t dim, int32_t V, int32_t fc,
                                                                const int32_t* __restrict__ col, int32_t min_reads, double alpha,
                                                                unsigned long long* __restrict__ ctr, ms_linkage_pair* __restrict__ out,
                                                                unsigned long long cap) {
    const int32_t v = blockIdx.x;
    const double m = static_cast<double>(ctr[0]);
    const double enough = 1.000001 * alpha / m;      // the tail only has to be exact below alpha / m_r (as in K2)
    for (int32_t w = max(v + 1, fc) + static_cast<int32_t>(threadIdx.x); w < V; w += kRareThreads) {
        const LinkTable t = link_table(G, dim, v, w);
        if (!rare_tested(col, t, v, w, min_reads)) continue;
        const uint32_t d = t.n - t.a - t.b - t.c;
        const double p = fisher_upper<true>(t.a, t.b, t.c, d, enough);
        if (!(p * m < alpha)) continue;
        const unsigned long long slot = atomicAdd(ctr + 1, 1ULL);
        if (slot >= cap) continue;
        ms_linkage_pair o;
        o.v = v; o.w = w;
        o.both = t.a; o.v_only = t.b; o.w_only = t.c; o.neither = d;
        linkage_measures(t.a, t.b, t.c, t.n, &o.d_prime, &o.r2);
        o.pvalue = p;
        o.relation = kLinkageLinked;
        out[slot] = o;
    }
}

// cnt[g] += reads with B = 1 at every key of set g, cnt[G + g] += reads with M = 1 at every key; the sets [g0, g0 + ng) of this
// launch are ent[off[i] .. off[i+1]) = (word, mask) for i = g - g0
__global__ void __launch_bounds__(256) rare_support_kernel(const uint32_t* __restrict__ B, const uint32_t* __restrict__ Mb, int64_t R,
                                                          int32_t vwords, const uint2* __restrict__ ent, const int32_t* __restrict__ off,
                                                          int32_t g0, int32_t ng, int32_t G, uint32_t* __restrict__ cnt) {
    extern __shared__ uint2 s_ent[];
    int32_t* s_off = reinterpret_cast<int32_t*>(s_ent + kRareSupportEntries);
    const int32_t nent = off[ng];
    for (int32_t i = threadIdx.x; i < nent; i += blockDim.x) s_ent[i] = ent[i];
    for (int32_t i = threadIdx.x; i <= ng; i += blockDim.x) s_off[i] = off[i];
    __syncthreads();
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool valid = r < R;
    const uint32_t* brow = B + (valid ? r : 0) * vwords;
    const uint32_t* mrow = Mb + (valid ? r : 0) * vwords;
    const int lane = threadIdx.x & 31;
    for (int32_t g = 0; g < ng; ++g) {
        bool car = valid, inf = valid;
        for (int32_t e = s_off[g]; e < s_off[g + 1]; ++e) {
            const uint2 x = s_ent[e];
            if (valid) {
                car = car && (brow[x.x] & x.y) == x.y;
                inf = inf && (mrow[x.x] & x.y) == x.y;
            }
        }
        const uint32_t bc = __ballot_sync(0xffffffffu, car), bi = __ballot_sync(0xffffffffu, inf);
        if (lane == 0) {
            if (bc) atomicAdd(cnt + g0 + g, static_cast<uint32_t>(__popc(bc)));
            if (bi) atomicAdd(cnt + G + g0 + g, static_cast<uint32_t>(__popc(bi)));
        }
    }
}

}  // namespace ms

extern "C" {

int ms_rare_linkage(ms_handle* h, int32_t first_candidate, const ms_linkage_params* prm, ms_linkage_pair* out, int64_t cap, int64_t* n,
                    int64_t* ntested) {
    MsRange nvtx_range("rare linkage");
    if (!h || !prm || !n || cap < 0 || (cap > 0 && !out) || !(prm->alpha > 0.0) || prm->min_reads < 0) return MS_ERR_ARG;
    if (first_candidate < 0 || first_candidate > h->V) MS_FAIL(h, MS_ERR_ARG, "ms_rare_linkage: first_candidate outside the keys");
    int32_t* G = nullptr;
    int32_t dim = 0;
    int rc = ms_linkage_device(h, &G, &dim);      // the (all-reduced, cached) stacked Gram matrix: a collective
    if (rc != MS_OK) return rc;
    const int32_t V = h->V;
    if (static_cast<int32_t>(h->link_col.size()) != V) MS_FAIL(h, MS_ERR_ARG, "ms_rare_linkage: key list changed");
    MS_CUDA(h, h->b_link_col.ensure(static_cast<size_t>(std::max(1, V)) * 4));
    if (V > 0) MS_CUDA(h, cudaMemcpyAsync(h->b_link_col.p, h->link_col.data(), static_cast<size_t>(V) * 4, cudaMemcpyHostToDevice, h->stream));
    const int32_t* col = h->b_link_col.as<int32_t>();
    rc = ms::phase_ensure_stage(h, 16);
    if (rc != MS_OK) return rc;
    uint64_t* st = static_cast<uint64_t*>(h->h_stage);
    size_t dev_cap = std::max<size_t>(1024, static_cast<size_t>(cap));
    bool counted = false;
    for (;;) {
        MS_CUDA(h, h->b_rare_pairs.ensure(64 + dev_cap * sizeof(ms_linkage_pair)));
        unsigned long long* ctr = h->b_rare_pairs.as<unsigned long long>();
        ms_linkage_pair* d_out = reinterpret_cast<ms_linkage_pair*>(h->b_rare_pairs.as<uint8_t>() + 64);
        if (!counted) {
            MS_CUDA(h, cudaMemsetAsync(ctr, 0, 16, h->stream));
            if (V > 1) {
                ms::rare_count_kernel<<<V - 1, ms::kRareThreads, 0, h->stream>>>(G, dim, V, first_candidate, col, prm->min_reads, ctr);
                h->launches++;
            }
            counted = true;
        } else {
            MS_CUDA(h, cudaMemsetAsync(ctr + 1, 0, 8, h->stream));
        }
        if (V > 1) {
            ms::rare_pair_kernel<<<V - 1, ms::kRareThreads, 0, h->stream>>>(G, dim, V, first_candidate, col, prm->min_reads, prm->alpha, ctr, d_out,
                                                                           dev_cap);
            h->launches++;
        }
        MS_CUDA(h, cudaGetLastError());
        MS_CUDA(h, cudaMemcpyAsync(st, ctr, 16, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        if (st[1] <= dev_cap) break;
        dev_cap = static_cast<size_t>(st[1]);
    }
    const int64_t m = static_cast<int64_t>(st[0]), nl = static_cast<int64_t>(st[1]);
    if (ntested) *ntested = m;
    *n = nl;
    const int64_t k = std::min(cap, nl);
    if (k > 0) {
        std::vector<ms_linkage_pair> v(static_cast<size_t>(nl));
        MS_CUDA(h, cudaMemcpyAsync(v.data(), h->b_rare_pairs.as<uint8_t>() + 64, static_cast<size_t>(nl) * sizeof(ms_linkage_pair),
                                   cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        std::sort(v.begin(), v.end(), [](const ms_linkage_pair& a, const ms_linkage_pair& b) { return a.v != b.v ? a.v < b.v : a.w < b.w; });
        std::copy(v.begin(), v.begin() + k, out);
    }
    return MS_OK;
}

int ms_rare_support(ms_handle* h, const uint32_t* masks, int64_t G, uint64_t* carriers, uint64_t* informative) {
    MsRange nvtx_range("rare support");
    if (!h || G < 0 || (G > 0 && (!masks || !carriers || !informative))) return MS_ERR_ARG;
    if (!h->b_bits.p) MS_FAIL(h, MS_ERR_ARG, "ms_rare_support: no phased reads");
    if (!h->link_ready) MS_FAIL(h, MS_ERR_ARG, "ms_rare_support: call ms_set_linkage(h, 1) before ms_phase_begin");
    if (G > (int64_t{1} << 30)) MS_FAIL(h, MS_ERR_ARG, "ms_rare_support: too many key sets");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t V = h->V, vw = h->vwords;
    // per set its non-zero words (bits >= V dropped); launches of at most kRareSupportSets sets and kRareSupportEntries entries
    std::vector<uint32_t> ent;                // (word, mask) pairs
    std::vector<int64_t> set_off(1, 0);
    for (int64_t g = 0; g < G; ++g) {
        int64_t ne = 0;
        for (int32_t w = 0; w < vw; ++w) {
            uint32_t x = masks[static_cast<size_t>(g) * vw + w];
            if (32 * w + 32 > V) x &= 32 * w >= V ? 0u : (1u << (V - 32 * w)) - 1u;
            if (x) { ent.push_back(static_cast<uint32_t>(w)); ent.push_back(x); ++ne; }
        }
        if (ne == 0) MS_FAIL(h, MS_ERR_ARG, "ms_rare_support: an empty key set");
        if (ne > ms::kRareSupportEntries) MS_FAIL(h, MS_ERR_ARG, "ms_rare_support: a key set spans too many words");
        set_off.push_back(set_off.back() + ne);
    }
    // device scratch: [2G counters | entries | per-launch offsets]
    const size_t cnt_bytes = (static_cast<size_t>(2 * G) * 4 + 15) & ~static_cast<size_t>(15);
    const size_t ent_bytes = std::max<size_t>(8, ent.size() * 4);
    std::vector<int32_t> offs;                // per launch ng + 1 offsets, relative to the launch's first entry
    std::vector<std::pair<int64_t, int64_t>> launches;   // (first set, sets)
    for (int64_t g = 0; g < G;) {
        int64_t e = g;
        while (e < G && e - g < ms::kRareSupportSets && set_off[e + 1] - set_off[g] <= ms::kRareSupportEntries) ++e;
        launches.emplace_back(g, e - g);
        for (int64_t i = g; i <= e; ++i) offs.push_back(static_cast<int32_t>(set_off[i] - set_off[g]));
        g = e;
    }
    MS_CUDA(h, h->b_rare_sup.ensure(cnt_bytes + ent_bytes + std::max<size_t>(4, offs.size() * 4)));
    uint8_t* base = h->b_rare_sup.as<uint8_t>();
    uint32_t* d_cnt = reinterpret_cast<uint32_t*>(base);
    uint2* d_ent = reinterpret_cast<uint2*>(base + cnt_bytes);
    int32_t* d_off = reinterpret_cast<int32_t*>(base + cnt_bytes + ent_bytes);
    if (G == 0) return MS_OK;
    MS_CUDA(h, cudaMemsetAsync(d_cnt, 0, static_cast<size_t>(2 * G) * 4, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(d_ent, ent.data(), ent.size() * 4, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(d_off, offs.data(), offs.size() * 4, cudaMemcpyHostToDevice, h->stream));
    const int64_t R = h->phase_n;
    const size_t smem = ms::kRareSupportEntries * sizeof(uint2) + (ms::kRareSupportSets + 1) * sizeof(int32_t);
    size_t oi = 0;
    for (const auto& l : launches) {
        if (R > 0) {
            const int64_t blocks = (R + 255) / 256;
            ms::rare_support_kernel<<<static_cast<unsigned>(blocks), 256, smem, h->stream>>>(
                h->b_bits.as<uint32_t>(), h->b_mbits.as<uint32_t>(), R, vw, d_ent + set_off[l.first], d_off + oi, static_cast<int32_t>(l.first),
                static_cast<int32_t>(l.second), static_cast<int32_t>(G), d_cnt);
            h->launches++;
        }
        oi += static_cast<size_t>(l.second) + 1;
    }
    MS_CUDA(h, cudaGetLastError());
    if (h->comm) {
        const int rc = ms_comm_allreduce_u32(h, d_cnt, static_cast<size_t>(2 * G));
        if (rc != MS_OK) return rc;
    }
    std::vector<uint32_t> c(static_cast<size_t>(2 * G));
    MS_CUDA(h, cudaMemcpyAsync(c.data(), d_cnt, c.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int64_t g = 0; g < G; ++g) { carriers[g] = c[g]; informative[g] = c[G + g]; }
    return MS_OK;
}

int ms_rare_groups(const ms_linkage_pair* pairs, int64_t npairs, int32_t first_candidate, int32_t V, int32_t* group) {
    if (V < 0 || npairs < 0 || (npairs > 0 && !pairs) || (V > 0 && !group) || first_candidate < 0 || first_candidate > V) return MS_ERR_ARG;
    std::vector<int32_t> parent(static_cast<size_t>(V));
    std::iota(parent.begin(), parent.end(), 0);
    auto find = [&](int32_t x) {
        while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; }
        return x;
    };
    for (int64_t i = 0; i < npairs; ++i) {
        const int32_t v = pairs[i].v, w = pairs[i].w;
        if (v < 0 || w < 0 || v >= V || w >= V) return MS_ERR_ARG;
        if (v < first_candidate || w < first_candidate || pairs[i].relation != MS_LINKED) continue;
        const int32_t a = find(v), b = find(w);
        if (a != b) parent[std::max(a, b)] = std::min(a, b);     // the root is the component's smallest key
    }
    std::vector<int32_t> size(static_cast<size_t>(V), 0), id(static_cast<size_t>(V), -1);
    for (int32_t k = 0; k < V; ++k) size[find(k)]++;
    int32_t ng = 0;
    for (int32_t k = 0; k < V; ++k) {          // roots in key order: groups numbered by their smallest key
        const int32_t r = find(k);
        if (size[r] < 2) { group[k] = -1; continue; }
        if (id[r] < 0) id[r] = ng++;
        group[k] = id[r];
    }
    return ng;
}

}  // extern "C"
