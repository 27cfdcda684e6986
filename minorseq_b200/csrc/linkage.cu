// linkage.cu -- pairwise variant linkage (restatement choice U14; include/minorseq_b200.h "pairwise variant linkage").
//
// Phasing drops a read that is damaged at ANY called codon; linkage asks, per pair of called variants, only for the reads
// whose two codons are clean.  Everything a pair needs sits in one Gram matrix: phase_bits_kernel<true> writes the clean-codon
// matrix M beside the phasing bits B, and the existing co-occurrence contraction (popcount-AND, or tcgen05 int8 at size) runs
// over the stacked transpose [B | M] -- so G = [B|M]^T [B|M] holds B^T B, M^T M and the full B^T M.  With a communicator the
// Gram matrix is summed over the ranks once per phased read set; it is cached, so a capacity retry of ms_linkage neither
// recomputes nor re-reduces it.
//
// Statistics, fp64, one thread per upper-triangle pair, a block per row v:
//   linkage_count_kernel   m = the number of tested pairs (|col_v - col_w| >= 3, n >= min_reads)
//   linkage_test_kernel    both Fisher tails (linkage_tails), the small one stopped once it reaches alpha/m -> a significance bit
//                          per pair and the row's count
//   linkage_scan_kernel    row offsets (exclusive scan)
//   linkage_emit_kernel    the significant pairs of each row in w order at the row's offset (table, D', r^2, p-value)
// The order (v ascending, then w) and every value depend on the integer counts only: the same bytes on every run and rank.
#include <algorithm>
#include <vector>
#include "linkage_core.h"
#include "phase_internal.cuh"

int ms_gram_dev(ms_handle* h, const uint32_t* const* mats, int nmat, int32_t dim, int32_t* G);
int ms_comm_allreduce_i32(ms_handle* h, int32_t* d, size_t count);

namespace ms {

constexpr int kLinkThreads = 128;

struct LinkTable { uint32_t a, b, c, n; };

// the 2x2 table of pair (v, w) from the stacked Gram matrix (dim x dim, half = dim / 2)
__device__ __forceinline__ LinkTable link_table(const int32_t* __restrict__ G, int32_t dim, int32_t v, int32_t w) {
    const int32_t half = dim >> 1;
    LinkTable t;
    t.a = static_cast<uint32_t>(G[static_cast<size_t>(v) * dim + w]);
    t.n = static_cast<uint32_t>(G[static_cast<size_t>(half + v) * dim + half + w]);
    t.b = static_cast<uint32_t>(G[static_cast<size_t>(v) * dim + half + w]) - t.a;     // B_v . M_w - a
    t.c = static_cast<uint32_t>(G[static_cast<size_t>(w) * dim + half + v]) - t.a;     // M_v . B_w - a
    return t;
}

__device__ __forceinline__ bool link_tested(const int32_t* __restrict__ col, const LinkTable& t, int32_t v, int32_t w, int32_t min_reads) {
    const int32_t dc = col[v] - col[w];
    return (dc >= kLinkageMinSpacing || -dc >= kLinkageMinSpacing) && t.n >= static_cast<uint32_t>(min_reads);
}

// relation of a tested pair: 0, kLinkageLinked or kLinkageExclusive; *p = the p-value of that relation
__device__ __forceinline__ int link_test(const LinkTable& t, double alpha, double m, double* p) {
    const uint32_t d = t.n - t.a - t.b - t.c;
    const double enough = 1.000001 * alpha / m;     // the tails only have to be exact below alpha / m (as in K2)
    double pt, pa;
    linkage_tails(t.a, t.b, t.c, d, enough, &pt, &pa);
    if (pt * m < alpha) { *p = pt; return kLinkageLinked; }
    if (pa * m < alpha) { *p = pa; return kLinkageExclusive; }
    return 0;
}

// sum over the block; every thread gets the total
__device__ __forceinline__ unsigned long long link_block_sum(unsigned long long x) {
    __shared__ unsigned long long s_part[kLinkThreads / 32];
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    __syncthreads();                                            // s_part may still be read from the previous call
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = x;
    __syncthreads();
    unsigned long long t = 0;
#pragma unroll
    for (int i = 0; i < kLinkThreads / 32; ++i) t += s_part[i];
    return t;
}

__global__ void __launch_bounds__(kLinkThreads) linkage_count_kernel(const int32_t* __restrict__ G, int32_t dim, int32_t V,
                                                                    const int32_t* __restrict__ col, int32_t min_reads,
                                                                    unsigned long long* __restrict__ ctr) {
    const int32_t v = blockIdx.x;
    unsigned long long k = 0;
    for (int32_t w = v + 1 + threadIdx.x; w < V; w += kLinkThreads) k += link_tested(col, link_table(G, dim, v, w), v, w, min_reads) ? 1 : 0;
    k = link_block_sum(k);
    if (threadIdx.x == 0 && k) atomicAdd(ctr, k);
}

// sig: V rows of sw words, bit w of row v = pair (v, w) is significant
__global__ void __launch_bounds__(kLinkThreads) linkage_test_kernel(const int32_t* __restrict__ G, int32_t dim, int32_t V,
                                                                   const int32_t* __restrict__ col, int32_t min_reads, double alpha,
                                                                   const unsigned long long* __restrict__ ctr, uint32_t* __restrict__ sig,
                                                                   int32_t sw, int32_t* __restrict__ row_cnt) {
    const int32_t v = blockIdx.x;
    const double m = static_cast<double>(*ctr);
    unsigned long long k = 0;
    for (int32_t w0 = (v + 1) & ~31; w0 < V; w0 += kLinkThreads) {     // whole 32-pair words, so that a ballot is a word of `sig`
        const int32_t w = w0 + static_cast<int32_t>(threadIdx.x);
        bool s = false;
        if (w > v && w < V) {
            const LinkTable t = link_table(G, dim, v, w);
            double p;
            s = link_tested(col, t, v, w, min_reads) && link_test(t, alpha, m, &p) != 0;
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, s);
        if ((threadIdx.x & 31) == 0 && (w >> 5) < sw) sig[static_cast<size_t>(v) * sw + (w >> 5)] = bal;
        k += s ? 1 : 0;
    }
    k = link_block_sum(k);
    if (threadIdx.x == 0) row_cnt[v] = static_cast<int32_t>(k);
}

// exclusive scan of the row counts (one block of 1024 threads, contiguous segments); total -> ctr[1]
__global__ void __launch_bounds__(1024) linkage_scan_kernel(const int32_t* __restrict__ row_cnt, int32_t V, int64_t* __restrict__ row_off,
                                                            unsigned long long* __restrict__ ctr) {
    __shared__ long long s[1024];
    const int t = threadIdx.x;
    const int32_t per = (V + 1023) / 1024;
    const int32_t b = min(V, t * per), e = min(V, b + per);
    long long x = 0;
    for (int32_t i = b; i < e; ++i) x += row_cnt[i];
    s[t] = x;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {          // Hillis-Steele inclusive scan
        const long long y = t >= o ? s[t - o] : 0;
        __syncthreads();
        s[t] += y;
        __syncthreads();
    }
    long long off = s[t] - x;
    for (int32_t i = b; i < e; ++i) { row_off[i] = off; off += row_cnt[i]; }
    if (t == 1023) ctr[1] = static_cast<unsigned long long>(s[1023]);
}

__global__ void __launch_bounds__(kLinkThreads) linkage_emit_kernel(const int32_t* __restrict__ G, int32_t dim, int32_t V, double alpha,
                                                                   const unsigned long long* __restrict__ ctr, const uint32_t* __restrict__ sig,
                                                                   int32_t sw, const int64_t* __restrict__ row_off, ms_linkage_pair* __restrict__ out) {
    __shared__ int32_t s_warp[kLinkThreads / 32];
    const int32_t v = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double m = static_cast<double>(ctr[0]);
    int64_t pos = row_off[v];
    for (int32_t w0 = (v + 1) & ~31; w0 < V; w0 += kLinkThreads) {
        const int32_t w = w0 + static_cast<int32_t>(threadIdx.x);
        const uint32_t word = (w >> 5) < sw ? sig[static_cast<size_t>(v) * sw + (w >> 5)] : 0u;
        const bool s = w > v && w < V && ((word >> lane) & 1u);
        const uint32_t bal = __ballot_sync(0xffffffffu, s);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int32_t before = 0, total = 0;
#pragma unroll
        for (int i = 0; i < kLinkThreads / 32; ++i) { before += i < warp ? s_warp[i] : 0; total += s_warp[i]; }
        if (s) {
            const LinkTable t = link_table(G, dim, v, w);
            double dp, r2, p = 0.0;
            linkage_measures(t.a, t.b, t.c, t.n, &dp, &r2);
            const int rel = link_test(t, alpha, m, &p);
            ms_linkage_pair* o = out + pos + before + __popc(bal & ((1u << lane) - 1u));
            o->v = v; o->w = w;
            o->both = t.a; o->v_only = t.b; o->w_only = t.c; o->neither = t.n - t.a - t.b - t.c;
            o->d_prime = dp; o->r2 = r2; o->pvalue = p; o->relation = rel;
        }
        pos += total;
        __syncthreads();                          // s_warp is rewritten by the next chunk
    }
}

}  // namespace ms

namespace {

// the stacked Gram matrix of the current read set, computed and (with a communicator) all-reduced once
int linkage_gram(ms_handle* h) {
    if (!h || !h->b_bits.p) return MS_ERR_ARG;
    if (!h->link_ready) MS_FAIL(h, MS_ERR_ARG, "pairwise linkage: call ms_set_linkage(h, 1) before ms_phase_begin");
    if (h->gram_valid) return MS_OK;
    const int32_t dim = 64 * h->vwords;
    MS_CUDA(h, h->b_link_gram.ensure(static_cast<size_t>(dim) * dim * 4));
    const uint32_t* mats[2] = {h->b_bits.as<uint32_t>(), h->b_mbits.as<uint32_t>()};
    int rc = ms_gram_dev(h, mats, 2, dim, h->b_link_gram.as<int32_t>());
    if (rc != MS_OK) return rc;
    if (h->comm) {
        rc = ms_comm_allreduce_i32(h, h->b_link_gram.as<int32_t>(), static_cast<size_t>(dim) * dim);
        if (rc != MS_OK) return rc;
    }
    h->gram_valid = true;
    return MS_OK;
}

}  // namespace

extern "C" {

void ms_linkage_params_default(ms_linkage_params* p) {
    if (!p) return;
    p->alpha = 0.01;
    p->min_reads = ms::kLinkageMinReads;
}

int ms_set_linkage(ms_handle* h, int on) {
    if (!h) return MS_ERR_ARG;
    h->linkage = on != 0;
    return MS_OK;
}

int ms_linkage_device(ms_handle* h, int32_t** d_gram, int32_t* dim) {
    MsRange nvtx_range("linkage Gram");
    if (!h || !d_gram || !dim) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    const int rc = linkage_gram(h);
    if (rc != MS_OK) return rc;
    *d_gram = h->b_link_gram.as<int32_t>();
    *dim = 64 * h->vwords;
    return MS_OK;
}

int ms_linkage(ms_handle* h, const ms_linkage_params* prm, ms_linkage_pair* out, int64_t cap, int64_t* n, int64_t* ntested) {
    MsRange nvtx_range("linkage");
    if (!h || !prm || !n || cap < 0 || (cap > 0 && !out) || !(prm->alpha > 0.0) || prm->min_reads < 0) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    int rc = linkage_gram(h);
    if (rc != MS_OK) return rc;
    const int32_t V = h->V, dim = 64 * h->vwords, sw = std::max(1, (V + 31) / 32);
    if (static_cast<int32_t>(h->link_col.size()) != V) MS_FAIL(h, MS_ERR_ARG, "pairwise linkage: variant list changed");
    MS_CUDA(h, h->b_link_col.ensure(static_cast<size_t>(std::max(1, V)) * 4));
    MS_CUDA(h, h->b_link_sig.ensure(static_cast<size_t>(std::max(1, V)) * sw * 4));
    // [ctr: 2 x u64 | row counts: V x i32 | row offsets: V x i64]
    const size_t off_cnt = 16, off_row = off_cnt + ((static_cast<size_t>(V) * 4 + 15) & ~static_cast<size_t>(15));
    MS_CUDA(h, h->b_link_rows.ensure(off_row + static_cast<size_t>(std::max(1, V)) * 8));
    uint8_t* rows = h->b_link_rows.as<uint8_t>();
    unsigned long long* ctr = reinterpret_cast<unsigned long long*>(rows);
    int32_t* row_cnt = reinterpret_cast<int32_t*>(rows + off_cnt);
    int64_t* row_off = reinterpret_cast<int64_t*>(rows + off_row);
    rc = ms::phase_ensure_stage(h, 16);
    if (rc != MS_OK) return rc;
    MS_CUDA(h, cudaMemsetAsync(ctr, 0, 16, h->stream));
    if (V > 0) MS_CUDA(h, cudaMemcpyAsync(h->b_link_col.p, h->link_col.data(), static_cast<size_t>(V) * 4, cudaMemcpyHostToDevice, h->stream));
    MS_STAGE_BEGIN(h, MS_STAGE_LINKAGE_STATS);
    if (V > 1) {
        const int32_t* G = h->b_link_gram.as<int32_t>();
        const int32_t* col = h->b_link_col.as<int32_t>();
        ms::linkage_count_kernel<<<V, ms::kLinkThreads, 0, h->stream>>>(G, dim, V, col, prm->min_reads, ctr);
        ms::linkage_test_kernel<<<V, ms::kLinkThreads, 0, h->stream>>>(G, dim, V, col, prm->min_reads, prm->alpha, ctr, h->b_link_sig.as<uint32_t>(), sw,
                                                                      row_cnt);
        ms::linkage_scan_kernel<<<1, 1024, 0, h->stream>>>(row_cnt, V, row_off, ctr);
        h->launches += 3;
    }
    MS_STAGE_END(h, MS_STAGE_LINKAGE_STATS);
    uint64_t* st = static_cast<uint64_t*>(h->h_stage);
    MS_CUDA(h, cudaMemcpyAsync(st, ctr, 16, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    MS_CUDA(h, cudaGetLastError());
    const int64_t m = static_cast<int64_t>(st[0]), nsig = static_cast<int64_t>(st[1]);
    if (ntested) *ntested = m;
    *n = nsig;
    const int64_t k = std::min(cap, nsig);
    if (k > 0) {
        MS_CUDA(h, h->b_link_out.ensure(static_cast<size_t>(nsig) * sizeof(ms_linkage_pair)));
        ms::linkage_emit_kernel<<<V, ms::kLinkThreads, 0, h->stream>>>(h->b_link_gram.as<int32_t>(), dim, V, prm->alpha, ctr,
                                                                      h->b_link_sig.as<uint32_t>(), sw, row_off, h->b_link_out.as<ms_linkage_pair>());
        h->launches++;
        MS_CUDA(h, cudaMemcpyAsync(out, h->b_link_out.p, static_cast<size_t>(k) * sizeof(ms_linkage_pair), cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        MS_CUDA(h, cudaGetLastError());
    }
    return MS_OK;
}

}  // extern "C"
