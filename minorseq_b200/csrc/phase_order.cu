// phase_order.cu -- K3, second half: haplotype merge over ranks, juliet's haplotype order and the per-read
// haplotype id, all on the device (SURVEY.md rows a12 and 8e "phasing merge").
//
// juliet reports the haplotypes with at least 10 reads, named A, B, ... in descending read count
// (/root/reference/doc/JULIET.md:198-211, :253-254) and only tallies the rest (:372-381).  A phasing stress run
// (BASELINE.json config 5) has a few dozen reported haplotypes among hundreds of thousands of distinct
// single-read patterns, so the full (pattern, count) list never leaves the GPU here: the ranks' compact lists are
// all-gathered, merged in a second hash table, ranked (count descending, then ascending pattern words -- a total
// order, so every rank computes the same one), and the host receives the first `cap` entries plus the tallies.
//
// Ranking: up to kSmallSort distinct patterns are ranked by counting (rank = number of entries that precede,
// one thread per entry, no host round trip to learn the count); more go through a bitonic sort of entry indices.
#include <algorithm>
#include <cstring>
#include "phase_internal.cuh"

int ms_comm_allgather_bytes(ms_handle* h, const void* d_send, void* d_recv, size_t bytes_per_rank);

namespace ms {

constexpr uint32_t kSentinel = 0xffffffffu;
constexpr int kLocalSpan = 2048;   // elements one CTA of bitonic_local_kernel sorts in shared memory

__device__ __forceinline__ unsigned long long warp_sum64(unsigned long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// entry i takes position r; the whole warp calls (inactive lanes contribute nothing)
__device__ __forceinline__ void emit_ranked(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ pat, int32_t nw, int64_t i, uint32_t r,
                                            bool active, const OrderOut& o) {
    const uint32_t c = active ? cnt[i] : 0u;
    const bool rep = active && c >= o.min_reads;
    if (active) {
        o.rank[i] = r;
        if (static_cast<int64_t>(r) < o.ocap) {
            o.o_cnt[r] = c;
            for (int32_t w = 0; w < nw; ++w) o.o_pat[static_cast<size_t>(r) * nw + w] = pat[static_cast<size_t>(i) * nw + w];
        }
    }
    const unsigned long long nrep = __popc(__ballot_sync(0xffffffffu, rep));
    const unsigned long long srep = warp_sum64(rep ? c : 0u), sins = warp_sum64(rep ? 0u : c);
    if ((threadIdx.x & 31) == 0) {
        if (nrep) atomicAdd(o.res + 1, nrep);
        if (srep) atomicAdd(o.res + 2, srep);
        if (sins) atomicAdd(o.res + 3, sins);
    }
}

// Counting rank for M <= kSmallSort entries (M is read on the device).  Also copies the ranks' 64-byte headers
// behind the result header so that one device->host read brings everything the host has to look at.
__global__ void __launch_bounds__(256) rank_small_kernel(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ pat, int32_t nw,
                                                         const unsigned long long* __restrict__ Mptr, int64_t bound,
                                                         const uint8_t* __restrict__ hdr_src, size_t hdr_stride, int32_t world, OrderOut o) {
    const int64_t gid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (gid < world * 8)
        o.res[8 + gid] = reinterpret_cast<const unsigned long long*>(hdr_src + static_cast<size_t>(gid >> 3) * hdr_stride)[gid & 7];
    const int64_t M = static_cast<int64_t>(*Mptr);
    if (M > bound || M > kSmallSort) {
        if (gid == 0) o.res[4] = 1ULL;
        return;
    }
    const bool active = gid < M;
    uint32_t r = 0;
    if (active) {
        const uint32_t ci = cnt[gid];
        const uint32_t* pi = pat + static_cast<size_t>(gid) * nw;
        const uint32_t p0 = pi[0];
        for (int64_t j = 0; j < M; ++j) {
            const uint32_t cj = cnt[j];
            if (cj > ci) ++r;
            else if (cj == ci && j != gid) {
                const uint32_t q0 = pat[static_cast<size_t>(j) * nw];
                if (q0 != p0) r += q0 < p0;
                else if (nw > 1) r += pattern_less(pat + static_cast<size_t>(j) * nw, pi, nw);
            }
        }
    }
    emit_ranked(cnt, pat, nw, gid, r, active, o);
}

// The sort runs on (64-bit key, entry index) pairs: key = (~count) << 32 | pattern word 0, so that almost every
// comparison is decided in registers / shared memory; only equal keys look at the remaining pattern words.
__global__ void order_init_kernel(uint32_t* __restrict__ ord, unsigned long long* __restrict__ key, const uint32_t* __restrict__ cnt,
                                  const uint32_t* __restrict__ pat, int32_t nw, int64_t n_pad, int64_t M) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    if (i < M) {
        ord[i] = static_cast<uint32_t>(i);
        key[i] = (static_cast<unsigned long long>(~cnt[i]) << 32) | pat[static_cast<size_t>(i) * nw];   // count >= 1, so never all ones
    } else {
        ord[i] = kSentinel;
        key[i] = ~0ULL;
    }
}

__device__ __forceinline__ bool key_precedes(const uint32_t* __restrict__ pat, int32_t nw, unsigned long long ka, uint32_t a,
                                             unsigned long long kb, uint32_t b) {
    if (ka != kb) return ka < kb;
    if (nw == 1 || a == kSentinel) return false;   // distinct patterns differ in word 0 when there is only one word
    const uint32_t *pa = pat + static_cast<size_t>(a) * nw, *pb = pat + static_cast<size_t>(b) * nw;
    if ((nw & 3) == 0 && (reinterpret_cast<uintptr_t>(pat) & 15) == 0) {
        // patterns of a phasing stress run share long prefixes (a strain's sites plus a few flipped bits): 16 bytes per load
        const uint4 *qa = reinterpret_cast<const uint4*>(pa), *qb = reinterpret_cast<const uint4*>(pb);
        for (int32_t i = 0; i < nw / 4; ++i) {
            const uint4 x = qa[i], y = qb[i];
            if (x.x != y.x) return x.x < y.x;
            if (x.y != y.y) return x.y < y.y;
            if (x.z != y.z) return x.z < y.z;
            if (x.w != y.w) return x.w < y.w;
        }
        return false;
    }
    return pattern_less(pa + 1, pb + 1, nw - 1);
}

// all compare-exchange stages with distance < kLocalSpan of the merges k_begin..k_end, one CTA per kLocalSpan elements
__global__ void __launch_bounds__(kLocalSpan / 2) bitonic_local_kernel(uint32_t* __restrict__ ord, unsigned long long* __restrict__ key,
                                                                       const uint32_t* __restrict__ pat, int32_t nw, int64_t k_begin, int64_t k_end) {
    __shared__ unsigned long long sk[kLocalSpan];
    __shared__ uint32_t s[kLocalSpan];
    const int64_t base = static_cast<int64_t>(blockIdx.x) * kLocalSpan;
    const int t = threadIdx.x;
    s[t] = ord[base + t];
    s[t + kLocalSpan / 2] = ord[base + t + kLocalSpan / 2];
    sk[t] = key[base + t];
    sk[t + kLocalSpan / 2] = key[base + t + kLocalSpan / 2];
    __syncthreads();
    for (int64_t k = k_begin; k <= k_end; k <<= 1) {
        for (int j = (k >> 1) < kLocalSpan / 2 ? static_cast<int>(k >> 1) : kLocalSpan / 2; j > 0; j >>= 1) {
            const int i = 2 * t - (t & (j - 1)), l = i + j;
            const bool asc = ((base + i) & k) == 0;
            const uint32_t a = s[i], b = s[l];
            const unsigned long long ka = sk[i], kb = sk[l];
            if (asc ? key_precedes(pat, nw, kb, b, ka, a) : key_precedes(pat, nw, ka, a, kb, b)) {
                s[i] = b; s[l] = a;
                sk[i] = kb; sk[l] = ka;
            }
            __syncthreads();
        }
    }
    ord[base + t] = s[t];
    ord[base + t + kLocalSpan / 2] = s[t + kLocalSpan / 2];
    key[base + t] = sk[t];
    key[base + t + kLocalSpan / 2] = sk[t + kLocalSpan / 2];
}

__global__ void bitonic_global_kernel(uint32_t* __restrict__ ord, unsigned long long* __restrict__ key, const uint32_t* __restrict__ pat,
                                      int32_t nw, int64_t n_pad, int64_t k, int64_t j) {
    const int64_t t = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (t >= n_pad / 2) return;
    const int64_t i = 2 * t - (t & (j - 1)), l = i + j;
    const bool asc = (i & k) == 0;
    const uint32_t a = ord[i], b = ord[l];
    const unsigned long long ka = key[i], kb = key[l];
    if (asc ? key_precedes(pat, nw, kb, b, ka, a) : key_precedes(pat, nw, ka, a, kb, b)) {
        ord[i] = b; ord[l] = a;
        key[i] = kb; key[l] = ka;
    }
}

__global__ void __launch_bounds__(256) emit_sorted_kernel(const uint32_t* __restrict__ ord, const uint32_t* __restrict__ cnt,
                                                          const uint32_t* __restrict__ pat, int32_t nw, int64_t M, OrderOut o) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool active = i < M;
    emit_ranked(cnt, pat, nw, active ? ord[i] : 0, static_cast<uint32_t>(i), active, o);
}

// table slot of this rank's k-th compacted pattern -> its position in the (merged) order
__global__ void local_rank_kernel(const int32_t* __restrict__ g_slot, const unsigned long long* __restrict__ ng_ptr, int64_t gcap,
                                  const uint32_t* __restrict__ rank, const int32_t* __restrict__ mslot, const uint32_t* __restrict__ mindex,
                                  const unsigned long long* __restrict__ res, bool after_sort, int32_t* __restrict__ slot_rank) {
    if (!after_sort && res[4] != 0ULL) return;   // the counting rank declined: positions are not there yet
    const int64_t k = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t ng = static_cast<int64_t>(*ng_ptr);
    if (k >= ng || k >= gcap) return;
    if (mslot && mslot[k] < 0) return;   // merge table overflow, reported through res[6]
    const int64_t idx = mslot ? static_cast<int64_t>(mindex[mslot[k]]) : k;
    slot_rank[g_slot[k]] = static_cast<int32_t>(rank[idx]);
}

__global__ void hap_assign_kernel(const int32_t* __restrict__ slot, const int32_t* __restrict__ slot_rank, int64_t R, int32_t* __restrict__ hap) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= R) return;
    hap[r] = slot[r] < 0 ? -1 : slot_rank[slot[r]];
}

__global__ void merge_insert_kernel(Gathered g, int64_t bound, uint64_t seed, unsigned long long* mt_key, uint32_t* mt_cnt,
                                    unsigned long long* mt_rep, int64_t mask, int32_t* __restrict__ mslot, unsigned long long* res) {
    const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= bound) return;
    const int64_t rnk = e / g.gcap;
    if (e - rnk * g.gcap >= g.ng(rnk)) { mslot[e] = -1; return; }
    const uint64_t key = pattern_hash(g.pat(e), g.nw, seed);
    int64_t probe = static_cast<int64_t>(key) & mask, idx = -1;
    for (int64_t step = 0; step <= mask; ++step) {
        const unsigned long long prev = atomicCAS(mt_key + probe, 0ULL, static_cast<unsigned long long>(key));
        if (prev == 0ULL || prev == key) { idx = probe; break; }
        probe = (probe + 1) & mask;
    }
    mslot[e] = static_cast<int32_t>(idx);
    if (idx < 0) { atomicAdd(res + 6, 1ULL); return; }
    atomicAdd(mt_cnt + idx, g.cnt(e));
    atomicMin(mt_rep + idx, static_cast<unsigned long long>(e));
}

__global__ void merge_verify_kernel(Gathered g, int64_t bound, const unsigned long long* __restrict__ mt_rep, const int32_t* __restrict__ mslot,
                                    unsigned long long* res) {
    const int64_t e = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= bound || mslot[e] < 0) return;
    const int64_t rep = static_cast<int64_t>(mt_rep[mslot[e]]);
    if (rep == e) return;
    const uint32_t *a = g.pat(e), *b = g.pat(rep);
    for (int32_t i = 0; i < g.nw; ++i)
        if (a[i] != b[i]) { atomicAdd(res + 5, 1ULL); return; }
}

__global__ void merge_compact_kernel(Gathered g, const uint32_t* __restrict__ mt_cnt, const unsigned long long* __restrict__ mt_rep, int64_t tsize,
                                     unsigned long long* res, uint32_t* __restrict__ m_cnt, uint32_t* __restrict__ m_pat,
                                     uint32_t* __restrict__ m_index) {
    const int64_t s = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (s >= tsize || mt_cnt[s] == 0) return;
    const unsigned long long k = atomicAdd(res + 0, 1ULL);
    m_cnt[k] = mt_cnt[s];
    m_index[s] = static_cast<uint32_t>(k);
    const uint32_t* src = g.pat(static_cast<int64_t>(mt_rep[s]));
    for (int32_t w = 0; w < g.nw; ++w) m_pat[k * g.nw + w] = src[w];
}

}  // namespace ms

namespace {

inline unsigned grid_for(int64_t n, int block) { return static_cast<unsigned>(std::max<int64_t>(1, (n + block - 1) / block)); }

}  // namespace

namespace ms {

int sort_big(ms_handle* h, const uint32_t* cnt, const uint32_t* pat, int32_t nw, int64_t M, int64_t* n_pad_out) {
    int64_t n_pad = ms::kLocalSpan;
    while (n_pad < M) n_pad <<= 1;
    MS_CUDA(h, h->b_ord.ensure(static_cast<size_t>(n_pad) * 4));
    MS_CUDA(h, h->b_keys.ensure(static_cast<size_t>(n_pad) * 8));
    uint32_t* ord = h->b_ord.as<uint32_t>();
    unsigned long long* key = h->b_keys.as<unsigned long long>();
    ms::order_init_kernel<<<grid_for(n_pad, 256), 256, 0, h->stream>>>(ord, key, cnt, pat, nw, n_pad, M);
    const unsigned nloc = static_cast<unsigned>(n_pad / ms::kLocalSpan);
    ms::bitonic_local_kernel<<<nloc, ms::kLocalSpan / 2, 0, h->stream>>>(ord, key, pat, nw, 2, ms::kLocalSpan);
    h->launches += 2;
    for (int64_t k = 2 * ms::kLocalSpan; k <= n_pad; k <<= 1) {
        for (int64_t j = k >> 1; j >= ms::kLocalSpan; j >>= 1) {
            ms::bitonic_global_kernel<<<grid_for(n_pad / 2, 256), 256, 0, h->stream>>>(ord, key, pat, nw, n_pad, k, j);
            h->launches++;
        }
        ms::bitonic_local_kernel<<<nloc, ms::kLocalSpan / 2, 0, h->stream>>>(ord, key, pat, nw, k, k);
        h->launches++;
    }
    MS_CUDA(h, cudaGetLastError());
    *n_pad_out = n_pad;
    return MS_OK;
}

}  // namespace ms

using ms::sort_big;

extern "C" int ms_phase_haplotypes(ms_handle* h, int32_t min_reads, uint32_t* patterns, uint64_t* counts, int64_t cap, int64_t* H,
                                   int64_t* nreported, ms_phase_counters* ctr, int32_t* hap_id) {
    MsRange nvtx_range("K3 haplotypes (merge + order)");
    if (!h || !h->b_bits.p || !H || cap < 0 || (cap > 0 && (!patterns || !counts)) || min_reads < 0) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t nw = h->vwords;
    const int world = h->comm ? h->world : 1;
    const int me = h->comm ? h->rank : 0;
    // the size of the exchanged block must be the same on every rank: the hint is reset when a communicator is attached
    // (ms_comm_init, a collective itself) and from then on only changes by values all ranks compute from the same headers
    int64_t gcap = std::max<int64_t>(4096, h->gcap_hint);
    int attempt = h->table_valid ? h->table_attempt : 0;
    int merge_attempt = 0;
    unsigned long long* lctr = ms::phase_ctr(h);
    uint64_t marg[4] = {0, 0, 0, 0};
    int64_t M = 0, ocap = 0;
    size_t out_bytes = 0, first_copy = 0, off_cnt = 0, off_pat = 0;
    for (;;) {
        if (!h->table_valid) {
            int rc = ms::phase_build_table(h, attempt);
            if (rc != MS_OK) return rc;
        }
        const int64_t bound = gcap * world;
        if (bound > 0x7fffffffLL) MS_FAIL(h, MS_ERR_CAPACITY, "too many distinct read patterns to order");
        ocap = std::min<int64_t>(cap, bound);
        const size_t block = 64 + static_cast<size_t>(gcap) * 4 * (1 + nw);
        off_cnt = 64 + static_cast<size_t>(world) * 64;
        off_pat = off_cnt + static_cast<size_t>(ocap) * 4;
        out_bytes = off_pat + static_cast<size_t>(ocap) * nw * 4;
        MS_CUDA(h, h->b_groups.ensure(block));
        MS_CUDA(h, h->b_gslot.ensure(static_cast<size_t>(gcap) * 4));
        MS_CUDA(h, h->b_m_rank.ensure(static_cast<size_t>(bound) * 4));
        MS_CUDA(h, h->b_rank.ensure(static_cast<size_t>(h->tab_size) * 4));
        MS_CUDA(h, h->b_out.ensure(out_bytes));
        int rc = ms::phase_ensure_stage(h, out_bytes);
        if (rc != MS_OK) return rc;
        uint8_t* blk = h->b_groups.as<uint8_t>();
        uint32_t* g_cnt = reinterpret_cast<uint32_t*>(blk + 64);
        uint32_t* g_pat = g_cnt + gcap;
        uint8_t* outb = h->b_out.as<uint8_t>();
        ms::OrderOut o;
        o.res = reinterpret_cast<unsigned long long*>(outb);
        o.rank = h->b_m_rank.as<uint32_t>();
        o.o_cnt = reinterpret_cast<uint32_t*>(outb + off_cnt);
        o.o_pat = reinterpret_cast<uint32_t*>(outb + off_pat);
        o.ocap = ocap;
        o.min_reads = static_cast<uint32_t>(min_reads);
        MS_CUDA(h, cudaMemsetAsync(o.res, 0, 64, h->stream));
        rc = ms::phase_compact(h, g_cnt, g_pat, h->b_gslot.as<int32_t>(), gcap);
        if (rc != MS_OK) return rc;
        if (world > 1) MS_CUDA(h, cudaMemcpyAsync(blk, h->b_ctr.p, 64, cudaMemcpyDeviceToDevice, h->stream));   // header of the block to exchange

        // the list the order is computed over: this rank's own, or the merge of everybody's
        const uint32_t *v_cnt = g_cnt, *v_pat = g_pat;
        const unsigned long long* Mptr = lctr + 5;
        const uint8_t* hdr_src = reinterpret_cast<const uint8_t*>(lctr);   // single rank: the counters themselves are the header
        size_t hdr_stride = 0;
        const int32_t* mslot_me = nullptr;
        int64_t tsize = 0;
        if (world > 1) {
            tsize = 1024;
            while (tsize < 2 * bound) tsize <<= 1;
            MS_CUDA(h, h->b_gather.ensure(block * world));
            MS_CUDA(h, h->b_mt_key.ensure(static_cast<size_t>(tsize) * 8));
            MS_CUDA(h, h->b_mt_cnt.ensure(static_cast<size_t>(tsize) * 4));
            MS_CUDA(h, h->b_mt_rep.ensure(static_cast<size_t>(tsize) * 8));
            MS_CUDA(h, h->b_mindex.ensure(static_cast<size_t>(tsize) * 4));
            MS_CUDA(h, h->b_mslot.ensure(static_cast<size_t>(bound) * 4));
            MS_CUDA(h, h->b_m_cnt.ensure(static_cast<size_t>(bound) * 4));
            MS_CUDA(h, h->b_m_pat.ensure(static_cast<size_t>(bound) * nw * 4));
            // the one exchange of the phasing step: every rank's compact (pattern, count) list and marginals
            MS_STAGE_BEGIN(h, MS_STAGE_HAPMERGE);
            rc = ms_comm_allgather_bytes(h, blk, h->b_gather.p, block);
            if (rc != MS_OK) return rc;
            MS_CUDA(h, cudaMemsetAsync(h->b_mt_key.p, 0, static_cast<size_t>(tsize) * 8, h->stream));
            MS_CUDA(h, cudaMemsetAsync(h->b_mt_cnt.p, 0, static_cast<size_t>(tsize) * 4, h->stream));
            MS_CUDA(h, cudaMemsetAsync(h->b_mt_rep.p, 0x7f, static_cast<size_t>(tsize) * 8, h->stream));
            ms::Gathered g{h->b_gather.as<uint8_t>(), block, gcap, nw};
            ms::merge_insert_kernel<<<grid_for(bound, 256), 256, 0, h->stream>>>(g, bound, ms::phase_seed(100 + merge_attempt),
                                                                               h->b_mt_key.as<unsigned long long>(), h->b_mt_cnt.as<uint32_t>(),
                                                                               h->b_mt_rep.as<unsigned long long>(), tsize - 1,
                                                                               h->b_mslot.as<int32_t>(), o.res);
            ms::merge_verify_kernel<<<grid_for(bound, 256), 256, 0, h->stream>>>(g, bound, h->b_mt_rep.as<unsigned long long>(),
                                                                               h->b_mslot.as<int32_t>(), o.res);
            ms::merge_compact_kernel<<<grid_for(tsize, 256), 256, 0, h->stream>>>(g, h->b_mt_cnt.as<uint32_t>(), h->b_mt_rep.as<unsigned long long>(),
                                                                                tsize, o.res, h->b_m_cnt.as<uint32_t>(), h->b_m_pat.as<uint32_t>(),
                                                                                h->b_mindex.as<uint32_t>());
            h->launches += 3;
            MS_STAGE_END(h, MS_STAGE_HAPMERGE);
            v_cnt = h->b_m_cnt.as<uint32_t>();
            v_pat = h->b_m_pat.as<uint32_t>();
            Mptr = o.res;
            hdr_src = h->b_gather.as<uint8_t>();
            hdr_stride = block;
            mslot_me = h->b_mslot.as<int32_t>() + static_cast<size_t>(me) * gcap;
        }
        ms::rank_small_kernel<<<grid_for(std::min<int64_t>(bound, ms::kSmallSort), 256), 256, 0, h->stream>>>(v_cnt, v_pat, nw, Mptr, bound, hdr_src,
                                                                                                           hdr_stride, world, o);
        ms::local_rank_kernel<<<grid_for(gcap, 256), 256, 0, h->stream>>>(h->b_gslot.as<int32_t>(), lctr + 5, gcap, o.rank, mslot_me,
                                                                         h->b_mindex.as<uint32_t>(), o.res, false, h->b_rank.as<int32_t>());
        h->launches += 2;
        MS_CUDA(h, cudaGetLastError());
        uint8_t* st = static_cast<uint8_t*>(h->h_stage);
        first_copy = std::min<size_t>(out_bytes, 96 * 1024);
        MS_CUDA(h, cudaMemcpyAsync(st, outb, first_copy, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));

        // every rank sees every header, so all ranks take the same branch below
        uint64_t res[8];
        memcpy(res, st, 64);
        bool any_collision = false, any_overflow = false;
        int64_t max_ng = 0;
        for (int r = 0; r < world; ++r) {
            uint64_t hc[8];
            memcpy(hc, st + 64 + static_cast<size_t>(r) * 64, 64);
            if ((hc[6] != 0 || hc[4] != 0) && (hc[7] & 0xff) != 0)   // rank r cannot recover (header's spare word, phase_build_table): every rank stops here
                MS_FAIL(h, MS_ERR_CUDA, hc[6] != 0 ? "haplotype table overflow at maximum size" : "haplotype hash collided under four seeds");
            if (hc[6] != 0) {
                any_overflow = true;
                if (r == me) { rc = ms::phase_grow_table(h); if (rc != MS_OK) return rc; }
            } else if (hc[4] != 0) {
                any_collision = true;
                if (r == me) {  // a 64-bit hash collision between different patterns here: re-hash with another seed
                    ++attempt;
                    h->table_valid = false;
                }
            } else if (r == me) {
                h->table_valid = true;
            }
            max_ng = std::max<int64_t>(max_ng, static_cast<int64_t>(hc[5]));
            if (r == 0) memset(marg, 0, sizeof marg);
            for (int i = 0; i < 4; ++i) marg[i] += hc[i];
        }
        if (any_collision || any_overflow) continue;
        if (max_ng > gcap) { gcap = (max_ng + 3) & ~int64_t(3); h->gcap_hint = gcap; continue; }   // multiple of 4: pattern rows stay 16-byte aligned
        if (res[6] != 0) MS_FAIL(h, MS_ERR_CUDA, "haplotype merge table overflow");
        if (res[5] != 0) {
            if (++merge_attempt >= 4) MS_FAIL(h, MS_ERR_CUDA, "haplotype merge hash collided under four seeds");
            continue;
        }
        M = world > 1 ? static_cast<int64_t>(res[0]) : max_ng;
        if (res[4] != 0) {
            // more than kSmallSort distinct patterns: sort the entry indices, then emit in order
            int64_t n_pad = 0;
            rc = sort_big(h, v_cnt, v_pat, nw, M, &n_pad);
            if (rc != MS_OK) return rc;
            ms::emit_sorted_kernel<<<grid_for(M, 256), 256, 0, h->stream>>>(h->b_ord.as<uint32_t>(), v_cnt, v_pat, nw, M, o);
            ms::local_rank_kernel<<<grid_for(gcap, 256), 256, 0, h->stream>>>(h->b_gslot.as<int32_t>(), lctr + 5, gcap, o.rank, mslot_me,
                                                                             h->b_mindex.as<uint32_t>(), o.res, true, h->b_rank.as<int32_t>());
            h->launches += 2;
            MS_CUDA(h, cudaGetLastError());
            MS_CUDA(h, cudaMemcpyAsync(st, outb, first_copy, cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
            memcpy(res, st, 64);
        }
        *H = M;
        if (nreported) *nreported = static_cast<int64_t>(res[1]);
        if (ctr) {
            ctr->reported = res[2]; ctr->insufficient = res[3];
            ctr->damaged = marg[0]; ctr->gaps = marg[1]; ctr->heteroduplex = marg[2]; ctr->partial = marg[3];
        }
        break;
    }
    // the ordered prefix the caller asked for
    const int64_t need = std::min<int64_t>(ocap, M);
    uint8_t* st = static_cast<uint8_t*>(h->h_stage);
    const uint8_t* outb = h->b_out.as<uint8_t>();
    bool pending = false;
    if (need > 0 && off_pat + static_cast<size_t>(need) * nw * 4 > first_copy) {
        if (off_cnt + static_cast<size_t>(need) * 4 > first_copy)
            MS_CUDA(h, cudaMemcpyAsync(st + off_cnt, outb + off_cnt, static_cast<size_t>(need) * 4, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(st + off_pat, outb + off_pat, static_cast<size_t>(need) * nw * 4, cudaMemcpyDeviceToHost, h->stream));
        pending = true;
    }
    if (hap_id && h->phase_n > 0) {
        MS_CUDA(h, h->b_hap.ensure(static_cast<size_t>(h->phase_n) * 4));
        ms::hap_assign_kernel<<<grid_for(h->phase_n, 256), 256, 0, h->stream>>>(h->b_slot.as<int32_t>(), h->b_rank.as<int32_t>(), h->phase_n,
                                                                               h->b_hap.as<int32_t>());
        h->launches++;
        MS_CUDA(h, cudaMemcpyAsync(hap_id, h->b_hap.p, static_cast<size_t>(h->phase_n) * 4, cudaMemcpyDeviceToHost, h->stream));
        pending = true;
    }
    if (pending) MS_CUDA(h, cudaStreamSynchronize(h->stream));
    MS_CUDA(h, cudaGetLastError());
    h->hap_ranked = true;
    h->hap_assigned = hap_id && h->phase_n > 0;
    if (need > 0) {
        memcpy(patterns, st + off_pat, static_cast<size_t>(need) * nw * 4);
        const uint32_t* c = reinterpret_cast<const uint32_t*>(st + off_cnt);
        for (int64_t i = 0; i < need; ++i) counts[i] = c[i];
    }
    return MS_OK;
}

// The per-read positions in the order of the last ms_phase_haplotypes, on the device (b_hap); hap_assign_kernel runs here when
// that call was made without hap_id.
extern "C" int ms_phase_hap_device(ms_handle* h, int32_t** d_hap, int64_t* R) {
    if (!h || !d_hap || !R) return MS_ERR_ARG;
    if (!h->hap_ranked) MS_FAIL(h, MS_ERR_ARG, "ms_phase_hap_device: call ms_phase_haplotypes on the phased reads first");
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, h->b_hap.ensure(static_cast<size_t>(std::max<int64_t>(1, h->phase_n)) * 4));
    if (!h->hap_assigned && h->phase_n > 0) {
        ms::hap_assign_kernel<<<grid_for(h->phase_n, 256), 256, 0, h->stream>>>(h->b_slot.as<int32_t>(), h->b_rank.as<int32_t>(), h->phase_n,
                                                                               h->b_hap.as<int32_t>());
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
        h->hap_assigned = true;
    }
    *d_hap = h->b_hap.as<int32_t>();
    *R = h->phase_n;
    return MS_OK;
}
