// abundance.cu -- haplotype abundance (restatement choice U18; include/minorseq_b200.h "haplotype abundance").
//
// Phasing counts a haplotype's reads among the reads that are clean at every key.  Abundance fits every phased read to the
// given patterns instead: read r is compatible with pattern h when they agree at every key where r is clean (M, the
// clean-codon matrix linkage added), and the frequencies are the maximum-likelihood estimate over those compatibility sets.
//
//   abundance_compat_kernel   one lane per read: its compatibility mask (ceil(H/32) words) and a flag byte, non-zero for
//                             the incompatible and the uninformative reads, which the EM does not need; their counts
//   phase_insert/verify/compact_kernel (phase.cu), on the masks at width ceil(H/32): the distinct masks ("classes") and
//                             their read counts.  The flag byte keeps the two skipped categories out of the table.
//   merge_*_kernel, rank_small_kernel / sort_big (phase_order.cu): the ranks' class lists all-gathered and merged, then
//                             totally ordered (count desc, then ascending mask words), as phasing orders its patterns
//   abundance_stats_kernel    per-haplotype compatible and unique reads from the ordered classes (integer sums)
//   abundance_denom_kernel    per class: sum of pi over its haplotypes, ascending h
//   abundance_sum_kernel      per haplotype: sum over the classes of count / denominator, fixed-order block sums over fixed
//                             class slices; the last block to finish adds the slices in order, updates pi and decides
//                             convergence on the device.  The host looks at the state every kEmBatch iterations.
//   abundance_loglik_kernel   sum over the classes of count * log(denominator), one block, fixed order
// No floating-point atomics, and launch shapes depend only on H and the number of classes: the result is bit-identical for
// any number of GPUs.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>
#include <vector>
#include "phase_internal.cuh"

int ms_comm_allgather_bytes(ms_handle* h, const void* d_send, void* d_recv, size_t bytes_per_rank);

namespace ms {

constexpr int kMaxPatterns = 4096;
constexpr int kCompatWarps = 4;     // 128 reads per CTA, one per lane
constexpr int kCompatAcc = 8;       // mask words a lane keeps in registers: 256 patterns per pass over the rows
constexpr int kCompatWords = 16;    // row words staged per step (64-byte row pieces, two reads per warp load)
constexpr int kEmThreads = 256;
constexpr int64_t kEmSlice = 2048;  // classes per block of abundance_sum_kernel
constexpr int kEmBatch = 32;        // iterations enqueued between two host looks at the EM state

// abundance counters, also the 64-byte header the ranks exchange (Gathered::ng reads word 5):
// [0] incompatible reads  [1] uninformative reads  [4] class hash collisions  [5] classes  [6] class table overflow
// [7] phase_clear_kernel's "last resort" word (unused here)

struct EmState {
    unsigned int arrive;   // blocks of abundance_sum_kernel done with this iteration
    int32_t iter, done, converged;
};

__global__ void __launch_bounds__(kCompatWarps * 32) abundance_compat_kernel(const uint32_t* __restrict__ B, const uint32_t* __restrict__ Mb,
                                                                             int64_t R, int32_t vwords, const uint32_t* __restrict__ pat, int32_t H,
                                                                             int32_t hw, uint32_t* __restrict__ mask, uint8_t* __restrict__ flag,
                                                                             unsigned long long* __restrict__ ctr) {
    __shared__ uint32_t sB[kCompatWarps][32][kCompatWords + 1], sM[kCompatWarps][32][kCompatWords + 1];
    __shared__ uint32_t sP[kCompatAcc * 32][kCompatWords];   // read as a broadcast: no padding
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t rw = static_cast<int64_t>(blockIdx.x) * (kCompatWarps * 32) + warp * 32;   // this warp's first read
    const int64_t r = rw + lane;
    int32_t pop = 0;
    for (int32_t h0 = 0; h0 < H; h0 += kCompatAcc * 32) {
        const int32_t nh = min(H - h0, kCompatAcc * 32);
        uint32_t acc[kCompatAcc];
#pragma unroll
        for (int k = 0; k < kCompatAcc; ++k) {
            const int32_t left = nh - k * 32;
            acc[k] = left >= 32 ? ~0u : left > 0 ? (1u << left) - 1u : 0u;
        }
        for (int32_t w0 = 0; w0 < vwords; w0 += kCompatWords) {
            const int32_t nw = min(kCompatWords, vwords - w0);
            __syncthreads();   // the previous step's rows and patterns are consumed
            for (int i = threadIdx.x; i < nh * kCompatWords; i += kCompatWarps * 32) {
                const int j = i / kCompatWords, w = i % kCompatWords;
                sP[j][w] = w < nw ? pat[static_cast<size_t>(h0 + j) * vwords + w0 + w] : 0u;
            }
            for (int i = lane >> 4; i < 32; i += 2) {
                const int w = lane & (kCompatWords - 1);
                const int64_t rr = rw + i;
                const bool ok = rr < R && w < nw;
                sB[warp][i][w] = ok ? B[static_cast<size_t>(rr) * vwords + w0 + w] : 0u;
                sM[warp][i][w] = ok ? Mb[static_cast<size_t>(rr) * vwords + w0 + w] : 0u;
            }
            __syncthreads();
            for (int w = 0; w < nw; ++w) {
                const uint32_t b = sB[warp][lane][w], m = sM[warp][lane][w];
                if (m == 0u) continue;
#pragma unroll
                for (int k = 0; k < kCompatAcc; ++k) {
                    if (k * 32 < nh) {
                        uint32_t a = acc[k];
#pragma unroll 8
                        for (int j = 0; j < 32; ++j) a &= ((b ^ sP[k * 32 + j][w]) & m) ? ~(1u << j) : ~0u;
                        acc[k] = a;
                    }
                }
            }
        }
        if (r < R) {
#pragma unroll
            for (int k = 0; k < kCompatAcc; ++k)
                if (k * 32 < nh) {
                    mask[static_cast<size_t>(r) * hw + (h0 >> 5) + k] = acc[k];
                    pop += __popc(acc[k]);
                }
        }
    }
    const bool incompatible = r < R && pop == 0, uninformative = r < R && H >= 2 && pop == H;
    if (r < R) flag[r] = (incompatible || uninformative) ? 1 : 0;
    const unsigned n0 = __popc(__ballot_sync(0xffffffffu, incompatible)), n1 = __popc(__ballot_sync(0xffffffffu, uninformative));
    if (lane == 0) {
        if (n0) atomicAdd(ctr + 0, static_cast<unsigned long long>(n0));
        if (n1) atomicAdd(ctr + 1, static_cast<unsigned long long>(n1));
    }
}

// per haplotype: reads of the classes that contain it, and of the classes that contain only it
__global__ void abundance_stats_kernel(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ pat, int32_t hw, int64_t M,
                                       unsigned long long* __restrict__ compat, unsigned long long* __restrict__ uniq) {
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= M) return;
    const uint32_t* p = pat + static_cast<size_t>(c) * hw;
    const unsigned long long n = cnt[c];
    int pop = 0;
    for (int32_t w = 0; w < hw; ++w) pop += __popc(p[w]);
    for (int32_t w = 0; w < hw; ++w)
        for (uint32_t x = p[w]; x; x &= x - 1) {
            const int h = w * 32 + __ffs(x) - 1;
            atomicAdd(compat + h, n);
            if (pop == 1) atomicAdd(uniq + h, n);
        }
}

// d[c] = sum of pi over the haplotypes of class c, ascending h
__global__ void abundance_denom_kernel(const uint32_t* __restrict__ pat, int32_t hw, int64_t M, const double* __restrict__ pi,
                                       double* __restrict__ d, const EmState* __restrict__ st, int always) {
    if (!always && st->done) return;
    const int64_t c = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= M) return;
    const uint32_t* p = pat + static_cast<size_t>(c) * hw;
    double s = 0.0;
    for (int32_t w = 0; w < hw; ++w)
        for (uint32_t x = p[w]; x; x &= x - 1) s += pi[w * 32 + __ffs(x) - 1];
    d[c] = s;
}

// grid (hw, slices): block (w, s) sums count / d over the classes of slice s for the 32 haplotypes of mask word w, into
// part[s][32 w + j]; the last block adds the slices in order: pi_h *= sum / N, and the convergence test
__global__ void __launch_bounds__(kEmThreads) abundance_sum_kernel(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ pat, int32_t hw,
                                                                   int64_t M, const double* __restrict__ d, double* __restrict__ part,
                                                                   double* __restrict__ pi, int32_t H, double N, double tol, int32_t max_it,
                                                                   EmState* __restrict__ st) {
    __shared__ double s_w[kEmThreads / 32][32];
    __shared__ bool s_last;
    if (st->done) return;
    const int32_t wi = blockIdx.x;
    const int64_t c0 = static_cast<int64_t>(blockIdx.y) * kEmSlice, c1 = min(M, c0 + kEmSlice);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double acc[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) acc[j] = 0.0;
    for (int64_t c = c0 + threadIdx.x; c < c1; c += kEmThreads) {
        const uint32_t x = pat[static_cast<size_t>(c) * hw + wi];
        if (!x) continue;
        const double wgt = static_cast<double>(cnt[c]) / d[c];
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] += ((x >> j) & 1u) ? wgt : 0.0;
    }
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        double v = acc[j];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == j) s_w[warp][j] = v;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < kEmThreads / 32; ++k) v += s_w[k][threadIdx.x];
        part[static_cast<size_t>(blockIdx.y) * hw * 32 + wi * 32 + threadIdx.x] = v;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&st->arrive, 1u) == gridDim.x * gridDim.y - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    __shared__ double s_max[kEmThreads];
    double mx = 0.0;
    const int32_t S = gridDim.y;
    for (int32_t h = threadIdx.x; h < H; h += kEmThreads) {
        double sum = 0.0;
        for (int32_t s = 0; s < S; ++s) sum += __ldcg(part + static_cast<size_t>(s) * hw * 32 + h);
        const double old = pi[h], nxt = old * sum / N;
        pi[h] = nxt;
        mx = fmax(mx, fabs(nxt - old));
    }
    s_max[threadIdx.x] = mx;
    __syncthreads();
    for (int o = kEmThreads / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) s_max[threadIdx.x] = fmax(s_max[threadIdx.x], s_max[threadIdx.x + o]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const int32_t it = st->iter + 1;
        st->iter = it;
        if (s_max[0] < tol) { st->converged = 1; st->done = 1; }
        else if (it >= max_it) st->done = 1;
        st->arrive = 0u;
        __threadfence();
    }
}

__global__ void __launch_bounds__(1024) abundance_loglik_kernel(const uint32_t* __restrict__ cnt, const double* __restrict__ d, int64_t M,
                                                                double* __restrict__ out) {
    __shared__ double s[1024];
    double x = 0.0;
    for (int64_t c = threadIdx.x; c < M; c += 1024) x += static_cast<double>(cnt[c]) * log(d[c]);
    s[threadIdx.x] = x;
    __syncthreads();
    for (int o = 512; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = s[0];
}

__global__ void abundance_init_kernel(double* __restrict__ pi, int32_t H, EmState* __restrict__ st) {
    const int32_t h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h < H) pi[h] = 1.0 / static_cast<double>(H);
    if (h == 0) { st->arrive = 0u; st->iter = 0; st->done = 0; st->converged = 0; }
}

}  // namespace ms

namespace {

inline unsigned grid_for(int64_t n, int block) { return static_cast<unsigned>(std::max<int64_t>(1, (n + block - 1) / block)); }
inline size_t align16(size_t x) { return (x + 15) & ~static_cast<size_t>(15); }

}  // namespace

extern "C" {

void ms_abundance_params_default(ms_abundance_params* p) {
    if (!p) return;
    p->tolerance = 1e-10;
    p->max_iterations = 10000;
}

int ms_set_abundance(ms_handle* h, int on) {
    if (!h) return MS_ERR_ARG;
    h->abundance = on != 0;
    return MS_OK;
}

int ms_haplotype_abundance(ms_handle* h, const ms_abundance_params* prm, const uint32_t* patterns, int64_t H, ms_abundance_row* rows,
                           int64_t cap, ms_abundance_counters* counters, int32_t* iterations, int32_t* converged, double* loglik) {
    MsRange nvtx_range("haplotype abundance");
    if (!h || !prm || H < 0 || (H > 0 && !patterns) || cap < 0 || (cap > 0 && !rows) || !(prm->tolerance >= 0.0) ||
        !std::isfinite(prm->tolerance) || prm->max_iterations < 1)
        return MS_ERR_ARG;
    if (H > ms::kMaxPatterns) MS_FAIL(h, MS_ERR_ARG, "haplotype abundance: more than 4096 patterns");
    if (!h->b_bits.p) MS_FAIL(h, MS_ERR_ARG, "haplotype abundance: no phased reads");
    if (!h->link_ready) MS_FAIL(h, MS_ERR_ARG, "haplotype abundance: call ms_set_abundance(h, 1) before ms_phase_begin");
    if (cap < H) MS_FAIL(h, MS_ERR_CAPACITY, "haplotype abundance: rows_out holds fewer rows than patterns");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t V = h->V, vw = h->vwords;
    const int32_t Hn = static_cast<int32_t>(H), hw = std::max(1, (Hn + 31) / 32);
    const int64_t R = h->phase_n;

    // the patterns with the bits >= V cleared; duplicates are refused
    std::vector<uint32_t> pat(static_cast<size_t>(H) * vw);
    for (int64_t k = 0; k < H; ++k)
        for (int32_t w = 0; w < vw; ++w) {
            const int32_t keep = std::min(32, std::max(0, V - 32 * w));
            const uint32_t m = keep >= 32 ? ~0u : (1u << keep) - 1u;
            pat[static_cast<size_t>(k) * vw + w] = patterns[static_cast<size_t>(k) * vw + w] & m;
        }
    {
        std::vector<int32_t> idx(static_cast<size_t>(H));
        std::iota(idx.begin(), idx.end(), 0);
        auto row = [&](int32_t k) { return pat.data() + static_cast<size_t>(k) * vw; };
        std::sort(idx.begin(), idx.end(), [&](int32_t a, int32_t b) { return ms::pattern_less(row(a), row(b), vw); });
        for (size_t i = 1; i < idx.size(); ++i)
            if (!ms::pattern_less(row(idx[i - 1]), row(idx[i]), vw)) MS_FAIL(h, MS_ERR_ARG, "haplotype abundance: duplicate patterns");
    }

    const int world = h->comm ? h->world : 1;
    const size_t hpad = static_cast<size_t>(hw) * 32;
    // EM buffer: [state 64 B | pi: 32 hw | compat, unique: u64 32 hw each | loglik | d: classes | part: slices x 32 hw]; the
    // pinned stage takes the patterns, the ranks' headers and the EM's results: sized once, nothing is in flight when it grows
    const size_t off_pi = 64, off_cmp = off_pi + hpad * 8, off_unq = off_cmp + hpad * 8, off_ll = off_unq + hpad * 8, off_d = off_ll + 16;
    int rc = ms::phase_ensure_stage(h, std::max({pat.size() * 4, 64 + static_cast<size_t>(world) * 64, off_d}));
    if (rc != MS_OK) return rc;
    MS_CUDA(h, h->b_ab_pat.ensure(std::max<size_t>(4, pat.size() * 4)));
    MS_CUDA(h, h->b_ab_mask.ensure(static_cast<size_t>(std::max<int64_t>(1, R)) * hw * 4));
    MS_CUDA(h, h->b_ab_flag.ensure(static_cast<size_t>(std::max<int64_t>(1, R))));
    MS_CUDA(h, h->b_ab_slot.ensure(static_cast<size_t>(std::max<int64_t>(1, R)) * 4));
    MS_CUDA(h, h->b_ab_ctr.ensure(64));
    unsigned long long* ctr = h->b_ab_ctr.as<unsigned long long>();
    if (!pat.empty()) {
        memcpy(h->h_stage, pat.data(), pat.size() * 4);
        MS_CUDA(h, cudaMemcpyAsync(h->b_ab_pat.p, h->h_stage, pat.size() * 4, cudaMemcpyHostToDevice, h->stream));
    }
    MS_CUDA(h, cudaMemsetAsync(ctr, 0, 64, h->stream));
    MS_STAGE_BEGIN(h, MS_STAGE_ABUNDANCE_COMPAT);
    if (R > 0) {
        ms::abundance_compat_kernel<<<grid_for(R, ms::kCompatWarps * 32), ms::kCompatWarps * 32, 0, h->stream>>>(
            h->b_bits.as<uint32_t>(), h->b_mbits.as<uint32_t>(), R, vw, h->b_ab_pat.as<uint32_t>(), Hn, hw, h->b_ab_mask.as<uint32_t>(),
            h->b_ab_flag.as<uint8_t>(), ctr);
        h->launches++;
    }
    MS_STAGE_END(h, MS_STAGE_ABUNDANCE_COMPAT);
    MS_CUDA(h, cudaGetLastError());

    // classes: group the masks (phasing's table), merge over the ranks, order.  Every rank sees every header, so every rank
    // takes the same turns through this loop.
    int64_t ts = 1024;
    while (ts < 2 * R) ts <<= 1;
    int64_t gcap = world == 1 ? std::max<int64_t>(4, (R + 3) & ~int64_t(3)) : 4096;   // a multiple of 4: rows stay 16-byte aligned
    int attempt = 0, merge_attempt = 0;
    int64_t M = 0;
    size_t off_cnt = 0, off_pat = 0;
    uint64_t cat[2] = {0, 0};   // incompatible, uninformative over all ranks
    uint64_t res[8];
    const uint32_t* v_cnt = nullptr;
    const uint32_t* v_pat = nullptr;
    ms::OrderOut o;
    for (;;) {
        const int64_t bound = gcap * world;
        if (bound > 0x7fffffffLL) MS_FAIL(h, MS_ERR_CAPACITY, "haplotype abundance: too many compatibility classes to order");
        const size_t block = 64 + static_cast<size_t>(gcap) * 4 * (1 + hw);
        off_cnt = 64 + static_cast<size_t>(world) * 64;
        off_pat = align16(off_cnt + static_cast<size_t>(bound) * 4);
        const size_t out_bytes = off_pat + static_cast<size_t>(bound) * hw * 4;
        MS_CUDA(h, h->b_ab_tab_key.ensure(static_cast<size_t>(ts) * 8));
        MS_CUDA(h, h->b_ab_tab_cnt.ensure(static_cast<size_t>(ts) * 4));
        MS_CUDA(h, h->b_ab_tab_rep.ensure(static_cast<size_t>(ts) * 8));
        MS_CUDA(h, h->b_ab_blk.ensure(block));
        MS_CUDA(h, h->b_ab_out.ensure(out_bytes));
        MS_CUDA(h, h->b_m_rank.ensure(static_cast<size_t>(bound) * 4));
        uint8_t* blk = h->b_ab_blk.as<uint8_t>();
        uint32_t* g_cnt = reinterpret_cast<uint32_t*>(blk + 64);
        uint32_t* g_pat = g_cnt + gcap;
        uint8_t* outb = h->b_ab_out.as<uint8_t>();
        o.res = reinterpret_cast<unsigned long long*>(outb);
        o.rank = h->b_m_rank.as<uint32_t>();
        o.o_cnt = reinterpret_cast<uint32_t*>(outb + off_cnt);
        o.o_pat = reinterpret_cast<uint32_t*>(outb + off_pat);
        o.ocap = bound;
        o.min_reads = 0;
        MS_CUDA(h, cudaMemsetAsync(o.res, 0, 64, h->stream));
        ms::phase_clear_kernel<<<static_cast<int>(std::min<int64_t>((ts + 255) / 256, static_cast<int64_t>(h->num_sms) * 8)), 256, 0, h->stream>>>(
            h->b_ab_tab_key.as<unsigned long long>(), h->b_ab_tab_cnt.as<uint32_t>(), h->b_ab_tab_rep.as<long long>(), ts, ctr, 0ULL);
        h->launches++;
        if (R > 0) {
            ms::phase_insert_kernel<<<grid_for(R, 256), 256, 0, h->stream>>>(h->b_ab_mask.as<uint32_t>(), h->b_ab_flag.as<uint8_t>(), R, hw,
                                                                             ms::phase_seed(200 + attempt), h->b_ab_tab_key.as<unsigned long long>(),
                                                                             h->b_ab_tab_cnt.as<uint32_t>(), h->b_ab_tab_rep.as<long long>(), ts - 1,
                                                                             h->b_ab_slot.as<int32_t>(), ctr + 6);
            ms::phase_verify_kernel<<<grid_for(R, 256), 256, 0, h->stream>>>(h->b_ab_mask.as<uint32_t>(), R, hw, h->b_ab_tab_rep.as<long long>(),
                                                                             h->b_ab_slot.as<int32_t>(), ctr + 4);
            h->launches += 2;
        }
        MS_CUDA(h, cudaMemsetAsync(ctr + 5, 0, 8, h->stream));
        ms::phase_compact_kernel<<<grid_for(ts, 256), 256, 0, h->stream>>>(h->b_ab_tab_cnt.as<uint32_t>(), h->b_ab_tab_rep.as<long long>(), ts,
                                                                           h->b_ab_mask.as<uint32_t>(), hw, ctr + 5, g_cnt, g_pat, nullptr, gcap);
        h->launches++;
        v_cnt = g_cnt;
        v_pat = g_pat;
        const unsigned long long* Mptr = ctr + 5;
        const uint8_t* hdr_src = reinterpret_cast<const uint8_t*>(ctr);
        size_t hdr_stride = 0;
        if (world > 1) {
            int64_t tsize = 1024;
            while (tsize < 2 * bound) tsize <<= 1;
            MS_CUDA(h, cudaMemcpyAsync(blk, ctr, 64, cudaMemcpyDeviceToDevice, h->stream));
            MS_CUDA(h, h->b_gather.ensure(block * world));
            MS_CUDA(h, h->b_mt_key.ensure(static_cast<size_t>(tsize) * 8));
            MS_CUDA(h, h->b_mt_cnt.ensure(static_cast<size_t>(tsize) * 4));
            MS_CUDA(h, h->b_mt_rep.ensure(static_cast<size_t>(tsize) * 8));
            MS_CUDA(h, h->b_mindex.ensure(static_cast<size_t>(tsize) * 4));
            MS_CUDA(h, h->b_mslot.ensure(static_cast<size_t>(bound) * 4));
            MS_CUDA(h, h->b_m_cnt.ensure(static_cast<size_t>(bound) * 4));
            MS_CUDA(h, h->b_m_pat.ensure(static_cast<size_t>(bound) * hw * 4));
            rc = ms_comm_allgather_bytes(h, blk, h->b_gather.p, block);
            if (rc != MS_OK) return rc;
            MS_CUDA(h, cudaMemsetAsync(h->b_mt_key.p, 0, static_cast<size_t>(tsize) * 8, h->stream));
            MS_CUDA(h, cudaMemsetAsync(h->b_mt_cnt.p, 0, static_cast<size_t>(tsize) * 4, h->stream));
            MS_CUDA(h, cudaMemsetAsync(h->b_mt_rep.p, 0x7f, static_cast<size_t>(tsize) * 8, h->stream));
            ms::Gathered g{h->b_gather.as<uint8_t>(), block, gcap, hw};
            ms::merge_insert_kernel<<<grid_for(bound, 256), 256, 0, h->stream>>>(g, bound, ms::phase_seed(300 + merge_attempt),
                                                                               h->b_mt_key.as<unsigned long long>(), h->b_mt_cnt.as<uint32_t>(),
                                                                               h->b_mt_rep.as<unsigned long long>(), tsize - 1, h->b_mslot.as<int32_t>(), o.res);
            ms::merge_verify_kernel<<<grid_for(bound, 256), 256, 0, h->stream>>>(g, bound, h->b_mt_rep.as<unsigned long long>(),
                                                                               h->b_mslot.as<int32_t>(), o.res);
            ms::merge_compact_kernel<<<grid_for(tsize, 256), 256, 0, h->stream>>>(g, h->b_mt_cnt.as<uint32_t>(), h->b_mt_rep.as<unsigned long long>(),
                                                                                tsize, o.res, h->b_m_cnt.as<uint32_t>(), h->b_m_pat.as<uint32_t>(),
                                                                                h->b_mindex.as<uint32_t>());
            h->launches += 3;
            v_cnt = h->b_m_cnt.as<uint32_t>();
            v_pat = h->b_m_pat.as<uint32_t>();
            Mptr = o.res;
            hdr_src = h->b_gather.as<uint8_t>();
            hdr_stride = block;
        }
        ms::rank_small_kernel<<<grid_for(std::min<int64_t>(bound, ms::kSmallSort), 256), 256, 0, h->stream>>>(v_cnt, v_pat, hw, Mptr, bound, hdr_src,
                                                                                                           hdr_stride, world, o);
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
        uint8_t* st = static_cast<uint8_t*>(h->h_stage);
        MS_CUDA(h, cudaMemcpyAsync(st, outb, 64 + static_cast<size_t>(world) * 64, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        memcpy(res, st, 64);
        bool any_collision = false, any_overflow = false;
        int64_t max_ng = 0;
        cat[0] = cat[1] = 0;
        for (int q = 0; q < world; ++q) {
            uint64_t hc[8];
            memcpy(hc, st + 64 + static_cast<size_t>(q) * 64, 64);
            any_overflow |= hc[6] != 0;
            any_collision |= hc[4] != 0;
            max_ng = std::max<int64_t>(max_ng, static_cast<int64_t>(hc[5]));
            cat[0] += hc[0];
            cat[1] += hc[1];
        }
        if (any_collision || any_overflow) {
            if (++attempt >= 4) MS_FAIL(h, MS_ERR_CUDA, "haplotype abundance: class table failed under four seeds");
            if (any_overflow) ts <<= 1;
            continue;
        }
        if (max_ng > gcap) { gcap = (max_ng + 3) & ~int64_t(3); continue; }
        if (res[6] != 0) MS_FAIL(h, MS_ERR_CUDA, "haplotype abundance: class merge table overflow");
        if (res[5] != 0) {
            if (++merge_attempt >= 4) MS_FAIL(h, MS_ERR_CUDA, "haplotype abundance: class merge hash collided under four seeds");
            continue;
        }
        M = world > 1 ? static_cast<int64_t>(res[0]) : max_ng;
        if (res[4] != 0) {   // more than kSmallSort classes: sort, then emit in order
            int64_t n_pad = 0;
            rc = ms::sort_big(h, v_cnt, v_pat, hw, M, &n_pad);
            if (rc != MS_OK) return rc;
            ms::emit_sorted_kernel<<<grid_for(M, 256), 256, 0, h->stream>>>(h->b_ord.as<uint32_t>(), v_cnt, v_pat, hw, M, o);
            h->launches++;
            MS_CUDA(h, cudaGetLastError());
            MS_CUDA(h, cudaMemcpyAsync(st, outb, 64, cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
            memcpy(res, st, 64);
        }
        break;
    }
    const uint64_t N = res[2];   // reads of the classes: the unique and ambiguous reads
    const uint32_t* c_cnt = o.o_cnt;
    const uint32_t* c_pat = o.o_pat;

    const int64_t S = std::max<int64_t>(1, (M + ms::kEmSlice - 1) / ms::kEmSlice);
    const size_t off_part = off_d + align16(static_cast<size_t>(std::max<int64_t>(1, M)) * 8);
    MS_CUDA(h, h->b_ab_em.ensure(off_part + static_cast<size_t>(S) * hpad * 8));
    uint8_t* em = h->b_ab_em.as<uint8_t>();
    ms::EmState* est = reinterpret_cast<ms::EmState*>(em);
    double* pi = reinterpret_cast<double*>(em + off_pi);
    unsigned long long* cmp = reinterpret_cast<unsigned long long*>(em + off_cmp);
    unsigned long long* unq = reinterpret_cast<unsigned long long*>(em + off_unq);
    double* ll = reinterpret_cast<double*>(em + off_ll);
    double* dd = reinterpret_cast<double*>(em + off_d);
    double* part = reinterpret_cast<double*>(em + off_part);
    MS_CUDA(h, cudaMemsetAsync(em, 0, off_d, h->stream));
    ms::abundance_init_kernel<<<grid_for(std::max<int64_t>(1, Hn), 256), 256, 0, h->stream>>>(pi, Hn, est);
    h->launches++;
    if (M > 0) {
        ms::abundance_stats_kernel<<<grid_for(M, 256), 256, 0, h->stream>>>(c_cnt, c_pat, hw, M, cmp, unq);
        h->launches++;
    }
    MS_CUDA(h, cudaGetLastError());
    int32_t it = 0, conv = 1;
    MS_STAGE_BEGIN(h, MS_STAGE_ABUNDANCE_EM);
    if (Hn > 0 && N > 0) {
        const dim3 sgrid(static_cast<unsigned>(hw), static_cast<unsigned>(S));
        ms::EmState* hst = static_cast<ms::EmState*>(h->h_stage);
        int32_t enqueued = 0;
        for (;;) {
            const int32_t k = std::min(ms::kEmBatch, prm->max_iterations - enqueued);
            for (int32_t i = 0; i < k; ++i) {
                ms::abundance_denom_kernel<<<grid_for(M, 256), 256, 0, h->stream>>>(c_pat, hw, M, pi, dd, est, 0);
                ms::abundance_sum_kernel<<<sgrid, ms::kEmThreads, 0, h->stream>>>(c_cnt, c_pat, hw, M, dd, part, pi, Hn, static_cast<double>(N),
                                                                                 prm->tolerance, prm->max_iterations, est);
            }
            h->launches += 2 * k;
            enqueued += k;
            MS_CUDA(h, cudaGetLastError());
            MS_CUDA(h, cudaMemcpyAsync(hst, est, sizeof(ms::EmState), cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
            if (hst->done || enqueued >= prm->max_iterations) break;
        }
        it = hst->iter;
        conv = hst->converged;
        ms::abundance_denom_kernel<<<grid_for(M, 256), 256, 0, h->stream>>>(c_pat, hw, M, pi, dd, est, 1);
        ms::abundance_loglik_kernel<<<1, 1024, 0, h->stream>>>(c_cnt, dd, M, ll);
        h->launches += 2;
    }
    MS_STAGE_END(h, MS_STAGE_ABUNDANCE_EM);
    MS_CUDA(h, cudaGetLastError());
    // [pi | compat | unique | loglik] in one copy
    uint8_t* st = static_cast<uint8_t*>(h->h_stage);
    MS_CUDA(h, cudaMemcpyAsync(st, em, off_d, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    const double* h_pi = reinterpret_cast<const double*>(st + off_pi);
    const uint64_t* h_cmp = reinterpret_cast<const uint64_t*>(st + off_cmp);
    const uint64_t* h_unq = reinterpret_cast<const uint64_t*>(st + off_unq);
    uint64_t nuniq = 0;
    for (int32_t k = 0; k < Hn; ++k) {
        rows[k].unique_reads = h_unq[k];
        rows[k].compatible_reads = h_cmp[k] + cat[1];
        rows[k].em_frequency = h_pi[k];
        nuniq += h_unq[k];
    }
    if (counters) {
        counters->unique = nuniq;
        counters->ambiguous = N - nuniq;
        counters->uninformative = cat[1];
        counters->incompatible = cat[0];
    }
    if (iterations) *iterations = it;
    if (converged) *converged = conv;
    if (loglik) *loglik = (Hn > 0 && N > 0) ? *reinterpret_cast<const double*>(st + off_ll) : 0.0;
    return MS_OK;
}

}  // extern "C"
