// group.cu -- grouped pile-up and per-group consensus (restatement choice U15, DESIGN.md "Haplotype consensus").
//
// What is the full sequence of each haplotype?  After phasing, every read carries its haplotype's position in juliet's
// order; the sequence of haplotype g is fuse's consensus over g's reads.  The pile-up is generic over int32 read labels:
//   1. a stable counting sort of the labels gives each group's list of read indices (ascending: consecutive reads of a
//      large group share the 128-byte lines of the tiles) and the group offsets; labels outside [0, ngroups) are skipped;
//   2. group_pileup_kernel: persistent CTAs walk work items (group, chunk of <= 2040 of its reads, column segment).  A
//      thread owns one 32-column block; it gathers that block of each listed read from the tiles with cp.async, two
//      batches of 8 reads ahead, forms K1's one-bit masks (P0, P1, P2, their pairwise ANDs, P3) and adds them into K1's
//      bit-sliced carry-save counters (pileup.cuh).  At the end of an item the sums decode into exact per-column counts
//      (reads that do not span a column drop out, as in K1's finalize) which are added into gcol[g][L][8] with RED;
//   3. the consensus: fuse's insertion tally (fuse.cuh) keyed by g * L + column, so every group is judged against its own
//      votes; the host applies the greedy spacing per group; one CTA per group computes the sequence length, and after
//      the prefix sum over the groups one CTA per group writes its sequence at its offset.
// Counts are integer sums: the order in which reads are visited changes locality, never a result.
#include <algorithm>
#include <climits>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>
#include "fuse.cuh"
#include "group.cuh"
#include "handle.h"

namespace ms {

constexpr int kGroupMasks = 7;                             // P0 P1 P2 P0&P1 P0&P2 P1&P2 P3
constexpr int kSortThreads = 256;
constexpr int64_t kSortHistMax = 1 << 22;                  // entries of the [chunk][group] histogram of the counting sort

__device__ __forceinline__ bool label_ok(int32_t g, int32_t ngroups) { return g >= 0 && g < ngroups; }

// ---------------------------------------------------------------- counting sort of the labels
// chunk c = reads [c*cs, (c+1)*cs): hist[c][g] = its reads labelled g
__global__ void __launch_bounds__(kSortThreads) label_hist_kernel(const int32_t* __restrict__ lab, int64_t R, int32_t ngroups, int64_t cs,
                                                                  uint32_t* __restrict__ hist) {
    const int64_t r0 = static_cast<int64_t>(blockIdx.x) * cs, r1 = min(R, r0 + cs);
    uint32_t* row = hist + static_cast<size_t>(blockIdx.x) * ngroups;
    const int lane = threadIdx.x & 31;
    for (int64_t base = r0; base < r1; base += blockDim.x) {
        const int64_t r = base + threadIdx.x;
        const int32_t g = r < r1 ? lab[r] : -1;
        const bool ok = label_ok(g, ngroups);
        const uint32_t peers = __match_any_sync(0xffffffffu, ok ? g : -1);
        if (ok && lane == __ffs(peers) - 1) atomicAdd(row + g, static_cast<uint32_t>(__popc(peers)));
    }
}

// one warp per group: hist[c][g] -> reads labelled g in chunks before c; tot[g] = all of them
__global__ void label_colscan_kernel(uint32_t* __restrict__ hist, int32_t nch, int32_t ngroups, uint32_t* __restrict__ tot) {
    const int64_t g = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= ngroups) return;
    uint32_t run = 0;
    for (int32_t c0 = 0; c0 < nch; c0 += 32) {
        const int32_t c = c0 + lane;
        const uint32_t v = c < nch ? hist[static_cast<size_t>(c) * ngroups + g] : 0u;
        uint32_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (c < nch) hist[static_cast<size_t>(c) * ngroups + g] = run + inc - v;
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) tot[g] = run;
}

// one CTA of 1024: goff = exclusive scan of tot (ngroups + 1 entries), ioff = the same over the work items ceil(tot / chunk)
__global__ void __launch_bounds__(1024) label_offsets_kernel(const uint32_t* __restrict__ tot, int32_t ngroups, int32_t* __restrict__ goff,
                                                             int32_t* __restrict__ ioff) {
    __shared__ uint32_t ws[2][32];
    __shared__ uint32_t carry[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry[0] = carry[1] = 0;
    __syncthreads();
    for (int32_t g0 = 0; g0 < ngroups; g0 += 1024) {
        const int32_t g = g0 + tid;
        const uint32_t n = g < ngroups ? tot[g] : 0u;
        uint32_t v[2] = {n, (n + kGroupChunk - 1) / kGroupChunk};
        uint32_t inc[2] = {v[0], v[1]};
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, inc[k], o);
                if (lane >= o) inc[k] += t;
            }
        }
        if (lane == 31) { ws[0][warp] = inc[0]; ws[1][warp] = inc[1]; }
        __syncthreads();
        if (warp == 0) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                uint32_t w = ws[k][lane], wi = w;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
                    if (lane >= o) wi += t;
                }
                ws[k][lane] = wi - w;   // exclusive prefix of the warps
            }
        }
        __syncthreads();
        if (g < ngroups) {
            goff[g] = static_cast<int32_t>(carry[0] + ws[0][warp] + inc[0] - v[0]);
            ioff[g] = static_cast<int32_t>(carry[1] + ws[1][warp] + inc[1] - v[1]);
        }
        __syncthreads();
        if (tid == 1023) { carry[0] += ws[0][warp] + inc[0]; carry[1] += ws[1][warp] + inc[1]; }
        __syncthreads();
    }
    if (tid == 0) { goff[ngroups] = static_cast<int32_t>(carry[0]); ioff[ngroups] = static_cast<int32_t>(carry[1]); }
}

// Stable scatter: the warps of a chunk take their turn in order, lanes of a warp by lane index, so that every group's list
// keeps the reads in ascending order.  hist[c][g] is chunk c's cursor into group g's list.
__global__ void __launch_bounds__(kSortThreads) label_scatter_kernel(const int32_t* __restrict__ lab, int64_t R, int32_t ngroups, int64_t cs,
                                                                     uint32_t* __restrict__ hist, const int32_t* __restrict__ goff,
                                                                     int32_t* __restrict__ list) {
    const int64_t r0 = static_cast<int64_t>(blockIdx.x) * cs, r1 = min(R, r0 + cs);
    uint32_t* row = hist + static_cast<size_t>(blockIdx.x) * ngroups;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int64_t base = r0; base < r1; base += blockDim.x) {
        const int64_t r = base + threadIdx.x;
        const int32_t g = r < r1 ? lab[r] : -1;
        const bool ok = label_ok(g, ngroups);
        const uint32_t peers = __match_any_sync(0xffffffffu, ok ? g : -1);
        const int leader = __ffs(peers) - 1;
        const uint32_t before = static_cast<uint32_t>(__popc(peers & ((1u << lane) - 1u)));
        for (int w = 0; w < nwarps; ++w) {
            if (w == warp) {
                uint32_t pos = 0;
                if (ok && lane == leader) pos = atomicAdd(row + g, static_cast<uint32_t>(__popc(peers)));
                pos = __shfl_sync(0xffffffffu, pos, leader);
                if (ok) list[goff[g] + static_cast<int64_t>(pos) + before] = static_cast<int32_t>(r);
            }
            __syncthreads();
        }
    }
}

// ---------------------------------------------------------------- grouped pile-up
struct GroupArgs {
    const uint4* tiles;        // reads in the tile layout (rows.cuh)
    const int32_t* list;       // read indices, grouped
    const int32_t* goff;       // [ngroups + 1] group offsets into list
    const int32_t* ioff;       // [ngroups + 1] first work item of each group (chunks of kGroupChunk reads)
    uint32_t* gcol;            // [ngroups][L][8]
    int32_t ngroups, L, nblk, nseg, seg_len;
};

// K1's masks of one read (kModeFuse's set)
__device__ __forceinline__ void group_masks(uint32_t addr, uint32_t /*stride*/, uint32_t (&m)[kGroupMasks]) {
    const uint4 q = lds128g(addr);
    m[0] = q.x;
    m[1] = q.y;
    m[2] = q.z;
    m[3] = q.x & q.y;
    m[4] = q.x & q.z;
    m[5] = q.y & q.z;
    m[6] = q.w;
}

// end of a work item (cold path, as K1's emit_slice): planes [mask][kPlanes] of n reads -> per-column integers, added into
// the group's columns [32 * blk, 32 * blk + ncols) with RED (zero counts are skipped)
__device__ __noinline__ void group_flush(const uint32_t* planes, uint32_t n, uint32_t* dst, int ncols) {
    uint32_t tr[kGroupMasks][16];
#pragma unroll
    for (int i = 0; i < kGroupMasks; ++i) {
        uint32_t acc[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[k] = k < kPlanes ? planes[i * kPlanes + k] : 0u;
        transpose16x2(acc);
#pragma unroll
        for (int k = 0; k < 16; ++k) tr[i][k] = acc[k];
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int colj = j + 16 * half;
            if (colj >= ncols) continue;
            uint32_t s[kGroupMasks];
#pragma unroll
            for (int i = 0; i < kGroupMasks; ++i) s[i] = half ? (tr[i][j] >> 16) : (tr[i][j] & 0xffffu);
            uint4 lo, hi;
            decode_counts(s, s[6], n, lo, hi);
            const uint32_t c[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (c[k]) atomicAdd(dst + colj * 8 + k, c[k]);
        }
    }
}

// the walk's policy (group.cuh): work item k belongs to the group g with ioff[g] <= k < ioff[g + 1]
struct GroupPolicy {
    static constexpr int NM = kGroupMasks, SLOTS = 1;
    GroupArgs a;
    __device__ __forceinline__ int32_t item(int32_t k, int32_t& r_begin, int32_t& r_end) const {
        int32_t lo = 0, hi = a.ngroups;
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (__ldg(a.ioff + mid) <= k) lo = mid;
            else hi = mid;
        }
        r_begin = __ldg(a.goff + lo) + (k - __ldg(a.ioff + lo)) * kGroupChunk;
        r_end = min(__ldg(a.goff + lo + 1), r_begin + kGroupChunk);
        return lo;
    }
    __device__ __forceinline__ int64_t read(int32_t idx) const { return __ldg(a.list + idx); }
    __device__ static __forceinline__ void masks(uint32_t addr, uint32_t stride, uint32_t (&m)[NM]) { group_masks(addr, stride, m); }
    __device__ __forceinline__ void flush(const uint32_t* planes, uint32_t n, int32_t g, int b) const {
        group_flush(planes, n, a.gcol + (static_cast<size_t>(g) * a.L + static_cast<size_t>(b) * 32) * 8, min(32, a.L - b * 32));
    }
};

__global__ void __launch_bounds__(kGroupMaxThreads) group_pileup_kernel(GroupArgs a) {
    csa_walk(GroupPolicy{a}, a.tiles, a.nblk, a.nseg, a.seg_len, static_cast<int64_t>(a.ioff[a.ngroups]) * a.nseg);
}

// ---------------------------------------------------------------- per-group consensus
// Column call of U15 (fuse's U6-U8 and the 'N' rule): 0 = the column is removed ('-' wins)
__device__ __forceinline__ char group_call(const uint32_t* hc, uint32_t min_cov) {
    const unsigned long long votes = static_cast<unsigned long long>(hc[0]) + hc[1] + hc[2] + hc[3] + hc[4];
    if (votes < min_cov) return 'N';
    int best = 0;
#pragma unroll
    for (int s = 1; s < 5; ++s)
        if (hc[s] > hc[best]) best = s;
    return best < 4 ? "ACGT"[best] : 0;
}

// one CTA per group: the kept span, first and last column with votes >= min_cov (lo > hi: nothing kept)
__global__ void __launch_bounds__(1024) group_span_kernel(const uint32_t* __restrict__ gcol, int32_t L, uint32_t min_cov, int2* __restrict__ span) {
    __shared__ int32_t wl[32], wh[32];
    const int g = blockIdx.x, tid = threadIdx.x;
    const uint32_t* col = gcol + static_cast<size_t>(g) * L * 8;
    int32_t lo = INT_MAX, hi = -1;
    for (int32_t j = tid; j < L; j += blockDim.x) {
        const uint32_t* hc = col + static_cast<size_t>(j) * 8;
        const unsigned long long votes = static_cast<unsigned long long>(hc[0]) + hc[1] + hc[2] + hc[3] + hc[4];
        if (votes >= min_cov) { lo = min(lo, j); hi = max(hi, j); }
    }
    lo = __reduce_min_sync(0xffffffffu, lo);
    hi = __reduce_max_sync(0xffffffffu, hi);
    if ((tid & 31) == 0) { wl[tid >> 5] = lo; wh[tid >> 5] = hi; }
    __syncthreads();
    if (tid < 32) {
        lo = tid < static_cast<int>(blockDim.x >> 5) ? wl[tid] : INT_MAX;
        hi = tid < static_cast<int>(blockDim.x >> 5) ? wh[tid] : -1;
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (tid == 0) span[g] = make_int2(lo, hi);
    }
}

struct GroupAcc {
    const int32_t* aoff;      // [ngroups + 1] accepted insertions of group g: [aoff[g], aoff[g + 1]), ascending column
    const int32_t* col;       // column the insertion follows
    const long long* off;     // its string: pool[off .. off + len)
    const int32_t* len;
    const char* pool;
};

// one CTA (1024 threads) per group over its kept span; EMIT = false: the length of each sequence, EMIT = true: the sequence
// at seq + seq_off[g]
template <bool EMIT>
__global__ void __launch_bounds__(1024) group_consensus_kernel(const uint32_t* __restrict__ gcol, int32_t L, uint32_t min_cov,
                                                               const int2* __restrict__ span, GroupAcc acc, long long* __restrict__ out_len,
                                                               const long long* __restrict__ seq_off, char* __restrict__ seq) {
    __shared__ long long part[1024];
    const int g = blockIdx.x, tid = threadIdx.x;
    const uint32_t* col = gcol + static_cast<size_t>(g) * L * 8;
    const int2 sp = span[g];
    const int32_t n = sp.y >= sp.x ? sp.y - sp.x + 1 : 0;
    const int32_t per = (n + 1023) / 1024;
    const int32_t j0 = sp.x + min(n, tid * per), j1 = sp.x + min(n, (tid + 1) * per);
    int32_t a = acc.aoff[g], ae = acc.aoff[g + 1];
    {   // first accepted insertion at a column >= j0
        int32_t hi = ae;
        while (a < hi) {
            const int32_t mid = (a + hi) >> 1;
            if (acc.col[mid] < j0) a = mid + 1;
            else hi = mid;
        }
    }
    const int32_t a0 = a;
    long long mine = 0;
    for (int32_t j = j0; j < j1; ++j) {
        mine += group_call(col + static_cast<size_t>(j) * 8, min_cov) ? 1 : 0;
        if (a < ae && acc.col[a] == j) mine += acc.len[a++];
    }
    part[tid] = mine;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // inclusive Hillis-Steele scan
        const long long t = tid >= o ? part[tid - o] : 0;
        __syncthreads();
        part[tid] += t;
        __syncthreads();
    }
    if (!EMIT) {
        if (tid == 1023) out_len[g] = part[1023];
        return;
    }
    char* out = seq + seq_off[g] + (part[tid] - mine);
    a = a0;
    for (int32_t j = j0; j < j1; ++j) {
        const char c = group_call(col + static_cast<size_t>(j) * 8, min_cov);
        if (c) *out++ = c;
        if (a < ae && acc.col[a] == j) {
            const char* s = acc.pool + acc.off[a];
            for (int32_t q = 0; q < acc.len[a]; ++q) *out++ = s[q];
            ++a;
        }
    }
}

}  // namespace ms

namespace {

inline unsigned blocks_for(int64_t n, int block) { return static_cast<unsigned>(std::max<int64_t>(1, (n + block - 1) / block)); }

// frees the temporaries of one call on every way out
struct TmpScope {
    std::vector<void*> ptrs;
    ~TmpScope() { for (void* p : ptrs) cudaFree(p); }
    template <class T> cudaError_t alloc(T** out, size_t bytes) {
        void* p = nullptr;
        const cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
        if (e == cudaSuccess) ptrs.push_back(p);
        *out = static_cast<T*>(p);
        return e;
    }
};

bool groups_ready(const ms_handle* h) { return h->label_groups >= 0 && h->label_L == h->L && h->L > 0; }

}  // namespace

void ms_group_set_smem_attr() {
    cudaFuncSetAttribute(ms::group_pileup_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         ms::kGroupRing * 8 * ms::kGroupMaxThreads * 16);
}

extern "C" {

int ms_set_groups(ms_handle* h, int32_t ngroups) {
    if (!h || ngroups < 0) return MS_ERR_ARG;
    if (h->L <= 0) MS_FAIL(h, MS_ERR_ARG, "ms_set_groups: call ms_set_layout first");
    MS_CUDA(h, cudaSetDevice(h->device));
    const size_t bytes = static_cast<size_t>(ngroups) * h->L * 8 * 4;
    MS_CUDA(h, h->b_gcol.ensure(std::max<size_t>(bytes, 4)));
    if (bytes) MS_CUDA(h, cudaMemsetAsync(h->b_gcol.p, 0, bytes, h->stream));
    h->label_groups = ngroups;
    h->label_L = h->L;
    return MS_OK;
}

int ms_group_pileup_dev(ms_handle* h, const uint32_t* d_packed, const int32_t* d_group, int64_t R) {
    MsRange nvtx_range("grouped pile-up");
    if (!h || R < 0 || (R > 0 && (!d_packed || !d_group))) return MS_ERR_ARG;
    if (!groups_ready(h)) MS_FAIL(h, MS_ERR_ARG, "ms_group_pileup_dev: call ms_set_groups after ms_set_layout first");
    if (R > INT32_MAX) MS_FAIL(h, MS_ERR_ARG, "ms_group_pileup_dev: more than 2^31 - 1 reads in one call");
    const int32_t G = h->label_groups;
    if (R == 0 || G == 0) return MS_OK;
    MS_CUDA(h, cudaSetDevice(h->device));
    // counting sort: chunks of the reads x groups histogram, bounded in size
    const int64_t nch = std::max<int64_t>(1, std::min<int64_t>((R + 2047) / 2048, ms::kSortHistMax / G));
    const int64_t cs = (R + nch - 1) / nch;
    MS_CUDA(h, h->b_ghist.ensure(static_cast<size_t>(nch) * G * 4));
    MS_CUDA(h, h->b_gtot.ensure(static_cast<size_t>(G) * 4));
    MS_CUDA(h, h->b_goff.ensure(static_cast<size_t>(G + 1) * 4));
    MS_CUDA(h, h->b_gioff.ensure(static_cast<size_t>(G + 1) * 4));
    MS_CUDA(h, h->b_glist.ensure(static_cast<size_t>(R) * 4));
    uint32_t* hist = h->b_ghist.as<uint32_t>();
    MS_CUDA(h, cudaMemsetAsync(hist, 0, static_cast<size_t>(nch) * G * 4, h->stream));
    ms::label_hist_kernel<<<static_cast<unsigned>(nch), ms::kSortThreads, 0, h->stream>>>(d_group, R, G, cs, hist);
    ms::label_colscan_kernel<<<blocks_for(static_cast<int64_t>(G) * 32, 256), 256, 0, h->stream>>>(hist, static_cast<int32_t>(nch), G,
                                                                                                   h->b_gtot.as<uint32_t>());
    ms::label_offsets_kernel<<<1, 1024, 0, h->stream>>>(h->b_gtot.as<uint32_t>(), G, h->b_goff.as<int32_t>(), h->b_gioff.as<int32_t>());
    ms::label_scatter_kernel<<<static_cast<unsigned>(nch), ms::kSortThreads, 0, h->stream>>>(d_group, R, G, cs, hist, h->b_goff.as<int32_t>(),
                                                                                              h->b_glist.as<int32_t>());
    h->launches += 4;
    // the pile-up: one thread per 32-column block of a segment, at most kGroupMaxThreads blocks per segment
    ms::GroupArgs a;
    a.tiles = reinterpret_cast<const uint4*>(d_packed);
    a.list = h->b_glist.as<int32_t>();
    a.goff = h->b_goff.as<int32_t>();
    a.ioff = h->b_gioff.as<int32_t>();
    a.gcol = h->b_gcol.as<uint32_t>();
    a.ngroups = G;
    a.L = h->L;
    a.nblk = h->nblk;
    a.nseg = (h->nblk + ms::kGroupMaxThreads - 1) / ms::kGroupMaxThreads;
    a.seg_len = (h->nblk + a.nseg - 1) / a.nseg;
    const int threads = (a.seg_len + 31) / 32 * 32;
    const int smem = ms::kGroupRing * 8 * threads * 16;
    int per_sm = 0;
    MS_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ms::group_pileup_kernel, threads, smem));
    // at most one CTA per work item; the item count is on the device: bound it by the reads
    const int64_t items_max = ((R + ms::kGroupChunk - 1) / ms::kGroupChunk + G) * a.nseg;
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(items_max, static_cast<int64_t>(std::max(1, per_sm)) * h->num_sms)));
    MS_STAGE_BEGIN(h, MS_STAGE_GROUP_PILEUP);
    ms::group_pileup_kernel<<<grid, threads, smem, h->stream>>>(a);
    MS_STAGE_END(h, MS_STAGE_GROUP_PILEUP);
    h->launches++;
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

int ms_get_group_counts(ms_handle* h, uint32_t* col) {
    if (!h || !col) return MS_ERR_ARG;
    if (!groups_ready(h)) MS_FAIL(h, MS_ERR_ARG, "ms_get_group_counts: no group counts (ms_set_groups)");
    MS_CUDA(h, cudaSetDevice(h->device));
    const size_t bytes = static_cast<size_t>(h->label_groups) * h->L * 8 * 4;
    if (bytes) MS_CUDA(h, cudaMemcpyAsync(col, h->b_gcol.p, bytes, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    return MS_OK;
}

int ms_group_consensus(ms_handle* h, const ms_fuse_params* prm, const int32_t* ins_group, const int32_t* ins_col, const int64_t* ins_off,
                       const int32_t* ins_len, int64_t nins, const char* ins_pool, int64_t pool_len, char* seq, int64_t cap,
                       int64_t* seq_off) {
    MsRange nvtx_range("group consensus");
    if (!h || !prm || !seq_off || nins < 0 || cap < 0 || pool_len < 0 || prm->min_coverage < 0 ||
        (nins > 0 && (!ins_group || !ins_col || !ins_off || !ins_len || !ins_pool)))
        return MS_ERR_ARG;
    if (!groups_ready(h)) MS_FAIL(h, MS_ERR_ARG, "ms_group_consensus: no group counts (ms_set_groups)");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t G = h->label_groups, L = h->L;
    seq_off[0] = 0;
    if (G == 0) return MS_OK;
    const uint32_t min_cov = static_cast<uint32_t>(std::max(1, prm->min_coverage));   // a column without votes is never called
    const uint32_t* gcol = h->b_gcol.as<uint32_t>();
    TmpScope tmp;
    int2* d_span = nullptr;
    MS_CUDA(h, tmp.alloc(&d_span, static_cast<size_t>(G) * sizeof(int2)));
    ms::group_span_kernel<<<G, 1024, 0, h->stream>>>(gcol, L, min_cov, d_span);
    h->launches++;
    std::vector<int2> span(G);
    MS_CUDA(h, cudaMemcpyAsync(span.data(), d_span, static_cast<size_t>(G) * sizeof(int2), cudaMemcpyDeviceToHost, h->stream));

    // insertions of the groups: key g * L + column, so that ins_eval_kernel reads group g's column from the flattened tensor
    std::vector<int32_t> acc_col, acc_len;
    std::vector<long long> acc_off;
    std::vector<int32_t> aoff(static_cast<size_t>(G) + 1, 0);
    char* d_pool = nullptr;
    std::vector<int64_t> keep;
    for (int64_t i = 0; i < nins; ++i) {
        if (ins_off[i] < 0 || ins_len[i] < 0 || ins_off[i] + ins_len[i] > pool_len) MS_FAIL(h, MS_ERR_ARG, "insertion event outside the pool");
        if (ins_group[i] >= 0 && ins_group[i] < G && ins_col[i] >= 0 && ins_col[i] < L) keep.push_back(i);
    }
    std::vector<ms::InsCand> cand;
    if (!keep.empty()) {
        if (static_cast<int64_t>(G) * L > INT32_MAX) MS_FAIL(h, MS_ERR_ARG, "ms_group_consensus: ngroups * L exceeds the insertion keys");
        const int64_t n = static_cast<int64_t>(keep.size());
        std::vector<int32_t> key(n), len(n);
        std::vector<long long> off(n);
        for (int64_t k = 0; k < n; ++k) {
            const int64_t i = keep[k];
            key[k] = ins_group[i] * L + ins_col[i];
            len[k] = ins_len[i];
            off[k] = ins_off[i];
        }
        int64_t ts = 1024;
        while (ts < 2 * n) ts <<= 1;
        int32_t* d_key = nullptr; long long* d_off = nullptr; int32_t* d_len = nullptr;
        unsigned long long* t_key = nullptr; uint32_t* t_cnt = nullptr; long long* t_rep = nullptr;
        ms::InsCand* d_cand = nullptr; unsigned long long* d_n = nullptr;
        MS_CUDA(h, tmp.alloc(&d_key, n * 4)); MS_CUDA(h, tmp.alloc(&d_off, n * 8)); MS_CUDA(h, tmp.alloc(&d_len, n * 4));
        MS_CUDA(h, tmp.alloc(&d_pool, std::max<int64_t>(1, pool_len)));
        MS_CUDA(h, tmp.alloc(&t_key, ts * 8)); MS_CUDA(h, tmp.alloc(&t_cnt, ts * 4)); MS_CUDA(h, tmp.alloc(&t_rep, ts * 8));
        MS_CUDA(h, tmp.alloc(&d_cand, n * sizeof(ms::InsCand))); MS_CUDA(h, tmp.alloc(&d_n, 8));
        MS_CUDA(h, cudaMemcpyAsync(d_key, key.data(), n * 4, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_off, off.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_len, len.data(), n * 4, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_pool, ins_pool, pool_len, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemsetAsync(t_key, 0, ts * 8, h->stream));
        MS_CUDA(h, cudaMemsetAsync(t_cnt, 0, ts * 4, h->stream));
        MS_CUDA(h, cudaMemsetAsync(t_rep, 0x7f, ts * 8, h->stream));
        MS_CUDA(h, cudaMemsetAsync(d_n, 0, 8, h->stream));
        ms::ins_tally_kernel<<<blocks_for(n, 256), 256, 0, h->stream>>>(d_key, d_off, d_len, n, d_pool, t_key, t_cnt, t_rep, ts - 1);
        ms::ins_eval_kernel<<<blocks_for(ts, 256), 256, 0, h->stream>>>(t_cnt, t_rep, ts, d_key, d_len, gcol, G * L, prm->ins_fraction, d_cand,
                                                                        d_n, n);
        h->launches += 2;
        unsigned long long nc = 0;
        MS_CUDA(h, cudaMemcpyAsync(&nc, d_n, 8, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        cand.resize(nc);
        if (nc) {
            MS_CUDA(h, cudaMemcpyAsync(cand.data(), d_cand, nc * sizeof(ms::InsCand), cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
        }
        // exactness guard against a 64-bit hash collision: recount the survivors' (key, string) over the events
        auto ident = [&](int32_t k, int64_t o, int32_t l) {
            std::string s(reinterpret_cast<const char*>(&k), 4);
            return s.append(ins_pool + o, static_cast<size_t>(l));
        };
        std::unordered_map<std::string, uint32_t> exact;
        for (ms::InsCand& c : cand) {
            c.rep = off[c.rep];                               // from here on: the string's offset in the pool
            exact.emplace(ident(c.col, c.rep, c.len), 0u);
        }
        if (!cand.empty())
            for (int64_t k = 0; k < n; ++k) {
                auto e = exact.find(ident(key[k], off[k], len[k]));
                if (e != exact.end()) ++e->second;
            }
        for (const ms::InsCand& c : cand)
            if (exact[ident(c.col, c.rep, c.len)] != c.cnt) MS_FAIL(h, MS_ERR_CUDA, "insertion hash collision");
        std::sort(cand.begin(), cand.end(), [&](const ms::InsCand& x, const ms::InsCand& y) {
            if (x.col != y.col) return x.col < y.col;
            if (x.len != y.len) return x.len < y.len;
            return memcmp(ins_pool + x.rep, ins_pool + y.rep, x.len) < 0;
        });
    } else {
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    // greedy spacing per group, left to right, over the candidates after a column of the group's kept span
    {
        int32_t cur = -1, last = -1;
        for (const ms::InsCand& c : cand) {
            const int32_t g = c.col / L, j = c.col % L;
            if (g != cur) { cur = g; last = -1; }
            if (j < span[g].x || j > span[g].y) continue;
            if (j == last) continue;                            // one insertion per column: the first in (length, string) order
            if (last >= 0 && j - last < prm->ins_distance) continue;
            acc_col.push_back(j); acc_off.push_back(c.rep); acc_len.push_back(c.len);
            ++aoff[g + 1];
            last = j;
        }
        for (int32_t g = 0; g < G; ++g) aoff[g + 1] += aoff[g];
    }
    const int64_t na = static_cast<int64_t>(acc_col.size());
    int32_t* d_aoff = nullptr; int32_t* d_acol = nullptr; long long* d_aoff_pool = nullptr; int32_t* d_alen = nullptr;
    long long* d_len = nullptr; long long* d_seq_off = nullptr;
    MS_CUDA(h, tmp.alloc(&d_aoff, static_cast<size_t>(G + 1) * 4));
    MS_CUDA(h, tmp.alloc(&d_acol, static_cast<size_t>(na) * 4)); MS_CUDA(h, tmp.alloc(&d_aoff_pool, static_cast<size_t>(na) * 8));
    MS_CUDA(h, tmp.alloc(&d_alen, static_cast<size_t>(na) * 4));
    MS_CUDA(h, tmp.alloc(&d_len, static_cast<size_t>(G) * 8)); MS_CUDA(h, tmp.alloc(&d_seq_off, static_cast<size_t>(G + 1) * 8));
    MS_CUDA(h, cudaMemcpyAsync(d_aoff, aoff.data(), static_cast<size_t>(G + 1) * 4, cudaMemcpyHostToDevice, h->stream));
    if (na) {
        MS_CUDA(h, cudaMemcpyAsync(d_acol, acc_col.data(), static_cast<size_t>(na) * 4, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_aoff_pool, acc_off.data(), static_cast<size_t>(na) * 8, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_alen, acc_len.data(), static_cast<size_t>(na) * 4, cudaMemcpyHostToDevice, h->stream));
    }
    ms::GroupAcc ga{d_aoff, d_acol, d_aoff_pool, d_alen, d_pool};
    ms::group_consensus_kernel<false><<<G, 1024, 0, h->stream>>>(gcol, L, min_cov, d_span, ga, d_len, nullptr, nullptr);
    h->launches++;
    std::vector<long long> glen(G);
    MS_CUDA(h, cudaMemcpyAsync(glen.data(), d_len, static_cast<size_t>(G) * 8, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    MS_CUDA(h, cudaGetLastError());
    for (int32_t g = 0; g < G; ++g) seq_off[g + 1] = seq_off[g] + glen[g];
    const int64_t total = seq_off[G];
    if (cap < total) MS_FAIL(h, MS_ERR_CAPACITY, "ms_group_consensus: seq holds fewer bytes than the sequences need (seq_off)");
    if (total == 0) return MS_OK;
    if (!seq) MS_FAIL(h, MS_ERR_ARG, "ms_group_consensus: seq is NULL");
    char* d_seq = nullptr;
    MS_CUDA(h, tmp.alloc(&d_seq, static_cast<size_t>(total)));
    MS_CUDA(h, cudaMemcpyAsync(d_seq_off, seq_off, static_cast<size_t>(G + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    ms::group_consensus_kernel<true><<<G, 1024, 0, h->stream>>>(gcol, L, min_cov, d_span, ga, nullptr, d_seq_off, d_seq);
    h->launches++;
    MS_CUDA(h, cudaMemcpyAsync(seq, d_seq, static_cast<size_t>(total), cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

}  // extern "C"
