// fuse.cu -- K4: fuse's column-majority consensus with its insertion rule.
//
// Replaces `fuse in.bam out.fasta` (/root/reference/doc/FUSE.md:17-24): "creation of a
// high-quality consensus sequence", "includes in-frame insertions with a certain distance
// to each other", "major deletions are being removed".  SURVEY.md rows a14, a15; the
// thresholds are restatement choices U6-U8 (ms_fuse_params).
//
// Device work: inserted strings are hashed and tallied per (column, string) in an
// open-addressing table, a per-slot kernel applies the in-frame + support rule against the
// all-reduced column votes, and one CTA emits the consensus (majority base per column,
// deletion-majority columns dropped, accepted insertions spliced in) with a block scan.
// The greedy left-to-right spacing pass over the handful of surviving candidates is
// sequential by definition and runs on the host between the two kernels.
#include <algorithm>
#include <cstring>
#include <vector>
#include "fuse.cuh"
#include "handle.h"

namespace ms {

__device__ __forceinline__ uint64_t mix64f(uint64_t x) {
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL;
    x ^= x >> 27; x *= 0x94d049bb133111ebULL;
    x ^= x >> 31;
    return x;
}

__global__ void ins_tally_kernel(const int32_t* __restrict__ col, const long long* __restrict__ off,
                                 const int32_t* __restrict__ len, int64_t nins, const char* __restrict__ pool,
                                 unsigned long long* tab_key, uint32_t* tab_cnt, long long* tab_rep, int64_t mask) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= nins) return;
    uint64_t hsh = mix64f(0x66757365ULL ^ (static_cast<uint64_t>(static_cast<uint32_t>(col[i])) << 32) ^ static_cast<uint32_t>(len[i]));
    const char* s = pool + off[i];
    for (int32_t k = 0; k < len[i]; ++k) hsh = mix64f(hsh ^ static_cast<uint8_t>(s[k]));
    if (!hsh) hsh = 1;
    int64_t idx = static_cast<int64_t>(hsh) & mask;
    for (;;) {
        const unsigned long long prev = atomicCAS(tab_key + idx, 0ULL, static_cast<unsigned long long>(hsh));
        if (prev == 0ULL || prev == hsh) break;
        idx = (idx + 1) & mask;
    }
    atomicAdd(tab_cnt + idx, 1u);
    atomicMin(tab_rep + idx, static_cast<long long>(i));
}

__global__ void ins_eval_kernel(const uint32_t* __restrict__ tab_cnt, const long long* __restrict__ tab_rep, int64_t tab_size,
                                const int32_t* __restrict__ col, const int32_t* __restrict__ len,
                                const uint32_t* __restrict__ colcnt, int32_t L, double frac,
                                InsCand* __restrict__ out, unsigned long long* nout, int64_t cap) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= tab_size || tab_cnt[i] == 0) return;
    const long long rep = tab_rep[i];
    const int32_t c = col[rep], l = len[rep];
    if (c < 0 || c >= L || l <= 0 || l % 3 != 0) return;
    const uint32_t* hc = colcnt + static_cast<size_t>(c) * 8;
    const unsigned long long votes = static_cast<unsigned long long>(hc[0]) + hc[1] + hc[2] + hc[3] + hc[4];
    if (!(static_cast<double>(tab_cnt[i]) > frac * static_cast<double>(votes))) return;
    const unsigned long long k = atomicAdd(nout, 1ULL);
    if (static_cast<int64_t>(k) < cap) { out[k].col = c; out[k].len = l; out[k].rep = rep; out[k].cnt = tab_cnt[i]; out[k].pad = 0; }
}

// acc_off[j] >= 0: an accepted insertion (offset into pool, acc_len[j]) follows column j
__global__ void __launch_bounds__(1024) consensus_kernel(const uint32_t* __restrict__ colcnt, int32_t L, int32_t min_cov,
                                                         const long long* __restrict__ acc_off, const int32_t* __restrict__ acc_len,
                                                         const char* __restrict__ pool, char* __restrict__ seq,
                                                         long long* __restrict__ out_len) {
    __shared__ long long part[1024];
    const int tid = threadIdx.x;
    const int per = (L + 1023) / 1024;
    const int j0 = tid * per, j1 = min(L, j0 + per);
    auto base_of = [&](int j) -> char {
        const uint32_t* hc = colcnt + static_cast<size_t>(j) * 8;
        const unsigned long long votes = static_cast<unsigned long long>(hc[0]) + hc[1] + hc[2] + hc[3] + hc[4];
        if (votes == 0 || votes < static_cast<unsigned long long>(min_cov)) return 0;
        int best = 0;
#pragma unroll
        for (int s = 1; s < 5; ++s)
            if (hc[s] > hc[best]) best = s;
        return best < 4 ? "ACGT"[best] : 0;
    };
    long long mine = 0;
    for (int j = j0; j < j1; ++j) mine += (base_of(j) ? 1 : 0) + (acc_off[j] >= 0 ? acc_len[j] : 0);
    part[tid] = mine;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {  // inclusive Hillis-Steele scan
        const long long v = tid >= o ? part[tid - o] : 0;
        __syncthreads();
        part[tid] += v;
        __syncthreads();
    }
    long long pos = part[tid] - mine;
    for (int j = j0; j < j1; ++j) {
        const char b = base_of(j);
        if (b) seq[pos++] = b;
        if (acc_off[j] >= 0)
            for (int k = 0; k < acc_len[j]; ++k) seq[pos++] = pool[acc_off[j] + k];
    }
    if (tid == 1023) *out_len = part[1023];
}

}  // namespace ms

namespace {
// frees every temporary of one ms_fuse call on every way out (errors included)
struct DevScope {
    std::vector<void*> ptrs;
    ~DevScope() { for (void* p : ptrs) cudaFree(p); }
    template <class T> cudaError_t alloc(T** out, size_t bytes) {
        void* p = nullptr;
        const cudaError_t e = cudaMalloc(&p, bytes ? bytes : 1);
        if (e == cudaSuccess) ptrs.push_back(p);
        *out = static_cast<T*>(p);
        return e;
    }
};
}  // namespace

extern "C" {

void ms_fuse_params_default(ms_fuse_params* p) {
    if (!p) return;
    p->min_coverage = 50; p->ins_fraction = 0.5; p->ins_distance = 20;
}

int ms_fuse(ms_handle* h, const ms_fuse_params* prm, const int32_t* ins_col, const int64_t* ins_off, const int32_t* ins_len,
            int64_t nins, const char* ins_pool, int64_t pool_len, char* seq, int64_t cap, int64_t* len) {
    MsRange nvtx_range("K4 fuse");
    if (!h || !h->d_counts || !prm || !len || nins < 0 || (nins > 0 && (!ins_col || !ins_off || !ins_len || !ins_pool)))
        return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t L = h->L;
    std::vector<long long> acc_off(L, -1);
    std::vector<int32_t> acc_len(L, 0);
    DevScope tmp;
    int32_t* d_col = nullptr; long long* d_off = nullptr; int32_t* d_len = nullptr; char* d_pool = nullptr;
    size_t extra = 0;
    if (nins > 0) {
        for (int64_t i = 0; i < nins; ++i)
            if (ins_off[i] < 0 || ins_len[i] < 0 || ins_off[i] + ins_len[i] > pool_len) MS_FAIL(h, MS_ERR_ARG, "insertion event outside the pool");
        int64_t ts = 1024;
        while (ts < 2 * nins) ts <<= 1;
        unsigned long long* t_key = nullptr; uint32_t* t_cnt = nullptr; long long* t_rep = nullptr;
        ms::InsCand* d_cand = nullptr; unsigned long long* d_n = nullptr;
        MS_CUDA(h, tmp.alloc(&d_col, nins * 4)); MS_CUDA(h, tmp.alloc(&d_off, nins * 8)); MS_CUDA(h, tmp.alloc(&d_len, nins * 4));
        MS_CUDA(h, tmp.alloc(&d_pool, std::max<int64_t>(1, pool_len)));
        MS_CUDA(h, tmp.alloc(&t_key, ts * 8)); MS_CUDA(h, tmp.alloc(&t_cnt, ts * 4)); MS_CUDA(h, tmp.alloc(&t_rep, ts * 8));
        MS_CUDA(h, tmp.alloc(&d_cand, nins * sizeof(ms::InsCand))); MS_CUDA(h, tmp.alloc(&d_n, 8));
        MS_CUDA(h, cudaMemcpyAsync(d_col, ins_col, nins * 4, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_off, ins_off, nins * 8, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_len, ins_len, nins * 4, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(d_pool, ins_pool, pool_len, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemsetAsync(t_key, 0, ts * 8, h->stream));
        MS_CUDA(h, cudaMemsetAsync(t_cnt, 0, ts * 4, h->stream));
        MS_CUDA(h, cudaMemsetAsync(t_rep, 0x7f, ts * 8, h->stream));
        MS_CUDA(h, cudaMemsetAsync(d_n, 0, 8, h->stream));
        ms::ins_tally_kernel<<<static_cast<int>((nins + 255) / 256), 256, 0, h->stream>>>(d_col, d_off, d_len, nins, d_pool, t_key, t_cnt, t_rep, ts - 1);
        ms::ins_eval_kernel<<<static_cast<int>((ts + 255) / 256), 256, 0, h->stream>>>(t_cnt, t_rep, ts, d_col, d_len, h->d_counts, L,
                                                                                     prm->ins_fraction, d_cand, d_n, nins);
        h->launches += 2;
        unsigned long long nc = 0;
        MS_CUDA(h, cudaMemcpyAsync(&nc, d_n, 8, cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        std::vector<ms::InsCand> cand(nc);
        if (nc) {
            MS_CUDA(h, cudaMemcpyAsync(cand.data(), d_cand, nc * sizeof(ms::InsCand), cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
        }
        // exactness guard against a 64-bit hash collision: recount the survivors' strings
        for (const ms::InsCand& c : cand) {
            uint32_t exact = 0;
            for (int64_t i = 0; i < nins; ++i)
                if (ins_col[i] == c.col && ins_len[i] == c.len && memcmp(ins_pool + ins_off[i], ins_pool + ins_off[c.rep], c.len) == 0) ++exact;
            if (exact != c.cnt) MS_FAIL(h, MS_ERR_CUDA, "insertion hash collision");
        }
        std::sort(cand.begin(), cand.end(), [&](const ms::InsCand& a, const ms::InsCand& b) {
            if (a.col != b.col) return a.col < b.col;
            if (a.len != b.len) return a.len < b.len;
            return memcmp(ins_pool + ins_off[a.rep], ins_pool + ins_off[b.rep], a.len) < 0;
        });
        int32_t last = -1;
        for (const ms::InsCand& c : cand) {  // greedy spacing, left to right
            if (acc_off[c.col] >= 0) continue;
            if (last >= 0 && c.col - last < prm->ins_distance) continue;
            acc_off[c.col] = ins_off[c.rep]; acc_len[c.col] = c.len; last = c.col;
            extra += static_cast<size_t>(c.len);
        }
    }
    long long* d_acc_off = nullptr; int32_t* d_acc_len = nullptr; long long* d_outlen = nullptr;
    MS_CUDA(h, tmp.alloc(&d_acc_off, static_cast<size_t>(L) * 8)); MS_CUDA(h, tmp.alloc(&d_acc_len, static_cast<size_t>(L) * 4));
    MS_CUDA(h, tmp.alloc(&d_outlen, 8));
    cudaFree(h->d_seq); h->d_seq = nullptr;
    MS_CUDA(h, cudaMalloc(&h->d_seq, static_cast<size_t>(L) + extra + 16));
    MS_CUDA(h, cudaMemcpyAsync(d_acc_off, acc_off.data(), static_cast<size_t>(L) * 8, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(d_acc_len, acc_len.data(), static_cast<size_t>(L) * 4, cudaMemcpyHostToDevice, h->stream));
    ms::consensus_kernel<<<1, 1024, 0, h->stream>>>(h->d_counts, L, prm->min_coverage, d_acc_off, d_acc_len, d_pool, h->d_seq, d_outlen);
    h->launches++;
    long long n = 0;
    MS_CUDA(h, cudaMemcpyAsync(&n, d_outlen, 8, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    if (seq && cap > 0 && n > 0)
        MS_CUDA(h, cudaMemcpy(seq, h->d_seq, static_cast<size_t>(std::min<int64_t>(cap, n)), cudaMemcpyDeviceToHost));
    MS_CUDA(h, cudaGetLastError());
    *len = n;
    return MS_OK;
}

}  // extern "C"
