// phase_internal.cuh -- pieces of K3 shared by phase.cu (bit-vectors, local grouping table) and
// phase_order.cu (cross-rank merge + ordering on the device).
#pragma once
#include "handle.h"

namespace ms {

__device__ __forceinline__ uint64_t mix64d(uint64_t x) {
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL;
    x ^= x >> 27; x *= 0x94d049bb133111ebULL;
    x ^= x >> 31;
    return x;
}

__device__ __forceinline__ uint64_t pattern_hash(const uint32_t* w, int32_t vwords, uint64_t seed) {
    uint64_t hsh = seed;
    for (int32_t i = 0; i < vwords; ++i) hsh = mix64d(hsh ^ (static_cast<uint64_t>(w[i]) + 0x9E3779B97F4A7C15ULL * (i + 1)));
    return hsh ? hsh : 1ULL;
}

// juliet's haplotype order among equal counts: ascending pattern words, word 0 first
__host__ __device__ __forceinline__ bool pattern_less(const uint32_t* a, const uint32_t* b, int32_t nw) {
    for (int32_t i = 0; i < nw; ++i)
        if (a[i] != b[i]) return a[i] < b[i];
    return false;
}

inline uint64_t phase_seed(int attempt) { return 0x6d696e6f72736571ULL + 0x9E3779B97F4A7C15ULL * static_cast<uint64_t>(attempt); }

// ctr layout (u64): [0] damaged [1] gaps [2] heteroduplex [3] partial [4] hash collisions [5] ngroups [6] table overflow [7] spare
inline unsigned long long* phase_ctr(ms_handle* h) { return h->b_ctr.as<unsigned long long>(); }

// Device-built phasing plan (phase_plan_kernel): the pooled variant list and the word stream of phase_bits_kernel made on the
// GPU from K2's output, so that the juliet pass needs no host round trip between the codon test and the bit-vectors.
// Covers the usual case -- at most 32 distinct (column, codon) keys from at most 64 calls; anything else sets `fallback`
// and the host builds the plan (ms_phase_begin) after all.
constexpr int kPlanMaxKeys = 32, kPlanMaxCalls = 64, kPlanMaxBlocks = 64, kPlanMaxLayers = 4;
constexpr int kPlanStreamWords = kPlanMaxBlocks * kPlanMaxLayers * 5 + kPlanMaxKeys;
struct PhasePlan {
    int32_t V, NB, nwords, partial_all, fallback, ncalls;
    int32_t key_col[kPlanMaxKeys], key_codon[kPlanMaxKeys];
};

// ---- grouping (phase.cu) and ordering (phase_order.cu) kernels; haplotype abundance (abundance.cu) runs them as well, on its
// per-read compatibility masks instead of the phasing bits ----
constexpr int64_t kSmallSort = 4096;   // up to this many distinct entries are ranked by counting, more are sorted

__global__ void __launch_bounds__(256) phase_clear_kernel(unsigned long long* __restrict__ tab_key, uint32_t* __restrict__ tab_cnt,
                                                          long long* __restrict__ tab_rep, int64_t tab_size, unsigned long long* __restrict__ ctr,
                                                          unsigned long long last_resort);
__global__ void phase_insert_kernel(const uint32_t* __restrict__ bits, const uint8_t* __restrict__ flags, int64_t R,
                                    int32_t vwords, uint64_t seed, unsigned long long* tab_key, uint32_t* tab_cnt,
                                    long long* tab_rep, int64_t mask, int32_t* __restrict__ slot, unsigned long long* overflow);
__global__ void phase_verify_kernel(const uint32_t* __restrict__ bits, int64_t R, int32_t vwords,
                                    const long long* __restrict__ tab_rep, const int32_t* __restrict__ slot,
                                    unsigned long long* collision);
__global__ void phase_compact_kernel(const uint32_t* __restrict__ tab_cnt, const long long* __restrict__ tab_rep,
                                     int64_t tab_size, const uint32_t* __restrict__ bits, int32_t vwords,
                                     unsigned long long* ngroups, uint32_t* __restrict__ g_cnt,
                                     uint32_t* __restrict__ g_pat, int32_t* __restrict__ g_slot, int64_t cap);

// result header (u64[8]) at the start of the out block:
// [0] merged distinct M (world > 1)  [1] nreported  [2] reported reads  [3] insufficient reads
// [4] "too many for counting rank"   [5] merge hash collisions  [6] merge table overflow
struct OrderOut {
    unsigned long long* res;
    uint32_t* rank;    // entry -> position in the order
    uint32_t* o_cnt;   // position -> count, first ocap positions
    uint32_t* o_pat;   // position -> pattern, first ocap positions
    int64_t ocap;
    uint32_t min_reads;
};

// ---- merge of the all-gathered compact lists: block r = [64-byte header | cnt u32[gcap] | pat u32[gcap*nw]] ----
struct Gathered {
    const uint8_t* base;
    size_t block;
    int64_t gcap;
    int32_t nw;
    __device__ __forceinline__ int64_t ng(int64_t rnk) const {
        const unsigned long long n = reinterpret_cast<const unsigned long long*>(base + rnk * block)[5];
        return n < static_cast<unsigned long long>(gcap) ? static_cast<int64_t>(n) : gcap;
    }
    __device__ __forceinline__ uint32_t cnt(int64_t e) const {
        const int64_t rnk = e / gcap;
        return reinterpret_cast<const uint32_t*>(base + rnk * block + 64)[e - rnk * gcap];
    }
    __device__ __forceinline__ const uint32_t* pat(int64_t e) const {
        const int64_t rnk = e / gcap;
        return reinterpret_cast<const uint32_t*>(base + rnk * block + 64) + gcap + static_cast<size_t>(e - rnk * gcap) * nw;
    }
};

__global__ void __launch_bounds__(256) rank_small_kernel(const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ pat, int32_t nw,
                                                         const unsigned long long* __restrict__ Mptr, int64_t bound,
                                                         const uint8_t* __restrict__ hdr_src, size_t hdr_stride, int32_t world, OrderOut o);
__global__ void __launch_bounds__(256) emit_sorted_kernel(const uint32_t* __restrict__ ord, const uint32_t* __restrict__ cnt,
                                                          const uint32_t* __restrict__ pat, int32_t nw, int64_t M, OrderOut o);
__global__ void merge_insert_kernel(Gathered g, int64_t bound, uint64_t seed, unsigned long long* mt_key, uint32_t* mt_cnt,
                                    unsigned long long* mt_rep, int64_t mask, int32_t* __restrict__ mslot, unsigned long long* res);
__global__ void merge_verify_kernel(Gathered g, int64_t bound, const unsigned long long* __restrict__ mt_rep, const int32_t* __restrict__ mslot,
                                    unsigned long long* res);
__global__ void merge_compact_kernel(Gathered g, const uint32_t* __restrict__ mt_cnt, const unsigned long long* __restrict__ mt_rep, int64_t tsize,
                                     unsigned long long* res, uint32_t* __restrict__ m_cnt, uint32_t* __restrict__ m_pat,
                                     uint32_t* __restrict__ m_index);
// bitonic sort of the entry indices 0..M-1 by (count desc, pattern asc); result in h->b_ord (n_pad entries, sentinels last)
int sort_big(ms_handle* h, const uint32_t* cnt, const uint32_t* pat, int32_t nw, int64_t M, int64_t* n_pad_out);

int phase_ensure_stage(ms_handle* h, size_t bytes);
int phase_build_table(ms_handle* h, int attempt);
// enqueue: distinct patterns of the local table -> g_cnt/g_pat (and the table slot of each in g_slot, may be null); count in ctr[5]
int phase_compact(ms_handle* h, uint32_t* g_cnt, uint32_t* g_pat, int32_t* g_slot, int64_t cap);
// after a host look at ctr[6]: grow the table (x8) for the next build; fails at the maximum size
int phase_grow_table(ms_handle* h);

}  // namespace ms
