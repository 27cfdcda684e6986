// pileup.cuh -- K1: juliet/fuse pileup over planar 4-bit packed reads (sm_100a).
//
// Replaces the per-column "MSA counts" and per-codon coverage/observed-codon
// counts juliet derives from the alignment (/root/reference/doc/JULIET.md:96-100,
// screenshot juliet_hiv-context.png) and fuse's per-column tallies
// (/root/reference/doc/FUSE.md:17-20).  SURVEY.md rows a4, a5.
//
// Design (DESIGN.md "K1"): at the HBM roofline one SM must absorb ~46 columns per
// clock, far beyond shared-memory atomic throughput, so nothing is counted with
// atomics.  A thread owns one 32-column block and walks down the reads; the four
// bit-planes of each read give 32-wide one-bit masks, which are summed with
// bit-sliced carry-save adders (Harley-Seal) into 11-plane vertical counters held
// in registers.  Codons: a per-column "pivot" base (majority of a read sample)
// turns "read carries the pivot codon" into three shifted ANDs; only the rare
// clean non-pivot codons go to the 64-bin histogram, with a global RED.
// Read tiles are staged into shared memory by cp.async.bulk (UBLKCP) behind an
// mbarrier full/empty ring driven by one producer lane.  At the end the row-groups
// of a CTA add their vertical counters bit-sliced through shared memory, one group
// bit-transposes them into per-column integers and stores the CTA's slice; a small
// finalize kernel sums the <=148 slices into the count tensor.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ms {

constexpr int kPlanes = 11;             // vertical counter planes held in registers
constexpr int kPlanesAll = 13;          // + two planes per mask in shared memory (HI instantiations)
constexpr int kMaxReadsPerFlush = 2047;     // reads of a row-group between flushes: register planes only ...
constexpr int kMaxReadsPerFlushHi = 8191;   // ... and with the two shared-memory planes
// shared memory in front of the chunk slots: mbarriers + release counters (2 KB); HI instantiations add the two upper
// counter planes (2 planes x up to 9 masks x 384 threads).  The plain kernel keeps the small header: the shared memory it
// does not claim stays L1, and K1 lost ~5 % at 1M x 3 kb with 27 KB less of it.
constexpr int kPileupHiOffset = 2048;
constexpr int kPileupSmemHeader = 2048;
constexpr int kPileupSmemHeaderHi = 2048 + 2 * 9 * 384 * 4;
constexpr int kPileupMaxThreads = 384;  // 12 warps = 3 per SM sub-partition -> 168 registers per thread

// which one-bit masks are counted
enum PileupMode { kModeJuliet = 0,  // 6 state sums + "not the pivot codon"
                  kModeFuse = 1,    // 6 state sums + insertion flag
                  kModeBoth = 2 };  // all 8

struct PileupArgs {
    const uint32_t* packed;   // R rows of row_words u32
    int64_t R;
    int32_t L;
    int32_t nblk;             // ceil(L/32)
    int32_t warps_per_group;  // W = ceil(nblk/32)
    int32_t groups;           // G row-groups per CTA
    int32_t nseg, seg_len;    // column segments: CTA c handles blocks [seg_len*(c%nseg), +seg_len) of its reads
    int32_t stages, stages_hi;   // ring depth of the plain and of the HI instantiation (smaller header / larger header)
    int32_t stage_bytes;      // G*8*row_bytes
    const uint2* pivot;       // [nblk+1] {r0, r1} planes of the pivot base
    const uint2* pivot2;      // [nblk+1] DENSE: planes of the designated base (runner-up of the sample where frequent, else the pivot)
    const uint32_t* start_mask; // [nblk] codon start columns
    uint32_t* codon;          // [L][64] global histogram (exceptions land here)
    uint32_t* part_col;       // [gridDim][nblk*32][8]
    uint32_t* part_piv;       // [gridDim][nblk*32]
    uint32_t* part_piv2;      // [gridDim][nblk*32] DENSE: designated-codon counts
    uint4* exc_list;          // [gridDim*blockDim][exc_cap] blocks of the reads logged for the exact codon pass (ExcLog, pileup.cu)
    uint32_t* exc_cnt;        // [gridDim*blockDim]
    uint32_t exc_cap;
    int64_t exc_lists;        // gridDim*blockDim of the pileup launch
};

template <int MODE, bool DENSE, bool SEG, bool HI>
__global__ void pileup_csa_kernel(PileupArgs a);

__global__ void pivot_sample_kernel(const uint32_t* packed, int64_t R, int32_t nblk, int32_t L,
                                    uint2* pivot, uint8_t* pivot_state, uint2* pivot2, uint8_t* pivot2_state, uint32_t* dense_stat);
__global__ void pileup_finalize_kernel(const uint32_t* part_col, const uint32_t* part_piv, const uint32_t* part_piv2, int32_t slices,
                                       int32_t nblk, int32_t L, const uint8_t* pivot_state, const uint8_t* pivot2_state,
                                       const uint32_t* start_mask, uint32_t* col, uint32_t* codon,
                                       int32_t count_codons, int32_t nseg, int32_t seg_len);
__global__ void pileup_atomic_kernel(const uint32_t* packed, int64_t R, int32_t L, int32_t nblk,
                                     const uint32_t* start_mask, uint32_t* col, uint32_t* codon,
                                     int32_t count_codons);
__global__ void coverage_kernel(uint32_t* col, int32_t L);

// ---------------------------------------------------------------- bit-sliced counting helpers
// Shared by K1 (pileup.cu) and the grouped pile-up (group.cu).
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// carry-save adder: (h,l) = a + b + c per bit position.  Two LOP3.
__device__ __forceinline__ void csa(uint32_t& h, uint32_t& l, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t u = a ^ b;
    h = (a & b) | (u & c);
    l = u ^ c;
}

template <int NM>
struct Vert {
    uint32_t c[NM][kPlanes];  // vertical counters, plane k has weight 2^k
    uint32_t p3[NM], p4[NM], p5[NM];  // pending carry-save inputs of weight 8, 16 and 32
};

// Planes kPlanes and kPlanes+1 (weights 2048 and 4096) live in shared memory, one word per thread and mask: a carry out of
// the register planes reaches them once per 2048 reads of a column, so they cost nothing in the hot loop and lift the
// capacity of a row-group from 2047 to 8191 reads -- which keeps the barrier-ordered mid-kernel flush out of every
// workload of ordinary size (it costs G serialised read-modify-write rounds over the CTA's slice).  HI is a template
// switch: K1 sits at its register limit, and carrying the two extra values cost the 1M x 3 kb kernel 5 %, so launches
// whose row-groups stay below 2048 reads use the instantiation without it.
struct HiPlanes {
    uint32_t base;     // shared-memory address of this thread's word of (plane kPlanes, mask 0)
    uint32_t stride;   // bytes between consecutive masks (= threads * 4); plane kPlanes+1 follows the NM masks of plane kPlanes
};
template <int NM>
__device__ __forceinline__ void hi_add(const HiPlanes& hp, int i, uint32_t x) {
    const uint32_t a0 = hp.base + static_cast<uint32_t>(i) * hp.stride;
    const uint32_t p = lds32(a0);
    sts32(a0, p ^ x);
    const uint32_t c = p & x;
    if (c) {
        const uint32_t a1 = a0 + static_cast<uint32_t>(NM) * hp.stride;
        sts32(a1, lds32(a1) ^ c);     // capacity checked by the caller (kMaxReadsPerFlush): no carry out of this one
    }
}

template <bool HI, int NM>
__device__ __forceinline__ void ripple(Vert<NM>& v, const HiPlanes& hp, int i, int level, uint32_t x) {
#pragma unroll
    for (int k = 0; k < kPlanes; ++k) {
        if (k >= level) {
            const uint32_t t = v.c[i][k] & x;
            v.c[i][k] ^= x;
            x = t;
        }
    }
    if (HI) {
        if (x) hi_add<NM>(hp, i, x);
    }
}

template <bool HI, int NM>
__device__ __forceinline__ void fold_pendings(Vert<NM>& v, const HiPlanes& hp, uint32_t bi) {
#pragma unroll
    for (int i = 0; i < NM; ++i) {
        if (bi & 1u) ripple<HI>(v, hp, i, 3, v.p3[i]);
        if (bi & 2u) ripple<HI>(v, hp, i, 4, v.p4[i]);
        if (bi & 4u) ripple<HI>(v, hp, i, 5, v.p5[i]);
    }
}

template <bool HI, int NM>
__device__ __forceinline__ void clear(Vert<NM>& v, const HiPlanes& hp) {
#pragma unroll
    for (int i = 0; i < NM; ++i) {
#pragma unroll
        for (int k = 0; k < kPlanes; ++k) v.c[i][k] = 0;
        v.p3[i] = v.p4[i] = v.p5[i] = 0;
        if (HI) {
            sts32(hp.base + static_cast<uint32_t>(i) * hp.stride, 0u);
            sts32(hp.base + static_cast<uint32_t>(NM + i) * hp.stride, 0u);
        }
    }
}

// 16 words x 32 bits holding two 16x16 bit matrices side by side: after the call, word j has
// bit k (low half) = old word k bit j, and bit 16+k (high half) = old word k bit 16+j.
__device__ __forceinline__ void transpose16x2(uint32_t (&a)[16]) {
#pragma unroll
    for (int s = 8; s >= 1; s >>= 1) {
        const uint32_t m = s == 8 ? 0x00FF00FFu : s == 4 ? 0x0F0F0F0Fu : s == 2 ? 0x33333333u : 0x55555555u;
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            if (k & s) continue;
            const uint32_t t = ((a[k] >> s) ^ a[k + s]) & m;
            a[k + s] ^= t;
            a[k] ^= t << s;
        }
    }
}

// Exact per-column counts {A,C,G,T} {-,N,ins,cov} of n reads from the column sums of the six state masks
// s0 = sum P0, s1 = sum P1, s2 = sum P2, s3 = sum P0&P1, s4 = sum P0&P2, s5 = sum P1&P2 (states A=000 C=001 G=010 T=011
// -=100 N=101 U=111).  Not-spanned reads (U) drop out: they are the reads of n that are not in cov.
template <int NS>
__device__ __forceinline__ void decode_counts(const uint32_t (&s)[NS], uint32_t ins, uint32_t n, uint4& lo, uint4& hi) {
    const uint32_t nU = s[5];
    const uint32_t nN = s[4] - nU;
    const uint32_t nT = s[3] - nU;
    const uint32_t nD = s[2] - nN - nU;
    const uint32_t nG = s[1] - nT - nU;
    const uint32_t nC = s[0] - nT - nN - nU;
    const uint32_t cov = n - nU;
    const uint32_t nA = cov - (nC + nG + nT + nD + nN);
    lo = make_uint4(nA, nC, nG, nT);
    hi = make_uint4(nD, nN, ins, cov);
}

void pileup_set_smem_attr(int max_smem);
void pileup_launch(int mode, bool dense, bool hi, int grid, int threads, int smem, cudaStream_t s, const PileupArgs& a);
void pileup_exceptions_launch(bool dense, int pileup_grid, int pileup_threads, cudaStream_t s, const PileupArgs& a);

}  // namespace ms
