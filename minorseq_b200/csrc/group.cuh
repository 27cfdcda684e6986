// group.cuh -- the grouped pile-up's walk (group.cu), shared with the in-frame indel counts (indel.cu).
//
// Persistent CTAs walk work items (a chunk of <= kGroupChunk reads, one column segment).  A thread owns one 32-column block;
// it gathers that block (and, for SLOTS = 2, the next one) of each read of the item from the tiles with cp.async, two batches
// of 8 reads ahead, forms the policy's one-bit masks and adds them into K1's bit-sliced carry-save counters (pileup.cuh).  At
// the end of an item the policy turns the counter planes into per-column integers and adds them into global memory with RED.
// Counts are integer sums: the order in which reads are visited changes locality, never a result.
//
// A policy P provides NM (masks per read), SLOTS (16-byte blocks per read: b, b+1, ...) and
//   int32_t item(int32_t k, int32_t& r_begin, int32_t& r_end)   the list positions of work item k, and a tag for flush
//   int64_t read(int32_t idx)                                    the read at list position idx
//   static void masks(uint32_t addr, uint32_t stride, uint32_t (&m)[NM])   masks of one read: block s at addr + s * stride
//   void flush(const uint32_t* planes, uint32_t n, int32_t tag, int b)     planes [NM][kPlanes] of n reads of block b
#pragma once
#include "pileup.cuh"

namespace ms {

constexpr int kGroupChunk = 8 * (kMaxReadsPerFlush / 8);   // reads per work item: whole batches of 8 within K1's counter capacity
constexpr int kGroupMaxThreads = 256;                      // one thread per 32-column block of a segment
constexpr int kGroupRing = 3;                              // batches of 8 reads per thread in the cp.async ring

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ uint4 lds128g(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint4 v) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// 8 reads (read i at addr + i * rstride) into the counters: K1's carry-save tree (pileup.cu, block8)
template <class P>
__device__ __forceinline__ void csa_add8(Vert<P::NM>& v, const HiPlanes& hp, uint32_t addr, uint32_t rstride, uint32_t stride, uint32_t bi) {
    constexpr int NM = P::NM;
    uint32_t m0[NM], m1[NM], twosA[NM], twosB[NM], foursA[NM], foursB[NM];
    P::masks(addr, stride, m0);
    P::masks(addr + rstride, stride, m1);
#pragma unroll
    for (int i = 0; i < NM; ++i) csa(twosA[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
    P::masks(addr + 2 * rstride, stride, m0);
    P::masks(addr + 3 * rstride, stride, m1);
#pragma unroll
    for (int i = 0; i < NM; ++i) {
        csa(twosB[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
        csa(foursA[i], v.c[i][1], v.c[i][1], twosA[i], twosB[i]);
    }
    P::masks(addr + 4 * rstride, stride, m0);
    P::masks(addr + 5 * rstride, stride, m1);
#pragma unroll
    for (int i = 0; i < NM; ++i) csa(twosA[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
    P::masks(addr + 6 * rstride, stride, m0);
    P::masks(addr + 7 * rstride, stride, m1);
#pragma unroll
    for (int i = 0; i < NM; ++i) {
        csa(twosB[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
        csa(foursB[i], v.c[i][1], v.c[i][1], twosA[i], twosB[i]);
        csa(twosA[i], v.c[i][2], v.c[i][2], foursA[i], foursB[i]);  // twosA now holds the weight-8 carry
    }
    if (bi & 1u) {
        if (bi & 2u) {
            if (bi & 4u) {
#pragma unroll
                for (int i = 0; i < NM; ++i) {
                    uint32_t x16, x32, x64;
                    csa(x16, v.c[i][3], v.c[i][3], v.p3[i], twosA[i]);
                    csa(x32, v.c[i][4], v.c[i][4], v.p4[i], x16);
                    csa(x64, v.c[i][5], v.c[i][5], v.p5[i], x32);
                    ripple<false>(v, hp, i, 6, x64);
                }
            } else {
#pragma unroll
                for (int i = 0; i < NM; ++i) {
                    uint32_t x16;
                    csa(x16, v.c[i][3], v.c[i][3], v.p3[i], twosA[i]);
                    csa(v.p5[i], v.c[i][4], v.c[i][4], v.p4[i], x16);
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < NM; ++i) csa(v.p4[i], v.c[i][3], v.c[i][3], v.p3[i], twosA[i]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < NM; ++i) v.p3[i] = twosA[i];
    }
}

// the body of a persistent walk kernel; dynamic shared memory: kGroupRing * 8 * P::SLOTS * blockDim * 16 bytes
template <class P>
__device__ __forceinline__ void csa_walk(const P& p, const uint4* __restrict__ tiles, int32_t nblk, int32_t nseg, int32_t seg_len,
                                         int64_t nitems) {
    extern __shared__ __align__(16) uint4 ring[];   // [kGroupRing * 8 * SLOTS][blockDim]: batch slot s, read i, block j at row (s * 8 + i) * SLOTS + j
    const int tid = threadIdx.x;
    const uint32_t stride = static_cast<uint32_t>(blockDim.x) * 16u;        // bytes between rows of the ring
    const uint32_t rstride = stride * P::SLOTS;                              // bytes between the reads of a batch
    const uint32_t ring0 = static_cast<uint32_t>(__cvta_generic_to_shared(ring)) + static_cast<uint32_t>(tid) * 16u;
    HiPlanes hp;
    hp.base = hp.stride = 0;
    Vert<P::NM> v;
    for (int64_t it = blockIdx.x; it < nitems; it += gridDim.x) {
        const int seg = static_cast<int>(it % nseg);
        const int32_t k = static_cast<int32_t>(it / nseg);
        const int b = seg * seg_len + tid;
        if (tid >= seg_len || b >= nblk) continue;          // no barriers below: idle lanes may leave the item
        int32_t r_begin, r_end;
        const int32_t tag = p.item(k, r_begin, r_end);
        const int32_t nb = (r_end - r_begin + 7) >> 3;      // batches of 8; the slots past r_end hold "not spanned" reads
        auto load = [&](int32_t batch) {
            const uint32_t slot = ring0 + static_cast<uint32_t>(batch % kGroupRing) * 8u * rstride;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int32_t idx = r_begin + batch * 8 + i;
#pragma unroll
                for (int j = 0; j < P::SLOTS; ++j) {
                    const uint32_t dst = slot + static_cast<uint32_t>(i) * rstride + static_cast<uint32_t>(j) * stride;
                    const int bj = b + j;
                    if (idx < r_end && bj < nblk) {
                        const int64_t r = p.read(idx);
                        cp_async16(dst, tiles + (((r >> 3) * nblk + bj) << 3) + ((r & 7) ^ (bj & 7)));
                    } else {
                        sts128(dst, make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0u));
                    }
                }
            }
        };
        clear<false>(v, hp);
#pragma unroll
        for (int q = 0; q < kGroupRing - 1; ++q) {
            if (q < nb) load(q);
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        uint32_t bi = 0;
        for (int32_t j = 0; j < nb; ++j) {
            if (j + kGroupRing - 1 < nb) load(j + kGroupRing - 1);   // into the slot batch j - 1 has left
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group %0;" ::"n"(kGroupRing - 1) : "memory");   // batch j has landed
            csa_add8<P>(v, hp, ring0 + static_cast<uint32_t>(j % kGroupRing) * 8u * rstride, rstride, stride, bi);
            ++bi;
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        fold_pendings<false>(v, hp, bi);
        uint32_t planes[P::NM * kPlanes];
#pragma unroll
        for (int i = 0; i < P::NM; ++i)
#pragma unroll
            for (int q = 0; q < kPlanes; ++q) planes[i * kPlanes + q] = v.c[i][q];
        p.flush(planes, static_cast<uint32_t>(nb) * 8u, tag, b);
    }
}

}  // namespace ms
