// pileup.cu -- K1 kernels.  See pileup.cuh for the design and reference citations.
#include "pileup.cuh"
#include "rows.cuh"

namespace ms {

// ---------------------------------------------------------------- PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
// bulk global->shared copy completing on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
        "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void consumer_barrier(int nthreads) {
    asm volatile("bar.sync 1, %0;" ::"r"(nthreads) : "memory");
}

// DENSE: a second bit-sliced codon count per start column -- the "designated" codon (runner-up base of the pivot sample
// wherever it holds > 2 % of the sample, the pivot base elsewhere), see the DENSE notes at read_masks.
template <int MODE, bool DENSE>
struct Traits {
    static constexpr int NM = (MODE == kModeBoth ? 8 : 7) + (DENSE ? 1 : 0);
    static constexpr bool CODON = MODE != kModeFuse;
    static constexpr bool INS = MODE != kModeJuliet;
    static constexpr int iINS = 6;
    static constexpr int iNP = MODE == kModeBoth ? 7 : 6;  // "not the pivot codon"
    static constexpr int iND = iNP + 1;                    // "not the designated codon" (DENSE only)
};

// ---------------------------------------------------------------- per-thread state (Vert, HiPlanes: pileup.cuh)
// Per-thread constants for codon work
struct CodonCtx {
    uint32_t r0, r1, r0n, r1n;  // pivot planes of this block and the next (the latter only for the rare path)
    uint32_t d0, d1, d0n, d1n;  // DENSE: planes of the designated base (second pivot where there is one)
    uint32_t start;             // codon start columns in this block
    uint32_t cols;              // columns of this block that belong to a codon starting in this block
    uint32_t lookcols;          // same for the first two columns of the next block (bits 0, 1)
    uint32_t* codon;            // this block's rows of the global [L][64] histogram
};

// exact masks (rare path): "codon starting at column j is not the clean pivot codon" and the clean ones among them
template <bool DENSE>
__device__ __forceinline__ void codon_masks(const uint4& q, const uint4& n, const CodonCtx& cx, uint32_t& np, uint32_t& e) {
    const uint32_t X = ((q.x ^ cx.r0) | q.z) | (q.y ^ cx.r1);  // column is not the clean pivot base
    const uint32_t Xn = ((n.x ^ cx.r0n) | n.z) | (n.y ^ cx.r1n);
    np = X | __funnelshift_r(X, Xn, 1) | __funnelshift_r(X, Xn, 2);
    const uint32_t dirty = q.z | __funnelshift_r(q.z, n.z, 1) | __funnelshift_r(q.z, n.z, 2);
    e = ~dirty & np & cx.start;  // clean codon that is not the pivot codon: rare
    if (DENSE) {                 // ... and not the designated codon either (that one is counted bit-sliced as well)
        const uint32_t D = ((q.x ^ cx.d0) | q.z) | (q.y ^ cx.d1);
        const uint32_t Dn = ((n.x ^ cx.d0n) | n.z) | (n.y ^ cx.d1n);
        e &= D | __funnelshift_r(D, Dn, 1) | __funnelshift_r(D, Dn, 2);
    }
}

// Build the one-bit masks of one read for this thread's 32 columns.
// Hot path of the codon work: the per-column mismatch mask X is computed once per block; the
// look-ahead into the next block comes from the neighbouring lane by shuffle (lane 31 of every
// warp but the last of a row is a pure look-ahead provider, see the lane mapping in pileup_body).
// A read is flagged for the exact rare path when a clean non-pivot BASE sits in a column that
// belongs to one of this block's codons -- a superset of "has a clean non-pivot codon".
// DENSE (frequent variants: a second codon in a sizeable share of the reads at many positions -- phasing stress data): the
// designated codon is counted exactly like the pivot codon, as one more carry-save mask, and a read is flagged for the rare
// path only when one of this block's start columns holds a clean codon that is NEITHER (exact, three more LOP3/SHF than the
// conservative trigger).  Results stay exact for any choice of the two bases per column.
template <int MODE, bool DENSE>
__device__ __forceinline__ void read_masks(uint32_t addr, const CodonCtx& cx, uint32_t (&m)[Traits<MODE, DENSE>::NM], uint32_t& pm,
                                           uint32_t rdbit) {
    using T = Traits<MODE, DENSE>;
    const uint4 q = lds128(addr);
    m[0] = q.x;
    m[1] = q.y;
    m[2] = q.z;
    m[3] = q.x & q.y;
    m[4] = q.x & q.z;
    m[5] = q.y & q.z;
    if (T::INS) m[T::iINS] = q.w;
    if (T::CODON) {
        const uint32_t X = ((q.x ^ cx.r0) | q.z) | (q.y ^ cx.r1);  // column is not the clean pivot base
        const uint32_t Xn = __shfl_down_sync(0xffffffffu, X, 1);
        const uint32_t zn = __shfl_down_sync(0xffffffffu, q.z, 1);
        const uint32_t np = X | __funnelshift_r(X, Xn, 1) | __funnelshift_r(X, Xn, 2);
        m[T::iNP] = np;
        if (DENSE) {
            const uint32_t D = ((q.x ^ cx.d0) | q.z) | (q.y ^ cx.d1);  // column is not the clean designated base
            const uint32_t Dn = __shfl_down_sync(0xffffffffu, D, 1);
            const uint32_t nd = D | __funnelshift_r(D, Dn, 1) | __funnelshift_r(D, Dn, 2);
            m[T::iND] = nd;
            const uint32_t dirty = q.z | __funnelshift_r(q.z, zn, 1) | __funnelshift_r(q.z, zn, 2);
            if (np & nd & ~dirty & cx.start) pm |= rdbit;
        } else {
            const uint32_t trig = (X & ~q.z & cx.cols) | (Xn & ~zn & cx.lookcols);
            if (trig) pm |= rdbit;
        }
    }
}

// Rare path: the reads flagged in pm may carry clean non-pivot codons; re-read them from the slot
// (still owned by this row-group) and add each such codon to the global 64-bin histogram.
// addr / naddr: this thread's block and the next one in the slot, swizzle folded in (read i at addr ^ 16 i).
template <bool DENSE>
__device__ __forceinline__ void codon_exceptions(uint32_t addr, uint32_t naddr, uint32_t pm, const CodonCtx& cx) {
    while (pm) {
        const int rd = __ffs(pm) - 1;
        pm &= pm - 1;
        const uint4 q = lds128(addr ^ (static_cast<uint32_t>(rd) << 4)), n = lds128(naddr ^ (static_cast<uint32_t>(rd) << 4));
        uint32_t np, e;
        codon_masks<DENSE>(q, n, cx, np, e);
        while (e) {
            const int j = __ffs(e) - 1;
            e &= e - 1;
            const uint32_t b0 = __funnelshift_r(q.x, n.x, j) & 7u;  // bit0 of the 3 states
            const uint32_t b1 = __funnelshift_r(q.y, n.y, j) & 7u;  // bit1 of the 3 states
            const uint32_t cod = ((b0 & 1u) << 4) | ((b1 & 1u) << 5) | ((b0 & 2u) << 1) | ((b1 & 2u) << 2) |
                                 ((b0 & 4u) >> 2) | ((b1 & 4u) >> 1);
            atomicAdd(cx.codon + (j * 64 + cod), 1u);
        }
    }
}

template <int MODE, bool DENSE, bool HI>
__device__ __forceinline__ uint32_t block8(uint32_t addr, const CodonCtx& cx, Vert<Traits<MODE, DENSE>::NM>& v, const HiPlanes& hp,
                                           uint32_t bi) {
    constexpr int NM = Traits<MODE, DENSE>::NM;
    uint32_t m0[NM], m1[NM], twosA[NM], twosB[NM], foursA[NM], foursB[NM];
    uint32_t pm = 0;
    // reads 0..3
    read_masks<MODE, DENSE>(addr, cx, m0, pm, 1u);   // read i of the tile sits at addr ^ 16 i (rows.cuh)
    read_masks<MODE, DENSE>(addr ^ 16u, cx, m1, pm, 2u);
#pragma unroll
    for (int i = 0; i < NM; ++i) csa(twosA[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
    read_masks<MODE, DENSE>(addr ^ 32u, cx, m0, pm, 4u);
    read_masks<MODE, DENSE>(addr ^ 48u, cx, m1, pm, 8u);
#pragma unroll
    for (int i = 0; i < NM; ++i) {
        csa(twosB[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
        csa(foursA[i], v.c[i][1], v.c[i][1], twosA[i], twosB[i]);
    }
    // reads 4..7
    read_masks<MODE, DENSE>(addr ^ 64u, cx, m0, pm, 16u);
    read_masks<MODE, DENSE>(addr ^ 80u, cx, m1, pm, 32u);
#pragma unroll
    for (int i = 0; i < NM; ++i) csa(twosA[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
    read_masks<MODE, DENSE>(addr ^ 96u, cx, m0, pm, 64u);
    read_masks<MODE, DENSE>(addr ^ 112u, cx, m1, pm, 128u);
#pragma unroll
    for (int i = 0; i < NM; ++i) {
        csa(twosB[i], v.c[i][0], v.c[i][0], m0[i], m1[i]);
        csa(foursB[i], v.c[i][1], v.c[i][1], twosA[i], twosB[i]);
        csa(twosA[i], v.c[i][2], v.c[i][2], foursA[i], foursB[i]);  // twosA now holds the weight-8 carry
    }
    // upper levels: combine the weight-8 words of successive blocks lazily (branches are CTA-uniform)
    if (bi & 1u) {
        if (bi & 2u) {
            if (bi & 4u) {
#pragma unroll
                for (int i = 0; i < NM; ++i) {
                    uint32_t x16, x32, x64;
                    csa(x16, v.c[i][3], v.c[i][3], v.p3[i], twosA[i]);
                    csa(x32, v.c[i][4], v.c[i][4], v.p4[i], x16);
                    csa(x64, v.c[i][5], v.c[i][5], v.p5[i], x32);
                    ripple<HI>(v, hp, i, 6, x64);
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
    return pm;  // reads of this block flagged for the exact codon pass
}

// Flagged reads are logged to this thread's private list in global memory (fire-and-forget stores)
// and resolved after the kernel by codon_exception_kernel with full parallelism; only when the
// list is full (dense-variation data) does the thread fall back to the in-kernel rare path.
// An entry is the flagged read's block itself -- planes P0 P1 P2 and, in the fourth word, the first two columns of the next
// block (2 bits of each plane) -- so the exception kernel never goes back to the rows: logging by reference made it re-read
// 256 bytes of row data per flagged read (403 MB at 1M x 3 kb, 85 us; 1.3 GB at 1M x 9.7 kb), the 16-byte entries are 27 MB.
struct ExcLog {
    uint4* list;
    uint32_t cnt, cap;
};
template <bool DENSE>
__device__ __forceinline__ void log_or_handle(uint32_t pm, ExcLog& lg, uint32_t addr, uint32_t naddr, const CodonCtx& cx) {
    if (lg.cnt + static_cast<uint32_t>(__popc(pm)) <= lg.cap) {
        while (pm) {
            const uint32_t rd = static_cast<uint32_t>(__ffs(pm) - 1);
            pm &= pm - 1;
            const uint4 q = lds128(addr ^ (rd << 4)), n = lds128(naddr ^ (rd << 4));
            lg.list[lg.cnt++] = make_uint4(q.x, q.y, q.z, (n.x & 3u) | ((n.y & 3u) << 2) | ((n.z & 3u) << 4));
        }
    } else {
        codon_exceptions<DENSE>(addr, naddr, pm, cx);
    }
}

// ---------------------------------------------------------------- flush (cold path)
// planes: this thread's counters (pendings already folded), [NM][NP] in local memory (NP = kPlanes, or kPlanesAll with the shared-memory planes).
// Adds the other groups' planes from shared memory (bit-sliced ripple-carry), transposes to
// per-column integers and stores / adds them into the CTA's slice.
template <int MODE, bool DENSE, int NP>
__device__ __noinline__ void emit_slice(const uint32_t* planes, uint32_t merge_base, int other_groups, uint32_t group_stride,
                                        uint32_t thread_stride, uint32_t n, uint32_t start, uint32_t* pc, uint32_t* pp, uint32_t* pd,
                                        bool add) {
    using T = Traits<MODE, DENSE>;
    constexpr int NM = T::NM;
    uint32_t tr[NM][16];
#pragma unroll
    for (int i = 0; i < NM; ++i) {
        uint32_t acc[16];
#pragma unroll
        for (int k = 0; k < 16; ++k) acc[k] = k < NP ? planes[i * NP + k] : 0u;
        for (int g = 0; g < other_groups; ++g) {
            uint32_t carry = 0;
            const uint32_t base = merge_base + static_cast<uint32_t>(g) * group_stride + static_cast<uint32_t>(i * NP) * thread_stride;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const uint32_t b = k < NP ? lds32(base + static_cast<uint32_t>(k) * thread_stride) : 0u;
                const uint32_t u = acc[k] ^ b;
                const uint32_t nc = (acc[k] & b) | (u & carry);
                acc[k] = u ^ carry;
                carry = nc;
            }
        }
        transpose16x2(acc);
#pragma unroll
        for (int k = 0; k < 16; ++k) tr[i][k] = acc[k];
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int colj = j + 16 * half;
            uint32_t s[NM];
#pragma unroll
            for (int i = 0; i < NM; ++i) s[i] = half ? (tr[i][j] >> 16) : (tr[i][j] & 0xffffu);
            uint4 lo, hi;
            decode_counts(s, T::INS ? s[T::iINS] : 0u, n, lo, hi);
            uint4* dst = reinterpret_cast<uint4*>(pc + colj * 8);
            if (add) {
                const uint4 x = dst[0], y = dst[1];
                lo.x += x.x; lo.y += x.y; lo.z += x.z; lo.w += x.w;
                hi.x += y.x; hi.y += y.y; hi.z += y.z; hi.w += y.w;
            }
            dst[0] = lo;
            dst[1] = hi;
            if (T::CODON) {
                uint32_t piv = ((start >> colj) & 1u) ? n - s[T::iNP] : 0u;
                if (add) piv += pp[colj];
                pp[colj] = piv;
                if (DENSE) {
                    uint32_t des = ((start >> colj) & 1u) ? n - s[T::iND] : 0u;
                    if (add) des += pd[colj];
                    pd[colj] = des;
                }
            }
        }
    }
}

// this thread's counters as kPlanesAll planes per mask: registers + the two shared-memory planes
template <bool HI, int NM>
__device__ __forceinline__ void gather_planes(const Vert<NM>& v, const HiPlanes& hp, uint32_t* planes) {
    constexpr int NP = HI ? kPlanesAll : kPlanes;
#pragma unroll
    for (int i = 0; i < NM; ++i) {
#pragma unroll
        for (int k = 0; k < kPlanes; ++k) planes[i * NP + k] = v.c[i][k];
        if (HI) {
            planes[i * NP + kPlanes] = lds32(hp.base + static_cast<uint32_t>(i) * hp.stride);
            planes[i * NP + kPlanes + 1] = lds32(hp.base + static_cast<uint32_t>(NM + i) * hp.stride);
        }
    }
}

template <int MODE, bool DENSE, bool SEG, bool HI>
__device__ __forceinline__ void pileup_body(const PileupArgs& a) {
    using T = Traits<MODE, DENSE>;
    constexpr int NM = T::NM;
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = a.warps_per_group, G = a.groups, S = HI ? a.stages_hi : a.stages;
    const int ncw = W * G;  // all warps are consumers; lane 0 of warp 0 also produces
    // Column segments: with nseg > 1 a CTA handles only the blocks [blk0, blk0 + seg_nblk) of its reads (plus one
    // look-ahead block of the next segment), so that row lengths whose warp count per row does not divide 12 still
    // fill the CTA with row-groups, and rows longer than 12 warps fit at all.  CTA c works on segment c % nseg.
    // SEG is a template parameter: the whole-row kernel must not carry any of this (K1 sits at its register limit and
    // lost 4 % to the mere presence of the segment arithmetic).
    const int nseg = SEG ? a.nseg : 1;
    const int seg = SEG ? static_cast<int>(blockIdx.x) % nseg : 0;
    const int cta_in_seg = SEG ? static_cast<int>(blockIdx.x) / nseg : static_cast<int>(blockIdx.x);
    const int ctas_in_seg = SEG ? (static_cast<int>(gridDim.x) - seg + nseg - 1) / nseg : static_cast<int>(gridDim.x);
    const int blk0 = SEG ? seg * a.seg_len : 0;
    const int seg_nblk = SEG ? (a.nblk - blk0 < a.seg_len ? a.nblk - blk0 : a.seg_len) : a.nblk;
    const int load_nblk = SEG ? seg_nblk + (blk0 + seg_nblk < a.nblk ? 1 : 0) : a.nblk;
    const size_t tile_bytes = static_cast<size_t>(a.nblk) * 128u;                 // one tile of 8 reads in global memory (rows.cuh)
    const uint32_t bar0 = smem_u32(smem);          // full barrier of slot (g,s) at bar0 + 8*(g*S+s)
    const uint32_t cnt0 = bar0 + 1024;             // release counter of slot (g,s) at cnt0 + 4*(g*S+s)
    const uint32_t data0 = bar0 + (HI ? kPileupSmemHeaderHi : kPileupSmemHeader);  // slot (g,s) at data0 + (g*S+s)*chunk_bytes
    const uint32_t chunk_bytes = static_cast<uint32_t>(load_nblk) * 128u;         // a slot = this segment's blocks of one tile
    const int64_t Tr = static_cast<int64_t>(G) * 8;  // reads per tile (one 8-read chunk per row-group)
    const int64_t ntiles = (a.R + Tr - 1) / Tr;

    if (threadIdx.x == 0) {
        for (int s = 0; s < S * G; ++s) {
            mbar_init(bar0 + 8 * s, 1);
            sts32(cnt0 + 4 * s, 0u);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    // ---------------- consumers: group g of W warps walks its 8 reads of every tile
    // Lane mapping: warp w of a row-group starts at block 31*w, so lane 31 of every warp but the last
    // re-reads the first block of the next warp and serves only as the look-ahead provider of lane 30
    // (its counters are ignored).  The last warp of the row uses all 32 lanes.
    const int group = warp / W;
    const int wig = warp - group * W;                // warp in group
    const int tig = wig * 32 + lane;                 // thread in group
    int lblk = wig * 31 + lane;                      // block within the segment (seg_nblk = the next segment's first: look-ahead only)
    const bool active = lblk < seg_nblk && (lane < 31 || wig == W - 1);
    if (lblk >= load_nblk) lblk = 0;
    const int blk = blk0 + lblk;                     // block within the reference
    // offsets of this thread's block and of the next one inside a slot, with the tile swizzle folded in (rows.cuh)
    const uint32_t blk_off = static_cast<uint32_t>(lblk) * 128u + (static_cast<uint32_t>(blk & 7) << 4);
    const uint32_t nblk_off = static_cast<uint32_t>(lblk + 1 < load_nblk ? lblk + 1 : lblk) * 128u + (static_cast<uint32_t>((blk + 1) & 7) << 4);

    CodonCtx cx;
    cx.codon = a.codon + static_cast<size_t>(blk) * 32 * 64;
    cx.r0 = cx.r1 = cx.r0n = cx.r1n = 0;
    cx.d0 = cx.d1 = cx.d0n = cx.d1n = 0;
    cx.start = cx.cols = cx.lookcols = 0;
    if (T::CODON) {
        const uint2 p = a.pivot[blk], pn = a.pivot[blk + 1];
        cx.r0 = p.x; cx.r1 = p.y; cx.r0n = pn.x; cx.r1n = pn.y;
        if (DENSE) {
            const uint2 d = a.pivot2[blk], dn = a.pivot2[blk + 1];
            cx.d0 = d.x; cx.d1 = d.y; cx.d0n = dn.x; cx.d1n = dn.y;
        }
        cx.start = active ? a.start_mask[blk] : 0u;
        cx.cols = cx.start | (cx.start << 1) | (cx.start << 2);
        cx.lookcols = ((cx.start >> 30) ? 1u : 0u) | ((cx.start >> 31) ? 2u : 0u);
    }

    const size_t list_id = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    ExcLog lg;
    lg.cap = a.exc_cap;
    lg.cnt = 0;
    lg.list = a.exc_list + list_id * a.exc_cap;   // (exc_cap = 0: no logging, everything in-kernel)

    // shared-memory planes kPlanes, kPlanes+1 of this thread's counters (in the header area)
    HiPlanes hp;
    hp.stride = HI ? static_cast<uint32_t>(blockDim.x) * 4u : 0u;
    hp.base = HI ? bar0 + kPileupHiOffset + static_cast<uint32_t>(threadIdx.x) * 4u : 0u;
    constexpr uint32_t kFlushAt = HI ? kMaxReadsPerFlushHi : kMaxReadsPerFlush;
    constexpr int NP = HI ? kPlanesAll : kPlanes;     // counter planes per mask

    Vert<NM> v;
    clear<HI>(v, hp);
    uint32_t bi = 0, n = 0, tiles_since_flush = 0;
    bool mid = false;
    uint32_t* pc = a.part_col + (static_cast<size_t>(blockIdx.x) * a.nblk + blk) * 256;
    uint32_t* pp = a.part_piv + (static_cast<size_t>(blockIdx.x) * a.nblk + blk) * 32;
    uint32_t* pd = DENSE ? a.part_piv2 + (static_cast<size_t>(blockIdx.x) * a.nblk + blk) * 32 : nullptr;
    const int nct = ncw * 32;

    // Chunk rings without a producer warp.  Every row-group owns S slots of 8 reads; the warp of the
    // group that arrives LAST at a slot's release counter knows the slot is free and refills it at
    // once (one cp.async.bulk), so S-1 chunks per group stay in flight, nobody blocks on an "empty"
    // barrier, and a slow group never holds back the others.
    auto issue_chunk = [&](int64_t k) {  // k = index among this CTA's tiles
        const int64_t t = static_cast<int64_t>(cta_in_seg) + k * ctas_in_seg;
        if (t >= ntiles) return;
        const int64_t r0 = t * Tr + group * 8;
        if (r0 >= a.R) return;
        const uint32_t slot = static_cast<uint32_t>(group * S + static_cast<int>(k % S));
        const uint32_t full = bar0 + 8 * slot;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy reads of the slot before the async write
        mbar_expect_tx(full, chunk_bytes);
        // the blocks [blk0, blk0 + load_nblk) of a tile are contiguous: one copy per chunk, whole rows or a segment
        // (a buffer holds whole tiles, so the last, partial tile is copied in full as well)
        const uint8_t* src = reinterpret_cast<const uint8_t*>(a.packed) + static_cast<size_t>(r0 >> 3) * tile_bytes + static_cast<size_t>(blk0) * 128u;
        bulk_g2s(data0 + slot * chunk_bytes, src, chunk_bytes, full);
    };
    if (tig == 0)
        for (int k = 0; k < S; ++k) issue_chunk(k);

    uint32_t stage = 0, phase = 0;
    int64_t kt = 0;
    for (int64_t t = cta_in_seg; t < ntiles; t += ctas_in_seg, ++kt) {
        if (8u * (tiles_since_flush + 1u) > kFlushAt) {
            // counters would overflow: every group adds its integers into the slice, one group at a time
            fold_pendings<HI>(v, hp, bi);
            uint32_t planes[NM * NP];
            gather_planes<HI>(v, hp, planes);
            for (int g = 0; g < G; ++g) {
                if (g == group && active) emit_slice<MODE, DENSE, NP>(planes, 0u, 0, 0u, 0u, n, cx.start, pc, pp, pd, mid || g > 0);
                consumer_barrier(nct);
            }
            clear<HI>(v, hp);
            bi = 0; n = 0; tiles_since_flush = 0; mid = true;
        }
        const int64_t r0 = t * Tr + group * 8;
        const int64_t left = a.R - r0;
        const int nv = left <= 0 ? 0 : (left > 8 ? 8 : static_cast<int>(left));
        const uint32_t slot = static_cast<uint32_t>(group * S) + stage;
        if (nv > 0) mbar_wait(bar0 + 8 * slot, phase);
        const uint32_t addr = data0 + slot * chunk_bytes + blk_off;   // read i of the tile at addr ^ 16 i
        const uint32_t naddr = data0 + slot * chunk_bytes + nblk_off; // same for the next block (rare path only)
        if (nv == 8) {
            const uint32_t pm = block8<MODE, DENSE, HI>(addr, cx, v, hp, bi);
            if (T::CODON && pm) log_or_handle<DENSE>(pm, lg, addr, naddr, cx);
            ++bi;
            n += 8;
        } else {
            for (int i = 0; i < nv; ++i) {
                uint32_t m[NM];
                uint32_t pm = 0;
                read_masks<MODE, DENSE>(addr ^ (static_cast<uint32_t>(i) << 4), cx, m, pm, 1u);
#pragma unroll
                for (int q = 0; q < NM; ++q) ripple<HI>(v, hp, q, 0, m[q]);
                if (T::CODON && pm) log_or_handle<DENSE>(1u << i, lg, addr, naddr, cx);
                ++n;
            }
        }
        ++tiles_since_flush;
        __syncwarp();
        if (lane == 0 && nv > 0) {
            __threadfence_block();
            const uint32_t cnt_addr = cnt0 + 4 * slot;
            uint32_t old;
            asm volatile("atom.shared.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(cnt_addr) : "memory");
            if (old == static_cast<uint32_t>(W - 1)) {  // last warp of the group out refills the slot
                __threadfence_block();
                sts32(cnt_addr, 0u);
                issue_chunk(kt + S);
            }
        }
        if (++stage == static_cast<uint32_t>(S)) { stage = 0; phase ^= 1u; }
    }

    if (T::CODON) a.exc_cnt[list_id] = lg.cnt;

    // ---------------- final merge: groups 1..G-1 hand their planes to group 0 through shared memory
    fold_pendings<HI>(v, hp, bi);
    // all tiles are consumed and every bulk copy has landed, so the stage ring is free to reuse
    consumer_barrier(nct);
    const uint32_t tg = static_cast<uint32_t>(W) * 32u;           // threads per group
    const uint32_t thread_stride = tg * 4u;                       // bytes between planes
    const uint32_t group_stride = static_cast<uint32_t>(NM * NP) * thread_stride;
    const uint32_t ncount0 = data0 + static_cast<uint32_t>(G - 1) * group_stride;  // n of groups 1..G-1
    if (group > 0) {
        const uint32_t base = data0 + static_cast<uint32_t>(group - 1) * group_stride + static_cast<uint32_t>(tig) * 4u;
#pragma unroll
        for (int i = 0; i < NM; ++i) {
#pragma unroll
            for (int k = 0; k < kPlanes; ++k) sts32(base + static_cast<uint32_t>(i * NP + k) * thread_stride, v.c[i][k]);
            if (HI) {
                sts32(base + static_cast<uint32_t>(i * NP + kPlanes) * thread_stride, lds32(hp.base + static_cast<uint32_t>(i) * hp.stride));
                sts32(base + static_cast<uint32_t>(i * NP + kPlanes + 1) * thread_stride, lds32(hp.base + static_cast<uint32_t>(NM + i) * hp.stride));
            }
        }
        if (tig == 0) sts32(ncount0 + static_cast<uint32_t>(group - 1) * 4u, n);
    }
    consumer_barrier(nct);
    if (group == 0 && active) {
        uint32_t ntot = n;
        for (int g = 1; g < G; ++g) ntot += lds32(ncount0 + static_cast<uint32_t>(g - 1) * 4u);
        uint32_t planes[NM * NP];
        gather_planes<HI>(v, hp, planes);
        emit_slice<MODE, DENSE, NP>(planes, data0 + static_cast<uint32_t>(tig) * 4u, G - 1, group_stride, thread_stride, ntot, cx.start,
                                    pc, pp, pd, mid);
    }
}

template <int MODE, bool DENSE, bool SEG, bool HI>
__global__ void __launch_bounds__(kPileupMaxThreads, 1) pileup_csa_kernel(PileupArgs a) {
    pileup_body<MODE, DENSE, SEG, HI>(a);
}

// launch = false: opt the instantiation in to the large dynamic shared memory on the current device (ms_create)
template <int MODE, bool DENSE>
static void launch_or_attr(bool launch, bool seg, bool hi, int grid, int threads, int smem, cudaStream_t s, const PileupArgs& a) {
#define MS_K1(SEG, HI)                                                                                                          \
    do {                                                                                                                        \
        if (launch) pileup_csa_kernel<MODE, DENSE, SEG, HI><<<grid, threads, smem, s>>>(a);                                     \
        else cudaFuncSetAttribute(pileup_csa_kernel<MODE, DENSE, SEG, HI>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);  \
    } while (0)
    if (!launch || (!seg && !hi)) MS_K1(false, false);
    if (!launch || (seg && !hi)) MS_K1(true, false);
    if (!launch || (!seg && hi)) MS_K1(false, true);
    if (!launch || (seg && hi)) MS_K1(true, true);
#undef MS_K1
}

static void dispatch(bool launch, int mode, bool dense, bool seg, bool hi, int grid, int threads, int smem, cudaStream_t s, const PileupArgs& a) {
    if (!launch || mode == kModeFuse) launch_or_attr<kModeFuse, false>(launch, seg, hi, grid, threads, smem, s, a);
    if (!launch || (mode == kModeJuliet && !dense)) launch_or_attr<kModeJuliet, false>(launch, seg, hi, grid, threads, smem, s, a);
    if (!launch || (mode == kModeJuliet && dense)) launch_or_attr<kModeJuliet, true>(launch, seg, hi, grid, threads, smem, s, a);
    if (!launch || (mode == kModeBoth && !dense)) launch_or_attr<kModeBoth, false>(launch, seg, hi, grid, threads, smem, s, a);
    if (!launch || (mode == kModeBoth && dense)) launch_or_attr<kModeBoth, true>(launch, seg, hi, grid, threads, smem, s, a);
}

void pileup_set_smem_attr(int max_smem) { dispatch(false, 0, false, false, false, 0, 0, max_smem, nullptr, PileupArgs()); }

// hi: the instantiation with the two shared-memory counter planes (row-groups of more than kMaxReadsPerFlush reads)
void pileup_launch(int mode, bool dense, bool hi, int grid, int threads, int smem, cudaStream_t s, const PileupArgs& a) {
    dispatch(true, mode, dense, a.nseg > 1, hi, grid, threads, smem, s, a);
}

// ---------------------------------------------------------------- logged exceptions
// One warp per logged list: every entry is the block of a read that may hold clean non-pivot codons (planes + the two
// look-ahead columns, see ExcLog).  The exact masks are recomputed from the entry and each such codon goes to the 64-bin
// histogram with a RED.  ~1.6 % of the (read, block) pairs at CCS error rates.
template <bool DENSE>
__global__ void __launch_bounds__(256) codon_exception_kernel(PileupArgs a, int threads_per_cta) {
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int64_t nlists = static_cast<int64_t>(a.exc_lists);
    if (warp >= nlists) return;
    uint32_t cnt = a.exc_cnt[warp];
    if (cnt > a.exc_cap) cnt = a.exc_cap;
    if (cnt == 0) return;
    const int tid = static_cast<int>(warp % threads_per_cta);
    const int w = tid >> 5, l = tid & 31;
    const int wig = w % a.warps_per_group;
    const int cta = static_cast<int>(warp / threads_per_cta);
    const int blk0 = (cta % a.nseg) * a.seg_len;
    const int seg_nblk = a.nblk - blk0 < a.seg_len ? a.nblk - blk0 : a.seg_len;
    if (wig * 31 + l >= seg_nblk) return;
    const int blk = blk0 + wig * 31 + l;
    CodonCtx cx;
    const uint2 p = a.pivot[blk], pn = a.pivot[blk + 1];
    cx.r0 = p.x; cx.r1 = p.y; cx.r0n = pn.x; cx.r1n = pn.y;
    cx.d0 = cx.d1 = cx.d0n = cx.d1n = 0;
    if (DENSE) {
        const uint2 d = a.pivot2[blk], dn = a.pivot2[blk + 1];
        cx.d0 = d.x; cx.d1 = d.y; cx.d0n = dn.x; cx.d1n = dn.y;
    }
    cx.start = a.start_mask[blk];
    cx.cols = cx.lookcols = 0;
    cx.codon = a.codon + static_cast<size_t>(blk) * 32 * 64;
    const uint4* list = a.exc_list + static_cast<size_t>(warp) * a.exc_cap;
    // lanes take consecutive entries.  Minor variants make many reads hit the SAME bin, so equal addresses within the warp
    // are merged (__match_any_sync) and only one lane issues the RED with the group's size.
    for (uint32_t i0 = 0; i0 < cnt; i0 += 32) {
        const uint32_t i = i0 + lane;
        uint32_t e = 0;
        uint4 q = make_uint4(0, 0, 0, 0), n = q;
        if (i < cnt) {
            const uint4 ent = list[i];
            q = make_uint4(ent.x, ent.y, ent.z, 0u);
            n = make_uint4(ent.w & 3u, (ent.w >> 2) & 3u, (ent.w >> 4) & 3u, 0u);     // columns 32, 33: only bits 0, 1 are ever shifted in
            uint32_t np;
            codon_masks<DENSE>(q, n, cx, np, e);
        }
        while (__any_sync(0xffffffffu, e != 0)) {
            uint32_t key = 0xffffffffu;
            if (e) {
                const int j = __ffs(e) - 1;
                e &= e - 1;
                const uint32_t b0 = __funnelshift_r(q.x, n.x, j) & 7u;
                const uint32_t b1 = __funnelshift_r(q.y, n.y, j) & 7u;
                const uint32_t cod = ((b0 & 1u) << 4) | ((b1 & 1u) << 5) | ((b0 & 2u) << 1) | ((b1 & 2u) << 2) |
                                     ((b0 & 4u) >> 2) | ((b1 & 4u) >> 1);
                key = static_cast<uint32_t>(j) * 64u + cod;
            }
            const uint32_t peers = __match_any_sync(0xffffffffu, key);
            if (key != 0xffffffffu && lane == __ffs(peers) - 1) atomicAdd(cx.codon + key, static_cast<uint32_t>(__popc(peers)));
        }
    }
}

void pileup_exceptions_launch(bool dense, int pileup_grid, int pileup_threads, cudaStream_t s, const PileupArgs& a) {
    const int64_t nlists = static_cast<int64_t>(pileup_grid) * pileup_threads;
    const unsigned grid = static_cast<unsigned>((nlists * 32 + 255) / 256);
    if (dense) codon_exception_kernel<true><<<grid, 256, 0, s>>>(a, pileup_threads);
    else codon_exception_kernel<false><<<grid, 256, 0, s>>>(a, pileup_threads);
}

// ---------------------------------------------------------------- pivot sampling
// One CTA per 32-column block; thread t looks at sample read t*R/blockDim.  Per column the
// majority of A/C/G/T among the sample becomes the pivot base.  The pivot only decides which
// codon is counted by the bit-sliced fast path; results are exact for any pivot.
__global__ void pivot_sample_kernel(const uint32_t* packed, int64_t R, int32_t nblk, int32_t L, uint2* pivot,
                                    uint8_t* pivot_state, uint2* pivot2, uint8_t* pivot2_state, uint32_t* dense_stat) {
    __shared__ uint32_t cnt[32][4];
    const int blk = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    if (tid < 128) cnt[tid >> 2][tid & 3] = 0;
    __syncthreads();
    const int64_t ns = R < blockDim.x ? R : blockDim.x;
    uint4 q = make_uint4(0, 0, 0xffffffffu, 0);  // state 4+: does not vote
    if (tid < ns) {
        const int64_t r = static_cast<int64_t>(tid) * R / ns;
        q = reinterpret_cast<const uint4*>(packed)[tile_slot(r, blk, nblk)];
    }
    for (int j = 0; j < 32; ++j) {
        const uint32_t st = ((q.x >> j) & 1u) | (((q.y >> j) & 1u) << 1) | (((q.z >> j) & 1u) << 2);
#pragma unroll
        for (uint32_t s = 0; s < 4; ++s) {
            const uint32_t b = __ballot_sync(0xffffffffu, st == s);
            if (lane == 0 && b) atomicAdd(&cnt[j][s], __popc(b));
        }
    }
    __syncthreads();
    if (tid < 32) {
        uint32_t best = 0;
#pragma unroll
        for (uint32_t s = 1; s < 4; ++s)
            if (cnt[tid][s] > cnt[tid][best]) best = s;
        const uint32_t r0 = __ballot_sync(0xffffffffu, best & 1u);
        const uint32_t r1 = __ballot_sync(0xffffffffu, best & 2u);
        if (tid == 0) pivot[blk] = make_uint2(r0, r1);
        if (blk * 32 + tid < L) pivot_state[blk * 32 + tid] = static_cast<uint8_t>(best);
        if (blk == 0 && tid == 0) { pivot[nblk] = make_uint2(0, 0); pivot2[nblk] = make_uint2(0, 0); }  // look-ahead of the last block
        uint32_t total = cnt[tid][0] + cnt[tid][1] + cnt[tid][2] + cnt[tid][3];
        // designated base of the DENSE kernel: the runner-up where it holds more than 2 % of the sampled clean bases
        // (a frequent variant), the pivot elsewhere
        uint32_t second = best;
        uint32_t second_cnt = 0;
#pragma unroll
        for (uint32_t s = 0; s < 4; ++s)
            if (s != best && cnt[tid][s] > second_cnt) { second = s; second_cnt = cnt[tid][s]; }
        if (second_cnt * 50u <= total) second = best;
        const uint32_t d0 = __ballot_sync(0xffffffffu, second & 1u);
        const uint32_t d1 = __ballot_sync(0xffffffffu, second & 2u);
        if (tid == 0) pivot2[blk] = make_uint2(d0, d1);
        if (blk * 32 + tid < L) pivot2_state[blk * 32 + tid] = static_cast<uint8_t>(second);
        // how often a sampled clean base is not the pivot: tells K1 whether non-pivot codons are rare (sequencing errors,
        // low-frequency variants) or the rule (dense high-frequency variants)
        uint32_t dev = total - cnt[tid][best];
        if (blk * 32 + tid >= L) total = dev = 0;
        total = __reduce_add_sync(0xffffffffu, total);
        dev = __reduce_add_sync(0xffffffffu, dev);
        if (tid == 0 && dense_stat) { atomicAdd(dense_stat, dev); atomicAdd(dense_stat + 1, total); }
    }
}

// ---------------------------------------------------------------- finalize
// counts += sum over the CTAs' slices; pivot-codon bin of every start column += its bit-sliced count.
// Four lanes share one output element and split the slices between them.
__global__ void pileup_finalize_kernel(const uint32_t* part_col, const uint32_t* part_piv, const uint32_t* part_piv2, int32_t slices,
                                       int32_t nblk, int32_t L, const uint8_t* pivot_state, const uint8_t* pivot2_state,
                                       const uint32_t* start_mask, uint32_t* col, uint32_t* codon,
                                       int32_t count_codons, int32_t nseg, int32_t seg_len) {
    const int64_t gt = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t i = gt >> 2;
    const int part = static_cast<int>(gt & 3);
    const int64_t ncol = static_cast<int64_t>(L) * 8;
    const size_t cstride = static_cast<size_t>(nblk) * 256, pstride = static_cast<size_t>(nblk) * 32;
    uint32_t s = 0, s2 = 0;
    bool is_col = i < ncol, is_piv = false;
    int64_t j = 0;
    // CTA k wrote the blocks of segment k % nseg only
    if (is_col) {
        const int sg = static_cast<int>((i >> 8) / seg_len);
        for (int k = sg + nseg * part; k < slices; k += 4 * nseg) s += part_col[k * cstride + i];
    } else if (count_codons && i < ncol + L) {
        j = i - ncol;
        is_piv = j + 2 < L && ((start_mask[j >> 5] >> (j & 31)) & 1u);
        const int sg = static_cast<int>((j >> 5) / seg_len);
        if (is_piv) {
            for (int k = sg + nseg * part; k < slices; k += 4 * nseg) s += part_piv[k * pstride + j];
            if (part_piv2)
                for (int k = sg + nseg * part; k < slices; k += 4 * nseg) s2 += part_piv2[k * pstride + j];
        }
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
    s2 += __shfl_xor_sync(0xffffffffu, s2, 2);
    if (part == 0) {
        if (is_col) col[i] += s;
        else if (is_piv) {
            const uint32_t cod = 16u * pivot_state[j] + 4u * pivot_state[j + 1] + pivot_state[j + 2];
            codon[j * 64 + cod] += s;
            if (part_piv2) {   // DENSE: the designated codon, where it is another codon than the pivot codon
                const uint32_t des = 16u * pivot2_state[j] + 4u * pivot2_state[j + 1] + pivot2_state[j + 2];
                if (des != cod) codon[j * 64 + des] += s2;
            }
        }
    }
}

// ---------------------------------------------------------------- A/B baseline
// The textbook histogram north_star describes: one thread per (read, 32-column block), shared-
// memory bins flushed once per CTA, codons straight to global atomics.  Kept only so ncu can
// show why K1 is not built this way (DESIGN.md); selected with ms_set_pileup_variant(h, 1).
__global__ void pileup_atomic_kernel(const uint32_t* packed, int64_t R, int32_t L, int32_t nblk,
                                     const uint32_t* start_mask, uint32_t* col, uint32_t* codon,
                                     int32_t count_codons) {
    extern __shared__ uint32_t bins[];  // [32 columns][8] of this CTA's column block
    const int blk = blockIdx.y;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) bins[i] = 0;
    __syncthreads();
    const uint32_t start = count_codons ? start_mask[blk] : 0u;
    for (int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; r < R;
         r += static_cast<int64_t>(gridDim.x) * blockDim.x) {
        const uint4 q = reinterpret_cast<const uint4*>(packed)[tile_slot(r, blk, nblk)];
        uint4 n = make_uint4(0, 0, 0xffffffffu, 0);
        if (blk + 1 < nblk) n = reinterpret_cast<const uint4*>(packed)[tile_slot(r, blk + 1, nblk)];
        for (int j = 0; j < 32; ++j) {
            const uint32_t st = ((q.x >> j) & 1u) | (((q.y >> j) & 1u) << 1) | (((q.z >> j) & 1u) << 2);
            if (st <= 5u) {
                atomicAdd(&bins[j * 8 + st], 1u);
                if ((q.w >> j) & 1u) atomicAdd(&bins[j * 8 + 6], 1u);
            }
            if ((start >> j) & 1u) {
                const uint32_t z = __funnelshift_r(q.z, n.z, j) & 7u;
                if (z == 0u) {
                    const uint32_t b0 = __funnelshift_r(q.x, n.x, j) & 7u, b1 = __funnelshift_r(q.y, n.y, j) & 7u;
                    const uint32_t cod = ((b0 & 1u) << 4) | ((b1 & 1u) << 5) | ((b0 & 2u) << 1) | ((b1 & 2u) << 2) |
                                         ((b0 & 4u) >> 2) | ((b1 & 4u) >> 1);
                    atomicAdd(codon + (static_cast<size_t>(blk * 32 + j) * 64 + cod), 1u);
                }
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        const int c = blk * 32 + (i >> 3);
        if (c < L && (i & 7) != 7 && bins[i]) atomicAdd(col + static_cast<size_t>(c) * 8 + (i & 7), bins[i]);
    }
}

// coverage column for the atomic variant (the CSA path writes it in its flush)
__global__ void coverage_kernel(uint32_t* col, int32_t L) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < L) {
        uint32_t* h = col + static_cast<size_t>(j) * 8;
        h[7] = h[0] + h[1] + h[2] + h[3] + h[4] + h[5];
    }
}

}  // namespace ms
