// phase.cu -- K3: read-level haplotype phasing.
//
// Replaces juliet --mode-phasing (/root/reference/doc/JULIET.md:192-211): for every
// read, which called variants it carries; reads with identical patterns form a
// haplotype; a read with a deletion (:278-288), a QV-filtered 'N' (:256-259) or
// missing coverage in any variant codon is unsuitable and only tallied in the three
// marginals of the tooltip (:372-381, screenshot juliet_haplotype-tooltip.png).
// SURVEY.md rows a11-a13.
//
// Kernels: phase_bits (one warp per read: stage the touched 32-column blocks in shared
// memory, one lane per variant, ballot -> bit-vector word), phase_insert (64-bit hash of
// the bit-vector into an open-addressing table with atomicCAS), phase_verify (exact compare
// against the slot's representative; a 64-bit collision triggers a re-hash with a new seed),
// compaction, and the popcount-AND co-occurrence over the transposed bit matrix.
#include <algorithm>
#include <cstring>
#include <numeric>
#include <vector>
#include "phase_internal.cuh"

namespace ms {

// The variant list as a word stream the kernel walks once per read (ms_phase_begin builds it; all lanes read the same
// word, so these are broadcast loads).  Per touched 32-column block, in block order, one or more LAYERS; a layer is a set of
// variants starting in that block whose codons agree on every column they share (different codons at the same site, or
// overlapping genes that disagree, go to further layers):
//   header, 5 words: [ slot in the block list (13 bits) | variants in this layer (11) << 13 | first layer of its block << 24 ],
//                    e0, e1  = bit-planes of the expected base per column (layer's codon columns; anything elsewhere),
//                    en      = the same for columns 32, 33 (a codon that starts at column 30 or 31): e0 in bits 0-1, e1 in bits 2-3,
//                    cover   = columns of this block that belong to ANY variant's codon (first layer only; damage flags)
//   then one word per variant: first column in the block (5 bits) | index in the caller's list << 5
//   -- or, when the layer's variants carry consecutive indices in column order (the usual sorted list; kHdrPacked), seven
//   words instead: the start-column mask, the five move masks of a parallel-suffix bit compress of that mask (Hacker's
//   Delight 7-4), and the first index.  The layer's bits then leave `hit` with 21 logic operations for all its variants
//   together instead of ~11 instructions per variant (phasing stress data: 11 variants per block).
constexpr uint32_t kHdrFirst = 1u << 24, kHdrPacked = 1u << 25;

constexpr int kPhaseWarps = 8;
constexpr int kPhaseChunkMax = 16;   // distinct blocks staged per pass (+1: the second block of a codon that straddles the chunk's end)

// Bit-vectors and damage flags, any number of variants, evaluated bit-sliced.  A lane owns a read, a warp four tiles
// (rows.cuh).  The touched blocks are staged `chunk` at a time into the warp's shared-memory slice -- per block one
// 16-byte load per lane, 128 contiguous bytes per tile, every byte of the line used, all loads of a chunk in flight
// together.  Per block and layer the lane then compares its 32 columns with the expected bases at once (2 LOP3 for the
// mismatch mask, 2 SHF + 1 LOP3 to spread it over the three columns of every possible codon start, exactly K1's pivot
// trick), and a variant costs one shift to pick its start column's bit and one to drop it into the lane's word of the
// bit-vector.  Damage (deletion / QV-filtered base / not spanned inside any variant codon) is three masked ORs per block.
// No ballots, no shuffles.  `ordered`: the stream visits the words of the bit-vector one after the other (the usual,
// sorted variant list), so a finished word is stored; otherwise it is ORed into the zeroed vector.  `partial_all`: some
// variant lies outside the reference, which makes every read partial.
// kClean (pairwise linkage, restatement choice U14): also the clean-codon matrix `mbits` (same row stride): bit v = the three
// columns of v's codon all hold A/C/G/T in this read.  It is `hit`'s construction on the state plane q.z instead of X, taken
// through the same compress / per-variant shift, so it costs a few logic operations per layer and one more store per word.
template <bool kClean>
__global__ void __launch_bounds__(kPhaseWarps * 32, 4) phase_bits_kernel(
    const uint4* __restrict__ packed, int64_t R, int32_t nblk, const int32_t* __restrict__ blocklist, int32_t NB, int32_t chunk, int32_t dbuf,
    const uint32_t* __restrict__ stream, int32_t nwords, int32_t vwords, int32_t ordered, int32_t partial_all,
    uint32_t* __restrict__ bits, uint8_t* __restrict__ flags, unsigned long long* __restrict__ ctr, const PhasePlan* __restrict__ plan,
    uint32_t* __restrict__ mbits) {
    extern __shared__ __align__(16) uint4 stage_sm[];   // [warp][chunk + 1][32]
    if (plan) {     // the sizes come from the device-built plan (one-word bit-vectors); a plan that gave up leaves everything to the host
        if (plan->fallback) return;
        NB = plan->NB; nwords = plan->nwords; partial_all = plan->partial_all; ordered = 1;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint4* sm = stage_sm + static_cast<size_t>(warp) * (dbuf ? 2 : 1) * (chunk + 1) * 32 + lane;
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kPhaseWarps;
    unsigned long long c_dam = 0, c_gap = 0, c_het = 0, c_par = 0;
    for (int64_t base = (static_cast<int64_t>(blockIdx.x) * kPhaseWarps + warp) * 32; base < R; base += nwarps * 32) {
        const int64_t r = base + lane;
        const bool live = r < R;
        const uint4* tile = packed + static_cast<size_t>(r >> 3) * nblk * 8;
        const uint32_t pos = static_cast<uint32_t>(r & 7);
        uint32_t fg = 0, fh = 0, fp = partial_all ? 1u : 0u;
        uint32_t word = 0, widx = 0xffffffffu;
        uint32_t mword = 0;      // kClean: the clean-codon bits of word widx
        uint32_t* myrow = bits + static_cast<size_t>(r) * vwords;
        uint32_t* mrow = kClean ? mbits + static_cast<size_t>(r) * vwords : nullptr;
        // store the finished word widx of both matrices
        auto flush = [&]() {
            if (ordered) myrow[widx] = word;
            else if (word) myrow[widx] |= word;
            if constexpr (kClean) {
                if (ordered) mrow[widx] = mword;
                else if (mword) mrow[widx] |= mword;
            }
        };
        int32_t p = 0;     // position in the stream
        // per-lane 16-byte asynchronous copies global -> shared (LDGSTS): every block of a chunk is in flight at once, no
        // registers in between.  A list of more than one chunk (dbuf) alternates between two buffers: chunk c + 1 is on its way
        // while chunk c is evaluated.
        auto stage_chunk = [&](int32_t c0s, uint4* buf) {
            const int32_t nbs = min(chunk + 1, NB - c0s);
#pragma unroll 4
            for (int32_t s2 = 0; s2 < nbs; ++s2) {
                const int32_t blk = blocklist[c0s + s2];
                const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(buf + s2 * 32));
                const uint4* src = tile + (blk * 8 + (pos ^ (blk & 7)));
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(live ? src : packed), "r"(live ? 16 : 0) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        };
        uint4* const sm0 = sm;
        uint4* const sm1 = sm + (dbuf ? (chunk + 1) * 32 : 0);
        stage_chunk(0, sm0);
        int32_t ci = 0;
        for (int32_t c0 = 0; c0 < NB; c0 += chunk, ++ci) {
            const int32_t nb = min(chunk + 1, NB - c0);
            uint4* const sm = (ci & 1) ? sm1 : sm0;
            if (c0 + chunk < NB) {
                if (dbuf) {
                    stage_chunk(c0 + chunk, (ci & 1) ? sm0 : sm1);
                    asm volatile("cp.async.wait_group 1;" ::: "memory");     // everything but the chunk just issued has landed
                } else {
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                }
            } else {
                asm volatile("cp.async.wait_group 0;" ::: "memory");
            }
            __syncwarp();
            while (p < nwords) {
                const uint32_t h0 = stream[p];
                const int32_t sa = static_cast<int32_t>(h0 & 0x1FFFu) - c0;
                if (sa >= chunk) break;                               // the next chunk's block
                const uint32_t e0 = stream[p + 1], e1 = stream[p + 2], en = stream[p + 3], cover = stream[p + 4];
                const int32_t nv = static_cast<int32_t>((h0 >> 13) & 0x7FFu);
                p += 5;
                const uint4 q = sm[sa * 32];
                const uint4 nx = sa + 1 < nb ? sm[(sa + 1) * 32] : make_uint4(0, 0, ~0u, 0);
                if (h0 & kHdrFirst) {
                    fg |= q.z & ~q.x & ~q.y & cover;      // 100  deletion
                    fh |= q.z & q.x & ~q.y & cover;       // 101  QV-filtered base
                    fp |= q.z & q.y & cover;              // 11x  not spanned
                }
                const uint32_t X = ((q.x ^ e0) | (q.y ^ e1)) | q.z;                       // column is not the clean expected base
                const uint32_t Xn = ((nx.x ^ en) | (nx.y ^ (en >> 2))) | nx.z;            // columns 32, 33 (bits 0, 1)
                const uint32_t hit = ~(X | __funnelshift_r(X, Xn, 1) | __funnelshift_r(X, Xn, 2));   // bit c: the codon starting at c matches
                uint32_t clean = 0;                                                       // bit c: the codon starting at c is all A/C/G/T
                if constexpr (kClean) clean = ~(q.z | __funnelshift_r(q.z, nx.z, 1) | __funnelshift_r(q.z, nx.z, 2));
                if (h0 & kHdrPacked) {
                    // compress the bits of `hit` at the start columns into the low nv bits (indices v0 .. v0 + nv - 1)
                    uint32_t x = hit & stream[p];
                    uint32_t xm = clean & stream[p];
#pragma unroll
                    for (int i = 0; i < 5; ++i) {
                        const uint32_t t = x & stream[p + 1 + i];
                        x = (x ^ t) | (t >> (1 << i));
                        if constexpr (kClean) {
                            const uint32_t tm = xm & stream[p + 1 + i];
                            xm = (xm ^ tm) | (tm >> (1 << i));
                        }
                    }
                    const uint32_t v0 = stream[p + 6];
                    p += 7;
                    const uint32_t sh = v0 & 31u;
                    if ((v0 >> 5) != widx) {
                        if (live && widx != 0xffffffffu) flush();
                        widx = v0 >> 5; word = 0;
                        if constexpr (kClean) mword = 0;
                    }
                    word |= x << sh;
                    if constexpr (kClean) mword |= xm << sh;
                    if (sh + static_cast<uint32_t>(nv) > 32u) {                             // the layer runs over into the next word
                        if (live) flush();
                        ++widx;
                        word = x >> (32u - sh);
                        if constexpr (kClean) mword = xm >> (32u - sh);
                    }
                    continue;
                }
                for (int32_t k = 0; k < nv; ++k) {
                    const uint32_t w = stream[p + k];
                    const uint32_t bit = __funnelshift_r(hit, 0u, w) & 1u;                 // shift by the low 5 bits of w: the start column
                    const uint32_t v = w >> 5;
                    if ((v >> 5) != widx) {                                                // warp-uniform: all lanes are at the same variant
                        if (live && widx != 0xffffffffu) flush();
                        widx = v >> 5; word = 0;
                        if constexpr (kClean) mword = 0;
                    }
                    word |= __funnelshift_l(0u, bit, v);                                    // bit << (v & 31)
                    if constexpr (kClean) mword |= __funnelshift_l(0u, __funnelshift_r(clean, 0u, w) & 1u, v);
                }
                p += nv;
            }
            __syncwarp();
            if (!dbuf && c0 + chunk < NB) stage_chunk(c0 + chunk, sm0);       // one buffer: the next chunk goes up after this one is done
        }
        if (live) {
            if (ordered && vwords == 1) {
                myrow[0] = word;                 // the only word: written whether or not any variant maps to it (no zeroing by the caller)
                if constexpr (kClean) mrow[0] = mword;
            } else if (widx != 0xffffffffu) {
                flush();
            }
            const uint32_t f = (fg ? MS_FLAG_GAP : 0) | (fh ? MS_FLAG_HET : 0) | (fp ? MS_FLAG_PARTIAL : 0);
            flags[r] = static_cast<uint8_t>(f);
            if (f) {
                ++c_dam;
                if (f & MS_FLAG_GAP) ++c_gap;
                if (f & MS_FLAG_HET) ++c_het;
                if (f & MS_FLAG_PARTIAL) ++c_par;
            }
        }
    }
    // warp totals -> one atomic per counter per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c_dam += __shfl_xor_sync(0xffffffffu, c_dam, o);
        c_gap += __shfl_xor_sync(0xffffffffu, c_gap, o);
        c_het += __shfl_xor_sync(0xffffffffu, c_het, o);
        c_par += __shfl_xor_sync(0xffffffffu, c_par, o);
    }
    if (lane == 0 && c_dam) {
        atomicAdd(ctr + 0, c_dam);
        atomicAdd(ctr + 1, c_gap);
        atomicAdd(ctr + 2, c_het);
        atomicAdd(ctr + 3, c_par);
    }
}

// The phasing plan on the device (PhasePlan, phase_internal.cuh): one warp turns K2's calls into the pooled, sorted,
// de-duplicated (column, codon) list juliet phases over (screenshot juliet_hiv-phasing.png: one variant list for all genes), the
// list of touched 32-column blocks and the block / layer / variant word stream phase_bits_kernel walks -- the same stream
// ms_phase_begin builds on the host.  Lanes own calls, then keys, then block slots; sorting is by rank counting (a few dozen
// items).  A few microseconds, and the pass keeps the GPU busy instead of waiting for a device -> host -> device round trip.
constexpr int kPlanSlotWords = kPlanMaxLayers * 5 + kPlanMaxKeys;

// first[i] = no earlier entry holds the same value; returns this lane's ranks among the distinct values (entries lane, lane + 32)
__device__ __forceinline__ void rank_distinct(const int32_t* vals, int n, int lane, int32_t* first, int (&rank)[2]) {
    for (int e = 0; e < 2; ++e) {
        const int i = lane + 32 * e;
        int f = 0;
        if (i < n && vals[i] != 0x7fffffff) {
            f = 1;
            for (int j = 0; j < i; ++j) f &= vals[j] != vals[i];
        }
        first[i] = f;
    }
    __syncwarp();
    for (int e = 0; e < 2; ++e) {
        const int i = lane + 32 * e;
        int r = 0;
        if (i < n)
            for (int j = 0; j < n; ++j) r += (first[j] && vals[j] < vals[i]) ? 1 : 0;
        rank[e] = r;
    }
}

__global__ void __launch_bounds__(32) phase_plan_kernel(const ms_variant* __restrict__ calls, const unsigned long long* __restrict__ ncalls_ptr,
                                                        int64_t calls_cap, int32_t L, PhasePlan* __restrict__ plan, int32_t* __restrict__ blocklist,
                                                        uint32_t* __restrict__ stream) {
    __shared__ int32_t s_key[kPlanMaxCalls], s_first[kPlanMaxCalls];
    __shared__ int32_t s_kc[kPlanMaxKeys], s_kk[kPlanMaxKeys];
    __shared__ int32_t s_cand[2 * kPlanMaxKeys], s_blk[kPlanMaxBlocks], s_nw[kPlanMaxBlocks];
    __shared__ uint32_t s_words[kPlanMaxBlocks][kPlanSlotWords];
    __shared__ int s_fail;
    const int lane = threadIdx.x;
    const unsigned long long n64 = *ncalls_ptr;
    if (lane == 0) {
        plan->ncalls = static_cast<int32_t>(n64 > 0x7fffffffULL ? 0x7fffffff : n64);
        plan->fallback = 1;
        plan->V = plan->NB = plan->nwords = plan->partial_all = 0;
        s_fail = 0;
    }
    if (n64 > static_cast<unsigned long long>(kPlanMaxCalls) || static_cast<int64_t>(n64) > calls_cap) return;
    const int n = static_cast<int>(n64);
    // pooled keys: distinct (column, codon), ascending
    for (int i = lane; i < kPlanMaxCalls; i += 32) s_key[i] = i < n ? ((calls[i].col << 6) | calls[i].codon) : 0x7fffffff;
    __syncwarp();
    int rank[2];
    rank_distinct(s_key, n, lane, s_first, rank);
    const int V = __popc(__ballot_sync(0xffffffffu, s_first[lane])) + __popc(__ballot_sync(0xffffffffu, s_first[lane + 32]));
    if (V > kPlanMaxKeys) return;
    for (int e = 0; e < 2; ++e) {
        const int i = lane + 32 * e;
        if (s_first[i]) { s_kc[rank[e]] = s_key[i] >> 6; s_kk[rank[e]] = s_key[i] & 63; }
    }
    __syncwarp();
    // touched blocks: distinct (col >> 5) and ((col + 2) >> 5) of the keys inside the reference, ascending
    const bool inside = lane < V && s_kc[lane] + 2 < L;
    const int partial = __any_sync(0xffffffffu, lane < V && !inside) ? 1 : 0;     // a variant outside the reference: no read spans it
    s_cand[2 * lane] = inside ? (s_kc[lane] >> 5) : 0x7fffffff;
    s_cand[2 * lane + 1] = inside ? ((s_kc[lane] + 2) >> 5) : 0x7fffffff;
    __syncwarp();
    rank_distinct(s_cand, 2 * kPlanMaxKeys, lane, s_first, rank);
    int NB = __popc(__ballot_sync(0xffffffffu, s_first[lane])) + __popc(__ballot_sync(0xffffffffu, s_first[lane + 32]));
    for (int e = 0; e < 2; ++e) {
        const int i = lane + 32 * e;
        if (s_first[i]) s_blk[rank[e]] = s_cand[i];
    }
    if (NB == 0) { if (lane == 0) s_blk[0] = 0; NB = 1; }
    __syncwarp();
    // per block slot: cover mask, greedy layers, the slot's words
    for (int e = 0; e < 2; ++e) {
        const int sl = lane + 32 * e;
        int nwords = 0;
        if (sl < NB) {
            const int32_t blk = s_blk[sl];
            uint32_t cover = 0;
            int8_t base[kPlanMaxLayers][34];
            uint8_t lv[kPlanMaxLayers][kPlanMaxKeys];
            int ln[kPlanMaxLayers];
            int nl = 0;
            bool fail = false;
            for (int v = 0; v < V; ++v) {
                const int32_t col = s_kc[v];
                if (col + 2 >= L) continue;
                for (int c = col; c < col + 3; ++c)
                    if ((c >> 5) == blk) cover |= 1u << (c & 31);
                if ((col >> 5) != blk) continue;
                const int c = col & 31;
                const int32_t kk = s_kk[v];
                const int8_t cod[3] = {static_cast<int8_t>((kk >> 4) & 3), static_cast<int8_t>((kk >> 2) & 3), static_cast<int8_t>(kk & 3)};
                int li = 0;
                for (; li < nl; ++li) {
                    bool ok = true;
                    for (int k = 0; k < 3; ++k) ok = ok && (base[li][c + k] < 0 || base[li][c + k] == cod[k]);
                    if (ok) break;
                }
                if (li == nl) {
                    if (nl == kPlanMaxLayers) { fail = true; break; }
                    for (int k = 0; k < 34; ++k) base[nl][k] = -1;
                    ln[nl] = 0; ++nl;
                }
                for (int k = 0; k < 3; ++k) base[li][c + k] = cod[k];
                lv[li][ln[li]++] = static_cast<uint8_t>(v);
            }
            if (fail) s_fail = 1;
            if (nl == 0) {                                        // spill-over block: damage flags only
                for (int k = 0; k < 34; ++k) base[0][k] = -1;
                ln[0] = 0; nl = 1;
            }
            if (!fail) {
                for (int li = 0; li < nl; ++li) {
                    uint32_t e0 = 0, e1 = 0, en = 0;
                    for (int c = 0; c < 32; ++c)
                        if (base[li][c] > 0) { e0 |= static_cast<uint32_t>(base[li][c] & 1) << c; e1 |= static_cast<uint32_t>((base[li][c] >> 1) & 1) << c; }
                    for (int c = 32; c < 34; ++c)
                        if (base[li][c] > 0) { en |= static_cast<uint32_t>(base[li][c] & 1) << (c - 32); en |= static_cast<uint32_t>((base[li][c] >> 1) & 1) << (c - 32 + 2); }
                    s_words[sl][nwords++] = static_cast<uint32_t>(sl) | (static_cast<uint32_t>(ln[li]) << 13) | (li == 0 ? kHdrFirst : 0u);
                    s_words[sl][nwords++] = e0; s_words[sl][nwords++] = e1; s_words[sl][nwords++] = en; s_words[sl][nwords++] = li == 0 ? cover : 0u;
                    for (int k = 0; k < ln[li]; ++k) s_words[sl][nwords++] = static_cast<uint32_t>(s_kc[lv[li][k]] & 31) | (static_cast<uint32_t>(lv[li][k]) << 5);
                }
            }
        }
        s_nw[sl] = nwords;
    }
    __syncwarp();
    if (s_fail) return;
    int total = 0;
    for (int e = 0; e < 2; ++e) {
        const int sl = lane + 32 * e;
        int off = 0;
        for (int t = 0; t < sl; ++t) off += s_nw[t];
        for (int k = 0; k < s_nw[sl]; ++k) stream[off + k] = s_words[sl][k];
        if (sl < NB) blocklist[sl] = s_blk[sl];
    }
    for (int t = 0; t < kPlanMaxBlocks; ++t) total += s_nw[t];
    if (lane < V) { plan->key_col[lane] = s_kc[lane]; plan->key_codon[lane] = s_kk[lane]; }
    __syncwarp();
    if (lane == 0) {
        plan->V = V; plan->NB = NB; plan->nwords = total; plan->partial_all = partial;
        __threadfence();
        plan->fallback = 0;
    }
}

// One launch instead of six memsets in front of every table build: empty keys, zero counts, "no representative yet", and the
// build's counters (ctr[4] collisions, ctr[6] overflow, ctr[7] "this build is the rank's last resort").
__global__ void __launch_bounds__(256) phase_clear_kernel(unsigned long long* __restrict__ tab_key, uint32_t* __restrict__ tab_cnt,
                                                          long long* __restrict__ tab_rep, int64_t tab_size, unsigned long long* __restrict__ ctr,
                                                          unsigned long long last_resort) {
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
    for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < tab_size; i += stride) {
        tab_key[i] = 0ULL;
        tab_cnt[i] = 0u;
        tab_rep[i] = 0x7f7f7f7f7f7f7f7fLL;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctr[4] = 0ULL; ctr[6] = 0ULL; ctr[7] = last_resort; }
}

// One thread per read; lanes of a warp that carry the same pattern elect a leader (lowest lane =
// lowest read index) which alone touches the table: one CAS probe, one count add, one rep min.
__global__ void phase_insert_kernel(const uint32_t* __restrict__ bits, const uint8_t* __restrict__ flags, int64_t R,
                                    int32_t vwords, uint64_t seed, unsigned long long* tab_key, uint32_t* tab_cnt,
                                    long long* tab_rep, int64_t mask, int32_t* __restrict__ slot, unsigned long long* overflow) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const bool valid = r < R && flags[r] == 0;
    if (r < R && !valid) slot[r] = -1;
    // the table already overflowed: this build is void (the host grows the table and rebuilds), so do not keep
    // probing it.  Decided per warp so that the match below still sees every lane of vmask.
    if (__any_sync(0xffffffffu, *reinterpret_cast<volatile unsigned long long*>(overflow) != 0ULL)) {
        if (r < R) slot[r] = -1;
        return;
    }
    const uint32_t vmask = __ballot_sync(0xffffffffu, valid);
    if (!valid) return;
    const uint64_t key = pattern_hash(bits + static_cast<size_t>(r) * vwords, vwords, seed);
    const uint32_t peers = __match_any_sync(vmask, static_cast<unsigned long long>(key));
    const int leader = __ffs(peers) - 1;
    int64_t idx = -1;
    if (lane == leader) {
        int64_t probe = static_cast<int64_t>(key) & mask;
        for (int step = 0; step < 256; ++step) {   // bounded: a (nearly) full table reports overflow instead of spinning
            const unsigned long long prev = atomicCAS(tab_key + probe, 0ULL, static_cast<unsigned long long>(key));
            if (prev == 0ULL || prev == key) { idx = probe; break; }
            probe = (probe + 1) & mask;
        }
        if (idx >= 0) {
            atomicAdd(tab_cnt + idx, static_cast<uint32_t>(__popc(peers)));
            atomicMin(tab_rep + idx, static_cast<long long>(r));
        } else {
            atomicAdd(overflow, 1ULL);
        }
    }
    idx = __shfl_sync(peers, idx, leader);
    slot[r] = static_cast<int32_t>(idx);
}

__global__ void phase_verify_kernel(const uint32_t* __restrict__ bits, int64_t R, int32_t vwords,
                                    const long long* __restrict__ tab_rep, const int32_t* __restrict__ slot,
                                    unsigned long long* collision) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= R || slot[r] < 0) return;
    const long long rep = tab_rep[slot[r]];
    if (rep == r) return;
    const uint32_t* a = bits + static_cast<size_t>(r) * vwords;
    const uint32_t* b = bits + static_cast<size_t>(rep) * vwords;
    for (int32_t i = 0; i < vwords; ++i)
        if (a[i] != b[i]) { atomicAdd(collision, 1ULL); return; }
}

// Distinct patterns out of the table: count + the representative's bit-vector, compacted.
__global__ void phase_compact_kernel(const uint32_t* __restrict__ tab_cnt, const long long* __restrict__ tab_rep,
                                     int64_t tab_size, const uint32_t* __restrict__ bits, int32_t vwords,
                                     unsigned long long* ngroups, uint32_t* __restrict__ g_cnt,
                                     uint32_t* __restrict__ g_pat, int32_t* __restrict__ g_slot, int64_t cap) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= tab_size || tab_cnt[i] == 0) return;
    const unsigned long long k = atomicAdd(ngroups, 1ULL);
    if (static_cast<int64_t>(k) < cap) {
        g_cnt[k] = tab_cnt[i];
        if (g_slot) g_slot[k] = static_cast<int32_t>(i);
        const uint32_t* src = bits + static_cast<size_t>(tab_rep[i]) * vwords;
        for (int32_t w = 0; w < vwords; ++w) g_pat[k * vwords + w] = src[w];
    }
}

// rank lookup for ms_phase_assign: ordered pattern -> its slot in this rank's table
__global__ void phase_rank_kernel(const uint32_t* __restrict__ ordered, int64_t H, int32_t vwords, uint64_t seed,
                                  const unsigned long long* __restrict__ tab_key, const long long* __restrict__ tab_rep,
                                  int64_t mask, const uint32_t* __restrict__ bits, int32_t* __restrict__ slot_rank) {
    const int64_t g = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (g >= H) return;
    const uint32_t* pat = ordered + static_cast<size_t>(g) * vwords;
    const uint64_t key = pattern_hash(pat, vwords, seed);
    int64_t idx = static_cast<int64_t>(key) & mask;
    for (;;) {
        const unsigned long long k = tab_key[idx];
        if (k == 0ULL) return;  // pattern not present on this rank
        if (k == key) {
            const uint32_t* b = bits + static_cast<size_t>(tab_rep[idx]) * vwords;
            bool same = true;
            for (int32_t i = 0; i < vwords; ++i) same = same && (b[i] == pat[i]);
            if (same) { slot_rank[idx] = static_cast<int32_t>(g); return; }
        }
        idx = (idx + 1) & mask;
    }
}

__global__ void phase_assign_kernel(const int32_t* __restrict__ slot, const int32_t* __restrict__ slot_rank, int64_t R,
                                    int32_t* __restrict__ hap) {
    const int64_t r = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (r >= R) return;
    hap[r] = slot[r] < 0 ? -1 : slot_rank[slot[r]];
}

// ---- co-occurrence: C = B^T B by popcount-AND over the transposed bit matrix ----
// transpose 32 reads x 32 variants per warp with ballots
__global__ void bits_transpose_kernel(const uint32_t* __restrict__ bits, int64_t R, int32_t vwords, int64_t rwords,
                                      uint32_t* __restrict__ bt) {
    const int64_t warp = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int64_t t = warp / vwords;   // read word
    const int32_t w = static_cast<int32_t>(warp - t * vwords);
    if (t >= rwords) return;
    const int64_t r = t * 32 + lane;
    const uint32_t x = r < R ? bits[static_cast<size_t>(r) * vwords + w] : 0u;
    uint32_t mine = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const uint32_t b = __ballot_sync(0xffffffffu, (x >> i) & 1u);
        if (lane == i) mine = b;
    }
    bt[static_cast<size_t>(w * 32 + lane) * rwords + t] = mine;
}

constexpr int kCoTile = 32, kCoChunk = 32;
__global__ void __launch_bounds__(256) cooccurrence_kernel(const uint32_t* __restrict__ bt, int32_t V, int64_t rwords,
                                                           int32_t* __restrict__ C) {
    __shared__ uint32_t A[kCoTile][kCoChunk + 1], B[kCoTile][kCoChunk + 1];
    const int tv = blockIdx.y * kCoTile, tw = blockIdx.x * kCoTile;
    if (tw < tv) return;  // symmetric: compute the upper triangle, mirror on write
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // ty 0..7
    int32_t acc[4] = {0, 0, 0, 0};
    for (int64_t t0 = 0; t0 < rwords; t0 += kCoChunk) {
        for (int i = ty; i < kCoTile; i += 8) {
            const int64_t t = t0 + tx;
            A[i][tx] = (tv + i < V && t < rwords) ? bt[static_cast<size_t>(tv + i) * rwords + t] : 0u;
            B[i][tx] = (tw + i < V && t < rwords) ? bt[static_cast<size_t>(tw + i) * rwords + t] : 0u;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < kCoChunk; ++k) {
            const uint32_t b = B[tx][k];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] += __popc(A[ty + 8 * q][k] & b);
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int v = tv + ty + 8 * q, w = tw + tx;
        if (v < V && w < V) {
            C[static_cast<size_t>(v) * V + w] = acc[q];
            C[static_cast<size_t>(w) * V + v] = acc[q];
        }
    }
}

}  // namespace ms

int ms_comm_allgather_bytes(ms_handle* h, const void* d_send, void* d_recv, size_t bytes_per_rank);
int ms_cooccurrence_tc_launch(ms_handle* h, const uint32_t* bt, int32_t V, int64_t rstride, int64_t R, int32_t* C);

namespace {

int phase_groups_copy_out(ms_handle* h, uint32_t* patterns, uint64_t* counts, int64_t cap, int64_t* H, ms_phase_counters* ctr);

constexpr int64_t kGroupCapInit = 4096;

}  // namespace

namespace ms {

int phase_ensure_stage(ms_handle* h, size_t bytes) {
    if (bytes <= h->h_stage_cap) return MS_OK;
    if (h->h_stage) cudaFreeHost(h->h_stage);
    h->h_stage = nullptr; h->h_stage_cap = 0;
    MS_CUDA(h, cudaMallocHost(&h->h_stage, bytes + bytes / 4 + 4096));
    h->h_stage_cap = bytes + bytes / 4 + 4096;
    return MS_OK;
}

int phase_build_table(ms_handle* h, int attempt) {
    const int64_t R = h->phase_n;
    h->hap_ranked = h->hap_assigned = false;   // new table slots: the order positions of ms_phase_haplotypes no longer apply
    unsigned long long* ctr = phase_ctr(h);
    // spare word of the exchanged header (ctr[7]): 1 = this build was this rank's last resort (table at its maximum size, or the
    // fourth hash seed), so that an overflow / a collision reported with it makes EVERY rank give up in the same iteration
    const unsigned long long last_resort = (h->tab_size >= h->tab_size_max || attempt >= 3) ? 1ULL : 0ULL;
    phase_clear_kernel<<<static_cast<int>(std::min<int64_t>((h->tab_size + 255) / 256, static_cast<int64_t>(h->num_sms) * 8)), 256, 0, h->stream>>>(
        h->b_tab_key.as<unsigned long long>(), h->b_tab_cnt.as<uint32_t>(), h->b_tab_rep.as<long long>(), h->tab_size, ctr, last_resort);
    h->launches++;
    if (R > 0) {
        const int grid = static_cast<int>((R + 255) / 256);
        phase_insert_kernel<<<grid, 256, 0, h->stream>>>(h->b_bits.as<uint32_t>(), h->b_flags.as<uint8_t>(), R, h->vwords,
                                                         phase_seed(attempt), h->b_tab_key.as<unsigned long long>(),
                                                         h->b_tab_cnt.as<uint32_t>(), h->b_tab_rep.as<long long>(),
                                                         h->tab_size - 1, h->b_slot.as<int32_t>(), ctr + 6);
        phase_verify_kernel<<<grid, 256, 0, h->stream>>>(h->b_bits.as<uint32_t>(), R, h->vwords, h->b_tab_rep.as<long long>(),
                                                         h->b_slot.as<int32_t>(), ctr + 4);
        h->launches += 2;
    }
    h->table_attempt = attempt;
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

int phase_compact(ms_handle* h, uint32_t* g_cnt, uint32_t* g_pat, int32_t* g_slot, int64_t cap) {
    MS_CUDA(h, cudaMemsetAsync(phase_ctr(h) + 5, 0, 8, h->stream));
    phase_compact_kernel<<<static_cast<int>((h->tab_size + 255) / 256), 256, 0, h->stream>>>(
        h->b_tab_cnt.as<uint32_t>(), h->b_tab_rep.as<long long>(), h->tab_size, h->b_bits.as<uint32_t>(), h->vwords, phase_ctr(h) + 5,
        g_cnt, g_pat, g_slot, cap);
    h->launches++;
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

int phase_grow_table(ms_handle* h) {
    if (h->tab_size >= h->tab_size_max) MS_FAIL(h, MS_ERR_CUDA, "haplotype table overflow at maximum size");
    h->tab_size = std::min<int64_t>(h->tab_size_max, h->tab_size * 8);
    h->tab_hint = h->tab_size;
    MS_CUDA(h, h->b_tab_key.ensure(static_cast<size_t>(h->tab_size) * 8));
    MS_CUDA(h, h->b_tab_cnt.ensure(static_cast<size_t>(h->tab_size) * 4));
    MS_CUDA(h, h->b_tab_rep.ensure(static_cast<size_t>(h->tab_size) * 8));
    h->table_valid = false;
    return MS_OK;
}

}  // namespace ms

namespace {

using ms::phase_seed;
inline unsigned long long* ctr_ptr(ms_handle* h) { return ms::phase_ctr(h); }
inline int ensure_stage(ms_handle* h, size_t bytes) { return ms::phase_ensure_stage(h, bytes); }
inline int build_table(ms_handle* h, int attempt) { return ms::phase_build_table(h, attempt); }

// hand the cached (pattern, count) lists of the last grouping pass to the caller (order: as compacted)
int phase_groups_copy_out(ms_handle* h, uint32_t* patterns, uint64_t* counts, int64_t cap, int64_t* H, ms_phase_counters* ctr) {
    const int32_t nw = h->vwords;
    const int64_t ng = static_cast<int64_t>(h->groups_cnt.size());
    const int64_t k = std::min<int64_t>(cap, ng);
    if (patterns && k > 0) memcpy(patterns, h->groups_pat.data(), static_cast<size_t>(k) * nw * 4);
    if (counts) for (int64_t i = 0; i < k; ++i) counts[i] = h->groups_cnt[i];
    *H = ng;
    if (ctr) {
        ctr->reported = 0; ctr->insufficient = 0;
        ctr->damaged = h->groups_marg[0]; ctr->gaps = h->groups_marg[1]; ctr->heteroduplex = h->groups_marg[2]; ctr->partial = h->groups_marg[3];
    }
    return MS_OK;
}

}  // namespace

// opt the bit-vector kernel in to its largest staging area (8 warps x 17 blocks x 512 B), on the current device (ms_create)
void ms_phase_set_smem_attr() {
    const int bytes = ms::kPhaseWarps * 2 * (ms::kPhaseChunkMax / 2 + 1) * 32 * static_cast<int>(sizeof(uint4)) >
                              ms::kPhaseWarps * (ms::kPhaseChunkMax + 1) * 32 * static_cast<int>(sizeof(uint4))
                          ? ms::kPhaseWarps * 2 * (ms::kPhaseChunkMax / 2 + 1) * 32 * static_cast<int>(sizeof(uint4))
                          : ms::kPhaseWarps * (ms::kPhaseChunkMax + 1) * 32 * static_cast<int>(sizeof(uint4));
    cudaFuncSetAttribute(ms::phase_bits_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    cudaFuncSetAttribute(ms::phase_bits_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}

extern "C" {

void ms_phase_free_internal(ms_handle* h) {
    DevBuf* all[] = {&h->b_plan, &h->b_var, &h->b_blocklist, &h->b_bits, &h->b_flags, &h->b_slot, &h->b_tab_key, &h->b_tab_cnt, &h->b_tab_rep,
                     &h->b_ctr, &h->b_groups, &h->b_gather, &h->b_rank, &h->b_hap, &h->b_pat, &h->b_cooc, &h->b_bits_t,
                     &h->b_gslot, &h->b_mt_key, &h->b_mt_cnt, &h->b_mt_rep, &h->b_mslot, &h->b_mindex, &h->b_m_cnt, &h->b_m_pat, &h->b_m_rank,
                     &h->b_ord, &h->b_keys, &h->b_out, &h->b_tc_tiles,
                     &h->b_nw_seq, &h->b_nw_hrow, &h->b_nw_hcol, &h->b_nw_dir,
                     &h->b_mbits, &h->b_link_gram, &h->b_link_col, &h->b_link_sig, &h->b_link_rows, &h->b_link_out};
    for (DevBuf* b : all) b->release();
    if (h->h_stage) cudaFreeHost(h->h_stage);
    h->h_stage = nullptr; h->h_stage_cap = 0;
    if (h->plan_stage) cudaFreeHost(h->plan_stage);
    h->plan_stage = nullptr;
    h->phase_cap = h->phase_n = 0; h->V = 0; h->vwords = 0; h->table_valid = false;
    h->link_ready = h->gram_valid = false;
    h->hap_ranked = h->hap_assigned = false;
}

int ms_phase_begin(ms_handle* h, const int32_t* var_col, const int32_t* var_codon, int32_t V, int64_t max_reads) {
    if (!h || h->L <= 0 || V < 0 || max_reads < 0 || (V > 0 && (!var_col || !var_codon))) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    h->V = V;
    h->vwords = std::max(1, (V + 31) / 32);
    h->phase_cap = std::max<int64_t>(1, max_reads);
    h->phase_n = 0;
    h->table_valid = false;
    h->groups_valid = false;
    h->gram_valid = false;
    h->link_ready = false;
    h->hap_ranked = h->hap_assigned = false;
    // distinct 32-column blocks the variants touch
    std::vector<int32_t> blocks;
    for (int32_t v = 0; v < V; ++v) {
        if (var_col[v] < 0 || var_codon[v] < 0 || var_codon[v] > 63) MS_FAIL(h, MS_ERR_ARG, "bad variant");
        if (var_col[v] + 2 < h->L) { blocks.push_back(var_col[v] >> 5); blocks.push_back((var_col[v] + 2) >> 5); }
    }
    std::sort(blocks.begin(), blocks.end());
    blocks.erase(std::unique(blocks.begin(), blocks.end()), blocks.end());
    if (blocks.empty()) blocks.push_back(0);
    h->nblocklist = static_cast<int32_t>(blocks.size());
    if (blocks.size() > 0x1FFF) MS_FAIL(h, MS_ERR_CAPACITY, "variants touch more than 8191 distinct 32-column blocks");
    // the word stream of phase_bits_kernel (layout documented there): per touched block its layers, per layer its variants
    const int32_t NBl = static_cast<int32_t>(blocks.size());
    std::vector<std::vector<int32_t>> by_block(static_cast<size_t>(NBl));      // variants starting in each listed block, by column
    std::vector<uint32_t> cover(static_cast<size_t>(NBl), 0u);
    h->phase_partial_all = false;
    {
        std::vector<int32_t> order;
        for (int32_t v = 0; v < V; ++v) {
            if (var_col[v] + 2 < h->L) order.push_back(v);
            else h->phase_partial_all = true;     // a variant outside the reference: no read spans it
        }
        std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return var_col[a] < var_col[b]; });
        for (int32_t v : order) {
            for (int32_t c = var_col[v]; c < var_col[v] + 3; ++c) {
                const int32_t sl = static_cast<int32_t>(std::lower_bound(blocks.begin(), blocks.end(), c >> 5) - blocks.begin());
                cover[sl] |= 1u << (c & 31);
            }
            by_block[std::lower_bound(blocks.begin(), blocks.end(), var_col[v] >> 5) - blocks.begin()].push_back(v);
        }
    }
    std::vector<uint32_t> vd;
    bool ordered = true;
    int64_t last_word = -1;
    std::vector<char> word_seen(static_cast<size_t>(h->vwords), 0);
    for (int32_t sl = 0; sl < NBl; ++sl) {
        // greedy layering: a variant joins the first layer whose expected bases agree with its codon on shared columns
        struct Layer { int8_t base[34]; std::vector<int32_t> vars; };
        std::vector<Layer> layers;
        for (int32_t v : by_block[sl]) {
            const int32_t c = var_col[v] & 31;
            const int8_t cod[3] = {static_cast<int8_t>((var_codon[v] >> 4) & 3), static_cast<int8_t>((var_codon[v] >> 2) & 3), static_cast<int8_t>(var_codon[v] & 3)};
            size_t li = 0;
            for (; li < layers.size(); ++li) {
                bool ok = true;
                for (int k = 0; k < 3; ++k) ok = ok && (layers[li].base[c + k] < 0 || layers[li].base[c + k] == cod[k]);
                if (ok) break;
            }
            if (li == layers.size()) { layers.emplace_back(); memset(layers.back().base, -1, sizeof layers.back().base); }
            for (int k = 0; k < 3; ++k) layers[li].base[c + k] = cod[k];
            layers[li].vars.push_back(v);
        }
        if (layers.empty()) { layers.emplace_back(); memset(layers.back().base, -1, sizeof layers.back().base); }   // spill-over block: flags only
        for (size_t li = 0; li < layers.size(); ++li) {
            const Layer& ly = layers[li];
            if (ly.vars.size() > 0x7FF) MS_FAIL(h, MS_ERR_CAPACITY, "more than 2047 variants start in one 32-column block");
            uint32_t e0 = 0, e1 = 0, en = 0;
            for (int c = 0; c < 32; ++c)
                if (ly.base[c] > 0) { e0 |= static_cast<uint32_t>(ly.base[c] & 1) << c; e1 |= static_cast<uint32_t>((ly.base[c] >> 1) & 1) << c; }
            for (int c = 32; c < 34; ++c)
                if (ly.base[c] > 0) { en |= static_cast<uint32_t>(ly.base[c] & 1) << (c - 32); en |= static_cast<uint32_t>((ly.base[c] >> 1) & 1) << (c - 32 + 2); }
            // packed form: consecutive indices on strictly increasing start columns (at least a few, or the 7 words do not pay)
            bool packed = ly.vars.size() >= 4 && ly.vars.size() <= 32;
            uint32_t smask = 0;
            for (size_t k = 0; k < ly.vars.size() && packed; ++k) {
                if (k > 0 && (ly.vars[k] != ly.vars[k - 1] + 1 || var_col[ly.vars[k]] <= var_col[ly.vars[k - 1]])) packed = false;
                smask |= 1u << (var_col[ly.vars[k]] & 31);
            }
            vd.push_back(static_cast<uint32_t>(sl) | (static_cast<uint32_t>(ly.vars.size()) << 13) | (li == 0 ? ms::kHdrFirst : 0u) |
                         (packed ? ms::kHdrPacked : 0u));
            vd.push_back(e0); vd.push_back(e1); vd.push_back(en); vd.push_back(li == 0 ? cover[sl] : 0u);
            if (packed) {
                // move masks of the parallel-suffix compress of smask (Hacker's Delight, "compress", figure 7-10)
                vd.push_back(smask);
                uint32_t m = smask, mk = ~m << 1;
                for (int i = 0; i < 5; ++i) {
                    uint32_t mp = mk ^ (mk << 1);
                    mp ^= mp << 2; mp ^= mp << 4; mp ^= mp << 8; mp ^= mp << 16;
                    const uint32_t mv = mp & m;
                    vd.push_back(mv);
                    m = (m ^ mv) | (mv >> (1 << i));
                    mk &= ~mp;
                }
                vd.push_back(static_cast<uint32_t>(ly.vars[0]));
            }
            for (int32_t v : ly.vars) {
                if (!packed) vd.push_back(static_cast<uint32_t>(var_col[v] & 31) | (static_cast<uint32_t>(v) << 5));
                const int64_t wi = v >> 5;
                if (wi != last_word) { if (word_seen[wi]) ordered = false; word_seen[wi] = 1; last_word = wi; }
            }
        }
    }
    h->phase_nrec = static_cast<int32_t>(vd.size());
    h->phase_ordered = ordered;
    if (vd.empty()) vd.push_back(0u);
    // The table starts small (distinct patterns are usually a few hundred) and is re-sized by
    // ms_phase_groups when an insert reports overflow; its upper bound is 2x the reads.
    int64_t ts_max = 1024;
    while (ts_max < 2 * h->phase_cap) ts_max <<= 1;
    h->tab_size_max = ts_max;
    int64_t ts = std::min<int64_t>(ts_max, std::max<int64_t>(1 << 16, h->tab_hint));   // last pass's grown size is the hint
    h->tab_size = ts;
    // the previous pass may still be reading these buffers on the stream if they have to move
    const bool grow = vd.size() * 4 > h->b_var.cap || blocks.size() * 4 > h->b_blocklist.cap ||
                      static_cast<size_t>(h->phase_cap) * h->vwords * 4 > h->b_bits.cap || static_cast<size_t>(h->phase_cap) > h->b_flags.cap ||
                      static_cast<size_t>(ts) * 8 > h->b_tab_key.cap || !h->b_ctr.p ||
                      ((h->linkage || h->abundance) && static_cast<size_t>(h->phase_cap) * h->vwords * 4 > h->b_mbits.cap);
    if (grow) MS_CUDA(h, cudaStreamSynchronize(h->stream));
    if (h->linkage || h->abundance) {   // the clean-codon matrix of pairwise linkage and haplotype abundance, same shape as the bit matrix
        MS_CUDA(h, h->b_mbits.ensure(static_cast<size_t>(h->phase_cap) * h->vwords * 4));
        h->link_col.assign(var_col, var_col + V);
        h->link_ready = true;
    }
    MS_CUDA(h, h->b_var.ensure(vd.size() * 4));
    MS_CUDA(h, h->b_blocklist.ensure(blocks.size() * 4));
    MS_CUDA(h, h->b_bits.ensure(static_cast<size_t>(h->phase_cap) * h->vwords * 4));
    MS_CUDA(h, h->b_flags.ensure(static_cast<size_t>(h->phase_cap)));
    MS_CUDA(h, h->b_slot.ensure(static_cast<size_t>(h->phase_cap) * 4));
    MS_CUDA(h, h->b_tab_key.ensure(static_cast<size_t>(ts) * 8));
    MS_CUDA(h, h->b_tab_cnt.ensure(static_cast<size_t>(ts) * 4));
    MS_CUDA(h, h->b_tab_rep.ensure(static_cast<size_t>(ts) * 8));
    MS_CUDA(h, h->b_ctr.ensure(64));
    int rc = ensure_stage(h, 1 << 20);
    if (rc != MS_OK) return rc;
    // pageable -> device copies of the small tables go through the pinned stage to stay asynchronous
    uint8_t* st = static_cast<uint8_t*>(h->h_stage);
    const size_t nb_var = vd.size() * 4, nb_blk = blocks.size() * 4;
    if (nb_var + nb_blk <= h->h_stage_cap) {
        memcpy(st, vd.data(), nb_var);
        memcpy(st + nb_var, blocks.data(), nb_blk);
        MS_CUDA(h, cudaMemcpyAsync(h->b_var.p, st, nb_var, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(h->b_blocklist.p, st + nb_var, nb_blk, cudaMemcpyHostToDevice, h->stream));
    } else {
        MS_CUDA(h, cudaMemcpy(h->b_var.p, vd.data(), nb_var, cudaMemcpyHostToDevice));
        MS_CUDA(h, cudaMemcpy(h->b_blocklist.p, blocks.data(), nb_blk, cudaMemcpyHostToDevice));
    }
    MS_CUDA(h, cudaMemsetAsync(h->b_ctr.p, 0, 64, h->stream));
    return MS_OK;
}

int ms_phase_dev(ms_handle* h, const uint32_t* d_packed, int64_t R) {
    MsRange nvtx_range("K3 phase bits");
    if (!h || !h->b_bits.p || R < 0 || (R > 0 && !d_packed)) return MS_ERR_ARG;
    if (h->phase_n + R > h->phase_cap) MS_FAIL(h, MS_ERR_CAPACITY, "more reads than ms_phase_begin(max_reads)");
    if (R == 0) return MS_OK;
    MS_CUDA(h, cudaSetDevice(h->device));
    h->table_valid = false;
    h->groups_valid = false;
    h->gram_valid = false;
    h->hap_ranked = h->hap_assigned = false;
    uint32_t* bits = h->b_bits.as<uint32_t>() + static_cast<size_t>(h->phase_n) * h->vwords;
    uint32_t* mbits = h->link_ready ? h->b_mbits.as<uint32_t>() + static_cast<size_t>(h->phase_n) * h->vwords : nullptr;
    uint8_t* flags = h->b_flags.as<uint8_t>() + h->phase_n;
    const uint4* pk = reinterpret_cast<const uint4*>(d_packed);
    const uint32_t* stream = h->b_var.as<uint32_t>();
    unsigned long long* ctr = ctr_ptr(h);
    if (!(h->phase_ordered && h->vwords == 1)) {   // one-word ordered vectors are written in full by the kernel
        MS_CUDA(h, cudaMemsetAsync(bits, 0, static_cast<size_t>(R) * h->vwords * 4, h->stream));   // words no variant maps to stay zero
        if (mbits) MS_CUDA(h, cudaMemsetAsync(mbits, 0, static_cast<size_t>(R) * h->vwords * 4, h->stream));
    }
    MS_STAGE_BEGIN(h, MS_STAGE_PHASE_BITS);
    {
        // up to 16 touched blocks: one chunk, all of it in flight at once; longer lists: chunks of 8, double-buffered
        const bool dbuf = h->nblocklist > ms::kPhaseChunkMax;
        const int chunk = dbuf ? ms::kPhaseChunkMax / 2 : std::min(ms::kPhaseChunkMax, h->nblocklist);
        const size_t smem = static_cast<size_t>(ms::kPhaseWarps) * (dbuf ? 2 : 1) * (chunk + 1) * 32 * sizeof(uint4);
        const int per_sm = std::max(1, std::min(6, static_cast<int>((h->max_smem + 1024) / (smem + 1024))));
        const int64_t want = (R + ms::kPhaseWarps * 32 - 1) / (ms::kPhaseWarps * 32);
        const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(want, static_cast<int64_t>(h->num_sms) * per_sm)));
        if (mbits)     // linkage or abundance was requested: the same walk also writes the clean-codon matrix
            ms::phase_bits_kernel<true><<<grid, ms::kPhaseWarps * 32, smem, h->stream>>>(pk, R, h->nblk, h->b_blocklist.as<int32_t>(), h->nblocklist, chunk,
                                                                                        dbuf ? 1 : 0, stream, h->phase_nrec, h->vwords,
                                                                                        h->phase_ordered ? 1 : 0, h->phase_partial_all ? 1 : 0, bits, flags,
                                                                                        ctr, nullptr, mbits);
        else
            ms::phase_bits_kernel<false><<<grid, ms::kPhaseWarps * 32, smem, h->stream>>>(pk, R, h->nblk, h->b_blocklist.as<int32_t>(), h->nblocklist, chunk, dbuf ? 1 : 0,
                                                                                         stream, h->phase_nrec, h->vwords, h->phase_ordered ? 1 : 0,
                                                                                         h->phase_partial_all ? 1 : 0, bits, flags, ctr, nullptr, nullptr);
    }
    MS_STAGE_END(h, MS_STAGE_PHASE_BITS);
    h->launches++;
    MS_CUDA(h, cudaGetLastError());
    h->phase_n += R;
    return MS_OK;
}

}  // extern "C"

// ---- the planned form of ms_phase_begin + ms_phase_dev used by the single-call pass (pass.cu): the variant list is still on
// the device (d_calls / d_ncalls, K2's output buffers); phase_plan_kernel builds the plan there, phase_bits_kernel reads its
// sizes from it.  One-word bit-vectors (V <= 32).  The caller reads the plan back with the pass's final download and, if it
// says `fallback`, runs the host-planned calls after all.
int ms_phase_planned_dev(ms_handle* h, const ms_variant* d_calls, const unsigned long long* d_ncalls, int64_t calls_cap,
                         const uint32_t* d_packed, int64_t R, ms::PhasePlan** d_plan_out) {
    if (!h || h->L <= 0 || R < 0 || !d_calls || !d_ncalls || (R > 0 && !d_packed)) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    h->V = 0;                       // known after the download of the plan (ms_phase_planned_adopt)
    h->vwords = 1;
    h->link_ready = h->gram_valid = false;   // this pass writes no clean-codon matrix
    h->hap_ranked = h->hap_assigned = false;
    h->phase_cap = std::max<int64_t>(1, R);
    h->phase_n = 0;
    h->table_valid = false;
    h->groups_valid = false;
    int64_t ts_max = 1024;
    while (ts_max < 2 * h->phase_cap) ts_max <<= 1;
    h->tab_size_max = ts_max;
    const int64_t ts = std::min<int64_t>(ts_max, std::max<int64_t>(1 << 16, h->tab_hint));
    h->tab_size = ts;
    const size_t plan_bytes = sizeof(ms::PhasePlan);
    const bool grow = static_cast<size_t>(ms::kPlanStreamWords) * 4 > h->b_var.cap || static_cast<size_t>(ms::kPlanMaxBlocks) * 4 > h->b_blocklist.cap ||
                      static_cast<size_t>(h->phase_cap) * 4 > h->b_bits.cap || static_cast<size_t>(h->phase_cap) > h->b_flags.cap ||
                      static_cast<size_t>(ts) * 8 > h->b_tab_key.cap || !h->b_ctr.p || plan_bytes > h->b_plan.cap;
    if (grow) MS_CUDA(h, cudaStreamSynchronize(h->stream));
    MS_CUDA(h, h->b_var.ensure(static_cast<size_t>(ms::kPlanStreamWords) * 4));
    MS_CUDA(h, h->b_blocklist.ensure(static_cast<size_t>(ms::kPlanMaxBlocks) * 4));
    MS_CUDA(h, h->b_bits.ensure(static_cast<size_t>(h->phase_cap) * 4));
    MS_CUDA(h, h->b_flags.ensure(static_cast<size_t>(h->phase_cap)));
    MS_CUDA(h, h->b_slot.ensure(static_cast<size_t>(h->phase_cap) * 4));
    MS_CUDA(h, h->b_tab_key.ensure(static_cast<size_t>(ts) * 8));
    MS_CUDA(h, h->b_tab_cnt.ensure(static_cast<size_t>(ts) * 4));
    MS_CUDA(h, h->b_tab_rep.ensure(static_cast<size_t>(ts) * 8));
    MS_CUDA(h, h->b_ctr.ensure(64));
    MS_CUDA(h, h->b_plan.ensure(plan_bytes));
    int rc = ensure_stage(h, 1 << 20);
    if (rc != MS_OK) return rc;
    ms::PhasePlan* d_plan = h->b_plan.as<ms::PhasePlan>();
    MS_CUDA(h, cudaMemsetAsync(h->b_ctr.p, 0, 64, h->stream));
    ms::phase_plan_kernel<<<1, 32, 0, h->stream>>>(d_calls, d_ncalls, calls_cap, h->L, d_plan, h->b_blocklist.as<int32_t>(), h->b_var.as<uint32_t>());
    h->launches++;
    if (R > 0) {
        MS_STAGE_BEGIN(h, MS_STAGE_PHASE_BITS);   // (one-word ordered vectors: no zeroing of the bit matrix needed)
        const int chunk = ms::kPhaseChunkMax;          // the block count is only known on the device: stage with the largest chunk
        const size_t smem = static_cast<size_t>(ms::kPhaseWarps) * (chunk + 1) * 32 * sizeof(uint4);
        const int per_sm = std::max(1, std::min(6, static_cast<int>((h->max_smem + 1024) / (smem + 1024))));
        const int64_t want = (R + ms::kPhaseWarps * 32 - 1) / (ms::kPhaseWarps * 32);
        const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(want, static_cast<int64_t>(h->num_sms) * per_sm)));
        ms::phase_bits_kernel<false><<<grid, ms::kPhaseWarps * 32, smem, h->stream>>>(reinterpret_cast<const uint4*>(d_packed), R, h->nblk,
                                                                                     h->b_blocklist.as<int32_t>(), 0, chunk, 0, h->b_var.as<uint32_t>(), 0, 1,
                                                                                     1, 0, h->b_bits.as<uint32_t>(), h->b_flags.as<uint8_t>(), ctr_ptr(h),
                                                                                     d_plan, nullptr);
        MS_STAGE_END(h, MS_STAGE_PHASE_BITS);
        h->launches++;
    }
    MS_CUDA(h, cudaGetLastError());
    h->phase_n = R;
    if (d_plan_out) *d_plan_out = d_plan;
    return MS_OK;
}

// after the plan has been read back: the handle learns the number of keys (ms_cooccurrence, ms_phase_device need it)
void ms_phase_planned_adopt(ms_handle* h, int32_t V) { h->V = V; }

// G (dim x dim int32, full symmetric) = S^T S over the phased reads, S = the nmat bit matrices mats[k] (R rows of h->vwords
// words each) side by side, matrix k's variants at rows 32 * vwords * k of the stacked transpose.  ms_cooccurrence is the
// one-matrix case (dim = V); pairwise linkage stacks the bit matrix and the clean-codon matrix (dim = 64 * vwords).  The
// contraction goes to the tensor cores when it is big enough to be one (cooc_tc.cu: V >= 256 variants and >= 32768 reads);
// the popcount-AND kernel serves the usual few-dozen-variant case, where the matrix is tiny.  Same integers either way.
int ms_gram_dev(ms_handle* h, const uint32_t* const* mats, int nmat, int32_t dim, int32_t* G) {
    const int32_t V = h->V, nw = h->vwords;
    const int64_t R = h->phase_n;
    const bool tensor = h->cooc_variant == 2 || (h->cooc_variant == 0 && V >= 256 && R >= 32768);
    // row stride of the transposed bit matrix: whole 128-read stages for the tensor path (zero padded)
    const int64_t rwords = tensor ? 4 * ((R + 127) / 128) : std::max<int64_t>(1, (R + 31) / 32);
    const size_t gbytes = std::max<size_t>(4, static_cast<size_t>(dim) * dim * 4);
    const size_t mat_words = static_cast<size_t>(nw) * 32 * rwords;
    MS_CUDA(h, h->b_bits_t.ensure(std::max<size_t>(16, nmat * mat_words * 4)));
    MS_CUDA(h, cudaMemsetAsync(G, 0, gbytes, h->stream));
    if (V > 0 && rwords > 0) {
        const int64_t nwarps = rwords * nw;
        for (int k = 0; k < nmat; ++k) {
            ms::bits_transpose_kernel<<<static_cast<unsigned>((nwarps * 32 + 255) / 256), 256, 0, h->stream>>>(mats[k], R, nw, rwords,
                                                                                                             h->b_bits_t.as<uint32_t>() + k * mat_words);
            h->launches++;
        }
        MS_STAGE_BEGIN(h, MS_STAGE_COOCCURRENCE);
        if (tensor) {
            int rc = ms_cooccurrence_tc_launch(h, h->b_bits_t.as<uint32_t>(), dim, rwords, R, G);
            if (rc != MS_OK) return rc;
        } else {
            dim3 grid((dim + ms::kCoTile - 1) / ms::kCoTile, (dim + ms::kCoTile - 1) / ms::kCoTile);
            ms::cooccurrence_kernel<<<grid, 256, 0, h->stream>>>(h->b_bits_t.as<uint32_t>(), dim, rwords, G);
            h->launches++;
        }
        MS_STAGE_END(h, MS_STAGE_COOCCURRENCE);
    }
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

extern "C" {

int ms_phase_groups(ms_handle* h, uint32_t* patterns, uint64_t* counts, int64_t cap, int64_t* H, ms_phase_counters* ctr) {
    MsRange nvtx_range("K3 grouping");
    if (!h || !h->b_bits.p || !H) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    if (h->groups_valid) return phase_groups_copy_out(h, patterns, counts, cap, H, ctr);   // same pass asked again (bigger cap)
    const int32_t nw = h->vwords;
    const int world = h->comm ? h->world : 1;
    int64_t gcap = kGroupCapInit;
    int attempt = h->table_valid ? h->table_attempt : 0;
    std::vector<uint32_t> all_cnt, all_pat;   // concatenation over ranks
    uint64_t marg[4] = {0, 0, 0, 0};
    for (;;) {
        if (!h->table_valid) {
            int rc = build_table(h, attempt);
            if (rc != MS_OK) return rc;
        }
        // block = [64-byte header (the 8 counters) | cnt u32[gcap] | pat u32[gcap*nw]]
        const size_t block = 64 + static_cast<size_t>(gcap) * 4 * (1 + nw);
        MS_CUDA(h, h->b_groups.ensure(block));
        if (world > 1) MS_CUDA(h, h->b_gather.ensure(block * world));
        int rc = ensure_stage(h, block * world);
        if (rc != MS_OK) return rc;
        uint8_t* blk = h->b_groups.as<uint8_t>();
        uint32_t* g_cnt = reinterpret_cast<uint32_t*>(blk + 64);
        uint32_t* g_pat = g_cnt + gcap;
        rc = ms::phase_compact(h, g_cnt, g_pat, nullptr, gcap);
        if (rc != MS_OK) return rc;
        MS_CUDA(h, cudaMemcpyAsync(blk, h->b_ctr.p, 64, cudaMemcpyDeviceToDevice, h->stream));
        uint8_t* st = static_cast<uint8_t*>(h->h_stage);
        if (world > 1) {
            // the only exchange of the phasing step: every rank's compact (pattern, count) list and marginals
            rc = ms_comm_allgather_bytes(h, blk, h->b_gather.p, block);
            if (rc != MS_OK) return rc;
            MS_CUDA(h, cudaMemcpyAsync(st, h->b_gather.p, block * world, cudaMemcpyDeviceToHost, h->stream));
        } else {
            MS_CUDA(h, cudaMemcpyAsync(st, blk, block, cudaMemcpyDeviceToHost, h->stream));
        }
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        // every rank sees every header, so all ranks take the same branch below
        bool any_collision = false, any_overflow = false;
        int64_t max_ng = 0;
        const int me = h->comm ? h->rank : 0;
        for (int r = 0; r < world; ++r) {
            uint64_t hc[8];
            memcpy(hc, st + static_cast<size_t>(r) * block, 64);
            if ((hc[6] != 0 || hc[4] != 0) && (hc[7] & 0xff) != 0)   // rank r cannot recover: every rank sees this header and stops here
                MS_FAIL(h, MS_ERR_CUDA, hc[6] != 0 ? "haplotype table overflow at maximum size" : "haplotype hash collided under four seeds");
            if (hc[6] != 0) {
                any_overflow = true;
                if (r == me) {  // table too small for this rank's distinct patterns: grow and rebuild
                    rc = ms::phase_grow_table(h);
                    if (rc != MS_OK) return rc;
                    h->table_valid = false;
                }
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
        }
        if (any_collision || any_overflow) continue;
        if (max_ng > gcap) { gcap = max_ng; continue; }
        all_cnt.clear(); all_pat.clear();
        for (int r = 0; r < world; ++r) {
            const uint8_t* base = st + static_cast<size_t>(r) * block;
            uint64_t hc[8];
            memcpy(hc, base, 64);
            for (int i = 0; i < 4; ++i) marg[i] += hc[i];
            const uint32_t* c = reinterpret_cast<const uint32_t*>(base + 64);
            const uint32_t* p = c + gcap;
            all_cnt.insert(all_cnt.end(), c, c + hc[5]);
            all_pat.insert(all_pat.end(), p, p + hc[5] * nw);
        }
        break;
    }
    h->groups_cnt.swap(all_cnt);
    h->groups_pat.swap(all_pat);
    for (int i = 0; i < 4; ++i) h->groups_marg[i] = marg[i];
    h->groups_valid = true;
    return phase_groups_copy_out(h, patterns, counts, cap, H, ctr);
}

int ms_haplotype_order(uint32_t* patterns, uint64_t* counts, int64_t H, int32_t V, int32_t min_reads, int64_t* Hmerged,
                       int64_t* nreported, ms_phase_counters* ctr) {
    if (H < 0 || (H > 0 && (!patterns || !counts)) || V < 0) return MS_ERR_ARG;
    const int32_t nw = std::max(1, (V + 31) / 32);
    auto pat = [&](int64_t i) { return patterns + static_cast<size_t>(i) * nw; };
    // 1. merge equal patterns (the same haplotype seen on several ranks) with a hash join: O(H)
    int64_t ts = 16;
    while (ts < 2 * H) ts <<= 1;
    std::vector<int64_t> table(ts, -1);
    std::vector<int64_t> first;        // merged group -> index of its first occurrence
    std::vector<uint64_t> mc;
    for (int64_t i = 0; i < H; ++i) {
        uint64_t hsh = 0x9E3779B97F4A7C15ULL;
        for (int32_t w = 0; w < nw; ++w) {
            hsh ^= pat(i)[w] + 0x9E3779B97F4A7C15ULL + (hsh << 6) + (hsh >> 2);
            hsh *= 0xbf58476d1ce4e5b9ULL;
            hsh ^= hsh >> 29;
        }
        int64_t slot = static_cast<int64_t>(hsh) & (ts - 1);
        for (;;) {
            const int64_t g = table[slot];
            if (g < 0) { table[slot] = static_cast<int64_t>(first.size()); first.push_back(i); mc.push_back(counts[i]); break; }
            if (memcmp(pat(first[g]), pat(i), static_cast<size_t>(nw) * 4) == 0) { mc[g] += counts[i]; break; }
            slot = (slot + 1) & (ts - 1);
        }
    }
    const int64_t M = static_cast<int64_t>(first.size());
    // 2. juliet's order for the reported ones: count descending, ties by ascending pattern words.
    //    The unreported rest follows; it is sorted the same way unless it is huge (phasing stress runs
    //    produce hundreds of thousands of single-read patterns nobody lists).
    std::vector<int64_t> rep, rest;
    uint64_t nrep_reads = 0, nins_reads = 0;
    for (int64_t g = 0; g < M; ++g) {
        if (mc[g] >= static_cast<uint64_t>(min_reads)) { rep.push_back(g); nrep_reads += mc[g]; }
        else { rest.push_back(g); nins_reads += mc[g]; }
    }
    auto by_order = [&](int64_t a, int64_t b) {
        if (mc[a] != mc[b]) return mc[a] > mc[b];
        return ms::pattern_less(pat(first[a]), pat(first[b]), nw);
    };
    std::sort(rep.begin(), rep.end(), by_order);
    if (rest.size() <= 65536) std::sort(rest.begin(), rest.end(), by_order);
    std::vector<uint32_t> op(static_cast<size_t>(M) * nw);
    std::vector<uint64_t> oc(M);
    int64_t k = 0;
    for (const std::vector<int64_t>* part : {&rep, &rest})
        for (int64_t g : *part) {
            memcpy(op.data() + static_cast<size_t>(k) * nw, pat(first[g]), static_cast<size_t>(nw) * 4);
            oc[k++] = mc[g];
        }
    if (M) { memcpy(patterns, op.data(), op.size() * 4); memcpy(counts, oc.data(), oc.size() * 8); }
    if (Hmerged) *Hmerged = M;
    if (nreported) *nreported = static_cast<int64_t>(rep.size());
    if (ctr) { ctr->reported = nrep_reads; ctr->insufficient = nins_reads; }
    return MS_OK;
}

void ms_haplotype_name(int64_t rank, char buf[3]) {
    if (rank < 26) { buf[0] = static_cast<char>('A' + rank); buf[1] = 0; return; }
    rank -= 26;
    buf[0] = static_cast<char>('A' + (rank / 26) % 26); buf[1] = static_cast<char>('a' + rank % 26); buf[2] = 0;
}

int ms_phase_assign(ms_handle* h, const uint32_t* ordered_patterns, int64_t H, int32_t* hap_id) {
    if (!h || !h->b_bits.p || H < 0 || (H > 0 && !ordered_patterns) || !hap_id) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    if (!h->table_valid) {
        // with a communicator the grouping pass is a collective: it must not be entered from here by some ranks only
        if (h->comm) MS_FAIL(h, MS_ERR_ARG, "ms_phase_assign: call ms_phase_groups (on every rank) first");
        int64_t dummy = 0;
        int rc = ms_phase_groups(h, nullptr, nullptr, 0, &dummy, nullptr);
        if (rc != MS_OK) return rc;
    }
    const int64_t R = h->phase_n;
    const int32_t nw = h->vwords;
    h->hap_ranked = h->hap_assigned = false;   // b_rank / b_hap now follow the caller's pattern list
    MS_CUDA(h, h->b_rank.ensure(static_cast<size_t>(h->tab_size) * 4));
    MS_CUDA(h, h->b_hap.ensure(static_cast<size_t>(std::max<int64_t>(1, R)) * 4));
    MS_CUDA(h, h->b_pat.ensure(static_cast<size_t>(std::max<int64_t>(1, H)) * nw * 4));
    MS_CUDA(h, cudaMemsetAsync(h->b_rank.p, 0xff, static_cast<size_t>(h->tab_size) * 4, h->stream));
    if (H > 0) {
        MS_CUDA(h, cudaMemcpyAsync(h->b_pat.p, ordered_patterns, static_cast<size_t>(H) * nw * 4, cudaMemcpyHostToDevice, h->stream));
        ms::phase_rank_kernel<<<static_cast<int>((H + 127) / 128), 128, 0, h->stream>>>(
            h->b_pat.as<uint32_t>(), H, nw, phase_seed(h->table_attempt), h->b_tab_key.as<unsigned long long>(),
            h->b_tab_rep.as<long long>(), h->tab_size - 1, h->b_bits.as<uint32_t>(), h->b_rank.as<int32_t>());
        h->launches++;
    }
    if (R > 0) {
        ms::phase_assign_kernel<<<static_cast<int>((R + 255) / 256), 256, 0, h->stream>>>(h->b_slot.as<int32_t>(), h->b_rank.as<int32_t>(), R,
                                                                                         h->b_hap.as<int32_t>());
        h->launches++;
        MS_CUDA(h, cudaMemcpyAsync(hap_id, h->b_hap.p, static_cast<size_t>(R) * 4, cudaMemcpyDeviceToHost, h->stream));
    }
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    MS_CUDA(h, cudaGetLastError());
    return MS_OK;
}

int ms_phase_device(ms_handle* h, uint32_t** d_bits, uint8_t** d_flags, int64_t* R) {
    if (!h || !h->b_bits.p) return MS_ERR_ARG;
    if (d_bits) *d_bits = h->b_bits.as<uint32_t>();
    if (d_flags) *d_flags = h->b_flags.as<uint8_t>();
    if (R) *R = h->phase_n;
    return MS_OK;
}

int ms_set_cooccurrence_variant(ms_handle* h, int32_t variant) {
    if (!h || variant < 0 || variant > 2) return MS_ERR_ARG;
    h->cooc_variant = variant;
    return MS_OK;
}

int ms_cooccurrence(ms_handle* h, int32_t** d_C) {
    MsRange nvtx_range("K3 co-occurrence");
    if (!h || !h->b_bits.p || !d_C) return MS_ERR_ARG;
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t V = h->V;
    const size_t cbytes = std::max<size_t>(4, static_cast<size_t>(V) * V * 4);
    MS_CUDA(h, h->b_cooc.ensure(cbytes));
    const uint32_t* mats[1] = {h->b_bits.as<uint32_t>()};
    const int rc = ms_gram_dev(h, mats, 1, V, h->b_cooc.as<int32_t>());
    if (rc != MS_OK) return rc;
    *d_C = h->b_cooc.as<int32_t>();
    return MS_OK;
}

}  // extern "C"
