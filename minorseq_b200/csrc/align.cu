// align.cu -- K6: overlap alignment of unaligned CCS reads to an amplicon reference (restatement choice U16).
//
// Seeds: the reference's unique 15-mers sit in an open-addressing hash table (built on the host once per reference,
// ms_align_set_reference).  align_seed_kernel gives each read one warp: for each strand the lanes look up the k-mers at
// q = 0 (mod 4), compact the hits' diagonals in q order into the warp's scratch, count for every hit the hits in the
// 65 diagonals ending at its own, and take the first hit (in q order) of the best window.
//
// Band: align_band_kernel is persistent, one warp per read.  Lane l owns the band cells p = 4l..4l+3 of an
// anti-diagonal k = i + j (read index i, reference index j, i = b_k + p).  The two previous anti-diagonals are held
// re-indexed to the current band, so every neighbour is a register or a one-lane shuffle; when the band moves down the
// arrays shift by one cell.  The read and reference bases of the cells shift the same way and cost one load per step.
// Two move bits per cell go to the warp's slab (lane l's byte of four consecutive anti-diagonals is one u32, so every
// fourth step the warp writes one 128-byte line), one band-move bit per anti-diagonal to a second array.  The same warp
// then walks back: 32 anti-diagonals (1 KB) of the slab at a time are staged in shared memory, and all lanes walk the
// path in lockstep, lane 0 writing the run-length CIGAR (reversed) into the read's slot.
#include <algorithm>
#include <cstring>
#include <vector>
#include "align_rule.h"
#include "handle.h"

namespace ms {

constexpr int kAlnW = MS_ALN_BAND;
constexpr int kAlnNeg = MS_ALN_NEG;
constexpr int kSeedWarps = 8, kBandWarps = 4;
constexpr int64_t kAlnChunkBases = int64_t(MS_ALN_CHUNK_MBASES) << 20, kAlnChunkReads = MS_ALN_CHUNK_READS;
constexpr size_t kAlnSlabBudget = size_t(4) << 30;   // move bits of the resident warps

static_assert(kAlnW == 128, "4 cells per lane of a warp");

__device__ __forceinline__ int base_code(char c) {
    return c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : c == 'T' ? 3 : -1;
}
// base i of the aligned read (strand 1: the reverse complement of the native read); 4 = not ACGT or outside
__device__ __forceinline__ int read_code(const char* s, int la, int strand, int i) {
    if (i < 0 || i >= la) return 4;
    const int x = base_code(strand ? s[la - 1 - i] : s[i]);
    return x < 0 ? 4 : (strand ? 3 - x : x);
}
// reference base j; 5 = not ACGT or outside (never equal to a read code, so such a pair is a mismatch)
__device__ __forceinline__ int ref_code(const char* r, int lb, int j) {
    if (j < 0 || j >= lb) return 5;
    const int x = base_code(r[j]);
    return x < 0 ? 5 : x;
}
__device__ __forceinline__ int lookup(const unsigned long long* tab, uint32_t mask, int bits, uint32_t kmer) {
    uint32_t s = (kmer * 0x9E3779B1u) >> (32 - bits);
    for (;;) {
        const unsigned long long e = tab[s];
        if (static_cast<uint32_t>(e) == 0u) return -1;
        if (static_cast<uint32_t>(e >> 32) == kmer) return static_cast<int>(static_cast<uint32_t>(e)) - 1;
        s = (s + 1) & mask;
    }
}

// seed[r] = {mapped, strand, d0, support}
__global__ void __launch_bounds__(kSeedWarps * 32) align_seed_kernel(const char* __restrict__ seq, const int64_t* __restrict__ off, int64_t R,
                                                                    const unsigned long long* __restrict__ tab, int bits, int lb, int min_seeds,
                                                                    int* __restrict__ scratch, int npos_max, int* __restrict__ ctr,
                                                                    int4* __restrict__ seed) {
    const int lane = threadIdx.x & 31;
    int* hits = scratch + static_cast<int64_t>(blockIdx.x * kSeedWarps + (threadIdx.x >> 5)) * npos_max;
    const uint32_t mask = (1u << bits) - 1u;
    for (;;) {
        int64_t r = 0;
        if (lane == 0) r = atomicAdd(ctr, 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r >= R) return;
        const char* s = seq + off[r];
        const int la = static_cast<int>(off[r + 1] - off[r]);
        const int npos = la >= MS_ALN_K ? (la - MS_ALN_K) / MS_ALN_STRIDE + 1 : 0;
        int best_sup = 0, best_strand = 0, best_d0 = 0;
        for (int strand = 0; strand < 2; ++strand) {
            int n = 0;
            for (int q0 = 0; q0 < npos; q0 += 32) {
                const int q = (q0 + lane) * MS_ALN_STRIDE;
                int t = -1;
                if (q0 + lane < npos) {
                    uint32_t kmer = 0;
                    bool ok = true;
                    for (int x = 0; x < MS_ALN_K; ++x) {
                        const int c = read_code(s, la, strand, q + x);
                        ok = ok && c < 4;
                        kmer = (kmer << 2) | static_cast<uint32_t>(c & 3);
                    }
                    if (ok) t = lookup(tab, mask, bits, kmer);
                }
                const unsigned hit = __ballot_sync(0xffffffffu, t >= 0);
                if (t >= 0) hits[n + __popc(hit & ((1u << lane) - 1u))] = t - q;
                n += __popc(hit);
            }
            __syncwarp();
            // support: for each hit e, the hits with diagonal in [d_e - 64, d_e]; the best window is the first by its top diagonal
            int sup = 0, top = 0x7fffffff;
            for (int e = lane; e < n; e += 32) {
                const int de = hits[e];
                int cnt = 0;
                for (int x = 0; x < n; ++x) {
                    const int dx = hits[x];
                    cnt += (dx <= de && dx >= de - (MS_ALN_WINDOW - 1)) ? 1 : 0;
                }
                if (cnt > sup || (cnt == sup && de < top)) { sup = cnt; top = de; }
            }
            for (int o = 16; o > 0; o >>= 1) {
                const int s2 = __shfl_xor_sync(0xffffffffu, sup, o), t2 = __shfl_xor_sync(0xffffffffu, top, o);
                if (s2 > sup || (s2 == sup && t2 < top)) { sup = s2; top = t2; }
            }
            // d0: the hit of that window with the smallest q (hits are in q order)
            int first = 0x7fffffff;
            for (int e = lane; e < n && first == 0x7fffffff; e += 32) {
                const int de = hits[e];
                if (de <= top && de >= top - (MS_ALN_WINDOW - 1)) first = e;
            }
            for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
            if (sup > best_sup) { best_sup = sup; best_strand = strand; best_d0 = n ? hits[first] : 0; }
            __syncwarp();
        }
        if (lane == 0) seed[r] = make_int4(best_sup >= min_seeds ? 1 : 0, best_strand, best_d0, best_sup);
    }
}

__global__ void __launch_bounds__(kBandWarps * 32) align_band_kernel(const char* __restrict__ seq, const int64_t* __restrict__ off, int64_t R,
                                                                    const char* __restrict__ ref, int lb, const int4* __restrict__ seed,
                                                                    uint32_t* __restrict__ slab, uint32_t* __restrict__ mbits, int64_t slab_words,
                                                                    int64_t mbits_words, int* __restrict__ ctr, uint32_t* __restrict__ cig,
                                                                    ms_read_alignment* __restrict__ res) {
    __shared__ uint32_t stage[kBandWarps][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = static_cast<int64_t>(blockIdx.x) * kBandWarps + wib;
    uint32_t* my_slab = slab + warp * slab_words;
    uint32_t* my_mb = mbits + warp * mbits_words;
    const int64_t off0 = off[0];
    for (;;) {
        int64_t r = 0;
        if (lane == 0) r = atomicAdd(ctr, 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r >= R) return;
        const int4 sd = seed[r];
        const int64_t slot = 2 * (off[r] - off0) + r;    // room for 2 la + 1 ops
        if (!sd.x) {
            if (lane == 0) {
                ms_read_alignment o;
                o.mapped = 0; o.strand = 0; o.pos = -1; o.score = 0; o.cigar_off = slot; o.ncigar = 0;
                res[r] = o;
            }
            continue;
        }
        const char* s = seq + off[r];
        const int la = static_cast<int>(off[r + 1] - off[r]), strand = sd.y, d0 = sd.z;
        const int i0 = d0 >= 0 ? 0 : -d0, k0 = d0 >= 0 ? d0 : -d0;
        int b = i0 - kAlnW / 2, k = k0;
        int h1[4], h2[4], ra[4], rb[4];
        int e1 = kAlnNeg, e2 = kAlnNeg;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int i = b + 4 * lane + c;
            h1[c] = kAlnNeg; h2[c] = kAlnNeg;
            ra[c] = read_code(s, la, strand, i - 1);
            rb[c] = ref_code(ref, lb, k - i - 1);
        }
        int best = kAlnNeg, bk = 0, bi = 0, bb = 0;     // this lane's best end cell
        uint32_t word = 0, mw = 0;
        int rel = 0;
        for (;; ++rel, ++k) {
            int up1 = __shfl_up_sync(0xffffffffu, h1[3], 1), up2 = __shfl_up_sync(0xffffffffu, h2[3], 1);
            if (lane == 0) { up1 = e1; up2 = e2; }
            int hn[4];
            uint32_t byte = 0;
            bool any = false;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int i = b + 4 * lane + c, j = k - i;
                const int pdiag = c ? h2[c - 1] : up2, pins = c ? h1[c - 1] : up1, pdel = h1[c];
                const bool in = i >= 0 && i <= la && j >= 0 && j <= lb;
                int hv = kAlnNeg;
                uint32_t mv = 3u;
                if (in && (i == 0 || j == 0)) {
                    hv = 0;
                } else if (in) {
                    hv = pdiag + (ra[c] == rb[c] ? MS_ALN_MATCH : MS_ALN_MISMATCH);
                    mv = 0u;
                    if (pins + MS_ALN_GAP > hv) { hv = pins + MS_ALN_GAP; mv = 1u; }
                    if (pdel + MS_ALN_GAP > hv) { hv = pdel + MS_ALN_GAP; mv = 2u; }
                    if (hv < kAlnNeg / 2) hv = kAlnNeg;
                }
                any = any || in;
                if (in && (i == la || j == lb) && hv > best && hv > kAlnNeg / 2) { best = hv; bk = k; bi = i; bb = b; }
                byte |= mv << (2 * c);
                hn[c] = hv;
            }
            word |= byte << (8 * (rel & 3));
            if ((rel & 3) == 3) { my_slab[static_cast<int64_t>(rel >> 2) * 32 + lane] = word; word = 0; }
            if (!__any_sync(0xffffffffu, any)) {
                if ((rel & 3) != 3) my_slab[static_cast<int64_t>(rel >> 2) * 32 + lane] = word;
                if (lane == 0 && (rel & 31) != 31) my_mb[rel >> 5] = mw;
                break;
            }
            const int top = __shfl_sync(0xffffffffu, hn[3], 31), bot = __shfl_sync(0xffffffffu, hn[0], 0);
            const bool down = top > bot;
            if (down) mw |= 1u << ((rel + 1) & 31);
            if (((rel + 1) & 31) == 31) { if (lane == 0) my_mb[(rel + 1) >> 5] = mw; mw = 0; }
            if (down) {
                const int h1lo = __shfl_sync(0xffffffffu, h1[0], 0), hnlo = __shfl_sync(0xffffffffu, hn[0], 0);
                const int h1n = __shfl_down_sync(0xffffffffu, h1[0], 1), hnn = __shfl_down_sync(0xffffffffu, hn[0], 1);
                const int ran = __shfl_down_sync(0xffffffffu, ra[0], 1);
#pragma unroll
                for (int c = 0; c < 3; ++c) { h2[c] = h1[c + 1]; h1[c] = hn[c + 1]; ra[c] = ra[c + 1]; }
                h2[3] = lane == 31 ? kAlnNeg : h1n;
                h1[3] = lane == 31 ? kAlnNeg : hnn;
                ra[3] = lane == 31 ? read_code(s, la, strand, b + kAlnW - 1) : ran;
                e2 = h1lo; e1 = hnlo;
                ++b;
            } else {
                const int rbn = __shfl_up_sync(0xffffffffu, rb[3], 1);
#pragma unroll
                for (int c = 3; c > 0; --c) rb[c] = rb[c - 1];
                rb[0] = lane == 0 ? ref_code(ref, lb, k - b) : rbn;
#pragma unroll
                for (int c = 0; c < 4; ++c) { h2[c] = h1[c]; h1[c] = hn[c]; }
                e2 = e1; e1 = kAlnNeg;
            }
        }
        // the warp's best end cell: highest score, then smallest k, then smallest i
        for (int o = 16; o > 0; o >>= 1) {
            const int s2 = __shfl_xor_sync(0xffffffffu, best, o), k2 = __shfl_xor_sync(0xffffffffu, bk, o);
            const int i2 = __shfl_xor_sync(0xffffffffu, bi, o), b2 = __shfl_xor_sync(0xffffffffu, bb, o);
            if (s2 > best || (s2 == best && (k2 < bk || (k2 == bk && i2 < bi)))) { best = s2; bk = k2; bi = i2; bb = b2; }
        }
        __syncwarp();
        uint32_t* out = cig + slot;
        int nops = 0, run_op = -1;
        uint32_t run = 0;
        auto push = [&](int op, uint32_t len) {
            if (op == run_op) { run += len; return; }
            if (run_op >= 0) { if (lane == 0) out[nops] = run << 4 | static_cast<uint32_t>(run_op); ++nops; }
            run_op = op; run = len;
        };
        if (best > kAlnNeg / 2) {
            if (la - bi > 0) push(4, static_cast<uint32_t>(la - bi));
            int i = bi, kk = bk, band = bb, chunk = -1;
            while (i > 0 && kk - i > 0) {
                const int rl = kk - k0;
                if ((rl >> 5) != chunk) {
                    chunk = rl >> 5;
                    __syncwarp();
                    const uint4* src = reinterpret_cast<const uint4*>(my_slab + static_cast<int64_t>(chunk) * 256);
                    reinterpret_cast<uint4*>(stage[wib])[lane] = src[lane];
                    reinterpret_cast<uint4*>(stage[wib])[lane + 32] = src[lane + 32];
                    __syncwarp();
                }
                const int p = i - band;
                const uint32_t w = stage[wib][((rl & 31) >> 2) * 32 + (p >> 2)];
                const uint32_t mv = (w >> (8 * (rl & 3) + 2 * (p & 3))) & 3u;
                const uint32_t mk = (my_mb[rl >> 5] >> (rl & 31)) & 1u;
                if (mv == 0u) {
                    const uint32_t mk1 = (my_mb[(rl - 1) >> 5] >> ((rl - 1) & 31)) & 1u;
                    const bool eq = read_code(s, la, strand, i - 1) == ref_code(ref, lb, kk - i - 1);
                    push(eq ? 7 : 8, 1);
                    --i; kk -= 2; band -= static_cast<int>(mk + mk1);
                } else if (mv == 1u) {
                    push(1, 1);
                    --i; --kk; band -= static_cast<int>(mk);
                } else {
                    push(2, 1);
                    --kk; band -= static_cast<int>(mk);
                }
            }
            if (i > 0) push(4, static_cast<uint32_t>(i));
            push(-1, 0);
            if (lane == 0) {
                ms_read_alignment o;
                o.mapped = 1; o.strand = strand; o.pos = kk - i; o.score = best; o.cigar_off = slot; o.ncigar = nops;
                res[r] = o;
            }
        } else if (lane == 0) {
            ms_read_alignment o;
            o.mapped = 0; o.strand = 0; o.pos = -1; o.score = 0; o.cigar_off = slot; o.ncigar = 0;
            res[r] = o;
        }
        __syncwarp();
    }
}

// one warp per read: its reversed ops from the slot -> forward order at the packed offset
__global__ void align_cigar_compact_kernel(const uint32_t* __restrict__ cig, const ms_read_alignment* __restrict__ res,
                                           const int64_t* __restrict__ dst_off, int64_t R, uint32_t* __restrict__ dst) {
    const int64_t r = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    const ms_read_alignment a = res[r];
    for (int x = lane; x < a.ncigar; x += 32) dst[dst_off[r] + x] = cig[a.cigar_off + a.ncigar - 1 - x];
}

}  // namespace ms

extern "C" void ms_align_params_default(ms_align_params* p) {
    if (p) p->min_seeds = MS_ALN_MIN_SEEDS;
}

extern "C" int ms_align_set_reference(ms_handle* h, const char* ref, int32_t L) {
    if (!h || L < 0 || (L > 0 && !ref)) return MS_ERR_ARG;
    if (L > MS_ALN_MAX_LEN) MS_FAIL(h, MS_ERR_ARG, "ms_align_set_reference: the reference is longer than 65535 columns");
    MsRange nvtx_range("K6 reference index");
    // every all-ACGT k-mer with its position; keep the ones that occur once
    std::vector<uint64_t> km;
    km.reserve(L);
    for (int32_t t = 0; t + MS_ALN_K <= L; ++t) {
        uint32_t x = 0;
        bool ok = true;
        for (int c = 0; c < MS_ALN_K && ok; ++c) {
            const char b = ref[t + c];
            const int v = b == 'A' ? 0 : b == 'C' ? 1 : b == 'G' ? 2 : b == 'T' ? 3 : -1;
            ok = v >= 0;
            x = (x << 2) | static_cast<uint32_t>(v & 3);
        }
        if (ok) km.push_back(static_cast<uint64_t>(x) << 32 | static_cast<uint32_t>(t));
    }
    std::sort(km.begin(), km.end());
    int bits = 4;
    while ((size_t(1) << bits) < 2 * km.size()) ++bits;
    const uint32_t mask = (1u << bits) - 1u;
    std::vector<uint64_t> tab(size_t(1) << bits, 0);
    for (size_t a = 0; a < km.size();) {
        size_t e = a + 1;
        while (e < km.size() && (km[e] >> 32) == (km[a] >> 32)) ++e;
        if (e == a + 1) {
            const uint32_t kmer = static_cast<uint32_t>(km[a] >> 32);
            uint32_t s = (kmer * 0x9E3779B1u) >> (32 - bits);
            while (tab[s]) s = (s + 1) & mask;
            tab[s] = static_cast<uint64_t>(kmer) << 32 | (static_cast<uint32_t>(km[a]) + 1u);
        }
        a = e;
    }
    MS_CUDA(h, cudaSetDevice(h->device));
    MS_CUDA(h, h->b_aln_ref.ensure(static_cast<size_t>(L) + 16));
    MS_CUDA(h, h->b_aln_idx.ensure(tab.size() * 8));
    if (L) MS_CUDA(h, cudaMemcpyAsync(h->b_aln_ref.p, ref, L, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(h->b_aln_idx.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));     // the host vectors go out of scope
    h->aln_L = L;
    h->aln_bits = bits;
    return MS_OK;
}

extern "C" int ms_align_reads(ms_handle* h, const ms_align_params* prm, const char* seq, const int64_t* off, int64_t R,
                              ms_read_alignment* out, uint32_t* cigar, int64_t cap, int64_t* ncigar) {
    if (!h || !prm || R < 0 || !ncigar || (R > 0 && (!off || !out)) || (cap > 0 && !cigar) || prm->min_seeds < 1) return MS_ERR_ARG;
    if (h->aln_L < 0) MS_FAIL(h, MS_ERR_ARG, "ms_align_reads: no reference (ms_align_set_reference)");
    for (int64_t r = 0; r < R; ++r)
        if (off[r + 1] < off[r] || off[r + 1] - off[r] > MS_ALN_MAX_LEN) MS_FAIL(h, MS_ERR_ARG, "ms_align_reads: read offsets decrease or a read is longer than 65535 bases");
    if (R > 0 && off[R] > off[0] && !seq) return MS_ERR_ARG;
    MsRange nvtx_range("K6 align reads");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int lb = h->aln_L;
    int64_t total = 0;
    std::vector<int64_t> rel, dst;
    for (int64_t r0 = 0; r0 < R;) {
        int64_t r1 = r0 + 1;
        while (r1 < R && r1 - r0 < ms::kAlnChunkReads && off[r1 + 1] - off[r0] <= ms::kAlnChunkBases) ++r1;
        const int64_t Rc = r1 - r0, bases = off[r1] - off[r0];
        int la_max = 0;
        rel.resize(Rc + 1);
        for (int64_t r = r0; r <= r1; ++r) rel[r - r0] = off[r] - off[r0];
        for (int64_t r = r0; r < r1; ++r) la_max = std::max<int>(la_max, static_cast<int>(off[r + 1] - off[r]));
        // seed scratch: one strand's hits per resident warp; slabs: move bits of la + lb + 2 anti-diagonals at most
        const int npos_max = std::max(1, la_max / MS_ALN_STRIDE + 1);
        const int64_t seed_warps = std::min<int64_t>(Rc, static_cast<int64_t>(h->num_sms) * 64);
        const int64_t nad_chunks = (static_cast<int64_t>(la_max) + lb + 2 + 31) / 32;
        const int64_t slab_words = nad_chunks * 256, mbits_words = nad_chunks + 1;
        const int64_t per_warp = (slab_words + mbits_words) * 4;
        int64_t band_warps = std::min<int64_t>(Rc, static_cast<int64_t>(h->num_sms) * 32);   // about what is resident (56 registers)
        band_warps = std::max<int64_t>(1, std::min<int64_t>(band_warps, static_cast<int64_t>(ms::kAlnSlabBudget) / per_warp));
        const int64_t seed_blocks = (seed_warps + ms::kSeedWarps - 1) / ms::kSeedWarps, band_blocks = (band_warps + ms::kBandWarps - 1) / ms::kBandWarps;
        MS_CUDA(h, h->b_aln_seq.ensure(static_cast<size_t>(bases) + 16));
        MS_CUDA(h, h->b_aln_off.ensure(static_cast<size_t>(Rc + 1) * 8));
        MS_CUDA(h, h->b_aln_seed.ensure(static_cast<size_t>(Rc) * sizeof(int4)));
        MS_CUDA(h, h->b_aln_scratch.ensure(static_cast<size_t>(seed_blocks) * ms::kSeedWarps * npos_max * 4));
        MS_CUDA(h, h->b_aln_slab.ensure(static_cast<size_t>(band_blocks) * ms::kBandWarps * slab_words * 4));
        MS_CUDA(h, h->b_aln_mbits.ensure(static_cast<size_t>(band_blocks) * ms::kBandWarps * mbits_words * 4));
        MS_CUDA(h, h->b_aln_cig.ensure(static_cast<size_t>(2 * bases + Rc) * 4));
        MS_CUDA(h, h->b_aln_res.ensure(static_cast<size_t>(Rc) * sizeof(ms_read_alignment)));
        MS_CUDA(h, h->b_aln_ctr.ensure(16));
        if (bases) MS_CUDA(h, cudaMemcpyAsync(h->b_aln_seq.p, seq + off[r0], static_cast<size_t>(bases), cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemcpyAsync(h->b_aln_off.p, rel.data(), static_cast<size_t>(Rc + 1) * 8, cudaMemcpyHostToDevice, h->stream));
        MS_CUDA(h, cudaMemsetAsync(h->b_aln_ctr.p, 0, 16, h->stream));
        const char* d_seq = h->b_aln_seq.as<char>();
        const int64_t* d_off = h->b_aln_off.as<int64_t>();
        MS_STAGE_BEGIN(h, MS_STAGE_ALIGN_SEED);
        ms::align_seed_kernel<<<static_cast<unsigned>(seed_blocks), ms::kSeedWarps * 32, 0, h->stream>>>(
            d_seq, d_off, Rc, h->b_aln_idx.as<unsigned long long>(), h->aln_bits, lb, prm->min_seeds, h->b_aln_scratch.as<int>(), npos_max,
            h->b_aln_ctr.as<int>(), h->b_aln_seed.as<int4>());
        MS_STAGE_END(h, MS_STAGE_ALIGN_SEED);
        h->launches++;
        MS_STAGE_BEGIN(h, MS_STAGE_ALIGN_BAND);
        ms::align_band_kernel<<<static_cast<unsigned>(band_blocks), ms::kBandWarps * 32, 0, h->stream>>>(
            d_seq, d_off, Rc, h->b_aln_ref.as<char>(), lb, h->b_aln_seed.as<int4>(), h->b_aln_slab.as<uint32_t>(), h->b_aln_mbits.as<uint32_t>(),
            slab_words, mbits_words, h->b_aln_ctr.as<int>() + 1, h->b_aln_cig.as<uint32_t>(), h->b_aln_res.as<ms_read_alignment>());
        MS_STAGE_END(h, MS_STAGE_ALIGN_BAND);
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
        MS_CUDA(h, cudaMemcpyAsync(out + r0, h->b_aln_res.p, static_cast<size_t>(Rc) * sizeof(ms_read_alignment), cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
        dst.resize(Rc);
        int64_t n = 0;
        for (int64_t r = 0; r < Rc; ++r) { dst[r] = n; n += out[r0 + r].ncigar; }
        if (total + n <= cap && n > 0) {
            MS_CUDA(h, h->b_aln_dst.ensure(static_cast<size_t>(Rc) * 8));
            MS_CUDA(h, h->b_aln_pack.ensure(static_cast<size_t>(n) * 4));
            MS_CUDA(h, cudaMemcpyAsync(h->b_aln_dst.p, dst.data(), static_cast<size_t>(Rc) * 8, cudaMemcpyHostToDevice, h->stream));
            ms::align_cigar_compact_kernel<<<static_cast<unsigned>((Rc * 32 + 255) / 256), 256, 0, h->stream>>>(
                h->b_aln_cig.as<uint32_t>(), h->b_aln_res.as<ms_read_alignment>(), h->b_aln_dst.as<int64_t>(), Rc, h->b_aln_pack.as<uint32_t>());
            h->launches++;
            MS_CUDA(h, cudaGetLastError());
            MS_CUDA(h, cudaMemcpyAsync(cigar + total, h->b_aln_pack.p, static_cast<size_t>(n) * 4, cudaMemcpyDeviceToHost, h->stream));
            MS_CUDA(h, cudaStreamSynchronize(h->stream));
        }
        for (int64_t r = 0; r < Rc; ++r) out[r0 + r].cigar_off = total + dst[r];
        total += n;
        r0 = r1;
    }
    *ncigar = total;
    return total > cap ? MS_ERR_CAPACITY : MS_OK;
}
