// phase_indel.cu -- in-frame indel keys in the phasing bit-vectors (restatement choice U20, DESIGN.md "Phasing indels").
//
// ms_phase_begin_indels puts the reported codon deletions and insertions after the V substitution keys:
//   deletion key s (bit V + k):        B = '-' at s, s+1, s+2;  M = B, or all three columns A/C/G/T;
//   insertion key (c, x) (bit V+ndel+i): M = c and c+1 both A/C/G/T;  B = M and the read's first insertion event at c is x.
// A read is damaged when some key is not informative (M = 0); the columns that make it so give the categories ('-' gaps,
// QV-filtered N heteroduplex, not spanned partial).  The columns of every deletion key are left out of phase_bits_kernel's
// damage mask (`cover`): its substitution bits do not depend on it, and the deletion key judges those columns here, so a read
// that carries the deletion in full is not damaged by them.
//
// phase_indel_kernel runs after phase_bits_kernel on the same reads: one lane per read, the touched 32-column blocks staged
// with 16-byte cp.async as in phase_bits_kernel, per key a 3- or 2-column window of the three state planes (the next block for
// windows that start at column 30 or 31).  It ORs B (deletions) and M into the lane's own rows, ORs the new damage into
// flags[r] and counts only the reads and categories that change.  phase_indel_ins_kernel then sets the insertion bits, one
// thread per kept insertion event of ms_indel_count_dev.
#include <algorithm>
#include <vector>
#include "phase_internal.cuh"
#include "rows.cuh"

namespace ms {

constexpr int kIndelWarps = 8;
constexpr int kIndelChunk = 8;   // distinct blocks staged at a time (+1: the second block of a window that crosses the last one)

// key words: [ column in the block (5 bits) | insertion << 5 | slot in the block list << 6 ], then the key's bit index
template <bool kClean>
__global__ void __launch_bounds__(kIndelWarps * 32) phase_indel_kernel(
    const uint4* __restrict__ packed, int64_t R, int32_t nblk, const int32_t* __restrict__ blocklist, int32_t NB, int32_t chunk,
    const uint32_t* __restrict__ keys, int32_t nkeys, int32_t vwords, uint32_t* __restrict__ bits, uint32_t* __restrict__ mbits,
    uint8_t* __restrict__ flags, unsigned long long* __restrict__ ctr) {
    extern __shared__ __align__(16) uint4 stage_sm[];   // [warp][chunk + 1][32]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint4* const sm = stage_sm + static_cast<size_t>(warp) * (chunk + 1) * 32 + lane;
    const int64_t nwarps = static_cast<int64_t>(gridDim.x) * kIndelWarps;
    unsigned long long c_dam = 0, c_gap = 0, c_het = 0, c_par = 0;
    for (int64_t base = (static_cast<int64_t>(blockIdx.x) * kIndelWarps + warp) * 32; base < R; base += nwarps * 32) {
        const int64_t r = base + lane;
        const bool live = r < R;
        const uint4* tile = packed + static_cast<size_t>(r >> 3) * nblk * 8;
        const uint32_t pos = static_cast<uint32_t>(r & 7);
        uint32_t fg = 0, fh = 0, fp = 0;
        uint32_t word = 0, mword = 0, widx = 0xffffffffu;
        uint32_t* myrow = bits + static_cast<size_t>(r) * vwords;
        uint32_t* mrow = kClean ? mbits + static_cast<size_t>(r) * vwords : nullptr;
        auto flush = [&]() {      // the words were written by phase_bits_kernel: OR the indel bits in
            if (word) myrow[widx] |= word;
            if constexpr (kClean) { if (mword) mrow[widx] |= mword; }
        };
        int32_t s0 = 0, ns = 0;   // staged: slots [s0, s0 + ns)
        for (int32_t k = 0; k < nkeys; ++k) {
            const uint32_t w0 = keys[2 * k], bit = keys[2 * k + 1];
            const int32_t slot = static_cast<int32_t>(w0 >> 6);
            const uint32_t j = w0 & 31u, ins = (w0 >> 5) & 1u;
            const int32_t last = slot + static_cast<int32_t>((j + (ins ? 1u : 2u)) >> 5);   // the window's last block
            if (slot < s0 || last >= s0 + ns) {     // warp-uniform: every lane walks the same keys
                __syncwarp();
                s0 = slot;
                ns = min(chunk + 1, NB - slot);
                for (int32_t t = 0; t < ns; ++t) {
                    const int32_t blk = blocklist[s0 + t];
                    const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(sm + t * 32));
                    const uint4* src = tile + (blk * 8 + (pos ^ (blk & 7)));
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(live ? src : packed), "r"(live ? 16 : 0) : "memory");
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
                asm volatile("cp.async.wait_group 0;" ::: "memory");
                __syncwarp();
            }
            const uint4 q = sm[(slot - s0) * 32];
            const uint4 nx = last > slot ? sm[(slot - s0 + 1) * 32] : q;     // only read by windows that cross the block
            const uint32_t msk = ins ? 3u : 7u;
            const uint32_t wx = __funnelshift_r(q.x, nx.x, j), wy = __funnelshift_r(q.y, nx.y, j), wz = __funnelshift_r(q.z, nx.z, j);
            const uint32_t gap = wz & ~wx & ~wy & msk;     // 100  '-'
            const uint32_t het = wz & wx & ~wy & msk;      // 101  QV-filtered base
            const uint32_t par = wz & wy & msk;            // 11x  not spanned
            const uint32_t b = (!ins && gap == 7u) ? 1u : 0u;
            const uint32_t m = (b || (wz & msk) == 0u) ? 1u : 0u;
            if (!m) { fg |= gap; fh |= het; fp |= par; }
            if ((bit >> 5) != widx) {
                if (live && widx != 0xffffffffu) flush();
                widx = bit >> 5; word = 0; mword = 0;
            }
            word |= b << (bit & 31u);
            if constexpr (kClean) mword |= m << (bit & 31u);
        }
        if (live) {
            if (widx != 0xffffffffu) flush();
            const uint32_t old = flags[r];
            const uint32_t f = old | (fg ? MS_FLAG_GAP : 0) | (fh ? MS_FLAG_HET : 0) | (fp ? MS_FLAG_PARTIAL : 0);
            if (f != old) {
                flags[r] = static_cast<uint8_t>(f);
                const uint32_t nw = f & ~old;
                if (!old) ++c_dam;
                if (nw & MS_FLAG_GAP) ++c_gap;
                if (nw & MS_FLAG_HET) ++c_het;
                if (nw & MS_FLAG_PARTIAL) ++c_par;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        c_dam += __shfl_xor_sync(0xffffffffu, c_dam, o);
        c_gap += __shfl_xor_sync(0xffffffffu, c_gap, o);
        c_het += __shfl_xor_sync(0xffffffffu, c_het, o);
        c_par += __shfl_xor_sync(0xffffffffu, c_par, o);
    }
    if (lane == 0) {
        if (c_dam) atomicAdd(ctr + 0, c_dam);
        if (c_gap) atomicAdd(ctr + 1, c_gap);
        if (c_het) atomicAdd(ctr + 2, c_het);
        if (c_par) atomicAdd(ctr + 3, c_par);
    }
}

// one thread per kept insertion event (local read, c, sid) of ms_indel_count_dev (the first event of its read at c, in frame,
// A/C/G/T): the read carries the key of sid when it is clean at c and c+1.  Keys of one word may be set by several events.
__global__ void phase_indel_ins_kernel(const uint4* __restrict__ packed, int32_t nblk, const int32_t* __restrict__ ev, int64_t n,
                                       const int32_t* __restrict__ sid_bit, int32_t nsid, int32_t vwords, uint32_t* __restrict__ bits) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t r = ev[3 * i], c = ev[3 * i + 1], sid = ev[3 * i + 2];
    const int32_t k = sid < nsid ? sid_bit[sid] : -1;
    if (k < 0) return;
    const uint32_t p0 = packed[tile_slot(r, c >> 5, nblk)].z, p1 = packed[tile_slot(r, (c + 1) >> 5, nblk)].z;
    if (!((p0 >> (c & 31)) & 1u) && !((p1 >> ((c + 1) & 31)) & 1u))
        atomicOr(bits + static_cast<size_t>(r) * vwords + (k >> 5), 1u << (k & 31));
}

int phase_indel_dev(ms_handle* h, const uint4* packed, int64_t R, uint32_t* bits, uint32_t* mbits, uint8_t* flags) {
    if (R == 0) return MS_OK;
    MsRange nvtx_range("K3 indel keys");
    const int chunk = std::min(kIndelChunk, h->pi_nblk);
    const size_t smem = static_cast<size_t>(kIndelWarps) * (chunk + 1) * 32 * sizeof(uint4);
    const int64_t want = (R + kIndelWarps * 32 - 1) / (kIndelWarps * 32);
    const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(want, static_cast<int64_t>(h->num_sms) * 6)));
    const int32_t* bl = h->b_pi_blocks.as<int32_t>();
    const uint32_t* keys = h->b_pi_keys.as<uint32_t>();
    if (mbits)
        phase_indel_kernel<true><<<grid, kIndelWarps * 32, smem, h->stream>>>(packed, R, h->nblk, bl, h->pi_nblk, chunk, keys, h->pi_nkeys,
                                                                              h->vwords, bits, mbits, flags, phase_ctr(h));
    else
        phase_indel_kernel<false><<<grid, kIndelWarps * 32, smem, h->stream>>>(packed, R, h->nblk, bl, h->pi_nblk, chunk, keys, h->pi_nkeys,
                                                                               h->vwords, bits, nullptr, flags, phase_ctr(h));
    h->launches++;
    MS_CUDA(h, cudaGetLastError());
    const int32_t nsid = static_cast<int32_t>(h->indel_col.size());
    if (h->indel_nev > 0 && nsid > 0) {
        phase_indel_ins_kernel<<<static_cast<unsigned>((h->indel_nev + 255) / 256), 256, 0, h->stream>>>(
            packed, h->nblk, h->b_indel_ev.as<int32_t>(), h->indel_nev, h->b_pi_sid.as<int32_t>(), nsid, h->vwords, bits);
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
    }
    return MS_OK;
}

}  // namespace ms

extern "C" {

int ms_phase_begin_indels(ms_handle* h, const int32_t* var_col, const int32_t* var_codon, int32_t V, const int32_t* del_col, int32_t ndel,
                          const int32_t* ins_sid, int32_t nins, int64_t max_reads) {
    if (!h || ndel < 0 || nins < 0 || (ndel > 0 && !del_col) || (nins > 0 && !ins_sid)) return MS_ERR_ARG;
    if (ndel == 0 && nins == 0) return ms_phase_begin(h, var_col, var_codon, V, max_reads);
    if (h->L <= 0 || h->indel_L != h->L) MS_FAIL(h, MS_ERR_ARG, "ms_phase_begin_indels: no indel counts (ms_indel_count_dev)");
    if (V < 0 || V > INT32_MAX - ndel - nins) return MS_ERR_ARG;
    const int32_t L = h->L, nsid = static_cast<int32_t>(h->indel_col.size());
    // the keys' columns (deletions: s; insertions: c), checked; the deletion columns leave phase_bits_kernel's damage mask
    std::vector<int32_t> kcol(static_cast<size_t>(ndel + nins));
    std::vector<uint32_t> exclude(static_cast<size_t>(h->nblk), 0u);
    std::vector<int32_t> sid_bit(static_cast<size_t>(std::max(1, nsid)), -1);
    for (int32_t k = 0; k < ndel; ++k) {
        const int32_t s = del_col[k];
        if (s < 0 || s + 2 >= L) MS_FAIL(h, MS_ERR_ARG, "ms_phase_begin_indels: deletion column outside the reference");
        for (int32_t c = s; c < s + 3; ++c) exclude[c >> 5] |= 1u << (c & 31);
        kcol[k] = s;
    }
    for (int32_t i = 0; i < nins; ++i) {
        const int32_t sid = ins_sid[i];
        if (sid < 0 || sid >= nsid) MS_FAIL(h, MS_ERR_ARG, "ms_phase_begin_indels: no such insertion string id");
        if (sid_bit[sid] >= 0) MS_FAIL(h, MS_ERR_ARG, "ms_phase_begin_indels: insertion string id given twice");
        sid_bit[sid] = V + ndel + i;
        kcol[ndel + i] = h->indel_col[sid];
    }
    {
        std::vector<int32_t> d(del_col, del_col + ndel);
        std::sort(d.begin(), d.end());
        if (std::adjacent_find(d.begin(), d.end()) != d.end()) MS_FAIL(h, MS_ERR_ARG, "ms_phase_begin_indels: deletion column given twice");
    }
    int rc = ms::phase_begin_keys(h, var_col, var_codon, V, kcol.data(), ndel + nins, exclude, max_reads);
    if (rc != MS_OK) return rc;
    // the indel kernel's block list and key words, keys in bit order
    std::vector<int32_t> blocks;
    for (int32_t k = 0; k < ndel + nins; ++k) {
        const int32_t c = kcol[k], span = k < ndel ? 2 : 1;
        blocks.push_back(c >> 5);
        blocks.push_back((c + span) >> 5);
    }
    std::sort(blocks.begin(), blocks.end());
    blocks.erase(std::unique(blocks.begin(), blocks.end()), blocks.end());
    std::vector<uint32_t> kw;
    for (int32_t k = 0; k < ndel + nins; ++k) {
        const int32_t c = kcol[k];
        const uint32_t slot = static_cast<uint32_t>(std::lower_bound(blocks.begin(), blocks.end(), c >> 5) - blocks.begin());
        kw.push_back(static_cast<uint32_t>(c & 31) | (k < ndel ? 0u : 32u) | (slot << 6));
        kw.push_back(static_cast<uint32_t>(V + k));
    }
    if (kw.size() * 4 > h->b_pi_keys.cap || blocks.size() * 4 > h->b_pi_blocks.cap || sid_bit.size() * 4 > h->b_pi_sid.cap)
        MS_CUDA(h, cudaStreamSynchronize(h->stream));   // the previous pass may still read the buffers that move
    MS_CUDA(h, h->b_pi_keys.ensure(kw.size() * 4));
    MS_CUDA(h, h->b_pi_blocks.ensure(blocks.size() * 4));
    MS_CUDA(h, h->b_pi_sid.ensure(sid_bit.size() * 4));
    MS_CUDA(h, cudaMemcpyAsync(h->b_pi_keys.p, kw.data(), kw.size() * 4, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(h->b_pi_blocks.p, blocks.data(), blocks.size() * 4, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(h->b_pi_sid.p, sid_bit.data(), sid_bit.size() * 4, cudaMemcpyHostToDevice, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));       // the sources are pageable host vectors
    h->pi_nkeys = ndel + nins;
    h->pi_nblk = static_cast<int32_t>(blocks.size());
    return MS_OK;
}

}  // extern "C"
