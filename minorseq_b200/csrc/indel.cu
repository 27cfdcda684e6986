// indel.cu -- in-frame codon deletions and insertions (restatement choice U19, DESIGN.md "In-frame indels").
//
// K2 tests substitutions only: a read with '-' in a codon, or with an insertion between two codons, never reaches its codon
// histogram.  This pass counts them per read, joint over the columns involved:
//   k_del[s] = reads with '-' at s, s+1 and s+2;
//   n_ins[c] = reads whose states at c and c+1 are both A/C/G/T;
//   tally[x] = those reads of n_ins[c] whose first insertion event at c is the in-frame A/C/G/T string x (one id per
//              (column, upper-cased string)).
// indel_count_kernel forms the two masks from each 32-column block and the next one and adds them into K1's carry-save
// counters through the grouped pile-up's walk (group.cuh); it counts every column, the call reads codon starts and
// boundaries only.  indel_ins_kernel checks the two columns of each candidate event in the tiles.  The test is K2's
// (U1-U3): e = min(n, ceil(n P)), the one-sided Fisher test of [[k, n-k], [e, n-e]], called iff p * ntests < alpha; for a
// deletion n = k_del + K2's coverage (the reads with a clean codon at s, the sum of K1's codon histogram).
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include "fisher_core.h"
#include "group.cuh"
#include "handle.h"
#include "rows.cuh"

namespace ms {

struct IndelCountArgs {
    const uint4* tiles;
    uint32_t* cnt;     // [L][2]: k_del, n_ins
    int64_t R;
    int32_t L, nblk, nseg, seg_len;
};

// end of a work item: planes [2][kPlanes] -> per-column integers, added into cnt[32 * b + j][0..1] with RED
__device__ __noinline__ void indel_flush(const uint32_t* planes, uint32_t* dst, int ncols) {
    uint32_t tr[2][16];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
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
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const uint32_t c = half ? (tr[i][j] >> 16) : (tr[i][j] & 0xffffu);
                if (c) atomicAdd(dst + colj * 2 + i, c);
            }
        }
    }
}

// the walk's policy: the reads in order, one chunk of kGroupChunk per work item; blocks b and b+1 of each read
struct IndelPolicy {
    static constexpr int NM = 2, SLOTS = 2;
    IndelCountArgs a;
    __device__ __forceinline__ int32_t item(int32_t k, int32_t& r_begin, int32_t& r_end) const {
        r_begin = k * kGroupChunk;
        r_end = static_cast<int32_t>(min(a.R, static_cast<int64_t>(r_begin) + kGroupChunk));
        return 0;
    }
    __device__ __forceinline__ int64_t read(int32_t idx) const { return idx; }
    // m[0]: '-' at j, j+1, j+2 (state 4 = P2 & ~P1 & ~P0); m[1]: A/C/G/T (~P2) at j and j+1.  Block b+1 supplies the
    // neighbours past bit 31; beyond the last block it reads as "not spanned".
    __device__ static __forceinline__ void masks(uint32_t addr, uint32_t stride, uint32_t (&m)[NM]) {
        const uint4 x = lds128g(addr), y = lds128g(addr + stride);
        const uint32_t gx = x.z & ~x.y & ~x.x, gy = y.z & ~y.y & ~y.x;
        m[0] = gx & ((gx >> 1) | (gy << 31)) & ((gx >> 2) | (gy << 30));
        const uint32_t cx = ~x.z, cy = ~y.z;
        m[1] = cx & ((cx >> 1) | (cy << 31));
    }
    __device__ __forceinline__ void flush(const uint32_t* planes, uint32_t, int32_t, int b) const {
        indel_flush(planes, a.cnt + static_cast<size_t>(b) * 32 * 2, min(32, a.L - b * 32));
    }
};

__global__ void __launch_bounds__(kGroupMaxThreads) indel_count_kernel(IndelCountArgs a) {
    csa_walk(IndelPolicy{a}, a.tiles, a.nblk, a.nseg, a.seg_len, (a.R + kGroupChunk - 1) / kGroupChunk * a.nseg);
}

// one thread per candidate insertion event (read, column c, string id): the read counts for its string when it is clean at
// c and c+1 (c+1 < L: c is a boundary)
__global__ void indel_ins_kernel(const uint4* __restrict__ tiles, int32_t nblk, const int32_t* __restrict__ ev, int64_t n,
                                 uint32_t* __restrict__ tally) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t r = ev[3 * i], c = ev[3 * i + 1], sid = ev[3 * i + 2];
    const uint32_t p0 = tiles[tile_slot(r, c >> 5, nblk)].z, p1 = tiles[tile_slot(r, (c + 1) >> 5, nblk)].z;
    if (!((p0 >> (c & 31)) & 1u) && !((p1 >> ((c + 1) & 31)) & 1u)) atomicAdd(tally + sid, 1u);
}

struct IndelCand {
    double P;                               // error probability of the event: deletion_rate^3 or insertion_rate^len
    int32_t gene, codon_index, col, kind, sid;
    int32_t ref0, ref1;                     // referenceSequence codons at s (and s+3 for an insertion); < 0: majority codon
    uint32_t ntests;
};

struct IndelConst {
    double alpha, min_perc, max_perc;
};

// the majority codon of a start column, lowest index on ties (U6); -1 when no read is clean there
__device__ int32_t major_codon(const uint32_t* h) {
    uint32_t bc = 0;
    int32_t bi = -1;
    for (int c = 0; c < 64; ++c)
        if (h[c] > bc) { bc = h[c]; bi = c; }
    return bi;
}

// one thread per candidate: K2's test on its (k, n), compacted output
__global__ void indel_test_kernel(const uint32_t* __restrict__ codon, const uint32_t* __restrict__ cnt, const uint32_t* __restrict__ tally,
                                  const IndelCand* __restrict__ cand, int64_t ncand, IndelConst cc, ms_indel* __restrict__ out,
                                  unsigned long long* __restrict__ nout) {
    const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= ncand) return;
    const IndelCand cd = cand[i];
    const int32_t s = cd.kind == MS_INDEL_DELETION ? cd.col : cd.col - 2;
    uint32_t k, n;
    if (cd.kind == MS_INDEL_DELETION) {
        k = cnt[2 * static_cast<size_t>(s)];
        uint32_t cov = 0;
        for (int c = 0; c < 64; ++c) cov += codon[static_cast<size_t>(s) * 64 + c];
        n = k + cov;
    } else {
        k = tally[cd.sid];
        n = cnt[2 * static_cast<size_t>(cd.col) + 1];
    }
    if (k == 0 || n == 0) return;
    const double ex = ceil(static_cast<double>(n) * cd.P);
    const uint32_t e = ex >= static_cast<double>(n) ? n : static_cast<uint32_t>(ex);
    if (k <= e && 0.5 * static_cast<double>(cd.ntests) >= cc.alpha) return;   // p >= 1/2 (call.cu)
    const double p = fisher_upper(k, n - k, e, n - e, 1.000001 * cc.alpha / static_cast<double>(cd.ntests));
    if (!(p * static_cast<double>(cd.ntests) < cc.alpha)) return;
    const double perc = 100.0 * static_cast<double>(k) / static_cast<double>(n);
    if (cc.min_perc >= 0.0 && !(perc > cc.min_perc)) return;
    if (cc.max_perc >= 0.0 && !(perc < cc.max_perc)) return;
    ms_indel v;
    v.gene = cd.gene; v.codon_index = cd.codon_index; v.col = cd.col; v.kind = cd.kind; v.sid = cd.sid;
    v.ref_codon = cd.ref0 >= 0 ? cd.ref0 : major_codon(codon + static_cast<size_t>(s) * 64);
    v.next_codon = cd.kind == MS_INDEL_DELETION ? -1 : (cd.ref1 >= 0 ? cd.ref1 : major_codon(codon + static_cast<size_t>(s + 3) * 64));
    v.count = k; v.coverage = n; v.expected = e; v.ntests = cd.ntests; v.pvalue = p;
    out[atomicAdd(nout, 1ULL)] = v;   // at most one record per candidate: the buffer holds ncand
}

static int base_code(char ch) {
    switch (ch) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return -1;
    }
}

static int ref_codon_at(const char* refseq, size_t reflen, int32_t s) {
    if (static_cast<size_t>(s) + 3 > reflen) return -1;
    const int b0 = base_code(refseq[s]), b1 = base_code(refseq[s + 1]), b2 = base_code(refseq[s + 2]);
    return (b0 >= 0 && b1 >= 0 && b2 >= 0) ? 16 * b0 + 4 * b1 + b2 : -1;
}

}  // namespace ms

int ms_comm_allreduce_u32(ms_handle* h, uint32_t* d, size_t count);   // comm.cu

namespace {

bool start_bit(const ms_handle* h, int32_t s) { return s >= 0 && s < h->L && ((h->h_start[s >> 5] >> (s & 31)) & 1u); }

}  // namespace

// the walk stages blocks b and b+1 of 8 reads per ring slot: up to 192 KB of dynamic shared memory
void ms_indel_set_smem_attr() {
    cudaFuncSetAttribute(ms::indel_count_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         ms::kGroupRing * 8 * 2 * ms::kGroupMaxThreads * 16);
}

extern "C" {

void ms_indel_params_default(ms_indel_params* p) {
    if (!p) return;
    p->deletion_rate = 3e-3; p->insertion_rate = 3e-3; p->alpha = 0.01;
    p->min_perc = -1.0; p->max_perc = -1.0; p->region_begin = 0; p->region_end = 0;
}

int ms_indel_count_dev(ms_handle* h, const uint32_t* d_packed, int64_t R, int64_t read0, const int64_t* ins_read, const int32_t* ins_col,
                       const int64_t* ins_off, const int32_t* ins_len, int64_t nins, const char* ins_pool, int64_t pool_len) {
    MsRange nvtx_range("indel counts");
    if (!h || R < 0 || read0 < 0 || nins < 0 || pool_len < 0 || (R > 0 && !d_packed) ||
        (nins > 0 && (!ins_read || !ins_col || !ins_off || !ins_len || !ins_pool)))
        return MS_ERR_ARG;
    if (!h->count_codons) MS_FAIL(h, MS_ERR_ARG, "ms_indel_count_dev: ms_set_layout was called without a codon start mask");
    if (R > INT32_MAX) MS_FAIL(h, MS_ERR_ARG, "ms_indel_count_dev: more than 2^31 - 1 reads in one call");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t L = h->L;
    // string ids over ALL events (every rank passes the same list and gets the same ids): events at a boundary c (c - 2 and
    // c + 1 codon starts), the first event of each (read, c) deciding, kept when its string is in frame and all A/C/G/T
    std::map<std::pair<int64_t, int32_t>, int64_t> first;   // (read, c) -> its first event
    for (int64_t i = 0; i < nins; ++i) {
        if (ins_off[i] < 0 || ins_len[i] < 0 || ins_off[i] + ins_len[i] > pool_len || ins_read[i] < 0)
            MS_FAIL(h, MS_ERR_ARG, "ms_indel_count_dev: insertion event outside the pool");
        const int32_t c = ins_col[i];
        if (!start_bit(h, c - 2) || !start_bit(h, c + 1)) continue;
        first.emplace(std::make_pair(ins_read[i], c), i);
    }
    std::map<std::pair<int32_t, std::string>, int32_t> ids;
    std::vector<std::pair<int64_t, std::pair<int32_t, std::string>>> kept;   // (read, (c, x))
    for (const auto& f : first) {
        const int64_t i = f.second;
        const int32_t len = ins_len[i];
        if (len < 3 || len % 3) continue;
        std::string x(ins_pool + ins_off[i], static_cast<size_t>(len));
        bool ok = true;
        for (char& ch : x) {
            const int b = ms::base_code(ch);
            if (b < 0) { ok = false; break; }
            ch = "ACGT"[b];
        }
        if (!ok) continue;
        ids.emplace(std::make_pair(ins_col[i], x), 0);
        kept.emplace_back(f.first.first, std::make_pair(ins_col[i], x));
    }
    h->indel_col.clear();
    h->indel_str.clear();
    for (auto& e : ids) {
        e.second = static_cast<int32_t>(h->indel_col.size());
        h->indel_col.push_back(e.first.first);
        h->indel_str.push_back(e.first.second);
    }
    const int64_t nsid = static_cast<int64_t>(h->indel_col.size());
    std::vector<int32_t> ev;   // this rank's events: (local read, c, sid)
    for (const auto& k : kept)
        if (k.first >= read0 && k.first < read0 + R)
            ev.insert(ev.end(), {static_cast<int32_t>(k.first - read0), k.second.first, ids[k.second]});
    const int64_t nev = static_cast<int64_t>(ev.size() / 3);
    const size_t words = static_cast<size_t>(L) * 2 + static_cast<size_t>(nsid);
    MS_CUDA(h, h->b_indel_cnt.ensure(words * 4));
    MS_CUDA(h, h->b_indel_ev.ensure(std::max<size_t>(4, ev.size() * 4)));
    uint32_t* cnt = h->b_indel_cnt.as<uint32_t>();
    MS_CUDA(h, cudaMemsetAsync(cnt, 0, words * 4, h->stream));
    h->indel_L = L;
    h->indel_reduced = false;
    if (R > 0) {
        ms::IndelCountArgs a;
        a.tiles = reinterpret_cast<const uint4*>(d_packed);
        a.cnt = cnt;
        a.R = R;
        a.L = L;
        a.nblk = h->nblk;
        a.nseg = (h->nblk + ms::kGroupMaxThreads - 1) / ms::kGroupMaxThreads;
        a.seg_len = (h->nblk + a.nseg - 1) / a.nseg;
        const int threads = (a.seg_len + 31) / 32 * 32;
        const int smem = ms::kGroupRing * 8 * 2 * threads * 16;
        int per_sm = 0;
        MS_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ms::indel_count_kernel, threads, smem));
        const int64_t items = (R + ms::kGroupChunk - 1) / ms::kGroupChunk * a.nseg;
        const int grid = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(items, static_cast<int64_t>(std::max(1, per_sm)) * h->num_sms)));
        MS_STAGE_BEGIN(h, MS_STAGE_INDELS);
        ms::indel_count_kernel<<<grid, threads, smem, h->stream>>>(a);
        MS_STAGE_END(h, MS_STAGE_INDELS);
        h->launches++;
        MS_CUDA(h, cudaGetLastError());
        if (nev > 0) {
            MS_CUDA(h, cudaMemcpyAsync(h->b_indel_ev.p, ev.data(), ev.size() * 4, cudaMemcpyHostToDevice, h->stream));
            ms::indel_ins_kernel<<<static_cast<unsigned>((nev + 255) / 256), 256, 0, h->stream>>>(
                a.tiles, h->nblk, h->b_indel_ev.as<int32_t>(), nev, cnt + static_cast<size_t>(L) * 2);
            h->launches++;
            MS_CUDA(h, cudaGetLastError());
            MS_CUDA(h, cudaStreamSynchronize(h->stream));   // the event list is pageable host memory
        }
    }
    return MS_OK;
}

int ms_indel_counts(ms_handle* h, uint32_t* cnt, uint32_t* tally, int64_t cap, int64_t* nstrings) {
    if (!h || !cnt || !nstrings || cap < 0 || (cap > 0 && !tally)) return MS_ERR_ARG;
    if (h->indel_L != h->L || h->L <= 0) MS_FAIL(h, MS_ERR_ARG, "ms_indel_counts: no indel counts (ms_indel_count_dev)");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int64_t nsid = static_cast<int64_t>(h->indel_col.size());
    *nstrings = nsid;
    const uint32_t* d = h->b_indel_cnt.as<uint32_t>();
    MS_CUDA(h, cudaMemcpyAsync(cnt, d, static_cast<size_t>(h->L) * 2 * 4, cudaMemcpyDeviceToHost, h->stream));
    const int64_t k = std::min(cap, nsid);
    if (k > 0) MS_CUDA(h, cudaMemcpyAsync(tally, d + static_cast<size_t>(h->L) * 2, static_cast<size_t>(k) * 4, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    return MS_OK;
}

int ms_indel_inserted(ms_handle* h, int32_t sid, int32_t* col, char* buf, int64_t cap, int64_t* len) {
    if (!h || !len || cap < 0 || (cap > 0 && !buf)) return MS_ERR_ARG;
    if (sid < 0 || static_cast<size_t>(sid) >= h->indel_str.size()) MS_FAIL(h, MS_ERR_ARG, "ms_indel_inserted: no such string id");
    const std::string& x = h->indel_str[sid];
    *len = static_cast<int64_t>(x.size());
    if (col) *col = h->indel_col[sid];
    if (cap < *len) MS_FAIL(h, MS_ERR_CAPACITY, "ms_indel_inserted: buffer too small (*len)");
    memcpy(buf, x.data(), x.size());
    return MS_OK;
}

int ms_indel_call(ms_handle* h, const ms_gene* genes, int32_t ngenes, const char* refseq, const ms_indel_params* prm, ms_indel* out,
                  int64_t cap, int64_t* n) {
    MsRange nvtx_range("indel call");
    if (!h || !genes || ngenes < 0 || !prm || !n || cap < 0 || (cap > 0 && !out)) return MS_ERR_ARG;
    *n = 0;
    if (h->indel_L != h->L || h->L <= 0 || !h->d_counts) MS_FAIL(h, MS_ERR_ARG, "ms_indel_call: no indel counts (ms_indel_count_dev)");
    MS_CUDA(h, cudaSetDevice(h->device));
    const int32_t L = h->L;
    const int64_t nsid = static_cast<int64_t>(h->indel_col.size());
    uint32_t* cnt = h->b_indel_cnt.as<uint32_t>();
    if (!h->indel_reduced) {
        // one sum of [L][2] | tally over the ranks (every rank holds the same string ids); once per ms_indel_count_dev
        if (h->comm) {
            const int rc = ms_comm_allreduce_u32(h, cnt, static_cast<size_t>(L) * 2 + static_cast<size_t>(nsid));
            if (rc != MS_OK) return rc;
        }
        h->indel_reduced = true;
    }
    const size_t reflen = refseq ? strnlen(refseq, static_cast<size_t>(L)) : 0;
    int32_t lo = 0, hi = L;
    if (prm->region_end > prm->region_begin) {
        lo = std::max(0, prm->region_begin - 1);
        hi = std::min(L, prm->region_end - 1);
    }
    // the string ids of each column, in (column, string) order
    std::vector<int32_t> sid_lo(static_cast<size_t>(L) + 1, 0);
    for (int32_t c : h->indel_col) ++sid_lo[c + 1];
    for (int32_t j = 0; j < L; ++j) sid_lo[j + 1] += sid_lo[j];
    double Pdel = 1.0;
    for (int i = 0; i < 3; ++i) Pdel *= prm->deletion_rate;
    std::vector<ms::IndelCand> cand;
    for (int32_t g = 0; g < ngenes; ++g) {
        const int32_t gb = genes[g].begin - 1, ge = std::min(genes[g].end - 1, L);
        const size_t first = cand.size();
        uint32_t nt = 0;
        for (int32_t s = gb, ci = 0; s + 3 <= ge; s += 3, ++ci) {
            if (!(s >= lo && s + 3 <= hi && s >= 0)) continue;
            if (!start_bit(h, s)) MS_FAIL(h, MS_ERR_ARG, "gene codon start not in the layout's start mask");
            ++nt;
            ms::IndelCand d;
            d.gene = g; d.codon_index = ci; d.col = s; d.kind = MS_INDEL_DELETION; d.sid = -1; d.P = Pdel; d.ntests = 0;
            d.ref0 = ms::ref_codon_at(refseq, reflen, s); d.ref1 = -1;
            cand.push_back(d);
            // the boundary after this codon, when the next codon of the gene is tested too
            const int32_t c = s + 2, t = s + 3;
            if (!(t + 3 <= ge && t + 3 <= hi)) continue;
            for (int32_t id = sid_lo[c]; id < sid_lo[c + 1]; ++id) {
                ms::IndelCand x = d;
                x.col = c; x.kind = MS_INDEL_INSERTION; x.sid = id;
                x.P = 1.0;
                for (size_t q = 0; q < h->indel_str[id].size(); ++q) x.P *= prm->insertion_rate;
                x.ref1 = ms::ref_codon_at(refseq, reflen, t);
                cand.push_back(x);
            }
        }
        for (size_t i = first; i < cand.size(); ++i) cand[i].ntests = nt;
    }
    const int64_t ncand = static_cast<int64_t>(cand.size());
    if (ncand == 0) return MS_OK;
    const size_t need = 64 + ncand * (sizeof(ms_indel) + sizeof(ms::IndelCand));
    MS_CUDA(h, h->b_indel_out.ensure(need));
    uint8_t* base = h->b_indel_out.as<uint8_t>();
    unsigned long long* d_n = reinterpret_cast<unsigned long long*>(base);
    ms_indel* d_out = reinterpret_cast<ms_indel*>(base + 64);
    ms::IndelCand* d_cand = reinterpret_cast<ms::IndelCand*>(base + 64 + ncand * sizeof(ms_indel));
    MS_CUDA(h, cudaMemsetAsync(d_n, 0, 8, h->stream));
    MS_CUDA(h, cudaMemcpyAsync(d_cand, cand.data(), ncand * sizeof(ms::IndelCand), cudaMemcpyHostToDevice, h->stream));
    ms::IndelConst cc;
    cc.alpha = prm->alpha; cc.min_perc = prm->min_perc; cc.max_perc = prm->max_perc;
    ms::indel_test_kernel<<<static_cast<unsigned>((ncand + 127) / 128), 128, 0, h->stream>>>(
        h->d_counts + static_cast<size_t>(L) * 8, cnt, cnt + static_cast<size_t>(L) * 2, d_cand, ncand, cc, d_out, d_n);
    h->launches++;
    MS_CUDA(h, cudaGetLastError());
    unsigned long long cnt_out = 0;
    MS_CUDA(h, cudaMemcpyAsync(&cnt_out, d_n, 8, cudaMemcpyDeviceToHost, h->stream));
    MS_CUDA(h, cudaStreamSynchronize(h->stream));
    std::vector<ms_indel> v(cnt_out);
    if (cnt_out) {
        MS_CUDA(h, cudaMemcpyAsync(v.data(), d_out, cnt_out * sizeof(ms_indel), cudaMemcpyDeviceToHost, h->stream));
        MS_CUDA(h, cudaStreamSynchronize(h->stream));
    }
    // (gene, codon, deletion before insertion, string): the string ids of a column are in string order
    std::sort(v.begin(), v.end(), [](const ms_indel& a, const ms_indel& b) {
        if (a.gene != b.gene) return a.gene < b.gene;
        if (a.codon_index != b.codon_index) return a.codon_index < b.codon_index;
        if (a.kind != b.kind) return a.kind < b.kind;
        return a.sid < b.sid;
    });
    *n = static_cast<int64_t>(cnt_out);
    for (int64_t i = 0; i < std::min<int64_t>(cap, *n); ++i) out[i] = v[i];
    if (*n > cap) MS_FAIL(h, MS_ERR_CAPACITY, "ms_indel_call: out holds fewer records than were called (*n)");
    return MS_OK;
}

}  // extern "C"
