// host_common.hpp -- what juliet and fuse share in front of the C ABI: the BAM loop, the ranks, the checks of the calls.
//
// For every record: admission filter (/root/reference/doc/JULIET.md:58), CIGAR walk into one packed row
// (:49-58, `M` rejected), rich-QV base filter -> 'N' (:256-259,:273-276), optional insertion events (fuse).
#pragma once
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <exception>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>
#include "../../include/minorseq_b200.h"
#include "bgzf_bam.hpp"
#if defined(__has_include)
#if __has_include(<nvtx3/nvToolsExt.h>)
#include <nvtx3/nvToolsExt.h>
#define MSHOST_RANGE(name) mshost::NvtxRange nvtx_range_(name)
namespace mshost { struct NvtxRange { explicit NvtxRange(const char* n) { nvtxRangePushA(n); } ~NvtxRange() { nvtxRangePop(); } }; }
#endif
#endif
#ifndef MSHOST_RANGE
#define MSHOST_RANGE(name) do {} while (0)     // built without the CUDA toolkit's headers: no NVTX ranges on the host stages
#endif

namespace mshost {

struct QvFilter {                      // restatement choice U4: which per-base tracks, which threshold
    std::vector<std::string> tags{"dq", "iq", "sq"};
    int threshold = 20;                // a base whose QV in any present track is below this becomes 'N'; 0 = off

    // mask[i] = 1 for every base of rec (SEQ orientation) whose value in any present per-base track is below the
    // threshold; returns false when no usable track exists (doc/JULIET.md:256-259,273-276: no filter then).  Tracks
    // are stored in native orientation, SEQ in reference orientation.  Works on the raw tag bytes: this runs once per
    // read and track on the decode path, which is what bounds the tools end to end.
    bool apply(const msbam::Record& rec, std::vector<uint8_t>& mask) const {
        if (threshold <= 0) return false;
        const size_t n = rec.seq.size();
        const bool rev = rec.flag & 0x10;
        bool any = false;
        for (const std::string& tg : tags) {
            const uint8_t* t = rec.find_tag(tg.c_str());
            if (!t || n == 0) continue;
            auto track = [&](auto value) {     // value(i) = QV of native base i; branch-free so that the loops vectorise
                if (!any) mask.assign(n, 0);
                any = true;
                uint8_t* m = mask.data();
                const int thr = threshold;
                if (rev) { for (size_t i = 0; i < n; ++i) m[n - 1 - i] |= static_cast<uint8_t>(value(i) < thr); }
                else { for (size_t i = 0; i < n; ++i) m[i] |= static_cast<uint8_t>(value(i) < thr); }
            };
            if (*t == 'Z') {
                const uint8_t* p = t + 1;
                if (strnlen(reinterpret_cast<const char*>(p), n + 1) != n) continue;
                track([&](size_t i) { return static_cast<int>(p[i]) - 33; });
            } else if (*t == 'B') {
                if (msbam::detail::u32(t + 2) != n) continue;
                const uint8_t* p = t + 6;
                switch (t[1]) {
                case 'c': track([&](size_t i) { return static_cast<int>(static_cast<int8_t>(p[i])); }); break;
                case 'C': track([&](size_t i) { return static_cast<int>(p[i]); }); break;
                case 's': track([&](size_t i) { return static_cast<int>(static_cast<int16_t>(msbam::detail::u16(p + 2 * i))); }); break;
                case 'S': track([&](size_t i) { return static_cast<int>(msbam::detail::u16(p + 2 * i)); }); break;
                default: break;
                }
            }
        }
        return any;
    }
};

struct Alignments {
    int32_t L = 0;
    int32_t ref_id = -1;
    std::string ref_name;
    int64_t nreads = 0, nskipped = 0;
    // The reads as EVENT ROWS against `base` (include/minorseq_b200.h, csrc/events.cu): span + event lists per read,
    // ~112 B instead of a 1504-byte plain row per 3 kb read -- what is kept in pinned memory and goes over the PCIe link;
    // the GPU expands them into tiles.  `base` is the configured referenceSequence, or the per-column majority of a sample
    // of the reads (any base is lossless, a close one is short).
    std::vector<uint8_t> base;         // L entries, 0..3
    ms_read_hdr* hdr = nullptr;        // pinned, nreads + 1 entries, sealed
    uint8_t* events = nullptr;         // pinned, ev_bytes
    int64_t ev_bytes = 0;
    std::vector<std::string> names;
    // insertion events (only when want_insertions); ins_read = the index of the event's read (in read order)
    std::vector<int32_t> ins_col, ins_len;
    std::vector<int64_t> ins_off, ins_read;
    std::string ins_pool;
    ~Alignments() { ms_free_pinned(hdr); ms_free_pinned(events); }
};

// The reads [r0, r1) of `a` as a sealed event-row array of their own (one rank's shard): `hdr_out` (pinned, r1 - r0 + 1 entries,
// owned by the caller: ms_free_pinned) with offsets relative to the returned events pointer.
inline const uint8_t* shard_events(const Alignments& a, int64_t r0, int64_t r1, ms_read_hdr** hdr_out) {
    const int64_t n = r1 - r0;
    ms_read_hdr* h = static_cast<ms_read_hdr*>(ms_alloc_pinned(static_cast<size_t>(n + 1) * sizeof(ms_read_hdr)));
    if (!h) throw std::runtime_error("cannot allocate pinned host memory for a shard's read headers");
    const uint32_t e0 = a.hdr[r0].ev_off;
    for (int64_t i = 0; i < n; ++i) { h[i] = a.hdr[r0 + i]; h[i].ev_off -= e0; }
    const int64_t bytes = static_cast<int64_t>(a.hdr[r1].ev_off) - e0;
    if (ms_events_seal(h, n, bytes, a.base.data(), a.L) != MS_OK) { ms_free_pinned(h); throw std::runtime_error("cannot seal a shard's event rows"); }
    *hdr_out = h;
    return a.events + e0;
}

inline void die(const std::string& m) {
    fprintf(stderr, "ERROR: %s\n", m.c_str());
    exit(1);
}

// throws "<what> failed: <the library's message>" unless rc is MS_OK
inline void check(ms_handle* h, int rc, const char* what) {
    if (rc != MS_OK) throw std::runtime_error(std::string(what) + " failed: " + ms_last_error(h));
}
#define CK(h, call) mshost::check((h), (call), #call)

// The list of one of the ABI's list calls: call(out, cap, &n) -> ms_status, first with initial_cap entries, then again with
// cap = n while the list did not fit.  Both conventions of the ABI count as "did not fit": MS_ERR_CAPACITY, and MS_OK with
// n > cap.  Any other failure throws as check() does.
template <class T, class Call>
inline std::vector<T> fetch(ms_handle* h, const char* what, int64_t initial_cap, Call call) {
    std::vector<T> out(static_cast<size_t>(initial_cap));
    int64_t n = 0;
    for (;;) {
        const int rc = call(out.data(), static_cast<int64_t>(out.size()), &n);
        if (rc == MS_ERR_CAPACITY || (rc == MS_OK && n > static_cast<int64_t>(out.size()))) { out.resize(static_cast<size_t>(n)); continue; }
        check(h, rc, what);
        out.resize(static_cast<size_t>(n));
        return out;
    }
}

// "in.bam" of "dir/in.bam": the input's name in the FASTA headers
inline std::string file_name(const std::string& path) { return path.substr(path.find_last_of('/') + 1); }

// rank r's contiguous range [r0, r1) of nreads reads over n ranks
inline std::pair<int64_t, int64_t> shard(int64_t nreads, int r, int n) { return {nreads * r / n, nreads * (r + 1) / n}; }

// f(rank) for rank 0..n-1: on this thread when n == 1, else one thread per rank (one rank per GPU; the ranks meet inside the
// library's collectives, so they have to run concurrently)
template <class F>
inline void run_ranks(int n, F f) {
    if (n <= 1) { f(0); return; }
    std::vector<std::thread> th;
    for (int r = 0; r < n; ++r) th.emplace_back([&f, r] { f(r); });
    for (std::thread& t : th) t.join();
}

// run_ranks where f may throw: a rank's thread must never exit() the process (the other ranks may be inside a collective),
// so each rank's exception is kept, and after the join the first failing rank's (in rank order) is rethrown on this thread
template <class F>
inline void for_ranks(int n, F f) {
    std::vector<std::exception_ptr> errs(static_cast<size_t>(n));
    run_ranks(n, [&](int r) { try { f(r); } catch (...) { errs[r] = std::current_exception(); } });
    for (const std::exception_ptr& e : errs)
        if (e) std::rethrow_exception(e);
}

// One handle per GPU (devices device..device+n-1, one thread each), sharing one NCCL communicator when n > 1.  Dies rather
// than throws: it runs while the BAM decode thread of load_alignments_overlapped is joinable.
inline std::vector<ms_handle*> open_ranks(int device, int n) {
    std::vector<ms_handle*> hs(static_cast<size_t>(n), nullptr);
    char id[128];
    if (n > 1 && ms_comm_unique_id(id) != MS_OK) die("NCCL is not available (libnccl.so.2): --gpus needs it");
    try {
        for_ranks(n, [&](int r) {
            // ms_create's error text is one for all threads, rewritten by each failing create: it is read after the join
            if (ms_create(device + r, &hs[r]) != MS_OK) throw std::runtime_error("");
            if (n > 1 && ms_comm_init(hs[r], id, r, n) != MS_OK) throw std::runtime_error(ms_last_error(hs[r]));
        });
    } catch (const std::exception& e) { die(*e.what() ? e.what() : ms_last_error(nullptr)); }   // there is no CPU path
    return hs;
}

// One record -> one packed row (+ optional insertion events appended to the caller's vectors).
inline void expand_record(const msbam::Record& rec, const QvFilter& qv, int32_t L, uint32_t* row, bool want_insertions,
                          std::vector<uint8_t>& mask, std::vector<int32_t>& ic, std::vector<int64_t>& io, std::vector<int32_t>& il,
                          std::string& pool, std::vector<int32_t>& out_col, std::vector<int32_t>& out_len, std::vector<int64_t>& out_off,
                          std::string& out_pool) {
    const uint8_t* maskp = qv.apply(rec, mask) ? mask.data() : nullptr;   // rich-QV filter
    int64_t ni = 0, pu = 0;
    int rc;
    for (;;) {
        ni = 0; pu = 0;
        rc = ms_expand_cigar(rec.cigar.data(), static_cast<int32_t>(rec.cigar.size()), rec.pos, rec.seq.data(), maskp,
                             static_cast<int32_t>(rec.seq.size()), L, row, want_insertions ? ic.data() : nullptr, io.data(), il.data(),
                             static_cast<int64_t>(ic.size()), &ni, want_insertions ? &pool[0] : nullptr, static_cast<int64_t>(pool.size()), &pu);
        if (rc != MS_ERR_CAPACITY) break;
        ic.resize(ic.size() * 2); io.resize(io.size() * 2); il.resize(il.size() * 2); pool.resize(pool.size() * 2);
    }
    // thrown, not die(): this runs on worker threads (an exit() from there would race the other workers)
    if (rc == MS_ERR_FORMAT) throw std::runtime_error("record " + rec.name + ": BAM files have to be PacBio-compliant, cigar M is forbidden");
    if (rc != MS_OK) throw std::runtime_error("record " + rec.name + ": cannot expand CIGAR");
    for (int64_t i = 0; i < ni; ++i) {
        out_col.push_back(ic[i]);
        out_len.push_back(il[i]);
        out_off.push_back(static_cast<int64_t>(out_pool.size()) + io[i]);
    }
    out_pool.append(pool.data(), static_cast<size_t>(pu));
}

// Whole-file loader in two phases so that the first one (no CUDA involved) can overlap the creation of the
// CUDA context: decode() = parallel BGZF inflate + record index + admission filter; expand() = all host
// threads parse and expand the admitted records straight into one pinned row buffer.
struct Decoded {
    msbam::Bytes u;
    msbam::BamIndexed bx;
    std::vector<size_t> keep;
    unsigned nt = 1;
};

inline void decode_alignments(const std::string& path, Decoded& d, Alignments& out) {
    MSHOST_RANGE("BAM inflate + index + admission");
    unsigned nt = std::thread::hardware_concurrency();
    if (const char* e = getenv("MS_HOST_THREADS")) nt = static_cast<unsigned>(atoi(e));
    if (nt < 1) nt = 1;
    d.nt = nt;
    d.u = msbam::inflate_file(path, nt);
    d.bx = msbam::index_stream(d.u);
    // admission (doc/JULIET.md:58) + one reference per run
    for (size_t i = 0; i < d.bx.records.size(); ++i) {
        const uint8_t* p = d.u.data() + d.bx.records[i].first;
        if (d.bx.records[i].second < 32) throw std::runtime_error("BAM record too small");
        const int32_t ref_id = msbam::detail::i32(p);
        const uint16_t flag = msbam::detail::u16(p + 14);
        if (!ms_read_admitted(flag) || ref_id < 0) { ++out.nskipped; continue; }
        if (out.ref_id < 0) {
            out.ref_id = ref_id;
            if (ref_id >= static_cast<int32_t>(d.bx.refs.size())) throw std::runtime_error("record refers to an unknown reference");
            out.L = d.bx.refs[ref_id].length;
            out.ref_name = d.bx.refs[ref_id].name;
            if (out.L < 3) throw std::runtime_error("reference too short");
        }
        if (ref_id != out.ref_id) { ++out.nskipped; continue; }
        d.keep.push_back(i);
    }
    out.nreads = static_cast<int64_t>(d.keep.size());
}

// refseq: the target configuration's referenceSequence ("" = none): the base the event rows are encoded against
inline void expand_alignments(const Decoded& d, const QvFilter& qv, bool want_names, bool want_insertions, const std::string& refseq,
                              Alignments& out) {
    MSHOST_RANGE("CIGAR expansion + QV filter + event encoding");
    const msbam::Bytes& u = d.u;
    const msbam::BamIndexed& bx = d.bx;
    const std::vector<size_t>& keep = d.keep;
    unsigned nt = d.nt;
    if (keep.empty()) return;
    const int32_t L = out.L;
    const int32_t rw = ms_row_words(L);
    if (L > 65535) throw std::runtime_error("reference longer than 65535 columns: event rows cannot address it");
    if (want_names) out.names.resize(keep.size());
    // ---- the base sequence: the configured reference, else the majority base per column over a sample of the reads
    out.base.assign(static_cast<size_t>(L), 0);
    bool have_base = refseq.size() >= static_cast<size_t>(L);
    for (int32_t c = 0; c < L && have_base; ++c) {
        switch (refseq[c]) {
        case 'A': case 'a': out.base[c] = 0; break;
        case 'C': case 'c': out.base[c] = 1; break;
        case 'G': case 'g': out.base[c] = 2; break;
        case 'T': case 't': out.base[c] = 3; break;
        default: have_base = false;
        }
    }
    if (!have_base) {
        const size_t ns = std::min<size_t>(keep.size(), 256);
        std::vector<uint32_t> votes(static_cast<size_t>(L) * 4, 0u), row(static_cast<size_t>(rw));
        msbam::Record rec;
        std::vector<uint8_t> mask;
        std::vector<int32_t> ic(4096), il(4096), oc, ol;
        std::vector<int64_t> io(4096), oo;
        std::string pool(1 << 16, '\0'), opool;
        for (size_t s = 0; s < ns; ++s) {
            const auto& rr = bx.records[keep[s * keep.size() / ns]];
            msbam::BamReader::parse_record(u.data() + rr.first, rr.second, rec);
            expand_record(rec, qv, L, row.data(), false, mask, ic, io, il, pool, oc, ol, oo, opool);
            for (int32_t c = 0; c < L; ++c) {
                const uint32_t* q = row.data() + 4 * (c >> 5);
                const int sh = c & 31;
                const uint32_t st = ((q[0] >> sh) & 1u) | (((q[1] >> sh) & 1u) << 1) | (((q[2] >> sh) & 1u) << 2);
                if (st < 4) ++votes[static_cast<size_t>(c) * 4 + st];
            }
        }
        for (int32_t c = 0; c < L; ++c) {
            uint32_t best = 0;
            for (uint32_t b = 1; b < 4; ++b)
                if (votes[static_cast<size_t>(c) * 4 + b] > votes[static_cast<size_t>(c) * 4 + best]) best = b;
            out.base[c] = static_cast<uint8_t>(best);
        }
    }
    std::vector<uint32_t> planes(2 * static_cast<size_t>((L + 31) / 32));
    if (ms_base_planes(out.base.data(), L, planes.data()) != MS_OK) throw std::runtime_error("ms_base_planes failed");
    // ---- every thread expands and encodes its contiguous range of the reads into buffers of its own
    struct Part {
        std::vector<int32_t> col, len; std::vector<int64_t> off, read; std::string pool;
        std::vector<ms_read_hdr> hdr; std::vector<uint8_t> ev; int64_t nbytes = 0;
    };
    nt = static_cast<unsigned>(std::min<size_t>(nt, keep.size()));
    std::vector<Part> parts(nt);
    const int64_t bound = ms_events_bound(L);
    for_ranks(static_cast<int>(nt), [&](int t) {      // a corrupt record throws on its worker: carried to the caller after the join
        const size_t i0 = keep.size() * t / nt, i1 = keep.size() * (t + 1) / nt;
        Part& P = parts[t];
        P.hdr.resize(i1 - i0);
        P.ev.resize(static_cast<size_t>(std::max<int64_t>(bound, static_cast<int64_t>(i1 - i0) * 192)));
        msbam::Record rec;
        std::vector<uint8_t> mask;
        std::vector<uint32_t> row(static_cast<size_t>(rw));
        std::vector<int32_t> ic(4096), il(4096);
        std::vector<int64_t> io(4096);
        std::string pool(1 << 16, '\0');
        for (size_t k = i0; k < i1; ++k) {
            const auto& rr = bx.records[keep[k]];
            msbam::BamReader::parse_record(u.data() + rr.first, rr.second, rec);
            expand_record(rec, qv, L, row.data(), want_insertions, mask, ic, io, il, pool, P.col, P.len, P.off, P.pool);
            P.read.resize(P.col.size(), static_cast<int64_t>(k));
            if (static_cast<int64_t>(P.ev.size()) - P.nbytes < bound) P.ev.resize(P.ev.size() * 2 + static_cast<size_t>(bound));
            if (ms_encode_row(row.data(), L, planes.data(), &P.hdr[k - i0], P.ev.data(), static_cast<int64_t>(P.ev.size()), &P.nbytes) != MS_OK)
                throw std::runtime_error("record " + rec.name + ": cannot encode the expanded row");
            if (want_names) out.names[k] = rec.name;
        }
    });
    // ---- one pinned header array and one pinned event array; the threads copy their parts into place
    std::vector<int64_t> ev0(nt + 1, 0);
    for (unsigned t = 0; t < nt; ++t) ev0[t + 1] = ev0[t] + parts[t].nbytes;
    out.ev_bytes = ev0[nt];
    if (out.ev_bytes > 0xffffffffLL) throw std::runtime_error("more than 4 GB of event rows in one run: split the input");
    out.hdr = static_cast<ms_read_hdr*>(ms_alloc_pinned((keep.size() + 1) * sizeof(ms_read_hdr)));
    out.events = static_cast<uint8_t*>(ms_alloc_pinned(static_cast<size_t>(out.ev_bytes) + 64));
    if (!out.hdr || !out.events) throw std::runtime_error("cannot allocate pinned host memory for the event rows");
    run_ranks(static_cast<int>(nt), [&](int t) {
        const size_t i0 = keep.size() * t / nt;
        const Part& P = parts[t];
        for (size_t k = 0; k < P.hdr.size(); ++k) {
            ms_read_hdr hd = P.hdr[k];
            hd.ev_off += static_cast<uint32_t>(ev0[t]);
            out.hdr[i0 + k] = hd;
        }
        if (P.nbytes) memcpy(out.events + ev0[t], P.ev.data(), static_cast<size_t>(P.nbytes));
    });
    if (ms_events_seal(out.hdr, static_cast<int64_t>(keep.size()), out.ev_bytes, out.base.data(), L) != MS_OK)
        throw std::runtime_error("ms_events_seal failed");
    for (const Part& p : parts) {   // read order is preserved: thread t holds a contiguous range
        const int64_t base = static_cast<int64_t>(out.ins_pool.size());
        out.ins_col.insert(out.ins_col.end(), p.col.begin(), p.col.end());
        out.ins_len.insert(out.ins_len.end(), p.len.begin(), p.len.end());
        out.ins_read.insert(out.ins_read.end(), p.read.begin(), p.read.end());
        for (int64_t o : p.off) out.ins_off.push_back(base + o);
        out.ins_pool += p.pool;
    }
}

// decode on a helper thread while the caller brings up the CUDA context, then expand
template <class CreateFn>
inline void load_alignments_overlapped(const std::string& path, const QvFilter& qv, bool want_names, bool want_insertions, const std::string& refseq,
                                       Alignments& out, CreateFn create_context) {
    Decoded d;
    std::string err;
    if (getenv("MS_SERIAL_LOAD")) {   // A/B switch for the overlap (tools/from_bam_timing.py)
        create_context();
        decode_alignments(path, d, out);
        expand_alignments(d, qv, want_names, want_insertions, refseq, out);
        return;
    }
    std::thread dec([&] { try { decode_alignments(path, d, out); } catch (const std::exception& e) { err = e.what(); } });
    create_context();      // dies with the CUDA error when there is no usable GPU: that message wins
    dec.join();
    if (!err.empty()) throw std::runtime_error(err);
    expand_alignments(d, qv, want_names, want_insertions, refseq, out);
}

// Rank r of n piles up its shard of the reads (event rows, ~112 B instead of 1504 B per 3 kb read on the link, expanded into
// tiles on the GPU) and all-reduces the counts; returns the rank's reads on its GPU (tiles, owned by the handle).
inline const uint32_t* pileup_shard(ms_handle* h, const Alignments& a, int r, int n) {
    const std::pair<int64_t, int64_t> s = shard(a.nreads, r, n);
    ms_read_hdr* hdr = a.hdr;
    const uint8_t* ev = a.events;
    if (n > 1) ev = shard_events(a, s.first, s.second, &hdr);
    const uint32_t* rows = nullptr;
    const int rc = ms_pileup_events_host(h, hdr, ev, s.second - s.first, &rows);
    if (n > 1) {
        if (rc == MS_OK) ms_synchronize(h);     // the shard's header copy is ours to free once the upload is done
        ms_free_pinned(hdr);
    }
    check(h, rc, "ms_pileup_events_host");
    CK(h, ms_allreduce_counts(h));
    CK(h, ms_synchronize(h));
    return rows;
}

}  // namespace mshost
