// align_main.cpp -- `align [--device n] [--min-seeds n] <reads.bam> <reference.fasta> <out.bam>`: overlap-align unaligned CCS
// reads to one amplicon reference on the GPU (K6, restatement choice U16) and write a BAM that juliet, fuse and cleric
// accept as it is (= X I D S CIGARs).  Secondary (0x100) and supplementary (0x800) records are dropped, every other record
// is written in input order, mapped or not.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <sstream>
#include <string>
#include <thread>
#include <vector>
#include "cleric.hpp"
#include "host_common.hpp"

#define CK(h, call)                                                                            \
    do {                                                                                       \
        int rc_ = (call);                                                                      \
        if (rc_ != MS_OK) mshost::die(std::string(#call) + " failed: " + ms_last_error(h));     \
    } while (0)

// IUPAC complement (the codes a BAM SEQ can hold: =ACMGRSVTWYHKDBN), so a stored-reverse record keeps every code
static char complement(char c) {
    switch (c) {
    case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A';
    case 'M': return 'K'; case 'K': return 'M'; case 'R': return 'Y'; case 'Y': return 'R';
    case 'V': return 'B'; case 'B': return 'V'; case 'H': return 'D'; case 'D': return 'H';
    default: return c;   // = S W N
    }
}
static std::string revcomp(const std::string& s) {
    std::string r(s.rbegin(), s.rend());
    for (char& c : r) c = complement(c);
    return r;
}

int main(int argc, char** argv) {
    int device = 0;
    ms_align_params prm;
    ms_align_params_default(&prm);
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        if (a == "-h" || a == "--help") {
            puts("Usage: align [--device n] [--min-seeds n] <reads.bam> <reference.fasta> <out.bam>");
            return 0;
        } else if (a == "--version") { puts("minorseq_b200 align 0.1.0 (B200-native overlap aligner, restatement choice U16)"); return 0; }
        else if (a == "--device") { if (i + 1 >= argc) mshost::die("option --device needs a value"); device = atoi(argv[++i]); }
        else if (a == "--min-seeds") {
            if (i + 1 >= argc) mshost::die("option --min-seeds needs a value");
            prm.min_seeds = atoi(argv[++i]);
            if (prm.min_seeds < 1) mshost::die("--min-seeds must be at least 1");
        } else if (!a.empty() && a[0] == '-') mshost::die("unknown option " + a);
        else pos.push_back(a);
    }
    if (pos.size() != 3) { puts("Usage: align [--device n] [--min-seeds n] <reads.bam> <reference.fasta> <out.bam>"); return 1; }
    try {
        unsigned nt = std::thread::hardware_concurrency();
        if (const char* e = getenv("MS_HOST_THREADS")) nt = static_cast<unsigned>(atoi(e));
        nt = std::max(1u, nt);
        msbam::Bytes stream;
        msbam::BamIndexed in;
        std::string read_err;
        std::thread reader([&] {
            try { stream = msbam::inflate_file(pos[0], nt); in = msbam::index_stream(stream); } catch (const std::exception& e) { read_err = e.what(); }
        });
        ms_handle* h = nullptr;
        const int create_rc = ms_create(device, &h);   // the alignment runs on the GPU; there is no CPU path
        reader.join();
        if (create_rc != MS_OK) mshost::die(ms_last_error(nullptr));
        if (!read_err.empty()) mshost::die(read_err);
        const std::vector<mscleric::Fasta> fa = mscleric::read_fasta(pos[1]);
        if (fa.size() != 1) mshost::die(pos[1] + ": the reference must hold exactly one sequence");
        const mscleric::Fasta& ref = fa[0];
        if (ref.seq.size() > 65535) mshost::die(pos[1] + ": references longer than 65535 bases are not supported");

        // records in input order, and the native orientation of every kept read
        std::vector<msbam::Record> recs(in.records.size());
        std::vector<std::string> native(recs.size());
        nt = std::max(1u, std::min<unsigned>(nt, static_cast<unsigned>(recs.size() / 256 + 1)));
        std::atomic<int> bad{0};
        std::string bad_msg;
        auto parse = [&](unsigned t) { try {
            for (size_t k = recs.size() * t / nt; k < recs.size() * (t + 1) / nt; ++k) {
                msbam::Record& r = recs[k];
                msbam::BamReader::parse_record(stream.data() + in.records[k].first, in.records[k].second, r);
                if (r.flag & 0x900) continue;
                if (r.seq.size() > 65535 && !bad.exchange(1)) bad_msg = r.name + ": reads longer than 65535 bases are not supported";
                native[k] = (r.flag & 0x10) ? revcomp(r.seq) : r.seq;
                if (r.flag & 0x10) std::reverse(r.qual.begin(), r.qual.end());
            }
        } catch (const std::exception& e) {
            if (!bad.exchange(2)) bad_msg = e.what();
        } };
        {
            std::vector<std::thread> th;
            for (unsigned t = 0; t < nt; ++t) th.emplace_back(parse, t);
            for (auto& x : th) x.join();
        }
        if (bad) mshost::die(bad_msg);
        std::vector<size_t> kept;
        std::string seq;
        std::vector<int64_t> off(1, 0);
        for (size_t k = 0; k < recs.size(); ++k) {
            if (recs[k].flag & 0x900) continue;
            kept.push_back(k);
            seq += native[k];
            off.push_back(static_cast<int64_t>(seq.size()));
        }
        const int64_t R = static_cast<int64_t>(kept.size());
        CK(h, ms_align_set_reference(h, ref.seq.data(), static_cast<int32_t>(ref.seq.size())));
        std::vector<ms_read_alignment> aln(static_cast<size_t>(R));
        std::vector<uint32_t> cig(static_cast<size_t>(R) * 16 + 16);
        int64_t ncig = 0;
        int rc = ms_align_reads(h, &prm, seq.data(), off.data(), R, aln.data(), cig.data(), static_cast<int64_t>(cig.size()), &ncig);
        if (rc == MS_ERR_CAPACITY) {
            cig.resize(static_cast<size_t>(ncig));
            rc = ms_align_reads(h, &prm, seq.data(), off.data(), R, aln.data(), cig.data(), ncig, &ncig);
        }
        if (rc != MS_OK) mshost::die(std::string("ms_align_reads failed: ") + ms_last_error(h));

        int64_t n_fwd = 0, n_rev = 0, n_un = 0;
        for (int64_t x = 0; x < R; ++x) {
            msbam::Record& r = recs[kept[x]];
            const ms_read_alignment& a = aln[x];
            msbam::strip_tags(r.aux, {"NM", "MD", "AS"});    // they describe an earlier alignment
            r.next_ref_id = -1; r.next_pos = -1; r.tlen = 0;
            if (a.mapped) {
                r.flag = static_cast<uint16_t>((r.flag & ~0x14) | (a.strand ? 0x10 : 0));
                r.ref_id = 0; r.pos = a.pos; r.mapq = 60;
                r.cigar.assign(cig.begin() + a.cigar_off, cig.begin() + a.cigar_off + a.ncigar);
                if (a.strand) { r.seq = revcomp(native[kept[x]]); std::reverse(r.qual.begin(), r.qual.end()); }
                else r.seq = native[kept[x]];
                const uint32_t as = static_cast<uint32_t>(a.score);
                const uint8_t tag[7] = {'A', 'S', 'i', static_cast<uint8_t>(as), static_cast<uint8_t>(as >> 8), static_cast<uint8_t>(as >> 16),
                                        static_cast<uint8_t>(as >> 24)};
                r.aux.insert(r.aux.end(), tag, tag + 7);
                ++(a.strand ? n_rev : n_fwd);
            } else {
                r.flag = static_cast<uint16_t>((r.flag & ~0x10) | 0x4);
                r.ref_id = -1; r.pos = -1; r.mapq = 0; r.cigar.clear();
                r.seq = native[kept[x]];
                ++n_un;
            }
        }

        // header: the input's, with the @SQ lines replaced by the reference, SO:unknown, and an @PG line for this step
        std::string text;
        {
            std::istringstream hs(in.text);
            std::string line;
            bool sq_done = false, hd = false;
            std::vector<std::string> pg_ids;   // an earlier align step keeps its @PG line; this one gets a fresh ID
            const std::string sq = "@SQ\tSN:" + ref.name + "\tLN:" + std::to_string(ref.seq.size()) + "\n";
            while (std::getline(hs, line)) {
                if (line.compare(0, 3, "@SQ") == 0) {
                    if (!sq_done) text += sq;
                    sq_done = true;
                } else if (line.compare(0, 3, "@HD") == 0) {
                    hd = true;
                    const size_t so = line.find("\tSO:");
                    if (so == std::string::npos) line += "\tSO:unknown";
                    else {
                        const size_t e = line.find('\t', so + 1);
                        line = line.substr(0, so) + "\tSO:unknown" + (e == std::string::npos ? "" : line.substr(e));
                    }
                    text += line + "\n";
                } else if (!line.empty()) {
                    if (line.compare(0, 3, "@PG") == 0) {
                        const size_t id = line.find("\tID:");
                        if (id != std::string::npos) pg_ids.push_back(line.substr(id + 4, line.find('\t', id + 1) - id - 4));
                    }
                    text += line + "\n";
                }
            }
            if (!sq_done) text += sq;
            if (!hd) text = "@HD\tVN:1.6\tSO:unknown\n" + text;
            std::string id = "align";
            for (int n = 1; std::find(pg_ids.begin(), pg_ids.end(), id) != pg_ids.end(); ++n) id = "align." + std::to_string(n);
            text += "@PG\tID:" + id + "\tPN:align\tVN:minorseq_b200-0.1.0";
            if (!pg_ids.empty()) text += "\tPP:" + pg_ids.back();
            text += "\n";
        }
        std::vector<const msbam::Record*> out;
        out.reserve(kept.size());
        for (size_t k : kept) out.push_back(&recs[k]);
        msbam::write_bam_parallel(pos[2], text, {{ref.name, static_cast<int32_t>(ref.seq.size())}}, out, nt);
        fprintf(stderr, "align: %lld mapped forward, %lld mapped reverse, %lld unmapped, %lld secondary/supplementary dropped (reference %s, %zu bases)\n",
                static_cast<long long>(n_fwd), static_cast<long long>(n_rev), static_cast<long long>(n_un),
                static_cast<long long>(recs.size() - kept.size()), ref.name.c_str(), ref.seq.size());
        ms_destroy(h);
    } catch (const std::exception& e) {
        mshost::die(e.what());
    }
    return 0;
}
