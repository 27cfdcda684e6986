// cleric_main.cpp -- `cleric in.bam reference.fasta new_ref.fasta out.bam` / `cleric in.bam combined.fasta out.bam`
// (/root/reference/doc/CLERIC.md:27-38): swap the reference of a BAM alignment.  The two references are aligned on the
// GPU (ms_align_refs, Needleman-Wunsch, N x M -- doc/CLERIC.md:41-44), every record is then re-expressed through that
// alignment on the host threads.  "The header of the original reference must match the reference name in the BAM"
// (doc/CLERIC.md:16-17); cigar M is refused (:14-15).
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <sstream>
#include <string>
#include <thread>
#include <vector>
#include "cleric.hpp"
#include "host_common.hpp"

int main(int argc, char** argv) {
    int device = 0;
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        if (a == "-h" || a == "--help") {
            puts("Usage: cleric [--device n] <in.bam> <reference.fasta> <new_ref.fasta> <out.bam>\n"
                 "       cleric [--device n] <in.bam> <combined.fasta> <out.bam>");
            return 0;
        } else if (a == "--version") { puts("minorseq_b200 cleric 0.1.0 (B200-native restatement; not PacBio cleric)"); return 0; }
        else if (a == "--device") { if (i + 1 >= argc) mshost::die("option --device needs a value"); device = atoi(argv[++i]); }
        else if (!a.empty() && a[0] == '-') mshost::die("unknown option " + a);
        else pos.push_back(a);
    }
    if (pos.size() != 3 && pos.size() != 4) { puts("Usage: cleric <in.bam> <reference.fasta> <new_ref.fasta> <out.bam>"); return 1; }
    try {
        unsigned nt = std::thread::hardware_concurrency();
        if (const char* e = getenv("MS_HOST_THREADS")) nt = static_cast<unsigned>(atoi(e));
        nt = std::max(1u, nt);
        // whole file: parallel BGZF inflate + record index on a helper thread while the CUDA context comes up
        msbam::Bytes stream;
        msbam::BamIndexed in;
        std::string read_err;
        std::thread reader([&] {
            try { stream = msbam::inflate_file(pos[0], nt); in = msbam::index_stream(stream); } catch (const std::exception& e) { read_err = e.what(); }
        });
        ms_handle* h = nullptr;
        const int create_rc = ms_create(device, &h);   // the alignment step runs on the GPU; there is no CPU path
        reader.join();
        if (create_rc != MS_OK) mshost::die(ms_last_error(nullptr));
        if (!read_err.empty()) mshost::die(read_err);
        std::vector<mscleric::Fasta> fa = mscleric::read_fasta(pos[1]);
        if (pos.size() == 4) {
            std::vector<mscleric::Fasta> fb = mscleric::read_fasta(pos[2]);
            fa.insert(fa.end(), fb.begin(), fb.end());
        }
        if (fa.size() != 2) mshost::die("two sequences have to be provided, either in individual files or combined in one");
        // the original reference is the one the BAM names
        int orig = -1, ref_id = -1;
        for (size_t r = 0; r < in.refs.size() && orig < 0; ++r)
            for (int k = 0; k < 2; ++k)
                if (in.refs[r].name == fa[k].name) { orig = k; ref_id = static_cast<int>(r); break; }
        if (orig < 0) mshost::die("the header of the original reference must match the reference name in the BAM");
        const mscleric::Fasta &A = fa[orig], &B = fa[1 - orig];
        if (static_cast<int64_t>(A.seq.size()) != in.refs[ref_id].length) mshost::die("the original reference's length differs from the BAM header's");
        std::string ops(A.seq.size() + B.seq.size() + 1, '\0');
        int64_t nops = 0, score = 0;
        CK(h, ms_align_refs(h, A.seq.data(), static_cast<int32_t>(A.seq.size()), B.seq.data(), static_cast<int32_t>(B.seq.size()), &ops[0],
                            static_cast<int64_t>(ops.size()), &nops, &score));
        ops.resize(static_cast<size_t>(nops));
        const mscleric::Path path(ops);

        std::vector<msbam::Record> recs(in.records.size());
        nt = std::max(1u, std::min<unsigned>(nt, static_cast<unsigned>(recs.size() / 256 + 1)));
        std::atomic<int64_t> n_ok{0}, n_unmapped{0}, n_other{0};
        std::atomic<int> bad{0};
        std::string bad_name;
        auto work = [&](unsigned t) { try {
            for (size_t k = recs.size() * t / nt; k < recs.size() * (t + 1) / nt; ++k) {
                msbam::Record& r = recs[k];
                msbam::BamReader::parse_record(stream.data() + in.records[k].first, in.records[k].second, r);
                if (r.ref_id < 0 || (r.flag & 0x4)) continue;                     // unmapped records pass through
                if (r.ref_id != ref_id) { ++n_other; r.ref_id = -2; continue; }   // aligned to something else: dropped
                switch (mscleric::project_read(path, B.seq, r)) {
                case mscleric::Projected::Ok:
                    r.ref_id = 0; ++n_ok;
                    msbam::strip_tags(r.aux, {"NM", "MD"});                      // they describe the alignment to the old reference
                    if (r.next_ref_id >= 0) { r.next_ref_id = -1; r.next_pos = -1; r.tlen = 0; }   // a mate's old coordinates mean nothing here
                    break;
                case mscleric::Projected::Unmapped:
                    r.ref_id = -1; r.pos = -1; r.cigar.clear(); r.flag |= 0x4; r.mapq = 0; ++n_unmapped;
                    msbam::strip_tags(r.aux, {"NM", "MD"});
                    break;
                case mscleric::Projected::Unsupported:
                    if (!bad.exchange(1)) bad_name = r.name + ": CIGAR ops other than = X I D S H are not supported (cigar M is forbidden)";
                    break;
                case mscleric::Projected::Inconsistent:
                    if (!bad.exchange(2)) bad_name = r.name + ": CIGAR, sequence and reference length disagree";
                    break;
                }
            }
        } catch (const std::exception& e) {     // a corrupt record: reported after the join, not std::terminate on this thread
            if (!bad.exchange(3)) bad_name = e.what();
        } };
        std::vector<std::thread> th;
        for (unsigned t = 0; t < nt; ++t) th.emplace_back(work, t);
        for (auto& x : th) x.join();
        if (bad) mshost::die(bad_name);

        // header: every @SQ line gives way to the target reference; a sort order survives only when no record lost its place
        // (the projection is monotone in POS, but a record that became unmapped now sits between placed ones); the rest is kept
        std::string text;
        {
            std::istringstream hs(in.text);
            std::string line;
            bool sq_done = false;
            while (std::getline(hs, line)) {
                if (line.compare(0, 3, "@SQ") == 0) {
                    if (!sq_done) text += "@SQ\tSN:" + B.name + "\tLN:" + std::to_string(B.seq.size()) + "\n";
                    sq_done = true;
                } else if (line.compare(0, 3, "@HD") == 0 && n_unmapped.load() > 0) {
                    const size_t so = line.find("\tSO:");
                    if (so != std::string::npos) {
                        const size_t e = line.find('\t', so + 1);
                        line = line.substr(0, so) + "\tSO:unknown" + (e == std::string::npos ? "" : line.substr(e));
                    }
                    text += line + "\n";
                } else if (!line.empty()) text += line + "\n";
            }
            if (!sq_done) text += "@SQ\tSN:" + B.name + "\tLN:" + std::to_string(B.seq.size()) + "\n";
            text += "@PG\tID:cleric\tPN:cleric\tVN:minorseq_b200-0.1.0\n";
        }
        {
            std::vector<const msbam::Record*> keep;
            for (const msbam::Record& r : recs)
                if (r.ref_id != -2) keep.push_back(&r);
            msbam::write_bam_parallel(pos.back(), text, {{B.name, static_cast<int32_t>(B.seq.size())}}, keep, nt);
        }
        fprintf(stderr, "cleric: %lld records re-expressed against %s (alignment score %lld), %lld became unmapped, %lld on other references dropped\n",
                static_cast<long long>(n_ok.load()), B.name.c_str(), static_cast<long long>(score), static_cast<long long>(n_unmapped.load()),
                static_cast<long long>(n_other.load()));
        ms_destroy(h);
    } catch (const std::exception& e) {
        mshost::die(e.what());
    }
    return 0;
}
