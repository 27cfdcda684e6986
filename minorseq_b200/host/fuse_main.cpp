// fuse_main.cpp -- `fuse in.bam out.fasta` on top of the C ABI (/root/reference/doc/FUSE.md:17-32):
// consensus of an alignment, in-frame insertions at a distance from each other included, major deletions
// removed, one FASTA record per input.  The thresholds are the restatement's choices U6-U8 (options).
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <string>
#include <vector>
#include <unistd.h>
#include "host_common.hpp"

int main(int argc, char** argv) {
    ms_fuse_params prm;
    ms_fuse_params_default(&prm);
    int device = 0, ngpus = 1;
    mshost::QvFilter qv;
    qv.threshold = 0;  // fuse takes every base
    std::vector<std::string> pos;
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto need = [&](const char* name) -> std::string {
            if (i + 1 >= argc) mshost::die(std::string("option ") + name + " needs a value");
            return argv[++i];
        };
        if (a == "-h" || a == "--help") {
            puts("Usage: fuse [--min-coverage n] [--ins-fraction f] [--ins-distance d] [--device n] [--gpus n] <in.bam> <out.fasta>\n"
                 "  --gpus n: shard the reads over n GPUs (devices n0..n0+n-1), one NCCL all-reduce of the column counts");
            return 0;
        } else if (a == "--version") { puts("minorseq_b200 fuse 0.1.0 (B200-native restatement; not PacBio fuse)"); return 0; }
        else if (a == "--min-coverage") prm.min_coverage = atoi(need("--min-coverage").c_str());
        else if (a == "--ins-fraction") prm.ins_fraction = atof(need("--ins-fraction").c_str());
        else if (a == "--ins-distance") prm.ins_distance = atoi(need("--ins-distance").c_str());
        else if (a == "--device") device = atoi(need("--device").c_str());
        else if (a == "--gpus") ngpus = atoi(need("--gpus").c_str());
        else if (!a.empty() && a[0] == '-') mshost::die("unknown option " + a);
        else pos.push_back(a);
    }
    if (pos.size() != 2) { puts("Usage: fuse <in.bam> <out.fasta>"); return 1; }
    if (ngpus < 1 || ngpus > 64) mshost::die("--gpus expects 1..64");
    try {
        // the CUDA contexts come up (~0.5 s, one thread per GPU) while a helper thread inflates and indexes the BAM
        std::vector<ms_handle*> hs;
        mshost::Alignments aln;
        mshost::load_alignments_overlapped(pos[0], qv, false, true, std::string(), aln, [&] { hs = mshost::open_ranks(device, ngpus); });
        if (aln.nreads == 0) mshost::die("no primary or supplementary alignments in " + pos[0]);
        // every rank piles up its contiguous range of the reads; the all-reduce leaves the column counts of all reads on rank 0
        mshost::for_ranks(ngpus, [&](int r) {
            CK(hs[r], ms_set_layout(hs[r], aln.L, nullptr));
            CK(hs[r], ms_set_base(hs[r], aln.base.data()));   // the reads as event rows (base = majority of a sample of them)
            mshost::pileup_shard(hs[r], aln, r, ngpus);
        });
        ms_handle* h = hs[0];
        std::string seq(static_cast<size_t>(aln.L) + aln.ins_pool.size() + 16, '\0');
        int64_t len = 0;
        CK(h, ms_fuse(h, &prm, aln.ins_col.data(), aln.ins_off.data(), aln.ins_len.data(), static_cast<int64_t>(aln.ins_col.size()),
                      aln.ins_pool.data(), static_cast<int64_t>(aln.ins_pool.size()), &seq[0], static_cast<int64_t>(seq.size()), &len));
        seq.resize(static_cast<size_t>(len));
        std::ofstream f(pos[1]);
        if (!f) mshost::die("cannot write " + pos[1]);
        f << ">" << mshost::file_name(pos[0]) << "|fuse|" << aln.ref_name << "\n";
        for (size_t i = 0; i < seq.size(); i += 70) f << seq.substr(i, 70) << "\n";
        fprintf(stderr, "fuse: %lld reads, consensus length %lld\n", static_cast<long long>(aln.nreads), static_cast<long long>(len));
        f.close();
        fflush(nullptr);
        if (!getenv("MS_FULL_TEARDOWN")) _exit(0);
        for (ms_handle* x : hs) ms_destroy(x);
    } catch (const std::exception& e) {
        mshost::die(e.what());
    }
    return 0;
}
