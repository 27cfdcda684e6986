// juliet_main.cpp -- `juliet [options] in.bam out.json|out.html ...` on top of the C ABI.
//
// Keeps the reference's process interface (/root/reference/doc/JULIET.md): outputs chosen by file
// extension, either or both (:61-66); --config/-c <HIV|ABL1|file.json> (:118-162); --region b-e (:270-271);
// --mode-phasing (:192-211); --min-perc / --max-perc (:342-354); --drm-only (:370).  The unpinned model
// constants (SURVEY App. B) are options with the restatement's defaults.  --linkage adds pairwise variant linkage
// (restatement choice U14): per pair of called variants, the reads clean at both codons, D', r^2 and two Fisher tests.
// A third output kind, out.fasta (with --mode-phasing), holds the consensus sequence of every reported haplotype (restatement
// choice U15): a grouped pile-up of each haplotype's reads on the GPU and fuse's column rule with thin columns written as 'N'.
// --haplotype-abundance (restatement choice U18) fits every phased read, damaged ones included, to the reported haplotypes and
// estimates their frequencies by EM over the reads' compatibility sets.  --indels (restatement choice U19) tests in-frame codon
// deletions and insertions between codons with K2's model and reports them in an "indels" block.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <ctime>
#include <fstream>
#include <map>
#include <string>
#include <thread>
#include <vector>
#include <unistd.h>
#include "host_common.hpp"
#include "report.hpp"
#include "target_config.hpp"

#define MS_VERSION "minorseq_b200 juliet 0.1.0 (B200-native restatement; not PacBio juliet)"

static void usage() {
    puts("Usage: juliet [options] <in.bam> <out.json|out.html|out.fasta> ...\n"
         "  outputs by extension, one or more: .json report, .html report, .fasta haplotype sequences (needs --mode-phasing)\n"
         "  -c, --config <HIV|ABL1|file.json>  target configuration (genes, DRMs, referenceSequence); the built-in HIV and ABL1\n"
         "                                     hold only what the public documentation shows (doc/JULIET.md:138-157 and the\n"
         "                                     target screenshot), not PacBio's full tables: pass the real config as a file\n"
         "      --region <begin-end>           1-based window to subset the target config\n"
         "      --mode-phasing                 phase variants into haplotypes\n"
         "      --linkage                      pairwise linkage of the called variants (reads clean at both codons; D', r^2,\n"
         "                                     Fisher tests for \"linked\" / \"exclusive\" after Bonferroni at --alpha)\n"
         "      --haplotype-abundance          with --mode-phasing: fit every read, damaged ones included, to the reported\n"
         "                                     haplotypes and estimate their frequencies by EM (\"haplotype_abundance\")\n"
         "      --indels                       also call in-frame codon deletions and whole-codon insertions between codons\n"
         "                                     (\"indels\"; DRM tokens such as 69ins, T69ins, 67del, D67del)\n"
         "      --min-perc <p>                 only variants with abundance > p %\n"
         "      --max-perc <p>                 only variants with abundance < p %\n"
         "      --drm-only                     only known drug-resistance mutations\n"
         "      --substitution-rate <r>        error model (default 5e-4)\n"
         "      --deletion-rate <r>            error model (default 3e-3)\n"
         "      --insertion-rate <r>           error model of --indels: an inserted string of n bases has probability r^n\n"
         "                                     (default 3e-3)\n"
         "      --alpha <a>                    significance after Bonferroni (default 0.01)\n"
         "      --min-haplotype-reads <n>      reads needed to report a haplotype (default 10)\n"
         "      --hap-min-coverage <n>         .fasta: a column with fewer votes of the haplotype's reads is written 'N'\n"
         "                                     (default 10; leading and trailing runs of such columns are trimmed)\n"
         "      --qv-threshold <q>             rich-QV base filter, 0 = off (default 20 on dq,iq,sq when present)\n"
         "      --device <n>                   first CUDA device (default 0)\n"
         "      --gpus <n>                     shard the reads over n GPUs (devices n0..n0+n-1) of this machine: contiguous read\n"
         "                                     ranges, one NCCL all-reduce of the count tensor, same report as with one GPU\n"
         "      --timing-json <file>           write the wall-clock time of every stage as JSON\n"
         "  -h, --help / --version");
}

static bool ends_with(const std::string& s, const std::string& e) { return s.size() >= e.size() && s.compare(s.size() - e.size(), e.size(), e) == 0; }

#define CK(h, call)                                                                            \
    do {                                                                                       \
        int rc_ = (call);                                                                      \
        if (rc_ != MS_OK) mshost::die(std::string(#call) + " failed: " + ms_last_error(h));     \
    } while (0)

int main(int argc, char** argv) {
    std::string config, region, cmdline, timing_json;
    bool phasing = false, drm_only = false, linkage = false, abundance = false, indels = false;
    double min_perc = -1, max_perc = -1, sub = 5e-4, del = 3e-3, alpha = 0.01, ins_rate = 3e-3;
    int min_hap = 10, device = 0, ngpus = 1, hap_min_cov = 10;
    const int link_min_reads = 10;   // reads clean at both codons that a tested pair needs (the haplotype default, F21)
    mshost::QvFilter qv;
    std::vector<std::string> pos;
    for (int i = 0; i < argc; ++i) cmdline += (i ? " " : "") + std::string(argv[i]);
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto need = [&](const char* name) -> std::string {
            if (i + 1 >= argc) mshost::die(std::string("option ") + name + " needs a value");
            return argv[++i];
        };
        if (a == "-h" || a == "--help") { usage(); return 0; }
        else if (a == "--version") { puts(MS_VERSION); return 0; }
        else if (a == "-c" || a == "--config") config = need("--config");
        else if (a == "--region") region = need("--region");
        else if (a == "--mode-phasing") phasing = true;
        else if (a == "--linkage") linkage = true;
        else if (a == "--haplotype-abundance") abundance = true;
        else if (a == "--indels") indels = true;
        else if (a == "--insertion-rate") ins_rate = atof(need("--insertion-rate").c_str());
        else if (a == "--drm-only") drm_only = true;
        else if (a == "--min-perc") min_perc = atof(need("--min-perc").c_str());
        else if (a == "--max-perc") max_perc = atof(need("--max-perc").c_str());
        else if (a == "--substitution-rate") sub = atof(need("--substitution-rate").c_str());
        else if (a == "--deletion-rate") del = atof(need("--deletion-rate").c_str());
        else if (a == "--alpha") alpha = atof(need("--alpha").c_str());
        else if (a == "--min-haplotype-reads") min_hap = atoi(need("--min-haplotype-reads").c_str());
        else if (a == "--hap-min-coverage") hap_min_cov = atoi(need("--hap-min-coverage").c_str());
        else if (a == "--qv-threshold") qv.threshold = atoi(need("--qv-threshold").c_str());
        else if (a == "--device") device = atoi(need("--device").c_str());
        else if (a == "--gpus") ngpus = atoi(need("--gpus").c_str());
        else if (a == "--timing-json") timing_json = need("--timing-json");
        else if (!a.empty() && a[0] == '-') mshost::die("unknown option " + a);
        else pos.push_back(a);
    }
    if (pos.size() < 2) { usage(); return 1; }
    if (ngpus < 1 || ngpus > 64) mshost::die("--gpus expects 1..64");
    std::string out_json, out_html, out_fasta;
    for (size_t i = 1; i < pos.size(); ++i) {
        if (ends_with(pos[i], ".json")) out_json = pos[i];
        else if (ends_with(pos[i], ".html")) out_html = pos[i];
        else if (ends_with(pos[i], ".fasta")) out_fasta = pos[i];
        else mshost::die("output must end in .json, .html or .fasta: " + pos[i]);
    }
    if (!out_fasta.empty() && !phasing) mshost::die("a .fasta output holds the haplotypes' sequences: it needs --mode-phasing");
    if (hap_min_cov < 0) mshost::die("--hap-min-coverage expects a count >= 0");
    if (abundance && !phasing) mshost::die("--haplotype-abundance fits the reads to the reported haplotypes: it needs --mode-phasing");
    int rb = 0, re = 0;
    if (!region.empty()) {
        if (sscanf(region.c_str(), "%d-%d", &rb, &re) != 2 || rb < 1 || re <= rb) mshost::die("--region expects <begin-end>");
    }

    const bool timing = getenv("MS_TIMING") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    auto t_prev = t_start;
    std::vector<std::pair<std::string, double>> laps;     // for --timing-json
    auto lap = [&](const char* what) {
        const auto now = std::chrono::steady_clock::now();
        const double ms = std::chrono::duration<double, std::milli>(now - t_prev).count();
        laps.emplace_back(what, ms);
        if (timing) fprintf(stderr, "[timing] %-28s %8.1f ms\n", what, ms);
        t_prev = now;
    };
    try {
        mscfg::TargetConfig cfg;
        if (!config.empty()) cfg = mscfg::load(config);

        // the CUDA contexts come up (~0.5 s each, one thread per GPU) while a helper thread inflates and indexes the BAM;
        // with --gpus N every GPU gets its own handle and the handles share one NCCL communicator (one rank per thread)
        std::vector<ms_handle*> hs(static_cast<size_t>(ngpus), nullptr);
        mshost::Alignments aln;
        const bool fasta = !out_fasta.empty();
        mshost::load_alignments_overlapped(pos[0], qv, phasing, fasta || indels, cfg.reference_sequence, aln, [&] {
            char id[128];
            if (ngpus > 1 && ms_comm_unique_id(id) != MS_OK) mshost::die("NCCL is not available (libnccl.so.2): --gpus needs it");
            std::vector<std::string> errs(static_cast<size_t>(ngpus));
            mshost::run_ranks(ngpus, [&](int r) {
                if (ms_create(device + r, &hs[r]) != MS_OK) { errs[r] = ms_last_error(nullptr); return; }   // there is no CPU path
                if (ngpus > 1 && ms_comm_init(hs[r], id, r, ngpus) != MS_OK) errs[r] = ms_last_error(hs[r]);
            });
            for (const std::string& e : errs)
                if (!e.empty()) mshost::die(e);
        });
        lap("CUDA context || BAM inflate + CIGAR expansion + event encoding");
        if (aln.nreads == 0) mshost::die("no primary or supplementary alignments in " + pos[0]);
        const int32_t L = aln.L;

        // genes: from the config, or one ORF labelled "unknown" (doc/JULIET.md:182-188)
        std::vector<mscfg::Gene> genes = cfg.genes;
        if (genes.empty()) {
            mscfg::Gene g;
            g.name = "unknown";
            g.begin = rb > 0 ? rb : 1;
            g.end = re > 0 ? re : L + 1;
            genes.push_back(g);
        }
        if (cfg.reference_name.empty()) cfg.reference_name = config.empty() ? "" : aln.ref_name;
        std::vector<uint32_t> start((L + 31) / 32, 0u);
        std::vector<ms_gene> mg;
        const int lo = rb > 0 ? rb - 1 : 0, hi = re > 0 ? std::min(L, re - 1) : L;
        for (const mscfg::Gene& g : genes) {
            mg.push_back({g.begin, g.end});
            for (int s = g.begin - 1; s + 3 <= std::min(g.end - 1, L); s += 3)
                if (s >= lo && s + 3 <= hi && s >= 0) start[s >> 5] |= 1u << (s & 31);
        }
        ms_call_params prm;
        ms_call_params_default(&prm);
        prm.substitution_rate = sub; prm.deletion_rate = del; prm.alpha = alpha;
        prm.min_perc = min_perc; prm.max_perc = max_perc; prm.region_begin = rb; prm.region_end = re;
        const char* ref = cfg.reference_sequence.size() >= static_cast<size_t>(L) ? cfg.reference_sequence.c_str() : nullptr;

        // Every rank piles up its contiguous range of the reads; after the all-reduce the counts, and with them the
        // variant list, are the same on every rank; phasing merges the ranks' pattern lists on the device and leaves the
        // per-read haplotype ids in the rank's slice of `hap`.  Rank 0's copy of the replicated results goes into the report.
        std::vector<msreport::VariantRow> rows;
        std::vector<uint32_t> col(static_cast<size_t>(L) * 8);
        std::vector<msreport::HaplotypeRow> haps;
        unsigned long long counters[6] = {0, 0, 0, 0, 0, 0};
        std::vector<int32_t> hap(phasing ? aln.nreads : 0);
        std::vector<std::pair<int, int>> keys;
        std::vector<uint32_t> pat;
        std::vector<uint64_t> cnt;
        int64_t nrep_all = 0;
        std::vector<ms_linkage_pair> link_pairs;
        int64_t link_tested = 0;
        std::vector<const uint32_t*> rows_dev(static_cast<size_t>(ngpus), nullptr);   // each rank's reads on its GPU (tiles)
        std::vector<std::string> errs(static_cast<size_t>(ngpus));
#define CKR(call)                                                                                      \
    do {                                                                                               \
        if ((call) != MS_OK) { errs[r] = std::string(#call) + " failed: " + ms_last_error(h); return; } \
    } while (0)
        mshost::run_ranks(ngpus, [&](int r) {
            ms_handle* h = hs[r];
            const int64_t r0 = aln.nreads * r / ngpus, r1 = aln.nreads * (r + 1) / ngpus;
            CKR(ms_set_layout(h, L, start.data()));
            CKR(ms_set_base(h, aln.base.data()));
            // this rank's reads as event rows (~112 B instead of 1504 B per 3 kb read on the link), expanded into tiles on the GPU
            const uint32_t* d_rows = nullptr;
            ms_read_hdr* my_hdr = ngpus > 1 ? nullptr : aln.hdr;
            const uint8_t* my_ev = aln.events;
            if (ngpus > 1) {
                try { my_ev = mshost::shard_events(aln, r0, r1, &my_hdr); } catch (const std::exception& e) { errs[r] = e.what(); return; }
            }
            const int prc = ms_pileup_events_host(h, my_hdr, my_ev, r1 - r0, &d_rows);
            if (prc == MS_OK && ngpus > 1) ms_synchronize(h);     // the shard's header copy is ours to free once the upload is done
            if (ngpus > 1) ms_free_pinned(my_hdr);
            if (prc != MS_OK) { errs[r] = std::string("ms_pileup_events_host failed: ") + ms_last_error(h); return; }
            rows_dev[r] = d_rows;
            CKR(ms_allreduce_counts(h));
            CKR(ms_synchronize(h));
            if (r == 0) lap(ngpus > 1 ? "H2D events + expand + pileup + all-reduce" : "H2D events + expand + pileup");

            std::vector<ms_variant> mv(4096);
            int64_t nv = 0;
            CKR(ms_call(h, mg.data(), static_cast<int32_t>(mg.size()), ref, &prm, mv.data(), static_cast<int64_t>(mv.size()), &nv));
            if (nv > static_cast<int64_t>(mv.size())) {
                mv.resize(nv);
                CKR(ms_call(h, mg.data(), static_cast<int32_t>(mg.size()), ref, &prm, mv.data(), static_cast<int64_t>(mv.size()), &nv));
            }
            mv.resize(nv);

            // DRM annotation and --drm-only (doc/JULIET.md:104-107,:370)
            std::vector<msreport::VariantRow> my_rows;
            for (const ms_variant& v : mv) {
                msreport::VariantRow vr;
                vr.gene = v.gene; vr.aa_pos = v.codon_index + 1; vr.col = v.col; vr.ref_codon = v.ref_codon; vr.codon = v.codon;
                vr.count = v.count; vr.coverage = v.coverage; vr.expected = v.expected; vr.ntests = v.ntests; vr.pvalue = v.pvalue;
                const char ra = mscfg::translate(v.ref_codon), va = mscfg::translate(v.codon);
                for (const mscfg::Drm& d : genes[v.gene].drms)
                    for (const mscfg::DrmPosition& p : d.positions)
                        if (mscfg::drm_matches(p, vr.aa_pos, ra, va)) { vr.drugs.push_back(d.name); break; }
                if (drm_only && vr.drugs.empty()) continue;
                my_rows.push_back(vr);
            }
            if (r == 0) {
                lap("call + DRM annotation");
                CKR(ms_get_counts(h, col.data(), nullptr));
            }
            if (phasing || linkage) {
                // one global variant list over all genes (screenshot juliet_hiv-phasing.png: same columns in every table)
                std::vector<std::pair<int, int>> my_keys;
                for (const msreport::VariantRow& vr : my_rows) my_keys.emplace_back(vr.col, vr.codon);
                std::sort(my_keys.begin(), my_keys.end());
                my_keys.erase(std::unique(my_keys.begin(), my_keys.end()), my_keys.end());
                const int32_t V = static_cast<int32_t>(my_keys.size());
                const int32_t nw = std::max(1, (V + 31) / 32);
                std::vector<int32_t> vc(V), vk(V);
                for (int32_t i = 0; i < V; ++i) { vc[i] = my_keys[i].first; vk[i] = my_keys[i].second; }
                CKR(ms_set_linkage(h, linkage ? 1 : 0));
                CKR(ms_set_abundance(h, abundance ? 1 : 0));
                CKR(ms_phase_begin(h, vc.data(), vk.data(), V, r1 - r0));
                CKR(ms_phase_dev(h, d_rows, r1 - r0));
                if (linkage) {
                    // every rank computes the same list from the all-reduced counts (a collective: all ranks call it)
                    ms_linkage_params lp;
                    ms_linkage_params_default(&lp);
                    lp.alpha = alpha;
                    lp.min_reads = link_min_reads;
                    std::vector<ms_linkage_pair> my_pairs(64);
                    int64_t np = 0, nt = 0;
                    for (;;) {
                        CKR(ms_linkage(h, &lp, my_pairs.data(), static_cast<int64_t>(my_pairs.size()), &np, &nt));
                        if (np <= static_cast<int64_t>(my_pairs.size())) break;
                        my_pairs.resize(np);
                    }
                    my_pairs.resize(np);
                    if (r == 0) { link_pairs.swap(my_pairs); link_tested = nt; }
                }
                if (phasing) {
                    // grouping, merge over the ranks, haplotype order and per-read ids in one device-side call; only the reported
                    // haplotypes are read back (every rank takes the same turns through this loop: nrep is a merged result)
                    int64_t H = 0, nrep = 0, cap = 256;
                    std::vector<uint32_t> my_pat;
                    std::vector<uint64_t> my_cnt;
                    ms_phase_counters c2;
                    for (;;) {
                        my_pat.assign(static_cast<size_t>(cap) * nw, 0u);
                        my_cnt.assign(cap, 0);
                        CKR(ms_phase_haplotypes(h, min_hap, my_pat.data(), my_cnt.data(), cap, &H, &nrep, &c2, hap.data() + r0));
                        if (nrep <= cap) break;
                        cap = nrep;
                    }
                    if (r == 0) {
                        counters[0] = c2.reported; counters[1] = c2.insufficient; counters[2] = c2.damaged;
                        counters[3] = c2.gaps; counters[4] = c2.heteroduplex; counters[5] = c2.partial;
                        pat.swap(my_pat); cnt.swap(my_cnt); nrep_all = nrep;
                    }
                }
                if (r == 0) keys.swap(my_keys);
            }
            if (r == 0) rows.swap(my_rows);
        });
        for (const std::string& e : errs)
            if (!e.empty()) mshost::die(e);
        ms_handle* h = hs[0];

        if (phasing) {
            const int32_t V = static_cast<int32_t>(keys.size());
            const int32_t nw = std::max(1, (V + 31) / 32);
            const int64_t nrep = nrep_all;
            haps.resize(nrep);
            for (int64_t k = 0; k < nrep; ++k) {
                char nb[3];
                ms_haplotype_name(k, nb);
                haps[k].name = nb;
                haps[k].reads = cnt[k];
                haps[k].frequency = counters[0] ? static_cast<double>(cnt[k]) / static_cast<double>(counters[0]) : 0.0;
                for (int32_t v = 0; v < V; ++v) {
                    char cb[4];
                    const bool on = (pat[static_cast<size_t>(k) * nw + (v >> 5)] >> (v & 31)) & 1u;
                    haps[k].codons.push_back(on ? mscfg::codon_string(keys[v].second, cb) : "");
                }
            }
            for (int64_t r = 0; r < aln.nreads; ++r)
                if (hap[r] >= 0 && hap[r] < nrep) haps[hap[r]].read_names.push_back(aln.names[r]);
            for (msreport::VariantRow& r : rows) {
                const int32_t v = static_cast<int32_t>(std::lower_bound(keys.begin(), keys.end(), std::make_pair(r.col, r.codon)) - keys.begin());
                r.haplotype_hit.resize(nrep);
                for (int64_t k = 0; k < nrep; ++k) r.haplotype_hit[k] = (pat[static_cast<size_t>(k) * nw + (v >> 5)] >> (v & 31)) & 1u;
            }
        }

        msreport::LinkageBlock link;
        if (linkage) {
            link.min_reads = link_min_reads;
            link.alpha = alpha;
            link.tested_pairs = link_tested;
            auto variant = [&](int32_t v) {
                msreport::LinkageVariant o;
                char cb[4];
                o.abs_pos = keys[v].first + 1;
                o.codon = mscfg::codon_string(keys[v].second, cb);
                for (const msreport::VariantRow& r : rows)
                    if (r.col == keys[v].first && r.codon == keys[v].second)
                        o.labels.push_back(genes[r.gene].name + " " + mscfg::translate(r.ref_codon) + std::to_string(r.aa_pos) + mscfg::translate(r.codon));
                return o;
            };
            for (const ms_linkage_pair& p : link_pairs) {
                msreport::LinkageRow lr;
                lr.a = variant(p.v);
                lr.b = variant(p.w);
                lr.reads = static_cast<unsigned long long>(p.both) + p.v_only + p.w_only + p.neither;
                lr.both = p.both; lr.a_only = p.v_only; lr.b_only = p.w_only; lr.neither = p.neither;
                lr.d_prime = p.d_prime; lr.r2 = p.r2; lr.pvalue = p.pvalue;
                lr.pvalue_corrected = std::min(1.0, p.pvalue * static_cast<double>(link_tested));
                lr.relation = p.relation == MS_LINKED ? "linked" : "exclusive";
                link.pairs.push_back(lr);
            }
        }

        lap(linkage ? "phasing + linkage" : "phasing");

        // in-frame indels: every rank counts its reads (string ids from all the run's insertion events, so that they agree), one
        // all-reduce inside ms_indel_call, the same list on every rank
        msreport::IndelBlock ind;
        if (indels) {
            ms_indel_params ip;
            ms_indel_params_default(&ip);
            ip.deletion_rate = del; ip.insertion_rate = ins_rate; ip.alpha = alpha;
            ip.min_perc = min_perc; ip.max_perc = max_perc; ip.region_begin = rb; ip.region_end = re;
            std::vector<ms_indel> calls;
            mshost::run_ranks(ngpus, [&](int r) {
                ms_handle* h = hs[r];
                const int64_t r0 = aln.nreads * r / ngpus, r1 = aln.nreads * (r + 1) / ngpus;
                CKR(ms_indel_count_dev(h, rows_dev[r], r1 - r0, r0, aln.ins_read.data(), aln.ins_col.data(), aln.ins_off.data(), aln.ins_len.data(),
                                       static_cast<int64_t>(aln.ins_read.size()), aln.ins_pool.data(), static_cast<int64_t>(aln.ins_pool.size())));
                std::vector<ms_indel> my(256);
                int64_t n = 0;
                for (;;) {
                    const int rc = ms_indel_call(h, mg.data(), static_cast<int32_t>(mg.size()), ref, &ip, my.data(), static_cast<int64_t>(my.size()), &n);
                    if (rc == MS_ERR_CAPACITY) { my.resize(n); continue; }
                    CKR(rc);
                    break;
                }
                my.resize(n);
                if (r == 0) calls.swap(my);
            });
            for (const std::string& e : errs)
                if (!e.empty()) mshost::die(e);
            ind.deletion_rate = del;
            ind.insertion_rate = ins_rate;
            for (const ms_indel& c : calls) {
                msreport::IndelRow row;
                const bool ins = c.kind == MS_INDEL_INSERTION;
                auto aa = [](int32_t codon) { return codon >= 0 ? mscfg::translate(codon) : '?'; };
                row.gene = c.gene;
                row.type = ins ? "insertion" : "deletion";
                row.ref_position = c.codon_index + 1;
                row.abs_pos = c.col + 1;
                row.count = c.count; row.coverage = c.coverage; row.expected = c.expected; row.ntests = c.ntests; row.pvalue = c.pvalue;
                row.label = std::string(1, aa(c.ref_codon)) + std::to_string(row.ref_position);
                if (ins) {
                    std::vector<char> buf(static_cast<size_t>(L) + 1);
                    int64_t len = 0;
                    for (;;) {
                        const int rc = ms_indel_inserted(h, c.sid, nullptr, buf.data(), static_cast<int64_t>(buf.size()), &len);
                        if (rc == MS_ERR_CAPACITY) { buf.resize(static_cast<size_t>(len)); continue; }
                        if (rc != MS_OK) mshost::die(std::string("ms_indel_inserted failed: ") + ms_last_error(h));
                        break;
                    }
                    row.inserted.assign(buf.data(), static_cast<size_t>(len));
                    row.label += "_" + std::string(1, aa(c.next_codon)) + std::to_string(row.ref_position + 1) + "ins";
                    for (size_t q = 0; q + 3 <= row.inserted.size(); q += 3) {
                        const int codon = 16 * (strchr("ACGT", row.inserted[q]) - "ACGT") + 4 * (strchr("ACGT", row.inserted[q + 1]) - "ACGT") +
                                          (strchr("ACGT", row.inserted[q + 2]) - "ACGT");
                        const char t = mscfg::translate(codon);
                        row.label += t == 'X' ? '*' : t;
                    }
                } else {
                    row.label += "del";
                }
                for (const mscfg::Drm& d : genes[c.gene].drms)
                    for (const mscfg::DrmPosition& p : d.positions)
                        if (mscfg::drm_matches_indel(p, row.ref_position, aa(c.ref_codon), ins)) { row.drugs.push_back(d.name); break; }
                if (drm_only && row.drugs.empty()) continue;
                ind.calls.push_back(row);
            }
            lap("indels");
        }

        // haplotype abundance: every rank fits its reads to the same reported patterns; classes and EM are merged inside the library
        msreport::AbundanceBlock ab;
        if (abundance) {
            const int64_t nrep = nrep_all;
            if (nrep > 4096)
                mshost::die("--haplotype-abundance handles at most 4096 haplotypes; this run reports " + std::to_string(nrep));
            ms_abundance_params ap;
            ms_abundance_params_default(&ap);
            ab.tolerance = ap.tolerance;
            ab.max_iterations = ap.max_iterations;
            std::vector<ms_abundance_row> arows(static_cast<size_t>(std::max<int64_t>(1, nrep)));
            ms_abundance_counters actr;
            int32_t it = 0, conv = 0;
            double ll = 0;
            mshost::run_ranks(ngpus, [&](int r) {
                ms_handle* h = hs[r];
                std::vector<ms_abundance_row> my_rows(arows.size());
                ms_abundance_counters my_ctr;
                int32_t my_it = 0, my_conv = 0;
                double my_ll = 0;
                CKR(ms_haplotype_abundance(h, &ap, pat.data(), nrep, my_rows.data(), nrep, &my_ctr, &my_it, &my_conv, &my_ll));
                if (r == 0) { arows.swap(my_rows); actr = my_ctr; it = my_it; conv = my_conv; ll = my_ll; }
            });
            for (const std::string& e : errs)
                if (!e.empty()) mshost::die(e);
            ab.iterations = it;
            ab.converged = conv != 0;
            ab.log_likelihood = ll;
            ab.unique = actr.unique; ab.ambiguous = actr.ambiguous; ab.uninformative = actr.uninformative; ab.incompatible = actr.incompatible;
            for (int64_t k = 0; k < nrep; ++k) {
                msreport::AbundanceRow row;
                row.name = haps[k].name;
                row.reads = haps[k].reads;
                row.unique_reads = arows[k].unique_reads;
                row.compatible_reads = arows[k].compatible_reads;
                row.em_frequency = arows[k].em_frequency;
                ab.haplotypes.push_back(row);
            }
            lap("haplotype abundance");
        }

        // haplotype sequences: every rank piles up its reads per haplotype (labels: the ranks' positions in the haplotype
        // order, on the device), one all-reduce sums the group counts, rank 0 calls them with all insertion events
        std::string fasta_text;
        if (fasta) {
            const int32_t nrep = static_cast<int32_t>(nrep_all);
            mshost::run_ranks(ngpus, [&](int r) {
                ms_handle* h = hs[r];
                const int64_t r0 = aln.nreads * r / ngpus, r1 = aln.nreads * (r + 1) / ngpus;
                int32_t* d_hap = nullptr;
                int64_t nh = 0;
                CKR(ms_phase_hap_device(h, &d_hap, &nh));
                if (nh != r1 - r0) { errs[r] = "ms_phase_hap_device: unexpected read count"; return; }
                CKR(ms_set_groups(h, nrep));
                CKR(ms_group_pileup_dev(h, rows_dev[r], d_hap, r1 - r0));
                CKR(ms_allreduce_group_counts(h));
                CKR(ms_synchronize(h));
            });
            for (const std::string& e : errs)
                if (!e.empty()) mshost::die(e);
            ms_fuse_params fp;
            ms_fuse_params_default(&fp);
            fp.min_coverage = hap_min_cov;
            std::vector<int32_t> ins_hap(aln.ins_read.size());
            for (size_t i = 0; i < ins_hap.size(); ++i) ins_hap[i] = hap[aln.ins_read[i]];
            std::vector<int64_t> seq_off(static_cast<size_t>(nrep) + 1, 0);
            std::string seqs(static_cast<size_t>(nrep) * (static_cast<size_t>(L) + 16), '\0');
            for (;;) {
                const int rc = ms_group_consensus(h, &fp, ins_hap.data(), aln.ins_col.data(), aln.ins_off.data(), aln.ins_len.data(),
                                                  static_cast<int64_t>(ins_hap.size()), aln.ins_pool.data(), static_cast<int64_t>(aln.ins_pool.size()),
                                                  seqs.empty() ? nullptr : &seqs[0], static_cast<int64_t>(seqs.size()), seq_off.data());
                if (rc == MS_ERR_CAPACITY) { seqs.resize(static_cast<size_t>(seq_off[nrep])); continue; }
                if (rc != MS_OK) mshost::die(std::string("ms_group_consensus failed: ") + ms_last_error(h));
                break;
            }
            std::string stem = pos[0];
            const size_t sl = stem.find_last_of('/');
            if (sl != std::string::npos) stem = stem.substr(sl + 1);
            for (int32_t k = 0; k < nrep; ++k) {
                char nb[3];
                ms_haplotype_name(k, nb);
                fasta_text += ">" + stem + "|haplotype_" + nb + "|" + aln.ref_name + " reads=" + std::to_string(cnt[k]) + "\n";
                for (int64_t i = seq_off[k]; i < seq_off[k + 1]; i += 70)
                    fasta_text += seqs.substr(static_cast<size_t>(i), static_cast<size_t>(std::min<int64_t>(70, seq_off[k + 1] - i))) + "\n";
            }
            lap("haplotype consensus");
        }
        char ts[40];
        const auto now = std::chrono::system_clock::now();
        const std::time_t tt = std::chrono::system_clock::to_time_t(now);
        const long ms = static_cast<long>(std::chrono::duration_cast<std::chrono::milliseconds>(now.time_since_epoch()).count() % 1000);
        std::tm tmv;
        gmtime_r(&tt, &tmv);
        char base[32];
        strftime(base, sizeof base, "%Y-%m-%dT%H:%M:%S", &tmv);
        snprintf(ts, sizeof ts, "%s.%03ldZ", base, ms);
        if (getenv("MS_FIXED_TIMESTAMP")) snprintf(ts, sizeof ts, "%s", getenv("MS_FIXED_TIMESTAMP"));

        const msjson::Value report = msreport::build(ts, pos[0], cmdline, MS_VERSION, cfg, L, genes, rows, col, L, phasing, haps, counters,
                                                     linkage ? &link : nullptr, abundance ? &ab : nullptr, indels ? &ind : nullptr);
        if (!out_json.empty()) {
            std::ofstream f(out_json);
            if (!f) mshost::die("cannot write " + out_json);
            f << msjson::dump(report);
        }
        if (!out_html.empty()) {
            std::ofstream f(out_html);
            if (!f) mshost::die("cannot write " + out_html);
            f << msreport::to_html(report);
        }
        if (fasta) {
            std::ofstream f(out_fasta);
            if (!f) mshost::die("cannot write " + out_fasta);
            f << fasta_text;
        }
        lap("report writing");
#undef CKR
        if (!timing_json.empty()) {
            msjson::Value t = msjson::Value::object();
            msjson::Value st = msjson::Value::array();
            for (const auto& l : laps) {
                msjson::Value e = msjson::Value::object();
                e.set("stage", msjson::Value::string(l.first));
                e.set("ms", msjson::Value::number(l.second));
                st.push(e);
            }
            t.set("reads", msjson::Value::integer(aln.nreads));
            t.set("stages", st);
            t.set("total_ms", msjson::Value::number(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count()));
            std::ofstream f(timing_json);
            if (!f) mshost::die("cannot write " + timing_json);
            f << msjson::dump(t);
        }
        fprintf(stderr, "juliet: %lld reads (%lld skipped), %zu variants%s\n", static_cast<long long>(aln.nreads),
                static_cast<long long>(aln.nskipped), rows.size(), phasing ? (", " + std::to_string(haps.size()) + " haplotypes").c_str() : "");
        fflush(nullptr);
        if (!getenv("MS_FULL_TEARDOWN")) _exit(0);   // outputs are written and closed; skip the ~0.2 s CUDA teardown
        for (ms_handle* x : hs) ms_destroy(x);
    } catch (const std::exception& e) {
        mshost::die(e.what());
    }
    return 0;
}
