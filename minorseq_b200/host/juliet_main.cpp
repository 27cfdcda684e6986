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
// deletions and insertions between codons with K2's model and reports them in an "indels" block.  --phase-indels (restatement
// choice U20) adds the reported indels to the phasing keys: haplotypes, linkage, abundance and the FASTA then see them.
// --rare-linkage (restatement choice U21) looks for minor strains below K2's threshold: codons that K2 does not call but whose
// uncorrected p is small, tested for linkage to each other and to the called variants on the reads clean at both codons.
// --control (restatement choice U22) piles up a control sample with the same layout and tests every codon of the sample against
// the control's count at the same position (two-sample Fisher), so that a systematic error is told apart from a minor strain.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <ctime>
#include <fstream>
#include <string>
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
         "      --phase-indels                 with --mode-phasing and --indels: phase the reported indels with the variants\n"
         "                                     (haplotypes, linkage, abundance and the .fasta carry them)\n"
         "      --rare-linkage                 sub-threshold variant linkage: uncalled codons with a small uncorrected p, tested\n"
         "                                     for linkage over the reads; linked groups and their reads (\"rare_linkage\")\n"
         "      --rare-min-reads <n>           reads a --rare-linkage candidate needs (default 5)\n"
         "      --rare-candidate-alpha <a>     uncorrected p a --rare-linkage candidate needs to stay below (default 0.1)\n"
         "      --control <control.bam>        test each codon against a control sample (same reference) at the same position:\n"
         "                                     two-sample one-sided Fisher, Bonferroni at --alpha (\"control\"; the rest of the\n"
         "                                     report is unchanged)\n"
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

struct Options {
    std::string input, config, region, cmdline, timing_json, out_json, out_html, out_fasta, control;
    bool phasing = false, drm_only = false, linkage = false, abundance = false, indels = false, phase_indels = false, rare_linkage = false;
    double min_perc = -1, max_perc = -1, sub = 5e-4, del = 3e-3, alpha = 0.01, ins_rate = 3e-3, rare_alpha = 0.1;
    int min_hap = 10, device = 0, ngpus = 1, hap_min_cov = 10, rare_min_reads = 5;
    int rb = 0, re = 0;                // --region, 0 = none
    mshost::QvFilter qv;
};
const int link_min_reads = 10;   // reads clean at both codons that a tested pair needs (the haplotype default, F21)

static Options parse_options(int argc, char** argv) {
    Options o;
    std::vector<std::string> pos;
    for (int i = 0; i < argc; ++i) o.cmdline += (i ? " " : "") + std::string(argv[i]);
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto need = [&](const char* name) -> std::string {
            if (i + 1 >= argc) mshost::die(std::string("option ") + name + " needs a value");
            return argv[++i];
        };
        if (a == "-h" || a == "--help") { usage(); exit(0); }
        else if (a == "--version") { puts(MS_VERSION); exit(0); }
        else if (a == "-c" || a == "--config") o.config = need("--config");
        else if (a == "--region") o.region = need("--region");
        else if (a == "--mode-phasing") o.phasing = true;
        else if (a == "--linkage") o.linkage = true;
        else if (a == "--haplotype-abundance") o.abundance = true;
        else if (a == "--indels") o.indels = true;
        else if (a == "--phase-indels") o.phase_indels = true;
        else if (a == "--rare-linkage") o.rare_linkage = true;
        else if (a == "--rare-min-reads") o.rare_min_reads = atoi(need("--rare-min-reads").c_str());
        else if (a == "--rare-candidate-alpha") o.rare_alpha = atof(need("--rare-candidate-alpha").c_str());
        else if (a == "--control") o.control = need("--control");
        else if (a == "--insertion-rate") o.ins_rate = atof(need("--insertion-rate").c_str());
        else if (a == "--drm-only") o.drm_only = true;
        else if (a == "--min-perc") o.min_perc = atof(need("--min-perc").c_str());
        else if (a == "--max-perc") o.max_perc = atof(need("--max-perc").c_str());
        else if (a == "--substitution-rate") o.sub = atof(need("--substitution-rate").c_str());
        else if (a == "--deletion-rate") o.del = atof(need("--deletion-rate").c_str());
        else if (a == "--alpha") o.alpha = atof(need("--alpha").c_str());
        else if (a == "--min-haplotype-reads") o.min_hap = atoi(need("--min-haplotype-reads").c_str());
        else if (a == "--hap-min-coverage") o.hap_min_cov = atoi(need("--hap-min-coverage").c_str());
        else if (a == "--qv-threshold") o.qv.threshold = atoi(need("--qv-threshold").c_str());
        else if (a == "--device") o.device = atoi(need("--device").c_str());
        else if (a == "--gpus") o.ngpus = atoi(need("--gpus").c_str());
        else if (a == "--timing-json") o.timing_json = need("--timing-json");
        else if (!a.empty() && a[0] == '-') mshost::die("unknown option " + a);
        else pos.push_back(a);
    }
    if (pos.size() < 2) { usage(); exit(1); }
    if (o.ngpus < 1 || o.ngpus > 64) mshost::die("--gpus expects 1..64");
    o.input = pos[0];
    for (size_t i = 1; i < pos.size(); ++i) {
        if (ends_with(pos[i], ".json")) o.out_json = pos[i];
        else if (ends_with(pos[i], ".html")) o.out_html = pos[i];
        else if (ends_with(pos[i], ".fasta")) o.out_fasta = pos[i];
        else mshost::die("output must end in .json, .html or .fasta: " + pos[i]);
    }
    if (!o.out_fasta.empty() && !o.phasing) mshost::die("a .fasta output holds the haplotypes' sequences: it needs --mode-phasing");
    if (o.hap_min_cov < 0) mshost::die("--hap-min-coverage expects a count >= 0");
    if (o.abundance && !o.phasing) mshost::die("--haplotype-abundance fits the reads to the reported haplotypes: it needs --mode-phasing");
    if (o.phase_indels && (!o.phasing || !o.indels))
        mshost::die("--phase-indels puts the reported indels into the haplotypes: it needs --mode-phasing and --indels");
    if (o.rare_min_reads < 1) mshost::die("--rare-min-reads expects a count >= 1");
    if (!(o.rare_alpha > 0.0 && o.rare_alpha <= 1.0)) mshost::die("--rare-candidate-alpha expects a value in (0, 1]");
    if (!o.region.empty()) {
        if (sscanf(o.region.c_str(), "%d-%d", &o.rb, &o.re) != 2 || o.rb < 1 || o.re <= o.rb) mshost::die("--region expects <begin-end>");
    }
    return o;
}

struct Laps {       // the wall-clock time of every stage, for --timing-json (and on stderr with MS_TIMING)
    const bool print = getenv("MS_TIMING") != nullptr;
    const std::chrono::steady_clock::time_point start = std::chrono::steady_clock::now();
    std::chrono::steady_clock::time_point prev = start;
    std::vector<std::pair<std::string, double>> laps;
    void operator()(const char* what) {
        const auto now = std::chrono::steady_clock::now();
        const double ms = std::chrono::duration<double, std::milli>(now - prev).count();
        laps.emplace_back(what, ms);
        if (print) fprintf(stderr, "[timing] %-28s %8.1f ms\n", what, ms);
        prev = now;
    }
};

// One run: what the stages share.  The rank pass leaves rank 0's copy of the ranks' replicated results here.
struct Run {
    const Options o;
    Laps lap;
    mscfg::TargetConfig cfg;
    std::vector<ms_gene> mg;                  // rep.genes as the library takes them
    std::vector<uint32_t> start;              // the codon starts inside --region
    ms_call_params prm;
    const char* ref = nullptr;                // the config's referenceSequence when it covers the reference
    mshost::Alignments aln;
    mshost::Alignments ctl;                   // --control: the control's reads
    std::vector<ms_handle*> hs;               // one handle per GPU (rank)
    std::vector<const uint32_t*> rows_dev;    // each rank's reads on its GPU (tiles)
    std::vector<std::pair<int, int>> keys;    // the called variants' (col, codon), sorted: phasing keys 0..V-1
    std::vector<int32_t> key_del, key_sid;    // --phase-indels: the keys V..: deletion columns, then insertion string ids
    std::vector<ms_indel> calls;
    std::vector<uint32_t> pat;                // the reported haplotypes' key bits, nw words each
    int32_t nw = 1;
    std::vector<uint64_t> cnt;
    int64_t nrep = 0;                         // reported haplotypes
    std::vector<int32_t> hap;                 // per read: its haplotype's position in the report order (-1 = none)
    std::vector<ms_linkage_pair> link_pairs;
    int64_t link_tested = 0;
    std::vector<ms_control_variant> control_rows;
    int64_t control_uncovered = 0;
    msreport::Report rep;
    bool carries(int64_t k, int32_t v) const { return (pat[static_cast<size_t>(k) * nw + (v >> 5)] >> (v & 31)) & 1u; }
    std::string gene_label(int gene, const std::string& label) const { return rep.genes[gene].name + " " + label; }
};

// "K65R": reference amino acid, 1-based amino-acid position, variant amino acid
static std::string aa_change(int ref_codon, int pos, int codon) {
    return std::string(1, mscfg::translate(ref_codon)) + std::to_string(pos) + mscfg::translate(codon);
}

static ms_linkage_params link_params(const Options& o) {
    ms_linkage_params lp;
    ms_linkage_params_default(&lp);
    lp.alpha = o.alpha;
    lp.min_reads = link_min_reads;
    return lp;
}

// the target config, the reads, the handles and the genes' codon starts
static void load(Run& run) {
    const Options& o = run.o;
    if (!o.config.empty()) run.cfg = mscfg::load(o.config);
    // the CUDA contexts come up (~0.5 s each, one thread per GPU) while a helper thread inflates and indexes the BAM;
    // with --gpus N every GPU gets its own handle and the handles share one NCCL communicator (one rank per thread)
    mshost::load_alignments_overlapped(o.input, o.qv, o.phasing, !o.out_fasta.empty() || o.indels, run.cfg.reference_sequence, run.aln,
                                       [&] { run.hs = mshost::open_ranks(o.device, o.ngpus); });
    run.lap("CUDA context || BAM inflate + CIGAR expansion + event encoding");
    if (run.aln.nreads == 0) mshost::die("no primary or supplementary alignments in " + o.input);
    const int32_t L = run.aln.L;
    if (!o.control.empty()) {
        // the control goes through the same admission rules and QV filter; it must be aligned to the sample's reference
        mshost::Decoded d;
        mshost::decode_alignments(o.control, d, run.ctl);
        if (run.ctl.nreads == 0) mshost::die("no primary or supplementary alignments in the control " + o.control);
        if (run.ctl.ref_name != run.aln.ref_name || run.ctl.L != L)
            mshost::die("the control " + o.control + " is aligned to " + run.ctl.ref_name + " (" + std::to_string(run.ctl.L) + " bp), the sample to " +
                        run.aln.ref_name + " (" + std::to_string(L) + " bp): --control needs the same reference");
        mshost::expand_alignments(d, o.qv, false, false, run.cfg.reference_sequence, run.ctl);
        run.lap("control BAM inflate + CIGAR expansion + event encoding");
    }

    // genes: from the config, or one ORF labelled "unknown" (doc/JULIET.md:182-188)
    std::vector<mscfg::Gene>& genes = run.rep.genes;
    genes = run.cfg.genes;
    if (genes.empty()) {
        mscfg::Gene g;
        g.name = "unknown";
        g.begin = o.rb > 0 ? o.rb : 1;
        g.end = o.re > 0 ? o.re : L + 1;
        genes.push_back(g);
    }
    if (run.cfg.reference_name.empty()) run.cfg.reference_name = o.config.empty() ? "" : run.aln.ref_name;
    run.start.assign((L + 31) / 32, 0u);
    const int lo = o.rb > 0 ? o.rb - 1 : 0, hi = o.re > 0 ? std::min(L, o.re - 1) : L;
    for (const mscfg::Gene& g : genes) {
        run.mg.push_back({g.begin, g.end});
        for (int s = g.begin - 1; s + 3 <= std::min(g.end - 1, L); s += 3)
            if (s >= lo && s + 3 <= hi && s >= 0) run.start[s >> 5] |= 1u << (s & 31);
    }
    ms_call_params_default(&run.prm);
    run.prm.substitution_rate = o.sub; run.prm.deletion_rate = o.del; run.prm.alpha = o.alpha;
    run.prm.min_perc = o.min_perc; run.prm.max_perc = o.max_perc; run.prm.region_begin = o.rb; run.prm.region_end = o.re;
    run.ref = run.cfg.reference_sequence.size() >= static_cast<size_t>(L) ? run.cfg.reference_sequence.c_str() : nullptr;
    run.rep.L = L;
    run.rep.col_counts.resize(static_cast<size_t>(L) * 8);
    run.rows_dev.resize(static_cast<size_t>(o.ngpus));
    run.hap.resize(o.phasing ? run.aln.nreads : 0);
}

// the DRMs of gene `gene` that a codon change at 1-based amino-acid position aa_pos matches (doc/JULIET.md:104-107)
static std::vector<std::string> variant_drugs(const Run& run, int gene, int aa_pos, int ref_codon, int codon) {
    std::vector<std::string> d;
    const char ra = mscfg::translate(ref_codon), va = mscfg::translate(codon);
    for (const mscfg::Drm& x : run.rep.genes[gene].drms)
        for (const mscfg::DrmPosition& p : x.positions)
            if (mscfg::drm_matches(p, aa_pos, ra, va)) { d.push_back(x.name); break; }
    return d;
}

static char indel_aa(int32_t codon) { return codon >= 0 ? mscfg::translate(codon) : '?'; }

static std::vector<std::string> indel_drugs(const Run& run, const ms_indel& c) {
    std::vector<std::string> d;
    for (const mscfg::Drm& x : run.rep.genes[c.gene].drms)
        for (const mscfg::DrmPosition& p : x.positions)
            if (mscfg::drm_matches_indel(p, c.codon_index + 1, indel_aa(c.ref_codon), c.kind == MS_INDEL_INSERTION)) { d.push_back(x.name); break; }
    return d;
}

// in-frame indels on rank r: the rank counts its reads (string ids from all the run's insertion events, so that they agree), one
// all-reduce inside ms_indel_call, the same list on every rank
static std::vector<ms_indel> call_indels(const Run& run, int r) {
    const Options& o = run.o;
    const mshost::Alignments& a = run.aln;
    ms_handle* h = run.hs[r];
    const std::pair<int64_t, int64_t> s = mshost::shard(a.nreads, r, o.ngpus);
    CK(h, ms_indel_count_dev(h, run.rows_dev[r], s.second - s.first, s.first, a.ins_read.data(), a.ins_col.data(), a.ins_off.data(), a.ins_len.data(),
                             static_cast<int64_t>(a.ins_read.size()), a.ins_pool.data(), static_cast<int64_t>(a.ins_pool.size())));
    ms_indel_params ip;
    ms_indel_params_default(&ip);
    ip.deletion_rate = o.del; ip.insertion_rate = o.ins_rate; ip.alpha = o.alpha;
    ip.min_perc = o.min_perc; ip.max_perc = o.max_perc; ip.region_begin = o.rb; ip.region_end = o.re;
    return mshost::fetch<ms_indel>(h, "ms_indel_call", 256, [&](ms_indel* out, int64_t cap, int64_t* n) {
        return ms_indel_call(h, run.mg.data(), static_cast<int32_t>(run.mg.size()), run.ref, &ip, out, cap, n);
    });
}

// Every rank piles up its contiguous range of the reads; after the all-reduce the counts, and with them the variant list, are
// the same on every rank; phasing merges the ranks' pattern lists on the device and leaves the per-read haplotype ids in the
// rank's slice of `hap`.  Rank 0's copy of the replicated results goes into the report.
static void rank_pass(Run& run) {
    const Options& o = run.o;
    mshost::for_ranks(o.ngpus, [&](int r) {
        ms_handle* h = run.hs[r];
        const std::pair<int64_t, int64_t> s = mshost::shard(run.aln.nreads, r, o.ngpus);
        const int64_t nr = s.second - s.first;
        CK(h, ms_set_layout(h, run.aln.L, run.start.data()));
        if (!o.control.empty()) {
            // the control first: the sample's reads have to stay on the device for phasing and indels
            CK(h, ms_set_base(h, run.ctl.base.data()));
            mshost::pileup_shard(h, run.ctl, r, o.ngpus);
            CK(h, ms_control_capture(h));
            CK(h, ms_reset_counts(h));
            if (r == 0) run.lap(o.ngpus > 1 ? "control: H2D events + expand + pileup + all-reduce" : "control: H2D events + expand + pileup");
        }
        CK(h, ms_set_base(h, run.aln.base.data()));
        run.rows_dev[r] = mshost::pileup_shard(h, run.aln, r, o.ngpus);
        if (r == 0) run.lap(o.ngpus > 1 ? "H2D events + expand + pileup + all-reduce" : "H2D events + expand + pileup");

        const std::vector<ms_variant> mv = mshost::fetch<ms_variant>(h, "ms_call", 4096, [&](ms_variant* out, int64_t cap, int64_t* n) {
            return ms_call(h, run.mg.data(), static_cast<int32_t>(run.mg.size()), run.ref, &run.prm, out, cap, n);
        });
        // DRM annotation and --drm-only (doc/JULIET.md:104-107,:370)
        std::vector<msreport::VariantRow> rows;
        std::vector<ms_variant> listed;       // the calls behind `rows`
        for (const ms_variant& v : mv) {
            msreport::VariantRow vr;
            vr.gene = v.gene; vr.aa_pos = v.codon_index + 1; vr.col = v.col; vr.ref_codon = v.ref_codon; vr.codon = v.codon;
            vr.count = v.count; vr.coverage = v.coverage; vr.expected = v.expected; vr.ntests = v.ntests; vr.pvalue = v.pvalue;
            vr.drugs = variant_drugs(run, v.gene, vr.aa_pos, v.ref_codon, v.codon);
            if (o.drm_only && vr.drugs.empty()) continue;
            rows.push_back(vr);
            listed.push_back(v);
        }
        if (r == 0) run.lap("call + DRM annotation");
        if (!o.control.empty()) {
            // replicated: every rank tests the same all-reduced counts against the same capture
            int64_t unc = 0;
            std::vector<ms_control_variant> cv = mshost::fetch<ms_control_variant>(h, "ms_control_call", 256, [&](ms_control_variant* out, int64_t cap, int64_t* n) {
                return ms_control_call(h, run.mg.data(), static_cast<int32_t>(run.mg.size()), run.ref, &run.prm, listed.data(),
                                       static_cast<int64_t>(listed.size()), out, cap, n, &unc);
            });
            if (r == 0) {
                run.control_rows.swap(cv);
                run.control_uncovered = unc;
                run.lap("control comparison");
            }
        }
        if (r == 0) CK(h, ms_get_counts(h, run.rep.col_counts.data(), nullptr));
        // one global variant list over all genes (screenshot juliet_hiv-phasing.png: same columns in every table)
        std::vector<std::pair<int, int>> keys;
        for (const msreport::VariantRow& vr : rows) keys.emplace_back(vr.col, vr.codon);
        std::sort(keys.begin(), keys.end());
        keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
        std::vector<ms_indel> calls;
        std::vector<int32_t> del, sid;
        if (o.phase_indels) {
            calls = call_indels(run, r);
            if (r == 0) run.lap("indels");
            for (const ms_indel& c : calls) {
                if (o.drm_only && indel_drugs(run, c).empty()) continue;
                if (c.kind == MS_INDEL_DELETION) del.push_back(c.col);
                else sid.push_back(c.sid);
            }
            for (std::vector<int32_t>* k : {&del, &sid}) {
                std::sort(k->begin(), k->end());
                k->erase(std::unique(k->begin(), k->end()), k->end());
            }
        }
        if (o.phasing || o.linkage) {
            const int32_t V = static_cast<int32_t>(keys.size());
            const int32_t nw = std::max(1, (V + static_cast<int32_t>(del.size() + sid.size()) + 31) / 32);
            std::vector<int32_t> vc(V), vk(V);
            for (int32_t i = 0; i < V; ++i) { vc[i] = keys[i].first; vk[i] = keys[i].second; }
            CK(h, ms_set_linkage(h, o.linkage ? 1 : 0));
            CK(h, ms_set_abundance(h, o.abundance ? 1 : 0));
            CK(h, ms_phase_begin_indels(h, vc.data(), vk.data(), V, del.data(), static_cast<int32_t>(del.size()), sid.data(),
                                        static_cast<int32_t>(sid.size()), nr));
            CK(h, ms_phase_dev(h, run.rows_dev[r], nr));
            if (o.linkage) {
                // every rank computes the same list from the all-reduced counts (a collective: all ranks call it)
                const ms_linkage_params lp = link_params(o);
                int64_t nt = 0;
                std::vector<ms_linkage_pair> pairs = mshost::fetch<ms_linkage_pair>(h, "ms_linkage", 64, [&](ms_linkage_pair* out, int64_t cap, int64_t* n) {
                    return ms_linkage(h, &lp, out, cap, n, &nt);
                });
                if (r == 0) { run.link_pairs.swap(pairs); run.link_tested = nt; }
            }
            if (o.phasing) {
                // grouping, merge over the ranks, haplotype order and per-read ids in one device-side call; only the reported
                // haplotypes are read back (every rank takes the same turns through this loop: nrep is a merged result)
                int64_t H = 0, nrep = 0, cap = 256;
                std::vector<uint32_t> pat;
                std::vector<uint64_t> cnt;
                ms_phase_counters c2;
                for (;;) {
                    pat.assign(static_cast<size_t>(cap) * nw, 0u);
                    cnt.assign(cap, 0);
                    CK(h, ms_phase_haplotypes(h, o.min_hap, pat.data(), cnt.data(), cap, &H, &nrep, &c2, run.hap.data() + s.first));
                    if (nrep <= cap) break;
                    cap = nrep;
                }
                if (r == 0) {
                    unsigned long long* ctr = run.rep.counters;
                    ctr[0] = c2.reported; ctr[1] = c2.insufficient; ctr[2] = c2.damaged; ctr[3] = c2.gaps; ctr[4] = c2.heteroduplex; ctr[5] = c2.partial;
                    run.pat.swap(pat); run.cnt.swap(cnt); run.nrep = nrep; run.nw = nw;
                }
            }
        }
        if (r == 0) { run.rep.variants.swap(rows); run.keys.swap(keys); run.key_del.swap(del); run.key_sid.swap(sid); run.calls.swap(calls); }
    });
}

// the report rows of the indel calls; with --phase-indels each row's key (V + position among the indel keys)
static msreport::IndelBlock indel_block(const Run& run) {
    const Options& o = run.o;
    ms_handle* h = run.hs[0];
    const int32_t V = static_cast<int32_t>(run.keys.size());
    msreport::IndelBlock ind;
    ind.deletion_rate = o.del;
    ind.insertion_rate = o.ins_rate;
    ind.phased = o.phase_indels;
    for (const ms_indel& c : run.calls) {
        msreport::IndelRow row;
        const bool ins = c.kind == MS_INDEL_INSERTION;
        row.gene = c.gene;
        row.type = ins ? "insertion" : "deletion";
        row.ref_position = c.codon_index + 1;
        row.abs_pos = c.col + 1;
        row.count = c.count; row.coverage = c.coverage; row.expected = c.expected; row.ntests = c.ntests; row.pvalue = c.pvalue;
        row.label = std::string(1, indel_aa(c.ref_codon)) + std::to_string(row.ref_position);
        if (ins) {
            const std::vector<char> buf = mshost::fetch<char>(h, "ms_indel_inserted", run.aln.L + 1, [&](char* out, int64_t cap, int64_t* len) {
                return ms_indel_inserted(h, c.sid, nullptr, out, cap, len);
            });
            row.inserted.assign(buf.begin(), buf.end());
            row.label += "_" + std::string(1, indel_aa(c.next_codon)) + std::to_string(row.ref_position + 1) + "ins";
            for (size_t q = 0; q + 3 <= row.inserted.size(); q += 3) {
                const int codon = 16 * (strchr("ACGT", row.inserted[q]) - "ACGT") + 4 * (strchr("ACGT", row.inserted[q + 1]) - "ACGT") +
                                  (strchr("ACGT", row.inserted[q + 2]) - "ACGT");
                const char t = mscfg::translate(codon);
                row.label += t == 'X' ? '*' : t;
            }
        } else {
            row.label += "del";
        }
        row.drugs = indel_drugs(run, c);
        if (o.drm_only && row.drugs.empty()) continue;
        if (o.phase_indels)
            row.key = ins ? V + static_cast<int>(run.key_del.size() + (std::lower_bound(run.key_sid.begin(), run.key_sid.end(), c.sid) - run.key_sid.begin()))
                          : V + static_cast<int>(std::lower_bound(run.key_del.begin(), run.key_del.end(), c.col) - run.key_del.begin());
        ind.calls.push_back(row);
    }
    return ind;
}

// phasing key v as a linkage variant: a called variant with the labels of its report rows, or an indel key ("---" or "+" and the
// inserted bases) with the labels of its calls
static msreport::LinkageVariant key_variant(const Run& run, int32_t v) {
    msreport::LinkageVariant o;
    if (v >= static_cast<int32_t>(run.keys.size())) {
        for (const msreport::IndelRow& row : run.rep.indels->calls)
            if (row.key == v) {
                o.abs_pos = row.abs_pos;
                o.codon = row.type == "deletion" ? "---" : "+" + row.inserted;
                o.labels.push_back(run.gene_label(row.gene, row.label));
            }
        return o;
    }
    char cb[4];
    o.abs_pos = run.keys[v].first + 1;
    o.codon = mscfg::codon_string(run.keys[v].second, cb);
    for (const msreport::VariantRow& r : run.rep.variants)
        if (r.col == run.keys[v].first && r.codon == run.keys[v].second) o.labels.push_back(run.gene_label(r.gene, aa_change(r.ref_codon, r.aa_pos, r.codon)));
    return o;
}

// one tested pair as a report row; m: the number of tests of the Bonferroni correction
static msreport::LinkageRow linkage_row(const ms_linkage_pair& p, msreport::LinkageVariant a, msreport::LinkageVariant b, int64_t m, const char* relation) {
    msreport::LinkageRow lr;
    lr.a = std::move(a);
    lr.b = std::move(b);
    lr.reads = static_cast<unsigned long long>(p.both) + p.v_only + p.w_only + p.neither;
    lr.both = p.both; lr.a_only = p.v_only; lr.b_only = p.w_only; lr.neither = p.neither;
    lr.d_prime = p.d_prime; lr.r2 = p.r2; lr.pvalue = p.pvalue;
    lr.pvalue_corrected = std::min(1.0, p.pvalue * static_cast<double>(m));
    lr.relation = relation;
    return lr;
}

// the reported haplotypes with their reads, and which of them carries each variant and (--phase-indels) indel row
static void haplotypes(Run& run) {
    msreport::Report& rep = run.rep;
    const int32_t V = static_cast<int32_t>(run.keys.size()), nkeys = V + static_cast<int32_t>(run.key_del.size() + run.key_sid.size());
    rep.haplotypes.resize(run.nrep);
    for (int64_t k = 0; k < run.nrep; ++k) {
        msreport::HaplotypeRow& hr = rep.haplotypes[k];
        char nb[3];
        ms_haplotype_name(k, nb);
        hr.name = nb;
        hr.reads = run.cnt[k];
        hr.frequency = rep.counters[0] ? static_cast<double>(run.cnt[k]) / static_cast<double>(rep.counters[0]) : 0.0;
        for (int32_t v = 0; v < V; ++v) {
            char cb[4];
            hr.codons.push_back(run.carries(k, v) ? mscfg::codon_string(run.keys[v].second, cb) : "");
        }
        for (int32_t v = V; v < nkeys; ++v)
            if (run.carries(k, v))
                for (const std::string& l : key_variant(run, v).labels) hr.indels.push_back(l);
    }
    if (rep.indels)
        for (msreport::IndelRow& row : rep.indels->calls) {
            row.haplotype_hit.resize(run.nrep);
            for (int64_t k = 0; k < run.nrep; ++k) row.haplotype_hit[k] = run.carries(k, row.key);
        }
    for (int64_t r = 0; r < run.aln.nreads; ++r)
        if (run.hap[r] >= 0 && run.hap[r] < run.nrep) rep.haplotypes[run.hap[r]].read_names.push_back(run.aln.names[r]);
    for (msreport::VariantRow& r : rep.variants) {
        const int32_t v = static_cast<int32_t>(std::lower_bound(run.keys.begin(), run.keys.end(), std::make_pair(r.col, r.codon)) - run.keys.begin());
        r.haplotype_hit.resize(run.nrep);
        for (int64_t k = 0; k < run.nrep; ++k) r.haplotype_hit[k] = run.carries(k, v);
    }
}

static msreport::LinkageBlock linkage_block(const Run& run) {
    msreport::LinkageBlock link;
    link.min_reads = link_min_reads;
    link.alpha = run.o.alpha;
    link.tested_pairs = run.link_tested;
    for (const ms_linkage_pair& p : run.link_pairs)
        link.pairs.push_back(linkage_row(p, key_variant(run, p.v), key_variant(run, p.w), run.link_tested, p.relation == MS_LINKED ? "linked" : "exclusive"));
    return link;
}

// haplotype abundance: every rank fits its reads to the same reported patterns; classes and EM are merged inside the library
static msreport::AbundanceBlock abundance_block(Run& run) {
    const int64_t nrep = run.nrep;
    if (nrep > 4096) mshost::die("--haplotype-abundance handles at most 4096 haplotypes; this run reports " + std::to_string(nrep));
    msreport::AbundanceBlock ab;
    ms_abundance_params ap;
    ms_abundance_params_default(&ap);
    ab.tolerance = ap.tolerance;
    ab.max_iterations = ap.max_iterations;
    struct Fit { std::vector<ms_abundance_row> rows; ms_abundance_counters ctr; int32_t it = 0, conv = 0; double ll = 0; };
    std::vector<Fit> fits(static_cast<size_t>(run.o.ngpus));     // each rank's copy of the merged result
    mshost::for_ranks(run.o.ngpus, [&](int r) {
        Fit& f = fits[r];
        f.rows.resize(static_cast<size_t>(std::max<int64_t>(1, nrep)));
        CK(run.hs[r], ms_haplotype_abundance(run.hs[r], &ap, run.pat.data(), nrep, f.rows.data(), nrep, &f.ctr, &f.it, &f.conv, &f.ll));
    });
    const Fit& f = fits[0];
    const std::vector<ms_abundance_row>& arows = f.rows;
    const ms_abundance_counters& actr = f.ctr;
    ab.iterations = f.it;
    ab.converged = f.conv != 0;
    ab.log_likelihood = f.ll;
    ab.unique = actr.unique; ab.ambiguous = actr.ambiguous; ab.uninformative = actr.uninformative; ab.incompatible = actr.incompatible;
    for (int64_t k = 0; k < nrep; ++k) {
        msreport::AbundanceRow row;
        row.name = run.rep.haplotypes[k].name;
        row.reads = run.rep.haplotypes[k].reads;
        row.unique_reads = arows[k].unique_reads;
        row.compatible_reads = arows[k].compatible_reads;
        row.em_frequency = arows[k].em_frequency;
        ab.haplotypes.push_back(row);
    }
    run.lap("haplotype abundance");
    return ab;
}

// haplotype sequences: every rank piles up its reads per haplotype (labels: the ranks' positions in the haplotype
// order, on the device), one all-reduce sums the group counts, rank 0 calls them with all insertion events
static std::string haplotype_fasta(Run& run) {
    const mshost::Alignments& a = run.aln;
    const int32_t nrep = static_cast<int32_t>(run.nrep);
    mshost::for_ranks(run.o.ngpus, [&](int r) {
        ms_handle* h = run.hs[r];
        const std::pair<int64_t, int64_t> s = mshost::shard(a.nreads, r, run.o.ngpus);
        int32_t* d_hap = nullptr;
        int64_t nh = 0;
        CK(h, ms_phase_hap_device(h, &d_hap, &nh));
        if (nh != s.second - s.first) throw std::runtime_error("ms_phase_hap_device: unexpected read count");
        CK(h, ms_set_groups(h, nrep));
        CK(h, ms_group_pileup_dev(h, run.rows_dev[r], d_hap, s.second - s.first));
        CK(h, ms_allreduce_group_counts(h));
        CK(h, ms_synchronize(h));
    });
    ms_handle* h = run.hs[0];
    ms_fuse_params fp;
    ms_fuse_params_default(&fp);
    fp.min_coverage = run.o.hap_min_cov;
    std::vector<int32_t> ins_hap(a.ins_read.size());
    for (size_t i = 0; i < ins_hap.size(); ++i) ins_hap[i] = run.hap[a.ins_read[i]];
    std::vector<int64_t> seq_off(static_cast<size_t>(nrep) + 1, 0);
    std::string seqs(static_cast<size_t>(nrep) * (static_cast<size_t>(a.L) + 16), '\0');
    for (;;) {
        const int rc = ms_group_consensus(h, &fp, ins_hap.data(), a.ins_col.data(), a.ins_off.data(), a.ins_len.data(),
                                          static_cast<int64_t>(ins_hap.size()), a.ins_pool.data(), static_cast<int64_t>(a.ins_pool.size()),
                                          seqs.empty() ? nullptr : &seqs[0], static_cast<int64_t>(seqs.size()), seq_off.data());
        if (rc == MS_ERR_CAPACITY) { seqs.resize(static_cast<size_t>(seq_off[nrep])); continue; }
        mshost::check(h, rc, "ms_group_consensus");
        break;
    }
    const std::string stem = mshost::file_name(run.o.input);
    std::string text;
    for (int32_t k = 0; k < nrep; ++k) {
        char nb[3];
        ms_haplotype_name(k, nb);
        text += ">" + stem + "|haplotype_" + nb + "|" + a.ref_name + " reads=" + std::to_string(run.cnt[k]) + "\n";
        for (int64_t i = seq_off[k]; i < seq_off[k + 1]; i += 70)
            text += seqs.substr(static_cast<size_t>(i), static_cast<size_t>(std::min<int64_t>(70, seq_off[k + 1] - i))) + "\n";
    }
    run.lap("haplotype consensus");
    return text;
}

// sub-threshold linkage: every rank phases the called keys and the candidates anew (the handle's phasing state is no longer
// needed by the steps above) and takes the same turns through the collectives: the Gram all-reduce, the support all-reduce
static msreport::RareBlock rare_block(Run& run) {
    const Options& o = run.o;
    const int32_t fc = static_cast<int32_t>(run.keys.size());
    ms_rare_params rp;
    ms_rare_params_default(&rp);
    rp.min_reads = o.rare_min_reads;
    rp.candidate_alpha = o.rare_alpha;
    const ms_linkage_params lp = link_params(o);
    std::vector<ms_variant> cands;
    std::vector<ms_linkage_pair> rpairs;
    std::vector<int32_t> rgroup;
    std::vector<uint64_t> rcar, rinf;
    int64_t rdropped = 0, rtested = 0;
    mshost::for_ranks(o.ngpus, [&](int r) {
        ms_handle* h = run.hs[r];
        const std::pair<int64_t, int64_t> s = mshost::shard(run.aln.nreads, r, o.ngpus);
        int64_t dropped = 0, nt = 0;
        std::vector<ms_variant> my_c = mshost::fetch<ms_variant>(h, "ms_rare_candidates", 256, [&](ms_variant* out, int64_t cap, int64_t* n) {
            return ms_rare_candidates(h, run.mg.data(), static_cast<int32_t>(run.mg.size()), run.ref, &run.prm, &rp, out, cap, n, &dropped);
        });
        const int32_t nc = static_cast<int32_t>(my_c.size()), V = fc + nc;
        std::vector<int32_t> vc(V), vk(V);
        for (int32_t i = 0; i < fc; ++i) { vc[i] = run.keys[i].first; vk[i] = run.keys[i].second; }
        for (int32_t i = 0; i < nc; ++i) { vc[fc + i] = my_c[i].col; vk[fc + i] = my_c[i].codon; }
        CK(h, ms_set_linkage(h, 1));
        CK(h, ms_phase_begin(h, vc.data(), vk.data(), V, s.second - s.first));
        CK(h, ms_phase_dev(h, run.rows_dev[r], s.second - s.first));
        std::vector<ms_linkage_pair> my_p = mshost::fetch<ms_linkage_pair>(h, "ms_rare_linkage", 64, [&](ms_linkage_pair* out, int64_t cap, int64_t* n) {
            return ms_rare_linkage(h, fc, &lp, out, cap, n, &nt);
        });
        std::vector<int32_t> grp(static_cast<size_t>(std::max(1, V)), -1);
        const int ng = ms_rare_groups(my_p.data(), static_cast<int64_t>(my_p.size()), fc, V, grp.data());
        if (ng < 0) throw std::runtime_error("ms_rare_groups failed");
        const int32_t nw = std::max(1, (V + 31) / 32);
        std::vector<uint32_t> masks(static_cast<size_t>(std::max(1, ng)) * nw, 0u);
        for (int32_t k = 0; k < V; ++k)
            if (grp[k] >= 0) masks[static_cast<size_t>(grp[k]) * nw + (k >> 5)] |= 1u << (k & 31);
        std::vector<uint64_t> car(static_cast<size_t>(std::max(1, ng))), inf(car.size());
        CK(h, ms_rare_support(h, masks.data(), ng, car.data(), inf.data()));
        if (r == 0) {
            cands.swap(my_c); rpairs.swap(my_p); rgroup.swap(grp); car.resize(ng); inf.resize(ng); rcar.swap(car); rinf.swap(inf);
            rdropped = dropped; rtested = nt;
        }
    });
    msreport::RareBlock rare;
    rare.min_reads = o.rare_min_reads;
    rare.candidate_alpha = o.rare_alpha;
    rare.alpha = o.alpha;
    rare.pair_min_reads = link_min_reads;
    rare.max_candidates = MS_RARE_MAX_CANDIDATES;
    rare.candidates_tested = static_cast<long long>(cands.size());
    rare.dropped_candidates = rdropped;
    rare.tested_pairs = rtested;
    auto cand_label = [&](const ms_variant& c) { return aa_change(c.ref_codon, c.codon_index + 1, c.codon); };
    auto variant = [&](int32_t k) {
        if (k < fc) return key_variant(run, k);
        const ms_variant& c = cands[k - fc];
        msreport::LinkageVariant v;
        char cb[4];
        v.abs_pos = c.col + 1;
        v.codon = mscfg::codon_string(c.codon, cb);
        v.labels.push_back(run.gene_label(c.gene, cand_label(c)));
        return v;
    };
    std::vector<std::vector<std::string>> linked_called(cands.size());
    std::vector<char> in_pair(cands.size(), 0);
    for (const ms_linkage_pair& p : rpairs) {
        rare.pairs.push_back(linkage_row(p, variant(p.v), variant(p.w), rtested, "linked"));
        in_pair[p.w - fc] = 1;
        if (p.v >= fc) in_pair[p.v - fc] = 1;
        else for (const std::string& l : rare.pairs.back().a.labels) linked_called[p.w - fc].push_back(l);
    }
    rare.groups.resize(rcar.size());
    for (size_t g = 0; g < rcar.size(); ++g) { rare.groups[g].carriers = rcar[g]; rare.groups[g].informative = rinf[g]; }
    for (size_t i = 0; i < cands.size(); ++i) {
        const ms_variant& c = cands[i];
        const int32_t g = rgroup[fc + i];
        if (g >= 0) rare.groups[g].members.push_back(run.gene_label(c.gene, cand_label(c)));
        if (!in_pair[i]) continue;
        msreport::RareCandidate rc;
        char cb[4];
        rc.gene = run.rep.genes[c.gene].name;
        rc.label = cand_label(c);
        rc.position = c.codon_index + 1;
        rc.abs_pos = c.col + 1;
        rc.ref_codon = mscfg::codon_string(c.ref_codon, cb);
        rc.codon = mscfg::codon_string(c.codon, cb);
        rc.count = c.count; rc.coverage = c.coverage; rc.expected = c.expected; rc.pvalue = c.pvalue;
        rc.group = g;
        rc.linked_called = linked_called[i];
        rare.candidates.push_back(rc);
    }
    run.lap("rare linkage");
    return rare;
}

// the control comparison's rows: the control calls and the report's variants, DRM-annotated (--drm-only drops the rest)
static msreport::ControlBlock control_block(const Run& run) {
    msreport::ControlBlock cb;
    cb.input_file = run.o.control;
    cb.reads = run.ctl.nreads;
    cb.alpha = run.o.alpha;
    cb.uncovered_positions = run.control_uncovered;
    for (const ms_control_variant& v : run.control_rows) {
        msreport::ControlRow row;
        char cb4[4];
        row.gene = run.rep.genes[v.gene].name;
        row.position = v.codon_index + 1;
        row.label = aa_change(v.ref_codon, row.position, v.codon);
        row.abs_pos = v.col + 1;
        row.ref_codon = mscfg::codon_string(v.ref_codon, cb4);
        row.codon = mscfg::codon_string(v.codon, cb4);
        row.count = v.count; row.coverage = v.coverage; row.control_count = v.control_count; row.control_coverage = v.control_coverage;
        row.pvalue = v.pvalue;
        row.pvalue_corrected = std::min(1.0, v.pvalue * static_cast<double>(v.ntests));
        row.control_call = v.called != 0;
        row.model_call = v.listed != 0;
        row.drugs = variant_drugs(run, v.gene, row.position, v.ref_codon, v.codon);
        if (run.o.drm_only && row.drugs.empty()) continue;
        cb.rows.push_back(row);
    }
    return cb;
}

static void write_file(const std::string& path, const std::string& text) {
    std::ofstream f(path);
    if (!f) mshost::die("cannot write " + path);
    f << text;
}

// the .json / .html report, the .fasta, and the --timing-json stage times
static void write_outputs(Run& run, const std::string& fasta) {
    const Options& o = run.o;
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

    msreport::Report& rep = run.rep;
    rep.timestamp = ts;
    rep.input_file = o.input;
    rep.command_line = o.cmdline;
    rep.version = MS_VERSION;
    rep.cfg = run.cfg;
    rep.phasing = o.phasing;
    const msjson::Value report = msreport::build(rep);
    if (!o.out_json.empty()) write_file(o.out_json, msjson::dump(report));
    if (!o.out_html.empty()) write_file(o.out_html, msreport::to_html(report));
    if (!o.out_fasta.empty()) write_file(o.out_fasta, fasta);
    run.lap("report writing");
    if (!o.timing_json.empty()) {
        msjson::Value t = msjson::Value::object();
        msjson::Value st = msjson::Value::array();
        for (const auto& l : run.lap.laps) {
            msjson::Value e = msjson::Value::object();
            e.set("stage", msjson::Value::string(l.first));
            e.set("ms", msjson::Value::number(l.second));
            st.push(e);
        }
        t.set("reads", msjson::Value::integer(run.aln.nreads));
        t.set("stages", st);
        t.set("total_ms", msjson::Value::number(std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - run.lap.start).count()));
        write_file(o.timing_json, msjson::dump(t));
    }
}

int main(int argc, char** argv) {
    const Options o = parse_options(argc, argv);
    try {
        Run run{o};
        load(run);
        rank_pass(run);                                   // pile-up, calls, [--phase-indels: indels,] phasing, linkage
        if (o.phase_indels) run.rep.indels = indel_block(run);
        if (o.phasing) haplotypes(run);
        if (o.linkage) run.rep.linkage = linkage_block(run);
        run.lap(o.linkage ? "phasing + linkage" : "phasing");
        if (o.indels && !o.phase_indels) {
            mshost::for_ranks(o.ngpus, [&](int r) {
                std::vector<ms_indel> calls = call_indels(run, r);
                if (r == 0) run.calls.swap(calls);
            });
            run.rep.indels = indel_block(run);
            run.lap("indels");
        }
        if (o.abundance) run.rep.abundance = abundance_block(run);
        const std::string fasta = o.out_fasta.empty() ? std::string() : haplotype_fasta(run);
        if (o.rare_linkage) run.rep.rare = rare_block(run);   // replaces the handles' phasing state: last
        if (!o.control.empty()) run.rep.control = control_block(run);
        write_outputs(run, fasta);
        fprintf(stderr, "juliet: %lld reads (%lld skipped), %zu variants%s\n", static_cast<long long>(run.aln.nreads),
                static_cast<long long>(run.aln.nskipped), run.rep.variants.size(),
                o.phasing ? (", " + std::to_string(run.rep.haplotypes.size()) + " haplotypes").c_str() : "");
        fflush(nullptr);
        if (!getenv("MS_FULL_TEARDOWN")) _exit(0);   // outputs are written and closed; skip the ~0.2 s CUDA teardown
        for (ms_handle* x : run.hs) ms_destroy(x);
    } catch (const std::exception& e) {
        mshost::die(e.what());
    }
    return 0;
}
