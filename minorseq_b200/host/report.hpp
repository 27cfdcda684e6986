// report.hpp -- juliet's JSON report and its 1:1 HTML rendering.
//
// "The HTML page is a 1:1 conversion of the JSON file" with four sections: Input data, Target config,
// Variant Discovery, Drug Summaries (/root/reference/doc/JULIET.md:68-107).  Per variant position: reference
// codon, reference amino acid, relative amino-acid position, mutated codon, mutated amino acid, coverage,
// affected drugs, and the -3..+5 MSA counts (:94-100, screenshot juliet_hiv-context.png).  With phasing each
// variant carries a `haplotype_hit` bool array and the root holds a haplotype block with counts and read
// names (:207-211); tooltips show reported / insufficient / unsuitable reads with the three marginals
// (:372-381).  The full schema is not documented (SURVEY U9): the field names below are this
// implementation's choice, mirroring the HTML tables column by column.
#pragma once
#include <algorithm>
#include <cstdio>
#include <map>
#include <string>
#include <vector>
#include "json.hpp"
#include "target_config.hpp"

namespace msreport {

using msjson::Value;

struct VariantRow {
    int gene = 0, aa_pos = 0, col = 0, ref_codon = 0, codon = 0;
    unsigned count = 0, coverage = 0, expected = 0, ntests = 0;
    double pvalue = 0;
    std::vector<std::string> drugs;
    std::vector<bool> haplotype_hit;
};

struct HaplotypeRow {
    std::string name;
    unsigned long long reads = 0;
    double frequency = 0;           // of the reported reads (screenshot juliet_hiv-phasing.png sums to 100)
    std::vector<std::string> codons;  // per variant column: codon string if carried, else ""
    std::vector<std::string> read_names;
};

// pairwise linkage of two called variants (--linkage, restatement choice U14): one row per significant pair
struct LinkageVariant {
    int abs_pos = 0;                  // 1-based first column of the codon
    std::string codon;
    std::vector<std::string> labels;  // the variant's report rows, e.g. "Reverse Transcriptase K65R"
};
struct LinkageRow {
    LinkageVariant a, b;
    unsigned long long reads = 0, both = 0, a_only = 0, b_only = 0, neither = 0;
    double d_prime = 0, r2 = 0, pvalue = 0, pvalue_corrected = 0;
    std::string relation;             // "linked" or "exclusive"
};
struct LinkageBlock {
    int min_reads = 0;
    double alpha = 0;
    long long tested_pairs = 0;
    std::vector<LinkageRow> pairs;
};

// haplotype abundance (--haplotype-abundance, restatement choice U18): every phased read fitted to the reported haplotypes
struct AbundanceRow {
    std::string name;
    unsigned long long reads = 0, unique_reads = 0, compatible_reads = 0;
    double em_frequency = 0;
};
struct AbundanceBlock {
    double tolerance = 0;
    int max_iterations = 0, iterations = 0;
    bool converged = false;
    double log_likelihood = 0;
    unsigned long long unique = 0, ambiguous = 0, uninformative = 0, incompatible = 0;
    std::vector<AbundanceRow> haplotypes;   // report order
};

// in-frame codon deletions and insertions (--indels, restatement choice U19)
struct IndelRow {
    int gene = 0;
    std::string type;          // "deletion" / "insertion"
    std::string label;         // D67del, T69_S70insSS
    int ref_position = 0;      // 1-based codon of the deletion / before the insertion
    int abs_pos = 0;           // 1-based column: the deleted codon's first, or the one the insertion follows
    std::string inserted;      // upper-cased inserted bases ("" for a deletion)
    unsigned count = 0, coverage = 0, expected = 0, ntests = 0;
    double pvalue = 0;
    std::vector<std::string> drugs;
};
struct IndelBlock {
    double deletion_rate = 0, insertion_rate = 0;
    std::vector<IndelRow> calls;   // (gene, codon, deletion first, inserted)
};

// "%": two significant digits as in the screenshots (1.1, 0.91, 98, 100)
inline std::string perc2(double p) {
    char b[32];
    snprintf(b, sizeof b, "%.2g", p);
    std::string s(b);
    if (s.find('e') != std::string::npos) { snprintf(b, sizeof b, "%.0f", p); s = b; }
    return s;
}
inline std::string perc1(double p) {  // haplotype %: one decimal, trailing ".0" dropped (92.5, 1.2, 1)
    char b[32];
    snprintf(b, sizeof b, "%.1f", p);
    std::string s(b);
    if (s.size() > 2 && s.compare(s.size() - 2, 2, ".0") == 0) s.resize(s.size() - 2);
    return s;
}

inline Value build(const std::string& timestamp, const std::string& input_file, const std::string& cmdline, const std::string& version,
                   const mscfg::TargetConfig& cfg, int ref_length, const std::vector<mscfg::Gene>& genes,
                   const std::vector<VariantRow>& variants, const std::vector<unsigned>& col_counts /* L*8 */, int L,
                   bool phasing, const std::vector<HaplotypeRow>& haps, const unsigned long long counters[6],
                   const LinkageBlock* linkage = nullptr, const AbundanceBlock* abundance = nullptr, const IndelBlock* indels = nullptr) {
    Value root = Value::object();
    Value& in = root.set("input", Value::object());
    in.set("timestamp", Value::string(timestamp));
    in.set("input_file", Value::string(input_file));
    in.set("command_line", Value::string(cmdline));
    in.set("juliet_version", Value::string(version));
    Value& tc = root.set("target_config", Value::object());
    tc.set("version", Value::string(cfg.version));
    tc.set("databaseVersion", Value::string(cfg.database_version));
    tc.set("referenceName", Value::string(cfg.reference_name));
    tc.set("referenceLength", Value::integer(ref_length));
    Value& tg = tc.set("genes", Value::array());
    for (const mscfg::Gene& g : genes) {
        Value& o = tg.push(Value::object());
        o.set("name", Value::string(g.name));
        o.set("begin", Value::integer(g.begin));
        o.set("end", Value::integer(g.end));
        Value& ds = o.set("drms", Value::array());
        for (const mscfg::Drm& d : g.drms) {
            Value& dd = ds.push(Value::object());
            dd.set("name", Value::string(d.name));
            Value& ps = dd.set("positions", Value::array());
            for (const mscfg::DrmPosition& p : d.positions) ps.push(Value::string(p.text));
        }
    }
    Value& gs = root.set("genes", Value::array());
    std::map<std::string, std::vector<std::string>> drug_summary;
    std::vector<std::string> drug_order;
    for (size_t gi = 0; gi < genes.size(); ++gi) {
        Value& go = gs.push(Value::object());
        go.set("name", Value::string(genes[gi].name));
        Value& vps = go.set("variant_positions", Value::array());
        for (size_t i = 0; i < variants.size();) {
            if (variants[i].gene != static_cast<int>(gi)) { ++i; continue; }
            size_t j = i;
            while (j < variants.size() && variants[j].gene == variants[i].gene && variants[j].col == variants[i].col) ++j;
            const VariantRow& f = variants[i];
            char cb[4];
            Value& vp = vps.push(Value::object());
            vp.set("ref_codon", Value::string(mscfg::codon_string(f.ref_codon, cb)));
            vp.set("ref_amino_acid", Value::string(std::string(1, mscfg::translate(f.ref_codon))));
            vp.set("ref_position", Value::integer(f.aa_pos));
            vp.set("coverage", Value::integer(f.coverage));
            // group the variant codons by amino acid (one position may carry several, SURVEY F18)
            Value& vaas = vp.set("variant_amino_acids", Value::array());
            for (size_t k = i; k < j; ++k) {
                const VariantRow& v = variants[k];
                const std::string aa(1, mscfg::translate(v.codon));
                Value* slot = nullptr;
                for (Value& e : vaas.arr) if (e.get_string("amino_acid") == aa) slot = &e;
                if (!slot) { slot = &vaas.push(Value::object()); slot->set("amino_acid", Value::string(aa)); slot->set("variant_codons", Value::array()); }
                Value& codons = const_cast<Value&>(*slot->get("variant_codons"));
                Value& vc = codons.push(Value::object());
                vc.set("codon", Value::string(mscfg::codon_string(v.codon, cb)));
                const double freq = static_cast<double>(v.count) / static_cast<double>(v.coverage);
                vc.set("frequency", Value::number(freq));
                vc.set("percentage", Value::string(perc2(100.0 * freq)));
                vc.set("count", Value::integer(v.count));
                vc.set("expected", Value::integer(v.expected));
                vc.set("pValue", Value::number(v.pvalue));
                vc.set("pValueCorrected", Value::number(std::min(1.0, v.pvalue * v.ntests)));
                std::string known;
                for (size_t d = 0; d < v.drugs.size(); ++d) known += (d ? " + " : "") + v.drugs[d];
                vc.set("known_drm", Value::string(known));
                if (phasing) {
                    Value& hh = vc.set("haplotype_hit", Value::array());
                    for (bool b : v.haplotype_hit) hh.push(Value::boolean(b));
                }
                const std::string label = std::string(1, mscfg::translate(v.ref_codon)) + std::to_string(v.aa_pos) + aa + " (" + genes[gi].name + ", " +
                                          perc2(100.0 * freq) + " %)";
                for (const std::string& d : v.drugs) {
                    if (!drug_summary.count(d)) drug_order.push_back(d);
                    drug_summary[d].push_back(label);
                }
            }
            // MSA context: relative positions -3..+5 around the codon's first column (screenshot juliet_hiv-context.png)
            Value& msa = vp.set("msa", Value::array());
            for (int rel = -3; rel <= 5; ++rel) {
                const int c = f.col + rel;
                if (c < 0 || c >= L) continue;
                Value& row = msa.push(Value::object());
                row.set("rel_pos", Value::integer(rel));
                row.set("abs_pos", Value::integer(c + 1));
                static const char* names[6] = {"A", "C", "G", "T", "-", "N"};
                for (int s = 0; s < 6; ++s) row.set(names[s], Value::integer(col_counts[static_cast<size_t>(c) * 8 + s]));
            }
            i = j;
        }
    }
    if (indels)
        for (const IndelRow& r : indels->calls) {
            const std::string label = r.label + " (" + genes[r.gene].name + ", " + perc2(100.0 * r.count / r.coverage) + " %)";
            for (const std::string& d : r.drugs) {
                if (!drug_summary.count(d)) drug_order.push_back(d);
                drug_summary[d].push_back(label);
            }
        }
    Value& dsum = root.set("drug_summaries", Value::array());
    for (const std::string& d : drug_order) {
        Value& o = dsum.push(Value::object());
        o.set("drug", Value::string(d));
        Value& vs = o.set("variants", Value::array());
        for (const std::string& l : drug_summary[d]) vs.push(Value::string(l));
    }
    if (phasing) {
        Value& hs = root.set("haplotypes", Value::array());
        for (const HaplotypeRow& h : haps) {
            Value& o = hs.push(Value::object());
            o.set("name", Value::string(h.name));
            o.set("reads", Value::integer(static_cast<long long>(h.reads)));
            o.set("frequency", Value::number(h.frequency));
            o.set("percentage", Value::string(perc1(100.0 * h.frequency)));
            Value& cs = o.set("codons", Value::array());
            for (const std::string& c : h.codons) cs.push(Value::string(c));
            Value& rn = o.set("read_names", Value::array());
            for (const std::string& n : h.read_names) rn.push(Value::string(n));
        }
        Value& hc = root.set("haplotype_read_categories", Value::object());
        static const char* names[6] = {"reported", "insufficient_coverage", "unsuitable", "unsuitable_gaps", "unsuitable_heteroduplex", "unsuitable_partial"};
        for (int i = 0; i < 6; ++i) hc.set(names[i], Value::integer(static_cast<long long>(counters[i])));
    }
    if (linkage) {
        Value& lk = root.set("linkage", Value::object());
        lk.set("min_reads", Value::integer(linkage->min_reads));
        lk.set("alpha", Value::number(linkage->alpha));
        lk.set("tested_pairs", Value::integer(linkage->tested_pairs));
        Value& ps = lk.set("pairs", Value::array());
        auto variant = [](const LinkageVariant& v) {
            Value o = Value::object();
            o.set("abs_pos", Value::integer(v.abs_pos));
            o.set("codon", Value::string(v.codon));
            Value& ls = o.set("labels", Value::array());
            for (const std::string& l : v.labels) ls.push(Value::string(l));
            return o;
        };
        for (const LinkageRow& r : linkage->pairs) {
            Value& o = ps.push(Value::object());
            o.set("a", variant(r.a));
            o.set("b", variant(r.b));
            o.set("reads", Value::integer(static_cast<long long>(r.reads)));
            o.set("both", Value::integer(static_cast<long long>(r.both)));
            o.set("a_only", Value::integer(static_cast<long long>(r.a_only)));
            o.set("b_only", Value::integer(static_cast<long long>(r.b_only)));
            o.set("neither", Value::integer(static_cast<long long>(r.neither)));
            o.set("d_prime", Value::number(r.d_prime));
            o.set("r2", Value::number(r.r2));
            o.set("pValue", Value::number(r.pvalue));
            o.set("pValueCorrected", Value::number(r.pvalue_corrected));
            o.set("relation", Value::string(r.relation));
        }
    }
    if (indels) {
        Value& ib = root.set("indels", Value::object());
        ib.set("deletion_rate", Value::number(indels->deletion_rate));
        ib.set("insertion_rate", Value::number(indels->insertion_rate));
        Value& cs = ib.set("calls", Value::array());
        for (const IndelRow& r : indels->calls) {
            Value& o = cs.push(Value::object());
            const double freq = static_cast<double>(r.count) / static_cast<double>(r.coverage);
            o.set("gene", Value::string(genes[r.gene].name));
            o.set("type", Value::string(r.type));
            o.set("label", Value::string(r.label));
            o.set("ref_position", Value::integer(r.ref_position));
            o.set("abs_pos", Value::integer(r.abs_pos));
            o.set("inserted", Value::string(r.inserted));
            o.set("count", Value::integer(r.count));
            o.set("coverage", Value::integer(r.coverage));
            o.set("frequency", Value::number(freq));
            o.set("percentage", Value::string(perc2(100.0 * freq)));
            o.set("expected", Value::integer(r.expected));
            o.set("pValue", Value::number(r.pvalue));
            o.set("pValueCorrected", Value::number(std::min(1.0, r.pvalue * r.ntests)));
            std::string known;
            for (size_t d = 0; d < r.drugs.size(); ++d) known += (d ? " + " : "") + r.drugs[d];
            o.set("known_drm", Value::string(known));
        }
    }
    if (abundance) {
        Value& ab = root.set("haplotype_abundance", Value::object());
        ab.set("tolerance", Value::number(abundance->tolerance));
        ab.set("max_iterations", Value::integer(abundance->max_iterations));
        ab.set("iterations", Value::integer(abundance->iterations));
        ab.set("converged", Value::boolean(abundance->converged));
        ab.set("log_likelihood", Value::number(abundance->log_likelihood));
        const unsigned long long used = abundance->unique + abundance->ambiguous;
        ab.set("reads_used", Value::integer(static_cast<long long>(used)));
        Value& rc = ab.set("read_categories", Value::object());
        rc.set("unique", Value::integer(static_cast<long long>(abundance->unique)));
        rc.set("ambiguous", Value::integer(static_cast<long long>(abundance->ambiguous)));
        rc.set("uninformative", Value::integer(static_cast<long long>(abundance->uninformative)));
        rc.set("incompatible", Value::integer(static_cast<long long>(abundance->incompatible)));
        Value& hs = ab.set("haplotypes", Value::array());
        for (const AbundanceRow& r : abundance->haplotypes) {
            Value& o = hs.push(Value::object());
            o.set("name", Value::string(r.name));
            o.set("reads", Value::integer(static_cast<long long>(r.reads)));
            o.set("unique_reads", Value::integer(static_cast<long long>(r.unique_reads)));
            o.set("compatible_reads", Value::integer(static_cast<long long>(r.compatible_reads)));
            o.set("em_reads", Value::number(r.em_frequency * static_cast<double>(used)));
            o.set("em_frequency", Value::number(r.em_frequency));
            char b[32];
            snprintf(b, sizeof b, "%.1f", 100.0 * r.em_frequency);
            o.set("em_percentage", Value::string(b));
        }
    }
    return root;
}

inline std::string esc(const std::string& s) {
    std::string o;
    for (char c : s) {
        switch (c) { case '<': o += "&lt;"; break; case '>': o += "&gt;"; break; case '&': o += "&amp;"; break; case '"': o += "&quot;"; break; default: o += c; }
    }
    return o;
}

// HTML from the JSON value only (never from internal state): the 1:1 conversion of doc/JULIET.md:68-69.
inline std::string to_html(const Value& root) {
    static const char* palette[] = {"#e6391e", "#f18f00", "#e8ff0c", "#55e400", "#4fc3ff", "#4a7dff", "#a639ff", "#de0062", "#e6391e", "#8c564b"};
    std::string h;
    h += "<!DOCTYPE html>\n<html><head><meta charset=\"utf-8\"><title>juliet</title>\n<style>\n"
         "body{font-family:Helvetica,Arial,sans-serif;margin:1.5em}details{border-left:3px solid #222;border-radius:8px;padding:.4em 1em;margin:.8em 0}"
         "summary{font-weight:bold;font-size:1.2em;cursor:pointer}table{border-collapse:collapse;margin:1em 0}"
         "th,td{padding:.35em .7em;text-align:center}th.gene{background:#3a3a3a;color:#fff;font-size:1.1em}"
         "tr.var td{background:#ddd;cursor:pointer}tr.var td.cov{background:#bbb}tr.var td.drug{background:#aaa;color:#fff}"
         "td.hap{background:#3a3a3a;min-width:2em;border-left:1px dotted #fff}tr.msa td{border-bottom:1px solid #222;background:#fff}"
         "tr.msa{display:none}tr.msa th{background:#3a3a3a;color:#fff}span.mut{color:#c00030}tt{font-size:1.05em}\n"
         "</style>\n<script>function tg(id){var r=document.getElementsByClassName(id);for(var i=0;i<r.length;i++){r[i].style.display=r[i].style.display=='table-row'?'none':'table-row';}}</script>\n"
         "</head><body>\n";
    const Value* in = root.get("input");
    h += "<details open><summary>Input data</summary><table>";
    if (in) {
        h += "<tr><td style=\"text-align:left\">Timestamp:</td><td style=\"text-align:left\"><tt>" + esc(in->get_string("timestamp")) + "</tt></td></tr>";
        h += "<tr><td style=\"text-align:left\">Input File:</td><td style=\"text-align:left\"><tt>" + esc(in->get_string("input_file")) + "</tt></td></tr>";
        h += "<tr><td style=\"text-align:left\">Command Line Call:</td><td style=\"text-align:left\"><tt>" + esc(in->get_string("command_line")) + "</tt></td></tr>";
        h += "<tr><td style=\"text-align:left\">Juliet Version:</td><td style=\"text-align:left\"><tt>" + esc(in->get_string("juliet_version")) + "</tt></td></tr>";
    }
    h += "</table></details>\n";
    const Value* tc = root.get("target_config");
    h += "<details><summary>Target config</summary>";
    if (tc) {
        h += "<p>Config Version: <tt>" + esc(tc->get_string("version")) + "</tt><br>Reference Name: <tt>" + esc(tc->get_string("referenceName")) +
             "</tt><br>Reference Length: <tt>" + std::to_string(static_cast<long long>(tc->get_number("referenceLength"))) + "</tt><br>Genes:</p><ul>";
        if (const Value* genes = tc->get("genes"))
            for (const Value& g : genes->arr) {
                h += "<li><b>" + esc(g.get_string("name")) + "</b> (" + std::to_string(static_cast<long long>(g.get_number("begin"))) + "-" +
                     std::to_string(static_cast<long long>(g.get_number("end"))) + ")";
                const Value* drms = g.get("drms");
                if (drms && !drms->arr.empty()) {
                    h += "<ul>";
                    for (const Value& d : drms->arr) {
                        h += "<li><tt>" + esc(d.get_string("name")) + ":";
                        if (const Value* ps = d.get("positions")) for (const Value& p : ps->arr) h += " " + esc(p.str);
                        h += "</tt></li>";
                    }
                    h += "</ul>";
                }
                h += "</li>";
            }
        h += "</ul>";
    }
    h += "</details>\n";
    const Value* haps = root.get("haplotypes");
    const size_t nh = haps ? haps->arr.size() : 0;
    const Value* cats = root.get("haplotype_read_categories");
    std::string cat_tip;
    if (cats) {
        cat_tip = "Reported: " + std::to_string(static_cast<long long>(cats->get_number("reported"))) +
                  " | Insufficient coverage: " + std::to_string(static_cast<long long>(cats->get_number("insufficient_coverage"))) +
                  " | Unsuitable: " + std::to_string(static_cast<long long>(cats->get_number("unsuitable"))) +
                  " (gaps " + std::to_string(static_cast<long long>(cats->get_number("unsuitable_gaps"))) +
                  ", heteroduplexes " + std::to_string(static_cast<long long>(cats->get_number("unsuitable_heteroduplex"))) +
                  ", partial " + std::to_string(static_cast<long long>(cats->get_number("unsuitable_partial"))) + ")";
    }
    const std::string refname = tc ? tc->get_string("referenceName") : "";
    h += "<details open><summary>Variant Discovery</summary>\n";
    int rowid = 0;
    if (const Value* genes = root.get("genes"))
        for (const Value& g : genes->arr) {
            const Value* vps = g.get("variant_positions");
            if (!vps || vps->arr.empty()) continue;
            h += "<table><tr><th class=\"gene\" colspan=\"8\">" + esc(g.get_string("name")) + "</th>";
            for (size_t k = 0; k < nh; ++k) h += "<th class=\"gene\" style=\"color:" + std::string(palette[k % 10]) + "\">" + esc(haps->arr[k].get_string("name")) + "</th>";
            h += "</tr><tr><th colspan=\"3\">" + esc(refname.empty() ? "Majority Call" : refname) + "</th><th colspan=\"5\">Sample Variants</th>";
            if (nh) h += "<th colspan=\"" + std::to_string(nh) + "\" title=\"" + esc(cat_tip) + "\">Haplotypes %</th>";
            h += "</tr><tr><th>Codon</th><th>AA</th><th>Pos</th><th>AA</th><th>Codon</th><th>%</th><th>Coverage</th><th>Affected Drugs</th>";
            for (size_t k = 0; k < nh; ++k)
                h += "<th title=\"" + std::to_string(static_cast<long long>(haps->arr[k].get_number("reads"))) + " reads\">" + esc(haps->arr[k].get_string("percentage")) + "</th>";
            h += "</tr>\n";
            for (const Value& vp : vps->arr) {
                const std::string refc = vp.get_string("ref_codon");
                bool first = true;
                const std::string id = "m" + std::to_string(rowid++);
                if (const Value* vaas = vp.get("variant_amino_acids"))
                    for (const Value& va : vaas->arr)
                        if (const Value* vcs = va.get("variant_codons"))
                            for (const Value& vc : vcs->arr) {
                                h += "<tr class=\"var\" onclick=\"tg('" + id + "')\">";
                                if (first) h += "<td><tt>" + esc(refc) + "</tt></td><td>" + esc(vp.get_string("ref_amino_acid")) + "</td><td><b>" +
                                                std::to_string(static_cast<long long>(vp.get_number("ref_position"))) + "</b></td>";
                                else h += "<td></td><td></td><td></td>";
                                first = false;
                                const std::string cod = vc.get_string("codon");
                                std::string cm;
                                for (size_t q = 0; q < cod.size(); ++q)
                                    cm += (q < refc.size() && cod[q] != refc[q]) ? "<span class=\"mut\">" + std::string(1, cod[q]) + "</span>" : std::string(1, cod[q]);
                                h += "<td>" + esc(va.get_string("amino_acid")) + "</td><td><tt>" + cm + "</tt></td><td>" + esc(vc.get_string("percentage")) +
                                     "</td><td class=\"cov\">" + std::to_string(static_cast<long long>(vp.get_number("coverage"))) + "</td><td class=\"drug\">" +
                                     esc(vc.get_string("known_drm")) + "</td>";
                                const Value* hh = vc.get("haplotype_hit");
                                for (size_t k = 0; k < nh; ++k) {
                                    const bool hit = hh && k < hh->arr.size() && hh->arr[k].b;
                                    h += hit ? "<td class=\"hap\" style=\"background:" + std::string(palette[k % 10]) + "\"></td>" : "<td class=\"hap\"></td>";
                                }
                                h += "</tr>\n";
                            }
                if (const Value* msa = vp.get("msa")) {
                    h += "<tr class=\"msa " + id + "\"><td colspan=\"3\"></td><th>Pos</th><th>A</th><th>C</th><th>G</th><th>T</th><th>-</th><th>N</th></tr>";
                    for (const Value& r : msa->arr) {
                        h += "<tr class=\"msa " + id + "\"><td colspan=\"3\"></td><td>" + std::to_string(static_cast<long long>(r.get_number("rel_pos"))) + "</td>";
                        for (const char* s : {"A", "C", "G", "T", "-", "N"}) h += "<td>" + std::to_string(static_cast<long long>(r.get_number(s))) + "</td>";
                        h += "</tr>";
                    }
                    h += "\n";
                }
            }
            h += "</table>\n";
        }
    if (tc && !tc->get_string("databaseVersion").empty()) h += "<p><sup>*</sup>" + esc(tc->get_string("databaseVersion")) + "</p>";
    h += "</details>\n<details><summary>Drug Summaries</summary>";
    if (const Value* ds = root.get("drug_summaries"))
        for (const Value& d : ds->arr) {
            h += "<p><b>" + esc(d.get_string("drug")) + "</b><br>";
            if (const Value* vs = d.get("variants")) for (const Value& v : vs->arr) h += esc(v.str) + "<br>";
            h += "</p>";
        }
    h += "</details>\n";
    if (const Value* lk = root.get("linkage")) {
        char b[64];
        snprintf(b, sizeof b, "%g", lk->get_number("alpha"));
        h += "<details open><summary>Variant Linkage</summary><p>Pairs of variants tested: " +
             std::to_string(static_cast<long long>(lk->get_number("tested_pairs"))) + " (at least " +
             std::to_string(static_cast<long long>(lk->get_number("min_reads"))) + " reads clean at both codons; significance " + b +
             " after Bonferroni)</p>";
        const Value* ps = lk->get("pairs");
        if (ps && !ps->arr.empty()) {
            h += "<table><tr><th>Variant A</th><th>Codon</th><th>Variant B</th><th>Codon</th><th>Reads</th><th>Both</th><th>A only</th>"
                 "<th>B only</th><th>Neither</th><th>D'</th><th>r&sup2;</th><th>p (corrected)</th><th>Relation</th></tr>\n";
            auto cell = [](const Value* v) {
                std::string t;
                if (const Value* ls = v ? v->get("labels") : nullptr)
                    for (const Value& l : ls->arr) t += (t.empty() ? "" : "<br>") + esc(l.str);
                if (t.empty() && v) t = "Pos " + std::to_string(static_cast<long long>(v->get_number("abs_pos")));
                return "<td>" + t + "</td><td><tt>" + esc(v ? v->get_string("codon") : "") + "</tt></td>";
            };
            for (const Value& r : ps->arr) {
                h += "<tr>" + cell(r.get("a")) + cell(r.get("b"));
                for (const char* k : {"reads", "both", "a_only", "b_only", "neither"})
                    h += "<td>" + std::to_string(static_cast<long long>(r.get_number(k))) + "</td>";
                snprintf(b, sizeof b, "<td>%.3f</td><td>%.3f</td><td>%.2e</td>", r.get_number("d_prime"), r.get_number("r2"), r.get_number("pValueCorrected"));
                h += b;
                h += "<td>" + esc(r.get_string("relation")) + "</td></tr>\n";
            }
            h += "</table>";
        }
        h += "</details>\n";
    }
    if (const Value* ab = root.get("haplotype_abundance")) {
        char b[160];
        const Value* rc = ab->get("read_categories");
        auto cat = [&](const char* k) { return std::to_string(static_cast<long long>(rc ? rc->get_number(k) : 0)); };
        snprintf(b, sizeof b, "%lld iterations (%s), log-likelihood %.6g", static_cast<long long>(ab->get_number("iterations")),
                 ab->get("converged") && ab->get("converged")->b ? "converged" : "not converged", ab->get_number("log_likelihood"));
        h += "<details open><summary>Haplotype Abundance</summary><p>Reads used: " +
             std::to_string(static_cast<long long>(ab->get_number("reads_used"))) + " (unique " + cat("unique") + ", ambiguous " + cat("ambiguous") +
             "; set aside: uninformative " + cat("uninformative") + ", incompatible " + cat("incompatible") + ")<br>EM: " + b + "</p>";
        h += "<table><tr><th>Haplotype</th><th>Reads</th><th>Unique</th><th>Compatible</th><th>EM reads</th><th>EM %</th></tr>\n";
        if (const Value* hs = ab->get("haplotypes"))
            for (const Value& r : hs->arr) {
                h += "<tr><td>" + esc(r.get_string("name")) + "</td>";
                for (const char* k : {"reads", "unique_reads", "compatible_reads"}) h += "<td>" + std::to_string(static_cast<long long>(r.get_number(k))) + "</td>";
                snprintf(b, sizeof b, "<td>%.1f</td>", r.get_number("em_reads"));
                h += b;
                h += "<td>" + esc(r.get_string("em_percentage")) + "</td></tr>\n";
            }
        h += "</table></details>\n";
    }
    if (const Value* ib = root.get("indels")) {
        char b[160];
        snprintf(b, sizeof b, "Error model: deletion rate %g, insertion rate %g", ib->get_number("deletion_rate"), ib->get_number("insertion_rate"));
        h += "<details open><summary>In-frame Insertions and Deletions</summary><p>" + std::string(b) + "</p>";
        const Value* cs = ib->get("calls");
        if (cs && !cs->arr.empty()) {
            h += "<table><tr><th>Gene</th><th>Indel</th><th>Pos</th><th>Inserted</th><th>%</th><th>Count</th><th>Coverage</th>"
                 "<th>p (corrected)</th><th>Affected Drugs</th></tr>\n";
            for (const Value& r : cs->arr) {
                snprintf(b, sizeof b, "<td>%.2e</td>", r.get_number("pValueCorrected"));
                h += "<tr><td>" + esc(r.get_string("gene")) + "</td><td>" + esc(r.get_string("label")) + "</td><td>" +
                     std::to_string(static_cast<long long>(r.get_number("abs_pos"))) + "</td><td><tt>" + esc(r.get_string("inserted")) + "</tt></td><td>" +
                     esc(r.get_string("percentage")) + "</td><td>" + std::to_string(static_cast<long long>(r.get_number("count"))) + "</td><td>" +
                     std::to_string(static_cast<long long>(r.get_number("coverage"))) + "</td>" + b + "<td>" + esc(r.get_string("known_drm")) + "</td></tr>\n";
            }
            h += "</table>";
        }
        h += "</details>\n";
    }
    h += "</body></html>\n";
    return h;
}

}  // namespace msreport
