// target_config.hpp -- juliet's target configuration (/root/reference/doc/JULIET.md:109-190).
//
// "The root child genes contains a list of coding regions, with begin and end, the name of the gene, and
// a list of drug resistent mutations drms ... All indices are with respect to the provided alignment
// space, 1-based, begin-inclusive and end-exclusive" (:129-136).  DRM position grammar :167-176.
// Predefined names (:126 `HIV`, `ABL1`; screenshot juliet_input.png also `HIV-PB`): the reference ships
// neither the HXB2 sequence nor the full HIVdb tables, so the built-in HIV config carries exactly what the
// documentation shows (gene intervals and the protease-inhibitor lists of screenshot juliet_target.png)
// and no referenceSequence (calls are then made against the major codon, :133-134); ABL1 is the example
// of :310-340.
#pragma once
#include <fstream>
#include <sstream>
#include <string>
#include <vector>
#include "json.hpp"

namespace mscfg {

// "M103LKA": ref aa (or '*'), position, allowed mutant aas (empty = '*', which also matches an indel there).
// "T69ins" / "69ins": an in-frame insertion after codon 69; "D67del" / "67del": a deletion of codon 67 (restatement choice U19).
enum DrmKind { kDrmSubstitution = 0, kDrmInsertion = 1, kDrmDeletion = 2 };
struct DrmPosition {
    char ref_aa = '*';
    int pos = 0;
    std::string mut_aas;
    std::string text;
    int kind = kDrmSubstitution;
};
struct Drm { std::string name; std::vector<DrmPosition> positions; };
struct Gene { std::string name; int begin = 0, end = 0; std::vector<Drm> drms; };
struct TargetConfig {
    std::vector<Gene> genes;
    std::string reference_name, reference_sequence, version, database_version;
    bool from_user = false;
};

inline DrmPosition parse_drm_position(const std::string& s) {
    DrmPosition p;
    p.text = s;
    size_t i = 0;
    if (i < s.size() && (s[i] < '0' || s[i] > '9')) p.ref_aa = s[i++];
    size_t j = i;
    while (j < s.size() && s[j] >= '0' && s[j] <= '9') ++j;
    if (j == i) throw std::runtime_error("DRM position without a number: " + s);
    p.pos = std::stoi(s.substr(i, j - i));
    p.mut_aas = s.substr(j);
    if (p.mut_aas == "ins" || p.mut_aas == "del") {
        p.kind = p.mut_aas == "ins" ? kDrmInsertion : kDrmDeletion;
        p.mut_aas.clear();
    }
    return p;
}

// does a variant (1-based amino-acid position in the gene, reference aa, variant aa) hit this DRM entry?
inline bool drm_matches(const DrmPosition& p, int aa_pos, char ref_aa, char var_aa) {
    if (p.kind != kDrmSubstitution || p.pos != aa_pos) return false;
    if (p.ref_aa != '*' && p.ref_aa != ref_aa) return false;
    return p.mut_aas.empty() || p.mut_aas.find(var_aa) != std::string::npos;
}

// does an in-frame indel hit this DRM entry?  aa_pos / ref_aa: the deleted codon, or the codon before the insertion
inline bool drm_matches_indel(const DrmPosition& p, int aa_pos, char ref_aa, bool insertion) {
    if (p.pos != aa_pos) return false;
    if (p.ref_aa != '*' && p.ref_aa != ref_aa) return false;
    if (p.kind == kDrmSubstitution) return p.mut_aas.empty();   // a bare position is a wildcard
    return p.kind == (insertion ? kDrmInsertion : kDrmDeletion);
}

inline TargetConfig from_json(const msjson::Value& root) {
    TargetConfig c;
    c.from_user = true;
    c.reference_name = root.get_string("referenceName");
    c.reference_sequence = root.get_string("referenceSequence");
    c.version = root.get_string("version");
    c.database_version = root.get_string("databaseVersion");
    const msjson::Value* genes = root.get("genes");
    if (!genes || genes->kind != msjson::Value::Array) throw std::runtime_error("target config: missing \"genes\"");
    for (const msjson::Value& g : genes->arr) {
        Gene gene;
        gene.name = g.get_string("name");
        gene.begin = static_cast<int>(g.get_number("begin"));
        gene.end = static_cast<int>(g.get_number("end"));
        if (gene.begin < 1 || gene.end <= gene.begin) throw std::runtime_error("target config: bad begin/end for gene " + gene.name);
        if (const msjson::Value* drms = g.get("drms")) {
            for (const msjson::Value& d : drms->arr) {
                Drm drm;
                drm.name = d.get_string("name");
                if (const msjson::Value* ps = d.get("positions"))
                    for (const msjson::Value& p : ps->arr) drm.positions.push_back(parse_drm_position(p.str));
                gene.drms.push_back(drm);
            }
        }
        c.genes.push_back(gene);
    }
    return c;
}

inline Drm make_drm(const std::string& name, const std::string& list) {
    Drm d;
    d.name = name;
    std::istringstream is(list);
    std::string tok;
    while (is >> tok) d.positions.push_back(parse_drm_position(tok));
    return d;
}

inline TargetConfig predefined_hiv() {
    TargetConfig c;
    c.reference_name = "HIV HXB2";
    c.version = "minorseq_b200 built-in: gene intervals and PI lists as shown in the minorseq documentation (juliet_target.png)";
    c.database_version = "partial: protease inhibitors only";
    auto gene = [&](const char* n, int b, int e) { Gene g; g.name = n; g.begin = b; g.end = e; c.genes.push_back(g); };
    gene("5'LTR", 1, 634); gene("p17", 790, 1186); gene("p24", 1186, 1879); gene("p2", 1879, 1921);
    gene("p7", 1921, 2086); gene("p1", 2086, 2134); gene("p6", 2134, 2292); gene("Protease", 2253, 2550);
    Gene& pr = c.genes.back();
    pr.drms.push_back(make_drm("ATV/r", "V32I L33F M46I M46L I47V G48V G48M I50L I54V I54T I54A I54L I54M V82A V82T V82F V82S I84V N88S L90M"));
    pr.drms.push_back(make_drm("DRV/r", "V32I L33F I47V I47A I50V I54L I54M L76V V8F I84V"));
    pr.drms.push_back(make_drm("FPV/r", "V32I L33F M46I M46L I47V I47A I50V I54V I54T I54A I54L I54M L76V V82A V82T V82F V82S I84V L90M"));
    pr.drms.push_back(make_drm("IDV/r", "V32I M46I M46L I47V I54V I54T I54A I54L I54M L76V V82A V82T V82F V82S I84V N88S L90M"));
    pr.drms.push_back(make_drm("NFV", "D30N L33F M46I M46L I47V G48V G48M I54V I54T I54A I54L I54M V82A V82T V82F V82S I84V N88D N88S L90M"));
    pr.drms.push_back(make_drm("SQV/r", "G48V G48M I54V I54T I54A I54L I54M V82A V82T I84V N88S L90M"));
    pr.drms.push_back(make_drm("TPV/r", "V32I L33F M46I M46L I47V I47A I54V I54A I54M V82T V82L I84V"));
    return c;
}

inline TargetConfig predefined_abl1() {
    TargetConfig c;
    c.reference_name = "NM_005157.5";
    c.version = "minorseq_b200 built-in: the ABL1 example of doc/JULIET.md:310-340";
    Gene g;
    g.name = "ABL1"; g.begin = 193; g.end = 3585;
    g.drms.push_back(make_drm("imatinib", "T315AI Y253H E255KV V299L F317AICLV F359CIV"));
    g.drms.push_back(make_drm("dasatinib", "T315AI V299L F317AICLV"));
    g.drms.push_back(make_drm("nilotinib", "T315AI Y253H E255KV F359CIV"));
    g.drms.push_back(make_drm("bosutinib", "T315AI"));
    c.genes.push_back(g);
    return c;
}

// --config <HIV|HIV-PB|ABL1|path.json>; empty = no target config (doc/JULIET.md:182-188)
inline TargetConfig load(const std::string& spec) {
    if (spec == "HIV" || spec == "HIV-PB") return predefined_hiv();
    if (spec == "ABL1") return predefined_abl1();
    std::ifstream in(spec);
    if (!in) throw std::runtime_error("cannot open target config " + spec);
    std::stringstream ss;
    ss << in.rdbuf();
    const std::string text = ss.str();
    return from_json(msjson::Parser(text).parse());
}

inline const char* codon_string(int c, char buf[4]) {
    static const char b[] = "ACGT";
    buf[0] = b[(c >> 4) & 3]; buf[1] = b[(c >> 2) & 3]; buf[2] = b[c & 3]; buf[3] = 0;
    return buf;
}

// standard genetic code; stop codons are reported as 'X' (screenshot juliet_hiv-hiv.png: CGA->TGA, R8X)
inline char translate(int c) {
    static const char ncbi[] = "FFLLSSSSYY**CC*WLLLLPPPPHHQQRRRRIIIMTTTTNNKKSSRRVVVVAAAADDEEGGGG";  // TCAG order
    static const int remap[4] = {2, 1, 3, 0};  // A,C,G,T -> index in TCAG
    const char aa = ncbi[16 * remap[(c >> 4) & 3] + 4 * remap[(c >> 2) & 3] + remap[c & 3]];
    return aa == '*' ? 'X' : aa;
}

}  // namespace mscfg
