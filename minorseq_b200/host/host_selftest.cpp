// host_selftest.cpp -- CPU-only checks of the C++ host layer (no GPU calls): BAM write/read round trip,
// aux tags, target-config JSON + DRM grammar, report JSON -> HTML, the rank and capacity helpers.  Exit code 0 = all good.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>
#include <zlib.h>
#include "bgzf_bam.hpp"
#include "host_common.hpp"
#include "json.hpp"
#include "report.hpp"
#include "target_config.hpp"

// the one library function the helpers under test reach (their error message); the self test runs without the library
extern "C" const char* ms_last_error(const ms_handle*) { return "fake library error"; }

#define REQUIRE(c)                                                          \
    do {                                                                    \
        if (!(c)) { fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } \
    } while (0)

int main(int argc, char** argv) {
    const std::string tmp = argc > 1 ? argv[1] : "/tmp/ms_selftest.bam";
    {   // ---- BAM writer: bin, mate fields, limits of the fixed-width fields, aux tag removal
        REQUIRE(msbam::BamWriter::reg2bin(0, 1) == 4681 && msbam::BamWriter::reg2bin(0, 1 << 14) == 4681);
        REQUIRE(msbam::BamWriter::reg2bin(0, (1 << 14) + 1) == 585 && msbam::BamWriter::reg2bin(1 << 14, (1 << 14) + 10) == 4682);
        REQUIRE(msbam::BamWriter::reg2bin(0, 1 << 29) == 0 && msbam::BamWriter::reg2bin((1 << 26) - 1, (1 << 26) + 1) == 0);
        msbam::Record r;
        r.ref_id = 0; r.pos = 16380; r.flag = 0x1 | 0x40; r.mapq = 7; r.name = "pair/1";
        r.next_ref_id = 0; r.next_pos = 20000; r.tlen = 3700;
        r.cigar = {(5u << 4) | 4u, (10u << 4) | 7u, (3u << 4) | 2u, (2u << 4) | 1u, (7u << 4) | 8u};      // 5S 10= 3D 2I 7X: 20 reference bases
        r.seq = std::string(24, 'A');
        std::vector<uint8_t> b;
        msbam::BamWriter::encode(r, b);
        msbam::Record back;
        msbam::BamReader::parse_record(b.data() + 4, static_cast<uint32_t>(b.size() - 4), back);
        REQUIRE(back.next_ref_id == 0 && back.next_pos == 20000 && back.tlen == 3700 && back.mapq == 7 && back.flag == (0x1 | 0x40));
        REQUIRE((b[4 + 10] | (b[4 + 11] << 8)) == 585);        // [16380, 16400) crosses a 16 kb boundary: a 128 kb bin
        r.pos = 100;
        b.clear();
        msbam::BamWriter::encode(r, b);
        REQUIRE((b[4 + 10] | (b[4 + 11] << 8)) == 4681);
        msbam::Record unplaced;
        unplaced.name = "u"; unplaced.flag = 4; unplaced.seq = "ACGT";
        b.clear();
        msbam::BamWriter::encode(unplaced, b);
        REQUIRE((b[4 + 10] | (b[4 + 11] << 8)) == 4680);
        bool threw = false;
        msbam::Record longname = r;
        longname.name.assign(255, 'x');
        try { b.clear(); msbam::BamWriter::encode(longname, b); } catch (const msbam::Error&) { threw = true; }
        REQUIRE(threw);
        longname.name.assign(254, 'x');
        b.clear();
        msbam::BamWriter::encode(longname, b);
        msbam::BamReader::parse_record(b.data() + 4, static_cast<uint32_t>(b.size() - 4), back);
        REQUIRE(back.name.size() == 254);
        threw = false;
        msbam::Record manyops = r;
        manyops.cigar.assign(65536, (1u << 4) | 7u);
        manyops.seq.assign(65536, 'C');
        try { b.clear(); msbam::BamWriter::encode(manyops, b); } catch (const msbam::Error&) { threw = true; }
        REQUIRE(threw);
        // the parallel whole-file writer reports the same error to its caller instead of terminating on a worker thread
        threw = false;
        try { msbam::write_bam_parallel(tmp, "@HD\tVN:1.5\n", {{"ref", 1000}}, {&r, &manyops, &r}, 3); } catch (const msbam::Error&) { threw = true; }
        REQUIRE(threw);
        threw = false;
        try { msbam::write_bam_parallel("/nonexistent-dir/x.bam", "@HD\tVN:1.5\n", {{"ref", 1000}}, {&r}, 2); } catch (const msbam::Error&) { threw = true; }
        REQUIRE(threw);
        std::vector<uint8_t> aux;
        msbam::BamWriter::aux_string(aux, "MD", "10A5");
        msbam::BamWriter::aux_float(aux, "rq", 0.5f);
        aux.insert(aux.end(), {'N', 'M', 'C', 3});
        msbam::BamWriter::aux_string(aux, "sq", "III");
        aux.insert(aux.end(), {'z', 'b', 'B', 's', 2, 0, 0, 0, 1, 0, 2, 0});
        std::vector<uint8_t> want;
        msbam::BamWriter::aux_float(want, "rq", 0.5f);
        msbam::BamWriter::aux_string(want, "sq", "III");
        want.insert(want.end(), {'z', 'b', 'B', 's', 2, 0, 0, 0, 1, 0, 2, 0});
        msbam::strip_tags(aux, {"NM", "MD"});
        REQUIRE(aux == want);
        std::vector<uint8_t> broken = want;
        broken.pop_back();                          // a cut 'B' array: left alone
        const std::vector<uint8_t> before = broken;
        msbam::strip_tags(broken, {"rq"});
        REQUIRE(broken == before);
    }
    {   // ---- BAM round trip over several BGZF blocks
        msbam::BamWriter w(tmp, "@HD\tVN:1.5\tSO:coordinate\n@SQ\tSN:ref\tLN:1000\n", {{"ref", 1000}});
        for (int i = 0; i < 3000; ++i) {
            msbam::Record r;
            r.ref_id = 0; r.pos = i % 50; r.flag = (i % 7 == 0) ? 0x100 : (i % 5 == 0 ? 0x10 : 0); r.mapq = 60;
            r.name = "m/" + std::to_string(i) + "/ccs";
            r.cigar = {(10u << 4) | 7u, (2u << 4) | 1u, (1u << 4) | 8u, (3u << 4) | 2u, (20u << 4) | 7u};
            r.seq = "ACGTACGTACGGTACGTACGTACGTACGTACGT";
            r.qual.assign(r.seq.size(), 40);
            msbam::BamWriter::aux_string(r.aux, "sq", std::string(r.seq.size(), i % 3 ? 'I' : '+'));
            msbam::BamWriter::aux_float(r.aux, "rq", 0.999f);
            w.write(r);
        }
        w.close();
        msbam::BamReader rd(tmp);
        REQUIRE(rd.refs().size() == 1 && rd.refs()[0].name == "ref" && rd.refs()[0].length == 1000);
        REQUIRE(rd.header_text().find("SN:ref") != std::string::npos);
        msbam::Record r;
        int n = 0;
        while (rd.next(r)) {
            REQUIRE(r.name == "m/" + std::to_string(n) + "/ccs");
            REQUIRE(r.pos == n % 50 && r.cigar.size() == 5 && (r.cigar[1] & 15u) == 1u && (r.cigar[1] >> 4) == 2u);
            REQUIRE(r.seq == "ACGTACGTACGGTACGTACGTACGTACGTACGT" && r.qual.size() == r.seq.size() && r.qual[0] == 40);
            std::vector<int> sq = r.tag_per_base("sq");
            REQUIRE(sq.size() == r.seq.size() && sq[0] == (n % 3 ? 'I' - 33 : '+' - 33));
            double rq = 0;
            REQUIRE(r.tag_number("rq", rq) && rq > 0.998 && rq < 1.0);
            REQUIRE(r.tag_per_base("zz").empty());
            ++n;
        }
        REQUIRE(n == 3000);
        // the whole-file path the tools use (parallel inflate with the project's decoder, record index, parse) sees the
        // same records as the sequential zlib reader -- with either decoder
        for (int use_zlib = 0; use_zlib < 2; ++use_zlib) {
            if (use_zlib) setenv("MS_ZLIB_INFLATE", "1", 1); else unsetenv("MS_ZLIB_INFLATE");
            const msbam::Bytes u = msbam::inflate_file(tmp, 3);
            const msbam::BamIndexed bx = msbam::index_stream(u);
            REQUIRE(bx.refs.size() == 1 && bx.refs[0].name == "ref" && bx.records.size() == 3000);
            msbam::BamReader again(tmp);
            msbam::Record a, b;
            for (size_t k = 0; k < bx.records.size(); ++k) {
                REQUIRE(again.next(a));
                msbam::BamReader::parse_record(u.data() + bx.records[k].first, bx.records[k].second, b);
                REQUIRE(a.name == b.name && a.pos == b.pos && a.flag == b.flag && a.cigar == b.cigar && a.seq == b.seq && a.qual == b.qual && a.aux == b.aux);
            }
        }
        unsetenv("MS_ZLIB_INFLATE");
        // truncated and corrupted files must end in msbam::Error, never in an out-of-bounds read: cut the file at many
        // lengths, shrink a block's BSIZE below its header size (would wrap the deflate length), inflate XLEN past the file end
        {
            FILE* f = fopen(tmp.c_str(), "rb");
            REQUIRE(f != nullptr);
            std::vector<uint8_t> whole;
            for (int ch; (ch = fgetc(f)) != EOF;) whole.push_back(static_cast<uint8_t>(ch));
            fclose(f);
            REQUIRE(whole.size() > 1000);
            const std::string bad = tmp + ".bad";
            auto attempt = [&](const std::vector<uint8_t>& bytes) -> int {      // 0 = loaded, 1 = rejected with msbam::Error
                FILE* g = fopen(bad.c_str(), "wb");
                if (!g) return -1;
                if (!bytes.empty()) fwrite(bytes.data(), 1, bytes.size(), g);
                fclose(g);
                try {
                    const msbam::Bytes u = msbam::inflate_file(bad, 2);
                    const msbam::BamIndexed bx = msbam::index_stream(u);
                    msbam::Record rec;
                    for (const auto& rr : bx.records) msbam::BamReader::parse_record(u.data() + rr.first, rr.second, rec);
                    return 0;
                } catch (const msbam::Error&) { return 1; } catch (const std::exception&) { return 1; }
            };
            for (size_t cut : {size_t(1), size_t(11), size_t(17), size_t(18), size_t(19), size_t(30), whole.size() / 3, whole.size() / 2, whole.size() - 29, whole.size() - 1}) {
                std::vector<uint8_t> part(whole.begin(), whole.begin() + static_cast<long>(cut));
                REQUIRE(attempt(part) >= 0);          // either outcome is fine, a crash is not
            }
            std::vector<uint8_t> v = whole;
            v[16] = 5; v[17] = 0;                     // BSIZE = 5: shorter than header + trailer
            REQUIRE(attempt(v) == 1);
            v = whole;
            v[10] = 0xff; v[11] = 0xff;               // XLEN = 65535: subfields would run far past the first block
            REQUIRE(attempt(v) == 1);
            v = whole;
            v.resize(40);                             // header says a full block follows, the file ends
            REQUIRE(attempt(v) == 1);
            remove(bad.c_str());
            // aux fields whose value runs past the record: never found, never read
            msbam::Record cr;
            cr.aux = {'d', 'q', 'B', 'C', 0xff, 0xff, 0xff, 0x7f, 1, 2, 3};       // B array claiming 2^31 elements
            REQUIRE(cr.find_tag("dq") == nullptr && cr.tag_per_base("dq").empty());
            cr.aux = {'r', 'q', 'f', 0, 0};                                       // float cut short
            double dummy = 0;
            REQUIRE(!cr.tag_number("rq", dummy));
            cr.aux = {'s', 'q', 'Z', 'I', 'I'};                                   // string without its terminator
            REQUIRE(cr.find_tag("sq") == nullptr);
        }
        // the parallel whole-file writer (cleric) produces a BAM the sequential reader reads back record for record
        {
            std::vector<msbam::Record> recs;
            msbam::BamReader src(tmp);
            msbam::Record r2;
            while (src.next(r2)) recs.push_back(r2);
            std::vector<const msbam::Record*> ptrs;
            for (const auto& x : recs) ptrs.push_back(&x);
            const std::string tmp2 = tmp + ".parallel.bam";
            msbam::write_bam_parallel(tmp2, "@HD\tVN:1.5\n@SQ\tSN:other\tLN:777\n", {{"other", 777}}, ptrs, 5);
            msbam::BamReader back(tmp2);
            REQUIRE(back.refs().size() == 1 && back.refs()[0].name == "other" && back.refs()[0].length == 777);
            size_t k = 0;
            while (back.next(r2)) {
                REQUIRE(k < recs.size());
                const msbam::Record& w0 = recs[k++];
                REQUIRE(r2.name == w0.name && r2.pos == w0.pos && r2.flag == w0.flag && r2.cigar == w0.cigar && r2.seq == w0.seq && r2.qual == w0.qual && r2.aux == w0.aux);
            }
            REQUIRE(k == recs.size());
            remove(tmp2.c_str());
        }
    }
    {   // ---- the project's DEFLATE decoder against zlib: every level and strategy, sizes around the edge cases
        uint64_t x = 88172645463325252ULL;
        auto rnd = [&]() { x ^= x << 13; x ^= x >> 7; x ^= x << 17; return x; };
        int tested = 0;
        for (int trial = 0; trial < 400; ++trial) {
            const size_t n = trial < 8 ? static_cast<size_t>(trial) : static_cast<size_t>(rnd() % 70000);
            std::vector<uint8_t> data(n);
            const int kind = trial % 5;            // random bytes / 4-letter text / long runs / BAM-like mix / all zero
            for (size_t i = 0; i < n; ++i) {
                switch (kind) {
                case 0: data[i] = static_cast<uint8_t>(rnd()); break;
                case 1: data[i] = "ACGT"[rnd() & 3]; break;
                case 2: data[i] = static_cast<uint8_t>((i / (1 + trial % 97)) & 0xff); break;
                case 3: data[i] = (i % 1000 < 500) ? "ACGT"[rnd() & 3] : static_cast<uint8_t>(33 + rnd() % 60); break;
                default: data[i] = 0;
                }
            }
            const int level = trial % 10, strategy = (trial / 10) % 5;     // Z_DEFAULT, FILTERED, HUFFMAN_ONLY, RLE, FIXED
            std::vector<uint8_t> comp(compressBound(static_cast<uLong>(n)) + 64);
            z_stream zs;
            memset(&zs, 0, sizeof zs);
            REQUIRE(deflateInit2(&zs, level, Z_DEFLATED, -15, 8, strategy) == Z_OK);
            zs.next_in = data.data(); zs.avail_in = static_cast<uInt>(n);
            zs.next_out = comp.data(); zs.avail_out = static_cast<uInt>(comp.size());
            REQUIRE(deflate(&zs, Z_FINISH) == Z_STREAM_END);
            const size_t clen = zs.total_out;
            deflateEnd(&zs);
            std::vector<uint8_t> back(n + 1, 0xAB);
            REQUIRE(msinflate::fast_inflate(comp.data(), clen, back.data(), n));
            REQUIRE((n == 0 || memcmp(back.data(), data.data(), n) == 0) && back[n] == 0xAB);
            // wrong expected size and truncated input must be refused, not crash
            if (n > 0) {
                REQUIRE(!msinflate::fast_inflate(comp.data(), clen, back.data(), n - 1));
                REQUIRE(!msinflate::fast_inflate(comp.data(), clen / 2, back.data(), n));
            }
            ++tested;
        }
        REQUIRE(tested == 400);
        // carry-less-multiply CRC-32 against zlib's, all lengths around the 16/64-byte boundaries and unaligned starts
        for (int t = 0; t < 1500; ++t) {
            const size_t n = t < 300 ? static_cast<size_t>(t) : static_cast<size_t>(rnd() % 70000);
            std::vector<uint8_t> buf(n + 3);
            for (auto& c : buf) c = static_cast<uint8_t>(rnd());
            const uint8_t* p = buf.data() + t % 3;
            REQUIRE(mscrc::crc32(p, n) == static_cast<uint32_t>(crc32(crc32(0L, Z_NULL, 0), p, static_cast<uInt>(n))));
        }
        // garbage input never reads or writes out of bounds (run under the sanitizers in development) and is refused or
        // caught by the caller's CRC check
        std::vector<uint8_t> junk(4096), sink(65536);
        for (int t = 0; t < 200; ++t) {
            for (auto& c : junk) c = static_cast<uint8_t>(rnd());
            (void)msinflate::fast_inflate(junk.data(), junk.size(), sink.data(), 1 + rnd() % sink.size());
        }
    }
    {   // ---- rich-QV filter (doc/JULIET.md:256-259): raw-byte implementation against the per-base accessor
        msbam::Record r;
        r.seq = "ACGTACGTACGTACGTACGTACGTA";
        const size_t n = r.seq.size();
        std::string dq(n, 'I'), sq(n, 'I');
        dq[2] = '+'; dq[7] = '4'; sq[7] = '5'; sq[20] = '!';            // QVs 10, 19 | 20, 0
        msbam::BamWriter::aux_string(r.aux, "dq", dq);
        msbam::BamWriter::aux_string(r.aux, "sq", sq);
        r.aux.insert(r.aux.end(), {'i', 'q', 'B', 'C'});                  // a B:C array track, one low value
        msbam::detail::put32(r.aux, static_cast<uint32_t>(n));
        for (size_t i = 0; i < n; ++i) r.aux.push_back(i == 11 ? 3 : 60);
        msbam::BamWriter::aux_string(r.aux, "xq", std::string(n - 1, '!'));   // wrong length: ignored
        mshost::QvFilter qv;
        qv.tags = {"dq", "iq", "sq", "xq", "zz"};
        for (int rev = 0; rev < 2; ++rev) {
            r.flag = rev ? 0x10 : 0;
            std::vector<uint8_t> want(n, 0), got;
            for (const std::string& t : qv.tags) {
                const std::vector<int> tr = r.tag_per_base(t.c_str());
                if (tr.size() != n) continue;
                for (size_t i = 0; i < n; ++i) if (tr[i] < qv.threshold) want[rev ? n - 1 - i : i] = 1;
            }
            REQUIRE(qv.apply(r, got) && got == want);
            REQUIRE(want[rev ? n - 1 - 2 : 2] == 1 && want[rev ? n - 1 - 7 : 7] == 1 && want[rev ? n - 1 - 11 : 11] == 1 && want[rev ? n - 1 - 20 : 20] == 1);
            size_t ones = 0; for (uint8_t m : want) ones += m;
            REQUIRE(ones == 4);
        }
        std::vector<uint8_t> m;
        mshost::QvFilter off; off.threshold = 0;
        REQUIRE(!off.apply(r, m));
        msbam::Record bare; bare.seq = "ACGT";
        REQUIRE(!qv.apply(bare, m));                                     // no tracks: no filtering
    }
    {   // ---- target config: the example of doc/JULIET.md:138-157 and the DRM grammar of :167-176
        const std::string text = R"({"genes":[{"begin":2550,"drms":[{"name":"fancy drug","positions":["M41L"]},
            {"name":"ATV/r","positions":["V32I","L33","46IL","I54VTALM","V82ATFS","84"]}],"end":2700,"name":"Reverse Transcriptase"}],
            "referenceName":"my seq","referenceSequence":"TGGAAGGGCT","version":"v","databaseVersion":"DrugDB"})";
        mscfg::TargetConfig c = mscfg::from_json(msjson::Parser(text).parse());
        REQUIRE(c.genes.size() == 1 && c.genes[0].begin == 2550 && c.genes[0].end == 2700 && c.genes[0].drms.size() == 2);
        const auto& atv = c.genes[0].drms[1].positions;
        REQUIRE(atv.size() == 6);
        REQUIRE(mscfg::drm_matches(atv[0], 32, 'V', 'I') && !mscfg::drm_matches(atv[0], 32, 'V', 'L') && !mscfg::drm_matches(atv[0], 32, 'A', 'I'));
        REQUIRE(mscfg::drm_matches(atv[1], 33, 'L', 'F') && mscfg::drm_matches(atv[1], 33, 'L', 'X'));          // "L33": any mutant
        REQUIRE(mscfg::drm_matches(atv[2], 46, 'M', 'I') && mscfg::drm_matches(atv[2], 46, 'Q', 'L') && !mscfg::drm_matches(atv[2], 46, 'M', 'V'));
        REQUIRE(mscfg::drm_matches(atv[3], 54, 'I', 'M') && !mscfg::drm_matches(atv[3], 54, 'I', 'K'));
        REQUIRE(mscfg::drm_matches(atv[5], 84, 'I', 'V') && mscfg::drm_matches(atv[5], 84, 'Z', 'Q') && !mscfg::drm_matches(atv[5], 85, 'I', 'V'));
        const mscfg::DrmPosition p1 = mscfg::parse_drm_position("103"), p2 = mscfg::parse_drm_position("M130"), p3 = mscfg::parse_drm_position("103LG");
        REQUIRE(p1.ref_aa == '*' && p1.pos == 103 && p1.mut_aas.empty());
        REQUIRE(p2.ref_aa == 'M' && p2.pos == 130 && p2.mut_aas.empty());
        REQUIRE(p3.ref_aa == '*' && p3.pos == 103 && p3.mut_aas == "LG");
        REQUIRE(mscfg::load("HIV").genes.size() == 8 && mscfg::load("HIV").genes[7].drms.size() == 7);
        REQUIRE(mscfg::load("ABL1").genes[0].drms.size() == 4);
        REQUIRE(mscfg::translate(0) == 'K' && mscfg::translate(63) == 'F' && mscfg::translate(16 * 3 + 4 * 2 + 0) == 'X');   // AAA, TTT, TGA
        REQUIRE(mscfg::translate(16 * 0 + 4 * 3 + 2) == 'M' && mscfg::translate(16 * 0 + 4 * 2 + 0) == 'R');                   // ATG, AGA
    }
    {   // ---- report: formatting rules read off the screenshots, JSON -> HTML
        REQUIRE(msreport::perc2(1.107) == "1.1" && msreport::perc2(0.912) == "0.91" && msreport::perc2(98.4) == "98" && msreport::perc2(100.0) == "100");
        REQUIRE(msreport::perc1(92.52) == "92.5" && msreport::perc1(1.0) == "1" && msreport::perc1(0.74) == "0.7");
        msreport::Report in;
        in.timestamp = "2017-05-16T11:00:12.187Z"; in.input_file = "in.bam"; in.command_line = "juliet in.bam out.json"; in.version = "test";
        in.cfg = mscfg::load("HIV");
        in.genes = in.cfg.genes;
        in.L = 9719;
        std::vector<msreport::VariantRow>& rows = in.variants;
        rows.resize(1);
        rows[0].gene = 7; rows[0].aa_pos = 46; rows[0].col = 2252 + 45 * 3; rows[0].ref_codon = 14; rows[0].codon = 12;  // ATG -> ATA (M46I)
        rows[0].count = 28; rows[0].coverage = 2529; rows[0].expected = 1; rows[0].ntests = 99; rows[0].pvalue = 5.2e-8;
        rows[0].drugs = {"ATV/r", "NFV"};
        rows[0].haplotype_hit = {false, true};
        in.col_counts.assign(9719 * 8, 7);
        in.phasing = true;
        std::vector<msreport::HaplotypeRow>& haps = in.haplotypes;
        haps.resize(2);
        haps[0].name = "A"; haps[0].reads = 900; haps[0].frequency = 0.9; haps[0].codons = {""}; haps[0].read_names = {"r1", "r2"};
        haps[1].name = "B"; haps[1].reads = 100; haps[1].frequency = 0.1; haps[1].codons = {"ATA"}; haps[1].read_names = {"r3"};
        const unsigned long long ctr[6] = {1000, 5, 20, 3, 15, 4};
        std::copy(ctr, ctr + 6, in.counters);
        const msjson::Value rep = msreport::build(in);
        const std::string js = msjson::dump(rep);
        const msjson::Value back = msjson::Parser(js).parse();
        REQUIRE(msjson::dump(back) == js);                                                   // writer/parser round trip
        REQUIRE(js.find("\"haplotype_hit\": [false, true]") != std::string::npos);
        REQUIRE(js.find("\"percentage\": \"1.1\"") != std::string::npos && js.find("\"known_drm\": \"ATV/r + NFV\"") != std::string::npos);
        REQUIRE(js.find("\"rel_pos\": -3") != std::string::npos && js.find("\"rel_pos\": 5") != std::string::npos);
        const std::string html = msreport::to_html(back);
        for (const char* needle : {"Input data", "Target config", "Variant Discovery", "Drug Summaries", "Haplotypes %", "ATV/r + NFV", "2017-05-16T11:00:12.187Z", "M46I"})
            REQUIRE(html.find(needle) != std::string::npos);
    }
    {   // ---- the rank and capacity helpers of the binaries, with fake library calls
        // fetch: both ways of the ABI to say "too small", a list that needs two growths, a failure
        int calls = 0;
        auto grows_by_status = [&](int* out, int64_t cap, int64_t* n) {   // MS_ERR_CAPACITY with the size it needs: 10, then 50
            ++calls;
            *n = calls == 1 ? 10 : 50;
            if (cap < *n) return static_cast<int>(MS_ERR_CAPACITY);
            for (int64_t i = 0; i < *n; ++i) out[i] = static_cast<int>(i);
            return static_cast<int>(MS_OK);
        };
        std::vector<int> got = mshost::fetch<int>(nullptr, "grows_by_status", 4, grows_by_status);
        REQUIRE(calls == 3 && got.size() == 50 && got[49] == 49);
        calls = 0;
        std::vector<int64_t> caps;
        auto grows_by_count = [&](int* out, int64_t cap, int64_t* n) {   // MS_OK with n > cap (out holds the first cap)
            caps.push_back(cap);
            *n = ++calls == 1 ? 7 : 20;
            for (int64_t i = 0; i < std::min(cap, *n); ++i) out[i] = static_cast<int>(100 + i);
            return static_cast<int>(MS_OK);
        };
        got = mshost::fetch<int>(nullptr, "grows_by_count", 4, grows_by_count);
        REQUIRE(calls == 3 && caps == std::vector<int64_t>({4, 7, 20}) && got.size() == 20 && got[19] == 119);
        got = mshost::fetch<int>(nullptr, "fits", 4, [](int*, int64_t, int64_t* n) { *n = 3; return static_cast<int>(MS_OK); });
        REQUIRE(got.size() == 3);
        std::string msg;
        try { mshost::fetch<int>(nullptr, "ms_broken", 4, [](int*, int64_t, int64_t*) { return static_cast<int>(MS_ERR_ARG); }); }
        catch (const std::exception& e) { msg = e.what(); }
        REQUIRE(msg == "ms_broken failed: fake library error");
        // for_ranks: every rank runs; of the failing ranks 1 and 2, rank 1's message reaches the caller
        std::vector<int> ran(3, 0);
        msg.clear();
        try {
            mshost::for_ranks(3, [&](int r) {
                ran[r] = 1;
                if (r == 2) throw std::runtime_error("rank 2 failed");
                if (r == 1) {
                    std::this_thread::sleep_for(std::chrono::milliseconds(50));    // rank 2 fails first in time
                    throw std::runtime_error("rank 1 failed");
                }
            });
        } catch (const std::exception& e) { msg = e.what(); }
        REQUIRE(msg == "rank 1 failed" && ran == std::vector<int>({1, 1, 1}));
        REQUIRE(mshost::shard(10, 0, 3).second == 3 && mshost::shard(10, 2, 3).first == 6 && mshost::shard(10, 2, 3).second == 10);
    }
    puts("host selftest ok");
    return 0;
}
