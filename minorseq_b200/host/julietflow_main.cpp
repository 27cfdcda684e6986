// julietflow_main.cpp -- `julietflow -i <ccs.bam> -r <reference.fasta> [-c <config>] [-k] [--device n]`: from unaligned CCS
// reads to juliet's report, running the sibling binaries of this directory in the documented order (SURVEY §3.4, blasr's
// two steps done by `align`):
//   1. align  ccs reference          -> tmp/<stem>/<stem>.ref.bam
//   2. fuse   <stem>.ref.bam         -> tmp/<stem>/<stem>.consensus.fasta
//   3. align  ccs consensus          -> tmp/<stem>/<stem>.consensus.bam
//   4. cleric <stem>.consensus.bam consensus reference -> tmp/<stem>/<stem>.cleric.bam
//   5. juliet [-c config] <stem>.cleric.bam -> <stem>.json, <stem>.html (working directory)
// stem = the input's file name without ".bam", then without ".ccs" (restatement choice U17).  Each step is fork/exec with an
// argument vector (no shell); its stderr passes through, and a failing step stops the flow with a non-zero exit.  The
// intermediates are removed at the end unless -k is given.
#include <sys/stat.h>
#include <sys/wait.h>
#include <unistd.h>
#include <cerrno>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

static void die(const std::string& m) {
    fprintf(stderr, "julietflow: %s\n", m.c_str());
    exit(1);
}

static std::string self_dir() {
    char buf[PATH_MAX];
    const ssize_t n = readlink("/proc/self/exe", buf, sizeof(buf) - 1);
    if (n <= 0) die("cannot locate the julietflow binary");
    std::string p(buf, static_cast<size_t>(n));
    return p.substr(0, p.rfind('/'));
}

static bool ends_with(const std::string& s, const std::string& e) {
    return s.size() >= e.size() && s.compare(s.size() - e.size(), e.size(), e) == 0;
}

static void run(const std::string& dir, const std::string& step, std::vector<std::string> args) {
    const std::string prog = dir + "/" + args[0];
    std::vector<char*> argv;
    for (std::string& a : args) argv.push_back(&a[0]);
    argv.push_back(nullptr);
    fflush(nullptr);
    const pid_t pid = fork();
    if (pid < 0) die(std::string("fork failed: ") + strerror(errno));
    if (pid == 0) {
        execv(prog.c_str(), argv.data());
        fprintf(stderr, "julietflow: cannot run %s: %s\n", prog.c_str(), strerror(errno));
        _exit(127);
    }
    int st = 0;
    while (waitpid(pid, &st, 0) < 0)
        if (errno != EINTR) die(std::string("waitpid failed: ") + strerror(errno));
    if (!WIFEXITED(st) || WEXITSTATUS(st) != 0)
        die("step " + step + " (" + args[0] + ") failed" + (WIFEXITED(st) ? " with exit code " + std::to_string(WEXITSTATUS(st)) : " on a signal"));
}

static void mkdir_p(const std::string& p) {
    if (mkdir(p.c_str(), 0777) != 0 && errno != EEXIST) die("cannot create " + p + ": " + strerror(errno));
}

int main(int argc, char** argv) {
    std::string in, ref, config, device;
    bool keep = false;
    const char* usage = "Usage: julietflow -i <ccs.bam> -r <reference.fasta> [-c <config>] [-k] [--device n]";
    for (int i = 1; i < argc; ++i) {
        const std::string a = argv[i];
        auto need = [&](const char* name) -> std::string {
            if (i + 1 >= argc) die(std::string("option ") + name + " needs a value");
            return argv[++i];
        };
        if (a == "-h" || a == "--help") { puts(usage); return 0; }
        else if (a == "-i") in = need("-i");
        else if (a == "-r") ref = need("-r");
        else if (a == "-c" || a == "--config") config = need("-c");
        else if (a == "-k") keep = true;
        else if (a == "--device") device = need("--device");
        else die("unknown argument " + a + "\n" + usage);
    }
    if (in.empty() || ref.empty()) die(std::string("-i and -r are required\n") + usage);
    struct stat sb;
    if (stat(in.c_str(), &sb) != 0) die("cannot read " + in);
    if (stat(ref.c_str(), &sb) != 0) die("cannot read " + ref);
    if (!config.empty() && config.find('/') != std::string::npos && stat(config.c_str(), &sb) != 0) die("cannot read " + config);

    std::string stem = in.substr(in.rfind('/') == std::string::npos ? 0 : in.rfind('/') + 1);
    if (ends_with(stem, ".bam")) stem.resize(stem.size() - 4);
    if (ends_with(stem, ".ccs")) stem.resize(stem.size() - 4);
    if (stem.empty()) die("cannot derive an output name from " + in);
    const std::string tmp = "tmp/" + stem, base = tmp + "/" + stem;
    mkdir_p("tmp");
    mkdir_p(tmp);
    const std::string bin = self_dir();
    std::vector<std::string> dev;
    if (!device.empty()) dev = {"--device", device};
    auto with_dev = [&](std::vector<std::string> v) {
        v.insert(v.begin() + 1, dev.begin(), dev.end());
        return v;
    };
    const std::string ref_bam = base + ".ref.bam", cons = base + ".consensus.fasta", cons_bam = base + ".consensus.bam",
                      cleric_bam = base + ".cleric.bam";
    run(bin, "1/5", with_dev({"align", in, ref, ref_bam}));
    run(bin, "2/5", with_dev({"fuse", ref_bam, cons}));
    run(bin, "3/5", with_dev({"align", in, cons, cons_bam}));
    run(bin, "4/5", with_dev({"cleric", cons_bam, cons, ref, cleric_bam}));
    std::vector<std::string> jl = {"juliet"};
    if (!config.empty()) jl.insert(jl.end(), {"-c", config});
    jl.insert(jl.end(), {cleric_bam, stem + ".json", stem + ".html"});
    run(bin, "5/5", with_dev(jl));
    if (!keep) {
        for (const std::string& f : {ref_bam, cons, cons_bam, cleric_bam}) unlink(f.c_str());
        rmdir(tmp.c_str());
        rmdir("tmp");        // only when nothing else is in it
    }
    return 0;
}
