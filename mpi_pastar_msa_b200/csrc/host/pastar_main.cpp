// pastar — drop-in CLI for the reference's ./bin/pastar (pastar/msa_pastar_main.cpp:56-193), GPU path.
//
//   pastar [-t N] [-s SHIFT] [-y FZORDER|FSUM|PZORDER|PSUM] [-v] [-h] [--memory_debug] file.fasta
//   new, optional: [-g/--gpus N] [--batch K] [--table_capacity SLOTS] [--max_expansions E] [--metrics_json FILE] [--weight W]
//                  [--incumbent FILE] [--anytime W1,W2,...]
//
// Same flags, exit codes (0 ok, 1 usage / not a regular file, -1 on exception) and stdout format as the reference
// (phase timers, "Final Score:", "Similarity:", wrapped alignment, "Total nodes count:" table).  No MPI: the
// reference's ranks x threads partitions map to GPUs of one box.
#include "pastar_host.hpp"

#include <algorithm>

namespace pastar {

int hash_shift = HASH_SHIFT;
hashType hash_type = HashFZorder;

// read_fasta_file_core, pastar/read_fasta.cpp:8-36: '>' lines and empty lines end a record; no validation
int read_fasta_file(const std::string &name)
{
    try {
        std::ifstream file(name.c_str());
        Sequences *sequences = Sequences::getInstance();
        if (!file.is_open()) {
            std::cout << "Can't open file " << name << std::endl;
            return -1;
        }
        while (!file.eof()) {
            std::string seq;
            while (!file.eof()) {
                std::string buf;
                getline(file, buf);
                if (!buf.empty() && buf.back() == '\r') buf.pop_back();
                if (buf.empty() || buf[0] == '>') break;
                seq.append(buf);
            }
            if (!seq.empty()) sequences->set_seq(seq);
        }
        return 0;
    } catch (std::exception &e) {
        std::cerr << "Reading file fatal error: " << e.what() << std::endl;
    } catch (...) {
        std::cerr << "Unknown fatal error while reading file!\n";
    }
    return -1;
}

static void usage(const char *argv0)
{
    std::cout << "Usage " << argv0 << " [OPTIONS] file.fasta:\n\n"
              << "Options:\n"
              << "  -v [ --version ]              print version string\n"
              << "  -h [ --help ]                 produce help message\n"
              << "  --memory_debug                memory debug option\n\n"
              << "Parallel Options:\n"
              << "  -t [ --threads ] arg          number of threads\n"
              << "  -s [ --hash_shift ] arg (=" << HASH_SHIFT << ")  Hash shift option value\n"
              << "  -y [ --hash_type ] arg (=FZORDER)\n"
              << "                                Hash type [FZORDER|FSUM|PZORDER|PSUM]\n\n"
              << "GPU Options:\n"
              << "  -g [ --gpus ] arg (=1)        hash-owned partitions, one per GPU\n"
              << "  --batch arg                   frontier nodes popped per round\n"
              << "  --table_capacity arg          closed/open table slots\n"
              << "  --max_expansions arg          stop after this many expansions\n"
              << "  --metrics_json arg            write the run's counters (total and per partition) as JSON\n"
              << "  --weight arg                  bounded-suboptimal search: cost at most W (1..16) x the optimum,\n"
              << "                                reported with a certified lower bound\n"
              << "  --incumbent arg               aligned FASTA of a known alignment of the input: find a cheaper one or\n"
              << "                                prove it optimal\n"
              << "  --anytime arg                 comma-separated weights (1..16), one search per weight, each bounded\n"
              << "                                by the best alignment so far (one GPU)\n"
              << std::endl;
}

// msa_options_core, pastar/msa_options.cpp:24-119, without Boost.ProgramOptions
static int options_core(int argc, char *argv[], std::string &filename, PAStarOpt &opt)
{
    std::string hash_read = "FZORDER";
    bool help = false, version = false, memory_debug = false, have_file = false;
    auto value = [&](int &i, const std::string &arg, const char *longname) -> std::string {
        const std::string eq = std::string("--") + longname + "=";
        if (arg.compare(0, eq.size(), eq) == 0) return arg.substr(eq.size());
        if (arg.size() > 2 && arg[0] == '-' && arg[1] != '-') return arg.substr(2); // -t4
        if (i + 1 >= argc) throw std::invalid_argument(std::string("the required argument for option '--") + longname + "' is missing");
        return argv[++i];
    };
    auto is = [](const std::string &a, char s, const char *l) {
        const std::string ll = std::string("--") + l;
        return (a.size() >= 2 && a[0] == '-' && a[1] == s) || a == ll || a.compare(0, ll.size() + 1, ll + "=") == 0;
    };
    // Boost.ProgramOptions' default style lets a long option be shortened to any unambiguous prefix ("--thr 4", "--hash_t=FSUM")
    static const char *const long_names[] = {"version", "help", "memory_debug", "threads", "hash_shift", "hash_type", "gpus",
                                             "batch", "table_capacity", "max_expansions", "metrics_json", "weight",
                                             "incumbent", "anytime"};
    auto canonical = [&](const std::string &arg) -> std::string {
        if (arg.size() < 3 || arg.compare(0, 2, "--") != 0) return arg;
        const size_t eq = arg.find('=');
        const std::string name = arg.substr(2, eq == std::string::npos ? std::string::npos : eq - 2);
        const char *hit = nullptr;
        int hits = 0;
        for (const char *l : long_names) {
            if (name == l) return arg;
            if (!name.empty() && std::string(l).compare(0, name.size(), name) == 0) {
                hit = l;
                hits++;
            }
        }
        if (hits > 1) throw std::invalid_argument("option '--" + name + "' is ambiguous");
        if (hits == 0) throw std::invalid_argument("unrecognised option '--" + name + "'");
        return std::string("--") + hit + (eq == std::string::npos ? "" : arg.substr(eq));
    };
    auto is_long = [](const std::string &a, const char *l) {
        const std::string ll = std::string("--") + l;
        return a == ll || a.compare(0, ll.size() + 1, ll + "=") == 0;
    };
    auto weight_num = [](const std::string &v, const char *longname) { // W in 1..16 as num / 1024, rounded up
        size_t used = 0;
        const double w = std::stod(v, &used);
        if (used != v.size() || !(w >= 1.0 && w <= 16.0))
            throw std::invalid_argument(std::string("the argument for option '--") + longname + "' must be a number in 1..16");
        return (int)std::ceil(w * 1024.0);
    };
    for (int i = 1; i < argc; i++) {
        const std::string a = canonical(argv[i]);
        if (a == "-v" || a == "--version") version = true;
        else if (a == "-h" || a == "--help") help = true;
        else if (a == "--memory_debug") memory_debug = true;
        else if (is(a, 't', "threads")) opt.threads_num = std::stoi(value(i, a, "threads"));
        else if (is(a, 's', "hash_shift")) opt.hash_shift = std::stoi(value(i, a, "hash_shift"));
        else if (is(a, 'y', "hash_type")) hash_read = value(i, a, "hash_type");
        else if (is(a, 'g', "gpus")) opt.gpus = std::stoi(value(i, a, "gpus"));
        else if (is_long(a, "batch")) opt.batch = std::stoll(value(i, a, "batch"));
        else if (is_long(a, "table_capacity")) opt.table_capacity = std::stoll(value(i, a, "table_capacity"));
        else if (is_long(a, "max_expansions")) opt.max_expansions = std::stoll(value(i, a, "max_expansions"));
        else if (is_long(a, "metrics_json")) opt.metrics_json = value(i, a, "metrics_json");
        else if (is_long(a, "weight")) opt.weight_num = weight_num(value(i, a, "weight"), "weight");
        else if (is_long(a, "incumbent")) opt.incumbent = value(i, a, "incumbent");
        else if (is_long(a, "anytime")) {
            const std::string v = value(i, a, "anytime");
            opt.anytime_num.clear();
            for (size_t at = 0;;) {
                const size_t comma = v.find(',', at);
                opt.anytime_num.push_back(weight_num(v.substr(at, comma == std::string::npos ? std::string::npos : comma - at), "anytime"));
                if (comma == std::string::npos) break;
                at = comma + 1;
            }
            if (opt.anytime_num.size() > 64) throw std::invalid_argument("the argument for option '--anytime' has more than 64 weights");
        }
        else if (!a.empty() && a[0] == '-' && a.size() > 1) throw std::invalid_argument("unrecognised option '" + a + "'");
        else {
            filename = a; // file.fasta is position independent
            have_file = true;
        }
    }
    if (hash_read == "FZORDER") opt.hash_type = HashFZorder;
    else if (hash_read == "FSUM") opt.hash_type = HashFSum;
    else if (hash_read == "PZORDER") opt.hash_type = HashPZorder;
    else if (hash_read == "PSUM") opt.hash_type = HashPSum;
    else throw std::invalid_argument("the argument for option '--hash_type' is invalid");
    if (!opt.anytime_num.empty() && opt.weight_num) throw std::invalid_argument("option '--anytime' cannot be combined with '--weight'");
    if (!opt.anytime_num.empty() && opt.gpus != 1) throw std::invalid_argument("option '--anytime' runs on one GPU (--gpus 1)");
    if (version) {
        std::cout << "msa_pastar, version 1.0\n";
        std::exit(0);
    }
    if (help || !have_file) {
        usage(argv[0]);
        return 1;
    }
    struct stat st;
    if (stat(filename.c_str(), &st) != 0 || !S_ISREG(st.st_mode)) {
        std::cout << "File: " << filename << " is not a regular file.\n";
        return 1;
    }
    opt.common_options.force_quit = !memory_debug;
    return 0;
}

int msa_pastar_options(int argc, char *argv[], std::string &filename, PAStarOpt &opt)
{
    try {
        return options_core(argc, argv, filename, opt);
    } catch (std::exception &e) {
        std::cerr << "Invalid argument: " << e.what() << std::endl;
    } catch (...) {
        std::cerr << "Unknown error\n";
    }
    return -1;
}

int get_print_size() // backtrace.cpp:20-35
{
    int size = 80;
    struct winsize w;
    if (!isatty(1)) return std::numeric_limits<int>::max();
    if ((ioctl(0, TIOCGWINSZ, &w) == 0) && (w.ws_col > 1)) size = w.ws_col - 1;
    return size;
}

void print_similarity(const std::vector<std::string> &rows) // backtrace.cpp:135-165
{
    long long total = 0, equal = 0;
    const size_t n = rows.size(), cols = rows.empty() ? 0 : rows[0].size();
    for (size_t c = 0; c < cols; c++)
        for (size_t i = 0; i < n; ++i)
            for (size_t j = i + 1; j < n; ++j) {
                if (rows[i][c] == rows[j][c]) ++equal;
                ++total;
            }
    float percent = (equal * 100) / (float)total;
    std::cout << "Similarity: " << std::fixed << std::setprecision(2) << percent << "%" << std::endl;
}

void print_alignment(const std::vector<std::string> &rows) // backtrace.cpp:171-191
{
    const int size = get_print_size();
    const size_t cols = rows.empty() ? 0 : rows[0].size();
    for (size_t at = 0; at < cols;) {
        const size_t take = std::min<size_t>((size_t)size, cols - at);
        std::cout << std::endl;
        for (size_t j = 0; j < rows.size(); j++) std::cout << rows[j].substr(at, take) << std::endl;
        at += take;
    }
}

// --incumbent FILE: an aligned FASTA (records as read_fasta_file reads them, '-' for gaps) with the input's records in
// the input's order.  Checked here, before any device call: the rows must be of equal length, spell the input sequences
// once their gaps are removed, and hold no column of gaps only.  Returns an empty string or what is wrong.
static std::string read_incumbent(const std::string &name, std::vector<std::string> &rows)
{
    struct stat st;
    if (stat(name.c_str(), &st) != 0 || !S_ISREG(st.st_mode)) return "not a regular file";
    std::ifstream file(name.c_str());
    if (!file.is_open()) return "cannot be opened";
    rows.clear();
    std::string cur, buf;
    while (getline(file, buf)) {
        if (!buf.empty() && buf.back() == '\r') buf.pop_back();
        if (buf.empty() || buf[0] == '>') {
            if (!cur.empty()) rows.push_back(cur);
            cur.clear();
        } else {
            cur += buf;
        }
    }
    if (!cur.empty()) rows.push_back(cur);
    const int n = Sequences::get_seq_num();
    if ((int)rows.size() != n) return std::to_string(rows.size()) + " records for " + std::to_string(n) + " input sequences";
    for (int i = 0; i < n; i++) {
        if (rows[i].size() != rows[0].size()) return "record " + std::to_string(i + 1) + " differs in length from record 1";
        std::string r = rows[i];
        r.erase(std::remove(r.begin(), r.end(), '-'), r.end());
        if (r != Sequences::getInstance()->get_seq(i)) return "record " + std::to_string(i + 1) + " does not spell input sequence " + std::to_string(i + 1);
    }
    for (size_t c = 0; c < rows[0].size(); c++) {
        bool gaps = true;
        for (int i = 0; i < n && gaps; i++) gaps = rows[i][c] == '-';
        if (gaps) return "column " + std::to_string(c + 1) + " holds gaps only";
    }
    return "";
}

static int pa_star_run_core(const PAStarOpt &opt) // msa_pastar_main.cpp:20-37
{
    HeuristicHPair::getInstance()->init();
    std::cout << "Performing search with Parallel A-Star.\n";
#define RUN_PASTAR(X) \
    case X:           \
        return PAStar<X>::pa_star(Sequences::get_initial_node<X>(), Sequences::get_final_coord<X>(), opt);
    switch (Sequences::get_seq_num()) {
        RUN_PASTAR(3) RUN_PASTAR(4) RUN_PASTAR(5) RUN_PASTAR(6) RUN_PASTAR(7) RUN_PASTAR(8) RUN_PASTAR(9) RUN_PASTAR(10) RUN_PASTAR(14)
            RUN_PASTAR(16) // max_seq_helper.h:9-19
    default:
        std::cerr << "Fatal error: Invalid number of sequences: " << Sequences::get_seq_num() << std::endl;
    }
    return -1;
}

static int pa_star_run(const PAStarOpt &opt) // msa_pastar_main.cpp:39-54
{
    try {
        return pa_star_run_core(opt);
    } catch (std::exception &e) {
        std::cerr << "Running fatal error: " << e.what() << std::endl;
    } catch (...) {
        std::cerr << "Unknown fatal error while running!\n";
    }
    return -1;
}

} // namespace pastar

int main(int argc, char *argv[])
{
    using namespace pastar;
    PAStarOpt opt;
    std::string filename;
    if (msa_pastar_options(argc, argv, filename, opt) != 0) return 1; // the reference MPI_Aborts with 1 here
    if (opt.gpus < 1 || opt.gpus > 16) {
        std::cerr << "Fatal error: --gpus must be between 1 and 16\n";
        return 1;
    }
    opt.mpiRank = 0;
    opt.mpiCommSize = 1;
    opt.mpiMin = 0;
    opt.mpiMax = opt.threads_num;
    opt.totalThreads = opt.mpiCommSize * opt.threads_num;
    if (read_fasta_file(filename) != 0) return 1;
    if (!opt.incumbent.empty()) {
        const std::string why = read_incumbent(opt.incumbent, opt.incumbent_rows);
        if (!why.empty()) {
            std::cerr << "Fatal error: --incumbent " << opt.incumbent << ": " << why << std::endl;
            return 1;
        }
    }
    const int ret = pa_star_run(opt);
    HeuristicHPair::getInstance()->destroyInstance();
    return ret;
}
