// Host-side mirror of the reference's interfaces for the PA-Star hot path, over the C ABI
// (include/pastar_gpu.h).  Same names, argument meaning and error behaviour as the reference so that code
// written against it (and the parity tests) read the same; every compute call goes to the GPU library.
//
//   reference                                                  here
//   Sequences            pastar/include/Sequences.h:16-40      Sequences      (singleton, set_seq/get_seq/...)
//   Cost                 pastar/include/Cost.h:9-50            Cost           (cost(), gap enums)
//   Coord<N>             pastar/include/Coord.h:30-81          Coord<N>       (operator[], neigh, parent, get_id)
//   Node<N>              pastar/include/Node.h:25-66           Node<N>        (ctor computes f, getNeigh, getters)
//   HeuristicHPair       pastar/include/HeuristicHPair.h:14-30 HeuristicHPair (init, calculate_h, weightMatrix)
//   PAStarOpt / PAStar   pastar/include/PAStar.h:87-117        PAStarOpt, PAStar<N>::pa_star
//   read_fasta_file      pastar/read_fasta.cpp:8-56            read_fasta_file
//   msa_pastar_options   pastar/msa_options.cpp:24-159         msa_pastar_options (hand parsed: Boost is not required)
//   TimeCounter          pastar/TimeCounter.cpp:10-27          TimeCounter
//   backtrace printing   pastar/backtrace.cpp:20-35,135-191    print_entire_backtrace
#pragma once
#include <sys/ioctl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iomanip>
#include <iostream>
#include <limits>
#include <stdexcept>
#include <string>
#include <vector>

#include "pastar_gpu.h"

#ifndef HASH_SHIFT
#define HASH_SHIFT 12 // pastar/include/CoordHash.h:11
#endif

namespace pastar {

enum hashType { HashFZorder, HashPZorder, HashFSum, HashPSum, HashLast }; // Coord.h:28

struct GpuError : std::runtime_error {
    int code;
    GpuError(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

// ---------------------------------------------------------------------------------------------------------
class TimeCounter { // RAII phase timer, prints "<msg>mm:ss.mmm s"
  public:
    explicit TimeCounter(const std::string &msg) : m_msg(msg), m_begin(std::chrono::high_resolution_clock::now()) {}
    ~TimeCounter()
    {
        auto dur = std::chrono::high_resolution_clock::now() - m_begin;
        auto ms = std::chrono::duration_cast<std::chrono::milliseconds>(dur).count() % 1000;
        auto s = std::chrono::duration_cast<std::chrono::seconds>(dur).count() % 60;
        auto m = std::chrono::duration_cast<std::chrono::minutes>(dur).count();
        std::cout << m_msg << std::setfill('0') << std::setw(2) << m << ":" << std::setfill('0') << std::setw(2) << s << "."
                  << std::setfill('0') << std::setw(3) << ms << " s" << std::endl;
    }

  private:
    std::string m_msg;
    std::chrono::high_resolution_clock::time_point m_begin;
};

// ---------------------------------------------------------------------------------------------------------
class Cost {
  public:
    enum { GapExtension = 30, GapOpen = 30, GapGap = GapOpen }; // Cost.h:13
    static int cost(const char r, const char l)
    {
        static int32_t table[90 * 90];
        static bool ready = false;
        if (!ready) {
            pg_default_cost_table(table);
            ready = true;
        }
        const unsigned a = (unsigned char)r, b = (unsigned char)l;
        return a < 90 && b < 90 ? table[a * 90 + b] : 0;
    }
};

template <int N>
class Coord;
template <int N>
class Node;

// ---------------------------------------------------------------------------------------------------------
class Sequences {
  public:
    static Sequences *getInstance()
    {
        static Sequences s;
        return &s;
    }
    int set_seq(const std::string &x)
    {
        seqs.push_back(x);
        if ((int)x.length() > max_length()) max_length() = (int)x.length();
        return ++get_seq_num();
    }
    const std::string &get_seq(int x) const { return seqs.at(x); }
    static int &get_seq_num()
    {
        static int n = 0;
        return n;
    }
    static int &max_length()
    {
        static int m = 0;
        return m;
    }
    const std::vector<std::string> &all() const { return seqs; }
    template <int N>
    static Coord<N> get_final_coord();
    template <int N>
    static Coord<N> get_initial_coord();
    template <int N>
    static Node<N> get_initial_node();
    template <int N>
    static bool is_final(const Coord<N> &c);

  private:
    std::vector<std::string> seqs;
};

// ---------------------------------------------------------------------------------------------------------
// The GPU context shared by the shims: the state the reference keeps in its Cost / Sequences /
// HeuristicHPair singletons and the two hash globals (CoordHash.cpp:17-18).
class HeuristicHPair {
  public:
    static HeuristicHPair *getInstance()
    {
        static HeuristicHPair h;
        return &h;
    }
    // HeuristicHPair::init, HeuristicHPair.cpp:47-67: pairwise tables (GPU) then pair weights (host)
    void init(int device = -1)
    {
        TimeCounter tp("Phase 1 - init heuristic: ");
        Sequences *seq = Sequences::getInstance();
        const int n = Sequences::get_seq_num();
        std::vector<const char *> ptr(n);
        std::vector<int> len(n);
        for (int i = 0; i < n; i++) {
            ptr[i] = seq->get_seq(i).data();
            len[i] = (int)seq->get_seq(i).size();
        }
        flat.assign((size_t)n * n, 0.0f);
        // the pair loop of weightAltschulsRationale2 runs on the device; very long sequences take the host routine
        int rc = pg_gpu_weights(n, ptr.data(), len.data(), device, flat.data(), nullptr);
        if (rc == PG_ERR_UNSUPPORTED) rc = pg_host_weights(n, ptr.data(), len.data(), flat.data());
        if (rc != PG_OK)
            throw GpuError(rc, std::string("pair weights (pg_gpu_weights / pg_host_weights) failed: ") +
                                   (rc == PG_ERR_CUDA  ? "CUDA failure or no CUDA device (there is no CPU fallback)"
                                    : rc == PG_ERR_ARG ? "bad input (empty sequence, or a residue outside the 90x90 cost table)"
                                                       : "status " + std::to_string(rc)));
        rows.resize(n);
        for (int i = 0; i < n; i++) rows[i] = flat.data() + (size_t)i * n;
        weightMatrix = rows.data();
        std::vector<int32_t> wint((size_t)n * n);
        for (size_t i = 0; i < wint.size(); i++) wint[i] = (int32_t)flat[i]; // (int) truncation, Node.cpp:226
        std::cout << "Starting pairwise alignments... " << std::flush;
        rc = pg_ctx_create(n, ptr.data(), len.data(), nullptr, Cost::GapOpen, Cost::GapExtension, Cost::GapGap, wint.data(), device, &ctx);
        check(rc, "pg_ctx_create");
        check(pg_build_pair_tables(ctx, &tables_ms), "pg_build_pair_tables");
        std::cout << "done!\n";
        wint_keep = wint;
    }
    // One more context per additional GPU: the reference recomputes the heuristic on every MPI rank
    // (HeuristicHPair.cpp:47-67 runs everywhere); here every device builds its own copy of the pair tables.
    std::vector<pg_ctx *> contexts(int gpus)
    {
        Sequences *seq = Sequences::getInstance();
        const int n = Sequences::get_seq_num();
        std::vector<const char *> ptr(n);
        std::vector<int> len(n);
        for (int i = 0; i < n; i++) {
            ptr[i] = seq->get_seq(i).data();
            len[i] = (int)seq->get_seq(i).size();
        }
        while ((int)more.size() + 1 < gpus) {
            pg_ctx *c = nullptr;
            const int dev = (int)more.size() + 1;
            int rc = pg_ctx_create(n, ptr.data(), len.data(), nullptr, Cost::GapOpen, Cost::GapExtension, Cost::GapGap, wint_keep.data(), dev, &c);
            if (rc != PG_OK) throw GpuError(rc, "pg_ctx_create on device " + std::to_string(dev) + " failed (are there that many GPUs?)");
            more.push_back(c);
            rc = pg_build_pair_tables(c, nullptr);
            if (rc != PG_OK) throw GpuError(rc, std::string("pg_build_pair_tables: ") + pg_last_error(c));
        }
        std::vector<pg_ctx *> all{ctx};
        for (int i = 0; i + 1 < gpus; i++) all.push_back(more[i]);
        return all;
    }
    void destroyInstance()
    {
        for (pg_ctx *c : more) pg_ctx_destroy(c);
        more.clear();
        if (ctx) pg_ctx_destroy(ctx);
        ctx = nullptr;
    }
    template <int N>
    int calculate_h(const Coord<N> &c) const;
    int getScore(int pair, int i, int j) // PairAlign::getScore, PairAlign.cpp:174-177
    {
        if ((int)tables.size() <= pair) tables.resize(pair + 1);
        int r = 0, c = 0;
        check(pg_pair_table_shape(ctx, pair, &r, &c), "pg_pair_table_shape");
        if (tables[pair].empty()) {
            tables[pair].resize((size_t)r * c);
            check(pg_copy_pair_table(ctx, pair, tables[pair].data()), "pg_copy_pair_table");
        }
        return tables[pair][(size_t)i * c + j];
    }
    void check(int rc, const char *what) const
    {
        if (rc == PG_OK) return;
        if (rc == PG_ERR_HASH_SHIFT) throw std::invalid_argument("Invalid Hash Shift"); // CoordHash.cpp:241
        throw GpuError(rc, std::string(what) + ": " + (ctx ? pg_last_error(ctx) : "no context (is a CUDA device present?)"));
    }
    float **weightMatrix = nullptr;
    pg_ctx *ctx = nullptr;
    float tables_ms = 0;
    ~HeuristicHPair() { destroyInstance(); }

  private:
    HeuristicHPair() {}
    std::vector<float> flat;
    std::vector<float *> rows;
    std::vector<std::vector<int32_t>> tables;
    std::vector<int32_t> wint_keep;
    std::vector<pg_ctx *> more; // contexts on devices 1 .. gpus-1
};

// ---------------------------------------------------------------------------------------------------------
extern int hash_shift;     // CoordHash.cpp:17
extern hashType hash_type; // CoordHash.cpp:18

template <int N>
class Coord {
  public:
    Coord(const int init = 0)
    {
        for (int i = 0; i < N; i++) m_coord[i] = (uint16_t)init;
    }
    bool operator!=(const Coord &rhs) const { return memcmp(m_coord, rhs.m_coord, sizeof(m_coord)) != 0; }
    bool operator==(const Coord &rhs) const { return !(*this != rhs); }
    bool operator<(const Coord &rhs) const // lexicographic, Coord.cpp:57-71
    {
        for (int i = 0; i < N; i++) {
            if (m_coord[i] < rhs.m_coord[i]) return true;
            if (m_coord[i] > rhs.m_coord[i]) return false;
        }
        return false;
    }
    const uint16_t &operator[](const uint16_t n) const { return m_coord[n]; }
    uint16_t &operator[](const uint16_t n) { return m_coord[n]; }
    Coord neigh(int n) const // Coord.cpp:92-106
    {
        Coord c(*this);
        for (int i = 0; n; n >>= 1, i++)
            if (n & 1) c[i] += 1;
        return c;
    }
    Coord parent(int n) const // Coord.cpp:112-126
    {
        Coord c(*this);
        for (int i = 0; n; n >>= 1, i++)
            if (n & 1) c[i] -= 1;
        return c;
    }
    static const char *get_hash_name()
    {
        static const char *const names[] = {"Full-Zorder", "Partial-Zorder", "Full-Sum", "Partial-Sum"};
        return names[hash_type];
    }
    static int get_hash_shift() { return hash_shift; }
    static void configure_hash(hashType type, int shift) // CoordHash.cpp:260-265 (globals) + push to the device context
    {
        hash_type = type;
        hash_shift = shift;
        HeuristicHPair *h = HeuristicHPair::getInstance();
        if (h->ctx) h->check(pg_configure_hash(h->ctx, (int)type, shift), "pg_configure_hash");
    }
    unsigned int get_id(const int size) const // CoordHash.cpp:190-245; throws invalid_argument on a bad shift
    {
        if (hash_shift < 0 || hash_shift > 21) throw std::invalid_argument("Invalid Hash Shift");
        HeuristicHPair *h = HeuristicHPair::getInstance();
        uint32_t out = 0;
        h->check(pg_owner(h->ctx, m_coord, 1, size, &out), "pg_owner");
        return out;
    }
    const uint16_t *data() const { return m_coord; }

  private:
    uint16_t m_coord[N];
};

template <int N>
std::ostream &operator<<(std::ostream &lhs, const Coord<N> &rhs) // Coord.cpp:29-40
{
    lhs << "(" << rhs[0];
    for (int i = 1; i < N; i++) lhs << " " << rhs[i];
    lhs << ")";
    return lhs;
}

template <int N>
int HeuristicHPair::calculate_h(const Coord<N> &c) const
{
    int32_t h = 0;
    check(pg_calculate_h(ctx, c.data(), 1, &h), "pg_calculate_h");
    return h;
}

// ---------------------------------------------------------------------------------------------------------
template <int N>
class Node { // memory layout == reference Node<N> == pg_node: pos, m_f, m_g, parenti
  public:
    Coord<N> pos;
    int m_f;
    Node() : m_f(0), m_g(0), parenti(0) {}
    Node(const int g, const Coord<N> &pos, const int &parenti) : pos(pos), m_g(g), parenti(parenti)
    {
        m_f = m_g + HeuristicHPair::getInstance()->calculate_h(pos); // Node.cpp:32-39
    }
    // Node<N>::getNeigh, Node.cpp:205-248: appends to a[owner], never clears, returns 0
    int getNeigh(std::vector<Node> a[], int vec_size = 1)
    {
        static_assert(sizeof(Node) == (size_t)(((2 * N + 3) & ~3) + 12), "Node<N> must match pg_node");
        HeuristicHPair *h = HeuristicHPair::getInstance();
        const int S = (1 << N) - 1, stride = pg_succ_stride(N);
        std::vector<unsigned char> buf((size_t)S * stride);
        int32_t count = 0;
        h->check(pg_expand_batch(h->ctx, this, 1, vec_size, buf.data(), &count), "pg_expand_batch");
        // the reference appends bucket by bucket in ascending mask order; ours are in ascending mask order already
        for (int k = 0; k < count; k++) {
            const unsigned char *r = buf.data() + (size_t)k * stride;
            Node nd;
            memcpy((void *)&nd, r, sizeof(Node));
            uint32_t owner;
            memcpy(&owner, r + sizeof(Node), 4);
            a[owner].push_back(nd);
        }
        return 0;
    }
    int get_g() const { return m_g; }
    int get_f() const { return m_f; }
    int get_h() const { return m_f - m_g; }
    int get_parenti() const { return parenti; }
    Coord<N> get_parent() const { return pos.parent(parenti); }
    void set(int g, int f, int par)
    {
        m_g = g;
        m_f = f;
        parenti = par;
    }

  private:
    int m_g;
    int parenti;
};

template <int N>
std::ostream &operator<<(std::ostream &lhs, const Node<N> &rhs) // Node.cpp:41-47
{
    lhs << rhs.pos << "\tg - " << rhs.get_g() << " (h - " << rhs.get_h() << " f - " << rhs.get_f() << ")";
    return lhs;
}

template <int N>
Coord<N> Sequences::get_final_coord()
{
    Coord<N> c;
    for (int i = 0; i < N; ++i) c[i] = (uint16_t)getInstance()->get_seq(i).length();
    return c;
}
template <int N>
Coord<N> Sequences::get_initial_coord()
{
    return Coord<N>();
}
template <int N>
Node<N> Sequences::get_initial_node() // Sequences.cpp:70-77
{
    return Node<N>(0, Sequences::get_initial_coord<N>(), (1 << N) - 1);
}
template <int N>
bool Sequences::is_final(const Coord<N> &c)
{
    return c == get_final_coord<N>();
}

// ---------------------------------------------------------------------------------------------------------
struct AStarOpt {
    bool force_quit = true;
};
struct PAStarOpt { // PAStar.h:87-112, plus the GPU-side knobs (new, do not change the existing ones)
    AStarOpt common_options;
    hashType hash_type = HashFZorder;
    int hash_shift = HASH_SHIFT;
    int threads_num = 1;
    int mpiRank = 0, mpiCommSize = 1, mpiMin = 0, mpiMax = 1, totalThreads = 1;
    int gpus = 1;
    long long batch = 0, table_capacity = 0, max_expansions = 0;
    std::string metrics_json; // --metrics_json FILE: counters of the run as one JSON object (PAStarSyncData.cpp's gather, machine-readable)
    int weight_num = 0;       // --weight W: bounded-suboptimal search with weight weight_num / 1024 (0 = not given: exact search)
    std::string incumbent;                  // --incumbent FILE: aligned FASTA of a known alignment (upper bound of the search)
    std::vector<std::string> incumbent_rows; // its rows, checked against the input before any device call
    std::vector<int32_t> anytime_num;        // --anytime W1,W2,...: one weighted phase per weight, num / 1024 (empty: not given)
};

int read_fasta_file(const std::string &name);
int msa_pastar_options(int argc, char *argv[], std::string &filename, PAStarOpt &opt);
int get_print_size();
void print_similarity(const std::vector<std::string> &rows);
void print_alignment(const std::vector<std::string> &rows);

template <int N>
class PAStar {
  public:
    // PAStar<N>::pa_star, PAStar.cpp:626-673
    static int pa_star(const Node<N> &node_zero, const Coord<N> &coord_final, const PAStarOpt &options)
    {
        (void)node_zero;
        if (options.threads_num <= 0) throw std::invalid_argument("Invalid number of threads");
        Coord<N>::configure_hash(options.hash_type, options.hash_shift);
        std::cout << "Running PAStar with: " << options.totalThreads << " threads (" << options.mpiCommSize << " machines with "
                  << options.threads_num << " threads each)," << Coord<N>::get_hash_name() << " hash, " << Coord<N>::get_hash_shift()
                  << " shift.\n";
        if (options.gpus > 1) std::cout << "Hash-owned partitions: " << options.gpus << " (one per GPU)\n";
        HeuristicHPair *h = HeuristicHPair::getInstance();
        pg_search_config cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.n_parts = 1;
        cfg.batch_target = options.batch;
        cfg.table_capacity = options.table_capacity;
        cfg.max_expansions = options.max_expansions;
        pg_result res;
        const int gpus = options.gpus > 0 ? options.gpus : 1;
        std::vector<pg_result> parts(gpus);
        size_t total = 1;
        for (int i = 0; i < N; i++) total += coord_final[i];
        std::vector<std::vector<char>> bufs(N, std::vector<char>(total));
        std::vector<char *> rowp(N);
        for (int i = 0; i < N; i++) rowp[i] = bufs[i].data();
        const int wden = 1024;
        int32_t lower_bound = 0;
        const bool bounded = options.weight_num || !options.incumbent_rows.empty() || !options.anytime_num.empty();
        std::vector<const char *> inc(N);
        for (int i = 0; i < (int)options.incumbent_rows.size(); i++) inc[i] = options.incumbent_rows[i].c_str();
        const int inc_cols = options.incumbent_rows.empty() ? 0 : (int)options.incumbent_rows[0].size();
        int64_t inc_cost = 0;
        const int n_phases = (int)options.anytime_num.size();
        std::vector<pg_result> phase_res(n_phases);
        std::vector<int32_t> phase_lb(n_phases, -1);
        if (inc_cols) h->check(pg_score_alignment(h->ctx, inc.data(), inc_cols, &inc_cost), "pg_score_alignment");
        if (gpus == 1) {
            if (options.weight_num) h->check(pg_search_set_weight(h->ctx, options.weight_num, wden), "pg_search_set_weight");
            if (inc_cols) h->check(pg_search_set_incumbent(h->ctx, inc.data(), inc_cols), "pg_search_set_incumbent");
            TimeCounter t("Phase 2: PA-Star running time: ");
            if (n_phases) {
                const std::vector<int32_t> dens(n_phases, wden);
                h->check(pg_search_anytime(h->ctx, &cfg, options.anytime_num.data(), dens.data(), n_phases, &res, phase_res.data(),
                                           phase_lb.data(), rowp.data()),
                         "pg_search_anytime");
            } else {
                h->check(pg_search(h->ctx, &cfg, &res, rowp.data()), "pg_search");
            }
            parts[0] = res;
            if (bounded) h->check(pg_search_lower_bound(h->ctx, &lower_bound), "pg_search_lower_bound");
        } else {
            // one hash-owned partition per GPU (the reference: one per thread x MPI rank, PAStar.cpp:107-117)
            std::vector<pg_ctx *> ctxs = h->contexts(gpus);
            for (pg_ctx *c : ctxs) h->check(pg_configure_hash(c, (int)options.hash_type, options.hash_shift), "pg_configure_hash");
            if (options.weight_num)
                for (pg_ctx *c : ctxs) h->check(pg_search_set_weight(c, options.weight_num, wden), "pg_search_set_weight");
            if (inc_cols)
                for (pg_ctx *c : ctxs) h->check(pg_search_set_incumbent(c, inc.data(), inc_cols), "pg_search_set_incumbent");
            TimeCounter t("Phase 2: PA-Star running time: ");
            h->check(pg_multi_search(ctxs.data(), gpus, &cfg, &res, parts.data(), rowp.data()), "pg_multi_search");
            if (bounded) h->check(pg_search_lower_bound(ctxs[0], &lower_bound), "pg_search_lower_bound");
        }
        // weighted, incumbent-bounded and anytime search: the optimum is at least the lower bound, so g / bound is the
        // certified ratio to it (1: the alignment is proved optimal)
        auto print_bound = [&]() {
            if (!(options.weight_num > wden || inc_cols || n_phases)) return;
            std::cout << "Lower bound: " << lower_bound;
            if (res.finished) std::cout << "\tg / lower bound: " << std::fixed << std::setprecision(4) << (double)res.g / lower_bound;
            std::cout << std::endl;
            for (int k = 0; k < n_phases; k++)
                if (phase_lb[k] >= 0)
                    std::cout << "Anytime phase " << k + 1 << ": weight " << std::defaultfloat << std::setprecision(6) << (double)options.anytime_num[k] / wden
                              << ", score " << phase_res[k].g << ", lower bound " << phase_lb[k] << ", expansions " << phase_res[k].expansions
                              << std::endl;
        };
        if (!res.finished) {
            std::cout << "Search stopped at the expansion budget: " << res.expansions << " expansions, no alignment.\n";
            print_bound();
        } else {
            TimeCounter *t = new TimeCounter("Phase 3 - backtrace: ");
            Node<N> fin;
            fin.pos = coord_final;
            fin.set(res.g, res.f, 0);
            std::cout << "Final Score: " << fin << std::endl; // PAStarDistributedBacktrace.cpp:47
            print_bound();
            std::vector<std::string> rows(N);
            for (int i = 0; i < N; i++) rows[i] = rowp[i];
            delete t;
            print_similarity(rows);
            print_alignment(rows);
        }
        // print_nodes_count, PAStar.cpp:591-619: one "tid" row per partition
        std::cout << "Total nodes count:" << std::endl;
        for (int i = 0; i < gpus; i++)
            std::cout << "tid " << i << "\tOpenList:" << parts[i].open_size << "\tClosedList:" << parts[i].closed_size << "\tReopen:" << parts[i].reopen
                      << "\tTotal: " << parts[i].pops << std::endl;
        std::cout << "Sum\tOpenList:" << res.open_size << "\tClosedList:" << res.closed_size << "\tReopen:" << res.reopen
                  << "\tTotal: " << res.pops << std::endl;
        std::cout << "GPU: " << res.expansions << " expansions, " << res.generated << " successors, " << res.rounds << " rounds, "
                  << std::fixed << std::setprecision(3) << res.kernel_ms << " ms on device ("
                  << (res.kernel_ms > 0 ? res.expansions / res.kernel_ms / 1e3 : 0.0) << " M expansions/s); pairwise tables "
                  << h->tables_ms << " ms" << std::endl;
        if (!options.metrics_json.empty()) {
            std::ofstream js(options.metrics_json);
            auto one = [&](const pg_result &r) {
                js << "{\"pops\": " << r.pops << ", \"expansions\": " << r.expansions << ", \"generated\": " << r.generated
                   << ", \"probed\": " << r.probed << ", \"pushed\": " << r.pushed << ", \"inserted\": " << r.inserted
                   << ", \"reopen\": " << r.reopen << ", \"open_size\": " << r.open_size << ", \"closed_size\": " << r.closed_size << "}";
            };
            js << "{\"finished\": " << res.finished << ", \"g\": " << res.g << ", \"f\": " << res.f << ", \"align_len\": " << res.align_len
               << ", \"rounds\": " << res.rounds << ", \"gpus\": " << gpus << ", \"search_ms\": " << res.kernel_ms
               << ", \"pair_tables_ms\": " << h->tables_ms << ", \"hash_type\": \"" << Coord<N>::get_hash_name() << "\", \"hash_shift\": "
               << Coord<N>::get_hash_shift();
            if (options.weight_num)
                js << ", \"weight\": " << std::setprecision(10) << (double)options.weight_num / wden;
            if (bounded) js << ", \"lower_bound\": " << lower_bound;
            if (inc_cols) js << ", \"incumbent\": " << inc_cost;
            if (n_phases) {
                js << ", \"phases\": [";
                bool first = true;
                for (int k = 0; k < n_phases; k++) {
                    if (phase_lb[k] < 0) continue;
                    js << (first ? "" : ", ") << "{\"weight\": " << std::setprecision(10) << (double)options.anytime_num[k] / wden
                       << ", \"g\": " << phase_res[k].g << ", \"lower_bound\": " << phase_lb[k] << ", \"expansions\": "
                       << phase_res[k].expansions << ", \"finished\": " << phase_res[k].finished << "}";
                    first = false;
                }
                js << "]";
            }
            js << ", \"total\": ";
            one(res);
            js << ", \"partitions\": [";
            for (int i = 0; i < gpus; i++) {
                if (i) js << ", ";
                one(parts[i]);
            }
            js << "]}\n";
        }
        return 0;
    }
};

} // namespace pastar
