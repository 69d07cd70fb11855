// Host drivers of the search (no kernels): whole searches built on the step-wise machinery of pg_search.cu.
//   pg_search          one partition on one GPU, rounds in groups replayed as CUDA graphs
//   pg_search_anytime  weighted searches with falling weights, each bounded by the best alignment so far
//   pg_search_layered  breadth-first heuristic search level by level (the level passes are in pg_layered.cu)
//   pg_search_beam     breadth-first beam search over the same level passes, one phase per width
//   pg_multi_search    the hash-partitioned search over the GPUs of one box, one host thread per GPU
// plus what they share: alignment scoring and the incumbent, the search weight, the lower bound and the result.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstring>
#include <thread>
#include <vector>

#include "pg_internal.cuh"

namespace {

pg_search_config config_or_zero(const pg_search_config *cfg_in)
{
    pg_search_config cfg;
    if (cfg_in)
        cfg = *cfg_in;
    else
        memset(&cfg, 0, sizeof(cfg));
    return cfg;
}

// a search weight num / den that pg_search_set_weight accepts
bool weight_ok(int32_t num, int32_t den)
{
    return den >= 1 && den <= 1024 && (den & (den - 1)) == 0 && num >= den && num <= 16 * den;
}

// the settings of a step-wise search (pg_search_begin) stay as they were while it is active
int refuse_while_stepwise(pg_ctx *ctx, const char *fn)
{
    if (ctx->search && ctx->search->active && ctx->search->stepwise)
        return pg_fail(ctx, PG_ERR_STATE, std::string(fn) + ": a step-wise search is active (pg_search_end first)");
    return PG_OK;
}

// the counts of `part` added to `total` (not the rounds, not the timings)
void add_counts(pg_result *total, const pg_result *part)
{
    total->pops += part->pops;
    total->expansions += part->expansions;
    total->generated += part->generated;
    total->reopen += part->reopen;
    total->open_size += part->open_size;
    total->closed_size += part->closed_size;
    total->probed += part->probed;
    total->pushed += part->pushed;
    total->inserted += part->inserted;
    total->survivors += part->survivors;
}

// Lower bound on the optimal cost from this partition's state (the control block read at the last sync, no records in
// flight): min of (a) g + h over the open entries, (b) the dropped successors' bound (weighted search only), (c) the best
// goal, (d) the all-advance cost and (e) the incumbent's cost U.  The first node of an optimal path that is not closed
// with its optimal g is open with that g or was dropped, so the minimum is at most the optimum.  Successors dropped for
// the incumbent have g + h >= U, and U >= the optimum since U is the cost of an alignment.
long long partition_lb(const SearchState *s, long long open_lb)
{
    const SearchCtrl *c = s->h_ctrl;
    return std::min(std::min(std::min(open_lb, (long long)s->ub), std::min((long long)c->drop_lb, (long long)c->best_goal)), s->inc);
}

// Move masks (origin first) of the alignment `rows`: N NUL-terminated rows of `cols` characters each, every row with its
// '-' removed spelling the context's sequence, no column of gaps only.  PG_ERR_ARG with a message otherwise.
int alignment_masks(pg_ctx *ctx, const char *const *rows, int32_t cols, std::vector<uint32_t> &masks)
{
    if (cols < 1) return pg_fail(ctx, PG_ERR_ARG, "alignment: cols must be positive");
    masks.assign((size_t)cols, 0u);
    for (int i = 0; i < ctx->n; i++) {
        const char *r = rows[i];
        if (!r) return pg_fail(ctx, PG_ERR_ARG, "alignment: row " + std::to_string(i) + " is NULL");
        int at = 0;
        for (int c = 0; c < cols; c++) {
            if (r[c] == 0) return pg_fail(ctx, PG_ERR_ARG, "alignment: row " + std::to_string(i) + " is shorter than cols");
            if (r[c] == '-') continue;
            if (at >= ctx->len[i] || r[c] != ctx->seqs[i][at])
                return pg_fail(ctx, PG_ERR_ARG, "alignment: row " + std::to_string(i) + " does not spell sequence " + std::to_string(i));
            at++;
            masks[c] |= 1u << i;
        }
        if (r[cols] != 0) return pg_fail(ctx, PG_ERR_ARG, "alignment: row " + std::to_string(i) + " is longer than cols");
        if (at != ctx->len[i])
            return pg_fail(ctx, PG_ERR_ARG, "alignment: row " + std::to_string(i) + " does not spell sequence " + std::to_string(i));
    }
    for (int c = 0; c < cols; c++)
        if (masks[c] == 0) return pg_fail(ctx, PG_ERR_ARG, "alignment: column " + std::to_string(c) + " holds gaps only");
    return PG_OK;
}

// The incumbent as a search result: g = f = U, its rows when the caller wants them.
void emit_incumbent(const pg_ctx *ctx, pg_result *res, char *const *rows)
{
    res->g = res->f = (int32_t)ctx->inc_cost;
    res->align_len = (int32_t)ctx->inc_rows[0].size();
    if (rows)
        for (int i = 0; i < ctx->n; i++) memcpy(rows[i], ctx->inc_rows[i].c_str(), ctx->inc_rows[i].size() + 1);
}

// The alignment spelled by `masks` (origin first) as a search result: its length, its rows when the caller wants them
// (backtrace.cpp:54-66) and, for a weighted search, its cost: an ancestor of the goal improved after the goal was found
// (h_w is not consistent) makes the parent chain cheaper than the best goal.
void emit_alignment(const pg_ctx *ctx, const std::vector<uint32_t> &masks, pg_result *res, char *const *rows)
{
    const int cols = (int)masks.size();
    res->align_len = cols;
    if (ctx->wnum > 1) res->g = res->f = (int32_t)pg_path_cost(ctx, masks);
    if (!rows) return;
    std::vector<int> at(ctx->n, 0);
    for (int i = 0; i < ctx->n; i++) rows[i][cols] = 0;
    for (int c = 0; c < cols; c++)
        for (int i = 0; i < ctx->n; i++) rows[i][c] = ((masks[c] >> i) & 1) ? ctx->seqs[i][at[i]++] : '-';
}
} // namespace

long long pg_path_cost(const pg_ctx *ctx, const std::vector<uint32_t> &masks)
{
    const DevProblem &p = ctx->dp;
    std::vector<int> at(ctx->n, 0);
    unsigned prev = (1u << ctx->n) - 1u; // initial parenti: all ones (Sequences.cpp:75)
    long long sum = 0;
    for (uint32_t m : masks) {
        for (int pr = 0; pr < p.npairs; pr++) {
            const int x = p.pa[pr], y = p.pb[pr];
            const int mx = (m >> x) & 1, my = (m >> y) & 1;
            int c;
            if (mx && my)
                c = ctx->cost[(unsigned char)ctx->seqs[x][at[x]] * 90 + (unsigned char)ctx->seqs[y][at[y]]];
            else if (mx)
                c = ((prev >> y) & 1) ? p.gap_open : p.gap_ext;
            else if (my)
                c = ((prev >> x) & 1) ? p.gap_open : p.gap_ext;
            else
                c = p.gap_gap;
            sum += (long long)c * p.w[pr];
        }
        for (int i = 0; i < ctx->n; i++) at[i] += (m >> i) & 1;
        prev = m;
    }
    return sum;
}

extern "C" int pg_score_alignment(pg_ctx *ctx, const char *const *rows, int32_t cols, int64_t *cost)
{
    if (!ctx || !rows || !cost) return PG_ERR_ARG;
    std::vector<uint32_t> masks;
    const int rc = alignment_masks(ctx, rows, cols, masks);
    if (rc != PG_OK) return rc;
    *cost = (int64_t)pg_path_cost(ctx, masks);
    return PG_OK;
}

extern "C" int pg_search_set_incumbent(pg_ctx *ctx, const char *const *rows, int32_t cols)
{
    if (!ctx) return PG_ERR_ARG;
    int rc = refuse_while_stepwise(ctx, "pg_search_set_incumbent");
    if (rc != PG_OK) return rc;
    if (!rows) {
        ctx->inc_rows.clear();
        ctx->inc_cost = -1;
        return PG_OK;
    }
    int64_t cost = 0;
    if ((rc = pg_score_alignment(ctx, rows, cols, &cost)) != PG_OK) return rc;
    if (cost < 0 || cost >= INT_MAX) return pg_fail(ctx, PG_ERR_ARG, "pg_search_set_incumbent: the alignment's cost is outside 0..2^31-2");
    ctx->inc_rows.assign(rows, rows + ctx->n);
    ctx->inc_cost = cost;
    return PG_OK;
}

extern "C" int pg_search(pg_ctx *ctx, const pg_search_config *cfg_in, pg_result *res, char *const *rows)
{
    if (!ctx || !res) return PG_ERR_ARG;
    pg_search_config cfg = config_or_zero(cfg_in);
    if (cfg.n_parts == 0) cfg.n_parts = 1;
    if (cfg.n_parts != 1) return pg_fail(ctx, PG_ERR_ARG, "pg_search runs one partition; use the step-wise calls for n_parts > 1");
    memset(res, 0, sizeof(*res));
    res->g = res->f = -1;
    auto t0 = std::chrono::steady_clock::now();
    int rc = pg_search_begin(ctx, &cfg);
    if (rc != PG_OK) return rc;
    SearchState *s = ctx->search;
    s->stepwise = false;
    const int per_sync = cfg.rounds_per_sync > 0 ? cfg.rounds_per_sync : 8;
    PG_CUDA(ctx, cudaEventRecord(s->ev0, ctx->stream));
    // Every round is the same four launches with the same arguments (all per-round state lives in the device control
    // block), so after a first, ordinary group of rounds the group is captured once into a CUDA graph and replayed: small
    // inputs (kinase.fasta: ~10 us of kernel time per round) are bound by launch overhead, not by the kernels.
    const bool try_graph = !s->profile && !getenv("PG_NO_GRAPH");
    // h(start) >= U: no alignment is cheaper than the incumbent, and no round needs to run to know it
    const bool at_once = s->f0 >= s->inc;
    if (at_once) rc = sync_ctrl(ctx);
    for (long group = 0; !at_once; group++) {
        if ((rc = pg_run_rounds(ctx, per_sync, INT_MAX, per_sync, group > 0 && try_graph)) != PG_OK) return rc;
        if ((rc = sync_ctrl(ctx)) != PG_OK) break;
        if (s->h_ctrl->done) break;
        if (cfg.max_expansions > 0 && (int64_t)s->h_ctrl->expansions >= cfg.max_expansions) break;
    }
    if (rc != PG_OK) return rc;
    PG_CUDA(ctx, cudaEventRecord(s->ev1, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    PG_CUDA(ctx, cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    s->kernel_ms = ms;
    fill_counters(s, res);
    res->finished = s->h_ctrl->done == 1 ? 1 : 0;
    if (s->inc != LLONG_MAX && (at_once || s->h_ctrl->done == 2)) // exhausted below U: the incumbent stands
        res->finished = 2;

    // ---- open / closed census (the reference's final report, PAStar.cpp:591-619) and the search's lower bound
    long long open_lb = 0;
    if ((rc = pg_census(ctx, &res->open_size, &res->closed_size, &open_lb)) != PG_OK) return rc;
    const long long lb = partition_lb(s, open_lb);

    if (res->finished == 2) {
        emit_incumbent(ctx, res, rows);
    } else if (res->finished) {
        res->g = res->f = s->h_ctrl->best_goal; // h(goal) = 0
        std::vector<uint32_t> masks;
        int goal_g = 0;
        if ((rc = pg_backtrace(ctx, masks, &goal_g)) != PG_OK) return rc;
        if (ctx->wnum <= 1 && goal_g != res->g) return pg_fail(ctx, PG_ERR_STATE, "goal entry does not hold the best goal cost");
        emit_alignment(ctx, masks, res, rows);
    }
    ctx->lower_bound = (int32_t)lb;
    ctx->lb_valid = true;
    res->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return PG_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// pg_search_layered: breadth-first heuristic search (Zhou & Hansen, AIJ 2006) with an iteratively raised bound (BFIDA*)
// and divide-and-conquer reconstruction over relay nodes.  The level passes are in pg_layered.cu; DESIGN.md §4.4c.
// ---------------------------------------------------------------------------------------------------------------------
namespace {

// c(pos, mask) under the context's cost model with gap_open == gap_ext (the incoming move does not matter)
long long move_cost(const pg_ctx *ctx, const int *pos, uint32_t m)
{
    const DevProblem &p = ctx->dp;
    long long sum = 0;
    for (int pr = 0; pr < p.npairs; pr++) {
        const int x = p.pa[pr], y = p.pb[pr];
        const int mx = (m >> x) & 1, my = (m >> y) & 1;
        const int c = mx && my ? ctx->cost[(unsigned char)ctx->seqs[x][pos[x]] * 90 + (unsigned char)ctx->seqs[y][pos[y]]]
                               : (mx || my ? p.gap_ext : p.gap_gap);
        sum += (long long)c * p.w[pr];
    }
    return sum;
}

// The refusals shared by the level-pass searches (pg_search_layered, pg_search_beam)
int level_search_refusals(pg_ctx *ctx, const char *fn)
{
    int rc = refuse_while_stepwise(ctx, fn);
    if (rc != PG_OK) return rc;
    if (!ctx->tables_built) return pg_fail(ctx, PG_ERR_STATE, std::string(fn) + ": pg_build_pair_tables has not run");
    if (ctx->dp.gap_open != ctx->dp.gap_ext)
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, std::string(fn) + ": gap_open != gap_ext (a coordinate is then not a state)");
    if (ctx->wnum != 1 || ctx->wsh != 0) return pg_fail(ctx, PG_ERR_ARG, std::string(fn) + ": exact search only (search weight 1)");
    if (ctx->n * ctx->dp.key_bits > 127) return pg_fail(ctx, PG_ERR_UNSUPPORTED, "packed coordinate key exceeds 127 bits");
    return PG_OK;
}

// cost of the alignment whose column c advances every sequence longer than c: the search's UB, as pg_search_begin
long long all_advance_cost(const pg_ctx *ctx)
{
    std::vector<uint32_t> all_advance;
    for (int c = 0, mx = *std::max_element(ctx->len, ctx->len + ctx->n); c < mx; c++) {
        uint32_t m = 0;
        for (int i = 0; i < ctx->n; i++) m |= (uint32_t)(c < ctx->len[i]) << i;
        all_advance.push_back(m);
    }
    return pg_path_cost(ctx, all_advance);
}

// Bin width of a top-level pass at bound U: the bins below the last one span 2 (U - h(start)), so the bound can at most
// triple its distance from h(start) in one step.
int bin_width(long long U, long long h0)
{
    return (int)std::max(1LL, (2 * std::max(1LL, U - h0) + PG_LAYERED_BINS - 2) / (PG_LAYERED_BINS - 1));
}

// The next bound of the top-level passes: the least bin edge U + (b + 1) w below which the failed pass pruned at least
// sqrt(expansions x generated) records, else the top of the bins, or f_min + 1 when every pruned record lies above them;
// at most `cap`.  Always above the pass's f_min.  (On kinase a target of `expansions` records grew the passes by about
// 10 % each, 89 passes; a target of `generated` overshot C* by 2.4 % and expanded ten times the nodes below it.)
long long next_bound(const LayPassOut &o, int U, int w, long long cap)
{
    unsigned long long cum = 0;
    const int nb = (int)o.hist.size();
    const unsigned long long target = std::max<unsigned long long>(1, (unsigned long long)std::sqrt((double)o.expansions * (double)o.generated));
    for (int b = 0; b + 1 < nb; b++) {
        cum += o.hist[b];
        if (cum >= target) return std::min(cap, (long long)U + (long long)(b + 1) * w);
    }
    return std::min(cap, std::max((long long)U + (long long)(nb - 1) * w, (long long)o.fmin + 1));
}

struct Layered {
    pg_ctx *ctx;
    LayeredState *L = nullptr;
    int retain_levels = 0;
    int C = 0;                 // the optimum, bound of every reconstruction pass
    int64_t budget = 0, used = 0;
    bool out_of_budget = false;
    pg_result *res;
    pg_layered_stats st;

    int pass(const LayPassIn &in, LayPassOut &o)
    {
        if (budget > 0 && used >= budget) {
            o = LayPassOut();
            out_of_budget = true;
            return PG_OK;
        }
        const int rc = pg_layered_pass(ctx, L, in, budget > 0 ? budget - used : 0, o);
        if (rc != PG_OK) return rc;
        used += o.expansions;
        res->expansions += o.expansions;
        res->generated += o.generated;
        res->inserted += o.inserted;
        st.passes++;
        st.levels += o.levels;
        st.max_level_nodes = std::max(st.max_level_nodes, o.max_level_nodes);
        st.max_held = std::max(st.max_held, o.max_held);
        if (o.aborted || (budget > 0 && used >= budget && !o.reached)) out_of_budget = true;
        return PG_OK;
    }

    // append the moves of an optimal path from s (g*(s) = gs) to t (g*(t) = gt), both on an optimal alignment
    int solve(const int *s, const int *t, int gs, int gt, int depth, std::vector<uint32_t> &masks)
    {
        int ls = 0, lt = 0;
        for (int i = 0; i < ctx->n; i++) {
            ls += s[i];
            lt += t[i];
        }
        if (ls == lt) return PG_OK;
        st.depth = std::max(st.depth, depth);
        LayPassIn in;
        memcpy(in.s, s, sizeof(in.s));
        memcpy(in.t, t, sizeof(in.t));
        in.g0 = gs;
        in.U = C;
        in.hist_w = 1;
        in.strict = false;
        in.retain = lt - ls + 1 <= retain_levels;
        in.mid = (ls + lt) / 2;
        LayPassOut o;
        int rc = pass(in, o);
        if (rc != PG_OK || out_of_budget) return rc;
        if (!o.reached || o.goal_g != gt)
            return pg_fail(ctx, PG_ERR_STATE, "pg_search_layered: a reconstruction pass missed the optimal g of its corner");
        if (in.retain) {
            std::vector<uint32_t> m;
            if ((rc = pg_layered_trace(ctx, L, in, m)) != PG_OK) return rc;
            masks.insert(masks.end(), m.begin(), m.end());
            return PG_OK;
        }
        return split(s, t, gs, gt, o, depth, masks);
    }

    // s .. p, the crossing move p -> x, x .. t, with x = o's relay
    int split(const int *s, const int *t, int gs, int gt, const LayPassOut &o, int depth, std::vector<uint32_t> &masks)
    {
        int p[PG_MAX_SEQ] = {0};
        for (int i = 0; i < ctx->n; i++) p[i] = o.relay[i] - ((o.relay_mask >> i) & 1);
        const int gp = (int)(o.relay_g - move_cost(ctx, p, o.relay_mask));
        int rc = solve(s, p, gs, gp, depth + 1, masks);
        if (rc != PG_OK || out_of_budget) return rc;
        masks.push_back(o.relay_mask);
        return solve(o.relay, t, o.relay_g, gt, depth + 1, masks);
    }
};

} // namespace

extern "C" int pg_search_layered(pg_ctx *ctx, const pg_search_config *cfg_in, pg_result *res, pg_layered_stats *stats, char *const *rows)
{
    if (!ctx || !res) return PG_ERR_ARG;
    int rc = level_search_refusals(ctx, "pg_search_layered");
    if (rc != PG_OK) return rc;
    const pg_search_config cfg = config_or_zero(cfg_in);
    if (cfg.table_capacity < 0 || cfg.max_expansions < 0) return pg_fail(ctx, PG_ERR_ARG, "pg_search_layered: negative capacity or budget");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    memset(res, 0, sizeof(*res));
    res->g = res->f = -1;
    ctx->lb_valid = false;
    const auto t0 = std::chrono::steady_clock::now();
    const int n = ctx->n;
    int origin[PG_MAX_SEQ] = {0}, goal[PG_MAX_SEQ] = {0}, D = 0;
    for (int i = 0; i < n; i++) {
        goal[i] = ctx->len[i];
        D += ctx->len[i];
    }
    std::vector<uint16_t> zero(n, 0);
    int32_t h0 = 0;
    if ((rc = pg_calculate_h(ctx, zero.data(), 1, &h0)) != PG_OK) return rc;
    const long long ub = all_advance_cost(ctx);
    const bool has_inc = ctx->inc_cost >= 0;
    const long long cap = has_inc ? ctx->inc_cost : ub + 1; // strict bounds: the last pass keeps g + h < cap
    if (cap > INT_MAX - 1) return pg_fail(ctx, PG_ERR_UNSUPPORTED, "pg_search_layered: the upper bound does not fit 31 bits");

    // PG_LAYERED_DEEP: recurse down to single moves; PG_LAYERED_RETAIN: reconstruct in one retain pass over the lattice
    const bool deep = getenv("PG_LAYERED_DEEP") != nullptr, retain_all = getenv("PG_LAYERED_RETAIN") != nullptr;
    Layered S;
    S.ctx = ctx;
    S.res = res;
    memset(&S.st, 0, sizeof(S.st));
    S.retain_levels = retain_all ? D + 1 : (deep ? 1 : 4 * (n + 1));
    S.budget = cfg.max_expansions;
    const int64_t capacity = cfg.table_capacity > 0 ? cfg.table_capacity : (1LL << 22);
    if ((rc = pg_layered_open(ctx, std::max<int64_t>(1, capacity / (n + 1)), S.retain_levels, 0, &S.L)) != PG_OK) {
        pg_layered_close(ctx, S.L);
        return rc;
    }
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    auto finish = [&](int code) {
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        pg_layered_close(ctx, S.L);
        return code;
    };
#define LAY_CHECK(expr)                 \
    do {                                \
        if ((rc = (expr)) != PG_OK)     \
            return finish(rc);          \
    } while (0)
    if (cudaEventCreate(&ev0) != cudaSuccess || cudaEventCreate(&ev1) != cudaSuccess || cudaEventRecord(ev0, ctx->stream) != cudaSuccess)
        return finish(pg_fail(ctx, PG_ERR_CUDA, "pg_search_layered: event set-up failed"));

    // ---- top level: strict bounds U_0 < U_1 < ... up to cap
    long long lb = h0;  // C* >= f_min of every failed pass
    int finished = 0, cstar = -1;
    LayPassOut top;
    if (h0 >= cap) { // h(start) >= U: nothing is cheaper than the incumbent
        finished = 2;
        lb = cap;
    }
    for (long long U = std::min<long long>((long long)h0 + 1, cap); !finished;) {
        LayPassIn in;
        memcpy(in.s, origin, sizeof(in.s));
        memcpy(in.t, goal, sizeof(in.t));
        in.g0 = 0;
        in.U = (int)U;
        in.hist_w = bin_width(U, h0);
        in.strict = true;
        in.retain = false;
        in.mid = D / 2;
        LAY_CHECK(S.pass(in, top));
        if (S.st.iterations == 0) S.st.first_bound = (int32_t)U;
        S.st.iterations++;
        S.st.last_bound = (int32_t)U;
        S.st.top_expansions = top.expansions;
        if (top.reached) {
            cstar = top.goal_g;
            finished = 1;
            lb = cstar;
            break;
        }
        if (top.aborted || (S.out_of_budget && top.levels == 0)) break; // the budget ran out inside (or before) the pass
        const long long fmin = top.fmin == INT_MAX ? cap : top.fmin;
        lb = std::max(lb, std::min(fmin, cap));
        if (fmin >= cap) {
            if (!has_inc) return finish(pg_fail(ctx, PG_ERR_STATE, "pg_search_layered: no path below the all-advance cost"));
            finished = 2; // nothing below U = the incumbent's cost: it is optimal
            lb = cap;
            break;
        }
        if (S.out_of_budget) break;
        U = next_bound(top, (int)U, in.hist_w, cap);
    }

    // ---- reconstruction: the top pass's relay splits the alignment, each half solved by narrower passes
    std::vector<uint32_t> masks;
    if (finished == 1 && rows) {
        S.C = cstar;
        if (retain_all)
            LAY_CHECK(S.solve(origin, goal, 0, cstar, 1, masks));
        else
            LAY_CHECK(S.split(origin, goal, 0, cstar, top, 0, masks));
        if (S.out_of_budget) {
            finished = 0; // C* is proved (lower bound == C*), but the alignment is not complete: no rows
            masks.clear();
        } else if (pg_path_cost(ctx, masks) != cstar) {
            return finish(pg_fail(ctx, PG_ERR_STATE, "pg_search_layered: the reconstructed alignment does not cost C*"));
        }
    }
    if (cudaEventRecord(ev1, ctx->stream) != cudaSuccess || cudaEventSynchronize(ev1) != cudaSuccess)
        return finish(pg_fail(ctx, PG_ERR_CUDA, "pg_search_layered: event failed"));
    float ms = 0;
    cudaEventElapsedTime(&ms, ev0, ev1);
    res->kernel_ms = ms;
    res->rounds = S.st.levels;
    res->finished = finished;
    if (finished == 2) {
        emit_incumbent(ctx, res, rows);
    } else if (finished == 1) {
        res->g = res->f = cstar;
        if (rows) emit_alignment(ctx, masks, res, rows);
    }
    if (finished == 0 && cstar >= 0) lb = cstar;
    if (has_inc) lb = std::min(lb, (long long)ctx->inc_cost);
    ctx->lower_bound = (int32_t)lb;
    ctx->lb_valid = true;
    S.st.peak_bytes = pg_layered_bytes(S.L);
    if (stats) *stats = S.st;
    res->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return finish(PG_OK);
#undef LAY_CHECK
}

// ---------------------------------------------------------------------------------------------------------------------
// pg_search_beam: breadth-first beam search over the lattice levels: strict level passes under the best alignment so far
// that keep the W least (f, packed key) of every level, one phase per width.  The cut is in pg_layered.cu; DESIGN.md §4.4d.
// ---------------------------------------------------------------------------------------------------------------------
namespace {

// Coordinates of the lattice on each level 0 .. D: the coefficients of prod_i (1 + x + ... + x^len_i), saturated at 2^62.
// Every coefficient is capped at 2^100 before the window sums, so a window that holds a capped term is itself >= 2^100.
std::vector<int64_t> level_sizes(const pg_ctx *ctx)
{
    typedef unsigned __int128 u128;
    const u128 CAP = (u128)1 << 100;
    std::vector<u128> c(1, 1);
    for (int i = 0; i < ctx->n; i++) {
        const size_t L = (size_t)ctx->len[i];
        std::vector<u128> pre(c.size() + 1, 0), nc(c.size() + L);
        for (size_t d = 0; d < c.size(); d++) pre[d + 1] = pre[d] + c[d];
        for (size_t d = 0; d < nc.size(); d++) {
            const size_t hi = std::min(d + 1, c.size()), lo = d >= L ? d - L : 0;
            nc[d] = std::min(CAP, pre[hi] - pre[lo]);
        }
        c.swap(nc);
    }
    std::vector<int64_t> out(c.size());
    for (size_t d = 0; d < c.size(); d++) out[d] = (int64_t)std::min(c[d], (u128)1 << 62);
    return out;
}

} // namespace

extern "C" int pg_search_beam(pg_ctx *ctx, const pg_search_config *cfg_in, const int64_t *widths, int n_widths, pg_result *res,
                              pg_result *phase_res, int32_t *phase_lb, pg_beam_stats *stats, char *const *rows)
{
    if (!ctx || !res || !widths) return PG_ERR_ARG;
    if (n_widths < 1 || n_widths > 64) return pg_fail(ctx, PG_ERR_ARG, "pg_search_beam: n_widths must be in 1..64");
    for (int k = 0; k < n_widths; k++)
        if (widths[k] <= 0) return pg_fail(ctx, PG_ERR_ARG, "pg_search_beam: width " + std::to_string(k) + " is not positive");
    int rc = level_search_refusals(ctx, "pg_search_beam");
    if (rc != PG_OK) return rc;
    const pg_search_config cfg = config_or_zero(cfg_in);
    if (cfg.table_capacity < 0 || cfg.max_expansions < 0) return pg_fail(ctx, PG_ERR_ARG, "pg_search_beam: negative capacity or budget");
    const int n = ctx->n;
    int origin[PG_MAX_SEQ] = {0}, goal[PG_MAX_SEQ] = {0}, D = 0;
    for (int i = 0; i < n; i++) {
        goal[i] = ctx->len[i];
        D += ctx->len[i];
    }
    const long long ub = all_advance_cost(ctx);
    if (ctx->inc_cost < 0 && ub + 1 > INT_MAX - 1)
        return pg_fail(ctx, PG_ERR_UNSUPPORTED, "pg_search_beam: the upper bound does not fit 31 bits");

    // memory: the retained array holds at most min(W, |level d|) nodes of every level expanded; the N + 1 level tables
    // hold the candidates before the cut, by default 64 W per level (at least 2^16), never more than the widest level
    const std::vector<int64_t> sizes = level_sizes(ctx);
    const int64_t wmax = *std::max_element(widths, widths + n_widths);
    unsigned __int128 retained = 0;
    for (int d = 0; d < D; d++) retained += (unsigned __int128)std::min(wmax, sizes[d]);
    if (retained > 0xffffffffu)
        return pg_fail(ctx, PG_ERR_CAPACITY, "pg_search_beam: the widest beam retains more than 2^32 - 1 nodes");
    const int64_t widest = *std::max_element(sizes.begin(), sizes.end());
    const int64_t level_cap = cfg.table_capacity > 0 ? std::max<int64_t>(1, cfg.table_capacity / (n + 1))
                                                     : std::min(widest, std::max<int64_t>(1LL << 16, 64 * std::min<int64_t>(wmax, 1LL << 40)));

    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    memset(res, 0, sizeof(*res));
    res->g = res->f = -1;
    for (int k = 0; k < n_widths; k++) {
        if (phase_res) {
            memset(&phase_res[k], 0, sizeof(pg_result));
            phase_res[k].g = phase_res[k].f = -1;
        }
        if (phase_lb) phase_lb[k] = -1;
    }
    pg_beam_stats st;
    memset(&st, 0, sizeof(st));
    st.best_phase = -1;
    st.retained = (int64_t)retained;
    ctx->lb_valid = false;
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<uint16_t> zero(n, 0);
    int32_t h0 = 0;
    if ((rc = pg_calculate_h(ctx, zero.data(), 1, &h0)) != PG_OK) return rc;

    LayeredState *L = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    auto finish = [&](int code) {
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        pg_layered_close(ctx, L);
        return code;
    };
    if ((rc = pg_layered_open(ctx, level_cap, 0, (int64_t)retained, &L)) != PG_OK) return finish(rc);
    if (cudaEventCreate(&ev0) != cudaSuccess || cudaEventCreate(&ev1) != cudaSuccess || cudaEventRecord(ev0, ctx->stream) != cudaSuccess)
        return finish(pg_fail(ctx, PG_ERR_CUDA, "pg_search_beam: event set-up failed"));

    size_t total = 1;
    for (int i = 0; i < n; i++) total += (size_t)ctx->len[i];
    std::vector<std::vector<char>> bufs(n, std::vector<char>(total));
    std::vector<char *> rowp(n);
    for (int i = 0; i < n; i++) rowp[i] = bufs[i].data();
    bool improved = false, any = false;
    long long lb = h0; // the maximum over the phases of their certified bounds
    for (int k = 0; k < n_widths; k++) {
        const bool has_best = ctx->inc_cost >= 0;
        if (has_best && lb >= ctx->inc_cost) break; // the best alignment is proved optimal
        if (cfg.max_expansions > 0 && res->expansions >= cfg.max_expansions) break;
        LayPassIn in;
        memcpy(in.s, origin, sizeof(in.s));
        memcpy(in.t, goal, sizeof(in.t));
        in.g0 = 0;
        in.U = (int)(has_best ? ctx->inc_cost : ub + 1);
        in.hist_w = 1;
        in.strict = true;
        in.retain = false;
        in.mid = D; // no crossing level: every successor carries its parent's retained index
        in.width = widths[k];
        LayPassOut o;
        if ((rc = pg_layered_pass(ctx, L, in, cfg.max_expansions > 0 ? cfg.max_expansions - res->expansions : 0, o)) != PG_OK) {
            // as pg_search_anytime: a phase that runs out of table ends the loop, and the best alignment so far stands
            if (rc == PG_ERR_CAPACITY && any) rc = PG_OK;
            break;
        }
        st.phases++;
        st.levels += o.levels;
        st.kept += o.kept;
        st.dropped += o.dropped;
        st.max_candidates = std::max(st.max_candidates, o.max_cand);
        res->expansions += o.expansions;
        res->generated += o.generated;
        res->inserted += o.inserted;
        res->rounds += o.levels;
        res->closed_size += o.kept;
        res->open_size += o.dropped;
        if (phase_res) {
            pg_result &pr = phase_res[k];
            pr.finished = o.reached && !o.aborted;
            pr.g = pr.f = pr.finished ? o.goal_g : -1;
            pr.expansions = o.expansions;
            pr.generated = o.generated;
            pr.inserted = o.inserted;
            pr.rounds = o.levels;
            pr.closed_size = o.kept;
            pr.open_size = o.dropped;
        }
        if (o.aborted) break; // the budget ran out inside the phase: it certifies nothing
        // LB: the first node of an optimal path that was not kept was dropped by the cut (f <= C*) or pruned by the
        // bound (U <= C*); when there is none, the goal was reached with g = C*
        long long plb = std::min<long long>(in.U, o.drop_fmin);
        if (o.reached) plb = std::min<long long>(plb, o.goal_g);
        lb = std::max(lb, plb);
        any = true;
        if (phase_lb) phase_lb[k] = (int32_t)plb;
        if (o.reached) { // g < U: a strict improvement, the next phases' incumbent
            std::vector<uint32_t> masks;
            if ((rc = pg_beam_trace(ctx, L, in, o.goal_parent, masks)) != PG_OK) return finish(rc);
            if (pg_path_cost(ctx, masks) != o.goal_g)
                return finish(pg_fail(ctx, PG_ERR_STATE, "pg_search_beam: the traced alignment does not cost the goal's g"));
            pg_result tmp;
            memset(&tmp, 0, sizeof(tmp));
            emit_alignment(ctx, masks, &tmp, rowp.data());
            if ((rc = pg_search_set_incumbent(ctx, rowp.data(), (int32_t)masks.size())) != PG_OK) return finish(rc);
            improved = true;
            st.best_phase = k;
        }
    }
    if (rc != PG_OK) return finish(rc);
    if (cudaEventRecord(ev1, ctx->stream) != cudaSuccess || cudaEventSynchronize(ev1) != cudaSuccess)
        return finish(pg_fail(ctx, PG_ERR_CUDA, "pg_search_beam: event failed"));
    float ms = 0;
    cudaEventElapsedTime(&ms, ev0, ev1);
    res->kernel_ms = ms;
    if (ctx->inc_cost >= 0) {
        emit_incumbent(ctx, res, rows);
        res->finished = improved && lb >= ctx->inc_cost ? 1 : 2;
    }
    ctx->lower_bound = (int32_t)lb;
    ctx->lb_valid = true;
    st.peak_bytes = pg_layered_bytes(L);
    if (stats) *stats = st;
    res->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return finish(PG_OK);
}

extern "C" int pg_search_set_weight(pg_ctx *ctx, int32_t num, int32_t den)
{
    if (!ctx) return PG_ERR_ARG;
    if (!weight_ok(num, den))
        return pg_fail(ctx, PG_ERR_ARG, "pg_search_set_weight: den must be a power of two in 1..1024 and den <= num <= 16 den");
    const int rc = refuse_while_stepwise(ctx, "pg_search_set_weight");
    if (rc != PG_OK) return rc;
    int sh = 0;
    while ((1 << sh) < den) sh++;
    while (sh > 0 && (num & 1) == 0) { // reduced: weight 1 is (1, 0) whatever num = den was given
        num >>= 1;
        sh--;
    }
    ctx->wnum = num;
    ctx->wsh = sh;
    return PG_OK;
}

extern "C" int pg_search_lower_bound(pg_ctx *ctx, int32_t *lower_bound)
{
    if (!ctx || !lower_bound) return PG_ERR_ARG;
    if (ctx->lb_valid) {
        *lower_bound = ctx->lower_bound;
        return PG_OK;
    }
    if (!ctx->search || !ctx->search->active) return pg_fail(ctx, PG_ERR_STATE, "pg_search_lower_bound: no search has run on this context");
    long long open_lb = 0;
    int rc = pg_census(ctx, nullptr, nullptr, &open_lb);
    if (rc == PG_OK) rc = sync_ctrl(ctx);
    if (rc != PG_OK) return rc;
    *lower_bound = (int32_t)partition_lb(ctx->search, open_lb);
    return PG_OK;
}

extern "C" int pg_search_anytime(pg_ctx *ctx, const pg_search_config *cfg_in, const int32_t *weight_num, const int32_t *weight_den,
                                 int n_phases, pg_result *res, pg_result *phase_res, int32_t *phase_lb, char *const *rows)
{
    if (!ctx || !res || !weight_num || !weight_den) return PG_ERR_ARG;
    if (n_phases < 1 || n_phases > 64) return pg_fail(ctx, PG_ERR_ARG, "pg_search_anytime: n_phases must be in 1..64");
    for (int k = 0; k < n_phases; k++)
        if (!weight_ok(weight_num[k], weight_den[k]))
            return pg_fail(ctx, PG_ERR_ARG, "pg_search_anytime: phase " + std::to_string(k) + ": den must be a power of two in 1..1024 and den <= num <= 16 den");
    int rc = refuse_while_stepwise(ctx, "pg_search_anytime");
    if (rc != PG_OK) return rc;
    const pg_search_config cfg = config_or_zero(cfg_in);
    memset(res, 0, sizeof(*res));
    res->g = res->f = -1;
    for (int k = 0; k < n_phases; k++) {
        if (phase_res) memset(&phase_res[k], 0, sizeof(pg_result));
        if (phase_lb) phase_lb[k] = -1;
    }
    const auto t0 = std::chrono::steady_clock::now();
    const int wnum0 = ctx->wnum, wsh0 = ctx->wsh;
    size_t total = 1;
    for (int i = 0; i < ctx->n; i++) total += (size_t)ctx->len[i];
    std::vector<std::vector<char>> bufs(ctx->n, std::vector<char>(total));
    std::vector<char *> rowp(ctx->n);
    for (int i = 0; i < ctx->n; i++) rowp[i] = bufs[i].data();
    bool any = false;
    long long lb = 0; // the maximum over the phases of their certified bounds
    for (int k = 0; k < n_phases; k++) {
        if (any && ctx->inc_cost >= 0 && lb >= ctx->inc_cost) break; // the incumbent is proved optimal
        pg_search_config pc = cfg;
        if (cfg.max_expansions > 0) {
            if (res->expansions >= cfg.max_expansions) break;
            pc.max_expansions = cfg.max_expansions - res->expansions;
        }
        if ((rc = pg_search_set_weight(ctx, weight_num[k], weight_den[k])) != PG_OK) break;
        pg_result pr;
        if ((rc = pg_search(ctx, &pc, &pr, rowp.data())) != PG_OK) {
            // a phase that runs out of table ends the loop as the budget does: a lower weight keeps more nodes, so the
            // later phases would too.  The best alignment so far stands (pg_last_error says why the loop stopped).
            if (rc == PG_ERR_CAPACITY && any) rc = PG_OK;
            break;
        }
        // a phase that finishes found an alignment cheaper than the incumbent: it is the next phase's incumbent
        if (pr.finished == 1 && (rc = pg_search_set_incumbent(ctx, rowp.data(), pr.align_len)) != PG_OK) break;
        lb = any ? std::max(lb, (long long)ctx->lower_bound) : (long long)ctx->lower_bound;
        any = true;
        if (phase_res) phase_res[k] = pr;
        if (phase_lb) phase_lb[k] = ctx->lower_bound;
        add_counts(res, &pr);
        res->rounds += pr.rounds;
        res->kernel_ms += pr.kernel_ms;
        res->expand_ms += pr.expand_ms;
        res->select_ms += pr.select_ms;
        res->claim_ms += pr.claim_ms;
        res->insert_ms += pr.insert_ms;
        res->inbox_ms += pr.inbox_ms;
        if (pr.finished == 0) break; // the expansion budget is spent
    }
    ctx->wnum = wnum0;
    ctx->wsh = wsh0;
    if (rc != PG_OK) return rc;
    if (ctx->inc_cost >= 0) {
        emit_incumbent(ctx, res, rows);
        res->finished = any && lb >= ctx->inc_cost ? 1 : 2;
    }
    ctx->lower_bound = (int32_t)lb;
    ctx->lb_valid = any;
    res->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return PG_OK;
}

// ---------------------------------------------------------------------------------------------------------------------
// pg_multi_search: the hash-partitioned search over G GPUs of one box, driven by ONE host process (the pastar CLI).
// Replaces PAStar<N>::pa_star with threads x MPI ranks (PAStar.cpp:626-673) plus sender / receiver / decoder threads
// (pastar_functions/*.cpp) and check_stop's allreduces (PAStar.cpp:502-519): one partition per GPU, parent forwarding
// over peer-mapped inboxes (cudaDeviceEnablePeerAccess: NVLink), the per-round cross-GPU barrier is a set of
// cudaStreamWaitEvent edges (no host blocking), the stop test runs every few rounds on the host from the partitions'
// control blocks.  torch / NCCL are not involved.
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int pg_multi_search(pg_ctx *const *ctxs, int n_gpus, const pg_search_config *cfg_in, pg_result *total, pg_result *parts,
                               char *const *rows)
{
    if (!ctxs || n_gpus < 1 || n_gpus > 16 || !total) return PG_ERR_ARG;
    for (int i = 0; i < n_gpus; i++)
        if (!ctxs[i]) return PG_ERR_ARG;
    pg_ctx *c0 = ctxs[0];
    for (int i = 1; i < n_gpus; i++)
        if (ctxs[i]->wnum != c0->wnum || ctxs[i]->wsh != c0->wsh)
            return pg_fail(c0, PG_ERR_ARG, "pg_multi_search: the contexts' search weights differ (pg_search_set_weight)");
    for (int i = 1; i < n_gpus; i++)
        if (ctxs[i]->inc_cost != c0->inc_cost)
            return pg_fail(c0, PG_ERR_ARG, "pg_multi_search: the contexts' incumbent costs differ (pg_search_set_incumbent)");
    if (n_gpus == 1) {
        int rc = pg_search(c0, cfg_in, total, rows);
        if (rc == PG_OK && parts) parts[0] = *total;
        return rc;
    }
    const pg_search_config cfg = config_or_zero(cfg_in);
    memset(total, 0, sizeof(*total));
    total->g = total->f = -1;
    auto t0 = std::chrono::steady_clock::now();
    const int G = n_gpus;
    std::vector<void *> inbox(G, nullptr), counts(G, nullptr);
    // two events per device: rounds alternate, so a peer one round ahead does not re-record the one being waited for
    std::vector<cudaEvent_t> ev(G, nullptr), ev2(G, nullptr);
    int rc = PG_OK;
    auto cleanup = [&]() {
        for (int i = 0; i < G; i++) {
            cudaSetDevice(ctxs[i]->device);
            if (ctxs[i]->search) cudaStreamSynchronize(ctxs[i]->stream);
            cudaFree(inbox[i]);
            cudaFree(counts[i]);
            if (ev[i]) cudaEventDestroy(ev[i]);
            if (ev2[i]) cudaEventDestroy(ev2[i]);
        }
    };
#define MG_CHECK(i, expr)                                  \
    do {                                                   \
        rc = (expr);                                       \
        if (rc != PG_OK) {                                 \
            if (ctxs[i] != c0) c0->err = ctxs[i]->err;     \
            cleanup();                                     \
            return rc;                                     \
        }                                                  \
    } while (0)
#define MG_CUDA(i, expr)                                                                                         \
    do {                                                                                                         \
        cudaError_t e__ = (expr);                                                                                \
        if (e__ != cudaSuccess) {                                                                                \
            rc = pg_fail(c0, PG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));                  \
            cleanup();                                                                                           \
            return rc;                                                                                           \
        }                                                                                                        \
    } while (0)

    // ---- peer access between every pair of devices; one search state, inbox and count array per device
    for (int i = 0; i < G; i++) {
        MG_CUDA(i, cudaSetDevice(ctxs[i]->device));
        for (int j = 0; j < G; j++) {
            if (ctxs[j]->device == ctxs[i]->device) continue;
            int can = 0;
            MG_CUDA(i, cudaDeviceCanAccessPeer(&can, ctxs[i]->device, ctxs[j]->device));
            if (!can) {
                rc = pg_fail(c0, PG_ERR_UNSUPPORTED, "pg_multi_search: the devices cannot access each other's memory");
                cleanup();
                return rc;
            }
            const cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[j]->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) MG_CUDA(i, e);
            cudaGetLastError();
        }
    }
    {   // search state, inbox and count array of every device, set up concurrently (tens of GB to allocate and clear each)
        std::vector<int> brc(G, PG_OK);
        auto begin_one = [&](int i) {
            pg_search_config ci = cfg;
            ci.n_parts = G;
            ci.part = i;
            ci.reserved = 2; // parent forwarding
            if ((brc[i] = pg_search_begin(ctxs[i], &ci)) != PG_OK) return;
            const size_t bytes = 2 * (size_t)G * ctxs[i]->search->region_bytes;
            cudaError_t e = cudaSetDevice(ctxs[i]->device);
            if (e == cudaSuccess) e = cudaMalloc(&inbox[i], bytes);
            if (e == cudaSuccess) e = cudaMalloc(&counts[i], 2 * (size_t)G * 8);
            if (e == cudaSuccess) e = cudaMemset(counts[i], 0, 2 * (size_t)G * 8);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming);
            if (e != cudaSuccess) brc[i] = pg_fail(ctxs[i], PG_ERR_CUDA, std::string("pg_multi_search set-up: ") + cudaGetErrorString(e));
        };
        std::vector<std::thread> th;
        for (int i = 1; i < G; i++) th.emplace_back(begin_one, i);
        begin_one(0);
        for (std::thread &t : th) t.join();
        for (int i = 0; i < G; i++) MG_CHECK(i, brc[i]);
    }
    // Device-side data-flow synchronisation (default): the counts carry the exchange round and the receiver waits for them
    // on the device, so a round needs no host hand-shake and a group of rounds replays as a CUDA graph.  PG_DEVICE_SYNC=0:
    // the event edges below (one cudaStreamWaitEvent per peer and round, recorded / waited for by the host threads).
    const bool stamped = !(getenv("PG_DEVICE_SYNC") && atoi(getenv("PG_DEVICE_SYNC")) == 0);
    for (int i = 0; i < G; i++) {
        MG_CHECK(i, pg_search_set_peers(ctxs[i], inbox.data(), G));
        MG_CHECK(i, pg_search_set_peer_counts(ctxs[i], counts.data(), G, 2));
        if (stamped) MG_CHECK(i, pg_search_set_device_sync(ctxs[i], 1));
    }

    // ---- rounds.  One host thread per device runs that device's whole loop (the reference: one worker thread per
    // partition, PAStar.cpp:650-651).  Inside a round a thread only waits, spinning on a host flag, until its peers have
    // RECORDED this round's "forwarded" event - the wait for the event itself happens on the GPU stream - and the
    // threads meet at a host barrier for the stop test every few rounds.
    const int per_sync = cfg.rounds_per_sync > 0 ? cfg.rounds_per_sync : (stamped ? 8 : 4);
    int best = INT_MAX, min_open = INT_MAX;
    bool finished = false;
    // every partition empty with no goal below the incumbent's cost U (or h(start) >= U, when no round runs): it stands
    const long long inc = c0->search->inc;
    bool exhausted = c0->search->f0 >= inc;
    std::vector<pg_result> pr(G);
    for (int i = 0; i < G; i++) {
        MG_CUDA(i, cudaSetDevice(ctxs[i]->device));
        MG_CUDA(i, cudaEventCreateWithFlags(&ev2[i], cudaEventDisableTiming));
    }
    if (!exhausted) {
        std::atomic<int> fail(-1), arrive(0), gsense(0), stop(0);
        std::vector<std::atomic<long>> recorded(G);
        for (auto &r : recorded) r.store(-1);
        std::vector<int> fail_rc(G, PG_OK);
        std::vector<int32_t> mn_v(G, INT_MAX), bg_v(G, INT_MAX);
        int shared_best = INT_MAX;
        auto failed = [&]() { return fail.load(std::memory_order_acquire) >= 0; };
        auto relax = [](unsigned &n) {
            if (++n & 1023u) return;
            std::this_thread::yield();
        };
        auto barrier = [&](int &sense) -> bool { // sense-reversing; gives up when a peer has failed
            sense ^= 1;
            if (arrive.fetch_add(1, std::memory_order_acq_rel) + 1 == G) {
                arrive.store(0, std::memory_order_relaxed);
                gsense.store(sense, std::memory_order_release);
            } else {
                unsigned n = 0;
                while (gsense.load(std::memory_order_acquire) != sense && !failed()) relax(n);
            }
            return !failed();
        };
        auto worker = [&](int i) {
            auto bail = [&](int e) {
                fail_rc[i] = e;
                int expect = -1;
                fail.compare_exchange_strong(expect, i);
            };
            int sense = 0, my_best = INT_MAX;
            long round = 0;
            // stamped mode: a group of per_sync rounds (even: the double-buffered inboxes repeat with period 2) is captured
            // once per value of the goal bound and replayed; the first group runs as plain launches (per-device kernel
            // attributes are set on first use)
            GraphExec exec;
            int exec_best = 0;
            const bool graph_ok = stamped && (per_sync % 2) == 0 && !getenv("PG_NO_GRAPH");
            for (;;) {
                bool replayed = false;
                if (graph_ok && round >= per_sync) {
                    if (cudaSetDevice(ctxs[i]->device) != cudaSuccess) return bail(pg_fail(ctxs[i], PG_ERR_CUDA, "cudaSetDevice failed"));
                    if (!exec || exec_best != my_best) {
                        const int e = pg_capture(ctxs[i], [&] {
                            int e = PG_OK;
                            for (int r = 0; r < per_sync && e == PG_OK; r++) {
                                e = pg_search_round_async(ctxs[i], my_best);
                                if (e == PG_OK) e = pg_search_insert_inbox_async(ctxs[i]);
                            }
                            return e;
                        }, &exec);
                        if (e != PG_OK) return bail(e);
                        if (!exec) return bail(pg_fail(ctxs[i], PG_ERR_CUDA, "capturing a group of rounds failed"));
                        exec_best = my_best;
                    }
                    if (cudaGraphLaunch(exec.exec, ctxs[i]->stream) != cudaSuccess) return bail(pg_fail(ctxs[i], PG_ERR_CUDA, "cudaGraphLaunch failed"));
                    pg_search_note_rounds(ctxs[i], per_sync);
                    round += per_sync;
                    replayed = true;
                }
                for (int r = 0; r < per_sync && !replayed; r++, round++) {
                    int e = pg_search_round_async(ctxs[i], my_best); // parents and counts are on their way when the event fires
                    if (e != PG_OK) return bail(e);
                    if (stamped) { // the receiver waits for the counts on the device
                        if ((e = pg_search_insert_inbox_async(ctxs[i])) != PG_OK) return bail(e);
                        continue;
                    }
                    cudaEvent_t mine = (round & 1) ? ev2[i] : ev[i];
                    if (cudaEventRecord(mine, ctxs[i]->stream) != cudaSuccess) return bail(pg_fail(ctxs[i], PG_ERR_CUDA, "cudaEventRecord failed"));
                    recorded[i].store(round, std::memory_order_release);
                    for (int q = 0; q < G; q++) { // barrier on the stream: nobody reads its inbox before every partition has forwarded
                        if (q == i) continue;
                        unsigned n = 0;
                        while (recorded[q].load(std::memory_order_acquire) < round && !failed()) relax(n);
                        if (failed()) return;
                        if (cudaStreamWaitEvent(ctxs[i]->stream, (round & 1) ? ev2[q] : ev[q], 0) != cudaSuccess)
                            return bail(pg_fail(ctxs[i], PG_ERR_CUDA, "cudaStreamWaitEvent failed"));
                    }
                    if ((e = pg_search_insert_inbox_async(ctxs[i])) != PG_OK) return bail(e);
                }
                // stop test (PAStar.cpp:410-547): nothing is in flight once every stream has drained
                int e = pg_search_sync(ctxs[i]);
                if (e == PG_OK) e = pg_search_status(ctxs[i], &mn_v[i], &bg_v[i], &pr[i]);
                if (e != PG_OK) return bail(e);
                if (!barrier(sense)) return;
                if (i == 0) {
                    int mo = INT_MAX, bs = shared_best;
                    int64_t expansions = 0;
                    for (int q = 0; q < G; q++) {
                        mo = std::min(mo, (int)mn_v[q]);
                        bs = std::min(bs, (int)bg_v[q]);
                        expansions += pr[q].expansions;
                    }
                    shared_best = bs;
                    min_open = mo;
                    if (mo >= bs || mo == INT_MAX) {
                        finished = bs != INT_MAX;
                        exhausted = !finished && inc != LLONG_MAX;
                        stop.store(1);
                    } else if (cfg.max_expansions > 0 && expansions >= cfg.max_expansions) {
                        stop.store(1);
                    }
                }
                if (!barrier(sense)) return;
                my_best = shared_best;
                if (stop.load()) return;
            }
        };
        const auto tr0 = std::chrono::steady_clock::now();
        std::vector<std::thread> th;
        for (int i = 1; i < G; i++) th.emplace_back(worker, i);
        worker(0);
        for (std::thread &t : th) t.join();
        total->kernel_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tr0).count();
        best = shared_best;
        const int bad = fail.load();
        if (bad >= 0) {
            rc = fail_rc[bad];
            if (ctxs[bad] != c0) c0->err = ctxs[bad]->err;
            cleanup();
            return rc;
        }
    } else {
        for (int i = 0; i < G; i++) MG_CHECK(i, pg_search_status(ctxs[i], nullptr, nullptr, &pr[i]));
    }

    // ---- results: counters per partition and summed; open / closed census (PAStar.cpp:591-619); the lower bound is the
    // minimum over the partitions
    long long lb = LLONG_MAX;
    for (int i = 0; i < G; i++) {
        long long open_lb = 0;
        MG_CHECK(i, pg_census(ctxs[i], &pr[i].open_size, &pr[i].closed_size, &open_lb));
        lb = std::min(lb, partition_lb(ctxs[i]->search, open_lb));
        pr[i].finished = finished ? 1 : 0;
        add_counts(total, &pr[i]);
        total->rounds = pr[i].rounds;
        if (parts) parts[i] = pr[i];
    }
    total->finished = finished ? 1 : (exhausted ? 2 : 0);
    if (exhausted) {
        for (int i = 0; i < G; i++) pr[i].finished = 2;
        emit_incumbent(c0, total, rows);
    } else if (finished) {
        total->g = total->f = best;
        // distributed backtrace (PAStarDistributedBacktrace.cpp:18-214): the owner of each coordinate answers
        const int n = c0->n;
        std::vector<uint16_t> pos(n);
        for (int i = 0; i < n; i++) pos[i] = (uint16_t)c0->len[i];
        std::vector<uint32_t> masks; // goal-first
        for (;;) {
            bool origin = true;
            for (int i = 0; i < n; i++) origin = origin && pos[i] == 0;
            if (origin) break;
            uint32_t own = 0;
            MG_CHECK(0, pg_owner(c0, pos.data(), 1, G, &own));
            int32_t found = 0, g = 0, parenti = 0;
            MG_CHECK((int)own, pg_search_lookup(ctxs[own], pos.data(), &found, &g, &parenti));
            if (!found || parenti == 0) {
                rc = pg_fail(c0, PG_ERR_STATE, "backtrace lost the parent chain");
                cleanup();
                return rc;
            }
            masks.push_back((uint32_t)parenti);
            for (int i = 0; i < n; i++) pos[i] = (uint16_t)(pos[i] - ((parenti >> i) & 1));
        }
        std::reverse(masks.begin(), masks.end());
        emit_alignment(c0, masks, total, rows);
    }
    for (int i = 0; i < G; i++) {
        pr[i].g = total->g;
        pr[i].f = total->f;
        if (parts) parts[i] = pr[i];
    }
    cleanup();
    for (int i = 0; i < G; i++) {
        pg_search_end(ctxs[i]);
        ctxs[i]->lower_bound = (int32_t)lb;
        ctxs[i]->lb_valid = true;
    }
    total->seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return PG_OK;
#undef MG_CHECK
#undef MG_CUDA
}
