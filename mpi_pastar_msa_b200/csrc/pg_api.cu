// C ABI of libpastar_gpu (include/pastar_gpu.h): context management and the
// host-pointer entry points.  No CPU fallback: every compute entry point
// launches a CUDA kernel or fails.
#include <algorithm>
#include <cstring>

#include "pg_internal.cuh"

int pg_fail(pg_ctx *ctx, int code, const std::string &msg)
{
    if (ctx) ctx->err = msg;
    return code;
}

extern "C" int pg_abi_version(void) { return PG_ABI_VERSION; }

// ---- measured ceiling of the closed/open-table probe: random 16-byte loads over `bytes` of HBM, 8 in flight per thread
namespace {
__global__ void gather_probe_kernel(const unsigned long long *tab, unsigned long long mask, int iters, unsigned long long *out)
{
    unsigned long long tid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
    unsigned long long acc = 0, seed = tid * 0x1234567ull + 1;
    for (int it = 0; it < iters; it++) {
        unsigned long long a[8], b[8];
#pragma unroll
        for (int j = 0; j < 8; j++) {
            seed = (seed + j) * 0x9E3779B97F4A7C15ull;
            seed ^= seed >> 32;
            seed *= 0xD6E8FEB86659FD93ull;
            seed ^= seed >> 29;
            asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(a[j]), "=l"(b[j]) : "l"(tab + 2 * (seed & mask)) : "memory");
        }
#pragma unroll
        for (int j = 0; j < 8; j++) acc += a[j] ^ b[j];
    }
    if (acc == 0x1234) out[0] = acc;
}
} // namespace

extern "C" int pg_bench_random_gather(int device, int64_t bytes, double *loads_per_sec)
{
    if (!loads_per_sec || bytes < (1 << 20)) return PG_ERR_ARG;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return PG_ERR_CUDA;
    unsigned long long entries = 1;
    while (entries * 2 * 16 <= (unsigned long long)bytes) entries *= 2;
    unsigned long long *tab = nullptr, *out = nullptr;
    if (cudaMalloc(&tab, entries * 16) != cudaSuccess) return PG_ERR_CUDA;
    if (cudaMalloc(&out, 64) != cudaSuccess) {
        cudaFree(tab);
        return PG_ERR_CUDA;
    }
    cudaMemset(tab, 0, entries * 16);
    cudaDeviceProp prop;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaGetDeviceProperties(&prop, dev);
    const int blocks = prop.multiProcessorCount * 4, threads = 256, iters = 64;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    gather_probe_kernel<<<blocks, threads>>>(tab, entries - 1, iters, out);
    cudaDeviceSynchronize();
    float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        cudaEventRecord(e0);
        gather_probe_kernel<<<blocks, threads>>>(tab, entries - 1, iters, out);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaError_t err = cudaGetLastError();
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(tab);
    cudaFree(out);
    if (err != cudaSuccess) return PG_ERR_CUDA;
    *loads_per_sec = (double)blocks * threads * iters * 8 / (best * 1e-3);
    return PG_OK;
}

// ---- measured integer peak for the pairwise DP's roofline: the DP cell is three adds and one three-input minimum
// (IADD x3 + VIMNMX3); this kernel issues exactly that mix in 8 independent chains per thread, so it measures how
// many DP-cell instruction groups per second the integer pipes sustain when nothing else limits them.
namespace {
__global__ void int_peak_kernel(int iters, int seed, int *out)
{
    int v[8], c = seed + (int)threadIdx.x;
#pragma unroll
    for (int k = 0; k < 8; k++) v[k] = seed * (k + 1) + (int)threadIdx.x;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int k = 0; k < 8; k++) v[k] = __vimin3_s32(v[k] + 30, v[(k + 1) & 7] + 29, v[(k + 3) & 7] + c); // one DP cell
    }
    int acc = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) acc ^= v[k];
    if (acc == 0x7fffffff) out[0] = acc;
}
} // namespace

extern "C" int pg_bench_int_peak(int device, double *cells_per_sec)
{
    if (!cells_per_sec) return PG_ERR_ARG;
    if (device >= 0 && cudaSetDevice(device) != cudaSuccess) return PG_ERR_CUDA;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return PG_ERR_CUDA;
    int *out = nullptr;
    if (cudaMalloc(&out, 64) != cudaSuccess) return PG_ERR_CUDA;
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    int_peak_kernel<<<blocks, threads>>>(iters, 1, out);
    cudaDeviceSynchronize();
    float best = 1e30f;
    for (int r = 0; r < 3; r++) {
        cudaEventRecord(e0);
        int_peak_kernel<<<blocks, threads>>>(iters, r + 2, out);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    const cudaError_t err = cudaGetLastError();
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(out);
    if (err != cudaSuccess) return PG_ERR_CUDA;
    *cells_per_sec = (double)blocks * threads * iters * 8 / (best * 1e-3);
    return PG_OK;
}

extern "C" const char *pg_last_error(const pg_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int pg_stage(pg_ctx *ctx, int which, size_t bytes, void **out)
{
    if (ctx->stage_bytes[which] < bytes) {
        if (ctx->d_stage[which]) cudaFree(ctx->d_stage[which]);
        ctx->d_stage[which] = nullptr;
        ctx->stage_bytes[which] = 0;
        size_t want = std::max(bytes, (size_t)1 << 20);
        PG_CUDA(ctx, cudaMalloc(&ctx->d_stage[which], want));
        ctx->stage_bytes[which] = want;
    }
    *out = ctx->d_stage[which];
    return PG_OK;
}

static bool g_extended_n = false; // explicit opt-in, process-wide: sequence counts the reference cannot run (SURVEY 8f N4)
extern "C" int pg_allow_extended_n(int enable)
{
    g_extended_n = enable != 0;
    return PG_OK;
}
static bool supported_n(int n)
{
    if ((n >= 3 && n <= 10) || n == 14 || n == 16) return true; // max_seq_helper.h:9-19
    return g_extended_n && n >= 11 && n <= 15;                  // 11, 12, 13, 15: one GPU only (no partitioned kernels built)
}

extern "C" int pg_ctx_create(int n_seq, const char *const *seqs, const int *lens, const int32_t *cost90x90, int gap_open,
                             int gap_ext, int gap_gap, const int32_t *w_int, int device, pg_ctx **out)
{
    if (!out) return PG_ERR_ARG;
    *out = nullptr;
    if (!seqs || !lens || !supported_n(n_seq)) return PG_ERR_ARG;
    for (int i = 0; i < n_seq; i++)
        if (lens[i] < 1 || lens[i] > 65534 || !seqs[i]) return PG_ERR_ARG; // Coord is uint16 (Coord.h:68)
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return PG_ERR_CUDA; // no CPU fallback
    pg_ctx *ctx = new pg_ctx();
    if (device >= 0) {
        if (cudaSetDevice(device) != cudaSuccess) {
            delete ctx;
            return PG_ERR_CUDA;
        }
    }
    cudaGetDevice(&ctx->device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ctx->device) != cudaSuccess) {
        delete ctx;
        return PG_ERR_CUDA;
    }
    ctx->sm_count = prop.multiProcessorCount;
    ctx->n = n_seq;
    ctx->npairs = n_seq * (n_seq - 1) / 2;
    *out = ctx; // from here on errors leave a context whose message can be read; caller destroys it

    DevProblem &dp = ctx->dp;
    memset(&dp, 0, sizeof(dp));
    dp.n = n_seq;
    dp.npairs = ctx->npairs;
    dp.gap_open = gap_open;
    dp.gap_ext = gap_ext;
    dp.gap_gap = gap_gap;
    dp.hash_type = PG_HASH_FZORDER; // CoordHash.cpp:17-18 defaults
    dp.hash_shift = 12;

    PG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    PG_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));

    // residues: one arena, each sequence padded with a trailing 0 (Node.cpp:225 reads seq[len], SURVEY F14)
    size_t seq_bytes = 0;
    std::vector<size_t> seq_off(n_seq);
    int max_len = 0;
    for (int i = 0; i < n_seq; i++) {
        ctx->len[i] = dp.len[i] = lens[i];
        ctx->seqs.emplace_back(seqs[i], seqs[i] + lens[i]);
        for (int j = 0; j < lens[i]; j++)
            if ((unsigned char)seqs[i][j] >= 90)
                return pg_fail(ctx, PG_ERR_ARG, "residue outside the 90x90 cost table (Cost.h:49: pam250['Z']['Z'])");
        seq_off[i] = seq_bytes;
        seq_bytes += ((size_t)lens[i] + 1 + 15) & ~size_t(15);
        max_len = std::max(max_len, lens[i]);
    }
    std::vector<uint8_t> hseq(seq_bytes, 0);
    for (int i = 0; i < n_seq; i++) memcpy(hseq.data() + seq_off[i], seqs[i], (size_t)lens[i]);
    PG_CUDA(ctx, cudaMalloc(&ctx->d_seq, seq_bytes));
    PG_CUDA(ctx, cudaMemcpy(ctx->d_seq, hseq.data(), seq_bytes, cudaMemcpyHostToDevice));
    for (int i = 0; i < n_seq; i++) dp.seq[i] = ctx->d_seq + seq_off[i];

    // cost table
    std::vector<int32_t> hcost(90 * 90);
    if (cost90x90)
        memcpy(hcost.data(), cost90x90, sizeof(int32_t) * 8100);
    else
        pg_default_cost_table(hcost.data());
    bool nonneg = gap_open >= 0 && gap_ext >= 0;
    for (int32_t v : hcost) nonneg = nonneg && v >= 0;
    ctx->cost_u8 = true;
    for (int32_t v : hcost) ctx->cost_u8 = ctx->cost_u8 && v >= 0 && v <= 255;
    {
        bool seen[90] = {false};
        for (const std::string &q : ctx->seqs)
            for (unsigned char ch : q) seen[ch] = true;
        ctx->n_alpha = 0;
        for (bool b : seen) ctx->n_alpha += b ? 1 : 0;
    }
    ctx->cost = hcost;
    PG_CUDA(ctx, cudaMalloc(&ctx->d_cost, sizeof(int32_t) * 8100));
    PG_CUDA(ctx, cudaMemcpy(ctx->d_cost, hcost.data(), sizeof(int32_t) * 8100, cudaMemcpyHostToDevice));
    dp.cost = ctx->d_cost;

    // packed-key geometry
    int kb = 1;
    while ((1 << kb) <= max_len) kb++;
    dp.key_bits = kb;
    if (n_seq * kb > 128) return pg_fail(ctx, PG_ERR_UNSUPPORTED, "packed coordinate key exceeds 128 bits");

    // pair geometry + table arena; a cell never exceeds the all-gaps path cost
    long long bound = 0;
    size_t cells = 0;
    int k = 0;
    for (int i = 0; i < n_seq - 1; i++) {
        for (int j = i + 1; j < n_seq; j++, k++) { // HeuristicHPair.cpp:54-61 order
            PairGeom g;
            g.a = i;
            g.b = j;
            g.rows = lens[i] + 1;
            g.cols = lens[j] + 1;
            g.pitch = (g.cols + 7) & ~7;
            g.offset = cells;
            cells += ((size_t)g.rows * g.pitch + 127) & ~size_t(127);
            ctx->pairs.push_back(g);
            dp.pa[k] = (uint8_t)i;
            dp.pb[k] = (uint8_t)j;
            dp.cols[k] = g.pitch;
            dp.w[k] = w_int ? w_int[i * n_seq + j] : 1;
            bound = std::max(bound, (long long)std::max(gap_open, gap_ext) * (lens[i] + lens[j]));
        }
    }
    ctx->table_cells = cells;
    dp.cell16 = (nonneg && bound < 65536) ? 1 : 0;
    const size_t cell_bytes = dp.cell16 ? 2 : 4;
    PG_CUDA(ctx, cudaMalloc(&ctx->d_tables, cells * cell_bytes));
    for (int p = 0; p < ctx->npairs; p++) dp.table[p] = (const char *)ctx->d_tables + ctx->pairs[p].offset * cell_bytes;
    return PG_OK;
}

extern "C" void pg_ctx_destroy(pg_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    pg_search_free(ctx);
    if (ctx->d_seq) cudaFree(ctx->d_seq);
    if (ctx->d_cost) cudaFree(ctx->d_cost);
    if (ctx->d_tables) cudaFree(ctx->d_tables);
    for (int i = 0; i < 2; i++)
        if (ctx->d_stage[i]) cudaFree(ctx->d_stage[i]);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    delete ctx;
}

extern "C" int pg_ctx_set_stream(pg_ctx *ctx, void *stream)
{
    if (!ctx) return PG_ERR_ARG;
    // NULL is the legacy default stream, as everywhere in CUDA (torch's default stream has handle 0); (void*)-1 = own
    ctx->stream = stream == (void *)-1 ? ctx->own_stream : (stream ? (cudaStream_t)stream : cudaStreamLegacy);
    return PG_OK;
}

extern "C" int pg_build_pair_tables(pg_ctx *ctx, float *kernel_ms)
{
    if (!ctx) return PG_ERR_ARG;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = pg_launch_pair_dp(ctx, kernel_ms);
    if (rc == PG_OK) ctx->tables_built = true;
    return rc;
}

extern "C" int pg_pair_table_shape(const pg_ctx *ctx, int pair, int *rows, int *cols)
{
    if (!ctx || pair < 0 || pair >= ctx->npairs || !rows || !cols) return PG_ERR_ARG;
    *rows = ctx->pairs[pair].rows;
    *cols = ctx->pairs[pair].cols;
    return PG_OK;
}

extern "C" int pg_copy_pair_table(pg_ctx *ctx, int pair, int32_t *out)
{
    if (!ctx || pair < 0 || pair >= ctx->npairs || !out) return PG_ERR_ARG;
    if (!ctx->tables_built) return pg_fail(ctx, PG_ERR_STATE, "pg_build_pair_tables has not run");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    const PairGeom &g = ctx->pairs[pair];
    const size_t n = (size_t)g.rows * g.cols;
    if (ctx->dp.cell16) { // stored rows are pitched: gather the logical rows x cols
        std::vector<uint16_t> tmp(n);
        PG_CUDA(ctx, cudaMemcpy2D(tmp.data(), (size_t)g.cols * 2, ctx->dp.table[pair], (size_t)g.pitch * 2, (size_t)g.cols * 2, g.rows, cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < n; i++) out[i] = tmp[i];
    } else {
        PG_CUDA(ctx, cudaMemcpy2D(out, (size_t)g.cols * 4, ctx->dp.table[pair], (size_t)g.pitch * 4, (size_t)g.cols * 4, g.rows, cudaMemcpyDeviceToHost));
    }
    return PG_OK;
}

extern "C" int pg_calculate_h(pg_ctx *ctx, const uint16_t *coords, int64_t n, int32_t *out)
{
    if (!ctx || n < 0 || (n > 0 && (!coords || !out))) return PG_ERR_ARG;
    if (!ctx->tables_built) return pg_fail(ctx, PG_ERR_STATE, "pg_build_pair_tables has not run");
    if (n == 0) return PG_OK;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    void *d_in, *d_out;
    int rc;
    if ((rc = pg_stage(ctx, 0, (size_t)n * ctx->n * 2, &d_in)) != PG_OK) return rc;
    if ((rc = pg_stage(ctx, 1, (size_t)n * 4, &d_out)) != PG_OK) return rc;
    PG_CUDA(ctx, cudaMemcpyAsync(d_in, coords, (size_t)n * ctx->n * 2, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = pg_launch_calc_h(ctx, (const uint16_t *)d_in, n, (int32_t *)d_out, ctx->stream)) != PG_OK) return rc;
    PG_CUDA(ctx, cudaMemcpyAsync(out, d_out, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PG_OK;
}

extern "C" int pg_configure_hash(pg_ctx *ctx, int hash_type, int hash_shift)
{
    if (!ctx || hash_type < 0 || hash_type > 3) return PG_ERR_ARG;
    if (hash_shift < 0 || hash_shift > 21) return pg_fail(ctx, PG_ERR_HASH_SHIFT, "Invalid Hash Shift"); // CoordHash.cpp:241
    ctx->dp.hash_type = hash_type;
    ctx->dp.hash_shift = hash_shift;
    return PG_OK;
}

extern "C" int pg_owner(pg_ctx *ctx, const uint16_t *coords, int64_t n, int size, uint32_t *out)
{
    if (!ctx || n < 0 || size < 1 || (n > 0 && (!coords || !out))) return PG_ERR_ARG;
    if (n == 0) return PG_OK;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    void *d_in, *d_out;
    int rc;
    if ((rc = pg_stage(ctx, 0, (size_t)n * ctx->n * 2, &d_in)) != PG_OK) return rc;
    if ((rc = pg_stage(ctx, 1, (size_t)n * 4, &d_out)) != PG_OK) return rc;
    PG_CUDA(ctx, cudaMemcpyAsync(d_in, coords, (size_t)n * ctx->n * 2, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = pg_launch_owner(ctx, (const uint16_t *)d_in, n, size, (uint32_t *)d_out, ctx->stream)) != PG_OK) return rc;
    PG_CUDA(ctx, cudaMemcpyAsync(out, d_out, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return PG_OK;
}

extern "C" int pg_expand_batch_dev(pg_ctx *ctx, const void *d_parents, int64_t k, int vec_size, void *d_out_succ,
                                   int32_t *d_out_counts, void *stream)
{
    if (!ctx || k < 0 || vec_size < 1 || vec_size > 64 || (k > 0 && (!d_parents || !d_out_succ || !d_out_counts))) return PG_ERR_ARG;
    if (!ctx->tables_built) return pg_fail(ctx, PG_ERR_STATE, "pg_build_pair_tables has not run");
    if (((uintptr_t)d_out_succ & 15) || ((uintptr_t)d_parents & 3)) return pg_fail(ctx, PG_ERR_ARG, "device buffers must be 16-byte aligned");
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    return pg_launch_expand(ctx, d_parents, k, vec_size, d_out_succ, d_out_counts, (cudaStream_t)stream); // NULL = the legacy default stream, as in CUDA
}

// Host-pointer form: chunks of parents are copied in, expanded and copied out,
// two chunks in flight on two streams so copies overlap the kernel when the
// host buffers are pinned.
extern "C" int pg_expand_batch(pg_ctx *ctx, const void *parents, int64_t k, int vec_size, void *out_succ, int32_t *out_counts)
{
    if (!ctx || k < 0 || vec_size < 1 || vec_size > 64 || (k > 0 && (!parents || !out_succ || !out_counts))) return PG_ERR_ARG;
    if (!ctx->tables_built) return pg_fail(ctx, PG_ERR_STATE, "pg_build_pair_tables has not run");
    if (k == 0) return PG_OK;
    PG_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t nstride = pg_node_stride(ctx->n), sstride = pg_succ_stride(ctx->n);
    const size_t S = ((size_t)1 << ctx->n) - 1;
    // chunk so that one chunk's records are about 64 MiB
    int64_t chunk = std::max<int64_t>(1, (int64_t)((64u << 20) / (S * sstride)));
    chunk = std::min<int64_t>(chunk, k);
    const size_t in_b = (size_t)chunk * nstride, out_b = (size_t)chunk * S * sstride, cnt_b = (size_t)chunk * 4;
    const size_t in_off = 0, cnt_off = (in_b + 255) & ~size_t(255), out_off = (cnt_off + cnt_b + 255) & ~size_t(255);
    const size_t per = out_off + out_b;
    cudaStream_t st[2] = {ctx->stream, ctx->stream2};
    char *buf[2];
    int rc;
    for (int i = 0; i < 2; i++) {
        void *pbuf;
        if ((rc = pg_stage(ctx, i, per, &pbuf)) != PG_OK) return rc;
        buf[i] = (char *)pbuf;
    }
    int which = 0;
    for (int64_t off = 0; off < k; off += chunk, which ^= 1) {
        const int64_t m = std::min(chunk, k - off);
        char *b = buf[which];
        cudaStream_t s = st[which];
        PG_CUDA(ctx, cudaMemcpyAsync(b + in_off, (const char *)parents + off * nstride, (size_t)m * nstride, cudaMemcpyHostToDevice, s));
        if ((rc = pg_launch_expand(ctx, b + in_off, m, vec_size, b + out_off, (int32_t *)(b + cnt_off), s)) != PG_OK) return rc;
        PG_CUDA(ctx, cudaMemcpyAsync((char *)out_succ + (size_t)off * S * sstride, b + out_off, (size_t)m * S * sstride,
                                     cudaMemcpyDeviceToHost, s));
        PG_CUDA(ctx, cudaMemcpyAsync(out_counts + off, b + cnt_off, (size_t)m * 4, cudaMemcpyDeviceToHost, s));
    }
    PG_CUDA(ctx, cudaStreamSynchronize(st[0]));
    PG_CUDA(ctx, cudaStreamSynchronize(st[1]));
    return PG_OK;
}
