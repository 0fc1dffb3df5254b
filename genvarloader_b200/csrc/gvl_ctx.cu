// gvl_ctx.cu -- context, workspace and error plumbing of the C ABI (include/gvl_b200.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "gvl_internal.cuh"

namespace gvl {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

template <typename T>
static int regrow(T *&p, int64_t need) {
    if (p) GVL_CUDA(cudaFree(p));
    p = nullptr;
    GVL_CUDA(cudaMalloc(&p, sizeof(T) * (size_t)need));
    return GVL_OK;
}

int ensure_rows(gvl_ctx *ctx, gvl_workspace &ws, int64_t n_work) {
    (void)ctx;
    if (n_work <= ws.rows_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());  // nothing may still be reading the old buffers
    int64_t cap = n_work + n_work / 2 + 64;
    int rc;
    if ((rc = regrow(ws.rows, cap))) return rc;
    if ((rc = regrow(ws.tile_off, cap + 1))) return rc;
    if ((rc = regrow(ws.row_len, cap))) return rc;
    if ((rc = regrow(ws.m_off, cap))) return rc;
    if ((rc = regrow(ws.m_len, cap))) return rc;
    ws.rows_cap = cap;
    return GVL_OK;
}

int ensure_records(gvl_ctx *ctx, gvl_workspace &ws, int64_t n_rec) {
    (void)ctx;
    if (n_rec <= ws.rec_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    int64_t cap = n_rec + n_rec / 2 + 1024;
    int rc;
    if ((rc = regrow(ws.rec.a, cap))) return rc;
    if ((rc = regrow(ws.rec.n, cap))) return rc;
    if ((rc = regrow(ws.rec.src, cap))) return rc;
    if ((rc = regrow(ws.rec.resume, cap))) return rc;
    if ((rc = regrow(ws.rec.vidx, cap))) return rc;
    if ((rc = regrow(ws.rec.vpos, cap))) return rc;
    ws.rec_cap = cap;
    return GVL_OK;
}

int ensure_merged(gvl_ctx *ctx, gvl_workspace &ws, int64_t n) {
    (void)ctx;
    if (n <= ws.m_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    int64_t cap = n + n / 2 + 1024;
    int rc;
    if ((rc = regrow(ws.m_pos, cap))) return rc;
    if ((rc = regrow(ws.m_key, cap))) return rc;
    ws.m_cap = cap;
    return GVL_OK;
}

int ensure_dir(gvl_ctx *ctx, gvl_workspace &ws, int64_t n) {
    (void)ctx;
    if (n <= ws.dir_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    int64_t cap = n + n / 2 + 1024;
    int rc;
    if ((rc = regrow(ws.dir, cap))) return rc;
    ws.dir_cap = cap;
    return GVL_OK;
}

int ensure_trecs(gvl_ctx *ctx, gvl_workspace &ws, int64_t n) {
    (void)ctx;
    if (n <= ws.trec_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    int64_t cap = n + n / 2 + 1024;
    if (ws.trecs) GVL_CUDA(cudaFree(ws.trecs));
    ws.trecs = nullptr;
    GVL_CUDA(cudaMalloc(&ws.trecs, 32 * (size_t)cap + 64));  // (32-byte records + slack for aligned bulk copies)
    ws.trec_cap = cap;
    return GVL_OK;
}

int ensure_tdesc(gvl_ctx *ctx, gvl_workspace &ws, int64_t n) {
    (void)ctx;
    if (n <= ws.tdesc_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    int64_t cap = n + n / 2 + 256;
    if (ws.tdesc) GVL_CUDA(cudaFree(ws.tdesc));
    ws.tdesc = nullptr;
    ws.tdesc_cap = ws.tdesc_bytes = 0;
    GVL_CUDA(cudaMalloc(&ws.tdesc, GVL_TILE_DESC_BYTES * (size_t)cap));
    ws.tdesc_cap = cap;
    ws.tdesc_bytes = GVL_TILE_DESC_BYTES * cap;
    return GVL_OK;
}

static void free_workspace(gvl_workspace &ws) {
    cudaFree(ws.tdesc);
    cudaFree(ws.trecs);
    cudaFree(ws.dir);
    cudaFree(ws.m_pos);
    cudaFree(ws.m_key);
    cudaFree(ws.m_off);
    cudaFree(ws.m_len);
    cudaFree(ws.rows);
    cudaFree(ws.tile_off);
    cudaFree(ws.row_len);
    cudaFree(ws.rec.a);
    cudaFree(ws.rec.n);
    cudaFree(ws.rec.src);
    cudaFree(ws.rec.resume);
    cudaFree(ws.rec.vidx);
    cudaFree(ws.rec.vpos);
}

}  // namespace gvl

using namespace gvl;

extern "C" {

const char *gvl_last_error(void) { return g_err; }

int64_t gvl_launch_count(int reset) {
    return reset ? g_launches.exchange(0) : g_launches.load();
}

int gvl_ctx_create(int device, gvl_ctx **out) {
    if (!out) return fail(GVL_ERR_ARG, "gvl_ctx_create: out is NULL");
    int n = 0;
    GVL_CUDA(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(GVL_ERR_ARG, "gvl_ctx_create: device %d of %d", device, n);
    GVL_CUDA(cudaSetDevice(device));
    gvl_ctx *ctx = new gvl_ctx();
    ctx->device = device;
    ctx->own_stream = nullptr;
    memset(&ctx->hap, 0, sizeof(ctx->hap));
    memset(&ctx->trk, 0, sizeof(ctx->trk));
    ctx->dev_words = nullptr;
    ctx->host_words = nullptr;
    ctx->trk_desc = nullptr;
    ctx->plan_valid = false;
    ctx->n_work = 0;
    ctx->fixed_len = -1;
    ctx->total = -1;
    ctx->plan_out_offsets = nullptr;
    ctx->last_exec_kernel = 0;
    ctx->zeros = nullptr;
    ctx->trk_params = nullptr;
    ctx->trk_plan_valid = false;
    ctx->zeros_bytes = 0;
    ctx->pinned = nullptr;
    ctx->pinned_bytes = 0;
    ctx->host_out_offsets_dev = nullptr;
    memset(&ctx->host_tab, 0, sizeof(ctx->host_tab));
    cudaError_t e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->dev_words, sizeof(int64_t) * 2 * W_COUNT);
    if (e == cudaSuccess) e = cudaMemset(ctx->dev_words, 0, sizeof(int64_t) * 2 * W_COUNT);
    if (e == cudaSuccess) e = cudaMalloc(&ctx->trk_desc, GVL_TRK_DESC_BYTES);
    if (e == cudaSuccess) e = cudaHostAlloc(&ctx->host_words, sizeof(int64_t) * 2 * W_COUNT, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        gvl_ctx_destroy(ctx);
        return fail(GVL_ERR_CUDA, "gvl_ctx_create: %s", cudaGetErrorString(e));
    }
    *out = ctx;
    return GVL_OK;
}

void gvl_ctx_destroy(gvl_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    free_workspace(ctx->hap);
    free_workspace(ctx->trk);
    cudaFree(ctx->dev_words);
    cudaFree(ctx->trk_desc);
    cudaFree(ctx->zeros);
    cudaFree(ctx->var_scratch);
    cudaFree(ctx->itv_counts);
    cudaFree(ctx->ritv_ws);
    free(ctx->trk_params);
    if (ctx->host_words) cudaFreeHost(ctx->host_words);
    for (auto &kv : ctx->statics) cudaFree(kv.second.dev);
    for (auto &kv : ctx->packed_refs) cudaFree(kv.second);
    for (auto &s : ctx->scratch) cudaFree(s.first);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (auto &sl : ctx->stage) {
        if (sl.host) cudaFreeHost(sl.host);
        if (sl.ev) cudaEventDestroy(sl.ev);
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

int gvl_ctx_check(gvl_ctx *ctx, gvl_stream stream) {
    if (!ctx) return fail(GVL_ERR_ARG, "gvl_ctx_check: ctx is NULL");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    GVL_CUDA(cudaMemcpyAsync(ctx->host_words, ctx->dev_words, sizeof(int64_t) * 2 * W_COUNT, cudaMemcpyDeviceToHost, st));
    GVL_CUDA(cudaStreamSynchronize(st));
    if (ctx->host_words[W_STATUS] != 0 || ctx->host_words[W_COUNT + W_STATUS] != 0) {
        int64_t s = ctx->host_words[W_STATUS] | ctx->host_words[W_COUNT + W_STATUS];
        cudaMemsetAsync(ctx->dev_words + W_STATUS, 0, sizeof(int64_t), st);
        cudaMemsetAsync(ctx->dev_words + W_COUNT + W_STATUS, 0, sizeof(int64_t), st);
        return fail(GVL_ERR_CAPACITY, "device workspace overflow (status=%lld): raise max_records", (long long)s);
    }
    return GVL_OK;
}

}  // extern "C"
