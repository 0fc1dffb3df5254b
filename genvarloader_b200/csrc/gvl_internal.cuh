// gvl_internal.cuh -- helpers private to the library (not part of the C ABI).
#pragma once
#include "gvl_common.cuh"

namespace gvl {

int fail(int code, const char *fmt, ...);
void count_launch(int n = 1);
int ensure_rows(gvl_ctx *ctx, gvl_workspace &ws, int64_t n_work);
int ensure_records(gvl_ctx *ctx, gvl_workspace &ws, int64_t n_rec);
int ensure_merged(gvl_ctx *ctx, gvl_workspace &ws, int64_t n);
int ensure_dir(gvl_ctx *ctx, gvl_workspace &ws, int64_t n);
int ensure_trecs(gvl_ctx *ctx, gvl_workspace &ws, int64_t n);
int ensure_tdesc(gvl_ctx *ctx, gvl_workspace &ws, int64_t n);
int ensure_zeros(gvl_ctx *ctx, int64_t bytes, cudaStream_t st);
int ensure_var_scratch(gvl_ctx *ctx, int64_t bytes);
// off[0] = 0, off[i + 1] = lengths[0] + ... + lengths[i]: the offset scan of the variants tail (gvl_variants.cu) over a
// device array of lengths
int scan_lengths(gvl_ctx *ctx, const int64_t *lengths, int64_t n, int64_t *off, cudaStream_t st);

#define GVL_CUDA(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return gvl::fail(GVL_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
    } while (0)

#define GVL_LAUNCH_CHECK()                                                                              \
    do {                                                                                                \
        cudaError_t _e = cudaGetLastError();                                                            \
        if (_e != cudaSuccess)                                                                          \
            return gvl::fail(GVL_ERR_CUDA, "%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
        gvl::count_launch();                                                                            \
    } while (0)

// A plan kernel's rows take their record space from words[W_CURSOR] (and the svar2 merge from words[W_MERGE_CURSOR]).
// The row that finishes LAST puts both cursors and the counter back to zero, so the words need no memset (or zeroing
// kernel) before the next plan: one node less per batch on the stream, and safe under CUDA-graph replay because every
// launch leaves the words as it found them.  Called by one thread per row, after the row's last global write.
__device__ __forceinline__ void plan_row_done(int64_t *words, int64_t n_work) {
    __threadfence();
    const unsigned long long prev = atomicAdd((unsigned long long *)&words[W_DONE], 1ull);
    if (prev + 1 == (unsigned long long)n_work) {
        words[W_CURSOR] = 0;
        words[W_MERGE_CURSOR] = 0;
        words[W_DONE] = 0;
        __threadfence();
    }
}

// ---- where a row's variant list comes from -------------------------------------------
struct RowVars {
    const int32_t *gv;    // SVAR1: variant indices of the row; merged lists: keys of the row
    const int32_t *mpos;  // merged lists: positions of the row (NULL for SVAR1)
    int64_t nvar;
};

__device__ __forceinline__ RowVars row_vars(const gvl_sparse_tables &tab, const MergedLists &M, const int64_t *goi,
                                            int64_t k) {
    RowVars r;
    if (M.key) {
        const int64_t o = M.off[k];
        r.gv = M.key + o;
        r.mpos = M.pos + o;
        r.nvar = M.len[k];
    } else {
        const int64_t o_idx = goi[k];
        const int64_t o_s = tab.geno_starts[o_idx];
        r.gv = tab.geno_v_idxs + o_s;
        r.mpos = nullptr;
        r.nvar = imax64(tab.geno_stops[o_idx] - o_s, 0);
    }
    return r;
}

// variant i of a row: table index vi, position
__device__ __forceinline__ int64_t var_pos(const gvl_sparse_tables &tab, const RowVars &r, int64_t i, int32_t vi) {
    return r.mpos ? (int64_t)r.mpos[i] : (int64_t)tab.v_starts[vi];
}

// ALT bytes of variant (i, vi): offset into alt_alleles (>= 0) or, for a pure deletion of the svar2 source
// (empty ALT, src/reconstruct/mod.rs:720-733), the anchor base ref[pos] encoded as ~(absolute ref offset)
__device__ __forceinline__ void var_alt(const gvl_sparse_tables &tab, const RowVars &r, int32_t vi, int64_t pos,
                                        int64_t c_s, int64_t &aoff, int64_t &alen) {
    aoff = tab.alt_offsets[vi];
    alen = tab.alt_offsets[vi + 1] - aoff;
    if (r.mpos && alen == 0) {
        aoff = ~(c_s + pos);
        alen = 1;
    }
}

// ---- TMA 1-D bulk copy (cp.async.bulk, SASS: UBLKCP) + mbarrier --------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // make the init visible to the async proxy
}

__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// global -> shared bulk copy; dst, src 16-byte aligned, bytes a multiple of 16; completes on `bar`
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// Ampere-style asynchronous 16-byte copy global -> shared (SASS: LDGSTS), per-thread completion groups
__device__ __forceinline__ void cp_async16(uint32_t smem_dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t smem_dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// ---- small device helpers ----------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// last index i in [lo, hi) with arr[i] <= key, or lo-1 if none.  Warp-cooperative 32-ary search:
// every lane must call it with identical arguments; every lane gets the result.
__device__ __forceinline__ int64_t warp_upper_le(const int32_t *__restrict__ arr, int64_t lo, int64_t hi, int32_t key) {
    // invariant: answer in [lo-1, hi-1]
    const int lane = lane_id();
    while (hi - lo > 32) {
        int64_t step = (hi - lo + 31) / 32;  // 32 probes at lo + (lane+1)*step - 1 (clamped)
        int64_t idx = lo + (int64_t)(lane + 1) * step - 1;
        bool ok = (idx < hi) ? (arr[idx] <= key) : false;
        unsigned m = __ballot_sync(0xffffffffu, ok);
        int cnt = __popc(m);  // probes are monotone: first `cnt` lanes are <= key
        int64_t new_lo = lo + (int64_t)cnt * step;
        int64_t new_hi = imin64(hi, lo + (int64_t)(cnt + 1) * step - 1);
        // elements [lo, new_lo) are all <= key; element at new_hi (if < hi) is > key
        lo = new_lo;
        hi = new_hi;
        if (lo > hi) hi = lo;
    }
    int64_t idx = lo + lane;
    bool ok = (idx < hi) ? (arr[idx] <= key) : false;
    unsigned m = __ballot_sync(0xffffffffu, ok);
    return lo + __popc(m) - 1;
}

}  // namespace gvl
