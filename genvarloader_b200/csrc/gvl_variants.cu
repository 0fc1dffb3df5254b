// gvl_variants.cu -- the `variants` / `variant-windows` outputs (SURVEY.md §8 f4 tail): per (region, sample, ploid) row the
// variant indices, positions, indel lengths and allele byte strings themselves instead of the reconstructed haplotype.
//   src/variants/mod.rs:6-49      gather_rows_{i32,f32}      rows of a sparse-genotype CSR, back to back
//   src/variants/mod.rs:52-78     gather_alleles             allele byte strings of the selected variants
//   src/variants/mod.rs:90-108    rc_alleles_inplace         reverse-complement the alleles of negative-strand rows
//   src/variants/mod.rs:112-153   compact_keep_{i32,f32}     drop filtered variants (AF filter), rebuild row offsets
//   src/variants/mod.rs:157-329   fill_empty_{scalar,fixed,seq}   one dummy variant for every empty row
//   src/variants/windows.rs:9-296 tokenize / fetch_windows / slice_flanks / assemble_alt_window / assemble_*_mode
//
// Every one of them is "lengths -> exclusive scan -> ragged copy".  On the device that is ONE pattern:
//   * scan_offsets<F>: three launches (per-block sums of F(i), spine, per-block rescan + write) -- no atomics, so the
//     offsets are reproducible bit for bit and the kernels can sit in a CUDA graph;
//   * seg_emit_kernel<F>: one thread per OUTPUT element, which finds its segment with a binary search over the offsets
//     (they are L1/L2 resident: a few KB to a few MB) -- stores are perfectly coalesced and the work per thread does not
//     depend on how the lengths are distributed (allele strings are 1-50 bytes, genotype rows 0-5,000 entries).
// The byte volume is tiny next to reconstruction (tens of bytes per variant); the point is that the whole batch stays on
// the device and in this library.
#include <cstring>

#include "gvl_internal.cuh"

using namespace gvl;

namespace {

constexpr int SCAN_T = 256;             // threads per scan CTA
constexpr int SCAN_I = 8;               // consecutive items per thread
constexpr int SCAN_B = SCAN_T * SCAN_I;  // items per CTA
constexpr int SPINE_T = 1024;

// ---- block-wide inclusive scan of one int64 per thread (256 threads) ----
__device__ __forceinline__ int64_t block_incl_scan(int64_t x, int64_t *s_warp, int64_t &block_total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int64_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < SCAN_T / 32; w++) {
        const int64_t v = s_warp[w];
        if (w < warp) before += v;
        total += v;
    }
    block_total = total;
    return x + before;
}

template <class F>
__global__ void __launch_bounds__(SCAN_T) scan_sums_kernel(F f, int64_t n, int64_t *__restrict__ sums) {
    __shared__ int64_t s_warp[SCAN_T / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_B + (int64_t)threadIdx.x * SCAN_I;
    int64_t t = 0;
#pragma unroll
    for (int j = 0; j < SCAN_I; j++)
        if (base + j < n) t += f(base + j);
    int64_t total;
    block_incl_scan(t, s_warp, total);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

// exclusive scan of the block sums in place; one CTA, chunks of 1024 with a running carry
__global__ void __launch_bounds__(SPINE_T) scan_spine_kernel(int64_t *__restrict__ sums, int64_t nb) {
    __shared__ int64_t s_warp[SPINE_T / 32];
    __shared__ int64_t s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int64_t b0 = 0; b0 < nb; b0 += SPINE_T) {
        const int64_t k = b0 + tid;
        const int64_t v = k < nb ? sums[k] : 0;
        int64_t x = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        if (lane == 31) s_warp[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int64_t w = s_warp[lane];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int64_t y = __shfl_up_sync(0xffffffffu, w, d);
                if (lane >= d) w += y;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const int64_t incl = s_carry + (warp ? s_warp[warp - 1] : 0) + x;
        if (k < nb) sums[k] = incl - v;
        __syncthreads();
        if (tid == SPINE_T - 1) s_carry = incl;
        __syncthreads();
    }
}

template <class F>
__global__ void __launch_bounds__(SCAN_T) scan_write_kernel(F f, int64_t n, const int64_t *__restrict__ sums,
                                                            int64_t *__restrict__ off) {
    __shared__ int64_t s_warp[SCAN_T / 32];
    const int64_t base = (int64_t)blockIdx.x * SCAN_B + (int64_t)threadIdx.x * SCAN_I;
    int64_t v[SCAN_I];
    int64_t t = 0;
#pragma unroll
    for (int j = 0; j < SCAN_I; j++) {
        v[j] = base + j < n ? f(base + j) : 0;
        t += v[j];
    }
    int64_t total;
    int64_t run = sums[blockIdx.x] + block_incl_scan(t, s_warp, total) - t;  // elements before this thread's first item
    if (blockIdx.x == 0 && threadIdx.x == 0) off[0] = 0;
#pragma unroll
    for (int j = 0; j < SCAN_I; j++) {
        run += v[j];
        if (base + j < n) off[base + j + 1] = run;
    }
}

}  // namespace

namespace gvl {

int ensure_var_scratch(gvl_ctx *ctx, int64_t bytes) {
    if (bytes <= ctx->var_scratch_bytes) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    if (ctx->var_scratch) GVL_CUDA(cudaFree(ctx->var_scratch));
    ctx->var_scratch = nullptr;
    ctx->var_scratch_bytes = 0;
    const int64_t cap = ((imax64(bytes * 2, 65536) + 255) / 256) * 256;
    GVL_CUDA(cudaMalloc(&ctx->var_scratch, (size_t)cap));
    ctx->var_scratch_bytes = cap;
    return GVL_OK;
}

}  // namespace gvl

namespace {

// off[0] = 0, off[i + 1] = f(0) + ... + f(i) for i < n
template <class F>
int scan_offsets(gvl_ctx *ctx, F f, int64_t n, int64_t *off, cudaStream_t st) {
    if (n == 0) {
        GVL_CUDA(cudaMemsetAsync(off, 0, sizeof(int64_t), st));
        return GVL_OK;
    }
    const int64_t nb = (n + SCAN_B - 1) / SCAN_B;
    if (nb > 0x7fffffff) return fail(GVL_ERR_ARG, "variants: %lld items in one call", (long long)n);
    int rc;
    if ((rc = ensure_var_scratch(ctx, sizeof(int64_t) * nb))) return rc;
    int64_t *sums = (int64_t *)ctx->var_scratch;
    scan_sums_kernel<F><<<(unsigned)nb, SCAN_T, 0, st>>>(f, n, sums);
    GVL_LAUNCH_CHECK();
    scan_spine_kernel<<<1, SPINE_T, 0, st>>>(sums, nb);
    GVL_LAUNCH_CHECK();
    scan_write_kernel<F><<<(unsigned)nb, SCAN_T, 0, st>>>(f, n, sums, off);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

struct ArrayLen {
    const int64_t *len;
    __device__ int64_t operator()(int64_t i) const { return __ldg(len + i); }
};

// last segment s in [0, n_seg) with off[s] <= e (off[0] = 0 <= e always): empty segments are skipped
__device__ __forceinline__ int64_t seg_of(const int64_t *__restrict__ off, int64_t n_seg, int64_t e) {
    int64_t lo = 0, hi = n_seg;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(off + mid) <= e) lo = mid;
        else hi = mid;
    }
    return lo;
}

// one thread per element e of a ragged layout (`inner` consecutive elements per offset unit): f(segment, unit inside the
// segment, element inside the unit, e)
template <class F>
__global__ void __launch_bounds__(256) seg_emit_kernel(F f, const int64_t *__restrict__ off, int64_t n_seg, int64_t total,
                                                       int64_t inner) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t u = inner == 1 ? e : e / inner;
        const int64_t s = seg_of(off, n_seg, u);
        f(s, u - __ldg(off + s), e - u * inner, e);
    }
}

template <class F>
int seg_emit(F f, const int64_t *off, int64_t n_seg, int64_t total, int64_t inner, cudaStream_t st) {
    if (total <= 0 || n_seg <= 0) return GVL_OK;
    const int64_t blocks = imin64((total + 255) / 256, 148 * 16);
    seg_emit_kernel<F><<<(unsigned)blocks, 256, 0, st>>>(f, off, n_seg, total, inner);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

// one thread per item i < n: f(i)
template <class F>
__global__ void __launch_bounds__(256) for_each_kernel(F f, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) f(i);
}

template <class F>
int for_each(F f, int64_t n, cudaStream_t st) {
    if (n <= 0) return GVL_OK;
    const int64_t blocks = imin64((n + 255) / 256, 148 * 16);
    for_each_kernel<F><<<(unsigned)blocks, 256, 0, st>>>(f, n);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

// src/reverse.rs:45-53: A <-> T, C <-> G, every other byte unchanged
__device__ __forceinline__ uint8_t comp_byte(uint8_t v) {
    const uint8_t at = (v == 'A') | (v == 'T') ? 21 : 0;
    const uint8_t cg = (v == 'C') | (v == 'G') ? 4 : 0;
    return v ^ at ^ cg;
}

// ---------------------------------------------------------------- functors: lengths
struct RowLen {  // src/variants/mod.rs:14-17
    const int64_t *goi, *o_starts, *o_stops;
    __device__ int64_t operator()(int64_t i) const {
        const int64_t g = goi[i];
        return o_stops[g] - o_starts[g];
    }
};
struct AlleleLen {  // :59-62
    const int32_t *v;
    const int64_t *aoff;
    __device__ int64_t operator()(int64_t i) const {
        const int64_t x = v[i];
        return aoff[x + 1] - aoff[x];
    }
};
struct KeepLen {  // :120-127
    const uint8_t *keep;
    __device__ int64_t operator()(int64_t j) const { return keep[j] ? 1 : 0; }
};
struct NonEmptyLen {  // :166-169, :213-216, :268-271: an empty row becomes one dummy variant
    const int64_t *off;
    __device__ int64_t operator()(int64_t i) const {
        const int64_t ln = off[i + 1] - off[i];
        return ln > 0 ? ln : 1;
    }
};
struct SrcSeqLen {  // :275-288
    const int64_t *src_var, *seq_off;
    int64_t dummy_len;
    __device__ int64_t operator()(int64_t e) const {
        const int64_t s = src_var[e];
        return s < 0 ? dummy_len : seq_off[s + 1] - seq_off[s];
    }
};
struct WindowLen {  // windows.rs:110-120 (reference window), :73-76 (flank5 . alt . flank3)
    const int32_t *v, *ilens;
    const int64_t *alt_off;
    int64_t flank;
    int alt;
    __device__ int64_t operator()(int64_t i) const {
        const int64_t x = v[i];
        if (alt) return 2 * flank + (alt_off[x + 1] - alt_off[x]);
        return 2 * flank + 1 - imin64((int64_t)ilens[x], 0);
    }
};

// ---------------------------------------------------------------- functors: element emitters
struct EmitRows {  // :19-27
    const int64_t *goi, *o_starts;
    const uint32_t *data;
    uint32_t *out;
    __device__ void operator()(int64_t s, int64_t k, int64_t, int64_t e) const { out[e] = __ldg(data + o_starts[goi[s]] + k); }
};
struct EmitVariantRows {  // EmitRows + the `table[v_idxs]` takes of start / ilen in the same pass (_flat_variants.py:948-953)
    const int64_t *goi, *o_starts;
    const int32_t *geno_v_idxs, *v_starts, *ilens;
    int32_t *v_out, *start_out, *ilen_out;
    __device__ void operator()(int64_t s, int64_t k, int64_t, int64_t e) const {
        const int32_t v = __ldg(geno_v_idxs + o_starts[goi[s]] + k);
        v_out[e] = v;
        if (start_out) start_out[e] = __ldg(v_starts + v);
        if (ilen_out) ilen_out[e] = __ldg(ilens + v);
    }
};
template <typename Tok, bool LUT>
struct EmitAlleles {  // :64-76 (+ windows.rs:9-22 tokenize)
    const int32_t *v;
    const int64_t *aoff;
    const uint8_t *bytes;
    const Tok *lut;
    Tok *out;
    __device__ void operator()(int64_t s, int64_t k, int64_t, int64_t e) const {
        const uint8_t b = __ldg(bytes + aoff[v[s]] + k);
        out[e] = LUT ? lut[b] : (Tok)b;
    }
};
struct EmitRc {  // :90-108: each thread of the first half of an allele swaps one pair
    uint8_t *data;
    const int64_t *seq_off, *var_off;
    const uint8_t *to_rc;
    int64_t n_rows;
    __device__ void operator()(int64_t a, int64_t k, int64_t, int64_t) const {
        const int64_t s0 = seq_off[a], len = seq_off[a + 1] - s0;
        if (k >= (len + 1) / 2) return;
        if (!to_rc[seg_of(var_off, n_rows, a)]) return;
        const int64_t i0 = s0 + k, i1 = s0 + len - 1 - k;
        const uint8_t x = data[i0], y = data[i1];
        data[i0] = comp_byte(y);
        data[i1] = comp_byte(x);
    }
};
struct EmitFillFixed {  // :218-232
    const uint32_t *data;
    const int64_t *off;
    uint32_t fill;
    int64_t inner;
    uint32_t *out;
    __device__ void operator()(int64_t row, int64_t k, int64_t j, int64_t e) const {
        const int64_t s = off[row];
        out[e] = off[row + 1] == s ? fill : __ldg(data + (s + k) * inner + j);
    }
};
struct EmitSrcVar {  // source variant of every variant of the filled layout (-1 = the dummy)
    const int64_t *var_off;
    int64_t *src_var;
    __device__ void operator()(int64_t row, int64_t k, int64_t, int64_t e) const {
        const int64_t s = var_off[row];
        src_var[e] = var_off[row + 1] == s ? -1 : s + k;
    }
};
template <typename T>
struct EmitFillSeq {  // :290-307
    const T *data, *dummy;
    const int64_t *src_var, *seq_off;
    T *out;
    __device__ void operator()(int64_t nv, int64_t k, int64_t, int64_t e) const {
        const int64_t s = src_var[nv];
        out[e] = s < 0 ? dummy[k] : __ldg(data + seq_off[s] + k);
    }
};

// byte w of the reference window [start - L, end + L) of variant x on contig c; outside the contig: pad (windows.rs:98-134)
struct Window {
    const int32_t *v, *v_contigs, *v_starts, *ilens;
    const uint8_t *ref;
    const int64_t *ref_off;
    int64_t flank;
    uint8_t pad;
    __device__ uint8_t at(int64_t i, int64_t x, int64_t w) const {
        const int64_t c = v_contigs ? v_contigs[i] : 0;
        const int64_t c_s = ref_off[c], c_len = ref_off[c + 1] - c_s;
        const int64_t pos = (int64_t)v_starts[x] - flank + w;
        return pos >= 0 && pos < c_len ? __ldg(ref + c_s + pos) : pad;
    }
    __device__ int64_t span(int64_t x) const { return 1 - imin64((int64_t)ilens[x], 0); }  // end - start
};
template <typename Tok>
struct EmitRefWindow {  // windows.rs:268-271
    Window W;
    const Tok *lut;
    Tok *out;
    __device__ void operator()(int64_t i, int64_t k, int64_t, int64_t e) const { out[e] = lut[W.at(i, W.v[i], k)]; }
};
template <typename Tok>
struct EmitAltWindow {  // windows.rs:55-90, :281-291
    Window W;
    const uint8_t *alt;
    const int64_t *alt_off;
    const Tok *lut;
    Tok *out;
    __device__ void operator()(int64_t i, int64_t k, int64_t, int64_t e) const {
        const int64_t x = W.v[i], L = W.flank, a0 = alt_off[x], alen = alt_off[x + 1] - a0;
        uint8_t b;
        if (k < L) b = W.at(i, x, k);
        else if (k < L + alen) b = __ldg(alt + a0 + k - L);
        else b = W.at(i, x, L + W.span(x) + (k - L - alen));
        out[e] = lut[b];
    }
};
template <typename Tok>
struct EmitFlanks {  // windows.rs:27-52, :196-214: [flank5 | flank3], 2L tokens per variant
    Window W;
    const Tok *lut;
    Tok *out;
    __device__ void operator()(int64_t e) const {
        const int64_t L = W.flank, i = e / (2 * L), k = e - i * 2 * L, x = W.v[i];
        out[e] = lut[k < L ? W.at(i, x, k) : W.at(i, x, L + W.span(x) + (k - L))];
    }
};

struct CompactOffsets {  // mod.rs:118-127: kept values before every row boundary
    const int64_t *pos, *row_off;
    int64_t *new_off;
    __device__ void operator()(int64_t i) const { new_off[i] = pos[row_off[i]] - pos[row_off[0]]; }
};
struct CompactScatter {  // mod.rs:128-133
    const uint32_t *src;
    const uint8_t *keep;
    const int64_t *pos;
    uint32_t *dst;
    __device__ void operator()(int64_t j) const {
        if (keep[j]) dst[pos[j]] = src[j];
    }
};
struct EmitExpand {  // np.repeat(values, np.diff(offsets)): the row's value for every variant of the row
    const uint32_t *values;
    uint32_t *out;
    __device__ void operator()(int64_t row, int64_t, int64_t, int64_t e) const { out[e] = values[row]; }
};
struct TakeU32 {
    const uint32_t *t;
    const int32_t *v;
    uint32_t *o;
    __device__ void operator()(int64_t i) const { o[i] = __ldg(t + v[i]); }
};

// ---------------------------------------------------------------- sizing and ring offsets
// One warp per genotype row: the lanes stride over the row's slice and reduce with a fixed shuffle tree, so a row of
// thousands of variants costs its warp ~len / 32 steps and an empty row costs one.  Integer sums: exact and reproducible.
constexpr int SIZE_T = 256;
constexpr int SIZE_ROWS = SIZE_T / 32;  // rows per CTA

__global__ void __launch_bounds__(SIZE_T)
    variant_row_sizes_kernel(const int64_t *__restrict__ goi, int64_t n_rows, const int64_t *__restrict__ o_starts,
                             const int64_t *__restrict__ o_stops, const int32_t *__restrict__ geno_v_idxs,
                             const int32_t *__restrict__ keep, const int64_t *__restrict__ alt_off,
                             const int64_t *__restrict__ ref_off, const int32_t *__restrict__ ilens, int64_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    for (int64_t r = (int64_t)blockIdx.x * SIZE_ROWS + (threadIdx.x >> 5); r < n_rows; r += (int64_t)gridDim.x * SIZE_ROWS) {
        const int64_t g = goi[r], lo = o_starts[g], hi = o_stops[g];
        int64_t n = 0, alt = 0, ref = 0, span = 0;
        for (int64_t k = lo + lane; k < hi; k += 32) {
            const int32_t v = __ldg(geno_v_idxs + k);
            if (keep && !__ldg(keep + v)) continue;
            n += 1;
            alt += __ldg(alt_off + v + 1) - __ldg(alt_off + v);
            if (ref_off) ref += __ldg(ref_off + v + 1) - __ldg(ref_off + v);
            span += 1 - imin64((int64_t)__ldg(ilens + v), 0);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            n += __shfl_xor_sync(0xffffffffu, n, d);
            alt += __shfl_xor_sync(0xffffffffu, alt, d);
            ref += __shfl_xor_sync(0xffffffffu, ref, d);
            span += __shfl_xor_sync(0xffffffffu, span, d);
        }
        if (lane < 4) out[r * 4 + lane] = lane == 0 ? n : lane == 1 ? alt : lane == 2 ? ref : span;
    }
}

// start of batch i of a ring: s_i = min(i * stride, n) over the items, or bounds[min(i * stride, n_bounds)]
struct RingBounds {
    const int64_t *bounds;
    int64_t stride, n, n_bounds;
    __device__ int64_t operator()(int64_t i) const {
        if (!bounds) return imin64(i * stride, n);
        return __ldg(bounds + imin64(i * stride, n_bounds));
    }
};

// batch i owns out[s_i + i .. s_{i+1} + i]: the last batch i with s_i + i <= e (K is tens: a short binary search)
__global__ void __launch_bounds__(256) rebase_offsets_kernel(const int64_t *__restrict__ off, RingBounds B, int64_t n_batches,
                                                             int64_t n_out, int64_t *__restrict__ out) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n_out; e += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = n_batches;
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (B(mid) + mid <= e) lo = mid;
            else hi = mid;
        }
        out[e] = __ldg(off + e - lo) - __ldg(off + B(lo));
    }
}

inline cudaStream_t S(gvl_stream s) { return (cudaStream_t)s; }

}  // namespace

namespace gvl {

int scan_lengths(gvl_ctx *ctx, const int64_t *lengths, int64_t n, int64_t *off, cudaStream_t st) {
    return scan_offsets(ctx, ArrayLen{lengths}, n, off, st);
}

}  // namespace gvl

#define VARG(cond, name) \
    if (!(cond)) return fail(GVL_ERR_ARG, name ": NULL argument or bad size")

extern "C" {

int gvl_dev_gather_rows_offsets(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_rows, const int64_t *o_starts,
                                const int64_t *o_stops, int64_t *out_offsets, gvl_stream stream) {
    VARG(ctx && out_offsets && n_rows >= 0 && (n_rows == 0 || (geno_offset_idx && o_starts && o_stops)),
         "gvl_dev_gather_rows_offsets");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return scan_offsets(ctx, RowLen{geno_offset_idx, o_starts, o_stops}, n_rows, out_offsets, S(stream));
}

int gvl_dev_gather_rows(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_rows, const int64_t *o_starts, const void *data,
                        const int64_t *out_offsets, int64_t total, void *out, gvl_stream stream) {
    VARG(ctx && n_rows >= 0 && total >= 0, "gvl_dev_gather_rows");
    if (n_rows == 0 || total == 0) return GVL_OK;
    VARG(geno_offset_idx && o_starts && data && out_offsets && out, "gvl_dev_gather_rows");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return seg_emit(EmitRows{geno_offset_idx, o_starts, (const uint32_t *)data, (uint32_t *)out}, out_offsets, n_rows, total, 1,
                    S(stream));
}

int gvl_dev_gather_variant_rows(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int64_t *geno_offset_idx, int64_t n_rows,
                                const int64_t *out_offsets, int64_t total, int32_t *v_idxs, int32_t *starts, int32_t *ilens,
                                gvl_stream stream) {
    VARG(ctx && tab && n_rows >= 0 && total >= 0, "gvl_dev_gather_variant_rows");
    if (n_rows == 0 || total == 0) return GVL_OK;
    VARG(geno_offset_idx && out_offsets && v_idxs && tab->geno_starts && tab->geno_v_idxs && (!starts || tab->v_starts) &&
             (!ilens || tab->ilens),
         "gvl_dev_gather_variant_rows");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return seg_emit(EmitVariantRows{geno_offset_idx, tab->geno_starts, tab->geno_v_idxs, tab->v_starts, tab->ilens, v_idxs, starts,
                                    ilens},
                    out_offsets, n_rows, total, 1, S(stream));
}

int gvl_dev_gather_alleles_offsets(gvl_ctx *ctx, const int32_t *v_idxs, int64_t n, const int64_t *allele_offsets,
                                   int64_t *seq_offsets, gvl_stream stream) {
    VARG(ctx && seq_offsets && n >= 0 && (n == 0 || (v_idxs && allele_offsets)), "gvl_dev_gather_alleles_offsets");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return scan_offsets(ctx, AlleleLen{v_idxs, allele_offsets}, n, seq_offsets, S(stream));
}

int gvl_dev_gather_alleles(gvl_ctx *ctx, const int32_t *v_idxs, int64_t n, const uint8_t *allele_bytes,
                           const int64_t *allele_offsets, const int64_t *seq_offsets, int64_t total, const void *lut,
                           int tok_bytes, void *out, gvl_stream stream) {
    VARG(ctx && n >= 0 && total >= 0, "gvl_dev_gather_alleles");
    if (lut && tok_bytes != 1 && tok_bytes != 4) return fail(GVL_ERR_ARG, "gvl_dev_gather_alleles: tokens of 1 or 4 bytes");
    if (n == 0 || total == 0) return GVL_OK;
    VARG(v_idxs && allele_bytes && allele_offsets && seq_offsets && out, "gvl_dev_gather_alleles");
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (!lut)
        return seg_emit(EmitAlleles<uint8_t, false>{v_idxs, allele_offsets, allele_bytes, nullptr, (uint8_t *)out}, seq_offsets, n,
                        total, 1, S(stream));
    if (tok_bytes == 1)
        return seg_emit(EmitAlleles<uint8_t, true>{v_idxs, allele_offsets, allele_bytes, (const uint8_t *)lut, (uint8_t *)out},
                        seq_offsets, n, total, 1, S(stream));
    return seg_emit(EmitAlleles<int32_t, true>{v_idxs, allele_offsets, allele_bytes, (const int32_t *)lut, (int32_t *)out},
                    seq_offsets, n, total, 1, S(stream));
}

int gvl_dev_rc_alleles(gvl_ctx *ctx, uint8_t *byte_data, const int64_t *seq_offsets, int64_t n_alleles,
                       const int64_t *var_offsets, int64_t n_rows, const uint8_t *to_rc_row, int64_t total_bytes,
                       gvl_stream stream) {
    VARG(ctx && n_alleles >= 0 && n_rows >= 0 && total_bytes >= 0, "gvl_dev_rc_alleles");
    if (n_alleles == 0 || n_rows == 0 || total_bytes == 0) return GVL_OK;
    VARG(byte_data && seq_offsets && var_offsets && to_rc_row, "gvl_dev_rc_alleles");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return seg_emit(EmitRc{byte_data, seq_offsets, var_offsets, to_rc_row, n_rows}, seq_offsets, n_alleles, total_bytes, 1,
                    S(stream));
}

int gvl_dev_compact_keep_offsets(gvl_ctx *ctx, const uint8_t *keep, int64_t n, const int64_t *row_offsets, int64_t n_rows,
                                 int64_t *pos, int64_t *new_offsets, gvl_stream stream) {
    VARG(ctx && pos && new_offsets && row_offsets && n >= 0 && n_rows >= 0 && (n == 0 || keep), "gvl_dev_compact_keep_offsets");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = scan_offsets(ctx, KeepLen{keep}, n, pos, S(stream)))) return rc;
    return for_each(CompactOffsets{pos, row_offsets, new_offsets}, n_rows + 1, S(stream));
}

int gvl_dev_compact_keep(gvl_ctx *ctx, const void *values, const uint8_t *keep, int64_t n, const int64_t *pos, void *out,
                         gvl_stream stream) {
    VARG(ctx && n >= 0, "gvl_dev_compact_keep");
    if (n == 0) return GVL_OK;
    VARG(values && keep && pos, "gvl_dev_compact_keep");
    GVL_CUDA(cudaSetDevice(ctx->device));
    // (out may be NULL when nothing is kept: never dereferenced then)
    return for_each(CompactScatter{(const uint32_t *)values, keep, pos, (uint32_t *)out}, n, S(stream));
}

int gvl_dev_fill_empty_offsets(gvl_ctx *ctx, const int64_t *offsets, int64_t n_rows, int64_t *new_offsets, gvl_stream stream) {
    VARG(ctx && offsets && new_offsets && n_rows >= 0, "gvl_dev_fill_empty_offsets");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return scan_offsets(ctx, NonEmptyLen{offsets}, n_rows, new_offsets, S(stream));
}

int gvl_dev_fill_empty_fixed(gvl_ctx *ctx, const void *data, const int64_t *offsets, int64_t n_rows, const int64_t *new_offsets,
                             int64_t new_total, int64_t inner, uint32_t fill_bits, void *out, gvl_stream stream) {
    VARG(ctx && n_rows >= 0 && new_total >= 0 && inner >= 0, "gvl_dev_fill_empty_fixed");
    if (n_rows == 0 || new_total == 0 || inner == 0) return GVL_OK;
    VARG(offsets && new_offsets && out, "gvl_dev_fill_empty_fixed");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return seg_emit(EmitFillFixed{(const uint32_t *)data, offsets, fill_bits, inner, (uint32_t *)out}, new_offsets, n_rows,
                    new_total * inner, inner, S(stream));
}

int gvl_dev_fill_empty_seq_offsets(gvl_ctx *ctx, const int64_t *var_offsets, int64_t n_rows, const int64_t *seq_offsets,
                                   int64_t dummy_len, const int64_t *new_var_offsets, int64_t n_new_vars, int64_t *src_var,
                                   int64_t *new_seq_offsets, gvl_stream stream) {
    VARG(ctx && var_offsets && new_var_offsets && new_seq_offsets && n_rows >= 0 && n_new_vars >= 0 && dummy_len >= 0 &&
             (n_new_vars == 0 || (src_var && seq_offsets)),
         "gvl_dev_fill_empty_seq_offsets");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = seg_emit(EmitSrcVar{var_offsets, src_var}, new_var_offsets, n_rows, n_new_vars, 1, S(stream)))) return rc;
    return scan_offsets(ctx, SrcSeqLen{src_var, seq_offsets, dummy_len}, n_new_vars, new_seq_offsets, S(stream));
}

int gvl_dev_fill_empty_seq(gvl_ctx *ctx, const void *data, int itemsize, const int64_t *seq_offsets, const void *dummy,
                           const int64_t *src_var, const int64_t *new_seq_offsets, int64_t n_new_vars, int64_t total, void *out,
                           gvl_stream stream) {
    VARG(ctx && n_new_vars >= 0 && total >= 0, "gvl_dev_fill_empty_seq");
    if (itemsize != 1 && itemsize != 4) return fail(GVL_ERR_ARG, "gvl_dev_fill_empty_seq: items of 1 or 4 bytes");
    if (n_new_vars == 0 || total == 0) return GVL_OK;
    VARG(src_var && new_seq_offsets && seq_offsets && out, "gvl_dev_fill_empty_seq");
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (itemsize == 1)
        return seg_emit(EmitFillSeq<uint8_t>{(const uint8_t *)data, (const uint8_t *)dummy, src_var, seq_offsets, (uint8_t *)out},
                        new_seq_offsets, n_new_vars, total, 1, S(stream));
    return seg_emit(EmitFillSeq<uint32_t>{(const uint32_t *)data, (const uint32_t *)dummy, src_var, seq_offsets, (uint32_t *)out},
                    new_seq_offsets, n_new_vars, total, 1, S(stream));
}

int gvl_dev_variant_windows_offsets(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *v_idxs, int64_t n,
                                    int64_t flank_len, int kind, int64_t *win_offsets, gvl_stream stream) {
    VARG(ctx && tab && win_offsets && n >= 0 && flank_len >= 0 && (n == 0 || v_idxs), "gvl_dev_variant_windows_offsets");
    if (kind != GVL_WINDOW_REF && kind != GVL_WINDOW_ALT)
        return fail(GVL_ERR_ARG, "gvl_dev_variant_windows_offsets: kind must be GVL_WINDOW_REF or GVL_WINDOW_ALT");
    if (n && (kind == GVL_WINDOW_ALT ? !tab->alt_offsets : !tab->ilens))
        return fail(GVL_ERR_ARG, "gvl_dev_variant_windows_offsets: variant table is NULL");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return scan_offsets(ctx, WindowLen{v_idxs, tab->ilens, tab->alt_offsets, flank_len, kind == GVL_WINDOW_ALT}, n, win_offsets,
                        S(stream));
}

int gvl_dev_variant_windows(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *v_idxs, const int32_t *v_contigs,
                            int64_t n, int64_t flank_len, int kind, uint8_t pad_char, const void *lut, int tok_bytes,
                            const int64_t *win_offsets, int64_t total, void *out, gvl_stream stream) {
    VARG(ctx && tab && n >= 0 && flank_len >= 0 && total >= 0, "gvl_dev_variant_windows");
    if (kind != GVL_WINDOW_REF && kind != GVL_WINDOW_ALT && kind != GVL_WINDOW_FLANKS)
        return fail(GVL_ERR_ARG, "gvl_dev_variant_windows: unknown kind");
    if (tok_bytes != 1 && tok_bytes != 4) return fail(GVL_ERR_ARG, "gvl_dev_variant_windows: tokens of 1 or 4 bytes");
    if (kind == GVL_WINDOW_FLANKS) total = n * 2 * flank_len;
    if (n == 0 || total == 0) return GVL_OK;
    VARG(v_idxs && lut && out && tab->v_starts && tab->ilens && tab->ref && tab->ref_offsets, "gvl_dev_variant_windows");
    if (kind != GVL_WINDOW_FLANKS && !win_offsets) return fail(GVL_ERR_ARG, "gvl_dev_variant_windows: win_offsets is NULL");
    if (kind == GVL_WINDOW_ALT && (!tab->alt_alleles || !tab->alt_offsets))
        return fail(GVL_ERR_ARG, "gvl_dev_variant_windows: ALT table is NULL");
    GVL_CUDA(cudaSetDevice(ctx->device));
    const Window W{v_idxs, v_contigs, tab->v_starts, tab->ilens, tab->ref, tab->ref_offsets, flank_len, pad_char};
    cudaStream_t st = S(stream);
    if (tok_bytes == 1) {
        const uint8_t *l = (const uint8_t *)lut;
        uint8_t *o = (uint8_t *)out;
        if (kind == GVL_WINDOW_REF) return seg_emit(EmitRefWindow<uint8_t>{W, l, o}, win_offsets, n, total, 1, st);
        if (kind == GVL_WINDOW_ALT)
            return seg_emit(EmitAltWindow<uint8_t>{W, tab->alt_alleles, tab->alt_offsets, l, o}, win_offsets, n, total, 1, st);
        return for_each(EmitFlanks<uint8_t>{W, l, o}, total, st);
    }
    const int32_t *l = (const int32_t *)lut;
    int32_t *o = (int32_t *)out;
    if (kind == GVL_WINDOW_REF) return seg_emit(EmitRefWindow<int32_t>{W, l, o}, win_offsets, n, total, 1, st);
    if (kind == GVL_WINDOW_ALT)
        return seg_emit(EmitAltWindow<int32_t>{W, tab->alt_alleles, tab->alt_offsets, l, o}, win_offsets, n, total, 1, st);
    return for_each(EmitFlanks<int32_t>{W, l, o}, total, st);
}

// np.repeat(values, np.diff(offsets)) for 4-byte values: the contig of every gathered variant from the contig of its row
// (_flat_variants.py:985-989)
int gvl_dev_expand_rows_u32(gvl_ctx *ctx, const void *values, const int64_t *offsets, int64_t n_rows, int64_t total, void *out,
                            gvl_stream stream) {
    VARG(ctx && n_rows >= 0 && total >= 0, "gvl_dev_expand_rows_u32");
    if (n_rows == 0 || total == 0) return GVL_OK;
    VARG(values && offsets && out, "gvl_dev_expand_rows_u32");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return seg_emit(EmitExpand{(const uint32_t *)values, (uint32_t *)out}, offsets, n_rows, total, 1, S(stream));
}

// table[v_idxs[i]] for a 4-byte table (start / ilen / info fields of the selected variants: `np.asarray(x)[v_idxs]`,
// python/genvarloader/_dataset/_flat_variants.py:948-953)
int gvl_dev_take_u32(gvl_ctx *ctx, const void *table, const int32_t *v_idxs, int64_t n, void *out, gvl_stream stream) {
    VARG(ctx && n >= 0, "gvl_dev_take_u32");
    if (n == 0) return GVL_OK;
    VARG(table && v_idxs && out, "gvl_dev_take_u32");
    GVL_CUDA(cudaSetDevice(ctx->device));
    return for_each(TakeU32{(const uint32_t *)table, v_idxs, (uint32_t *)out}, n, S(stream));
}

int gvl_dev_variant_row_sizes(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int64_t *geno_offset_idx, int64_t n_rows,
                              const int32_t *keep_table, const int64_t *ref_offsets, int64_t *out_sizes, gvl_stream stream) {
    VARG(ctx && tab && n_rows >= 0, "gvl_dev_variant_row_sizes");
    if (n_rows == 0) return GVL_OK;
    VARG(geno_offset_idx && out_sizes && tab->geno_starts && tab->geno_stops && tab->geno_v_idxs && tab->alt_offsets && tab->ilens,
         "gvl_dev_variant_row_sizes");
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t blocks = imin64((n_rows + SIZE_ROWS - 1) / SIZE_ROWS, 148 * 16);
    variant_row_sizes_kernel<<<(unsigned)blocks, SIZE_T, 0, S(stream)>>>(geno_offset_idx, n_rows, tab->geno_starts, tab->geno_stops,
                                                                          tab->geno_v_idxs, keep_table, tab->alt_offsets,
                                                                          ref_offsets, tab->ilens, out_sizes);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

int gvl_dev_rebase_offsets(gvl_ctx *ctx, const int64_t *offsets, int64_t n, const int64_t *bounds, int64_t n_bounds,
                           int64_t stride, int64_t n_batches, int64_t *out, gvl_stream stream) {
    VARG(ctx && n >= 0 && n_batches >= 1 && stride >= 0 && (!bounds || n_bounds >= 0), "gvl_dev_rebase_offsets");
    VARG(offsets && out, "gvl_dev_rebase_offsets");
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_out = n + n_batches;
    const int64_t blocks = imin64((n_out + 255) / 256, 148 * 16);
    rebase_offsets_kernel<<<(unsigned)blocks, 256, 0, S(stream)>>>(offsets, RingBounds{bounds, stride, n, n_bounds}, n_batches,
                                                                   n_out, out);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

}  // extern "C"
