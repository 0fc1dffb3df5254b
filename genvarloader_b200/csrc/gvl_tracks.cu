// gvl_tracks.cu -- indel-aware track realignment on sm_100a (include/gvl_b200.h:
// gvl_dev_realign_tracks, gvl_dev_intervals_to_tracks).
//
// Reference path replaced: intervals_and_realign_track_fused (src/ffi/mod.rs:2553-2672) =
// intervals_to_tracks (src/intervals.rs:19-126) into a dense scratch -> shift_and_realign_tracks_sparse
// (src/tracks/mod.rs:224-406, 495-667) -> reverse_flat_rows_inplace (src/reverse.rs:25-38), called
// once per track from a Python loop (_dataset/_reconstruct.py:228-290).
//
// Here: ONE plan launch per batch (the variant state machine does not depend on the track), one tile-preparation
// launch and ONE execute launch for all tracks.  Each execute CTA owns a tile of TRK_TILE output values of one
// (track, row): it turns the tile's records and the stored intervals that reach into it into value markers in output
// coordinates (no dense scratch in HBM), then every thread writes chunks of 16 consecutive output values with 32-byte
// stores (source span copies, deletion/insertion fills, trailing zeros, reversal for negative strands).  Unsorted
// variant lists and dense sources resolve every value on its own.  gvl_tracks_exec.cuh has the details.
// The output is float32, bfloat16 or float16 (GVL_TRACK_*): one execute instantiation per type, values narrowed at the
// store.
//
// gvl_dev_track_intervals returns the stored intervals themselves instead of painting them: a count kernel (one warp per
// row, two 32-ary searches), the offset scan of the variants tail, and an emit kernel that copies each row's run.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <cstring>
#include <vector>

#include "gvl_internal.cuh"

namespace gvl {

constexpr int TRK_TILE = 8192;  // output values per execute CTA (one tile of one (track, row))

// =====================================================================================
// plan: the scan-based plan kernel of the haplotype path in track mode (gvl_plan_par.cuh, hap_plan_par_kernel<NT, true>;
// launched through gvl_trk_plan_launch, gvl_hap.cu) -- the same offset scan serves both paths
// =====================================================================================
// identity plan for intervals_to_tracks: one row per query, no records, source window = row
__global__ void paint_plan_kernel(int64_t n, const int32_t *__restrict__ starts, const int64_t *__restrict__ out_offsets,
                                  const uint8_t *__restrict__ to_rc, RowPlan *rows, int32_t *row_len) {
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n) return;
    int64_t length = imax64(out_offsets[q + 1] - out_offsets[q], 0);
    RowPlan rp;
    rp.out_off = out_offsets[q];
    rp.ref_base = 0;
    rp.rec_off = 0;
    rp.length = (int32_t)length;
    rp.contig_len = (int32_t)length;
    rp.lead_pad = 0;
    rp.ref0 = 0;
    rp.n_rec = 0;
    rp.rc = (to_rc && to_rc[q]) ? 1 : 0;  // negative-strand rows come out reversed (src/reverse.rs:25-38)
    rp.diff = 0;
    rp.q_start = starts[q];
    rows[q] = rp;
    row_len[q] = (int32_t)length;
}

// tile map for TRK_TILE-sized tiles (same scan as the haplotype path, different tile size)
__global__ void __launch_bounds__(1024) trk_tile_scan_kernel(int64_t n_work, const int32_t *__restrict__ row_len,
                                                             int64_t *tile_off) {
    __shared__ int64_t s_tile[32];
    __shared__ int64_t carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < n_work; base += 1024) {
        int64_t k = base + tid;
        int64_t til = (k < n_work) ? ((int64_t)row_len[k] + TRK_TILE - 1) / TRK_TILE : 0;
        int64_t x = til;
        for (int o = 1; o < 32; o <<= 1) {
            int64_t y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        if (lane == 31) s_tile[warp] = x;
        __syncthreads();
        if (warp == 0) {
            int64_t w = s_tile[lane];
            for (int o = 1; o < 32; o <<= 1) {
                int64_t y = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += y;
            }
            s_tile[lane] = w;
        }
        __syncthreads();
        if (k < n_work) tile_off[k] = carry + (warp ? s_tile[warp - 1] : 0) + x - til;
        __syncthreads();
        if (tid == 0) carry += s_tile[31];
        __syncthreads();
    }
    if (tid == 0) tile_off[n_work] = carry;
}

// =====================================================================================
// execute
// =====================================================================================
constexpr int MAX_TRACKS = 64;

struct TrkDesc {
    const int32_t *itv_starts;
    const int32_t *itv_ends;
    const float *itv_values;
    const int64_t *itv_offsets;
    const float *dense;            // non-NULL: dense f32 source windows instead of intervals
    const int64_t *dense_offsets;  //           i64[n_queries+1] offsets of each query's window
    int32_t strategy;
    double param;
};

struct TrkExecParams {
    const RowPlan *rows;
    const TRec *trecs;
    const int64_t *tile_off;   // [n_work+1]
    int64_t n_work, ploidy;
    int64_t grid_per_track;    // CTAs per track (upper bound on tiles)
    int64_t total_per_track;   // output values per track
    int64_t n_tracks;
    int32_t layout_btp;        // 0: out is track-major (t, b, p, ~l); 1: (b, t, p, ~l), every query's tracks adjacent
    const int64_t *offset_idxs;  // [n_tracks * n_queries]
    int64_t n_queries;
    const int64_t *query_seed;   // optional [n_queries]
    uint64_t base_seed;
    const uint64_t *base_seed_dev;  // optional: the seed(s) live in device memory (CUDA-graph replays with new batches)
    int64_t sub_batch;              // > 0: queries per logical batch (seed and FlankSample row index are per logical batch)
    void *out;                   // elements of the call's output type (trk_execute picks the instantiation)
    const TrkDesc *tracks;       // device array [n_tracks], or NULL: the descriptors travel in `inl`
    TrkDesc inl[8];              // (kernel parameters are captured by value: CUDA-graph safe)
};

#include "gvl_tracks_exec.cuh"

__global__ void prng_kernel(uint64_t a, uint64_t b, uint64_t c, uint64_t d, int which, uint64_t *out) {
    *out = which ? hash4(a, b, c, d) : xorshift64(a);
}

// =====================================================================================
// intervals: a slot's stored intervals over one window per row, clipped (gvl_dev_track_intervals)
// =====================================================================================
constexpr int ITV_THREADS = 256;  // 8 warps per CTA, one warp per row

struct ItvRows {
    gvl_intervals tracks[MAX_TRACKS];  // (by value: 40 bytes each, the parameters stay under 4 KB)
    int64_t n_tracks;
    const int64_t *slot;
    const int32_t *track, *w0, *w1;
    int64_t n_rows;
};

// The intervals of row q that reach into its window [w0, w1): [lo, lo + n) of its track's arrays, or n = 0 (also for a
// slot or track out of range).  A slot is sorted and free of overlaps, so its starts and its ends are both sorted: lo is
// the first interval with end > w0 and lo + n the first with start >= w1.  `count` = false skips the second search.
// Every lane of the warp calls it for the same row.
__device__ __forceinline__ const gvl_intervals *itv_row(const ItvRows &R, int64_t q, bool count, int64_t &lo, int64_t &n) {
    lo = n = 0;
    const int32_t t = __ldg(R.track + q), w0 = __ldg(R.w0 + q), w1 = __ldg(R.w1 + q);
    const int64_t slot = __ldg(R.slot + q);
    if (t < 0 || t >= R.n_tracks || w1 <= w0) return nullptr;
    const gvl_intervals *I = &R.tracks[t];
    if (slot < 0 || slot >= I->n_slots) return nullptr;
    const int64_t s1 = __ldg(I->itv_offsets + slot + 1);
    lo = warp_upper_le(I->itv_ends, __ldg(I->itv_offsets + slot), s1, w0) + 1;
    if (count) n = warp_upper_le(I->itv_starts, lo, s1, w1 - 1) + 1 - lo;
    else n = s1 - lo;  // (an upper bound: the caller knows the count)
    return I;
}

__global__ void __launch_bounds__(ITV_THREADS) itv_count_kernel(const __grid_constant__ ItvRows R, int64_t *__restrict__ counts) {
    const int64_t n_warps = (int64_t)gridDim.x * (ITV_THREADS / 32);
    for (int64_t q = ((int64_t)blockIdx.x * ITV_THREADS + threadIdx.x) / 32; q < R.n_rows; q += n_warps) {
        int64_t lo, n;
        itv_row(R, q, true, lo, n);
        if (lane_id() == 0) counts[q] = n;
    }
}

// Row q's intervals go to [off[q], off[q + 1]): lanes copy consecutive intervals (coalesced loads and stores), the first
// and the last one clipped to the window, values narrowed to T at the store as in the track execute (to_out).  A row that
// does not fit `cap` or its slot is left unwritten.
template <class T>
__global__ void __launch_bounds__(ITV_THREADS) itv_emit_kernel(const __grid_constant__ ItvRows R, const int64_t *__restrict__ off,
                                                               int64_t cap, int32_t *__restrict__ o_starts,
                                                               int32_t *__restrict__ o_ends, T *__restrict__ o_values) {
    const int lane = lane_id();
    const int64_t n_warps = (int64_t)gridDim.x * (ITV_THREADS / 32);
    for (int64_t q = ((int64_t)blockIdx.x * ITV_THREADS + threadIdx.x) / 32; q < R.n_rows; q += n_warps) {
        const int64_t o = __ldg(off + q), n = __ldg(off + q + 1) - o;
        if (n <= 0 || o < 0 || o + n > cap) continue;
        int64_t lo, avail;
        const gvl_intervals *I = itv_row(R, q, false, lo, avail);
        if (!I || n > avail) continue;
        const int32_t w0 = __ldg(R.w0 + q), w1 = __ldg(R.w1 + q);
        for (int64_t i = lane; i < n; i += 32) {
            int32_t s = __ldg(I->itv_starts + lo + i), e = __ldg(I->itv_ends + lo + i);
            if (i == 0) s = max(s, w0);
            if (i == n - 1) e = min(e, w1);
            o_starts[o + i] = s;
            o_ends[o + i] = e;
            o_values[o + i] = to_out<T>(__ldg(I->itv_values + lo + i));
        }
    }
}

}  // namespace gvl

using namespace gvl;

static bool track_dtype_ok(int32_t dtype) { return dtype == GVL_TRACK_F32 || dtype == GVL_TRACK_BF16 || dtype == GVL_TRACK_F16; }

static int trk_execute(gvl_ctx *ctx, void *out, int32_t dtype, cudaStream_t st) {
    if (!ctx->trk_plan_valid || !ctx->trk_params) return fail(GVL_ERR_STATE, "track execute without a track plan");
    if (!out || ((uintptr_t)out & 3)) return fail(GVL_ERR_ARG, "track output must be an aligned buffer");
    TrkExecParams P;
    memcpy(&P, ctx->trk_params, sizeof(P));
    P.out = out;
    const dim3 grid((unsigned)P.grid_per_track, (unsigned)P.n_tracks);
    const TileDesc *tdesc = (const TileDesc *)ctx->trk.tdesc;
    switch (dtype) {
        case GVL_TRACK_F32: trk_exec3_kernel<float><<<grid, T2_THREADS, 0, st>>>(P, tdesc); break;
        case GVL_TRACK_BF16: trk_exec3_kernel<__nv_bfloat16><<<grid, T2_THREADS, 0, st>>>(P, tdesc); break;
        case GVL_TRACK_F16: trk_exec3_kernel<__half><<<grid, T2_THREADS, 0, st>>>(P, tdesc); break;
        default: return fail(GVL_ERR_ARG, "unknown track dtype %d", (int)dtype);
    }
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

static int launch_trk_exec(gvl_ctx *ctx, int64_t n_work, int64_t ploidy, int64_t n_queries, int64_t n_tracks,
                           const TrkDesc *host_desc, const int64_t *offset_idxs, int64_t total_per_track,
                           const int64_t *query_seed, uint64_t base_seed, void *out, int layout_btp, cudaStream_t st,
                           const uint64_t *base_seed_dev = nullptr, int64_t sub_batch = 0, const int64_t *row_dst = nullptr,
                           const int64_t *row_tstride = nullptr, int32_t dtype = GVL_TRACK_F32) {
    if (n_tracks > MAX_TRACKS) return fail(GVL_ERR_ARG, "at most %d tracks per call", MAX_TRACKS);
    static_assert(sizeof(TrkDesc) * MAX_TRACKS <= GVL_TRK_DESC_BYTES, "descriptor buffer too small");
    TrkDesc *d_desc = nullptr;
    if (n_tracks > 8) {  // (not CUDA-graph safe: the copy reads the caller's host array at replay time)
        d_desc = reinterpret_cast<TrkDesc *>(ctx->trk_desc);
        GVL_CUDA(cudaMemcpyAsync(d_desc, host_desc, sizeof(TrkDesc) * (size_t)n_tracks, cudaMemcpyHostToDevice, st));
    }
    trk_tile_scan_kernel<<<1, 1024, 0, st>>>(n_work, ctx->trk.row_len, ctx->trk.tile_off);
    GVL_LAUNCH_CHECK();
    TrkExecParams P;
    P.rows = ctx->trk.rows;
    P.trecs = (const TRec *)ctx->trk.trecs;
    P.tile_off = ctx->trk.tile_off;
    P.n_work = n_work;
    P.ploidy = ploidy;
    P.grid_per_track = total_per_track / TRK_TILE + n_work;
    P.total_per_track = total_per_track;
    P.n_tracks = n_tracks;
    P.layout_btp = layout_btp;
    P.offset_idxs = offset_idxs;
    P.n_queries = n_queries;
    P.query_seed = query_seed;
    P.base_seed = base_seed;
    P.base_seed_dev = base_seed_dev;
    P.sub_batch = sub_batch;
    P.out = out;
    P.tracks = d_desc;
    if (!d_desc)
        for (int64_t t = 0; t < n_tracks; t++) P.inl[t] = host_desc[t];
    const int64_t grid = P.grid_per_track * n_tracks;
    if (grid > INT32_MAX) return fail(GVL_ERR_ARG, "too many track tiles");
    int rc;
    if ((rc = ensure_tdesc(ctx, ctx->trk, grid))) return rc;
    if (grid * (int64_t)sizeof(TileDesc) > ctx->trk.tdesc_bytes)  // tile prep writes one descriptor per CTA of the grid
        return fail(GVL_ERR_STATE, "track tile descriptors: %lld bytes needed, %lld allocated", (long long)(grid * (int64_t)sizeof(TileDesc)),
                    (long long)ctx->trk.tdesc_bytes);
    TileDesc *tdesc = (TileDesc *)ctx->trk.tdesc;
    trk_tile_prep_kernel<<<(unsigned)((grid + 3) / 4), 128, 0, st>>>(P, row_dst, row_tstride, tdesc);  // one warp per tile
    GVL_LAUNCH_CHECK();
    // the execute launch may follow later, on another stream (gvl_dev_realign_tracks_exec): keep its parameters
    if (!ctx->trk_params) ctx->trk_params = malloc(sizeof(TrkExecParams));
    if (!ctx->trk_params) return fail(GVL_ERR_ARG, "out of host memory");
    memcpy(ctx->trk_params, &P, sizeof(P));
    ctx->trk_plan_valid = true;
    if (!out) return GVL_OK;  // plan only
    return trk_execute(ctx, out, dtype, st);
}

// the scan-based plan kernel in track mode (gvl_hap.cu)
int gvl_trk_plan_launch(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl::MergedLists *merged, const int32_t *regions,
                        const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy,
                        const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc, const int32_t *track_lengths,
                        const int64_t *out_offsets, int64_t max_records, int64_t *words, cudaStream_t st);

// svar2 two-channel merge (gvl_svar2.cu)
int gvl_svar2_merge_launch(gvl_ctx *ctx, gvl_workspace *ws, int64_t *words, const gvl_svar2_channels *ch, int64_t batch,
                           int64_t ploidy, int64_t max_merged, cudaStream_t st);

extern "C" {

static int realign_impl(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2, const int32_t *regions,
                        const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy,
                        const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                        int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                        const float *dense, const int64_t *dense_offsets,
                        const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                        const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                        const int64_t *query_seed, int64_t max_records, float *out, gvl_stream stream,
                        int layout_btp = 0, const uint64_t *base_seed_dev = nullptr, int64_t sub_batch = 0,
                        bool plan_only = false, const int64_t *row_dst = nullptr, const int64_t *row_tstride = nullptr) {
    if (!ctx || !tab || !regions || !shifts || !(geno_offset_idx || svar2) || !(itv || dense) || !(offset_idxs || dense) ||
        !track_lengths || !out_offsets || !strategy_ids || !params)
        return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_work = batch * ploidy;
    ctx->trk_plan_valid = false;
    if (n_work == 0 || n_tracks == 0 || total_per_track == 0) return GVL_OK;
    if (!plan_only && (!out || ((uintptr_t)out & 15))) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks: out must be 16-byte aligned");
    if (plan_only) out = nullptr;
    // every argument is checked before the first launch: a rejected call leaves no half-planned state behind
    if (n_tracks < 0 || n_tracks > MAX_TRACKS) return fail(GVL_ERR_ARG, "at most %d tracks per call", MAX_TRACKS);
    for (int64_t t = 0; t < n_tracks; t++) {
        if (strategy_ids[t] < 0 || strategy_ids[t] > GVL_FILL_INTERPOLATE)
            return fail(GVL_ERR_ARG, "unknown insertion-fill strategy %d", strategy_ids[t]);
        if (strategy_ids[t] == GVL_FILL_INTERPOLATE && !(params[t] >= 1 && params[t] <= 3))
            return fail(GVL_ERR_ARG, "Interpolate order must be 1, 2 or 3");
    }
    int rc;
    if ((rc = ensure_rows(ctx, ctx->trk, n_work))) return rc;
    if ((rc = ensure_trecs(ctx, ctx->trk, max_records + n_work))) return rc;
    int64_t *words = ctx->dev_words + W_COUNT;  // (left at zero by the previous plan, see plan_row_done)
    MergedLists merged{nullptr, nullptr, nullptr, nullptr};
    if (svar2) {  // merged two-channel variant lists (src/svar2/mod.rs:45-66), same merge as the haplotype path
        if ((rc = ensure_merged(ctx, ctx->trk, max_records))) return rc;
        if ((rc = gvl_svar2_merge_launch(ctx, &ctx->trk, words, svar2, batch, ploidy, max_records, st))) return rc;
        merged = MergedLists{ctx->trk.m_pos, ctx->trk.m_key, ctx->trk.m_off, ctx->trk.m_len};
    }
    if ((rc = gvl_trk_plan_launch(ctx, tab, svar2 ? &merged : nullptr, regions, shifts, geno_offset_idx, batch, ploidy, keep,
                                  keep_offsets, to_rc, track_lengths, out_offsets, max_records, words, st)))
        return rc;
    TrkDesc desc[MAX_TRACKS];
    for (int64_t t = 0; t < n_tracks; t++) {
        desc[t].itv_starts = itv ? itv[t].itv_starts : nullptr;
        desc[t].itv_ends = itv ? itv[t].itv_ends : nullptr;
        desc[t].itv_values = itv ? itv[t].itv_values : nullptr;
        desc[t].itv_offsets = itv ? itv[t].itv_offsets : nullptr;
        desc[t].dense = dense;
        desc[t].dense_offsets = dense_offsets;
        desc[t].strategy = strategy_ids[t];
        desc[t].param = params[t];
    }
    return launch_trk_exec(ctx, n_work, ploidy, batch, n_tracks, desc, offset_idxs, total_per_track, query_seed,
                           base_seed, out, layout_btp, st, base_seed_dev, sub_batch, row_dst, row_tstride);
}

int gvl_dev_realign_tracks(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *regions,
                           const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy,
                           const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                           int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                           const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                           const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                           const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed, int64_t max_records,
                           float *out, gvl_stream stream) {
    if (!itv || !offset_idxs) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks: NULL argument");
    return realign_impl(ctx, tab, nullptr, regions, shifts, geno_offset_idx, batch, ploidy, keep, keep_offsets, to_rc, n_tracks,
                        itv, offset_idxs, nullptr, nullptr, track_lengths, out_offsets, total_per_track, strategy_ids,
                        params, base_seed, query_seed, max_records, out, stream, 0, base_seed_dev, sub_batch);
}

int gvl_dev_realign_tracks_btp(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *regions,
                               const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy,
                               const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                               int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                               const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                               const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                               const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed,
                               int64_t max_records, float *out, gvl_stream stream) {
    if (!itv || !offset_idxs) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_btp: NULL argument");
    return realign_impl(ctx, tab, nullptr, regions, shifts, geno_offset_idx, batch, ploidy, keep, keep_offsets, to_rc, n_tracks,
                        itv, offset_idxs, nullptr, nullptr, track_lengths, out_offsets, total_per_track, strategy_ids,
                        params, base_seed, query_seed, max_records, out, stream, 1, base_seed_dev, sub_batch);
}

int gvl_dev_realign_tracks_plan(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                                const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const uint8_t *keep,
                                const int64_t *keep_offsets, const uint8_t *to_rc, int64_t n_tracks, const gvl_intervals *itv,
                                const int64_t *offset_idxs, const int32_t *track_lengths, const int64_t *out_offsets,
                                int64_t total_per_track, const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                                const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed,
                                int64_t max_records, int layout_btp, gvl_stream stream) {
    if (!itv || !offset_idxs) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_plan: NULL argument");
    if (svar2 && (!svar2->vk_off || !svar2->dense_range || !svar2->dense_present_off))
        return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_plan: NULL channel");
    return realign_impl(ctx, tab, svar2, regions, shifts, geno_offset_idx, batch, ploidy, keep, keep_offsets, to_rc, n_tracks,
                        itv, offset_idxs, nullptr, nullptr, track_lengths, out_offsets, total_per_track, strategy_ids,
                        params, base_seed, query_seed, max_records, nullptr, stream, layout_btp ? 1 : 0, base_seed_dev, sub_batch,
                        true);
}

int gvl_dev_realign_tracks_plan_rows(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                                     const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
                                     int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                                     int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                                     const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                                     const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                                     const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed,
                                     int64_t max_records, const int64_t *row_dst, const int64_t *row_tstride, gvl_stream stream) {
    if (!itv || !offset_idxs || !row_dst || !row_tstride) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_plan_rows: NULL argument");
    if (svar2 && (!svar2->vk_off || !svar2->dense_range || !svar2->dense_present_off))
        return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_plan_rows: NULL channel");
    return realign_impl(ctx, tab, svar2, regions, shifts, geno_offset_idx, batch, ploidy, keep, keep_offsets, to_rc, n_tracks,
                        itv, offset_idxs, nullptr, nullptr, track_lengths, out_offsets, total_per_track, strategy_ids,
                        params, base_seed, query_seed, max_records, nullptr, stream, 0, base_seed_dev, sub_batch, true, row_dst,
                        row_tstride);
}

int gvl_dev_realign_tracks_exec_dtype(gvl_ctx *ctx, void *out, int32_t dtype, gvl_stream stream) {
    if (!ctx) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_exec: ctx is NULL");
    if (!track_dtype_ok(dtype)) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_exec: unknown track dtype %d", (int)dtype);
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->trk_plan_valid) return GVL_OK;  // (the plan was empty: nothing to write)
    if ((uintptr_t)out & 15) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_exec: out must be 16-byte aligned");
    return trk_execute(ctx, out, dtype, (cudaStream_t)stream);
}

int gvl_dev_realign_tracks_exec(gvl_ctx *ctx, float *out, gvl_stream stream) {
    return gvl_dev_realign_tracks_exec_dtype(ctx, out, GVL_TRACK_F32, stream);
}

int gvl_dev_shift_and_realign_tracks(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *regions,
                                     const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
                                     int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets,
                                     const uint8_t *to_rc, const float *tracks, const int64_t *track_offsets,
                                     const int32_t *track_lengths, const int64_t *out_offsets, int64_t total,
                                     int32_t strategy_id, double param, uint64_t base_seed,
                                     const int64_t *query_seed, int64_t max_records, float *out, gvl_stream stream) {
    if (!tracks || !track_offsets) return fail(GVL_ERR_ARG, "gvl_dev_shift_and_realign_tracks: NULL argument");
    return realign_impl(ctx, tab, nullptr, regions, shifts, geno_offset_idx, batch, ploidy, keep, keep_offsets, to_rc, 1, nullptr,
                        nullptr, tracks, track_offsets, track_lengths, out_offsets, total, &strategy_id, &param,
                        base_seed, query_seed, max_records, out, stream);
}


int gvl_dev_shift_and_realign_tracks_svar2(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *ch,
                                           const int32_t *regions, const int32_t *shifts, int64_t batch, int64_t ploidy,
                                           const uint8_t *to_rc, const float *tracks, const int64_t *track_offsets,
                                           const int32_t *track_lengths, const int64_t *out_offsets, int64_t total,
                                           int32_t strategy_id, double param, uint64_t base_seed,
                                           const int64_t *query_seed, int64_t max_merged, float *out, gvl_stream stream) {
    if (!ch || !ch->vk_off || !ch->dense_range || !ch->dense_present_off || !tracks || !track_offsets)
        return fail(GVL_ERR_ARG, "gvl_dev_shift_and_realign_tracks_svar2: NULL argument");
    return realign_impl(ctx, tab, ch, regions, shifts, nullptr, batch, ploidy, nullptr, nullptr, to_rc, 1, nullptr, nullptr,
                        tracks, track_offsets, track_lengths, out_offsets, total, &strategy_id, &param, base_seed,
                        query_seed, max_merged, out, stream);
}

int gvl_dev_intervals_to_tracks(gvl_ctx *ctx, const gvl_intervals *itv, const int64_t *offset_idxs,
                                const int32_t *starts, int64_t n_queries, const int64_t *out_offsets,
                                int64_t total, float *out, gvl_stream stream) {
    if (!ctx || !itv || !offset_idxs || !starts || !out_offsets)
        return fail(GVL_ERR_ARG, "gvl_dev_intervals_to_tracks: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (n_queries == 0 || total == 0) return GVL_OK;
    if (!out || ((uintptr_t)out & 15)) return fail(GVL_ERR_ARG, "gvl_dev_intervals_to_tracks: out must be 16-byte aligned");
    int rc;
    if ((rc = ensure_rows(ctx, ctx->trk, n_queries))) return rc;
    if ((rc = ensure_trecs(ctx, ctx->trk, 1))) return rc;
    paint_plan_kernel<<<(unsigned)((n_queries + 255) / 256), 256, 0, st>>>(n_queries, starts, out_offsets, nullptr,
                                                                            ctx->trk.rows, ctx->trk.row_len);
    GVL_LAUNCH_CHECK();
    TrkDesc desc;
    desc.itv_starts = itv->itv_starts;
    desc.itv_ends = itv->itv_ends;
    desc.itv_values = itv->itv_values;
    desc.itv_offsets = itv->itv_offsets;
    desc.dense = nullptr;
    desc.dense_offsets = nullptr;
    desc.strategy = GVL_FILL_REPEAT_5P;
    desc.param = 0.0;
    return launch_trk_exec(ctx, n_queries, 1, n_queries, 1, &desc, offset_idxs, total, nullptr, 0, out, 0, st);
}

static int paint_impl(const char *who, gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                      const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                      const uint8_t *to_rc, void *out, gvl_stream stream, const int64_t *row_dst = nullptr,
                      const int64_t *row_tstride = nullptr, int32_t dtype = GVL_TRACK_F32) {
    if (!ctx || !itv || !offset_idxs || !starts || !out_offsets) return fail(GVL_ERR_ARG, "%s: NULL argument", who);
    if (n_tracks < 0 || n_tracks > MAX_TRACKS) return fail(GVL_ERR_ARG, "%s: 0..%d tracks per call", who, MAX_TRACKS);
    if (!track_dtype_ok(dtype)) return fail(GVL_ERR_ARG, "%s: unknown track dtype %d", who, (int)dtype);
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (n_queries == 0 || n_tracks == 0 || total_per_track == 0) return GVL_OK;
    if (!out || ((uintptr_t)out & 15)) return fail(GVL_ERR_ARG, "%s: out must be 16-byte aligned", who);
    int rc;
    if ((rc = ensure_rows(ctx, ctx->trk, n_queries))) return rc;
    if ((rc = ensure_trecs(ctx, ctx->trk, 1))) return rc;
    paint_plan_kernel<<<(unsigned)((n_queries + 255) / 256), 256, 0, st>>>(n_queries, starts, out_offsets, to_rc,
                                                                            ctx->trk.rows, ctx->trk.row_len);
    GVL_LAUNCH_CHECK();
    TrkDesc desc[MAX_TRACKS];
    for (int64_t t = 0; t < n_tracks; t++) {
        desc[t].itv_starts = itv[t].itv_starts;
        desc[t].itv_ends = itv[t].itv_ends;
        desc[t].itv_values = itv[t].itv_values;
        desc[t].itv_offsets = itv[t].itv_offsets;
        desc[t].dense = nullptr;
        desc[t].dense_offsets = nullptr;
        desc[t].strategy = GVL_FILL_REPEAT_5P;
        desc[t].param = 0.0;
    }
    return launch_trk_exec(ctx, n_queries, 1, n_queries, n_tracks, desc, offset_idxs, total_per_track, nullptr, 0, out, 1, st,
                           nullptr, 0, row_dst, row_tstride, dtype);
}

int gvl_dev_paint_tracks(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                         const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                         const uint8_t *to_rc, float *out, gvl_stream stream) {
    return paint_impl("gvl_dev_paint_tracks", ctx, n_tracks, itv, offset_idxs, starts, n_queries, out_offsets, total_per_track,
                      to_rc, out, stream);
}

int gvl_dev_paint_tracks_rows(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                              const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                              const uint8_t *to_rc, const int64_t *row_dst, const int64_t *row_tstride, float *out,
                              gvl_stream stream) {
    if (!row_dst || !row_tstride) return fail(GVL_ERR_ARG, "gvl_dev_paint_tracks_rows: NULL argument");
    return paint_impl("gvl_dev_paint_tracks_rows", ctx, n_tracks, itv, offset_idxs, starts, n_queries, out_offsets,
                      total_per_track, to_rc, out, stream, row_dst, row_tstride);
}

int gvl_dev_paint_tracks_dtype(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                               const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                               const uint8_t *to_rc, const int64_t *row_dst, const int64_t *row_tstride, void *out, int32_t dtype,
                               gvl_stream stream) {
    if (!row_dst != !row_tstride) return fail(GVL_ERR_ARG, "gvl_dev_paint_tracks_dtype: row_dst and row_tstride go together");
    return paint_impl("gvl_dev_paint_tracks_dtype", ctx, n_tracks, itv, offset_idxs, starts, n_queries, out_offsets,
                      total_per_track, to_rc, out, stream, row_dst, row_tstride, dtype);
}

static int ensure_itv_counts(gvl_ctx *ctx, int64_t n) {
    if (n <= ctx->itv_counts_cap) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    if (ctx->itv_counts) GVL_CUDA(cudaFree(ctx->itv_counts));
    ctx->itv_counts = nullptr;
    ctx->itv_counts_cap = 0;
    const int64_t cap = imax64(2 * n, 4096);
    GVL_CUDA(cudaMalloc(&ctx->itv_counts, sizeof(int64_t) * (size_t)cap));
    ctx->itv_counts_cap = cap;
    return GVL_OK;
}

int gvl_dev_track_intervals(gvl_ctx *ctx, const gvl_intervals *tracks, int64_t n_tracks, const int64_t *row_slot,
                            const int32_t *row_track, const int32_t *row_w0, const int32_t *row_w1, int64_t n_rows,
                            int64_t *out_offsets, int64_t cap, int32_t *out_starts, int32_t *out_ends, void *out_values,
                            int32_t track_dtype, gvl_stream stream) {
    const char *who = "gvl_dev_track_intervals";
    if (!ctx || !out_offsets || n_rows < 0 || cap < 0) return fail(GVL_ERR_ARG, "%s: NULL argument or negative size", who);
    if (n_tracks < 0 || n_tracks > MAX_TRACKS) return fail(GVL_ERR_ARG, "%s: 0..%d tracks per call", who, MAX_TRACKS);
    if (!track_dtype_ok(track_dtype)) return fail(GVL_ERR_ARG, "%s: unknown track dtype %d", who, (int)track_dtype);
    if (n_tracks && !tracks) return fail(GVL_ERR_ARG, "%s: NULL tracks", who);
    for (int64_t t = 0; t < n_tracks; t++)
        if (!tracks[t].itv_starts || !tracks[t].itv_ends || !tracks[t].itv_values || !tracks[t].itv_offsets || tracks[t].n_slots < 0)
            return fail(GVL_ERR_ARG, "%s: track %lld has a NULL array", who, (long long)t);
    if (n_rows && (!row_slot || !row_track || !row_w0 || !row_w1)) return fail(GVL_ERR_ARG, "%s: NULL row array", who);
    if (cap && (!out_starts || !out_ends || !out_values)) return fail(GVL_ERR_ARG, "%s: NULL output with cap > 0", who);
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    ItvRows R;
    memset(&R, 0, sizeof(R));
    for (int64_t t = 0; t < n_tracks; t++) R.tracks[t] = tracks[t];
    R.n_tracks = n_tracks;
    R.slot = row_slot;
    R.track = row_track;
    R.w0 = row_w0;
    R.w1 = row_w1;
    R.n_rows = n_rows;
    const unsigned blocks = (unsigned)imin64(imax64((n_rows + ITV_THREADS / 32 - 1) / (ITV_THREADS / 32), 1), 148 * 32);
    if (cap == 0) {  // sizing call: counts, then their offsets
        int rc;
        if (n_rows) {
            if ((rc = ensure_itv_counts(ctx, n_rows))) return rc;
            itv_count_kernel<<<blocks, ITV_THREADS, 0, st>>>(R, ctx->itv_counts);
            GVL_LAUNCH_CHECK();
        }
        return scan_lengths(ctx, ctx->itv_counts, n_rows, out_offsets, st);
    }
    if (n_rows == 0) return GVL_OK;
    switch (track_dtype) {
        case GVL_TRACK_F32:
            itv_emit_kernel<float><<<blocks, ITV_THREADS, 0, st>>>(R, out_offsets, cap, out_starts, out_ends, (float *)out_values);
            break;
        case GVL_TRACK_BF16:
            itv_emit_kernel<__nv_bfloat16><<<blocks, ITV_THREADS, 0, st>>>(R, out_offsets, cap, out_starts, out_ends,
                                                                           (__nv_bfloat16 *)out_values);
            break;
        default:
            itv_emit_kernel<__half><<<blocks, ITV_THREADS, 0, st>>>(R, out_offsets, cap, out_starts, out_ends, (__half *)out_values);
    }
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

static int run_prng(gvl_ctx *ctx, uint64_t a, uint64_t b, uint64_t c, uint64_t d, int which, uint64_t *out) {
    if (!ctx || !out) return fail(GVL_ERR_ARG, "gvl_debug prng: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    uint64_t *dv = (uint64_t *)(ctx->dev_words + 2 * W_COUNT - 1);
    prng_kernel<<<1, 1, 0, ctx->own_stream>>>(a, b, c, d, which, dv);
    GVL_LAUNCH_CHECK();
    GVL_CUDA(cudaMemcpyAsync(out, dv, sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    return GVL_OK;
}

int gvl_debug_hash4(gvl_ctx *ctx, uint64_t a, uint64_t b, uint64_t c, uint64_t d, uint64_t *out) {
    return run_prng(ctx, a, b, c, d, 1, out);
}

int gvl_debug_xorshift64(gvl_ctx *ctx, uint64_t x, uint64_t *out) { return run_prng(ctx, x, 0, 0, 0, 0, out); }

int gvl_debug_track_tiles(gvl_ctx *ctx, int32_t *out, int64_t n_max, int64_t *n_tiles, int64_t *tdesc_bytes) {
    if (!ctx || !n_tiles || !tdesc_bytes || n_max < 0 || (!out && n_max > 0))
        return fail(GVL_ERR_ARG, "gvl_debug_track_tiles: bad argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    GVL_CUDA(cudaDeviceSynchronize());
    *tdesc_bytes = ctx->trk.tdesc_bytes;
    *n_tiles = 0;
    if (!ctx->trk_params) return GVL_OK;
    const TrkExecParams *P = (const TrkExecParams *)ctx->trk_params;
    const int64_t grid = P->grid_per_track * P->n_tracks;
    *n_tiles = grid;
    if (n_max == 0) return GVL_OK;
    if (grid * (int64_t)sizeof(TileDesc) > ctx->trk.tdesc_bytes)
        return fail(GVL_ERR_STATE, "gvl_debug_track_tiles: %lld descriptors do not fit the buffer", (long long)grid);
    std::vector<TileDesc> h((size_t)grid);
    GVL_CUDA(cudaMemcpy(h.data(), ctx->trk.tdesc, sizeof(TileDesc) * (size_t)grid, cudaMemcpyDeviceToHost));
    int64_t k = 0;
    for (int64_t g = 0; g < grid && k < n_max; g++) {
        const TileDesc &D = h[(size_t)g];
        if (D.row < 0) continue;
        int32_t *o = out + 7 * k++;
        o[0] = (int32_t)(g / P->grid_per_track), o[1] = D.row, o[2] = D.h0, o[3] = D.h1, o[4] = D.flags, o[5] = D.m, o[6] = D.cnt;
    }
    for (; k < n_max; k++)
        for (int f = 0; f < 7; f++) out[7 * k + f] = -1;
    return GVL_OK;
}

}  // extern "C"
