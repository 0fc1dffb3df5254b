// gvl_batch.cu -- device-side preparation of a (region, sample) batch.
//
// The reference prepares every batch on the host with numpy: region rows + read-time jitter
// (python/genvarloader/_dataset/_query.py:161-175), geno_offset_idx = ravel of (region, sample, ploid)
// (_dataset/_haps.py:757-768), the per-row strand mask (_haps.py:838-843, _reconstruct.py:251-256) and the
// interval slot of every (track, query) (_reconstruct.py:233-236).  Here the same O(batch) arithmetic is one
// small kernel over the flat dataset indices, so a batch needs ONE host->device copy (its indices) and the
// whole chain prep -> plan -> execute can be captured in a CUDA graph and replayed with new indices.
#include <cstring>

#include "gvl_internal.cuh"

using namespace gvl;

namespace {

struct PrepParams {
    const int32_t *full_regions;  // (R, 4)
    const int64_t *ds_idx;        // (b) flat index r * n_samples + s over the FULL grid
    const int32_t *jitter;        // (b) or NULL
    int64_t batch, n_samples, ploidy, rows_p, ref_slot, n_tracks, sub_batch;
    uint32_t annot_mask;
    int32_t rc_neg;
    int32_t *regions;
    int32_t *shifts;
    int64_t *goi;
    uint8_t *to_rc;
    uint8_t *to_rc_q;
    int64_t *offset_idxs;
    uint64_t *base_seed;
    int32_t *starts;
};

// Indices of a small batch passed BY VALUE with the launch (kernel parameter space): no staging copy, no event.
constexpr int INLINE_MAX = 256;
struct InlineIdx {
    int64_t idx[INLINE_MAX];
    int32_t jit[INLINE_MAX];
};

template <class IdxOf, class JitOf>
__device__ __forceinline__ void batch_prep_body(const PrepParams &P, IdxOf idx_of, JitOf jit_of) {
    if (P.base_seed) {
        // deterministic fill seed of every logical batch: xor-reduce of its dataset indices as u64
        // (_reconstruct.py:215-218); one warp per logical batch, warps stride over them
        const int lane = threadIdx.x & 31;
        const int64_t n_sub = (P.batch + P.sub_batch - 1) / P.sub_batch;
        const int64_t n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
        for (int64_t sb = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); sb < n_sub; sb += n_warps) {
            const int64_t lo = sb * P.sub_batch, hi = imin64(lo + P.sub_batch, P.batch);
            uint64_t x = 0;
            for (int64_t i = lo + lane; i < hi; i += 32) x ^= (uint64_t)idx_of(i);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x ^= __shfl_xor_sync(0xffffffffu, x, o);
            if (lane == 0) P.base_seed[sb] = x;
        }
    }
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= P.batch) return;
    const int64_t idx = idx_of(q);
    const int64_t r = idx / P.n_samples;
    const int4 reg = *reinterpret_cast<const int4 *>(P.full_regions + 4 * r);  // contig, start, end, strand
    const int32_t len = reg.z - reg.y;
    const int32_t start = reg.y + jit_of(q);  // _query.py:165-171
    P.regions[3 * q + 0] = reg.x;
    P.regions[3 * q + 1] = start;
    P.regions[3 * q + 2] = start + len;
    if (P.starts) P.starts[q] = start;
    const uint8_t rc = (P.rc_neg && reg.w == -1) ? 1 : 0;  // _query.py:173-175
    if (P.to_rc_q) P.to_rc_q[q] = rc;
    for (int64_t h = 0; h < P.rows_p; h++) {
        const int64_t k = q * P.rows_p + h;
        P.goi[k] = P.ref_slot >= 0 ? P.ref_slot : idx * P.ploidy + h;  // _haps.py:757-768
        P.shifts[k] = 0;
        P.to_rc[k] = rc;                                                  // _haps.py:838-843
    }
    for (int64_t t = 0; t < P.n_tracks; t++)  // SAMPLE tracks: dataset index; ANNOT tracks: region index (_reconstruct.py:233-236)
        P.offset_idxs[t * P.batch + q] = ((P.annot_mask >> t) & 1u) ? r : idx;
}

__global__ void __launch_bounds__(128) batch_prep_kernel(PrepParams P) {
    batch_prep_body(P, [&](int64_t i) { return P.ds_idx[i]; }, [&](int64_t i) { return P.jitter ? P.jitter[i] : 0; });
}

__global__ void __launch_bounds__(128) batch_prep_inline_kernel(PrepParams P, const __grid_constant__ InlineIdx I) {
    batch_prep_body(P, [&](int64_t i) { return I.idx[i]; }, [&](int64_t i) { return P.jitter ? I.jit[i] : 0; });
}

__global__ void __launch_bounds__(128) track_lengths_kernel(const int32_t *__restrict__ regions,
                                                            const int32_t *__restrict__ diffs, int64_t batch,
                                                            int64_t ploidy, int32_t *__restrict__ out) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= batch) return;
    int32_t m = 0;
    for (int64_t h = 0; h < ploidy; h++) m = min(m, diffs[q * ploidy + h]);
    out[q] = regions[3 * q + 2] - regions[3 * q + 1] - m;
}

}  // namespace

extern "C" {

// ds_idx / jitter are device arrays, or -- inline_host -- host arrays of <= INLINE_MAX entries passed with the launch
static int launch_batch_prep(gvl_ctx *ctx, const gvl_dataset_view *view, const int64_t *ds_idx, const int32_t *jitter,
                             bool inline_host, int64_t batch, int64_t sub_batch, int64_t ref_slot, int64_t n_tracks,
                             uint32_t annot_mask, const gvl_batch_args *args, gvl_stream stream) {
    if (!ctx || !view || !args) return fail(GVL_ERR_ARG, "gvl_dev_batch_prep: NULL argument");
    if (batch == 0) return GVL_OK;
    if (!ds_idx || !view->full_regions || !args->regions || !args->shifts || !args->goi || !args->to_rc)
        return fail(GVL_ERR_ARG, "gvl_dev_batch_prep: NULL buffer");
    if (n_tracks < 0 || n_tracks > 32 || (n_tracks > 0 && !args->offset_idxs))
        return fail(GVL_ERR_ARG, "gvl_dev_batch_prep: 0..32 tracks, offset_idxs required when n_tracks > 0");
    if (view->n_samples < 1 || view->ploidy < 1) return fail(GVL_ERR_ARG, "gvl_dev_batch_prep: bad dataset view");
    if ((uintptr_t)view->full_regions & 15) return fail(GVL_ERR_ARG, "gvl_dev_batch_prep: full_regions must be 16-byte aligned");
    GVL_CUDA(cudaSetDevice(ctx->device));
    PrepParams P;
    P.full_regions = view->full_regions;
    P.ds_idx = ds_idx;
    P.jitter = jitter;
    P.batch = batch;
    P.sub_batch = (sub_batch > 0 && sub_batch < batch) ? sub_batch : batch;
    P.n_samples = view->n_samples;
    P.ploidy = view->ploidy;
    P.rows_p = ref_slot >= 0 ? 1 : view->ploidy;
    P.ref_slot = ref_slot;
    P.n_tracks = n_tracks;
    P.annot_mask = annot_mask;
    P.rc_neg = view->rc_neg;
    P.regions = args->regions;
    P.shifts = args->shifts;
    P.goi = args->goi;
    P.to_rc = args->to_rc;
    P.to_rc_q = args->to_rc_q;
    P.offset_idxs = args->offset_idxs;
    P.base_seed = args->base_seed;
    P.starts = args->starts;
    const unsigned grid = (unsigned)((batch + 127) / 128);
    if (inline_host) {
        if (batch > INLINE_MAX) return fail(GVL_ERR_ARG, "gvl_dev_batch_prep: inline batch too large");
        const int64_t n_rows = view->n_regions * view->n_samples;
        InlineIdx I;
        for (int64_t i = 0; i < batch; i++) {
            if (ds_idx[i] < 0 || ds_idx[i] >= n_rows) return fail(GVL_ERR_ARG, "dataset index %lld out of range", (long long)ds_idx[i]);
            I.idx[i] = ds_idx[i];
        }
        if (jitter) memcpy(I.jit, jitter, (size_t)batch * 4);
        batch_prep_inline_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(P, I);
    } else {
        batch_prep_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(P);
    }
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

int gvl_dev_batch_prep(gvl_ctx *ctx, const gvl_dataset_view *view, const int64_t *ds_idx, const int32_t *jitter,
                       int64_t batch, int64_t sub_batch, int64_t ref_slot, int64_t n_tracks, uint32_t annot_mask,
                       const gvl_batch_args *args, gvl_stream stream) {
    return launch_batch_prep(ctx, view, ds_idx, jitter, false, batch, sub_batch, ref_slot, n_tracks, annot_mask, args, stream);
}

// track_lengths[q] = (end - start) - min(0, min_h diffs[q, h]): the source window of a realigned track grows by the
// longest net deletion among the query's haplotypes (HapsTracks.__call__, _dataset/_reconstruct.py:191-196)
int gvl_dev_track_lengths(gvl_ctx *ctx, const int32_t *regions, const int32_t *diffs, int64_t batch, int64_t ploidy,
                          int32_t *track_lengths, gvl_stream stream) {
    if (!ctx || batch < 0 || ploidy < 1) return fail(GVL_ERR_ARG, "gvl_dev_track_lengths: bad argument");
    if (batch == 0) return GVL_OK;
    if (!regions || !diffs || !track_lengths) return fail(GVL_ERR_ARG, "gvl_dev_track_lengths: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    track_lengths_kernel<<<(unsigned)((batch + 127) / 128), 128, 0, (cudaStream_t)stream>>>(regions, diffs, batch, ploidy,
                                                                                            track_lengths);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

// Asynchronous host -> device copy on the caller's stream (the pipelined loader stages a ring's indices with one copy;
// `host` should be page-locked, gvl_host_alloc).
int gvl_dev_upload(gvl_ctx *ctx, void *dev, const void *host, int64_t bytes, gvl_stream stream) {
    if (!ctx || (bytes > 0 && (!dev || !host)) || bytes < 0) return fail(GVL_ERR_ARG, "gvl_dev_upload: bad argument");
    if (bytes == 0) return GVL_OK;
    GVL_CUDA(cudaSetDevice(ctx->device));
    GVL_CUDA(cudaMemcpyAsync(dev, host, (size_t)bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return GVL_OK;
}

// ---- one fixed-length batch, end to end (the C side of Dataset.__getitem__ / the loader's device calls) ----

// everything of gvl_dev_fixed_plan after the batch prep: the haplotype plan (what = 1), the track plan (what = 2) or both
static int fixed_plan_prepared(gvl_ctx *ctx, const gvl_fixed_job *J, int64_t n, int64_t sub_batch, gvl_stream stream, int what) {
    int rc;
    const gvl_batch_args &A = J->args;
    const uint8_t *to_rc = J->rc_neg ? A.to_rc : NULL;
    const int64_t cap = J->ref_slot < 0 ? n * J->rows_p * (J->max_slot_len > 1 ? J->max_slot_len : 1) : 0;
    gvl_svar2_channels ch;
    const bool sv = J->svar2 != NULL && J->ref_slot < 0;
    if (sv) {
        ch = *J->svar2;
        ch.row_slot = A.goi;
    }
    // every row's list is bounded by max_slot_len: static record slices (no allocation atomics in the plan kernels)
    ctx->row_stride_hint = J->ref_slot < 0 ? (J->max_slot_len > 1 ? J->max_slot_len : 1) + 1 : 1;
    struct Unhint {
        gvl_ctx *c;
        ~Unhint() { c->row_stride_hint = 0; }
    } unhint{ctx};
    if ((what & 1) && J->mode >= 0) {
        if (sv)
            rc = gvl_dev_hap_plan_svar2(ctx, J->tab, &ch, A.regions, A.shifts, n, J->rows_p, to_rc, J->output_length, cap,
                                        J->out_offsets, J->diffs, stream);
        else
            rc = gvl_dev_hap_plan(ctx, J->tab, A.regions, A.shifts, A.goi, n, J->rows_p, NULL, NULL, to_rc, J->output_length, cap,
                                  J->out_offsets, J->diffs, stream);
        if (rc) return rc;
        if (J->typ_slot_len > 0) ctx->rec_bound_per_row = imin64(ctx->rec_bound_per_row, J->typ_slot_len);  // (tile-length hint)
    }
    if ((what & 2) && J->realign) {
        rc = gvl_dev_track_lengths(ctx, A.regions, J->diffs, n, J->ploidy, J->track_lengths, stream);
        if (rc) return rc;
        rc = gvl_dev_realign_tracks(ctx, J->tab, sv ? &ch : NULL, A.regions, A.shifts, A.goi, n, J->ploidy, NULL, NULL, to_rc,
                                    J->n_tracks, J->itv, A.offset_idxs, J->track_lengths, J->out_offsets,
                                    n * J->ploidy * J->output_length, J->strategy_ids, J->params, 0, A.base_seed, sub_batch, NULL,
                                    cap, GVL_TRACK_LAYOUT_BTP, NULL, NULL, NULL, J->track_dtype, stream);  // (plan only)
        if (rc) return rc;
    }
    return GVL_OK;
}

// batch prep + the plans `what` selects (as in fixed_plan_prepared); ds_idx / jitter as in launch_batch_prep
static int fixed_plan(gvl_ctx *ctx, const gvl_fixed_job *J, const int64_t *ds_idx, const int32_t *jitter, bool inline_host,
                      int64_t n, int64_t sub_batch, int what, gvl_stream stream) {
    if (!ctx || !J || !J->view || !J->tab) return fail(GVL_ERR_ARG, "gvl_dev_fixed_plan: NULL argument");
    if (J->realign && (J->mode < 0 || J->ref_slot >= 0 || !J->diffs || !J->track_lengths))
        return fail(GVL_ERR_ARG, "gvl_dev_fixed_plan: realigned tracks need haplotypes, diffs and track_lengths scratch");
    if (J->track_dtype != GVL_TRACK_F32 && J->track_dtype != GVL_TRACK_BF16 && J->track_dtype != GVL_TRACK_F16)
        return fail(GVL_ERR_ARG, "gvl_dev_fixed_plan: unknown track dtype %d", (int)J->track_dtype);
    if (J->track_bin < 0 || J->track_bin > GVL_TRACK_BIN_MAX || (J->track_bin & (J->track_bin - 1)) ||
        (J->track_reduce != GVL_TRACK_REDUCE_MEAN && J->track_reduce != GVL_TRACK_REDUCE_SUM && J->track_reduce != GVL_TRACK_REDUCE_MAX))
        return fail(GVL_ERR_ARG, "gvl_dev_fixed_plan: bad track bin %d / reduction %d", (int)J->track_bin, (int)J->track_reduce);
    int rc = launch_batch_prep(ctx, J->view, ds_idx, jitter, inline_host, n, sub_batch, J->ref_slot, J->n_tracks, J->annot_mask,
                               &J->args, stream);
    if (rc) return rc;
    return fixed_plan_prepared(ctx, J, n, sub_batch, stream, what);
}

int gvl_dev_fixed_plan(gvl_ctx *ctx, const gvl_fixed_job *J, const int64_t *ds_idx, const int32_t *jitter, int64_t n,
                       int64_t sub_batch, gvl_stream stream) {
    return fixed_plan(ctx, J, ds_idx, jitter, false, n, sub_batch, 3, stream);
}

// One stage of a fixed-length batch, for callers that spread a device call over two streams (the track plan -- a chain of
// small latency-bound kernels -- next to the bandwidth-bound haplotype execute): GVL_STAGE_HAP_PLAN = batch prep +
// haplotype plan, GVL_STAGE_TRK_PLAN (needs the diffs of HAP_PLAN), GVL_STAGE_HAP_EXEC, GVL_STAGE_TRK_EXEC (needs TRK_PLAN).
int gvl_dev_fixed_stage(gvl_ctx *ctx, const gvl_fixed_job *J, int stage, const int64_t *ds_idx, const int32_t *jitter, int64_t n,
                        int64_t sub_batch, uint8_t *seq, int32_t *annot_v, int32_t *annot_pos, void *trk, gvl_stream stream) {
    if (!ctx || !J || !J->tab) return fail(GVL_ERR_ARG, "gvl_dev_fixed_stage: NULL argument");
    switch (stage) {
        case GVL_STAGE_HAP_PLAN:
            return fixed_plan(ctx, J, ds_idx, jitter, false, n, sub_batch, 1, stream);
        case GVL_STAGE_TRK_PLAN:
            return fixed_plan_prepared(ctx, J, n, sub_batch, stream, 2);
        case GVL_STAGE_HAP_EXEC:
            if (J->mode < 0) return GVL_OK;
            if (!seq) return fail(GVL_ERR_ARG, "gvl_dev_fixed_stage: sequence output missing");
            return gvl_dev_hap_exec(ctx, J->tab, J->mode, J->pad_char, seq, annot_v, annot_pos, stream);
        case GVL_STAGE_TRK_EXEC:
            if (J->n_tracks <= 0) return GVL_OK;
            if (!trk) return fail(GVL_ERR_ARG, "gvl_dev_fixed_stage: track output missing");
            if (J->realign) return gvl_dev_realign_tracks_exec_binned(ctx, trk, J->track_dtype, J->track_bin, J->track_reduce, stream);
            return gvl_dev_paint_tracks_binned(ctx, J->n_tracks, J->itv, J->args.offset_idxs, J->args.starts, n, J->paint_offsets,
                                               n * J->output_length, J->rc_neg ? J->args.to_rc_q : NULL, GVL_TRACK_LAYOUT_BTP, NULL,
                                               NULL, trk, J->track_dtype, J->track_bin, J->track_reduce, stream);
        default: return fail(GVL_ERR_ARG, "gvl_dev_fixed_stage: unknown stage %d", stage);
    }
}

int gvl_dev_fixed_exec(gvl_ctx *ctx, const gvl_fixed_job *J, int64_t n, uint8_t *seq, int32_t *annot_v, int32_t *annot_pos,
                       void *trk, gvl_stream stream) {
    int rc = gvl_dev_fixed_stage(ctx, J, GVL_STAGE_HAP_EXEC, NULL, NULL, n, 0, seq, annot_v, annot_pos, trk, stream);
    if (rc) return rc;
    return gvl_dev_fixed_stage(ctx, J, GVL_STAGE_TRK_EXEC, NULL, NULL, n, 0, seq, annot_v, annot_pos, trk, stream);
}

int gvl_dev_fixed_run(gvl_ctx *ctx, const gvl_fixed_job *J, const int64_t *ds_idx, const int32_t *jitter, int64_t n,
                      int64_t *idx_dev, int32_t *jitter_dev, uint8_t *seq, int32_t *annot_v, int32_t *annot_pos, void *trk,
                      gvl_stream stream) {
    if (!ctx || !J || n < 0 || (n > 0 && (!ds_idx || !idx_dev)) || (jitter && !jitter_dev))
        return fail(GVL_ERR_ARG, "gvl_dev_fixed_run: bad argument");
    if (n == 0) return GVL_OK;
    GVL_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (n <= INLINE_MAX) {  // small batch: the indices travel with the prep launch
        int rc = fixed_plan(ctx, J, ds_idx, jitter, true, n, 0, 3, stream);
        if (rc) return rc;
        return gvl_dev_fixed_exec(ctx, J, n, seq, annot_v, annot_pos, trk, stream);
    }
    // stage the (pageable) indices through a rotating pinned slot: the host never waits for the previous call's copy
    gvl_ctx::StageSlot &S = ctx->stage[ctx->stage_k];
    ctx->stage_k = (ctx->stage_k + 1) % 8;
    if (S.used) GVL_CUDA(cudaEventSynchronize(S.ev));
    const int64_t need = n * 12;
    if (S.bytes < need) {
        if (S.host) cudaFreeHost(S.host);
        S.host = nullptr;
        S.bytes = 0;
        int64_t cap = 4096;
        while (cap < need) cap *= 2;
        GVL_CUDA(cudaMallocHost(&S.host, (size_t)cap));
        S.bytes = cap;
    }
    if (!S.ev) GVL_CUDA(cudaEventCreateWithFlags(&S.ev, cudaEventDisableTiming));
    {
        const int64_t n_rows = J->view ? J->view->n_regions * J->view->n_samples : 0;
        int64_t *dst = (int64_t *)S.host;
        for (int64_t i = 0; i < n; i++) {
            if (ds_idx[i] < 0 || ds_idx[i] >= n_rows) return fail(GVL_ERR_ARG, "dataset index %lld out of range", (long long)ds_idx[i]);
            dst[i] = ds_idx[i];
        }
    }
    GVL_CUDA(cudaMemcpyAsync(idx_dev, S.host, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    if (jitter) {
        memcpy((char *)S.host + n * 8, jitter, (size_t)n * 4);
        GVL_CUDA(cudaMemcpyAsync(jitter_dev, (char *)S.host + n * 8, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    }
    GVL_CUDA(cudaEventRecord(S.ev, st));
    S.used = true;
    int rc = gvl_dev_fixed_plan(ctx, J, idx_dev, jitter ? jitter_dev : NULL, n, 0, stream);
    if (rc) return rc;
    return gvl_dev_fixed_exec(ctx, J, n, seq, annot_v, annot_pos, trk, stream);
}

}  // extern "C"
