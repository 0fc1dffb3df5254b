// gvl_tracks.cu -- indel-aware track realignment on sm_100a (include/gvl_b200.h:
// gvl_dev_realign_tracks, gvl_dev_shift_and_realign_tracks, gvl_dev_paint_tracks).
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
// The output is float32, bfloat16 or float16 (GVL_TRACK_*: one execute instantiation per type, values narrowed at the
// store), each row placed by the tile preparation as the call's GVL_TRACK_LAYOUT_* says.
//
// gvl_dev_track_intervals returns the stored intervals themselves instead of painting them: a count kernel (one warp per
// row, two 32-ary searches), the offset scan of the variants tail, and an emit kernel that copies each row's run.
// gvl_dev_realigned_track_intervals cuts the rows of a track plan into intervals instead of executing them: a count kernel
// over the rows' items (one warp each), offset scans, and an emit kernel with one thread per output interval.
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
// identity plan for painting (gvl_dev_paint_tracks): one row per query, no records, source window = row
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

// =====================================================================================
// realigned intervals: the rows of a track plan cut into intervals (gvl_dev_realigned_track_intervals)
// =====================================================================================
// Every output position p of a planned row has a source, resolved as t2_generic_value resolves it, and the source has an
// IDENTITY: the index of the stored interval that holds it (none outside every interval and outside the window); one per
// record for Repeat5pNormalized / Constant fills; one per position for Interpolate fills; FlankSample positions take the
// identity of the position they sample.  The row's intervals are the maximal runs of one identity other than none.
//
// Row k of track t ("pair" t * n_work + k) is split into ITEMS in output order: the copy span before the first record, then
// for every record its own span and the copy span after it -- 1 + 2 n_rec items, contiguous and covering [0, L).  A copy
// span reads consecutive source positions, so its runs are the stored intervals that overlap its source range (two 32-ary
// searches); a record span is one run or none, except FlankSample and Interpolate spans (a step per position).  A run that
// crosses items belongs to the item where it starts: an item whose first identity equals that of the position before it
// is MERGED and does not count that run.
//   ritv_count_kernel  one warp per item: its geometry, pieces and merge flag into an RItem, its count into `counts`;
//   (offset scans)     items -> per-pair totals -> the caller's out_offsets;
//   ritv_emit_kernel   one thread per output interval (seg_emit_kernel of gvl_variants.cu): finds its item and pair with
//                      two binary searches over the offsets, writes (start, end, value); the end of a run that reaches the
//                      end of its item is read from the RItems of the items it crosses.
constexpr int RI_COPY = 0, RI_SPAN = 1, RI_ONE = 2, RI_INTERP = 3, RI_FLANK = 4;  // RItem.flags & 7
constexpr int RI_MERGED = 8;  // the run at p0 continues a run of an earlier item (not counted here)
constexpr int RI_OPEN = 16;   // the run at p0 has an interval identity and covers [p0, p1)

struct __align__(16) RItem {
    int64_t lo;        // COPY: first stored interval that reaches the span; SPAN: the source's interval (-1: none);
                       // fills: the record (index in the row)
    int32_t p0, p1;    // output positions of the item
    int32_t s0;        // COPY: relative source position feeding p0; SPAN: the variant's source position
    int32_t flags;     // kind | RI_MERGED | RI_OPEN
    int32_t head_end;  // end of the run that starts at p0 (meaningful with an interval identity at p0)
    int32_t pad;
};
static_assert(sizeof(RItem) == 32, "RItem is 32 bytes");

struct RItvParams {
    TrkExecParams P;           // the plan's saved execute parameters: rows, records, track descriptors, seeds
    const int64_t *item_base;  // [n_pairs + 1] first item of each pair
    const int64_t *item_off;   // [item_cap + 1] first output interval of each item (emit)
    const int64_t *row_out;    // optional [n_pairs]: output row of each pair
    int64_t n_pairs, item_cap;
    RItem *items;              // [item_cap]
};

// what a pair needs to resolve its positions (the execute kernel's TileCtx, for one row of one track)
struct RRow {
    const TRec *recs;
    int32_t n_rec, L, ref0, q_start, track_n, strategy;
    double param;
    SrcGlobal src;
    uint64_t base_seed, qseed, hap;
};

__device__ __forceinline__ RRow ritv_row(const RItvParams &R, int64_t pair) {
    const TrkExecParams &P = R.P;
    const int64_t t = pair / P.n_work, k = pair - t * P.n_work, query = k / P.ploidy;
    const RowPlan rp = P.rows[k];
    const TrkDesc &T = P.tracks ? P.tracks[t] : P.inl[t];
    RRow w;
    w.recs = P.trecs + rp.rec_off;
    w.n_rec = rp.n_rec, w.L = rp.length, w.ref0 = rp.ref0, w.q_start = rp.q_start, w.track_n = rp.contig_len;
    w.strategy = T.strategy, w.param = T.param;
    const int64_t slot = P.offset_idxs[t * P.n_queries + query];
    w.src.its = T.itv_starts, w.src.ite = T.itv_ends, w.src.itv = T.itv_values, w.src.dense = nullptr;
    w.src.itv_lo = T.itv_offsets[slot], w.src.itv_hi = T.itv_offsets[slot + 1], w.src.q_start = rp.q_start;
    w.src.track_n = rp.contig_len;
    // seeds of the fills exactly as trk_exec3_kernel takes them
    const uint32_t sub = P.sub_batch > 0 ? (uint32_t)P.sub_batch : 0u;
    const uint32_t q_blk = sub ? (uint32_t)query / sub : 0u;
    w.hap = (uint64_t)(k - query * P.ploidy);
    w.qseed = P.query_seed ? (uint64_t)P.query_seed[query] : (uint64_t)(sub ? (uint32_t)query - q_blk * sub : (uint32_t)query);
    w.base_seed = P.base_seed_dev ? P.base_seed_dev[q_blk] : P.base_seed;
    return w;
}

__device__ __forceinline__ int64_t ritv_out_row(const RItvParams &R, int64_t pair) {
    if (R.row_out) return __ldg(R.row_out + pair);
    const int64_t t = pair / R.P.n_work, k = pair - t * R.P.n_work, q = k / R.P.ploidy;
    return (q * R.P.n_tracks + t) * R.P.ploidy + (k - q * R.P.ploidy);  // (query, track, ploid)
}

// warp_upper_le over any non-decreasing sequence at(lo .. hi - 1): last index with at(i) <= key, or lo - 1
template <class F>
__device__ __forceinline__ int64_t warp_last_le(F at, int64_t lo, int64_t hi, int64_t key) {
    const int lane = lane_id();
    while (hi - lo > 32) {
        const int64_t step = (hi - lo + 31) / 32;
        const int64_t idx = lo + (int64_t)(lane + 1) * step - 1;
        const int cnt = __popc(__ballot_sync(0xffffffffu, idx < hi && at(idx) <= key));
        const int64_t nlo = lo + (int64_t)cnt * step;
        hi = imin64(hi, lo + (int64_t)(cnt + 1) * step - 1);
        lo = nlo;
        if (lo > hi) hi = lo;
    }
    const int64_t idx = lo + lane;
    return lo + __popc(__ballot_sync(0xffffffffu, idx < hi && at(idx) <= key)) - 1;
}

// last i in [0, n) with off[i] <= e (off non-decreasing, off[0] <= e): one thread
__device__ __forceinline__ int64_t last_le_i64(const int64_t *__restrict__ off, int64_t n, int64_t e) {
    int64_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (__ldg(off + mid) <= e) lo = mid; else hi = mid;
    }
    return lo;
}

// identity of relative source position s: the stored interval that holds it, -1 = none (also outside [0, track_n))
__device__ __forceinline__ int64_t ritv_src_id_warp(const RRow &w, int64_t s) {
    if (s < 0 || s >= w.track_n) return -1;
    const int64_t g = (int64_t)w.q_start + s;
    const int64_t i = warp_upper_le(w.src.its, w.src.itv_lo, w.src.itv_hi, (int32_t)g);
    return (i >= w.src.itv_lo && (int64_t)__ldg(w.src.ite + i) > g) ? i : -1;
}
__device__ __forceinline__ int64_t ritv_src_id(const RRow &w, int64_t s) {  // (one thread)
    if (s < 0 || s >= w.track_n) return -1;
    const int64_t g = (int64_t)w.q_start + s;
    int64_t a = w.src.itv_lo, b = w.src.itv_hi;
    while (a < b) {
        const int64_t mid = (a + b) >> 1;
        if ((int64_t)__ldg(w.src.its + mid) <= g) a = mid + 1; else b = mid;
    }
    return (a > w.src.itv_lo && (int64_t)__ldg(w.src.ite + a - 1) > g) ? a - 1 : -1;
}

// source position that FlankSample output position p of record r samples (insertion_fill_value)
__device__ __forceinline__ int64_t ritv_flank_src(const RRow &w, const TRec &r, int32_t p) {
    const int64_t width = (int64_t)w.param;
    const int64_t pool_lo = imax64((int64_t)r.vrel - width, 0), pool_hi = imin64((int64_t)r.vrel + width, (int64_t)w.track_n - 1);
    const uint64_t pool_size = (uint64_t)(pool_hi - pool_lo + 1);
    return pool_lo + (int64_t)(hash4(w.base_seed, w.qseed, w.hap, (uint64_t)p) % pool_size);
}

__device__ __forceinline__ bool ritv_is_fill(const RRow &w, const TRec &r) { return r.vdiff > 0 && w.strategy != GVL_FILL_REPEAT_5P; }

// identity of output position p (warp): >= 0 a stored interval, -1 none, -2 an identity of its own (fills)
__device__ int64_t ritv_ident_warp(const RRow &w, int32_t p) {
    const TRec *__restrict__ recs = w.recs;
    const int64_t i = warp_last_le([&](int64_t j) { return (int64_t)recs[j].a; }, 0, w.n_rec, p);
    int64_t s;
    if (i < 0) {
        s = (int64_t)w.ref0 + p;
    } else {
        const TRec r = recs[i];
        if (p < r.e) {
            if (ritv_is_fill(w, r)) {
                if (w.strategy != GVL_FILL_FLANK_SAMPLE) return -2;
                s = ritv_flank_src(w, r, p);
            } else {
                s = r.vrel;
            }
        } else {
            s = (int64_t)r.resume + (p - r.e);
        }
    }
    return ritv_src_id_warp(w, s);
}

// geometry of item u of a row: positions [p0, p1), kind, source of p0, record
__device__ __forceinline__ RItem ritv_geom(const RRow &w, int64_t u) {
    auto A = [&](int64_t i) { return i < w.n_rec ? min(max(w.recs[i].a, 0), w.L) : w.L; };  // where record i takes over
    RItem o;
    o.pad = 0;
    if (u == 0) {
        o.p0 = 0, o.p1 = A(0), o.s0 = w.ref0, o.flags = RI_COPY, o.lo = -1;
    } else {
        const int64_t i = (u - 1) >> 1;
        const TRec r = w.recs[i];
        const int32_t a0 = A(i), a1 = max(A(i + 1), a0);
        const int32_t e = min(max(r.e, a0), a1);
        o.lo = i;
        if (u & 1) {  // the variant's own values
            o.p0 = a0, o.p1 = e, o.s0 = r.vrel;
            o.flags = !ritv_is_fill(w, r) ? RI_SPAN
                      : w.strategy == GVL_FILL_FLANK_SAMPLE ? RI_FLANK
                      : w.strategy == GVL_FILL_INTERPOLATE ? RI_INTERP : RI_ONE;
        } else {      // the copy after it
            o.p0 = e, o.p1 = a1, o.s0 = r.resume + (e - r.e), o.flags = RI_COPY;
        }
    }
    o.head_end = o.p0;
    return o;
}

__global__ void __launch_bounds__(ITV_THREADS) ritv_count_kernel(const __grid_constant__ RItvParams R, int64_t *__restrict__ counts) {
    const int lane = lane_id();
    const int64_t n_items = __ldg(R.item_base + R.n_pairs);
    const int64_t n_warps = (int64_t)gridDim.x * (ITV_THREADS / 32);
    for (int64_t it = ((int64_t)blockIdx.x * ITV_THREADS + threadIdx.x) / 32; it < R.item_cap; it += n_warps) {
        if (it >= n_items) {  // (slots beyond the plan's items)
            if (lane == 0) counts[it] = 0;
            continue;
        }
        const int64_t pair = warp_last_le([&](int64_t j) { return __ldg(R.item_base + j); }, 0, R.n_pairs, it);
        const RRow w = ritv_row(R, pair);
        RItem o = ritv_geom(w, it - __ldg(R.item_base + pair));
        const int kind = o.flags;
        int64_t n = 0, id0 = -2;  // pieces of the item, identity at p0
        if (o.p1 > o.p0) {
            if (kind == RI_COPY) {  // the stored intervals that overlap the source range, clipped to the window
                const int64_t c0 = imax64(o.s0, 0), c1 = imin64((int64_t)o.s0 + (o.p1 - o.p0), w.track_n);
                id0 = -1;
                if (c1 > c0) {
                    const int64_t g0 = (int64_t)w.q_start + c0, g1 = (int64_t)w.q_start + c1;
                    const int64_t a = warp_upper_le(w.src.ite, w.src.itv_lo, w.src.itv_hi, (int32_t)g0) + 1;
                    const int64_t b = warp_upper_le(w.src.its, a, w.src.itv_hi, (int32_t)(g1 - 1)) + 1;
                    n = b - a;
                    o.lo = a;
                    if (n > 0 && o.s0 >= 0 && (int64_t)__ldg(w.src.its + a) <= g0) {
                        id0 = a;
                        o.head_end = (int32_t)(o.p0 + (imin64(__ldg(w.src.ite + a), g1) - g0));
                    }
                }
            } else if (kind == RI_SPAN) {  // one source position for the whole span
                id0 = ritv_src_id_warp(w, o.s0);
                n = id0 >= 0;
                o.lo = id0;
                o.head_end = o.p1;
            } else if (kind == RI_ONE) {
                n = 1;
            } else if (kind == RI_INTERP) {
                n = o.p1 - o.p0;
            } else {  // FlankSample: the identity of every position, 32 at a time
                const TRec r = w.recs[o.lo];
                int64_t prev = -3;  // identity before the chunk (-3: the item starts there)
                bool head = false;
                for (int32_t p = o.p0; p < o.p1; p += 32) {
                    const int32_t q = p + lane;
                    const int64_t id = q < o.p1 ? ritv_src_id(w, ritv_flank_src(w, r, q)) : -1;
                    int64_t before = __shfl_up_sync(0xffffffffu, id, 1);
                    if (lane == 0) before = prev;
                    n += __popc(__ballot_sync(0xffffffffu, q < o.p1 && id >= 0 && id != before));
                    if (p == o.p0) id0 = __shfl_sync(0xffffffffu, id, 0);
                    const unsigned brk = __ballot_sync(0xffffffffu, q < o.p1 && id != id0);
                    if (!head && brk) {
                        o.head_end = p + __ffs(brk) - 1;
                        head = true;
                    }
                    prev = __shfl_sync(0xffffffffu, id, 31);
                }
                if (!head) o.head_end = o.p1;
            }
        }
        if (id0 >= 0 && o.head_end == o.p1) o.flags |= RI_OPEN;
        if (id0 >= 0 && o.p0 > 0 && ritv_ident_warp(w, o.p0 - 1) == id0) {  // the run began in an earlier item
            o.flags |= RI_MERGED;
            n--;
        }
        if (lane == 0) {
            R.items[it] = o;
            counts[it] = n;
        }
    }
}

// per output row: its intervals = those of its pair's items
__global__ void ritv_rows_kernel(const __grid_constant__ RItvParams R, int64_t *__restrict__ row_cnt) {
    const int64_t pair = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= R.n_pairs) return;
    const int64_t row = ritv_out_row(R, pair);
    if (row < 0 || row >= R.n_pairs) return;
    row_cnt[row] = __ldg(R.item_off + __ldg(R.item_base + pair + 1)) - __ldg(R.item_off + __ldg(R.item_base + pair));
}

// end of a run that reaches the end p1 of item `slot`: it goes on through the merged items that follow
__device__ __forceinline__ int32_t ritv_run_end(const RItvParams &R, int64_t slot, int32_t end, int64_t n_items) {
    for (int64_t s = slot + 1; s < n_items; s++) {
        const RItem x = R.items[s];
        if (x.p1 == x.p0) continue;
        if (!(x.flags & RI_MERGED)) break;
        end = x.head_end;
        if (!(x.flags & RI_OPEN)) break;
    }
    return end;
}

template <class T>
__device__ __forceinline__ void ritv_store(int32_t *o_starts, int32_t *o_ends, T *o_values, int64_t o, int32_t w0, int32_t s,
                                           int32_t e, float v) {
    o_starts[o] = w0 + s;
    o_ends[o] = w0 + e;
    o_values[o] = to_out<T>(v);
}

template <class T>
__global__ void __launch_bounds__(256) ritv_emit_kernel(const __grid_constant__ RItvParams R, const int64_t *__restrict__ out_off,
                                                        int64_t cap, int32_t *__restrict__ o_starts, int32_t *__restrict__ o_ends,
                                                        T *__restrict__ o_values) {
    const int64_t total = imin64(__ldg(R.item_off + R.item_cap), cap);
    const int64_t n_items = __ldg(R.item_base + R.n_pairs);
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
        const int64_t slot = last_le_i64(R.item_off, R.item_cap, g);
        const int64_t pair = last_le_i64(R.item_base, R.n_pairs, slot);
        const int64_t row = ritv_out_row(R, pair);
        if (row < 0 || row >= R.n_pairs) continue;
        const int64_t o = __ldg(out_off + row) + (g - __ldg(R.item_off + __ldg(R.item_base + pair)));
        const int64_t j = g - __ldg(R.item_off + slot);  // the item's j-th interval
        const RRow w = ritv_row(R, pair);
        const RItem it = R.items[slot];
        const int kind = it.flags & 7;
        const int64_t raw = j + ((it.flags & RI_MERGED) ? 1 : 0);  // its j-th piece that is not a continued run
        int32_t s, e;
        float v;
        if (kind == RI_COPY) {
            const int64_t i = it.lo + raw;
            const int64_t g0 = (int64_t)w.q_start + imax64(it.s0, 0);
            const int64_t g1 = (int64_t)w.q_start + imin64((int64_t)it.s0 + (it.p1 - it.p0), w.track_n);
            const int64_t base = (int64_t)w.q_start + it.s0 - it.p0;  // position p reads source q_start + p + (s0 - p0)
            s = (int32_t)(imax64(__ldg(w.src.its + i), g0) - base);
            e = (int32_t)(imin64(__ldg(w.src.ite + i), g1) - base);
            v = __ldg(w.src.itv + i);
        } else if (kind == RI_SPAN) {
            s = it.p0, e = it.p1, v = __ldg(w.src.itv + it.lo);
        } else if (kind == RI_ONE || kind == RI_INTERP) {
            const TRec r = w.recs[it.lo];
            s = kind == RI_ONE ? it.p0 : it.p0 + (int32_t)raw;
            e = kind == RI_ONE ? it.p1 : s + 1;
            v = insertion_fill_value(w.src, w.strategy, w.param, r.vlen, r.vrel, s - r.a, s, w.base_seed, w.qseed, w.hap);
        } else {  // FlankSample: the thread of the item's first interval writes all of them (fills are short)
            if (j != 0) continue;
            const int64_t n = __ldg(R.item_off + slot + 1) - __ldg(R.item_off + slot);
            if (o + n > cap) continue;
            const TRec r = w.recs[it.lo];
            int64_t prev = -3, k = 0;
            int32_t run0 = it.p0;
            for (int32_t p = it.p0; p <= it.p1; p++) {
                const int64_t id = p < it.p1 ? ritv_src_id(w, ritv_flank_src(w, r, p)) : -3;
                if (id == prev) continue;
                if (prev >= 0 && !(run0 == it.p0 && (it.flags & RI_MERGED))) {
                    const int32_t end = p == it.p1 ? ritv_run_end(R, slot, p, n_items) : p;
                    ritv_store(o_starts, o_ends, o_values, o + k++, w.q_start, run0, end, __ldg(w.src.itv + prev));
                }
                run0 = p;
                prev = id;
            }
            continue;
        }
        if (o < 0 || o >= cap) continue;
        if (e == it.p1) e = ritv_run_end(R, slot, e, n_items);
        ritv_store(o_starts, o_ends, o_values, o, w.q_start, s, e, v);
    }
}

}  // namespace gvl

using namespace gvl;

static bool track_dtype_ok(int32_t dtype) { return dtype == GVL_TRACK_F32 || dtype == GVL_TRACK_BF16 || dtype == GVL_TRACK_F16; }

// layout, destination table and element type of gvl_dev_realign_tracks / gvl_dev_paint_tracks
static int check_track_output(const char *who, int32_t layout, const int64_t *row_dst, const int64_t *row_tstride,
                              int32_t dtype) {
    if (layout != GVL_TRACK_LAYOUT_TBP && layout != GVL_TRACK_LAYOUT_BTP && layout != GVL_TRACK_LAYOUT_ROWS)
        return fail(GVL_ERR_ARG, "%s: unknown track layout %d", who, (int)layout);
    const bool rows = layout == GVL_TRACK_LAYOUT_ROWS;
    if (rows != (row_dst != nullptr) || rows != (row_tstride != nullptr))
        return fail(GVL_ERR_ARG, "%s: row_dst and row_tstride go with GVL_TRACK_LAYOUT_ROWS, and only with it", who);
    if (!track_dtype_ok(dtype)) return fail(GVL_ERR_ARG, "%s: unknown track dtype %d", who, (int)dtype);
    return GVL_OK;
}

// bin 0 or 1: unbinned; else a power of two in [2, GVL_TRACK_BIN_MAX]
static int check_track_bin(const char *who, int32_t bin, int32_t reduce) {
    if (bin < 0 || bin > GVL_TRACK_BIN_MAX || (bin & (bin - 1)))
        return fail(GVL_ERR_ARG, "%s: track bin %d is not 0, 1 or a power of two up to %d", who, (int)bin, GVL_TRACK_BIN_MAX);
    if (reduce != GVL_TRACK_REDUCE_MEAN && reduce != GVL_TRACK_REDUCE_SUM && reduce != GVL_TRACK_REDUCE_MAX)
        return fail(GVL_ERR_ARG, "%s: unknown track reduction %d", who, (int)reduce);
    return GVL_OK;
}

static int trk_execute(gvl_ctx *ctx, void *out, int32_t dtype, int32_t bin, int32_t reduce, cudaStream_t st) {
    if (!ctx->trk_plan_valid || !ctx->trk_params) return fail(GVL_ERR_STATE, "track execute without a track plan");
    if (!out || ((uintptr_t)out & 15)) return fail(GVL_ERR_ARG, "track output must be a 16-byte aligned buffer");
    TrkExecParams P;
    memcpy(&P, ctx->trk_params, sizeof(P));
    P.out = out;
    const dim3 grid((unsigned)P.grid_per_track, (unsigned)P.n_tracks);
    const TileDesc *tdesc = (const TileDesc *)ctx->trk.tdesc;
    const TrkBin bn{bin > 1 ? __builtin_ctz((unsigned)bin) : 0, reduce};
    if (bin > 1) {
        switch (dtype) {
            case GVL_TRACK_F32: trk_exec3_kernel<float, true><<<grid, T2_THREADS, 0, st>>>(P, tdesc, bn); break;
            case GVL_TRACK_BF16: trk_exec3_kernel<__nv_bfloat16, true><<<grid, T2_THREADS, 0, st>>>(P, tdesc, bn); break;
            case GVL_TRACK_F16: trk_exec3_kernel<__half, true><<<grid, T2_THREADS, 0, st>>>(P, tdesc, bn); break;
            default: return fail(GVL_ERR_ARG, "unknown track dtype %d", (int)dtype);
        }
    } else {
        switch (dtype) {
            case GVL_TRACK_F32: trk_exec3_kernel<float, false><<<grid, T2_THREADS, 0, st>>>(P, tdesc, bn); break;
            case GVL_TRACK_BF16: trk_exec3_kernel<__nv_bfloat16, false><<<grid, T2_THREADS, 0, st>>>(P, tdesc, bn); break;
            case GVL_TRACK_F16: trk_exec3_kernel<__half, false><<<grid, T2_THREADS, 0, st>>>(P, tdesc, bn); break;
            default: return fail(GVL_ERR_ARG, "unknown track dtype %d", (int)dtype);
        }
    }
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

// Everything of a planned call (rows and records in ctx->trk) up to the execute launch: descriptor copy, tile map, per-tile
// descriptors, and the execute launch's parameters, kept in ctx so that trk_execute may follow later, on another stream.
static int trk_prepare(gvl_ctx *ctx, int64_t n_work, int64_t ploidy, int64_t n_queries, int64_t n_tracks,
                       const TrkDesc *host_desc, const int64_t *offset_idxs, int64_t total_per_track, const int64_t *query_seed,
                       uint64_t base_seed, const uint64_t *base_seed_dev, int64_t sub_batch, int32_t layout,
                       const int64_t *row_dst, const int64_t *row_tstride, cudaStream_t st) {
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
    P.layout_btp = layout == GVL_TRACK_LAYOUT_BTP;
    P.offset_idxs = offset_idxs;
    P.n_queries = n_queries;
    P.query_seed = query_seed;
    P.base_seed = base_seed;
    P.base_seed_dev = base_seed_dev;
    P.sub_batch = sub_batch;
    P.out = nullptr;
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
    if (!ctx->trk_params) ctx->trk_params = malloc(sizeof(TrkExecParams));
    if (!ctx->trk_params) return fail(GVL_ERR_ARG, "out of host memory");
    memcpy(ctx->trk_params, &P, sizeof(P));
    ctx->trk_plan_valid = true;
    return GVL_OK;
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

// gvl_dev_realign_tracks (interval sources `itv`) and gvl_dev_shift_and_realign_tracks (one track, `dense` source)
static int realign_impl(const char *who, gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                        const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
                        int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                        int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                        const float *dense, const int64_t *dense_offsets,
                        const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                        const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                        const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed, int64_t max_records,
                        int32_t layout, const int64_t *row_dst, const int64_t *row_tstride, void *out, int32_t dtype,
                        gvl_stream stream) {
    if (!ctx) return fail(GVL_ERR_ARG, "%s: NULL argument", who);
    // every argument is checked before the first launch: a rejected call leaves no plan behind, not even the previous one
    ctx->trk_plan_valid = false;
    if (!tab || !regions || !shifts || !(geno_offset_idx || svar2) || (itv ? !offset_idxs : !(dense && dense_offsets)) ||
        !track_lengths || !out_offsets || !strategy_ids || !params)
        return fail(GVL_ERR_ARG, "%s: NULL argument", who);
    if (svar2 && (!svar2->vk_off || !svar2->dense_range || !svar2->dense_present_off))
        return fail(GVL_ERR_ARG, "%s: NULL channel", who);
    int rc;
    if ((rc = check_track_output(who, layout, row_dst, row_tstride, dtype))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_work = batch * ploidy;
    if (n_work == 0 || n_tracks == 0 || total_per_track == 0) return GVL_OK;
    if (n_tracks < 0 || n_tracks > MAX_TRACKS) return fail(GVL_ERR_ARG, "at most %d tracks per call", MAX_TRACKS);
    for (int64_t t = 0; t < n_tracks; t++) {
        if (strategy_ids[t] < 0 || strategy_ids[t] > GVL_FILL_INTERPOLATE)
            return fail(GVL_ERR_ARG, "unknown insertion-fill strategy %d", strategy_ids[t]);
        if (strategy_ids[t] == GVL_FILL_INTERPOLATE && !(params[t] >= 1 && params[t] <= 3))
            return fail(GVL_ERR_ARG, "Interpolate order must be 1, 2 or 3");
    }
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
    if ((rc = trk_prepare(ctx, n_work, ploidy, batch, n_tracks, desc, offset_idxs, total_per_track, query_seed, base_seed,
                          base_seed_dev, sub_batch, layout, row_dst, row_tstride, st)))
        return rc;
    return out ? trk_execute(ctx, out, dtype, 0, GVL_TRACK_REDUCE_MEAN, st) : GVL_OK;  // (out == NULL: plan only)
}

int gvl_dev_realign_tracks(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                           const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
                           int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                           int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                           const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                           const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                           const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed, int64_t max_records,
                           int32_t layout, const int64_t *row_dst, const int64_t *row_tstride, void *out, int32_t dtype,
                           gvl_stream stream) {
    return realign_impl("gvl_dev_realign_tracks", ctx, tab, svar2, regions, shifts, geno_offset_idx, batch, ploidy, keep,
                        keep_offsets, to_rc, n_tracks, itv, offset_idxs, nullptr, nullptr, track_lengths, out_offsets,
                        total_per_track, strategy_ids, params, base_seed, base_seed_dev, sub_batch, query_seed, max_records,
                        layout, row_dst, row_tstride, out, dtype, stream);
}

int gvl_dev_realign_tracks_exec(gvl_ctx *ctx, void *out, int32_t dtype, gvl_stream stream) {
    if (!ctx) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_exec: ctx is NULL");
    if (!track_dtype_ok(dtype)) return fail(GVL_ERR_ARG, "gvl_dev_realign_tracks_exec: unknown track dtype %d", (int)dtype);
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->trk_plan_valid) return GVL_OK;  // (an empty or rejected plan: nothing to write)
    return trk_execute(ctx, out, dtype, 0, GVL_TRACK_REDUCE_MEAN, (cudaStream_t)stream);
}

int gvl_dev_realign_tracks_exec_binned(gvl_ctx *ctx, void *out, int32_t dtype, int32_t bin, int32_t reduce, gvl_stream stream) {
    const char *who = "gvl_dev_realign_tracks_exec_binned";
    if (!ctx) return fail(GVL_ERR_ARG, "%s: ctx is NULL", who);
    if (!track_dtype_ok(dtype)) return fail(GVL_ERR_ARG, "%s: unknown track dtype %d", who, (int)dtype);
    int rc;
    if ((rc = check_track_bin(who, bin, reduce))) return rc;
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (!ctx->trk_plan_valid) return GVL_OK;
    return trk_execute(ctx, out, dtype, bin, reduce, (cudaStream_t)stream);
}

int gvl_dev_shift_and_realign_tracks(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                                     const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx,
                                     int64_t batch, int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets,
                                     const uint8_t *to_rc, const float *tracks, const int64_t *track_offsets,
                                     const int32_t *track_lengths, const int64_t *out_offsets, int64_t total,
                                     int32_t strategy_id, double param, uint64_t base_seed,
                                     const int64_t *query_seed, int64_t max_records, float *out, gvl_stream stream) {
    return realign_impl("gvl_dev_shift_and_realign_tracks", ctx, tab, svar2, regions, shifts, geno_offset_idx, batch, ploidy,
                        keep, keep_offsets, to_rc, 1, nullptr, nullptr, tracks, track_offsets, track_lengths, out_offsets,
                        total, &strategy_id, &param, base_seed, nullptr, 0, query_seed, max_records, GVL_TRACK_LAYOUT_TBP,
                        nullptr, nullptr, out, GVL_TRACK_F32, stream);
}

static int paint_impl(const char *who, gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                      const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                      const uint8_t *to_rc, int32_t layout, const int64_t *row_dst, const int64_t *row_tstride, void *out,
                      int32_t dtype, int32_t bin, int32_t reduce, gvl_stream stream) {
    if (!ctx) return fail(GVL_ERR_ARG, "%s: NULL argument", who);
    ctx->trk_plan_valid = false;  // (as in realign_impl)
    if (!itv || !offset_idxs || !starts || !out_offsets) return fail(GVL_ERR_ARG, "%s: NULL argument", who);
    if (n_tracks < 0 || n_tracks > MAX_TRACKS) return fail(GVL_ERR_ARG, "%s: 0..%d tracks per call", who, MAX_TRACKS);
    int rc;
    if ((rc = check_track_output(who, layout, row_dst, row_tstride, dtype))) return rc;
    if ((rc = check_track_bin(who, bin, reduce))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (n_queries == 0 || n_tracks == 0 || total_per_track == 0) return GVL_OK;
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
    if ((rc = trk_prepare(ctx, n_queries, 1, n_queries, n_tracks, desc, offset_idxs, total_per_track, nullptr, 0, nullptr, 0,
                          layout, row_dst, row_tstride, st)))
        return rc;
    return trk_execute(ctx, out, dtype, bin, reduce, st);
}

int gvl_dev_paint_tracks(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                         const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                         const uint8_t *to_rc, int32_t layout, const int64_t *row_dst, const int64_t *row_tstride, void *out,
                         int32_t dtype, gvl_stream stream) {
    return paint_impl("gvl_dev_paint_tracks", ctx, n_tracks, itv, offset_idxs, starts, n_queries, out_offsets, total_per_track,
                      to_rc, layout, row_dst, row_tstride, out, dtype, 0, GVL_TRACK_REDUCE_MEAN, stream);
}

int gvl_dev_paint_tracks_binned(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                                const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                                const uint8_t *to_rc, int32_t layout, const int64_t *row_dst, const int64_t *row_tstride,
                                void *out, int32_t dtype, int32_t bin, int32_t reduce, gvl_stream stream) {
    return paint_impl("gvl_dev_paint_tracks_binned", ctx, n_tracks, itv, offset_idxs, starts, n_queries, out_offsets,
                      total_per_track, to_rc, layout, row_dst, row_tstride, out, dtype, bin, reduce, stream);
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

// ---- gvl_dev_realigned_track_intervals ----
__global__ void ritv_pair_items_kernel(const RowPlan *__restrict__ rows, int64_t n_work, int64_t n_pairs, int64_t *__restrict__ items) {
    const int64_t pair = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (pair < n_pairs) items[pair] = 1 + 2 * (int64_t)rows[pair % n_work].n_rec;
}

// the workspace of one sizing call, kept in ctx->ritv_ws for its emit call: per-pair item counts (later per-row interval
// counts), item_base, per-item interval counts, item_off, the RItems
struct RitvWs {
    int64_t *pair_cnt, *item_base, *item_cnt, *item_off;
    RItem *items;
};

static RitvWs ritv_ws_layout(void *base, int64_t n_pairs, int64_t item_cap) {
    RitvWs w;
    w.items = (RItem *)base;  // (32-byte aligned first)
    w.pair_cnt = (int64_t *)(w.items + item_cap);
    w.item_base = w.pair_cnt + n_pairs;
    w.item_cnt = w.item_base + n_pairs + 1;
    w.item_off = w.item_cnt + item_cap;
    return w;
}

static int ensure_ritv_ws(gvl_ctx *ctx, int64_t bytes) {
    if (bytes <= ctx->ritv_ws_bytes) return GVL_OK;
    GVL_CUDA(cudaDeviceSynchronize());
    if (ctx->ritv_ws) GVL_CUDA(cudaFree(ctx->ritv_ws));
    ctx->ritv_ws = nullptr;
    ctx->ritv_ws_bytes = 0;
    const int64_t cap = imax64(bytes + bytes / 2, 1 << 16);
    GVL_CUDA(cudaMalloc(&ctx->ritv_ws, (size_t)cap));
    ctx->ritv_ws_bytes = cap;
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

int gvl_dev_realigned_track_intervals(gvl_ctx *ctx, const int64_t *row_out, int64_t *out_offsets, int64_t cap, int32_t *out_starts,
                                      int32_t *out_ends, void *out_values, int32_t track_dtype, gvl_stream stream) {
    const char *who = "gvl_dev_realigned_track_intervals";
    if (!ctx || !out_offsets || cap < 0) return fail(GVL_ERR_ARG, "%s: NULL argument or negative size", who);
    if (!track_dtype_ok(track_dtype)) return fail(GVL_ERR_ARG, "%s: unknown track dtype %d", who, (int)track_dtype);
    if (cap && (!out_starts || !out_ends || !out_values)) return fail(GVL_ERR_ARG, "%s: NULL output with cap > 0", who);
    if (!ctx->trk_plan_valid || !ctx->trk_params) return fail(GVL_ERR_STATE, "%s: no track plan", who);
    RItvParams R;
    memset(&R, 0, sizeof(R));
    memcpy(&R.P, ctx->trk_params, sizeof(R.P));
    if (!R.P.tracks && R.P.inl[0].dense) return fail(GVL_ERR_STATE, "%s: the plan reads a dense source, not intervals", who);
    R.n_pairs = R.P.n_tracks * R.P.n_work;
    R.row_out = row_out;
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    if (cap == 0) {  // sizing call: items, their counts, per-row totals, out_offsets
        // item slots: 1 + 2 n_rec per pair, and the plan's records lie in the record buffer
        R.item_cap = R.P.n_tracks * (R.P.n_work + 2 * ctx->trk.trec_cap);
        const int64_t bytes = (int64_t)sizeof(RItem) * R.item_cap + 8 * (2 * R.n_pairs + 1 + 2 * R.item_cap + 1);
        if ((rc = ensure_ritv_ws(ctx, bytes))) return rc;
        const RitvWs W = ritv_ws_layout(ctx->ritv_ws, R.n_pairs, R.item_cap);
        ctx->ritv_pairs = -1;
        const unsigned pb = (unsigned)((R.n_pairs + 255) / 256);
        ritv_pair_items_kernel<<<pb, 256, 0, st>>>(R.P.rows, R.P.n_work, R.n_pairs, W.pair_cnt);
        GVL_LAUNCH_CHECK();
        if ((rc = scan_lengths(ctx, W.pair_cnt, R.n_pairs, W.item_base, st))) return rc;
        R.item_base = W.item_base;
        R.items = W.items;
        const unsigned blocks = (unsigned)imin64((R.item_cap + ITV_THREADS / 32 - 1) / (ITV_THREADS / 32), 148 * 32);
        ritv_count_kernel<<<blocks, ITV_THREADS, 0, st>>>(R, W.item_cnt);
        GVL_LAUNCH_CHECK();
        if ((rc = scan_lengths(ctx, W.item_cnt, R.item_cap, W.item_off, st))) return rc;
        R.item_off = W.item_off;
        GVL_CUDA(cudaMemsetAsync(W.pair_cnt, 0, sizeof(int64_t) * (size_t)R.n_pairs, st));
        ritv_rows_kernel<<<pb, 256, 0, st>>>(R, W.pair_cnt);
        GVL_LAUNCH_CHECK();
        if ((rc = scan_lengths(ctx, W.pair_cnt, R.n_pairs, out_offsets, st))) return rc;
        ctx->ritv_pairs = R.n_pairs;
        ctx->ritv_item_cap = R.item_cap;
        return GVL_OK;
    }
    if (ctx->ritv_pairs != R.n_pairs) return fail(GVL_ERR_STATE, "%s: no sizing call (cap = 0) over this plan", who);
    R.item_cap = ctx->ritv_item_cap;
    const RitvWs W = ritv_ws_layout(ctx->ritv_ws, R.n_pairs, R.item_cap);
    R.item_base = W.item_base, R.item_off = W.item_off, R.items = W.items;
    const unsigned blocks = (unsigned)imin64((cap + 255) / 256, 148 * 16);
    switch (track_dtype) {
        case GVL_TRACK_F32:
            ritv_emit_kernel<float><<<blocks, 256, 0, st>>>(R, out_offsets, cap, out_starts, out_ends, (float *)out_values);
            break;
        case GVL_TRACK_BF16:
            ritv_emit_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(R, out_offsets, cap, out_starts, out_ends, (__nv_bfloat16 *)out_values);
            break;
        default:
            ritv_emit_kernel<__half><<<blocks, 256, 0, st>>>(R, out_offsets, cap, out_starts, out_ends, (__half *)out_values);
    }
    GVL_LAUNCH_CHECK();
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
