/*
 * gvl_b200.h -- C ABI of the B200-native haplotype-reconstruction path.
 *
 * Drop-in boundary for GenVarLoader's PyO3 extension module `genvarloader.genvarloader`
 * (reference: src/lib.rs:17-89, src/ffi/mod.rs).  Plain pointers and sizes only; no torch,
 * numpy or C++ types cross this boundary.  Every entry returns a status code
 * (0 = GVL_OK) and leaves a message retrievable with gvl_last_error() on failure -- the
 * reference panics/raises instead (src/ffi/mod.rs:45-55), the binding maps codes to
 * exceptions.
 *
 * Two layers:
 *   gvl_*      HOST-buffer entries with the argument lists of the reference's #[pyfunction]s
 *              (what a cgo/ctypes/PyO3 stub binds 1:1).  Sample-scale static arrays
 *              (reference, variant table, genotype CSR, interval SoA) are uploaded once and
 *              cached by host address (gvl_pin_static); O(batch)
 *              arrays are copied per call; results are copied back to host buffers.
 *   gvl_dev_*  DEVICE-pointer entries used by the Python `Dataset` host: inputs/outputs are
 *              device buffers owned by the caller (torch tensors), work is enqueued on the
 *              caller's stream, no host synchronisation except where stated.
 *
 * All arrays are C-contiguous with the reference's exact dtypes: i32 regions/shifts/positions,
 * i64 offsets/indices, u8 bytes/bools, f32 tracks, f64 params.
 */
#ifndef GVL_B200_H
#define GVL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define GVL_OK 0
#define GVL_ERR_CUDA 1      /* a CUDA runtime call failed                                   */
#define GVL_ERR_ARG 2       /* contract violation detectable on the host                   */
#define GVL_ERR_CAPACITY 3  /* device workspace overflow reported by a kernel              */
#define GVL_ERR_STATE 4     /* call sequence error (e.g. exec without plan)                */

/* Output encodings of the fused epilogue (a6 + a14 in SURVEY.md section 8). */
#define GVL_MODE_U8 0        /* ASCII haplotype bytes, what reconstruct_haplotypes_fused returns       */
#define GVL_MODE_ONEHOT 1    /* uint8 (L,4) one-hot, alphabet ACGT  (seqpro.DNA.ohe of the bytes)      */
#define GVL_MODE_ANNOTATED 2 /* bytes + int32 variant index + int32 reference coordinate per base      */
#define GVL_MODE_ONEHOT_CF 3 /* uint8 (4,L) channels-first one-hot ("alphabet length" layout)          */

/* Insertion-fill strategies, python/genvarloader/_dataset/_insertion_fill.py:9-13. */
#define GVL_FILL_REPEAT_5P 0
#define GVL_FILL_REPEAT_5P_NORM 1
#define GVL_FILL_CONSTANT 2
#define GVL_FILL_FLANK_SAMPLE 3
#define GVL_FILL_INTERPOLATE 4

typedef struct gvl_ctx gvl_ctx;
typedef void *gvl_stream; /* cudaStream_t / CUstream; NULL = legacy default stream */

/* ---- context ---------------------------------------------------------------------- */
int gvl_ctx_create(int device, gvl_ctx **out);
void gvl_ctx_destroy(gvl_ctx *ctx);
const char *gvl_last_error(void);
/* Number of kernels this library has launched since the counter was last reset. */
int64_t gvl_launch_count(int reset);
/* Blocks until the stream is idle, then reports any device-side status flag
 * (GVL_ERR_CAPACITY) raised by kernels of this context. */
int gvl_ctx_check(gvl_ctx *ctx, gvl_stream stream);

/* SVAR1-style static tables: reference + global variant table + sparse genotype CSR.
 * Replaces the cached `_HapsFfiStatic` (python/genvarloader/_dataset/_haps.py:233-247,330-348)
 * and the memmapped `genotypes.data/offsets` passed to every FFI call (_haps.py:844-866).
 * Device pointers for gvl_dev_*; `ref` must be readable up to the next multiple of 16 bytes. */
typedef struct {
    const uint8_t *ref;          /* u8[ref_offsets[n_contigs]]                 */
    const int64_t *ref_offsets;  /* i64[n_contigs+1]                           */
    int64_t n_contigs;
    const int32_t *v_starts;     /* i32[n_variants]                            */
    const int32_t *ilens;        /* i32[n_variants]                            */
    const uint8_t *alt_alleles;  /* u8[alt_offsets[n_variants]]                */
    const int64_t *alt_offsets;  /* i64[n_variants+1]                          */
    int64_t n_variants;
    const int32_t *geno_v_idxs;  /* i32[G]                                     */
    const int64_t *geno_starts;  /* i64[n_geno]  row 0 of the (2,n) offsets    */
    const int64_t *geno_stops;   /* i64[n_geno]  row 1                         */
    int64_t n_geno;
    /* Optional (NULL = absent): the reference and the ALT alleles re-encoded by gvl_dev_pack_reference, one 4-bit
     * one-hot code per base.  When BOTH are present, GVL_MODE_ONEHOT executes over them (8 positions per lane,
     * 256-bit stores); results are identical with and without them. */
    const uint32_t *ref_packed;  /* u32[gvl_packed_reference_words(ref_offsets[n_contigs])], 16-byte aligned */
    const uint32_t *alt_packed;  /* u32[gvl_packed_reference_words(alt_offsets[n_variants])], 16-byte aligned */
} gvl_sparse_tables;

/* Packed form of the reference for the one-hot execute path: base r of the concatenated reference is nibble r&7
 * (low nibble first) of word r>>3, code A=1 C=2 G=4 T=8, any other byte 0.  Built once per dataset replica on the
 * device (a static-table transform like the upload itself; the reference keeps ASCII only, _reference.py:53-120). */
int64_t gvl_packed_reference_words(int64_t n_bases);
int gvl_dev_pack_reference(gvl_ctx *ctx, const uint8_t *ref, int64_t n_bases, uint32_t *ref_packed, gvl_stream stream);

/* Per-track interval SoA (python/genvarloader/_dataset/_tracks.py:327-339).  Device layer: the three arrays are 16-byte
 * aligned and readable up to the next multiple of 16 bytes; every slot is sorted by start and free of overlaps
 * (gvl_flatten_intervals). */
typedef struct {
    const int32_t *itv_starts;
    const int32_t *itv_ends;
    const float *itv_values;
    const int64_t *itv_offsets; /* i64[n_slots+1] */
    int64_t n_slots;
} gvl_intervals;

/* ---- device layer: haplotypes ------------------------------------------------------ */
/*
 * Phase A ("plan").  One launch: per (query, hap) row runs get_diffs_sparse
 * (src/genotypes/mod.rs:15-125) and the variant state machine of reconstruct_haplotype_core
 * (src/reconstruct/mod.rs:39-256), emitting a compact segment table into the context's
 * workspace, then sizes rows exactly as src/ffi/mod.rs:794-811.
 *   regions (b,3) i32, shifts (b,p) i32, geno_offset_idx (b,p) i64, keep/keep_offsets/to_rc optional (NULL)
 *   output_length  >=0 fixed; -1 ragged, sized from the diffs; -2 rows sized by the caller:
 *                  out_offsets is then an INPUT (gap-free, non-decreasing), as in the un-fused
 *                  reconstruct_haplotypes_from_sparse (src/ffi/mod.rs:634-655)
 *   max_records    upper bound on the summed per-row variant counts (workspace capacity)
 *   out_offsets    device i64[b*p+1], written (read when output_length == -2)
 *   diffs          optional device i32[b*p], written (get_diffs_sparse result)
 * No host sync.
 */
int gvl_dev_hap_plan(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *regions, const int32_t *shifts,
                     const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const uint8_t *keep,
                     const int64_t *keep_offsets, const uint8_t *to_rc, int64_t output_length, int64_t max_records,
                     int64_t *out_offsets, int32_t *diffs, gvl_stream stream);

/* svar2 two-channel variant source, flat per-call layout of the reference's `FlatChannels`
 * (src/svar2/mod.rs:150-160; consumed by reconstruct_haplotypes_from_svar2, src/reconstruct/mod.rs:620-826).
 * Device pointers.  Keys are indices into a DECODED key table that stands for svar2_codec::decode_key +
 * decode_alt (src/svar2/mod.rs:17-28; third-party codec, parity unpinned): the table is passed as
 * gvl_sparse_tables.{ilens, alt_offsets, alt_alleles, n_variants}; an empty ALT means a pure deletion whose
 * anchor base is taken from ref[pos] (src/reconstruct/mod.rs:720-733).  Both channels are position-sorted. */
typedef struct {
    const int32_t *vk_pos;            /* per-hap var_key channel: positions                           */
    const int32_t *vk_key;            /*                          keys                                */
    const int64_t *vk_off;            /* i64[b*p+1] CSR offsets by flat row k = query*ploidy + hap    */
    const int32_t *dense_pos;         /* shared dense channel: positions                              */
    const int32_t *dense_key;         /*                       keys                                   */
    const int32_t *dense_range;       /* i32[b,2] window [ds, de) of each query                       */
    const uint8_t *dense_present;     /* presence bits over the window, LSB first                     */
    const int64_t *dense_present_off; /* i64[b*p+1] BIT offsets by flat row                           */
    /* Optional (NULL / 0 = the per-call flat layout above).  A dataset replica keeps the two channels RESIDENT instead
     * of gathering them per call (the range cache of docs/source/format.md:88-96, `_svar2_haps.py:1269-1313`): the
     * per-row arrays are then tables over all (region, sample, ploid) slots and the per-query one over all regions. */
    const int64_t *vk_stop;           /* row i holds var_key entries [vk_off[i], vk_stop[i])           */
    const int64_t *row_slot;          /* i64[b*p]: row k reads entry row_slot[k] of vk_off / vk_stop / dense_present_off */
    int64_t query_div;                /* > 0: query q reads dense_range[row_slot[q*p] / query_div] (slots per region) */
} gvl_svar2_channels;

/* gvl_dev_hap_plan for the svar2 source: merges each row's two channels on the device (stable by position,
 * var_key first on ties, src/svar2/mod.rs:45-66), then plans exactly like the SVAR1 source.  Variant indices
 * written by the annotated mode are LOCAL to the row (src/reconstruct/mod.rs:734).
 *   max_merged = sum over rows of (var_key entries + dense window size)  (workspace capacity) */
int gvl_dev_hap_plan_svar2(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *ch,
                           const int32_t *regions, const int32_t *shifts, int64_t batch, int64_t ploidy,
                           const uint8_t *to_rc, int64_t output_length, int64_t max_merged, int64_t *out_offsets,
                           int32_t *diffs, gvl_stream stream);

/* hap_diffs_svar2, src/svar2/mod.rs:73-146 (the core of hap_diffs_from_svar2_readbound, src/ffi/mod.rs:1414-1427): the
 * clipped length differences of get_diffs_sparse over each row's MERGED two-channel list.  Only tab->ilens (the decoded
 * key table's ILEN column) is read.  diffs: device i32[batch*ploidy].  Leaves the current haplotype plan intact. */
int gvl_dev_hap_diffs_svar2(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *ch, const int32_t *regions,
                            int64_t batch, int64_t ploidy, int64_t max_merged, int32_t *diffs, gvl_stream stream);

/* Total number of output positions of the current plan (= out_offsets[-1]).  Fixed-length plans
 * answer from the host; ragged plans synchronise the stream once (the reference sizes its
 * allocation at the same point, src/ffi/mod.rs:814). */
int gvl_dev_hap_total(gvl_ctx *ctx, gvl_stream stream, int64_t *total);

/*
 * Phase B ("execute").  One launch over output tiles: copies reference spans, scatters ALT
 * bytes, pads, reverse-complements masked rows (src/reverse.rs:45-69) and encodes, writing each
 * output byte exactly once.  Buffers are device pointers, 16-byte aligned:
 *   GVL_MODE_U8         out u8[total]
 *   GVL_MODE_ONEHOT     out u8[total*4]           (row-major (L,4) per row)
 *   GVL_MODE_ONEHOT_CF  out u8[total*4]           ((4,L) per row; fixed-length plans only)
 *   GVL_MODE_ANNOTATED  out u8[total], annot_v i32[total], annot_pos i32[total]
 */
int gvl_dev_hap_exec(gvl_ctx *ctx, const gvl_sparse_tables *tab, int mode, uint8_t pad_char, uint8_t *out,
                     int32_t *annot_v, int32_t *annot_pos, gvl_stream stream);

/* Standalone get_diffs_sparse on device (src/ffi/mod.rs:145-157).  q_starts/q_ends/v_starts may
 * be NULL together (unclipped sum).  diffs: device i32[n_queries*ploidy]. */
int gvl_dev_get_diffs_sparse(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int64_t *geno_offset_idx,
                             int64_t n_queries, int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets,
                             const int32_t *q_starts, const int32_t *q_ends, int use_v_starts, int32_t *diffs,
                             gvl_stream stream);

/* ---- device layer: tracks ---------------------------------------------------------- */
/* Element type of a track output.  Values are computed in float32 as for GVL_TRACK_F32 and narrowed at the store with
 * round-to-nearest-even (cvt.rn, no flush to zero: subnormals are kept, values beyond the float16 range become +-inf, NaN
 * becomes the device's canonical NaN): bit for bit the float32 output cast to the type on the device.  Only the output
 * changes: stored intervals stay float32. */
#define GVL_TRACK_F32 0
#define GVL_TRACK_BF16 1
#define GVL_TRACK_F16 2

/* Binned track output (gvl_dev_realign_tracks_exec_binned, gvl_dev_paint_tracks_binned, gvl_fixed_job.track_bin): every
 * row is cut into bins of `bin` output positions (a power of two, 2..GVL_TRACK_BIN_MAX; 0 or 1 = unbinned) and one value
 * per bin is stored: bin k of a row covers its output positions [k*bin, (k+1)*bin), so a reversed row's bins are its
 * forward bins reversed.  Row lengths and row offsets (out_offsets, row_dst, row_tstride) stay in unbinned positions and
 * must be multiples of `bin`: a row whose values start at element o of the unbinned layout has its bins at o / bin, and
 * `out` holds n_tracks * total_per_track / bin elements.  The reduction runs on the float32 values:
 *   SUM   the bin's values summed in float64, rounded to float32, then narrowed to the dtype like every value;
 *   MEAN  that float64 sum divided by bin in float64, with the same roundings;
 *   MAX   the largest value, narrowed.
 * A NaN in the bin makes it NaN for all three.  The float64 order is fixed by the row alone, so a row's bins have the same
 * bits in every call.  An unknown bin or reduction is GVL_ERR_ARG before any launch. */
#define GVL_TRACK_REDUCE_MEAN 0
#define GVL_TRACK_REDUCE_SUM 1
#define GVL_TRACK_REDUCE_MAX 2
#define GVL_TRACK_BIN_MAX 4096

/* Where the rows of a track call land in `out` (n_tracks * total_per_track elements).  Row k (= q*p + h; p = 1 when
 * painting) has out_offsets[k+1] - out_offsets[k] values, written reversed on masked rows in every layout. */
#define GVL_TRACK_LAYOUT_TBP 0  /* track-major (t, b, p, ~l): the reference's flat buffer (_reconstruct.py:238); row k of
                                   track t starts at t * total_per_track + out_offsets[k] */
#define GVL_TRACK_LAYOUT_BTP 1  /* (b, t, p, ~l): every query's tracks adjacent, the order the reference's offsets describe
                                   (_reconstruct.py:292-300) and what Dataset returns; row (q, t, h) starts at n_tracks *
                                   out_offsets[q*p] + t * (out_offsets[(q+1)*p] - out_offsets[q*p]) + out_offsets[q*p + h] -
                                   out_offsets[q*p].  out_offsets must be gap-free. */
#define GVL_TRACK_LAYOUT_ROWS 2 /* row k of track t starts at row_dst[k] + t * row_tstride[k] (device i64[b*p] each).  The
                                   caller guarantees that the ranges of all (row, track) pairs are disjoint and lie inside
                                   [0, n_tracks*total_per_track): every value is then written exactly once when they cover
                                   the buffer.  out_offsets still gives each row's length and must be gap-free.  Used for
                                   spliced output: the elements of a splice row are separate rows written straight into
                                   their place in the concatenation. */
/* row_dst and row_tstride are both given with GVL_TRACK_LAYOUT_ROWS and both NULL with the other layouts; an unknown layout
 * or dtype (GVL_TRACK_*) is GVL_ERR_ARG.  These checks run before the first launch: a rejected call plans nothing and
 * drops the plan of the call before it.  `out` is device memory, 16-byte aligned. */

/*
 * intervals_and_realign_track_fused (src/ffi/mod.rs:2553-2672) for ALL tracks of a batch in one
 * plan launch + one execute launch: paints stored intervals (src/intervals.rs:19-126) and
 * realigns them to haplotype coordinates (src/tracks/mod.rs:224-406) without the dense scratch.
 *   svar2                NULL: the variants come from the SVAR1 tables of `tab`; non-NULL: from the svar2 two-channel
 *                        source (merged on the device like gvl_dev_hap_plan_svar2; geno_offset_idx and the keep mask are
 *                        then ignored, max_records = max_merged)
 *   n_tracks             tracks realigned in this call (<= 64)
 *   itv[t]               HOST array of n_tracks descriptors holding DEVICE pointers
 *   offset_idxs          device i64[n_tracks*b]: interval slot per (track, query) (dataset idx for
 *                        SAMPLE tracks, region idx for ANNOT tracks, _reconstruct.py:233-236)
 *   track_lengths        device i32[b]: source window length per query (_reconstruct.py:191)
 *   out_offsets          device i64[b*p+1] per-track row offsets (same for every track), input
 *   total_per_track      out_offsets[b*p] (host value)
 *   strategy_ids/params  HOST arrays, one per track (python/genvarloader/_dataset/_insertion_fill.py:89)
 *   base_seed_dev        optional device u64[1]: when non-NULL the seed is read from device memory at run time instead of
 *                        `base_seed` (a CUDA graph captured once then serves batches with different seeds)
 *   sub_batch            > 0: the call holds several logical batches of this many queries: query q belongs to batch
 *                        q / sub_batch, its FlankSample row index is q % sub_batch and its seed base_seed_dev[q / sub_batch];
 *                        <= 0: one batch (seed base_seed_dev[0] or base_seed)
 *   query_seed           optional device i64[b]: global batch row used as the FlankSample seed
 *                        component when one logical batch is split over several calls / GPUs
 *                        (src/tracks/mod.rs:696-702); NULL = local row index
 *   layout, row_dst, row_tstride   GVL_TRACK_LAYOUT_*
 *   out, dtype           `dtype` elements (GVL_TRACK_*) written in `layout`.  out == NULL plans the call without executing
 *                        it: gvl_dev_realign_tracks_exec writes the values later, on the same stream or another (a
 *                        pipeline runs the latency-bound part -- variant plan, tile map, per-tile searches -- on one stream
 *                        and the bandwidth-bound execute launch on another; the caller orders the two).
 */
int gvl_dev_realign_tracks(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                           const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
                           int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                           int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                           const int32_t *track_lengths, const int64_t *out_offsets, int64_t total_per_track,
                           const int32_t *strategy_ids, const double *params, uint64_t base_seed,
                           const uint64_t *base_seed_dev, int64_t sub_batch, const int64_t *query_seed, int64_t max_records,
                           int32_t layout, const int64_t *row_dst, const int64_t *row_tstride, void *out, int32_t dtype,
                           gvl_stream stream);

/* The execute launch of the last call planned on this context: writes elements of `dtype` (GVL_TRACK_*; any other value:
 * GVL_ERR_ARG) into `out` (device, n_tracks * total_per_track elements, 16-byte aligned).  Writes nothing after an empty or
 * rejected plan. */
int gvl_dev_realign_tracks_exec(gvl_ctx *ctx, void *out, int32_t dtype, gvl_stream stream);
/* The same launch with a binned store (GVL_TRACK_REDUCE_*): `out` holds n_tracks * total_per_track / bin elements. */
int gvl_dev_realign_tracks_exec_binned(gvl_ctx *ctx, void *out, int32_t dtype, int32_t bin, int32_t reduce, gvl_stream stream);

/* shift_and_realign_tracks_sparse (src/ffi/mod.rs:2439-2458) and shift_and_realign_tracks_from_svar2
 * (src/tracks/mod.rs:705-856) on device: ONE track whose source is a dense f32 window per query (`tracks` ragged by
 * `track_offsets` i64[b+1]) instead of intervals, written track-major as float32.  svar2 as in gvl_dev_realign_tracks
 * (`tab` then carries the decoded key table in ilens / n_variants; max_records = max_merged = sum over rows of (var_key
 * entries + dense window size)).  track_lengths[q] = track_offsets[q+1]-track_offsets[q] as device i32[b]. */
int gvl_dev_shift_and_realign_tracks(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                                     const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx,
                                     int64_t batch, int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets,
                                     const uint8_t *to_rc, const float *tracks, const int64_t *track_offsets,
                                     const int32_t *track_lengths, const int64_t *out_offsets, int64_t total,
                                     int32_t strategy_id, double param, uint64_t base_seed,
                                     const int64_t *query_seed, int64_t max_records, float *out, gvl_stream stream);

/* intervals_to_tracks for ALL tracks of a batch in one launch (the un-realigned track read, Tracks._call_float32
 * python/genvarloader/_dataset/_tracks.py:370-420; src/ffi/mod.rs:190-201 is the one-track GVL_TRACK_LAYOUT_TBP case):
 * itv is a HOST array of n_tracks descriptors, offset_idxs device i64[n_tracks*n_queries], out_offsets device
 * i64[n_queries+1] (per track, gap-free), to_rc optional device u8[n_queries] (masked rows are written reversed,
 * src/reverse.rs:25-38).  One row per query; layout, row_dst, row_tstride, out and dtype as in gvl_dev_realign_tracks
 * (`out` is required). */
int gvl_dev_paint_tracks(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                         const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                         const uint8_t *to_rc, int32_t layout, const int64_t *row_dst, const int64_t *row_tstride, void *out,
                         int32_t dtype, gvl_stream stream);
/* gvl_dev_paint_tracks with a binned store (GVL_TRACK_REDUCE_*): `out` holds n_tracks * total_per_track / bin elements. */
int gvl_dev_paint_tracks_binned(gvl_ctx *ctx, int64_t n_tracks, const gvl_intervals *itv, const int64_t *offset_idxs,
                                const int32_t *starts, int64_t n_queries, const int64_t *out_offsets, int64_t total_per_track,
                                const uint8_t *to_rc, int32_t layout, const int64_t *row_dst, const int64_t *row_tstride,
                                void *out, int32_t dtype, int32_t bin, int32_t reduce, gvl_stream stream);

/* The stored intervals of one slot over one window per row (the "intervals" kind of Dataset.with_tracks).  tracks is a
 * HOST array of n_tracks (<= 64) descriptors; row k (device arrays of n_rows entries) reads slot row_slot[k] of track
 * row_track[k] over the window [row_w0[k], row_w1[k]): the intervals with end > w0 and start < w1, in stored order, the
 * first one's start raised to w0 and the last one's end lowered to w1.  An empty window (w1 <= w0), or a slot or track
 * out of range, gives no intervals.  Two calls over the same rows:
 *   cap == 0: writes out_offsets (device i64[n_rows + 1], row k's intervals at [out_offsets[k], out_offsets[k + 1])) and
 *             nothing else; the caller reads out_offsets[n_rows] to size the outputs;
 *   cap > 0:  reads those out_offsets and writes out_starts / out_ends (device i32[cap]) and out_values (device, cap
 *             elements of track_dtype, GVL_TRACK_*: the float32 values narrowed as by gvl_dev_realign_tracks_exec).
 *             A row whose intervals would end past cap is not written. */
int gvl_dev_track_intervals(gvl_ctx *ctx, const gvl_intervals *tracks, int64_t n_tracks, const int64_t *row_slot,
                            const int32_t *row_track, const int32_t *row_w0, const int32_t *row_w1, int64_t n_rows,
                            int64_t *out_offsets, int64_t cap, int32_t *out_starts, int32_t *out_ends, void *out_values,
                            int32_t track_dtype, gvl_stream stream);

/* The rows of the last track plan on this context (gvl_dev_realign_tracks with out == NULL) cut into intervals instead of
 * executed (the "realigned-intervals" kind of Dataset.with_tracks).  Every output position p of a planned row has the
 * source the execute resolves for it; the source's identity is the stored interval that holds it (none outside every
 * interval and outside the track window), one per record for Repeat5pNormalized / Constant insertion fills, one per
 * position for Interpolate fills, and that of the sampled position for FlankSample fills.  A row's intervals are the
 * maximal runs of one identity other than none, in ascending order: (w0 + first, w0 + last + 1, value), w0 = the row's
 * query start (regions[q, 1]), value = the float32 value the execute computes there narrowed to track_dtype.  Strand
 * reverses nothing.  row_out (device i64[n_tracks * n_work], or NULL) gives the output row of (track t, plan row k) at
 * t * n_work + k, a permutation; NULL = (query, track, ploid) order.  Two calls over the same plan:
 *   cap == 0: writes out_offsets (device i64[n_tracks * n_work + 1]) and nothing else; keeps its item table on the context;
 *   cap > 0:  writes out_starts / out_ends (device i32[cap]) and out_values (cap elements of track_dtype), reading the
 *             out_offsets of the sizing call, which must be the last one on this context.
 * GVL_ERR_STATE without a valid plan (or for a plan of gvl_dev_shift_and_realign_tracks), or for cap > 0 without its
 * sizing call.  A record overflow of the plan is reported by gvl_ctx_check, as for the execute. */
int gvl_dev_realigned_track_intervals(gvl_ctx *ctx, const int64_t *row_out, int64_t *out_offsets, int64_t cap, int32_t *out_starts,
                                      int32_t *out_ends, void *out_values, int32_t track_dtype, gvl_stream stream);

/* ---- device layer: the small entries either side of reconstruction ------------------ */
/* choose_exonic_variants, src/ffi/mod.rs:229-238 -> src/genotypes/mod.rs:132-176: for every (query, hap) row,
 * keep_offsets[k+1] - keep_offsets[k] = size of its genotype slice and keep[keep_offsets[k] + i] = 1 iff variant i
 * lies fully inside [starts[q], ends[q]) (v_pos >= start && v_pos - min(ilen,0) + 1 <= end).
 *   starts/ends i32[n_queries], geno_offset_idx i64[n_queries*ploidy], keep u8[keep_cap] (may be NULL: offsets only),
 *   keep_offsets i64[n_queries*ploidy + 1].  Entries beyond keep_cap are not written; the caller compares
 *   keep_offsets[n_work] with keep_cap (the host entry below does).  No host sync. */
int gvl_dev_choose_exonic_variants(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *starts, const int32_t *ends,
                                   const int64_t *geno_offset_idx, int64_t n_queries, int64_t ploidy, uint8_t *keep,
                                   int64_t keep_cap, int64_t *keep_offsets, gvl_stream stream);

/* get_reference, src/ffi/mod.rs:2402-2411 -> src/reference/mod.rs:56-120: row i = contig regions[i,0] from
 * regions[i,1] on, positions outside the contig filled with pad_char, masked rows reverse-complemented
 * (src/reverse.rs:45-69).  Runs as the zero-variant case of the haplotype plan + execute kernels, so GVL_MODE_ONEHOT
 * (with tab->ref_packed: the packed kernel) is available besides GVL_MODE_U8.  Only tab->{ref, ref_offsets,
 * n_contigs, ref_packed} are read.
 *   row_length >= 0: every row has that length, out_offsets (device i64[n+1]) is written, no host sync;
 *   row_length == -1: rows are sized by the caller's out_offsets (an input; the reference requires
 *                     out_offsets[i+1] - out_offsets[i] == end - start), one stream sync like every ragged plan. */
int gvl_dev_get_reference(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *regions, int64_t *out_offsets,
                          int64_t n_regions, int64_t row_length, const uint8_t *to_rc, int mode, uint8_t pad_char,
                          uint8_t *out, gvl_stream stream);

/* ragged_to_padded, src/ragged/mod.rs:7-23 (seqpro-core Ragged::to_padded_into): copies min(len_r, out_len) items of
 * row r to out[r, :]; `out` is (n_rows, out_len) items of `itemsize` bytes PRE-FILLED with the pad value by the
 * caller, exactly like the reference.  Device pointers, any alignment. */
int gvl_dev_ragged_to_padded(gvl_ctx *ctx, const void *data, const int64_t *offsets, int64_t n_rows, void *out,
                             int64_t itemsize, int64_t out_len, gvl_stream stream);
/* The same with the padding written by the kernel: `out` may be uninitialised, `pad_item` is a HOST pointer to one item
 * (itemsize <= 8 bytes).  One pass over the output instead of pre-fill + copy. */
int gvl_dev_ragged_to_padded_fill(gvl_ctx *ctx, const void *data, const int64_t *offsets, int64_t n_rows, void *out,
                                  int64_t itemsize, int64_t out_len, const void *pad_item, gvl_stream stream);

/* ---- device layer: batch preparation (the host prep of the reference, on the device) --- */
/* Per-replica region table for gvl_dev_batch_prep: the reference's `_full_regions` (int32 (R,4): contig index, start,
 * end, strand in {+1,-1}; python/genvarloader/_dataset/_open.py:146-164) resident in HBM. */
typedef struct {
    const int32_t *full_regions; /* device i32[n_regions*4], 16-byte aligned */
    int64_t n_regions, n_samples, ploidy;
    int32_t rc_neg;              /* reverse(-complement) negative-strand regions (Dataset.with_settings(rc_neg=)) */
} gvl_dataset_view;

/* Device buffers of one prepared batch (caller-owned; b = batch, p = ploidy, or 1 when ref_slot >= 0). */
typedef struct {
    int32_t *regions;     /* i32[b*3]   contig, start (+ jitter), end                    */
    int32_t *shifts;      /* i32[b*p]   zero (deterministic shifts, _haps.py:720-730)    */
    int64_t *goi;         /* i64[b*p]   geno_offset_idx                                  */
    uint8_t *to_rc;       /* u8[b*p]    per-row strand mask                              */
    uint8_t *to_rc_q;     /* u8[b]      per-query strand mask (un-realigned tracks), may be NULL */
    int64_t *offset_idxs; /* i64[n_tracks*b] interval slot per (track, query), NULL when n_tracks == 0 */
    uint64_t *base_seed;  /* u64[n logical batches] xor-reduce of ds_idx: the deterministic insertion-fill seed (_reconstruct.py:215-218), may be NULL */
    int32_t *starts;      /* i32[b] = regions[:,1], contiguous (gvl_dev_paint_tracks takes it), may be NULL */
} gvl_batch_args;

/* O(batch) arguments of plan / realign / paint from flat dataset indices, on the device: what
 * `_getitem_unspliced` (_dataset/_query.py:161-175), `Haps._get_geno_offset_idx` (_haps.py:757-768), the strand masks
 * (_haps.py:838-843, _reconstruct.py:251-256) and the interval-slot choice (_reconstruct.py:233-236) compute with numpy.
 *   ds_idx      device i64[batch]: r * n_samples + s over the FULL (regions, samples) grid (_indexing.py:237-245)
 *   jitter      optional device i32[batch]: per-query start offset drawn by the caller's generator (_query.py:165-171)
 *   sub_batch   > 0: the call holds several LOGICAL batches of this many queries (a loader reading ahead); fill seeds
 *               are then per logical batch (args->base_seed has ceil(batch / sub_batch) words); <= 0: one batch
 *   ref_slot    >= 0: "reference" rows -- one row per query that points at this (empty) genotype slot; < 0: haplotypes
 *   annot_mask  bit t set: track t is an ANNOT track (slot = region index) instead of a SAMPLE track (dataset index)
 * No host sync; safe to capture in a CUDA graph (all arguments are captured by value). */
int gvl_dev_batch_prep(gvl_ctx *ctx, const gvl_dataset_view *view, const int64_t *ds_idx, const int32_t *jitter,
                       int64_t batch, int64_t sub_batch, int64_t ref_slot, int64_t n_tracks, uint32_t annot_mask,
                       const gvl_batch_args *args, gvl_stream stream);
/* track_lengths[q] = (end - start) - min(0, min_h diffs[q,h]) (HapsTracks.__call__, _dataset/_reconstruct.py:191-196): the
 * source-window length of every query of a realigned-track call.  regions i32[b*3], diffs i32[b*p], out i32[b]; device. */
int gvl_dev_track_lengths(gvl_ctx *ctx, const int32_t *regions, const int32_t *diffs, int64_t batch, int64_t ploidy,
                          int32_t *track_lengths, gvl_stream stream);
/* cudaMemcpyAsync(host -> device) on the caller's stream: one copy stages the indices of a whole ring of batches. */
int gvl_dev_upload(gvl_ctx *ctx, void *dev, const void *host, int64_t bytes, gvl_stream stream);

/* ---- device layer: one fixed-length (region, sample) batch, end to end ------------------ */
/* What `Dataset.__getitem__` (_dataset/_impl.py:2074-2121 -> _query.py:66-204 -> Haps.__call__ _haps.py:578-870 /
 * HapsTracks.__call__ _reconstruct.py:132-307) does for a dataset state with a FIXED output length, as two calls over
 * prepared state: everything that does not change from batch to batch lives in a `gvl_fixed_job` the caller fills once.
 * All pointers are device pointers unless noted; `args`, `out_offsets`, `diffs`, `track_lengths` are scratch sized for
 * the largest batch the job will see.  No host sync; graph-capturable. */
typedef struct gvl_fixed_job {
    const gvl_dataset_view *view;     /* HOST pointer */
    const gvl_sparse_tables *tab;     /* HOST pointer */
    const gvl_svar2_channels *svar2;  /* HOST pointer or NULL (sparse CSR source); its row_slot is ignored: rows read slot args.goi[k] */
    gvl_batch_args args;
    int64_t *out_offsets;             /* i64[cap*rows_p + 1] */
    int32_t *diffs;                   /* i32[cap*ploidy]   realigned tracks only, else NULL */
    int32_t *track_lengths;           /* i32[cap]          realigned tracks only, else NULL */
    const int64_t *paint_offsets;     /* i64[cap + 1] = q * output_length: un-realigned tracks only, else NULL */
    const gvl_intervals *itv;         /* HOST pointer, n_tracks entries (NULL when n_tracks == 0) */
    const int32_t *strategy_ids;      /* HOST i32[n_tracks] insertion-fill strategy per track */
    const double *params;             /* HOST f64[n_tracks] */
    int64_t ploidy, rows_p;           /* rows_p = 1 for "reference" / track-only reads, else ploidy */
    int64_t output_length;
    int64_t ref_slot;                 /* >= 0: every row reads this (empty) genotype slot; < 0: haplotypes */
    int64_t n_tracks;
    int64_t max_slot_len;             /* upper bound of one row's variant-list length: the plan workspace is rows * (this + 1) and every
                                       * row owns a static slice of it (no allocation atomics in the plan kernels) */
    int64_t typ_slot_len;             /* typical (about twice the mean) variant-list length of a row: a HINT for the one-hot execute
                                       * kernel's tile length where the bound is loose (svar2: the bound counts the cohort's whole dense
                                       * window); 0 = use the bound */
    uint32_t annot_mask;
    int32_t mode;                     /* GVL_MODE_* of the sequence output; < 0: no sequence output */
    int32_t realign;                  /* tracks are realigned to the haplotypes (needs mode >= 0 and ref_slot < 0) */
    int32_t rc_neg;                   /* reverse(-complement) rows of negative-strand regions */
    uint8_t pad_char;
    int32_t track_dtype;              /* GVL_TRACK_* element type of `trk` (0 = float32) */
    int32_t track_bin, track_reduce;  /* binned tracks (0 = unbinned; output_length must be a multiple of track_bin) */
} gvl_fixed_job;
/* batch prep + variant plan (+ track plan and tile prep) of `n` queries; sub_batch as in gvl_dev_batch_prep. */
int gvl_dev_fixed_plan(gvl_ctx *ctx, const gvl_fixed_job *job, const int64_t *ds_idx, const int32_t *jitter, int64_t n,
                       int64_t sub_batch, gvl_stream stream);
/* the bandwidth-bound launches of the batch planned last on `ctx`: seq u8[n*rows_p*L (*4 one-hot)], annot_* i32[n*rows_p*L]
 * (GVL_MODE_ANNOTATED), trk [n*n_tracks*(ploidy|1)*L] elements of job->track_dtype in (b, t, p, L) / (b, t, L) order
 * (binned: L / track_bin per row).
 * Unused outputs NULL. */
int gvl_dev_fixed_exec(gvl_ctx *ctx, const gvl_fixed_job *job, int64_t n, uint8_t *seq, int32_t *annot_v, int32_t *annot_pos,
                       void *trk, gvl_stream stream);
/* One stage of gvl_dev_fixed_plan / _exec, for callers that spread a device call over two streams: the track plan (a chain of
 * small latency-bound kernels) can run next to the bandwidth-bound haplotype execute.  Order: HAP_PLAN (batch prep +
 * haplotype plan) -> { HAP_EXEC, TRK_PLAN (reads the diffs of HAP_PLAN) } -> TRK_EXEC (after TRK_PLAN). */
#define GVL_STAGE_HAP_PLAN 1
#define GVL_STAGE_TRK_PLAN 2
#define GVL_STAGE_HAP_EXEC 3
#define GVL_STAGE_TRK_EXEC 4
int gvl_dev_fixed_stage(gvl_ctx *ctx, const gvl_fixed_job *job, int stage, const int64_t *ds_idx, const int32_t *jitter, int64_t n,
                        int64_t sub_batch, uint8_t *seq, int32_t *annot_v, int32_t *annot_pos, void *trk, gvl_stream stream);
/* The whole of a fixed-length `Dataset.__getitem__` in one call: ds_idx i64[n] / jitter i32[n] (optional) are HOST arrays
 * (pageable is fine, the caller may reuse them at once).  Up to 256 queries they travel BY VALUE with the batch-prep launch
 * (kernel parameter space: no copy, no event); larger batches are staged through a rotating pool of pinned slots owned by the
 * context into idx_dev / jitter_dev (device scratch, n entries), so the host never waits for earlier calls.  Indices are
 * range-checked against the view (GVL_ERR_ARG).  Then gvl_dev_fixed_plan + gvl_dev_fixed_exec on `stream`. */
int gvl_dev_fixed_run(gvl_ctx *ctx, const gvl_fixed_job *job, const int64_t *ds_idx, const int32_t *jitter, int64_t n,
                      int64_t *idx_dev, int32_t *jitter_dev, uint8_t *seq, int32_t *annot_v, int32_t *annot_pos, void *trk,
                      gvl_stream stream);

/* ---- host layer: reference-shaped entries (host pointers in, host pointers out) ------ */
/* Upload (or refresh) a static array and cache it by host address; later gvl_* calls that see
 * the same (ptr, bytes) use the device copy.  The caller must not mutate or free the host array
 * while it is pinned.  Arrays that were NOT pinned are uploaded for the duration of the call
 * (correct, but pays the copy every time).  Replaces the zero-copy memmap crossing that
 * `_ffi_array` guards (python/genvarloader/_dataset/_utils.py:13-35). */
int gvl_pin_static(gvl_ctx *ctx, const void *host_ptr, int64_t bytes);
int gvl_unpin_static(gvl_ctx *ctx, const void *host_ptr);
/* Overlapping intervals.  The reference paints a slot's intervals in stored order, later ones overwriting earlier ones
 * (src/intervals.rs:64-85), so overlaps are legal data (annotation tables are sorted by start, never merged).  The
 * execute kernel paints a run-length code over DISJOINT intervals: gvl_flatten_intervals rewrites every overlapping slot
 * as the equivalent disjoint, sorted list (other slots are copied).  Host arrays; out arrays need room for out_cap
 * intervals (2 * n_itv always suffices; GVL_ERR_CAPACITY with *out_n = the size needed otherwise), out_offsets i64[n_slots+1].
 * The gvl_* host entries do this themselves for the slots a call touches; callers of gvl_dev_* upload flattened tables
 * (`Engine.add_track` does). */
int gvl_intervals_overlap(const int32_t *itv_starts, const int32_t *itv_ends, const int64_t *itv_offsets, int64_t n_slots,
                          int64_t *n_overlapping);
int gvl_flatten_intervals(const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
                          const int64_t *itv_offsets, int64_t n_slots, int32_t *out_starts, int32_t *out_ends,
                          float *out_values, int64_t *out_offsets, int64_t out_cap, int64_t *out_n);
/* Page-locked host memory for per-call inputs/outputs (full PCIe rate on the D2H copies). */
int gvl_host_alloc(int64_t bytes, void **out);
int gvl_host_free(void *p);

/* reconstruct_haplotypes_fused, src/ffi/mod.rs:724-860 (mode U8) -- also serves
 * reconstruct_annotated_haplotypes_fused, src/ffi/mod.rs:2239-2397 (mode ANNOTATED) and the
 * fused one-hot encodings.  Two calls, like every C API that returns a variable-size buffer:
 *   gvl_reconstruct_haplotypes_fused_begin  runs plan, fills out_offsets (host i64[b*p+1]),
 *                                           returns the element count in *total
 *   gvl_reconstruct_haplotypes_fused_finish executes into caller-owned host buffers
 *                                           (out: total bytes, or total*4 for one-hot)
 */
int gvl_reconstruct_haplotypes_fused_begin(
    gvl_ctx *ctx, const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
    int64_t ploidy, const int64_t *geno_offsets /* (2,n_geno) */, int64_t n_geno, const int32_t *geno_v_idxs,
    int64_t n_geno_v, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants, const uint8_t *alt_alleles,
    const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets, int64_t n_contigs,
    int64_t output_length, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
    int64_t *out_offsets, int64_t *total);
int gvl_reconstruct_haplotypes_fused_finish(gvl_ctx *ctx, int mode, uint8_t pad_char, uint8_t *out, int32_t *annot_v,
                                            int32_t *annot_pos);

/* reconstruct_haplotypes_from_svar2, src/ffi/mod.rs:874-893 (sizes rows like the fused SVAR1 entry; finish with
 * gvl_reconstruct_haplotypes_fused_finish).  The reference passes codec keys + the long-allele LUT; this entry
 * takes the DECODED key table (key_ilen, key_alt, key_alt_off) -- see gvl_svar2_channels.  Host pointers. */
int gvl_reconstruct_haplotypes_from_svar2_begin(
    gvl_ctx *ctx, const int32_t *regions, const int32_t *shifts, int64_t batch, int64_t ploidy, const int32_t *vk_pos,
    const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos, const int32_t *dense_key, int64_t n_dense,
    const int32_t *dense_range, const uint8_t *dense_present, const int64_t *dense_present_off, const int32_t *key_ilen,
    const uint8_t *key_alt, const int64_t *key_alt_off, int64_t n_keys, const uint8_t *ref_, const int64_t *ref_offsets,
    int64_t n_contigs, int64_t output_length, const uint8_t *to_rc, int64_t *out_offsets, int64_t *total);

/* hap_diffs_svar2 (see gvl_dev_hap_diffs_svar2), host pointers.  diffs: host i32[batch*ploidy]. */
int gvl_hap_diffs_svar2(gvl_ctx *ctx, const int32_t *regions, int64_t batch, int64_t ploidy, const int32_t *vk_pos,
                        const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos, const int32_t *dense_key,
                        int64_t n_dense, const int32_t *dense_range, const uint8_t *dense_present,
                        const int64_t *dense_present_off, const int32_t *key_ilen, int64_t n_keys, int32_t *diffs);

/* reconstruct_haplotypes_from_sparse, src/ffi/mod.rs:634-655: caller-sized rows, writes `out`
 * (and the optional annotation buffers) in place.  out: host u8[out_offsets[b*p]]. */
int gvl_reconstruct_haplotypes_from_sparse(
    gvl_ctx *ctx, uint8_t *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const int64_t *geno_offsets, int64_t n_geno,
    const int32_t *geno_v_idxs, int64_t n_geno_v, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
    const uint8_t *alt_alleles, const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets,
    int64_t n_contigs, uint8_t pad_char, const uint8_t *keep, const int64_t *keep_offsets, int32_t *annot_v_idxs,
    int32_t *annot_ref_pos);

/* reconstruct_haplotypes_spliced_fused, src/ffi/mod.rs:1983-2071, and (annot_v/annot_pos non-NULL)
 * reconstruct_annotated_haplotypes_spliced_fused, src/ffi/mod.rs:2097-2211: the splice plan's permuted elements are
 * rows of ploidy 1 sized by the caller's out_offsets (i64[n_perm+1], input); masked elements are reverse-complemented
 * (annotation rows reversed).  out: host u8[out_offsets[n_perm]]; annotations host i32 of the same length. */
int gvl_reconstruct_haplotypes_spliced_fused(
    gvl_ctx *ctx, uint8_t *out, int32_t *annot_v, int32_t *annot_pos, const int32_t *permuted_regions,
    const int32_t *flat_shifts, const int64_t *flat_geno_offset_idx, int64_t n_perm, const int64_t *out_offsets,
    const int64_t *geno_offsets, int64_t n_geno, const int32_t *geno_v_idxs, int64_t n_geno_v, const int32_t *v_starts,
    const int32_t *ilens, int64_t n_variants, const uint8_t *alt_alleles, const int64_t *alt_offsets, const uint8_t *ref_,
    const int64_t *ref_offsets, int64_t n_contigs, uint8_t pad_char, const uint8_t *keep, const int64_t *keep_offsets,
    const uint8_t *to_rc);

/* choose_exonic_variants, src/ffi/mod.rs:229-238.  keep: host u8[keep_cap] with keep_cap >= the summed slice sizes
 * (GVL_ERR_CAPACITY otherwise; keep_offsets is valid either way, so a caller may size with keep_cap = 0 first). */
int gvl_choose_exonic_variants(gvl_ctx *ctx, const int32_t *starts, const int32_t *ends, const int64_t *geno_offset_idx,
                               int64_t n_queries, int64_t ploidy, const int32_t *geno_v_idxs, int64_t n_geno_v,
                               const int64_t *geno_offsets, int64_t n_geno, const int32_t *v_starts, const int32_t *ilens,
                               int64_t n_variants, uint8_t *keep, int64_t keep_cap, int64_t *keep_offsets);

/* get_reference, src/ffi/mod.rs:2402-2411.  out: host u8[out_offsets[n_regions]] (x4 for GVL_MODE_ONEHOT). */
int gvl_get_reference(gvl_ctx *ctx, const int32_t *regions, const int64_t *out_offsets, int64_t n_regions,
                      const uint8_t *reference, const int64_t *ref_offsets, int64_t n_contigs, uint8_t pad_char,
                      const uint8_t *to_rc, int mode, uint8_t *out);

/* ragged_to_padded, src/ragged/mod.rs:7-23.  out: host, (n_rows, out_len) items, pre-filled by the caller. */
int gvl_ragged_to_padded(gvl_ctx *ctx, const void *data, const int64_t *offsets, int64_t n_rows, void *out,
                         int64_t itemsize, int64_t out_len);

/* get_diffs_sparse, src/ffi/mod.rs:145-157.  diffs: host i32[n_queries*ploidy]. */
int gvl_get_diffs_sparse(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_queries, int64_t ploidy,
                         const int32_t *geno_v_idxs, int64_t n_geno_v, const int64_t *geno_offsets, int64_t n_geno,
                         const int32_t *ilens, int64_t n_variants, const uint8_t *keep, const int64_t *keep_offsets,
                         const int32_t *q_starts, const int32_t *q_ends, const int32_t *v_starts, int32_t *diffs);

/* intervals_and_realign_track_fused, src/ffi/mod.rs:2553-2672 (one track per call, like the
 * reference's Python loop at _reconstruct.py:228-290).  out: host f32[out_offsets[b*p]]. */
int gvl_intervals_and_realign_track_fused(
    gvl_ctx *ctx, float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const int32_t *geno_v_idxs, int64_t n_geno_v,
    const int64_t *geno_offsets, int64_t n_geno, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
    const int64_t *offset_idxs, const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
    int64_t n_itv, const int64_t *itv_offsets, int64_t n_slots, const int64_t *track_offsets, const double *params,
    int64_t strategy_id, uint64_t base_seed, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc);

/* shift_and_realign_tracks_from_svar2: the core behind src/ffi/mod.rs:1836-1960 (src/tracks/mod.rs:705-856) -- dense f32
 * source windows, svar2 two-channel variant source, decoded key table (key_ilen) instead of the codec's LUT.  Rows are
 * sized by the caller (`out_offsets` is an input, e.g. the offsets gvl_reconstruct_haplotypes_from_svar2_begin returns
 * for output_length = -1, which are hap_diffs_svar2's); `out` is written in place.  query_seed optional (i64[batch]). */
int gvl_shift_and_realign_tracks_from_svar2(
    gvl_ctx *ctx, float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts, int64_t batch,
    int64_t ploidy, const int32_t *vk_pos, const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos,
    const int32_t *dense_key, int64_t n_dense, const int32_t *dense_range, const uint8_t *dense_present,
    const int64_t *dense_present_off, const int32_t *key_ilen, int64_t n_keys, const float *tracks,
    const int64_t *track_offsets, const double *params, int64_t strategy_id, uint64_t base_seed,
    const int64_t *query_seed);

/* shift_and_realign_tracks_sparse, src/ffi/mod.rs:2439-2458 (dense source, writes `out` in place). */
int gvl_shift_and_realign_tracks_sparse(
    gvl_ctx *ctx, float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const int32_t *geno_v_idxs, int64_t n_geno_v,
    const int64_t *geno_offsets, int64_t n_geno, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
    const float *tracks, const int64_t *track_offsets, const double *params, const uint8_t *keep,
    const int64_t *keep_offsets, int64_t strategy_id, uint64_t base_seed);

/* intervals_to_tracks, src/ffi/mod.rs:190-201.  out: host f32[out_offsets[n_queries]]. */
int gvl_intervals_to_tracks(gvl_ctx *ctx, const int64_t *offset_idxs, const int32_t *starts, int64_t n_queries,
                            const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
                            int64_t n_itv, const int64_t *itv_offsets, int64_t n_slots, float *out,
                            const int64_t *out_offsets);

/* _debug_xorshift64 / _debug_hash4, src/ffi/mod.rs:2824-2834 (evaluated on the device). */
int gvl_debug_hash4(gvl_ctx *ctx, uint64_t a, uint64_t b, uint64_t c, uint64_t d, uint64_t *out);
int gvl_debug_xorshift64(gvl_ctx *ctx, uint64_t x, uint64_t *out);
/* Which execute kernel the last gvl_dev_hap_exec of this context launched: 0 byte-oriented, 1 packed one-hot
 * (tests assert that the intended kernel ran). */
int gvl_debug_last_exec_kernel(gvl_ctx *ctx);

/* The launch configuration the last plans and execute of this context chose, recorded on the host when each choice is
 * made (so also while a CUDA graph is being captured).  Fills out[0 .. min(n, GVL_LAUNCH_FIELDS)), in this order:
 *   GVL_LAUNCH_PLAN_THREADS      threads per row of the last haplotype plan (32, 256 or 512)
 *   GVL_LAUNCH_PLAN_STATIC       1 if that plan used static record slices (a bounded list length per row), else 0
 *   GVL_LAUNCH_EXEC_KERNEL       the last gvl_dev_hap_exec's kernel: one of GVL_EXEC_*
 *   GVL_LAUNCH_TILE_LEN          its output positions per tile
 *   GVL_LAUNCH_TILES_PER_ROW     its tiles per row (0 for ragged plans)
 *   GVL_LAUNCH_REC_BOUND         the record bound per row it chose from (after the typical-slot-length clamp)
 *   GVL_LAUNCH_TRK_PLAN_THREADS  threads per row of the last track plan (32, 256 or 512)
 *   GVL_LAUNCH_TRK_PLAN_STATIC   1 if that track plan used static record slices, else 0
 * Values of a step that has not run yet on this context are 0.  A gvl_dev_hap_exec that has nothing to launch (no rows,
 * no output positions, no tiles) returns before the choice and leaves the previous call's values in place.  Tests use it
 * to assert which configuration they reach. */
#define GVL_LAUNCH_PLAN_THREADS 0
#define GVL_LAUNCH_PLAN_STATIC 1
#define GVL_LAUNCH_EXEC_KERNEL 2
#define GVL_LAUNCH_TILE_LEN 3
#define GVL_LAUNCH_TILES_PER_ROW 4
#define GVL_LAUNCH_REC_BOUND 5
#define GVL_LAUNCH_TRK_PLAN_THREADS 6
#define GVL_LAUNCH_TRK_PLAN_STATIC 7
#define GVL_LAUNCH_FIELDS 8
#define GVL_EXEC_BYTES 0          /* byte-oriented kernel (bytes, annotated, channels-first, one-hot without a packed reference) */
#define GVL_EXEC_PACKED_2WARP 1   /* packed one-hot, 2-warp CTAs: one tile of <= 8,192 positions per row                  */
#define GVL_EXEC_PACKED_UNROLL4 2 /* packed one-hot, 4 groups per warp in flight: long sparse rows, ragged plans          */
#define GVL_EXEC_PACKED_UNROLL2 3 /* packed one-hot, 2 groups per warp in flight: everything else                         */
int gvl_debug_last_launch(gvl_ctx *ctx, int64_t *out, int n);

/* The tile descriptors of the last track execute this context prepared (every entry that realigns or paints tracks).
 * Synchronizes the device, then copies the descriptors back.  *n_tiles = descriptors of that call's grid (tiles per
 * track, an upper bound, times the tracks); *tdesc_bytes = bytes allocated for descriptors (at least *n_tiles times the
 * descriptor size).  out: int32[7 * n_max]; entry k = (track, row, h0, h1, flags, m, cnt) of the k-th tile that exists,
 * in grid order, where [h0, h1) is the tile in haplotype coordinates, flags a mask of GVL_TILE_*, m the records the tile
 * stages (its carry included) and cnt the stored intervals it needs; entries past the last tile are -1.  n_max = 0 only
 * reports the two counts.  Tests use it to assert which execute path every tile takes. */
#define GVL_TILE_RC 1       /* the row is written reversed (negative strand)                                          */
#define GVL_TILE_GENERIC 2  /* every value resolved on its own: unsorted variant list or dense source                  */
#define GVL_TILE_BIG 4      /* more records or stored intervals than one pass stages: finished in sub-passes           */
int gvl_debug_track_tiles(gvl_ctx *ctx, int32_t *out, int64_t n_max, int64_t *n_tiles, int64_t *tdesc_bytes);

/* ====================================================================================
 * `variants` / `variant-windows` outputs (SURVEY.md section 8 f4): the variants of every (region, sample, ploid) row
 * themselves -- indices, positions, indel lengths, allele byte strings, flank / window tokens -- instead of the
 * reconstructed haplotype.  Reference: src/variants/mod.rs, src/variants/windows.rs; callers
 * python/genvarloader/_dataset/_flat_variants.py:869-1112 (get_variants_flat), _rag_variants.py:300-325.
 * Every entry is "lengths -> exclusive scan -> ragged copy": an `_offsets` call writes the (n + 1) offsets on the device,
 * the caller reads offsets[n] (its one synchronisation, as for every ragged output), allocates, and calls the fill.
 * 4-byte items (i32 variant indices / positions, f32 dosages) move as raw 32-bit words: bit-exact for floats.
 * ==================================================================================== */
#define GVL_WINDOW_REF 0    /* tokens of the reference window [start - L, end + L), end = start - min(ilen, 0) + 1 */
#define GVL_WINDOW_ALT 1    /* tokens of flank5 . ALT . flank3                                                     */
#define GVL_WINDOW_FLANKS 2 /* tokens of [flank5 | flank3], 2 L per variant (the `flank_tokens` field)             */

/* gather_rows_{i32,f32}, src/ffi/mod.rs:255-288 -> src/variants/mod.rs:6-49: row i = data[o_starts[g] .. o_stops[g]) with
 * g = geno_offset_idx[i].  out_offsets i64[n_rows + 1]. */
int gvl_dev_gather_rows_offsets(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_rows, const int64_t *o_starts,
                                const int64_t *o_stops, int64_t *out_offsets, gvl_stream stream);
int gvl_dev_gather_rows(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_rows, const int64_t *o_starts, const void *data,
                        const int64_t *out_offsets, int64_t total, void *out, gvl_stream stream);
/* gvl_dev_gather_rows over the genotype CSR of `tab` with the positions and indel lengths of the gathered variants taken in
 * the same pass: v_idxs[e] = geno_v_idxs[...], starts[e] = v_starts[v_idxs[e]], ilens[e] = ilens[v_idxs[e]] (starts / ilens
 * may be NULL).  One launch for the three fields every `variants` read asks for. */
int gvl_dev_gather_variant_rows(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int64_t *geno_offset_idx, int64_t n_rows,
                                const int64_t *out_offsets, int64_t total, int32_t *v_idxs, int32_t *starts, int32_t *ilens,
                                gvl_stream stream);
/* table[v_idxs[i]] for a 4-byte table: start / ilen / info fields of the gathered variants (_flat_variants.py:948-953). */
int gvl_dev_take_u32(gvl_ctx *ctx, const void *table, const int32_t *v_idxs, int64_t n, void *out, gvl_stream stream);

/* np.repeat(values, np.diff(offsets)) for 4-byte values: e.g. the contig of every gathered variant from the contig of its
 * row (_flat_variants.py:985-989), which gvl_dev_variant_windows takes as v_contigs. */
int gvl_dev_expand_rows_u32(gvl_ctx *ctx, const void *values, const int64_t *offsets, int64_t n_rows, int64_t total, void *out,
                            gvl_stream stream);

/* gather_alleles, src/ffi/mod.rs:291-304 -> src/variants/mod.rs:52-78.  seq_offsets i64[n + 1].  With lut != NULL the
 * bytes are tokenised on the way out (windows.rs:9-22): out[e] = lut[byte], lut = 256 tokens of tok_bytes (1 or 4). */
int gvl_dev_gather_alleles_offsets(gvl_ctx *ctx, const int32_t *v_idxs, int64_t n, const int64_t *allele_offsets,
                                   int64_t *seq_offsets, gvl_stream stream);
int gvl_dev_gather_alleles(gvl_ctx *ctx, const int32_t *v_idxs, int64_t n, const uint8_t *allele_bytes,
                           const int64_t *allele_offsets, const int64_t *seq_offsets, int64_t total, const void *lut,
                           int tok_bytes, void *out, gvl_stream stream);

/* rc_alleles, src/ffi/mod.rs:2808 -> src/variants/mod.rs:90-108: reverse-complement, in place, every allele of the
 * (b*p) rows with to_rc_row != 0 (src/reverse.rs:45-53).  seq_offsets i64[n_alleles + 1] (seq_offsets[0] = 0),
 * var_offsets i64[n_rows + 1], total_bytes = seq_offsets[n_alleles]. */
int gvl_dev_rc_alleles(gvl_ctx *ctx, uint8_t *byte_data, const int64_t *seq_offsets, int64_t n_alleles,
                       const int64_t *var_offsets, int64_t n_rows, const uint8_t *to_rc_row, int64_t total_bytes,
                       gvl_stream stream);

/* compact_keep_{i32,f32}, src/ffi/mod.rs:308-333 -> src/variants/mod.rs:112-153.  pos i64[n + 1] is caller scratch that
 * receives the exclusive scan of keep (pos[n] = values kept); new_offsets i64[n_rows + 1]. */
int gvl_dev_compact_keep_offsets(gvl_ctx *ctx, const uint8_t *keep, int64_t n, const int64_t *row_offsets, int64_t n_rows,
                                 int64_t *pos, int64_t *new_offsets, gvl_stream stream);
int gvl_dev_compact_keep(gvl_ctx *ctx, const void *values, const uint8_t *keep, int64_t n, const int64_t *pos, void *out,
                         gvl_stream stream);

/* fill_empty_{scalar,fixed}_{i32,f32}, src/ffi/mod.rs:336-388 -> src/variants/mod.rs:157-256: every empty row receives one
 * dummy variant of `inner` items equal to fill_bits (scalar: inner = 1).  new_offsets i64[n_rows + 1] count variants;
 * new_total = new_offsets[n_rows]; out holds new_total * inner items. */
int gvl_dev_fill_empty_offsets(gvl_ctx *ctx, const int64_t *offsets, int64_t n_rows, int64_t *new_offsets, gvl_stream stream);
int gvl_dev_fill_empty_fixed(gvl_ctx *ctx, const void *data, const int64_t *offsets, int64_t n_rows, const int64_t *new_offsets,
                             int64_t new_total, int64_t inner, uint32_t fill_bits, void *out, gvl_stream stream);

/* fill_empty_seq_{u8,i32}, src/ffi/mod.rs:391-445 -> src/variants/mod.rs:259-329: two-level ragged (rows -> variants ->
 * items); every empty row receives one dummy sequence.  new_var_offsets comes from gvl_dev_fill_empty_offsets
 * (n_new_vars = new_var_offsets[n_rows]); src_var i64[n_new_vars] is caller scratch (source variant of every new variant,
 * -1 = dummy); new_seq_offsets i64[n_new_vars + 1]; total = new_seq_offsets[n_new_vars]. */
int gvl_dev_fill_empty_seq_offsets(gvl_ctx *ctx, const int64_t *var_offsets, int64_t n_rows, const int64_t *seq_offsets,
                                   int64_t dummy_len, const int64_t *new_var_offsets, int64_t n_new_vars, int64_t *src_var,
                                   int64_t *new_seq_offsets, gvl_stream stream);
int gvl_dev_fill_empty_seq(gvl_ctx *ctx, const void *data, int itemsize, const int64_t *seq_offsets, const void *dummy,
                           const int64_t *src_var, const int64_t *new_seq_offsets, int64_t n_new_vars, int64_t total, void *out,
                           gvl_stream stream);

/* Flank / window tokens, src/variants/windows.rs:27-134, 196-214, 262-291 (fetch_windows + slice_flanks +
 * assemble_alt_window + tokenize in one pass; the intermediate window bytes are never materialised).  Reads
 * tab->{v_starts, ilens, alt_alleles, alt_offsets, ref, ref_offsets}; v_contigs i32[n] = contig of every selected variant
 * (NULL: contig 0); positions outside the contig read as pad_char; lut = 256 tokens of tok_bytes (1 or 4).
 * GVL_WINDOW_FLANKS needs no offsets (2 * flank_len tokens per variant). */
int gvl_dev_variant_windows_offsets(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *v_idxs, int64_t n,
                                    int64_t flank_len, int kind, int64_t *win_offsets, gvl_stream stream);
int gvl_dev_variant_windows(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *v_idxs, const int32_t *v_contigs,
                            int64_t n, int64_t flank_len, int kind, uint8_t pad_char, const void *lut, int tok_bytes,
                            const int64_t *win_offsets, int64_t total, void *out, gvl_stream stream);

/* Every buffer length of a variants read, from four sums per genotype row r (slot g = geno_offset_idx[r], the variants
 * geno_v_idxs[geno_starts[g] .. geno_stops[g]) of the row, those with keep_table[v] == 0 left out; keep_table = per-variant
 * int32 AF flags, NULL keeps every variant): out_sizes i64[n_rows * 4], row r = (variants kept, sum of their ALT lengths,
 * sum of their REF lengths from ref_offsets (0 when NULL), sum of their reference spans 1 - min(ilen, 0)).  One warp per
 * row, no atomics: reproducible, and safe to capture in a graph. */
int gvl_dev_variant_row_sizes(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int64_t *geno_offset_idx, int64_t n_rows,
                              const int32_t *keep_table, const int64_t *ref_offsets, int64_t *out_sizes, gvl_stream stream);
/* Batch-local offsets of K consecutive batches read as one call.  offsets i64[n + 1] run over the items of the whole ring;
 * batch i owns items [s_i, s_{i+1}) with s_i = min(i * stride, n) when bounds is NULL, else s_i = bounds[min(i * stride,
 * n_bounds)] (bounds i64[n_bounds + 1], e.g. the ring's row offsets: a batch's rows turned into its variants).  s_0 must be
 * 0 and s_K must be n.  Writes offsets[s_i .. s_{i+1}] - offsets[s_i] to out[s_i + i .. s_{i+1} + i]: out i64[n + K], every
 * batch's offsets starting at 0, one launch for all K batches. */
int gvl_dev_rebase_offsets(gvl_ctx *ctx, const int64_t *offsets, int64_t n, const int64_t *bounds, int64_t n_bounds,
                           int64_t stride, int64_t n_batches, int64_t *out, gvl_stream stream);

/* ---- host layer of the same entries: the reference's #[pyfunction] argument lists, host pointers in.  The reference
 * returns arrays it allocates; here a call leaves its results on the device, reports their sizes, and the caller copies
 * each one out with gvl_variants_fetch(which) into a buffer of exactly that size (results stay valid until the next
 * host-layer variants call on the context).  Offsets that size other results are also written straight to host. */
int gvl_variants_fetch(gvl_ctx *ctx, int which, void *host_out, int64_t bytes);
/* result 0: data (4 * total bytes).  geno_offsets is the (2, n_geno) starts / stops array. */
int gvl_gather_rows(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_rows, const int64_t *geno_offsets, int64_t n_geno,
                    const void *data, int64_t n_data, int64_t *out_offsets, int64_t *total);
/* result 0: bytes (total). */
int gvl_gather_alleles(gvl_ctx *ctx, const int32_t *v_idxs, int64_t n, const uint8_t *allele_bytes, int64_t n_bytes,
                       const int64_t *allele_offsets, int64_t n_table, int64_t *seq_offsets, int64_t *total);
/* in place on the caller's host buffer. */
int gvl_rc_alleles(gvl_ctx *ctx, uint8_t *byte_data, int64_t n_bytes, const int64_t *seq_offsets, int64_t n_alleles,
                   const int64_t *var_offsets, int64_t n_rows, const uint8_t *to_rc_row);
/* result 0: kept values (4 * total bytes). */
int gvl_compact_keep(gvl_ctx *ctx, const void *values, int64_t n, const int64_t *row_offsets, int64_t n_rows,
                     const uint8_t *keep, int64_t *new_offsets, int64_t *total);
/* result 0: data (4 * new_total * inner bytes); fill_empty_scalar = inner 1. */
int gvl_fill_empty_fixed(gvl_ctx *ctx, const void *data, int64_t n_data, const int64_t *offsets, int64_t n_rows, int64_t inner,
                         uint32_t fill_bits, int64_t *new_offsets, int64_t *new_total);
/* result 0: data (itemsize * total bytes), result 1: new_seq_offsets (8 * (n_new_vars + 1) bytes). */
int gvl_fill_empty_seq(gvl_ctx *ctx, const void *data, int itemsize, int64_t n_data, const int64_t *var_offsets, int64_t n_rows,
                       const int64_t *seq_offsets, int64_t n_vars, const void *dummy, int64_t dummy_len,
                       int64_t *new_var_offsets, int64_t *n_new_vars, int64_t *total);
/* assemble_variant_buffers_{u8,i32}, src/ffi/mod.rs:460-630.  Up to three fields come back in the reference's order:
 * field_kind[j] in {0 alt, 1 ref, 2 flank_tokens, 3 ref_window, 4 alt_window}, field_items[j] = items of its data,
 * field_tok[j] = bytes per item; data = result 2 j, seq offsets = result 2 j + 1 (i64[n + 1]; flank_tokens has none: its
 * offsets are the caller's row_offsets).  lut may be NULL when no tokens are requested. */
int gvl_assemble_variant_buffers(gvl_ctx *ctx, int64_t mode, const int32_t *v_idxs, int64_t n, const uint8_t *alt_global,
                                 const int64_t *alt_off_global, const uint8_t *ref_global, const int64_t *ref_off_global,
                                 int64_t n_variants, int want_ref_bytes, int want_flank, int64_t ref_mode, int64_t alt_mode,
                                 int64_t flank_len, const void *lut, int tok_bytes, const int32_t *v_contigs,
                                 const int32_t *v_starts, const int32_t *ilens, const uint8_t *reference,
                                 const int64_t *ref_offsets, int64_t n_contigs, uint8_t pad_char, int32_t *n_fields,
                                 int32_t *field_kind, int64_t *field_items, int32_t *field_tok);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* GVL_B200_H */
