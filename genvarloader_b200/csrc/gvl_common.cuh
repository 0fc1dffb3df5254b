// gvl_common.cuh -- shared declarations of the B200 haplotype path (device structs, ctx).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/gvl_b200.h"
#include "gvl_plan.cuh"

namespace gvl {

// Per-(query, hap) row header written by the plan kernels and read by the execute kernels.
struct __align__(16) RowPlan {
    int64_t out_off;     // first element of this row in the flat output
    int64_t ref_base;    // ref_offsets[contig]                       (haps)   | slot base of intervals (tracks)
    int64_t rec_off;     // first record of this row in the record arrays
    int32_t length;      // output positions in this row
    int32_t contig_len;  // contig length (haps) | source window length (tracks)
    int32_t lead_pad;    // leading pad positions, clamped to length (haps)
    int32_t ref0;        // reference/track position feeding the first span
    int32_t n_rec;       // records of this row
    int32_t rc;          // reverse(-complement) this row
    int32_t diff;        // get_diffs_sparse value of the row
    int32_t q_start;     // regions[q,1]
};

// Record arrays (SoA).  Haplotypes use a, n, src, resume, vidx, vpos; tracks reuse
// a, n, resume, vpos (= v_rel_pos), vidx (= v_len handed to the fill) and src (= ilen).
struct RecArrays {
    int32_t *a;
    int32_t *n;
    int64_t *src;
    int32_t *resume;
    int32_t *vidx;
    int32_t *vpos;
};

// One record of a TRACK row (32 bytes, AoS so that a tile's records are one contiguous read): the variant writes
// output positions [a, e) -- DEL: track[vrel] once; INS: e - a of vlen fill values -- and the source resumes at `resume`
// (positions relative to the query start).
struct __align__(16) TRec {
    int32_t a;       // output (haplotype) position of the variant's values
    int32_t e;       // a + values written (writable_length, src/tracks/mod.rs:329)
    int32_t resume;  // source position after the variant (v_rel_end, :267)
    int32_t vrel;    // v_rel_pos (:264)
    int32_t vlen;    // (possibly shift-trimmed) v_len handed to the fill (:306, :338)
    int32_t vdiff;   // ilen
    int32_t pad0, pad1;
};
static_assert(sizeof(TRec) == 32, "TRec is a 32-byte record");
constexpr int FLAG_JUMPS = 1;  // RowPlan.lead_pad of a track row: the row has jump records (unsorted variant list)

// Optional per-call MERGED variant lists: the svar2 two-channel source (var_key + dense/presence,
// src/svar2/mod.rs:45-66) after the device merge.  Row k's list is key/pos[off[k] .. off[k]+len[k]); keys
// index the decoded-key table that is passed as gvl_sparse_tables.ilens / alt_offsets / alt_alleles.
struct MergedLists {
    const int32_t *pos;
    const int32_t *key;
    const int64_t *off;
    const int32_t *len;
};

// Device status words (ctx->dev_words).
enum { W_CURSOR = 0, W_STATUS = 1, W_TOTAL = 2, W_TILES = 3, W_MERGE_CURSOR = 4, W_DONE = 5, W_COUNT = 8 };

constexpr int EXEC_THREADS = 128;
constexpr int EXEC_MIN_CTAS = 12;        // resident CTAs per SM the execute kernels are compiled for (<= 40 registers)
constexpr int EXEC_UNIT = EXEC_THREADS * 4;  // positions covered by one CTA-wide step (4 per thread)
constexpr int TILE = 4096;       // haplotype positions per execute CTA for ragged plans (fixed plans pick theirs)
constexpr int REC_CAP = 128;     // records staged in shared memory per pass
constexpr int EXEC_MAX_UNITS = 16;  // haplotype positions per CTA of the byte kernel, in units of 512
constexpr int DIR_Q = 1024;      // haplotype positions per directory entry (execute tiles are multiples of it)
constexpr int64_t ALT_PAD = INT64_MIN;  // RecArrays.src sentinel: "ALT piece" is padding (leading pad)

}  // namespace gvl

#define GVL_TRK_DESC_BYTES 4096
// bytes of one tile descriptor of the track execute (gvl_tracks_exec.cuh: TileDesc, which static_asserts this size)
#define GVL_TILE_DESC_BYTES 112

struct gvl_static_entry {
    void *dev;
    int64_t bytes;
};

// Plan workspace: row headers + record arrays + tile map.  One for haplotypes, one for tracks, so a
// track plan never invalidates a haplotype plan that has not been executed yet.
struct gvl_workspace {
    gvl::RowPlan *rows;
    int64_t rows_cap;
    gvl::RecArrays rec;
    int64_t rec_cap;
    int64_t *tile_off;  // i64[rows_cap+1] (ragged plans)
    int32_t *row_len;   // i32[rows_cap]
    // svar2 merge output
    int32_t *m_pos, *m_key;
    int64_t m_cap;
    int64_t *m_off;     // i64[rows_cap]
    int32_t *m_len;     // i32[rows_cap]
    // fixed-length plans: per-row checkpoint directory, dir[row * stride + q] = records with a < q * DIR_Q
    int32_t *dir;
    int64_t dir_cap;
    // track plans: 32-byte AoS records (gvl_tracks.cu: TrkRec)
    void *trecs;
    int64_t trec_cap;
    void *tdesc;        // per (track, tile) descriptors of the track execute kernel (GVL_TILE_DESC_BYTES each)
    int64_t tdesc_cap;  // descriptors it holds
    int64_t tdesc_bytes;  // bytes allocated (checked against every tile-prep launch)
};

struct gvl_ctx {
    int device;
    cudaStream_t own_stream;  // used by the host layer
    gvl_workspace hap, trk;
    void *trk_desc;       // device buffer for per-track descriptors (GVL_TRK_DESC_BYTES)
    int64_t *dev_words;   // 2 * W_COUNT words (haps, tracks)
    int64_t *host_words;  // pinned mirror
    // current haplotype plan
    bool plan_valid;
    int64_t n_work;
    int64_t fixed_len;  // >=0 fixed, -1 ragged
    int64_t row_stride_hint = 0;    // set around a plan by callers that bound the variant-list length per row (gvl_batch.cu)
    int64_t rec_bound_per_row = 0;  // the plan's record bound / rows (tile length of the one-hot kernel)
    int64_t dir_stride; // directory entries per row of the current plan (0 = no directory)
    int64_t total;      // -1 = unknown (ragged before sync)
    int64_t *plan_out_offsets;  // device pointer supplied at plan time
    int last_exec_kernel;       // 0 byte-oriented, 1 packed one-hot (gvl_debug_last_exec_kernel)
    int64_t last_launch[GVL_LAUNCH_FIELDS] = {};  // launch choices of the last plans / execute (gvl_debug_last_launch)
    void *trk_params;           // parameters of the pending track execute launch (gvl_tracks.cu)
    bool trk_plan_valid;
    // gvl_dev_fixed_run: rotating pinned staging slots for the per-call index upload (gvl_batch.cu)
    struct StageSlot {
        void *host = nullptr;
        int64_t bytes = 0;
        cudaEvent_t ev = nullptr;
        bool used = false;
    } stage[8];
    int stage_k = 0;
    void *zeros;                // device zeros (gvl_aux.cu: rows without genotypes)
    int64_t zeros_bytes;
    void *var_scratch = nullptr;    // block sums of the offset scans (gvl_variants.cu)
    int64_t var_scratch_bytes = 0;
    int64_t *itv_counts = nullptr;  // per-row interval counts of gvl_dev_track_intervals (gvl_tracks.cu)
    int64_t itv_counts_cap = 0;
    void *ritv_ws = nullptr;        // item table, counts and offsets of gvl_dev_realigned_track_intervals (gvl_tracks.cu)
    int64_t ritv_ws_bytes = 0;
    int64_t ritv_pairs = -1;        // (track, row) pairs and item slots of its last sizing call (-1: none yet)
    int64_t ritv_item_cap = 0;
    std::vector<std::pair<void *, int64_t>> var_results;  // device results of the last host-layer variants entry (gvl_variants_fetch)
    // host layer
    std::map<const void *, gvl_static_entry> statics;
    std::map<const void *, void *> packed_refs;  // device ASCII reference (pinned static) -> its packed copy
    std::vector<std::pair<void *, int64_t>> scratch;  // per-call device scratch (name-less pool)
    void *pinned;
    int64_t pinned_bytes;
    gvl_sparse_tables host_tab;  // device pointers resolved by the last host-layer plan
    int64_t *host_out_offsets_dev;
};
