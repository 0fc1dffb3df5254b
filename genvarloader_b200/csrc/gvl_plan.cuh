// gvl_plan.cuh -- the per-(query, hap) variant state machines as small step functions.
//
// The reference walks each haplotype's variant list with a sequential state machine
// (src/reconstruct/mod.rs:39-256 for bytes, src/tracks/mod.rs:224-406 for tracks,
// src/genotypes/mod.rs:15-125 for the length diff).  Here the same state machines are
// expressed as `init / step / finish` functions over plain integers so that the serial device
// plan routines (rows with unsorted lists) can drive them in lock-step across a warp,
// one variant per step with operands broadcast by shuffles, emitting a compact segment table
// instead of copying bytes.  (The scan-based kernel of gvl_plan_par.cuh restates the same rules
// as block-wide scans.)
// The execute kernels never see variants -- only the records emitted here.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GVL_HD __host__ __device__ __forceinline__
#else
#define GVL_HD inline
#endif

namespace gvl {

GVL_HD int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }
GVL_HD int64_t imax64(int64_t a, int64_t b) { return a > b ? a : b; }

enum { STEP_SKIP = 0, STEP_EMIT = 1, STEP_BREAK = 2 };

// ------------------------------------------------------------------------------------
// Haplotype bytes: reconstruct_haplotype_core, src/reconstruct/mod.rs:39-256.
//
// Output of a row = [lead_pad x pad] then, for each emitted record r (in order),
//   reference bytes  ref[prev_resume .. )  up to output position a_r,
//   ALT bytes        alt[src_r + trim_r .. +n_r)  at output positions [a_r, a_r + n_r),
// then reference bytes from resume_last (pad once the contig is exhausted).  `prev_resume`
// of the first record is `ref0`.
// ------------------------------------------------------------------------------------
struct HapState {
    int64_t ref_start, shift, length;
    int64_t ref_idx, out_idx, shifted;
    int64_t lead_pad;
};

struct HapRec {
    int64_t a;         // output position where the ALT bytes start        (out_idx after the ref span)
    int64_t n;         // ALT bytes written (writable_length)
    int64_t trim;      // ALT bytes consumed by the shift (allele_start_idx)
    int64_t resume;    // reference position after the variant (v_ref_end)
    int64_t span_src;  // reference position where the preceding ref span starts (ref_idx at copy time)
};

GVL_HD void hap_init(HapState &s, int64_t ref_start, int64_t shift, int64_t length) {
    s.ref_start = ref_start;
    s.shift = shift;
    s.length = length;
    s.ref_idx = ref_start;  // :61
    s.out_idx = 0;          // :63
    s.shifted = 0;          // :65
    s.lead_pad = 0;
    if (s.ref_idx < 0) {  // :68-83
        int64_t pad_len_raw = -s.ref_idx;
        s.shifted = imin64(shift, pad_len_raw);
        int64_t pad_len = pad_len_raw - s.shifted;
        s.lead_pad = pad_len;
        s.out_idx += pad_len;
        s.ref_idx = 0;
    }
}

// One kept variant (the caller applies the keep mask, :86-90).
GVL_HD int hap_step(HapState &s, int64_t v_pos, int64_t v_diff, int64_t v_len_full, HapRec &rec) {
    int64_t v_ref_end = v_pos - imin64(0, v_diff) + 1;  // :96
    if (v_pos < s.ref_start && v_diff < 0 && v_ref_end >= s.ref_start) {  // :99-102
        s.ref_idx = v_ref_end;
        return STEP_SKIP;
    }
    if (v_pos < s.ref_idx) return STEP_SKIP;  // :108-110
    int64_t allele_start_idx = 0;             // :114
    if (s.shifted < s.shift) {                // :115-146
        int64_t ref_shift_dist = v_pos - s.ref_idx;
        if (s.shifted + ref_shift_dist + v_len_full < s.shift) {
            return STEP_SKIP;  // :118-121 (ref_idx NOT advanced)
        } else if (s.shifted + ref_shift_dist >= s.shift) {
            s.ref_idx += s.shift - s.shifted;  // :123-128
            s.shifted = s.shift;
        } else {
            allele_start_idx = s.shift - s.shifted - ref_shift_dist;  // :132
            s.shifted = s.shift;
            if (allele_start_idx == v_len_full) {  // :135-140
                s.ref_idx = v_ref_end;
                return STEP_SKIP;
            }
            s.ref_idx = v_pos;  // :143
        }
    }
    int64_t v_len = v_len_full - allele_start_idx;             // :149-150
    int64_t ref_len = v_pos - s.ref_idx;                       // :153
    if (s.out_idx + ref_len >= s.length) return STEP_BREAK;    // :154-158
    rec.span_src = s.ref_idx;
    s.out_idx += ref_len;                                      // :175
    int64_t writable_length = imin64(v_len, s.length - s.out_idx);  // :178
    rec.a = s.out_idx;
    rec.n = writable_length;
    rec.trim = allele_start_idx;
    rec.resume = v_ref_end;
    s.out_idx += writable_length;  // :190
    s.ref_idx = v_ref_end;         // :193
    return STEP_EMIT;              // caller breaks when out_idx >= length (:195-197)
}

GVL_HD void hap_finish(HapState &s, int64_t contig_len) {  // :200-205
    if (s.shifted < s.shift) {
        s.ref_idx += s.shift - s.shifted;
        s.ref_idx = imin64(s.ref_idx, contig_len);
        s.shifted = s.shift;
    }
}

// ------------------------------------------------------------------------------------
// Length diff: get_diffs_sparse, src/genotypes/mod.rs:48-86 (query-clipped branch) --
// also hap_diffs_svar2, src/svar2/mod.rs:116-143.
// ------------------------------------------------------------------------------------
struct DiffState {
    int64_t q_start, q_end, ref_idx, acc;
};

GVL_HD void diff_init(DiffState &d, int64_t q_start, int64_t q_end) {
    d.q_start = q_start;
    d.q_end = q_end;
    d.ref_idx = q_start;
    d.acc = 0;
}

// returns false when the reference loop `break`s
GVL_HD bool diff_step(DiffState &d, int64_t v_start, int64_t v_ilen) {
    int64_t v_end = v_start - imin64(v_ilen, 0) + 1;
    if (v_end <= d.q_start) return true;                           // :69-71
    if (v_start >= d.q_end) return false;                          // :72-74
    if (v_start >= d.q_start && v_start < d.ref_idx) return true;  // :75-77
    d.ref_idx = imax64(d.ref_idx, v_end);                          // :78
    if (v_ilen < 0) v_ilen += imax64(d.q_start - v_start - 1, 0);  // :79-81
    v_ilen += imax64(v_end - d.q_end, 0);                          // :82
    d.acc += v_ilen;
    return true;
}

// ------------------------------------------------------------------------------------
// Tracks: shift_and_realign_track_core, src/tracks/mod.rs:224-406.
//
// Output of a row = for each emitted record r: source values track[prev_resume ..) up to
// output position a_r, then n_r values produced by the variant (DEL: track[v_rel_pos] once;
// INS: the insertion fill over v_len values, of which n_r are written), then source values
// from resume_last, 0.0 once the source window is exhausted.  prev_resume of the first
// record is `track0`.
// ------------------------------------------------------------------------------------
struct TrkState {
    int64_t shift, length;
    int64_t track_idx, out_idx, shifted;
};

struct TrkRec {
    int64_t a;          // output position of the variant's values
    int64_t n;          // values written (writable_length)
    int64_t v_len;      // (possibly shift-trimmed) v_len handed to the fill (:306, :338)
    int64_t v_rel_pos;  // variant position relative to the query start
    int64_t v_diff;     // ilen
    int64_t resume;     // v_rel_end
    int64_t span_src;   // track_idx at copy time
};

GVL_HD void trk_init(TrkState &s, int64_t shift, int64_t length) {
    s.shift = shift;
    s.length = length;
    s.track_idx = 0;  // :249-251
    s.out_idx = 0;
    s.shifted = 0;
}

GVL_HD int trk_step(TrkState &s, int64_t v_rel_pos, int64_t v_diff, TrkRec &rec) {
    int64_t v_rel_end = v_rel_pos - imin64(v_diff, 0) + 1;  // :267
    if (v_diff < 0 && v_rel_pos < 0 && v_rel_end >= 0) {     // :271-274
        s.track_idx = v_rel_end;
        return STEP_SKIP;
    }
    if (v_rel_pos < s.track_idx) return STEP_SKIP;  // :277-279
    int64_t v_len = imax64(v_diff, 0) + 1;           // :282
    if (s.shifted < s.shift) {                       // :285-308
        int64_t ref_shift_dist = v_rel_pos - s.track_idx;
        if (s.shifted + ref_shift_dist + v_len < s.shift) {
            return STEP_SKIP;
        } else if (s.shifted + ref_shift_dist >= s.shift) {
            s.track_idx += s.shift - s.shifted;
            s.shifted = s.shift;
        } else {
            int64_t allele_start_idx = s.shift - s.shifted - ref_shift_dist;
            s.shifted = s.shift;
            if (allele_start_idx == v_len) {
                s.track_idx = v_rel_end;
                return STEP_SKIP;
            }
            s.track_idx = v_rel_pos;
            v_len -= allele_start_idx;
        }
    }
    if (v_diff == 0) return STEP_SKIP;  // :312-314 SNPs write nothing
    int64_t track_len = v_rel_pos - s.track_idx;               // :317
    if (s.out_idx + track_len >= s.length) return STEP_BREAK;  // :319-321
    rec.span_src = s.track_idx;
    s.out_idx += track_len;
    int64_t writable_length = imin64(v_len, s.length - s.out_idx);  // :329
    rec.a = s.out_idx;
    rec.n = writable_length;
    rec.v_len = v_len;
    rec.v_rel_pos = v_rel_pos;
    rec.v_diff = v_diff;
    rec.resume = v_rel_end;
    s.out_idx += writable_length;
    s.track_idx = v_rel_end;  // :356
    return STEP_EMIT;
}

GVL_HD void trk_finish(TrkState &s, int64_t track_n) {  // :365-369
    if (s.shifted < s.shift) {
        s.track_idx += s.shift - s.shifted;
        s.track_idx = imin64(s.track_idx, track_n);
    }
}

// ------------------------------------------------------------------------------------
// PRNG, src/tracks/mod.rs:31-54.
// ------------------------------------------------------------------------------------
GVL_HD uint64_t xorshift64(uint64_t x) {
    x ^= x << 13;
    x ^= x >> 7;
    x ^= x << 17;
    return x;
}

GVL_HD uint64_t hash4(uint64_t a, uint64_t b, uint64_t c, uint64_t d) {
    uint64_t h = a;
    h = xorshift64(h ^ b);
    h = xorshift64(h ^ c);
    h = xorshift64(h ^ d);
    return h;
}

}  // namespace gvl
