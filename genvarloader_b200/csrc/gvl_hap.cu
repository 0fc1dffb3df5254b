// gvl_hap.cu -- haplotype reconstruction on sm_100a: plan + execute kernels and their
// device-pointer C entries (include/gvl_b200.h: gvl_dev_hap_plan / _total / _exec,
// gvl_dev_get_diffs_sparse).
//
// Reference path replaced: src/ffi/mod.rs:724-860 (reconstruct_haplotypes_fused) and
// :2239-2397 (annotated) = get_diffs_sparse -> prefix sum -> alloc ->
// reconstruct_haplotypes_from_sparse -> rc_flat_rows_inplace, plus the one-hot transform the
// reference leaves to seqpro (docs/source/index.md:108-119).
//
// Data flow (all in HBM, nothing on the host):
//   plan    one warp per (query, hap) row walks the row's sparse variant list in chunks of 32
//           (coalesced index loads, gathered table loads) and drives the reference's state
//           machine (gvl_plan.cuh) in lock-step; emits <= n_variants records
//           (alt_out_start, alt_len, alt_src, ref_resume, variant_idx, variant_pos) + a row header.
//   scan    (ragged plans only) single-CTA exclusive scan of row lengths -> out_offsets, tile map.
//   execute one CTA per 4096-position output tile; records of the tile are staged in shared
//           memory; every thread produces 4 consecutive output positions per step: 4 reference
//           bytes with two aligned 32-bit loads + funnel shift, ALT/pad bytes patched in,
//           reverse-complement and the encoding fused, one 16-byte store (one-hot) per step.
//           Every output byte is written exactly once; no intermediate haplotype in HBM.
#include "gvl_internal.cuh"

namespace gvl {

// =====================================================================================
// plan
// =====================================================================================
struct HapPlanParams {
    gvl_sparse_tables tab;
    MergedLists merged;  // all-NULL for the SVAR1 CSR source
    const int32_t *regions;
    const int32_t *shifts;
    const int64_t *goi;
    const uint8_t *keep;
    const int64_t *keep_off;
    const uint8_t *to_rc;
    int64_t n_work, ploidy, output_length, rec_cap;
    RowPlan *rows;
    RecArrays rec;
    int64_t *words;
    int64_t *out_offsets;
    int32_t *diffs;
    int32_t *row_len;
    int32_t *dir;        // fixed-length plans: checkpoint directory (NULL otherwise)
    int64_t dir_stride;  // entries per row = ceil(length / DIR_Q) + 1
    // > 0: every row owns record slots [k * row_stride, (k + 1) * row_stride) (callers that bound the list length PER ROW: no
    // cursor atomic, and -- without merged lists -- no completion count either); 0: rows take space from words[W_CURSOR]
    int64_t row_stride;
    // track mode (hap_plan_par_kernel<NT, true>): 32-byte records, per-query source window lengths
    TRec *trecs;
    const int32_t *track_lengths;
};

constexpr int PLAN_WARPS = 4;

// Checkpoint directory of a row, written by the NT threads that planned it once its records are in
// global memory: dir[q] = number of records whose ALT starts before haplotype position q * DIR_Q.
// The execute kernels read their tile's record range from it instead of searching the record list.
template <int NT>
__device__ __forceinline__ void write_dir(const HapPlanParams &P, int64_t k, int64_t rec_off, int64_t n_rec, int t) {
    if (!P.dir) return;
    if (NT == 32) __syncwarp(); else __syncthreads();  // the row's records are visible to the whole group
    int32_t *__restrict__ d = P.dir + k * P.dir_stride;
    const int64_t nq = P.dir_stride - 1;
    if (n_rec == 0) {
        for (int64_t q = t; q <= nq; q += NT) d[q] = 0;
        return;
    }
    const int32_t *a = P.rec.a + rec_off;
    for (int64_t i = t; i < n_rec; i += NT) {
        const int64_t q_lo = i == 0 ? 0 : (int64_t)a[i - 1] / DIR_Q + 1;
        const int64_t q_hi = imin64((int64_t)a[i] / DIR_Q, nq);
        for (int64_t q = q_lo; q <= q_hi; q++) d[q] = (int32_t)i;
        if (i == n_rec - 1)
            for (int64_t q = q_hi + 1; q <= nq; q++) d[q] = (int32_t)n_rec;
    }
}

// Serial (lock-step) plan of one row by ONE warp: the reference's loop, one variant per step.
// Exact for any input order; the scan-based kernel (gvl_plan_par.cuh) calls it for rows whose
// variant list is not position-sorted and handles everything else itself.
__device__ void plan_row_serial(const HapPlanParams &P, const int64_t k, const int64_t rec_off_in = -1) {
    const int lane = lane_id();
    const int64_t query = k / P.ploidy;
    const RowVars rv = row_vars(P.tab, P.merged, P.goi, k);
    const int64_t nvar = rv.nvar;
    const int64_t c_idx = P.regions[query * 3 + 0];
    const int64_t c_s = P.tab.ref_offsets[c_idx];
    const int64_t contig_len = P.tab.ref_offsets[c_idx + 1] - c_s;
    const int64_t q_start = P.regions[query * 3 + 1];
    const int64_t q_end = P.regions[query * 3 + 2];
    const int64_t shift = P.shifts[k];
    const int64_t keep_base = (P.keep && P.keep_off) ? P.keep_off[k] : 0;
    const bool has_keep = (P.keep && P.keep_off);
    const int32_t *__restrict__ gv = rv.gv;

    // ---- get_diffs_sparse (src/genotypes/mod.rs:48-86), needed first for ragged sizing ----
    DiffState ds;
    diff_init(ds, q_start, q_end);
    bool diff_live = nvar > 0;  // :46-47
    const bool ragged = P.output_length < 0;      // row lengths vary: offsets come from the scan kernel
    const bool sized = P.output_length == -1;     // ... and are sized here from the diffs
    if (sized) {
        for (int64_t base = 0; base < nvar && diff_live; base += 32) {
            int64_t i = base + lane;
            int32_t pos = 0, il = 0;
            bool kp = false;
            if (i < nvar) {
                int32_t vi = gv[i];
                pos = (int32_t)var_pos(P.tab, rv, i, vi);
                il = P.tab.ilens[vi];
                kp = has_keep ? (P.keep[keep_base + i] != 0) : true;
            }
            unsigned mask = __ballot_sync(0xffffffffu, kp);
            while (mask) {
                int t = __ffs(mask) - 1;
                mask &= mask - 1;
                int32_t p = __shfl_sync(0xffffffffu, pos, t), l = __shfl_sync(0xffffffffu, il, t);
                if (!diff_step(ds, p, l)) {
                    diff_live = false;
                    break;
                }
            }
        }
        diff_live = false;
    }
    int64_t length;
    if (sized) {
        length = imax64((q_end - q_start) + (int64_t)(int32_t)ds.acc, 0);  // src/ffi/mod.rs:801-807
    } else if (ragged) {
        length = imax64(P.out_offsets[k + 1] - P.out_offsets[k], 0);  // caller-supplied row bounds
    } else {
        length = P.output_length;
    }

    // ---- workspace for this row's records: nvar + 1 slots ----
    int64_t rec_off = rec_off_in;
    if (rec_off_in < 0) {
        if (lane == 0) rec_off = (int64_t)atomicAdd((unsigned long long *)&P.words[W_CURSOR], (unsigned long long)(nvar + 1));
        rec_off = __shfl_sync(0xffffffffu, rec_off, 0);
    }
    const bool overflow = rec_off + nvar + 1 > P.rec_cap;
    if (overflow && lane == 0) atomicMax((unsigned long long *)&P.words[W_STATUS], (unsigned long long)(rec_off + nvar + 1));

    // ---- reconstruct_haplotype_core state machine (src/reconstruct/mod.rs:39-256) ----
    HapState hs;
    hap_init(hs, q_start, shift, length);
    int64_t n_emit = 0, ref0 = 0, prev_resume = 0;
    bool done = false;
    for (int64_t base = 0; base < nvar && (!done || diff_live); base += 32) {
        int64_t i = base + lane;
        int32_t pos = 0, il = 0, alen = 0, vi = 0;
        int64_t aoff = 0;
        bool kp = false;
        if (i < nvar) {
            vi = gv[i];
            pos = (int32_t)var_pos(P.tab, rv, i, vi);
            il = P.tab.ilens[vi];
            int64_t alen64;
            var_alt(P.tab, rv, vi, pos, c_s, aoff, alen64);
            alen = (int32_t)alen64;
            kp = has_keep ? (P.keep[keep_base + i] != 0) : true;
            if (rv.mpos) vi = (int32_t)i;  // svar2 annotates with the LOCAL index (src/reconstruct/mod.rs:734)
        }
        unsigned mask = __ballot_sync(0xffffffffu, kp);
        while (mask && (!done || diff_live)) {
            int t = __ffs(mask) - 1;
            mask &= mask - 1;
            int32_t p = __shfl_sync(0xffffffffu, pos, t);
            int32_t l = __shfl_sync(0xffffffffu, il, t);
            int32_t al = __shfl_sync(0xffffffffu, alen, t);
            if (diff_live && !diff_step(ds, p, l)) diff_live = false;
            if (done) continue;
            HapRec r;
            int act = hap_step(hs, p, l, al, r);
            if (act == STEP_BREAK) {
                done = true;
            } else if (act == STEP_EMIT) {
                if (n_emit == 0) ref0 = r.span_src;
                if (n_emit > 0 && r.span_src != prev_resume) {
                    // unsorted input moved ref_idx between emissions: zero-length "jump" record.
                    // span start (output coordinate) of this record = r.a - (v_pos - span_src)
                    int64_t span_out = r.a - ((int64_t)p - r.span_src);
                    if (lane == t && !overflow) {
                        int64_t w = rec_off + n_emit;
                        P.rec.a[w] = (int32_t)span_out;
                        P.rec.n[w] = 0;
                        P.rec.src[w] = 0;
                        P.rec.resume[w] = (int32_t)r.span_src;
                        P.rec.vidx[w] = -1;
                        P.rec.vpos[w] = -1;
                    }
                    n_emit++;
                }
                if (lane == t && !overflow) {
                    int64_t w = rec_off + n_emit;
                    P.rec.a[w] = (int32_t)r.a;
                    P.rec.n[w] = (int32_t)r.n;
                    P.rec.src[w] = aoff + r.trim;
                    P.rec.resume[w] = (int32_t)r.resume;
                    P.rec.vidx[w] = vi;
                    P.rec.vpos[w] = p;
                }
                n_emit++;
                prev_resume = r.resume;
                if (hs.out_idx >= hs.length) done = true;  // :195-197
            }
        }
    }
    hap_finish(hs, contig_len);
    if (n_emit == 0) {
        ref0 = hs.ref_idx;
    } else if (hs.ref_idx != prev_resume) {  // unsorted input: trailing jump
        if (lane == 0 && !overflow) {
            int64_t w = rec_off + n_emit;
            P.rec.a[w] = (int32_t)imin64(hs.out_idx, length);
            P.rec.n[w] = 0;
            P.rec.src[w] = 0;
            P.rec.resume[w] = (int32_t)hs.ref_idx;
            P.rec.vidx[w] = -1;
            P.rec.vpos[w] = -1;
        }
        n_emit++;
    }

    if (lane == 0) {
        RowPlan rp;
        rp.out_off = ragged ? 0 : k * length;
        rp.ref_base = c_s;
        rp.rec_off = rec_off;
        rp.length = (int32_t)length;
        rp.contig_len = (int32_t)contig_len;
        rp.lead_pad = (int32_t)imin64(hs.lead_pad, length);
        rp.ref0 = (int32_t)ref0;
        rp.n_rec = overflow ? 0 : (int32_t)n_emit;
        rp.rc = (P.to_rc && P.to_rc[k]) ? 1 : 0;
        rp.diff = nvar > 0 ? (int32_t)ds.acc : 0;
        rp.q_start = (int32_t)q_start;
        P.rows[k] = rp;
        if (P.diffs) P.diffs[k] = rp.diff;
        if (ragged) {
            P.row_len[k] = (int32_t)length;
        } else {
            P.out_offsets[k] = k * length;
            if (k == P.n_work - 1) P.out_offsets[P.n_work] = P.n_work * length;
        }
    }
    write_dir<32>(P, k, rec_off, overflow ? 0 : n_emit, lane);
}

#include "gvl_trk_plan.cuh"
#include "gvl_plan_par.cuh"

// Threads per (query, hap) row of the parallel plan kernel, from the mean list-length bound: one warp for short lists; one
// 256-thread CTA up to ~4,000 variants (cfg3's ~600-variant rows: 52 us per 640 rows against 63 us with 512 threads -- a
// half-empty second chunk costs more than a third pass; cfg2d's ~1,300-variant rows: 125 vs 144 us); 512 beyond.
static int plan_width(int64_t max_records, int64_t n_work) {
    if (max_records <= 40 * n_work) return 32;
    return max_records <= 4096 * n_work ? 256 : 512;
}

// ragged plans: exclusive scan of row lengths -> out_offsets, RowPlan.out_off, tile map, totals.
__global__ void __launch_bounds__(1024) row_scan_kernel(int64_t n_work, const int32_t *__restrict__ row_len,
                                                        RowPlan *rows, int64_t *out_offsets, int64_t *tile_off,
                                                        int64_t *words) {
    __shared__ int64_t s_len[32], s_tile[32];
    __shared__ int64_t carry_len, carry_tile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        carry_len = 0;
        carry_tile = 0;
    }
    __syncthreads();
    for (int64_t base = 0; base < n_work; base += 1024) {
        int64_t k = base + tid;
        int64_t len = (k < n_work) ? (int64_t)row_len[k] : 0;
        int64_t til = (len + TILE - 1) / TILE;
        int64_t xl = len, xt = til;
        for (int o = 1; o < 32; o <<= 1) {
            int64_t yl = __shfl_up_sync(0xffffffffu, xl, o), yt = __shfl_up_sync(0xffffffffu, xt, o);
            if (lane >= o) {
                xl += yl;
                xt += yt;
            }
        }
        if (lane == 31) {
            s_len[warp] = xl;
            s_tile[warp] = xt;
        }
        __syncthreads();
        if (warp == 0) {
            int64_t wl = s_len[lane], wt = s_tile[lane];
            for (int o = 1; o < 32; o <<= 1) {
                int64_t yl = __shfl_up_sync(0xffffffffu, wl, o), yt = __shfl_up_sync(0xffffffffu, wt, o);
                if (lane >= o) {
                    wl += yl;
                    wt += yt;
                }
            }
            s_len[lane] = wl;
            s_tile[lane] = wt;
        }
        __syncthreads();
        int64_t pre_l = carry_len + (warp ? s_len[warp - 1] : 0) + xl - len;
        int64_t pre_t = carry_tile + (warp ? s_tile[warp - 1] : 0) + xt - til;
        if (k < n_work) {
            if (out_offsets) out_offsets[k] = pre_l;
            rows[k].out_off = pre_l;
            tile_off[k] = pre_t;
        }
        __syncthreads();
        if (tid == 0) {
            carry_len += s_len[31];
            carry_tile += s_tile[31];
        }
        __syncthreads();
    }
    if (tid == 0) {
        if (out_offsets) out_offsets[n_work] = carry_len;
        tile_off[n_work] = carry_tile;
        words[W_TOTAL] = carry_len;
        words[W_TILES] = carry_tile;
    }
}

// =====================================================================================
// execute
// =====================================================================================
struct HapExecParams {
    const RowPlan *rows;
    RecArrays rec;
    const uint8_t *ref;
    const uint32_t *ref_packed;  // optional 4-bit codes (gvl_hap_oh.cuh)
    const uint32_t *alt_packed;  // optional 4-bit codes of alt_alleles
    const uint8_t *alt;
    int64_t n_work;
    int64_t tiles_per_row;    // >0: fixed-length plan
    const int64_t *tile_off;  // ragged plan: first tile of each row
    int32_t tile_len;         // haplotype positions per CTA (multiple of EXEC_UNIT)
    const int32_t *dir;       // fixed-length plans: checkpoint directory (write_dir), else NULL
    int64_t dir_stride;
    int64_t fixed_len;
    uint8_t *out;
    int32_t *annot_v;
    int32_t *annot_pos;
    uint32_t pad_char;
};

struct TileRecs {
    int32_t a[REC_CAP + 1];       // ALT start (haplotype coordinate); a[m] sentinel
    int32_t e[REC_CAP];           // ALT end = start of the following reference span
    int32_t resume[REC_CAP];      // reference position at e[]
    int64_t src[REC_CAP];         // ALT source (offset into alt_alleles), ALT_PAD for the leading pad
    int32_t vidx[REC_CAP];
    int32_t vpos[REC_CAP];
};

// complement one base: A<->T (xor 0x15), C<->G (xor 0x04), everything else unchanged
// (src/reverse.rs:45-53).
__device__ __forceinline__ uint32_t comp1(uint32_t b) {
    uint32_t at = (b == 'A' || b == 'T') ? 0x15u : 0u;
    uint32_t cg = (b == 'C' || b == 'G') ? 0x04u : 0u;
    return b ^ at ^ cg;
}

// complement 4 packed bases (SWAR form of comp1)
__device__ __forceinline__ uint32_t comp4(uint32_t v) {
    uint32_t at = __vcmpeq4(v, 0x41414141u) | __vcmpeq4(v, 0x54545454u);
    uint32_t cg = __vcmpeq4(v, 0x43434343u) | __vcmpeq4(v, 0x47474747u);
    return v ^ (at & 0x15151515u) ^ (cg & 0x04040404u);
}

// one-hot of a single base: byte c of the word is (b == "ACGT"[c]).
__device__ __forceinline__ uint32_t onehot1(uint32_t b) {
    return (b == 'A' ? 1u : 0u) | (b == 'C' ? 0x100u : 0u) | (b == 'G' ? 0x10000u : 0u) | (b == 'T' ? 0x1000000u : 0u);
}

// last staged entry i in [0, m) with a[i] <= p (entry 0 always qualifies)
__device__ __forceinline__ int find_rec(const TileRecs &S, int m, int32_t p) {
    int lo = 0, hi = m;
    while (hi - lo > 1) {
        int mid = (lo + hi) >> 1;
        if (S.a[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
}

constexpr int COUNT_MAX = 2048;  // rows with more records locate their tile range by 32-ary search

template <int MODE>
__global__ void __launch_bounds__(EXEC_THREADS, EXEC_MIN_CTAS) hap_exec_kernel(HapExecParams P) {
    constexpr bool ANNOT = (MODE == GVL_MODE_ANNOTATED);
    constexpr bool OH = (MODE == GVL_MODE_ONEHOT || MODE == GVL_MODE_ONEHOT_CF);
    __shared__ TileRecs S;
    __shared__ __align__(16) uint32_t s_lut[OH ? 512 : 4];  // [0,256): one-hot(b); [256,512): one-hot(complement(b))
    __shared__ int64_t s_lo, s_hi;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // ---- tile -> (row, tile-in-row) ----
    int64_t row, tile;
    if (P.tiles_per_row > 0) {
        tile = blockIdx.x;
        row = (int64_t)blockIdx.y + (int64_t)blockIdx.z * 65535;
        if (row >= P.n_work) return;
    } else {
        int64_t b = blockIdx.x;
        if (b >= P.tile_off[P.n_work]) return;
        int64_t lo = 0, hi = P.n_work;  // last row with tile_off[row] <= b
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (P.tile_off[mid] <= b) lo = mid; else hi = mid;
        }
        row = lo;
        tile = b - P.tile_off[row];
    }
    const RowPlan rp = P.rows[row];
    const int32_t L = rp.length;
    // tiles are cut in HAPLOTYPE coordinates; a reversed row writes them back to front
    const int64_t h0_64 = tile * (int64_t)P.tile_len;
    if (h0_64 >= L) return;
    const int32_t h0 = (int32_t)h0_64;
    const int32_t h1 = (int32_t)imin64(h0_64 + P.tile_len, L);
    const bool rc = rp.rc != 0;

    if (OH) reinterpret_cast<uint4 *>(s_lut)[tid] = make_uint4(0u, 0u, 0u, 0u);  // 128 threads x 16 B = the whole table
    __syncthreads();
    if (OH && tid < 8) {  // the only non-zero entries: ACGT (and their complements in the second half)
        const int i = tid & 3;
        const uint32_t letter = (0x54474341u >> (8 * i)) & 0xffu;  // 'A','C','G','T'
        s_lut[(tid < 4 ? 0 : 256) + letter] = 1u << (8 * (tid < 4 ? i : 3 - i));
    }

    // ---- records of this tile: r_lo = last with a <= h0 (or -1), r_hi = first with a >= h1 ----
    // (warp 0 only: the other warps have nothing to do until the records are staged)
    const int32_t *__restrict__ ra = P.rec.a + rp.rec_off;
    if (warp == 0) {
        int64_t r_lo, r_hi0;
        if (rp.n_rec <= COUNT_MAX) {
            int c0 = 0, c1 = 0;  // sorted array: counts are indices
            for (int i = lane; i < rp.n_rec; i += 32) {
                const int32_t a = ra[i];
                c0 += (a <= h0);
                c1 += (a < h1);
            }
            r_lo = (int64_t)__reduce_add_sync(0xffffffffu, c0) - 1;
            r_hi0 = __reduce_add_sync(0xffffffffu, c1);
        } else {
            r_lo = warp_upper_le(ra, 0, rp.n_rec, h0);
            r_hi0 = warp_upper_le(ra, imax64(r_lo, 0), rp.n_rec, h1 - 1) + 1;
        }
        if (lane == 0) {
            s_lo = r_lo;
            s_hi = r_hi0;
        }
    }
    __syncthreads();
    const int64_t r_hi = s_hi;
    int64_t r = s_lo;
    int32_t cur = h0;
    const uint8_t *__restrict__ refrow = P.ref + rp.ref_base;
    uint8_t *__restrict__ out_row = P.out + (OH ? 4 : 1) * rp.out_off;  // position j of the row lives at out_row[(4*)j]
    const uint32_t lut_a = smem_u32(s_lut);   // byte address of the table in shared memory
    const uint32_t lut_rc = rc ? 1024u : 0u;  // second half = one-hot of the complement

    // one 4-position chunk made only of reference bytes: v holds the bytes in OUTPUT order (not yet
    // complemented), r0 = reference position of the chunk's lowest haplotype position
    auto emit_ref4 = [&](int32_t j, uint32_t v, int32_t r0) {
        if (OH) {
            uint4 o;
            // table offset of base i = (byte_i * 4) | half: one shift + one 3-input logic op each (hand-written
            // shared-memory addressing: +2 % over indexing the table, profiles/)
            o.x = lds_u32(lut_a + (((v << 2) & 0x3fcu) | lut_rc));
            o.y = lds_u32(lut_a + (((v >> 6) & 0x3fcu) | lut_rc));
            o.z = lds_u32(lut_a + (((v >> 14) & 0x3fcu) | lut_rc));
            o.w = lds_u32(lut_a + (((v >> 22) & 0x3fcu) | lut_rc));
            if (MODE == GVL_MODE_ONEHOT) {
                *reinterpret_cast<uint4 *>(out_row + 4 * (int64_t)j) = o;
            } else {
                uint8_t *op = out_row + j;  // (4, L) block of this row
                const uint32_t xy0 = __byte_perm(o.x, o.y, 0x5140), xy1 = __byte_perm(o.x, o.y, 0x7362);
                const uint32_t zw0 = __byte_perm(o.z, o.w, 0x5140), zw1 = __byte_perm(o.z, o.w, 0x7362);
                *reinterpret_cast<uint32_t *>(op) = __byte_perm(xy0, zw0, 0x5410);
                *reinterpret_cast<uint32_t *>(op + L) = __byte_perm(xy0, zw0, 0x7632);
                *reinterpret_cast<uint32_t *>(op + 2 * (int64_t)L) = __byte_perm(xy1, zw1, 0x5410);
                *reinterpret_cast<uint32_t *>(op + 3 * (int64_t)L) = __byte_perm(xy1, zw1, 0x7632);
            }
        } else {
            if (rc) v = comp4(v);
            *reinterpret_cast<uint32_t *>(out_row + j) = v;
            if (ANNOT) {
                const int64_t g = rp.out_off + j;
                *reinterpret_cast<int4 *>(P.annot_v + g) = make_int4(-1, -1, -1, -1);
                *reinterpret_cast<int4 *>(P.annot_pos + g) =
                    rc ? make_int4(r0 + 3, r0 + 2, r0 + 1, r0) : make_int4(r0, r0 + 1, r0 + 2, r0 + 3);
            }
        }
    };

    while (cur < h1) {
        // ---- stage entry 0 (carry) + up to REC_CAP-1 following records ----
        const int m_new = (int)imin64(REC_CAP - 1, r_hi - (r + 1));
        const int m = m_new + 1;
        const int32_t seg_end = (r + 1 + m_new < r_hi) ? ra[r + 1 + m_new] : h1;
        __syncthreads();  // previous pass finished reading S
        for (int i = tid; i < m; i += EXEC_THREADS) {  // (m is a handful of records: effectively warp 0)
            int64_t idx = r + i;
            if (idx < 0) {  // virtual record: leading pad, then reference from ref0
                S.a[0] = 0;
                S.e[0] = rp.lead_pad;
                S.resume[0] = rp.ref0;
                S.src[0] = ALT_PAD;
                S.vidx[0] = -1;
                S.vpos[0] = -1;
            } else {
                int64_t g = rp.rec_off + idx;
                int32_t a = P.rec.a[g], n = P.rec.n[g];
                S.a[i] = a;
                S.e[i] = a + n;
                S.resume[i] = P.rec.resume[g];
                S.src[i] = P.rec.src[g];
                if (ANNOT) {
                    S.vidx[i] = P.rec.vidx[g];
                    S.vpos[i] = P.rec.vpos[g];
                }
            }
        }
        if (tid == 0) S.a[m] = INT32_MAX;
        __syncthreads();

        // ---- output range of this pass, chunked by 4 on the GLOBAL flat index ----
        // chunk c covers row positions j0+4c .. j0+4c+3; a GROUP is 32 chunks (one per lane: 128
        // positions, one 512-byte one-hot store per warp), a BLOCK is 4 groups.  Warp w owns blocks
        // w, w+4, ...
        const int32_t jo_lo = rc ? L - seg_end : cur;
        const int32_t jo_hi = rc ? L - cur : seg_end;
        const int64_t g0 = (rp.out_off + jo_lo) & ~(int64_t)3;
        const int32_t j0 = (int32_t)(g0 - rp.out_off);  // row-relative position of chunk 0 (may be < jo_lo)
        const int32_t n_chunks = (jo_hi - j0 + 3) >> 2;
        const int32_t n_blocks = (n_chunks + 127) >> 7;
        int ic = rc ? (m - 1) : 0;  // warp-uniform record cursor (blocks are visited in monotone order)

        for (int32_t blk = warp; blk < n_blocks; blk += EXEC_THREADS / 32) {
            const int32_t jb = j0 + 512 * blk;  // first row position of the block
            if (jb >= jo_lo && jb + 512 <= jo_hi) {
                // ---- whole block inside the pass: one warp-uniform test against the records ----
                const int32_t p_lo = rc ? (L - 512 - jb) : jb;  // lowest haplotype position of the block
                if (!rc) {
                    while (S.a[ic + 1] <= p_lo) ic++;
                } else {
                    while (S.a[ic] > p_lo) ic--;
                }
                const int32_t e_i = S.e[ic];
                const int64_t rpos_lo = (int64_t)S.resume[ic] + (p_lo - e_i);
                if (p_lo >= e_i && p_lo + 511 < S.a[ic + 1] && rpos_lo + 511 < rp.contig_len) {
                    // 512 reference bytes in a row: all 8 loads first, then 4 encodes + stores
                    const int32_t r_lane = (int32_t)rpos_lo + (rc ? 508 - 4 * lane : 4 * lane);
                    const uintptr_t addr = reinterpret_cast<uintptr_t>(refrow + r_lane);
                    const unsigned sh = (unsigned)(addr & 3) * 8u;
                    uint32_t w0[4], w1[4];
                    const uint32_t *w = reinterpret_cast<const uint32_t *>(addr & ~(uintptr_t)3);
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int off = rc ? -32 * k : 32 * k;  // group k of the OUTPUT lies 128 bytes further (back)
                        w0[k] = __ldg(w + off);
                        w1[k] = __ldg(w + off + 1);  // (readable: buffers carry >= 16 B of slack)
                    }
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        uint32_t v = __funnelshift_r(w0[k], w1[k], sh);  // byte i = haplotype position p0+i
                        if (rc) v = __byte_perm(v, 0, 0x0123);            // byte i = output position j+i
                        emit_ref4(jb + 128 * k + 4 * lane, v, r_lane + (rc ? -128 * k : 128 * k));
                    }
                    continue;
                }
            }
            {
            // ---- block with variants / pads / pass edges: group by group ----
            int ig = (jb >= jo_lo && jb + 512 <= jo_hi) ? ic : -1;  // cursor for the block's lowest position, if known
#pragma unroll 1
            for (int k = 0; k < 4; k++) {
                const int32_t cg = blk * 128 + 32 * k;  // first chunk of the group
                if (cg >= n_chunks) break;
                const int32_t jg = j0 + 4 * cg;
                const int32_t j = jg + 4 * lane;
                if (jg >= jo_lo && jg + 128 <= jo_hi) {
                    const int32_t p_lo = rc ? (L - 128 - jg) : jg;
                    if (ig < 0) ig = find_rec(S, m, p_lo);
                    while (S.a[ig + 1] <= p_lo) ig++;  // forward rows: groups ascend
                    while (S.a[ig] > p_lo) ig--;       // reversed rows: groups descend
                    const int32_t e_i = S.e[ig];
                    const int64_t rpos_lo = (int64_t)S.resume[ig] + (p_lo - e_i);
                    if (p_lo >= e_i && p_lo + 127 < S.a[ig + 1] && rpos_lo + 127 < rp.contig_len) {
                        const int32_t r_lane = (int32_t)rpos_lo + (rc ? 124 - 4 * lane : 4 * lane);
                        const uintptr_t addr = reinterpret_cast<uintptr_t>(refrow + r_lane);
                        uint32_t x0, x1;
                        const uint32_t *w = reinterpret_cast<const uint32_t *>(addr & ~(uintptr_t)3);
                        x0 = __ldg(w);
                        x1 = __ldg(w + 1);
                        uint32_t v = __funnelshift_r(x0, x1, (unsigned)(addr & 3) * 8u);
                        if (rc) v = __byte_perm(v, 0, 0x0123);
                        emit_ref4(j, v, r_lane);
                        continue;
                    }
                }
                // ---- generic chunk: resolve each position against the records ----
                if (cg + lane >= n_chunks) continue;
                const int32_t pa = rc ? (L - 4 - j) : j;  // haplotype position of byte t=0 (ascending in t)
                const bool full = (j >= jo_lo) && (j + 4 <= jo_hi);
                uint32_t v = 0;          // byte t = haplotype position pa+t (raw, not complemented)
                int32_t av[4], ap[4];    // annotations in haplotype order
                int il = -1;
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    av[t] = -1;
                    ap[t] = -1;
                    const int32_t jj = rc ? (j + 3 - t) : (j + t);
                    if (!full && (jj < jo_lo || jj >= jo_hi)) continue;
                    const int32_t p = pa + t;
                    if (il < 0) il = find_rec(S, m, p);
                    while (S.a[il + 1] <= p) il++;
                    uint32_t b;
                    if (p < S.e[il]) {
                        const int64_t src = S.src[il];
                        if (src == ALT_PAD) {
                            b = P.pad_char;  // leading pad (src/reconstruct/mod.rs:75-80): annotations (-1, -1)
                        } else {
                            // (src < 0: pure-deletion anchor of the svar2 source, taken from the reference)
                            b = src >= 0 ? P.alt[src + (p - S.a[il])] : P.ref[~src + (p - S.a[il])];
                            if (ANNOT) {
                                av[t] = S.vidx[il];
                                ap[t] = S.vpos[il];
                            }
                        }
                    } else {
                        const int64_t rpos = (int64_t)S.resume[il] + (p - S.e[il]);
                        if (rpos < rp.contig_len) {
                            b = refrow[rpos];
                            ap[t] = (int32_t)rpos;
                        } else {
                            b = P.pad_char;
                            ap[t] = INT32_MAX;  // trailing pad (:248-253)
                        }
                    }
                    v |= b << (8 * t);
                }
                if (rc) v = __byte_perm(v, 0, 0x0123);  // byte i = output position j+i
                if (full) {
                    if (OH) {
                        emit_ref4(j, v, 0);
                    } else {
                        if (rc) v = comp4(v);
                        *reinterpret_cast<uint32_t *>(out_row + j) = v;
                        if (ANNOT) {
                            const int64_t g = rp.out_off + j;
                            *reinterpret_cast<int4 *>(P.annot_v + g) =
                                rc ? make_int4(av[3], av[2], av[1], av[0]) : make_int4(av[0], av[1], av[2], av[3]);
                            *reinterpret_cast<int4 *>(P.annot_pos + g) =
                                rc ? make_int4(ap[3], ap[2], ap[1], ap[0]) : make_int4(ap[0], ap[1], ap[2], ap[3]);
                        }
                    }
                } else {
                    // chunk cut by a pass / row boundary: position-wise stores
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int32_t jj = j + q;
                        if (jj < jo_lo || jj >= jo_hi) continue;
                        uint32_t b = (v >> (8 * q)) & 0xffu;
                        if (rc) b = comp1(b);
                        if (MODE == GVL_MODE_ONEHOT) {
                            *reinterpret_cast<uint32_t *>(out_row + 4 * (int64_t)jj) = onehot1(b);
                        } else if (MODE == GVL_MODE_ONEHOT_CF) {
                            uint8_t *op = out_row + jj;
                            op[0] = (b == 'A');
                            op[L] = (b == 'C');
                            op[2 * (int64_t)L] = (b == 'G');
                            op[3 * (int64_t)L] = (b == 'T');
                        } else {
                            out_row[jj] = (uint8_t)b;
                            if (ANNOT) {
                                P.annot_v[rp.out_off + jj] = av[rc ? 3 - q : q];
                                P.annot_pos[rp.out_off + jj] = ap[rc ? 3 - q : q];
                            }
                        }
                    }
                }
            }
            }
        }
        cur = seg_end;
        r += m_new;
    }
}

}  // namespace gvl
#include "gvl_hap_oh.cuh"
namespace gvl {

// standalone get_diffs_sparse (all four branches of src/genotypes/mod.rs:46-104)
struct DiffParams {
    gvl_sparse_tables tab;
    MergedLists merged;  // svar2 source: merged per-row lists (key == NULL: SVAR1 CSR through goi)
    int64_t q_stride;    // element stride of q_starts / q_ends (3: columns 1 and 2 of a (b,3) regions array)
    const int64_t *goi;
    const uint8_t *keep;
    const int64_t *keep_off;
    const int32_t *q_starts;
    const int32_t *q_ends;
    int use_v_starts;
    int64_t n_work, ploidy;
    int32_t *diffs;
};

__global__ void __launch_bounds__(PLAN_WARPS * 32) diffs_kernel(DiffParams P) {
    const int lane = lane_id();
    const int64_t k = (int64_t)blockIdx.x * PLAN_WARPS + (threadIdx.x >> 5);
    if (k >= P.n_work) return;
    const int64_t query = k / P.ploidy;
    const RowVars rv = row_vars(P.tab, P.merged, P.goi, k);
    const int64_t nvar = rv.nvar;
    const bool has_query = P.q_starts && P.q_ends && P.use_v_starts;
    const bool has_keep = P.keep && P.keep_off;
    const int64_t keep_base = has_keep ? P.keep_off[k] : 0;
    const int32_t *__restrict__ gv = rv.gv;
    int64_t acc = 0;
    if (has_query) {
        DiffState ds;
        diff_init(ds, P.q_starts[query * P.q_stride], P.q_ends[query * P.q_stride]);
        bool live = true;
        for (int64_t base = 0; base < nvar && live; base += 32) {
            int64_t i = base + lane;
            int32_t pos = 0, il = 0;
            bool kp = false;
            if (i < nvar) {
                int32_t vi = gv[i];
                pos = rv.mpos ? rv.mpos[i] : P.tab.v_starts[vi];
                il = P.tab.ilens[vi];
                kp = has_keep ? (P.keep[keep_base + i] != 0) : true;
            }
            unsigned mask = __ballot_sync(0xffffffffu, kp);
            while (mask) {
                int t = __ffs(mask) - 1;
                mask &= mask - 1;
                int32_t p = __shfl_sync(0xffffffffu, pos, t), l = __shfl_sync(0xffffffffu, il, t);
                if (!diff_step(ds, p, l)) {
                    live = false;
                    break;
                }
            }
        }
        acc = ds.acc;
    } else {
        int64_t part = 0;
        for (int64_t i = lane; i < nvar; i += 32) {
            bool kp = has_keep ? (P.keep[keep_base + i] != 0) : true;
            if (kp) part += P.tab.ilens[gv[i]];
        }
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        acc = part;
    }
    if (lane == 0) P.diffs[k] = (int32_t)acc;
}

}  // namespace gvl

using namespace gvl;

// resident CTAs of the execute kernel on this device (one wave)
static int64_t exec_capacity(gvl_ctx *ctx, int mode) {
    static int64_t cache[8][4] = {};
    if (ctx->device < 8 && cache[ctx->device][mode & 3]) return cache[ctx->device][mode & 3];
    int sms = 148, per_sm = 8;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device);
    switch (mode) {
        case GVL_MODE_U8: cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hap_exec_kernel<GVL_MODE_U8>, EXEC_THREADS, 0); break;
        case GVL_MODE_ONEHOT: cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hap_exec_kernel<GVL_MODE_ONEHOT>, EXEC_THREADS, 0); break;
        case GVL_MODE_ONEHOT_CF: cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hap_exec_kernel<GVL_MODE_ONEHOT_CF>, EXEC_THREADS, 0); break;
        default: cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hap_exec_kernel<GVL_MODE_ANNOTATED>, EXEC_THREADS, 0); break;
    }
    int64_t cap = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
    if (ctx->device < 8) cache[ctx->device][mode & 3] = cap;
    return cap;
}

// Merge of the svar2 two-channel source (gvl_svar2.cu); fills ctx->hap.m_* for n_work rows.
int gvl_svar2_merge_launch(gvl_ctx *ctx, gvl_workspace *ws, int64_t *words, const gvl_svar2_channels *ch, int64_t batch,
                           int64_t ploidy, int64_t max_merged, cudaStream_t st);

// merge-only callers (no plan kernel follows that would do it): put the cursors back to zero, keep the status word
__global__ void reset_cursors_kernel(int64_t *words) {
    words[W_CURSOR] = 0;
    words[W_MERGE_CURSOR] = 0;
    words[W_DONE] = 0;
}

static int hap_plan_impl(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *svar2,
                         const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
                         int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
                         int64_t output_length, int64_t max_records, int64_t *out_offsets, int32_t *diffs,
                         gvl_stream stream) {
    if (!ctx || !tab || !regions || !shifts || !(geno_offset_idx || svar2) || !out_offsets)
        return fail(GVL_ERR_ARG, "gvl_dev_hap_plan: NULL argument");
    if (batch < 0 || ploidy < 1) return fail(GVL_ERR_ARG, "gvl_dev_hap_plan: batch=%lld ploidy=%lld", (long long)batch, (long long)ploidy);
    if (output_length > INT32_MAX) return fail(GVL_ERR_ARG, "gvl_dev_hap_plan: output_length too large");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_work = batch * ploidy;
    ctx->plan_valid = false;
    int rc;
    if ((rc = ensure_rows(ctx, ctx->hap, n_work))) return rc;
    if ((rc = ensure_records(ctx, ctx->hap, max_records + n_work))) return rc;
    // (no memset of the status words: every plan leaves its cursors at zero, see plan_row_done)
    ctx->n_work = n_work;
    ctx->fixed_len = output_length >= 0 ? output_length : -1;
    ctx->rec_bound_per_row = n_work > 0 ? max_records / n_work : 0;
    ctx->plan_out_offsets = out_offsets;
    if (n_work == 0) {
        GVL_CUDA(cudaMemsetAsync(out_offsets, 0, sizeof(int64_t), st));
        ctx->total = 0;
        ctx->plan_valid = true;
        return GVL_OK;
    }
    HapPlanParams P;
    P.tab = *tab;
    P.merged = MergedLists{nullptr, nullptr, nullptr, nullptr};
    if (svar2) {
        if ((rc = ensure_merged(ctx, ctx->hap, max_records))) return rc;
        if ((rc = gvl_svar2_merge_launch(ctx, &ctx->hap, ctx->dev_words, svar2, batch, ploidy, max_records, st))) return rc;
        P.merged = MergedLists{ctx->hap.m_pos, ctx->hap.m_key, ctx->hap.m_off, ctx->hap.m_len};
    }
    P.regions = regions;
    P.shifts = shifts;
    P.goi = geno_offset_idx;
    P.keep = keep;
    P.keep_off = keep_offsets;
    P.to_rc = to_rc;
    P.n_work = n_work;
    P.ploidy = ploidy;
    P.output_length = output_length >= 0 ? output_length : (output_length == -2 ? -2 : -1);
    P.rec_cap = ctx->hap.rec_cap;
    P.row_stride = (ctx->row_stride_hint > 0 && ctx->row_stride_hint * n_work <= ctx->hap.rec_cap) ? ctx->row_stride_hint : 0;
    P.rows = ctx->hap.rows;
    P.rec = ctx->hap.rec;
    P.words = ctx->dev_words;
    P.out_offsets = out_offsets;
    P.diffs = diffs;
    P.row_len = ctx->hap.row_len;
    P.dir = nullptr;
    P.dir_stride = 0;
    P.trecs = nullptr;
    P.track_lengths = nullptr;
    ctx->dir_stride = 0;
    if (output_length >= 0) {
        const int64_t stride = (output_length + DIR_Q - 1) / DIR_Q + 1;
        if ((rc = ensure_dir(ctx, ctx->hap, n_work * stride))) return rc;
        P.dir = ctx->hap.dir;
        P.dir_stride = ctx->dir_stride = stride;
    }
    const int nt = plan_width(max_records, n_work);
    ctx->last_launch[GVL_LAUNCH_PLAN_THREADS] = nt;
    ctx->last_launch[GVL_LAUNCH_PLAN_STATIC] = P.row_stride > 0;
    if (nt == 32) {  // short lists: one warp per row, 4 rows per CTA
        hap_plan_par_kernel<32, false><<<(unsigned)((n_work + 3) / 4), 128, 0, st>>>(P);
    } else if (nt == 256) {  // one 256-thread CTA per row
        hap_plan_par_kernel<256, false><<<(unsigned)n_work, 256, 0, st>>>(P);
    } else {  // long lists: 512 variants per sequential chunk
        hap_plan_par_kernel<512, false><<<(unsigned)n_work, 512, 0, st>>>(P);
    }
    GVL_LAUNCH_CHECK();
    if (output_length >= 0) {
        ctx->total = n_work * output_length;
    } else {
        row_scan_kernel<<<1, 1024, 0, st>>>(n_work, ctx->hap.row_len, ctx->hap.rows,
                                            output_length == -2 ? nullptr : out_offsets, ctx->hap.tile_off, ctx->dev_words);
        GVL_LAUNCH_CHECK();
        ctx->total = -1;
    }
    ctx->plan_valid = true;
    return GVL_OK;
}

// The track plan: the same kernel in track mode over the TRACK workspace of the context (rows sized by the caller's
// out_offsets; merged svar2 lists when `merged` is set).  Called by gvl_tracks.cu.
int gvl_trk_plan_launch(gvl_ctx *ctx, const gvl_sparse_tables *tab, const MergedLists *merged, const int32_t *regions,
                        const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy,
                        const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc, const int32_t *track_lengths,
                        const int64_t *out_offsets, int64_t max_records, int64_t *words, cudaStream_t st) {
    const int64_t n_work = batch * ploidy;
    HapPlanParams P;
    P.tab = *tab;
    P.merged = merged ? *merged : MergedLists{nullptr, nullptr, nullptr, nullptr};
    P.regions = regions;
    P.shifts = shifts;
    P.goi = geno_offset_idx;
    P.keep = keep;
    P.keep_off = keep_offsets;
    P.to_rc = to_rc;
    P.n_work = n_work;
    P.ploidy = ploidy;
    P.output_length = -2;  // rows sized by the caller's offsets
    P.rec_cap = ctx->trk.trec_cap;
    P.row_stride = (ctx->row_stride_hint > 0 && ctx->row_stride_hint * n_work <= ctx->trk.trec_cap) ? ctx->row_stride_hint : 0;
    P.rows = ctx->trk.rows;
    P.rec = RecArrays{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    P.words = words;
    P.out_offsets = const_cast<int64_t *>(out_offsets);  // (read only in this mode)
    P.diffs = nullptr;
    P.row_len = ctx->trk.row_len;
    P.dir = nullptr;
    P.dir_stride = 0;
    P.trecs = (TRec *)ctx->trk.trecs;
    P.track_lengths = track_lengths;
    const int nt = plan_width(max_records, n_work);
    ctx->last_launch[GVL_LAUNCH_TRK_PLAN_THREADS] = nt;
    ctx->last_launch[GVL_LAUNCH_TRK_PLAN_STATIC] = P.row_stride > 0;
    if (nt == 32) hap_plan_par_kernel<32, true><<<(unsigned)((n_work + 3) / 4), 128, 0, st>>>(P);
    else if (nt == 256) hap_plan_par_kernel<256, true><<<(unsigned)n_work, 256, 0, st>>>(P);
    else hap_plan_par_kernel<512, true><<<(unsigned)n_work, 512, 0, st>>>(P);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

extern "C" {

int gvl_dev_hap_plan(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int32_t *regions, const int32_t *shifts,
                     const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const uint8_t *keep,
                     const int64_t *keep_offsets, const uint8_t *to_rc, int64_t output_length, int64_t max_records,
                     int64_t *out_offsets, int32_t *diffs, gvl_stream stream) {
    if (!geno_offset_idx) return fail(GVL_ERR_ARG, "gvl_dev_hap_plan: NULL argument");
    return hap_plan_impl(ctx, tab, nullptr, regions, shifts, geno_offset_idx, batch, ploidy, keep, keep_offsets, to_rc,
                         output_length, max_records, out_offsets, diffs, stream);
}

int gvl_dev_hap_plan_svar2(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *ch,
                           const int32_t *regions, const int32_t *shifts, int64_t batch, int64_t ploidy,
                           const uint8_t *to_rc, int64_t output_length, int64_t max_merged, int64_t *out_offsets,
                           int32_t *diffs, gvl_stream stream) {
    if (!ch || !ch->vk_off || !ch->dense_range || !ch->dense_present_off)
        return fail(GVL_ERR_ARG, "gvl_dev_hap_plan_svar2: NULL channel");
    return hap_plan_impl(ctx, tab, ch, regions, shifts, nullptr, batch, ploidy, nullptr, nullptr, to_rc, output_length,
                         max_merged, out_offsets, diffs, stream);
}

int gvl_dev_hap_total(gvl_ctx *ctx, gvl_stream stream, int64_t *total) {
    if (!ctx || !total) return fail(GVL_ERR_ARG, "gvl_dev_hap_total: NULL argument");
    if (!ctx->plan_valid) return fail(GVL_ERR_STATE, "gvl_dev_hap_total: no plan");
    if (ctx->total < 0) {
        int rc = gvl_ctx_check(ctx, stream);  // syncs, mirrors the status words
        if (rc) return rc;
        ctx->total = ctx->host_words[W_TOTAL];
    }
    *total = ctx->total;
    return GVL_OK;
}

int gvl_dev_hap_exec(gvl_ctx *ctx, const gvl_sparse_tables *tab, int mode, uint8_t pad_char, uint8_t *out,
                     int32_t *annot_v, int32_t *annot_pos, gvl_stream stream) {
    if (!ctx || !tab) return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: NULL argument");
    if (!ctx->plan_valid) return fail(GVL_ERR_STATE, "gvl_dev_hap_exec: no plan");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    if (ctx->n_work == 0 || ctx->total == 0) return GVL_OK;
    if (!out) return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: out is NULL");
    if (((uintptr_t)out & 15) || ((uintptr_t)annot_v & 15) || ((uintptr_t)annot_pos & 15))
        return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: output buffers must be 16-byte aligned");
    if ((uintptr_t)tab->ref & 15) return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: the reference buffer must be 16-byte aligned");
    if (mode == GVL_MODE_ANNOTATED && (!annot_v || !annot_pos))
        return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: annotated mode needs annot_v and annot_pos");
    HapExecParams P;
    P.rows = ctx->hap.rows;
    P.rec = ctx->hap.rec;
    P.ref = tab->ref;
    P.ref_packed = tab->ref_packed;
    P.alt_packed = tab->alt_packed;
    P.dir = ctx->dir_stride > 0 ? ctx->hap.dir : nullptr;
    P.dir_stride = ctx->dir_stride;
    P.fixed_len = ctx->fixed_len;
    P.alt = tab->alt_alleles;
    P.n_work = ctx->n_work;
    P.out = out;
    P.annot_v = annot_v;
    P.annot_pos = annot_pos;
    P.pad_char = pad_char;
    // one-hot over the packed reference (gvl_hap_oh.cuh) when the caller supplied it
    const bool packed = mode == GVL_MODE_ONEHOT && tab->ref_packed && tab->alt_packed &&
                        !((uintptr_t)out & 31) && !((uintptr_t)tab->ref_packed & 15) && !((uintptr_t)tab->alt_packed & 15);
    int64_t grid;
    if (ctx->fixed_len >= 0 && packed) {
        // Tiles as long as they can be (<= OH_MAX_TILE) while the batch still gives every SM ~3 CTAs: a CTA's fixed
        // cost (two dependent round trips before its first store) is amortised over more positions, and a launch
        // that leaves CTA slots free lets the next batch's launch (another stream) overlap its latency phases
        // with this one's store stream (measured: profiles/r1_packed.md).
        const int64_t q = imax64((OH_THREADS / 32) * OH_GROUP, DIR_Q);  // whole groups per warp, whole directory quanta
        static const int sms = [] {
            int n = 148, dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
            return n;
        }();
        const int64_t target_ctas = 3 * (int64_t)sms;
        int64_t tl = ctx->fixed_len * ctx->n_work / target_ctas;
        // tiles beyond 16,384 positions only where the plan's record bound promises one staging pass per tile (REC_CAP = 128:
        // about 100 records per tile); denser -- or loosely bounded, like the svar2 source whose bound counts the whole
        // cohort's dense window -- lists keep the 16,384 of round 1 (cfg2d: 8,192 -> 336 us, 16,384 -> 352, 32,768 -> 373)
        if (tl > 16384 && !(ctx->rec_bound_per_row > 0 && ctx->rec_bound_per_row * (int64_t)OH_MAX_TILE <= 100 * ctx->fixed_len))
            tl = 16384;
        // lists so dense that a 16,384-position tile needs a second staging pass (REC_CAP = 128): 8,192 (cfg2d: 304 -> 285 us)
        if (tl > 8192 && ctx->fixed_len > 0 && ctx->rec_bound_per_row * (int64_t)16384 > (int64_t)REC_CAP * ctx->fixed_len) tl = 8192;
        tl = imax64(q, imin64(tl / q * q, OH_MAX_TILE));
        P.tile_len = (int32_t)tl;
        P.tiles_per_row = (ctx->fixed_len + P.tile_len - 1) / P.tile_len;
        P.tile_off = nullptr;
        grid = P.tiles_per_row * ctx->n_work;
    } else if (ctx->fixed_len >= 0) {
        // pick the tile length so that the whole batch is ONE wave of CTAs when it can be
        const int64_t units_per_row = (ctx->fixed_len + EXEC_UNIT - 1) / EXEC_UNIT;
        const int64_t tiles_target = imax64(1, exec_capacity(ctx, mode) / ctx->n_work);
        int64_t units_per_tile = (units_per_row + tiles_target - 1) / tiles_target;
        units_per_tile = (units_per_tile + 3) & ~(int64_t)3;  // whole 512-position blocks for each of the 4 warps
        units_per_tile = imax64(4, imin64(units_per_tile, EXEC_MAX_UNITS));
        P.tile_len = (int32_t)(units_per_tile * EXEC_UNIT);
        P.tiles_per_row = (ctx->fixed_len + P.tile_len - 1) / P.tile_len;
        P.tile_off = nullptr;
        grid = P.tiles_per_row * ctx->n_work;
    } else {
        P.tile_len = TILE;
        if (ctx->total < 0) return fail(GVL_ERR_STATE, "gvl_dev_hap_exec: ragged plan needs gvl_dev_hap_total first");
        if (mode == GVL_MODE_ONEHOT_CF) return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: channels-first one-hot needs a fixed length");
        P.tiles_per_row = 0;
        P.tile_off = ctx->hap.tile_off;
        grid = ctx->host_words[W_TILES];
    }
    if (grid == 0) return GVL_OK;
    if (grid > INT32_MAX) return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: too many tiles");
    dim3 grid3((unsigned)grid, 1, 1);
    if (ctx->fixed_len >= 0) {  // (tile, row) grid: no division in the kernel
        const int64_t gy = imin64(ctx->n_work, 65535);
        grid3 = dim3((unsigned)P.tiles_per_row, (unsigned)gy, (unsigned)((ctx->n_work + 65534) / 65535));
    }
    if (mode == GVL_MODE_ONEHOT_CF && (ctx->fixed_len & 3))
        return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: channels-first one-hot needs output_length %% 4 == 0");
    int64_t kind = GVL_EXEC_BYTES;
    switch (mode) {
        case GVL_MODE_U8: hap_exec_kernel<GVL_MODE_U8><<<grid3, EXEC_THREADS, 0, st>>>(P); break;
        case GVL_MODE_ONEHOT:
            if (packed) {
                // loads of 4 groups in flight per warp for long, sparse rows; 2 where the record bound says "dense" (the tile
                // length above stayed at 16,384 for that reason) or a warp has fewer than 8 groups to walk
                const bool sparse = ctx->fixed_len > 0 && ctx->rec_bound_per_row > 0 &&
                                    ctx->rec_bound_per_row * (int64_t)OH_MAX_TILE <= 100 * ctx->fixed_len;
                const int64_t groups_per_warp = (imin64(P.tile_len, ctx->fixed_len) / OH_GROUP) / (OH_THREADS / 32);
                if (imin64(P.tile_len, ctx->fixed_len) <= 8192 && P.tiles_per_row == 1) {  // short rows: one tile per row, 2-warp CTAs
                    hap_exec_oh_kernel<2, 64><<<grid3, 64, 0, st>>>(P);
                    kind = GVL_EXEC_PACKED_2WARP;
                } else if (ctx->fixed_len < 0 || (sparse && groups_per_warp >= 8)) {  // (ragged plans: as in round 1)
                    hap_exec_oh_kernel<OH_UNROLL_LONG, OH_THREADS><<<grid3, OH_THREADS, 0, st>>>(P);
                    kind = GVL_EXEC_PACKED_UNROLL4;
                } else {
                    hap_exec_oh_kernel<2, OH_THREADS><<<grid3, OH_THREADS, 0, st>>>(P);
                    kind = GVL_EXEC_PACKED_UNROLL2;
                }
            }
            else hap_exec_kernel<GVL_MODE_ONEHOT><<<grid3, EXEC_THREADS, 0, st>>>(P);
            break;
        case GVL_MODE_ONEHOT_CF: hap_exec_kernel<GVL_MODE_ONEHOT_CF><<<grid3, EXEC_THREADS, 0, st>>>(P); break;
        case GVL_MODE_ANNOTATED: hap_exec_kernel<GVL_MODE_ANNOTATED><<<grid3, EXEC_THREADS, 0, st>>>(P); break;
        default: return fail(GVL_ERR_ARG, "gvl_dev_hap_exec: unknown mode %d", mode);
    }
    GVL_LAUNCH_CHECK();
    ctx->last_exec_kernel = packed ? 1 : 0;
    ctx->last_launch[GVL_LAUNCH_EXEC_KERNEL] = kind;
    ctx->last_launch[GVL_LAUNCH_TILE_LEN] = P.tile_len;
    ctx->last_launch[GVL_LAUNCH_TILES_PER_ROW] = P.tiles_per_row;
    ctx->last_launch[GVL_LAUNCH_REC_BOUND] = ctx->rec_bound_per_row;
    return GVL_OK;
}

int gvl_debug_last_exec_kernel(gvl_ctx *ctx) { return ctx ? ctx->last_exec_kernel : -1; }

int gvl_debug_last_launch(gvl_ctx *ctx, int64_t *out, int n) {
    if (!ctx || (!out && n > 0) || n < 0) return fail(GVL_ERR_ARG, "gvl_debug_last_launch: bad argument");
    for (int i = 0; i < n && i < GVL_LAUNCH_FIELDS; i++) out[i] = ctx->last_launch[i];
    return GVL_OK;
}

int64_t gvl_packed_reference_words(int64_t n_bases) { return (imax64(n_bases, 0) + 7) / 8 + 4; }  // + zeroed slack

int gvl_dev_pack_reference(gvl_ctx *ctx, const uint8_t *ref, int64_t n_bases, uint32_t *ref_packed, gvl_stream stream) {
    if (!ctx || !ref_packed || (!ref && n_bases > 0) || n_bases < 0)
        return fail(GVL_ERR_ARG, "gvl_dev_pack_reference: bad argument");
    if (((uintptr_t)ref & 15) || ((uintptr_t)ref_packed & 15))
        return fail(GVL_ERR_ARG, "gvl_dev_pack_reference: buffers must be 16-byte aligned");
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_words = gvl_packed_reference_words(n_bases);
    const unsigned grid = (unsigned)imax64(1, imin64((n_words + 255) / 256, 148 * 16));
    pack_ref_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(ref, n_bases, ref_packed, n_words);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

int gvl_dev_get_diffs_sparse(gvl_ctx *ctx, const gvl_sparse_tables *tab, const int64_t *geno_offset_idx,
                             int64_t n_queries, int64_t ploidy, const uint8_t *keep, const int64_t *keep_offsets,
                             const int32_t *q_starts, const int32_t *q_ends, int use_v_starts, int32_t *diffs,
                             gvl_stream stream) {
    if (!ctx || !tab || !geno_offset_idx || !diffs) return fail(GVL_ERR_ARG, "gvl_dev_get_diffs_sparse: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t n_work = n_queries * ploidy;
    if (n_work == 0) return GVL_OK;
    DiffParams P;
    P.tab = *tab;
    P.merged = MergedLists{nullptr, nullptr, nullptr, nullptr};
    P.q_stride = 1;
    P.goi = geno_offset_idx;
    P.keep = keep;
    P.keep_off = keep_offsets;
    P.q_starts = q_starts;
    P.q_ends = q_ends;
    P.use_v_starts = use_v_starts;
    P.n_work = n_work;
    P.ploidy = ploidy;
    P.diffs = diffs;
    diffs_kernel<<<(unsigned)((n_work + PLAN_WARPS - 1) / PLAN_WARPS), PLAN_WARPS * 32, 0, st>>>(P);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

int gvl_dev_hap_diffs_svar2(gvl_ctx *ctx, const gvl_sparse_tables *tab, const gvl_svar2_channels *ch, const int32_t *regions,
                            int64_t batch, int64_t ploidy, int64_t max_merged, int32_t *diffs, gvl_stream stream) {
    if (!ctx || !tab || !tab->ilens || !ch || !ch->vk_off || !ch->dense_range || !ch->dense_present_off)
        return fail(GVL_ERR_ARG, "gvl_dev_hap_diffs_svar2: NULL argument");
    if (batch < 0 || ploidy < 1 || max_merged < 0) return fail(GVL_ERR_ARG, "gvl_dev_hap_diffs_svar2: bad sizes");
    const int64_t n_work = batch * ploidy;
    if (n_work == 0) return GVL_OK;
    if (!regions || !diffs) return fail(GVL_ERR_ARG, "gvl_dev_hap_diffs_svar2: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    GVL_CUDA(cudaSetDevice(ctx->device));
    // merged lists go to the TRACK workspace (never holds a plan across calls), so a haplotype plan that has not been
    // executed yet stays valid
    int rc;
    if ((rc = ensure_rows(ctx, ctx->trk, n_work))) return rc;
    if ((rc = ensure_merged(ctx, ctx->trk, max_merged))) return rc;
    int64_t *words = ctx->dev_words + W_COUNT;  // (cursors are zero between calls, see plan_row_done)
    if ((rc = gvl_svar2_merge_launch(ctx, &ctx->trk, words, ch, batch, ploidy, max_merged, st))) return rc;
    DiffParams P;
    P.tab = *tab;
    P.merged = MergedLists{ctx->trk.m_pos, ctx->trk.m_key, ctx->trk.m_off, ctx->trk.m_len};
    P.q_stride = 3;
    P.goi = nullptr;
    P.keep = nullptr;
    P.keep_off = nullptr;
    P.q_starts = regions + 1;
    P.q_ends = regions + 2;
    P.use_v_starts = 1;
    P.n_work = n_work;
    P.ploidy = ploidy;
    P.diffs = diffs;
    diffs_kernel<<<(unsigned)((n_work + PLAN_WARPS - 1) / PLAN_WARPS), PLAN_WARPS * 32, 0, st>>>(P);
    GVL_LAUNCH_CHECK();
    reset_cursors_kernel<<<1, 1, 0, st>>>(words);
    GVL_LAUNCH_CHECK();
    return GVL_OK;
}

}  // extern "C"
