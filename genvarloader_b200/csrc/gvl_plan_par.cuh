// gvl_plan_par.cuh -- scan-based parallel haplotype plan (included by gvl_hap.cu).
//
// The reference walks a haplotype's variants one by one (src/reconstruct/mod.rs:85-198).  For a
// position-sorted list the walk decomposes into data-parallel steps over a chunk of NT variants
// (one per thread), with the state (ref_idx R, out_idx O, shifted) carried between chunks:
//
//  A  variants left of the window: only a deletion spanning the window start acts (:99-102); the
//     LAST such deletion in list order sets R.                                   -> block max
//  B  while the shift is not consumed (:115-146) neither R nor `shifted` change until the first
//     variant j* with shifted + (pos - R) + alt_len >= shift; everything before it is skipped
//     without side effects.                                                       -> block min
//  C  afterwards a variant is applied iff pos >= R_current, where R_current is the end of the last
//     APPLIED variant (:108-110, first ALT wins).  A variant whose pos is >= every earlier end
//     (and >= R) is certainly applied ("head").  Variants between heads overlap something and are
//     resolved by a short serial walk started at each head (clusters are tiny in practice; the
//     walk is exact for any size).                                                -> max-scan + walk
//  D  reference gap before each applied variant = pos - end(previous applied)      -> max-scan
//     output position of its ALT bytes = O + sum(gaps + ALT lengths before) + gap  -> sum-scan
//     the loop `break`s (:154-158) at the first applied variant whose ALT would start at or
//     beyond `length`; positions are monotone, so validity is a prefix.          -> sum-scan (rank)
//
// Unsorted lists (out of contract for the reference's writers, but legal inputs of the kernel) are
// detected and replanned by plan_row_serial, which is exact for any order.
// get_diffs_sparse (src/genotypes/mod.rs:48-86) has the same shape: a variant counts iff it starts
// left of the window or at/after the running maximum end of counted variants.
#pragma once
// (included from inside `namespace gvl` in gvl_hap.cu)

template <int NT>
__device__ __forceinline__ void grp_sync() {
    if (NT == 32) __syncwarp(); else __syncthreads();
}

// inclusive scan over the NT threads of a group (a warp, or the whole CTA) -- OP in {max, add}
template <int NT, bool IS_MAX>
__device__ __forceinline__ int64_t grp_scan_incl(int64_t x, int64_t *s_warp /* >= NT/32 + 1 slots */) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int64_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = IS_MAX ? imax64(x, y) : x + y;
    }
    if (NT == 32) return x;
    const int warp = threadIdx.x >> 5;
    __syncthreads();  // s_warp may still be read by the previous scan
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int64_t pre = IS_MAX ? INT64_MIN : 0;
    for (int w = 0; w < warp; w++) pre = IS_MAX ? imax64(pre, s_warp[w]) : pre + s_warp[w];
    return IS_MAX ? imax64(x, pre) : x + pre;
}

// reduction to ALL threads of the group
template <int NT, bool IS_MAX>
__device__ __forceinline__ int64_t grp_reduce(int64_t x, int64_t *s_warp) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        int64_t y = __shfl_xor_sync(0xffffffffu, x, o);
        x = IS_MAX ? imax64(x, y) : imin64(x, y);
    }
    if (NT == 32) return x;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = x;
    __syncthreads();
    int64_t r = s_warp[0];
    for (int w = 1; w < NT / 32; w++) r = IS_MAX ? imax64(r, s_warp[w]) : imin64(r, s_warp[w]);
    return r;
}

// One-barrier block scan: inclusive result, the value of the thread before (`excl`, identity for thread 0) and the
// group's aggregate (`total`), for 32- or 64-bit operands.  Consecutive scans alternate between two staging buffers
// (`sb` toggles uniformly), so the buffer a scan writes was last read two scans -- at least one barrier -- ago.
template <class T, bool IS_MAX> struct ScanId;
template <> struct ScanId<int32_t, true> { static constexpr int32_t v = INT32_MIN; };
template <> struct ScanId<int64_t, true> { static constexpr int64_t v = INT64_MIN; };
template <> struct ScanId<int32_t, false> { static constexpr int32_t v = 0; };
template <> struct ScanId<int64_t, false> { static constexpr int64_t v = 0; };

template <int NT, bool IS_MAX, class T>
__device__ __forceinline__ T grp_scan_x(T x, int64_t (*bufs)[NT / 32 + 1], int &sb, T &excl, T &total) {
    const int lane = threadIdx.x & 31;
    constexpr T ID = ScanId<T, IS_MAX>::v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x = IS_MAX ? (x > y ? x : y) : x + y;
    }
    T ex = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) ex = ID;
    if (NT == 32) {
        excl = ex;
        total = __shfl_sync(0xffffffffu, x, 31);
        return x;
    }
    T *s = reinterpret_cast<T *>(bufs[sb]);
    sb ^= 1;
    const int warp = threadIdx.x >> 5;
    if (lane == 31) s[warp] = x;
    __syncthreads();
    T pre = ID, tot = ID;
#pragma unroll
    for (int w = 0; w < NT / 32; w++) {
        const T v = s[w];
        if (w < warp) pre = IS_MAX ? (pre > v ? pre : v) : pre + v;
        tot = IS_MAX ? (tot > v ? tot : v) : tot + v;
    }
    excl = IS_MAX ? (ex > pre ? ex : pre) : ex + pre;
    total = tot;
    return IS_MAX ? (x > pre ? x : pre) : x + pre;
}

// number of threads of the group whose predicate holds, to all threads (one barrier)
template <int NT>
__device__ __forceinline__ int grp_count(bool p) {
    if (NT == 32) return __popc(__ballot_sync(0xffffffffu, p));
    return __syncthreads_count(p);
}

template <int NT>
struct PlanSmem {
    int32_t pos[NT];
    int32_t end[NT];
    uint8_t elig[NT];
    uint8_t head[NT];
    uint8_t applied[NT];
    int64_t warp[NT / 32 + 1];
    int64_t scan[2][NT / 32 + 1];  // grp_scan_x staging (double-buffered)
    int64_t st[2];                  // carried state broadcast (output cursor, reference cursor)
    int flag;
};

// TRK = false: haplotype rows (reconstruct_haplotype_core).  TRK = true: track rows (shift_and_realign_track_core,
// src/tracks/mod.rs:224-406) -- the SAME offset scan with the track core's three differences: the "ALT length" of a
// variant is max(ilen, 0) + 1 (:282), SNPs take part in the shift bookkeeping only and otherwise change nothing
// (:310-314), and there is no leading-pad clause (the source window is query-relative, positions left of it just read 0).
// Records go out as 32-byte TRec (output range, resume point, anchor, fill length, ilen) in window-relative coordinates.
// PLAN_OCC = resident threads per SM the register allocation aims for (1,280 or 1,536 spill and gain nothing:
// profiles/r2_plan.md)
constexpr int PLAN_OCC = 1024;
template <int NT, bool TRK>
__global__ void __launch_bounds__(NT == 32 ? 128 : NT, PLAN_OCC / (NT == 32 ? 128 : NT)) hap_plan_par_kernel(HapPlanParams P) {
    constexpr int ROWS_PER_CTA = (NT == 32) ? 4 : 1;
    __shared__ PlanSmem<NT> s_all[ROWS_PER_CTA];
    PlanSmem<NT> &S = s_all[(NT == 32) ? (threadIdx.x >> 5) : 0];
    const int t = (NT == 32) ? (threadIdx.x & 31) : threadIdx.x;  // index within the row's group
    const int64_t k = (NT == 32) ? ((int64_t)blockIdx.x * 4 + (threadIdx.x >> 5)) : (int64_t)blockIdx.x;
    if (k >= P.n_work) return;  // (NT == 32: whole warps exit; NT == 256: whole CTA)

    const int64_t query = k / P.ploidy;
    const RowVars rv = row_vars(P.tab, P.merged, P.goi, k);
    const int64_t nvar = rv.nvar;
    const int64_t c_idx = P.regions[query * 3 + 0];
    const int64_t c_s = TRK ? 0 : P.tab.ref_offsets[c_idx];
    const int64_t q_start = P.regions[query * 3 + 1];
    // (tracks: the "contig" is the source window [q_start, q_start + track_n), _reconstruct.py:191-196)
    const int64_t contig_len = TRK ? q_start + (int64_t)P.track_lengths[query] : P.tab.ref_offsets[c_idx + 1] - c_s;
    const int64_t q_end = P.regions[query * 3 + 2];
    const int64_t shift = P.shifts[k];
    const bool has_keep = (P.keep && P.keep_off);
    const int64_t keep_base = has_keep ? P.keep_off[k] : 0;
    const int32_t *__restrict__ gv = rv.gv;
    const bool ragged = P.output_length < 0;
    const bool sized = P.output_length == -1;
    const bool want_diff = !TRK && (sized || (P.diffs != nullptr));

    // record workspace of the row: one atomic per row.  Its round trip overlaps with the first gathers: the value
    // stays in thread 0 until the first chunk's loads are in flight (bcast_off below).
    int64_t rec_off = 0;
    const bool static_rows = P.row_stride > 0;  // the row owns a fixed slice: no atomic (81,920 same-address atomics cost cfg4 ~90 us)
    if (static_rows) rec_off = k * P.row_stride;
    else if (t == 0) rec_off = (int64_t)atomicAdd((unsigned long long *)&P.words[W_CURSOR], (unsigned long long)(nvar + 1));
    // (rows of a statically sliced plan that reads no merged lists leave the cursors untouched: nothing to put back)
    const bool count_done = !static_rows || P.merged.off != nullptr;
    bool have_off = false, overflow = false;
    auto bcast_off = [&]() {
        if (have_off) return;
        if (static_rows) {
            overflow = nvar + 1 > P.row_stride;
            if (overflow && t == 0) atomicMax((unsigned long long *)&P.words[W_STATUS], (unsigned long long)(P.rec_cap + nvar + 1));
            have_off = true;
            return;
        }
        if (NT == 32) {
            rec_off = __shfl_sync(0xffffffffu, rec_off, 0);
        } else {
            if (t == 0) S.warp[NT / 32] = rec_off;
            __syncthreads();
            rec_off = S.warp[NT / 32];
        }
        overflow = rec_off + nvar + 1 > P.rec_cap;
        if (overflow && t == 0) atomicMax((unsigned long long *)&P.words[W_STATUS], (unsigned long long)(rec_off + nvar + 1));
        have_off = true;
    };

    // ---------------------------------------------------------------- pass 1: diffs (only if needed)
    bool unsorted = false;
    int64_t diff_acc = 0;
    if (want_diff && nvar > 0) {
        int64_t d_ref = q_start;  // running max end of counted variants (src/genotypes/mod.rs:57,78)
        int64_t last_pos = INT64_MIN;
        int sb1 = 0;
        for (int64_t base = 0; base < nvar; base += NT) {
            const int64_t i = base + t;
            int64_t pos = INT64_MAX, il = 0;
            bool kept = false;
            if (i < nvar) {
                const int32_t vi = gv[i];
                pos = var_pos(P.tab, rv, i, vi);
                il = P.tab.ilens[vi];
                kept = has_keep ? (P.keep[keep_base + i] != 0) : true;
            }
            const int64_t end = (i < nvar) ? pos - imin64(il, 0) + 1 : INT64_MIN;
            // sortedness (of the whole list, kept or not)
            const int nv = (int)imin64(NT, nvar - base);  // entries of this chunk
            const int32_t end32 = (int32_t)imax64(imin64(end, INT32_MAX), INT32_MIN);
            S.pos[t] = (int32_t)imin64(pos, INT32_MAX);
            S.end[t] = end32;
            grp_sync<NT>();
            const int64_t prev = (t > 0) ? (int64_t)S.pos[t - 1] : last_pos;
            bool bad = (i < nvar) && (pos < prev);
            if (NT == 32) bad = __any_sync(0xffffffffu, bad); else bad = __syncthreads_or(bad);
            if (bad) {
                unsorted = true;
                break;
            }
            last_pos = S.pos[nv - 1];
            // variants that take part at all: :69-74 (the `break` is a suffix cut for sorted input)
            const bool in = kept && (end > q_start) && (pos < q_end);
            int32_t mx_excl32, tot32;
            grp_scan_x<NT, true, int32_t>(in ? end32 : INT32_MIN, S.scan, sb1, mx_excl32, tot32);
            const int64_t mx_excl = imax64((int64_t)mx_excl32, d_ref);
            const bool left = in && pos < q_start;          // always counted
            const bool head = in && !left && pos >= mx_excl;  // certainly counted, resets the running max
            S.elig[t] = in ? (left ? 2 : 1) : 0;
            S.head[t] = head;
            S.applied[t] = (left || head);
            grp_sync<NT>();
            // cluster walks: from every head, and from the chunk start (virtual head with cur = d_ref)
            if (head || t == 0) {
                int64_t cur = head ? end : d_ref;
                int u = head ? t + 1 : 0;
                for (; u < nv && !S.head[u]; u++) {
                    const int e = S.elig[u];
                    if (e == 0) continue;
                    if (e == 2) {
                        cur = imax64(cur, S.end[u]);
                    } else if ((int64_t)S.pos[u] >= cur) {
                        S.applied[u] = 1;
                        cur = imax64(cur, S.end[u]);
                    }
                }
            }
            grp_sync<NT>();
            const bool counted = S.applied[t] != 0;
            int64_t adj = 0;
            if (counted) {
                adj = il;
                if (il < 0) adj += imax64(q_start - pos - 1, 0);  // :79-81
                adj += imax64(end - q_end, 0);                     // :82
            }
            // chunk totals: sum of the adjustments, maximum end of the counted variants
            int64_t adj_excl, chunk_sum;
            grp_scan_x<NT, false, int64_t>(adj, S.scan, sb1, adj_excl, chunk_sum);
            int32_t cm_excl, chunk_max;
            grp_scan_x<NT, true, int32_t>(counted ? end32 : INT32_MIN, S.scan, sb1, cm_excl, chunk_max);
            diff_acc += chunk_sum;
            d_ref = imax64(d_ref, (int64_t)chunk_max);
        }
    }

    int64_t length;
    if (sized) {
        length = imax64((q_end - q_start) + (int64_t)(int32_t)diff_acc, 0);  // src/ffi/mod.rs:801-807
    } else if (ragged) {
        length = imax64(P.out_offsets[k + 1] - P.out_offsets[k], 0);
    } else {
        length = P.output_length;
    }

    // ---------------------------------------------------------------- pass 2: haplotype records
    HapState hs;
    hap_init(hs, q_start, shift, length);  // leading pad, :68-83
    if (TRK) {  // src/tracks/mod.rs:249-251: no pad clause, the cursor starts at the window start
        hs.ref_idx = q_start;
        hs.out_idx = 0;
        hs.shifted = 0;
        hs.lead_pad = 0;
    }
    int64_t R = hs.ref_idx, O = hs.out_idx, shifted = hs.shifted;
    int64_t n_emit = 0, ref0 = 0;
    int sb = 0;
    bool done = false;
    int64_t last_pos = INT64_MIN;
    for (int64_t base = 0; base < nvar && !done && !unsorted; base += NT) {
        const int64_t i = base + t;
        int64_t pos = INT64_MAX, il = 0, alen = 0, aoff = 0;
        int32_t vi = 0;
        bool kept = false;
        if (i < nvar) {
            vi = gv[i];
            pos = var_pos(P.tab, rv, i, vi);
            il = P.tab.ilens[vi];
            if (TRK) alen = imax64(il, 0) + 1;  // v_len, src/tracks/mod.rs:282
            else var_alt(P.tab, rv, vi, pos, c_s, aoff, alen);
            kept = has_keep ? (P.keep[keep_base + i] != 0) : true;
            if (rv.mpos) vi = (int32_t)i;  // svar2 annotates with the LOCAL index (src/reconstruct/mod.rs:734)
        }
        bcast_off();  // (first chunk only; the gathers above are already in flight)
        const int64_t end = (i < nvar) ? pos - imin64(il, 0) + 1 : INT64_MIN;
        const int nv = (int)imin64(NT, nvar - base);  // entries of this chunk
        // (every read of S.pos / S.end of the previous chunk is followed by at least one barrier of that chunk)
        const int32_t end32 = (int32_t)imax64(imin64(end, INT32_MAX), INT32_MIN);
        S.pos[t] = (int32_t)imin64(pos, INT32_MAX);
        S.end[t] = end32;
        grp_sync<NT>();
        {
            const int64_t prev = (t > 0) ? (int64_t)S.pos[t - 1] : last_pos;
            bool bad = (i < nvar) && (pos < prev);
            if (NT == 32) bad = __any_sync(0xffffffffu, bad); else bad = __syncthreads_or(bad);
            if (bad) {
                unsorted = true;
                break;
            }
            last_pos = S.pos[nv - 1];  // sorted: the chunk's last entry is its maximum
        }
        // -- A: deletions spanning the window start (:99-102): the last one sets R.  Only chunks that begin left of
        // the window can hold one (sorted list).
        const bool span = kept && pos < q_start && il < 0 && end >= q_start;
        if ((int64_t)S.pos[0] < q_start) {
            const int64_t last_span = grp_reduce<NT, true>(span ? (int64_t)t : -1, S.warp);
            if (last_span >= 0) R = S.end[last_span];
        }
        bool elig = kept && pos >= q_start;  // everything else is skipped without side effects
        // -- B: shift phase (:115-146)
        int64_t start = 0, trim_at = -1, trim = 0;
        if (shifted < shift) {
            const bool cand = elig && pos >= R && (shifted + (pos - R) + alen >= shift);
            const int64_t js = grp_reduce<NT, false>(cand ? (int64_t)t : INT64_MAX, S.warp);
            if (js == INT64_MAX) continue;  // the whole chunk is skipped; R and shifted unchanged
            // operands of j*: broadcast through shared memory
            grp_sync<NT>();
            if (t == js) {
                S.warp[0] = pos;
                S.warp[1] = alen;
                S.warp[2] = end;
            }
            grp_sync<NT>();
            const int64_t jpos = S.warp[0], jalen = S.warp[1], jend = S.warp[2];
            grp_sync<NT>();
            const int64_t d = jpos - R;
            if (shifted + d >= shift) {  // :123-128
                R += shift - shifted;
                start = js;
            } else {
                const int64_t tr = shift - shifted - d;  // :132
                if (tr == jalen) {                        // :135-140
                    R = jend;
                    start = js + 1;
                } else {
                    R = jpos;  // :143
                    start = js;
                    trim_at = js;
                    trim = tr;
                }
            }
            shifted = shift;
        }
        elig = elig && t >= start;
        if (TRK) elig = elig && il != 0;  // a SNP "writes nothing" and does not move the cursor (src/tracks/mod.rs:310-314)
        // -- C: applied set.  Ends are compared as saturated 32-bit values (coordinates are int32 throughout the ABI).
        int32_t mx_excl32, tot32;
        grp_scan_x<NT, true, int32_t>(elig ? end32 : INT32_MIN, S.scan, sb, mx_excl32, tot32);
        const int64_t mx_excl = imax64((int64_t)mx_excl32, R);
        const bool head = elig && pos >= mx_excl;
        // (S.elig / S.head / S.applied of the previous chunk were last read before that chunk's later barriers)
        S.elig[t] = elig;
        S.head[t] = head;
        S.applied[t] = head;
        grp_sync<NT>();
        if (head || t == 0) {
            int64_t cur = head ? end : R;
            int u = head ? t + 1 : 0;
            for (; u < nv && !S.head[u]; u++) {
                if (S.elig[u] && (int64_t)S.pos[u] >= cur) {  // :108-110
                    S.applied[u] = 1;
                    cur = S.end[u];
                }
            }
        }
        grp_sync<NT>();
        const bool applied = S.applied[t] != 0;
        // -- D: gaps, output positions, validity
        int32_t pe_excl32;
        grp_scan_x<NT, true, int32_t>(applied ? end32 : INT32_MIN, S.scan, sb, pe_excl32, tot32);
        const int64_t prev_end = imax64((int64_t)pe_excl32, R);
        const int64_t my_trim = (t == trim_at) ? trim : 0;
        const int64_t ref_len = applied ? pos - prev_end : 0;
        const int64_t alen_eff = applied ? alen - my_trim : 0;
        // one scan for the output positions and the rank among applied variants: lengths << 10 | applied (<= 512 per chunk)
        int64_t pk_excl, pk_tot;
        const int64_t pk_incl = grp_scan_x<NT, false, int64_t>(((ref_len + alen_eff) << 10) | (applied ? 1 : 0), S.scan, sb, pk_excl, pk_tot);
        const int64_t c_incl = pk_incl >> 10;
        const int64_t a = O + (c_incl - (ref_len + alen_eff)) + ref_len;  // ALT start in the output
        const bool valid = applied && a < length;                         // :154-158 (a prefix of the applied variants)
        const int64_t n = valid ? imin64(alen_eff, length - a) : 0;     // :178
        const int64_t rank_incl = pk_incl & 1023;                        // (= rank among VALID ones for a valid variant)
        if (valid && !overflow) {
            const int64_t w = rec_off + n_emit + rank_incl - 1;
            if (TRK) {
                TRec r;
                r.a = (int32_t)a, r.e = (int32_t)(a + n), r.resume = (int32_t)(end - q_start), r.vrel = (int32_t)(pos - q_start);
                r.vlen = (int32_t)alen_eff, r.vdiff = (int32_t)il, r.pad0 = 0, r.pad1 = 0;
                P.trecs[w] = r;
            } else {
                P.rec.a[w] = (int32_t)a;
                P.rec.n[w] = (int32_t)n;
                P.rec.src[w] = aoff + my_trim;
                P.rec.resume[w] = (int32_t)end;
                P.rec.vidx[w] = vi;
                P.rec.vpos[w] = (int32_t)pos;
            }
        }
        // carried state: the chunk's last valid record
        const int n_valid = grp_count<NT>(valid);
        const bool any_broke = (int64_t)n_valid < (pk_tot & 1023);
        if (n_valid > 0) {
            if (valid && rank_incl == n_valid) {
                S.st[0] = a + n;
                S.st[1] = end;
            }
            grp_sync<NT>();
            if (n_emit == 0) ref0 = R;  // the first applied variant's gap starts at R (after the shift)
            O = S.st[0];
            R = S.st[1];
            n_emit += n_valid;
        }
        if (any_broke || O >= length) done = true;  // :154-158, :195-197
    }

    bcast_off();
    if (unsorted) {
        // exact replan in list order by one warp (rare; out of the writers' contract)
        if (NT == 32 || threadIdx.x < 32) {
            if (TRK) trk_plan_row_serial(P, k, rec_off);
            else plan_row_serial(P, k, rec_off);
        }
        if (t == 0 && count_done) plan_row_done(P.words, P.n_work);
        return;
    }
    if (TRK) {
        if (nvar == 0) {
            R = q_start;  // src/tracks/mod.rs:240-246: an EMPTY variant list copies track[:length], whatever the shift
        } else if (shifted < shift) {
            R = imin64(R + (shift - shifted), contig_len);  // :365-369
        }
        if (n_emit == 0) ref0 = R;
        if (t == 0) {
            RowPlan rp;
            rp.out_off = P.out_offsets[k];
            rp.ref_base = 0;
            rp.rec_off = rec_off;
            rp.length = (int32_t)length;
            rp.contig_len = (int32_t)(contig_len - q_start);
            rp.lead_pad = 0;  // (flags of a track row: no jump records on this path)
            rp.ref0 = (int32_t)(ref0 - q_start);
            rp.n_rec = overflow ? 0 : (int32_t)n_emit;
            rp.rc = (P.to_rc && P.to_rc[k]) ? 1 : 0;
            rp.diff = 0;
            rp.q_start = (int32_t)q_start;
            P.rows[k] = rp;
            P.row_len[k] = (int32_t)length;
            if (count_done) plan_row_done(P.words, P.n_work);
        }
        return;
    }

    if (shifted < shift) {  // :200-205
        R = imin64(R + (shift - shifted), contig_len);
    }
    if (n_emit == 0) ref0 = R;
    if (t == 0) {
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
        rp.diff = (int32_t)diff_acc;
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
    write_dir<NT>(P, k, rec_off, overflow ? 0 : n_emit, t);
    if (t == 0 && count_done) plan_row_done(P.words, P.n_work);
}

