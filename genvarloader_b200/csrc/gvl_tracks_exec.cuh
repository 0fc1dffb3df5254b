// gvl_tracks_exec.cuh -- tile preparation + execute kernels of the track path (included by gvl_tracks.cu, inside
// `namespace gvl`).
//
// Reference path replaced: intervals_to_tracks (src/intervals.rs:19-126) into a dense scratch, then
// shift_and_realign_track_core (src/tracks/mod.rs:224-406) + apply_insertion_fill (:87-190) + the reversal of
// negative-strand rows (src/reverse.rs:25-38).
//
// The output of one (track, row) is cut into TILES of T3_TILE values; every tile is independent:
//
//   trk_tile_prep_kernel   one WARP per (track, tile): finds the tile's record cursor, the first stored interval that
//                          reaches into it and the value in effect at its first position (32-ary searches, a probe per
//                          lane, thousands of them in parallel) and leaves a 112-byte descriptor.  All searching of the
//                          path lives here.
//   trk_exec3_kernel       one CTA per tile, no loop, two barriers.  It never materialises the source window: the stored
//                          intervals are painted DIRECTLY IN OUTPUT COORDINATES as a run-length code --
//       load     the descriptor (one broadcast load), then the tile's records and its slice of the interval SoA
//                (coalesced, two intervals per thread, kept in registers and mirrored in shared memory);
//       markers  one thread per stored interval maps its two boundaries from source to haplotype coordinates (a
//                translation per reference span; boundaries inside a deletion vanish) and drops a marker -- the value
//                in effect from there on -- into `val[]` plus a bit into a two-level bitmap; one thread per record
//                drops the value in effect right after the variant; insertion fills other than Repeat5p are computed
//                one value per thread and dropped as markers too;
//       output   every lane owns chunks of 16 consecutive output values: it finds the last marker before its chunk with
//                two bitmap probes (no block-wide scan), walks its 16 marker bits in registers, and writes the chunk
//                with 256-bit stores (float: two, lanes 64 bytes apart; bfloat16 / float16: one of packed pairs).
//     The values themselves never travel through shared memory.  A tile whose source range holds more stored intervals
//     (or records) than are staged at once is finished in further sub-passes (rare: intervals of a few bp).
// The output element type T is float, __nv_bfloat16 or __half: every value is computed in float32 exactly as for float
// output and narrowed at the store (cvt.rn, no .ftz: round to nearest even, overflow to inf, subnormals kept, NaN the
// canonical one) -- bit for bit what a device-side cast of the float32 output gives.
// Rows that need the reference's sequential semantics literally (variant lists that are not position-sorted leave
// "jump" records) and dense f32 sources (shift_and_realign_tracks_sparse) take `t2_generic_segment`: every value
// resolved on its own against the row's records and the source -- slow, exact for any input.
// Binned output (trk_exec3_kernel<T, true>, `t3_bin_pass`): the same values are reduced per bin of 2..4096 output
// positions before the store, so only one value per bin is written.  A bin never straddles a tile (tiles start at
// multiples of T3_TILE in the row), but may straddle the sub-passes of a TD_BIG tile: the open bin's partial result
// carries to the next sub-pass in shared memory.
#pragma once

constexpr int T3_TILE = TRK_TILE;           // output values per execute CTA
constexpr int T2_THREADS = 256;
constexpr int T3_ITV = 512;                 // stored intervals staged per sub-pass (two per thread)
constexpr int T3_REC = 96;                  // records staged per sub-pass (carry + new ones + sentinel)
constexpr int T3_WORDS = T3_TILE / 32;
constexpr int TD_RC = 1, TD_GENERIC = 2, TD_BIG = 4;  // TileDesc.flags
static_assert(TD_RC == GVL_TILE_RC && TD_GENERIC == GVL_TILE_GENERIC && TD_BIG == GVL_TILE_BIG, "gvl_debug_track_tiles reports these flags");

// What trk_tile_prep_kernel leaves for one (track, tile); row < 0 = no such tile.
struct __align__(16) TileDesc {
    int64_t out_base;   // flat index of the row's value 0 in the output buffer
    int64_t it0;        // first stored interval (absolute index) whose end lies beyond the source position feeding h0
    int64_t it_lo, it_hi;  // the slot's intervals (dense source: the query's window offsets)
    int64_t rec_base;   // absolute index of the row's first record
    int32_t n_rec, r;   // records of the row; carry record of the tile (last with a <= h0, -1: none)
    int32_t L, h0, h1;  // row length; the tile in haplotype coordinates
    int32_t q_start, track_n, ref0;
    int32_t flags, row;
    float val0;         // value in effect at h0
    int32_t src_lo, src_hi;  // relative source positions feeding h0 / h1 (sources in [src_lo, src_hi) reach the tile)
    int32_t m, cnt;     // records (carry included) / stored intervals the tile needs; TD_BIG when either exceeds the staging
    int32_t query;      // row / ploidy (hap = row - query * ploidy)
};
static_assert(sizeof(TileDesc) == GVL_TILE_DESC_BYTES, "TileDesc must be GVL_TILE_DESC_BYTES (ensure_tdesc sizes the buffer with it)");

struct T3Smem {
    float val[T3_TILE];             // marker values by tile-relative haplotype position
    TRec rec[T3_REC];               // staged records
    int32_t its[T3_ITV], ite[T3_ITV];  // staged intervals (the record threads and the fills search them)
    float itv[T3_ITV];
    uint32_t mk[T3_WORDS + 1];      // marker bitmap (+ one zero word so that a funnel shift may read past the end)
    uint32_t mk2[T3_WORDS / 32];    // second level: bit w = word w of mk is non-zero
    int32_t fill_list[T3_REC];      // staged records whose insertion fill has to be computed
    int32_t n_fill;
    int32_t bc_i32[4];              // broadcast slots of the (rare) sub-pass hand-over; binned: [0, 1] = the TrkBin
    int64_t bc_i64[2];              // binned: [1] = the open bin's partial result (a double) carried to the next sub-pass
    float bc_f32;
    alignas(16) unsigned char big_ctx[128];  // TileCtx handed to the out-of-line sub-pass variant
};

__device__ __forceinline__ void stg_f8(float *p, float a, float b, float c, float d, float e, float f, float g, float h) {
    asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "f"(e),
                 "f"(f), "f"(g), "f"(h)
                 : "memory");
}

// sixteen 16-bit values as eight packed pairs (lower address = lower half): one 256-bit store
__device__ __forceinline__ void stg_b8(void *p, const uint32_t (&w)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
                 "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
                 : "memory");
}

// a track value as output element T (the only place where the output type matters to the value)
template <class T> __device__ __forceinline__ T to_out(float v);
template <> __device__ __forceinline__ float to_out<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 to_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half to_out<__half>(float v) { return __float2half_rn(v); }

// two values as one packed pair of 16-bit elements, a in the lower half (cvt.rn.{bf16,f16}x2.f32: the rounding of to_out)
template <class T> __device__ __forceinline__ uint32_t pack2(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float a, float b) {
    const __nv_bfloat162 x = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&x);
}
template <> __device__ __forceinline__ uint32_t pack2<__half>(float a, float b) {
    const __half2 x = __floats2half2_rn(a, b);
    return *reinterpret_cast<const uint32_t *>(&x);
}

// ---- sources ---------------------------------------------------------------------------------------------
// source seen by the generic path and the fall-backs: the global arrays.  Value of the painted source track at relative
// position tp: dense windows, or the last interval with start <= q_start + tp if it also ends after it (intervals of a
// slot are sorted by start and do not overlap: overlapping slots are flattened when the track is uploaded)
struct SrcGlobal {
    const int32_t *its, *ite;  // the track's interval SoA (global memory)
    const float *itv;
    const float *dense;        // non-NULL: dense f32 source windows instead
    int64_t itv_lo, itv_hi, q_start, track_n;
    __device__ __forceinline__ float at(int64_t tp) const {
        if (tp < 0 || tp >= track_n) return 0.0f;  // out of contract in the reference (index panic)
        if (dense) return dense[itv_lo + tp];      // dense source: `itv_lo` is the window's offset
        const int64_t g = q_start + tp;
        int64_t a = itv_lo, b = itv_hi;  // last i in [lo, hi) with starts[i] <= g
        while (a < b) {
            const int64_t mid = (a + b) >> 1;
            if ((int64_t)its[mid] <= g) a = mid + 1; else b = mid;
        }
        const int64_t i = a - 1;
        if (i < itv_lo) return 0.0f;
        return ((int64_t)ite[i] > g) ? itv[i] : 0.0f;
    }
};

// source seen by the fast path: the pass's staged intervals first (shared memory), the global arrays otherwise
struct SrcStaged {
    const int32_t *its, *ite;  // staged arrays, already offset to the first staged interval
    const float *itv;
    int cnt;
    bool more, from_first;     // intervals follow the staged ones / the staged ones start at the slot's first interval
    const SrcGlobal &G;
    int64_t track_n;
    __device__ __forceinline__ float at(int64_t tp) const {
        if (tp < 0 || tp >= track_n) return 0.0f;
        const int64_t g = G.q_start + tp;
        if (cnt > 0 && g >= (int64_t)its[0]) {
            int lo = 0, hi = cnt;  // last staged interval with start <= g
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if ((int64_t)its[mid] <= g) lo = mid; else hi = mid;
            }
            if ((int64_t)ite[lo] > g) return itv[lo];
            if (lo < cnt - 1 || !more) return 0.0f;  // the next interval starts beyond g, or there is none
        } else if (from_first && (cnt > 0 || !more)) {
            return 0.0f;  // left of the slot's first interval (or the slot is empty)
        }
        return G.at(tp);
    }
};

// Lagrange interpolation through K anchors on each side of the insertion (src/tracks/mod.rs:138-188), evaluated at
// index i of the written values; same operation order as the reference (term = y_a * prod_b (x - x_b) / (x_a - x_b)).
template <int K, class Src>
__device__ __forceinline__ float lagrange_fill(const Src &S, int64_t v_len, int64_t v_rel_pos, int64_t i) {
    double xs[2 * K], ys[2 * K];
#pragma unroll
    for (int j = 0; j < K; j++) {
        xs[j] = -(double)j;
        ys[j] = (double)S.at(imax64(v_rel_pos - j, 0));
        xs[K + j] = (double)v_len + (double)j;
        ys[K + j] = (double)S.at(imin64(v_rel_pos + 1 + j, S.track_n - 1));
    }
    const double x = (double)i;
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 2 * K; a++) {
        double term = ys[a];
#pragma unroll
        for (int b = 0; b < 2 * K; b++) {
            if (b == a) continue;
            term = __dmul_rn(term, __ddiv_rn(__dsub_rn(x, xs[b]), __dsub_rn(xs[a], xs[b])));
        }
        acc = __dadd_rn(acc, term);
    }
    return (float)acc;
}

// apply_insertion_fill, src/tracks/mod.rs:87-190, for ONE written value (index i within the write).
template <class Src>
__device__ __forceinline__ float insertion_fill_value(const Src &S, int strategy, double param, int64_t v_len, int64_t v_rel_pos,
                                                   int64_t i, int64_t out_pos, uint64_t base_seed, uint64_t query, uint64_t hap) {
    if (strategy == GVL_FILL_REPEAT_5P) {
        return S.at(v_rel_pos);
    } else if (strategy == GVL_FILL_REPEAT_5P_NORM) {
        return __fdiv_rn(S.at(v_rel_pos), (float)v_len);  // :115
    } else if (strategy == GVL_FILL_CONSTANT) {
        return (float)param;  // :121
    } else if (strategy == GVL_FILL_FLANK_SAMPLE) {  // :125-137
        int64_t width = (int64_t)param;
        int64_t pool_lo = imax64(v_rel_pos - width, 0);
        int64_t pool_hi = imin64(v_rel_pos + width, S.track_n - 1);
        uint64_t pool_size = (uint64_t)(pool_hi - pool_lo + 1);
        uint64_t seed = hash4(base_seed, query, hap, (uint64_t)out_pos);
        int64_t offset = (int64_t)(seed % pool_size);
        return S.at(pool_lo + offset);
    } else {  // GVL_FILL_INTERPOLATE :138-188
        const int64_t order = (int64_t)param;
        const int64_t k = (order + 1 + 1) / 2;
        // k anchors on each side: 2 anchors for order 1, 4 for orders 2 and 3 -- fixed-size instantiations keep the
        // anchors in registers and let the divisions overlap; the operation order is the reference's
        return k == 1 ? lagrange_fill<1>(S, v_len, v_rel_pos, i) : lagrange_fill<2>(S, v_len, v_rel_pos, i);
    }
}

// ---- generic path ------------------------------------------------------------------------------------------
// output value at haplotype position p of a row, resolved against the row's records in GLOBAL memory.  `hint` caches
// the record found last (positions of one thread advance monotonically).
__device__ float t2_generic_value(const TRec *__restrict__ recs, int32_t n_rec, int32_t ref0, const SrcGlobal &src,
                                  int strategy, double param, int32_t p, uint64_t base_seed, uint64_t qseed, uint64_t hap, int32_t &hint) {
    // i = last record with a <= p, -1 = before every record (the virtual record: span from ref0)
    int32_t i = hint;
    if (!(i >= -1 && i < n_rec && (i < 0 || recs[i].a <= p) && (i + 1 >= n_rec || recs[i + 1].a > p))) {
        int32_t lo = -1, hi = n_rec;
        while (hi - lo > 1) {
            const int32_t mid = (lo + hi) >> 1;
            if (recs[mid].a <= p) lo = mid; else hi = mid;
        }
        i = lo;
    }
    hint = i;
    if (i < 0) return src.at((int64_t)ref0 + p);
    const TRec r = recs[i];
    if (p < r.e) {  // values written by the variant itself (src/tracks/mod.rs:329-354)
        if (r.vdiff > 0 && strategy != GVL_FILL_REPEAT_5P)
            return insertion_fill_value(src, strategy, param, r.vlen, r.vrel, p - r.a, p, base_seed, qseed, hap);
        return src.at(r.vrel);
    }
    const int64_t tp = (int64_t)r.resume + (p - r.e);
    return tp < src.track_n ? src.at(tp) : 0.0f;  // :381-404 trailing zeros
}

template <class T>
__device__ __noinline__ void t2_generic_segment(const TRec *__restrict__ recs, int32_t n_rec, int32_t ref0, SrcGlobal src,
                                                int strategy, double param, T *__restrict__ out_row, int32_t L, bool rc, int32_t t0, int32_t t1,
                                   uint64_t base_seed, uint64_t qseed, uint64_t hap) {
    int32_t hint = -2;
    for (int32_t j = t0 + (int32_t)threadIdx.x; j < t1; j += T2_THREADS) {
        const int32_t p = rc ? (L - 1 - j) : j;
        // (one element per store: a 16-bit value never touches its neighbour)
        out_row[j] = to_out<T>(t2_generic_value(recs, n_rec, ref0, src, strategy, param, p, base_seed, qseed, hap, hint));
    }
}

// ---- fast path helpers -------------------------------------------------------------------------------------
// haplotype position at which relative source position x appears, given the staged records R[0..m) (R[0] = carry).
// dropped = x is not copied (inside a deletion, or behind the carry span); the returned position is then the first
// one whose source lies beyond x.
__device__ __forceinline__ int32_t t2_map(const TRec *R, int m, int32_t x, bool &dropped) {
    if (x < R[0].resume) {
        dropped = true;
        return R[0].e;
    }
    int lo = 0, hi = m;  // last staged record with resume <= x
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (R[mid].resume <= x) lo = mid; else hi = mid;
    }
    if (lo + 1 < m && x > R[lo + 1].vrel) {  // deleted by the next record
        dropped = true;
        return R[lo + 1].e;
    }
    dropped = false;
    return R[lo].e + (x - R[lo].resume);
}

__device__ __forceinline__ void t2_set_bit(uint32_t *mk, uint32_t *mk2, int u) {
    const uint32_t old = atomicOr(&mk[u >> 5], 1u << (u & 31));
    if (old == 0) atomicOr(&mk2[u >> 10], 1u << ((u >> 5) & 31));
}

// ---- binned store ------------------------------------------------------------------------------------------
// Bins of B = 1 << shift output positions; bin k of a row covers its positions [k B, (k + 1) B) and is stored at
// out_bins[k].  Values are combined in float64 (sum, mean) or as float32 values held in float64 (max, NaN first), in an
// order fixed by the row alone: sequentially over each 16-position chunk of the row (haplotype order), then a fixed
// tree over the chunks of a bin (xor shuffles, then warps in order), and across the sub-passes of a TD_BIG tile in
// haplotype order.  The tile geometry is a function of the row, so a row's bins have the same bits in every call.
struct TrkBin {
    int32_t shift, reduce;  // log2 of the bin size; GVL_TRACK_REDUCE_*
};

__device__ __forceinline__ double bin_op(int32_t reduce, double a, double b) {
    if (reduce != GVL_TRACK_REDUCE_MAX) return __dadd_rn(a, b);
    if (a != a) return a;  // NaN propagates
    if (b != b) return b;
    return b > a ? b : a;
}

// One (sub-)pass [cur, pass_end) (haplotype positions) of a tile, binned.  The CTA walks the pass in row-aligned chunks
// of 16 output positions, T2_THREADS chunks per round (whole bins: B divides 16 * T2_THREADS), every thread calling
// begin(j) for its chunk at output position j and then next(i, valid) for i = 0..15: the value at haplotype position
// (RC ? L - 16 - j : j) + i.  Every thread runs the same rounds (the barriers of bins that span warps).
template <class T, class Begin, class Next>
__device__ __forceinline__ void t3_bin_pass(T3Smem &S, T *__restrict__ out_bins, bool rc, int32_t L, int32_t cur, int32_t pass_end,
                                            TrkBin bn, Begin &&begin, Next &&next) {
    const int tid = threadIdx.x, lane = tid & 31;
    const int32_t B = 1 << bn.shift;
    const int32_t jo_lo = rc ? L - pass_end : cur, jo_hi = rc ? L - cur : pass_end;  // the pass in output positions
    const int32_t jb = jo_lo & ~(max(B, 16) - 1);
    const int32_t n_chunks = (jo_hi - jb + 15) >> 4;
    const double id = bn.reduce == GVL_TRACK_REDUCE_MAX ? __longlong_as_double((long long)0xfff0000000000000ull) : 0.0;  // -inf
    // a sub-pass that starts inside a bin continues the previous one's partial result; one that ends inside a bin leaves it
    const bool contd = (cur & (B - 1)) != 0, open = (pass_end & (B - 1)) != 0;
    const int32_t k_in = (rc ? L - 1 - cur : cur) >> bn.shift, k_out = (rc ? L - pass_end : pass_end - 1) >> bn.shift;
    double *carry = reinterpret_cast<double *>(&S.bc_i64[1]);
    const double carry_in = contd ? *carry : id;
    if (contd && open) __syncthreads();  // (read before it is rewritten)
    auto finish = [&](int32_t bs, double v) {  // the bin at output position bs, reduced over the pass's positions in it
        if (bs >= jo_hi || bs + B <= jo_lo || bs + B > L) return;
        const int32_t k = bs >> bn.shift;
        if (contd && k == k_in) v = bin_op(bn.reduce, carry_in, v);
        if (open && k == k_out) {
            *carry = v;
            return;
        }
        if (bn.reduce == GVL_TRACK_REDUCE_MEAN) v = __ddiv_rn(v, (double)B);
        out_bins[k] = to_out<T>((float)v);
    };
    double *wpart = reinterpret_cast<double *>(S.itv);  // per-warp results (the staged intervals are no longer read)
    const int n_rounds = (n_chunks + T2_THREADS - 1) / T2_THREADS;
    for (int it = 0; it < n_rounds; it++) {
        const int32_t j = jb + 16 * (it * T2_THREADS + tid);
        const int32_t vlo = max(jo_lo - j, 0), vhi = min(jo_hi - j, 16);  // chunk values inside the pass
        double acc = id;
        if (vlo < vhi) {
            begin(j);
#pragma unroll
            for (int i = 0; i < 16; i++) {
                const int32_t o = rc ? 15 - i : i;  // output position j + o
                const bool valid = o >= vlo && o < vhi;
                const float x = next(i, valid);
                if (valid) acc = bin_op(bn.reduce, acc, (double)x);
                if (B < 16 && ((i + 1) & (B - 1)) == 0) {
                    finish(rc ? j + 15 - i : j + i + 1 - B, acc);
                    acc = id;
                }
            }
        }
        if (B >= 16) {
            const int G = min(B >> 4, 32);  // chunks of a bin within a warp
            for (int o = 1; o < G; o <<= 1) acc = bin_op(bn.reduce, acc, __shfl_xor_sync(0xffffffffu, acc, o));
            if (B <= 512) {
                if ((lane & (G - 1)) == 0) finish(j, acc);
            } else {
                if (lane == 0) wpart[tid >> 5] = acc;
                __syncthreads();
                const int W = B >> 9;  // warps of a bin
                if (tid < (T2_THREADS / 32) / W) {
                    double v = wpart[tid * W];
                    for (int w = 1; w < W; w++) v = bin_op(bn.reduce, v, wpart[tid * W + w]);
                    finish(jb + 16 * (it * T2_THREADS + tid * W * 32), v);
                }
                __syncthreads();
            }
        }
    }
}

// t2_generic_segment, binned: the tile [h0, h1) (haplotype positions) in one pass
template <class T>
__device__ __noinline__ void t2_generic_bins(const TRec *__restrict__ recs, int32_t n_rec, int32_t ref0, SrcGlobal src, int strategy,
                                             double param, T3Smem *S, T *__restrict__ out_bins, int32_t L, bool rc, int32_t h0,
                                             int32_t h1, uint64_t base_seed, uint64_t qseed, uint64_t hap, TrkBin bn) {
    int32_t hint = -2, hb = 0;
    t3_bin_pass<T>(*S, out_bins, rc, L, h0, h1, bn, [&](int32_t j) { hb = rc ? L - 16 - j : j; },
                   [&](int i, bool valid) {
                       return valid ? t2_generic_value(recs, n_rec, ref0, src, strategy, param, hb + i, base_seed, qseed, hap, hint) : 0.0f;
                   });
}

// =====================================================================================
// tile preparation: one warp per (track, tile)
// =====================================================================================
// row_dst / row_tstride (GVL_TRACK_LAYOUT_ROWS): explicit destination of every row, out_base = row_dst[row] + track *
// row_tstride[row]; NULL row_dst = the fixed layout of P.layout_btp.  (Kernel arguments of their own, not members of
// TrkExecParams: the execute kernel takes the same struct, and a larger struct would move its tdesc argument.)
__global__ void __launch_bounds__(128) trk_tile_prep_kernel(TrkExecParams P, const int64_t *__restrict__ row_dst,
                                                            const int64_t *__restrict__ row_tstride, TileDesc *__restrict__ tdesc) {
    // one WARP per (track, tile): the searches are 32-ary (a probe per lane), the record counts one strided pass
    const int lane = threadIdx.x & 31;
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (g >= P.grid_per_track * P.n_tracks) return;
    const int64_t track = g / P.grid_per_track;
    const int64_t b = g % P.grid_per_track;
    TileDesc D;
    D.row = -1;
    if (b < P.tile_off[P.n_work]) {
        int64_t lo = 0, hi = P.n_work;  // row of the tile: last row with tile_off[row] <= b
        while (hi - lo > 1) {           // (32-ary: lane l probes the l-th of 32 cut points)
            const int64_t step = (hi - lo + 31) / 32;
            const int64_t idx = lo + (int64_t)(lane + 1) * step;
            const bool ok = idx < hi && P.tile_off[idx] <= b;
            const int cnt = __popc(__ballot_sync(0xffffffffu, ok));  // probes are monotone
            const int64_t nlo = lo + (int64_t)cnt * step;
            hi = imin64(hi, nlo + step);
            lo = nlo;
        }
        const int64_t row = lo, tile = b - P.tile_off[row];
        const RowPlan rp = P.rows[row];
        const int32_t L = rp.length;
        const int32_t t0 = (int32_t)(tile * T3_TILE);
        if (t0 < L) {
            const int32_t t1 = (int32_t)imin64((int64_t)t0 + T3_TILE, L);
            const bool rc = rp.rc != 0;
            const int64_t query = row / P.ploidy;
            const TrkDesc &T = P.tracks ? P.tracks[track] : P.inl[track];
            D.row = (int32_t)row;
            D.L = L;
            D.h0 = rc ? L - t1 : t0;  // the tile in haplotype coordinates
            D.h1 = rc ? L - t0 : t1;
            D.q_start = rp.q_start;
            D.track_n = rp.contig_len;
            D.ref0 = rp.ref0;
            D.rec_base = rp.rec_off;
            D.n_rec = rp.n_rec;
            D.flags = (rc ? TD_RC : 0) | ((T.dense || (rp.lead_pad & FLAG_JUMPS)) ? TD_GENERIC : 0);
            D.query = (int32_t)query;
            D.src_lo = D.src_hi = 0;
            D.m = 1;
            D.cnt = 0;
            int64_t row_base = track * P.total_per_track + rp.out_off;  // flat index of the row's first value
            if (row_dst) {
                row_base = row_dst[row] + track * row_tstride[row];
            } else if (P.layout_btp) {  // all tracks of a query adjacent: block of the query, then track, then the row inside the block
                const int64_t k0 = query * P.ploidy;
                const int64_t blk0 = P.rows[k0].out_off;
                const int64_t blk_len = P.rows[k0 + P.ploidy - 1].out_off + P.rows[k0 + P.ploidy - 1].length - blk0;
                row_base = P.n_tracks * blk0 + track * blk_len + (rp.out_off - blk0);
            }
            D.out_base = row_base;
            if (T.dense) {
                D.it_lo = T.dense_offsets[query];
                D.it_hi = T.dense_offsets[query + 1];
                D.it0 = D.it_lo;
                D.r = -1;
                D.val0 = 0.0f;
            } else {
                const int64_t slot = P.offset_idxs[track * P.n_queries + query];
                D.it_lo = T.itv_offsets[slot];
                D.it_hi = T.itv_offsets[slot + 1];
                // carry record (last with a <= h0) and last record that starts inside the tile (a < h1): one strided
                // pass over the row's sorted records (independent loads)
                const TRec *__restrict__ recs = P.trecs + rp.rec_off;
                int c0 = 0, c1 = 0;
                for (int i = lane; i < rp.n_rec; i += 32) {
                    const int32_t a = recs[i].a;
                    c0 += (a <= D.h0);
                    c1 += (a < D.h1);
                }
                const int32_t rl = __reduce_add_sync(0xffffffffu, c0) - 1;
                const int32_t el = max(__reduce_add_sync(0xffffffffu, c1) - 1, rl);
                D.r = rl;
                int64_t src = (int64_t)rp.ref0 + D.h0;  // source position that feeds h0
                if (rl >= 0) {
                    const TRec cr = recs[rl];
                    src = D.h0 < cr.e ? (int64_t)cr.vrel : (int64_t)cr.resume + (D.h0 - cr.e);
                }
                D.m = 1 + (el - rl);
                int64_t src_hi = (int64_t)rp.ref0 + D.h1;  // ... and the one that feeds h1
                if (el >= 0) {
                    const TRec cr = recs[el];
                    src_hi = D.h1 <= cr.e ? (int64_t)cr.vrel + 1 : (int64_t)cr.resume + (D.h1 - cr.e);
                }
                D.src_lo = (int32_t)src;
                D.src_hi = (int32_t)src_hi;
                // first interval whose end lies beyond src (ends are sorted: the slot's intervals do not overlap) ...
                const int64_t gpos = (int64_t)rp.q_start + src;
                const int64_t a = warp_upper_le(T.itv_ends, D.it_lo, D.it_hi, (int32_t)imax64(imin64(gpos, INT32_MAX), INT32_MIN)) + 1;
                D.it0 = a;
                D.val0 = (src >= 0 && src < (int64_t)rp.contig_len && a < D.it_hi && (int64_t)T.itv_starts[a] <= gpos) ? T.itv_values[a] : 0.0f;
                // ... and the first one that starts at or beyond src_hi: the tile needs the intervals in between
                const int64_t ghi = (int64_t)rp.q_start + src_hi;
                const int64_t c = warp_upper_le(T.itv_starts, a, D.it_hi, (int32_t)imax64(imin64(ghi - 1, INT32_MAX), INT32_MIN)) + 1;
                D.cnt = (int32_t)imin64(c - a, INT32_MAX);
                if (D.m > T3_REC || c - a > T3_ITV) D.flags |= TD_BIG;
                // the execute CTA of this tile reads these next: have them in L2 by then
                const int64_t n_pf = imin64(c - a, T3_ITV);
                for (int64_t o = ((a * 4) & ~(int64_t)127) + 128 * lane; o < (a + n_pf) * 4; o += 128 * 32) {
                    asm volatile("prefetch.global.L2 [%0];" ::"l"((const char *)T.itv_starts + o));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"((const char *)T.itv_ends + o));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"((const char *)T.itv_values + o));
                }
            }
        }
    }
    if (lane == 0) tdesc[g] = D;
}

// =====================================================================================
// execute: one CTA per tile
// =====================================================================================
// the output phase of a (sub-)pass: see the header comment
template <bool RC, class T>
__device__ __forceinline__ void t3_write_chunks(const T3Smem &S, T *__restrict__ out_row, int32_t j0, int32_t n_chunks,
                                                int32_t jo_lo, int32_t jo_hi, int32_t L, int32_t cur) {
    // Every thread owns 16 consecutive output values (float: 64 bytes, two 256-bit stores; lanes 64 bytes apart still run
    // at the full store rate on B200, 128 bytes per lane do not -- profiles/microbench/fill.py), so the search for the
    // value in effect before the chunk is paid once per 16 values and the walk carries it in a register.
    // 16-bit output keeps the 16 values per thread: ONE 256-bit store of packed pairs, lanes 32 bytes apart (a warp
    // instruction still writes 1 KiB of contiguous output).  32 values per thread would halve the chunk searches but
    // double the marker walk each thread runs before its first store and halve the threads that store a tile; the
    // kernel is bound by that per-tile latency chain, not by the searches, and one chunk geometry for every T keeps the
    // walk, the bitmap reads and the tile-edge handling the same code.
    const uint32_t *mk = S.mk, *mk2 = S.mk2;
    const int tid = threadIdx.x;
    int32_t j = j0 + 16 * tid;                          // first output position of the thread's chunk
    int32_t u_lo = (RC ? (L - 16 - j) : j) - cur;       // its lowest tile-relative haplotype position
    T *dst = out_row + j;
    for (int32_t c = tid; c < n_chunks; c += T2_THREADS, j += 16 * T2_THREADS, u_lo += RC ? -16 * T2_THREADS : 16 * T2_THREADS,
                 dst += 16 * T2_THREADS) {
        uint32_t bits;
        if (u_lo >= 0) {
            const int w = u_lo >> 5;
            bits = __funnelshift_r(mk[w], mk[w + 1], u_lo & 31) & 0xffffu;
        } else {
            bits = (mk[0] << (-u_lo)) & 0xffffu;
        }
        float cv = 0.0f;
        const int q = max(u_lo, 0) - 1;  // last position before the chunk (position 0 always holds a marker)
        if (q >= 0) {
            int w = q >> 5;
            uint32_t mm = mk[w] & (0xffffffffu >> (31 - (q & 31)));
            if (mm == 0u) {
                int w2 = w >> 5;
                uint32_t m2 = mk2[w2] & ((1u << (w & 31)) - 1u);
                while (m2 == 0u) m2 = mk2[--w2];
                w = 32 * w2 + 31 - __clz(m2);
                mm = mk[w];
            }
            cv = S.val[32 * w + 31 - __clz(mm)];
        }
        const bool whole = j >= jo_lo && j + 16 <= jo_hi;
        if constexpr (sizeof(T) == 2) {
            float x[16];  // in OUTPUT order: haplotype position u_lo + i is output RC ? 15 - i : i of the chunk
#pragma unroll
            for (int i = 0; i < 16; i++) {
                if ((bits >> i) & 1u) cv = S.val[u_lo + i];
                x[RC ? 15 - i : i] = cv;
            }
            if (whole) {
                uint32_t w[8];
#pragma unroll
                for (int k = 0; k < 8; k++) w[k] = pack2<T>(x[2 * k], x[2 * k + 1]);
                stg_b8(dst, w);
            } else {  // chunk cut by the tile / row ends: one 16-bit store per value of the range, nothing outside it
#pragma unroll
                for (int t = 0; t < 16; t++) {
                    const int32_t jj = j + t;
                    if (jj >= jo_lo && jj < jo_hi) dst[t] = to_out<T>(x[t]);
                }
            }
        } else {
#pragma unroll
            for (int h = 0; h < 2; h++) {  // two halves of 8 in HAPLOTYPE order; the reversed row stores them back to front
                float x[8];                // in OUTPUT order: haplotype position u_lo + 8h + t is output RC ? 7 - t : t of its half
#pragma unroll
                for (int t = 0; t < 8; t++) {
                    if ((bits >> (8 * h + t)) & 1u) cv = S.val[u_lo + 8 * h + t];
                    x[RC ? 7 - t : t] = cv;
                }
                const int off = RC ? 8 * (1 - h) : 8 * h;
                if (whole) {
                    stg_f8(reinterpret_cast<float *>(dst + off), x[0], x[1], x[2], x[3], x[4], x[5], x[6], x[7]);
                } else {  // chunk cut by the tile / row ends
#pragma unroll
                    for (int t = 0; t < 8; t++) {
                        const int32_t jj = j + off + t;
                        if (jj >= jo_lo && jj < jo_hi) dst[off + t] = to_out<T>(x[t]);
                    }
                }
            }
        }
    }
}

// what a tile needs beyond its descriptor (built once by the kernel; small enough to travel by value)
template <class T>
struct TileCtx {
    const TRec *recs;      // the row's records
    T *out_row;            // the row's value 0
    int64_t base_elems;    // its address in elements of T (alignment of the 16-value chunks: 64 bytes for float, 32 for 16-bit)
    SrcGlobal srcg;
    uint64_t base_seed, qseed, hap;
    double param;
    int32_t strategy;
};

// One tile.  BIG = false: everything the tile needs fits the staging (the descriptor says how much of it): one pass,
// extents known.  BIG = true: sub-passes, each as long as the staged records / intervals reach.
template <bool BIG, class T, bool BIN = false>
__device__ __forceinline__ void t3_tile(const TileCtx<T> &X, const TileDesc &D, T3Smem &S, TrkBin bn = TrkBin{0, 0}) {
    const int tid = threadIdx.x;
    const int32_t L = D.L;
    const bool rc = (D.flags & TD_RC) != 0;
    const uint64_t hap = X.hap, qseed = X.qseed, base_seed = X.base_seed;
    const int64_t track_n = D.track_n, q_start = D.q_start;
    const TRec *__restrict__ recs = X.recs;
    const SrcGlobal &srcg = X.srcg;
    T *__restrict__ out_row = X.out_row;
    const int64_t base_elems = X.base_elems;
    const int32_t h1 = D.h1;
    int32_t cur = D.h0;
    int64_t r = D.r, it0 = D.it0;  // cursors: carry record (relative to the row, -1 = virtual), first staged interval
    float val0 = D.val0;
    for (;;) {
        // ---- load: two intervals per thread (registers + shared memory), the records, clean bitmaps ----
        const int cnt = BIG ? (int)imin64((int64_t)T3_ITV, imax64(D.it_hi - it0, 0)) : D.cnt;
        const bool more_itv = BIG && it0 + cnt < D.it_hi;  // (BIG = false: what follows the staged intervals lies beyond the tile)
        int32_t is[2], ie[2];
        float iv[2];
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int k = tid + q * T2_THREADS;
            is[q] = ie[q] = 0, iv[q] = 0.0f;
            if (k < cnt) {
                is[q] = __ldg(srcg.its + it0 + k);
                ie[q] = __ldg(srcg.ite + it0 + k);
                iv[q] = __ldg(srcg.itv + it0 + k);
            }
        }
        const int dst0 = r < 0 ? 1 : 0;
        const int64_t src0 = r < 0 ? 0 : r;
        const int n_ld = BIG ? (int)imin64((int64_t)(T3_REC - dst0), imax64((int64_t)D.n_rec - src0, 0)) : D.m - 1 + (1 - dst0);
        const int m = dst0 + n_ld;
        const bool more_rec = BIG && src0 + n_ld < (int64_t)D.n_rec;
        if (tid < n_ld) S.rec[dst0 + tid] = recs[src0 + tid];
        if (tid == 0 && dst0) {  // virtual carry: nothing written yet, the span starts at ref0
            TRec v;
            v.a = 0, v.e = 0, v.resume = D.ref0, v.vrel = D.ref0, v.vlen = 1, v.vdiff = 0, v.pad0 = 0, v.pad1 = 0;
            S.rec[0] = v;
        }
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int k = tid + q * T2_THREADS;
            S.its[k] = is[q], S.ite[k] = ie[q], S.itv[k] = iv[q];
        }
        for (int i = tid; i < T3_WORDS + 1; i += T2_THREADS) S.mk[i] = 0u;
        if (tid < T3_WORDS / 32) S.mk2[tid] = 0u;
        if (tid == 0) S.n_fill = 0;
        __syncthreads();

        // ---- extent of the sub-pass ----
        const TRec *R = S.rec;
        int32_t pass_end = h1;
        int m_eff = m;
        if (more_rec) {  // the last staged record is a sentinel: the sub-pass stops where it starts
            m_eff = m - 1;
            pass_end = min(pass_end, R[m - 1].a);
        }
        int32_t src_lo = D.src_lo, src_hi = D.src_hi;  // sources in [src_lo, src_hi) reach the (sub-)pass
        int m_pass = m;  // staged records that start inside the sub-pass (+ the carry): the only ones the mapping needs
        if (BIG) {
            const int32_t e0 = R[0].e;
            src_lo = cur < e0 ? R[0].vrel : R[0].resume + (cur - e0);
            if (more_itv) {  // likewise the last staged interval: nothing beyond its start is known
                bool dr;
                const int32_t hl = t2_map(R, m_eff, (int32_t)imax64((int64_t)S.its[cnt - 1] - q_start, 0), dr);
                pass_end = min(pass_end, max(hl, cur + 1));
            }
            int lo = 0, hi = m_eff;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (R[mid].a < pass_end) lo = mid; else hi = mid;
            }
            m_pass = lo + 1;
            const TRec rl = R[m_pass - 1];
            src_hi = pass_end <= rl.e ? rl.vrel + 1 : rl.resume + (pass_end - rl.e);
        }
        const int32_t plen = pass_end - cur;
        const SrcStaged src{S.its, S.ite, S.itv, cnt, BIG ? more_itv : (it0 + cnt < D.it_hi), it0 == D.it_lo, srcg, track_n};
        uint32_t *mk = S.mk, *mk2 = S.mk2;

        // ---- markers: intervals ----
        auto place = [&](int32_t x, float v) {
            bool dr;
            const int32_t h = t2_map(R, m_pass, x, dr);
            const int32_t u = h - cur;
            if (dr || u <= 0 || u >= plen) return;
            S.val[u] = v;
            t2_set_bit(mk, mk2, u);
        };
#pragma unroll
        for (int q = 0; q < 2; q++) {
            const int k = tid + q * T2_THREADS;
            if (k >= cnt) continue;
            // (clipped to the source window in 64 bits, 32-bit arithmetic from here on)
            const int32_t s = (int32_t)imin64(imax64((int64_t)is[q] - q_start, 0), track_n);
            const int32_t e = (int32_t)imax64(imin64((int64_t)ie[q] - q_start, track_n), 0);
            if (e <= s || e <= src_lo || s >= src_hi) continue;  // empty after clipping, behind the sub-pass, beyond it
            if (s > src_lo) place(s, iv[q]);  // (an interval that covers the first position is the start marker's)
            const bool adjacent = (k + 1 < cnt) && ((int64_t)S.its[k + 1] - q_start == (int64_t)e);  // the next interval starts right there
            if (!adjacent && e < src_hi) place(e, 0.0f);
        }
        // ---- markers: records (threads from the top of the CTA) + the first position ----
        bool need_fill = false;
        {
            const int i = T2_THREADS - 1 - tid;
            if (i < m_pass) {
                const TRec rr = R[i];
                const bool live = i == 0 ? (cur < rr.e) : true;
                if (live) {
                    if (rr.vdiff > 0 && X.strategy != GVL_FILL_REPEAT_5P) {
                        S.fill_list[atomicAdd(&S.n_fill, 1)] = i;
                        need_fill = true;
                    }
                    if (rr.e < pass_end && rr.e > cur) {  // value in effect right after the variant
                        S.val[rr.e - cur] = src.at(rr.resume);
                        t2_set_bit(mk, mk2, rr.e - cur);
                    }
                }
            } else if (i == m_pass) {
                S.val[0] = val0;
                t2_set_bit(mk, mk2, 0);
            }
        }
        // ---- insertion fills other than Repeat5p: one value per thread, dropped as markers ----
        if (__syncthreads_or(need_fill)) {
            const int warp = tid >> 5, lane = tid & 31;
            for (int f = warp; f < S.n_fill; f += T2_THREADS / 32) {
                const TRec rr = R[S.fill_list[f]];
                const int32_t lo = max(rr.a, cur), hi = min(rr.e, pass_end);
                for (int32_t p = lo + lane; p < hi; p += 32) {
                    S.val[p - cur] = insertion_fill_value(src, X.strategy, X.param, rr.vlen, rr.vrel, p - rr.a, p, base_seed, qseed, hap);
                    t2_set_bit(mk, mk2, p - cur);
                }
            }
            __syncthreads();
        }

        if constexpr (BIN) {
            // ---- binned output: chunks of 16 values on 16-position aligned ROW positions, the walk of t3_write_chunks ----
            int32_t u_lo = 0;
            uint32_t bits = 0u;
            float cv = 0.0f;
            t3_bin_pass<T>(S, out_row, rc, L, cur, pass_end, bn,
                           [&](int32_t j) {
                               u_lo = (rc ? (L - 16 - j) : j) - cur;
                               const uint32_t *mk = S.mk, *mk2 = S.mk2;
                               if (u_lo >= 0) {
                                   const int w = u_lo >> 5;
                                   bits = __funnelshift_r(mk[w], mk[w + 1], u_lo & 31) & 0xffffu;
                               } else {
                                   bits = (mk[0] << (-u_lo)) & 0xffffu;
                               }
                               cv = 0.0f;
                               const int q = max(u_lo, 0) - 1;
                               if (q >= 0) {
                                   int w = q >> 5;
                                   uint32_t mm = mk[w] & (0xffffffffu >> (31 - (q & 31)));
                                   if (mm == 0u) {
                                       int w2 = w >> 5;
                                       uint32_t m2 = mk2[w2] & ((1u << (w & 31)) - 1u);
                                       while (m2 == 0u) m2 = mk2[--w2];
                                       w = 32 * w2 + 31 - __clz(m2);
                                       mm = mk[w];
                                   }
                                   cv = S.val[32 * w + 31 - __clz(mm)];
                               }
                           },
                           [&](int i, bool) {
                               if ((bits >> i) & 1u) cv = S.val[u_lo + i];
                               return cv;
                           });
        } else {
        // ---- output: chunks of 16 values on 16-element (float: 64-byte, 16-bit: 32-byte) aligned addresses ----
        const int32_t jo_lo = rc ? L - pass_end : cur;
        const int32_t jo_hi = rc ? L - cur : pass_end;
        const int32_t j0 = (int32_t)(((base_elems + jo_lo) & ~(int64_t)15) - base_elems);  // may be < jo_lo
        const int32_t n_chunks = (jo_hi - j0 + 15) >> 4;
        // (the two directions are separate instantiations: the walk then writes its registers in output order)
        if (rc) t3_write_chunks<true, T>(S, out_row, j0, n_chunks, jo_lo, jo_hi, L, cur);
        else t3_write_chunks<false, T>(S, out_row, j0, n_chunks, jo_lo, jo_hi, L, cur);
        }
        if (!BIG || pass_end >= h1) break;

        // ---- (rare) the tile goes on: cursors of the next sub-pass ----
        // next carry = last staged record with a <= pass_end; staged intervals that end at or before the source
        // position feeding pass_end are history
        int lo = 0;
        {
            int hi = m;
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (R[mid].a <= pass_end) lo = mid; else hi = mid;
            }
        }
        const TRec cr = R[lo];
        const int64_t src_next = pass_end < cr.e ? (int64_t)cr.vrel : (int64_t)cr.resume + (pass_end - cr.e);
        src_lo = (int32_t)src_next;
        int behind = 0;
#pragma unroll
        for (int q = 0; q < 2; q++)
            behind += (tid + q * T2_THREADS < cnt && (int64_t)ie[q] - q_start <= src_next) ? 1 : 0;
        const int n_behind = __syncthreads_count(behind > 0) + __syncthreads_count(behind > 1);  // (also: everyone is done with S)
        if (tid == 0) {
            int64_t it_next = it0 + n_behind;
            if (n_behind == cnt && more_itv) {  // a long deletion skipped every staged interval: search the slot
                int64_t a = it_next, bb = D.it_hi;
                const int64_t gpos = q_start + src_next;
                while (a < bb) {
                    const int64_t mid = (a + bb) >> 1;
                    if ((int64_t)srcg.ite[mid] <= gpos) a = mid + 1; else bb = mid;
                }
                it_next = a;
            }
            S.bc_i64[0] = it_next;
            S.bc_f32 = srcg.at(src_next);  // value in effect at the first position of the next sub-pass
        }
        __syncthreads();
        it0 = S.bc_i64[0];
        val0 = S.bc_f32;
        r += lo;  // staged index i <-> row index r + i (staged[0] is the carry, also when it is the virtual one, r = -1)
        cur = pass_end;
        __syncthreads();  // the broadcast slots are read before the next sub-pass rewrites shared memory
    }
}

// (the rare sub-pass variant is kept out of line: its register needs must not weigh on the common path)
// (it takes its context from shared memory and re-reads the descriptor: structs passed by value or reference would
//  make every thread of EVERY tile spill them to local memory before the branch)
template <class T, bool BIN>
__device__ __noinline__ void t3_tile_big(T3Smem *S, const TileDesc *__restrict__ dp) {
    const TileCtx<T> X = *reinterpret_cast<const TileCtx<T> *>(S->big_ctx);
    const TileDesc D = *dp;
    if constexpr (BIN) {
        const TrkBin bn{S->bc_i32[0], S->bc_i32[1]};
        __syncthreads();  // everyone holds its copy before shared memory is reused
        t3_tile<true, T, true>(X, D, *S, bn);
    } else {
        __syncthreads();  // everyone holds its copy before shared memory is reused
        t3_tile<true, T>(X, D, *S);
    }
}
static_assert(sizeof(TileCtx<float>) <= 128, "TileCtx must fit T3Smem::big_ctx");

// 5 CTAs per SM (48 registers, 80 bytes of spills; shared memory allows no more): the kernel is bound by the latency chain of a
// tile, so the fifth tile in flight pays (tracks step of a 20-batch ring 63.7 -> 60.3 us) although a single 134 MB call gains little
constexpr int T3_MIN_CTAS = 5;
// BIN: the binned store (bn); the row's bins start at out + out_base / B (row offsets are multiples of B)
template <class T, bool BIN>
__global__ void __launch_bounds__(T2_THREADS, T3_MIN_CTAS) trk_exec3_kernel(TrkExecParams P, const TileDesc *__restrict__ tdesc, TrkBin bn) {
    __shared__ __align__(16) T3Smem S;
    const unsigned track = blockIdx.y;
    const TileDesc *dp = tdesc + ((size_t)track * (size_t)P.grid_per_track + blockIdx.x);
    const TileDesc D = *dp;  // (same address in every thread: one broadcast load)
    if (D.row < 0) return;
    const TrkDesc *Tp = P.tracks ? P.tracks + track : nullptr;
    TileCtx<T> X;
    {
        const int64_t query = D.query;
        // (queries and logical batch sizes are < 2^31: 32-bit division, the 64-bit one was 8 % of the kernel's instructions)
        const uint32_t sub = P.sub_batch > 0 ? (uint32_t)P.sub_batch : 0u;
        const uint32_t q_blk = sub ? (uint32_t)D.query / sub : 0u;
        X.hap = (uint64_t)(D.row - D.query * (int32_t)P.ploidy);
        X.qseed = P.query_seed ? (uint64_t)P.query_seed[query] : (uint64_t)(sub ? (uint32_t)D.query - q_blk * sub : (uint32_t)D.query);
        X.base_seed = P.base_seed_dev ? P.base_seed_dev[q_blk] : P.base_seed;
        X.recs = P.trecs + D.rec_base;
        X.out_row = static_cast<T *>(P.out) + (BIN ? D.out_base >> bn.shift : D.out_base);
        X.base_elems = (int64_t)(reinterpret_cast<uintptr_t>(P.out) / sizeof(T)) + D.out_base;
        // (kernel parameters are indexed with a compile-time subscript: a run-time one would copy them to local memory)
        const TrkDesc *Td = Tp;
#define GVL_TRK_PICK(i) case i: if (!Tp) { X.srcg.its = P.inl[i].itv_starts; X.srcg.ite = P.inl[i].itv_ends; X.srcg.itv = P.inl[i].itv_values; \
                                           X.srcg.dense = P.inl[i].dense; X.strategy = P.inl[i].strategy; X.param = P.inl[i].param; } break;
        switch (track) {
            GVL_TRK_PICK(0) GVL_TRK_PICK(1) GVL_TRK_PICK(2) GVL_TRK_PICK(3) GVL_TRK_PICK(4) GVL_TRK_PICK(5) GVL_TRK_PICK(6) GVL_TRK_PICK(7)
            default: break;
        }
#undef GVL_TRK_PICK
        if (Td) {
            X.srcg.its = Td->itv_starts, X.srcg.ite = Td->itv_ends, X.srcg.itv = Td->itv_values, X.srcg.dense = Td->dense;
            X.strategy = Td->strategy, X.param = Td->param;
        }
        X.srcg.itv_lo = D.it_lo, X.srcg.itv_hi = D.it_hi, X.srcg.q_start = D.q_start, X.srcg.track_n = D.track_n;
    }
    if (D.flags & TD_GENERIC) {
        const int32_t L = D.L;
        const bool rc = (D.flags & TD_RC) != 0;
        const int32_t t0 = rc ? L - D.h1 : D.h0, t1 = rc ? L - D.h0 : D.h1;
        if constexpr (BIN)
            t2_generic_bins(X.recs, D.n_rec, D.ref0, X.srcg, X.strategy, X.param, &S, X.out_row, L, rc, D.h0, D.h1, X.base_seed, X.qseed,
                            X.hap, bn);
        else
            t2_generic_segment(X.recs, D.n_rec, D.ref0, X.srcg, X.strategy, X.param, X.out_row, L, rc, t0, t1, X.base_seed, X.qseed, X.hap);
        return;
    }
    if (D.flags & TD_BIG) {
        if (threadIdx.x == 0) {
            *reinterpret_cast<TileCtx<T> *>(S.big_ctx) = X;
            if constexpr (BIN) S.bc_i32[0] = bn.shift, S.bc_i32[1] = bn.reduce;
        }
        __syncthreads();
        t3_tile_big<T, BIN>(&S, dp);
    } else {
        t3_tile<false, T, BIN>(X, D, S, bn);
    }
}
