// gvl_hap_oh.cuh -- execute kernel for the (L,4) one-hot output over the PACKED reference.
//
// The packed reference holds one 4-bit code per base (A=1, C=2, G=4, T=8, anything else 0; base r of the
// concatenated reference is nibble r&7 of word r>>3, low nibble first).  It is built once per dataset from the
// ASCII reference (pack_ref_kernel, gvl_dev_pack_reference) and makes the fused epilogue of
// reconstruct_haplotypes_fused + seqpro.DNA.ohe (src/ffi/mod.rs:724-860, docs/source/index.md:108-119) cheap:
//   * one lane owns 8 consecutive output positions: two aligned 32-bit loads + one funnel shift fetch their 8 codes
//     whatever the indel shift of the row is;
//   * reverse-complement of the 8 positions (src/reverse.rs:45-69) is ONE bit reversal (brev): reversing the nibble
//     order reverses the positions, reversing the bits inside a nibble swaps A<->T and C<->G;
//   * a 256-entry shared-memory table maps a byte (2 codes) to its 8 one-hot bytes: 4 lookups per lane, at swizzled
//     indices so that the bytes of A/C/G/T fall into distinct banks (oh_swizzle);
//   * the lane's 32 output bytes leave with one 256-bit store (STG.256): a warp writes 1 KiB per instruction.
// Groups of 256 positions that are plain reference (the common case) take exactly that path; groups that contain
// a variant, a pad or a tile edge classify every lane on its own, and only the lanes that straddle a record edge
// rebuild their 8 codes piecewise (ALT bytes come from the ASCII allele buffer) before the common epilogue.
//
// Included by gvl_hap.cu (shares HapExecParams / find_rec with the byte-oriented kernel, which keeps serving the
// u8, annotated and channels-first modes and callers without a packed reference).
#pragma once

namespace gvl {

constexpr int OH_GROUP = 256;                                  // positions per warp step (8 per lane)
// (round 1 capped tiles at 16,384: its launches were single batches.  A ring launch has thousands of CTAs, and a CTA's fixed
//  cost -- ~3.3 us of dependent round trips and barriers before its first store -- is worth amortising over twice the positions:
//  cfg3 execute 272 -> 259 us per 20 batches.  The launch code shortens tiles again when variants are dense.)
constexpr int OH_MAX_TILE_WANTED = 32768;                      // haplotype positions per CTA, at most

constexpr int OH_THREADS = 128;                                // threads per CTA of the packed kernel
// 4-warp CTAs per SM the register budget is sized for (64 registers at 8, 72 at 6).  The unroll-4 kernel of long sparse rows
// runs faster at 6 (cfg3: 384 -> 380 us per 32-batch launch; 5 CTAs: 414 us, 10 CTAs at 48 registers: 425 us), the unroll-2
// kernel of dense rows needs the 8 to hide its record lookups (cfg2d at 6: 994 us per launch against 877 us for the kernel
// before the swizzle, in one call) -- profiles/r3_oh_swizzle.md
constexpr int OH_MIN_CTAS = 8;
constexpr int OH_MIN_CTAS_LONG = 6;
// one thread per group builds the group table: a pass may not touch more groups than the CTA has threads
constexpr int OH_MAX_TILE = OH_MAX_TILE_WANTED < (OH_THREADS - 2) * OH_GROUP ? OH_MAX_TILE_WANTED : (OH_THREADS - 2) * OH_GROUP / 1024 * 1024;
constexpr int OH_MAX_GROUPS = OH_MAX_TILE / OH_GROUP + 2;      // groups a pass can touch (+ misaligned edges)
static_assert(OH_MAX_GROUPS <= OH_THREADS && OH_MAX_TILE >= 1024, "group table: one thread per group");
constexpr int OH_UNROLL_LONG = 4;                              // groups per warp whose loads are issued together (long sparse rows)

struct OhRecs {
    int32_t a[REC_CAP + 2];   // ALT start (haplotype coordinate); a[m], a[m+1] sentinels
    int32_t e[REC_CAP];       // ALT end = start of the following reference span
    int32_t resume[REC_CAP];  // reference position at e[]
    int64_t src[REC_CAP];     // ALT source (offset into alt_alleles), ALT_PAD for the leading pad
};

// 4-bit one-hot code of an ASCII base
__host__ __device__ __forceinline__ uint32_t nib_code(uint32_t b) {
    return (b == 'A' ? 1u : 0u) | (b == 'C' ? 2u : 0u) | (b == 'G' ? 4u : 0u) | (b == 'T' ? 8u : 0u);
}

__global__ void __launch_bounds__(256) pack_ref_kernel(const uint8_t *__restrict__ ref, int64_t n_bases,
                                                       uint32_t *__restrict__ out, int64_t n_words) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += stride) {
        const int64_t b0 = w * 8;
        uint32_t v = 0;
        if (b0 + 8 <= n_bases) {
            const uint2 x = *reinterpret_cast<const uint2 *>(ref + b0);  // (ref is 16-byte aligned)
#pragma unroll
            for (int t = 0; t < 4; t++) {
                v |= nib_code((x.x >> (8 * t)) & 0xffu) << (4 * t);
                v |= nib_code((x.y >> (8 * t)) & 0xffu) << (4 * (t + 4));
            }
        } else {
            for (int t = 0; t < 8; t++)
                if (b0 + t < n_bases) v |= nib_code(ref[b0 + t]) << (4 * t);
        }
        out[w] = v;
    }
}

// Index of the one-hot table entry of each byte of x (two codes per byte; bytes are independent).  The 8-byte entries sit
// in 16 bank pairs, entry i in pair i mod 16, and the low code of an ACGT byte takes only 4 values (1, 2, 4, 8): with the
// byte as index, the 16 ACGT x ACGT bytes share 4 bank pairs and a warp's lookup of random sequence replays to ~7
// shared-memory wavefronts.  XOR-ing bits of the high code into the low nibble puts those 16 bytes into 16 distinct bank
// pairs (2 wavefronts, the minimum for 32 lanes x 8 bytes).  A bijection on 0..255: the high nibble is kept, and for a
// fixed high nibble the low one maps by a triangular XOR (bit 0 ^= bit 3; bits 1..3 ^= bits of the high nibble).
__host__ __device__ __forceinline__ uint32_t oh_swizzle(uint32_t x) {
    return x ^ ((x >> 3) & 0x0F0F0F0Fu) ^ ((x >> 4) & 0x0E0E0E0Eu);
}

__device__ __forceinline__ uint2 lds_u64(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}

__device__ __forceinline__ void stg_256(void *p, const uint2 &o0, const uint2 &o1, const uint2 &o2, const uint2 &o3) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(o0.x), "r"(o0.y), "r"(o1.x),
                 "r"(o1.y), "r"(o2.x), "r"(o2.y), "r"(o3.x), "r"(o3.y)
                 : "memory");
}

// 8 codes starting at absolute base index n of the packed reference (nibble t = base n + t)
__device__ __forceinline__ uint32_t load_codes(const uint32_t *__restrict__ nib, int64_t n) {
    const uint32_t *w = nib + (n >> 3);
    return __funnelshift_r(__ldg(w), __ldg(w + 1), (uint32_t)n << 2);
}

// Codes of the haplotype positions [ps, pe) of a unit that starts at p_lo (nibble t = position p_lo + t), built
// piece by piece from the staged records; `il` = last staged record with a <= ps.  Semantics of the generic
// path of hap_exec_kernel (ALT bytes, leading pad, pure-deletion anchors, trailing pad past the contig end).
__device__ __noinline__ uint32_t oh_slow_unit(const OhRecs &S, const uint8_t *__restrict__ alt,
                                              const uint8_t *__restrict__ ref, const uint32_t *__restrict__ nib,
                                              int64_t ref_base, int32_t contig_len, uint32_t padnib, int il,
                                              int32_t p_lo, int32_t ps, int32_t pe) {
    uint32_t v = 0;
    int32_t p = ps;
    while (p < pe) {
        while (S.a[il + 1] <= p) il++;
        const int32_t e_i = S.e[il];
        if (p < e_i) {
            const int64_t src = S.src[il];
            const int32_t a_i = S.a[il];
            const int32_t q = min(e_i, pe);
            for (; p < q; p++) {
                uint32_t c;
                if (src == ALT_PAD) {
                    c = padnib & 15u;  // leading pad (src/reconstruct/mod.rs:75-80)
                } else {
                    // (src < 0: pure-deletion anchor of the svar2 source, taken from the reference)
                    c = nib_code(src >= 0 ? alt[src + (p - a_i)] : ref[~src + (p - a_i)]);
                }
                v |= c << (4 * (p - p_lo));
            }
        } else {
            const int32_t q = min(S.a[il + 1], pe);
            const int32_t cnt = q - p;  // 1..8 positions of reference
            const int64_t rpos = (int64_t)S.resume[il] + (p - e_i);
            const int32_t valid = (int32_t)imax64(0, imin64((int64_t)contig_len - rpos, cnt));
            uint32_t x = padnib;  // trailing pad past the contig end (:248-253)
            if (valid > 0) {
                const uint32_t keep = valid >= 8 ? 0xffffffffu : ((1u << (4 * valid)) - 1u);
                x = (load_codes(nib, ref_base + rpos) & keep) | (padnib & ~keep);
            }
            const uint32_t cm = cnt >= 8 ? 0xffffffffu : ((1u << (4 * cnt)) - 1u);
            v |= (x & cm) << (4 * (p - p_lo));
            p = q;
        }
    }
    return v;
}


// ---- EDGE units: units of 8 positions with a record boundary strictly inside --------------------------
// Every staged record owns two "boundaries" (its ALT start a and its ALT end e); one thread per boundary
// assembles the unit that contains it (if no earlier boundary lies in the same unit).  All other units of the
// pass are a single run (reference or ALT interior) and are streamed by the lanes of the group loop.
enum { U_SKIP = 0, U_PATCH = 2, U_SLOW = 3 };

// Shape of a PATCH unit: [0, x1) reference with delta dlA | [x1, x2) ALT codes starting at base index `alt` of the
// packed allele buffer (ALT_PAD: pad codes; < 0: ~index into the packed reference, the svar2 pure-deletion
// anchor) | [x2, 8) reference with delta dlB.
struct UnitShape {
    int x1, x2;
    int32_t dlA, dlB;
    int64_t alt;
};

__device__ __forceinline__ uint32_t nib_mask(int k) { return k >= 8 ? 0xffffffffu : ((1u << (4 * k)) - 1u); }

// valid leading codes of an 8-code window that starts at reference position rpos (trailing pad past the contig end)
__device__ __forceinline__ int n_valid(int32_t contig_len, int64_t rpos) {
    return (int)imax64(0, imin64((int64_t)contig_len - rpos, 8));
}

// il = last staged record with a <= p_lo; the unit [p_lo, p_lo + 8) lies inside the pass
__device__ __forceinline__ int oh_classify(const OhRecs &S, int il, int32_t p_lo, int64_t ref_base, UnitShape &U) {
    const int32_t end = p_lo + 8, e_i = S.e[il], a1 = S.a[il + 1];
    U.dlA = S.resume[il] - e_i;
    if (p_lo >= e_i) {  // starts in the reference run of record il; record il+1 starts inside
        if (S.a[il + 2] < end) return U_SLOW;  // two records start inside the unit
        const int32_t e1 = S.e[il + 1];
        U.x1 = a1 - p_lo;
        U.x2 = min(e1, end) - p_lo;
        U.dlB = S.resume[il + 1] - e1;
        U.alt = S.src[il + 1];
        if (ref_base + p_lo + U.dlB < 0) return U_SLOW;  // (the 8-code window would start before the buffer)
    } else {  // starts inside the ALT of record il, which ends inside
        if (a1 < end) return U_SLOW;
        U.x1 = 0;
        U.x2 = e_i - p_lo;
        U.dlB = U.dlA;
        const int64_t src = S.src[il], off = p_lo - S.a[il];
        U.alt = src == ALT_PAD ? ALT_PAD : (src >= 0 ? src + off : ~(~src + off));
        if (ref_base + p_lo + U.dlA < 0) return U_SLOW;
    }
    return U_PATCH;
}

// OH_UNROLL = groups per warp whose loads are issued together: 4 for long sparse rows (cfg3: 259 us per 20 batches against 270
// with 2), 2 where most groups take the mixed path or a warp has only a handful of groups (cfg2d: 358 -> 304 us, cfg4: 613 ->
// 551 us) -- the launch code picks (profiles/r2_plan.md).
// NT = threads per CTA: 128, or 64 for rows of at most 8,192 positions (one tile per row: twelve 2-warp CTAs per SM keep more
// rows in flight against the ~3.3 us of fixed latency per CTA than eight 4-warp ones -- cfg4: 551 -> 479 us per 20 batches).
template <int OH_UNROLL, int NT>
__global__ void __launch_bounds__(NT, NT == 64 ? 12 : OH_UNROLL == OH_UNROLL_LONG ? OH_MIN_CTAS_LONG : OH_MIN_CTAS) hap_exec_oh_kernel(HapExecParams P) {
    constexpr int EDGE_ROUNDS = (2 * REC_CAP + 2 + NT - 1) / NT;  // edge slots per thread and pass
    __shared__ OhRecs S;
    __shared__ __align__(16) uint2 s_lut[256];         // byte (2 codes) -> 8 one-hot bytes
    __shared__ __align__(8) uint2 s_grp[OH_MAX_GROUPS];  // per group: {reference delta, idx | cnt << 8 | plain << 31}
    // per thread and round (2 * REC_CAP + 2 slots over NT threads): 6 staged code words of an edge unit, descriptor, position
    __shared__ uint32_t s_edge[EDGE_ROUNDS][8][NT];
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
    // ---- records of this tile: r = last with a < h0 (or -1, the virtual leading-pad record), r_hi = first with
    //      a >= h1.  Fixed-length plans read both from the plan's checkpoint directory -- the two loads do not
    //      depend on the row header, so the prologue is ONE round trip; ragged plans count (sorted array). ----
    int32_t d_lo = 0, d_hi = 0;
    if (P.dir) {
        const int64_t h0d = tile * (int64_t)P.tile_len;
        const int64_t h1d = imin64(h0d + P.tile_len, P.fixed_len);
        const int32_t *__restrict__ d = P.dir + row * P.dir_stride;
        d_lo = __ldg(d + h0d / DIR_Q);
        d_hi = __ldg(d + (h1d + DIR_Q - 1) / DIR_Q);  // (h1 is a multiple of DIR_Q or the row end = last entry)
    }
    const RowPlan rp = P.rows[row];
    const int32_t L = rp.length;
    const int64_t h0_64 = tile * (int64_t)P.tile_len;  // tiles are cut in HAPLOTYPE coordinates
    if (h0_64 >= L) return;
    const int32_t h0 = (int32_t)h0_64;
    const int32_t h1 = (int32_t)imin64(h0_64 + P.tile_len, L);
    const bool rc = rp.rc != 0;

    // ---- warm L2 with the packed reference window of this tile while the records travel: the window starts near
    //      ref0 + (h0 - lead_pad) (exact up to the indels before h0); +-1 Ki bases of slack, 128-byte lines ----
    if (warp == 1) {
        const int64_t est = (int64_t)rp.ref0 + (h0 - rp.lead_pad);
        const int64_t b_lo = imax64(est - 1024, 0), b_hi = imin64(est + (h1 - h0) + 1024, rp.contig_len);
        const char *base = reinterpret_cast<const char *>(P.ref_packed);
        for (int64_t line = ((rp.ref_base + b_lo) >> 8) + lane; line <= ((rp.ref_base + b_hi) >> 8); line += 32)
            if (b_hi > b_lo) asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (line << 7)));
    }

    // spread(n): byte c = bit c of the 4-bit code n   (n * 0x204081 puts bit c at bit 8c, no carries); entry of byte i at
    // oh_swizzle(i) (a bijection on bytes)
    for (int i = tid; i < 256; i += NT)
        s_lut[oh_swizzle(i)] = make_uint2(((i & 15) * 0x204081u) & 0x01010101u, ((i >> 4) * 0x204081u) & 0x01010101u);

    const int32_t *__restrict__ ra = P.rec.a + rp.rec_off;
    if (!P.dir && warp == 0) {
        int64_t r_lo, r_hi0;
        if (rp.n_rec <= 2048) {
            int c0 = 0, c1 = 0;
            for (int i0 = 0; i0 < rp.n_rec; i0 += 256) {  // 8 independent loads per lane and trip
                int32_t a[8];
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    const int i = i0 + 32 * u + lane;
                    a[u] = i < rp.n_rec ? ra[i] : INT32_MAX;
                }
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    c0 += (a[u] < h0);
                    c1 += (a[u] < h1);
                }
            }
            r_lo = (int64_t)__reduce_add_sync(0xffffffffu, c0) - 1;
            r_hi0 = __reduce_add_sync(0xffffffffu, c1);
        } else {
            r_lo = h0 > 0 ? warp_upper_le(ra, 0, rp.n_rec, h0 - 1) : -1;
            r_hi0 = warp_upper_le(ra, imax64(r_lo, 0), rp.n_rec, h1 - 1) + 1;
        }
        if (lane == 0) {
            s_lo = r_lo;
            s_hi = r_hi0;
        }
    }
    if (P.dir && tid == 0) {
        s_lo = (int64_t)d_lo - 1;
        s_hi = rp.n_rec ? d_hi : 0;
    }
    __syncthreads();
    const int64_t r_hi = s_hi;
    int64_t r = s_lo;
    int32_t cur = h0;
    uint8_t *__restrict__ out_row = P.out + 4 * rp.out_off;  // position j of the row lives at out_row[4*j]
    const uint32_t padnib = nib_code(P.pad_char) * 0x11111111u;
    const int32_t lane_off = 8 * (rc ? 31 - lane : lane);  // haplotype offset of the lane's unit inside its group
    // (reference base index + 2 * table address): (x >> 1) & ~3 is then the byte address of the word that holds
    // base x, and the low 3 bits still count nibbles (the table is 16-byte aligned)
    const int64_t nb2 = rp.ref_base + lane_off + 2 * (int64_t)reinterpret_cast<uintptr_t>(P.ref_packed);

    // common epilogue of a full unit: 8 codes (output order) -> 32 one-hot bytes, one 256-bit store
    auto emit8 = [&](uint8_t *dst, uint32_t v) {
        v = oh_swizzle(v);  // each byte to its table index
        const char *lut = reinterpret_cast<const char *>(s_lut);  // (a link-time constant: folds into the LDS offset)
        const uint2 o0 = *reinterpret_cast<const uint2 *>(lut + ((v << 3) & 0x7f8u));
        const uint2 o1 = *reinterpret_cast<const uint2 *>(lut + ((v >> 5) & 0x7f8u));
        const uint2 o2 = *reinterpret_cast<const uint2 *>(lut + ((v >> 13) & 0x7f8u));
        const uint2 o3 = *reinterpret_cast<const uint2 *>(lut + ((v >> 21) & 0x7f8u));
        stg_256(dst, o0, o1, o2, o3);
    };
    // reverse-complement of 8 codes = bit reversal of the word (rows that are not reversed pass through)
    auto rc8 = [&](uint32_t v) {
        uint32_t r_;
        asm("brev.b32 %0, %1;" : "=r"(r_) : "r"(v));
        return rc ? r_ : v;
    };

    while (cur < h1) {
        // ---- stage entry 0 (carry) + up to REC_CAP-1 following records ----
        const int m_new = (int)imin64(REC_CAP - 1, r_hi - (r + 1));
        const int m = m_new + 1;
        const int32_t seg_end = (r + 1 + m_new < r_hi) ? ra[r + 1 + m_new] : h1;
        __syncthreads();  // previous pass finished reading S
        for (int i = tid; i < m; i += NT) {
            const int64_t idx = r + i;
            if (idx < 0) {  // virtual record: leading pad, then reference from ref0
                S.a[0] = 0;
                S.e[0] = rp.lead_pad;
                S.resume[0] = rp.ref0;
                S.src[0] = ALT_PAD;
            } else {
                const int64_t g = rp.rec_off + idx;
                const int32_t a = P.rec.a[g];
                S.a[i] = a;
                S.e[i] = a + P.rec.n[g];
                S.resume[i] = P.rec.resume[g];
                S.src[i] = P.rec.src[g];
            }
        }
        if (tid == 0) S.a[m] = S.a[m + 1] = INT32_MAX;
        __syncthreads();

        // ---- output range of the pass in units of 8 positions aligned on the GLOBAL flat index (32-byte
        //      aligned stores); a group is 32 units (one per lane), warp w owns groups w, w+4, ... ----
        const int32_t jo_lo = rc ? L - seg_end : cur;
        const int32_t jo_hi = rc ? L - cur : seg_end;
        const int64_t g0 = (rp.out_off + jo_lo) & ~(int64_t)7;
        const int32_t j0 = (int32_t)(g0 - rp.out_off);  // row-relative position of unit 0 (may be < jo_lo)
        const int32_t n_groups = (jo_hi - j0 + OH_GROUP - 1) / OH_GROUP;

        // ---- group table: one thread per group ----
        if (tid < n_groups) {
            const int32_t jg = j0 + OH_GROUP * tid;
            const bool full = jg >= jo_lo && jg + OH_GROUP <= jo_hi;
            const int32_t pg = rc ? (L - OH_GROUP - jg) : jg;  // lowest haplotype position of the group
            int idx = 0;
            {
                const int32_t ps = max(pg, cur);
                int hi = m;
                while (hi - idx > 1) {
                    const int mid = (idx + hi) >> 1;
                    if (S.a[mid] <= ps) idx = mid; else hi = mid;
                }
            }
            const int32_t phi = min(pg + OH_GROUP, seg_end);
            int cnt = 0;
            while (S.a[idx + 1 + cnt] < phi) cnt++;
            const int32_t e_i = S.e[idx];
            const int32_t dl = S.resume[idx] - e_i;
            const bool plain = full && cnt == 0 && pg >= e_i && (int64_t)pg + dl + OH_GROUP <= rp.contig_len;
            s_grp[tid] = make_uint2((uint32_t)dl, (uint32_t)idx | ((uint32_t)cnt << 8) | (plain ? 0x80000000u : 0u));
        }
        __syncthreads();

        uint8_t *const out_lane = out_row + 4 * ((int64_t)j0 + 8 * lane);
        const int32_t pg0 = rc ? (L - OH_GROUP - j0) : j0;  // lowest haplotype position of group 0
        const int32_t pg_step = rc ? -OH_GROUP : OH_GROUP;
        const int32_t gofs = (rc ? L - j0 : j0) & 7;        // units start at haplotype positions == gofs (mod 8)

        // ---- edge slots, part 1: classify + start the loads.  Slot s < 2m is the boundary a (s even) / e (s odd)
        //      of staged record s >> 1; slots 2m and 2m+1 are the units cut by the two ends of the pass. ----
        const int n_slots = 2 * m + 2;
        auto edge_locate = [&](int s_, int &kind, int32_t &p_lo, int &il) {
            kind = U_SKIP;
            if (s_ >= 2 * m) {  // partial units at the pass ends (first: s_ == 2m, last: 2m+1)
                const int32_t jf = j0, jl = j0 + (((jo_hi - 1 - j0) >> 3) << 3);
                const int32_t j = s_ == 2 * m ? jf : jl;
                if ((s_ == 2 * m + 1 && jl == jf) || (j >= jo_lo && j + 8 <= jo_hi)) return;
                p_lo = rc ? L - 8 - j : j;
                kind = U_SLOW;
            } else {
                const int32_t b = (s_ & 1) ? S.e[s_ >> 1] : S.a[s_ >> 1];
                const int32_t in = (b - gofs) & 7;
                if (in == 0) return;  // boundary on a unit edge: both neighbours are single runs
                p_lo = b - in;
                const int32_t j = rc ? L - 8 - p_lo : p_lo;
                if (!(j >= jo_lo && j + 8 <= jo_hi)) return;  // outside this pass, or cut by it (slots 2m, 2m+1)
                if (s_ > 0 && (((s_ - 1) & 1) ? S.e[(s_ - 1) >> 1] : S.a[(s_ - 1) >> 1]) > p_lo) return;  // an earlier boundary owns the unit
                kind = U_PATCH;
            }
            il = min(s_ >> 1, m - 1);
            const int32_t ps = max(p_lo, cur);
            while (il > 0 && S.a[il] > ps) il--;
        };
        // (the code words travel with asynchronous 4-byte copies into the thread's own shared-memory slots, so no
        //  register stays live across the group loop; part 2 reads them back after it)
        auto edge_begin = [&](int s_, int rd) {
            int e_kind, e_il = 0;
            int32_t e_p = 0;
            uint32_t e_desc = 0;
            edge_locate(s_, e_kind, e_p, e_il);
            if (e_kind == U_PATCH) {
                UnitShape U;
                e_kind = oh_classify(S, e_il, e_p, rp.ref_base, U);
                if (e_kind == U_PATCH) {
                    const uint32_t slot = smem_u32(&s_edge[rd][0][tid]);
                    const int64_t nA = rp.ref_base + e_p + U.dlA;
                    const int vA = n_valid(rp.contig_len, (int64_t)e_p + U.dlA);
                    e_desc = (uint32_t)U.x1 << 2 | (uint32_t)U.x2 << 6 | (uint32_t)vA << 10 | ((uint32_t)nA & 7u) << 18;
                    if (vA > 0 && (U.x1 > 0 || U.x2 < 8)) {
                        const uint32_t *w = P.ref_packed + (nA >> 3);
                        cp_async4(slot, w);
                        cp_async4(slot + 4 * NT, w + 1);
                    }
                    if (U.x1 > 0 && U.x2 < 8) {  // a record starts inside the unit: reference resumes with its own delta
                        const int64_t nB = rp.ref_base + e_p + U.dlB;
                        const int vB = n_valid(rp.contig_len, (int64_t)e_p + U.dlB);
                        e_desc |= (uint32_t)vB << 14 | ((uint32_t)nB & 7u) << 21;
                        if (vB > 0) {
                            const uint32_t *w = P.ref_packed + (nB >> 3);
                            cp_async4(slot + 8 * NT, w);
                            cp_async4(slot + 12 * NT, w + 1);
                        }
                    }
                    if (U.alt == ALT_PAD) {
                        e_desc |= 1u << 27;
                    } else {  // ALT codes, or the svar2 pure-deletion anchor from the packed reference
                        const int64_t nC = U.alt >= 0 ? U.alt : ~U.alt;
                        const uint32_t *w = (U.alt >= 0 ? P.alt_packed : P.ref_packed) + (nC >> 3);
                        e_desc |= ((uint32_t)nC & 7u) << 24;
                        cp_async4(slot + 16 * NT, w);
                        cp_async4(slot + 20 * NT, w + 1);
                    }
                }
            }
            s_edge[rd][6][tid] = e_desc | (uint32_t)e_kind;
            s_edge[rd][7][tid] = (uint32_t)e_p;
        };
        for (int s_ = tid, rd = 0; s_ < n_slots; s_ += NT, rd++) edge_begin(s_, rd);  // (one round unless variants are dense)
        cp_async_commit();

        // ---- the group loop: every lane streams the units that are a single run ----
        for (int gb = warp; gb < n_groups; gb += OH_UNROLL * (NT / 32)) {
            uint8_t *const out_it = out_lane + (int64_t)gb * (4 * OH_GROUP);  // the lane's unit in group gb
            // phase 1: all loads of the warp's next OH_UNROLL groups (2 per lane and group in flight)
            uint32_t w0[OH_UNROLL], w1[OH_UNROLL], sh[OH_UNROLL];
            unsigned nvs = 0;      // per LANE, 4 bits per group: valid codes 0..8, 15 = not this lane's unit
            unsigned mixmask = 0;  // per warp
#pragma unroll
            for (int u = 0; u < OH_UNROLL; u++) {
                const int g = gb + u * (NT / 32);
                w0[u] = w1[u] = sh[u] = 0;
                unsigned nv = 15;
                if (g < n_groups) {
                    const uint2 meta = s_grp[g];
                    if (meta.y & 0x80000000u) {  // plain: one delta for the whole group
                        nv = 8;
                        const int64_t x = nb2 + (int32_t)(pg0 + pg_step * g + (int32_t)meta.x);
                        const uint32_t *w = reinterpret_cast<const uint32_t *>((uintptr_t)(x >> 1) & ~(uintptr_t)3);
                        w0[u] = __ldg(w);
                        w1[u] = __ldg(w + 1);
                        sh[u] = (uint32_t)x << 2;
                    } else {  // variants / pads / edges: the lane looks at its own unit
                        mixmask |= 1u << u;
                        const int32_t j = j0 + OH_GROUP * g + 8 * lane;  // first output position of the lane's unit
                        const int32_t p_lo = pg0 + pg_step * g + lane_off;
                        if (j >= jo_lo && j + 8 <= jo_hi) {
                            const int idx = meta.y & 0xff, cnt = (meta.y >> 8) & 0xff;
                            int il = idx;
                            for (int q = 1; q <= cnt; q++) il += (S.a[idx + q] <= p_lo);
                            const int32_t e_i = S.e[il];
                            const uint32_t *base = P.ref_packed;
                            int64_t n = -1;
                            if (p_lo >= e_i) {
                                if (p_lo + 8 <= S.a[il + 1]) {  // reference run (trailing pad past the contig end, :248-253)
                                    const int64_t rpos = (int64_t)p_lo + (S.resume[il] - e_i);
                                    nv = (unsigned)n_valid(rp.contig_len, rpos);
                                    n = rp.ref_base + rpos;
                                }
                            } else if (p_lo + 8 <= e_i) {  // interior of an ALT (long insertion, leading pad)
                                const int64_t src = S.src[il];
                                nv = src == ALT_PAD ? 0 : 8;  // (pad codes need no load)
                                n = (src >= 0 ? src : ~src) + (p_lo - S.a[il]);
                                if (src >= 0) base = P.alt_packed;
                            }
                            if (nv >= 1 && nv <= 8) {
                                const uint32_t *w = base + (n >> 3);
                                w0[u] = __ldg(w);
                                w1[u] = __ldg(w + 1);
                                sh[u] = (uint32_t)n << 2;
                            }
                        }
                    }
                }
                nvs |= nv << (4 * u);
            }
            // phase 2: encode + store
#pragma unroll
            for (int u = 0; u < OH_UNROLL; u++) {
                const unsigned nv = (nvs >> (4 * u)) & 15u;
                if (nv != 15) {
                    uint32_t v = __funnelshift_r(w0[u], w1[u], sh[u]);  // nibble t = haplotype position p_lo + t
                    if (mixmask & (1u << u)) {
                        const uint32_t mk = nib_mask((int)nv);
                        v = (v & mk) | (padnib & ~mk);
                    }
                    emit8(out_it + u * (NT / 32) * (4 * OH_GROUP), rc8(v));  // rc: nibble t = output position j + t, complemented
                }
            }
        }

        // ---- edge slots, part 2: blend (the copies were started before the group loop) + store ----
        cp_async_wait<0>();
#pragma unroll 1
        for (int s_ = tid, rd = 0; s_ < n_slots; s_ += NT, rd++) {
            int e_kind, e_il = 0;
            int32_t e_p;
            uint32_t e_desc = 0;
            const uint32_t(*sl)[NT] = s_edge[rd];
            e_desc = sl[6][tid];
            e_kind = e_desc & 3u;
            e_p = (int32_t)sl[7][tid];
            if (e_kind == U_SLOW) {  // piecewise units are done start to finish here
                edge_locate(s_, e_kind, e_p, e_il);
                if (e_kind == U_PATCH) e_kind = U_SLOW;
            }
            if (e_kind == U_SKIP) continue;
            const int32_t j = rc ? L - 8 - e_p : e_p;
            uint32_t v;
            if (e_kind == U_PATCH) {
                const int x1 = (e_desc >> 2) & 15, x2 = (e_desc >> 6) & 15;
                const uint32_t mA = nib_mask((e_desc >> 10) & 15);
                const uint32_t A = (__funnelshift_r(sl[0][tid], sl[1][tid], ((e_desc >> 18) & 7u) * 4u) & mA) | (padnib & ~mA);
                uint32_t B = A;
                if (x1 > 0) {
                    const uint32_t mB = nib_mask((e_desc >> 14) & 15);
                    B = (__funnelshift_r(sl[2][tid], sl[3][tid], ((e_desc >> 21) & 7u) * 4u) & mB) | (padnib & ~mB);
                }
                uint32_t alt = padnib;  // leading pad (src/reconstruct/mod.rs:75-80)
                if (!(e_desc & (1u << 27))) alt = __funnelshift_r(sl[4][tid], sl[5][tid], ((e_desc >> 24) & 7u) * 4u);
                const uint32_t m1 = nib_mask(x1), m2 = nib_mask(x2);
                v = (A & m1) | ((alt << (4 * x1)) & m2 & ~m1) | (B & ~m2);
            } else {
                v = oh_slow_unit(S, P.alt, P.ref, P.ref_packed, rp.ref_base, rp.contig_len, padnib, e_il, e_p,
                                 max(e_p, cur), min(e_p + 8, seg_end));
            }
            v = rc8(v);
            uint8_t *dst = out_row + 4 * (int64_t)j;
            if (j >= jo_lo && j + 8 <= jo_hi) {
                emit8(dst, v);
            } else {  // unit cut by a pass / tile / row boundary: position-wise stores
#pragma unroll 1
                for (int q = 0; q < 8; q++) {
                    const int32_t jj = j + q;
                    if (jj >= jo_lo && jj < jo_hi)
                        *reinterpret_cast<uint32_t *>(dst + 4 * q) = (((v >> (4 * q)) & 15u) * 0x204081u) & 0x01010101u;
                }
            }
        }
        cur = seg_end;
        r += m_new;
    }
}

}  // namespace gvl
