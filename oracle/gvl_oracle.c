/*
 * gvl_oracle.c -- CPU restatement of GenVarLoader's haplotype-reconstruction hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under genvarloader_b200/ may import, link or call
 * this file.  It is used by tests/, by __graft_entry__.smoke() as the checker, and by
 * bench.py's cpu_baseline / --impl reference legs as the timed CPU stand-in.
 *
 * The reference's own implementation is Rust (cargo/rustc are absent here), so this is a
 * "port" oracle.  It is PINNED: tests/test_oracle_golden.py replays every frozen golden
 * vector the reference's parity suite holds for this path (the .npz files under tests/parity/golden,
 * converted by tests/golden/make_golden.py) plus the known-answer vectors of the Rust
 * in-file unit tests, and tests/golden/make_pyref_golden.py cross-checks it against the
 * reference's own pure-Python fallbacks.
 *
 * Every function cites the reference file:line (relative to /root/reference) it follows.
 * The statement order, integer widths (i64 state, i32 stores) and float promotion points
 * of the reference are kept so results are bit-identical.
 *
 * Build: gcc -O3 -march=native -fPIC -shared -pthread -o oracle/libgvl_oracle.so oracle/gvl_oracle.c
 */
#include <math.h>
#include <pthread.h>
#include <stdatomic.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define GVL_API __attribute__((visibility("default")))

static inline int64_t i64min(int64_t a, int64_t b) { return a < b ? a : b; }
static inline int64_t i64max(int64_t a, int64_t b) { return a > b ? a : b; }

/* ------------------------------------------------------------------------------------
 * persistent fork-join pool: one task per work item pulled from an atomic counter.  Same
 * decomposition as rayon `into_par_iter` over (query, hap) items
 * (src/reconstruct/mod.rs:531-538); like rayon's process-global pool
 * (python/genvarloader/_threads.py:102-115) the workers are created once and parked between
 * calls, so a call pays a wake-up, not a thread creation.  Scheduling never affects results
 * (disjoint outputs).
 * ---------------------------------------------------------------------------------- */
typedef void (*gvl_task_fn)(void *ctx, int64_t k);
typedef struct {
    gvl_task_fn fn;
    void *ctx;
    int64_t n;
    atomic_llong next;
    int64_t grain;
} gvl_job;

static void gvl_run_job(gvl_job *job) {
    for (;;) {
        int64_t s = atomic_fetch_add(&job->next, job->grain);
        if (s >= job->n) break;
        int64_t e = i64min(s + job->grain, job->n);
        for (int64_t k = s; k < e; k++) job->fn(job->ctx, k);
    }
}

#define GVL_MAX_THREADS 256
static int g_threads = 1;
static struct {
    pthread_mutex_t mu;
    pthread_cond_t wake, done;
    pthread_t th[GVL_MAX_THREADS];
    int n_workers;        /* threads alive (excluding the caller) */
    int n_active;         /* workers that take part in the current job */
    int n_running;        /* workers that have not finished the current job yet */
    unsigned generation;  /* bumped once per job */
    gvl_job *job;
    int init;
} g_pool = {PTHREAD_MUTEX_INITIALIZER, PTHREAD_COND_INITIALIZER, PTHREAD_COND_INITIALIZER, {0}, 0, 0, 0, 0, NULL, 0};

static void *gvl_pool_worker(void *p) {
    const int id = (int)(intptr_t)p;
    unsigned seen = 0;
    pthread_mutex_lock(&g_pool.mu);
    for (;;) {
        while (g_pool.generation == seen) pthread_cond_wait(&g_pool.wake, &g_pool.mu);
        seen = g_pool.generation;
        if (id >= g_pool.n_active) continue; /* this job uses fewer threads */
        gvl_job *job = g_pool.job;
        pthread_mutex_unlock(&g_pool.mu);
        gvl_run_job(job);
        pthread_mutex_lock(&g_pool.mu);
        if (--g_pool.n_running == 0) pthread_cond_signal(&g_pool.done);
    }
    return NULL;
}

GVL_API void gvl_oracle_set_threads(int n) { g_threads = n < 1 ? 1 : (n > GVL_MAX_THREADS ? GVL_MAX_THREADS : n); }
GVL_API int gvl_oracle_get_threads(void) { return g_threads; }

static void gvl_parallel_for(gvl_task_fn fn, void *ctx, int64_t n, int parallel, int64_t grain) {
    int nt = parallel ? g_threads : 1;
    if (nt > n) nt = (int)n;
    if (nt <= 1) {
        for (int64_t k = 0; k < n; k++) fn(ctx, k);
        return;
    }
    gvl_job job;
    job.fn = fn;
    job.ctx = ctx;
    job.n = n;
    job.grain = grain < 1 ? 1 : grain;
    atomic_init(&job.next, 0);
    pthread_mutex_lock(&g_pool.mu);
    while (g_pool.n_workers < nt - 1) { /* grow the pool on demand; workers never exit */
        const int id = g_pool.n_workers;
        if (pthread_create(&g_pool.th[id], NULL, gvl_pool_worker, (void *)(intptr_t)id) != 0) break;
        pthread_detach(g_pool.th[id]);
        g_pool.n_workers++;
    }
    const int helpers = g_pool.n_workers < nt - 1 ? g_pool.n_workers : nt - 1;
    g_pool.job = &job;
    g_pool.n_active = helpers;
    g_pool.n_running = helpers;
    g_pool.generation++;
    pthread_cond_broadcast(&g_pool.wake);
    pthread_mutex_unlock(&g_pool.mu);
    gvl_run_job(&job); /* the caller works too */
    pthread_mutex_lock(&g_pool.mu);
    while (g_pool.n_running > 0) pthread_cond_wait(&g_pool.done, &g_pool.mu);
    g_pool.job = NULL;
    pthread_mutex_unlock(&g_pool.mu);
}

/* ====================================================================================
 * a1  reconstruct_haplotype_core                     src/reconstruct/mod.rs:39-256
 * ==================================================================================== */
typedef struct {
    int64_t v_pos;
    int64_t v_diff;
    const uint8_t *allele;
    int64_t allele_len;
    int32_t annot_id;
} gvl_var;

typedef void (*gvl_provide_fn)(const void *src, int64_t v, gvl_var *out);

static void reconstruct_haplotype_core(int64_t n_variants, gvl_provide_fn provide, const void *src,
                                       int64_t shift, const uint8_t *ref_, int64_t ref_len_total,
                                       int64_t ref_start, uint8_t *out, int64_t length,
                                       uint8_t pad_char, const uint8_t *keep, int32_t *annot_v,
                                       int32_t *annot_pos) {
    int64_t ref_idx = ref_start; /* :61 */
    int64_t out_idx = 0;         /* :63 */
    int64_t shifted = 0;         /* :65 */

    if (ref_idx < 0) { /* :68-83 leading pad */
        int64_t pad_len_raw = -ref_idx;
        shifted = i64min(shift, pad_len_raw);
        int64_t pad_len = pad_len_raw - shifted;
        /* Rust would panic on pad_len > length (out of contract); clamp like numpy slicing
         * in the reference's pure-Python twin (_genotypes.py:159). */
        int64_t e = i64min(out_idx + pad_len, length);
        for (int64_t j = out_idx; j < e; j++) out[j] = pad_char;
        if (annot_v) for (int64_t j = out_idx; j < e; j++) annot_v[j] = -1;
        if (annot_pos) for (int64_t j = out_idx; j < e; j++) annot_pos[j] = -1;
        out_idx += pad_len;
        ref_idx = 0;
    }

    for (int64_t v = 0; v < n_variants; v++) { /* :85 */
        if (keep && !keep[v]) continue;        /* :86-90 */
        gvl_var var;
        provide(src, v, &var); /* :92 */
        int64_t v_pos = var.v_pos, v_diff = var.v_diff;
        int64_t v_len_full = var.allele_len;
        int64_t v_ref_end = v_pos - i64min(0, v_diff) + 1; /* :96 */

        if (v_pos < ref_start && v_diff < 0 && v_ref_end >= ref_start) { /* :99-102 */
            ref_idx = v_ref_end;
            continue;
        }
        if (v_pos < ref_idx) continue; /* :108-110 first ALT wins */

        int64_t allele_start_idx = 0; /* :114 */
        if (shifted < shift) {        /* :115-146 */
            int64_t ref_shift_dist = v_pos - ref_idx;
            if (shifted + ref_shift_dist + v_len_full < shift) {
                continue; /* :118-121 */
            } else if (shifted + ref_shift_dist >= shift) {
                ref_idx += shift - shifted; /* :123-128 */
                shifted = shift;
            } else {
                allele_start_idx = shift - shifted - ref_shift_dist; /* :132 */
                shifted = shift;
                if (allele_start_idx == v_len_full) { /* :135-140 */
                    ref_idx = v_ref_end;
                    continue;
                }
                ref_idx = v_pos; /* :143 */
            }
        }
        const uint8_t *allele = var.allele + allele_start_idx; /* :149 */
        int64_t v_len = v_len_full - allele_start_idx;

        int64_t ref_len = v_pos - ref_idx;       /* :153 */
        if (out_idx + ref_len >= length) break;  /* :154-158 */
        memcpy(out + out_idx, ref_ + ref_idx, (size_t)ref_len); /* :164 */
        if (annot_v) for (int64_t j = 0; j < ref_len; j++) annot_v[out_idx + j] = -1;
        if (annot_pos) for (int64_t j = 0; j < ref_len; j++) annot_pos[out_idx + j] = (int32_t)(ref_idx + j);
        out_idx += ref_len; /* :175 */

        int64_t writable_length = i64min(v_len, length - out_idx); /* :178 */
        memcpy(out + out_idx, allele, (size_t)writable_length);    /* :182 */
        if (annot_v) for (int64_t j = 0; j < writable_length; j++) annot_v[out_idx + j] = var.annot_id;
        if (annot_pos) for (int64_t j = 0; j < writable_length; j++) annot_pos[out_idx + j] = (int32_t)v_pos;
        out_idx += writable_length; /* :190 */

        ref_idx = v_ref_end;           /* :193 */
        if (out_idx >= length) break;  /* :195-197 */
    }

    if (shifted < shift) { /* :200-205 */
        ref_idx += shift - shifted;
        ref_idx = i64min(ref_idx, ref_len_total);
        shifted = shift;
    }

    int64_t unfilled_length = length - out_idx; /* :209 */
    if (unfilled_length > 0) {
        int64_t writable_ref = i64min(unfilled_length, ref_len_total - ref_idx); /* :213 */
        int64_t out_end_idx;
        if (writable_ref > 0) { /* :215-233 */
            memcpy(out + out_idx, ref_ + ref_idx, (size_t)writable_ref);
            if (annot_v) for (int64_t j = 0; j < writable_ref; j++) annot_v[out_idx + j] = -1;
            if (annot_pos) for (int64_t j = 0; j < writable_ref; j++) annot_pos[out_idx + j] = (int32_t)(ref_idx + j);
            out_end_idx = out_idx + writable_ref;
        } else {
            out_end_idx = out_idx; /* :234-241 */
        }
        if (out_end_idx < length) { /* :244-254 right pad */
            for (int64_t j = out_end_idx; j < length; j++) out[j] = pad_char;
            if (annot_v) for (int64_t j = out_end_idx; j < length; j++) annot_v[j] = -1;
            if (annot_pos) for (int64_t j = out_end_idx; j < length; j++) annot_pos[j] = INT32_MAX;
        }
    }
}

/* a2  SVAR1 variant source                            src/reconstruct/mod.rs:280-319 */
typedef struct {
    const int32_t *v_idxs;
    const int32_t *v_starts;
    const int32_t *ilens;
    const uint8_t *alt_alleles;
    const int64_t *alt_offsets;
} sparse_src;

static void provide_sparse(const void *p, int64_t v, gvl_var *out) {
    const sparse_src *s = (const sparse_src *)p;
    int64_t variant = s->v_idxs[v];
    int64_t ao_s = s->alt_offsets[variant], ao_e = s->alt_offsets[variant + 1];
    out->v_pos = s->v_starts[variant];
    out->v_diff = s->ilens[variant];
    out->allele = s->alt_alleles + ao_s;
    out->allele_len = ao_e - ao_s;
    out->annot_id = (int32_t)variant;
}

/* a3  reconstruct_haplotypes_from_sparse (batch)      src/reconstruct/mod.rs:348-583 */
typedef struct {
    uint8_t *out;
    const int64_t *out_offsets;
    const int32_t *regions; /* (b,3) */
    const int32_t *shifts;  /* (b,p) */
    const int64_t *geno_offset_idx;
    const int64_t *go_starts, *go_stops;
    const int32_t *geno_v_idxs;
    sparse_src tab;
    const uint8_t *ref_;
    const int64_t *ref_offsets;
    uint8_t pad_char;
    const uint8_t *keep;
    const int64_t *keep_offsets;
    int32_t *annot_v, *annot_pos;
    int64_t ploidy;
} recon_ctx;

static void recon_task(void *p, int64_t k) {
    recon_ctx *c = (recon_ctx *)p;
    int64_t query = k / c->ploidy; /* :380-381 */
    int64_t o_idx = c->geno_offset_idx[k];
    int64_t o_s = c->go_starts[o_idx], o_e = c->go_stops[o_idx]; /* :384-387 */
    sparse_src s = c->tab;
    s.v_idxs = c->geno_v_idxs + o_s;
    const uint8_t *qh_keep = (c->keep && c->keep_offsets) ? c->keep + c->keep_offsets[k] : NULL; /* :390-397 */
    int64_t c_idx = c->regions[query * 3 + 0];                                                  /* :400-405 */
    int64_t c_s = c->ref_offsets[c_idx], c_e = c->ref_offsets[c_idx + 1];
    int64_t ref_start = c->regions[query * 3 + 1];
    int64_t shift = c->shifts[k];
    int64_t os = c->out_offsets[k], oe = c->out_offsets[k + 1];
    reconstruct_haplotype_core(o_e - o_s, provide_sparse, &s, shift, c->ref_ + c_s, c_e - c_s, ref_start,
                               c->out + os, oe - os, c->pad_char, qh_keep,
                               c->annot_v ? c->annot_v + os : NULL, c->annot_pos ? c->annot_pos + os : NULL);
}

GVL_API void gvl_oracle_reconstruct_haplotypes_from_sparse(
    uint8_t *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, const int64_t *go_starts, const int64_t *go_stops,
    const int32_t *geno_v_idxs, const int32_t *v_starts, const int32_t *ilens, const uint8_t *alt_alleles,
    const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets, uint8_t pad_char,
    const uint8_t *keep, const int64_t *keep_offsets, int32_t *annot_v, int32_t *annot_pos, int64_t batch,
    int64_t ploidy, int parallel) {
    recon_ctx c = {out, out_offsets, regions, shifts, geno_offset_idx, go_starts, go_stops, geno_v_idxs,
                   {NULL, v_starts, ilens, alt_alleles, alt_offsets}, ref_, ref_offsets, pad_char, keep,
                   keep_offsets, annot_v, annot_pos, ploidy};
    gvl_parallel_for(recon_task, &c, batch * ploidy, parallel, 1);
}

/* ====================================================================================
 * a4  get_diffs_sparse                                src/genotypes/mod.rs:15-125
 * ==================================================================================== */
typedef struct {
    const int64_t *geno_offset_idx;
    const int32_t *geno_v_idxs;
    const int64_t *o_starts, *o_stops;
    const int32_t *ilens;
    const uint8_t *keep;
    const int64_t *keep_offsets;
    const int32_t *q_starts, *q_ends, *v_starts;
    int64_t q_stride; /* stride (in elements) of q_starts/q_ends so regions[:,1] can be passed */
    int64_t ploidy;
    int32_t *diffs;
} diffs_ctx;

static void diffs_task(void *p, int64_t k) {
    diffs_ctx *c = (diffs_ctx *)p;
    int64_t query = k / c->ploidy;
    int64_t o_idx = c->geno_offset_idx[k];
    int64_t o_s = c->o_starts[o_idx], o_e = c->o_stops[o_idx];
    int has_query = c->q_starts && c->q_ends && c->v_starts; /* :35 */
    int has_keep = c->keep && c->keep_offsets;               /* :36 */
    int64_t acc = 0;
    if (o_e - o_s == 0) { /* :46-47 */
        acc = 0;
    } else if (has_query) { /* :48-86 */
        int64_t q_start = c->q_starts[query * c->q_stride], q_end = c->q_ends[query * c->q_stride];
        int64_t ref_idx = q_start;
        for (int64_t v = o_s; v < o_e; v++) {
            if (has_keep && !c->keep[c->keep_offsets[k] + (v - o_s)]) continue;
            int64_t v_idx = c->geno_v_idxs[v];
            int64_t v_start = c->v_starts[v_idx];
            int64_t v_ilen = c->ilens[v_idx];
            int64_t v_end = v_start - i64min(v_ilen, 0) + 1;
            if (v_end <= q_start) continue;                      /* :69-71 */
            if (v_start >= q_end) break;                         /* :72-74 */
            if (v_start >= q_start && v_start < ref_idx) continue; /* :75-77 */
            ref_idx = i64max(ref_idx, v_end);                    /* :78 */
            if (v_ilen < 0) v_ilen += i64max(q_start - v_start - 1, 0); /* :79-81 */
            v_ilen += i64max(v_end - q_end, 0);                  /* :82 */
            acc += v_ilen;
        }
    } else if (has_keep) { /* :87-97 */
        int64_t k_s = c->keep_offsets[k];
        for (int64_t v = o_s; v < o_e; v++)
            if (c->keep[k_s + (v - o_s)]) acc += c->ilens[c->geno_v_idxs[v]];
    } else { /* :98-104 */
        for (int64_t v = o_s; v < o_e; v++) acc += c->ilens[c->geno_v_idxs[v]];
    }
    c->diffs[k] = (int32_t)acc;
}

GVL_API void gvl_oracle_get_diffs_sparse(const int64_t *geno_offset_idx, const int32_t *geno_v_idxs,
                                         const int64_t *o_starts, const int64_t *o_stops, const int32_t *ilens,
                                         const uint8_t *keep, const int64_t *keep_offsets,
                                         const int32_t *q_starts, const int32_t *q_ends, int64_t q_stride,
                                         const int32_t *v_starts, int64_t n_queries, int64_t ploidy,
                                         int parallel, int32_t *diffs) {
    diffs_ctx c = {geno_offset_idx, geno_v_idxs, o_starts, o_stops, ilens, keep, keep_offsets,
                   q_starts, q_ends, v_starts, q_stride, ploidy, diffs};
    gvl_parallel_for(diffs_task, &c, n_queries * ploidy, parallel, 16);
}

/* choose_exonic_variants                              src/genotypes/mod.rs:132-176
 * keep_offsets has n_regions*ploidy+1 entries; keep has keep_offsets[-1] entries (caller
 * sizes it with a first call passing keep == NULL). */
GVL_API void gvl_oracle_choose_exonic_variants(const int32_t *starts, const int32_t *ends,
                                               const int64_t *geno_offset_idx, const int32_t *geno_v_idxs,
                                               const int64_t *o_starts, const int64_t *o_stops,
                                               const int32_t *v_starts, const int32_t *ilens, int64_t n_regions,
                                               int64_t ploidy, uint8_t *keep, int64_t *keep_offsets) {
    int64_t acc = 0;
    keep_offsets[0] = 0;
    for (int64_t k = 0; k < n_regions * ploidy; k++) {
        int64_t o_idx = geno_offset_idx[k];
        acc += i64max(o_stops[o_idx] - o_starts[o_idx], 0);
        keep_offsets[k + 1] = acc;
    }
    if (!keep) return;
    for (int64_t query = 0; query < n_regions; query++) {
        int64_t ref_start = starts[query], ref_end = ends[query];
        for (int64_t hap = 0; hap < ploidy; hap++) {
            int64_t k = query * ploidy + hap;
            int64_t o_idx = geno_offset_idx[k];
            int64_t o_s = o_starts[o_idx], o_e = o_stops[o_idx], k_s = keep_offsets[k];
            for (int64_t v = o_s; v < o_e; v++) {
                int64_t v_idx = geno_v_idxs[v];
                int64_t v_pos = v_starts[v_idx];
                int64_t v_ref_end = v_pos - i64min((int64_t)ilens[v_idx], 0) + 1;
                keep[k_s + (v - o_s)] = (v_pos >= ref_start && v_ref_end <= ref_end);
            }
        }
    }
}

/* ====================================================================================
 * a5  reverse / reverse-complement                    src/reverse.rs:9-84
 * ==================================================================================== */
static inline uint8_t comp_byte(uint8_t v) { /* :45-53 */
    uint8_t at = (uint8_t)(-(uint8_t)((v == 'A') | (v == 'T')));
    uint8_t cg = (uint8_t)(-(uint8_t)((v == 'C') | (v == 'G')));
    return (uint8_t)(v ^ (at & 21) ^ (cg & 4));
}

static void rc_row(uint8_t *row, int64_t n) {
    for (int64_t i = 0, j = n - 1; i < j; i++, j--) {
        uint8_t t = row[i];
        row[i] = row[j];
        row[j] = t;
    }
    for (int64_t i = 0; i < n; i++) row[i] = comp_byte(row[i]);
}

GVL_API void gvl_oracle_rc_flat_rows_inplace(uint8_t *data, const int64_t *offsets, const uint8_t *to_rc,
                                             int64_t n_rows) { /* :56-69 (serial, like the reference) */
    for (int64_t i = 0; i < n_rows; i++) {
        if (!to_rc[i]) continue;
        rc_row(data + offsets[i], offsets[i + 1] - offsets[i]);
    }
}

GVL_API void gvl_oracle_reverse_flat_rows_inplace_32(uint32_t *data, const int64_t *offsets, const uint8_t *to_rc,
                                                    int64_t n_rows) { /* :25-38 for f32 / i32 */
    for (int64_t r = 0; r < n_rows; r++) {
        if (!to_rc[r]) continue;
        uint32_t *row = data + offsets[r];
        int64_t n = offsets[r + 1] - offsets[r];
        for (int64_t i = 0, j = n - 1; i < j; i++, j--) {
            uint32_t t = row[i];
            row[i] = row[j];
            row[j] = t;
        }
    }
}

/* ====================================================================================
 * get_reference / padded_slice                        src/reference/mod.rs:9-120
 * ==================================================================================== */
static void padded_slice(const uint8_t *arr, int64_t len, int64_t start, int64_t stop, uint8_t pad_val,
                         uint8_t *out, int64_t out_len) {
    if (start >= stop) return; /* :16-18 */
    if (stop < 0) {            /* :19-22 */
        memset(out, pad_val, (size_t)out_len);
        return;
    }
    int64_t pad_left = i64max(-start, 0), pad_right = i64max(stop - len, 0);
    if (pad_left == 0 && pad_right == 0) {
        memcpy(out, arr + start, (size_t)(stop - start));
        return;
    }
    if (pad_left > 0 && pad_right > 0) {
        int64_t out_stop = out_len - pad_right;
        memset(out, pad_val, (size_t)pad_left);
        memcpy(out + pad_left, arr, (size_t)len);
        memset(out + out_stop, pad_val, (size_t)(out_len - out_stop));
    } else if (pad_left > 0) {
        memset(out, pad_val, (size_t)pad_left);
        memcpy(out + pad_left, arr, (size_t)stop);
    } else {
        int64_t out_stop = out_len - pad_right;
        memcpy(out, arr + start, (size_t)(len - start));
        memset(out + out_stop, pad_val, (size_t)(out_len - out_stop));
    }
}

GVL_API void gvl_oracle_get_reference(const int32_t *regions, const int64_t *out_offsets, const uint8_t *reference,
                                      const int64_t *ref_offsets, uint8_t pad_char, const uint8_t *to_rc,
                                      int64_t n, uint8_t *out) {
    for (int64_t i = 0; i < n; i++) {
        int64_t c_idx = regions[i * 3], start = regions[i * 3 + 1], end = regions[i * 3 + 2];
        int64_t c_s = ref_offsets[c_idx], c_e = ref_offsets[c_idx + 1];
        padded_slice(reference + c_s, c_e - c_s, start, end, pad_char, out + out_offsets[i],
                     out_offsets[i + 1] - out_offsets[i]);
    }
    if (to_rc) gvl_oracle_rc_flat_rows_inplace(out, out_offsets, to_rc, n);
}

/* ====================================================================================
 * a6  fused entries                                   src/ffi/mod.rs:724-860, 2239-2397
 * out_offsets (n_work+1) is computed first (steps 1-2); the caller allocates `total`
 * elements and calls the _fill half (steps 3-4b).  gvl_oracle_reconstruct_fused_alloc does
 * both with a malloc'ed (uninitialised, like uninit_output :17-35) buffer for timing.
 * ==================================================================================== */
GVL_API int64_t gvl_oracle_fused_out_offsets(const int32_t *regions, const int64_t *geno_offset_idx,
                                             const int64_t *go_starts, const int64_t *go_stops,
                                             const int32_t *geno_v_idxs, const int32_t *v_starts,
                                             const int32_t *ilens, int64_t output_length, const uint8_t *keep,
                                             const int64_t *keep_offsets, int64_t batch, int64_t ploidy,
                                             int parallel, int64_t *out_offsets, int32_t *diffs_out) {
    int64_t n_work = batch * ploidy;
    int32_t *diffs = diffs_out ? diffs_out : (int32_t *)malloc(sizeof(int32_t) * (size_t)(n_work ? n_work : 1));
    /* :776-788 q_starts = regions[:,1], q_ends = regions[:,2] */
    gvl_oracle_get_diffs_sparse(geno_offset_idx, geno_v_idxs, go_starts, go_stops, ilens, keep, keep_offsets,
                                regions + 1, regions + 2, 3, v_starts, batch, ploidy, parallel, diffs);
    int64_t acc = 0; /* :794-811 serial prefix sum */
    out_offsets[0] = 0;
    for (int64_t k = 0; k < n_work; k++) {
        int64_t query = k / ploidy;
        int64_t len;
        if (output_length >= 0) {
            len = output_length;
        } else {
            int64_t ref_len = (int64_t)(regions[query * 3 + 2] - regions[query * 3 + 1]);
            len = i64max(ref_len + (int64_t)diffs[k], 0);
        }
        acc += len;
        out_offsets[k + 1] = acc;
    }
    if (!diffs_out) free(diffs);
    return acc;
}

GVL_API void gvl_oracle_fused_fill(uint8_t *out, int32_t *annot_v, int32_t *annot_pos, const int64_t *out_offsets,
                                   const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx,
                                   const int64_t *go_starts, const int64_t *go_stops, const int32_t *geno_v_idxs,
                                   const int32_t *v_starts, const int32_t *ilens, const uint8_t *alt_alleles,
                                   const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets,
                                   uint8_t pad_char, const uint8_t *keep, const int64_t *keep_offsets,
                                   const uint8_t *to_rc, int64_t batch, int64_t ploidy, int parallel) {
    gvl_oracle_reconstruct_haplotypes_from_sparse(out, out_offsets, regions, shifts, geno_offset_idx, go_starts,
                                                  go_stops, geno_v_idxs, v_starts, ilens, alt_alleles, alt_offsets,
                                                  ref_, ref_offsets, pad_char, keep, keep_offsets, annot_v,
                                                  annot_pos, batch, ploidy, parallel);
    if (to_rc) { /* :842-853 / :2363-2385 -- serial, as in the reference */
        int64_t n_work = batch * ploidy;
        gvl_oracle_rc_flat_rows_inplace(out, out_offsets, to_rc, n_work);
        if (annot_v) gvl_oracle_reverse_flat_rows_inplace_32((uint32_t *)annot_v, out_offsets, to_rc, n_work);
        if (annot_pos) gvl_oracle_reverse_flat_rows_inplace_32((uint32_t *)annot_pos, out_offsets, to_rc, n_work);
    }
}

/* One-crossing form used by the timed CPU baseline: sizes, allocates (uninitialised),
 * fills and reverse-complements exactly like reconstruct_haplotypes_fused.  Returns the
 * malloc'ed data pointer (free with gvl_oracle_free); *total_out receives the byte count. */
GVL_API uint8_t *gvl_oracle_reconstruct_haplotypes_fused(
    const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, const int64_t *go_starts,
    const int64_t *go_stops, const int32_t *geno_v_idxs, const int32_t *v_starts, const int32_t *ilens,
    const uint8_t *alt_alleles, const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets,
    uint8_t pad_char, int64_t output_length, const uint8_t *keep, const int64_t *keep_offsets,
    const uint8_t *to_rc, int64_t batch, int64_t ploidy, int parallel, int64_t *out_offsets, int64_t *total_out) {
    int64_t total = gvl_oracle_fused_out_offsets(regions, geno_offset_idx, go_starts, go_stops, geno_v_idxs,
                                                 v_starts, ilens, output_length, keep, keep_offsets, batch, ploidy,
                                                 parallel, out_offsets, NULL);
    uint8_t *out = (uint8_t *)malloc((size_t)(total ? total : 1));
    gvl_oracle_fused_fill(out, NULL, NULL, out_offsets, regions, shifts, geno_offset_idx, go_starts, go_stops,
                          geno_v_idxs, v_starts, ilens, alt_alleles, alt_offsets, ref_, ref_offsets, pad_char, keep,
                          keep_offsets, to_rc, batch, ploidy, parallel);
    *total_out = total;
    return out;
}

GVL_API void gvl_oracle_free(void *p) { free(p); }

/* ====================================================================================
 * a14  one-hot (seqpro.DNA.ohe; third-party, parity unpinned -- see DESIGN.md)
 * out[j, c] = (in[j] == "ACGT"[c]), uint8, layout (n, 4).
 * ==================================================================================== */
typedef struct {
    const uint8_t *in;
    uint8_t *out;
    int64_t n;
    int64_t chunk;
} ohe_ctx;

static void ohe_task(void *p, int64_t k) {
    ohe_ctx *c = (ohe_ctx *)p;
    int64_t s = k * c->chunk, e = i64min(s + c->chunk, c->n);
    for (int64_t j = s; j < e; j++) {
        uint8_t b = c->in[j];
        uint8_t *o = c->out + 4 * j;
        o[0] = (b == 'A');
        o[1] = (b == 'C');
        o[2] = (b == 'G');
        o[3] = (b == 'T');
    }
}

GVL_API void gvl_oracle_onehot(const uint8_t *in, int64_t n, uint8_t *out, int parallel) {
    ohe_ctx c = {in, out, n, 1 << 16};
    gvl_parallel_for(ohe_task, &c, (n + c.chunk - 1) / c.chunk, parallel, 1);
}

/* ====================================================================================
 * a7  intervals_to_tracks                             src/intervals.rs:19-126
 * ==================================================================================== */
typedef struct {
    const int64_t *offset_idxs;
    const int32_t *starts;
    int64_t starts_stride;
    const int32_t *itv_starts, *itv_ends;
    const float *itv_values;
    const int64_t *itv_offsets;
    float *out;
    const int64_t *out_offsets;
} paint_ctx;

static void paint_task(void *p, int64_t query) {
    paint_ctx *c = (paint_ctx *)p;
    int64_t idx = c->offset_idxs[query];
    int64_t itv_s = c->itv_offsets[idx], itv_e = c->itv_offsets[idx + 1];
    if (itv_s == itv_e) return; /* :58-61 */
    float *out_chunk = c->out + c->out_offsets[query];
    int64_t length = c->out_offsets[query + 1] - c->out_offsets[query];
    int64_t query_start = c->starts[query * c->starts_stride];
    for (int64_t it = itv_s; it < itv_e; it++) {
        int64_t start = (int64_t)c->itv_starts[it] - query_start; /* :68-70 */
        int64_t end = (int64_t)c->itv_ends[it] - query_start;
        float value = c->itv_values[it];
        if (start >= length) break; /* :72-76 */
        int64_t s = i64max(start, 0), e = i64min(end, length);
        for (int64_t j = s; j < e; j++) out_chunk[j] = value; /* :84-86 */
    }
}

GVL_API void gvl_oracle_intervals_to_tracks(const int64_t *offset_idxs, const int32_t *starts,
                                            int64_t starts_stride, const int32_t *itv_starts,
                                            const int32_t *itv_ends, const float *itv_values,
                                            const int64_t *itv_offsets, float *out, const int64_t *out_offsets,
                                            int64_t n_queries, int parallel) {
    int64_t total = out_offsets[n_queries];
    memset(out, 0, sizeof(float) * (size_t)total); /* :45-49 out[:] = 0.0 */
    paint_ctx c = {offset_idxs, starts, starts_stride, itv_starts, itv_ends, itv_values, itv_offsets, out, out_offsets};
    gvl_parallel_for(paint_task, &c, n_queries, parallel, 1);
}

/* ====================================================================================
 * a9  PRNG + insertion fill                           src/tracks/mod.rs:31-54, 87-190
 * ==================================================================================== */
GVL_API uint64_t gvl_oracle_xorshift64(uint64_t x) { /* :31-36 */
    x ^= x << 13;
    x ^= x >> 7;
    x ^= x << 17;
    return x;
}

GVL_API uint64_t gvl_oracle_hash4(uint64_t a, uint64_t b, uint64_t c, uint64_t d) { /* :48-54 */
    uint64_t h = a;
    h = gvl_oracle_xorshift64(h ^ b);
    h = gvl_oracle_xorshift64(h ^ c);
    h = gvl_oracle_xorshift64(h ^ d);
    return h;
}

enum { REPEAT_5P = 0, REPEAT_5P_NORM = 1, CONSTANT = 2, FLANK_SAMPLE = 3, INTERPOLATE = 4 }; /* :15-19 */

/* A track value at relative source position i of a window of n values.  Positions outside the window are out of
 * the reference's contract (a slice index past the track panics, src/tracks/mod.rs:102-188, :317-404); they read 0
 * here, as past the end of a row (:400-404) and as the track kernels do. */
static inline float trk_at(const float *track, int64_t n, int64_t i) { return (i >= 0 && i < n) ? track[i] : 0.0f; }

/* `double` arithmetic below must not be contracted into FMAs: build with -ffp-contract=off. */
static void apply_insertion_fill(float *out, int64_t out_idx, int64_t writable_length, int64_t v_len,
                                 const float *track, int64_t track_len, int64_t v_rel_pos, int64_t strategy_id,
                                 const double *params, uint64_t base_seed, uint64_t query, uint64_t hap) {
    if (strategy_id == REPEAT_5P) { /* :102-108 */
        float val = trk_at(track, track_len, v_rel_pos);
        for (int64_t i = 0; i < writable_length; i++) out[out_idx + i] = val;
    } else if (strategy_id == REPEAT_5P_NORM) { /* :109-118 f32 / f32 */
        float val = trk_at(track, track_len, v_rel_pos) / (float)v_len;
        for (int64_t i = 0; i < writable_length; i++) out[out_idx + i] = val;
    } else if (strategy_id == CONSTANT) { /* :119-124 */
        float val = (float)params[0];
        for (int64_t i = 0; i < writable_length; i++) out[out_idx + i] = val;
    } else if (strategy_id == FLANK_SAMPLE) { /* :125-137 */
        int64_t width = (int64_t)params[0];
        int64_t pool_lo = i64max(v_rel_pos - width, 0);
        int64_t pool_hi = i64min(v_rel_pos + width, track_len - 1);
        uint64_t pool_size = (uint64_t)(pool_hi - pool_lo + 1);
        for (int64_t i = 0; i < writable_length; i++) {
            uint64_t seed = gvl_oracle_hash4(base_seed, query, hap, (uint64_t)(out_idx + i));
            int64_t offset = (int64_t)(seed % pool_size);
            out[out_idx + i] = trk_at(track, track_len, pool_lo + offset);
        }
    } else if (strategy_id == INTERPOLATE) { /* :138-188 */
        int64_t order = (int64_t)params[0];
        int64_t k = (order + 1 + 1) / 2;
        int64_t n_anchors = 2 * k;
        double xs[8], ys[8];
        for (int64_t j = 0; j < k; j++) { /* 5' side :153-157 */
            int64_t ri = i64max(v_rel_pos - j, 0);
            xs[j] = -(double)j;
            ys[j] = (double)trk_at(track, track_len, ri);
        }
        for (int64_t j = 0; j < k; j++) { /* 3' side :160-164 */
            int64_t ri = i64min(v_rel_pos + 1 + j, track_len - 1);
            xs[k + j] = (double)v_len + (double)j;
            ys[k + j] = (double)trk_at(track, track_len, ri);
        }
        for (int64_t i = 0; i < writable_length; i++) { /* :168-188 */
            double x = (double)i;
            double acc = 0.0;
            for (int64_t a = 0; a < n_anchors; a++) {
                double term = ys[a];
                for (int64_t b = 0; b < n_anchors; b++) {
                    if (b == a) continue;
                    term *= (x - xs[b]) / (xs[a] - xs[b]);
                }
                acc += term;
            }
            out[out_idx + i] = (float)acc;
        }
    }
}

/* ====================================================================================
 * a8  shift_and_realign_track_core                    src/tracks/mod.rs:224-406
 * ==================================================================================== */
typedef void (*gvl_provide_track_fn)(const void *src, int64_t v, int64_t *v_start, int64_t *v_diff);

static void shift_and_realign_track_core(int64_t n_variants, gvl_provide_track_fn provide, const void *src,
                                         int64_t shift, const float *track, int64_t track_n, int64_t query_start,
                                         float *out, int64_t length, const double *params, const uint8_t *keep,
                                         int64_t strategy_id, uint64_t base_seed, uint64_t query, uint64_t hap) {
    if (n_variants == 0) { /* :240-246 */
        for (int64_t i = 0; i < length; i++) out[i] = trk_at(track, track_n, i);
        return;
    }
    int64_t track_idx = 0, out_idx = 0, shifted = 0; /* :249-251 */
    for (int64_t v = 0; v < n_variants; v++) {
        if (keep && !keep[v]) continue; /* :255-259 */
        int64_t v_start, v_diff;
        provide(src, v, &v_start, &v_diff);
        int64_t v_rel_pos = v_start - query_start;              /* :264 */
        int64_t v_rel_end = v_rel_pos - i64min(v_diff, 0) + 1; /* :267 */
        if (v_diff < 0 && v_rel_pos < 0 && v_rel_end >= 0) {    /* :271-274 */
            track_idx = v_rel_end;
            continue;
        }
        if (v_rel_pos < track_idx) continue;     /* :277-279 */
        int64_t v_len = i64max(v_diff, 0) + 1;   /* :282 */
        if (shifted < shift) {                   /* :285-308 */
            int64_t ref_shift_dist = v_rel_pos - track_idx;
            if (shifted + ref_shift_dist + v_len < shift) {
                continue;
            } else if (shifted + ref_shift_dist >= shift) {
                track_idx += shift - shifted;
                shifted = shift;
            } else {
                int64_t allele_start_idx = shift - shifted - ref_shift_dist;
                shifted = shift;
                if (allele_start_idx == v_len) {
                    track_idx = v_rel_end;
                    continue;
                }
                track_idx = v_rel_pos;
                v_len -= allele_start_idx;
            }
        }
        if (v_diff == 0) continue; /* :312-314 SNPs match the reference track */
        int64_t track_len = v_rel_pos - track_idx;   /* :317 */
        if (out_idx + track_len >= length) break;    /* :319-321 */
        for (int64_t i = 0; i < track_len; i++) out[out_idx + i] = trk_at(track, track_n, track_idx + i);
        out_idx += track_len;
        int64_t writable_length = i64min(v_len, length - out_idx); /* :329 */
        if (v_diff > 0 && strategy_id != REPEAT_5P) {              /* :333-346 */
            apply_insertion_fill(out, out_idx, writable_length, v_len, track, track_n, v_rel_pos, strategy_id,
                                 params, base_seed, query, hap);
        } else { /* :347-354 */
            float val = trk_at(track, track_n, v_rel_pos);
            for (int64_t i = 0; i < writable_length; i++) out[out_idx + i] = val;
        }
        out_idx += writable_length;
        track_idx = v_rel_end;          /* :356 */
        if (out_idx >= length) break;   /* :359-361 */
    }
    if (shifted < shift) { /* :365-369 */
        track_idx += shift - shifted;
        track_idx = i64min(track_idx, track_n);
    }
    int64_t unfilled_length = length - out_idx; /* :373 */
    if (unfilled_length > 0) {
        int64_t writable_ref = i64min(unfilled_length, track_n - track_idx); /* :381 */
        int64_t out_end_idx;
        if (writable_ref > 0) {
            for (int64_t i = 0; i < writable_ref; i++) out[out_idx + i] = track[track_idx + i];
            out_end_idx = out_idx + writable_ref;
        } else {
            out_end_idx = out_idx;
        }
        for (int64_t i = out_end_idx; i < length; i++) out[i] = 0.0f; /* :400-404 */
    }
}

typedef struct {
    const int32_t *v_idxs;
    const int32_t *v_starts;
    const int32_t *ilens;
} sparse_track_src;

static void provide_track_sparse(const void *p, int64_t v, int64_t *v_start, int64_t *v_diff) {
    const sparse_track_src *s = (const sparse_track_src *)p; /* :453-456 */
    int64_t variant = s->v_idxs[v];
    *v_start = s->v_starts[variant];
    *v_diff = s->ilens[variant];
}

/* batch shift_and_realign_tracks_sparse               src/tracks/mod.rs:495-667 */
typedef struct {
    float *out;
    const int64_t *out_offsets;
    const int32_t *regions;
    const int32_t *shifts;
    const int64_t *geno_offset_idx;
    const int32_t *geno_v_idxs;
    const int64_t *go_starts, *go_stops;
    const int32_t *v_starts, *ilens;
    const float *tracks;
    const int64_t *track_offsets;
    const double *params;
    const uint8_t *keep;
    const int64_t *keep_offsets;
    int64_t strategy_id;
    uint64_t base_seed;
    int64_t ploidy;
} realign_ctx;

static void realign_task(void *p, int64_t k) {
    realign_ctx *c = (realign_ctx *)p;
    int64_t query = k / c->ploidy, hap = k % c->ploidy;
    int64_t t_s = c->track_offsets[query], t_e = c->track_offsets[query + 1];
    int64_t q_start = c->regions[query * 3 + 1];
    int64_t o_idx = c->geno_offset_idx[k];
    int64_t o_s = c->go_starts[o_idx], o_e = c->go_stops[o_idx];
    sparse_track_src s = {c->geno_v_idxs + o_s, c->v_starts, c->ilens};
    const uint8_t *qh_keep = (c->keep && c->keep_offsets) ? c->keep + c->keep_offsets[k] : NULL;
    int64_t os = c->out_offsets[k], oe = c->out_offsets[k + 1];
    shift_and_realign_track_core(o_e - o_s, provide_track_sparse, &s, c->shifts[k], c->tracks + t_s, t_e - t_s,
                                 q_start, c->out + os, oe - os, c->params, qh_keep, c->strategy_id, c->base_seed,
                                 (uint64_t)query, (uint64_t)hap);
}

GVL_API void gvl_oracle_shift_and_realign_tracks_sparse(
    float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, const int32_t *geno_v_idxs, const int64_t *go_starts, const int64_t *go_stops,
    const int32_t *v_starts, const int32_t *ilens, const float *tracks, const int64_t *track_offsets,
    const double *params, const uint8_t *keep, const int64_t *keep_offsets, int64_t strategy_id,
    uint64_t base_seed, int64_t n_regions, int64_t ploidy, int parallel) {
    realign_ctx c = {out, out_offsets, regions, shifts, geno_offset_idx, geno_v_idxs, go_starts, go_stops,
                     v_starts, ilens, tracks, track_offsets, params, keep, keep_offsets, strategy_id, base_seed,
                     ploidy};
    gvl_parallel_for(realign_task, &c, n_regions * ploidy, parallel, 1);
}

/* a10 intervals_and_realign_track_fused               src/ffi/mod.rs:2553-2672 */
GVL_API void gvl_oracle_intervals_and_realign_track_fused(
    float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, const int32_t *geno_v_idxs, const int64_t *go_starts, const int64_t *go_stops,
    const int32_t *v_starts, const int32_t *ilens, const int64_t *offset_idxs, const int32_t *itv_starts,
    const int32_t *itv_ends, const float *itv_values, const int64_t *itv_offsets, const int64_t *track_offsets,
    const double *params, int64_t strategy_id, uint64_t base_seed, const uint8_t *keep,
    const int64_t *keep_offsets, const uint8_t *to_rc, int64_t batch, int64_t ploidy, int parallel) {
    int64_t scratch_len = track_offsets[batch]; /* :2608 */
    float *scratch = (float *)malloc(sizeof(float) * (size_t)(scratch_len ? scratch_len : 1));
    gvl_oracle_intervals_to_tracks(offset_idxs, regions + 1, 3, itv_starts, itv_ends, itv_values, itv_offsets,
                                   scratch, track_offsets, batch, parallel); /* :2622-2632 */
    gvl_oracle_shift_and_realign_tracks_sparse(out, out_offsets, regions, shifts, geno_offset_idx, geno_v_idxs,
                                               go_starts, go_stops, v_starts, ilens, scratch, track_offsets, params,
                                               keep, keep_offsets, strategy_id, base_seed, batch, ploidy,
                                               parallel); /* :2635-2654 */
    if (to_rc) /* :2657-2668 reverse only */
        gvl_oracle_reverse_flat_rows_inplace_32((uint32_t *)out, out_offsets, to_rc, batch * ploidy);
    free(scratch);
}

/* ====================================================================================
 * a11  svar2 two-channel source                       src/svar2/mod.rs:17-146,
 *                                                     src/reconstruct/mod.rs:620-826,
 *                                                     src/tracks/mod.rs:705-856
 *
 * The 32-bit key codec (svar2-codec @ genoray 66ba734, decode_key) is a third-party
 * dependency absent from /root/reference: PARITY UNPINNED at the key-bit level.  This
 * restatement works at the DECODED level: a key is an index into a decoded-key table
 * (key_ilen[K], key_alt_off[K+1], key_alt bytes) that stands for decode_alt()'s result
 * (src/svar2/mod.rs:17-28): Inline/Lookup -> (alt.len()-1, alt); PureDel -> (ilen, empty).
 * Merge order, presence bits, diff semantics and the pure-DEL anchor are the reference's.
 * ==================================================================================== */
typedef struct {
    uint32_t pos;
    uint32_t key;
} pk_t;

static inline int present_bit(const uint8_t *dense_present, int64_t base_bit, int64_t j) { /* :35-38 */
    int64_t bit = base_bit + j;
    return (dense_present[bit / 8] >> (bit % 8)) & 1;
}

/* merge_hap :45-66 -- vk entries first, then set-bit dense entries, then STABLE sort by pos. */
static int64_t merge_hap(const int32_t *vk_pos, const int32_t *vk_key, int64_t vk_lo, int64_t vk_hi,
                         const int32_t *dense_pos, const int32_t *dense_key, int64_t ds, int64_t de,
                         const uint8_t *dense_present, int64_t base_bit, pk_t *a) {
    int64_t n = 0;
    for (int64_t i = vk_lo; i < vk_hi; i++) {
        a[n].pos = (uint32_t)vk_pos[i];
        a[n].key = (uint32_t)vk_key[i];
        n++;
    }
    for (int64_t j = ds, k = 0; j < de; j++, k++) {
        if (present_bit(dense_present, base_bit, k)) {
            a[n].pos = (uint32_t)dense_pos[j];
            a[n].key = (uint32_t)dense_key[j];
            n++;
        }
    }
    /* stable insertion sort by pos (inputs are two nearly-sorted runs; n is small) */
    for (int64_t i = 1; i < n; i++) {
        pk_t x = a[i];
        int64_t j = i - 1;
        while (j >= 0 && a[j].pos > x.pos) {
            a[j + 1] = a[j];
            j--;
        }
        a[j + 1] = x;
    }
    return n;
}

typedef struct {
    const pk_t *merged;
    const int32_t *key_ilen;
    const uint8_t *key_alt;
    const int64_t *key_alt_off;
    const uint8_t *contig_ref;
} svar2_src;

static void provide_svar2(const void *p, int64_t v, gvl_var *out) { /* reconstruct/mod.rs:711-735 */
    const svar2_src *s = (const svar2_src *)p;
    uint32_t pos = s->merged[v].pos, key = s->merged[v].key;
    int64_t a_s = s->key_alt_off[key], a_e = s->key_alt_off[key + 1];
    out->v_pos = (int64_t)pos;
    out->v_diff = s->key_ilen[key];
    if (a_e == a_s) { /* pure DEL: anchor base = ref[pos] (:720-733) */
        out->allele = s->contig_ref + pos;
        out->allele_len = 1;
    } else {
        out->allele = s->key_alt + a_s;
        out->allele_len = a_e - a_s;
    }
    out->annot_id = (int32_t)v;
}

static void provide_track_svar2(const void *p, int64_t v, int64_t *v_start, int64_t *v_diff) {
    const svar2_src *s = (const svar2_src *)p; /* tracks/mod.rs:705-856 provide closure */
    *v_start = (int64_t)s->merged[v].pos;
    *v_diff = s->key_ilen[s->merged[v].key];
}

typedef struct {
    uint8_t *out;
    float *out_f;
    const int64_t *out_bounds; /* (n_work,2) */
    const int32_t *regions, *shifts;
    const int32_t *vk_pos, *vk_key;
    const int64_t *vk_off;
    const int32_t *dense_pos, *dense_key, *dense_range;
    const uint8_t *dense_present;
    const int64_t *dense_present_off;
    const int32_t *key_ilen;
    const uint8_t *key_alt;
    const int64_t *key_alt_off;
    const uint8_t *ref_;
    const int64_t *ref_offsets;
    uint8_t pad_char;
    int64_t ploidy;
    int filter_exonic;
    /* tracks */
    const float *tracks;
    const int64_t *track_offsets;
    const double *params;
    int64_t strategy_id;
    uint64_t base_seed;
    const int64_t *query_seed;
    int32_t *diffs;
} svar2_ctx;

static int64_t svar2_merge_row(const svar2_ctx *c, int64_t k, pk_t **buf) {
    int64_t query = k / c->ploidy;
    int64_t vk_lo = c->vk_off[k], vk_hi = c->vk_off[k + 1];
    int64_t ds = c->dense_range[query * 2], de = c->dense_range[query * 2 + 1];
    pk_t *a = (pk_t *)malloc(sizeof(pk_t) * (size_t)((vk_hi - vk_lo) + (de - ds) + 1));
    *buf = a;
    return merge_hap(c->vk_pos, c->vk_key, vk_lo, vk_hi, c->dense_pos, c->dense_key, ds, de, c->dense_present,
                     c->dense_present_off[k], a);
}

static int64_t svar2_filter_exonic(const svar2_ctx *c, pk_t *a, int64_t n, int64_t ref_start, int64_t ref_end) {
    int64_t m = 0; /* reconstruct/mod.rs:700-708 */
    for (int64_t i = 0; i < n; i++) {
        int64_t v_start = a[i].pos, v_ilen = c->key_ilen[a[i].key];
        int64_t v_end = v_start - i64min(v_ilen, 0) + 1;
        if (v_start >= ref_start && v_end <= ref_end) a[m++] = a[i];
    }
    return m;
}

static void svar2_recon_task(void *p, int64_t k) {
    svar2_ctx *c = (svar2_ctx *)p;
    int64_t query = k / c->ploidy;
    int64_t c_idx = c->regions[query * 3];
    int64_t c_s = c->ref_offsets[c_idx], c_e = c->ref_offsets[c_idx + 1];
    int64_t ref_start = c->regions[query * 3 + 1];
    pk_t *a;
    int64_t n = svar2_merge_row(c, k, &a);
    if (c->filter_exonic) n = svar2_filter_exonic(c, a, n, ref_start, c->regions[query * 3 + 2]);
    svar2_src s = {a, c->key_ilen, c->key_alt, c->key_alt_off, c->ref_ + c_s};
    int64_t os = c->out_bounds[k * 2], oe = c->out_bounds[k * 2 + 1];
    reconstruct_haplotype_core(n, provide_svar2, &s, c->shifts[k], c->ref_ + c_s, c_e - c_s, ref_start,
                               c->out + os, oe - os, c->pad_char, NULL, NULL, NULL);
    free(a);
}

GVL_API void gvl_oracle_reconstruct_haplotypes_from_svar2(
    uint8_t *out, const int64_t *out_bounds, const int32_t *regions, const int32_t *shifts, const int32_t *vk_pos,
    const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos, const int32_t *dense_key,
    const int32_t *dense_range, const uint8_t *dense_present, const int64_t *dense_present_off,
    const int32_t *key_ilen, const uint8_t *key_alt, const int64_t *key_alt_off, const uint8_t *ref_,
    const int64_t *ref_offsets, uint8_t pad_char, int64_t batch, int64_t ploidy, int parallel, int filter_exonic) {
    svar2_ctx c;
    memset(&c, 0, sizeof(c));
    c.out = out; c.out_bounds = out_bounds; c.regions = regions; c.shifts = shifts;
    c.vk_pos = vk_pos; c.vk_key = vk_key; c.vk_off = vk_off;
    c.dense_pos = dense_pos; c.dense_key = dense_key; c.dense_range = dense_range;
    c.dense_present = dense_present; c.dense_present_off = dense_present_off;
    c.key_ilen = key_ilen; c.key_alt = key_alt; c.key_alt_off = key_alt_off;
    c.ref_ = ref_; c.ref_offsets = ref_offsets; c.pad_char = pad_char; c.ploidy = ploidy;
    c.filter_exonic = filter_exonic;
    gvl_parallel_for(svar2_recon_task, &c, batch * ploidy, parallel, 1);
}

/* hap_diffs_svar2                                     src/svar2/mod.rs:73-146 */
static void svar2_diffs_task(void *p, int64_t k) {
    svar2_ctx *c = (svar2_ctx *)p;
    int64_t query = k / c->ploidy;
    pk_t *a;
    int64_t n = svar2_merge_row(c, k, &a);
    int64_t acc = 0;
    if (n > 0) {
        int64_t q_start = c->regions[query * 3 + 1], q_end = c->regions[query * 3 + 2];
        int64_t ref_idx = q_start;
        for (int64_t i = 0; i < n; i++) {
            int64_t v_start = a[i].pos, v_ilen = c->key_ilen[a[i].key];
            int64_t v_end = v_start - i64min(v_ilen, 0) + 1;
            if (c->filter_exonic && (v_start < q_start || v_end > q_end)) continue;
            if (v_end <= q_start) continue;
            if (v_start >= q_end) break;
            if (v_start >= q_start && v_start < ref_idx) continue;
            ref_idx = i64max(ref_idx, v_end);
            if (v_ilen < 0) v_ilen += i64max(q_start - v_start - 1, 0);
            v_ilen += i64max(v_end - q_end, 0);
            acc += v_ilen;
        }
    }
    c->diffs[k] = (int32_t)acc;
    free(a);
}

GVL_API void gvl_oracle_hap_diffs_svar2(const int32_t *regions, int64_t batch, int64_t ploidy, const int32_t *vk_pos,
                                        const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos,
                                        const int32_t *dense_key, const int32_t *dense_range,
                                        const uint8_t *dense_present, const int64_t *dense_present_off,
                                        const int32_t *key_ilen, int filter_exonic, int32_t *diffs) {
    svar2_ctx c;
    memset(&c, 0, sizeof(c));
    c.regions = regions; c.ploidy = ploidy; c.vk_pos = vk_pos; c.vk_key = vk_key; c.vk_off = vk_off;
    c.dense_pos = dense_pos; c.dense_key = dense_key; c.dense_range = dense_range;
    c.dense_present = dense_present; c.dense_present_off = dense_present_off; c.key_ilen = key_ilen;
    c.filter_exonic = filter_exonic; c.diffs = diffs;
    gvl_parallel_for(svar2_diffs_task, &c, batch * ploidy, 0, 1); /* serial in the reference */
}

/* shift_and_realign_tracks_from_svar2                 src/tracks/mod.rs:705-856 */
static void svar2_track_task(void *p, int64_t k) {
    svar2_ctx *c = (svar2_ctx *)p;
    int64_t query = k / c->ploidy, hap = k % c->ploidy;
    int64_t t_s = c->track_offsets[query], t_e = c->track_offsets[query + 1];
    int64_t q_start = c->regions[query * 3 + 1];
    pk_t *a;
    int64_t n = svar2_merge_row(c, k, &a);
    svar2_src s = {a, c->key_ilen, c->key_alt, c->key_alt_off, NULL};
    int64_t os = c->out_bounds[k], oe = c->out_bounds[k + 1]; /* 1-D out_offsets here (:707) */
    uint64_t qseed = c->query_seed ? (uint64_t)c->query_seed[query] : (uint64_t)query;
    shift_and_realign_track_core(n, provide_track_svar2, &s, c->shifts[k], c->tracks + t_s, t_e - t_s, q_start,
                                 c->out_f + os, oe - os, c->params, NULL, c->strategy_id, c->base_seed, qseed,
                                 (uint64_t)hap);
    free(a);
}

GVL_API void gvl_oracle_shift_and_realign_tracks_from_svar2(
    float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts, const int32_t *vk_pos,
    const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos, const int32_t *dense_key,
    const int32_t *dense_range, const uint8_t *dense_present, const int64_t *dense_present_off,
    const int32_t *key_ilen, const float *tracks, const int64_t *track_offsets, const double *params,
    int64_t strategy_id, uint64_t base_seed, const int64_t *query_seed, int64_t batch, int64_t ploidy,
    int parallel) {
    svar2_ctx c;
    memset(&c, 0, sizeof(c));
    c.out_f = out; c.out_bounds = out_offsets; c.regions = regions; c.shifts = shifts;
    c.vk_pos = vk_pos; c.vk_key = vk_key; c.vk_off = vk_off;
    c.dense_pos = dense_pos; c.dense_key = dense_key; c.dense_range = dense_range;
    c.dense_present = dense_present; c.dense_present_off = dense_present_off; c.key_ilen = key_ilen;
    c.tracks = tracks; c.track_offsets = track_offsets; c.params = params; c.strategy_id = strategy_id;
    c.base_seed = base_seed; c.query_seed = query_seed; c.ploidy = ploidy;
    gvl_parallel_for(svar2_track_task, &c, batch * ploidy, parallel, 1);
}

/* ====================================================================================
 * a13  ragged_to_padded                               src/ragged/mod.rs:7-23
 * (seqpro-core 0.1.0 Ragged::to_padded_into: copy min(len, out_len) items of each row into
 * a PRE-FILLED (n_rows, out_len) buffer; the pad value is whatever the caller filled.)
 * ==================================================================================== */
GVL_API void gvl_oracle_ragged_to_padded(const uint8_t *data, const int64_t *offsets, int64_t n_rows, uint8_t *out,
                                         int64_t itemsize, int64_t out_len) {
    for (int64_t r = 0; r < n_rows; r++) {
        int64_t n = i64min(offsets[r + 1] - offsets[r], out_len);
        memcpy(out + r * out_len * itemsize, data + offsets[r] * itemsize, (size_t)(n * itemsize));
    }
}
