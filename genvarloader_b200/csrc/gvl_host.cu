// gvl_host.cu -- HOST-buffer entries of the C ABI: same argument lists as the reference's
// #[pyfunction]s (src/ffi/mod.rs), host pointers in, host pointers out.
//
// Static arrays (reference, variant table, genotype CSR, interval SoA) are uploaded once and
// cached by host address; O(batch) arrays travel through one pinned staging buffer and one
// H2D copy per call; outputs come back with one D2H copy per array.
#include <cstring>

#include "gvl_internal.cuh"

namespace gvl {

static inline int64_t round16(int64_t x) { return (x + 15) & ~(int64_t)15; }

// scratch slot i: a growable device buffer private to the host layer
static int scratch(gvl_ctx *ctx, size_t slot, int64_t bytes, void **dev);

// upload a static array into its own allocation and register it by host address
static int pin_static(gvl_ctx *ctx, const void *host, int64_t bytes, const void **dev) {
    void *d = nullptr;
    const int64_t cap = round16(bytes) + 16;  // slack: 32-bit loads may touch up to the next 16 B
    GVL_CUDA(cudaMalloc(&d, (size_t)cap));
    GVL_CUDA(cudaMemsetAsync((char *)d + (bytes / 16) * 16, 0, (size_t)(cap - (bytes / 16) * 16), ctx->own_stream));
    if (bytes) GVL_CUDA(cudaMemcpyAsync(d, host, (size_t)bytes, cudaMemcpyHostToDevice, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    ctx->statics[host] = gvl_static_entry{d, bytes};
    if (dev) *dev = d;
    return GVL_OK;
}

// device view of a sample-scale host array: the pinned copy when the caller registered it with
// gvl_pin_static (same address and size), otherwise a per-call upload into scratch slot `slot`.
static int static_dev(gvl_ctx *ctx, const void *host, int64_t bytes, size_t slot, const void **dev) {
    if (!host) {
        *dev = nullptr;
        return GVL_OK;
    }
    auto it = ctx->statics.find(host);
    if (it != ctx->statics.end() && it->second.bytes == bytes) {
        *dev = it->second.dev;
        return GVL_OK;
    }
    void *d;
    int rc;
    if ((rc = scratch(ctx, slot, bytes + 32, &d))) return rc;
    GVL_CUDA(cudaMemsetAsync((char *)d + (bytes / 16) * 16, 0, 32, ctx->own_stream));
    if (bytes) GVL_CUDA(cudaMemcpyAsync(d, host, (size_t)bytes, cudaMemcpyHostToDevice, ctx->own_stream));
    *dev = d;
    return GVL_OK;
}

// packed (4-bit) copy of a PINNED reference, built on first use and kept until the reference is unpinned;
// references uploaded per call keep the byte-oriented kernel (packing would cost more than it saves)
static int packed_ref(gvl_ctx *ctx, const void *host_ref, const uint8_t *dev_ref, int64_t n_bases,
                      const uint32_t **out) {
    *out = nullptr;
    auto st = ctx->statics.find(host_ref);
    if (st == ctx->statics.end() || st->second.dev != (void *)dev_ref) return GVL_OK;
    auto it = ctx->packed_refs.find(dev_ref);
    if (it == ctx->packed_refs.end()) {
        void *d = nullptr;
        GVL_CUDA(cudaMalloc(&d, sizeof(uint32_t) * (size_t)gvl_packed_reference_words(n_bases)));
        int rc = gvl_dev_pack_reference(ctx, dev_ref, n_bases, (uint32_t *)d, ctx->own_stream);
        if (rc) {
            cudaFree(d);
            return rc;
        }
        it = ctx->packed_refs.emplace(dev_ref, d).first;
    }
    *out = (const uint32_t *)it->second;
    return GVL_OK;
}

static void drop_packed(gvl_ctx *ctx, const void *dev_ref) {
    auto it = ctx->packed_refs.find(dev_ref);
    if (it != ctx->packed_refs.end()) {
        cudaFree(it->second);
        ctx->packed_refs.erase(it);
    }
}

static int scratch(gvl_ctx *ctx, size_t slot, int64_t bytes, void **dev) {
    if (ctx->scratch.size() <= slot) ctx->scratch.resize(slot + 1, {nullptr, 0});
    auto &s = ctx->scratch[slot];
    if (s.second < bytes || !s.first) {
        if (s.first) GVL_CUDA(cudaFree(s.first));
        s.first = nullptr;
        int64_t cap = round16(bytes + bytes / 4) + 256;
        GVL_CUDA(cudaMalloc(&s.first, (size_t)cap));
        s.second = cap;
    }
    *dev = s.first;
    return GVL_OK;
}

static int pinned(gvl_ctx *ctx, int64_t bytes, void **p) {
    if (ctx->pinned_bytes < bytes) {
        if (ctx->pinned) GVL_CUDA(cudaFreeHost(ctx->pinned));
        ctx->pinned = nullptr;
        int64_t cap = round16(bytes * 2) + 4096;
        GVL_CUDA(cudaHostAlloc(&ctx->pinned, (size_t)cap, cudaHostAllocDefault));
        ctx->pinned_bytes = cap;
    }
    *p = ctx->pinned;
    return GVL_OK;
}

// Pack several small host arrays into the pinned buffer, upload with ONE copy, hand back device pointers.
struct Packer {
    struct Item {
        const void *host;
        int64_t bytes;
        int64_t off;
    };
    std::vector<Item> items;
    int64_t total = 0;
    size_t add(const void *host, int64_t bytes) {
        Item it{host, host ? bytes : 0, total};
        if (host) total += round16(bytes) + 16;
        items.push_back(it);
        return items.size() - 1;
    }
    char *dev_base = nullptr;
    int upload(gvl_ctx *ctx, size_t slot) {
        void *pin, *dev;
        int rc;
        if ((rc = pinned(ctx, total + 16, &pin))) return rc;
        if ((rc = scratch(ctx, slot, total + 16, &dev))) return rc;
        for (auto &it : items)
            if (it.host && it.bytes) memcpy((char *)pin + it.off, it.host, (size_t)it.bytes);
        if (total) GVL_CUDA(cudaMemcpyAsync(dev, pin, (size_t)total, cudaMemcpyHostToDevice, ctx->own_stream));
        dev_base = (char *)dev;
        return GVL_OK;
    }
    template <typename T>
    const T *ptr(size_t i) const {
        return items[i].host ? reinterpret_cast<const T *>(dev_base + items[i].off) : nullptr;
    }
};

static int64_t sum_variants(const int64_t *geno_offsets, int64_t n_geno, const int64_t *goi, int64_t n_work) {
    int64_t s = 0;
    for (int64_t k = 0; k < n_work; k++) {
        int64_t o = goi[k];
        int64_t d = geno_offsets[n_geno + o] - geno_offsets[o];
        if (d > 0) s += d;
    }
    return s;
}

// ---- svar2 two-channel source: host arrays -> device channel struct (three entries share this) ----
struct Svar2Host {
    const int32_t *vk_pos, *vk_key;
    const int64_t *vk_off;
    const int32_t *dense_pos, *dense_key;
    int64_t n_dense;
    const int32_t *dense_range;
    const uint8_t *dense_present;
    const int64_t *dense_present_off;
};

struct Svar2Slots {
    size_t vp, vk, vo, dr, dp, dpo;
    int64_t max_merged;  // sum over rows of (var_key entries + dense window size): the merge workspace
};

// the shared dense channel is sample-scale: pinned copy when registered, per-call upload otherwise
static int svar2_static(gvl_ctx *ctx, const Svar2Host &h, gvl_svar2_channels *ch) {
    int rc;
    const void *d;
    memset(ch, 0, sizeof(*ch));  // (per-call flat layout: no resident-table indirection)
    if ((rc = static_dev(ctx, h.dense_pos, sizeof(int32_t) * h.n_dense, 16, &d))) return rc;
    ch->dense_pos = (const int32_t *)d;
    if ((rc = static_dev(ctx, h.dense_key, sizeof(int32_t) * h.n_dense, 17, &d))) return rc;
    ch->dense_key = (const int32_t *)d;
    return GVL_OK;
}

// the O(batch) channel arrays join the call's single staged upload (NULL arrays of empty channels get a placeholder)
static Svar2Slots svar2_add(Packer &pk, const Svar2Host &h, int64_t batch, int64_t ploidy) {
    const int64_t n_work = batch * ploidy;
    const int64_t n_vk = h.vk_off[n_work];
    const int64_t n_bits = h.dense_present_off[n_work];
    Svar2Slots s;
    s.max_merged = n_vk;
    for (int64_t q = 0; q < batch; q++) {
        const int64_t w = (int64_t)h.dense_range[2 * q + 1] - h.dense_range[2 * q];
        if (w > 0) s.max_merged += ploidy * w;
    }
    s.vp = pk.add(h.vk_pos ? (const void *)h.vk_pos : (const void *)h.vk_off, sizeof(int32_t) * n_vk);
    s.vk = pk.add(h.vk_key ? (const void *)h.vk_key : (const void *)h.vk_off, sizeof(int32_t) * n_vk);
    s.vo = pk.add(h.vk_off, sizeof(int64_t) * (n_work + 1));
    s.dr = pk.add(h.dense_range, sizeof(int32_t) * 2 * batch);
    s.dp = pk.add(h.dense_present ? (const void *)h.dense_present : (const void *)h.vk_off, (n_bits + 7) / 8);
    s.dpo = pk.add(h.dense_present_off, sizeof(int64_t) * (n_work + 1));
    return s;
}

static void svar2_resolve(const Packer &pk, const Svar2Slots &s, gvl_svar2_channels *ch) {
    ch->vk_pos = pk.ptr<int32_t>(s.vp);
    ch->vk_key = pk.ptr<int32_t>(s.vk);
    ch->vk_off = pk.ptr<int64_t>(s.vo);
    ch->dense_range = pk.ptr<int32_t>(s.dr);
    ch->dense_present = pk.ptr<uint8_t>(s.dp);
    ch->dense_present_off = pk.ptr<int64_t>(s.dpo);
}

}  // namespace gvl

using namespace gvl;

namespace gvl {
// ---- overlapping intervals ---------------------------------------------------------------------------------
// The reference paints a slot's intervals in stored order, later intervals overwriting earlier ones
// (src/intervals.rs:64-85); annotation tables are sorted by start but never merged, so overlaps are legal data.  The
// execute kernel paints a run-length code and needs disjoint intervals: a slot with overlaps is replaced by the
// equivalent disjoint, sorted list ("last write wins" resolved once, here on the host).
static bool slot_overlaps(const int32_t *s, const int32_t *e, int64_t n) {
    int32_t reach = INT32_MIN;  // furthest end of the non-empty intervals seen so far
    for (int64_t i = 0; i < n; i++) {
        if (e[i] <= s[i]) continue;
        if (s[i] < reach) return true;
        reach = e[i] > reach ? e[i] : reach;
    }
    return false;
}

static void flatten_slot(const int32_t *s, const int32_t *e, const float *v, int64_t n, std::vector<int32_t> &os,
                         std::vector<int32_t> &oe, std::vector<float> &ov) {
    const size_t base = os.size();  // pieces of this slot live in [base, os.size()): sorted, disjoint
    std::vector<int32_t> ts, te;
    std::vector<float> tv;
    for (int64_t i = 0; i < n; i++) {
        const int32_t a = s[i], b = e[i];
        if (b <= a) continue;
        size_t k = os.size();  // first piece whose end lies beyond a (ends are sorted: search from the tail)
        while (k > base && oe[k - 1] > a) k--;
        ts.clear(), te.clear(), tv.clear();
        for (size_t j = k; j < os.size(); j++) {  // what the new interval leaves of the pieces it meets
            if (os[j] < a) ts.push_back(os[j]), te.push_back(a), tv.push_back(ov[j]);
        }
        ts.push_back(a), te.push_back(b), tv.push_back(v[i]);
        for (size_t j = k; j < os.size(); j++) {
            if (oe[j] > b) ts.push_back(os[j] > b ? os[j] : b), te.push_back(oe[j]), tv.push_back(ov[j]);
        }
        os.resize(k), oe.resize(k), ov.resize(k);
        os.insert(os.end(), ts.begin(), ts.end());
        oe.insert(oe.end(), te.begin(), te.end());
        ov.insert(ov.end(), tv.begin(), tv.end());
    }
}

}  // namespace gvl
using namespace gvl;

extern "C" {

int gvl_intervals_overlap(const int32_t *itv_starts, const int32_t *itv_ends, const int64_t *itv_offsets, int64_t n_slots,
                          int64_t *n_overlapping) {
    if (!itv_offsets || !n_overlapping || (n_slots > 0 && itv_offsets[n_slots] > 0 && (!itv_starts || !itv_ends)))
        return fail(GVL_ERR_ARG, "gvl_intervals_overlap: NULL argument");
    int64_t c = 0;
    for (int64_t k = 0; k < n_slots; k++)
        c += slot_overlaps(itv_starts + itv_offsets[k], itv_ends + itv_offsets[k], itv_offsets[k + 1] - itv_offsets[k]) ? 1 : 0;
    *n_overlapping = c;
    return GVL_OK;
}

int gvl_flatten_intervals(const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
                          const int64_t *itv_offsets, int64_t n_slots, int32_t *out_starts, int32_t *out_ends,
                          float *out_values, int64_t *out_offsets, int64_t out_cap, int64_t *out_n) {
    if (!itv_offsets || !out_offsets || !out_n) return fail(GVL_ERR_ARG, "gvl_flatten_intervals: NULL argument");
    std::vector<int32_t> os, oe;
    std::vector<float> ov;
    out_offsets[0] = 0;
    for (int64_t k = 0; k < n_slots; k++) {
        const int64_t lo = itv_offsets[k], n = itv_offsets[k + 1] - lo;
        if (slot_overlaps(itv_starts + lo, itv_ends + lo, n)) {
            flatten_slot(itv_starts + lo, itv_ends + lo, itv_values + lo, n, os, oe, ov);
        } else {
            os.insert(os.end(), itv_starts + lo, itv_starts + lo + n);
            oe.insert(oe.end(), itv_ends + lo, itv_ends + lo + n);
            ov.insert(ov.end(), itv_values + lo, itv_values + lo + n);
        }
        out_offsets[k + 1] = (int64_t)os.size();
    }
    *out_n = (int64_t)os.size();
    if ((int64_t)os.size() > out_cap) return fail(GVL_ERR_CAPACITY, "gvl_flatten_intervals: %lld intervals, capacity %lld",
                                                  (long long)os.size(), (long long)out_cap);
    if (!os.empty()) {
        if (!out_starts || !out_ends || !out_values) return fail(GVL_ERR_ARG, "gvl_flatten_intervals: NULL output");
        memcpy(out_starts, os.data(), sizeof(int32_t) * os.size());
        memcpy(out_ends, oe.data(), sizeof(int32_t) * oe.size());
        memcpy(out_values, ov.data(), sizeof(float) * ov.size());
    }
    return GVL_OK;
}

int gvl_host_alloc(int64_t bytes, void **out) {
    if (!out) return fail(GVL_ERR_ARG, "gvl_host_alloc: out is NULL");
    GVL_CUDA(cudaHostAlloc(out, (size_t)(bytes > 0 ? bytes : 1), cudaHostAllocDefault));
    return GVL_OK;
}

int gvl_host_free(void *p) {
    if (p) GVL_CUDA(cudaFreeHost(p));
    return GVL_OK;
}

int gvl_pin_static(gvl_ctx *ctx, const void *host_ptr, int64_t bytes) {
    if (!ctx || !host_ptr) return fail(GVL_ERR_ARG, "gvl_pin_static: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    auto it = ctx->statics.find(host_ptr);
    if (it != ctx->statics.end()) {  // refresh
        GVL_CUDA(cudaDeviceSynchronize());
        drop_packed(ctx, it->second.dev);
        cudaFree(it->second.dev);
        ctx->statics.erase(it);
    }
    return pin_static(ctx, host_ptr, bytes, nullptr);
}

int gvl_unpin_static(gvl_ctx *ctx, const void *host_ptr) {
    if (!ctx) return fail(GVL_ERR_ARG, "gvl_unpin_static: ctx is NULL");
    auto it = ctx->statics.find(host_ptr);
    if (it == ctx->statics.end()) return GVL_OK;
    GVL_CUDA(cudaSetDevice(ctx->device));
    GVL_CUDA(cudaDeviceSynchronize());
    drop_packed(ctx, it->second.dev);
    cudaFree(it->second.dev);
    ctx->statics.erase(it);
    return GVL_OK;
}

static int resolve_tables(gvl_ctx *ctx, const int64_t *geno_offsets, int64_t n_geno, const int32_t *geno_v_idxs,
                          int64_t n_geno_v, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
                          const uint8_t *alt_alleles, const int64_t *alt_offsets, const uint8_t *ref_,
                          const int64_t *ref_offsets, int64_t n_contigs, gvl_sparse_tables *t) {
    int rc;
    const void *d;
    memset(t, 0, sizeof(*t));
    if ((rc = static_dev(ctx, geno_offsets, sizeof(int64_t) * 2 * n_geno, 8, &d))) return rc;
    t->geno_starts = (const int64_t *)d;
    t->geno_stops = t->geno_starts ? t->geno_starts + n_geno : nullptr;
    t->n_geno = n_geno;
    if ((rc = static_dev(ctx, geno_v_idxs, sizeof(int32_t) * n_geno_v, 9, &d))) return rc;
    t->geno_v_idxs = (const int32_t *)d;
    if ((rc = static_dev(ctx, v_starts, sizeof(int32_t) * n_variants, 10, &d))) return rc;
    t->v_starts = (const int32_t *)d;
    if ((rc = static_dev(ctx, ilens, sizeof(int32_t) * n_variants, 11, &d))) return rc;
    t->ilens = (const int32_t *)d;
    t->n_variants = n_variants;
    if (alt_offsets) {
        if ((rc = static_dev(ctx, alt_offsets, sizeof(int64_t) * (n_variants + 1), 12, &d))) return rc;
        t->alt_offsets = (const int64_t *)d;
        if ((rc = static_dev(ctx, alt_alleles, alt_offsets[n_variants], 13, &d))) return rc;
        t->alt_alleles = (const uint8_t *)d;
        if ((rc = packed_ref(ctx, alt_alleles, t->alt_alleles, alt_offsets[n_variants], &t->alt_packed))) return rc;
    }
    if (ref_offsets) {
        if ((rc = static_dev(ctx, ref_offsets, sizeof(int64_t) * (n_contigs + 1), 14, &d))) return rc;
        t->ref_offsets = (const int64_t *)d;
        if ((rc = static_dev(ctx, ref_, ref_offsets[n_contigs], 15, &d))) return rc;
        t->ref = (const uint8_t *)d;
        t->n_contigs = n_contigs;
        if ((rc = packed_ref(ctx, ref_, t->ref, ref_offsets[n_contigs], &t->ref_packed))) return rc;
    }
    return GVL_OK;
}

static int hap_begin(
    gvl_ctx *ctx, const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
    int64_t ploidy, const int64_t *geno_offsets, int64_t n_geno, const int32_t *geno_v_idxs, int64_t n_geno_v,
    const int32_t *v_starts, const int32_t *ilens, int64_t n_variants, const uint8_t *alt_alleles,
    const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets, int64_t n_contigs,
    int64_t output_length, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
    int64_t *out_offsets, int64_t *total) {
    if (!ctx || !regions || !shifts || !geno_offset_idx || !geno_offsets || !geno_v_idxs || !v_starts || !ilens ||
        !alt_offsets || !ref_offsets || !out_offsets || !total)
        return fail(GVL_ERR_ARG, "gvl_reconstruct_haplotypes_fused_begin: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t n_work = batch * ploidy;
    if ((rc = resolve_tables(ctx, geno_offsets, n_geno, geno_v_idxs, n_geno_v, v_starts, ilens, n_variants, alt_alleles,
                             alt_offsets, ref_, ref_offsets, n_contigs, &ctx->host_tab)))
        return rc;
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * batch);
    size_t i_sh = pk.add(shifts, sizeof(int32_t) * n_work);
    size_t i_goi = pk.add(geno_offset_idx, sizeof(int64_t) * n_work);
    size_t i_ko = pk.add(keep_offsets, sizeof(int64_t) * (n_work + 1));
    size_t i_kp = pk.add(keep, keep_offsets ? keep_offsets[n_work] : 0);
    size_t i_rc = pk.add(to_rc, n_work);
    if ((rc = pk.upload(ctx, 0))) return rc;
    void *oo_dev;
    if ((rc = scratch(ctx, 1, sizeof(int64_t) * (n_work + 1), &oo_dev))) return rc;
    ctx->host_out_offsets_dev = (int64_t *)oo_dev;
    if (output_length == -2)  // caller-sized rows: offsets are an input
        GVL_CUDA(cudaMemcpyAsync(oo_dev, out_offsets, sizeof(int64_t) * (n_work + 1), cudaMemcpyHostToDevice, ctx->own_stream));
    const int64_t max_rec = sum_variants(geno_offsets, n_geno, geno_offset_idx, n_work);
    if ((rc = gvl_dev_hap_plan(ctx, &ctx->host_tab, pk.ptr<int32_t>(i_reg), pk.ptr<int32_t>(i_sh), pk.ptr<int64_t>(i_goi),
                               batch, ploidy, keep && keep_offsets ? pk.ptr<uint8_t>(i_kp) : nullptr,
                               keep && keep_offsets ? pk.ptr<int64_t>(i_ko) : nullptr, pk.ptr<uint8_t>(i_rc),
                               output_length, max_rec, ctx->host_out_offsets_dev, nullptr, ctx->own_stream)))
        return rc;
    if (output_length != -2)
        GVL_CUDA(cudaMemcpyAsync(out_offsets, oo_dev, sizeof(int64_t) * (n_work + 1), cudaMemcpyDeviceToHost, ctx->own_stream));
    if ((rc = gvl_ctx_check(ctx, ctx->own_stream))) return rc;  // syncs; reports workspace overflow
    if (ctx->total < 0) ctx->total = ctx->host_words[W_TOTAL];
    *total = ctx->total;
    return GVL_OK;
}

int gvl_reconstruct_haplotypes_fused_begin(
    gvl_ctx *ctx, const int32_t *regions, const int32_t *shifts, const int64_t *geno_offset_idx, int64_t batch,
    int64_t ploidy, const int64_t *geno_offsets, int64_t n_geno, const int32_t *geno_v_idxs, int64_t n_geno_v,
    const int32_t *v_starts, const int32_t *ilens, int64_t n_variants, const uint8_t *alt_alleles,
    const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets, int64_t n_contigs,
    int64_t output_length, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc,
    int64_t *out_offsets, int64_t *total) {
    if (output_length < -1) return fail(GVL_ERR_ARG, "output_length must be >= -1");
    return hap_begin(ctx, regions, shifts, geno_offset_idx, batch, ploidy, geno_offsets, n_geno, geno_v_idxs, n_geno_v,
                     v_starts, ilens, n_variants, alt_alleles, alt_offsets, ref_, ref_offsets, n_contigs, output_length,
                     keep, keep_offsets, to_rc, out_offsets, total);
}

int gvl_reconstruct_haplotypes_from_svar2_begin(
    gvl_ctx *ctx, const int32_t *regions, const int32_t *shifts, int64_t batch, int64_t ploidy, const int32_t *vk_pos,
    const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos, const int32_t *dense_key, int64_t n_dense,
    const int32_t *dense_range, const uint8_t *dense_present, const int64_t *dense_present_off, const int32_t *key_ilen,
    const uint8_t *key_alt, const int64_t *key_alt_off, int64_t n_keys, const uint8_t *ref_, const int64_t *ref_offsets,
    int64_t n_contigs, int64_t output_length, const uint8_t *to_rc, int64_t *out_offsets, int64_t *total) {
    if (!ctx || !regions || !shifts || !vk_off || !dense_range || !dense_present_off || !key_ilen || !key_alt_off ||
        !ref_offsets || !out_offsets || !total)
        return fail(GVL_ERR_ARG, "gvl_reconstruct_haplotypes_from_svar2_begin: NULL argument");
    if (output_length < -1) return fail(GVL_ERR_ARG, "output_length must be >= -1");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t n_work = batch * ploidy;
    const void *d;
    gvl_sparse_tables &t = ctx->host_tab;
    memset(&t, 0, sizeof(t));
    if ((rc = static_dev(ctx, key_ilen, sizeof(int32_t) * n_keys, 11, &d))) return rc;
    t.ilens = (const int32_t *)d;
    t.v_starts = t.ilens;  // unused by the merged-list source
    t.n_variants = n_keys;
    if ((rc = static_dev(ctx, key_alt_off, sizeof(int64_t) * (n_keys + 1), 12, &d))) return rc;
    t.alt_offsets = (const int64_t *)d;
    if ((rc = static_dev(ctx, key_alt, key_alt_off[n_keys], 13, &d))) return rc;
    t.alt_alleles = (const uint8_t *)d;
    if ((rc = packed_ref(ctx, key_alt, t.alt_alleles, key_alt_off[n_keys], &t.alt_packed))) return rc;
    if ((rc = static_dev(ctx, ref_offsets, sizeof(int64_t) * (n_contigs + 1), 14, &d))) return rc;
    t.ref_offsets = (const int64_t *)d;
    if ((rc = static_dev(ctx, ref_, ref_offsets[n_contigs], 15, &d))) return rc;
    t.ref = (const uint8_t *)d;
    if ((rc = packed_ref(ctx, ref_, t.ref, ref_offsets[n_contigs], &t.ref_packed))) return rc;
    t.n_contigs = n_contigs;
    const Svar2Host sh{vk_pos, vk_key, vk_off, dense_pos, dense_key, n_dense, dense_range, dense_present, dense_present_off};
    gvl_svar2_channels ch;
    if ((rc = svar2_static(ctx, sh, &ch))) return rc;
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * batch);
    size_t i_sh = pk.add(shifts, sizeof(int32_t) * n_work);
    size_t i_rc = pk.add(to_rc, n_work);
    const Svar2Slots ss = svar2_add(pk, sh, batch, ploidy);
    const int64_t max_merged = ss.max_merged;
    if ((rc = pk.upload(ctx, 0))) return rc;
    svar2_resolve(pk, ss, &ch);
    void *oo_dev;
    if ((rc = scratch(ctx, 1, sizeof(int64_t) * (n_work + 1), &oo_dev))) return rc;
    ctx->host_out_offsets_dev = (int64_t *)oo_dev;
    if ((rc = gvl_dev_hap_plan_svar2(ctx, &t, &ch, pk.ptr<int32_t>(i_reg), pk.ptr<int32_t>(i_sh), batch, ploidy,
                                     pk.ptr<uint8_t>(i_rc), output_length, max_merged, ctx->host_out_offsets_dev, nullptr,
                                     ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out_offsets, oo_dev, sizeof(int64_t) * (n_work + 1), cudaMemcpyDeviceToHost, ctx->own_stream));
    if ((rc = gvl_ctx_check(ctx, ctx->own_stream))) return rc;
    if (ctx->total < 0) ctx->total = ctx->host_words[W_TOTAL];
    *total = ctx->total;
    return GVL_OK;
}

int gvl_hap_diffs_svar2(gvl_ctx *ctx, const int32_t *regions, int64_t batch, int64_t ploidy, const int32_t *vk_pos,
                        const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos, const int32_t *dense_key,
                        int64_t n_dense, const int32_t *dense_range, const uint8_t *dense_present,
                        const int64_t *dense_present_off, const int32_t *key_ilen, int64_t n_keys, int32_t *diffs) {
    if (!ctx || !vk_off || !dense_range || !dense_present_off || !key_ilen)
        return fail(GVL_ERR_ARG, "gvl_hap_diffs_svar2: NULL argument");
    if (batch < 0 || ploidy < 1) return fail(GVL_ERR_ARG, "gvl_hap_diffs_svar2: bad sizes");
    const int64_t n_work = batch * ploidy;
    if (n_work == 0) return GVL_OK;
    if (!regions || !diffs) return fail(GVL_ERR_ARG, "gvl_hap_diffs_svar2: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const void *d;
    gvl_sparse_tables t;
    memset(&t, 0, sizeof(t));
    if ((rc = static_dev(ctx, key_ilen, sizeof(int32_t) * n_keys, 11, &d))) return rc;
    t.ilens = (const int32_t *)d;
    t.v_starts = t.ilens;  // unused by the merged-list source
    t.n_variants = n_keys;
    const Svar2Host sh{vk_pos, vk_key, vk_off, dense_pos, dense_key, n_dense, dense_range, dense_present, dense_present_off};
    gvl_svar2_channels ch;
    if ((rc = svar2_static(ctx, sh, &ch))) return rc;
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * batch);
    const Svar2Slots ss = svar2_add(pk, sh, batch, ploidy);
    const int64_t max_merged = ss.max_merged;
    if ((rc = pk.upload(ctx, 0))) return rc;
    svar2_resolve(pk, ss, &ch);
    void *d_diffs;
    if ((rc = scratch(ctx, 1, sizeof(int32_t) * n_work, &d_diffs))) return rc;
    if ((rc = gvl_dev_hap_diffs_svar2(ctx, &t, &ch, pk.ptr<int32_t>(i_reg), batch, ploidy, max_merged, (int32_t *)d_diffs,
                                      ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(diffs, d_diffs, sizeof(int32_t) * n_work, cudaMemcpyDeviceToHost, ctx->own_stream));
    return gvl_ctx_check(ctx, ctx->own_stream);  // syncs; reports a merged-list overflow
}

int gvl_reconstruct_haplotypes_from_sparse(
    gvl_ctx *ctx, uint8_t *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const int64_t *geno_offsets, int64_t n_geno,
    const int32_t *geno_v_idxs, int64_t n_geno_v, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
    const uint8_t *alt_alleles, const int64_t *alt_offsets, const uint8_t *ref_, const int64_t *ref_offsets,
    int64_t n_contigs, uint8_t pad_char, const uint8_t *keep, const int64_t *keep_offsets, int32_t *annot_v_idxs,
    int32_t *annot_ref_pos) {
    int64_t total = 0;
    int rc = hap_begin(ctx, regions, shifts, geno_offset_idx, batch, ploidy, geno_offsets, n_geno, geno_v_idxs, n_geno_v,
                       v_starts, ilens, n_variants, alt_alleles, alt_offsets, ref_, ref_offsets, n_contigs, -2, keep,
                       keep_offsets, nullptr, const_cast<int64_t *>(out_offsets), &total);
    if (rc) return rc;
    const bool annot = annot_v_idxs && annot_ref_pos;
    return gvl_reconstruct_haplotypes_fused_finish(ctx, annot ? GVL_MODE_ANNOTATED : GVL_MODE_U8, pad_char, out,
                                                   annot_v_idxs, annot_ref_pos);
}

int gvl_reconstruct_haplotypes_fused_finish(gvl_ctx *ctx, int mode, uint8_t pad_char, uint8_t *out, int32_t *annot_v,
                                            int32_t *annot_pos) {
    if (!ctx) return fail(GVL_ERR_ARG, "gvl_reconstruct_haplotypes_fused_finish: ctx is NULL");
    if (!ctx->plan_valid) return fail(GVL_ERR_STATE, "gvl_reconstruct_haplotypes_fused_finish: begin was not called");
    GVL_CUDA(cudaSetDevice(ctx->device));
    const int64_t total = ctx->total;
    if (total == 0) return GVL_OK;
    if (!out) return fail(GVL_ERR_ARG, "gvl_reconstruct_haplotypes_fused_finish: out is NULL");
    const bool oh = (mode == GVL_MODE_ONEHOT || mode == GVL_MODE_ONEHOT_CF);
    const int64_t out_bytes = oh ? total * 4 : total;
    int rc;
    void *d_out, *d_av = nullptr, *d_ap = nullptr;
    if ((rc = scratch(ctx, 2, out_bytes, &d_out))) return rc;
    if (mode == GVL_MODE_ANNOTATED) {
        if (!annot_v || !annot_pos) return fail(GVL_ERR_ARG, "annotated mode needs annot_v and annot_pos");
        if ((rc = scratch(ctx, 3, total * 4, &d_av))) return rc;
        if ((rc = scratch(ctx, 4, total * 4, &d_ap))) return rc;
    }
    if ((rc = gvl_dev_hap_exec(ctx, &ctx->host_tab, mode, pad_char, (uint8_t *)d_out, (int32_t *)d_av, (int32_t *)d_ap,
                               ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)out_bytes, cudaMemcpyDeviceToHost, ctx->own_stream));
    if (mode == GVL_MODE_ANNOTATED) {
        GVL_CUDA(cudaMemcpyAsync(annot_v, d_av, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->own_stream));
        GVL_CUDA(cudaMemcpyAsync(annot_pos, d_ap, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->own_stream));
    }
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    return GVL_OK;
}

int gvl_reconstruct_haplotypes_spliced_fused(
    gvl_ctx *ctx, uint8_t *out, int32_t *annot_v, int32_t *annot_pos, const int32_t *permuted_regions,
    const int32_t *flat_shifts, const int64_t *flat_geno_offset_idx, int64_t n_perm, const int64_t *out_offsets,
    const int64_t *geno_offsets, int64_t n_geno, const int32_t *geno_v_idxs, int64_t n_geno_v, const int32_t *v_starts,
    const int32_t *ilens, int64_t n_variants, const uint8_t *alt_alleles, const int64_t *alt_offsets, const uint8_t *ref_,
    const int64_t *ref_offsets, int64_t n_contigs, uint8_t pad_char, const uint8_t *keep, const int64_t *keep_offsets,
    const uint8_t *to_rc) {
    if ((annot_v == nullptr) != (annot_pos == nullptr))
        return fail(GVL_ERR_ARG, "gvl_reconstruct_haplotypes_spliced_fused: annot_v and annot_pos go together");
    int64_t total = 0;
    int rc = hap_begin(ctx, permuted_regions, flat_shifts, flat_geno_offset_idx, n_perm, 1, geno_offsets, n_geno,
                       geno_v_idxs, n_geno_v, v_starts, ilens, n_variants, alt_alleles, alt_offsets, ref_, ref_offsets,
                       n_contigs, -2, keep, keep_offsets, to_rc, const_cast<int64_t *>(out_offsets), &total);
    if (rc) return rc;
    return gvl_reconstruct_haplotypes_fused_finish(ctx, annot_v ? GVL_MODE_ANNOTATED : GVL_MODE_U8, pad_char, out, annot_v,
                                                   annot_pos);
}

int gvl_choose_exonic_variants(gvl_ctx *ctx, const int32_t *starts, const int32_t *ends, const int64_t *geno_offset_idx,
                               int64_t n_queries, int64_t ploidy, const int32_t *geno_v_idxs, int64_t n_geno_v,
                               const int64_t *geno_offsets, int64_t n_geno, const int32_t *v_starts, const int32_t *ilens,
                               int64_t n_variants, uint8_t *keep, int64_t keep_cap, int64_t *keep_offsets) {
    if (!ctx || !geno_offsets || !keep_offsets) return fail(GVL_ERR_ARG, "gvl_choose_exonic_variants: NULL argument");
    if (n_queries < 0 || ploidy < 1 || keep_cap < 0) return fail(GVL_ERR_ARG, "gvl_choose_exonic_variants: bad sizes");
    const int64_t n_work = n_queries * ploidy;
    if (n_work && (!starts || !ends || !geno_offset_idx || !geno_v_idxs || !v_starts || !ilens))
        return fail(GVL_ERR_ARG, "gvl_choose_exonic_variants: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    gvl_sparse_tables t;
    if ((rc = resolve_tables(ctx, geno_offsets, n_geno, geno_v_idxs, n_geno_v, v_starts, ilens, n_variants, nullptr,
                             nullptr, nullptr, nullptr, 0, &t)))
        return rc;
    Packer pk;
    size_t i_st = pk.add(starts, sizeof(int32_t) * n_queries);
    size_t i_en = pk.add(ends, sizeof(int32_t) * n_queries);
    size_t i_goi = pk.add(geno_offset_idx, sizeof(int64_t) * n_work);
    if ((rc = pk.upload(ctx, 0))) return rc;
    void *d_ko, *d_keep = nullptr;
    if ((rc = scratch(ctx, 1, sizeof(int64_t) * (n_work + 1), &d_ko))) return rc;
    if (keep && keep_cap && (rc = scratch(ctx, 2, keep_cap, &d_keep))) return rc;
    if ((rc = gvl_dev_choose_exonic_variants(ctx, &t, pk.ptr<int32_t>(i_st), pk.ptr<int32_t>(i_en), pk.ptr<int64_t>(i_goi),
                                             n_queries, ploidy, (uint8_t *)d_keep, d_keep ? keep_cap : 0, (int64_t *)d_ko,
                                             ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(keep_offsets, d_ko, sizeof(int64_t) * (n_work + 1), cudaMemcpyDeviceToHost, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    const int64_t n = keep_offsets[n_work];
    if (n > (d_keep ? keep_cap : 0))
        return fail(GVL_ERR_CAPACITY, "gvl_choose_exonic_variants: keep holds %lld entries, %lld needed", (long long)keep_cap,
                    (long long)n);
    if (n) {
        GVL_CUDA(cudaMemcpyAsync(keep, d_keep, (size_t)n, cudaMemcpyDeviceToHost, ctx->own_stream));
        GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    }
    return GVL_OK;
}

int gvl_get_reference(gvl_ctx *ctx, const int32_t *regions, const int64_t *out_offsets, int64_t n_regions,
                      const uint8_t *reference, const int64_t *ref_offsets, int64_t n_contigs, uint8_t pad_char,
                      const uint8_t *to_rc, int mode, uint8_t *out) {
    if (!ctx || !out_offsets || !reference || !ref_offsets) return fail(GVL_ERR_ARG, "gvl_get_reference: NULL argument");
    if (n_regions < 0 || n_contigs < 0) return fail(GVL_ERR_ARG, "gvl_get_reference: bad sizes");
    if (n_regions && !regions) return fail(GVL_ERR_ARG, "gvl_get_reference: regions is NULL");
    if (mode != GVL_MODE_U8 && mode != GVL_MODE_ONEHOT) return fail(GVL_ERR_ARG, "gvl_get_reference: mode must be u8 or one-hot");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const void *d;
    gvl_sparse_tables t;
    memset(&t, 0, sizeof(t));
    if ((rc = static_dev(ctx, ref_offsets, sizeof(int64_t) * (n_contigs + 1), 14, &d))) return rc;
    t.ref_offsets = (const int64_t *)d;
    if ((rc = static_dev(ctx, reference, ref_offsets[n_contigs], 15, &d))) return rc;
    t.ref = (const uint8_t *)d;
    t.n_contigs = n_contigs;
    if ((rc = packed_ref(ctx, reference, t.ref, ref_offsets[n_contigs], &t.ref_packed))) return rc;
    const int64_t total = out_offsets[n_regions];
    if (total == 0) return GVL_OK;
    if (!out) return fail(GVL_ERR_ARG, "gvl_get_reference: out is NULL");
    // equal rows take the fixed-length plan (no sync between plan and execute, packed one-hot kernel eligible)
    int64_t row_length = out_offsets[1] - out_offsets[0];
    for (int64_t i = 1; i < n_regions && row_length >= 0; i++)
        if (out_offsets[i + 1] - out_offsets[i] != row_length) row_length = -1;
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * n_regions);
    size_t i_oo = pk.add(out_offsets, sizeof(int64_t) * (n_regions + 1));
    size_t i_rc = pk.add(to_rc, n_regions);
    if ((rc = pk.upload(ctx, 0))) return rc;
    const int64_t out_bytes = mode == GVL_MODE_ONEHOT ? total * 4 : total;
    void *d_out;
    if ((rc = scratch(ctx, 2, out_bytes, &d_out))) return rc;
    if ((rc = gvl_dev_get_reference(ctx, &t, pk.ptr<int32_t>(i_reg), const_cast<int64_t *>(pk.ptr<int64_t>(i_oo)), n_regions,
                                    row_length, pk.ptr<uint8_t>(i_rc), mode, pad_char, (uint8_t *)d_out, ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)out_bytes, cudaMemcpyDeviceToHost, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    return GVL_OK;
}

int gvl_ragged_to_padded(gvl_ctx *ctx, const void *data, const int64_t *offsets, int64_t n_rows, void *out,
                         int64_t itemsize, int64_t out_len) {
    if (!ctx) return fail(GVL_ERR_ARG, "gvl_ragged_to_padded: ctx is NULL");
    if (n_rows < 0 || itemsize < 1 || out_len < 0) return fail(GVL_ERR_ARG, "gvl_ragged_to_padded: bad sizes");
    if (n_rows == 0 || out_len == 0) return GVL_OK;
    if (!data || !offsets || !out) return fail(GVL_ERR_ARG, "gvl_ragged_to_padded: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t lo = offsets[0], hi = offsets[n_rows];  // only [lo, hi) of `data` is read
    const int64_t out_bytes = n_rows * out_len * itemsize;
    void *d_data, *d_off, *d_out;
    if ((rc = scratch(ctx, 0, (hi - lo) * itemsize + 16, &d_data))) return rc;
    if ((rc = scratch(ctx, 1, sizeof(int64_t) * (n_rows + 1), &d_off))) return rc;
    if ((rc = scratch(ctx, 2, out_bytes, &d_out))) return rc;
    if (hi > lo)
        GVL_CUDA(cudaMemcpyAsync(d_data, (const char *)data + lo * itemsize, (size_t)((hi - lo) * itemsize),
                                 cudaMemcpyHostToDevice, ctx->own_stream));
    GVL_CUDA(cudaMemcpyAsync(d_off, offsets, sizeof(int64_t) * (n_rows + 1), cudaMemcpyHostToDevice, ctx->own_stream));
    GVL_CUDA(cudaMemcpyAsync(d_out, out, (size_t)out_bytes, cudaMemcpyHostToDevice, ctx->own_stream));  // the pre-fill
    // the device copy of `data` starts at item lo: shift the base pointer instead of rewriting the offsets
    if ((rc = gvl_dev_ragged_to_padded(ctx, (const char *)d_data - lo * itemsize, (const int64_t *)d_off, n_rows, d_out,
                                       itemsize, out_len, ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)out_bytes, cudaMemcpyDeviceToHost, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    return GVL_OK;
}

int gvl_get_diffs_sparse(gvl_ctx *ctx, const int64_t *geno_offset_idx, int64_t n_queries, int64_t ploidy,
                         const int32_t *geno_v_idxs, int64_t n_geno_v, const int64_t *geno_offsets, int64_t n_geno,
                         const int32_t *ilens, int64_t n_variants, const uint8_t *keep, const int64_t *keep_offsets,
                         const int32_t *q_starts, const int32_t *q_ends, const int32_t *v_starts, int32_t *diffs) {
    if (!ctx || !geno_offset_idx || !geno_v_idxs || !geno_offsets || !ilens || !diffs)
        return fail(GVL_ERR_ARG, "gvl_get_diffs_sparse: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t n_work = n_queries * ploidy;
    gvl_sparse_tables t;
    if ((rc = resolve_tables(ctx, geno_offsets, n_geno, geno_v_idxs, n_geno_v, v_starts ? v_starts : ilens, ilens,
                             n_variants, nullptr, nullptr, nullptr, nullptr, 0, &t)))
        return rc;
    Packer pk;
    size_t i_goi = pk.add(geno_offset_idx, sizeof(int64_t) * n_work);
    size_t i_ko = pk.add(keep_offsets, sizeof(int64_t) * (n_work + 1));
    size_t i_kp = pk.add(keep, keep_offsets ? keep_offsets[n_work] : 0);
    size_t i_qs = pk.add(q_starts, sizeof(int32_t) * n_queries);
    size_t i_qe = pk.add(q_ends, sizeof(int32_t) * n_queries);
    if ((rc = pk.upload(ctx, 0))) return rc;
    void *d_diffs;
    if ((rc = scratch(ctx, 1, sizeof(int32_t) * (n_work + 1), &d_diffs))) return rc;
    if ((rc = gvl_dev_get_diffs_sparse(ctx, &t, pk.ptr<int64_t>(i_goi), n_queries, ploidy,
                                       keep && keep_offsets ? pk.ptr<uint8_t>(i_kp) : nullptr,
                                       keep && keep_offsets ? pk.ptr<int64_t>(i_ko) : nullptr, pk.ptr<int32_t>(i_qs),
                                       pk.ptr<int32_t>(i_qe), v_starts != nullptr, (int32_t *)d_diffs, ctx->own_stream)))
        return rc;
    if (n_work) GVL_CUDA(cudaMemcpyAsync(diffs, d_diffs, sizeof(int32_t) * n_work, cudaMemcpyDeviceToHost, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    return GVL_OK;
}

}  // extern "C"

// ---- tracks ----------------------------------------------------------------------------------
extern "C" {

static int resolve_intervals(gvl_ctx *ctx, const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
                             int64_t n_itv, const int64_t *itv_offsets, int64_t n_slots, gvl_intervals *iv) {
    int rc;
    const void *d;
    if ((rc = static_dev(ctx, itv_starts, sizeof(int32_t) * n_itv, 16, &d))) return rc;
    iv->itv_starts = (const int32_t *)d;
    if ((rc = static_dev(ctx, itv_ends, sizeof(int32_t) * n_itv, 17, &d))) return rc;
    iv->itv_ends = (const int32_t *)d;
    if ((rc = static_dev(ctx, itv_values, sizeof(float) * n_itv, 18, &d))) return rc;
    iv->itv_values = (const float *)d;
    if ((rc = static_dev(ctx, itv_offsets, sizeof(int64_t) * (n_slots + 1), 19, &d))) return rc;
    iv->itv_offsets = (const int64_t *)d;
    iv->n_slots = n_slots;
    return GVL_OK;
}

// Intervals of ONE call: the caller's arrays when none of the slots the call touches overlaps (the normal case:
// one scan of those slots, O(the call's own work)); otherwise a private, flattened copy of the touched slots -- one
// slot per query, `flat_idx` = 0..n_queries-1 replaces the caller's offset_idxs (see the flatten helpers above).
struct CallIntervals {
    gvl_intervals iv;
    std::vector<int32_t> s, e;
    std::vector<float> v;
    std::vector<int64_t> off, flat_idx;
    bool flattened = false;
};

static int resolve_call_intervals(gvl_ctx *ctx, const int64_t *offset_idxs, int64_t n_queries, const int32_t *itv_starts,
                                  const int32_t *itv_ends, const float *itv_values, int64_t n_itv,
                                  const int64_t *itv_offsets, int64_t n_slots, CallIntervals *ci) {
    bool any = false;
    for (int64_t q = 0; q < n_queries && !any; q++) {
        const int64_t k = offset_idxs[q];
        if (k < 0 || k >= n_slots) return fail(GVL_ERR_ARG, "interval slot %lld of %lld", (long long)k, (long long)n_slots);
        any = slot_overlaps(itv_starts + itv_offsets[k], itv_ends + itv_offsets[k], itv_offsets[k + 1] - itv_offsets[k]);
    }
    if (!any) return resolve_intervals(ctx, itv_starts, itv_ends, itv_values, n_itv, itv_offsets, n_slots, &ci->iv);
    ci->flattened = true;
    ci->off.assign(1, 0);
    for (int64_t q = 0; q < n_queries; q++) {
        const int64_t k = offset_idxs[q], lo = itv_offsets[k];
        flatten_slot(itv_starts + lo, itv_ends + lo, itv_values + lo, itv_offsets[k + 1] - lo, ci->s, ci->e, ci->v);
        ci->off.push_back((int64_t)ci->s.size());
        ci->flat_idx.push_back(q);
    }
    return resolve_intervals(ctx, ci->s.data(), ci->e.data(), ci->v.data(), (int64_t)ci->s.size(), ci->off.data(), n_queries,
                             &ci->iv);
}

int gvl_intervals_and_realign_track_fused(
    gvl_ctx *ctx, float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const int32_t *geno_v_idxs, int64_t n_geno_v,
    const int64_t *geno_offsets, int64_t n_geno, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
    const int64_t *offset_idxs, const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
    int64_t n_itv, const int64_t *itv_offsets, int64_t n_slots, const int64_t *track_offsets, const double *params,
    int64_t strategy_id, uint64_t base_seed, const uint8_t *keep, const int64_t *keep_offsets, const uint8_t *to_rc) {
    if (!ctx || !out_offsets || !regions || !shifts || !geno_offset_idx || !geno_v_idxs || !geno_offsets || !v_starts ||
        !ilens || !offset_idxs || !itv_offsets || !track_offsets || !params)
        return fail(GVL_ERR_ARG, "gvl_intervals_and_realign_track_fused: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t n_work = batch * ploidy;
    const int64_t total = out_offsets[n_work];
    if (n_work == 0 || total == 0) return GVL_OK;
    if (!out) return fail(GVL_ERR_ARG, "gvl_intervals_and_realign_track_fused: out is NULL");
    gvl_sparse_tables t;
    if ((rc = resolve_tables(ctx, geno_offsets, n_geno, geno_v_idxs, n_geno_v, v_starts, ilens, n_variants, nullptr,
                             nullptr, nullptr, nullptr, 0, &t)))
        return rc;
    CallIntervals ci;
    if ((rc = resolve_call_intervals(ctx, offset_idxs, batch, itv_starts, itv_ends, itv_values, n_itv, itv_offsets, n_slots, &ci)))
        return rc;
    const gvl_intervals &iv = ci.iv;
    if (ci.flattened) offset_idxs = ci.flat_idx.data();
    std::vector<int32_t> tl((size_t)batch);
    for (int64_t q = 0; q < batch; q++) tl[q] = (int32_t)(track_offsets[q + 1] - track_offsets[q]);
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * batch);
    size_t i_sh = pk.add(shifts, sizeof(int32_t) * n_work);
    size_t i_goi = pk.add(geno_offset_idx, sizeof(int64_t) * n_work);
    size_t i_ko = pk.add(keep_offsets, sizeof(int64_t) * (n_work + 1));
    size_t i_kp = pk.add(keep, keep_offsets ? keep_offsets[n_work] : 0);
    size_t i_rc = pk.add(to_rc, n_work);
    size_t i_oi = pk.add(offset_idxs, sizeof(int64_t) * batch);
    size_t i_tl = pk.add(tl.data(), sizeof(int32_t) * batch);
    size_t i_oo = pk.add(out_offsets, sizeof(int64_t) * (n_work + 1));
    if ((rc = pk.upload(ctx, 0))) return rc;
    void *d_out;
    if ((rc = scratch(ctx, 2, total * 4, &d_out))) return rc;
    const int32_t strat = (int32_t)strategy_id;
    const int64_t max_rec = sum_variants(geno_offsets, n_geno, geno_offset_idx, n_work);
    if ((rc = gvl_dev_realign_tracks(ctx, &t, nullptr, pk.ptr<int32_t>(i_reg), pk.ptr<int32_t>(i_sh), pk.ptr<int64_t>(i_goi),
                                     batch, ploidy, keep && keep_offsets ? pk.ptr<uint8_t>(i_kp) : nullptr,
                                     keep && keep_offsets ? pk.ptr<int64_t>(i_ko) : nullptr, pk.ptr<uint8_t>(i_rc), 1, &iv,
                                     pk.ptr<int64_t>(i_oi), pk.ptr<int32_t>(i_tl), pk.ptr<int64_t>(i_oo), total, &strat,
                                     params, base_seed, nullptr, 0, nullptr, max_rec, GVL_TRACK_LAYOUT_TBP, nullptr, nullptr,
                                     d_out, GVL_TRACK_F32, ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->own_stream));
    return gvl_ctx_check(ctx, ctx->own_stream);
}

int gvl_shift_and_realign_tracks_sparse(
    gvl_ctx *ctx, float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts,
    const int64_t *geno_offset_idx, int64_t batch, int64_t ploidy, const int32_t *geno_v_idxs, int64_t n_geno_v,
    const int64_t *geno_offsets, int64_t n_geno, const int32_t *v_starts, const int32_t *ilens, int64_t n_variants,
    const float *tracks, const int64_t *track_offsets, const double *params, const uint8_t *keep,
    const int64_t *keep_offsets, int64_t strategy_id, uint64_t base_seed) {
    if (!ctx || !out_offsets || !regions || !shifts || !geno_offset_idx || !geno_v_idxs || !geno_offsets || !v_starts ||
        !ilens || !track_offsets || !params)
        return fail(GVL_ERR_ARG, "gvl_shift_and_realign_tracks_sparse: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t n_work = batch * ploidy;
    const int64_t total = out_offsets[n_work];
    if (n_work == 0 || total == 0) return GVL_OK;
    if (!out || !tracks) return fail(GVL_ERR_ARG, "gvl_shift_and_realign_tracks_sparse: NULL buffer");
    gvl_sparse_tables t;
    if ((rc = resolve_tables(ctx, geno_offsets, n_geno, geno_v_idxs, n_geno_v, v_starts, ilens, n_variants, nullptr,
                             nullptr, nullptr, nullptr, 0, &t)))
        return rc;
    const void *d_tracks;
    if ((rc = static_dev(ctx, tracks, sizeof(float) * track_offsets[batch], 16, &d_tracks))) return rc;
    std::vector<int32_t> tl((size_t)batch);
    for (int64_t q = 0; q < batch; q++) tl[q] = (int32_t)(track_offsets[q + 1] - track_offsets[q]);
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * batch);
    size_t i_sh = pk.add(shifts, sizeof(int32_t) * n_work);
    size_t i_goi = pk.add(geno_offset_idx, sizeof(int64_t) * n_work);
    size_t i_ko = pk.add(keep_offsets, sizeof(int64_t) * (n_work + 1));
    size_t i_kp = pk.add(keep, keep_offsets ? keep_offsets[n_work] : 0);
    size_t i_to = pk.add(track_offsets, sizeof(int64_t) * (batch + 1));
    size_t i_tl = pk.add(tl.data(), sizeof(int32_t) * batch);
    size_t i_oo = pk.add(out_offsets, sizeof(int64_t) * (n_work + 1));
    if ((rc = pk.upload(ctx, 0))) return rc;
    void *d_out;
    if ((rc = scratch(ctx, 2, total * 4, &d_out))) return rc;
    const int64_t max_rec = sum_variants(geno_offsets, n_geno, geno_offset_idx, n_work);
    if ((rc = gvl_dev_shift_and_realign_tracks(
             ctx, &t, nullptr, pk.ptr<int32_t>(i_reg), pk.ptr<int32_t>(i_sh), pk.ptr<int64_t>(i_goi), batch, ploidy,
             keep && keep_offsets ? pk.ptr<uint8_t>(i_kp) : nullptr, keep && keep_offsets ? pk.ptr<int64_t>(i_ko) : nullptr,
             nullptr, (const float *)d_tracks, pk.ptr<int64_t>(i_to), pk.ptr<int32_t>(i_tl), pk.ptr<int64_t>(i_oo), total,
             (int32_t)strategy_id, params[0], base_seed, nullptr, max_rec, (float *)d_out, ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->own_stream));
    return gvl_ctx_check(ctx, ctx->own_stream);
}

int gvl_shift_and_realign_tracks_from_svar2(
    gvl_ctx *ctx, float *out, const int64_t *out_offsets, const int32_t *regions, const int32_t *shifts, int64_t batch,
    int64_t ploidy, const int32_t *vk_pos, const int32_t *vk_key, const int64_t *vk_off, const int32_t *dense_pos,
    const int32_t *dense_key, int64_t n_dense, const int32_t *dense_range, const uint8_t *dense_present,
    const int64_t *dense_present_off, const int32_t *key_ilen, int64_t n_keys, const float *tracks,
    const int64_t *track_offsets, const double *params, int64_t strategy_id, uint64_t base_seed,
    const int64_t *query_seed) {
    if (!ctx || !out_offsets || !regions || !shifts || !vk_off || !dense_range || !dense_present_off || !key_ilen ||
        !track_offsets || !params)
        return fail(GVL_ERR_ARG, "gvl_shift_and_realign_tracks_from_svar2: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t n_work = batch * ploidy;
    const int64_t total = out_offsets[n_work];
    if (n_work == 0 || total == 0) return GVL_OK;
    if (!out || !tracks) return fail(GVL_ERR_ARG, "gvl_shift_and_realign_tracks_from_svar2: NULL buffer");
    const void *d;
    gvl_sparse_tables t;
    memset(&t, 0, sizeof(t));
    if ((rc = static_dev(ctx, key_ilen, sizeof(int32_t) * n_keys, 11, &d))) return rc;
    t.ilens = (const int32_t *)d;
    t.v_starts = t.ilens;  // unused by the merged-list source
    t.n_variants = n_keys;
    const Svar2Host sh{vk_pos, vk_key, vk_off, dense_pos, dense_key, n_dense, dense_range, dense_present, dense_present_off};
    gvl_svar2_channels ch;
    if ((rc = svar2_static(ctx, sh, &ch))) return rc;
    const void *d_tracks;
    if ((rc = static_dev(ctx, tracks, sizeof(float) * track_offsets[batch], 18, &d_tracks))) return rc;
    std::vector<int32_t> tl((size_t)batch);
    for (int64_t q = 0; q < batch; q++) tl[q] = (int32_t)(track_offsets[q + 1] - track_offsets[q]);
    Packer pk;
    size_t i_reg = pk.add(regions, sizeof(int32_t) * 3 * batch);
    size_t i_sh = pk.add(shifts, sizeof(int32_t) * n_work);
    const Svar2Slots ss = svar2_add(pk, sh, batch, ploidy);
    const int64_t max_merged = ss.max_merged;
    size_t i_to = pk.add(track_offsets, sizeof(int64_t) * (batch + 1));
    size_t i_tl = pk.add(tl.data(), sizeof(int32_t) * batch);
    size_t i_oo = pk.add(out_offsets, sizeof(int64_t) * (n_work + 1));
    size_t i_qs = pk.add(query_seed, sizeof(int64_t) * batch);
    if ((rc = pk.upload(ctx, 0))) return rc;
    svar2_resolve(pk, ss, &ch);
    void *d_out;
    if ((rc = scratch(ctx, 2, total * 4, &d_out))) return rc;
    if ((rc = gvl_dev_shift_and_realign_tracks(
             ctx, &t, &ch, pk.ptr<int32_t>(i_reg), pk.ptr<int32_t>(i_sh), nullptr, batch, ploidy, nullptr, nullptr, nullptr,
             (const float *)d_tracks, pk.ptr<int64_t>(i_to), pk.ptr<int32_t>(i_tl), pk.ptr<int64_t>(i_oo), total,
             (int32_t)strategy_id, params[0], base_seed, query_seed ? pk.ptr<int64_t>(i_qs) : nullptr, max_merged, (float *)d_out, ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->own_stream));
    return gvl_ctx_check(ctx, ctx->own_stream);
}

int gvl_intervals_to_tracks(gvl_ctx *ctx, const int64_t *offset_idxs, const int32_t *starts, int64_t n_queries,
                            const int32_t *itv_starts, const int32_t *itv_ends, const float *itv_values,
                            int64_t n_itv, const int64_t *itv_offsets, int64_t n_slots, float *out,
                            const int64_t *out_offsets) {
    if (!ctx || !offset_idxs || !starts || !itv_offsets || !out_offsets)
        return fail(GVL_ERR_ARG, "gvl_intervals_to_tracks: NULL argument");
    GVL_CUDA(cudaSetDevice(ctx->device));
    int rc;
    const int64_t total = out_offsets[n_queries];
    if (n_queries == 0 || total == 0) return GVL_OK;
    if (!out) return fail(GVL_ERR_ARG, "gvl_intervals_to_tracks: out is NULL");
    CallIntervals ci;
    if ((rc = resolve_call_intervals(ctx, offset_idxs, n_queries, itv_starts, itv_ends, itv_values, n_itv, itv_offsets, n_slots,
                                     &ci)))
        return rc;
    const gvl_intervals &iv = ci.iv;
    if (ci.flattened) offset_idxs = ci.flat_idx.data();
    Packer pk;
    size_t i_oi = pk.add(offset_idxs, sizeof(int64_t) * n_queries);
    size_t i_st = pk.add(starts, sizeof(int32_t) * n_queries);
    size_t i_oo = pk.add(out_offsets, sizeof(int64_t) * (n_queries + 1));
    if ((rc = pk.upload(ctx, 0))) return rc;
    void *d_out;
    if ((rc = scratch(ctx, 2, total * 4, &d_out))) return rc;
    if ((rc = gvl_dev_paint_tracks(ctx, 1, &iv, pk.ptr<int64_t>(i_oi), pk.ptr<int32_t>(i_st), n_queries, pk.ptr<int64_t>(i_oo),
                                   total, nullptr, GVL_TRACK_LAYOUT_TBP, nullptr, nullptr, d_out, GVL_TRACK_F32, ctx->own_stream)))
        return rc;
    GVL_CUDA(cudaMemcpyAsync(out, d_out, (size_t)total * 4, cudaMemcpyDeviceToHost, ctx->own_stream));
    GVL_CUDA(cudaStreamSynchronize(ctx->own_stream));
    return GVL_OK;
}

}  // extern "C"

#include "gvl_host_variants.cuh"
