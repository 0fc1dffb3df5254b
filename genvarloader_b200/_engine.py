"""Device-resident engine: static tables in HBM as torch tensors + thin calls into the gvl_dev_*
layer of include/gvl_b200.h on torch's current CUDA stream.

torch is plumbing here (device memory, streams); all compute is in the CUDA library.
"""
from __future__ import annotations

import ctypes as C
import warnings

import numpy as np
import torch

from . import _ffi
from ._ffi import (MODE_ANNOTATED, MODE_ONEHOT, MODE_ONEHOT_CF, MODE_U8, TRACK_BF16, TRACK_F16, TRACK_F32, DatasetView, Intervals,
                   SparseTables, Svar2Channels, c_i32, c_i64, c_u8, c_u64, c_vp, check, lib, ptr)

_SVAR2_VARIANTS = ("`variants` output is built for the SVAR1 genotype CSR; the svar2 source decodes variants through its "
                   "store (decode_variants_from_svar2_readbound, src/ffi/mod.rs:1692)")
MODES = {"haplotypes": MODE_U8, "u8": MODE_U8, "onehot": MODE_ONEHOT, "onehot_cf": MODE_ONEHOT_CF,
         "annotated": MODE_ANNOTATED}
# element types of track outputs (GVL_TRACK_*): values are computed in float32 and narrowed at the kernel's store
TRACK_DTYPES = {torch.float32: TRACK_F32, torch.bfloat16: TRACK_BF16, torch.float16: TRACK_F16}


def track_dtype_code(dtype) -> int:
    """GVL_TRACK_* code of a torch dtype; ValueError for anything but float32, bfloat16 and float16."""
    code = TRACK_DTYPES.get(dtype) if isinstance(dtype, torch.dtype) else None
    if code is None:
        raise ValueError(f"track dtype must be torch.float32, torch.bfloat16 or torch.float16, got {dtype!r}")
    return code


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)  # ~1 us; torch.cuda.current_stream() costs ~15 us
if _raw_stream is None:  # pragma: no cover  (older torch)
    def _raw_stream(device_index: int) -> int:
        return torch.cuda.current_stream(device_index).cuda_stream


def _stream() -> c_vp:
    """torch's current CUDA stream of the current device as a raw handle."""
    return c_vp(_raw_stream(torch._C._cuda_getDevice()))


def _dev(a, dtype, device, pad: int = 0) -> torch.Tensor:
    """Upload a host array (numpy / memmap) as a device tensor, optionally with `pad` spare elements
    (the reference buffer must be readable up to the next multiple of 16 bytes)."""
    a = np.ascontiguousarray(a, dtype)
    t = torch.empty(a.size + pad, dtype=torch.from_numpy(np.empty(0, dtype)).dtype, device=device)
    if pad:
        t[a.size:].zero_()
    if a.size:
        with warnings.catch_warnings():  # read-only memmaps (datasets opened from disk) are only read here
            warnings.filterwarnings("ignore", message="The given NumPy array is not writable")
            t[: a.size].copy_(torch.from_numpy(a.reshape(-1)), non_blocking=False)
    return t


class Engine:
    """Static tables of one dataset replica on one GPU (SVAR1-style: reference + variant table +
    sparse genotype CSR [+ interval tracks]) -- the device-side counterpart of `_HapsFfiStatic`
    (python/genvarloader/_dataset/_haps.py:233-247) plus the memmapped genotype/interval arrays."""

    def __init__(self, device, reference, ref_offsets, v_starts, ilens, alt_alleles, alt_offsets, geno_v_idxs,
                 geno_offsets, pad_char: int = ord("N"), pack_reference: bool = True):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("genvarloader_b200 needs a CUDA device; there is no CPU path")
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.device = torch.device("cuda", idx)
        self.ctx = _ffi.Ctx(idx)
        self.pad_char = int(pad_char)
        go = np.asarray(geno_offsets)
        if go.ndim == 1:
            go = np.stack([go[:-1], go[1:]])
        # one extra, EMPTY slot at the end: rows that must carry no variants ("reference" sequences) point at it
        go = np.concatenate([np.ascontiguousarray(go, np.int64), np.zeros((2, 1), np.int64)], 1)
        self.empty_slot = go.shape[1] - 1
        self.geno_offsets_host = np.ascontiguousarray(go, np.int64)  # O(batch) capacity sums stay on the host
        # longest variant list of any (region, sample, ploid) slot: workspace capacity of graph-replayed batches
        self.max_slot_len = int(np.maximum(go[1] - go[0], 0).max()) if go.shape[1] else 0
        self.typ_slot_len = 0  # (the CSR bound is tight enough; svar2 sources set a hint, set_svar2)
        self._views: dict = {}
        with torch.cuda.device(self.device):
            self.ref = _dev(reference, np.uint8, self.device, pad=32)
            self.ref_offsets = _dev(ref_offsets, np.int64, self.device)
            self.v_starts = _dev(v_starts, np.int32, self.device)
            self.ilens = _dev(ilens, np.int32, self.device)
            self.alt_alleles = _dev(alt_alleles, np.uint8, self.device, pad=16)
            self.alt_offsets = _dev(alt_offsets, np.int64, self.device)
            self.geno_v_idxs = _dev(geno_v_idxs, np.int32, self.device, pad=4)
            self.geno_starts = _dev(self.geno_offsets_host[0], np.int64, self.device)
            self.geno_stops = _dev(self.geno_offsets_host[1], np.int64, self.device)
        self.n_contigs = int(np.asarray(ref_offsets).size - 1)
        # 4-bit-per-base copy of the reference for the one-hot execute kernel (gvl_dev_pack_reference)
        self.ref_packed = self.alt_packed = None
        if pack_reference:
            def pack(t: torch.Tensor, n_bases: int) -> torch.Tensor:
                n_words = int(lib.gvl_packed_reference_words(c_i64(n_bases)))
                with torch.cuda.device(self.device):
                    out = torch.empty(n_words, dtype=torch.int32, device=self.device)
                    check(lib.gvl_dev_pack_reference(self.ctx.handle, ptr(t), c_i64(n_bases), ptr(out), _stream()))
                return out

            self.ref_packed = pack(self.ref, int(np.asarray(reference).size))
            self.alt_packed = pack(self.alt_alleles, int(np.asarray(alt_alleles).size))
        self.tab = SparseTables(
            ptr(self.ref), ptr(self.ref_offsets), self.n_contigs, ptr(self.v_starts), ptr(self.ilens),
            ptr(self.alt_alleles), ptr(self.alt_offsets), int(self.v_starts.numel()), ptr(self.geno_v_idxs),
            ptr(self.geno_starts), ptr(self.geno_stops), int(self.geno_starts.numel()), ptr(self.ref_packed),
            ptr(self.alt_packed))
        self.tracks: dict[str, tuple] = {}
        self.svar2 = None  # resident svar2 two-channel source (set_svar2)
        self.ref_alleles = None  # (bytes, offsets) of the REF allele strings (set_variant_fields)
        self.var_info: dict[str, torch.Tensor] = {}   # 4-byte info columns on the device (output fields)
        self.var_info_host: dict[str, np.ndarray] = {}  # every info column (the AF filter is evaluated per variant on the host)
        self._af_tables: dict = {}
        self._consts: dict = {}
        self.dosages = None
        self._n_work = 0
        self._fixed = -1

    # ------------------------------------------------------------------ svar2 source
    @classmethod
    def from_svar2(cls, device, reference, ref_offsets, sv: dict, n_slots: int, pad_char: int = ord("N")) -> "Engine":
        """Engine over a RESIDENT svar2 two-channel source (`synth.to_svar2_dataset` layout; the reference keeps the same
        information as range tables into the .svar2 store, docs/source/format.md:88-96, `_svar2_haps.py:1269-1313`).
        The variant table of the engine is the DECODED key table (ilen, ALT bytes); the SVAR1 genotype CSR is empty."""
        eng = cls(device, reference, ref_offsets, np.zeros(sv["key_ilen"].size, np.int32), sv["key_ilen"], sv["key_alt"],
                  sv["key_alt_off"], np.zeros(0, np.int32), np.zeros(n_slots + 1, np.int64), pad_char=pad_char)
        eng.set_svar2(sv)
        return eng

    def set_svar2(self, sv: dict) -> None:
        d = self.device
        with torch.cuda.device(d):
            t = dict(vk_pos=_dev(sv["vk_pos"], np.int32, d, pad=4), vk_key=_dev(sv["vk_key"], np.int32, d, pad=4),
                     vk_lo=_dev(sv["vk_range"][0], np.int64, d), vk_hi=_dev(sv["vk_range"][1], np.int64, d),
                     dense_pos=_dev(sv["dense_pos"], np.int32, d, pad=4), dense_key=_dev(sv["dense_key"], np.int32, d, pad=4),
                     dense_range=_dev(sv["dense_range"], np.int32, d, pad=2), dense_present=_dev(sv["dense_present"], np.uint8, d, pad=16),
                     present_off=_dev(sv["present_off"], np.int64, d))
        vk_len = np.asarray(sv["vk_range"][1] - sv["vk_range"][0], np.int64)
        win = np.asarray(sv["dense_range"][:, 1] - sv["dense_range"][:, 0], np.int64)
        spr = int(sv["slots_per_region"])
        self.svar2 = dict(t=t, spr=spr, vk_len=vk_len, win=win)
        # longest merged list of any slot (var_key entries + the whole dense window): workspace capacity per row
        self.max_slot_len = int((vk_len.max() if vk_len.size else 0) + (win.max() if win.size else 0))
        # typical merged length (hint for the execute kernel's tile length; the bound above counts the whole cohort's window)
        n_present = int(np.bitwise_count(np.asarray(sv["dense_present"], np.uint8)).sum(dtype=np.int64))
        self.typ_slot_len = int(2 * (vk_len.sum() + n_present) / max(vk_len.size, 1)) + 1

    def svar2_channels(self, geno_offset_idx) -> Svar2Channels:
        """gvl_svar2_channels over the resident tables; row k reads slot geno_offset_idx[k] (device i64 (b, p))."""
        t, spr = self.svar2["t"], self.svar2["spr"]
        return Svar2Channels(ptr(t["vk_pos"]), ptr(t["vk_key"]), ptr(t["vk_lo"]), ptr(t["dense_pos"]), ptr(t["dense_key"]),
                             ptr(t["dense_range"]), ptr(t["dense_present"]), ptr(t["present_off"]), ptr(t["vk_hi"]),
                             ptr(geno_offset_idx), spr)

    def fork(self) -> "Engine":
        """A second planning context (own workspace) over the SAME device tables -- one per pipeline
        slot, so several batches can be in flight on different streams."""
        e = object.__new__(Engine)
        e.__dict__.update(self.__dict__)
        e.ctx = _ffi.Ctx(self.device.index)
        e._n_work, e._fixed = 0, -1
        return e

    # ------------------------------------------------------------------ device-side batch preparation
    def dataset_view(self, full_regions: np.ndarray, n_samples: int, ploidy: int, rc_neg: bool) -> DatasetView:
        """gvl_dataset_view over a device copy of `full_regions` (uploaded once per distinct table)."""
        key = (full_regions.ctypes.data, full_regions.shape)
        ent = self._views.get(key)
        if ent is None:
            ent = self._views[key] = (_dev(np.ascontiguousarray(full_regions, np.int32).reshape(-1, 4), np.int32, self.device, pad=4),
                                      full_regions)
        return DatasetView(ptr(ent[0]), int(full_regions.shape[0]), int(n_samples), int(ploidy), 1 if rc_neg else 0)

    def batch_prep(self, view: DatasetView, ds_idx, jitter, batch: int, ref_slot: int, n_tracks: int, annot_mask: int, args,
                   sub_batch: int = 0):
        """gvl_dev_batch_prep: regions / genotype slots / strand masks / interval slots / fill seed from flat indices."""
        check(lib.gvl_dev_batch_prep(self.ctx.handle, C.byref(view), ptr(ds_idx), ptr(jitter), c_i64(int(batch)),
                                     c_i64(int(sub_batch)), c_i64(int(ref_slot)), c_i64(int(n_tracks)), C.c_uint32(int(annot_mask)), C.byref(args),
                                     _stream()))

    def track_lengths(self, regions, diffs, batch: int, ploidy: int, out):
        check(lib.gvl_dev_track_lengths(self.ctx.handle, ptr(regions), ptr(diffs), c_i64(int(batch)), c_i64(int(ploidy)),
                                        ptr(out), _stream()))

    def choose_exonic_variants(self, starts, ends, geno_offset_idx, keep_cap: int):
        """gvl_dev_choose_exonic_variants (src/genotypes/mod.rs:132-176): keep mask of the variants that lie fully
        inside [starts, ends).  `keep_cap` = `max_records(geno_offset_idx)`; returns device (keep u8, keep_offsets i64)."""
        n_q, ploidy = geno_offset_idx.shape
        keep = torch.empty(max(int(keep_cap), 1), dtype=torch.uint8, device=self.device)
        keep_offsets = torch.empty(n_q * ploidy + 1, dtype=torch.int64, device=self.device)
        check(lib.gvl_dev_choose_exonic_variants(self.ctx.handle, C.byref(self.tab), ptr(starts), ptr(ends),
                                                 ptr(geno_offset_idx), c_i64(n_q), c_i64(ploidy), ptr(keep),
                                                 c_i64(int(keep_cap)), ptr(keep_offsets), _stream()))
        return keep, keep_offsets

    # ------------------------------------------------------------------ `variants` output (csrc/gvl_variants.cu)
    def set_variant_fields(self, ref_alleles=None, info: dict | None = None, dosages=None) -> None:
        """Optional columns of the `variants` output: REF allele strings `(bytes, offsets)`, per-variant info columns
        (`_Variants.ref` / `.info`, _haps.py:139-157: any numeric dtype can drive `min_af` / `max_af`; 4-byte columns can
        also be requested as output fields) and per-call dosages (float32, parallel to `geno_v_idxs`; `Haps.dosages`)."""
        with torch.cuda.device(self.device):
            if ref_alleles is not None:
                self.ref_alleles = (_dev(ref_alleles[0], np.uint8, self.device, pad=16), _dev(ref_alleles[1], np.int64, self.device))
            for k, v in (info or {}).items():
                v = np.ascontiguousarray(v)
                if v.shape != (int(self.v_starts.numel()),):
                    raise ValueError(f"info column {k!r}: one value per variant expected, got shape {v.shape}")
                self.var_info_host[k] = v
                if v.dtype.itemsize == 4 and v.dtype.kind in "if":
                    self.var_info[k] = _dev(v, v.dtype, self.device)
                self._af_tables.clear()
            if dosages is not None:
                dz = np.ascontiguousarray(dosages, np.float32)
                if dz.size != int(self.geno_v_idxs.numel()) - 4:  # (geno_v_idxs carries 4 spare elements)
                    raise ValueError("dosages: one float32 per sparse genotype entry expected")
                self.dosages = _dev(dz, np.float32, self.device, pad=4)

    def _af_keep_table(self, min_af, max_af) -> torch.Tensor:
        """Per-VARIANT keep flags of the AF filter (int32 0 / 1), evaluated once per (min_af, max_af) on the host in the
        column's own dtype: `(af >= min_af)[v_idxs]` is what `af[v_idxs] >= min_af` computes (_flat_variants.py:899-909)."""
        key = (min_af, max_af)
        if key not in self._af_tables:
            if "AF" not in self.var_info_host:
                raise ValueError("min_af / max_af need the variants' AF column (variant_info={'AF': ...})")
            af = self.var_info_host["AF"]
            keep = np.ones(af.shape, np.bool_)
            if min_af is not None:
                keep &= af >= min_af
            if max_af is not None:
                keep &= af <= max_af
            with torch.cuda.device(self.device):
                self._af_tables[key] = _dev(keep.astype(np.int32), np.int32, self.device)
        return self._af_tables[key]

    def _const(self, a: np.ndarray) -> torch.Tensor:
        """Device copy of a small constant array (token table, dummy allele), uploaded once: a pageable upload per read
        would wait for the stream."""
        key = (a.dtype.str, a.tobytes())
        t = self._consts.get(key)
        if t is None:
            with torch.cuda.device(self.device):
                t = self._consts[key] = _dev(a, a.dtype, self.device)
        return t

    def variant_row_sizes(self, geno_offset_idx: torch.Tensor, min_af=None, max_af=None) -> np.ndarray:
        """gvl_dev_variant_row_sizes over the genotype rows `geno_offset_idx` (device i64) and one device-to-host copy: host
        int64 (n_rows, 4) = (variants kept by the AF filter, sum of their ALT lengths, of their REF lengths -- 0 without
        REF strings -- and of their reference spans).  The one wait of a variants read: it waits for the current stream."""
        if self.svar2 is not None:
            raise NotImplementedError(_SVAR2_VARIANTS)
        goi = geno_offset_idx.reshape(-1)
        n = goi.numel()
        host = torch.empty((n, 4), dtype=torch.int64, pin_memory=True)
        if n:
            keep = self._af_keep_table(min_af, max_af) if (min_af is not None or max_af is not None) else None
            ref_off = self.ref_alleles[1] if self.ref_alleles is not None else None
            with torch.cuda.device(self.device):
                out = torch.empty((n, 4), dtype=torch.int64, device=self.device)
                check(lib.gvl_dev_variant_row_sizes(self.ctx.handle, C.byref(self.tab), ptr(goi), c_i64(n), ptr(keep), ptr(ref_off),
                                                    ptr(out), _stream()))
                host.copy_(out, non_blocking=True)
                torch.cuda.current_stream(self.device).synchronize()
        return host.numpy()

    def rebase_offsets(self, offsets: torch.Tensor, n_batches: int, stride: int, bounds: torch.Tensor | None = None) -> torch.Tensor:
        """gvl_dev_rebase_offsets: the offsets of `n_batches` consecutive batches read as one call, each batch's own offsets
        starting at 0, back to back: batch i owns items [s_i, s_{i+1}) of `offsets` (n + 1 entries), s_i = min(i * stride, n),
        or bounds[min(i * stride, len(bounds) - 1)] given device `bounds`.  Returns int64 (n + n_batches,)."""
        n = offsets.numel() - 1
        out = torch.empty(n + n_batches, dtype=torch.int64, device=self.device)
        nb = bounds.numel() - 1 if bounds is not None else 0
        check(lib.gvl_dev_rebase_offsets(self.ctx.handle, ptr(offsets), c_i64(n), ptr(bounds), c_i64(nb), c_i64(int(stride)),
                                         c_i64(int(n_batches)), ptr(out), _stream()))
        return out

    def gather_variants(self, geno_offset_idx: torch.Tensor, to_rc_row, fields, sizes, n_gathered: int, dummy=None, min_af=None,
                        max_af=None, fold: int = 1, tokens: dict | None = None, row_contigs=None) -> dict:
        """The tail of `get_variants_flat` (python/genvarloader/_dataset/_flat_variants.py:869-1112) on the device: per
        (b*p) row the variant indices of its genotype slice (gather_rows, src/variants/mod.rs:6-49), optional AF
        compaction (:112-153), positions / indel lengths / info columns (`table[v_idxs]`), ALT / REF allele strings
        (:52-78), reverse complement of the alleles of negative-strand rows (:90-108) and one dummy variant per empty row
        (:157-329).  `geno_offset_idx`: device i64, flat (b*p); `to_rc_row`: device u8 (b*p) or None; `fold` = ploidy
        folds the rows of one (region, sample) into one (`unphased_union`, _flat_variants.py:925-938).
        `tokens` = {"lut": 256-entry uint8 / int32 array, "unk": int, "L": flank length, "ref": 0 | 1 window | 2 allele,
        "alt": likewise, "flank": bool} adds the token buffers of `assemble_variant_buffers` (src/variants/windows.rs:162-296):
        `flank_tokens` for the variants tail, `ref_window` / `alt_window` / tokenised `ref` / `alt` for the windows tail
        (then `alt` / `ref` in `fields` are skipped and nothing is reverse-complemented: windows are reference-oriented);
        `row_contigs`: device i32, contig of every (b*p) row.  `sizes`: the `VariantSizes` of these rows and settings
        (`_variant_sizes.variant_buffer_sizes` over `variant_row_sizes`), `n_gathered`: the rows' summed genotype slice
        lengths (`max_records`, from the host copy of the genotype offsets): every buffer is sized from them, so nothing
        here waits for the device.
        Returns {"row_offsets": i64, "v_idxs": i32, name: tensor | (data, seq_offsets)}."""
        if self.svar2 is not None:
            raise NotImplementedError(_SVAR2_VARIANTS)
        h, dev, st = self.ctx.handle, self.device, _stream
        goi = geno_offset_idx.reshape(-1).contiguous()
        n_rows = goi.numel()
        i64 = lambda n: torch.empty(n, dtype=torch.int64, device=dev)
        with torch.cuda.device(dev):
            row_off = i64(n_rows + 1)
            check(lib.gvl_dev_gather_rows_offsets(h, ptr(goi), c_i64(n_rows), ptr(self.geno_starts), ptr(self.geno_stops), ptr(row_off), st()))
            n = int(n_gathered)
            filtered = min_af is not None or max_af is not None
            v_idxs = torch.empty(n, dtype=torch.int32, device=dev)
            # positions and indel lengths ride along with the row gather (they are re-taken after an AF compaction)
            pre = {k: torch.empty(n, dtype=torch.int32, device=dev) for k in ("start", "ilen") if k in fields and not filtered}
            check(lib.gvl_dev_gather_variant_rows(h, C.byref(self.tab), ptr(goi), c_i64(n_rows), ptr(row_off), c_i64(n), ptr(v_idxs),
                                                  ptr(pre.get("start")), ptr(pre.get("ilen")), st()))

            def take(table: torch.Tensor) -> torch.Tensor:
                out = torch.empty(n, dtype=table.dtype, device=dev)
                check(lib.gvl_dev_take_u32(h, ptr(table), ptr(v_idxs), c_i64(n), ptr(out), st()))
                return out

            dosage = None
            if "dosage" in fields:  # parallel to the genotypes: same offset ranges (_flat_variants.py:911-921)
                if self.dosages is None:
                    raise ValueError("Missing variant fields: ['dosage']")
                dosage = torch.empty(n, dtype=torch.float32, device=dev)
                check(lib.gvl_dev_gather_rows(h, ptr(goi), c_i64(n_rows), ptr(self.geno_starts), ptr(self.dosages), ptr(row_off), c_i64(n),
                                              ptr(dosage), st()))
            if min_af is not None or max_af is not None:  # _flat_variants.py:899-923
                keep = (take(self._af_keep_table(min_af, max_af)) != 0).view(torch.uint8)
                pos, new_off = i64(n + 1), i64(n_rows + 1)
                check(lib.gvl_dev_compact_keep_offsets(h, ptr(keep), c_i64(n), ptr(row_off), c_i64(n_rows), ptr(pos), ptr(new_off), st()))
                n_keep = sizes.total("variants", filled=False)
                kept = torch.empty(n_keep, dtype=torch.int32, device=dev)
                check(lib.gvl_dev_compact_keep(h, ptr(v_idxs), ptr(keep), c_i64(n), ptr(pos), ptr(kept), st()))
                if dosage is not None:  # compacted with the SAME mask (:923-926)
                    kd = torch.empty(n_keep, dtype=torch.float32, device=dev)
                    check(lib.gvl_dev_compact_keep(h, ptr(dosage), ptr(keep), c_i64(n), ptr(pos), ptr(kd), st()))
                    dosage = kd
                v_idxs, row_off, n = kept, new_off, n_keep
            if fold > 1:
                row_off = row_off[::fold].contiguous()
                if to_rc_row is not None:
                    to_rc_row = to_rc_row[::fold].contiguous()
                n_rows //= fold

            out = {"v_idxs": v_idxs}
            alleles = {}
            windows_mode = tokens is not None and (tokens.get("ref") or tokens.get("alt"))
            tok_fixed = {}   # flank_tokens: tokens per variant (fixed inner axis: returned without seq offsets)
            tok_dummy = {}   # window field -> dummy window length
            if tokens is not None:
                lut_np = np.ascontiguousarray(tokens["lut"])
                tdt = torch.uint8 if lut_np.dtype == np.uint8 else torch.int32
                tb = lut_np.dtype.itemsize
                d_lut = self._const(lut_np)
                L = int(tokens["L"])
                if fold > 1 and row_contigs is not None:
                    row_contigs = row_contigs[::fold].contiguous()
                v_contigs = None
                if row_contigs is not None:  # _flat_variants.py:985-989
                    v_contigs = torch.empty(n, dtype=torch.int32, device=dev)
                    check(lib.gvl_dev_expand_rows_u32(h, ptr(row_contigs), ptr(row_off), c_i64(n_rows), c_i64(n), ptr(v_contigs), st()))

                def window(kind: int):
                    if kind == 2:  # GVL_WINDOW_FLANKS: 2 L tokens per variant, no offsets
                        data = torch.empty(n * 2 * L, dtype=tdt, device=dev)
                        check(lib.gvl_dev_variant_windows(h, C.byref(self.tab), ptr(v_idxs), ptr(v_contigs), c_i64(n), c_i64(L), C.c_int(2),
                                                          c_u8(self.pad_char), ptr(d_lut), C.c_int(tb), c_vp(0), c_i64(n * 2 * L), ptr(data), st()))
                        return data
                    w_off = i64(n + 1)
                    check(lib.gvl_dev_variant_windows_offsets(h, C.byref(self.tab), ptr(v_idxs), c_i64(n), c_i64(L), C.c_int(kind), ptr(w_off), st()))
                    nt = sizes.total("alt_window" if kind == 1 else "ref_window", filled=False)
                    data = torch.empty(nt, dtype=tdt, device=dev)
                    check(lib.gvl_dev_variant_windows(h, C.byref(self.tab), ptr(v_idxs), ptr(v_contigs), c_i64(n), c_i64(L), C.c_int(kind),
                                                      c_u8(self.pad_char), ptr(d_lut), C.c_int(tb), ptr(w_off), c_i64(nt), ptr(data), st()))
                    return data, w_off

                def tok_alleles(name, ab, ao):
                    seq_off = i64(n + 1)
                    check(lib.gvl_dev_gather_alleles_offsets(h, ptr(v_idxs), c_i64(n), ptr(ao), ptr(seq_off), st()))
                    nb = sizes.total(name, filled=False)
                    data = torch.empty(nb, dtype=tdt, device=dev)
                    check(lib.gvl_dev_gather_alleles(h, ptr(v_idxs), c_i64(n), ptr(ab), ptr(ao), ptr(seq_off), c_i64(nb), ptr(d_lut),
                                                     C.c_int(tb), ptr(data), st()))
                    return data, seq_off

                if windows_mode:  # windows.rs:227-296 (ref side first, like the reference's field order)
                    d_alt = len(dummy.alt) if dummy is not None else 0
                    d_ref = len(dummy.ref) if dummy is not None else 0
                    if tokens.get("ref") == 1:
                        alleles["ref_window"], tok_dummy["ref_window"] = window(0), 2 * L + d_ref
                    elif tokens.get("ref") == 2:
                        if self.ref_alleles is None:
                            raise ValueError("VarWindowOpt(ref='allele') needs the REF allele strings (ref_alleles=)")
                        alleles["ref"], tok_dummy["ref"] = tok_alleles("ref", *self.ref_alleles), d_ref
                    if tokens.get("alt") == 1:
                        alleles["alt_window"], tok_dummy["alt_window"] = window(1), 2 * L + d_alt
                    elif tokens.get("alt") == 2:
                        alleles["alt"], tok_dummy["alt"] = tok_alleles("alt", self.alt_alleles, self.alt_offsets), d_alt
                    to_rc_row = None
                elif tokens.get("flank") and L > 0:
                    # 2 L tokens per variant; carried as a two-level ragged with constant strides so that the dummy fill
                    # below is the same fill_empty_seq pass for 1- and 4-byte tokens
                    alleles["flank_tokens"] = (window(2), torch.arange(0, (n + 1) * 2 * L, 2 * L, dtype=torch.int64, device=dev))
                    tok_dummy["flank_tokens"] = tok_fixed["flank_tokens"] = 2 * L
            for name in fields:
                if name in ("alt", "ref") and windows_mode:
                    continue
                if name in ("alt", "ref"):
                    if name == "ref" and self.ref_alleles is None:
                        raise ValueError("Missing variant fields: ['ref']")
                    ab, ao = (self.alt_alleles, self.alt_offsets) if name == "alt" else self.ref_alleles
                    seq_off = i64(n + 1)
                    check(lib.gvl_dev_gather_alleles_offsets(h, ptr(v_idxs), c_i64(n), ptr(ao), ptr(seq_off), st()))
                    nb = sizes.total(name, filled=False)
                    data = torch.empty(nb, dtype=torch.uint8, device=dev)
                    check(lib.gvl_dev_gather_alleles(h, ptr(v_idxs), c_i64(n), ptr(ab), ptr(ao), ptr(seq_off), c_i64(nb), c_vp(0),
                                                     C.c_int(1), ptr(data), st()))
                    alleles[name] = (data, seq_off)
                elif name == "dosage":
                    out[name] = dosage
                elif name == "start":
                    out[name] = pre[name] if name in pre else take(self.v_starts)
                elif name == "ilen":
                    out[name] = pre[name] if name in pre else take(self.ilens)
                elif name in self.var_info:
                    out[name] = take(self.var_info[name])
                else:
                    raise ValueError(f"Missing variant fields: [{name!r}]")
            def rc(alleles_: dict, n_var: int, var_off: torch.Tensor) -> None:
                # negative-strand rows: reverse-complement their alleles in place (applied after the dummy fill, like
                # `_query.py:485-529` after `get_variants_flat`)
                if to_rc_row is None:
                    return
                for data, seq_off in alleles_.values():
                    check(lib.gvl_dev_rc_alleles(h, ptr(data), ptr(seq_off), c_i64(n_var), ptr(var_off), c_i64(n_rows), ptr(to_rc_row),
                                                 c_i64(data.numel()), st()))

            if dummy is None:
                rc({k: v for k, v in alleles.items() if k not in tok_dummy}, n, row_off)
                out["row_offsets"] = row_off
                out.update({k: (v[0] if k in tok_fixed else v) for k, v in alleles.items()})
                return out
            # ---- one dummy variant per empty row (fill_empty_groups, _flat_variants.py:501-535) ----
            new_off = i64(n_rows + 1)
            check(lib.gvl_dev_fill_empty_offsets(h, ptr(row_off), c_i64(n_rows), ptr(new_off), st()))
            n_new = sizes.total("variants")
            for name in list(out):
                t = out[name]
                np_dt = np.float32 if t.dtype == torch.float32 else np.int32
                fill = -1 if name == "v_idxs" else dummy.scalar_for(name, np_dt)
                bits = int(np.array(fill, np_dt).view(np.uint32))
                filled = torch.empty(n_new, dtype=t.dtype, device=dev)
                check(lib.gvl_dev_fill_empty_fixed(h, ptr(t), ptr(row_off), c_i64(n_rows), ptr(new_off), c_i64(n_new), c_i64(1),
                                                   C.c_uint32(bits), ptr(filled), st()))
                out[name] = filled
            src_var = i64(max(n_new, 1))
            for name, (data, seq_off) in alleles.items():
                if name in tok_dummy:  # token windows / flank tokens: all-unknown tokens (:385-393, :527-534)
                    db = np.full(tok_dummy[name], tokens["unk"], np.uint8 if data.dtype == torch.uint8 else np.int32)
                else:
                    db = np.frombuffer(dummy.alt if name == "alt" else dummy.ref, np.uint8)
                d_dummy = self._const(db)
                new_seq = i64(n_new + 1)
                check(lib.gvl_dev_fill_empty_seq_offsets(h, ptr(row_off), c_i64(n_rows), ptr(seq_off), c_i64(db.size), ptr(new_off),
                                                         c_i64(n_new), ptr(src_var), ptr(new_seq), st()))
                nb = sizes.total(name)
                filled = torch.empty(nb, dtype=data.dtype, device=dev)
                check(lib.gvl_dev_fill_empty_seq(h, ptr(data), C.c_int(data.element_size()), ptr(seq_off), ptr(d_dummy), ptr(src_var),
                                                 ptr(new_seq), c_i64(n_new), c_i64(nb), ptr(filled), st()))
                alleles[name] = (filled, new_seq)
            rc({k: v for k, v in alleles.items() if k not in tok_dummy}, n_new, new_off)
            out.update({k: (v[0] if k in tok_fixed else v) for k, v in alleles.items()})
            out["row_offsets"] = new_off
            return out

    # ------------------------------------------------------------------ tracks
    def add_track(self, name: str, itv_starts, itv_ends, itv_values, itv_offsets) -> None:
        """Upload one track's interval SoA.  Slots whose intervals overlap (legal: the reference paints in stored order,
        last write wins, src/intervals.rs:64-85) are flattened into the equivalent disjoint list first."""
        st, en = np.ascontiguousarray(itv_starts, np.int32), np.ascontiguousarray(itv_ends, np.int32)
        off = np.ascontiguousarray(itv_offsets, np.int64)
        n_bad = c_i64(0)
        check(lib.gvl_intervals_overlap(ptr(st), ptr(en), ptr(off), c_i64(off.size - 1), C.byref(n_bad)))
        if n_bad.value:
            va = np.ascontiguousarray(itv_values, np.float32)
            cap = 2 * st.size + 16
            o_s, o_e, o_v = np.empty(cap, np.int32), np.empty(cap, np.int32), np.empty(cap, np.float32)
            o_off, n_out = np.empty(off.size, np.int64), c_i64(0)
            check(lib.gvl_flatten_intervals(ptr(st), ptr(en), ptr(va), ptr(off), c_i64(off.size - 1), ptr(o_s), ptr(o_e), ptr(o_v),
                                            ptr(o_off), c_i64(cap), C.byref(n_out)))
            itv_starts, itv_ends, itv_values, itv_offsets = o_s[: n_out.value], o_e[: n_out.value], o_v[: n_out.value], o_off
        with torch.cuda.device(self.device):
            t = (_dev(itv_starts, np.int32, self.device, pad=4), _dev(itv_ends, np.int32, self.device, pad=4),
                 _dev(itv_values, np.float32, self.device, pad=4), _dev(itv_offsets, np.int64, self.device))
        self.tracks[name] = t + (Intervals(ptr(t[0]), ptr(t[1]), ptr(t[2]), ptr(t[3]), int(t[3].numel() - 1)),)

    # ------------------------------------------------------------------ capacity
    def max_records(self, geno_offset_idx_host: np.ndarray) -> int:
        """Upper bound on the summed per-row variant counts (host O(batch) gather)."""
        g = np.asarray(geno_offset_idx_host).reshape(-1)
        if self.svar2 is not None and g.size and int(g.max()) < self.empty_slot:
            sv = self.svar2  # merged lists: own var_key entries + the region's whole dense window
            return int(sv["vk_len"][g].sum() + sv["win"][g // sv["spr"]].sum())
        d = self.geno_offsets_host[1, g] - self.geno_offsets_host[0, g]
        return int(np.maximum(d, 0).sum())

    # ------------------------------------------------------------------ haplotypes
    def plan(self, regions: torch.Tensor, shifts: torch.Tensor, geno_offset_idx: torch.Tensor, output_length: int,
             max_records: int, keep=None, keep_offsets=None, to_rc=None, out_offsets=None, diffs=None, use_svar2=True):
        """gvl_dev_hap_plan.  All tensors live on this engine's device; nothing synchronises."""
        batch, ploidy = geno_offset_idx.shape
        n_work = batch * ploidy
        if out_offsets is None:
            out_offsets = torch.empty(n_work + 1, dtype=torch.int64, device=self.device)
        if self.svar2 is not None and use_svar2:
            if keep is not None:
                raise NotImplementedError("keep masks (var_filter) are not supported with the svar2 source")
            ch = self.svar2_channels(geno_offset_idx)
            check(lib.gvl_dev_hap_plan_svar2(self.ctx.handle, C.byref(self.tab), C.byref(ch), ptr(regions), ptr(shifts),
                                             c_i64(batch), c_i64(ploidy), ptr(to_rc), c_i64(int(output_length)),
                                             c_i64(int(max_records)), ptr(out_offsets), ptr(diffs), _stream()))
            self._n_work, self._fixed = n_work, int(output_length)
            return out_offsets
        check(lib.gvl_dev_hap_plan(self.ctx.handle, C.byref(self.tab), ptr(regions), ptr(shifts), ptr(geno_offset_idx),
                                   c_i64(batch), c_i64(ploidy), ptr(keep), ptr(keep_offsets), ptr(to_rc),
                                   c_i64(int(output_length)), c_i64(int(max_records)), ptr(out_offsets), ptr(diffs),
                                   _stream()))
        self._n_work, self._fixed = n_work, int(output_length)
        return out_offsets

    def total(self) -> int:
        t = c_i64(0)
        check(lib.gvl_dev_hap_total(self.ctx.handle, _stream(), C.byref(t)))
        return int(t.value)

    def execute(self, mode: str = "haplotypes", out=None, annot_v=None, annot_pos=None):
        """gvl_dev_hap_exec into (pre)allocated tensors.  Returns the flat buffers."""
        m = MODES[mode]
        total = self.total()
        mult = 4 if m in (MODE_ONEHOT, MODE_ONEHOT_CF) else 1
        if out is None:
            out = torch.empty(total * mult, dtype=torch.uint8, device=self.device)
        if m == MODE_ANNOTATED:
            if annot_v is None:
                annot_v = torch.empty(total, dtype=torch.int32, device=self.device)
            if annot_pos is None:
                annot_pos = torch.empty(total, dtype=torch.int32, device=self.device)
        check(lib.gvl_dev_hap_exec(self.ctx.handle, C.byref(self.tab), C.c_int(m), c_u8(self.pad_char), ptr(out),
                                   ptr(annot_v), ptr(annot_pos), _stream()))
        if m == MODE_ANNOTATED:
            return out, annot_v, annot_pos
        return out

    def get_diffs(self, geno_offset_idx, q_starts=None, q_ends=None, keep=None, keep_offsets=None, clipped=True, regions=None,
                  max_records: int = 0):
        n_q, ploidy = geno_offset_idx.shape
        diffs = torch.empty((n_q, ploidy), dtype=torch.int32, device=self.device)
        if self.svar2 is not None:  # hap_diffs_svar2 over the merged lists (src/svar2/mod.rs:73-146)
            ch = self.svar2_channels(geno_offset_idx)
            check(lib.gvl_dev_hap_diffs_svar2(self.ctx.handle, C.byref(self.tab), C.byref(ch), ptr(regions), c_i64(n_q),
                                              c_i64(ploidy), c_i64(int(max_records)), ptr(diffs), _stream()))
            return diffs
        check(lib.gvl_dev_get_diffs_sparse(self.ctx.handle, C.byref(self.tab), ptr(geno_offset_idx), c_i64(n_q),
                                           c_i64(ploidy), ptr(keep), ptr(keep_offsets), ptr(q_starts), ptr(q_ends),
                                           C.c_int(1 if clipped else 0), ptr(diffs), _stream()))
        return diffs

    # ------------------------------------------------------------------ tracks
    def track_descs(self, names, strategy_ids=None, params=None):
        """Descriptor arrays of a track call: the interval table of every track in `names` and, for realignment, its
        insertion-fill id and parameter (None, None when painting)."""
        n = len(names)
        itv = (Intervals * n)(*[self.tracks[x][4] for x in names])
        if strategy_ids is None:
            return itv, None, None
        return itv, (c_i32 * n)(*[int(s) for s in strategy_ids]), (C.c_double * n)(*[float(p) for p in params])

    def _realign_args(self, names, regions, shifts, geno_offset_idx, offset_idxs, track_lengths, out_offsets, total_per_track,
                      strategy_ids, params, base_seed, max_records, keep, keep_offsets, to_rc, query_seed, base_seed_dev, batch,
                      sub_batch):
        """The arguments every gvl_dev_realign_tracks* entry takes after its variant source and before its layout."""
        b_cap, ploidy = geno_offset_idx.shape
        batch = b_cap if batch is None else int(batch)  # (a prefix of preallocated buffers)
        itv, sid, par = self.track_descs(names, strategy_ids, params)
        return (ptr(regions), ptr(shifts), ptr(geno_offset_idx), c_i64(batch), c_i64(ploidy), ptr(keep), ptr(keep_offsets),
                ptr(to_rc), c_i64(len(names)), itv, ptr(offset_idxs), ptr(track_lengths), ptr(out_offsets),
                c_i64(int(total_per_track)), sid, par, c_u64(int(base_seed)), ptr(base_seed_dev), c_i64(int(sub_batch)),
                ptr(query_seed), c_i64(int(max_records)))

    def realign_tracks(self, names, regions, shifts, geno_offset_idx, offset_idxs, track_lengths, out_offsets,
                       total_per_track: int, strategy_ids, params, base_seed: int, max_records: int, keep=None,
                       keep_offsets=None, to_rc=None, query_seed=None, out=None, layout="tbp", base_seed_dev=None,
                       batch=None, sub_batch: int = 0, row_dst=None, row_tstride=None, dtype=torch.float32):
        """gvl_dev_realign_tracks: all `names` in one plan + one execute launch.
        offset_idxs: int64 (n_tracks, batch) device; out: `dtype` (n_tracks * total_per_track,), track-major
        (layout="tbp", the reference's flat buffer), with every query's tracks adjacent (layout="btp",
        gvl_dev_realign_tracks_btp: the order the reference's (b, t, p, ~l) offsets describe) or wherever the
        per-row table puts each row (layout="rows": row k of track t starts at row_dst[k] + t * row_tstride[k],
        device int64 (batch * ploidy,) each; gvl_dev_realign_tracks_plan_rows).  `dtype` (of `out` when given): float32,
        or bfloat16 / float16 -- the float32 values rounded to nearest even by the execute kernel's stores."""
        if out is None:
            track_dtype_code(dtype)
            out = torch.empty(len(names) * total_per_track, dtype=dtype, device=self.device)
        if self.svar2 is not None or layout == "rows" or out.dtype != torch.float32:
            self.realign_tracks_plan(names, regions, shifts, geno_offset_idx, offset_idxs, track_lengths, out_offsets,
                                     total_per_track, strategy_ids, params, base_seed, max_records, keep, keep_offsets, to_rc,
                                     query_seed, layout, base_seed_dev, batch, sub_batch, row_dst, row_tstride)
            return self.realign_tracks_exec(out)
        args = self._realign_args(names, regions, shifts, geno_offset_idx, offset_idxs, track_lengths, out_offsets,
                                  total_per_track, strategy_ids, params, base_seed, max_records, keep, keep_offsets, to_rc,
                                  query_seed, base_seed_dev, batch, sub_batch)
        fn = lib.gvl_dev_realign_tracks_btp if layout == "btp" else lib.gvl_dev_realign_tracks
        check(fn(self.ctx.handle, C.byref(self.tab), *args, ptr(out), _stream()))
        return out

    def realign_tracks_plan(self, names, regions, shifts, geno_offset_idx, offset_idxs, track_lengths, out_offsets,
                            total_per_track: int, strategy_ids, params, base_seed: int, max_records: int, keep=None,
                            keep_offsets=None, to_rc=None, query_seed=None, layout="tbp", base_seed_dev=None, batch=None,
                            sub_batch: int = 0, row_dst=None, row_tstride=None):
        """gvl_dev_realign_tracks_plan (layout="rows": gvl_dev_realign_tracks_plan_rows): everything of `realign_tracks`
        but the execute launch (variant plan, tile map, per-tile searches); `realign_tracks_exec(out)` writes the values,
        possibly on another stream."""
        if layout == "rows" and (row_dst is None or row_tstride is None):
            raise ValueError('layout="rows" needs row_dst and row_tstride')
        args = self._realign_args(names, regions, shifts, geno_offset_idx, offset_idxs, track_lengths, out_offsets,
                                  total_per_track, strategy_ids, params, base_seed, max_records, keep, keep_offsets, to_rc,
                                  query_seed, base_seed_dev, batch, sub_batch)
        ch = self.svar2_channels(geno_offset_idx) if self.svar2 is not None else None
        src = C.byref(ch) if ch is not None else c_vp(0)
        if layout == "rows":
            check(lib.gvl_dev_realign_tracks_plan_rows(self.ctx.handle, C.byref(self.tab), src, *args, ptr(row_dst),
                                                       ptr(row_tstride), _stream()))
        else:
            check(lib.gvl_dev_realign_tracks_plan(self.ctx.handle, C.byref(self.tab), src, *args,
                                                  C.c_int(1 if layout == "btp" else 0), _stream()))

    def realign_tracks_exec(self, out):
        """gvl_dev_realign_tracks_exec_dtype: the planned call's values into `out`, in out's dtype (float32, bfloat16,
        float16)."""
        check(lib.gvl_dev_realign_tracks_exec_dtype(self.ctx.handle, ptr(out), track_dtype_code(out.dtype), _stream()))
        return out

    def intervals_to_tracks(self, name, offset_idxs, starts, out_offsets, total: int, out=None):
        """gvl_dev_intervals_to_tracks: paint one track's stored intervals into dense windows."""
        n_q = int(starts.numel())
        if out is None:
            out = torch.empty(total, dtype=torch.float32, device=self.device)
        check(lib.gvl_dev_intervals_to_tracks(self.ctx.handle, C.byref(self.tracks[name][4]), ptr(offset_idxs), ptr(starts),
                                              c_i64(n_q), ptr(out_offsets), c_i64(int(total)), ptr(out), _stream()))
        return out

    def paint_tracks(self, names, offset_idxs, starts, out_offsets, total_per_track: int, to_rc=None, out=None,
                     n_queries=None, layout="btp", row_dst=None, row_tstride=None, dtype=torch.float32):
        """gvl_dev_paint_tracks: stored intervals of all `names` painted in one launch, (b, t, ~l) order,
        masked rows reversed.  offset_idxs: int64 (n_tracks, batch) device.  layout="rows"
        (gvl_dev_paint_tracks_rows): query q of track t starts at row_dst[q] + t * row_tstride[q] instead.
        `dtype` (of `out` when given): float32, bfloat16 or float16 (gvl_dev_paint_tracks_dtype)."""
        n_tracks, n_q = len(names), int(starts.numel() if n_queries is None else n_queries)
        itv = self.track_descs(names)[0]
        if out is None:
            track_dtype_code(dtype)
            out = torch.empty(n_tracks * int(total_per_track), dtype=dtype, device=self.device)
        if layout == "rows" and (row_dst is None or row_tstride is None):
            raise ValueError('layout="rows" needs row_dst and row_tstride')
        if out.dtype != torch.float32:
            rows = layout == "rows"
            check(lib.gvl_dev_paint_tracks_dtype(self.ctx.handle, n_tracks, itv, ptr(offset_idxs), ptr(starts), n_q,
                                                 ptr(out_offsets), int(total_per_track), ptr(to_rc), ptr(row_dst if rows else None),
                                                 ptr(row_tstride if rows else None), ptr(out), track_dtype_code(out.dtype),
                                                 _stream()))
            return out
        if layout == "rows":
            check(lib.gvl_dev_paint_tracks_rows(self.ctx.handle, n_tracks, itv, ptr(offset_idxs), ptr(starts), n_q,
                                                ptr(out_offsets), int(total_per_track), ptr(to_rc), ptr(row_dst),
                                                ptr(row_tstride), ptr(out), _stream()))
            return out
        check(lib.gvl_dev_paint_tracks(self.ctx.handle, c_i64(n_tracks), itv, ptr(offset_idxs), ptr(starts), c_i64(n_q),
                                       ptr(out_offsets), c_i64(int(total_per_track)), ptr(to_rc), ptr(out), _stream()))
        return out

    def track_intervals(self, names, row_slot, row_track, row_w0, row_w1, dtype=torch.float32):
        """gvl_dev_track_intervals: row k = the stored intervals of slot row_slot[k] (device i64) of track
        names[row_track[k]] (device i32) that overlap [row_w0[k], row_w1[k]) (device i32), clipped to it.  A sizing call,
        ONE wait for the total, then the emit call into buffers of exactly that size.  Returns (offsets i64 (n + 1,),
        starts i32, ends i32, values of `dtype`): float32, or bfloat16 / float16 narrowed at the kernel's store."""
        code = track_dtype_code(dtype)
        n = int(row_slot.numel())
        itv = self.track_descs(names)[0]
        dev = self.device
        offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
        rows = (ptr(row_slot), ptr(row_track), ptr(row_w0), ptr(row_w1), c_i64(n), ptr(offsets))
        check(lib.gvl_dev_track_intervals(self.ctx.handle, itv, len(names), *rows, 0, None, None, None, code, _stream()))
        total = int(offsets[-1])  # the read's one wait
        starts = torch.empty(total, dtype=torch.int32, device=dev)
        ends = torch.empty(total, dtype=torch.int32, device=dev)
        values = torch.empty(total, dtype=dtype, device=dev)
        if total:
            check(lib.gvl_dev_track_intervals(self.ctx.handle, itv, len(names), *rows, total, ptr(starts), ptr(ends), ptr(values),
                                              code, _stream()))
        return offsets, starts, ends, values

    def check(self) -> None:
        """Synchronise and surface device-side status flags (workspace overflow)."""
        self.ctx.check(torch.cuda.current_stream().cuda_stream)
