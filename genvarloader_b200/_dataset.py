"""GPU-resident `Dataset`: the reference's `gvl.Dataset` surface for the haplotype / track hot path.

Mirrors (names, argument meaning, error behaviour, return shapes):
  * `Dataset` state + `with_settings / with_len / with_seqs / with_tracks / with_insertion_fill /
    with_output_format / subset_to / __getitem__`      python/genvarloader/_dataset/_impl.py:78-2121
  * index parsing (`DatasetIndexer.parse_idx`)          python/genvarloader/_dataset/_indexing.py:208-264
  * read-time prep: jitter, strand mask, shifts, seeds   _dataset/_query.py:153-204, _haps.py:678-768,
                                                         _reconstruct.py:168-226
  * output shaping (to_fixed / pad / ragged, squeeze)    _dataset/_query.py:94-127

Host work per call is O(batch) numpy (index maths, RNG draws in the reference's order); everything
sample-scale lives on the GPU inside `Engine`.  Results are torch CUDA tensors.
Not supported (outside the hot-path scope, raise): fixed-length or jittered spliced output.
"""
from __future__ import annotations

from dataclasses import dataclass, field, replace
from typing import Literal

import numpy as np
import torch

from ._engine import Engine, track_dtype_code
from ._insertion_fill import InsertionFill, Repeat5p, lower
from ._variant_sizes import variant_buffer_sizes
from ._types import (AnnotatedHaps, DummyVariant, Ragged, RaggedAlleles, RaggedAnnotatedHaps, RaggedIntervals, RaggedVariants,
                     VarWindowOpt, build_token_lut)

SeqKind = Literal["reference", "haplotypes", "annotated"]
N_CHAR = ord("N")


def _idx_to_array(idx, n: int) -> np.ndarray:
    if isinstance(idx, slice):
        return np.arange(n, dtype=np.int64)[idx]
    a = np.asarray(idx)
    if a.dtype == np.bool_:
        if a.shape != (n,):
            raise IndexError(f"boolean index of shape {a.shape} does not match axis of size {n}")
        return np.flatnonzero(a).astype(np.int64)
    a = a.astype(np.int64)
    if ((a < -n) | (a >= n)).any():
        raise IndexError(f"index out of bounds for axis of size {n}")
    return np.where(a < 0, a + n, a)


@dataclass(frozen=True)
class Dataset:
    """Effective shape `(n_regions, n_samples, [tracks], [ploidy], output_length)`; indexable on the
    first two axes like a 2-D array (reference docstring, _impl.py:80-115)."""

    engine: Engine
    full_regions: np.ndarray            # int32 (R, 4): contig_idx, start, end, strand
    sample_names: tuple
    ploidy: int
    max_jitter: int = 0
    track_kinds: dict = field(default_factory=dict)   # name -> "sample" | "annot"
    # ---- settings (reference defaults: _impl.py:119-162) ----
    output_length: object = "ragged"                  # "ragged" | "variable" | int
    sequence_type: object = "haplotypes"              # "reference" | "haplotypes" | "annotated" | None
    active_tracks: tuple = ()
    track_output: str = "tracks"                      # with_tracks(kind=...): "tracks" (values) | "intervals"
    insertion_fill: dict = field(default_factory=dict)
    jitter: int = 0
    deterministic: bool = True
    rc_neg: bool = True
    var_filter: object = None                         # None | "exonic"
    realign_tracks: bool = True
    output_format: str = "ragged"                     # "ragged" | "flat"  (with_output_format)
    encoding: str = "bytes"                           # "bytes" | "onehot" | "onehot_cf"  (this build's fused one-hot)
    track_dtype: torch.dtype = torch.float32          # element type of track outputs (with_track_dtype, this build's extension)
    var_fields: tuple = ("alt", "ilen", "start")      # fields of the "variants" output (_haps.py:268)
    dummy_variant: object = None                      # DummyVariant for empty (region, sample, ploid) groups, or None
    unphased_union: bool = False                      # fold the ploidy rows of a (region, sample) into one (_flat_variants.py:925-938)
    min_af: object = None                             # AF filter of the "variants" output (_flat_variants.py:899-923)
    max_af: object = None
    window_opt: object = None                         # VarWindowOpt of with_seqs("variant-windows", ...)
    flank_length: int = 0                             # "variants": flank tokens around every variant (with a token alphabet)
    token_alphabet: object = None                     # bytes; with unknown_token defines the byte -> token table
    unknown_token: object = None
    rng: np.random.Generator = field(default_factory=np.random.default_rng)
    region_subset: object = None
    sample_subset: object = None
    region_map: object = None                         # input-BED row -> storage row (datasets opened from disk)
    splice_rows: object = None                        # spliced: tuple of int64 arrays of STORAGE region indices, one per splice row
    splice_names: object = None                       # spliced: names of the splice rows (or None)
    bed_columns: object = None                        # opened datasets: extra input-BED columns (name -> array, input order)
    _cache: dict = field(default_factory=dict, compare=False, repr=False)  # per-state lazies (fixed-length pipeline)

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_arrays(cls, device, reference, ref_offsets, v_starts, ilens, alt_alleles, alt_offsets, geno_v_idxs,
                    geno_offsets, regions, n_samples: int, ploidy: int, max_jitter: int = 0, tracks: dict | None = None,
                    track_kinds: dict | None = None, sample_names=None, rng=None, ref_alleles=None,
                    variant_info: dict | None = None, dosages=None) -> "Dataset":
        """In-memory dataset (the GPU counterpart of `get_dummy_dataset`, python/genvarloader/_dummy.py).
        `tracks`: name -> (itv_starts, itv_ends, itv_values, itv_offsets); SAMPLE tracks have one interval slot
        per (region, sample), ANNOT tracks one per region (_reconstruct.py:233-236).  `ref_alleles` = (bytes, offsets) of
        the REF strings, `variant_info` = {name: numeric column, one value per variant} and `dosages` (float32, parallel to
        `geno_v_idxs`) feed the "variants" output (`var_fields`, AF filter)."""
        eng = Engine(device, reference, ref_offsets, v_starts, ilens, alt_alleles, alt_offsets, geno_v_idxs, geno_offsets)
        if ref_alleles is not None or variant_info or dosages is not None:
            eng.set_variant_fields(ref_alleles, variant_info, dosages)
        return cls._from_engine(eng, regions, n_samples, ploidy, max_jitter, tracks, track_kinds, sample_names, rng)

    @classmethod
    def from_synth(cls, device, d, rng=None, svar2=None) -> "Dataset":
        """From a `genvarloader_b200.synth.SynthData`; `svar2`: a `synth.to_svar2_dataset(d)` dict = keep the variants as
        a resident svar2 two-channel source instead of the SVAR1 CSR."""
        if svar2 is not None:
            return cls.from_svar2_arrays(device, d.reference, d.ref_offsets, svar2, d.regions, d.n_samples, d.ploidy,
                                         d.max_jitter, d.tracks, rng=rng)
        return cls.from_arrays(device, d.reference, d.ref_offsets, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                               d.geno_v_idxs, d.geno_offsets, d.regions, d.n_samples, d.ploidy, d.max_jitter, d.tracks,
                               rng=rng)

    @classmethod
    def from_svar2_arrays(cls, device, reference, ref_offsets, sv: dict, regions, n_samples: int, ploidy: int,
                          max_jitter: int = 0, tracks: dict | None = None, track_kinds: dict | None = None,
                          sample_names=None, rng=None) -> "Dataset":
        """In-memory dataset over a resident svar2 two-channel variant source -- the GPU counterpart of `Svar2Haps`
        (python/genvarloader/_dataset/_svar2_haps.py:183): per-(region, sample, ploid) var_key ranges, per-region dense
        windows and presence bits (docs/source/format.md:88-96) stay in HBM, every read merges the two channels on the
        device (src/svar2/mod.rs:45-66).  `sv`: see `synth.to_svar2_dataset` for the arrays."""
        eng = Engine.from_svar2(device, reference, ref_offsets, sv, len(regions) * int(n_samples) * int(ploidy))
        return cls._from_engine(eng, regions, n_samples, ploidy, max_jitter, tracks, track_kinds, sample_names, rng)

    @classmethod
    def open(cls, path, reference=None, device="cuda", jitter: int = 0, rng=None, deterministic: bool = True,
             rc_neg: bool = True, svar=None) -> "Dataset":
        """Open a dataset directory written by `gvl.write` (reference `Dataset.open`, _impl.py:164-226 ->
        `_open.py:62-345`; layout: docs/source/format.md:8-49) and upload it to `device`.

        `reference`: FASTA path (plain / gzip / bgzip) or a `genvarloader_b200.Reference`; required when the dataset
        has genotypes.  Regions are addressed in the ORDER OF THE INPUT BED, like the reference (`r_idx_map`).
        Datasets linked to a `.svar` (SVAR1) store are followed (`svar=` overrides the stored path, like the reference);
        `.svar2`-backed datasets are refused (third-party store format)."""
        from ._open import Reference, read_dataset_arrays

        a = read_dataset_arrays(path, reference, svar)
        ref = a["reference"]
        n_regions, samples = len(a["full_regions"]), a["samples"]
        has_geno = "geno_v_idxs" in a
        ploidy = int(a["ploidy"]) if has_geno else 1
        if has_geno and ref is None:
            raise ValueError("this dataset has genotypes: pass `reference=` (FASTA path or Reference) to reconstruct haplotypes")
        if ref is None:  # tracks only: contig extents are never read
            ref = Reference.from_arrays(np.zeros(0, np.uint8), np.zeros(len(a["contigs"]) + 1, np.int64), a["contigs"])
        if has_geno:
            eng = Engine(device, ref.reference, ref.offsets, a["v_starts"], a["ilens"], a["alt_alleles"], a["alt_offsets"],
                         a["geno_v_idxs"], a["geno_offsets"], pad_char=ref.pad_char)
        else:
            eng = Engine(device, ref.reference, ref.offsets, np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.uint8),
                         np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(n_regions * len(samples) * ploidy + 1, np.int64),
                         pad_char=ref.pad_char)
        if has_geno and (a.get("ref_alleles") is not None or a.get("variant_info")):
            eng.set_variant_fields(a.get("ref_alleles"), a.get("variant_info"))  # "variants" output: REF strings, INFO columns
        ds = cls._from_engine(eng, a["full_regions"], len(samples), ploidy, a["max_jitter"], a["tracks"], a["track_kinds"],
                              samples, rng, sequence_type="haplotypes" if has_geno else None,
                              region_map=np.ascontiguousarray(a["region_map"], np.int64), bed_columns=a.get("bed_columns"))
        return ds.with_settings(jitter=jitter, deterministic=deterministic, rc_neg=rc_neg)

    @classmethod
    def _from_engine(cls, eng, regions, n_samples: int, ploidy: int, max_jitter: int, tracks, track_kinds, sample_names, rng,
                     **settings) -> "Dataset":
        """The common tail of the constructors: register `tracks` on `eng` (kind "sample" unless `track_kinds` says
        otherwise), give 3-column regions a + strand, name the samples s0, s1, ... unless named."""
        kinds = {}
        for name, t in (tracks or {}).items():
            eng.add_track(name, *t)
            kinds[name] = (track_kinds or {}).get(name, "sample")
        regions = np.ascontiguousarray(regions, np.int32)
        if regions.shape[1] == 3:
            regions = np.concatenate([regions, np.ones((len(regions), 1), np.int32)], 1)
        names = tuple(sample_names) if sample_names is not None else tuple(f"s{i}" for i in range(n_samples))
        return cls(engine=eng, full_regions=regions, sample_names=names, ploidy=int(ploidy), max_jitter=int(max_jitter),
                   track_kinds=kinds, active_tracks=tuple(kinds), rng=np.random.default_rng(rng), **settings)

    # ------------------------------------------------------------------ properties (reference: _impl.py:954-1110)
    @property
    def n_regions(self) -> int:
        """Number of regions -- of SPLICE ROWS when the dataset is spliced (reference _impl.py:1001-1005)."""
        return len(self.splice_rows) if self.splice_rows is not None else len(self._r_idx)

    @property
    def n_samples(self) -> int:
        return len(self._s_idx)

    @property
    def samples(self) -> list:
        return [self.sample_names[i] for i in self._s_idx]

    @property
    def shape(self) -> tuple:
        return (self.n_regions, self.n_samples)

    @property
    def full_shape(self) -> tuple:
        return (len(self.full_regions), len(self.sample_names))

    @property
    def available_var_fields(self) -> list:
        """Reference: `Haps.available_var_fields`, _haps.py:313-319."""
        eng = self.engine
        return (["alt", "ilen", "start"] + (["ref"] if eng.ref_alleles is not None else [])
                + (["dosage"] if eng.dosages is not None else []) + sorted(eng.var_info))

    @property
    def available_tracks(self) -> list:
        return list(self.track_kinds)

    @property
    def is_subset(self) -> bool:
        return self.region_subset is not None or self.sample_subset is not None

    # ---- what the dataset holds (reference: _impl.py:954-1110, 1234-1340, 1848-1895) ----
    @property
    def has_reference(self) -> bool:
        return True  # (an Engine always holds a reference; datasets without one are not opened here)

    @property
    def has_genotypes(self) -> bool:
        return self.engine.svar2 is not None or int(self.engine.alt_offsets.numel()) > 1  # (a variant table with entries)

    @property
    def has_intervals(self) -> bool:
        return bool(self.track_kinds)

    def __repr__(self) -> str:
        return (f"GVL dataset (B200-resident) with shape {self.shape}: sequences={self.sequence_type!r}, tracks={list(self.active_tracks)}, "
                f"output_length={self.output_length!r}, jitter={self.jitter} (max {self.max_jitter}), deterministic={self.deterministic}, "
                f"rc_neg={self.rc_neg}, is_subset={self.is_subset}, is_spliced={self.is_spliced}, track_dtype={self.track_dtype}")

    def _shape_counts(self, x: np.ndarray, squeeze: bool, out_reshape):
        if squeeze:
            x = x.squeeze(0)
        if out_reshape is not None:
            x = x.reshape(*out_reshape, x.shape[-1])
        return x

    def _counts(self, regions, samples, per_index) -> np.ndarray:
        """Counts of the selected (region, sample) pairs shaped like `ds[regions, samples]`: `per_index(ds_idx)` gives int32
        (n, k) per dataset index.  A spliced (splice row, sample) sums the counts of its elements."""
        idx = (slice(None) if regions is None else regions, slice(None) if samples is None else samples)
        if self.splice_rows is None:
            ds_idx, squeeze, out_reshape = self._parse_idx(idx)
            return self._shape_counts(per_index(ds_idx), squeeze, out_reshape)
        _, ds_idx_e, _, e_first, outer, squeeze = self._spliced_batch(idx)
        n = per_index(ds_idx_e)
        x = np.add.reduceat(n, e_first[:-1], axis=0).astype(np.int32).reshape(*outer, n.shape[1])
        return x.reshape(n.shape[1]) if squeeze else x

    def n_variants(self, regions=None, samples=None) -> np.ndarray:
        """`Dataset.n_variants`, _impl.py:1293-1340: variants per (region, sample, ploid) -> int32 (..., ploidy).  Spliced:
        per (splice row, sample, ploid), the sum over the row's elements."""
        if self.engine.svar2 is not None:
            raise NotImplementedError("n_variants of an svar2-backed dataset needs the presence-bit popcounts (not kept on the host)")
        p, go = self.ploidy, self.engine.geno_offsets_host

        def per_index(ds_idx):
            goi = ds_idx[:, None] * p + np.arange(p, dtype=np.int64)[None, :]
            return np.maximum(go[1, goi] - go[0, goi], 0).astype(np.int32)

        return self._counts(regions, samples, per_index)

    def n_intervals(self, regions=None, samples=None) -> np.ndarray:
        """`Dataset.n_intervals`, _impl.py:1848-1895: stored intervals per (region, sample) and ACTIVE track -> int32 (..., tracks).
        Spliced: per (splice row, sample, track), the sum over the row's elements (annotation tracks read the element's slot)."""
        offs = []
        for name in self.active_tracks:
            off = self._cache.get(("itv_off", name))
            if off is None:
                off = self._cache[("itv_off", name)] = self.engine.tracks[name][3].cpu().numpy()
            offs.append((off, self.track_kinds[name] == "annot"))

        def per_index(ds_idx):
            r_idx = ds_idx // len(self.sample_names)
            cols = []
            for off, annot in offs:
                slot = r_idx if annot else ds_idx
                cols.append((off[slot + 1] - off[slot]).astype(np.int32))
            return np.stack(cols, -1) if cols else np.zeros((len(ds_idx), 0), np.int32)

        return self._counts(regions, samples, per_index)

    def haplotype_lengths(self, regions=None, samples=None):
        """`Dataset.haplotype_lengths`, _impl.py:1234-1291: lengths of the JITTER-EXTENDED haplotypes -> int32 (..., ploidy);
        None when the lengths are not a fixed property of the dataset (no genotypes, random shifts)."""
        if self.splice_rows is not None:
            raise NotImplementedError("Haplotype lengths are not yet implemented for spliced datasets.")
        if not self.has_genotypes or not self.deterministic:
            return None
        ds_idx, squeeze, out_reshape = self._parse_idx((slice(None) if regions is None else regions,
                                                        slice(None) if samples is None else samples))
        eng, dev, p = self.engine, self.engine.device, self.ploidy
        reg = self.full_regions[ds_idx // len(self.sample_names)].copy()
        reg[:, 1] -= self.jitter
        reg[:, 2] += self.jitter
        goi = ds_idx[:, None] * p + np.arange(p, dtype=np.int64)[None, :]
        t_reg = torch.from_numpy(np.ascontiguousarray(reg[:, :3])).to(dev)
        t_goi = torch.from_numpy(goi).to(dev)
        keep = keep_off = None
        if self.var_filter == "exonic":
            keep, keep_off = self._exonic_keep(t_goi, t_reg, goi)
        d = eng.get_diffs(t_goi, t_reg[:, 1].contiguous(), t_reg[:, 2].contiguous(), keep, keep_off, regions=t_reg,
                          max_records=eng.max_records(goi)).cpu().numpy()
        lens = ((reg[:, 2] - reg[:, 1])[:, None] + d).astype(np.int32)
        return self._shape_counts(lens, squeeze, out_reshape)

    def to_torch_dataset(self, return_indices: bool = False, transform=None):
        """`Dataset.to_torch_dataset`, _impl.py:1940-1961 -> `TorchDataset`, _torch.py:272-307: a map-style dataset over the flat
        (region, sample) index; an int or a list of ints selects a batch (the batches are CUDA tensors)."""
        return _MapDataset(self, bool(return_indices), transform)

    @property
    def regions(self) -> np.ndarray:
        return self.full_regions[self._r_idx]

    def __len__(self) -> int:
        return self.n_regions * self.n_samples

    @property
    def _r_idx(self) -> np.ndarray:
        v = self._cache.get("r_idx")
        if v is None:
            if self.region_subset is not None:
                v = self.region_subset
            else:
                v = np.arange(len(self.full_regions)) if self.region_map is None else self.region_map
            v = self._cache["r_idx"] = np.ascontiguousarray(v, np.int64)
        return v

    @property
    def _s_idx(self) -> np.ndarray:
        v = self._cache.get("s_idx")
        if v is None:
            v = np.arange(len(self.sample_names)) if self.sample_subset is None else self.sample_subset
            v = self._cache["s_idx"] = np.ascontiguousarray(v, np.int64)
        return v

    # ------------------------------------------------------------------ with_* (immutable evolution)
    def _check_valid_state(self) -> None:
        """Same checks and messages as the reference's `_check_valid_state` (_impl.py:501-568) for this scope."""
        if self.jitter < 0:
            raise ValueError(f"Jitter ({self.jitter}) must be a non-negative integer.")
        if self.jitter > self.max_jitter:
            raise ValueError(f"Jitter ({self.jitter}) must be less than or equal to the maximum jitter of the dataset ({self.max_jitter}).")
        if isinstance(self.output_length, (int, np.integer)) and not isinstance(self.output_length, bool):
            if self.output_length < 1:
                raise ValueError(f"Output length ({self.output_length}) must be a positive integer.")
            min_r_len = int((self.full_regions[:, 2] - self.full_regions[:, 1]).min())
            max_output_length = min_r_len + 2 * self.max_jitter
            eff_length = int(self.output_length) + 2 * self.jitter
            if eff_length > max_output_length:
                raise ValueError(
                    f"Effective length (out_len={self.output_length}) + 2 * ({self.jitter=}) = {eff_length} must be less"
                    f" than or equal to the maximum output length of the dataset ({max_output_length})."
                    f" The maximum output length is the minimum region length ({min_r_len}) + 2 * (max_jitter={self.max_jitter}).")
        elif self.output_length not in ("ragged", "variable"):
            raise ValueError(f"Output length must be 'ragged', 'variable' or a positive integer, got {self.output_length!r}")
        if self.unphased_union and self.sequence_type in ("haplotypes", "annotated"):
            raise ValueError("unphased_union is incompatible with 'haplotypes'/'annotated' output (a union of phased sequences is "
                             "ill-defined). Use 'variant-windows' or 'variants', or clear the flag with "
                             "with_settings(unphased_union=False).")  # _impl.py:769-779
        if (self.min_af is not None or self.max_af is not None) and self.sequence_type not in ("variants", "variant-windows"):
            raise NotImplementedError("Filtering by AF is not supported for haplotype output yet.")  # _haps.py:695-698
        if self.track_output == "intervals" and self._realigns:
            raise ValueError("kind='intervals' returns the stored intervals, which are not realigned to haplotypes: set "
                             "with_settings(realign_tracks=False), or use with_seqs('reference') or with_seqs(None).")
        if self.encoding != "bytes" and self.sequence_type not in ("haplotypes", "reference"):
            raise ValueError("one-hot encoding applies to 'haplotypes' / 'reference' sequences only")
        if self.encoding == "onehot_cf":
            if not isinstance(self.output_length, (int, np.integer)):
                raise ValueError("channels-first one-hot needs a fixed output length")
            if int(self.output_length) % 4:
                raise ValueError("channels-first one-hot needs an output length that is a multiple of 4")

    def _evolve(self, **kw) -> "Dataset":
        ds = replace(self, **kw, _cache={})
        ds._check_valid_state()
        return ds

    def with_settings(self, jitter=None, rng=None, deterministic=None, rc_neg=None, var_filter=None, realign_tracks=None,
                      min_af=None, max_af=None, splice_info=None, **unsupported) -> "Dataset":
        """Reference: `Dataset.with_settings`, _impl.py:228-499 (hot-path settings only)."""
        kw = {}
        if min_af is not None:
            kw["min_af"] = None if min_af is False else float(min_af)
        if max_af is not None:
            kw["max_af"] = None if max_af is False else float(max_af)
        ta, ut = unsupported.pop("token_alphabet", None), unsupported.pop("unknown_token", None)
        if ta is not None or ut is not None:  # _impl.py:432-441
            if ta is None or ut is None:
                raise ValueError("token_alphabet and unknown_token must be set together.")
            kw["token_alphabet"] = ta.encode("ascii") if isinstance(ta, str) else bytes(ta)
            kw["unknown_token"] = int(ut)
        fl = unsupported.pop("flank_length", None)
        if fl is not None:
            if fl is not False and kw.get("token_alphabet", self.token_alphabet) is None:
                raise ValueError("flank_length requires a token LUT; pass token_alphabet and unknown_token to with_settings(...)"
                                 " (in this or a prior call).")  # _impl.py:442-446
            kw["flank_length"] = 0 if fl is False else int(fl)
        for name in ("var_fields", "dummy_variant", "unphased_union"):
            if name in unsupported:
                v = unsupported.pop(name)
                if v is None:
                    continue
                if name == "var_fields":
                    avail = self.available_var_fields
                    missing = sorted(set(v) - set(avail))
                    if missing:
                        raise ValueError(f"Missing variant fields: {missing}")  # _impl.py:343-346
                    v = tuple(v)
                elif name == "dummy_variant":
                    v = None if v is False else v
                else:
                    v = bool(v)
                kw[name] = v
        if splice_info is False:
            kw["splice_rows"], kw["splice_names"] = None, None
        elif splice_info is not None:
            kw["splice_rows"], kw["splice_names"] = self._build_splice_rows(splice_info)
        if unsupported:
            raise NotImplementedError(f"settings outside the hot-path scope: {sorted(unsupported)}")
        if jitter is not None:
            kw["jitter"] = int(jitter)
        if rng is not None:
            kw["rng"] = np.random.default_rng(rng)
        if deterministic is not None:
            kw["deterministic"] = bool(deterministic)
        if rc_neg is not None:
            kw["rc_neg"] = bool(rc_neg)
        if var_filter not in (None, False) and self.engine.svar2 is not None:
            raise NotImplementedError("var_filter is not supported with the svar2 source")
        if var_filter is not None:
            if var_filter not in (False, "exonic"):
                raise ValueError(f"var_filter must be False or 'exonic', got {var_filter!r}")
            kw["var_filter"] = None if var_filter is False else "exonic"
        if realign_tracks is not None:
            kw["realign_tracks"] = bool(realign_tracks)
        return self._evolve(**kw)

    def with_len(self, output_length) -> "Dataset":
        """Reference: `Dataset.with_len`, _impl.py:570-647."""
        if isinstance(output_length, (int, np.integer)) and not isinstance(output_length, bool):
            if output_length < 1:
                raise ValueError(f"Output length ({output_length}) must be a positive integer.")
            output_length = int(output_length)
        return self._evolve(output_length=output_length)

    def with_seqs(self, kind, window_opt=None) -> "Dataset":
        """Reference: `Dataset.with_seqs`, _impl.py:649-783."""
        if kind in ("variants", "variant-windows") and getattr(self.engine, "svar2", None) is not None:
            raise NotImplementedError(f"with_seqs({kind!r}) needs the SVAR1 genotype CSR (the svar2 source decodes variants "
                                      "through its store)")
        if kind not in (None, "reference", "haplotypes", "annotated", "variants", "variant-windows"):
            raise ValueError(f"Unknown sequence type {kind!r}")
        kw = {}
        if kind == "variant-windows":
            if not isinstance(window_opt, VarWindowOpt):
                raise ValueError("with_seqs('variant-windows') requires window_opt=VarWindowOpt(...)")  # _impl.py:741-747
            kw["window_opt"] = window_opt
        elif window_opt is not None:
            raise ValueError("window_opt only applies to with_seqs('variant-windows')")
        enc = self.encoding if kind in ("haplotypes", "reference") else "bytes"
        return self._evolve(sequence_type=kind, encoding=enc, **kw)

    def with_encoding(self, encoding: str) -> "Dataset":
        """Fused one-hot output (this build's extension; the reference leaves one-hot to `seqpro.DNA.ohe`,
        docs/source/index.md:108-119).  "onehot": uint8 (..., L, 4); "onehot_cf": uint8 (..., 4, L); alphabet ACGT."""
        if encoding not in ("bytes", "onehot", "onehot_cf"):
            raise ValueError(f"Unknown encoding {encoding!r}")
        return self._evolve(encoding=encoding)

    def with_track_dtype(self, dtype) -> "Dataset":
        """Element type of the track outputs (this build's extension, like `with_encoding`): `torch.float32` (the default),
        `torch.bfloat16` or `torch.float16`.  Values are computed in float32 as always and rounded to nearest even by the
        track kernels' stores, so every read returns bit for bit `x.to(dtype)` of its float32 output `x` cast on the device
        (float16 overflows to +-inf, subnormals are kept, NaN is the device's canonical NaN) -- without a second pass over
        the batch, and with half the bytes written.  Shapes, offsets, padding and fills do not change."""
        if not self.track_kinds:
            raise ValueError("Dataset has no tracks; cannot set a track dtype.")
        track_dtype_code(dtype)
        return self._evolve(track_dtype=dtype)

    def with_tracks(self, tracks=None, kind=None) -> "Dataset":
        """Reference: `Dataset.with_tracks`, _impl.py:785-839.  `False`/`[]` disables tracks.  `kind`: None keeps the
        current output kind; "tracks" returns base-pair values (painted or realigned), "intervals" the stored intervals
        that overlap each read's window, clipped to it (`RaggedIntervals`, one cell per (..., track); DESIGN.md §7).
        Intervals are not realigned: with haplotypes, set `with_settings(realign_tracks=False)` first."""
        if kind not in (None, "tracks", "intervals"):
            raise ValueError(f"Unknown track kind {kind!r}: 'tracks' or 'intervals'")
        if tracks is None:
            names = tuple(self.track_kinds)
        elif tracks is False:
            names = ()
        else:
            names = (tracks,) if isinstance(tracks, str) else tuple(tracks)
        missing = [t for t in names if t not in self.track_kinds]
        if missing:
            raise ValueError(f"Track(s) {missing} not found. Available tracks: {self.available_tracks}")
        return self._evolve(active_tracks=names, track_output=self.track_output if kind is None else kind)

    def with_insertion_fill(self, strategy) -> "Dataset":
        """Reference: `Dataset.with_insertion_fill`, _impl.py:841-878 (one strategy for all tracks or a dict)."""
        if not self.track_kinds:
            raise ValueError("Dataset has no tracks; cannot configure insertion fill.")
        if self.track_output == "intervals":
            raise ValueError("with_insertion_fill has no effect on kind='intervals' (intervals are not realigned); use "
                             "with_tracks(kind='tracks') first.")
        if self.sequence_type not in ("haplotypes", "annotated"):
            raise ValueError("with_insertion_fill is only meaningful for datasets with both haplotypes and tracks "
                             "(use with_seqs to activate haplotypes first).")
        if not self.active_tracks:
            raise ValueError("with_insertion_fill is only meaningful when tracks are active (use with_tracks to activate tracks first).")
        if not self.realign_tracks:
            raise ValueError("with_insertion_fill has no effect when realign_tracks=False (insertion fill only applies during "
                             "track re-alignment). Set with_settings(realign_tracks=True) first, or drop the call.")
        if isinstance(strategy, InsertionFill):
            fills = {name: strategy for name in self.track_kinds}
        else:
            fills = dict(self.insertion_fill)
            for name, s in dict(strategy).items():
                if name not in self.track_kinds:
                    raise ValueError(f"Track {name!r} not found. Available tracks: {self.available_tracks}")
                if not isinstance(s, InsertionFill):
                    raise TypeError("strategies must be InsertionFill instances")
                fills[name] = s
        return self._evolve(insertion_fill=fills)

    def with_output_format(self, fmt: str) -> "Dataset":
        """Reference: `Dataset.with_output_format`, _impl.py:880-952.  "flat" returns `Ragged` triples untouched."""
        if fmt not in ("ragged", "flat"):
            raise ValueError(f"Unknown output format {fmt!r}")
        return self._evolve(output_format=fmt)

    def subset_to(self, regions=None, samples=None) -> "Dataset":
        """Reference: `Dataset.subset_to`, _impl.py:1153-1221 (integer / slice / boolean / sample-name selectors)."""
        kw = {}
        if regions is not None:
            if self.splice_rows is not None:
                raise ValueError("subset_to(regions=...) on a spliced dataset would mix splice rows with regions: subset first, "
                                 "then with_settings(splice_info=...)")
            kw["region_subset"] = self._r_idx[_idx_to_array(regions, self.n_regions)]
        if samples is not None:
            if isinstance(samples, str) or (np.ndim(samples) > 0 and len(samples) and isinstance(samples[0], str)):
                names = [samples] if isinstance(samples, str) else list(samples)
                lut = {n: i for i, n in enumerate(self.sample_names)}
                try:
                    kw["sample_subset"] = np.array([lut[n] for n in names], np.int64)
                except KeyError as e:
                    raise KeyError(f"Sample {e.args[0]!r} not found") from None
            else:
                kw["sample_subset"] = self._s_idx[_idx_to_array(samples, self.n_samples)]
        return self._evolve(**kw)

    def to_full_dataset(self) -> "Dataset":
        return self._evolve(region_subset=None, sample_subset=None)

    # ------------------------------------------------------------------ indexing
    def _parse_idx(self, idx):
        """`DatasetIndexer.parse_idx`, _indexing.py:208-264: flat dataset indices (row-major over the FULL
        (regions, samples) grid), squeeze flag, optional outer reshape -- "basic" (ints / slices), "adv" (two
        arrays, paired) and "combo" (one array, one basic -> outer product) indexing."""
        if not isinstance(idx, tuple):
            r, s = idx, slice(None)
        elif len(idx) == 1:
            r, s = idx[0], slice(None)
        elif len(idx) == 2:
            r, s = idx
        else:
            raise IndexError("a Dataset is indexed by (regions, samples)")
        if (type(r) is np.ndarray and type(s) is np.ndarray and r.ndim == 1 and s.shape == r.shape
                and r.dtype.kind in "iu" and s.dtype.kind in "iu"):
            # the loader's case, two paired 1-D integer arrays: fancy indexing does the bounds check, the negative wrap
            # and the subset mapping in one step each
            flat = self._r_idx[r] * len(self.sample_names) + self._s_idx[s]
            return (flat if flat.dtype == np.int64 else flat.astype(np.int64)), False, None
        is_basic = lambda x: isinstance(x, (int, np.integer, slice))
        is_int = lambda x: isinstance(x, (int, np.integer))
        n_s = len(self.sample_names)
        r_raw = self._r_idx[_idx_to_array(r, self.n_regions)]
        s_raw = self._s_idx[_idx_to_array(s, self.n_samples)]
        squeeze, out_reshape = False, None
        if is_basic(r) and is_basic(s):
            squeeze = is_int(r) and is_int(s)
            ri, si = np.atleast_1d(r_raw), np.atleast_1d(s_raw)
            flat = (ri[:, None] * n_s + si[None, :]).squeeze()
            if isinstance(r, slice) and isinstance(s, slice):
                out_reshape = (len(ri), len(si))
            if flat.ndim > 1:
                out_reshape = flat.shape
        elif not is_basic(r) and not is_basic(s):
            ri, si = np.broadcast_arrays(r_raw, s_raw)
            flat = ri * n_s + si
            if flat.ndim > 1:
                out_reshape = flat.shape
        else:
            flat = r_raw.ravel()[:, None] * n_s + s_raw.ravel()[None, :]
            if r_raw.ndim > 1 or s_raw.ndim > 1:
                out_reshape = (*r_raw.shape, *s_raw.shape)
            else:
                out_reshape = flat.shape
        return np.asarray(flat, np.int64).ravel(), squeeze, out_reshape

    # ------------------------------------------------------------------ splicing (reference: _splice.py, _query.py:206-330)
    def _build_splice_rows(self, splice_info):
        """Splice rows = ordered lists of regions (e.g. the exons of a transcript) whose haplotypes are concatenated.

        `splice_info` follows the reference (`SpliceMap.from_bed`, _splice.py:163-230) for datasets opened from disk:
        a column name of the input BED (rows with the same value form a splice row, in BED order) or a
        `(id_column, order_column)` pair (elements sorted by the second column).  In-memory datasets -- and any
        dataset -- may pass the mapping directly: `{name: [region indices]}` or a sequence of index sequences
        (indices address regions like `ds[r, s]` does)."""
        r_map = self._r_idx
        names = None
        by_column = isinstance(splice_info, str) or (isinstance(splice_info, tuple) and len(splice_info) == 2
                                                     and all(isinstance(x, str) for x in splice_info))
        if by_column:
            cols = self.bed_columns or {}
            id_col, order_col = (splice_info, None) if isinstance(splice_info, str) else splice_info
            for c in (id_col, order_col):
                if c is not None and c not in cols:
                    raise ValueError(f"column {c!r} is not in the dataset's input BED (available: {sorted(cols)})")
            ids = np.asarray(cols[id_col])
            groups: dict = {}
            for i, v in enumerate(ids.tolist()):
                groups.setdefault(v, []).append(i)
            if order_col is not None:
                order = np.asarray(cols[order_col])
                groups = {k: sorted(v, key=lambda i: order[i]) for k, v in groups.items()}
            # BED columns are in INPUT order: rows map to storage through region_map (not through a subset); with a region
            # subset active, elements outside it drop out and rows left empty disappear
            full_map = self.region_map if self.region_map is not None else np.arange(len(self.full_regions), dtype=np.int64)
            allowed = None if self.region_subset is None else set(np.asarray(self.region_subset).tolist())
            names, rows = [], []
            for k, v in groups.items():
                st = [int(full_map[i]) for i in v]
                if allowed is not None:
                    st = [x for x in st if x in allowed]
                if st:
                    names.append(k)
                    rows.append(np.asarray(st, np.int64))
            if not rows:
                raise ValueError("no splice row is left after subsetting")
            return tuple(rows), tuple(names)
        elif isinstance(splice_info, dict):
            names, lists = list(splice_info), list(splice_info.values())
        else:
            lists = list(splice_info)
        rows = []
        for l in lists:
            a = _idx_to_array(np.asarray(l, np.int64), len(r_map))
            if a.ndim != 1 or a.size == 0:
                raise ValueError("every splice row needs at least one region index")
            rows.append(np.ascontiguousarray(r_map[a], np.int64))
        return tuple(rows), (tuple(names) if names is not None else None)

    @property
    def is_spliced(self) -> bool:
        return self.splice_rows is not None

    def _spliced_batch(self, idx):
        """The element batch E of a spliced selection `idx` (the index forms of `ds[...]`): every (element region, sample)
        of the selected (splice row, sample) pairs, pairs in output order and a pair's elements in splice-row order ->
        (e_reg, ds_idx_e, n_el, e_first, outer, squeeze).  Two paired arrays select pairs, `outer = (pairs,)`; any other
        form selects the outer product, `outer = (rows, samples)`, squeezed away by an int/int index."""
        if not isinstance(idx, tuple):
            idx = (idx, slice(None))
        r_sel, s_sel = idx
        rows_all = self.splice_rows
        ri = np.atleast_1d(_idx_to_array(r_sel, len(rows_all)))
        si = np.atleast_1d(self._s_idx[_idx_to_array(s_sel, len(self._s_idx))])
        is_int = lambda x: isinstance(x, (int, np.integer))
        is_basic = lambda x: isinstance(x, (int, np.integer, slice))
        if not is_basic(r_sel) and not is_basic(s_sel):  # paired
            ri, si = (a.ravel() for a in np.broadcast_arrays(ri, si))
            outer = (ri.size,)
        else:
            outer = (ri.size, si.size)
            ri, si = np.repeat(ri.ravel(), si.size), np.tile(si.ravel(), ri.size)
        elems = [rows_all[r] for r in ri.tolist()]
        n_el = np.array([len(e) for e in elems], np.int64)                # K_c
        e_first = np.concatenate([[0], np.cumsum(n_el)]).astype(np.int64)  # first element of pair c in E
        e_reg = np.concatenate(elems).astype(np.int64)
        ds_idx_e = e_reg * len(self.sample_names) + np.repeat(si, n_el)
        return e_reg, ds_idx_e, n_el, e_first, outer, is_int(r_sel) and is_int(s_sel)

    def _getitem_spliced(self, idx):
        """One ragged sequence per (splice row, sample[, ploid]) and, with tracks active, one ragged track per (splice row,
        sample, track[, ploid]): a spliced cell is the concatenation, in splice-row order, of its elements' unspliced
        outputs (jitter 0, ragged length).

        Sequences: the row's elements are reconstructed as separate kernel rows, laid out in (row, sample, ploid, element)
        order (the reference's permuted write, _splice.py:56-160 / _haps.py:872-919), so the concatenation is free and the
        group offsets are the kernel's row offsets sampled at cell boundaries.  Negative-strand elements are
        reverse-complemented one by one (_query.py:269-288).  "reference" sequences are the zero-variant case (no ploidy axis).

        Tracks: the element batch E lists every (element region, sample) of the selected pairs in output order.  One track
        call covers all of E and all active tracks -- realigned to the element haplotypes (rows (e, ploid)) or painted over
        the element regions (rows e) -- and writes every row straight into its place in the concatenated output through a
        per-row destination table (gvl_dev_realign_tracks_plan_rows / gvl_dev_paint_tracks_rows).  The values are those of
        one unspliced call over E: the same fill seed (of E's dataset indices), FlankSample rows and track lengths.

        Variants: the genotype rows of E are gathered in cell order -- (pair, ploid, element), or (pair, element, ploid)
        under `unphased_union` so that the p rows folded into one belong to one element -- with every element's own strand
        and contig, so each element row is its unspliced variants row (AF filter, dummy variant, strand, tokens) and a cell
        is a contiguous run of rows: its offsets are the gathered row offsets sampled at cell boundaries."""
        if self.jitter or isinstance(self.output_length, (int, np.integer)):
            raise ValueError("spliced datasets return ragged haplotypes: use with_len('ragged') and jitter=0")
        seq = self.sequence_type
        if seq is not None and self.encoding == "onehot_cf":
            raise ValueError("channels-first one-hot needs a fixed output length; spliced output is ragged")
        e_reg, ds_idx_e, n_el, e_first, outer, squeeze = self._spliced_batch(idx)
        eng, dev, p = self.engine, self.engine.device, self.ploidy
        is_ref = seq == "reference"
        is_var = seq in ("variants", "variant-windows")
        fold = is_var and self.unphased_union
        rows_p = 1 if is_ref else p  # sequence rows per element
        t = len(self.active_tracks)
        realign = self._realigns

        # ---- the element batch E: (pair, element) in output order
        n_pairs = n_el.size
        e_pair = np.repeat(np.arange(n_pairs, dtype=np.int64), n_el)
        e_k = np.arange(e_reg.size, dtype=np.int64) - e_first[e_pair]
        regions = self.full_regions[e_reg]
        to_rc_e = (regions[:, 3] == -1) if self.rc_neg else None
        e_len = (regions[:, 2] - regions[:, 1]).astype(np.int64)
        n_e = e_reg.size

        # sequence row of (e, h): pair c holds rows rows_p * e_first[c] ..., ploid-major, element-minor
        q = ((rows_p * e_first[e_pair])[:, None] + np.arange(rows_p, dtype=np.int64)[None, :] * n_el[e_pair][:, None]
             + e_k[:, None])
        goi_e = ds_idx_e[:, None] * p + np.arange(p, dtype=np.int64)[None, :]
        pk = _Packer(dev)
        if seq is not None:
            if fold:  # variant rows (pair, element, ploid), folded to one per element: cell c = elements of pair c
                inv = np.repeat(np.arange(n_e, dtype=np.int64), p)
                s_goi = goi_e.reshape(-1, 1)
                cell_starts = e_first
            else:
                inv = np.empty(n_e * rows_p, np.int64)  # element of every sequence row
                inv[q.ravel()] = np.repeat(np.arange(n_e, dtype=np.int64), rows_p)
                if is_ref:
                    s_goi = np.full((n_e, 1), eng.empty_slot, np.int64)
                else:
                    s_goi = np.empty((n_e * p, 1), np.int64)
                    s_goi[q.ravel(), 0] = goi_e.ravel()
                cell_starts = (rows_p * e_first[:-1, None] + np.arange(rows_p, dtype=np.int64)[None, :] * n_el[:, None]).ravel()
                cell_starts = np.append(cell_starts, rows_p * e_first[-1])
            i_sgoi = pk.add(s_goi, np.int64)
            i_src = pk.add(to_rc_e[inv], np.uint8) if to_rc_e is not None else None
            i_cs = pk.add(cell_starts, np.int64)
            if not is_var:
                i_sreg = pk.add(regions[inv, :3], np.int32)
                i_ssh = pk.add(np.zeros((len(s_goi), 1), np.int32), np.int32)
        if t:
            oi = np.stack([ds_idx_e if self.track_kinds[n] == "sample" else e_reg for n in self.active_tracks])
            i_oi = pk.add(oi, np.int64)
            if realign:
                i_reg = pk.add(regions[:, :3], np.int32)
                i_len = pk.add(e_len, np.int64)
                i_goi_e = pk.add(goi_e, np.int64)
                i_sh_e = pk.add(np.zeros((n_e, p), np.int32), np.int32)
                i_rc_e = pk.add(np.repeat(to_rc_e, p), np.uint8) if to_rc_e is not None else None
                i_q = pk.add(q, np.int64)
                i_pf = pk.add(rows_p * e_first[e_pair], np.int64)       # first sequence row of the element's pair
                i_pn = pk.add(rows_p * e_first[e_pair + 1], np.int64)   # ... and of the next pair
            elif self.track_output == "intervals":
                # rows (pair, track, element), each element over its own region: cell (pair, track) is a run of rows
                tt = np.arange(t, dtype=np.int64)
                row_of = (t * e_first[e_pair])[:, None] + tt[None, :] * n_el[e_pair][:, None] + e_k[:, None]
                slot, tw = _interval_rows(oi, regions[:, 1], regions[:, 2], row_of)
                i_islot, i_itw = pk.add(slot, np.int64), pk.add(tw, np.int32)
                i_icells = pk.add(np.append((t * e_first[:-1, None] + tt[None, :] * n_el[:, None]).ravel(), t * e_first[-1]),
                                  np.int64)
            else:
                # painted: lengths are the element region lengths, known here -- the whole table is built on the host
                off_e = np.concatenate([[0], np.cumsum(e_len)]).astype(np.int64)
                base_c = off_e[e_first]                                   # B_c (and the end of E at [n_pairs])
                len_c = base_c[1:] - base_c[:-1]                          # L_c
                i_off_e = pk.add(off_e, np.int64)
                i_dst = pk.add(t * base_c[e_pair] + (off_e[:-1] - base_c[e_pair]), np.int64)
                i_ts = pk.add(len_c[e_pair], np.int64)
                i_rc_q = pk.add(to_rc_e, np.uint8) if to_rc_e is not None else None
                i_st = pk.add(regions[:, 1], np.int32)
                i_toff = pk.add(np.concatenate([[0], np.cumsum(np.repeat(len_c, t))]), np.int64)
        pk.upload()

        results = []
        max_rec = 0 if is_ref else eng.max_records(goi_e)
        oo = group_offsets = total = None
        if is_var:
            results.append(self._get_variants(pk.get(i_sgoi), pk.get(i_src) if i_src is not None else None, regions[inv, 0],
                                              max_rec, (*outer, 1 if fold else p, None), cells=pk.get(i_cs)))
        elif seq is not None:
            keep = keep_off = None
            if self.var_filter == "exonic" and not is_ref:
                keep, keep_off = self._exonic_keep(pk.get(i_sgoi), pk.get(i_sreg), s_goi)
            oo, total, diffs = self._plan_seqs(pk.get(i_sreg), pk.get(i_ssh), pk.get(i_sgoi), -1, max_rec, keep, keep_off,
                                               pk.get(i_src) if i_src is not None else None)
            group_offsets = oo[pk.get(i_cs)]
            results.append(self._execute_seqs(group_offsets, (*outer, None) if is_ref else (*outer, p, None), total))
        if t and realign:
            # rows (e, h) of E; their haplotypes are sequence rows q[e, h] of the plan above
            t_q = pk.get(i_q)
            row_len = (oo[1:] - oo[:-1])[t_q].reshape(-1)
            out_offsets = torch.zeros(n_e * p + 1, dtype=torch.int64, device=dev)
            torch.cumsum(row_len, 0, out=out_offsets[1:])
            base = oo[pk.get(i_pf)][:, None]  # B_c of the element's pair: cell (c, track, h) starts at t * B_c + ...
            row_dst = (t * base + oo[t_q] - base).reshape(-1)
            row_tstride = (oo[pk.get(i_pn)] - base[:, 0]).repeat_interleave(p)  # (a materialised copy: the kernel reads it by index)
            keep = keep_off = None
            if self.var_filter == "exonic":
                keep, keep_off = self._exonic_keep(pk.get(i_goi_e), pk.get(i_reg), goi_e)
            results.append(self._realigned_tracks(
                ds_idx_e, pk.get(i_reg), pk.get(i_sh_e), pk.get(i_goi_e), pk.get(i_oi), pk.get(i_len), diffs.view(-1)[t_q],
                out_offsets, total, max_rec, keep, keep_off, pk.get(i_rc_e) if i_rc_e is not None else None, group_offsets,
                (*outer, t, p, None), row_dst=row_dst, row_tstride=row_tstride))
        elif t and self.track_output == "intervals":
            results.append(self._track_intervals(pk.get(i_islot), pk.get(i_itw), (*outer, t, None), cells=pk.get(i_icells)))
        elif t:
            results.append(self._painted_tracks(pk.get(i_oi), pk.get(i_st), pk.get(i_off_e), int(off_e[-1]),
                                                pk.get(i_rc_q) if i_rc_q is not None else None, pk.get(i_toff),
                                                (*outer, t, None), row_dst=pk.get(i_dst), row_tstride=pk.get(i_ts)))
        if self.output_length == "variable" and self.output_format != "flat":  # pad like the unspliced path (_query.py:94-127)
            results = [self._shape_output(o, None, False) for o in results]
        if squeeze:
            results = [o.squeeze(0).squeeze(0) for o in results]
        return results[0] if len(results) == 1 else tuple(results)

    # ------------------------------------------------------------------ iteration (reference: to_dataloader, _impl.py:1963-2072)
    def to_dataloader(self, batch_size: int = 1, shuffle: bool = False, sampler=None, num_workers: int = 0, collate_fn=None,
                      pin_memory: bool = False, drop_last: bool = False, generator=None, *, return_indices: bool = False,
                      transform=None, mode=None, copy: bool = True, ring: int = 0, to_host: bool = False, **ignored):
        """Batches over the flat `(region, sample)` index like the reference's DataLoader (which wraps its sampler in a
        `BatchSampler` so that the dataset is indexed with lists of indices, _torch.py:160-228).  The batches are born on
        the GPU, so there are no workers, no pinning and no collation: `num_workers`, `pin_memory`, `collate_fn`,
        `buffer_bytes` ... are accepted and ignored.  `generator`: seed / numpy Generator / torch.Generator for `shuffle`.

        `mode=None`: one synchronous `ds[r, s]` per batch (any output kind).
        `mode="buffered"` / `"double_buffered"` (reference: `_impl.py:2029-2046`, prefetching producers): the GPU-side
        analogue for fixed-length output -- the loader reads `ring` batches ahead with ONE device call per ring (0: sized
        for ~256 MiB of output), two ring halves produced alternately while the other is consumed (`_pipeline.py`).  `copy=False` hands out zero-copy
        views into the ring that stay valid until `ring` more batches have been drawn (the reference's `copy=False`
        contract: "only valid until the next batch is yielded"); `copy=True` (default) clones every batch.
        `to_host=True` (pipelined modes): batches are delivered as NUMPY arrays in pinned host memory -- every ring is copied
        device-to-host on a copy stream while the next one is produced, so a CPU consumer sees the PCIe copy rate instead of
        copy + compute + launch latency per batch (`copy=False`: views valid until the half comes around again).  float16
        tracks arrive as numpy float16; bfloat16 tracks raise ValueError (numpy has no bfloat16).
        `variants` / `variant-windows` (unspliced, no tracks, no var_filter, on the device): the same modes read `ring`
        batches per device call (`_variants_loader.py`): one sizing pass over the ring's genotype rows and one wait, then
        one variants tail over all of them, every batch a RaggedVariants with its own offsets starting at 0.  `ring=0`
        targets about 2**20 variants per ring, estimated from the dataset's mean variants per genotype row (1 to 64 batches).
        Rings alternate between two streams, so one is produced while the other is read; every ring gets fresh buffers, so
        `copy=False` views stay valid for as long as they are held (at least until `ring` more batches have been drawn).
        Other datasets the pipelines cannot serve (ragged / variable-length haplotypes, random shifts, splicing, var_filter,
        track intervals) fall back to `mode=None`."""
        if sampler is not None and shuffle:
            raise ValueError("sampler option is mutually exclusive with shuffle")
        if mode not in (None, "buffered", "double_buffered"):
            raise ValueError(f"Unknown dataloader mode {mode!r}")
        if mode is not None:
            from . import _pipeline

            if _pipeline.supports(self) is None:
                return _pipeline.PipelinedLoader(self, int(batch_size), bool(shuffle), sampler, bool(drop_last), generator,
                                                 bool(return_indices), transform, bool(copy), ring, to_host=bool(to_host))
            from . import _variants_loader

            if not to_host and _variants_loader.supports(self) is None:
                return _variants_loader.VariantsLoader(self, int(batch_size), bool(shuffle), sampler, bool(drop_last), generator,
                                                       bool(return_indices), transform, bool(copy), ring)
        return BatchLoader(self, int(batch_size), bool(shuffle), sampler, bool(drop_last), generator, bool(return_indices), transform)

    # ------------------------------------------------------------------ the hot path
    def __getitem__(self, idx):
        """Reference: `Dataset.__getitem__` _impl.py:2074-2121 -> `_query.getitem` _query.py:66-204."""
        if self.sequence_type is None and not self.active_tracks:
            raise ValueError("Dataset has neither sequences nor tracks active.")
        if self.splice_rows is not None:
            return self._getitem_spliced(idx)
        ds_idx, squeeze, out_reshape = self._parse_idx(idx)
        pipe = self._eager_pipeline(len(ds_idx))
        if pipe is not None:
            # fixed-length fast path: the O(batch) prep runs on the device (gvl_dev_batch_prep), one small H2D copy per call
            jit = self.rng.integers(-self.jitter, self.jitter + 1, size=len(ds_idx), dtype=np.int32) if self.jitter else None
            out = pipe.run_eager(ds_idx, jit)
            if out_reshape is None and not squeeze and type(out) is torch.Tensor:
                return out  # (paired array indices, sequences only: nothing to reshape)
            out = out if isinstance(out, tuple) else (out,)
            out = tuple(self._shape_output(o, out_reshape, squeeze) for o in out)
            return out[0] if len(out) == 1 else out
        S = len(self.sample_names)
        r_idx, s_idx = ds_idx // S, ds_idx % S

        # ---- _getitem_unspliced, _query.py:161-175 ----
        regions = self.full_regions[r_idx].copy()
        lengths = regions[:, 2] - regions[:, 1]
        jitter_off = self.rng.integers(-self.jitter, self.jitter + 1, size=len(regions), dtype=np.int32)
        regions[:, 1] += jitter_off
        regions[:, 2] = regions[:, 1] + lengths

        out = self._reconstruct(ds_idx, r_idx, s_idx, regions)
        out = tuple(self._shape_output(o, out_reshape, squeeze) for o in out)
        return out[0] if len(out) == 1 else out

    def _eager_pipeline(self, n: int):
        """The fixed-length pipeline serving `__getitem__` (None when this dataset state needs the general path)."""
        c = self._cache
        if "fast" not in c:
            from . import _pipeline

            c["fast"] = _pipeline.supports(self) is None
        if not c["fast"] or n == 0:
            return None
        pipe = c.get("pipe")
        if pipe is None or pipe.b < n:
            from . import _pipeline

            cap = max(n, 2 * pipe.b if pipe is not None else 0)
            pipe = c["pipe"] = _pipeline.FixedPipeline(self, cap, ring=0)
        return pipe

    # ---- reconstructors: Haps / HapsTracks / Tracks (_haps.py:578-870, _reconstruct.py:132-307, _tracks.py:370-420)
    def _reconstruct(self, ds_idx, r_idx, s_idx, regions):
        eng, dev, p = self.engine, self.engine.device, self.ploidy
        b = len(ds_idx)
        fixed = isinstance(self.output_length, (int, np.integer))
        want_seqs = self.sequence_type is not None
        want_tracks = len(self.active_tracks) > 0
        is_ref = self.sequence_type == "reference"
        to_rc_q = (self.full_regions[r_idx, 3] == -1) if self.rc_neg else None
        lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)

        # geno_offset_idx = ravel (region, sample, ploid), _haps.py:757-768.  "reference" rows use the engine's
        # empty CSR slot: the zero-variant case of the same kernels (get_reference, src/reference/mod.rs:56-120).
        rows_p = 1 if is_ref else p
        out_len_q = np.full(b, int(self.output_length), np.int64) if fixed else lengths  # painted track / interval window
        if is_ref:
            goi = np.full((b, 1), eng.empty_slot, np.int64)
        else:
            goi = ds_idx[:, None] * p + np.arange(p, dtype=np.int64)[None, :]
        to_rc = None if to_rc_q is None else np.repeat(to_rc_q, rows_p)  # _haps.py:838-843

        pk = _Packer(dev)  # one pinned staging buffer, one H2D copy for all O(batch) arrays
        i_reg = pk.add(regions[:, :3], np.int32)
        i_goi = pk.add(goi, np.int64)
        i_rc = pk.add(to_rc, np.uint8) if to_rc is not None else None
        i_sh = pk.add(np.zeros((b, rows_p), np.int32), np.int32)
        i_tr = i_trc = i_islot = i_itw = None
        if want_tracks:
            oi = np.stack([ds_idx if self.track_kinds[n] == "sample" else r_idx for n in self.active_tracks])
            if self.track_output == "intervals":  # rows (q, track)
                slot, tw = _interval_rows(oi, regions[:, 1], regions[:, 1] + out_len_q, np.arange(b * len(oi)).reshape(b, len(oi)))
                i_islot, i_itw = pk.add(slot, np.int64), pk.add(tw, np.int32)
            else:
                i_tr = pk.add(oi, np.int64)
                if to_rc_q is not None:
                    i_trc = pk.add(to_rc_q, np.uint8)
        pk.upload()
        t_reg, t_goi, t_shifts = pk.get(i_reg), pk.get(i_goi), pk.get(i_sh)
        t_rc = pk.get(i_rc) if i_rc is not None else None

        max_rec = 0 if is_ref else eng.max_records(goi)
        keep = keep_off = None
        if self.var_filter == "exonic" and not is_ref:
            keep, keep_off = self._exonic_keep(t_goi, t_reg, goi)

        results = []
        oo = total = diffs = None
        if self.sequence_type in ("variants", "variant-windows"):
            # Haps._get_variants -> get_variants_flat (_haps.py:602-609, _flat_variants.py:869-1112), on the device
            results.append(self._get_variants(t_goi, t_rc, np.repeat(regions[:, 0], p), max_rec,
                                              (b, 1 if self.unphased_union else p, None)))
            want_seqs = False
        if want_seqs:
            out_len = int(self.output_length) if fixed else -1
            if fixed and not self.deterministic and not is_ref:
                # random shifts need the diffs first (_haps.py:720-730): one extra device pass + sync; the
                # draw itself stays on the host generator so seeded runs follow the reference's RNG order
                dd = eng.get_diffs(t_goi, t_reg[:, 1].contiguous(), t_reg[:, 2].contiguous(), keep, keep_off, regions=t_reg,
                                   max_records=max_rec).cpu().numpy()
                max_shift = dd.clip(min=0) + (lengths - out_len).clip(min=0)[:, None]
                t_shifts = torch.from_numpy(self.rng.integers(0, max_shift + 1, dtype=np.int32)).to(dev)
            oo, total, diffs = self._plan_seqs(t_reg, t_shifts, t_goi, out_len, max_rec, keep, keep_off, t_rc)
            # Ref has no ploidy axis (_dataset/_ref.py)
            results.append(self._execute_seqs(oo, (b, None) if is_ref else (b, p, None), total))
        if want_tracks:
            t = len(self.active_tracks)
            if self._realigns:
                results.append(self._realigned_tracks(ds_idx, t_reg, t_shifts, t_goi, pk.get(i_tr), torch.from_numpy(lengths).to(dev),
                                                      diffs, oo, total, max_rec, keep, keep_off, t_rc, oo, (b, t, p, None)))
            elif i_islot is not None:
                results.append(self._track_intervals(pk.get(i_islot), pk.get(i_itw), (b, t, None)))
            else:
                offs = np.concatenate([[0], np.cumsum(out_len_q)]).astype(np.int64)
                d_off = torch.from_numpy(offs).to(dev)
                results.append(self._painted_tracks(pk.get(i_tr), t_reg[:, 1].contiguous(), d_off, int(offs[-1]),
                                                    pk.get(i_trc) if i_trc is not None else None, _cell_offsets(d_off, t),
                                                    (b, t, None)))
        return tuple(results)

    # ---- read steps shared by the unspliced (_reconstruct) and spliced (_getitem_spliced) reads
    @property
    def _realigns(self) -> bool:
        """Tracks are realigned to the haplotypes; otherwise their stored intervals are painted over the regions."""
        return bool(self.active_tracks) and self.sequence_type in ("haplotypes", "annotated") and self.realign_tracks

    def _fills(self, names) -> tuple:
        """(strategy ids, parameters) of the insertion fills of the tracks `names` (Repeat5p unless set)."""
        return lower([self.insertion_fill.get(n, Repeat5p()) for n in names])

    def _fill_seed(self, ds_idx) -> int:
        """Base seed of a realignment call over the dataset indices `ds_idx`."""
        if self.deterministic:
            return int(np.bitwise_xor.reduce(ds_idx.astype(np.uint64)))  # _reconstruct.py:215-218
        return int(self.rng.integers(0, np.iinfo(np.uint64).max, dtype=np.uint64))  # :219-222

    def _plan_seqs(self, t_reg, t_shifts, t_goi, out_len: int, max_rec: int, keep, keep_off, t_rc):
        """Plan one sequence row per entry of `t_goi`: (row offsets, total length, per-row diffs for realigned tracks or
        None)."""
        eng = self.engine
        diffs = torch.empty(tuple(t_goi.shape), dtype=torch.int32, device=eng.device) if self._realigns else None
        oo = eng.plan(t_reg, t_shifts, t_goi, out_len, max_rec, keep, keep_off, t_rc, diffs=diffs,
                      use_svar2=self.sequence_type != "reference")
        return oo, eng.total(), diffs

    def _execute_seqs(self, offsets, shape, total: int):
        """Execute the planned rows in this dataset's sequence output: ragged over `offsets` with `shape`, or dense
        (`shape` without its ragged axis) for channels-first one-hot."""
        eng = self.engine
        if self.sequence_type == "annotated":
            h, av, ap = eng.execute("annotated")
            return RaggedAnnotatedHaps(Ragged(h, offsets, shape), Ragged(av, offsets, shape), Ragged(ap, offsets, shape))
        if self.encoding == "bytes":
            return Ragged(eng.execute("haplotypes"), offsets, shape)
        if self.encoding == "onehot":
            return Ragged(eng.execute("onehot").view(total, 4), offsets, shape)
        return eng.execute("onehot_cf").view(*shape[:-1], 4, int(self.output_length))

    def _realigned_tracks(self, ds_idx, t_reg, t_shifts, t_goi, t_oi, lengths, diffs, row_offsets, total: int, max_rec: int,
                          keep, keep_off, t_rc, seq_offsets, shape, **rows) -> Ragged:
        """All active tracks realigned to planned haplotype rows in one call (HapsTracks.__call__, _reconstruct.py:182-300).
        One query per row of `t_goi` (dataset indices `ds_idx`, region `lengths`, planned `diffs`); its values go to
        `row_offsets` in (query, track, ploid) order or, given `row_dst` / `row_tstride`, where that table puts them.
        The (cell, track, ploid) rows take the lengths of the sequence rows at `seq_offsets`."""
        names = list(self.active_tracks)
        ids, params = self._fills(names)
        # a query's track window is its region less its longest net deletion (_reconstruct.py:191-196)
        track_lengths = (lengths - diffs.clamp(max=0).min(1).values.to(torch.int64)).to(torch.int32)
        # the reference's flat buffer is track-major (_reconstruct.py:238) while its offsets describe (b, t, p, ~l)
        # (:292-300); the kernel writes the latter directly so data and offsets agree for t > 1
        out = self.engine.realign_tracks(names, t_reg, t_shifts, t_goi, t_oi, track_lengths, row_offsets, total, ids, params,
                                         self._fill_seed(ds_idx), max_rec, keep, keep_off, t_rc,
                                         layout="rows" if rows else "btp", dtype=self.track_dtype, **rows)
        return Ragged(out, _cell_offsets(seq_offsets, len(names), self.ploidy), shape)

    def _painted_tracks(self, t_oi, starts, row_offsets, total: int, t_rc, offsets, shape, **rows) -> Ragged:
        """The stored intervals of all active tracks painted in one launch (Tracks._call_float32, _tracks.py:370-420),
        negative-strand rows reversed, in (query, track) order or, given `row_dst` / `row_tstride`, where that table puts
        each row.  `offsets`: of the output cells."""
        out = self.engine.paint_tracks(list(self.active_tracks), t_oi, starts, row_offsets, total, t_rc,
                                       layout="rows" if rows else "btp", dtype=self.track_dtype, **rows)
        return Ragged(out, offsets, shape)

    def _track_intervals(self, row_slot, row_tw, shape, cells=None) -> RaggedIntervals:
        """The stored intervals of the active tracks over one window per row (gvl_dev_track_intervals): row k reads slot
        `row_slot[k]` (device int64) of track `row_tw[0, k]` over [`row_tw[1, k]`, `row_tw[2, k]`) (device int32 (3, n),
        `_interval_rows`), clipped to it.  Strand changes nothing: coordinates stay on the reference.  `cells`: device
        indices into the row offsets at which the output cells start, the last one = the end; None = one cell per row."""
        off, starts, ends, values = self.engine.track_intervals(list(self.active_tracks), row_slot, row_tw[0], row_tw[1],
                                                                row_tw[2], dtype=self.track_dtype)
        if cells is not None:
            off = off[cells]
        return RaggedIntervals(Ragged(starts, off, shape), Ragged(ends, off, shape), Ragged(values, off, shape))

    def _get_variants(self, t_goi, t_rc, contigs, n_variants: int, shape, cells=None) -> RaggedVariants:
        """The variants of the genotype rows `t_goi` (device strand flags `t_rc`, host `contigs` of every row) as a
        RaggedVariants of `shape`.  `n_variants` = the sum of the rows' genotype slice lengths, known from the host copy of
        the offsets.  `cells`: device indices into the gathered row offsets (rows folded under `unphased_union`) at which
        the output cells start, the last one = the end; None = one cell per row."""
        row_contigs = None
        if self._variant_tokens() is not None:  # contig of every row (_flat_variants.py:985-989)
            row_contigs = torch.from_numpy(np.ascontiguousarray(contigs, np.int32)).to(self.engine.device)
        g, _ = self._gather_variants(self.engine, t_goi, t_rc, row_contigs, n_variants)
        off = g["row_offsets"] if cells is None else g["row_offsets"][cells]
        return self._variants_result(g, off, shape)

    def _variant_tokens(self):
        """The token settings of the variants tail (Engine.gather_variants `tokens`), None without flank / window tokens."""
        if self.sequence_type == "variant-windows":
            o = self.window_opt
            lut, _ = build_token_lut(o.token_alphabet, o.unknown_token)
            return dict(lut=lut, unk=o.unknown_token, L=o.flank_length, ref=1 if o.ref == "window" else 2,
                        alt=1 if o.alt == "window" else 2)
        if self.flank_length and self.token_alphabet is not None:
            lut, _ = build_token_lut(self.token_alphabet, self.unknown_token)
            return dict(lut=lut, unk=self.unknown_token, L=self.flank_length, flank=True)
        return None

    def _gather_variants(self, eng, t_goi, t_rc, row_contigs, n_variants: int):
        """The variants tail over the genotype rows `t_goi` on `eng` (this dataset's engine or a fork of it) and the current
        stream: the sizing pass and its one wait, then every buffer allocated at its final size -> (gather_variants dict,
        VariantSizes with one cell per output row)."""
        fold = self.ploidy if self.unphased_union else 1
        tokens = self._variant_tokens()
        sums = eng.variant_row_sizes(t_goi, self.min_af, self.max_af)
        sizes = variant_buffer_sizes(sums, fold, self.dummy_variant, tokens["L"] if tokens is not None else 0)
        g = eng.gather_variants(t_goi, t_rc, self.var_fields, sizes, n_variants, self.dummy_variant, self.min_af, self.max_af, fold,
                                tokens, row_contigs)
        return g, sizes

    def _variant_field_names(self, g) -> list:
        """The fields of a RaggedVariants in output order; `flank_tokens` last when present."""
        windows = self.sequence_type == "variant-windows"
        names = [n for n in self.var_fields if not (windows and n in ("alt", "ref"))]
        names += [n for n in ("ref_window", "alt_window", "ref", "alt") if windows and n in g]  # token buffers of the windows tail
        return names + (["flank_tokens"] if "flank_tokens" in g else [])

    def _variants_result(self, g, off, shape) -> RaggedVariants:
        fields = {}
        for name in self._variant_field_names(g):
            v = g[name]
            if name == "flank_tokens":  # (b, p, ~v, 2 L): the trailing token axis stays on `data`
                fields[name] = Ragged(v.view(-1, 2 * self.flank_length), off, shape)
            else:
                fields[name] = RaggedAlleles(v[0], v[1], off, shape) if isinstance(v, tuple) else Ragged(v, off, shape)
        return RaggedVariants(fields, off, shape)

    def _exonic_keep(self, t_goi, t_reg, goi):
        """choose_exonic_variants (src/genotypes/mod.rs:132-176): variants fully inside the query, on the device."""
        eng = self.engine
        return eng.choose_exonic_variants(t_reg[:, 1].contiguous(), t_reg[:, 2].contiguous(), t_goi, eng.max_records(goi))

    # ---- output shaping, _query.py:94-127 ----
    def _shape_output(self, o, out_reshape, squeeze):
        if (isinstance(o, (torch.Tensor, AnnotatedHaps, RaggedVariants, RaggedIntervals)) or self.output_format == "flat"
                or self.output_length == "ragged"):
            # already dense (fixed-length pipeline, channels-first one-hot), ragged by nature (variants, intervals: the
            # ragged axis counts items, not positions); "flat"/"ragged" hand the flat triple back
            res = o
        elif self.output_length == "variable":
            if isinstance(o, RaggedAnnotatedHaps):
                res = o.to_padded()
            elif o.data.is_floating_point():
                res = o.to_padded(0.0)                               # tracks (any track dtype) pad with 0 (_query.py:545-548)
            else:
                res = o.to_padded(0 if o.data.dim() > 1 else N_CHAR)  # bytes pad with N; one-hot with zeros
        else:
            res = o.to_fixed(int(self.output_length))
        if out_reshape is not None:
            if isinstance(res, torch.Tensor):
                res = res.reshape(*out_reshape, *res.shape[1:])
            elif isinstance(res, AnnotatedHaps):
                res = res.reshape((*out_reshape, *res.haps.shape[1:]))
            else:
                res = res.reshape((*out_reshape, *(d for d in res.shape[1:] if d is not None)))
        if squeeze:
            res = res.squeeze(0)  # (1 [p] l) -> ([p] l), _query.py:120-122
        return res


def _interval_rows(oi: np.ndarray, w0: np.ndarray, w1: np.ndarray, row_of: np.ndarray):
    """Host rows of a `_track_intervals` read: (element e, track t) reads slot oi[t, e] over [w0[e], w1[e]) as row
    row_of[e, t] -> (slots int64 (n,), int32 (3, n) of track, w0, w1)."""
    n_e, t = row_of.shape
    slot = np.empty(n_e * t, np.int64)
    tw = np.empty((3, n_e * t), np.int32)
    slot[row_of] = oi.T
    tw[0, row_of] = np.arange(t, dtype=np.int32)[None, :]
    tw[1, row_of] = np.asarray(w0)[:, None]
    tw[2, row_of] = np.asarray(w1)[:, None]
    return slot, tw


def _cell_offsets(row_offsets: torch.Tensor, t: int, p: int = 1) -> torch.Tensor:
    """Offsets of track cells (n, t, p) whose lengths are those of the sequence rows (n, p) at `row_offsets`."""
    n = (row_offsets.numel() - 1) // p
    lens = (row_offsets[1:] - row_offsets[:-1]).view(n, 1, p).expand(n, t, p).reshape(-1)
    offsets = torch.zeros(n * t * p + 1, dtype=torch.int64, device=row_offsets.device)
    torch.cumsum(lens, 0, out=offsets[1:])
    return offsets


class _Packer:
    """All O(batch) host arrays of one call in ONE pinned buffer and ONE async H2D copy."""

    def __init__(self, device):
        self.device = device
        self.items = []
        self.total = 0
        self.dev = None

    def add(self, arr, dtype) -> int:
        a = np.ascontiguousarray(arr, dtype)
        self.items.append((a, self.total))
        self.total += (a.nbytes + 15) & ~15
        return len(self.items) - 1

    def upload(self) -> None:
        host = torch.empty(max(self.total, 16), dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        for a, off in self.items:
            hv[off: off + a.nbytes] = a.reshape(-1).view(np.uint8)
        self.dev = host.to(self.device, non_blocking=True)
        self._host = host  # keep the pinned buffer alive until the copy has been consumed

    def get(self, i: int) -> torch.Tensor:
        a, off = self.items[i]
        tdt = torch.from_numpy(np.empty(0, a.dtype)).dtype
        return self.dev[off: off + a.nbytes].view(tdt).view(a.shape)


class BatchLoader:
    """Re-iterable batch iterator over a `Dataset` (see `Dataset.to_dataloader`)."""

    def __init__(self, ds: Dataset, batch_size: int, shuffle: bool, sampler, drop_last: bool, generator, return_indices: bool,
                 transform):
        if batch_size < 1:
            raise ValueError("batch_size must be a positive integer")
        self.ds, self.batch_size, self.shuffle, self.sampler = ds, batch_size, shuffle, sampler
        self.drop_last, self.return_indices, self.transform = drop_last, return_indices, transform
        self._rng = _as_rng(generator)

    def __len__(self) -> int:
        n = len(self.sampler) if self.sampler is not None else len(self.ds)
        return n // self.batch_size if self.drop_last else -(-n // self.batch_size)

    def __iter__(self):
        order = epoch_order(self.ds, self.sampler, self.shuffle, self._rng)
        n_s = self.ds.n_samples
        for lo in range(0, len(order), self.batch_size):
            idx = order[lo: lo + self.batch_size]
            if len(idx) < self.batch_size and self.drop_last:
                return
            r, s_ = idx // n_s, idx % n_s  # np.unravel_index(idx, dataset.shape), _torch.py:293
            yield _batch_tail(self.ds[r, s_], (r, s_) if self.return_indices else None, self.transform)


class _MapDataset:
    """Map-style view of a Dataset (reference `TorchDataset`, _torch.py:272-307); usable with torch.utils.data.DataLoader
    (batch_size=None + a BatchSampler, as the reference's own loader does)."""

    def __init__(self, dataset: Dataset, include_indices: bool, transform):
        self.dataset, self.include_indices, self.transform = dataset, include_indices, transform

    def __len__(self) -> int:
        return len(self.dataset)

    def __getitem__(self, idx):
        r_idx, s_idx = np.unravel_index(idx, self.dataset.shape)
        return _batch_tail(self.dataset[r_idx, s_idx], (r_idx, s_idx) if self.include_indices else None, self.transform)


def _as_rng(generator) -> np.random.Generator:
    """The numpy generator of a loader's `generator` argument: None / a seed, a numpy Generator or a torch.Generator."""
    if generator is None or isinstance(generator, (int, np.integer)):
        return np.random.default_rng(generator)
    if isinstance(generator, np.random.Generator):
        return generator
    return np.random.default_rng(int(generator.initial_seed()))  # torch.Generator


def epoch_order(ds, sampler, shuffle, rng) -> np.ndarray:
    """Flat (region, sample) indices of one epoch, in the order the loader reads them."""
    if sampler is not None:
        if isinstance(sampler, np.ndarray):  # (an index array is its own sampler: no per-element iteration)
            return np.ascontiguousarray(sampler, np.int64).ravel()
        return np.fromiter(iter(sampler), np.int64)
    if shuffle:
        return rng.permutation(len(ds)).astype(np.int64)
    return np.arange(len(ds), dtype=np.int64)


def _batch_tail(batch, indices, transform):
    """What a loader yields for one batch: its outputs, then the (region, sample) `indices` it was read with unless None
    (_torch.py:299-300), passed through `transform` (_torch.py:302-303); a lone output is returned bare."""
    if not isinstance(batch, tuple):
        batch = (batch,)
    if indices is not None:
        batch = (*batch, *indices)
    if transform is not None:
        return transform(*batch)
    return batch[0] if len(batch) == 1 else batch
