"""A numpy restatement of a `Dataset` track read, with the CPU oracle underneath, and the host references of the
outputs derived from it (16-bit stores, binned tracks).

The read follows the reference's read-time prep: jittered regions (python/genvarloader/_dataset/_query.py:161-175),
strand masks and genotype rows (_haps.py:757-768, :838-843), keep masks and diffs, random shifts (_haps.py:720-730),
the fill seed (_reconstruct.py:215-222), output and track offsets (_reconstruct.py:182-300), the per-track interval slot
(_reconstruct.py:233-236), then per track the oracle's realignment (`intervals_and_realign_track_fused`) or painting
(`intervals_to_tracks` + `reverse_flat_rows_inplace`).  It never calls into `Dataset` or `Engine`: its inputs are the
dataset's arrays, the read state, the (region, sample) pairs and the generator seed.

Draws from `np.random.default_rng(seed)`, in this order and only when they happen:
  1. jitter, one int32 per read in [-jitter, jitter] (when jitter > 0);
  2. random shifts, one int32 per haplotype row in [0, max_shift] (fixed-length haplotype or annotated reads with
     deterministic=False);
  3. the fill seed, one uint64 in [0, 2**64 - 1) (realigned tracks with deterministic=False; otherwise the xor of the
     dataset indices).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

FILL_IDS = {"Repeat5p": 0, "Repeat5pNormalized": 1, "Constant": 2, "FlankSample": 3, "Interpolate": 4}
ARITH_FILLS = (1, 4)  # fills that compute values (NaNs they produce are compared as NaN only)


# ---------------------------------------------------------------------------------------------------------------------
# the read state
# ---------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class ReadState:
    """The settings of a `Dataset` that a track read depends on.  `fills`: track name -> (strategy id, parameter), for
    realigned reads (Repeat5p when absent)."""

    seqs: object = "haplotypes"           # "haplotypes" | "annotated" | "reference" | None
    realign: bool = True
    length: object = "ragged"             # int | "ragged" | "variable"
    jitter: int = 0
    deterministic: bool = True
    rc_neg: bool = True
    exonic: bool = False
    tracks: tuple = ()
    fills: dict = field(default_factory=dict)

    @property
    def realigns(self) -> bool:
        return bool(self.tracks) and self.seqs in ("haplotypes", "annotated") and self.realign

    @property
    def fixed(self) -> bool:
        return isinstance(self.length, (int, np.integer)) and not isinstance(self.length, bool)


@dataclass
class TrackRead:
    """The float32 values of one read: `data` holds every (read, track[, ploid]) cell in that order, cell c at
    data[offsets[c]:offsets[c + 1]]; `cells` is the outer shape; `nan_class` marks the values whose NaNs are compared
    as NaN only (those an arithmetic fill writes at insertions); `w0` the window start of every cell and `rc` its
    strand mask."""

    data: np.ndarray
    offsets: np.ndarray
    cells: tuple
    nan_class: np.ndarray
    w0: np.ndarray
    rc: np.ndarray
    draws: dict

    def cell(self, c: int) -> np.ndarray:
        return self.data[self.offsets[c]:self.offsets[c + 1]]

    def dense(self) -> np.ndarray:
        """Fixed-length cells as (*cells, L); variable-length cells padded with +0.0 to the longest."""
        lens = np.diff(self.offsets)
        L = int(lens.max()) if lens.size else 0
        out = np.zeros((lens.size, L), np.float32)
        mask = np.arange(L)[None, :] < lens[:, None]
        out[mask] = self.data
        return out.reshape(*self.cells, L)


def _gather_cells(bufs, row_off, rows_of_cell, track_of_cell):
    """Concatenate the rows rows_of_cell[c] of track buffers bufs[track_of_cell[c]] -> (data, offsets)."""
    total = int(row_off[-1])
    big = np.concatenate(bufs) if bufs else np.zeros(0, np.float32)  # (float32 values or bool masks)
    lens = (row_off[rows_of_cell + 1] - row_off[rows_of_cell]).astype(np.int64)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    src0 = track_of_cell.astype(np.int64) * total + row_off[rows_of_cell]
    idx = np.repeat(src0 - offsets[:-1], lens) + np.arange(int(offsets[-1]), dtype=np.int64)
    return big[idx], offsets


def read_tracks(O, d, kinds: dict, st: ReadState, ds_idx, seed) -> TrackRead:
    """The track output of a read of `d` in state `st` at flat dataset indices `ds_idx` (row-major over the full
    (regions, samples) grid), with the generator `np.random.default_rng(seed)`.  `kinds`: track name -> "sample" |
    "annot".  The variants are those of the SVAR1 arrays of `d` (an svar2 re-expression of them carries the same
    haplotypes)."""
    rng = np.random.default_rng(seed)
    ds_idx = np.asarray(ds_idx, np.int64)
    S, p = d.n_samples, d.ploidy
    b = ds_idx.size
    r_idx = ds_idx // S
    draws = {}

    # 1. jittered regions: the window keeps its length, its start moves
    regions = np.ascontiguousarray(d.regions[r_idx, :3], np.int32).copy()
    lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)
    if st.jitter:
        jit = rng.integers(-st.jitter, st.jitter + 1, size=b, dtype=np.int32)
        draws["jitter"] = jit
        regions[:, 1] += jit
        regions[:, 2] = regions[:, 1] + lengths.astype(np.int32)

    # 2. strand masks and genotype rows
    rc_q = (d.regions[r_idx, 3] == -1) if st.rc_neg else np.zeros(b, bool)
    goi = ds_idx[:, None] * p + np.arange(p, dtype=np.int64)[None, :]
    hap_seqs = st.seqs in ("haplotypes", "annotated")

    # 3. keep masks and diffs
    keep = ko = None
    diffs = np.zeros((b, p), np.int32)
    if hap_seqs:
        if st.exonic:
            keep, ko = O.choose_exonic_variants(regions[:, 1], regions[:, 2], goi, d.geno_v_idxs, d.geno_offsets,
                                                d.v_starts, d.ilens)
        diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, keep, ko, regions[:, 1], regions[:, 2],
                                   d.v_starts)

    # 4. random shifts
    shifts = np.zeros((b, p), np.int32)
    if st.fixed and hap_seqs and not st.deterministic:
        max_shift = diffs.clip(min=0) + (lengths - int(st.length)).clip(min=0)[:, None]
        shifts = rng.integers(0, max_shift + 1, dtype=np.int32)
        draws["shifts"] = shifts

    # 5. fill seed
    seed_ = 0
    if st.realigns:
        if st.deterministic:
            seed_ = int(np.bitwise_xor.reduce(ds_idx.astype(np.uint64)))
        else:
            seed_ = int(rng.integers(0, np.iinfo(np.uint64).max, dtype=np.uint64))
            draws["fill_seed"] = seed_

    names = list(st.tracks)
    t = len(names)
    # 7. per-track slots: the dataset index of a sample track, the region of an annotation track
    slots = [ds_idx if kinds[n] == "sample" else r_idx for n in names]
    bufs, nan_class = [], []
    if st.realigns:
        # 6. one row per (read, ploid): L, or the haplotype's length; track windows lose the longest net deletion
        row_len = np.full((b, p), int(st.length), np.int64) if st.fixed else lengths[:, None] + diffs
        row_off = np.concatenate([[0], np.cumsum(row_len.ravel())]).astype(np.int64)
        trk_off = np.concatenate([[0], np.cumsum(lengths - diffs.clip(max=0).min(1))]).astype(np.int64)
        to_rc = np.repeat(rc_q, p)

        def realign(n, sl, sid, par):
            s, e, v, io = d.tracks[n]
            buf = np.zeros(int(row_off[-1]), np.float32)
            O.intervals_and_realign_track_fused(buf, row_off, regions, shifts, goi, d.geno_v_idxs, d.geno_offsets, d.v_starts,
                                                d.ilens, sl, s, e, v, io, trk_off, np.array([par], np.float64), sid, seed_,
                                                keep, ko, to_rc)
            return buf

        for n, sl in zip(names, slots):
            sid, par = st.fills.get(n, (0, 0.0))
            bufs.append(realign(n, sl, sid, par))
            if sid in ARITH_FILLS:
                # the positions an insertion fill writes: where two Constant fills differ; everywhere else the value is
                # copied from the stored intervals and must keep its bits
                nan_class.append(realign(n, sl, 2, 1.0) != realign(n, sl, 2, 2.0))
            else:
                nan_class.append(np.zeros(bufs[-1].size, bool))
        q = np.repeat(np.arange(b, dtype=np.int64), t * p)
        tt = np.tile(np.repeat(np.arange(t, dtype=np.int64), p), b)
        hh = np.tile(np.arange(p, dtype=np.int64), b * t)
        rows = q * p + hh
        cells = (b, t, p)
    else:
        # 6. painted: one row per read over [start, start + L) (fixed) or the region
        row_len = np.full(b, int(st.length), np.int64) if st.fixed else lengths
        row_off = np.concatenate([[0], np.cumsum(row_len)]).astype(np.int64)
        for n, sl in zip(names, slots):
            s, e, v, io = d.tracks[n]
            buf = np.zeros(int(row_off[-1]), np.float32)
            O.intervals_to_tracks(sl, regions[:, 1], s, e, v, io, buf, row_off)
            O.reverse_flat_rows_inplace(buf, row_off, rc_q)
            bufs.append(buf)
            nan_class.append(np.zeros(buf.size, bool))
        q = np.repeat(np.arange(b, dtype=np.int64), t)
        tt = np.tile(np.arange(t, dtype=np.int64), b)
        rows = q
        cells = (b, t)
    data, offsets = _gather_cells(bufs, row_off, rows, tt)
    nan_mask, _ = _gather_cells(nan_class, row_off, rows, tt)
    return TrackRead(data, offsets, cells, nan_mask, regions[q, 1].astype(np.int64), rc_q[q], draws)


def assert_f32(got: np.ndarray, exp: np.ndarray, nan_class: np.ndarray, what=""):
    """Bit equality, except that a NaN the oracle computed (nan_class) only needs a NaN."""
    got = np.ascontiguousarray(got, np.float32).reshape(-1)
    exp = np.ascontiguousarray(exp, np.float32).reshape(-1)
    assert got.shape == exp.shape, (what, got.shape, exp.shape)
    ok = got.view(np.uint32) == exp.view(np.uint32)
    ok |= np.broadcast_to(nan_class, ok.shape) & np.isnan(exp) & np.isnan(got)
    if not ok.all():
        k = np.flatnonzero(~ok)
        raise AssertionError(f"{what}: {k.size} of {ok.size} values differ, first at {k[:5]}: got "
                             f"{got[k[:5]].view(np.uint32)} expected {exp[k[:5]].view(np.uint32)}")


# ---------------------------------------------------------------------------------------------------------------------
# 16-bit stores
# ---------------------------------------------------------------------------------------------------------------------
def bf16_bits(x) -> np.ndarray:
    """float32 -> bfloat16 bits, rounded to nearest even on the bit pattern (NaN -> a quiet NaN of the same sign)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)
    nan = np.isnan(np.asarray(x, np.float32))
    return np.where(nan, ((u >> 16) | 0x40).astype(np.uint16), r)


def f16_bits(x) -> np.ndarray:
    """float32 -> float16 bits, rounded to nearest even (subnormals kept, overflow to inf)."""
    with np.errstate(over="ignore"):
        return np.ascontiguousarray(x, np.float32).astype(np.float16).view(np.uint16)


def narrow_bits(x, dtype_name: str) -> np.ndarray:
    if dtype_name == "float32":
        return np.ascontiguousarray(x, np.float32).view(np.uint32)
    return bf16_bits(x) if dtype_name == "bfloat16" else f16_bits(x)


def bits_are_nan(bits: np.ndarray, dtype_name: str) -> np.ndarray:
    if dtype_name == "float32":
        return np.isnan(bits.view(np.float32))
    exp_mask, man_mask = (0x7F80, 0x007F) if dtype_name == "bfloat16" else (0x7C00, 0x03FF)
    return ((bits & exp_mask) == exp_mask) & ((bits & man_mask) != 0)


def assert_narrowed(got_bits: np.ndarray, exp32: np.ndarray, dtype_name: str, what=""):
    """A 16-bit (or float32) store of `exp32`: equal bits, a NaN wherever the float32 value is a NaN (the device writes
    its canonical NaN)."""
    exp = narrow_bits(exp32, dtype_name).reshape(-1)
    got_bits = got_bits.reshape(-1)
    en, gn = bits_are_nan(exp, dtype_name), bits_are_nan(got_bits, dtype_name)
    assert np.array_equal(en, gn), (what, "NaNs in different places", np.flatnonzero(en != gn)[:5])
    bad = ~en & (got_bits != exp)
    if bad.any():
        k = np.flatnonzero(bad)
        raise AssertionError(f"{what}: {k.size} values differ, first at {k[:5]}: got {got_bits[k[:5]]} expected {exp[k[:5]]} "
                             f"(float32 {exp32.reshape(-1)[k[:5]]})")


# ---------------------------------------------------------------------------------------------------------------------
# binned tracks: the definition, exactly
# ---------------------------------------------------------------------------------------------------------------------
def f32_parts(x: np.ndarray):
    """Finite float32 values as (integer significand m, exponent e) with x = m * 2**e exactly; e is the value's ulp
    (2**-149 for subnormals and zeros)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.int64)
    sign = np.where(u >> 31, -1, 1)
    ex = (u >> 23) & 0xFF
    man = u & 0x7FFFFF
    m = np.where(ex > 0, man | 0x800000, man) * sign
    e = np.where(ex > 0, ex - 150, -149)
    return m, e


def round_f32(num: int, e: int) -> np.float32:
    """num * 2**e (exact, integers) rounded once to float32, to nearest even; +-inf past the largest finite value."""
    if num == 0:
        return np.float32(0.0)
    sign = -1.0 if num < 0 else 1.0
    a = abs(num)
    top = a.bit_length() - 1 + e                  # exponent of the leading bit
    qe = max(top - 23, -149)                      # exponent of the float32 ulp at that magnitude
    shift = qe - e
    if shift > 0:
        q, r = divmod(a, 1 << shift)
        half = 1 << (shift - 1)
        if r > half or (r == half and q & 1):
            q += 1
    else:
        q = a << -shift
    v = float(q) * 2.0 ** qe                      # exact in float64 (q <= 2**24)
    if v >= 2.0 ** 128:
        return np.float32(sign * np.inf)
    return np.float32(sign * v)


def exactly_summable(vals: np.ndarray) -> bool:
    """Every partial sum of the finite float32 values `vals` is exact in float64: sum |x| / (the smallest ulp among the
    non-zero values) < 2**53.  Bins holding a NaN or an infinity are not."""
    vals = np.asarray(vals, np.float32)
    if not np.isfinite(vals).all():
        return False
    nz = vals[vals != 0]
    if nz.size == 0:
        return True
    m, e = f32_parts(nz)
    e0 = int(e.min())
    total = sum(abs(int(mi)) << (int(ei) - e0) for mi, ei in zip(m, e))
    return total < (1 << 53)


def exact_bin(vals: np.ndarray, reduce: str) -> np.float32:
    """The definition of one bin on float32 values: "sum" -- the exact sum rounded once to float32; "mean" -- the exact
    sum / len rounded once (len a power of two); "max" -- the largest value.  A NaN, or +inf with -inf, makes it NaN."""
    vals = np.asarray(vals, np.float32)
    if np.isnan(vals).any():
        return np.float32(np.nan)
    if reduce == "max":
        return vals.max()
    pinf, ninf = (vals == np.inf).any(), (vals == -np.inf).any()
    if pinf and ninf:
        return np.float32(np.nan)
    if pinf or ninf:
        return np.float32(np.inf if pinf else -np.inf)
    m, e = f32_parts(vals)
    e0 = int(e.min())
    total = sum(int(mi) << (int(ei) - e0) for mi, ei in zip(m, e))
    B = vals.size
    assert B & (B - 1) == 0
    return round_f32(total, e0 - (B.bit_length() - 1 if reduce == "mean" else 0))


def value_class(bits: np.ndarray, dtype_name: str) -> np.ndarray:
    """0 finite, 1 +inf, 2 -inf, 3 NaN."""
    if dtype_name == "float32":
        x = bits.view(np.float32)
    else:
        x = (bits.view(np.float16).astype(np.float32) if dtype_name == "float16"
             else (bits.astype(np.uint32) << 16).view(np.float32))
    return np.where(np.isnan(x), 3, np.where(x == np.inf, 1, np.where(x == -np.inf, 2, 0)))


def assert_bins(got_bits: np.ndarray, x32: np.ndarray, B: int, reduce: str, dtype_name: str, what=""):
    """Binned cells `got_bits` (cells, L // B) of the dtype against the definition on the oracle's float32 cells `x32`
    (cells, L).  Exactly summable bins (and every bin of `max`, +-0 equal) must match bit for bit.  In the others the
    float64 order may move a finite result across the dtype's overflow threshold, so only what no order changes is
    checked: NaN where the definition gives NaN, and the infinity of a bin holding one.  Returns (bins, exactly checked
    bins)."""
    xb = np.asarray(x32, np.float32).reshape(-1, B)
    got_bits = got_bits.reshape(-1)
    assert got_bits.size == xb.shape[0], (what, got_bits.size, xb.shape)
    exp32 = np.array([exact_bin(v, reduce) for v in xb], np.float32)
    exp_bits = narrow_bits(exp32, dtype_name)
    exact = np.array([reduce == "max" or exactly_summable(v) for v in xb], bool)
    ecls, gcls = value_class(exp_bits, dtype_name), value_class(got_bits, dtype_name)
    fixed_cls = exact | (ecls == 3) | (gcls == 3) | np.isinf(xb).any(1)
    bad_cls = fixed_cls & (ecls != gcls)
    assert not bad_cls.any(), (what, "value classes differ", np.flatnonzero(bad_cls)[:5])
    same = got_bits == exp_bits
    if reduce == "max":  # +0 and -0 are both the largest value of a bin holding both
        zero = 0x7FFFFFFF if dtype_name == "float32" else 0x7FFF
        same |= ((got_bits & zero) == 0) & ((exp_bits & zero) == 0)
    bad = exact & (ecls != 3) & ~same
    if bad.any():
        k = np.flatnonzero(bad)
        raise AssertionError(f"{what}: {k.size} bins differ, first at {k[:5]}: got {got_bits[k[:5]]} expected "
                             f"{exp_bits[k[:5]]}, bin values {xb[k[0]]}")
    return xb.shape[0], int(exact.sum())


# ---------------------------------------------------------------------------------------------------------------------
# the edge-valued track
# ---------------------------------------------------------------------------------------------------------------------
def _f(bits: int) -> np.float32:
    return np.array([bits], np.uint32).view(np.float32)[0]


EDGE_SPECIALS = np.array([
    0.0, -0.0, -1.5, -3.25, -1e-3, -7.0e20,             # +-0, negative normals
    1e-40, -1.4e-45,                                     # float32 subnormals
    6e-8, 1e-7, 65504.0, 65519.996, 65520.0,             # float16: subnormals, largest finite, last below inf, inf
    _f(0x3F808000), _f(0x3F818000),                      # bfloat16 ties (to even: down, up)
    np.finfo(np.float32).max, -np.finfo(np.float32).max, np.inf, -np.inf,
    _f(0x7FC00001), _f(0xFFC00000),                      # quiet NaNs: a payload, a sign
], np.float32)
EDGE_NEGATIVE = np.array([-1.5, -3.25, -0.75, -2.0e-3, -6.0e4, -1.0e30], np.float32)


def big_fraction_values(n: int, rng) -> np.ndarray:
    """2**20 + k/8: exact in float32, while the sum of two of them needs more than float32's 24 bits."""
    return (np.float32(2.0 ** 20) + rng.integers(1, 8 * 1024, n).astype(np.float32) / np.float32(8)).astype(np.float32)


def make_edge_track(rng, regions, n_slots_per_region, max_jitter=0, headroom=64):
    """Interval SoA per slot covering the expanded region with no holes, built from runs of three kinds: short
    intervals holding EDGE_SPECIALS in turn (so every fill meets them as anchors next to insertions), long runs
    of negative values (whole bins all negative) and runs of 2**20 + k/8 values (bins exactly summable in float64 but
    not in float32)."""
    starts, ends, values, counts = [], [], [], []
    n_spec = EDGE_SPECIALS.size
    k_spec = 0
    for r in range(regions.shape[0]):
        s0 = int(regions[r, 1]) - max_jitter
        e0 = int(regions[r, 2]) + max_jitter + headroom
        for _ in range(n_slots_per_region):
            pos, n = s0, 0
            kind = int(rng.integers(0, 3))
            while pos < e0:
                if kind == 0:  # the next 4-8 specials, 1-4 positions each
                    vs = [EDGE_SPECIALS[(k_spec + i) % n_spec] for i in range(int(rng.integers(4, 9)))]
                    k_spec += len(vs)
                    ln = None
                elif kind == 1:  # one negative run of 40-140 positions, in 1-4 intervals
                    ln = int(rng.integers(40, 141))
                    vs = list(rng.choice(EDGE_NEGATIVE, int(rng.integers(1, 5))))
                else:  # 2**20 + k/8 values, 1-4 positions each, 8-24 of them
                    vs = list(big_fraction_values(int(rng.integers(8, 25)), rng))
                    ln = None
                for v in vs:
                    w = int(rng.integers(1, 5)) if ln is None else max(1, ln // len(vs))
                    w = min(w, e0 - pos)
                    if w <= 0:
                        break
                    starts.append(pos)
                    ends.append(pos + w)
                    values.append(v)
                    pos += w
                    n += 1
                kind = (kind + 1 + int(rng.integers(0, 2))) % 3
            counts.append(n)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return (np.array(starts, np.int32), np.array(ends, np.int32), np.array(values, np.float32), off)
