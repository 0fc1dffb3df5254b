"""Buffer lengths of a `variants` / `variant-windows` read, on the host, from four sums per genotype row.

`gvl_dev_variant_row_sizes` gives, for every genotype row r, `(n, alt, ref, span)`: the variants the AF filter keeps, the
sum of their ALT lengths, of their REF lengths and of their reference spans `1 - min(ilen, 0)`.  Every length of the read
follows from these: `unphased_union` folds `fold` consecutive rows into one cell (a cell's sums are its rows' sums), the
dummy fill gives every empty cell one variant with the dummy's ALT / REF, windows are `2 L` tokens longer than the ALT
allele or the reference span, and flank tokens are `2 L` per variant.  Pure numpy: the read (`Dataset.__getitem__`) and
the read-ahead loader both size their buffers here and never read an offsets array back from the device.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

# per-cell lengths: the variants, then the items of every two-level field (bytes or tokens, one sequence per variant)
FIELDS = ("variants", "alt", "ref", "ref_window", "alt_window", "flank_tokens")


@dataclass(frozen=True)
class VariantSizes:
    """Per-cell lengths (int64 arrays, one entry per cell) of every buffer of a variants read: `raw` before the dummy
    fill, `out` as returned (the same arrays when there is no dummy variant)."""

    raw: dict
    out: dict

    @property
    def n_cells(self) -> int:
        return int(self.out["variants"].size)

    def total(self, name: str, filled: bool = True) -> int:
        return int((self.out if filled else self.raw)[name].sum())

    def bounds(self, name: str, cells_per_batch: int) -> np.ndarray:
        """Start of every batch of `cells_per_batch` cells in the returned `name` buffer, and its end: int64 (K + 1,)."""
        cum = np.zeros(self.n_cells + 1, np.int64)
        np.cumsum(self.out[name], out=cum[1:])
        return cum[np.append(np.arange(0, self.n_cells, cells_per_batch, dtype=np.int64), self.n_cells)]


def variant_buffer_sizes(row_sums, fold: int = 1, dummy=None, flank_len: int = 0) -> VariantSizes:
    """`row_sums`: int64 (n_rows, 4) from gvl_dev_variant_row_sizes; `fold`: rows per cell (the ploidy under
    `unphased_union`, else 1); `dummy`: the DummyVariant given to every empty cell, or None; `flank_len`: L of the flank /
    window tokens (0 when the read has none)."""
    s = np.asarray(row_sums, np.int64).reshape(-1, 4)
    if s.shape[0] % fold:
        raise ValueError(f"{s.shape[0]} genotype rows do not fold by {fold}")
    cell = s.reshape(-1, fold, 4).sum(1)
    n, alt, ref, span = (np.ascontiguousarray(cell[:, j]) for j in range(4))
    L2 = 2 * int(flank_len)
    raw = {"variants": n, "alt": alt, "ref": ref, "ref_window": L2 * n + span, "alt_window": L2 * n + alt, "flank_tokens": L2 * n}
    if dummy is None:
        return VariantSizes(raw, raw)
    empty = (n == 0).astype(np.int64)
    d_alt, d_ref = len(dummy.alt), len(dummy.ref)
    out = {"variants": n + empty, "alt": alt + empty * d_alt, "ref": ref + empty * d_ref,
           "ref_window": raw["ref_window"] + empty * (L2 + d_ref), "alt_window": raw["alt_window"] + empty * (L2 + d_alt),
           "flank_tokens": L2 * (n + empty)}
    return VariantSizes(raw, out)
