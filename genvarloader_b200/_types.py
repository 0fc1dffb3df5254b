"""Return containers of the GPU `Dataset` -- torch-tensor counterparts of the reference's
`_Flat` (python/genvarloader/_flat.py:26-214), `AnnotatedHaps` (python/genvarloader/_types.py:26) and
`RaggedAnnotatedHaps` (python/genvarloader/_ragged.py)."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Any

import numpy as np
import torch

INT32_MAX = int(np.iinfo(np.int32).max)


@dataclass(frozen=True)
class Ragged:
    """Flat `(data, offsets, shape)` ragged array on the device (exactly one ragged axis, last).

    `data` is the flat buffer the kernels wrote, `offsets` int64 `(n_rows + 1,)`, `shape` the outer
    fixed dims followed by `None`.  For one-hot data the trailing alphabet axis of 4 is kept on `data`
    (`data.shape == (total, 4)`)."""

    data: torch.Tensor
    offsets: torch.Tensor
    shape: tuple

    @property
    def n_rows(self) -> int:
        return int(np.prod([d for d in self.shape if d is not None], dtype=np.int64))

    @property
    def lengths(self) -> torch.Tensor:
        outer = tuple(d for d in self.shape if d is not None)
        return (self.offsets[1:] - self.offsets[:-1]).reshape(outer)

    def reshape(self, shape) -> "Ragged":
        if isinstance(shape, int):
            shape = (shape,)
        return Ragged(self.data, self.offsets, tuple(shape) + (None,))

    def squeeze(self, axis: int | None = None) -> "Ragged":
        outer = [d for d in self.shape if d is not None]
        if axis is None:
            outer = [d for d in outer if d != 1]
        else:
            if outer[axis] != 1:
                raise ValueError(f"cannot squeeze axis {axis} with size {outer[axis]}")
            del outer[axis]
        return Ragged(self.data, self.offsets, (*outer, None))

    def to_fixed(self, length: int) -> torch.Tensor:
        """Every row has exactly `length` elements: pure reshape (reference `_Flat.to_fixed`, _flat.py:54-57)."""
        outer = tuple(d for d in self.shape if d is not None)
        return self.data.reshape(*outer, length, *self.data.shape[1:])

    def to_padded(self, pad_value: Any) -> torch.Tensor:
        """Right-pad every row to the longest one (reference `to_padded`, _ragged.py:281-314 ->
        src/ragged/mod.rs:7-23): gvl_dev_ragged_to_padded_fill copies the rows and writes the pad item behind them in one pass."""
        import ctypes as C

        from ._engine import _stream
        from ._ffi import check, lib, ptr
        from ._kernels import default_ctx

        outer = tuple(d for d in self.shape if d is not None)
        lens = self.offsets[1:] - self.offsets[:-1]
        n_rows = lens.numel()
        max_len = int(lens.max().item()) if n_rows else 0
        dev = self.data.device
        # one pass: the kernel copies the rows AND writes the pad item behind them (no torch.full pre-fill of the whole output)
        out = torch.empty((n_rows, max_len, *self.data.shape[1:]), dtype=self.data.dtype, device=dev)
        if n_rows and max_len:
            data, offsets = self.data.contiguous(), self.offsets.contiguous()
            itemsize = data.element_size() * int(np.prod(data.shape[1:], dtype=np.int64))  # one-hot rows: 4 bytes per position
            if data.dtype in (torch.bfloat16, torch.float16):  # 16-bit tracks (numpy has no bfloat16: torch gives the bits)
                pad_item = torch.full(tuple(data.shape[1:]) or (1,), pad_value, dtype=data.dtype).view(torch.int16).numpy().tobytes()
            else:
                np_dt = {torch.uint8: np.uint8, torch.int32: np.int32, torch.float32: np.float32, torch.int64: np.int64}[data.dtype]
                pad_item = np.full(tuple(data.shape[1:]) or (1,), pad_value, np_dt).tobytes()
            with torch.cuda.device(dev):
                if len(pad_item) <= 8:
                    check(lib.gvl_dev_ragged_to_padded_fill(default_ctx(dev.index or 0).handle, ptr(data), ptr(offsets),
                                                            C.c_int64(n_rows), ptr(out), C.c_int64(itemsize), C.c_int64(max_len),
                                                            C.c_char_p(pad_item), _stream()))
                else:  # (items wider than 8 bytes: pre-fill, then copy)
                    out.fill_(pad_value)
                    check(lib.gvl_dev_ragged_to_padded(default_ctx(dev.index or 0).handle, ptr(data), ptr(offsets),
                                                       C.c_int64(n_rows), ptr(out), C.c_int64(itemsize), C.c_int64(max_len),
                                                       _stream()))
        return out.reshape(*outer, max_len, *self.data.shape[1:])

    def to_numpy(self):
        return self.data.cpu().numpy(), self.offsets.cpu().numpy(), self.shape


@dataclass(frozen=True)
class AnnotatedHaps:
    """Dense annotated haplotypes (reference `AnnotatedHaps`, python/genvarloader/_types.py:26-60)."""

    haps: torch.Tensor        # uint8  (..., L)
    var_idxs: torch.Tensor    # int32  (..., L)   -1 = reference / pad
    ref_coords: torch.Tensor  # int32  (..., L)   -1 = leading pad, INT32_MAX = trailing pad

    @property
    def shape(self):
        return tuple(self.haps.shape)

    def reshape(self, shape):
        return AnnotatedHaps(self.haps.reshape(shape), self.var_idxs.reshape(shape), self.ref_coords.reshape(shape))

    def squeeze(self, axis=None):
        f = (lambda t: t.squeeze()) if axis is None else (lambda t: t.squeeze(axis))
        return AnnotatedHaps(f(self.haps), f(self.var_idxs), f(self.ref_coords))


@dataclass(frozen=True)
class RaggedAnnotatedHaps:
    haps: Ragged
    var_idxs: Ragged
    ref_coords: Ragged

    @property
    def shape(self):
        return self.haps.shape

    def reshape(self, shape):
        return RaggedAnnotatedHaps(self.haps.reshape(shape), self.var_idxs.reshape(shape), self.ref_coords.reshape(shape))

    def squeeze(self, axis=None):
        return RaggedAnnotatedHaps(self.haps.squeeze(axis), self.var_idxs.squeeze(axis), self.ref_coords.squeeze(axis))

    def to_fixed(self, length: int) -> AnnotatedHaps:
        return AnnotatedHaps(self.haps.to_fixed(length), self.var_idxs.to_fixed(length), self.ref_coords.to_fixed(length))

    def to_padded(self) -> AnnotatedHaps:
        # pad values: python/genvarloader/_flat.py:207-214
        return AnnotatedHaps(self.haps.to_padded(ord("N")), self.var_idxs.to_padded(-1), self.ref_coords.to_padded(INT32_MAX))


@dataclass(frozen=True)
class DummyVariant:
    """Per-field values of the dummy variant inserted into empty (region, sample, ploid) groups (reference
    `DummyVariant`, python/genvarloader/_dataset/_flat_variants.py:39-68): unspecified info fields default to 0 for
    integer columns and NaN for float columns."""

    start: int = -1
    ilen: int = 0
    dosage: float = 0.0
    ref: bytes = b"N"
    alt: bytes = b"N"
    info: Any = None

    def scalar_for(self, name: str, dtype):
        dt = np.dtype(dtype)
        if name == "start":
            return dt.type(self.start)
        if name == "ilen":
            return dt.type(self.ilen)
        if name == "dosage":
            return dt.type(self.dosage)
        if self.info and name in self.info:
            return dt.type(self.info[name])
        return dt.type(np.nan) if np.issubdtype(dt, np.floating) else dt.type(0)


@dataclass(frozen=True)
class RaggedAlleles:
    """Two-level ragged allele strings on the device (reference `_FlatAlleles`, _flat_variants.py:70-188): allele a of
    the batch is `data[seq_offsets[a]:seq_offsets[a+1]]`, row r owns alleles `var_offsets[r]:var_offsets[r+1]`."""

    data: torch.Tensor         # uint8 bytes
    seq_offsets: torch.Tensor  # int64 (n_alleles + 1,)
    var_offsets: torch.Tensor  # int64 (n_rows + 1,)
    shape: tuple

    def reshape(self, shape) -> "RaggedAlleles":
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        return RaggedAlleles(self.data, self.seq_offsets, self.var_offsets, shape + (None,))

    def to_list(self) -> list:
        """Host copy as nested lists of `bytes` (tests, debugging)."""
        d, so, vo = self.data.cpu().numpy().tobytes(), self.seq_offsets.cpu().numpy(), self.var_offsets.cpu().numpy()
        return [[d[so[a]:so[a + 1]] for a in range(vo[r], vo[r + 1])] for r in range(len(vo) - 1)]


@dataclass(frozen=True)
class RaggedVariants:
    """The `variants` output (reference `RaggedVariants` / `_FlatVariants`, _rag_variants.py, _flat_variants.py:405-535):
    one ragged field per requested name, all sharing `offsets` (variants per (b, p) row).  Scalar fields are `Ragged`
    (int32 `start`, `ilen`; 4-byte info columns), `alt` / `ref` are `RaggedAlleles`."""

    fields: dict
    offsets: torch.Tensor
    shape: tuple

    def __getitem__(self, name: str):
        return self.fields[name]

    def __getattr__(self, name: str):
        f = object.__getattribute__(self, "fields")
        if name in f:
            return f[name]
        raise AttributeError(name)

    @property
    def lengths(self) -> torch.Tensor:
        outer = tuple(d for d in self.shape if d is not None)
        return (self.offsets[1:] - self.offsets[:-1]).reshape(outer)

    def reshape(self, shape) -> "RaggedVariants":
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        return RaggedVariants({k: v.reshape(shape) for k, v in self.fields.items()}, self.offsets, shape + (None,))

    def squeeze(self, axis=None) -> "RaggedVariants":
        outer = [d for d in self.shape if d is not None]
        if axis is None:
            outer = [d for d in outer if d != 1]
        else:
            if outer[axis] != 1:
                raise ValueError(f"cannot squeeze axis {axis} with size {outer[axis]}")
            del outer[axis]
        return self.reshape(tuple(outer))


@dataclass(frozen=True)
class RaggedIntervals:
    """The `with_tracks(kind="intervals")` output: per (..., track) cell, the stored intervals that overlap the read's
    window, in ascending position, clipped to it, in absolute 0-based reference coordinates.  Three `Ragged` fields share
    `offsets` (intervals per cell): `starts` and `ends` int32, `values` of the dataset's track dtype."""

    starts: Ragged
    ends: Ragged
    values: Ragged

    @property
    def offsets(self) -> torch.Tensor:
        return self.starts.offsets

    @property
    def shape(self) -> tuple:
        return self.starts.shape

    @property
    def lengths(self) -> torch.Tensor:
        return self.starts.lengths

    def reshape(self, shape) -> "RaggedIntervals":
        return RaggedIntervals(self.starts.reshape(shape), self.ends.reshape(shape), self.values.reshape(shape))

    def squeeze(self, axis=None) -> "RaggedIntervals":
        return RaggedIntervals(self.starts.squeeze(axis), self.ends.squeeze(axis), self.values.squeeze(axis))

    def to_list(self) -> list:
        """Host copy: one list of (start, end, value) per cell, cells in row-major order (tests, debugging)."""
        s, e = self.starts.data.cpu().tolist(), self.ends.data.cpu().tolist()
        v, o = self.values.data.float().cpu().tolist(), self.offsets.cpu().tolist()
        return [list(zip(s[a:b], e[a:b], v[a:b])) for a, b in zip(o[:-1], o[1:])]


def build_token_lut(alphabet, unknown_token: int):
    """256-entry byte -> token table (reference `build_token_lut`, _flat_flanks.py:23-40): byte i of the alphabet maps to
    token i, every other byte (N, padding outside the contig) to `unknown_token`; uint8 when every token fits, else int32."""
    alphabet = alphabet.encode("ascii") if isinstance(alphabet, str) else bytes(alphabet)
    max_token = max(len(alphabet) - 1, int(unknown_token))
    dtype = np.uint8 if max_token <= 255 else np.int32
    lut = np.full(256, unknown_token, dtype=dtype)
    for i, b in enumerate(alphabet):
        lut[b] = i
    return lut, np.dtype(dtype)


@dataclass(frozen=True)
class VarWindowOpt:
    """Options of `with_seqs("variant-windows")` (reference `VarWindowOpt`, _flat_variants.py:291-321): "window" emits the
    flanked, tokenised window (ref: the reference read [start - L, end + L); alt: flank5 . alt . flank3), "allele" the bare
    tokenised allele."""

    flank_length: int
    token_alphabet: Any
    unknown_token: int
    ref: str = "window"
    alt: str = "window"

    def __post_init__(self):
        a = self.token_alphabet
        object.__setattr__(self, "token_alphabet", a.encode("ascii") if isinstance(a, str) else bytes(a))
        if self.ref not in ("window", "allele") or self.alt not in ("window", "allele"):
            raise ValueError("VarWindowOpt.ref / .alt must be 'window' or 'allele'")
