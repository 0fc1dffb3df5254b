"""Read-ahead loader for the `variants` / `variant-windows` outputs (`Dataset.to_dataloader(mode="buffered" |
"double_buffered")` on an unspliced variants state).

A variants read does a few microseconds of device work and hundreds of microseconds of host work (launches, allocations,
the wait for its sizes), so a batch-by-batch loader is bound by the host.  This loader amortises that host time over
`ring` batches: their genotype rows are read as ONE call -- one sizing pass (`gvl_dev_variant_row_sizes`) and its one
wait, then one variants tail over all K*b*p rows with every buffer sized on the host (`_variant_sizes.py`).  Rows are
independent and every step of the tail works per row or per folded cell, so batch i is cells [i*C, (i+1)*C) of the ring
(C = b*p, or b under `unphased_union`).  `gvl_dev_rebase_offsets` turns the ring's row offsets and each per-variant offsets
array into batch-local offsets, one launch per array.

Two rings are in flight, on two streams with a planning context each: while the consumer reads the batches of one ring,
the next one is produced.  Every ring gets freshly allocated buffers (a ring may hold more variants than the one before);
they are marked as used by the consumer's stream, so the allocator hands their memory out again only after the consumer's
work on them has finished.
"""
from __future__ import annotations

import numpy as np
import torch

from ._dataset import _as_rng, _batch_tail, _Packer, epoch_order

RING_VARIANTS = 1 << 20  # ring=0: batches per ring for about this many variants
RING_MAX = 64


def supports(ds) -> str | None:
    """None when `ds` can use the read-ahead variants loader, else the reason it cannot."""
    if ds.sequence_type not in ("variants", "variant-windows"):
        return "not a variants output"
    if ds.splice_rows is not None:
        return "spliced output"
    if ds.var_filter is not None:
        return "var_filter"
    if ds.active_tracks:
        return "tracks are active"
    if ds.engine.svar2 is not None:
        return "variants of the svar2 source"
    return None


def default_ring(ds, batch_size: int) -> int:
    """Batches per ring for about RING_VARIANTS variants, from the dataset's mean variants per genotype row (1 to
    RING_MAX)."""
    go = ds.engine.geno_offsets_host[:, :-1]  # (without the engine's empty slot)
    mean = float(np.maximum(go[1] - go[0], 0).mean()) if go.shape[1] else 0.0
    per_batch = batch_size * ds.ploidy * mean
    return int(min(max(np.ceil(RING_VARIANTS / max(per_batch, 1.0)), 1), RING_MAX))


class _Ring:
    """One device call: the tail's outputs over the ring's rows, the batch-local offsets and the host sizes."""

    __slots__ = ("g", "sizes", "off", "seq", "done", "chunk", "n_batches", "cells")


class VariantsLoader:
    """Re-iterable loader over an unspliced variants `Dataset` (see the module docstring and `Dataset.to_dataloader`)."""

    def __init__(self, ds, batch_size, shuffle, sampler, drop_last, generator, return_indices, transform, copy, ring):
        why = supports(ds)
        if why is not None:
            raise ValueError(f"the read-ahead variants loader does not apply: {why}")
        if batch_size < 1:
            raise ValueError("batch_size must be a positive integer")
        self.ds, self.batch_size, self.shuffle, self.sampler = ds, int(batch_size), shuffle, sampler
        self.drop_last, self.return_indices, self.transform, self.copy = drop_last, return_indices, transform, copy
        self._rng = _as_rng(generator)
        ring = int(ring) if ring else default_ring(ds, self.batch_size)
        self.ring = max(1, min(ring, -(-len(self) // 2)))  # (no more than half an epoch: both streams get work)
        self.dev = ds.engine.device
        self.cells_per_query = 1 if ds.unphased_union else ds.ploidy
        with torch.cuda.device(self.dev):
            self._halves = [(ds.engine.fork(), torch.cuda.Stream(self.dev)) for _ in range(2)]

    def __len__(self) -> int:
        n = len(self.sampler) if self.sampler is not None else len(self.ds)
        return n // self.batch_size if self.drop_last else -(-n // self.batch_size)

    def __iter__(self):
        b, K = self.batch_size, self.ring
        order = epoch_order(self.ds, self.sampler, self.shuffle, self._rng)
        n_batches = len(self)
        order = order[: n_batches * b]
        n_rings = -(-n_batches // K)
        rings = {i: self._submit(i % 2, order[i * K * b: (i + 1) * K * b]) for i in range(min(2, n_rings))}
        n_s = self.ds.n_samples
        for i in range(n_rings):
            ring = rings.pop(i)
            for j, batch in enumerate(self._acquire(ring)):
                c = ring.chunk[j * b: (j + 1) * b]
                yield _batch_tail(batch, (c // n_s, c % n_s) if self.return_indices else None, self.transform)
            if i + 2 < n_rings:
                rings[i + 2] = self._submit(i % 2, order[(i + 2) * K * b: (i + 3) * K * b])

    def _submit(self, h: int, chunk: np.ndarray) -> _Ring:
        """Produce the ring of the flat (subset) indices `chunk` on half h's stream; returns once its tail is enqueued."""
        ds, b, p = self.ds, self.batch_size, self.ds.ploidy
        eng, stream = self._halves[h]
        for lo in range(0, len(chunk), b):  # one jitter draw per batch, in batch order, as ds[r, s] makes them
            ds.rng.integers(-ds.jitter, ds.jitter + 1, size=min(b, len(chunk) - lo), dtype=np.int32)
        n_s = ds.n_samples
        r_full = ds._r_idx[chunk // n_s]
        goi = (r_full * len(ds.sample_names) + ds._s_idx[chunk % n_s])[:, None] * p + np.arange(p, dtype=np.int64)[None, :]
        pk = _Packer(self.dev)
        i_goi = pk.add(goi, np.int64)
        i_rc = pk.add(np.repeat(ds.full_regions[r_full, 3] == -1, p), np.uint8) if ds.rc_neg else None
        i_ct = pk.add(np.repeat(ds.full_regions[r_full, 0], p), np.int32) if ds._variant_tokens() is not None else None
        R = _Ring()
        R.chunk, R.n_batches, R.cells = chunk, -(-len(chunk) // b), b * self.cells_per_query
        with torch.cuda.device(self.dev), torch.cuda.stream(stream):
            pk.upload()
            get = lambda i: pk.get(i) if i is not None else None
            R.g, R.sizes = ds._gather_variants(eng, pk.get(i_goi), get(i_rc), get(i_ct), eng.max_records(goi))
            row_off = R.g["row_offsets"]
            R.off = eng.rebase_offsets(row_off, R.n_batches, R.cells)
            R.seq = {k: eng.rebase_offsets(v[1], R.n_batches, R.cells, bounds=row_off) for k, v in R.g.items() if isinstance(v, tuple)}
            R.done = torch.cuda.Event()
            R.done.record(stream)
        return R

    def _acquire(self, R: _Ring) -> list:
        """The batches of ring R for the current stream, which first waits for the ring."""
        cur = torch.cuda.current_stream(self.dev)
        cur.wait_event(R.done)
        for v in (*R.g.values(), R.off, *R.seq.values()):
            for t in v if isinstance(v, tuple) else (v,):
                t.record_stream(cur)
        ds, C, cp = self.ds, R.cells, self.cells_per_query
        n_cells = R.sizes.n_cells
        names = ds._variant_field_names(R.g)
        two_level = [k for k in names if isinstance(R.g[k], tuple)]
        vb = R.sizes.bounds("variants", C)
        ib = {k: R.sizes.bounds(k, C) for k in two_level}
        L2 = 2 * ds.flank_length if "flank_tokens" in names else 0
        cp_ = (lambda t: t.clone()) if self.copy else (lambda t: t)
        out = []
        for i in range(R.n_batches):
            c0, c1 = i * C, min((i + 1) * C, n_cells)
            v0, v1 = int(vb[i]), int(vb[i + 1])
            g = {}
            for k in names:
                x = R.g[k]
                if k in ib:
                    g[k] = (cp_(x[0][ib[k][i]: ib[k][i + 1]]), cp_(R.seq[k][v0 + i: v1 + i + 1]))
                elif k == "flank_tokens":
                    g[k] = cp_(x[v0 * L2: v1 * L2])
                else:
                    g[k] = cp_(x[v0:v1])
            off = cp_(R.off[c0 + i: c1 + i + 1])
            out.append(ds._variants_result(g, off, ((c1 - c0) // cp, cp, None)))
        return out
