"""Track outputs in bfloat16 and float16 (`Dataset.with_track_dtype`, GVL_TRACK_*).

One rule, checked everywhere: a 16-bit read returns bit for bit `x.to(dtype)` of the float32 output `x` of the same call,
cast on the device (round to nearest even, float16 overflow to inf, subnormals kept, the device's canonical NaN).  Every
comparison is `torch.equal` on the raw 16 bits.  Where the float32 path has an oracle, the oracle's float32 values cast on
the device are compared as well.

  1. every tile path of the track execute (single pass at tile edges, TD_BIG sub-passes and the hand-over after a long
     deletion, TD_GENERIC, all five fills, 9 tracks, per-row destinations, painted rows), asserted through
     gvl_debug_track_tiles, on the geometry dataset of tests/test_gpu_track_paths.py;
  2. stores stay inside their rows: rows at every residue mod 16 elements, separated by guard elements;
  3. every Dataset read path: fixed length (haplotypes, annotated, tracks only, reference), jitter and negative strands,
     ragged and variable, spliced, svar2, the read-ahead loader and host delivery;
  4. one full-size batch of the cfg3t shape;
  5. the API: invalid dtypes, datasets without tracks, float32 unchanged, an unknown dtype code at the C ABI."""
from __future__ import annotations

import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from tests.test_gpu_track_paths import (BOTH, CROSS, EDGE_F, EDGE_F_END, EDGE_RC1, EDGE_RC2, EDGE_RC3, EMPTY, LIM_A_F,
                                        LIM_A_RC, LIM_B_F, LIM_B_RC, LONG_INS_F, LONG_INS_RC, N_TRACKS, SHORT_RC, TD_BIG,
                                        TD_GENERIC, TD_RC, TILE, WIDE_RC, _fast, _fills, _tiles, _with_jumps,
                                        geometry_dataset, handover_tiles, tiles)

pytestmark = pytest.mark.gpu
DTYPES = [torch.bfloat16, torch.float16]
IDS = ["bf16", "f16"]
SENT16 = 0x7FA1  # a NaN in both 16-bit types that no kernel writes (not the canonical one)


@pytest.fixture(scope="module")
def O():
    from oracle import oracle

    return oracle


@pytest.fixture(scope="module")
def G():
    return geometry_dataset()


def _bits(x: torch.Tensor) -> torch.Tensor:
    return x.contiguous().view(torch.int16)


def assert_cast(got, ref, dtype):
    """`got` (16-bit track output: Ragged or tensor) is `ref` (the same read in float32) cast on the device."""
    from genvarloader_b200._types import Ragged

    if isinstance(ref, Ragged):
        assert isinstance(got, Ragged) and got.shape == ref.shape and torch.equal(got.offsets, ref.offsets)
        got, ref = got.data, ref.data
    assert ref.dtype == torch.float32 and got.dtype == dtype and got.shape == ref.shape, (got.dtype, got.shape, ref.shape)
    assert got.device.type == "cuda" and ref.device.type == "cuda"
    assert torch.equal(_bits(got), _bits(ref.to(dtype)))


def _same(a, b) -> bool:
    """Exact equality of non-track outputs (tensors, Ragged, annotated haplotypes)."""
    if isinstance(a, torch.Tensor):
        return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)
    if dataclasses.is_dataclass(a):
        return type(a) is type(b) and all(_same(getattr(a, f.name), getattr(b, f.name)) for f in dataclasses.fields(a))
    return a == b


def read_both(ds, idx, dtype):
    """ds[idx] in float32 and in `dtype`; asserts the rule on the tracks (the last output) and equality of the rest."""
    ref, got = ds[idx], ds.with_track_dtype(dtype)[idx]
    ref = ref if isinstance(ref, tuple) else (ref,)
    got = got if isinstance(got, tuple) else (got,)
    assert len(ref) == len(got)
    for a, b in zip(ref[:-1], got[:-1]):
        assert _same(a, b)
    assert_cast(got[-1], ref[-1], dtype)
    return got[-1], ref[-1]


def _oracle_cast(exp, dtype):
    """Oracle float32 buffers cast on the device, widened back to float32 (exact), for the float32 row checkers."""
    return [torch.from_numpy(e).cuda().to(dtype).float().cpu().numpy() for e in exp]


def _widened(r):
    from genvarloader_b200._types import Ragged

    return Ragged(r.data.float(), r.offsets, r.shape)


# ---------------------------------------------------------------------------------------------------------------------
# 1. every tile path
# ---------------------------------------------------------------------------------------------------------------------
def _geometry_ds(dev, d, names, fills):
    from genvarloader_b200._dataset import Dataset

    return Dataset.from_synth(dev, d, rng=0).with_tracks(names).with_insertion_fill(dict(zip(names, fills)))


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
def test_tile_paths_realigned(cuda_device, G, O, dtype):
    """9 tracks with every fill (Constant with its default NaN, Interpolate of orders 1-3) over rows that put tiles on
    edges of forward and reverse rows, at and past the staging limits (TD_BIG), and the hand-over after a deletion that
    skips every staged interval; then the same slots as spliced rows (per-row destinations)."""
    import genvarloader_b200 as m
    from tests.test_gpu_spliced_tracks import _check_realigned, _element_batch, _oracle_realigned, _seed

    d, slots = G
    names = [f"t{i}" for i in range(N_TRACKS)]
    fills = _fills(m, N_TRACKS)
    fills[2] = m.Constant()  # the default value: NaN
    assert np.isnan(fills[2].value) and {type(f).__name__ for f in fills} >= {"Repeat5p", "Repeat5pNormalized", "Constant",
                                                                              "FlankSample", "Interpolate"}
    ds = _geometry_ds(cuda_device, d, names, fills)
    ks = np.array([EDGE_F, EDGE_RC1, EDGE_RC2, EDGE_RC3, SHORT_RC, WIDE_RC, EDGE_F_END, EMPTY, LIM_A_F, LIM_A_RC, LIM_B_F,
                   LIM_B_RC, BOTH, CROSS, LONG_INS_F, LONG_INS_RC])
    r, s = ks // 2, ks % 2
    got, _ = read_both(ds, (r, s), dtype)
    t = _tiles(ds.engine.ctx.handle)
    assert set(t[:, 0].tolist()) == set(range(N_TRACKS))
    t0 = t[t[:, 0] == 0]
    rc_rows = {int(x[1]) for x in t0 if x[4] & TD_RC}
    for q in range(4):  # the edge rows: every tile a single pass, reversed exactly on the negative strand
        for h in range(2):
            row = 2 * q + h
            rt = t0[t0[:, 1] == row]
            assert len(rt) and all(_fast(x) for x in rt) and (row in rc_rows) == (d.regions[r[q], 3] == -1), row
    assert (t0[:, 4] & TD_BIG).any() and ((t0[:, 4] & TD_GENERIC) == 0).all()
    both_q = int(np.flatnonzero(ks == BOTH)[0])
    for p in range(2):  # the hand-over tile of the BOTH slot is finished in sub-passes
        assert 2 * TILE in handover_tiles(d, slots, BOTH, p)
        sel = t0[(t0[:, 1] == 2 * both_q + p) & (t0[:, 2] == 2 * TILE)]
        assert len(sel) == 1 and sel[0][4] & TD_BIG, sel
    exp, oo = _oracle_realigned(d, O, r, s, fills, names, _seed(r, s, d.n_samples))
    assert np.isnan(exp[2]).any()  # the NaN fill is written somewhere
    _check_realigned(_widened(got), _oracle_cast(exp, dtype), oo, np.ones(ks.size, np.int64), d.ploidy)

    rows = {"a": [0, 4], "b": [2, 1, 6], "c": [3], "d": [7, 5, 0]}
    pairs = [(0, 0), (1, 1), (2, 0), (3, 1), (1, 0)]
    idx = ([p[0] for p in pairs], [p[1] for p in pairs])
    got, _ = read_both(ds.with_settings(splice_info=rows), idx, dtype)
    t = _tiles(ds.engine.ctx.handle)
    assert (t[:, 4] & TD_BIG).any() and (t[:, 4] & TD_RC).any()
    e_reg, e_s, n_el = _element_batch(d, rows, pairs)
    exp, oo = _oracle_realigned(d, O, e_reg, e_s, fills, names, _seed(e_reg, e_s, d.n_samples))
    _check_realigned(_widened(got), _oracle_cast(exp, dtype), oo, n_el, d.ploidy)


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
def test_tile_paths_generic(cuda_device, G, O, dtype):
    """Variant lists out of position order (jump records): those rows take TD_GENERIC in every tile, per value."""
    import genvarloader_b200 as m
    from tests.test_gpu_spliced_tracks import _check_realigned, _oracle_realigned, _seed

    d, _ = G
    ks = np.array([LIM_A_F, WIDE_RC, BOTH, CROSS])
    dj = _with_jumps(d, ks[:3])
    names, fills = ["t0", "t4"], [m.Interpolate(2), m.FlankSample(5)]
    ds = _geometry_ds(cuda_device, dj, names, fills)
    r, s = ks // 2, ks % 2
    got, _ = read_both(ds, (r, s), dtype)
    t = _tiles(ds.engine.ctx.handle)
    for row in range(2 * len(ks)):
        rt = t[(t[:, 0] == 0) & (t[:, 1] == row)]
        want = row % 2 == 0 and row < 6
        assert len(rt) and all(bool(x[4] & TD_GENERIC) == want for x in rt), (row, rt)
    exp, oo = _oracle_realigned(dj, O, r, s, fills, names, _seed(r, s, d.n_samples))
    _check_realigned(_widened(got), _oracle_cast(exp, dtype), oo, np.ones(ks.size, np.int64), d.ploidy)


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
def test_tile_paths_painted(cuda_device, G, O, dtype):
    """Painted rows at tile edges, reversed, 9 tracks: the (b, t, ~l) layout and spliced rows (per-row destinations)."""
    from genvarloader_b200._dataset import Dataset
    from tests.test_gpu_spliced_tracks import _check_painted, _element_batch, _oracle_painted

    d, _ = G
    names = [f"t{i}" for i in range(N_TRACKS)]
    ds = Dataset.from_synth(cuda_device, d, rng=0).with_tracks(names).with_settings(realign_tracks=False)
    q = np.array([EDGE_F, EDGE_RC1, EDGE_RC2, WIDE_RC, EMPTY, SHORT_RC, LIM_A_RC])
    r, sm = q // 2, q % 2
    got, _ = read_both(ds, (r, sm), dtype)
    t = _tiles(ds.engine.ctx.handle)
    for row, k in enumerate(q):
        rc = bool(d.regions[k // 2, 3] == -1)
        L = int(d.regions[k // 2, 2] - d.regions[k // 2, 1])
        rt = t[(t[:, 0] == 0) & (t[:, 1] == row)]
        assert sorted((int(x[2]), int(x[3])) for x in rt) == sorted(tiles(L, rc))
        assert all(bool(x[4] & TD_RC) == rc and _fast(x) for x in rt)
    exp, offs = _oracle_painted(d, O, r, sm, names)
    _check_painted(_widened(got), _oracle_cast(exp, dtype), offs, np.ones(q.size, np.int64))
    rows = {"a": [1, 4, 2], "b": [5], "c": [0, 3]}
    pairs = [(0, 1), (1, 0), (2, 1), (0, 0)]
    got, _ = read_both(ds.with_settings(splice_info=rows, realign_tracks=False), ([p[0] for p in pairs], [p[1] for p in pairs]),
                       dtype)
    e_reg, e_s, n_el = _element_batch(d, rows, pairs)
    exp, offs_e = _oracle_painted(d, O, e_reg, e_s, names)
    _check_painted(_widened(got), _oracle_cast(exp, dtype), offs_e, n_el)


# ---------------------------------------------------------------------------------------------------------------------
# 2. stores stay inside their rows
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
def test_stores_stay_in_bounds(cuda_device, G, dtype):
    """Painted rows written through a destination table that leaves 1-16 guard elements after every row and puts row
    starts and ends at every residue mod 16 elements (so every row starts and ends inside a 16-value chunk): every row value is
    written (no sentinel left) and equals the float32 call cast on the device; no guard element changes."""
    from genvarloader_b200._dataset import Dataset

    d, _ = G
    ds = Dataset.from_synth(cuda_device, d, rng=0).with_tracks(["t2"])
    eng = ds.engine
    rng = np.random.default_rng(11)
    n = 64
    k = rng.integers(0, 16, n)
    i = np.arange(n)
    base = rng.integers(16, 60, n)
    base[::4] = rng.integers(TILE - 20, 2 * TILE + 20, base[::4].size)  # rows over tile edges too
    L = base - base % 16 + (i // 4 - i) % 16  # row i ends at residue i // 4 ...
    dst = np.zeros(n, np.int64)
    for k_ in range(1, n):  # ... and starts at residue i, after 1 to 16 guard elements
        end = int(dst[k_ - 1] + L[k_ - 1])
        dst[k_] = end + ((k_ - end) % 16 or 16)
    assert set((dst % 16).tolist()) == set(range(16)) and set(((dst + L) % 16).tolist()) == set(range(16))
    size = int(dst[-1] + L[-1]) + 40
    starts = (d.regions[k // 2, 1] + rng.integers(-30, 30, n)).astype(np.int32)
    to_rc = (d.regions[k // 2, 3] == -1).astype(np.uint8)
    oo = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    args = (["t2"], dv(k.astype(np.int64)[None, :]), dv(starts), dv(oo), size, dv(to_rc))
    rows = dict(layout="rows", row_dst=dv(dst), row_tstride=torch.zeros(n, dtype=torch.int64, device=cuda_device))
    ref = torch.empty(size, dtype=torch.float32, device=cuda_device)
    ref.view(torch.int32).fill_(0x7FBADBAD)
    eng.paint_tracks(*args, out=ref, **rows)
    got = torch.empty(size, dtype=dtype, device=cuda_device)
    got.view(torch.int16).fill_(SENT16)
    eng.paint_tracks(*args, out=got, **rows)
    torch.cuda.synchronize()
    inside = np.zeros(size, bool)
    for a, b in zip(dst, dst + L):
        inside[a:b] = True
    inside_t = torch.from_numpy(inside).to(cuda_device)
    assert not (ref.view(torch.int32)[inside_t] == 0x7FBADBAD).any()  # float32: every row value written
    assert (ref.view(torch.int32)[~inside_t] == 0x7FBADBAD).all()
    g16 = got.view(torch.int16)
    assert not (g16[inside_t] == SENT16).any()  # every row value written ...
    assert (g16[~inside_t] == SENT16).all()  # ... and nothing around it
    assert torch.equal(g16[inside_t], _bits(ref[inside_t].to(dtype)))


# ---------------------------------------------------------------------------------------------------------------------
# 3. every Dataset read path
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env(cuda_device):
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset

    d = synth.make_dataset(91, 300_000, 4, 11, 2000 + 2 * 12, 6.0, max_jitter=12, neg_strand_frac=0.5, straddle_ends=False,
                           n_tracks=2, max_indel=15, snp_frac=0.5)
    import genvarloader_b200 as m

    ds = Dataset.from_synth(cuda_device, d, rng=5).with_insertion_fill({"track0": m.Interpolate(3), "track1": m.FlankSample(3)})
    return d, ds


IDX = (np.array([0, 3, 5, 7, 10, 2]), np.array([1, 0, 3, 2, 1, 0]))


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
@pytest.mark.parametrize("kind", ["haplotypes", "annotated", None, "reference"])
def test_fixed_length(env, dtype, kind):
    """Fixed-length __getitem__ (the device-side batch path): haplotypes + tracks, annotated + tracks, tracks only and
    reference + tracks (painted); with jitter and negative strands; array, scalar and slice indices."""
    _, ds = env
    base = ds.with_seqs(kind).with_len(1500)
    for settings in (dict(rng=1), dict(jitter=12, rng=2), dict(jitter=7, rng=3, rc_neg=False)):
        dsx = base.with_settings(**settings)
        for idx in (IDX, (4, 1), (slice(2, 6), slice(None))):
            # (two datasets with the same seed: both reads draw the same jitter)
            a = dsx.with_settings(rng=settings["rng"])
            b = dsx.with_track_dtype(dtype).with_settings(rng=settings["rng"])
            ra, rb = a[idx], b[idx]
            ra, rb = (ra if isinstance(ra, tuple) else (ra,)), (rb if isinstance(rb, tuple) else (rb,))
            for x, y in zip(ra[:-1], rb[:-1]):
                assert _same(x, y)
            assert_cast(rb[-1], ra[-1], dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
@pytest.mark.parametrize("length", ["ragged", "variable"])
def test_ragged_and_variable(env, dtype, length):
    """Ragged and variable-length reads, realigned and painted: `variable` pads tracks with 0 in the track dtype."""
    _, ds = env
    for dsx in (ds.with_len(length), ds.with_len(length).with_settings(realign_tracks=False), ds.with_len(length).with_seqs(None),
                ds.with_len(length).with_settings(jitter=9)):
        # (two datasets with the same seed: both reads draw the same jitter)
        a = dsx.with_settings(rng=4)[IDX]
        b = dsx.with_track_dtype(dtype).with_settings(rng=4)[IDX]
        a, b = (a if isinstance(a, tuple) else (a,)), (b if isinstance(b, tuple) else (b,))
        assert all(_same(x, y) for x, y in zip(a[:-1], b[:-1]))
        assert_cast(b[-1], a[-1], dtype)  # variable: the float32 read pads with 0.0, so the padding is +0 in the dtype
        assert isinstance(b[-1], torch.Tensor) == (length == "variable")


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
def test_spliced(env, dtype):
    """Spliced datasets, realigned and painted tracks: every cell the concatenation of its elements, in the dtype."""
    _, ds = env
    rows = {"a": [3, 0, 7], "b": [5], "c": [10, 2, 10], "d": [1, 4, 9, 6]}
    sp = ds.with_settings(splice_info=rows)
    for dsx in (sp, sp.with_settings(realign_tracks=False), sp.with_seqs(None), sp.with_seqs("reference")):
        read_both(dsx, ([0, 2, 3, 1], [1, 0, 3, 2]), dtype)
        read_both(dsx, (slice(None), slice(None)), dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
def test_svar2_source(cuda_device, dtype):
    """An svar2-backed dataset with tracks: fixed length (device batch path) and ragged (plan + execute entries)."""
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset

    d = synth.make_dataset(23, 400_000, 4, 10, 3000 + 2 * 8, 6.0, max_jitter=8, neg_strand_frac=0.5, straddle_ends=False,
                           n_tracks=1, max_indel=20, snp_frac=0.5)
    sv = synth.to_svar2_dataset(d, dense_frac=0.5, seed=4)
    ds = Dataset.from_synth(cuda_device, d, rng=9, svar2=sv)
    idx = (np.array([0, 4, 9, 2]), np.array([3, 1, 0, 2]))
    read_both(ds.with_len(2000), idx, dtype)
    read_both(ds.with_len("ragged"), idx, dtype)
    read_both(ds.with_len("variable").with_settings(realign_tracks=False), idx, dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=IDS)
@pytest.mark.parametrize("copy", [False, True])
def test_loader(env, dtype, copy):
    """to_dataloader(mode="double_buffered"): rings in the dtype, batch for batch equal to __getitem__ of the same indices
    (and that to the float32 read cast on the device)."""
    _, ds = env
    for dsx in (ds.with_len(1200), ds.with_len(1200).with_seqs("reference"), ds.with_len(1200).with_seqs(None)):
        d16 = dsx.with_track_dtype(dtype)
        n = 0
        for batch in d16.to_dataloader(batch_size=5, mode="double_buffered", copy=copy, ring=2, return_indices=True):
            *outs, r, s = batch
            assert outs[-1].dtype == dtype
            ref16 = d16[r, s]
            ref16 = ref16 if isinstance(ref16, tuple) else (ref16,)
            assert all(_same(x, y) for x, y in zip(outs, ref16))
            ref32 = dsx[r, s]
            assert_cast(outs[-1], (ref32 if isinstance(ref32, tuple) else (ref32,))[-1], dtype)
            n += len(r)
        assert n == len(dsx)


def test_to_host(env):
    """to_host=True: float16 tracks arrive as numpy float16 equal to the device read; bfloat16 raises (numpy has none)."""
    _, ds = env
    dsx = ds.with_len(1000)
    h16 = dsx.with_track_dtype(torch.float16)
    for batch in h16.to_dataloader(batch_size=4, mode="double_buffered", copy=True, ring=2, to_host=True, return_indices=True):
        *outs, r, s = batch
        assert isinstance(outs[-1], np.ndarray) and outs[-1].dtype == np.float16
        ref = h16[r, s][-1]
        assert np.array_equal(outs[-1].view(np.int16), _bits(ref).cpu().numpy())
        assert np.array_equal(outs[0], dsx[r, s][0].cpu().numpy())
    with pytest.raises(ValueError, match="bfloat16"):
        dsx.with_track_dtype(torch.bfloat16).to_dataloader(batch_size=4, mode="double_buffered", to_host=True)


# ---------------------------------------------------------------------------------------------------------------------
# 4. one full-size batch
# ---------------------------------------------------------------------------------------------------------------------
def test_full_size_batch(cuda_device):
    """The cfg3t shape: 16 (region, sample) pairs x ploidy 2 = 32 rows x 524,288 values x 2 realigned tracks (Repeat5p,
    Interpolate(1)), jitter 128, half the regions on the negative strand; in bfloat16 and float16."""
    import genvarloader_b200 as m
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset

    L = 524_288
    d = synth.make_dataset(3, 4_000_000, 4, 6, L + 2 * 128, 1.0, max_jitter=128, snp_frac=0.8, neg_strand_frac=0.5,
                           straddle_ends=False, n_tracks=2, fast_tracks=True)
    ds = (Dataset.from_synth(cuda_device, d, rng=0).with_len(L).with_encoding("onehot")
          .with_insertion_fill({"track0": m.Repeat5p(), "track1": m.Interpolate(1)}))
    rng = np.random.default_rng(1)
    r, s = rng.integers(0, d.n_regions, 16), rng.integers(0, d.n_samples, 16)
    for dtype in DTYPES:
        a = ds.with_settings(jitter=128, rng=5)[r, s]
        b = ds.with_track_dtype(dtype).with_settings(jitter=128, rng=5)[r, s]
        assert b[1].shape == (16, 2, 2, L)
        assert _same(a[0], b[0])
        assert_cast(b[1], a[1], dtype)


# ---------------------------------------------------------------------------------------------------------------------
# 5. the API
# ---------------------------------------------------------------------------------------------------------------------
def test_api(env, cuda_device):
    from genvarloader_b200 import _ffi, synth
    from genvarloader_b200._dataset import Dataset
    from genvarloader_b200._engine import _stream
    from genvarloader_b200._pipeline import FixedPipeline

    d, ds = env
    for bad in (torch.float64, torch.int16, torch.uint8, "bfloat16", np.float16, None):
        with pytest.raises(ValueError, match="track dtype"):
            ds.with_track_dtype(bad)
    d0 = synth.make_dataset(5, 100_000, 2, 3, 500, 2.0)
    with pytest.raises(ValueError, match="no tracks"):
        Dataset.from_synth(cuda_device, d0).with_track_dtype(torch.bfloat16)
    # float32 is the default: the same dataset state, the same bytes
    f32 = ds.with_track_dtype(torch.float32)
    assert f32 == ds and ds.track_dtype == torch.float32 and "track_dtype=torch.float32" in repr(ds)
    assert "track_dtype=torch.bfloat16" in repr(ds.with_track_dtype(torch.bfloat16))
    for dsx, idx in ((ds.with_len(900), IDX), (ds, IDX), (ds.with_settings(splice_info={"a": [1, 2]}), (0, 1))):
        x, y = dsx.with_settings(rng=3)[idx], dsx.with_track_dtype(torch.float32).with_settings(rng=3)[idx]
        assert all(_same(p, q) for p, q in zip(x, y))
    # unknown dtype codes at the C ABI
    h = ds.engine.ctx.handle
    buf = torch.empty(64, dtype=torch.float32, device=cuda_device)
    for code in (3, -1):
        assert _ffi.lib.gvl_dev_realign_tracks_exec_dtype(h, _ffi.ptr(buf), code, _stream()) == 2
        assert b"unknown track dtype" in _ffi.lib.gvl_last_error()
    itv = ds.engine.track_descs(["track0"])[0]
    z64 = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    z32 = torch.zeros(1, dtype=torch.int32, device=cuda_device)
    rc = _ffi.lib.gvl_dev_paint_tracks_dtype(h, 1, itv, _ffi.ptr(z64), _ffi.ptr(z32), 1, _ffi.ptr(z64), 1, None, None, None,
                                             _ffi.ptr(buf), 7, _stream())
    assert rc == 2 and b"unknown track dtype" in _ffi.lib.gvl_last_error()
    pipe = FixedPipeline(ds.with_len(800).with_track_dtype(torch.float16), 4)
    job = pipe._scr0.job
    assert job.track_dtype == _ffi.TRACK_F16
    job.track_dtype = 5
    try:
        rc = _ffi.lib.gvl_dev_fixed_plan(pipe.eng.ctx.handle, C.addressof(job), pipe._idx0.data_ptr(), None, 4, 0, _stream())
        assert rc == 2 and b"unknown track dtype" in _ffi.lib.gvl_last_error()
    finally:
        job.track_dtype = _ffi.TRACK_F16
