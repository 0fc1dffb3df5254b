"""Binned tracks (`Dataset.with_track_bins`, the binned store of the track execute) on the GPU.

Every binned read is compared with the definition (DESIGN.md §7) applied to the unbinned float32 read of the same
dataset state and generator state: bin j of a row covers its output positions [j*bin, (j+1)*bin); `sum` = float64 sum
rounded to float32, `mean` = that sum / bin in float64 rounded to float32, `max` = the largest value, NaN first; then
narrowed to the track dtype.  `sum` and `mean` must lie within one unit in the last place of the output dtype (the
float64 order differs), `max` must be equal with NaNs in the same places.  Different paths of one state must agree bit
for bit."""
from __future__ import annotations

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REDUCES = ["mean", "sum", "max"]
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DT_IDS = ["f32", "bf16", "f16"]
IDX = (np.array([0, 3, 5, 7, 2, 6, 1]), np.array([1, 0, 3, 2, 1, 0, 2]))


def _int_view(x):
    return x.view(torch.int32) if x.dtype == torch.float32 else x.view(torch.int16)


def reference(x32: torch.Tensor, B: int, reduce: str, dtype) -> torch.Tensor:
    """The definition on an unbinned float32 output (last axis = output positions)."""
    assert x32.dtype == torch.float32
    xb = x32.unflatten(-1, (x32.shape[-1] // B, B))
    if reduce == "max":
        v = xb.amax(-1)  # (propagates NaN)
    else:
        s = xb.double().sum(-1)
        v = (s / B if reduce == "mean" else s).float()
    return v.to(dtype)


def assert_bins(got: torch.Tensor, x32: torch.Tensor, B: int, reduce: str, dtype):
    ref = reference(x32, B, reduce, dtype)
    assert got.dtype == dtype and got.shape == ref.shape, (got.dtype, got.shape, ref.shape)
    gn, rn = torch.isnan(got), torch.isnan(ref)
    assert torch.equal(gn, rn), "NaNs in different places"
    g, r = got[~gn], ref[~rn]
    if reduce == "max":
        assert torch.equal(g, r)
        return
    same = g == r
    # one unit in the last place: adjacent bit patterns of one sign
    gi, ri = _int_view(g.contiguous()).long(), _int_view(r.contiguous()).long()
    adjacent = ((gi - ri).abs() <= 1) & ((g >= 0) == (r >= 0))
    bad = ~(same | adjacent)
    assert not bad.any(), (g[bad][:8], r[bad][:8])


def _tracks_of(out):
    return out[-1] if isinstance(out, tuple) else out


def read_pair(ds, idx, B, reduce, dtype, seed=3):
    """(binned read, unbinned float32 read) of the same state and generator state."""
    x32 = _tracks_of(ds.with_track_dtype(torch.float32).with_settings(rng=seed)[idx])
    got_all = ds.with_track_dtype(dtype).with_track_bins(B, reduce).with_settings(rng=seed)[idx]
    return got_all, x32


@pytest.fixture(scope="module")
def env(cuda_device):
    """5 tracks (every insertion fill: Repeat5p, Repeat5pNormalized, Constant with its default NaN, FlankSample,
    Interpolate) plus one annotation track, mixed strands, regions long enough for two execute tiles."""
    import genvarloader_b200 as m
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset

    d = synth.make_dataset(17, 400_000, 4, 10, 16384 + 2 * 16, 6.0, max_jitter=16, neg_strand_frac=0.5, straddle_ends=False,
                           n_tracks=5, max_indel=15, snp_frac=0.5)
    rng = np.random.default_rng(4)
    d.tracks["annot0"] = synth.make_track(rng, d.regions, 1, 16, mean_run=12)
    kinds = {n: ("annot" if n == "annot0" else "sample") for n in d.tracks}
    fills = {"track0": m.Repeat5p(), "track1": m.Repeat5pNormalized(), "track2": m.Constant(), "track3": m.FlankSample(4),
             "track4": m.Interpolate(3)}
    assert np.isnan(fills["track2"].value)
    ds = Dataset.from_arrays(cuda_device, d.reference, d.ref_offsets, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                             d.geno_v_idxs, d.geno_offsets, d.regions, d.n_samples, d.ploidy, d.max_jitter, d.tracks,
                             track_kinds=kinds, rng=0)
    return d, ds.with_insertion_fill(fills).with_settings(jitter=5)


# ---------------------------------------------------------------------------------------------------------------------
# the definition: reductions x dtypes x bins, realigned and painted, on the fixed-length pipeline
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [2, 8, 32, 128, 4096])
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
@pytest.mark.parametrize("reduce", REDUCES)
def test_definition(env, reduce, dtype, B):
    _, ds = env
    ds = ds.with_len(16384)
    got, x32 = read_pair(ds, IDX, B, reduce, dtype)
    assert _tracks_of(got).shape == (len(IDX[0]), 6, 2, 16384 // B)
    assert torch.isnan(x32).any()  # the Constant fill's NaN reaches some bins
    assert_bins(_tracks_of(got), x32, B, reduce, dtype)


@pytest.mark.parametrize("kind", ["reference", None, "painted", "annotated"])
@pytest.mark.parametrize("reduce", REDUCES)
def test_kinds(env, kind, reduce):
    """Painted tracks (with_seqs(None), "reference", realign_tracks=False) and annotated haplotypes; the sequences of the
    same read are unchanged."""
    _, ds = env
    ds = ds.with_len(8192 + 1024)
    if kind == "painted":
        ds = ds.with_settings(realign_tracks=False)
    elif kind == "annotated":
        ds = ds.with_seqs("annotated")
    else:
        ds = ds.with_seqs(kind)
    for dtype in (torch.float32, torch.bfloat16):
        got, x32 = read_pair(ds, IDX, 64, reduce, dtype)
        realigned = kind == "annotated"
        assert _tracks_of(got).shape == ((7, 6, 2, 144) if realigned else (7, 6, 144))
        assert_bins(_tracks_of(got), x32, 64, reduce, dtype)
        if isinstance(got, tuple):
            ref = ds.with_settings(rng=3)[IDX]
            a, b = got[0], ref[0]
            a, b = (a.haps, b.haps) if kind == "annotated" else (a, b)
            assert torch.equal(a, b)


def test_length_not_a_multiple_of_16(env):
    """L % 16 == 8 with bin 8: the last 16-value chunk of every row is half outside the row."""
    _, ds = env
    ds = ds.with_len(8200)
    for reduce in REDUCES:
        for dtype in DTYPES:
            got, x32 = read_pair(ds, IDX, 8, reduce, dtype)
            assert_bins(_tracks_of(got), x32, 8, reduce, dtype)
            got, x32 = read_pair(ds.with_seqs(None), IDX, 8, reduce, dtype)
            assert_bins(_tracks_of(got), x32, 8, reduce, dtype)


def test_index_forms(env):
    _, ds = env
    b = ds.with_len(4096).with_track_bins(32)
    assert _tracks_of(b[3, 1]).shape == (6, 2, 128)
    assert _tracks_of(b[2:4, 1:3]).shape == (2, 2, 6, 2, 128)
    assert _tracks_of(b.with_seqs(None)[3, 1]).shape == (6, 128)


# ---------------------------------------------------------------------------------------------------------------------
# paths: the pipeline and the general path give identical bits
# ---------------------------------------------------------------------------------------------------------------------
def _general(ds):
    """The same state read through the general path (the fixed-length pipeline switched off for this dataset)."""
    ds._cache["fast"] = False
    return ds


@pytest.mark.parametrize("reduce", REDUCES)
def test_pipeline_and_general_path_agree(env, reduce):
    _, ds = env
    for seqs in ("haplotypes", "annotated", None):
        for dtype in (torch.float32, torch.float16):
            b = ds.with_len(8192 + 2048).with_seqs(seqs).with_track_dtype(dtype).with_track_bins(128, reduce)
            fast = _tracks_of(b.with_settings(rng=9)[IDX])
            gen = _tracks_of(_general(b.with_settings(rng=9))[IDX])
            assert torch.equal(_int_view(fast), _int_view(gen))


@pytest.mark.parametrize("reduce", REDUCES)
def test_general_path_states(env, reduce):
    """States the pipeline declines, against the definition: var_filter="exonic", deterministic=False, 9 tracks."""
    from genvarloader_b200 import _pipeline

    d, ds = env
    base = ds.with_len(4096 + 512)
    states = [base.with_settings(var_filter="exonic"), base.with_settings(deterministic=False)]
    nine = base.with_tracks(list(ds.track_kinds) + ["track0", "track1", "track2"])
    assert len(nine.active_tracks) == 9
    states.append(nine)
    for st in states:
        assert _pipeline.supports(st) is not None
        got, x32 = read_pair(st, IDX, 32, reduce, torch.bfloat16)
        assert_bins(_tracks_of(got), x32, 32, reduce, torch.bfloat16)
    # 9 tracks: the first 6 are those of the 6-track read of the pipeline, bit for bit
    a = _tracks_of(nine.with_track_bins(32, reduce).with_settings(rng=3)[IDX])
    b = _tracks_of(base.with_track_bins(32, reduce).with_settings(rng=3)[IDX])
    assert torch.equal(_int_view(a[:, :6]), _int_view(b))


@pytest.mark.parametrize("reduce", REDUCES)
def test_svar2_source(cuda_device, reduce):
    import genvarloader_b200 as m
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset

    d = synth.make_dataset(23, 200_000, 3, 6, 4096 + 64, 8.0, max_jitter=8, neg_strand_frac=0.5, straddle_ends=False,
                           n_tracks=2, max_indel=12)
    ds = Dataset.from_synth(cuda_device, d, rng=1, svar2=synth.to_svar2_dataset(d))
    ds = ds.with_insertion_fill({"track0": m.Interpolate(2), "track1": m.Constant()}).with_len(4096)
    idx = (np.array([0, 1, 2, 3, 4, 5]), np.array([0, 1, 2, 0, 1, 2]))
    for dtype in (torch.float32, torch.float16):
        got, x32 = read_pair(ds, idx, 16, reduce, dtype)
        assert_bins(_tracks_of(got), x32, 16, reduce, dtype)
        b = ds.with_track_dtype(dtype).with_track_bins(16, reduce)
        fast = _tracks_of(b.with_settings(rng=2)[idx])
        gen = _tracks_of(_general(b.with_settings(rng=2))[idx])
        assert torch.equal(_int_view(fast), _int_view(gen))


# ---------------------------------------------------------------------------------------------------------------------
# the read-ahead loader
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("copy", [False, True])
def test_loader(env, copy):
    _, ds = env
    for dsx in (ds.with_len(4096).with_settings(jitter=0), ds.with_len(4096).with_seqs(None).with_settings(jitter=0)):
        for dtype, reduce in ((torch.float32, "mean"), (torch.bfloat16, "max")):
            b = dsx.with_track_dtype(dtype).with_track_bins(64, reduce)
            n = 0
            for batch in b.to_dataloader(batch_size=6, mode="double_buffered", copy=copy, ring=2, return_indices=True):
                *outs, r, s = batch
                ref = b[r, s]
                ref = ref if isinstance(ref, tuple) else (ref,)
                assert outs[-1].shape[-1] == 64
                for x, y in zip(outs, ref):
                    assert torch.equal(_int_view(x) if x.is_floating_point() else x, _int_view(y) if y.is_floating_point() else y)
                n += len(r)
            assert n == len(dsx)


def test_loader_to_host(env):
    _, ds = env
    b = ds.with_len(4096).with_settings(jitter=0).with_track_dtype(torch.float16).with_track_bins(32, "sum")
    for batch in b.to_dataloader(batch_size=5, mode="double_buffered", copy=True, ring=2, to_host=True, return_indices=True):
        *outs, r, s = batch
        assert isinstance(outs[-1], np.ndarray) and outs[-1].dtype == np.float16 and outs[-1].shape[-1] == 128
        ref = b[r, s][-1]
        assert np.array_equal(outs[-1].view(np.int16), ref.view(torch.int16).cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------
# forced tile paths: TD_BIG sub-passes (bins straddle them) and TD_GENERIC
# ---------------------------------------------------------------------------------------------------------------------
def test_big_and_generic_tiles(cuda_device):
    """A track of 1-3 bp runs (thousands of stored intervals per tile: every tile is finished in sub-passes, TD_BIG) and
    rows whose variant lists leave jump records (`_with_jumps` of the tile-path tests: TD_GENERIC), asserted through
    gvl_debug_track_tiles."""
    import genvarloader_b200 as m
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset
    from tests.test_gpu_track_paths import TD_BIG, TD_GENERIC, _tiles, _with_jumps

    d = synth.make_dataset(31, 200_000, 2, 6, 12288 + 32, 10.0, max_jitter=16, neg_strand_frac=0.5, straddle_ends=False,
                           n_tracks=1, max_indel=10)
    d.tracks["fine"] = synth.make_track(np.random.default_rng(6), d.regions, d.n_samples, 16, mean_run=2)
    ks = np.array([0, 3, 6])
    dj = _with_jumps(d, ks)
    ds = Dataset.from_synth(cuda_device, dj, rng=0).with_insertion_fill({"track0": m.FlankSample(3), "fine": m.Interpolate(1)})
    ds = ds.with_len(12288)  # two tiles per row
    r = np.arange(12) // 2
    s = np.arange(12) % 2
    for B in (2, 16, 512, 4096):
        for reduce in REDUCES:
            got, x32 = read_pair(ds, (r, s), B, reduce, torch.float32)
            assert_bins(_tracks_of(got), x32, B, reduce, torch.float32)
            t = _tiles(ds.engine.ctx.handle)
            assert (t[:, 4] & TD_BIG).any() and (t[:, 4] & TD_GENERIC).any()
            for row in range(24):  # rows 2k (ploid 0) of the jump slots take the generic path
                rt = t[t[:, 1] == row]
                want = row % 2 == 0 and row // 2 in ks.tolist()
                assert len(rt) and all(bool(x[4] & TD_GENERIC) == want for x in rt), (row, rt)
            big = t[(t[:, 0] == 1) & ((t[:, 4] & TD_GENERIC) == 0)]
            assert len(big) and (big[:, 4] & TD_BIG).all()


# ---------------------------------------------------------------------------------------------------------------------
# stores stay inside the binned rows
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [2, 32, 4096])
def test_guard(env, cuda_device, B):
    """Painted rows through a destination table with guard elements between them: every bin is written and no guard
    element changes."""
    d, ds = env
    eng = ds.engine
    rng = np.random.default_rng(2)
    n = 12
    k = rng.integers(0, d.n_regions * d.n_samples, n)
    L = (rng.integers(1, 5, n) * max(B, 16) * 4).astype(np.int64)
    L[::3] = 8192 + B * (2 if B < 4096 else 1)
    gaps = rng.integers(1, 4, n) * B
    dst = np.zeros(n, np.int64)
    for i in range(1, n):
        dst[i] = dst[i - 1] + L[i - 1] + gaps[i]
    size = int(dst[-1] + L[-1] + 4 * B)
    starts = (d.regions[k // d.n_samples, 1]).astype(np.int32)
    to_rc = (d.regions[k // d.n_samples, 3] == -1).astype(np.uint8)
    oo = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    dv = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda_device)
    args = (["track0"], dv(k.astype(np.int64)[None, :]), dv(starts), dv(oo), size, dv(to_rc))
    rows = dict(layout="rows", row_dst=dv(dst), row_tstride=torch.zeros(n, dtype=torch.int64, device=cuda_device))
    x32 = eng.paint_tracks(*args, **rows)
    for dtype in (torch.float32, torch.bfloat16):
        out = torch.empty(size // B, dtype=dtype, device=cuda_device)
        iv = _int_view(out)
        iv.fill_(0x7FBADBAD if dtype == torch.float32 else 0x7FA1)
        sentinel = int(iv[0])
        eng.paint_tracks(*args, out=out, bin=B, reduce="sum", **rows)
        torch.cuda.synchronize()
        inside = np.zeros(size // B, bool)
        for a, l in zip(dst, L):
            inside[a // B:(a + l) // B] = True
        ins = torch.from_numpy(inside).to(cuda_device)
        assert not (iv[ins] == sentinel).any()
        assert (iv[~ins] == sentinel).all()
        for a, l in zip(dst, L):
            assert_bins(out[a // B:(a + l) // B], x32[a:a + l], B, "sum", dtype)


# ---------------------------------------------------------------------------------------------------------------------
# the C entries reject bad bins before any launch
# ---------------------------------------------------------------------------------------------------------------------
def test_bad_bins_at_the_c_entries(env, cuda_device):
    from genvarloader_b200 import _ffi

    _, ds = env
    h = ds.engine.ctx.handle
    out = torch.empty(64, device=cuda_device)
    for bin_, red in ((3, 0), (8192, 0), (-2, 0), (32, 3), (32, -1)):
        assert _ffi.lib.gvl_dev_realign_tracks_exec_binned(h, out.data_ptr(), 0, bin_, red, None) == 2
        assert b"track" in _ffi.lib.gvl_last_error()
