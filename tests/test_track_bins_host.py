"""Binned tracks (`Dataset.with_track_bins`) without a GPU: the state rules and their messages, the shapes a binned read
returns, and the C ABI surface (GVL_TRACK_REDUCE_*, the two binned entries, the trailing fields of gvl_fixed_job)."""
import ctypes
import re
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")
from genvarloader_b200._dataset import Dataset  # noqa: E402
from genvarloader_b200._types import Ragged  # noqa: E402
from genvarloader_b200 import _pipeline  # noqa: E402

ROOT = Path(__file__).resolve().parent.parent


def _ds(R=6, S=3, L=4200, max_jitter=4, tracks=True):
    regions = np.stack([np.zeros(R), np.arange(R) * 10_000, np.arange(R) * 10_000 + L, np.ones(R)], 1).astype(np.int32)
    kinds = {"t0": "sample", "t1": "annot"} if tracks else {}
    return Dataset(engine=None, full_regions=regions, sample_names=tuple(f"s{i}" for i in range(S)), ploidy=2,
                   max_jitter=max_jitter, track_kinds=kinds, active_tracks=tuple(kinds))


def test_defaults_and_evolution():
    ds = _ds()
    assert (ds.track_bin, ds.track_reduce) == (1, "mean")
    assert "track_bins" not in repr(ds)
    b = ds.with_len(4096).with_track_bins(32, "max")
    assert (b.track_bin, b.track_reduce) == (32, "max") and (ds.track_bin, ds.track_reduce) == (1, "mean")
    assert "track_bins=32 (max)" in repr(b)
    assert b.with_track_bins(32).track_reduce == "mean"
    assert b.with_track_bins(1).track_bin == 1
    # other settings keep it
    assert b.with_seqs("reference").with_settings(jitter=2).with_track_dtype(torch.float16).track_bin == 32
    # bin 1 restores the unbinned default in every state, also those that refuse bins
    assert _ds().with_track_bins(1).track_bin == 1


@pytest.mark.parametrize("bad", [0, 3, 6, 48, 8192, -2, 2.0, True, "32", None])
def test_bin_size_must_be_a_power_of_two_up_to_4096(bad):
    ds = _ds().with_len(4096)
    with pytest.raises(ValueError, match="power of two from 2 to 4096"):
        ds.with_track_bins(bad)


@pytest.mark.parametrize("bin_size", [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096])
def test_every_power_of_two_is_accepted(bin_size):
    assert _ds().with_len(4096).with_track_bins(bin_size).track_bin == bin_size


@pytest.mark.parametrize("bad", ["median", "min", "MEAN", None, 0])
def test_reduction_must_be_mean_sum_or_max(bad):
    with pytest.raises(ValueError, match='"mean", "sum" or "max"'):
        _ds().with_len(4096).with_track_bins(32, bad)


def test_needs_tracks():
    with pytest.raises(ValueError, match="no tracks"):
        _ds(tracks=False).with_len(4096).with_track_bins(32)


def test_needs_a_fixed_length_first():
    ds = _ds()
    for length in ("ragged", "variable"):
        with pytest.raises(ValueError, match=r"with_len\(<multiple of 32>\) before with_track_bins\(32\)"):
            ds.with_len(length).with_track_bins(32)
    b = ds.with_len(4096).with_track_bins(32)
    for length in ("ragged", "variable"):
        with pytest.raises(ValueError, match="fixed output length"):
            b.with_len(length)
    assert b.with_track_bins(1).with_len("ragged").output_length == "ragged"


def test_length_must_be_a_multiple_of_the_bin():
    ds = _ds()
    with pytest.raises(ValueError, match=r"multiple of the track bin size \(32\): use with_len\(4128\)"):
        ds.with_len(4100).with_track_bins(32)
    b = ds.with_len(4096).with_track_bins(32)
    with pytest.raises(ValueError, match="multiple of the track bin size"):
        b.with_len(4010)
    assert b.with_len(4064).output_length == 4064
    assert ds.with_len(4100).with_track_bins(4).track_bin == 4


def test_only_kind_tracks():
    ds = _ds().with_len(4096).with_settings(realign_tracks=False)
    with pytest.raises(ValueError, match="kind='tracks' only"):
        ds.with_tracks(kind="intervals").with_track_bins(32)
    with pytest.raises(ValueError, match="kind='tracks' only"):
        ds.with_track_bins(32).with_tracks(kind="intervals")
    with pytest.raises(ValueError, match="kind='tracks' only"):
        ds.with_settings(realign_tracks=True).with_seqs("haplotypes").with_track_bins(32).with_tracks(kind="realigned-intervals")


def test_not_spliced():
    ds = _ds().with_len(4096)
    b = ds.with_track_bins(32)
    with pytest.raises(ValueError, match="spliced output is ragged"):
        b.with_settings(splice_info={"a": [0, 1], "b": [2]})


def test_ffi_codes():
    from genvarloader_b200._engine import track_bin_codes

    assert track_bin_codes(1, "mean") == (1, 0)
    assert track_bin_codes(32, "sum") == (32, 1)
    assert track_bin_codes(np.int64(4096), "max") == (4096, 2)


# ---- shapes ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seqs,realign", [("haplotypes", True), ("annotated", True), ("haplotypes", False), ("reference", False),
                                          (None, False)])
@pytest.mark.parametrize("bin_size", [2, 128])
def test_pipeline_buffers_and_views(seqs, realign, bin_size):
    """The fixed-length pipeline's track buffers hold L // bin values per row and its results view them as
    (b, t, p, L // bin) realigned or (b, t, L // bin) painted tracks; sequences keep L."""
    L, b = 1024, 3
    ds = _ds().with_len(L).with_seqs(seqs).with_settings(realign_tracks=realign).with_track_bins(bin_size)
    sp = _pipeline._Spec(ds)
    assert sp.realign == (realign and seqs in ("haplotypes", "annotated")) and sp.Lt == L // bin_size
    out = _pipeline._Out(sp, b, torch.device("cpu"))
    res = out.result()
    trk = res[-1] if isinstance(res, tuple) else res
    assert trk.shape == ((b, 2, 2, L // bin_size) if sp.realign else (b, 2, L // bin_size))
    if seqs is not None:
        seq = res[0].haps if seqs == "annotated" else res[0]
        assert seq.shape[-1] == L


def test_general_path_shapes():
    """The general path's Ragged tracks (offsets already divided by the bin) become (..., L // bin); sequences keep L."""
    L, B, b, t, p = 64, 8, 2, 2, 2
    ds = _ds().with_len(L).with_track_bins(B)
    trk = Ragged(torch.arange(b * t * p * L // B, dtype=torch.float32), torch.arange(b * t * p + 1) * (L // B), (b, t, p, None))
    assert ds._shape_output(trk, None, False).shape == (b, t, p, L // B)
    assert ds._shape_output(trk, (1, 2), False).shape == (1, 2, t, p, L // B)
    one = Ragged(torch.zeros(t * p * L // B, dtype=torch.bfloat16), torch.arange(t * p + 1) * (L // B), (1, t, p, None))
    assert ds._shape_output(one, None, True).shape == (t, p, L // B)
    seq = Ragged(torch.zeros(b * p * L, dtype=torch.uint8), torch.arange(b * p + 1) * L, (b, p, None))
    assert ds._shape_output(seq, None, False).shape == (b, p, L)


# ---- C ABI -----------------------------------------------------------------------------------------------------
def _header():
    return re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "gvl_b200.h").read_text(), flags=re.S)


def _n_params(name):
    m = re.search(rf"\b{name}\s*\(([^)]*)\)\s*;", _header())
    assert m, f"{name} is not declared in gvl_b200.h"
    return len(m.group(1).split(","))


def test_constants_match_the_header():
    from genvarloader_b200 import _ffi

    h = (ROOT / "include" / "gvl_b200.h").read_text()
    val = lambda n: int(re.search(rf"#define {n} (\d+)", h).group(1))
    assert (val("GVL_TRACK_REDUCE_MEAN"), val("GVL_TRACK_REDUCE_SUM"), val("GVL_TRACK_REDUCE_MAX")) == (
        _ffi.TRACK_REDUCE_MEAN, _ffi.TRACK_REDUCE_SUM, _ffi.TRACK_REDUCE_MAX)
    assert val("GVL_TRACK_BIN_MAX") == _ffi.TRACK_BIN_MAX == 4096


@pytest.mark.parametrize("name,n", [("gvl_dev_realign_tracks_exec_binned", 6), ("gvl_dev_paint_tracks_binned", 17)])
def test_binned_entries_are_declared_and_exported(name, n):
    from genvarloader_b200 import _ffi

    assert _n_params(name) == n
    fn = getattr(_ffi.lib, name)
    assert len(fn.argtypes) == n
    # the entries they extend keep their prototypes
    base = name.replace("_binned", "")
    assert _n_params(base) == n - 2 and len(getattr(_ffi.lib, base).argtypes) == n - 2


def test_binned_entries_reject_a_null_context():
    from genvarloader_b200 import _ffi

    for name in ("gvl_dev_realign_tracks_exec_binned", "gvl_dev_paint_tracks_binned"):
        fn = getattr(_ffi.lib, name)
        args = [0 if t in (ctypes.c_int64, ctypes.c_int32) else None for t in fn.argtypes]
        assert fn(*args) == 2, name
        assert b"NULL" in _ffi.lib.gvl_last_error(), name


def test_fixed_job_matches_the_header():
    """_ffi.FixedJob mirrors gvl_fixed_job field by field, the two binning fields last."""
    from genvarloader_b200 import _ffi

    body = re.search(r"typedef struct gvl_fixed_job \{(.*?)\} gvl_fixed_job;", _header(), flags=re.S).group(1)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?\w+\s*\**", "", decl)  # drop the type
        names += [re.sub(r"[\s*]", "", n) for n in decl.split(",")]
    assert names == [f[0] for f in _ffi.FixedJob._fields_]
    assert names[-2:] == ["track_bin", "track_reduce"]
    assert _ffi.FixedJob.track_bin.size == 4 and _ffi.FixedJob.track_reduce.size == 4
    job = _ffi.FixedJob()
    assert (job.track_bin, job.track_reduce) == (0, 0)  # zero = unbinned
