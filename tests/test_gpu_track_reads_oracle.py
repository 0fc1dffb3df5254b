"""Dense track reads of a `Dataset` against the oracle (tests/_track_reads.py), over a seeded sweep of read states.

Every case reads one state twice -- on whichever path serves it (the fixed-length pipeline when
`_pipeline.supports(ds)` is None, else the general path) and on the general path forced -- and compares both with the
restatement at 0 ulp: float32 bits, except NaNs computed by an arithmetic insertion fill (Repeat5pNormalized,
Interpolate), which are compared as NaN.  Subsets of the cases also check the outputs derived from the dense read
against the oracle's values: 16-bit stores (host rounding), binned tracks (the exact definition) and the two interval
kinds (painted back).

The dataset has six sample tracks, two annotation tracks and the `edge` track (edge float32 values, long negative runs,
2**20 + k/8 runs).  The annotation tracks hold one slot per (region, sample) of which the first n_regions are read, so a
read that took a dataset index as an annotation slot would read other values, not outside the table."""
from __future__ import annotations

import numpy as np
import pytest

from tests import _track_reads as TR

pytestmark = pytest.mark.gpu

N_REGIONS, N_SAMPLES, REGION_LEN, MAX_JITTER = 10, 4, 320, 8
SAMPLE_TRACKS = tuple(f"track{i}" for i in range(6))
ANNOT_TRACKS = ("annot0", "annot1")
ALL_TRACKS = SAMPLE_TRACKS + ANNOT_TRACKS + ("edge",)
FIXED = (256, 257, 264, 320, 321, 328, 336)      # below / equal to / above the region; L % 16 of 0, 1 and 8
LENGTHS = FIXED + ("ragged", "variable")
FILLS = ("Repeat5p", "Repeat5pNormalized", "Constant(nan)", "Constant(-2.5)", "FlankSample", "Interpolate(1)",
         "Interpolate(2)", "Interpolate(3)")
READS = ("pairs", "grid", "int", "subset", "batch<=256", "batch>256")
SEQS = ("haplotypes", "annotated", None, "reference")


# ---------------------------------------------------------------------------------------------------------------------
# the cases
# ---------------------------------------------------------------------------------------------------------------------
def _valid(c: dict) -> dict:
    """Make a case a valid state: the window fits the jitter, exonic filtering needs the SVAR1 source."""
    if isinstance(c["length"], int):
        while c["length"] + 2 * c["jitter"] > REGION_LEN + 2 * MAX_JITTER:
            c["jitter"] = {MAX_JITTER: 1, 1: 0}[c["jitter"]]
    if c["exonic"]:
        c["source"] = "svar1"
    return c


def _random_case(k: int) -> dict:
    rng = np.random.default_rng(7000 + k)
    pick = lambda xs: xs[int(rng.integers(0, len(xs)))]
    n_t = 9 if rng.random() < 0.1 else int(rng.integers(1, 4))
    tracks = ALL_TRACKS if n_t == 9 else tuple(rng.choice(ALL_TRACKS, n_t, replace=False).tolist())
    return _valid(dict(name=f"random{k}", source="svar2" if rng.random() < 0.25 else "svar1", seqs=pick(SEQS),
                       realign=bool(rng.random() < 0.75), length=pick(LENGTHS), jitter=pick((0, 1, MAX_JITTER)),
                       deterministic=bool(rng.random() < 0.5), rc_neg=bool(rng.random() < 0.7),
                       exonic=bool(rng.random() < 0.2), tracks=tracks,
                       fills=tuple(pick(FILLS) for _ in tracks), read=pick(READS), seed=int(rng.integers(0, 1 << 30))))


_BASE = dict(source="svar1", seqs="haplotypes", realign=True, length=320, jitter=1, deterministic=True, rc_neg=True,
             exonic=False, tracks=("track0", "annot0", "edge"), fills=("Repeat5p", "Interpolate(2)", "Constant(nan)"),
             read="pairs", seed=11)


def _named_cases() -> list:
    """For every value of every axis, one case built around it on the fast path where it can be (the fixed-length
    pipeline) and one on the general path; the sweep adds the combinations."""
    out = []
    axes = dict(source=("svar1", "svar2"), seqs=SEQS, realign=(True, False), length=LENGTHS, jitter=(0, 1, MAX_JITTER),
                deterministic=(True, False), rc_neg=(True, False), exonic=(False, True), n_tracks=(1, 2, 3, 9),
                kind=("sample", "annot", "edge"), fill=FILLS, read=READS)
    for axis, values in axes.items():
        for v in values:
            for general in (False, True):
                c = dict(_BASE, name=f"{axis}={v}{'-general' if general else ''}", seed=100 + len(out))
                if axis == "n_tracks":
                    c["tracks"] = ALL_TRACKS if v == 9 else ("edge", "annot1", "track3")[:v]
                elif axis == "kind":
                    c["tracks"] = {"sample": ("track2",), "annot": ("annot1",), "edge": ("edge",)}[v]
                elif axis == "fill":
                    c["tracks"], c["fills"] = ("edge", "track1"), (v, v)
                else:
                    c[axis] = v
                if axis == "deterministic" and not v and not general:
                    c["seqs"] = None  # random shifts leave the fast path; random draws without them do not
                if general and axis not in ("length", "exonic") and not (axis == "n_tracks" and v == 9):
                    c["length"] = "ragged" if c["seqs"] in ("haplotypes", "annotated") else "variable"
                c = _valid(c)
                c["fills"] = tuple(c["fills"][i % len(c["fills"])] for i in range(len(c["tracks"])))
                out.append(c)
    # random shifts: fixed-length realigned haplotypes with deterministic=False (general path), below and above the region
    for L in (264, 336):
        out.append(_valid(dict(_BASE, name=f"shifts-{L}", length=L, jitter=MAX_JITTER, deterministic=False,
                               seed=200 + L)))
    # the loader's cases: one per kind of sequence, jitter 0, deterministic
    for s in SEQS:
        out.append(dict(_BASE, name=f"loader-{s}", seqs=s, jitter=0, length=264, loader=True, seed=5))
    return out


CASES = _named_cases() + [_random_case(k) for k in range(120)]


def _fill(name: str):
    import genvarloader_b200 as G

    if name.startswith("Constant"):
        return G.Constant(float(name[9:-1]))
    if name.startswith("Interpolate"):
        return G.Interpolate(int(name[12]))
    if name == "FlankSample":
        return G.FlankSample(3)
    return getattr(G, name)()


def expect_fast(c: dict) -> bool:
    """The fixed-length pipeline serves fixed-length, unfiltered reads of at most 8 tracks, without random shifts."""
    hap = c["seqs"] in ("haplotypes", "annotated")
    return (isinstance(c["length"], int) and not c["exonic"] and len(c["tracks"]) <= 8
            and not (hap and not c["deterministic"]))


def _realigns(c: dict) -> bool:
    return c["seqs"] in ("haplotypes", "annotated") and c["realign"]


def _axis_values(c: dict) -> set:
    vals = {("source", c["source"]), ("seqs", c["seqs"]), ("length", c["length"]), ("jitter", c["jitter"]),
            ("deterministic", c["deterministic"]), ("rc_neg", c["rc_neg"]), ("exonic", c["exonic"]),
            ("n_tracks", len(c["tracks"])), ("read", c["read"])}
    if c["seqs"] in ("haplotypes", "annotated"):
        vals.add(("realign", c["realign"]))
    if isinstance(c["length"], int):  # realigned and painted reads each at every place of the length against the region
        place = "below" if c["length"] < REGION_LEN else "equal" if c["length"] == REGION_LEN else "above"
        vals.add(("realigned length", (_realigns(c), place)))
    if _realigns(c) and isinstance(c["length"], int) and not c["deterministic"]:
        vals.add(("random shifts", True))
    for t in c["tracks"]:
        vals.add(("kind", "edge" if t == "edge" else "annot" if t.startswith("annot") else "sample"))
    if _realigns(c):
        vals |= {("fill", f) for f in c["fills"]}
    return vals


def test_every_axis_value_on_every_path():
    """Every axis value occurs in some case (every case is also read on the general path) and, where the fixed-length
    pipeline can serve it, in a case it serves."""
    every = {("source", v) for v in ("svar1", "svar2")} | {("seqs", v) for v in SEQS} | {("realign", v) for v in (True, False)}
    every |= {("length", v) for v in LENGTHS} | {("jitter", v) for v in (0, 1, MAX_JITTER)}
    every |= {(a, v) for a in ("deterministic", "rc_neg", "exonic") for v in (True, False)}
    every |= {("n_tracks", v) for v in (1, 2, 3, 9)} | {("kind", v) for v in ("sample", "annot", "edge")}
    every |= {("fill", v) for v in FILLS} | {("read", v) for v in READS}
    every |= {("realigned length", (r, p)) for r in (True, False) for p in ("below", "equal", "above")}
    every |= {("random shifts", True)}
    not_fast = {("length", "ragged"), ("length", "variable"), ("exonic", True), ("n_tracks", 9), ("random shifts", True)}
    seen = {"fast": set(), "general": set()}
    for c in CASES:
        v = _axis_values(c)
        seen["general"] |= v
        if expect_fast(c):
            seen["fast"] |= v
    assert not every - seen["general"], sorted(every - seen["general"], key=str)
    assert not (every - not_fast) - seen["fast"], sorted((every - not_fast) - seen["fast"], key=str)
    assert sum(1 for c in CASES if c["name"].startswith("random")) == 120


# ---------------------------------------------------------------------------------------------------------------------
# the dataset
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def env(cuda_device):
    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset
    from oracle import oracle as O

    d = synth.make_dataset(41, 60_000, N_SAMPLES, N_REGIONS, REGION_LEN, 8.0, max_jitter=MAX_JITTER, neg_strand_frac=0.5,
                           straddle_ends=False, n_tracks=len(SAMPLE_TRACKS), max_indel=12, snp_frac=0.5)
    rng = np.random.default_rng(43)
    for name in ANNOT_TRACKS:
        d.tracks[name] = synth.make_track(rng, d.regions, N_SAMPLES, MAX_JITTER, mean_run=17)
    d.tracks["edge"] = TR.make_edge_track(rng, d.regions, N_SAMPLES, MAX_JITTER)
    kinds = {n: ("annot" if n in ANNOT_TRACKS else "sample") for n in d.tracks}
    assert tuple(d.tracks) == ALL_TRACKS
    ds1 = Dataset.from_arrays(cuda_device, d.reference, d.ref_offsets, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                              d.geno_v_idxs, d.geno_offsets, d.regions, N_SAMPLES, d.ploidy, MAX_JITTER, d.tracks,
                              track_kinds=kinds)
    ds2 = Dataset.from_svar2_arrays(cuda_device, d.reference, d.ref_offsets, synth.to_svar2_dataset(d), d.regions, N_SAMPLES,
                                    d.ploidy, MAX_JITTER, d.tracks, track_kinds=kinds)
    return d, kinds, {"svar1": ds1, "svar2": ds2}, O


def _state(c: dict) -> TR.ReadState:
    fills = {}
    for t, f in zip(c["tracks"], c["fills"]):
        s = _fill(f)
        fills[t] = (s.strategy_id, s.param())
    return TR.ReadState(seqs=c["seqs"], realign=c["realign"], length=c["length"], jitter=c["jitter"],
                        deterministic=c["deterministic"], rc_neg=c["rc_neg"], exonic=c["exonic"], tracks=tuple(c["tracks"]),
                        fills=fills if _realigns(c) else {})


def _dataset(env, c: dict):
    _, _, dss, _ = env
    ds = dss[c["source"]].with_seqs(c["seqs"]).with_tracks(list(c["tracks"]), kind="tracks").with_len(c["length"])
    ds = ds.with_settings(jitter=c["jitter"], deterministic=c["deterministic"], rc_neg=c["rc_neg"],
                          var_filter="exonic" if c["exonic"] else False, realign_tracks=c["realign"])
    if _realigns(c):
        ds = ds.with_insertion_fill({t: _fill(f) for t, f in zip(c["tracks"], c["fills"])})
    return ds


def _index(c: dict):
    """(dataset view to read, index, flat dataset indices over the full grid, outer shape of the output)."""
    rng = np.random.default_rng(c["seed"] + 1)
    S = N_SAMPLES
    read = c["read"]
    if read == "grid":
        r0, s0 = int(rng.integers(0, N_REGIONS - 2)), int(rng.integers(0, S - 1))
        r1, s1 = int(rng.integers(r0 + 1, N_REGIONS + 1)), int(rng.integers(s0 + 1, S + 1))
        ds_idx = (np.arange(r0, r1)[:, None] * S + np.arange(s0, s1)[None, :]).ravel()
        return None, (slice(r0, r1), slice(s0, s1)), ds_idx, (r1 - r0, s1 - s0)
    if read == "int":
        r, s = int(rng.integers(0, N_REGIONS)), int(rng.integers(0, S))
        return None, (r, s), np.array([r * S + s]), ()
    if read == "subset":
        ri = rng.permutation(N_REGIONS)[: int(rng.integers(2, N_REGIONS))]
        si = rng.permutation(S)[: int(rng.integers(1, S + 1))]
        n = int(rng.integers(1, 30))
        r, s = rng.integers(0, ri.size, n), rng.integers(0, si.size, n)
        return (ri, si), (r, s), ri[r] * S + si[s], (n,)
    n = {"pairs": int(rng.integers(1, 40)), "batch<=256": int(rng.integers(255, 257)),
         "batch>256": int(rng.integers(257, 261))}[read]
    r, s = rng.integers(0, N_REGIONS, n), rng.integers(0, S, n)
    return None, (r, s), r * S + s, (n,)


def _tracks(out):
    return out[-1] if isinstance(out, tuple) else out


def _got(trk, exp: TR.TrackRead, outer, length, bits=False):
    """The read's values in the restatement's cell order -> flat float32 (or the raw bits of any dtype), checking the
    shape and, for ragged reads, the offsets."""
    import torch

    def raw(x):
        x = x.contiguous()
        if bits:
            return x.view(torch.int32 if x.dtype == torch.float32 else torch.int16).cpu().numpy().view(
                np.uint32 if x.dtype == torch.float32 else np.uint16)
        return x.cpu().numpy()

    inner = exp.cells[1:]
    if length == "ragged":
        assert tuple(trk.shape) == (*outer, *inner, None), (trk.shape, outer, inner)
        assert np.array_equal(trk.offsets.cpu().numpy(), exp.offsets)
        return raw(trk.data).reshape(-1), exp.data
    want = exp.dense()
    assert tuple(trk.shape) == (*outer, *inner, want.shape[-1]), (tuple(trk.shape), outer, want.shape)
    return raw(trk).reshape(-1), want.reshape(-1)


def _nan_class(exp: TR.TrackRead, length):
    if length != "variable":
        return exp.nan_class
    lens = np.diff(exp.offsets)
    L = int(lens.max())
    out = np.zeros((lens.size, L), bool)
    out[np.arange(L)[None, :] < lens[:, None]] = exp.nan_class
    return out.reshape(-1)


def _read(ds, sub, idx, seed, fast: bool | None):
    from genvarloader_b200 import _pipeline

    if sub is not None:
        ds = ds.subset_to(regions=sub[0], samples=sub[1])
    ds = ds.with_settings(rng=seed)
    if fast is False:
        ds._cache["fast"] = False
    else:
        fast = _pipeline.supports(ds) is None
    out = ds[idx]
    assert ds._cache.get("fast") == fast and (("pipe" in ds._cache) == fast), ds._cache.keys()
    return out, fast


def _check(env, c: dict, ds, sub, idx, ds_idx, outer, st, exp):
    fast = None
    for force in (None, False):
        out, served = _read(ds, sub, idx, c["seed"], force)
        if force is None:
            assert served == expect_fast(c), (c["name"], served)
            fast = served
        got, want = _got(_tracks(out), exp, outer, c["length"])
        TR.assert_f32(got, want, _nan_class(exp, c["length"]), f"{c['name']} fast={force is None and fast}")
    return fast


# ---------------------------------------------------------------------------------------------------------------------
# the sweep
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_dense_read_matches_oracle(env, c):
    import torch

    d, kinds, _, O = env
    ds = _dataset(env, c)
    sub, idx, ds_idx, outer = _index(c)
    st = _state(c)
    exp = TR.read_tracks(O, d, kinds, st, ds_idx, c["seed"])
    _check(env, c, ds, sub, idx, ds_idx, outer, st, exp)
    k = CASES.index(c)

    # 16-bit stores: a host rounding of the oracle's float32 values
    if k % 3 == 0:
        for dt, name in ((torch.bfloat16, "bfloat16"), (torch.float16, "float16")):
            out, _ = _read(ds.with_track_dtype(dt), sub, idx, c["seed"], None)
            got_bits, want = _got(_tracks(out), exp, outer, c["length"], bits=True)
            TR.assert_narrowed(got_bits, want, name, f"{c['name']} {name}")

    # binned tracks: the exact definition on the oracle's values
    L = c["length"]
    if isinstance(L, int) and len(ds_idx) <= 64 and k % 2 == 0:
        divs = [B for B in (2, 4, 8, 16, 32, 64) if L % B == 0]
        if divs:
            B = divs[k % len(divs)]
            reduce = ("sum", "mean", "max")[k % 3]
            dt, name = ((torch.float32, "float32"), (torch.bfloat16, "bfloat16"), (torch.float16, "float16"))[(k // 3) % 3]
            for force in (None, False):
                out, _ = _read(ds.with_track_dtype(dt).with_track_bins(B, reduce), sub, idx, c["seed"], force)
                trk = _tracks(out)
                assert tuple(trk.shape) == (*outer, *exp.cells[1:], L // B)
                raw = trk.contiguous()
                raw = raw.view(torch.int32 if dt == torch.float32 else torch.int16).cpu().numpy()
                raw = raw.view(np.uint32 if dt == torch.float32 else np.uint16).reshape(-1)
                TR.assert_bins(raw, exp.data.reshape(-1, L), B, reduce, name, f"{c['name']} bins {B} {reduce} {name}")
                if force is None:
                    first = raw
                else:
                    assert np.array_equal(first, raw), "the two paths' bins differ"

    # intervals, painted back over each cell's window
    if k % 3 == 1 and c["read"] != "int":
        _check_intervals(env, c, ds, sub, idx, outer, exp)


def _check_intervals(env, c, ds, sub, idx, outer, exp):
    from genvarloader_b200._types import RaggedIntervals

    _, _, _, O = env
    kind = "realigned-intervals" if _realigns(c) else "intervals"
    if kind == "intervals" and c["seqs"] in ("haplotypes", "annotated"):
        ds = ds.with_settings(realign_tracks=False)
    if c["length"] == "variable" and kind == "intervals":
        return
    out, _ = _read(ds.with_tracks(list(c["tracks"]), kind=kind), sub, idx, c["seed"], None)
    got = _tracks(out)
    assert isinstance(got, RaggedIntervals)
    n_cells = int(np.prod(exp.cells))
    off = got.offsets.cpu().numpy().reshape(-1)
    assert off.size == n_cells + 1
    buf = np.zeros(int(exp.offsets[-1]), np.float32)
    O.intervals_to_tracks(np.arange(n_cells), exp.w0, got.starts.data.cpu().numpy(), got.ends.data.cpu().numpy(),
                          got.values.data.cpu().numpy(), off, buf, exp.offsets)
    O.reverse_flat_rows_inplace(buf, exp.offsets, exp.rc)
    TR.assert_f32(buf, exp.data, exp.nan_class, f"{c['name']} {kind}")


# ---------------------------------------------------------------------------------------------------------------------
# the loader: every batch against the oracle for its indices
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seqs", SEQS, ids=[str(s) for s in SEQS])
def test_loader_batches_match_oracle(env, seqs):
    d, kinds, _, O = env
    c = next(c for c in CASES if c["name"] == f"loader-{seqs}")
    ds = _dataset(env, c)
    st = _state(c)
    n = 0
    for batch in ds.to_dataloader(batch_size=7, shuffle=True, generator=3, return_indices=True):
        r, s = batch[-2], batch[-1]
        ds_idx = np.asarray(r) * N_SAMPLES + np.asarray(s)
        exp = TR.read_tracks(O, d, kinds, st, ds_idx, 0)
        got, want = _got(batch[-3], exp, (len(ds_idx),), c["length"])
        TR.assert_f32(got, want, exp.nan_class, f"loader {seqs}")
        n += len(ds_idx)
    assert n == N_REGIONS * N_SAMPLES


# ---------------------------------------------------------------------------------------------------------------------
# the edge track, binned: all-negative bins, bins exact in float64 but not in float32
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype_name", ["float32", "bfloat16", "float16"])
@pytest.mark.parametrize("reduce", ["sum", "mean", "max"])
@pytest.mark.parametrize("realign", [True, False])
def test_edge_track_bins(env, realign, reduce, dtype_name):
    import torch

    d, kinds, dss, O = env
    c = dict(_BASE, name="edge-bins", tracks=("edge",), fills=("Repeat5p",), realign=realign, length=256, jitter=0,
             read="pairs", seed=3)
    ds = _dataset(env, c)
    r = np.repeat(np.arange(N_REGIONS), N_SAMPLES)
    s = np.tile(np.arange(N_SAMPLES), N_REGIONS)
    exp = TR.read_tracks(O, d, kinds, _state(c), r * N_SAMPLES + s, 3)
    x = exp.data.reshape(-1, 8)
    assert (x < 0).all(1).sum() > 50, "too few all-negative bins"
    assert sum(TR.exactly_summable(v) and (v >= 2.0 ** 20).all() for v in x) > 50, "too few 2**20 + k/8 bins"
    dt = getattr(torch, dtype_name)
    totals = []
    for B in (8, 16):
        out, _ = _read(ds.with_track_dtype(dt).with_track_bins(B, reduce), None, (r, s), 3, None)
        raw = _tracks(out).contiguous()
        raw = raw.view(torch.int32 if dt == torch.float32 else torch.int16).cpu().numpy()
        raw = raw.view(np.uint32 if dt == torch.float32 else np.uint16).reshape(-1)
        totals.append(TR.assert_bins(raw, exp.data.reshape(-1, 256), B, reduce, dtype_name, f"edge {B} {reduce}"))
    assert all(exact > 0 for _, exact in totals)


@pytest.mark.parametrize("length", [328, 336])
def test_realigned_rows_past_the_track_window(env, length):
    """A fixed length above the region length (possible when jitter < max_jitter) makes realigned rows longer than
    the track window of their query (the region less its longest net deletion); large random shifts carry rows past it
    too.  Past the window a row reads 0.0 (src/tracks/mod.rs:381-404), also where the stored interval that ends at the
    window's end is followed by one that starts there."""
    d, kinds, _, O = env
    c = _valid(dict(_BASE, name=f"past-window-{length}", length=length, jitter=0, tracks=("edge", "track0", "annot0")))
    ds = _dataset(env, c)
    sub, idx, ds_idx, outer = _index(c)
    exp = TR.read_tracks(O, d, kinds, _state(c), ds_idx, c["seed"])
    assert (exp.dense()[..., REGION_LEN + 4:] == 0).any()  # rows reach past their window
    for force in (None, False):
        out, _ = _read(ds, sub, idx, c["seed"], force)
        got, want = _got(_tracks(out), exp, outer, length)
        TR.assert_f32(got, want, exp.nan_class, c["name"])


def test_edge_values_reach_every_read(env):
    """The edge track's stored values come back bit for bit from a painted read of every slot (NaN payloads, -0.0,
    subnormals and infinities included): neither the upload nor the kernels change them."""
    d, kinds, dss, O = env
    s_, e_, v_, io = d.tracks["edge"]
    for ds in dss.values():
        out = ds.with_seqs(None).with_tracks(["edge"]).with_settings(rc_neg=False)[:, :]
        got = out.data.cpu().numpy().view(np.uint32)
        seen = set(got.tolist())
        for x in TR.EDGE_SPECIALS:
            assert int(np.float32(x).view(np.uint32)) in seen, hex(int(np.float32(x).view(np.uint32)))
