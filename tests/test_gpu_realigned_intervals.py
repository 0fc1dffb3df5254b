"""`with_tracks(kind="realigned-intervals")` (gvl_dev_realigned_track_intervals): every realigned row cut into the maximal
runs of positions that take their value from one stored interval or one insertion fill (DESIGN.md §7).  Checked exactly
against the numpy restatement of the definition (tests/_realigned_intervals.py), and through the painting invariant: the
intervals painted into zeros over each haplotype row and reversed where the strand mask is set are, bit for bit, the
`kind="tracks"` output of the same read from the same generator state."""
import numpy as np
import pytest

from tests import _realigned_intervals as RI

pytestmark = pytest.mark.gpu

MAX_JITTER = 8


def _overlap_track(rng, regions, n_slots_per_region, n=40):
    """Overlapping intervals in stored order (flattened at upload)."""
    s, e, counts = [], [], []
    for r in range(len(regions)):
        a, b = int(regions[r, 1]) - MAX_JITTER, int(regions[r, 2]) + MAX_JITTER
        for _ in range(n_slots_per_region):
            st = rng.integers(a - 20, b, n)
            s.append(st)
            e.append(st + rng.integers(1, 60, n))
            counts.append(n)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    s, e = np.concatenate(s).astype(np.int32), np.concatenate(e).astype(np.int32)
    return s, e, (rng.integers(1, 1000, s.size) / 8).astype(np.float32), off


@pytest.fixture(scope="module")
def env(cuda_device):
    from genvarloader_b200 import Dataset, synth

    d = synth.make_dataset(17, 60_000, 3, 12, 400, 6.0, neg_strand_frac=0.5, straddle_ends=True, n_tracks=3, max_indel=6)
    d.max_jitter = MAX_JITTER
    rng = np.random.default_rng(3)
    kinds = {f"track{i}": "sample" for i in range(3)}
    d.tracks["annot0"], kinds["annot0"] = synth.make_track(rng, d.regions, 1, MAX_JITTER, mean_run=12), "annot"
    d.tracks["short"], kinds["short"] = synth.make_track(rng, d.regions, d.n_samples, MAX_JITTER, mean_run=3), "sample"
    d.tracks["overlap"], kinds["overlap"] = _overlap_track(rng, d.regions, d.n_samples), "sample"
    ds = Dataset.from_arrays(cuda_device, d.reference, d.ref_offsets, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                             d.geno_v_idxs, d.geno_offsets, d.regions, d.n_samples, d.ploidy, d.max_jitter, d.tracks,
                             track_kinds=kinds, rng=0).with_seqs("haplotypes")
    return d, ds, kinds


R_IDX = np.array([0, 11, 4, 6, 1, 11, 9, 3, 0, 8])
S_IDX = np.array([0, 1, 2, 1, 0, 2, 2, 0, 1, 1])


def _jitter(ds, n, seed):
    return np.random.default_rng(seed).integers(-ds.jitter, ds.jitter + 1, size=n, dtype=np.int32)


def _values(x):
    import torch

    return x.to(torch.float32).cpu().numpy() if x.dtype != torch.float32 else x.cpu().numpy()


def _strip(out):
    """The track part of a read that returns (sequences, tracks)."""
    return out[1] if isinstance(out, tuple) else out


def _check_painting(got, trk, w0_cells, rc_cells):
    """Invariant 1: `got` (RaggedIntervals, cells in row-major order) painted into zeros of each cell's length (that of the
    tracks output `trk`, Ragged or dense), reversed on masked cells, is `trk` bit for bit.  Returns the interval count."""
    import torch

    if isinstance(trk, torch.Tensor):
        n_cells = int(np.prod(trk.shape[:-1]))
        L = trk.shape[-1]
        t_off = np.arange(n_cells + 1, dtype=np.int64) * L
        t_data = _values(trk.reshape(-1))
    else:
        t_off = trk.offsets.cpu().numpy().reshape(-1)
        t_data = _values(trk.data)
        n_cells = t_off.size - 1
    off = got.offsets.cpu().numpy().reshape(-1)
    assert off.size == n_cells + 1
    st, en, va = got.starts.data.cpu().numpy(), got.ends.data.cpu().numpy(), _values(got.values.data)
    assert got.starts.data.dtype == torch.int32 and got.ends.data.dtype == torch.int32
    for c in range(n_cells):
        a, b = off[c], off[c + 1]
        L = int(t_off[c + 1] - t_off[c])
        s, e = st[a:b], en[a:b]
        w0 = int(w0_cells[c])
        assert (e > s).all() and (s[1:] >= e[:-1]).all() and (s >= w0).all() and (e <= w0 + L).all(), c
        p = _paint(s, e, va[a:b], w0, L, bool(rc_cells[c]))
        assert np.array_equal(p.view(np.uint32), t_data[t_off[c]:t_off[c + 1]].view(np.uint32)), c
    return int(off[-1])


def _paint(s, e, v, w0, L, rc):
    """RI.paint without a Python loop over the intervals (sorted and disjoint)."""
    out = np.zeros(L, np.float32)
    n = (e - s).astype(np.int64)
    if n.size:
        first = np.concatenate([[0], np.cumsum(n)[:-1]])
        pos = np.arange(int(n.sum())) - np.repeat(first - (s.astype(np.int64) - w0), n)
        out[pos] = np.repeat(v, n)
    return out[::-1].copy() if rc else out


def _read_both(ds_, r, s, seed):
    trk = _strip(ds_.with_tracks(kind="tracks").with_settings(rng=seed)[r, s])
    got = _strip(ds_.with_tracks(kind="realigned-intervals").with_settings(rng=seed)[r, s])
    return got, trk


def _cells(d, ds_, r, seed, t, p, rc_neg):
    """Per (read, track, ploid) cell: w0 and the strand mask."""
    w0 = d.regions[r, 1].astype(np.int64) + _jitter(ds_, len(r), seed)
    rc = (d.regions[r, 3] == -1) if rc_neg else np.zeros(len(r), bool)
    return np.repeat(w0, t * p), np.repeat(rc, t * p)


@pytest.mark.parametrize("length", ["ragged", 300])
@pytest.mark.parametrize("jitter", [0, MAX_JITTER])
@pytest.mark.parametrize("rc_neg", [True, False])
def test_painting_invariant(env, length, jitter, rc_neg):
    d, ds, kinds = env
    ds_ = ds.with_len(length).with_settings(jitter=jitter, rc_neg=rc_neg)
    got, trk = _read_both(ds_, R_IDX, S_IDX, 5)
    t, p = len(kinds), d.ploidy
    assert got.shape == (len(R_IDX), t, p, None)
    w0, rc = _cells(d, ds_, R_IDX, 5, t, p, rc_neg)
    assert _check_painting(got, trk, w0, rc) > 100


def test_variable_length_returns_the_ragged_intervals(env):
    d, ds, kinds = env
    a = ds.with_len("variable").with_tracks(kind="realigned-intervals")[R_IDX, S_IDX][1]
    b = ds.with_len("ragged").with_tracks(kind="realigned-intervals")[R_IDX, S_IDX][1]
    assert a.to_list() == b.to_list()
    one = ds.with_tracks(kind="realigned-intervals")[3, 1][1]
    assert one.shape == (len(kinds), d.ploidy, None)
    assert one.to_list() == ds.with_tracks(kind="realigned-intervals")[[3], [1]][1].to_list()


@pytest.mark.parametrize("fill", ["Repeat5p", "Repeat5pNormalized", "Constant", "FlankSample", "Interpolate"])
@pytest.mark.parametrize("deterministic", [True, False])
def test_every_fill(env, fill, deterministic):
    import genvarloader_b200 as G

    d, ds, kinds = env
    strat = {"Repeat5p": G.Repeat5p(), "Repeat5pNormalized": G.Repeat5pNormalized(), "Constant": G.Constant(0.75),
             "FlankSample": G.FlankSample(5), "Interpolate": G.Interpolate(3)}[fill]
    ds_ = ds.with_insertion_fill(strat).with_settings(jitter=MAX_JITTER, deterministic=deterministic, rc_neg=True).with_len(
        "ragged" if deterministic else 300)
    got, trk = _read_both(ds_, R_IDX, S_IDX, 9)
    w0, rc = _cells(d, ds_, R_IDX, 9, len(kinds), d.ploidy, True)
    _check_painting(got, trk, w0, rc)


@pytest.mark.parametrize("dtype_name", ["bfloat16", "float16"])
def test_16_bit_values(env, dtype_name):
    import torch

    import genvarloader_b200 as G

    d, ds, kinds = env
    dt = getattr(torch, dtype_name)
    ds_ = ds.with_insertion_fill(G.Interpolate(1)).with_settings(jitter=MAX_JITTER)
    got16, trk16 = _read_both(ds_.with_track_dtype(dt), R_IDX, S_IDX, 4)
    got32 = _strip(ds_.with_tracks(kind="realigned-intervals").with_settings(rng=4)[R_IDX, S_IDX])
    assert got16.values.data.dtype == dt
    assert got16.offsets.cpu().tolist() == got32.offsets.cpu().tolist()  # runs are decided on identity
    assert torch.equal(got16.starts.data, got32.starts.data) and torch.equal(got16.ends.data, got32.ends.data)
    assert torch.equal(got16.values.data.view(torch.int16), got32.values.data.to(dt).view(torch.int16))
    w0, rc = _cells(d, ds_, R_IDX, 4, len(kinds), d.ploidy, True)
    _check_painting(got16, trk16, w0, rc)


def test_annotated_and_exonic(env):
    d, ds, kinds = env
    for ds_ in (ds.with_seqs("annotated"), ds.with_settings(var_filter="exonic"),
                ds.with_seqs("annotated").with_settings(var_filter="exonic", jitter=3)):
        got, trk = _read_both(ds_, R_IDX, S_IDX, 6)
        w0, rc = _cells(d, ds_, R_IDX, 6, len(kinds), d.ploidy, True)
        _check_painting(got, trk, w0, rc)


def _expect(d, kinds, names, r, s, w0, lengths_rows, fills=None):
    """The restatement over a read's rows (svar1 lists, no filter, no shift): cells (read, track, ploid)."""
    from oracle import oracle as O

    p = d.ploidy
    ds_idx = r * d.n_samples + s
    goi = ds_idx[:, None] * p + np.arange(p)[None, :]
    go = np.asarray(d.geno_offsets)
    gs, ge = (go[:-1], go[1:]) if go.ndim == 1 else (go[0], go[1])
    length = (d.regions[r, 2] - d.regions[r, 1]).astype(np.int64)
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, q_starts=w0, q_ends=w0 + length, v_starts=d.v_starts)
    track_n = length - np.minimum(diffs.min(1), 0)
    base_seed = int(np.bitwise_xor.reduce(ds_idx.astype(np.uint64)))
    S, E, V, n = [], [], [], []
    for q in range(len(r)):
        for ti, name in enumerate(names):
            ts, te, tv, io = d.tracks[name]
            slot = ds_idx[q] if kinds[name] == "sample" else r[q]
            sl = RI.Slot(ts[io[slot]:io[slot + 1]], te[io[slot]:io[slot + 1]], tv[io[slot]:io[slot + 1]], w0[q], track_n[q])
            strat, par = fills[ti] if fills else (0, 0.0)
            for h in range(p):
                vi = d.geno_v_idxs[gs[goi[q, h]]:ge[goi[q, h]]]
                a, b, c = RI.realigned_intervals_row(d.v_starts[vi], d.ilens[vi], None, 0, sl, int(lengths_rows[q * p + h]),
                                                     strat, par, base_seed, q, h)
                S.append(a), E.append(b), V.append(c), n.append(len(a))
    return (np.concatenate(S).astype(np.int32), np.concatenate(E).astype(np.int32), np.concatenate(V).astype(np.float32),
            np.concatenate([[0], np.cumsum(n)]).astype(np.int64))


def _assert_exact(got, exp):
    s, e, v, off = exp
    assert got.offsets.cpu().numpy().reshape(-1).tolist() == off.tolist()
    assert np.array_equal(got.starts.data.cpu().numpy(), s) and np.array_equal(got.ends.data.cpu().numpy(), e)
    assert np.array_equal(got.values.data.cpu().numpy().view(np.uint32), v.view(np.uint32))


@pytest.mark.parametrize("jitter", [0, MAX_JITTER])
@pytest.mark.parametrize("fill", [None, "Constant", "FlankSample", "Interpolate"])
def test_matches_the_restatement(env, jitter, fill):
    import genvarloader_b200 as G

    d, ds, kinds = env
    names = [n for n in kinds if n != "overlap"]  # stored intervals that are already free of overlaps
    ds_ = ds.with_tracks(names).with_settings(jitter=jitter, rc_neg=True)
    fills = None
    if fill is not None:
        strat = {"Constant": G.Constant(-1.5), "FlankSample": G.FlankSample(4), "Interpolate": G.Interpolate(2)}[fill]
        ds_ = ds_.with_insertion_fill({"track1": strat, "short": strat})
        code = {"Constant": (2, -1.5), "FlankSample": (3, 4.0), "Interpolate": (4, 2.0)}[fill]
        fills = [code if n in ("track1", "short") else (0, 0.0) for n in names]
    seqs, got = ds_.with_tracks(names, kind="realigned-intervals").with_settings(rng=7)[R_IDX, S_IDX]
    w0 = d.regions[R_IDX, 1].astype(np.int64) + _jitter(ds_, len(R_IDX), 7)
    rows_len = np.diff(seqs.offsets.cpu().numpy().reshape(-1))
    _assert_exact(got, _expect(d, kinds, names, R_IDX, S_IDX, w0, rows_len, fills))


def test_rows_without_indels_are_the_stored_intervals(env):
    """Invariant 2: a row with no applied indel and no shift returns what kind="intervals" returns for the read."""
    d, ds, kinds = env
    names = list(kinds)
    got = ds.with_tracks(kind="realigned-intervals")[R_IDX, S_IDX][1].to_list()
    ref = ds.with_settings(realign_tracks=False).with_tracks(kind="intervals")[R_IDX, S_IDX][1].to_list()
    go = np.asarray(d.geno_offsets)
    gs, ge = (go[:-1], go[1:]) if go.ndim == 1 else (go[0], go[1])
    p, t, n = d.ploidy, len(names), 0
    for q, (r, s) in enumerate(zip(R_IDX, S_IDX)):
        a, b = int(d.regions[r, 1]), int(d.regions[r, 2])
        for h in range(p):
            k = (r * d.n_samples + s) * p + h
            vi = d.geno_v_idxs[gs[k]:ge[k]]
            if ((d.ilens[vi] != 0) & (d.v_starts[vi] < b) & (d.v_starts[vi] - np.minimum(d.ilens[vi], 0) >= a - 1)).any():
                continue
            for ti in range(t):
                assert got[(q * t + ti) * p + h] == ref[q * t + ti], (q, ti, h)
                n += 1
    assert n > 0


def test_spliced_cells_concatenate_elements(env):
    d, ds, kinds = env
    t, p = len(kinds), d.ploidy
    rows = {"a": [3, 0, 7], "b": [5], "c": [11, 2, 11], "d": [1, 4, 9, 6, 8]}
    base = ds.with_tracks(kind="realigned-intervals").with_settings(rc_neg=True)
    sp = base.with_settings(splice_info=rows)
    memo = {}

    def elem(e, s):  # (row lengths per ploid, t * p cells) of one unspliced element read
        if (e, s) not in memo:
            seqs, iv = base[e, s]
            memo[e, s] = (np.diff(seqs.offsets.cpu().numpy().reshape(-1)), iv.to_list())
        return memo[e, s]

    out = sp[:, :][1]
    assert out.shape == (4, d.n_samples, t, p, None)
    cells = out.to_list()
    for c, (_, elems) in enumerate(rows.items()):
        for s in range(d.n_samples):
            el = [elem(e, s)[1] for e in elems]  # (t * p cells each)
            for k in range(t * p):
                assert cells[(c * d.n_samples + s) * t * p + k] == sum((x[k] for x in el), [])
    # painted back, element by element, the spliced tracks
    trk = sp.with_tracks(kind="tracks")[:, :][1]
    t_off, t_data = trk.offsets.cpu().numpy().reshape(-1), _values(trk.data)
    ci = 0
    for c, (_, elems) in enumerate(rows.items()):
        for s in range(d.n_samples):
            for k in range(t * p):
                parts = []
                for e in elems:
                    L, iv = int(elem(e, s)[0][k % p]), elem(e, s)[1][k]
                    a0 = int(d.regions[e, 1])
                    parts.append(RI.paint([x[0] for x in iv], [x[1] for x in iv], np.float32([x[2] for x in iv]), a0, L,
                                          bool(d.regions[e, 3] == -1)))
                want = t_data[t_off[ci]:t_off[ci + 1]]
                assert np.array_equal(np.concatenate(parts).view(np.uint32), want.view(np.uint32)), ci
                ci += 1


def test_svar2_dataset_matches_svar1_twin(cuda_device):
    from genvarloader_b200 import Dataset, synth

    d = synth.make_dataset(29, 80_000, 4, 10, 900, 5.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=3, max_indel=7)
    sv = synth.to_svar2_dataset(d, dense_frac=0.5, seed=2)
    r, s = np.arange(10), np.arange(10) % 4
    out = []
    for ds in (Dataset.from_synth(cuda_device, d, rng=1, svar2=sv), Dataset.from_synth(cuda_device, d, rng=1)):
        out.append(ds.with_seqs("haplotypes").with_tracks(kind="realigned-intervals")[r, s])
    assert np.array_equal(out[0][0].data.cpu().numpy(), out[1][0].data.cpu().numpy())
    assert out[0][1].to_list() == out[1][1].to_list() and out[0][1].offsets[-1] > 0


def test_opened_dataset(cuda_device, tmp_path):
    from genvarloader_b200 import Dataset, synth
    from tests._gvl_disk import write_fasta, write_gvl_dataset

    d = synth.make_dataset(23, 150_000, 3, 10, 2000, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=3, max_indel=9)
    order = np.random.default_rng(1).permutation(d.n_regions)
    write_gvl_dataset(tmp_path / "ds", d, ["chr1"], ["a", "b", "c"], order)
    write_fasta(tmp_path / "ref.fa", d.reference, d.ref_offsets, ["chr1"])
    dsk = Dataset.open(tmp_path / "ds", tmp_path / "ref.fa", device=cuda_device).with_seqs("haplotypes")
    got = _strip(dsk.with_tracks(kind="realigned-intervals")[:, :])
    trk = _strip(dsk.with_tracks(kind="tracks")[:, :])
    assert got.shape == (10, 3, 3, 2, None)
    ds_idx = (order[:, None] * 3 + np.arange(3)[None, :]).ravel()
    reg = d.regions[ds_idx // 3]
    t = len(dsk.active_tracks)
    rc = np.repeat(reg[:, 3] == -1, t * 2) if dsk.rc_neg else np.zeros(len(ds_idx) * t * 2, bool)
    assert _check_painting(got, trk, np.repeat(reg[:, 1].astype(np.int64), t * 2), rc) > 0


def test_large_read_many_items_and_scan_blocks(cuda_device):
    """600 reads x 2 tracks x 2 ploids = 2,400 output rows (two blocks of the offset scan), 10 kb rows with hundreds of
    records each (items beyond one 32-lane chunk), 3 bp runs crossing many indels."""
    from genvarloader_b200 import Dataset, synth

    d = synth.make_dataset(41, 400_000, 8, 16, 10_000, 20.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=0, max_indel=5,
                           snp_frac=0.3)
    rng = np.random.default_rng(4)
    d.tracks["long"] = synth.make_track_fast(rng, d.regions, d.n_samples, mean_run=400)
    d.tracks["short"] = synth.make_track_fast(rng, d.regions, d.n_samples, mean_run=3)
    ds = Dataset.from_synth(cuda_device, d, rng=2).with_seqs("haplotypes")
    r, s = rng.integers(0, d.n_regions, 600), rng.integers(0, d.n_samples, 600)
    got, trk = _read_both(ds.with_settings(rc_neg=True), r, s, 3)
    w0, rc = _cells(d, ds, r, 3, 2, 2, True)
    assert _check_painting(got, trk, w0, rc) > 500_000


def test_entry_rejects_bad_calls(env):
    import ctypes

    import torch
    from genvarloader_b200 import _ffi

    d, ds, kinds = env
    eng = ds.engine
    lib = _ffi.lib
    off = torch.zeros(16, dtype=torch.int64, device=eng.device)
    ptr = ctypes.c_void_p(off.data_ptr())
    # a rejected track call leaves no plan
    assert lib.gvl_dev_paint_tracks(eng.ctx.handle, 1, None, None, None, 0, None, 0, None, 0, None, None, None, 0, None) == 2
    assert lib.gvl_dev_realigned_track_intervals(eng.ctx.handle, None, ptr, 0, None, None, None, 0, None) == 4
    assert b"plan" in lib.gvl_last_error()
    assert lib.gvl_dev_realigned_track_intervals(eng.ctx.handle, None, ptr, 0, None, None, None, 7, None) == 2
    assert lib.gvl_dev_realigned_track_intervals(eng.ctx.handle, None, ptr, 5, None, None, None, 0, None) == 2
    # a valid read afterwards
    got, trk = _read_both(ds, R_IDX[:3], S_IDX[:3], 1)
    assert got.offsets[-1] > 0
