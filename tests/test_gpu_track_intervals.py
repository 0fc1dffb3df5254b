"""`with_tracks(kind="intervals")`: per (read, track) cell the stored intervals that overlap the read's window, clipped to it
(gvl_dev_track_intervals).  Checked exactly against a numpy mask-and-clip restatement of the definition on non-overlapping
synthetic intervals, and through the painting invariant (DESIGN.md §7): the returned intervals painted into zeros over the
window and reversed where the strand mask is set are, bit for bit, the `kind="tracks"` output of the same read."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MAX_JITTER = 8


def _edge_track(rng, regions, n_slots_per_region):
    """Per slot, non-overlapping intervals placed on the edges of its region [a, b): one ending at a (excluded from an
    unjittered read) and one starting there, or one straddling a; a few inside; one straddling b, or one ending at b and
    one starting there (excluded); every 5th slot is empty."""
    s, e, counts = [], [], []
    for r in range(len(regions)):
        a, b = int(regions[r, 1]), int(regions[r, 2])
        for k in range(n_slots_per_region):
            if (r * n_slots_per_region + k) % 5 == 3:
                counts.append(0)
                continue
            cuts = np.sort(rng.choice(np.arange(a + 10, b - 10), 6, replace=False))
            iv = [(a - 9, a), (a, a + 3)] if k % 2 == 0 else [(a - 9, a - 4), (a - 4, a + 3)]
            iv += [(int(cuts[i]), int(cuts[i + 1])) for i in range(0, 6, 2)]
            iv += [(b - 3, b + 6), (b + 6, b + 11)] if k % 2 == 0 else [(b - 3, b), (b, b + 6)]
            s += [x for x, _ in iv]
            e += [y for _, y in iv]
            counts.append(len(iv))
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return (np.asarray(s, np.int32), np.asarray(e, np.int32), rng.gamma(2.0, 2.0, len(s)).astype(np.float32), off)


def _overlap_track(rng, regions, n_slots_per_region, n=40):
    """Overlapping intervals in stored order (painted last-write-wins; flattened at upload)."""
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

    # straddle_ends: the first region starts before the contig, the last ends past it (windows past both ends)
    d = synth.make_dataset(17, 60_000, 3, 12, 400, 4.0, neg_strand_frac=0.5, straddle_ends=True, n_tracks=6, max_indel=6)
    d.max_jitter = MAX_JITTER
    rng = np.random.default_rng(3)
    kinds = {f"track{i}": "sample" for i in range(6)}
    for i in range(3):
        d.tracks[f"annot{i}"] = synth.make_track(rng, d.regions, 1, MAX_JITTER)
        kinds[f"annot{i}"] = "annot"
    d.tracks["edges"], kinds["edges"] = _edge_track(rng, d.regions, d.n_samples), "sample"
    d.tracks["annot_edges"], kinds["annot_edges"] = _edge_track(rng, d.regions, 1), "annot"
    d.tracks["overlap"], kinds["overlap"] = _overlap_track(rng, d.regions, d.n_samples), "sample"
    ds = Dataset.from_arrays(cuda_device, d.reference, d.ref_offsets, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                             d.geno_v_idxs, d.geno_offsets, d.regions, d.n_samples, d.ploidy, d.max_jitter, d.tracks,
                             track_kinds=kinds, rng=0)
    names = [n for n in kinds if n != "overlap"]  # 11 tracks with non-overlapping stored intervals
    iv = ds.with_seqs(None).with_tracks(names, kind="intervals")
    return d, ds, iv, kinds, names


def _expect_rows(tracks, slots, w0, w1):
    """Mask-and-clip restatement of the definition for rows (tracks[k], slots[k], [w0[k], w1[k])): the intervals with
    end > w0 and start < w1 of a non-empty window, clipped -> (starts, ends, values f32, offsets)."""
    st, en, va, n = [np.zeros(0, np.int32)], [np.zeros(0, np.int32)], [np.zeros(0, np.float32)], []
    for (s, e, v, io), slot, a0, a1 in zip(tracks, slots, w0, w1):
        a, b = io[slot], io[slot + 1]
        keep = (e[a:b] > a0) & (s[a:b] < a1) if a1 > a0 else np.zeros(b - a, bool)
        st.append(np.maximum(s[a:b][keep], a0))
        en.append(np.minimum(e[a:b][keep], a1))
        va.append(v[a:b][keep])
        n.append(int(keep.sum()))
    return (np.concatenate(st).astype(np.int32), np.concatenate(en).astype(np.int32), np.concatenate(va).astype(np.float32),
            np.concatenate([[0], np.cumsum(n)]).astype(np.int64))


def _expect(d, kinds, names, ds_idx, w0, w1):
    """`_expect_rows` of a read: rows (read, track), a SAMPLE track's slot is the dataset index, an ANNOT track's the
    region."""
    t = len(names)
    slots = np.stack([ds_idx if kinds[n] == "sample" else ds_idx // d.n_samples for n in names], 1).ravel()
    return _expect_rows([d.tracks[n] for n in names] * len(ds_idx), slots, np.repeat(w0, t), np.repeat(w1, t))


def _windows(d, ds, ds_idx, seed, length):
    """The read's windows: jittered start (the read's one draw per query) and the painted track's length."""
    reg = d.regions[ds_idx // d.n_samples]
    jit = np.random.default_rng(seed).integers(-ds.jitter, ds.jitter + 1, size=len(ds_idx), dtype=np.int32)
    w0 = reg[:, 1].astype(np.int64) + jit
    w1 = w0 + (length if isinstance(length, int) else reg[:, 2] - reg[:, 1])
    return w0, w1


def _assert_equal(got, exp, dtype=None):
    import torch

    s, e, v, off = exp
    assert got.offsets.cpu().numpy().tolist() == off.tolist()
    assert got.starts.data.dtype == torch.int32 and got.ends.data.dtype == torch.int32
    assert (got.starts.data.cpu().numpy() == s).all() and (got.ends.data.cpu().numpy() == e).all()
    dtype = dtype or torch.float32
    assert got.values.data.dtype == dtype
    want = torch.from_numpy(v).to(got.values.data.device).to(dtype)  # cast on the device
    bits = torch.int32 if dtype == torch.float32 else torch.int16
    assert torch.equal(got.values.data.view(bits), want.view(bits))


@pytest.mark.parametrize("length", ["ragged", "variable", 300])
@pytest.mark.parametrize("jitter", [0, MAX_JITTER])
def test_matches_definition(env, length, jitter):
    d, ds, iv, kinds, names = env
    ds_ = iv.with_len(length).with_settings(jitter=jitter, rng=11)
    r = np.array([0, 11, 3, 5, 0, 7, 11, 2, 9])
    s = np.array([1, 2, 0, 2, 0, 1, 0, 2, 1])
    got = ds_[r, s]
    ds_idx = r * d.n_samples + s
    w0, w1 = _windows(d, ds_, ds_idx, 11, length)
    assert got.shape == (len(r), len(names), None)
    _assert_equal(got, _expect(d, kinds, names, ds_idx, w0, w1))
    # the edge tracks: the intervals ending at w0 / starting at w1 are left out, the straddling ones are clipped
    if jitter == 0 and length != 300:
        cells = got.reshape(len(r) * len(names)).to_list()
        for q in range(len(r)):
            a, b = int(w0[q]), int(w1[q])
            for name in ("edges", "annot_edges"):
                c = cells[q * len(names) + names.index(name)]
                if c:
                    assert c[0][0] == a and c[-1][1] == b and all(a < y and x < b for x, y, _ in c)


def test_strand_changes_nothing(env):
    d, ds, iv, kinds, names = env
    r = np.arange(d.n_regions)
    assert (d.regions[:, 3] == -1).any() and (d.regions[:, 3] == 1).any()
    a, b = iv.with_settings(rc_neg=True)[r, r % 3], iv.with_settings(rc_neg=False)[r, r % 3]
    for f in ("starts", "ends", "values"):
        assert np.array_equal(getattr(a, f).data.cpu().numpy(), getattr(b, f).data.cpu().numpy())
    assert np.array_equal(a.offsets.cpu().numpy(), b.offsets.cpu().numpy())


def test_index_forms_and_shapes(env):
    d, ds, iv, kinds, names = env
    t = len(names)
    S = d.n_samples

    painted = iv.with_tracks(names, kind="tracks")

    def exp(ds_idx):
        reg = d.regions[ds_idx // S]
        return _expect(d, kinds, names, ds_idx, reg[:, 1], reg[:, 2])

    one = iv[4, 2]  # scalar: (t, ~n)
    assert one.shape == (t, None) == painted[4, 2].shape
    _assert_equal(one, exp(np.array([4 * S + 2])))
    sl = iv[2:6, 1:3]  # two slices: (n, m, t, ~n)
    assert sl.shape == (4, 2, t, None) == painted[2:6, 1:3].shape
    _assert_equal(sl, exp((np.arange(2, 6)[:, None] * S + np.arange(1, 3)[None, :]).ravel()))
    combo = iv[[7, 1], 0]
    assert combo.shape == painted[[7, 1], 0].shape
    _assert_equal(combo, exp(np.array([7 * S, 1 * S])))
    sub = iv.subset_to(regions=[9, 3, 10], samples=["s2", "s0"])
    got = sub[1:, :]
    assert got.shape == (2, 2, t, None) == painted.subset_to(regions=[9, 3, 10], samples=["s2", "s0"])[1:, :].shape
    _assert_equal(got, exp(np.array([3 * S + 2, 3 * S, 10 * S + 2, 10 * S])))
    # "flat" hands back the same object; "variable" does not pad intervals
    flat = iv.with_output_format("flat")[[1, 2], [0, 1]]
    var = iv.with_len("variable")[[1, 2], [0, 1]]
    for o in (flat, var):
        assert o.shape == (2, t, None)
        _assert_equal(o, exp(np.array([1 * S, 2 * S + 1])))


@pytest.mark.parametrize("dtype_name", ["bfloat16", "float16"])
def test_16_bit_values(env, dtype_name):
    import torch

    d, ds, iv, kinds, names = env
    dtype = getattr(torch, dtype_name)
    r, s = np.arange(12), np.arange(12) % 3
    got = iv.with_track_dtype(dtype)[r, s]
    ref = iv[r, s]
    assert torch.equal(got.starts.data, ref.starts.data) and torch.equal(got.offsets, ref.offsets)
    assert torch.equal(got.values.data.view(torch.int16), ref.values.data.to(dtype).view(torch.int16))
    reg = d.regions[r]
    _assert_equal(got, _expect(d, kinds, names, r * d.n_samples + s, reg[:, 1], reg[:, 2]), dtype)


def _paint(got, w0, w1, to_rc):
    """The intervals of every (read, track) cell painted into zeros over its window, masked rows reversed: f32 flat."""
    from oracle import oracle as O

    outer = got.lengths.shape
    n_cells = int(np.prod(outer))
    q_of = np.repeat(np.arange(len(w0)), n_cells // len(w0))
    lens = (w1 - w0)[q_of]
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    buf = np.zeros(int(offs[-1]), np.float32)
    O.intervals_to_tracks(np.arange(n_cells), w0[q_of], got.starts.data.cpu().numpy(), got.ends.data.cpu().numpy(),
                          got.values.data.cpu().numpy(), got.offsets.cpu().numpy(), buf, offs)
    if to_rc is not None:
        O.reverse_flat_rows_inplace(buf, offs, to_rc[q_of])
    return buf, offs


@pytest.mark.parametrize("seqs", [None, "reference", "haplotypes"])
@pytest.mark.parametrize("length", ["ragged", 300])
@pytest.mark.parametrize("rc_neg", [True, False])
def test_painting_invariant(env, seqs, length, rc_neg):
    """All 12 tracks, the overlapping one included: painting the intervals gives the painted tracks bit for bit."""
    d, ds, iv, kinds, names = env
    base = ds.with_seqs(seqs).with_settings(realign_tracks=False, rc_neg=rc_neg, jitter=MAX_JITTER).with_len(length)
    r = np.array([0, 11, 4, 6, 1, 11, 9, 3, 0, 8])
    s = np.array([0, 1, 2, 1, 0, 2, 2, 0, 1, 1])
    trk = base.with_settings(rng=5)[r, s]
    got = base.with_tracks(kind="intervals").with_settings(rng=5)[r, s]
    if seqs is not None:
        seq_t, trk = trk
        seq_i, got = got
        a = seq_t.data if hasattr(seq_t, "data") else seq_t
        b = seq_i.data if hasattr(seq_i, "data") else seq_i
        assert np.array_equal(a.cpu().numpy(), b.cpu().numpy())  # the sequences do not change
    t = len(kinds)
    assert got.shape == (len(r), t, None)
    ds_idx = r * d.n_samples + s
    w0, w1 = _windows(d, base, ds_idx, 5, length)
    # sorted, disjoint and inside the window
    st, en, off = got.starts.data.cpu().numpy(), got.ends.data.cpu().numpy(), got.offsets.cpu().numpy()
    q_of = np.repeat(np.repeat(np.arange(len(r)), t), np.diff(off))
    assert (st >= w0[q_of]).all() and (en <= w1[q_of]).all() and (st <= en).all()
    inner = np.ones(st.size, bool)
    inner[off[:-1][off[:-1] < st.size]] = False  # first interval of a cell
    assert (st[1:][inner[1:]] >= en[:-1][inner[1:]]).all()
    to_rc = (d.regions[r, 3] == -1) if rc_neg else None
    buf, offs = _paint(got, w0, w1, to_rc)
    exp = (trk.data if hasattr(trk, "offsets") else trk).reshape(-1).cpu().numpy()
    assert buf.view(np.uint32).tolist() == exp.view(np.uint32).tolist()


def test_spliced_cells_concatenate_elements(env):
    d, ds, iv, kinds, names = env
    rows = {"a": [3, 0, 7], "b": [5], "c": [11, 2, 11], "d": [1, 4, 9, 6, 8]}
    for seqs in (None, "reference"):
        base = ds.with_seqs(seqs).with_tracks(names, kind="intervals")
        sp = base.with_settings(splice_info=rows)
        painted = sp.with_tracks(names, kind="tracks")
        t = len(names)
        itv = (lambda o: o[1]) if seqs is not None else (lambda o: o)
        out = itv(sp[:, :])
        assert out.shape == (4, d.n_samples, t, None) == itv(painted[:, :]).shape
        cells = out.to_list()
        for c, (_, elems) in enumerate(rows.items()):
            for s in range(d.n_samples):
                el = [itv(base[e, s]).to_list() for e in elems]  # (t cells each)
                for k in range(t):
                    assert cells[(c * d.n_samples + s) * t + k] == sum((x[k] for x in el), [])
        one = itv(sp[3, 1])
        assert one.shape == (t, None) == itv(painted[3, 1]).shape
        assert one.to_list() == cells[(3 * d.n_samples + 1) * t:(3 * d.n_samples + 2) * t]
        paired = itv(sp[np.array([2, 0]), np.array([1, 2])])
        assert paired.shape == (2, t, None)
        assert paired.to_list() == (cells[(2 * d.n_samples + 1) * t:(2 * d.n_samples + 2) * t]
                                    + cells[(0 * d.n_samples + 2) * t:(0 * d.n_samples + 3) * t])


def test_loader_reads_through_getitem(env):
    from genvarloader_b200._dataset import BatchLoader

    d, ds, iv, kinds, names = env
    ds_ = iv.with_len(300)
    for mode in (None, "buffered", "double_buffered"):
        dl = ds_.to_dataloader(batch_size=5, mode=mode, return_indices=True)
        assert isinstance(dl, BatchLoader)
        n = 0
        for got, r, s in dl:
            assert got.to_list() == ds_[r, s].to_list()
            n += len(r)
        assert n == len(ds_)


def test_svar2_dataset_matches_svar1_twin(cuda_device):
    from genvarloader_b200 import Dataset, synth

    d = synth.make_dataset(29, 80_000, 4, 10, 900, 5.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=3, max_indel=7)
    sv = synth.to_svar2_dataset(d, dense_frac=0.5, seed=2)
    r, s = np.arange(10), np.arange(10) % 4
    out = []
    for ds in (Dataset.from_synth(cuda_device, d, rng=1, svar2=sv), Dataset.from_synth(cuda_device, d, rng=1)):
        out.append(ds.with_settings(realign_tracks=False).with_tracks(kind="intervals")[r, s])
    assert np.array_equal(out[0][0].data.cpu().numpy(), out[1][0].data.cpu().numpy())
    assert out[0][1].to_list() == out[1][1].to_list()
    reg = d.regions[r]
    _assert_equal(out[0][1], _expect(d, {n: "sample" for n in d.tracks}, list(d.tracks), r * 4 + s, reg[:, 1], reg[:, 2]))


def test_opened_dataset(cuda_device, tmp_path):
    from genvarloader_b200 import Dataset, synth
    from tests._gvl_disk import write_fasta, write_gvl_dataset

    d = synth.make_dataset(23, 150_000, 3, 10, 2000, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=3, max_indel=9)
    d.tracks["track2"] = synth.make_track(np.random.default_rng(0), d.regions, 1)
    order = np.random.default_rng(1).permutation(d.n_regions)
    write_gvl_dataset(tmp_path / "ds", d, ["chr1"], ["a", "b", "c"], order, annot_tracks=("track2",))
    write_fasta(tmp_path / "ref.fa", d.reference, d.ref_offsets, ["chr1"])
    dsk = Dataset.open(tmp_path / "ds", tmp_path / "ref.fa", device=cuda_device)
    got = dsk.with_settings(realign_tracks=False).with_tracks(kind="intervals")[:, :][1]
    assert got.shape == (10, 3, 3, None)
    ds_idx = (order[:, None] * 3 + np.arange(3)[None, :]).ravel()  # input row i is storage region order[i]
    reg = d.regions[ds_idx // 3]
    assert dsk.track_kinds["track2"] == "annot"
    _assert_equal(got, _expect(d, dsk.track_kinds, list(dsk.active_tracks), ds_idx, reg[:, 1], reg[:, 2]))


def test_engine_rows(env):
    """Rows given directly: empty and inverted windows, a window in a gap or before every interval, the whole slot,
    an empty slot, slots of several tracks in one call, no rows at all."""
    import torch

    d, ds, iv, kinds, names = env
    eng, dev = ds.engine, ds.engine.device
    use = ["track0", "annot1", "edges"]
    s, e, v, io = d.tracks["track0"]
    slot = 4
    a, b = int(s[io[slot]]), int(e[io[slot + 1] - 1])
    gap = next(k for k in range(io[slot], io[slot + 1] - 1) if e[k] < s[k + 1])
    es, ee, _, eio = d.tracks["edges"]
    empty = int(np.flatnonzero(np.diff(eio) == 0)[0])
    rows = [(0, slot, a + 5, a + 5), (0, slot, a + 9, a + 2), (0, slot, a - 100, a - 50), (0, slot, int(e[gap]), int(s[gap + 1])),
            (0, slot, a - 1000, b + 1000), (0, slot, int(s[gap]) + 1, int(s[gap]) + 2), (1, 7, -50, 10_000_000),
            (2, empty, -50, 10_000_000), (2, 5, int(ee[eio[5]]), int(es[eio[6] - 1])), (1, 0, 100, 99)]
    tk = np.array([r[0] for r in rows], np.int32)
    slots = np.array([r[1] for r in rows], np.int64)
    w0 = np.array([r[2] for r in rows], np.int32)
    w1 = np.array([r[3] for r in rows], np.int32)
    cu = lambda x: torch.from_numpy(x).to(dev)
    off, st, en, va = eng.track_intervals(use, cu(slots), cu(tk), cu(w0), cu(w1))
    exp = _expect_rows([d.tracks[use[k]] for k in tk], slots, w0, w1)
    assert np.diff(exp[3]).tolist()[:4] == [0, 0, 0, 0] and exp[3][-1] > 0
    assert off.cpu().tolist() == exp[3].tolist()
    assert st.cpu().numpy().tolist() == exp[0].tolist() and en.cpu().numpy().tolist() == exp[1].tolist()
    assert va.cpu().numpy().view(np.uint32).tolist() == exp[2].view(np.uint32).tolist()
    z = torch.zeros(0, dtype=torch.int64, device=dev)
    off, st, en, va = eng.track_intervals(use, z, z.int(), z.int(), z.int(), dtype=torch.bfloat16)
    assert off.cpu().tolist() == [0] and st.numel() == en.numel() == va.numel() == 0 and va.dtype == torch.bfloat16


def test_large_read_spans_many_scan_blocks(cuda_device):
    """2,048 reads x 8 tracks = 16,384 rows (8 blocks of the offset scan), about 2,000 intervals per slot."""
    from genvarloader_b200 import Dataset, synth

    d = synth.make_dataset(31, 2_000_000, 8, 16, 60_000, 0.5, straddle_ends=False, n_tracks=0)
    rng = np.random.default_rng(4)
    for i in range(8):
        d.tracks[f"t{i}"] = synth.make_track_fast(rng, d.regions, d.n_samples, mean_run=30)
    ds = Dataset.from_synth(cuda_device, d, rng=2).with_seqs(None).with_tracks(kind="intervals")
    r, s = rng.integers(0, d.n_regions, 2048), rng.integers(0, d.n_samples, 2048)
    got = ds.with_len(50_000).with_settings(jitter=0)[r, s]
    ds_idx = r * d.n_samples + s
    w0 = d.regions[r, 1].astype(np.int64)
    exp = _expect(d, {n: "sample" for n in d.tracks}, list(d.tracks), ds_idx, w0, w0 + 50_000)
    assert np.diff(exp[3]).max() > 1000 and exp[0].size > 10_000_000
    _assert_equal(got, exp)
