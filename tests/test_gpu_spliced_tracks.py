"""Tracks of spliced datasets: a spliced cell is the concatenation, in splice-row order, of its elements' unspliced outputs
(jitter 0, ragged length).  The element batch E lists the selected (splice row, sample) pairs in output order and, inside a
pair, the row's elements; the expected values are one oracle call over E, regrouped -- bit-exact.  Also: the per-row
destination layout of the track entries (GVL_TRACK_LAYOUT_ROWS) against the fixed layouts it restates."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
N = ord("N")
SENTINEL = np.array([0x7FBADBAD], np.uint32).view(np.float32)[0]  # a NaN no kernel writes


@pytest.fixture(scope="module")
def env(cuda_device):
    from genvarloader_b200 import Dataset, synth
    from oracle import oracle as O

    d = synth.make_dataset(41, 400_000, 3, 14, 9_000, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=10,
                           max_indel=12, snp_frac=0.5)
    # element lengths: longer than one 8,192-value track tile, a few hundred values, and shorter than 8
    lens = np.array([9000, 8300, 700, 5, 1200, 3, 9000, 450, 7, 2500, 9000, 640, 6, 1000])
    d.regions[:, 2] = d.regions[:, 1] + lens
    d.regions[:, 3] = np.where(np.arange(d.n_regions) % 3 == 1, -1, 1)
    ds = Dataset.from_synth(cuda_device, d, rng=7)
    rows = {"a": [3, 0, 7, 1], "b": [5], "c": [11, 2, 11], "d": [1, 4, 9, 6, 8], "e": [13, 12], "f": [10]}
    return d, ds, rows, O


def _element_batch(d, rows, pairs):
    row_list = list(rows.values())
    e_reg = np.concatenate([row_list[r] for r, _ in pairs]).astype(np.int64)
    e_s = np.concatenate([[s] * len(row_list[r]) for r, s in pairs]).astype(np.int64)
    n_el = np.array([len(row_list[r]) for r, _ in pairs])
    return e_reg, e_s, n_el


def _oracle_realigned(d, O, e_reg, e_s, fills, names, seed, exonic=False, rc_neg=True):
    """One oracle call per track over E: flat buffers and the (e, h) row offsets."""
    p = d.ploidy
    ds_idx = e_reg * d.n_samples + e_s
    regions = np.ascontiguousarray(d.regions[e_reg, :3])
    goi = ds_idx[:, None] * p + np.arange(p)[None, :]
    to_rc = np.repeat(d.regions[e_reg, 3] == -1, p) if rc_neg else None
    keep = ko = None
    if exonic:
        keep, ko = O.choose_exonic_variants(regions[:, 1], regions[:, 2], goi, d.geno_v_idxs, d.geno_offsets, d.v_starts, d.ilens)
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, keep, ko, regions[:, 1], regions[:, 2], d.v_starts)
    lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)
    oo = np.concatenate([[0], np.cumsum(np.maximum(lengths[:, None] + diffs, 0).ravel())]).astype(np.int64)
    to = np.concatenate([[0], np.cumsum(lengths - diffs.clip(max=0).min(1))]).astype(np.int64)
    sh = np.zeros(goi.shape, np.int32)
    out = []
    for name, fill in zip(names, fills):
        s, e, v, io = d.tracks[name]
        buf = np.zeros(int(oo[-1]), np.float32)
        O.intervals_and_realign_track_fused(buf, oo, regions, sh, goi, d.geno_v_idxs, d.geno_offsets, d.v_starts, d.ilens,
                                            ds_idx, s, e, v, io, to, np.array([fill.param()]), fill.strategy_id, seed, keep, ko,
                                            to_rc)
        out.append(buf)
    return out, oo


def _oracle_painted(d, O, e_reg, e_s, names, rc_neg=True):
    ds_idx = e_reg * d.n_samples + e_s
    regions = d.regions[e_reg]
    offs = np.concatenate([[0], np.cumsum(regions[:, 2] - regions[:, 1])]).astype(np.int64)
    out = []
    for name in names:
        s, e, v, io = d.tracks[name]
        buf = np.zeros(int(offs[-1]), np.float32)
        O.intervals_to_tracks(ds_idx, regions[:, 1], s, e, v, io, buf, offs)
        if rc_neg:
            O.reverse_flat_rows_inplace(buf, offs, regions[:, 3] == -1)
        out.append(buf)
    return out, offs


def _check_realigned(got, exp, oo, n_el, p):
    """got: Ragged (pairs..., t, p, None); exp[t]: flat over E rows (e, h)."""
    data, offs = got.data.cpu().numpy().view(np.uint32), got.offsets.cpu().numpy()
    t = len(exp)
    assert offs[-1] == t * oo[-1] and data.size == offs[-1]
    e0, cell = 0, 0
    for k in n_el:
        for ti in range(t):
            for h in range(p):
                want = np.concatenate([exp[ti][oo[e * p + h]: oo[e * p + h + 1]] for e in range(e0, e0 + k)]).view(np.uint32)
                assert (data[offs[cell]: offs[cell + 1]] == want).all(), (e0, ti, h)
                cell += 1
        e0 += k


def _check_painted(got, exp, offs_e, n_el):
    data, offs = got.data.cpu().numpy().view(np.uint32), got.offsets.cpu().numpy()
    t = len(exp)
    assert offs[-1] == t * offs_e[-1] and data.size == offs[-1]
    e0, cell = 0, 0
    for k in n_el:
        for ti in range(t):
            want = exp[ti][offs_e[e0]: offs_e[e0 + k]].view(np.uint32)
            assert (data[offs[cell]: offs[cell + 1]] == want).all(), (e0, ti)
            cell += 1
        e0 += k


def _seed(e_reg, e_s, n_samples):
    return int(np.bitwise_xor.reduce((e_reg * n_samples + e_s).astype(np.uint64)))


# ---------------------------------------------------------------------------------------------------- the ABI
def test_rows_entries_restate_the_fixed_layouts(env):
    """A destination table restating the (b, t, p, ~l) / (b, t, ~l) layout gives the bytes of GVL_TRACK_LAYOUT_BTP in
    gvl_dev_realign_tracks / gvl_dev_paint_tracks; a permutation of the query blocks permutes the output; every value is
    written (NaN sentinel)."""
    import torch

    from genvarloader_b200 import Constant, FlankSample, Interpolate, Repeat5p, Repeat5pNormalized
    from genvarloader_b200._insertion_fill import lower

    d, ds, _, _ = env
    eng, dev, p = ds.engine, ds.engine.device, d.ploidy
    names = [f"track{i}" for i in range(10)]  # > 8 tracks: descriptors in the device buffer
    fills = [Repeat5p(), Repeat5pNormalized(), Constant(-2.5), FlankSample(3), Interpolate(1), Interpolate(2), Interpolate(3),
             FlankSample(1), Repeat5p(), Interpolate(2)]
    ids, params = lower(fills)
    b = 9
    rng = np.random.default_rng(3)
    r_idx, s_idx = rng.integers(0, d.n_regions, b), rng.integers(0, d.n_samples, b)
    ds_idx = r_idx * d.n_samples + s_idx
    regions = np.ascontiguousarray(d.regions[r_idx, :3])
    goi = ds_idx[:, None] * p + np.arange(p)[None, :]
    T = len(names)
    t_reg, t_goi = torch.from_numpy(regions).to(dev), torch.from_numpy(goi).to(dev)
    t_sh = torch.zeros(goi.shape, dtype=torch.int32, device=dev)
    t_rc = torch.from_numpy(np.repeat(d.regions[r_idx, 3] == -1, p).astype(np.uint8)).to(dev)
    t_oi = torch.from_numpy(np.stack([ds_idx] * T)).to(dev)
    diffs = eng.get_diffs(t_goi, t_reg[:, 1].contiguous(), t_reg[:, 2].contiguous())
    lengths = torch.from_numpy((regions[:, 2] - regions[:, 1]).astype(np.int64)).to(dev)
    track_lengths = (lengths - diffs.clamp(max=0).min(1).values.to(torch.int64)).to(torch.int32)
    row_len = (lengths[:, None] + diffs).clamp(min=0).reshape(-1)
    oo = torch.zeros(b * p + 1, dtype=torch.int64, device=dev)
    torch.cumsum(row_len, 0, out=oo[1:])
    total = int(oo[-1])
    mr = eng.max_records(goi)
    args = (names, t_reg, t_sh, t_goi, t_oi, track_lengths, oo, total, ids, params, 1234567, mr)
    ref = eng.realign_tracks(*args, to_rc=t_rc, layout="btp")
    oo_h = oo.cpu().numpy()
    blk0, blk1 = oo_h[0:-1:p], oo_h[p::p]  # block of query q: [blk0[q], blk1[q])
    q_of_row = np.repeat(np.arange(b), p)

    def table(block_base):
        dst = block_base[q_of_row] + (oo_h[:-1] - blk0[q_of_row])
        ts = (blk1 - blk0)[q_of_row]
        return torch.from_numpy(dst.astype(np.int64)).to(dev), torch.from_numpy(ts.astype(np.int64)).to(dev)

    perm = rng.permutation(b)
    blk_len = T * (blk1 - blk0)
    perm_base = np.empty(b, np.int64)
    perm_base[perm] = np.concatenate([[0], np.cumsum(blk_len[perm])[:-1]])  # block of query perm[j] is j-th
    ref_h = ref.cpu().numpy().view(np.uint32)
    for base, want in ((T * blk0, ref_h),
                       (perm_base, np.concatenate([ref_h[T * blk0[q]: T * blk1[q]] for q in perm]))):
        dst, ts = table(base)
        out = torch.empty(T * total, dtype=torch.float32, device=dev)
        out.view(torch.int32).fill_(int(np.array(SENTINEL).view(np.int32)))
        eng.realign_tracks(*args, to_rc=t_rc, out=out, layout="rows", row_dst=dst, row_tstride=ts)
        assert (out.cpu().numpy().view(np.uint32) == want).all()
    # painted: one row per query
    offs = np.concatenate([[0], np.cumsum(regions[:, 2] - regions[:, 1])]).astype(np.int64)
    d_off = torch.from_numpy(offs).to(dev)
    starts = t_reg[:, 1].contiguous()
    q_rc = torch.from_numpy((d.regions[r_idx, 3] == -1).astype(np.uint8)).to(dev)
    ref_p = eng.paint_tracks(names, t_oi, starts, d_off, int(offs[-1]), q_rc).cpu().numpy().view(np.uint32)
    lens = offs[1:] - offs[:-1]
    pb = np.empty(b, np.int64)
    pb[perm] = np.concatenate([[0], np.cumsum(T * lens[perm])[:-1]])
    for base, want in ((T * offs[:-1], ref_p), (pb, np.concatenate([ref_p[T * offs[q]: T * offs[q + 1]] for q in perm]))):
        out = torch.empty(T * int(offs[-1]), dtype=torch.float32, device=dev)
        out.view(torch.int32).fill_(int(np.array(SENTINEL).view(np.int32)))
        eng.paint_tracks(names, t_oi, starts, d_off, int(offs[-1]), q_rc, out=out, layout="rows",
                         row_dst=torch.from_numpy(base.astype(np.int64)).to(dev), row_tstride=torch.from_numpy(lens).to(dev))
        assert (out.cpu().numpy().view(np.uint32) == want).all()


def test_rejected_layouts_leave_no_plan(env):
    """An unknown layout, GVL_TRACK_LAYOUT_ROWS without both tables and a fixed layout with them are argument errors of
    gvl_dev_realign_tracks and gvl_dev_paint_tracks, found before any launch.  A rejected call also drops the plan of the
    call before it: the execute that follows writes nothing."""
    import ctypes as C

    import torch

    from genvarloader_b200._engine import _stream
    from genvarloader_b200._ffi import lib, ptr

    d, ds, _, _ = env
    eng, dev, p = ds.engine, ds.engine.device, int(d.ploidy)
    names, b = ["track0", "track1"], 6
    T = len(names)
    r_idx, s_idx = np.arange(b), np.arange(b) % d.n_samples
    ds_idx = r_idx * d.n_samples + s_idx
    regions = np.ascontiguousarray(d.regions[r_idx, :3])
    goi = ds_idx[:, None] * p + np.arange(p)[None, :]
    t_reg, t_goi = torch.from_numpy(regions).to(dev), torch.from_numpy(goi).to(dev)
    t_sh = torch.zeros(goi.shape, dtype=torch.int32, device=dev)
    t_oi = torch.from_numpy(np.stack([ds_idx] * T)).to(dev)
    diffs = eng.get_diffs(t_goi, t_reg[:, 1].contiguous(), t_reg[:, 2].contiguous())
    lengths = torch.from_numpy((regions[:, 2] - regions[:, 1]).astype(np.int64)).to(dev)
    track_lengths = (lengths - diffs.clamp(max=0).min(1).values.to(torch.int64)).to(torch.int32)
    oo = torch.zeros(b * p + 1, dtype=torch.int64, device=dev)
    torch.cumsum((lengths[:, None] + diffs).clamp(min=0).reshape(-1), 0, out=oo[1:])
    total, mr = int(oo[-1]), int(eng.max_records(goi))
    starts = t_reg[:, 1].contiguous()
    p_off = torch.from_numpy(np.concatenate([[0], np.cumsum(regions[:, 2] - regions[:, 1])]).astype(np.int64)).to(dev)
    itv, sid, par = eng.track_descs(names, [0] * T, [0.0] * T)
    h, table = eng.ctx.handle, torch.zeros(b * p, dtype=torch.int64, device=dev)

    def realign(layout, dst=None, ts=None, out=None):  # out = None: plan only
        return lib.gvl_dev_realign_tracks(h, C.byref(eng.tab), None, ptr(t_reg), ptr(t_sh), ptr(t_goi), b, p, None, None, None,
                                          T, itv, ptr(t_oi), ptr(track_lengths), ptr(oo), total, sid, par, 1, None, 0, None, mr,
                                          layout, ptr(dst), ptr(ts), ptr(out), 0, _stream())

    def paint(layout, dst=None, ts=None, out=None):
        return lib.gvl_dev_paint_tracks(h, T, itv, ptr(t_oi), ptr(starts), b, ptr(p_off), int(p_off[-1]), None, layout, ptr(dst),
                                        ptr(ts), ptr(out), 0, _stream())

    def sentinel_buffer():
        buf = torch.empty(T * total, dtype=torch.float32, device=dev)
        buf.view(torch.int32).fill_(int(np.array(SENTINEL).view(np.int32)))
        return buf

    def untouched(buf):
        return bool((buf.view(torch.int32) == int(np.array(SENTINEL).view(np.int32))).all())

    out = sentinel_buffer()
    for call in (realign, paint):
        for args in ((2,), (2, table), (2, None, table), (1, table, table), (0, table, table), (3,), (-1,)):
            assert call(*args, out=out) == 2, (call.__name__, args)
            assert b"layout" in lib.gvl_last_error().lower(), (call.__name__, args)
    assert untouched(out)
    # a valid plan executes into the whole buffer ...
    assert realign(1) == 0
    assert lib.gvl_dev_realign_tracks_exec(h, ptr(out), 0, _stream()) == 0
    torch.cuda.synchronize()
    assert not (out.view(torch.int32) == int(np.array(SENTINEL).view(np.int32))).any()
    # ... and into nothing once a rejected call of either entry followed it
    for reject in (lambda: realign(3), lambda: paint(2), lambda: realign(1, table, table)):
        assert realign(1) == 0 and reject() == 2
        buf = sentinel_buffer()
        assert lib.gvl_dev_realign_tracks_exec(h, ptr(buf), 0, _stream()) == 0
        torch.cuda.synchronize()
        assert untouched(buf)


# ---------------------------------------------------------------------------------------------------- Dataset vs the oracle
FILLS = {
    "repeat5p": lambda m: m.Repeat5p(),
    "repeat5p_norm": lambda m: m.Repeat5pNormalized(),
    "constant": lambda m: m.Constant(-2.5),
    "flank": lambda m: m.FlankSample(4),
    "interp1": lambda m: m.Interpolate(1),
    "interp2": lambda m: m.Interpolate(2),
    "interp3": lambda m: m.Interpolate(3),
}


@pytest.mark.parametrize("seqs", ["haplotypes", "annotated"])
@pytest.mark.parametrize("fill", list(FILLS))
def test_realigned_tracks_vs_oracle(env, seqs, fill):
    import genvarloader_b200 as m

    d, ds, rows, O = env
    names = ["track0", "track3"]
    f = FILLS[fill](m)
    sp = ds.with_seqs(seqs).with_tracks(names).with_insertion_fill(f).with_settings(splice_info=rows)
    r_sel, s_sel = [0, 2, 3, 1, 4, 5], [1, 0, 2, 2, 1, 0]
    seq_out, trk = sp[r_sel, s_sel]
    assert trk.shape == (6, 2, d.ploidy, None)
    pairs = list(zip(r_sel, s_sel))
    e_reg, e_s, n_el = _element_batch(d, rows, pairs)
    exp, oo = _oracle_realigned(d, O, e_reg, e_s, [f, f], names, _seed(e_reg, e_s, d.n_samples))
    _check_realigned(trk, exp, oo, n_el, d.ploidy)
    # the tracks have the lengths of the sequences they come with
    h = seq_out.haps if seqs == "annotated" else seq_out
    assert (trk.lengths.cpu() == h.lengths.cpu()[:, None, :]).all()


def test_spliced_tracks_equal_one_unspliced_call_over_the_elements(env):
    """Structural check: ds_spliced[...] == the regrouped tracks of ds[E_r, E_s] (FlankSample seeds included)."""
    from genvarloader_b200 import FlankSample, Interpolate

    d, ds, rows, _ = env
    base = ds.with_tracks(["track1", "track2", "track5"]).with_insertion_fill(
        {"track1": FlankSample(6), "track2": Interpolate(3), "track5": FlankSample(2)})
    sp = base.with_settings(splice_info=rows)
    h_sp, t_sp = sp[:, 1:]
    pairs = [(r, s) for r in range(len(rows)) for s in range(1, d.n_samples)]
    e_reg, e_s, n_el = _element_batch(d, rows, pairs)
    h_un, t_un = base[e_reg, e_s]
    p, T = d.ploidy, 3
    assert t_sp.shape == (len(rows), d.n_samples - 1, T, p, None)
    du, ou = t_un.data.cpu().numpy().view(np.uint32), t_un.offsets.cpu().numpy()
    ds_, os_ = t_sp.data.cpu().numpy().view(np.uint32), t_sp.offsets.cpu().numpy()
    hu, hou = h_un.data.cpu().numpy(), h_un.offsets.cpu().numpy()
    hs, hos = h_sp.data.cpu().numpy(), h_sp.offsets.cpu().numpy()
    e0, cell = 0, 0
    for c, k in enumerate(n_el):
        for h in range(p):
            want = np.concatenate([hu[hou[e * p + h]: hou[e * p + h + 1]] for e in range(e0, e0 + k)])
            assert (hs[hos[c * p + h]: hos[c * p + h + 1]] == want).all()
        for ti in range(T):
            for h in range(p):
                want = np.concatenate([du[ou[(e * T + ti) * p + h]: ou[(e * T + ti) * p + h + 1]] for e in range(e0, e0 + k)])
                assert (ds_[os_[cell]: os_[cell + 1]] == want).all(), (c, ti, h)
                cell += 1
        e0 += k


def test_more_than_8_tracks_and_exonic_filter(env):
    import genvarloader_b200 as m

    d, ds, rows, O = env
    names = [f"track{i}" for i in range(10)]
    fills = [FILLS[k](m) for k in ("repeat5p", "repeat5p_norm", "constant", "flank", "interp1", "interp2", "interp3",
                                   "flank", "repeat5p", "interp1")]
    for exonic in (False, True):
        sp = ds.with_tracks(names).with_insertion_fill(dict(zip(names, fills))).with_settings(
            splice_info=rows, var_filter="exonic" if exonic else False)
        r_sel, s_sel = [3, 0, 2, 5, 1], [0, 2, 1, 1, 0]
        _, trk = sp[r_sel, s_sel]
        e_reg, e_s, n_el = _element_batch(d, rows, list(zip(r_sel, s_sel)))
        exp, oo = _oracle_realigned(d, O, e_reg, e_s, fills, names, _seed(e_reg, e_s, d.n_samples), exonic=exonic)
        _check_realigned(trk, exp, oo, n_el, d.ploidy)


def test_painted_tracks_reference_and_tracks_only(env):
    """realign_tracks=False, "reference" sequences and tracks only: painted stored intervals over every element region,
    reversed element by element on negative strands, (pairs..., t, ~l) -- no ploidy axis."""
    d, ds, rows, O = env
    names = ["track4", "track0", "track9"]
    r_sel, s_sel = [2, 0, 4, 1], [1, 1, 0, 2]
    e_reg, e_s, n_el = _element_batch(d, rows, list(zip(r_sel, s_sel)))
    exp, offs_e = _oracle_painted(d, O, e_reg, e_s, names)
    base = ds.with_tracks(names)
    h, trk = base.with_settings(splice_info=rows, realign_tracks=False)[r_sel, s_sel]
    assert h.shape == (4, d.ploidy, None) and trk.shape == (4, 3, None)
    _check_painted(trk, exp, offs_e, n_el)
    for enc in ("bytes", "onehot"):
        seq, trk = base.with_seqs("reference").with_encoding(enc).with_settings(splice_info=rows)[r_sel, s_sel]
        assert seq.shape == (4, None) and trk.shape == (4, 3, None)
        _check_painted(trk, exp, offs_e, n_el)
        regions = d.regions[e_reg]
        e_ref = O.get_reference(np.ascontiguousarray(regions[:, :3]), offs_e, d.reference, d.ref_offsets, N, False,
                                regions[:, 3] == -1)
        got = seq.data.cpu().numpy()
        assert (got == (O.onehot(e_ref) if enc == "onehot" else e_ref)).all()
        assert (seq.offsets.cpu().numpy() == offs_e[np.concatenate([[0], np.cumsum(n_el)])]).all()
    trk = base.with_seqs(None).with_settings(splice_info=rows)[r_sel, s_sel]
    _check_painted(trk, exp, offs_e, n_el)
    # rc_neg=False: nothing is reversed
    exp_f, _ = _oracle_painted(d, O, e_reg, e_s, names, rc_neg=False)
    _check_painted(base.with_seqs(None).with_settings(splice_info=rows, rc_neg=False)[r_sel, s_sel], exp_f, offs_e, n_el)


def test_single_element_rows_and_output_shapes(env):
    import torch

    d, ds, rows, _ = env
    names = ["track2", "track6"]
    base = ds.with_tracks(names)
    sp = base.with_settings(splice_info=rows)
    # a one-element row equals the unspliced dataset at that region
    for r_row, region in ((1, 5), (5, 10)):
        for s in range(d.n_samples):
            (h1, t1), (h0, t0) = sp[r_row, s], base[region, s]
            assert t1.shape == (2, d.ploidy, None) and h1.shape == (d.ploidy, None)
            assert (t1.data.view(torch.int32) == t0.data.view(torch.int32)).all() and (t1.offsets == t0.offsets).all()
            assert (h1.data == h0.data).all()
    # int/int squeezes like the sequences; slices and outer indexing keep (rows, samples)
    h, t = sp[2, 0]
    assert t.shape == (2, d.ploidy, None)
    h, t = sp[1:4, [0, 2]]
    assert t.shape == (3, 2, 2, d.ploidy, None) and h.shape == (3, 2, d.ploidy, None)
    h2, t2 = sp[[1, 2, 3], [2, 2, 2]]
    whole = t.data.view(torch.int32)
    assert t2.shape == (3, 2, d.ploidy, None)
    o, o2 = t.offsets.cpu().numpy(), t2.offsets.cpu().numpy()
    per = 2 * d.ploidy  # cells of one (row, sample)
    for j in range(3):  # pair j of the paired call is cell (j, 1) of the outer call
        a = whole[o[(2 * j + 1) * per]: o[(2 * j + 2) * per]]
        b = t2.data.view(torch.int32)[o2[j * per]: o2[(j + 1) * per]]
        assert (a == b).all()
    # "variable": tracks pad with 0.0, sequences with N
    hv, tv = sp.with_len("variable")[1:4, [0, 2]]
    lens = t.lengths.cpu().numpy().reshape(-1)
    assert tuple(tv.shape) == (3, 2, 2, d.ploidy, int(lens.max()))
    flat = tv.reshape(-1, tv.shape[-1]).cpu().numpy()
    for k in range(lens.size):
        assert (flat[k, : lens[k]].view(np.uint32) == t.data[o[k]: o[k + 1]].cpu().numpy().view(np.uint32)).all()
        assert (flat[k, lens[k]:] == 0.0).all()
    assert (hv.reshape(-1, hv.shape[-1])[:, -1:] == N).any()
    # "flat": the Ragged triple, untouched
    hf, tf = sp.with_output_format("flat").with_len("variable")[1:4, [0, 2]]
    assert (tf.data.view(torch.int32) == whole).all() and (tf.offsets == t.offsets).all()


def test_open_bed_column_splice_rows_with_an_annotation_track(env, cuda_device, tmp_path):
    """Splice rows from input-BED columns of an opened dataset with one sample track and one annotation track (one interval
    slot per region): the annotation track reads slot r_k of every element."""
    import pyarrow as pa
    import pyarrow.ipc as ipc

    from genvarloader_b200 import Dataset, synth
    from tests._gvl_disk import write_fasta, write_gvl_dataset

    d = synth.make_dataset(43, 150_000, 3, 10, 1500, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=1, max_indel=9)
    d.tracks["annot"] = synth.make_track(np.random.default_rng(5), d.regions, 1)
    rows = {"tA": [3, 0, 7], "tB": [5], "tC": [9, 8, 2]}
    order = np.arange(d.n_regions)
    write_gvl_dataset(tmp_path / "ds", d, ["chr1"], ["a", "b", "c"], order, annot_tracks=("annot",))
    with pa.memory_map(str(tmp_path / "ds" / "input_regions.arrow"), "r") as src:
        bed = ipc.open_file(src).read_all()
    tid, rank = ["x"] * d.n_regions, [0] * d.n_regions
    for name, idxs in rows.items():
        for k, r in enumerate(idxs):
            tid[r], rank[r] = name, k
    bed = bed.append_column("transcript", pa.array(tid)).append_column("exon", pa.array(rank))
    with pa.OSFile(str(tmp_path / "bed.new"), "wb") as f, ipc.new_file(f, bed.schema) as w:
        w.write_table(bed)
    del bed
    (tmp_path / "bed.new").replace(tmp_path / "ds" / "input_regions.arrow")
    write_fasta(tmp_path / "ref.fa", d.reference, d.ref_offsets, ["chr1"])
    dsk = Dataset.open(tmp_path / "ds", tmp_path / "ref.fa", device=cuda_device)
    assert dsk.track_kinds == {"track0": "sample", "annot": "annot"}
    spd = dsk.with_tracks(["annot", "track0"]).with_settings(splice_info=("transcript", "exon"))
    names = list(spd.splice_names)
    O = env[3]
    for row in ("tA", "tC"):
        for s in range(3):
            _, trk = spd[names.index(row), s]
            e_reg = np.array(rows[row], np.int64)
            e_s = np.full(e_reg.size, s, np.int64)
            seed = _seed(e_reg, e_s, d.n_samples)
            p = d.ploidy
            ds_idx = e_reg * d.n_samples + e_s
            regions = np.ascontiguousarray(d.regions[e_reg, :3])
            goi = ds_idx[:, None] * p + np.arange(p)[None, :]
            diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2],
                                       d.v_starts)
            lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)
            oo = np.concatenate([[0], np.cumsum(np.maximum(lengths[:, None] + diffs, 0).ravel())]).astype(np.int64)
            to = np.concatenate([[0], np.cumsum(lengths - diffs.clip(max=0).min(1))]).astype(np.int64)
            exp = []
            for name, slots in (("annot", e_reg), ("track0", ds_idx)):
                st, en, v, io = d.tracks[name]
                buf = np.zeros(int(oo[-1]), np.float32)
                O.intervals_and_realign_track_fused(buf, oo, regions, np.zeros(goi.shape, np.int32), goi, d.geno_v_idxs,
                                                    d.geno_offsets, d.v_starts, d.ilens, slots, st, en, v, io, to,
                                                    np.array([0.0]), 0, seed, None, None, np.repeat(d.regions[e_reg, 3] == -1, p))
                exp.append(buf)
            _check_realigned(trk.reshape((1, 2, p)), exp, oo, [e_reg.size], p)


def test_to_dataloader_yields_the_tracks(env):
    d, ds, rows, _ = env
    sp = ds.with_tracks(["track1", "track7"]).with_settings(splice_info=rows)
    n = 0
    for k, (h, t) in enumerate(sp.to_dataloader(batch_size=4)):
        idx = np.arange(4 * k, min(4 * k + 4, len(sp)))
        eh, et = sp[idx // sp.n_samples, idx % sp.n_samples]
        assert (h.data == eh.data).all() and (h.offsets == eh.offsets).all()
        assert (t.data.view(-1).view(dtype=__import__("torch").int32) == et.data.view(dtype=__import__("torch").int32)).all()
        assert (t.offsets == et.offsets).all() and t.shape == et.shape
        n += len(idx)
    assert n == len(sp)


def test_library_calls_do_not_grow_with_the_batch(env, monkeypatch):
    """One track call per ds[...]: the number of library calls does not depend on the number of pairs, elements or tracks."""
    from genvarloader_b200 import _engine

    d, ds, rows, _ = env
    calls = []

    class Counting:
        def __init__(self, lib):
            self._lib = lib

        def __getattr__(self, name):
            fn = getattr(self._lib, name)

            def wrapped(*a):
                calls.append(name)
                return fn(*a)

            return wrapped

    monkeypatch.setattr(_engine, "lib", Counting(_engine.lib))

    def count(ds_, idx):
        calls.clear()
        ds_[idx]
        return list(calls)

    for realign in (True, False):
        small = ds.with_tracks(["track0"]).with_settings(splice_info=rows, realign_tracks=realign)
        big = ds.with_tracks([f"track{i}" for i in range(10)]).with_settings(splice_info=rows, realign_tracks=realign)
        a = count(small, ([1], [0]))
        b = count(big, (slice(None), slice(None)))
        assert a == b and len(a) <= 6, (a, b)


def test_svar2_source(cuda_device):
    """Spliced haplotypes and realigned tracks over a resident svar2 source: the oracle's svar2 composition over E
    (dense source windows painted from the intervals, shift_and_realign_tracks_from_svar2, reversal of negative rows)."""
    from genvarloader_b200 import Dataset, FlankSample, synth
    from oracle import oracle as O

    d = synth.make_dataset(47, 300_000, 3, 8, 2500, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=1, max_indel=15,
                           snp_frac=0.5)
    sv = synth.to_svar2_dataset(d, dense_frac=0.5, seed=2)
    rows = [[2, 0, 5], [7], [1, 3, 3]]
    ds2 = Dataset.from_synth(cuda_device, d, rng=1, svar2=sv).with_insertion_fill(FlankSample(3))
    ds1 = Dataset.from_synth(cuda_device, d, rng=1).with_insertion_fill(FlankSample(3))
    r_sel, s_sel = [0, 2, 1, 0], [1, 0, 2, 2]
    (h2, t2) = ds2.with_settings(splice_info=rows)[r_sel, s_sel]
    (h1, t1) = ds1.with_settings(splice_info=rows)[r_sel, s_sel]
    assert (h2.data == h1.data).all() and (h2.offsets == h1.offsets).all()
    e_reg = np.concatenate([rows[r] for r in r_sel]).astype(np.int64)
    e_s = np.concatenate([[s] * len(rows[r]) for r, s in zip(r_sel, s_sel)]).astype(np.int64)
    n_el = [len(rows[r]) for r in r_sel]
    ds_idx = e_reg * d.n_samples + e_s
    p = d.ploidy
    regions = np.ascontiguousarray(d.regions[e_reg, :3])
    ch = synth.svar2_batch_channels(sv, ds_idx, p, d.n_samples)
    cargs = (ch["vk_pos"], ch["vk_key"], ch["vk_off"], ch["dense_pos"], ch["dense_key"], ch["dense_range"], ch["dense_present"],
             ch["dense_present_off"])
    diffs = O.hap_diffs_svar2(regions, p, *cargs, ch["key_ilen"])
    lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)
    oo = np.concatenate([[0], np.cumsum(np.maximum(lengths[:, None] + diffs, 0).ravel())]).astype(np.int64)
    to = np.concatenate([[0], np.cumsum(lengths - diffs.clip(max=0).min(1))]).astype(np.int64)
    s, e, v, io = d.tracks["track0"]
    dense = np.zeros(int(to[-1]), np.float32)
    O.intervals_to_tracks(ds_idx, regions[:, 1], s, e, v, io, dense, to)
    exp = np.zeros(int(oo[-1]), np.float32)
    O.shift_and_realign_tracks_from_svar2(exp, oo, regions, np.zeros((len(e_reg), p), np.int32), *cargs, ch["key_ilen"], dense, to,
                                          np.array([3.0]), 3, _seed(e_reg, e_s, d.n_samples))
    O.reverse_flat_rows_inplace(exp, oo, np.repeat(d.regions[e_reg, 3] == -1, p))
    _check_realigned(t2, [exp], oo, n_el, p)
    assert (t2.data.cpu().numpy().view(np.uint32) == t1.data.cpu().numpy().view(np.uint32)).all()
