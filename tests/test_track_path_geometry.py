"""The geometry of tests/test_gpu_track_paths.py, checked with the C oracle alone: every indel of `geometry_dataset` lies at
the haplotype position its slot names, every chosen interval boundary changes the realigned track exactly at the output
position it was placed for, and the tiles aimed at the staging limits hold the intended numbers of records and stored
intervals.  (No GPU: the builder is verified before any device time is spent on it.)"""
import numpy as np
import pytest

from tests import test_gpu_track_paths as T


@pytest.fixture(scope="module")
def G():
    from oracle import oracle

    d, slots = T.geometry_dataset()
    return d, slots, oracle


def _host_value(d, k: int, x, track="t0"):
    """Value of the painted source of slot k at relative source position x (None: an insertion's value)."""
    if x is None:
        return None
    s, e, v, io = d.tracks[track]
    s0 = int(d.regions[k // 2, 1])
    lo, hi = int(io[k]), int(io[k + 1])
    i = lo + int(np.searchsorted(s[lo:hi], s0 + x, "right")) - 1
    return np.float32(v[i]) if i >= lo and e[i] > s0 + x else np.float32(0)


def test_records_lie_at_their_haplotype_positions(G):
    from genvarloader_b200 import synth

    d, slots, O = G
    ks = np.arange(len(slots))
    regions, goi, _, _ = synth.batch_args(d, ks // 2, ks % 2)
    args = (regions, np.zeros(goi.shape, np.int32), goi, d.geno_offsets, d.geno_v_idxs, d.v_starts, d.ilens, d.alt_alleles,
            d.alt_offsets, d.reference, d.ref_offsets, ord("N"), -1)
    hap, oo = O.reconstruct_haplotypes_fused(*args, None, None, None)
    ref = d.reference
    n_checked = 0
    for k, sl in enumerate(slots):
        for p in range(2):
            row = hap[oo[2 * k + p]: oo[2 * k + p + 1]]
            recs = T._slot_records(sl.ev[p], int(regions[k, 1]), T.GEOM_CONTIG)
            first = int(d.geno_offsets[0, 2 * k + p])
            for j, ((h, il), (pos, _, il2)) in enumerate(zip(sl.ev[p], recs)):
                vi = int(d.geno_v_idxs[first + j])
                assert il == il2 == d.ilens[vi] and pos == d.v_starts[vi]
                alt = d.alt_alleles[d.alt_offsets[vi]: d.alt_offsets[vi + 1]]
                assert row[h] == ref[pos], (k, p, h)
                if il > 0:
                    assert (row[h: h + il + 1] == alt).all(), (k, p, h)
                elif h + 1 < row.size:
                    assert row[h + 1] == ref[pos - il + 1], (k, p, h)
                n_checked += 1
    assert n_checked == sum(len(sl.ev[0]) + len(sl.ev[1]) for sl in slots)


def test_boundaries_change_the_track_where_placed(G):
    from genvarloader_b200 import synth

    d, slots, O = G
    ks = np.array([k for k, sl in enumerate(slots) if sl.L])
    regions, goi, _, ds_idx = synth.batch_args(d, ks // 2, ks % 2)
    lens = np.array([[slots[k].L] * 2 for k in ks], np.int64)
    oo = np.concatenate([[0], np.cumsum(lens.ravel())]).astype(np.int64)
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2], d.v_starts)
    to = np.concatenate([[0], np.cumsum((regions[:, 2] - regions[:, 1]) - diffs.clip(max=0).min(1))]).astype(np.int64)
    s, e, v, io = d.tracks["t0"]
    out = np.zeros(int(oo[-1]), np.float32)
    O.intervals_and_realign_track_fused(out, oo, regions, np.zeros(goi.shape, np.int32), goi, d.geno_v_idxs, d.geno_offsets,
                                        d.v_starts, d.ilens, ds_idx, s, e, v, io, to, np.array([0.0]), 0, 0, None, None, None)
    n_changes = 0
    for q, k in enumerate(ks):
        sl = slots[k]
        row = out[oo[2 * q]: oo[2 * q + 1]]  # ploid 0, forward: output position = haplotype position
        track_n = int(to[q + 1] - to[q])
        for h in sl.cuts:
            for x in (h - 1, h, h + 1):
                if 0 <= x < row.size and T.src_of(sl.ev[0], x) is not None and T.src_of(sl.ev[0], x) < track_n:
                    assert row[x] == _host_value(d, k, T.src_of(sl.ev[0], x)), (k, h, x)
            if h in sl.keep and 0 < h < row.size:
                assert row[h - 1] != row[h] and row[h] != 0, (k, h)  # two kept intervals meet at h
                n_changes += 1
    assert n_changes >= 8
    if slots[T.EMPTY].empty:
        q = int(np.flatnonzero(ks == T.EMPTY)[0])
        assert not out[oo[2 * q]: oo[2 * q + 2]].any()


def _reaching(d, k, ev, h0, h1, track="t0"):
    """Stored intervals of slot k that reach the source feeding [h0, h1) of a row without records before h1."""
    s, e, _, io = d.tracks[track]
    s0 = int(d.regions[k // 2, 1])
    lo, hi = int(io[k]), int(io[k + 1])
    a, b = T.src_of(ev, h0), T.src_of(ev, h1 - 1) + 1
    return int(((e[lo:hi] > s0 + a) & (s[lo:hi] < s0 + b)).sum())


def test_tiles_at_the_staging_limits(G):
    d, slots, _ = G
    TILE, REC, ITV = T.TILE, T.T3_REC, T.T3_ITV
    for k, extra, recs in ((T.LIM_A_F, 0, (REC - 1, REC)), (T.LIM_A_RC, 0, (REC - 1, REC)),
                           (T.LIM_B_F, 1, (130, REC + 1)), (T.LIM_B_RC, 1, (130, REC + 1))):
        sl = slots[k]
        assert sl.L == 3 * TILE
        for p in range(2):
            hs = np.array([h for h, _ in sl.ev[p]])
            assert not (hs <= TILE).any() and int(((hs > TILE) & (hs < 2 * TILE)).sum()) == recs[p], (k, p)
            assert _reaching(d, k, sl.ev[p], 0, TILE) == ITV + extra
    # the long insertion of the records-limited tile is its last staged record (virtual carry + T3_REC - 1 records)
    h, il = slots[T.LIM_B_F].ev[0][REC - 2]
    assert il == 300 and TILE < h and h + il < 2 * TILE
    ev0 = slots[T.BOTH].ev[0]
    hs = np.array([h for h, _ in ev0])
    assert int(((hs > TILE) & (hs < 2 * TILE)).sum()) > REC
    for p in range(2):
        assert T.handover_tiles(d, slots, T.BOTH, p) == [2 * TILE]
    # the long insertions cover a whole tile; the deletions are longer than one
    for k in (T.LONG_INS_F, T.LONG_INS_RC, T.CROSS):
        (h, il), = slots[k].ev[0]
        assert il > TILE
        (h, il), = slots[k].ev[1]
        assert -il > TILE
