"""`with_tracks(kind="realigned-intervals")` without a GPU: the numpy restatement of the definition (tests/_realigned_intervals.py)
painted back into zeros is, bit for bit, the oracle's realigned track (intervals_and_realign_track_fused) on seeded cases
with every insertion fill, shifts, unsorted variant lists and windows past both ends of the stored intervals; hand-written
answers for intervals that span indels; and the state rules of the kind."""
import numpy as np
import pytest

from tests import _realigned_intervals as RI

torch = pytest.importorskip("torch")
from genvarloader_b200 import Constant, FlankSample, Interpolate, Repeat5p  # noqa: E402
from genvarloader_b200._dataset import BatchLoader, Dataset  # noqa: E402
from genvarloader_b200 import _pipeline, _variants_loader  # noqa: E402

FILLS = [(RI.REPEAT_5P, 0.0), (RI.REPEAT_5P_NORM, 0.0), (RI.CONSTANT, 2.5), (RI.FLANK_SAMPLE, 3.0), (RI.INTERPOLATE, 1.0),
         (RI.INTERPOLATE, 3.0)]


def _case(seed, unsorted=False, shifts=False):
    """Six queries x two ploids over windows that start before and end past the stored intervals; per query one slot of
    non-overlapping intervals (gaps, adjacent pairs, 1 bp ones) and per row a random list of indels and SNPs."""
    rng = np.random.default_rng(seed)
    n_q, p = 6, 2
    starts = np.array([-7, 40, 200, 415, 600, 820], np.int64)
    lens = rng.integers(30, 90, n_q)
    regions = np.stack([np.zeros(n_q), starts, starts + lens], 1).astype(np.int32)
    itv_s, itv_e, itv_v, counts = [], [], [], []
    for q in range(n_q):
        a = int(starts[q]) + 3  # nothing stored at the window's first positions: the window reaches past the slot
        pos = a
        n = 0
        while pos < int(starts[q] + lens[q]) - 4:  # ... and none at its last ones
            pos += int(rng.integers(0, 4))
            w = int(rng.integers(1, 9))
            itv_s.append(pos)
            itv_e.append(pos + w)
            itv_v.append(float(rng.integers(1, 64)) / 8)
            pos += w
            n += 1
        counts.append(n)
    itv_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    v_starts, ilens, rows = [], [], []
    for k in range(n_q * p):
        q = k // p
        n = int(rng.integers(0, 9))
        ps = np.sort(rng.integers(int(starts[q]) - 6, int(starts[q] + lens[q]) + 4, n))
        if unsorted and n > 2:
            rng.shuffle(ps)
        row = []
        for x in ps:
            v_starts.append(int(x))
            ilens.append(int(rng.choice([-5, -3, -1, 0, 0, 1, 2, 4, 7])))
            row.append(len(v_starts) - 1)
        rows.append(row)
    geno_offsets = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    geno_v_idxs = np.concatenate([np.asarray(r, np.int32) for r in rows] + [np.zeros(0, np.int32)])
    sh = rng.integers(0, 6, (n_q, p)).astype(np.int32) if shifts else np.zeros((n_q, p), np.int32)
    row_len = np.repeat(lens, p) - (rng.integers(0, 4, n_q * p) if shifts else 0)
    track_n = lens + 16  # (generous source windows: the oracle reads its painted scratch without bounds checks)
    return dict(n_q=n_q, p=p, regions=regions, v_starts=np.asarray(v_starts, np.int32), ilens=np.asarray(ilens, np.int32),
                geno_v_idxs=geno_v_idxs, geno_offsets=geno_offsets, rows=rows, shifts=sh, row_len=row_len.astype(np.int64),
                track_n=track_n.astype(np.int64), itv=(np.asarray(itv_s, np.int32), np.asarray(itv_e, np.int32),
                                                      np.asarray(itv_v, np.float32), itv_off),
                to_rc=np.arange(n_q * p) % 3 == 1)


def _oracle(c, strategy, param, base_seed):
    from oracle import oracle as O

    out_offsets = np.concatenate([[0], np.cumsum(c["row_len"])]).astype(np.int64)
    out = np.zeros(int(out_offsets[-1]), np.float32)
    goi = np.arange(c["n_q"] * c["p"], dtype=np.int64).reshape(c["n_q"], c["p"])
    s, e, v, io = c["itv"]
    O.intervals_and_realign_track_fused(out, out_offsets, c["regions"], c["shifts"], goi, c["geno_v_idxs"], c["geno_offsets"],
                                        c["v_starts"], c["ilens"], np.arange(c["n_q"]), s, e, v, io,
                                        np.concatenate([[0], np.cumsum(c["track_n"])]), np.array([param]), strategy, base_seed,
                                        to_rc=c["to_rc"].astype(np.uint8))
    return out, out_offsets


def _row(c, k, strategy, param, base_seed):
    q, h = divmod(k, c["p"])
    s, e, v, io = c["itv"]
    slot = RI.Slot(s[io[q]:io[q + 1]], e[io[q]:io[q + 1]], v[io[q]:io[q + 1]], c["regions"][q, 1], c["track_n"][q])
    r = c["rows"][k]
    return slot, RI.realigned_intervals_row(c["v_starts"][r], c["ilens"][r], None, int(c["shifts"][q, h]), slot,
                                            int(c["row_len"][k]), strategy, param, base_seed, q, h)


@pytest.mark.parametrize("strategy,param", FILLS)
@pytest.mark.parametrize("unsorted,shifts", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_restatement_paints_the_oracle(strategy, param, unsorted, shifts, seed):
    pytest.importorskip("oracle.oracle")
    c = _case(seed, unsorted, shifts)
    base_seed = 977 * seed
    out, oo = _oracle(c, strategy, param, base_seed)
    n_itv = 0
    for k in range(c["n_q"] * c["p"]):
        slot, (s, e, v) = _row(c, k, strategy, param, base_seed)
        L = int(c["row_len"][k])
        assert (np.diff(s) > 0).all() and (e > s).all() and (s[1:] >= e[:-1]).all()
        assert ((s >= slot.q_start) & (e <= slot.q_start + L)).all()
        got = RI.paint(s, e, v, slot.q_start, L, bool(c["to_rc"][k]))
        assert np.array_equal(got.view(np.int32), out[oo[k]:oo[k + 1]].view(np.int32)), k
        n_itv += len(s)
    assert n_itv > 0


def _one(v_starts, ilens, strategy=RI.REPEAT_5P, param=0.0, length=None):
    """One row over the window [90, 130) of a slot holding [80, 86) = 1.0 and [100, 120) = 2.0."""
    slot = RI.Slot([80, 100], [86, 120], [1.0, 2.0], 90, 40)
    L = 40 + sum(ilens) if length is None else length
    s, e, v = RI.realigned_intervals_row(np.asarray(v_starts), np.asarray(ilens), None, 0, slot, L, strategy, param)
    return list(zip(s.tolist(), e.tolist(), v.tolist()))


def test_an_interval_across_a_deletion_is_one_shorter_interval():
    assert _one([], []) == [(100, 120, 2.0)]
    assert _one([105], [-3]) == [(100, 117, 2.0)]
    assert _one([105, 110], [-3, -2]) == [(100, 115, 2.0)]
    # a deletion that removes the interval's end, or its start
    assert _one([117], [-5]) == [(100, 118, 2.0)]
    assert _one([97], [-5]) == [(98, 115, 2.0)]


def test_an_insertion_under_repeat5p_lengthens_the_interval():
    assert _one([105], [4]) == [(100, 124, 2.0)]
    assert _one([105, 112], [4, 2]) == [(100, 126, 2.0)]
    # the same insertion under a fill of its own cuts the interval around the inserted values
    assert _one([105], [4], RI.CONSTANT, 0.5) == [(100, 105, 2.0), (105, 110, 0.5), (110, 124, 2.0)]
    assert _one([105], [4], RI.REPEAT_5P_NORM) == [(100, 105, 2.0), (105, 110, float(np.float32(0.4))), (110, 124, 2.0)]
    # an insertion in a gap: Repeat5p repeats nothing, a constant fill is an interval of its own
    assert _one([95], [3]) == [(103, 123, 2.0)]
    assert _one([95], [3], RI.CONSTANT, 7.0) == [(95, 99, 7.0), (103, 123, 2.0)]


def _ds(R=6, S=3, L=100, max_jitter=4):
    regions = np.stack([np.zeros(R), np.arange(R) * 1000, np.arange(R) * 1000 + L, np.ones(R)], 1).astype(np.int32)
    return Dataset(engine=None, full_regions=regions, sample_names=tuple(f"s{i}" for i in range(S)), ploidy=2,
                   max_jitter=max_jitter, track_kinds={"t0": "sample", "t1": "annot"}, active_tracks=("t0", "t1"))


def test_kind_is_accepted_and_kept():
    ds = _ds().with_seqs("haplotypes")
    ri = ds.with_tracks(kind="realigned-intervals")
    assert ri.track_output == "realigned-intervals"
    assert ri.with_tracks("t1").track_output == "realigned-intervals"
    assert ri.with_seqs("annotated").with_len(50).with_settings(jitter=2).track_output == "realigned-intervals"
    assert ri.with_tracks(kind="tracks").track_output == "tracks"
    with pytest.raises(ValueError, match="realigned-intervals"):
        ds.with_tracks(kind="realigned_intervals")


@pytest.mark.parametrize("seqs", [None, "reference", "variants"])
def test_states_that_do_not_realign_refuse_the_kind(seqs):
    with pytest.raises(ValueError, match="kind='intervals'"):
        _ds().with_seqs(seqs).with_tracks(kind="realigned-intervals")
    ri = _ds().with_seqs("haplotypes").with_tracks(kind="realigned-intervals")
    with pytest.raises(ValueError, match="kind='intervals'"):
        ri.with_settings(realign_tracks=False)
    with pytest.raises(ValueError, match="kind='intervals'"):
        ri.with_seqs(seqs)
    # no active track: nothing to cut
    assert ri.with_tracks(False).with_seqs(seqs).active_tracks == ()


def test_intervals_kind_still_refuses_realigning_states():
    with pytest.raises(ValueError, match="realign_tracks=False"):
        _ds().with_seqs("haplotypes").with_tracks(kind="intervals")


def test_insertion_fill_is_accepted():
    ri = _ds().with_seqs("haplotypes").with_tracks(kind="realigned-intervals")
    fills = ri.with_insertion_fill(Constant(1.0)).with_insertion_fill({"t1": FlankSample(4)})
    assert fills.track_output == "realigned-intervals"
    assert isinstance(fills.insertion_fill["t0"], Constant) and isinstance(fills.insertion_fill["t1"], FlankSample)
    assert ri.with_insertion_fill(Interpolate(2)).with_insertion_fill(Repeat5p()).insertion_fill


@pytest.mark.parametrize("length", [64, "ragged", "variable"])
@pytest.mark.parametrize("seqs", ["haplotypes", "annotated"])
@pytest.mark.parametrize("mode", ["buffered", "double_buffered"])
def test_loaders_decline_the_kind(length, seqs, mode):
    ds = _ds().with_seqs(seqs).with_len(length)
    ri = ds.with_tracks(kind="realigned-intervals")
    assert _pipeline.supports(ri) is not None
    assert _variants_loader.supports(ri) is not None
    assert isinstance(ri.to_dataloader(batch_size=4, mode=mode), BatchLoader)
    if length == 64 and seqs == "haplotypes":  # the dense twin of a fixed-length state is served by the pipeline
        assert _pipeline.supports(ds) is None


def test_entry_declares_every_argument_and_rejects_a_null_context():
    import ctypes
    import re
    from pathlib import Path

    from genvarloader_b200 import _ffi

    header = re.sub(r"/\*.*?\*/", "", (Path(__file__).resolve().parent.parent / "include" / "gvl_b200.h").read_text(), flags=re.S)
    m = re.search(r"\bgvl_dev_realigned_track_intervals\s*\(([^)]*)\)\s*;", header)
    assert m
    fn = _ffi.lib.gvl_dev_realigned_track_intervals
    assert len(fn.argtypes) == len(m.group(1).split(",")) == 9
    args = [0 if t in (ctypes.c_int64, ctypes.c_int32) else None for t in fn.argtypes]
    assert fn(*args) == 2
    assert b"NULL" in _ffi.lib.gvl_last_error()
