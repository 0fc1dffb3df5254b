"""State rules of `with_tracks(kind="intervals")` and the `RaggedIntervals` container (no GPU needed): the kind is
validated and kept, intervals are never realigned (the realigning states and `with_insertion_fill` refuse), and the
read-ahead loaders leave interval reads to the batch-by-batch loader."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
from genvarloader_b200 import RaggedIntervals, Repeat5p  # noqa: E402
from genvarloader_b200._dataset import BatchLoader, Dataset  # noqa: E402
from genvarloader_b200._types import Ragged  # noqa: E402
from genvarloader_b200 import _pipeline, _variants_loader  # noqa: E402


def _ds(R=6, S=3, L=100, max_jitter=4):
    regions = np.stack([np.zeros(R), np.arange(R) * 1000, np.arange(R) * 1000 + L, np.ones(R)], 1).astype(np.int32)
    return Dataset(engine=None, full_regions=regions, sample_names=tuple(f"s{i}" for i in range(S)), ploidy=2,
                   max_jitter=max_jitter, track_kinds={"t0": "sample", "t1": "annot"}, active_tracks=("t0", "t1"))


def test_kind_is_validated():
    ds = _ds().with_settings(realign_tracks=False)
    for bad in ("painted", "bigwig", 1, True):
        with pytest.raises(ValueError, match="track kind"):
            ds.with_tracks(kind=bad)
    assert ds.track_output == "tracks"
    assert ds.with_tracks(kind="tracks").track_output == "tracks"
    assert ds.with_tracks(kind="intervals").track_output == "intervals"


def test_kind_none_keeps_the_current_kind():
    ds = _ds().with_settings(realign_tracks=False).with_tracks(kind="intervals")
    assert ds.with_tracks().track_output == "intervals"
    assert ds.with_tracks("t1").track_output == "intervals"
    assert ds.with_tracks("t1").active_tracks == ("t1",)
    assert ds.with_tracks(kind="tracks").with_tracks("t0").track_output == "tracks"
    # the other with_* keep it as well
    assert ds.with_len(50).with_seqs("reference").with_settings(jitter=2).track_output == "intervals"


@pytest.mark.parametrize("seqs", ["haplotypes", "annotated"])
def test_realigning_states_refuse_intervals(seqs):
    ds = _ds().with_seqs(seqs)
    assert ds.realign_tracks
    with pytest.raises(ValueError, match="realign_tracks=False"):
        ds.with_tracks(kind="intervals")
    iv = ds.with_settings(realign_tracks=False).with_tracks(kind="intervals")
    assert iv.sequence_type == seqs
    with pytest.raises(ValueError, match="realign_tracks=False"):
        iv.with_settings(realign_tracks=True)
    # states that paint accept intervals
    for s in (None, "reference", "variants"):
        assert _ds().with_seqs(s).with_tracks(kind="intervals").track_output == "intervals"
    # no active track: nothing would be realigned
    assert ds.with_tracks(False, kind="intervals").active_tracks == ()


def test_insertion_fill_refuses_intervals():
    ds = _ds().with_settings(realign_tracks=False).with_tracks(kind="intervals")
    with pytest.raises(ValueError, match="kind='intervals'"):
        ds.with_insertion_fill(Repeat5p())
    assert _ds().with_insertion_fill(Repeat5p()).insertion_fill  # (the painted-value states are unchanged)


@pytest.mark.parametrize("length", [64, "ragged", "variable"])
@pytest.mark.parametrize("seqs", [None, "reference", "haplotypes"])
@pytest.mark.parametrize("mode", ["buffered", "double_buffered"])
def test_pipelined_loaders_fall_back_to_batch_loader(length, seqs, mode):
    ds = _ds().with_seqs(seqs).with_settings(realign_tracks=False).with_len(length)
    iv = ds.with_tracks(kind="intervals")
    assert _pipeline.supports(iv) is not None
    assert _variants_loader.supports(iv) is not None
    assert isinstance(iv.to_dataloader(batch_size=4, mode=mode), BatchLoader)
    if length == 64:  # the painted twin of a fixed-length state is served by the pipeline
        assert _pipeline.supports(ds) is None
    assert _variants_loader.supports(ds.with_seqs("variants").with_tracks(kind="intervals")) is not None


def test_ragged_intervals_container():
    off = torch.tensor([0, 2, 2, 3, 6, 6, 7])
    s = torch.arange(7, dtype=torch.int32) * 10
    v = torch.linspace(0, 1, 7).to(torch.bfloat16)
    ri = RaggedIntervals(Ragged(s, off, (1, 3, 2, None)), Ragged(s + 5, off, (1, 3, 2, None)), Ragged(v, off, (1, 3, 2, None)))
    assert ri.shape == (1, 3, 2, None) and ri.offsets is off
    assert ri.lengths.tolist() == [[[2, 0], [1, 3], [0, 1]]]
    sq = ri.squeeze(0)
    assert sq.shape == (3, 2, None) and sq.ends.shape == (3, 2, None) and sq.values.shape == (3, 2, None)
    assert ri.reshape((6,)).shape == (6, None) and ri.reshape(6).values.shape == (6, None)
    cells = ri.to_list()
    assert len(cells) == 6 and [len(c) for c in cells] == [2, 0, 1, 3, 0, 1]
    assert cells[3] == [(30, 35, float(v[3])), (40, 45, float(v[4])), (50, 55, float(v[5]))]
