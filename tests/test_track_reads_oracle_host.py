"""Host pieces of the track-read oracle (tests/_track_reads.py): the 16-bit rounding, the exact bin reference, the edge
track and the draw order of the restatement."""
from fractions import Fraction

import numpy as np
import pytest

from tests import _track_reads as TR


def _f(bits):
    return np.array(bits, np.uint32).view(np.float32)


def test_bf16_rounds_to_nearest_even_on_the_bits():
    x = _f([0x3F808000, 0x3F818000, 0x3F808001, 0x3F807FFF, 0x7F7FFFFF, 0xFF7FFFFF, 0x00000001, 0x80000000,
            0x7F800000, 0x3F800000, 0x477FE000])
    want = [0x3F80, 0x3F82, 0x3F81, 0x3F80, 0x7F80, 0xFF80, 0x0000, 0x8000, 0x7F80, 0x3F80, 0x4780]
    assert TR.bf16_bits(x).tolist() == want
    nan = TR.bf16_bits(_f([0x7FC00001, 0xFFC00000]))
    assert TR.bits_are_nan(nan, "bfloat16").all() and (nan >> 15).tolist() == [0, 1]


def test_f16_edges():
    x = np.array([6e-8, 1e-7, 65504.0, 65519.996, 65520.0, -0.0, 1e-40], np.float32)
    assert TR.f16_bits(x).tolist() == [0x0001, 0x0002, 0x7BFF, 0x7BFF, 0x7C00, 0x8000, 0x0000]


def test_round_f32_is_one_rounding():
    assert TR.round_f32(1, -149) == _f(1)                                      # smallest subnormal
    assert TR.round_f32(1, -150) == 0.0                                        # a tie at half of it: to even (zero)
    assert TR.round_f32(3, -150).view(np.uint32) == 2                          # 1.5 units: to even (2)
    assert TR.round_f32((1 << 24) + 1, 0) == np.float32(1 << 24)               # tie below: even
    assert TR.round_f32((1 << 24) + 3, 0) == np.float32((1 << 24) + 4)         # tie above: even
    assert TR.round_f32((1 << 128) - (1 << 103), 0) == np.inf                  # the overflow threshold (a tie)
    assert TR.round_f32((1 << 128) - (1 << 103) - 1, 0) == np.finfo(np.float32).max
    assert TR.round_f32(-5, -1) == np.float32(-2.5)


def test_exactly_summable_and_the_exact_bin():
    big = np.float32(2.0 ** 60)
    bin_ = np.array([big, 1.0, -big, 0.0], np.float32)
    # 2**60 / 1 (the smallest ulp: of the value 1.0 is 2**-23) is far beyond 2**53: the order decides the float64 sum
    assert not TR.exactly_summable(bin_)
    assert TR.exact_bin(bin_, "sum") == np.float32(1.0)
    assert (big + 1.0) - big == 0.0 and (big - big) + 1.0 == 1.0  # {2^60, 1, -2^60}: 0 in one order, 1 in another
    assert TR.exact_bin(bin_, "mean") == np.float32(0.25)
    v = np.float32(2.0 ** 20) + np.arange(1, 9, dtype=np.float32) / np.float32(8)
    assert TR.exactly_summable(v)
    s = sum(Fraction(float(a)) for a in v)
    assert TR.exact_bin(v, "sum") == np.float32(float(s)) == np.float32(8 * 2 ** 20 + 4.5)
    acc = np.float32(0)
    for a in v:
        acc = np.float32(acc + a)  # a float32 accumulator loses the eighths
    assert acc != TR.exact_bin(v, "sum")
    assert TR.exactly_summable(np.array([1e-40, -1.4e-45, 0.0, -0.0], np.float32))
    assert TR.exact_bin(np.array([-1.5, -3.25], np.float32), "max") == np.float32(-1.5)
    assert np.isnan(TR.exact_bin(np.array([1.0, np.nan], np.float32), "max"))
    assert np.isnan(TR.exact_bin(np.array([np.inf, -np.inf], np.float32), "sum"))
    assert TR.exact_bin(np.array([np.inf, 1.0], np.float32), "mean") == np.inf
    m = np.finfo(np.float32).max
    assert TR.exact_bin(np.array([m, m], np.float32), "sum") == np.inf
    assert TR.exact_bin(np.array([m, m], np.float32), "mean") == m


def test_assert_bins_flags_a_float32_accumulator():
    v = (np.float32(2.0 ** 20) + np.arange(1, 17, dtype=np.float32) / np.float32(8)).astype(np.float32)
    exp = TR.narrow_bits(np.array([TR.exact_bin(v, "sum")], np.float32), "float32")
    assert TR.assert_bins(exp, v, 16, "sum", "float32") == (1, 1)
    acc = np.float32(0)
    for a in v:
        acc = np.float32(acc + a)
    with pytest.raises(AssertionError):
        TR.assert_bins(np.array([acc], np.float32).view(np.uint32), v, 16, "sum", "float32")
    # max: a bin of negative values is not 0
    neg = np.full(8, -1.5, np.float32)
    with pytest.raises(AssertionError):
        TR.assert_bins(np.zeros(1, np.uint32), neg, 8, "max", "float32")


def test_edge_track_holds_every_listed_value():
    rng = np.random.default_rng(0)
    regions = np.array([[0, 100, 420, 1], [0, 600, 920, -1]], np.int32)
    s, e, v, off = TR.make_edge_track(rng, regions, 3, 8)
    assert off[-1] == s.size == v.size and (e > s).all()
    bits = set(v.view(np.uint32).tolist())
    listed = [0x00000000, 0x80000000, 0x3F808000, 0x3F818000, 0x7F7FFFFF, 0xFF7FFFFF, 0x7F800000, 0xFF800000,
              0x7FC00001, 0xFFC00000]
    listed += [int(np.float32(x).view(np.uint32)) for x in (1e-40, -1.4e-45, 6e-8, 1e-7, 65504.0, 65519.996, 65520.0)]
    assert not set(listed) - bits, [hex(b) for b in set(listed) - bits]
    assert np.float32(65519.996).astype(np.float16) == np.float16(65504)
    assert (v < 0).any() and (v[v < 0] > -np.inf).any()
    assert ((v >= 2.0 ** 20) & (v < 2.0 ** 21) & (v != np.floor(v))).sum() > 10
    for k in range(off.size - 1):  # every slot covers its expanded region without holes
        a, b = off[k], off[k + 1]
        assert (s[a + 1:b] == e[a:b - 1]).all()


class _Recorder:
    """Stands in for the oracle module: records nothing, returns zero diffs and writes zeros."""

    def __init__(self, diffs):
        self.diffs = diffs

    def get_diffs_sparse(self, goi, *a, **k):
        return self.diffs[: goi.shape[0]].copy()

    def choose_exonic_variants(self, *a, **k):
        raise AssertionError("not used")

    def intervals_and_realign_track_fused(self, *a, **k):
        pass

    def intervals_to_tracks(self, *a, **k):
        pass

    def reverse_flat_rows_inplace(self, *a, **k):
        pass


def _tiny():
    from genvarloader_b200 import synth

    d = synth.make_dataset(3, 5000, 3, 4, 100, 5.0, max_jitter=6, n_tracks=1)
    return d, {"track0": "sample"}


@pytest.mark.parametrize("jitter", [0, 6])
def test_draw_order_matches_a_hand_replay(jitter):
    d, kinds = _tiny()
    ds_idx = np.array([0, 5, 7, 11, 2])
    diffs = np.array([[3, -2], [0, 4], [-1, -1], [2, 0], [0, 0]], np.int32)
    st = TR.ReadState(seqs="haplotypes", length=90, jitter=jitter, deterministic=False, tracks=("track0",))
    got = TR.read_tracks(_Recorder(diffs), d, kinds, st, ds_idx, 77)
    rng = np.random.default_rng(77)
    jit = rng.integers(-jitter, jitter + 1, size=5, dtype=np.int32)  # 1. jitter (a zero range draws nothing)
    if jitter:
        assert np.array_equal(got.draws["jitter"], jit)
    else:
        assert "jitter" not in got.draws
    max_shift = diffs.clip(min=0) + (100 - 90)                      # 2. shifts: diffs + what the window leaves
    assert np.array_equal(got.draws["shifts"], rng.integers(0, max_shift + 1, dtype=np.int32))
    assert got.draws["fill_seed"] == int(rng.integers(0, np.iinfo(np.uint64).max, dtype=np.uint64))  # 3. fill seed
    # a zero-range integer draw consumes nothing, so drawing jitter 0 or not leaves the same state behind
    a, b = np.random.default_rng(5), np.random.default_rng(5)
    a.integers(0, 1, size=9, dtype=np.int32)
    assert a.integers(0, 1 << 30) == b.integers(0, 1 << 30)


def test_draws_only_where_the_read_makes_them():
    d, kinds = _tiny()
    ds_idx = np.array([1, 4])
    diffs = np.zeros((2, 2), np.int32)
    for st, keys in [(TR.ReadState(seqs="haplotypes", length="ragged", deterministic=False, tracks=("track0",)), {"fill_seed"}),
                     (TR.ReadState(seqs=None, length=90, jitter=2, deterministic=False, tracks=("track0",)), {"jitter"}),
                     (TR.ReadState(seqs="haplotypes", realign=False, length=90, deterministic=False, tracks=("track0",)),
                      {"shifts"}),
                     (TR.ReadState(seqs="reference", length=90, deterministic=False, tracks=("track0",)), set())]:
        assert set(TR.read_tracks(_Recorder(diffs), d, kinds, st, ds_idx, 1).draws) == keys, st
    det = TR.read_tracks(_Recorder(diffs), d, kinds, TR.ReadState(length=90, tracks=("track0",)), np.array([5, 11]), 1)
    assert det.draws == {}
