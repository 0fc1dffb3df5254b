"""Host sizing of a variants read (genvarloader_b200/_variant_sizes.py, no GPU): the per-cell lengths it derives from the
four sums per genotype row equal the lengths of the buffers the numpy oracle's composition of `get_variants_flat` builds
(gather_rows -> compact_keep -> fold -> gather_alleles / assemble_variant_buffers -> fill_empty_*), for every field, fold,
dummy, flank and window mode."""
import numpy as np
import pytest

from genvarloader_b200._types import DummyVariant
from genvarloader_b200._variant_sizes import variant_buffer_sizes
from oracle import variants_oracle as O


def _tables(seed=0, n_var=400, n_slots=120, p=2):
    rng = np.random.default_rng(seed)
    contig_lens = [3000, 2000]
    ref_off = np.concatenate([[0], np.cumsum(contig_lens)]).astype(np.int64)
    reference = rng.choice(np.frombuffer(b"ACGTN", np.uint8), ref_off[-1])
    v_starts = np.sort(rng.integers(0, 2000, n_var)).astype(np.int32)
    ilens = rng.integers(-20, 21, n_var).astype(np.int32)
    alt_off = np.concatenate([[0], np.cumsum(np.where(ilens > 0, ilens + 1, 1))]).astype(np.int64)
    rfo = np.concatenate([[0], np.cumsum(np.where(ilens < 0, 1 - ilens, 1))]).astype(np.int64)
    alt = rng.choice(np.frombuffer(b"ACGT", np.uint8), alt_off[-1])
    rfa = rng.choice(np.frombuffer(b"ACGT", np.uint8), rfo[-1])
    glen = rng.integers(0, 12, n_slots)
    glen[rng.random(n_slots) < 0.35] = 0
    geno_off = np.concatenate([[0], np.cumsum(glen)]).astype(np.int64)
    geno_v = np.concatenate([np.sort(rng.choice(n_var, k, replace=False)) for k in glen]).astype(np.int32)
    af = rng.random(n_var).astype(np.float32)
    goi = rng.integers(0, n_slots, 60 * p)
    contig_rows = np.repeat(rng.integers(0, 2, 60), p).astype(np.int32)
    return dict(reference=reference, ref_off=ref_off, v_starts=v_starts, ilens=ilens, alt=alt, alt_off=alt_off, rfa=rfa, rfo=rfo,
                geno_off=geno_off, geno_v=geno_v, af=af, goi=goi, contig_rows=contig_rows)


def _row_sums(t, keep_v):
    """The four sums per genotype row, as gvl_dev_variant_row_sizes computes them."""
    out = np.zeros((len(t["goi"]), 4), np.int64)
    a_len, r_len, span = np.diff(t["alt_off"]), np.diff(t["rfo"]), 1 - np.minimum(t["ilens"].astype(np.int64), 0)
    for i, g in enumerate(t["goi"]):
        v = t["geno_v"][t["geno_off"][g]: t["geno_off"][g + 1]]
        v = v[keep_v[v]]
        out[i] = (len(v), a_len[v].sum(), r_len[v].sum(), span[v].sum())
    return out


def _cell_items(var_off, seq_off):
    return seq_off[var_off[1:]] - seq_off[var_off[:-1]]


@pytest.mark.parametrize("fold", [1, 2])
@pytest.mark.parametrize("dummy", [None, DummyVariant(alt=b"ACG", ref=b"T")])
@pytest.mark.parametrize("filtered", [False, True])
@pytest.mark.parametrize("L", [0, 4])
def test_sizes_match_oracle_composition(fold, dummy, filtered, L):
    t = _tables(seed=fold + 2 * filtered + 4 * L)
    keep_v = (t["af"] >= 0.3) & (t["af"] <= 0.8) if filtered else np.ones(len(t["af"]), bool)
    sizes = variant_buffer_sizes(_row_sums(t, keep_v), fold, dummy, L)

    go = np.stack([t["geno_off"][:-1], t["geno_off"][1:]])
    v, off = O.gather_rows(t["goi"], go, t["geno_v"])
    contigs = np.repeat(t["contig_rows"], np.diff(off))
    if filtered:
        keep = keep_v[v]
        contigs, _ = O.compact_keep(contigs, off, keep)
        v, off = O.compact_keep(v, off, keep)
    off = off[::fold].copy()
    n_cells = len(off) - 1
    assert n_cells == sizes.n_cells and (np.diff(off) == 0).any() and (np.diff(off) > 0).any()
    np.testing.assert_array_equal(sizes.raw["variants"], np.diff(off))

    lut = np.arange(256, dtype=np.uint8)
    common = (L, lut, contigs, t["v_starts"], t["ilens"], t["reference"], t["ref_off"], ord("N"))
    bufs = dict(O.assemble_variant_buffers(0, v, off, t["alt"], t["alt_off"], t["rfa"], t["rfo"], True, L > 0, 0, 0, *common))
    bufs.update(O.assemble_variant_buffers(1, v, off, t["alt"], t["alt_off"], t["rfa"], t["rfo"], False, False, 1, 1, *common))
    assert set(bufs) == ({"alt", "ref", "ref_window", "alt_window"} | ({"flank_tokens"} if L else set()))
    dummy_len = {} if dummy is None else {"alt": len(dummy.alt), "ref": len(dummy.ref), "alt_window": 2 * L + len(dummy.alt),
                                          "ref_window": 2 * L + len(dummy.ref)}
    for name, (data, so) in bufs.items():
        if name == "flank_tokens":  # 2 L tokens per variant, offsets per row
            np.testing.assert_array_equal(sizes.raw[name], 2 * L * np.diff(off))
            assert sizes.total(name, filled=False) == data.size
            if dummy is not None:
                filled, _ = O.fill_empty_fixed(data, off, 2 * L, np.uint8(0))
                assert sizes.total(name) == filled.size
            continue
        np.testing.assert_array_equal(sizes.raw[name], _cell_items(off, so), err_msg=name)
        assert sizes.total(name, filled=False) == data.size
        if dummy is not None:
            data, vo, so = O.fill_empty_seq(data, off, so, np.zeros(dummy_len[name], np.uint8))
        else:
            vo = off
        np.testing.assert_array_equal(sizes.out[name], _cell_items(vo, so), err_msg=name)
        assert sizes.total(name) == data.size
    if dummy is not None:
        _, new_off = O.fill_empty_scalar(np.zeros(int(off[-1]), np.int32), off, np.int32(0))
        np.testing.assert_array_equal(sizes.out["variants"], np.diff(new_off))
        np.testing.assert_array_equal(sizes.out["flank_tokens"], 2 * L * np.diff(new_off))
    else:
        assert sizes.out is sizes.raw


def test_batch_bounds():
    sums = np.zeros((7, 4), np.int64)
    sums[:, 0] = [1, 0, 2, 3, 0, 0, 4]
    sums[:, 1] = [5, 0, 2, 3, 0, 0, 1]
    s = variant_buffer_sizes(sums, 1, DummyVariant(alt=b"AC"), 0)
    np.testing.assert_array_equal(s.out["variants"], [1, 1, 2, 3, 1, 1, 4])
    np.testing.assert_array_equal(s.bounds("variants", 3), [0, 4, 9, 13])  # two full batches of 3 cells, one of 1
    np.testing.assert_array_equal(s.bounds("alt", 7), [0, 17])
    np.testing.assert_array_equal(s.bounds("alt", 2), [0, 7, 12, 16, 17])
    with pytest.raises(ValueError):
        variant_buffer_sizes(sums, 2)
