"""The read-ahead loader of the `variants` / `variant-windows` outputs (genvarloader_b200/_variants_loader.py) and the
sizing pass it and every variants read share: gvl_dev_variant_row_sizes against numpy, gvl_dev_rebase_offsets against
numpy, and every loader batch against `ds[r, s]` of the same indices, field by field and bit for bit, offsets included."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

R, S, P = 40, 6, 2


def _arrays(seed=0):
    rng = np.random.default_rng(seed)
    contig_lens = [6000, 4000]
    ref_off = np.concatenate([[0], np.cumsum(contig_lens)]).astype(np.int64)
    reference = rng.choice(np.frombuffer(b"ACGTN", np.uint8), ref_off[-1])
    n_var = 900
    v_starts = np.sort(rng.integers(0, 4000, n_var)).astype(np.int32)
    v_starts[:2], v_starts[-2:] = [0, 1], [3998, 3999]
    ilens = rng.integers(-15, 16, n_var).astype(np.int32)
    alt_off = np.concatenate([[0], np.cumsum(np.where(ilens > 0, ilens + 1, 1))]).astype(np.int64)
    rfo = np.concatenate([[0], np.cumsum(np.where(ilens < 0, 1 - ilens, 1))]).astype(np.int64)
    alt = rng.choice(np.frombuffer(b"ACGT", np.uint8), alt_off[-1])
    rfa = rng.choice(np.frombuffer(b"ACGT", np.uint8), rfo[-1])
    regions = np.stack([rng.integers(0, 2, R), rng.integers(0, 3500, R), np.zeros(R, np.int64),
                        np.where(rng.random(R) < 0.5, -1, 1)], 1)
    regions[:, 2] = regions[:, 1] + 300
    # slot lengths 0..60, a third empty; the last regions carry far more variants (a later ring needs more space)
    glen = rng.integers(0, 20, R * S * P)
    glen[rng.random(R * S * P) < 0.33] = 0
    glen[(R - 8) * S * P:] = rng.integers(100, 400, 8 * S * P)
    geno_off = np.concatenate([[0], np.cumsum(glen)]).astype(np.int64)
    geno_v = np.concatenate([np.sort(rng.choice(n_var, k, replace=False)) for k in glen]).astype(np.int32)
    af = rng.random(n_var).astype(np.float32)
    dz = rng.random(len(geno_v)).astype(np.float32)
    return dict(reference=reference, ref_off=ref_off, v_starts=v_starts, ilens=ilens, alt=alt, alt_off=alt_off, rfa=rfa, rfo=rfo,
                regions=regions.astype(np.int32), geno_off=geno_off, geno_v=geno_v, af=af, dz=dz)


@pytest.fixture(scope="module")
def A():
    return _arrays()


def _dataset(dev, a, with_ref=True, rng=0):
    from genvarloader_b200._dataset import Dataset

    return Dataset.from_arrays(dev, a["reference"], a["ref_off"], a["v_starts"], a["ilens"], a["alt"], a["alt_off"], a["geno_v"],
                               a["geno_off"], a["regions"], S, P, max_jitter=5, rng=rng,
                               ref_alleles=(a["rfa"], a["rfo"]) if with_ref else None, variant_info={"AF": a["af"]},
                               dosages=a["dz"])


@pytest.fixture(scope="module")
def DS(cuda_device, A):
    return _dataset(cuda_device, A)


# ---------------------------------------------------------------- kernels
@pytest.mark.parametrize("with_ref", [False, True])
def test_row_sizes_vs_numpy(cuda_device, A, with_ref):
    """Empty slots, AF bounds equal to variants' own AF values, REF strings absent and present, 50,000 rows (more rows than
    one pass of the grid covers)."""
    ds = _dataset(cuda_device, A, with_ref)
    eng = ds.engine
    rng = np.random.default_rng(7)
    n_slots = len(A["geno_off"]) - 1
    goi = rng.integers(0, n_slots + 1, 50_000)  # (n_slots = the engine's empty slot)
    af = A["af"]
    lo, hi = np.sort(af)[[100, 800]]
    d_goi = torch.from_numpy(goi).to(cuda_device)
    a_len, r_len = np.diff(A["alt_off"]), np.diff(A["rfo"])
    span = 1 - np.minimum(A["ilens"].astype(np.int64), 0)
    go = np.append(A["geno_off"], A["geno_off"][-1])
    for min_af, max_af in ((None, None), (float(lo), float(hi)), (float(lo), None)):
        keep_v = np.ones(len(af), bool)
        if min_af is not None:
            keep_v &= af >= np.float32(min_af)
        if max_af is not None:
            keep_v &= af <= np.float32(max_af)
        assert (af == np.float32(lo)).any() and keep_v[af == np.float32(lo)].all()
        got = eng.variant_row_sizes(d_goi, min_af, max_af)
        exp = np.zeros((len(goi), 4), np.int64)
        for i, g in enumerate(goi):
            v = A["geno_v"][go[g]: go[g + 1]]
            v = v[keep_v[v]]
            exp[i] = (len(v), a_len[v].sum(), r_len[v].sum() if with_ref else 0, span[v].sum())
        assert (exp[:, 0] == 0).any() and (exp[:, 0] > 100).any()
        np.testing.assert_array_equal(got, exp)


def test_rebase_offsets_vs_numpy(DS):
    eng, dev = DS.engine, DS.engine.device
    rng = np.random.default_rng(3)
    rows = np.concatenate([[0], np.cumsum(rng.integers(0, 4, 23))]).astype(np.int64)  # 23 rows, some empty
    items = np.concatenate([[0], np.cumsum(rng.integers(0, 9, rows[-1]))]).astype(np.int64)
    d_rows, d_items = torch.from_numpy(rows).to(dev), torch.from_numpy(items).to(dev)
    for stride in (1, 5, 23, 40):
        K = -(-23 // stride)
        cut = np.minimum(np.arange(K + 1) * stride, 23)
        exp_rows = np.concatenate([rows[a: b + 1] - rows[a] for a, b in zip(cut[:-1], cut[1:])])
        np.testing.assert_array_equal(eng.rebase_offsets(d_rows, K, stride).cpu().numpy(), exp_rows)
        vc = rows[cut]
        exp_items = np.concatenate([items[a: b + 1] - items[a] for a, b in zip(vc[:-1], vc[1:])])
        np.testing.assert_array_equal(eng.rebase_offsets(d_items, K, stride, bounds=d_rows).cpu().numpy(), exp_items)


# ---------------------------------------------------------------- loader batches == ds[r, s]
def _eq_t(tag, a, b):
    assert a.dtype == b.dtype and tuple(a.shape) == tuple(b.shape), (tag, a.dtype, b.dtype, a.shape, b.shape)
    assert torch.equal(a.view(torch.uint8) if a.dtype.is_floating_point else a, b.view(torch.uint8) if b.dtype.is_floating_point else b), tag


def _same(got, exp):
    from genvarloader_b200._types import RaggedAlleles

    assert got.shape == exp.shape and list(got.fields) == list(exp.fields)
    _eq_t("offsets", got.offsets, exp.offsets)
    for k, e in exp.fields.items():
        g = got.fields[k]
        assert g.shape == e.shape
        if isinstance(e, RaggedAlleles):
            _eq_t(f"{k}.data", g.data, e.data)
            _eq_t(f"{k}.seq_offsets", g.seq_offsets, e.seq_offsets)
            _eq_t(f"{k}.var_offsets", g.var_offsets, e.var_offsets)
        else:
            _eq_t(f"{k}.data", g.data, e.data)
            _eq_t(f"{k}.offsets", g.offsets, e.offsets)


def _states(ds):
    from genvarloader_b200 import DummyVariant, VarWindowOpt

    dummy = DummyVariant(start=-5, ilen=9, alt=b"AC", ref=b"G", dosage=0.5, info={"AF": 0.25})
    v = ds.with_seqs("variants")
    every = ["alt", "start", "ref", "ilen", "dosage", "AF"]
    return {
        "default": v,
        "fields_dummy_af": v.with_settings(var_fields=every, dummy_variant=dummy, min_af=0.2, max_af=0.9),
        "union_dummy": v.with_settings(var_fields=every, dummy_variant=dummy, unphased_union=True, min_af=0.1),
        "no_rc": v.with_settings(var_fields=every, rc_neg=False),
        "flank_u8": v.with_settings(token_alphabet="ACGT", unknown_token=4, flank_length=6, dummy_variant=dummy),
        "flank_i32": v.with_settings(token_alphabet="ACGT", unknown_token=300, flank_length=3),
        "win_window": ds.with_seqs("variant-windows", VarWindowOpt(5, "ACGT", 4)).with_settings(dummy_variant=dummy),
        "win_allele": ds.with_seqs("variant-windows", VarWindowOpt(4, "ACGT", 300, ref="allele", alt="allele")),
        "win_mixed_union": ds.with_seqs("variant-windows", VarWindowOpt(2, "ACGT", 4, ref="allele")).with_settings(
            unphased_union=True, dummy_variant=dummy),
        "subset": v.with_settings(var_fields=every).subset_to(regions=np.arange(3, 37, 2), samples=[5, 0, 2]),
    }


def _check_epoch(ds, loader, n_expected):
    n = 0
    for batch, r, s in loader:
        _same(batch, ds[r, s])
        n += 1
    assert n == n_expected


@pytest.mark.parametrize("state", ["default", "fields_dummy_af", "union_dummy", "no_rc", "flank_u8", "flank_i32", "win_window",
                                   "win_allele", "win_mixed_union", "subset"])
def test_loader_batches_equal_getitem(DS, state):
    from genvarloader_b200._variants_loader import VariantsLoader

    ds = _states(DS)[state]
    n = len(ds)
    for b, ring, copy in ((7, 2, False), (16, 0, True)):
        ld = ds.to_dataloader(b, mode="double_buffered", copy=copy, ring=ring, return_indices=True)
        assert isinstance(ld, VariantsLoader)
        _check_epoch(ds, ld, -(-n // b))


@pytest.mark.parametrize("ring", [1, 2, 0])
@pytest.mark.parametrize("copy", [False, True])
def test_loader_shuffle_drop_last_rings(DS, ring, copy):
    """Shuffle with a generator, drop_last, a partial last ring; two epochs over one loader (a new order each epoch, the
    same order as the batch-by-batch loader with the same generator)."""
    ds = _states(DS)["fields_dummy_af"]
    b = 13
    for drop_last in (False, True):
        ld = ds.to_dataloader(b, shuffle=True, generator=11, mode="buffered", ring=ring, copy=copy, drop_last=drop_last,
                              return_indices=True)
        ref = ds.to_dataloader(b, shuffle=True, generator=11, drop_last=drop_last, return_indices=True)
        n_batches = len(ds) // b if drop_last else -(-len(ds) // b)
        assert len(ld) == n_batches
        orders = []
        for _ in range(2):
            got = [(r, s) for _, r, s in ld]
            exp = [(r, s) for _, r, s in ref]
            assert len(got) == n_batches
            for (r1, s1), (r2, s2) in zip(got, exp):
                np.testing.assert_array_equal(r1, r2)
                np.testing.assert_array_equal(s1, s2)
            orders.append(np.concatenate([r * ds.n_samples + s for r, s in got]))
        assert not np.array_equal(orders[0], orders[1])
        _check_epoch(ds, ld, n_batches)


def test_loader_sampler_and_transform(DS):
    ds = _states(DS)["default"]
    order = np.random.default_rng(2).permutation(len(ds))[:50]
    seen = []
    ld = ds.to_dataloader(8, sampler=order, mode="double_buffered", ring=2, transform=lambda v, r, s: (v.offsets.numel(), r, s),
                          return_indices=True)
    for n_off, r, s in ld:
        seen.append(r * ds.n_samples + s)
        assert n_off == len(r) * P + 1
    np.testing.assert_array_equal(np.concatenate(seen), order)


def test_growing_ring_keeps_earlier_views(DS):
    """Rings of growing size (the last regions carry 100-400 variants per slot): views of an earlier ring, copy=False, stay
    intact while later, larger rings are produced."""
    ds = _states(DS)["fields_dummy_af"]
    order = np.arange(len(ds))  # in order: the heavy regions come last
    ld = ds.to_dataloader(12, sampler=order, mode="double_buffered", ring=2, copy=False, return_indices=True)
    held = []
    sizes = []
    for batch, r, s in ld:
        held.append((batch, r, s))
        sizes.append(int(batch.offsets[-1]))
    assert max(sizes[-4:]) > 10 * max(sizes[:4])
    torch.cuda.synchronize()
    for batch, r, s in held:
        _same(batch, ds[r, s])


def test_one_sizing_wait_per_read_and_per_ring(DS, monkeypatch):
    """No variants read reads a value back from the device (no `.item()` / `.cpu()` / `.tolist()` of an offsets total); one
    sizing wait per ds[idx] and one per ring of the loader."""
    from genvarloader_b200._engine import Engine

    def boom(self, *a, **k):
        raise AssertionError("a device value read back in a variants read")

    calls = []
    real = Engine.variant_row_sizes

    def counted(self, *a, **k):
        calls.append(1)
        return real(self, *a, **k)

    for name in ("item", "cpu", "tolist"):
        monkeypatch.setattr(torch.Tensor, name, boom)
    monkeypatch.setattr(Engine, "variant_row_sizes", counted)
    for name, ds in _states(DS).items():
        calls.clear()
        ds[np.arange(3), np.arange(3)]
        ds[3, 2]
        assert len(calls) == 2, name
        calls.clear()
        ld = ds.to_dataloader(9, mode="double_buffered", ring=3)
        n_batches = sum(1 for _ in ld)
        assert len(calls) == -(-n_batches // 3), name


def test_jitter_draws_match_batch_loader(cuda_device, A):
    ds1 = _dataset(cuda_device, A, rng=5).with_seqs("variants").with_settings(jitter=3)
    ds2 = _dataset(cuda_device, A, rng=5).with_seqs("variants").with_settings(jitter=3)
    for _ in ds1.to_dataloader(11, shuffle=True, generator=1, mode="double_buffered", ring=2):
        pass
    for _ in ds2.to_dataloader(11, shuffle=True, generator=1):
        pass
    assert ds1.rng.bit_generator.state == ds2.rng.bit_generator.state
    assert ds1.rng.integers(0, 2**31) == ds2.rng.integers(0, 2**31)


def test_fallbacks(DS):
    from genvarloader_b200._dataset import BatchLoader

    v = DS.with_seqs("variants")
    assert isinstance(v.to_dataloader(4), BatchLoader)  # mode=None
    assert isinstance(v.to_dataloader(4, mode="double_buffered", to_host=True), BatchLoader)
    assert isinstance(v.with_settings(var_filter="exonic").to_dataloader(4, mode="double_buffered"), BatchLoader)
