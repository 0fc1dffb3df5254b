"""`variants` / `variant-windows` outputs of spliced datasets: a spliced cell is the concatenation, in splice-row order, of its
elements' unspliced outputs (jitter 0, ragged).  Cell (c, s, h) holds the variants rows (r_0, s, h), (r_1, s, h), ... of the
row's elements -- each with its own AF filter, dummy variant, strand and contig -- and under `unphased_union` cell (c, s) holds
every element's union row in turn.  The expected values are one oracle call over the element batch E (the selected pairs in
output order, a pair's elements in splice-row order), regrouped into cells -- bit-exact."""
import numpy as np
import pytest

from tests._golden import eq
from tests.test_gpu_variants import _check_variants, _expected_variants

pytestmark = pytest.mark.gpu
N = ord("N")
ROWS = {"a": [3, 0, 7, 1], "b": [5], "c": [11, 2, 11], "d": [1, 4, 9, 6, 8], "e": [13, 12], "f": [10]}


def _ref_alleles(rng, ilens):
    rfo = np.concatenate([[0], np.cumsum(np.where(ilens < 0, 1 - ilens, 1))]).astype(np.int64)
    return rng.choice(np.frombuffer(b"ACGT", np.uint8), rfo[-1]), rfo


@pytest.fixture(scope="module")
def O():
    from oracle import variants_oracle

    return variants_oracle


@pytest.fixture(scope="module")
def env(cuda_device):
    """Mixed strands, two contigs, a repeated element in one row, one-element rows, elements without variants (regions 4
    and 12 in every sample, ploid 1 of region 9), REF strings, an AF column and dosages."""
    from genvarloader_b200 import Dataset, synth

    d = synth.make_dataset(41, 400_000, 3, 14, 9_000, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=2,
                           max_indel=12, snp_frac=0.5)
    R, S, P = d.n_regions, d.n_samples, d.ploidy
    lens = np.array([9000, 8300, 700, 5, 1200, 3, 9000, 450, 7, 2500, 9000, 640, 6, 1000])
    d.regions[:, 2] = d.regions[:, 1] + lens
    d.regions[:, 3] = np.where(np.arange(R) % 3 == 1, -1, 1)
    rng = np.random.default_rng(9)
    contig_len = int(d.ref_offsets[-1])
    d.reference = np.concatenate([d.reference, synth.ACGT[rng.integers(0, 4, contig_len)]])
    d.ref_offsets = np.array([0, contig_len, 2 * contig_len], np.int64)
    d.regions[[2, 6, 9, 13], 0] = 1
    go = np.array(d.geno_offsets, copy=True)
    slots = np.concatenate([np.arange(r * S * P, (r + 1) * S * P) for r in (4, 12)] + [9 * S * P + np.arange(S) * P + 1])
    go[1, slots] = go[0, slots]
    d.geno_offsets = go
    rfa, rfo = _ref_alleles(rng, d.ilens)
    af = rng.random(d.v_starts.size).astype(np.float32)
    dz = rng.random(d.geno_v_idxs.size).astype(np.float32)
    ds = Dataset.from_arrays(cuda_device, d.reference, d.ref_offsets, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                             d.geno_v_idxs, d.geno_offsets, d.regions, S, P, tracks=d.tracks, rng=7, ref_alleles=(rfa, rfo),
                             variant_info={"AF": af}, dosages=dz)
    return d, ds, dict(ref=(rfa, rfo), af=af, dz=dz)


def _element_batch(rows, pairs):
    row_list = list(rows.values())
    e_reg = np.concatenate([row_list[r] for r, _ in pairs]).astype(np.int64)
    e_s = np.concatenate([[s] * len(row_list[r]) for r, s in pairs]).astype(np.int64)
    return e_reg, e_s, [len(row_list[r]) for r, _ in pairs]


def _cell_rows(n_el, p, fold):
    """Rows of a call over E (e * p + h, or e under unphased_union) that make up every spliced cell, cells in output order."""
    cells, e0 = [], 0
    for k in n_el:
        els = np.arange(e0, e0 + k)
        cells += [els] if fold else [els * p + h for h in range(p)]
        e0 += k
    return cells


def _regroup(fields, off, cells):
    """Fields over the rows of a call over E -> the same fields over the spliced cells: (fields, cell offsets)."""
    rows = np.concatenate(cells)
    var = np.concatenate([np.arange(off[r], off[r + 1]) for r in rows]).astype(np.int64)
    new_off = np.concatenate([[0], np.cumsum([sum(off[r + 1] - off[r] for r in c) for c in cells])]).astype(np.int64)
    out = {}
    for name, f in fields.items():
        if isinstance(f, tuple):
            data, so = f
            take = np.concatenate([np.arange(so[v], so[v + 1]) for v in var] + [np.zeros(0, np.int64)]).astype(np.int64)
            out[name] = (data[take], np.concatenate([[0], np.cumsum((so[1:] - so[:-1])[var])]).astype(np.int64))
        else:
            out[name] = f[var]
    return out, new_off


def _rows(rv):
    """Per output row (outer axes flattened) and field: the bytes of every variant of the row."""
    from genvarloader_b200._types import RaggedAlleles

    off = rv.offsets.cpu().numpy()
    out = {}
    for name, f in rv.fields.items():
        if isinstance(f, RaggedAlleles):
            data, so = f.data.cpu().numpy(), f.seq_offsets.cpu().numpy()
            per_var = [data[so[a]: so[a + 1]].tobytes() for a in range(so.size - 1)]
        else:
            per_var = [x.tobytes() for x in f.data.cpu().numpy()]
        out[name] = [per_var[off[r]: off[r + 1]] for r in range(off.size - 1)]
    return out


def _same(a, b):
    ra, rb = _rows(a), _rows(b)
    assert a.shape == b.shape and list(ra) == list(rb)
    assert ra == rb


# ---------------------------------------------------------------------------------------------------- vs the oracle
def test_variants_vs_oracle(env, O):
    from genvarloader_b200 import DummyVariant

    d, ds, x = env
    p, S = d.ploidy, d.n_samples
    sp = ds.with_tracks(False).with_seqs("variants").with_settings(splice_info=ROWS)

    def expected(pairs, fields, dummy, fold=False, rc_neg=True, **kw):
        e_reg, e_s, n_el = _element_batch(ROWS, pairs)
        to_rc = (d.regions[e_reg, 3] == -1) if rc_neg else np.zeros(e_reg.size, bool)
        exp, off = _expected_variants(O, d, e_reg * S + e_s, to_rc, fields, dummy, x["ref"], x["af"], fold=fold,
                                      dosages=x["dz"], **kw)
        return (off, *_regroup(exp, off, _cell_rows(n_el, p, fold)))

    # default fields, paired pairs: elements without variants contribute nothing
    r_sel, s_sel = [0, 2, 3, 1, 4, 5, 3], [1, 0, 2, 2, 1, 0, 0]
    e_off, exp, off = expected(list(zip(r_sel, s_sel)), ("alt", "ilen", "start"), None)
    assert (np.diff(e_off) == 0).any() and (np.diff(e_off) > 3).any()
    _check_variants(sp[r_sel, s_sel], exp, off, (7, p, None))

    # every field + a dummy variant per element row, with and without the strand pass
    dummy = DummyVariant(start=-5, ilen=9, alt=b"AC", ref=b"G", dosage=0.5, info={"AF": 0.25})
    every = ("alt", "start", "ref", "ilen", "dosage", "AF")
    full = sp.with_settings(var_fields=list(every), dummy_variant=dummy)
    pairs = [(r, s) for r in range(len(ROWS)) for s in range(S)]
    for rc_neg in (True, False):
        e_off, exp, off = expected(pairs, every, dummy, rc_neg=rc_neg)
        assert (np.diff(e_off) >= 1).all()
        _check_variants(full.with_settings(rc_neg=rc_neg)[:, :], exp, off, (len(ROWS), S, p, None))

    # AF filter + unphased union + dummy: each element's union row (ploid 0, then ploid 1), element after element
    flt = sp.with_settings(min_af=0.2, max_af=0.9, unphased_union=True, dummy_variant=DummyVariant(),
                           var_fields=["alt", "ilen", "start", "dosage", "AF"])
    _, exp, off = expected(pairs, ("alt", "ilen", "start", "dosage", "AF"), DummyVariant(), fold=True, min_af=0.2, max_af=0.9)
    _check_variants(flt[:, :], exp, off, (len(ROWS), S, 1, None))


@pytest.mark.parametrize("alphabet,unk", [("ACGT", 4), ("ACGT", 300)])
def test_variant_windows_and_flank_tokens_vs_oracle(env, O, alphabet, unk):
    """Windows in window and allele modes (reference-oriented: no strand pass) and flank tokens next to reverse-complemented
    alleles, with tokens of two contigs; unk = 300 makes the tokens int32."""
    from genvarloader_b200 import DummyVariant, VarWindowOpt
    from genvarloader_b200._types import build_token_lut

    d, ds, x = env
    p, S = d.ploidy, d.n_samples
    rfa, rfo = x["ref"]
    lut, tok_dt = build_token_lut(alphabet, unk)
    r_sel, s_sel = [3, 0, 2, 5, 1, 4, 3], [0, 2, 1, 1, 0, 2, 1]
    e_reg, e_s, n_el = _element_batch(ROWS, list(zip(r_sel, s_sel)))
    goi = ((e_reg * S + e_s)[:, None] * p + np.arange(p)[None, :]).reshape(-1)
    v, off = O.gather_rows(goi, d.geno_offsets, d.geno_v_idxs)
    v_contigs = np.repeat(np.repeat(d.regions[e_reg, 0], p), np.diff(off)).astype(np.int32)
    assert set(v_contigs.tolist()) == {0, 1}
    tail = (lut, v_contigs, d.v_starts, d.ilens, d.reference, d.ref_offsets, N)
    cells = _cell_rows(n_el, p, False)
    L = 6
    dummy = DummyVariant(alt=b"NN", ref=b"N")
    base = ds.with_tracks(False).with_settings(splice_info=ROWS)
    for ref_kind, alt_kind in (("window", "window"), ("allele", "window"), ("window", "allele"), ("allele", "allele")):
        opt = VarWindowOpt(L, alphabet, unk, ref=ref_kind, alt=alt_kind)
        win = O.assemble_variant_buffers(1, v, off, d.alt_alleles, d.alt_offsets, rfa, rfo, False, False,
                                         1 if ref_kind == "window" else 2, 1 if alt_kind == "window" else 2, L, *tail)
        for dv in (None, dummy):
            got = base.with_seqs("variant-windows", opt).with_settings(dummy_variant=dv if dv is not None else False)[r_sel, s_sel]
            exp, e_off = {"ilen": d.ilens[v], "start": d.v_starts[v]}, off
            for name in ("ilen", "start"):
                if dv is not None:
                    exp[name], e_off = O.fill_empty_scalar(exp[name], off, dv.scalar_for(name, np.int32))
            for name, (data, so) in win.items():
                if dv is not None:
                    wl = len(dv.alt if name in ("alt", "alt_window") else dv.ref) + (2 * L if name.endswith("_window") else 0)
                    data, _, so = O.fill_empty_seq(data, off, so, np.full(wl, unk, tok_dt))
                exp[name] = (data, so)
            assert sorted(got.fields) == sorted(exp)
            exp, c_off = _regroup(exp, e_off, cells)
            _check_variants(got, exp, c_off, (7, p, None))
    # variants + flank tokens: alleles reverse-complemented per element strand, tokens reference-oriented
    got = base.with_seqs("variants").with_settings(token_alphabet=alphabet, unknown_token=unk, flank_length=L,
                                                    dummy_variant=dummy)[r_sel, s_sel]
    fl = O.assemble_variant_buffers(0, v, off, d.alt_alleles, d.alt_offsets, None, None, False, True, 0, 0, L, *tail)
    tok, e_off = O.fill_empty_fixed(fl["flank_tokens"][0], off, 2 * L, tok_dt.type(unk))
    a_data, a_vo, a_so = O.fill_empty_seq(fl["alt"][0], off, fl["alt"][1], np.frombuffer(b"NN", np.uint8))
    exp = {"alt": (O.rc_alleles(a_data, a_so, a_vo, np.repeat(d.regions[e_reg, 3] == -1, p)), a_so),
           "ilen": O.fill_empty_scalar(d.ilens[v], off, np.int32(0))[0],
           "start": O.fill_empty_scalar(d.v_starts[v], off, np.int32(-1))[0], "flank_tokens": tok.reshape(-1, 2 * L)}
    assert sorted(got.fields) == sorted(exp)
    exp, c_off = _regroup(exp, e_off, cells)
    _check_variants(got, exp, c_off, (7, p, None))


# ---------------------------------------------------------------------------------------------------- structure and shapes
def test_cells_are_the_concatenated_unspliced_reads(env):
    """Every spliced cell equals the concatenation of the unspliced ds[r_k, s] outputs, field by field."""
    from genvarloader_b200 import DummyVariant, VarWindowOpt

    d, ds, _ = env
    p, S = d.ploidy, d.n_samples
    base = ds.with_tracks(False)
    dummy = DummyVariant(start=-5, ilen=9, alt=b"AC", ref=b"G", dosage=0.5, info={"AF": 0.25})
    states = [base.with_seqs("variants").with_settings(var_fields=["alt", "start", "ref", "ilen", "dosage", "AF"],
                                                         dummy_variant=dummy),
              base.with_seqs("variants").with_settings(min_af=0.1, max_af=0.7, unphased_union=True, dummy_variant=DummyVariant()),
              base.with_seqs("variants").with_settings(token_alphabet="ACGT", unknown_token=4, flank_length=3),
              base.with_seqs("variant-windows", VarWindowOpt(4, "ACGT", 4, ref="allele")).with_settings(dummy_variant=dummy)]
    row_list = list(ROWS.values())
    for st in states:
        got = _rows(st.with_settings(splice_info=ROWS)[:, :])
        n_h = 1 if st.unphased_union else p
        cell = 0
        for r in range(len(row_list)):
            for s in range(S):
                parts = [_rows(st[int(e), s]) for e in row_list[r]]
                for h in range(n_h):
                    for name in got:
                        assert got[name][cell] == [v for u in parts for v in u[name][h]], (r, s, h, name)
                    cell += 1
        assert cell == len(got["start"])


def test_index_forms_and_output_shapes(env):
    d, ds, _ = env
    p, S = d.ploidy, d.n_samples
    base = ds.with_tracks(False).with_seqs("variants").with_settings(var_fields=["alt", "ref", "start"])
    sp = base.with_settings(splice_info=ROWS)
    # a one-element row equals the unspliced read of its region
    for r_row, region in ((1, 5), (5, 10)):
        for s in range(S):
            _same(sp[r_row, s], base[region, s])
    # int/int squeezes; slices and outer indexing keep (rows, samples); paired arrays give (pairs,)
    assert sp[2, 0].shape == (p, None)
    _same(sp[2, 0], sp[[2], [0]].squeeze(0))
    outer = sp[1:4, [0, 2]]
    assert outer.shape == (3, 2, p, None)
    paired = sp[[1, 2, 3], [2, 2, 2]]
    assert paired.shape == (3, p, None)
    ro, rp = _rows(outer), _rows(paired)
    for name in ro:
        for j in range(3):  # pair j of the paired call is cell (j, 1) of the outer call
            assert rp[name][j * p: (j + 1) * p] == ro[name][(2 * j + 1) * p: (2 * j + 2) * p]
    assert sp[:, 1].shape == (len(ROWS), 1, p, None)
    assert sp.with_settings(unphased_union=True)[1:4, :].shape == (3, S, 1, None)
    # "flat" and "variable" hand the RaggedVariants back unchanged
    for st in (sp.with_output_format("flat"), sp.with_len("variable"), sp.with_output_format("flat").with_len("variable")):
        _same(st[1:4, [0, 2]], outer)


def test_with_painted_tracks(env):
    """Variants with tracks active: (variants, tracks), the tracks painted over the element regions exactly as a tracks-only
    spliced read returns them (tracks are never realigned to a variants output)."""
    import torch

    d, ds, _ = env
    names = ["track1", "track0"]
    r_sel, s_sel = [0, 3, 2, 5], [2, 1, 0, 1]
    for realign in (True, False):
        sp = ds.with_tracks(names).with_settings(splice_info=ROWS, realign_tracks=realign)
        v, t = sp.with_seqs("variants")[r_sel, s_sel]
        t_only = sp.with_seqs(None)[r_sel, s_sel]
        assert t.shape == t_only.shape == (4, 2, None)
        assert (t.data.view(torch.int32) == t_only.data.view(torch.int32)).all() and (t.offsets == t_only.offsets).all()
        _same(v, sp.with_seqs("variants").with_tracks(False)[r_sel, s_sel])


def test_to_dataloader_yields_what_getitem_returns(env):
    d, ds, _ = env
    sp = ds.with_tracks(False).with_seqs("variants").with_settings(splice_info=ROWS, var_fields=["alt", "ilen", "start", "AF"])
    n = 0
    for k, v in enumerate(sp.to_dataloader(batch_size=4)):
        idx = np.arange(4 * k, min(4 * k + 4, len(sp)))
        _same(v, sp[idx // sp.n_samples, idx % sp.n_samples])
        n += len(idx)
    assert n == len(sp)


def test_library_calls_do_not_grow_with_the_batch(env, monkeypatch):
    from genvarloader_b200 import DummyVariant, VarWindowOpt, _engine

    d, ds, _ = env
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

    base = ds.with_tracks(False).with_settings(splice_info=ROWS)
    for st in (base.with_seqs("variants"),
               base.with_seqs("variants").with_settings(var_fields=["alt", "ref", "start", "dosage", "AF"], min_af=0.1,
                                                         unphased_union=True, dummy_variant=DummyVariant()),
               base.with_seqs("variant-windows", VarWindowOpt(8, "ACGT", 4))):
        a = count(st, ([1], [0]))
        b = count(st, (slice(None), slice(None)))
        assert a == b, (a, b)


# ---------------------------------------------------------------------------------------------------- counts
def test_counts_sum_over_the_elements(env):
    d, ds, _ = env
    p, S = d.ploidy, d.n_samples
    sp = ds.with_settings(splice_info=ROWS)
    go = d.geno_offsets
    row_list = list(ROWS.values())
    exp_v = np.zeros((len(ROWS), S, p), np.int32)
    exp_i = np.zeros((len(ROWS), S, 2), np.int32)
    for r, els in enumerate(row_list):
        for s in range(S):
            for e in els:
                slot = (e * S + s) * p + np.arange(p)
                exp_v[r, s] += (go[1, slot] - go[0, slot]).astype(np.int32)
                for ti, name in enumerate(("track0", "track1")):
                    io = d.tracks[name][3]
                    exp_i[r, s, ti] += io[e * S + s + 1] - io[e * S + s]
    eq("n_variants", 0, sp.n_variants(), exp_v)
    eq("n_intervals", 0, sp.n_intervals(), exp_i)
    # the cell lengths of the variants output without AF filter and dummy
    lens = sp.with_tracks(False).with_seqs("variants")[:, :].lengths.cpu().numpy()
    assert (lens == exp_v).all()
    # the index forms and shapes of ds[...]
    eq("n_variants[2, 1]", 0, sp.n_variants(2, 1), exp_v[2, 1])
    eq("n_variants paired", 0, sp.n_variants([0, 3], [1, 1]), exp_v[[0, 3], [1, 1]])
    eq("n_variants outer", 0, sp.n_variants(slice(1, 4), [0, 2]), exp_v[1:4][:, [0, 2]])
    eq("n_intervals", 1, sp.with_tracks(["track1"]).n_intervals(slice(1, 3)), exp_i[1:3, :, 1:])
    eq("n_intervals", 2, sp.with_tracks(False).n_intervals(4, 0), np.zeros(0, np.int32))


# ---------------------------------------------------------------------------------------------------- opened datasets
def test_opened_dataset_with_bed_column_splice_rows(O, cuda_device, tmp_path):
    """Splice rows from input-BED columns of an opened dataset whose variant table carries REF strings and a 4-byte INFO
    column (AF: a field and the filter's column); its annotation track counts slot r_k of every element."""
    import pyarrow as pa
    import pyarrow.ipc as ipc

    from genvarloader_b200 import Dataset, DummyVariant, synth
    from tests._gvl_disk import write_fasta, write_gvl_dataset

    d = synth.make_dataset(43, 150_000, 3, 10, 1500, 6.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=1, max_indel=9)
    d.tracks["annot"] = synth.make_track(np.random.default_rng(5), d.regions, 1)
    rows = {"tA": [3, 0, 7], "tB": [5], "tC": [9, 8, 2]}
    write_gvl_dataset(tmp_path / "ds", d, ["chr1"], ["a", "b", "c"], np.arange(d.n_regions), annot_tracks=("annot",))
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
    rng = np.random.default_rng(6)
    rfa, rfo = _ref_alleles(rng, d.ilens)
    af = rng.random(d.v_starts.size).astype(np.float32)
    vpath = tmp_path / "ds" / "genotypes" / "variants.arrow"
    with pa.memory_map(str(vpath), "r") as src:
        vt = ipc.open_file(src).read_all()
    refs = [rfa[rfo[i]: rfo[i + 1]].tobytes().decode() for i in range(d.v_starts.size)]
    vt = vt.drop_columns(["AF"]).append_column("REF", pa.array(refs)).append_column("AF", pa.array(af))
    with pa.OSFile(str(tmp_path / "vt.new"), "wb") as f, ipc.new_file(f, vt.schema) as w:
        w.write_table(vt)
    del vt
    (tmp_path / "vt.new").replace(vpath)
    write_fasta(tmp_path / "ref.fa", d.reference, d.ref_offsets, ["chr1"])
    dsk = Dataset.open(tmp_path / "ds", tmp_path / "ref.fa", device=cuda_device)
    assert {"ref", "AF"} <= set(dsk.available_var_fields)
    fields = ("alt", "ref", "start", "ilen", "AF")
    dummy = DummyVariant(ref=b"T", info={"AF": 0.5})
    sp = dsk.with_tracks(False).with_seqs("variants").with_settings(splice_info=("transcript", "exon"), var_fields=list(fields),
                                                                     dummy_variant=dummy, min_af=0.15)
    names = list(sp.splice_names)
    p = d.ploidy
    for row in rows:
        for s in range(3):
            e_reg = np.array(rows[row], np.int64)
            exp, off = _expected_variants(O, d, e_reg * d.n_samples + s, d.regions[e_reg, 3] == -1, fields, dummy, (rfa, rfo), af,
                                          min_af=0.15)
            exp, c_off = _regroup(exp, off, _cell_rows([e_reg.size], p, False))
            _check_variants(sp[names.index(row), s], exp, c_off, (p, None))
    # counts: the annotation track reads slot r_k, the sample track slot (r_k, s)
    spt = dsk.with_tracks(["annot", "track0"]).with_settings(splice_info=("transcript", "exon"))
    got = spt.n_intervals()
    for row in rows:
        for s in range(3):
            e_reg = np.array(rows[row], np.int64)
            ia, it = d.tracks["annot"][3], d.tracks["track0"][3]
            want = [int((ia[e_reg + 1] - ia[e_reg]).sum()), int((it[e_reg * 3 + s + 1] - it[e_reg * 3 + s]).sum())]
            assert got[names.index(row), s].tolist() == want
