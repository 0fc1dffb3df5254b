"""Every launch configuration of the haplotype execute, pinned bit for bit to the oracle.

`gvl_dev_hap_exec` picks the packed one-hot kernel's instantiation and tile length at launch time from the output length,
the rows of the call, the plan's record bound per row and the SM count; the plans pick 32, 256 or 512 threads per row and
static or dynamic record slices.  A tile-boundary or staging bug in one configuration only shows where that configuration
runs, so each case here:

  * computes its shape from the device's SM count and the tuning constants of gvl_common.cuh / gvl_hap_oh.cuh (parsed from
    the sources), through `_packed_choice`, a restatement of the selection in gvl_hap.cu;
  * asserts through gvl_debug_last_launch that the library reached the configuration the case targets, so a retune makes
    the case fail loudly instead of quietly testing something else;
  * compares every output byte with the oracle.

The variant tables come from `boundary_dataset`: clusters of records at every multiple of DIR_Q output positions (every
tile and directory boundary is one), net-zero in length so that output and reference coordinates stay aligned between
clusters, with some rows drifting.  The last part runs the fixed-length job and its rings at the benchmark's shapes."""
from __future__ import annotations

import dataclasses
import re
from pathlib import Path

import numpy as np
import pytest

from tests import _golden

pytestmark = pytest.mark.gpu

N = ord("N")
_CSRC = Path(__file__).resolve().parent.parent / "genvarloader_b200" / "csrc"


def _constants() -> dict:
    text = (_CSRC / "gvl_common.cuh").read_text() + (_CSRC / "gvl_hap_oh.cuh").read_text() + (_CSRC / "gvl_hap.cu").read_text()
    c = {m.group(1): int(m.group(2)) for m in re.finditer(r"constexpr int (\w+) = (-?\d+);", text)}
    c["EXEC_UNIT"] = c["EXEC_THREADS"] * 4  # (gvl_common.cuh: 4 positions per thread)
    # OH_MAX_TILE as gvl_hap_oh.cuh derives it: the wanted length, unless the group table (one thread per group) caps it
    cap = (c["OH_THREADS"] - 2) * c["OH_GROUP"]
    c["OH_MAX_TILE"] = c["OH_MAX_TILE_WANTED"] if c["OH_MAX_TILE_WANTED"] < cap else cap // 1024 * 1024
    return c


C_ = _constants()
DIR_Q, REC_CAP, OH_MAX_TILE = C_["DIR_Q"], C_["REC_CAP"], C_["OH_MAX_TILE"]


def _sms() -> int:
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def _plan_width(max_records: int, n_work: int) -> int:
    """gvl_hap.cu plan_width."""
    if max_records <= 40 * n_work:
        return 32
    return 256 if max_records <= 4096 * n_work else 512


def _packed_choice(L: int, n_work: int, rb: int, sms: int):
    """(kernel, tile_len, tiles_per_row) of the packed one-hot execute for a fixed-length plan: gvl_dev_hap_exec."""
    q = max((C_["OH_THREADS"] // 32) * C_["OH_GROUP"], DIR_Q)
    tl = L * n_work // (3 * sms)
    sparse = rb > 0 and rb * OH_MAX_TILE <= 100 * L
    if tl > 16384 and not sparse:
        tl = 16384
    if tl > 8192 and L > 0 and rb * 16384 > REC_CAP * L:
        tl = 8192
    tl = max(q, min(tl // q * q, OH_MAX_TILE))
    tiles = -(-L // tl)
    gpw = (min(tl, L) // C_["OH_GROUP"]) // (C_["OH_THREADS"] // 32)
    if min(tl, L) <= 8192 and tiles == 1:
        kind = "packed_2warp"
    elif sparse and gpw >= 8:
        kind = "packed_unroll4"
    else:
        kind = "packed_unroll2"
    return kind, tl, tiles


def _launch(handle) -> dict:
    from genvarloader_b200 import _ffi

    return _ffi.last_launch(handle)


# ---------------------------------------------------------------------------------------------------------------------
# variant tables with records where the execute kernels split work
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Pattern:
    every: int = 1          # a cluster at every `every`-th multiple of DIR_Q output positions
    fill: int = 0           # plus one SNP every `fill` positions between clusters (0: none)
    far: int = 0            # plus SNPs outside the window: they count in the record bound, never in a tile
    drift: float = 0.15     # probability that a cluster is not net-zero in length
    mnp: bool = True        # multi-base substitutions (ALT of 4 bases over 4 reference bases)
    unsorted: bool = False  # the slot's list is not in position order (the plans' serial fallback)


def _slot(rng, s0: int, L: int, rc: bool, C: int, pat: Pattern):
    """(pos, alt_len, ilen) records of one slot and the haplotype position of each, in list order."""
    recs, hpos = [], []
    st = {"g": 0, "nxt": 1}  # output positions gained so far; first reference position free for the next record

    def add(h, alt_len, ilen):
        pos = s0 + h - st["g"]
        used = 1 - min(ilen, 0)
        if h < 0 or h >= L or pos < st["nxt"] or pos + used >= C - 2:
            return
        recs.append((pos, alt_len, ilen))
        hpos.append(h)
        st["g"] += alt_len - used
        st["nxt"] = pos + used

    def cur_h():
        return st["nxt"] - s0 + st["g"]

    step = DIR_Q * pat.every
    cs = sorted((L - B) if rc else B for B in range(step, L + 1, step))
    cs = [c for c in cs if 8 <= c <= L - 8]
    for c in cs + [None]:
        if pat.fill:
            stop = (c - 12) if c is not None else L - 1
            for h in range(max(cur_h(), 0) + 3, stop, pat.fill):
                add(h, 1, 0)
        if c is None:
            break
        k = int(rng.integers(3, 13))
        t = int(rng.integers(0, 4 if pat.mnp else 3))
        if t == 0:  # SNPs at boundary - 1 and at the boundary, two records inside one 8-position unit, then +k / -k
            add(c - 1, 1, 0)
            add(c, 1, 0)
            u = (c + 16) // 8 * 8
            add(u + 1, 1, 0)
            add(u + 4, 1, -2)
            add(c + 30, 1 + k, k)
            add(c + 31 + k + 20, 1, -k)
        elif t == 1:  # an insertion whose ALT crosses the boundary, then the deletion that restores the alignment
            add(c - 2, 1 + k, k)
            add(c + k + 25, 1, -k)
        elif t == 2:  # a deletion spanning the boundary, a SNP right after it, the restoring insertion
            add(c - 3, 1, -k)
            add(c, 1, 0)
            add(c + 25, 1 + k, k)
        else:  # a multi-base substitution over the boundary and two SNPs in the next unit
            add(c - 2, 4, -3)
            add(c + 3, 1, 0)
            add(c + 5, 1, 0)
        if rng.random() < pat.drift:  # not net-zero: the offsets drift from here on
            kd = int(rng.integers(1, 10))
            add(c + 95, 1 + kd, kd) if rng.random() < 0.5 else add(c + 95, 1, -kd)
    if pat.far:
        after = s0 + L + 3000
        if after + 3 * pat.far < C - 2:
            far = [(after + 3 * i, 1, 0) for i in range(pat.far)]
            recs, hpos = recs + far, hpos + [L + 3000] * pat.far
        elif s0 - 3000 - 3 * pat.far > 0:
            far = [(s0 - 3000 - 3 * (pat.far - i), 1, 0) for i in range(pat.far)]
            recs, hpos = far + recs, [-1] * pat.far + hpos
    return recs, hpos


def boundary_dataset(seed: int, L: int, n_regions: int, n_samples: int, pattern, contig_len: int | None = None,
                     rc_frac: float = 0.5, ends: bool = True, n_tracks: int = 0):
    """A `synth.SynthData` (ploidy 2, one contig) whose every (region, sample, ploid) slot follows `pattern(r, s, p)`.
    `ends`: the first window hangs over the contig's start, the last over its end.  Returns (data, haplotype positions
    of every slot's records, in list order)."""
    from genvarloader_b200 import synth

    rng = np.random.default_rng(seed)
    C = contig_len or (3 * L + 60_000)
    ref, ref_off = synth.make_reference(rng, [C])
    starts = np.sort(rng.integers(0, max(C - L, 1), n_regions)).astype(np.int64)
    if ends and n_regions >= 3:
        starts[0] = -37
        starts[-1] = C - L + 53
    strand = np.where(rng.random(n_regions) < rc_frac, -1, 1)
    regions = np.stack([np.zeros(n_regions, np.int64), starts, starts + L, strand], 1).astype(np.int32)
    slots, hpos = [], []
    for r in range(n_regions):
        for s in range(n_samples):
            for p in range(2):
                recs, h = _slot(rng, int(starts[r]), L, bool(strand[r] == -1), C, pattern(r, s, p))
                slots.append(recs)
                hpos.append(np.array(h, np.int64))
    pos = np.array([x[0] for sl in slots for x in sl], np.int64)
    alen = np.array([x[1] for sl in slots for x in sl], np.int64)
    ilen = np.array([x[2] for sl in slots for x in sl], np.int32)
    order = np.argsort(pos, kind="stable")
    new_idx = np.empty(order.size, np.int64)
    new_idx[order] = np.arange(order.size)
    alt_off = np.concatenate([[0], np.cumsum(alen[order])]).astype(np.int64)
    alt = synth.ACGT[rng.integers(0, 4, int(alt_off[-1]), dtype=np.uint8)]
    anchor = (ilen[order] != 0) | (alen[order] == 1)  # indels and SNP-free anchors start with the reference base
    alt[alt_off[:-1][anchor]] = ref[pos[order][anchor]]
    snp = (alen[order] == 1) & (ilen[order] == 0)
    alt[alt_off[:-1][snp]] = synth.ACGT[(np.searchsorted(synth.ACGT, ref[pos[order][snp]]) + 1) % 4]  # a real change
    lists, lens, k = [], [], 0
    for si, sl in enumerate(slots):
        idx = new_idx[k:k + len(sl)]
        k += len(sl)
        pat = pattern(si // (2 * n_samples), (si // 2) % n_samples, si % 2)
        if pat.unsorted and idx.size >= 6:  # swap neighbours in the middle third
            a, b = idx.size // 3, 2 * idx.size // 3
            mid = idx[a:b].copy()
            mid[: mid.size // 2 * 2] = mid[: mid.size // 2 * 2].reshape(-1, 2)[:, ::-1].ravel()
            idx = np.concatenate([idx[:a], mid, idx[b:]])
            hpos[si] = np.concatenate([hpos[si][:a], hpos[si][a:b][: mid.size // 2 * 2].reshape(-1, 2)[:, ::-1].ravel(),
                                       hpos[si][a + mid.size // 2 * 2:]])
        lists.append(idx)
        lens.append(idx.size)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    gv = np.concatenate(lists).astype(np.int32) if lists else np.empty(0, np.int32)
    d = synth.SynthData(ref, ref_off, pos[order].astype(np.int32), ilen[order], alt, alt_off, gv,
                        np.ascontiguousarray(np.stack([off[:-1], off[1:]])), regions, n_samples, 2, 0)
    for t in range(n_tracks):
        d.tracks[f"track{t}"] = synth.make_track(rng, regions, n_samples, 0)
    return d, hpos


def _max_per_tile(hpos, L: int, tl: int) -> int:
    """Most records of one row inside one tile of `tl` output positions (haplotype positions of forward and reverse
    rows alike: a reverse row's tiles are the same intervals counted from the other end)."""
    best = 0
    for h in hpos:
        h = h[(h >= 0) & (h < L)]
        if h.size:
            best = max(best, int(np.bincount(h // tl).max()), int(np.bincount((L - 1 - h) // tl).max()))
    return best


def _all_pairs(d):
    r = np.repeat(np.arange(d.n_regions), d.n_samples)
    s = np.tile(np.arange(d.n_samples), d.n_regions)
    return r, s


# ---------------------------------------------------------------------------------------------------------------------
# fixtures
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def K(cuda_device):
    from genvarloader_b200 import _kernels

    return _kernels


@pytest.fixture(scope="module")
def O():
    from oracle import oracle

    return oracle


def _host_args(d, regions, shifts, goi, pad, L):
    return (regions, shifts, goi, d.geno_offsets, d.geno_v_idxs, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
            d.reference, d.ref_offsets, pad, L)


def _rows_mean(d, goi) -> int:
    g = goi.ravel()
    return int((d.geno_offsets[1, g] - d.geno_offsets[0, g]).clip(min=0).sum()) // g.size


# ---------------------------------------------------------------------------------------------------------------------
# 1. packed one-hot, fixed length and ragged, through the host layer (record bound = the rows' list lengths)
# ---------------------------------------------------------------------------------------------------------------------
def _sparse(every):
    return lambda r, s, p: Pattern(every=every)


# name: (target kernel, target tile (None: from the shape), L, rows wanted as a function of the SM count, pattern maker)
def _packed_cases():
    def p_2warp(r, s, p):  # every 4th row dense: one tile holds several hundred records
        return Pattern(fill=9) if (r + s + p) % 4 == 0 else Pattern(every=1)

    def p_u4_long(r, s, p):  # 1 row in 8 dense (multi-pass staging at 31,744); the others only at tile boundaries
        return Pattern(fill=70) if (2 * r + p) % 8 == 0 else Pattern(every=31, drift=0.5)

    def p_u4_mid(r, s, p):
        return Pattern(every=1, drift=0.3) if p == 0 else Pattern(every=3)

    def p_dense_bound(r, s, p):  # dense bound (far variants) and one dense row in four
        return Pattern(fill=25, far=300) if (r + p) % 4 == 0 else Pattern(every=1, far=420)

    def p_loose(r, s, p):  # bound between "sparse" and "dense", rows themselves sparse
        return Pattern(every=1, far=300, drift=0.3)

    def p_min(r, s, p):
        return Pattern(every=1, fill=40 if p else 0, drift=0.4)

    return {
        # a 2-warp CTA per row: rows of <= 8,192 positions, enough rows for 3 CTAs per SM
        "2warp": ("packed_2warp", None, 6997, lambda sms: 8192 * 3 * sms // 6997 + 2, p_2warp),
        "unroll4_31744": ("packed_unroll4", OH_MAX_TILE, 100_003, lambda sms: OH_MAX_TILE * 3 * sms // 100_003 + 2, p_u4_long),
        "unroll4_12288": ("packed_unroll4", 12288, 50_001, lambda sms: 12800 * 3 * sms // 50_001, p_u4_mid),
        "unroll2_8192_dense": ("packed_unroll2", 8192, 40_003, lambda sms: 12000 * 3 * sms // 40_003, p_dense_bound),
        "unroll2_16384_loose": ("packed_unroll2", 16384, 120_001, lambda sms: 20000 * 3 * sms // 120_001, p_loose),
        "unroll2_1024_min": ("packed_unroll2", 1024, 5003, lambda sms: 8, p_min),
    }


_PACKED = _packed_cases()
# cases whose densest tile must need more than one staging pass (REC_CAP records)
_MULTI_PASS = {"2warp", "unroll4_31744", "unroll2_8192_dense"}


def _packed_data(name, sms):
    target, tl_target, L, rows_of, pat = _PACKED[name]
    n_q = -(-rows_of(sms) // 2)
    n_s = 4
    n_r = -(-n_q // n_s)
    d, hpos = boundary_dataset(sum(name.encode()), L, n_r, n_s, pat)
    r, s = _all_pairs(d)
    return d, hpos, r[:n_q], s[:n_q], L, target, tl_target


@pytest.mark.parametrize("name", list(_PACKED))
def test_packed_fixed_configurations(K, O, name):
    from genvarloader_b200 import synth

    sms = _sms()
    d, hpos, r, s, L, target, tl_target = _packed_data(name, sms)
    regions, goi, to_rc, _ = synth.batch_args(d, r, s)
    rb = _rows_mean(d, goi)
    kind, tl, tiles = _packed_choice(L, goi.size, rb, sms)
    assert kind == target and (tl_target is None or tl == tl_target), f"{name}: shape reaches {kind} at {tl}"
    if name in _MULTI_PASS:
        assert _max_per_tile(hpos, L, tl) > REC_CAP, f"{name}: no tile needs a second staging pass"
    sh = np.zeros(goi.shape, np.int32)
    pad = ord("A") if name.endswith("dense") else N  # a pad byte that is a base: complemented in reverse rows
    args = _host_args(d, regions, sh, goi, pad, L)
    e_out, _ = O.reconstruct_haplotypes_fused(*args, None, None, to_rc, parallel=True)
    exp = O.onehot(e_out, parallel=True)
    K.pin_static(d.reference, d.alt_alleles)
    try:
        got, _ = K.reconstruct_haplotypes_fused(*args, None, None, to_rc, mode="onehot")
        cfg = _launch(K.default_ctx().handle)
    finally:
        K.unpin_static(d.reference, d.alt_alleles)
    assert (cfg["exec_kernel"], cfg["tile_len"], cfg["tiles_per_row"], cfg["rec_bound"]) == (kind, tl, tiles, rb), cfg
    bad = np.flatnonzero((got != exp).any(1))
    _golden.eq(f"{name}[{cfg}] first bad row {bad[0] // L if bad.size else -1}", 0, got, exp)


def test_packed_ragged_configuration(K, O):
    """ragged rows: unroll-4 over the fixed ragged tile, multi-pass tiles, RC rows, both contig ends."""
    from genvarloader_b200 import synth

    L = 21_003
    d, hpos = boundary_dataset(5, L, 5, 4, lambda r, s, p: Pattern(fill=14) if p else Pattern(every=1, drift=0.5))
    r, s = _all_pairs(d)
    regions, goi, to_rc, _ = synth.batch_args(d, r, s)
    assert _max_per_tile(hpos, L, C_["TILE"]) > REC_CAP
    args = _host_args(d, regions, np.zeros(goi.shape, np.int32), goi, ord("G"), -1)
    e_out, e_oo = O.reconstruct_haplotypes_fused(*args, None, None, to_rc, parallel=True)
    K.pin_static(d.reference, d.alt_alleles)
    try:
        got, g_oo = K.reconstruct_haplotypes_fused(*args, None, None, to_rc, mode="onehot")
        cfg = _launch(K.default_ctx().handle)
    finally:
        K.unpin_static(d.reference, d.alt_alleles)
    assert (cfg["exec_kernel"], cfg["tile_len"], cfg["tiles_per_row"]) == ("packed_unroll4", C_["TILE"], 0), cfg
    _golden.eq("ragged.offsets", 0, g_oo, e_oo)
    _golden.eq(f"ragged.onehot[{cfg}]", 0, got, O.onehot(e_out, parallel=True))


# ---------------------------------------------------------------------------------------------------------------------
# 2. byte, annotated and channels-first kernels across the tile range, and rows beyond COUNT_MAX records
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["few_rows", "many_rows", "count_max"])
def test_byte_kernels(K, O, case):
    from genvarloader_b200 import synth

    sms = _sms()
    unit, max_units = C_["EXEC_UNIT"], C_["EXEC_MAX_UNITS"]
    if case == "few_rows":  # many tiles per row wanted: the shortest tile (4 units)
        L, n_r, n_s, pat = 20_004, 2, 1, lambda r, s, p: Pattern(every=1, drift=0.4)
        want = 4 * unit
    elif case == "many_rows":  # at least one row per resident CTA: the longest tile
        L, n_r, n_s, pat = 8196, -(-16 * sms // 8), 4, lambda r, s, p: Pattern(every=1, fill=60 if r % 5 == 0 else 0)
        want = max_units * unit
    else:  # rows with more than COUNT_MAX records: the 32-ary tile search
        L, n_r, n_s, pat = 30_004, 3, 2, lambda r, s, p: Pattern(fill=9, drift=0.3) if p == 0 else Pattern(every=1)
        want = None
    d, hpos = boundary_dataset(17 + len(case), L, n_r, n_s, pat)
    r, s = _all_pairs(d)
    regions, goi, to_rc, _ = synth.batch_args(d, r, s)
    if case == "count_max":
        assert max(int((h < L).sum()) for h in hpos) > C_["COUNT_MAX"]
    h = K.default_ctx().handle
    for out_len in ([L, -1] if case == "count_max" else [L]):
        args = _host_args(d, regions, np.zeros(goi.shape, np.int32), goi, N, out_len)
        e_out, e_oo = O.reconstruct_haplotypes_fused(*args, None, None, to_rc, parallel=True)
        g_out, g_oo = K.reconstruct_haplotypes_fused(*args, None, None, to_rc)
        cfg = _launch(h)
        assert cfg["exec_kernel"] == "bytes", cfg
        if out_len >= 0:
            assert unit * 4 <= cfg["tile_len"] <= unit * max_units and cfg["tiles_per_row"] == -(-L // cfg["tile_len"]), cfg
            if want is not None:
                assert cfg["tile_len"] == want, cfg
        tag = f"{case}[{out_len}][{cfg}]"
        _golden.eq(tag + ".offsets", 0, g_oo, e_oo)
        _golden.eq(tag + ".u8", 0, g_out, e_out)
        e = O.reconstruct_annotated_haplotypes_fused(*args, None, None, to_rc, parallel=True)
        g = K.reconstruct_annotated_haplotypes_fused(*args, None, None, to_rc)
        assert _launch(h)["exec_kernel"] == "bytes"
        for j, nm in enumerate(["out", "annot_v", "annot_pos", "offsets"]):
            _golden.eq(f"{tag}.annot.{nm}", 0, g[j], e[j])
        oh, _ = K.reconstruct_haplotypes_fused(*args, None, None, to_rc, mode="onehot")  # reference not pinned: bytes kernel
        assert _launch(h)["exec_kernel"] == "bytes"
        exp_oh = O.onehot(e_out, parallel=True)
        _golden.eq(tag + ".onehot", 0, oh, exp_oh)
        if out_len >= 0:
            cf, _ = K.reconstruct_haplotypes_fused(*args, None, None, to_rc, mode="onehot_cf")
            assert _launch(h)["exec_kernel"] == "bytes"
            _golden.eq(tag + ".onehot_cf", 0, cf, exp_oh.reshape(goi.size, L, 4).transpose(0, 2, 1))


# ---------------------------------------------------------------------------------------------------------------------
# 3. plan widths: dynamic record slices (host layer: keep mask, shifts, unsorted lists; the track plan too)
# ---------------------------------------------------------------------------------------------------------------------
def _width_pattern(nt):
    if nt == 32:
        return lambda r, s, p: Pattern(every=4, unsorted=(r + s) % 3 == 0, drift=0.4)
    if nt == 256:
        return lambda r, s, p: Pattern(every=1, fill=120, unsorted=(r + s) % 3 == 0)
    return lambda r, s, p: Pattern(every=1, fill=60, far=4200, unsorted=(r + s) % 3 == 0)


@pytest.mark.parametrize("nt", [32, 256, 512])
def test_plan_widths_host_layer(K, O, nt):
    from genvarloader_b200 import synth

    L = 16_005
    d, _ = boundary_dataset(40 + nt, L, 4, 3, _width_pattern(nt), n_tracks=1)
    r, s = _all_pairs(d)
    regions, goi, to_rc, ds_idx = synth.batch_args(d, r, s)
    rows = goi.size
    g = goi.ravel()
    n_var = (d.geno_offsets[1, g] - d.geno_offsets[0, g]).clip(min=0)
    assert _plan_width(int(n_var.sum()), rows) == nt
    rng = np.random.default_rng(nt)
    keep_off = np.concatenate([[0], np.cumsum(n_var)]).astype(np.int64)
    keep = rng.random(int(keep_off[-1])) < 0.8
    # shifts that walk over several variants (the densest rows have one every ~60 positions)
    sh = rng.integers(0, 400, goi.shape).astype(np.int32)
    h = K.default_ctx().handle
    for out_len in (L, -1):
        shifts = sh if out_len >= 0 else np.zeros_like(sh)
        args = _host_args(d, regions, shifts, goi, N, out_len)
        for kp, ko in ((None, None), (keep, keep_off)):
            e_out, e_oo = O.reconstruct_haplotypes_fused(*args, kp, ko, to_rc, parallel=True)
            g_out, g_oo = K.reconstruct_haplotypes_fused(*args, kp, ko, to_rc)
            cfg = _launch(h)
            assert (cfg["plan_threads"], cfg["plan_static"]) == (nt, 0), cfg
            tag = f"width{nt}[{out_len}][keep={kp is not None}]"
            _golden.eq(tag + ".offsets", 0, g_oo, e_oo)
            _golden.eq(tag + ".u8", 0, g_out, e_out)
    # the track plan: the same kernel in track mode
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2], d.v_starts)
    lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)
    out_offsets = (np.arange(rows + 1) * L).astype(np.int64)
    track_offsets = np.concatenate([[0], np.cumsum(lengths - diffs.clip(max=0).min(1))]).astype(np.int64)
    st, en, va, io = d.tracks["track0"]
    for kp, ko in ((None, None), (keep, keep_off)):
        a = (out_offsets, regions, sh, goi, d.geno_v_idxs, d.geno_offsets, d.v_starts, d.ilens, ds_idx, st, en, va, io,
             track_offsets, np.array([1.0], np.float64), 4, 99, kp, ko, to_rc)
        exp = np.zeros(int(out_offsets[-1]), np.float32)
        O.intervals_and_realign_track_fused(exp, *a)
        got = np.full(int(out_offsets[-1]), 7.0, np.float32)
        K.intervals_and_realign_track_fused(got, *a)
        cfg = _launch(h)
        assert (cfg["trk_plan_threads"], cfg["trk_plan_static"]) == (nt, 0), cfg
        _golden.eq(f"width{nt}.track[keep={kp is not None}]", 0, got, exp)


# ---------------------------------------------------------------------------------------------------------------------
# 4. plan widths with static record slices: the fixed-length job of a Dataset (longest slot bounds every row)
# ---------------------------------------------------------------------------------------------------------------------
def _track_oracle(O, d, regions, goi, to_rc, ds_idx, L, names_params):
    """Realigned tracks of fixed-length rows as the Dataset writes them, one array (rows * L) per track."""
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2], d.v_starts)
    lengths = (regions[:, 2] - regions[:, 1]).astype(np.int64)
    out_offsets = (np.arange(goi.size + 1) * L).astype(np.int64)
    track_offsets = np.concatenate([[0], np.cumsum(lengths - diffs.clip(max=0).min(1))]).astype(np.int64)
    res = []
    for name, strategy, param in names_params:
        s, e, v, io = d.tracks[name]
        exp = np.zeros(int(out_offsets[-1]), np.float32)
        O.intervals_and_realign_track_fused(exp, out_offsets, regions, np.zeros(goi.shape, np.int32), goi, d.geno_v_idxs,
                                            d.geno_offsets, d.v_starts, d.ilens, ds_idx, s, e, v, io, track_offsets,
                                            np.array([param], np.float64), strategy, 0, None, None, to_rc)
        res.append(exp)
    return res


@pytest.mark.parametrize("nt", [32, 256, 512])
def test_plan_widths_fixed_job(cuda_device, O, nt):
    import torch

    from genvarloader_b200 import Interpolate, Repeat5p, synth
    from genvarloader_b200._dataset import Dataset

    L = 16_005 if nt != 512 else 40_003
    if nt == 512:  # one slot longer than 4,096 variants
        pat = lambda r, s, p: Pattern(fill=8, unsorted=True) if (r, s, p) == (1, 1, 0) else Pattern(every=1, unsorted=s == 2)
    else:
        pat = _width_pattern(nt)
    d, _ = boundary_dataset(60 + nt, L, 4, 3, pat, n_tracks=2)
    max_slot = int((d.geno_offsets[1] - d.geno_offsets[0]).max())
    assert _plan_width(max_slot, 1) == nt
    ds = Dataset.from_synth(cuda_device, d, rng=1).with_len(L).with_insertion_fill({"track0": Repeat5p(), "track1": Interpolate(1)})
    r, s = _all_pairs(d)
    regions, goi, to_rc, ds_idx = synth.batch_args(d, r, s)
    seq, trk = ds[r, s]
    torch.cuda.synchronize()
    cfg = _launch(ds.engine.ctx.handle)
    assert (cfg["plan_threads"], cfg["plan_static"], cfg["trk_plan_threads"], cfg["trk_plan_static"]) == (nt, 1, nt, 1), cfg
    assert cfg["rec_bound"] == max_slot, cfg
    e_out, _ = O.reconstruct_haplotypes_fused(*_host_args(d, regions, np.zeros(goi.shape, np.int32), goi, N, L), None, None,
                                              to_rc, parallel=True)
    _golden.eq(f"job{nt}.u8[{cfg}]", 0, seq.cpu().numpy().ravel(), e_out)
    exp_t = _track_oracle(O, d, regions, goi, to_rc, ds_idx, L, [("track0", 0, 0.0), ("track1", 4, 1.0)])
    got_t = trk.cpu().numpy()  # (b, t, p, L)
    for ti in range(2):
        _golden.eq(f"job{nt}.track{ti}", 0, np.ascontiguousarray(got_t[:, ti]).ravel(), exp_t[ti])
    # one-hot through the packed kernel under the static-slice bound
    oh = ds.with_tracks(False).with_encoding("onehot")[r, s]
    torch.cuda.synchronize()
    cfg = _launch(ds.engine.ctx.handle)
    assert cfg["exec_kernel"] != "bytes" and cfg["plan_static"] == 1, cfg
    _golden.eq(f"job{nt}.onehot[{cfg}]", 0, oh.cpu().numpy().reshape(-1, 4), O.onehot(e_out, parallel=True))


# ---------------------------------------------------------------------------------------------------------------------
# 5. the svar2 source under the typical-slot-length hint: long tiles chosen for rows that are in fact dense
# ---------------------------------------------------------------------------------------------------------------------
def test_svar2_hint_long_tiles_dense_rows(cuda_device, O):
    import torch

    from genvarloader_b200 import synth
    from genvarloader_b200._dataset import Dataset
    from tests.test_gpu_svar2_dataset import _oracle_haps

    sms = _sms()
    L = 100_003
    n_r, n_s = 32, 8
    dense = {(3, 1), (11, 5), (20, 0)}  # (region, sample) pairs whose haplotypes carry ~one variant every 20 bp
    pat = lambda r, s, p: Pattern(fill=20, mnp=False, drift=0.0) if (r, s) in dense else Pattern(every=31, mnp=False, drift=0.0)
    d, hpos = boundary_dataset(77, L, n_r, n_s, pat, rc_frac=0.5)
    sv = synth.to_svar2_dataset(d, dense_frac=0.5, seed=2)
    ds = Dataset.from_synth(cuda_device, d, rng=3, svar2=sv).with_tracks(False).with_len(L).with_encoding("onehot")
    n_q = -(-OH_MAX_TILE * 3 * sms // L // 2) + 2
    rng = np.random.default_rng(1)
    r = rng.integers(0, n_r, n_q)
    s = rng.integers(0, n_s, n_q)
    r[:3], s[:3] = zip(*sorted(dense))
    out = ds[r, s]
    torch.cuda.synchronize()
    cfg = _launch(ds.engine.ctx.handle)
    eng = ds.engine
    assert 0 < eng.typ_slot_len < eng.max_slot_len
    assert cfg["rec_bound"] == eng.typ_slot_len and cfg["plan_static"] == 1, cfg  # the clamp decided
    kind, tl, tiles = _packed_choice(L, 2 * n_q, eng.typ_slot_len, sms)
    assert (kind, tl) == ("packed_unroll4", OH_MAX_TILE), (kind, tl)
    assert (cfg["exec_kernel"], cfg["tile_len"], cfg["tiles_per_row"]) == (kind, tl, tiles), cfg
    assert _max_per_tile([hpos[(rr * n_s + ss) * 2] for rr, ss in dense], L, tl) > REC_CAP
    exp, *_ = _oracle_haps(O, synth, d, sv, r, s, L)
    _golden.eq(f"svar2_hint[{cfg}]", 0, out.cpu().numpy().reshape(-1, 4), O.onehot(exp, parallel=True))


# ---------------------------------------------------------------------------------------------------------------------
# 6. the fixed-length job and its rings at the benchmark's shapes
# ---------------------------------------------------------------------------------------------------------------------
_BENCH_CACHE: dict = {}


def _bench_workload(name):
    import bench

    base = "cfg3" if name == "cfg3t" else name  # (the same data: cfg3 carries the tracks cfg3t reads)
    if base not in _BENCH_CACHE:
        _BENCH_CACHE.clear()  # one large workload in host memory at a time
        _BENCH_CACHE[base] = bench.build_workload(base, 3)
    return bench.WORKLOADS[name], _BENCH_CACHE[base][1]


def _bench_ring(w, mode: str, n_tracks: int, steps: int = 20) -> int:
    """The ring bench.run_b200 picks for `--steps steps` with its default --ring / --ring-gib / --min-calls."""
    out_bytes_step = w["pairs"] * 2 * w["window"] * ({"onehot": 4, "u8": 1, "annotated": 9}[mode] + 4 * n_tracks)
    cap = max(1, min(128, int(12.0 * (1 << 30)) // (2 * out_bytes_step), max(1, (2 << 30) // out_bytes_step)))
    return max((r for r in range(1, cap + 1) if steps % r == 0 and steps // r >= 1), default=1)


def _bench_ring_tracks(w, n_tracks: int, steps: int = 20) -> int:
    """The ring of bench.run_b200's track leg (cfg3t: the cfg3 timed block with realigned tracks) for `--steps steps`."""
    ring = _bench_ring(w, "onehot", 0, steps)
    bp_per_step = w["pairs"] * 2 * w["window"]
    return max((r for r in range(1, ring + 1) if steps % r == 0 and r * 2 * bp_per_step * (4 + 4 * n_tracks) <= 12.0 * (1 << 30)),
               default=1)


def _bench_oracle(O, d, idx, L, annotated=False):
    from genvarloader_b200 import synth
    from tests.test_gpu_svar2_dataset import _oracle_haps

    r, s = idx // d.n_samples, idx % d.n_samples
    if getattr(d, "svar2", None) is not None:
        return _oracle_haps(O, synth, d, d.svar2, r, s, L)[0]
    regions, goi, to_rc, _ = synth.batch_args(d, r, s)
    args = _host_args(d, regions, np.zeros(goi.shape, np.int32), goi, N, L)
    if annotated:
        return O.reconstruct_annotated_haplotypes_fused(*args, None, None, to_rc, parallel=True)[:3]
    return O.reconstruct_haplotypes_fused(*args, None, None, to_rc, parallel=True)[0]


_TRACK_FILLS = [("track0", 0, 0.0), ("track1", 4, 1.0)]  # Repeat5p and Interpolate(1), as bench.py fills cfg3t


def _check_batch(O, d, L, sel, res, n_tracks, mode, tag):
    """One batch of the fixed-length job (queries `sel`, results as the pipeline hands them out) against the oracle."""
    from genvarloader_b200 import synth

    seq, trk = res if n_tracks else (res, None)
    if mode == "annotated":
        e_out, e_v, e_p = _bench_oracle(O, d, sel, L, annotated=True)
        _golden.eq(tag + ".haps", 0, seq.haps.cpu().numpy().ravel(), e_out)
        _golden.eq(tag + ".var_idxs", 0, seq.var_idxs.cpu().numpy().ravel(), e_v)
        _golden.eq(tag + ".ref_coords", 0, seq.ref_coords.cpu().numpy().ravel(), e_p)
    else:
        e_out = _bench_oracle(O, d, sel, L)
        _golden.eq(tag + ".onehot", 0, seq.cpu().numpy().reshape(-1, 4), O.onehot(e_out, parallel=True))
    if n_tracks:
        regions, goi, to_rc, ds_idx = synth.batch_args(d, sel // d.n_samples, sel % d.n_samples)
        exp_t = _track_oracle(O, d, regions, goi, to_rc, ds_idx, L, _TRACK_FILLS[:n_tracks])
        got_t = trk.cpu().numpy()  # (b, t, p, L)
        for ti in range(n_tracks):
            _golden.eq(f"{tag}.track{ti}", 0, np.ascontiguousarray(got_t[:, ti]).ravel(), exp_t[ti])


def _check_config(cfg, eng, L, rows, mode, n_tracks):
    """The configuration a call of the fixed-length job over `rows` rows must reach: static slices bounded by the longest
    slot (clamped to the typical slot of an svar2 source for the tile choice) and the tile choice of gvl_dev_hap_exec."""
    rb = max(eng.max_slot_len, 1)
    if getattr(eng, "typ_slot_len", 0) > 0:
        rb = min(rb, eng.typ_slot_len)
    nt = _plan_width(rows * max(eng.max_slot_len, 1), rows)
    assert (cfg["plan_threads"], cfg["plan_static"], cfg["rec_bound"]) == (nt, 1, rb), cfg
    if n_tracks:
        assert (cfg["trk_plan_threads"], cfg["trk_plan_static"]) == (nt, 1), cfg
    if mode == "onehot":
        assert (cfg["exec_kernel"], cfg["tile_len"], cfg["tiles_per_row"]) == _packed_choice(L, rows, rb, _sms()), cfg
    else:
        assert cfg["exec_kernel"] == "bytes", cfg


@pytest.mark.parametrize("name,mode", [("cfg1", "onehot"), ("cfg2", "onehot"), ("cfg2d", "onehot"), ("cfg3", "onehot"),
                                       ("cfg3t", "onehot"), ("cfg4", "onehot"), ("cfg4", "annotated")])
def test_bench_shapes_ring_vs_oracle(cuda_device, O, name, mode):
    import torch

    import bench
    from genvarloader_b200 import Interpolate, Repeat5p
    from genvarloader_b200._dataset import Dataset
    from genvarloader_b200._pipeline import FixedPipeline
    from genvarloader_b200._types import AnnotatedHaps

    w, d = _bench_workload(name)
    L, pairs = w["window"], w["pairs"]
    n_tracks = w.get("tracks", 0)
    ds = Dataset.from_synth(cuda_device, d, rng=10, svar2=getattr(d, "svar2", None)).with_len(L)  # (jitter 0)
    ds = ds.with_seqs("annotated") if mode == "annotated" else ds.with_encoding("onehot")
    if n_tracks:
        ds = ds.with_tracks([f"track{i}" for i in range(n_tracks)]).with_insertion_fill({"track0": Repeat5p(), "track1": Interpolate(1)})
        R = _bench_ring_tracks(bench.WORKLOADS["cfg3"], n_tracks)
    else:
        ds = ds.with_tracks(False)
        R = _bench_ring(w, mode, 0)
    idx = bench.draw_indices(d, R * pairs, 103)
    pipe = FixedPipeline(ds, pairs, ring=R)
    try:
        pipe.submit(0, idx)
        out = pipe.acquire(0)
        torch.cuda.synchronize()
        pipe.check()
        cfg = _launch(pipe.halves[0].eng.ctx.handle)
        _check_config(cfg, ds.engine, L, 2 * pairs * R, mode, n_tracks)
        if name in ("cfg3", "cfg3t"):
            assert (cfg["exec_kernel"], cfg["tile_len"], cfg["plan_static"]) == ("packed_unroll4", OH_MAX_TILE, 1), cfg
        for k in (0, R - 1):
            _check_batch(O, d, L, idx[k * pairs:(k + 1) * pairs], out.result(k * pairs, pairs), n_tracks, mode,
                         f"{name}.{mode}.ring{R}.batch{k}[{cfg}]")
    finally:
        del pipe
        torch.cuda.empty_cache()
    # one __getitem__ of 264 queries: more than 256 take the staged index upload instead of travelling with the launch.  The
    # whole call runs on the device; queries on both sides of 256 are compared (all 264 of cfg3 would be 1.1 GB of one-hot).
    sel = bench.draw_indices(d, 264, 7)
    res = ds[sel // d.n_samples, sel % d.n_samples]
    torch.cuda.synchronize()
    cfg = _launch(ds.engine.ctx.handle)
    _check_config(cfg, ds.engine, L, 2 * 264, mode, n_tracks)
    sub = np.array([0, 1, 255, 256, 263])
    ts = torch.from_numpy(sub).to(cuda_device)

    def pick(x):
        if isinstance(x, AnnotatedHaps):
            return AnnotatedHaps(x.haps[ts], x.var_idxs[ts], x.ref_coords[ts])
        return x[ts]

    _check_batch(O, d, L, sel[sub], pick(res) if not n_tracks else tuple(pick(x) for x in res), n_tracks, mode,
                 f"{name}.{mode}.getitem264[{cfg}]")
    del res
    torch.cuda.empty_cache()
