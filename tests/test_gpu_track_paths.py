"""Every tile path of the track execute, pinned bit for bit to the oracle.

`trk_tile_prep_kernel` cuts every (track, row) into tiles of TRK_TILE output values and sends each tile down one of
three paths (gvl_tracks_exec.cuh): the single pass (at most T3_REC staged records, carry included, and T3_ITV staged
intervals), TD_BIG sub-passes when a tile needs more, and TD_GENERIC per-value resolution for unsorted variant lists and
dense sources.  A mistake in one path only shows in the tiles that take it, so every case here:

  * places records and interval boundaries at chosen OUTPUT positions -- tile edges of forward and reverse rows, exactly
    at and one past the staging limits, insertions and deletions longer than a tile -- through a variant table and an
    interval SoA built for it (`geometry_dataset`; tests/test_track_path_geometry.py checks the builder on the CPU);
  * asserts through gvl_debug_track_tiles that its target tiles took the intended path with the intended record and
    interval counts, with the constants parsed from the sources, so a retune fails loudly instead of quietly testing
    something else;
  * compares every float with the oracle at 0 ulp.

Haplotype positions: on an unshifted row, output position h of a forward row (L - 1 - h of a reverse row) holds the
track value of haplotype position h (DESIGN section 4.1).  Only indels are track records (a SNP changes no position)."""
from __future__ import annotations

import dataclasses
import re
from pathlib import Path

import numpy as np
import pytest

from tests import _golden

pytestmark = pytest.mark.gpu

_CSRC = Path(__file__).resolve().parent.parent / "genvarloader_b200" / "csrc"


def _constants() -> dict:
    ex = (_CSRC / "gvl_tracks_exec.cuh").read_text()
    tr = (_CSRC / "gvl_tracks.cu").read_text()
    c = {m.group(1): int(m.group(2)) for m in re.finditer(r"constexpr int (\w+) = (-?\d+);", ex + tr)}
    c.update({m.group(1): int(m.group(2)) for m in re.finditer(r"\b(TD_[A-Z]+) = (\d+)", ex)})
    c["TILE_DESC_BYTES"] = int(re.search(r"#define GVL_TILE_DESC_BYTES (\d+)", (_CSRC / "gvl_common.cuh").read_text()).group(1))
    assert re.search(r"static_assert\(sizeof\(TileDesc\) == GVL_TILE_DESC_BYTES", ex)
    grow = re.search(r"int ensure_tdesc\(.*?int64_t cap = n \+ n / (\d+) \+ (\d+);", (_CSRC / "gvl_ctx.cu").read_text(), re.S)
    c["GROW_DIV"], c["GROW_ADD"] = int(grow.group(1)), int(grow.group(2))
    return c


C_ = _constants()
TILE, T3_REC, T3_ITV = C_["TRK_TILE"], C_["T3_REC"], C_["T3_ITV"]
TD_RC, TD_GENERIC, TD_BIG = C_["TD_RC"], C_["TD_GENERIC"], C_["TD_BIG"]


def tdesc_cap(n: int) -> int:
    """Descriptors ensure_tdesc allocates when a call needs n (gvl_ctx.cu)."""
    return n + n // C_["GROW_DIV"] + C_["GROW_ADD"]


# ---------------------------------------------------------------------------------------------------------------------
# geometry: variant tables and interval SoAs with records and boundaries at chosen output positions
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Slot:
    """One (region, sample) slot.  `ev[p]`: indels of ploid p as (haplotype position, ilen), sorted (ilen > 0: an
    insertion writing ilen + 1 values from h on; ilen < 0: a deletion whose anchor at h is followed by the source after
    the deleted bases).  `cuts`: haplotype positions of ploid 0 where an interval boundary lies; `src_cuts`: boundaries
    given as source positions relative to the region start; `quiet`: relative source ranges with no other boundary and
    every interval kept; `keep`: haplotype cut positions whose neighbouring intervals are kept; `bg`: mean spacing of
    the other boundaries (0: none); `empty`: the slot has no interval."""
    ev: tuple = ((), ())
    cuts: tuple = ()
    src_cuts: tuple = ()
    quiet: tuple = ()
    keep: tuple = ()
    bg: int = 90
    empty: bool = False
    L: int | None = None  # the row length the slot is laid out for (reverse rows: tile edges count from the row's end)


def src_of(ev, h: int):
    """Source position (relative to the region start) written at haplotype position h, None inside an insertion."""
    g = 0
    for he, il in ev:
        if h < he:
            break
        if il > 0 and h <= he + il:
            return None
        if h == he:  # a deletion's anchor: still the source before the deleted bases
            return h - g
        g += il
    return h - g


def edges(L: int, rc: bool):
    """Tile edges of a row in haplotype coordinates (forward rows: multiples of TILE; reverse rows: from the row's end)."""
    return [L - k * TILE if rc else k * TILE for k in range(1, -(-L // TILE))]


def tiles(L: int, rc: bool):
    """(h0, h1) of every tile of a row, in output order."""
    out = []
    for t0 in range(0, L, TILE):
        t1 = min(t0 + TILE, L)
        out.append((L - t1, L - t0) if rc else (t0, t1))
    return out


def edge_slot(L: int, rc: bool, mode0: int) -> Slot:
    """Records and interval boundaries around every tile edge B, four patterns in turn: boundaries at B - 1, B, B + 1
    (adjacent intervals meeting at B); an insertion across B (the tile starts on a live carry); a deletion across B with a
    boundary inside the deleted bases; boundaries at B - 1 and B (an interval ends on the tile end)."""
    ev = ([], [])
    cuts, src_cuts, keep = [0, 1, L - 1, L], [], []
    for p in range(2):
        for i, B in enumerate(edges(L, rc)):
            if not 16 <= B <= L - 16:
                continue
            mode = (mode0 + i + p) % 4
            if mode == 1:
                ev[p].append((B - 3, 6))
            elif mode == 2:
                ev[p].append((B - 2, -5))
    ev = (sorted(ev[0]), sorted(ev[1]))
    for i, B in enumerate(edges(L, rc)):
        if not 16 <= B <= L - 16:
            continue
        mode = (mode0 + i) % 4
        if mode == 0:
            cuts += [B - 1, B, B + 1]
            keep += [B]
        elif mode == 1:
            cuts += [B - 8, B + 6]
        elif mode == 2:
            cuts += [B, B + 2]
            src_cuts += [src_of(ev[0], B - 2) + 3]  # inside the deleted bases: the boundary vanishes
        else:
            cuts += [B - 1, B]
            keep += [B]
    return Slot(ev=(tuple(sorted(ev[0])), tuple(sorted(ev[1]))), cuts=tuple(cuts), src_cuts=tuple(src_cuts), keep=tuple(keep),
                L=L)


def dense_indels(h: int, n: int, gap: int = 20, long_at: int = -1, long_k: int = 300):
    """n indels from haplotype position h on (insertions of 2 and deletions of 2 in turn, `gap` copied values apart); the
    `long_at`-th is an insertion of `long_k`."""
    ev = []
    for i in range(n):
        il = long_k if i == long_at else (2 if i % 2 == 0 else -2)
        ev.append((h, il))
        h += (il + 1 if il > 0 else 1) + gap
    return ev


def lim_slot(extra_itv: int, rec: tuple) -> Slot:
    """Rows of 3 TILE values: the tile [0, TILE) holds exactly T3_ITV + extra_itv stored intervals and no record; the
    tile [TILE, 2 TILE) holds rec[p] records on ploid p (virtual carry: m = 1 + rec[p]; a tuple: dense_indels arguments)."""
    step = TILE // T3_ITV
    cuts = list(range(0, TILE + 1, step)) + [step // 2 + step * i for i in range(extra_itv)]
    ev = tuple(tuple(dense_indels(TILE + 40, n, gap=60)) if not isinstance(n, tuple) else tuple(dense_indels(TILE + 30, *n))
               for n in rec)
    return Slot(ev=ev, cuts=tuple(sorted(set(cuts))), quiet=((0, TILE),), keep=(0, TILE), L=3 * TILE)


def both_slot() -> Slot:
    """Tile [TILE, 2 TILE): more records than staged (ploid 0) and 2-bp intervals; tile [2 TILE, 3 TILE): a deletion of
    3,000 bases over 2-bp intervals, so that a sub-pass ends with every staged interval behind the deletion."""
    d_at = 2 * TILE + 200
    ev0 = tuple(dense_indels(TILE + 30, 120)) + ((d_at, -3000),)
    ev1 = ((d_at, -3000),)
    lo, hi = src_of(ev0, TILE), src_of(ev0, d_at) + 3000 + 400
    return Slot(ev=(ev0, ev1), src_cuts=tuple(range(lo, hi + 1, 2)), quiet=((lo, hi),), L=3 * TILE)


def long_ins_slot(at: int = 3000, k: int = 20000) -> Slot:
    """Ploid 0: an insertion of k values (covering whole tiles); ploid 1: a deletion longer than a tile.  1-bp intervals
    around the insertion's source position: every Interpolate / FlankSample anchor has a value of its own."""
    ev0 = ((at, k),)
    ev1 = ((6000, -9000),)
    v = src_of(ev0, at - 1) + 1  # the insertion's own source position (v_rel_pos)
    return Slot(ev=(ev0, ev1), src_cuts=tuple(range(v - 8, v + 9)), quiet=((v - 8, v + 8),), L=3 * TILE + 64)


def cross_slot() -> Slot:
    """Ploid 0: an insertion longer than a tile that starts before the first tile edge; ploid 1: a deletion of 9,000
    bases anchored two positions before it."""
    ev0 = ((TILE - 1200, 9000),)
    ev1 = ((TILE - 2, -9000),)
    v = src_of(ev0, TILE - 1201) + 1
    return Slot(ev=(ev0, ev1), src_cuts=tuple(range(v - 8, v + 9)), cuts=(TILE + 9000,), quiet=((v - 8, v + 8),),
                L=3 * TILE + 64)


def wide_slot(L: int) -> Slot:
    """One interval over several whole tiles (no boundary in between), an insertion across the first edge of a reverse
    row."""
    B = L - TILE
    return Slot(ev=(((B - 4, 7),), ()), cuts=(100, L - 300), quiet=((100, L - 300),), keep=(100,), L=L)


# (region start, region length, strand) and the slots of sample 0 / sample 1
def _layout(C: int):
    R = 3 * TILE + 64
    return [
        (-37, R, 1, lambda: edge_slot(R, False, 0), lambda: long_ins_slot()),
        (40_000, 3 * TILE, -1, lambda: lim_slot(0, (T3_REC - 1, T3_REC)), lambda: lim_slot(1, ((130, 20, T3_REC - 2), T3_REC + 1))),
        (80_000, 3 * TILE, 1, lambda: lim_slot(0, (T3_REC - 1, T3_REC)), lambda: lim_slot(1, ((130, 20, T3_REC - 2), T3_REC + 1))),
        (120_000, 3 * TILE, 1, both_slot, cross_slot),
        (170_000, 3 * TILE + 1, -1, lambda: edge_slot(3 * TILE + 1, True, 1), lambda: edge_slot(3 * TILE - 1, True, 2)),
        (210_000, TILE + 1, -1, lambda: edge_slot(TILE + 1, True, 3), lambda: Slot(cuts=(1, 2, 7, 8, 15, 16), L=TILE)),
        (250_000, R, -1, lambda: long_ins_slot(), lambda: wide_slot(R)),
        (C - R + 53, R, 1, lambda: edge_slot(R, False, 2), lambda: Slot(empty=True, L=R)),
    ]


GEOM_CONTIG = 320_000
N_TRACKS = 9


def _slot_records(ev, s0: int, C: int, nxt: int = 1):
    """(pos, alt_len, ilen) of a slot's indels."""
    out, g = [], 0
    for h, il in ev:
        pos = s0 + h - g
        used = 1 - min(il, 0)
        assert pos >= nxt and pos + used < C - 2, (h, il, pos)
        out.append((pos, 1 + max(il, 0), il))
        g += il
        nxt = pos + used
    return out


def _slot_intervals(sl: Slot, s0: int, R: int, C: int, rng):
    """Interval SoA of one slot (genomic coordinates), sorted and non-overlapping."""
    if sl.empty:
        return np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32)
    lo, hi = max(-300, -s0), min(R + 12_000, C - s0)
    pts = {src_of(sl.ev[0], h) for h in sl.cuts} | set(sl.src_cuts)
    assert None not in pts, "an interval boundary inside an insertion"
    keep_src = {src_of(sl.ev[0], h) for h in sl.keep}
    if sl.bg:
        x = lo
        while x < hi:
            x += int(rng.integers(1, 2 * sl.bg))
            if not any(a <= x <= b for a, b in sl.quiet):
                pts.add(x)
    pts = np.array(sorted(p for p in pts if lo <= p <= hi), np.int64)
    st, en = pts[:-1], pts[1:]
    quiet = np.zeros(st.size, bool)
    for a, b in sl.quiet:
        quiet |= (st >= a) & (en <= b)
    forced = np.isin(st, list(keep_src)) | np.isin(en, list(keep_src)) | quiet
    kept = forced | (rng.random(st.size) > 0.25)
    vals = rng.normal(size=st.size).astype(np.float32)
    vals[vals == 0] = 1.0
    return (st[kept] + s0).astype(np.int32), (en[kept] + s0).astype(np.int32), vals[kept]


def geometry_dataset(seed: int = 0):
    """The slots of `_layout` as a `synth.SynthData` (one contig, 8 regions, 2 samples, ploidy 2) with N_TRACKS tracks
    t0..t8 (the same chosen boundaries, different other boundaries and values).  Returns (data, slots)."""
    from genvarloader_b200 import synth

    rng = np.random.default_rng(seed)
    C = GEOM_CONTIG
    ref, ref_off = synth.make_reference(rng, [C], n_frac=0.0)
    lay = _layout(C)
    regions = np.array([[0, s, s + R, strand] for s, R, strand, *_ in lay], np.int32)
    slots = [mk() for *_, m0, m1 in lay for mk in (m0, m1)]
    recs = []
    for k, sl in enumerate(slots):
        s0 = int(regions[k // 2, 1])
        for p in range(2):
            recs.append(_slot_records(sl.ev[p], s0, C))
    pos = np.array([x[0] for r in recs for x in r], np.int64)
    alen = np.array([x[1] for r in recs for x in r], np.int64)
    ilen = np.array([x[2] for r in recs for x in r], np.int32)
    order = np.argsort(pos, kind="stable")
    new_idx = np.empty(order.size, np.int64)
    new_idx[order] = np.arange(order.size)
    alt_off = np.concatenate([[0], np.cumsum(alen[order])]).astype(np.int64)
    alt = synth.ACGT[rng.integers(0, 4, int(alt_off[-1]), dtype=np.uint8)]
    alt[alt_off[:-1]] = ref[pos[order]]  # indels start with the reference base
    lens = [len(r) for r in recs]
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    gv = new_idx.astype(np.int32)
    d = synth.SynthData(ref, ref_off, pos[order].astype(np.int32), ilen[order], alt, alt_off, gv,
                        np.ascontiguousarray(np.stack([off[:-1], off[1:]])), regions, 2, 2, 0)
    for t in range(N_TRACKS):
        trng = np.random.default_rng([seed, t])
        parts = [_slot_intervals(sl, int(regions[k // 2, 1]), int(regions[k // 2, 2] - regions[k // 2, 1]), C, trng)
                 for k, sl in enumerate(slots)]
        io = np.concatenate([[0], np.cumsum([p[0].size for p in parts])]).astype(np.int64)
        d.tracks[f"t{t}"] = tuple(np.concatenate([p[i] for p in parts]) for i in range(3)) + (io,)
    return d, slots


# slot index (region * 2 + sample) of every role
EDGE_F, LONG_INS_F, LIM_A_RC, LIM_B_RC, LIM_A_F, LIM_B_F, BOTH, CROSS = range(8)
EDGE_RC1, EDGE_RC2, EDGE_RC3, SHORT_RC, LONG_INS_RC, WIDE_RC, EDGE_F_END, EMPTY = range(8, 16)
FWD_LENGTHS = [1, 15, 16, TILE - 1, TILE, TILE + 1, 3 * TILE - 1, 3 * TILE + 1]
SHORT_LENGTHS = [1, 15, 16, TILE - 1, TILE]


def handover_tiles(d, slots, k: int, p: int, track: str = "t0"):
    """Tiles (h0) of slot k, ploid p, in which a sub-pass must end with every staged interval behind a deletion: the first
    T3_ITV intervals that reach the tile all end before the deletion's source resumes, and the last of them starts inside
    the deleted bases."""
    s, e, _, io = d.tracks[track]
    s0 = int(d.regions[k // 2, 1])
    ev = slots[k].ev[p]
    lo, hi = int(io[k]), int(io[k + 1])
    out = []
    for h0, h1 in tiles(slots[k].L, d.regions[k // 2, 3] == -1):
        dels = [(h, -il) for h, il in ev if il < 0 and h0 < h < h1]
        if not dels or src_of(ev, h0) is None:
            continue
        it0 = lo + int(np.searchsorted(e[lo:hi], s0 + src_of(ev, h0), "right"))
        if it0 + T3_ITV > hi:
            continue
        for h, k_del in dels:
            vrel = src_of(ev, h)
            if e[it0 + T3_ITV - 1] <= s0 + vrel + k_del + 1 and s[it0 + T3_ITV - 1] > s0 + vrel:
                out.append(h0)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# device calls
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def K(cuda_device):
    from genvarloader_b200 import _kernels

    return _kernels


@pytest.fixture(scope="module")
def O():
    from oracle import oracle

    return oracle


@pytest.fixture(scope="module")
def G():
    return geometry_dataset()


def _tiles(handle):
    """Tiles of the last track call of a context, each checked to fit the descriptor buffer."""
    from genvarloader_b200 import _ffi

    assert (_ffi.TILE_RC, _ffi.TILE_GENERIC, _ffi.TILE_BIG) == (TD_RC, TD_GENERIC, TD_BIG)
    t, n, nb = _ffi.track_tiles(handle)
    assert nb >= n * C_["TILE_DESC_BYTES"], (n, nb)
    return t


def _row_tiles(t, row: int, track: int = 0):
    sel = t[(t[:, 0] == track) & (t[:, 1] == row)]
    return {(int(x[2]), int(x[3])): x for x in sel}


def _fused(K, O, d, ks, lens, strategy=0, param=0.0, track="t0", tag=""):
    """The host fused entry over slots `ks` (one query each) with row lengths lens[q][p]; compared with the oracle.
    Returns the tiles of the call."""
    from genvarloader_b200 import synth

    ks = np.asarray(ks)
    regions, goi, to_rc, ds_idx = synth.batch_args(d, ks // 2, ks % 2)
    lens = np.asarray(lens, np.int64).reshape(goi.shape)
    oo = np.concatenate([[0], np.cumsum(lens.ravel())]).astype(np.int64)
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2], d.v_starts)
    to = np.concatenate([[0], np.cumsum((regions[:, 2] - regions[:, 1]) - diffs.clip(max=0).min(1))]).astype(np.int64)
    s, e, v, io = d.tracks[track]
    a = (oo, regions, np.zeros(goi.shape, np.int32), goi, d.geno_v_idxs, d.geno_offsets, d.v_starts, d.ilens, ds_idx, s, e, v, io,
         to, np.array([param], np.float64), strategy, 1234, None, None, to_rc)
    exp = np.zeros(int(oo[-1]), np.float32)
    O.intervals_and_realign_track_fused(exp, *a)
    got = np.full(int(oo[-1]), 7.0, np.float32)
    K.intervals_and_realign_track_fused(got, *a)
    t = _tiles(K.default_ctx().handle)
    bad = np.flatnonzero(got.view(np.uint32) != exp.view(np.uint32))
    row = int(np.searchsorted(oo, bad[0], "right") - 1) if bad.size else -1
    _golden.eq(f"{tag}[strategy {strategy}, param {param}] first bad row {row} at {bad[0] - oo[row] if bad.size else -1}", 0,
               got, exp)
    return t, to_rc


def _fast(x):
    return (int(x[4]) & (TD_BIG | TD_GENERIC)) == 0


# ---------------------------------------------------------------------------------------------------------------------
# 1. the single pass at tile edges, forward and reverse rows
# ---------------------------------------------------------------------------------------------------------------------
def test_fast_path_at_tile_edges(K, O, G):
    """Rows of 1 ... 3 TILE + 1 values (ragged: chunks cut by row ends), edges of forward and reverse rows, windows over
    both contig ends, an interval over whole tiles, an empty slot -- every tile a single pass."""
    d, slots = G
    F = FWD_LENGTHS
    ks = [EDGE_F] * 4 + [EDGE_F_END] * 4 + [EDGE_RC1, EDGE_RC2, EDGE_RC3, WIDE_RC, EMPTY] + [SHORT_RC] * 3
    lens = [[F[i], F[7 - i]] for i in range(4)] + [[F[i + 4], F[3 - i]] for i in range(4)]
    lens += [[slots[k].L] * 2 for k in (EDGE_RC1, EDGE_RC2, EDGE_RC3, WIDE_RC)] + [[3 * TILE, 5]]
    lens += [[SHORT_LENGTHS[i], SHORT_LENGTHS[4 - i]] for i in range(3)]
    t, to_rc = _fused(K, O, d, ks, lens, tag="edges")
    for row, L in enumerate(np.asarray(lens).ravel()):
        rt = _row_tiles(t, row)
        assert sorted(rt) == sorted(tiles(int(L), bool(to_rc[row]))), row
        for x in rt.values():
            assert _fast(x) and bool(x[4] & TD_RC) == bool(to_rc[row]), (row, x)


@pytest.mark.parametrize("strategy,param", [(0, 0.0), (1, 0.0), (2, -2.5), (3, 4.0), (4, 1.0), (4, 2.0), (4, 3.0)])
def test_records_across_tiles(K, O, G, strategy, param):
    """Insertions longer than a tile (a tile wholly inside one: one record, one interval, fills whose anchors lie in other
    tiles or beyond the staged intervals), an insertion across an edge, deletions longer than a tile -- every fill."""
    d, slots = G
    ks = [LONG_INS_F, LONG_INS_RC, CROSS, EDGE_F]
    lens = [[slots[k].L] * 2 for k in ks[:3]] + [[3 * TILE + 1, 3 * TILE - 1]]
    t, to_rc = _fused(K, O, d, ks, lens, strategy, param, track=f"t{strategy + 2 * (param == 3.0)}", tag="across")
    for row in range(len(ks) * 2):
        assert all(_fast(x) for x in _row_tiles(t, row).values()), row
    ins_at, k = slots[LONG_INS_F].ev[0][0]
    for row in (0, 2):  # ploid 0 of the long insertion, forward and reverse: the tile [TILE, 2 TILE) lies inside it
        x = _row_tiles(t, row)[(TILE, 2 * TILE)] if row == 0 else _row_tiles(t, row)[(slots[LONG_INS_RC].L - 2 * TILE,
                                                                                     slots[LONG_INS_RC].L - TILE)]
        assert ins_at < x[2] and x[3] <= ins_at + k and (x[5], x[6]) == (1, 1), x


# ---------------------------------------------------------------------------------------------------------------------
# 2. staging limits and sub-passes
# ---------------------------------------------------------------------------------------------------------------------
def test_staging_limits(K, O, G):
    """T3_REC records (carry included) and T3_ITV intervals fit one pass, one more of either does not; dense records,
    1-bp-scale intervals and both at once; a sub-pass that ends where a long insertion starts; the hand-over after a
    deletion that skips every staged interval."""
    d, slots = G
    ks = [LIM_A_F, LIM_A_RC, LIM_B_F, LIM_B_RC, BOTH]
    t, _ = _fused(K, O, d, ks, [[3 * TILE] * 2] * 5, tag="limits")
    first, second = (0, TILE), (TILE, 2 * TILE)
    for q in range(4):
        for p in range(2):
            rt = _row_tiles(t, 2 * q + p)
            x0, x1 = rt[first], rt[second]
            if ks[q] in (LIM_A_F, LIM_A_RC):
                assert _fast(x0) and x0[6] == T3_ITV, x0
                want = T3_REC if p == 0 else T3_REC + 1
                assert x1[5] == want and _fast(x1) == (want <= T3_REC), x1
            else:
                assert x0[4] & TD_BIG and x0[6] == T3_ITV + 1, x0  # BIG from intervals
                assert x1[4] & TD_BIG and x1[5] > T3_REC and x1[6] <= T3_ITV, x1  # BIG from records
    b0, b1 = _row_tiles(t, 8), _row_tiles(t, 9)
    assert b0[second][4] & TD_BIG and b0[second][5] > T3_REC and b0[second][6] > T3_ITV, b0[second]  # both at once
    assert b1[second][4] & TD_BIG and b1[second][5] <= T3_REC and b1[second][6] > T3_ITV, b1[second]
    for p, rt in ((0, b0), (1, b1)):
        ho = handover_tiles(d, slots, BOTH, p)
        assert 2 * TILE in ho, (p, ho)
        assert rt[(2 * TILE, 3 * TILE)][4] & TD_BIG
    # the sub-pass of the long-insertion slot ends where the insertion starts: it is the last staged record
    ev = slots[LIM_B_F].ev[0]
    assert ev[T3_REC - 2][1] == 300 and TILE < ev[T3_REC - 2][0] < 2 * TILE


# ---------------------------------------------------------------------------------------------------------------------
# 3. per-value resolution
# ---------------------------------------------------------------------------------------------------------------------
def _with_jumps(d, ks):
    """A copy of `d` whose slots `ks` (ploid 0) end their variant list with a deletion that starts before the region and
    reaches into it: listed after the slot's other indels, it moves the source back (src/tracks/mod.rs:271-274), so the
    plan leaves a jump record and the row is resolved value by value."""
    import copy

    d = copy.copy(d)
    gv, go = list(d.geno_v_idxs), d.geno_offsets.copy()
    vs, il, ao, alt = list(d.v_starts), list(d.ilens), list(d.alt_offsets), list(d.alt_alleles)
    for k in ks:
        pos = int(d.regions[k // 2, 1]) - 3
        vs.append(pos), il.append(-10), alt.append(d.reference[pos]), ao.append(ao[-1] + 1)
        g = 2 * k
        lst = gv[go[0, g]: go[1, g]] + [len(vs) - 1]
        go[0, g], go[1, g] = len(gv), len(gv) + len(lst)
        gv += lst
    d.geno_v_idxs, d.geno_offsets = np.array(gv, np.int32), go
    d.v_starts, d.ilens = np.array(vs, np.int32), np.array(il, np.int32)
    d.alt_alleles, d.alt_offsets = np.array(alt, np.uint8), np.array(ao, np.int64)
    return d


def test_generic_unsorted_lists(K, O, G):
    """Variant lists out of position order that move the source back (jump records), with intervals: those rows take
    TD_GENERIC in every tile, the others do not."""
    d, slots = G
    ks = [LIM_A_F, WIDE_RC, BOTH, CROSS]
    dj = _with_jumps(d, ks[:3])
    t, _ = _fused(K, O, dj, ks, [[slots[k].L] * 2 for k in ks], 4, 2.0, tag="unsorted")
    for row in range(2 * len(ks)):
        rt = _row_tiles(t, row)
        want = row % 2 == 0 and row < 6
        assert rt and all(bool(x[4] & TD_GENERIC) == want for x in rt.values()), (row, rt)


def _dense_windows(O, d, ks, rng, extra=40):
    from genvarloader_b200 import synth

    regions, goi, to_rc, ds_idx = synth.batch_args(d, ks // 2, ks % 2)
    diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2], d.v_starts)
    lens = np.maximum((regions[:, 2] - regions[:, 1])[:, None] + diffs, 0)
    oo = np.concatenate([[0], np.cumsum(lens.ravel())]).astype(np.int64)
    tl = (regions[:, 2] - regions[:, 1]) - np.minimum(diffs.min(1), 0) + extra
    to = np.concatenate([[0], np.cumsum(tl)]).astype(np.int64)
    return regions, goi, to_rc, ds_idx, oo, to, rng.standard_normal(int(to[-1])).astype(np.float32)


@pytest.mark.parametrize("strategy,param", [(0, 0.0), (3, 4.0), (4, 3.0)])
def test_generic_dense_sources(K, O, G, strategy, param):
    """Dense f32 source windows (shift_and_realign_tracks_sparse) and the svar2 dense source: rows over several tiles,
    every tile TD_GENERIC."""
    from genvarloader_b200 import synth

    d, slots = G
    ks = np.array([EDGE_F, LONG_INS_F, BOTH, CROSS, EDGE_RC1, LONG_INS_RC, LIM_B_RC])
    rng = np.random.default_rng(strategy)
    regions, goi, to_rc, ds_idx, oo, to, tracks = _dense_windows(O, d, ks, rng)
    a = (oo, regions, np.zeros(goi.shape, np.int32), goi, d.geno_v_idxs, d.geno_offsets, d.v_starts, d.ilens, tracks, to,
         np.array([param]), None, None, strategy, 77)
    exp, got = np.zeros(int(oo[-1]), np.float32), np.full(int(oo[-1]), 7.0, np.float32)
    O.shift_and_realign_tracks_sparse(exp, *a)
    K.shift_and_realign_tracks_sparse(got, *a)
    t = _tiles(K.default_ctx().handle)
    assert t.shape[0] == sum(-(-int(n) // TILE) for n in np.diff(oo)) and (t[:, 4] & TD_GENERIC).all()
    _golden.eq(f"dense[{strategy}]", 0, got, exp)
    ch = synth.to_svar2_channels(d, regions, ds_idx, dense_frac=0.5, seed=strategy)
    qs = rng.integers(0, 1000, ks.size).astype(np.int64)
    a = (oo, regions, np.zeros(goi.shape, np.int32), ch["vk_pos"], ch["vk_key"], ch["vk_off"], ch["dense_pos"], ch["dense_key"],
         ch["dense_range"], ch["dense_present"], ch["dense_present_off"], ch["key_ilen"], tracks, to, np.array([param]), strategy,
         91, qs)
    exp, got = np.zeros(int(oo[-1]), np.float32), np.full(int(oo[-1]), 7.0, np.float32)
    O.shift_and_realign_tracks_from_svar2(exp, *a)
    K.shift_and_realign_tracks_from_svar2(got, *a)
    t = _tiles(K.default_ctx().handle)
    assert t.shape[0] == sum(-(-int(n) // TILE) for n in np.diff(oo)) and (t[:, 4] & TD_GENERIC).all()
    _golden.eq(f"svar2[{strategy}]", 0, got, exp)


# ---------------------------------------------------------------------------------------------------------------------
# 4. layouts and track descriptors
# ---------------------------------------------------------------------------------------------------------------------
FILL_KEYS = ["repeat5p", "repeat5p_norm", "constant", "flank", "interp1", "interp2", "interp3", "flank", "constant"]


def _fills(m, n):
    from tests.test_gpu_spliced_tracks import FILLS

    f = [FILLS[k](m) for k in FILL_KEYS[:n]]
    if n > 7:  # two more fills that differ from the first ones by their parameter
        f[7] = m.FlankSample(9)
    if n > 8:
        f[8] = m.Constant(3.0)
    return f


def _same_tiles_every_track(t, n_tracks):
    def key(x):  # (row, h0, h1, reversed, records): the interval counts and with them TD_BIG differ between tracks
        return int(x[1]), int(x[2]), int(x[3]), int(x[4]) & TD_RC, int(x[5])

    base = {key(x) for x in t[t[:, 0] == 0]}
    assert base and all({key(x) for x in t[t[:, 0] == k]} == base for k in range(n_tracks))
    assert set(t[:, 0].tolist()) == set(range(n_tracks))


@pytest.mark.parametrize("n_tracks", [8, 9])
def test_dataset_layouts_many_tracks(cuda_device, O, G, n_tracks):
    """(b, t, p, ~l) rows of different lengths through Dataset.__getitem__ (descriptors inline for <= 8 tracks, a device
    array above), then the same slots as spliced rows (per-row destinations, gvl_dev_realign_tracks_plan_rows); every
    track with intervals and a fill of its own, so a mix-up of track indices shows."""
    import genvarloader_b200 as m
    from genvarloader_b200._dataset import Dataset
    from tests.test_gpu_spliced_tracks import _check_realigned, _element_batch, _oracle_realigned, _seed

    d, slots = G
    names = [f"t{i}" for i in range(n_tracks)]
    fills = _fills(m, n_tracks)
    ds = Dataset.from_synth(cuda_device, d, rng=0).with_tracks(names).with_insertion_fill(dict(zip(names, fills)))
    ks = np.array([EDGE_F, EDGE_RC1, LIM_B_F, BOTH, LONG_INS_RC, CROSS, EDGE_RC3, WIDE_RC, EMPTY])
    r, s = ks // 2, ks % 2
    _, trk = ds[r, s]
    t = _tiles(ds.engine.ctx.handle)
    _same_tiles_every_track(t, n_tracks)
    assert (t[:, 4] & TD_BIG).any()
    exp, oo = _oracle_realigned(d, O, r, s, fills, names, _seed(r, s, d.n_samples))
    _check_realigned(trk, exp, oo, np.ones(ks.size, np.int64), d.ploidy)
    rows = {"a": [0, 4], "b": [2, 1, 6], "c": [3], "d": [7, 5, 0]}
    sp = ds.with_settings(splice_info=rows)
    pairs = [(0, 0), (1, 1), (2, 0), (3, 1), (1, 0)]
    _, trk = sp[[p[0] for p in pairs], [p[1] for p in pairs]]
    t = _tiles(ds.engine.ctx.handle)
    _same_tiles_every_track(t, n_tracks)
    e_reg, e_s, n_el = _element_batch(d, rows, pairs)
    exp, oo = _oracle_realigned(d, O, e_reg, e_s, fills, names, _seed(e_reg, e_s, d.n_samples))
    _check_realigned(trk, exp, oo, n_el, d.ploidy)


def test_painted_rows(K, O, cuda_device, G):
    """Painted (identity-plan) rows at tile edges, reversed: the host paint entry (one track), then 9 tracks through a
    Dataset with realign_tracks=False, unspliced ((b, t, ~l) layout) and spliced (per-row destinations)."""
    from genvarloader_b200._dataset import Dataset
    from tests.test_gpu_spliced_tracks import _check_painted, _element_batch, _oracle_painted

    d, slots = G
    rng = np.random.default_rng(5)
    q = np.array([EDGE_F, EDGE_RC1, EDGE_RC2, WIDE_RC, EMPTY, SHORT_RC, LIM_A_RC])
    starts = d.regions[q // 2, 1].astype(np.int32) + np.array([0, 0, 3, -5, 0, 0, 1], np.int32)
    lens = np.array([3 * TILE + 1, TILE, TILE + 1, 2 * TILE - 1, 17, 15, 3 * TILE])
    oo = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    s, e, v, io = d.tracks["t1"]
    exp, got = np.zeros(int(oo[-1]), np.float32), np.full(int(oo[-1]), 7.0, np.float32)
    O.intervals_to_tracks(q, starts, s, e, v, io, exp, oo)
    K.intervals_to_tracks(q, starts, s, e, v, io, got, oo)
    t = _tiles(K.default_ctx().handle)
    for row, L in enumerate(lens):
        assert sorted(_row_tiles(t, row)) == tiles(int(L), False)
    _golden.eq("paint.host", 0, got, exp)
    names = [f"t{i}" for i in range(N_TRACKS)]
    ds = Dataset.from_synth(cuda_device, d, rng=0).with_tracks(names).with_settings(realign_tracks=False)
    r, sm = q // 2, q % 2
    _, trk = ds[r, sm]
    t = _tiles(ds.engine.ctx.handle)
    _same_tiles_every_track(t, N_TRACKS)
    for row, k in enumerate(q):
        rc = bool(d.regions[k // 2, 3] == -1)
        L = int(d.regions[k // 2, 2] - d.regions[k // 2, 1])
        rt = _row_tiles(t, row)
        assert sorted(rt) == sorted(tiles(L, rc)) and all(bool(x[4] & TD_RC) == rc and _fast(x) for x in rt.values())
    exp, offs = _oracle_painted(d, O, r, sm, names)
    _check_painted(trk, exp, offs, np.ones(q.size, np.int64))
    rows = {"a": [1, 4, 2], "b": [5], "c": [0, 3]}
    pairs = [(0, 1), (1, 0), (2, 1), (0, 0)]
    _, trk = ds.with_settings(splice_info=rows, realign_tracks=False)[[p[0] for p in pairs], [p[1] for p in pairs]]
    _same_tiles_every_track(_tiles(ds.engine.ctx.handle), N_TRACKS)
    e_reg, e_s, n_el = _element_batch(d, rows, pairs)
    exp, offs_e = _oracle_painted(d, O, e_reg, e_s, names)
    _check_painted(trk, exp, offs_e, n_el)


# ---------------------------------------------------------------------------------------------------------------------
# 5. the descriptor workspace: reused for smaller grids, regrown for larger ones
# ---------------------------------------------------------------------------------------------------------------------
def _paint_call(K, O, ctx, d, n_rows: int, grid: int, rng, tag):
    """One host paint call of n_rows rows whose grid (total // TILE + rows) is `grid`; checked against the oracle."""
    total = (grid - n_rows) * TILE
    lens = np.full(n_rows, total // n_rows, np.int64)
    lens[: total % n_rows] += 1
    lens[-1] += int(rng.integers(0, TILE // 2))  # (still below the next multiple of TILE of the total)
    q = rng.integers(0, 16, n_rows)
    starts = (d.regions[q // 2, 1] + rng.integers(-50, 50, n_rows)).astype(np.int32)
    oo = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    s, e, v, io = d.tracks["t3"]
    exp, got = np.zeros(int(oo[-1]), np.float32), np.full(int(oo[-1]), 7.0, np.float32)
    O.intervals_to_tracks(q, starts, s, e, v, io, exp, oo)
    K.intervals_to_tracks(q, starts, s, e, v, io, got, oo, ctx=ctx)
    from genvarloader_b200 import _ffi

    t, n, nb = _ffi.track_tiles(ctx.handle)
    assert n == grid and nb >= n * C_["TILE_DESC_BYTES"], (tag, n, nb)
    assert t.shape[0] == sum(-(-int(x) // TILE) for x in lens)
    _golden.eq(tag, 0, got, exp)
    return nb


def test_descriptor_workspace_growth(K, O, G):
    """On a fresh context: a first call sizes the buffer (cap descriptors); calls whose grid lies in (96/112 cap, cap] --
    the window a 96-byte descriptor buffer would have overrun -- reuse it; a larger call regrows it, a smaller one
    follows."""
    from genvarloader_b200 import _ffi

    d, _ = G
    rng = np.random.default_rng(8)
    ctx = _ffi.Ctx(0)
    try:
        g1 = 94
        nb = _paint_call(K, O, ctx, d, 16, g1, rng, "grow.first")
        cap = tdesc_cap(g1)
        assert nb == cap * C_["TILE_DESC_BYTES"]
        lo = cap * 96 // C_["TILE_DESC_BYTES"] + 1
        for g, n_rows in ((lo, 44), ((lo + cap) // 2, 30), (cap, 61)):
            assert g * C_["TILE_DESC_BYTES"] > 96 * cap and g <= cap  # more than a 96-byte-per-descriptor buffer holds
            assert _paint_call(K, O, ctx, d, n_rows, g, rng, f"grow.window[{g} of {cap}]") == nb
        g2 = cap + 1
        nb2 = _paint_call(K, O, ctx, d, 20, g2, rng, "grow.regrow")
        assert nb2 == tdesc_cap(g2) * C_["TILE_DESC_BYTES"]
        assert _paint_call(K, O, ctx, d, 9, 40, rng, "grow.after") == nb2
    finally:
        ctx.close()


def test_descriptor_workspace_growth_dataset(cuda_device, O, G):
    """The same through Dataset.__getitem__ with two realigned tracks: a batch, then a larger one inside the window."""
    import genvarloader_b200 as m
    from genvarloader_b200 import _ffi, synth
    from genvarloader_b200._dataset import Dataset
    from tests.test_gpu_spliced_tracks import _check_realigned, _oracle_realigned, _seed

    d, _ = G
    names = ["t0", "t5"]
    fills = [m.Interpolate(2), m.FlankSample(3)]
    ds = Dataset.from_synth(cuda_device, d, rng=0).with_tracks(names).with_insertion_fill(dict(zip(names, fills)))
    rng = np.random.default_rng(2)

    def grid_of(k):
        regions, goi, _, _ = synth.batch_args(d, k // 2, k % 2)
        diffs = O.get_diffs_sparse(goi, d.geno_v_idxs, d.geno_offsets, d.ilens, None, None, regions[:, 1], regions[:, 2],
                                   d.v_starts)
        total = int(np.maximum((regions[:, 2] - regions[:, 1])[:, None] + diffs, 0).sum())
        return (total // TILE + goi.size) * len(names)

    k1 = rng.integers(0, 16, 12)
    cap = tdesc_cap(grid_of(k1))
    lo = cap * 96 // C_["TILE_DESC_BYTES"] + 1
    k2 = None
    for n in range(12, 200):
        for _ in range(20):
            k = rng.integers(0, 16, n)
            if lo <= grid_of(k) <= cap:
                k2 = k
                break
        if k2 is not None:
            break
    assert k2 is not None
    for k, tag in ((k1, "first"), (k2, "window")):
        _, trk = ds[k // 2, k % 2]
        t, n, nb = _ffi.track_tiles(ds.engine.ctx.handle)
        assert n == grid_of(k) and nb >= n * C_["TILE_DESC_BYTES"], (tag, n, nb, cap)
        if tag == "window":
            assert lo <= n <= cap and nb == cap * C_["TILE_DESC_BYTES"], (n, nb, cap)
        exp, oo = _oracle_realigned(d, O, k // 2, k % 2, fills, names, _seed(k // 2, k % 2, d.n_samples))
        _check_realigned(trk, exp, oo, np.ones(k.size, np.int64), d.ploidy)
