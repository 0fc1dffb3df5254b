"""numpy/ctypes front end of the CPU oracle (oracle/gvl_oracle.c).

TEST INFRASTRUCTURE ONLY -- the product package (genvarloader_b200/) never imports this.
Allowed importers: tests/, __graft_entry__.smoke(), bench.py (cpu_baseline / --impl reference).

Function names, positional argument order and dtypes follow the reference's PyO3 module
(src/ffi/mod.rs; line numbers in each docstring) so parity tests read like the
reference's own tests/parity/*.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_SRC = _HERE / "gvl_oracle.c"


def _cpu_tag() -> str:
    """-march=native objects are only valid on the CPU model they were built on: key the .so by
    the CPU feature flags so the build container and the GPU box each get their own."""
    import hashlib

    try:
        flags = next(l for l in open("/proc/cpuinfo") if l.startswith("flags"))
    except Exception:
        flags = "generic"
    return hashlib.md5(flags.encode()).hexdigest()[:8]


_LIB = _HERE / f"libgvl_oracle_{_cpu_tag()}.so"

# -ffp-contract=off: the f64 Lagrange arithmetic of Interpolate must not be fused into FMAs.
_CFLAGS = ["-O3", "-march=native", "-ffp-contract=off", "-fPIC", "-shared", "-pthread"]


def build(force: bool = False, out: Path = _LIB) -> Path:
    """Compile the C restatement (gcc only; no reference sources involved)."""
    if force or not out.exists() or out.stat().st_mtime < _SRC.stat().st_mtime:
        subprocess.check_call(["gcc", *_CFLAGS, "-o", str(out), str(_SRC)])
    return out


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        path = _LIB
        if not _LIB.exists() and not os.access(_HERE, os.W_OK):
            # read-only source tree and no library for this CPU yet: compile into a temporary directory
            import tempfile

            path = build(out=Path(tempfile.mkdtemp(prefix="gvl_oracle_")) / _LIB.name)
        else:
            try:
                build()
            except Exception:
                if not _LIB.exists():
                    raise
        _lib = C.CDLL(str(path))
        _lib.gvl_oracle_xorshift64.restype = C.c_uint64
        _lib.gvl_oracle_xorshift64.argtypes = [C.c_uint64]
        _lib.gvl_oracle_hash4.restype = C.c_uint64
        _lib.gvl_oracle_hash4.argtypes = [C.c_uint64] * 4
        _lib.gvl_oracle_fused_out_offsets.restype = C.c_int64
        _lib.gvl_oracle_reconstruct_haplotypes_fused.restype = C.c_void_p
        _lib.gvl_oracle_get_threads.restype = C.c_int
    return _lib


def set_threads(n: int) -> None:
    """GVL_NUM_THREADS equivalent (python/genvarloader/_threads.py:92-115)."""
    lib().gvl_oracle_set_threads(C.c_int(int(n)))


def get_threads() -> int:
    return int(lib().gvl_oracle_get_threads())


def default_threads() -> int:
    env = os.environ.get("GVL_NUM_THREADS")
    if env:
        return max(1, int(env))
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:  # pragma: no cover
        return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------
def _p(a):
    """ctypes pointer for an optional contiguous array."""
    if a is None:
        return C.c_void_p(0)
    assert a.flags.c_contiguous, "oracle wants C-contiguous arrays"
    return C.c_void_p(a.ctypes.data)


def _c(a, dt):
    return None if a is None else np.ascontiguousarray(a, dt)


def _i64(x):
    return C.c_int64(int(x))


def _split_offsets(geno_offsets):
    """(2, n) starts/stops; a 1-D (n+1,) offsets array is normalised like
    python/genvarloader/_dataset/_genotypes.py:13-22."""
    go = np.asarray(geno_offsets)
    if go.ndim == 1:
        go = np.stack([go[:-1], go[1:]])
    go = np.ascontiguousarray(go, np.int64)
    return go, go[0], go[1]


# ------------------------------------------------------------------ PRNG (debug exports)
def _debug_xorshift64(x: int) -> int:
    """src/ffi/mod.rs:2824 / src/tracks/mod.rs:31."""
    return int(lib().gvl_oracle_xorshift64(C.c_uint64(int(x))))


def _debug_hash4(a: int, b: int, c: int, d: int) -> int:
    """src/ffi/mod.rs:2830 / src/tracks/mod.rs:48."""
    return int(lib().gvl_oracle_hash4(*(C.c_uint64(int(v)) for v in (a, b, c, d))))


# ------------------------------------------------------------------ genotypes
def get_diffs_sparse(geno_offset_idx, geno_v_idxs, geno_offsets, ilens, keep=None, keep_offsets=None,
                     q_starts=None, q_ends=None, v_starts=None, parallel=False):
    """src/ffi/mod.rs:145-157 -> src/genotypes/mod.rs:15-125.  Returns i32 (n_queries, ploidy)."""
    goi = _c(geno_offset_idx, np.int64)
    n_q, ploidy = goi.shape
    go, gs, ge = _split_offsets(geno_offsets)
    gv, il = _c(geno_v_idxs, np.int32), _c(ilens, np.int32)
    kp, ko = _c(keep, np.bool_), _c(keep_offsets, np.int64)
    qs, qe, vs = _c(q_starts, np.int32), _c(q_ends, np.int32), _c(v_starts, np.int32)
    diffs = np.zeros((n_q, ploidy), np.int32)
    lib().gvl_oracle_get_diffs_sparse(_p(goi), _p(gv), _p(gs), _p(ge), _p(il), _p(kp), _p(ko), _p(qs), _p(qe),
                                      _i64(1), _p(vs), _i64(n_q), _i64(ploidy), C.c_int(bool(parallel)), _p(diffs))
    return diffs


def choose_exonic_variants(starts, ends, geno_offset_idx, geno_v_idxs, geno_offsets, v_starts, ilens):
    """src/ffi/mod.rs:229-238 -> src/genotypes/mod.rs:132-176.  Returns (keep bool, keep_offsets i64)."""
    goi = _c(geno_offset_idx, np.int64)
    n_r, ploidy = goi.shape
    go, gs, ge = _split_offsets(geno_offsets)
    st, en = _c(starts, np.int32), _c(ends, np.int32)
    gv, vs, il = _c(geno_v_idxs, np.int32), _c(v_starts, np.int32), _c(ilens, np.int32)
    koff = np.zeros(n_r * ploidy + 1, np.int64)
    args = [_p(st), _p(en), _p(goi), _p(gv), _p(gs), _p(ge), _p(vs), _p(il), _i64(n_r), _i64(ploidy)]
    lib().gvl_oracle_choose_exonic_variants(*args, C.c_void_p(0), _p(koff))
    keep = np.zeros(int(koff[-1]), np.bool_)
    lib().gvl_oracle_choose_exonic_variants(*args, _p(keep), _p(koff))
    return keep, koff


# ------------------------------------------------------------------ haplotypes
def reconstruct_haplotypes_from_sparse(out, out_offsets, regions, shifts, geno_offset_idx, geno_offsets,
                                       geno_v_idxs, v_starts, ilens, alt_alleles, alt_offsets, ref_, ref_offsets,
                                       pad_char, keep=None, keep_offsets=None, annot_v_idxs=None,
                                       annot_ref_pos=None, parallel=False):
    """src/ffi/mod.rs:634-655 -> src/reconstruct/mod.rs:348-583.  Writes `out` (and annotations) in place."""
    assert out.dtype == np.uint8 and out.flags.c_contiguous
    oo = _c(out_offsets, np.int64)
    rg, sh = _c(regions, np.int32), _c(shifts, np.int32)
    goi = _c(geno_offset_idx, np.int64)
    batch, ploidy = goi.shape
    go, gs, ge = _split_offsets(geno_offsets)
    gv, vs, il = _c(geno_v_idxs, np.int32), _c(v_starts, np.int32), _c(ilens, np.int32)
    aa, ao = _c(alt_alleles, np.uint8), _c(alt_offsets, np.int64)
    rf, ro = _c(ref_, np.uint8), _c(ref_offsets, np.int64)
    kp, ko = _c(keep, np.bool_), _c(keep_offsets, np.int64)
    for a in (annot_v_idxs, annot_ref_pos):
        assert a is None or (a.dtype == np.int32 and a.flags.c_contiguous)
    lib().gvl_oracle_reconstruct_haplotypes_from_sparse(
        _p(out), _p(oo), _p(rg), _p(sh), _p(goi), _p(gs), _p(ge), _p(gv), _p(vs), _p(il), _p(aa), _p(ao), _p(rf),
        _p(ro), C.c_uint8(int(pad_char)), _p(kp), _p(ko), _p(annot_v_idxs), _p(annot_ref_pos), _i64(batch),
        _i64(ploidy), C.c_int(bool(parallel)))


def _fused(annotated, regions, shifts, geno_offset_idx, geno_offsets, geno_v_idxs, v_starts, ilens, alt_alleles,
           alt_offsets, ref_, ref_offsets, pad_char, output_length, keep, keep_offsets, to_rc, parallel):
    rg, sh = _c(regions, np.int32), _c(shifts, np.int32)
    goi = _c(geno_offset_idx, np.int64)
    batch, ploidy = goi.shape
    go, gs, ge = _split_offsets(geno_offsets)
    gv, vs, il = _c(geno_v_idxs, np.int32), _c(v_starts, np.int32), _c(ilens, np.int32)
    aa, ao = _c(alt_alleles, np.uint8), _c(alt_offsets, np.int64)
    rf, ro = _c(ref_, np.uint8), _c(ref_offsets, np.int64)
    kp, ko = _c(keep, np.bool_), _c(keep_offsets, np.int64)
    rc = _c(to_rc, np.bool_)
    par = C.c_int(bool(parallel))
    out_offsets = np.zeros(batch * ploidy + 1, np.int64)
    total = lib().gvl_oracle_fused_out_offsets(_p(rg), _p(goi), _p(gs), _p(ge), _p(gv), _p(vs), _p(il),
                                               _i64(output_length), _p(kp), _p(ko), _i64(batch), _i64(ploidy), par,
                                               _p(out_offsets), C.c_void_p(0))
    out = np.empty(int(total), np.uint8)
    av = np.empty(int(total), np.int32) if annotated else None
    ap = np.empty(int(total), np.int32) if annotated else None
    lib().gvl_oracle_fused_fill(_p(out), _p(av), _p(ap), _p(out_offsets), _p(rg), _p(sh), _p(goi), _p(gs), _p(ge),
                                _p(gv), _p(vs), _p(il), _p(aa), _p(ao), _p(rf), _p(ro), C.c_uint8(int(pad_char)),
                                _p(kp), _p(ko), _p(rc), _i64(batch), _i64(ploidy), par)
    return out, av, ap, out_offsets


def reconstruct_haplotypes_fused(regions, shifts, geno_offset_idx, geno_offsets, geno_v_idxs, v_starts, ilens,
                                 alt_alleles, alt_offsets, ref_, ref_offsets, pad_char, output_length, keep=None,
                                 keep_offsets=None, to_rc=None, parallel=False):
    """src/ffi/mod.rs:724-860.  Returns (out_data u8, out_offsets i64)."""
    out, _, _, oo = _fused(False, regions, shifts, geno_offset_idx, geno_offsets, geno_v_idxs, v_starts, ilens,
                           alt_alleles, alt_offsets, ref_, ref_offsets, pad_char, output_length, keep, keep_offsets,
                           to_rc, parallel)
    return out, oo


def reconstruct_annotated_haplotypes_fused(regions, shifts, geno_offset_idx, geno_offsets, geno_v_idxs, v_starts,
                                           ilens, alt_alleles, alt_offsets, ref_, ref_offsets, pad_char,
                                           output_length, keep=None, keep_offsets=None, to_rc=None, parallel=False):
    """src/ffi/mod.rs:2239-2397.  Returns (out_data u8, annot_v i32, annot_pos i32, out_offsets i64)."""
    return _fused(True, regions, shifts, geno_offset_idx, geno_offsets, geno_v_idxs, v_starts, ilens, alt_alleles,
                  alt_offsets, ref_, ref_offsets, pad_char, output_length, keep, keep_offsets, to_rc, parallel)


class FusedTimer:
    """Pre-marshalled one-crossing call of gvl_oracle_reconstruct_haplotypes_fused (+ optional one-hot pass)
    for the timed CPU baseline: sizes, mallocs, fills, RCs in C exactly like the reference's fused entry."""

    def __init__(self, regions, shifts, geno_offset_idx, geno_offsets, geno_v_idxs, v_starts, ilens, alt_alleles,
                 alt_offsets, ref_, ref_offsets, pad_char, output_length, to_rc=None, onehot=True):
        self.a = dict(rg=_c(regions, np.int32), sh=_c(shifts, np.int32), goi=_c(geno_offset_idx, np.int64))
        self.batch, self.ploidy = self.a["goi"].shape
        self.go, self.gs, self.ge = _split_offsets(geno_offsets)
        self.gv, self.vs, self.il = _c(geno_v_idxs, np.int32), _c(v_starts, np.int32), _c(ilens, np.int32)
        self.aa, self.ao = _c(alt_alleles, np.uint8), _c(alt_offsets, np.int64)
        self.rf, self.ro = _c(ref_, np.uint8), _c(ref_offsets, np.int64)
        self.rc = _c(to_rc, np.bool_)
        self.pad, self.L, self.onehot = int(pad_char), int(output_length), onehot
        self.out_offsets = np.zeros(self.batch * self.ploidy + 1, np.int64)
        self.ohe = None

    def __call__(self, parallel=True):
        L = lib()
        total = C.c_int64(0)
        par = C.c_int(bool(parallel))
        a = self.a
        ptr = L.gvl_oracle_reconstruct_haplotypes_fused(
            _p(a["rg"]), _p(a["sh"]), _p(a["goi"]), _p(self.gs), _p(self.ge), _p(self.gv), _p(self.vs), _p(self.il),
            _p(self.aa), _p(self.ao), _p(self.rf), _p(self.ro), C.c_uint8(self.pad), _i64(self.L), C.c_void_p(0),
            C.c_void_p(0), _p(self.rc), _i64(self.batch), _i64(self.ploidy), par, _p(self.out_offsets),
            C.byref(total))
        n = int(total.value)
        if self.onehot:
            # the separate pass a seqpro.DNA.ohe user pays (docs/source/index.md:108-119); fresh output each call
            self.ohe = np.empty((n, 4), np.uint8)
            L.gvl_oracle_onehot(C.c_void_p(ptr), _i64(n), _p(self.ohe), par)
        L.gvl_oracle_free(C.c_void_p(ptr))
        return n


def get_reference(regions, out_offsets, reference, ref_offsets, pad_char, parallel=False, to_rc=None):
    """src/ffi/mod.rs:2402-2411 -> src/reference/mod.rs:56-120."""
    rg, oo = _c(regions, np.int32), _c(out_offsets, np.int64)
    rf, ro, rc = _c(reference, np.uint8), _c(ref_offsets, np.int64), _c(to_rc, np.bool_)
    out = np.zeros(int(oo[-1]), np.uint8)
    lib().gvl_oracle_get_reference(_p(rg), _p(oo), _p(rf), _p(ro), C.c_uint8(int(pad_char)), _p(rc),
                                   _i64(rg.shape[0]), _p(out))
    return out


def rc_flat_rows_inplace(data, offsets, to_rc):
    """src/reverse.rs:56-69."""
    oo, rc = _c(offsets, np.int64), _c(to_rc, np.bool_)
    assert data.dtype == np.uint8 and data.flags.c_contiguous
    lib().gvl_oracle_rc_flat_rows_inplace(_p(data), _p(oo), _p(rc), _i64(len(rc)))


def reverse_flat_rows_inplace(data, offsets, to_rc):
    """src/reverse.rs:25-38 for 4-byte elements (f32 tracks, i32 annotations)."""
    oo, rc = _c(offsets, np.int64), _c(to_rc, np.bool_)
    assert data.dtype.itemsize == 4 and data.flags.c_contiguous
    lib().gvl_oracle_reverse_flat_rows_inplace_32(_p(data), _p(oo), _p(rc), _i64(len(rc)))


def onehot(haps, parallel=False):
    """seqpro.DNA.ohe semantics (third-party; PARITY UNPINNED): (...,) u8 -> (..., 4) u8, alphabet ACGT."""
    h = np.ascontiguousarray(haps).view(np.uint8)
    out = np.empty(h.shape + (4,), np.uint8)
    lib().gvl_oracle_onehot(_p(h), _i64(h.size), _p(out), C.c_int(bool(parallel)))
    return out


# ------------------------------------------------------------------ tracks
def intervals_to_tracks(offset_idxs, starts, itv_starts, itv_ends, itv_values, itv_offsets, out, out_offsets,
                        parallel=False):
    """src/ffi/mod.rs:190-201 -> src/intervals.rs:19-126.  Writes `out` in place."""
    oi, st = _c(offset_idxs, np.int64), _c(starts, np.int32)
    s, e, v = _c(itv_starts, np.int32), _c(itv_ends, np.int32), _c(itv_values, np.float32)
    io, oo = _c(itv_offsets, np.int64), _c(out_offsets, np.int64)
    assert out.dtype == np.float32 and out.flags.c_contiguous
    lib().gvl_oracle_intervals_to_tracks(_p(oi), _p(st), _i64(1), _p(s), _p(e), _p(v), _p(io), _p(out), _p(oo),
                                         _i64(len(st)), C.c_int(bool(parallel)))


def shift_and_realign_tracks_sparse(out, out_offsets, regions, shifts, geno_offset_idx, geno_v_idxs, geno_offsets,
                                    v_starts, ilens, tracks, track_offsets, params, keep=None, keep_offsets=None,
                                    strategy_id=0, base_seed=0, parallel=False):
    """src/ffi/mod.rs:2439-2458 -> src/tracks/mod.rs:495-667.  Writes `out` in place."""
    assert out.dtype == np.float32 and out.flags.c_contiguous
    oo, rg, sh = _c(out_offsets, np.int64), _c(regions, np.int32), _c(shifts, np.int32)
    goi = _c(geno_offset_idx, np.int64)
    n_q, ploidy = goi.shape
    go, gs, ge = _split_offsets(geno_offsets)
    gv, vs, il = _c(geno_v_idxs, np.int32), _c(v_starts, np.int32), _c(ilens, np.int32)
    tr, to, pa = _c(tracks, np.float32), _c(track_offsets, np.int64), _c(params, np.float64)
    kp, ko = _c(keep, np.bool_), _c(keep_offsets, np.int64)
    lib().gvl_oracle_shift_and_realign_tracks_sparse(
        _p(out), _p(oo), _p(rg), _p(sh), _p(goi), _p(gv), _p(gs), _p(ge), _p(vs), _p(il), _p(tr), _p(to), _p(pa),
        _p(kp), _p(ko), _i64(strategy_id), C.c_uint64(int(base_seed)), _i64(n_q), _i64(ploidy),
        C.c_int(bool(parallel)))


def intervals_and_realign_track_fused(out, out_offsets, regions, shifts, geno_offset_idx, geno_v_idxs, geno_offsets,
                                      v_starts, ilens, offset_idxs, itv_starts, itv_ends, itv_values, itv_offsets,
                                      track_offsets, params, strategy_id, base_seed, keep=None, keep_offsets=None,
                                      to_rc=None, parallel=False):
    """src/ffi/mod.rs:2553-2672.  Writes `out` in place."""
    assert out.dtype == np.float32 and out.flags.c_contiguous
    oo, rg, sh = _c(out_offsets, np.int64), _c(regions, np.int32), _c(shifts, np.int32)
    goi = _c(geno_offset_idx, np.int64)
    batch, ploidy = goi.shape
    go, gs, ge = _split_offsets(geno_offsets)
    gv, vs, il = _c(geno_v_idxs, np.int32), _c(v_starts, np.int32), _c(ilens, np.int32)
    oi = _c(offset_idxs, np.int64)
    s, e, v = _c(itv_starts, np.int32), _c(itv_ends, np.int32), _c(itv_values, np.float32)
    io, to, pa = _c(itv_offsets, np.int64), _c(track_offsets, np.int64), _c(params, np.float64)
    kp, ko, rc = _c(keep, np.bool_), _c(keep_offsets, np.int64), _c(to_rc, np.bool_)
    lib().gvl_oracle_intervals_and_realign_track_fused(
        _p(out), _p(oo), _p(rg), _p(sh), _p(goi), _p(gv), _p(gs), _p(ge), _p(vs), _p(il), _p(oi), _p(s), _p(e),
        _p(v), _p(io), _p(to), _p(pa), _i64(strategy_id), C.c_uint64(int(base_seed)), _p(kp), _p(ko), _p(rc),
        _i64(batch), _i64(ploidy), C.c_int(bool(parallel)))


# ------------------------------------------------------------------ svar2 two-channel source (decoded level)
def reconstruct_haplotypes_from_svar2(out, out_bounds, regions, shifts, vk_pos, vk_key, vk_off, dense_pos, dense_key,
                                      dense_range, dense_present, dense_present_off, key_ilen, key_alt, key_alt_off,
                                      ref_, ref_offsets, pad_char, parallel=False, filter_exonic=False):
    """src/reconstruct/mod.rs:620-826 with decode_alt replaced by the decoded-key table (see gvl_oracle.c a11)."""
    assert out.dtype == np.uint8 and out.flags.c_contiguous
    ob, rg, sh = _c(out_bounds, np.int64), _c(regions, np.int32), _c(shifts, np.int32)
    batch, ploidy = sh.shape
    a = [_c(vk_pos, np.int32), _c(vk_key, np.int32), _c(vk_off, np.int64), _c(dense_pos, np.int32),
         _c(dense_key, np.int32), _c(dense_range, np.int32), _c(dense_present, np.uint8),
         _c(dense_present_off, np.int64), _c(key_ilen, np.int32), _c(key_alt, np.uint8), _c(key_alt_off, np.int64),
         _c(ref_, np.uint8), _c(ref_offsets, np.int64)]
    lib().gvl_oracle_reconstruct_haplotypes_from_svar2(
        _p(out), _p(ob), _p(rg), _p(sh), *[_p(x) for x in a], C.c_uint8(int(pad_char)), _i64(batch), _i64(ploidy),
        C.c_int(bool(parallel)), C.c_int(bool(filter_exonic)))


def hap_diffs_svar2(regions, ploidy, vk_pos, vk_key, vk_off, dense_pos, dense_key, dense_range, dense_present,
                    dense_present_off, key_ilen, filter_exonic=False):
    """src/svar2/mod.rs:73-146."""
    rg = _c(regions, np.int32)
    batch = rg.shape[0]
    a = [_c(vk_pos, np.int32), _c(vk_key, np.int32), _c(vk_off, np.int64), _c(dense_pos, np.int32),
         _c(dense_key, np.int32), _c(dense_range, np.int32), _c(dense_present, np.uint8),
         _c(dense_present_off, np.int64), _c(key_ilen, np.int32)]
    diffs = np.zeros((batch, ploidy), np.int32)
    lib().gvl_oracle_hap_diffs_svar2(_p(rg), _i64(batch), _i64(ploidy), *[_p(x) for x in a],
                                     C.c_int(bool(filter_exonic)), _p(diffs))
    return diffs


def shift_and_realign_tracks_from_svar2(out, out_offsets, regions, shifts, vk_pos, vk_key, vk_off, dense_pos,
                                        dense_key, dense_range, dense_present, dense_present_off, key_ilen, tracks,
                                        track_offsets, params, strategy_id, base_seed, query_seed=None,
                                        parallel=False):
    """src/tracks/mod.rs:705-856 (decoded-key table instead of decode_alt)."""
    assert out.dtype == np.float32 and out.flags.c_contiguous
    oo, rg, sh = _c(out_offsets, np.int64), _c(regions, np.int32), _c(shifts, np.int32)
    batch, ploidy = sh.shape
    a = [_c(vk_pos, np.int32), _c(vk_key, np.int32), _c(vk_off, np.int64), _c(dense_pos, np.int32),
         _c(dense_key, np.int32), _c(dense_range, np.int32), _c(dense_present, np.uint8),
         _c(dense_present_off, np.int64), _c(key_ilen, np.int32), _c(tracks, np.float32),
         _c(track_offsets, np.int64), _c(params, np.float64)]
    qs = _c(query_seed, np.int64)
    lib().gvl_oracle_shift_and_realign_tracks_from_svar2(
        _p(out), _p(oo), _p(rg), _p(sh), *[_p(x) for x in a], _i64(strategy_id), C.c_uint64(int(base_seed)), _p(qs),
        _i64(batch), _i64(ploidy), C.c_int(bool(parallel)))


def ragged_to_padded(data, offsets, out, itemsize, out_len):
    """src/ragged/mod.rs:7-23 (seqpro-core Ragged::to_padded_into)."""
    d, oo = np.ascontiguousarray(data).view(np.uint8), _c(offsets, np.int64)
    assert out.flags.c_contiguous
    lib().gvl_oracle_ragged_to_padded(_p(d), _p(oo), _i64(len(oo) - 1), _p(out.view(np.uint8)), _i64(itemsize),
                                      _i64(out_len))
