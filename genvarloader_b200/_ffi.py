"""ctypes binding of the C ABI declared in include/gvl_b200.h.

There is no CPU fallback: importing this module without the built CUDA library raises.
Build it with ``python -m genvarloader_b200._build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
import os

LIB_PATH = _PKG / "_lib" / os.environ.get("GVL_LIB_NAME", "libgvl_b200.so")  # (variant builds for A/B profiling)

GVL_OK = 0
MODE_U8, MODE_ONEHOT, MODE_ANNOTATED, MODE_ONEHOT_CF = 0, 1, 2, 3
TRACK_F32, TRACK_BF16, TRACK_F16 = 0, 1, 2  # GVL_TRACK_*: element type of a track output
TRACK_REDUCE_MEAN, TRACK_REDUCE_SUM, TRACK_REDUCE_MAX = 0, 1, 2  # GVL_TRACK_REDUCE_*: reduction of a binned track output
TRACK_BIN_MAX = 4096  # GVL_TRACK_BIN_MAX

c_i64, c_i32, c_u8, c_u64, c_vp = C.c_int64, C.c_int32, C.c_uint8, C.c_uint64, C.c_void_p


class GvlError(RuntimeError):
    """A gvl_* entry returned a non-zero status (the reference would panic / raise,
    src/ffi/mod.rs:45-55)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"[gvl_b200 status {code}] {msg}")
        self.code = code


class SparseTables(C.Structure):
    """gvl_sparse_tables (include/gvl_b200.h)."""

    _fields_ = [
        ("ref", c_vp), ("ref_offsets", c_vp), ("n_contigs", c_i64),
        ("v_starts", c_vp), ("ilens", c_vp), ("alt_alleles", c_vp), ("alt_offsets", c_vp), ("n_variants", c_i64),
        ("geno_v_idxs", c_vp), ("geno_starts", c_vp), ("geno_stops", c_vp), ("n_geno", c_i64),
        ("ref_packed", c_vp), ("alt_packed", c_vp),
    ]


class Intervals(C.Structure):
    """gvl_intervals (include/gvl_b200.h)."""

    _fields_ = [("itv_starts", c_vp), ("itv_ends", c_vp), ("itv_values", c_vp), ("itv_offsets", c_vp),
                ("n_slots", c_i64)]


class Svar2Channels(C.Structure):
    """gvl_svar2_channels (include/gvl_b200.h)."""

    _fields_ = [("vk_pos", c_vp), ("vk_key", c_vp), ("vk_off", c_vp), ("dense_pos", c_vp), ("dense_key", c_vp),
                ("dense_range", c_vp), ("dense_present", c_vp), ("dense_present_off", c_vp), ("vk_stop", c_vp),
                ("row_slot", c_vp), ("query_div", c_i64)]


class DatasetView(C.Structure):
    """gvl_dataset_view (include/gvl_b200.h)."""

    _fields_ = [("full_regions", c_vp), ("n_regions", c_i64), ("n_samples", c_i64), ("ploidy", c_i64), ("rc_neg", c_i32)]


class BatchArgs(C.Structure):
    """gvl_batch_args (include/gvl_b200.h)."""

    _fields_ = [("regions", c_vp), ("shifts", c_vp), ("goi", c_vp), ("to_rc", c_vp), ("to_rc_q", c_vp),
                ("offset_idxs", c_vp), ("base_seed", c_vp), ("starts", c_vp)]


class FixedJob(C.Structure):
    """gvl_fixed_job (include/gvl_b200.h)."""

    _fields_ = [("view", c_vp), ("tab", c_vp), ("svar2", c_vp), ("args", BatchArgs), ("out_offsets", c_vp), ("diffs", c_vp),
                ("track_lengths", c_vp), ("paint_offsets", c_vp), ("itv", c_vp), ("strategy_ids", c_vp), ("params", c_vp),
                ("ploidy", c_i64), ("rows_p", c_i64), ("output_length", c_i64), ("ref_slot", c_i64), ("n_tracks", c_i64),
                ("max_slot_len", c_i64), ("typ_slot_len", c_i64), ("annot_mask", C.c_uint32), ("mode", c_i32), ("realign", c_i32), ("rc_neg", c_i32),
                ("pad_char", c_u8), ("track_dtype", c_i32), ("track_bin", c_i32), ("track_reduce", c_i32)]


def _load() -> C.CDLL:
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension is not built. Run `python -m genvarloader_b200._build` "
            "(needs nvcc). genvarloader_b200 has no CPU fallback."
        )
    lib = C.CDLL(str(LIB_PATH))
    lib.gvl_last_error.restype = C.c_char_p
    lib.gvl_launch_count.restype = c_i64
    lib.gvl_launch_count.argtypes = [C.c_int]
    lib.gvl_packed_reference_words.restype = c_i64
    lib.gvl_packed_reference_words.argtypes = [c_i64]
    lib.gvl_debug_last_launch.argtypes = [c_vp, c_vp, C.c_int]
    lib.gvl_debug_track_tiles.argtypes = [c_vp, c_vp, c_i64, c_vp, c_vp]
    # the per-batch entries of the fixed-length path take plain ints (no per-call ctypes objects)
    lib.gvl_dev_fixed_plan.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]
    lib.gvl_dev_fixed_exec.argtypes = [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.gvl_dev_fixed_stage.argtypes = [c_vp, c_vp, C.c_int, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]
    lib.gvl_dev_fixed_run.argtypes = [c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
    # the track entries (up to 30 arguments: a wrong count must fail here, not reach the device)
    lib.gvl_dev_realign_tracks.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_vp,
                                           c_vp, c_vp, c_i64, c_vp, c_vp, c_u64, c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp,
                                           c_i32, c_vp]
    lib.gvl_dev_realign_tracks_exec.argtypes = [c_vp, c_vp, c_i32, c_vp]
    lib.gvl_dev_realign_tracks_exec_binned.argtypes = [c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]
    lib.gvl_dev_shift_and_realign_tracks.argtypes = [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp,
                                                     c_vp, c_vp, c_vp, c_i64, c_i32, C.c_double, c_u64, c_vp, c_i64, c_vp, c_vp]
    lib.gvl_dev_paint_tracks.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i32, c_vp, c_vp, c_vp, c_i32,
                                         c_vp]
    lib.gvl_dev_paint_tracks_binned.argtypes = [c_vp, c_i64, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_i32, c_vp, c_vp, c_vp,
                                                c_i32, c_i32, c_i32, c_vp]
    lib.gvl_dev_track_intervals.argtypes = [c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_i32,
                                            c_vp]
    lib.gvl_dev_realigned_track_intervals.argtypes = [c_vp, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_i32, c_vp]
    return lib


lib = _load()


def check(code: int) -> None:
    if code != GVL_OK:
        raise GvlError(code, (lib.gvl_last_error() or b"").decode())


def launch_count(reset: bool = False) -> int:
    return int(lib.gvl_launch_count(1 if reset else 0))


# gvl_debug_last_launch: field names in the order of GVL_LAUNCH_* (include/gvl_b200.h), kernel names in the order of GVL_EXEC_*
LAUNCH_FIELDS = ("plan_threads", "plan_static", "exec_kernel", "tile_len", "tiles_per_row", "rec_bound", "trk_plan_threads",
                 "trk_plan_static")
EXEC_KERNELS = ("bytes", "packed_2warp", "packed_unroll4", "packed_unroll2")


def last_launch(handle) -> dict:
    """The launch configuration the last plans and execute of a context chose (gvl_debug_last_launch), by field name;
    `exec_kernel` is given by name."""
    out = (C.c_int64 * len(LAUNCH_FIELDS))()
    check(lib.gvl_debug_last_launch(handle, out, len(LAUNCH_FIELDS)))
    d = dict(zip(LAUNCH_FIELDS, (int(x) for x in out)))
    d["exec_kernel"] = EXEC_KERNELS[d["exec_kernel"]]
    return d


# gvl_debug_track_tiles: fields of one tile entry, flag bits (GVL_TILE_* in include/gvl_b200.h)
TILE_FIELDS = ("track", "row", "h0", "h1", "flags", "m", "cnt")
TILE_RC, TILE_GENERIC, TILE_BIG = 1, 2, 4


def track_tiles(handle):
    """Tile descriptors of the last track execute a context prepared (gvl_debug_track_tiles): ``(tiles, n_tiles,
    tdesc_bytes)`` with ``tiles`` an int32 array (tiles that exist, in grid order) x TILE_FIELDS, ``n_tiles`` the
    descriptors of the call's grid and ``tdesc_bytes`` the bytes allocated for them.  Synchronizes the device."""
    import numpy as np

    n, nb = c_i64(0), c_i64(0)
    check(lib.gvl_debug_track_tiles(handle, None, 0, C.byref(n), C.byref(nb)))
    out = np.empty((max(n.value, 1), len(TILE_FIELDS)), np.int32)
    check(lib.gvl_debug_track_tiles(handle, out.ctypes.data, n.value, C.byref(n), C.byref(nb)))
    return out[: n.value][out[: n.value, 1] >= 0], int(n.value), int(nb.value)


def ptr(x) -> C.c_void_p:
    """Pointer of a torch tensor / numpy array / None."""
    if x is None:
        return c_vp(0)
    if hasattr(x, "data_ptr"):
        return c_vp(x.data_ptr())
    return c_vp(x.ctypes.data)


class Ctx:
    """Owner of a gvl_ctx (device workspace, host-layer upload cache)."""

    def __init__(self, device: int = 0):
        self._h = c_vp(0)
        check(lib.gvl_ctx_create(C.c_int(int(device)), C.byref(self._h)))
        self.device = int(device)

    @property
    def handle(self) -> C.c_void_p:
        if not self._h:
            raise GvlError(4, "context was destroyed")
        return self._h

    def close(self) -> None:
        if self._h:
            lib.gvl_ctx_destroy(self._h)
            self._h = c_vp(0)

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def check(self, stream: int = 0) -> None:
        check(lib.gvl_ctx_check(self.handle, c_vp(stream)))
