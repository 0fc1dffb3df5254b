"""Fixed-length batch pipeline: the GPU-side analogue of the reference's buffered / double-buffered loaders
(`Dataset.to_dataloader(mode=...)`, python/genvarloader/_dataset/_impl.py:1963-2072, `_double_buffered_loader.py`).

A fixed-length, deterministic batch needs nothing from the host but its flat dataset indices (and the jitter draws):
`gvl_dev_batch_prep` derives the regions, genotype slots, strand masks, interval slots and the fill seeds on the device,
then plan -> execute (-> tracks) run as in `Dataset.__getitem__`.  Two users:

  * `FixedPipeline.run_eager`  -- one batch on the current stream: the fast path of `Dataset.__getitem__` (one small
                                  H2D copy, no per-call pinned allocation).
  * `FixedPipeline` rings      -- the loader reads AHEAD: `ring` consecutive batches are reconstructed as ONE device
                                  call (rows of all batches in one plan launch and one execute launch, so every launch
                                  fills the GPU for hundreds of microseconds instead of ~10), into two buffer halves.
                                  Each half owns one CUDA graph (prep -> plan -> execute [-> tracks]) replayed on the
                                  half's own stream: while the consumer reads the batches of one half, the other is being
                                  produced, and the plan of one call overlaps the execute of the other half's call.  Rows
                                  are independent (src/reconstruct/mod.rs:374-422), so batch i of a ring is simply rows
                                  [i*b*p, (i+1)*b*p) of the ring's output.  `PipelinedLoader` drives it.

Batches of a ring are views into the ring's output buffers (zero-copy, like `copy=False` of the reference's
double-buffered mode: valid until the ring is refilled); `copy=True` hands out clones.
"""
from __future__ import annotations

import ctypes as C
import gc
import os

import numpy as np
import torch

from . import _ffi
from ._dataset import _as_rng, _batch_tail, epoch_order
from ._engine import MODES, Engine, _raw_stream, _stream, track_dtype_code
from ._ffi import BatchArgs, DatasetView, FixedJob, c_i64, c_u8, c_u64, c_vp, check, lib, ptr
from ._types import AnnotatedHaps


class PinnedArray:
    """Page-locked host array (gvl_host_alloc) viewed as numpy."""

    def __init__(self, shape, dtype):
        self.nbytes = int(np.prod(shape, dtype=np.int64)) * np.dtype(dtype).itemsize
        self._p = c_vp(0)
        check(lib.gvl_host_alloc(c_i64(max(self.nbytes, 16)), C.byref(self._p)))
        raw = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(max(self.nbytes, 16),))
        self.array = raw[: self.nbytes].view(dtype).reshape(shape)
        self.ptr = int(self._p.value)

    def close(self):
        if self._p:
            lib.gvl_host_free(self._p)
            self._p = c_vp(0)

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


class _Spec:
    """What a dataset state asks of a fixed-length batch (resolved once per pipeline)."""

    def __init__(self, ds):
        self.L = int(ds.output_length)
        self.p = int(ds.ploidy)
        self.want_seqs = ds.sequence_type is not None
        self.is_ref = ds.sequence_type == "reference"
        self.annotated = ds.sequence_type == "annotated"
        self.names = list(ds.active_tracks)
        self.t = len(self.names)
        self.realign = ds._realigns
        self.rows_p = 1 if (self.is_ref or not self.want_seqs) else self.p
        self.rc_neg = bool(ds.rc_neg)
        self.jitter = int(ds.jitter)
        if self.annotated:
            self.mode = "annotated"
        elif ds.encoding == "bytes":
            self.mode = "haplotypes"
        else:
            self.mode = ds.encoding  # "onehot" | "onehot_cf"
        self.annot_mask = 0
        for i, n in enumerate(self.names):
            if ds.track_kinds[n] == "annot":
                self.annot_mask |= 1 << i
        self.fill_ids, self.fill_params = ds._fills(self.names)
        self.track_dtype = ds.track_dtype


def supports(ds) -> str | None:
    """None when `ds` can use the fixed pipeline, else the reason it cannot."""
    if not isinstance(ds.output_length, (int, np.integer)) or isinstance(ds.output_length, bool):
        return "output_length is not fixed"
    if ds.splice_rows is not None:
        return "spliced output"
    if ds.sequence_type in ("variants", "variant-windows"):
        return "the variants output is ragged by nature"
    if ds.var_filter is not None:
        return "var_filter needs per-batch keep masks"
    if not ds.deterministic and ds.sequence_type in ("haplotypes", "annotated"):
        return "random shifts (deterministic=False) are drawn on the host from the batch's diffs"
    if ds.sequence_type is None and not ds.active_tracks:
        return "nothing to read"
    if ds.track_output == "intervals" and ds.active_tracks:
        return "track intervals are ragged by nature"
    if len(ds.active_tracks) > 8:
        return "more than 8 tracks"
    return None


class _Scratch:
    """Device buffers holding the prepared arguments of ONE batch in flight."""

    def __init__(self, spec: _Spec, b: int, dev, n_sub: int = 1):
        rp, t = spec.rows_p, spec.t
        i32, i64, u8 = torch.int32, torch.int64, torch.uint8
        self.regions = torch.empty((b, 3), dtype=i32, device=dev)
        self.starts = torch.empty(b, dtype=i32, device=dev)
        self.shifts = torch.empty((b, rp), dtype=i32, device=dev)
        self.goi = torch.empty((b, rp), dtype=i64, device=dev)
        self.to_rc = torch.empty(b * rp, dtype=u8, device=dev)
        self.to_rc_q = torch.empty(b, dtype=u8, device=dev)
        self.offset_idxs = torch.empty((max(t, 1), b), dtype=i64, device=dev)
        self.base_seed = torch.zeros(max(n_sub, 1), dtype=i64, device=dev)  # one fill seed per logical batch
        self.out_offsets = torch.empty(b * rp + 1, dtype=i64, device=dev)
        self.diffs = torch.empty((b, rp), dtype=i32, device=dev) if spec.realign else None
        self.track_lengths = torch.empty(b, dtype=i32, device=dev) if spec.realign else None
        self.args = BatchArgs(ptr(self.regions), ptr(self.shifts), ptr(self.goi), ptr(self.to_rc), ptr(self.to_rc_q),
                              ptr(self.offset_idxs) if t else c_vp(0), ptr(self.base_seed), ptr(self.starts))


class _Out:
    """Output buffers of one batch + the objects handed to the user."""

    def __init__(self, spec: _Spec, b: int, dev):
        L, p, rp, t = spec.L, spec.p, spec.rows_p, spec.t
        self.seq = self.av = self.ap = self.trk = None
        if spec.want_seqs:
            mult = 4 if spec.mode in ("onehot", "onehot_cf") else 1
            self.seq = torch.empty(b * rp * L * mult, dtype=torch.uint8, device=dev)
            if spec.annotated:
                self.av = torch.empty(b * rp * L, dtype=torch.int32, device=dev)
                self.ap = torch.empty(b * rp * L, dtype=torch.int32, device=dev)
        if t:
            self.trk = torch.empty(b * t * (p if spec.realign else 1) * L, dtype=spec.track_dtype, device=dev)
        self.spec, self.b = spec, b

    def result(self, lo: int = 0, n: int | None = None, clone: bool = False):
        """Queries [lo, lo + n) as `Dataset.__getitem__` returns them for array indices: dense tensors, `(seqs, tracks)`
        when both are active."""
        sp, b = self.spec, self.b
        L, p, t = sp.L, sp.p, sp.t
        n = b - lo if n is None else n
        if lo == 0 and n == b and not clone:
            f = lambda x: x
        else:
            f = (lambda x: x[lo: lo + n].clone()) if clone else (lambda x: x[lo: lo + n])
        res = []
        if sp.want_seqs:
            lead = (b,) if sp.is_ref else (b, p)
            if sp.mode == "onehot":
                s = f(self.seq.view(*lead, L, 4))
            elif sp.mode == "onehot_cf":
                s = f(self.seq.view(*lead, 4, L))
            else:
                s = f(self.seq.view(*lead, L))
            if sp.annotated:
                s = AnnotatedHaps(s, f(self.av.view(*lead, L)), f(self.ap.view(*lead, L)))
            res.append(s)
        if t:
            res.append(f(self.trk.view(b, t, p, L) if sp.realign else self.trk.view(b, t, L)))
        return res[0] if len(res) == 1 else tuple(res)


class FixedPipeline:
    """See the module docstring.  `batch_size` = queries per logical batch, `ring` = batches per device call (0: eager
    single batches only), `halves` = ring buffers produced alternately."""

    fused = True  # a device call of a ring half is one graph on one stream (bench.py reads this)

    def __init__(self, ds, batch_size: int, ring: int = 0, halves: int = 2, graph: bool = True):
        why = supports(ds)
        if why is not None:
            raise ValueError(f"the fixed-length pipeline does not apply: {why}")
        self.ds, self.b = ds, int(batch_size)
        self.eng: Engine = ds.engine
        self.dev = self.eng.device
        self.spec = sp = _Spec(ds)
        self.view = self.eng.dataset_view(ds.full_regions, len(ds.sample_names), ds.ploidy, ds.rc_neg)
        self.ref_slot = self.eng.empty_slot if (sp.is_ref or not sp.want_seqs) else -1
        self.ring, self.n_halves = int(ring), int(halves)
        self.use_graph = bool(graph) and os.environ.get("GVL_PIPE_GRAPH", "1") != "0"  # (0: eager launches, for tool runs)
        b, dev = self.b, self.dev
        with torch.cuda.device(dev):
            # eager path (Dataset.__getitem__): one scratch set, one pinned index buffer
            self._keep = []
            self._paint_off = torch.arange(max(self.ring, 1) * b + 1, dtype=torch.int64, device=dev) * sp.L
            self._scr0 = _Scratch(sp, b, dev)
            self._scr0.job = self._make_job(self._scr0)
            self._idx0 = torch.zeros(b + (b + 1) // 2, dtype=torch.int64, device=dev)
            self._jit0 = self._idx0[b:].view(torch.int32)
            self._ctx_handle, self._job0_adr = self.eng.ctx.handle, C.addressof(self._scr0.job)
            self._simple_shape = None
            if sp.want_seqs and not sp.annotated and not sp.t:
                lead = () if sp.is_ref else (sp.p,)
                self._simple_shape = {"onehot": (*lead, sp.L, 4), "onehot_cf": (*lead, 4, sp.L)}.get(sp.mode, (*lead, sp.L))
            self._idx0_ptr, self._jit0_ptr = self._idx0.data_ptr(), self._jit0.data_ptr()
        self.halves = []
        if self.ring > 0:
            self._build_rings()

    def _cap(self, n_queries: int) -> int:
        """Plan workspace (records) for `n_queries`: what gvl_dev_fixed_plan derives from the job."""
        return n_queries * self.spec.rows_p * max(self.eng.max_slot_len, 1) if self.ref_slot < 0 else 0

    def _make_job(self, scr: _Scratch) -> FixedJob:
        """gvl_fixed_job over one scratch set: everything `gvl_dev_fixed_plan/_exec` need that does not change per batch.
        The host-side structs it points to are kept alive on `self._keep`."""
        sp, eng = self.spec, self.eng
        keep = self._keep
        keep.append(self.view)
        sv = None
        if eng.svar2 is not None:
            sv = eng.svar2_channels(None)
            keep.append(sv)
        itv = sid = par = None
        if sp.t:
            itv, sid, par = eng.track_descs(sp.names, sp.fill_ids, sp.fill_params)
            keep.extend([itv, sid, par])
        adr = lambda x: c_vp(C.addressof(x)) if x is not None else c_vp(0)
        mode = MODES[sp.mode] if sp.want_seqs else -1
        return FixedJob(adr(self.view), adr(eng.tab), adr(sv), scr.args, ptr(scr.out_offsets), ptr(scr.diffs), ptr(scr.track_lengths),
                        ptr(self._paint_off) if (sp.t and not sp.realign) else c_vp(0), adr(itv), adr(sid), adr(par),
                        sp.p, sp.rows_p, sp.L, self.ref_slot, sp.t, max(eng.max_slot_len, 1), int(getattr(eng, "typ_slot_len", 0)), sp.annot_mask, mode,
                        1 if sp.realign else 0, 1 if sp.rc_neg else 0, eng.pad_char, track_dtype_code(sp.track_dtype))

    # ------------------------------------------------------------------ one device call over n queries
    # Stage P ("plan"): batch prep + variant plan (+ track plan / tile prep).  Stage E ("execute"): the bandwidth-bound
    # kernels.  The eager path runs both on the current stream (gvl_dev_fixed_run); a ring half runs both on its own stream
    # (_stages_fused), so the plan of one half's call (latency-bound, few CTAs) overlaps the execute of the other's.
    def _stage_plan(self, eng: Engine, scr: _Scratch, idx_dev, jit_dev, n: int, sub_batch: int = 0):
        check(lib.gvl_dev_fixed_plan(eng.ctx.handle, C.addressof(scr.job), idx_dev.data_ptr(),
                                     jit_dev.data_ptr() if jit_dev is not None else None, n, sub_batch, _stream()))

    def _stage_exec(self, eng: Engine, scr: _Scratch, out: _Out, n: int, sub_batch: int = 0):
        dp = lambda x: x.data_ptr() if x is not None else None
        check(lib.gvl_dev_fixed_exec(eng.ctx.handle, C.addressof(scr.job), n, dp(out.seq), dp(out.av), dp(out.ap), dp(out.trk),
                                     _stream()))

    def run_eager(self, ds_idx: np.ndarray, jitter: np.ndarray | None):
        """One batch (len(ds_idx) <= batch_size) on the current stream; returns freshly allocated outputs.  Host side:
        the output allocation and ONE library call (gvl_dev_fixed_run: staged index upload + prep + plan + execute)."""
        n = len(ds_idx)
        if n > self.b:
            raise ValueError("batch larger than the pipeline's batch size")
        dev = self.dev
        guard = torch._C._cuda_getDevice() != dev.index
        if guard:
            prev = torch.cuda.current_device()
            torch.cuda.set_device(dev)
        try:
            shp = self._simple_shape
            if shp is not None:  # sequences only (bytes / one-hot): allocate the result in its final shape, no wrapper objects
                seq = torch.empty((n, *shp), dtype=torch.uint8, device=dev)
                rc = lib.gvl_dev_fixed_run(self._ctx_handle, self._job0_adr, ds_idx.__array_interface__["data"][0],
                                           jitter.__array_interface__["data"][0] if jitter is not None else None, n,
                                           self._idx0_ptr, self._jit0_ptr, seq.data_ptr(), None, None, None, _raw_stream(dev.index))
                if rc:
                    check(rc)
                return seq
            out = _Out(self.spec, n, dev)
            seq, av, ap, trk = out.seq, out.av, out.ap, out.trk
            rc = lib.gvl_dev_fixed_run(self._ctx_handle, self._job0_adr, ds_idx.ctypes.data,
                                       jitter.ctypes.data if jitter is not None else None, n, self._idx0_ptr, self._jit0_ptr,
                                       seq.data_ptr() if seq is not None else None, av.data_ptr() if av is not None else None,
                                       ap.data_ptr() if ap is not None else None, trk.data_ptr() if trk is not None else None,
                                       _raw_stream(dev.index))
            if rc:
                check(rc)
        finally:
            if guard:
                torch.cuda.set_device(prev)
        return out.result()

    # ------------------------------------------------------------------ rings
    def _build_rings(self):
        sp, b, dev, K = self.spec, self.b, self.dev, self.ring
        n = K * b
        with torch.cuda.device(dev):
            self.s_plan, self.s_exec = torch.cuda.Stream(dev), torch.cuda.Stream(dev)  # the streams of even / odd halves
            for h in range(self.n_halves):
                H = type("Half", (), {})()
                H.eng = self.eng.fork()
                H.scr = _Scratch(sp, n, dev, n_sub=K)
                H.scr.job = self._make_job(H.scr)
                H.out = _Out(sp, n, dev)
                H.pin = PinnedArray((n + (n + 1) // 2,), np.int64)  # [ds_idx i64[n]][jitter i32[n]]
                H.pin_jit = H.pin.array[n:].view(np.int32)
                H.idx = torch.zeros(n + (n + 1) // 2, dtype=torch.int64, device=dev)
                H.jit = H.idx[n:].view(torch.int32)
                H.done, H.uploaded = torch.cuda.Event(), torch.cuda.Event()
                H.free = None
                H.g_plan = None
                self.halves.append(H)
            jit = (lambda H: H.jit if sp.jitter else None)
            # warm once outside capture: workspace growth allocates
            _ffi.launch_count(reset=True)
            for H in self.halves:
                with torch.cuda.stream(self.s_plan):
                    self._stage_plan(H.eng, H.scr, H.idx, jit(H), n, sub_batch=b)
                    self._stage_exec(H.eng, H.scr, H.out, n, sub_batch=b)
            self.launches_per_ring = _ffi.launch_count() // max(len(self.halves), 1)
            torch.cuda.synchronize(dev)
            for H in self.halves:
                H.eng.check()
            # ONE graph per half -- prep -> plan -> execute -- replayed on the half's own stream, so a device call is one graph
            # launch and the plan of the next call (other half, other stream) still overlaps this call's execute.
            for i, H in enumerate(self.halves):
                H.stream = (self.s_plan, self.s_exec)[i % 2]
                H.side = torch.cuda.Stream(dev, priority=-1)  # (its small kernels go first when SM slots free up)
            if self.use_graph:
                # No garbage collection while a graph is being captured: collecting a dead context or pinned buffer of
                # an earlier dataset frees device / host memory, which a capture does not permit (the capture fails).
                # Collect first, then keep the collector off until the captures are done.
                gc.collect()
                gc_was_on = gc.isenabled()
                gc.disable()
                try:
                    for H in self.halves:
                        H.g_plan = torch.cuda.CUDAGraph()
                        with torch.cuda.graph(H.g_plan, stream=H.stream):
                            self._stages_fused(H, jit(H), n, b)
                finally:
                    if gc_was_on:
                        gc.enable()

    def _stages_fused(self, H, jit_dev, n: int, b: int):
        """One device call of half H on the current stream (= H.stream).  With realigned tracks the call forks: the track
        plan (variant walk, tile scan, per-tile searches: ~120 us of small latency-bound kernels for a 20-batch ring) runs
        on a side stream next to the bandwidth-bound haplotype execute, and joins before the track execute.  Inside a
        capture the fork / join become graph edges."""
        sp = self.spec
        if not (sp.realign and sp.want_seqs):
            self._stage_plan(H.eng, H.scr, H.idx, jit_dev, n, sub_batch=b)
            self._stage_exec(H.eng, H.scr, H.out, n, sub_batch=b)
            return
        h, job = H.eng.ctx.handle, C.addressof(H.scr.job)
        idx, jit = H.idx.data_ptr(), (jit_dev.data_ptr() if jit_dev is not None else None)
        o = H.out
        dp = lambda x: x.data_ptr() if x is not None else None
        args = (idx, jit, n, b, dp(o.seq), dp(o.av), dp(o.ap), dp(o.trk))
        main = torch.cuda.current_stream(self.dev)
        check(lib.gvl_dev_fixed_stage(h, job, 1, *args, _stream()))  # batch prep + haplotype plan
        fork, join = torch.cuda.Event(), torch.cuda.Event()
        fork.record(main)
        H.side.wait_event(fork)
        with torch.cuda.stream(H.side):
            check(lib.gvl_dev_fixed_stage(h, job, 2, *args, _stream()))  # track plan
            join.record(H.side)
        check(lib.gvl_dev_fixed_stage(h, job, 3, *args, _stream()))  # haplotype execute
        main.wait_event(join)
        check(lib.gvl_dev_fixed_stage(h, job, 4, *args, _stream()))  # track execute

    def wait_all(self, event):
        """Every stream of the pipeline waits for `event` (bench: one start event for a timed block)."""
        self.s_plan.wait_event(event)
        self.s_exec.wait_event(event)

    def submit(self, h: int, ds_idx=None, jitter=None):
        """Produce half `h`.  `ds_idx`: int64 (ring * b) indices -- a numpy array (staged through pinned memory, one H2D
        copy), a device tensor (device-to-device copy) or None (replay with the indices already in place); `jitter`
        likewise (int32)."""
        H = self.halves[h]
        n = self.ring * self.b
        sp = self.spec
        s_in = H.stream  # the stream the indices arrive on and the device call runs on
        with torch.cuda.device(self.dev):
            if isinstance(ds_idx, np.ndarray):
                H.uploaded.synchronize()  # the previous copy out of the pinned buffer has finished
                H.pin.array[:n] = ds_idx
                if jitter is not None:
                    H.pin_jit[:n] = jitter
                check(lib.gvl_dev_upload(self.eng.ctx.handle, ptr(H.idx), c_vp(H.pin.ptr), c_i64(H.pin.nbytes),
                                         c_vp(s_in.cuda_stream)))
                H.uploaded.record(s_in)
            elif ds_idx is not None:
                with torch.cuda.stream(s_in):
                    if ds_idx.numel() == H.idx.numel():  # already in the staging layout [ds_idx][jitter]: one copy
                        H.idx.copy_(ds_idx, non_blocking=True)
                    else:
                        H.idx[:n].copy_(ds_idx, non_blocking=True)
                        if jitter is not None:
                            H.jit[:n].copy_(jitter, non_blocking=True)
            if H.free is not None:
                s_in.wait_event(H.free)  # the consumer has let go of this half's output buffers
            with torch.cuda.stream(s_in):
                if H.g_plan is not None:
                    H.g_plan.replay()
                else:
                    self._stages_fused(H, H.jit if sp.jitter else None, n, self.b)
            H.done.record(s_in)

    def acquire(self, h: int) -> _Out:
        """Make the current stream wait for half `h`; returns its `_Out` (batch i = queries [i*b, (i+1)*b))."""
        H = self.halves[h]
        torch.cuda.current_stream(self.dev).wait_event(H.done)
        return H.out

    def release(self, h: int):
        """The consumer is done with half `h` (everything it enqueued so far on the current stream)."""
        H = self.halves[h]
        if H.free is None:
            H.free = torch.cuda.Event()
        H.free.record(torch.cuda.current_stream(self.dev))

    def check(self):
        for H in self.halves:
            H.eng.check()
        self.eng.check()


class PipelinedLoader:
    """Re-iterable loader over a `Dataset` backed by a `FixedPipeline` (see `Dataset.to_dataloader(mode=...)`)."""

    def __init__(self, ds, batch_size, shuffle, sampler, drop_last, generator, return_indices, transform, copy, ring, to_host=False):
        if to_host and ds.active_tracks and ds.track_dtype == torch.bfloat16:
            raise ValueError("to_host=True delivers numpy arrays and numpy has no bfloat16: read bfloat16 tracks on the device, "
                             "or use with_track_dtype(torch.float16) / torch.float32 for host delivery")
        self.ds, self.batch_size, self.shuffle, self.sampler = ds, int(batch_size), shuffle, sampler
        self.drop_last, self.return_indices, self.transform, self.copy = drop_last, return_indices, transform, copy
        self._rng = _as_rng(generator)
        n_batches = len(self)
        if not ring:  # ~256 MiB of output per half, at least one batch, no more than half an epoch
            per_batch = self.batch_size * max(ds.ploidy, 1) * int(ds.output_length) * (4 + 4 * len(ds.active_tracks))
            ring = max(1, min((256 << 20) // max(per_batch, 1), 64))
        ring = max(1, min(int(ring), -(-n_batches // 2)))
        self.pipe = FixedPipeline(ds, self.batch_size, ring=ring)
        self._views = {}
        # host delivery (`to_host=True`): every ring is copied into a pinned host twin of its half on a copy stream while the other
        # half is produced; batches are numpy views of that buffer (valid until the half comes around again)
        self.to_host = bool(to_host)
        self._host = {}
        self._copy_stream = torch.cuda.Stream(self.pipe.dev) if self.to_host else None

    def __len__(self) -> int:
        n = len(self.sampler) if self.sampler is not None else len(self.ds)
        return n // self.batch_size if self.drop_last else -(-n // self.batch_size)

    def __iter__(self):
        ds, pipe, b, K = self.ds, self.pipe, self.batch_size, self.pipe.ring
        order = epoch_order(ds, self.sampler, self.shuffle, self._rng)
        n_batches = len(self)
        if self.drop_last:
            order = order[: n_batches * b]
        n_s, S_full = ds.n_samples, len(ds.sample_names)
        r_map, s_map = ds._r_idx, ds._s_idx
        n_rings = -(-n_batches // K)
        jit = ds.jitter

        def fill(ring_i):
            chunk = order[ring_i * K * b: (ring_i + 1) * K * b]
            r, s = chunk // n_s, chunk % n_s
            flat = np.zeros(K * b, np.int64)
            flat[: len(chunk)] = r_map[r] * S_full + s_map[s]
            j = None
            if jit:
                j = np.zeros(K * b, np.int32)
                for lo in range(0, len(chunk), b):  # one draw per batch, like the reference (_query.py:165-171)
                    m = min(b, len(chunk) - lo)
                    j[lo: lo + m] = ds.rng.integers(-jit, jit + 1, size=m, dtype=np.int32)
            return flat, j, chunk

        chunks = {}
        for ring_i in range(min(pipe.n_halves, n_rings)):
            flat, j, chunks[ring_i] = fill(ring_i)
            pipe.submit(ring_i % pipe.n_halves, flat, j)
        plain = not self.return_indices and self.transform is None
        if self.to_host:
            yield from self._iter_host(pipe, chunks, fill, n_rings, K, b, n_s)
            return
        for ring_i in range(n_rings):
            h = ring_i % pipe.n_halves
            out = pipe.acquire(h)
            chunk = chunks.pop(ring_i)
            if plain and not self.copy and len(chunk) == K * b:
                # zero-copy views of a full ring are the same tensors every time the half comes around: built once
                views = self._views.get(h)
                if views is None:
                    views = self._views[h] = [out.result(lo, b) for lo in range(0, K * b, b)]
                yield from views
                pipe.release(h)
                nxt = ring_i + pipe.n_halves
                if nxt < n_rings:
                    flat, j, chunks[nxt] = fill(nxt)
                    pipe.submit(h, flat, j)
                continue
            for lo in range(0, len(chunk), b):
                c = chunk[lo: lo + b]
                yield _batch_tail(out.result(lo, len(c), clone=self.copy), (c // n_s, c % n_s) if self.return_indices else None,
                                  self.transform)
            pipe.release(h)
            nxt = ring_i + pipe.n_halves
            if nxt < n_rings:
                flat, j, chunks[nxt] = fill(nxt)
                pipe.submit(h, flat, j)

    # ------------------------------------------------------------------ host delivery
    def _host_half(self, h: int):
        """Pinned host twin of half h's output buffers (+ the event of its last copy)."""
        ent = self._host.get(h)
        if ent is None:
            out = self.pipe.halves[h].out
            bufs = {k: torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for k in ("seq", "av", "ap", "trk")
                    if (t := getattr(out, k)) is not None}
            twin = _Out.__new__(_Out)
            twin.spec, twin.b = out.spec, out.b
            twin.seq, twin.av, twin.ap, twin.trk = (bufs.get(k) for k in ("seq", "av", "ap", "trk"))
            ent = self._host[h] = (twin, torch.cuda.Event(), bufs)
        return ent

    def _iter_host(self, pipe, chunks, fill, n_rings, K, b, n_s):
        cs = self._copy_stream

        def start_copy(h):  # device half -> pinned twin, on the copy stream, as soon as the half is produced
            H = pipe.halves[h]
            twin, ev, bufs = self._host_half(h)
            cs.wait_event(H.done)
            with torch.cuda.stream(cs):
                for k, dst in bufs.items():
                    dst.copy_(getattr(H.out, k), non_blocking=True)
            ev.record(cs)
            H.free = ev  # the device half may be refilled once its copy has left

        for ring_i in range(min(pipe.n_halves, n_rings)):
            start_copy(ring_i % pipe.n_halves)
        for ring_i in range(n_rings):
            h = ring_i % pipe.n_halves
            twin, ev, _ = self._host_half(h)
            ev.synchronize()  # the ring is in host memory
            chunk = chunks.pop(ring_i)
            for lo in range(0, len(chunk), b):
                c = chunk[lo: lo + b]
                batch = twin.result(lo, len(c), clone=self.copy)
                batch = tuple(x.numpy() if isinstance(x, torch.Tensor) else x for x in (batch if isinstance(batch, tuple) else (batch,)))
                yield _batch_tail(batch, (c // n_s, c % n_s) if self.return_indices else None, self.transform)
            nxt = ring_i + pipe.n_halves
            if nxt < n_rings:  # (the consumer is past every batch of this half: its pinned twin may be overwritten)
                flat, j, chunks[nxt] = fill(nxt)
                pipe.submit(h, flat, j)
                start_copy(h)
