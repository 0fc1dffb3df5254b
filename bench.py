#!/usr/bin/env python
"""bench.py -- haplotype bp/s (one-hot) of the B200-native path, with roofline, CPU baseline, API and e2e legs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg3|cfg2|cfg1|cfg4|...]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over ONE batch of synthetic (region, sample) pairs: device-side batch prep,
plan (variant state machine -> segment table) and execute (fused copy / ALT scatter / pad / RC / one-hot), with every
input already resident in HBM.  The product path is the read-ahead loader (`genvarloader_b200._pipeline`): `ring`
consecutive batches are reconstructed by one device call (one CUDA graph: prep -> plan -> execute), two ring halves alternate
on two streams -- the timed region replays exactly that machinery for K batches.  Default workload = BASELINE.json configs[2] / the north-star target:
524,288-bp indel-bearing windows, 32 haplotypes per batch, 512 regions on a 300 Mb contig (packed reference 150 MB >
126 MB L2).  `--workload cfg2` = configs[1].

Printed JSON line (rank 0): the driver's contract + `roofline`, `cpu_baseline`, `api`, `e2e`, `clocks`, `gpu_launches`
(+ `tracks` on cfg3: the same batches with 2 realigned float tracks).  See DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

N_CHAR = ord("N")
ALG_BYTES_PER_BP = 5.0        # 1 reference byte read + 4 one-hot bytes written (SURVEY.md 8d)
ALG_BYTES_PER_VARIANT = 29.0  # 4 v_idx + 4 pos + 4 ilen + 16 alt_offsets + >=1 ALT
ALG_BYTES_PER_ROW = 56.0


# ----------------------------------------------------------------------------------------------
# workloads (SURVEY.md 8d / BASELINE.json configs)
# ----------------------------------------------------------------------------------------------
WORKLOADS = {
    "cfg1": dict(desc="configs[0]: 1 Mb contig, 8 diploid samples, ~1 variant/kb, 1,000 regions x 16,384 bp, 64 haplotypes/batch",
                 contig_len=1_000_000, n_samples=8, n_regions=1000, window=16_384, pairs=32, vkb=1.0),
    "cfg2": dict(desc="configs[1]: 50 Mb contig, 2,504 diploid samples, ~1 variant/kb/haplotype (~0.55 M variant table) in an "
                      "svar2 two-channel store (half of the variants dense + presence bits), 64 regions x 131,072 bp, "
                      "64 haplotypes/batch",
                 contig_len=50_000_000, n_samples=2504, n_regions=64, window=131_072, pairs=32, vkb=1.0, source="svar2"),
    "cfg3": dict(desc="configs[2] (haplotype part): 524,288-bp indel-bearing windows (20% indels), 512 regions on a 300 Mb contig, "
                      "32 haplotypes/batch, jitter 128, 50% negative strand (reverse-complemented)",
                 contig_len=300_000_000, n_samples=4, n_regions=512, window=524_288, pairs=16, vkb=1.0, neg=0.5, jitter=128,
                 tracks_avail=2),
    "cfg3t": dict(desc="configs[2]: cfg3 PLUS 2 realigned float tracks per haplotype (intervals with a mean run of 50 bp; fills "
                       "Repeat5p and Interpolate(1))",
                  contig_len=300_000_000, n_samples=4, n_regions=512, window=524_288, pairs=16, vkb=1.0, neg=0.5, jitter=128,
                  tracks_avail=2, tracks=2),
    "cfg2d": dict(desc="configs[4] dense cell: 131,072-bp windows, 64 haplotypes/batch, ~10 variants/kb/haplotype",
                  contig_len=50_000_000, n_samples=16, n_regions=256, window=131_072, pairs=32, vkb=10.0, neg=0.5),
    "cfg4": dict(desc="configs[3] (one-hot instead of annotated): 6,144-bp windows, 4,096 haplotypes/batch",
                 contig_len=5_000_000, n_samples=64, n_regions=512, window=6_144, pairs=2048, vkb=1.0),
}


# (profiles/sweep_cfg5_r2.py: one extra workload described by the environment, e.g. a cell of the configs[4] sweep)
if os.environ.get("GVL_BENCH_CUSTOM"):
    WORKLOADS["custom"] = json.loads(os.environ["GVL_BENCH_CUSTOM"])


def build_workload(name: str, seed: int):
    from genvarloader_b200 import synth

    w = WORKLOADS[name]
    j = w.get("jitter", 0)
    d = synth.make_dataset(seed, w["contig_len"], w["n_samples"], w["n_regions"], w["window"] + 2 * j, w["vkb"],
                           max_jitter=j, neg_strand_frac=w.get("neg", 0.0), straddle_ends=False,
                           n_tracks=w.get("tracks_avail", w.get("tracks", 0)), fast_tracks=True)
    d.svar2 = synth.to_svar2_dataset(d, dense_frac=0.5, seed=seed) if w.get("source") == "svar2" else None
    return w, d


def draw_indices(d, n: int, seed: int, rank: int = 0, world: int = 1) -> np.ndarray:
    """`n` flat dataset indices (r * n_samples + s) of this rank: every GLOBAL batch is drawn from one shared seed and cut
    into contiguous per-rank blocks (genvarloader_b200._dist.shard_bounds) -- weak scaling, no communication."""
    from genvarloader_b200._dist import shard_bounds

    rng = np.random.default_rng(seed)
    r = rng.integers(0, d.n_regions, n * world)
    s = rng.integers(0, d.n_samples, n * world)
    lo, hi = shard_bounds(n * world, rank, world)
    return (r[lo:hi] * d.n_samples + s[lo:hi]).astype(np.int64)


def host_batches(d, w, n_batches: int, seed: int, rank: int = 0, world: int = 1):
    """Host-side (reference-shaped) arguments of distinct batches, built like the reference's Python prep."""
    from genvarloader_b200 import synth

    rng = np.random.default_rng(seed + 17)
    out = []
    for i in range(n_batches):
        idx = draw_indices(d, w["pairs"], seed + 1000 + i, rank, world)
        regions, goi, to_rc, ds_idx = synth.batch_args(d, idx // d.n_samples, idx % d.n_samples, rng, jitter=w.get("jitter", 0))
        regions[:, 2] = regions[:, 1] + w["window"]  # (the fused entry pads / truncates to output_length anyway)
        shifts = np.zeros(goi.shape, np.int32)
        nvar = int((d.geno_offsets[1, goi.ravel()] - d.geno_offsets[0, goi.ravel()]).sum())
        b = dict(regions=regions, goi=goi, to_rc=to_rc, shifts=shifts, nvar=nvar, ds_idx=ds_idx)
        if getattr(d, "svar2", None) is not None:  # the per-call flat channels the reference slices out of its range cache
            b["ch"] = synth.svar2_batch_channels(d.svar2, ds_idx, d.ploidy, d.n_samples)
        out.append(b)
    return out


# ----------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.idx)], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)  # a run that fails before stop() does not leave the sampler behind
        except Exception:
            self.p = None

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [s for s, p in zip(sm, pw) if p > (min(pw) + 0.25 * (max(pw) - min(pw)) if pw else 0)] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons)}


def measured_peak_gbs() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def alg_bytes(w, nvar: float, mode: str = "onehot", n_batches: int = 1) -> float:
    rows = w["pairs"] * 2
    per_bp = {"onehot": ALG_BYTES_PER_BP, "u8": 2.0, "annotated": 10.0}[mode]  # SURVEY.md 8d
    return n_batches * (rows * w["window"] * per_bp + nvar * ALG_BYTES_PER_VARIANT + rows * ALG_BYTES_PER_ROW)


def track_bytes(w, n_tracks: int) -> float:
    """4 B per realigned value written (SURVEY.md 8d; the intervals read add 12 B each, not counted)."""
    return 4.0 * n_tracks * w["pairs"] * 2 * w["window"]


DUMP_BYTES = 64_000_000  # all files of one --dump-outputs, .npy headers included
NPY_HEADER_BYTES = 256


def dump_outputs(out_dir: Path, result, mode: str, budget: int = DUMP_BYTES, seed: int = 0) -> dict:
    """Write one batch as a caller of the pipeline receives it (`FixedPipeline` / `Dataset.to_dataloader`) to
    `out_dir/<name>.npy`: `haplotypes` (or `haps`, `var_idxs`, `ref_coords` when annotated) and `tracks` when realigned
    tracks are on.  uint8 and float32 outputs are written as float32, int32 ones as float64 (exact).  When the files would
    take more than `budget` bytes, every array keeps the same seeded sample of window positions (sorted), all other axes whole.
    Returns {name: written shape}."""
    import torch

    seq, tracks = result if isinstance(result, tuple) else (result, None)
    if mode == "annotated":
        arrays = {"haps": (seq.haps, -1), "var_idxs": (seq.var_idxs, -1), "ref_coords": (seq.ref_coords, -1)}
    else:
        arrays = {"haplotypes": (seq, -2 if mode == "onehot" else -1)}
    if tracks is not None:
        arrays["tracks"] = (tracks, -1)
    dtypes = {k: np.float64 if t.dtype in (torch.int32, torch.int64) else np.float32 for k, (t, _) in arrays.items()}
    L = {t.shape[ax] for t, ax in arrays.values()}.pop()
    per_pos = sum(t.numel() // L * np.dtype(dtypes[k]).itemsize for k, (t, _) in arrays.items())
    keep = max(1, min(L, (budget - NPY_HEADER_BYTES * len(arrays)) // per_pos))
    pos = None
    if keep < L:
        pos = np.sort(np.random.default_rng(seed).choice(L, keep, replace=False))
    out_dir.mkdir(parents=True, exist_ok=True)
    shapes = {}
    for k, (t, ax) in arrays.items():
        if pos is not None:
            t = t.index_select(ax % t.dim(), torch.from_numpy(pos).to(t.device))
        a = t.cpu().numpy().astype(dtypes[k])
        np.save(out_dir / f"{k}.npy", a)
        shapes[k] = a.shape
    return shapes


# ----------------------------------------------------------------------------------------------
# CPU arm: the oracle (C restatement of the reference's Rust/rayon path) on the host cores
# ----------------------------------------------------------------------------------------------
class Svar2Timer:
    """One batch through the oracle's svar2 path: reconstruct_haplotypes_from_svar2 (merge + reconstruct, one task per
    (query, hap)) into a fresh fixed-length buffer, reverse-complement, then the separate one-hot pass."""

    def __init__(self, O, d, w, b):
        self.O, self.d, self.w, self.b = O, d, w, b
        rows = b["goi"].size
        self.oo = (np.arange(rows + 1) * w["window"]).astype(np.int64)
        self.bounds = np.ascontiguousarray(np.stack([self.oo[:-1], self.oo[1:]], 1))

    def __call__(self, parallel=True):
        O, d, b, ch = self.O, self.d, self.b, self.b["ch"]
        out = np.empty(int(self.oo[-1]), np.uint8)
        O.reconstruct_haplotypes_from_svar2(out, self.bounds, b["regions"], b["shifts"], ch["vk_pos"], ch["vk_key"], ch["vk_off"],
                                            ch["dense_pos"], ch["dense_key"], ch["dense_range"], ch["dense_present"],
                                            ch["dense_present_off"], ch["key_ilen"], ch["key_alt"], ch["key_alt_off"],
                                            d.reference, d.ref_offsets, N_CHAR, parallel=parallel)
        O.rc_flat_rows_inplace(out, self.oo, b["to_rc"])
        O.onehot(out, parallel=parallel)
        return out.size


def _timers(O, d, w, batches):
    if getattr(d, "svar2", None) is not None:
        return [Svar2Timer(O, d, w, b) for b in batches]
    return [O.FusedTimer(b["regions"], b["shifts"], b["goi"], d.geno_offsets, d.geno_v_idxs, d.v_starts, d.ilens,
                         d.alt_alleles, d.alt_offsets, d.reference, d.ref_offsets, N_CHAR, w["window"], b["to_rc"],
                         onehot=True) for b in batches]


def cpu_arm(d, w, batches, budget_s: float, threads: int, min_reps: int = 2):
    """Times reconstruct_haplotypes_fused (+ the separate one-hot pass a seqpro user pays) exactly as the
    reference runs it: one crossing per batch, rayon-style (query, hap) tasks on `threads` threads."""
    from oracle import oracle as O

    O.set_threads(threads)
    timers = _timers(O, d, w, batches[:4])
    timers[0](parallel=threads > 1)  # warm-up (page faults, thread start)
    t0 = time.perf_counter()
    n, bp = 0, 0
    while True:
        bp += timers[n % len(timers)](parallel=threads > 1)
        n += 1
        el = time.perf_counter() - t0
        if (el > budget_s and n >= min_reps) or n >= 4096:
            break
    return bp / el, n, el


def reference_gate(w) -> dict:
    """What the reference's own `should_parallelize` (python/genvarloader/_threads.py:122-127) would choose for one
    batch of this workload: parallel only above n_threads x 1 MiB of output."""
    out_bytes = w["pairs"] * 2 * w["window"]
    return {"batch_output_bytes": out_bytes, "rule": "parallel iff output bytes >= n_threads * 1 MiB (_threads.py:122-127)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O

    w, d = build_workload(args.workload, args.seed)
    batches = host_batches(d, w, 8, args.seed + 1)
    threads = O.default_threads()
    O.set_threads(threads)
    timers = _timers(O, d, w, batches)
    for i in range(max(args.warmup, 1)):
        timers[i % len(timers)](parallel=threads > 1)
    t0 = time.perf_counter()
    bp = 0
    for i in range(args.steps):
        bp += timers[i % len(timers)](parallel=threads > 1)
    el = time.perf_counter() - t0
    v = bp / el
    gate = reference_gate(w)
    gate["reference_would_run_parallel"] = bool(gate["batch_output_bytes"] >= threads * (1 << 20))
    line = {
        "impl": "reference", "metric": "haplotype bp/s (one-hot)", "value": v, "unit": "bp/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.workload, w, batches[0]["nvar"], "onehot"),
        "cpu_baseline": {"value": v, "unit": "bp/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} batches of {w['pairs'] * 2} haplotypes x {w['window']} bp: C restatement of "
                                   "reconstruct_haplotypes_fused + separate one-hot pass, one task per (query, hap), persistent "
                                   "thread pool, forced parallel", "thread_gate": gate},
        "e2e": {"value": v, "unit": "bp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(name, w, nvar, mode, n_tracks=0):
    """The `config` object: identical keys and values for both arms (the driver compares them)."""
    return {"workload": f"{name}: {w['desc']}", "window_bp": w["window"], "haplotypes_per_batch": w["pairs"] * 2,
            "variants_per_batch": int(nvar),
            "output": {"onehot": "uint8 one-hot (L,4)", "u8": "uint8 haplotype bytes",
                       "annotated": "uint8 bytes + int32 variant index + int32 reference coordinate"}[mode]
            + (f" + {n_tracks} float32 tracks (b, t, p, L)" if n_tracks else ""),
            "source": "svar2 two-channel source (var_key ranges + dense windows + presence bits, decoded key table)"
            if w.get("source") == "svar2" else "SVAR1-style sparse CSR", "jitter": w.get("jitter", 0)}


# ----------------------------------------------------------------------------------------------
def run_b200(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_

        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from genvarloader_b200 import Interpolate, Repeat5p, _ffi, _kernels
    from genvarloader_b200._dataset import Dataset
    from genvarloader_b200._pipeline import FixedPipeline

    w, d = build_workload(args.workload, args.seed)  # every rank holds a full replica (SURVEY.md 8e)
    L, rows, pairs = w["window"], w["pairs"] * 2, w["pairs"]
    bp_per_step = rows * L
    mode = args.mode
    ds0 = Dataset.from_synth(dev, d, rng=args.seed + 7 + rank, svar2=d.svar2)
    ds0 = ds0.with_len(L).with_settings(jitter=w.get("jitter", 0))
    if mode == "annotated":
        ds0 = ds0.with_seqs("annotated")
    elif mode == "onehot":
        ds0 = ds0.with_encoding("onehot")
    ds = ds0.with_tracks(False)
    n_tracks_main = w.get("tracks", 0)
    if n_tracks_main:
        ds = ds0.with_tracks([f"track{i}" for i in range(n_tracks_main)]).with_insertion_fill(
            {"track0": Repeat5p(), "track1": Interpolate(1)})

    # ---- ring geometry: K steps = n_sub device calls of `ring` batches each, alternating between two halves ----
    out_bytes_step = bp_per_step * ({"onehot": 4, "u8": 1, "annotated": 9}[mode] + 4 * n_tracks_main)
    # (at most ~2 GiB of output per device call: longer calls gain nothing and delay the first batch)
    ring_cap = max(1, min(args.ring, int(args.ring_gib * (1 << 30)) // (2 * out_bytes_step), max(1, (2 << 30) // out_bytes_step)))
    ring = max((r for r in range(1, ring_cap + 1) if args.steps % r == 0 and args.steps // r >= min(args.min_calls, args.steps)), default=1)
    n_sub = args.steps // ring
    pipe = FixedPipeline(ds, pairs, ring=ring)
    n_q = ring * pairs
    # distinct index sets on the device (inputs resident in HBM): every device call reads different windows
    n_sets = max(8, 2 * n_sub)
    idx_sets = torch.from_numpy(np.stack([draw_indices(d, n_q, args.seed + 100 + i, rank, world) for i in range(n_sets)])).to(dev)
    jit_sets = None
    if w.get("jitter", 0):
        jr = np.random.default_rng(args.seed + 5 + rank)
        jit_sets = torch.from_numpy(jr.integers(-w["jitter"], w["jitter"] + 1, size=(n_sets, n_q), dtype=np.int32)).to(dev)
    nvar_per_step = float(np.mean([np.asarray(d.geno_offsets[1] - d.geno_offsets[0])[
        (draw_indices(d, n_q, args.seed + 100 + i, rank, world)[:, None] * 2 + np.arange(2)[None, :]).ravel()].sum()
        for i in range(2)])) / ring
    # resident inputs in the layout the loader's pinned staging buffer has ([ds_idx i64[n]][jitter i32[n]]), so that a device
    # call of the timed block starts with one copy, like the loader's one H2D copy per ring
    comb_sets = torch.zeros((n_sets, n_q + (n_q + 1) // 2), dtype=torch.int64, device=dev)
    comb_sets[:, :n_q] = idx_sets
    if jit_sets is not None:
        comb_sets[:, n_q:].view(torch.int32)[:, :n_q] = jit_sets
    main = torch.cuda.current_stream()
    set_i = [0]

    def submit_resident(pl, h):
        """One device call of half h over the next resident index set (a device-to-device copy of the indices, then the
        captured prep -> plan chain on the plan stream and execute [-> tracks] on the execute stream)."""
        k = set_i[0] % n_sets
        set_i[0] += 1
        pl.submit(h, comb_sets[k])  # indices + jitter draws in the staging layout of a ring half: ONE device-to-device copy

    def timed_block(pl, sync_ranks=True) -> float:
        """Exactly `steps` steps: n_sub device calls alternating between the two halves; device time between one start
        event both half streams wait on and one end event that waits on both."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        if dist is not None and sync_ranks:
            dist.barrier()
            torch.cuda.synchronize()
        if n_sub == 1 and getattr(pl, "fused", False):
            # one device call: both events go on the stream the call is launched on (no cross-stream hop on either side)
            st = pl.halves[0].stream
            e0.record(st)
            submit_resident(pl, 0)
            e1.record(st)
            torch.cuda.synchronize()
            return e0.elapsed_time(e1)  # ms
        e0.record(main)
        pl.wait_all(e0)
        for i in range(n_sub):
            submit_resident(pl, i % pl.n_halves)
        for h in range(min(n_sub, pl.n_halves)):  # every half that ran (their streams are independent)
            main.wait_event(pl.halves[h].done)
        e1.record(main)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)  # ms

    def measure(pl, warm_ms=60.0, max_warm=400):
        """Warm-up blocks (at least `--warmup` steps, and about `warm_ms` of device time so that clocks and caches are in
        steady state), then ONE timed block: exactly `--steps` steps.  The timed block starts from the first resident index
        set whatever the warm-up did, so its inputs, and what its last step computes, are the same from run to run."""
        n_warm = max(1, -(-max(args.warmup, 3) // args.steps))
        last = 0.0
        for _ in range(n_warm):
            last = timed_block(pl)
        more = max(0, int(min(max_warm, np.ceil(warm_ms / max(last, 1e-3)))) - n_warm)
        if dist is not None:  # same block count on every rank (the blocks contain barriers)
            t = torch.tensor([more], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            more = int(t.item())
        for _ in range(more):
            timed_block(pl)
        set_i[0] = 0
        ms = timed_block(pl)
        if dist is not None:  # the slowest rank
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            per_rank = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
            dist.all_gather(per_rank, torch.tensor([ms], device=dev, dtype=torch.float64))
            return float(t.item()), [float(x.item()) for x in per_rank], n_warm + more
        return ms, [ms], n_warm + more

    def last_step(pl):
        """What the last step of the timed block returned to its caller: batch `ring - 1` of the last device call."""
        return pl.halves[(n_sub - 1) % pl.n_halves].out.result((ring - 1) * pairs, pairs)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms, per_rank_ms, warm_blocks = measure(pipe)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_step(pipe), mode)
    value = world * args.steps * bp_per_step / (ms * 1e-3)
    launches = pipe.launches_per_ring * n_sub

    # ---- roofline of the dominant kernel: ONE execute launch over a ring (events on its own stream) ----
    H = pipe.halves[0]
    exec_ms = plan_ms = None
    with torch.cuda.stream(pipe.s_exec):
        sp = pipe.spec
        durs, pdurs = [], []
        for i in range(12):
            k = i % n_sets
            H.idx[:n_q].copy_(idx_sets[k])
            if jit_sets is not None:
                H.jit[:n_q].copy_(jit_sets[k])
            # the same library calls the pipeline's graph holds (gvl_dev_fixed_plan / gvl_dev_fixed_exec over the half's job)
            a0, a1, a2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            a0.record(pipe.s_exec)
            pipe._stage_plan(H.eng, H.scr, H.idx, H.jit if sp.jitter else None, n_q, sub_batch=pairs)  # batch prep + plan (+ svar2 merge)
            a1.record(pipe.s_exec)
            pipe._stage_exec(H.eng, H.scr, H.out, n_q, sub_batch=pairs)
            a2.record(pipe.s_exec)
            pipe.s_exec.synchronize()
            if i >= 2:
                pdurs.append(a0.elapsed_time(a1))
                durs.append(a1.elapsed_time(a2))
        exec_ms, plan_ms = float(np.median(durs)), float(np.median(pdurs))
    packed_ran = int(_ffi.lib.gvl_debug_last_exec_kernel(H.eng.ctx.handle)) == 1
    kernel_name = "hap_exec_oh_kernel (one-hot over the packed reference)" if packed_ran else f"hap_exec_kernel<{mode}> (byte reference)"
    peak, peak_src = measured_peak_gbs()
    ab_launch = alg_bytes(w, nvar_per_step, mode, ring)
    achieved = ab_launch / (exec_ms * 1e-3) / 1e9
    step_bytes = alg_bytes(w, nvar_per_step, mode) + track_bytes(w, n_tracks_main)
    step_achieved = step_bytes * args.steps / (ms * 1e-3) / 1e9  # per GPU
    traffic, traffic_note = None, None
    tp = ROOT / "profiles" / "ncu_exec_traffic.json"
    if tp.exists():
        try:
            tj = json.loads(tp.read_text()).get(args.workload) or {}
            if tj.get("dram_bytes_per_bp") is not None:
                traffic = float(tj["dram_bytes_per_bp"]) * bp_per_step * ring
                traffic_note = tj.get("note")
        except Exception:
            traffic = None

    # ---- tracks (cfg3 only): the same batches with 2 realigned float tracks, same machinery ----
    tracks_line = None
    if not n_tracks_main and w.get("tracks_avail", 0) and mode == "onehot" and not args.no_tracks:
        nt = w["tracks_avail"]
        dst = ds0.with_tracks([f"track{i}" for i in range(nt)]).with_insertion_fill({"track0": Repeat5p(), "track1": Interpolate(1)})
        ring_t = max((r for r in range(1, ring + 1) if args.steps % r == 0 and args.steps // r >= min(args.min_calls, args.steps) and
                      r * 2 * bp_per_step * (4 + 4 * nt) <= args.ring_gib * (1 << 30)), default=1)
        if ring_t == ring:
            pipe_t = FixedPipeline(dst, pairs, ring=ring_t)
            t_ms, _, _ = measure(pipe_t, warm_ms=40.0, max_warm=100)
            tb = alg_bytes(w, nvar_per_step, mode) + track_bytes(w, nt)
            tracks_line = {"n_tracks": nt, "value": world * args.steps * bp_per_step / (t_ms * 1e-3), "unit": "bp/s",
                           "ms_per_step": t_ms / args.steps, "track_values_per_s": world * args.steps * nt * bp_per_step / (t_ms * 1e-3),
                           "alg_bytes_per_step": tb, "whole_step_frac": tb * args.steps / (t_ms * 1e-3) / 1e9 / peak,
                           "fills": ["Repeat5p", "Interpolate(1)"], "gpu_launches": pipe_t.launches_per_ring * n_sub,
                           "how": "cfg3t: the same timed block with 2 realigned float32 tracks per haplotype written as (b, t, p, L)"}
            del pipe_t

    # ---- api: the public loader, host index prep + H2D of the indices inside the timed region, outputs stay in HBM ----
    n_api_batches = ring * max(4, min(16, int(np.ceil(200.0 / max(ms / n_sub, 1e-3)))))
    order = draw_indices(d, n_api_batches * pairs, args.seed + 999, rank, world)
    # (indices address the dataset's (region, sample) grid: flat = r * n_samples + s, the loader's own convention)
    loader = ds.to_dataloader(batch_size=pairs, sampler=order, mode="double_buffered", copy=False, ring=ring)
    for _ in loader:  # warm-up epoch (builds nothing new: the pipeline exists since construction)
        pass
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    nb = 0
    for batch in loader:
        nb += 1
    torch.cuda.synchronize()
    api_s = time.perf_counter() - t0
    api_t = torch.tensor([api_s], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(api_t, op=dist.ReduceOp.MAX)
    api = {"value": world * nb * bp_per_step / float(api_t.item()), "unit": "bp/s", "batches": nb, "ring": ring,
           "h2d_bytes_per_step": pairs * (8 + (4 if w.get("jitter", 0) else 0)), "d2h_bytes_per_step": 0,
           "path": "for batch in Dataset.to_dataloader(batch_size, sampler=..., mode='double_buffered', copy=False): host index "
                   "prep + one pinned H2D copy per ring inside the timed region; batches are CUDA tensors (views into the ring)"}
    del loader

    # ---- e2e: the reference-shaped host-buffer call (numpy in, pinned numpy out), copies included; every rank ----
    eng0 = ds.engine
    batches = host_batches(d, w, 8, args.seed + 1, rank, world)
    e2e_bytes_out = rows * L * 4  # the e2e leg always returns the one-hot (the headline metric)
    pinned = _kernels.PinnedBuffer(e2e_bytes_out)
    if d.svar2 is not None:
        sv = d.svar2
        _kernels.pin_static(d.reference, d.ref_offsets, sv["key_ilen"], sv["key_alt"], sv["key_alt_off"], ctx=eng0.ctx)

        def e2e_step(b):
            ch = b["ch"]
            _kernels.reconstruct_haplotypes_from_svar2(b["regions"], b["shifts"], ch["vk_pos"], ch["vk_key"], ch["vk_off"],
                                                       ch["dense_pos"], ch["dense_key"], ch["dense_range"], ch["dense_present"],
                                                       ch["dense_present_off"], sv["key_ilen"], sv["key_alt"], sv["key_alt_off"],
                                                       d.reference, d.ref_offsets, N_CHAR, L, to_rc=b["to_rc"], mode="onehot",
                                                       out=pinned.array, ctx=eng0.ctx)
    else:
        _kernels.pin_static(d.geno_offsets, d.geno_v_idxs, d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets,
                            d.reference, d.ref_offsets, ctx=eng0.ctx)

        def e2e_step(b):
            _kernels.reconstruct_haplotypes_fused(b["regions"], b["shifts"], b["goi"], d.geno_offsets, d.geno_v_idxs,
                                                  d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets, d.reference,
                                                  d.ref_offsets, N_CHAR, L, None, None, b["to_rc"], mode="onehot",
                                                  out=pinned.array, ctx=eng0.ctx)

    for i in range(3):
        e2e_step(batches[i % len(batches)])
    n_e2e = max(3, min(max(args.steps, 20), int(2.0 / max(e2e_bytes_out / 20e9, 1e-4))))
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(n_e2e):
        e2e_step(batches[i % len(batches)])
    e2e_t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    h2d = int(sum(batches[0][k].nbytes for k in ("regions", "shifts", "goi", "to_rc")))
    if d.svar2 is not None:  # the batch's gathered channels travel too (the reference slices them from its range cache)
        h2d = int(sum(batches[0][k].nbytes for k in ("regions", "shifts", "to_rc")) + sum(
            batches[0]["ch"][k].nbytes for k in ("vk_pos", "vk_key", "vk_off", "dense_pos", "dense_key", "dense_range",
                                                 "dense_present", "dense_present_off")))
    e2e = {"value": world * n_e2e * bp_per_step / float(e2e_t.item()), "unit": "bp/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": int(e2e_bytes_out + (rows + 1) * 8), "steps": n_e2e, "ranks": world,
           "path": ("genvarloader_b200._kernels.reconstruct_haplotypes_from_svar2(mode='onehot') -> gvl_reconstruct_haplotypes_from_svar2_begin / "
                    "gvl_reconstruct_haplotypes_fused_finish" if d.svar2 is not None else
                    "genvarloader_b200._kernels.reconstruct_haplotypes_fused(mode='onehot') -> gvl_reconstruct_haplotypes_fused_begin/_finish")
                   + ", host numpy in, pinned host numpy out; every rank runs it on its own PCIe link, value = all ranks' bp / max time"}

    # ---- e2e_loader: the loader delivering into pinned HOST memory (the reference's DataLoader hands out host batches too):
    #      every ring is copied device-to-host on a copy stream while the next one is produced ----
    ring_h = max(1, min(ring, int((256 << 20) // max(rows * L * 4, 1))))
    n_h = ring_h * max(4, min(64, int(np.ceil(1.5e9 / max(ring_h * rows * L * 4, 1)))))
    order_h = draw_indices(d, n_h * pairs, args.seed + 555, rank, world)
    loader_h = ds.to_dataloader(batch_size=pairs, sampler=order_h, mode="double_buffered", copy=False, ring=ring_h, to_host=True)
    for _ in loader_h:  # warm-up epoch: allocates the pinned twins
        pass
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    nbh = 0
    for hb in loader_h:
        nbh += 1
    eh_t = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(eh_t, op=dist.ReduceOp.MAX)
    e2e_loader = {"value": world * nbh * bp_per_step / float(eh_t.item()), "unit": "bp/s", "batches": nbh, "ring": ring_h,
                  "h2d_bytes_per_step": pairs * (8 + (4 if w.get("jitter", 0) else 0)), "d2h_bytes_per_step": int(rows * L * 4),
                  "path": "for batch in Dataset.to_dataloader(batch_size, sampler=..., mode='double_buffered', copy=False, to_host=True): "
                          "numpy batches in pinned host memory; the device-to-host copy of ring n overlaps the production of ring n+1"}
    del loader_h

    # ---- single-consumer gather over NCCL / NVLink (reported apart from the roofline, SURVEY.md 8e) ----
    gather = None
    if dist is not None:
        from genvarloader_b200._dist import gather_rows

        # a whole device call's output (ring batches) per rank: large enough to show the link rate
        g_rows = rows * ring
        out_t = pipe.halves[0].out.seq[: g_rows * L * 4].view(g_rows * L, 4) if mode == "onehot" else pipe.halves[0].out.seq[: g_rows * L]
        offs = torch.arange(g_rows + 1, device=dev, dtype=torch.int64) * L
        for _ in range(2):
            gather_rows(out_t, offs, dst=0)
        torch.cuda.synchronize()
        dist.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_g = 5
        g0.record()
        for _ in range(n_g):
            gather_rows(out_t, offs, dst=0)
        g1.record()
        torch.cuda.synchronize()
        g_ms = torch.tensor([g0.elapsed_time(g1) / n_g], device=dev, dtype=torch.float64)
        dist.all_reduce(g_ms, op=dist.ReduceOp.MAX)
        recv = (world - 1) * out_t.numel() * out_t.element_size()
        gather = {"ms_per_device_call": float(g_ms.item()), "batches": ring, "consumer_ingest_GBps": recv / (float(g_ms.item()) * 1e-3) / 1e9,
                  "bytes_received_by_consumer": recv, "how": "genvarloader_b200._dist.gather_rows: every rank's batch output "
                  "(one-hot rows) sent to rank 0 over NCCL point-to-point; not on the hot path, not part of the roofline"}
    clk = clocks.stop() if rank == 0 else None
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    # ---- CPU baseline (bounded sample of the same workload; rank 0, after the GPU legs) ----
    from oracle import oracle as O

    threads = O.default_threads()
    cpu_batches = host_batches(d, w, 4, args.seed + 1)
    cpu_v, cpu_n, cpu_s = cpu_arm(d, w, cpu_batches, budget_s=args.cpu_seconds, threads=threads)
    cpu1_v, cpu1_n, _ = cpu_arm(d, w, cpu_batches, budget_s=min(args.cpu_seconds, 4.0), threads=1)
    gate = reference_gate(w)
    gate["reference_would_run_parallel"] = bool(gate["batch_output_bytes"] >= threads * (1 << 20))

    # `config` is identical in both arms (the driver compares them); how THIS arm runs the workload goes to `pipeline`
    cfg = workload_config(args.workload, w, host_batches(d, w, 1, args.seed + 1)[0]["nvar"], mode, n_tracks_main)
    pipeline = {"batches_per_device_call": ring, "device_calls_per_timed_block": n_sub, "halves": pipe.n_halves,
                "cuda_graph": pipe.use_graph, "warmup_blocks": warm_blocks, "launches_per_device_call": pipe.launches_per_ring,
                "l2": f"{n_sets} resident index sets over {d.n_regions} regions of a {w['contig_len'] / 1e6:.0f} Mb contig (packed reference "
                      f"{w['contig_len'] / 2e6:.0f} MB); every device call writes {ring * out_bytes_step >> 20} MiB into its half "
                      "(> 126 MB L2 per call)",
                "parallelism": f"dp{world} (replicated tables, (region,sample) shards, no collective)"}
    line = {
        "metric": "haplotype bp/s (%s)" % {"onehot": "one-hot", "u8": "uint8 bytes", "annotated": "annotated"}[mode],
        "value": value, "unit": "bp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": cfg, "pipeline": pipeline, "timed_block_ms": ms, "per_rank_ms": per_rank_ms,
        "output_GBps": value * {"onehot": 4, "u8": 1, "annotated": 9}[mode] / 1e9, "algorithmic_GBps": step_achieved * world,
        "whole_step_frac": step_achieved / peak,
        "roofline": {"bound": "hbm", "kernel": kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src,
                     "alg_bytes_per_launch": ab_launch, "launch_ms": exec_ms, "plan_kernel_ms": plan_ms,
                     "batches_per_launch": ring,
                     "plan_note": "plan_kernel_ms = batch prep + plan (+ svar2 merge) of the same device call between two events on an "
                                  "otherwise idle stream (includes the launch latencies of its 2-3 kernels)",
                     "how": f"one execute launch covers the {ring} batches of a device call; its duration is the time between two CUDA "
                            "events around that single launch on the stream it runs on (median of 10, nothing else on the GPU)",
                     "frac_of_nominal_8TBps": achieved / 8000.0,
                     "bytes_note": "algorithmic bytes = SURVEY.md 8d (5 B/bp: 1 reference byte + 4 one-hot bytes); the packed reference "
                                   "moves 0.5 B/bp; the peak is a read+write copy figure, so a nearly write-only kernel can land a "
                                   "little above 1.0",
                     "whole_step_frac": step_achieved / peak},
        "cpu_baseline": {"value": cpu_v, "unit": "bp/s", "cores": threads, "kind": "port",
                         "sample": f"{cpu_n} batches ({cpu_s:.1f} s) of the same workload; C restatement of the reference's "
                                   "reconstruct_haplotypes_fused + separate one-hot pass (oracle/gvl_oracle.c), persistent thread pool",
                         "single_thread_value": cpu1_v, "thread_gate": gate},
        "api": api, "e2e": e2e, "e2e_loader": e2e_loader, "gpu_launches": int(launches), "clocks": clk,
    }
    if tracks_line:
        line["tracks"] = tracks_line
    if gather:
        line["gather"] = gather
    print(json.dumps(line))


def main():
    sys.dont_write_bytecode = True  # the benchmark writes nothing into the source tree (it may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=640)
    ap.add_argument("--warmup", type=int, default=64)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--mode", default="onehot", choices=["onehot", "u8", "annotated"],
                    help="output of the execute kernel (the headline metric is one-hot)")
    ap.add_argument("--ring", type=int, default=128, help="batches per device call, at most (the largest divisor of --steps)")
    ap.add_argument("--min-calls", type=int, default=1, help="device calls per timed block, at least")
    ap.add_argument("--ring-gib", type=float, default=12.0, help="output memory of the two ring halves, at most")
    ap.add_argument("--no-tracks", action="store_true", help="skip the cfg3t extra leg")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", type=Path, metavar="DIR",
                    help="write the last timed step's batch to DIR/<name>.npy (float32 / float64, at most 64 MB: a fixed "
                         "seeded sample of window positions when larger); the same arguments give the same arrays")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
