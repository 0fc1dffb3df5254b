"""What a bfloat16 track output saves a training loop: the read-ahead loader on the cfg3t shape (16 (region, sample) pairs
x ploidy 2 = 32 rows x 524,288 values per batch, one-hot haplotypes + 2 realigned tracks, Repeat5p and Interpolate(1),
jitter 128, half the regions on the negative strand) through `to_dataloader(mode="double_buffered", copy=False)` at the
default ring, three variants:

  f32        float32 tracks (the default);
  bf16       `with_track_dtype(torch.bfloat16)`: the track kernels store bfloat16;
  f32+cast   float32 tracks and the per-batch `.to(torch.bfloat16)` a user pays without the option.

Each variant's loader is built once and warmed by one pass; then the variants alternate in one process, REPEATS passes
each.  A pass of N_BATCHES batches is timed with CUDA events (start before the iteration, end after the consumer's last
operation) and reported as µs per batch.  A separate pass under torch.profiler (CUDA activities) takes the execute
kernel's time per dtype and the cast kernel's time.  The card's name, power limit and max SM clock are read in the same
run.  Not a bench.py number; context for DESIGN.md section 4.3.

    python profiles/probe_track_dtype.py [out.json]      (default: profiles/probe_track_dtype.json)
"""
from __future__ import annotations

import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import genvarloader_b200 as gvl  # noqa: E402
from genvarloader_b200 import synth  # noqa: E402
from genvarloader_b200._dataset import Dataset  # noqa: E402

L, PAIRS, N_BATCHES, REPEATS = 524_288, 16, 48, 7
VARIANTS = ("f32", "bf16", "f32+cast")


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in (q.stdout.strip().split(",") + ["?", "?", "?"])[:3])
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def build(dev):
    d = synth.make_dataset(3, 20_000_000, 4, 32, L + 2 * 128, 1.0, max_jitter=128, snp_frac=0.8, neg_strand_frac=0.5,
                           straddle_ends=False, n_tracks=2, fast_tracks=True)
    ds = (Dataset.from_synth(dev, d, rng=7).with_len(L).with_encoding("onehot").with_settings(jitter=128)
          .with_tracks(["track0", "track1"]).with_insertion_fill({"track0": gvl.Repeat5p(), "track1": gvl.Interpolate(1)}))
    order = np.random.default_rng(11).integers(0, len(ds), N_BATCHES * PAIRS)
    return ds, order


def loader(ds, order, variant: str):
    dsx = ds.with_track_dtype(torch.bfloat16) if variant == "bf16" else ds
    return dsx.to_dataloader(batch_size=PAIRS, sampler=order, mode="double_buffered", copy=False)


def one_pass(dl, variant: str) -> float:
    """µs per batch of one pass over N_BATCHES batches."""
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    n = 0
    for seq, trk in dl:
        if variant == "f32+cast":
            trk = trk.to(torch.bfloat16)
        n += 1
    e.record()
    torch.cuda.synchronize()
    assert n == N_BATCHES and trk.dtype == (torch.float32 if variant == "f32" else torch.bfloat16)
    return a.elapsed_time(e) * 1e3 / n


def kernel_times(loaders) -> dict:
    """Mean device time per launch of the track execute kernel (per dtype) and of the cast, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    out = {}
    for variant in VARIANTS:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            one_pass(loaders[variant], variant)
        ex, cast = [], []
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            us = ev.time_range.elapsed_us()
            if "trk_exec3_kernel" in ev.name:
                ex.append((ev.name, us))
            elif variant == "f32+cast" and ("copy" in ev.name.lower() or "elementwise" in ev.name.lower()) and "gvl" not in ev.name:
                cast.append(us)
        names = sorted({n for n, _ in ex})
        out[variant] = {"exec_kernel": names, "exec_launches": len(ex),
                        "exec_us_mean": statistics.fmean([u for _, u in ex]) if ex else None}
        if variant == "f32+cast":
            out[variant].update(cast_launches=len(cast), cast_us_mean=statistics.fmean(cast) if cast else None)
    return out


def main():
    dst = Path(sys.argv[1]) if len(sys.argv) > 1 else Path(__file__).resolve().parent / "probe_track_dtype.json"
    if not torch.cuda.is_available():
        raise SystemExit("probe_track_dtype.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    ds, order = build(dev)
    loaders = {v: loader(ds, order, v) for v in VARIANTS}
    ring = {v: loaders[v].pipe.ring for v in VARIANTS}
    for v in VARIANTS:  # warm-up: modules, graphs, allocator
        one_pass(loaders[v], v)
    times = {v: [] for v in VARIANTS}
    for _ in range(REPEATS):
        for v in VARIANTS:
            times[v].append(one_pass(loaders[v], v))
    res = {"gpu": info, "shape": {"pairs": PAIRS, "ploidy": 2, "rows": 2 * PAIRS, "values_per_row": L, "tracks": 2,
                                  "batches_per_pass": N_BATCHES, "repeats": REPEATS, "ring": ring},
           "how": "to_dataloader(batch_size=16, mode='double_buffered', copy=False) at the default ring, one loader per variant "
                  "built and warmed once; CUDA events around one pass (iteration start to the consumer's last op) per "
                  "repeat; variants alternated",
           "us_per_batch": {v: {"median": statistics.median(t), "min": min(t), "max": max(t), "all": t} for v, t in times.items()},
           "kernels": kernel_times(loaders)}
    dst.parent.mkdir(parents=True, exist_ok=True)
    dst.write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({v: res["us_per_batch"][v]["median"] for v in VARIANTS}), info)


if __name__ == "__main__":
    main()
