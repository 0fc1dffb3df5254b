"""What binned tracks save a training step: the cfg3t shape (16 (region, sample) pairs x ploidy 2 = 32 rows x 524,288
values per batch, one-hot haplotypes + 2 realigned float32 tracks, Repeat5p and Interpolate(1), jitter 128, half the
regions on the negative strand), for bins of 32 and 128 bp, two ways of getting mean-binned tracks:

  pool    an unbinned float32 read, then `x.unflatten(-1, (L // bin, bin)).mean(-1)` in torch;
  binned  `with_track_bins(bin, "mean")`: the track kernels store one value per bin.

Both through `ds[r, s]` (one synchronous read per batch) and through `to_dataloader(mode="double_buffered", copy=False)`
at the default ring.  Loaders are built and warmed once; then the variants alternate, REPEATS passes each.  A pass of
N_BATCHES batches is timed with CUDA events (before the iteration to after the consumer's last operation) and reported
as µs per batch.  A separate loader pass under torch.profiler (CUDA activities) gives the execute kernel's mean time.
Bytes written per batch by the track kernels are computed from the shapes.  The card's name, power limit and max SM
clock are read in the same run.  Not a bench.py number; context for DESIGN.md section 4.3.

    python profiles/probe_track_bins.py [out.json]      (default: profiles/probe_track_bins.json)
"""
from __future__ import annotations

import json
import statistics
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
from probe_track_dtype import L, N_BATCHES, PAIRS, build, gpu_info  # noqa: E402

REPEATS = 5
BINS = (32, 128)


def variants():
    return [(b, how) for b in BINS for how in ("pool", "binned")]


def pooled(trk, b):
    return trk.unflatten(-1, (L // b, b)).mean(-1)


def timed(fn) -> float:
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    n = fn()
    e.record()
    torch.cuda.synchronize()
    return a.elapsed_time(e) * 1e3 / n


def loader_pass(dl, b, how) -> int:
    n = 0
    for seq, trk in dl:
        if how == "pool":
            trk = pooled(trk, b)
        n += 1
    assert n == N_BATCHES and trk.shape[-1] == L // b
    return n


def getitem_pass(ds, order, b, how) -> int:
    for i in range(N_BATCHES):
        k = order[i * PAIRS:(i + 1) * PAIRS]
        r, s = k // ds.n_samples, k % ds.n_samples
        seq, trk = ds[r, s]
        if how == "pool":
            trk = pooled(trk, b)
    assert trk.shape[-1] == L // b
    return N_BATCHES


def exec_kernel_us(dl, b, how) -> dict:
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loader_pass(dl, b, how)
    ex, pool = [], []
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.time_range.elapsed_us()
        if "trk_exec3_kernel" in ev.name:
            ex.append(us)
        elif how == "pool" and "gvl" not in ev.name and ("reduce" in ev.name.lower() or "mean" in ev.name.lower()):
            pool.append(us)
    return {"exec_launches": len(ex), "exec_us_mean": statistics.fmean(ex) if ex else None,
            "pool_launches": len(pool), "pool_us_mean": statistics.fmean(pool) if pool else None}


def main():
    dst = Path(sys.argv[1]) if len(sys.argv) > 1 else Path(__file__).resolve().parent / "probe_track_bins.json"
    if not torch.cuda.is_available():
        raise SystemExit("probe_track_bins.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    ds, order = build(dev)
    dss = {(b, how): ds.with_track_bins(b, "mean") if how == "binned" else ds for b, how in variants()}
    loaders = {v: dss[v].to_dataloader(batch_size=PAIRS, sampler=order, mode="double_buffered", copy=False) for v in variants()}
    # one batch: the binned read is the definition (float64 mean of the unbinned read, rounded to float32) within one unit
    # in the last place; torch's float32 pooling is another rounding of the same mean (its largest difference is reported)
    k = order[:PAIRS]
    agree = {}
    for b in BINS:
        x = ds.with_settings(rng=5)[k // ds.n_samples, k % ds.n_samples][1]  # (the same jitter draws)
        y = dss[(b, "binned")].with_settings(rng=5)[k // ds.n_samples, k % ds.n_samples][1]
        ref = x.double().unflatten(-1, (L // b, b)).mean(-1).float()
        fin = ~torch.isnan(ref)
        assert torch.equal(fin, ~torch.isnan(y)), b
        ulps = (ref[fin].view(torch.int32).long() - y[fin].view(torch.int32).long()).abs()
        assert int(ulps.max()) <= 1, (b, int(ulps.max()))
        agree[f"bin{b}"] = {"max_ulps_vs_definition": int(ulps.max()),
                            "max_abs_diff_torch_pool": float((pooled(x, b) - y)[fin].abs().max())}
    for v in variants():  # warm-up: modules, graphs, allocator, the eager pipelines
        loader_pass(loaders[v], *v)
        getitem_pass(dss[v], order, *v)
    t_loader = {v: [] for v in variants()}
    t_get = {v: [] for v in variants()}
    for _ in range(REPEATS):
        for v in variants():
            t_loader[v].append(timed(lambda: loader_pass(loaders[v], *v)))
            t_get[v].append(timed(lambda: getitem_pass(dss[v], order, *v)))
    rows = 2 * PAIRS * 2  # (row, track) pairs per batch
    key = lambda v: f"bin{v[0]}_{v[1]}"
    res = {"gpu": info, "shape": {"pairs": PAIRS, "ploidy": 2, "rows": 2 * PAIRS, "values_per_row": L, "tracks": 2,
                                  "batches_per_pass": N_BATCHES, "repeats": REPEATS,
                                  "ring": {key(v): loaders[v].pipe.ring for v in variants()}},
           "how": "ds[r, s] per batch and to_dataloader(batch_size=16, mode='double_buffered', copy=False) at the default ring; "
                  "'pool' = unbinned float32 read + torch unflatten().mean(-1), 'binned' = with_track_bins(bin, 'mean'); CUDA "
                  "events around one pass per repeat, variants alternated",
           "agreement": agree,
           "track_bytes_written_per_batch": {key(v): rows * (L if v[1] == "pool" else L // v[0]) * 4 for v in variants()},
           "loader_us_per_batch": {key(v): {"median": statistics.median(t), "min": min(t), "max": max(t)} for v, t in t_loader.items()},
           "getitem_us_per_batch": {key(v): {"median": statistics.median(t), "min": min(t), "max": max(t)} for v, t in t_get.items()},
           "kernels": {key(v): exec_kernel_us(loaders[v], *v) for v in variants()}}
    dst.parent.mkdir(parents=True, exist_ok=True)
    dst.write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({"loader": {k: v["median"] for k, v in res["loader_us_per_batch"].items()},
                      "getitem": {k: v["median"] for k, v in res["getitem_us_per_batch"].items()}}), info)


if __name__ == "__main__":
    main()
