"""What `with_tracks(kind="realigned-intervals")` costs against the realigned-tracks read it replaces, on two shapes:

  cfg3t   16 (region, sample) pairs x ploidy 2 = 32 rows x 524,288 values x 2 tracks (~50 bp runs), jitter 128, half the
          regions on the negative strand, ~1 variant/kb/haplotype, Repeat5p and Interpolate(1);
  cfg2d   32 pairs x ploidy 2 = 64 rows x 131,072 values x 2 tracks, ~10 variants/kb/haplotype (the bench's dense cell).

For each shape one dataset serves both kinds (`kind="tracks"` and `"realigned-intervals"`, same haplotype sequences): every
kind is warmed, then the two alternate, REPEATS timed `ds[r, s]` reads each, CUDA events from before the call to after a
synchronise.  A separate pass under torch.profiler (CUDA activities) takes the device time of the count and emit kernels
and of the track execute.  Output bytes are those of the returned track part.  The card's name, power limit and max SM
clock are read in the same run.  Not a bench.py number; context for DESIGN.md section 4.3.

    python profiles/probe_realigned_intervals.py [out.json]      (default: profiles/probe_realigned_intervals.json)
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

REPEATS, WARMUP = 15, 3
KINDS = ("tracks", "realigned-intervals")


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clock = (x.strip() for x in (q.stdout.strip().split(",") + ["?", "?", "?"])[:3])
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def shape(name: str, dev):
    if name == "cfg3t":
        L, pairs, jit = 524_288, 16, 128
        d = synth.make_dataset(3, 20_000_000, 4, 32, L + 2 * jit, 1.0, max_jitter=jit, snp_frac=0.8, neg_strand_frac=0.5,
                               straddle_ends=False, n_tracks=2, fast_tracks=True)
    else:
        L, pairs, jit = 131_072, 32, 0
        d = synth.make_dataset(2, 5_000_000, 8, 64, L, 10.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=2,
                               fast_tracks=True)
    ds = (Dataset.from_synth(dev, d, rng=7).with_seqs("haplotypes").with_len(L).with_settings(jitter=jit)
          .with_tracks(["track0", "track1"]).with_insertion_fill({"track0": gvl.Repeat5p(), "track1": gvl.Interpolate(1)}))
    rng = np.random.default_rng(11)
    r, s = rng.integers(0, d.n_regions, pairs), rng.integers(0, d.n_samples, pairs)
    return ds, r, s, {"pairs": pairs, "ploidy": 2, "rows": 2 * pairs, "values_per_row": L, "tracks": 2, "jitter": jit}


def nbytes(out) -> int:
    trk = out[1]
    if isinstance(trk, torch.Tensor):
        return trk.numel() * trk.element_size()
    if hasattr(trk, "starts"):
        return sum(x.data.numel() * x.data.element_size() for x in (trk.starts, trk.ends, trk.values)) + trk.offsets.numel() * 8
    return trk.data.numel() * trk.data.element_size() + trk.offsets.numel() * 8


def timed(ds, r, s) -> float:
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = ds[r, s]
    e.record()
    torch.cuda.synchronize()
    del out
    return a.elapsed_time(e) * 1e3


def kernel_times(views, r, s) -> dict:
    from torch.profiler import ProfilerActivity, profile

    res = {}
    for k, ds in views.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(3):
                ds[r, s]
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            nm = ev.name
            key = next((x for x in ("ritv_count_kernel", "ritv_emit_kernel", "trk_exec3_kernel", "trk_tile_prep_kernel",
                                    "hap_plan_par_kernel", "scan_") if x in nm), None)
            if key is not None:
                per.setdefault(key, []).append(ev.time_range.elapsed_us())
        res[k] = {n: {"launches_per_read": len(v) / 3, "us_per_read": sum(v) / 3} for n, v in sorted(per.items())}
    return res


def main():
    dst = Path(sys.argv[1]) if len(sys.argv) > 1 else Path(__file__).resolve().parent / "probe_realigned_intervals.json"
    if not torch.cuda.is_available():
        raise SystemExit("probe_realigned_intervals.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "how": "ds[r, s] timed with CUDA events from before the call to after a synchronise; kinds "
                                     "alternated after a warm-up; profiler pass separate", "shapes": {}}
    for name in ("cfg3t", "cfg2d"):
        ds, r, s, geo = shape(name, dev)
        views = {k: ds.with_tracks(kind=k) for k in KINDS}
        byt = {k: nbytes(views[k][r, s]) for k in KINDS}
        for _ in range(WARMUP):
            for k in KINDS:
                timed(views[k], r, s)
        t = {k: [] for k in KINDS}
        for _ in range(REPEATS):
            for k in KINDS:
                t[k].append(timed(views[k], r, s))
        n_itv = int(views["realigned-intervals"][r, s][1].offsets[-1])
        res["shapes"][name] = {"shape": geo, "intervals": n_itv, "output_bytes": byt,
                               "us_per_read": {k: {"median": statistics.median(v), "min": min(v), "max": max(v)}
                                               for k, v in t.items()},
                               "kernels": kernel_times(views, r, s)}
        print(name, {k: round(statistics.median(v)) for k, v in t.items()}, byt, n_itv)
    dst.parent.mkdir(parents=True, exist_ok=True)
    dst.write_text(json.dumps(res, indent=1) + "\n")
    print(res["gpu"])


if __name__ == "__main__":
    main()
