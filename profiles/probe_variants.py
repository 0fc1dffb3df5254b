"""`Dataset.with_seqs("variants")` on the bench workloads' shapes.

Leg 1, `ds[r, s]`: time per call (device drained) and variants per second.  A call is the sizing pass (one wait) ->
gather_rows -> take(start, ilen) -> gather_alleles -> rc_alleles [-> dummy fill].
Leg 2, the loader: batches/s and variants/s of one epoch of `to_dataloader(b, sampler=..., mode=None)` (one `ds[r, s]` per
batch) against `mode="double_buffered", copy=False` (rings of batches per device call, `_variants_loader.py`), the consumer
doing nothing with the batches; device drained at the end of the epoch, after one untimed warm-up epoch.
Prints the card's name and power limit first.  Not a bench.py number; context for DESIGN.md sections 4.5 and 4.7."""
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import bench  # noqa: E402
from genvarloader_b200 import Dataset, DummyVariant  # noqa: E402

q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
print(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit: {q.stdout.strip().splitlines()[0] if q.stdout else 'n/a'}")

N_LOADER_BATCHES = 48

for name, pairs in (("cfg2d", None), ("cfg4", None), ("cfg1", 8000)):
    w, d = bench.build_workload(name, 2)
    pairs = pairs or w["pairs"]
    if getattr(d, "geno_v_idxs", None) is None:
        continue
    try:
        ds = Dataset.from_synth(torch.device("cuda", 0), d, rng=0).with_tracks(False).with_seqs("variants")
    except NotImplementedError as e:  # (cfg2 is built on the svar2 source)
        print(f"{name}: {e}")
        continue
    rng = np.random.default_rng(0)
    idx = [(rng.integers(0, ds.n_regions, pairs), rng.integers(0, ds.n_samples, pairs)) for _ in range(8)]
    for label, dsv in (("alt,ilen,start", ds), ("+ dummy fill", ds.with_settings(dummy_variant=DummyVariant()))):
        for r, s in idx[:3]:
            out = dsv[r, s]
        torch.cuda.synchronize()
        n = 40
        t0 = time.perf_counter()
        for k in range(n):
            r, s = idx[k % len(idx)]
            out = dsv[r, s]
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / n
        nv = int(out.offsets[-1].item())
        nb = int(out["alt"].data.numel())
        print(f"{name} variants [{label}]: {pairs} pairs x {d.ploidy} rows, {nv} variants, {nb} ALT bytes per call: "
              f"{dt * 1e6:.0f} us per call = {nv / dt / 1e6:.1f} M variants/s")

    # ---- loader leg
    sampler = np.random.default_rng(1).integers(0, len(ds), N_LOADER_BATCHES * pairs)
    for label, dsv in (("alt,ilen,start", ds), ("+ dummy fill", ds.with_settings(dummy_variant=DummyVariant()))):
        n_var = sum(int(b.offsets[-1]) for b in dsv.to_dataloader(pairs, sampler=sampler))
        res = {}
        for mode in (None, "double_buffered"):
            ld = dsv.to_dataloader(pairs, sampler=sampler, mode=mode, copy=False)
            for _ in ld:  # warm-up epoch
                pass
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nb = 0
            for _ in ld:
                nb += 1
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            res[mode] = dt
            ring = getattr(ld, "ring", "-")
            print(f"{name} loader [{label}] mode={mode} (ring {ring}): {nb} batches of {pairs} pairs, {n_var} variants in "
                  f"{dt * 1e3:.1f} ms = {nb / dt:.0f} batches/s = {n_var / dt / 1e6:.1f} M variants/s")
        print(f"{name} loader [{label}]: double_buffered / mode=None = {res[None] / res['double_buffered']:.2f}x")
