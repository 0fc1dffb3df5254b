"""Cost of tracks and variants on spliced datasets: time per `ds[...]` of one spliced batch with two realigned tracks
(Repeat5p and Interpolate(1)) next to the same batch with `with_tracks(False)`; the `variants` output (default fields) and
`variant-windows` (VarWindowOpt(32, "ACGT", 4), window mode) of the same batch, next to the unspliced `variants` read of its
element batch E (`ds[e_reg, e_s]`: the same rows, one cell per element); plus the library calls each makes.

Shape: 512 regions of 150-3,000 bp (exon-like), 16 samples, 64 splice rows of 8 elements; one batch = 32 rows x 8 samples
= 256 (row, sample) pairs = 2,048 elements, ~6.4 M haplotype bases per call.  Each leg is timed over `--iters` calls
ending in a device synchronise (host clock), the legs alternating over `--rounds` rounds after a warm-up of each.
Not a bench.py number; run as `python profiles/probe_spliced.py [--out DIR]`."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from genvarloader_b200 import Dataset, Interpolate, Repeat5p, VarWindowOpt, _engine, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--iters", type=int, default=50)
ap.add_argument("--rounds", type=int, default=3)
ap.add_argument("--out", default=None)
a = ap.parse_args()

dev = torch.device("cuda", 0)
rng = np.random.default_rng(11)
d = synth.make_dataset(17, 4_000_000, 16, 512, 3000, 2.0, neg_strand_frac=0.5, straddle_ends=False, n_tracks=2,
                       fast_tracks=True)
d.regions[:, 2] = d.regions[:, 1] + rng.integers(150, 3001, d.n_regions)
rows = [np.sort(rng.choice(d.n_regions, 8, replace=False)) for _ in range(64)]
ds = Dataset.from_synth(dev, d, rng=0).with_insertion_fill({"track0": Repeat5p(), "track1": Interpolate(1)})
sp_t = ds.with_settings(splice_info=rows)
sp_n = sp_t.with_tracks(False)
idx = (slice(0, 32), slice(0, 8))
sp_v = sp_n.with_seqs("variants")
sp_w = sp_n.with_seqs("variant-windows", VarWindowOpt(32, "ACGT", 4))
e_reg = np.concatenate([rows[r] for r in range(32) for _ in range(8)]).astype(np.int64)
e_s = np.concatenate([np.full(len(rows[r]), s, np.int64) for r in range(32) for s in range(8)])
un_v = ds.with_tracks(False).with_seqs("variants")
legs = {"tracks": (sp_t, idx), "no_tracks": (sp_n, idx), "variants": (sp_v, idx), "variant_windows": (sp_w, idx),
        "unspliced_variants_over_E": (un_v, (e_reg, e_s))}


class Counting:
    def __init__(self, lib):
        self.lib, self.calls = lib, []

    def __getattr__(self, name):
        fn = getattr(self.lib, name)

        def wrapped(*args):
            self.calls.append(name)
            return fn(*args)

        return wrapped


def n_calls(ds_, ix):
    lib = _engine.lib
    _engine.lib = c = Counting(lib)
    try:
        ds_[ix]
    finally:
        _engine.lib = lib
    return len(c.calls)


def timed(ds_, ix) -> float:
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.iters):
        ds_[ix]
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / a.iters * 1e3


for x, ix in legs.values():  # warm-up: module loads, allocator, pinned staging
    for _ in range(5):
        x[ix]
res = {k: [] for k in legs}
for _ in range(a.rounds):
    for k, (x, ix) in legs.items():
        res[k].append(timed(x, ix))
h, t = sp_t[idx]
v = sp_v[idx]
assert (v.offsets[-1] == un_v[e_reg, e_s].offsets[-1]).item()
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
out = {
    "gpu": gpu or torch.cuda.get_device_name(0),
    "pairs": 32 * 8, "elements": int(sum(len(rows[r]) for r in range(32)) * 8),
    "haplotype_bases": int(h.offsets[-1]), "track_values": int(t.offsets[-1]),
    "variants": int(v.offsets[-1]),
    **{f"ms_per_call_{k}": r for k, r in res.items()},
    "library_calls": {"tracks_1_pair": n_calls(sp_t, ([0], [0])), "tracks_256_pairs": n_calls(sp_t, idx),
                      "no_tracks_1_pair": n_calls(sp_n, ([0], [0])), "no_tracks_256_pairs": n_calls(sp_n, idx),
                      "variants_1_pair": n_calls(sp_v, ([0], [0])), "variants_256_pairs": n_calls(sp_v, idx),
                      "variant_windows_1_pair": n_calls(sp_w, ([0], [0])), "variant_windows_256_pairs": n_calls(sp_w, idx),
                      "unspliced_variants_over_E": n_calls(un_v, (e_reg, e_s))},
}
print(json.dumps(out))
if a.out:
    Path(a.out).mkdir(parents=True, exist_ok=True)
    (Path(a.out) / "probe_spliced.json").write_text(json.dumps(out, indent=1) + "\n")
