"""bench.py's reference arm runs on the host cores alone: check the JSON contract (keys the driver reads) without a GPU.
The device arm's `--dump-outputs` is checked on the GPU."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "4",
                        "--warmup", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["unit"] == "bp/s" and j["higher_is_better"] is True
    for k in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in j, k
    assert j["steps"] == 4 and j["value"] > 0 and j["vs_baseline"] is None
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "bp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["config"]["workload"].startswith("cfg1") and j["config"]["window_bp"] == 16384


def test_ranks_other_than_zero_stay_silent():
    import os

    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "2",
                        "--warmup", "1", "--gpus", "2"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    assert not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_is_a_seeded_sample_within_budget(tmp_path):
    """--dump-outputs: float32 for uint8 / float32 outputs, float64 for int32 ones, and one seeded sample of window positions
    shared by every array when the batch would exceed the byte budget."""
    import numpy as np
    import torch

    import bench
    from genvarloader_b200._types import AnnotatedHaps

    rng = np.random.default_rng(1)
    L = 1000
    oh = torch.from_numpy(rng.integers(0, 2, (3, 2, L, 4), dtype=np.uint8))
    trk = torch.from_numpy(rng.standard_normal((3, 2, 2, L)).astype(np.float32))
    assert bench.dump_outputs(tmp_path / "full", (oh, trk), "onehot") == {"haplotypes": (3, 2, L, 4), "tracks": (3, 2, 2, L)}
    assert (np.load(tmp_path / "full" / "haplotypes.npy") == oh.numpy()).all()

    # 144 B per window position (24 uint8 + 12 float32 values, all written as float32) and two .npy headers: 250 positions
    budget = 144 * 250 + 2 * bench.NPY_HEADER_BYTES + 50
    for d in ("a", "b"):
        assert bench.dump_outputs(tmp_path / d, (oh, trk), "onehot", budget=budget) == {"haplotypes": (3, 2, 250, 4),
                                                                                        "tracks": (3, 2, 2, 250)}
    pos = np.sort(np.random.default_rng(0).choice(L, 250, replace=False))
    for name, full, ax in (("haplotypes", oh.numpy(), 2), ("tracks", trk.numpy(), 3)):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and (a == b).all()
        assert (a == np.take(full, pos, axis=ax)).all()
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= budget

    big = np.int32(2**31 - 1)
    ann = AnnotatedHaps(torch.from_numpy(rng.integers(0, 255, (2, 2, L), dtype=np.uint8)),
                        torch.from_numpy(rng.integers(-1, 10**7, (2, 2, L), dtype=np.int32)),
                        torch.full((2, 2, L), big, dtype=torch.int32))
    bench.dump_outputs(tmp_path / "ann", ann, "annotated")
    assert np.load(tmp_path / "ann" / "haps.npy").dtype == np.float32
    for name in ("var_idxs", "ref_coords"):
        a = np.load(tmp_path / "ann" / f"{name}.npy")
        assert a.dtype == np.float64 and (a == getattr(ann, name).numpy()).all()


def test_dump_outputs_needs_the_b200_arm(tmp_path):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(cuda_device, tmp_path):
    """Exactly --steps steps are timed, and --dump-outputs holds the last one's batch: the same whatever the warm-up, and
    equal to the oracle on that step's (region, sample) pairs."""
    import numpy as np

    import bench
    from genvarloader_b200 import synth
    from oracle import oracle as O

    lines = {}
    for warmup in (1, 9):
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--workload", "cfg1", "--steps", "4", "--warmup", str(warmup),
                            "--min-calls", "2", "--cpu-seconds", "0.1", "--dump-outputs", str(tmp_path / f"w{warmup}")],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        lines[warmup] = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    j = lines[1]
    ring, calls = j["pipeline"]["batches_per_device_call"], j["pipeline"]["device_calls_per_timed_block"]
    assert j["steps"] == 4 and (ring, calls) == (2, 2) and j["timed_block_ms"] > 0
    assert lines[9]["pipeline"]["warmup_blocks"] >= 3
    got = np.load(tmp_path / "w1" / "haplotypes.npy")
    assert got.dtype == np.float32 and (got == np.load(tmp_path / "w9" / "haplotypes.npy")).all()

    seed = 3  # bench.py's default --seed
    w, d = bench.build_workload("cfg1", seed)
    pairs, L = w["pairs"], w["window"]
    idx = bench.draw_indices(d, ring * pairs, seed + 100 + calls - 1)[(ring - 1) * pairs:]
    regions, goi, to_rc, _ = synth.batch_args(d, idx // d.n_samples, idx % d.n_samples, jitter=0)
    regions[:, 2] = regions[:, 1] + L
    exp, _ = O.reconstruct_haplotypes_fused(regions, np.zeros(goi.shape, np.int32), goi, d.geno_offsets, d.geno_v_idxs,
                                            d.v_starts, d.ilens, d.alt_alleles, d.alt_offsets, d.reference, d.ref_offsets,
                                            ord("N"), L, None, None, to_rc)
    assert got.shape == (pairs, d.ploidy, L, 4)
    assert (got == O.onehot(exp).reshape(got.shape)).all()
