"""Golden vectors for the `variants` cores produced by EXECUTING the reference's own pure-numpy twins.

Needs a checkout of the original GenVarLoader project:

    python tests/golden/make_pyref_variants_golden.py <genvarloader checkout>

The reference keeps dtype-preserving numpy fallbacks next to its Rust cores (python/genvarloader/_dataset/_flat_variants.py:
`_gather_rows_numpy` :545, `_compact_keep_numpy` :567, `_fill_empty_scalar_numpy` :624, `_fill_empty_seq_numpy` :660,
`_fill_empty_fixed_numpy` :721) and the numba / numpy originals of the window assembly (`_flat_flanks.py`: `build_token_lut`
:23, `_slice_flanks` :43, `_assemble_alt_windows` :96).  Their modules import the compiled extension, so the function bodies
are lifted with `ast` and executed with numpy only -- nothing is re-implemented here.  The cases are larger and more ragged
than the frozen hypothesis goldens (rows of up to 150 variants, runs of empty rows, empty first / last rows, alleles of up to 24 items).

Output (pickle-free, same c{case}_a{arg} / c{case}_g{j} layout as make_golden.py): tests/golden/ref_pyref_<name>.npz.
"""
from __future__ import annotations

import ast
import sys
from pathlib import Path

import numpy as np

REF_SUBDIR = Path("python/genvarloader/_dataset")
# no fixture file may exceed 1 MB: `fill_empty_seq` keeps only the cases of at most this many bytes (71 of 80)
MAX_CASE_BYTES = {"fill_empty_seq": 100_000}
DST = Path(__file__).parent


def _lift(path: Path, names: set) -> dict:
    tree = ast.parse(path.read_text())
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    assert {n.name for n in body} == names, names - {n.name for n in body}
    ns: dict = {"np": np, "_normalize_token_alphabet": lambda a: a.encode("ascii") if isinstance(a, str) else bytes(a)}
    exec(compile(ast.Module(body=body, type_ignores=[]), str(path), "exec"), ns)
    return ns


def _save(name: str, cases: list) -> None:
    cap = MAX_CASE_BYTES.get(name)
    if cap is not None:
        cases = [c for c in cases if sum(np.asarray(a).nbytes for a in (*c[0], *c[1])) <= cap]
    out = {"n_cases": np.array(len(cases), np.int64), "n_args": np.array(len(cases[0][0]), np.int64),
           "n_gold": np.array(len(cases[0][1]), np.int64)}
    for ci, (args, gold) in enumerate(cases):
        for j, a in enumerate(args):
            out[f"c{ci}_a{j}"] = np.asarray(a)
        out[f"c{ci}_none"] = np.zeros(0, np.int64)
        for j, g in enumerate(gold):
            out[f"c{ci}_g{j}"] = np.asarray(g)
    np.savez_compressed(DST / f"ref_pyref_{name}.npz", **out)
    print(f"{name}: {len(cases)} cases -> ref_pyref_{name}.npz")


def _offsets(rng, n, max_len, empty_frac):
    ln = rng.integers(1, max_len + 1, n)
    ln[rng.random(n) < empty_frac] = 0
    if n > 6:  # a run of consecutive empty rows, an empty first and last row
        ln[2:5] = 0
        ln[0] = ln[-1] = 0
    return np.concatenate([[0], np.cumsum(ln)]).astype(np.int64)


def main(ref: Path) -> None:
    fv = _lift(ref / "_flat_variants.py", {"_gather_rows_numpy", "_compact_keep_numpy", "_fill_empty_scalar_numpy",
                                           "_fill_empty_seq_numpy", "_fill_empty_fixed_numpy"})
    ff = _lift(ref / "_flat_flanks.py", {"build_token_lut", "_slice_flanks", "_assemble_alt_windows"})
    rng = np.random.default_rng(20260)
    gather, compact, fscalar, fseq, ffixed, alt_win = [], [], [], [], [], []
    for ci in range(40):
        n_rows = int(rng.integers(1, 60))
        n_slots = 2 * n_rows + 2
        so = _offsets(rng, n_slots, int(rng.choice([3, 40, 150])), 0.3)
        go = np.stack([so[:-1], so[1:]])
        goi = rng.integers(0, n_slots, n_rows).astype(np.int64)
        for dt in (np.int32, np.float32):
            data = (rng.integers(-2**31, 2**31 - 1, so[-1]).astype(np.int32) if dt is np.int32
                    else rng.standard_normal(so[-1]).astype(np.float32))
            gather.append(((goi, go, data), fv["_gather_rows_numpy"](goi, go, data)))
        off = _offsets(rng, n_rows, int(rng.choice([2, 30, 100])), float(rng.choice([0.0, 0.4, 0.9])))
        n = int(off[-1])
        keep = rng.random(n) < rng.choice([0.0, 0.5, 1.0])
        for dt in (np.int32, np.float32):
            vals = rng.integers(-99, 99, n).astype(dt)
            compact.append(((vals, off, keep), fv["_compact_keep_numpy"](vals, off, keep)))
            fill = dt(rng.integers(-9, 9))
            fscalar.append(((vals, off, fill), fv["_fill_empty_scalar_numpy"](vals, off, fill)))
            inner = int(rng.integers(1, 9))
            fx = rng.integers(-99, 99, n * inner).astype(dt)
            ffixed.append(((fx, off, np.int64(inner), fill), fv["_fill_empty_fixed_numpy"](fx, off, inner, fill)))
        seq_off = np.concatenate([[0], np.cumsum(rng.integers(0, 25, n))]).astype(np.int64)
        for dt, dummy in ((np.uint8, np.frombuffer(b"NN", np.uint8)), (np.int32, np.array([4, 4, 4], np.int32))):
            data = rng.integers(0, 200, seq_off[-1]).astype(dt)
            fseq.append(((data, off, seq_off, dummy), fv["_fill_empty_seq_numpy"](data, off, seq_off, dummy)))
        # flank5 . alt . flank3 from per-variant reference windows (the byte level of `alt_window`)
        L = int(rng.integers(0, 12))
        nv = int(rng.integers(0, 50))
        span = rng.integers(1, 20, nv)
        rw_off = np.concatenate([[0], np.cumsum(span + 2 * L)]).astype(np.int64)
        rw = rng.integers(65, 90, rw_off[-1]).astype(np.uint8)
        a_off = np.concatenate([[0], np.cumsum(rng.integers(1, 30, nv))]).astype(np.int64)
        a_data = rng.integers(65, 90, a_off[-1]).astype(np.uint8)
        f5, f3 = ff["_slice_flanks"](rw, rw_off, L)
        alt_win.append(((rw, rw_off, a_data, a_off, np.int64(L)),
                        ff["_assemble_alt_windows"](f5.reshape(-1), f3.reshape(-1), a_data, a_off, L)))
    luts = []
    for alphabet, unk in ((b"ACGT", 4), ("ACGTN", 0), (b"ACGT", 1000), (bytes(range(65, 91)), 255)):
        lut, dt = ff["build_token_lut"](alphabet, unk)
        luts.append(((np.frombuffer(alphabet.encode() if isinstance(alphabet, str) else alphabet, np.uint8), np.int64(unk)), (lut,)))
    for name, cases in (("gather_rows", gather), ("compact_keep", compact), ("fill_empty_scalar", fscalar),
                        ("fill_empty_fixed", ffixed), ("fill_empty_seq", fseq), ("alt_windows", alt_win), ("token_lut", luts)):
        _save(name, cases)


if __name__ == "__main__":
    ref = Path(sys.argv[1]) / REF_SUBDIR if len(sys.argv) > 1 else None
    if ref is None or not ref.is_dir():
        sys.exit("usage: make_pyref_variants_golden.py <genvarloader checkout>")
    main(ref)
