"""Generate tests/golden/*.npz from the UNMODIFIED reference -- TEST INFRASTRUCTURE ONLY.

Runs only where the reference is at hand (PTWT_REFERENCE_SRC); the fixtures are committed so that a
machine without the reference can still check the CUDA path and the oracle port against numbers
the reference itself produced.

    PTWT_REFERENCE_SRC=<reference checkout>/src python -m oracle.make_golden
"""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np
import torch

from oracle.ref_import import import_reference

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"

CASES = [
    # family, dtype, wavelet, mode, level, shape, axes
    ("wavedec", "float32", "haar", "zero", 2, (16,), None),          # BASELINE.json configs[0] (README example)
    ("wavedec", "float64", "db2", "reflect", 3, (2, 65), None),
    ("wavedec", "float32", "db4", "symmetric", None, (3, 64), None),
    ("wavedec", "float64", "sym5", "periodic", 2, (2, 3, 50), None),
    ("wavedec", "float64", "db3", "constant", 2, (4, 31, 3), -2),
    ("wavedec", "float64", "db5", "symmetric", 1, (2, 7), None),      # symmetric pad longer than the signal
    ("wavedec2", "float32", "db4", "reflect", 2, (2, 64, 64), None),
    ("wavedec2", "float64", "db2", "zero", 2, (33, 31), None),
    ("wavedec2", "float64", "sym4", "periodic", None, (2, 3, 40, 56), None),
    ("wavedec2", "float32", "haar", "constant", 3, (1, 32, 48), None),
    ("wavedec2", "float64", "db3", "symmetric", 2, (2, 30, 5, 37), (1, 3)),
    ("wavedec3", "float32", "sym4", "zero", 2, (2, 32, 32, 32), None),
    ("wavedec3", "float64", "db2", "reflect", 2, (17, 18, 19), None),
    ("wavedec3", "float64", "haar", "periodic", None, (2, 16, 20, 24), None),
    ("wavedec3", "float64", "db2", "symmetric", 1, (2, 12, 3, 14, 16), (1, 3, 4)),
    ("matrix", "float64", "haar", "zero", 2, (2, 32), None),
    ("matrix", "float64", "db6", "zero", None, (3, 256), None),
    ("matrix", "float32", "db4", "zero", 3, (2, 128), None),
    ("matrix", "float64", "db2", "reflect", 3, (2, 101), None),        # odd lengths -> padded levels
    ("matrix", "float64", "sym5", "zero", 2, (4, 64), None),
    ("matrix_gs", "float64", "db4", "zero", 2, (2, 64), None),         # gramschmidt orthogonalisation
    # separable 2-D / 3-D boundary-wavelet transforms (SURVEY.md section 8f row 2); appended so that the
    # random inputs of the cases above stay what they were
    ("matrix2", "float64", "db2", "zero", 2, (2, 32, 24), None),
    ("matrix2", "float64", "db3", "reflect", 2, (3, 33, 27), None),    # odd extents -> padded levels
    ("matrix2", "float32", "haar", "zero", 3, (1, 32, 32), None),
    ("matrix2", "float64", "sym4", "symmetric", 2, (2, 37, 3, 40), (1, 3)),
    ("matrix3", "float64", "db2", "zero", 2, (2, 16, 20, 24), None),
    ("matrix3", "float64", "haar", "constant", 2, (9, 10, 11), None),  # odd extents, no batch dimension
]


def _flatten(coeffs):
    out = []
    for el in coeffs:
        if isinstance(el, torch.Tensor):
            out.append(el)
        elif isinstance(el, dict):
            out.extend(el[k] for k in ("aad", "ada", "add", "daa", "dad", "dda", "ddd"))
        else:
            out.extend(el)
    return out


def main() -> None:
    ptwt = import_reference()
    OUT.mkdir(parents=True, exist_ok=True)
    arrays = {}
    manifest = []
    g = torch.Generator().manual_seed(20260923)
    for i, (family, dtype, wav, mode, level, shape, axes) in enumerate(CASES):
        dt = getattr(torch, dtype)
        if i == 0:
            x = torch.tensor([0, 1, 2, 3, 4, 5, 6, 7, 7, 6, 5, 4, 3, 2, 1, 0], dtype=dt)
        else:
            x = torch.randn(shape, generator=g, dtype=torch.float64).to(dt)
        if family == "wavedec":
            kw = {} if axes is None else {"axis": axes}
            c = ptwt.wavedec(x, wav, mode=mode, level=level, **kw)
            r = ptwt.waverec(c, wav, **kw)
        elif family == "wavedec2":
            kw = {} if axes is None else {"axes": axes}
            c = ptwt.wavedec2(x, wav, mode=mode, level=level, **kw)
            r = ptwt.waverec2(c, wav, **kw)
        elif family == "wavedec3":
            kw = {} if axes is None else {"axes": axes}
            c = ptwt.wavedec3(x, wav, mode=mode, level=level, **kw)
            r = ptwt.waverec3(c, wav, **kw)
        elif family == "matrix2":
            kw = {} if axes is None else {"axes": axes}
            c = ptwt.MatrixWavedec2(wav, level, odd_coeff_padding_mode=mode, **kw)(x)
            r = ptwt.MatrixWaverec2(wav, **kw)(c)
        elif family == "matrix3":
            kw = {} if axes is None else {"axes": axes}
            c = ptwt.MatrixWavedec3(wav, level, odd_coeff_padding_mode=mode, **kw)(x)
            r = ptwt.MatrixWaverec3(wav, **kw)(c)
        else:
            meth = "gramschmidt" if family == "matrix_gs" else "qr"
            c = ptwt.MatrixWavedec(wav, level, orthogonalization=meth, odd_coeff_padding_mode=mode)(x)
            r = ptwt.MatrixWaverec(wav, orthogonalization=meth)(c)
        flat = _flatten(c)
        arrays[f"c{i}_x"] = x.numpy()
        for j, t in enumerate(flat):
            arrays[f"c{i}_o{j}"] = t.contiguous().numpy()
        arrays[f"c{i}_rec"] = r.contiguous().numpy()
        manifest.append({"id": i, "family": family, "dtype": dtype, "wavelet": wav, "mode": mode, "level": level,
                         "shape": list(shape), "axes": axes if axes is None or isinstance(axes, int) else list(axes),
                         "n_out": len(flat)})
    # boundary operators themselves (small sizes), dense
    for wav, n in (("db2", 16), ("db4", 32), ("db6", 64)):
        a = ptwt.matmul_transform.construct_boundary_a(wav, n, dtype=torch.float64).to_dense()
        s = ptwt.matmul_transform.construct_boundary_s(wav, n, dtype=torch.float64).to_dense()
        arrays[f"A_{wav}_{n}"] = a.numpy()
        arrays[f"S_{wav}_{n}"] = s.numpy()
    np.savez_compressed(OUT / "reference_vectors.npz", **arrays)
    (OUT / "reference_vectors.json").write_text(json.dumps({
        "generated_by": "oracle/make_golden.py",
        "reference_commit": "6c3b62c1fe02ddca0f0d8662d73582e9f9be48e5",
        "torch": torch.__version__,
        "cases": manifest,
    }, indent=1))
    print("wrote", OUT / "reference_vectors.npz", sum(v.nbytes for v in arrays.values()), "bytes raw")


if __name__ == "__main__":
    main()
