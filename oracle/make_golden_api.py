"""Generate tests/golden/reference_api.* from the UNMODIFIED reference -- TEST INFRASTRUCTURE ONLY.

What the CPU tests used to ask the reference itself at run time, recorded once so that they run anywhere: the
signatures of the public callables, the stderr warning of the separable matrix level walk, the packet orders, the
outputs of the convolution transforms (as SHA-256 digests of the exact bytes: the port must be bit-identical) and of
the boundary-wavelet and fully separable transforms (a fixed sample of each output, compared against a tolerance).
The inputs are drawn from seeded torch generators and recorded by digest, so a changed random stream is reported as
such instead of as a wrong transform.

    PTWT_REFERENCE_SRC=<reference checkout>/src python -m oracle.make_golden_api
"""
from __future__ import annotations

import contextlib
import hashlib
import inspect
import io
import json
from pathlib import Path

import numpy as np
import torch

from oracle.ref_import import import_reference

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"

SIGNATURE_FUNCTIONS = ("wavedec", "waverec", "wavedec2", "waverec2", "wavedec3", "waverec3", "fswavedec2", "fswavedec3",
                       "fswaverec2", "fswaverec3")
SIGNATURE_CLASSES = ("MatrixWavedec", "MatrixWaverec", "MatrixWavedec2", "MatrixWaverec2", "MatrixWavedec3",
                     "MatrixWaverec3")
PACKET_CLASSES = ("WaveletPacket", "WaveletPacket2D")
MODES = ("zero", "constant", "reflect", "periodic", "symmetric")


def params(fn):
    """[name, kind, repr(default)] of every parameter but self and **kwargs (the form the tests compare)."""
    return [[n, p.kind.name, repr(p.default)] for n, p in inspect.signature(fn).parameters.items()
            if n != "self" and p.kind is not inspect.Parameter.VAR_KEYWORD]


def digest(t: torch.Tensor) -> str:
    t = t.detach().contiguous()
    return f"{str(t.dtype)}{tuple(t.shape)}:" + hashlib.sha256(t.numpy().tobytes()).hexdigest()


#: values kept per output tensor of the tolerance comparisons (evenly spaced, first and last included)
SAMPLE = 128


def sample_index(numel: int) -> np.ndarray:
    return np.unique(np.linspace(0, numel - 1, min(numel, SAMPLE)).round().astype(np.int64))


def sample(t: torch.Tensor) -> np.ndarray:
    flat = t.detach().contiguous().reshape(-1).numpy()
    return flat[sample_index(flat.size)]


def flatten(coeffs):
    out = []
    for el in coeffs:
        if isinstance(el, torch.Tensor):
            out.append(el)
        elif isinstance(el, dict):
            out.extend(el[k] for k in sorted(el))
        else:
            out.extend(el)
    return out


def conv_cases(ptwt) -> dict:
    """Digests of the convolution transforms for the inputs test_port_equals_the_reference draws (seed 7)."""
    g = torch.Generator().manual_seed(7)
    out = {}
    for dtype in (torch.float32, torch.float64):
        for mode in MODES:
            key = f"{str(dtype)[6:]}_{mode}"
            x = torch.randn(2, 37, 40, generator=g, dtype=torch.float64).to(dtype)
            r = ptwt.wavedec2(x, "db2", mode=mode, level=2)
            x3 = torch.randn(2, 13, 14, 15, generator=g, dtype=torch.float64).to(dtype)
            r3 = ptwt.wavedec3(x3, "db2", mode=mode, level=1)
            out[key] = {
                "x": digest(x), "x3": digest(x3),
                "wavedec": [digest(t) for t in flatten(ptwt.wavedec(x, "db3", mode=mode, level=2))],
                "wavedec2": [digest(t) for t in flatten(r)], "waverec2": digest(ptwt.waverec2(r, "db2")),
                "wavedec3": [digest(t) for t in flatten(r3)], "waverec3": digest(ptwt.waverec3(r3, "db2")),
            }
    return out


def put(arrays: dict, shapes: dict, key: str, t: torch.Tensor) -> None:
    arrays[key] = sample(t)
    shapes[key] = list(t.shape)


def matrix_cases(ptwt, arrays: dict, shapes: dict) -> None:
    """Boundary-wavelet transforms, 1-D .. 3-D, every padding mode of odd extents (seed 8)."""
    g = torch.Generator().manual_seed(8)
    x = torch.randn(3, 96, generator=g, dtype=torch.float64)
    r = ptwt.MatrixWavedec("db4", 3)(x)
    shapes["m1_x"] = digest(x)
    for j, t in enumerate(r):
        put(arrays, shapes, f"m1_o{j}", t)
    put(arrays, shapes, "m1_rec", ptwt.MatrixWaverec("db4")(r))
    for mode in MODES:
        x2 = torch.randn(2, 27, 34, generator=g, dtype=torch.float64)
        r = ptwt.MatrixWavedec2("db3", 2, odd_coeff_padding_mode=mode)(x2)
        shapes[f"m2_{mode}_x"] = digest(x2)
        for j, t in enumerate(flatten(r)):
            put(arrays, shapes, f"m2_{mode}_o{j}", t)
        put(arrays, shapes, f"m2_{mode}_rec", ptwt.MatrixWaverec2("db3")(r))
        x3 = torch.randn(2, 9, 12, 11, generator=g, dtype=torch.float64)
        r = ptwt.MatrixWavedec3("db2", 2, odd_coeff_padding_mode=mode)(x3)
        shapes[f"m3_{mode}_x"] = digest(x3)
        for j, t in enumerate(flatten(r)):
            put(arrays, shapes, f"m3_{mode}_o{j}", t)
        put(arrays, shapes, f"m3_{mode}_rec", ptwt.MatrixWaverec3("db2")(r))


def separable_cases(ptwt, arrays: dict, shapes: dict) -> dict:
    """fswavedec2 / fswavedec3 bands and reconstructions, with the band keys in the reference's order."""
    g = torch.Generator().manual_seed(9)
    keys = {}
    x = torch.randn(2, 33, 40, generator=g, dtype=torch.float64)
    shapes["fs2_x"] = digest(x)
    for mode in ("zero", "reflect", "constant", "periodic"):
        fs = ptwt.fswavedec2(x, "db2", mode=mode, level=2)
        put(arrays, shapes, f"fs2_{mode}_a", fs[0])
        for lv, d in enumerate(fs[1:], 1):
            keys["fs2"] = list(d.keys())
            for k, t in d.items():
                put(arrays, shapes, f"fs2_{mode}_{lv}{k}", t)
        put(arrays, shapes, f"fs2_{mode}_rec", ptwt.fswaverec2(fs, "db2"))
    x3 = torch.randn(2, 12, 13, 14, generator=g, dtype=torch.float64)
    fs = ptwt.fswavedec3(x3, "db2", mode="zero", level=1)
    shapes["fs3_x"] = digest(x3)
    keys["fs3"] = list(fs[1].keys())
    for k, t in fs[1].items():
        put(arrays, shapes, f"fs3_{k}", t)
    return keys


def level_walk_warnings(ptwt) -> list[str]:
    """stderr of the reference's MatrixWavedec3 / MatrixWavedec2 when the level walk stops early."""
    errs = []
    for make, shape in ((lambda: ptwt.MatrixWavedec3("db2", 3), (12, 9, 16)),
                        (lambda: ptwt.MatrixWavedec2("db3", 3), (20, 12))):
        buf = io.StringIO()
        with contextlib.redirect_stderr(buf):
            make()(torch.randn(shape, dtype=torch.float64))
        errs.append(buf.getvalue())
    return errs


def main() -> None:
    ptwt = import_reference()
    arrays, shapes = {}, {}
    matrix_cases(ptwt, arrays, shapes)
    manifest = {
        "generated_by": "oracle/make_golden_api.py",
        "reference_commit": "6c3b62c1fe02ddca0f0d8662d73582e9f9be48e5",
        "torch": torch.__version__,
        "signatures": {name: params(getattr(ptwt, name)) for name in SIGNATURE_FUNCTIONS}
        | {name: params(inspect.unwrap(getattr(ptwt, name).__init__)) for name in SIGNATURE_CLASSES}
        | {name: [p[0] for p in params(inspect.unwrap(getattr(ptwt, name).__init__))] for name in PACKET_CLASSES},
        "level_walk_stderr": level_walk_warnings(ptwt),
        "packet_orders": {str(lev): {"gray": ptwt.WaveletPacket.get_level(lev),
                                     "natural": ptwt.WaveletPacket.get_level(lev, "natural"),
                                     "freq_2d": ptwt.WaveletPacket2D.get_freq_order(lev),
                                     "natural_2d": ptwt.WaveletPacket2D.get_natural_order(lev)} for lev in (0, 1, 2, 3)},
        "conv_digests": conv_cases(ptwt),
        "separable_keys": separable_cases(ptwt, arrays, shapes),
        "sampled_shapes": shapes,          # output key -> shape; input key (*_x) -> digest
    }
    np.savez_compressed(OUT / "reference_api.npz", **arrays)
    (OUT / "reference_api.json").write_text(json.dumps(manifest, indent=1) + "\n")
    print("wrote", OUT / "reference_api.npz", sum(v.nbytes for v in arrays.values()), "bytes raw")


if __name__ == "__main__":
    main()
