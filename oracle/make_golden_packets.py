"""Generate tests/golden/packet_vectors.* from the UNMODIFIED reference's WaveletPacket / WaveletPacket2D --
TEST INFRASTRUCTURE ONLY (needs the reference, named by PTWT_REFERENCE_SRC).

    PTWT_REFERENCE_SRC=<reference checkout>/src python -m oracle.make_golden_packets
"""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np
import torch

from oracle.ref_import import import_reference

OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"

CASES = [
    # dim, dtype, wavelet, mode, maxlevel, shape, axes, separable
    (1, "float32", "db2", "reflect", 3, (2, 64), None, False),
    (1, "float64", "haar", "zero", 3, (3, 32), None, False),
    (1, "float64", "db3", "boundary", 2, (2, 64), None, False),
    (1, "float64", "db2", "symmetric", 2, (2, 40, 3), -2, False),
    (1, "float64", "db4", "periodic", 2, (65,), None, False),
    (2, "float32", "db2", "reflect", 2, (2, 32, 32), None, False),
    (2, "float64", "haar", "zero", 2, (1, 16, 24), None, True),
    (2, "float64", "db2", "boundary", 2, (2, 32, 32), None, True),
    (2, "float64", "db2", "constant", 2, (2, 20, 3, 24), (1, 3), False),
    (2, "float64", "db3", "symmetric", 2, (33, 31), None, True),
]


def main() -> None:
    ptwt = import_reference()
    arrays, manifest = {}, []
    g = torch.Generator().manual_seed(20260924)
    for i, (dim, dtype, wav, mode, maxlevel, shape, axes, separable) in enumerate(CASES):
        x = torch.randn(shape, generator=g, dtype=torch.float64).to(getattr(torch, dtype))
        if dim == 1:
            kw = {} if axes is None else {"axis": axes}
            wp = ptwt.WaveletPacket(x, wav, mode=mode, maxlevel=maxlevel, **kw)
            keys = wp.get_level(maxlevel, "natural")
        else:
            kw = {} if axes is None else {"axes": axes}
            wp = ptwt.WaveletPacket2D(x, wav, mode=mode, maxlevel=maxlevel, separable=separable, **kw)
            keys = wp.get_natural_order(maxlevel)
        wp.initialize(keys)
        every = sorted(k for k in wp.keys() if k != "")
        for k in every:
            arrays[f"p{i}_{k}"] = wp[k].contiguous().numpy()
        rec = wp.reconstruct()[""]
        arrays[f"p{i}_x"] = x.numpy()
        arrays[f"p{i}_rec"] = rec.contiguous().numpy()
        manifest.append({"id": i, "dim": dim, "dtype": dtype, "wavelet": wav, "mode": mode, "maxlevel": maxlevel,
                         "shape": list(shape), "axes": axes if axes is None or isinstance(axes, int) else list(axes),
                         "separable": separable, "keys": every})
    np.savez_compressed(OUT / "packet_vectors.npz", **arrays)
    (OUT / "packet_vectors.json").write_text(json.dumps({
        "generated_by": "oracle/make_golden_packets.py", "torch": torch.__version__, "cases": manifest}, indent=1))
    print("wrote", OUT / "packet_vectors.npz", sum(v.nbytes for v in arrays.values()), "bytes raw")


if __name__ == "__main__":
    main()
