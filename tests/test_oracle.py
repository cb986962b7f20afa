"""The oracle is pinned: port == golden vectors produced by the unmodified reference, port == what the
reference computed from the same seeded inputs, closed form == port, known-answer tests that the
reference's own test-suite holds (no GPU needed)."""
from __future__ import annotations

import json

import numpy as np
import pytest
import torch

from conftest import GOLDEN, flatten_coeffs
from oracle import closed_form as CF
from oracle import ptwt_port as P
from oracle import make_golden_api as G
from pytorch_wavelet_toolbox_b200._wavelets import BuiltinWavelet, as_wavelet


def reference_api() -> dict:
    ref = json.loads((GOLDEN / "reference_api.json").read_text())
    ref["arrays"] = np.load(GOLDEN / "reference_api.npz")
    return ref


def digest(t: torch.Tensor) -> str:
    return G.digest(t)


def check_sampled(ref, key: str, got: torch.Tensor, tol: float | None = None) -> None:
    """An input: its digest equals the one recorded.  An output: its shape equals the reference's, and at the
    recorded sample of elements |got - reference| <= tol."""
    want = ref["sampled_shapes"][key]
    if tol is None:
        assert digest(got) == want, f"{key}: torch's seeded random stream changed"
        return
    assert list(got.shape) == want, (key, tuple(got.shape), want)
    err = np.abs(G.sample(got) - ref["arrays"][key]).max()
    assert err < tol, (key, err)


def _run_port(case, x):
    fam, wav, mode, level, axes = case["family"], case["wavelet"], case["mode"], case["level"], case["axes"]
    if isinstance(axes, list):
        axes = tuple(axes)
    if fam == "wavedec":
        kw = {} if axes is None else {"axis": axes}
        c = P.wavedec(x, wav, mode=mode, level=level, **kw)
        return c, P.waverec(c, wav, **kw)
    if fam == "wavedec2":
        kw = {} if axes is None else {"axes": axes}
        c = P.wavedec2(x, wav, mode=mode, level=level, **kw)
        return c, P.waverec2(c, wav, **kw)
    if fam == "wavedec3":
        kw = {} if axes is None else {"axes": axes}
        c = P.wavedec3(x, wav, mode=mode, level=level, **kw)
        return c, P.waverec3(c, wav, **kw)
    if fam in ("matrix2", "matrix3"):
        kw = {} if axes is None else {"axes": axes}
        dec, rec = ((P.MatrixWavedec2, P.MatrixWaverec2) if fam == "matrix2" else (P.MatrixWavedec3, P.MatrixWaverec3))
        c = dec(wav, level, odd_coeff_padding_mode=mode, **kw)(x)
        return c, rec(wav, **kw)(c)
    meth = "gramschmidt" if fam == "matrix_gs" else "qr"
    c = P.MatrixWavedec(wav, level, orthogonalization=meth, odd_coeff_padding_mode=mode)(x)
    return c, P.MatrixWaverec(wav, orthogonalization=meth)(c)


def test_port_reproduces_golden_vectors(golden):
    manifest, arrays = golden
    for case in manifest["cases"]:
        i = case["id"]
        x = torch.from_numpy(arrays[f"c{i}_x"])
        c, rec = _run_port(case, x)
        flat = flatten_coeffs(c)
        assert len(flat) == case["n_out"]
        exact = not case["family"].startswith("matrix")
        for j, t in enumerate(flat):
            want = arrays[f"c{i}_o{j}"]
            if exact:  # same torch ops in the same order -> bit-identical
                assert np.array_equal(t.numpy(), want), (case, j)
            else:      # sparse vs dense construction of the same operator
                tol = 1e-5 if case["dtype"] == "float32" else 1e-12
                assert np.abs(t.numpy() - want).max() <= tol, (case, j)
        tol = 1e-4 if case["dtype"] == "float32" else 1e-11
        assert np.abs(rec.numpy() - arrays[f"c{i}_rec"]).max() <= tol


def test_port_boundary_operators_match_golden(golden):
    _, arrays = golden
    for wav, n in (("db2", 16), ("db4", 32), ("db6", 64)):
        w = as_wavelet(wav)
        lo = torch.tensor(w.dec_lo, dtype=torch.float64)
        hi = torch.tensor(w.dec_hi, dtype=torch.float64)
        a = P.boundary_matrix(lo, hi, n)
        assert np.abs(a.numpy() - arrays[f"A_{wav}_{n}"]).max() < 1e-13
        rlo = torch.tensor(w.rec_lo, dtype=torch.float64).flip(0)
        rhi = torch.tensor(w.rec_hi, dtype=torch.float64).flip(0)
        s = P.boundary_matrix(rlo, rhi, n).T
        assert np.abs(s.numpy() - arrays[f"S_{wav}_{n}"]).max() < 1e-13
        # reference tests/test_matrix_fwt.py:91-121: orthogonal, inverse error < 1e-8
        eye = torch.eye(n, dtype=torch.float64)
        assert (a @ a.T - eye).abs().max() < 1e-8
        assert (s @ a - eye).abs().max() < 1e-8


def test_port_equals_the_reference():
    """The port against what the unmodified reference computed from the same seeded inputs (tests/golden/
    reference_api.*): the convolution transforms bit for bit (SHA-256 of the exact bytes), the boundary-wavelet
    transforms within rounding at a fixed sample of every output."""
    ref = reference_api()
    g = torch.Generator().manual_seed(7)
    for dtype in (torch.float32, torch.float64):
        for mode in ("zero", "constant", "reflect", "periodic", "symmetric"):
            want = ref["conv_digests"][f"{str(dtype)[6:]}_{mode}"]
            x = torch.randn(2, 37, 40, generator=g, dtype=torch.float64).to(dtype)
            x3 = torch.randn(2, 13, 14, 15, generator=g, dtype=torch.float64).to(dtype)
            assert digest(x) == want["x"] and digest(x3) == want["x3"], "torch's seeded random stream changed"
            assert [digest(t) for t in G.flatten(P.wavedec(x, "db3", mode=mode, level=2))] == want["wavedec"], mode
            p = P.wavedec2(x, "db2", mode=mode, level=2)
            assert [digest(t) for t in G.flatten(p)] == want["wavedec2"], mode
            assert digest(P.waverec2(p, "db2")) == want["waverec2"], mode
            p = P.wavedec3(x3, "db2", mode=mode, level=1)
            assert [digest(t) for t in G.flatten(p)] == want["wavedec3"], mode
            assert digest(P.waverec3(p, "db2")) == want["waverec3"], mode
    g = torch.Generator().manual_seed(8)
    x = torch.randn(3, 96, generator=g, dtype=torch.float64)
    p = P.MatrixWavedec("db4", 3)(x)
    check_sampled(ref, "m1_x", x)
    for j, t in enumerate(p):
        check_sampled(ref, f"m1_o{j}", t, 1e-13)
    check_sampled(ref, "m1_rec", P.MatrixWaverec("db4")(p), 1e-12)
    # separable 2-D / 3-D boundary-wavelet transforms (SURVEY 8f row 2): even and odd extents, every mode of the
    # odd-sample padding
    for odd_mode in ("zero", "constant", "reflect", "periodic", "symmetric"):
        x2 = torch.randn(2, 27, 34, generator=g, dtype=torch.float64)
        p = P.MatrixWavedec2("db3", 2, odd_coeff_padding_mode=odd_mode)(x2)
        check_sampled(ref, f"m2_{odd_mode}_x", x2)
        for j, t in enumerate(G.flatten(p)):
            check_sampled(ref, f"m2_{odd_mode}_o{j}", t, 1e-12)
        check_sampled(ref, f"m2_{odd_mode}_rec", P.MatrixWaverec2("db3")(p), 1e-11)
        x3 = torch.randn(2, 9, 12, 11, generator=g, dtype=torch.float64)
        p = P.MatrixWavedec3("db2", 2, odd_coeff_padding_mode=odd_mode)(x3)
        check_sampled(ref, f"m3_{odd_mode}_x", x3)
        for j, t in enumerate(G.flatten(p)):
            check_sampled(ref, f"m3_{odd_mode}_o{j}", t, 1e-12)
        check_sampled(ref, f"m3_{odd_mode}_rec", P.MatrixWaverec3("db2")(p), 1e-11)


def test_known_answer_ripples_haar():
    """Unscaled Haar, 'Ripples in Mathematics' p.7 -- the reference's tests/test_convolution_fwt.py:98-118."""

    class MyHaar:
        name = "unscaled Haar"
        filter_bank = ([0.5, 0.5], [-0.5, 0.5], [0.5, 0.5], [0.5, -0.5])
        dec_lo, dec_hi, rec_lo, rec_hi = filter_bank
        dec_len = rec_len = 2

        def __len__(self):
            return 2

    x = torch.tensor([56.0, 40.0, 8.0, 24.0, 48.0, 48.0, 40.0, 16.0])
    c = P.wavedec(x, MyHaar(), level=3)
    want = [[35.0], [-3.0], [16.0, 10.0], [8.0, -8.0, 0.0, 12.0]]
    for got, w in zip(c, want):
        assert torch.equal(got.reshape(-1), torch.tensor(w))


def test_known_answer_readme_example():
    """The reference's README.rst:77-87 (BASELINE.json configs[0])."""
    x = torch.tensor([0, 1, 2, 3, 4, 5, 6, 7, 7, 6, 5, 4, 3, 2, 1, 0], dtype=torch.float32)
    c = P.wavedec(x, "haar", mode="zero", level=2)
    assert torch.allclose(c[0], torch.tensor([3.0, 11.0, 11.0, 3.0]), atol=1e-6)
    assert torch.allclose(c[1], torch.tensor([-2.0, -2.0, 2.0, 2.0]), atol=1e-6)
    s = 0.5 ** 0.5
    assert torch.allclose(c[2], torch.tensor([-s] * 4 + [s] * 4), atol=1e-6)
    assert (P.waverec(c, "haar") - x).abs().max() < 1e-6


def test_symmetric_extension_matches_numpy():
    """The reference's tests/test_util.py:54-73."""
    rng = np.random.default_rng(0)
    for size in (5, 6, 9):
        x = rng.standard_normal(size)
        for pads in ((2, 2), (0, 0), (1, 0), (0, 1), (2, 1), (1, 2), (10, 10), (23, 4)):
            want = np.pad(x, pads, mode="symmetric")
            got = [x[CF.ext_index(j, size, "symmetric")] for j in range(-pads[0], size + pads[1])]
            assert np.array_equal(np.array(got), want)
            t = P._sym_pad_axis(torch.from_numpy(x), 0, *pads)
            assert np.array_equal(t.numpy(), want)
    for mode, npmode in (("reflect", "reflect"), ("constant", "edge"), ("periodic", "wrap")):
        x = rng.standard_normal(7)
        want = np.pad(x, (5, 6), mode=npmode)
        got = [x[CF.ext_index(j, 7, mode)] for j in range(-5, 13)]
        assert np.array_equal(np.array(got), want)


def test_closed_form_equals_port():
    rng = np.random.default_rng(1)
    for wav in ("haar", "db2", "db4"):
        w = as_wavelet(wav)
        for mode in ("zero", "constant", "reflect", "periodic", "symmetric"):
            x = rng.standard_normal((2, 21))
            if mode == "reflect" and 21 <= len(w.dec_lo) - 2 + 1:
                continue
            lo, hi = CF.dwt_axis(x, w.dec_lo, w.dec_hi, mode)
            ref = P.wavedec(torch.from_numpy(x), wav, mode=mode, level=1)
            assert np.abs(lo - ref[0].numpy()).max() < 1e-13
            assert np.abs(hi - ref[1].numpy()).max() < 1e-13
            rec = CF.idwt_axis(lo, hi, w.rec_lo, w.rec_hi)
            assert np.abs(rec - P.waverec(ref, wav).numpy()).max() < 1e-13
            x2 = rng.standard_normal((2, 11, 14))
            bands = CF.dwt_nd_level(x2, w.dec_lo, w.dec_hi, mode, 2)
            r2 = P.wavedec2(torch.from_numpy(x2), wav, mode=mode, level=1)
            assert np.abs(bands[0] - r2[0].numpy()).max() < 1e-13
            assert np.abs(bands[2] - r2[1].horizontal.numpy()).max() < 1e-13
            assert np.abs(bands[1] - r2[1].vertical.numpy()).max() < 1e-13
            assert np.abs(bands[3] - r2[1].diagonal.numpy()).max() < 1e-13


def test_builtin_wavelet_table_is_orthonormal():
    from pytorch_wavelet_toolbox_b200._wavelet_table import REC_LO

    for name, taps in REC_LO.items():
        h = np.array(taps)
        assert abs(h.sum() - np.sqrt(2)) < 1e-14
        for s in range(0, len(h), 2):
            v = np.dot(h[s:], h[: len(h) - s])
            assert abs(v - (1.0 if s == 0 else 0.0)) < 1e-14, name
    # cross-check values quoted in SURVEY.md appendix A
    db2 = [0.48296291314453416, 0.8365163037378078, 0.22414386804201342, -0.1294095225512604]
    assert np.abs(np.array(REC_LO["db2"]) - db2).max() < 1e-15
    sym4 = [0.0322231006040427, -0.012603967262037833, -0.09921954357684722, 0.29785779560527736,
            0.8037387518059161, 0.49761866763201545, -0.02963552764599851, -0.07576571478927333]
    assert np.abs(np.array(REC_LO["sym4"]) - sym4).max() < 1e-11
    w = BuiltinWavelet("db2", REC_LO["db2"])
    assert w.dec_lo == w.rec_lo[::-1] and w.dec_hi == w.rec_hi[::-1]


def test_separable_containers_are_a_repackaging_of_wavedec2_3():
    """The claim behind pytorch_wavelet_toolbox_b200.separable: the reference's fswavedec2/3 bands (tests/golden/
    reference_api.*) equal the wavedec2/3 bands ('da' = horizontal, 'ad' = vertical, 'dd' = diagonal; 3-D keys
    unchanged)."""
    ref = reference_api()
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 33, 40, generator=g, dtype=torch.float64)
    check_sampled(ref, "fs2_x", x)
    assert ref["separable_keys"]["fs2"] == ["da", "ad", "dd"]
    for mode in ("zero", "reflect", "constant", "periodic"):
        wd = P.wavedec2(x, "db2", mode=mode, level=2)
        check_sampled(ref, f"fs2_{mode}_a", wd[0], 1e-12)
        for lv, t in enumerate(wd[1:], 1):
            check_sampled(ref, f"fs2_{mode}_{lv}da", t.horizontal, 1e-12)
            check_sampled(ref, f"fs2_{mode}_{lv}ad", t.vertical, 1e-12)
            check_sampled(ref, f"fs2_{mode}_{lv}dd", t.diagonal, 1e-12)
        check_sampled(ref, f"fs2_{mode}_rec", P.waverec2(wd, "db2"), 1e-12)
    x3 = torch.randn(2, 12, 13, 14, generator=g, dtype=torch.float64)
    check_sampled(ref, "fs3_x", x3)
    wd = P.wavedec3(x3, "db2", mode="zero", level=1)
    assert ref["separable_keys"]["fs3"] == ["daa", "ada", "dda", "aad", "dad", "add", "ddd"]
    for k in ref["separable_keys"]["fs3"]:
        check_sampled(ref, f"fs3_{k}", wd[1][k], 1e-12)
