"""Host-side contract of the drop-in API: validation, extents, layout, error behaviour (no GPU).

Mirrors the error cases of the reference's tests (tests/test_convolution_fwt.py:303-314, :391-402;
tests/test_convolution_fwt_3.py:167-178; tests/test_matrix_fwt.py:242-245)."""
from __future__ import annotations

import json
import sys

import numpy as np
import pytest
import torch

import pytorch_wavelet_toolbox_b200 as wt
from pytorch_wavelet_toolbox_b200 import _native, _shape
from pytorch_wavelet_toolbox_b200 import fwt as F
from pytorch_wavelet_toolbox_b200.matrix_fwt import _level_blocks, _analysis_taps, _level_sizes
from conftest import GOLDEN

no_gpu = not torch.cuda.is_available()


def reference_api() -> dict:
    return json.loads((GOLDEN / "reference_api.json").read_text())


def stand_in_ptwt(monkeypatch):
    """A ``ptwt`` with the reference's module layout (names bound by value in ``ptwt.packets``), computing with the
    oracle port -- the reference's own operator sequence -- for install() to find in sys.modules."""
    import types

    from oracle import ptwt_port as P

    ptwt = types.ModuleType("ptwt")
    ptwt.packets = types.ModuleType("ptwt.packets")
    ptwt.wavedec = ptwt.packets.wavedec = P.wavedec
    monkeypatch.setitem(sys.modules, "ptwt", ptwt)
    monkeypatch.setitem(sys.modules, "ptwt.packets", ptwt.packets)
    return ptwt


def test_public_surface_and_signatures():
    import inspect

    for name in wt.HOT_PATH_NAMES:
        assert hasattr(wt, name)
    sig = inspect.signature(wt.wavedec)
    assert list(sig.parameters) == ["data", "wavelet", "mode", "level", "axis"]
    assert sig.parameters["mode"].default == "reflect" and sig.parameters["mode"].kind is inspect.Parameter.KEYWORD_ONLY
    assert inspect.signature(wt.wavedec2).parameters["axes"].default == (-2, -1)
    s3 = inspect.signature(wt.wavedec3)
    assert s3.parameters["mode"].default == "zero" and s3.parameters["axes"].default == (-3, -2, -1)
    assert list(inspect.signature(wt.waverec2).parameters) == ["coeffs", "wavelet", "axes"]
    sm = inspect.signature(wt.MatrixWavedec.__init__)
    assert sm.parameters["orthogonalization"].default == "qr"
    assert sm.parameters["odd_coeff_padding_mode"].default == "zero"


@pytest.mark.parametrize("fn,shape", [(wt.wavedec, (4, 32)), (wt.wavedec2, (32, 32)), (wt.wavedec3, (16, 16, 16))])
def test_unsupported_dtype_raises_value_error(fn, shape):
    with pytest.raises(ValueError):
        fn(torch.zeros(shape, dtype=torch.int32), "haar", level=1)
    with pytest.raises(ValueError):
        fn(torch.zeros(shape, dtype=torch.float16), "haar", level=1)


def test_too_few_dims():
    with pytest.raises(ValueError):
        wt.wavedec2(torch.zeros(32), "haar", level=1)
    with pytest.raises(ValueError):
        wt.wavedec3(torch.zeros(32, 32), "haar", level=1)


def test_axes_errors():
    x = torch.zeros(4, 16, 16, 16)
    with pytest.raises(ValueError):
        wt.wavedec2(x, "haar", level=1, axes=(1, 1))
    with pytest.raises(ValueError):
        wt.wavedec2(x, "haar", level=1, axes=(1, 2, 3))
    with pytest.raises(ValueError):
        wt.wavedec3(x, "haar", level=1, axes=(1, 2))
    with pytest.raises(ValueError):
        wt.wavedec(x, "haar", level=1, axis=(1, 2))
    with pytest.raises(ValueError):
        wt.waverec2((x,), "haar", axes=(0, 0))


def test_unknown_mode():
    with pytest.raises(ValueError):
        wt.wavedec(torch.zeros(2, 32), "haar", mode="nope", level=1)


def test_level_zero_returns_input_unchanged():
    x = torch.randn(3, 20)
    out = wt.wavedec(x, "db2", level=0)
    assert isinstance(out, list) and len(out) == 1 and torch.equal(out[0], x)
    out2 = wt.wavedec2(torch.randn(2, 8, 8), "db2", level=0)
    assert isinstance(out2, tuple) and len(out2) == 1
    assert torch.equal(wt.waverec([x], "db2"), x)


def test_reflect_padding_larger_than_signal_raises_like_torch():
    with pytest.raises(RuntimeError):
        wt.wavedec(torch.zeros(2, 6), "db4", mode="reflect", level=1)
    with pytest.raises(RuntimeError):
        wt.wavedec(torch.zeros(2, 5), "db4", mode="periodic", level=1)


@pytest.mark.skipif(not no_gpu, reason="only meaningful on a machine without CUDA")
def test_no_cuda_device_fails_loudly():
    with pytest.raises(RuntimeError, match="CUDA"):
        wt.wavedec(torch.zeros(2, 32), "haar", level=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        wt.MatrixWavedec("haar", 1)(torch.zeros(2, 32))


def test_waverec2_malformed_containers():
    a = torch.zeros(2, 8, 8)
    with pytest.raises(ValueError):
        wt.waverec2((a, (a, a)), "haar")
    with pytest.raises(ValueError):
        wt.waverec2((a, a), "haar")
    with pytest.raises(ValueError):
        wt.waverec2((a, wt.WaveletDetailTuple2d(a, a, torch.zeros(2, 8, 9))), "haar")
    with pytest.raises(ValueError):
        wt.waverec2(([1, 2], (a, a, a)), "haar")
    with pytest.raises(ValueError):
        wt.waverec3((torch.zeros(2, 4, 4, 4), {"aad": torch.zeros(2, 4, 4, 4)}), "haar")
    with pytest.raises(ValueError):
        wt.waverec2((a, (a, a, a.double())), "haar")


def test_waverec_padding_mismatch_is_assertion_error():
    # the next detail must have the reconstructed length or one less (reference _util.py:231-244)
    with pytest.raises(AssertionError):
        wt.waverec([torch.zeros(2, 8), torch.zeros(2, 8), torch.zeros(2, 20)], "haar")


def test_packed_layout_is_aligned_and_matches_reference_extents():
    plan = F._make_plan((4096, 4096), 8, 4, 4)
    assert [lv.dims for lv in plan.levels] == [(2051, 2051), (1029, 1029), (518, 518), (262, 262)]
    for lv in plan.levels:
        assert lv.pitch % 4 == 0 and lv.pitch >= lv.dims[-1] and lv.plane % 32 == 0
        assert lv.det_off % 32 == 0
    n_coeff = 262 * 262 + 3 * sum(d * d for d in (262, 518, 1029, 2051))
    assert n_coeff == 16_875_874  # SURVEY.md section 8(a3)
    assert plan.item_elems >= n_coeff
    plan3 = F._make_plan((256, 256, 256), 8, 3, 4)
    assert [lv.dims[0] for lv in plan3.levels] == [131, 69, 38]
    assert plan3.levels[0].strides == (131 * 132, 132, 1)


def test_fold_unfold_roundtrip():
    x = torch.arange(2 * 3 * 4 * 5 * 6).reshape(2, 3, 4, 5, 6).float()
    for ndim, axes in ((1, 2), (2, (1, 3)), (3, (4, 0, 2)), (2, None), (1, -1)):
        t, f = _shape.fold(x, ndim, axes)
        assert t.dim() == ndim + 1
        assert torch.equal(_shape.unfold(t, f), x)
    t, f = _shape.fold(torch.zeros(7), 1, None)
    assert t.shape == (1, 7) and _shape.unfold(t, f).shape == (7,)


def test_matrix_argument_errors_and_deprecation():
    with pytest.raises(NotImplementedError):
        wt.MatrixWavedec("haar", 2, orthogonalization="nope")
    with pytest.raises(NotImplementedError):
        wt.MatrixWaverec("haar", orthogonalization="nope")
    with pytest.warns(DeprecationWarning):
        wt.MatrixWavedec("haar", 2, boundary="qr")
    with pytest.warns(DeprecationWarning):
        wt.MatrixWaverec("haar", boundary="qr")
    with pytest.raises(ValueError):
        wt.MatrixWavedec("haar", 0)(torch.zeros(2, 32))
    with pytest.raises(ValueError):
        wt.MatrixWavedec("haar", 2)(torch.zeros(2, 32, dtype=torch.int64))
    with pytest.raises(ValueError):
        wt.MatrixWavedec("haar", 2, axis=(0, 1))


def test_boundary_operators_match_reference_fixtures(golden):
    """construct_boundary_a / _s == the matrices the reference built (tests/golden)."""
    _, arrays = golden
    for wav, n in (("db2", 16), ("db4", 32), ("db6", 64)):
        a = wt.construct_boundary_a(wav, n, dtype=torch.float64).to_dense().numpy()
        s = wt.construct_boundary_s(wav, n, dtype=torch.float64).to_dense().numpy()
        assert np.abs(a - arrays[f"A_{wav}_{n}"]).max() < 1e-13
        assert np.abs(s - arrays[f"S_{wav}_{n}"]).max() < 1e-13
        eye = np.eye(n)
        assert np.abs(a @ a.T - eye).max() < 1e-8 and np.abs(s @ a - eye).max() < 1e-8


@pytest.mark.parametrize("wav,n", [("db2", 24), ("db4", 64), ("db6", 128), ("db8", 256)])
def test_boundary_blocks_shape_and_independence_of_n(wav, n):
    """Corner blocks are confined to the first / last L-1 columns and do not depend on n
    (SURVEY.md section 8(a7)); counts are ceil((L-2)/4) top and floor(L/4) bottom."""
    lo, hi = _analysis_taps(wav, torch.float64)
    L = lo.shape[0]
    b1 = _level_blocks(lo, hi, torch.float64, n, "qr")
    b2 = _level_blocks(lo, hi, torch.float64, 4 * n, "qr")
    assert b1.nb_top == -(-(L - 2) // 4) and b1.nb_bot == L // 4
    assert b1.w_left <= L - 1 and b1.w_right <= L - 1
    for name in ("lo_left", "lo_right", "hi_left", "hi_right"):
        assert (getattr(b1, name) - getattr(b2, name)).abs().max() < 1e-14


def test_level_sizes_bookkeeping():
    sizes, pads, last = _level_sizes(101 + 1, 3, 4)  # odd input already padded to 102 by the caller
    assert sizes == [102, 52, 26] and pads == [False, True, False] and last == 13
    sizes, pads, last = _level_sizes(65536, 12, 12)
    assert sizes[-1] == 32 and last == 16 and not any(pads)


def test_install_is_a_noop_without_ptwt():
    import importlib.util

    if importlib.util.find_spec("ptwt") is None:
        if torch.cuda.is_available():
            with pytest.raises(ModuleNotFoundError):
                wt.install()
        else:
            with pytest.warns(RuntimeWarning):       # no CUDA device: nothing is rebound, not even looked up
                assert wt.install() == []


def test_separable_matrix_nd_argument_errors():
    """MatrixWavedec2/3 mirror the reference's constructor checks (matmul_transform_2.py:329-341,
    matmul_transform_3.py:121-128); the non-separable operator is declared out of scope."""
    import pytorch_wavelet_toolbox_b200 as wt

    with pytest.raises(NotImplementedError):
        wt.MatrixWavedec2("haar", 2, orthogonalization="cholesky")
    with pytest.raises(NotImplementedError):
        wt.MatrixWavedec3("haar", 2, orthogonalization="cholesky")
    with pytest.raises(ValueError):
        wt.MatrixWavedec2("haar", 2, axes=(1, 1))
    with pytest.raises(ValueError):
        wt.MatrixWaverec3("haar", axes=(0, 1))
    with pytest.raises(NotImplementedError):
        wt.MatrixWavedec2("haar", 2, separable=False)(torch.zeros(2, 8, 8))
    with pytest.raises(NotImplementedError):
        wt.MatrixWavedec2("haar", 2).sparse_fwt_operator
    with pytest.raises(ValueError):
        wt.MatrixWavedec2("haar", 0)(torch.zeros(2, 8, 8))
    with pytest.raises(ValueError):
        wt.MatrixWaverec2("haar")((torch.zeros(2, 4, 4), [torch.zeros(2, 4, 4)] * 3))
    with pytest.raises(ValueError):
        wt.MatrixWaverec3("haar")((torch.zeros(2, 4, 4, 4), (torch.zeros(2, 4, 4, 4),)))
    with pytest.warns(DeprecationWarning):
        wt.MatrixWavedec2("haar", 2, boundary="qr")


def test_separable_matrix_level_walk_matches_the_reference_warning(capsys):
    """The level walk of MatrixWavedec2/3 (operator sizes, padded axes, early stop with the reference's
    stderr warning, matmul_transform_2.py:381-405 / matmul_transform_3.py:163-196) is host logic: check it
    here, and against the warnings the unmodified reference printed (tests/golden/reference_api.json)."""
    from pytorch_wavelet_toolbox_b200.matrix_fwt_nd import _level_sizes

    sizes, pads = _level_sizes((33, 20), 4, 2, 2)
    assert sizes == [(34, 20), (18, 10)] and pads == [(True, False), (True, False)]
    assert capsys.readouterr().err == ""
    sizes, pads = _level_sizes((12, 9, 16), 4, 3, 3)
    assert sizes == [(12, 10, 16), (6, 6, 8)] and pads == [(False, True, False), (False, True, False)]
    ours = capsys.readouterr().err
    assert "only computed up to the decomposition level 2" in ours and "(3, 3,4)" in ours

    ref = reference_api()["level_walk_stderr"]          # MatrixWavedec3("db2", 3) on (12, 9, 16), MatrixWavedec2("db3", 3)
    assert ref[0] == ours                               # on (20, 12)
    _level_sizes((20, 12), 6, 3, 2)
    assert capsys.readouterr().err == ref[1]


def test_signatures_equal_the_reference_functions():
    """Every public callable has the parameter names, kinds and defaults of the reference function of the same name
    (as the unmodified reference declared them, tests/golden/reference_api.json)."""
    from oracle.make_golden_api import PACKET_CLASSES, SIGNATURE_CLASSES, SIGNATURE_FUNCTIONS, params

    ref = reference_api()["signatures"]
    for name in SIGNATURE_FUNCTIONS:
        assert params(getattr(wt, name)) == ref[name], name
    for name in SIGNATURE_CLASSES:
        assert params(getattr(wt, name).__init__) == ref[name], name
    for name in PACKET_CLASSES:
        assert [q[0] for q in params(getattr(wt, name).__init__)] == ref[name], name


def test_install_leaves_a_cpu_only_machine_alone(monkeypatch):
    """Without a CUDA device install() must not turn a working CPU ptwt into a failing one (ADVICE round 1)."""
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    ptwt = stand_in_ptwt(monkeypatch)
    before = ptwt.wavedec
    with pytest.warns(RuntimeWarning):
        assert wt.install() == []
    assert ptwt.wavedec is before and ptwt.packets.wavedec is before
    c = ptwt.wavedec(torch.arange(16.0), "haar", mode="zero", level=2)
    assert [t.shape[-1] for t in c] == [4, 4, 8]


def test_fold_extension_is_the_adjoint_of_the_boundary_extension():
    """The differentiable path extends inside the kernel on the forward pass and folds the gradient of the extended
    signal back on the backward pass (_autograd.fold_extension).  Pure torch, so checked here against autograd of the
    extension itself: every mode, 1-D .. 3-D, even / odd lengths, extensions longer than the signal."""
    import torch
    from pytorch_wavelet_toolbox_b200._autograd import extend, fold_extension

    g = torch.Generator().manual_seed(5)
    checked = 0
    for mode in ("reflect", "constant", "periodic", "symmetric"):
        for filt_len in (2, 4, 8, 12):
            for dims in ((5,), (7,), (8,), (33,), (5, 6), (16, 9), (4, 5, 6), (13, 8, 7)):
                x = torch.randn((2,) + dims, generator=g, dtype=torch.float64, requires_grad=True)
                try:
                    xp = extend(x, len(dims), filt_len, mode)
                except RuntimeError:          # torch refuses reflect / circular pads longer than the signal
                    continue
                gy = torch.randn(xp.shape, generator=g, dtype=torch.float64)
                (want,) = torch.autograd.grad(xp, x, gy)
                got = fold_extension(gy, dims, filt_len, mode)
                assert got.shape == want.shape and float((got - want).abs().max()) < 1e-12, (mode, filt_len, dims)
                checked += 1
    assert checked > 80
