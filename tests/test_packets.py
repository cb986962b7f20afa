"""Wavelet packets with level-wise batched expansion (SURVEY.md section 8f, row 4).

CPU: the dictionary semantics, orders and errors of the reference classes (tests/test_packets.py of the reference:
partial expansion :333-405, access errors :433-463, orders :243-330).  GPU: the numbers of the unmodified reference
(fixtures from oracle/make_golden_packets.py) and one launch per tree level.
"""
from __future__ import annotations

import json

import numpy as np
import pytest
import torch

import pytorch_wavelet_toolbox_b200 as wt
from conftest import GOLDEN, assert_close_rel


def test_orders_match_the_reference_definitions():
    assert wt.WaveletPacket.get_level(0) == [""]
    assert wt.WaveletPacket.get_level(2) == ["aa", "ad", "dd", "da"]                       # Gray code
    assert wt.WaveletPacket.get_level(2, "natural") == ["aa", "ad", "da", "dd"]
    assert wt.WaveletPacket.get_level(3)[:4] == ["aaa", "aad", "add", "ada"]
    with pytest.raises(ValueError):
        wt.WaveletPacket.get_level(2, "nope")
    nat = wt.WaveletPacket2D.get_natural_order(2)
    assert len(nat) == 16 and nat[:5] == ["aa", "ah", "av", "ad", "ha"]
    assert wt.WaveletPacket2D.get_freq_order(1) == [["a", "v"], ["h", "d"]]
    f2 = wt.WaveletPacket2D.get_freq_order(2)
    assert [len(r) for r in f2] == [4, 4, 4, 4] and f2[0][0] == "aa" and sorted(sum(f2, [])) == sorted(nat)
    ref = json.loads((GOLDEN / "reference_api.json").read_text())["packet_orders"]   # the unmodified reference's
    for lev in (0, 1, 2, 3):
        assert wt.WaveletPacket.get_level(lev) == ref[str(lev)]["gray"]
        assert wt.WaveletPacket.get_level(lev, "natural") == ref[str(lev)]["natural"]
        assert wt.WaveletPacket2D.get_freq_order(lev) == ref[str(lev)]["freq_2d"]
        assert wt.WaveletPacket2D.get_natural_order(lev) == ref[str(lev)]["natural_2d"]


def test_access_errors_without_touching_the_device():
    wp = wt.WaveletPacket(None, "haar")
    with pytest.raises(ValueError):
        wp["a"]
    wp.transform(torch.zeros(2, 32), maxlevel=2)
    with pytest.raises(KeyError):
        wp["aaa"]
    with pytest.raises(ValueError):
        wp["x"]
    assert wp[""].shape == (2, 32) and wp.maxlevel == 2
    wp2 = wt.WaveletPacket2D(torch.zeros(2, 16, 16), "haar", maxlevel=1)
    with pytest.raises(KeyError):
        wp2["aa"]
    with pytest.raises(ValueError):
        wp2["q"]
    with pytest.raises(NotImplementedError):
        wt.WaveletPacket(None, "haar", orthogonalization="cholesky")
    with pytest.warns(DeprecationWarning):
        wt.WaveletPacket(None, "haar", boundary_orthogonalization="qr")
    assert wt.WaveletPacket(torch.zeros(3, 64), "db2").maxlevel == 4           # floor(log2(64 / 3))
    with pytest.raises(KeyError):
        wt.WaveletPacket(torch.zeros(3, 64), "db2", maxlevel=1).reconstruct()   # leaves never initialised


def _cases():
    man = json.loads((GOLDEN / "packet_vectors.json").read_text())
    arr = np.load(GOLDEN / "packet_vectors.npz")
    return man["cases"], arr


def _make(case, x):
    if case["dim"] == 1:
        kw = {} if case["axes"] is None else {"axis": case["axes"]}
        return wt.WaveletPacket(x, case["wavelet"], mode=case["mode"], maxlevel=case["maxlevel"], **kw)
    kw = {} if case["axes"] is None else {"axes": tuple(case["axes"])}
    return wt.WaveletPacket2D(x, case["wavelet"], mode=case["mode"], maxlevel=case["maxlevel"],
                              separable=case["separable"], **kw)


@pytest.mark.gpu
def test_packets_equal_the_unmodified_reference_and_launch_once_per_level():
    from pytorch_wavelet_toolbox_b200 import _native

    cases, arr = _cases()
    for case in cases:
        i = case["id"]
        x = torch.from_numpy(arr[f"p{i}_x"]).cuda()
        wp = _make(case, x)
        leaves = (wp.get_level(case["maxlevel"], "natural") if case["dim"] == 1
                  else wp.get_natural_order(case["maxlevel"]))
        _native.launch_count_reset()
        wp.initialize(leaves)
        launches = _native.launch_count()
        assert sorted(k for k in wp.keys() if k != "") == case["keys"]
        scale = max(float(np.abs(arr[f"p{i}_{k}"]).max()) for k in case["keys"])
        for k in case["keys"]:
            assert_close_rel(wp[k], torch.from_numpy(arr[f"p{i}_{k}"]), scale=scale, what=f"packet case {i} node {k}")
        if case["mode"] != "boundary":
            # one launch per tree level (2-D separable: one per axis pass and level); the reference needs one per node
            per_level = 1 if not case["separable"] else 4
            assert launches <= per_level * case["maxlevel"], (case, launches)
        rec = wp.reconstruct()[""]
        want = torch.from_numpy(arr[f"p{i}_rec"])
        assert_close_rel(rec, want, scale=float(want.abs().max()), what=f"packet case {i} reconstruction")


@pytest.mark.gpu
def test_packets_partial_expansion_is_lazy_like_the_reference():
    """reference tests/test_packets.py:333-405: only the requested branches exist."""
    x = torch.randn(2, 64, device="cuda")
    wp = wt.WaveletPacket(x, "db2", mode="reflect", maxlevel=3)
    full = wp.get_level(3)
    assert not any(k in wp for k in full)
    wp.initialize(["aad", "aa", "d"])
    assert all(k in wp for k in ("a", "d", "aa", "ad", "aaa", "aad")) and "da" not in wp and "ada" not in wp
    wp["dda"]
    assert "dd" in wp and "da" in wp and "ddd" in wp and "daa" not in wp
    wp.initialize(full)
    assert all(k in wp for k in full)
    x2 = torch.randn(2, 32, 32, device="cuda")
    wp2 = wt.WaveletPacket2D(x2, "haar", maxlevel=2)
    wp2.initialize(["ah", "v"])
    assert all(k in wp2 for k in ("a", "h", "v", "d", "aa", "ah", "av", "ad")) and "ha" not in wp2
    full2 = wp2.get_natural_order(2)
    wp2.initialize(full2)
    assert all(k in wp2 for k in full2)
    # a modified leaf changes the reconstruction, an untouched tree reconstructs the input
    rec = wt.WaveletPacket2D(x2, "haar", maxlevel=2)
    rec.initialize(full2)
    assert float((rec.reconstruct()[""] - x2).abs().max()) < 1e-5
