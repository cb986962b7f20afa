"""install() / uninstall(): rebinding in ptwt and in the modules that captured the names by value, against a stand-in
with the reference's module layout; the REAL reference package (oracle/_ref, installed by oracle/make_ref.py when the
reference is at hand) for its own packet classes and learnable filters running on the new kernels."""
from __future__ import annotations

import sys
import types

import pytest
import torch

import pytorch_wavelet_toolbox_b200 as wt

pytestmark = pytest.mark.gpu


@pytest.fixture
def ptwt():
    from oracle.make_ref import import_ref

    mod = import_ref()
    if mod is None:
        pytest.skip("the reference package is not installed in oracle/_ref (PTWT_REFERENCE_SRC=... python -m oracle.make_ref)")
    yield mod
    wt.uninstall()


@pytest.fixture
def stand_in_ptwt(monkeypatch):
    """``ptwt`` with the reference's layout: the names defined in conv_transform(_2) / matmul_transform, re-exported by
    the package and bound by value in packets (packets.py:34-37) and separable_conv_transform (:33); every function is
    the oracle port, the reference's own operator sequence."""
    from oracle import ptwt_port as P

    mods = {name: types.ModuleType(name) for name in ("ptwt", "ptwt.conv_transform", "ptwt.conv_transform_2",
                                                       "ptwt.matmul_transform", "ptwt.packets",
                                                       "ptwt.separable_conv_transform")}
    defined = {"ptwt.conv_transform": ("wavedec", "waverec"), "ptwt.conv_transform_2": ("wavedec2", "waverec2"),
               "ptwt.matmul_transform": ("MatrixWavedec", "MatrixWaverec")}
    for modname, names in defined.items():
        for name in names:
            setattr(mods[modname], name, getattr(P, name))
            setattr(mods["ptwt"], name, getattr(P, name))
    mods["ptwt.packets"].wavedec = mods["ptwt.separable_conv_transform"].wavedec = P.wavedec
    for modname, mod in mods.items():
        monkeypatch.setitem(sys.modules, modname, mod)
        if modname != "ptwt":
            setattr(mods["ptwt"], modname.split(".")[1], mod)
    yield mods["ptwt"]
    wt.uninstall()


def test_install_rebinds_and_uninstall_restores(stand_in_ptwt):
    ptwt = stand_in_ptwt
    packets, sep = ptwt.packets, ptwt.separable_conv_transform
    ref_wavedec, ref_packets_wavedec, ref_sep_wavedec = ptwt.wavedec, packets.wavedec, sep.wavedec
    replaced = wt.install()
    assert "ptwt.wavedec" in replaced and "ptwt.packets.wavedec" in replaced
    assert ptwt.wavedec is wt.wavedec and packets.wavedec is wt.wavedec and sep.wavedec is wt.wavedec
    assert ptwt.conv_transform_2.wavedec2 is wt.wavedec2 and ptwt.matmul_transform.MatrixWavedec is wt.MatrixWavedec
    x = torch.randn(2, 3, 64, 48, device="cuda")
    got = ptwt.wavedec2(x, "db2", level=2)                      # the reference's name, our kernels
    wt.uninstall()
    assert ptwt.wavedec is ref_wavedec and packets.wavedec is ref_packets_wavedec and sep.wavedec is ref_sep_wavedec
    want = ptwt.wavedec2(x.cpu(), "db2", level=2)               # the reference's operator sequence on the CPU
    flat = lambda c: [c[0]] + [b for lv in c[1:] for b in lv]   # noqa: E731
    scale = max(float(t.abs().max()) for t in flat(want))
    for a, b in zip(flat(got), flat(want)):
        assert a.is_cuda and float((a.cpu() - b).abs().max()) <= 1e-5 * scale


def test_reference_packet_classes_ride_on_the_installed_kernels(ptwt):
    """The reference's own WaveletPacket captured wavedec by value (packets.py:34-37): after install() it runs every node
    through our level-1 kernels and still produces the reference's numbers."""
    import ptwt.packets as packets

    ref_cls = packets.WaveletPacket
    x = torch.randn(3, 128, dtype=torch.float64)
    want = ref_cls(x, "db3", mode="reflect", maxlevel=3)
    keys = want.get_level(3)
    want_nodes = {k: want[k] for k in keys}
    wt.install()
    assert packets.wavedec is wt.wavedec
    got = ref_cls(x.cuda(), "db3", mode="reflect", maxlevel=3)   # the reference's class, not ours
    scale = max(float(t.abs().max()) for t in want_nodes.values())
    for k in keys:
        assert got[k].is_cuda and float((got[k].cpu() - want_nodes[k]).abs().max()) <= 1e-11 * scale
    ours = ptwt.WaveletPacket(x.cuda(), "db3", mode="reflect", maxlevel=3)   # rebound to the batched class
    assert type(ours) is wt.WaveletPacket
    ours.initialize(keys)
    for k in keys:
        assert float((ours[k].cpu() - want_nodes[k]).abs().max()) <= 1e-11 * scale


def test_reference_learnable_filters_train_through_the_installed_backend(ptwt):
    """ptwt.wavelets_learnable.ProductFilter (nn.Parameters behind filter_bank, wavelets_learnable.py:167-199) through
    ptwt.wavedec / waverec after install(): the four filters and the data receive the reference's gradients
    (the pattern of examples/network_compression/wavelet_linear.py:118,150)."""
    from ptwt.wavelets_learnable import ProductFilter

    def make():
        fb = wt.WaveletTensorTuple.from_wavelet(wt._wavelets.as_wavelet("db3"), torch.float64)
        return ProductFilter(*[t.clone() for t in fb])

    g = torch.Generator().manual_seed(3)
    x = torch.randn(4, 96, generator=g, dtype=torch.float64)
    w = torch.randn(4, 96, generator=g, dtype=torch.float64)

    def loss_of(mod, wav, data, weight):
        c = mod.wavedec(data, wav, level=3, mode="reflect")
        rec = mod.waverec(c, wav)[..., :96]
        return sum((t * t).sum() for t in c) + (rec * weight).sum() + wav.wavelet_loss()

    ref_wav = make()
    xr = x.clone().requires_grad_(True)
    loss_ref = loss_of(ptwt, ref_wav, xr, w)
    loss_ref.backward()
    wt.install()
    our_wav = make()
    xo = x.clone().cuda().requires_grad_(True)
    loss_our = loss_of(ptwt, our_wav, xo, w.cuda())
    loss_our.backward()
    assert abs(float(loss_our) - float(loss_ref)) <= 1e-10 * abs(float(loss_ref))
    assert float((xo.grad.cpu() - xr.grad).abs().max()) <= 1e-10 * float(xr.grad.abs().max())
    for name in ("dec_lo", "dec_hi", "rec_lo", "rec_hi"):
        a, b = getattr(our_wav, name).grad, getattr(ref_wav, name).grad
        assert a is not None, name
        assert float((a - b).abs().max()) <= 1e-9 * float(b.abs().max()), name
