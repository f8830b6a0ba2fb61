"""The oracle restatement vs. the REAL reference (bit-for-bit).

Where an output of the reference is stored under tests/golden/ (written from the reference
objects by tests/golden/make_golden.py), the case compares against it and runs everywhere:
the 2-D tables at ngp_1d = 2, 3, 4, the 3-D tables at ngp_1d = 2, and the Gauss-point
evaluations and loss bodies.  The cases no stored output covers (the 3-D tables at ngp_1d = 3,
the default constructor arguments, checkpoints) import the reference module itself
(oracle/refload.py) and skip where it is not importable.
"""
import numpy as np
import pytest
import torch

from oracle import losses as L
from oracle.fem import Q1Oracle
from oracle.refload import load_reference, reference_available


@pytest.fixture(scope="module")
def ref():
    if not reference_available():
        pytest.skip("the reference package is not importable (DIFFNET_REFERENCE_ROOT)")
    return load_reference()


def _same_tables(o, r, names):
    for n in names:
        a, b = getattr(o, n), getattr(r, n)
        if isinstance(a, list):
            assert len(a) == len(b)
            for x, y in zip(a, b):
                assert x.shape == y.shape and torch.equal(x, y.detach()), n
        else:
            assert torch.equal(torch.as_tensor(a), torch.as_tensor(b)), n


def _same_gp(o, g, u, keys):
    """The oracle's gauss_pt_evaluation* of u equal the reference's stored outputs bit for bit."""
    for m, k in keys:
        assert np.array_equal(getattr(o, m)(u).numpy(), g[k]), k


def _same_loss_and_grad(body, o, u, args, g, key):
    uo = u.clone().requires_grad_(True)
    lo = body(o, uo, *args)
    lo.backward()
    assert np.array_equal(lo.detach().numpy(), g[key + ".loss"]), key
    assert np.array_equal(uo.grad.numpy(), g[key + ".grad"]), key


@pytest.mark.parametrize("ngp", [2, 3, 4])
def test_tables_2d_bit_exact(golden, ngp):
    if ngp == 2:     # ref_2d_rect: 12 x 9 nodes on 1.5 x 1.0
        g = golden("ref_2d_rect")
        o = Q1Oracle(nsd=2, domain_sizes=(12, 9, 1), domain_lengths=(1.5, 1.0, 1.0), domain_size=12,
                     domain_length=1.5, ngp_1d=ngp)
        assert o.h == float(g["h"]) and o.hs == (float(g["hx"]), float(g["hy"]))
        _same_gp(o, g, g.t("u"), [("gauss_pt_evaluation", "gp.N"), ("gauss_pt_evaluation_der_x", "gp.dx"),
                                  ("gauss_pt_evaluation_der_y", "gp.dy")])
    else:            # ref_2d_ngp: 10 x 10 nodes on the unit square
        g = golden("ref_2d_ngp")
        o = Q1Oracle(nsd=2, domain_size=10, ngp_1d=ngp)
        assert np.array_equal(o.gpw.numpy(), g[f"gpw_ngp{ngp}"])
        _same_gp(o, g, g.t("u"), [("gauss_pt_evaluation", f"gp.N_ngp{ngp}"),
                                  ("gauss_pt_evaluation_der_x", f"gp.dx_ngp{ngp}")])


@pytest.mark.parametrize("ngp", [2, 3])
def test_tables_3d_bit_exact(golden, request, ngp):
    kw = dict(domain_sizes=(7, 6, 5), domain_lengths=(1.0, 0.8, 0.5), domain_size=7, ngp_1d=ngp)
    o = Q1Oracle(nsd=3, **kw)
    if ngp == 2:     # ref_3d_box: the reference's Gauss-point evaluations on this mesh
        g = golden("ref_3d_box")
        assert tuple(g["sizes"]) == (7, 6, 5) and tuple(g["lengths"]) == (1.0, 0.8, 0.5)
        _same_gp(o, g, g.t("u"), [("gauss_pt_evaluation", "gp.N"), ("gauss_pt_evaluation_der_x", "gp.dx"),
                                  ("gauss_pt_evaluation_der_y", "gp.dy"), ("gauss_pt_evaluation_der_z", "gp.dz")])
        return
    r = request.getfixturevalue("ref").DiffNet3DFEM(None, nsd=3, **kw)
    _same_tables(o, r, ["gpw", "N_gp", "dN_x_gp", "dN_y_gp", "dN_z_gp", "Nvalues", "dN_x_values",
                        "dN_y_values", "dN_z_values", "xx", "yy", "zz", "xgp", "ygp", "zgp"])
    assert (o.hs[0], o.hs[1], o.hs[2]) == (r.hx, r.hy, r.hz)


def test_default_kwargs_match(ref):
    r = ref.DiffNet2DFEM(None)
    o = Q1Oracle(nsd=2)
    assert o.sizes == (r.domain_sizeX, r.domain_sizeY) == (64, 64)
    assert o.h == r.h and torch.equal(o.N_gp[0], r.N_gp[0].detach())


def test_gp_eval_and_losses_bit_exact(golden):
    """The three 2-D loss bodies on the reference's 12 x 9 mesh: fp32 loss and gradient equal the
    reference's (ref_2d_rect: E2 = 0_base.py, E1 = 12_klsum.py energy, resmin = its residual form)."""
    g = golden("ref_2d_rect")
    o = Q1Oracle(nsd=2, domain_sizes=(12, 9, 1), domain_lengths=(1.5, 1.0, 1.0), domain_size=12, domain_length=1.5)
    u, inputs, f = g.t("u"), g.t("inputs"), g.t("forcing")
    _same_gp(o, g, u, [("gauss_pt_evaluation", "gp.N"), ("gauss_pt_evaluation_der_x", "gp.dx"),
                       ("gauss_pt_evaluation_der_y", "gp.dy")])
    for key, body in (("E2", L.body_0_base), ("E1", L.body_klsum_energy), ("resmin", L.body_klsum_resmin)):
        _same_loss_and_grad(body, o, u, (inputs, f), g, key)


def test_3d_losses_bit_exact(golden):
    """IBN_3D's loss body on the reference's 7 x 6 x 5 mesh (ref_3d_box)."""
    g = golden("ref_3d_box")
    o = Q1Oracle(nsd=3, domain_sizes=(7, 6, 5), domain_lengths=(1.0, 0.8, 0.5), domain_size=7)
    u = g.t("u")
    _same_gp(o, g, u, [("gauss_pt_evaluation_der_z", "gp.dz")])
    _same_loss_and_grad(L.body_ibn3d, o, u, (g.t("source"), g.t("sink"), g.t("forcing")), g, "ibn3d")


def test_reference_checkpoints_load_strictly(ref):
    """A state_dict written by the reference's DiffNet2DFEM / DiffNet3DFEM / UNet loads into the
    diffnet_b200 classes with strict=True (same keys, same shapes, same table values), and back."""
    import importlib
    from diffnet_b200 import DiffNet2DFEM, DiffNet3DFEM
    from diffnet_b200.networks import UNet
    for ours, theirs in ((DiffNet2DFEM(None, domain_size=16), ref.DiffNet2DFEM(None, domain_size=16)),
                         (DiffNet3DFEM(None, domain_size=8), ref.DiffNet3DFEM(None, domain_size=8, nsd=3))):
        sd = theirs.state_dict()
        assert set(sd) == set(ours.state_dict())
        for k, v in ours.state_dict().items():
            assert torch.equal(v, sd[k]), k
        ours.load_state_dict(sd, strict=True)
        theirs.load_state_dict(ours.state_dict(), strict=True)
    unets = importlib.import_module("DiffNet.networks.unets")
    torch.manual_seed(0)
    rnet, net = unets.UNet(3, 1).eval(), UNet(3, 1).eval()
    net.load_state_dict(rnet.state_dict(), strict=True)
    x = torch.rand(2, 3, 64, 64)
    with torch.no_grad():
        assert torch.equal(net(x), rnet(x))
    rnet.load_state_dict(net.reference_state_dict(), strict=True)
