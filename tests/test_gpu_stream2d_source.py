"""The streaming 2-D kernel's nodal source stencil at its edges.

The streaming kernel (k_fem2d_tma) takes the nodal-f source term per node, as the separable stencil
-kf (M_y (x) M_x) f of the 1-D element mass M, while the general kernel (k_fem2d, DN_2D_PATH=warp)
integrates it per element.  Both are compared with each other and with the fp64 oracle where the
stencil has edges: the image's first/last row and column, chunk seams, warp seams, one-warp and
two-lane widths, odd row counts (a trailing half stage), Dirichlet sets with scalar values, a value
field and a nu mask, every Gauss rule, and both loss forms (energy, and the residual form in which
the source share enters the residual before it is squared).
"""
import os

import pytest
import torch

from conftest import rel_l2, rel_scalar
from helpers import assert_parity, oracle_energy, oracle_residual
from diffnet_b200 import DiffNet2DFEM

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (B, ny, nx): two lanes and one stage; odd ny; three warps (warp seams); many chunks per image
# (chunk seams, balanced split) with odd ny; a wide image with a partly idle last warp
SIZES = [(3, 2, 8), (2, 9, 8), (2, 33, 264), (1, 67, 520), (2, 16, 1000)]


def _inputs(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(B, 1, H, W, generator=g)
    nu = torch.exp(0.5 * torch.randn(B, 1, H, W, generator=g))
    f = torch.randn(B, 1, H, W, generator=g)
    left = torch.zeros(B, 1, H, W); left[..., 0] = 1
    right = torch.zeros(B, 1, H, W); right[..., -1] = 1
    top = torch.zeros(B, 1, H, W); top[:, :, 0, :] = 1
    blob = (torch.rand(B, 1, H, W, generator=g) > 0.8).float()
    ubc = torch.randn(B, 1, H, W, generator=g)
    return [t.to(DEV) for t in (u, nu, f, left, right, top, blob, ubc)]


def _cases(nu, f, left, right, top, blob, ubc):
    return {
        "f": dict(f=f),
        "nu_f_2mask": dict(nu=nu, f=f, dirichlet=[(left, 1.0), (right, 0.0)]),
        "f_3mask": dict(f=f, dirichlet=[(left, 1.0), (right, 0.0), (top, 0.25)]),
        "nu_f_valuefield": dict(nu=nu, f=f, dirichlet=[(blob, ubc)]),
        "nu_f_numask": dict(nu=nu, f=f, nu_zero_mask=top, dirichlet=[(left, 1.0), (right, 0.0)]),
    }


def _both_paths(fn):
    os.environ.pop("DN_2D_PATH", None)
    stream = fn()
    os.environ["DN_2D_PATH"] = "warp"
    try:
        general = fn()
    finally:
        os.environ.pop("DN_2D_PATH", None)
    return stream, general


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("B,H,W", SIZES)
def test_energy_source_stencil_edges(B, H, W, ngp):
    fem = DiffNet2DFEM(None, domain_sizes=(W, H, 1), domain_lengths=(1.3, 0.9, 1.0), domain_size=W, ngp_1d=ngp)
    u, nu, f, left, right, top, blob, ubc = _inputs(B, H, W, seed=H * 7 + W + ngp)
    for name, kw in _cases(nu, f, left, right, top, blob, ubc).items():
        (ls, gs), (lw, gw) = _both_paths(lambda: fem.energy_loss_and_grad(u, **kw))
        what = f"{name} {B}x{H}x{W} ngp={ngp}"
        assert rel_scalar(ls, lw) < 2e-6, (what, float(ls), float(lw))
        assert rel_l2(gs, gw) < 2e-6, what
        if B * H * W <= 40_000:
            lref, gref = oracle_energy(fem, u.cpu(), **{k: v for k, v in kw.items()})
            masks = [m for m, _ in kw.get("dirichlet", [])]
            assert_parity(ls, gs, lref, gref, masks=masks, what=what)


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("B,H,W", SIZES)
def test_residual_source_stencil_edges(B, H, W, ngp):
    fem = DiffNet2DFEM(None, domain_sizes=(W, H, 1), domain_size=W, ngp_1d=ngp)
    u, nu, f, left, right, top, blob, ubc = _inputs(B, H, W, seed=H * 11 + W + ngp)
    cases = {"f": dict(f=f), "nu_f_2mask": dict(nu=nu, f=f, dirichlet=[(left, 1.0), (right, 0.0)])}
    for name, kw in cases.items():
        def run():
            ud = u.clone().requires_grad_(True)
            loss = fem.residual_loss(ud, jac=(0.5 * fem.h) ** 2, **kw)
            loss.backward()
            return loss.detach(), ud.grad.detach()
        (ls, gs), (lw, gw) = _both_paths(run)
        what = f"residual {name} {B}x{H}x{W} ngp={ngp}"
        assert rel_scalar(ls, lw) < 2e-6, (what, float(ls), float(lw))
        assert rel_l2(gs, gw) < 2e-6, what
        if B * H * W <= 40_000:
            lref, gref = oracle_residual(fem, u.cpu(), jac=(0.5 * fem.h) ** 2, **kw)
            assert rel_scalar(ls, lref) <= 1e-5, (what, float(ls), float(lref))
            assert rel_l2(gs.cpu(), gref.reshape(gs.shape)) <= 1e-4, what
