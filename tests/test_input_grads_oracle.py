"""The closed forms the input-gradient kernels implement, pinned to the fp64 autograd of oracle.losses (CPU).

dn_fem_{energy,residual}_input_grads_* compute each gradient as a nodal operator (include/diffnet_fem.h):
the separable Q1 mass stencil M, the stiffness K(nu) and Gauss-point products, with the Dirichlet value fields
taking the gradient where their mask is the last one that fires.  Here those formulas are evaluated with the
oracle's own gp-eval convolutions (transposes by autograd of the linear gp-eval alone) and compared with what
autograd gives the reference's loss() bodies.
"""
import pytest
import torch

from oracle import losses as OL
from oracle.fem import Q1Oracle


def _mass(fem, X):
    """M X with M = (x)_d (W1/4)[[1+t, 1-t], [1-t, 1+t]] per element, t = sum w x^2 / W1, assembled."""
    x, w = [torch.as_tensor(v, dtype=torch.float64) for v in (fem.gpx_1d, fem.gpw_1d)]
    W1 = float(w.sum())
    t = float((w * x * x).sum()) / W1
    a, c = 0.25 * W1 * (1 + t), 0.25 * W1 * (1 - t)
    out = X
    for ax in range(2, X.dim()):                          # one separable 1-D mass per direction
        lo = out.narrow(ax, 0, out.shape[ax] - 1)
        hi = out.narrow(ax, 1, out.shape[ax] - 1)
        pad = [0, 0] * (X.dim() - 1 - ax)
        res = torch.nn.functional.pad(a * lo + c * hi, pad + [0, 1]) + torch.nn.functional.pad(c * lo + a * hi, pad + [1, 0])
        out = res
    return out


def _eq(got, want):
    """Max-norm agreement.  The oracle's basis tables and weights are the reference's fp32 roundings, so its
    autograd differs from the fp64 closed forms in the 7th digit."""
    err = float((got - want).abs().max() / want.abs().max().clamp_min(1e-300))
    assert err <= 1e-5, err


def _tables(fem):
    return [fem.gauss_pt_evaluation_der_x, fem.gauss_pt_evaluation_der_y] + (
        [fem.gauss_pt_evaluation_der_z] if fem.nsd == 3 else [])


def _gpw(fem):
    return fem.gpw.double().reshape((1, -1) + (1,) * fem.nsd)


def _transpose(op, cot, like):
    """op^T cot for a linear gp-eval op (autograd of the op alone)."""
    with torch.enable_grad():
        y = torch.zeros_like(like, requires_grad=True)
        (g,) = torch.autograd.grad((op(y) * cot).sum(), y)
    return g


def _stiff(fem, nu, X):
    """K(nu) X = sum_d D_d^T (w nu_g D_d X)."""
    nug = fem.gauss_pt_evaluation(nu) if nu is not None else 1.0
    return sum(_transpose(D, _gpw(fem) * nug * D(X), X) for D in _tables(fem))


def _last_mask(dirichlet, k):
    fire = dirichlet[k][0] > 0.5
    for m, _ in dirichlet[k + 1:]:
        fire = fire & ~(m > 0.5)
    return fire


def _setup(nsd, ngp, seed):
    torch.manual_seed(seed)
    shape = (7, 9) if nsd == 2 else (5, 6, 7)
    sizes = tuple(reversed(shape)) + ((1,) if nsd == 2 else ())
    fem = Q1Oracle(nsd=nsd, domain_size=sizes[0], domain_sizes=sizes, domain_lengths=(1.3, 0.9, 1.1),
                   ngp_1d=ngp, dtype=torch.float64)
    sp = (2, 1) + shape
    d = lambda: torch.randn(sp, dtype=torch.float64)   # noqa: E731
    m0 = (torch.rand(sp) > 0.6).double()
    m1 = (torch.rand(sp) > 0.6).double()
    return fem, sp, d, m0, m1


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("nsd", [2, 3])
def test_energy_input_gradient_formulas(nsd, ngp):
    fem, sp, d, m0, m1 = _setup(nsd, ngp, 10 * nsd + ngp)
    u, f, v0, v1 = d(), d(), d(), d()
    nu = torch.exp(0.3 * d())
    numask = (torch.rand(sp) > 0.8).double()
    scale, c_k, c_f = 0.7, 1.3, 0.9
    count = sp[0] * torch.tensor(sp[2:]).sub(1).prod().item()
    S = scale / count
    f = f.requires_grad_(True)
    v0, v1 = v0.requires_grad_(True), v1.requires_grad_(True)
    dirichlet = [(m0, v0), (m1, v1)]
    L = OL.energy_loss(fem, u, nu=nu, f=f, dirichlet=dirichlet, nu_zero_mask=numask, c_k=c_k, c_f=c_f, scale=scale)
    gf, g0, g1 = torch.autograd.grad(L, [f, v0, v1])
    with torch.no_grad():
        up = OL._dirichlet(u, [(m0, v0.detach()), (m1, v1.detach())])
        nup = torch.where(numask > 0.5, 0.0 * nu, nu)
        ghat = S * (2 * c_k * _stiff(fem, nup, up) - c_f * _mass(fem, f.detach()))
        _eq(gf, -S * c_f * _mass(fem, up))
        _eq(g0, torch.where(_last_mask(dirichlet, 0), ghat, 0.0))
        _eq(g1, torch.where(_last_mask(dirichlet, 1), ghat, 0.0))

    # forcing at the Gauss points: dL/df_gp = -S c_f w_G u'_G, and the source part of g-hat is -c_f N^T (w f_gp)
    fgp = torch.randn((sp[0], fem.ngp_total) + tuple(s - 1 for s in sp[2:]), dtype=torch.float64, requires_grad=True)
    v0 = v0.detach().requires_grad_(True)
    L = OL.energy_loss(fem, u, nu=nu, f_gp=fgp, dirichlet=[(m0, v0)], c_k=c_k, c_f=c_f, scale=scale)
    gfgp, g0 = torch.autograd.grad(L, [fgp, v0])
    with torch.no_grad():
        up = OL._dirichlet(u, [(m0, v0.detach())])
        _eq(gfgp, -S * c_f * _gpw(fem) * fem.gauss_pt_evaluation(up))
        src = _transpose(fem.gauss_pt_evaluation, _gpw(fem) * fgp.detach(), up)
        ghat = S * (2 * c_k * _stiff(fem, nu, up) - c_f * src)
        _eq(g0, torch.where(m0 > 0.5, ghat, 0.0))


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("nsd", [2, 3])
def test_residual_input_gradient_formulas(nsd, ngp):
    fem, sp, d, m0, m1 = _setup(nsd, ngp, 20 * nsd + ngp)
    u, f, v0, v1 = d(), d(), d(), d()
    nu = torch.exp(0.3 * d()).requires_grad_(True)
    f = f.requires_grad_(True)
    v0, v1 = v0.requires_grad_(True), v1.requires_grad_(True)
    jac = 0.37
    dirichlet = [(m0, v0), (m1, v1)]
    L = OL.residual_loss(fem, u, nu=nu, f=f, dirichlet=dirichlet, jac=jac)
    gnu, gf, g0, g1 = torch.autograd.grad(L, [nu, f, v0, v1])
    with torch.no_grad():
        R = OL.residual_vector(fem, u, nu=nu.detach(), f=f.detach(),
                               dirichlet=[(m0, v0.detach()), (m1, v1.detach())], jac=jac)
        up = OL._dirichlet(u, [(m0, v0.detach()), (m1, v1.detach())])
        dot = sum(D(up) * D(R) for D in _tables(fem))
        _eq(gnu, 2 * jac * _transpose(fem.gauss_pt_evaluation, _gpw(fem) * dot, up))
        _eq(gf, -2 * jac * _mass(fem, R))
        KR = 2 * jac * _stiff(fem, nu.detach(), R)
        _eq(g0, torch.where(_last_mask(dirichlet, 0), KR, 0.0))
        _eq(g1, torch.where(_last_mask(dirichlet, 1), KR, 0.0))
