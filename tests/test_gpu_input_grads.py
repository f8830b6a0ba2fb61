"""Gradients of the fused losses with respect to f, f_gp, the Dirichlet value fields and (residual form) nu.

Every gradient is compared with the fp64 autograd of oracle.losses (the reference's loss() bodies), across streaming
and general 2-D sizes, 3-D shapes, Gauss rules 2-4, broadcast / strided / bare input layouts and non-default
constants; then the autograd plumbing, bit-identity of the default path, identities at the benchmark sizes, and a
short Adam run against the oracle.
"""
import pytest
import torch

from conftest import rel_l2, rel_scalar
from helpers import GRAD_MAX_RTOL, GRAD_RTOL, LOSS_RTOL, oracle_for, to64
from oracle import losses as OL
from diffnet_b200 import DiffNet2DFEM, DiffNet3DFEM, ops
from diffnet_b200._lib import DiffNetFEMError

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _fem(shape, ngp):
    if len(shape) == 2:
        H, W = shape
        return DiffNet2DFEM(None, domain_sizes=(W, H, 1), domain_lengths=(1.3, 0.9, 1.0), domain_size=W, ngp_1d=ngp)
    D, H, W = shape
    return DiffNet3DFEM(None, domain_sizes=(W, H, D), domain_lengths=(1.1, 0.9, 1.2), domain_size=W, ngp_1d=ngp)


def _fields(B, shape, seed, ngp=2):
    g = torch.Generator().manual_seed(seed)
    sp = (B, 1) + tuple(shape)
    u = torch.randn(sp, generator=g)
    nu = torch.exp(0.5 * torch.randn(sp, generator=g))
    f = torch.randn(sp, generator=g)
    left = torch.zeros(sp); left[..., 0] = 1
    right = torch.zeros(sp); right[..., -1] = 1
    blob = (torch.rand(sp, generator=g) > 0.7).float()
    ubc = torch.randn(sp, generator=g)
    numask = (torch.rand(sp, generator=g) > 0.85).float()
    elems = tuple(s - 1 for s in shape)
    fgp = torch.randn((B, ngp ** len(shape)) + elems, generator=g)
    return dict(u=u, nu=nu, f=f, left=left, right=right, blob=blob, ubc=ubc, numask=numask, fgp=fgp)


def _close(g, gref, what):
    g = g.detach().cpu().double()
    gref = gref.detach().double().reshape(g.shape)
    e = rel_l2(g, gref)
    assert e <= GRAD_RTOL, f"{what}: rel-L2 {e:.3e}"
    em = float((g - gref).abs().max() / gref.abs().max().clamp_min(1e-300))
    assert em <= GRAD_MAX_RTOL, f"{what}: max-norm {em:.3e}"


def _leafs(kw, names):
    """Copies of the inputs (device) with requires_grad on the named ones; names may index values as 'v0', 'v1'."""
    out = {}
    for k, v in kw.items():
        if k == "dirichlet":
            out[k] = [(m, (val.detach().clone().requires_grad_(f"v{i}" in names) if torch.is_tensor(val) else val))
                      for i, (m, val) in enumerate(v)]
        elif torch.is_tensor(v):
            out[k] = v.detach().clone().requires_grad_(k in names)
        else:
            out[k] = v
    return out


def _wrt(kw, names):
    ts = [kw[n] for n in names if not n.startswith("v")]
    ts += [val for i, (_, val) in enumerate(kw.get("dirichlet", ())) if f"v{i}" in names]
    return ts


def _check(fem, loss_fn, oracle_fn, u, kw, names, what, **fixed):
    dev_kw = _leafs({k: (v.to(DEV) if torch.is_tensor(v) else
                         [(m.to(DEV), val.to(DEV) if torch.is_tensor(val) else val) for m, val in v]
                         if k == "dirichlet" else v) for k, v in kw.items()}, names)
    ud = u.to(DEV).requires_grad_(True)
    loss = loss_fn(ud, **dev_kw, **fixed)
    loss.backward()
    ref_kw = _leafs({k: (to64(v) if k != "dirichlet" else [(to64(m), to64(val)) for m, val in v])
                     for k, v in kw.items()}, names)
    u64 = to64(u).requires_grad_(True)
    nsd = len(fem.geometry.spatial)
    call_kw = {k: (v[None, None] if torch.is_tensor(v) and v.dim() == nsd else v) for k, v in ref_kw.items()}
    lref = oracle_fn(oracle_for(fem), u64, **call_kw, **fixed)
    refs = torch.autograd.grad(lref, [u64] + _wrt(ref_kw, names))
    assert rel_scalar(loss.detach().cpu(), lref.detach()) <= LOSS_RTOL, what
    _close(ud.grad, refs[0], what + " du")
    for n, t, r in zip(names, _wrt(dev_kw, names), refs[1:]):
        assert t.grad is not None, f"{what}: no gradient for {n}"
        assert t.grad.shape == t.shape, (what, n, t.grad.shape, t.shape)
        _close(t.grad, r, f"{what} d{n}")


SHAPES = [(2, (32, 64)), (2, (21, 37)), (1, (9, 200)), (2, (16, 16, 16)), (1, (9, 7, 13))]


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("B,shape", SHAPES)
def test_energy_input_grads_parity(B, shape, ngp):
    fem = _fem(shape, ngp)
    x = _fields(B, shape, seed=sum(shape) * 13 + ngp, ngp=ngp)
    two = [(x["left"], 1.0), (x["right"], 0.0)]
    cases = [
        ("f", dict(f=x["f"], dirichlet=two), ["f"], {}),
        ("nu_numask_f_sum", dict(nu=x["nu"], nu_zero_mask=x["numask"], f=x["f"], dirichlet=two), ["f"],
         dict(reduction="sum", scale=0.37, c_k=1.7, c_f=0.6)),
        ("valuefield", dict(nu=x["nu"], f=x["f"], dirichlet=[(x["blob"], x["ubc"])]), ["f", "v0"],
         dict(scale=2.5, c_k=0.5, c_f=1.3)),
        ("f_bcast", dict(f=x["f"][:1], dirichlet=two), ["f"], {}),
        ("f_bare", dict(f=x["f"][0, 0].clone(), dirichlet=two), ["f"], {}),
        ("f_gp", dict(nu=x["nu"], f_gp=x["fgp"], dirichlet=[(x["blob"], x["ubc"])]), ["f_gp", "v0"],
         dict(c_f=0.8)),
        ("f_gp_bcast", dict(f_gp=x["fgp"][:1], dirichlet=two), ["f_gp"], dict(reduction="sum")),
    ]
    for name, kw, names, fixed in cases:
        _check(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, names, f"energy {name} {B}x{shape} ngp={ngp}",
               **fixed)


@pytest.mark.parametrize("B,shape", SHAPES)
def test_energy_f_gp_without_load_vector(B, shape, monkeypatch):
    monkeypatch.setattr(ops, "USE_LOAD_VECTOR", False)
    fem = _fem(shape, 2)
    x = _fields(B, shape, seed=5 + sum(shape))
    kw = dict(nu=x["nu"], f_gp=x["fgp"], dirichlet=[(x["blob"], x["ubc"])])
    _check(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, ["f_gp", "v0"], f"energy f_gp no-lv {shape}")


@pytest.mark.parametrize("shape", [(24, 40), (9, 7, 13)])
def test_energy_strided_channel_view(shape):
    fem = _fem(shape, 2)
    g = torch.Generator().manual_seed(3)
    inputs = torch.randn((3, 4) + shape, generator=g)
    u = torch.randn((3, 1) + shape, generator=g)
    x = _fields(3, shape, seed=4)
    ud = u.to(DEV).requires_grad_(True)
    inp = inputs.to(DEV).requires_grad_(True)
    dirichlet = [(x["left"].to(DEV), 1.0), (x["right"].to(DEV), 0.0)]
    loss = fem.energy_loss(ud, nu=inp[:, 0:1].exp(), f=inp[:, 2:3], dirichlet=dirichlet)
    loss.backward()
    i64 = to64(inputs).requires_grad_(True)
    lref = OL.energy_loss(oracle_for(fem), to64(u), nu=i64[:, 0:1].exp(), f=i64[:, 2:3],
                          dirichlet=[(to64(m), v) for m, v in dirichlet])
    (gi,) = torch.autograd.grad(lref, [i64])
    assert torch.count_nonzero(inp.grad[:, [1, 3]]) == 0
    _close(inp.grad[:, 2], gi[:, 2], "energy strided f view")


@pytest.mark.parametrize("shape", [(21, 37), (9, 7, 13)])
def test_batch_expanded_inputs(shape):
    """Fields given as one (1, ...) parameter expanded over the batch (stride_b = 0 with batch B): the parameter gets
    the batch sum and the expanded tensor its per-sample gradient, as autograd gives the reference."""
    B = 3
    fem = _fem(shape, 2)
    x = _fields(B, shape, seed=23)
    sp = (B, 1) + tuple(shape)

    def leaves(dev, dtype):
        ps = [x[k][:1].to(dev, dtype).clone().requires_grad_(True) for k in ("f", "ubc", "nu")]
        es = [p.expand(sp) for p in ps]
        for e in es:
            e.retain_grad()
        return ps, es

    def run(dev, dtype, energy, residual):
        ps, es = leaves(dev, dtype)
        u = x["u"].to(dev, dtype).requires_grad_(True)
        blob, left = x["blob"].to(dev, dtype), x["left"].to(dev, dtype)
        loss = energy(u, nu=x["nu"].to(dev, dtype), f=es[0], dirichlet=[(blob, es[1])], c_k=0.7, c_f=1.2)
        loss = loss + residual(u, nu=es[2], f=es[0], dirichlet=[(left, 1.0)], jac=0.4)
        loss.backward()
        return [t.grad for t in ps + es + [u]]

    o = oracle_for(fem)
    got = run(DEV, torch.float32, fem.energy_loss, fem.residual_loss)
    ref = run("cpu", torch.float64, lambda u, **kw: OL.energy_loss(o, u, **kw),
              lambda u, **kw: OL.residual_loss(o, u, **kw))
    names = ["f", "u_bc", "nu", "f expanded", "u_bc expanded", "nu expanded", "u"]
    for n, a, b in zip(names, got, ref):
        assert a.shape == b.shape, (n, a.shape, b.shape)
        _close(a, b, f"expanded {n} {shape}")


def test_overlapping_value_fields_last_mask_wins():
    """Two overlapping masks, both with value fields, through the input-gradient launch itself (the fused forward
    takes one value field): at the overlap only the later mask's field gets the gradient."""
    for shape in [(21, 37), (9, 7, 13)]:
        fem = _fem(shape, 3)
        x = _fields(2, shape, seed=17)
        m0 = x["blob"]
        m1 = (torch.rand(x["blob"].shape, generator=torch.Generator().manual_seed(9)) > 0.6).float()
        v0, v1 = x["ubc"], torch.randn(x["ubc"].shape, generator=torch.Generator().manual_seed(10))
        dev = [t.to(DEV) for t in (x["u"], x["nu"], x["f"], m0, m1, v0, v1)]
        u, nu, f, dm0, dm1, dv0, dv1 = dev
        _, _, (g0, g1) = ops.energy_input_grads_raw(fem.geometry, u, nu=nu, f=f, dirichlet=[(dm0, dv0), (dm1, dv1)],
                                                    scale=0.7, c_k=1.2, c_f=0.9, want_values=(True, True))
        r0, r1 = to64(v0).requires_grad_(True), to64(v1).requires_grad_(True)
        lref = OL.energy_loss(oracle_for(fem), to64(x["u"]), nu=to64(x["nu"]), f=to64(x["f"]),
                              dirichlet=[(to64(m0), r0), (to64(m1), r1)], scale=0.7, c_k=1.2, c_f=0.9)
        gr0, gr1 = torch.autograd.grad(lref, [r0, r1])
        assert torch.count_nonzero(gr0[(m0 > 0.5) & (m1 > 0.5)]) == 0
        _close(g0, gr0, f"overlap v0 {shape}")
        _close(g1, gr1, f"overlap v1 {shape}")
        _, _, (h0, h1) = ops.residual_input_grads_raw(
            fem.geometry, u, *_residual_R(fem, u, nu, f, [(dm0, dv0), (dm1, dv1)], 0.3), nu=nu, f=f,
            dirichlet=[(dm0, dv0), (dm1, dv1)], jac=0.3, want_values=(True, True))
        r0, r1 = to64(v0).requires_grad_(True), to64(v1).requires_grad_(True)
        lref = OL.residual_loss(oracle_for(fem), to64(x["u"]), nu=to64(x["nu"]), f=to64(x["f"]),
                                dirichlet=[(to64(m0), r0), (to64(m1), r1)], jac=0.3)
        gr0, gr1 = torch.autograd.grad(lref, [r0, r1])
        _close(h0, gr0, f"residual overlap v0 {shape}")
        _close(h1, gr1, f"residual overlap v1 {shape}")


def _residual_R(fem, u, nu, f, dirichlet, jac):
    """R of the oracle in fp32 on the device (the fused residual takes one value field)."""
    R = OL.residual_vector(oracle_for(fem), to64(u), nu=to64(nu), f=to64(f),
                           dirichlet=[(to64(m), to64(v)) for m, v in dirichlet], jac=jac)
    return (R[:, 0].float().to(DEV).contiguous(),)


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("B,shape", SHAPES)
def test_residual_input_grads_parity(B, shape, ngp):
    fem = _fem(shape, ngp)
    x = _fields(B, shape, seed=sum(shape) * 7 + ngp)
    two = [(x["left"], 1.0), (x["right"], 0.0)]
    u = x["u"]
    cases = [
        ("nu_f", u, dict(nu=x["nu"], f=x["f"], dirichlet=two), ["nu", "f"], dict(jac=0.37)),
        ("valuefield", u, dict(nu=x["nu"], f=x["f"], dirichlet=[(x["blob"], x["ubc"])]), ["nu", "v0"], {}),
        ("nu_bcast_f_bare", u, dict(nu=x["nu"][:1], f=x["f"][0, 0].clone(), dirichlet=two), ["nu", "f"],
         dict(jac=1.9)),
        # only the value field carries the batch: the launch batch is taken from it, as in the energy form
        ("valuefield_batched_only", u[:1], dict(nu=x["nu"][:1], f=x["f"][:1], dirichlet=[(x["blob"][:1], x["ubc"])]),
         ["nu", "v0"], dict(jac=0.8)),
    ]
    for name, u0, kw, names, fixed in cases:
        _check(fem, fem.residual_loss, OL.residual_loss, u0, kw, names,
               f"residual {name} {B}x{shape} ngp={ngp}", **fixed)


# ---------------------------------------------------------------------------------------------- autograd plumbing
def _energy_grads(fem, x, mult=1.0, twice=False):
    u = x["u"].to(DEV).requires_grad_(True)
    f = x["f"].to(DEV).requires_grad_(True)
    v = x["ubc"].to(DEV).requires_grad_(True)
    kw = dict(nu=x["nu"].to(DEV), dirichlet=[(x["blob"].to(DEV), v)])
    loss = mult * fem.energy_loss(u, f=f, **kw)
    if twice:
        loss = loss + fem.residual_loss(u, f=f, **kw)
    loss.backward()
    return u.grad, f.grad, v.grad


def test_autograd_scaling_accumulation_and_determinism():
    fem = _fem((33, 40), 2)
    x = _fields(2, (33, 40), seed=1)
    g1 = _energy_grads(fem, x)
    g1b = _energy_grads(fem, x)
    for a, b in zip(g1, g1b):
        assert torch.equal(a, b)
    g37 = _energy_grads(fem, x, mult=3.7)
    for a, b in zip(g37, g1):
        assert rel_l2(a.cpu(), 3.7 * b.cpu()) < 1e-6
    gsum = _energy_grads(fem, x, twice=True)
    u = x["u"].to(DEV).requires_grad_(True)
    f = x["f"].to(DEV).requires_grad_(True)
    v = x["ubc"].to(DEV).requires_grad_(True)
    fem.residual_loss(u, nu=x["nu"].to(DEV), f=f, dirichlet=[(x["blob"].to(DEV), v)]).backward()
    for a, b, c in zip(gsum, g1, (u.grad, f.grad, v.grad)):
        assert rel_l2(a.cpu(), (b + c).cpu()) < 1e-6


def test_inplace_edit_between_forward_and_backward_raises():
    fem = _fem((16, 24), 2)
    x = _fields(1, (16, 24), seed=2)
    f = x["f"].to(DEV).requires_grad_(True)
    fw = f * 1.0
    loss = fem.energy_loss(x["u"].to(DEV), f=fw)
    fw.add_(1.0)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        loss.backward()


def test_z_own_with_input_grads_raises():
    fem = _fem((9, 8, 8), 2)
    x = _fields(1, (9, 8, 8), seed=3)
    f = x["f"].to(DEV).requires_grad_(True)
    with pytest.raises(DiffNetFEMError):
        ops.fem_energy(fem.geometry, x["u"].to(DEV), f=f, z_own=(1, 5))


# ---------------------------------------------------------------------------------------------- default path
@pytest.mark.parametrize("B,shape", [(64, (256, 256)), (16, (64, 64, 64))])
def test_default_path_bit_identical(B, shape):
    fem = _fem(shape, 2)
    g = torch.Generator(device=DEV).manual_seed(0)
    sp = (B, 1) + shape
    u0 = torch.randn(sp, generator=g, device=DEV)
    nu = torch.rand(sp, generator=g, device=DEV) + 0.5
    f = torch.randn(sp, generator=g, device=DEV)
    m0 = torch.zeros(sp, device=DEV); m0[..., 0] = 1
    ubc = torch.randn(sp, generator=g, device=DEV)

    def run(f_grad, v_grad):
        u = u0.clone().requires_grad_(True)
        ff = f.clone().requires_grad_(f_grad)
        vv = ubc.clone().requires_grad_(v_grad)
        loss = fem.energy_loss(u, nu=nu, f=ff, dirichlet=[(m0, vv)])
        loss.backward()
        return loss.detach(), u.grad

    l0, g0 = run(False, False)
    for fg, vg in ((True, False), (False, True)):
        l1, g1 = run(fg, vg)
        assert torch.equal(l0, l1) and torch.equal(g0, g1)


@pytest.mark.parametrize("B,shape", [(64, (256, 256)), (16, (64, 64, 64))])
def test_identities_at_benchmark_sizes(B, shape):
    fem = _fem(shape, 2)
    g = torch.Generator(device=DEV).manual_seed(1)
    sp = (B, 1) + shape
    u = torch.randn(sp, generator=g, device=DEV)
    nu = torch.rand(sp, generator=g, device=DEV) + 0.5
    f = torch.randn(sp, generator=g, device=DEV).requires_grad_(True)
    m0 = torch.zeros(sp, device=DEV); m0[..., 0] = 1
    d = [(m0, 1.0)]
    # c_k keeps the stiffness term (|grad u|^2 ~ (2/h)^2 for a random u) near the source term, so that L(u, f) -
    # L(u, 0) is not lost to the fp32 rounding of the element energies; both losses from the fp64 reduction
    kw = dict(nu=nu, dirichlet=d, reduction="sum", c_k=1e-6)
    fem.energy_loss(u, f=f, **kw).backward()
    L1 = float(ops.energy_raw(fem.geometry, u, f=f.detach(), want_grad=False, want_double=True, **kw)[3])
    L0 = float(ops.energy_raw(fem.geometry, u, want_grad=False, want_double=True, **kw)[3])
    lhs = float((f.grad.double() * f.detach().double()).sum())
    assert abs(lhs - (L1 - L0)) <= 1e-5 * abs(L1 - L0), (lhs, L1, L0)
    nup = nu.clone().requires_grad_(True)
    R = fem.residual_loss(u, nu=nup, dirichlet=d)
    R.backward()
    lhs = float((nup.grad.double() * nu.double()).sum())
    assert abs(lhs - 2 * float(R)) <= 1e-5 * 2 * float(R), (lhs, float(R))


def test_adam_on_u_and_f_matches_oracle():
    shape = (17, 23)
    fem = _fem(shape, 2)
    x = _fields(2, shape, seed=11)
    dirichlet = [(x["left"], 1.0), (x["right"], 0.0)]

    def run(device, loss_fn, dtype):
        u = x["u"].to(device, dtype).clone().requires_grad_(True)
        f = x["f"].to(device, dtype).clone().requires_grad_(True)
        opt = torch.optim.Adam([u, f], lr=1e-2)
        d = [(m.to(device, dtype), v) for m, v in dirichlet]
        for _ in range(5):
            opt.zero_grad()
            loss = loss_fn(u, nu=x["nu"].to(device, dtype), f=f, dirichlet=d) + (f ** 2).mean()
            loss.backward()
            opt.step()
        return u.detach().cpu().double(), f.detach().cpu().double()

    o = oracle_for(fem)
    ug, fg = run(DEV, fem.energy_loss, torch.float32)
    uo, fo = run("cpu", lambda u, **kw: OL.energy_loss(o, u, **kw), torch.float64)
    assert rel_l2(ug, uo) <= 1e-4 and rel_l2(fg, fo) <= 1e-4
