"""The CUDA entry points at their launch-geometry limits.

The launchers switch on size limits that the small shapes of the other suites never reach:

* batches past the 65535 limit of a grid's y / z axis (B = 70001 on tiny meshes): the fused losses under every
  reduction, their input gradients (the 2-D input-gradient launch puts one sample per grid z and slices the batch),
  gauss_pt_evaluation_all and its adjoint, the load vector and the per-sample scaling;
* the batch slices of the 3-D gp-eval launches (grid z = samples x element layers / node planes) and meshes of more
  than 65535 layers (the forward then runs the flat general-basis kernel, the y-march adjoint one sample and a slice
  of its node planes per launch);
* fields whose later samples start past 2^31 bytes and 2^31 elements, with a sample that straddles each boundary
  inside a node row, and the adj3 <-> y-march switch at ngp^3 * elements = 2^31.

Each case is compared with the fp64 oracle on the samples at the boundaries and with a B = 1 launch of the same
sample (bit-exact for the fused 2-D u gradient, 2e-6 relative otherwise); per-sample losses are compared with the
per-sample oracle.  The large cases check the free device memory first and skip, with the amount, when it is short;
none needs more than ~27 GiB.
"""
import math

import pytest
import torch

from conftest import rel_scalar
from helpers import GRAD_MAX_RTOL, GRAD_RTOL, LOSS_RTOL, oracle_for, to64
from oracle import losses as OL
from diffnet_b200 import DiffNet2DFEM, DiffNet3DFEM, ops

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
B1_RTOL = 2e-6            # a B = 1 launch of the same sample, where the plan changes the summation order


@pytest.fixture(autouse=True)
def _release_memory():
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _need(gib):
    free, _ = torch.cuda.mem_get_info()
    if free < gib * 2 ** 30:
        pytest.skip(f"needs {gib} GiB of free device memory, {free / 2 ** 30:.1f} GiB free")


def _fem(shape, ngp=2):
    if len(shape) == 2:
        H, W = shape
        return DiffNet2DFEM(None, domain_sizes=(W, H, 1), domain_lengths=(1.3, 0.9, 1.0), domain_size=W, ngp_1d=ngp)
    D, H, W = shape
    return DiffNet3DFEM(None, domain_sizes=(W, H, D), domain_lengths=(1.1, 0.9, 1.2), domain_size=W, ngp_1d=ngp)


def _rel_max(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double().reshape(a.shape)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _close(g, gref, what):
    g = g.detach().cpu().double()
    gref = gref.detach().cpu().double().reshape(g.shape)
    e = float(torch.linalg.norm(g - gref) / torch.linalg.norm(gref).clamp_min(1e-300))
    assert e <= GRAD_RTOL, f"{what}: rel-L2 {e:.3e}"
    em = _rel_max(g, gref)
    assert em <= GRAD_MAX_RTOL, f"{what}: max-norm {em:.3e}"


def _same_b1(big, one, exact, what):
    if exact:
        assert torch.equal(big, one), f"{what}: differs from the B = 1 launch"
    else:
        e = _rel_max(big, one)
        assert e <= B1_RTOL, f"{what}: {e:.3e} from the B = 1 launch"


# ============================================================================ batches past the grid axes
B_BIG = 70001
IDX = [0, 65534, 65535, 65536, B_BIG - 1]
TINY = {
    "2d_stream": ((8, 8), {}),
    "2d_warp": ((8, 8), {"DN_2D_PATH": "warp"}),
    "2d_general": ((7, 9), {}),
    "3d_stream": ((4, 4, 8), {}),
    "3d_tile": ((4, 4, 8), {"DN_3D_PATH": "tile"}),
}


def _tiny_fields(shape, seed, ngp=2):
    g = torch.Generator().manual_seed(seed)
    sp = (B_BIG, 1) + tuple(shape)
    left = torch.zeros((1, 1) + tuple(shape)); left[..., 0] = 1
    right = torch.zeros((1, 1) + tuple(shape)); right[..., -1] = 1
    elems = tuple(s - 1 for s in shape)
    return dict(u=torch.randn(sp, generator=g), nu=torch.exp(0.5 * torch.randn(sp, generator=g)),
                f=torch.randn(sp, generator=g), left=left, right=right,
                blob=(torch.rand(sp, generator=g) > 0.7).float(), ubc=torch.randn(sp, generator=g),
                fgp=torch.randn((B_BIG, ngp ** len(shape)) + elems, generator=g))


def _leaves(kw, names, fn):
    out = {}
    for k, v in kw.items():
        if k == "dirichlet":
            out[k] = [(fn(m), fn(val).requires_grad_(f"v{i}" in names) if torch.is_tensor(val) else val)
                      for i, (m, val) in enumerate(v)]
        else:
            out[k] = fn(v).requires_grad_(k in names)
    return out


def _wrt(kw, names):
    return [kw[n] for n in names if not n.startswith("v")] + \
        [val for i, (_, val) in enumerate(kw.get("dirichlet", ())) if f"v{i}" in names]


def _sample_rows(kw, rows):
    """The inputs of the given samples: a batched tensor is indexed, a shared (batch-1) one is kept."""
    cut = lambda t: t[rows] if t.shape[0] > 1 else t
    return {k: ([(cut(m), cut(v) if torch.is_tensor(v) else v) for m, v in kw[k]] if k == "dirichlet" else cut(kw[k]))
            for k in kw}


def _oracle_per_sample(fem, form, u64, kw64, fixed):
    """fp64 per-sample losses of the batch u64 (reduction="none": the energy of a sample is the mean over its
    elements, the residual loss the sum of its R^2), and the number of elements of one sample."""
    o = oracle_for(fem)
    if form == "energy":
        return OL.energy_density(o, u64, **kw64, **fixed).flatten(1).mean(1), math.prod(fem.geometry.elems)
    return (OL.residual_vector(o, u64, **kw64, **fixed) ** 2).flatten(1).sum(1), 1


def _total(form, red, per, nel, w):
    """The batch loss of a reduction from per-sample losses (a subset of the batch gives the same gradients at its
    samples, the mean still dividing by the whole batch)."""
    if red == "none":
        return (per * w).sum()
    if red == "mean":
        return per.sum() / B_BIG
    return per.sum() * nel


def _check_batch_past_axes(fem, form, kw, names, reductions, what, seed, fixed, b1=True):
    """Every per-sample loss against the oracle; the gradients of u and of the named inputs at the samples of IDX
    (a shared input: its whole batch-summed gradient); and the same samples launched alone."""
    loss_fn = fem.energy_loss if form == "energy" else fem.residual_loss
    u = kw.pop("u")
    w = torch.randn(B_BIG, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)
    with torch.no_grad():
        kw64 = _leaves(kw, (), to64)
        per_all, nel = _oracle_per_sample(fem, form, to64(u), kw64, fixed)
        floor = per_all.abs()
        if form == "energy":      # the non-negative stiffness part of each sample's energy
            floor = floor + _oracle_per_sample(fem, form, to64(u), {k: v for k, v in kw64.items()
                                                                   if k not in ("f", "f_gp")},
                                               {**fixed, "c_f": 0.0})[0]
    # oracle gradients: of the IDX samples alone, or of the whole batch when a shared input is differentiated
    shared = any(t.shape[0] == 1 for t in _wrt(kw, names))
    rows = list(range(B_BIG)) if shared else IDX
    pick = IDX if shared else list(range(len(IDX)))
    sub = _sample_rows(kw, rows)
    u64 = to64(u[rows]).requires_grad_(True)
    ref_kw = _leaves(sub, names, lambda t: to64(t).clone())
    per, _ = _oracle_per_sample(fem, form, u64, ref_kw, fixed)
    for red in reductions:
        dev_kw = _leaves(kw, names, lambda t: t.detach().to(DEV).clone())
        ud = u.to(DEV).requires_grad_(True)
        loss = loss_fn(ud, **dev_kw, reduction=red, **fixed)
        if red == "none":
            assert loss.shape == (B_BIG,), (what, loss.shape)
            (loss * w.float().to(DEV)).sum().backward()
            err = (loss.detach().cpu().double() - per_all).abs() / floor
            bad = int(err.argmax())
            assert float(err[bad]) <= LOSS_RTOL, f"{what} none: loss[{bad}] {float(loss[bad])} vs {float(per_all[bad])}"
        else:
            loss.backward()
            lref = _total(form, red, per_all, nel, w)
            assert rel_scalar(loss.detach().cpu(), lref) <= LOSS_RTOL, f"{what} {red}: loss"
        refs = torch.autograd.grad(_total(form, red, per, nel, w[rows]), [u64] + _wrt(ref_kw, names),
                                   retain_graph=True)
        _close(ud.grad[IDX], refs[0][pick], f"{what} {red} du")
        for n, t, r in zip(names, _wrt(dev_kw, names), refs[1:]):
            assert t.grad is not None and t.grad.shape == t.shape, (what, red, n)
            if t.shape[0] > 1:
                _close(t.grad[IDX], r[pick], f"{what} {red} d{n}")
            else:
                _close(t.grad, r, f"{what} {red} d{n} (shared)")
        if red == "sum" and b1:
            for b in IDX:
                one_kw = _leaves(_sample_rows(kw, [b]), names, lambda t: t.detach().to(DEV).clone())
                u1 = u[b:b + 1].to(DEV).requires_grad_(True)
                loss_fn(u1, **one_kw, reduction="sum", **fixed).backward()
                _same_b1(ud.grad[b:b + 1], u1.grad, fem.nsd == 2 and form == "energy", f"{what} du[{b}]")
                for n, t, t1 in zip(names, _wrt(dev_kw, names), _wrt(one_kw, names)):
                    if t.shape[0] > 1:
                        _same_b1(t.grad[b:b + 1], t1.grad, False, f"{what} d{n}[{b}]")
    kw["u"] = u


@pytest.mark.parametrize("cfg", list(TINY))
def test_fused_losses_past_grid_axes(cfg, monkeypatch):
    shape, env = TINY[cfg]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    fem = _fem(shape)
    x = _tiny_fields(shape, seed=len(cfg) * 7 + sum(shape))
    two = [(x["left"], 1.0), (x["right"], 0.0)]
    fixed = dict(c_k=0.7, c_f=1.3, scale=0.37)
    # energy: u and nu (fused), f (the input-gradient launch), batched
    _check_batch_past_axes(fem, "energy", dict(u=x["u"], nu=x["nu"], f=x["f"], dirichlet=two), ["nu", "f"],
                           ("mean", "sum", "none"), f"{cfg} energy", 1, fixed)
    # energy: f_gp and a value field, batched
    _check_batch_past_axes(fem, "energy", dict(u=x["u"], nu=x["nu"], f_gp=x["fgp"], dirichlet=[(x["blob"], x["ubc"])]),
                           ["f_gp", "v0"], ("mean", "none"), f"{cfg} energy f_gp/value", 2, dict(c_f=0.8), b1=False)
    # energy: shared f and value field (one batch-summed gradient; "none" expands them over the batch)
    _check_batch_past_axes(fem, "energy", dict(u=x["u"], f=x["f"][:1], dirichlet=[(x["left"], x["ubc"][:1])]),
                           ["f", "v0"], ("sum", "none"), f"{cfg} energy shared", 3, {}, b1=False)
    # residual: nu, f and a value field, batched; then nu and f shared
    _check_batch_past_axes(fem, "residual", dict(u=x["u"], nu=x["nu"], f=x["f"], dirichlet=[(x["blob"], x["ubc"])]),
                           ["nu", "f", "v0"], ("sum", "none"), f"{cfg} residual", 4, dict(jac=0.4))
    _check_batch_past_axes(fem, "residual", dict(u=x["u"], nu=x["nu"][:1], f=x["f"][:1], dirichlet=two),
                           ["nu", "f"], ("sum", "none"), f"{cfg} residual shared", 5, {}, b1=False)


def _gp_ref(fem, t64, whichs):
    o = oracle_for(fem)
    fn = {"N": o.gauss_pt_evaluation, "dx": o.gauss_pt_evaluation_der_x, "dy": o.gauss_pt_evaluation_der_y,
          "dz": getattr(o, "gauss_pt_evaluation_der_z", None)}
    return [fn[w](t64) for w in whichs]


def _load_vector_ref(fem, f_gp):
    o = oracle_for(fem)
    u = torch.zeros((f_gp.shape[0], 1) + fem.geometry.spatial, dtype=torch.float64, requires_grad=True)
    w = o.gpw.double().reshape((1, -1) + (1,) * fem.nsd)
    (b,) = torch.autograd.grad((w * f_gp.double() * o.gauss_pt_evaluation(u)).sum(), u)
    return b[:, 0]


def _check_gp_family(fem, t, samples, what, adj_env=(None,), monkeypatch=None, lv=True):
    """gauss_pt_evaluation_all and its adjoint (autograd backward with random cotangents), the load vector, at the
    given samples: against the oracle and against a B = 1 launch of the same sample."""
    whichs = ("N", "dx", "dy") + (("dz",) if fem.nsd == 3 else ())
    B = t.shape[0]
    outs = fem.gauss_pt_evaluation_all(t)
    g = torch.Generator(device=DEV).manual_seed(B)
    cots = [torch.randn(o.shape, generator=g, device=DEV) for o in outs]
    ts = t[samples].cpu()
    refs = _gp_ref(fem, to64(ts), whichs)
    for w, o, r in zip(whichs, outs, refs):
        _close(o[samples], r, f"{what} gp {w}")
    for b in samples:
        for w, o, o1 in zip(whichs, outs, fem.gauss_pt_evaluation_all(t[b:b + 1])):
            _same_b1(o[b:b + 1], o1, False, f"{what} gp {w}[{b}]")
    t64 = to64(ts).requires_grad_(True)
    (gref,) = torch.autograd.grad(sum((r * to64(c[samples])).sum() for r, c in zip(_gp_ref(fem, t64, whichs), cots)),
                                  t64)
    for env in adj_env:
        if env is not None:
            monkeypatch.setenv("DN_GP_ADJ3", env)
        leaf = t.detach().clone().requires_grad_(True)
        torch.autograd.backward(fem.gauss_pt_evaluation_all(leaf), cots)
        _close(leaf.grad[samples], gref, f"{what} gp adjoint (DN_GP_ADJ3={env})")
        for b in samples:
            l1 = t[b:b + 1].detach().clone().requires_grad_(True)
            torch.autograd.backward(fem.gauss_pt_evaluation_all(l1), [c[b:b + 1] for c in cots])
            _same_b1(leaf.grad[b:b + 1], l1.grad, False, f"{what} gp adjoint[{b}] (DN_GP_ADJ3={env})")
        del leaf
    if lv:
        fgp = cots[0]
        for env in adj_env:
            if env is not None:
                monkeypatch.setenv("DN_GP_ADJ3", env)
            bvec = ops.load_vector(fem.geometry, fgp)
            _close(bvec[samples], _load_vector_ref(fem, fgp[samples].cpu()), f"{what} load vector (DN_GP_ADJ3={env})")
            for b in samples:
                _same_b1(bvec[b:b + 1], ops.load_vector(fem.geometry, fgp[b:b + 1]), False, f"{what} load vector[{b}]")


@pytest.mark.parametrize("shape", [(8, 8), (7, 9), (4, 4, 8)])
def test_gp_eval_load_vector_and_scaling_past_grid_axes(shape, monkeypatch):
    fem = _fem(shape)
    g = torch.Generator(device=DEV).manual_seed(sum(shape))
    t = torch.randn((B_BIG, 1) + shape, generator=g, device=DEV)
    _check_gp_family(fem, t, IDX, f"B={B_BIG} {shape}", ("1", "0") if len(shape) == 3 else (None,), monkeypatch)
    # x[b] *= factors[b] (the backward of every reduction="none" loss): every sample
    x = torch.randn((B_BIG,) + shape, generator=g, device=DEV)
    fac = torch.randn(B_BIG, generator=g, device=DEV)
    want = x * fac.reshape((-1,) + (1,) * len(shape))
    assert torch.equal(ops.scale_per_sample_(x, fac), want)


# ============================================================================ batch / layer slices of 3-D gp-eval
@pytest.mark.parametrize("layout", ["dense", "broadcast", "channel"])
def test_gp_eval_3d_batch_slices(layout, monkeypatch):
    """(nz, ny, nx) = (1000, 4, 6), B = 70: 999 element layers put 65 samples in the first slice of the forward and
    of the y-march adjoint, 5 in the second."""
    shape, B = (1000, 4, 6), 70
    fem = _fem(shape)
    g = torch.Generator(device=DEV).manual_seed(7)
    if layout == "dense":
        t = torch.randn((B, 1) + shape, generator=g, device=DEV)
    elif layout == "broadcast":
        t = torch.randn((1, 1) + shape, generator=g, device=DEV).expand((B, 1) + shape)
    else:
        t = torch.randn((B, 3) + shape, generator=g, device=DEV)[:, 1:2]
    _check_gp_family(fem, t, [0, 1, 64, 65, 66, B - 1], f"{layout} {shape} B={B}", ("1", "0"), monkeypatch,
                     lv=layout == "dense")


def test_gp_eval_3d_more_layers_than_grid_z(monkeypatch):
    """nz = 65538: 65537 element layers and 65538 node planes, more than grid z holds, in the forward and both
    adjoints (the z-marching adj3 and the y-march)."""
    shape, B = (65538, 3, 5), 2
    fem = _fem(shape)
    t = torch.randn((B, 1) + shape, generator=torch.Generator(device=DEV).manual_seed(3), device=DEV)
    _check_gp_family(fem, t, [0, 1], f"{shape} B={B}", ("1", "0"), monkeypatch)


# ============================================================================ offsets past 2^31
BOUNDS = (2 ** 29, 2 ** 30, 2 ** 31)        # elements: 2^31 bytes, 2^32 bytes, 2^31 elements


def _straddlers(stride, B, per=None):
    """Samples whose data crosses an element offset of BOUNDS (a sample b covers [b stride, b stride + per)), their
    neighbours and the last sample."""
    per = per or stride
    s = {B - 1}
    for bd in BOUNDS:
        b = bd // stride
        if bd - b * stride < per:
            s |= {b - 1, b, b + 1}
    return sorted(b for b in s if 0 <= b < B)


def _big_batch(per):
    """The smallest batch whose last sample starts past 2^31 elements, plus a few."""
    return 2 ** 31 // per + 12


LARGE = {
    # (256, 252): 2^31 elements fall inside node row 32 of sample 33288, 2^30 inside row 16 of 16644
    "2d_stream": ((256, 252), {}),
    "2d_warp": ((256, 252), {"DN_2D_PATH": "warp"}),
    "3d_stream": ((60, 64, 68), {}),
    "3d_tile": ((60, 64, 68), {"DN_3D_PATH": "tile"}),
}


def _per_sample_oracle(fem, u, kw, b):
    """loss[b] and its gradient with respect to u of sample b alone (reduction="none")."""
    o = oracle_for(fem)
    u64 = to64(u[b:b + 1]).requires_grad_(True)
    kw64 = {k: ([(to64(m[b:b + 1] if m.shape[0] > 1 else m), v) for m, v in val] if k == "dirichlet" else
                to64(val[b:b + 1] if val.shape[0] > 1 else val)) for k, val in kw.items()}
    loss = OL.energy_density(o, u64, **kw64).flatten(1).mean(1)[0]
    (g,) = torch.autograd.grad(loss, u64)
    return loss.detach(), g


@pytest.mark.parametrize("cfg", list(LARGE))
def test_fused_energy_past_2_31(cfg, monkeypatch):
    shape, env = LARGE[cfg]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    per = math.prod(shape)
    B = _big_batch(per)
    _need(2 * 4 * B * per / 2 ** 30 + 2)
    fem = _fem(shape)
    g = torch.Generator(device=DEV).manual_seed(per)
    u = torch.randn((B, 1) + shape, generator=g, device=DEV)
    one = (1, 1) + shape
    nu = torch.rand(one, generator=g, device=DEV) + 0.5
    f = torch.randn(one, generator=g, device=DEV)
    left = torch.zeros(one, device=DEV); left[..., 0] = 1
    kw = dict(nu=nu, f=f, dirichlet=[(left, 1.0)])
    loss, grad = fem.energy_loss_and_grad(u, reduction="none", **kw)
    for b in _straddlers(per, B):
        lref, gref = _per_sample_oracle(fem, u, kw, b)
        assert rel_scalar(loss[b].item(), lref) <= LOSS_RTOL, f"{cfg}: loss[{b}]"
        _close(grad[b], gref, f"{cfg} du[{b}]")
        l1, g1 = fem.energy_loss_and_grad(u[b:b + 1], reduction="none", **kw)
        _same_b1(grad[b:b + 1], g1, fem.nsd == 2, f"{cfg} du[{b}]")
        assert rel_scalar(loss[b].item(), l1.item()) <= B1_RTOL


@pytest.mark.parametrize("shape", [(256, 252), (60, 64, 68)])
def test_input_grads_past_2_31(shape):
    """dL/df of the energy, f batched: the input-gradient kernels read u and f and write grad f past 2^31."""
    per = math.prod(shape)
    B = _big_batch(per)
    _need(3 * 4 * B * per / 2 ** 30 + 2)
    fem = _fem(shape)
    g = torch.Generator(device=DEV).manual_seed(per + 1)
    u = torch.randn((B, 1) + shape, generator=g, device=DEV)
    f = torch.randn((B, 1) + shape, generator=g, device=DEV)
    left = torch.zeros((1, 1) + shape, device=DEV); left[..., 0] = 1
    kw = dict(dirichlet=[(left, 1.0)], reduction="sum", c_f=1.3)
    gf, _, _ = ops.energy_input_grads_raw(fem.geometry, u, f=f, want_f=True, **kw)
    o = oracle_for(fem)
    for b in _straddlers(per, B):
        f64 = to64(f[b:b + 1]).requires_grad_(True)
        lref = OL.energy_loss(o, to64(u[b:b + 1]), f=f64, dirichlet=[(to64(left), 1.0)], reduction="sum", c_f=1.3)
        (gref,) = torch.autograd.grad(lref, f64)
        _close(gf[b], gref, f"{shape} df[{b}]")
        g1, _, _ = ops.energy_input_grads_raw(fem.geometry, u[b:b + 1], f=f[b:b + 1], want_f=True, **kw)
        _same_b1(gf[b:b + 1], g1, False, f"{shape} df[{b}]")


def test_channel_slices_past_2_31():
    """nu, f and a mask as channel slices of one (B, 3, H, W) tensor: stride_b = 3 H W, so every field crosses 2^31
    elements at a third of the batch; the fused loss, and dL/df through the input-gradient launch."""
    shape = (256, 252)
    per = math.prod(shape)
    B = 2 ** 31 // (3 * per) + 12
    _need(4 * B * per * 6 / 2 ** 30 + 2)
    fem = _fem(shape)
    g = torch.Generator(device=DEV).manual_seed(5)
    inp = torch.empty((B, 3) + shape, device=DEV)
    inp[:, 0].uniform_(0.5, 1.5, generator=g)
    inp[:, 1].normal_(generator=g)
    inp[:, 2] = (torch.rand((B,) + shape, generator=g, device=DEV) > 0.8).float()
    u = torch.randn((B, 1) + shape, generator=g, device=DEV)
    kw = dict(nu=inp[:, 0:1], f=inp[:, 1:2], dirichlet=[(inp[:, 2:3], 1.0)])
    loss, grad = fem.energy_loss_and_grad(u, reduction="none", **kw)
    gf, _, _ = ops.energy_input_grads_raw(fem.geometry, u, want_f=True, reduction="none", **kw)
    o = oracle_for(fem)
    for b in _straddlers(3 * per, B, 3 * per):
        kb = dict(nu=inp[b:b + 1, 0:1], f=inp[b:b + 1, 1:2], dirichlet=[(inp[b:b + 1, 2:3], 1.0)])
        u64 = to64(u[b:b + 1]).requires_grad_(True)
        f64 = to64(kb["f"]).requires_grad_(True)
        lref = OL.energy_density(o, u64, nu=to64(kb["nu"]), f=f64, dirichlet=[(to64(inp[b:b + 1, 2:3]), 1.0)])
        lref = lref.flatten(1).mean(1)[0]
        gu, gfr = torch.autograd.grad(lref, [u64, f64])
        assert rel_scalar(loss[b].item(), lref.item()) <= LOSS_RTOL, f"channel slices: loss[{b}]"
        _close(grad[b], gu, f"channel slices du[{b}]")
        _close(gf[b], gfr, f"channel slices df[{b}]")
        l1, g1 = fem.energy_loss_and_grad(u[b:b + 1], reduction="none", **kb)
        _same_b1(grad[b:b + 1], g1, True, f"channel slices du[{b}]")
        gf1, _, _ = ops.energy_input_grads_raw(fem.geometry, u[b:b + 1], want_f=True, reduction="none", **kb)
        _same_b1(gf[b:b + 1], gf1, False, f"channel slices df[{b}]")


def test_gp_eval_2d_past_2_31():
    """256^2 x B: the (B, 4, 255, 255) Gauss-point tensor passes 2^31 elements; the forward and its adjoint (with the
    forward's own output as the cotangent)."""
    shape = (256, 256)
    fem = _fem(shape)
    per_gp = 4 * 255 * 255
    B = 2 ** 31 // per_gp + 12
    _need(4 * B * (per_gp + 2 * 65536) / 2 ** 30 + 2)
    t = torch.randn((B, 1) + shape, generator=torch.Generator(device=DEV).manual_seed(8), device=DEV)
    out = ops.gp_eval(fem.geometry, t, "N")
    gin = ops._gp_adj_raw(fem.geometry, out, 0)
    o = oracle_for(fem)
    samples = sorted(set(_straddlers(per_gp, B)) | set(_straddlers(65536, B)))
    for b in samples:
        t64 = to64(t[b:b + 1]).requires_grad_(True)
        r = o.gauss_pt_evaluation(t64)
        _close(out[b], r[0], f"gp 2-D past 2^31 [{b}]")
        (gref,) = torch.autograd.grad((r * to64(out[b:b + 1])).sum(), t64)
        _close(gin[b], gref[0, 0], f"gp adjoint 2-D past 2^31 [{b}]")
        _same_b1(out[b:b + 1], ops.gp_eval(fem.geometry, t[b:b + 1], "N"), False, f"gp 2-D [{b}]")
        _same_b1(gin[b:b + 1], ops._gp_adj_raw(fem.geometry, out[b:b + 1], 0), False, f"gp adjoint 2-D [{b}]")


@pytest.mark.parametrize("nelx,adj3", [(1023, True), (1025, False)])
def test_gp_adjoint_3d_at_the_adj3_threshold(nelx, adj3, monkeypatch):
    """(nelz, nely) = (256, 1024): 8 nelz nely nelx = 2^31 - 2^21 with nelx = 1023 (the z-marching adj3 runs, and the
    y-march forced by DN_GP_ADJ3=0 must agree with it), 2^31 + 2^21 with nelx = 1025 (adj3 gives way to the y-march).
    The cotangent is zero but on a few elements at the far corner and one in the middle, so the oracle runs on crops
    and every other node must come out exactly 0 (outputs are NaN-poisoned: an unwritten node is not)."""
    shape = (257, 1025, nelx + 1)
    fem = _fem(shape)
    nel = 256 * 1024 * nelx
    assert (8 * nel < 2 ** 31) == adj3
    _need(4 * (8 * nel + 2 * math.prod(shape)) / 2 ** 30 + 2)
    gout = torch.zeros((1, 8, 256, 1024, nelx), device=DEV)
    g = torch.Generator(device=DEV).manual_seed(nelx)
    corner = (slice(253, 256), slice(1019, 1024), slice(nelx - 6, nelx))
    mid = (slice(128, 129), slice(512, 513), slice(nelx // 2, nelx // 2 + 1))
    for c in (corner, mid):
        gout[(0, slice(None)) + c] = torch.randn((8,) + tuple(s.stop - s.start for s in c), generator=g, device=DEV)
    runs = [("default", None)] + ([("y-march", "0")] if adj3 else [])
    got = {}
    for name, env in runs:
        if env is not None:
            monkeypatch.setenv("DN_GP_ADJ3", env)
        gin = ops._gp_adj_raw(fem.geometry, gout, 0)
        for c in (corner, mid):
            nodes = tuple(slice(s.start, s.stop + 1) for s in c)
            cfem = _fem(tuple(s.stop - s.start for s in nodes))
            u64 = torch.zeros((1, 1) + tuple(s.stop - s.start for s in nodes), dtype=torch.float64,
                              requires_grad=True)
            r = oracle_for(cfem).gauss_pt_evaluation(u64)
            (gref,) = torch.autograd.grad((r * to64(gout[(0, slice(None)) + c])[None]).sum(), u64)
            _close(gin[(0,) + nodes], gref[0, 0], f"adj3 threshold nelx={nelx} {name}")
        nz = int(torch.count_nonzero(gin))
        inside = sum(int(torch.count_nonzero(gin[(0,) + tuple(slice(s.start, s.stop + 1) for s in c)]))
                     for c in (corner, mid))
        assert nz == inside, f"adj3 threshold nelx={nelx} {name}: {nz - inside} nodes outside the support"
        got[name] = gin[(0,) + tuple(slice(s.start, s.stop + 1) for s in corner)].clone()
        del gin
    if adj3:
        _same_b1(got["default"], got["y-march"], False, "adj3 against the y-march")
