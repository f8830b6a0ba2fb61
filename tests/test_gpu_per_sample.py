"""Per-sample fused losses: reduction="none" for the energy and residual forms.

Every per-sample loss and every gradient of a weighted sum of them is compared with the fp64 oracle applied to
one-sample slices, over both 2-D and both 3-D kernel families, the source forms, the Dirichlet variants and Gauss
rules 2-4.  Then the identities with the "mean" launch at the benchmark sizes, bit-reproducibility, the workspace
contract, the C-ABI refusals, the autograd plumbing and CUDA-graph capture of a prepared call.
"""
import ctypes as C

import pytest
import torch

from conftest import rel_l2, rel_scalar
from helpers import GRAD_MAX_RTOL, GRAD_RTOL, LOSS_RTOL, oracle_for, to64
from oracle import losses as OL
from diffnet_b200 import DiffNet2DFEM, DiffNet3DFEM, ops
from diffnet_b200 import _lib as L

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CONSTS = dict(c_k=0.7, c_f=1.3, scale=0.37)


def _fem(shape, ngp=2, lengths=None):
    if len(shape) == 2:
        H, W = shape
        return DiffNet2DFEM(None, domain_sizes=(W, H, 1), domain_lengths=lengths or (1.3, 0.9, 1.0), domain_size=W,
                            ngp_1d=ngp)
    D, H, W = shape
    return DiffNet3DFEM(None, domain_sizes=(W, H, D), domain_lengths=lengths or (1.1, 0.9, 1.2), domain_size=W,
                        ngp_1d=ngp)


def _fields(B, shape, seed, ngp=2):
    g = torch.Generator().manual_seed(seed)
    sp = (B, 1) + tuple(shape)
    left = torch.zeros(sp); left[..., 0] = 1
    right = torch.zeros(sp); right[..., -1] = 1
    elems = tuple(s - 1 for s in shape)
    return dict(u=torch.randn(sp, generator=g), nu=torch.exp(0.5 * torch.randn(sp, generator=g)),
                f=torch.randn(sp, generator=g), left=left, right=right,
                blob=(torch.rand(sp, generator=g) > 0.7).float(), ubc=torch.randn(sp, generator=g),
                numask=(torch.rand(sp, generator=g) > 0.85).float(),
                fgp=torch.randn((B, ngp ** len(shape)) + elems, generator=g))


def _sample(x, b, nsd):
    """Sample b of an input: a batched (B, 1|ngp, ...) tensor is sliced, a batch-1 one is shared."""
    if torch.is_tensor(x):
        return x[b:b + 1] if x.dim() == nsd + 2 and x.shape[0] > 1 else x
    if isinstance(x, dict):
        return {k: _sample(v, b, nsd) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return type(x)(_sample(v, b, nsd) for v in x)
    return x


def _map(kw, fn, names):
    """kw with every tensor passed through fn; requires_grad on the named inputs ('v0'.. index the values)."""
    out = {}
    for k, v in kw.items():
        if k == "dirichlet":
            out[k] = [(fn(m), fn(val).requires_grad_(f"v{i}" in names) if torch.is_tensor(val) else val)
                      for i, (m, val) in enumerate(v)]
        elif torch.is_tensor(v):
            out[k] = fn(v).requires_grad_(k in names)
        else:
            out[k] = v
    return out


def _wrt(kw, names):
    return [kw[n] for n in names if not n.startswith("v")] + \
        [val for i, (_, val) in enumerate(kw.get("dirichlet", ())) if f"v{i}" in names]


def _close(g, gref, what):
    g = g.detach().cpu().double()
    gref = gref.detach().double().reshape(g.shape)
    assert rel_l2(g, gref) <= GRAD_RTOL, f"{what}: rel-L2 {rel_l2(g, gref):.3e}"
    em = float((g - gref).abs().max() / gref.abs().max().clamp_min(1e-300))
    assert em <= GRAD_MAX_RTOL, f"{what}: max-norm {em:.3e}"


def _oracle_losses(fem, oracle_fn, u64, kw64, fixed):
    """fp64 oracle per sample: oracle_fn on every one-sample slice -> (B,) (mean over one sample's elements for the
    energy, sum of R^2 for the residual)."""
    o, nsd = oracle_for(fem), fem.nsd
    return torch.stack([oracle_fn(o, u64[b:b + 1], **_sample(kw64, b, nsd), **fixed) for b in range(u64.shape[0])])


def _check(fem, loss_fn, oracle_fn, u, kw, names, what, seed=0, **fixed):
    """loss[b] against the oracle per sample, and the gradient of sum_b w_b loss[b] for a random w w.r.t. u and the
    named inputs (exactly zero on Dirichlet nodes)."""
    B = u.shape[0]
    w = torch.randn(B, generator=torch.Generator().manual_seed(seed + 11), dtype=torch.float64)
    dev_kw = _map(kw, lambda t: t.detach().to(DEV).clone(), names)
    ud = u.to(DEV).requires_grad_(True)
    loss = loss_fn(ud, **dev_kw, reduction="none", **fixed)
    assert loss.shape == (B,) and loss.dtype == torch.float32, (what, loss.shape)
    (loss * w.float().to(DEV)).sum().backward()
    ref_kw = _map(kw, lambda t: to64(t).clone(), names)
    u64 = to64(u).requires_grad_(True)
    lref = _oracle_losses(fem, oracle_fn, u64, ref_kw, fixed)
    for b in range(B):
        e = rel_scalar(loss[b].item(), lref[b].item())
        assert e <= LOSS_RTOL, f"{what}: loss[{b}] rel {e:.3e} ({loss[b].item()} vs {lref[b].item()})"
    refs = torch.autograd.grad((lref * w).sum(), [u64] + _wrt(ref_kw, names))
    _close(ud.grad, refs[0], what + " du")
    for m, _ in kw.get("dirichlet", ()):
        hit = (m.to(DEV) > 0.5).expand_as(ud.grad)
        assert torch.count_nonzero(ud.grad[hit]) == 0, f"{what}: du not exactly 0 on Dirichlet nodes"
    for n, t, r in zip(names, _wrt(dev_kw, names), refs[1:]):
        assert t.grad is not None and t.grad.shape == t.shape, (what, n)
        _close(t.grad, r, f"{what} d{n}")


def _plan(B, shape, nfields, has_nu=0):
    """dn_debug_plan of the streaming planner for this shape (148 SMs, the B200's)."""
    nsd = len(shape)
    g = ops._geom_struct(ops.Geometry(nsd, shape[-1], shape[-2], shape[0] if nsd == 3 else 1, 1.0, 1.0, 1.0), B)
    out = (C.c_int64 * 16)()
    L.check(L.lib().dn_debug_plan(C.byref(g), nfields, has_nu, out), "dn_debug_plan")
    return list(out)


def _streams(B, shape, nfields, has_nu=0):
    """(eligible, grid) of the streaming planner for this shape."""
    out = _plan(B, shape, nfields, has_nu)
    return out[0], out[2]


def _check_on_fresh_workspace(fem, loss_fn, oracle_fn, u, kw, names, what, **fixed):
    """_check on a stream of its own (a fresh workspace), then: the workspace is all zero again."""
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        _check(fem, loss_fn, oracle_fn, u, kw, names, what, **fixed)
        s.synchronize()
        ws = ops._workspaces[(torch.device(DEV).index, s.cuda_stream)]
        assert torch.count_nonzero(ws) == 0, f"{what}: workspace not zero after a reduction='none' call"


# d/dnu is checked where the kernels produce it: the general 2-D kernel has no d/dnu with nu_zero_mask or f_gp.  A 2-D
# energy call that wants d/dnu runs on the general kernel; the cases without it take the "stream" path's kernel.
CASES = {
    "no_nu_one_mask": (lambda x: dict(dirichlet=[(x["left"], 1.0)]), []),
    "no_mask_nu_f": (lambda x: dict(nu=x["nu"], f=x["f"]), ["nu"]),
    "numask_two_masks": (lambda x: dict(nu=x["nu"], f=x["f"], nu_zero_mask=x["numask"],
                                         dirichlet=[(x["left"], 1.0), (x["right"], 0.0)]), []),
    "three_overlapping": (lambda x: dict(nu=x["nu"], f=x["f"],
                                          dirichlet=[(x["left"], 1.0), (x["blob"], -0.5), (x["right"], 0.25)]), ["nu"]),
    "value_field": (lambda x: dict(nu=x["nu"], f=x["f"], dirichlet=[(x["blob"], x["ubc"])]), ["nu"]),
    "f_gp": (lambda x: dict(nu=x["nu"], f_gp=x["fgp"], dirichlet=[(x["left"], 1.0)]), []),
}
PATHS_2D = [("stream", (64, 128), 5), ("general", (37, 45), 3), ("warp", (32, 64), 5)]


@pytest.mark.parametrize("ngp", [2, 3, 4])
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("path,shape,B", PATHS_2D)
def test_energy_2d(path, shape, B, case, ngp, monkeypatch):
    if path == "warp":
        monkeypatch.setenv("DN_2D_PATH", "warp")
    if path == "stream":
        ok, grid = _streams(B, shape, 4)
        assert ok and grid >= 2 * B, "the streaming case must cut every image into several chunks"
    fem = _fem(shape, ngp)
    x = _fields(B, shape, seed=ngp + len(case), ngp=ngp)
    build, names = CASES[case]
    _check(fem, fem.energy_loss, OL.energy_loss, x["u"], build(x), names, f"2-D {path} {case} ngp={ngp}",
           seed=ngp, **CONSTS)


def test_energy_2d_balanced_split_with_remainder(monkeypatch):
    """The streaming 2-D kernel's balanced one-wave split with bal_rem > 0: images [0, bal_rem) own bal_q + 1 chunks,
    the others bal_q -- both branches of the slot -> sample map."""
    monkeypatch.setenv("DN_T2_FILL_PCT", "0")    # every resident slot gets a CTA ...
    monkeypatch.setenv("DN_T2_CPS", "1")         # ... and there is one per SM: 148 slots over 9 images
    shape, B = (160, 64), 9
    if torch.cuda.get_device_properties(DEV).multi_processor_count != 148:
        pytest.skip("the split below is planned for 148 SMs")
    out = _plan(B, shape, 5, 1)
    assert out[0] == 1 and out[7] == 16 and out[8] == 4, out[:9]
    fem = _fem(shape)
    x = _fields(B, shape, seed=13)
    kw = dict(nu=x["nu"], f=x["f"], dirichlet=[(x["left"], 1.0), (x["right"], 0.0)])
    # no d/dnu here: it sends a 2-D energy call to the general kernel
    _check_on_fresh_workspace(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, [], "2-D balanced rem", **CONSTS)
    _check_on_fresh_workspace(fem, fem.residual_loss, OL.residual_loss, x["u"], kw, ["nu", "f"], "2-D balanced rem R",
                              jac=0.8)


def test_energy_3d_tile_block_smaller_than_a_warp():
    """A 5 x 5 x 200 volume runs on k_fem3d with 25-thread blocks and 50 z-chunks per sample: the finishing warp has
    fewer lanes than its sample has slots, and must still sum and zero every slot."""
    shape, B = (200, 5, 5), 2
    fem = _fem(shape)
    x = _fields(B, shape, seed=17)
    kw = dict(nu=x["nu"], f=x["f"], dirichlet=[(x["left"], 1.0), (x["right"], 0.0)])
    _check_on_fresh_workspace(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, ["nu"], "3-D 25-thread tile",
                              **CONSTS)
    _check_on_fresh_workspace(fem, fem.residual_loss, OL.residual_loss, x["u"], kw, ["nu", "f"],
                              "3-D 25-thread tile R", jac=0.8)


@pytest.mark.parametrize("shape", [(64, 128), (37, 45)])
def test_energy_2d_f_gp_without_load_vector(shape, monkeypatch):
    monkeypatch.setattr(ops, "USE_LOAD_VECTOR", False)
    fem = _fem(shape, 3)
    x = _fields(4, shape, seed=3, ngp=3)
    kw = dict(nu=x["nu"], f_gp=x["fgp"], dirichlet=[(x["left"], 1.0), (x["blob"], 0.0)])
    _check(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, ["f_gp"], f"2-D f_gp no-lv {shape}", **CONSTS)


def test_energy_2d_channel_slice_views():
    """u and nu as channel slices of (B, 3, H, W) tensors: strided views, the general kernel."""
    shape, B = (24, 40), 4
    fem = _fem(shape)
    x = _fields(B, shape, seed=21)
    packed = torch.cat([x["u"], x["nu"], x["f"]], 1)
    kw = dict(nu=packed[:, 1:2], f=packed[:, 2:3], dirichlet=[(x["left"], 1.0), (x["right"], 0.0)])
    _check(fem, fem.energy_loss, OL.energy_loss, packed[:, 0:1].contiguous(), kw, ["nu"], "2-D channel slices",
           **CONSTS)


CASES_3D = {
    "nu1": (lambda x: dict(f=x["f"], dirichlet=[(x["left"], 0.0), (x["right"], 1.0)]), []),
    "nu_nodal": (lambda x: dict(nu=x["nu"], f=x["f"], dirichlet=[(x["left"], 0.0), (x["right"], 1.0)]), ["nu"]),
}
SHAPES_3D = [("stream_iso", (16, 16, 16), (1.0, 1.0, 1.0), 3), ("stream_aniso", (16, 12, 20), None, 3),
             ("tile_odd", (9, 7, 13), None, 2), ("tile_aniso", (16, 12, 20), None, 3)]


@pytest.mark.parametrize("case", sorted(CASES_3D))
@pytest.mark.parametrize("name,shape,lengths,B", SHAPES_3D)
def test_energy_3d(name, shape, lengths, B, case, monkeypatch):
    if name.startswith("tile"):
        monkeypatch.setenv("DN_3D_PATH", "tile")
    fem = _fem(shape, 2, lengths)
    x = _fields(B, shape, seed=7 + B)
    build, names = CASES_3D[case]
    _check(fem, fem.energy_loss, OL.energy_loss, x["u"], build(x), names, f"3-D {name} {case}", **CONSTS)


@pytest.mark.parametrize("shape,B", [((64, 128), 5), ((37, 45), 3), ((16, 12, 20), 3), ((9, 7, 13), 2)])
def test_residual(shape, B):
    """per-sample sum(R^2) and the weighted backward, including d/dnu and d/df (residual input-gradient launch)."""
    fem = _fem(shape)
    x = _fields(B, shape, seed=5 + B)
    kw = dict(nu=x["nu"], f=x["f"], dirichlet=[(x["left"], 1.0), (x["right"], 0.0)])
    _check(fem, fem.residual_loss, OL.residual_loss, x["u"], kw, ["nu", "f"], f"residual {shape}", jac=0.8)


@pytest.mark.parametrize("shape,B", [((64, 128), 4), ((37, 45), 3), ((16, 12, 20), 2)])
@pytest.mark.parametrize("shared", [False, True])
def test_input_grads(shape, B, shared):
    """d/df, d/df_gp, d/d(value field) and residual d/dnu under "none", per-sample fields and fields shared by the
    batch (a (1, ...) field: the weighted sum over the samples)."""
    fem = _fem(shape)
    x = _fields(B, shape, seed=31 + B)
    one = (lambda t: t[:1].clone()) if shared else (lambda t: t)
    kw = dict(nu=x["nu"], f=one(x["f"]), dirichlet=[(x["blob"], one(x["ubc"]))])
    _check(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, ["f", "v0"], f"energy df dv shared={shared}", **CONSTS)
    kw = dict(nu=one(x["nu"]), f_gp=one(x["fgp"]), dirichlet=[(x["left"], 1.0)])
    _check(fem, fem.energy_loss, OL.energy_loss, x["u"], kw, ["f_gp"], f"energy df_gp shared={shared}", **CONSTS)
    kw = dict(nu=one(x["nu"]), f=one(x["f"]), dirichlet=[(x["blob"], one(x["ubc"]))])
    _check(fem, fem.residual_loss, OL.residual_loss, x["u"], kw, ["nu", "f", "v0"],
           f"residual dnu df dv shared={shared}", jac=1.1)


def _bench_inputs(shape, B, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    sp = (B, 1) + tuple(shape)
    u = torch.randn(sp, generator=g, device=DEV)
    nu = torch.exp(0.5 * torch.randn(sp, generator=g, device=DEV))
    f = torch.randn(sp, generator=g, device=DEV)
    left = torch.zeros(sp, device=DEV); left[..., 0] = 1
    right = torch.zeros(sp, device=DEV); right[..., -1] = 1
    return u, dict(nu=nu, f=f, dirichlet=[(left, 1.0), (right, 0.0)])


@pytest.mark.parametrize("shape,B", [((256, 256), 64), ((512, 512), 16), ((64, 64, 64), 16)])
def test_identities_at_benchmark_sizes(shape, B):
    fem = _fem(shape, 2, (1.0,) * 3)
    geom = fem.geometry
    u, kw = _bench_inputs(shape, B)
    lm, gm, _, lm64 = ops.energy_raw(geom, u, **kw, want_double=True)
    ln, gn, _, ln64 = ops.energy_raw(geom, u, **kw, reduction="none", want_double=True)
    assert ln64.shape == (B,)
    assert abs(float(ln64.mean()) - float(lm64)) <= 1e-12 * abs(float(lm64))
    assert rel_l2(gn / B, gm) <= 1e-6                  # the gradient of loss_none.mean()
    # sample b of the batch against a launch of that sample alone (another launch shape)
    for b in (0, B // 2, B - 1):
        l1, g1, _, l164 = ops.energy_raw(geom, u[b:b + 1], **_sample_kw(kw, b), reduction="none", want_double=True)
        assert rel_scalar(float(l164[0]), float(ln64[b])) <= 1e-6
        assert rel_l2(g1[0], gn[b]) <= 1e-6
    # a one-hot cotangent: exactly zero gradient on every other sample
    k = B // 3
    ud = u.clone().requires_grad_(True)
    loss = fem.energy_loss(ud, **kw, reduction="none")
    loss[k].backward()
    others = torch.cat([ud.grad[:k], ud.grad[k + 1:]])
    assert torch.count_nonzero(others) == 0
    assert rel_l2(ud.grad[k], gn[k]) == 0.0
    # two identical launches: bit-identical per-sample values and gradients
    ln2, gn2, _, ln642 = ops.energy_raw(geom, u, **kw, reduction="none", want_double=True)
    assert torch.equal(ln64, ln642) and torch.equal(ln, ln2) and torch.equal(gn, gn2)


def _sample_kw(kw, b):
    return {k: ([(m[b:b + 1], v) for m, v in val] if k == "dirichlet" else val[b:b + 1]) for k, val in kw.items()}


@pytest.mark.parametrize("shape,B,env", [((256, 256), 8, {}), ((37, 45), 5, {}), ((32, 64), 6, {"DN_2D_PATH": "warp"}),
                                         ((16, 16, 16), 4, {}), ((9, 7, 13), 3, {})])
def test_workspace_contract(shape, B, env, monkeypatch):
    """After a "none" call the workspace is all zero again: a "mean" call on it is bit-identical to one on a fresh
    workspace, and (with DN_POISON_OUTPUTS=1, set by the suite) all B loss values are written."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    fem = _fem(shape, 2, (1.0,) * 3)
    u, kw = _bench_inputs(shape, B, seed=3)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        ln, _, _ = ops.energy_raw(fem.geometry, u, **kw, reduction="none")
        rn, _ = ops.residual_raw(fem.geometry, u, **{k: v for k, v in kw.items() if k != "f"}, reduction="none")
        torch.cuda.current_stream().synchronize()
        assert torch.isfinite(ln).all() and torch.isfinite(rn).all()
        ws = ops._workspaces[(torch.device(DEV).index, s1.cuda_stream)]
        assert torch.count_nonzero(ws) == 0, "workspace not zero after a reduction='none' call"
        lm1, gm1, _ = ops.energy_raw(fem.geometry, u, **kw)
    with torch.cuda.stream(s2):
        lm2, gm2, _ = ops.energy_raw(fem.geometry, u, **kw)
    torch.cuda.synchronize()
    assert torch.equal(lm1, lm2) and torch.equal(gm1, gm2)


def test_c_abi_refusals():
    """The C entry points refuse reduction = none with mean_count, z-slab ownership or a bad residual reduction."""
    lib = L.lib()
    fem = _fem((16, 32))
    u = torch.randn(2, 16, 32, device=DEV)
    fld = L.dn_field(u.data_ptr(), u.stride(0), 0, u.stride(1))
    grad = torch.empty_like(u)
    loss = torch.empty(2, device=DEV)
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cs = L.dn_consts(1.0, 1.0, 1.0, L.DN_REDUCE_NONE, 0)
    for kw in (dict(mean_count=5.0), dict(z_own=(1, 8))):
        g = ops._geom_struct(fem.geometry, 2, kw.get("z_own"), kw.get("mean_count", 0.0))
        rc = lib.dn_fem_energy_2d_f32(C.byref(fld), None, None, None, None, 0, None, C.byref(g), C.byref(cs),
                                      C.c_void_p(grad.data_ptr()), None, C.c_void_p(ws.data_ptr()), ws.numel(), None,
                                      C.c_void_p(loss.data_ptr()), stream)
        assert rc == L.DN_EINVAL and b"none" in lib.dn_last_error(), kw
    g = ops._geom_struct(fem.geometry, 2)
    rc = lib.dn_fem_residual_reduce_2d_f32(C.byref(fld), None, None, None, 0, 1, C.byref(g), 1.0,
                                           C.c_void_p(grad.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), None,
                                           C.c_void_p(loss.data_ptr()), stream, 0)
    assert rc == L.DN_EINVAL


def test_scale_per_sample():
    x = torch.randn(5, 7, 13, device=DEV)               # 91 floats per sample: unaligned rows after sample 0
    fac = torch.tensor([0.5, -2.0, 1.0, 0.0, 3.0], device=DEV)
    want = x * fac[:, None, None]
    ops.scale_per_sample_(x, fac)
    assert torch.equal(x, want)
    # more samples than a grid has rows in y: the kernel walks the samples
    x = torch.randn(70001, 3, device=DEV)
    fac = torch.randn(70001, device=DEV)
    want = x * fac[:, None]
    ops.scale_per_sample_(x, fac)
    assert torch.equal(x, want)


def test_autograd_plumbing():
    shape, B = (64, 128), 6
    fem = _fem(shape)
    x = _fields(B, shape, seed=41)
    u = x["u"].to(DEV)
    kw = dict(nu=x["nu"].to(DEV), f=x["f"].to(DEV), dirichlet=[(x["left"].to(DEV), 1.0)])
    _, g, _ = ops.energy_raw(fem.geometry, u, **kw, reduction="none")
    w = torch.randn(B, device=DEV)
    for name, reduce, scale in (("sum", lambda l: l.sum(), torch.ones(B, device=DEV)),
                                ("weighted", lambda l: (w * l).sum(), w)):
        ud = u.clone().requires_grad_(True)
        reduce(fem.energy_loss(ud, **kw, reduction="none")).backward()
        assert rel_l2(ud.grad, g * scale[:, None, None]) <= 1e-6, name
    # the (loss, grad) pair outside autograd: grad is the gradient of loss.sum()
    l2, g2 = fem.energy_loss_and_grad(u, **kw, reduction="none")
    assert l2.shape == (B,) and torch.equal(g2, g)
    # a second backward through the same node still raises
    ud = u.clone().requires_grad_(True)
    loss = fem.energy_loss(ud, **kw, reduction="none")
    loss.sum().backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already run"):
        loss.sum().backward()


def test_prepared_energy_graph_capture():
    shape, B = (64, 128), 5
    fem = _fem(shape)
    x = _fields(B, shape, seed=43)
    u = x["u"].to(DEV)
    kw = dict(nu=x["nu"].to(DEV), f=x["f"].to(DEV), dirichlet=[(x["left"].to(DEV), 1.0), (x["right"].to(DEV), 0.0)])
    call = fem.prepare_energy(u, **kw, reduction="none")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        call()                                           # warm-up on the capture stream (workspace allocated here)
    torch.cuda.current_stream().wait_stream(s)
    loss_e, grad_e = (t.clone() for t in ops.energy_raw(fem.geometry, u, **kw, reduction="none")[:2])
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        loss, grad = call()
    call.loss.zero_(); call.grad.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert loss.shape == (B,)
    assert torch.equal(loss, loss_e) and torch.equal(grad, grad_e)
