"""torch.autograd.Function wrappers over the C ABI (the drop-in seam for DiffNet's loss()).

  fem_energy(...)    fused Poisson energy loss, differentiable w.r.t. u, nu, f, f_gp and Dirichlet value fields
  fem_residual(...)  assembled-residual loss  sum(R^2), differentiable w.r.t. u, nu, f and Dirichlet value fields
  gp_eval(...)       gauss_pt_evaluation{,_der_x,_der_y,_der_z}, differentiable w.r.t. its input

Everything runs on the CUDA stream torch considers current; there is no host sync inside and no
CPU path (CPU tensors raise).  See include/diffnet_fem.h for the C side.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib as L


@dataclass(frozen=True)
class Geometry:
    """Mesh description shared by every call (mirrors the reference's kwargs -> attributes,
    DiffNet/base.py:16-32, DiffNetFEM.py:42-51)."""
    nsd: int
    nx: int
    ny: int
    nz: int
    hx: float
    hy: float
    hz: float
    ngp_1d: int = 2

    @property
    def spatial(self) -> Tuple[int, ...]:
        return (self.ny, self.nx) if self.nsd == 2 else (self.nz, self.ny, self.nx)

    @property
    def elems(self) -> Tuple[int, ...]:
        return tuple(s - 1 for s in self.spatial)


# ------------------------------------------------------------------------------ marshalling
def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise L.DiffNetFEMError(
            f"{name} is on {t.device}: the FEM ops are CUDA (sm_100a) only, there is no CPU fallback")


def _nodal(t: torch.Tensor, nsd: int, name: str) -> torch.Tensor:
    """View `t` as (Bt, *nodes) with x contiguous.  Accepted layouts: bare nodes, (B, *nodes) and (B, 1, *nodes)
    -- what the reference's where()/conv broadcasting accepts (solve_in_object_3d.py:198-199 passes a bare (D,H,W)
    parameter)."""
    if t.dim() == nsd + 2:
        if t.shape[1] != 1:
            raise L.DiffNetFEMError(f"{name}: expected one channel, got shape {tuple(t.shape)}")
        t = t[:, 0]
    elif t.dim() == nsd:
        t = t.unsqueeze(0)
    elif t.dim() != nsd + 1:
        raise L.DiffNetFEMError(f"{name}: bad shape {tuple(t.shape)} for a {nsd}-D nodal field")
    if t.stride(-1) != 1:
        t = t.contiguous()
    return t


def _canon(t: torch.Tensor, geom: Geometry, name: str) -> torch.Tensor:
    """`_nodal` view of a CUDA fp32 field on the mesh nodes (bool / uint8 masks are converted)."""
    _require_cuda(t, name)
    if t.dtype != torch.float32:
        if t.dtype in (torch.bool, torch.uint8):
            t = t.to(torch.float32)
        else:
            raise L.DiffNetFEMError(f"{name} must be float32 (got {t.dtype})")
    t = _nodal(t, geom.nsd, name)
    if tuple(t.shape[1:]) != geom.spatial:
        raise L.DiffNetFEMError(f"{name}: spatial shape {tuple(t.shape[1:])} != mesh nodes {geom.spatial}")
    return t


def _field(t: Optional[torch.Tensor], B: int, nsd: int) -> L.dn_field:
    if t is None:
        return L.dn_field(None, 0, 0, 0)
    bt = t.shape[0]
    if bt != B and bt != 1:
        raise L.DiffNetFEMError(f"batch {bt} does not broadcast to {B}")
    sb = t.stride(0) if (bt == B and B > 1) else 0
    if nsd == 2:
        return L.dn_field(t.data_ptr(), sb, 0, t.stride(1))
    return L.dn_field(t.data_ptr(), sb, t.stride(1), t.stride(2))


def _geom_struct(geom: Geometry, B: int, z_own=None, mean_count=0.0) -> L.dn_geom:
    zo = z_own or (0, 0)
    return L.dn_geom(geom.nsd, B, geom.nx, geom.ny, geom.nz if geom.nsd == 3 else 1, geom.ngp_1d,
                     geom.hx, geom.hy, geom.hz if geom.nsd == 3 else 0.0, int(zo[0]), int(zo[1]),
                     float(mean_count))


def _new_out(shape, device, dtype=torch.float32) -> torch.Tensor:
    """Output buffer.  With DN_POISON_OUTPUTS=1 (set by the test-suite) it is NaN-filled first so
    that a node the kernel failed to write can never pass a parity check by accident."""
    if os.environ.get("DN_POISON_OUTPUTS"):
        return torch.full(shape, float("nan"), dtype=dtype, device=device)
    return torch.empty(shape, dtype=dtype, device=device)


_workspaces = {}
_ws_bytes = {}


class _on_device:
    """`with torch.cuda.device(dev)` costs ~10 us per call; skip it when `dev` is already current
    (the one-process-per-GPU case)."""

    def __init__(self, dev):
        self.ctx = None if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def _workspace_for(lib, g, geom, B, device, stream_ptr):
    key = (geom.nsd, B, geom.nx, geom.ny, geom.nz)
    n = _ws_bytes.get(key)
    if n is None:
        n = _ws_bytes[key] = lib.dn_fem_workspace_bytes(C.byref(g))
    return _workspace(device, stream_ptr, n)


def _workspace(device: torch.device, stream_ptr: int, nbytes: int) -> torch.Tensor:
    """Zero-initialised scratch (ticket counter + per-CTA partials), one per device and stream;
    the kernels leave it ready for the next call."""
    key = (device.index, stream_ptr)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.zeros(max(nbytes, 1 << 16), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


_REDUCTION = {"mean": 0, "sum": 1, "none": L.DN_REDUCE_NONE}


def _check_none(reduction, z_own=None, mean_count=0.0, link=None):
    """``reduction="none"`` gives one loss per sample, so a launch must hold whole samples: refuse what splits one."""
    if reduction != "none":
        return
    if z_own is not None:
        raise L.DiffNetFEMError("reduction='none' is not available with z_own: a z-slab holds part of a sample")
    if mean_count:
        raise L.DiffNetFEMError("reduction='none' takes no mean_count (each sample is divided by its element count)")
    if link is not None:
        raise L.DiffNetFEMError("reduction='none' is not available for a linked (z-slab) launch")


def _consts(c_k, c_f, scale, reduction, flags=0, z_own=None, mean_count=0.0, link=None) -> L.dn_consts:
    """``reduction``: "mean", "sum" or "none" (a (B,) loss, one value per sample)."""
    if reduction not in _REDUCTION:
        raise L.DiffNetFEMError("reduction must be 'mean', 'sum' or 'none'")
    _check_none(reduction, z_own, mean_count, link)
    return L.dn_consts(float(c_k), float(c_f), float(scale), _REDUCTION[reduction], flags)


def _loss_shape(reduction, B):
    return (B,) if reduction == "none" else ()


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check_f_gp(geom: Geometry, f_gp) -> torch.Tensor:
    _require_cuda(f_gp, "f_gp")
    ngp = geom.ngp_1d ** geom.nsd
    fg = f_gp if f_gp.dim() == geom.nsd + 2 else f_gp.unsqueeze(0)
    if tuple(fg.shape[1:]) != (ngp,) + geom.elems or fg.dtype != torch.float32:
        raise L.DiffNetFEMError(
            f"f_gp must be float32 (B|1, {ngp}, {geom.elems}); got {tuple(f_gp.shape)} {f_gp.dtype}")
    return fg


def _per_sample(t: Optional[torch.Tensor], B: int, expand: bool = False) -> Optional[torch.Tensor]:
    """The canonical view of a field whose gradient is wanted.  The launch writes ONE (1, ...) gradient summed over
    the batch for a field it reads with stride_b = 0.  A field that spans the batch with stride_b = 0 (``expand``)
    needs a gradient per sample (autograd's expand backward sums it), so its values are materialised here.
    ``expand=True`` (reduction="none": every sample's gradient gets its own weight) materialises a batch-1 field
    over the batch as well, at B times its memory."""
    if t is not None and B > 1 and t.shape[0] == B and t.stride(0) == 0:
        return t.contiguous()
    if expand and t is not None and B > 1 and t.shape[0] == 1:
        return t.expand((B,) + tuple(t.shape[1:])).contiguous()
    return t


class _Args:
    """The inputs of one fused-loss launch, canonicalised once (``_canon``, ``_check_f_gp``).

    ``B`` is the batch of the launch: the largest batch among all inputs (every other one is 1 or ``B``).  The ctypes
    arguments are ``c_u``, ``c_nu``, ``c_f``, ``c_fgp``, ``c_nzm``, ``c_R`` (``C.byref(dn_field)``, or None for an
    absent input) and ``marr``, ``nm`` (the ``dn_mask`` array and its length); this object holds the views they point
    into.  ``want`` names the fields (``"nu"``, ``"f"``, ``"f_gp"``) and ``want_values`` flags the tensor Dirichlet
    values (list order) whose gradient the launch writes: those take the ``_per_sample`` view (``per_sample=True``:
    a gradient per sample even for a field shared by the batch).  ``bind=True`` (a prepared call, which reads the
    same storage on every later call) refuses an input that would have to be copied."""

    def __init__(self, geom: Geometry, u=None, nu=None, f=None, f_gp=None, dirichlet=(), nu_zero_mask=None, R=None,
                 want=(), want_values=(), bind=False, per_sample=False):
        def canon(t, name):
            if t is None:
                return None
            c = _canon(t, geom, name)
            if bind and c.data_ptr() != t.data_ptr():
                raise L.DiffNetFEMError(
                    f"prepare_energy: {name} would have to be copied (dtype {t.dtype}, strides {tuple(t.stride())}); "
                    "a prepared call binds storage -- pass float32 tensors whose x axis is contiguous")
            return c

        n = len(dirichlet)
        if n > L.DN_MAX_MASKS:
            raise L.DiffNetFEMError(f"at most {L.DN_MAX_MASKS} Dirichlet conditions per call (got {n})")
        self.u, self.nu, self.f = canon(u, "u"), canon(nu, "nu"), canon(f, "f")
        self.nzm, self.R = canon(nu_zero_mask, "nu_zero_mask"), canon(R, "R")
        self.fg = None
        if f_gp is not None:
            self.fg = _check_f_gp(geom, f_gp)
            if not self.fg.is_contiguous():
                if bind:
                    raise L.DiffNetFEMError("prepare_energy: f_gp must be contiguous (a prepared call binds storage)")
                self.fg = self.fg.contiguous()
        masks = [canon(m, f"dirichlet[{i}].mask") for i, (m, _) in enumerate(dirichlet)]
        values = [canon(v, f"dirichlet[{i}].value") if torch.is_tensor(v) else None
                  for i, (_, v) in enumerate(dirichlet)]
        B = 1
        for t in (self.u, self.nu, self.f, self.nzm, self.R, self.fg, *masks, *values):
            if t is not None:
                B = max(B, t.shape[0])
        self.B = B
        if "nu" in want:
            self.nu = _per_sample(self.nu, B, per_sample)
        if "f" in want:
            self.f = _per_sample(self.f, B, per_sample)
        if "f_gp" in want:
            self.fg = _per_sample(self.fg, B, per_sample)
        flags = iter(want_values)
        self.want_v = [i for i, v in enumerate(values) if v is not None and next(flags, False)]
        for i in self.want_v:
            values[i] = _per_sample(values[i], B, per_sample)
        self.masks, self.values = masks, values
        self.dev = (self.u if self.u is not None else self.fg).device

        nsd = geom.nsd
        ref = lambda t: None if t is None else C.byref(_field(t, B, nsd))
        self.c_u, self.c_nu, self.c_f, self.c_nzm, self.c_R = map(ref, (self.u, self.nu, self.f, self.nzm, self.R))
        self.c_fgp = None
        if self.fg is not None:
            fg = self.fg
            self.c_fgp = C.byref(L.dn_field(fg.data_ptr(), fg.stride(0) if (fg.shape[0] == B and B > 1) else 0, 0, 0))
        self.marr, self.nm = (L.dn_mask * max(n, 1))(), n
        for i, (m, (_, v)) in enumerate(zip(masks, dirichlet)):
            self.marr[i].mask = _field(m, B, nsd)
            if values[i] is not None:
                self.marr[i].value_field = _field(values[i], B, nsd)
                self.marr[i].value = 0.0
            else:
                self.marr[i].value_field = L.dn_field(None, 0, 0, 0)
                self.marr[i].value = float(v)

    def grad_out(self, t: torch.Tensor, tail) -> torch.Tensor:
        """Gradient buffer for the canonical input ``t``: per sample, or one (1, ...) sum when ``t`` is broadcast."""
        return _new_out((self.B if (self.B > 1 and t.shape[0] == self.B) else 1,) + tuple(tail), self.dev)

    def value_grads(self, spatial):
        """Buffers for the wanted value-field gradients: (pointer array for the C call, [buffer | None per tensor
        value, list order])."""
        ptrs = (C.c_void_p * max(self.nm, 1))()
        bufs = {}
        for i in self.want_v:
            bufs[i] = self.grad_out(self.values[i], spatial)
            ptrs[i] = bufs[i].data_ptr()
        return ptrs, [bufs.get(i) for i, v in enumerate(self.values) if v is not None]


def load_vector(geom: Geometry, f_gp: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Assembled load vector b (Bf, *nodes) of a forcing given at the Gauss points (Bf = f_gp's batch, 1 when it is
    shared by the batch): b_a = sum over elements and Gauss points of w_g N_a(g) f_gp.  The forcing term of the
    reference's f_gp form (e8_2d_poisson_mms.py:154-175) is linear in u, so sum_g w_g f_g u_g = sum_a b_a u_a:
    pass ``b`` as ``f`` with ``load_vector=True`` and the fused kernels stream 4 bytes per node instead of
    4 * ngp bytes per element."""
    a = _Args(geom, f_gp=f_gp)
    if out is None:
        out = _new_out((a.B,) + geom.spatial, a.dev)
    g = _geom_struct(geom, a.B)
    with _on_device(a.dev):
        rc = L.lib().dn_fem_load_vector_f32(a.c_fgp, C.byref(g), C.c_void_p(out.data_ptr()),
                                            C.c_void_p(torch.cuda.current_stream(a.dev).cuda_stream))
    L.check(rc, "dn_fem_load_vector_f32")
    return out


# f_gp -> load vector, remembered per tensor OBJECT and version counter (an in-place update of f_gp re-assembles; a
# new tensor at a recycled address is a different object and misses).  Small: a training loop has one or two f_gp.
_LV_CACHE = []          # [(weakref(f_gp), version, geom key, b)]
_LV_CACHE_MAX = 8
USE_LOAD_VECTOR = os.environ.get("DN_LOAD_VECTOR", "1") != "0"


def _cached_load_vector(geom: Geometry, f_gp: torch.Tensor) -> torch.Tensor:
    import weakref
    key = (geom.nsd, geom.spatial, geom.ngp_1d)
    for i, (ref, ver, k, b) in enumerate(_LV_CACHE):
        if ref() is f_gp and k == key:
            if ver == f_gp._version:
                return b
            _LV_CACHE.pop(i)
            break
    _LV_CACHE[:] = [e for e in _LV_CACHE if e[0]() is not None][-(_LV_CACHE_MAX - 1):]
    b = load_vector(geom, f_gp)
    _LV_CACHE.append((weakref.ref(f_gp), f_gp._version, key, b))
    return b


def energy_raw(geom: Geometry, u, nu=None, f=None, f_gp=None, dirichlet=(), nu_zero_mask=None,
               c_k=1.0, c_f=1.0, scale=1.0, reduction="mean", want_grad=True, want_grad_nu=False,
               z_own=None, mean_count=0.0, want_double=False, load_vector=False):
    """One fused launch.  Returns (loss 0-dim fp32, grad_u (B,*spatial) or None,
    grad_nu or None[, loss fp64 0-dim]).  With ``reduction="none"`` both losses are (B,), one per sample, and the
    gradients are each sample's own.

    ``load_vector=True``: ``f`` is an assembled load vector (``load_vector()``), not a nodal source.  A call with
    ``f_gp`` takes that route by itself (assembling b once per f_gp tensor and version) whenever the streaming
    kernels can run the launch, and reads f_gp in the general kernels otherwise."""
    cs = _consts(c_k, c_f, scale, reduction, L.DN_F_LOAD_VECTOR if load_vector else 0, z_own, mean_count)
    if (f_gp is not None and f is None and USE_LOAD_VECTOR and not load_vector and z_own is None
            and not want_grad_nu):
        _check_f_gp(geom, f_gp)
        try:
            return energy_raw(geom, u, nu=nu, f=_cached_load_vector(geom, f_gp), dirichlet=dirichlet,
                              nu_zero_mask=nu_zero_mask, c_k=c_k, c_f=c_f, scale=scale, reduction=reduction,
                              want_grad=want_grad, want_grad_nu=False, mean_count=mean_count,
                              want_double=want_double, load_vector=True)
        except L.DiffNetFEMError as e:
            if e.code != L.DN_ENOSTREAM:
                raise                      # anything else is a real error; DN_ENOSTREAM: the general kernels read f_gp
    a = _Args(geom, u, nu, f, f_gp, dirichlet, nu_zero_mask)
    if load_vector and (a.f is None or a.fg is not None):
        raise L.DiffNetFEMError("load_vector=True: pass the assembled vector as f (and no f_gp)")
    B, dev = a.B, a.dev
    g = _geom_struct(geom, B, z_own, mean_count)
    grad = _new_out((B,) + geom.spatial, dev) if want_grad else None
    grad_nu = _new_out((B,) + geom.spatial, dev) if want_grad_nu else None
    loss = _new_out(_loss_shape(reduction, B), dev)
    loss64 = torch.empty(_loss_shape(reduction, B), dtype=torch.float64, device=dev) if want_double else None
    lib = L.lib()
    stream = torch.cuda.current_stream(dev).cuda_stream
    with _on_device(dev):
        ws = _workspace_for(lib, g, geom, B, dev, stream)
        fn = lib.dn_fem_energy_2d_f32 if geom.nsd == 2 else lib.dn_fem_energy_3d_f32
        rc = fn(a.c_u, a.c_nu, a.c_f, a.c_fgp, a.marr, a.nm, a.c_nzm, C.byref(g), C.byref(cs), _ptr(grad),
                _ptr(grad_nu), C.c_void_p(ws.data_ptr()), ws.numel(), _ptr(loss64), _ptr(loss), C.c_void_p(stream))
    L.check(rc, f"dn_fem_energy_{geom.nsd}d_f32")
    out = (loss, grad, grad_nu)
    return out + (loss64,) if want_double else out


class PreparedEnergy:
    """A fused energy call bound to fixed tensors: all marshalling (views, strides, ctypes
    structs, workspace, output buffers) is done once; ``__call__`` is one C call (~5 us of host
    time instead of ~50).  For loops that evaluate the loss on the SAME storage every iteration:
    u-as-parameter solves (solve_in_object_3d.py, LBFGS closures), the z-slab steps, benchmarks.

    The returned ``(loss, grad)`` are the SAME tensors on every call (overwritten in place):
    consume or copy them before calling again.  ``reduction="none"``: ``loss`` is a (B,) buffer.  In-place updates of the bound tensors are seen
    (pointers, not values, are captured); re-prepare if a tensor is reallocated."""

    def __init__(self, geom: Geometry, u, nu=None, f=None, f_gp=None, dirichlet=(), nu_zero_mask=None,
                 c_k=1.0, c_f=1.0, scale=1.0, reduction="mean", z_own=None, mean_count=0.0, link=None):
        """``link``: a ``_lib.dn_slab_link`` (3-D only, see include/diffnet_fem.h) -- the launch then also
        exchanges the z-halo planes of u with the neighbouring ranks and pushes the loss partial."""
        cs = _consts(c_k, c_f, scale, reduction, 0, z_own, mean_count, link)
        if link is not None and (geom.nsd != 3 or f_gp is not None):
            raise L.DiffNetFEMError("a linked (z-slab) call is 3-D with a nodal source term")
        if f is not None and f_gp is not None:
            raise L.DiffNetFEMError("give f or f_gp, not both")
        self.geom = geom
        self._a = a = _Args(geom, u, nu, f, f_gp, dirichlet, nu_zero_mask, bind=True)
        self.device, self._B = a.dev, a.B
        self._g = g = _geom_struct(geom, a.B, z_own, mean_count)
        self.grad = _new_out((a.B,) + geom.spatial, a.dev)
        self.loss = _new_out(_loss_shape(reduction, a.B), a.dev)
        self._loss_ptr = C.c_void_p(self.loss.data_ptr())
        grad = C.c_void_p(self.grad.data_ptr())
        lib = L.lib()
        fn, name = (lib.dn_fem_energy_2d_f32, "dn_fem_energy_2d_f32") if geom.nsd == 2 else \
            (lib.dn_fem_energy_3d_f32, "dn_fem_energy_3d_f32")
        # each call: (C function, arguments before the workspace, name); the workspace, loss and stream follow
        self._plain = (fn, (a.c_u, a.c_nu, a.c_f, a.c_fgp, a.marr, a.nm, a.c_nzm, C.byref(g), C.byref(cs), grad,
                            None), name)
        self._call = self._plain
        if link is not None:
            self._call = (lib.dn_fem_energy_3d_linked_f32,
                          (a.c_u, a.c_nu, a.c_f, a.marr, a.nm, a.c_nzm, C.byref(g), C.byref(cs), C.byref(link), grad),
                          "dn_fem_energy_3d_linked_f32")
        # f_gp: the assembled load vector is what the streaming kernels read (re-assembled when f_gp's version
        # counter moves); the first call falls back to the general kernels for good if they refuse the launch
        self._lv = None
        if a.fg is not None and link is None and z_own is None and USE_LOAD_VECTOR:
            bvec = load_vector(geom, a.fg)
            self._lv = (a.fg, a.fg._version, bvec)
            cs_lv = _consts(c_k, c_f, scale, reduction, L.DN_F_LOAD_VECTOR)
            self._call = (fn, (a.c_u, a.c_nu, C.byref(_field(bvec, a.B, geom.nsd)), None, a.marr, a.nm, a.c_nzm,
                               C.byref(g), C.byref(cs_lv), grad, None), name)
        self._ws = {}

    def __call__(self):
        dev = self.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        with _on_device(dev):
            ws = self._ws.get(stream)
            if ws is None:
                ws = self._ws[stream] = _workspace_for(L.lib(), self._g, self.geom, self._B, dev, stream)
            tail = (C.c_void_p(ws.data_ptr()), ws.numel(), None, self._loss_ptr, C.c_void_p(stream))
            if self._lv is not None and self._lv[0]._version != self._lv[1]:
                fg, _, bvec = self._lv
                load_vector(self.geom, fg, out=bvec)
                self._lv = (fg, fg._version, bvec)
            fn, head, name = self._call
            rc = fn(*head, *tail)
            if rc == L.DN_ENOSTREAM and self._lv is not None:     # the general kernels read f_gp from now on
                self._lv = None
                fn, head, name = self._call = self._plain
                rc = fn(*head, *tail)
        L.check(rc, name)
        return self.loss, self.grad


def residual_raw(geom: Geometry, u, nu=None, f=None, dirichlet=(), jac=1.0, apply_masks_to_input=True,
                 reduction="sum"):
    """R = jac*(K(nu) u' - F(f)) masked, and sum(R^2).  Returns (loss 0-dim, R (B,*spatial));
    ``reduction="none"``: loss (B,), the sum of R^2 over each sample."""
    if reduction not in ("sum", "none"):
        raise L.DiffNetFEMError("residual reduction must be 'sum' or 'none'")
    a = _Args(geom, u, nu, f, dirichlet=dirichlet)
    B, dev = a.B, a.dev
    g = _geom_struct(geom, B)
    R = _new_out((B,) + geom.spatial, dev)
    loss = _new_out(_loss_shape(reduction, B), dev)
    lib = L.lib()
    stream = torch.cuda.current_stream(dev).cuda_stream
    with _on_device(dev):
        ws = _workspace_for(lib, g, geom, B, dev, stream)
        fn = lib.dn_fem_residual_reduce_2d_f32 if geom.nsd == 2 else lib.dn_fem_residual_reduce_3d_f32
        rc = fn(a.c_u, a.c_nu, a.c_f, a.marr, a.nm, 1 if apply_masks_to_input else 0, C.byref(g), float(jac),
                _ptr(R), C.c_void_p(ws.data_ptr()), ws.numel(), None, _ptr(loss), C.c_void_p(stream),
                _REDUCTION[reduction])
    L.check(rc, f"dn_fem_residual_reduce_{geom.nsd}d_f32")
    return loss, R


def energy_input_grads_raw(geom: Geometry, u, nu=None, f=None, f_gp=None, dirichlet=(), nu_zero_mask=None,
                           c_k=1.0, c_f=1.0, scale=1.0, reduction="mean", mean_count=0.0, want_f=False,
                           want_f_gp=False, want_values=()):
    """dL/df, dL/df_gp and dL/d(value field) of the energy loss in ONE launch (dn_fem_energy_input_grads_*).
    ``want_values``: one flag per tensor Dirichlet value, in list order.  Returns (grad_f | None,
    grad_f_gp | None, [grad per tensor value | None]); a gradient of a field broadcast over the batch is (1, ...).
    ``reduction="none"``: every gradient is per sample, (B, ...), the gradient of that sample's loss."""
    cs = _consts(c_k, c_f, scale, reduction, 0, None, mean_count)
    want = ("f",) * want_f + ("f_gp",) * want_f_gp
    a = _Args(geom, u, nu, f, f_gp, dirichlet, nu_zero_mask, want=want, want_values=want_values,
              per_sample=reduction == "none")
    g = _geom_struct(geom, a.B, None, mean_count)
    gf = a.grad_out(a.f, geom.spatial) if want_f else None
    gfg = a.grad_out(a.fg, (geom.ngp_1d ** geom.nsd,) + geom.elems) if want_f_gp else None
    ptrs, gv = a.value_grads(geom.spatial)
    with _on_device(a.dev):
        lib = L.lib()
        fn = lib.dn_fem_energy_input_grads_2d_f32 if geom.nsd == 2 else lib.dn_fem_energy_input_grads_3d_f32
        rc = fn(a.c_u, a.c_nu, a.c_f, a.c_fgp, a.marr, a.nm, a.c_nzm, C.byref(g), C.byref(cs), _ptr(gf), _ptr(gfg),
                ptrs, C.c_void_p(torch.cuda.current_stream(a.dev).cuda_stream))
    L.check(rc, f"dn_fem_energy_input_grads_{geom.nsd}d_f32")
    return gf, gfg, gv


def residual_input_grads_raw(geom: Geometry, u, R, nu=None, f=None, dirichlet=(), jac=1.0, want_nu=False,
                             want_f=False, want_values=(), per_sample=False):
    """dL/dnu, dL/df and dL/d(value field) of the residual loss sum(R^2) in ONE launch
    (dn_fem_residual_input_grads_*); ``R`` is the residual the forward returned.  Returns (grad_nu | None,
    grad_f | None, [grad per tensor value | None]).  ``per_sample=True``: every gradient is (B, ...), the gradient
    of its sample's sum(R^2), also for a field shared by the batch."""
    want = ("nu",) * want_nu + ("f",) * want_f
    a = _Args(geom, u, nu, f, dirichlet=dirichlet, R=R, want=want, want_values=want_values, per_sample=per_sample)
    g = _geom_struct(geom, a.B)
    gnu = a.grad_out(a.nu, geom.spatial) if want_nu else None
    gf = a.grad_out(a.f, geom.spatial) if want_f else None
    ptrs, gv = a.value_grads(geom.spatial)
    with _on_device(a.dev):
        lib = L.lib()
        fn = lib.dn_fem_residual_input_grads_2d_f32 if geom.nsd == 2 else lib.dn_fem_residual_input_grads_3d_f32
        rc = fn(a.c_u, a.c_nu, a.c_f, a.c_R, a.marr, a.nm, C.byref(g), float(jac), _ptr(gnu), _ptr(gf), ptrs,
                C.c_void_p(torch.cuda.current_stream(a.dev).cuda_stream))
    L.check(rc, f"dn_fem_residual_input_grads_{geom.nsd}d_f32")
    return gnu, gf, gv


def scale_inplace_(x: torch.Tensor, factor: torch.Tensor) -> torch.Tensor:
    """x *= factor (0-dim device tensor), free when factor == 1 (checked on the device)."""
    _require_cuda(x, "x")
    assert x.is_contiguous() and x.dtype == torch.float32
    fac = factor.detach().to(device=x.device, dtype=torch.float32).reshape(())
    stream = torch.cuda.current_stream(x.device).cuda_stream
    with _on_device(x.device):
        rc = L.lib().dn_scale_inplace_f32(C.c_void_p(x.data_ptr()), x.numel(),
                                          C.c_void_p(fac.data_ptr()), C.c_void_p(stream))
    L.check(rc, "dn_scale_inplace_f32")
    return x


def scale_per_sample_(x: torch.Tensor, factors: torch.Tensor) -> torch.Tensor:
    """x[b] *= factors[b] for a (B, ...) tensor and a (B,) device tensor of factors, no host sync."""
    _require_cuda(x, "x")
    assert x.is_contiguous() and x.dtype == torch.float32
    B = x.shape[0]
    fac = factors.detach().to(device=x.device, dtype=torch.float32).reshape(B).contiguous()
    stream = torch.cuda.current_stream(x.device).cuda_stream
    with _on_device(x.device):
        rc = L.lib().dn_scale_per_sample_f32(C.c_void_p(x.data_ptr()), B, x.numel() // max(B, 1),
                                             C.c_void_p(fac.data_ptr()), C.c_void_p(stream))
    L.check(rc, "dn_scale_per_sample_f32")
    return x


def _scale(x: torch.Tensor, gout: torch.Tensor) -> torch.Tensor:
    """x *= grad_output: one factor (reduction "mean" / "sum"), or one per sample (reduction "none", gout (B,))."""
    return scale_inplace_(x, gout) if gout.dim() == 0 else scale_per_sample_(x, gout)


def _like_input(grad_b: torch.Tensor, ref: torch.Tensor, geom: Geometry) -> torch.Tensor:
    """Reduce/reshape a dense (B,*spatial) gradient to the shape of the tensor the user passed."""
    if ref.dim() == geom.nsd:                       # bare field broadcast over the batch
        return grad_b.sum(0) if grad_b.shape[0] > 1 else grad_b[0]
    bt = ref.shape[0]
    g = grad_b
    if bt == 1 and g.shape[0] > 1:
        g = g.sum(0, keepdim=True)
    return g.reshape(ref.shape)


# ------------------------------------------------------------------------------ autograd
class FEMEnergyFunction(torch.autograd.Function):
    """loss = energy(u, nu, ...); backward returns grad_output * dloss/du (and dloss/dnu).  With reduction="none"
    the loss is (B,) and grad_output weighs each sample's gradient (dn_scale_per_sample_f32).

    Forward AND gradient come from the single fused launch in forward(); backward only scales
    (in place, skipped on the device when grad_output == 1).  First-order only
    (once_differentiable), which is all Adam / LBFGS need.

    The gradient buffer is handed to autograd, not copied, and scaling it in place consumes it: a
    SECOND backward through the same node (``retain_graph=True``, or ``autograd.grad`` followed by
    ``backward``) raises instead of silently returning ``grad_output**2 * dL/du`` -- re-run the
    forward (one launch) to differentiate again.

    The tensor Dirichlet values follow the fixed arguments (``*values``, list order) so that autograd tracks them.
    When ``f``, ``f_gp`` or a value requires grad, backward runs ONE more launch (dn_fem_energy_input_grads_*) for
    those gradients; the inputs it reads are saved for backward, so an in-place change between forward and
    backward raises torch's version-counter error."""

    @staticmethod
    def forward(ctx, u, nu, geom, f, f_gp, dirichlet, nu_zero_mask, c_k, c_f, scale, reduction,
                z_own, mean_count, *values):
        need_u = ctx.needs_input_grad[0]
        need_nu = nu is not None and ctx.needs_input_grad[1]
        need_f = f is not None and ctx.needs_input_grad[3]
        need_fgp = f_gp is not None and ctx.needs_input_grad[4]
        need_v = tuple(ctx.needs_input_grad[13:])
        extra = need_f or need_fgp or any(need_v)
        if extra and z_own is not None:
            raise L.DiffNetFEMError("gradients w.r.t. f, f_gp or a Dirichlet value field are not available with "
                                    "z_own: a z-slab only holds a partial gradient")
        loss, grad, grad_nu = energy_raw(
            geom, u.detach(), None if nu is None else nu.detach(), f, f_gp, dirichlet,
            nu_zero_mask, c_k, c_f, scale, reduction, want_grad=need_u or need_nu,
            want_grad_nu=need_nu, z_own=z_own, mean_count=mean_count)
        ctx.geom = geom
        ctx.u_ref = u if need_u else None
        ctx.nu_ref = nu if need_nu else None
        head = [t for t in (grad if need_u else None, grad_nu) if t is not None]
        ctx.has = (need_u, need_nu)
        ctx.consumed = False
        ctx.nvalues = len(values)
        ctx.extra = None
        if extra:
            ctx.extra = (need_f, need_fgp, need_v, len(head), dirichlet, c_k, c_f, scale, reduction, mean_count)
            head += [u, nu, f, f_gp, nu_zero_mask] + [m for m, _ in dirichlet] + list(values)
        ctx.save_for_backward(*head)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        if ctx.consumed:
            raise RuntimeError(
                "FEMEnergyFunction: backward was already run through this node; its gradient buffer was scaled "
                "in place and handed to autograd.  Evaluate the loss again (one fused launch) for another backward.")
        ctx.consumed = True
        saved = list(ctx.saved_tensors)
        gu = gnu = None
        if ctx.has[0]:
            gu = _like_input(_scale(saved.pop(0), gout), ctx.u_ref, ctx.geom)
        if ctx.has[1]:
            gnu = _like_input(_scale(saved.pop(0), gout), ctx.nu_ref, ctx.geom)
        if ctx.extra is None:
            return (gu, gnu) + (None,) * (11 + ctx.nvalues)
        need_f, need_fgp, need_v, _, dirichlet, c_k, c_f, scale, reduction, mean_count = ctx.extra
        u, nu, f, f_gp, nzm = saved[:5]
        values = saved[5 + len(dirichlet):]
        gf, gfg, gv = energy_input_grads_raw(ctx.geom, u, nu, f, f_gp, dirichlet, nzm, c_k, c_f, scale, reduction,
                                             mean_count, want_f=need_f, want_f_gp=need_fgp, want_values=need_v)
        if gf is not None:
            gf = _like_input(_scale(gf, gout), f, ctx.geom)
        if gfg is not None:
            gfg = _scale(gfg, gout)
            if gfg.shape[0] > 1 and (f_gp.dim() == ctx.geom.nsd + 1 or f_gp.shape[0] == 1):
                gfg = gfg.sum(0, keepdim=True)    # reduction="none": per-sample gradients of a shared f_gp
            gfg = gfg.reshape(f_gp.shape)
        gv = [None if g is None else _like_input(_scale(g, gout), v, ctx.geom) for g, v in zip(gv, values)]
        return (gu, gnu, None, gf, gfg) + (None,) * 8 + tuple(gv)


class FEMResidualFunction(torch.autograd.Function):
    """loss = sum(R^2); dL/du = mask( K(nu) (2R) ) -- one more pass of the same operator
    (K is symmetric; R is already zero on the Dirichlet nodes).  reduction="none": loss[b] = sum of R^2 over sample
    b, and a (B,) grad_output weighs each sample's gradient.

    The tensor Dirichlet values follow the fixed arguments (``*values``).  When ``nu``, ``f`` or a value requires
    grad, backward runs ONE more launch (dn_fem_residual_input_grads_*) for those gradients."""

    @staticmethod
    def forward(ctx, u, geom, nu, f, dirichlet, jac, reduction, *values):
        loss, R = residual_raw(geom, u.detach(), nu, f, dirichlet, jac, True, reduction)
        ctx.geom, ctx.nu, ctx.dirichlet, ctx.jac, ctx.u_ref = geom, nu, dirichlet, jac, u
        ctx.per_sample = reduction == "none"
        ctx.nvalues = len(values)
        need_nu = nu is not None and ctx.needs_input_grad[2]
        need_f = f is not None and ctx.needs_input_grad[3]
        need_v = tuple(ctx.needs_input_grad[7:])
        ctx.extra = None
        if need_nu or need_f or any(need_v):
            ctx.extra = (need_nu, need_f, need_v)
            ctx.save_for_backward(R, u, nu, f, *[m for m, _ in dirichlet], *values)
        else:
            ctx.save_for_backward(R)
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        saved = ctx.saved_tensors
        R = saved[0]
        if ctx.extra is None:
            _, KR = residual_raw(ctx.geom, R, ctx.nu, None, ctx.dirichlet, ctx.jac, False)
            g = KR.mul_(2.0)
            g = _scale(g, gout)
            return (_like_input(g, ctx.u_ref, ctx.geom),) + (None,) * (6 + ctx.nvalues)
        need_nu, need_f, need_v = ctx.extra
        u, nu, f = saved[1:4]
        values = saved[4 + len(ctx.dirichlet):]
        gu = None
        if ctx.needs_input_grad[0]:
            _, KR = residual_raw(ctx.geom, R, nu, None, ctx.dirichlet, ctx.jac, False)
            gu = _like_input(_scale(KR.mul_(2.0), gout), ctx.u_ref, ctx.geom)
        gnu, gf, gv = residual_input_grads_raw(ctx.geom, u, R, nu, f, ctx.dirichlet, ctx.jac, want_nu=need_nu,
                                               want_f=need_f, want_values=need_v, per_sample=ctx.per_sample)
        if gnu is not None:
            gnu = _like_input(_scale(gnu, gout), nu, ctx.geom)
        if gf is not None:
            gf = _like_input(_scale(gf, gout), f, ctx.geom)
        gv = [None if g is None else _like_input(_scale(g, gout), v, ctx.geom) for g, v in zip(gv, values)]
        return (gu, None, gnu, gf, None, None, None) + tuple(gv)


_WHICH = {"N": 0, "dx": 1, "dy": 2, "dz": 3}


def _gp_raw(geom: Geometry, t: torch.Tensor, which: int) -> torch.Tensor:
    tc = _canon(t, geom, "tensor")
    B = tc.shape[0]
    g = _geom_struct(geom, B)
    out = _new_out((B, geom.ngp_1d ** geom.nsd) + geom.elems, tc.device)
    fld = _field(tc, B, geom.nsd)
    stream = torch.cuda.current_stream(tc.device).cuda_stream
    lib = L.lib()
    fn = lib.dn_fem_gp_eval_2d_f32 if geom.nsd == 2 else lib.dn_fem_gp_eval_3d_f32
    with _on_device(tc.device):
        rc = fn(C.byref(fld), C.byref(g), which, _ptr(out), C.c_void_p(stream))
    L.check(rc, "dn_fem_gp_eval")
    return out


def _gp_adj_raw(geom: Geometry, gout: torch.Tensor, which: int) -> torch.Tensor:
    """Transpose of `_gp_raw`: cotangent (B, ngp, elems) -> nodes (B, *spatial)."""
    gout = gout.contiguous()
    B = gout.shape[0]
    g = _geom_struct(geom, B)
    gin = _new_out((B,) + geom.spatial, gout.device)
    stream = torch.cuda.current_stream(gout.device).cuda_stream
    lib = L.lib()
    fn = lib.dn_fem_gp_eval_adj_2d_f32 if geom.nsd == 2 else lib.dn_fem_gp_eval_adj_3d_f32
    with _on_device(gout.device):
        rc = fn(_ptr(gout), C.byref(g), which, _ptr(gin), C.c_void_p(stream))
    L.check(rc, "dn_fem_gp_eval_adj")
    return gin


class GaussPointEvalFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, t, geom, which):
        ctx.geom, ctx.which, ctx.t_ref = geom, which, t
        return _gp_raw(geom, t.detach(), which)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        return _like_input(_gp_adj_raw(ctx.geom, gout, ctx.which), ctx.t_ref, ctx.geom), None, None


def _gp_multi_raw(geom: Geometry, t: torch.Tensor, whichs: Sequence[int]):
    """Several tables in one call (dn_fem_gp_eval_multi_*): a tuple of (B, ngp, elems) tensors."""
    tc = _canon(t, geom, "tensor")
    B = tc.shape[0]
    g = _geom_struct(geom, B)
    outs = [_new_out((B, geom.ngp_1d ** geom.nsd) + geom.elems, tc.device) for _ in whichs]
    fld = _field(tc, B, geom.nsd)
    stream = torch.cuda.current_stream(tc.device).cuda_stream
    lib = L.lib()
    fn = lib.dn_fem_gp_eval_multi_2d_f32 if geom.nsd == 2 else lib.dn_fem_gp_eval_multi_3d_f32
    n = len(whichs)
    wh = (C.c_int * n)(*whichs)
    ptrs = (C.c_void_p * n)(*[o.data_ptr() for o in outs])
    with _on_device(tc.device):
        rc = fn(C.byref(fld), C.byref(g), n, wh, ptrs, C.c_void_p(stream))
    L.check(rc, "dn_fem_gp_eval_multi")
    return tuple(outs)


class GaussPointEvalMultiFunction(torch.autograd.Function):
    """gauss_pt_evaluation + its derivatives of ONE nodal field in one launch; backward sums the
    cotangents of all tables in one adjoint launch."""

    @staticmethod
    def forward(ctx, t, geom, whichs):
        ctx.geom, ctx.whichs, ctx.t_ref = geom, tuple(whichs), t
        return _gp_multi_raw(geom, t.detach(), whichs)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *gouts):
        geom = ctx.geom
        used = [(w, g.contiguous()) for w, g in zip(ctx.whichs, gouts) if g is not None]
        if not used:
            return None, None, None
        B = used[0][1].shape[0]
        g = _geom_struct(geom, B)
        dev = used[0][1].device
        gin = _new_out((B,) + geom.spatial, dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        lib = L.lib()
        fn = lib.dn_fem_gp_eval_multi_adj_2d_f32 if geom.nsd == 2 else lib.dn_fem_gp_eval_multi_adj_3d_f32
        n = len(used)
        wh = (C.c_int * n)(*[w for w, _ in used])
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for _, t in used])
        with _on_device(dev):
            rc = fn(ptrs, C.byref(g), n, wh, _ptr(gin), C.c_void_p(stream))
        L.check(rc, "dn_fem_gp_eval_multi_adj")
        return _like_input(gin, ctx.t_ref, geom), None, None


class GaussPointEvalGeneralFunction(torch.autograd.Function):
    """gauss_pt_eval for any tensor-product Lagrange basis / rule in 1-3 dimensions
    (dn_fem_gp_eval_general_f32): the degree 2 / 3 bases and the 1-D surface stencils."""

    @staticmethod
    def forward(ctx, t, nsd, nb, ng, factors):
        _require_cuda(t, "tensor")
        if t.dtype != torch.float32:
            raise L.DiffNetFEMError(f"tensor must be float32 (got {t.dtype})")
        tc = _nodal(t.detach(), nsd, "tensor")
        B = tc.shape[0]
        sp = tuple(tc.shape[1:])                                   # ([nz, ny,] nx)
        if any((n - 1) % (nb - 1) for n in sp):
            raise L.DiffNetFEMError(f"nodes {sp}: (n - 1) must be a multiple of the basis degree {nb - 1}")
        nel = tuple((n - 1) // (nb - 1) for n in sp)
        n3 = (1,) * (3 - nsd) + sp                                 # (nz, ny, nx)
        fac = np.ascontiguousarray(np.asarray(factors, dtype=np.float32).reshape(nsd, ng, nb))
        out = _new_out((B, ng ** nsd) + nel, tc.device)
        fld = L.dn_field(tc.data_ptr(), tc.stride(0), tc.stride(1) if nsd == 3 else 0,
                         tc.stride(nsd - 1) if nsd >= 2 else 0)
        stream = torch.cuda.current_stream(tc.device).cuda_stream
        with _on_device(tc.device):
            rc = L.lib().dn_fem_gp_eval_general_f32(C.byref(fld), nsd, B, n3[2], n3[1], n3[0], nb, ng,
                                                    fac.ctypes.data_as(C.POINTER(C.c_float)), _ptr(out), C.c_void_p(stream))
        L.check(rc, "dn_fem_gp_eval_general_f32")
        ctx.meta = (nsd, nb, ng, fac, n3, B, sp)
        ctx.t_shape = tuple(t.shape)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        nsd, nb, ng, fac, n3, B, sp = ctx.meta
        gout = gout.contiguous()
        gin = _new_out((B,) + sp, gout.device)
        stream = torch.cuda.current_stream(gout.device).cuda_stream
        with _on_device(gout.device):
            rc = L.lib().dn_fem_gp_eval_general_adj_f32(_ptr(gout), nsd, B, n3[2], n3[1], n3[0], nb, ng,
                                                        fac.ctypes.data_as(C.POINTER(C.c_float)), _ptr(gin), C.c_void_p(stream))
        L.check(rc, "dn_fem_gp_eval_general_adj_f32")
        return gin.reshape(ctx.t_shape), None, None, None, None


def gp_eval_general(t: torch.Tensor, nsd: int, nbf_1d: int, ngp_1d: int, factors) -> torch.Tensor:
    """``factors[d][g][b]``, d = 0 (x) .. nsd-1: the 1-D basis value (or derivative * 2/h) of local node b at
    Gauss point g.  Returns (B, ngp_1d^nsd, elements...)."""
    return GaussPointEvalGeneralFunction.apply(t, nsd, nbf_1d, ngp_1d, factors)


# ------------------------------------------------------------------------------ public functional API
def fem_energy(geom: Geometry, u, nu=None, f=None, f_gp=None, dirichlet: Sequence = (),
               nu_zero_mask=None, c_k=1.0, c_f=1.0, scale=1.0, reduction="mean", z_own=None,
               mean_count=0.0) -> torch.Tensor:
    """Fused Poisson energy loss (SURVEY.md App. A.4), differentiable w.r.t. u, nu, f, f_gp and the tensor
    Dirichlet values (the last three not with ``z_own``).  ``reduction``: "mean", "sum" or "none" (a (B,) loss,
    loss[b] = scale / elements * the sum over sample b, so that its mean is the "mean" loss)."""
    _consts(c_k, c_f, scale, reduction, 0, z_own, mean_count)     # refuses a bad reduction before any launch
    dirichlet = tuple(dirichlet)
    return FEMEnergyFunction.apply(u, nu, geom, f, f_gp, dirichlet, nu_zero_mask, c_k, c_f, scale, reduction,
                                   z_own, mean_count, *(v for _, v in dirichlet if torch.is_tensor(v)))


def fem_energy_and_grad(geom: Geometry, u, **kw):
    """(loss, dloss/du) from ONE launch, outside autograd (LBFGS closures, benchmarks)."""
    loss, grad, _ = energy_raw(geom, u, **kw)
    return loss, grad


def fem_residual(geom: Geometry, u, nu=None, f=None, dirichlet: Sequence = (), jac=1.0,
                 reduction="sum") -> torch.Tensor:
    """sum(R^2) of the assembled residual, differentiable w.r.t. u, nu, f and the tensor Dirichlet values.
    ``reduction="none"``: a (B,) loss, the sum of R^2 over each sample."""
    if reduction not in ("sum", "none"):
        raise L.DiffNetFEMError("residual reduction must be 'sum' or 'none'")
    dirichlet = tuple(dirichlet)
    return FEMResidualFunction.apply(u, geom, nu, f, dirichlet, jac, reduction,
                                     *(v for _, v in dirichlet if torch.is_tensor(v)))


def gp_eval(geom: Geometry, t: torch.Tensor, which: str = "N") -> torch.Tensor:
    return GaussPointEvalFunction.apply(t, geom, _WHICH[which])


def gp_eval_multi(geom: Geometry, t: torch.Tensor, which: Sequence[str] = ("N", "dx", "dy")):
    """(gauss_pt_evaluation(t), ..._der_x(t), ...) for the listed tables from ONE call (and one backward pass over all cotangents)."""
    whichs = tuple(_WHICH[w] for w in which)
    if not 1 <= len(whichs) <= 4 or (geom.nsd == 2 and 3 in whichs):
        raise ValueError(f"which={which!r}: 1..4 tables out of N, dx, dy" + (", dz" if geom.nsd == 3 else ""))
    return GaussPointEvalMultiFunction.apply(t, geom, whichs)
