"""DiffNetFEM / DiffNet2DFEM / DiffNet3DFEM on the fused sm_100a kernels.

Public surface of reference ``DiffNet/DiffNetFEM.py`` kept: constructor ``(network, **kwargs)``,
attributes ``ngp_1d, ngp_total, nbf_1d, nbf_total, gpx_1d, gpw_1d, gpw, nelem{,X,Y,Z},
h{,x,y,z}, N_gp, dN_x_gp, dN_y_gp, dN_z_gp, Nvalues, dN_{x,y,z}_values, xx, yy, zz,
xgp, ygp, zgp`` and methods ``gauss_pt_evaluation{,_der_x,_der_y,_der_z}``, ``calc_l2_err``.
New: ``energy_loss`` / ``residual_loss`` -- the whole reference ``loss()`` body as ONE kernel:

    def loss(self, u, inputs_tensor, forcing_tensor):             # 0_base.py:31-56 in 3 lines
        nu, bc1, bc2 = inputs_tensor[:, 0:1], inputs_tensor[:, 1:2], inputs_tensor[:, 2:3]
        return self.energy_loss(u, nu=nu, f=forcing_tensor, dirichlet=[(bc1, 1.0), (bc2, 0.0)],
                                scale=0.5 * (0.5 * self.h) ** 2)

The tables are host-side metadata (numpy, float64 -> float32 like the reference); all field
arithmetic happens in libdiffnet_fem.so.  CPU tensors are rejected: there is no fallback.
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

from . import ops
from .base import PDE

# 1-D Gauss rules, constants as in DiffNetFEM.py:128-141 (kept truncated where the reference
# truncates them: the kernels integrate with the moments of exactly these rules)
_RULES = {
    1: ([0.0], [2.0]),
    2: ([-0.5773502691896258, 0.5773502691896258], [1.0, 1.0]),
    3: ([-0.774596669, 0.0, 0.774596669], [5.0 / 9.0, 8.0 / 9.0, 5.0 / 9.0]),
    4: ([-0.861136, -0.339981, 0.339981, 0.861136], [0.347855, 0.652145, 0.652145, 0.347855]),
}


class DiffNetFEM(PDE):
    def __init__(self, network, **kwargs):
        super().__init__(network, **kwargs)
        self.fem_basis_deg = kwargs.get("fem_basis_deg", 1)
        if self.fem_basis_deg in (2, 3):
            self._init_high_order(kwargs)
            return
        if self.fem_basis_deg != 1:
            raise NotImplementedError("fem_basis_deg must be 1, 2 or 3 (DiffNetFEM.py:53-126)")
        self.ngp_1d = max(int(kwargs.get("ngp_1d", 2)), 2)       # DiffNetFEM.py:29-38
        self.ngp_total = self.ngp_1d ** self.nsd
        self.gpx_1d, self.gpw_1d = self.gauss_guadrature_scheme(self.ngp_1d)
        self.nbf_1d = 2
        self.nbf_total = self.nbf_1d ** self.nsd

        self.nelemX = int(self.domain_sizeX - 1)
        self.nelemY = int(self.domain_sizeY - 1)
        self.nelem = int(self.domain_size - 1)
        self.hx = self.domain_lengthX / self.nelemX
        self.hy = self.domain_lengthY / self.nelemY
        self.h = self.domain_length / self.nelem
        if self.nsd == 3:
            self.nelemZ = int(self.domain_sizeZ - 1)
            self.hz = self.domain_lengthZ / self.nelemZ

        self.bf_1d = lambda x: np.array([0.5 * (1.0 - x), 0.5 * (1.0 + x)])
        self.bf_1d_der = lambda x: np.array([-0.5, 0.5])
        self.bf_1d_der2 = lambda x: np.array([0.0, 0.0])

        self.geometry = ops.Geometry(
            nsd=self.nsd, nx=int(self.domain_sizeX), ny=int(self.domain_sizeY),
            nz=int(self.domain_sizeZ) if self.nsd == 3 else 1,
            hx=float(self.hx), hy=float(self.hy), hz=float(self.hz) if self.nsd == 3 else 0.0,
            ngp_1d=self.ngp_1d)
        self._build_tables()

    # ---------------------------------------------------------------- quadratic / cubic bases
    def _init_high_order(self, kwargs):
        """fem_basis_deg 2 / 3 (DiffNetFEM.py:66-126; upstream these crash on numpy >= 1.24 because of
        ``dtype=np.float`` -- the polynomials are restated here).  Elements span ``deg`` node intervals,
        ``(size - 1) % deg == 0``.  The Gauss-point evaluation family runs on the general-basis CUDA ops
        (``dn_fem_gp_eval_general_f32``); the FUSED energy / residual kernels are Q1 only."""
        deg = self.fem_basis_deg
        self.ngp_1d = max(int(kwargs.get("ngp_1d", 2)), 3)        # DiffNetFEM.py:27-38: both need >= 3 points
        self.ngp_total = self.ngp_1d ** self.nsd
        self.gpx_1d, self.gpw_1d = self.gauss_guadrature_scheme(self.ngp_1d)
        self.nbf_1d = deg + 1
        self.nbf_total = self.nbf_1d ** self.nsd
        sizes = [self.domain_sizeX, self.domain_sizeY] + ([self.domain_sizeZ] if self.nsd == 3 else [])
        if any((int(n) - 1) % deg for n in sizes):
            raise AssertionError(f"(domain_size - 1) % {deg} != 0")   # the reference asserts the same (:67, :101)
        self.nelemX = int((self.domain_sizeX - 1) / deg)
        self.nelemY = int((self.domain_sizeY - 1) / deg)
        self.nelem = int((self.domain_size - 1) / deg)
        self.hx = self.domain_lengthX / self.nelemX
        self.hy = self.domain_lengthY / self.nelemY
        self.h = self.domain_length / self.nelem
        if self.nsd == 3:
            self.nelemZ = int((self.domain_sizeZ - 1) / deg)
            self.hz = self.domain_lengthZ / self.nelemZ
        if deg == 2:
            self.bf_1d = lambda x: np.array([0.5 * x * (x - 1.0), 1.0 - x ** 2, 0.5 * x * (x + 1.0)], dtype=float)
            self.bf_1d_der = lambda x: np.array([0.5 * (2.0 * x - 1.0), -2.0 * x, 0.5 * (2.0 * x + 1.0)], dtype=float)
            self.bf_1d_der2 = lambda x: np.array([1.0, -2.0, 1.0], dtype=float)
        else:
            self.bf_1d = lambda x: np.array([
                (-9.0 / 16.0) * (x ** 3 - x ** 2 - (1.0 / 9.0) * x + (1.0 / 9.0)),
                (27.0 / 16.0) * (x ** 3 - (1.0 / 3.0) * x ** 2 - x + (1.0 / 3.0)),
                (-27.0 / 16.0) * (x ** 3 + (1.0 / 3.0) * x ** 2 - x - (1.0 / 3.0)),
                (9.0 / 16.0) * (x ** 3 + x ** 2 - (1.0 / 9.0) * x - (1.0 / 9.0))], dtype=float)
            self.bf_1d_der = lambda x: np.array([
                (-9.0 / 16.0) * (3 * x ** 2 - 2 * x - (1.0 / 9.0)),
                (27.0 / 16.0) * (3 * x ** 2 - (2.0 / 3.0) * x - 1),
                (-27.0 / 16.0) * (3 * x ** 2 + (2.0 / 3.0) * x - 1),
                (9.0 / 16.0) * (3 * x ** 2 + 2 * x - (1.0 / 9.0))], dtype=float)
            self.bf_1d_der2 = lambda x: np.array([
                (-9.0 / 16.0) * (6.0 * x - 2.0), (27.0 / 16.0) * (6.0 * x - (2.0 / 3.0)),
                (-27.0 / 16.0) * (6.0 * x + (2.0 / 3.0)), (9.0 / 16.0) * (6.0 * x + 2.0)], dtype=float)
        self.geometry = None                                       # Q1 kernels do not apply
        nsd, ng, nb = self.nsd, self.ngp_1d, self.nbf_1d
        val = np.stack([self.bf_1d(x) for x in self.gpx_1d])       # [gp][bf]
        der = np.stack([self.bf_1d_der(x) for x in self.gpx_1d])
        scl = [2.0 / self.hx, 2.0 / self.hy] + ([2.0 / self.hz] if nsd == 3 else [])
        axes = "xyz"[:nsd]
        names = ["N_gp"] + [f"dN_{a}_gp" for a in axes]
        vnames = ["Nvalues"] + [f"dN_{a}_values" for a in axes]
        lists = {n: nn.ParameterList() for n in names}
        tail = (1,) * nsd
        values = {n: torch.ones((1, self.nbf_total, self.ngp_total) + tail) for n in vnames}
        self.gpw = torch.zeros(self.ngp_total)
        for G, gp in enumerate(np.ndindex(*(ng,) * nsd)):           # gp = ([kg,] jg, ig)
            gp_xyz = gp[::-1]
            self.gpw[G] = float(np.prod([self.gpw_1d[g] for g in gp_xyz]))
            for t, (name, vname) in enumerate(zip(names, vnames)):
                fac = [der[gp_xyz[d]] if t == d + 1 else val[gp_xyz[d]] for d in range(nsd)]
                tab = fac[0]
                for d in range(1, nsd):
                    tab = fac[d].reshape((nb,) + (1,) * d) * tab
                if t > 0:
                    tab = tab * scl[t - 1]
                t32 = torch.from_numpy(np.ascontiguousarray(tab)).to(torch.float32)
                lists[name].append(nn.Parameter(t32[None, None].clone(), requires_grad=False))
                values[vname][0, :, G] = t32.reshape((self.nbf_total,) + tail)
        for n in names:
            setattr(self, n, lists[n])
        for n in vnames:
            setattr(self, n, values[n])
        if nsd == 2:
            self.gpw_surf = torch.tensor([float(w) for w in self.gpw_1d], dtype=torch.float32)
            self.N_gp_surf = nn.ParameterList([nn.Parameter(torch.tensor(val[g], dtype=torch.float32)[None, None].clone(),
                                                            requires_grad=False) for g in range(ng)])
        # 1-D factor tables of the general-basis ops: [which][d][g][b], which = 0: N, 1 + d: d/dx_d
        self._factors = {}
        for w, key in enumerate(["N"] + ["d" + a for a in axes]):
            self._factors[key] = np.stack([(der * scl[d]) if w == d + 1 else val for d in range(nsd)]).astype(np.float32)
        self._surf_factors = val.astype(np.float32)[None]
        x = np.linspace(0, self.domain_lengthX, self.domain_sizeX)
        y = np.linspace(0, self.domain_lengthY, self.domain_sizeY)
        if nsd == 2:
            xx, yy = np.meshgrid(x, y)
            grids = {"xx": xx, "yy": yy}
        else:
            z = np.linspace(0, self.domain_lengthZ, self.domain_sizeZ)
            zz, yy, xx = np.meshgrid(z, y, x, indexing="ij")
            grids = {"xx": xx, "yy": yy, "zz": zz}
        for k, v in grids.items():
            setattr(self, k, torch.FloatTensor(np.ascontiguousarray(v)))
        # Gauss-point coordinates: the Lagrange basis reproduces the (linear) coordinate exactly
        nels = [self.nelemX, self.nelemY] + ([self.nelemZ] if nsd == 3 else [])
        lens = [self.domain_lengthX, self.domain_lengthY] + ([self.domain_lengthZ] if nsd == 3 else [])
        elems = tuple(nels[::-1])
        for a, name in enumerate(("xgp", "ygp", "zgp")[:nsd]):
            hh = lens[a] / nels[a]
            lo = hh * np.arange(nels[a])
            per_gp = np.stack([lo + 0.5 * (1.0 + float(self.gpx_1d[g])) * hh for g in range(ng)])    # [g][elem]
            out = np.zeros((1, self.ngp_total) + elems)
            for G, gp in enumerate(np.ndindex(*(ng,) * nsd)):
                shape = [1] * nsd
                shape[nsd - 1 - a] = -1
                out[0, G] = per_gp[gp[::-1][a]].reshape(shape)
            setattr(self, name, torch.FloatTensor(out))

    def _general(self, tensor, key):
        return ops.gp_eval_general(tensor, self.nsd, self.nbf_1d, self.ngp_1d, self._factors[key])

    # name kept (typo included) for drop-in compatibility: DiffNetFEM.py:128
    def gauss_guadrature_scheme(self, ngp_1d):
        x, w = _RULES[ngp_1d]
        return np.array(x), np.array(w)

    # ---------------------------------------------------------------- tables (host metadata)
    def _build_tables(self):
        nsd, ng = self.nsd, self.ngp_1d
        val = np.stack([self.bf_1d(x) for x in self.gpx_1d])        # [gp][bf]
        der = np.stack([self.bf_1d_der(x) for x in self.gpx_1d])
        scl = [2.0 / self.hx, 2.0 / self.hy] + ([2.0 / self.hz] if nsd == 3 else [])
        axes = "xyz"[:nsd]
        names = ["N_gp"] + [f"dN_{a}_gp" for a in axes]
        vnames = ["Nvalues"] + [f"dN_{a}_values" for a in axes]
        lists = {n: nn.ParameterList() for n in names}
        tail = (1,) * nsd
        values = {n: torch.ones((1, self.nbf_total, self.ngp_total) + tail) for n in vnames}
        self.gpw = torch.zeros(self.ngp_total)
        # gp index tuples in (z,) y, x order -> G = ((kg)*ng + jg)*ng + ig
        for G, gp in enumerate(np.ndindex(*(ng,) * nsd)):
            gp_xyz = gp[::-1]                                         # (ig, jg[, kg])
            self.gpw[G] = float(np.prod([self.gpw_1d[g] for g in gp_xyz]))
            for t, (name, vname) in enumerate(zip(names, vnames)):
                # 1-D factor per direction d: derivative for the differentiated one
                fac = [der[gp_xyz[d]] if t == d + 1 else val[gp_xyz[d]] for d in range(nsd)]
                tab = fac[0]                                          # x, innermost
                for d in range(1, nsd):
                    tab = fac[d].reshape((2,) + (1,) * d) * tab       # (.. y, x): same product order as ref
                if t > 0:
                    tab = tab * scl[t - 1]
                t32 = torch.from_numpy(np.ascontiguousarray(tab)).to(torch.float32)
                lists[name].append(nn.Parameter(t32[None, None].clone(), requires_grad=False))
                values[vname][0, :, G] = t32.reshape((self.nbf_total,) + tail)
        for n in names:
            setattr(self, n, lists[n])          # registered: appear in state_dict like the reference
        for n in vnames:
            setattr(self, n, values[n])
        # The reference also registers the second-derivative stencils (identically zero for Q1) and, in
        # 2-D, the 1-D surface stencils (DiffNetFEM.py:187-195,244-269, 391-403): they are part of its
        # state_dict, so a checkpoint written by the reference loads here with strict=True and vice versa.
        # d2N_{x,y,z} are identically zero for Q1; the mixed ones are not.  In 3-D the reference writes
        # them with TRANSPOSED local indices [ibf, jbf, kbf] (DiffNetFEM.py:430-435, SURVEY App. B): kept,
        # the point is an identical state_dict.
        D = [-0.5, 0.5]
        gx = [float(x) for x in self.gpx_1d]
        bf = lambda x, i: float(self.bf_1d(x)[i])       # noqa: E731
        mixed = {}
        zero = lambda: [torch.zeros((2,) * nsd) for _ in range(self.ngp_total)]   # noqa: E731
        if nsd == 2:
            second = ["d2N_x_gp", "d2N_y_gp", "d2N_xy_gp"]
            mixed["d2N_xy_gp"] = zero()
            for G in range(self.ngp_total):
                for jb in range(2):
                    for ib in range(2):
                        mixed["d2N_xy_gp"][G][jb, ib] = D[ib] * D[jb] * (2 / self.hx) * (2 / self.hy)
        else:
            second = ["d2N_x_gp", "d2N_y_gp", "d2N_z_gp", "d2N_xy_gp", "d2N_yz_gp", "d2N_zx_gp"]
            for n in ("d2N_xy_gp", "d2N_yz_gp", "d2N_zx_gp"):
                mixed[n] = zero()
            for G, (kg, jg, ig) in enumerate(np.ndindex(ng, ng, ng)):
                for kb in range(2):
                    for jb in range(2):
                        for ib in range(2):
                            mixed["d2N_xy_gp"][G][ib, jb, kb] = D[ib] * D[jb] * bf(gx[kg], kb) * (2 / self.hx) * (2 / self.hy)
                            mixed["d2N_yz_gp"][G][ib, jb, kb] = bf(gx[ig], ib) * D[jb] * D[kb] * (2 / self.hy) * (2 / self.hz)
                            mixed["d2N_zx_gp"][G][ib, jb, kb] = D[ib] * bf(gx[jg], jb) * D[kb] * (2 / self.hz) * (2 / self.hx)
        for n in second:
            tabs = mixed.get(n) or zero()
            setattr(self, n, nn.ParameterList([nn.Parameter(t[None, None].clone(), requires_grad=False) for t in tabs]))
        if nsd == 2:
            self.gpw_surf = torch.tensor([float(w) for w in self.gpw_1d], dtype=torch.float32)
            surf = {"N_gp_surf": [], "dN_x_gp_surf": [], "dN_y_gp_surf": []}
            self.Nvalues_surf = torch.ones((1, self.nbf_1d, ng, 1))
            self.dN_x_values_surf = torch.ones((1, self.nbf_1d, ng, 1))
            self.dN_y_values_surf = torch.ones((1, self.nbf_1d, ng, 1))
            for igp in range(ng):
                row = {"N_gp_surf": torch.tensor(val[igp], dtype=torch.float32),
                       "dN_x_gp_surf": torch.tensor(der[igp] * (2.0 / self.hx), dtype=torch.float32),
                       "dN_y_gp_surf": torch.tensor(der[igp] * (2.0 / self.hy), dtype=torch.float32)}
                self.Nvalues_surf[0, :, igp, 0] = row["N_gp_surf"]
                self.dN_x_values_surf[0, :, igp, 0] = row["dN_x_gp_surf"]
                self.dN_y_values_surf[0, :, igp, 0] = row["dN_y_gp_surf"]
                for k, v in row.items():
                    surf[k].append(nn.Parameter(v[None, None].clone(), requires_grad=False))
            for k, v in surf.items():
                setattr(self, k, nn.ParameterList(v))

        x = np.linspace(0, self.domain_lengthX, self.domain_sizeX)
        y = np.linspace(0, self.domain_lengthY, self.domain_sizeY)
        if nsd == 2:
            xx, yy = np.meshgrid(x, y)
            grids = {"xx": xx, "yy": yy}
        else:
            z = np.linspace(0, self.domain_lengthZ, self.domain_sizeZ)
            zz, yy, xx = np.meshgrid(z, y, x, indexing="ij")          # (P, N, M): cuboid_mesh.py:8-25
            grids = {"xx": xx, "yy": yy, "zz": zz}
        for k, v in grids.items():
            setattr(self, k, torch.FloatTensor(np.ascontiguousarray(v)))
        # Gauss-point coordinates (DiffNetFEM.py:229-235, 455-465): closed form of interpolating
        # a linear coordinate -- host metadata, evaluated once in float64
        for a, (name, n1, L1) in enumerate(zip(("xgp", "ygp", "zgp")[:nsd],
                                               self.geometry.spatial[::-1],
                                               (self.domain_lengthX, self.domain_lengthY,
                                                getattr(self, "domain_lengthZ", 1.0)))):
            nodes = np.linspace(0, L1, n1)
            lo, hi = nodes[:-1], nodes[1:]
            per_gp = np.stack([val[g][0] * lo + val[g][1] * hi for g in range(ng)])   # [g][elem]
            out = np.zeros((1, self.ngp_total) + self.geometry.elems)
            for G, gp in enumerate(np.ndindex(*(ng,) * nsd)):
                g1 = gp[::-1][a]
                shape = [1] * nsd
                shape[nsd - 1 - a] = -1
                out[0, G] = per_gp[g1].reshape(shape)
            setattr(self, name, torch.FloatTensor(out))

    # ---------------------------------------------------------------- reference methods
    def gauss_pt_evaluation(self, tensor, stride=1):
        if self.fem_basis_deg != 1:
            return self._general(tensor, "N")
        return ops.gp_eval(self.geometry, tensor, "N")

    def gauss_pt_evaluation_der_x(self, tensor, stride=1):
        if self.fem_basis_deg != 1:
            return self._general(tensor, "dx")
        return ops.gp_eval(self.geometry, tensor, "dx")

    def gauss_pt_evaluation_der_y(self, tensor, stride=1):
        if self.fem_basis_deg != 1:
            return self._general(tensor, "dy")
        return ops.gp_eval(self.geometry, tensor, "dy")

    def gauss_pt_evaluation_der_z(self, tensor, stride=1):
        if self.nsd != 3:
            raise ValueError("gauss_pt_evaluation_der_z needs nsd == 3")
        if self.fem_basis_deg != 1:
            return self._general(tensor, "dz")
        return ops.gp_eval(self.geometry, tensor, "dz")

    def gauss_pt_evaluation_surf(self, tensor, stride=1):
        """Boundary-line evaluation of a 2-D mesh (DiffNetFEM.py:146-147): ``tensor`` (B, 1, n) nodal values along
        one edge -> (B, ngp_1d, n_elements) values at the edge's Gauss points."""
        if self.nsd != 2:
            raise ValueError("gauss_pt_evaluation_surf is defined for nsd == 2 (the reference builds N_gp_surf in 2-D only)")
        if self.fem_basis_deg == 1:
            fac = np.stack([self.bf_1d(x) for x in self.gpx_1d]).astype(np.float32)[None]
        else:
            fac = self._surf_factors
        return ops.gp_eval_general(tensor, 1, self.nbf_1d, self.ngp_1d, fac)

    def gauss_pt_evaluation_all(self, tensor, which=None):
        """(gauss_pt_evaluation(t), _der_x(t), _der_y(t)[, _der_z(t)]) from ONE call (new; the
        reference makes one conv sweep per table, DiffNetFEM.py:143-156)."""
        which = which or (("N", "dx", "dy") + (("dz",) if self.nsd == 3 else ()))
        if self.fem_basis_deg != 1:
            return tuple(self._general(tensor, w) for w in which)
        return ops.gp_eval_multi(self.geometry, tensor, which)

    # ---------------------------------------------------------------- fused ops (new)
    def energy_loss(self, u, nu=None, f=None, f_gp=None, dirichlet=(), nu_zero_mask=None,
                    c_k=1.0, c_f=1.0, scale=1.0, reduction="mean"):
        """scale * sum_g gpw_g (c_k nu_g |grad u|_g^2 - c_f u_g f_g), mean/sum over batch x elements,
        with u = where(mask > 0.5, value, u) applied for each (mask, value) of `dirichlet` in order.
        ``reduction="none"``: one loss per sample, a (B,) tensor whose mean is the "mean" loss."""
        self._q1_only("energy_loss")
        return ops.fem_energy(self.geometry, u, nu=nu, f=f, f_gp=f_gp, dirichlet=dirichlet,
                              nu_zero_mask=nu_zero_mask, c_k=c_k, c_f=c_f, scale=scale,
                              reduction=reduction)

    def energy_loss_and_grad(self, u, **kw):
        """(loss, dloss/du) in one launch, outside autograd.  With ``reduction="none"`` loss is (B,) and dloss/du the
        gradient of loss.sum(): each sample's own gradient."""
        self._q1_only("energy_loss_and_grad")
        return ops.fem_energy_and_grad(self.geometry, u, **kw)

    def prepare_energy(self, u, **kw):
        """Bind a fused energy call to fixed tensors (see ops.PreparedEnergy): ``call = fem.prepare_energy(u,
        nu=..., ...)``, then ``loss, grad = call()`` costs one C call per evaluation."""
        self._q1_only("prepare_energy")
        return ops.PreparedEnergy(self.geometry, u, **kw)

    def residual_loss(self, u, nu=None, f=None, dirichlet=(), jac=1.0, reduction="sum"):
        """sum(R^2) of the assembled, Dirichlet-zeroed Galerkin residual (12_klsum.py:80-132); ``reduction="none"``:
        one sum per sample, a (B,) tensor."""
        self._q1_only("residual_loss")
        return ops.fem_residual(self.geometry, u, nu=nu, f=f, dirichlet=dirichlet, jac=jac, reduction=reduction)

    def _q1_only(self, what):
        if self.fem_basis_deg != 1:
            raise NotImplementedError(
                f"{what}: the fused kernels are Q1 (fem_basis_deg=1); with degree {self.fem_basis_deg} write the loss body "
                "on gauss_pt_evaluation* (general-basis CUDA ops), as the reference's scripts do")

    def calc_l2_err(self, u_sol):
        """||u_sol - u_exact||_L2 by Gauss quadrature (DiffNetFEM.py:348-379, 560-591); returns
        (eL2, uL2, u_exL2) instead of printing.  Needs ``self.exact_solution(xgp, ygp[, zgp])``."""
        u_gp = self.gauss_pt_evaluation(u_sol)
        coords = [self.xgp, self.ygp] + ([self.zgp] if self.nsd == 3 else [])
        u_ex_gp = self.exact_solution(*coords).to(u_gp)
        jac = float(np.prod([0.5 * h for h in (self.hx, self.hy) + ((self.hz,) if self.nsd == 3 else ())]))
        JxW = (self.gpw.to(u_gp) * jac).reshape((1, -1) + (1,) * self.nsd)
        e = torch.sqrt(torch.sum((u_gp - u_ex_gp) ** 2 * JxW))
        return e, torch.sqrt(torch.sum(u_gp ** 2 * JxW)), torch.sqrt(torch.sum(u_ex_gp ** 2 * JxW))


class DiffNet2DFEM(DiffNetFEM):
    def __init__(self, network, **kwargs):
        super().__init__(network, **kwargs)
        assert self.nsd == 2


class DiffNet3DFEM(DiffNetFEM):
    def __init__(self, network, **kwargs):
        kwargs.setdefault("nsd", 3)
        super().__init__(network, **kwargs)
        assert self.nsd == 3
