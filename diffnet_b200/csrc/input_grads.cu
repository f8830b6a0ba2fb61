// input_grads.cu -- see input_grads.cuh.
//
// The fused losses differentiate with respect to u (and nu of the energy form) inside their own launch.  The other
// inputs a user may optimise -- the source f, the forcing at the Gauss points f_gp, the Dirichlet value fields, and
// nu of the residual form -- get their gradients here, in ONE launch per backward.  Every such gradient is a nodal
// operator applied to one field X of the forward pass (X = u' for the energy, X = R for the residual):
//
//   slot 0   cM * M X                                    energy dL/df, residual dL/df       (mass stencil)
//   slot 1   cK * K(nu) X + cS * (M f | sum_g w N f_gp)  energy g-hat, residual 2 jac K(nu) R  (-> value fields)
//   slot 2   cN * sum_g w_g N grad u' . grad R           residual dL/dnu
//   per element and Gauss point G:  cG * w_G X_G         energy dL/df_gp
//
// M = the separable Q1 mass (1-D element mass (W1/4)[[1+t, 1-t], [1-t, 1+t]] per direction, closed form); the other
// terms are Gauss sums, evaluated by sum factorisation (z-, y-, x-stages forward, x-, y-, z-stages back to the
// corners).  A value field k receives slot 1 at the nodes where mask k is the LAST firing mask, 0 elsewhere.
//
// Decomposition and gather (no atomics, bit-reproducible):
//   2-D  a warp covers 31 node columns plus one provider lane on its left and MARCHES in y: each node row is loaded
//        once, the x-neighbour's value comes from the next lane by one shuffle, element rows contribute to the node
//        rows above and below through a register carry, the left element's share arrives by one shuffle (the
//        layout of k_gp_eval_adj, gp_eval.cu).
//   3-D  a CTA is LXW lanes (x) by kIg3Rows rows (y) and marches UP in z; a thread owns one element column and one
//        node column, shares meet through a register carry in z and one double-buffered shared-memory exchange per
//        layer (the layout of k_gp_eval_adj3).  Later tiles overlap their predecessor by one provider lane / row.
// A gradient of a field broadcast over the batch (stride_b = 0) is one (1, ...) field: the launch then has no batch
// dimension, every thread walks b = 0 .. B-1 in order and adds into the node it owns (fixed order, no atomics).
#include <algorithm>

#include "input_grads.cuh"

namespace dn {

namespace {

struct Flags {
  bool s0, s1, s2;   // slots wanted (grad_f; any value field; grad_nu)
  bool fo;           // grad_fgp wanted (energy)
  bool srcf, srcg;   // slot 1 carries the source term: nodal f / f at the Gauss points (energy)
  bool dir;          // u' / last firing mask needed at the nodes
};

struct NV {
  float X, NU, F, UP;
  int last;
};

__device__ __forceinline__ float at(const Field& F, int b, int z, int y, int x) {
  return __ldg(F.p + (long long)b * F.sb + (long long)z * F.sz + (long long)y * F.sy + x);
}

// The raw loads of one node, issued one row ahead of their use by the 2-D march (its loads then overlap the
// arithmetic of the element row in flight), and the node values derived from them.
struct Raw {
  float u, R, nu, nz, f;
  float m[DN_MAX_MASKS], vf[DN_MAX_MASKS];
  bool ok;
};

template <int MODE>
__device__ __forceinline__ void load_raw(const InGrad& q, const Flags& fl, int b, int z, int y, int x, bool ok,
                                         Raw& r) {
  r.ok = ok;
  r.u = (ok && fl.dir && (MODE == 0 || fl.s2)) ? at(q.u, b, z, y, x) : 0.f;
#pragma unroll
  for (int k = 0; k < DN_MAX_MASKS; ++k) {
    const bool mk = ok && fl.dir && k < q.nmasks;
    r.m[k] = mk ? at(q.mk[k].m, b, z, y, x) : 0.f;
    r.vf[k] = (mk && q.mk[k].vf.p) ? at(q.mk[k].vf, b, z, y, x) : 0.f;
  }
  r.R = (ok && MODE == 1) ? at(q.R, b, z, y, x) : 0.f;
  r.nu = (ok && fl.s1 && q.nu.p) ? at(q.nu, b, z, y, x) : 1.f;
  r.nz = (ok && fl.s1 && MODE == 0 && q.numask.p) ? at(q.numask, b, z, y, x) : 0.f;
  r.f = (ok && MODE == 0 && fl.srcf) ? at(q.f, b, z, y, x) : 0.f;
}

template <int MODE>
__device__ __forceinline__ void finish_node(const InGrad& q, const Raw& r, NV& o) {
  float up = r.u;
  int last = -1;
#pragma unroll
  for (int k = 0; k < DN_MAX_MASKS; ++k) {          // torch.where in list order: the last firing mask wins
    if (k < q.nmasks && r.m[k] > 0.5f) {
      up = q.mk[k].vf.p ? r.vf[k] : q.mk[k].v;
      last = k;
    }
  }
  o.UP = r.ok ? up : 0.f;
  o.last = r.ok ? last : -1;
  o.X = (MODE == 0) ? o.UP : r.R;
  o.NU = r.ok ? (r.nz > 0.5f ? 0.f : r.nu) : 0.f;
  o.F = r.f;
}

// Loads and derived values at once (the 3-D march holds four corners per plane: no registers for a plane ahead).
template <int MODE>
__device__ __forceinline__ void load_node(const InGrad& q, const Flags& fl, int b, int z, int y, int x, bool ok,
                                          NV& o) {
  o.X = o.NU = o.F = o.UP = 0.f;
  o.last = -1;
  if (!ok) return;
  if (fl.dir) {
    float up = (MODE == 0 || fl.s2) ? at(q.u, b, z, y, x) : 0.f;
    for (int k = 0; k < q.nmasks; ++k) {
      if (at(q.mk[k].m, b, z, y, x) > 0.5f) {
        up = q.mk[k].vf.p ? at(q.mk[k].vf, b, z, y, x) : q.mk[k].v;
        o.last = k;
      }
    }
    o.UP = up;
  }
  o.X = (MODE == 0) ? o.UP : at(q.R, b, z, y, x);
  if (fl.s1) {
    float nu = q.nu.p ? at(q.nu, b, z, y, x) : 1.f;
    if (MODE == 0 && q.numask.p && at(q.numask, b, z, y, x) > 0.5f) nu = 0.f;
    o.NU = nu;
    if (MODE == 0 && fl.srcf) o.F = at(q.f, b, z, y, x);
  }
}

// O += c * M V  (separable Q1 mass, closed form)
template <int NZ>
__device__ __forceinline__ void mass(const InGrad& q, const float (&V)[NZ][2][2], float c, float (&O)[NZ][2][2]) {
  const float a = q.ma, m = q.mc;
  float t[NZ][2][2];
#pragma unroll
  for (int kb = 0; kb < NZ; ++kb)
#pragma unroll
    for (int jb = 0; jb < 2; ++jb) {
      const float x0 = a * V[kb][jb][0] + m * V[kb][jb][1];
      const float x1 = m * V[kb][jb][0] + a * V[kb][jb][1];
      t[kb][jb][0] = x0;
      t[kb][jb][1] = x1;
    }
#pragma unroll
  for (int kb = 0; kb < NZ; ++kb)
#pragma unroll
    for (int ib = 0; ib < 2; ++ib) {
      const float y0 = a * t[kb][0][ib] + m * t[kb][1][ib];
      const float y1 = m * t[kb][0][ib] + a * t[kb][1][ib];
      t[kb][0][ib] = y0;
      t[kb][1][ib] = y1;
    }
#pragma unroll
  for (int jb = 0; jb < 2; ++jb)
#pragma unroll
    for (int ib = 0; ib < 2; ++ib) {
      if constexpr (NZ == 2) {
        O[0][jb][ib] += c * (a * t[0][jb][ib] + m * t[1][jb][ib]);
        O[1][jb][ib] += c * (m * t[0][jb][ib] + a * t[1][jb][ib]);
      } else {
        O[0][jb][ib] += c * t[0][jb][ib];
      }
    }
}

// One element: its shares Q[slot][kb][jb][ib] of the nodal outputs, and its grad_fgp values.
//   fg_in:  f_gp of this element at G = 0 (fl.srcg), fg_out: grad_fgp of this element at G = 0 (fl.fo), gs: the
//   stride between Gauss points; fg_acc: add to what fg_out holds (broadcast f_gp, not the first b).
template <int NZ, int NG, int MODE>
__device__ __forceinline__ void element(const InGrad& q, const Flags& fl, const float (&X)[NZ][2][2],
                                        const float (&NU)[NZ][2][2], const float (&F)[NZ][2][2],
                                        const float (&UP)[NZ][2][2], const float* fg_in, float* fg_out,
                                        bool fg_acc, long long gs, float (&Q)[3][NZ][2][2]) {
  if (fl.s0) mass<NZ>(q, X, q.cM, Q[0]);
  if (MODE == 0 && fl.s1 && fl.srcf) mass<NZ>(q, F, q.cS, Q[1]);
  const bool s2 = (MODE == 1) && fl.s2;
  if (!(fl.s1 || s2 || fl.fo)) return;
  const float dx = q.d[0], dy = q.d[1], dz = q.d[2];
#pragma unroll
  for (int kg = 0; kg < (NZ == 2 ? NG : 1); ++kg) {
    const float zw = (NZ == 2) ? q.w[kg] : 1.f;
    const float zn0 = (NZ == 2) ? 0.5f * (1.f - q.x[kg]) : 1.f, zn1 = 0.5f * (1.f + q.x[kg]);
    // z-stage: values and z-derivatives on the element's (jb, ib) edge lines at height kg
    float Xz[2][2], Xdz[2][2], Nz[2][2], Uz[2][2], Udz[2][2];
#pragma unroll
    for (int jb = 0; jb < 2; ++jb)
#pragma unroll
      for (int ib = 0; ib < 2; ++ib) {
        if constexpr (NZ == 2) {
          Xz[jb][ib] = zn0 * X[0][jb][ib] + zn1 * X[1][jb][ib];
          Xdz[jb][ib] = dz * (X[1][jb][ib] - X[0][jb][ib]);
          Nz[jb][ib] = zn0 * NU[0][jb][ib] + zn1 * NU[1][jb][ib];
          Uz[jb][ib] = zn0 * UP[0][jb][ib] + zn1 * UP[1][jb][ib];
          Udz[jb][ib] = dz * (UP[1][jb][ib] - UP[0][jb][ib]);
        } else {
          Xz[jb][ib] = X[0][jb][ib];
          Xdz[jb][ib] = 0.f;
          Nz[jb][ib] = NU[0][jb][ib];
          Uz[jb][ib] = UP[0][jb][ib];
          Udz[jb][ib] = 0.f;
        }
      }
    float A1[2][2] = {{0.f, 0.f}, {0.f, 0.f}}, Z1[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    float A2[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
    for (int jg = 0; jg < NG; ++jg) {
      const float yw = q.w[jg], yn0 = 0.5f * (1.f - q.x[jg]), yn1 = 0.5f * (1.f + q.x[jg]);
      float Xy[2], Xdy[2], Xyz[2], Ny[2], Uy[2], Udy[2], Uyz[2];
#pragma unroll
      for (int ib = 0; ib < 2; ++ib) {
        Xy[ib] = yn0 * Xz[0][ib] + yn1 * Xz[1][ib];
        Xdy[ib] = dy * (Xz[1][ib] - Xz[0][ib]);
        Xyz[ib] = yn0 * Xdz[0][ib] + yn1 * Xdz[1][ib];
        Ny[ib] = yn0 * Nz[0][ib] + yn1 * Nz[1][ib];
        Uy[ib] = yn0 * Uz[0][ib] + yn1 * Uz[1][ib];
        Udy[ib] = dy * (Uz[1][ib] - Uz[0][ib]);
        Uyz[ib] = yn0 * Udz[0][ib] + yn1 * Udz[1][ib];
      }
      // x-stage accumulators: value-weighted (P), d/dx-weighted (sqx), d/dy- (Y1) and d/dz-weighted (Zx)
      float P1[2] = {0.f, 0.f}, Y1[2] = {0.f, 0.f}, Zx[2] = {0.f, 0.f}, P2[2] = {0.f, 0.f};
      float sqx = 0.f;
#pragma unroll
      for (int ig = 0; ig < NG; ++ig) {
        const float xn0 = 0.5f * (1.f - q.x[ig]), xn1 = 0.5f * (1.f + q.x[ig]);
        const float W = zw * yw * q.w[ig];
        const long long G = (kg * NG + jg) * NG + ig;
        const float gx = dx * (Xy[1] - Xy[0]);
        const float gy = xn0 * Xdy[0] + xn1 * Xdy[1];
        const float gz = xn0 * Xyz[0] + xn1 * Xyz[1];
        if (fg_out) {
          float v = q.cG * W * (xn0 * Xy[0] + xn1 * Xy[1]);
          float* p = fg_out + G * gs;
          if (fg_acc) v += *p;
          *p = v;
        }
        if (fl.s1) {
          const float c = q.cK * W * (xn0 * Ny[0] + xn1 * Ny[1]);
          sqx += c * gx;
          Y1[0] += xn0 * (c * gy);
          Y1[1] += xn1 * (c * gy);
          if constexpr (NZ == 2) {
            Zx[0] += xn0 * (c * gz);
            Zx[1] += xn1 * (c * gz);
          }
          if (MODE == 0 && fl.srcg) {
            const float p = q.cS * W * __ldg(fg_in + G * gs);
            P1[0] += xn0 * p;
            P1[1] += xn1 * p;
          }
        }
        if (s2) {
          const float ux = dx * (Uy[1] - Uy[0]);
          const float uy = xn0 * Udy[0] + xn1 * Udy[1];
          float dot = ux * gx + uy * gy;
          if constexpr (NZ == 2) dot += (xn0 * Uyz[0] + xn1 * Uyz[1]) * gz;
          const float p = q.cN * W * dot;
          P2[0] += xn0 * p;
          P2[1] += xn1 * p;
        }
      }
      P1[0] -= dx * sqx;
      P1[1] += dx * sqx;
#pragma unroll
      for (int jb = 0; jb < 2; ++jb) {
        const float yn = jb ? yn1 : yn0, dd = jb ? dy : -dy;
#pragma unroll
        for (int ib = 0; ib < 2; ++ib) {
          A1[jb][ib] += yn * P1[ib] + dd * Y1[ib];
          if constexpr (NZ == 2) Z1[jb][ib] += yn * Zx[ib];
          A2[jb][ib] += yn * P2[ib];
        }
      }
    }
#pragma unroll
    for (int kb = 0; kb < NZ; ++kb) {
      const float zn = kb ? zn1 : zn0, ddz = kb ? dz : -dz;
#pragma unroll
      for (int jb = 0; jb < 2; ++jb)
#pragma unroll
        for (int ib = 0; ib < 2; ++ib) {
          if (fl.s1) Q[1][kb][jb][ib] += (NZ == 2) ? zn * A1[jb][ib] + ddz * Z1[jb][ib] : A1[jb][ib];
          if (s2) Q[2][kb][jb][ib] += zn * A2[jb][ib];
        }
    }
  }
}

__device__ __forceinline__ void put(float* o, bool bc, bool first, int b, long long per_b, long long i, float v) {
  float* p = o + (bc ? 0 : (long long)b * per_b) + i;
  if (bc && !first) v += *p;
  *p = v;
}

template <int MODE>
__device__ __forceinline__ void store_node(const InGrad& q, const Flags& fl, int b, bool first, long long nodes,
                                           long long i, const float (&n)[3], int last) {
  if (fl.s0) put(q.g_f, q.bc & 1u, first, b, nodes, i, n[0]);
  if (MODE == 1 && fl.s2) put(q.g_nu, q.bc & 4u, first, b, nodes, i, n[2]);
  if (fl.s1) {
#pragma unroll
    for (int k = 0; k < DN_MAX_MASKS; ++k)
      if (k < q.nmasks && q.g_v[k]) put(q.g_v[k], q.bc & (8u << k), first, b, nodes, i, last == k ? n[1] : 0.f);
  }
}

// ---- 2-D ------------------------------------------------------------------------------------------------------------
constexpr int kIgWarps = 4;

template <int NG, int MODE>
__global__ void __launch_bounds__(32 * kIgWarps, 4) k_input_grads_2d(InGrad q, Flags fl, int RY, int ball) {
  constexpr int NS = MODE ? 3 : 2;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nx = q.nx, ny = q.ny, nelx = nx - 1, nely = ny - 1;
  const int e = (int)blockIdx.x * 31 - 1 + lane;              // element column of this lane, node column it stores
  const bool ev = e >= 0 && e < nelx;
  const bool sv = lane >= 1 && e < nx;
  const bool c0 = e >= 0 && e < nx;
  const bool c1 = lane == 31 && e + 1 < nx;                   // lane 31 loads column e + 1 itself
  const int y0 = ((int)blockIdx.y * kIgWarps + warp) * RY;
  if (y0 >= ny) return;                                       // warp-uniform; the kernel has no CTA barrier
  const int y1 = min(ny, y0 + RY);
  const long long nodes = (long long)nx * ny, nel = (long long)nelx * nely, ngpe = (long long)NG * NG * nel;
  const int bb = ball ? 0 : (int)blockIdx.z, be = ball ? q.B : (int)blockIdx.z + 1;
  const unsigned full = 0xffffffffu;

  for (int b = bb; b < be; ++b) {
    const bool first = (b == bb);
    // raw loads of node row y: column e, and column e + 1 on lane 31 (the other lanes get it by a shuffle)
    auto issue_row = [&](int y, Raw& r0, Raw& r1) {
      const bool yv = y >= 0 && y < ny;
      load_raw<MODE>(q, fl, b, 0, y, e, yv && c0, r0);
      load_raw<MODE>(q, fl, b, 0, y, e + 1, yv && c1, r1);
    };
    auto finish_row = [&](const Raw& r0, const Raw& r1, NV& o0, NV& o1) {
      finish_node<MODE>(q, r0, o0);
      NV t;
      finish_node<MODE>(q, r1, t);
      o1.X = __shfl_down_sync(full, o0.X, 1);
      o1.NU = fl.s1 ? __shfl_down_sync(full, o0.NU, 1) : 0.f;
      o1.F = (MODE == 0 && fl.srcf) ? __shfl_down_sync(full, o0.F, 1) : 0.f;
      o1.UP = (MODE == 1 && fl.s2) ? __shfl_down_sync(full, o0.UP, 1) : 0.f;
      o1.last = -1;
      if (lane == 31) o1 = t;
    };
    Raw ra0, ra1, rb0, rb1;
    issue_row(y0 - 1, ra0, ra1);
    issue_row(y0, rb0, rb1);
    NV a0, a1;
    finish_row(ra0, ra1, a0, a1);
    float carry[3] = {0.f, 0.f, 0.f};
    for (int ej = y0 - 1; ej < y1; ++ej) {
      Raw rc0, rc1;
      issue_row(ej + 2, rc0, rc1);                          // in flight during element row ej
      NV b0, b1;
      finish_row(rb0, rb1, b0, b1);
      float Q[3][1][2][2] = {};
      if (ev && ej >= 0 && ej < nely) {
        const float X[1][2][2] = {{{a0.X, a1.X}, {b0.X, b1.X}}};
        const float NU[1][2][2] = {{{a0.NU, a1.NU}, {b0.NU, b1.NU}}};
        const float F[1][2][2] = {{{a0.F, a1.F}, {b0.F, b1.F}}};
        const float UP[1][2][2] = {{{a0.UP, a1.UP}, {b0.UP, b1.UP}}};
        const long long el = (long long)ej * nelx + e;
        const float* fg_in = fl.srcg ? q.fgp + (long long)b * q.fgp_sb + el : nullptr;
        // an element is formed twice where warps / chunks overlap: only its owner writes grad_fgp
        const bool own = lane >= 1 && ej >= y0;
        float* fg_out = (fl.fo && own) ? q.g_fgp + ((q.bc & 2u) ? 0 : (long long)b * ngpe) + el : nullptr;
        element<1, NG, MODE>(q, fl, X, NU, F, UP, fg_in, fg_out, (q.bc & 2u) && !first, nel, Q);
      }
      // node (ej, e): own share (jb 0, ib 0) + the left lane's (jb 0, ib 1) + the carry of element row ej - 1
      float n[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const float l0 = __shfl_up_sync(full, Q[s][0][0][1], 1);
        const float l1 = __shfl_up_sync(full, Q[s][0][1][1], 1);
        n[s] = carry[s] + Q[s][0][0][0] + l0;
        carry[s] = Q[s][0][1][0] + l1;
      }
      if (ej >= y0 && sv) store_node<MODE>(q, fl, b, first, nodes, (long long)ej * nx + e, n, a0.last);
      a0 = b0;
      a1 = b1;
      rb0 = rc0;
      rb1 = rc1;
    }
  }
}

// ---- 3-D ------------------------------------------------------------------------------------------------------------
constexpr int kIg3Rows = 8;
// lanes per tile row at most: 64 for the 2-point rule (512 threads fit 128 registers without spilling), 32 for the
// 3- and 4-point rules, whose Gauss loops need more registers
template <int NG>
constexpr int kIg3MaxLanes = NG == 2 ? 64 : 32;

template <int NG, int MODE>
__global__ void __launch_bounds__(kIg3MaxLanes<NG> * kIg3Rows) k_input_grads_3d(InGrad q, Flags fl, int LXW, int ZC,
                                                                            int ntx, int nty, int ball) {
  constexpr int NS = MODE ? 3 : 2;
  extern __shared__ float2 xch[];                       // [2 buffers][3 kinds][NS][kIg3Rows * LXW]
  const int lx = threadIdx.x % LXW, r = threadIdx.x / LXW;
  const int nx = q.nx, ny = q.ny, nz = q.nz, nelx = nx - 1, nely = ny - 1, nelz = nz - 1;
  int w_ = blockIdx.x;
  const int tx = w_ % ntx; w_ /= ntx;
  const int ty = w_ % nty; w_ /= nty;
  const int nzc = (nz + ZC - 1) / ZC;
  const int zc = w_ % nzc;
  const int bz = w_ / nzc;
  const int e = (tx == 0) ? lx : LXW + (tx - 1) * (LXW - 1) - 1 + lx;              // element column == node column
  const int ej = (ty == 0) ? r : kIg3Rows + (ty - 1) * (kIg3Rows - 1) - 1 + r;    // element row == node row
  const bool st = (tx == 0 || lx >= 1) && e < nx && (ty == 0 || r >= 1) && ej < ny;
  const bool ev = e < nelx && ej < nely;
  const bool hasL = lx > 0, hasU = r > 0;
  const int z0 = zc * ZC, z1 = min(nz, z0 + ZC);
  const int ek0 = max(z0 - 1, 0);
  const long long plane = (long long)nx * ny, nodes = plane * nz;
  const long long nel = (long long)nelx * nely * nelz, ngpe = (long long)NG * NG * NG * nel;
  const int kind = kIg3Rows * LXW;
  const int bb = ball ? 0 : bz, be = ball ? q.B : bz + 1;
  int buf = 0;

  for (int b = bb; b < be; ++b) {
    const bool first = (b == bb);
    NV c[2][2][2];                                      // [plane ek / ek + 1][jb][ib]
    auto load_plane = [&](int z, NV (&o)[2][2]) {
#pragma unroll
      for (int jb = 0; jb < 2; ++jb)
#pragma unroll
        for (int ib = 0; ib < 2; ++ib)
          load_node<MODE>(q, fl, b, z, ej + jb, e + ib, z < nz && ej + jb < ny && e + ib < nx, o[jb][ib]);
    };
    load_plane(ek0, c[0]);
    float carry[3] = {0.f, 0.f, 0.f};
    for (int ek = ek0; ek < z1; ++ek) {
      load_plane(ek + 1, c[1]);
      float Q[3][2][2][2] = {};
      if (ev && ek < nelz) {
        float X[2][2][2], NU[2][2][2], F[2][2][2], UP[2][2][2];
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int jb = 0; jb < 2; ++jb)
#pragma unroll
            for (int ib = 0; ib < 2; ++ib) {
              X[kb][jb][ib] = c[kb][jb][ib].X;
              NU[kb][jb][ib] = c[kb][jb][ib].NU;
              F[kb][jb][ib] = c[kb][jb][ib].F;
              UP[kb][jb][ib] = c[kb][jb][ib].UP;
            }
        const long long el = ((long long)ek * nely + ej) * nelx + e;
        const float* fg_in = fl.srcg ? q.fgp + (long long)b * q.fgp_sb + el : nullptr;
        // an element is formed twice where tiles / z-chunks overlap: only its owner writes grad_fgp
        const bool own = (tx == 0 || lx >= 1) && (ty == 0 || r >= 1) && ek >= z0;
        float* fg_out = (fl.fo && own) ? q.g_fgp + ((q.bc & 2u) ? 0 : (long long)b * ngpe) + el : nullptr;
        element<2, NG, MODE>(q, fl, X, NU, F, UP, fg_in, fg_out, (q.bc & 2u) && !first, nel, Q);
      }
      float2* cur = xch + (long long)buf * 3 * NS * kind + threadIdx.x;
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        cur[(0 * NS + s) * kind] = make_float2(Q[s][0][0][1], Q[s][1][0][1]);   // for the right neighbour
        cur[(1 * NS + s) * kind] = make_float2(Q[s][0][1][0], Q[s][1][1][0]);   // for the thread below
        cur[(2 * NS + s) * kind] = make_float2(Q[s][0][1][1], Q[s][1][1][1]);   // for the thread below-right
      }
      __syncthreads();
      const float2 zero = make_float2(0.f, 0.f);
      float n[3] = {0.f, 0.f, 0.f};
#pragma unroll
      for (int s = 0; s < NS; ++s) {
        const float2 fl_ = hasL ? cur[(0 * NS + s) * kind - 1] : zero;
        const float2 fu = hasU ? cur[(1 * NS + s) * kind - LXW] : zero;
        const float2 ful = (hasL && hasU) ? cur[(2 * NS + s) * kind - LXW - 1] : zero;
        n[s] = carry[s] + (Q[s][0][0][0] + fl_.x + (fu.x + ful.x));            // plane ek: complete
        carry[s] = Q[s][1][0][0] + fl_.y + (fu.y + ful.y);                    // plane ek + 1: waits a layer
      }
      buf ^= 1;
      if (ek >= z0 && st)
        store_node<MODE>(q, fl, b, first, nodes, (long long)ek * plane + (long long)ej * nx + e, n, c[0][0][0].last);
#pragma unroll
      for (int jb = 0; jb < 2; ++jb)
#pragma unroll
        for (int ib = 0; ib < 2; ++ib) c[0][jb][ib] = c[1][jb][ib];
    }
  }
}

template <int NG, int MODE>
cudaError_t launch(const InGrad& q, const Flags& fl, int nsd, int sms, cudaStream_t s) {
  const int ball = q.bc != 0;
  const long long bgrid = ball ? 1 : q.B;
  if (nsd == 2) {
    const long long ntx = (q.nx + 30) / 31;
    // rows per warp: enough warps for ~48 per SM, but at least 8 rows (the halo row costs 1/RY), at most 64
    long long ry = (q.ny * ntx * bgrid + sms * 48LL - 1) / (sms * 48LL);
    ry = std::min(64LL, std::max(8LL, ry));
    const long long nch = (q.ny + ry - 1) / ry;
    const dim3 grid((unsigned)ntx, (unsigned)((nch + kIgWarps - 1) / kIgWarps), (unsigned)bgrid);
    k_input_grads_2d<NG, MODE><<<grid, 32 * kIgWarps, 0, s>>>(q, fl, (int)ry, ball);
    return cudaGetLastError();
  }
  constexpr int NS = MODE ? 3 : 2;
  constexpr int ML = kIg3MaxLanes<NG>;
  const int ntx = q.nx <= ML ? 1 : (q.nx - 1 + ML - 2) / (ML - 1);
  const int lxw = (q.nx - 1 + ntx - 1) / ntx + 1;                      // 1 + ntx (lxw - 1) >= nx
  const int nty = q.ny <= kIg3Rows ? 1 : 1 + (q.ny - kIg3Rows + kIg3Rows - 2) / (kIg3Rows - 1);
  const long long tiles = (long long)ntx * nty * bgrid;
  // planes per chunk: ~4 CTAs per SM, but at least 8 planes (a chunk re-runs the layer below its first plane)
  long long zc = (q.nz * tiles + sms * 4LL - 1) / (sms * 4LL);
  zc = std::min<long long>(q.nz, std::max(8LL, zc));
  const long long nzc = (q.nz + zc - 1) / zc;
  const size_t smem = sizeof(float2) * 2 * 3 * NS * kIg3Rows * lxw;
  cudaError_t e = cudaFuncSetAttribute(k_input_grads_3d<NG, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem);
  if (e != cudaSuccess) return e;
  k_input_grads_3d<NG, MODE><<<(unsigned)(tiles * nzc), lxw * kIg3Rows, smem, s>>>(q, fl, lxw, (int)zc, ntx, nty,
                                                                                 ball);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_input_grads(const InGrad& q, int nsd, int sms, cudaStream_t s) {
  Flags fl;
  bool anyv = false;
  for (int k = 0; k < q.nmasks; ++k) anyv = anyv || q.g_v[k];
  fl.s0 = q.g_f != nullptr;
  fl.s1 = anyv;
  fl.s2 = q.mode == 1 && q.g_nu != nullptr;
  fl.fo = q.mode == 0 && q.g_fgp != nullptr;
  fl.srcf = q.mode == 0 && anyv && q.f.p != nullptr && q.cS != 0.f;
  fl.srcg = q.mode == 0 && anyv && q.fgp != nullptr && q.cS != 0.f;
  fl.dir = q.mode == 0 || fl.s2 || anyv;
  const int key = q.ng * 2 + q.mode;
  switch (key) {
    case 4: return launch<2, 0>(q, fl, nsd, sms, s);
    case 5: return launch<2, 1>(q, fl, nsd, sms, s);
    case 6: return launch<3, 0>(q, fl, nsd, sms, s);
    case 7: return launch<3, 1>(q, fl, nsd, sms, s);
    case 8: return launch<4, 0>(q, fl, nsd, sms, s);
    case 9: return launch<4, 1>(q, fl, nsd, sms, s);
  }
  return cudaErrorInvalidValue;
}

}  // namespace dn
