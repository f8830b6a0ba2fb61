// fem2d.cuh -- fused 2-D Q1 Poisson energy / residual + adjoint, sm_100a.
//
// Replaces, in one pass over HBM, the reference's 20 conv2d + ~25 pointwise/reduction launches
// forward and 12 convolution_backward + pointwise launches backward
// (DiffNet/DiffNetFEM.py:7-18,143-153 + e.g. examples/poisson/single_instance/0_base.py:31-56).
//
// Mapping (DESIGN.md section 4):  one WARP owns a strip of 32*V consecutive node columns and
// marches down R node rows of one image.  Each lane owns V (=4: one 16-byte load) consecutive
// nodes and the V elements to their right.  Nodal values of the two rows bounding the current
// element row live in registers; the right neighbour's first node comes by warp shuffle, the
// node beyond the strip by one predicated scalar load in lane 31, and the element left of the
// strip (needed to complete the gradient of the strip's first node) is recomputed by lane 0.
// The gradient is gathered without atomics: per element row each lane accumulates the
// contributions to its V+1 top nodes (T) and bottom nodes (Bt); T is completed by one shuffle
// from the left neighbour and stored (one 16-byte store per lane), Bt becomes T of the next row.
//
// Element math: closed form of the Gauss sum for bilinear u, nu, f (exact for any symmetric rule
// with >= 2 points; `t` is the rule's second moment), written on un-normalised Hadamard
// coefficients A = (a+b+c+d, xi, eta, xi*eta), see DESIGN.md.
#pragma once
#include "dn_common.cuh"

namespace dn {

struct P2D {
  Field u, nu, f, fgp, numask;
  Mask mk[DN_MAX_MASKS];
  int B, nx, ny;
  Consts k;
  Rule rule;
  int R, nchunks, ntx, nitems;
  float* grad;          // dense (B, ny, nx); nullable (forward only)
  float* grad_nu;       // dense (B, ny, nx); nullable
  Reduce red;
  int mode;             // 0: loss = energy; 1: loss = sum(out^2) (residual form)
  int mask_input;       // substitute Dirichlet values into u (0 only for the resmin backward op)
};

template <int V, int NM>
struct Raw2D {
  float u[V], nu[V], f[V], nm[V];
  float m[NM > 0 ? NM : 1][V], mv[V];
  float hu, hnu, hf, hnm, hm[NM > 0 ? NM : 1], hmv;   // halo node of this lane (lane 0 / 31 only)
};

template <int V>
struct Row2D {
  float u[V + 1], nu[V + 1], f[V + 1];   // own V nodes + right neighbour
  float uL, nuL, fL;                      // node left of the strip (lane 0)
  unsigned fixed;                         // bit e: Dirichlet node
  unsigned nzero;                         // bit e: nu zeroed by nu_zero_mask
};

template <int V, int NM, bool VF, bool HAS_NU, int FM, bool NUMASK>
__device__ __forceinline__ void load_raw2d(const P2D& p, int b, int j, int x0, bool act, bool halo,
                                           int xh, Raw2D<V, NM>& r) {
  const long long ob = (long long)b, oj = (long long)j;
  ldv<V>(p.u.p + ob * p.u.sb + oj * p.u.sy + x0, act, r.u);
  r.hu = lds1(p.u.p + ob * p.u.sb + oj * p.u.sy + xh, halo);
  if constexpr (HAS_NU) {
    ldv<V>(p.nu.p + ob * p.nu.sb + oj * p.nu.sy + x0, act, r.nu);
    r.hnu = lds1(p.nu.p + ob * p.nu.sb + oj * p.nu.sy + xh, halo);
  }
  if constexpr (FM == 1) {
    ldv<V>(p.f.p + ob * p.f.sb + oj * p.f.sy + x0, act, r.f);
    r.hf = lds1(p.f.p + ob * p.f.sb + oj * p.f.sy + xh, halo);
  }
  if constexpr (NUMASK) {
    ldv<V>(p.numask.p + ob * p.numask.sb + oj * p.numask.sy + x0, act, r.nm);
    r.hnm = lds1(p.numask.p + ob * p.numask.sb + oj * p.numask.sy + xh, halo);
  }
#pragma unroll
  for (int k = 0; k < NM; ++k) {
    const Field& m = p.mk[k].m;
    ldv<V>(m.p + ob * m.sb + oj * m.sy + x0, act, r.m[k]);
    r.hm[k] = lds1(m.p + ob * m.sb + oj * m.sy + xh, halo);
  }
  if constexpr (VF) {   // NM == 1 by construction
    const Field& m = p.mk[0].vf;
    ldv<V>(m.p + ob * m.sb + oj * m.sy + x0, act, r.mv);
    r.hmv = lds1(m.p + ob * m.sb + oj * m.sy + xh, halo);
  }
}

// Dirichlet substitution  u = where(mask > 0.5, value, u)  in array order (later wins).
template <int NM, bool VF>
__device__ __forceinline__ float apply_masks(const P2D& p, float u, const float (&m)[NM > 0 ? NM : 1],
                                             float mv, bool& fixed) {
  fixed = false;
#pragma unroll
  for (int k = 0; k < NM; ++k) {
    const bool hit = m[k] > 0.5f;
    const float val = VF ? mv : p.mk[k].v;
    u = (hit && p.mask_input) ? val : u;
    fixed = fixed || hit;
  }
  return u;
}

template <int V, int NM, bool VF, bool HAS_NU, int FM, bool NUMASK>
__device__ __forceinline__ void make_row2d(const P2D& p, const Raw2D<V, NM>& r, int lane,
                                           Row2D<V>& o) {
  o.fixed = 0u;
  o.nzero = 0u;
#pragma unroll
  for (int e = 0; e < V; ++e) {
    float mk[NM > 0 ? NM : 1];
#pragma unroll
    for (int k = 0; k < NM; ++k) mk[k] = r.m[k][e];
    bool fx;
    o.u[e] = apply_masks<NM, VF>(p, r.u[e], mk, r.mv[e], fx);
    o.fixed |= fx ? (1u << e) : 0u;
    if constexpr (HAS_NU) o.nu[e] = (NUMASK && r.nm[e] > 0.5f) ? 0.f : r.nu[e];
    if constexpr (NUMASK) o.nzero |= (r.nm[e] > 0.5f) ? (1u << e) : 0u;
    if constexpr (FM == 1) o.f[e] = r.f[e];
  }
  bool fx;
  const float hu = apply_masks<NM, VF>(p, r.hu, r.hm, r.hmv, fx);
  const float hnu = HAS_NU ? ((NUMASK && r.hnm > 0.5f) ? 0.f : r.hnu) : 0.f;
  const float hf = (FM == 1) ? r.hf : 0.f;
  // right neighbour = first node of lane+1; lane 31 uses its halo load (0 if beyond the row)
  float un = __shfl_down_sync(0xffffffffu, o.u[0], 1);
  o.u[V] = (lane == 31) ? hu : un;
  if constexpr (HAS_NU) {
    float nn = __shfl_down_sync(0xffffffffu, o.nu[0], 1);
    o.nu[V] = (lane == 31) ? hnu : nn;
  }
  if constexpr (FM == 1) {
    float fn = __shfl_down_sync(0xffffffffu, o.f[0], 1);
    o.f[V] = (lane == 31) ? hf : fn;
  }
  o.uL = hu; o.nuL = hnu; o.fL = hf;   // meaningful in lane 0 only
}

// Effective modal source B = (B0, t*Bxi, t*Beta, t^2*Bxieta) of one element, pre-multiplied by kf.
template <int FM>
__device__ __forceinline__ void source2d(const P2D& p, float kf, float fa, float fb, float fc,
                                         float fd, int b, int j, int x, float (&kB)[4]) {
  if constexpr (FM == 1) {
    const float st = fa + fb, dt = fb - fa, sb = fc + fd, db = fd - fc;
    const float t = p.k.t;
    kB[0] = kf * (st + sb);
    kB[1] = kf * t * (dt + db);        // xi
    kB[2] = kf * t * (sb - st);        // eta
    kB[3] = kf * t * t * (db - dt);    // xi*eta
  } else if constexpr (FM == 2) {
    // f given at the Gauss points: moments of w_g f_g against (1, xi, eta, xi*eta)
    const int n = p.rule.n, nelx = p.nx - 1, nely = p.ny - 1;
    const float* base = p.fgp.p + (long long)b * p.fgp.sb + (long long)j * nelx + x;
    const long long gs = (long long)nely * nelx;
    float M0 = 0.f, Mx = 0.f, Me = 0.f, Mxe = 0.f;
    for (int jg = 0; jg < n; ++jg) {
      float r0 = 0.f, r1 = 0.f;
      for (int ig = 0; ig < n; ++ig) {
        const float v = __ldg(base + (long long)(jg * n + ig) * gs) * p.rule.w[ig];
        r0 += v; r1 += v * p.rule.x[ig];
      }
      const float wj = p.rule.w[jg], ej = p.rule.x[jg];
      M0 += wj * r0; Mx += wj * r1; Me += wj * ej * r0; Mxe += wj * ej * r1;
    }
    const float s = kf * p.rule.fscale;
    kB[0] = s * M0; kB[1] = s * Mx; kB[2] = s * Me; kB[3] = s * Mxe;
  } else {
    kB[0] = kB[1] = kB[2] = kB[3] = 0.f;
  }
}

// One Q1 element: nodes a=(j,i) b=(j,i+1) c=(j+1,i) d=(j+1,i+1).  Returns the element energy and
// d(energy)/d(nodal u) in g[4]; if GN, also d(energy)/d(nodal nu) in gn[4].
template <bool HAS_NU, int FM, bool GN>
__device__ __forceinline__ float elem2d(float kx, float ky, float t, const float (&kB)[4],
                                        float ua, float ub, float uc, float ud,
                                        float na, float nb, float nc, float nd,
                                        float (&g)[4], float (&gn)[4]) {
  const float st = ua + ub, dt = ub - ua, sb = uc + ud, db = ud - uc;
  const float A0 = st + sb, Ae = sb - st, Ax = dt + db, Axe = db - dt;
  float C0, Cx, Ce;
  if constexpr (HAS_NU) {
    const float ns = na + nb, nd_ = nb - na, ms = nc + nd, md = nd - nc;
    C0 = ns + ms; Ce = ms - ns; Cx = nd_ + md;
  } else {
    C0 = 4.f; Cx = 0.f; Ce = 0.f;
  }
  const float tAxe = t * Axe;
  // x-derivative part: kx [ C0 (Ax^2 + t Axe^2) + 2 t Ce Ax Axe ]
  const float c0x = 2.f * kx * C0, c1x = 2.f * kx * t * Ce;
  float gAx = c0x * Ax + c1x * Axe;
  float gAxe = c0x * tAxe + c1x * Ax;
  // y-derivative part: ky [ C0 (Ae^2 + t Axe^2) + 2 t Cx Ae Axe ]
  const float c0y = 2.f * ky * C0, c1y = 2.f * ky * t * Cx;
  float gAe = c0y * Ae + c1y * Axe;
  gAxe += c0y * tAxe + c1y * Ae;
  float E = 0.5f * (Ax * gAx + Ae * gAe + Axe * gAxe);   // Euler: quadratic form
  float g0 = 0.f;
  if constexpr (FM != 0) {
    E -= A0 * kB[0] + Ax * kB[1] + Ae * kB[2] + Axe * kB[3];
    g0 = -kB[0]; gAx -= kB[1]; gAe -= kB[2]; gAxe -= kB[3];
  }
  const float m0 = g0 - gAe, m1 = g0 + gAe, n0 = gAx - gAxe, n1 = gAx + gAxe;
  g[0] = m0 - n0; g[1] = m0 + n0; g[2] = m1 - n1; g[3] = m1 + n1;
  if constexpr (GN && HAS_NU) {
    // dE/dC0 = kx (Ax^2 + t Axe^2) + ky (Ae^2 + t Axe^2); dE/dCe = 2 kx t Ax Axe; dE/dCx = 2 ky t Ae Axe
    const float q = tAxe * Axe;
    const float h0 = kx * (Ax * Ax + q) + ky * (Ae * Ae + q);
    const float he = 2.f * kx * tAxe * Ax, hx = 2.f * ky * tAxe * Ae;
    gn[0] = h0 - hx - he; gn[1] = h0 + hx - he; gn[2] = h0 - hx + he; gn[3] = h0 + hx + he;
  }
  return E;
}

template <int V, int NM, bool VF, bool HAS_NU, int FM, bool NUMASK, bool GN>
__global__ void __launch_bounds__(128) k_fem2d(const P2D p) {
  __shared__ double s_red[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int wpc = blockDim.x >> 5;
  const int item = blockIdx.x * wpc + warp;
  double acc = 0.0;

  if (item < p.nitems) {
    const int tx = item % p.ntx;
    const int rest = item / p.ntx;
    const int ch = rest % p.nchunks, b = rest / p.nchunks;
    const int x0 = (tx * 32 + lane) * V;
    const bool act = x0 < p.nx;
    const bool left = (lane == 0) && (tx > 0);              // strip has a left neighbour strip
    const bool right = (lane == 31) && (x0 + V < p.nx);      // node beyond the strip exists
    const bool halo = left || right;
    const int xh = left ? (x0 - 1) : (x0 + V);
    const int r_begin = ch * p.R, r_end = min(p.ny, r_begin + p.R);
    const int j_first = max(r_begin - 1, 0), j_last = min(r_end, p.ny - 1);
    const float t = p.k.t;
    // validity of this lane's last element (x0+V-1 -> x0+V); others are valid whenever act
    const bool lastvalid = (x0 + V) < p.nx;

    Raw2D<V, NM> raw;
    Row2D<V> top, bot;
    load_raw2d<V, NM, VF, HAS_NU, FM, NUMASK>(p, b, j_first, x0, act, halo, xh, raw);
    make_row2d<V, NM, VF, HAS_NU, FM, NUMASK>(p, raw, lane, top);
    if (j_first < j_last)
      load_raw2d<V, NM, VF, HAS_NU, FM, NUMASK>(p, b, j_first + 1, x0, act, halo, xh, raw);

    float T[V + 1], Tn[V + 1];
#pragma unroll
    for (int e = 0; e <= V; ++e) { T[e] = 0.f; Tn[e] = 0.f; }

    for (int j = j_first; j < j_last; ++j) {
      make_row2d<V, NM, VF, HAS_NU, FM, NUMASK>(p, raw, lane, bot);
      if (j + 2 <= j_last)   // prefetch the next node row while this element row is computed
        load_raw2d<V, NM, VF, HAS_NU, FM, NUMASK>(p, b, j + 2, x0, act, halo, xh, raw);

      float Bt[V + 1], Bn[V + 1];
#pragma unroll
      for (int e = 0; e <= V; ++e) { Bt[e] = 0.f; Bn[e] = 0.f; }
      float erow = 0.f;
#pragma unroll
      for (int e = 0; e < V; ++e) {
        const bool valid = act && (e < V - 1 || lastvalid);
        const float w = valid ? 1.f : 0.f;
        float kB[4], g[4], gn[4];
        source2d<FM>(p, p.k.kf * w, top.f[e], top.f[e + 1], bot.f[e], bot.f[e + 1], b, j,
                     valid ? x0 + e : 0, kB);
        const float E = elem2d<HAS_NU, FM, GN>(p.k.kx * w, p.k.ky * w, t, kB,
                                               top.u[e], top.u[e + 1], bot.u[e], bot.u[e + 1],
                                               top.nu[e], top.nu[e + 1], bot.nu[e], bot.nu[e + 1],
                                               g, gn);
        erow += E;
        T[e] += g[0]; T[e + 1] += g[1]; Bt[e] += g[2]; Bt[e + 1] += g[3];
        if constexpr (GN) { Tn[e] += gn[0]; Tn[e + 1] += gn[1]; Bn[e] += gn[2]; Bn[e + 1] += gn[3]; }
      }
      if (left) {   // element left of the strip: only its right-hand nodes belong to this strip
        float kB[4], g[4], gn[4];
        source2d<FM>(p, p.k.kf, top.fL, top.f[0], bot.fL, bot.f[0], b, j, x0 - 1, kB);
        elem2d<HAS_NU, FM, GN>(p.k.kx, p.k.ky, t, kB, top.uL, top.u[0], bot.uL, bot.u[0],
                               top.nuL, top.nu[0], bot.nuL, bot.nu[0], g, gn);
        T[0] += g[1]; Bt[0] += g[3];
        if constexpr (GN) { Tn[0] += gn[1]; Bn[0] += gn[3]; }
      }
      // complete the first node with the left lane's contribution to it
      {
        const float fromL = __shfl_up_sync(0xffffffffu, T[V], 1);
        if (lane > 0) T[0] += fromL;
        if constexpr (GN) {
          const float nL = __shfl_up_sync(0xffffffffu, Tn[V], 1);
          if (lane > 0) Tn[0] += nL;
        }
      }
      if (j >= r_begin) {   // row j is owned by this chunk: count its energy, emit its gradient
        float G[V];
        float sq = 0.f;
#pragma unroll
        for (int e = 0; e < V; ++e) {
          G[e] = ((top.fixed >> e) & 1u) ? 0.f : T[e];
          sq += G[e] * G[e];
        }
        if (act) {
          if (p.grad) stv<V>(p.grad + ((long long)b * p.ny + j) * p.nx + x0, G);
          if constexpr (GN) {
            float Gn[V];
#pragma unroll
            for (int e = 0; e < V; ++e) Gn[e] = ((top.nzero >> e) & 1u) ? 0.f : Tn[e];
            stv<V>(p.grad_nu + ((long long)b * p.ny + j) * p.nx + x0, Gn);
          }
        }
        acc += (double)(p.mode == 0 ? erow : (act ? sq : 0.f));
      }
#pragma unroll
      for (int e = 0; e <= V; ++e) { T[e] = Bt[e]; if constexpr (GN) Tn[e] = Bn[e]; }
      top = bot;
    }
    // last node row of the image: no element row below it
    if (r_end == p.ny) {
      const float fromL = __shfl_up_sync(0xffffffffu, T[V], 1);
      if (lane > 0) T[0] += fromL;
      float G[V];
      float sq = 0.f;
#pragma unroll
      for (int e = 0; e < V; ++e) {
        G[e] = ((top.fixed >> e) & 1u) ? 0.f : T[e];
        sq += G[e] * G[e];
      }
      if constexpr (GN) {
        const float nL = __shfl_up_sync(0xffffffffu, Tn[V], 1);
        if (lane > 0) Tn[0] += nL;
      }
      if (act) {
        if (p.grad) stv<V>(p.grad + ((long long)b * p.ny + (p.ny - 1)) * p.nx + x0, G);
        if constexpr (GN) {
          float Gn[V];
#pragma unroll
          for (int e = 0; e < V; ++e) Gn[e] = ((top.nzero >> e) & 1u) ? 0.f : Tn[e];
          stv<V>(p.grad_nu + ((long long)b * p.ny + (p.ny - 1)) * p.nx + x0, Gn);
        }
        if (p.mode != 0) acc += (double)sq;
      }
    }
  }

  acc = warp_sum(acc);
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  double cta = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < wpc; ++w) cta += s_red[w];
  __syncthreads();
  finish_loss(p.red, cta, s_red);
}

// The kernel of one fem2d_combos.h variant (MK as in dn_launch.h), instantiated by fem2d_inst.cu.
template <int V, int MK, bool HAS_NU, int FM, bool NUMASK, bool GN>
const void* kernel2d();

}  // namespace dn
