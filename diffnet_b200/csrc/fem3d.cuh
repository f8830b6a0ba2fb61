// fem3d.cuh -- fused 3-D Q1 (hex) Poisson energy / residual + adjoint, sm_100a.
//
// Replaces the reference's 48 conv3d + ~25 pointwise/reduction launches forward and 32
// convolution_backward launches backward (DiffNet/DiffNetFEM.py:7-18,143-156 +
// IBN/poisson-3d/parametric/IBN_3D.py:114-136, IBN/poisson-3d/non-parametric/
// solve_in_object_3d.py:75-102) with one pass over HBM.
//
// Mapping (DESIGN.md section 5).  A CTA owns a (y,x) tile and marches up a chunk of z planes.
// Thread (r, lx) of the (TY+1) x LX block owns V (=4: one 16-byte load) consecutive nodes of
// node row y0+r in every plane and, for r < TY, the V hexahedra to their right/below/above.
// Per plane each thread loads its own nodes once (software-prefetched one plane ahead), applies
// the Dirichlet masks, and publishes them to shared memory; the row below and the node to the
// right are read back from there.  The nodal values of the lower plane stay in registers.
// Gradient: each thread accumulates its elements' contributions to the 2 x (V+1) nodes of the
// lower plane (`Dn`, complete in z after this layer) and of the upper plane (`Up`, carried to
// the next layer).  The lateral sum (row above, lane to the left, and the diagonal) goes through
// shared memory in the same barrier interval as the next plane's nodal exchange: ONE
// __syncthreads per plane, double-buffered.  No atomics; tile seams are closed by one halo row
// (r = 0), one halo column (lx = 0) and one halo plane per chunk, recomputed.
#pragma once
#include "dn_common.cuh"

namespace dn {

#define DN_MAXT_3D 512

// floats of dynamic shared memory per buffer for a (TY+1) x LX block of lane width V
inline int smem_floats_3d(int LX, int TY, int V) {
  const int NR = TY + 1, nvs = NR * LX * V;
  return (4 * nvs + 3 * NR + 2 * NR * LX + 3) & ~3;
}

struct P3D {
  Field u, nu, f, fgp, numask;
  Mask mk[DN_MAX_MASKS];
  int B, nx, ny, nz;
  Consts k;
  Rule rule;
  int LX, TY, ZC, ntx, nty, nzc;
  int zloss_lo, zloss_hi;   // element layers whose energy counts (z-slab ownership)
  float* grad;              // dense (B, nz, ny, nx); nullable
  Reduce red;
  int mode, mask_input;
};

template <int V, int NM>
struct Raw3D {
  float u[V], nu[V], f[V], nm[V];
  float m[NM > 0 ? NM : 1][V], mv[V];
  float hu, hnu, hf, hnm, hm[NM > 0 ? NM : 1], hmv;   // node right of the tile (lx == LX-1 only)
};

template <int NM, bool VF>
__device__ __forceinline__ float apply_masks3(const P3D& p, float u,
                                              const float (&m)[NM > 0 ? NM : 1], float mv,
                                              bool& fixed) {
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
__device__ __forceinline__ void load_raw3d(const P3D& p, int b, int z, int y, int x0, bool act,
                                           bool halo, Raw3D<V, NM>& r) {
  const long long ob = b, oz = z, oy = y;
  const int xh = x0 + V;
  {
    const float* q = p.u.p + ob * p.u.sb + oz * p.u.sz + oy * p.u.sy;
    ldv<V>(q + x0, act, r.u);
    r.hu = lds1(q + xh, halo);
  }
  if constexpr (HAS_NU) {
    const float* q = p.nu.p + ob * p.nu.sb + oz * p.nu.sz + oy * p.nu.sy;
    ldv<V>(q + x0, act, r.nu);
    r.hnu = lds1(q + xh, halo);
  }
  if constexpr (FM == 1) {
    const float* q = p.f.p + ob * p.f.sb + oz * p.f.sz + oy * p.f.sy;
    ldv<V>(q + x0, act, r.f);
    r.hf = lds1(q + xh, halo);
  }
  if constexpr (NUMASK) {
    const float* q = p.numask.p + ob * p.numask.sb + oz * p.numask.sz + oy * p.numask.sy;
    ldv<V>(q + x0, act, r.nm);
    r.hnm = lds1(q + xh, halo);
  }
#pragma unroll
  for (int k = 0; k < NM; ++k) {
    const Field& m = p.mk[k].m;
    const float* q = m.p + ob * m.sb + oz * m.sz + oy * m.sy;
    ldv<V>(q + x0, act, r.m[k]);
    r.hm[k] = lds1(q + xh, halo);
  }
  if constexpr (VF) {
    const Field& m = p.mk[0].vf;
    const float* q = m.p + ob * m.sb + oz * m.sz + oy * m.sy;
    ldv<V>(q + x0, act, r.mv);
    r.hmv = lds1(q + xh, halo);
  }
}

// In-place 2x2x2 Hadamard-like transform: index bit0 = x, bit1 = y, bit2 = z; a set bit means
// "difference along that axis" (v1 - v0), a clear bit "sum".
__device__ __forceinline__ void had8(float (&v)[8]) {
#pragma unroll
  for (int n = 0; n < 8; n += 2) { const float s = v[n] + v[n + 1], d = v[n + 1] - v[n]; v[n] = s; v[n + 1] = d; }
#pragma unroll
  for (int n = 0; n < 8; ++n) if (!(n & 2)) { const float s = v[n] + v[n + 2], d = v[n + 2] - v[n]; v[n] = s; v[n + 2] = d; }
#pragma unroll
  for (int n = 0; n < 4; ++n) { const float s = v[n] + v[n + 4], d = v[n + 4] - v[n]; v[n] = s; v[n + 4] = d; }
}

// Transposed transform (modal gradient -> nodal gradient).
__device__ __forceinline__ void had8_t(float (&g)[8]) {
#pragma unroll
  for (int n = 0; n < 4; ++n) { const float a = g[n] - g[n + 4], b = g[n] + g[n + 4]; g[n] = a; g[n + 4] = b; }
#pragma unroll
  for (int n = 0; n < 8; ++n) if (!(n & 2)) { const float a = g[n] - g[n + 2], b = g[n] + g[n + 2]; g[n] = a; g[n + 2] = b; }
#pragma unroll
  for (int n = 0; n < 8; n += 2) { const float a = g[n] - g[n + 1], b = g[n] + g[n + 1]; g[n] = a; g[n + 1] = b; }
}

// Directional stiffness term  k [ c0 (P0^2 + t P1^2 + t P2^2 + t^2 P3^2) + t c1 (2 P0 P1 + 2 t P2 P3)
//   + t c2 (2 P0 P2 + 2 t P1 P3) + t^2 c12 (2 P0 P3 + 2 P1 P2) ]  and its P-gradient; returns the term.
__device__ __forceinline__ float dir_term(float k, float t, float c0, float c1, float c2, float c12,
                                          float P0, float P1, float P2, float P3, float& g0,
                                          float& g1, float& g2, float& g3) {
  const float k2 = 2.f * k, kt = k2 * t;
  const float d0 = k2 * c0, d1 = kt * c1, d2 = kt * c2, d3 = kt * t * c12;
  const float Q1 = t * P1, Q2 = t * P2, Q3 = t * P3;
  g0 = d0 * P0 + d1 * P1 + d2 * P2 + d3 * P3;
  g1 = d0 * Q1 + d1 * P0 + d2 * Q3 + d3 * P2;
  g2 = d0 * Q2 + d1 * Q3 + d2 * P0 + d3 * P1;
  g3 = d0 * (t * Q3) + d1 * Q2 + d2 * Q1 + d3 * P0;
  return 0.5f * (P0 * g0 + P1 * g1 + P2 * g2 + P3 * g3);
}

// One Q1 hexahedron.  Node order n = 4*kb + 2*jb + ib (z, y, x).  u/nu/f are overwritten by
// their modal coefficients; g returns d(energy)/d(nodal u).
template <bool HAS_NU, int FM>
__device__ __forceinline__ float elem3d(const Consts& k, float w, float (&u)[8], float (&nu)[8],
                                        const float (&kB)[8], float (&g)[8]) {
  had8(u);
  float C0, C1, C2, C3, C4, C5, C6;
  if constexpr (HAS_NU) {
    had8(nu);
    C0 = nu[0]; C1 = nu[1]; C2 = nu[2]; C3 = nu[3]; C4 = nu[4]; C5 = nu[5]; C6 = nu[6];
  } else {
    C0 = 8.f; C1 = C2 = C3 = C4 = C5 = C6 = 0.f;
  }
  const float t = k.t;
  float gx0, gx1, gx2, gx3, gy0, gy1, gy2, gy3, gz0, gz1, gz2, gz3;
  // d/dx: P = (xi, xi*eta, xi*zeta, xi*eta*zeta); nu modes (1, eta, zeta, eta*zeta)
  float E = dir_term(k.kx * w, t, C0, C2, C4, C6, u[1], u[3], u[5], u[7], gx0, gx1, gx2, gx3);
  // d/dy: P = (eta, xi*eta, eta*zeta, xi*eta*zeta); nu modes (1, xi, zeta, xi*zeta)
  E += dir_term(k.ky * w, t, C0, C1, C4, C5, u[2], u[3], u[6], u[7], gy0, gy1, gy2, gy3);
  // d/dz: P = (zeta, xi*zeta, eta*zeta, xi*eta*zeta); nu modes (1, xi, eta, xi*eta)
  E += dir_term(k.kz * w, t, C0, C1, C2, C3, u[4], u[5], u[6], u[7], gz0, gz1, gz2, gz3);
  g[0] = 0.f;
  g[1] = gx0;
  g[2] = gy0;
  g[3] = gx1 + gy1;
  g[4] = gz0;
  g[5] = gx2 + gz1;
  g[6] = gy2 + gz2;
  g[7] = gx3 + gy3 + gz3;
  if constexpr (FM != 0) {
    float Ef = 0.f;
#pragma unroll
    for (int m = 0; m < 8; ++m) { Ef += u[m] * kB[m]; g[m] -= kB[m]; }
    E -= Ef;
  }
  had8_t(g);
  return E;
}

// kB[m] = kf * t^order(m) * B[m] from nodal f (FM 1) or from f at the Gauss points (FM 2).
template <int FM>
__device__ __forceinline__ void source3d(const P3D& p, float kf, float (&f)[8], int b, int z, int y,
                                         int x, float (&kB)[8]) {
  const float t = p.k.t;
  if constexpr (FM == 1) {
    had8(f);
    const float k1 = kf * t, k2 = k1 * t, k3 = k2 * t;
    kB[0] = kf * f[0];
    kB[1] = k1 * f[1]; kB[2] = k1 * f[2]; kB[4] = k1 * f[4];
    kB[3] = k2 * f[3]; kB[5] = k2 * f[5]; kB[6] = k2 * f[6];
    kB[7] = k3 * f[7];
  } else if constexpr (FM == 2) {
    const int n = p.rule.n;
    const long long nelx = p.nx - 1, nely = p.ny - 1, nelz = p.nz - 1;
    const long long gs = nelx * nely * nelz;
    const float* base = p.fgp.p + (long long)b * p.fgp.sb + ((long long)z * nely + y) * nelx + x;
    float M[8];
#pragma unroll
    for (int m = 0; m < 8; ++m) M[m] = 0.f;
    for (int kg = 0; kg < n; ++kg) {
      float s[4] = {0.f, 0.f, 0.f, 0.f};
      for (int jg = 0; jg < n; ++jg) {
        float r0 = 0.f, r1 = 0.f;
        for (int ig = 0; ig < n; ++ig) {
          const float v = __ldg(base + (long long)((kg * n + jg) * n + ig) * gs) * p.rule.w[ig];
          r0 += v; r1 += v * p.rule.x[ig];
        }
        const float wj = p.rule.w[jg], ej = wj * p.rule.x[jg];
        s[0] += wj * r0; s[1] += wj * r1; s[2] += ej * r0; s[3] += ej * r1;
      }
      const float wk = p.rule.w[kg], ek = wk * p.rule.x[kg];
#pragma unroll
      for (int q = 0; q < 4; ++q) { M[q] += wk * s[q]; M[4 + q] += ek * s[q]; }
    }
    const float sc = kf * p.rule.fscale;
#pragma unroll
    for (int m = 0; m < 8; ++m) kB[m] = sc * M[m];
  } else {
#pragma unroll
    for (int m = 0; m < 8; ++m) kB[m] = 0.f;
  }
}

template <int V, int NM, bool VF, bool HAS_NU, int FM, bool NUMASK>
__global__ void __launch_bounds__(DN_MAXT_3D) k_fem3d(const P3D p) {
  extern __shared__ __align__(16) float smem[];
  __shared__ double s_red[32];

  const int LX = p.LX, TY = p.TY, NR = TY + 1;
  const int lx = threadIdx.x, r = threadIdx.y;
  const int tid = r * LX + lx;
  // ---- decode the work item: (b, z-chunk, y-tile, x-tile)
  int w_ = blockIdx.x;
  const int itx = w_ % p.ntx; w_ /= p.ntx;
  const int ity = w_ % p.nty; w_ /= p.nty;
  const int izc = w_ % p.nzc;
  const int b = w_ / p.nzc;

  const int col = (p.ntx > 1 ? itx * (LX - 1) : 0) + lx;
  const int x0 = col * V;
  const int y = ity * (TY - 1) + r;
  const bool act = (x0 < p.nx) && (y < p.ny);
  const bool rhalo = act && (lx == LX - 1) && (x0 + V < p.nx);
  const bool crow = (r < TY) && act && (y + 1 < p.ny);          // this thread computes elements
  const bool own_x = (lx >= 1) || (itx == 0);
  // rows 1..TY-1 (plus row 0 of the first tile); the domain's last node row has no element row
  // below it, so when it lands on the loader row of the LAST tile that tile owns it too
  const bool own_y = ((r <= TY - 1) && ((r >= 1) || (ity == 0))) ||
                     ((r == TY) && (y == p.ny - 1) && (ity == p.nty - 1));
  const bool own = act && own_x && own_y;
  const bool lastvalid = (x0 + V) < p.nx;

  const int z0 = izc * p.ZC, z1 = min(p.nz, z0 + p.ZC);          // owned planes [z0, z1)
  const int zf = max(z0 - 1, 0), zl = min(z1, p.nz - 1);          // planes loaded: zf..zl

  // ---- shared memory carve-up (per buffer), vector regions first so they stay 16-byte aligned:
  //      [u][nu][f] nodal, [NR][LX][V] each; gradient exchange Dn[1][0..V) [NR][LX][V];
  //      then scalars: halo u,nu,f [3][NR]; Dn[1][V] [NR][LX]; Dn[0][V] [NR][LX]
  const int nvs = NR * LX * V;
  const int off_gxv = 3 * nvs, off_h = 4 * nvs, off_gxa = off_h + 3 * NR, off_gxb = off_gxa + NR * LX;
  const int per_buf_al = (off_gxb + NR * LX + 3) & ~3;

  auto publish_nv = [&](int buf, const float (&uu)[V], const float (&nn)[V], const float (&ff)[V],
                        float hu, float hnu, float hf) {
    float* s = smem + buf * per_buf_al;
    stv<V>(s + tid * V, uu);
    if constexpr (HAS_NU) stv<V>(s + nvs + tid * V, nn);
    if constexpr (FM == 1) stv<V>(s + 2 * nvs + tid * V, ff);
    if (lx == LX - 1) {
      float* h = s + off_h;
      h[r] = hu;
      if constexpr (HAS_NU) h[NR + r] = hnu;
      if constexpr (FM == 1) h[2 * NR + r] = hf;
    }
  };

  // gather rows (r, r+1) x cols (0..V) of one field from shared memory
  auto gather = [&](int buf, int field, const float (&own_v)[V], float own_h, float (&o)[2][V + 1]) {
    const float* s = smem + buf * per_buf_al + field * nvs;
    const float* h = smem + buf * per_buf_al + off_h + field * NR;
#pragma unroll
    for (int e = 0; e < V; ++e) o[0][e] = own_v[e];
    if constexpr (V == 4) {
      const float4 q = *reinterpret_cast<const float4*>(s + (tid + LX) * V);
      o[1][0] = q.x; o[1][1] = q.y; o[1][2] = q.z; o[1][3] = q.w;
    } else {
#pragma unroll
      for (int e = 0; e < V; ++e) o[1][e] = s[(tid + LX) * V + e];
    }
    if (lx == LX - 1) {
      o[0][V] = own_h;
      o[1][V] = h[r + 1];
    } else {
      o[0][V] = s[(tid + 1) * V];
      o[1][V] = s[(tid + 1 + LX) * V];
    }
  };

  Raw3D<V, NM> raw;
  float lowU[2][V + 1], lowN[2][V + 1], lowF[2][V + 1];
  float Done[2][V + 1], Up[2][V + 1];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int e = 0; e <= V; ++e) { Done[a][e] = 0.f; Up[a][e] = 0.f; lowU[a][e] = 0.f; lowN[a][e] = 0.f; lowF[a][e] = 0.f; }
  unsigned fixed_hist = 0u;   // bits [0,V): plane being published; [V,2V): one back; [2V,3V): two back
  double acc = 0.0;
  int buf = 0;

  // masked nodal values of the plane held in `raw`
  float cu[V], cn[V], cf[V], chu, chn, chf;
  auto mask_plane = [&]() {
    unsigned fx = 0u;
#pragma unroll
    for (int e = 0; e < V; ++e) {
      float mk[NM > 0 ? NM : 1];
#pragma unroll
      for (int k = 0; k < NM; ++k) mk[k] = raw.m[k][e];
      bool f_;
      cu[e] = apply_masks3<NM, VF>(p, raw.u[e], mk, raw.mv[e], f_);
      fx |= f_ ? (1u << e) : 0u;
      cn[e] = HAS_NU ? ((NUMASK && raw.nm[e] > 0.5f) ? 0.f : raw.nu[e]) : 0.f;
      cf[e] = (FM == 1) ? raw.f[e] : 0.f;
    }
    bool f_;
    chu = apply_masks3<NM, VF>(p, raw.hu, raw.hm, raw.hmv, f_);
    chn = HAS_NU ? ((NUMASK && raw.hnm > 0.5f) ? 0.f : raw.hnu) : 0.f;
    chf = (FM == 1) ? raw.hf : 0.f;
    fixed_hist = (fixed_hist << V) | fx;
  };

  // finalize + store the gradient of plane `zp` from Done (own) and the neighbours' exchange
  auto publish_gx = [&](int bufi) {
    float* s = smem + bufi * per_buf_al;
    float v1[V];
#pragma unroll
    for (int e = 0; e < V; ++e) v1[e] = Done[1][e];
    stv<V>(s + off_gxv + tid * V, v1);
    s[off_gxa + tid] = Done[1][V];
    s[off_gxb + tid] = Done[0][V];
  };
  auto finalize = [&](int bufi, int zp, int hist_shift) {
    if (!own) return;
    const float* s = smem + bufi * per_buf_al;
    float G[V];
#pragma unroll
    for (int e = 0; e < V; ++e) G[e] = Done[0][e];
    if (r >= 1) {
#pragma unroll
      for (int e = 0; e < V; ++e) G[e] += s[off_gxv + (tid - LX) * V + e];
    }
    if (lx >= 1) {
      G[0] += s[off_gxb + tid - 1];
      if (r >= 1) G[0] += s[off_gxa + tid - LX - 1];
    }
    const unsigned fx = (fixed_hist >> hist_shift) & ((1u << V) - 1u);
    float sq = 0.f;
#pragma unroll
    for (int e = 0; e < V; ++e) {
      G[e] = ((fx >> e) & 1u) ? 0.f : G[e];
      sq += G[e] * G[e];
    }
    if (zp >= z0 && zp < z1) {
      if (p.grad) stv<V>(p.grad + (((long long)b * p.nz + zp) * p.ny + y) * p.nx + x0, G);
      if (p.mode != 0) acc += (double)sq;
    }
  };

  // ---- prologue: first plane
  load_raw3d<V, NM, VF, HAS_NU, FM, NUMASK>(p, b, zf, y, x0, act, rhalo, raw);
  mask_plane();
  publish_nv(buf, cu, cn, cf, chu, chn, chf);
  __syncthreads();
  if (r < TY) {
    gather(buf, 0, cu, chu, lowU);
    if constexpr (HAS_NU) gather(buf, 1, cn, chn, lowN);
    if constexpr (FM == 1) gather(buf, 2, cf, chf, lowF);
  }
  buf ^= 1;
  if (zf < zl) load_raw3d<V, NM, VF, HAS_NU, FM, NUMASK>(p, b, zf + 1, y, x0, act, rhalo, raw);

  for (int s = zf; s < zl; ++s) {
    // ---- phase A: publish plane s+1 nodal values and the finished gradient partials of plane s-1
    mask_plane();
    publish_nv(buf, cu, cn, cf, chu, chn, chf);
    if (s > zf) publish_gx(buf);
    __syncthreads();
    // ---- phase B
    if (s > zf) finalize(buf, s - 1, 2 * V);
    float upU[2][V + 1], upN[2][V + 1], upF[2][V + 1];
    if (r < TY) {
      gather(buf, 0, cu, chu, upU);
      if constexpr (HAS_NU) gather(buf, 1, cn, chn, upN);
      if constexpr (FM == 1) gather(buf, 2, cf, chf, upF);
    }
    buf ^= 1;
    if (s + 2 <= zl) load_raw3d<V, NM, VF, HAS_NU, FM, NUMASK>(p, b, s + 2, y, x0, act, rhalo, raw);
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int e = 0; e <= V; ++e) { Done[a][e] = Up[a][e]; Up[a][e] = 0.f; }
    if (crow) {
      float esum = 0.f;
#pragma unroll
      for (int e = 0; e < V; ++e) {
        const bool valid = (e < V - 1) || lastvalid;
        const float w = valid ? 1.f : 0.f;
        float eu[8], en[8], ef[8], kB[8], g[8];
        eu[0] = lowU[0][e]; eu[1] = lowU[0][e + 1]; eu[2] = lowU[1][e]; eu[3] = lowU[1][e + 1];
        eu[4] = upU[0][e];  eu[5] = upU[0][e + 1];  eu[6] = upU[1][e];  eu[7] = upU[1][e + 1];
        if constexpr (HAS_NU) {
          en[0] = lowN[0][e]; en[1] = lowN[0][e + 1]; en[2] = lowN[1][e]; en[3] = lowN[1][e + 1];
          en[4] = upN[0][e];  en[5] = upN[0][e + 1];  en[6] = upN[1][e];  en[7] = upN[1][e + 1];
        }
        if constexpr (FM == 1) {
          ef[0] = lowF[0][e]; ef[1] = lowF[0][e + 1]; ef[2] = lowF[1][e]; ef[3] = lowF[1][e + 1];
          ef[4] = upF[0][e];  ef[5] = upF[0][e + 1];  ef[6] = upF[1][e];  ef[7] = upF[1][e + 1];
        }
        source3d<FM>(p, p.k.kf * w, ef, b, s, y, valid ? x0 + e : 0, kB);
        const float E = elem3d<HAS_NU, FM>(p.k, w, eu, en, kB, g);
        esum += E;
        Done[0][e] += g[0]; Done[0][e + 1] += g[1]; Done[1][e] += g[2]; Done[1][e + 1] += g[3];
        Up[0][e] += g[4];   Up[0][e + 1] += g[5];   Up[1][e] += g[6];   Up[1][e + 1] += g[7];
      }
      if (own && s >= z0 && s >= p.zloss_lo && s < p.zloss_hi && p.mode == 0) acc += (double)esum;
    }
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int e = 0; e <= V; ++e) { lowU[a][e] = upU[a][e]; lowN[a][e] = upN[a][e]; lowF[a][e] = upF[a][e]; }
  }

  // ---- epilogue: plane zl-1 is complete in Done; the domain's top plane is complete in Up
  if (zl > zf) {
    publish_gx(buf);
    __syncthreads();
    finalize(buf, zl - 1, V);
    buf ^= 1;
  }
  if (z1 == p.nz) {   // top node plane of the domain: no element layer above it
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int e = 0; e <= V; ++e) Done[a][e] = Up[a][e];
    publish_gx(buf);
    __syncthreads();
    finalize(buf, p.nz - 1, 0);
  }

  // ---- loss reduction
  acc = warp_sum(acc);
  const int nthreads = LX * NR, warp = tid >> 5, lane = tid & 31;
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  double cta = 0.0;
  if (tid == 0)
    for (int w2 = 0; w2 < (nthreads + 31) / 32; ++w2) cta += s_red[w2];
  if (p.red.seg_q) {     // reduction = none: a CTA is one work item of one sample, one slot per CTA
    if (warp == 0) finish_sample_warp(p.red, blockIdx.x, cta, lane, nthreads < 32 ? nthreads : 32);
    return;
  }
  __syncthreads();
  // finish_loss indexes threads by threadIdx.x: re-linearise through a 1-D view
  {
    __shared__ bool is_last;
    if (tid == 0) {
      p.red.partials[blockIdx.x] = cta;
      __threadfence();
      const unsigned int ticket = atomicAdd(p.red.counter, 1u);
      is_last = (ticket == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
      __threadfence();
      double sacc = 0.0;
      for (unsigned int i = tid; i < gridDim.x; i += nthreads) {
        sacc += __ldcg(p.red.partials + i);
        __stcg(p.red.partials + i, 0.0);     // zero on exit: the streaming kernels read zero as "not yet written"
      }
      sacc = warp_sum(sacc);
      if (lane == 0) s_red[warp] = sacc;
      __syncthreads();
      if (tid == 0) {
        double tot = 0.0;
        for (int w2 = 0; w2 < (nthreads + 31) / 32; ++w2) tot += s_red[w2];
        if (p.red.loss_out) *p.red.loss_out = tot;
        if (p.red.loss_f32) *p.red.loss_f32 = (float)tot;
        *p.red.counter = 0u;
      }
    }
  }
}

// The kernel of one fem3d_combos.h variant (MK as in dn_launch.h), instantiated by fem3d_inst.cu.
template <int V, int MK, bool HAS_NU, int FM, bool NUMASK>
const void* kernel3d();

}  // namespace dn
