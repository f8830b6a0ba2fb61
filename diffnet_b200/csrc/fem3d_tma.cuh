// fem3d_tma.cuh -- the streaming 3-D Q1 (hex) Poisson energy/residual + adjoint kernel (sm_100a).
//
// Same operator as fem3d.cuh (which stays as the general path: odd sizes, unaligned or
// non-contiguous views, nx > 256, f at Gauss points), rebuilt around the two facts the profile of
// the first kernel showed: the 3-D element is ISSUE-bound (about 8x the arithmetic of the 2-D
// one per byte), and its loads must not sit in registers.
//
//   * A CTA owns a (TY rows) x (LXo element pairs) tile of a chunk of ZC node planes and marches
//     up in z.  Plane tiles with their halos ((TY+2) x (2 LXT + 2) nodes) travel HBM -> shared
//     memory through a ring of S stages filled by TMA tensor copies (cp.async.bulk.tensor.4d, SASS
//     UTMALDG; one instruction per field per plane, out-of-range nodes zero-filled by the TMA unit)
//     completing on one mbarrier per stage.  Any x-contiguous strided view is accepted.
//   * Thread (r, lx) owns ONE PAIR of hexahedra: element row r of the tile, columns 2lx, 2lx+1,
//     in every layer.  All element arithmetic is packed f32x2 (FFMA2/FADD2/FMUL2): the two
//     elements of the pair share every issue slot.
//   * The 2x2x2 modal (Hadamard) transform is hierarchical: x-sums/differences per node row,
//     y-stage per element face, z-stage per element.  The face below an element is the face above
//     the previous one: it is carried in registers, so each plane is read once per thread.
//     The transposed transform (modal gradient -> nodes) is hierarchical the same way and the
//     z-carry of the gradient is kept in face-mode space (one transposed y-stage per plane).
//   * Gradient gather without atomics: per plane each thread publishes its lower-row partial sums
//     to shared memory; after ONE __syncthreads (which also releases the consumed ring stage) the
//     owner of each node row adds the three neighbour shares, masks Dirichlet nodes and stores.
//   * Seams: one halo row above/below the tile, one halo pair column left of it and one halo
//     plane below/above the chunk are re-read (L2) and their elements recomputed:
//     (TY+1)/TY x (LXo+1)/LXo x (ZC+1)/ZC arithmetic (14 x 32 tiles: 1.07 x 1.03).
#pragma once
#include <cuda.h>

#include "fem2d_tma.cuh"

namespace dn {

#define DN_T3_MAXT 640      // largest CTA of any variant
// Register budgets (__maxnreg__; one CTA per SM).  Registers are granted per warp in units of 1024
// (measured: 112 registers/thread admit no more warps than 128), so the useful budgets are 96 and
// 128: nu == 1 variants fit 96 without spills -> 640-thread CTAs (20 warps/SM, +4 % measured);
// variable-nu variants need 128 -> 512-thread CTAs (96 registers spill: -4 %)
#define DN_T3_MAXT_OF(HAS_NU) ((HAS_NU) ? 512 : 640)
#define DN_T3_REGS_OF(HAS_NU) ((HAS_NU) ? 128 : 96)

// pair-replicated constants (half-gradient convention: k, not 2k)
struct K3 {
  float2 kx, ky, kz, kxt, kyt, kzt, kxtt, kytt, kztt, t, tt, nkf, nkft, nkftt, nkfttt, c0x, c0y, c0z;
  // Isotropic spacing (hx == hy == hz, every BASELINE grid): the stiffness part of E and g is linear
  // in k, so k is applied once per NODE (kscale, folded into the Dirichlet keep factor) and once per
  // thread (the energy weight) instead of 12 times per element; the source constants are divided
  // by k to compensate.  iso == 0: kscale == 1 and the per-direction constants above are used.
  float kscale;
  // nu == 1 on an isotropic grid: the three directional forms collapse to ONE product per mode,
  // q_m = n_m t^(order(m) - 1) c0 u_m with n_m = the number of directions mode m is differentiated in
  // (1, 2, 3 for the first-, second-, third-order modes): 7 products instead of 20 products + 5 sums.
  float2 c0_2t, c0_3tt;
  // assembled load vector (FK == 2): nkb = -(S c_f) weighs the nodal energy b u, nkb_pre = nkb / kscale the nodal
  // gradient share (added before the keep factor applies kscale)
  float nkb;
  float2 nkb_pre;
};

// Linked z-slab launch (include/diffnet_fem.h: dn_slab_link): the halo exchange of u and the loss
// all-reduce ride inside the FEM launch.  nput == 0: not linked.
struct Link3 {
  CUtensorMap tmh[2];           // (x, y, 1, 1) maps over the staged halo planes [below, above]
  const int* hflag[2];          // local flag words the neighbours release; null = no neighbour on that side
  float4* pdst[2];              // neighbour's staging plane (peer-mapped); null = none
  const float4* psrc[2];        // my first / last owned plane of u
  int* pflag[2];                // neighbour's flag word (peer-mapped)
  long long pn4;                // float4 per plane
  int nput;                     // CTAs that copy one side's plane (the launch is 2 * nput CTAs larger)
  unsigned int* tickets;        // [2] zero-initialised scratch
  int* status;                  // set to 1 if a device-side wait ran out of polls
  long long max_spins;
  int dbg;                      // timing experiments only (DN_SLAB_DBG): 1 skip the plane copy, 2 skip the flag wait, 4 skip the loss push
};

struct P3T {
  CUtensorMap tm[DN_T2_MAXF];   // one 4-D (x, y, z, b) tiled map per field; slot order: u, [nu], [f], [numask], masks..., [value field]
  int bmul[DN_T2_MAXF];         // 1: the field has a batch dimension, 0: broadcast over the batch
  float mval[DN_MAX_MASKS];
  int nf;
  int B, nx, ny, nz;
  int LXT, LXo, hl, ntx;        // lanes per tile row, owned pairs per tile, halo lanes (0/1), x tiles
  int rows, TY, nty;            // thread rows (element rows) per tile, owned node rows per tile, y tiles
  int ZC, nzc, S;               // planes per chunk, chunks, ring stages
  int BX, BY, fstride;          // box (nodes) and floats between fields in a stage (128-byte multiple)
  int zloss_lo, zloss_hi;       // element layers whose energy counts (z-slab ownership)
  K3 k3;
  float* grad;                  // dense (B, nz, ny, nx); nullable
  Reduce red;
  int mode;                     // 0: loss = energy; 1: loss = sum(out^2)
  Link3 lk;
};

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}

// Shared-memory accesses by 32-bit shared-window address (one register per address, [R + imm] forms).
// volatile: they keep their program order relative to the mbarrier waits and the CTA barrier.
__device__ __forceinline__ float2 lds64(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts64(uint32_t a, float2 v) {
  asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v.x), "f"(v.y));
}
__device__ __forceinline__ void sts32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v)); }
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "DN_WAIT3:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DN_DONE3;\n"
      "bra DN_WAIT3;\n"
      "DN_DONE3:\n"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}

// Face modes of one field for a pair of elements; index bit0 = x, bit1 = y; set bit = difference.
struct Face {
  float2 m0, m1, m2, m3;
};

// one direction of the stiffness form:  q = M(c) P  (half gradient),  P = 4 modal coefficients
// carrying the differentiated direction, c = the 4 nu modes that survive the integration.
// Q1,Q2,Q3 = t P1, t P2, t P3 and Q33 = t^2 P3 are shared between directions by the caller.
__device__ __forceinline__ void dir_q(float2 d0, float2 d1, float2 d2, float2 d3, float2 P0, float2 P1,
                                      float2 P2, float2 P3, float2 Q1, float2 Q2, float2 Q3, float2 Q33,
                                      float2& q0, float2& q1, float2& q2, float2& q3) {
  // ordered by nu mode: four consecutive FMAs share d_i (operand reuse cache: 2.3 instead of 3.0 dispatch
  // cycles per FFMA2, tools/micro/reuse.cu)
  q0 = mul2(d0, P0);       q1 = mul2(d0, Q1);       q2 = mul2(d0, Q2);       q3 = mul2(d0, Q33);
  q0 = fma2(d1, P1, q0);   q1 = fma2(d1, P0, q1);   q2 = fma2(d1, Q3, q2);   q3 = fma2(d1, Q2, q3);
  q0 = fma2(d2, P2, q0);   q1 = fma2(d2, Q3, q1);   q2 = fma2(d2, P0, q2);   q3 = fma2(d2, Q1, q3);
  q0 = fma2(d3, P3, q0);   q1 = fma2(d3, P2, q1);   q2 = fma2(d3, P1, q2);   q3 = fma2(d3, P0, q3);
}

// FK: 0 no source term, 1 nodal source, 2 `f` is an assembled load vector (see Fem2T): its term is added per
// node when the node's plane is gathered (finalize), not per element.
template <int NM, bool VF, bool HAS_NU, int FK, bool NUMASK, bool MI = true, bool ISO = false>
struct Fem3T {
  static constexpr bool HAS_F = (FK == 1), LV = (FK == 2);
  static constexpr int NF = 1 + (HAS_NU ? 1 : 0) + (FK ? 1 : 0) + (NUMASK ? 1 : 0) + NM + (VF ? 1 : 0);
  static constexpr int F_U = 0, F_NU = 1, F_F = F_NU + (HAS_NU ? 1 : 0), F_NM = F_F + (FK ? 1 : 0),
                       F_M = F_NM + (NUMASK ? 1 : 0), F_VF = F_M + NM;

  // x-stage of one node row (3 nodes -> 2 elements): s = (v0+v1, v1+v2), d = (v1-v0, v2-v1)
  static __device__ __forceinline__ void xs(const float (&v)[3], float2& s, float2& d) {
    s = f2(v[0] + v[1], v[1] + v[2]);
    d = f2(v[1] - v[0], v[2] - v[1]);
  }

  // Read node rows a (local row r) and b (r+1) of one plane from its ring stage, apply the
  // Dirichlet conditions / nu mask, and reduce to the face modes of u, nu, f.
  // `a0` = shared-window address of (row r, node x0) of field 0; `fs4` / `bx4` = bytes between
  // fields / rows.  keep = kscale at free nodes of row a, 0 at Dirichlet nodes.
  // `edge_warp` is warp-uniform: a phantom element (beyond the last node of a row, or the row below
  // the domain) lives in this warp; the common warps skip that work with one branch.
  static __device__ __forceinline__ void load_faces(const P3T& p, uint32_t a0, uint32_t bx4, uint32_t fs4,
                                                    bool has_right, bool phantom, bool edge_warp, Face& Uu,
                                                    Face& Un, Face& Uf, float2& keep, float2& lb, float& lE) {
    float2 su[2], du[2], sn[2], dn_[2], sf[2], df[2];
#pragma unroll
    for (int row = 0; row < 2; ++row) {
      float v[NF][3];
#pragma unroll
      for (int f = 0; f < NF; ++f) {
        const uint32_t q = a0 + f * fs4 + row * bx4;
        const float2 t = lds64(q);
        v[f][0] = t.x; v[f][1] = t.y;
        v[f][2] = lds32(q + 8u);            // beyond the last node the TMA unit has written zeros
      }
      float ub[3], nb[3], fb[3];
      bool fx[3];
#pragma unroll
      for (int e = 0; e < 3; ++e) {
        float u = v[F_U][e];
        fx[e] = false;
#pragma unroll
        for (int m = 0; m < NM; ++m) {
          const bool hit = v[F_M + m][e] > 0.5f;
          if constexpr (MI) u = hit ? (VF ? v[F_VF][e] : p.mval[m]) : u;   // MI = false: operator apply
          fx[e] = fx[e] || hit;
        }
        ub[e] = u;
        if constexpr (HAS_NU) {
          float n = v[F_NU][e];
          if constexpr (NUMASK) n = (v[F_NM][e] > 0.5f) ? 0.f : n;
          nb[e] = n;
        }
        if constexpr (HAS_F || LV) fb[e] = v[F_F][e];
      }
      if (row == 0) keep = f2(fx[0] ? 0.f : p.k3.kscale, fx[1] ? 0.f : p.k3.kscale);
      if constexpr (LV) {
        if (row == 0) {      // the two nodes of row a this thread gathers and stores
          lb = mul2(p.k3.nkb_pre, f2(fb[0], fb[1]));
          lE = p.k3.nkb * (fb[0] * ub[0] + fb[1] * ub[1]);
        }
      }
      xs(ub, su[row], du[row]);
      if constexpr (HAS_NU) xs(nb, sn[row], dn_[row]);
      if constexpr (HAS_F) xs(fb, sf[row], df[row]);
    }
    // a phantom element must not contribute: E and g are linear in (nu, f), so zeroing their
    // x-sums/differences removes it (nu == 1 uses the weight vw instead)
    if constexpr (HAS_NU || HAS_F) {
      if (edge_warp) {
#pragma unroll
        for (int row = 0; row < 2; ++row) {
          if constexpr (HAS_NU) {
            if (!has_right || phantom) { sn[row].y = 0.f; dn_[row].y = 0.f; }
            if (phantom) { sn[row].x = 0.f; dn_[row].x = 0.f; }
          }
          if constexpr (HAS_F) {
            if (!has_right || phantom) { sf[row].y = 0.f; df[row].y = 0.f; }
            if (phantom) { sf[row].x = 0.f; df[row].x = 0.f; }
          }
        }
      }
    }
    Uu.m0 = add2(su[0], su[1]); Uu.m1 = add2(du[0], du[1]);
    Uu.m2 = sub2(su[1], su[0]); Uu.m3 = sub2(du[1], du[0]);
    if constexpr (HAS_NU) {
      Un.m0 = add2(sn[0], sn[1]); Un.m1 = add2(dn_[0], dn_[1]);
      Un.m2 = sub2(sn[1], sn[0]); Un.m3 = sub2(dn_[1], dn_[0]);
    }
    if constexpr (HAS_F) {
      Uf.m0 = add2(sf[0], sf[1]); Uf.m1 = add2(df[0], df[1]);
      Uf.m2 = sub2(sf[1], sf[0]); Uf.m3 = sub2(df[1], df[0]);
    }
  }

  // z-stage of one pair of hexahedra: the 8 modes of u (and of nu, f) from the face modes of the lower (L*)
  // and upper (U*) faces; modes m = 4*zbit + 2*ybit + xbit.  After it the lower faces are dead.
  struct Modes {
    float2 u0, u1, u2, u3, u4, u5, u6, u7;
    float2 C0, C1, C2, C3, C4, C5, C6;
    float2 F0, F1, F2, F3, F4, F5, F6, F7;
  };
  static __device__ __forceinline__ void zstage(const Face& Lu, const Face& Uu, const Face& Ln, const Face& Un,
                                                const Face& Lf, const Face& Uf, Modes& M) {
    if constexpr (HAS_F) M.u0 = add2(Lu.m0, Uu.m0);
    M.u1 = add2(Lu.m1, Uu.m1); M.u2 = add2(Lu.m2, Uu.m2); M.u3 = add2(Lu.m3, Uu.m3);
    M.u4 = sub2(Uu.m0, Lu.m0); M.u5 = sub2(Uu.m1, Lu.m1); M.u6 = sub2(Uu.m2, Lu.m2); M.u7 = sub2(Uu.m3, Lu.m3);
    if constexpr (HAS_NU) {
      M.C0 = add2(Ln.m0, Un.m0); M.C1 = add2(Ln.m1, Un.m1); M.C2 = add2(Ln.m2, Un.m2); M.C3 = add2(Ln.m3, Un.m3);
      M.C4 = sub2(Un.m0, Ln.m0); M.C5 = sub2(Un.m1, Ln.m1); M.C6 = sub2(Un.m2, Ln.m2);
    }
    if constexpr (HAS_F) {
      M.F0 = add2(Lf.m0, Uf.m0); M.F1 = add2(Lf.m1, Uf.m1); M.F2 = add2(Lf.m2, Uf.m2); M.F3 = add2(Lf.m3, Uf.m3);
      M.F4 = sub2(Uf.m0, Lf.m0); M.F5 = sub2(Uf.m1, Lf.m1); M.F6 = sub2(Uf.m2, Lf.m2); M.F7 = sub2(Uf.m3, Lf.m3);
    }
  }

  // One pair of hexahedra between the lower faces L* and the upper faces U*.  Returns the energy
  // pair; gLo / gUp = gradient w.r.t. the face modes of u on the lower / upper face.
  static __device__ __forceinline__ float2 elem_pair(const K3& k, const Face& Lu, const Face& Uu,
                                                     const Face& Ln, const Face& Un, const Face& Lf,
                                                     const Face& Uf, float2 vw, Face& gLo, Face& gUp) {
    Modes M;
    zstage(Lu, Uu, Ln, Un, Lf, Uf, M);
    return elem_modes(k, M, vw, gLo, gUp);
  }

  // The element in modal space (everything after the z-stage).
  static __device__ __forceinline__ float2 elem_modes(const K3& k, const Modes& M, float2 vw, Face& gLo, Face& gUp) {
    const float2 u1 = M.u1, u2 = M.u2, u3 = M.u3, u4 = M.u4, u5 = M.u5, u6 = M.u6, u7 = M.u7;
    float2 q1, q2, q3, q4, q5, q6, q7;          // half gradient per mode
    if constexpr (HAS_NU) {
      float2 qx0, qx1, qx2, qx3, qy0, qy1, qy2, qy3, qz0, qz1, qz2, qz3;
      const float2 Q3 = mul2(k.t, u3), Q5 = mul2(k.t, u5), Q6 = mul2(k.t, u6), Q7 = mul2(k.t, u7),
                   Q77 = mul2(k.tt, u7);
      const float2 C0 = M.C0, C1 = M.C1, C2 = M.C2, C3 = M.C3, C4 = M.C4, C5 = M.C5, C6 = M.C6;
      float2 dx0, dx1, dx2, dx3, dy0, dy1, dy2, dy3, dz0, dz1, dz2, dz3;
      if constexpr (ISO) {   // k is applied per node / per thread (K3::kscale): 6 products instead of 12
        const float2 T1 = mul2(k.t, C1), T2 = mul2(k.t, C2), T4 = mul2(k.t, C4);
        dx0 = C0; dx1 = T2; dx2 = T4; dx3 = mul2(k.tt, C6);
        dy0 = C0; dy1 = T1; dy2 = T4; dy3 = mul2(k.tt, C5);
        dz0 = C0; dz1 = T1; dz2 = T2; dz3 = mul2(k.tt, C3);
      } else {
        dx0 = mul2(k.kx, C0); dx1 = mul2(k.kxt, C2); dx2 = mul2(k.kxt, C4); dx3 = mul2(k.kxtt, C6);
        dy0 = mul2(k.ky, C0); dy1 = mul2(k.kyt, C1); dy2 = mul2(k.kyt, C4); dy3 = mul2(k.kytt, C5);
        dz0 = mul2(k.kz, C0); dz1 = mul2(k.kzt, C1); dz2 = mul2(k.kzt, C2); dz3 = mul2(k.kztt, C3);
      }
      // d/dx: P = (xi, xi eta, xi zeta, xi eta zeta); nu modes (1, eta, zeta, eta zeta)
      dir_q(dx0, dx1, dx2, dx3, u1, u3, u5, u7, Q3, Q5, Q7, Q77, qx0, qx1, qx2, qx3);
      // d/dy: P = (eta, xi eta, eta zeta, xi eta zeta); nu modes (1, xi, zeta, xi zeta)
      dir_q(dy0, dy1, dy2, dy3, u2, u3, u6, u7, Q3, Q6, Q7, Q77, qy0, qy1, qy2, qy3);
      // d/dz: P = (zeta, xi zeta, eta zeta, xi eta zeta); nu modes (1, xi, eta, xi eta)
      dir_q(dz0, dz1, dz2, dz3, u4, u5, u6, u7, Q5, Q6, Q7, Q77, qz0, qz1, qz2, qz3);
      q1 = qx0; q2 = qy0; q3 = add2(qx1, qy1); q4 = qz0; q5 = add2(qx2, qz1);
      q6 = add2(qy2, qz2); q7 = add2(qx3, add2(qy3, qz3));
    } else if constexpr (ISO) {
      // nu == 1, hx == hy == hz: C0 = 8 (times the validity weight of the element), every direction has the same
      // constant; the per-thread products with vw are loop invariants
      const float2 d = mul2(k.c0x, vw), d2 = mul2(k.c0_2t, vw), d3 = mul2(k.c0_3tt, vw);
      q1 = mul2(d, u1); q2 = mul2(d, u2); q4 = mul2(d, u4);
      q3 = mul2(d2, u3); q5 = mul2(d2, u5); q6 = mul2(d2, u6);
      q7 = mul2(d3, u7);
    } else {
      // nu == 1: C0 = 8 (times the validity weight of the element), all other modes 0
      const float2 Q3 = mul2(k.t, u3), Q5 = mul2(k.t, u5), Q6 = mul2(k.t, u6), Q77 = mul2(k.tt, u7);
      const float2 dx = mul2(k.c0x, vw), dy = mul2(k.c0y, vw), dz = mul2(k.c0z, vw);
      q1 = mul2(dx, u1); q2 = mul2(dy, u2); q4 = mul2(dz, u4);
      q3 = add2(mul2(dx, Q3), mul2(dy, Q3)); q5 = add2(mul2(dx, Q5), mul2(dz, Q5));
      q6 = add2(mul2(dy, Q6), mul2(dz, Q6)); q7 = add2(mul2(dx, Q77), add2(mul2(dy, Q77), mul2(dz, Q77)));
    }
    float2 E, g0, g1, g2, g3, g4, g5, g6, g7;
    if constexpr (HAS_F) {
      const float2 u0 = M.u0;
      // t_m = q_m + nb_m with nb_m = -kf t^order(m) f_m, fused: one FFMA2 per mode
      const float2 nb0 = mul2(k.nkf, M.F0);
      const float2 t1 = fma2(k.nkft, M.F1, q1), t2 = fma2(k.nkft, M.F2, q2), t4 = fma2(k.nkft, M.F4, q4);
      const float2 t3 = fma2(k.nkftt, M.F3, q3), t5 = fma2(k.nkftt, M.F5, q5), t6 = fma2(k.nkftt, M.F6, q6);
      const float2 t7 = fma2(k.nkfttt, M.F7, q7);
      E = fma2(u0, nb0, fma2(u1, t1, fma2(u2, t2, fma2(u3, t3, fma2(u4, t4, fma2(u5, t5, fma2(u6, t6,
               mul2(u7, t7))))))));
      g0 = nb0; g1 = add2(q1, t1); g2 = add2(q2, t2); g3 = add2(q3, t3); g4 = add2(q4, t4);
      g5 = add2(q5, t5); g6 = add2(q6, t6); g7 = add2(q7, t7);
    } else {
      E = fma2(u1, q1, fma2(u2, q2, fma2(u3, q3, fma2(u4, q4, fma2(u5, q5, fma2(u6, q6, mul2(u7, q7)))))));
      g0 = f2(0.f); g1 = add2(q1, q1); g2 = add2(q2, q2); g3 = add2(q3, q3); g4 = add2(q4, q4);
      g5 = add2(q5, q5); g6 = add2(q6, q6); g7 = add2(q7, q7);
    }
    // transposed z-stage
    gLo.m0 = sub2(g0, g4); gLo.m1 = sub2(g1, g5); gLo.m2 = sub2(g2, g6); gLo.m3 = sub2(g3, g7);
    gUp.m0 = add2(g0, g4); gUp.m1 = add2(g1, g5); gUp.m2 = add2(g2, g6); gUp.m3 = add2(g3, g7);
    return E;
  }
};

// Row-space gradient of one face: (sum, difference) coefficients of node rows a (upper y) and b.
struct RowG {
  float2 sa, da, sb, db;
};
__device__ __forceinline__ RowG face_to_rows(const Face& g) {   // transposed y-stage
  RowG o;
  o.sa = sub2(g.m0, g.m2); o.da = sub2(g.m1, g.m3);
  o.sb = add2(g.m0, g.m2); o.db = add2(g.m1, g.m3);
  return o;
}

// One lane of the warp, chosen by the hardware (the branch around it must be warp-uniform).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(pred));
  return pred != 0;
}

// Exchange area (gradient gather between thread rows / lanes), FIXED geometry so that every
// address in the main loop is [thread register + immediate].  Per parity, in floats:
//   nb  float2[XPRE + MAXT]  row-b partial sums of thread i at slot XPRE + i; the reader (one tile row
//                            below) reads slot XPRE + i - LXT: row 0 lands in the never-written, zero prefix
//   hb  float [XPRE + MAXT + 4], ha likewise: right-neighbour shares of row b / row a.  The last
//       lane of every tile row (its right neighbour belongs to another tile or does not exist) and
//       lanes that hold no pair store to the trash word at the end of each array, so the slot the
//       first lane of a row reads stays zero: no predicates in the gather.
constexpr int kXPre = 132;                                   // >= LXT + 1 (BX <= 256 -> LXT <= 126)
constexpr int kXNb = 0, kXHb = 2 * (kXPre + DN_T3_MAXT), kXHa = kXHb + kXPre + DN_T3_MAXT + 4;
constexpr int kXParity = kXHa + kXPre + DN_T3_MAXT + 4;      // floats per parity
constexpr int kXTrash = kXPre + DN_T3_MAXT + 2;              // slot index (within hb / ha) nobody reads
__host__ __device__ constexpr int xbuf_bytes() { return 2 * kXParity * 4; }

// Linked z-slab launch: wait (bounded) until the neighbour has released this step's halo plane, then make its
// stores visible to the TMA unit.  Executed by the WHOLE producer warp, convergently (one broadcast load per
// poll), as ONE opaque asm statement, at most twice per CTA.  The same loop under the elected-lane branch of the
// producer -- as C++, as a call or as asm -- made the compiler give up the uniform datapath for the whole main
// loop (ncu on the loopback harness: +15 % instructions -- per-thread IMAD/ISETP, BSSY/BSYNC/YIELD around every
// refill, spills).
__device__ __forceinline__ void wait_halo_flag(const int* flag, const int* step, long long max_spins, int* status,
                                               int dbg) {
  const int want = (dbg & 2) ? (int)0x80000000 : *step + 1;   // the step counter advances only in the finisher's epilogue
  int seen;
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      ".reg .s64 n;\n"
      "mov.s64 n, 0;\n"
      "DN_HSPIN:\n"
      "ld.acquire.sys.global.s32 %0, [%1];\n"
      "setp.ge.s32 P1, %0, %2;\n"
      "@P1 bra DN_HDONE;\n"
      "nanosleep.u32 32;\n"
      "add.s64 n, n, 1;\n"
      "setp.lt.s64 P1, n, %3;\n"
      "@P1 bra DN_HSPIN;\n"
      "DN_HDONE:\n"
      "fence.proxy.async.global;\n"
      "}"
      : "=r"(seen)
      : "l"(flag), "r"(want), "l"(max_spins)
      : "memory");
  if (seen < want) *status = 1;
}

// LK: linked z-slab launch (dn_slab_link) -- separate instantiations, so that the plain kernels carry none of it
template <int NM, bool VF, bool HAS_NU, int FK, bool NUMASK, bool MI, bool ISO, bool LK>
__global__ void __maxnreg__(DN_T3_REGS_OF(HAS_NU)) k_fem3d_tma(const __grid_constant__ P3T p) {
  using F = Fem3T<NM, VF, HAS_NU, FK, NUMASK, MI, ISO>;
  constexpr int NF = F::NF;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double s_red[DN_T3_MAXT / 32];
  __shared__ unsigned int s_ticket;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform by construction
  const int NT = blockDim.x;                                // >= LXT * rows, multiple of 32
  const int nx = p.nx, LXT = p.LXT, S = p.S, BX = p.BX, fstride = p.fstride;
  const int stage_floats = NF * fstride;
  float* const ring = reinterpret_cast<float*>(smem_raw);                                   // [S][NF][fstride]
  uint64_t* const full = reinterpret_cast<uint64_t*>(ring + (size_t)S * stage_floats);      // [S] + 1: the layer barrier
  float* const xbuf = reinterpret_cast<float*>(full + S + 1);                               // [2][kXParity]

  // ---- linked z-slab launch: the first 2 * nput CTAs push this rank's boundary planes of u into the
  // neighbours' staging buffers (plain vectorised stores over NVLink), release the neighbours' flag
  // words (system scope, last CTA of a side through a ticket) and are done
  const int nputc = LK ? 2 * p.lk.nput : 0;
  if (nputc) {
    pdl_wait();
    if ((int)blockIdx.x < nputc) {
      const int want = *p.red.step + 1;
      if (tid == 0) s_ticket = draw_start_ticket(p.red, 0);
      const int side = (int)blockIdx.x / p.lk.nput, part = (int)blockIdx.x - side * p.lk.nput;
      if (p.lk.pdst[side]) {
        float4* dst = p.lk.pdst[side];
        const float4* src = p.lk.psrc[side];
        if (!(p.lk.dbg & 1))
          for (long long i = (long long)part * NT + tid; i < p.lk.pn4; i += (long long)p.lk.nput * NT) dst[i] = src[i];
        __threadfence_system();
        __syncthreads();
        if (tid == 0) {
          const unsigned int t = atomicAdd(p.lk.tickets + side, 1u);
          if (t == (unsigned)p.lk.nput - 1) {          // every CTA of this side has fenced its stores
            p.lk.tickets[side] = 0u;
            __threadfence_system();
            *reinterpret_cast<volatile int*>(p.lk.pflag[side]) = want;
          }
        }
      }
      finish_loss_w0<8>(p.red, 0.0, s_ticket);
      return;
    }
  }

  // ---- work item: (b, z-chunk, y-tile, x-tile)
  int w_ = (int)blockIdx.x - nputc;
  const int itx = w_ % p.ntx; w_ /= p.ntx;
  const int ity = w_ % p.nty; w_ /= p.nty;
  const int izc = w_ % p.nzc;
  const int b = w_ / p.nzc;
  const int ty0 = ity * p.TY, ty1 = min(p.ny, ty0 + p.TY);      // owned node rows [ty0, ty1)
  const int jf = max(ty0 - 1, 0), jl = min(ty1, p.ny - 1);       // node rows needed: jf..jl
  // element rows of this tile; the tile that holds the domain's last node row runs one PHANTOM
  // element row below it (nodes beyond the domain are zero-filled by the TMA unit, its nu / f / weight
  // are zeroed), so that the last node row is gathered and stored like every other row
  const int TRr = jl - jf, TR = TRr + (ty1 == p.ny ? 1 : 0);
  const int z0 = izc * p.ZC, z1 = min(p.nz, z0 + p.ZC);          // owned node planes [z0, z1)
  const int zf = max(z0 - 1, 0), zl = min(z1, p.nz - 1);         // planes loaded: zf..zl
  const int npl = zl - zf + 1;                                   // >= 2
  const int pfirst = itx * p.LXo - p.hl;                         // pair handled by lane 0 (-1: none)
  // the TMA unit wants the innermost start coordinate 16-byte aligned: the box starts at the
  // multiple of 4 nodes at or below the first node of lane 0
  const int xs = (2 * pfirst) & ~3, xoff = 2 * pfirst - xs;

  // Linked launch, chunk that starts at the lower halo plane: march DOWN instead of up, so that the plane
  // the neighbour sends is needed last and its arrival hides behind the whole chunk.  The element code is
  // untouched: fed (upper, lower) instead of (lower, upper) it solves the z-mirrored problem, whose energy
  // and nodal gradients are the same numbers (every operation is sign-symmetric).
  const bool rev = LK && nputc && p.lk.hflag[0] && izc == 0 && (p.nzc > 1 || !p.lk.hflag[1]);
  // ---- producer: one elected lane of warp 0 issues one tensor copy per field per plane
  int issued = 0, ist = 0;
  auto issue_plane = [&]() {         // warp 0 only (warp-uniform)
    const int zpl = rev ? zl - issued : zf + issued;
    const int hs = (LK && nputc) ? ((zpl == 0 && p.lk.hflag[0]) ? 0 : ((zpl == p.nz - 1 && p.lk.hflag[1]) ? 1 : -1)) : -1;
    if (hs >= 0) wait_halo_flag(p.lk.hflag[hs], p.red.step, p.lk.max_spins, p.lk.status, p.lk.dbg);   // the whole warp polls (one broadcast load)
    if (elect_one()) {
      uint64_t* bar = full + ist;
      float* dst = ring + ist * stage_floats;
      mbar_arrive_expect_tx(bar, (uint32_t)(NF * BX * p.BY * 4));
      const CUtensorMap* tm0 = &p.tm[0];
      int c2 = zpl, c3 = b * p.bmul[0];
      if (hs >= 0) { tm0 = &p.lk.tmh[hs]; c2 = 0; c3 = 0; }
      tma_load_4d(dst, tm0, xs, jf, c2, c3, bar);
#pragma unroll
      for (int f = 1; f < NF; ++f)
        tma_load_4d(dst + f * fstride, &p.tm[f], xs, jf, zpl, b * p.bmul[f], bar);
    }
    ++issued;
    ist = (ist + 1 == S) ? 0 : ist + 1;
  };
  if (tid == 0) {
    for (int s = 0; s < S; ++s) mbar_init(full + s, 1);
    mbar_init(full + S, NT >> 5);                  // split-phase CTA barrier: one arrival per warp and layer
    fence_mbar_init();
  }
  for (int i = tid; i < 2 * kXParity; i += NT) xbuf[i] = 0.f;
  pdl_wait();
  __syncthreads();
  if (warp == 0) {
    const int n0 = min(S, npl);
    for (int q = 0; q < n0; ++q) issue_plane();
  }
  if (tid == 0) s_ticket = draw_start_ticket(p.red, b);   // its round trip hides behind the first plane loads

  // ---- thread geometry
  const int r_raw = tid / LXT, lx = tid - r_raw * LXT;
  const int pp = pfirst + lx;                    // this thread's element pair (global index)
  const bool lvalid = (pp >= 0) && (2 * pp + 1 < nx);
  const bool rvalid = (r_raw < TR) && lvalid;
  const int r = (r_raw < TR) ? r_raw : 0;        // idle threads shadow a valid position (results dropped)
  const int x0 = 2 * pp;
  const bool has_right = (x0 + 2) < nx;
  const bool phantom = (r >= TRr);               // the element row below the domain's last node row
  // the phantom last element of a row / the phantom row is in this warp (the common warps skip that work)
  const bool edge_warp = __any_sync(0xffffffffu, !has_right || phantom);
  const int er = jf + r;                         // element row == its upper node row (a); b = er + 1
  const bool own_a = rvalid && (lx >= p.hl) && (er >= ty0);   // node row a is stored by this thread; element row owned
  const float2 vw = f2(phantom ? 0.f : 1.f, (has_right && !phantom) ? 1.f : 0.f);
  const K3& k = p.k3;
  float* gptr = p.grad ? p.grad + ((((long long)b * p.nz + (rev ? zl : zf)) * p.ny + er) * nx + (lvalid ? x0 : 0)) : nullptr;
  const long long plane_elems = rev ? -(long long)p.ny * nx : (long long)p.ny * nx;   // towards the next plane of the march
  const bool st_a = own_a && (gptr != nullptr);
  const float ew = (own_a && !phantom) ? k.kscale : 0.f;   // energy weight of this thread's element row
  const int elo = max(z0, p.zloss_lo), ecnt = p.zloss_hi - elo;
  const bool resid = (p.mode != 0);

  // ---- shared-window addresses (bytes): the ring row of this thread, its exchange slots
  const uint32_t fs4 = 4u * fstride, bx4 = 4u * BX, stage4 = 4u * stage_floats;
  const uint32_t row0 = smem_u32(ring) + 4u * (r * BX + xoff + 2 * (lvalid ? lx : p.hl));   // (row a, node x0), stage 0
  uint32_t cur = row0;
  uint32_t cbar = smem_u32(full);
  const uint32_t xb0 = smem_u32(xbuf);
  const uint32_t a_nw = xb0 + 8u * (kXPre + tid);                 // nb[tid]      (write)
  const uint32_t a_nr = a_nw - 8u * LXT;                          // nb[tid-LXT]  (read: row r-1, same lane)
  const uint32_t a_t4 = xb0 + 4u * (kXHb + kXPre + tid);          // hb[tid]; ha[tid] is 4 (kXHa - kXHb) further
  const uint32_t a_r4 = a_t4 - 4u * LXT;                          // hb[tid-LXT]
  const uint32_t a_hw = ((lx == LXT - 1) || !lvalid) ? xb0 + 4u * (kXHb + kXTrash) : a_t4;   // where the shares go
  constexpr uint32_t kHA = 4u * (kXHa - kXHb), kPAR = 4u * kXParity;

  // node planes alternate between two register sets: the upper faces of one layer are the
  // lower faces of the next (no copies)
  struct Plane { Face u, n, f; float2 keep, lb; float lE; };
  Plane PA, PB;
  Face up;                                       // z-carry of the gradient (face-mode space), upper plane
  up.m0 = up.m1 = up.m2 = up.m3 = f2(0.f);
  double acc = 0.0;
  float e32 = 0.f;
  int st = 0;
  uint32_t phase = 0;

  // The per-layer CTA barrier is SPLIT (an mbarrier, one arrival per warp): a warp arrives as soon as
  // its partial sums of plane s are published, then already fetches plane s+2 and reduces it to face
  // modes (into the register set of the plane it has just finished with) and only then waits for the
  // other warps, refills the ring and gathers plane s.  Warps that finish the element math early thus
  // run their load/mask phase while the others still compute: the two phases overlap across warps
  // instead of every warp stalling on the same latency at the same time.
  const uint32_t lbar = smem_u32(full + S);
  uint32_t lphase = 0;
  auto arrive = [&]() {
    __syncwarp();
    if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(lbar) : "memory");
  };
  auto wait_all = [&]() {
    mbar_wait_u32(lbar, lphase);
    lphase ^= 1u;
  };
  auto load_next = [&](Plane& U) {               // next ring stage: wait for its plane (long since requested), read it
    ++st; cur += stage4; cbar += 8u;
    if (st == S) { st = 0; cur = row0; cbar -= 8u * S; phase ^= 1u; }
    mbar_wait_u32(cbar, phase);
    F::load_faces(p, cur, bx4, fs4, has_right, phantom, edge_warp, U.u, U.n, U.f, U.keep, U.lb, U.lE);
  };
  auto refill = [&]() {                          // after the layer barrier: the oldest stage is free again
    if (warp == 0 && issued < npl) issue_plane();
  };
  // publish the row-b partial sums and the right-neighbour shares of a finished plane; returns the
  // part of node row a this thread already holds
  auto publish = [&](const RowG& d, const uint32_t po) -> float2 {
    const float2 loa = sub2(d.sa, d.da), hia = add2(d.sa, d.da);
    const float2 lob = sub2(d.sb, d.db), hib = add2(d.sb, d.db);
    sts64(a_nw + po, f2(lob.x, lob.y + hib.x));
    sts32(a_hw + po, hib.y);
    sts32(a_hw + kHA + po, hia.y);
    return f2(loa.x, loa.y + hia.x);
  };
  // after the barrier: gather the neighbours' shares for node row a, mask, store
  auto finalize = [&](float2 Na01, float2 keep, const uint32_t po, const bool sto, const float2 lb, const float lE) {
    const float2 nb = lds64(a_nr + po);                            // row r-1, same lane
    const float ha = lds32(a_t4 + kHA - 4u + po);                  // row a from lane lx-1   (thread tid-1)
    const float hb = lds32(a_r4 - 4u + po);                        // row b of row r-1 from lane lx-1 (thread tid-LXT-1)
    float2 G = f2(Na01.x + nb.x + (ha + hb), Na01.y + nb.y);
    if constexpr (F::LV) G = add2(G, lb);                          // load vector: -(c_f / kscale) b of the two nodes
    G = mul2(G, keep);
    if (sto) {
      if (st_a) *reinterpret_cast<float2*>(gptr) = G;
      if (resid && own_a) e32 += G.x * G.x + G.y * G.y;
      if constexpr (F::LV) e32 += (!resid && own_a) ? lE : 0.f;    // ... and their energy -c_f b u, once, by the owner
    }
    gptr += plane_elems;
  };

  // ---- first two planes of the march (npl >= 2): nothing before the first
  mbar_wait_u32(cbar, phase);
  F::load_faces(p, cur, bx4, fs4, has_right, phantom, edge_warp, PA.u, PA.n, PA.f, PA.keep, PA.lb, PA.lE);
  arrive();
  load_next(PB);
  wait_all();
  refill();                  // the stage of the first plane

  // element layer between the plane in L and the next plane of the march in U (both in registers).
  // `s` counts the layers from zf upwards; going up it IS the layer's index in the mesh (= its lower
  // plane) and the plane gathered and stored afterwards; going down (rev) those are mirrored in the chunk.
  auto layer = [&](Plane& L, Plane& U, const int s, const uint32_t po) {
    int sl = s, pl = s;
    if constexpr (LK) {
      if (rev) { sl = zl - 1 - (s - zf); pl = zl - (s - zf); }
    }
    Face gLo, gUp;
    const float2 E = F::elem_pair(k, L.u, U.u, L.n, U.n, L.f, U.f, vw, gLo, gUp);
    const float wl = (!resid && (unsigned)(sl - elo) < (unsigned)ecnt) ? ew : 0.f;
    e32 = fmaf(wl, E.x + E.y, e32);
    Face dF;                 // plane L is complete: carry from the layer below + this layer's lower face
    dF.m0 = add2(up.m0, gLo.m0); dF.m1 = add2(up.m1, gLo.m1);
    dF.m2 = add2(up.m2, gLo.m2); dF.m3 = add2(up.m3, gLo.m3);
    up = gUp;
    const float2 Na01 = publish(face_to_rows(dF), po);
    arrive();              // this warp has read the stage of the U plane and published its sums of the L plane
    const float2 keepL = L.keep, lbL = L.lb;
    const float lEL = L.lE;
    if (s + 2 <= zl) load_next(L);      // the plane after U replaces L in registers
    wait_all();            // every warp has arrived: partial sums visible, the oldest stage is free
    refill();
    if constexpr (LK) finalize(Na01, keepL, po, pl >= z0 && pl < z1, lbL, lEL);
    else finalize(Na01, keepL, po, s >= z0, lbL, lEL);
  };
  int s = zf;
  for (; s + 1 < zl; s += 2) {
    layer(PA, PB, s, 0u);
    layer(PB, PA, s + 1, kPAR);
    acc += (double)e32;
    e32 = 0.f;
  }
  const bool odd = s < zl;
  if (odd) layer(PA, PB, s, 0u);

  // ---- the last plane of the march when this chunk owns it (top plane of the domain going up, bottom
  // plane going down): no element layer beyond it
  if (rev ? (z0 == 0) : (z1 == p.nz)) {
    const uint32_t po = odd ? kPAR : 0u;
    const float2 Na01 = publish(face_to_rows(up), po);
    arrive();
    wait_all();
    finalize(Na01, odd ? PB.keep : PA.keep, po, true, odd ? PB.lb : PA.lb, odd ? PB.lE : PA.lE);
  }
  acc += (double)e32;

  pdl_trigger();
  acc = warp_sum(acc);
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  double cta = 0.0;
  if (tid == 0)
    for (int w = 0; w < (NT >> 5); ++w) cta += s_red[w];
  finish_loss_w0<8>(p.red, cta, s_ticket);   // 3-D grids are a few hundred CTAs
}

// The kernel of one fem3d_tma_combos.h variant (MK as in dn_launch.h), instantiated by fem3d_tma_inst.cu.
template <int MK, int NUK, int FK, bool NUMASK, bool LK>
const void* kernel3t();

}  // namespace dn
