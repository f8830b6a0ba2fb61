// fem2d_tma.cuh -- the streaming 2-D Q1 Poisson energy/residual + adjoint kernel (sm_100a).
//
// Same operator as fem2d.cuh (which stays as the general path: odd sizes, unaligned views,
// f at Gauss points, d/dnu), restructured for the B200 memory system:
//
//   * A CTA owns one chunk of R node rows of one image at FULL row width; thread t owns the four
//     nodes x0 = 4t .. 4t+3 of every row and the four elements to their right.
//   * Node rows of all NF input fields travel HBM -> shared memory through a ring of S stages
//     filled by bulk-async copies (cp.async.bulk, SASS UBLKCP) that complete on one mbarrier per
//     stage.  The bytes in flight live in shared memory, not in registers: S rows x NF fields per
//     CTA, 6-8 CTAs per SM, independent of how far the arithmetic has got.
//   * Each node row is read from shared memory exactly once (one 16-byte load per field plus the
//     right neighbour), masked, and reduced to its x-sums / x-differences, which serve both the
//     element row above and the one below.  The element math is the closed form of DESIGN.md 4
//     evaluated on float2 PAIRS of elements with FFMA2/FADD2/FMUL2 (two elements per issue slot).
//     The source term is linear in u: it enters per node, as a separable stencil, when a row closes.
//   * Gradient gather without atomics: contributions to the top nodes are completed by one
//     shuffle from the left lane (one shared-memory word across warp seams), contributions to
//     the bottom nodes are carried in registers to the next row.  One __syncthreads per row
//     releases the consumed ring stage and publishes the seam words.
//   * Chunk seams: one halo row above and below is re-read (from L2) and the element row above
//     the chunk recomputed; (R+2)/R reads, (R+1)/R arithmetic.
#pragma once
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "dn_common.cuh"

namespace dn {

#define DN_T2_MAXF 8        // u, nu, f, numask, masks[3] | mask+value_field
#define DN_T2_MAXT 512      // threads per CTA -> nx <= 2048

// Packed constants of one launch (see prepare(): kx, ky carry S c_k W (2/h)^2 / 64, kf = S c_f W / 16)
struct K2 {
  float2 kx, ky, kxt, kyt, t, c0x_const, c0y_const;
  // FK == 1, the nodal source stencil (Fem2T::load_row / src_share): 1-D element mass [[1+t, 1-t], [1-t, 1+t]]
  float2 nfc, nfw;   // x-stencil: -kf (1-t) per row neighbour, -kf 2(1+t) own weight
  float2 fmir;       // -(1+t)/(1-t): the missing neighbour of an image edge node, in units of the node's own f
  float2 yc, yw;     // y-stencil: (1-t) per neighbour row, 2(1+t) own weight (half of it in the image's top/bottom row)
  float2 nkb;        // -(S c_f): weight of an assembled load vector (FK == 2)
};

struct P2T {
  Field fld[DN_T2_MAXF];    // slot order: u, [nu], [f], [numask], masks..., [value field]
  float mval[DN_MAX_MASKS];
  int nf;
  int B, nx, ny;
  int R, nchunks, S;
  int bal_q, bal_rem;       // bal_q > 0: balanced one-wave split -- images [0, bal_rem) have bal_q + 1 equal chunks, the rest bal_q
  K2 k2;                    // packed (pair-replicated) constants, read straight from the constant bank
  float* grad;              // dense (B, ny, nx); nullable (forward only)
  Reduce red;
  int mode;                 // 0: loss = energy; 1: loss = sum(out^2) (residual form)
};

// ---- PTX wrappers: mbarrier + bulk async copy ------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
// Programmatic dependent launch (a no-op for a grid launched without the attribute):
// pdl_trigger() lets the NEXT grid in the stream begin launching while this one still runs;
// pdl_wait() blocks until the PREVIOUS grid has completed and its memory is visible.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "DN_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DN_DONE;\n"
      "bra DN_WAIT;\n"
      "DN_DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// predicated shared-memory store: no divergent branch around a one-lane store
__device__ __forceinline__ void sts_if(bool pred, float* p, float v) {
  asm volatile("{\n.reg .pred P;\nsetp.ne.u32 P, %0, 0;\n@P st.shared.f32 [%1], %2;\n}" ::"r"((unsigned)pred), "r"(smem_u32(p)), "f"(v)
               : "memory");
}

// ---- float2 helpers (FADD2 / FMUL2 / FFMA2) --------------------------------------------------
__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
  return __fadd2_rn(a, make_float2(-b.x, -b.y));   // the negation folds into the operand modifier
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }

// x-sums and x-differences of one masked node row: s[e] = v[e] + v[e+1], d[e] = v[e+1] - v[e]
struct RowSD {
  float2 s01, s23, d01, d23;
};
__device__ __forceinline__ RowSD row_sd(const float (&v)[5]) {
  RowSD o;
  o.s01 = f2(v[0] + v[1], v[1] + v[2]);
  o.s23 = f2(v[2] + v[3], v[3] + v[4]);
  o.d01 = f2(v[1] - v[0], v[2] - v[1]);
  o.d23 = f2(v[3] - v[2], v[4] - v[3]);
  return o;
}


// Two Q1 elements at once.  Inputs: x-sums/differences of u (top st,dt / bottom sb,db) and of nu.
// Outputs: energy pair E and the nodal gradient pairs ga (top-left), gb (top-right),
// gc (bottom-left), gd (bottom-right).  Quadratic part in the half-gradient convention
// q = (1/2) dE/dA, so E = sum A q and g = 2 q.  The source term is not part of the element pair: it
// is linear in u and enters per node (Fem2T::src_share).
template <bool HAS_NU>
__device__ __forceinline__ float2 elem_pair(const K2& k, float2 st, float2 dt, float2 sb, float2 db,
                                            float2 nst, float2 ndt, float2 nsb, float2 ndb,
                                            float2 vw, float2& ga, float2& gb, float2& gc,
                                            float2& gd) {
  const float2 Ae = sub2(sb, st), Ax = add2(dt, db), Axe = sub2(db, dt);
  float2 c0x, c0y, qx, qe, qxe;
  const float2 tAxe = mul2(k.t, Axe);
  if constexpr (HAS_NU) {
    const float2 C0 = add2(nst, nsb), Ce = sub2(nsb, nst), Cx = add2(ndt, ndb);
    c0x = mul2(k.kx, C0);
    c0y = mul2(k.ky, C0);
    const float2 c1x = mul2(k.kxt, Ce), c1y = mul2(k.kyt, Cx);
    qx = fma2(c0x, Ax, mul2(c1x, Axe));
    qe = fma2(c0y, Ae, mul2(c1y, Axe));
    qxe = fma2(add2(c0x, c0y), tAxe, fma2(c1x, Ax, mul2(c1y, Ae)));
  } else {
    // nu == 1: C0 = 4 (times the validity weight of the element), Cx = Ce = 0
    c0x = mul2(k.c0x_const, vw);
    c0y = mul2(k.c0y_const, vw);
    qx = mul2(c0x, Ax);
    qe = mul2(c0y, Ae);
    qxe = mul2(add2(c0x, c0y), tAxe);
  }
  const float2 E = fma2(Ax, qx, fma2(Ae, qe, mul2(Axe, qxe)));
  const float2 gx = add2(qx, qx), ge = add2(qe, qe), gxe = add2(qxe, qxe);
  const float2 n0 = sub2(gx, gxe), n1 = add2(gx, gxe);
  // m0 = -ge, m1 = +ge
  ga = sub2(f2(-ge.x, -ge.y), n0); gb = sub2(n0, ge); gc = sub2(ge, n1); gd = add2(ge, n1);
  return E;
}

// Per-thread state of one masked node row: x-sums / x-differences of u and nu, the 0/1
// "free node" multipliers (0 where a Dirichlet mask fired) and what the source term needs.
struct Row2T {
  RowSD u, n;
  float2 keep01, keep23;
  float2 lb01, lb23;   // FK == 2: -(S c_f) b of the 4 own nodes (their gradient share), and
  float lE;            //          their energy share sum(-(S c_f) b u)
  float2 fx01, fx23;   // FK == 1: -kf (M_x f) of the 4 own nodes (x-stencil of f)
};
// Gradient accumulators of one node row: own nodes 0..3 and the right neighbour's node 0.
struct Acc2T {
  float2 a01, a23;
  float a4;
};

// FK: 0 no source term, 1 nodal source f (interpolated to the Gauss points), 2 `f` is an ASSEMBLED load vector
// b_a = sum_e sum_g w_g N_a(g) f_g (dn_fem_load_vector_f32): the term -c_f sum_a b_a u_a is added per node when its
// row closes -- what the reference's f-at-Gauss-points form (e8_2d_poisson_mms.py:154-175) costs once b exists.
//
// FK == 1 takes the same per-node route.  The element source energy -kf (A0 B0 + t (Ax Bxi + Ae Beta) + t^2 Axe Bxieta)
// is the tensor product of the 1-D element mass M = [[1+t, 1-t], [1-t, 1+t]] in x and in y (A0 = s_x s_y u,
// Ax = d_x s_y u, ...; s s' + t d d' = a^T M b), so the assembled term is -kf u^T (M_y (x) M_x) f: node a's gradient
// share is the separable stencil g_a = -kf (M_y (M_x f))_a and the energy is sum_a u_a g_a.  M_x f is taken when a row
// is loaded (Row2T::fx), the y-combination when the row closes (src_share).  A node on the image's edge has one
// element in that direction, i.e. own weight (1+t): in x a mirrored neighbour (K2::fmir) gives it, in y the weight wy.
template <int NM, bool VF, bool HAS_NU, int FK, bool NUMASK, bool MI = true>
struct Fem2T {
  static constexpr bool HAS_F = (FK == 1), LV = (FK == 2);
  static constexpr bool NODAL = HAS_F || LV;      // a per-node source share (Row2T::lb, lE) enters when a row closes
  static constexpr int NF = 1 + (HAS_NU ? 1 : 0) + (FK ? 1 : 0) + (NUMASK ? 1 : 0) + NM + (VF ? 1 : 0);
  static constexpr int F_U = 0, F_NU = 1, F_F = F_NU + (HAS_NU ? 1 : 0), F_NM = F_F + (FK ? 1 : 0),
                       F_M = F_NM + (NUMASK ? 1 : 0), F_VF = F_M + NM;

  // Read one node row from its ring stage (own 4 nodes + right neighbour of every field), apply
  // the Dirichlet conditions (array order: later masks win) and the nu mask, reduce to x-sums.
  // FK == 1: also the left neighbour of f and the x-stencil of f.
  static __device__ __forceinline__ void load_row(const P2T& p, const float* __restrict__ sp, int fstride,
                                                  bool has_left, bool has_right, Row2T& o) {
    float v[NF][5];
#pragma unroll
    for (int f = 0; f < NF; ++f) {
      const float* q = sp + f * fstride;
      const float4 t = *reinterpret_cast<const float4*>(q);
      const float h = q[4];            // in-bounds of the ring for every thread (padded), masked below
      v[f][0] = t.x; v[f][1] = t.y; v[f][2] = t.z; v[f][3] = t.w; v[f][4] = has_right ? h : 0.f;
    }
    float fl = 0.f;                    // f left of node 0: the ring holds the whole row (x0 = 0: the u field's last word)
    if constexpr (HAS_F) fl = sp[F_F * fstride - 1];
    float ub[5], nb[5], fb[5], kp[4];
#pragma unroll
    for (int e = 0; e < 5; ++e) {
      float u = v[F_U][e];
      bool fx = false;
#pragma unroll
      for (int m = 0; m < NM; ++m) {
        const bool hit = v[F_M + m][e] > 0.5f;
        if constexpr (MI) u = hit ? (VF ? v[F_VF][e] : p.mval[m]) : u;   // MI = false: operator apply, values not substituted
        fx = fx || hit;
      }
      ub[e] = u;
      if (e < 4) kp[e] = fx ? 0.f : 1.f;
      if constexpr (HAS_NU) {
        float n = v[F_NU][e];
        if constexpr (NUMASK) n = (v[F_NM][e] > 0.5f) ? 0.f : n;
        nb[e] = n;
      }
      if constexpr (HAS_F || LV) fb[e] = v[F_F][e];
    }
    o.keep01 = f2(kp[0], kp[1]);
    o.keep23 = f2(kp[2], kp[3]);
    if constexpr (LV) {
      o.lb01 = mul2(p.k2.nkb, f2(fb[0], fb[1]));
      o.lb23 = mul2(p.k2.nkb, f2(fb[2], fb[3]));
      const float2 le = fma2(o.lb01, f2(ub[0], ub[1]), mul2(o.lb23, f2(ub[2], ub[3])));
      o.lE = le.x + le.y;
    }
    if constexpr (HAS_F) {
      // -kf (M_x f): (1-t) per neighbour node, 2(1+t) own.  A row end has one element: (1+t) own, which the
      // mirrored neighbour fmir f gives ((1-t) fmir + 2(1+t) = 1+t) with the interior weights unchanged.
      fl = has_left ? fl : p.k2.fmir.x * fb[0];
      const float fr = has_right ? fb[4] : p.k2.fmir.x * fb[3];
      o.fx01 = fma2(p.k2.nfc, f2(fl + fb[1], fb[0] + fb[2]), mul2(p.k2.nfw, f2(fb[0], fb[1])));
      o.fx23 = fma2(p.k2.nfc, f2(fb[1] + fb[3], fb[2] + fr), mul2(p.k2.nfw, f2(fb[2], fb[3])));
    }
    o.u = row_sd(ub);
    // the last element of a row does not exist: E and g are linear in nu, so zeroing its
    // x-sums/differences for that element removes it (nu == 1 uses the weight vw instead)
    if constexpr (HAS_NU) {
      o.n = row_sd(nb);
      if (!has_right) { o.n.s23.y = 0.f; o.n.d23.y = 0.f; }
    }
  }

  // FK == 1: node row `row` closes between the rows above (x-stencil xa) and below (xb) -- zero where the image
  // ends, and then wy = (1+t) instead of 2(1+t).  Fills row.lb (gradient share) and row.lE (energy share).  The
  // energy share sum_a u_a lb_a is taken from the row's u x-sums / x-differences (u0 = (s0 - d0) / 2, u1 = (s0 + d0) / 2,
  // the same for u2, u3): no register holds the row's u itself until it closes.
  static __device__ __forceinline__ void src_share(const K2& k, float2 xa01, float2 xa23, float2 xb01,
                                                   float2 xb23, float2 wy, Row2T& row) {
    row.lb01 = fma2(k.yc, add2(xa01, xb01), mul2(wy, row.fx01));
    row.lb23 = fma2(k.yc, add2(xa23, xb23), mul2(wy, row.fx23));
    const float2 ls = f2(row.lb01.x + row.lb01.y, row.lb23.x + row.lb23.y);
    const float2 ld = f2(row.lb01.y - row.lb01.x, row.lb23.y - row.lb23.x);
    const float2 le = fma2(f2(row.u.s01.x, row.u.s23.x), ls, mul2(f2(row.u.d01.x, row.u.d23.x), ld));
    row.lE = 0.5f * (le.x + le.y);
  }

  // Element row between `top` and `bot`: adds its gradient to At (top nodes) and WRITES Ab
  // (bottom nodes); returns the row's energy of this lane's 4 elements.
  static __device__ __forceinline__ float elem_row(const K2& k, const Row2T& top, const Row2T& bot,
                                                   float2 vw01, float2 vw23, Acc2T& At, Acc2T& Ab) {
    float2 ga, gb, gc, gd;
    const float2 E0 = elem_pair<HAS_NU>(k, top.u.s01, top.u.d01, bot.u.s01, bot.u.d01,
                                        top.n.s01, top.n.d01, bot.n.s01, bot.n.d01, vw01,
                                        ga, gb, gc, gd);
    At.a01 = add2(At.a01, ga);
    At.a01.y += gb.x; At.a23.x += gb.y;
    Ab.a01 = gc; Ab.a01.y += gd.x;
    const float carry = gd.y;
    const float2 E1 = elem_pair<HAS_NU>(k, top.u.s23, top.u.d23, bot.u.s23, bot.u.d23,
                                        top.n.s23, top.n.d23, bot.n.s23, bot.n.d23, vw23,
                                        ga, gb, gc, gd);
    At.a23 = add2(At.a23, ga);
    At.a23.y += gb.x; At.a4 += gb.y;
    Ab.a23 = gc; Ab.a23.x += carry; Ab.a23.y += gd.x;
    Ab.a4 = gd.y;
    const float2 Es = add2(E0, E1);
    return Es.x + Es.y;
  }
};

// Loss epilogue for the streaming kernels.  Only warp 0 takes part (the other warps retire at once) and
// no CTA waits for a fence or an atomic round trip at its end:
//   * at its START (after pdl_wait) thread 0 of every CTA draws a ticket (draw_start_ticket; the answer is
//     not needed before the epilogue, so its latency hides behind the first tile loads).  The CTA that
//     drew the LAST ticket is the finisher: every other CTA has started by then, so waiting for them
//     cannot deadlock, and it is among the last to finish.
//   * a CTA publishes its partial with ONE 8-byte store whose bit pattern is never zero (+-0.0 is stored
//     as -0.0): the value is its own "ready" flag, so no fence / ticket separates data and flag.
//   * the finisher polls the slots until none is zero (one batched L2 round trip per sweep), sums them in
//     a fixed order (lane-strided, then an xor butterfly: bit-reproducible), and zeroes slots and counter
//     again: the workspace contract (zero on entry, zero on exit) is unchanged.
__device__ __forceinline__ unsigned int draw_start_ticket(const Reduce& r) { return atomicAdd(r.counter, 1u); }

__device__ __forceinline__ long long ld_relaxed_b64(const void* p) {
  long long v;
  asm volatile("ld.relaxed.gpu.global.b64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// NB = slots per lane fetched per sweep (all of them are live registers while the sweep is checked)
template <int NB = 40>
__device__ __forceinline__ void finish_loss_w0(const Reduce& r, double cta_value, unsigned int start_ticket) {
  if (threadIdx.x >= 32) return;
  const int lane = threadIdx.x;
  unsigned fin = 0u;
  if (lane == 0) {
    long long bits = __double_as_longlong(cta_value);
    if ((bits << 1) == 0) bits = (long long)0x8000000000000000ull;      // +-0.0 -> -0.0: never the "empty" pattern
    __stcg(reinterpret_cast<long long*>(r.partials + blockIdx.x), bits);
    fin = (start_ticket == gridDim.x - 1) ? 1u : 0u;
  }
  fin = __shfl_sync(0xffffffffu, fin, 0);
  if (!fin) return;
  const unsigned n = gridDim.x;
  double s = 0.0;
  for (unsigned base = 0; base < n; base += 32 * NB) {   // up to NB independent L2 loads per lane in flight
    long long v[NB];
    bool all;
    do {
      all = true;
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        const unsigned i = base + q * 32 + lane;
        v[q] = (i < n) ? ld_relaxed_b64(r.partials + i) : (long long)0x8000000000000000ull;
        all = all && (v[q] != 0);
      }
      all = __all_sync(0xffffffffu, all);
    } while (!all);
#pragma unroll
    for (int q = 0; q < NB; ++q) {
      const unsigned i = base + q * 32 + lane;
      s += __longlong_as_double(v[q]);                    // out-of-range slots hold -0.0
      if (i < n) __stcg(reinterpret_cast<long long*>(r.partials + i), 0ll);   // self-reset
    }
  }
  s = warp_sum(s) + 0.0;                                  // -0.0 (all partials zero) -> +0.0
  if (r.peer_slots) {      // linked z-slab launch: push the rank total to every rank (NVLink stores), then the flags
    const int want = *r.step + 1;
    if (lane < r.world) {
      double* slots = r.peer_slots[lane];
      *reinterpret_cast<volatile double*>(slots + r.rank) = s;
      __threadfence_system();
      *reinterpret_cast<volatile int*>(reinterpret_cast<int*>(slots + r.world) + r.rank) = want;
    }
    __syncwarp();
    if (lane == 0) *r.step = want;
  }
  if (lane == 0) {
    if (r.loss_out) *r.loss_out = s;
    if (r.loss_f32) *r.loss_f32 = (float)s;
    *r.counter = 0u;   // self-reset: the workspace is ready for the next call
  }
}

// TB = max threads per CTA, MINB = min resident CTAs per SM the register allocation must allow.
template <int NM, bool VF, bool HAS_NU, int FK, bool NUMASK, bool MI, int TB, int MINB>
__global__ void __launch_bounds__(TB, MINB) k_fem2d_tma(const __grid_constant__ P2T p) {
  using F = Fem2T<NM, VF, HAS_NU, FK, NUMASK, MI>;
  constexpr int NF = F::NF;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ double s_red[TB / 32];
  __shared__ unsigned int s_ticket;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const int nx = p.nx, S = p.S;
  const int stage_floats = NF * 2 * nx;                                               // 2 node rows per stage
  float* ring = reinterpret_cast<float*>(smem_raw);                                   // [S][NF][2][nx] (+16 B pad)
  uint64_t* full = reinterpret_cast<uint64_t*>(ring + (size_t)S * stage_floats + 4);  // [S]
  float* seam = reinterpret_cast<float*>(full + S);                                   // [2 parities][2 rows][nw]

  int b, r_begin, r_end;
  if (p.bal_q > 0) {
    const int c = (int)blockIdx.x, hi = p.bal_rem * (p.bal_q + 1);
    int n, ch;
    if (c < hi) { n = p.bal_q + 1; b = c / n; ch = c - b * n; }
    else { n = p.bal_q; const int c2 = c - hi; b = c2 / n; ch = c2 - b * n; b += p.bal_rem; }
    r_begin = (int)((long long)ch * p.ny / n);
    r_end = (int)((long long)(ch + 1) * p.ny / n);
    // every chunk then streams an EVEN number of node rows (its own + the halo rows): whole two-row stages, no
    // half-empty last stage on the CTA's serial chain.  Interior cuts at odd rows do that when ny is even.
    if (!(p.ny & 1)) {
      if (ch > 0) r_begin |= 1;
      if (ch + 1 < n) r_end |= 1;
    }
  } else {
    b = blockIdx.x / p.nchunks;
    const int ch = blockIdx.x - b * p.nchunks;
    r_begin = ch * p.R;
    r_end = min(p.ny, r_begin + p.R);
  }
  const int j_first = max(r_begin - 1, 0), j_last = min(r_end, p.ny - 1);
  const int nrows = j_last - j_first + 1;          // node rows streamed: >= 2
  const int nst = (nrows + 1) >> 1;                // stages streamed (the last may hold one row)

  // ---- producer: thread 0 copies, per stage, two rows of every field (one bulk copy per field).  The source rows
  // of the next stage start where the last stage's ended (stride_y == nx is an eligibility condition of this path):
  // the field addresses are set up once and advance by two rows per stage.
  const uint32_t row_bytes = (uint32_t)(nx * 4);
  const float* src[NF];
#pragma unroll
  for (int f = 0; f < NF; ++f) src[f] = p.fld[f].p + (long long)b * p.fld[f].sb + (long long)j_first * nx;
  int issued = 0, ist = 0;
  auto issue_stage = [&]() {
    if (tid == 0) {
      const uint32_t nr_bytes = (issued + 1 < nst || !(nrows & 1)) ? 2 * row_bytes : row_bytes;
      uint64_t* bar = full + ist;
      float* dst = ring + ist * stage_floats;
      mbar_arrive_expect_tx(bar, (uint32_t)NF * nr_bytes);
#pragma unroll
      for (int f = 0; f < NF; ++f) bulk_g2s(dst + f * 2 * nx, src[f], nr_bytes, bar);
    }
#pragma unroll
    for (int f = 0; f < NF; ++f) src[f] += 2 * nx;
    ++issued;
    ist = (ist + 1 == S) ? 0 : ist + 1;
  };
  if (tid == 0) {
    for (int s = 0; s < S; ++s) mbar_init(full + s, 1);
    fence_mbar_init();
  }
  pdl_wait();            // everything above overlaps the tail of the previous grid in the stream
  {
    const int n0 = min(S, nst);
    for (int q = 0; q < n0; ++q) issue_stage();     // thread 0 only; the others just count
  }
  if (tid == 0) s_ticket = draw_start_ticket(p.red);  // its round trip hides behind the first tile loads
  __syncthreads();                                   // barriers initialised before anyone waits

  const bool act = tid * 4 < nx;
  const int x0 = act ? tid * 4 : 0;          // idle lanes of the last warp shadow lane 0 (results dropped)
  const bool has_right = (x0 + 4) < nx, has_left = x0 > 0;
  const float2 vw01 = f2(1.f, 1.f);
  const float2 vw23 = f2(1.f, has_right ? 1.f : 0.f);
  const K2& k = p.k2;
  // FK == 1: the y-stencil's own weight in the image's top and bottom row, and the x-stencil of the row above the
  // next row to close (zero above row 0)
  const float2 wy_edge = mul2(f2(0.5f), k.yw);
  float2 xc01 = f2(0.f), xc23 = f2(0.f);
  const bool seam_in = (lane == 0) && (warp > 0);

  double acc = 0.0;
  int st = 0;                // stage being consumed
  uint32_t phase = 0;        // its mbarrier parity
  const float* sbase = ring + x0;
  float* gout = p.grad ? p.grad + ((long long)b * p.ny + j_first) * nx + x0 : nullptr;

  // Node row `jr` is complete in A except for the share of the left neighbour: take it from the
  // left lane now (across a warp seam it arrives through shared memory after the barrier).
  auto close_row = [&](const Acc2T& A, const Row2T& row, float4& G) {
    const float fromL = __shfl_up_sync(0xffffffffu, A.a4, 1);
    float2 g01 = A.a01, g23 = A.a23;
    if (lane > 0) g01.x += fromL;
    if constexpr (F::NODAL) { g01 = add2(g01, row.lb01); g23 = add2(g23, row.lb23); }
    g01 = mul2(g01, row.keep01);
    g23 = mul2(g23, row.keep23);
    G = make_float4(g01.x, g01.y, g23.x, g23.y);
  };
  // branch-free: a predicated 16-byte store; the residual form's square sum (RES) or the row's source energy
  // selected into `pend` (added to the fp64 accumulator together with the next stage's energy).  `inr`: the row
  // is owned by this chunk -- a compile-time true everywhere but in the first stage.
  const bool wr = act && (gout != nullptr);
  float pend = 0.f;
  auto store_row = [&](auto res_c, float4 G, float keep0, float seam_v, const int jr, const bool inr, const float le) {
    G.x += seam_in ? seam_v * keep0 : 0.f;
    if (inr && wr) *reinterpret_cast<float4*>(gout + (long long)(jr - j_first) * nx) = G;
    if constexpr (decltype(res_c)::value) {
      const float sq = G.x * G.x + G.y * G.y + G.z * G.z + G.w * G.w;
      pend += (inr && act) ? sq : 0.f;
    } else if constexpr (F::NODAL) {
      pend += (inr && act) ? le : 0.f;     // the row's source energy, once, by its owner
    }
  };

  Row2T rowA, rowB;          // even node rows of the chunk live in A, odd ones in B
  Acc2T accA, accB;
  accA.a01 = accA.a23 = f2(0.f); accA.a4 = 0.f;
  accB = accA;

  // One stage = two node rows.  The body exists three times: the FIRST stage (no element row above its even
  // row, the only place a halo row must not be stored), the steady loop (every check of the general body is a
  // compile-time constant there: one straight-line block per stage between the data wait and the CTA barrier,
  // so the two rows' shared loads, masks and element pairs can be scheduled across each other), and the trailing
  // half stage of a chunk that streams an odd number of rows.  RES (res_c): the loss is the residual form.
  auto stage = [&](auto first_c, auto odd_c, auto res_c, const int q) {
    constexpr bool FIRST = decltype(first_c)::value, HAS_ODD = decltype(odd_c)::value, RES = decltype(res_c)::value;
    mbar_wait(full + st, phase);
    const float* sp = sbase + st * stage_floats;
    const int r0 = 2 * q;                              // even row of this stage (chunk-relative)
    const int par = q & 1;
    float4 G0 = make_float4(0.f, 0.f, 0.f, 0.f), G1 = G0;
    float kp0 = 0.f, kp1 = 0.f, e = 0.f, le0 = 0.f, le1 = 0.f;

    // ---- even row -> A; element row (B above, A below); node row r0-1 (B) closes
    F::load_row(p, sp, 2 * nx, has_left, has_right, rowA);
    if constexpr (!FIRST) {
      const float e0 = F::elem_row(k, rowB, rowA, vw01, vw23, accB, accA);
      e += (j_first + r0 - 1 >= r_begin) ? e0 : 0.f;
      sts_if(lane == 31, seam + (par * 2 + 0) * nw + warp, accB.a4);
      if constexpr (F::HAS_F) {
        F::src_share(k, xc01, xc23, rowA.fx01, rowA.fx23, k.yw, rowB);
        xc01 = rowB.fx01; xc23 = rowB.fx23;
      }
      close_row(accB, rowB, G0);
      kp0 = rowB.keep01.x;
      if constexpr (F::NODAL) le0 = rowB.lE;
    }
    // ---- odd row -> B; element row (A above, B below); node row r0 (A) closes
    if constexpr (HAS_ODD) {
      F::load_row(p, sp + nx, 2 * nx, has_left, has_right, rowB);
      const float e1 = F::elem_row(k, rowA, rowB, vw01, vw23, accA, accB);
      e += (j_first + r0 >= r_begin) ? e1 : 0.f;
      sts_if(lane == 31, seam + (par * 2 + 1) * nw + warp, accA.a4);
      if constexpr (F::HAS_F) {
        // FIRST: row j_first is the image's top row, or a halo row this chunk does not store
        F::src_share(k, xc01, xc23, rowB.fx01, rowB.fx23, FIRST ? wy_edge : k.yw, rowA);
        xc01 = rowA.fx01; xc23 = rowA.fx23;
      }
      close_row(accA, rowA, G1);
      kp1 = rowA.keep01.x;
      if constexpr (F::NODAL) le1 = rowA.lE;
    }
    acc += (double)(((!RES && act) ? e : 0.f) + pend);
    pend = 0.f;
    __syncthreads();      // stage consumed by every thread; seam words of both rows visible
    if (issued < nst) issue_stage();
    ++st;
    if (st == S) { st = 0; phase ^= 1u; }
    // unconditional loads from a valid slot (warp 0 reads its own), selected away where there is no seam
    const int wl = warp > 0 ? warp - 1 : 0;
    const float s0 = seam[(par * 2 + 0) * nw + wl];
    const float s1 = seam[(par * 2 + 1) * nw + wl];
    if constexpr (!FIRST) store_row(res_c, G0, kp0, s0, j_first + r0 - 1, true, le0);
    if constexpr (HAS_ODD) store_row(res_c, G1, kp1, s1, j_first + r0, FIRST ? (j_first >= r_begin) : true, le1);
  };
  // The whole march exists once per loss form (one uniform branch on p.mode): the energy march carries no square
  // sums, the residual march no element energies.
  auto march = [&](auto res_c) {
    const int nfull = nrows >> 1;                        // >= 1: a chunk streams at least two rows
    stage(std::true_type{}, std::true_type{}, res_c, 0);
    for (int q = 1; q < nfull; ++q) stage(std::false_type{}, std::true_type{}, res_c, q);
    if (nrows & 1) stage(std::false_type{}, std::false_type{}, res_c, nfull);

    // ---- last node row of the image: no element row below it; its sum is already complete
    if (r_end == p.ny) {
      const bool lastB = (nrows & 1) == 0;             // the last streamed row is odd -> lives in B
      const Acc2T& A = lastB ? accB : accA;
      Row2T row = lastB ? rowB : rowA;
      const int par = nst & 1;
      if (lane == 31) seam[(par * 2) * nw + warp] = A.a4;
      if constexpr (F::HAS_F) F::src_share(k, xc01, xc23, f2(0.f), f2(0.f), wy_edge, row);
      float4 G;
      close_row(A, row, G);
      __syncthreads();
      const float sv = seam_in ? seam[(par * 2) * nw + warp - 1] : 0.f;
      float le = 0.f;
      if constexpr (F::NODAL) le = row.lE;
      store_row(res_c, G, row.keep01.x, sv, p.ny - 1, true, le);
    }
  };
  if (p.mode != 0) march(std::true_type{});
  else march(std::false_type{});
  acc += (double)pend;

  // all streaming done: the next grid in the stream may start launching behind our epilogue
  // (its own pdl_wait() still holds it until this grid has completed and flushed)
  pdl_trigger();
  acc = warp_sum(acc);
  if (lane == 0) s_red[warp] = acc;
  __syncthreads();
  double cta = 0.0;
  if (tid == 0)
    for (int w = 0; w < nw; ++w) cta += s_red[w];
  finish_loss_w0(p.red, cta, s_ticket);
}

// ---- dispatch (fem2d_tma_dispatch.cu) --------------------------------------------------------
// MK encodes the Dirichlet set: 0..3 scalar-valued masks; 4 = one mask with a nodal value field.
typedef cudaError_t (*launch2t_fn)(const P2T&, dim3, dim3, size_t, cudaStream_t);
typedef int (*occ2t_fn)(int, size_t);
launch2t_fn get_launch2t(int MK, int NU, int F, int NUMASK);
occ2t_fn get_occ2t(int MK, int NU, int F, int NUMASK);

// DN_PDL=0 disables programmatic dependent launch (default on)
inline bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("DN_PDL"); v = (e && *e == '0') ? 0 : 1; }
  return v == 1;
}

constexpr int kMaxDynSmem = 226 * 1024;   // 227 KB per CTA minus the kernels' static shared memory

// One register budget (<= 128 registers, CTAs of up to 512 threads).  A tighter variant
// (<= 96 registers, 10 instead of 8 resident 64-thread CTAs per SM) measured 10% SLOWER on
// 256^2 x 64: more CTAs per wave means shorter row chunks and more seam work (profiles/).
template <int MK, bool HAS_NU, int FK, bool NUMASK>
struct Kern2T {
  // MK 0..3: that many scalar-valued masks; 4: one mask with a value field; 5..7: 1..3 masks whose
  // values are NOT substituted into u (mask_input = 0: the operator v -> mask(K v) of the resmin backward)
  static constexpr int NM = (MK == 4) ? 1 : (MK >= 5 ? MK - 4 : MK);
  static auto get() { return k_fem2d_tma<NM, (MK == 4), HAS_NU, FK, NUMASK, (MK < 5), DN_T2_MAXT, 1>; }
};

template <int MK, bool HAS_NU, int FK, bool NUMASK>
cudaError_t prep2t() {
  // opt in to the full dynamic shared memory once per device
  static bool done[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev >= 0 && dev < 64 && done[dev]) return cudaSuccess;
  e = cudaFuncSetAttribute(Kern2T<MK, HAS_NU, FK, NUMASK>::get(),
                           cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem);
  if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev] = true;
  return e;
}

template <int MK, bool HAS_NU, int FK, bool NUMASK>
cudaError_t launch2t(const P2T& p, dim3 grid, dim3 block, size_t smem, cudaStream_t s) {
  cudaError_t e = prep2t<MK, HAS_NU, FK, NUMASK>();
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  if (pdl_enabled()) { cfg.attrs = at; cfg.numAttrs = 1; }
  return cudaLaunchKernelEx(&cfg, Kern2T<MK, HAS_NU, FK, NUMASK>::get(), p);
}

// resident CTAs per SM for a block of `threads` threads and `smem` bytes of dynamic shared memory
template <int MK, bool HAS_NU, int FK, bool NUMASK>
int occ2t(int threads, size_t smem) {
  if (prep2t<MK, HAS_NU, FK, NUMASK>() != cudaSuccess) return 0;
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, Kern2T<MK, HAS_NU, FK, NUMASK>::get(),
                                                    threads, smem) != cudaSuccess)
    return 0;
  return n;
}

}  // namespace dn
