// gp_eval.cu -- see gp_eval.cuh.
//
// Un-fused gauss_pt_evaluation* (DiffNet/DiffNetFEM.py:7-18,143-156) and its adjoint for user loss() bodies that
// are not one of the fused forms.  Both are pure streaming operators: the forward writes ngp values per element
// and table (write-bound: 4 B read, 4 ngp B written per node), the adjoint reads them back (read-bound).
//
//   * A thread owns one element column (forward) / node column (adjoint) and MARCHES in y: the node row shared by
//     two element rows is loaded once and kept in registers, element rows contribute to the node rows above and
//     below through a register carry.  Lanes run along x: every load and store instruction of a warp covers 32
//     consecutive floats.  No integer division in the loop (the grid is (x chunks, y chunks, plane * batch)).
//   * Several tables (N, d/dx, d/dy, d/dz) are requested in ONE call (GpMulti).  The kernels can evaluate them in one
//     pass over the input, but the op is write-bound and one table per pass measured faster (launch_gp_eval).
//   * Outputs are write-once: streaming stores (st.global.cs), so they do not evict the inputs from L2.
//   * Adjoint: the x-neighbour's share travels by one warp shuffle per node row; a warp covers 31 node columns
//     plus one provider lane on its left, so there are no shared-memory seams and no atomics (deterministic).
#include <cstdlib>

#include "gp_eval.cuh"

namespace dn {

constexpr int kGpThreads = 128;

// ---- forward ---------------------------------------------------------------------------------------------------
// out_w[b, G, (k,) j, i] = sum_a T_w[G][a] * in[b, (k+kb,) j+jb, i+ib],  G = (kg*n + jg)*n + ig.
template <int NSD, int NG>
__global__ void __launch_bounds__(kGpThreads) k_gp_eval(Field in, int nx, int ny, int nz, GpMulti m, int RY) {
  constexpr int NZ = (NSD == 3) ? 2 : 1;
  constexpr int NGP = (NSD == 3) ? NG * NG * NG : NG * NG;
  const int nelx = nx - 1, nely = ny - 1, nelz = (NSD == 3) ? nz - 1 : 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nelx) return;
  const int j0 = blockIdx.y * RY, j1 = min(nely, j0 + RY);
  const int k = (NSD == 3) ? (int)(blockIdx.z % nelz) : 0;
  const int b = (NSD == 3) ? (int)(blockIdx.z / nelz) : (int)blockIdx.z;
  const long long nel = (long long)nelx * nely * nelz;
  const float* base = in.p + (long long)b * in.sb + (NSD == 3 ? (long long)k * in.sz : 0) + (long long)j0 * in.sy + i;
  const long long obase = (long long)b * NGP * nel + ((long long)k * nely + j0) * nelx + i;

  // node rows j (jb = 0) and j + 1 (jb = 1) of the element row in flight, plus row j + 2 prefetched one
  // iteration ahead: its loads are issued before the arithmetic and the stores of element row j
  float v[NZ][2][2];       // [kb][jb][ib]
  float nx2[NZ][2];        // row j + 2
#pragma unroll
  for (int kb = 0; kb < NZ; ++kb) {
    const float* q = base + (long long)kb * in.sz;
    v[kb][0][0] = __ldg(q);
    v[kb][0][1] = __ldg(q + 1);
    v[kb][1][0] = __ldg(q + in.sy);
    v[kb][1][1] = __ldg(q + in.sy + 1);
  }
  base += 2 * in.sy;
  for (int j = j0; j < j1; ++j) {
    const bool more = (j + 2 <= nely);                    // node row j + 2 exists (it is row nely at most)
#pragma unroll
    for (int kb = 0; kb < NZ; ++kb) {
      const float* q = base + (long long)kb * in.sz;
      nx2[kb][0] = more ? __ldg(q) : 0.f;
      nx2[kb][1] = more ? __ldg(q + 1) : 0.f;
    }
    base += in.sy;
    const long long orow = obase + (long long)(j - j0) * nelx;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      if (w >= m.nw) break;
      const GpTables& tb = m.tb[w];
      float* o = m.out[w] + orow;
#pragma unroll
      for (int kg = 0; kg < (NSD == 3 ? NG : 1); ++kg) {
        float wz[2][2];
#pragma unroll
        for (int jb = 0; jb < 2; ++jb)
#pragma unroll
          for (int ib = 0; ib < 2; ++ib)
            wz[jb][ib] = (NSD == 3) ? tb.c[2][kg][0] * v[0][jb][ib] + tb.c[2][kg][1] * v[NZ - 1][jb][ib] : v[0][jb][ib];
#pragma unroll
        for (int jg = 0; jg < NG; ++jg) {
          const float r0 = tb.c[1][jg][0] * wz[0][0] + tb.c[1][jg][1] * wz[1][0];
          const float r1 = tb.c[1][jg][0] * wz[0][1] + tb.c[1][jg][1] * wz[1][1];
#pragma unroll
          for (int ig = 0; ig < NG; ++ig) {
            const int G = (kg * NG + jg) * NG + ig;
            __stcs(o + (long long)G * nel, tb.c[0][ig][0] * r0 + tb.c[0][ig][1] * r1);
          }
        }
      }
    }
#pragma unroll
    for (int kb = 0; kb < NZ; ++kb) {
      v[kb][0][0] = v[kb][1][0]; v[kb][0][1] = v[kb][1][1];
      v[kb][1][0] = nx2[kb][0];  v[kb][1][1] = nx2[kb][1];
    }
  }
}

// ---- adjoint ---------------------------------------------------------------------------------------------------
// gin[b, node] = sum_w sum over the elements e around the node and all Gauss points G of
//                T_w[G][a(node in e)] * gout_w[b, G, e]          (gather form: no atomics, deterministic).
// Lane l of a warp works on element column e = xw - 1 + l and (for l >= 1) stores node column x = e.
// 3-D: grid z = (sample, node plane z0 + 0 .. nzl - 1) of this launch's slice.
template <int NSD, int NG>
__global__ void __launch_bounds__(kGpThreads) k_gp_eval_adj(GpMultiAdj m, int nx, int ny, int nz, int RY,
                                                            float* __restrict__ gin, int z0, int nzl) {
  constexpr int NZ = (NSD == 3) ? 2 : 1;
  constexpr int NGP = (NSD == 3) ? NG * NG * NG : NG * NG;
  const int nelx = nx - 1, nely = ny - 1, nelz = (NSD == 3) ? nz - 1 : 1;
  const int nzz = (NSD == 3) ? nz : 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int xw = (blockIdx.x * (blockDim.x >> 5) + warp) * 31;          // first node column of this warp
  if (xw >= nx) return;                                                  // warp-uniform
  const int e = xw - 1 + lane;                                           // element column of this lane
  const bool ev = (e >= 0) && (e < nelx);
  const int x = e;                                                       // node column stored by lanes >= 1
  const bool sv = (lane >= 1) && (x < nx);
  const int y0 = blockIdx.y * RY, y1 = min(ny, y0 + RY);                 // node rows [y0, y1)
  const int z = (NSD == 3) ? z0 + (int)(blockIdx.z % nzl) : 0;
  const int b = (NSD == 3) ? (int)(blockIdx.z / nzl) : (int)blockIdx.z;
  const long long nel = (long long)nelx * nely * nelz;
  const long long gb = (long long)b * NGP * nel + (ev ? e : 0);
  float* orow = gin + (((long long)b * nzz + z) * ny + y0) * nx + (sv ? x : 0);

  // byte offset of (b, G = 0, layer z, element row ej, column e) inside a cotangent tensor: advanced by one element
  // row per iteration (recomputing it from (b, ej) cost 45 integer instructions per row -- more than the arithmetic)
  const long long rowb = 4LL * nelx, layerb = rowb * nely, gstepb = 4 * nel;
  long long offb = 4 * gb + ((long long)(NSD == 3 ? z : 0) * nely + (y0 - 1)) * rowb;
  float carry = 0.f;                      // contribution of element row ej - 1 to node row ej (jb = 1), own + left share
  for (int ej = y0 - 1; ej < y1; ++ej, offb += rowb) {
    // Q[jb][ib]: this element column's contribution (both layers around plane z, all tables) to its node
    // row jb (0: row ej, 1: row ej + 1) and node column ib (0: x = e, 1: x = e + 1)
    float Q[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    if (ev && ej >= 0 && ej < nely) {
#pragma unroll
      for (int kb = 0; kb < NZ; ++kb) {
        const int ek = z - kb;
        if (NSD == 3 && (ek < 0 || ek >= nelz)) continue;
        const long long ob = offb - kb * layerb;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          if (w >= m.nw) break;
          const GpTables& tb = m.tb[w];
          const char* ge = reinterpret_cast<const char*>(m.gout[w]) + ob;
#pragma unroll
          for (int kg = 0; kg < (NSD == 3 ? NG : 1); ++kg) {
            const float cz = (NSD == 3) ? tb.c[2][kg][kb] : 1.f;
#pragma unroll
            for (int jg = 0; jg < NG; ++jg) {
              float s0 = 0.f, s1 = 0.f;
#pragma unroll
              for (int ig = 0; ig < NG; ++ig) {
                const float gv = __ldg(reinterpret_cast<const float*>(ge + ((kg * NG + jg) * NG + ig) * gstepb));
                s0 += tb.c[0][ig][0] * gv;
                s1 += tb.c[0][ig][1] * gv;
              }
              const float c0 = cz * tb.c[1][jg][0], c1 = cz * tb.c[1][jg][1];
              Q[0][0] += c0 * s0; Q[0][1] += c0 * s1;
              Q[1][0] += c1 * s0; Q[1][1] += c1 * s1;
            }
          }
        }
      }
    }
    // node (ej, x): own element's (jb = 0, ib = 0) + left element's (jb = 0, ib = 1) + the carry of row ej - 1
    const float l0 = __shfl_up_sync(0xffffffffu, Q[0][1], 1);
    const float l1 = __shfl_up_sync(0xffffffffu, Q[1][1], 1);
    if (ej >= y0) {
      if (sv) __stcs(orow, carry + Q[0][0] + l0);
      orow += nx;
    }
    carry = Q[1][0] + l1;
  }
}

// ---- 3-D adjoint, z-marching --------------------------------------------------------------------------------------
// The y-march above visits every element layer twice in 3-D (once per node plane it touches: 16 loads and two
// passes of the table products per node; ncu: 491 thread instructions per node, issue-bound at 0.24 of the HBM
// peak).  Here a thread owns ONE element column (e, ej) and marches UP in z: each element's ngp^3 values are loaded
// once, reduced by the separable x-, y-, z-stages to the 8 corner shares Q[kb][jb][ib] (48 FMAs per table for
// ngp = 2), and the shares meet at the nodes through
//   z: a register carry (the kb = 1 shares of layer ek wait one iteration for plane ek + 1),
//   x, y: one shared-memory exchange per layer (three 8-byte words per thread: the shares for the right, lower and
//         lower-right neighbour threads; double-buffered, ONE __syncthreads per layer).
// A CTA is LXW lanes (x) by kAdjR rows (y).  Its thread (lx, r) stores node (x = e, y = ej); in the first tile of
// each direction every thread stores (node 0 has no element on its left / above it), later tiles overlap their
// predecessor by one provider lane / row.  z-chunks re-run the layer below their first plane for the carry.
constexpr int kAdjR = 8;

// keep a loop invariant in a register (ptxas otherwise re-derives strides from the kernel parameters with a chain of
// integer multiplies in every iteration: 75 of the 220 instructions per layer of the first version)
__device__ __forceinline__ long long pinned(long long v) {
  asm volatile("" : "+l"(v));
  return v;
}

template <int NG>
__global__ void __launch_bounds__(64 * kAdjR) k_gp_eval_adj3(GpMultiAdj m, int nx, int ny, int nz, int ZC, int ntx,
                                                             int nty, float* __restrict__ gin) {
  constexpr int NGP = NG * NG * NG;
  extern __shared__ float2 xch[];                       // [2 buffers][3 kinds][kAdjR][LXW]
  const int LXW = blockDim.x / kAdjR;
  const int lx = threadIdx.x % LXW, r = threadIdx.x / LXW;
  const int nelx = nx - 1, nely = ny - 1, nelz = nz - 1;
  int w_ = blockIdx.x;
  const int tx = w_ % ntx; w_ /= ntx;
  const int ty = w_ % nty; w_ /= nty;
  const int nzc = (nz + ZC - 1) / ZC;
  const int zc = w_ % nzc;
  const int b = w_ / nzc;
  const int e = (tx == 0) ? lx : LXW + (tx - 1) * (LXW - 1) - 1 + lx;        // element column == node column stored
  const int ej = (ty == 0) ? r : kAdjR + (ty - 1) * (kAdjR - 1) - 1 + r;     // element row == node row stored
  const bool st = (tx == 0 || lx >= 1) && e < nx && (ty == 0 || r >= 1) && ej < ny;
  const bool ev = e < nelx && ej < nely;
  const bool hasL = lx > 0, hasU = r > 0;
  const int z0 = zc * ZC, z1 = min(nz, z0 + ZC);
  const long long nel = (long long)nelx * nely * nelz;
  const int ek0 = max(z0 - 1, 0);
  // byte strides / offsets (NGP * nel < 2^31 elements: checked by the launcher)
  const long long gsb = pinned(4 * nel);                                     // between Gauss points
  const long long layerb = pinned(4LL * nelx * nely);                        // between element layers
  const long long planeb = pinned(4LL * ny * nx);                            // between node planes
  long long offb = 4 * ((long long)b * NGP * nel + (long long)ek0 * nelx * nely + (ev ? ej * nelx + e : 0));
  const char* p0 = reinterpret_cast<const char*>(m.gout[0]) + offb;          // table 0, layer ek, this element column
  char* out = reinterpret_cast<char*>(gin + (((long long)b * nz + z0) * ny + (st ? ej : 0)) * nx + (st ? e : 0));
  const int kind = kAdjR * LXW;
  float2* cur = xch + (r * LXW + lx) + (ek0 & 1) * 3 * kind;                 // this thread's slot in the layer's buffer
  int flip = (ek0 & 1) ? -3 * kind : 3 * kind;                               // to the other buffer

  float g[NG == 2 ? NGP : 1];                           // table 0 of the next layer (ngp = 2), loaded one layer ahead
  if constexpr (NG == 2) {
    const bool v0 = ev && ek0 < nelz;
    const char* a = p0;
#pragma unroll
    for (int G = 0; G < NGP; ++G, a += gsb) g[G] = v0 ? __ldg(reinterpret_cast<const float*>(a)) : 0.f;
  }
  float carry = 0.f;
  for (int ek = ek0; ek < z1; ++ek) {
    float Q[2][2][2] = {{{0.f, 0.f}, {0.f, 0.f}}, {{0.f, 0.f}, {0.f, 0.f}}};
    const bool lv = ev && ek < nelz;                    // the top plane of the domain has no layer above it
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      if (w >= m.nw) break;
      const GpTables& tb = m.tb[w];
      const char* aw = reinterpret_cast<const char*>(m.gout[w]) + offb;
      float t[NG][2][2];                                // [kg][jb][ib]: x- and y-stages done
#pragma unroll
      for (int kg = 0; kg < NG; ++kg) {
        t[kg][0][0] = t[kg][0][1] = t[kg][1][0] = t[kg][1][1] = 0.f;
#pragma unroll
        for (int jg = 0; jg < NG; ++jg) {
          float s0 = 0.f, s1 = 0.f;
#pragma unroll
          for (int ig = 0; ig < NG; ++ig) {
            const int G = (kg * NG + jg) * NG + ig;
            float gv;
            if (NG == 2 && w == 0) gv = g[NG == 2 ? G : 0];
            else gv = lv ? __ldg(reinterpret_cast<const float*>(aw + G * gsb)) : 0.f;
            s0 = fmaf(tb.c[0][ig][0], gv, s0);
            s1 = fmaf(tb.c[0][ig][1], gv, s1);
          }
          t[kg][0][0] = fmaf(tb.c[1][jg][0], s0, t[kg][0][0]); t[kg][0][1] = fmaf(tb.c[1][jg][0], s1, t[kg][0][1]);
          t[kg][1][0] = fmaf(tb.c[1][jg][1], s0, t[kg][1][0]); t[kg][1][1] = fmaf(tb.c[1][jg][1], s1, t[kg][1][1]);
        }
      }
#pragma unroll
      for (int kg = 0; kg < NG; ++kg)
#pragma unroll
        for (int kb = 0; kb < 2; ++kb)
#pragma unroll
          for (int jb = 0; jb < 2; ++jb)
#pragma unroll
            for (int ib = 0; ib < 2; ++ib) Q[kb][jb][ib] = fmaf(tb.c[2][kg][kb], t[kg][jb][ib], Q[kb][jb][ib]);
    }
    p0 += layerb;
    offb += layerb;
    if constexpr (NG == 2) {                            // next layer's loads fly during the exchange
      const bool nv = ev && ek + 1 < nelz && ek + 1 < z1;
      const char* a = p0;
#pragma unroll
      for (int G = 0; G < NGP; ++G, a += gsb) g[G] = nv ? __ldg(reinterpret_cast<const float*>(a)) : 0.f;
    }
    cur[0] = make_float2(Q[0][0][1], Q[1][0][1]);                    // for the right neighbour (same row)
    cur[kind] = make_float2(Q[0][1][0], Q[1][1][0]);                 // for the thread below (same column)
    cur[2 * kind] = make_float2(Q[0][1][1], Q[1][1][1]);             // for the thread below-right
    __syncthreads();
    const float2 zero = make_float2(0.f, 0.f);
    const float2 fl = hasL ? cur[-1] : zero;
    const float2 fu = hasU ? cur[kind - LXW] : zero;
    const float2 ful = (hasL && hasU) ? cur[2 * kind - LXW - 1] : zero;
    cur += flip;
    flip = -flip;
    const float n0 = Q[0][0][0] + fl.x + (fu.x + ful.x);             // plane ek: complete with the carry
    const float n1 = Q[1][0][0] + fl.y + (fu.y + ful.y);             // plane ek + 1: waits for the next layer
    if (ek >= z0) {
      if (st) __stcs(reinterpret_cast<float*>(out), carry + n0);
      out += planeb;
    }
    carry = n1;
  }
}

__global__ void __launch_bounds__(256) k_scale(float* __restrict__ x, size_t n,
                                               const float* __restrict__ factor) {
  const float f = __ldg(factor);
  if (f == 1.0f) return;   // loss.backward() with the default grad_output: nothing to do
  const size_t n4 = (((uintptr_t)x % 16) == 0) ? n / 4 : 0;
  float4* x4 = reinterpret_cast<float4*>(x);
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 v = x4[i];
    v.x *= f; v.y *= f; v.z *= f; v.w *= f;
    x4[i] = v;
  }
  for (size_t i = n4 * 4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += stride)
    x[i] *= f;
}

static int sm_count() {
  static int sms[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!sms[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n < 1) n = 148;
    sms[dev] = n;
  }
  return sms[dev];
}

// Rows per chunk: long enough that the re-read halo row is cheap (1/RY), short enough that the grid has
// several CTAs per SM slot.
static int rows_per_chunk(long long columns_ctas, int rows, int dflt_per_sm = 32) {
  // these kernels are latency-bound at low occupancy (ncu: 0.54 waves, long_scoreboard 9 per issue with
  // 8 CTAs per SM in the grid): fill the machine -- 16 resident 128-thread CTAs per SM, two waves of them
  const char* ev = getenv("DN_GP_CTAS_PER_SM");
  const int per_sm = (ev && atoi(ev) > 0) ? atoi(ev) : dflt_per_sm;
  const long long want = (long long)per_sm * sm_count();   // CTAs in the grid
  long long chunks = (want + columns_ctas - 1) / columns_ctas;
  if (chunks < 1) chunks = 1;
  int ry = (int)((rows + chunks - 1) / chunks);
  if (ry < 4) ry = 4;
  if (ry > rows) ry = rows;
  return ry < 1 ? 1 : ry;
}

template <int NSD>
static cudaError_t launch_fwd(Field in, int B, int nx, int ny, int nz, GpMulti m, cudaStream_t s) {
  const int nelx = nx - 1, nely = ny - 1, nelz = (NSD == 3) ? nz - 1 : 1;
  const int NG = m.tb[0].n;
  const long long per_b = (long long)(NSD == 3 ? NG * NG * NG : NG * NG) * nelx * nely * nelz;
  const int threads = nelx >= kGpThreads ? kGpThreads : ((nelx + 31) / 32) * 32;
  const int gx = (nelx + threads - 1) / threads;
  const int bmax = 65535 / nelz;                       // gridDim.z = batch slice * element layers
  if (bmax < 1) return cudaErrorInvalidConfiguration;
  for (int b0 = 0; b0 < B; b0 += bmax) {
    const int nb = (B - b0 < bmax) ? B - b0 : bmax;
    const long long gz = (long long)nb * nelz;
    const int RY = rows_per_chunk((long long)gx * gz, nely, NSD == 3 ? 64 : 32);   // measured: 3-D 37.7 -> 35.6 us at 64
    dim3 grid(gx, (nely + RY - 1) / RY, (unsigned)gz);
    switch (NG) {
      case 2: k_gp_eval<NSD, 2><<<grid, threads, 0, s>>>(in, nx, ny, nz, m, RY); break;
      case 3: k_gp_eval<NSD, 3><<<grid, threads, 0, s>>>(in, nx, ny, nz, m, RY); break;
      case 4: k_gp_eval<NSD, 4><<<grid, threads, 0, s>>>(in, nx, ny, nz, m, RY); break;
      default: return cudaErrorInvalidValue;
    }
    in.p += (long long)nb * in.sb;
    for (int w = 0; w < m.nw; ++w) m.out[w] += (long long)nb * per_b;
  }
  return cudaGetLastError();
}

cudaError_t launch_gp_eval(Field in, int B, int nx, int ny, int nz, int nsd, const GpMulti& m, cudaStream_t s) {
  // Tables per pass over the input (DN_GP_TABLES_PER_PASS, default 1).  The forward is WRITE-bound (4 B read against
  // 4 ngp B written per node and table), so sharing the read buys little, and a pass that writes 12-32 output streams
  // per thread runs at a lower fraction of the peak: measured 256^2 x 64, 3 tables: 70.4 / 65.6 / 61.7 us with
  // 4 / 2 / 1 tables per pass; 64^3 x 16, 4 tables: 204.7 / 164.8 / 136.1 us.
  if (nsd == 3 && nz - 1 > 65535) {
    // more element layers than grid z holds (launch_fwd puts samples x layers there): the general-basis kernel, a
    // flat grid-stride loop, evaluates the Q1 tables one at a time
    for (int w = 0; w < m.nw; ++w) {
      const int ng = m.tb[w].n;
      float fac[3 * 4 * 2];
      for (int d = 0; d < 3; ++d)
        for (int g = 0; g < ng; ++g)
          for (int a = 0; a < 2; ++a) fac[(d * ng + g) * 2 + a] = m.tb[w].c[d][g][a];
      int bad = 0;
      const cudaError_t e = launch_gp_eval_general(in, B, 3, nx, ny, nz, 2, ng, fac, m.out[w], s, &bad);
      if (e != cudaSuccess) return e;
      if (bad) return cudaErrorInvalidValue;
    }
    return cudaSuccess;
  }
  const char* ev = getenv("DN_GP_TABLES_PER_PASS");
  int per = (ev && atoi(ev) > 0) ? atoi(ev) : 1;
  for (int w0 = 0; w0 < m.nw; w0 += per) {
    GpMulti part;
    part.nw = (m.nw - w0 < per) ? m.nw - w0 : per;
    for (int w = 0; w < part.nw; ++w) { part.tb[w] = m.tb[w0 + w]; part.out[w] = m.out[w0 + w]; }
    cudaError_t e = nsd == 2 ? launch_fwd<2>(in, B, nx, ny, 1, part, s) : launch_fwd<3>(in, B, nx, ny, nz, part, s);
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// z-marching 3-D adjoint; false: not applicable (the y-march takes the call)
static bool launch_adj3(int B, int nx, int ny, int nz, const GpMultiAdj& m, float* gin, cudaStream_t s, cudaError_t* err) {
  const int NG = m.tb[0].n;
  const long long nel = (long long)(nx - 1) * (ny - 1) * (nz - 1);
  if (env_int("DN_GP_ADJ3", 1) == 0 || NG * NG * NG * nel >= (1LL << 31)) return false;
  const int LXW = nx <= 32 ? 32 : 64;
  const int ntx = nx <= LXW ? 1 : 1 + (nx - LXW + LXW - 2) / (LXW - 1);
  const int nty = ny <= kAdjR ? 1 : 1 + (ny - kAdjR + kAdjR - 2) / (kAdjR - 1);
  // z chunks: a CTA costs (ZC + 1 layers + a prologue worth ~3 layers) and the grid runs in ceil(grid / slots) waves.
  // Measured at 64^3 x 16 (144 tiles, 444 slots): ZC = 22 (432 CTAs, one full wave) 37.8 us, 11 (1.95 waves) 39.3,
  // 32 (0.65) 41.9, 8 (2.59) 42.8, 16 (1.30) 43.8 -- the order of this cost.
  const long long tiles = (long long)B * ntx * nty;
  const size_t smem = (size_t)2 * 3 * kAdjR * LXW * sizeof(float2);
  static int occ_cache[64][3][2] = {};                 // [device][NG - 2][LXW == 64]
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); dev = 0; }
  if (NG < 2 || NG > 4) return false;
  int& per_sm = occ_cache[dev][NG - 2][LXW == 64];
  cudaError_t oe = cudaSuccess;
  if (per_sm < 1) switch (NG) {
    case 2: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gp_eval_adj3<2>, LXW * kAdjR, smem); break;
    case 3: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gp_eval_adj3<3>, LXW * kAdjR, smem); break;
    case 4: oe = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_gp_eval_adj3<4>, LXW * kAdjR, smem); break;
    default: return false;
  }
  if (oe != cudaSuccess || per_sm < 1) { cudaGetLastError(); per_sm = 1; }
  const long long slots = (long long)per_sm * sm_count();
  int ZC = nz;
  long long best = -1;
  for (int nzc = 1; nzc <= (nz + 3) / 4; ++nzc) {
    const int zc = (nz + nzc - 1) / nzc;
    const long long grid = tiles * ((nz + zc - 1) / zc);
    const long long cost = ((grid + slots - 1) / slots) * (zc + 4);
    if (best < 0 || cost < best) { best = cost; ZC = zc; }
  }
  ZC = env_int("DN_GP_ADJ3_ZC", ZC);
  if (ZC < 1) ZC = 1;
  if (ZC > nz) ZC = nz;
  const long long grid = tiles * ((nz + ZC - 1) / ZC);
  if (grid > 0x7fffffffLL) return false;
  const dim3 g((unsigned)grid), blk(LXW * kAdjR);
  switch (NG) {
    case 2: k_gp_eval_adj3<2><<<g, blk, smem, s>>>(m, nx, ny, nz, ZC, ntx, nty, gin); break;
    case 3: k_gp_eval_adj3<3><<<g, blk, smem, s>>>(m, nx, ny, nz, ZC, ntx, nty, gin); break;
    case 4: k_gp_eval_adj3<4><<<g, blk, smem, s>>>(m, nx, ny, nz, ZC, ntx, nty, gin); break;
    default: return false;
  }
  *err = cudaGetLastError();
  return true;
}

template <int NSD>
static cudaError_t launch_adj(int B, int nx, int ny, int nz, GpMultiAdj m, float* gin, cudaStream_t s) {
  if (NSD == 3) {
    cudaError_t err = cudaSuccess;
    if (launch_adj3(B, nx, ny, nz, m, gin, s, &err)) return err;
  }
  const int nzz = (NSD == 3) ? nz : 1;
  const int nelx = nx - 1, nely = ny - 1, nelz = (NSD == 3) ? nz - 1 : 1;
  const int NG = m.tb[0].n;
  const long long per_b = (long long)(NSD == 3 ? NG * NG * NG : NG * NG) * nelx * nely * nelz;
  const int warps_needed = (nx + 30) / 31;
  const int wpc = warps_needed >= kGpThreads / 32 ? kGpThreads / 32 : warps_needed;
  const int gx = (warps_needed + wpc - 1) / wpc;
  // gridDim.z = batch slice * node planes (<= 65535): a mesh of more planes runs one sample and a slice of its planes
  // per launch
  const int zs = nzz < 65535 ? nzz : 65535;
  const int bmax = 65535 / zs;
  for (int b0 = 0; b0 < B; b0 += bmax) {
    const int nb = (B - b0 < bmax) ? B - b0 : bmax;
    for (int z0 = 0; z0 < nzz; z0 += zs) {
      const int nzl = (nzz - z0 < zs) ? nzz - z0 : zs;
      const long long gz = (long long)nb * nzl;
      const int RY = rows_per_chunk((long long)gx * gz, ny);
      dim3 grid(gx, (ny + RY - 1) / RY, (unsigned)gz);
      switch (NG) {
        case 2: k_gp_eval_adj<NSD, 2><<<grid, wpc * 32, 0, s>>>(m, nx, ny, nz, RY, gin, z0, nzl); break;
        case 3: k_gp_eval_adj<NSD, 3><<<grid, wpc * 32, 0, s>>>(m, nx, ny, nz, RY, gin, z0, nzl); break;
        case 4: k_gp_eval_adj<NSD, 4><<<grid, wpc * 32, 0, s>>>(m, nx, ny, nz, RY, gin, z0, nzl); break;
        default: return cudaErrorInvalidValue;
      }
    }
    gin += (long long)nb * nzz * ny * nx;
    for (int w = 0; w < m.nw; ++w) m.gout[w] += (long long)nb * per_b;
  }
  return cudaGetLastError();
}

cudaError_t launch_gp_eval_adj(int B, int nx, int ny, int nz, int nsd, const GpMultiAdj& m, float* gin,
                               cudaStream_t s) {
  return nsd == 2 ? launch_adj<2>(B, nx, ny, 1, m, gin, s) : launch_adj<3>(B, nx, ny, nz, m, gin, s);
}

cudaError_t launch_scale(float* x, size_t n, const float* factor_dev, cudaStream_t s) {
  long long g = ((long long)(n + 3) / 4 + 255) / 256;
  const long long cap = 16LL * sm_count();
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  k_scale<<<(int)g, 256, 0, s>>>(x, n, factor_dev);
  return cudaGetLastError();
}

// x[b, :] *= factors[b]: blockIdx.y walks the samples (b = blockIdx.y, + gridDim.y, ...), and a CTA reads the factor
// of each sample it scales once; 16-byte accesses when the sample's row is aligned (n % 4 == 0 and x aligned), else
// scalar ones.
__global__ void __launch_bounds__(256) k_scale_per_sample(float* __restrict__ x, int batch, size_t n,
                                                          const float* __restrict__ factors) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (int b = blockIdx.y; b < batch; b += gridDim.y) {
    const float f = __ldg(factors + b);
    float* xb = x + (size_t)b * n;
    const size_t n4 = (((uintptr_t)xb % 16) == 0) ? n / 4 : 0;
    float4* x4 = reinterpret_cast<float4*>(xb);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += stride) {
      float4 v = x4[i];
      v.x *= f; v.y *= f; v.z *= f; v.w *= f;
      x4[i] = v;
    }
    for (size_t i = n4 * 4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += stride)
      xb[i] *= f;
  }
}

cudaError_t launch_scale_per_sample(float* x, int batch, size_t n, const float* factors_dev, cudaStream_t s) {
  long long g = ((long long)(n + 3) / 4 + 255) / 256;
  long long cap = 16LL * sm_count() / batch;          // ~16 CTAs per SM over the whole launch
  if (cap < 1) cap = 1;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  const int gy = batch < 65535 ? batch : 65535;       // the grid's y limit: larger batches loop in the kernel
  k_scale_per_sample<<<dim3((unsigned)g, (unsigned)gy), 256, 0, s>>>(x, batch, n, factors_dev);
  return cudaGetLastError();
}

}  // namespace dn

// ---- general basis / rule / dimension ---------------------------------------------------------------------------
// gauss_pt_eval for any tensor-product Lagrange basis (nbf_1d = degree + 1 nodes per direction, element stride
// nbf_1d - 1: DiffNetFEM.py:7-18 with stride = nbf_1d - 1, :66-126 for the degree 2 / 3 bases) and for the 1-D
// "surface" stencils of a 2-D mesh (gauss_pt_evaluation_surf, :146-147, 244-269: nsd - 1 = 1).  The caller passes
// the 1-D factors f[d][g][b] (basis value, or derivative * 2/h for the differentiated direction): the kernels know
// nothing about the basis.  One thread per element (forward) / node (adjoint, gather form: deterministic).
// These are the rarely used corners of the operator family (no BASELINE config uses them): simple, not tuned.
namespace dn {

struct GpGeneral {
  int nsd, nb, ng;            // dimensions, nodes per direction per element, Gauss points per direction
  int n[3], nel[3];           // nodes / elements per direction, index 0 = x (innermost)
  float f[3][4][4];           // [d][g][b]
};

__global__ void __launch_bounds__(128) k_gp_eval_general(Field in, int B, GpGeneral q, float* __restrict__ out) {
  const int nb = q.nb, ng = q.ng, nsd = q.nsd;
  const long long nel = (long long)q.nel[0] * q.nel[1] * q.nel[2];
  const long long total = nel * B;
  const int ngp = (nsd == 3) ? ng * ng * ng : (nsd == 2 ? ng * ng : ng);
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ei = (int)(idx % q.nel[0]);
    long long r = idx / q.nel[0];
    const int ej = (int)(r % q.nel[1]);
    r /= q.nel[1];
    const int ek = (int)(r % q.nel[2]);
    const int b = (int)(r / q.nel[2]);
    const int s = nb - 1;
    const float* base = in.p + (long long)b * in.sb + (long long)(ek * s) * in.sz + (long long)(ej * s) * in.sy + ei * s;
    float v[4][4][4];
    for (int kb = 0; kb < (nsd == 3 ? nb : 1); ++kb)
      for (int jb = 0; jb < (nsd >= 2 ? nb : 1); ++jb)
        for (int ib = 0; ib < nb; ++ib)
          v[kb][jb][ib] = __ldg(base + (long long)kb * in.sz + (long long)jb * in.sy + ib);
    float* o = out + (long long)b * ngp * nel + ((long long)ek * q.nel[1] + ej) * q.nel[0] + ei;
    for (int kg = 0; kg < (nsd == 3 ? ng : 1); ++kg) {
      float wz[4][4];
      for (int jb = 0; jb < (nsd >= 2 ? nb : 1); ++jb)
        for (int ib = 0; ib < nb; ++ib) {
          float a = v[0][jb][ib];
          if (nsd == 3) {
            a = 0.f;
            for (int kb = 0; kb < nb; ++kb) a += q.f[2][kg][kb] * v[kb][jb][ib];
          }
          wz[jb][ib] = a;
        }
      for (int jg = 0; jg < (nsd >= 2 ? ng : 1); ++jg) {
        float wy[4];
        for (int ib = 0; ib < nb; ++ib) {
          float a = wz[0][ib];
          if (nsd >= 2) {
            a = 0.f;
            for (int jb = 0; jb < nb; ++jb) a += q.f[1][jg][jb] * wz[jb][ib];
          }
          wy[ib] = a;
        }
        for (int ig = 0; ig < ng; ++ig) {
          float a = 0.f;
          for (int ib = 0; ib < nb; ++ib) a += q.f[0][ig][ib] * wy[ib];
          const int G = (kg * (nsd >= 2 ? ng : 1) + jg) * ng + ig;
          o[(long long)G * nel] = a;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(128) k_gp_eval_general_adj(const float* __restrict__ gout, int B, GpGeneral q,
                                                             float* __restrict__ gin) {
  const int nb = q.nb, ng = q.ng, nsd = q.nsd, s = nb - 1;
  const long long nel = (long long)q.nel[0] * q.nel[1] * q.nel[2];
  const long long nodes = (long long)q.n[0] * q.n[1] * q.n[2];
  const long long total = nodes * B;
  const int ngp = (nsd == 3) ? ng * ng * ng : (nsd == 2 ? ng * ng : ng);
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    int c[3];
    c[0] = (int)(idx % q.n[0]);
    long long r = idx / q.n[0];
    c[1] = (int)(r % q.n[1]);
    r /= q.n[1];
    c[2] = (int)(r % q.n[2]);
    const int b = (int)(r / q.n[2]);
    // per direction: the (element, local node) pairs this node belongs to (two for a node shared by neighbours)
    int el[3][2], lb[3][2], cnt[3];
    for (int d = 0; d < 3; ++d) {
      cnt[d] = 0;
      if (d >= nsd) { el[d][0] = 0; lb[d][0] = 0; cnt[d] = 1; continue; }
      const int e = c[d] / s, l = c[d] - e * s;
      if (e < q.nel[d]) { el[d][cnt[d]] = e; lb[d][cnt[d]] = l; ++cnt[d]; }
      if (l == 0 && e > 0) { el[d][cnt[d]] = e - 1; lb[d][cnt[d]] = s; ++cnt[d]; }
    }
    const float* gb = gout + (long long)b * ngp * nel;
    float acc = 0.f;
    for (int pk = 0; pk < cnt[2]; ++pk)
      for (int pj = 0; pj < cnt[1]; ++pj)
        for (int pi = 0; pi < cnt[0]; ++pi) {
          const float* ge = gb + ((long long)el[2][pk] * q.nel[1] + el[1][pj]) * q.nel[0] + el[0][pi];
          for (int kg = 0; kg < (nsd == 3 ? ng : 1); ++kg) {
            const float cz = (nsd == 3) ? q.f[2][kg][lb[2][pk]] : 1.f;
            for (int jg = 0; jg < (nsd >= 2 ? ng : 1); ++jg) {
              const float czy = (nsd >= 2) ? cz * q.f[1][jg][lb[1][pj]] : cz;
              float t = 0.f;
              for (int ig = 0; ig < ng; ++ig) {
                const int G = (kg * (nsd >= 2 ? ng : 1) + jg) * ng + ig;
                t += q.f[0][ig][lb[0][pi]] * __ldg(ge + (long long)G * nel);
              }
              acc += czy * t;
            }
          }
        }
    gin[idx] = acc;
  }
}

static int general_setup(int nsd, int nx, int ny, int nz, int nbf_1d, int ngp_1d, const float* factors, GpGeneral* q) {
  if (nsd < 1 || nsd > 3 || nbf_1d < 2 || nbf_1d > 4 || ngp_1d < 1 || ngp_1d > 4 || !factors) return 1;
  const int n[3] = {nx, nsd >= 2 ? ny : 1, nsd == 3 ? nz : 1};
  q->nsd = nsd; q->nb = nbf_1d; q->ng = ngp_1d;
  for (int d = 0; d < 3; ++d) {
    q->n[d] = n[d];
    q->nel[d] = 1;
    if (d < nsd) {
      if (n[d] < nbf_1d || (n[d] - 1) % (nbf_1d - 1)) return 2;      // (size - 1) % degree == 0, DiffNetFEM.py:67,101
      q->nel[d] = (n[d] - 1) / (nbf_1d - 1);
    }
    for (int g = 0; g < 4; ++g)
      for (int b = 0; b < 4; ++b)
        q->f[d][g][b] = (d < nsd && g < ngp_1d && b < nbf_1d) ? factors[((size_t)d * ngp_1d + g) * nbf_1d + b] : 0.f;
  }
  return 0;
}

cudaError_t launch_gp_eval_general(Field in, int B, int nsd, int nx, int ny, int nz, int nbf_1d, int ngp_1d,
                                   const float* factors, float* out, cudaStream_t s, int* bad) {
  GpGeneral q;
  *bad = general_setup(nsd, nx, ny, nz, nbf_1d, ngp_1d, factors, &q);
  if (*bad) return cudaSuccess;
  const long long total = (long long)B * q.nel[0] * q.nel[1] * q.nel[2];
  long long g = (total + 127) / 128;
  const long long cap = 32LL * sm_count();
  k_gp_eval_general<<<(int)(g > cap ? cap : (g < 1 ? 1 : g)), 128, 0, s>>>(in, B, q, out);
  return cudaGetLastError();
}

cudaError_t launch_gp_eval_general_adj(const float* gout, int B, int nsd, int nx, int ny, int nz, int nbf_1d,
                                       int ngp_1d, const float* factors, float* gin, cudaStream_t s, int* bad) {
  GpGeneral q;
  *bad = general_setup(nsd, nx, ny, nz, nbf_1d, ngp_1d, factors, &q);
  if (*bad) return cudaSuccess;
  const long long total = (long long)B * q.n[0] * q.n[1] * q.n[2];
  long long g = (total + 127) / 128;
  const long long cap = 32LL * sm_count();
  k_gp_eval_general_adj<<<(int)(g > cap ? cap : (g < 1 ? 1 : g)), 128, 0, s>>>(gout, B, q, gin);
  return cudaGetLastError();
}

}  // namespace dn

// ---- dL/dnu on 3-D meshes -----------------------------------------------------------------------------------------
// dL/dnu[n] = S c_k sum over the elements e around node n and their Gauss points g of  w_g N_n(g) |grad u'|^2_g,
// u' = u with the Dirichlet conditions applied, zero where the nu mask fired (16_topopt.py:124,153 differentiates a
// 2-D loss w.r.t. nu; the 2-D kernels emit it in the fused launch, this is the 3-D counterpart as a separate gather
// launch: one thread per node, each adjacent element re-evaluated -- no scratch tensor, no atomics, deterministic;
// a side path, not tuned).
namespace dn {

__device__ __forceinline__ float masked_u(const GradNu3& q, int b, int z, int y, int x) {
  const long long off = (long long)z * q.u.sz + (long long)y * q.u.sy + x;
  float v = __ldg(q.u.p + (long long)b * q.u.sb + off);
  for (int m = 0; m < q.nmasks; ++m) {
    const Field& f = q.mk[m].m;
    const float mv = __ldg(f.p + (long long)b * f.sb + (long long)z * f.sz + (long long)y * f.sy + x);
    if (mv > 0.5f) {
      const Field& vf = q.mk[m].vf;
      v = (q.has_vf && vf.p) ? __ldg(vf.p + (long long)b * vf.sb + (long long)z * vf.sz + (long long)y * vf.sy + x) : q.mk[m].v;
    }
  }
  return v;
}

__global__ void __launch_bounds__(128) k_grad_nu_3d(GradNu3 q, float* __restrict__ out) {
  const long long total = (long long)q.B * q.nz * q.ny * q.nx;
  const int ng = q.ng;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(idx % q.nx);
    long long r = idx / q.nx;
    const int y = (int)(r % q.ny);
    r /= q.ny;
    const int z = (int)(r % q.nz);
    const int b = (int)(r / q.nz);
    float acc = 0.f;
    bool dead = false;
    if (q.numask.p)
      dead = __ldg(q.numask.p + (long long)b * q.numask.sb + (long long)z * q.numask.sz + (long long)y * q.numask.sy + x) > 0.5f;
    if (!dead) {
      for (int kb = 0; kb < 2; ++kb) {
        const int ek = z - kb;
        if (ek < 0 || ek >= q.nz - 1 || ek < q.zlo || ek >= q.zhi) continue;
        for (int jb = 0; jb < 2; ++jb) {
          const int ej = y - jb;
          if (ej < 0 || ej >= q.ny - 1) continue;
          for (int ib = 0; ib < 2; ++ib) {
            const int ei = x - ib;
            if (ei < 0 || ei >= q.nx - 1) continue;
            float v[2][2][2];
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
              for (int bq = 0; bq < 2; ++bq)
#pragma unroll
                for (int a = 0; a < 2; ++a) v[c][bq][a] = masked_u(q, b, ek + c, ej + bq, ei + a);
            for (int kg = 0; kg < ng; ++kg)
              for (int jg = 0; jg < ng; ++jg)
                for (int ig = 0; ig < ng; ++ig) {
                  float g3[3];
#pragma unroll
                  for (int d = 0; d < 3; ++d) {
                    const GpTables& t = q.tb[d + 1];
                    float s = 0.f;
#pragma unroll
                    for (int c = 0; c < 2; ++c)
#pragma unroll
                      for (int bq = 0; bq < 2; ++bq)
#pragma unroll
                        for (int a = 0; a < 2; ++a) s += t.c[2][kg][c] * t.c[1][jg][bq] * t.c[0][ig][a] * v[c][bq][a];
                    g3[d] = s;
                  }
                  const float Nn = q.tb[0].c[2][kg][kb] * q.tb[0].c[1][jg][jb] * q.tb[0].c[0][ig][ib];
                  acc += q.w[kg] * q.w[jg] * q.w[ig] * Nn * (g3[0] * g3[0] + g3[1] * g3[1] + g3[2] * g3[2]);
                }
          }
        }
      }
    }
    out[idx] = q.coef * acc;
  }
}

cudaError_t launch_grad_nu_3d(const GradNu3& q, float* out, cudaStream_t s) {
  const long long total = (long long)q.B * q.nz * q.ny * q.nx;
  long long g = (total + 127) / 128;
  const long long cap = 64LL * sm_count();
  k_grad_nu_3d<<<(int)(g > cap ? cap : (g < 1 ? 1 : g)), 128, 0, s>>>(q, out);
  return cudaGetLastError();
}

}  // namespace dn
