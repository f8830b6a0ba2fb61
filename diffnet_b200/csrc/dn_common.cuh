// dn_common.cuh -- shared device/host plumbing of libdiffnet_fem (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/diffnet_fem.h"

namespace dn {

constexpr int kWarpsPerCta2D = 4;

#define DN_T2_MAXF 8        // field slots of a streaming launch: u, nu, f, numask, masks[3] | mask+value_field

struct Field {
  const float* p;
  long long sb, sz, sy;
};

struct Mask {
  Field m;
  Field vf;
  float v;
};

// Reduction epilogue shared by every loss kernel: per-CTA double partials, a ticket counter,
// and a fixed-order final sum done by whichever CTA draws the last ticket (bit-reproducible:
// the order of the final sum depends only on the grid, never on arrival order).
struct Reduce {
  double* partials;      // [gridDim.x]; all-zero bits on entry and on exit (see finish_loss_w0, fem2d_tma.cuh)
  unsigned int* counter; // zero on entry, zero on exit
  double* loss_out;      // nullable
  float* loss_f32;       // nullable
  // linked z-slab launches (dn_slab_link): the rank's total is also stored into slot `rank` of every
  // rank's receive area (double[world] + int32[world] flags, peer-mapped) and the launch counter is
  // advanced -- the all-reduce of the loss without a collective launch.  All null/0 otherwise.
  double* const* peer_slots;
  int* step;             // this rank's launch counter of the current parity (device word)
  int rank, world;
  // reduction = none (DN_REDUCE_NONE): one loss per sample, loss_out[b].  Sample b owns the partial slots
  // [seg_lo(b), seg_lo(b) + seg_len(b)) and the ticket counter seg_counter[b] (zero on entry, zero on exit); the
  // kernel that writes the slot knows its sample.  seg_q == 0: one loss for the whole launch.
  unsigned int* seg_counter;
  int seg_q, seg_rem;    // every sample owns seg_q slots, samples [0, seg_rem) one more
};

__device__ __forceinline__ int seg_lo(const Reduce& r, int b) { return b * r.seg_q + min(b, r.seg_rem); }
__device__ __forceinline__ int seg_len(const Reduce& r, int b) { return r.seg_q + (b < r.seg_rem ? 1 : 0); }
// the sample that owns slot i (the inverse of seg_lo): the finishers recompute it rather than keep it live
__device__ __forceinline__ int seg_of(const Reduce& r, int i) {
  const int hi = r.seg_rem * (r.seg_q + 1);
  return i < hi ? i / (r.seg_q + 1) : r.seg_rem + (i - hi) / r.seg_q;
}

// Folded constants of the closed-form Q1 energy (DESIGN.md "element math"):
//   kd[d] = S * c_k * W1^nsd * (2/h_d)^2 / 4^nsd(=norm of C) / ... (see host code), kf likewise,
//   t = second moment of the 1-D Gauss rule (1/3 for the 2-point rule).
struct Consts {
  float kx, ky, kz, kf, t;
  float kb;   // S c_f: weight of an assembled load vector
  int lv;     // `f` is an assembled load vector (dn_consts.flags & DN_F_LOAD_VECTOR): streaming kernels only
};

// 1-D quadrature tables, only used by the f-at-Gauss-points path.
struct Rule {
  int n;          // ngp_1d
  float x[4];     // abscissae
  float w[4];     // weights
  float fscale;   // 4/W1^2 (2-D) or 8/W1^3 (3-D): turns moments into "effective modal f"
};

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Called by all threads of the CTA. `cta_value` must be valid in thread 0.
// smem: at least blockDim.x/32 doubles.
__device__ __forceinline__ void finish_loss(const Reduce& r, double cta_value, double* smem) {
  __shared__ bool is_last;
  if (threadIdx.x == 0) {
    r.partials[blockIdx.x] = cta_value;
    __threadfence();
    unsigned int ticket = atomicAdd(r.counter, 1u);
    is_last = (ticket == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // fixed-order strided partial sums, then a fixed tree over warps
  double s = 0.0;
  for (unsigned int i = threadIdx.x; i < gridDim.x; i += blockDim.x) {
    s += __ldcg(r.partials + i);
    __stcg(r.partials + i, 0.0);     // the streaming kernels read an all-zero slot as "not yet written"
  }
  s = warp_sum(s);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) smem[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int w = 0; w < nw; ++w) tot += smem[w];
    if (r.loss_out) *r.loss_out = tot;
    if (r.loss_f32) *r.loss_f32 = (float)tot;
    *r.counter = 0u;   // self-reset: the workspace is ready for the next call
  }
}

// reduction = none in the general kernels: one warp publishes the partial `v` (valid in lane 0) into slot `slot`.
// The warp that draws the last ticket of the slot's sample b sums the sample's slots in a fixed order (strided over
// the warp's lanes, then a shuffle tree: bit-reproducible for a given launch shape) and writes loss[b].  Called by
// the `nlanes` (1..32) threads lanes 0..nlanes-1 of the warp: a 3-D tile block can have fewer than 32 threads.
__device__ __forceinline__ void finish_sample_warp(const Reduce& r, int slot, double v, int lane, int nlanes) {
  const unsigned live = nlanes >= 32 ? 0xffffffffu : (1u << nlanes) - 1u;
  const int b = seg_of(r, slot);
  unsigned last = 0u;
  if (lane == 0) {
    r.partials[slot] = v;
    __threadfence();
    last = (atomicAdd(r.seg_counter + b, 1u) == (unsigned)seg_len(r, b) - 1u) ? 1u : 0u;
  }
  if (!__shfl_sync(live, last, 0)) return;
  __threadfence();
  const int lo = seg_lo(r, b), n = seg_len(r, b);
  double s = 0.0;
  for (int i = lane; i < n; i += nlanes) {     // every slot of the sample is read and zeroed
    s += __ldcg(r.partials + lo + i);
    __stcg(r.partials + lo + i, 0.0);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double t = __shfl_down_sync(live, s, o);   // from a lane beyond nlanes: undefined, and not used
    if (lane + o < nlanes) s += t;
  }
  if (lane == 0) {
    if (r.loss_out) r.loss_out[b] = s;
    if (r.loss_f32) r.loss_f32[b] = (float)s;
    r.seg_counter[b] = 0u;
  }
}

// ---- vector loads -------------------------------------------------------------------------
template <int V>
__device__ __forceinline__ void ldv(const float* __restrict__ p, bool pred, float (&o)[V]) {
  if constexpr (V == 4) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (pred) v = __ldg(reinterpret_cast<const float4*>(p));
    o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
  } else if constexpr (V == 2) {
    float2 v = make_float2(0.f, 0.f);
    if (pred) v = __ldg(reinterpret_cast<const float2*>(p));
    o[0] = v.x; o[1] = v.y;
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) o[i] = pred ? __ldg(p + i) : 0.f;
  }
}

template <int V>
__device__ __forceinline__ void stv(float* __restrict__ p, const float (&v)[V]) {
  if constexpr (V == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else if constexpr (V == 2) {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
  } else {
#pragma unroll
    for (int i = 0; i < V; ++i) p[i] = v[i];
  }
}

__device__ __forceinline__ float lds1(const float* __restrict__ p, bool pred) {
  return pred ? __ldg(p) : 0.f;
}

}  // namespace dn

// ---- host-side error plumbing (dn_api.cu owns the storage) ---------------------------------
namespace dn {
int fail(int code, const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);
// Integer tuning knob from the environment, `dflt` when unset or empty.  Read on every call (DESIGN.md §10b).
int env_int(const char* name, int dflt);
}  // namespace dn
