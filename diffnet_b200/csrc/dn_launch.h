// dn_launch.h -- host interface between the fused-loss entry points (dn_api.cu) and the launchers of the four
// kernel families (fem{2d,2d_tma,3d,3d_tma}_dispatch.cu).
#pragma once
#include <atomic>
#include <cstdlib>
#include <cstring>

#include "dn_common.cuh"

namespace dn {

#define DN_T2_MAXT 512                    // threads per streaming 2-D CTA -> nx <= 2048
constexpr int kMaxDynSmem = 226 * 1024;   // 227 KB per CTA minus the kernels' static shared memory

// One validated fused-loss call (dn_api.cu: prepare): fields, Dirichlet set, folded constants, launch options.
struct Common {
  Field u, nu, f, fgp, numask;
  Mask mk[DN_MAX_MASKS];
  int nmasks, MK;            // MK: Dirichlet variant, see mk_nmasks
  Consts k;
  Rule rule;
  bool vec4;                 // every field allows 16-byte row loads
  int mode;                  // 0: energy, 1: residual
  int mask_input;            // 0: the mask values are not substituted into the input (operator apply)
  int sms;
  const dn_slab_link* link;  // linked z-slab launch (3-D streaming kernel only), else null
};

// Where a launch writes.
struct Out {
  float* grad;               // dL/du (energy) or R (residual)
  float* grad_nu;            // dL/dnu, 2-D only (the 3-D entry point launches it separately)
  double* loss_out;
  float* loss_f32;
  void* workspace;
  size_t wsb;
  void* stream;
};

// Workspace of a `grid`-CTA launch: the ticket counter, then one double partial per CTA.
inline size_t ws_bytes_for_grid(long long grid) { return 64 + 8 * (size_t)grid; }

// Checks the workspace for a `grid`-CTA launch and points the reduction epilogue at it and at the loss outputs.
inline int reduce_into(const Out& o, long long grid, Reduce* r) {
  const size_t need = ws_bytes_for_grid(grid);
  if (!o.workspace || o.wsb < need) return fail(DN_EWORKSPACE, "workspace too small: %zu < %zu", o.wsb, need);
  if ((uintptr_t)o.workspace % 16) return fail(DN_EWORKSPACE, "workspace must be 16-byte aligned");
  r->counter = (unsigned int*)o.workspace;
  r->partials = (double*)((char*)o.workspace + 64);
  r->loss_out = o.loss_out;
  r->loss_f32 = o.loss_f32;
  return DN_OK;
}

// The Dirichlet variant MK, a template parameter of every kernel family.  prepare() encodes 0..3 for that many
// scalar-valued masks and 4 for one mask with a nodal value field; stream_variant() adds 5..7 for 1..3 scalar-valued
// masks whose values are not substituted into the input (mask_input == 0, which the general kernels take at run time).
constexpr int mk_nmasks(int MK) { return MK == 4 ? 1 : MK >= 5 ? MK - 4 : MK; }
constexpr bool mk_value_field(int MK) { return MK == 4; }
constexpr bool mk_mask_input(int MK) { return MK < 5; }

// Dirichlet variant of a streaming launch, or -1 when none is instantiated.  An operator apply (mask_input == 0)
// only exists without a source term or nu_zero_mask, with plain masks: variants 5..7 for 1..3 masks.
inline int stream_variant(const Common& c, bool source, bool numask) {
  if (c.mask_input || c.MK == 0) return c.MK;
  return (c.MK <= 3 && !source && !numask) ? c.MK + 4 : -1;
}

// Field slots of a streaming launch in the order the kernels read them: u, [nu], [f], [nu_zero_mask], masks...,
// [value field].  Fills `fld` (DN_T2_MAXF slots) and the mask values; returns the number of slots.
inline int stream_fields(const Common& c, Field* fld, float* mval) {
  int nf = 0;
  fld[nf++] = c.u;
  if (c.nu.p) fld[nf++] = c.nu;
  if (c.f.p) fld[nf++] = c.f;
  if (c.numask.p) fld[nf++] = c.numask;
  for (int i = 0; i < c.nmasks; ++i) { fld[nf++] = c.mk[i].m; mval[i] = c.mk[i].v; }
  if (mk_value_field(c.MK)) fld[nf++] = c.mk[0].vf;
  return nf;
}

// One instantiated kernel of a family (the `const void*` of its __global__ function) and the devices (bit d) on
// which it may use kMaxDynSmem bytes of dynamic shared memory.
struct Kernel {
  const void* fn;
  std::atomic<uint64_t> optin{0};
};

// Raises k's dynamic shared memory limit to kMaxDynSmem on the current device, once per kernel and device.
inline cudaError_t opt_in(Kernel& k) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const uint64_t bit = dev < 64 ? 1ull << dev : 0;
  if (k.optin.load(std::memory_order_relaxed) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem);
  if (e == cudaSuccess) k.optin.fetch_or(bit, std::memory_order_relaxed);
  return e;
}

// DN_PDL=0 disables programmatic dependent launch (default on); read once per process.
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("DN_PDL"); return !(e && *e == '0'); }();
  return on;
}

// Launches k with `params` (the kernel's one parameter struct).  `pdl`: with programmatic stream serialisation,
// when pdl_enabled().
inline cudaError_t launch(Kernel& k, const void* params, dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                          bool pdl) {
  cudaError_t e = opt_in(k);
  if (e != cudaSuccess) return e;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  if (pdl && pdl_enabled()) { cfg.attrs = at; cfg.numAttrs = 1; }
  void* args[1] = {const_cast<void*>(params)};
  e = cudaLaunchKernelExC(&cfg, k.fn, args);
  if (e != cudaSuccess) cudaGetLastError();   // reported to the caller, not left for the next CUDA error check
  return e;
}

// Resident CTAs per SM of k for a block of `threads` threads and `smem` bytes of dynamic shared memory; 0 on error.
inline int occupancy(Kernel& k, int threads, size_t smem) {
  int n = 0;
  if (opt_in(k) != cudaSuccess || cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k.fn, threads, smem) != cudaSuccess)
    return 0;
  return n;
}

// Launchers: the streaming kernel when it takes the call (run*t sets *handled), else the general kernel.
int run2d(const Common& c, const dn_geom* g, const Out& o);
int run2t(const Common& c, const dn_geom* g, const Out& o, bool* handled);
int run3d(const Common& c, const dn_geom* g, const Out& o);
int run3t(const Common& c, const dn_geom* g, const Out& o, bool* handled);

// Upper bounds of the grid sizes the planners may pick (workspace sizing) and the streaming planners' choices.
long long plan2d_max_ctas(const dn_geom* g, int sms);
long long plan3d_max_ctas(const dn_geom* g);
long long plan3t_max_ctas(const dn_geom* g);
int debug_plan2t(const dn_geom* g, int nfields, int64_t* out);
int debug_plan3t(const dn_geom* g, int nfields, int has_nu, int64_t* out);

}  // namespace dn
