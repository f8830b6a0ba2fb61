// dn_launch.h -- host interface between the fused-loss entry points (dn_api.cu) and the launchers of the four
// kernel families (fem{2d,2d_tma,3d,3d_tma}_dispatch.cu).
#pragma once
#include <cstring>

#include "dn_common.cuh"

namespace dn {

// One validated fused-loss call (dn_api.cu: prepare): fields, Dirichlet set, folded constants, launch options.
struct Common {
  Field u, nu, f, fgp, numask;
  Mask mk[DN_MAX_MASKS];
  int nmasks, MK;            // MK: 0..3 scalar-valued masks, 4 = one mask with a value field
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

// Dirichlet variant of a streaming launch, or -1 when none is instantiated.  An operator apply (mask_input == 0)
// only exists without a source term or nu_zero_mask, with plain masks: variants 5..7 for 1..3 masks.
inline int stream_variant(const Common& c, bool source, bool numask) {
  if (c.mask_input || c.MK == 0) return c.MK;
  return (c.MK <= 3 && !source && !numask) ? c.MK + 4 : -1;
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
