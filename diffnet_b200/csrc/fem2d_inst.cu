// One (V, MK) slice of the k_fem2d variants: build.py compiles this file once per slice with -DDN_V=.. -DDN_MK=..,
// so that the kernels compile in parallel.
#if !defined(DN_V) || !defined(DN_MK)
#error "fem2d_inst.cu needs -DDN_V=<lane width> -DDN_MK=<Dirichlet variant> (see diffnet_b200/build.py)"
#endif
#include "dn_launch.h"
#include "fem2d.cuh"
#include "fem2d_combos.h"
namespace dn {
template <int V, int MK, bool HAS_NU, int FM, bool NUMASK, bool GN>
const void* kernel2d() {
  return (const void*)k_fem2d<V, mk_nmasks(MK), mk_value_field(MK), HAS_NU, FM, NUMASK, GN>;
}
#define DN_INST(V, MK, NU, FM, NMK, GN) template const void* kernel2d<V, MK, NU, FM, NMK, GN>();
DN2D_COMBOS(DN_INST, DN_V, DN_MK)
#undef DN_INST
}  // namespace dn
