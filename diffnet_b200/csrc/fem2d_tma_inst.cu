// One MK slice of the k_fem2d_tma variants: build.py compiles this file once per Dirichlet variant with -DDN_MK=..,
// so that the kernels compile in parallel.
#if !defined(DN_MK)
#error "fem2d_tma_inst.cu needs -DDN_MK=<Dirichlet variant> (see diffnet_b200/build.py)"
#endif
#include "dn_launch.h"
#include "fem2d_tma.cuh"
#include "fem2d_tma_combos.h"
namespace dn {
// One register budget (<= 128 registers, CTAs of up to 512 threads).  A tighter variant
// (<= 96 registers, 10 instead of 8 resident 64-thread CTAs per SM) measured 10% SLOWER on
// 256^2 x 64: more CTAs per wave means shorter row chunks and more seam work (profiles/).
template <int MK, bool HAS_NU, int FK, bool NUMASK>
const void* kernel2t() {
  return (const void*)k_fem2d_tma<mk_nmasks(MK), mk_value_field(MK), HAS_NU, FK, NUMASK, mk_mask_input(MK),
                                  DN_T2_MAXT, 1>;
}
#define DN_INST(MK, NU, F, NMK) template const void* kernel2t<MK, NU, F, NMK>();
DN2T_COMBOS(DN_INST, DN_MK)
#undef DN_INST
}  // namespace dn
