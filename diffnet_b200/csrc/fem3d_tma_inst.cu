// One MK slice of the k_fem3d_tma variants: build.py compiles this file once per Dirichlet variant with -DDN_MK=..,
// so that the kernels compile in parallel.
#if !defined(DN_MK)
#error "fem3d_tma_inst.cu needs -DDN_MK=<Dirichlet variant> (see diffnet_b200/build.py)"
#endif
#include "dn_launch.h"
#include "fem3d_tma.cuh"
#include "fem3d_tma_combos.h"
namespace dn {
// NUK (fem3d_tma_combos.h): 1, 2 variable nu; 2, 3 isotropic grid
template <int MK, int NUK, int FK, bool NUMASK, bool LK>
const void* kernel3t() {
  return (const void*)k_fem3d_tma<mk_nmasks(MK), mk_value_field(MK), (NUK == 1 || NUK == 2), FK, NUMASK,
                                  mk_mask_input(MK), (NUK >= 2), LK>;
}
#define DN_INST(MK, NU, F, NMK, LK) template const void* kernel3t<MK, NU, F, NMK, LK>();
DN3T_COMBOS(DN_INST, DN_MK)
#undef DN_INST
}  // namespace dn
