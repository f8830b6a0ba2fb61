// Instantiation list of k_fem3d_tma: X(MK, NUK, HAS_F, NUMASK, LK).
//   MK    Dirichlet set (0..3 scalar-valued masks, 4 = one mask with a nodal value field,
//         5..7 = 1..3 masks with mask_input = 0)
//   NUK   0: nu == 1, 1: nodal nu, 2: nodal nu on an isotropic grid (hx == hy == hz: k applied per node),
//         3: nu == 1 on an isotropic grid (one product per mode)
#pragma once
//   F     0 no source, 1 (true) nodal source, 2 assembled load vector (plain launches, no nu mask)
//   LK    linked z-slab launch (dn_slab_link): scalar-valued Dirichlet sets (MK 0..3), no nu mask
#define DN3T_COMBOS_PLAIN(X, MK)                                                                        \
  X(MK, 0, false, false, false) X(MK, 0, true, false, false) X(MK, 1, false, false, false)              \
  X(MK, 1, true, false, false) X(MK, 1, false, true, false) X(MK, 1, true, true, false)                 \
  X(MK, 2, false, false, false) X(MK, 2, true, false, false) X(MK, 2, false, true, false) X(MK, 2, true, true, false) \
  X(MK, 3, false, false, false) X(MK, 3, true, false, false)                                            \
  X(MK, 0, 2, false, false) X(MK, 1, 2, false, false) X(MK, 2, 2, false, false) X(MK, 3, 2, false, false)
#define DN3T_COMBOS_LINKED(X, MK)                                                                       \
  X(MK, 0, false, false, true) X(MK, 0, true, false, true) X(MK, 1, false, false, true)                 \
  X(MK, 1, true, false, true) X(MK, 2, false, false, true) X(MK, 2, true, false, true)                  \
  X(MK, 3, false, false, true) X(MK, 3, true, false, true)
#define DN3T_COMBOS_0(X) DN3T_COMBOS_PLAIN(X, 0) DN3T_COMBOS_LINKED(X, 0)
#define DN3T_COMBOS_1(X) DN3T_COMBOS_PLAIN(X, 1) DN3T_COMBOS_LINKED(X, 1)
#define DN3T_COMBOS_2(X) DN3T_COMBOS_PLAIN(X, 2) DN3T_COMBOS_LINKED(X, 2)
#define DN3T_COMBOS_3(X) DN3T_COMBOS_PLAIN(X, 3) DN3T_COMBOS_LINKED(X, 3)
#define DN3T_COMBOS_4(X) DN3T_COMBOS_PLAIN(X, 4)
// MK 5..7 (mask_input = 0, the resmin backward operator): no source term, no nu mask
#define DN3T_COMBOS_OP(X, MK) \
  X(MK, 0, false, false, false) X(MK, 1, false, false, false) X(MK, 2, false, false, false) X(MK, 3, false, false, false)
#define DN3T_COMBOS_5(X) DN3T_COMBOS_OP(X, 5)
#define DN3T_COMBOS_6(X) DN3T_COMBOS_OP(X, 6)
#define DN3T_COMBOS_7(X) DN3T_COMBOS_OP(X, 7)
// DN3T_COMBOS(X, MK) is one slice (one object file, see build.py), DN3T_ALL(X) all of them.
#define DN3T_CAT_(a, b) a##b
#define DN3T_COMBOS(X, MK) DN3T_CAT_(DN3T_COMBOS_, MK)(X)
#define DN3T_ALL(X)                                                                              \
  DN3T_COMBOS(X, 0) DN3T_COMBOS(X, 1) DN3T_COMBOS(X, 2) DN3T_COMBOS(X, 3) DN3T_COMBOS(X, 4)             \
  DN3T_COMBOS(X, 5) DN3T_COMBOS(X, 6) DN3T_COMBOS(X, 7)
