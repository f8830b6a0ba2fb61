// Instantiation list of k_fem2d_tma: X(MK, HAS_NU, FK, NUMASK).
//   FK    0 no source, 1 (true) nodal source, 2 assembled load vector (no nu mask variants)
//   MK    Dirichlet set (0..3 scalar-valued masks, 4 = one mask with a nodal value field,
//         5..7 = 1..3 masks with mask_input = 0)
// DN2T_COMBOS(X, MK) is one slice (one object file, see build.py), DN2T_ALL(X) all of them.
#pragma once
#define DN2T_COMBOS_PLAIN(X, MK)                                                 \
  X(MK, false, false, false) X(MK, false, true, false) X(MK, true, false, false) \
  X(MK, true, true, false) X(MK, true, false, true) X(MK, true, true, true)        \
  X(MK, false, 2, false) X(MK, true, 2, false)
// MK 5..7 (mask_input = 0, the resmin backward operator): no source term, no nu mask
#define DN2T_COMBOS_OP(X, MK) X(MK, false, false, false) X(MK, true, false, false)
#define DN2T_COMBOS_0(X) DN2T_COMBOS_PLAIN(X, 0)
#define DN2T_COMBOS_1(X) DN2T_COMBOS_PLAIN(X, 1)
#define DN2T_COMBOS_2(X) DN2T_COMBOS_PLAIN(X, 2)
#define DN2T_COMBOS_3(X) DN2T_COMBOS_PLAIN(X, 3)
#define DN2T_COMBOS_4(X) DN2T_COMBOS_PLAIN(X, 4)
#define DN2T_COMBOS_5(X) DN2T_COMBOS_OP(X, 5)
#define DN2T_COMBOS_6(X) DN2T_COMBOS_OP(X, 6)
#define DN2T_COMBOS_7(X) DN2T_COMBOS_OP(X, 7)
#define DN2T_CAT_(a, b) a##b
#define DN2T_COMBOS(X, MK) DN2T_CAT_(DN2T_COMBOS_, MK)(X)
#define DN2T_ALL(X)                                                                              \
  DN2T_COMBOS(X, 0) DN2T_COMBOS(X, 1) DN2T_COMBOS(X, 2) DN2T_COMBOS(X, 3) DN2T_COMBOS(X, 4)             \
  DN2T_COMBOS(X, 5) DN2T_COMBOS(X, 6) DN2T_COMBOS(X, 7)
