// Instantiation list of k_fem2d: X(V, MK, HAS_NU, FM, NUMASK, GN).
//   V   lane width (4 = 16-byte loads, 1 = unaligned/odd sizes)
//   MK  Dirichlet set (0..3 scalar-valued masks, 4 = one mask with a nodal value field)
//   FM  source term (0 none, 1 nodal f, 2 f at Gauss points)
//   NUMASK  nu zeroed under a mask (Neumann IBN);  GN  also emit d(loss)/d(nu)
// DN2D_COMBOS(X, V, MK) is one slice (one object file, see build.py), DN2D_ALL(X) all of them.
#pragma once
#define DN2D_COMBOS(X, V, MK)                                                          \
  X(V, MK, false, 0, false, false) X(V, MK, false, 1, false, false)                    \
  X(V, MK, false, 2, false, false) X(V, MK, true, 0, false, false)                     \
  X(V, MK, true, 1, false, false) X(V, MK, true, 2, false, false)                      \
  X(V, MK, true, 0, true, false) X(V, MK, true, 1, true, false)                        \
  X(V, MK, true, 0, false, true) X(V, MK, true, 1, false, true)
#define DN2D_ALL(X)                                                                     \
  DN2D_COMBOS(X, 4, 0) DN2D_COMBOS(X, 4, 1) DN2D_COMBOS(X, 4, 2) DN2D_COMBOS(X, 4, 3)  \
  DN2D_COMBOS(X, 4, 4) DN2D_COMBOS(X, 1, 0) DN2D_COMBOS(X, 1, 1) DN2D_COMBOS(X, 1, 2)  \
  DN2D_COMBOS(X, 1, 3) DN2D_COMBOS(X, 1, 4)
