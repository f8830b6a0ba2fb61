// Instantiation list of k_fem3d: X(V, MK, HAS_NU, FM, NUMASK) -- see fem2d_combos.h for the codes.
// DN3D_COMBOS(X, V, MK) is one slice (one object file, see build.py), DN3D_ALL(X) all of them.
#pragma once
#define DN3D_COMBOS(X, V, MK)                                                         \
  X(V, MK, false, 0, false) X(V, MK, false, 1, false) X(V, MK, false, 2, false)       \
  X(V, MK, true, 0, false) X(V, MK, true, 1, false) X(V, MK, true, 2, false)          \
  X(V, MK, true, 0, true) X(V, MK, true, 1, true)
#define DN3D_ALL(X)                                                                    \
  DN3D_COMBOS(X, 4, 0) DN3D_COMBOS(X, 4, 1) DN3D_COMBOS(X, 4, 2) DN3D_COMBOS(X, 4, 3) \
  DN3D_COMBOS(X, 4, 4) DN3D_COMBOS(X, 1, 0) DN3D_COMBOS(X, 1, 1) DN3D_COMBOS(X, 1, 2) \
  DN3D_COMBOS(X, 1, 3) DN3D_COMBOS(X, 1, 4)
