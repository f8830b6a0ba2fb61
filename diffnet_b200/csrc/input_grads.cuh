// input_grads.cuh -- gradients of the fused losses with respect to their OTHER inputs (the source f, the forcing
// at the Gauss points f_gp, the Dirichlet value fields, and nu of the residual form).  One launch per backward
// produces every requested one; gather form, no atomics (see input_grads.cu).
#pragma once
#include "dn_common.cuh"

namespace dn {

struct InGrad {
  int mode;                     // 0: energy, 1: residual
  int B, nx, ny, nz;            // nz = 1 in 2-D
  Field u, nu, f, numask, R;    // R: the residual of the forward pass (mode 1)
  const float* fgp;             // dense (B|1, ngp, elems); fgp_sb = 0 broadcasts
  long long fgp_sb;
  Mask mk[DN_MAX_MASKS];
  int nmasks;
  int ng;                       // ngp_1d
  float x[4], w[4];             // 1-D rule
  float d[3];                   // derivative of the 1-D basis in x, y, z: (2/h) / 2
  float ma, mc;                 // 1-D element mass (W1/4) [[1+t, 1-t], [1-t, 1+t]]
  // folded constants (host, fp64 -> fp32)
  float cM;                     // slot 0 = cM * M X
  float cK, cS;                 // slot 1 = cK * K(nu) X + cS * (M f | sum_g w_g N f_gp)
  float cN;                     // slot 2 = cN * sum_g w_g N grad u' . grad R
  float cG;                     // grad_fgp = cG * w_G X_G
  // outputs (NULL = not wanted); bit k of bc set: output k is one (1, ...) field summed over the batch
  float* g_f;                   // bit 0
  float* g_fgp;                 // bit 1
  float* g_nu;                  // bit 2
  float* g_v[DN_MAX_MASKS];     // bit 3 + k
  unsigned bc;
};

cudaError_t launch_input_grads(const InGrad& q, int nsd, int sms, cudaStream_t s);

}  // namespace dn
