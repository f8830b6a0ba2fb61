// gp_eval.cuh -- standalone Gauss-point evaluation (gauss_pt_eval, DiffNet/DiffNetFEM.py:7-18)
// and its adjoint (autograd's convolution_backward w.r.t. the input), plus the in-place
// gradient scaling used by the autograd wrapper.  Generic in ngp_1d (2..4); these serve
// user-written loss() bodies that are not one of the fused forms.
#pragma once
#include "dn_common.cuh"

namespace dn {

// 1-D factors: c[d][q][a] for direction d (0=x,1=y,2=z), Gauss point q, basis function a:
// shape-function value, or derivative*(2/h) for the differentiated direction.
struct GpTables {
  int n;
  float c[3][4][2];
};

// Up to four tables evaluated in one pass over the input (N, d/dx, d/dy, d/dz in any subset / order).
struct GpMulti {
  int nw;
  GpTables tb[4];
  float* out[4];          // each dense (B, ngp, [nz-1,] ny-1, nx-1)
};
struct GpMultiAdj {
  int nw;
  GpTables tb[4];
  const float* gout[4];   // cotangents of the outputs above
};

cudaError_t launch_gp_eval(Field in, int B, int nx, int ny, int nz, int nsd, const GpMulti& m, cudaStream_t s);
cudaError_t launch_gp_eval_adj(int B, int nx, int ny, int nz, int nsd, const GpMultiAdj& m, float* gin,
                               cudaStream_t s);
// any tensor-product Lagrange basis / rule / 1..3 dimensions; factors = host [nsd][ngp_1d][nbf_1d]; *bad != 0: rejected
cudaError_t launch_gp_eval_general(Field in, int B, int nsd, int nx, int ny, int nz, int nbf_1d, int ngp_1d,
                                   const float* factors, float* out, cudaStream_t s, int* bad);
cudaError_t launch_gp_eval_general_adj(const float* gout, int B, int nsd, int nx, int ny, int nz, int nbf_1d,
                                       int ngp_1d, const float* factors, float* gin, cudaStream_t s, int* bad);
struct GradNu3 {
  Field u, numask;
  Mask mk[DN_MAX_MASKS];
  int nmasks, has_vf;
  int B, nx, ny, nz, ng;
  int zlo, zhi;                 // element layers whose energy counts
  float coef;                   // S * c_k
  float w[4];                   // 1-D weights
  GpTables tb[4];               // N, d/dx, d/dy, d/dz factor tables
};

cudaError_t launch_grad_nu_3d(const GradNu3& q, float* out, cudaStream_t s);

cudaError_t launch_scale(float* x, size_t n, const float* factor_dev, cudaStream_t s);
cudaError_t launch_scale_per_sample(float* x, int batch, size_t n, const float* factors_dev, cudaStream_t s);

}  // namespace dn
