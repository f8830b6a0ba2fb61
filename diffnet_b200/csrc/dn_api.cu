// dn_api.cu -- extern "C" entry points of libdiffnet_fem.so (see include/diffnet_fem.h).
// Validation and constant folding; the fused-loss launches are planned in the dispatch files (dn_launch.h).
// No device state.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "dn_common.cuh"
#include "dn_launch.h"
#include "gp_eval.cuh"
#include "input_grads.cuh"

namespace dn {
cudaError_t launch_peer_put(float* dst_peer, const float* src, size_t n, int* remote_flag, int* local_counter,
                            unsigned int* ticket, cudaStream_t s);
cudaError_t launch_peer_wait(float* halo, const float* staged, size_t n, const int* flag, int* expect,
                             long long max_spins, int* status, cudaStream_t s);
cudaError_t launch_peer_loss_sum(const double* slots, int world, const int* step, long long max_spins, int* status,
                                 float* out, cudaStream_t s);
cudaError_t launch_peer_allreduce(const float* partial, float* out, double* slots, double* const* peer_slots,
                                  int rank, int world, int* counter, long long max_spins, int* status,
                                  cudaStream_t s);
}  // namespace dn

namespace dn {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return DN_OK;
  return fail(DN_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

// One device query per process and device.
struct DevInfo { int checked, ok, sms; };
static DevInfo g_dev[64];

static int device_ok(int* sms) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return check_cuda(e, "cudaGetDevice");
  if (dev < 0 || dev >= 64) return fail(DN_EINVAL, "device index %d out of range", dev);
  if (!g_dev[dev].checked) {
    int major = 0, minor = 0, n = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    g_dev[dev].ok = (major == 10 && minor == 0);
    g_dev[dev].sms = n;
    g_dev[dev].checked = 1;
    if (!g_dev[dev].ok)
      return fail(DN_EARCH, "device %d is sm_%d%d; libdiffnet_fem is built for sm_100a (B200) only",
                  dev, major, minor);
  }
  if (!g_dev[dev].ok) return fail(DN_EARCH, "device %d is not sm_100", dev);
  if (sms) *sms = g_dev[dev].sms;
  return DN_OK;
}

// 1-D Gauss rule with the reference's own (truncated) constants, DiffNetFEM.py:128-141, zero beyond n, and its
// moments W1 = sum w, t = sum w x^2 / W1.  n is 2..4 (check_geom).
struct Gauss { double x[4], w[4], W1, t; };

static Gauss gauss_rule(int n) {
  Gauss r = {{0, 0, 0, 0}, {0, 0, 0, 0}, 0, 0};
  double* x = r.x;
  double* w = r.w;
  switch (n) {
    case 2: x[0] = -0.5773502691896258; x[1] = 0.5773502691896258; w[0] = w[1] = 1.0; break;
    case 3: x[0] = -0.774596669; x[1] = 0.0; x[2] = 0.774596669;
            w[0] = 5.0 / 9.0; w[1] = 8.0 / 9.0; w[2] = 5.0 / 9.0; break;
    case 4: x[0] = -0.861136; x[1] = -0.339981; x[2] = 0.339981; x[3] = 0.861136;
            w[0] = 0.347855; w[1] = 0.652145; w[2] = 0.652145; w[3] = 0.347855; break;
  }
  double m2 = 0;
  for (int i = 0; i < n; ++i) { r.W1 += w[i]; m2 += w[i] * x[i] * x[i]; }
  r.t = m2 / r.W1;
  return r;
}

// The mesh checks of every entry point that takes a dn_geom.  `spacing`: the call uses hx, hy (, hz).
static int check_geom(const dn_geom* g, int nsd, bool spacing = true) {
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  if (g->nsd != nsd) return fail(DN_EINVAL, "geom.nsd=%d but the %d-D entry point was called", g->nsd, nsd);
  if (g->batch < 1 || g->nx < 2 || g->ny < 2 || (nsd == 3 && g->nz < 2))
    return fail(DN_EINVAL, "need batch >= 1 and >= 2 nodes per direction (B=%d nx=%d ny=%d nz=%d)",
                g->batch, g->nx, g->ny, g->nz);
  if (spacing && (!(g->hx > 0) || !(g->hy > 0) || (nsd == 3 && !(g->hz > 0))))
    return fail(DN_EINVAL, "element sizes must be positive");
  if (g->ngp_1d < 2 || g->ngp_1d > 4) return fail(DN_EINVAL, "ngp_1d=%d (2..4)", g->ngp_1d);
  return DN_OK;
}

// Divisor of the loss: 1 for reduction = sum; for mean g->mean_count, else B times the elements the call owns; for
// none (DN_REDUCE_NONE, which check_per_sample admits only without mean_count and z-slab ownership) the elements of
// one sample.
static double loss_count(const dn_geom* g, int nsd, int reduction) {
  const bool none = (reduction == DN_REDUCE_NONE);
  if (reduction != 0 && !none) return 1.0;
  if (!none && g->mean_count > 0) return g->mean_count;
  double nelz = 1.0;
  if (nsd == 3) {
    const int hi = g->z_own_hi < g->nz - 1 ? g->z_own_hi : g->nz - 1;
    nelz = (g->z_own_hi > g->z_own_lo) ? (double)(hi - g->z_own_lo) : (double)(g->nz - 1);
  }
  return (none ? 1.0 : (double)g->batch) * (g->nx - 1) * (double)(g->ny - 1) * nelz;
}

// reduction = none: every sample's loss has to come out of this launch whole, so it refuses what splits a sample
// (a z-slab holds part of one) or redefines the divisor.
static int check_per_sample(const dn_geom* g, const dn_slab_link* link) {
  if (link) return fail(DN_EINVAL, "reduction = none is not available for a linked z-slab launch");
  if (g->z_own_lo != 0 || g->z_own_hi != 0)
    return fail(DN_EINVAL, "reduction = none is not available under z-slab ownership (z_own_lo/hi set): a slab holds "
                           "part of a sample");
  if (g->mean_count != 0) return fail(DN_EINVAL, "reduction = none takes no mean_count");
  return DN_OK;
}

static Field to_field(const dn_field* f) {
  Field o{nullptr, 0, 0, 0};
  if (f && f->ptr) { o.p = f->ptr; o.sb = f->stride_b; o.sz = f->stride_z; o.sy = f->stride_y; }
  return o;
}

static bool aligned4(const Field& f, bool use_z) {
  if (!f.p) return true;
  return ((uintptr_t)f.p % 16 == 0) && (f.sb % 4 == 0) && (f.sy % 4 == 0) && (!use_z || f.sz % 4 == 0);
}

// Validates one fused-loss call and folds its constants; the caller sets mode, mask_input, sms and link.
static int prepare(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                   const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask, const dn_geom* g,
                   const dn_consts& cs, Common* c) {
  if (int rc = check_geom(g, nsd)) return rc;
  if (!u || !u->ptr) return fail(DN_EINVAL, "u is NULL");
  if (f && f->ptr && fgp && fgp->ptr) return fail(DN_EINVAL, "give f or fgp, not both");
  if ((cs.flags & DN_F_LOAD_VECTOR) && !(f && f->ptr)) return fail(DN_EINVAL, "DN_F_LOAD_VECTOR needs the load vector in f");
  if (nmasks < 0 || nmasks > DN_MAX_MASKS)
    return fail(DN_EINVAL, "nmasks=%d (max %d)", nmasks, DN_MAX_MASKS);
  if (nmasks > 0 && !masks) return fail(DN_EINVAL, "masks is NULL");

  memset(c, 0, sizeof(*c));
  c->u = to_field(u); c->nu = to_field(nu); c->f = to_field(f); c->fgp = to_field(fgp);
  c->numask = to_field(nu_zero_mask);
  if (c->numask.p && !c->nu.p) return fail(DN_EINVAL, "nu_zero_mask needs nu");
  c->nmasks = nmasks;
  int nvf = 0;
  for (int i = 0; i < nmasks; ++i) {
    if (!masks[i].mask.ptr) return fail(DN_EINVAL, "masks[%d].mask is NULL", i);
    c->mk[i].m = to_field(&masks[i].mask);
    c->mk[i].vf = to_field(&masks[i].value_field);
    c->mk[i].v = masks[i].value;
    nvf += c->mk[i].vf.p ? 1 : 0;
  }
  if (nvf > 0 && nmasks != 1)
    return fail(DN_EINVAL, "a Dirichlet value_field is supported only as the single mask");
  c->MK = nvf ? 4 : nmasks;

  const Gauss r = gauss_rule(g->ngp_1d);
  const double S = cs.scale / loss_count(g, nsd, cs.reduction);
  const double Wn = (nsd == 2) ? r.W1 * r.W1 : r.W1 * r.W1 * r.W1;
  const double nrm = (nsd == 2) ? 64.0 : 512.0;     // (2^nsd)^2 from un-normalised C * A^2
  c->k.kx = (float)(S * cs.c_k * Wn * (2.0 / g->hx) * (2.0 / g->hx) / nrm);
  c->k.ky = (float)(S * cs.c_k * Wn * (2.0 / g->hy) * (2.0 / g->hy) / nrm);
  c->k.kz = (nsd == 3) ? (float)(S * cs.c_k * Wn * (2.0 / g->hz) * (2.0 / g->hz) / nrm) : 0.f;
  c->k.kf = (float)(S * cs.c_f * Wn / ((nsd == 2) ? 16.0 : 64.0));
  c->k.t = (float)r.t;
  c->k.kb = (float)(S * cs.c_f);
  c->k.lv = (cs.flags & DN_F_LOAD_VECTOR) ? 1 : 0;
  c->rule.n = g->ngp_1d;
  for (int i = 0; i < 4; ++i) {
    c->rule.x[i] = (float)r.x[i];
    c->rule.w[i] = (float)r.w[i];
  }
  c->rule.fscale = (float)(((nsd == 2) ? 4.0 : 8.0) / Wn);

  bool v4 = (g->nx % 4 == 0);
  const bool z = (nsd == 3);
  v4 = v4 && aligned4(c->u, z) && aligned4(c->nu, z) && aligned4(c->f, z) && aligned4(c->numask, z);
  for (int i = 0; i < nmasks; ++i) v4 = v4 && aligned4(c->mk[i].m, z) && aligned4(c->mk[i].vf, z);
  if (env_int("DN_FORCE_SCALAR", 0)) v4 = false;
  c->vec4 = v4;
  return DN_OK;
}

static int gp_common(const dn_geom* g, int which, int nsd, GpTables* tb) {
  if (int rc = check_geom(g, nsd, false)) return rc;
  if (which < 0 || which > (nsd == 2 ? 2 : 3)) return fail(DN_EINVAL, "which=%d", which);
  const Gauss r = gauss_rule(g->ngp_1d);
  // 1-D factors per Gauss point: value table N1[gp][bf] and derivative table D1[bf] * (2/h).
  // The reference stores the fp32 rounding of the f64 product including 2/h
  // (DiffNetFEM.py:198-215, 405-453); the separable evaluation here agrees to 1 ulp-ish.
  tb->n = g->ngp_1d;
  const double s[3] = {2.0 / g->hx, 2.0 / g->hy, nsd == 3 ? 2.0 / g->hz : 0.0};
  for (int d = 0; d < 3; ++d) {
    const bool der = (which == d + 1);
    for (int q = 0; q < 4; ++q) {
      const double x = r.x[q];
      tb->c[d][q][0] = (float)(der ? -0.5 * s[d] : 0.5 * (1.0 - x));
      tb->c[d][q][1] = (float)(der ? +0.5 * s[d] : 0.5 * (1.0 + x));
    }
  }
  return DN_OK;
}

// dn_fem_energy_{2d,3d}_f32 and, with `link`, dn_fem_energy_3d_linked_f32.
static int energy(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                  const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask, const dn_geom* g,
                  const dn_consts* c, const dn_slab_link* link, const Out& o) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!c) return fail(DN_EINVAL, "consts is NULL");
  dn_consts cs = *c;
  if (link) cs.flags = 0;       // a linked launch streams a nodal source
  Common cm;
  if (int rc = prepare(nsd, u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, cs, &cm)) return rc;
  if (o.grad_nu && !cm.nu.p) return fail(DN_EINVAL, "grad_nu requested without nu");
  cm.per_sample = (cs.reduction == DN_REDUCE_NONE);
  if (cm.per_sample)
    if (int rc = check_per_sample(g, link)) return rc;
  cm.mask_input = 1; cm.sms = sms; cm.link = link;
  if (nsd == 2) return run2d(cm, g, o);
  if (int rc = run3d(cm, g, o)) return rc;
  if (!o.grad_nu) return DN_OK;
  // dL/dnu: a separate gather launch (gp_eval.cu: k_grad_nu_3d)
  GradNu3 q;
  memset(&q, 0, sizeof(q));
  q.u = cm.u; q.numask = cm.numask;
  for (int i = 0; i < DN_MAX_MASKS; ++i) q.mk[i] = cm.mk[i];
  q.nmasks = cm.nmasks; q.has_vf = (cm.MK == 4) ? 1 : 0;
  q.B = g->batch; q.nx = g->nx; q.ny = g->ny; q.nz = g->nz; q.ng = g->ngp_1d;
  q.zlo = 0; q.zhi = g->nz - 1;
  if (g->z_own_hi > g->z_own_lo) { q.zlo = g->z_own_lo; q.zhi = g->z_own_hi < g->nz - 1 ? g->z_own_hi : g->nz - 1; }
  q.coef = (float)(c->scale / loss_count(g, 3, c->reduction) * c->c_k);
  const Gauss r = gauss_rule(g->ngp_1d);
  for (int i = 0; i < 4; ++i) q.w[i] = (float)r.w[i];
  for (int w = 0; w < 4; ++w)
    if (int rc = gp_common(g, w, 3, &q.tb[w])) return rc;
  return check_cuda(launch_grad_nu_3d(q, o.grad_nu, (cudaStream_t)o.stream), "grad_nu launch");
}

// dn_fem_residual_reduce_{2d,3d}_f32; reduction 1 (sum) or DN_REDUCE_NONE
static int residual(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f, const dn_mask* masks,
                    int nmasks, int apply_masks_to_input, const dn_geom* g, double jac, int reduction, const Out& o) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!o.grad) return fail(DN_EINVAL, "residual output is NULL");
  if (reduction != 1 && reduction != DN_REDUCE_NONE)
    return fail(DN_EINVAL, "residual reduction=%d (1 = sum, %d = none)", reduction, DN_REDUCE_NONE);
  // R = d/du [ sum_e sum_g jac w_g ( 1/2 nu |grad u|^2 - u f ) ]
  const dn_consts cs = {0.5 * jac, jac, 1.0, 1, 0};
  Common cm;
  if (int rc = prepare(nsd, u, nu, f, nullptr, masks, nmasks, nullptr, g, cs, &cm)) return rc;
  cm.per_sample = (reduction == DN_REDUCE_NONE);
  if (cm.per_sample)
    if (int rc = check_per_sample(g, nullptr)) return rc;
  cm.mode = 1; cm.mask_input = apply_masks_to_input ? 1 : 0; cm.sms = sms;
  return nsd == 2 ? run2d(cm, g, o) : run3d(cm, g, o);
}

}  // namespace dn

using namespace dn;

extern "C" {

int dn_abi_version(void) { return DN_ABI_VERSION; }
const char* dn_last_error(void) { return g_err; }
int dn_device_check(void) { return device_ok(nullptr); }

size_t dn_fem_workspace_bytes(const dn_geom* g) {
  if (!g) return 0;
  // upper bound over both lane widths and any env override; grids are <= items.  Host-only query: the SM count of
  // the current device when there is one, else the B200's 148
  int sms = 148;
  {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      sms = n;
    cudaGetLastError();
  }
  const long long worst = (g->nsd == 2) ? plan2d_max_ctas(g, sms) : plan3d_max_ctas(g);
  // + one ticket counter per sample for reduction = none (reduce_into)
  return ws_bytes_for_grid(worst + 1024) + 4 * (size_t)(g->batch > 0 ? g->batch : 0);
}

int dn_debug_plan(const dn_geom* g, int nfields, int has_nu, int64_t out[16]) {
  if (!g || !out) return fail(DN_EINVAL, "NULL pointer");
  for (int i = 0; i < 16; ++i) out[i] = 0;
  if (nfields < 1 || nfields > DN_T2_MAXF) return fail(DN_EINVAL, "nfields=%d", nfields);
  if (g->nsd == 2) return debug_plan2t(g, nfields, out);
  if (g->nsd == 3) return debug_plan3t(g, nfields, has_nu, out);
  return fail(DN_EINVAL, "nsd=%d", g->nsd);
}

int dn_fem_energy_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                         const dn_field* fgp, const dn_mask* masks, int nmasks,
                         const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                         float* grad_u, float* grad_nu, void* workspace, size_t workspace_bytes,
                         double* loss_out, float* loss_out_f32, void* stream) {
  return energy(2, u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, c, nullptr,
                Out{grad_u, grad_nu, loss_out, loss_out_f32, workspace, workspace_bytes, stream});
}

int dn_fem_energy_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                         const dn_field* fgp, const dn_mask* masks, int nmasks,
                         const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                         float* grad_u, float* grad_nu, void* workspace, size_t workspace_bytes,
                         double* loss_out, float* loss_out_f32, void* stream) {
  return energy(3, u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, c, nullptr,
                Out{grad_u, grad_nu, loss_out, loss_out_f32, workspace, workspace_bytes, stream});
}

int dn_fem_energy_3d_linked_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask,
                                const dn_geom* g, const dn_consts* c, const dn_slab_link* link,
                                float* grad_u, void* workspace, size_t workspace_bytes,
                                double* loss_out, float* loss_out_f32, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!link) return fail(DN_EINVAL, "link is NULL");
  return energy(3, u, nu, f, nullptr, masks, nmasks, nu_zero_mask, g, c, link,
                Out{grad_u, nullptr, loss_out, loss_out_f32, workspace, workspace_bytes, stream});
}

int dn_fem_residual_reduce_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                  const dn_mask* masks, int nmasks, int apply_masks_to_input,
                                  const dn_geom* g, double jac, float* residual_out, void* workspace,
                                  size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                                  void* stream, int reduction) {
  return residual(2, u, nu, f, masks, nmasks, apply_masks_to_input, g, jac, reduction,
                  Out{residual_out, nullptr, loss_out, loss_out_f32, workspace, workspace_bytes, stream});
}

int dn_fem_residual_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                           const dn_mask* masks, int nmasks, int apply_masks_to_input,
                           const dn_geom* g, double jac, float* residual_out, void* workspace,
                           size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                           void* stream) {
  return dn_fem_residual_reduce_2d_f32(u, nu, f, masks, nmasks, apply_masks_to_input, g, jac, residual_out,
                                       workspace, workspace_bytes, loss_out, loss_out_f32, stream, 1);
}

int dn_fem_residual_reduce_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                  const dn_mask* masks, int nmasks, int apply_masks_to_input,
                                  const dn_geom* g, double jac, float* residual_out, void* workspace,
                                  size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                                  void* stream, int reduction) {
  return residual(3, u, nu, f, masks, nmasks, apply_masks_to_input, g, jac, reduction,
                  Out{residual_out, nullptr, loss_out, loss_out_f32, workspace, workspace_bytes, stream});
}

int dn_fem_residual_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                           const dn_mask* masks, int nmasks, int apply_masks_to_input,
                           const dn_geom* g, double jac, float* residual_out, void* workspace,
                           size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                           void* stream) {
  return dn_fem_residual_reduce_3d_f32(u, nu, f, masks, nmasks, apply_masks_to_input, g, jac, residual_out,
                                       workspace, workspace_bytes, loss_out, loss_out_f32, stream, 1);
}

int dn_peer_loss_sum_f32(const double* slots, int world, const int32_t* step, int64_t max_spins,
                         int32_t* status, float* out, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!slots || !step || !status || !out) return fail(DN_EINVAL, "NULL pointer");
  if (world < 1 || world > 32) return fail(DN_EINVAL, "world %d (1..32)", world);
  return check_cuda(launch_peer_loss_sum(slots, world, step, max_spins > 0 ? max_spins : (1LL << 26), status, out,
                                         (cudaStream_t)stream), "peer_loss_sum launch");
}

// ------------------------------------------------------------------------------------ input gradients
static int ingrad_common(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                         const dn_mask* masks, int nmasks, const dn_geom* g, float* const* grad_values, InGrad* q) {
  if (int rc = check_geom(g, nsd)) return rc;
  if (g->z_own_hi > g->z_own_lo)
    return fail(DN_EINVAL, "input gradients are not available under z-slab ownership (z_own_lo/hi set): a slab "
                           "would only hold a partial gradient");
  if (!u || !u->ptr) return fail(DN_EINVAL, "u is NULL");
  if (nmasks < 0 || nmasks > DN_MAX_MASKS) return fail(DN_EINVAL, "nmasks=%d (max %d)", nmasks, DN_MAX_MASKS);
  if (nmasks > 0 && !masks) return fail(DN_EINVAL, "masks is NULL");
  memset(q, 0, sizeof(*q));
  const bool bat = g->batch > 1;
  q->B = g->batch; q->nx = g->nx; q->ny = g->ny; q->nz = (nsd == 3) ? g->nz : 1;
  q->u = to_field(u); q->nu = to_field(nu); q->f = to_field(f);
  if (fgp && fgp->ptr) {
    const long long nel = (long long)(g->nx - 1) * (g->ny - 1) * (nsd == 3 ? g->nz - 1 : 1);
    long long ngp = 1;
    for (int d = 0; d < nsd; ++d) ngp *= g->ngp_1d;
    if (bat && fgp->stride_b != 0 && fgp->stride_b != ngp * nel)
      return fail(DN_EINVAL, "fgp must be dense (stride_b = ngp * elems, or 0)");
    q->fgp = fgp->ptr;
    q->fgp_sb = bat ? fgp->stride_b : 0;
  }
  q->nmasks = nmasks;
  for (int i = 0; i < nmasks; ++i) {
    if (!masks[i].mask.ptr) return fail(DN_EINVAL, "masks[%d].mask is NULL", i);
    q->mk[i] = Mask{to_field(&masks[i].mask), to_field(&masks[i].value_field), masks[i].value};
    q->g_v[i] = grad_values ? grad_values[i] : nullptr;
    if (q->g_v[i] && !q->mk[i].vf.p) return fail(DN_EINVAL, "grad_values[%d] needs masks[%d].value_field", i, i);
    if (q->g_v[i] && bat && q->mk[i].vf.sb == 0) q->bc |= 8u << i;
  }
  q->ng = g->ngp_1d;
  const Gauss r = gauss_rule(g->ngp_1d);
  for (int i = 0; i < 4; ++i) { q->x[i] = (float)r.x[i]; q->w[i] = (float)r.w[i]; }
  q->ma = (float)(0.25 * r.W1 * (1.0 + r.t));
  q->mc = (float)(0.25 * r.W1 * (1.0 - r.t));
  q->d[0] = (float)(1.0 / g->hx); q->d[1] = (float)(1.0 / g->hy); q->d[2] = nsd == 3 ? (float)(1.0 / g->hz) : 0.f;
  return DN_OK;
}

static int energy_input_grads(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                              const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask, const dn_geom* g,
                              const dn_consts* c, float* grad_f, float* grad_fgp, float* const* grad_values,
                              void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!c) return fail(DN_EINVAL, "consts is NULL");
  if (c->flags & DN_F_LOAD_VECTOR) return fail(DN_EINVAL, "input gradients take f_gp itself, not DN_F_LOAD_VECTOR");
  if (f && f->ptr && fgp && fgp->ptr) return fail(DN_EINVAL, "give f or fgp, not both");
  InGrad q;
  if (int rc = ingrad_common(nsd, u, nu, f, fgp, masks, nmasks, g, grad_values, &q)) return rc;
  if (c->reduction == DN_REDUCE_NONE)
    if (int rc = check_per_sample(g, nullptr)) return rc;
  q.numask = to_field(nu_zero_mask);
  if (q.numask.p && !q.nu.p) return fail(DN_EINVAL, "nu_zero_mask needs nu");
  if (grad_f && !q.f.p) return fail(DN_EINVAL, "grad_f requested without f");
  if (grad_fgp && !q.fgp) return fail(DN_EINVAL, "grad_fgp requested without fgp");
  const double S = c->scale / loss_count(g, nsd, c->reduction);
  q.mode = 0;
  q.cM = q.cS = q.cG = (float)(-S * c->c_f);
  q.cK = (float)(2.0 * S * c->c_k);
  q.g_f = grad_f;
  q.g_fgp = grad_fgp;
  if (grad_f && g->batch > 1 && q.f.sb == 0) q.bc |= 1u;
  if (grad_fgp && g->batch > 1 && q.fgp_sb == 0) q.bc |= 2u;
  bool any = grad_f || grad_fgp;
  for (int k = 0; k < nmasks; ++k) any = any || q.g_v[k];
  if (!any) return DN_OK;
  return check_cuda(launch_input_grads(q, nsd, sms, (cudaStream_t)stream), "energy input-gradient launch");
}

static int residual_input_grads(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f,
                                const dn_field* residual, const dn_mask* masks, int nmasks, const dn_geom* g,
                                double jac, float* grad_nu, float* grad_f, float* const* grad_values, void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  InGrad q;
  if (int rc = ingrad_common(nsd, u, nu, f, nullptr, masks, nmasks, g, grad_values, &q)) return rc;
  if (!residual || !residual->ptr) return fail(DN_EINVAL, "residual is NULL");
  q.R = to_field(residual);
  if (grad_nu && !q.nu.p) return fail(DN_EINVAL, "grad_nu requested without nu");
  if (grad_f && !q.f.p) return fail(DN_EINVAL, "grad_f requested without f");
  q.mode = 1;
  q.cM = (float)(-2.0 * jac);
  q.cK = q.cN = (float)(2.0 * jac);
  q.g_f = grad_f;
  q.g_nu = grad_nu;
  if (grad_f && g->batch > 1 && q.f.sb == 0) q.bc |= 1u;
  if (grad_nu && g->batch > 1 && q.nu.sb == 0) q.bc |= 4u;
  bool any = grad_f || grad_nu;
  for (int k = 0; k < nmasks; ++k) any = any || q.g_v[k];
  if (!any) return DN_OK;
  return check_cuda(launch_input_grads(q, nsd, sms, (cudaStream_t)stream), "residual input-gradient launch");
}

int dn_fem_energy_input_grads_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                                     const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask, const dn_geom* g,
                                     const dn_consts* c, float* grad_f, float* grad_fgp, float* const* grad_values,
                                     void* stream) {
  return energy_input_grads(2, u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, c, grad_f, grad_fgp, grad_values,
                            stream);
}
int dn_fem_energy_input_grads_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                                     const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask, const dn_geom* g,
                                     const dn_consts* c, float* grad_f, float* grad_fgp, float* const* grad_values,
                                     void* stream) {
  return energy_input_grads(3, u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, c, grad_f, grad_fgp, grad_values,
                            stream);
}
int dn_fem_residual_input_grads_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                       const dn_field* residual, const dn_mask* masks, int nmasks, const dn_geom* g,
                                       double jac, float* grad_nu, float* grad_f, float* const* grad_values,
                                       void* stream) {
  return residual_input_grads(2, u, nu, f, residual, masks, nmasks, g, jac, grad_nu, grad_f, grad_values, stream);
}
int dn_fem_residual_input_grads_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                       const dn_field* residual, const dn_mask* masks, int nmasks, const dn_geom* g,
                                       double jac, float* grad_nu, float* grad_f, float* const* grad_values,
                                       void* stream) {
  return residual_input_grads(3, u, nu, f, residual, masks, nmasks, g, jac, grad_nu, grad_f, grad_values, stream);
}

static int gp_forward(const dn_field* in, const dn_geom* g, int nsd, int nwhich, const int* which,
                      float* const* outs, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (nwhich < 1 || nwhich > 4 || !which || !outs) return fail(DN_EINVAL, "1..4 tables per call");
  GpMulti m;
  m.nw = nwhich;
  for (int w = 0; w < nwhich; ++w) {
    if (int rc = gp_common(g, which[w], nsd, &m.tb[w])) return rc;
    if (!outs[w]) return fail(DN_EINVAL, "NULL output %d", w);
    m.out[w] = outs[w];
  }
  if (!in || !in->ptr) return fail(DN_EINVAL, "NULL input");
  return check_cuda(launch_gp_eval(to_field(in), g->batch, g->nx, g->ny, nsd == 3 ? g->nz : 1, nsd, m,
                                   (cudaStream_t)stream), "gp_eval launch");
}

static int gp_adjoint(const float* const* grad_outs, const dn_geom* g, int nsd, int nwhich, const int* which,
                      float* grad_in, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (nwhich < 1 || nwhich > 4 || !which || !grad_outs) return fail(DN_EINVAL, "1..4 tables per call");
  GpMultiAdj m;
  m.nw = nwhich;
  for (int w = 0; w < nwhich; ++w) {
    if (int rc = gp_common(g, which[w], nsd, &m.tb[w])) return rc;
    if (!grad_outs[w]) return fail(DN_EINVAL, "NULL cotangent %d", w);
    m.gout[w] = grad_outs[w];
  }
  if (!grad_in) return fail(DN_EINVAL, "NULL output");
  return check_cuda(launch_gp_eval_adj(g->batch, g->nx, g->ny, nsd == 3 ? g->nz : 1, nsd, m, grad_in,
                                       (cudaStream_t)stream), "gp_eval_adj launch");
}

int dn_fem_gp_eval_2d_f32(const dn_field* in, const dn_geom* g, int which, float* out, void* stream) {
  return gp_forward(in, g, 2, 1, &which, &out, stream);
}
int dn_fem_gp_eval_3d_f32(const dn_field* in, const dn_geom* g, int which, float* out, void* stream) {
  return gp_forward(in, g, 3, 1, &which, &out, stream);
}
int dn_fem_gp_eval_adj_2d_f32(const float* grad_out, const dn_geom* g, int which, float* grad_in, void* stream) {
  return gp_adjoint(&grad_out, g, 2, 1, &which, grad_in, stream);
}
int dn_fem_gp_eval_adj_3d_f32(const float* grad_out, const dn_geom* g, int which, float* grad_in, void* stream) {
  return gp_adjoint(&grad_out, g, 3, 1, &which, grad_in, stream);
}
int dn_fem_gp_eval_multi_2d_f32(const dn_field* in, const dn_geom* g, int nwhich, const int* which,
                                float* const* outs, void* stream) {
  return gp_forward(in, g, 2, nwhich, which, outs, stream);
}
int dn_fem_gp_eval_multi_3d_f32(const dn_field* in, const dn_geom* g, int nwhich, const int* which,
                                float* const* outs, void* stream) {
  return gp_forward(in, g, 3, nwhich, which, outs, stream);
}
int dn_fem_gp_eval_multi_adj_2d_f32(const float* const* grad_outs, const dn_geom* g, int nwhich, const int* which,
                                    float* grad_in, void* stream) {
  return gp_adjoint(grad_outs, g, 2, nwhich, which, grad_in, stream);
}
int dn_fem_gp_eval_multi_adj_3d_f32(const float* const* grad_outs, const dn_geom* g, int nwhich, const int* which,
                                    float* grad_in, void* stream) {
  return gp_adjoint(grad_outs, g, 3, nwhich, which, grad_in, stream);
}

int dn_fem_gp_eval_general_f32(const dn_field* in, int nsd, int batch, int nx, int ny, int nz, int nbf_1d,
                               int ngp_1d, const float* factors, float* out, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!in || !in->ptr || !out || batch < 1) return fail(DN_EINVAL, "gp_eval_general: NULL input/output");
  int bad = 0;
  cudaError_t e = launch_gp_eval_general(to_field(in), batch, nsd, nx, ny, nz, nbf_1d, ngp_1d, factors, out,
                                         (cudaStream_t)stream, &bad);
  if (bad) return fail(DN_EINVAL, "gp_eval_general: nsd 1..3, nbf_1d 2..4, ngp_1d 1..4, (nodes - 1) %% (nbf_1d - 1) == 0");
  return check_cuda(e, "gp_eval_general launch");
}

int dn_fem_gp_eval_general_adj_f32(const float* grad_out, int nsd, int batch, int nx, int ny, int nz, int nbf_1d,
                                   int ngp_1d, const float* factors, float* grad_in, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!grad_out || !grad_in || batch < 1) return fail(DN_EINVAL, "gp_eval_general_adj: NULL input/output");
  int bad = 0;
  cudaError_t e = launch_gp_eval_general_adj(grad_out, batch, nsd, nx, ny, nz, nbf_1d, ngp_1d, factors, grad_in,
                                             (cudaStream_t)stream, &bad);
  if (bad) return fail(DN_EINVAL, "gp_eval_general_adj: nsd 1..3, nbf_1d 2..4, ngp_1d 1..4, (nodes - 1) %% (nbf_1d - 1) == 0");
  return check_cuda(e, "gp_eval_general_adj launch");
}

int dn_fem_load_vector_f32(const dn_field* fgp, const dn_geom* g, float* out, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (int rc = check_geom(g, g && g->nsd == 3 ? 3 : 2, false)) return rc;
  if (!fgp || !fgp->ptr || !out) return fail(DN_EINVAL, "load_vector: NULL input/output");
  const Gauss r = gauss_rule(g->ngp_1d);
  // b = N^T (w f_gp): the transpose of the Gauss-point interpolation with the quadrature weights folded into the
  // 1-D factors -- the tuned adjoint kernels (gp_eval.cu) do the assembly
  GpMultiAdj m;
  memset(&m, 0, sizeof(m));
  m.nw = 1;
  m.tb[0].n = g->ngp_1d;
  for (int d = 0; d < 3; ++d)
    for (int i = 0; i < g->ngp_1d; ++i) {
      m.tb[0].c[d][i][0] = (float)(r.w[i] * 0.5 * (1.0 - r.x[i]));
      m.tb[0].c[d][i][1] = (float)(r.w[i] * 0.5 * (1.0 + r.x[i]));
    }
  m.gout[0] = (const float*)fgp->ptr;
  const int B = (fgp->stride_b == 0) ? 1 : g->batch;
  const long long per_b = (long long)(g->nx - 1) * (g->ny - 1) * (g->nsd == 3 ? g->nz - 1 : 1);
  long long ngp = 1;
  for (int d = 0; d < g->nsd; ++d) ngp *= g->ngp_1d;
  if (B > 1 && fgp->stride_b != ngp * per_b) return fail(DN_EINVAL, "load_vector: fgp must be dense (stride_b = ngp * elems)");
  return check_cuda(launch_gp_eval_adj(B, g->nx, g->ny, g->nsd == 3 ? g->nz : 1, g->nsd, m, out, (cudaStream_t)stream),
                    "load_vector launch");
}

int dn_peer_alloc(size_t bytes, void** ptr) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!ptr || bytes == 0) return fail(DN_EINVAL, "dn_peer_alloc: bad arguments");
  if (int rc = check_cuda(cudaMalloc(ptr, bytes), "cudaMalloc")) return rc;
  return check_cuda(cudaMemset(*ptr, 0, bytes), "cudaMemset");
}

int dn_peer_free(void* ptr) { return ptr ? check_cuda(cudaFree(ptr), "cudaFree") : DN_OK; }

int dn_peer_export(void* ptr, unsigned char handle[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (!ptr || !handle) return fail(DN_EINVAL, "NULL pointer");
  cudaIpcMemHandle_t h;
  if (int rc = check_cuda(cudaIpcGetMemHandle(&h, ptr), "cudaIpcGetMemHandle")) return rc;
  memcpy(handle, &h, 64);
  return DN_OK;
}

int dn_peer_import(const unsigned char handle[64], void** ptr) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!ptr || !handle) return fail(DN_EINVAL, "NULL pointer");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  return check_cuda(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle");
}

int dn_peer_unimport(void* ptr) { return ptr ? check_cuda(cudaIpcCloseMemHandle(ptr), "cudaIpcCloseMemHandle") : DN_OK; }

int dn_peer_put_f32(float* dst_peer, const float* src, size_t n, int32_t* remote_flag, int32_t* local_counter,
                    uint32_t* ticket, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!dst_peer || !src || !remote_flag || !local_counter || !ticket) return fail(DN_EINVAL, "NULL pointer");
  if (n % 4 || (uintptr_t)dst_peer % 16 || (uintptr_t)src % 16)
    return fail(DN_EINVAL, "peer planes must be 16-byte aligned with n %% 4 == 0");
  return check_cuda(launch_peer_put(dst_peer, src, n, remote_flag, local_counter, ticket, (cudaStream_t)stream),
                    "peer_put launch");
}

int dn_peer_wait_f32(float* halo, const float* staged, size_t n, const int32_t* flag, int32_t* expect,
                     int64_t max_spins, int32_t* status, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!halo || !staged || !flag || !expect || !status) return fail(DN_EINVAL, "NULL pointer");
  if (n % 4 || (uintptr_t)halo % 16 || (uintptr_t)staged % 16)
    return fail(DN_EINVAL, "peer planes must be 16-byte aligned with n %% 4 == 0");
  return check_cuda(launch_peer_wait(halo, staged, n, flag, expect, max_spins > 0 ? max_spins : (1LL << 22), status,
                                     (cudaStream_t)stream), "peer_wait launch");
}

int dn_peer_allreduce_f32(const float* partial, float* out, double* slots, double* const* peer_slots, int rank,
                          int world, int32_t* counter, int64_t max_spins, int32_t* status, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!partial || !out || !slots || !peer_slots || !counter || !status) return fail(DN_EINVAL, "NULL pointer");
  if (world < 1 || world > 32 || rank < 0 || rank >= world) return fail(DN_EINVAL, "bad rank/world %d/%d", rank, world);
  return check_cuda(launch_peer_allreduce(partial, out, slots, peer_slots, rank, world, counter,
                                          max_spins > 0 ? max_spins : (1LL << 22), status, (cudaStream_t)stream),
                    "peer_allreduce launch");
}

int dn_scale_inplace_f32(float* x, size_t n, const float* factor_dev, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!x || !factor_dev) return fail(DN_EINVAL, "NULL pointer");
  if (n == 0) return DN_OK;
  return check_cuda(launch_scale(x, n, factor_dev, (cudaStream_t)stream), "scale launch");
}

int dn_scale_per_sample_f32(float* x, int batch, size_t n_per_sample, const float* factors_dev, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!x || !factors_dev) return fail(DN_EINVAL, "NULL pointer");
  if (batch < 1) return fail(DN_EINVAL, "batch=%d", batch);
  if (n_per_sample == 0) return DN_OK;
  return check_cuda(launch_scale_per_sample(x, batch, n_per_sample, factors_dev, (cudaStream_t)stream),
                    "scale_per_sample launch");
}

}  // extern "C"
