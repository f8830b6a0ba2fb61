// dn_api.cu -- extern "C" entry points of libdiffnet_fem.so (see include/diffnet_fem.h).
// Validation, constant folding, launch planning and template dispatch; no device state.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "dn_common.cuh"
#include "fem2d.cuh"
#include "fem2d_tma.cuh"
#include "fem3d.cuh"
#include "gp_eval.cuh"
#include "input_grads.cuh"

namespace dn {
int debug_plan3t(const dn_geom* g, int nfields, int has_nu, int64_t* out);
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

static int env_int(const char* name, int dflt) {
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

// 1-D Gauss rules with the reference's own (truncated) constants, DiffNetFEM.py:128-141.
static int gauss_rule(int n, double* x, double* w) {
  switch (n) {
    case 2: x[0] = -0.5773502691896258; x[1] = 0.5773502691896258; w[0] = w[1] = 1.0; return 0;
    case 3: x[0] = -0.774596669; x[1] = 0.0; x[2] = 0.774596669;
            w[0] = 5.0 / 9.0; w[1] = 8.0 / 9.0; w[2] = 5.0 / 9.0; return 0;
    case 4: x[0] = -0.861136; x[1] = -0.339981; x[2] = 0.339981; x[3] = 0.861136;
            w[0] = 0.347855; w[1] = 0.652145; w[2] = 0.652145; w[3] = 0.347855; return 0;
  }
  return -1;
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

struct Common {
  Field u, nu, f, fgp, numask;
  Mask mk[DN_MAX_MASKS];
  int nmasks, MK;
  Consts k;
  Rule rule;
  bool vec4;
};

static int prepare(const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                   const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask,
                   const dn_geom* g, double c_k, double c_f, double S, int nsd, Common* c, int flags = 0) {
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  if (g->nsd != nsd) return fail(DN_EINVAL, "geom.nsd=%d but the %d-D entry point was called", g->nsd, nsd);
  if (g->batch < 1 || g->nx < 2 || g->ny < 2 || (nsd == 3 && g->nz < 2))
    return fail(DN_EINVAL, "need batch >= 1 and >= 2 nodes per direction (B=%d nx=%d ny=%d nz=%d)",
                g->batch, g->nx, g->ny, g->nz);
  if (!(g->hx > 0) || !(g->hy > 0) || (nsd == 3 && !(g->hz > 0)))
    return fail(DN_EINVAL, "element sizes must be positive");
  if (!u || !u->ptr) return fail(DN_EINVAL, "u is NULL");
  if (f && f->ptr && fgp && fgp->ptr) return fail(DN_EINVAL, "give f or fgp, not both");
  if ((flags & DN_F_LOAD_VECTOR) && !(f && f->ptr)) return fail(DN_EINVAL, "DN_F_LOAD_VECTOR needs the load vector in f");
  if (nmasks < 0 || nmasks > DN_MAX_MASKS)
    return fail(DN_EINVAL, "nmasks=%d (max %d)", nmasks, DN_MAX_MASKS);
  if (nmasks > 0 && !masks) return fail(DN_EINVAL, "masks is NULL");
  double gx[4], gw[4];
  if (gauss_rule(g->ngp_1d, gx, gw)) return fail(DN_EINVAL, "ngp_1d=%d (2..4)", g->ngp_1d);

  c->u = to_field(u); c->nu = to_field(nu); c->f = to_field(f); c->fgp = to_field(fgp);
  c->numask = to_field(nu_zero_mask);
  if (c->numask.p && !c->nu.p) return fail(DN_EINVAL, "nu_zero_mask needs nu");
  c->nmasks = nmasks;
  int nvf = 0;
  for (int i = 0; i < DN_MAX_MASKS; ++i) c->mk[i] = Mask{{nullptr, 0, 0, 0}, {nullptr, 0, 0, 0}, 0.f};
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

  // rule moments: W1 = sum w, t = sum w x^2 / W1
  double W1 = 0, m2 = 0;
  for (int i = 0; i < g->ngp_1d; ++i) { W1 += gw[i]; m2 += gw[i] * gx[i] * gx[i]; }
  const double t = m2 / W1;
  const double Wn = (nsd == 2) ? W1 * W1 : W1 * W1 * W1;
  const double nrm = (nsd == 2) ? 64.0 : 512.0;     // (2^nsd)^2 from un-normalised C * A^2
  c->k.kx = (float)(S * c_k * Wn * (2.0 / g->hx) * (2.0 / g->hx) / nrm);
  c->k.ky = (float)(S * c_k * Wn * (2.0 / g->hy) * (2.0 / g->hy) / nrm);
  c->k.kz = (nsd == 3) ? (float)(S * c_k * Wn * (2.0 / g->hz) * (2.0 / g->hz) / nrm) : 0.f;
  c->k.kf = (float)(S * c_f * Wn / ((nsd == 2) ? 16.0 : 64.0));
  c->k.t = (float)t;
  c->k.kb = (float)(S * c_f);
  c->k.lv = (flags & DN_F_LOAD_VECTOR) ? 1 : 0;
  c->rule.n = g->ngp_1d;
  for (int i = 0; i < 4; ++i) {
    c->rule.x[i] = i < g->ngp_1d ? (float)gx[i] : 0.f;
    c->rule.w[i] = i < g->ngp_1d ? (float)gw[i] : 0.f;
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

// ------------------------------------------------------------------------------------ 2-D
struct Plan2D { int V, R, nchunks, ntx, nitems, wpc, grid; };

static Plan2D plan2d(const dn_geom* g, bool vec4, int sms) {
  Plan2D pl;
  pl.V = vec4 ? 4 : 1;
  pl.ntx = (g->nx + 32 * pl.V - 1) / (32 * pl.V);
  // enough warps to give every SM ~16, but chunks of at least 8 rows (halo rows are re-read
  // from L2 and their elements recomputed: (R+1)/R work, (R+2)/R loads)
  const long long target = (long long)sms * env_int("DN_WARPS_PER_SM_2D", 16);
  long long per_row_items = (long long)g->batch * pl.ntx;
  long long want = (target + per_row_items - 1) / per_row_items;
  if (want < 1) want = 1;
  int R = (int)((g->ny + want - 1) / want);
  const int Rmin = env_int("DN_RMIN_2D", 8);
  if (R < Rmin) R = Rmin;
  if (R > g->ny) R = g->ny;
  R = env_int("DN_R_2D", R);
  pl.R = R;
  pl.nchunks = (g->ny + R - 1) / R;
  pl.nitems = g->batch * pl.nchunks * pl.ntx;
  pl.wpc = env_int("DN_WPC_2D", pl.ntx == 2 ? 2 : 4);
  pl.grid = (pl.nitems + pl.wpc - 1) / pl.wpc;
  return pl;
}

static size_t ws_bytes_for_grid(long long grid) { return 64 + 8 * (size_t)grid; }

// ---- streaming (bulk-async) 2-D path -------------------------------------------------------
struct Plan2T { int ok, threads, S, R, nchunks, nf, bal_q, bal_rem; long long grid; size_t smem; };

static size_t smem_2t(int S, int nf, int nx, int threads) {
  return (size_t)S * nf * 2 * nx * 4 + 16 + (size_t)S * 8 + 4 * (size_t)(threads / 32) * 4;
}

// Eligibility + launch shape.  `occ` (resident CTAs per SM) may be null: then only the upper
// bound of the grid matters (workspace sizing).
static Plan2T plan2t(const dn_geom* g, int nf, int sms, occ2t_fn occ) {
  Plan2T pl;
  memset(&pl, 0, sizeof(pl));
  if (g->nx % 4 != 0 || g->nx < 8) return pl;
  const int lanes = g->nx / 4;
  pl.threads = (lanes + 31) / 32 * 32;
  if (pl.threads > DN_T2_MAXT) return pl;
  pl.nf = nf;
  int S = env_int("DN_T2_STAGES", 2);           // stages of two node rows each
  if (S < 2) S = 2;
  if (S > 16) S = 16;
  while (S > 2 && smem_2t(S, nf, g->nx, pl.threads) > (size_t)64 * 1024) --S;   // keep >= 3 CTAs/SM
  pl.S = S;
  pl.smem = smem_2t(S, nf, g->nx, pl.threads);
  if (pl.smem > (size_t)kMaxDynSmem) return pl;
  int cps = occ ? occ(pl.threads, pl.smem) : 8;
  if (cps < 1) return pl;
  const int cap = env_int("DN_T2_CPS", 0);
  if (cap > 0 && cps > cap) cps = cap;
  // one wave: B * nchunks <= resident slots, chunks of >= Rmin rows (halo rows are re-read
  // from L2 and their element row recomputed: (R+2)/R reads, (R+1)/R arithmetic)
  const long long slots = (long long)sms * cps;
  long long nch = slots / g->batch;
  if (nch < 1) nch = 1;
  int R = (int)((g->ny + nch - 1) / nch);
  int Rmin = env_int("DN_T2_RMIN", 8);
  if (Rmin < 4) Rmin = 4;
  if (R < Rmin) R = Rmin;
  // with more work than one wave, long chunks stop paying: 32-row chunks in several waves measured
  // 0.85 (B = 256) and 0.96 (B = 1024) of the HBM peak against 0.77 / 0.93 for one wave of 64- /
  // 256-row chunks (fewer, longer-lived CTAs expose every ring refill)
  const int Rmax = env_int("DN_T2_RMAX", 32);
  if (R > Rmax && Rmax >= Rmin) R = Rmax;
  const int Rforced = env_int("DN_T2_R", 0);
  if (Rforced > 0) R = Rforced;
  if (R < 4) R = 4;
  if (R > g->ny) R = g->ny;
  pl.R = R;
  pl.nchunks = (g->ny + R - 1) / R;
  pl.grid = (long long)g->batch * pl.nchunks;
  // One wave, balanced: uniform R-row chunks leave a short last chunk per image (256 rows / 15 -> 17 chunks + a
  // 1-row chunk) and fewer CTAs than slots (1152 of 1184: 32 SMs run 7 CTAs, the rest 8 -- the kernel ends with the
  // busiest SM).  Instead every slot gets one CTA: the first `rem` images are cut into q + 1 chunks, the others into
  // q, each image into equal parts (rows differ by at most one).
  if (Rforced <= 0 && env_int("DN_T2_BALANCE", 1) && pl.grid <= slots && slots <= (long long)g->batch * (g->ny / Rmin)) {
    long long q = slots / g->batch, rem = slots % g->batch;
    // Measured (256^2 x 64 and 512^2 x 16, sweeps of the chunk count): the best one-wave shape fills ~70 % of the
    // resident slots (13 / 26 chunks per image: 0.72 / 0.73 of the HBM peak against 0.70 / 0.72 with every slot
    // taken) -- fewer CTAs per SM make every stage round shorter and the longer chunks have fewer seams.
    const int fill = env_int("DN_T2_FILL_PCT", 70);
    if (fill > 0 && fill < 100) {
      const long long q2 = (slots * fill / 100 + g->batch / 2) / g->batch;
      if (q2 >= 1 && g->ny / (q2 + 1) >= Rmin && (g->ny + q2 - 1) / q2 <= Rmax) { q = q2; rem = 0; }
    }
    const int qf = env_int("DN_T2_Q", 0);            // experiments: exactly qf equal chunks per image
    if (qf > 0 && qf <= slots / g->batch) { q = qf; rem = 0; }
    if (q >= 1 && g->ny / (q + 1) >= Rmin && (g->ny + q - 1) / q <= Rmax) {
      pl.bal_q = (int)q; pl.bal_rem = (int)rem;
      pl.grid = q * g->batch + rem;
      pl.nchunks = (int)q + (rem ? 1 : 0);
      pl.R = (int)((g->ny + q - 1) / q);
    }
  }
  pl.ok = 1;
  return pl;
}

static int run2t(const Common& c, const dn_geom* g, float* grad, int mode, int mask_input, void* workspace,
                 size_t wsb, double* loss_out, float* loss_f32, void* stream, int sms, bool* handled) {
  *handled = false;
  const char* path = getenv("DN_2D_PATH");
  if (path && !strcmp(path, "warp")) return DN_OK;
  if (!c.vec4 || c.fgp.p || ((uintptr_t)grad % 16 != 0)) return DN_OK;
  const int NU = c.nu.p ? 1 : 0, F = c.f.p ? (c.k.lv ? 2 : 1) : 0, NMK = c.numask.p ? 1 : 0;
  if (g->nx % 4 != 0 || g->nx / 4 > DN_T2_MAXT) return DN_OK;
  int MKx = c.MK;
  if (!mask_input) {                     // operator apply: only the plain-mask, no-source variants exist
    if (c.MK == 0) MKx = 0;              // nothing to substitute anyway
    else if (c.MK >= 1 && c.MK <= 3 && !F && !NMK) MKx = c.MK + 4;
    else return DN_OK;
  }
  launch2t_fn fn = get_launch2t(MKx, NU, F, NMK);
  occ2t_fn occ = get_occ2t(MKx, NU, F, NMK);
  if (!fn || !occ) return DN_OK;
  P2T p;
  memset(&p, 0, sizeof(p));
  int nf = 0;
  p.fld[nf++] = c.u;
  if (NU) p.fld[nf++] = c.nu;
  if (F) p.fld[nf++] = c.f;
  if (NMK) p.fld[nf++] = c.numask;
  for (int i = 0; i < c.nmasks; ++i) { p.fld[nf++] = c.mk[i].m; p.mval[i] = c.mk[i].v; }
  if (c.MK == 4) p.fld[nf++] = c.mk[0].vf;
  for (int i = 0; i < nf; ++i)
    if (p.fld[i].sy != g->nx) return DN_OK;      // bulk copies take whole runs of rows
  Plan2T pl = plan2t(g, nf, sms, occ);
  if (!pl.ok) { cudaGetLastError(); return DN_OK; }
  if (pl.grid > 0x7fffffffLL) return DN_OK;
  if (!workspace || wsb < ws_bytes_for_grid(pl.grid))
    return fail(DN_EWORKSPACE, "workspace too small: %zu < %zu", wsb, ws_bytes_for_grid(pl.grid));
  if ((uintptr_t)workspace % 16) return fail(DN_EWORKSPACE, "workspace must be 16-byte aligned");
  p.nf = nf;
  p.B = g->batch; p.nx = g->nx; p.ny = g->ny;
  p.R = pl.R; p.nchunks = pl.nchunks; p.S = pl.S;
  p.bal_q = pl.bal_q; p.bal_rem = pl.bal_rem;
  const float kx = c.k.kx, ky = c.k.ky, kf = c.k.kf, t = c.k.t;
  p.k2.kx = make_float2(kx, kx); p.k2.ky = make_float2(ky, ky); p.k2.t = make_float2(t, t);
  p.k2.kxt = make_float2(kx * t, kx * t); p.k2.kyt = make_float2(ky * t, ky * t);
  // nodal source stencil (FK == 1): 1-D element mass [[1+t, 1-t], [1-t, 1+t]] in x (times -kf) and in y
  const float fc = 1.f - t, fw = 2.f * (1.f + t);
  p.k2.nfc = make_float2(-kf * fc, -kf * fc); p.k2.nfw = make_float2(-kf * fw, -kf * fw);
  p.k2.yc = make_float2(fc, fc); p.k2.yw = make_float2(fw, fw);
  p.k2.fmir = make_float2(-(1.f + t) / fc, -(1.f + t) / fc);
  p.k2.c0x_const = make_float2(4.f * kx, 4.f * kx); p.k2.c0y_const = make_float2(4.f * ky, 4.f * ky);
  p.k2.nkb = make_float2(-c.k.kb, -c.k.kb);
  p.grad = grad;
  p.red.counter = (unsigned int*)workspace;
  p.red.partials = (double*)((char*)workspace + 64);
  p.red.loss_out = loss_out; p.red.loss_f32 = loss_f32;
  p.mode = mode;
  *handled = true;
  return check_cuda(fn(p, dim3((unsigned)pl.grid), dim3(pl.threads), pl.smem, (cudaStream_t)stream),
                    "fem2d_tma launch");
}

static int run2d(const Common& c, const dn_geom* g, float* grad, float* grad_nu, int mode,
                 int mask_input, void* workspace, size_t wsb, double* loss_out, float* loss_f32,
                 void* stream, int sms) {
  if (!grad_nu) {   // streaming path: common aligned cases (the rest stays on k_fem2d)
    bool handled = false;
    int rc = run2t(c, g, grad, mode, mask_input, workspace, wsb, loss_out, loss_f32, stream, sms, &handled);
    if (rc != DN_OK || handled) return rc;
  }
  if (c.k.lv)
    return fail(DN_ENOSTREAM, "DN_F_LOAD_VECTOR: the streaming 2-D kernel cannot take this launch (nx %% 4, nx <= %d, "
                "16-byte aligned dense rows, no grad_nu); pass f_gp instead", 4 * DN_T2_MAXT);
  bool vec4 = c.vec4 && ((uintptr_t)grad % 16 == 0) && ((uintptr_t)grad_nu % 16 == 0);
  Plan2D pl = plan2d(g, vec4, sms);
  if (!workspace || wsb < ws_bytes_for_grid(pl.grid))
    return fail(DN_EWORKSPACE, "workspace too small: %zu < %zu", wsb, ws_bytes_for_grid(pl.grid));
  if ((uintptr_t)workspace % 16) return fail(DN_EWORKSPACE, "workspace must be 16-byte aligned");
  P2D p;
  memset(&p, 0, sizeof(p));
  p.u = c.u; p.nu = c.nu; p.f = c.f; p.fgp = c.fgp; p.numask = c.numask;
  for (int i = 0; i < DN_MAX_MASKS; ++i) p.mk[i] = c.mk[i];
  p.B = g->batch; p.nx = g->nx; p.ny = g->ny;
  p.k = c.k; p.rule = c.rule;
  p.R = pl.R; p.nchunks = pl.nchunks; p.ntx = pl.ntx; p.nitems = pl.nitems;
  p.grad = grad; p.grad_nu = grad_nu;
  p.red.counter = (unsigned int*)workspace;
  p.red.partials = (double*)((char*)workspace + 64);
  p.red.loss_out = loss_out; p.red.loss_f32 = loss_f32;
  p.mode = mode; p.mask_input = mask_input;
  const int FM = c.f.p ? 1 : (c.fgp.p ? 2 : 0);
  launch2d_fn fn = get_launch2d(pl.V, c.MK, c.nu.p ? 1 : 0, FM, c.numask.p ? 1 : 0, grad_nu ? 1 : 0);
  if (!fn)
    return fail(DN_EINVAL, "unsupported option combination (V=%d MK=%d nu=%d fmode=%d numask=%d grad_nu=%d)",
                pl.V, c.MK, c.nu.p ? 1 : 0, FM, c.numask.p ? 1 : 0, grad_nu ? 1 : 0);
  return check_cuda(fn(p, dim3(pl.grid), dim3(32 * pl.wpc), (cudaStream_t)stream), "fem2d launch");
}

}  // namespace dn

using namespace dn;

extern "C" {

static int gp_common(const dn_geom* g, int which, int nsd, GpTables* tb);

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
  long long worst = 0;
  if (g->nsd == 2) {
    for (int v = 0; v < 2; ++v) {
      Plan2D pl = plan2d(g, v == 1, sms);
      if (pl.nitems > worst) worst = pl.nitems;
    }
    const long long t2 = (long long)g->batch * ((g->ny + 3) / 4);   // streaming path, R >= 4
    if (t2 > worst) worst = t2;
  } else {
    worst = plan3d_max_ctas(g);
  }
  return ws_bytes_for_grid(worst + 1024);
}

int dn_debug_plan(const dn_geom* g, int nfields, int has_nu, int64_t out[16]) {
  if (!g || !out) return fail(DN_EINVAL, "NULL pointer");
  for (int i = 0; i < 16; ++i) out[i] = 0;
  if (nfields < 1 || nfields > DN_T2_MAXF) return fail(DN_EINVAL, "nfields=%d", nfields);
  if (g->nsd == 2) {
    Plan2T pl = plan2t(g, nfields, 148, nullptr);
    out[0] = pl.ok;
    if (pl.ok) {
      out[1] = pl.threads; out[2] = pl.grid; out[3] = (int64_t)pl.smem; out[4] = pl.S;
      out[5] = pl.R; out[6] = pl.nchunks; out[7] = pl.bal_q; out[8] = pl.bal_rem;
    }
    return DN_OK;
  }
  if (g->nsd == 3) return debug_plan3t(g, nfields, has_nu, out);
  return fail(DN_EINVAL, "nsd=%d", g->nsd);
}

int dn_fem_energy_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                         const dn_field* fgp, const dn_mask* masks, int nmasks,
                         const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                         float* grad_u, float* grad_nu, void* workspace, size_t workspace_bytes,
                         double* loss_out, float* loss_out_f32, void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!c) return fail(DN_EINVAL, "consts is NULL");
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  const double count = (c->reduction == 0)
      ? (g->mean_count > 0 ? g->mean_count : (double)g->batch * (g->nx - 1) * (double)(g->ny - 1))
      : 1.0;
  Common cm;
  if (int rc = prepare(u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, c->c_k, c->c_f,
                       c->scale / count, 2, &cm, c->flags)) return rc;
  if (grad_nu && !cm.nu.p) return fail(DN_EINVAL, "grad_nu requested without nu");
  return run2d(cm, g, grad_u, grad_nu, 0, 1, workspace, workspace_bytes, loss_out, loss_out_f32,
               stream, sms);
}

int dn_fem_residual_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                           const dn_mask* masks, int nmasks, int apply_masks_to_input,
                           const dn_geom* g, double jac, float* residual, void* workspace,
                           size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                           void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!residual) return fail(DN_EINVAL, "residual output is NULL");
  Common cm;
  // R = d/du [ sum_e sum_g jac w_g ( 1/2 nu |grad u|^2 - u f ) ]
  if (int rc = prepare(u, nu, f, nullptr, masks, nmasks, nullptr, g, 0.5 * jac, jac, 1.0, 2, &cm))
    return rc;
  return run2d(cm, g, residual, nullptr, 1, apply_masks_to_input ? 1 : 0, workspace,
               workspace_bytes, loss_out, loss_out_f32, stream, sms);
}

int dn_fem_energy_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                         const dn_field* fgp, const dn_mask* masks, int nmasks,
                         const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                         float* grad_u, float* grad_nu, void* workspace, size_t workspace_bytes,
                         double* loss_out, float* loss_out_f32, void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!c) return fail(DN_EINVAL, "consts is NULL");
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  double count = 1.0;
  if (c->reduction == 0) {
    long long nelz = g->nz - 1;
    if (g->z_own_hi > g->z_own_lo) {
      const int hi = g->z_own_hi < g->nz - 1 ? g->z_own_hi : g->nz - 1;
      nelz = hi - g->z_own_lo;
    }
    count = g->mean_count > 0 ? g->mean_count
                              : (double)g->batch * (g->nx - 1) * (double)(g->ny - 1) * (double)nelz;
  }
  Common cm;
  if (int rc = prepare(u, nu, f, fgp, masks, nmasks, nu_zero_mask, g, c->c_k, c->c_f,
                       c->scale / count, 3, &cm, c->flags)) return rc;
  if (grad_nu && !cm.nu.p) return fail(DN_EINVAL, "grad_nu requested without nu");
  if (int rc = run3d(cm.u, cm.nu, cm.f, cm.fgp, cm.numask, cm.mk, cm.MK, cm.k, cm.rule, cm.vec4, g,
                     grad_u, 0, 1, workspace, workspace_bytes, loss_out, loss_out_f32, stream, sms)) return rc;
  if (grad_nu) {        // dL/dnu: a separate gather launch (gp_eval.cu: k_grad_nu_3d)
    GradNu3 q;
    memset(&q, 0, sizeof(q));
    q.u = cm.u; q.numask = cm.numask;
    for (int i = 0; i < DN_MAX_MASKS; ++i) q.mk[i] = cm.mk[i];
    q.nmasks = cm.nmasks; q.has_vf = (cm.MK == 4) ? 1 : 0;
    q.B = g->batch; q.nx = g->nx; q.ny = g->ny; q.nz = g->nz; q.ng = g->ngp_1d;
    q.zlo = 0; q.zhi = g->nz - 1;
    if (g->z_own_hi > g->z_own_lo) { q.zlo = g->z_own_lo; q.zhi = g->z_own_hi < g->nz - 1 ? g->z_own_hi : g->nz - 1; }
    q.coef = (float)(c->scale / count * c->c_k);
    double gx[4], gw[4];
    gauss_rule(g->ngp_1d, gx, gw);
    for (int i = 0; i < 4; ++i) q.w[i] = i < g->ngp_1d ? (float)gw[i] : 0.f;
    for (int w = 0; w < 4; ++w)
      if (int rc = gp_common(g, w, 3, &q.tb[w])) return rc;
    return check_cuda(launch_grad_nu_3d(q, grad_nu, (cudaStream_t)stream), "grad_nu launch");
  }
  return DN_OK;
}

int dn_fem_energy_3d_linked_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask,
                                const dn_geom* g, const dn_consts* c, const dn_slab_link* link,
                                float* grad_u, void* workspace, size_t workspace_bytes,
                                double* loss_out, float* loss_out_f32, void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!c || !g || !link) return fail(DN_EINVAL, "consts / geom / link is NULL");
  double count = 1.0;
  if (c->reduction == 0) {
    long long nelz = g->nz - 1;
    if (g->z_own_hi > g->z_own_lo) {
      const int hi = g->z_own_hi < g->nz - 1 ? g->z_own_hi : g->nz - 1;
      nelz = hi - g->z_own_lo;
    }
    count = g->mean_count > 0 ? g->mean_count
                              : (double)g->batch * (g->nx - 1) * (double)(g->ny - 1) * (double)nelz;
  }
  Common cm;
  if (int rc = prepare(u, nu, f, nullptr, masks, nmasks, nu_zero_mask, g, c->c_k, c->c_f,
                       c->scale / count, 3, &cm)) return rc;
  return run3d(cm.u, cm.nu, cm.f, cm.fgp, cm.numask, cm.mk, cm.MK, cm.k, cm.rule, cm.vec4, g,
               grad_u, 0, 1, workspace, workspace_bytes, loss_out, loss_out_f32, stream, sms, link);
}

int dn_peer_loss_sum_f32(const double* slots, int world, const int32_t* step, int64_t max_spins,
                         int32_t* status, float* out, void* stream) {
  if (int rc = device_ok(nullptr)) return rc;
  if (!slots || !step || !status || !out) return fail(DN_EINVAL, "NULL pointer");
  if (world < 1 || world > 32) return fail(DN_EINVAL, "world %d (1..32)", world);
  return check_cuda(launch_peer_loss_sum(slots, world, step, max_spins > 0 ? max_spins : (1LL << 26), status, out,
                                         (cudaStream_t)stream), "peer_loss_sum launch");
}

int dn_fem_residual_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                           const dn_mask* masks, int nmasks, int apply_masks_to_input,
                           const dn_geom* g, double jac, float* residual, void* workspace,
                           size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                           void* stream) {
  int sms = 0;
  if (int rc = device_ok(&sms)) return rc;
  if (!residual) return fail(DN_EINVAL, "residual output is NULL");
  Common cm;
  if (int rc = prepare(u, nu, f, nullptr, masks, nmasks, nullptr, g, 0.5 * jac, jac, 1.0, 3, &cm))
    return rc;
  return run3d(cm.u, cm.nu, cm.f, cm.fgp, cm.numask, cm.mk, cm.MK, cm.k, cm.rule, cm.vec4, g,
               residual, 1, apply_masks_to_input ? 1 : 0, workspace, workspace_bytes, loss_out,
               loss_out_f32, stream, sms);
}

// ------------------------------------------------------------------------------------ input gradients
static double mean_count(const dn_geom* g, int nsd, int reduction) {
  if (reduction != 0) return 1.0;
  if (g->mean_count > 0) return g->mean_count;
  return (double)g->batch * (g->nx - 1) * (double)(g->ny - 1) * (nsd == 3 ? (double)(g->nz - 1) : 1.0);
}

static int ingrad_common(int nsd, const dn_field* u, const dn_field* nu, const dn_field* f, const dn_field* fgp,
                         const dn_mask* masks, int nmasks, const dn_geom* g, float* const* grad_values, InGrad* q) {
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  if (g->nsd != nsd) return fail(DN_EINVAL, "geom.nsd=%d but the %d-D entry point was called", g->nsd, nsd);
  if (g->batch < 1 || g->nx < 2 || g->ny < 2 || (nsd == 3 && g->nz < 2))
    return fail(DN_EINVAL, "need batch >= 1 and >= 2 nodes per direction (B=%d nx=%d ny=%d nz=%d)",
                g->batch, g->nx, g->ny, g->nz);
  if (!(g->hx > 0) || !(g->hy > 0) || (nsd == 3 && !(g->hz > 0)))
    return fail(DN_EINVAL, "element sizes must be positive");
  if (g->z_own_hi > g->z_own_lo)
    return fail(DN_EINVAL, "input gradients are not available under z-slab ownership (z_own_lo/hi set): a slab "
                           "would only hold a partial gradient");
  if (!u || !u->ptr) return fail(DN_EINVAL, "u is NULL");
  if (nmasks < 0 || nmasks > DN_MAX_MASKS) return fail(DN_EINVAL, "nmasks=%d (max %d)", nmasks, DN_MAX_MASKS);
  if (nmasks > 0 && !masks) return fail(DN_EINVAL, "masks is NULL");
  double gx[4], gw[4];
  if (gauss_rule(g->ngp_1d, gx, gw)) return fail(DN_EINVAL, "ngp_1d=%d (2..4)", g->ngp_1d);
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
  double W1 = 0, m2 = 0;
  for (int i = 0; i < 4; ++i) {
    q->x[i] = i < g->ngp_1d ? (float)gx[i] : 0.f;
    q->w[i] = i < g->ngp_1d ? (float)gw[i] : 0.f;
    if (i < g->ngp_1d) { W1 += gw[i]; m2 += gw[i] * gx[i] * gx[i]; }
  }
  const double t = m2 / W1;
  q->ma = (float)(0.25 * W1 * (1.0 + t));
  q->mc = (float)(0.25 * W1 * (1.0 - t));
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
  q.numask = to_field(nu_zero_mask);
  if (q.numask.p && !q.nu.p) return fail(DN_EINVAL, "nu_zero_mask needs nu");
  if (grad_f && !q.f.p) return fail(DN_EINVAL, "grad_f requested without f");
  if (grad_fgp && !q.fgp) return fail(DN_EINVAL, "grad_fgp requested without fgp");
  const double S = c->scale / mean_count(g, nsd, c->reduction);
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

static int gp_common(const dn_geom* g, int which, int nsd, GpTables* tb) {
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  if (g->nsd != nsd) return fail(DN_EINVAL, "geom.nsd mismatch");
  if (g->batch < 1 || g->nx < 2 || g->ny < 2 || (nsd == 3 && g->nz < 2))
    return fail(DN_EINVAL, "need >= 2 nodes per direction");
  if (which < 0 || which > (nsd == 2 ? 2 : 3)) return fail(DN_EINVAL, "which=%d", which);
  double gx[4], gw[4];
  if (gauss_rule(g->ngp_1d, gx, gw)) return fail(DN_EINVAL, "ngp_1d=%d (2..4)", g->ngp_1d);
  // 1-D factors per Gauss point: value table N1[gp][bf] and derivative table D1[bf] * (2/h).
  // The reference stores the fp32 rounding of the f64 product including 2/h
  // (DiffNetFEM.py:198-215, 405-453); the separable evaluation here agrees to 1 ulp-ish.
  tb->n = g->ngp_1d;
  const double s[3] = {2.0 / g->hx, 2.0 / g->hy, nsd == 3 ? 2.0 / g->hz : 0.0};
  for (int d = 0; d < 3; ++d) {
    const bool der = (which == d + 1);
    for (int q = 0; q < 4; ++q) {
      const double x = q < g->ngp_1d ? gx[q] : 0.0;
      tb->c[d][q][0] = (float)(der ? -0.5 * s[d] : 0.5 * (1.0 - x));
      tb->c[d][q][1] = (float)(der ? +0.5 * s[d] : 0.5 * (1.0 + x));
    }
  }
  return DN_OK;
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
  if (!g) return fail(DN_EINVAL, "geom is NULL");
  if (!fgp || !fgp->ptr || !out) return fail(DN_EINVAL, "load_vector: NULL input/output");
  if ((g->nsd != 2 && g->nsd != 3) || g->batch < 1 || g->nx < 2 || g->ny < 2 || (g->nsd == 3 && g->nz < 2))
    return fail(DN_EINVAL, "load_vector: nsd 2 or 3, batch >= 1, >= 2 nodes per direction");
  double gx[4], gw[4];
  if (gauss_rule(g->ngp_1d, gx, gw)) return fail(DN_EINVAL, "ngp_1d=%d (2..4)", g->ngp_1d);
  // b = N^T (w f_gp): the transpose of the Gauss-point interpolation with the quadrature weights folded into the
  // 1-D factors -- the tuned adjoint kernels (gp_eval.cu) do the assembly
  GpMultiAdj m;
  memset(&m, 0, sizeof(m));
  m.nw = 1;
  m.tb[0].n = g->ngp_1d;
  for (int d = 0; d < 3; ++d)
    for (int i = 0; i < g->ngp_1d; ++i) {
      m.tb[0].c[d][i][0] = (float)(gw[i] * 0.5 * (1.0 - gx[i]));
      m.tb[0].c[d][i][1] = (float)(gw[i] * 0.5 * (1.0 + gx[i]));
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

}  // extern "C"
