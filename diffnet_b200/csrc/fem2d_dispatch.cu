// Launch planning and runtime -> compile-time dispatch of the 2-D kernel family (instantiated by fem2d_inst.cu).
#include "dn_launch.h"
#include "fem2d.cuh"
#include "fem2d_combos.h"
namespace dn {

// The kernel of a variant of fem2d_combos.h, or null when it is not instantiated.
static Kernel* find2d(int V, int MK, int NU, int FM, int NUMASK, int GN) {
  static struct { int V, MK, NU, FM, NUMASK, GN; Kernel k; } tab[] = {
#define DN_ROW(V_, MK_, NU_, FM_, NMK_, GN_) {V_, MK_, NU_, FM_, NMK_, GN_, {kernel2d<V_, MK_, NU_, FM_, NMK_, GN_>()}},
      DN2D_ALL(DN_ROW)
#undef DN_ROW
  };
  for (auto& r : tab)
    if (r.V == V && r.MK == MK && r.NU == NU && r.FM == FM && r.NUMASK == NUMASK && r.GN == GN) return &r.k;
  return nullptr;
}

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

long long plan2d_max_ctas(const dn_geom* g, int sms) {
  long long worst = 0;
  for (int v = 0; v < 2; ++v) {      // grids are <= items
    Plan2D pl = plan2d(g, v == 1, sms);
    if (pl.nitems > worst) worst = pl.nitems;
  }
  const long long t2 = (long long)g->batch * ((g->ny + 3) / 4);   // streaming path, R >= 4
  return t2 > worst ? t2 : worst;
}

int run2d(const Common& c, const dn_geom* g, const Out& o) {
  if (!o.grad_nu) {   // streaming path: common aligned cases (the rest stays on k_fem2d)
    bool handled = false;
    int rc = run2t(c, g, o, &handled);
    if (rc != DN_OK || handled) return rc;
  }
  if (c.k.lv)
    return fail(DN_ENOSTREAM, "DN_F_LOAD_VECTOR: the streaming 2-D kernel cannot take this launch (nx %% 4, nx <= %d, "
                "16-byte aligned dense rows, no grad_nu); pass f_gp instead", 4 * DN_T2_MAXT);
  bool vec4 = c.vec4 && ((uintptr_t)o.grad % 16 == 0) && ((uintptr_t)o.grad_nu % 16 == 0);
  Plan2D pl = plan2d(g, vec4, c.sms);
  P2D p;
  memset(&p, 0, sizeof(p));
  // reduction = none: one slot per item (warp), not per CTA -- the wpc items of a CTA can span two samples
  if (int rc = reduce_into(c, o, g, pl.grid, pl.ntx * pl.nchunks, 0, &p.red)) return rc;
  p.u = c.u; p.nu = c.nu; p.f = c.f; p.fgp = c.fgp; p.numask = c.numask;
  for (int i = 0; i < DN_MAX_MASKS; ++i) p.mk[i] = c.mk[i];
  p.B = g->batch; p.nx = g->nx; p.ny = g->ny;
  p.k = c.k; p.rule = c.rule;
  p.R = pl.R; p.nchunks = pl.nchunks; p.ntx = pl.ntx; p.nitems = pl.nitems;
  p.grad = o.grad; p.grad_nu = o.grad_nu;
  p.mode = c.mode; p.mask_input = c.mask_input;
  const int FM = c.f.p ? 1 : (c.fgp.p ? 2 : 0);
  Kernel* k = find2d(pl.V, c.MK, c.nu.p ? 1 : 0, FM, c.numask.p ? 1 : 0, o.grad_nu ? 1 : 0);
  if (!k)
    return fail(DN_EINVAL, "unsupported option combination (V=%d MK=%d nu=%d fmode=%d numask=%d grad_nu=%d)",
                pl.V, c.MK, c.nu.p ? 1 : 0, FM, c.numask.p ? 1 : 0, o.grad_nu ? 1 : 0);
  return check_cuda(launch(*k, &p, dim3(pl.grid), dim3(32 * pl.wpc), 0, (cudaStream_t)o.stream, false),
                    "fem2d launch");
}

}  // namespace dn
