// Launch planning and runtime -> compile-time dispatch of the 3-D kernel family (instantiated by fem3d_inst.cu).
#include "dn_launch.h"
#include "fem3d.cuh"
#include "fem3d_combos.h"

namespace dn {

// The kernel of a variant of fem3d_combos.h, or null when it is not instantiated.
static Kernel* find3d(int V, int MK, int NU, int FM, int NUMASK) {
  static struct { int V, MK, NU, FM, NUMASK; Kernel k; } tab[] = {
#define DN_ROW(V_, MK_, NU_, FM_, NMK_) {V_, MK_, NU_, FM_, NMK_, {kernel3d<V_, MK_, NU_, FM_, NMK_>()}},
      DN3D_ALL(DN_ROW)
#undef DN_ROW
  };
  for (auto& r : tab)
    if (r.V == V && r.MK == MK && r.NU == NU && r.FM == FM && r.NUMASK == NUMASK) return &r.k;
  return nullptr;
}

struct Plan3D { int V, LX, TY, ZC, ntx, nty, nzc; long long grid; size_t smem; };

static Plan3D plan3d(const dn_geom* g, bool vec4, int sms) {
  Plan3D pl;
  pl.V = vec4 ? 4 : 1;
  const int nxv = (g->nx + pl.V - 1) / pl.V;           // lane columns per row
  const int lxmax = env_int("DN_LXMAX_3D", 64);
  if (nxv <= lxmax) { pl.LX = nxv; pl.ntx = 1; }
  else {
    pl.ntx = (nxv - 1 + (lxmax - 2)) / (lxmax - 1);
    pl.LX = (nxv - 1 + pl.ntx - 1) / pl.ntx + 1;
    pl.ntx = (nxv - 1 + (pl.LX - 2)) / (pl.LX - 1);
  }
  // rows: fill ~DN_THREADS_3D threads; at least 2 compute rows
  const int target = env_int("DN_THREADS_3D", 288);
  int rows = target / pl.LX;
  if (rows < 3) rows = 3;
  if (rows * pl.LX > DN_MAXT_3D) rows = DN_MAXT_3D / pl.LX;
  if (rows > g->ny) rows = g->ny;                       // one tile covers all rows
  if (rows < 2) rows = 2;
  rows = env_int("DN_ROWS_3D", rows);
  pl.TY = rows - 1;
  pl.nty = (pl.TY >= g->ny - 1) ? 1 : ((g->ny - 1) + (pl.TY - 2)) / (pl.TY - 1);
  // z chunks: aim at >= 2 CTAs per SM, chunks of at least 4 planes
  const long long tiles = (long long)g->batch * pl.ntx * pl.nty;
  long long want = ((long long)sms * env_int("DN_CTAS_PER_SM_3D", 2) + tiles - 1) / tiles;
  if (want < 1) want = 1;
  int ZC = (int)((g->nz + want - 1) / want);
  const int zmin = env_int("DN_ZCMIN_3D", 4);
  if (ZC < zmin) ZC = zmin;
  if (ZC > g->nz) ZC = g->nz;
  ZC = env_int("DN_ZC_3D", ZC);
  pl.ZC = ZC;
  pl.nzc = (g->nz + ZC - 1) / ZC;
  pl.grid = tiles * pl.nzc;
  pl.smem = (size_t)2 * smem_floats_3d(pl.LX, pl.TY, pl.V) * sizeof(float);
  return pl;
}

long long plan3d_max_ctas(const dn_geom* g) {
  long long worst = 0;
  for (int v = 0; v < 2; ++v) {
    Plan3D pl = plan3d(g, v == 1, 148);
    if (pl.grid > worst) worst = pl.grid;
  }
  // streaming path: tiles own >= 1 row... bounded by its planner's minimum chunk (ZCmin >= 1)
  const long long t3 = plan3t_max_ctas(g);
  if (t3 > worst) worst = t3;
  return worst;
}

int run3d(const Common& c, const dn_geom* g, const Out& o) {
  {   // streaming path: common aligned cases (the rest stays on k_fem3d)
    bool handled = false;
    int rc = run3t(c, g, o, &handled);
    if (rc != DN_OK || handled) return rc;
    if (c.link) return fail(DN_EINVAL, "a linked z-slab launch needs the streaming path (nx %% 4 == 0, aligned x-contiguous fields)");
    if (c.k.lv)
      return fail(DN_ENOSTREAM, "DN_F_LOAD_VECTOR: the streaming 3-D kernel cannot take this launch (nx %% 4, aligned "
                  "x-contiguous fields, whole-domain ownership); pass f_gp instead");
  }
  const bool vec4 = c.vec4 && ((uintptr_t)o.grad % 16 == 0);
  Plan3D pl = plan3d(g, vec4, c.sms);
  if (pl.TY < 1 || (pl.nty > 1 && pl.TY < 2) || (pl.ntx > 1 && pl.LX < 2))
    return fail(DN_EINVAL, "bad 3-D launch plan (LX=%d TY=%d)", pl.LX, pl.TY);
  if ((long long)pl.LX * (pl.TY + 1) > DN_MAXT_3D)
    return fail(DN_EINVAL, "3-D block of %d x %d threads exceeds %d", pl.LX, pl.TY + 1, DN_MAXT_3D);
  if (pl.smem > 200 * 1024) return fail(DN_EINVAL, "3-D tile needs %zu B of shared memory", pl.smem);
  P3D p;
  memset(&p, 0, sizeof(p));
  if (int rc = reduce_into(o, pl.grid, &p.red)) return rc;
  if (pl.grid > 0x7fffffffLL) return fail(DN_EINVAL, "grid too large");
  p.u = c.u; p.nu = c.nu; p.f = c.f; p.fgp = c.fgp; p.numask = c.numask;
  for (int i = 0; i < DN_MAX_MASKS; ++i) p.mk[i] = c.mk[i];
  p.B = g->batch; p.nx = g->nx; p.ny = g->ny; p.nz = g->nz;
  p.k = c.k; p.rule = c.rule;
  p.LX = pl.LX; p.TY = pl.TY; p.ZC = pl.ZC; p.ntx = pl.ntx; p.nty = pl.nty; p.nzc = pl.nzc;
  if (g->z_own_hi > g->z_own_lo) { p.zloss_lo = g->z_own_lo; p.zloss_hi = g->z_own_hi; }
  else { p.zloss_lo = 0; p.zloss_hi = g->nz; }
  p.grad = o.grad;
  p.mode = c.mode; p.mask_input = c.mask_input;
  const int FM = c.f.p ? 1 : (c.fgp.p ? 2 : 0);
  Kernel* k = find3d(pl.V, c.MK, c.nu.p ? 1 : 0, FM, c.numask.p ? 1 : 0);
  if (!k)
    return fail(DN_EINVAL, "unsupported option combination (V=%d MK=%d nu=%d fmode=%d numask=%d)",
                pl.V, c.MK, c.nu.p ? 1 : 0, FM, c.numask.p ? 1 : 0);
  return check_cuda(launch(*k, &p, dim3((unsigned)pl.grid), dim3(pl.LX, pl.TY + 1), pl.smem,
                           (cudaStream_t)o.stream, false), "fem3d launch");
}

}  // namespace dn
