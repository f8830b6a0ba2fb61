// Launch planning and runtime -> compile-time dispatch of the streaming 3-D kernel family (instantiated by
// fem3d_tma_inst.cu).
#include <cstdio>
#include <cstdlib>

#include "dn_launch.h"
#include "fem3d.cuh"
#include "fem3d_tma.cuh"
#include "fem3d_tma_combos.h"

namespace dn {

// The kernel of a variant of fem3d_tma_combos.h, or null when it is not instantiated.
static Kernel* find3t(int MK, int NU, int F, int NUMASK, int LK) {
  static struct { int MK, NU, F, NUMASK, LK; Kernel k; } tab[] = {
#define DN_ROW(MK_, NU_, F_, NMK_, LK_) {MK_, NU_, F_, NMK_, LK_, {kernel3t<MK_, NU_, F_, NMK_, LK_>()}},
      DN3T_ALL(DN_ROW)
#undef DN_ROW
  };
  for (auto& r : tab)
    if (r.MK == MK && r.NU == NU && r.F == F && r.NUMASK == NUMASK && r.LK == LK) return &r.k;
  return nullptr;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no libcuda link dependency)
typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                              const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                              CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static encode_fn get_encode() {
  static encode_fn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (encode_fn)ptr;
    else
      cudaGetLastError();
  }
  return fn;
}

// 4-D map (x, y, z, b) over one strided fp32 field; box = BX x BY x 1 x 1, zero fill outside
static bool make_map(CUtensorMap* tm, const Field& f, const dn_geom* g, int BX, int BY, int* bmul) {
  encode_fn enc = get_encode();
  if (!enc) return false;
  const bool bc = (f.sb == 0) || (g->batch == 1);
  *bmul = bc ? 0 : 1;
  cuuint64_t dims[4] = {(cuuint64_t)g->nx, (cuuint64_t)g->ny, (cuuint64_t)g->nz, (cuuint64_t)(bc ? 1 : g->batch)};
  const cuuint64_t plane = (cuuint64_t)g->ny * g->nx * 4, vol = plane * (cuuint64_t)g->nz;
  cuuint64_t strides[3] = {(cuuint64_t)f.sy * 4, g->nz > 1 ? (cuuint64_t)f.sz * 4 : plane,
                           bc ? vol : (cuuint64_t)f.sb * 4};
  for (int i = 0; i < 3; ++i)
    if (strides[i] == 0 || strides[i] % 16) return false;
  cuuint32_t box[4] = {(cuuint32_t)BX, (cuuint32_t)BY, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void*)f.p, dims, strides, box, es,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct Plan3T {
  int ok, LXT, LXo, hl, ntx, rows, TY, nty, threads, ZC, nzc, S, BX, BY, fstride;
  long long grid;
  size_t smem;
};

static size_t smem_3t(int S, int nf, int fstride) {
  return (size_t)S * nf * fstride * 4 + (size_t)(S + 1) * 8 + (size_t)xbuf_bytes() + 64;
}

// Launch shape search.  Candidates: x-tile width (owned element pairs per tile row) x thread rows
// per tile (threads = LXT * rows <= 512) x number of z-chunks.  Cost model (the kernel is FP32-pipe
// bound; CTAs on one SM share the pipe):
//   SM time ~ ceil(grid / SMs) * threads * (ZC + 1)   [thread-layers executed by the busiest SM]
// with a penalty when fewer than 12 warps per SM are resident and a mild preference for one wave.
// `k` may be null (workspace sizing): then the register bound is assumed instead of its occupancy.
static Plan3T plan3t(const dn_geom* g, int nf, int sms, Kernel* k, int maxt_variant, long long min_grid = 0) {
  Plan3T best;
  memset(&best, 0, sizeof(best));
  if (g->nx % 4 != 0 || g->nx < 8) return best;
  const int npairs = g->nx / 2;
  int maxt = env_int("DN_T3_THREADS", maxt_variant);
  if (maxt > maxt_variant) maxt = maxt_variant;
  const int lx_forced = env_int("DN_T3_LX", 0), ty_forced = env_int("DN_T3_TY", 0), zc_forced = env_int("DN_T3_ZC", 0);
  int zmin = env_int("DN_T3_ZCMIN", 4);
  if (zmin < 1) zmin = 1;
  int S0 = env_int("DN_T3_STAGES", 4);
  if (S0 < 2) S0 = 2;
  if (S0 > 8) S0 = 8;
  double best_cost = 0.0;
  const int cand[5] = {npairs, 16, 32, 64, 128};
  for (int ci = 0; ci < 5; ++ci) {
    int LXo = cand[ci];
    if (lx_forced > 0) { if (ci > 0) break; LXo = lx_forced; }
    if (LXo > npairs) LXo = npairs;
    if (ci > 0 && LXo >= npairs) continue;             // same as the full-width candidate
    const int ntx = (npairs + LXo - 1) / LXo;
    const int hl = ntx > 1 ? 1 : 0;
    const int LXT = LXo + hl;
    if (LXT * 2 > maxt) continue;
    const int BX = (2 * LXT + 2 + 2 * hl + 3) / 4 * 4;   // + alignment slack when the tile starts at an odd pair
    if (BX > 256) continue;
    for (int rows = 2; rows * LXT <= maxt; ++rows) {
      int TYmax = rows - 1;
      if (ty_forced > 0) { if (ty_forced > TYmax) continue; TYmax = ty_forced; }
      const int nty = (g->ny + TYmax - 1) / TYmax;
      const int TY = (g->ny + nty - 1) / nty;
      // thread rows a tile needs: TY owned node rows + the halo element row above (tiles below the
      // first); the tile with the domain's last node row runs a phantom element row below it instead
      int need = nty >= 2 ? TY + 1 : TY;
      if (need < 1) need = 1;
      if (ty_forced <= 0 && rows != need && !(need < 2 && rows == 2)) continue;   // a smaller block covers it
      if (rows < need) continue;
      const int BY = TY + 2;
      if (BY > 256) continue;
      const int threads = (rows * LXT + 31) / 32 * 32;
      if (threads > maxt_variant) continue;
      const int fstride = (BX * BY + 31) / 32 * 32;
      int S = S0;
      while (S > 2 && smem_3t(S, nf, fstride) > (size_t)kMaxDynSmem) --S;
      const size_t smem = smem_3t(S, nf, fstride);
      if (smem > (size_t)kMaxDynSmem) continue;
      int cps = k ? occupancy(*k, threads, smem) : (int)(65536 / (threads * (maxt_variant > 512 ? 96 : 128)));
      if (env_int("DN_DEBUG_PLAN", 0) >= 2)
        fprintf(stderr, "[plan3t] candidate LXT=%d rows=%d TY=%d threads=%d smem=%zu -> %d CTA/SM\n", LXT, rows, TY,
                threads, smem, cps);
      if (cps < 1) continue;
      const long long tiles = (long long)g->batch * nty * ntx;
      const int nzc_max = zc_forced > 0 ? 1 : (g->nz + zmin - 1) / zmin;
      for (int nzc_try = 1; nzc_try <= nzc_max; ++nzc_try) {
        int ZC = zc_forced > 0 ? zc_forced : (g->nz + nzc_try - 1) / nzc_try;
        if (ZC > g->nz) ZC = g->nz;
        if (ZC < 1) ZC = 1;
        const int nzc = (g->nz + ZC - 1) / ZC;
        if (zc_forced <= 0 && nzc != nzc_try) continue;
        const long long grid = tiles * nzc;
        if (grid < min_grid && nzc_try < nzc_max) continue;          // linked launches want >= 2 waves (see the kernel)
        const long long per_sm = (grid + sms - 1) / sms;             // CTAs the busiest SM runs
        const long long resident = per_sm < cps ? per_sm : cps;
        const double waves = (double)((per_sm + cps - 1) / cps);
        const double warps = (double)resident * threads / 32.0;
        double cost = (double)per_sm * threads * (ZC + 1);
        if (warps < 12.0) cost *= 1.0 + 0.4 * (12.0 - warps) / 12.0;
        if (LXT % 32) cost *= 1.2;      // warps straddling tile rows: measured 15-20 % slower per thread-layer
        cost *= 1.0 + 0.05 * (waves - 1.0);
        if (!best.ok || cost < best_cost) {
          best_cost = cost;
          best.ok = 1; best.LXT = LXT; best.LXo = LXo; best.hl = hl; best.ntx = ntx; best.rows = rows;
          best.TY = TY; best.nty = nty; best.threads = threads; best.ZC = ZC; best.nzc = nzc; best.S = S;
          best.BX = BX; best.BY = BY; best.fstride = fstride; best.grid = grid; best.smem = smem;
        }
        if (grid > 64LL * sms) break;                                 // finer chunks only add seams
      }
    }
  }
  return best;
}

long long plan3t_max_ctas(const dn_geom* g) {
  if (g->nx % 4 != 0 || g->nx < 8) return 0;
  // workspace sizing: an upper bound on what the planner may pick -- x tiles of >= 16 pairs,
  // y tiles owning >= 1 row, chunks of >= 4 planes (the DN_T3_ZCMIN default).  Capped to keep
  // the workspace small; a knob setting that needs more is refused with DN_EWORKSPACE.
  const long long ntx = (g->nx / 2 + 15) / 16, nty = g->ny, nzc = (g->nz + 3) / 4;
  long long n = (long long)g->batch * ntx * nty * nzc;
  const long long cap = 1LL << 22;
  return n < cap ? n : cap;
}

int debug_plan3t(const dn_geom* g, int nfields, int has_nu, int64_t* out) {
  Plan3T pl = plan3t(g, nfields, 148, nullptr, DN_T3_MAXT_OF(has_nu));
  out[0] = pl.ok;
  if (pl.ok) {
    out[1] = pl.threads; out[2] = pl.grid; out[3] = (int64_t)pl.smem; out[4] = pl.S;
    out[5] = pl.TY; out[6] = pl.nty; out[7] = pl.LXT; out[8] = pl.ntx; out[9] = pl.ZC; out[10] = pl.nzc;
    out[11] = pl.BX; out[12] = pl.BY; out[13] = pl.rows; out[14] = pl.LXo; out[15] = pl.hl;
  }
  return DN_OK;
}

int run3t(const Common& c, const dn_geom* g, const Out& o, bool* handled) {
  *handled = false;
  const char* path = getenv("DN_3D_PATH");
  if (path && !strcmp(path, "tile")) return DN_OK;
  if (!c.vec4 || c.fgp.p || ((uintptr_t)o.grad % 16 != 0)) return DN_OK;
  const Field& u = c.u;
  const Consts& k = c.k;
  const dn_slab_link* link = c.link;
  const int sms = c.sms;
  const bool iso = c.nu.p && k.kx == k.ky && k.kx == k.kz && k.kx != 0.f && env_int("DN_T3_ISO", 1);
  const bool iso1 = !c.nu.p && k.kx == k.ky && k.kx == k.kz && env_int("DN_T3_ISO", 1);
  const int NU = c.nu.p ? (iso ? 2 : 1) : (iso1 ? 3 : 0), F = c.f.p ? (k.lv ? 2 : 1) : 0, NMK = c.numask.p ? 1 : 0;
  // the load-vector term is nodal: with z-slab ownership a node plane has no single owner
  if (k.lv && (link || g->z_own_hi > g->z_own_lo)) return DN_OK;
  Kernel* kern = find3t(stream_variant(c, F, NMK), NU, F, NMK, link ? 1 : 0);
  if (!kern || !get_encode()) return DN_OK;
  Field fl[DN_T2_MAXF];
  P3T p;
  memset(&p, 0, sizeof(p));
  const int nf = stream_fields(c, fl, p.mval);
  const long long min_grid = (link && link->halo_plane[0] && env_int("DN_SLAB_WAVES", 0)) ? (long long)(1.9 * sms) : 0;
  Plan3T pl = plan3t(g, nf, sms, kern, DN_T3_MAXT_OF(c.nu.p != nullptr), min_grid);
  if (!pl.ok) { cudaGetLastError(); return DN_OK; }
  if (pl.grid > 0x7fffffffLL) return DN_OK;
  int nput = 0;
  if (link) {
    nput = env_int("DN_SLAB_NPUT", 2);
    if (nput < 1) nput = 1;
    if (nput > 16) nput = 16;
    pl.grid += 2 * nput;
  }
  // a CTA is one (x-tile, y-tile, z-chunk) work item of one sample; the items of a sample are consecutive CTAs
  if (int rc = reduce_into(c, o, g, pl.grid, pl.ntx * pl.nty * pl.nzc, 0, &p.red)) return rc;
  for (int i = 0; i < nf; ++i)
    if (!make_map(&p.tm[i], fl[i], g, pl.BX, pl.BY, &p.bmul[i])) return DN_OK;   // general kernel takes it
  p.nf = nf;
  p.B = g->batch; p.nx = g->nx; p.ny = g->ny; p.nz = g->nz;
  p.LXT = pl.LXT; p.LXo = pl.LXo; p.hl = pl.hl; p.ntx = pl.ntx;
  p.rows = pl.rows; p.TY = pl.TY; p.nty = pl.nty;
  p.ZC = pl.ZC; p.nzc = pl.nzc; p.S = pl.S;
  p.BX = pl.BX; p.BY = pl.BY; p.fstride = pl.fstride;
  if (g->z_own_hi > g->z_own_lo) { p.zloss_lo = g->z_own_lo; p.zloss_hi = g->z_own_hi; }
  else { p.zloss_lo = 0; p.zloss_hi = g->nz; }
  const float t = k.t;
  auto pr = [](float v) { return make_float2(v, v); };
  p.k3.kx = pr(k.kx); p.k3.ky = pr(k.ky); p.k3.kz = pr(k.kz);
  p.k3.kxt = pr(k.kx * t); p.k3.kyt = pr(k.ky * t); p.k3.kzt = pr(k.kz * t);
  p.k3.kxtt = pr(k.kx * t * t); p.k3.kytt = pr(k.ky * t * t); p.k3.kztt = pr(k.kz * t * t);
  p.k3.t = pr(t); p.k3.tt = pr(t * t);
  p.k3.nkf = pr(-k.kf); p.k3.nkft = pr(-k.kf * t); p.k3.nkftt = pr(-k.kf * t * t);
  p.k3.nkfttt = pr(-k.kf * t * t * t);
  p.k3.c0x = pr(8.f * k.kx); p.k3.c0y = pr(8.f * k.ky); p.k3.c0z = pr(8.f * k.kz);
  p.k3.kscale = 1.f;
  p.k3.c0_2t = pr(2.f * 8.f * k.kx * t); p.k3.c0_3tt = pr(3.f * 8.f * k.kx * t * t);
  if (iso) {
    // isotropic spacing: k moves out of the element (see K3); the source constants absorb 1/k
    p.k3.kscale = k.kx;
    const float kf = k.kf / k.kx;
    p.k3.nkf = pr(-kf); p.k3.nkft = pr(-kf * t); p.k3.nkftt = pr(-kf * t * t); p.k3.nkfttt = pr(-kf * t * t * t);
  }
  p.k3.nkb = -k.kb;
  p.k3.nkb_pre = pr(-k.kb / p.k3.kscale);
  p.grad = o.grad;
  p.mode = c.mode;
  if (link) {
    if (g->batch != 1) return fail(DN_EINVAL, "linked z-slab launches are for one field (batch 1)");
    if (!link->step || !link->tickets || !link->status) return fail(DN_EINVAL, "dn_slab_link: step / tickets / status missing");
    dn_geom gp = *g;
    gp.nz = 1; gp.batch = 1;
    const long long plane = (long long)g->ny * g->nx;
    for (int sd = 0; sd < 2; ++sd) {
      if (link->halo_plane[sd]) {
        if (!link->halo_flag[sd]) return fail(DN_EINVAL, "dn_slab_link: halo_flag[%d] missing", sd);
        Field hf;
        hf.p = link->halo_plane[sd]; hf.sb = plane; hf.sz = plane; hf.sy = g->nx;
        int bm = 0;
        if (!make_map(&p.lk.tmh[sd], hf, &gp, pl.BX, pl.BY, &bm))
          return fail(DN_EINVAL, "dn_slab_link: halo_plane[%d] is not TMA-addressable (16-byte alignment)", sd);
        p.lk.hflag[sd] = link->halo_flag[sd];
      }
      if (link->put_dst[sd]) {
        if (!link->put_flag[sd] || link->put_plane[sd] < 0 || link->put_plane[sd] >= g->nz)
          return fail(DN_EINVAL, "dn_slab_link: put_flag / put_plane[%d] invalid", sd);
        if (u.sy != g->nx || u.sz != plane || plane % 4 || ((uintptr_t)u.p % 16) || ((uintptr_t)link->put_dst[sd] % 16))
          return fail(DN_EINVAL, "dn_slab_link: u must be a contiguous, 16-byte aligned slab (ny*nx %% 4 == 0)");
        p.lk.pdst[sd] = (float4*)link->put_dst[sd];
        p.lk.psrc[sd] = (const float4*)(u.p + (long long)link->put_plane[sd] * plane);
        p.lk.pflag[sd] = link->put_flag[sd];
      }
    }
    p.lk.pn4 = plane / 4;
    p.lk.nput = nput;
    p.lk.tickets = link->tickets;
    p.lk.status = link->status;
    p.lk.max_spins = link->max_spins > 0 ? link->max_spins : (1LL << 26);
    p.red.step = link->step;
    p.lk.dbg = env_int("DN_SLAB_DBG", 0);
    p.red.peer_slots = link->loss_slots;
    p.red.rank = link->rank; p.red.world = (p.lk.dbg & 4) ? 0 : link->world;
    if (link->loss_slots && (link->world < 1 || link->world > 32 || link->rank < 0 || link->rank >= link->world))
      return fail(DN_EINVAL, "dn_slab_link: rank %d / world %d (world <= 32)", link->rank, link->world);
  }
  if (env_int("DN_DEBUG_PLAN", 0))
    fprintf(stderr, "[plan3t] B=%d n=(%d,%d,%d) LXT=%d LXo=%d hl=%d ntx=%d rows=%d TY=%d nty=%d ZC=%d nzc=%d S=%d BX=%d BY=%d "
            "fstride=%d threads=%d grid=%lld smem=%zu\n", g->batch, g->nx, g->ny, g->nz, pl.LXT, pl.LXo, pl.hl, pl.ntx,
            pl.rows, pl.TY, pl.nty, pl.ZC, pl.nzc, pl.S, pl.BX, pl.BY, pl.fstride, pl.threads, pl.grid, pl.smem);
  *handled = true;
  return check_cuda(launch(*kern, &p, dim3((unsigned)pl.grid), dim3(pl.threads), pl.smem, (cudaStream_t)o.stream, true),
                    "fem3d_tma launch");
}

}  // namespace dn
