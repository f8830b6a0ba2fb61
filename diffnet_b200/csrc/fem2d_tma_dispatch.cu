// Launch planning and runtime -> compile-time dispatch of the streaming 2-D kernel family (instantiated by
// fem2d_tma_inst.cu).
#include "dn_launch.h"
#include "fem2d_tma.cuh"
#include "fem2d_tma_combos.h"
namespace dn {

// The kernel of a variant of fem2d_tma_combos.h, or null when it is not instantiated.
static Kernel* find2t(int MK, int NU, int F, int NUMASK) {
  static struct { int MK, NU, F, NUMASK; Kernel k; } tab[] = {
#define DN_ROW(MK_, NU_, F_, NMK_) {MK_, NU_, F_, NMK_, {kernel2t<MK_, NU_, F_, NMK_>()}},
      DN2T_ALL(DN_ROW)
#undef DN_ROW
  };
  for (auto& r : tab)
    if (r.MK == MK && r.NU == NU && r.F == F && r.NUMASK == NUMASK) return &r.k;
  return nullptr;
}

struct Plan2T { int ok, threads, S, R, nchunks, nf, bal_q, bal_rem; long long grid; size_t smem; };

static size_t smem_2t(int S, int nf, int nx, int threads) {
  return (size_t)S * nf * 2 * nx * 4 + 16 + (size_t)S * 8 + 4 * (size_t)(threads / 32) * 4;
}

// Eligibility + launch shape.  `k` (whose occupancy bounds the grid) may be null: then only the upper
// bound of the grid matters (workspace sizing).
static Plan2T plan2t(const dn_geom* g, int nf, int sms, Kernel* k) {
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
  int cps = k ? occupancy(*k, pl.threads, pl.smem) : 8;
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

int debug_plan2t(const dn_geom* g, int nfields, int64_t* out) {
  Plan2T pl = plan2t(g, nfields, 148, nullptr);
  out[0] = pl.ok;
  if (pl.ok) {
    out[1] = pl.threads; out[2] = pl.grid; out[3] = (int64_t)pl.smem; out[4] = pl.S;
    out[5] = pl.R; out[6] = pl.nchunks; out[7] = pl.bal_q; out[8] = pl.bal_rem;
  }
  return DN_OK;
}

int run2t(const Common& c, const dn_geom* g, const Out& o, bool* handled) {
  *handled = false;
  const char* path = getenv("DN_2D_PATH");
  if (path && !strcmp(path, "warp")) return DN_OK;
  if (!c.vec4 || c.fgp.p || ((uintptr_t)o.grad % 16 != 0)) return DN_OK;
  const int NU = c.nu.p ? 1 : 0, F = c.f.p ? (c.k.lv ? 2 : 1) : 0, NMK = c.numask.p ? 1 : 0;
  if (g->nx % 4 != 0 || g->nx / 4 > DN_T2_MAXT) return DN_OK;
  Kernel* k = find2t(stream_variant(c, F, NMK), NU, F, NMK);
  if (!k) return DN_OK;
  P2T p;
  memset(&p, 0, sizeof(p));
  const int nf = stream_fields(c, p.fld, p.mval);
  for (int i = 0; i < nf; ++i)
    if (p.fld[i].sy != g->nx) return DN_OK;      // bulk copies take whole runs of rows
  Plan2T pl = plan2t(g, nf, c.sms, k);
  if (!pl.ok) { cudaGetLastError(); return DN_OK; }
  if (pl.grid > 0x7fffffffLL) return DN_OK;
  if (int rc = reduce_into(o, pl.grid, &p.red)) return rc;
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
  p.grad = o.grad;
  p.mode = c.mode;
  *handled = true;
  return check_cuda(launch(*k, &p, dim3((unsigned)pl.grid), dim3(pl.threads), pl.smem, (cudaStream_t)o.stream, true),
                    "fem2d_tma launch");
}

}  // namespace dn
