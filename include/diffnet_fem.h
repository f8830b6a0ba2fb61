/*
 * diffnet_fem.h -- C ABI of libdiffnet_fem.so: the B200 (sm_100a) FEM-loss hot path of DiffNet.
 *
 * The reference (adityabalu/DiffNet) has no FFI; its seam is a Python method contract
 * (SURVEY.md 8b).  Each entry point below names the reference code it replaces:
 *
 *   dn_fem_energy_{2d,3d}_f32   the user loss() body built from gauss_pt_evaluation{,_der_x,
 *                               _der_y,_der_z} (DiffNet/DiffNetFEM.py:7-18,143-156) + torch.where
 *                               Dirichlet masking + the energy integrand + sum over Gauss points +
 *                               mean over elements, AND its autograd backward w.r.t. u (and nu):
 *                               examples/poisson/single_instance/0_base.py:31-56,
 *                               12_klsum.py:53-78, IBN/poisson-2d/parametric/
 *                               e1_complex_immersed_background.py:33-58, e2_..._neumann.py:33-60,
 *                               IBN/poisson-3d/parametric/IBN_3D.py:114-136,
 *                               IBN/poisson-3d/non-parametric/solve_in_object_3d.py:75-102.
 *   dn_fem_residual_{2d,3d}_f32 the assembled-residual ("resmin") body: per-element residual,
 *                               Q1 scatter-add assembly, Dirichlet zeroing, sum(R^2):
 *                               12_klsum.py:46-51,80-132; tests/test.py:36-79; tests/test3D.py:36-85.
 *   dn_fem_gp_eval_{2d,3d}_f32  gauss_pt_eval / gauss_pt_evaluation* themselves
 *   dn_fem_gp_eval_adj_*        (DiffNetFEM.py:7-18,143-156) and their autograd backward
 *                               (convolution_backward = scatter-transpose).
 *   dn_fem_{energy,residual}_input_grads_*  the same bodies' autograd backward w.r.t. the source, the forcing at
 *                               the Gauss points, the Dirichlet value fields and (residual) nu.
 *   dn_scale_inplace_f32        autograd's  grad_input = grad_output * dL/du.
 *   dn_scale_per_sample_f32     the same with one grad_output per sample (reduction = none).
 *   dn_peer_{put,wait}_f32      (no reference counterpart) one-plane halo exchange of the z-slab
 *                               decomposition through NVLink peer memory.
 *
 * Conventions
 *   - All pointers in dn_field / outputs are DEVICE pointers, fp32, x (innermost) contiguous.
 *     Nodal fields are (B, nz, ny, nx) [nz = 1 in 2-D]; strides are in ELEMENTS and arbitrary
 *     (channel slices of a (B,3,H,W) tensor are passed as-is: stride_b = 3*H*W); stride_b = 0
 *     broadcasts one field over the batch.
 *   - Outputs (grad_u, grad_nu, residual, gp-eval results) are dense/contiguous.
 *   - Every call is asynchronous on `stream` (a cudaStream_t passed as void*), re-entrant,
 *     allocates nothing and keeps no device state.  The caller owns all buffers.  (Only
 *     dn_peer_alloc/dn_peer_import hand out memory; they are synchronous set-up calls.)
 *   - `workspace`: at least dn_fem_workspace_bytes() bytes, 16-byte aligned, and ZERO-FILLED
 *     BEFORE ITS FIRST USE; a call leaves it zero-filled-equivalent for the next call on the same
 *     stream (the ticket counter self-resets).  Do not share one workspace between streams.
 *   - Return value: DN_OK or a negative dn_status; dn_last_error() gives the text (thread-local).
 *   - No CPU fallback: non-sm_100 devices get DN_EARCH.
 */
#ifndef DIFFNET_FEM_H_
#define DIFFNET_FEM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DN_ABI_VERSION 1
#define DN_MAX_MASKS 3

typedef enum dn_status {
  DN_OK = 0,
  DN_EINVAL = -1,      /* bad shape / stride / null pointer / unsupported option */
  DN_EARCH = -2,       /* device is not sm_100 (B200) */
  DN_ECUDA = -3,       /* CUDA launch/runtime error, see dn_last_error() */
  DN_EWORKSPACE = -4,  /* workspace missing or too small */
  DN_ENOSTREAM = -5    /* an option only the streaming kernels implement (DN_F_LOAD_VECTOR) was asked for a launch they
                          cannot take (odd nx, unaligned or non-contiguous views, z-slab ownership): use f_gp instead */
} dn_status;

/* One fp32 field on the mesh nodes.  ptr == NULL means "absent". */
typedef struct dn_field {
  const float* ptr;
  int64_t stride_b;    /* batch stride (0 = broadcast) */
  int64_t stride_z;    /* plane stride (ignored in 2-D) */
  int64_t stride_y;    /* row stride */
} dn_field;

/* Dirichlet condition  u = where(mask > 0.5, value [+ value_field], u)   (0_base.py:41-42,
 * e8_2d_poisson_mms.py:165).  Conditions are applied in array order: where masks overlap the
 * LAST one wins; dL/du is exactly 0 wherever any mask fired. */
typedef struct dn_mask {
  dn_field mask;         /* fp32 0/1 field, strict > 0.5 */
  dn_field value_field;  /* optional nodal Dirichlet values; ptr NULL -> use `value` */
  float value;
  int32_t _pad;
} dn_mask;

typedef struct dn_geom {
  int32_t nsd;           /* 2 or 3 */
  int32_t batch;         /* B */
  int32_t nx, ny, nz;    /* NODES per direction (domain_sizeX/Y/Z); nz = 1 in 2-D */
  int32_t ngp_1d;        /* 2, 3 or 4 (DiffNetFEM.py:128-141); Q1 basis only */
  double hx, hy, hz;     /* element sizes (DiffNetFEM.py:47-51) */
  /* z-slab decomposition (3-D only, SURVEY.md 8e); all zero = whole domain is local.
   * Local planes [0,nz) hold global planes [z_global0, z_global0+nz); the loss sums elements
   * whose lower plane is in [z_own_lo, z_own_hi) (local indices); gradients are written for all
   * local planes but are complete only on owned ones. */
  int32_t z_own_lo, z_own_hi;
  double mean_count;     /* divisor of reduction=mean; 0 -> B * (local element count) */
} dn_geom;

typedef struct dn_consts {
  double c_k;            /* multiplies nu * |grad u|^2      (SURVEY.md App. A.4) */
  double c_f;            /* multiplies u * f */
  double scale;          /* overall factor s (e.g. 0.5*(h/2)^2 in 0_base.py:51-52) */
  int32_t reduction;     /* 0 = mean over batch x elements, 1 = sum, DN_REDUCE_NONE = one loss per sample */
  int32_t flags;         /* DN_F_* bits; 0 = the reference's forms */
} dn_consts;

/* dn_consts.reduction (and the `reduction` of dn_fem_residual_reduce_*): one loss per sample instead of one for the
 * launch.  loss_out / loss_out_f32 then point to g->batch values each, and
 *   energy:    loss[b] = scale / (elements of one sample) * sum_{e in sample b} sum_g w_g (...),
 *              so the mean of loss[] is the reduction = 0 loss and its sum times the element count the reduction = 1 one;
 *   residual:  loss[b] = sum_{nodes of sample b} R^2, whose sum is the reduction = 1 loss.
 * The gradients written are those of loss[b] with respect to the inputs of sample b.  The per-sample values are
 * summed in a fixed order that depends only on the launch shape (bit-reproducible run to run).  Not available with
 * mean_count != 0, z-slab ownership (z_own_lo/hi) or a linked launch: DN_EINVAL. */
#define DN_REDUCE_NONE 2

/* dn_consts.flags: `f` is not a nodal source but an ASSEMBLED load vector b_a = sum_e sum_g w_g N_a(g) f_g
 * (dn_fem_load_vector_f32; reference-element weights, |J| stays in `scale`): the source term becomes
 * -scale c_f sum_a b_a u_a.  Same loss and gradient as passing f_gp
 * (the reference's forcing-at-Gauss-points form, e8_2d_poisson_mms.py:154-175) up to fp32 summation order, at 4
 * instead of 4 ngp^nsd bytes per node and step when f_gp does not change between steps. */
#define DN_F_LOAD_VECTOR 1

/* which table a gp-eval call uses (DiffNetFEM.py:143-156) */
typedef enum dn_gp_which { DN_GP_N = 0, DN_GP_DX = 1, DN_GP_DY = 2, DN_GP_DZ = 3 } dn_gp_which;

int dn_abi_version(void);
const char* dn_last_error(void);
/* DN_OK if the current CUDA device is sm_100, DN_EARCH / DN_ECUDA otherwise. */
int dn_device_check(void);

size_t dn_fem_workspace_bytes(const dn_geom* g);

/* Launch shape the streaming planners pick for `g` with `nfields` input fields (u, nu, f, masks ...),
 * using the static register bound instead of a device occupancy query, so it runs WITHOUT a GPU
 * (tests of the planners).  out[0] = 1 if the streaming path is eligible by shape, then
 * out[1..] = {threads per CTA, grid, dynamic shared memory bytes, ring stages,
 *             2-D: rows per chunk R, chunks per image | 3-D: owned rows per tile TY, y tiles,
 *             lanes per tile row LXT, x tiles, planes per chunk ZC, z chunks, box BX, box BY}. */
int dn_debug_plan(const dn_geom* g, int nfields, int has_nu, int64_t out[16]);

/*
 * Fused energy loss + gradient.
 *   loss = S * sum_{b,e} sum_g w_g ( c_k nu_g |grad u'|_g^2 - c_f u'_g f_g ),  S = scale / count
 *   u'   = u with the Dirichlet conditions applied;  nu' = where(nu_zero_mask > 0.5, 0, nu)
 *   grad_u[b,node] = dloss/du  (0 at Dirichlet nodes);  grad_nu likewise (optional).
 * nu == NULL means nu == 1 (IBN_3D.py:132); f and fgp NULL means no source term; at most one of
 * f (nodal, (B|1,nz,ny,nx)) and fgp (at Gauss points, dense (B|1, ngp, elems), stride_b given,
 * other strides ignored; e8_2d_poisson_mms.py:47,154) may be set.
 * loss_out: device double[1] (nullable); loss_out_f32: device float[1] (nullable); double[B] / float[B] with
 * c->reduction == DN_REDUCE_NONE.
 * grad_u NULL -> forward only.
 */
int dn_fem_energy_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                         const dn_field* fgp, const dn_mask* masks, int nmasks,
                         const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                         float* grad_u, float* grad_nu, void* workspace, size_t workspace_bytes,
                         double* loss_out, float* loss_out_f32, void* stream);
int dn_fem_energy_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                         const dn_field* fgp, const dn_mask* masks, int nmasks,
                         const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                         float* grad_u, float* grad_nu, void* workspace, size_t workspace_bytes,
                         double* loss_out, float* loss_out_f32, void* stream);

/*
 * Linked z-slab step (3-D, one process per GPU; SURVEY.md 8e -- new functionality, the reference runs
 * solve_in_object_3d.py:191-200 on one GPU): ONE launch per rank and step does the halo exchange of
 * u, the fused loss + gradient on the slab and the all-reduce of the loss, over NVLink peer memory:
 *   - the first CTAs of the launch store this rank's first / last owned plane of u into the
 *     neighbours' staging planes (put_dst, peer-mapped) and release their flag words (put_flag) with
 *     the launch number (system scope);
 *   - the kernel reads local plane 0 / nz-1 of u (the halos) from halo_plane[0] / [1] instead of from
 *     `u`; only the CTAs whose z-chunk touches a halo plane wait -- on the device, bounded by
 *     max_spins polls -- until *halo_flag >= launch number; all other CTAs start at once, so the
 *     exchange overlaps the interior planes;
 *   - the CTA that finishes the loss reduction stores the rank total into slot `rank` of every
 *     rank's receive area (loss_slots[r]: double[world] then int32[world] flags) and increments
 *     *step; dn_peer_loss_sum_f32 adds the slots up (rank order) whenever the value is wanted.
 * `step` is a device word counting the launches of this link (start at 0); consecutive launches
 * must alternate between two sets {staging planes, flags, loss areas, step} (parity) so that a rank
 * one step ahead never overwrites data its neighbour still reads.  Pointers of a missing neighbour
 * are NULL.  All ranks must launch the same sequence.  Needs the streaming path (nx % 4 == 0,
 * 16-byte aligned x-contiguous fields, nodal f); DN_EINVAL otherwise.  *status becomes 1 if a wait
 * ran out of polls (the launch then finishes with stale halos: check it when you synchronise).
 */
typedef struct dn_slab_link {
  const float* halo_plane[2];   /* [below, above] local staging plane, ny*nx floats, 16-byte aligned */
  const int32_t* halo_flag[2];  /* local flag words released by the neighbours */
  float* put_dst[2];            /* the neighbours' staging planes (peer-mapped) */
  int32_t* put_flag[2];         /* the neighbours' flag words (peer-mapped) */
  int32_t put_plane[2];         /* local plane index of u sent below / above (first / last owned) */
  double* const* loss_slots;    /* DEVICE array[world] of receive areas as mapped here; NULL = no loss exchange */
  int32_t* step;                /* local device word: launches so far with this set */
  uint32_t* tickets;            /* 2 zero-initialised local device words (scratch) */
  int32_t* status;              /* local device word */
  int64_t max_spins;
  int32_t rank, world;
} dn_slab_link;

int dn_fem_energy_3d_linked_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                const dn_mask* masks, int nmasks, const dn_field* nu_zero_mask,
                                const dn_geom* g, const dn_consts* c, const dn_slab_link* link,
                                float* grad_u, void* workspace, size_t workspace_bytes,
                                double* loss_out, float* loss_out_f32, void* stream);
/* Sum (rank order, bit-identical everywhere) of the loss slots of launch number `want` once every
 * rank's flag has reached it (bounded device-side wait); out: device float[1]. */
int dn_peer_loss_sum_f32(const double* slots, int world, const int32_t* step, int64_t max_spins,
                         int32_t* status, float* out, void* stream);

/*
 * Assembled residual  R = jac * ( K(nu) u' - F(f) ), zeroed at Dirichlet nodes, and
 * loss = sum(R^2)  (12_klsum.py:80-132).  `residual` (dense (B,nz,ny,nx)) is required: it is
 * what the backward pass consumes.  If apply_masks_to_input == 0 the Dirichlet VALUES are not
 * substituted into u (only the output is zeroed): that is the operator  v -> mask(K(nu) v)
 * the backward pass needs (dL/du = mask( K(nu) (2R) )).
 */
int dn_fem_residual_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                           const dn_mask* masks, int nmasks, int apply_masks_to_input,
                           const dn_geom* g, double jac, float* residual, void* workspace,
                           size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                           void* stream);
int dn_fem_residual_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                           const dn_mask* masks, int nmasks, int apply_masks_to_input,
                           const dn_geom* g, double jac, float* residual, void* workspace,
                           size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                           void* stream);
/* The same with reduction = 1 (sum, what dn_fem_residual_* do) or DN_REDUCE_NONE (loss_out / loss_out_f32 then hold
 * g->batch values: the sum of R^2 over each sample's nodes). */
int dn_fem_residual_reduce_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                  const dn_mask* masks, int nmasks, int apply_masks_to_input,
                                  const dn_geom* g, double jac, float* residual, void* workspace,
                                  size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                                  void* stream, int reduction);
int dn_fem_residual_reduce_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                  const dn_mask* masks, int nmasks, int apply_masks_to_input,
                                  const dn_geom* g, double jac, float* residual, void* workspace,
                                  size_t workspace_bytes, double* loss_out, float* loss_out_f32,
                                  void* stream, int reduction);

/*
 * Gradients of the fused losses with respect to their OTHER inputs -- what autograd gives the reference's loss()
 * bodies for a source, forcing, Dirichlet value field or diffusivity that requires grad (inverse problems, optimal
 * control, coefficient identification).  ONE launch produces every requested output; each output pointer may be NULL
 * (not wanted).  Notation of dn_fem_energy_*: S = scale / count, u' = u with the Dirichlet conditions applied,
 * M / K(nu) = Q1 mass / stiffness matrices with the rule's reference-element weights (K includes (2/h)^2).
 * "mask k is the last firing mask at n": mask k fires at n and no later mask of the list does.
 *
 * dn_fem_energy_input_grads_*   (the autograd backward of the loss() bodies listed at dn_fem_energy_*, w.r.t.
 *                               forcing_tensor / f_gp / a value field, e8_2d_poisson_mms.py:154-175)
 *   grad_f[b,n]       = -S c_f (M u')[b,n]                          (f required; NOT zeroed at Dirichlet nodes)
 *   grad_fgp[b,G,e]   = -S c_f w_G u'_G(e)                          (fgp required; dense like fgp)
 *   grad_values[k][b,n] = [k last firing at n] * S (2 c_k K(nu') u' - c_f (M f | sum_e sum_g w_g N_n f_gp))[b,n]
 *                                                                   (masks[k].value_field required)
 *   With c->reduction == DN_REDUCE_NONE, S = scale / (elements of one sample): the gradients of loss[b].
 * dn_fem_residual_input_grads_* (the autograd backward of 12_klsum.py:80-132 w.r.t. nu, forcing, a value field)
 *   residual: the R that dn_fem_residual_*_f32 returned for the same inputs (dense (B, nz, ny, nx))
 *   grad_nu[b,n]      = 2 jac sum_{e around n} sum_g w_g N_n(g) grad u'_g . grad R_g     (nu required)
 *   grad_f[b,n]       = -2 jac (M R)[b,n]                                                (f required)
 *   grad_values[k][b,n] = [k last firing at n] * 2 jac (K(nu) R)[b,n]
 * Output shapes: dense (B, nz, ny, nx) -- or (1, nz, ny, nx), summed over the batch in a fixed order, when the
 * differentiated field has stride_b == 0 and batch > 1.  grad_values is a HOST array of nmasks pointers (or NULL).
 * Gather form, no atomics: bit-reproducible.  No workspace.  z-slab ownership (z_own_lo/hi set) and
 * DN_F_LOAD_VECTOR are rejected with DN_EINVAL (pass f_gp itself).
 */
int dn_fem_energy_input_grads_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                     const dn_field* fgp, const dn_mask* masks, int nmasks,
                                     const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                                     float* grad_f, float* grad_fgp, float* const* grad_values, void* stream);
int dn_fem_energy_input_grads_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                     const dn_field* fgp, const dn_mask* masks, int nmasks,
                                     const dn_field* nu_zero_mask, const dn_geom* g, const dn_consts* c,
                                     float* grad_f, float* grad_fgp, float* const* grad_values, void* stream);
int dn_fem_residual_input_grads_2d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                       const dn_field* residual, const dn_mask* masks, int nmasks,
                                       const dn_geom* g, double jac, float* grad_nu, float* grad_f,
                                       float* const* grad_values, void* stream);
int dn_fem_residual_input_grads_3d_f32(const dn_field* u, const dn_field* nu, const dn_field* f,
                                       const dn_field* residual, const dn_mask* masks, int nmasks,
                                       const dn_geom* g, double jac, float* grad_nu, float* grad_f,
                                       float* const* grad_values, void* stream);

/*
 * Gauss-point evaluation  out[b, G, elem] = sum_a T_which[G][a] * in[b, node(elem,a)]
 * (gauss_pt_eval, DiffNetFEM.py:7-18), G = ngp_1d*jgp + igp (2-D), ngp_1d^2*kgp + ngp_1d*jgp + igp
 * (3-D); out dense (B, ngp_1d^nsd, [nz-1,] ny-1, nx-1).  The adjoint scatters a cotangent of that
 * shape back to the nodes: grad_in dense (B, nz, ny, nx) (fully overwritten).
 */
int dn_fem_gp_eval_2d_f32(const dn_field* in, const dn_geom* g, int which, float* out,
                          void* stream);
int dn_fem_gp_eval_3d_f32(const dn_field* in, const dn_geom* g, int which, float* out,
                          void* stream);
int dn_fem_gp_eval_adj_2d_f32(const float* grad_out, const dn_geom* g, int which, float* grad_in,
                              void* stream);
int dn_fem_gp_eval_adj_3d_f32(const float* grad_out, const dn_geom* g, int which, float* grad_in,
                              void* stream);
/*
 * Several tables in ONE call (one table per pass by default: the op is write-bound, see gp_eval.cu): which[w] in {0: N, 1: d/dx, 2: d/dy, 3: d/dz}, nwhich <= 4,
 * outs[w] / grad_outs[w] dense as above.  A user loss() body that calls gauss_pt_evaluation(u),
 * gauss_pt_evaluation_der_x(u), gauss_pt_evaluation_der_y(u) (e.g. examples/poisson/single_instance/
 * 14_helmholtz_mms.py:50-59) streams u once; the adjoint sums the cotangents of all tables in one launch.
 * `which`, `outs`, `grad_outs` are HOST arrays (read during the call).
 */
int dn_fem_gp_eval_multi_2d_f32(const dn_field* in, const dn_geom* g, int nwhich, const int* which,
                                float* const* outs, void* stream);
int dn_fem_gp_eval_multi_3d_f32(const dn_field* in, const dn_geom* g, int nwhich, const int* which,
                                float* const* outs, void* stream);
int dn_fem_gp_eval_multi_adj_2d_f32(const float* const* grad_outs, const dn_geom* g, int nwhich,
                                    const int* which, float* grad_in, void* stream);
int dn_fem_gp_eval_multi_adj_3d_f32(const float* const* grad_outs, const dn_geom* g, int nwhich,
                                    const int* which, float* grad_in, void* stream);

/*
 * gauss_pt_eval for ANY tensor-product Lagrange basis and rule, in 1, 2 or 3 dimensions: the quadratic / cubic bases
 * (fem_basis_deg 2 / 3: nbf_1d = 3 / 4 nodes per direction, elements every nbf_1d - 1 nodes -- DiffNetFEM.py:7-18 with
 * stride = nbf_1d - 1, :66-126) and the 1-D surface stencils of a 2-D mesh (gauss_pt_evaluation_surf, :146-147,
 * 244-269: nsd = 1).  factors = HOST array [nsd][ngp_1d][nbf_1d] of the 1-D factors per direction (0 = x): basis value
 * at the Gauss point, or derivative * 2/h for the differentiated direction.  in: nodes (B, [nz, ny,] nx) through its
 * strides; out dense (B, ngp_1d^nsd, elements...), G = (kg ngp + jg) ngp + ig; grad_in dense nodes (overwritten).
 * (nodes - 1) % (nbf_1d - 1) == 0 per direction.  Q1 meshes in 2-D / 3-D take the tuned dn_fem_gp_eval_* above.
 */
int dn_fem_gp_eval_general_f32(const dn_field* in, int nsd, int batch, int nx, int ny, int nz, int nbf_1d,
                               int ngp_1d, const float* factors, float* out, void* stream);
int dn_fem_gp_eval_general_adj_f32(const float* grad_out, int nsd, int batch, int nx, int ny, int nz, int nbf_1d,
                                   int ngp_1d, const float* factors, float* grad_in, void* stream);

/*
 * Load-vector assembly for the forcing-at-Gauss-points form (e8_2d_poisson_mms.py:154-175: f_gp * u_gp summed with
 * the quadrature weights).  The term is LINEAR in u, so it equals sum_a b_a u_a with
 *     b_a = sum over the elements e around node a, over Gauss points g:  w_g N_a(g) f_gp[e, g]
 * (reference-element weights).  This call assembles b once; every later loss call passes it as `f` with
 * dn_consts.flags = DN_F_LOAD_VECTOR and the streaming kernels read 4 bytes per node instead of 4 ngp^nsd per element.
 * fgp: dense (B|1, ngp_1d^nsd, elems), stride_b = 0 -> one b for the whole batch; out: dense nodes
 * (stride_b == 0 ? 1 : g->batch, [nz,] ny, nx), overwritten.  Uses g->nsd, batch, nx, ny, nz, ngp_1d.
 */
int dn_fem_load_vector_f32(const dn_field* fgp, const dn_geom* g, float* out, void* stream);

/*
 * Device-side producers of the path's INPUT tensors (what the reference's dataset classes build on the host with
 * numpy and ship through a DataLoader every step).  Outputs: `inputs` dense (B, 3, [N,] H, W) fp32 =
 * [nu or domain, bc1, bc2] and `forcing` dense (B, 1, ...) zero-filled (nullable), the layout loss() slices
 * (examples/poisson/parametric/2_klsum_fem.py:36-38).  All pointers are device pointers unless said otherwise.
 *
 * dn_gen_kl_inputs_f32     KLSumStochastic (DiffNet/datasets/parametric/klsum.py:10-46) over
 *                          generate_diffusivity_tensor (DiffNet/gen_input_calc.py:74-181): nu = exp(KL sum of `nterms`
 *                          modes), bc1 = first column, bc2 = last column.  coeffs: (B, nterms) fp64 (the Sobol
 *                          samples); omega: HOST array of the nterms roots for `eta` (calculate_omega_based_on_eta);
 *                          evaluated in fp64 without fma contraction, rounded to fp32 at the end like the reference.
 *                          nsd == 3: `inputs` is the (B, 1, N, N, N) diffusivity only (the reference has no 3-D KL
 *                          dataset class), axes (y, x, z) as np.meshgrid orders them.  `tables`: device scratch of
 *                          dn_gen_kl_table_bytes(nterms, size) bytes.  size % 4 == 0.
 * dn_gen_image_inputs_f32  ImageIMBack (DiffNet/datasets/parametric/images.py:9-49): img = (B, H, W) greyscale bytes
 *                          (PIL convert('L')); domain = 1 - (img > 0), bc1 = (img > 0), bc2 = the four edges.
 * dn_gen_voxel_inputs_f32  VoxelIMBackRAW / load_raw (DiffNet/datasets/single_instances/voxels.py:8-61): raw = the bytes
 *                          of <name>inouts.raw (Fortran order over numDiv = (d0, d1, d2)); inside = raw / 254.0 > 0.25;
 *                          the block sits at `offset` (the reference hard-codes 32) in a domain_size^3 box; one sample.
 * dn_gen_star_inputs_f32, dn_gen_box_masks_3d_f32
 *                          synthetic immersed geometries for benchmarks / tests (no reference counterpart: stand-ins
 *                          for its image and SIMP-topology datasets).  params: 11 floats per sample (cx, cy, r0,
 *                          a[4], phase[4]) / 19 ints per sample (n, lo[3][3], hi[3][3]).
 */
size_t dn_gen_kl_table_bytes(int nterms, int size);
int dn_gen_kl_inputs_f32(const double* coeffs, int batch, int nterms, const double* omega, double eta, int nsd,
                         int size, void* tables, size_t table_bytes, float* inputs, float* forcing, void* stream);
int dn_gen_image_inputs_f32(const unsigned char* img, int batch, int height, int width, float* inputs,
                            float* forcing, void* stream);
int dn_gen_voxel_inputs_f32(const unsigned char* raw, int d0, int d1, int d2, int domain_size, int offset,
                            float* inputs, float* forcing, void* stream);
int dn_gen_star_inputs_f32(const float* params, int batch, int size, float* inputs, float* forcing, void* stream);
int dn_gen_box_masks_3d_f32(const int* params, int batch, int size, float* source, float* sink, float* forcing,
                            void* stream);

/* x[i] *= *factor_dev for i < n, skipping all memory traffic when *factor_dev == 1.0f
 * (the usual loss.backward() case).  factor_dev is a device pointer: no host sync. */
int dn_scale_inplace_f32(float* x, size_t n, const float* factor_dev, void* stream);
/* x[b, i] *= factors_dev[b] for b < batch, i < n_per_sample (x dense (batch, n_per_sample)): the backward of a
 * reduction = none loss with a (B,) grad_output.  factors_dev is a device pointer: no host sync. */
int dn_scale_per_sample_f32(float* x, int batch, size_t n_per_sample, const float* factors_dev, void* stream);

/*
 * Halo planes over NVLink peer memory (z-slab decomposition of one 3-D field over several GPUs,
 * one process per GPU; new functionality, SURVEY.md 8e -- the reference is single-GPU there).
 *
 * dn_peer_put_f32: copy n floats (n % 4 == 0, 16-byte aligned) from `src` (local) to `dst_peer`
 *   (a buffer of the neighbouring GPU mapped into this process, e.g. through CUDA IPC) with
 *   stores over NVLink, then publish ++(*local_counter) in `*remote_flag` (a word in the
 *   neighbour's memory) with system-scope release ordering.  `ticket`: a zero-initialised local
 *   device word (scratch).
 * dn_peer_wait_f32: wait (on the device, bounded by max_spins polls; no host involvement) until
 *   *flag >= ++(*expect), then copy the staged plane into `halo` (both local).  `status`: two
 *   zero-initialised local device ints; status[0] becomes 1 if the wait timed out.
 * Both are asynchronous on `stream` and may be captured in a CUDA graph.
 */
/* Receive buffers for the peer transport.  They are the one thing this library allocates (a raw
 * cudaMalloc on the current device, zero-filled, owned by the caller through dn_peer_free): a CUDA
 * IPC handle must name a whole allocation, which a framework's caching allocator does not hand
 * out.  dn_peer_export writes the 64-byte IPC handle; dn_peer_import maps a neighbour's buffer
 * into THIS process for access from the CURRENT device (peer access is enabled as needed);
 * dn_peer_unimport unmaps it. */
int dn_peer_alloc(size_t bytes, void** ptr);
int dn_peer_free(void* ptr);
int dn_peer_export(void* ptr, unsigned char handle[64]);
int dn_peer_import(const unsigned char handle[64], void** ptr);
int dn_peer_unimport(void* ptr);
int dn_peer_put_f32(float* dst_peer, const float* src, size_t n, int32_t* remote_flag,
                    int32_t* local_counter, uint32_t* ticket, void* stream);
int dn_peer_wait_f32(float* halo, const float* staged, size_t n, const int32_t* flag, int32_t* expect,
                     int64_t max_spins, int32_t* status, void* stream);

/*
 * All-reduce (sum) of one float per rank through peer memory, summed in rank order (bit-identical
 * on every rank).  `slots`: local receive area = double[world] followed by int32[world], zero-
 * initialised, 8-byte aligned; `peer_slots`: DEVICE array of `world` pointers to the same area of
 * every rank as mapped in this process (entry `rank` ignored); `counter`, `status`: local device
 * words (zero-initialised).  Consecutive calls must alternate between two slot areas (parity) so a
 * fast rank cannot overwrite values a slow rank has not read yet.  world <= 32.
 */
int dn_peer_allreduce_f32(const float* partial, float* out, double* slots, double* const* peer_slots,
                          int rank, int world, int32_t* counter, int64_t max_spins, int32_t* status,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFNET_FEM_H_ */
