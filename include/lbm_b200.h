/* lbm_b200.h — C ABI of the B200-native D2Q9 lattice-Boltzmann time step.
 *
 * Drop-in boundary for the hot path of cristian-jfv/lattice-boltzmann-method: the reference has no
 * FFI layer of its own (its callable surface is C++ on torch::Tensor: src/solver.hpp:8-36,
 * src/domain.hpp:5-15, src/colour.hpp:9-42, src/differential.hpp:6-53, src/ibm.hpp:9-34,
 * src/params.hpp:9-49, plus the loop bodies of test/<driver>.cpp), so this header is what a cgo-/ctypes-/
 * C++-side binding of that surface binds to.  Each entry point cites the reference interface it
 * replaces.  INTEGRATION.md shows the reference-side stubs.
 *
 * Conventions
 *   - every function returns an lbm_status (0 = ok); lbm_last_error() gives the message of the
 *     last failure on the calling thread.  No C++ exception crosses this boundary (the reference
 *     throws std::runtime_error / c10::Error instead: src/params.cpp:13, src/colour.cpp:45).
 *   - "AoS" buffers use the reference layout: fp64, shape {X,Y,Q} row-major, axis 0 = x ("rows"),
 *     axis 1 = y ("columns"), Q innermost (src/domain.cpp:7-11).  Direction order and weights are
 *     solver::c / solver::E (src/solver.cpp:12-21).
 *   - host pointers unless a name ends in _dev.  The caller owns host buffers, the library owns
 *     all device memory.  There is NO CPU fallback: without a CUDA device every compute entry
 *     point fails with LBM_ERR_CUDA.
 *   - one lbm_domain = one slab (rows [x0,x1) of the global grid) on one GPU, the unit the
 *     reference calls `struct domain` (src/domain.hpp:5-15, test/decompose_domain.cpp:101-104).
 */
#ifndef LBM_B200_H
#define LBM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lbm_domain lbm_domain;

typedef enum
{
  LBM_OK = 0,
  LBM_ERR_INVALID = 1,     /* bad argument / inconsistent description */
  LBM_ERR_CUDA = 2,        /* CUDA runtime failure or no device */
  LBM_ERR_CONFIG = 3,      /* missing / malformed TOML key (message mirrors the reference's) */
  LBM_ERR_UNSUPPORTED = 4, /* valid request outside what this build implements */
  LBM_ERR_COMM = 5         /* NCCL failure */
} lbm_status;

const char* lbm_last_error(void);
/* library version string, e.g. "lbm_b200 0.1 (sm_100a)" */
const char* lbm_version(void);

/* ------------------------------------------------------------------------------------------------
 * Models (one fused collide+stream kernel family per model)
 * ---------------------------------------------------------------------------------------------- */
typedef enum
{
  LBM_MODEL_BGK = 0,     /* single lattice: drivers 10-14 (test/horizontal_poiseuille_test.cpp, cylinder_test.cpp,
                            free_stream_test.cpp, specular_boundary_test.cpp, gravity_test.cpp) */
  LBM_MODEL_BGK_ADE = 1, /* fluid + advection-diffusion lattice: test/rectangle_sedimentation_test.cpp */
  LBM_MODEL_MRTCG = 2,   /* MRT colour gradient: test/mrtcg_rayleigh_taylor.cpp, test/mrtcg_static_droplet.cpp */
  LBM_MODEL_RK = 3,      /* Rothman-Keller droplet: test/rk_static_droplet_test.cpp */
  LBM_MODEL_MRT_CSF = 5, /* MRT colour gradient with a continuum-surface-force perturbation: test/mrt_rayleigh_taylor.cpp
                            (curvature of the interface normal, interfacial tension carried into the next velocity) */
  LBM_MODEL_KBC = 4      /* entropic central-moment collision ulbm::d2q9::kbc (src/ulbm.hpp:11-90, src/ulbm.cpp):
                            test/ulbm_double_shear_flow.cpp, test/ulbm_poiseuille.cpp; omega = the class's s2 */
} lbm_model;

typedef enum
{
  LBM_EQ_COMPRESSIBLE = 0,  /* solver::equilibrium        src/solver.cpp:51-62 */
  LBM_EQ_INCOMPRESSIBLE = 1, /* solver::incomp_equilibrium src/solver.cpp:39-49 */
  /* lbm_init_equilibrium only: kbc::eval_equilibrium (src/ulbm.cpp:246-262) */
  LBM_EQ_KBC = 2,            /* with ux2 = ux^2, uy2 = uy^2 */
  LBM_EQ_KBC_FRESH = 3       /* as called on a fresh object (test/ulbm_double_shear_flow.cpp:97): the members ux2, uy2,
                                which only collide() refreshes, are still zero */
} lbm_equilibrium_kind;

typedef enum
{
  LBM_FORCE_NONE = 0,
  LBM_FORCE_UNIFORM = 1, /* test/gravity_test.cpp:143-160: u += Fg, source term with ics2=1/3, ics4=1/9 */
  LBM_FORCE_IBM = 2      /* test/cylinder_test.cpp:110-127: ROI force field from the immersed boundary */
} lbm_force_kind;

typedef struct
{
  double rho_0, alpha, A, nu, beta; /* [red]/[blue] tables: src/colour.cpp:11-21 */
} lbm_colour_desc;

typedef struct
{
  int model;          /* lbm_model */
  int X, Y;           /* GLOBAL grid (rows, columns) */
  int x0, x1;         /* rows of the global grid owned by this domain, [x0,x1); x0=0,x1=X for one GPU */
  int device;         /* CUDA device ordinal */
  /* --- BGK / BGK_ADE */
  double omega;       /* 1/tau (params::lattice::omega, src/params.cpp:57) */
  int equilibrium;    /* lbm_equilibrium_kind */
  int force;          /* lbm_force_kind */
  double Fg[2];       /* LBM_FORCE_UNIFORM; MRTCG: gravity vector (mrtcg_rayleigh_taylor.cpp:403) */
  double w_s;         /* BGK_ADE: settling velocity added to BOTH components (rectangle_sedimentation_test.cpp:125) */
  double omega_g;     /* BGK_ADE: relaxation of the second lattice (lp.omega/1.0, :131) */
  /* --- MRTCG / RK */
  lbm_colour_desc red, blue;
  double sigma;       /* MRTCG: [general].sigma (RT) or 0.1 (droplet) */
  double delta;       /* interface half-width of the relaxation blend: 0.1 (MRTCG), 0.98 (RK) */
  int add_force;      /* MRTCG: 1 = RT driver (:463-464), 0 = droplet driver (source not added) */
} lbm_config;

/* fills *cfg with zeros and the defaults (model BGK, compressible, no force, delta 0.1, device 0) */
void lbm_config_default(lbm_config* cfg);

/* replaces `domain::domain(R,C,Q)` (src/domain.cpp:3-12) and the per-driver tensor allocations
 * (e.g. test/cylinder_test.cpp:49-53): allocates the SoA device state of one slab. */
int lbm_create(const lbm_config* cfg, lbm_domain** out);
int lbm_destroy(lbm_domain* d);

/* ------------------------------------------------------------------------------------------------
 * Boundary conditions.  The reference writes them as ordered slice assignments after
 * solver::advect (post-stream, e.g. test/horizontal_poiseuille_test.cpp:146-152) or on f_coll
 * before it (pre-stream, e.g. :140, rectangle_sedimentation_test.cpp:138-141).  An lbm_bc_op is
 * ONE such assignment; ops are applied in the order added, so later ops win where regions
 * overlap, exactly like the reference.  Slices use torch semantics (negative = from the end,
 * LBM_END = "None").  Coordinates are GLOBAL; each slab keeps the part it owns.
 * ---------------------------------------------------------------------------------------------- */
#define LBM_END 2147483647

typedef enum
{
  /* post-stream: f_adve[region, dst_q] = coef * f_coll[src_node(region), src_q] + cst */
  LBM_BC_LINEAR = 0,
  /* post-stream anti-bounce-back with a fixed wall velocity (test/cylinder_test.cpp:135-154):
   *   f_adve[region, opp(src_q)] = -f_coll[region, src_q] + (2 + 9 (c.uw)^2 - 3 uw.uw) w     */
  LBM_BC_ABB_FIXED = 1,
  /* same with uw = 1.5 u[.., -1] - 0.5 u[.., -2] of the previous moments
   * (test/rectangle_sedimentation_test.cpp:163-172); region must be a column                      */
  LBM_BC_ABB_EXTRAPOLATED = 2,
  /* ADE inlet (rectangle_sedimentation_test.cpp:204-218): lattice 1,
   *   g_adve[region, opp(src_q)] = -g_coll[region, src_q] + 2 geq_q(u + w_s, C_w[x])               */
  LBM_BC_ADE_INLET = 3,
  /* pre-stream pressure-periodic rows (test/horizontal_poiseuille_test.cpp:25-45):
   *   f_coll[row] = feq(rho_bc, u[src_row]) + f_coll[src_row] - f_equi[src_row]                    */
  LBM_BC_PRESSURE_PERIODIC = 4,
  /* pre-stream copy (zero gradient, rectangle_sedimentation_test.cpp:138-141):
   *   f_coll[region, :] = f_coll[src_node(region), :]                                              */
  LBM_BC_COPY_PRE = 5
} lbm_bc_kind;

typedef enum
{
  LBM_SRC_SAME_NODE = 0, /* f_coll at the node being written */
  LBM_SRC_SHIFT = 1,     /* node + (src_a, src_b) */
  LBM_SRC_ROW = 2,       /* same column, absolute row src_a (negative = from the end) */
  LBM_SRC_COL = 3        /* same row, absolute column src_a (negative = from the end) */
} lbm_bc_src;

typedef struct
{
  int kind;                 /* lbm_bc_kind */
  int lattice;              /* 0 = f / red, 1 = g / blue, -1 = both lattices */
  int x_begin, x_end;       /* row slice   [x_begin, x_end) */
  int y_begin, y_end;       /* column slice [y_begin, y_end) */
  int dst_q;                /* population written; -1 = all nine, each from the same q of the source */
  int src_q;                /* population read */
  int src_mode;             /* lbm_bc_src */
  int src_a, src_b;
  double coef, cst;         /* LBM_BC_LINEAR */
  double uw[2];             /* LBM_BC_ABB_FIXED */
  double rho_bc;            /* LBM_BC_PRESSURE_PERIODIC */
  const double* per_row;    /* LBM_BC_ADE_INLET: C_w[X] (global rows), copied at add time */
} lbm_bc_op;

void lbm_bc_op_default(lbm_bc_op* op);
int lbm_bc_clear(lbm_domain* d);
int lbm_bc_add(lbm_domain* d, const lbm_bc_op* op);
/* Half-way bounce-back around an arbitrary (staircase) solid body: solid = {X,Y} GLOBAL mask, non-zero = solid.
 * For every node n and direction q whose upstream neighbour n - c_q (periodic, like solver::advect) lies on the other
 * side of the surface: f_adve[n, q] = f_coll[n, opp(q)] — the link-wise rule of the reference's obstacle walls
 * (test/rectangle_sedimentation_test.cpp:186-196; BASELINE.json configs[1] "cylinder ... with bounce-back").
 * Appends ordinary LBM_BC_LINEAR ops (one per run of columns); call lbm_bc_commit afterwards.  X, Y must be the
 * domain's global size. */
int lbm_bc_add_solid(lbm_domain* d, int lattice, const unsigned char* solid, int X, int Y);
/* compiles the op list into per-node programs (must be called once before stepping) */
int lbm_bc_commit(lbm_domain* d);
/* bit-exact introspection of the compiled masks (SURVEY §8: "boundary-node masks ... bit-exact"):
 * for lattice l, mask[(x*Y + y)*9 + q] = 1 + index of the post-stream op that owns (x,y,q), 0 = plain pull.
 * x runs over the slab's own rows.  */
int lbm_bc_get_mask(lbm_domain* d, int lattice, int32_t* mask);

/* Ready-made rule lists: each one is the ordered list of slice assignments of one reference driver,
 * expressed with lbm_bc_add and committed (lbm_bc_clear + adds + lbm_bc_commit).
 *   lbm_preset_poiseuille        test/horizontal_poiseuille_test.cpp:140,146-152 (also gravity_test.cpp:163-176,
 *                                decompose_domain.cpp:155-178 once the slabs are linked)
 *   lbm_preset_specular_channel  test/specular_boundary_test.cpp:116,122-128
 *   lbm_preset_free_stream       test/free_stream_test.cpp:106-134, test/cylinder_test.cpp:135-163
 *   lbm_preset_sedimentation     test/rectangle_sedimentation_test.cpp:138-141,150-196,204-236
 *   lbm_preset_mrtcg             test/mrtcg_rayleigh_taylor.cpp:495-533
 *   lbm_preset_rk                test/rk_static_droplet_test.cpp:204-211                              */
int lbm_preset_poiseuille(lbm_domain* d, double rho_in, double rho_out);
int lbm_preset_specular_channel(lbm_domain* d, double rho_in, double rho_out);
int lbm_preset_free_stream(lbm_domain* d, double uwx, double uwy);
int lbm_preset_sedimentation(lbm_domain* d, double u_lb, const double* C_w, int R23, int C28, int C38);
int lbm_preset_mrtcg(lbm_domain* d);
int lbm_preset_rk(lbm_domain* d);
/* fully periodic box (solver::advect alone): no rules */
int lbm_preset_periodic(lbm_domain* d);

/* ------------------------------------------------------------------------------------------------
 * State import / export in the reference layout
 * ---------------------------------------------------------------------------------------------- */
/* f_adve of one lattice, AoS {x1-x0, Y, 9}  (replaces direct tensor access, e.g. cylinder_test.cpp:86) */
int lbm_set_f(lbm_domain* d, int lattice, const double* f_aos);
int lbm_get_f(lbm_domain* d, int lattice, double* f_aos);
/* moments of the CURRENT post-stream state, as the next loop iteration of the reference would
 * compute them: rho {X,Y,1} (solver::calc_rho), u {X,Y,2} (calc_u / calc_incomp_u, plus the
 * model's force shift).  Either pointer may be NULL.  BGK_ADE: lattice 1 gives C in rho.          */
int lbm_get_moments(lbm_domain* d, int lattice, double* rho, double* u);
/* Snapshot without stalling the time loop (SURVEY §8(f) rank 1; the reference copies CUDA->CPU tensors
 * synchronously, e.g. test/cylinder_test.cpp:94-98): the fields of the CURRENT state are staged on the
 * domain's stream and copied to the caller's buffers on a separate copy stream while later lbm_step calls
 * run.  rho {X,Y,1}, u {X,Y,2}, phase {X,Y} (two-phase models only); any may be NULL.  Pinned host memory
 * gives a true overlap.  The buffers are valid after lbm_snapshot_wait; a second snapshot (or lbm_get_*)
 * issued earlier waits for the first copy on the device, not on the host.                          */
int lbm_snapshot_async(lbm_domain* d, int lattice, double* rho, double* u, double* phase);
int lbm_snapshot_wait(lbm_domain* d);
/* two-phase fields of the current state: phase {X,Y} (eval_phase_field), rho_r, rho_b {X,Y}     */
int lbm_get_phase(lbm_domain* d, double* phase, double* rho_r, double* rho_b);
/* LBM_MODEL_MRT_CSF: interf_tension {X,Y,2} of the last step (the driver snapshots it: mrt_rayleigh_taylor.cpp:485-486) */
int lbm_get_interfacial_tension(lbm_domain* d, double* Fs_aos);
/* LBM_MODEL_RK: the diagnostic fields test/rk_static_droplet_test.cpp snapshots at the top of every iteration (:546-600) —
 * functions of the CURRENT state only, none feeds the step (it uses grad and |grad| alone, :213-237).  Call before
 * lbm_step(d, 1) to reproduce iteration t of the driver.  Host buffers in the reference's tensor layouts; NULL = skip.
 *   phase {X,Y} (rhons)   grad {X,Y,2} (gradxs, gradys: [0] = the driver's partial.x, along axis 1)   norm {X,Y} (norms)
 *   n {X,Y,2} (nxs, nys) = -normalize(grad where |grad| > 0.1 max|grad|, else 0)   K {X,Y} (Ks, eval_local_curvature :440-446)
 *   Fs {X,Y,2} (Fsxs, Fsys) = sigma/2 K grad   eta {X,Y,9} (eval_eta :398-413)   kappa {X,Y,9} (kappas, eval_kappa :415-438)
 *   rparams {X,Y} = 1/tau(phase)   omega1, omega2, omega3 {X,Y,9}: the RED colour's operators (:255-262, :239-245, :232-236)
 * Monolithic domains, or every rank of an lbm_comm_init ring at once (the cut's max|grad| is reduced over the ring, the
 * normal planes swap halos: SURVEY 8(e)); LBM_ERR_UNSUPPORTED on linked slabs of one process.                              */
typedef struct lbm_rk_diag
{
  double *phase, *grad, *norm, *n, *K, *Fs, *eta, *kappa, *rparams, *omega1, *omega2, *omega3;
} lbm_rk_diag;
int lbm_rk_diagnostics(lbm_domain* d, double sigma, const lbm_rk_diag* out);
/* two-phase models carry u between steps (mrtcg_rayleigh_taylor.cpp:476-477); initial value.      */
int lbm_set_u(lbm_domain* d, const double* u_aos);
/* LBM_MODEL_KBC: the class keeps m0 / m1 as members that its first collide() reads before they are recomputed
 * from the populations (test/ulbm_poiseuille.cpp:93 starts from adve_f = 0, m0 = 1, m1 = 0).  After an import,
 * the FIRST step takes rho {X,Y,1}, u {X,Y,2} from here instead of the moments of the imported populations.  */
int lbm_set_moments(lbm_domain* d, const double* rho, const double* u);
/* initial condition helpers that mirror the drivers' own initialisation:
 *   BGK       f = incomp_equilibrium(u0, rho0)              (cylinder_test.cpp:86)
 *   two-phase adv_f = eq(rho_r, rho_b, u)                   (mrtcg_rayleigh_taylor.cpp:407-410)
 * lbm_init_equilibrium returns once the HOST buffers have been read (they may be reused); the copy runs on its own stream,
 * beside whatever the domain is still doing, and the equilibrium kernel is ordered behind both — feeding one initial state
 * after the other overlaps the copy with the previous run's steps and with its asynchronous snapshot. */
int lbm_init_equilibrium(lbm_domain* d, int lattice, int equilibrium_kind, const double* rho, const double* u);
int lbm_init_two_phase(lbm_domain* d, const double* rho_r, const double* rho_b, const double* u);

/* ------------------------------------------------------------------------------------------------
 * Immersed boundary (src/ibm.hpp:21-34, src/ibm.cpp:60-190)
 * ---------------------------------------------------------------------------------------------- */
/* replaces `ibm ib{tbl, name, dev}`: marker coordinates in GLOBAL lattice units.  With slabs, hand EVERY slab the same
 * list: a slab that owns none of the ROI rows ignores it (LBM_OK, no body), slabs that share the ROI exchange the moments
 * of their own ROI nodes every step and keep identical force fields.  The ROI columns must be interior ([2, Y-2)). */
int lbm_ibm_set_markers(lbm_domain* d, const double* xs, const double* ys, int n_markers, int m_max);
/* A constant body force on a rectangle of nodes, entering through the source term only (no velocity shift):
 *   f_coll[region] += (1 - omega/2) ((ics2 + ics4 u.c_q)(F.c_q) - ics2 u.F) w_q
 * test/decompose_domain_loop.cpp:66-69,151-158 (F = (3e-3, 0), ics2 = 3, ics4 = 9, rows L/4+5 .. L/4+55 of block A).
 * Slices are GLOBAL with torch semantics (clamped).  Occupies the force-field slot of the immersed boundary: the domain
 * must have been created with force = LBM_FORCE_IBM, and markers and a region force exclude each other. */
int lbm_set_force_region(lbm_domain* d, int x_begin, int x_end, int y_begin, int y_end, double Fx, double Fy, double ics2,
                         double ics4);
/* ib.rows / ib.cols: roi = {row_start,row_stop,col_start,col_stop} */
int lbm_ibm_get_roi(lbm_domain* d, long* roi4);
/* last Eulerian force density F {roi_rows, roi_cols, 2} computed inside lbm_step (cylinder_test.cpp:110) */
int lbm_ibm_get_force(lbm_domain* d, double* F_aos);
/* stand-alone ibm::eulerian_force_density(u, rho) on AoS inputs {X,Y,2}, {X,Y,1} (src/ibm.cpp:158-190) */
int lbm_ibm_force(lbm_domain* d, const double* u_aos, const double* rho_aos, double* F_aos);

/* ------------------------------------------------------------------------------------------------
 * Force on a body, recorded on the device every step — replaces the accumulation of F_s that test/cylinder_test.cpp:112
 * snapshots for an offline sum.  Each domain records the force that the fluid on ITS rows exerts on one body, in lattice
 * units, for the step that advances f_coll(t) to f_adve(t+1); the parts of linked slabs / ring ranks add up to the total.
 *   bounce-back body: momentum exchange F = sum 2 c_opp(q) f_coll(t)[n, opp(q)] over the links (n, q) with n a fluid node
 *                     of this slab and n - c_q solid (periodic wrap, as lbm_bc_add_solid)
 *   immersed body:    F = -sum F_euler over the ROI nodes of this slab's rows (F_euler: the field the step adds)
 * The sum is deterministic (no floating-point atomics) and lands in a device ring; nothing crosses to the host until
 * lbm_body_force_read.  Single-phase models only (two-phase: LBM_ERR_UNSUPPORTED).  Without a record the step is unchanged.
 * ---------------------------------------------------------------------------------------------- */
/* solid != NULL: the staircase body of lbm_bc_add_solid(d, 0, solid, X, Y) ({X,Y} GLOBAL mask); needs lbm_bc_commit first,
 *                and every counted link must be owned by a plain bounce-back LBM_BC_LINEAR op (same node, src_q = opp(q),
 *                coef 1, cst 0), else LBM_ERR_INVALID.  A later lbm_bc_commit / lbm_bc_clear ends the record.
 * solid == NULL: the immersed body of lbm_ibm_set_markers (F_s of test/cylinder_test.cpp:112, sign flipped); X, Y are
 *                ignored.  A later lbm_ibm_set_markers / lbm_set_force_region ends the record.
 * capacity = steps kept in the device ring.  Calling it again replaces the record and restarts the count. */
int lbm_body_force_record(lbm_domain* d, const unsigned char* solid, int X, int Y, int capacity);
/* Force on the body from the last min(recorded, capacity, max_steps) steps, in step order.
 * F[2k] is along axis 0 (x, rows) and F[2k+1] along axis 1.  *first_step is the index of entry 0,
 * counted from the record call.  Synchronises the domain's stream. */
int lbm_body_force_read(lbm_domain* d, double* F, int max_steps, int* n_steps, long long* first_step);
int lbm_body_force_stop(lbm_domain* d);

/* ------------------------------------------------------------------------------------------------
 * Time stepping — replaces the loop body of each driver (SURVEY §3.1-3.3)
 * ---------------------------------------------------------------------------------------------- */
/* advance n_steps; asynchronous on the domain's stream */
int lbm_step(lbm_domain* d, int n_steps);
int lbm_synchronize(lbm_domain* d);
/* device time of the last lbm_step call in milliseconds (CUDA events on the domain's stream) */
int lbm_last_step_ms(lbm_domain* d, float* ms);
/* number of kernels launched by this domain so far */
int lbm_kernel_launches(lbm_domain* d, long long* n);
/* the cudaStream_t the domain runs on (as void*) */
int lbm_get_stream(lbm_domain* d, void** stream);
/* capture one step into a CUDA graph and replay it in lbm_step (launch-bound small grids) */
int lbm_use_graph(lbm_domain* d, int enable);
/* per-kernel-class device timing with CUDA events on the domain's stream (the reference has no
 * timers at all, SURVEY §5).  enable != 0 starts a fresh recording; lbm_profile_read synchronises
 * and returns the summed duration and the launch count of one class since then. */
typedef enum
{
  LBM_PROF_INTERIOR = 0, /* fused collide+stream over the interior nodes (the dominant kernel) */
  LBM_PROF_BOUNDARY = 1, /* table-driven boundary-node kernel */
  LBM_PROF_FIXUP = 2,    /* pre-stream rules */
  LBM_PROF_GHOST = 3,    /* ghost-row wrap / exchange */
  LBM_PROF_IBM = 4,      /* immersed-boundary pre-pass */
  LBM_PROF_MOMENTS = 5,  /* two-phase models: stream + moments kernel */
  LBM_PROF_EARLY = 6,    /* single-phase family: the same kernel over the EARLY rows, on the side stream beside the bulk launch */
  LBM_PROF_CLASSES = 7
} lbm_prof_class;
int lbm_profile_enable(lbm_domain* d, int enable);
int lbm_profile_read(lbm_domain* d, int prof_class, double* total_ms, long long* launches);
/* single-phase family: how the step splits the slab's rows between the early launch (first / last row, rows with listed nodes
 * in interior columns or feeding a stage, the immersed body's ROI rows) and the bulk launch; both run k_bgk_interior */
int lbm_row_split(lbm_domain* d, int* n_early_rows, int* n_bulk_rows);

/* ------------------------------------------------------------------------------------------------
 * Multi-GPU slabs (test/decompose_domain.cpp:181-187 generalised to P slabs along axis 0)
 * ---------------------------------------------------------------------------------------------- */
#define LBM_UNIQUE_ID_BYTES 128
/* rank 0 creates the id, the launcher broadcasts it (torch.distributed / MPI / file) */
int lbm_comm_unique_id(char id[LBM_UNIQUE_ID_BYTES]);
/* joins the slab ring: neighbours are rank-1 and rank+1 (periodic, like solver::advect).
 * Call order: lbm_create -> lbm_comm_init -> rules / markers -> state import -> lbm_step.  A two-phase domain that
 * already holds state is refused (LBM_ERR_INVALID): its imports swap the moment-plane halos of the cuts when they run. */
int lbm_comm_init(lbm_domain* d, const char id[LBM_UNIQUE_ID_BYTES], int n_ranks, int rank);
/* d joins the ring `member` belongs to, on member's communicator (no second ncclCommInitRank: seconds on eight ranks).  For
 * drivers that keep several domains on the same slabs — the reference's drivers hold fluid, sediment and colour lattices in
 * separate tensors over one decomposition (test/decompose_domain.cpp:60-95) — and for running cases one after the other.
 * Same device, same decomposition rule and call order as lbm_comm_init; step the sharing domains one at a time. */
int lbm_comm_share(lbm_domain* d, lbm_domain* member);
/* Collective consistency check of the ring (optional; every rank calls it after its setup, before the first lbm_step):
 * grids, model, force mode, and that every slab owning rows of an immersed body's ROI was handed that body's marker list —
 * the misuse that otherwise leaves ranks waiting for a row exchange nobody posts.  LBM_ERR_COMM on every rank, with the
 * difference in lbm_last_error(), instead of a hang.  LBM_OK without a communicator.                                    */
int lbm_comm_check(lbm_domain* d);
/* single-process alternative: link two domains on the same host process; ghost rows are exchanged with
 * cudaMemcpyPeerAsync (what decompose_domain.cpp's "bind" does between tensors) */
int lbm_link_neighbours(lbm_domain* d, lbm_domain* lower, lbm_domain* upper);
/* advance a set of linked slabs in lock step (what decompose_domain.cpp's loop does for A and B) */
int lbm_step_group(lbm_domain* const* domains, int n_domains, int n_steps);
/* Multi-block binding across a COLUMN face — the "Bind the domains" lines of test/decompose_domain_loop.cpp:232-261, one
 * call per direction.  The three populations that enter block d through its edge column (`side` 0 = first column,
 * populations 2, 5, 6; `side` 1 = last column, populations 4, 7, 8) on rows [row_begin, row_begin + n_rows) stream in from
 * the facing edge column of `other` (its last column for side 0, its first for side 1), rows
 * [other_row_begin, other_row_begin + n_rows):
 *   f_adve[row_begin + k, col, q] = other.f_coll[other_row_begin + k - c_qx, col', q]     for 0 <= k - c_qx < n_rows,
 * i.e. the diagonal populations keep the block's own (wall) rule at the two ends of the face, as in the reference.
 * Blocks keep their own coordinates and rule lists (like the reference's `domain A{L, L4}; domain B{L4, L2}; ...`), must own
 * all their rows, and are advanced together with lbm_step_group.  Call lbm_bc_commit after the last binding. */
int lbm_link_face(lbm_domain* d, int side, int row_begin, int n_rows, lbm_domain* other, int other_row_begin);
/* The same binding between blocks that live in DIFFERENT processes (one block per GPU), over NCCL send/recv:
 *   lbm_comm_init_blocks   joins the block communicator (rank 0 makes the id with lbm_comm_unique_id); unlike lbm_comm_init
 *                          the members are independent grids, there is no slab ring
 *   lbm_link_face_rank     like lbm_link_face, the facing block named by the rank that owns it; one call per direction ON THE
 *                          READING RANK only
 *   lbm_comm_faces_commit  collective, after the last lbm_link_face_rank of every rank and before lbm_bc_commit / lbm_step:
 *                          the ranks exchange their link lists, so that each learns which rows of its edge columns the others
 *                          read and sends them every step
 * then plain lbm_step on every rank, the same number of steps everywhere (each step holds one grouped exchange).
 * test/decompose_domain_loop.cpp:232-261 with A, B, C, D on four ranks. */
int lbm_comm_init_blocks(lbm_domain* d, const char id[LBM_UNIQUE_ID_BYTES], int n_ranks, int rank);
int lbm_link_face_rank(lbm_domain* d, int side, int row_begin, int n_rows, int peer_rank, int peer_row_begin);
int lbm_comm_faces_commit(lbm_domain* d);
/* bit-exact decomposition indexing: rows [x0,x1) for `rank` of `n_ranks` over X rows */
int lbm_decompose_rows(int X, int n_ranks, int rank, int* x0, int* x1);

/* ------------------------------------------------------------------------------------------------
 * Granular operators, one-to-one with namespace solver (src/solver.hpp:11-36) and class
 * differential (src/differential.hpp:48-51), on AoS host buffers; each runs a CUDA kernel.
 * ---------------------------------------------------------------------------------------------- */
int lbm_calc_rho(const double* f, int X, int Y, double* rho);
int lbm_calc_u(const double* f, const double* rho, int X, int Y, double* u);
int lbm_calc_incomp_u(const double* f, int X, int Y, double* u);
int lbm_equilibrium(const double* u, const double* rho, int X, int Y, double* feq);
int lbm_incomp_equilibrium(const double* u, const double* rho, int X, int Y, double* feq);
int lbm_collision(const double* f, const double* feq, double omega, int X, int Y, double* fcoll);
int lbm_advect(const double* f, int X, int Y, double* g);
/* 5x5 isotropic differences, replicate padding: dx along axis 0, dy along axis 1 */
int lbm_differential(const double* psi, int R, int C, double* dx, double* dy);
/* the RK driver's 3x3 operator (test/rk_static_droplet_test.cpp:48-107): its "x" is along axis 1 */
int lbm_differential3(const double* psi, int R, int C, double* dx, double* dy);

/* ------------------------------------------------------------------------------------------------
 * parameters.toml surface (src/params.cpp, src/colour.cpp) — host-only scalar code
 * ---------------------------------------------------------------------------------------------- */
typedef struct
{
  /* params::flow (src/params.cpp:7-29) */
  double flow_nu, flow_u, flow_l, flow_rho_0, flow_Re;
  /* params::lattice (src/params.cpp:31-66) */
  double tau, omega, Re, nu, dx, dt, u;
  int l, T, X, Y;
  /* params::simulation (src/params.cpp:95-120); valid only when has_simulation */
  int has_simulation;
  double stop_time, snapshot_period;
  int total_steps, snapshot_steps, total_snapshots;
  char file_prefix[256];
} lbm_params;

/* parses [flow], [lattice] and, when require_simulation != 0, [simulation]; a missing key gives
 * LBM_ERR_CONFIG with the reference's message "<key> not defined in parameters file" */
int lbm_params_from_toml(const char* path, int require_simulation, lbm_params* out);

typedef struct
{
  double rho_0, alpha, A, nu, mu, beta, cs2, ics2, rlx; /* src/colour.cpp:11-39 */
  double phi[9], eta[9];                                /* :49-64 */
} lbm_colour;
int lbm_colour_from_toml(const char* path, const char* table, lbm_colour* out);

typedef struct
{
  int rows, columns, time_steps, nr_snapshots, period_snapshots; /* mrtcg_rayleigh_taylor.cpp:103-117 */
  int has_general;
  double sigma, gravity_magnitude;                              /* :360-361 */
  char name[256];                                               /* :362 */
} lbm_two_phase_params;
int lbm_two_phase_from_toml(const char* path, int require_general, lbm_two_phase_params* out);

/* boundary file `[name] x=[..] y=[..]` (src/ibm.cpp:78-102).  Call with xs=ys=NULL to get the count. */
int lbm_markers_from_toml(const char* path, const char* name, double* xs, double* ys, int* n);

/* ------------------------------------------------------------------------------------------------
 * Snapshot output in the reference's on-disk format (SURVEY §8(f) rank 1)
 * ---------------------------------------------------------------------------------------------- */
/* replaces `torch::save(tensor, path)` of a contiguous CPU fp64 tensor (test/horizontal_poiseuille_test.cpp:157-160,
 * test/cylinder_test.cpp:168-172, test/mrtcg_rayleigh_taylor.cpp:481-485): writes the same TorchScript archive
 * (ZIP of stored entries, one parameter "0"), readable by torch.jit.load / torch.load / torch::load.
 * shape[ndim] row-major; ZIP64 when the storage exceeds 4 GiB.  Host-only, needs no CUDA device.           */
int lbm_save_pt(const char* path, const double* data, const long long* shape, int ndim);

#ifdef __cplusplus
}
#endif
#endif
