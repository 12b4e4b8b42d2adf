/*
 * eicos_b200.h - C ABI of the B200-native batched SOCP interior-point engine.
 *
 * Drop-in boundary for ONE path of EmbersArc/EiCOS: EiCOS::Solver construction ->
 * solve() -> updateData() -> solution(), plus a batched overload for many instances that
 * share a sparsity pattern.  Plain pointers and sizes only; no C++/torch types.
 * "reference" below = /root/reference (EmbersArc/EiCOS).
 *
 * Problem form (reference README.md:20-50):   min c'x  s.t.  A x = b,  G x + s = h,  s in K,
 * K = R+^l x Q^{q_1} x ... x Q^{q_ncones}; G, A in CSC (0-based int indices, rows ascending in a
 * column), rows of G ordered LP rows first, then cone 1, cone 2, ...
 *
 * Exit codes are the reference's `exitcode` values (include/eicos.hpp:8-21):
 *   0 optimal, 1 primal infeasible, 2 dual infeasible, -1 maxit, -2 numerics, -3 outcone,
 *   -7 fatal, +10 = "close to" variants.
 *
 * Every function needs a CUDA device (sm_100a); there is no CPU fallback.  On failure the
 * constructors return NULL and the int functions return a negative EICOS_ERR_* code;
 * eicos_last_error() gives the message (thread-local).
 */
#ifndef EICOS_B200_H
#define EICOS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define EICOS_ERR_INVALID (-100) /* bad argument */
#define EICOS_ERR_DEVICE (-101)  /* CUDA failure (no device, out of memory, launch error) */

/* Mirrors EiCOS::Information (reference include/eicos.hpp:49-73); std::optional fields are
 * (has_*, value) pairs. */
typedef struct eicos_info
{
    double pcost, dcost, pres, dres;
    double pinfres, dinfres, gap, relgap;
    double sigma, mu, step, step_aff, kapovert;
    int pinf, dinf;
    int has_pinfres, has_dinfres, has_relgap;
    int iter, iter_max, nitref1, nitref2, nitref3;
} eicos_info;

/* Solver settings (the run-time fields of EiCOS::Settings, reference include/eicos.hpp:23-47).  Every handle
 * holds one set, which applies to every instance of every later solve on it.  A setter checks every field and
 * rejects bad input with EICOS_ERR_INVALID, naming the field in eicos_last_error() and keeping the handle's
 * settings as they were.  Valid values: every double finite; the tolerances, linsysacc and irerrfact > 0;
 * 0 < gamma <= 1; 0 < stepmin <= stepmax <= 1; 0 <= sigmamin <= sigmamax <= 1; safeguard >= 1;
 * 0 <= nitref <= 32; 1 <= iter_max <= 1000.
 * deltastat (7e-8) and equil_iters (3) stay fixed: they enter the KKT values, the programs' constants and the
 * equilibration when the handle is set up.  delta, eps and maxit are not read by the reference either. */
typedef struct eicos_settings
{
    double feastol, abstol, reltol;                   /* exit tolerances (1e-8 each) */
    double feastol_inacc, abstol_inacc, reltol_inacc; /* reduced tolerances for "close to" exits (1e-4, 5e-5, 5e-5) */
    double linsysacc, irerrfact;                      /* iterative refinement: accuracy 1e-14, error factor 6 */
    double gamma, stepmin, stepmax;                   /* step scaling 0.99, line-search clamp [1e-6, 0.999] */
    double sigmamin, sigmamax;                        /* centering parameter clamp [1e-4, 1] */
    double safeguard;                                 /* restore the best iterate when pres grows by this factor (500) */
    int nitref, iter_max;                             /* refinement rounds per KKT solve (9), iteration limit (100) */
} eicos_settings;

/* the reference's default values */
void eicos_default_settings(eicos_settings *out);

/* ------------------------------------------------------------------ single instance ---- */
typedef struct eicos_solver eicos_solver;

/* replaces EiCOS::Solver::Solver(int n,int m,int p,int l,int ncones,int* q, double* Gpr,...)
 * (reference include/eicos.hpp:151-154, src/eicos.cpp:91-120) and ECOS_setup of the test shim
 * (test/ecos.h:11-17).  `l` is ignored like there (l = m - sum q).  NULL (Gpr,Gjc,Gir) / (Apr,
 * Ajc,Air) triples mean "no G" / "no A".  All inputs are copied.  device = CUDA ordinal. */
eicos_solver *eicos_setup(int n, int m, int p, int l, int ncones, const int *q,
                          const double *Gpr, const int *Gjc, const int *Gir,
                          const double *Apr, const int *Ajc, const int *Air,
                          const double *c, const double *h, const double *b, int device);

/* replaces Solver::updateData(double* Gpr,double* Apr,double* c,double* h,double* b)
 * (include/eicos.hpp:155-156, src/eicos.cpp:2053-2082) / ECOS_updateData (test/ecos.h:24-29).
 * NULL = keep; as in the reference h is only read when Gpr is given and b only when Apr is. */
int eicos_update_data(eicos_solver *s, const double *Gpr, const double *Apr,
                      const double *c, const double *h, const double *b);

/* settings of every later eicos_solve (see eicos_settings; they survive eicos_update_data) */
int eicos_set_settings(eicos_solver *s, const eicos_settings *settings);
int eicos_get_settings(const eicos_solver *s, eicos_settings *out);

/* replaces Solver::updateData(const SparseMatrix& G, A, const VectorXd& c, h, b)
 * (include/eicos.hpp:144-148, src/eicos.cpp:2032-2051): all five value arrays are required. */
int eicos_update_data_full(eicos_solver *s, const double *Gpr, const double *Apr,
                           const double *c, const double *h, const double *b);

/* replaces Solver::solve (include/eicos.hpp:158, src/eicos.cpp:848-1262) / ECOS_solve. */
int eicos_solve(eicos_solver *s);

/* replaces Solver::solution() (include/eicos.hpp:160): pointer to n doubles owned by the solver,
 * valid until the next solve/update/cleanup. */
const double *eicos_solution(const eicos_solver *s);
/* y (p), z (m), s (m): private members of `w` in the reference (include/eicos.hpp:176); exposed
 * for parity checks.  Any pointer may be NULL. */
int eicos_get_duals(const eicos_solver *s, double *y, double *z, double *slack);
/* replaces Solver::getInfo() (include/eicos.hpp:163). */
int eicos_get_info(const eicos_solver *s, eicos_info *out);
/* replaces ~Solver / ECOS_cleanup (test/ecos.h:31-34). */
void eicos_cleanup(eicos_solver *s);

/* ------------------------------------------------------------------ batched ------------ */
typedef struct eicos_batch eicos_batch;

/* One sparsity pattern + the matrix VALUES shared by every instance of the batch (the MPC /
 * updateData use case: the reference would construct one Solver and call updateData + solve per
 * instance).  Symbolic analysis (KKT pattern src/eicos.cpp:1734-1988, AMD ordering + elimination
 * tree = Eigen analyzePattern at src/eicos.cpp:897) runs here, once.  c/h/b are the default
 * vectors for instances that do not override them.
 * capacity = number of instances resident at once (0 = choose from free memory); larger
 * batches are processed in chunks.  workers = warps per CTA (0 = default). */
eicos_batch *eicos_batch_setup(int n, int m, int p, int l, int ncones, const int *q,
                               const double *Gpr, const int *Gjc, const int *Gir,
                               const double *Apr, const int *Ajc, const int *Air,
                               const double *c, const double *h, const double *b,
                               int device, long long capacity, int workers);

/* The same with flags.  EICOS_BATCH_INSTANCE_MATRICES: every instance may bring its own G / A VALUES
 * (same pattern) - what the reference does with updateData(Gpr, Apr, c, h, b) + solve per instance
 * (src/eicos.cpp:2053-2082): the matrices are equilibrated per instance on the device
 * (setEquilibration, src/eicos.cpp:302-374) and the KKT programs read them per instance. */
#define EICOS_BATCH_INSTANCE_MATRICES 1
eicos_batch *eicos_batch_setup_ex(int n, int m, int p, int l, int ncones, const int *q,
                                  const double *Gpr, const int *Gjc, const int *Gir,
                                  const double *Apr, const int *Ajc, const int *Air,
                                  const double *c, const double *h, const double *b,
                                  int device, long long capacity, int workers, int flags);

/* New shared matrix values for the whole batch (both or either; NULL = keep the last raw
 * values); re-equilibrates and refreshes the KKT values like updateData (src/eicos.cpp:2076-2081). */
int eicos_batch_update_matrices(eicos_batch *bt, const double *Gpr, const double *Apr);

/* updateData + solve for `batch` instances with HOST buffers.  cs/hs/bs: instance-major stacked
 * vectors [batch x n], [batch x m], [batch x p]; NULL = every instance uses the setup vector.
 * Outputs (any may be NULL): x [batch x n], y [batch x p], z [batch x m], s [batch x m],
 * exitflag [batch], info [batch].  Host<->device copies are part of the call. */
int eicos_batch_solve(eicos_batch *bt, int batch,
                      const double *cs, const double *hs, const double *bs,
                      double *x, double *y, double *z, double *s,
                      int *exitflag, eicos_info *info);

/* eicos_batch_solve with per-instance matrix values: Gs [batch x nnzG], As [batch x nnzA], instance-major,
 * in the CSC order of the setup matrices; NULL = the setup values for every instance.  Needs a handle
 * from eicos_batch_setup_ex(..., EICOS_BATCH_INSTANCE_MATRICES). */
int eicos_batch_solve_matrices(eicos_batch *bt, int batch, const double *Gs, const double *As,
                               const double *cs, const double *hs, const double *bs,
                               double *x, double *y, double *z, double *s,
                               int *exitflag, eicos_info *info);

/* Same with DEVICE buffers (already resident in HBM; results stay on the device).
 * iters may be NULL.  Runs on the engine's own stream and returns after it has drained. */
int eicos_batch_solve_device(eicos_batch *bt, int batch,
                             const double *d_cs, const double *d_hs, const double *d_bs,
                             double *d_x, double *d_y, double *d_z, double *d_s,
                             int *d_exitflag, int *d_iters);

/* eicos_batch_solve_matrices with DEVICE buffers: d_Gs [batch x nnzG], d_As [batch x nnzA] instance-major
 * raw values in HBM (NULL = the setup values for every instance). */
int eicos_batch_solve_matrices_device(eicos_batch *bt, int batch, const double *d_Gs, const double *d_As,
                                      const double *d_cs, const double *d_hs, const double *d_bs,
                                      double *d_x, double *d_y, double *d_z, double *d_s,
                                      int *d_exitflag, int *d_iters);

typedef struct eicos_batch_stats
{
    int chunks, ipm_iterations;
    long long launches;
    unsigned long long ir_rounds;
    double ms_total, ms_factor, ms_solve, ms_other; /* device time (CUDA events) of the last solve */
    long long factor_launch_tiles, solve_launch_tiles;
    int factor_launches, solve_launches;
    int compactions; /* active-set compactions performed */
    /* SM clock cycles the tiles spent in the phases of eicos_solve_kkt, summed over tiles and launches:
     * right-hand-side norm, forward sweep, backward sweep, refinement residual, bookkeeping */
    unsigned long long kkt_phase_cycles[5];
    /* part of ms_other: eicos_residuals (computeResiduals) and the three per-iteration vector kernels
     * (eicos_iter_head / _mid / _tail), with the tiles their launches covered */
    double ms_resid, ms_vector;
    long long resid_launch_tiles, vector_launch_tiles;
    int resid_launches, vector_launches;
    unsigned long long lane_rounds; /* solve rounds the instances needed themselves (ir_rounds counts whole tiles) */
} eicos_batch_stats;

/* Per-kernel-class device timing of the LAST eicos_batch_solve* call (enable first). */
int eicos_batch_set_timing(eicos_batch *bt, int enabled);
/* Active-set compaction (on by default): when at most 3/4 of the resident instances are still
 * iterating, results of the finished ones are written out and the survivors are packed into fewer
 * tiles.  Results do not depend on it. */
int eicos_batch_set_compaction(eicos_batch *bt, int enabled);
int eicos_batch_get_stats(const eicos_batch *bt, eicos_batch_stats *out);

typedef struct eicos_batch_dims
{
    int n, m, p, l, ncones, dim_K, nnzK, nnzL, nnzV, nnzG, nnzA;
    int etree_height, max_col, tile_width, workers;
    long long ldl_fma; /* multiply-adds of one numeric factorisation */
    long long capacity;
    long long workspace_bytes, rows_per_instance;
} eicos_batch_dims;
int eicos_batch_get_dims(const eicos_batch *bt, eicos_batch_dims *out);

/* What the host-side program compiler produced for this pattern (eicos_b200/csrc/streams.cpp): the
 * factorisation, the triangular sweeps and the KKT mat-vecs run as programs whose intermediate values
 * live in shared-memory slots and whose global reads are known in advance (load lists). */
typedef struct eicos_program_stats
{
    int sw_slots, fa_slots; /* shared-memory slots used by the sweeps + mat-vec / by the factorisation */
    int fa_fast;            /* 1: record-form factor program (narrow columns), 0: general form */
    long long sw_far, sw_direct, fa_home; /* operands served by far gathers / direct global loads / home rows */
    int fw_loads, bw_loads, fa_loads, mv_loads; /* rows each program reads from HBM per run */
} eicos_program_stats;
int eicos_batch_get_program_stats(const eicos_batch *bt, eicos_program_stats *out);

/* Symbolic results for parity checks (any pointer may be NULL): pinv[dim_K] = original KKT index
 * of the k-th pivot (what Eigen's AMDOrdering returns), parent[dim_K] = elimination tree,
 * Lp[dim_K+1]/Li[nnzL] = pattern of L, Kp[dim_K+1]/Ki[nnzK] = upper KKT pattern. */
int eicos_batch_get_symbolic(const eicos_batch *bt, int *pinv, int *parent, int *Lp, int *Li, int *Kp, int *Ki);

/* Debug: initial factorisation (V = identity-like, src/eicos.cpp:855-900) and the two initial KKT
 * solves for `batch` instances; host outputs, instance-major, any may be NULL:
 * Lx [batch x nnzL], D [batch x dim_K], sol1/sol2 [batch x dim_K], nitref [batch x 2]. */
int eicos_batch_debug_init(eicos_batch *bt, int batch, const double *cs, const double *hs, const double *bs,
                           double *Lx, double *D, double *sol1, double *sol2, int *nitref);
/* ---- several GPUs of one node behind one handle (SURVEY.md 8b / 8e).  Instances are independent (no reduction
 * across instances anywhere in src/eicos.cpp:848-1262), so the batch is cut into contiguous slices, one per
 * device; every device gets its own eicos_batch (symbolic data and programs replicated, ~1 MB) and its own host
 * thread; results land in the caller's buffers by per-device copies - no collective.
 * devices: ngpu CUDA ordinals, or NULL for 0 .. ngpu-1; an ordinal may be listed several times: every mention is a
 * slice with its own stream, staging buffers and host thread, so that the copies of one slice overlap the kernels
 * of the others.  capacity: instances resident per slice (0 = default: an equal share of what fits the device). */
typedef struct eicos_multi eicos_multi;
eicos_multi *eicos_multi_setup(int n, int m, int p, int l, int ncones, const int *q,
                               const double *Gpr, const int *Gjc, const int *Gir,
                               const double *Apr, const int *Ajc, const int *Air,
                               const double *c, const double *h, const double *b,
                               int ngpu, const int *devices, long long capacity, int workers, int flags);
/* Host buffers, instance-major, as eicos_batch_solve_matrices (any input NULL = the setup data for every instance). */
int eicos_multi_solve(eicos_multi *mt, int batch, const double *Gs, const double *As,
                      const double *cs, const double *hs, const double *bs,
                      double *x, double *y, double *z, double *s, int *exitflag, eicos_info *info);
int eicos_multi_ngpu(const eicos_multi *mt);
/* slice of device k in a batch of `batch` instances: [*first, *first + *count) */
int eicos_multi_slice(const eicos_multi *mt, int batch, int k, int *first, int *count);
/* settings of every slice (see eicos_settings) */
int eicos_multi_set_settings(eicos_multi *mt, const eicos_settings *settings);
int eicos_multi_get_settings(const eicos_multi *mt, eicos_settings *out);
void eicos_multi_cleanup(eicos_multi *mt);

/* Test hook: lineSearch (reference src/eicos.cpp:1380-1469) on caller data - lambda, ds, dz instance-major in z
 * order [batch x m], scalars = tau, dtau, kap, dkap per instance [batch x 4], alpha out [batch] (host pointers). */
int eicos_batch_debug_line_search(eicos_batch *bt, int batch, const double *lambda, const double *ds, const double *dz,
                                  const double *scalars, double *alpha);

/* Test hook: cap the interior-point iterations of this handle at min(iter_max, 100) (the reference's
 * Settings::iter_max, include/eicos.hpp:45).  A capped solve ends with exit flag -1 (maxit) and the iterate
 * src/eicos.cpp:1082-1106 returns after `iter_max` iterations, which the parity tests compare with a CPU solve
 * under the same cap: a check of every kernel's result iteration by iteration.  iter_max <= 0 restores 100. */
int eicos_batch_debug_set_iter_max(eicos_batch *bt, int iter_max);

/* settings of every later solve on this handle, every chunk of it (see eicos_settings).  The test hook above
 * writes the same iter_max. */
int eicos_batch_set_settings(eicos_batch *bt, const eicos_settings *settings);
int eicos_batch_get_settings(const eicos_batch *bt, eicos_settings *out);

void *eicos_batch_stream(const eicos_batch *bt); /* cudaStream_t the engine launches on */
void eicos_batch_cleanup(eicos_batch *bt);

const char *eicos_last_error(void);
int eicos_device_count(void);

#ifdef __cplusplus
}
#endif
#endif
