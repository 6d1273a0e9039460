/* mseetc_b200 -- C ABI of the B200-native batched multiple-shooting OCP solver.
 *
 * Drop-in boundary for the NLP build-and-solve of dkouzoup/ms-eetc:
 *   - mseetc_create       replaces what casadiSolver.__init__ hands to ca.nlpsol (mseetc/ocp.py:288-290):
 *                         the problem *structure* (flags fixed by train/options, ocp.py:101-102,184,216).
 *   - mseetc_solve_batch  replaces self.solver(lbx=,ubx=,lbg=,ubg=,x0=) (mseetc/ocp.py:359) for a whole batch
 *                         of instances; it returns, per instance, what ocp.py:360-362 reads back:
 *                         zOpt, f, return_status, iter_count.
 *   - mseetc_eval_interval  kernel-level parity hook for TrainIntegrator.solve (mseetc/train.py:347-364).
 *
 * Plain pointers and sizes only.  Every `*_dev` pointer is a CUDA device pointer owned by the caller
 * (torch tensors in the Python shim); the library never allocates or frees per call.  Calls on one handle
 * must be serialised by the caller.  Work is enqueued on `stream`; mseetc_solve_batch synchronises the
 * stream before returning (it polls a device-side completion counter).
 *
 * Return value: 0 ok, <0 usage error, >0 cudaError_t.  mseetc_last_error() gives the message.
 * Per-instance solver outcomes are *never* an error return: see status_out.
 */
#ifndef MSEETC_B200_H
#define MSEETC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MSEETC_B200_VERSION 100
#define MSEETC_KERNEL_CLASSES 8

/* per-instance parameter planes: params_dev[field * n_instances + instance], specific units (ocp.py:96-116) */
enum mseetc_param {
    MSEETC_P_SR0 = 0,   /* r0/(mass*rho)                      train.py:181 */
    MSEETC_P_SR1,       /* r1/(mass*rho)                      train.py:182 */
    MSEETC_P_SR2,       /* r2/(mass*rho)                      train.py:183 */
    MSEETC_P_FEL_LO,    /* forceMin/M or 0 (no regen brake)   ocp.py:107,175 */
    MSEETC_P_FEL_UP,    /* forceMax/M                         ocp.py:106,176 */
    MSEETC_P_FPB_LO,    /* forceMinPn/M                       ocp.py:108,175 */
    MSEETC_P_POW_LO,    /* -|lowerBound|                      ocp.py:187,192 */
    MSEETC_P_POW_UP,    /* |upperBound|                       ocp.py:186,191 */
    MSEETC_P_ACC_LO,    /* accMin                             ocp.py:114 */
    MSEETC_P_ACC_UP,    /* accMax                             ocp.py:113 */
    MSEETC_P_LOSS_TR,   /* (1-etaT)/etaT  (static map)        train.py:204 */
    MSEETC_P_LOSS_RG,   /* (1-etaR)                           train.py:204 */
    MSEETC_P_BMIN,      /* minimumVelocity^2                  ocp.py:271 */
    MSEETC_P_OBJ_SCALE, /* scalingFactorObjective             ocp.py:276-284 */
    MSEETC_P_T_END,     /* terminalTime                       ocp.py:353 */
    MSEETC_P_T_START,   /* initialTime                        ocp.py:347 */
    MSEETC_P_B_START,   /* clipped v0^2                       ocp.py:343,348 */
    MSEETC_P_B_END,     /* clipped vN^2                       ocp.py:344,349 */
    MSEETC_P_MASS,      /* mass*rho                           ocp.py:97 */
    MSEETC_P_DYN_AUX,   /* auxiliaries [W]        (loss_kind 2, efficiency.py:101) */
    MSEETC_P_DYN_ETAG,  /* etaGear                (efficiency.py:101) */
    MSEETC_P_DYN_FMAX,  /* forceMax of the measured drive [N]  (efficiency.py:64) */
    MSEETC_P_DYN_PMAX,  /* powerMax of the measured drive [W]  (efficiency.py:65) */
    MSEETC_P_DYN_SCALE, /* scale of the measured loss table (1 = reference map) */
    MSEETC_PARAM_COUNT
};

/* per-instance status_out codes; the Python shim maps them to IPOPT's return_status strings (ocp.py:362) */
enum mseetc_status {
    MSEETC_SOLVE_SUCCEEDED = 0,
    MSEETC_MAXIMUM_ITERATIONS_EXCEEDED = 1,
    MSEETC_RESTORATION_FAILED = 2,
    MSEETC_ERROR_IN_STEP_COMPUTATION = 3,
    MSEETC_INFEASIBLE_PROBLEM_DETECTED = 4,
    MSEETC_INVALID_NUMBER_DETECTED = 5,
    MSEETC_SOLVED_TO_ACCEPTABLE_LEVEL = 6   /* IPOPT's acceptable_tol 1e-6 for 15 iterations: success in CasADi's stats() */
};

typedef struct mseetc_problem {
    int32_t n_intervals_max;    /* largest numIntervals in any batch solved with this handle (ocp.py:88) */
    int32_t with_pn_brake;      /* train.forceMinPn != 0                 ocp.py:102 */
    int32_t with_power_rows;    /* powerMax or powerMin present          ocp.py:184 */
    int32_t energy_optimal;     /* opts.energyOptimal                    ocp.py:146,216 */
    int32_t loss_kind;          /* 0 none / 1 static efficiencies (train.py:204) / 2 dynamic map (efficiency.py) */
    int32_t num_steps;          /* OptionsRK.numSteps                    train.py:463 */
    int32_t num_approx_steps;   /* OptionsRK.numApproxSteps              train.py:465 */
    int32_t max_iterations;     /* opts.maxIterations -> ipopt max_iter  ocp.py:290 */
    double tol;                 /* IPOPT tol (default 1e-8) */
    double mu_init;             /* IPOPT mu_init (default 0.1) */
    int32_t initial_guess;      /* 0: the reference's starting point (ocp.py:325-339); 1: dynamically consistent
                                 * speed-envelope profile built on the device (same optimum, about half the iterations) */
    int32_t stall_iterations;   /* > 0: stop an instance (status MAXIMUM_ITERATIONS_EXCEEDED) after that many trial evaluations without
                                 * a 10 % gain of its best KKT error -- keeps one cycling instance from holding a whole batch;
                                 * 0 = run to max_iterations like the reference */
} mseetc_problem;

typedef struct mseetc_solver* mseetc_handle;

int mseetc_version(void);
const char* mseetc_last_error(void);

int mseetc_create(const mseetc_problem* problem, mseetc_handle* out);
int mseetc_destroy(mseetc_handle h);

/* Dynamic loss map (loss_kind 2): the cubic tensor-product B-spline that efficiency.createSpline builds
 * (efficiency.py:23-51): knots over load [%] (n_load+4) and speed [m/s] (n_speed+4), coefficients [n_load][n_speed].
 * Host pointers; the library keeps a device copy until mseetc_destroy. */
int mseetc_set_loss_map(mseetc_handle h, int32_t n_load, int32_t n_speed, const double* knots_load,
                        const double* knots_speed, const double* coef);

/* Kernel-level parity hook for the loss rows: G(Fel, b_k, b_{k+1}) = PL{tr,rgb}(Fel, vMid)/vMid with gradient and
 * Hessian.  in_dev planes [3*n]: Fel, b_k, b_{k+1}; params_dev planes [MSEETC_PARAM_COUNT*n];
 * out_dev planes [20*n]: traction row (value, dFel, db0, db1, FF, F0, F1, 00, 01, 11) then the braking row. */
int mseetc_eval_loss_rows(mseetc_handle h, int32_t n, const double* in_dev, const double* params_dev, double* out_dev,
                          void* cuda_stream);

/* bytes of device workspace needed to solve `n_instances` at once */
size_t mseetc_workspace_bytes(mseetc_handle h, int32_t n_instances);

/* Solve a batch.
 *   params_dev        [MSEETC_PARAM_COUNT * n_instances] planes (see enum mseetc_param)
 *   n_intervals_dev   [n_instances]  numIntervals of each instance (<= n_intervals_max)
 *   track_of_inst_dev [n_instances]  index of the track table an instance runs on
 *   track_offset_dev  [n_tracks+1]   interval offsets (CSR) into ds/c0; node arrays use offset+track index
 *   ds_dev, c0_dev    [sum N_j]      interval length; g*grad/rho + curvRes/rho   (ocp.py:125, train.py:252-254)
 *   bmax_dev          [sum (N_j+1)]  min(limit_i, vmax, limit_{i-1})^2 at the nodes (ocp.py:266-272)
 *   tmin_dev          [n_instances] or NULL: known minimum trip duration of each instance (from a time-optimal
 *                     solve of the same problem).  Instances with T_END - T_START below it are infeasible
 *                     (terminalTime is an upper bound on t_N, ocp.py:260-261) and are reported as
 *                     MSEETC_INFEASIBLE_PROBLEM_DETECTED without iterating.  An entry of 0 means "not known yet": the
 *                     array is re-read once per iteration, so the minimum times may be produced concurrently (another
 *                     stream / thread) while this call is running.  Passing the array (even all zeros) also switches on
 *                     the envelope screening: an instance whose available time is more than 1 % below a speed-envelope
 *                     lower bound on the trip duration gets the same status before its first iteration (iterations 0).
 *                     The caller is expected to confirm such flags with the exact minimum time once it is known (the
 *                     Python layer does, and re-solves with tmin_dev = NULL should one not be confirmed).  A negative entry
 *                     exempts an instance from both screenings (the caller asserts that it is feasible).
 * outputs (device, caller-owned; each may be NULL except status_out):
 *   z_out_dev    [n_instances * (n_intervals_max*(3+nu)+2)]  reference variable order (ocp.py:166-181,248-249)
 *   lam_g_out_dev[n_instances * n_intervals_max*rows]        multipliers of g in reference row order
 *   obj_out_dev, kkt_out_dev [n_instances]; iters_out_dev, status_out_dev [n_instances]
 */
int mseetc_solve_batch(mseetc_handle h, int32_t n_instances,
                       const double* params_dev, const int32_t* n_intervals_dev,
                       const int32_t* track_of_inst_dev, const int32_t* track_offset_dev,
                       const double* ds_dev, const double* c0_dev, const double* bmax_dev, const double* tmin_dev,
                       double* z_out_dev, double* lam_g_out_dev, double* obj_out_dev, double* kkt_out_dev,
                       int32_t* iters_out_dev, int32_t* status_out_dev,
                       void* workspace_dev, size_t workspace_bytes, void* cuda_stream);

/* Host-side preprocessing of MANY tracks in one call (no device work): the grid of computeDiscretizationPoints
 * (mseetc/track.py:91-107 with mergeDataFrames :377-383) -- per track the union of numpy.linspace(0, length, N + 1 - (M - 1)) and the
 * M merged section starts, which must have exactly N + 1 points (error[t] = 1 otherwise, the reference raises ValueError), and
 * the forward-filled speed limit / gradient / curvature at those points.  Step functions in CSR form (offsets [n_tracks+1],
 * ascending positions, first position 0); node outputs indexed like bmax_dev: out_off[t] + t + k with out_off = cumsum(n_int).
 * All pointers are HOST pointers. */
int mseetc_discretize_tracks(int32_t n_tracks, const double* length, const int32_t* n_int,
                             const int32_t* lim_off, const double* lim_pos, const double* lim_val,
                             const int32_t* grd_off, const double* grd_pos, const double* grd_val,
                             const int32_t* crv_off, const double* crv_pos, const double* crv_val,
                             const int32_t* out_off, double* pos_nodes, double* limit_nodes, double* grad_nodes, double* curv_nodes,
                             int32_t* error);

/* Trajectory tables of a batch: what utils.postProcessDataFrame (mseetc/utils.py:223-336, called at ocp.py:407) adds to every
 * returned solution, for all instances at once, incl. the time-domain re-simulation columns (utils.py:164-194; RK4 with
 * Richardson extrapolation in place of CVODES).  table_out_dev: [n_instances][n_intervals_max+1][mseetc_table_columns()],
 * row-major, columns in the reference's order with the index column 'Time [s]' first; rows beyond an instance's last node and
 * all rows of failed instances (status_dev, may be NULL) are NaN.  node_tables_dev: four planes (position [m], speed limit
 * [m/s], gradient [permil], curvature [1/m]) of [sum (N_j+1)] doubles, node_plane_stride doubles apart, indexed like bmax_dev;
 * mass_dev [n_instances]: train.mass without the rotating-mass factor (utils.py:294).  The other arguments are those of
 * mseetc_solve_batch.  Synchronises the stream. */
int mseetc_table_columns(void);
int mseetc_postprocess_batch(mseetc_handle h, int32_t n_instances, const double* z_dev, const double* params_dev,
                             const int32_t* n_intervals_dev, const int32_t* track_of_inst_dev, const int32_t* track_offset_dev,
                             const double* ds_dev, const double* c0_dev, const double* node_tables_dev, size_t node_plane_stride,
                             const double* mass_dev, const int32_t* status_dev, double* table_out_dev, void* cuda_stream);

/* Sweep variant (replaces MUMPS behind mseetc/ocp.py:359): 1 = sequential Riccati sweeps, one thread per instance (default of
 * a new handle); 8, 16 or 32 = parallel-in-time sweeps with that many chunk lanes per instance (chunk elements from reference
 * Riccati recursions, sequential chain of the chunk-end value functions, exact in-chunk recursions, a-posteriori consistency
 * check with sequential fallback per instance; see csrc/pit.cuh); 0 = chosen per call from n_intervals_max and the batch size
 * (what the Python layer sets): 16 lanes from 96 intervals, 32 from 1024, sequential sweeps beyond 4096 instances per call. */
int mseetc_set_sweep_lanes(mseetc_handle h, int lanes);
int mseetc_last_sweep_lanes(mseetc_handle h);          /* lanes the last mseetc_solve_batch on h ran with */
/* compaction passes launched in the last solve (running instances moved into the slots of finished ones so that they fill whole
 * warps; csrc/compact.cuh; results do not depend on it; mseetc_set_compaction(h, 0) switches it off) */
int mseetc_last_compactions(mseetc_handle h);
int mseetc_last_compaction_moves(mseetc_handle h);     /* instances moved by those passes */
int mseetc_set_compaction(mseetc_handle h, int on);
/* instances x iterations of the last solve that fell back to the sequential sweeps; reasons (out3): reference recursion of a
 * chunk not positive definite / chain step numerically singular / chain and recursion disagreed */
long long mseetc_last_sweep_fallbacks(mseetc_handle h);
int mseetc_last_sweep_fallback_reasons(mseetc_handle h, int32_t* out3);

/* number of solver ticks (lock-step rounds) and kernel launches of the last mseetc_solve_batch on h */
int mseetc_last_ticks(mseetc_handle h);
int mseetc_last_launches(mseetc_handle h);

/* Per-kernel accounting of the last mseetc_solve_batch (measurement support for bench.py):
 *   kernel classes: 0 cell_trial, 1 inst_decide, 2 cell_eval, 3 inst_step (Riccati sweeps), 4 setup/init/extract,
 *                   5 cell_step, 6 inst_alpha, 7 inst_kkt (MSEETC_KERNEL_CLASSES = 8 entries in every array)
 *   ms_out[8]        summed device time per class, from cudaEvent pairs recorded on the launch stream
 *                    (only when profiling was switched on with mseetc_set_profiling; else zeros)
 *   launches_out[8]  launches per class
 *   cells_out[8]     (interval, instance) cells actually processed per class (idle/finished instances excluded)
 *   mseetc_bytes_per_cell(h, cls): algorithmic HBM bytes one processed cell costs in that class (see DESIGN.md) */
int mseetc_set_profiling(mseetc_handle h, int on);
int mseetc_last_profile(mseetc_handle h, double* ms_out, int32_t* launches_out, int64_t* cells_out);
double mseetc_bytes_per_cell(mseetc_handle h, int kernel_class);
/* Diagnostic: the launches of the last solve on `h` as (class, start_ms, end_ms) triples in out[3*max_entries], times taken
 * from the same event pairs relative to the first launch of the last solve on `origin` (another handle of the same device,
 * e.g. the first stream of a pool, or `h` itself).  Returns the number of entries written; needs profiling switched on. */
int mseetc_last_timeline(mseetc_handle h, mseetc_handle origin, double* out, int32_t max_entries);

/* Measurement aid (SURVEY 8d: the FP64 roofline denominator is not in MEASURED_PEAKS.json): sustained DFMA throughput of the
 * current device in GFLOP/s (FMA = 2), from a kernel of independent FMA chains timed with CUDA events on the given stream. */
int mseetc_measure_fp64_peak(double* gflops_out, void* cuda_stream);

/* One shooting interval for n points (train.py:347-364): tau = t1 - t0 and b1, with first and second
 * sensitivities w.r.t. (b0, F).  in_dev planes [7*n]: b0, F, ds, c0, sr0, sr1, sr2; out_dev planes [12*n]:
 * tau, dtau/db, dtau/dF, d2tau/dbb, d2tau/dbF, d2tau/dFF, then the same six for b1. */
int mseetc_eval_interval(int32_t n, int32_t num_steps, int32_t num_approx_steps,
                         const double* in_dev, double* out_dev, void* cuda_stream);

/* Shooting integrator of the handle (TrainIntegrator, mseetc/train.py:282-322).  The default is the explicit branch
 * (ca.simpleRK, train.py:294-301).  stages >= 1 selects collocation steps (ca.simpleIRK, train.py:303-310): `A` [stages*stages,
 * row-major] and `w` [stages] are HOST arrays with the Runge-Kutta coefficients of the collocation method on the chosen points
 * (A_ij = int_0^{c_i} l_j, w_j = int_0^1 l_j), `max_newton` the iteration limit of the stage solve (OptionsIRK.maxIter,
 * train.py:494).  The number of steps and the time approximation stay the num_steps and num_approx_steps of the problem structure.
 * The 'CVODES' branch (train.py:312-322) is served by the same entry point with a high-order Gauss tableau, see DESIGN.md.
 * stages = 0 returns to the explicit steps. */
int mseetc_set_integrator(mseetc_handle h, int32_t stages, const double* A, const double* w, int32_t max_newton);

/* integrateLosses = True of the reference (OptionsCasadiSolver, mseetc/ocp.py:28,118-120,231-241): the two epigraph rows of every
 * interval bound s_k from below by the traction / regenerative-braking loss ENERGY of the interval, integrated in the time domain
 * (TrainIntegrator.calcLosses, train.py:367-413), and the objective becomes sum(ds_k Fel_k + s_k).  Energy-optimal mode with the
 * constant-efficiency or the spline loss model, any integrator of mseetc_set_integrator.  lam_out holds the multipliers of the reference's
 * formulation (rows on t_{k+1} - t_k).  See DESIGN.md section 2 for the formulation solved on the device. */
int mseetc_set_integrate_losses(mseetc_handle h, int on);

/* mseetc_eval_interval with collocation steps (same planes in and out; A, w: host arrays as above). */
int mseetc_eval_interval_irk(int32_t n, int32_t num_steps, int32_t num_approx_steps, int32_t stages, const double* A,
                             const double* w, int32_t max_newton, const double* in_dev, double* out_dev, void* cuda_stream);

#ifdef __cplusplus
}
#endif
#endif
