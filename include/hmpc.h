/* hmpc.h -- C ABI of libhmpc_b200.so: batched hopper MPC hot path on NVIDIA B200 (sm_100a).
 *
 * The reference (bbokser/hopper-mpc-inertial) is pure Python and has no FFI; this header is the
 * boundary a maintainer would bind with ctypes (see INTEGRATION.md).  Each entry point names the
 * reference interface it replaces (file:line into the reference's src/).
 *
 * Conventions
 *  - Every function returns 0 on success or a negative hmpc_error; hmpc_last_error() gives text.
 *    Nothing throws or aborts across the boundary.
 *  - All array arguments are DEVICE pointers (e.g. torch tensor.data_ptr()) unless the name ends
 *    in _host.  Layout is structure-of-arrays with the hopper (batch) index FASTEST:
 *    an array documented as [R][C][B] stores element (r,c,b) at ((r*C)+c)*B + b.
 *  - Element type is double (FP64) for every floating-point array at the boundary, whatever the
 *    internal solver precision (hmpc_config.precision).
 *  - A handle is bound to one device and one stream (a multi-tick hmpc_rollout also uses a second stream the
 *    handle owns, joined back into the handle's stream before the call's work ends); calls are stream-asynchronous; a handle is
 *    not thread-safe.  The library allocates only its own opaque workspace.
 *  - There is no CPU fallback: creating a handle without a usable CUDA device fails.
 */
#ifndef HMPC_H
#define HMPC_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMPC_ABI_VERSION 2
#define HMPC_INF 1e30          /* "no bound" marker (same convention as OSQP's OSQP_INFTY) */
#define HMPC_NX 12             /* Euler MPC state  [p, rpy, pdot_w, omega_w]  (mpc_cvx_euler_3f.py:21) */
#define HMPC_NU 6              /* control [f(3), tau_body(3)]                 (mpc_cvx_euler_3f.py:22) */
#define HMPC_NXSIM 13          /* simulator state [p, q(wxyz), v_b, omega_b]  (robotrunner.py:50)      */
#define HMPC_MAX_N 64          /* contact schedule is shipped as one 64-bit mask per hopper            */

typedef enum hmpc_error {
    HMPC_OK = 0,
    HMPC_ERR_BAD_ARG = -1,
    HMPC_ERR_CUDA = -2,
    HMPC_ERR_UNSUPPORTED = -3,
    HMPC_ERR_NO_DEVICE = -4,
    HMPC_ERR_ALLOC = -5
} hmpc_error;

/* per-hopper solve status (device int32 arrays) */
typedef enum hmpc_status {
    HMPC_SOLVED = 0,           /* exact optimum: passed the KKT test of the original QP                */
    HMPC_MAX_ITER = 1,
    HMPC_PRIMAL_INFEASIBLE = 2,/* some height row x[k,2] >= z_min cannot be met by any admissible
                                  input (includes the u-independent rows k = 0, 1, SURVEY App. D2);
                                  the reference raises "QP FAILED" (mpc_cvx_euler_3f.py:158-159)       */
    HMPC_NON_FINITE = 3,
    HMPC_SOLVED_INEXACT = 4    /* residual test met (ADMM eps_abs/eps_rel, or interior-point tolerance)
                                  but the point did not pass the exact KKT verification                */
} hmpc_status;

/* which branch of the solver produced the result (hmpc_solve_stats) */
enum { HMPC_PATH_NONE = 0, HMPC_PATH_WARM = 1, HMPC_PATH_IPM_POLISH = 2, HMPC_PATH_IPM = 3, HMPC_PATH_ADMM = 4 };

enum { HMPC_DYN_2F = 2, HMPC_DYN_3F = 3 };                 /* mpc_cvx_euler_2f / mpc_cvx_euler_3f      */
enum { HMPC_FP64 = 0, HMPC_FP32 = 1 };
enum { HMPC_UREF_ALIASED = 0, HMPC_UREF_PER_STAGE = 1 };   /* SURVEY App. D1                           */
enum { HMPC_SOLVER_EXACT = 0, HMPC_SOLVER_ADMM = 1 };
enum { HMPC_MODE_EARLY_EXIT = 0, HMPC_MODE_FIXED_ITER = 1 };
enum { HMPC_INFEASIBLE_HOLD = 0, HMPC_INFEASIBLE_RESPAWN = 1 };
enum { HMPC_HOT_AUTO = 0, HMPC_HOT_CTA = 1 };

/* Constants of Mpc.__init__ (mpc_cvx_euler_3f.py:12-39), Runner.__init__ (robotrunner.py:37-79) and
 * the literals inside build_qp (mpc_cvx_euler_3f.py:113-146), plus solver settings. */
typedef struct hmpc_config {
    int32_t abi_version;   /* = HMPC_ABI_VERSION */
    int32_t device;        /* CUDA device ordinal */
    int32_t batch;         /* B: hoppers handled by this handle */
    int32_t dyn;           /* HMPC_DYN_2F | HMPC_DYN_3F */
    int32_t N;             /* horizon (robotrunner.py:46 uses 60; benches 10/20/40) */
    int32_t mpc_factor;    /* sim steps per MPC tick (robotrunner.py:48) = 20 */
    int32_t precision;     /* HMPC_FP64 | HMPC_FP32.  FP32 = mixed precision: the factorisations and substitutions
                              run in FP32 (factor stored as float), QP data / iterates / residuals stay FP64 and the
                              refinement loops recover the accuracy; same acceptance test on the original QP */
    int32_t uref_mode;     /* HMPC_UREF_ALIASED (reference-faithful) | HMPC_UREF_PER_STAGE */
    int32_t solver;        /* HMPC_SOLVER_EXACT: warm-started verified active-set refinement with an
                              interior-point fallback -> the exact optimum (default);
                              HMPC_SOLVER_ADMM: OSQP-style ADMM (cvxpy's settings below) */
    int32_t mode;          /* ADMM: HMPC_MODE_EARLY_EXIT | HMPC_MODE_FIXED_ITER */
    int32_t max_iter;      /* ADMM iteration cap (cvxpy passes 10000) / exact iteration count in FIXED_ITER */
    int32_t check_interval;/* ADMM residual-test / rho-adaptation cadence after the first check (OSQP: 25) */
    int32_t first_check;   /* ADMM iterations before the first residual test */
    int32_t polish;        /* ADMM: 1 = verified active-set polish after termination (OSQP polish=True) */
    int32_t adaptive_rho;  /* ADMM: OSQP residual-balancing rho update at check time */
    int32_t warm_start;    /* 1: start from the time-shifted previous solution / active set */
    int32_t polish_retries;/* active-set refinements per polish attempt */
    int32_t ipm_max_iter;  /* interior-point iteration cap */
    int32_t on_infeasible; /* rollout: HMPC_INFEASIBLE_HOLD (apply U = 0) | HMPC_INFEASIBLE_RESPAWN
                              (reset the hopper onto its reference at the next tick and re-initialise) */
    int32_t sqp_sweeps;    /* relinearisation sweeps per (non-first) tick: 1 = the reference's single linearisation
                              about the time-shifted previous solution (mpc_cvx_euler_3f.py:59-68); k > 1 relinearises
                              about the sweep's own solution and solves again (the SQP the reference's docstring
                              gestures at, mpc_cvx_euler_3f.py:41-46).  0 is treated as 1 */
    int32_t hot_path;      /* HMPC_HOT_AUTO: warm ticks run the warp-per-hopper kernel, hoppers it cannot finish (and
                              first calls, ADMM, FP32, sqp_sweeps > 1, long horizons) the CTA-per-hopper kernel;
                              HMPC_HOT_CTA: CTA-per-hopper kernel only (round-1 path, kept for A/B measurements) */
    double mpc_dt;         /* robotrunner.py:47  0.02  */
    double sim_dt;         /* run.py:24          1e-3  */
    double m, g, mu;       /* robotrunner.py:37,42,68 */
    double J[9];           /* row-major inertia (robotrunner.py:38-40) */
    double Jinv[9];        /* robotrunner.py:41 */
    double rh[3];          /* robotrunner.py:42 */
    double tau_max[3];     /* mpc_cvx_euler_3f.py:123-128  7.78, 7.78, 4 */
    double fz_max;         /* mpc_cvx_euler_3f.py:20,146   206 */
    double z_min;          /* mpc_cvx_euler_3f.py:129      0.1 */
    double kf;             /* terminal state-cost factor, mpc_cvx_euler_3f.py:113 (100); input factor kuf=0 */
    double eps_abs, eps_rel;   /* ADMM residual test (cvxpy: 1e-5 each) */
    double rho0, sigma, alpha; /* OSQP defaults 0.1, 1e-6, 1.6 */
    double kkt_eps;            /* relative regularisation of the row block of the quasi-definite polish system
                                  (removed by refinement); FP32 mode uses at least 1e-3 */
    double polish_tol;         /* relative KKT acceptance tolerance of the verification, default 1e-9 */
    double ipm_tol;            /* interior-point residual / complementarity tolerance, default 1e-6 (the verified
                                  polish that follows lands on the exact optimum) */
} hmpc_config;

typedef struct hmpc_handle hmpc_handle;

/* Fill a config with the reference's constants and OSQP/cvxpy solver defaults. */
int hmpc_default_config(hmpc_config* cfg);

/* Replaces Mpc.__init__ (mpc_cvx_euler_3f.py:12-39 / mpc_cvx_euler_2f.py:12-38) for a batch. */
int hmpc_create(const hmpc_config* cfg, hmpc_handle** out);
int hmpc_destroy(hmpc_handle* h);
int hmpc_set_stream(hmpc_handle* h, void* cuda_stream);
int hmpc_synchronize(hmpc_handle* h);

/* Per-hopper gains: the public Mpc.Q / Mpc.R attributes (mpc_cvx_euler_3f.py:34-37), diagonals only.
 * Qdiag [12][B], Rdiag [6][B].  Defaults are the reference's values for every hopper. */
int hmpc_set_gains(hmpc_handle* h, const double* Qdiag, const double* Rdiag);

/* Per-hopper body: the arguments of Mpc(t, N, m, g, mu, Jinv, rh) (mpc_cvx_euler_3f.py:12-39) and the simulator's own
 * m, J, Jinv, rh (robotrunner.py:37-42,76), one set per hopper instead of the config's scalars -- for domain randomisation,
 * and for model mismatch (the MPC plans with one body while the simulator integrates another).
 *   HMPC_BODY_MODEL  what the MPC plans with: m, Jinv, rh, mu     (linearisation, condensing, friction cones, u_ref)
 *   HMPC_BODY_PLANT  what hmpc_rk4 / the rollouts integrate: m, J, Jinv, rh   (dynamics_ct, HMPC_GATE_DETECT's leg vector)
 *   HMPC_BODY_BOTH   both from the same arrays
 * m [B], J [9][B] (row-major 3x3 per hopper), Jinv [9][B], rh [3][B], mu [B], device arrays, copied (stream-ordered)
 * into storage the handle owns.  A NULL array: that quantity takes the config's scalar for every hopper; each call
 * replaces the whole target.  All NULL: the target goes back to the config's scalars.  J with HMPC_BODY_MODEL and mu
 * with HMPC_BODY_PLANT have no effect and are rejected.  Nothing derives Jinv from J here: pass both.
 * The values are checked (m > 0, mu >= 0, all finite; the call synchronises the stream): on failure HMPC_ERR_BAD_ARG,
 * hmpc_last_error() names the first offending hopper and the handle is unchanged.  Takes effect from the next solve or
 * rollout; warm starts stay valid (every accepted point is verified against the QP built with the new body).
 * g, tau_max, fz_max, z_min, kf, dt and N stay per handle. */
enum { HMPC_BODY_MODEL = 1, HMPC_BODY_PLANT = 2, HMPC_BODY_BOTH = 3 };
int hmpc_set_body_params(hmpc_handle* h, int which, const double* m, const double* J, const double* Jinv,
                         const double* rh, const double* mu);

/* convert (robotrunner.py:19-28): X [13][B] -> x [12][B]. */
int hmpc_convert(hmpc_handle* h, const double* X, double* x);

/* rk4_normalized repeated nsteps times with a zero-order-hold control (robotrunner.py:154-164,
 * dynamics_ct :126-152).  X [13][B] in/out, U [6][B], pf [3][B]; X_steps [nsteps][13][B] optional
 * (may be NULL): the state after every step (X_traj rows, robotrunner.py:113). */
int hmpc_rk4(hmpc_handle* h, double* X, const double* U, const double* pf, int nsteps, double* X_steps);

/* gen_dt_dynamics (mpc_cvx_euler_3f.py:71-94 / 2f:70-94): x_guess [N+1][12][B], pf [N][3][B] ->
 * Ad [N][12][12][B], Bd [N][12][6][B].  Exposed for parity tests; the solver never materialises these. */
int hmpc_linearize(hmpc_handle* h, const double* x_guess, const double* pf, double* Ad, double* Bd);

/* Condensed QP data for parity tests: given the linearisation point, emit
 * H [n][n][B], g [n][B], lo/hi [m][B] in the slot layout  rows = [6N box | 4N friction | N height]
 * (n = 6N, m = 11N; see DESIGN.md).  Built from build_qp (mpc_cvx_euler_3f.py:96-153).
 * Height row k >= 2 is normalised by its largest coefficient dt^2 (k-1)/m, so its bound reads
 * lo = (z_min - c_z[k]) m / (dt^2 (k-1)).  infeasible [B] (int32, may be NULL): 1 when some height row
 * cannot be met by any admissible input. */
int hmpc_condense(hmpc_handle* h, const double* x_in, const double* x_guess, const double* x_ref,
                  const double* pf, const uint64_t* Cbits, double* H, double* g, double* lo, double* hi,
                  int32_t* infeasible);

/* Mpc.mpcontrol (mpc_cvx_euler_3f.py:41-69): linearise, build and solve the QP for every hopper.
 *   x_in  [12][B]        convert()ed current state
 *   x_ref [N][12][B]     reference window (path_plan_grab, robotrunner.py:228-230)
 *   pf    [N][3][B]      footstep window
 *   Cbits [B]            contact schedule, bit k = C[k] != 0 (gait_map, robotrunner.py:172-180)
 *   init                 1: first call (two solves, x_guess[1:] = x_ref);  0: time-shift the handle's
 *                        previous solution (mpc_cvx_euler_3f.py:50-62)
 *   U     [N][6][B]      out: u.value
 *   Xsol  [N+1][12][B]   out: x.value (also kept inside the handle for the next time shift)
 *   status, iters [B]    out: hmpc_status and solver iterations (ADMM or interior-point; 0 when the
 *                        warm-started active-set refinement succeeded) (int32)
 */
int hmpc_solve(hmpc_handle* h, const double* x_in, const double* x_ref, const double* pf,
               const uint64_t* Cbits, int init, double* U, double* Xsol, int32_t* status,
               int32_t* iters);

/* Closed loop of Runner.run (robotrunner.py:96-113) for n_ticks MPC ticks, state resident in HBM:
 * per tick: convert -> mpcontrol -> mpc_factor x rk4 with ZOH U[0].
 *   X        [13][B]               in/out simulator state
 *   xref_tab [T+N][12][B]          MPC-rate reference rows (row j = x_ref[j*mpc_factor])
 *   pf_tab   [T+N][3][B]           MPC-rate footstep rows
 *   C_tab    [T][B]                contact masks per tick
 *   pf_switch[T][B] (uint8)        sim step within the tick at which pf_ref changes from row t to t+1
 *                                  (mpc_factor = never)  -- reproduces pf_ref[k] at 1 kHz
 *   tick0                          index of the first tick in the tables; init = 1 on the run's first tick
 *   X_log    [n_ticks+1][13][B]    optional (may be NULL): state at every tick boundary
 *   U_log    [n_ticks][6][B]       optional: applied control per tick (f_hist, robotrunner.py:111)
 *   status   [B], iters [B]        first non-zero status / accumulated iterations over the ticks
 * A hopper whose QP is infeasible gets U = 0 for that tick (HOLD) or is put back onto its reference
 * (RESPAWN, hmpc_config.on_infeasible); hmpc_solve_stats reports how often that happened.
 */
int hmpc_rollout(hmpc_handle* h, double* X, const double* xref_tab, const double* pf_tab,
                 const uint64_t* C_tab, const uint8_t* pf_switch, int tick0, int n_ticks, int init,
                 double* X_log, double* U_log, int32_t* status, int32_t* iters);

/* ---- the caller side of the path on the device: path_plan_init / path_plan_grab / gait_map ------------------------
 * (robotrunner.py:166-230).  Every hopper follows the reference's planner between its own start x0 and goal xf,
 * optionally with the --curve profile, and enters the run at its own tick.  What depends only on the common clock is
 * passed as small HOST tables (computed with the reference's summation order, planner.global_tables in the Python
 * package); the per-hopper rows are generated on the device, bit-identical to the numpy planner. */
typedef struct hmpc_plan_config {
    int32_t N_run;        /* simulator steps of the run (robotrunner.py:183) */
    int32_t n_sim;        /* entries of sin_tab / pf_idx (N_run + N * mpc_factor) */
    int32_t max_tick;     /* entries of cmask / sw_glob */
    int32_t reserved;
    double t_p;           /* gait period (robotrunner.py:43); the height wave has amplitude t_p / 4 (:207) */
    double curve_psi1, curve_psi2;   /* yaw knots of --curve: -0.4 sin(45 deg), -sin(45 deg) (robotrunner.py:197) */
} hmpc_plan_config;

/* x0, xf [12][B] (device), curve, tick_offset [B] int32 (device); HOST tables: sin_tab [n_sim] = sin(2 pi / t_p (k dt)
 * + 3 pi / 2) (robotrunner.py:210), pf_idx [n_sim] = simulator index whose reference xy is the footstep in force at
 * step k (:214-224), cmask [max_tick] = contact mask of global tick j (gait_map on the run clock, :97-102,172-180),
 * sw_glob [max_tick] = simulator step inside tick j at which the footstep changes (mpc_factor = never).  The
 * per-hopper arrays are referenced, not copied: they must stay alive while the plan is in use. */
int hmpc_plan_set(hmpc_handle* h, const hmpc_plan_config* pc, const double* x0, const double* xf, const int32_t* curve,
                  const int32_t* tick_offset, const double* sin_tab_host, const int32_t* pf_idx_host,
                  const uint64_t* cmask_host, const uint8_t* sw_glob_host);

/* path_plan_grab for ticks [tick0, tick0 + n_ticks): the tables hmpc_rollout takes, written by the device:
 * xref_tab [n_ticks+N][12][B], pf_tab [n_ticks+N+1][3][B], C_tab [n_ticks][B], pf_switch [n_ticks][B] (uint8). */
int hmpc_plan_tables(hmpc_handle* h, int tick0, int n_ticks, double* xref_tab, double* pf_tab, uint64_t* C_tab,
                     uint8_t* pf_switch);

/* hmpc_rollout without tables: every tick generates its own reference window (N+1 rows), footsteps, contact mask
 * and switch step on the device just before the solve (about 1.4 KB written per hopper-tick instead of table rows
 * read).  Same results as hmpc_rollout on the tables of hmpc_plan_tables, bit for bit. */
int hmpc_rollout_planned(hmpc_handle* h, double* X, int tick0, int n_ticks, int init, double* X_log, double* U_log,
                         int32_t* status, int32_t* iters);

/* ---- contact gate of the applied control (SURVEY 8 row f4, second half) --------------------------------------------
 * The reference computes the scheduled contact s = gait_scheduler(t, t0) at every simulator step and logs it
 * (robotrunner.py:99,112) but applies the control ungated: `f_hist[k, :] = U[0, :]  # * s` (robotrunner.py:111).
 *   HMPC_GATE_OFF       (default) the reference as shipped: U[0] is held over the whole tick
 *   HMPC_GATE_SCHEDULE  the commented-out factor switched on: simulator step i of a tick applies U[0] * s_i with s_i
 *                       the scheduled contact at that step's time (1 kHz gait clock, robotrunner.py:97-99,166-171)
 *   HMPC_GATE_DETECT    contact detected from the state instead of the clock: s_i = 1 while the leg vector of
 *                       dynamics_ct, r = rh + R(q)'(pf - p) (robotrunner.py:143), is no longer than leg_max, else 0
 * gate_tab  [T][B] uint32 (device, referenced not copied; used by hmpc_rollout): bit i of entry (tick, b) = s at
 *           simulator step i of that tick, indexed like C_tab;
 * gate_glob [max_tick] uint32 (HOST, copied; used by hmpc_rollout_planned): the same masks on the common clock,
 *           hopper b reads entry tick_offset[b] + tick (planner.global_tables: gate_glob).
 * Either may be NULL when the corresponding rollout flavour is not used (that flavour then returns HMPC_ERR_BAD_ARG).
 * HMPC_GATE_SCHEDULE requires mpc_factor <= 32.  The MPC itself is unchanged: it keeps planning on the schedule. */
enum { HMPC_GATE_OFF = 0, HMPC_GATE_SCHEDULE = 1, HMPC_GATE_DETECT = 2 };
int hmpc_set_contact_gate(hmpc_handle* h, int mode, const uint32_t* gate_tab, const uint32_t* gate_glob_host, int max_tick,
                          double leg_max);

/* Per-hopper statistics of the most recent hmpc_solve (or accumulated over the most recent
 * hmpc_rollout): nfac [B] = matrix factorisations, path [B] = HMPC_PATH_* of the last solve,
 * n_infeasible [B] = ticks flagged HMPC_PRIMAL_INFEASIBLE (device int32 arrays), flops [B] = algorithmic
 * floating-point operations of the solver kernel (device double array; FMA = 2).  Each may be NULL. */
int hmpc_solve_stats(hmpc_handle* h, int32_t* nfac, int32_t* path, int32_t* n_infeasible, double* flops);

/* Per-kernel device timing of hmpc_rollout: when enabled, CUDA events are recorded on the handle's stream
 * around every launch.  hmpc_kernel_times synchronises the stream and returns the summed durations (ms)
 * of the solver kernel and of the simulator kernel over the most recent hmpc_rollout and its tick count.
 * In a multi-tick rollout on the warp-per-hopper path the deferred hoppers' solver and simulator kernels run on a
 * second stream of the handle, beside the next tick's work (DESIGN.md section 5); their own event intervals are added
 * to the tick's solver and simulator times.  These intervals overlap: they no longer add up to the tick's duration. */
int hmpc_set_timing(hmpc_handle* h, int enable);
int hmpc_kernel_times(hmpc_handle* h, double* mpc_ms, double* sim_ms, int* n_ticks);
/* The same per tick: mpc_ms / sim_ms are HOST arrays of at least cap doubles (either may be NULL); *n_ticks receives
 * the tick count of the most recent timed hmpc_rollout.  Used for the p50 QP-solve latency of BASELINE.json's metric:
 * one entry is the solver kernels' time for the WHOLE batch of that tick. */
int hmpc_tick_times(hmpc_handle* h, double* mpc_ms_host, double* sim_ms_host, int cap, int* n_ticks);

/* The warp-per-hopper hot path of this handle (hmpc_config.hot_path): resident warps (= hoppers in flight) per SM,
 * the cap on the order of the compact KKT system it keeps in shared memory, registers per thread, and how many
 * hopper-ticks of the most recent hmpc_solve / hmpc_rollout it handed to the CTA-per-hopper kernel (host value;
 * synchronises the stream).  warps_per_sm = 0 when the handle's configuration does not use the warp kernel.
 * Each pointer may be NULL. */
int hmpc_hot_path_info(hmpc_handle* h, int* warps_per_sm, int* kcap, int* regs, int64_t* n_deferred);

/* Counters since handle creation: kernels launched by this library (for bench gpu_launches). */
int hmpc_launch_count(hmpc_handle* h, int64_t* n_launches);

/* FP64 FMA peak microbenchmark (roofline denominator, SURVEY 8d): returns TFLOP/s measured with a
 * dependent-chain-free DFMA kernel on the handle's device. */
int hmpc_measure_fp64_peak(hmpc_handle* h, double* tflops);

const char* hmpc_last_error(void);
int hmpc_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* HMPC_H */
