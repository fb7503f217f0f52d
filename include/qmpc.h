/*
 * include/qmpc.h — C-ABI of libqmpc.so: batched RTI-MPC + recursive-GP control step on B200 (sm_100a).
 *
 * Drop-in boundary for the per-control-step loop of smidmatej/mpc_quad_ros
 * (reference src/execute_trajectory.py:196-277).  In the reference that loop reaches native code through
 * acados' ctypes wrapper (`AcadosOcpSolver.set / solve / get / get_cost`, call sites
 * src/quad_opt.py:286,290,311,315,328-333,342-350,404) for ONE vehicle with host double* buffers, and
 * through numpy for the RGP (src/gp/RGP.py:303-330).  Here one handle owns B vehicles on one GPU.
 *
 * Conventions
 *   - every array argument is a DEVICE pointer to fp64 unless marked `host`;
 *   - arrays are vehicle-major and C-contiguous (`[B][N][13]` means vehicle b's record is contiguous):
 *     one warp owns one vehicle, so per-vehicle-contiguous records are the coalesced layout;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every call returns 0 on success, <0 on error (qmpc_last_error() gives the text);
 *     nothing synchronises the host except the functions documented as such;
 *   - a handle is bound to one device and is not thread-safe; independent handles are.
 * State ordering x = [p(3), q(w,x,y,z), v(3, world), r(3, body)], inputs u in [lbu,ubu]^4.
 */
#ifndef QMPC_H
#define QMPC_H

#ifdef __cplusplus
extern "C" {
#endif

#define QMPC_NX 13
#define QMPC_NU 4
#define QMPC_NY 17

#define QMPC_OK 0
#define QMPC_ERR_ARG (-1)
#define QMPC_ERR_CUDA (-2)
#define QMPC_ERR_ALLOC (-3)

/* per-vehicle solver status written by qmpc_solve */
#define QMPC_STATUS_OK 0        /* exact active set verified, or IPM converged below ipm_mu_tol */
#define QMPC_STATUS_MAXITER 1   /* ipm_max_iter reached (reference: qp_solver_iter_max = 50)  */
#define QMPC_STATUS_NAN 2       /* NaN/Inf met                                                */

typedef struct qmpc_solver *qmpc_handle_t;
typedef struct qrgp_model *qrgp_handle_t;

/* OCP definition: replaces AcadosOcp setup in quad_optimizer.__init__ (src/quad_opt.py:36-160) and
 * src/_acados_ocp.json.  quad[] follows Quadrotor3D (src/quad.py:41-94). */
typedef struct {
    int batch;           /* B vehicles handled by this handle                                        */
    int n_nodes;         /* N (acados dims.N, quad_opt.py:98)                                        */
    int n_basis;         /* M RGP basis points per axis; 0 = nominal model (gpe=None)                */
    int precision;       /* 64: fp64 solver (default) ; 32: fp32 Riccati/IPM (RGP stays fp64)        */
    int device;          /* CUDA device ordinal                                                       */
    int ipm_max_iter;    /* <=0 -> 50                                                                  */
    int refine_max_rounds; /* active-set refinement rounds after the IPM: 0 -> 20 (fp32: 10), <0 -> off     */
    int warm_start_rounds; /* refinement rounds tried first from the previous solve's active set: 0 -> 6,
                              <0 -> off (cold IPM every step, in every kernel of the solver)                  */
    double ipm_mu_tol;   /* <=0 -> 1e-13 (fp64) / 1e-6 (fp32): complementarity target of the pure IPM     */
    double ipm_mu_switch; /* <=0 -> 1e-4: the IPM hands over to the active-set refinement below this          */
    double t_horizon;    /* tf ; dt = t_horizon / n_nodes (quad_opt.py:43)                            */
    double quad[20];     /* mass, max_thrust, J[3], x_f[4], y_f[4], z_l_tau[4], g[3]                  */
    double w_diag[17];   /* LINEAR_LS stage weights diag(W) (quad_opt.py:122-129); scaled by dt inside */
    double we_diag[13];  /* terminal weights diag(W_e) (quad_opt.py:130)                               */
    double lbu, ubu;     /* input box (quad_opt.py:142-143)                                            */
    double gp_theta[9];  /* per axis (L, sigma_f, sigma_n) (RGP.py:106)                                */
    const double *gp_X;  /* host [3][M] basis points, may be NULL when n_basis == 0.  Any layout is accepted; an axis
                            whose points are equispaced (linspace, what GPEnsemble.fromrange builds: GPE.py:127-150) is
                            detected here and its M kernel values are evaluated from 3 exps by recurrence            */
    /* ---- solver policy, per handle (every field: 0 -> library default).  The reference has no counterpart: acados
     * cold-starts HPIPM every step and ignores its status (quad_opt.py:333, _acados_ocp.json qp_solver_warm_start 0). */
    int solver_variant;    /* 0 -> auto: Riccati screening launch + dense condensed launch for fp64 with N <= 21, the
                              Riccati kernel alone otherwise; 1 -> Riccati kernel alone; 2 -> screening + dense */
    int reset_on_fail;     /* 0 -> on: a vehicle whose last solve failed (status != 0) restarts its SQP iterate on the new
                              reference and, from the second failure in a row, gets a bounded attempt per step;
                              <0 -> off: keep whatever the solver left, as the reference does */
    int screen_rounds;     /* active-set rounds the screening launch tries before it hands an OCP over: 0 -> 3 */
    int dense_warm_rounds; /* rounds the dense kernel continues from the handed-over guess before its IPM: 0 -> 8, <0 -> none */
    int bail_round;        /* round (0-based) from which a non-contracting change count ends a warm attempt: 0 -> 2 */
    int bail_changed;      /* a warm round that still moves more inputs than this ends the attempt: 0 -> never */
    int final_rollout;     /* >0 -> always re-roll the horizon at the end of a solve (A/B knob): 0 -> reuse the last sweep */
    int dense_grid;        /* persistent CTAs of the dense launch: 0 -> min(resident CTAs, max(32, B/3)) */
    int screen_rounds_busy; /* round limit of the screening launch in a BUSY step: 0 -> 8, <0 -> same as screen_rounds.  A step
                              is busy when the previous step left more than screen_busy_pct % of the vehicles unsettled
                              after screen_rounds rounds (start-up transients, aggressive references): the dense launch
                              would need several waves then, and a Riccati round is cheaper than the dense condensing */
    int screen_busy_pct;   /* 0 -> 25 */
} qmpc_config;

const char *qmpc_last_error(void);
int qmpc_version(void);

/* ---- solver life cycle: AcadosOcpSolver(ocp) / capsule free (quad_opt.py:156) */
int qmpc_create(const qmpc_config *cfg, qmpc_handle_t *out);
int qmpc_destroy(qmpc_handle_t h);

/* ---- inputs.  Each copies (device->device, async on `stream`) into handle-owned storage. */
/* solver.set(j,"yref",.) j<N and solver.set(N,"yref",.) (quad_opt.py:311,315): yref [B][N][17], yref_e [B][13] */
int qmpc_set_yref(qmpc_handle_t h, const double *yref, const double *yref_e, void *stream);
/* quad_optimizer.set_reference_trajectory (quad_opt.py:295-317): x_ref [B][N][13], u_ref [B][N][4] or NULL
 * (NULL -> 0.16 hover, quad_opt.py:304); terminal reference = x_ref[:, N-1] (quad_opt.py:314). */
int qmpc_set_reference(qmpc_handle_t h, const double *x_ref, const double *u_ref, void *stream);
/* solver.set(0,'lbx',x); solver.set(0,'ubx',x) (quad_opt.py:328-329): x0 [B][13] */
int qmpc_set_x0(qmpc_handle_t h, const double *x0, void *stream);
/* solver.set(ii,'p',rgp_params) (quad_opt.py:402-404): mu [B][3][M] RGP means; the handle forms
 * alpha = K_x^-1 mu per axis (the constant product of RGP.py:252-254) with Kx_inv [3][M][M] device. */
int qmpc_set_params(qmpc_handle_t h, const double *mu, const double *Kx_inv, void *stream);
/* the same, when alpha [B][3][M] is already available (qrgp_get_alpha) */
int qmpc_set_alpha(qmpc_handle_t h, const double *alpha, void *stream);
/* the same without a copy: later solves read alpha from the caller's device buffer (stride = doubles between vehicles:
 * 3*M, or 0 when one shared model serves every vehicle); NULL returns to the handle's own storage.  Host-side switch,
 * takes effect for solves queued afterwards (used by the shared-swarm mode to double-buffer the model). */
int qmpc_bind_alpha(qmpc_handle_t h, const double *alpha, int stride);
/* persistent SQP iterate (acados keeps it inside the capsule; zero after create, SURVEY A.3):
 * x [B][N+1][13], u [B][N][4] */
int qmpc_set_iterate(qmpc_handle_t h, const double *x, const double *u, void *stream);
int qmpc_get_iterate(qmpc_handle_t h, double *x, double *u, void *stream);

/* ---- solver.solve() (quad_opt.py:333): one SQP-RTI iteration for all B vehicles.
 * Kernels: qmpc_linearize (RK4 + forward sensitivities incl. GP Jacobian) -> qmpc_ipm (Riccati Mehrotra IPM,
 * full step, cost).  Asynchronous. */
int qmpc_solve(qmpc_handle_t h, void *stream);

/* ---- outputs: solver.get(i,"u"), get(i,"x"), get_cost() (quad_opt.py:342-350) */
int qmpc_get_u0(qmpc_handle_t h, double *u0 /*[B][4]*/, void *stream);
int qmpc_get_x(qmpc_handle_t h, double *x /*[B][N+1][13]*/, void *stream);
int qmpc_get_u(qmpc_handle_t h, double *u /*[B][N][4]*/, void *stream);
int qmpc_get_cost(qmpc_handle_t h, double *cost /*[B]*/, void *stream);
int qmpc_get_status(qmpc_handle_t h, int *status /*[B]*/, int *iters /*[B]*/, void *stream);
/* consecutive failed solves per vehicle (0 = last solve fine); all zero when reset_on_fail is off */
int qmpc_get_fail_streak(qmpc_handle_t h, int *streak /*[B]*/, void *stream);
/* active-set refinement rounds of the last solve (warm-start rounds + rounds after the IPM), [B] */
int qmpc_get_refine_rounds(qmpc_handle_t h, int *rounds /*[B]*/, void *stream);
/* OCPs the screening launch of the last solve handed to the dense launch (host value; synchronises `stream`) */
int qmpc_get_hard_count(qmpc_handle_t h, int *count_host, void *stream);
/* active sets remembered for the warm start, device u8 [B][4N]: 0 free, 1 at lbu, 2 at ubu, 255 unknown.  They steer
 * which path a solve takes (warm rounds / IPM), never its answer; exposed for replaying a solve elsewhere. */
int qmpc_get_active_set(qmpc_handle_t h, unsigned char *act, void *stream);
int qmpc_set_active_set(qmpc_handle_t h, const unsigned char *act, void *stream);
/* forget the active sets remembered for the warm start (the next solve starts from the cold IPM) */
int qmpc_reset_warm_start(qmpc_handle_t h, void *stream);
/* sum over vehicles of IPM iterations of the last solve (host value; synchronises `stream`) */
int qmpc_iters_total(qmpc_handle_t h, long long *total, void *stream);

/* acados eval_param_sens(field "ex") + get(k, "sens_x" / "sens_u") for every vehicle and every x0 component at once:
 * derivatives of the last solve's x[k], u[k] w.r.t. x0 at the active set the handle holds (after a solve: that solve's),
 * k < n_stages (1..N).  sens_x [B][n_stages+1][13][13] (may be NULL), sens_u [B][n_stages][4][13], row-major,
 * column = x0 component.  NaN for vehicles whose active set is unknown.  Reads the stage tiles of the last solve:
 * valid until the next qmpc_solve / qmpc_step on the handle.  Asynchronous.
 * The linearisation of an RTI step does not read x0, so x0 -> (x, u) is the box-QP's solution map (piecewise affine):
 * these are its exact derivatives on the active set, i.e. the closed loop of the LQR with the inputs flagged 1/2 pinned
 * (their rows are 0), taken w.r.t. the 13 raw components of x0.  sens_u[:, 0] is the feedback gain K0 = du0/dx0.
 * A solve that ended on the IPM alone (status 0) leaves the IPM's classification of the bounds; the sensitivities refer
 * to that set.  Returns QMPC_ERR_ARG before the handle's first solve and for fp32 handles. */
int qmpc_eval_sens_x0(qmpc_handle_t h, int n_stages, double *sens_x, double *sens_u, void *stream);

/* Reverse mode of the same solution map, now w.r.t. x0 AND the reference, for every vehicle at once: for cotangents
 * x_bar [B][N+1][13] and u_bar [B][N][4] of the last solve's x, u (either may be NULL = zero), the gradients of
 * <x_bar, x> + <u_bar, u> w.r.t. x0 -> x0_bar [B][13], yref -> yref_bar [B][N][17] and yref_e -> yref_e_bar [B][13]
 * (any of the three may be NULL; outputs are overwritten, not accumulated).  The linearisation reads the reference only
 * in the linear cost term, so on the active set of the last solve these are exact: with (xh, uh) the minimiser of the
 * pinned LQR with linear costs -x_bar, -u_bar from xh_0 = 0,  yref_bar[k] = (Qd xh_k, Rd uh_k) (Qd = dt w_diag[0:13],
 * Rd = dt w_diag[13:17]; its stage-0 state part and pinned input entries are exactly 0), yref_e_bar = we_diag xh_N and
 * x0_bar = sum_k sens_x[k]^T x_bar[k] + sens_u[k]^T u_bar[k].  Cotangents on pinned inputs have no effect.  NaN for
 * vehicles whose active set is unknown.  With reset_on_fail on, a vehicle whose PREVIOUS solve failed was linearised
 * at a point built from the reference: its result is the derivative at that fixed linearisation.  One pinned
 * factorisation and two vector sweeps; reads the stage tiles and active set: valid until the next solve.  Asynchronous.
 * Returns QMPC_ERR_ARG, launching nothing, before the handle's first solve, for fp32 handles, with both cotangents NULL
 * and with all three outputs NULL. */
int qmpc_eval_adjoint(qmpc_handle_t h, const double *x_bar, const double *u_bar, double *x0_bar, double *yref_bar,
                      double *yref_e_bar, void *stream);

/* host counter that changes whenever the data qmpc_eval_sens_x0 / qmpc_eval_adjoint read may change: every solve
 * (qmpc_solve, qmpc_step, qmpc_step_dt, qmpc_closed_loop_step), qmpc_set_active_set and qmpc_reset_warm_start.  The
 * sensitivity calls leave it alone.  A deferred backward compares it to refuse stale tiles. */
int qmpc_get_sens_epoch(qmpc_handle_t h, long long *epoch);

/* ---- stateless helpers of the loop (any B) */
/* quad_optimizer.discrete_dynamics (quad_opt.py:353-377): nominal RK4 step, optional body-frame velocity.
 * x [B][13], u [B][4] -> x_next [B][13] */
int qmpc_predict_nominal(const double *quad /*host[20]*/, int B, const double *x, const double *u, double dt,
                         int body_frame, double *x_next, void *stream);
/* utils.compute_a_drag (utils.py:934-950): x_now, x_pred [B][13] -> v_body, a_drag [B][3] */
int qmpc_compute_a_drag(int B, const double *x_now, const double *x_pred, double dt,
                        double *v_body, double *a_drag, void *stream);
/* utils.get_reference_chunk (utils.py:897-931): traj [B][K][13], idx (same for all) -> chunk [B][N][13] */
int qmpc_reference_chunk(int B, int K, const double *traj, int idx, int N, int skip, double *chunk, void *stream);
/* the same chunk without a stored trajectory: the reference generators evaluated on the device at the sample times
 * (row * dt, rows chosen like get_reference_chunk, rows past K-1 repeat row K-1).  params device [B][QMPC_REFGEN_NPAR]:
 * kind 0 sum of three sinusoids per axis (amp[3][3], f[3][3] Hz, phase[3][3], scale, p0[3], z0), kind 1 lemniscate
 * (phase, yaw, w, a, z0, p0x, p0y, ramp time), kind 2 accelerating circle of TrajectoryGenerator.py:41-74 (radius, v_max,
 * n samples, start[3], csv-rounding flag).  q = (1,0,0,0), r = 0 as TrajectoryGenerator.load_trajectory leaves them. */
#define QMPC_REFGEN_NPAR 32
int qmpc_reference_generate(int kind, int B, const double *params, int K, int idx, int N, int skip, double dt,
                            double *chunk, void *stream);
/* Quadrotor3D.update repeated over one control period (quad.py:234-277, execute_trajectory.py:232-243):
 * plant[4] = aero_drag, rotor_drag xyz (host); x [B][13] in/out; u [B][4]; n_sub sub-steps of sim_dt */
int qmpc_plant_period(const double *quad /*host[20]*/, const double *plant /*host[4]*/, int B, double *x,
                      const double *u, double sim_dt, int n_sub, void *stream);

/* ---- RGP ensemble: GPEnsemble of 3 RGPs per vehicle (src/gp/GPE.py:34, src/gp/RGP.py:104) */
/* RGP.__init__ x3 (RGP.py:106-157; GPE.fromrange GPE.py:127-150): X host [3][M], theta host [3][3],
 * Kx, Kx_inv host [3][M][M] (computed by the caller exactly as the reference does, np.linalg.inv).
 * State: mu = 0, C = K_x for every vehicle. */
int qrgp_create(int batch, int n_basis, const double *X, const double *theta, const double *Kx,
                const double *Kx_inv, int device, qrgp_handle_t *out);
int qrgp_destroy(qrgp_handle_t g);
/* GPEnsemble.regress with one sample per axis (GPE.py:244-268 -> RGP.py:303-330): xt, yt [B][3] */
int qrgp_regress(qrgp_handle_t g, const double *xt, const double *yt, void *stream);
/* fused utils.compute_a_drag + regress (execute_trajectory.py:255-256): x_now, x_pred_prev [B][13] */
int qrgp_regress_from_states(qrgp_handle_t g, const double *x_now, const double *x_pred_prev, double dt,
                             double *v_body /*[B][3] or NULL*/, double *a_drag /*[B][3] or NULL*/, void *stream);
/* state access: mu [B][3][M], C [B][3][M][M]; alpha = K_x^-1 mu [B][3][M] */
int qrgp_get_mu(qrgp_handle_t g, double *mu, void *stream);
int qrgp_get_C(qrgp_handle_t g, double *C, void *stream);
int qrgp_set_state(qrgp_handle_t g, const double *mu, const double *C, void *stream);
int qrgp_get_alpha(qrgp_handle_t g, double *alpha, void *stream);
const double *qrgp_Kx_inv_device(qrgp_handle_t g);
const double *qrgp_mu_device(qrgp_handle_t g);
/* RGP.predict (RGP.py:195-229): xs [B][3][m] -> mean [B][3][m], var [B][3][m] (var may be NULL) */
int qrgp_predict(qrgp_handle_t g, int m, const double *xs, double *mean, double *var, void *stream);
/* RGP.predict_using_y numpy branch (RGP.py:264-300): xs [B][3][m], y [B][3][M] -> mean [B][3][m] */
int qrgp_predict_using_y(qrgp_handle_t g, int m, const double *xs, const double *y, double *mean, void *stream);
/* RGP.predict(cov=True, return_Jt=True) (RGP.py:195-229): gains Jt [B][3][m][M] and full posterior covariance [B][3][m][m] */
int qrgp_predict_cov(qrgp_handle_t g, int m, const double *xs, double *Jt, double *cov, void *stream);

/* ---- shared-swarm mode (BASELINE config 3): ONE RGP for all vehicles on all GPUs.
 * Each rank accumulates the information-form contributions of its vehicles,
 *   Lambda_d = sum_v j_v^T j_v / r_v,  eta_d = sum_v j_v^T y_v / r_v,  r_v = b_v + sigma_n^2,
 * into info [3][M*M+M] (device), the host all-reduces `info` (NCCL sum), then every rank applies the
 * identical posterior update C <- (C^-1 + Lambda)^-1, mu <- C (C_old^-1 mu_old + eta). */
int qrgp_shared_accumulate(qrgp_handle_t g, int B, const double *xt, const double *yt, double *info, void *stream);
int qrgp_shared_apply(qrgp_handle_t g, const double *info, void *stream);

/* ---- fused control step for the closed loop (execute_trajectory.py:196-277), all on `stream`:
 *   set_reference(x_ref chunk) ; set_x0(x_now) ; solve (alpha of the previous step) ; u0 ;
 *   x_pred = nominal RK4(x_now,u0,dt) ; if g: residual(x_now, x_pred_prev) -> regress -> alpha for the next solve.
 * x_pred_prev [B][13] is updated in place with x_pred (pass x_now for the very first step). */
int qmpc_step(qmpc_handle_t h, qrgp_handle_t g, const double *x_now, const double *x_ref,
              double *x_pred_prev, int first_step, double *u0_out, void *stream);

/* the ROS node's variant of the same step (src/mpc_controller_node.py:298,315): the nominal prediction and the drag
 * residual use the odometry period instead of the OCP's dt (odometry_dt <= 0 -> the OCP's dt = qmpc_step); the caller cuts
 * x_ref with skip = control_freq_factor (qmpc_reference_chunk / qmpc_reference_generate, node :278) */
int qmpc_step_dt(qmpc_handle_t h, qrgp_handle_t g, const double *x_now, const double *x_ref,
                 double *x_pred_prev, int first_step, double *u0_out, double odometry_dt, void *stream);

/* the whole closed-loop step in one call: qmpc_reference_chunk(traj, idx) -> qmpc_step -> qmpc_plant_period(x, u0).
 * traj [B][K][13]; x [B][13] plant state in/out; chunk [B][N][13] and u0 [B][4] caller-owned scratch/outputs. */
int qmpc_closed_loop_step(qmpc_handle_t h, qrgp_handle_t g, const double *traj, int K, int idx, double *x,
                          double *x_pred_prev, double *chunk, double *u0, const double *plant /*host[4]*/, double sim_dt,
                          int n_sub, void *stream);

/* when `g` is a shared model (created with batch == 1) qmpc_step leaves the residual samples of its B vehicles
 * (v_body, a_drag: [B][3] each) in handle-owned buffers for qrgp_shared_accumulate */
const double *qmpc_residual_x_device(qmpc_handle_t h);
const double *qmpc_residual_y_device(qmpc_handle_t h);

/* ---- RGP* hyper-parameter learning: RGP.learn (src/gp/RGP.py:332-482, sigma points :485-505) for n_models independent
 * 1-D models on one basis grid X[n_basis] (host) with initial hyper-parameters theta[3] = (L, sigma_f, sigma_n) (host).
 * State per model as RGP.__init__ leaves it (:141-157): mu_g = 0, C_g = K_x, mu_eta = theta, C_eta = I, C_g_eta = 0,
 * K_x_inv = inv(K(X,X) + sigma_n^2 I).  The reference never calls learn from its control loop; neither does qmpc_step. */
typedef struct qrgpl_model *qrgpl_handle_t;
int qrgpl_create(int n_models, int n_basis, const double *X, const double *theta, int device, qrgpl_handle_t *out);
int qrgpl_destroy(qrgpl_handle_t g);
/* one learn() call per model: xt, yt device [n_models]; optional outputs mu_z [n][M+3], C_z [n][M+3][M+3] (device, may be NULL) */
int qrgpl_learn(qrgpl_handle_t g, const double *xt, const double *yt, double *mu_z, double *C_z, void *stream);
/* device copies of the state; any pointer may be NULL: mu_g [n][M], C_g [n][M][M], mu_eta [n][3], C_eta [n][3][3], Kx_inv [n][M][M] */
int qrgpl_get_state(qrgpl_handle_t g, double *mu_g, double *C_g, double *mu_eta, double *C_eta, double *Kx_inv, void *stream);
int qrgpl_set_state(qrgpl_handle_t g, const double *mu_g, const double *C_g, const double *mu_eta, const double *C_eta,
                    const double *C_g_eta /*[n][M][3]*/, const double *Kx_inv, void *stream);
/* per-model status of the last learn (device int [n]): 0 ok, 1 singular K_x */
int qrgpl_get_status(qrgpl_handle_t g, int *status, void *stream);

/* ---- measurement hooks (bench.py roofline leg; not part of the control path) */
/* cudaEvents around the two kernels of qmpc_solve: enable, run solves, read summed device times (synchronises). */
int qmpc_timing_enable(qmpc_handle_t h, int on);
int qmpc_timing_read(qmpc_handle_t h, double *ms_linearize, double *ms_ipm, int *count);
/* part of ms_ipm spent in the dense kernel (the solver is a screening launch followed by a dense launch); call before
 * qmpc_timing_enable(h, 0) */
int qmpc_timing_read_dense(qmpc_handle_t h, double *ms_dense);
/* per-vehicle timeline of the solver kernel: when enabled, every OCP records %globaltimer (ns) when its warp starts
 * and when it has written its result; read copies [batch][2] (start, end) of the LAST solve to the host (synchronises). */
int qmpc_timeline_enable(qmpc_handle_t h, int on);
int qmpc_timeline_read(qmpc_handle_t h, long long *start_end_host);
/* register-resident FMA microbenchmark: measured non-tensor FMA peak (TFLOP/s); precision 64 or 32; synchronises */
int qmpc_fma_peak(int precision, double *tflops, void *stream);

/* number of kernels launched by this library since load (for bench.py's gpu_launches) */
long long qmpc_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* QMPC_H */
