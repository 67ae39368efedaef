/*
 * libm4q -- C ABI of the B200-native MPC4quantum hot path.
 *
 * The reference (andgoldschmidt/MPC4quantum) is pure Python and has no FFI; its seam is the module API of
 * mpc4quantum/{mpc,optimize,linearize,vectorize,experiment}.py.  Each entry point below names the reference
 * function (file:line) whose arithmetic it replaces.  INTEGRATION.md shows the ctypes stub a maintainer of the
 * reference would add.
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer unless its name ends in _host.  The caller owns all buffers; the
 *     library allocates nothing persistent and frees nothing it did not allocate.
 *   - complex128 is interleaved (re, im) doubles, matrices row-major -- exactly numpy / torch.complex128.
 *   - vec(rho) is row-major (reference: x0.reshape(H0.shape), experiment.py:203, :211).
 *   - All work is enqueued on `stream` (a cudaStream_t passed as void*); no host synchronisation inside.
 *   - Return value: 0 on success, negative on argument / CUDA error (text via m4q_last_error()).
 *   - Per-member solver status uses the reference's exit codes (mpc.py:131, :195, :202, :291):
 *       0 normal, 1 exit condition met, 2 QP solver could not certify its solution, 3 non-finite objective.
 */
#ifndef M4Q_H
#define M4Q_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define M4Q_VERSION 100

/* observable maps between plant state and model state (experiment.py:29-37, 225-235, 248-306) */
#define M4Q_LIFT_IDENTITY 0
#define M4Q_LIFT_COUPLED  1   /* QCoupledExperiment: stacked partial traces / Kronecker product */
#define M4Q_LIFT_TRUNC32  2   /* QExperiment32: qubit block of a qutrit, trace-normalised        */
#define M4Q_LIFT_PROCESS  3   /* QSynthesis: plant state = propagator U, model state = vec(U (x) U^*) */

/* controller model (m4q_mpc_problem.model_mode) */
#define M4Q_MODEL_TAYLOR 0    /* reference: order-k Taylor blocks [A, N_1..N_p] (vectorize.py:8-49)            */
#define M4Q_MODEL_EXACT  1    /* extension: x+ = expm((L_0 + sum u_i L_i) dt) x, A_blocks = the m + 1 generators */

/* QP solver settings (replaces the cvxpy->OSQP call at optimize.py:59) */
typedef struct {
    double rho;          /* ADMM penalty on u = z                        (default 0.1)  */
    double alpha;        /* over-relaxation                              (default 1.6)  */
    double eps;          /* ADMM stopping: max(prim, dual) inf-norm      (default 1e-2 with polish, 1e-5 without) */
    int32_t max_admm;    /* ADMM iterations per block                    (default 400)  */
    int32_t polish;      /* 1: active-set polish + KKT certificate (tight mode); 0: OSQP-equivalent mode */
    int32_t max_polish;  /* active-set rounds per polish                 (default 8)    */
    int32_t admm_first;  /* tight mode only. 0: warm-started active-set rounds first, ADMM block as fallback (default);
                            1: always run an ADMM block to eps before the active-set rounds */
    int32_t adaptive_rho;/* 0 / 1: rho is rescaled from the primal / dual residual ratio at a few check points, with a
                            re-factorisation, as OSQP's adaptive_rho does (default); -1: fixed rho */
    int32_t kkt_fallback;/* tight mode only.  0: a QP that the Riccati-based active set cannot certify ends with status 2
                            (default).  1: such a QP is handed to a pivoted stage-wise KKT solve (states and costates as
                            unknowns of one almost-block-diagonal system, row partial pivoting) with primal-dual active-set
                            rounds from an empty working set -- what the reference's sparse solver does, and the only thing
                            that works for the order-1 model at H = 100, where the cost-to-go leaves the fp64 range.
                            2: the same as soon as the Riccati path breaks down numerically (a settled working set whose
                            solve is not stationary or not finite, or a rollout that grows by more than 1e3 over the
                            horizon), and from then on for every QP of that member, across the launches of a
                            split run too (the switch is part of the state m4q_mpc_closed_loop carries).
                            4: every QP goes to the KKT solve (no Riccati attempt): slow; for cross-checking the two
                            solvers against each other on any problem.  Needs H (2n+m)(4n+2m+2) doubles per resident warp (n = 2c), which
                            m4q_mpc_table_bytes / m4q_qp_workspace_bytes_kkt include when this is set. */
} m4q_qp_settings;

/* Problem description of the closed loop (mpc.py:128-304).  Shared (member-independent) data. */
typedef struct {
    int32_t c;             /* complex model-state dimension dim_x                               */
    int32_t m;             /* number of controls dim_u                                           */
    int32_t p;             /* number of control monomials (model.py:95-103: A = [A_x | A_u])     */
    int32_t d;             /* plant Hilbert-space dimension (plant state is d*d complex); 0 = external plant */
    int32_t horizon;       /* StepClock.horizon  (mpc.py:17)                                     */
    int32_t n_steps;       /* StepClock.n_steps  (mpc.py:18)                                     */
    int32_t measure_freq;  /* StepClock.measure_freq (mpc.py:19, :252)                           */
    int32_t warm_start;    /* mpc(..., warm_start) (mpc.py:208)                                  */
    int32_t max_iter;      /* mpc(..., max_iter) SQP iterations per step (mpc.py:173)            */
    int32_t lift_mode;     /* M4Q_LIFT_*                                                         */
    int32_t has_du;        /* 0: du=None (optimize.py:29)                                        */
    int32_t n_targ;        /* columns of X_targ (>= n_steps + horizon + 1)                       */
    double dt;             /* StepClock.dt                                                       */
    double sat;            /* control saturation (optimize.py:43)                                */
    double du;             /* bound on |u_0 - u_prev| (optimize.py:30)                           */
    double exit_infidelity;/* >0: built-in exit condition 1 - Re<fid_vec, x> < value (mpc.py:289-292); <=0 off */
    const double *A_blocks;   /* [p+1][c][c] complex: block 0 = A_x, block k = N_k (linearize.py:32)   */
    const int32_t *powers;    /* [p][m] exponents of the monomials (linearize.py:113-116)              */
    const double *Q;          /* [c][c] complex  (mpc.py:149)                                          */
    const double *Qf;         /* [c][c] complex  (mpc.py:150)                                          */
    const double *R;          /* [m][m] real     (mpc.py:151)                                          */
    const double *X_targ;     /* [c][n_targ] complex (mpc.py:145, :276)                                */
    const double *U_targ;     /* [m][n_targ-1] real   (mpc.py:146, :277)                               */
    const double *fid_vec;    /* [d*d] complex or NULL: fidelity[k] = Re sum conj(fid_vec) * x_final   */
    m4q_qp_settings qp;
    int32_t model_per_member; /* 0: A_blocks is one model shared by all members; 1: A_blocks is [N][p+1][c][c],
                                 member k controls with its own (perturbed) model -- e.g. the output of
                                 m4q_taylor_discretize_batched regrouped per block                           */
    int32_t model_mode;       /* M4Q_MODEL_TAYLOR (default) or M4Q_MODEL_EXACT (then p == m, measure_freq == 1) */
    /* measurement noise of QExperiment.set_sigma (experiment.py:193-194, :212): every measured plant state gets
       sigma * (N(0,1) + i N(0,1)) added per component, and -- as in the reference, which restarts the next simulate()
       from the stored measurement (mpc.py:259) -- the plant continues from the noisy state.  Counter-based generator
       (Philox4x32-10) keyed by (noise_seed, member), counter (step, component): results do not depend on the launch
       geometry.  noise_sigma = 0 switches it off. */
    double noise_sigma;
    uint64_t noise_seed;
    /* streaming model update (mpc.py:281-285 with OnlineDMDc.fit_iteration, model.py:295-313), per member, after every
       MPC step: z = [x; phi(u) (x) x], gamma = 1 / (1 + z^T P z), A += gamma (y - A z)(P z)^T, P = (P - gamma P z (P z)^T)
       / discount.  As in the reference the controller keeps linearising the operators captured before the loop; the
       updated A is used by the model steps between measurements (measure_freq > 1) and returned.
       streaming = 0: off.  stream_A [N][c][c (p+1)] complex (in: initial model of every member, out: final),
       stream_P [N][c (p+1)][c (p+1)] complex (in: initial P, out: final). */
    int32_t streaming;
    int32_t fidelity_sqrt;    /* 0: fidelity = Re<fid_vec, x> (= <psi|rho|psi> for a pure target); 1: its square root,
                                 qutip.fidelity's convention (tests/test_mpc4quantum.py:590, :691) */
    double stream_discount;   /* OnlineDMDc.discount (model.py:28), 1 = none */
    double *stream_A;
    double *stream_P;
    int64_t member_offset;    /* global index of member 0 of this launch: the noise stream of a member depends on its global
                                 index only, so a sharded ensemble draws the same noise as an unsharded one */
} m4q_mpc_problem;

int m4q_version(void);
const char *m4q_last_error(void);

/* 1 if the (c, m) pair has a compiled kernel instantiation: c in {4, 8, 9, 16} with m in {1, 2, 3, 4}. */
int m4q_supported(int32_t c, int32_t m);

/*
 * Plant step(s): rho <- U rho U^dagger, U = expm(-i (H0 + sum_k u_k H1_k) dt), n_seg consecutive segments.
 * Replaces QExperiment.simulate (experiment.py:202-212, qutip.mesolve) for the piecewise-constant control that
 * mpc.py:256-260 builds.  One thread per member with the matrices in registers (d <= 4, N >= 4096), else one warp
 * per member.
 *   H0 [N][d][d] c128, H1 [N][m][d][d] c128 (member stride 0 allowed via h_stride_members = 0),
 *   u [N][n_seg][m] f64, rho_in [N][d*d] c128, rho_out [N][n_seg][d*d] c128 (state after each segment),
 *   prop_out [N][n_seg][d][d] c128 or NULL (the propagators, for the 1e-10 parity check).
 */
int m4q_expm_step_batched(int64_t N, int32_t d, int32_t m, int32_t n_seg, double dt,
                          const double *H0, const double *H1, int32_t shared_hamiltonian,
                          const double *u, const double *rho_in, double *rho_out, double *prop_out,
                          void *stream);

/*
 * Order-k Taylor blocks of exp((L0 + sum u_i L_i) dt) grouped by control monomial.
 * Replaces discretize_homogeneous (vectorize.py:8-49).  L [N][m+1][c][c] c128 -> out [N][c][c*(p+1)] c128
 * (the reference's hstack layout), powers [p+1][m] int32 including the constant row.
 */
int m4q_taylor_discretize_batched(int64_t N, int32_t c, int32_t m, int32_t order, int32_t p1, double dt,
                                  const double *L, const int32_t *powers, double *out, void *stream);

/*
 * Local linearisation along a guess trajectory.  Replaces WrapModel.get_model_along_traj (linearize.py:61-70):
 *   A_t = A + sum_p phi_p(u_t) N_p, B_t = df/du, Delta_t = f - A_t x_t - B_t u_t, t < H.
 *   Xg [N][c][H+1] c128, Ug [N][m][H] f64 (reference layouts) ->
 *   A_out [N][H][c][c] c128, B_out [N][H][c][m] c128, D_out [N][H][c] c128.
 */
int m4q_linearize_batched(int64_t N, int32_t c, int32_t m, int32_t p, int32_t H,
                          const double *A_blocks, const int32_t *powers,
                          const double *Xg, const double *Ug,
                          double *A_out, double *B_out, double *D_out, void *stream);

/*
 * Exact-discretisation model mode (no counterpart in the reference, whose model is the order-k Taylor expansion of
 * vectorize.py:8-49): x+ = expm(G(u) dt) x with the continuous-time generators G(u) = L_0 + sum_i u_i L_i.
 *   A_t = expm(G(u_t) dt), B_t[:, i] = d/du_i [expm(G(u) dt)] x_t (Frechet derivative applied to x_t),
 *   Delta_t = -B_t u_t.  generators [m+1][c][c] c128 (shared by all instances); other layouts as above.
 */
int m4q_exact_linearize_batched(int64_t N, int32_t c, int32_t m, int32_t H, double dt, const double *generators,
                                const double *Xg, const double *Ug,
                                double *A_out, double *B_out, double *D_out, void *stream);

/*
 * Horizon QP.  Replaces optimize.quad_program (optimize.py:12-60; cvxpy -> OSQP):
 *   min sum_t Re[(x_t-r_t)^H Q_t (x_t-r_t)] + (u_t-ub_t)^T R_t (u_t-ub_t) + terminal
 *   s.t. x_0 = x_init, x_{t+1} = Delta_t + A_t x_t + B_t u_t, |u_t| <= sat, |u_0 - u_prev| <= du.
 * Batched over N independent instances, one warp each; ADMM on the control box whose inner linear system is a
 * time-varying Riccati recursion held in shared memory.
 *   x_init [N][c] c128, X_bm [N][c][H+1] c128, U_bm [N][m][H] f64, Q_ls [N][H+1][c][c] c128, R_ls [N][H][m][m] f64,
 *   A_ls [N][H][c][c] c128, B_ls [N][H][c][m] c128, D_ls [N][H][c] c128, u_prev [N][m] f64 or NULL,
 *   -> X_out [N][c][H+1] c128, U_out [N][m][H] f64, obj_out [N] f64, status_out [N] int32 (0 ok, 2, 3),
 *      iters_out [N][2] int32 (ADMM iterations, Riccati factorisations).
 *   workspace: m4q_qp_workspace_bytes(N, c, m, H) bytes of device memory.
 */
int64_t m4q_qp_workspace_bytes(int64_t N, int32_t c, int32_t m, int32_t H);
int64_t m4q_qp_workspace_bytes_kkt(int64_t N, int32_t c, int32_t m, int32_t H);   /* with settings.kkt_fallback != 0 */
int m4q_qp_admm_batched(int64_t N, int32_t c, int32_t m, int32_t H,
                        const double *x_init, const double *X_bm, const double *U_bm,
                        const double *Q_ls, const double *R_ls,
                        const double *A_ls, const double *B_ls, const double *D_ls,
                        const double *u_prev, double sat, double du, int32_t has_du,
                        const m4q_qp_settings *settings_host,
                        double *X_out, double *U_out, double *obj_out, int32_t *status_out, int32_t *iters_out,
                        void *workspace, void *stream);
/* Launch geometry m4q_qp_admm_batched chooses for N instances (N <= 0: the widest launch, which sizes the KKT
   workspaces of m4q_qp_workspace_bytes_kkt). */
int m4q_qp_launch_info(int64_t N, int32_t c, int32_t m, int32_t H, int32_t *warps_per_cta, int32_t *ctas,
                       int32_t *smem_bytes);

/*
 * Line search of the iterative QP.  Replaces iqp_line_search (mpc.py:101-125), including its pairing of a
 * time-major metric with state-major vectors.  Q_ls [H+1][c][c] c128, R_ls [H][m][m] f64, X_ref [c][H+1] c128 and
 * U_ref [m][H] f64 are shared by the N instances (they are in mpc.py); Xg/Xo [N][c][H+1] c128, Ug/Uo [N][m][H] f64.
 * alpha_out [N], step_out [N].  workspace: m4q_line_search_workspace_bytes(c, m, H) bytes of device memory.
 */
int64_t m4q_line_search_workspace_bytes(int32_t c, int32_t m, int32_t H);
int m4q_line_search_batched(int64_t N, int32_t c, int32_t m, int32_t H,
                            const double *Q_ls, const double *R_ls,
                            const double *X_ref, const double *U_ref,
                            const double *Xg, const double *Ug, const double *Xo, const double *Uo,
                            double *alpha_out, double *step_out, void *workspace, void *stream);

/*
 * The closed loop.  Replaces mpc() (mpc.py:128-304) for N ensemble members that share the model, cost and
 * targets and differ in plant Hamiltonian and/or initial state.  One warp per member; all MPC steps in
 * [step_begin, step_end) run on the device with no host round trip.
 *   x0 [N or 1][d*d] c128 (x0_stride_members = 0 broadcasts), H0 [N][d][d], H1 [N][m][d][d] c128
 *   xs [N][d*d][S+1] c128 (reference layout of data[0]); us [N][m][S] f64 (data[1]);
 *   exit_code [N] int32; steps_done [N] int32; qp_count [N][S] int32 (QP solves per MPC step);
 *   counters [N][4] int32 (ADMM iterations, Riccati factorisations, polish rounds, QP solves);
 *   fidelity [N] f64 or NULL.
 *   external_plant != 0 (with prob.d = 0): the kernel does not propagate the plant; xs is [N][c][S+1] and holds
 *   LIFTED model states which the caller writes into xs[:, :, step_begin] before each single-step launch
 *   (host-stepped mode for a user-defined Experiment.simulate / exit_condition; mpc.py:247-292 stay on the host).
 *   state: m4q_mpc_state_bytes(prob, N) bytes, carries each member between launches: per member the guesses Xg and
 *   Ug, the ADMM duals z and y, the measured plant state and, last, one flags word (the KKT switch of
 *   kkt_fallback = 2), so that a run split into step ranges computes what one launch computes.  A member whose exit
 *   code is not 0 when a launch with step_begin > 0 starts is left untouched by that launch: its exit code, steps,
 *   counters, fidelity and state keep the values of the launch it stopped in.
 *   noise_sigma > 0 is refused for the process lift (M4Q_LIFT_PROCESS), which measures a propagator.
 *   tables: m4q_mpc_table_bytes(prob) bytes of device memory, owned by the caller, re-usable across launches of the
 *   same problem: the member-independent tables (realified costs, targets) followed by one L2-resident workspace
 *   per resident warp (stage records [K | S^-1 | dv | B | D | A_t | x - r] and the state trajectories of the member
 *   the warp is working on; sized for the widest launch on the current device, independent of N).
 *   Environment (measurement aids): M4Q_MAX_WARPS caps the members per CTA; M4Q_L2_PERSIST=0 disables the
 *   persisting-L2 access-policy window that the launch sets on `stream` for the workspaces; M4Q_HERM_FACTOR=0 keeps
 *   every Riccati factorisation in realified coordinates (m4q_mpc_herm_sigma).
 */
int64_t m4q_mpc_state_bytes(const m4q_mpc_problem *prob_host, int64_t N);
int64_t m4q_mpc_table_bytes(const m4q_mpc_problem *prob_host);
int m4q_mpc_closed_loop(const m4q_mpc_problem *prob_host, int64_t N,
                        const double *x0, int32_t x0_shared,
                        const double *H0, const double *H1, int32_t shared_hamiltonian,
                        int32_t step_begin, int32_t step_end, int32_t external_plant,
                        double *xs, double *us, int32_t *exit_code, int32_t *steps_done,
                        int32_t *qp_count, int32_t *counters, double *fidelity,
                        void *state, void *tables, void *stream);

/* The index involution sigma of the problem's lift (sigma [c]): a Hermitian plant state lifts to x with
   x[sigma[k]] = conj(x[k]).  Returns 1 if the lift has one, 0 if not, -1 on error.  When the model blocks and costs are
   sigma-symmetric and a QP's guess trajectory is sigma-conjugate-symmetric, the closed loop runs that QP's Riccati
   factorisations in the c real coordinates of the Hermitian subspace instead of the 2c realified ones (c = 9). */
int m4q_mpc_herm_sigma(const m4q_mpc_problem *prob_host, int32_t *sigma);
/* Byte offset, inside the tables, of two uint64 counters of the last launch: Riccati factorisations run in Hermitian
   coordinates and in realified coordinates, summed over the members. */
int64_t m4q_mpc_factor_counts_offset(const m4q_mpc_problem *prob_host);

/* Launch geometry chosen for a problem and N members (N <= 0: the widest launch, which sizes the tables);
   for reporting / roofline accounting. */
int m4q_mpc_launch_info(const m4q_mpc_problem *prob_host, int64_t N, int32_t *warps_per_cta, int32_t *ctas,
                        int32_t *smem_bytes);

/* 256-bin (or nbins) histogram of fidelities on [lo, hi]; counts [nbins] int64 are ADDED to (NCCL all-reduce later). */
int m4q_hist_fidelity(int64_t N, const double *fidelity, double lo, double hi, int32_t nbins,
                      int64_t *counts, void *stream);

/*
 * Measurement aid: `ctas` CTAs of 256 threads each run `iters` x 16 independent fp64 FMAs per thread
 * (2 * 16 * iters * 256 * ctas flops).  Timed by the caller with events on `stream`; gives the fp64 roofline
 * denominator on the part the benchmark runs on.  scratch: >= 8 bytes of device memory.
 */
int m4q_fp64_fma_probe(int32_t ctas, int64_t iters, double *scratch, void *stream);
/* same for the fp64 tensor-core path: each warp issues 8 * iters mma.sync.m8n8k4.f64 (512 flops each) */
int m4q_fp64_dmma_probe(int32_t ctas, int64_t iters, double *scratch, void *stream);

#ifdef __cplusplus
}
#endif
#endif
