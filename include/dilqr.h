/* dilqr.h -- C ABI of libdilqr (B200 / sm_100a batched differentiable iLQR-MPC).
 *
 * This is the drop-in boundary for the hot path of josef-w/Differentiable-iLQR
 * (a pure PyTorch reference; it has no FFI of its own, so each entry point
 * below names the *Python* function it replaces, file:line relative to the
 * reference root).  Plain pointers and sizes only: no torch types.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated otherwise; tensors are
 *     contiguous, time-major, batch-second exactly as in the reference
 *     (mpc.py:185-186): C[T,B,n,n] c[T,B,n] F[T-1,B,ns,n] f[T-1,B,ns]
 *     x[T,B,ns] u[T,B,nc] x_init[B,ns], n = ns + nc;
 *   - `dtype` selects float (DILQR_F32) or double (DILQR_F64) for ALL float
 *     tensors of a call;
 *   - the caller owns every buffer including the workspace; the library never
 *     allocates, frees or synchronises; all work is enqueued on `stream`
 *     (a cudaStream_t passed as void*);
 *   - return value: 0 on success, negative DILQR_E* on error (nothing enqueued);
 *     numerical non-convergence is data (status block), never an error.
 */
#ifndef DILQR_H_
#define DILQR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { DILQR_F32 = 0, DILQR_F64 = 1 };

/* Where F_t comes from / what the rollouts integrate. */
enum {
  DILQR_DYN_LINDX    = 0, /* definitions.py:4  LinDx(F,f): x' = F_t [x;u] (+ f_t)      */
  DILQR_DYN_PENDULUM = 1, /* env_dx/pendulum.py:60-95, Jacobian 444-475             */
  DILQR_DYN_CARTPOLE = 2, /* env_dx/cartpole.py:64-97, Jacobian 790-839             */
  DILQR_DYN_ROCKET   = 3, /* env_dx/rocket.py:82-164,  Jacobian 324-426             */
  DILQR_DYN_NN       = 4, /* dynamics.py:15-130 NNDynamics, one or two hidden layers
                             (dyn_aux, dyn_ai); compiled shapes only                   */
  DILQR_DYN_LINDX_RT = 5, /* LinDx through the runtime-dimension kernels (rt_kernels.cuh):
                             any n_state >= 1, n_ctrl >= 1 with n_state + n_ctrl <= 32, both
                             dtypes; same problem struct and entry points as DILQR_DYN_LINDX.
                             Replays the pnqp trace (never the group sweep); dilqr_mpc_gains
                             and the DiLQR backward calls do not serve it.  Select it with
                             dilqr_lindx_kernels.                                         */
  DILQR_DYN_NN_RT    = 6  /* NNDynamics through the runtime-dimension kernels: any n_state >= 1,
                             n_ctrl >= 1 with n_state + n_ctrl <= 32, both dtypes; the same
                             network limits, DilqrSolve fields (dyn_aux, dyn_ai) and entry points
                             as DILQR_DYN_NN.  Replays the pnqp trace (never the group sweep);
                             dilqr_mpc_gains does not serve it and dilqr_kkt_grads rejects it (the
                             gradient of a network solve is a LinDx KKT problem at the solution).
                             Select it with dilqr_nn_kernels.                                   */
};

/* How unconstrained multi-input gains are solved (the reference copies differ). */
enum {
  DILQR_GAIN_PLAIN    = 0, /* lqr_step.py:88-94 (pinverse of an SPD Quu == inverse)  */
  DILQR_GAIN_CHOL_REG = 1  /* lqr_step_backup.py:202-205 (Cholesky of Quu + 1e-6 I)  */
};

enum { DILQR_BOUNDS_NONE = 0, DILQR_BOUNDS_SCALAR = 1, DILQR_BOUNDS_TENSOR = 2 };

enum {
  DILQR_OK = 0,
  DILQR_EINVAL = -1,       /* bad dims / null pointer / bad enum                   */
  DILQR_EUNSUPPORTED = -2, /* (dtype, n_state, n_ctrl, dynamics) not instantiated  */
  DILQR_EALIGN = -3,       /* a pointer is not 16-byte aligned                      */
  DILQR_EWORKSPACE = -4,   /* workspace too small                                   */
  DILQR_ECUDA = -5,        /* kernel launch failed (cudaGetLastError != success)    */
  DILQR_ELOCKSTEP = -6     /* group sweep: the batch does not fit the device at once */
};

#define DILQR_PNQP_MAX_ITER 20   /* pnqp.py:5  n_iter=20 (lqr_step.py:137)           */

/* Host-visible solver status, written by dilqr_mpc_commit into DEVICE memory
 * (`status` below); the host copies it back once per iLQR iteration to apply
 * the stop rule of mpc.py:299-301. */
typedef struct DilqrStatus {
  uint32_t trace_match;     /* 1: pnqp control-flow guess == votes (iteration valid) */
  uint32_t any_improved;    /* any problem improved its best cost (mpc.py:280-281)   */
  uint32_t n_total_qp_iter; /* sum_t (1 + n_qp_iter_t)            (lqr_step.py:140)  */
  uint32_t pnqp_unconverged;/* #timesteps where pnqp hit n_iter   (pnqp.py:81)       */
  double   max_full_du;     /* max_b ||u - u_new||_2              (mpc.py:299)       */
  double   mean_alpha;      /* mean_b alpha_b                     (lqr_step.py:259)  */
  double   mean_best_cost;  /* mean_b best cost (verbose table,   mpc.py:288)        */
  uint32_t first_mismatch;  /* slot index of first trace mismatch (debug)            */
  uint32_t n_active;        /* solo == 2: problems whose own stop rule has not fired */
  uint32_t reserved[4];
} DilqrStatus;

/* Optional device-resident outer-loop state: with `control` set in DilqrSolve the
 * caller may enqueue ALL iterations (iterate+commit pairs, status = one DilqrStatus per
 * iteration) without synchronising; the stop rule of mpc.py:299-301 and the trace
 * check run on the device and later launches turn into no-ops once `halt` is set.
 * The host reads the block once at the end: halt == 2 means iteration `iters_done`
 * must be re-enqueued (its pnqp trace guess was wrong and has been corrected). */
typedef struct DilqrControl {
  uint32_t halt;            /* 0 running, 1 stop rule fired, 2 pnqp trace mismatch     */
  uint32_t iters_done;      /* committed iLQR iterations                               */
  uint32_t n_not_improved;  /* mpc.py:245,266,281                                      */
  uint32_t not_improved_lim;/* mpc.py:141                                              */
  double   eps;             /* mpc.py:131, already rounded to the data dtype           */
  uint32_t reserved[10];
} DilqrControl;

/* One batched MPC / LQR problem instance.  Unused pointers may be NULL. */
typedef struct DilqrSolve {
  int32_t n_state, n_ctrl, T, n_batch;
  int32_t dtype;            /* DILQR_F32 / DILQR_F64                                */
  int32_t dynamics;         /* DILQR_DYN_*                                          */
  int32_t gain_solve;       /* DILQR_GAIN_*                                         */
  int32_t bounds_kind;      /* DILQR_BOUNDS_*                                       */
  int32_t solo;             /* 0: batch-global pnqp control flow (== reference on
                               the same batch); 1: per-problem pnqp / Armijo flags
                               (== reference B=1 for one LQR step); 2: additionally the
                               outer loop per problem -- own ||du||, own n_not_improved,
                               own stop rule (mpc.py:266,281,299-301): every problem ==
                               the reference called with n_batch=1 (il_env.py:96-151).
                               2 needs `control` for the stop thresholds             */
  int32_t max_linesearch_iter; /* mpc.py:135                                        */
  int32_t iteration;        /* 0-based iLQR iteration index of this iterate/commit call
                               (0: first -> best := new, mpc.py:271; parity selects
                               the ping-pong trajectory buffer)                      */
  int32_t has_f;            /* LinDx: f present (util.py:121)                        */
  int32_t gains_only;       /* iterate: only lqr_backward (K_out,k_out), no rollout --
                               the final no-op LQR pass of lqr_step_explicit.py:604-618 */
  int32_t C_bcast, c_bcast; /* cost layout (mpc.py:205-219): 0 dense C[T,B,n,n] / c[T,B,n];
                               1 batch-broadcast C[T,n,n] / c[T,n]; 2 C[n,n] / c[n] -- the
                               kernels read the single shared block, nothing is tiled   */
  double  linesearch_decay; /* mpc.py:134                                           */
  double  u_lower, u_upper; /* scalar bounds (mpc.py:81-82)                         */
  double  best_cost_eps;    /* mpc.py:142                                           */
  double  dyn_params[8];    /* env parameters theta (pendulum g,m,l; cartpole
                               g,m_c,m_p,l; rocket Jx,Jy,Jz,mass,l), host copy      */
  /* inputs */
  const void* x_init;       /* [B,ns]                                               */
  const void* C;            /* [T,B,n,n]  (or [T,n,n] / [n,n], see C_bcast)          */
  const void* c;            /* [T,B,n]    (or [T,n] / [n], see c_bcast)              */
  const void* F;            /* [T-1,B,ns,n]  (LinDx)                                */
  const void* f;            /* [T-1,B,ns]    (LinDx, optional)                      */
  const void* u_init;       /* [T,B,nc] or NULL (zeros, mpc.py:230-231)             */
  const void* x_cur;        /* [T,B,ns] current trajectory (single LQR step only)    */
  const void* u_lower_t;    /* [T,B,nc] tensor bounds (lqr_step.py:264-272)         */
  const void* u_upper_t;
  const uint8_t* u_zero_I;  /* [T,B,nc] bool mask or NULL (lqr_step.py:99-127)      */
  /* outputs */
  void* x_out;              /* [T,B,ns]                                             */
  void* u_out;              /* [T,B,nc]                                             */
  void* cost_out;           /* [B]                                                  */
  void* du_out;             /* [B]  full_du_norm                                    */
  void* alpha_out;          /* [B]  accepted line-search step (lqr_step only)       */
  void* K_out;              /* [T,B,nc,ns] gains, FORWARD time order (optional)     */
  void* k_out;              /* [T,B,nc]    (optional)                               */
  DilqrStatus* status;      /* device; the block this iteration's commit writes      */
  DilqrControl* control;    /* device, optional (see DilqrControl)                   */
  /* scratch */
  void*  workspace;
  size_t workspace_bytes;
  /* DILQR_DYN_NN / DILQR_DYN_NN_RT only: the network of dynamics.NNDynamics(hidden_sizes=[H] or
     [H1,H2]) */
  const void* dyn_aux;      /* device, packed in the call's dtype, layer by layer:
                               weight[out][in] then bias[out] (fc0, fc1[, fc2])        */
  int32_t dyn_ai[4];        /* {H1 | H2 << 16 (H2 = 0: one hidden layer; two layers need
                               H1 <= 128, H1 < 65536 otherwise), activation (0 sigmoid /
                               1 relu), passthrough,
                               linearisation: 0 analytic (grad_input), 1 central
                               differences eps=1e-4 (GradMethods.FINITE_DIFF)}       */
  /* trust region on the control change of one LQR step (mpc.py:93, lqr_step.py:132-134,
     204-211); needs box constraints (lqr_step.py:195) */
  double  delta_u;
  int32_t has_delta_u;
  int32_t gains_guess_reset; /* dilqr_mpc_gains keeps its own pnqp trace guess in the workspace,
                                carried from call to call (a training loop revisits nearly the
                                same solutions, so the guess of the previous step is right);
                                1: start from the default guess (first use of a workspace)      */
  int32_t keep_trace_guess;  /* dilqr_mpc_begin: 1 keeps the pnqp trace guess the previous solve in
                                this workspace ended with (same shape; steady-state loops) instead
                                of resetting it to the default                                    */
  int32_t group_sweep;       /* written by dilqr_mpc_plan.  1: iterate runs the Riccati / pnqp sweep
                                with the batch-synchronous thread-group kernel
                                (csrc/group_kernels.cuh): G lanes per problem, every batch-global pnqp
                                decision a grid barrier, no trace replay.  0: one thread per problem,
                                replaying a guessed trace.  dilqr_workspace_bytes depends on it      */
} DilqrSolve;

const char* dilqr_version(void);

/* 1 if kernels for this combination are compiled in, else 0.  DILQR_DYN_LINDX_RT and
 * DILQR_DYN_NN_RT: 1 for every shape of their range, compiled-in shapes included. */
int dilqr_supported(int dtype, int n_state, int n_ctrl, int dynamics);

/* Which kernels serve a LinDx problem of this shape: DILQR_DYN_LINDX if the shape is compiled in,
 * else DILQR_DYN_LINDX_RT if n_state + n_ctrl <= 32, else DILQR_EUNSUPPORTED; DILQR_EINVAL for a
 * bad dtype or a non-positive dimension.  Put the result into DilqrSolve.dynamics /
 * DilqrKkt.dynamics. */
int dilqr_lindx_kernels(int dtype, int n_state, int n_ctrl);

/* The same choice for a network (NNDynamics) problem: DILQR_DYN_NN if the shape is compiled in,
 * else DILQR_DYN_NN_RT if n_state + n_ctrl <= 32, else DILQR_EUNSUPPORTED; DILQR_EINVAL for a bad
 * dtype or a non-positive dimension.  Put the result into DilqrSolve.dynamics. */
int dilqr_nn_kernels(int dtype, int n_state, int n_ctrl);

/* Choose how dilqr_mpc_iterate resolves pnqp's batch-global decisions and write it to
 * s->group_sweep.  Reads only dtype, n_state, n_ctrl, dynamics, bounds_kind, solo and n_batch;
 * call it before dilqr_workspace_bytes.  The group sweep runs shapes whose matrices do not fit
 * one thread's registers, and box-constrained (solo == 0) multi-input batches, wherever the
 * shape has it and the batch fits the current device at once; everything else replays a
 * guessed trace.  DILQR_DYN_LINDX_RT and DILQR_DYN_NN_RT always replay (group_sweep = 0) and
 * never query the device.  DILQR_EUNSUPPORTED: the shape is not compiled in (the runtime ids: out
 * of their range). */
int dilqr_mpc_plan(DilqrSolve* s);

/* Bytes of workspace the dilqr_mpc_* calls need. */
size_t dilqr_workspace_bytes(const DilqrSolve* s);

/* What the solve leaves in its workspace for the backward pass (valid until the workspace is
 * reused): the gains Kk warp-blocked [T][ceil(B/32)][nc*ns+nc][32] (K then k; written by
 * iterate / dilqr_mpc_gains), the packed upper triangle of C [T][ceil(B/32)][n(n+1)/2][32]
 * with its validity word (1: every C[t,b] was bitwise symmetric and the copy exists). */
typedef struct DilqrWsView {
  void* Kk;
  const void* Cpk;
  const uint32_t* cpk_state;
  int32_t n_warps;          /* ceil(B/32) */
  int32_t reserved;
} DilqrWsView;
int dilqr_workspace_view(const DilqrSolve* s, DilqrWsView* view);

/* ---- iLQR outer loop, MPC.forward (mpc.py:184-337, mpc_explicit.py:182-358) -- */

/* Initial nominal rollout x = get_traj(u_init) (util.py:104-127) and its cost
 * (util.py:130-153); resets the best-iterate record and the pnqp trace guess. */
int dilqr_mpc_begin(const DilqrSolve* s, void* stream);

/* One fused iLQR iteration = LQRStepFn.forward (lqr_step.py:277-309):
 * c_back (289-295) + analytic linearisation (mpc_explicit.py:516-546) +
 * Riccati backward with pnqp (lqr_step.py:52-160, pnqp.py:5-82) + line-search
 * rollout over the true dynamics (lqr_step.py:164-261).  Results are staged;
 * nothing is committed until dilqr_mpc_commit. */
int dilqr_mpc_iterate(const DilqrSolve* s, void* stream);

/* Verify the pnqp control-flow trace, then per problem the best-iterate
 * bookkeeping of mpc.py:271-285 and the batch reductions of mpc.py:299-301;
 * writes *s->status.  If status.trace_match == 0 nothing was committed: call
 * dilqr_mpc_iterate + dilqr_mpc_commit again (the guess has been corrected). */
int dilqr_mpc_commit(const DilqrSolve* s, void* stream);

/* Gather the best iterate into x_out,u_out,cost_out,du_out (mpc.py:304-306). */
int dilqr_mpc_finish(const DilqrSolve* s, void* stream);

/* Gains of the final no-op LQR pass at the solution (lqr_step_explicit.py:604-618) and the
 * primal costates (lqr_step.py:355-369) in ONE sweep over s->x_out, s->u_out (the solution as
 * dilqr_mpc_finish returned it), C read from the packed workspace copy when valid.  Writes
 * the gains into the workspace (DilqrWsView.Kk) and lam_blk [T][ceil(B/32)][ns][32]
 * (optional); verifies the pnqp trace into *s->status like dilqr_mpc_commit.  Staged env_dx
 * shapes only (DILQR_EUNSUPPORTED otherwise: use the LQR-step call sequence below). */
int dilqr_mpc_gains(const DilqrSolve* s, void* lam_blk, void* stream);

/* A single LQR step, LQRStep(...)(x_init,C,c,F,f) (lqr_step.py:22-38,277-309), is
 * the same call sequence with `x_cur` (and `u_init` = current u) set: dilqr_mpc_begin
 * then loads the given trajectory instead of rolling it out, one
 * dilqr_mpc_iterate + dilqr_mpc_commit (iteration = 0) runs the step, and
 * dilqr_mpc_finish returns the new iterate (x_out,u_out,cost_out,du_out,
 * alpha_out) and, if requested, the gains K_out,k_out of lqr_backward. */

/* ---- standalone pnqp (pnqp.py:5-82) --------------------------------------
 * H[B,n,n] q[B,n] lower[B,n] upper[B,n] x_init[B,n] (or NULL: unconstrained
 * minimiser, pnqp.py:14-19) -> x[B,n], lu[B,n,n] + pivots[B,n] (LAPACK getrf layout
 * of the masked Hessian H_ + 1e-11 I of the last iteration, what Tensor.lu() returns;
 * n == 1: the scalar H_), If[B,n] (float 0/1).  `trace`: 40 device words (20-word
 * control-flow guess, zero-initialised by the caller before the first call, then
 * 20 vote words).  After the call status->trace_match tells whether the replayed
 * batch-global control flow was right; if 0, call again (the guess was corrected).
 * status->n_total_qp_iter - 1 is the returned iteration count `i`,
 * status->pnqp_unconverged != 0 the "[WARNING] pnqp warning" case (pnqp.py:81).
 * Compiled for n in {1,2,3,4,6,8} and n_iter = DILQR_PNQP_MAX_ITER (else DILQR_EUNSUPPORTED);
 * every other size up to 256 and budget up to 1024 is served by dilqr_pnqp_rt below. */
int dilqr_pnqp(int dtype, int n, int n_batch, const void* H, const void* q, const void* lower,
               const void* upper, const void* x_init, void* x, void* lu, int32_t* pivots,
               void* If, uint32_t* trace, int solo, DilqrStatus* status, void* stream);

/* Which kernels serve a standalone pnqp of size n with budget n_iter: DILQR_PNQP_COMPILED
 * (dilqr_pnqp) for n in {1,2,3,4,6,8} with n_iter == DILQR_PNQP_MAX_ITER, else DILQR_PNQP_RT
 * (dilqr_pnqp_rt) for n <= DILQR_PNQP_RT_MAX_N and n_iter <= DILQR_PNQP_RT_MAX_ITER, else
 * DILQR_EUNSUPPORTED; DILQR_EINVAL for a bad dtype or n <= 0 or n_iter <= 0. */
enum { DILQR_PNQP_COMPILED = 0, DILQR_PNQP_RT = 1 };
#define DILQR_PNQP_RT_MAX_N 256
#define DILQR_PNQP_RT_MAX_ITER 1024
int dilqr_pnqp_kernels(int dtype, int n, int n_iter);

/* dilqr_pnqp with n and the iteration budget n_iter at run time (csrc/pnqp_rt.cuh, one warp per
 * problem): any 1 <= n <= DILQR_PNQP_RT_MAX_N, 1 <= n_iter <= DILQR_PNQP_RT_MAX_ITER, both dtypes,
 * the compiled sizes included (where it returns bitwise what dilqr_pnqp returns).  Same
 * arguments, outputs and status fields as dilqr_pnqp, except that `trace` holds 2 * n_iter
 * words (n_iter guess words, zero-initialised by the caller before the first call, then n_iter
 * vote words) and needs only 4-byte alignment.  DILQR_EINVAL for a null pointer, n_batch <= 0,
 * n <= 0 or n_iter <= 0, DILQR_EUNSUPPORTED beyond the limits, DILQR_EALIGN for a misaligned
 * `trace`; nothing is enqueued then. */
int dilqr_pnqp_rt(int dtype, int n, int n_iter, int n_batch, const void* H, const void* q,
                  const void* lower, const void* upper, const void* x_init, void* x, void* lu,
                  int32_t* pivots, void* If, uint32_t* trace, int solo, DilqrStatus* status,
                  void* stream);

/* ---- analytic linearisation (mpc_explicit.py:516-546) --------------------
 * x[T,B,ns], u[T,B,nc] -> F[T-1,B,ns,n], f[T-1,B,ns] (f may be NULL). */
int dilqr_linearize(int dtype, int dynamics, const double* dyn_params, int T,
                    int n_batch, const void* x, const void* u, void* F, void* f,
                    void* stream);

/* ---- nominal rollout, util.get_traj (util.py:104-127) for env dynamics ---- */
int dilqr_rollout(int dtype, int dynamics, const double* dyn_params, int T,
                  int n_batch, const void* x_init, const void* u, void* x,
                  void* stream);

/* ---- KKT / adjoint-LQR backward, LQRStepFn.backward (lqr_step.py:312-407) --
 * Given the adjoint solution (dx,du) of the masked LQR (computed with
 * dilqr_mpc_* on cost (C,-r), LinDx(F,None), x_init=0, u_zero_I=active set),
 * the two costate recursions and outer products:
 *   dC[T,B,n,n] dc[T,B,n] dF[T-1,B,ns,n] df[T-1,B,ns] dx_init[B,ns].
 * Any output pointer may be NULL to skip it. */
typedef struct DilqrKkt {
  int32_t n_state, n_ctrl, T, n_batch, dtype;
  int32_t dynamics;             /* DILQR_DYN_LINDX (compiled shapes) or DILQR_DYN_LINDX_RT
                                   (dilqr_lindx_kernels); other values: DILQR_EINVAL */
  const void *C, *c, *F;        /* problem data                               */
  const void *x, *u;            /* solution  x*[T,B,ns], u*[T,B,nc]           */
  const void *dx, *du;          /* adjoint solution                           */
  const void *r;                /* [T,B,n] = cat(dl_dx, dl_du)                 */
  void *dC, *dc, *dF, *df, *dx_init;
} DilqrKkt;
int dilqr_kkt_grads(const DilqrKkt* k, void* stream);

/* ---- DiLQR implicit (fixed-point) gradient, LQRStepFn.backward +
 * fix_point_equ (lqr_step_explicit.py:652-712, 458-598), matrix-free -------- */

/* Primal costates lam[T,B,ns] (lqr_step_explicit.py:305-319) and contracted
 * second-order tables Lam_t[k][j] = sum_i lam_{t+1}[i] dD_t[i][j]/dtau_k with dD/dtau
 * from get_matrices (cartpole.py:425-613, pendulum.py:152-382).  packed == 0: dense
 * Lam[T-1,B,n,n] (for dilqr_richardson_update); packed == 1: only the structurally
 * non-zero entries, warp-blocked [T-1][ceil(B/32)][dilqr_lam_pack_size()][32] (for
 * dilqr_adjoint_pass). */
int dilqr_lam_pack_size(int dynamics);
int dilqr_costate_tables(int dtype, int dynamics, const double* dyn_params, int T, int n_batch,
                         const void* C, const void* c, const void* x, const void* u, void* lam,
                         void* Lam, int C_bcast, int c_bcast, int packed, void* stream);

/* The contracted second-order tables alone, from tau* and the warp-blocked costates of
 * dilqr_mpc_gains: one thread per (t, problem) -- no recursion in t is left.  Lam is the packed
 * layout of dilqr_costate_tables(packed = 1). */
int dilqr_lam_tables(int dtype, int dynamics, const double* dyn_params, int T, int n_batch,
                     const void* x, const void* u, const void* lam_blk, void* Lam, void* stream);

/* One Richardson update of A' w = g:  w_t = g_t - Lam_t dtau_t (t < T-1),
 * w_{T-1} = g_{T-1}; writes w and -w, and resid[0] = max|w_new - w_old|,
 * resid[1] = max|w_new| (two doubles, device).  (dx,du) is the adjoint LQR
 * solution for r = w_old (lqr_step_explicit.py:276-303). */
int dilqr_richardson_update(int dtype, int n_state, int n_ctrl, int T, int n_batch, const void* g,
                            const void* Lam, const void* dx, const void* du, void* w, void* negw,
                            void* resid, void* stream);

/* get_matrices (cartpole.py:105-716, pendulum.py:152-382, rocket.py:258-261) as
 * materialised tensors for n sample rows x[n,ns], u[n,nc]; out[0..6] =
 * D[n,ns,N], D_grad_params[n,ns,N,nth], D_grad_x[n,ns,N,ns], D_grad_u[n,ns,N,nc],
 * x_grad_theta[n,ns,nth], x_grad_xtm1[n,ns,ns], x_grad_utm1[n,ns,nc]. */
int dilqr_env_tables(int dtype, int dynamics, const double* dyn_params, int n, const void* x,
                     const void* u, void* const* out, void* stream);

/* Adjoint (KKT) LQR solves of the DiLQR backward for env_dx dynamics, factored
 * once and replayed per Richardson pass (lqr_step_explicit.py:276-303 restated;
 * see csrc/adjoint_kernels.cuh).  F_t = D(x*_t,u*_t) is re-derived on the fly. */
typedef struct DilqrAdjoint {
  int32_t n_state, n_ctrl, T, n_batch, dtype, dynamics;
  int32_t bounds_kind;   /* NONE: no active set; SCALAR: I = |u*-bound| <= 1e-8 (:690-691) */
  int32_t gain_solve;    /* DILQR_GAIN_CHOL_REG for the explicit variant (mpc_backup)      */
  int32_t C_bcast, c_bcast; /* cost layout as in DilqrSolve; for a broadcast C (c) the final
                               pass writes per-warp PARTIAL sums of the gradient:
                               dC[T][ceil(B/32)][n*n] (mode 1) or [ceil(B/32)][n*n] (mode 2),
                               to be summed over the warp axis by the caller            */
  double u_lower, u_upper;
  double dyn_params[8];
  const void *C;         /* [T,B,n,n]                                                  */
  const void *x, *u;     /* solution tau* [T,B,ns], [T,B,nc]                           */
  const void *gx, *gu;   /* upstream gradient g = [dl_dx; dl_du] as its two halves [T,B,ns]
                            (NULL: zero) and [T,B,nc] -- never concatenated               */
  const void *Lam;       /* packed Lam from dilqr_costate_tables(packed = 1) / dilqr_lam_tables */
  void *w;               /* [T,B,n]  Richardson iterate; with first_pass = 1 the solve reads
                            its right-hand side from g and w is only written               */
  void *dC, *dc, *df;    /* final pass outputs: [T,B,n,n], [T,B,n], [T-1,B,ns]         */
  void *dx_out, *du_out; /* final pass: adjoint solution (optional)                    */
  void *resid;           /* device, 3 x 8 bytes: max|dw|, max|w| (doubles), #problems
                            whose adjoint step the reference's line search would reject */
  void *workspace;
  size_t workspace_bytes;
  /* --- fused-backward options (all optional, zero = round-1 behaviour) ------------------ */
  const void *Cpk;       /* packed symmetric copy of C the forward solve left in its workspace */
  const uint32_t *cpk_state; /* device word, 1: Cpk valid (dilqr_workspace_view)              */
  int32_t first_pass;    /* the Richardson iterate equals g (first solve): no w <- g copy      */
  int32_t want_resid;    /* pass: reduce resid[0..1] (one extra read of w per pass)            */
  int32_t reduce_tile;   /* final: gradient of the TILED DIAGONAL cost of il_env.py:159-162
                            instead of dC, dc: red_out[ceil(B/32)][2n] per-warp partial sums of
                            sum_{t,b} diag(dC) and sum_{t,b} dc (sum over axis 0 = dq, dp)    */
  int32_t reserved0;
  void *red_out;
  void *df_blk;          /* final: df warp-blocked [T-1][ceil(B/32)][ns][32] for
                            dilqr_sens_theta_adjoint (instead of df)                          */
} DilqrAdjoint;
size_t dilqr_adjoint_workspace_bytes(const DilqrAdjoint* a);
/* Byte offset, inside the adjoint workspace, of the adjoint solution the final pass keeps:
 * dtau warp-blocked [T][ceil(B/32)][n][32] (input of dilqr_sens_theta_adjoint). */
size_t dilqr_adjoint_dtau_offset(const DilqrAdjoint* a);
/* Masked Riccati sweep at tau*: gains and the r-independent blocks.  Needs only C, x, u,
 * bounds, dyn_params, resid and the workspace (not w, g, Lam or the outputs), so it can be
 * enqueued right behind the forward solve, before any upstream gradient exists. */
int dilqr_adjoint_factor(const DilqrAdjoint* a, void* stream);
/* One Richardson pass: adjoint solve with r = w fused with w <- g - Lam dtau. */
int dilqr_adjoint_pass(const DilqrAdjoint* a, void* stream);
/* Adjoint solve with r = w, then costates and dC, dc, df (lqr_step.py:346-402). */
int dilqr_adjoint_final(const DilqrAdjoint* a, void* stream);

/* dtheta[B,n_theta] = sum_t <dF_w, dD_t/dtheta> + <df_w, dd_t/dtheta> with the
 * closed-loop sensitivity rollout grad_input (cartpole.py:717-788, pendulum.py:
 * 383-443) contracted on the fly.  K[T,B,nc,ns]: gains of the final LQR pass in
 * forward time order; df[T-1,B,ns] = -dlam_{t+1} from dilqr_kkt_grads. */
int dilqr_sens_theta(int dtype, int dynamics, const double* dyn_params, int T, int n_batch,
                     const void* x, const void* u, const void* K, const void* lam, const void* dx,
                     const void* du, const void* df, void* dtheta, void* stream);

/* Same sum in adjoint form (one reverse sweep carrying n_state scalars per problem instead of
 * the n_state x n_theta sensitivity matrix; the second-order tables enter through
 * Lam_packed [T-1][ceil(B/32)][dilqr_lam_pack_size][32] of dilqr_lam_tables), with every
 * solver-internal operand in the warp-blocked layout it was produced in: Kk (DilqrWsView),
 * lam_blk (dilqr_mpc_gains), dtau_blk (adjoint workspace + dilqr_adjoint_dtau_offset), df_blk
 * (DilqrAdjoint.df_blk).  Pendulum and cartpole.  Replaces the loop of cartpole.py:755-782 / pendulum.py:412-437 contracted with
 * dF, df (lqr_step_explicit.py:700-708). */
int dilqr_sens_theta_adjoint(int dtype, int dynamics, const double* dyn_params, int T, int n_batch,
                             const void* x, const void* u, const void* Kk, const void* lam_blk,
                             const void* dtau_blk, const void* df_blk, const void* Lam_packed,
                             void* dtheta, void* stream);

/* Kernels the most recent successful dilqr_mpc_iterate enqueued: 1 for the fused sweep +
 * rollout, 2 when that kernel is enqueued as a symmetric / general pair (one exits at once),
 * 2 for the group sweep + its rollout, 1 for the group sweep with gains_only -- launch
 * accounting of the host bindings only. */
int dilqr_last_iterate_launches(void);

/* The cost plumbing either side of the solve in the imitation-learning loop.
 * dilqr_tile_cost: C[T,B,n,n] = diag(q), c[T,B,n] = p for every (t, b) -- what
 * il_env.py:159-162 builds with .repeat (C or c may be NULL to skip one).
 * dilqr_tile_cost_grad: the adjoint of that tiling, dq[i] = sum_{t,b} dC[t,b,i,i],
 * dp[i] = sum_{t,b} dc[t,b,i] (what autograd computes for il_exp.py:373), one pass over
 * dC, dc with a fixed summation order; workspace: dilqr_tile_cost_grad_workspace_bytes(n). */
int dilqr_tile_cost(int dtype, int n, int T, int n_batch, const void* q, const void* p, void* C,
                    void* c, void* stream);
size_t dilqr_tile_cost_grad_workspace_bytes(int n);
int dilqr_tile_cost_grad(int dtype, int n, int T, int n_batch, const void* dC, const void* dc,
                         void* dq, void* dp, void* workspace, size_t workspace_bytes,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DILQR_H_ */
