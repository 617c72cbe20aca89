// dispatch.cu -- the extern "C" surface declared in include/dilqr.h; routes on
// dtype to the per-scalar objects built from api.cu.
#include "../../include/dilqr.h"

namespace dilqr {
// shape-specialised entry points: one copy per (dtype, shape group)
#define DECL_G(sfx)                                                                       \
  int supported_##sfx(int, int, int);                                                     \
  int mpc_plan_##sfx(DilqrSolve*);                                                        \
  int mpc_begin_##sfx(const DilqrSolve*, void*);                                          \
  int mpc_iterate_##sfx(const DilqrSolve*, void*);                                        \
  int mpc_commit_##sfx(const DilqrSolve*, void*);                                         \
  int mpc_finish_##sfx(const DilqrSolve*, void*);                                         \
  int mpc_gains_##sfx(const DilqrSolve*, void*, void*);                                   \
  int kkt_grads_##sfx(const DilqrKkt*, void*);                                            \
  int richardson_update_##sfx(int, int, int, int, const void*, const void*, const void*,   \
                              const void*, void*, void*, void*, void*);
// shape-independent entry points: group 0 only
#define DECL_0(sfx)                                                                       \
  size_t workspace_bytes_##sfx(const DilqrSolve*);                                        \
  int linearize_##sfx(int, const double*, int, int, const void*, const void*, void*, void*, \
                      void*);                                                             \
  int rollout_##sfx(int, const double*, int, int, const void*, const void*, void*, void*); \
  int costate_tables_##sfx(int, const double*, int, int, const void*, const void*, const void*, \
                           const void*, void*, void*, int, int, int, void*);              \
  int lam_pack_size_##sfx(int);                                                           \
  int sens_theta_##sfx(int, const double*, int, int, const void*, const void*, const void*, \
                       const void*, const void*, const void*, const void*, void*, void*); \
  int env_tables_##sfx(int, const double*, int, const void*, const void*, void* const*, void*); \
  int pnqp_##sfx(int, int, const void*, const void*, const void*, const void*, const void*, \
                 void*, void*, int32_t*, void*, uint32_t*, int, DilqrStatus*, void*);     \
  int pnqp_rt_##sfx(int, int, int, const void*, const void*, const void*, const void*,    \
                    const void*, void*, void*, int32_t*, void*, uint32_t*, int, DilqrStatus*, \
                    void*);                                                               \
  size_t adjoint_workspace_bytes_##sfx(const DilqrAdjoint*);                              \
  size_t adjoint_dtau_offset_##sfx(const DilqrAdjoint*);                                  \
  int workspace_view_##sfx(const DilqrSolve*, DilqrWsView*);                              \
  int lam_tables_##sfx(int, const double*, int, int, const void*, const void*, const void*, \
                       void*, void*);                                                     \
  int sens_theta_adjoint_##sfx(int, const double*, int, int, const void*, const void*,    \
                               const void*, const void*, const void*, const void*, const void*, \
                               void*, void*);                                             \
  int adjoint_run_##sfx(const DilqrAdjoint*, int, void*);                                \
  size_t krylov_workspace_bytes_##sfx(const DilqrKrylov*);                                \
  int krylov_run_##sfx(const DilqrKrylov*, int, void*);
DECL_G(f32_g0) DECL_G(f32_g1) DECL_G(f32_g2) DECL_G(f32_g3)
DECL_G(f64_g0) DECL_G(f64_g1) DECL_G(f64_g2) DECL_G(f64_g3)
DECL_0(f32_g0) DECL_0(f64_g0)
#undef DECL_G
#undef DECL_0
}  // namespace dilqr

extern "C" int g_dilqr_iterate_launches;
int g_dilqr_iterate_launches = 1;
int dilqr_last_iterate_launches(void) { return g_dilqr_iterate_launches; }

#define ROUTE(dtype, call32, call64)                   \
  ((dtype) == DILQR_F32 ? (call32) : ((dtype) == DILQR_F64 ? (call64) : DILQR_EINVAL))

// try the shape groups in turn until one has the (n_state, n_ctrl, dynamics) kernels
#define TRY_GROUPS(T, fn, ...)                                   \
  do {                                                           \
    int rc_ = dilqr::fn##_##T##_g0(__VA_ARGS__);                 \
    if (rc_ == DILQR_EUNSUPPORTED) rc_ = dilqr::fn##_##T##_g1(__VA_ARGS__); \
    if (rc_ == DILQR_EUNSUPPORTED) rc_ = dilqr::fn##_##T##_g2(__VA_ARGS__); \
    if (rc_ == DILQR_EUNSUPPORTED) rc_ = dilqr::fn##_##T##_g3(__VA_ARGS__); \
    return rc_;                                                  \
  } while (0)
#define BY_DTYPE_GROUPS(dtype, fn, ...)                          \
  do {                                                           \
    if ((dtype) == DILQR_F32) TRY_GROUPS(f32, fn, __VA_ARGS__);  \
    if ((dtype) == DILQR_F64) TRY_GROUPS(f64, fn, __VA_ARGS__);  \
    return DILQR_EINVAL;                                         \
  } while (0)

extern "C" {

const char* dilqr_version(void) { return "dilqr-b200 0.1 (sm_100a)"; }

int dilqr_supported(int dtype, int ns, int nc, int dyn) {
  if (dtype == DILQR_F32)
    return dilqr::supported_f32_g0(ns, nc, dyn) | dilqr::supported_f32_g1(ns, nc, dyn) |
           dilqr::supported_f32_g2(ns, nc, dyn) | dilqr::supported_f32_g3(ns, nc, dyn);
  if (dtype == DILQR_F64)
    return dilqr::supported_f64_g0(ns, nc, dyn) | dilqr::supported_f64_g1(ns, nc, dyn) |
           dilqr::supported_f64_g2(ns, nc, dyn) | dilqr::supported_f64_g3(ns, nc, dyn);
  return 0;
}

// the compiled kernels of a shape where they exist, else the runtime-dimension family
static int kernels_for(int dtype, int ns, int nc, int compiled, int runtime) {
  if ((dtype != DILQR_F32 && dtype != DILQR_F64) || ns <= 0 || nc <= 0) return DILQR_EINVAL;
  if (dilqr_supported(dtype, ns, nc, compiled)) return compiled;
  if (dilqr_supported(dtype, ns, nc, runtime)) return runtime;
  return DILQR_EUNSUPPORTED;
}

int dilqr_lindx_kernels(int dtype, int ns, int nc) {
  return kernels_for(dtype, ns, nc, DILQR_DYN_LINDX, DILQR_DYN_LINDX_RT);
}

int dilqr_nn_kernels(int dtype, int ns, int nc) {
  return kernels_for(dtype, ns, nc, DILQR_DYN_NN, DILQR_DYN_NN_RT);
}

int dilqr_mpc_plan(DilqrSolve* s) {
  if (!s) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(s->dtype, mpc_plan, s);
}

size_t dilqr_workspace_bytes(const DilqrSolve* s) {
  if (!s) return 0;
  return s->dtype == DILQR_F32 ? dilqr::workspace_bytes_f32_g0(s) : dilqr::workspace_bytes_f64_g0(s);
}

int dilqr_mpc_begin(const DilqrSolve* s, void* st) {
  if (!s) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(s->dtype, mpc_begin, s, st);
}
int dilqr_mpc_iterate(const DilqrSolve* s, void* st) {
  if (!s) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(s->dtype, mpc_iterate, s, st);
}
int dilqr_mpc_commit(const DilqrSolve* s, void* st) {
  if (!s) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(s->dtype, mpc_commit, s, st);
}
int dilqr_mpc_finish(const DilqrSolve* s, void* st) {
  if (!s) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(s->dtype, mpc_finish, s, st);
}
int dilqr_mpc_gains(const DilqrSolve* s, void* lam_blk, void* st) {
  if (!s) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(s->dtype, mpc_gains, s, lam_blk, st);
}
int dilqr_workspace_view(const DilqrSolve* s, DilqrWsView* v) {
  if (!s || !v) return DILQR_EINVAL;
  return ROUTE(s->dtype, dilqr::workspace_view_f32_g0(s, v), dilqr::workspace_view_f64_g0(s, v));
}
int dilqr_lam_tables(int dtype, int dyn, const double* dp, int T, int B, const void* x,
                     const void* u, const void* lam_blk, void* Lam, void* st) {
  return ROUTE(dtype, dilqr::lam_tables_f32_g0(dyn, dp, T, B, x, u, lam_blk, Lam, st),
               dilqr::lam_tables_f64_g0(dyn, dp, T, B, x, u, lam_blk, Lam, st));
}
int dilqr_sens_theta_adjoint(int dtype, int dyn, const double* dp, int T, int B, const void* x,
                             const void* u, const void* Kk, const void* lam_blk,
                             const void* dtau_blk, const void* df_blk, const void* Lam_packed,
                             void* dtheta, void* st) {
  return ROUTE(dtype,
               dilqr::sens_theta_adjoint_f32_g0(dyn, dp, T, B, x, u, Kk, lam_blk, dtau_blk, df_blk,
                                                Lam_packed, dtheta, st),
               dilqr::sens_theta_adjoint_f64_g0(dyn, dp, T, B, x, u, Kk, lam_blk, dtau_blk, df_blk,
                                                Lam_packed, dtheta, st));
}
size_t dilqr_adjoint_dtau_offset(const DilqrAdjoint* a) {
  if (!a) return 0;
  return a->dtype == DILQR_F32 ? dilqr::adjoint_dtau_offset_f32_g0(a)
                               : dilqr::adjoint_dtau_offset_f64_g0(a);
}
int dilqr_kkt_grads(const DilqrKkt* k, void* st) {
  if (!k) return DILQR_EINVAL;
  if (k->dynamics != DILQR_DYN_LINDX && k->dynamics != DILQR_DYN_LINDX_RT) return DILQR_EINVAL;
  BY_DTYPE_GROUPS(k->dtype, kkt_grads, k, st);
}
int dilqr_linearize(int dtype, int dyn, const double* dp, int T, int B, const void* x,
                    const void* u, void* F, void* f, void* st) {
  return ROUTE(dtype, dilqr::linearize_f32_g0(dyn, dp, T, B, x, u, F, f, st),
               dilqr::linearize_f64_g0(dyn, dp, T, B, x, u, F, f, st));
}
int dilqr_rollout(int dtype, int dyn, const double* dp, int T, int B, const void* x0,
                  const void* u, void* x, void* st) {
  return ROUTE(dtype, dilqr::rollout_f32_g0(dyn, dp, T, B, x0, u, x, st),
               dilqr::rollout_f64_g0(dyn, dp, T, B, x0, u, x, st));
}

int dilqr_costate_tables(int dtype, int dyn, const double* dp, int T, int B, const void* C,
                         const void* c, const void* x, const void* u, void* lam, void* Lam,
                         int C_bcast, int c_bcast, int packed, void* st) {
  return ROUTE(dtype,
               dilqr::costate_tables_f32_g0(dyn, dp, T, B, C, c, x, u, lam, Lam, C_bcast, c_bcast,
                                            packed, st),
               dilqr::costate_tables_f64_g0(dyn, dp, T, B, C, c, x, u, lam, Lam, C_bcast, c_bcast,
                                            packed, st));
}
int dilqr_lam_pack_size(int dynamics) { return dilqr::lam_pack_size_f64_g0(dynamics);
}
int dilqr_sens_theta(int dtype, int dyn, const double* dp, int T, int B, const void* x,
                     const void* u, const void* K, const void* lam, const void* dx,
                     const void* du, const void* df, void* dtheta, void* st) {
  return ROUTE(dtype, dilqr::sens_theta_f32_g0(dyn, dp, T, B, x, u, K, lam, dx, du, df, dtheta, st),
               dilqr::sens_theta_f64_g0(dyn, dp, T, B, x, u, K, lam, dx, du, df, dtheta, st));
}
int dilqr_richardson_update(int dtype, int ns, int nc, int T, int B, const void* g,
                            const void* Lam, const void* dx, const void* du, void* w, void* negw,
                            void* resid, void* st) {
  BY_DTYPE_GROUPS(dtype, richardson_update, ns, nc, T, B, g, Lam, dx, du, w, negw, resid, st);
}

int dilqr_env_tables(int dtype, int dyn, const double* dp, int n, const void* x, const void* u,
                     void* const* out, void* st) {
  return ROUTE(dtype, dilqr::env_tables_f32_g0(dyn, dp, n, x, u, out, st),
               dilqr::env_tables_f64_g0(dyn, dp, n, x, u, out, st));
}

int dilqr_pnqp(int dtype, int n, int B, const void* H, const void* q, const void* lower,
               const void* upper, const void* x_init, void* x, void* lu, int32_t* pivots, void* If,
               uint32_t* trace, int solo, DilqrStatus* status, void* st) {
  return ROUTE(dtype,
               dilqr::pnqp_f32_g0(n, B, H, q, lower, upper, x_init, x, lu, pivots, If, trace, solo, status, st),
               dilqr::pnqp_f64_g0(n, B, H, q, lower, upper, x_init, x, lu, pivots, If, trace, solo, status, st));
}

int dilqr_pnqp_kernels(int dtype, int n, int n_iter) {
  if ((dtype != DILQR_F32 && dtype != DILQR_F64) || n <= 0 || n_iter <= 0) return DILQR_EINVAL;
  // the sizes DILQR_SUFFIX(pnqp) (api.cu) instantiates, at their fixed budget
  const bool compiled = n == 1 || n == 2 || n == 3 || n == 4 || n == 6 || n == 8;
  if (compiled && n_iter == DILQR_PNQP_MAX_ITER) return DILQR_PNQP_COMPILED;
  if (n <= DILQR_PNQP_RT_MAX_N && n_iter <= DILQR_PNQP_RT_MAX_ITER) return DILQR_PNQP_RT;
  return DILQR_EUNSUPPORTED;
}

int dilqr_pnqp_rt(int dtype, int n, int n_iter, int B, const void* H, const void* q,
                  const void* lower, const void* upper, const void* x_init, void* x, void* lu,
                  int32_t* pivots, void* If, uint32_t* trace, int solo, DilqrStatus* status,
                  void* st) {
  return ROUTE(dtype,
               dilqr::pnqp_rt_f32_g0(n, n_iter, B, H, q, lower, upper, x_init, x, lu, pivots, If,
                                     trace, solo, status, st),
               dilqr::pnqp_rt_f64_g0(n, n_iter, B, H, q, lower, upper, x_init, x, lu, pivots, If,
                                     trace, solo, status, st));
}

size_t dilqr_adjoint_workspace_bytes(const DilqrAdjoint* a) {
  if (!a) return 0;
  return a->dtype == DILQR_F32 ? dilqr::adjoint_workspace_bytes_f32_g0(a)
                               : dilqr::adjoint_workspace_bytes_f64_g0(a);
}
int dilqr_adjoint_factor(const DilqrAdjoint* a, void* st) {
  if (!a) return DILQR_EINVAL;
  return ROUTE(a->dtype, dilqr::adjoint_run_f32_g0(a, 0, st), dilqr::adjoint_run_f64_g0(a, 0, st));
}
int dilqr_adjoint_pass(const DilqrAdjoint* a, void* st) {
  if (!a) return DILQR_EINVAL;
  return ROUTE(a->dtype, dilqr::adjoint_run_f32_g0(a, 1, st), dilqr::adjoint_run_f64_g0(a, 1, st));
}
int dilqr_adjoint_final(const DilqrAdjoint* a, void* st) {
  if (!a) return DILQR_EINVAL;
  return ROUTE(a->dtype, dilqr::adjoint_run_f32_g0(a, 2, st), dilqr::adjoint_run_f64_g0(a, 2, st));
}

size_t dilqr_krylov_workspace_bytes(const DilqrKrylov* k) {
  if (!k) return 0;
  return k->dtype == DILQR_F32 ? dilqr::krylov_workspace_bytes_f32_g0(k)
       : k->dtype == DILQR_F64 ? dilqr::krylov_workspace_bytes_f64_g0(k) : 0;
}
int dilqr_krylov_cycle_steps(const DilqrKrylov* k, int cycle) {
  if (!k || k->restart < 1 || k->max_iter < 1 || cycle < 0) return DILQR_EINVAL;
  const long long left = (long long)k->max_iter - (long long)cycle * k->restart;
  return left <= 0 ? 0 : (int)(left < k->restart ? left : k->restart);
}
int dilqr_krylov_start(const DilqrKrylov* k, void* st) {
  if (!k) return DILQR_EINVAL;
  return ROUTE(k->dtype, dilqr::krylov_run_f32_g0(k, 0, st), dilqr::krylov_run_f64_g0(k, 0, st));
}
int dilqr_krylov_arnoldi(const DilqrKrylov* k, void* st) {
  if (!k) return DILQR_EINVAL;
  return ROUTE(k->dtype, dilqr::krylov_run_f32_g0(k, 1, st), dilqr::krylov_run_f64_g0(k, 1, st));
}
int dilqr_krylov_update(const DilqrKrylov* k, void* st) {
  if (!k) return DILQR_EINVAL;
  return ROUTE(k->dtype, dilqr::krylov_run_f32_g0(k, 2, st), dilqr::krylov_run_f64_g0(k, 2, st));
}
int dilqr_krylov_restart(const DilqrKrylov* k, void* st) {
  if (!k) return DILQR_EINVAL;
  return ROUTE(k->dtype, dilqr::krylov_run_f32_g0(k, 3, st), dilqr::krylov_run_f64_g0(k, 3, st));
}

}  // extern "C"
