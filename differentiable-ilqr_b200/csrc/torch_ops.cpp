// torch_ops.cpp -- TORCH_LIBRARY(dilqr, ...): the hot path as dispatcher-visible torch
// custom ops, a THIN layer over the C ABI of include/dilqr.h (every kernel launch below is
// a libdilqr entry point; torch supplies device memory, the current stream and autograd).
//
//   torch.ops.dilqr.mpc_solve       MPC.forward            mpc.py:184-337, mpc_explicit.py:182-358
//   torch.ops.dilqr.dilqr_backward  LQRStepFn.backward     lqr_step_explicit.py:652-712
//   torch.ops.dilqr.lqr_kkt_backward  LQRStepFn.backward   lqr_step.py:312-407 (LinDx problems)
//
// The call sites they serve in the reference: il_env.py:174-187 (IL_Env.mpc builds
// mpc_explicit.MPC(...)(xinit, QuadCost(Q, p), dx)) and mpc.py:339-361 (solve_lqr_subproblem).
// Autograd formulas are registered from Python (torch_ops.py) on top of these ops.
#include <ATen/ATen.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <cstring>
#include <tuple>
#include <vector>

#include "../../include/dilqr.h"

namespace {

using at::Tensor;
using c10::optional;

int dtype_of(const Tensor& t) {
  TORCH_CHECK(t.scalar_type() == at::kFloat || t.scalar_type() == at::kDouble,
              "dilqr: float32 / float64 tensors only");
  return t.scalar_type() == at::kDouble ? DILQR_F64 : DILQR_F32;
}

void check_rc(int rc, const char* what) {
  TORCH_CHECK(rc == DILQR_OK, "dilqr: ", what, " failed with code ", rc,
              rc == DILQR_EUNSUPPORTED ? " (shape not compiled in: see DILQR_CONFIGS in csrc/api.cu)" : "");
}

// cost layouts of mpc.py:205-219: [n,n] / [T,n,n] / [T,B,n,n]
int cost_mode(const Tensor& C, int64_t tail) {
  if (C.dim() == tail) return 2;
  if (C.dim() == tail + 1) return 1;
  TORCH_CHECK(C.dim() == tail + 2, "dilqr: unexpected cost shape");
  return 0;
}

void host_theta(const Tensor& theta, double* out) {
  Tensor h = theta.detach().to(at::kCPU, at::kDouble).contiguous();
  TORCH_CHECK(h.numel() <= 8, "dilqr: at most 8 dynamics parameters");
  for (int i = 0; i < 8; ++i) out[i] = i < h.numel() ? h.data_ptr<double>()[i] : 0.0;
}

struct Problem {
  DilqrSolve s;
  std::vector<Tensor> keep;
  Tensor ws, pipe, pipe_host;
};

// Fill a DilqrSolve for (x_init, C, c, dynamics) -- the argument handling of MPC.forward.
void make_problem(Problem& P, const Tensor& x_init, const Tensor& C, const Tensor& c,
                  const optional<Tensor>& F, const optional<Tensor>& f,
                  const optional<Tensor>& u_init, const Tensor& theta, int64_t dynamics, int64_t T,
                  optional<double> u_lower, optional<double> u_upper, int64_t max_ls, double decay,
                  double best_cost_eps, int64_t solo, int64_t max_iters) {
  DilqrSolve& s = P.s;
  std::memset(&s, 0, sizeof(s));
  TORCH_CHECK(x_init.is_cuda() && C.is_cuda() && c.is_cuda(), "dilqr: CUDA tensors only (no CPU path)");
  TORCH_CHECK(x_init.dim() == 2, "dilqr: x_init must be [B, n_state]");
  const auto dt = x_init.scalar_type();
  auto own = [&](const Tensor& t) {
    Tensor r = t.detach().to(dt).contiguous();
    P.keep.push_back(r);
    return r.data_ptr();
  };
  s.n_batch = (int)x_init.size(0);
  s.n_state = (int)x_init.size(1);
  s.n_ctrl = (int)C.size(-1) - s.n_state;
  s.T = (int)T;
  s.dtype = dtype_of(x_init);
  s.dynamics = (int)dynamics;
  if (dynamics == DILQR_DYN_LINDX) {   // the library picks compiled or runtime-dimension kernels
    s.dynamics = dilqr_lindx_kernels(s.dtype, s.n_state, s.n_ctrl);
    TORCH_CHECK(s.dynamics != DILQR_EUNSUPPORTED, "dilqr: LinDx n_state=", s.n_state, " n_ctrl=",
                s.n_ctrl, " is not supported: at most 32 variables (n_state + n_ctrl)");
    check_rc(s.dynamics < 0 ? s.dynamics : 0, "dilqr_lindx_kernels");
  }
  s.gain_solve = DILQR_GAIN_PLAIN;
  s.solo = (int)solo;
  s.max_linesearch_iter = (int)max_ls;
  s.linesearch_decay = decay;
  s.best_cost_eps = best_cost_eps;
  s.C_bcast = cost_mode(C, 2);
  s.c_bcast = cost_mode(c, 1);
  s.x_init = own(x_init);
  s.C = own(C);
  s.c = own(c);
  if (dynamics == DILQR_DYN_LINDX) {
    TORCH_CHECK(F.has_value(), "dilqr: LinDx needs F");
    s.F = own(*F);
    if (f.has_value() && f->numel() > 0) {
      s.f = own(*f);
      s.has_f = 1;
    }
  } else {
    host_theta(theta, s.dyn_params);
  }
  if (u_init.has_value()) {
    Tensor u0 = *u_init;
    if (u0.dim() == 2) u0 = u0.unsqueeze(1).expand({T, s.n_batch, s.n_ctrl});
    s.u_init = own(u0);
  }
  if (u_lower.has_value()) {
    TORCH_CHECK(u_upper.has_value(), "dilqr: u_lower and u_upper come together (mpc.py:146)");
    s.bounds_kind = DILQR_BOUNDS_SCALAR;
    s.u_lower = *u_lower;
    s.u_upper = *u_upper;
  }
  const int rc = dilqr_mpc_plan(&s);   // the library chooses how pnqp's decisions are resolved
  TORCH_CHECK(rc != DILQR_EUNSUPPORTED, "dilqr: no kernel compiled for n_state=", s.n_state,
              " n_ctrl=", s.n_ctrl, " dynamics=", s.dynamics);
  check_rc(rc, "dilqr_mpc_plan");
  auto bytes = at::TensorOptions().dtype(at::kByte).device(x_init.device());
  P.ws = at::empty({(int64_t)dilqr_workspace_bytes(&s)}, bytes);
  P.pipe = at::zeros({64 * (1 + max_iters)}, bytes);
  P.pipe_host = at::empty({64 * (1 + max_iters)}, at::TensorOptions().dtype(at::kByte).pinned_memory(true));
  s.workspace = P.ws.data_ptr();
  s.workspace_bytes = (size_t)P.ws.numel();
}

// iLQR outer loop with the stop rule on the device (DilqrControl): all iterations enqueued
// back to back, one host sync; a wrong pnqp trace guess halts the queue and is re-enqueued.
int64_t run_iterations(Problem& P, int64_t n_loops, double eps, int64_t not_improved_lim,
                       cudaStream_t st, std::vector<int64_t>* qp_iters) {
  DilqrSolve& s = P.s;
  DilqrControl ctl;
  std::memset(&ctl, 0, sizeof(ctl));
  ctl.eps = s.dtype == DILQR_F32 ? (double)(float)eps : eps;   // python float vs tensor dtype (mpc.py:299)
  ctl.not_improved_lim = (uint32_t)not_improved_lim;
  char* base = static_cast<char*>(P.pipe.data_ptr());
  std::memcpy(P.pipe_host.data_ptr(), &ctl, sizeof(ctl));
  C10_CUDA_CHECK(cudaMemcpyAsync(base, P.pipe_host.data_ptr(), 64, cudaMemcpyHostToDevice, st));
  s.control = reinterpret_cast<DilqrControl*>(base);
  int64_t start = 0;
  const size_t nbytes = 64 * (1 + n_loops);
  DilqrControl got;
  for (int attempt = 0; attempt < 256; ++attempt) {
    for (int64_t j = start; j < n_loops; ++j) {
      s.iteration = (int)j;
      s.status = reinterpret_cast<DilqrStatus*>(base + 64 * (1 + j));
      check_rc(dilqr_mpc_iterate(&s, st), "dilqr_mpc_iterate");
      check_rc(dilqr_mpc_commit(&s, st), "dilqr_mpc_commit");
    }
    C10_CUDA_CHECK(cudaMemcpyAsync(P.pipe_host.data_ptr(), base, nbytes, cudaMemcpyDeviceToHost, st));
    C10_CUDA_CHECK(cudaStreamSynchronize(st));
    std::memcpy(&got, P.pipe_host.data_ptr(), sizeof(got));
    if (got.halt != 2) break;
    start = got.iters_done;            // trace mismatch: redo that iteration (guess corrected)
    C10_CUDA_CHECK(cudaMemsetAsync(base, 0, 4, st));
    TORCH_CHECK(attempt < 255, "dilqr: pnqp control-flow trace did not stabilise");
  }
  if (qp_iters) {
    const char* h = static_cast<const char*>(P.pipe_host.data_ptr());
    for (uint32_t j = 0; j < got.iters_done; ++j) {
      DilqrStatus stt;
      std::memcpy(&stt, h + 64 * (1 + j), sizeof(stt));
      qp_iters->push_back(stt.n_total_qp_iter);
    }
  }
  s.iteration = (int)got.iters_done - 1;
  s.control = nullptr;
  s.status = reinterpret_cast<DilqrStatus*>(base + 64);
  return got.iters_done;
}

// ------------------------------------------------------------------ mpc_solve
std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor> mpc_solve(
    const Tensor& x_init, const Tensor& C, const Tensor& c, const optional<Tensor>& F,
    const optional<Tensor>& f, const optional<Tensor>& u_init, const Tensor& theta, int64_t dynamics,
    int64_t T, optional<double> u_lower, optional<double> u_upper, int64_t lqr_iter, double eps,
    double linesearch_decay, int64_t max_linesearch_iter, int64_t not_improved_lim,
    double best_cost_eps, int64_t solo) {
  c10::cuda::CUDAGuard guard(x_init.device());
  cudaStream_t st = c10::cuda::getCurrentCUDAStream();
  Problem P;
  make_problem(P, x_init, C, c, F, f, u_init, theta, dynamics, T, u_lower, u_upper,
               max_linesearch_iter, linesearch_decay, best_cost_eps, solo, lqr_iter);
  DilqrSolve& s = P.s;
  s.status = reinterpret_cast<DilqrStatus*>(static_cast<char*>(P.pipe.data_ptr()) + 64);
  check_rc(dilqr_mpc_begin(&s, st), "dilqr_mpc_begin");
  std::vector<int64_t> qp;
  run_iterations(P, lqr_iter, eps, not_improved_lim, st, &qp);
  auto opt = x_init.options();
  Tensor x = at::empty({T, s.n_batch, s.n_state}, opt), u = at::empty({T, s.n_batch, s.n_ctrl}, opt);
  Tensor costs = at::empty({s.n_batch}, opt), du = at::empty({s.n_batch}, opt);
  s.x_out = x.data_ptr();
  s.u_out = u.data_ptr();
  s.cost_out = costs.data_ptr();
  s.du_out = du.data_ptr();
  check_rc(dilqr_mpc_finish(&s, st), "dilqr_mpc_finish");
  // n_total_qp_iter of every iteration that ran, -1 for the ones the stop rule skipped
  Tensor qpt = at::full({lqr_iter}, -1, at::kLong);
  for (size_t i = 0; i < qp.size() && (int64_t)i < lqr_iter; ++i) qpt.data_ptr<int64_t>()[i] = qp[i];
  return {x, u, costs, du, qpt};
}

// ------------------------------------------------------------------ KKT backward (LinDx)
// LQRStepFn.backward (lqr_step.py:312-407): adjoint LQR solve on (C, -r, LinDx(F), u_zero_I =
// active set), then the costate recursions and outer products.
std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor> lqr_kkt_backward(
    const optional<Tensor>& gx, const Tensor& gu, const Tensor& x_init, const Tensor& C,
    const Tensor& c, const Tensor& F, const Tensor& x, const Tensor& u, optional<double> u_lower,
    optional<double> u_upper) {
  c10::cuda::CUDAGuard guard(x.device());
  cudaStream_t st = c10::cuda::getCurrentCUDAStream();
  const int64_t T = x.size(0), B = x.size(1), ns = x.size(2), nc = u.size(2), n = ns + nc;
  Tensor gxx = gx.has_value() ? *gx : at::zeros_like(x);
  Tensor r = at::cat({gxx, gu}, 2).contiguous();
  Tensor negr = r.neg();
  Tensor Cd = C.detach().expand({T, B, n, n}).contiguous(), cd = c.detach().expand({T, B, n}).contiguous();
  Tensor zero = at::zeros_like(x_init);
  Problem P;
  make_problem(P, zero, Cd, negr, F, c10::nullopt, c10::nullopt, zero, DILQR_DYN_LINDX, T,
               c10::nullopt, c10::nullopt, 10, 0.2, 1e-4, 0, 1);
  DilqrSolve& s = P.s;
  Tensor I;
  if (u_lower.has_value()) {     // lqr_step.py:325-326
    I = ((u - *u_lower).abs().le(1e-8)).logical_or((u - *u_upper).abs().le(1e-8)).to(at::kByte).contiguous();
    s.u_zero_I = I.data_ptr<uint8_t>();
  }
  s.status = reinterpret_cast<DilqrStatus*>(static_cast<char*>(P.pipe.data_ptr()) + 64);
  check_rc(dilqr_mpc_begin(&s, st), "dilqr_mpc_begin");
  s.iteration = 0;
  check_rc(dilqr_mpc_iterate(&s, st), "dilqr_mpc_iterate");
  check_rc(dilqr_mpc_commit(&s, st), "dilqr_mpc_commit");
  auto opt = x.options();
  Tensor dx = at::empty({T, B, ns}, opt), du = at::empty({T, B, nc}, opt), cst = at::empty({B}, opt),
         dun = at::empty({B}, opt);
  s.x_out = dx.data_ptr();
  s.u_out = du.data_ptr();
  s.cost_out = cst.data_ptr();
  s.du_out = dun.data_ptr();
  check_rc(dilqr_mpc_finish(&s, st), "dilqr_mpc_finish");
  DilqrKkt k;
  std::memset(&k, 0, sizeof(k));
  k.n_state = (int)ns; k.n_ctrl = (int)nc; k.T = (int)T; k.n_batch = (int)B; k.dtype = dtype_of(x);
  k.dynamics = s.dynamics;   // the kernels make_problem chose for this shape (dilqr_lindx_kernels)
  Tensor Fc = F.detach().contiguous(), xc = x.detach().contiguous(), uc = u.detach().contiguous();
  k.C = Cd.data_ptr(); k.c = cd.data_ptr(); k.F = Fc.data_ptr(); k.x = xc.data_ptr(); k.u = uc.data_ptr();
  k.dx = dx.data_ptr(); k.du = du.data_ptr(); k.r = r.data_ptr();
  Tensor dC = at::empty({T, B, n, n}, opt), dc = at::empty({T, B, n}, opt),
         dF = at::empty({T - 1, B, ns, n}, opt), df = at::empty({T - 1, B, ns}, opt),
         dx0 = at::empty({B, ns}, opt);
  k.dC = dC.data_ptr(); k.dc = dc.data_ptr(); k.dF = dF.data_ptr(); k.df = df.data_ptr();
  k.dx_init = dx0.data_ptr();
  check_rc(dilqr_kkt_grads(&k, st), "dilqr_kkt_grads");
  return {dx0, dC, dc, dF, df};
}

// ------------------------------------------------------------------ DiLQR implicit backward
// (dC, dc, dtheta[B, n_theta]) at a solution (x, u) of an env_dx problem: gains of the final
// no-op LQR pass, costates + second-order tables, factored adjoint solves (n_passes
// Richardson passes + the final one), closed-loop sensitivity rollout.
std::tuple<Tensor, Tensor, Tensor> dilqr_backward(
    const optional<Tensor>& gx, const Tensor& gu, const Tensor& x_init, const Tensor& C,
    const Tensor& c, const Tensor& x, const Tensor& u, const Tensor& theta, int64_t dynamics,
    optional<double> u_lower, optional<double> u_upper, int64_t n_passes, int64_t max_ls,
    double decay) {
  c10::cuda::CUDAGuard guard(x.device());
  cudaStream_t st = c10::cuda::getCurrentCUDAStream();
  TORCH_CHECK(dynamics == DILQR_DYN_PENDULUM || dynamics == DILQR_DYN_CARTPOLE,
              "dilqr::dilqr_backward: factored adjoint kernels exist for pendulum / cartpole; use "
              "the Python mpc_explicit.MPC for other models");
  const int64_t T = x.size(0), B = x.size(1), ns = x.size(2), nc = u.size(2), n = ns + nc;
  auto opt = x.options();
  const int dt = dtype_of(x);
  Tensor xc = x.detach().contiguous(), uc = u.detach().contiguous();
  // (1) gains of the final LQR pass at tau* (lqr_step_explicit.py:604-618): one LQR step
  Problem P;
  make_problem(P, x_init, C, c, c10::nullopt, c10::nullopt, uc, theta, dynamics, T, u_lower, u_upper,
               1, decay, 1e-4, 0, 1);
  (void)max_ls;
  DilqrSolve& s = P.s;
  s.x_cur = xc.data_ptr();
  s.gains_only = 1;
  char* base = static_cast<char*>(P.pipe.data_ptr());
  s.status = reinterpret_cast<DilqrStatus*>(base + 64);
  check_rc(dilqr_mpc_begin(&s, st), "dilqr_mpc_begin");
  s.iteration = 0;
  for (int attempt = 0;; ++attempt) {
    check_rc(dilqr_mpc_iterate(&s, st), "dilqr_mpc_iterate");
    check_rc(dilqr_mpc_commit(&s, st), "dilqr_mpc_commit");
    C10_CUDA_CHECK(cudaMemcpyAsync(P.pipe_host.data_ptr(), base + 64, 64, cudaMemcpyDeviceToHost, st));
    C10_CUDA_CHECK(cudaStreamSynchronize(st));
    DilqrStatus stt;
    std::memcpy(&stt, P.pipe_host.data_ptr(), sizeof(stt));
    if (stt.trace_match) break;
    TORCH_CHECK(attempt < 64, "dilqr: pnqp control-flow trace did not stabilise");
  }
  Tensor K = at::empty({T, B, nc, ns}, opt), kk = at::empty({T, B, nc}, opt);
  s.K_out = K.data_ptr();
  s.k_out = kk.data_ptr();
  check_rc(dilqr_mpc_finish(&s, st), "dilqr_mpc_finish");
  // (2) costates + packed second-order tables
  double th[8];
  host_theta(theta, th);
  const int64_t nW = (B + 31) / 32;
  Tensor lam = at::empty({T, B, ns}, opt);
  Tensor Lam = at::empty({T - 1, nW, (int64_t)dilqr_lam_pack_size((int)dynamics), 32}, opt);
  Tensor Cc = C.detach().contiguous(), cc = c.detach().contiguous();
  const int Cb = cost_mode(C, 2), cb = cost_mode(c, 1);
  check_rc(dilqr_costate_tables(dt, (int)dynamics, th, (int)T, (int)B, Cc.data_ptr(), cc.data_ptr(),
                                xc.data_ptr(), uc.data_ptr(), lam.data_ptr(), Lam.data_ptr(), Cb, cb, 1,
                                st),
           "dilqr_costate_tables");
  // (3) factored adjoint solves
  DilqrAdjoint a;
  std::memset(&a, 0, sizeof(a));
  a.n_state = (int)ns; a.n_ctrl = (int)nc; a.T = (int)T; a.n_batch = (int)B; a.dtype = dt;
  a.dynamics = (int)dynamics;
  a.bounds_kind = u_lower.has_value() ? DILQR_BOUNDS_SCALAR : DILQR_BOUNDS_NONE;
  a.gain_solve = DILQR_GAIN_CHOL_REG;
  a.C_bcast = Cb; a.c_bcast = cb;
  if (u_lower.has_value()) { a.u_lower = *u_lower; a.u_upper = *u_upper; }
  for (int i = 0; i < 8; ++i) a.dyn_params[i] = th[i];
  Tensor resid = at::zeros({3}, opt.dtype(at::kDouble));
  Tensor guc = gu.detach().to(x.scalar_type()).contiguous(), gxc;
  if (gx.has_value()) gxc = gx->detach().to(x.scalar_type()).contiguous();
  Tensor w = at::empty({T, B, n}, opt);
  a.C = Cc.data_ptr(); a.x = xc.data_ptr(); a.u = uc.data_ptr(); a.Lam = Lam.data_ptr();
  a.gx = gx.has_value() ? gxc.data_ptr() : nullptr;
  a.gu = guc.data_ptr();
  a.w = w.data_ptr();
  a.resid = resid.data_ptr();
  Tensor aws = at::empty({(int64_t)dilqr_adjoint_workspace_bytes(&a)}, opt.dtype(at::kByte));
  a.workspace = aws.data_ptr();
  a.workspace_bytes = (size_t)aws.numel();
  check_rc(dilqr_adjoint_factor(&a, st), "dilqr_adjoint_factor");
  for (int64_t i = 0; i < n_passes; ++i) {
    a.first_pass = i == 0;
    check_rc(dilqr_adjoint_pass(&a, st), "dilqr_adjoint_pass");
  }
  a.first_pass = n_passes == 0;
  const std::vector<int64_t> shC = Cb == 0 ? std::vector<int64_t>{T, B, n, n}
                                 : Cb == 1 ? std::vector<int64_t>{T, nW, n, n} : std::vector<int64_t>{nW, n, n};
  const std::vector<int64_t> shc = cb == 0 ? std::vector<int64_t>{T, B, n}
                                 : cb == 1 ? std::vector<int64_t>{T, nW, n} : std::vector<int64_t>{nW, n};
  Tensor dC = at::empty(shC, opt), dc = at::empty(shc, opt), df = at::empty({T - 1, B, ns}, opt),
         dxa = at::empty({T, B, ns}, opt), dua = at::empty({T, B, nc}, opt);
  a.dC = dC.data_ptr(); a.dc = dc.data_ptr(); a.df = df.data_ptr();
  a.dx_out = dxa.data_ptr(); a.du_out = dua.data_ptr();
  check_rc(dilqr_adjoint_final(&a, st), "dilqr_adjoint_final");
  // (4) dtheta through the closed-loop sensitivity rollout
  Tensor dtheta = at::empty({B, theta.numel()}, opt);
  check_rc(dilqr_sens_theta(dt, (int)dynamics, th, (int)T, (int)B, xc.data_ptr(), uc.data_ptr(),
                            K.data_ptr(), lam.data_ptr(), dxa.data_ptr(), dua.data_ptr(), df.data_ptr(),
                            dtheta.data_ptr(), st),
           "dilqr_sens_theta");
  Tensor rh = resid.cpu();
  int64_t n_rej;
  std::memcpy(&n_rej, rh.data_ptr<double>() + 2, sizeof(n_rej));
  TORCH_CHECK(n_rej == 0, "dilqr::dilqr_backward: the reference's line search would reject an adjoint "
                          "step for ", n_rej, " problem(s) (non-convex model); use the Python "
                          "mpc_explicit.MPC, which falls back to the line-searching kernels");
  if (Cb) dC = dC.sum(Cb == 1 ? 1 : 0);
  if (cb) dc = dc.sum(cb == 1 ? 1 : 0);
  return {dC, dc, dtheta};
}

}  // namespace

TORCH_LIBRARY(dilqr, m) {
  m.def("mpc_solve(Tensor x_init, Tensor C, Tensor c, Tensor? F, Tensor? f, Tensor? u_init, "
        "Tensor theta, int dynamics, int T, float? u_lower, float? u_upper, int lqr_iter, float eps, "
        "float linesearch_decay, int max_linesearch_iter, int not_improved_lim, float best_cost_eps, "
        "int solo) -> (Tensor, Tensor, Tensor, Tensor, Tensor)");
  m.def("dilqr_backward(Tensor? gx, Tensor gu, Tensor x_init, Tensor C, Tensor c, Tensor x, Tensor u, "
        "Tensor theta, int dynamics, float? u_lower, float? u_upper, int n_passes, "
        "int max_linesearch_iter, float linesearch_decay) -> (Tensor, Tensor, Tensor)");
  m.def("lqr_kkt_backward(Tensor? gx, Tensor gu, Tensor x_init, Tensor C, Tensor c, Tensor F, Tensor x, "
        "Tensor u, float? u_lower, float? u_upper) -> (Tensor, Tensor, Tensor, Tensor, Tensor)");
}

TORCH_LIBRARY_IMPL(dilqr, CUDA, m) {
  m.impl("mpc_solve", &mpc_solve);
  m.impl("dilqr_backward", &dilqr_backward);
  m.impl("lqr_kkt_backward", &lqr_kkt_backward);
}
