// api.cu -- extern "C" entry points of libdilqr (see include/dilqr.h).
// Compiled once per scalar type (-DDILQR_SCALAR_F64=0/1) into separate objects;
// dispatch.cu routes on DilqrSolve::dtype.
#include <cuda_runtime.h>
#include <atomic>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/dilqr.h"
#include "ilqr_kernels.cuh"
#include "misc_kernels.cuh"
#include "dilqr_backward.cuh"
#include "adjoint_kernels.cuh"
#include "group_kernels.cuh"
#include "rt_kernels.cuh"
#if !defined(DILQR_GROUP) || DILQR_GROUP == 0
#include "pnqp_rt.cuh"
#endif

namespace dilqr {

// Compiled once per (scalar type, shape group): -DDILQR_SCALAR_F64=0/1 -DDILQR_GROUP=0..3.
// The shape-specialised kernels are split over four groups purely to parallelise the
// build; group 0 also carries every entry point that does not depend on (ns, nc).
#ifndef DILQR_GROUP
#define DILQR_GROUP 0
#endif
#define DILQR_PASTE2(a, b, c) a##_##b##_g##c
#define DILQR_PASTE(a, b, c) DILQR_PASTE2(a, b, c)
#if DILQR_SCALAR_F64
using Scalar = double;
#define DILQR_SUFFIX(name) DILQR_PASTE(name, f64, DILQR_GROUP)
#else
using Scalar = float;
#define DILQR_SUFFIX(name) DILQR_PASTE(name, f32, DILQR_GROUP)
#endif

// (n_state, n_ctrl, dynamics) combinations compiled into this group.
#ifdef DILQR_FAST_BUILD   // developer builds: a handful of shapes, all in group 0
#if DILQR_GROUP == 0
#define DILQR_CONFIGS(X)       \
  X(3, 1, DYN_LINDX)           \
  X(4, 2, DYN_LINDX)           \
  X(5, 1, DYN_LINDX)           \
  X(6, 2, DYN_LINDX)           \
  X(13, 3, DYN_LINDX)          \
  X(3, 1, DYN_PENDULUM)        \
  X(5, 1, DYN_CARTPOLE)        \
  X(13, 3, DYN_ROCKET)         \
  X(3, 1, DYN_NN)
#else
#define DILQR_CONFIGS(X)
#endif
#elif DILQR_GROUP == 0
#define DILQR_CONFIGS(X)       \
  X(3, 1, DYN_LINDX)           \
  X(5, 1, DYN_LINDX)           \
  X(3, 1, DYN_PENDULUM)        \
  X(5, 1, DYN_CARTPOLE)        \
  X(13, 3, DYN_ROCKET)
#elif DILQR_GROUP == 1
#define DILQR_CONFIGS(X)       \
  X(2, 1, DYN_LINDX)           \
  X(2, 2, DYN_LINDX)           \
  X(6, 2, DYN_LINDX)           \
  X(4, 1, DYN_LINDX)           \
  X(4, 2, DYN_LINDX)           \
  X(4, 4, DYN_LINDX)           \
  X(8, 1, DYN_LINDX)           \
  X(8, 2, DYN_LINDX)
#elif DILQR_GROUP == 2
#define DILQR_CONFIGS(X)       \
  X(8, 4, DYN_LINDX)           \
  X(13, 3, DYN_LINDX)          \
  X(16, 1, DYN_LINDX)
#else
#define DILQR_CONFIGS(X)       \
  X(16, 2, DYN_LINDX)          \
  X(16, 4, DYN_LINDX)          \
  X(3, 1, DYN_NN)              \
  X(4, 2, DYN_NN)              \
  X(5, 1, DYN_NN)
#endif

constexpr size_t kStageBudget = 56 * 1024;  // per-warp staging budget (>= 4 warps / SM)

template <class S, int NS, int NC, int DYN>
constexpr bool staged_v() {
  constexpr int N = NS + NC;
  constexpr bool env = DYN != DYN_LINDX;
  size_t per = (size_t)kWarp * sizeof(S) * (N * N + N + (env ? 0 : NS * N + NS));
  return per * kStages <= kStageBudget;
}

}  // namespace dilqr
extern "C" int g_dilqr_iterate_launches;   // dispatch.cu: kernels of the last dilqr_mpc_iterate
namespace dilqr {
#define g_iterate_launches g_dilqr_iterate_launches

// shapes whose sweeps exist in a symmetric-Riccati form next to the general one
template <class S, int NS, int NC, int DYN>
constexpr bool sym_pair_v() {
  return kSymRiccatiOn && kChainFmaOn && staged_v<S, NS, NC, DYN>() &&
         (DYN == DYN_PENDULUM || DYN == DYN_CARTPOLE);
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct WsLayout {
  size_t traj[2], best, Kk, cost_cur, cost_new, cost_best, du_new, du_best, alpha_new, dusq, take,
      guess, votes, guess_gains, cpk_state, gs_barrier, commit_ticket, commit_part, Cpk, gsQ, gsG, total;
  int Bp;
};

static WsLayout ws_layout(const DilqrSolve* s, size_t esz) {
  WsLayout w;
  const int N = s->n_state + s->n_ctrl;
  const int NK = s->n_ctrl * s->n_state + s->n_ctrl;
  w.Bp = (int)align_up((size_t)s->n_batch, 32);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  w.traj[0] = take((size_t)s->T * N * w.Bp * esz);
  w.traj[1] = take((size_t)s->T * N * w.Bp * esz);
  w.best = take((size_t)s->T * N * w.Bp * esz);
  w.Kk = take((size_t)s->T * NK * w.Bp * esz);
  w.cost_cur = take((size_t)w.Bp * esz);
  w.cost_new = take((size_t)w.Bp * esz);
  w.cost_best = take((size_t)w.Bp * esz);
  w.du_new = take((size_t)w.Bp * esz);
  w.du_best = take((size_t)w.Bp * esz);
  w.alpha_new = take((size_t)w.Bp * esz);
  w.dusq = take((size_t)s->T * s->n_ctrl * w.Bp * esz);
  w.take = take((size_t)w.Bp * sizeof(int));
  w.guess = take((size_t)s->T * kPnqpMaxIter * sizeof(uint32_t));
  w.votes = take((size_t)s->T * kPnqpMaxIter * sizeof(uint32_t));
  w.guess_gains = take((size_t)s->T * kPnqpMaxIter * sizeof(uint32_t));
  w.cpk_state = take(sizeof(uint32_t));
  w.gs_barrier = take(sizeof(uint32_t));
  w.commit_ticket = take(sizeof(uint32_t));
  w.commit_part = take((size_t)((w.Bp + 127) / 128) * sizeof(CommitPart));
  // packed symmetric copy of C: only shapes whose sweeps are staged use it (staged_v)
  {
    const bool env = s->dynamics != DILQR_DYN_LINDX;
    const size_t per = (size_t)kWarp * esz *
                       ((size_t)N * N + N + (env ? 0 : (size_t)s->n_state * N + s->n_state));
    const bool staged = per * kStages <= kStageBudget;
    (void)staged;   // every shape keeps the packed copy (staged: TMA chunks; else: coalesced reads)
    w.Cpk = take(!s->C_bcast ? (size_t)s->T * w.Bp * (N * (N + 1) / 2) * esz : 0);
  }
  // group sweep: one Q_t / q_t record per problem
  w.gsQ = take(s->group_sweep ? (size_t)w.Bp * ((size_t)N * N + N) * esz : 0);
  w.gsG = take(s->group_sweep ? (size_t)w.Bp * ((size_t)s->n_ctrl * N + s->n_ctrl) * esz : 0);
  w.total = off;
  return w;
}

// `role`: 0 = begin (writes the current iterate), 1 = iterate / commit / finish of
// iLQR iteration s->iteration (reads buffer it&1, writes buffer (it+1)&1).
static IterParams<Scalar> make_params(const DilqrSolve* s, int role = 1) {
  using S = Scalar;
  IterParams<S> p;
  memset(&p, 0, sizeof(p));
  const WsLayout w = ws_layout(s, sizeof(S));
  char* ws = static_cast<char*>(s->workspace);
  p.T = s->T;
  p.B = s->n_batch;
  p.Bp = w.Bp;
  p.bounds_kind = s->bounds_kind;
  p.solo = s->solo;
  p.gain_solve = s->gain_solve;
  p.max_ls = s->max_linesearch_iter;
  p.has_f = s->has_f && s->f != nullptr;
  p.first_iteration = s->iteration == 0;
  p.nW = w.Bp / 32;
  p.lo = (S)s->u_lower;
  p.hi = (S)s->u_upper;
  p.decay = (S)s->linesearch_decay;
  p.delta_u = (S)s->delta_u;
  p.has_delta = s->has_delta_u && s->bounds_kind != DILQR_BOUNDS_NONE;
  p.best_cost_eps = (S)s->best_cost_eps;
  p.lo_t = static_cast<const S*>(s->u_lower_t);
  p.hi_t = static_cast<const S*>(s->u_upper_t);
  p.zeroI = s->u_zero_I;
  p.x_init = static_cast<const S*>(s->x_init);
  p.C = static_cast<const S*>(s->C);
  p.c = static_cast<const S*>(s->c);
  p.F = static_cast<const S*>(s->F);
  p.f = static_cast<const S*>(s->f);
  p.u_init = static_cast<const S*>(s->u_init);
  p.x_cur = static_cast<const S*>(s->x_cur);
  {
    const int cur = role == 0 ? 1 : (s->iteration & 1);   // begin "writes new" = buffer 0
    p.traj_cur = reinterpret_cast<const S*>(ws + w.traj[cur]);
    p.traj_new = reinterpret_cast<S*>(ws + w.traj[cur ^ 1]);
    p.traj_best = reinterpret_cast<S*>(ws + w.best);
    p.traj_buf[0] = reinterpret_cast<S*>(ws + w.traj[0]);
    p.traj_buf[1] = reinterpret_cast<S*>(ws + w.traj[1]);
  }
  p.Kk = reinterpret_cast<S*>(ws + w.Kk);
  p.cost_cur = reinterpret_cast<S*>(ws + w.cost_cur);
  p.cost_new = reinterpret_cast<S*>(ws + w.cost_new);
  p.cost_best = reinterpret_cast<S*>(ws + w.cost_best);
  p.du_new = reinterpret_cast<S*>(ws + w.du_new);
  p.du_best = reinterpret_cast<S*>(ws + w.du_best);
  p.alpha_new = reinterpret_cast<S*>(ws + w.alpha_new);
  p.dusq = reinterpret_cast<S*>(ws + w.dusq);
  p.take = reinterpret_cast<int*>(ws + w.take);
  p.cpk_state = reinterpret_cast<uint32_t*>(ws + w.cpk_state);
  p.Cpk = reinterpret_cast<S*>(ws + w.Cpk);
  p.gains_only = s->gains_only;
  p.C_bcast = s->C_bcast;
  p.c_bcast = s->c_bcast;
  p.votes_are_trace = s->group_sweep;   // the group sweep decides at barriers: nothing to replay
  p.gsQ = reinterpret_cast<S*>(ws + w.gsQ);
  p.gsG = reinterpret_cast<S*>(ws + w.gsG);
  p.gs_barrier = reinterpret_cast<unsigned int*>(ws + w.gs_barrier);
  p.guess = reinterpret_cast<uint32_t*>(ws + w.guess);
  p.votes = reinterpret_cast<uint32_t*>(ws + w.votes);
  p.status = s->status;
  p.control = s->control;
  p.halt = s->control ? &s->control->halt : nullptr;
  p.x_out = static_cast<S*>(s->x_out);
  p.u_out = static_cast<S*>(s->u_out);
  p.cost_out = static_cast<S*>(s->cost_out);
  p.du_out = static_cast<S*>(s->du_out);
  p.alpha_out = static_cast<S*>(s->alpha_out);
  p.K_out = static_cast<S*>(s->K_out);
  p.k_out = static_cast<S*>(s->k_out);
  for (int i = 0; i < 8; ++i) p.dyn.p[i] = (S)s->dyn_params[i];
  p.dyn.aux = static_cast<const S*>(s->dyn_aux);
  for (int i = 0; i < 4; ++i) p.dyn.ai[i] = s->dyn_ai[i];
  return p;
}

static int check(const DilqrSolve* s, bool need_ws) {
  if (!s || s->n_state <= 0 || s->n_ctrl <= 0 || s->T <= 0 || s->n_batch <= 0) return DILQR_EINVAL;
  if (!s->x_init || !s->C || !s->c) return DILQR_EINVAL;
  if ((s->dynamics == DILQR_DYN_LINDX || s->dynamics == DILQR_DYN_LINDX_RT) && s->T > 1 && !s->F)
    return DILQR_EINVAL;
  if ((s->dynamics == DILQR_DYN_NN || s->dynamics == DILQR_DYN_NN_RT) &&
      (!s->dyn_aux || s->dyn_ai[0] < 1 || (s->dyn_ai[0] & 0xffff) < 1 ||
       ((s->dyn_ai[0] >> 16) > 0 && (s->dyn_ai[0] & 0xffff) > 128) ||   /* two layers: H1 <= 128 */
       s->dyn_ai[1] < 0 || s->dyn_ai[1] > 1 ||
       s->dyn_ai[3] < 0 || s->dyn_ai[3] > 1))
    return DILQR_EINVAL;
  if (s->bounds_kind == DILQR_BOUNDS_TENSOR && (!s->u_lower_t || !s->u_upper_t)) return DILQR_EINVAL;
  if (s->bounds_kind < 0 || s->bounds_kind > 2) return DILQR_EINVAL;
  if (s->has_delta_u && (s->bounds_kind == DILQR_BOUNDS_NONE || !(s->delta_u > 0.0)))
    return DILQR_EINVAL;                      /* lqr_step.py:195 */
  if (s->C_bcast < 0 || s->C_bcast > 2 || s->c_bcast < 0 || s->c_bcast > 2) return DILQR_EINVAL;
  auto mis = [](const void* p) { return p && (reinterpret_cast<uintptr_t>(p) & 15u); };
  if (mis(s->C) || mis(s->c) || mis(s->F) || mis(s->f) || mis(s->workspace)) return DILQR_EALIGN;
  if (need_ws) {
    if (!s->workspace || !s->status) return DILQR_EINVAL;
    if (s->workspace_bytes < ws_layout(s, sizeof(Scalar)).total) return DILQR_EWORKSPACE;
  }
  return DILQR_OK;
}

// launch geometry for the warp-per-32-problems kernels
template <class S, int NS, int NC, int DYN>
struct Geometry {
  static constexpr bool STAGED = staged_v<S, NS, NC, DYN>();
  using IK = IterKernel<S, NS, NC, DYN, STAGED>;
  static int warps_per_block() {
    if (!STAGED) return 4;
    const size_t per = IK::smem_per_warp();
    int w = (int)((112 * 1024) / per);  // <= ~112 KB / block so two blocks fit one SM
    if (w > 4) w = 4;
    if (w < 1) w = 1;
    return w;
  }
  static size_t smem(int wpb) { return STAGED ? IK::smem_per_warp() * wpb : 0; }
};

// Workspace state a begin kernel starts from.  `packs_C`: the kernels keep a packed copy of C
// (ilqr_kernels.cuh); without it the packed-C state word stays 0 (no copy).
static void begin_state(const DilqrSolve* s, const IterParams<Scalar>& p, bool packs_C,
                        cudaStream_t st) {
  // default pnqp trace guess: at t = T-1 nothing moves (x_init=None is the exact
  // minimiser); at t < T-1 one Newton step then convergence (SURVEY a-5).
  const WsLayout w = ws_layout(s, sizeof(Scalar));
  static_assert(kPnqpMaxIter == DILQR_PNQP_MAX_ITER, "trace width");
  if (!s->keep_trace_guess) {
    cudaMemsetAsync(p.guess, 0, (size_t)p.T * kPnqpMaxIter * sizeof(uint32_t), st);
    if (p.T > 1)
      cudaMemset2DAsync(p.guess, kPnqpMaxIter * sizeof(uint32_t), 3, 1, p.T - 1, st);
  }
  // 1: begin packs the upper triangle of C for the sweeps (ilqr_kernels.cuh), 0: dense
  const bool pack = packs_C && !p.C_bcast && !(p.gains_only && p.x_cur);
  cudaMemsetAsync(p.cpk_state, 0, sizeof(uint32_t), st);
  if (pack) cudaMemsetAsync(p.cpk_state, 1, 1, st);   // little-endian: word value 1
  // 3: broadcast C, symmetry of the shared block(s) to be verified by begin
  if (packs_C && p.C_bcast && !(p.gains_only && p.x_cur)) cudaMemsetAsync(p.cpk_state, 3, 1, st);
  // ticket counter of the one-launch commit (returns to zero after every commit)
  cudaMemsetAsync(static_cast<char*>(s->workspace) + w.commit_ticket, 0, sizeof(uint32_t), st);
}

template <int NS, int NC, int DYN>
static int launch_begin(const DilqrSolve* s, cudaStream_t st) {
  using S = Scalar;
  using G = Geometry<S, NS, NC, DYN>;
  IterParams<S> p = make_params(s, 0);
  const int wpb = G::warps_per_block();
  const int warps = (p.B + kWarp - 1) / kWarp;
  const int blocks = (warps + wpb - 1) / wpb;
  const size_t smem = G::smem(wpb);
  auto kern = ilqr_begin_kernel<S, NS, NC, DYN, G::STAGED>;
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  begin_state(s, p, true, st);
  kern<<<blocks, wpb * kWarp, smem, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

// Shapes the batch-synchronous group sweep (group_kernels.cuh) is compiled for: everything
// too large for one thread per problem, and every multi-input shape (whose box-constrained
// batches otherwise need the whole batch co-resident or a replayed trace).
template <class S, int NS, int NC, int DYN>
constexpr bool group_sweep_v() {
  return (DYN == DYN_LINDX || DYN == DYN_ROCKET) && (!staged_v<S, NS, NC, DYN>() || NC > 1);
}

// Largest batch the group sweep holds on the current device (0: no group sweep for the shape):
// one phase-B thread per problem, every block co-resident.  Queried once per (device, shape);
// the query also raises the kernel's dynamic shared-memory limit on that device, which every
// later launch there relies on.
template <int NS, int NC, int DYN>
static int group_sweep_capacity() {
  using S = Scalar;
  if constexpr (!group_sweep_v<S, NS, NC, DYN>()) {
    return 0;
  } else {
    constexpr int kMaxDevices = 64;
    static std::atomic<int> cached[kMaxDevices];   // capacity + 1; 0: not queried yet
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (dev < kMaxDevices && cached[dev].load() > 0) return cached[dev].load() - 1;
    using GS = GroupSweep<S, NS, NC, DYN>;
    auto kern = group_sweep_kernel<S, NS, NC, DYN>;
    const size_t smem = GS::smem_bytes();
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int per_sm = 0, sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, GS::kThreads, smem) != cudaSuccess)
      return 0;
    const int cap = per_sm * sms * GS::kThreads;
    if (dev < kMaxDevices) cached[dev].store(cap + 1);
    return cap;
  }
}

// dilqr_mpc_plan: the group sweep for shapes too large for one thread per problem and for
// box-constrained multi-input batches, as long as the batch fits the device; trace replay
// otherwise.  The compile-time tests come first, so most shapes never query the device.
template <int NS, int NC, int DYN>
static int plan(DilqrSolve* s) {
  using S = Scalar;
  const bool boxed_multi = s->bounds_kind != DILQR_BOUNDS_NONE && s->solo == 0 && NC > 1;
  s->group_sweep = group_sweep_v<S, NS, NC, DYN>() && (!staged_v<S, NS, NC, DYN>() || boxed_multi) &&
                   s->n_batch > 0 && s->n_batch <= group_sweep_capacity<NS, NC, DYN>();
  return DILQR_OK;
}

template <int NS, int NC, int DYN>
static int launch_group_sweep(const DilqrSolve* s, IterParams<Scalar>& p, cudaStream_t st) {
  using S = Scalar;
  if constexpr (!group_sweep_v<S, NS, NC, DYN>()) {
    return DILQR_EUNSUPPORTED;
  } else {
    using GS = GroupSweep<S, NS, NC, DYN>;
    const int cap = group_sweep_capacity<NS, NC, DYN>();
    if (p.B > cap) return DILQR_ELOCKSTEP;
    const int max_blocks = cap / GS::kThreads;
    const int need_b = (p.B + GS::kThreads - 1) / GS::kThreads;       // phase B: thread per problem
    const int want_ac = (p.B + GS::GPB - 1) / GS::GPB;               // phase AC: group per problem
    int blocks = want_ac < max_blocks ? want_ac : max_blocks;
    if (blocks < need_b) blocks = need_b;
    if (p.bounds_kind && !p.solo)
      cudaMemsetAsync(p.votes, 0, (size_t)p.T * kPnqpMaxIter * sizeof(uint32_t), st);
    cudaMemsetAsync(p.gs_barrier, 0, sizeof(unsigned int), st);
    auto kern = group_sweep_kernel<S, NS, NC, DYN>;
    void* args[] = {(void*)&p};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)kern, dim3(blocks), dim3(GS::kThreads), args,
                                                GS::smem_bytes(), st);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return DILQR_ELOCKSTEP;
    }
    (void)s;
    return DILQR_OK;
  }
}

template <int NS, int NC, int DYN>
static int launch_iterate(const DilqrSolve* s, cudaStream_t st) {
  using S = Scalar;
  using G = Geometry<S, NS, NC, DYN>;
  IterParams<S> p = make_params(s);
  const int wpb = G::warps_per_block();
  const int warps = (p.B + kWarp - 1) / kWarp;
  const int blocks = (warps + wpb - 1) / wpb;
  const size_t smem = G::smem(wpb);
  g_iterate_launches = 0;
  if (s->group_sweep) {
    // Riccati / pnqp sweep by thread groups, all problems in step; then the line-search
    // rollout (one thread per problem: its state is small) as a second launch
    int rc = launch_group_sweep<NS, NC, DYN>(s, p, st);
    if (rc != DILQR_OK) return rc;
    g_iterate_launches = 1;
    if (p.gains_only) return DILQR_OK;
    if constexpr (group_sweep_v<S, NS, NC, DYN>()) {
      auto fwd = ilqr_iter_kernel<S, NS, NC, DYN, G::STAGED, true>;
      if (smem > 48 * 1024)
        cudaFuncSetAttribute(fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      fwd<<<blocks, wpb * kWarp, smem, st>>>(p);
      g_iterate_launches = 2;
    }
    return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
  }
  if (p.bounds_kind && !p.solo)
    cudaMemsetAsync(p.votes, 0, (size_t)p.T * kPnqpMaxIter * sizeof(uint32_t), st);
  g_iterate_launches = 1;
  auto kern = ilqr_iter_kernel<S, NS, NC, DYN, G::STAGED>;
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if constexpr (sym_pair_v<S, NS, NC, DYN>()) {
    // symmetric Riccati update when the packed copy of C is valid (ilqr_kernels.cuh, kSym): the
    // flag is on the device, so both kernels of the pair are enqueued and one exits at once
    auto ksym = ilqr_iter_kernel<S, NS, NC, DYN, G::STAGED, false, true>;
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(ksym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    p.sym_pair = 1;
    ksym<<<blocks, wpb * kWarp, smem, st>>>(p);
    g_iterate_launches = 2;
  }
  kern<<<blocks, wpb * kWarp, smem, st>>>(p);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

// gains of the final no-op LQR pass + costates at the solution (ilqr_gains_kernel)
template <int NS, int NC, int DYN>
static int launch_gains(const DilqrSolve* s, void* lam_blk, cudaStream_t st) {
  using S = Scalar;
  using G = Geometry<S, NS, NC, DYN>;
  if constexpr (!G::STAGED || DYN == DYN_LINDX || DYN == DYN_NN) {
    return DILQR_EUNSUPPORTED;
  } else {
    if (!s->x_out || !s->u_out) return DILQR_EINVAL;
    if (s->u_zero_I || (s->bounds_kind && !s->solo && NC > 1)) return DILQR_EUNSUPPORTED;
    IterParams<S> p = make_params(s);
    p.gains_only = 1;
    p.lam_blk = static_cast<S*>(lam_blk);
    using IK = typename G::IK;
    size_t per = IK::smem_per_warp(true);
    int wpb = (int)((112 * 1024) / per);
    if (wpb > 4) wpb = 4;
    if (wpb < 1) wpb = 1;
    const int warps = (p.B + kWarp - 1) / kWarp;
    const int blocks = (warps + wpb - 1) / wpb;
    const size_t smem = per * wpb;
    auto kern = ilqr_gains_kernel<S, NS, NC, DYN, G::STAGED>;
    if (smem > 48 * 1024)
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    // pnqp trace guess: this sweep's own, kept in the workspace from call to call (the
    // correction a mismatching call leaves is the right guess for the next call / step)
    p.guess = reinterpret_cast<uint32_t*>(static_cast<char*>(s->workspace) +
                                          ws_layout(s, sizeof(S)).guess_gains);
    if (s->gains_guess_reset) {   // default: nothing moves at T-1, one Newton step elsewhere
      cudaMemsetAsync(p.guess, 0, (size_t)p.T * kPnqpMaxIter * sizeof(uint32_t), st);
      if (p.T > 1) cudaMemset2DAsync(p.guess, kPnqpMaxIter * sizeof(uint32_t), 3, 1, p.T - 1, st);
    }
    if (p.bounds_kind && !p.solo)
      cudaMemsetAsync(p.votes, 0, (size_t)p.T * kPnqpMaxIter * sizeof(uint32_t), st);
    if constexpr (sym_pair_v<S, NS, NC, DYN>()) {
      auto ksym = ilqr_gains_kernel<S, NS, NC, DYN, G::STAGED, true>;
      if (smem > 48 * 1024)
        cudaFuncSetAttribute(ksym, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      p.sym_pair = 1;
      ksym<<<blocks, wpb * kWarp, smem, st>>>(p);
    }
    kern<<<blocks, wpb * kWarp, smem, st>>>(p);
    trace_verify_kernel<<<1, 256, 0, st>>>(p.guess, p.votes, p.T, p.bounds_kind != 0, p.solo,
                                           s->status);
    return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
  }
}

template <int NS, int NC>
static int launch_commit(const DilqrSolve* s, cudaStream_t st) {
  using S = Scalar;
  IterParams<S> p = make_params(s);
  const WsLayout w = ws_layout(s, sizeof(S));
  char* ws = static_cast<char*>(s->workspace);
  CommitAux aux;
  aux.part = reinterpret_cast<CommitPart*>(ws + w.commit_part);
  aux.ticket = reinterpret_cast<unsigned int*>(ws + w.commit_ticket);
  aux.ctrl = s->control;
  aux.votes_are_trace = p.votes_are_trace;
  aux.iteration = s->iteration;
  aux.nc = s->n_ctrl;
  commit_kernel<S, NS + NC, NC><<<(p.B + 127) / 128, 128, 0, st>>>(p, aux);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

template <int NS, int NC>
static int launch_finish(const DilqrSolve* s, cudaStream_t st) {
  using S = Scalar;
  IterParams<S> p = make_params(s);
  dim3 grid((p.B + 127) / 128, p.T);
  finish_kernel<S, NS, NC><<<grid, 128, 0, st>>>(p, s->n_state, s->n_ctrl);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

template <int NS, int NC>
static int launch_kkt(const DilqrKkt* k, cudaStream_t st) {
  using S = Scalar;
  kkt_grads_kernel<S, NS, NC><<<(k->n_batch + 127) / 128, 128, 0, st>>>(*k);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

// ------------------------------------------------------------------ dispatch
enum Op { OP_BEGIN, OP_ITERATE, OP_COMMIT, OP_FINISH };

#if DILQR_GROUP == 0
// DILQR_DYN_LINDX_RT / DILQR_DYN_NN_RT (rt_kernels.cuh): one warp per problem, the warp's
// shared-memory slice sized for (n_state, n_ctrl) and, for a network, its hidden widths; commit
// and finish are the compiled family's kernels with runtime dimensions.
static bool rt_dynamics(int dynamics) {
  return dynamics == DILQR_DYN_LINDX_RT || dynamics == DILQR_DYN_NN_RT;
}

static int rt_launch(const DilqrSolve* s, Op op, cudaStream_t st) {
  using S = Scalar;
  const int ns = s->n_state, nc = s->n_ctrl;
  if (!rt_shape_ok(ns, nc)) return DILQR_EUNSUPPORTED;
  if (op == OP_COMMIT) return launch_commit<0, 0>(s, st);
  if (op == OP_FINISH) return launch_finish<0, 0>(s, st);
  IterParams<S> p = make_params(s, op == OP_BEGIN ? 0 : 1);
  const bool nn = s->dynamics == DILQR_DYN_NN_RT;
  const size_t per = nn ? rt_nn_slice_bytes<S>(ns, nc, s->dyn_ai[0]) : RtSmem<S>::bytes(ns, nc);
  int wpb = (int)((96 * 1024) / per);   // <= 96 KB a block: two blocks fit one SM
  if (wpb > 4) wpb = 4;
  if (wpb < 1) wpb = 1;
  const int blocks = (p.B + wpb - 1) / wpb;
  const size_t smem = per * wpb;
  auto kern = op == OP_BEGIN ? (nn ? rt_nn_begin_kernel<S> : rt_begin_kernel<S>)
                             : (nn ? rt_nn_iter_kernel<S> : rt_iter_kernel<S>);
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (op == OP_BEGIN) {
    begin_state(s, p, false, st);
  } else {
    if (p.bounds_kind && !p.solo)
      cudaMemsetAsync(p.votes, 0, (size_t)p.T * kPnqpMaxIter * sizeof(uint32_t), st);
    g_iterate_launches = 1;
  }
  kern<<<blocks, wpb * kWarp, smem, st>>>(p, ns, nc);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}
#endif

static int dispatch(const DilqrSolve* s, Op op, cudaStream_t st) {
#if DILQR_GROUP == 0
  if (rt_dynamics(s->dynamics)) return rt_launch(s, op, st);
#endif
#define X(NS_, NC_, DYN_)                                                            \
  if (s->n_state == NS_ && s->n_ctrl == NC_ && s->dynamics == DYN_) {                \
    switch (op) {                                                                    \
      case OP_BEGIN: return launch_begin<NS_, NC_, DYN_>(s, st);                     \
      case OP_ITERATE: return launch_iterate<NS_, NC_, DYN_>(s, st);                 \
      case OP_COMMIT: return launch_commit<NS_, NC_>(s, st);                         \
      case OP_FINISH: return launch_finish<NS_, NC_>(s, st);                         \
    }                                                                                \
  }
  DILQR_CONFIGS(X)
#undef X
  return DILQR_EUNSUPPORTED;
}

int DILQR_SUFFIX(mpc_plan)(DilqrSolve* s) {
#if DILQR_GROUP == 0
  if (rt_dynamics(s->dynamics)) {   // replays the pnqp trace; never asks the device
    if (!rt_shape_ok(s->n_state, s->n_ctrl)) return DILQR_EUNSUPPORTED;
    s->group_sweep = 0;
    return DILQR_OK;
  }
#endif
#define X(NS_, NC_, DYN_) \
  if (s->n_state == NS_ && s->n_ctrl == NC_ && s->dynamics == DYN_) return plan<NS_, NC_, DYN_>(s);
  DILQR_CONFIGS(X)
#undef X
  return DILQR_EUNSUPPORTED;
}

int DILQR_SUFFIX(supported)(int n_state, int n_ctrl, int dynamics) {
#if DILQR_GROUP == 0
  if (rt_dynamics(dynamics)) return rt_shape_ok(n_state, n_ctrl) ? 1 : 0;
#endif
#define X(NS_, NC_, DYN_) \
  if (n_state == NS_ && n_ctrl == NC_ && dynamics == DYN_) return 1;
  DILQR_CONFIGS(X)
#undef X
  return 0;
}

#if DILQR_GROUP == 0
size_t DILQR_SUFFIX(workspace_bytes)(const DilqrSolve* s) {
  return ws_layout(s, sizeof(Scalar)).total;
}
int DILQR_SUFFIX(workspace_view)(const DilqrSolve* s, DilqrWsView* v) {
  if (!s->workspace) return DILQR_EINVAL;
  const WsLayout w = ws_layout(s, sizeof(Scalar));
  if (s->workspace_bytes < w.total) return DILQR_EWORKSPACE;
  char* ws = static_cast<char*>(s->workspace);
  v->Kk = ws + w.Kk;
  v->Cpk = ws + w.Cpk;
  v->cpk_state = reinterpret_cast<const uint32_t*>(ws + w.cpk_state);
  v->n_warps = w.Bp / 32;
  v->reserved = 0;
  return DILQR_OK;
}

#endif

int DILQR_SUFFIX(mpc_begin)(const DilqrSolve* s, void* stream) {
  int e = check(s, true);
  if (e) return e;
  return dispatch(s, OP_BEGIN, static_cast<cudaStream_t>(stream));
}
int DILQR_SUFFIX(mpc_iterate)(const DilqrSolve* s, void* stream) {
  int e = check(s, true);
  if (e) return e;
  return dispatch(s, OP_ITERATE, static_cast<cudaStream_t>(stream));
}
int DILQR_SUFFIX(mpc_commit)(const DilqrSolve* s, void* stream) {
  int e = check(s, true);
  if (e) return e;
  return dispatch(s, OP_COMMIT, static_cast<cudaStream_t>(stream));
}
int DILQR_SUFFIX(mpc_finish)(const DilqrSolve* s, void* stream) {
  int e = check(s, true);
  if (e) return e;
  return dispatch(s, OP_FINISH, static_cast<cudaStream_t>(stream));
}
int DILQR_SUFFIX(mpc_gains)(const DilqrSolve* s, void* lam_blk, void* stream) {
  int e = check(s, true);
  if (e) return e;
#define X(NS_, NC_, DYN_)                                                       \
  if (s->n_state == NS_ && s->n_ctrl == NC_ && s->dynamics == DYN_)             \
    return launch_gains<NS_, NC_, DYN_>(s, lam_blk, static_cast<cudaStream_t>(stream));
  DILQR_CONFIGS(X)
#undef X
  return DILQR_EUNSUPPORTED;
}

int DILQR_SUFFIX(kkt_grads)(const DilqrKkt* k, void* stream) {
  if (!k || !k->C || !k->c || !k->x || !k->u || !k->dx || !k->du || !k->r) return DILQR_EINVAL;
  if (k->T > 1 && !k->F) return DILQR_EINVAL;
#if DILQR_GROUP == 0
  if (k->dynamics == DILQR_DYN_LINDX_RT) {
    if (k->T <= 0 || k->n_batch <= 0) return DILQR_EINVAL;
    if (!rt_shape_ok(k->n_state, k->n_ctrl)) return DILQR_EUNSUPPORTED;
    rt_kkt_kernel<Scalar><<<(k->n_batch + 3) / 4, 128, 0, static_cast<cudaStream_t>(stream)>>>(*k);
    return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
  }
#endif
#define X(NS_, NC_, DYN_)                                                                 \
  if (DYN_ == DYN_LINDX && k->dynamics == DILQR_DYN_LINDX && k->n_state == NS_ &&          \
      k->n_ctrl == NC_)                                                                    \
    return launch_kkt<NS_, NC_>(k, static_cast<cudaStream_t>(stream));
  DILQR_CONFIGS(X)
#undef X
  return DILQR_EUNSUPPORTED;
}

#if DILQR_GROUP == 0
template <int DYN>
static int launch_linearize(const double* dp, int T, int B, const void* x, const void* u, void* F,
                            void* f, cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  if (T < 2) return DILQR_OK;
  dim3 grid((B + 127) / 128, T - 1);
  linearize_kernel<S, DYN><<<grid, 128, 0, st>>>(P, T, B, static_cast<const S*>(x),
                                                  static_cast<const S*>(u), static_cast<S*>(F),
                                                  static_cast<S*>(f));
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(linearize)(int dynamics, const double* dp, int T, int B, const void* x,
                            const void* u, void* F, void* f, void* stream) {
  if (!dp || !x || !u || !F || T <= 0 || B <= 0) return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_linearize<DYN_PENDULUM>(dp, T, B, x, u, F, f, st);
  if (dynamics == DYN_CARTPOLE) return launch_linearize<DYN_CARTPOLE>(dp, T, B, x, u, F, f, st);
  if (dynamics == DYN_ROCKET) return launch_linearize<DYN_ROCKET>(dp, T, B, x, u, F, f, st);
  return DILQR_EUNSUPPORTED;
}

template <int DYN>
static int launch_rollout(const double* dp, int T, int B, const void* x0, const void* u, void* x,
                          cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  rollout_kernel<S, DYN><<<(B + 127) / 128, 128, 0, st>>>(P, T, B, static_cast<const S*>(x0),
                                                           static_cast<const S*>(u),
                                                           static_cast<S*>(x));
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(rollout)(int dynamics, const double* dp, int T, int B, const void* x0,
                          const void* u, void* x, void* stream) {
  if (!dp || !x0 || !u || !x || T <= 0 || B <= 0) return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_rollout<DYN_PENDULUM>(dp, T, B, x0, u, x, st);
  if (dynamics == DYN_CARTPOLE) return launch_rollout<DYN_CARTPOLE>(dp, T, B, x0, u, x, st);
  if (dynamics == DYN_ROCKET) return launch_rollout<DYN_ROCKET>(dp, T, B, x0, u, x, st);
  return DILQR_EUNSUPPORTED;
}

// ------------------------------------------------- standalone pnqp
template <int N>
static int launch_pnqp(int B, const void* H, const void* q, const void* lo, const void* hi,
                       const void* x0, void* x, void* lu, int32_t* piv, void* If, uint32_t* trace,
                       int solo, DilqrStatus* status, cudaStream_t st) {
  using S = Scalar;
  uint32_t* guess = trace;
  uint32_t* votes = trace + kPnqpMaxIter;
  cudaMemsetAsync(votes, 0, kPnqpMaxIter * sizeof(uint32_t), st);
  pnqp_kernel<S, N><<<(B + 127) / 128, 128, 0, st>>>(
      B, static_cast<const S*>(H), static_cast<const S*>(q), static_cast<const S*>(lo),
      static_cast<const S*>(hi), static_cast<const S*>(x0), static_cast<S*>(x),
      static_cast<S*>(lu), piv, static_cast<S*>(If), guess, votes, solo);
  trace_verify_kernel<<<1, 32, 0, st>>>(guess, votes, 1, 1, solo, status);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(pnqp)(int n, int B, const void* H, const void* q, const void* lo, const void* hi,
                       const void* x0, void* x, void* lu, int32_t* piv, void* If, uint32_t* trace,
                       int solo, DilqrStatus* status, void* stream) {
  if (!H || !q || !lo || !hi || !x || !lu || !piv || !If || !trace || !status || B <= 0)
    return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (n) {
    case 1: return launch_pnqp<1>(B, H, q, lo, hi, x0, x, lu, piv, If, trace, solo, status, st);
    case 2: return launch_pnqp<2>(B, H, q, lo, hi, x0, x, lu, piv, If, trace, solo, status, st);
    case 3: return launch_pnqp<3>(B, H, q, lo, hi, x0, x, lu, piv, If, trace, solo, status, st);
    case 4: return launch_pnqp<4>(B, H, q, lo, hi, x0, x, lu, piv, If, trace, solo, status, st);
    case 6: return launch_pnqp<6>(B, H, q, lo, hi, x0, x, lu, piv, If, trace, solo, status, st);
    case 8: return launch_pnqp<8>(B, H, q, lo, hi, x0, x, lu, piv, If, trace, solo, status, st);
    default: return DILQR_EUNSUPPORTED;
  }
}

// n and the iteration budget at run time (pnqp_rt.cuh): one warp per problem, the warp's
// shared-memory slice sized for n.
int DILQR_SUFFIX(pnqp_rt)(int n, int n_iter, int B, const void* H, const void* q, const void* lo,
                          const void* hi, const void* x0, void* x, void* lu, int32_t* piv, void* If,
                          uint32_t* trace, int solo, DilqrStatus* status, void* stream) {
  if (!H || !q || !lo || !hi || !x || !lu || !piv || !If || !trace || !status || B <= 0 ||
      n <= 0 || n_iter <= 0)
    return DILQR_EINVAL;
  if (!pnqp_rt_ok(n, n_iter)) return DILQR_EUNSUPPORTED;
  if (reinterpret_cast<uintptr_t>(trace) % sizeof(uint32_t)) return DILQR_EALIGN;
  using S = Scalar;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint32_t* guess = trace;
  uint32_t* votes = trace + n_iter;
  const size_t per = PnqpRtSmem<S>::bytes(n);
  int wpb = (int)((96 * 1024) / per);   // <= 96 KB a block: two blocks fit one SM
  if (wpb > 4) wpb = 4;
  const size_t smem = per * wpb;
  if (smem > 48 * 1024)
    cudaFuncSetAttribute(pnqp_rt_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  cudaMemsetAsync(votes, 0, (size_t)n_iter * sizeof(uint32_t), st);
  pnqp_rt_kernel<S><<<(B + wpb - 1) / wpb, wpb * kWarp, smem, st>>>(
      B, n, n_iter, static_cast<const S*>(H), static_cast<const S*>(q), static_cast<const S*>(lo),
      static_cast<const S*>(hi), static_cast<const S*>(x0), static_cast<S*>(x), static_cast<S*>(lu),
      piv, static_cast<S*>(If), guess, votes, solo);
  pnqp_rt_verify_kernel<<<1, 32, 0, st>>>(guess, votes, n_iter, solo, status);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

// ------------------------------------------------- factored adjoint solves
struct AdjLayout {
  size_t fac, kvec, dtau, total;
  int Bp;
};
template <int DYN>
static AdjLayout adj_layout(const DilqrAdjoint* a) {
  using A = Adj<Scalar, DYN>;
  AdjLayout w;
  w.Bp = (int)align_up((size_t)a->n_batch, 32);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off = align_up(off + bytes, 256);
    return o;
  };
  w.fac = take((size_t)a->T * A::NFAC * w.Bp * sizeof(Scalar));
  w.kvec = take((size_t)a->T * A::NC * w.Bp * sizeof(Scalar));
  w.dtau = take((size_t)a->T * A::N * w.Bp * sizeof(Scalar));
  w.total = off;
  return w;
}

template <int DYN>
static int adj_run(const DilqrAdjoint* a, int what, cudaStream_t st) {
  using S = Scalar;
  using A = Adj<S, DYN>;
  if (a->n_state != A::NS || a->n_ctrl != A::NC) return DILQR_EINVAL;
  const AdjLayout w = adj_layout<DYN>(a);
  if (!a->workspace || a->workspace_bytes < w.total) return DILQR_EWORKSPACE;
  AdjParams<S> p;
  memset(&p, 0, sizeof(p));
  char* ws = static_cast<char*>(a->workspace);
  p.T = a->T;
  p.B = a->n_batch;
  p.Bp = w.Bp;
  p.bounds_kind = a->bounds_kind;
  p.gain_solve = a->gain_solve;
  p.final_pass = what == 2;
  p.C_bcast = a->C_bcast;
  p.c_bcast = a->c_bcast;
  p.lo = (S)a->u_lower;
  p.hi = (S)a->u_upper;
  p.C = static_cast<const S*>(a->C);
  p.x = static_cast<const S*>(a->x);
  p.u = static_cast<const S*>(a->u);
  p.gx = static_cast<const S*>(a->gx);
  p.gu = static_cast<const S*>(a->gu);
  p.Cpk = static_cast<const S*>(a->Cpk);
  p.cpk_state = a->cpk_state;
  p.first = a->first_pass;
  p.want_resid = a->want_resid;
  p.reduce_tile = (what == 2) ? a->reduce_tile : 0;
  p.red_out = static_cast<S*>(a->red_out);
  p.df_blk = static_cast<S*>(a->df_blk);
  p.Lam = static_cast<const S*>(a->Lam);
  p.w = static_cast<S*>(a->w);
  p.fac = reinterpret_cast<S*>(ws + w.fac);
  p.kvec = reinterpret_cast<S*>(ws + w.kvec);
  p.dtau = reinterpret_cast<S*>(ws + w.dtau);
  p.dC = static_cast<S*>(a->dC);
  p.dc = static_cast<S*>(a->dc);
  p.df = static_cast<S*>(a->df);
  p.dx_out = static_cast<S*>(a->dx_out);
  p.du_out = static_cast<S*>(a->du_out);
  p.resid = static_cast<unsigned long long*>(a->resid);
  for (int i = 0; i < 8; ++i) p.dyn.p[i] = (S)a->dyn_params[i];
  const int warps = (p.B + kWarp - 1) / kWarp;
  constexpr int N = A::N;
  const uint32_t e1[1] = {N * N};
  if (what == 0) {
    const int wpb = 4;
    const size_t smem = (WarpStager<S>::bytes_per_warp(1, e1) + kStages * sizeof(uint64_t)) * wpb;
    auto kern = adjoint_factor_kernel<S, DYN>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<(warps + wpb - 1) / wpb, wpb * kWarp, smem, st>>>(p);
  } else if (what == 1) {
    const int wpb = 1;
    const size_t smem = AdjStage<S, DYN>::smem_per_warp(false) * wpb;
    auto kern = adjoint_pass_kernel<S, DYN, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (p.want_resid) cudaMemsetAsync(p.resid, 0, 16, st);   // max|dw|, max|w|; the reject counter accumulates
    kern<<<(warps + wpb - 1) / wpb, wpb * kWarp, smem, st>>>(p);
  } else {
    const int wpb = 1;
    const size_t smem = AdjStage<S, DYN>::smem_per_warp(true) * wpb;
    auto kern = p.reduce_tile ? adjoint_pass_kernel<S, DYN, true, true>
                              : adjoint_pass_kernel<S, DYN, true, false>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<(warps + wpb - 1) / wpb, wpb * kWarp, smem, st>>>(p);
  }
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

static int adj_check(const DilqrAdjoint* a, int what) {
  if (!a || a->T < 2 || a->n_batch <= 0 || !a->C || !a->x || !a->u || !a->resid)
    return DILQR_EINVAL;
  if (what != 0 && !a->gu) return DILQR_EINVAL;    // the factorisation needs no right-hand side
  if (what == 1 && (!a->w || !a->Lam)) return DILQR_EINVAL;
  if (what == 2 && !a->first_pass && !a->w) return DILQR_EINVAL;
  if (what == 2 && a->reduce_tile && (!a->red_out || a->C_bcast || a->c_bcast)) return DILQR_EINVAL;
  if (a->bounds_kind != DILQR_BOUNDS_NONE && a->bounds_kind != DILQR_BOUNDS_SCALAR)
    return DILQR_EINVAL;
  auto mis = [](const void* p) { return p && (reinterpret_cast<uintptr_t>(p) & 15u); };
  if (mis(a->C) || mis(a->gx) || mis(a->gu) || mis(a->w) || mis(a->Lam) || mis(a->dC) ||
      mis(a->dc) || mis(a->workspace) || mis(a->Cpk))
    return DILQR_EALIGN;
  return DILQR_OK;
}

size_t DILQR_SUFFIX(adjoint_workspace_bytes)(const DilqrAdjoint* a) {
  if (!a) return 0;
  if (a->dynamics == DYN_PENDULUM) return adj_layout<DYN_PENDULUM>(a).total;
  if (a->dynamics == DYN_CARTPOLE) return adj_layout<DYN_CARTPOLE>(a).total;
  return 0;
}

size_t DILQR_SUFFIX(adjoint_dtau_offset)(const DilqrAdjoint* a) {
  if (!a) return 0;
  if (a->dynamics == DYN_PENDULUM) return adj_layout<DYN_PENDULUM>(a).dtau;
  if (a->dynamics == DYN_CARTPOLE) return adj_layout<DYN_CARTPOLE>(a).dtau;
  return 0;
}

int DILQR_SUFFIX(lam_pack_size)(int dynamics) {
  if (dynamics == DYN_PENDULUM) return LamPack<Scalar, DYN_PENDULUM>::NLAM;
  if (dynamics == DYN_CARTPOLE) return LamPack<Scalar, DYN_CARTPOLE>::NLAM;
  if (dynamics == DYN_ROCKET) return LamPack<Scalar, DYN_ROCKET>::NLAM;
  return 0;
}

int DILQR_SUFFIX(adjoint_run)(const DilqrAdjoint* a, int what, void* stream) {
  int e = adj_check(a, what);
  if (e) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (a->dynamics == DYN_PENDULUM) return adj_run<DYN_PENDULUM>(a, what, st);
  if (a->dynamics == DYN_CARTPOLE) return adj_run<DYN_CARTPOLE>(a, what, st);
  return DILQR_EUNSUPPORTED;
}

// ------------------------------------------------- DiLQR implicit backward
template <int DYN>
static int launch_costate(const double* dp, int T, int B, const void* C, const void* c,
                          const void* x, const void* u, void* lam, void* Lam, int Cb, int cb,
                          int packed, cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  const int wpb = CostateStage<S, DYN>::smem_per_warp() * 2 <= 200 * 1024 ? 2 : 1;
  const size_t smem = CostateStage<S, DYN>::smem_per_warp() * wpb;
  if (smem > 227 * 1024) return DILQR_EUNSUPPORTED;
  auto kern = packed ? costate_tables_kernel<S, DYN, true> : costate_tables_kernel<S, DYN, false>;
  cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  const int warps = (B + kWarp - 1) / kWarp;
  kern<<<(warps + wpb - 1) / wpb, wpb * kWarp, smem, st>>>(
      P, T, B, static_cast<const S*>(C), static_cast<const S*>(c), static_cast<const S*>(x),
      static_cast<const S*>(u), static_cast<S*>(lam), static_cast<S*>(Lam), Cb, cb);
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(costate_tables)(int dynamics, const double* dp, int T, int B, const void* C,
                                 const void* c, const void* x, const void* u, void* lam,
                                 void* Lam, int Cb, int cb, int packed, void* stream) {
  if (!dp || !C || !c || !x || !u || !lam || !Lam || T <= 0 || B <= 0) return DILQR_EINVAL;
  if (Cb < 0 || Cb > 2 || cb < 0 || cb > 2) return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_costate<DYN_PENDULUM>(dp, T, B, C, c, x, u, lam, Lam, Cb, cb, packed, st);
  if (dynamics == DYN_CARTPOLE) return launch_costate<DYN_CARTPOLE>(dp, T, B, C, c, x, u, lam, Lam, Cb, cb, packed, st);
  if (dynamics == DYN_ROCKET) return launch_costate<DYN_ROCKET>(dp, T, B, C, c, x, u, lam, Lam, Cb, cb, packed, st);
  return DILQR_EUNSUPPORTED;
}

template <int DYN>
static int launch_lam_tables(const double* dp, int T, int B, const void* x, const void* u,
                             const void* lam_blk, void* Lam, cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  memset(&P, 0, sizeof(P));
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  if (T < 2) return DILQR_OK;
  const int Bp = (B + kWarp - 1) / kWarp * kWarp;
  dim3 grid((Bp + 127) / 128, T - 1);
  lam_tables_kernel<S, DYN><<<grid, 128, 0, st>>>(P, T, B, static_cast<const S*>(x),
                                                   static_cast<const S*>(u),
                                                   static_cast<const S*>(lam_blk),
                                                   static_cast<S*>(Lam));
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(lam_tables)(int dynamics, const double* dp, int T, int B, const void* x,
                             const void* u, const void* lam_blk, void* Lam, void* stream) {
  if (!dp || !x || !u || !lam_blk || !Lam || T <= 0 || B <= 0) return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_lam_tables<DYN_PENDULUM>(dp, T, B, x, u, lam_blk, Lam, st);
  if (dynamics == DYN_CARTPOLE) return launch_lam_tables<DYN_CARTPOLE>(dp, T, B, x, u, lam_blk, Lam, st);
  if (dynamics == DYN_ROCKET) return launch_lam_tables<DYN_ROCKET>(dp, T, B, x, u, lam_blk, Lam, st);
  return DILQR_EUNSUPPORTED;
}

template <int DYN>
static int launch_sens_adjoint(const double* dp, int T, int B, const void* x, const void* u,
                               const void* Kk, const void* lam, const void* dtau, const void* df,
                               const void* Lam, void* dtheta, cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  memset(&P, 0, sizeof(P));
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  const int Bp = (B + kWarp - 1) / kWarp * kWarp;
  sens_theta_adjoint_kernel<S, DYN><<<(Bp + 63) / 64, 64, 0, st>>>(
      P, T, B, static_cast<const S*>(x), static_cast<const S*>(u), static_cast<const S*>(Kk),
      static_cast<const S*>(lam), static_cast<const S*>(dtau), static_cast<const S*>(df),
      static_cast<const S*>(Lam), static_cast<S*>(dtheta));
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(sens_theta_adjoint)(int dynamics, const double* dp, int T, int B, const void* x,
                                     const void* u, const void* Kk, const void* lam,
                                     const void* dtau, const void* df, const void* Lam,
                                     void* dtheta, void* stream) {
  if (!dp || !x || !u || !Kk || !lam || !dtau || !df || !Lam || !dtheta || T <= 1 || B <= 0)
    return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_sens_adjoint<DYN_PENDULUM>(dp, T, B, x, u, Kk, lam, dtau, df, Lam, dtheta, st);
  if (dynamics == DYN_CARTPOLE) return launch_sens_adjoint<DYN_CARTPOLE>(dp, T, B, x, u, Kk, lam, dtau, df, Lam, dtheta, st);
  return DILQR_EUNSUPPORTED;
}

template <int DYN>
static int launch_sens(const double* dp, int T, int B, const void* x, const void* u,
                       const void* K, const void* lam, const void* dx, const void* du,
                       const void* df, void* dtheta, cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  sens_theta_kernel<S, DYN><<<(B + 63) / 64, 64, 0, st>>>(
      P, T, B, static_cast<const S*>(x), static_cast<const S*>(u), static_cast<const S*>(K),
      static_cast<const S*>(lam), static_cast<const S*>(dx), static_cast<const S*>(du),
      static_cast<const S*>(df), static_cast<S*>(dtheta));
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(sens_theta)(int dynamics, const double* dp, int T, int B, const void* x,
                             const void* u, const void* K, const void* lam, const void* dx,
                             const void* du, const void* df, void* dtheta, void* stream) {
  if (!dp || !x || !u || !K || !lam || !dx || !du || !df || !dtheta || T <= 1 || B <= 0)
    return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_sens<DYN_PENDULUM>(dp, T, B, x, u, K, lam, dx, du, df, dtheta, st);
  if (dynamics == DYN_CARTPOLE) return launch_sens<DYN_CARTPOLE>(dp, T, B, x, u, K, lam, dx, du, df, dtheta, st);
  if (dynamics == DYN_ROCKET) return launch_sens<DYN_ROCKET>(dp, T, B, x, u, K, lam, dx, du, df, dtheta, st);
  return DILQR_EUNSUPPORTED;
}

template <int DYN>
static int launch_tables(const double* dp, int n, const void* x, const void* u, void* const* out,
                         cudaStream_t st) {
  using S = Scalar;
  DynParams<S> P;
  for (int i = 0; i < 8; ++i) P.p[i] = (S)dp[i];
  env_tables_kernel<S, DYN><<<(n + 63) / 64, 64, 0, st>>>(
      P, n, static_cast<const S*>(x), static_cast<const S*>(u), static_cast<S*>(out[0]),
      static_cast<S*>(out[1]), static_cast<S*>(out[2]), static_cast<S*>(out[3]),
      static_cast<S*>(out[4]), static_cast<S*>(out[5]), static_cast<S*>(out[6]));
  return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;
}

int DILQR_SUFFIX(env_tables)(int dynamics, const double* dp, int n, const void* x, const void* u,
                             void* const* out, void* stream) {
  if (!dp || !x || !u || !out || n <= 0) return DILQR_EINVAL;
  for (int i = 0; i < 7; ++i)
    if (!out[i]) return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dynamics == DYN_PENDULUM) return launch_tables<DYN_PENDULUM>(dp, n, x, u, out, st);
  if (dynamics == DYN_CARTPOLE) return launch_tables<DYN_CARTPOLE>(dp, n, x, u, out, st);
  if (dynamics == DYN_ROCKET) return launch_tables<DYN_ROCKET>(dp, n, x, u, out, st);
  return DILQR_EUNSUPPORTED;
}

#endif  // DILQR_GROUP == 0

int DILQR_SUFFIX(richardson_update)(int ns, int nc, int T, int B, const void* g, const void* Lam,
                                    const void* dx, const void* du, void* w, void* negw,
                                    void* resid, void* stream) {
  using S = Scalar;
  if (!g || !Lam || !dx || !du || !w || !negw || !resid || T <= 0 || B <= 0) return DILQR_EINVAL;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid((B + 127) / 128, T);
  cudaMemsetAsync(resid, 0, 16, st);
#define X(NS_, NC_, DYN_)                                                                   \
  if (DYN_ == DYN_LINDX && ns == NS_ && nc == NC_) {                                        \
    richardson_update_kernel<S, NS_, NC_><<<grid, 128, 0, st>>>(                            \
        T, B, static_cast<const S*>(g), static_cast<const S*>(Lam), static_cast<const S*>(dx), \
        static_cast<const S*>(du), static_cast<S*>(w), static_cast<S*>(negw),               \
        static_cast<unsigned long long*>(resid));                                           \
    return cudaGetLastError() == cudaSuccess ? DILQR_OK : DILQR_ECUDA;                      \
  }
  DILQR_CONFIGS(X)
#undef X
  return DILQR_EUNSUPPORTED;
}

}  // namespace dilqr
