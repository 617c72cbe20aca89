// misc_kernels.cuh -- bookkeeping kernels around the fused iLQR iteration:
// trace verification, best-iterate commit, gather to the API layout, analytic
// linearisation, nominal rollout, and the KKT gradient assembly.
#pragma once
#include "../../include/dilqr.h"
#include "ilqr_kernels.cuh"

namespace dilqr {

// ---------------------------------------------------------------------------
// Verify the replayed pnqp control-flow trace (one block).  votes == guess up
// to the first wrong guess; on mismatch the votes become the next guess.
// Also derives n_total_qp_iter = sum_t (1 + n_qp_iter_t)  (lqr_step.py:140) and
// resets the reduction fields of the status block.  W words per timestep (the
// pnqp iteration budget n_iter): W_CT when > 0, else W_RT.  trace_verify_kernel
// passes W_CT = kPnqpMaxIter and compiles to the code it had before the runtime
// budget existed.
// ---------------------------------------------------------------------------
template <int W_CT>
DILQR_DEVICE void trace_verify_block(uint32_t* __restrict__ guess, const uint32_t* __restrict__ votes,
                                     int T, int W_RT, int boxed, int solo, DilqrStatus* status,
                                     DilqrControl* ctrl) {
  const int W = W_CT > 0 ? W_CT : W_RT;
  if (ctrl && ctrl->halt) return;   // uniform: whole block leaves
  __shared__ int s_first;
  __shared__ unsigned s_nqp, s_unconv;
  const int n = T * W;
  if (threadIdx.x == 0) {
    s_first = n;
    s_nqp = 0;
    s_unconv = 0;
  }
  __syncthreads();
  if (boxed && !solo) {
    // Normalised vote of a slot: if nobody was moving the sweep left the slot
    // right there, so Armijo bits voted under a wrong "moving" guess are void.
    // Processing order of the sweep is t = T-1 .. 0, it = 0 .. 19.
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int t = T - 1 - i / W, it = i % W;
      const int slot = t * W + it;
      uint32_t v = votes[slot];
      if (!(v & 1u)) v = 0;
      if (guess[slot] != v) atomicMin(&s_first, i);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      int it = 0;
      while (it < W && (votes[t * W + it] & 1u)) ++it;
      if (it == W) {
        atomicAdd(&s_unconv, 1u);
        it = W - 1;   // pnqp.py:82 returns i = n_iter-1
      }
      atomicAdd(&s_nqp, 1u + (unsigned)it);
    }
    __syncthreads();
    if (s_first < n) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        uint32_t v = votes[i];
        if (!(v & 1u)) v = 0;
        // moving, but the sweep exited here on a wrong guess so no Armijo pass was
        // observed: guess the overwhelmingly common "exit after the first pass".
        else if (!(guess[i] & 1u)) v = 3u;
        guess[i] = v;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    status->trace_match = (s_first >= n) ? 1u : 0u;
    status->first_mismatch = (uint32_t)s_first;
    status->any_improved = 0;
    status->n_active = 0;
    status->n_total_qp_iter = s_nqp;
    status->pnqp_unconverged = s_unconv;
    status->max_full_du = 0.0;
    status->mean_alpha = 0.0;
    status->mean_best_cost = 0.0;
    if (ctrl && s_first < n) ctrl->halt = 2u;
  }
}

static __global__ void trace_verify_kernel(uint32_t* __restrict__ guess, const uint32_t* __restrict__ votes,
                                    int T, int boxed, int solo, DilqrStatus* status,
                                    DilqrControl* ctrl = nullptr) {
  trace_verify_block<kPnqpMaxIter>(guess, votes, T, 0, boxed, solo, status, ctrl);
}

// ---------------------------------------------------------------------------
// Commit of one iLQR iteration, ONE launch (round 1 used three: trace_verify<<<1,256>>>,
// commit<<<B/128,128>>>, control<<<1,1>>>):
//   1. every block checks the replayed pnqp trace against the votes on its own (a few KB of
//      L2-resident words), so no block waits for a verdict;
//   2. per-problem best-iterate bookkeeping (mpc.py:271-285), block-level partial reductions
//      written to `part[blockIdx]`;
//   3. the block that finishes last (ticket counter) folds the partials in a fixed order,
//      corrects the trace guess on a mismatch, fills the status block and runs the stop rule
//      of the outer loop (mpc.py:266,281,299-301).
// ---------------------------------------------------------------------------
struct CommitPart {
  double du, al, bc;
  uint32_t flags;   // bit 0: some problem improved, bit 1: NaN in ||du||
  uint32_t n_active;
};
struct CommitAux {
  CommitPart* part;         // one record per block
  unsigned int* ticket;     // zero between launches
  DilqrControl* ctrl;       // may be nullptr
  int votes_are_trace;      // group sweep: the votes ARE the trace, nothing to compare
  int iteration;
  int nc;                   // n_ctrl of the runtime-dimension family (commit_kernel<S, 0, 0>)
};

template <class S, int N, int NCc>
__global__ void __launch_bounds__(128) commit_kernel(const __grid_constant__ IterParams<S> p,
                                                     const CommitAux aux) {
  const int nc = NCc ? NCc : aux.nc;
  DilqrStatus* status = reinterpret_cast<DilqrStatus*>(p.status);
  if (p.halt && *reinterpret_cast<const volatile uint32_t*>(p.halt)) return;   // uniform
  __shared__ int s_first;
  __shared__ unsigned s_nqp, s_unconv, s_last;
  __shared__ double s_du[4], s_al[4], s_bc[4];
  __shared__ unsigned s_fl[4], s_act[4];
  const int n = p.T * kPnqpMaxIter;
  const bool traced = p.bounds_kind != 0 && !p.solo;
  if (threadIdx.x == 0) {
    s_first = n;
    s_nqp = 0;
    s_unconv = 0;
  }
  __syncthreads();
  if (traced && !aux.votes_are_trace) {
    // Normalised vote of a slot: if nobody was moving the sweep left the slot right there, so
    // Armijo bits voted under a wrong "moving" guess are void.  Processing order of the sweep
    // is t = T-1 .. 0, it = 0 .. 19.
    int first = n;
#pragma unroll 4
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      const int t = p.T - 1 - i / kPnqpMaxIter, it = i % kPnqpMaxIter;
      const int slot = t * kPnqpMaxIter + it;
      uint32_t v = p.votes[slot];
      if (!(v & 1u)) v = 0;
      if (p.guess[slot] != v && i < first) first = i;
    }
    if (first < n) atomicMin(&s_first, first);
    __syncthreads();
  }
  const bool match = s_first >= n;

  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  double du = 0.0, al = 0.0, bc = 0.0;
  bool improved = false;
  bool active = false;
  if (match && b < p.B && p.solo == 2) {
    // Every problem is its own batch of one (the closed-loop driver il_env.py:96-151 calls
    // MPC with n_batch = 1): plain per-problem ||du||, and the stop rule mpc.py:266,281,
    // 299-301 per problem.  take[b]: bit 0 = take, bits 8..29 = n_not_improved, bit 30 =
    // stopped (a stopped problem keeps iterating with the others but is never taken again).
    const int state = p.take[b];
    const bool frozen = (state >> 30) & 1;
    int nni = (state >> 8) & 0x3fffff;
    S acc = S(0);
    for (int k = 0; k < p.T * nc; ++k) acc = acc + p.dusq[(size_t)k * p.B + b];
    const S dn = sqrtS<S>(acc);
    const S cn = p.cost_new[b];
    bool take = false, stop = frozen;
    if (!frozen) {
      p.du_new[b] = dn;
      nni += 1;
      if (p.first_iteration) {
        take = true;
      } else if (cn <= p.cost_best[b] + p.best_cost_eps) {
        take = true;
        improved = true;
        nni = 0;
      }
      if (take) {
        p.cost_best[b] = cn;
        p.du_best[b] = dn;
      }
      if (aux.ctrl) stop = (double)dn < aux.ctrl->eps || (uint32_t)nni > aux.ctrl->not_improved_lim;
      active = !stop;
      du = (double)dn;
      al = (double)p.alpha_new[b];
    }
    p.take[b] = (take ? 1 : 0) | (nni << 8) | (stop ? (1 << 30) : 0);
    p.cost_cur[b] = cn;
    bc = (double)p.cost_best[b];
  } else if (match && b < p.B) {
    // full_du_norm[b]: norm of row b of the [T,nc,B] squares re-read as [B, T*nc]
    // (lqr_step.py:243-245, see the note in forward_linesearch)
    {
      const int row = p.T * nc;
      const S* src = p.dusq + (size_t)b * row;
      S acc = S(0);
      int k = 0;
      for (; k + 8 <= row; k += 8) {   // eight loads in flight, summed in the same order
        S v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = src[k + j];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc = acc + v[j];
      }
      for (; k < row; ++k) acc = acc + src[k];
      p.du_new[b] = sqrtS<S>(acc);
    }
    const S cn = p.cost_new[b];
    bool take = false;
    if (p.first_iteration) {
      take = true;
    } else if (cn <= p.cost_best[b] + p.best_cost_eps) {  // mpc.py:280
      take = true;
      improved = true;
    }
    if (take) {   // best <- new   (mpc.py:272-285); the trajectory copy is deferred:
      p.cost_best[b] = cn;   // the next sweep (or finish) moves it, see IterParams::take
      p.du_best[b] = p.du_new[b];
    }
    p.take[b] = take ? 1 : 0;
    p.cost_cur[b] = cn;
    du = (double)p.du_new[b];
    al = (double)p.alpha_new[b];
    bc = (double)p.cost_best[b];
  }
  // warp reductions -> block partial
  const bool nan_du = du != du;
  for (int o = 16; o > 0; o >>= 1) {
    du = fmax(du, __shfl_xor_sync(kFull, du, o));
    al += __shfl_xor_sync(kFull, al, o);
    bc += __shfl_xor_sync(kFull, bc, o);
  }
  const unsigned imp = __ballot_sync(kFull, improved);
  const unsigned nn = __ballot_sync(kFull, nan_du);
  const unsigned act = __ballot_sync(kFull, active);
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) {
    s_du[w] = du;
    s_al[w] = al;
    s_bc[w] = bc;
    s_fl[w] = (imp ? 1u : 0u) | (nn ? 2u : 0u);
    s_act[w] = (unsigned)__popc(act);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    CommitPart r;
    r.du = fmax(fmax(s_du[0], s_du[1]), fmax(s_du[2], s_du[3]));
    r.al = (s_al[0] + s_al[1]) + (s_al[2] + s_al[3]);
    r.bc = (s_bc[0] + s_bc[1]) + (s_bc[2] + s_bc[3]);
    r.flags = s_fl[0] | s_fl[1] | s_fl[2] | s_fl[3];
    r.n_active = s_act[0] + s_act[1] + s_act[2] + s_act[3];
    aux.part[blockIdx.x] = r;
    __threadfence();
    s_last = (atomicAdd(aux.ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();

  // ---- last block: fold the partials, finish the trace bookkeeping, status + stop rule
  if (traced) {
    for (int t = threadIdx.x; t < p.T; t += blockDim.x) {
      int it = 0;
      while (it < kPnqpMaxIter && (p.votes[t * kPnqpMaxIter + it] & 1u)) ++it;
      if (it == kPnqpMaxIter) {
        atomicAdd(&s_unconv, 1u);
        it = kPnqpMaxIter - 1;   // pnqp.py:82 returns i = n_iter-1
      }
      atomicAdd(&s_nqp, 1u + (unsigned)it);
    }
    if (!match) {
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        uint32_t v = p.votes[i];
        if (!(v & 1u)) v = 0;
        // moving, but the sweep exited here on a wrong guess so no Armijo pass was
        // observed: guess the overwhelmingly common "exit after the first pass".
        else if (!(p.guess[i] & 1u)) v = 3u;
        p.guess[i] = v;
      }
    }
  }
  du = 0.0; al = 0.0; bc = 0.0;
  unsigned fl = 0, na = 0;
#pragma unroll 4
  for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) {
    const CommitPart* r = &aux.part[i];   // written by other blocks: read through L2
    du = fmax(du, __ldcg(&r->du));
    al += __ldcg(&r->al);
    bc += __ldcg(&r->bc);
    fl |= __ldcg(&r->flags);
    na += __ldcg(&r->n_active);
  }
  for (int o = 16; o > 0; o >>= 1) {
    du = fmax(du, __shfl_xor_sync(kFull, du, o));
    al += __shfl_xor_sync(kFull, al, o);
    bc += __shfl_xor_sync(kFull, bc, o);
    fl |= __shfl_xor_sync(kFull, fl, o);
    na += __shfl_xor_sync(kFull, na, o);
  }
  if ((threadIdx.x & 31) == 0) {
    s_du[w] = du;
    s_al[w] = al;
    s_bc[w] = bc;
    s_fl[w] = fl;
    s_act[w] = na;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  du = fmax(fmax(s_du[0], s_du[1]), fmax(s_du[2], s_du[3]));
  al = (s_al[0] + s_al[1]) + (s_al[2] + s_al[3]);
  bc = (s_bc[0] + s_bc[1]) + (s_bc[2] + s_bc[3]);
  fl = s_fl[0] | s_fl[1] | s_fl[2] | s_fl[3];
  na = s_act[0] + s_act[1] + s_act[2] + s_act[3];
  if (fl & 2u) du = __longlong_as_double(0x7ff8000000000000LL);  // propagate NaN like python max()
  *aux.ticket = 0u;
  status->trace_match = match ? 1u : 0u;
  status->first_mismatch = (uint32_t)s_first;
  status->n_total_qp_iter = s_nqp;
  status->pnqp_unconverged = s_unconv;
  status->any_improved = match ? (fl & 1u) : 0u;
  status->n_active = match ? na : 0u;
  status->max_full_du = match ? du : 0.0;
  status->mean_alpha = match ? al / p.B : 0.0;
  status->mean_best_cost = match ? bc / p.B : 0.0;
  DilqrControl* ctrl = aux.ctrl;
  if (!ctrl) return;
  if (!match) {
    ctrl->halt = 2u;
    return;
  }
  // device-side stop rule of the outer loop (mpc.py:266,281,299-301)
  if (p.solo == 2) {   // per-problem stop rule above; halt once nobody is left
    ctrl->iters_done = (uint32_t)aux.iteration + 1u;
    if (na == 0u) ctrl->halt = 1u;
    return;
  }
  uint32_t nni = ctrl->n_not_improved + 1u;
  if (aux.iteration > 0 && (fl & 1u)) nni = 0u;
  ctrl->n_not_improved = nni;
  ctrl->iters_done = (uint32_t)aux.iteration + 1u;
  // the comparison of mpc.py:299 is on the python max() of the batch: NaN never compares below eps
  if (du < ctrl->eps || nni > ctrl->not_improved_lim) ctrl->halt = 1u;
}

// ---------------------------------------------------------------------------
// Gather the best iterate into the API (AoS) layout  (mpc.py:304-306).
// One thread per (t, b); workspace reads are coalesced, the AoS writes are
// contiguous per warp (consecutive b).
// ---------------------------------------------------------------------------
// NS_ = NC_ = 0: the runtime-dimension family (rt_kernels.cuh), shape given as ns_rt, nc_rt
template <class S, int NS_, int NC_>
__global__ void finish_kernel(const __grid_constant__ IterParams<S> p, int ns_rt, int nc_rt) {
  const int NS = NS_ ? NS_ : ns_rt, NC = NC_ ? NC_ : nc_rt;
  const int N = NS + NC;
  const int NK = NC * NS + NC;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int t = blockIdx.y;
  if (b >= p.B) return;
  // best iterate: parked in traj_best, or still the latest trajectory (take flag).  With a
  // device-side outer loop (DilqrControl) the host may not know yet how many iterations were
  // committed: the latest trajectory is the one iteration iters_done-1 wrote.
  const S* latest = p.traj_new;
  if (p.control) {
    const int it = (int)reinterpret_cast<const DilqrControl*>(p.control)->iters_done - 1;
    latest = p.traj_buf[(it + 1) & 1];
  }
  const S* src = ((p.take[b] & 1) ? latest : p.traj_best) + bidx(t, 0, N, b, p.nW);
  if (p.x_out) {
#pragma unroll
    for (int i = 0; i < NS; ++i) p.x_out[((size_t)t * p.B + b) * NS + i] = src[i * kWarp];
  }
  if (p.u_out) {
#pragma unroll
    for (int a = 0; a < NC; ++a) p.u_out[((size_t)t * p.B + b) * NC + a] = src[(NS + a) * kWarp];
  }
  const S* ks = p.Kk + bidx(t, 0, NK, b, p.nW);
  if (p.K_out) {
#pragma unroll
    for (int e = 0; e < NC * NS; ++e) p.K_out[((size_t)t * p.B + b) * (NC * NS) + e] = ks[e * kWarp];
  }
  if (p.k_out) {
#pragma unroll
    for (int a = 0; a < NC; ++a)
      p.k_out[((size_t)t * p.B + b) * NC + a] = ks[(NC * NS + a) * kWarp];
  }
  if (t == 0) {
    if (p.cost_out) p.cost_out[b] = p.cost_best[b];
    if (p.du_out) p.du_out[b] = p.du_best[b];
    if (p.alpha_out) p.alpha_out[b] = p.alpha_new[b];
  }
}

// ---------------------------------------------------------------------------
// Analytic linearisation F_t = D(x_t,u_t), f_t = step(x_t,u_t) - D tau_t
// (mpc_explicit.py:516-546) for t < T-1.  One thread per (t, b).
// ---------------------------------------------------------------------------
template <class S, int DYN>
__global__ void linearize_kernel(DynParams<S> P, int T, int B, const S* __restrict__ x,
                                 const S* __restrict__ u, S* __restrict__ F, S* __restrict__ f) {
  using D = Dyn<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC, N = D::N;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int t = blockIdx.y;
  if (b >= B || t >= T - 1) return;
  S tau[N], xn[NS], Fm[NS][N];
#pragma unroll
  for (int i = 0; i < NS; ++i) tau[i] = x[((size_t)t * B + b) * NS + i];
#pragma unroll
  for (int a = 0; a < NC; ++a) tau[NS + a] = u[((size_t)t * B + b) * NC + a];
  D::step(P, tau, &tau[NS], xn);
  D::jacobian(P, tau, xn, Fm);   // sin/cos of the new angle come from xn (same rollout)
  S* Fo = F + ((size_t)t * B + b) * (NS * N);
#pragma unroll
  for (int i = 0; i < NS; ++i) {
    S acc = S(0);
#pragma unroll
    for (int j = 0; j < N; ++j) {
      Fo[i * N + j] = Fm[i][j];
      acc = fmaS<S>(Fm[i][j], tau[j], acc);
    }
    if (f) f[((size_t)t * B + b) * NS + i] = xn[i] - acc;
  }
}

// nominal rollout (util.py:104-127), one thread per problem
template <class S, int DYN>
__global__ void rollout_kernel(DynParams<S> P, int T, int B, const S* __restrict__ x_init,
                               const S* __restrict__ u, S* __restrict__ x) {
  using D = Dyn<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  S xc[NS], uc[NC], xn[NS];
#pragma unroll
  for (int i = 0; i < NS; ++i) xc[i] = x_init[(size_t)b * NS + i];
  for (int t = 0; t < T; ++t) {
#pragma unroll
    for (int i = 0; i < NS; ++i) x[((size_t)t * B + b) * NS + i] = xc[i];
    if (t < T - 1) {
#pragma unroll
      for (int a = 0; a < NC; ++a) uc[a] = u[((size_t)t * B + b) * NC + a];
      D::step(P, xc, uc, xn);
#pragma unroll
      for (int i = 0; i < NS; ++i) xc[i] = xn[i];
    }
  }
}

// ---------------------------------------------------------------------------
// KKT gradient assembly (lqr_step.py:343-404): costates lambda / dlambda by a
// reverse sweep, then
//   dC_t = -1/2 (dtau tau' + tau dtau')   dc_t = -dtau
//   dF_t = -(dlam_{t+1} tau_t' + lam_{t+1} dtau_t')   df_t = -dlam_{t+1}
//   dx_init = -dlam_0.
// One thread per problem.
// ---------------------------------------------------------------------------
template <class S, int NS, int NC>
__global__ void __launch_bounds__(128) kkt_grads_kernel(const __grid_constant__ DilqrKkt k) {
  constexpr int N = NS + NC;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int T = k.T, B = k.n_batch;
  if (b >= B) return;
  const S* C = static_cast<const S*>(k.C);
  const S* c = static_cast<const S*>(k.c);
  const S* F = static_cast<const S*>(k.F);
  const S* x = static_cast<const S*>(k.x);
  const S* u = static_cast<const S*>(k.u);
  const S* dx = static_cast<const S*>(k.dx);
  const S* du = static_cast<const S*>(k.du);
  const S* r = static_cast<const S*>(k.r);
  S* dC = static_cast<S*>(k.dC);
  S* dc = static_cast<S*>(k.dc);
  S* dF = static_cast<S*>(k.dF);
  S* df = static_cast<S*>(k.df);
  S* dx0 = static_cast<S*>(k.dx_init);
  S lam[NS], dlam[NS];
  for (int t = T - 1; t >= 0; --t) {
    const size_t tb = (size_t)t * B + b;
    S tau[N], dtau[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      tau[i] = x[tb * NS + i];
      dtau[i] = dx[tb * NS + i];
    }
#pragma unroll
    for (int a = 0; a < NC; ++a) {
      tau[NS + a] = u[tb * NC + a];
      dtau[NS + a] = du[tb * NC + a];
    }
    // gradients that pair step t with the costates of t+1 (held in lam/dlam)
    if (t < T - 1) {
      if (dF) {
#pragma unroll
        for (int i = 0; i < NS; ++i)
#pragma unroll
          for (int j = 0; j < N; ++j)
            dF[tb * (NS * N) + i * N + j] = -(dlam[i] * tau[j] + lam[i] * dtau[j]);
      }
      if (df) {
#pragma unroll
        for (int i = 0; i < NS; ++i) df[tb * NS + i] = -dlam[i];
      }
    }
    if (dC) {
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j)
          dC[tb * (N * N) + i * N + j] = S(-0.5) * (dtau[i] * tau[j] + tau[i] * dtau[j]);
    }
    if (dc) {
#pragma unroll
      for (int i = 0; i < N; ++i) dc[tb * N + i] = -dtau[i];
    }
    // lam_t = Cxx x + Cxu u + c_x + Fx' lam_{t+1}   (lqr_step.py:355-369)
    S nl[NS], ndl[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      S a1 = S(0), a2 = S(0), d1 = S(0), d2 = S(0);
#pragma unroll
      for (int j = 0; j < NS; ++j) {
        const S cij = C[tb * (N * N) + i * N + j];
        a1 = fmaS<S>(cij, tau[j], a1);
        d1 = fmaS<S>(cij, dtau[j], d1);
      }
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        const S cij = C[tb * (N * N) + i * N + NS + a];
        a2 = fmaS<S>(cij, tau[NS + a], a2);
        d2 = fmaS<S>(cij, dtau[NS + a], d2);
      }
      nl[i] = (a1 + a2) + c[tb * N + i];
      ndl[i] = (d1 + d2) - r[tb * N + i];
    }
    if (t < T - 1) {
#pragma unroll
      for (int i = 0; i < NS; ++i) {
        S a1 = S(0), d1 = S(0);
#pragma unroll
        for (int l = 0; l < NS; ++l) {
          const S fli = F[tb * (NS * N) + l * N + i];
          a1 = fmaS<S>(fli, lam[l], a1);
          d1 = fmaS<S>(fli, dlam[l], d1);
        }
        nl[i] = nl[i] + a1;
        ndl[i] = ndl[i] + d1;
      }
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      lam[i] = nl[i];
      dlam[i] = ndl[i];
    }
  }
  if (dx0) {
#pragma unroll
    for (int i = 0; i < NS; ++i) dx0[(size_t)b * NS + i] = -dlam[i];
  }
}

}  // namespace dilqr

namespace dilqr {

// ---------------------------------------------------------------------------
// Standalone projected-Newton box QP (pnqp.py:5-82), one thread per problem,
// batch-global control flow replayed from a 20-word trace exactly like the fused
// sweep.  Outputs: x[B,n], LU[B,n,n] + pivots[B,n] (LAPACK getrf layout, 1-based
// pivots == what Tensor.lu() returns; for n == 1 LU is the scalar H_), If[B,n].
// ---------------------------------------------------------------------------
template <class S, int N>
__global__ void pnqp_kernel(int B, const S* __restrict__ H, const S* __restrict__ q,
                            const S* __restrict__ lower, const S* __restrict__ upper,
                            const S* __restrict__ x_init, S* __restrict__ x_out,
                            S* __restrict__ lu_out, int32_t* __restrict__ piv_out,
                            S* __restrict__ if_out, const uint32_t* __restrict__ guess,
                            uint32_t* __restrict__ votes, int solo) {
  const int lane = threadIdx.x & 31;
  const int b0 = (blockIdx.x * blockDim.x + threadIdx.x) - lane;
  if (b0 >= B) return;
  const bool active = b0 + lane < B;
  const int b = active ? b0 + lane : b0;
  S Hm[N][N], qv[N], lo[N], hi[N], x[N];
  bool If[N];
#pragma unroll
  for (int i = 0; i < N; ++i) {
#pragma unroll
    for (int j = 0; j < N; ++j) Hm[i][j] = H[((size_t)b * N + i) * N + j];
    qv[i] = q[(size_t)b * N + i];
    lo[i] = lower[(size_t)b * N + i];
    hi[i] = upper[(size_t)b * N + i];
    x[i] = x_init ? x_init[(size_t)b * N + i] : S(0);
  }
  LUpp<S, N> lu;
  const uint4 gpre = solo ? make_uint4(0, 0, 0, 0) : __ldg(reinterpret_cast<const uint4*>(guess));
  pnqp_thread<S, N>(Hm, qv, lo, hi, x_init != nullptr, x, If, lu, guess, gpre, votes, solo != 0,
                    active, lane);
  if (!active) return;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    x_out[(size_t)b * N + i] = x[i];
    if_out[(size_t)b * N + i] = If[i] ? S(1) : S(0);
    piv_out[(size_t)b * N + i] = (N == 1) ? 1 : lu.piv[i] + 1;
#pragma unroll
    for (int j = 0; j < N; ++j) lu_out[((size_t)b * N + i) * N + j] = lu.a[i][j];
  }
}

}  // namespace dilqr
