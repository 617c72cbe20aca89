// ilqr_kernels.cuh -- the batched box-constrained iLQR iteration for sm_100a.
//
// Mapping: ONE THREAD PER MPC PROBLEM (n_tau <= ~10: the whole Riccati state of
// a problem -- V, v, Q, q, K, k -- lives in that thread's registers), warps are
// fully independent (no block-level synchronisation), and each warp streams the
// API's time-major AoS tensors (C, c, F, f) one timestep at a time through a
// double-buffered shared-memory stage filled by 1-D bulk TMA copies
// (cp.async.bulk + mbarrier, see WarpStager).  Everything private to the solver
// (trajectories, gains, per-problem bookkeeping) is kept in a warp-blocked SoA
// workspace [T][B/32][component][32]: per-thread accesses are perfectly coalesced
// AND the chunk a warp needs for one timestep is contiguous, so it rides the same
// TMA stage as the API slabs -- every per-timestep operand of the sweep arrives in
// shared memory one step ahead of its use.
//
// Tensor cores are deliberately not used: the per-problem matrices are at most
// ~16x16, strictly sequential in t, and every problem has different operands.
//
// Reference semantics implemented here (file:line relative to the reference):
//   LQRStepFn.forward            lqr_step.py:277-309
//   lqr_backward (Riccati)       lqr_step.py:52-160, lqr_step_backup.py:163-259
//   pnqp                         pnqp.py:5-82
//   lqr_forward (line search)    lqr_step.py:164-261
//   get_traj / get_cost          util.py:104-153
//   ANALYTIC linearisation       mpc_explicit.py:516-546
//   best-iterate bookkeeping     mpc.py:271-285
//
// Batch-global control flow.  pnqp terminates, and runs its Armijo loop, on
// batch-wide reductions (pnqp.py:56-59,65,75).  Threads cannot see the batch, so
// the kernel REPLAYS a guessed control-flow trace (one 32-bit word per
// (timestep, pnqp iteration): bit0 = "some problem still moving", bit 1+c =
// "Armijo loop exits after pass c") and every warp ORs what it actually observed
// into a vote array.  The commit step compares votes with the guess; they are
// equal up to the first wrong guess, so after at most a few re-runs (normally
// zero: the trace of the previous iLQR iteration is the next guess) the result
// is exactly what the reference computes on the whole batch.
#pragma once
#include "common.cuh"
#include "dynamics.cuh"
#include "env_tables_gen.cuh"
#include "smallmat.cuh"

namespace dilqr {

template <class S>
struct IterParams {
  int sym_pair;      // this launch is one of a (symmetric, general) pair: see IterKernel::kSym
  int T, B, Bp;
  int bounds_kind;   // 0 none, 1 scalar, 2 tensor
  int solo;
  int gain_solve;
  int max_ls;
  int has_f;
  int first_iteration;
  S lo, hi;
  S delta_u;        // trust region on the control change (lqr_step.py:132-134,204-211)
  int has_delta;
  S decay;
  S best_cost_eps;
  const S* lo_t;
  const S* hi_t;
  const uint8_t* zeroI;
  const S* x_init;
  const S* C;
  const S* c;
  const S* F;
  const S* f;
  const S* u_init;
  const S* x_cur;
  S* Cpk;             // [T][Bp/32][N(N+1)/2][32] upper triangle of C, written by begin when
                      // every C[t,b] is bitwise symmetric (see cpk_state)
  uint32_t* cpk_state;  // 1: Cpk is valid and the sweeps stream it instead of the dense C
  const S* traj_cur;  // [T][Bp/32][N][32]  current iterate (read)
  S* traj_new;        // [T][Bp/32][N][32]  new iterate (written)
  S* traj_best;       // [T][Bp/32][N][32]  best iterate so far
  S* traj_buf[2];     // the two ping-pong buffers (finish picks by the device-side iteration count)
  S* Kk;              // [T][Bp/32][NC*NS+NC][32]
  int nW;             // Bp / 32
  S* dusq;            // [T][NC][B] squared control changes of the first line-search pass
  int* take;          // [Bp] 1: the problem's best iterate is the CURRENT trajectory and
                      //         has not been copied to traj_best yet (lazy best tracking)
  int gains_only;     // skip the line-search rollout (only K,k are wanted)
  int votes_are_trace;  // the group sweep resolved the pnqp decisions at barriers: no replay
  int C_bcast, c_bcast;  // cost layout: 0 dense [T,B,..], 1 batch-broadcast [T,..], 2 [..] only
  S* cost_cur;    // [Bp]
  S* cost_new;
  S* cost_best;
  S* du_new;
  S* du_best;
  S* alpha_new;
  uint32_t* guess;  // [T][kPnqpMaxIter]
  uint32_t* votes;  // [T][kPnqpMaxIter]
  void* status;     // DilqrStatus*
  const uint32_t* halt;  // DilqrControl::halt (or nullptr): non-zero -> this launch is a no-op
  void* control;    // DilqrControl*
  S* x_out;
  S* u_out;
  S* cost_out;
  S* du_out;
  S* alpha_out;
  S* K_out;
  S* k_out;
  S* lam_blk;   // gains-at-the-solution sweep: primal costates [T][Bp/32][NS][32] (optional)
  S* gsQ;       // group sweep (group_kernels.cuh): per-problem record Q_t[N][N], q_t[N]
  S* gsG;       // group sweep: rows n_state.. of Q_t and q_u, lane-interleaved [Bp/32][NC*N+NC][32]
  unsigned int* gs_barrier;   // group sweep: SubBarrier counter (zeroed before the launch)
  DynParams<S> dyn;
};

// ---------------------------------------------------------------------------
// stage cost  0.5 tau' C tau + c' tau   (util.py:145-147: bquad then bdot)
// C, c are this lane's blocks in shared memory (row-major).
// ---------------------------------------------------------------------------
// Source of the cost block(s) of timestep t for the warp starting at problem b0
// (dense: the warp's slab; broadcast: the single shared block, mpc.py:205-219).
template <class S>
DILQR_DEVICE const S* cost_src(const S* base, int bcast, int t, int B, int b0, int elems) {
  return bcast == 0 ? base + ((size_t)t * B + b0) * elems
                    : (bcast == 1 ? base + (size_t)t * elems : base);
}

template <class S, int N>
DILQR_DEVICE S stage_cost(const S* __restrict__ Cs, const S* __restrict__ cs, const S* tau) {
  S quad = S(0);
#pragma unroll
  for (int j = 0; j < N; ++j) {
    S row = S(0);
#pragma unroll
    for (int i = 0; i < N; ++i) row = fmaS<S>(tau[i], Cs[i * N + j], row);
    quad = fmaS<S>(row, tau[j], quad);
  }
  S dot = S(0);
#pragma unroll
  for (int i = 0; i < N; ++i) dot = fmaS<S>(tau[i], cs[i], dot);
  return S(0.5) * quad + dot;
}

// Slot of C[i][j] in the packed upper triangle (row-major over i <= j).
template <int N>
DILQR_DEVICE constexpr int pk_idx(int i, int j) {
  return i <= j ? i * N - (i * (i - 1)) / 2 + (j - i) : j * N - (j * (j - 1)) / 2 + (i - j);
}

// stage_cost on the packed, lane-interleaved copy: the same operations in the same order
// (C[j][i] is read from the slot of C[i][j]; the two are bitwise equal when Cpk is valid).
template <class S, int N>
DILQR_DEVICE S stage_cost_packed(const S* __restrict__ Cp, const S* __restrict__ cs, const S* tau) {
  S quad = S(0);
#pragma unroll
  for (int j = 0; j < N; ++j) {
    S row = S(0);
#pragma unroll
    for (int i = 0; i < N; ++i) row = fmaS<S>(tau[i], Cp[pk_idx<N>(i, j) * kWarp], row);
    quad = fmaS<S>(row, tau[j], quad);
  }
  S dot = S(0);
#pragma unroll
  for (int i = 0; i < N; ++i) dot = fmaS<S>(tau[i], cs[i], dot);
  return S(0.5) * quad + dot;
}

// LinDx step  x' = F tau (+ f)    (util.py:117-121)
template <class S, int NS, int N>
DILQR_DEVICE void lin_step(const S* __restrict__ Fs, const S* __restrict__ fs, bool has_f,
                           const S* tau, S* xn) {
#pragma unroll
  for (int i = 0; i < NS; ++i) {
    S acc = S(0);
#pragma unroll
    for (int j = 0; j < N; ++j) acc = fmaS<S>(Fs[i * N + j], tau[j], acc);
    if (has_f) acc = acc + fs[i];
    xn[i] = acc;
  }
}

// ---------------------------------------------------------------------------
// pnqp for one problem, replaying / voting the batch-global control flow.
// (pnqp.py:5-82).  On return x is the solution, If the free-set mask and lu the
// LU factors (N>1) or scalar (N==1, lu.a[0][0]) of the masked Hessian of the
// last evaluated iteration -- exactly what lqr_backward consumes
// (lqr_step.py:135-148).
// ---------------------------------------------------------------------------
// Barrier among the first `n` blocks of a (co-resident) grid: one monotonically increasing
// counter in global memory, episode k is complete once it reaches k * n.  Used by the group
// sweep for the pnqp decisions, which only involve the blocks that own problems (a fraction
// of the grid, so it is cheaper than a full grid.sync and the other blocks stay out of it).
// Fire-and-forget OR into a vote word: a RED has no destination register, so nothing in the
// sweep ever waits for the L2 round trip of the (heavily shared) word.
DILQR_DEVICE void vote_or(uint32_t* word, uint32_t bits) {
  asm volatile("red.relaxed.gpu.global.or.b32 [%0], %1;" ::"l"(word), "r"(bits) : "memory");
}

struct SubBarrier {
  unsigned int* counter;   // zeroed before the launch
  unsigned int n;
  unsigned int episode;
  DILQR_DEVICE void sync() {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned int target = (++episode) * n;
      atomicAdd(counter, 1u);
      while (*reinterpret_cast<volatile unsigned int*>(counter) < target) {
      }
      __threadfence();
    }
    __syncthreads();
  }
};

// BARRIER: false replays a guessed trace; true decides with a SubBarrier (`sb`).
template <class S, int N, bool BARRIER = false>
DILQR_DEVICE void pnqp_thread(const S (&H)[N][N], const S (&q)[N], const S (&lo)[N],
                              const S (&hi)[N], bool have_init, S (&x)[N], bool (&If)[N],
                              LUpp<S, N>& lu, const uint32_t* __restrict__ guess, uint4 gpre,
                              uint32_t* __restrict__ votes, bool solo, bool active, int lane,
                              S* rinv_out = nullptr, SubBarrier* sb = nullptr) {
  // N == 1: 1 / (masked Hessian) of the last evaluated iteration, handed to the caller
  // (which needs the same quotient for K, lqr_step.py:144-146) and reused across
  // iterations while the operand is unchanged -- same value, one division instead of three.
  S h_last = S(0), r_last = S(0);
  bool have_r = false;
  // BARRIER: every batch-global decision is an atomicOr into the vote word + a barrier over
  // the whole batch (no guessing, no re-runs) -- the better trade when the control-flow
  // trace is long and unstable (multi-input problems with many active constraints).
  auto grid_decide = [&](uint32_t* word, uint32_t mine) -> uint32_t {
    if constexpr (BARRIER) {
      if (mine && lane == 0) atomicOr(word, mine);
      sb->sync();
      return *reinterpret_cast<volatile uint32_t*>(word);
    } else {
      return 0u;
    }
  };
  // gpre.x/.y = guess[0..1], obtained by the caller without a global load at this point (the
  // common case never looks past the first two words; an L2 round trip here would sit on the
  // critical path of the sweep).
  auto gword_at = [&](int it) -> uint32_t {
    return it == 0 ? gpre.x : it == 1 ? gpre.y : __ldg(&guess[it]);
  };
  const S GAMMA = S(0.1);
  if (!have_init) {  // pnqp.py:14-19
    if (N == 1) {
      x[0] = -(S(1) / H[0][0]) * q[0];
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) lu.a[i][j] = H[i][j];
        x[i] = q[i];
      }
      lu.factor();
      lu.solve(x);
#pragma unroll
      for (int i = 0; i < N; ++i) x[i] = -x[i];
    }
  }
#pragma unroll
  for (int i = 0; i < N; ++i) x[i] = eclamp<S>(x[i], lo[i], hi[i]);  // pnqp.py:23

  for (int it = 0; it < kPnqpMaxIter; ++it) {
    S g[N], dx[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {  // g = H x + q   (pnqp.py:29)
      S acc = S(0);
#pragma unroll
      for (int j = 0; j < N; ++j) acc = fmaS<S>(H[i][j], x[j], acc);
      g[i] = acc + q[i];
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {  // pnqp.py:32-33
      const bool Ic = ((x[i] == lo[i]) && (g[i] > S(0))) || ((x[i] == hi[i]) && (g[i] < S(0)));
      If[i] = !Ic;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {  // pnqp.py:44-48
#pragma unroll
      for (int j = 0; j < N; ++j) {
        S h = (If[i] && If[j]) ? H[i][j] : S(0);
        if (i == j) h = h + S(1e-11);
        lu.a[i][j] = h;
      }
      dx[i] = If[i] ? g[i] : S(0);
    }
    if (N == 1) {  // pnqp.py:50-51
      if (!(have_r && lu.a[0][0] == h_last)) {
        h_last = lu.a[0][0];
        r_last = S(1) / h_last;
        have_r = true;
      }
      if (rinv_out) *rinv_out = r_last;
      dx[0] = -r_last * dx[0];
    } else {
      lu.factor();
      lu.solve(dx);
#pragma unroll
      for (int i = 0; i < N; ++i) dx[i] = -dx[i];
    }
    S nrm2 = S(0);
#pragma unroll
    for (int i = 0; i < N; ++i) nrm2 = fmaS<S>(dx[i], dx[i], nrm2);
    // pnqp.py:56.  N == 1: sqrt(dx*dx) == |dx| exactly (correctly rounded square root of a
    // correctly rounded square; in the under/overflow ranges both sides of the test agree)
    const bool J = (N == 1) ? (absS<S>(dx[0]) >= S(1e-4)) : (sqrtS<S>(nrm2) >= S(1e-4));
    uint32_t vote = 0;
    bool any_moving;
    if (solo) {
      any_moving = J;
    } else if (BARRIER) {
      if (__ballot_sync(kFull, active && J)) vote |= 1u;
      any_moving = (grid_decide(&votes[it], vote) & 1u) != 0;
    } else {
      if (__ballot_sync(kFull, active && J)) vote |= 1u;
      any_moving = (gword_at(it) & 1u) != 0;
    }
    if (!any_moving) {  // pnqp.py:57-59
      if (!solo && !BARRIER && vote && lane == 0) vote_or(&votes[it], vote);
      return;
    }
    // Armijo backtracking with a batch-global exit test (pnqp.py:61-76).
    S fx = S(0);
    {
      S quad = S(0), dot = S(0);
#pragma unroll
      for (int j = 0; j < N; ++j) {
        S row = S(0);
#pragma unroll
        for (int i = 0; i < N; ++i) row = fmaS<S>(x[i], H[i][j], row);
        quad = fmaS<S>(row, x[j], quad);
      }
#pragma unroll
      for (int i = 0; i < N; ++i) dot = fmaS<S>(q[i], x[i], dot);
      fx = S(0.5) * quad + dot;
    }
    S alpha = S(1);
    S mx[N];
    const uint32_t gword = (solo || BARRIER) ? 0u : gword_at(it);
    for (int cnt = 0; cnt < kArmijoMax; ++cnt) {
#pragma unroll
      for (int i = 0; i < N; ++i) mx[i] = eclamp<S>(x[i] + alpha * dx[i], lo[i], hi[i]);
      S arm = GAMMA + S(1e-6);
      if (J) {
        S quad = S(0), dot = S(0), gd = S(0);
#pragma unroll
        for (int j = 0; j < N; ++j) {
          S row = S(0);
#pragma unroll
          for (int i = 0; i < N; ++i) row = fmaS<S>(mx[i], H[i][j], row);
          quad = fmaS<S>(row, mx[j], quad);
        }
#pragma unroll
        for (int i = 0; i < N; ++i) dot = fmaS<S>(q[i], mx[i], dot);
#pragma unroll
        for (int i = 0; i < N; ++i) gd = fmaS<S>(g[i], x[i] - mx[i], gd);
        arm = (fx - (S(0.5) * quad + dot)) / gd;
      }
      const bool small = arm <= GAMMA;   // pnqp.py:73
      if (small) alpha = alpha * S(0.1);
      bool exit_loop;
      if (solo) {
        exit_loop = !small;
      } else if (BARRIER) {
        const uint32_t mine = __ballot_sync(kFull, active && !small) ? (2u << cnt) : 0u;
        exit_loop = (grid_decide(&votes[it], mine) >> (1 + cnt)) & 1u;
      } else {
        // max_armijo > GAMMA  <=>  some problem has !(arm <= GAMMA)
        if (__ballot_sync(kFull, active && !small)) vote |= (2u << cnt);
        exit_loop = (gword >> (1 + cnt)) & 1u;
      }
      if (exit_loop) break;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) x[i] = mx[i];  // pnqp.py:78
    if (!solo && !BARRIER && vote && lane == 0) vote_or(&votes[it], vote);
  }
  // fell through n_iter iterations: the reference returns the factors / If of the
  // last iteration together with the stepped x (pnqp.py:81-82).
}

// ---------------------------------------------------------------------------
// The fused iLQR iteration.
// ---------------------------------------------------------------------------
// Association of the Riccati update.  0: every product of lqr_step.py:66-70,155-158 is rounded
// on its own and the terms are added in the reference's order (what torch computes op by
// op).  1: the same terms accumulated as ONE fused-multiply-add chain per entry (the addend
// C_ij / q_i / Q_ij opens the chain): ~14 % fewer FP64 instructions in the sweep and fewer
// roundings; results differ from mode 0 by a few ulp (both are within the rounding error of
// the reference's own BLAS-ordered sums).
#ifndef DILQR_CHAIN_FMA
#define DILQR_CHAIN_FMA 1
#endif
constexpr bool kChainFmaOn = DILQR_CHAIN_FMA != 0;
// Symmetric Riccati update (env models, with the chained association): Q_t and V_t are formed
// for j >= i only and mirrored.  C_t comes from the packed copy (bitwise symmetric), F'VF and the
// V update are symmetric in exact arithmetic; the reference's batched matmuls round Q_ij and Q_ji
// independently (differences of an ulp), which this makes unobservable.  Only valid when C_t
// is symmetric: the SYM kernels run iff begin found every block bitwise symmetric (packed copy
// valid); the host enqueues the pair (SYM, general) and the one that does not apply exits at
// once (the flag lives on the device, the host never reads it).  15 % fewer FP64 instructions
// in the sweep, 242 -> 206 registers.
#ifndef DILQR_SYM_RICCATI
#define DILQR_SYM_RICCATI 1
#endif
constexpr bool kSymRiccatiOn = DILQR_SYM_RICCATI != 0;

template <class S, int NS, int NC, int DYN, bool STAGED, bool SYM = false>
struct IterKernel {
  static constexpr int N = NS + NC;
  static constexpr int NK = NC * NS + NC;
  static constexpr bool kEnv = (DYN != DYN_LINDX);
  // env_dx models only: user-supplied LinDx problems keep the op-by-op association (their
  // parity tests pin pnqp iteration counts on borderline |dx| >= 1e-4 decisions)
  static constexpr bool kChainFma = kChainFmaOn && kEnv;
  static constexpr bool kSym = SYM && kSymRiccatiOn && kChainFma && STAGED;
  using D = Dyn<S, DYN>;
  // stage segments: 0 C[n*n]  1 c[n]  2 F[ns*n]  3 f[ns]  (API slabs)
  //                 4 traj_cur[t] chunk [N][32]   5 Kk[t] chunk [NK][32]   (workspace)
  static constexpr int kNSeg = 6;
  static constexpr uint32_t kFullMask = (1u << 4) | (1u << 5);
  static constexpr int NP = N * (N + 1) / 2;   // packed symmetric C

  // Does this launch stream the packed copy of C?  (uniform over the grid)
  DILQR_DEVICE static bool use_packed(const IterParams<S>& p) {
    return STAGED && p.cpk_state && !p.C_bcast && *reinterpret_cast<const volatile uint32_t*>(p.cpk_state) == 1u;
  }

  // Is every C block known to be bitwise symmetric?  (state 1: begin packed the dense tensor and
  // found it symmetric; state 3: begin checked the broadcast block(s).)  Uniform over the grid.
  DILQR_DEVICE static bool sym_ok(const IterParams<S>& p) {
    if (!STAGED || !p.cpk_state) return false;
    const uint32_t v = *reinterpret_cast<const volatile uint32_t*>(p.cpk_state);
    return p.C_bcast ? v == 3u : v == 1u;
  }

  // Same question for the kernels that read their operands straight from global memory.
  DILQR_DEVICE static bool use_packed_direct(const IterParams<S>& p) {
    return !p.C_bcast && p.cpk_state &&
           *reinterpret_cast<const volatile uint32_t*>(p.cpk_state) == 1u;
  }

  // Non-staged rollout: ask L2 for the operands of timestep t (this warp's chunks / slabs)
  // one timestep before they are loaded -- the loads then cost an L2 hit, not a DRAM round trip.
  DILQR_DEVICE static void prefetch_span_l2(const void* base, size_t bytes, int lane) {
    const char* pc = static_cast<const char*>(base);
    for (size_t o = (size_t)lane * 128; o < bytes; o += 32 * 128)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(pc + o));
  }
  DILQR_DEVICE static void prefetch_step_l2(const IterParams<S>& p, const WarpStager<S>& st, int t,
                                            int b0, int lane) {
    const int nvalid = min(kWarp, p.B - b0);
    if ((st.seg_full >> 0) & 1u)
      prefetch_span_l2(p.Cpk + bidx(t, 0, NP, b0, p.nW), (size_t)NP * kWarp * sizeof(S), lane);
    else if (!p.C_bcast)
      prefetch_span_l2(cost_src<S>(p.C, 0, t, p.B, b0, N * N), (size_t)nvalid * N * N * sizeof(S), lane);
    if (!p.c_bcast)
      prefetch_span_l2(cost_src<S>(p.c, 0, t, p.B, b0, N), (size_t)nvalid * N * sizeof(S), lane);
    prefetch_span_l2(p.traj_cur + bidx(t, 0, N, b0, p.nW), (size_t)N * kWarp * sizeof(S), lane);
    prefetch_span_l2(p.Kk + bidx(t, 0, NK, b0, p.nW), (size_t)NK * kWarp * sizeof(S), lane);
  }

  // sol: the sweep runs at a given solution handed over in the API layout (x_out[T,B,ns],
  // u_out[T,B,nc]): segments 2 / 3 carry those slabs, the workspace chunks are not staged
  static __host__ __device__ void seg_elems(uint32_t* e, bool sol = false) {
    e[0] = N * N;
    e[1] = N;
    e[2] = sol ? NS : (kEnv ? 0 : NS * N);
    e[3] = sol ? NC : (kEnv ? 0 : NS);
    e[4] = sol ? 0 : N;
    e[5] = sol ? 0 : NK;
  }
  static __host__ __device__ size_t smem_per_warp(bool sol = false) {
    if (!STAGED) return 0;
    uint32_t e[kNSeg];
    seg_elems(e, sol);
    return WarpStager<S>::bytes_per_warp(kNSeg, e) + kStages * sizeof(uint64_t);
  }

  // Per-lane view of the operands of timestep t: staged copies in shared memory, or
  // (shapes too large to stage) straight global memory.  C,c,F,f are this lane's
  // row-major blocks; tau / Kk are lane-interleaved (element e at [e * tstride]).
  struct Blk {
    const S* C;       // dense: this lane's row-major block; packed: slot e at C[e * 32]
    bool packed;
    const S* c;
    const S* F;
    const S* f;
    const S* tau;
    const S* Kk;
    const S* xs;      // SOL sweeps: this lane's x_t[NS] / u_t[NC] of the API slabs
    const S* us;
    int tstride;
  };
  template <bool SOL = false>
  DILQR_DEVICE static Blk blocks(const IterParams<S>& p, const WarpStager<S>& st, int sg, int t,
                                 int b, int bw, int lane) {
    Blk k;
    k.packed = STAGED && ((st.seg_full >> 0) & 1u);
    k.xs = k.us = nullptr;
    if (STAGED && SOL) {
      k.C = k.packed ? st.seg_ptr(sg, 0) + lane : st.lane_ptr(sg, 0);
      k.c = st.lane_ptr(sg, 1);
      k.F = k.f = k.tau = k.Kk = nullptr;
      k.xs = st.lane_ptr(sg, 2);
      k.us = st.lane_ptr(sg, 3);
    } else if (STAGED) {
      k.C = k.packed ? st.seg_ptr(sg, 0) + lane : st.lane_ptr(sg, 0);
      k.c = st.lane_ptr(sg, 1);
      k.F = kEnv ? nullptr : st.lane_ptr(sg, 2);
      k.f = kEnv ? nullptr : st.lane_ptr(sg, 3);
      k.tau = st.seg_ptr(sg, 4) + lane;
      k.Kk = st.seg_ptr(sg, 5) + lane;
    } else {
      // shapes too large to stage: the packed, lane-interleaved copy of C (written by begin)
      // turns the per-thread reads of a 2 KB row-major block into coalesced ones
      k.packed = (st.seg_full >> 0) & 1u;   // set once per kernel (use_packed_direct)
      k.C = k.packed ? p.Cpk + bidx(t, 0, NP, bw, p.nW)
                     : cost_src<S>(p.C, p.C_bcast, t, p.B, b, N * N);
      k.c = cost_src<S>(p.c, p.c_bcast, t, p.B, b, N);
      k.F = (kEnv || t >= p.T - 1) ? nullptr : p.F + ((size_t)t * p.B + b) * (NS * N);
      k.f = (kEnv || !p.has_f || t >= p.T - 1) ? nullptr : p.f + ((size_t)t * p.B + b) * NS;
      k.tau = p.traj_cur + bidx(t, 0, N, bw, p.nW);
      k.Kk = p.Kk + bidx(t, 0, NK, bw, p.nW);
    }
    k.tstride = kWarp;
    return k;
  }

  DILQR_DEVICE static void bounds_at(const IterParams<S>& p, int t, int b, S* lo, S* hi) {
    if (p.bounds_kind == 2) {
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        lo[a] = __ldg(p.lo_t + ((size_t)t * p.B + b) * NC + a);
        hi[a] = __ldg(p.hi_t + ((size_t)t * p.B + b) * NC + a);
      }
    } else {
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        lo[a] = p.lo;
        hi[a] = p.hi;
      }
    }
  }

  // Tell the stager where this warp's slabs / chunks of each segment live (once per
  // kernel): address of timestep 0 and the byte stride between timesteps.
  template <bool SOL = false>
  DILQR_DEVICE static void bind_sources(WarpStager<S>& st, const IterParams<S>& p, int b0) {
    if (!STAGED) return;
    const long long sz = (long long)sizeof(S);
    if ((st.seg_full >> 0) & 1u)
      st.bind(0, p.Cpk + bidx(0, 0, NP, b0, p.nW), (long long)p.nW * NP * kWarp * sz);
    else
      st.bind(0, cost_src<S>(p.C, p.C_bcast, 0, p.B, b0, N * N),
              p.C_bcast == 0 ? (long long)p.B * N * N * sz : (p.C_bcast == 1 ? (long long)N * N * sz : 0));
    st.bind(1, cost_src<S>(p.c, p.c_bcast, 0, p.B, b0, N),
            p.c_bcast == 0 ? (long long)p.B * N * sz : (p.c_bcast == 1 ? (long long)N * sz : 0));
    if (SOL) {
      st.bind(2, p.x_out + (size_t)b0 * NS, (long long)p.B * NS * sz);
      st.bind(3, p.u_out + (size_t)b0 * NC, (long long)p.B * NC * sz);
      return;
    }
    if (!kEnv) {
      st.bind(2, p.F ? p.F + (size_t)b0 * (NS * N) : nullptr, (long long)p.B * NS * N * sz);
      st.bind(3, (p.has_f && p.f) ? p.f + (size_t)b0 * NS : nullptr, (long long)p.B * NS * sz);
    }
    st.bind(4, p.traj_cur + bidx(0, 0, N, b0, p.nW), (long long)p.nW * N * kWarp * sz);
    st.bind(5, p.Kk + bidx(0, 0, NK, b0, p.nW), (long long)p.nW * NK * kWarp * sz);
  }

  // issue the operands of timestep t for this warp into `stage`
  template <bool SOL = false>
  DILQR_DEVICE static void issue_t(WarpStager<S>& st, const IterParams<S>& p, int stage, int t,
                                   int b0, bool want_f, bool want_traj, bool want_K) {
    if (!STAGED) return;
    uint32_t mask = 3u;   // C, c
    if (SOL) {
      st.issue_bound(stage, t, mask | (1u << 2) | (1u << 3));
      return;
    }
    if (!kEnv && t < p.T - 1) {
      if (p.F) mask |= 1u << 2;
      if (want_f && p.has_f && p.f) mask |= 1u << 3;
    }
    if (want_traj) mask |= 1u << 4;
    if (want_K) mask |= 1u << 5;
    st.issue_bound(stage, t, mask);
  }

  // ======================================================================
  // Phase A: c_back + Riccati backward sweep with gains (and pnqp).
  // ======================================================================
  // b: problem index for the API tensors (clamped for padded lanes); bw: this
  // lane's own column of the (padded) workspace.
  // SOL (gains at the solution, lqr_step_explicit.py:604-618): tau* comes from the API
  // slabs x_out / u_out, nothing of the solver state is touched except the gains, and the
  // primal costates lam_t = C_xx x + C_xu u + c_x + F_x' lam_{t+1} (lqr_step.py:355-369) ride
  // along (p.lam_blk) -- they need exactly the operands this sweep has in hand.
  template <bool SOL = false>
  DILQR_DEVICE static void backward_sweep(const IterParams<S>& p, WarpStager<S>& st, int b0,
                                          int b, int bw, bool active, int lane) {
    S V[NS][NS], v[NS];
    S lam[SOL ? NS : 1];
    S kprev[NC];
    S xnext[NS];  // x_{t+1} of the nominal trajectory (trig reuse for env Jacobians)
    bool have_prev = false;
    const int T = p.T;
    // lazy best-iterate tracking (mpc.py:272-285): if the previous iteration made the
    // current trajectory this problem's best, park it in traj_best while it streams by.
    const bool flush = !SOL && (p.take[bw] & 1) != 0;
    issue_t<SOL>(st, p, 0, T - 1, b0, false, true, false);
    // First two words of the guessed pnqp trace: lane l keeps those of timestep (t & ~31) + l
    // (one 8-byte load per lane per 32 timesteps), the sweep fetches its timestep's pair with
    // two shuffles.  A global load per timestep -- wherever it is placed -- costs an exposed L2
    // round trip: ptxas makes an unrelated instruction next to it wait on the shared scoreboard
    // (ncu: 400 cycles per timestep, profiles/r2_iter_stalls.txt).
    const bool use_guess = p.bounds_kind && !p.solo;
    uint2 glane = make_uint2(0, 0);
    for (int t = T - 1; t >= 0; --t) {
      const int sg = (T - 1 - t) & 1;
      if (t > 0) issue_t<SOL>(st, p, sg ^ 1, t - 1, b0, false, true, false);
      if (use_guess && (t == T - 1 || (t & 31) == 31)) {
        const int tt = (t & ~31) + lane;
        glane = tt < T ? __ldg(reinterpret_cast<const uint2*>(p.guess + (size_t)tt * kPnqpMaxIter))
                       : make_uint2(0, 0);
      }
      if (STAGED) st.wait(sg);
      const Blk blk = blocks<SOL>(p, st, sg, t, b, bw, lane);
      const S* Cs = blk.C;
      const S* cs = blk.c;
      S tau[N];
      if constexpr (SOL) {
#pragma unroll
        for (int i = 0; i < NS; ++i) tau[i] = blk.xs[i];
#pragma unroll
        for (int a = 0; a < NC; ++a) tau[NS + a] = blk.us[a];
      } else {
#pragma unroll
        for (int i = 0; i < N; ++i) tau[i] = blk.tau[i * kWarp];
      }
      if (flush) {
        S* bo = p.traj_best + bidx(t, 0, N, bw, p.nW);
#pragma unroll
        for (int i = 0; i < N; ++i) bo[i * kWarp] = tau[i];
      }

      S Q[N][N], qv[N];
      if (blk.packed) {
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = 0; j < N; ++j) Q[i][j] = Cs[pk_idx<N>(i, j) * kWarp];
      } else {
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = 0; j < N; ++j) Q[i][j] = Cs[i * N + j];
      }
#pragma unroll
      for (int i = 0; i < N; ++i) {  // c_back = C tau + c   (lqr_step.py:294)
        S acc = kChainFma ? cs[i] : S(0);
#pragma unroll
        for (int j = 0; j < N; ++j) acc = fmaS<S>(Q[i][j], tau[j], acc);
        qv[i] = kChainFma ? acc : acc + cs[i];
      }
      S nl[SOL ? NS : 1];
      if constexpr (SOL) {   // cost part of lam_t, same association as costate_tables_kernel
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          S a1 = S(0), a2 = S(0);
#pragma unroll
          for (int j = 0; j < NS; ++j) a1 = fmaS<S>(Q[i][j], tau[j], a1);
#pragma unroll
          for (int a = 0; a < NC; ++a) a2 = fmaS<S>(Q[i][NS + a], tau[NS + a], a2);
          nl[i] = (a1 + a2) + cs[i];
        }
      }
      if (t < T - 1) {
        S Fm[NS][N];
        if constexpr (kEnv) {
          D::jacobian(p.dyn, tau, xnext, Fm);
        } else {
          const S* Fs = blk.F;
#pragma unroll
          for (int i = 0; i < NS; ++i)
#pragma unroll
            for (int j = 0; j < N; ++j) Fm[i][j] = Fs[i * N + j];
        }
        // Q = C + (F' V) F ; q = c~ + F' v     (lqr_step.py:66-70).  Structurally
        // zero entries of the env Jacobians are skipped at compile time (exact).
#pragma unroll
        for (int i = 0; i < N; ++i) {
          S M[NS];
#pragma unroll
          for (int k = 0; k < NS; ++k) {
            S acc = S(0);
#pragma unroll
            for (int l = 0; l < NS; ++l)
              if (D::nz(l, i)) acc = fmaS<S>(Fm[l][i], V[l][k], acc);
            M[k] = acc;
          }
#pragma unroll
          for (int j = 0; j < N; ++j) {
            if (kSym && j < i) continue;
            S acc = kChainFma ? Q[i][j] : S(0);
#pragma unroll
            for (int k = 0; k < NS; ++k)
              if (D::nz(k, j)) acc = fmaS<S>(M[k], Fm[k][j], acc);
            Q[i][j] = kChainFma ? acc : Q[i][j] + acc;
          }
          S acc = kChainFma ? qv[i] : S(0);
#pragma unroll
          for (int l = 0; l < NS; ++l)
            if (D::nz(l, i)) acc = fmaS<S>(Fm[l][i], v[l], acc);
          qv[i] = kChainFma ? acc : qv[i] + acc;
        }
        if constexpr (kSym) {
#pragma unroll
          for (int i = 0; i < N; ++i)
#pragma unroll
            for (int j = 0; j < i; ++j) Q[i][j] = Q[j][i];
        }
        if constexpr (SOL) {
#pragma unroll
          for (int i = 0; i < NS; ++i) {
            S a1 = S(0);
#pragma unroll
            for (int l = 0; l < NS; ++l)
              if (D::nz(l, i)) a1 = fmaS<S>(Fm[l][i], lam[l], a1);
            nl[i] = nl[i] + a1;
          }
        }
      }
      if constexpr (SOL) {
        S* lo_ = p.lam_blk ? p.lam_blk + bidx(t, 0, NS, bw, p.nW) : nullptr;
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          lam[i] = nl[i];
          if (lo_) lo_[i * kWarp] = nl[i];
        }
      }
#pragma unroll
      for (int i = 0; i < NS; ++i) xnext[i] = tau[i];

      // ------------------------------------------------------------ gains
      S K[NC][NS], k[NC];
      if (p.bounds_kind == 0) {
        bool mask[NC];
#pragma unroll
        for (int a = 0; a < NC; ++a)
          mask[a] = p.zeroI ? (p.zeroI[((size_t)t * p.B + b) * NC + a] != 0) : false;
        if (NC == 1) {
          if (!p.zeroI) {  // lqr_step.py:84-86
            const S r = S(1) / Q[NS][NS];
#pragma unroll
            for (int j = 0; j < NS; ++j) K[0][j] = -(r * Q[NS][j]);
            k[0] = -(r * qv[NS]);
          } else {         // lqr_step.py:101-123
            const S quu_m = mask[0] ? S(1e-8) : Q[NS][NS];
            const S r = S(1) / quu_m;
#pragma unroll
            for (int j = 0; j < NS; ++j) K[0][j] = -(r * (mask[0] ? S(0) : Q[NS][j]));
            k[0] = -((S(1) / Q[NS][NS]) * (mask[0] ? S(0) : qv[NS]));
          }
        } else if (!p.zeroI && p.gain_solve == 1) {  // lqr_step_backup.py:202-205
          Chol<S, NC> ch;
#pragma unroll
          for (int a = 0; a < NC; ++a)
#pragma unroll
            for (int c2 = 0; c2 < NC; ++c2)
              ch.l[a][c2] = Q[NS + a][NS + c2] + (a == c2 ? S(1e-6) : S(0));
          ch.factor();
#pragma unroll
          for (int j = 0; j <= NS; ++j) {
            S rhs[NC];
#pragma unroll
            for (int a = 0; a < NC; ++a) rhs[a] = (j < NS) ? Q[NS + a][j] : qv[NS + a];
            ch.solve(rhs);
#pragma unroll
            for (int a = 0; a < NC; ++a) {
              if (j < NS) K[a][j] = -rhs[a];
              else k[a] = -rhs[a];
            }
          }
        } else {  // plain solve / u_zero_I-masked LU solve (lqr_step.py:88-94,101-127)
          LUpp<S, NC> lu;
#pragma unroll
          for (int a = 0; a < NC; ++a)
#pragma unroll
            for (int c2 = 0; c2 < NC; ++c2) {
              S h = (mask[a] || mask[c2]) ? S(0) : Q[NS + a][NS + c2];
              if (a == c2 && mask[a]) h = h + S(1e-8);
              lu.a[a][c2] = h;
            }
          lu.factor();
#pragma unroll
          for (int j = 0; j <= NS; ++j) {
            S rhs[NC];
#pragma unroll
            for (int a = 0; a < NC; ++a)
              rhs[a] = mask[a] ? S(0) : ((j < NS) ? Q[NS + a][j] : qv[NS + a]);
            lu.solve(rhs);
#pragma unroll
            for (int a = 0; a < NC; ++a) {
              if (j < NS) K[a][j] = -rhs[a];
              else k[a] = -rhs[a];
            }
          }
        }
      } else {  // box constraints: pnqp   (lqr_step.py:128-148)
        S lo[NC], hi[NC], H[NC][NC], qu[NC];
        bounds_at(p, t, b, lo, hi);
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          lo[a] = lo[a] - tau[NS + a];
          hi[a] = hi[a] - tau[NS + a];
          if (p.has_delta) {   // lqr_step.py:132-134
            if (lo[a] < -p.delta_u) lo[a] = -p.delta_u;
            if (hi[a] > p.delta_u) hi[a] = p.delta_u;
          }
          qu[a] = qv[NS + a];
#pragma unroll
          for (int c2 = 0; c2 < NC; ++c2) H[a][c2] = Q[NS + a][NS + c2];
          k[a] = have_prev ? kprev[a] : S(0);
        }
        bool If[NC];
        LUpp<S, NC> lu;
        S rinv = S(0);
        uint4 gpre = make_uint4(0, 0, 0, 0);
        if (use_guess) {
          gpre.x = __shfl_sync(kFull, glane.x, t & 31);
          gpre.y = __shfl_sync(kFull, glane.y, t & 31);
        }
        pnqp_thread<S, NC>(H, qu, lo, hi, have_prev, k, If, lu, p.guess + (size_t)t * kPnqpMaxIter,
                           gpre, p.votes + (size_t)t * kPnqpMaxIter, p.solo != 0, active, lane,
                           &rinv);
        have_prev = true;
#pragma unroll
        for (int a = 0; a < NC; ++a) kprev[a] = k[a];
        if (NC == 1) {  // lqr_step.py:144-146
          const S r = rinv;   // == 1 / lu.a[0][0], computed inside pnqp_thread
#pragma unroll
          for (int j = 0; j < NS; ++j) K[0][j] = -(r * (If[0] ? Q[NS][j] : S(0)));
        } else {        // lqr_step.py:148
#pragma unroll
          for (int j = 0; j < NS; ++j) {
            S rhs[NC];
#pragma unroll
            for (int a = 0; a < NC; ++a) rhs[a] = If[a] ? Q[NS + a][j] : S(0);
            lu.solve(rhs);
#pragma unroll
            for (int a = 0; a < NC; ++a) K[a][j] = -rhs[a];
          }
        }
      }
      {
        S* ko = p.Kk + bidx(t, 0, NK, bw, p.nW);   // padded lanes own their column: no guard
#pragma unroll
        for (int a = 0; a < NC; ++a) {
#pragma unroll
          for (int j = 0; j < NS; ++j) ko[(a * NS + j) * kWarp] = K[a][j];
          ko[(NC * NS + a) * kWarp] = k[a];
        }
      }
      // -------------------------------------------- value function update
      // V = Qxx + Qxu K + K' Qux + (K' Quu) K      (lqr_step.py:155)
      // v = qx + Qxu k + K' qu + (K' Quu) k        (lqr_step.py:156-158)
      S KQ[NS][NC];  // K' Quu
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          S acc = S(0);
#pragma unroll
          for (int c2 = 0; c2 < NC; ++c2) acc = fmaS<S>(K[c2][i], Q[NS + c2][NS + a], acc);
          KQ[i][a] = acc;
        }
#pragma unroll
      for (int i = 0; i < NS; ++i) {
#pragma unroll
        for (int j = 0; j < NS; ++j) {
          if (kSym && j < i) continue;
          if constexpr (kChainFma) {
            S acc = Q[i][j];
#pragma unroll
            for (int a = 0; a < NC; ++a) acc = fmaS<S>(Q[i][NS + a], K[a][j], acc);
#pragma unroll
            for (int a = 0; a < NC; ++a) acc = fmaS<S>(K[a][i], Q[NS + a][j], acc);
#pragma unroll
            for (int a = 0; a < NC; ++a) acc = fmaS<S>(KQ[i][a], K[a][j], acc);
            V[i][j] = acc;
          } else {
            S t1 = S(0), t2 = S(0), t3 = S(0);
#pragma unroll
            for (int a = 0; a < NC; ++a) {
              t1 = fmaS<S>(Q[i][NS + a], K[a][j], t1);
              t2 = fmaS<S>(K[a][i], Q[NS + a][j], t2);
              t3 = fmaS<S>(KQ[i][a], K[a][j], t3);
            }
            V[i][j] = ((Q[i][j] + t1) + t2) + t3;
          }
        }
        if constexpr (kChainFma) {
          S acc = qv[i];
#pragma unroll
          for (int a = 0; a < NC; ++a) acc = fmaS<S>(Q[i][NS + a], k[a], acc);
#pragma unroll
          for (int a = 0; a < NC; ++a) acc = fmaS<S>(K[a][i], qv[NS + a], acc);
#pragma unroll
          for (int a = 0; a < NC; ++a) acc = fmaS<S>(KQ[i][a], k[a], acc);
          v[i] = acc;
        } else {
          S t1 = S(0), t2 = S(0), t3 = S(0);
#pragma unroll
          for (int a = 0; a < NC; ++a) {
            t1 = fmaS<S>(Q[i][NS + a], k[a], t1);
            t2 = fmaS<S>(K[a][i], qv[NS + a], t2);
            t3 = fmaS<S>(KQ[i][a], k[a], t3);
          }
          v[i] = ((qv[i] + t1) + t2) + t3;
        }
      }
      if constexpr (kSym) {
#pragma unroll
        for (int i = 0; i < NS; ++i)
#pragma unroll
          for (int j = 0; j < i; ++j) V[i][j] = V[j][i];
      }
    }
  }

  // ======================================================================
  // Phase B: forward rollout with the affine control law + line search over
  // the true dynamics (lqr_step.py:164-261).
  // ======================================================================
  DILQR_DEVICE static void forward_linesearch(const IterParams<S>& p, WarpStager<S>& st, int b0,
                                              int b, int bw, bool active, int lane) {
    const int T = p.T;
    const S old_cost = p.cost_cur[b];
    S alpha = S(1);
    bool accepted = false;
    S res_cost = S(0), res_alpha = S(1);
    S x0[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) x0[i] = __ldg(p.x_init + (size_t)b * NS + i);
    // the gains written by phase A (generic-proxy stores) are read back through the
    // async proxy (TMA) below
    __threadfence();
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncwarp();

    for (int tr = 0; tr < p.max_ls; ++tr) {
      if (!__any_sync(kFull, active && !accepted)) break;
      const bool run = active && !accepted;
      S xh[NS];
#pragma unroll
      for (int i = 0; i < NS; ++i) xh[i] = x0[i];
      S cost = S(0);
      // two timesteps in flight: the stage of t is re-issued for t+2 as soon as its last
      // reader (the cost of t; the linear dynamics for LinDx) is done, i.e. before the
      // dynamics step -- a rollout timestep is shorter than a DRAM round trip under load
      issue_t(st, p, 0, 0, b0, true, true, true);
      if (T > 1) issue_t(st, p, 1, 1, b0, true, true, true);
      for (int t = 0; t < T; ++t) {
        const int sg = t & 1;
        if (STAGED) st.wait(sg);
        if (!STAGED && kEnv && t + 1 < T) prefetch_step_l2(p, st, t + 1, b0, lane);
        const Blk blk = blocks(p, st, sg, t, b, bw, lane);
        S tau[N];   // nominal (x_t, u_t)
#pragma unroll
        for (int i = 0; i < N; ++i) tau[i] = blk.tau[i * kWarp];
        S th[N];    // new (x^_t, u^_t)
#pragma unroll
        for (int i = 0; i < NS; ++i) th[i] = xh[i];
        S lo[NC], hi[NC];
        if (p.bounds_kind) bounds_at(p, t, b, lo, hi);
#pragma unroll
        for (int a = 0; a < NC; ++a) {  // lqr_step.py:192
          S acc = S(0);
          if (t > 0) {
#pragma unroll
            for (int j = 0; j < NS; ++j)
              acc = fmaS<S>(blk.Kk[(a * NS + j) * kWarp], xh[j] - tau[j], acc);
          }
          S un = (acc + tau[NS + a]) + alpha * blk.Kk[(NC * NS + a) * kWarp];
          if (p.zeroI && p.zeroI[((size_t)t * p.B + b) * NC + a]) un = S(0);  // :197-198
          if (p.bounds_kind) {
            S lb = lo[a], ub = hi[a];
            if (p.has_delta) {   // lqr_step.py:204-211
              const S l2 = tau[NS + a] - p.delta_u, u2 = tau[NS + a] + p.delta_u;
              lb = l2 < lb ? lb : l2;
              ub = u2 > ub ? ub : u2;
            }
            un = eclamp<S>(un, lb, ub);                                         // :213
          }
          th[NS + a] = un;
          // full_du_norm (lqr_step.py:243-245) is the row norm of
          // (u - new_u).transpose(1,2).contiguous().view(n_batch, -1): the [T,nc,B]
          // array re-read as [B, T*nc] -- rows mix problems and timesteps.  Mirror it:
          // store the squares in [T,nc,B] order, the commit kernel sums the rows.
          if (tr == 0 && active) {
            const S d = tau[NS + a] - un;
            p.dusq[((size_t)t * NC + a) * p.B + b] = d * d;
          }
        }
        if (!accepted) {   // padded lanes keep their own columns defined as well
          S* to = p.traj_new + bidx(t, 0, N, bw, p.nW);
#pragma unroll
          for (int i = 0; i < N; ++i) to[i * kWarp] = th[i];
        }
        cost = cost + (blk.packed ? stage_cost_packed<S, N>(blk.C, blk.c, th)
                                  : stage_cost<S, N>(blk.C, blk.c, th));
        if (kEnv && t + 2 < T) issue_t(st, p, sg, t + 2, b0, true, true, true);
        if (t < T - 1) {
          if constexpr (kEnv) {
            dyn_step<S, NS, NC, DYN>(p.dyn, th, &th[NS], xh);
          } else {
            lin_step<S, NS, N>(blk.F, blk.f, p.has_f != 0, th, xh);
          }
        }
        if (!kEnv && t + 2 < T) issue_t(st, p, sg, t + 2, b0, true, true, true);
      }
      if (run) {
        res_cost = cost;
        res_alpha = alpha;
        accepted = !(cost > old_cost);      // lqr_step.py:176-179,247
        if (!accepted) alpha = alpha * p.decay;
      }
    }
    if (active) {
      p.cost_new[b] = res_cost;
      p.alpha_new[b] = res_alpha;
    }
  }
};

// FP32, small env shapes: cap the registers at 128 (no extra spills) so that 16 warps fit
// one SM: a 65536-problem batch (2048 warps, 13.8 per SM) then runs as ONE wave instead of
// two, which saves a whole per-warp latency (cartpole: 0.445 -> 0.30 ms per launch).  The
// FP64 build needs 252 registers and 27.6 KB of stage per warp and stays at 8 warps/SM.
template <class S, int NS, int NC, int DYN, bool STAGED>
constexpr int iter_min_blocks() {
  return (sizeof(S) == 4 && STAGED && DYN != DYN_LINDX && NS + NC <= 6) ? 4 : 1;
}

// ROLLOUT_ONLY: the line-search rollout alone, behind the group sweep (api.cu)
template <class S, int NS, int NC, int DYN, bool STAGED, bool ROLLOUT_ONLY = false, bool SYM = false>
__global__ void __launch_bounds__(128, iter_min_blocks<S, NS, NC, DYN, STAGED>())
ilqr_iter_kernel(const __grid_constant__ IterParams<S> p) {
  using IK = IterKernel<S, NS, NC, DYN, STAGED, SYM>;
  if (SYM ? !IK::sym_ok(p) : (p.sym_pair && IK::sym_ok(p))) return;   // the other kernel of the pair runs
  extern __shared__ __align__(128) char smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int wpb = blockDim.x >> 5;
  const int b0 = (blockIdx.x * wpb + warp) * kWarp;
  if (b0 >= p.B) return;
  if (p.halt && *reinterpret_cast<const volatile uint32_t*>(p.halt)) return;  // pipelined loop stopped
  const int nvalid = min(kWarp, p.B - b0);
  const bool active = lane < nvalid;
  const int b = b0 + lane;   // padded lanes index their own (padded) workspace column

  const size_t per_warp = IK::smem_per_warp();
  char* wbase = smem + warp * per_warp;
  uint64_t* bars = reinterpret_cast<uint64_t*>(wbase);
  WarpStager<S> st;
  if (STAGED) {
    uint32_t e[IK::kNSeg];
    IK::seg_elems(e);
    const bool packed = IK::use_packed(p);
    if (packed) e[0] = IK::NP;     // segment 0 = warp-blocked packed chunk instead of the slab
    st.init(wbase + kStages * sizeof(uint64_t), bars, lane, nvalid, IK::kNSeg, e,
            IK::kFullMask | (packed ? 1u : 0u), (p.C_bcast ? 1u : 0u) | (p.c_bcast ? 2u : 0u));
    IK::bind_sources(st, p, b0);
  } else {
    st.seg_full = IK::use_packed_direct(p) ? 1u : 0u;   // blocks(): packed copy of C or the API tensor
  }
  // padded lanes (tail warp) read the API tensors of the warp's first problem
  const int bsafe = active ? b : b0;
  if (!ROLLOUT_ONLY) IK::backward_sweep(p, st, b0, bsafe, b, active, lane);
  if (!p.gains_only) IK::forward_linesearch(p, st, b0, bsafe, b, active, lane);
}

// ---------------------------------------------------------------------------
// Gains of the final no-op LQR pass at the solution (lqr_step_explicit.py:604-618:
// LQRStep(...)(x*, u*) whose new iterate is discarded) + the primal costates, straight
// from the solver's outputs x_out / u_out and the packed C the solve left in the
// workspace: no re-layout of the trajectory (begin) and no gather of the gains (finish).
// Writes Kk (workspace, blocked) and lam_blk.
// ---------------------------------------------------------------------------
template <class S, int NS, int NC, int DYN, bool STAGED, bool SYM = false>
__global__ void __launch_bounds__(128)
ilqr_gains_kernel(const __grid_constant__ IterParams<S> p) {
  using IK = IterKernel<S, NS, NC, DYN, STAGED, SYM>;
  if (SYM ? !IK::sym_ok(p) : (p.sym_pair && IK::sym_ok(p))) return;   // the other kernel of the pair runs
  extern __shared__ __align__(128) char smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int wpb = blockDim.x >> 5;
  const int b0 = (blockIdx.x * wpb + warp) * kWarp;
  if (b0 >= p.B) return;
  const int nvalid = min(kWarp, p.B - b0);
  const bool active = lane < nvalid;
  const int b = b0 + lane;
  const size_t per_warp = IK::smem_per_warp(true);
  char* wbase = smem + warp * per_warp;
  WarpStager<S> st;
  if (STAGED) {
    uint32_t e[IK::kNSeg];
    IK::seg_elems(e, true);
    const bool packed = IK::use_packed(p);
    if (packed) e[0] = IK::NP;
    st.init(wbase + kStages * sizeof(uint64_t), reinterpret_cast<uint64_t*>(wbase), lane, nvalid,
            IK::kNSeg, e, packed ? 1u : 0u, (p.C_bcast ? 1u : 0u) | (p.c_bcast ? 2u : 0u));
    IK::template bind_sources<true>(st, p, b0);
  }
  const int bsafe = active ? b : b0;
  IK::template backward_sweep<true>(p, st, b0, bsafe, b, active, lane);
}

// ---------------------------------------------------------------------------
// begin: nominal rollout of u_init (util.get_traj) + its cost (util.get_cost)
// into the current-trajectory buffer.  With p.x_cur != nullptr the given
// trajectory is loaded instead of rolled out (standalone LQRStep,
// lqr_step.py:164-169).
// ---------------------------------------------------------------------------
template <class S, int NS, int NC, int DYN, bool STAGED>
__global__ void __launch_bounds__(128)
ilqr_begin_kernel(const __grid_constant__ IterParams<S> p) {
  using IK = IterKernel<S, NS, NC, DYN, STAGED>;
  using D = Dyn<S, DYN>;
  constexpr int N = NS + NC;
  constexpr bool kEnv = (DYN != DYN_LINDX);
  extern __shared__ __align__(128) char smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int wpb = blockDim.x >> 5;
  const int b0 = (blockIdx.x * wpb + warp) * kWarp;
  if (b0 >= p.B) return;
  const int nvalid = min(kWarp, p.B - b0);
  const bool active = lane < nvalid;
  const int b = active ? b0 + lane : b0;
  const size_t per_warp = IK::smem_per_warp();
  char* wbase = smem + warp * per_warp;
  WarpStager<S> st;
  if (STAGED) {
    uint32_t e[IK::kNSeg];
    IK::seg_elems(e);
    st.init(wbase + kStages * sizeof(uint64_t), reinterpret_cast<uint64_t*>(wbase), lane, nvalid,
            IK::kNSeg, e, IK::kFullMask, (p.C_bcast ? 1u : 0u) | (p.c_bcast ? 2u : 0u));
    IK::bind_sources(st, p, b0);
  }
  const int T = p.T;
  S xh[NS];
#pragma unroll
  for (int i = 0; i < NS; ++i) xh[i] = __ldg(p.x_init + (size_t)b * NS + i);
  S cost = S(0);
  // gains_only (final no-op LQR pass): the trajectory is only re-laid-out, no cost, so
  // C and c are not streamed at all
  const bool want_cost = !(p.gains_only && p.x_cur);
  // the sweeps read C twice per iteration: when every block is bitwise symmetric they
  // stream this packed copy (N(N+1)/2 instead of N*N scalars) instead
  const bool do_pack = want_cost && !p.C_bcast && p.cpk_state &&
                       *reinterpret_cast<const volatile uint32_t*>(p.cpk_state) == 1u;
  // broadcast C (state 3, set by the launch): verify the shared block(s) so that the sweeps may
  // use the symmetric update for them too -- same arithmetic as for the dense tiling of that block
  const bool do_symchk = want_cost && p.C_bcast && p.cpk_state &&
                         *reinterpret_cast<const volatile uint32_t*>(p.cpk_state) == 3u;
  bool asym = false;
  if (want_cost) IK::issue_t(st, p, 0, 0, b0, true, false, false);
  for (int t = 0; t < T; ++t) {
    const int sg = t & 1;
    if (want_cost && t + 1 < T) IK::issue_t(st, p, sg ^ 1, t + 1, b0, true, false, false);
    S th[N];
    if (p.x_cur) {
#pragma unroll
      for (int i = 0; i < NS; ++i) th[i] = __ldg(p.x_cur + ((size_t)t * p.B + b) * NS + i);
    } else {
#pragma unroll
      for (int i = 0; i < NS; ++i) th[i] = xh[i];
    }
#pragma unroll
    for (int a = 0; a < NC; ++a)
      th[NS + a] = p.u_init ? __ldg(p.u_init + ((size_t)t * p.B + b) * NC + a) : S(0);
    {
      S* to = p.traj_new + bidx(t, 0, N, b0 + lane, p.nW);
#pragma unroll
      for (int i = 0; i < N; ++i) to[i * kWarp] = th[i];
    }
    if (!want_cost) continue;
    if (STAGED) st.wait(sg);
    typename IK::Blk blk = IK::blocks(p, st, sg, t, b, b0 + lane, lane);
    if (!STAGED) {   // begin WRITES the packed copy: it reads the dense API tensor itself
      blk.C = cost_src<S>(p.C, p.C_bcast, t, p.B, b, N * N);
      blk.packed = false;
    }
    cost = cost + stage_cost<S, N>(blk.C, blk.c, th);
    if (do_pack) {   // upper triangle into the warp-blocked workspace copy; symmetry check
      S* po = p.Cpk + bidx(t, 0, IK::NP, b0 + lane, p.nW);
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = i; j < N; ++j) {
          const S cij = blk.C[i * N + j];
          if (j > i && !(cij == blk.C[j * N + i])) asym = true;
          po[pk_idx<N>(i, j) * kWarp] = cij;
        }
    }
    if (do_symchk && (p.C_bcast == 1 || t == 0)) {
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = i + 1; j < N; ++j)
          if (!(blk.C[i * N + j] == blk.C[j * N + i])) asym = true;
    }
    if (t < T - 1 && !p.x_cur) {
      if constexpr (kEnv) {
        dyn_step<S, NS, NC, DYN>(p.dyn, th, &th[NS], xh);
      } else {
        lin_step<S, NS, N>(blk.F, blk.f, p.has_f != 0, th, xh);
      }
    }
  }
  if (active) p.cost_cur[b] = cost;
  p.take[b0 + lane] = 0;
  if ((do_pack || do_symchk) && __any_sync(kFull, asym && active) && lane == 0)
    atomicExch(p.cpk_state, 2u);
}

}  // namespace dilqr
