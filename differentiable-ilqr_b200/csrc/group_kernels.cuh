// group_kernels.cuh -- the Riccati / pnqp sweep for LARGE problems (n_tau >= 12: rocket
// 13+3, LinDx up to 16+4) and for multi-input box-constrained batches of any size.
//
// Why a second mapping.  One thread per problem keeps V, Q, F of a problem in that thread's
// registers; for n_tau = 16 that is 633 doubles -- they spill to local memory (6.5 KB per
// thread), 36.6 GB of DRAM traffic per launch against 3.8 GB algorithmic, 1.8 % of the HBM
// roofline (profiles/r1_iter_rocket_f64_g.txt).  And the batch-global pnqp decisions
// (pnqp.py:56-59,65,75) were resolved with grid barriers, which needs EVERY problem resident:
// 16 384 rocket problems x 5 KB of state is more than the chip's registers + shared memory.
//
// Here the sweep is BATCH-SYNCHRONOUS: a persistent cooperative grid walks the horizon once,
// all problems together, and per timestep alternates between
//   phase AC  a THREAD GROUP of G = 16 (32) lanes per problem: lane l owns row l of the
//             matrices; V_{t+1} = f(Q_{t+1}, K_{t+1}) and Q_t = C_t + F_t' V_{t+1} F_t are formed
//             with the operands every lane needs (F_t, V_{t+1}, K_{t+1}) broadcast from shared
//             memory and the lane's own rows in registers; a group loops over its share of
//             the batch, so residency no longer depends on the batch size;
//   phase B   ONE THREAD per problem on the n_ctrl x n_ctrl control QP: gains or pnqp, every
//             batch-global decision an atomicOr + grid barrier (the votes ARE the trace: no
//             guessing, no re-runs), warm start carried in registers along the horizon.
// The only state that crosses a phase boundary is Q_t, q_t (one record per problem, written
// and read once per timestep, L2-resident) and the gains, which the forward pass needs anyway.
//
// Reference semantics: lqr_step.py:52-160 (lqr_backward), pnqp.py:5-82, as in ilqr_kernels.cuh.
#pragma once
#include <cooperative_groups.h>

#include "ilqr_kernels.cuh"

namespace dilqr {

template <class S, int NS, int NC, int DYN>
struct GroupSweep {
  static constexpr int N = NS + NC;
  static constexpr int NK = NC * NS + NC;
  static constexpr int G = (N <= 16) ? 16 : 32;   // lanes per problem
  static constexpr int kThreads = 256;
  static constexpr int GPB = kThreads / G;        // groups per block
  static constexpr bool kEnv = (DYN != DYN_LINDX);
  static constexpr bool kChain = kChainFmaOn && kEnv;
  static constexpr int QREC = N * N + N;          // scratch record: Q_t[N][N], q_t[N]
  static constexpr int GIN = NC * N + NC;         // gains input: rows n_state.. of Q_t, q_u
  using D = Dyn<S, DYN>;

  struct alignas(16) Shared {
    S F[NS][N];
    S V[NS][NS];
    S v[NS];
    S tau[N];
    S xnext[NS];
    S K[NC][NS];
    S k[NC];
    S Qu[NC][N];   // rows n_state.. of Q_{t+1}
    S qu[NC];
    // The two (G = 16) groups of a warp broadcast-read the same field of their own block in
    // one instruction: keep the block size off the 128-byte bank period so the two
    // addresses fall into different banks (one wavefront instead of a 2-way conflict).
    S pad[((sizeof(S) * (NS * N + NS * NS + NS + N + NS + NC * NS + NC + NC * N + NC)) % 128 == 0) ? 2 : 0];
  };
  static __host__ __device__ size_t smem_bytes() { return sizeof(Shared) * GPB; }

  DILQR_DEVICE static void gsync(unsigned mask) { __syncwarp(mask); }

  // ---------------------------------------------------------------- phase AC, one problem
#ifdef DILQR_GS_TIMING
#define AC_TICK(i) { long long c_ = clock64(); tacc[i] += c_ - tprev; tprev = c_; }
#else
#define AC_TICK(i)
#endif
  DILQR_DEVICE static void phase_ac(const IterParams<S>& p, Shared& sm, int b, int t, int gl,
                                    unsigned gmask, long long* tacc = nullptr) {
    const int T = p.T;
#ifdef DILQR_GS_TIMING
    long long tprev = clock64();
#endif
    S* rec = p.gsQ + (size_t)b * QREC;
    // ---- (C) V_{t+1}, v_{t+1} from Q_{t+1} and the gains of t+1   (lqr_step.py:155-158)
    if (t < T - 1) {
      {
        // gains of t+1: K[a][j] at component a*NS + j of the blocked record, k[a] behind them
        const S* kb = p.Kk + bidx(t + 1, 0, NK, b, p.nW);
        S* Kflat = &sm.K[0][0];
#pragma unroll
        for (int e0 = 0; e0 < NC * NS; e0 += G)
          if (e0 + gl < NC * NS) Kflat[e0 + gl] = kb[(size_t)(e0 + gl) * kWarp];
        if (gl < NC) sm.k[gl] = kb[(size_t)(NC * NS + gl) * kWarp];
        // rows n_state.. of Q_{t+1} are contiguous in the record
        S* Quflat = &sm.Qu[0][0];
#pragma unroll
        for (int e0 = 0; e0 < NC * N; e0 += G)
          if (e0 + gl < NC * N) Quflat[e0 + gl] = rec[NS * N + e0 + gl];
        if (gl < NC) sm.qu[gl] = rec[N * N + NS + gl];
      }
      S Qrow[N], qme = S(0);
      if (gl < NS) {
#pragma unroll
        for (int j = 0; j < N; ++j) Qrow[j] = rec[gl * N + j];
        qme = rec[N * N + gl];
      }
      gsync(gmask);
      if (gl < NS) {
        S KQ[NC];
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          S acc = S(0);
#pragma unroll
          for (int c2 = 0; c2 < NC; ++c2) acc = fmaS<S>(sm.K[c2][gl], sm.Qu[c2][NS + a], acc);
          KQ[a] = acc;
        }
#pragma unroll
        for (int j = 0; j < NS; ++j) {
          S vrow_j;
          if constexpr (kChain) {
            S acc = Qrow[j];
#pragma unroll
            for (int a = 0; a < NC; ++a) acc = fmaS<S>(Qrow[NS + a], sm.K[a][j], acc);
#pragma unroll
            for (int a = 0; a < NC; ++a) acc = fmaS<S>(sm.K[a][gl], sm.Qu[a][j], acc);
#pragma unroll
            for (int a = 0; a < NC; ++a) acc = fmaS<S>(KQ[a], sm.K[a][j], acc);
            vrow_j = acc;
          } else {
            S t1 = S(0), t2 = S(0), t3 = S(0);
#pragma unroll
            for (int a = 0; a < NC; ++a) {
              t1 = fmaS<S>(Qrow[NS + a], sm.K[a][j], t1);
              t2 = fmaS<S>(sm.K[a][gl], sm.Qu[a][j], t2);
              t3 = fmaS<S>(KQ[a], sm.K[a][j], t3);
            }
            vrow_j = ((Qrow[j] + t1) + t2) + t3;
          }
          sm.V[gl][j] = vrow_j;   // nobody reads V before the group barrier below
        }
        S vv;
        if constexpr (kChain) {
          S acc = qme;
#pragma unroll
          for (int a = 0; a < NC; ++a) acc = fmaS<S>(Qrow[NS + a], sm.k[a], acc);
#pragma unroll
          for (int a = 0; a < NC; ++a) acc = fmaS<S>(sm.K[a][gl], sm.qu[a], acc);
#pragma unroll
          for (int a = 0; a < NC; ++a) acc = fmaS<S>(KQ[a], sm.k[a], acc);
          vv = acc;
        } else {
          S t1 = S(0), t2 = S(0), t3 = S(0);
#pragma unroll
          for (int a = 0; a < NC; ++a) {
            t1 = fmaS<S>(Qrow[NS + a], sm.k[a], t1);
            t2 = fmaS<S>(sm.K[a][gl], sm.qu[a], t2);
            t3 = fmaS<S>(KQ[a], sm.k[a], t3);
          }
          vv = ((qme + t1) + t2) + t3;
        }
        sm.v[gl] = vv;
      }
    }
    AC_TICK(0)
    // ---- (A) Q_t = C_t + F_t' V_{t+1} F_t,  q_t = C_t tau_t + c_t + F_t' v_{t+1}   (lqr_step.py:66-70,294)
    const bool flush = (p.take[b] & 1) != 0;   // lazy best-iterate tracking, see backward_sweep
    if (gl < N) {
      const S tv = p.traj_cur[bidx(t, gl, N, b, p.nW)];
      sm.tau[gl] = tv;
      if (flush) p.traj_best[bidx(t, gl, N, b, p.nW)] = tv;
    }
    if (kEnv && t < T - 1 && gl < NS) sm.xnext[gl] = p.traj_cur[bidx(t + 1, gl, N, b, p.nW)];
    gsync(gmask);
    AC_TICK(1)
    if (t < T - 1) {
      if constexpr (kEnv) {
        if (gl == 0) {   // one lane evaluates the analytic Jacobian straight into shared memory
          S tr[N], xn[NS];
#pragma unroll
          for (int i = 0; i < N; ++i) tr[i] = sm.tau[i];
#pragma unroll
          for (int i = 0; i < NS; ++i) xn[i] = sm.xnext[i];
          D::jacobian(p.dyn, tr, xn, sm.F);
        }
      } else {
        const S* Fg = p.F + ((size_t)t * p.B + b) * (NS * N);
        S* Fflat = &sm.F[0][0];
#pragma unroll
        for (int e0 = 0; e0 < NS * N; e0 += G)
          if (e0 + gl < NS * N) Fflat[e0 + gl] = __ldg(Fg + e0 + gl);
      }
    }
    AC_TICK(2)
    S Crow[N], cme = S(0);
    if (gl < N) {
      const S* Cg = cost_src<S>(p.C, p.C_bcast, t, p.B, b, N * N) + gl * N;
#pragma unroll
      for (int j = 0; j < N; ++j) Crow[j] = __ldg(Cg + j);
      cme = __ldg(cost_src<S>(p.c, p.c_bcast, t, p.B, b, N) + gl);
    }
    gsync(gmask);
    AC_TICK(3)
    if (gl < N) {
      S qv = kChain ? cme : S(0);
#pragma unroll
      for (int j = 0; j < N; ++j) qv = fmaS<S>(Crow[j], sm.tau[j], qv);
      if (!kChain) qv = qv + cme;
      if (t < T - 1) {
        // M[k] = sum_i F[i][l] V[i][k]: i outermost, so every step feeds NS independent
        // accumulators from one row of V (each M[k] still sums over i in ascending order);
        // the lane's column of F is re-read from shared memory rather than kept in registers
        S M[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) M[k] = S(0);
        S fv = kChain ? qv : S(0);
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          const S f = sm.F[i][gl];
#pragma unroll
          for (int k = 0; k < NS; ++k) M[k] = fmaS<S>(f, sm.V[i][k], M[k]);
          fv = fmaS<S>(f, sm.v[i], fv);
        }
        qv = kChain ? fv : qv + fv;
        if constexpr (kChain) {
#pragma unroll
          for (int k = 0; k < NS; ++k) {
#pragma unroll
            for (int j = 0; j < N; ++j)
              if (D::nz(k, j)) Crow[j] = fmaS<S>(M[k], sm.F[k][j], Crow[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < N; ++j) {
            S acc = S(0);
#pragma unroll
            for (int k = 0; k < NS; ++k)
              if (D::nz(k, j)) acc = fmaS<S>(M[k], sm.F[k][j], acc);
            Crow[j] = Crow[j] + acc;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < N; ++j) rec[gl * N + j] = Crow[j];
      rec[N * N + gl] = qv;
      if (gl >= NS) {
        // the control rows once more, lane-interleaved over the batch: what phase B (one
        // thread per problem) reads, coalesced
        S* gi = p.gsG + ((size_t)(b >> 5) * GIN) * kWarp + (b & 31);
        const int a = gl - NS;
#pragma unroll
        for (int j = 0; j < N; ++j) gi[(size_t)(a * N + j) * kWarp] = Crow[j];
        gi[(size_t)(NC * N + a) * kWarp] = qv;
      }
    }
    gsync(gmask);   // the shared block is reused by this group's next problem
    AC_TICK(4)
  }

  // ---------------------------------------------------------------- phase B, one thread per problem
  // Gains of timestep t from (Q_uu, Q_ux, q_u): plain / masked / regularised solves
  // (lqr_step.py:84-127, lqr_step_backup.py:202-205) or pnqp (lqr_step.py:128-148).
  DILQR_DEVICE static void phase_b(const IterParams<S>& p, int t, int b, bool active, int lane,
                                   S (&kprev)[NC], bool& have_prev, SubBarrier& sb) {
    const int bs = active ? b : 0;           // spare threads shadow problem 0 (never vote / write)
    const S* gi = p.gsG + ((size_t)(bs >> 5) * GIN) * kWarp + (bs & 31);
    // Q_uu, q_u and the columns of Q_ux come from the lane-interleaved record (coalesced);
    // every column of K is stored as soon as it is solved
    S H[NC][NC], qu[NC], tau_u[NC];
#pragma unroll
    for (int a = 0; a < NC; ++a) {
#pragma unroll
      for (int c2 = 0; c2 < NC; ++c2) H[a][c2] = gi[(size_t)(a * N + NS + c2) * kWarp];
      qu[a] = gi[(size_t)(NC * N + a) * kWarp];
      tau_u[a] = p.traj_cur[bidx(t, NS + a, N, bs, p.nW)];
    }
    auto qux = [&](int a, int j) -> S { return gi[(size_t)(a * N + j) * kWarp]; };
    S* ko = p.Kk + bidx(t, 0, NK, bs, p.nW);
    auto put_K = [&](int a, int j, S v) {
      if (active) ko[(a * NS + j) * kWarp] = v;
    };
    auto put_k = [&](int a, S v) {
      if (active) ko[(NC * NS + a) * kWarp] = v;
    };
    if (p.bounds_kind == 0) {
      bool mask[NC];
#pragma unroll
      for (int a = 0; a < NC; ++a)
        mask[a] = p.zeroI ? (p.zeroI[((size_t)t * p.B + bs) * NC + a] != 0) : false;
      if (NC == 1) {
        if (!p.zeroI) {  // lqr_step.py:84-86
          const S r = S(1) / H[0][0];
#pragma unroll
          for (int j = 0; j < NS; ++j) put_K(0, j, -(r * qux(0, j)));
          put_k(0, -(r * qu[0]));
        } else {         // lqr_step.py:101-123
          const S quu_m = mask[0] ? S(1e-8) : H[0][0];
          const S r = S(1) / quu_m;
#pragma unroll
          for (int j = 0; j < NS; ++j) put_K(0, j, -(r * (mask[0] ? S(0) : qux(0, j))));
          put_k(0, -((S(1) / H[0][0]) * (mask[0] ? S(0) : qu[0])));
        }
      } else if (!p.zeroI && p.gain_solve == 1) {  // lqr_step_backup.py:202-205
        Chol<S, NC> ch;
#pragma unroll
        for (int a = 0; a < NC; ++a)
#pragma unroll
          for (int c2 = 0; c2 < NC; ++c2) ch.l[a][c2] = H[a][c2] + (a == c2 ? S(1e-6) : S(0));
        ch.factor();
#pragma unroll
        for (int j = 0; j <= NS; ++j) {
          S rhs[NC];
#pragma unroll
          for (int a = 0; a < NC; ++a) rhs[a] = (j < NS) ? qux(a, j < NS ? j : 0) : qu[a];
          ch.solve(rhs);
#pragma unroll
          for (int a = 0; a < NC; ++a) {
            if (j < NS) put_K(a, j, -rhs[a]);
            else put_k(a, -rhs[a]);
          }
        }
      } else {  // plain solve / u_zero_I-masked LU solve (lqr_step.py:88-94,101-127)
        LUpp<S, NC> lu;
#pragma unroll
        for (int a = 0; a < NC; ++a)
#pragma unroll
          for (int c2 = 0; c2 < NC; ++c2) {
            S h = (mask[a] || mask[c2]) ? S(0) : H[a][c2];
            if (a == c2 && mask[a]) h = h + S(1e-8);
            lu.a[a][c2] = h;
          }
        lu.factor();
#pragma unroll
        for (int j = 0; j <= NS; ++j) {
          S rhs[NC];
#pragma unroll
          for (int a = 0; a < NC; ++a)
            rhs[a] = mask[a] ? S(0) : ((j < NS) ? qux(a, j < NS ? j : 0) : qu[a]);
          lu.solve(rhs);
#pragma unroll
          for (int a = 0; a < NC; ++a) {
            if (j < NS) put_K(a, j, -rhs[a]);
            else put_k(a, -rhs[a]);
          }
        }
      }
    } else {  // box constraints: pnqp   (lqr_step.py:128-148)
      S lo[NC], hi[NC], k[NC];
      if (p.bounds_kind == 2) {
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          lo[a] = __ldg(p.lo_t + ((size_t)t * p.B + bs) * NC + a);
          hi[a] = __ldg(p.hi_t + ((size_t)t * p.B + bs) * NC + a);
        }
      } else {
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          lo[a] = p.lo;
          hi[a] = p.hi;
        }
      }
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        lo[a] = lo[a] - tau_u[a];
        hi[a] = hi[a] - tau_u[a];
        if (p.has_delta) {   // lqr_step.py:132-134
          if (lo[a] < -p.delta_u) lo[a] = -p.delta_u;
          if (hi[a] > p.delta_u) hi[a] = p.delta_u;
        }
        k[a] = have_prev ? kprev[a] : S(0);
      }
      bool If[NC];
      LUpp<S, NC> lu;
      S rinv = S(0);
      pnqp_thread<S, NC, true>(H, qu, lo, hi, have_prev, k, If, lu,
                               p.guess + (size_t)t * kPnqpMaxIter, make_uint4(0, 0, 0, 0),
                               p.votes + (size_t)t * kPnqpMaxIter, p.solo != 0, active, lane, &rinv, &sb);
      have_prev = true;
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        kprev[a] = k[a];
        put_k(a, k[a]);
      }
      if (NC == 1) {  // lqr_step.py:144-146
#pragma unroll
        for (int j = 0; j < NS; ++j) put_K(0, j, -(rinv * (If[0] ? qux(0, j) : S(0))));
      } else {        // lqr_step.py:148
#pragma unroll
        for (int j = 0; j < NS; ++j) {
          S rhs[NC];
#pragma unroll
          for (int a = 0; a < NC; ++a) rhs[a] = If[a] ? qux(a, j) : S(0);
          lu.solve(rhs);
#pragma unroll
          for (int a = 0; a < NC; ++a) put_K(a, j, -rhs[a]);
        }
      }
    }
  }
};

// One Riccati / pnqp sweep over the whole batch (cooperative launch; gridDim.x * 256 >= B).
#ifndef DILQR_GS_MINBLOCKS
#define DILQR_GS_MINBLOCKS 2
#endif
template <class S, int NS, int NC, int DYN>
__global__ void __launch_bounds__(256, DILQR_GS_MINBLOCKS) group_sweep_kernel(const __grid_constant__ IterParams<S> p) {
  using GS = GroupSweep<S, NS, NC, DYN>;
  namespace cg = cooperative_groups;
  cg::grid_group grid = cg::this_grid();
  extern __shared__ __align__(16) char smem[];
  if (p.halt && *reinterpret_cast<const volatile uint32_t*>(p.halt)) return;   // uniform over the grid
  const int lane = threadIdx.x & 31;
  const int gi = threadIdx.x / GS::G, gl = threadIdx.x % GS::G;
  const unsigned gmask = (GS::G == 32) ? kFull : (0xffffu << (16 * (lane >> 4)));
  typename GS::Shared& sm = reinterpret_cast<typename GS::Shared*>(smem)[gi];
  const int n_groups = gridDim.x * GS::GPB;
  const int my_group = blockIdx.x * GS::GPB + gi;
  const int tid = blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = tid < p.B;
  // phase B involves only the blocks that own problems; their pnqp decisions synchronise
  // over a SubBarrier, the rest of the grid waits at the phase boundary
  const unsigned nb_b = (unsigned)((p.B + GS::kThreads - 1) / GS::kThreads);
  const bool in_b = blockIdx.x < nb_b;
  SubBarrier sb{p.gs_barrier, nb_b, 0u};
  S kprev[NC];
#pragma unroll
  for (int a = 0; a < NC; ++a) kprev[a] = S(0);
  bool have_prev = false;
#ifdef DILQR_GS_TIMING
  long long t_ac = 0, t_s1 = 0, t_b = 0, t_s2 = 0, c0, c1;
  long long tacc[5] = {0, 0, 0, 0, 0};
#define GS_TICK(acc) c1 = clock64(); acc += c1 - c0; c0 = c1;
  c0 = clock64();
#else
#define GS_TICK(acc)
#endif
  for (int t = p.T - 1; t >= 0; --t) {
    for (int b = my_group; b < p.B; b += n_groups) {
      // the rows this lane will need for the group's NEXT problem: on their way to L1 while
      // the current problem is worked on (every phase of phase_ac starts with dependent loads)
      const int bn = b + n_groups;
      if (bn < p.B && gl < GS::N) {
        prefetch_l1(p.gsQ + (size_t)bn * GS::QREC + gl * GS::N);
        if (!p.C_bcast) prefetch_l1(p.C + (((size_t)t * p.B + bn) * GS::N + gl) * GS::N);
        prefetch_l1(p.traj_cur + bidx(t, gl, GS::N, bn, p.nW));
      }
#ifdef DILQR_GS_TIMING
      GS::phase_ac(p, sm, b, t, gl, gmask, tacc);
#else
      GS::phase_ac(p, sm, b, t, gl, gmask);
#endif
    }
    GS_TICK(t_ac)
    grid.sync();
    GS_TICK(t_s1)
    if (in_b) GS::phase_b(p, t, tid, active, lane, kprev, have_prev, sb);
    GS_TICK(t_b)
    grid.sync();
    GS_TICK(t_s2)
  }
#ifdef DILQR_GS_TIMING
  if (threadIdx.x == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1 || blockIdx.x == nb_b))
    printf("gs block %d/%d: phase AC %lld  sync %lld  phase B %lld  sync %lld cycles (in_b %d) | AC parts: "
           "C %lld  tau %lld  F %lld  rows %lld  compute+store %lld\n",
           blockIdx.x, gridDim.x, t_ac, t_s1, t_b, t_s2, (int)in_b, tacc[0], tacc[1], tacc[2], tacc[3], tacc[4]);
#endif
}

}  // namespace dilqr
