// dilqr_backward.cuh -- kernels of the DiLQR implicit-differentiation backward
// pass (lqr_step_explicit.py:652-712 + fix_point_equ 458-598) in its matrix-free
// form (SURVEY Appendix C).
//
// With tau* the converged trajectory, the reference solves
//     A X = B,   A = I - (J_F dD/dtau + J_f dd/dtau)           (dense, (T n)^3)
// where J_F, J_f are Jacobians of the LQR solution wrt (F, f) obtained from T*n
// KKT adjoint solves.  Equivalent and matrix-free:  solve A' w = g by the
// Richardson iteration  w <- g + M' w;  M' w needs ONE adjoint LQR solve with
// r = w:  with dtau the adjoint solution and lambda the costates of the primal
// solution (lqr_step.py:355-369),
//     dF_w = -(dlam_{t+1} tau' + lam_{t+1} dtau'),  df_w = -dlam_{t+1}
//     (M' w)_t[k] = sum_ij (dF_w - df_w tau')[i,j] dD_t[i,j]/dtau_k
//                 = - sum_j Lam_t[k][j] dtau_t[j],
//     Lam_t[k][j] = sum_i lam_{t+1}[i] dD_t[i,j]/dtau_k          (independent of w).
// Finally dC, dc come from one more KKT pass with r = w (kkt_grads_kernel) and
//     dtheta_b = sum_t <dF_w, dD_t/dtheta> + <df_w, dd_t/dtheta>
// with the total derivatives dD/dtheta, dd/dtheta of the closed-loop
// sensitivity rollout grad_input (cartpole.py:717-788), contracted on the fly.
#pragma once
#include "common.cuh"
#include "dynamics.cuh"
#include "env_tables_gen.cuh"
#include "adjoint_kernels.cuh"

namespace dilqr {

// ---------------------------------------------------------------------------
// Primal costates lambda_t (lqr_step.py:355-369) and the contracted second-order
// tables Lam_t.  One thread per problem, reverse sweep.
//   lam  [T,B,ns]      Lam [T-1,B,n,n]  (row k = d/dtau_k, col j)
// ---------------------------------------------------------------------------
template <class S, int DYN>
struct CostateStage {
  using D = Dyn<S, DYN>;
  static constexpr int NS = D::NS, NC = D::NC, N = D::N;
  static constexpr int kNSeg = 4;   // C[N*N], c[N], x[NS], u[NC]
  static __host__ __device__ void seg_elems(uint32_t* e) {
    e[0] = N * N;
    e[1] = N;
    e[2] = NS;
    e[3] = NC;
  }
  static __host__ __device__ size_t out_bytes() {
    return ((size_t)kWarp * (N * N) * sizeof(S) + 15) & ~(size_t)15;
  }
  static __host__ __device__ size_t smem_per_warp() {
    uint32_t e[kNSeg];
    seg_elems(e);
    return WarpStager<S>::bytes_per_warp(kNSeg, e) + kStages * sizeof(uint64_t) + out_bytes();
  }
};

// PACKED: Lam_out is the packed, warp-blocked layout [T-1][B/32][NLAM][32] consumed by
// the factored adjoint passes; otherwise dense [T-1,B,n,n] (richardson_update_kernel).
template <class S, int DYN, bool PACKED>
__global__ void __launch_bounds__(64)
costate_tables_kernel(DynParams<S> P, int T, int B, const S* __restrict__ C,
                      const S* __restrict__ c, const S* __restrict__ x, const S* __restrict__ u,
                      S* __restrict__ lam_out, S* __restrict__ Lam_out, int C_bcast, int c_bcast) {
  using D = Dyn<S, DYN>;
  using TB = EnvTables<S, DYN>;
  using CS = CostateStage<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC, N = D::N, NTH = TB::NTH;
  extern __shared__ __align__(128) char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int b0 = (blockIdx.x * wpb + warp) * kWarp;
  if (b0 >= B) return;
  const int nvalid = min(kWarp, B - b0);
  const bool act = lane < nvalid;
  const int b = act ? b0 + lane : b0;
  char* wbase = smem + warp * CS::smem_per_warp();
  WarpStager<S> st;
  {
    uint32_t e[CS::kNSeg];
    CS::seg_elems(e);
    st.init(wbase + kStages * sizeof(uint64_t), reinterpret_cast<uint64_t*>(wbase), lane, nvalid,
            CS::kNSeg, e, 0, (C_bcast ? 1u : 0u) | (c_bcast ? 2u : 0u));
  }
  S* outL = reinterpret_cast<S*>(wbase + CS::smem_per_warp() - CS::out_bytes());
  auto issue = [&](int stage, int t) {
    const size_t o = (size_t)t * B + b0;
    const S* src[CS::kNSeg] = {cost_src<S>(C, C_bcast, t, B, b0, N * N),
                               cost_src<S>(c, c_bcast, t, B, b0, N), x + o * NS, u + o * NC};
    st.issue(stage, src, CS::kNSeg);
  };
  // a bulk store needs a 16-byte aligned destination: the slab of step t starts t * B rows in
  const bool bulk_out = !PACKED && (nvalid == kWarp) &&
                        ((((size_t)N * N * sizeof(S) * kWarp) & 15) == 0) &&
                        ((((size_t)B * N * N * sizeof(S)) & 15) == 0) &&
                        ((reinterpret_cast<uintptr_t>(Lam_out) & 15) == 0);
  using LP = LamPack<S, DYN>;
  const int nWp = (B + kWarp - 1) / kWarp;
  S lam[NS];
  issue(0, T - 1);
  for (int t = T - 1; t >= 0; --t) {
    const int sg = (T - 1 - t) & 1;
    if (t > 0) issue(sg ^ 1, t - 1);
    st.wait(sg);
    const S* Cs = st.lane_ptr(sg, 0);
    const S* cs = st.lane_ptr(sg, 1);
    const S* xs_ = st.lane_ptr(sg, 2);
    const S* us_ = st.lane_ptr(sg, 3);
    const size_t tb = (size_t)t * B + b;
    S tau[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) tau[i] = xs_[i];
#pragma unroll
    for (int a = 0; a < NC; ++a) tau[NS + a] = us_[a];
    S Dm[NS][N];
    if (t < T - 1) {
      S Dth[NS][N][NTH], Dx[NS][N][NS], Du[NS][N][NC], xth[NS][NTH], xx[NS][NS], xu[NS][NC];
      TB::eval(P, tau, &tau[NS], Dm, Dth, Dx, Du, xth, xx, xu);
      // Lam_t[k][j] = sum_i lam_{t+1}[i] dD[i][j]/dtau_k
      if (bulk_out) {
        bulk_wait_read0();
        __syncwarp();
      }
      S* Lo = bulk_out ? outL + lane * (N * N) : Lam_out + tb * (N * N);
      if (PACKED) Lo = Lam_out + bidx(t, 0, LP::NLAM, b0 + lane, nWp);   // own (padded) column
      if (act || bulk_out || PACKED) {
static_for<0, N>([&](auto KK) {
          constexpr int k = decltype(KK)::value;
          static_for<0, N>([&](auto JJ) {
            constexpr int j = decltype(JJ)::value;
            if constexpr (!PACKED || LP::nz(k, j)) {
              S acc = S(0);
#pragma unroll
              for (int i = 0; i < NS; ++i) {
                if (k < NS) {
                  if (TB::nz_Dx(i, j, k < NS ? k : 0))
                    acc = fmaS<S>(lam[i], Dx[i][j][k < NS ? k : 0], acc);
                } else {
                  if (TB::nz_Du(i, j, k < NS ? 0 : k - NS))
                    acc = fmaS<S>(lam[i], Du[i][j][k < NS ? 0 : k - NS], acc);
                }
              }
              if constexpr (PACKED) {
                constexpr int e = LP::idx(k, j);
                Lo[e * kWarp] = acc;
              } else {
                Lo[k * N + j] = acc;
              }
            }
          });
        });
      }
      if (bulk_out) {
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
          bulk_s2g(Lam_out + ((size_t)t * B + b0) * (N * N), outL, kWarp * N * N * sizeof(S));
          bulk_commit();
        }
      }
    }
    S nl[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      S a1 = S(0), a2 = S(0);
#pragma unroll
      for (int j = 0; j < NS; ++j) a1 = fmaS<S>(Cs[i * N + j], tau[j], a1);
#pragma unroll
      for (int a = 0; a < NC; ++a) a2 = fmaS<S>(Cs[i * N + NS + a], tau[NS + a], a2);
      nl[i] = (a1 + a2) + cs[i];
    }
    if (t < T - 1) {
#pragma unroll
      for (int i = 0; i < NS; ++i) {
        S a1 = S(0);
#pragma unroll
        for (int l = 0; l < NS; ++l)
          if (TB::nz_D(l, i)) a1 = fmaS<S>(Dm[l][i], lam[l], a1);
        nl[i] = nl[i] + a1;
      }
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      lam[i] = nl[i];
      if (act) lam_out[tb * NS + i] = nl[i];
    }
  }
  if (bulk_out) bulk_wait0();
}

// ---------------------------------------------------------------------------
// Contracted second-order tables alone: Lam_t (packed, warp-blocked) from tau*_t and
// lam_{t+1} (blocked [T][B/32][NS][32], written by the gains sweep).  No recursion in t is
// left once the costates are known, so this is ONE THREAD PER (t, problem): 50x the
// parallelism of the costate sweep, throughput- instead of latency-bound.
// ---------------------------------------------------------------------------
template <class S, int DYN>
__global__ void __launch_bounds__(128)
lam_tables_kernel(DynParams<S> P, int T, int B, const S* __restrict__ x, const S* __restrict__ u,
                  const S* __restrict__ lam_blk, S* __restrict__ Lam_out) {
  using D = Dyn<S, DYN>;
  using TB = EnvTables<S, DYN>;
  using LP = LamPack<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC, N = D::N, NTH = TB::NTH;
  const int bw = blockIdx.x * blockDim.x + threadIdx.x;   // own (padded) column
  const int t = blockIdx.y;
  const int nW = (B + kWarp - 1) / kWarp;
  if (bw >= nW * kWarp || t >= T - 1) return;
  const int b = bw < B ? bw : B - 1;
  const size_t tb = (size_t)t * B + b;
  S tau[N], lam[NS];
#pragma unroll
  for (int i = 0; i < NS; ++i) tau[i] = __ldg(x + tb * NS + i);
#pragma unroll
  for (int a = 0; a < NC; ++a) tau[NS + a] = __ldg(u + tb * NC + a);
  {
    const S* ls = lam_blk + bidx(t + 1, 0, NS, bw, nW);
#pragma unroll
    for (int i = 0; i < NS; ++i) lam[i] = ls[i * kWarp];
  }
  S Dm[NS][N], Dth[NS][N][NTH], Dx[NS][N][NS], Du[NS][N][NC], xth[NS][NTH], xx[NS][NS], xu[NS][NC];
  TB::eval(P, tau, &tau[NS], Dm, Dth, Dx, Du, xth, xx, xu);
  S* Lo = Lam_out + bidx(t, 0, LP::NLAM, bw, nW);
  static_for<0, N>([&](auto KK) {
    constexpr int k = decltype(KK)::value;
    static_for<0, N>([&](auto JJ) {
      constexpr int j = decltype(JJ)::value;
      if constexpr (LP::nz(k, j)) {
        S acc = S(0);
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          if (k < NS) {
            if (TB::nz_Dx(i, j, k < NS ? k : 0)) acc = fmaS<S>(lam[i], Dx[i][j][k < NS ? k : 0], acc);
          } else {
            if (TB::nz_Du(i, j, k < NS ? 0 : k - NS))
              acc = fmaS<S>(lam[i], Du[i][j][k < NS ? 0 : k - NS], acc);
          }
        }
        constexpr int e = LP::idx(k, j);
        Lo[e * kWarp] = acc;
      }
    });
  });
}

// ---------------------------------------------------------------------------
// Richardson update  w_t = g_t - Lam_t dtau_t  (t < T-1),  w_{T-1} = g_{T-1};
// also writes -w (the linear cost of the next adjoint solve) and reduces
// max|w_new - w_old| and max|w_new| into resid[0], resid[1] (ordered-uint max).
// One thread per (t, b).
// ---------------------------------------------------------------------------
template <class S, int NS, int NC>
__global__ void richardson_update_kernel(int T, int B, const S* __restrict__ g,
                                         const S* __restrict__ Lam, const S* __restrict__ dx,
                                         const S* __restrict__ du, S* __restrict__ w,
                                         S* __restrict__ negw,
                                         unsigned long long* __restrict__ resid) {
  constexpr int N = NS + NC;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  const int t = blockIdx.y;
  double dmax = 0.0, wmax = 0.0;
  if (b < B) {
    const size_t tb = (size_t)t * B + b;
    S dt[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) dt[i] = dx[tb * NS + i];
#pragma unroll
    for (int a = 0; a < NC; ++a) dt[NS + a] = du[tb * NC + a];
#pragma unroll
    for (int k = 0; k < N; ++k) {
      S acc = S(0);
      if (t < T - 1) {
#pragma unroll
        for (int j = 0; j < N; ++j) acc = fmaS<S>(Lam[tb * (N * N) + k * N + j], dt[j], acc);
      }
      const S wn = g[tb * N + k] - acc;
      const S wo = w[tb * N + k];
      dmax = fmax(dmax, fabs((double)wn - (double)wo));
      wmax = fmax(wmax, fabs((double)wn));
      w[tb * N + k] = wn;
      negw[tb * N + k] = -wn;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    dmax = fmax(dmax, __shfl_xor_sync(kFull, dmax, o));
    wmax = fmax(wmax, __shfl_xor_sync(kFull, wmax, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&resid[0], dbits(dmax));
    atomicMax(&resid[1], dbits(wmax));
  }
}

// ---------------------------------------------------------------------------
// dtheta: closed-loop sensitivity rollout (cartpole.py:755-782) contracted on
// the fly with the adjoint quantities.  One thread per problem, forward sweep.
//   K      [T,B,nc,ns]  gains of the final LQR pass in FORWARD time order; the
//                       reference indexes its reverse-time stack with t
//                       (SURVEY 8a-10 quirk), i.e. uses K_{T-1-t} at step t.
//   lam    [T,B,ns]     primal costates           dx,du: adjoint solution (r = w)
//   df     [T-1,B,ns]   = -dlam_{t+1}             dtheta [B,nth]
// ---------------------------------------------------------------------------
template <class S, int DYN>
__global__ void __launch_bounds__(128)
sens_theta_kernel(DynParams<S> P, int T, int B, const S* __restrict__ x,
                  const S* __restrict__ u, const S* __restrict__ K, const S* __restrict__ lam,
                  const S* __restrict__ dx, const S* __restrict__ du, const S* __restrict__ df,
                  S* __restrict__ dtheta) {
  using D = Dyn<S, DYN>;
  using TB = EnvTables<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC, N = D::N, NTH = TB::NTH;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  auto ldK = [&](int t, int e) -> S { return K[((size_t)t * B + b) * (NC * NS) + e]; };
  auto ldlam = [&](int t, int i) -> S { return lam[((size_t)t * B + b) * NS + i]; };
  auto lddtau = [&](int t, int i) -> S {
    return i < NS ? dx[((size_t)t * B + b) * NS + i] : du[((size_t)t * B + b) * NC + (i - NS)];
  };
  auto lddf = [&](int t, int i) -> S { return df[((size_t)t * B + b) * NS + i]; };
  S G[NS][NTH], Gp[NS][NTH], Dprev[NS][N], Kp[NC][NS];
  S acc[NTH];
#pragma unroll
  for (int q = 0; q < NTH; ++q) acc[q] = S(0);
#pragma unroll
  for (int i = 0; i < NS; ++i)
#pragma unroll
    for (int q = 0; q < NTH; ++q) G[i][q] = S(0);
  for (int t = 0; t < T; ++t) {
    const size_t tb = (size_t)t * B + b;
    if (t + 1 < T) {   // next step's operands on their way while this step's tables are evaluated
      const size_t nb = tb + B;
      prefetch_l1(x + nb * NS);
      prefetch_l1(u + nb * NC);
      prefetch_l1(dx + nb * NS);
      prefetch_l1(du + nb * NC);
      prefetch_l1(lam + nb * NS);
      prefetch_l1(df + tb * NS);
      if (t + 2 < T) prefetch_l1(K + ((size_t)(T - 2 - t) * B + b) * (NC * NS));
    }
    S tau[N], dtau[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) tau[i] = x[tb * NS + i];
#pragma unroll
    for (int a = 0; a < NC; ++a) tau[NS + a] = u[tb * NC + a];
#pragma unroll
    for (int i = 0; i < N; ++i) dtau[i] = lddtau(t, i);
    S Dm[NS][N], Dth[NS][N][NTH], Dx[NS][N][NS], Du[NS][N][NC], xth[NS][NTH], xx[NS][NS],
        xu[NS][NC];
    TB::eval(P, tau, &tau[NS], Dm, Dth, Dx, Du, xth, xx, xu);
    S Kt[NC][NS];   // K_ref[t] = K_{T-1-t}
#pragma unroll
    for (int a = 0; a < NC; ++a)
#pragma unroll
      for (int j = 0; j < NS; ++j) Kt[a][j] = ldK(T - 1 - t, a * NS + j);
    if (t > 0) {
      // G_t = xth + (xx + xu K_ref[t-1]) G_{t-1}                 (cartpole.py:768)
      S A[NS][NS];
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int j = 0; j < NS; ++j) {
          S s = S(0);
#pragma unroll
          for (int a = 0; a < NC; ++a)
            if (TB::nz_xu(i, a)) s = fmaS<S>(xu[i][a], Kp[a][j], s);
          A[i][j] = (TB::nz_xx(i, j) ? xx[i][j] : S(0)) + s;
        }
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int q = 0; q < NTH; ++q) Gp[i][q] = G[i][q];
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int q = 0; q < NTH; ++q) {
          S s = S(0);
#pragma unroll
          for (int j = 0; j < NS; ++j) s = fmaS<S>(A[i][j], Gp[j][q], s);
          G[i][q] = (TB::nz_xth(i, q) ? xth[i][q] : S(0)) + s;
        }
      // <df_{t-1}, G_t - D_{t-1} [G_{t-1}; K_ref[t-1] G_{t-1}]>   (cartpole.py:778-782)
      S Z[N][NTH];
#pragma unroll
      for (int q = 0; q < NTH; ++q) {
#pragma unroll
        for (int j = 0; j < NS; ++j) Z[j][q] = Gp[j][q];
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          S s = S(0);
#pragma unroll
          for (int j = 0; j < NS; ++j) s = fmaS<S>(Kp[a][j], Gp[j][q], s);
          Z[NS + a][q] = s;
        }
      }
#pragma unroll
      for (int i = 0; i < NS; ++i) {
        const S dfi = lddf(t - 1, i);
#pragma unroll
        for (int q = 0; q < NTH; ++q) {
          S s = S(0);
#pragma unroll
          for (int m = 0; m < N; ++m)
            if (TB::nz_D(i, m)) s = fmaS<S>(Dprev[i][m], Z[m][q], s);
          acc[q] = fmaS<S>(dfi, G[i][q] - s, acc[q]);
        }
      }
    }
    if (t < T - 1) {
      // sum_ij W[i][j] gradD_t[i][j][:],  W = -lam_{t+1} dtau_t'
      // gradD = Dth + (Dx + Du K_ref[t]) G_t                      (cartpole.py:773-775)
      S lm[NS];
#pragma unroll
      for (int i = 0; i < NS; ++i) lm[i] = ldlam(t + 1, i);
      S om[NS];   // om[k] = sum_ij W_ij (Dx[i][j][k] + sum_a Du[i][j][a] K[a][k])
#pragma unroll
      for (int k = 0; k < NS; ++k) om[k] = S(0);
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const S wij = -(lm[i] * dtau[j]);
#pragma unroll
          for (int q = 0; q < NTH; ++q)
            if (TB::nz_Dth(i, j, q)) acc[q] = fmaS<S>(wij, Dth[i][j][q], acc[q]);
#pragma unroll
          for (int k = 0; k < NS; ++k) {
            bool any = TB::nz_Dx(i, j, k);
            S e = any ? Dx[i][j][k] : S(0);
#pragma unroll
            for (int a = 0; a < NC; ++a)
              if (TB::nz_Du(i, j, a)) {
                e = fmaS<S>(Du[i][j][a], Kt[a][k], e);
                any = true;
              }
            if (any) om[k] = fmaS<S>(wij, e, om[k]);
          }
        }
#pragma unroll
      for (int k = 0; k < NS; ++k)
#pragma unroll
        for (int q = 0; q < NTH; ++q) acc[q] = fmaS<S>(om[k], G[k][q], acc[q]);
    }
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) Dprev[i][j] = Dm[i][j];
#pragma unroll
    for (int a = 0; a < NC; ++a)
#pragma unroll
      for (int j = 0; j < NS; ++j) Kp[a][j] = Kt[a][j];
  }
#pragma unroll
  for (int q = 0; q < NTH; ++q) dtheta[(size_t)b * NTH + q] = acc[q];
}

// ---------------------------------------------------------------------------
// dtheta again, in ADJOINT form: same sum as sens_theta_kernel, but the 5 x n_theta
// sensitivity matrix G_t of the forward rollout is never formed.  With (loop variables of
// sens_theta_kernel) A_t = xx_t + xu_t K_ref[t-1], G_t = xth_t + A_t G_{t-1}, G_0 = 0,
//   dtheta = sum_{t<=T-2} W_t : Dth_t + sum_t c_t' G_t,      W_t = -lam_{t+1} dtau_t',
//   c_t = [t>=1] df_{t-1} + [t<=T-2] (om_t - (D_t,x + D_t,u K_ref[t])' df_t),
//   om_t = -(Lam_t,x dtau_t + K_ref[t]' Lam_t,u dtau_t)          (Lam_t: lam_tables_kernel),
// and  sum_t c_t' G_t = sum_{t>=1} mu_t' xth_t  with the reverse recursion
//   mu_{T-1} = c_{T-1},  mu_t = c_t + A_{t+1}' mu_{t+1}.
// One reverse sweep per problem carrying a vector of n_state scalars; the second-order tables
// Dx, Du (the bulk of EnvTables::eval) are not evaluated at all -- their contraction with
// lam is the packed Lam the Richardson passes already use.  Every operand in its blocked
// workspace layout.  (cartpole.py:717-788, pendulum.py:383-443)
// ---------------------------------------------------------------------------
template <class S, int DYN>
__global__ void __launch_bounds__(64)
sens_theta_adjoint_kernel(DynParams<S> P, int T, int B, const S* __restrict__ x,
                          const S* __restrict__ u, const S* __restrict__ K,
                          const S* __restrict__ lam, const S* __restrict__ dtau_b,
                          const S* __restrict__ df, const S* __restrict__ Lam,
                          S* __restrict__ dtheta) {
  using D = Dyn<S, DYN>;
  using TB = EnvTables<S, DYN>;
  using LP = LamPack<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC, N = D::N, NTH = TB::NTH;
  constexpr int NK = NC * NS + NC;
  const int bw = blockIdx.x * blockDim.x + threadIdx.x;
  const int nW = (B + kWarp - 1) / kWarp;
  if (bw >= nW * kWarp) return;
  const int b = bw < B ? bw : B - 1;
  S acc[NTH], nu[NS], dfn[NS], Kt[NC][NS];
#pragma unroll
  for (int q = 0; q < NTH; ++q) acc[q] = S(0);
#pragma unroll
  for (int i = 0; i < NS; ++i) nu[i] = dfn[i] = S(0);
#pragma unroll
  for (int a = 0; a < NC; ++a)
#pragma unroll
    for (int j = 0; j < NS; ++j) Kt[a][j] = K[bidx(0, a * NS + j, NK, bw, nW)];   // K_ref[T-1] = K_0
  for (int t = T - 1; t >= 0; --t) {
    const size_t tb = (size_t)t * B + b;
    if (t > 0) {
      prefetch_l1(x + (tb - B) * NS);
      prefetch_l1(u + (tb - B) * NC);
    }
    S tau[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) tau[i] = x[tb * NS + i];
#pragma unroll
    for (int a = 0; a < NC; ++a) tau[NS + a] = u[tb * NC + a];
    S Dm[NS][N], Dth[NS][N][NTH], Dx[NS][N][NS], Du[NS][N][NC], xth[NS][NTH], xx[NS][NS],
        xu[NS][NC];
    TB::eval(P, tau, &tau[NS], Dm, Dth, Dx, Du, xth, xx, xu);   // Dx, Du unused: eliminated
    S dfm[NS], mu[NS];   // df_{t-1}
#pragma unroll
    for (int i = 0; i < NS; ++i) dfm[i] = t >= 1 ? df[bidx(t - 1, i, NS, bw, nW)] : S(0);
    if (t <= T - 2) {
      S dtau[N], lm[NS], Ld[N];
#pragma unroll
      for (int i = 0; i < N; ++i) dtau[i] = dtau_b[bidx(t, i, N, bw, nW)];
#pragma unroll
      for (int i = 0; i < NS; ++i) lm[i] = lam[bidx(t + 1, i, NS, bw, nW)];
      static_for<0, N>([&](auto KK) {
        constexpr int k = decltype(KK)::value;
        S s = S(0);
        static_for<0, N>([&](auto JJ) {
          constexpr int j = decltype(JJ)::value;
          if constexpr (LP::nz(k, j)) s = fmaS<S>(Lam[bidx(t, LP::idx(k, j), LP::NLAM, bw, nW)], dtau[j], s);
        });
        Ld[k] = s;
      });
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        S om = Ld[k];
#pragma unroll
        for (int a = 0; a < NC; ++a) om = fmaS<S>(Kt[a][k], Ld[NS + a], om);
        S s = S(0);   // ((D_x + D_u K_ref[t])' df_t)[k]
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          S e = TB::nz_D(i, k) ? Dm[i][k] : S(0);
#pragma unroll
          for (int a = 0; a < NC; ++a)
            if (TB::nz_D(i, NS + a)) e = fmaS<S>(Dm[i][NS + a], Kt[a][k], e);
          s = fmaS<S>(dfn[i], e, s);
        }
        mu[k] = (dfm[k] - (om + s)) + nu[k];
      }
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) {
          const S wij = -(lm[i] * dtau[j]);
#pragma unroll
          for (int q = 0; q < NTH; ++q)
            if (TB::nz_Dth(i, j, q)) acc[q] = fmaS<S>(wij, Dth[i][j][q], acc[q]);
        }
    } else {
#pragma unroll
      for (int k = 0; k < NS; ++k) mu[k] = dfm[k];
    }
    if (t >= 1) {
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int q = 0; q < NTH; ++q)
          if (TB::nz_xth(i, q)) acc[q] = fmaS<S>(mu[i], xth[i][q], acc[q]);
      // nu_{t-1} = (xx_t + xu_t K_ref[t-1])' mu_t ; K_ref[t-1] = K_{T-t}
#pragma unroll
      for (int a = 0; a < NC; ++a)
#pragma unroll
        for (int j = 0; j < NS; ++j) Kt[a][j] = K[bidx(T - t, a * NS + j, NK, bw, nW)];
#pragma unroll
      for (int k = 0; k < NS; ++k) {
        S s = S(0);
#pragma unroll
        for (int i = 0; i < NS; ++i) {
          bool any = TB::nz_xx(i, k);
          S e = any ? xx[i][k] : S(0);
#pragma unroll
          for (int a = 0; a < NC; ++a)
            if (TB::nz_xu(i, a)) {
              e = fmaS<S>(xu[i][a], Kt[a][k], e);
              any = true;
            }
          if (any) s = fmaS<S>(mu[i], e, s);
        }
        nu[k] = s;
      }
#pragma unroll
      for (int i = 0; i < NS; ++i) dfn[i] = dfm[i];
    }
  }
  if (bw < B) {
#pragma unroll
    for (int q = 0; q < NTH; ++q) dtheta[(size_t)b * NTH + q] = acc[q];
  }
}

}  // namespace dilqr

namespace dilqr {

// ---------------------------------------------------------------------------
// get_matrices (cartpole.py:105-716, pendulum.py:152-382, rocket.py:258-261) as
// materialised tensors, one thread per sample row of x[N_,ns], u[N_,nc]:
//   D[N_,ns,n]  Dth[N_,ns,n,nth]  Dx[N_,ns,n,ns]  Du[N_,ns,n,nc]
//   xth[N_,ns,nth]  xx[N_,ns,ns]  xu[N_,ns,nc]
// (API compatibility; the backward pass itself never materialises them.)
// ---------------------------------------------------------------------------
template <class S, int DYN>
__global__ void __launch_bounds__(64)
env_tables_kernel(DynParams<S> P, int Nrows, const S* __restrict__ x, const S* __restrict__ u,
                  S* __restrict__ oD, S* __restrict__ oDth, S* __restrict__ oDx,
                  S* __restrict__ oDu, S* __restrict__ oxth, S* __restrict__ oxx,
                  S* __restrict__ oxu) {
  using D = Dyn<S, DYN>;
  using TB = EnvTables<S, DYN>;
  constexpr int NS = D::NS, NC = D::NC, N = D::N, NTH = TB::NTH;
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= Nrows) return;
  S tau[N];
#pragma unroll
  for (int i = 0; i < NS; ++i) tau[i] = x[(size_t)r * NS + i];
#pragma unroll
  for (int a = 0; a < NC; ++a) tau[NS + a] = u[(size_t)r * NC + a];
  S Dm[NS][N], Dth[NS][N][NTH], Dx[NS][N][NS], Du[NS][N][NC], xth[NS][NTH], xx[NS][NS], xu[NS][NC];
  TB::eval(P, tau, &tau[NS], Dm, Dth, Dx, Du, xth, xx, xu);
#pragma unroll
  for (int i = 0; i < NS; ++i) {
#pragma unroll
    for (int j = 0; j < N; ++j) {
      oD[((size_t)r * NS + i) * N + j] = TB::nz_D(i, j) ? Dm[i][j] : S(0);
#pragma unroll
      for (int q = 0; q < NTH; ++q)
        oDth[(((size_t)r * NS + i) * N + j) * NTH + q] = TB::nz_Dth(i, j, q) ? Dth[i][j][q] : S(0);
#pragma unroll
      for (int k = 0; k < NS; ++k)
        oDx[(((size_t)r * NS + i) * N + j) * NS + k] = TB::nz_Dx(i, j, k) ? Dx[i][j][k] : S(0);
#pragma unroll
      for (int a = 0; a < NC; ++a)
        oDu[(((size_t)r * NS + i) * N + j) * NC + a] = TB::nz_Du(i, j, a) ? Du[i][j][a] : S(0);
    }
#pragma unroll
    for (int q = 0; q < NTH; ++q)
      oxth[((size_t)r * NS + i) * NTH + q] = TB::nz_xth(i, q) ? xth[i][q] : S(0);
#pragma unroll
    for (int k = 0; k < NS; ++k) oxx[((size_t)r * NS + i) * NS + k] = TB::nz_xx(i, k) ? xx[i][k] : S(0);
#pragma unroll
    for (int a = 0; a < NC; ++a) oxu[((size_t)r * NS + i) * NC + a] = TB::nz_xu(i, a) ? xu[i][a] : S(0);
  }
}

}  // namespace dilqr
