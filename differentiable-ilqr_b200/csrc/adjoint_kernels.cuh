// adjoint_kernels.cuh -- the adjoint (KKT) LQR solves of the DiLQR backward for
// env_dx dynamics, factored once and replayed per Richardson pass.
//
// The reference performs every adjoint solve as a full
//   mpc_backup.MPC(lqr_iter=1, u_zero_I=active set)(0, QuadCost(C,-r), LinDx(F,None))
// (lqr_step_explicit.py:276-303): Riccati sweep + rollout + line search.  For a
// fixed problem (C, F = D(tau*), active set) only the affine terms depend on r:
//   q_t = -r_t + F_t' v_{t+1},  k_t = -Hm_t^{-1} (q_u masked),
//   v_t = q_x + (Q_xu + K_t' Q_uu) k_t + K_t' q_u          (lqr_step.py:156-158)
// so the quadratic part (K_t, Hm_t^{-1}, Q_xu + K'Q_uu, Q_uu) is computed ONCE
// (adjoint_factor_kernel) and each Richardson pass only runs the cheap affine
// backward sweep + the linear rollout dx_{t+1} = F_t [dx_t; K_t dx_t + k_t], fused
// with the Richardson update w_t = g_t - Lam_t dtau_t (adjoint_pass_kernel).
// F_t is re-derived from (x*_t, u*_t) in registers instead of being read from HBM.
//
// Line search of the reference's adjoint MPC: the step alpha = 1 is the exact
// minimiser of the (masked) QP, whose optimal value sum_t (q_u'k + 1/2 k'Q_uu k) is
// <= 0 whenever Q_uu > 0 on the free set, so the reference accepts alpha = 1.  Each
// pass evaluates that value and counts the problems where it is positive (or NaN)
// into resid[2]; the host falls back to the generic (line-searching) kernels if the
// count is non-zero.
#pragma once
#include "common.cuh"
#include "dynamics.cuh"
#include "smallmat.cuh"
#include "ilqr_kernels.cuh"
#include "env_tables_gen.cuh"
#include "../../include/dilqr.h"

namespace dilqr {

DILQR_DEVICE void bulk_s2g(void* dst_global, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_global),
               "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
DILQR_DEVICE void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
DILQR_DEVICE void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
DILQR_DEVICE void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
DILQR_DEVICE void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Lam_t[k][j] = sum_i lam_{t+1}[i] dD_t[i][j]/dtau_k is structurally sparse (cartpole:
// D does not depend on x, dx and has constant columns) -- the factored path stores only
// the entries that can be non-zero, warp-blocked [T-1][B/32][NLAM][32].
template <class S, int DYN>
struct LamPack {
  using TB = EnvTables<S, DYN>;
  static constexpr int NS = Dyn<S, DYN>::NS, NC = Dyn<S, DYN>::NC, N = NS + NC;
  __host__ __device__ static constexpr bool nz(int k, int j) {
    for (int i = 0; i < NS; ++i)
      if (k < NS ? TB::nz_Dx(i, j, k < NS ? k : 0) : TB::nz_Du(i, j, k < NS ? 0 : k - NS)) return true;
    return false;
  }
  __host__ __device__ static constexpr int idx(int k, int j) {   // position of (k,j) in the pack
    int c = 0;
    for (int e = 0; e < k * N + j; ++e)
      if (nz(e / N, e % N)) ++c;
    return c;
  }
  static constexpr int NLAM = idx(N - 1, N - 1) + (nz(N - 1, N - 1) ? 1 : 0);
};

template <class S>
struct AdjParams {
  int T, B, Bp;
  int bounds_kind;   // 0: no active set; 1: scalar bounds -> I = |u - bound| <= 1e-8
  int gain_solve;
  int final_pass;
  int C_bcast, c_bcast;  // cost layout (0 dense, 1 [T,..], 2 [..]); for a broadcast C (c) the
                         // final pass writes per-warp partial sums of dC (dc) -- layout
                         // [T][n_warps][..] (mode 1) or [n_warps][..] (mode 2) -- instead of slabs
  S lo, hi;
  const S* C;
  const S* x;
  const S* u;
  const S* g;
  const S* Lam;
  S* w;
  S* fac;     // [T][NFAC][Bp]
  S* kvec;    // [T][NC][Bp]
  S* dtau;    // [T][N][Bp]
  S* dC;
  S* dc;
  S* df;
  S* dx_out;
  S* du_out;
  unsigned long long* resid;   // [0] max|dw| [1] max|w| (double bits), [2] #rejected problems
  const S* Cpk;                // packed symmetric copy of C left by the solve (optional) ...
  const uint32_t* cpk_state;   // ... valid iff *cpk_state == 1
  const S* gx;                 // [T,B,ns] upstream gradient wrt x (NULL: zero)
  const S* gu;                 // [T,B,nc] upstream gradient wrt u
  int first;                   // this solve's right-hand side is g itself (w == g)
  int want_resid;              // reduce max|dw|, max|w| (costs one extra read of w)
  int reduce_tile;             // final pass: red_out instead of dC, dc
  S* red_out;                  // [n_warps][2N]
  S* df_blk;                   // final pass: df warp-blocked [T-1][Bp/32][NS][32] (optional)
  DynParams<S> dyn;
};

template <class S, int DYN>
struct Adj {
  using D = Dyn<S, DYN>;
  static constexpr int NS = D::NS, NC = D::NC, N = D::N;
  // per (t, problem) factor record: K[NC][NS], G[NC][NC] (inverse of the masked
  // Q_uu), M[NS][NC] = Q_xu + K'Q_uu, Quu[NC][NC]
  static constexpr int OFF_K = 0, OFF_G = NC * NS, OFF_M = OFF_G + NC * NC,
                       OFF_Q = OFF_M + NS * NC, NFAC = OFF_Q + NC * NC;

  DILQR_DEVICE static bool active(const AdjParams<S>& p, S uv) {
    if (p.bounds_kind == 0) return false;
    return (absS<S>(uv - p.lo) <= S(1e-8)) || (absS<S>(uv - p.hi) <= S(1e-8));
  }

  // F_t = D(x_t, u_t); sin/cos of the new angle are components of x_{t+1}
  DILQR_DEVICE static void jac_at(const AdjParams<S>& p, const S* tau, const S* xnext,
                                  S (*F)[N]) {
    D::jacobian(p.dyn, tau, xnext, F);
  }

  DILQR_DEVICE static void load_tau(const AdjParams<S>& p, int t, int b, S* tau) {
    const size_t tb = (size_t)t * p.B + b;
#pragma unroll
    for (int i = 0; i < NS; ++i) tau[i] = __ldg(p.x + tb * NS + i);
#pragma unroll
    for (int a = 0; a < NC; ++a) tau[NS + a] = __ldg(p.u + tb * NC + a);
  }
};

// ---------------------------------------------------------------------------
// Factor: masked Riccati sweep at tau* (lqr_step.py:99-127 / lqr_step_backup.py:
// 196-228), storing what the affine passes need.
// ---------------------------------------------------------------------------
template <class S, int DYN>
__global__ void __launch_bounds__(128) adjoint_factor_kernel(const __grid_constant__ AdjParams<S> p) {
  using A = Adj<S, DYN>;
  constexpr int NS = A::NS, NC = A::NC, N = A::N, NFAC = A::NFAC;
  extern __shared__ __align__(128) char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int b0 = (blockIdx.x * wpb + warp) * kWarp;
  if (b0 >= p.B) return;
  const int nvalid = min(kWarp, p.B - b0);
  const bool act = lane < nvalid;
  const int b = act ? b0 + lane : b0;
  // the packed symmetric copy of C the solve left in its workspace (21 instead of 36 scalars
  // for cartpole), when the caller hands it over and it is valid
  constexpr int NP = N * (N + 1) / 2;
  const bool packedC = p.Cpk && p.cpk_state && !p.C_bcast &&
                       *reinterpret_cast<const volatile uint32_t*>(p.cpk_state) == 1u;
  const uint32_t elems_dense[1] = {N * N};
  const uint32_t elems[1] = {packedC ? (uint32_t)NP : (uint32_t)(N * N)};
  const size_t per_warp = WarpStager<S>::bytes_per_warp(1, elems_dense) + kStages * sizeof(uint64_t);
  char* wbase = smem + warp * per_warp;
  WarpStager<S> st;
  st.init(wbase + kStages * sizeof(uint64_t), reinterpret_cast<uint64_t*>(wbase), lane, nvalid, 1,
          elems, packedC ? 1u : 0u, p.C_bcast ? 1u : 0u);
  const int T = p.T;
  const int nWc = p.Bp / kWarp;
  auto issue = [&](int stage, int t) {
    const S* src[1] = {packedC ? p.Cpk + bidx(t, 0, NP, b0, nWc)
                               : cost_src<S>(p.C, p.C_bcast, t, p.B, b0, N * N)};
    st.issue(stage, src, 1);
  };
  S V[NS][NS], xnext[NS];
  issue(0, T - 1);
  for (int t = T - 1; t >= 0; --t) {
    const int sg = (T - 1 - t) & 1;
    if (t > 0) issue(sg ^ 1, t - 1);
    S tau[N];
    A::load_tau(p, t, b, tau);
    st.wait(sg);
    S Q[N][N];
    if (packedC) {
      const S* Cs = st.seg_ptr(sg, 0) + lane;
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) Q[i][j] = Cs[pk_idx<N>(i, j) * kWarp];
    } else {
      const S* Cs = st.lane_ptr(sg, 0);
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) Q[i][j] = Cs[i * N + j];
    }
    if (t < T - 1) {
      S Fm[NS][N];
      A::jac_at(p, tau, xnext, Fm);
#pragma unroll
      for (int i = 0; i < N; ++i) {
        S Mr[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) {
          S acc = S(0);
#pragma unroll
          for (int l = 0; l < NS; ++l) acc = fmaS<S>(Fm[l][i], V[l][k], acc);
          Mr[k] = acc;
        }
#pragma unroll
        for (int j = 0; j < N; ++j) {
          S acc = S(0);
#pragma unroll
          for (int k = 0; k < NS; ++k) acc = fmaS<S>(Mr[k], Fm[k][j], acc);
          Q[i][j] = Q[i][j] + acc;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) xnext[i] = tau[i];
    bool mask[NC];
#pragma unroll
    for (int a = 0; a < NC; ++a) mask[a] = A::active(p, tau[NS + a]);
    S K[NC][NS], G[NC][NC];
    if (NC == 1) {
      if (p.bounds_kind == 0) {                 // lqr_step.py:84-86
        const S r = S(1) / Q[NS][NS];
#pragma unroll
        for (int j = 0; j < NS; ++j) K[0][j] = -(r * Q[NS][j]);
        G[0][0] = r;
      } else {                                  // lqr_step.py:101-123
        const S r = S(1) / (mask[0] ? S(1e-8) : Q[NS][NS]);
#pragma unroll
        for (int j = 0; j < NS; ++j) K[0][j] = -(r * (mask[0] ? S(0) : Q[NS][j]));
        G[0][0] = S(1) / Q[NS][NS];             // k uses the UNMASKED Q_uu (lqr_step.py:123)
      }
    } else if (p.bounds_kind == 0 && p.gain_solve == 1) {   // lqr_step_backup.py:202-205
      Chol<S, NC> ch;
#pragma unroll
      for (int a = 0; a < NC; ++a)
#pragma unroll
        for (int c2 = 0; c2 < NC; ++c2)
          ch.l[a][c2] = Q[NS + a][NS + c2] + (a == c2 ? S(1e-6) : S(0));
      ch.factor();
#pragma unroll
      for (int j = 0; j < NS + NC; ++j) {
        S rhs[NC];
#pragma unroll
        for (int a = 0; a < NC; ++a) rhs[a] = (j < NS) ? Q[NS + a][j] : (a == j - NS ? S(1) : S(0));
        ch.solve(rhs);
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          if (j < NS) K[a][j] = -rhs[a];
          else G[a][j - NS < NC ? j - NS : 0] = rhs[a];
        }
      }
    } else {                                    // lqr_step.py:88-94 / 101-127
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
      for (int j = 0; j < NS + NC; ++j) {
        S rhs[NC];
#pragma unroll
        for (int a = 0; a < NC; ++a)
          rhs[a] = (j < NS) ? (mask[a] ? S(0) : Q[NS + a][j]) : (a == j - NS ? S(1) : S(0));
        lu.solve(rhs);
#pragma unroll
        for (int a = 0; a < NC; ++a) {
          if (j < NS) K[a][j] = -rhs[a];
          else G[a][j - NS < NC ? j - NS : 0] = rhs[a];
        }
      }
    }
    S KQ[NS][NC];
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        S acc = S(0);
#pragma unroll
        for (int c2 = 0; c2 < NC; ++c2) acc = fmaS<S>(K[c2][i], Q[NS + c2][NS + a], acc);
        KQ[i][a] = acc;
      }
    {
      S* f = p.fac + bidx(t, 0, NFAC, b0 + lane, p.Bp / kWarp);   // own (padded) column
#pragma unroll
      for (int a = 0; a < NC; ++a)
#pragma unroll
        for (int j = 0; j < NS; ++j) f[(A::OFF_K + a * NS + j) * kWarp] = K[a][j];
#pragma unroll
      for (int a = 0; a < NC; ++a)
#pragma unroll
        for (int c2 = 0; c2 < NC; ++c2) {
          f[(A::OFF_G + a * NC + c2) * kWarp] = G[a][c2];
          f[(A::OFF_Q + a * NC + c2) * kWarp] = Q[NS + a][NS + c2];
        }
#pragma unroll
      for (int i = 0; i < NS; ++i)
#pragma unroll
        for (int a = 0; a < NC; ++a) f[(A::OFF_M + i * NC + a) * kWarp] = Q[i][NS + a] + KQ[i][a];
    }
#pragma unroll
    for (int i = 0; i < NS; ++i)
#pragma unroll
      for (int j = 0; j < NS; ++j) {
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
}

// ---------------------------------------------------------------------------
// One adjoint solve with r = w (affine sweep + linear rollout).
//   FINAL == false: fused Richardson update  w_t <- g_t - Lam_t dtau_t.
//   FINAL == true : keeps dtau (workspace + optional AoS dx_out/du_out), then a
//                   costate sweep (lqr_step.py:371-385) produces dC, dc, df -- dense, or
//                   (reduce_tile) already reduced to the gradient of the tiled diagonal
//                   cost: sum_{t,b} diag(dC), sum_{t,b} dc, per-warp partial sums.
// Every per-timestep operand (w / g, x*, u*, factor record, Lam, k, dtau, C) is staged
// through shared memory by TMA one step ahead of its use; the segment table of the stage
// is re-laid out between the sweeps (WarpStager::reconfigure).
//   p.first: this is the first solve of the Richardson iteration, w == g: the right-hand
//            side is read from g (no w <- g copy is ever made).
//   g is handed over as its two halves gx[T,B,ns] (may be NULL: zero) and gu[T,B,nc],
//            the upstream gradients as autograd delivers them (no concatenation).
// ---------------------------------------------------------------------------
template <class S, int DYN>
struct AdjStage {
  using A = Adj<S, DYN>;
  static constexpr int NS = A::NS, NC = A::NC, N = A::N, NFAC = A::NFAC;
  static constexpr int NP = N * (N + 1) / 2;
  static constexpr int NLAM = LamPack<S, DYN>::NLAM;
  static constexpr int kNSeg = 8;
  using Stager = WarpStager<S, kNSeg>;
  // sweep A (affine backward): 0 w[N]  1 x[NS]  2 u[NC]  3 fac[NFAC]*  4 gx[NS]  5 gu[NC]
  // sweep B (rollout):         0 Lam[NLAM]*  1 x  2 u  3 K[NC*NS]* (prefix of the factor
  //                            record)  4 gx  5 gu  6 kvec[NC]*
  // sweep C (costates, FINAL): 0 C[N*N] (slab) or Cpk[NP]*  1 x  2 u  3 dtau[N]*  4 gx  5 gu
  //                            7 w[N]                                  (* = warp-blocked)
  static __host__ __device__ void elems_A(uint32_t* e) {
    e[0] = N; e[1] = NS; e[2] = NC; e[3] = NFAC; e[4] = NS; e[5] = NC; e[6] = 0; e[7] = 0;
  }
  static __host__ __device__ void elems_B(uint32_t* e, bool fin) {
    e[0] = fin ? 0 : NLAM; e[1] = NS; e[2] = NC; e[3] = NC * NS; e[4] = fin ? 0 : NS;
    e[5] = fin ? 0 : NC; e[6] = NC; e[7] = 0;
  }
  static __host__ __device__ void elems_C(uint32_t* e, bool packed) {
    e[0] = packed ? NP : N * N; e[1] = NS; e[2] = NC; e[3] = N; e[4] = NS; e[5] = NC; e[6] = 0;
    e[7] = N;
  }
  static __host__ __device__ size_t stage_bytes(bool fin) {
    uint32_t e[kNSeg];
    elems_A(e);
    size_t m = Stager::bytes_per_warp(kNSeg, e);
    elems_B(e, fin);
    size_t v = Stager::bytes_per_warp(kNSeg, e);
    m = v > m ? v : m;
    if (fin) {
      elems_C(e, false);
      v = Stager::bytes_per_warp(kNSeg, e);
      m = v > m ? v : m;
    }
    return m;
  }
  static __host__ __device__ size_t out_bytes(bool fin) {
    return fin ? (((size_t)kWarp * (N * N + N) * sizeof(S) + 15) & ~(size_t)15) : 0;
  }
  static __host__ __device__ size_t smem_per_warp(bool fin) {
    return stage_bytes(fin) + kStages * sizeof(uint64_t) + out_bytes(fin);
  }
};

template <class S, int DYN, bool FINAL, bool REDUCE = false>
__global__ void __launch_bounds__(64) adjoint_pass_kernel(const __grid_constant__ AdjParams<S> p) {
  using A = Adj<S, DYN>;
  using AS = AdjStage<S, DYN>;
  constexpr int NS = A::NS, NC = A::NC, N = A::N, NFAC = A::NFAC;
  extern __shared__ __align__(128) char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  const int b0 = (blockIdx.x * wpb + warp) * kWarp;
  if (b0 >= p.B) return;
  const int nvalid = min(kWarp, p.B - b0);
  const bool act = lane < nvalid;
  const int b = act ? b0 + lane : b0;     // API tensors
  const int bw = b0 + lane;               // own workspace column
  const int T = p.T;
  const int nW = p.Bp / kWarp;
  const size_t per_warp = AS::smem_per_warp(FINAL);
  char* wbase = smem + warp * per_warp;
  typename AS::Stager st;
  {
    uint32_t e[AS::kNSeg];
    AS::elems_A(e);
    st.init(wbase + kStages * sizeof(uint64_t), reinterpret_cast<uint64_t*>(wbase), lane, nvalid,
            AS::kNSeg, e, 1u << 3);
  }
  S* outC = reinterpret_cast<S*>(wbase + kStages * sizeof(uint64_t) + AS::stage_bytes(FINAL));
  S* outc = outC + kWarp * N * N;

  auto slab = [&](const S* base, int elems) {
    return base ? base + (size_t)b0 * elems : nullptr;
  };
  const long long sz = (long long)sizeof(S);
  const long long chunk = (long long)nW * kWarp * sz;   // bytes per timestep per component
  const bool first = p.first != 0;
  // right-hand side r_t of this solve: w_t, or (first) g_t = [gx_t; gu_t]
  const uint32_t rmask = first ? ((p.gx ? 1u << 4 : 0u) | (1u << 5)) : 1u;
  auto bind_common = [&]() {
    st.bind(1, slab(p.x, NS), (long long)p.B * NS * sz);
    st.bind(2, slab(p.u, NC), (long long)p.B * NC * sz);
    st.bind(4, slab(p.gx, NS), (long long)p.B * NS * sz);
    st.bind(5, slab(p.gu, NC), (long long)p.B * NC * sz);
  };
  // r_t[i] from the staged right-hand side
  auto rhs = [&](int sg, int wseg, S* r) {
    if (first) {
      const S* gxs = st.lane_ptr(sg, 4);
      const S* gus = st.lane_ptr(sg, 5);
#pragma unroll
      for (int i = 0; i < NS; ++i) r[i] = p.gx ? gxs[i] : S(0);
#pragma unroll
      for (int a = 0; a < NC; ++a) r[NS + a] = gus[a];
    } else {
      const S* ws_ = st.lane_ptr(sg, wseg);
#pragma unroll
      for (int i = 0; i < N; ++i) r[i] = ws_[i];
    }
  };

  // ---------------- affine backward sweep
  bind_common();
  st.bind(0, slab(p.w, N), (long long)p.B * N * sz);
  st.bind(3, p.fac + bidx(0, 0, NFAC, b0, nW), chunk * NFAC);
  auto issue_a = [&](int stage, int t) { st.issue_bound(stage, t, 0xeu | rmask); };
  S v[NS], xnext[NS];
  S pred = S(0);
  issue_a(0, T - 1);
  for (int t = T - 1; t >= 0; --t) {
    const int sg = (T - 1 - t) & 1;
    if (t > 0) issue_a(sg ^ 1, t - 1);
    st.wait(sg);
    const S* xs_ = st.lane_ptr(sg, 1);
    const S* us_ = st.lane_ptr(sg, 2);
    const S* f = st.seg_ptr(sg, 3) + lane;
    S tau[N], q[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) tau[i] = xs_[i];
#pragma unroll
    for (int a = 0; a < NC; ++a) tau[NS + a] = us_[a];
    rhs(sg, 0, q);
#pragma unroll
    for (int i = 0; i < N; ++i) q[i] = -q[i];
    if (t < T - 1) {
      S Fm[NS][N];
      A::jac_at(p, tau, xnext, Fm);
#pragma unroll
      for (int i = 0; i < N; ++i) {
        S acc = S(0);
#pragma unroll
        for (int l = 0; l < NS; ++l) acc = fmaS<S>(Fm[l][i], v[l], acc);
        q[i] = q[i] + acc;
      }
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) xnext[i] = tau[i];
    S qm[NC], k[NC];
#pragma unroll
    for (int a = 0; a < NC; ++a) qm[a] = A::active(p, tau[NS + a]) ? S(0) : q[NS + a];
#pragma unroll
    for (int a = 0; a < NC; ++a) {
      S acc = S(0);
#pragma unroll
      for (int c2 = 0; c2 < NC; ++c2) acc = fmaS<S>(f[(A::OFF_G + a * NC + c2) * kWarp], qm[c2], acc);
      k[a] = -acc;
    }
    // optimal value of the masked QP: sum_t q_u'k + 1/2 k'Q_uu k
#pragma unroll
    for (int a = 0; a < NC; ++a) {
      S hk = S(0);
#pragma unroll
      for (int c2 = 0; c2 < NC; ++c2) hk = fmaS<S>(f[(A::OFF_Q + a * NC + c2) * kWarp], k[c2], hk);
      pred = fmaS<S>(k[a], q[NS + a] + S(0.5) * hk, pred);
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      S t1 = S(0), t2 = S(0);
#pragma unroll
      for (int a = 0; a < NC; ++a) {
        t1 = fmaS<S>(f[(A::OFF_M + i * NC + a) * kWarp], k[a], t1);
        t2 = fmaS<S>(f[(A::OFF_K + a * NS + i) * kWarp], q[NS + a], t2);
      }
      v[i] = (q[i] + t1) + t2;
    }
    {
      S* ko = p.kvec + bidx(t, 0, NC, bw, nW);
#pragma unroll
      for (int a = 0; a < NC; ++a) ko[a * kWarp] = k[a];
    }
  }
  if (act && !(pred <= S(0))) atomicAdd(&p.resid[2], 1ull);
  // kvec (generic-proxy stores) is read back through TMA below
  __threadfence();
  asm volatile("fence.proxy.async;" ::: "memory");
  __syncwarp();

  // ---------------- linear rollout (+ Richardson update)
  {
    uint32_t e[AS::kNSeg];
    AS::elems_B(e, FINAL);
    st.reconfigure(AS::kNSeg, e, (1u << 0) | (1u << 3) | (1u << 6));
  }
  bind_common();
  if (!FINAL) st.bind(0, p.Lam + bidx(0, 0, AS::NLAM, b0, nW), chunk * AS::NLAM);
  st.bind(3, p.fac + bidx(0, 0, NFAC, b0, nW), chunk * NFAC);   // K = leading NC*NS components
  st.bind(6, p.kvec + bidx(0, 0, NC, b0, nW), chunk * NC);
  const uint32_t gmask = (p.gx ? 1u << 4 : 0u) | (1u << 5);
  auto issue_f = [&](int stage, int t) {
    st.issue_bound(stage, t, FINAL ? 0x4eu : (0x4eu | gmask | ((t < T - 1) ? 1u : 0u)));
  };
  S dt[N], tprev[N];
  double dmax = 0.0, wmax = 0.0;
  issue_f(0, 0);
  for (int t = 0; t < T; ++t) {
    const int sg = t & 1;
    if (t + 1 < T) issue_f(sg ^ 1, t + 1);
    st.wait(sg);
    const S* xs_ = st.lane_ptr(sg, 1);
    const S* us_ = st.lane_ptr(sg, 2);
    const S* f = st.seg_ptr(sg, 3) + lane;
    const S* kv = st.seg_ptr(sg, 6) + lane;
    // previous iterate w_t (only for the residual of the Richardson update): fetched now,
    // used at the end of the step, so the global-load latency hides behind the arithmetic
    S wold[N];
    if (!FINAL && p.want_resid) {
#pragma unroll
      for (int k2 = 0; k2 < N; ++k2) {
        S wv = S(0);
        if (act) {
          if (!first) wv = p.w[((size_t)t * p.B + b) * N + k2];
          else if (k2 < NS) wv = p.gx ? p.gx[((size_t)t * p.B + b) * NS + k2] : S(0);
          else wv = p.gu[((size_t)t * p.B + b) * NC + (k2 - NS)];
        }
        wold[k2] = wv;
      }
    }
    S tau[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) tau[i] = xs_[i];
#pragma unroll
    for (int a = 0; a < NC; ++a) tau[NS + a] = us_[a];
    // dx_t = F_{t-1} dtau_{t-1}; the trig of F_{t-1} is part of x_t (just arrived)
    S dx[NS];
    if (t > 0) {
      S Fm[NS][N];
      A::jac_at(p, tprev, tau, Fm);
#pragma unroll
      for (int i = 0; i < NS; ++i) {
        S acc = S(0);
#pragma unroll
        for (int j = 0; j < N; ++j) acc = fmaS<S>(Fm[i][j], dt[j], acc);
        dx[i] = acc;
      }
    } else {
#pragma unroll
      for (int i = 0; i < NS; ++i) dx[i] = S(0);
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) dt[i] = dx[i];
#pragma unroll
    for (int a = 0; a < NC; ++a) {
      S acc = S(0);
      if (t > 0) {
#pragma unroll
        for (int j = 0; j < NS; ++j) acc = fmaS<S>(f[(A::OFF_K + a * NS + j) * kWarp], dx[j], acc);
      }
      S un = acc + kv[a * kWarp];
      if (A::active(p, tau[NS + a])) un = S(0);          // lqr_step.py:197-198
      dt[NS + a] = un;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) tprev[i] = tau[i];
    if (FINAL) {
      S* dto = p.dtau + bidx(t, 0, N, bw, nW);
#pragma unroll
      for (int i = 0; i < N; ++i) dto[i * kWarp] = dt[i];
      if (act) {
        const size_t tb = (size_t)t * p.B + b;
        if (p.dx_out) {
#pragma unroll
          for (int i = 0; i < NS; ++i) p.dx_out[tb * NS + i] = dt[i];
        }
        if (p.du_out) {
#pragma unroll
          for (int a = 0; a < NC; ++a) p.du_out[tb * NC + a] = dt[NS + a];
        }
      }
    } else {
      const S* Ls = st.seg_ptr(sg, 0) + lane;     // packed Lam_t, lane-interleaved
      const S* gxs = st.lane_ptr(sg, 4);
      const S* gus = st.lane_ptr(sg, 5);
      const size_t tb = (size_t)t * p.B + b;
      using LP = LamPack<S, DYN>;
      static_for<0, N>([&](auto K2) {
        constexpr int k2 = decltype(K2)::value;
        S acc = S(0);
        if (t < T - 1) {
          static_for<0, N>([&](auto J) {
            constexpr int j = decltype(J)::value;
            if constexpr (LP::nz(k2, j)) {
              constexpr int e = LP::idx(k2, j);
              acc = fmaS<S>(Ls[e * kWarp], dt[j], acc);
            }
          });
        }
        const S gk = k2 < NS ? (p.gx ? gxs[k2 < NS ? k2 : 0] : S(0)) : gus[k2 < NS ? 0 : k2 - NS];
        const S wn = gk - acc;
        if (act) {
          if (p.want_resid) {
            const S wo = wold[k2];
            dmax = fmax(dmax, fabs((double)wn - (double)wo));
            wmax = fmax(wmax, fabs((double)wn));
          }
          p.w[tb * N + k2] = wn;
        }
      });
    }
  }
  if (!FINAL) {
    if (p.want_resid) {
      for (int o = 16; o > 0; o >>= 1) {
        dmax = fmax(dmax, __shfl_xor_sync(kFull, dmax, o));
        wmax = fmax(wmax, __shfl_xor_sync(kFull, wmax, o));
      }
      if (lane == 0) {
        atomicMax(&p.resid[0], dbits(dmax));
        atomicMax(&p.resid[1], dbits(wmax));
      }
    }
    return;
  }

  // ---------------- final pass: costate sweep + gradient assembly
  //   dlam_t = Cxx dx + Cxu du - r_x + Fx' dlam_{t+1}          (lqr_step.py:371-385)
  //   dC_t = -1/2 (dtau tau' + tau dtau'), dc_t = -dtau, df_t = -dlam_{t+1}
  __threadfence();
  asm volatile("fence.proxy.async;" ::: "memory");
  __syncwarp();
  const bool packedC = p.Cpk && p.cpk_state && !p.C_bcast &&
                       *reinterpret_cast<const volatile uint32_t*>(p.cpk_state) == 1u;
  {
    uint32_t e[AS::kNSeg];
    AS::elems_C(e, packedC);
    st.reconfigure(AS::kNSeg, e, (1u << 3) | (packedC ? 1u : 0u), p.C_bcast ? 1u : 0u);
  }
  bind_common();
  if (packedC)
    st.bind(0, p.Cpk + bidx(0, 0, AS::NP, b0, nW), chunk * AS::NP);
  else
    st.bind(0, cost_src<S>(p.C, p.C_bcast, 0, p.B, b0, N * N),
            p.C_bcast == 0 ? (long long)p.B * N * N * sz : (p.C_bcast == 1 ? (long long)N * N * sz : 0));
  st.bind(3, p.dtau + bidx(0, 0, N, b0, nW), chunk * N);
  st.bind(7, slab(p.w, N), (long long)p.B * N * sz);
  auto issue_b = [&](int stage, int t) {
    st.issue_bound(stage, t, 0xfu | (first ? rmask : (1u << 7)));
  };
  constexpr bool reduce = REDUCE;
  // a bulk store needs a 16-byte aligned destination: the slab of step t starts t * B rows in,
  // so the row stride B * N (N * N) scalars must be a 16-byte multiple too (FP32, N = 6 and an
  // odd B is not)
  const bool bulk_out = !reduce && (nvalid == kWarp) &&
                        ((((size_t)N * N * sizeof(S) * kWarp) & 15) == 0) &&
                        ((((size_t)N * sizeof(S) * kWarp) & 15) == 0) &&
                        ((((size_t)p.B * N * N * sizeof(S)) & 15) == 0) &&
                        ((((size_t)p.B * N * sizeof(S)) & 15) == 0) &&
                        ((reinterpret_cast<uintptr_t>(p.dC) & 15) == 0) &&
                        ((reinterpret_cast<uintptr_t>(p.dc) & 15) == 0) &&
                        (p.C_bcast == 0 || p.c_bcast == 0);
  const int gwarp = b0 / kWarp;
  auto warp_sum = [&](S v) -> S {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = v + __shfl_xor_sync(kFull, v, o);
    return v;
  };
  // mode-2 accumulators (sum over t of this lane's contributions); none in REDUCE mode
  S accC[REDUCE ? 1 : N][REDUCE ? 1 : N], accc[N];
  S redq[N];               // reduce_tile: sum over t of diag(dC_t)  (dc sums go to accc)
#pragma unroll
  for (int i = 0; i < N; ++i) {
    accc[i] = S(0);
    redq[i] = S(0);
  }
  if constexpr (!REDUCE) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) accC[i][j] = S(0);
  }
  S dlam[NS];
  issue_b(0, T - 1);
  for (int t = T - 1; t >= 0; --t) {
    const int sg = (T - 1 - t) & 1;
    if (t > 0) issue_b(sg ^ 1, t - 1);
    st.wait(sg);
    const S* Cs = packedC ? st.seg_ptr(sg, 0) + lane : st.lane_ptr(sg, 0);
    const S* xs_ = st.lane_ptr(sg, 1);
    const S* us_ = st.lane_ptr(sg, 2);
    const S* ds_ = st.seg_ptr(sg, 3) + lane;
    S tt[N], dtv[N], rv[N];
#pragma unroll
    for (int i = 0; i < NS; ++i) tt[i] = xs_[i];
#pragma unroll
    for (int a = 0; a < NC; ++a) tt[NS + a] = us_[a];
#pragma unroll
    for (int i = 0; i < N; ++i) dtv[i] = ds_[i * kWarp];
    rhs(sg, 7, rv);
    const size_t tb = (size_t)t * p.B + b;
    if (t < T - 1) {
      if (p.df_blk) {
        S* o = p.df_blk + bidx(t, 0, NS, bw, nW);
#pragma unroll
        for (int i = 0; i < NS; ++i) o[i * kWarp] = -dlam[i];
      } else if (p.df && act) {
#pragma unroll
        for (int i = 0; i < NS; ++i) p.df[tb * NS + i] = -dlam[i];
      }
    }
    if constexpr (reduce) {
      // gradient of the tiled diagonal cost (il_env.py:159-162): only diag(dC) and dc survive
      // the adjoint of the tiling -- accumulated here instead of writing dC, dc out
      if (act) {
#pragma unroll
        for (int i = 0; i < N; ++i) {
          redq[i] = redq[i] + S(-0.5) * (dtv[i] * tt[i] + tt[i] * dtv[i]);
          accc[i] = accc[i] + (-dtv[i]);
        }
      }
    } else {
    // dense outputs go through shared memory, one bulk store per warp slab
    if (bulk_out) {
      bulk_wait_read0();
      __syncwarp();
    }
    if (p.dC) {
      if (p.C_bcast == 0) {
        S* oC = bulk_out ? outC + lane * (N * N) : p.dC + tb * (N * N);
        if (act || bulk_out) {
#pragma unroll
          for (int i = 0; i < N; ++i)
#pragma unroll
            for (int j = 0; j < N; ++j) oC[i * N + j] = S(-0.5) * (dtv[i] * tt[j] + tt[i] * dtv[j]);
        }
      } else {   // gradient of a broadcast C: sum over the batch (and time)
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = 0; j < N; ++j) {
            const S v = act ? S(-0.5) * (dtv[i] * tt[j] + tt[i] * dtv[j]) : S(0);
            if (p.C_bcast == 2) {
              accC[i][j] = accC[i][j] + v;
            } else {
              const S r = warp_sum(v);
              if (lane == 0) p.dC[((size_t)t * gridDim.x * wpb + gwarp) * (N * N) + i * N + j] = r;
            }
          }
      }
    }
    if (p.dc) {
      if (p.c_bcast == 0) {
        S* oc = bulk_out ? outc + lane * N : p.dc + tb * N;
        if (act || bulk_out) {
#pragma unroll
          for (int i = 0; i < N; ++i) oc[i] = -dtv[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const S v = act ? -dtv[i] : S(0);
          if (p.c_bcast == 2) {
            accc[i] = accc[i] + v;
          } else {
            const S r = warp_sum(v);
            if (lane == 0) p.dc[((size_t)t * gridDim.x * wpb + gwarp) * N + i] = r;
          }
        }
      }
    }
    if (bulk_out) {
      fence_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (p.dC && p.C_bcast == 0)
          bulk_s2g(p.dC + ((size_t)t * p.B + b0) * (N * N), outC, kWarp * N * N * sizeof(S));
        if (p.dc && p.c_bcast == 0)
          bulk_s2g(p.dc + ((size_t)t * p.B + b0) * N, outc, kWarp * N * sizeof(S));
        bulk_commit();
      }
    }
    }
    S nd[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      S d1 = S(0), d2 = S(0);
      if (packedC) {
#pragma unroll
        for (int j = 0; j < NS; ++j) d1 = fmaS<S>(Cs[pk_idx<N>(i, j) * kWarp], dtv[j], d1);
#pragma unroll
        for (int a = 0; a < NC; ++a) d2 = fmaS<S>(Cs[pk_idx<N>(i, NS + a) * kWarp], dtv[NS + a], d2);
      } else {
#pragma unroll
        for (int j = 0; j < NS; ++j) d1 = fmaS<S>(Cs[i * N + j], dtv[j], d1);
#pragma unroll
        for (int a = 0; a < NC; ++a) d2 = fmaS<S>(Cs[i * N + NS + a], dtv[NS + a], d2);
      }
      nd[i] = (d1 + d2) - rv[i];
    }
    if (t < T - 1) {
      S Fm[NS][N];
      A::jac_at(p, tt, xnext, Fm);
#pragma unroll
      for (int i = 0; i < NS; ++i) {
        S d1 = S(0);
#pragma unroll
        for (int l = 0; l < NS; ++l) d1 = fmaS<S>(Fm[l][i], dlam[l], d1);
        nd[i] = nd[i] + d1;
      }
    }
#pragma unroll
    for (int i = 0; i < NS; ++i) {
      dlam[i] = nd[i];
      xnext[i] = tt[i];
    }
  }
  if (bulk_out) bulk_wait0();
  if constexpr (reduce) {
    // red_out[n_warps][2N]: per-warp partial sums, summed over the warp axis by the caller
    // (fixed order: deterministic)
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const S rq = warp_sum(redq[i]);
      const S rc = warp_sum(accc[i]);
      if (lane == 0) {
        p.red_out[(size_t)gwarp * (2 * N) + i] = rq;
        p.red_out[(size_t)gwarp * (2 * N) + N + i] = rc;
      }
    }
    return;
  } else {
  if (p.dC && p.C_bcast == 2) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) {
        const S r = warp_sum(accC[i][j]);
        if (lane == 0) p.dC[(size_t)gwarp * (N * N) + i * N + j] = r;
      }
  }
  if (p.dc && p.c_bcast == 2) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const S r = warp_sum(accc[i]);
      if (lane == 0) p.dc[(size_t)gwarp * N + i] = r;
    }
  }
  }
}

}  // namespace dilqr
