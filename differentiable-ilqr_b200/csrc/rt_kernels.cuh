// rt_kernels.cuh -- LinDx iLQR kernels whose dimensions are runtime values (DILQR_DYN_LINDX_RT).
//
// The compiled family (ilqr_kernels.cuh) keeps a problem's whole Riccati state in one thread's
// registers, so every (n_state, n_ctrl) has to be instantiated.  This family serves any shape
// with n_state + n_ctrl <= 32:
//   - ONE WARP PER PROBLEM, lane r owns row r of V, Q, F'V and the gains;
//   - V_{t+1}, F_t, Q_t, the n_ctrl x n_ctrl factor and the small vectors live in the warp's
//     slice of dynamic shared memory, every loop has a runtime bound;
//   - C[t,b] and F[t,b] are contiguous blocks of the API tensors: the warp copies them into
//     shared memory with coalesced loads;
//   - the workspace (trajectories, gains, per-problem bookkeeping) has the layout of the compiled
//     family, so commit_kernel / finish_kernel (misc_kernels.cuh) serve both.
//
// Arithmetic: every entry is produced by one lane with the operations, operands and order of
// the compiled LinDx kernels (op-by-op association, kChainFma off; LUpp / Chol of smallmat.cuh;
// pnqp_thread), so both families agree to the last bit on the shapes they share.  The
// factorisations and pnqp, which are sequential, run on lane 0; the triangular solves for the
// gain columns run one column per lane.
//
// pnqp's batch-global decisions replay the guessed trace exactly like the one-thread path: each
// problem reads the guess word of its timestep, ORs what it observed into the vote word, and
// commit_kernel verifies and corrects the guess.  There is no group sweep for this family.
//
// Network dynamics (DILQR_DYN_NN_RT) are a compile-time variant of the same kernels (NN = true):
// the sweep forms F_t as the network's Jacobian at the current trajectory instead of reading it,
// and the rollouts evaluate the network instead of F_t th + f_t.  Every value is formed with the
// operations and order of Dyn<S, DYN_NN> (dynamics.cuh), and the Riccati update uses the chained
// association of the compiled env kernels (kChainFma), so the two NN families agree to
// round-off.  The warp computes hidden units 32 at a time (one per lane) into its slice of shared
// memory; the outputs / Jacobian entries then accumulate over the hidden units in ascending order.
#pragma once
#include "ilqr_kernels.cuh"

namespace dilqr {

constexpr int kRtMaxN = 32;   // one lane per row

__host__ __device__ inline bool rt_shape_ok(int ns, int nc) {
  return ns >= 1 && nc >= 1 && ns + nc <= kRtMaxN;
}

// Network scratch of the NN variant, after the RtSmem slice of the warp: one chunk of hidden
// units, the central-difference input / outputs, and for two hidden layers the first layer's
// activations z1[H1] and the n_state x H1 product G = W3 diag(d2) W2 of jacobian2.
template <class S>
struct RtNetSmem {
  S *hz, *tp, *fp, *fm, *z1, *G;

  __host__ __device__ size_t carve(char* base, int ns, int nc, int ai0) {
    const int n = ns + nc, H1 = ai0 & 0xffff;
    const bool two = (ai0 >> 16) != 0;
    size_t off = 0;
    auto take = [&](int cnt) {
      S* ptr = base ? reinterpret_cast<S*>(base + off) : nullptr;
      off += (size_t)cnt * sizeof(S);
      return ptr;
    };
    hz = take(kWarp);
    tp = take(n);
    fp = take(ns);
    fm = take(ns);
    z1 = take(two ? H1 : 0);
    G = take(two ? ns * H1 : 0);
    return (off + 15) & ~(size_t)15;
  }
  __host__ __device__ static size_t bytes(int ns, int nc, int ai0) {
    RtNetSmem w;
    return w.carve(nullptr, ns, nc, ai0);
  }
};

// This warp's slice of shared memory.
template <class S>
struct RtSmem {
  S *V, *v, *Q, *q, *F, *M, *tau, *th, *xh, *row, *K, *k, *KQ, *R, *H, *LU, *lo, *hi, *g, *dx, *mx,
      *sc;
  int *piv, *flag;

  // Point the arrays into `base` (nullptr: only count); returns the bytes of one warp's slice.
  __host__ __device__ size_t carve(char* base, int ns, int nc) {
    const int n = ns + nc;
    size_t off = 0;
    auto take = [&](int cnt) {
      S* ptr = base ? reinterpret_cast<S*>(base + off) : nullptr;
      off += (size_t)cnt * sizeof(S);
      return ptr;
    };
    V = take(ns * ns);
    v = take(ns);
    Q = take(n * n);
    q = take(n);
    F = take(ns * n);
    M = take(n * ns);
    tau = take(n);
    th = take(n);
    xh = take(ns);
    row = take(n);
    K = take(nc * ns);
    k = take(nc);
    KQ = take(ns * nc);
    R = take((ns + 1) * nc);   // one right-hand side per gain column (lane)
    H = take(nc * nc);
    LU = take(nc * nc);
    lo = take(nc);
    hi = take(nc);
    g = take(nc);
    dx = take(nc);
    mx = take(nc);
    sc = take(2);
    piv = base ? reinterpret_cast<int*>(base + off) : nullptr;
    off += (size_t)nc * sizeof(int);
    flag = base ? reinterpret_cast<int*>(base + off) : nullptr;
    off += (size_t)nc * sizeof(int);
    return (off + 15) & ~(size_t)15;
  }
  __host__ __device__ static size_t bytes(int ns, int nc) {
    RtSmem m;
    return m.carve(nullptr, ns, nc);
  }
};

// One warp's slice of shared memory for the NN variant (ai0 = DynParams::ai[0]).
template <class S>
__host__ __device__ inline size_t rt_nn_slice_bytes(int ns, int nc, int ai0) {
  return RtSmem<S>::bytes(ns, nc) + RtNetSmem<S>::bytes(ns, nc, ai0);
}

// ---------------------------------------------------------------------------
// One-thread factorisations over row-major shared-memory matrices: LUpp / Chol of smallmat.cuh
// with runtime n, the same operations in the same order.
// ---------------------------------------------------------------------------
template <class S>
DILQR_DEVICE void rt_lu_factor(S* a, int* piv, int n) {
  for (int k = 0; k < n; ++k) {
    int p = k;
    S best = absS<S>(a[k * n + k]);
    for (int i = k + 1; i < n; ++i) {
      const S v = absS<S>(a[i * n + k]);
      if (v > best) {
        best = v;
        p = i;
      }
    }
    piv[k] = p;
    if (p != k) {
      for (int j = 0; j < n; ++j) {
        const S tmp = a[k * n + j];
        a[k * n + j] = a[p * n + j];
        a[p * n + j] = tmp;
      }
    }
    const S d = a[k * n + k];
    for (int i = k + 1; i < n; ++i) {
      const S m = a[i * n + k] / d;
      a[i * n + k] = m;
      for (int j = k + 1; j < n; ++j) a[i * n + j] = fmaS<S>(-m, a[k * n + j], a[i * n + j]);
    }
  }
}

template <class S>
DILQR_DEVICE void rt_lu_solve(const S* a, const int* piv, int n, S* b) {
  for (int k = 0; k < n; ++k) {
    const int p = piv[k];
    if (p != k) {
      const S tmp = b[k];
      b[k] = b[p];
      b[p] = tmp;
    }
  }
  for (int i = 1; i < n; ++i) {
    S acc = b[i];
    for (int j = 0; j < i; ++j) acc = fmaS<S>(-a[i * n + j], b[j], acc);
    b[i] = acc;
  }
  for (int i = n - 1; i >= 0; --i) {
    S acc = b[i];
    for (int j = i + 1; j < n; ++j) acc = fmaS<S>(-a[i * n + j], b[j], acc);
    b[i] = acc / a[i * n + i];
  }
}

template <class S>
DILQR_DEVICE void rt_chol_factor(S* l, int n) {
  for (int j = 0; j < n; ++j) {
    S d = l[j * n + j];
    for (int k = 0; k < j; ++k) d = fmaS<S>(-l[j * n + k], l[j * n + k], d);
    d = sqrtS<S>(d);
    l[j * n + j] = d;
    for (int i = j + 1; i < n; ++i) {
      S s = l[i * n + j];
      for (int k = 0; k < j; ++k) s = fmaS<S>(-l[i * n + k], l[j * n + k], s);
      l[i * n + j] = s / d;
    }
  }
}

template <class S>
DILQR_DEVICE void rt_chol_solve(const S* l, int n, S* b) {
  for (int i = 0; i < n; ++i) {
    S acc = b[i];
    for (int j = 0; j < i; ++j) acc = fmaS<S>(-l[i * n + j], b[j], acc);
    b[i] = acc / l[i * n + i];
  }
  for (int i = n - 1; i >= 0; --i) {
    S acc = b[i];
    for (int j = i + 1; j < n; ++j) acc = fmaS<S>(-l[j * n + i], b[j], acc);
    b[i] = acc / l[i * n + i];
  }
}

// ---------------------------------------------------------------------------
// pnqp (pnqp.py:5-82) for one problem on one thread: pnqp_thread with runtime N, operands in
// shared memory, the trace replayed from `guess` (this timestep's 20 words) and voted into
// `votes`.  On return x is the solution, If the free set, lu/piv the factors of the masked
// Hessian of the last evaluated iteration (N > 1) and *rinv 1 / that Hessian (N == 1).
// ---------------------------------------------------------------------------
template <class S>
DILQR_DEVICE void rt_pnqp(int N, const S* H, const S* q, const S* lo, const S* hi, bool have_init,
                          S* x, int* If, S* lu, int* piv, S* g, S* dx, S* mx,
                          const uint32_t* __restrict__ guess, uint32_t* __restrict__ votes,
                          bool solo, S* rinv) {
  S h_last = S(0), r_last = S(0);
  bool have_r = false;
  const S GAMMA = S(0.1);
  if (!have_init) {  // pnqp.py:14-19
    if (N == 1) {
      x[0] = -(S(1) / H[0]) * q[0];
    } else {
      for (int i = 0; i < N; ++i) {
        for (int j = 0; j < N; ++j) lu[i * N + j] = H[i * N + j];
        x[i] = q[i];
      }
      rt_lu_factor<S>(lu, piv, N);
      rt_lu_solve<S>(lu, piv, N, x);
      for (int i = 0; i < N; ++i) x[i] = -x[i];
    }
  }
  for (int i = 0; i < N; ++i) x[i] = eclamp<S>(x[i], lo[i], hi[i]);  // pnqp.py:23

  for (int it = 0; it < kPnqpMaxIter; ++it) {
    for (int i = 0; i < N; ++i) {  // g = H x + q   (pnqp.py:29)
      S acc = S(0);
      for (int j = 0; j < N; ++j) acc = fmaS<S>(H[i * N + j], x[j], acc);
      g[i] = acc + q[i];
    }
    for (int i = 0; i < N; ++i) {  // pnqp.py:32-33
      const bool Ic = ((x[i] == lo[i]) && (g[i] > S(0))) || ((x[i] == hi[i]) && (g[i] < S(0)));
      If[i] = !Ic;
    }
    for (int i = 0; i < N; ++i) {  // pnqp.py:44-48
      for (int j = 0; j < N; ++j) {
        S h = (If[i] && If[j]) ? H[i * N + j] : S(0);
        if (i == j) h = h + S(1e-11);
        lu[i * N + j] = h;
      }
      dx[i] = If[i] ? g[i] : S(0);
    }
    if (N == 1) {  // pnqp.py:50-51
      if (!(have_r && lu[0] == h_last)) {
        h_last = lu[0];
        r_last = S(1) / h_last;
        have_r = true;
      }
      *rinv = r_last;
      dx[0] = -r_last * dx[0];
    } else {
      rt_lu_factor<S>(lu, piv, N);
      rt_lu_solve<S>(lu, piv, N, dx);
      for (int i = 0; i < N; ++i) dx[i] = -dx[i];
    }
    S nrm2 = S(0);
    for (int i = 0; i < N; ++i) nrm2 = fmaS<S>(dx[i], dx[i], nrm2);
    const bool J = (N == 1) ? (absS<S>(dx[0]) >= S(1e-4)) : (sqrtS<S>(nrm2) >= S(1e-4));
    uint32_t vote = 0;
    bool any_moving;
    if (solo) {
      any_moving = J;
    } else {
      if (J) vote |= 1u;
      any_moving = (__ldg(&guess[it]) & 1u) != 0;
    }
    if (!any_moving) {  // pnqp.py:57-59
      if (!solo && vote) vote_or(&votes[it], vote);
      return;
    }
    // Armijo backtracking with a batch-global exit test (pnqp.py:61-76)
    S fx;
    {
      S quad = S(0), dot = S(0);
      for (int j = 0; j < N; ++j) {
        S row = S(0);
        for (int i = 0; i < N; ++i) row = fmaS<S>(x[i], H[i * N + j], row);
        quad = fmaS<S>(row, x[j], quad);
      }
      for (int i = 0; i < N; ++i) dot = fmaS<S>(q[i], x[i], dot);
      fx = S(0.5) * quad + dot;
    }
    S alpha = S(1);
    const uint32_t gword = solo ? 0u : __ldg(&guess[it]);
    for (int cnt = 0; cnt < kArmijoMax; ++cnt) {
      for (int i = 0; i < N; ++i) mx[i] = eclamp<S>(x[i] + alpha * dx[i], lo[i], hi[i]);
      S arm = GAMMA + S(1e-6);
      if (J) {
        S quad = S(0), dot = S(0), gd = S(0);
        for (int j = 0; j < N; ++j) {
          S row = S(0);
          for (int i = 0; i < N; ++i) row = fmaS<S>(mx[i], H[i * N + j], row);
          quad = fmaS<S>(row, mx[j], quad);
        }
        for (int i = 0; i < N; ++i) dot = fmaS<S>(q[i], mx[i], dot);
        for (int i = 0; i < N; ++i) gd = fmaS<S>(g[i], x[i] - mx[i], gd);
        arm = (fx - (S(0.5) * quad + dot)) / gd;
      }
      const bool small = arm <= GAMMA;   // pnqp.py:73
      if (small) alpha = alpha * S(0.1);
      bool exit_loop;
      if (solo) {
        exit_loop = !small;
      } else {
        if (!small) vote |= (2u << cnt);
        exit_loop = (gword >> (1 + cnt)) & 1u;
      }
      if (exit_loop) break;
    }
    for (int i = 0; i < N; ++i) x[i] = mx[i];  // pnqp.py:78
    if (!solo && vote) vote_or(&votes[it], vote);
  }
}

// ---------------------------------------------------------------------------
// Warp helpers shared by begin and the line-search rollout (same code => the cost of an
// unchanged trajectory is bitwise the cost begin recorded, lqr_step.py:176-179).
// ---------------------------------------------------------------------------
// stage cost 0.5 th' C th + c' th (util.py:145-147), the operation order of stage_cost: lane j
// forms column sum j (coalesced over the lanes), lane 0 folds them.  Returns on lane 0 only.
template <class S>
DILQR_DEVICE S rt_stage_cost(const RtSmem<S>& m, const S* __restrict__ Cg, const S* __restrict__ cg,
                             int n, int lane) {
  if (lane < n) {
    S r = S(0);
    for (int i = 0; i < n; ++i) r = fmaS<S>(m.th[i], __ldg(Cg + i * n + lane), r);
    m.row[lane] = r;
  }
  __syncwarp();
  S out = S(0);
  if (lane == 0) {
    S quad = S(0);
    for (int j = 0; j < n; ++j) quad = fmaS<S>(m.row[j], m.th[j], quad);
    S dot = S(0);
    for (int i = 0; i < n; ++i) dot = fmaS<S>(m.th[i], __ldg(cg + i), dot);
    out = S(0.5) * quad + dot;
  }
  __syncwarp();
  return out;
}

// x_{t+1} = F_t th (+ f_t) into m.xh (util.py:117-121, lin_step); F_t read from the API tensor.
template <class S>
DILQR_DEVICE void rt_lin_step(const IterParams<S>& p, const RtSmem<S>& m, int t, int b, int ns,
                              int nc, int lane) {
  const int n = ns + nc;
  const S* Fg = p.F + ((size_t)t * p.B + b) * (ns * n);
  for (int e = lane; e < ns * n; e += kWarp) m.F[e] = __ldg(Fg + e);
  __syncwarp();
  if (lane < ns) {
    S acc = S(0);
    for (int j = 0; j < n; ++j) acc = fmaS<S>(m.F[lane * n + j], m.th[j], acc);
    if (p.has_f) acc = acc + __ldg(p.f + ((size_t)t * p.B + b) * ns + lane);
    m.xh[lane] = acc;
  }
  __syncwarp();
}

// out[0..ns) = the network at in[0..n) (Dyn<S, DYN_NN>::step / step2).  The last hidden layer
// is computed 32 units at a time, one per lane, into w.hz; lane i < ns then accumulates output i
// over those units in ascending order.  Two hidden layers: the first goes to w.z1 beforehand.
template <class S>
DILQR_DEVICE void rt_nn_step(const DynParams<S>& P, const RtNetSmem<S>& w, const S* in, S* out,
                             int ns, int nc, int lane) {
  using D = Dyn<S, DYN_NN>;
  const int n = ns + nc, H1 = P.ai[0] & 0xffff, H2 = P.ai[0] >> 16, act = P.ai[1];
  const bool two = H2 != 0;
  const S* W1 = P.aux;
  const S* b1 = W1 + (size_t)H1 * n;
  const int HL = two ? H2 : H1;         // last hidden layer: HL units over KL inputs
  const int KL = two ? H1 : n;
  const S* WL = two ? b1 + H1 : W1;
  const S* bL = WL + (size_t)HL * KL;
  const S* Wo = bL + HL;                // output layer [ns][HL], bias [ns]
  const S* bo = Wo + (size_t)ns * HL;
  const S* src = two ? w.z1 : in;
  if (two) {
    for (int h = lane; h < H1; h += kWarp) {
      S a = S(0);
      for (int j = 0; j < n; ++j) a = fmaS<S>(__ldg(W1 + (size_t)h * n + j), in[j], a);
      w.z1[h] = D::act(a + __ldg(b1 + h), act);
    }
    __syncwarp();
  }
  S acc = S(0);
  for (int h0 = 0; h0 < HL; h0 += kWarp) {
    const int h = h0 + lane;
    if (h < HL) {
      S a = S(0);
      for (int j = 0; j < KL; ++j) a = fmaS<S>(__ldg(WL + (size_t)h * KL + j), src[j], a);
      w.hz[lane] = D::act(a + __ldg(bL + h), act);
    }
    __syncwarp();
    if (lane < ns) {
      const int cnt = min(kWarp, HL - h0);
      for (int q = 0; q < cnt; ++q)
        acc = fmaS<S>(__ldg(Wo + (size_t)lane * HL + h0 + q), w.hz[q], acc);
    }
    __syncwarp();
  }
  if (lane < ns) {
    S v = acc + __ldg(bo + lane);
    if (P.ai[2]) v = v + in[lane];
    out[lane] = v;
  }
  __syncwarp();
}

// F[ns][n] = d net / d tau at tau (Dyn<S, DYN_NN>::jacobian / jacobian2 / jacobian_fd).  Lane j
// < n owns column j; every entry accumulates over the hidden units in ascending order with the
// rounded products W1[h][j] * d_h of the compiled family.
template <class S>
DILQR_DEVICE void rt_nn_jacobian(const DynParams<S>& P, const RtNetSmem<S>& w, const S* tau, S* F,
                                 int ns, int nc, int lane) {
  using D = Dyn<S, DYN_NN>;
  const int n = ns + nc;
  if (P.ai[3] == 1) {   // central differences, eps = 1e-4: 2n network evaluations
    const S eps = S(1e-4), two_eps = S(2. * 1e-4);
    if (lane < n) w.tp[lane] = tau[lane];
    __syncwarp();
    for (int j = 0; j < n; ++j) {
      if (lane == 0) w.tp[j] = tau[j] + eps;
      __syncwarp();
      rt_nn_step<S>(P, w, w.tp, w.fp, ns, nc, lane);
      if (lane == 0) w.tp[j] = tau[j] - eps;
      __syncwarp();
      rt_nn_step<S>(P, w, w.tp, w.fm, ns, nc, lane);
      if (lane == 0) w.tp[j] = tau[j];
      if (lane < ns) F[lane * n + j] = (w.fp[lane] - w.fm[lane]) / two_eps;
      __syncwarp();
    }
    return;
  }
  const int H1 = P.ai[0] & 0xffff, H2 = P.ai[0] >> 16, act = P.ai[1];
  const S* W1 = P.aux;
  const S* b1 = W1 + (size_t)H1 * n;
  auto dact = [act](S z) { return act == 1 ? (z <= S(0) ? S(0) : S(1)) : z * (S(1) - z); };
  for (int e = lane; e < ns * n; e += kWarp) F[e] = S(0);
  if (H2 == 0) {
    const S* W2 = b1 + H1;
    for (int h0 = 0; h0 < H1; h0 += kWarp) {
      const int h = h0 + lane;
      if (h < H1) {
        S a = S(0);
        for (int j = 0; j < n; ++j) a = fmaS<S>(__ldg(W1 + (size_t)h * n + j), tau[j], a);
        w.hz[lane] = dact(D::act(a + __ldg(b1 + h), act));
      }
      __syncwarp();
      if (lane < n) {
        const int j = lane, cnt = min(kWarp, H1 - h0);
        for (int q = 0; q < cnt; ++q) {
          const S wj = __ldg(W1 + (size_t)(h0 + q) * n + j) * w.hz[q];
          for (int i = 0; i < ns; ++i)
            F[i * n + j] = fmaS<S>(__ldg(W2 + (size_t)i * H1 + h0 + q), wj, F[i * n + j]);
        }
      }
      __syncwarp();
    }
  } else {   // G = W3 (diag(d2) W2), then F = G (diag(d1) W1)
    const S* W2 = b1 + H1;
    const S* b2 = W2 + (size_t)H2 * H1;
    const S* W3 = b2 + H2;
    for (int h = lane; h < H1; h += kWarp) {
      S a = S(0);
      for (int j = 0; j < n; ++j) a = fmaS<S>(__ldg(W1 + (size_t)h * n + j), tau[j], a);
      w.z1[h] = D::act(a + __ldg(b1 + h), act);
      for (int i = 0; i < ns; ++i) w.G[i * H1 + h] = S(0);
    }
    __syncwarp();
    for (int k0 = 0; k0 < H2; k0 += kWarp) {
      const int k = k0 + lane;
      if (k < H2) {
        S a = S(0);
        for (int h = 0; h < H1; ++h) a = fmaS<S>(__ldg(W2 + (size_t)k * H1 + h), w.z1[h], a);
        w.hz[lane] = dact(D::act(a + __ldg(b2 + k), act));
      }
      __syncwarp();
      const int cnt = min(kWarp, H2 - k0);
      for (int h = lane; h < H1; h += kWarp)   // column h of G on one lane
        for (int q = 0; q < cnt; ++q) {
          const S wv = __ldg(W2 + (size_t)(k0 + q) * H1 + h) * w.hz[q];
          for (int i = 0; i < ns; ++i)
            w.G[i * H1 + h] = fmaS<S>(__ldg(W3 + (size_t)i * H2 + k0 + q), wv, w.G[i * H1 + h]);
        }
      __syncwarp();
    }
    if (lane < n) {
      const int j = lane;
      for (int h = 0; h < H1; ++h) {
        const S wj = __ldg(W1 + (size_t)h * n + j) * dact(w.z1[h]);
        for (int i = 0; i < ns; ++i) F[i * n + j] = fmaS<S>(w.G[i * H1 + h], wj, F[i * n + j]);
      }
    }
  }
  if (P.ai[2] && lane < ns) F[lane * n + lane] = F[lane * n + lane] + S(1);
  __syncwarp();
}

template <class S>
DILQR_DEVICE void rt_bounds(const IterParams<S>& p, int t, int b, int nc, int a, S* lo, S* hi) {
  if (p.bounds_kind == 2) {
    *lo = __ldg(p.lo_t + ((size_t)t * p.B + b) * nc + a);
    *hi = __ldg(p.hi_t + ((size_t)t * p.B + b) * nc + a);
  } else {
    *lo = p.lo;
    *hi = p.hi;
  }
}

// ---------------------------------------------------------------------------
// Phase A: c_back + Riccati backward sweep with gains and pnqp (lqr_step.py:52-160,289-295),
// the order of operations of IterKernel::backward_sweep for LinDx (NN: for DYN_NN, whose
// Riccati update uses the chained association kChainFma).
// ---------------------------------------------------------------------------
template <class S, bool NN>
DILQR_DEVICE void rt_backward_sweep(const IterParams<S>& p, const RtSmem<S>& m,
                                    const RtNetSmem<S>& w, int ns, int nc, int b, int lane) {
  constexpr bool kChain = NN && kChainFmaOn;
  const int n = ns + nc, NK = nc * ns + nc, T = p.T;
  // lazy best-iterate tracking (mpc.py:272-285), see IterParams::take
  const bool flush = (p.take[b] & 1) != 0;
  bool have_prev = false;
  for (int t = T - 1; t >= 0; --t) {
    const S* Cg = cost_src<S>(p.C, p.C_bcast, t, p.B, b, n * n);
    const S* cg = cost_src<S>(p.c, p.c_bcast, t, p.B, b, n);
    for (int e = lane; e < n * n; e += kWarp) m.Q[e] = __ldg(Cg + e);
    if (!NN && t < T - 1) {
      const S* Fg = p.F + ((size_t)t * p.B + b) * (ns * n);
      for (int e = lane; e < ns * n; e += kWarp) m.F[e] = __ldg(Fg + e);
    }
    if (lane < n) {
      const S tv = p.traj_cur[bidx(t, lane, n, b, p.nW)];
      m.tau[lane] = tv;
      if (flush) p.traj_best[bidx(t, lane, n, b, p.nW)] = tv;
    }
    __syncwarp();
    if constexpr (NN) {   // F_t = the network's Jacobian at tau_t (mpc_explicit.py:516-546)
      if (t < T - 1) rt_nn_jacobian<S>(p.dyn, w, m.tau, m.F, ns, nc, lane);
    }
    if (lane < n) {
      const int i = lane;
      S acc = kChain ? __ldg(cg + i) : S(0);  // c_back = C tau + c   (lqr_step.py:294)
      for (int j = 0; j < n; ++j) acc = fmaS<S>(m.Q[i * n + j], m.tau[j], acc);
      m.q[i] = kChain ? acc : acc + __ldg(cg + i);
      if (t < T - 1) {  // Q = C + (F' V) F ; q = c~ + F' v     (lqr_step.py:66-70)
        for (int k = 0; k < ns; ++k) {
          S a2 = S(0);
          for (int l = 0; l < ns; ++l) a2 = fmaS<S>(m.F[l * n + i], m.V[l * ns + k], a2);
          m.M[i * ns + k] = a2;
        }
        for (int j = 0; j < n; ++j) {
          S a2 = kChain ? m.Q[i * n + j] : S(0);
          for (int k = 0; k < ns; ++k) a2 = fmaS<S>(m.M[i * ns + k], m.F[k * n + j], a2);
          m.Q[i * n + j] = kChain ? a2 : m.Q[i * n + j] + a2;
        }
        S a3 = kChain ? m.q[i] : S(0);
        for (int l = 0; l < ns; ++l) a3 = fmaS<S>(m.F[l * n + i], m.v[l], a3);
        m.q[i] = kChain ? a3 : m.q[i] + a3;
      }
    }
    __syncwarp();

    // ------------------------------------------------------------ gains
    const S* Qu = m.Q + ns * n;   // rows n_state.. of Q
    if (p.bounds_kind == 0) {
      if (lane < nc) m.flag[lane] = p.zeroI ? (p.zeroI[((size_t)t * p.B + b) * nc + lane] != 0) : 0;
      __syncwarp();
      if (nc == 1) {
        if (!p.zeroI) {  // lqr_step.py:84-86
          const S r = S(1) / Qu[ns];
          if (lane < ns) m.K[lane] = -(r * Qu[lane]);
          if (lane == 0) m.k[0] = -(r * m.q[ns]);
        } else {         // lqr_step.py:101-123
          const bool mk = m.flag[0] != 0;
          const S quu_m = mk ? S(1e-8) : Qu[ns];
          const S r = S(1) / quu_m;
          if (lane < ns) m.K[lane] = -(r * (mk ? S(0) : Qu[lane]));
          if (lane == 0) m.k[0] = -((S(1) / Qu[ns]) * (mk ? S(0) : m.q[ns]));
        }
      } else {
        const bool chol = !p.zeroI && p.gain_solve == 1;   // lqr_step_backup.py:202-205
        if (lane == 0) {
          for (int a = 0; a < nc; ++a)
            for (int c2 = 0; c2 < nc; ++c2) {
              S h;
              if (chol) {
                h = Qu[a * n + ns + c2] + (a == c2 ? S(1e-6) : S(0));
              } else {   // plain / u_zero_I-masked LU solve (lqr_step.py:88-94,101-127)
                h = (m.flag[a] || m.flag[c2]) ? S(0) : Qu[a * n + ns + c2];
                if (a == c2 && m.flag[a]) h = h + S(1e-8);
              }
              m.LU[a * nc + c2] = h;
            }
          if (chol) rt_chol_factor<S>(m.LU, nc);
          else rt_lu_factor<S>(m.LU, m.piv, nc);
        }
        __syncwarp();
        if (lane <= ns) {   // column `lane` of [K | k]
          const int j = lane;
          S* rhs = m.R + j * nc;
          for (int a = 0; a < nc; ++a) {
            const S val = (j < ns) ? Qu[a * n + j] : m.q[ns + a];
            rhs[a] = (!chol && m.flag[a]) ? S(0) : val;
          }
          if (chol) rt_chol_solve<S>(m.LU, nc, rhs);
          else rt_lu_solve<S>(m.LU, m.piv, nc, rhs);
          for (int a = 0; a < nc; ++a) {
            if (j < ns) m.K[a * ns + j] = -rhs[a];
            else m.k[a] = -rhs[a];
          }
        }
      }
    } else {  // box constraints: pnqp   (lqr_step.py:128-148)
      if (lane == 0) {
        for (int a = 0; a < nc; ++a) {
          S lo, hi;
          rt_bounds<S>(p, t, b, nc, a, &lo, &hi);
          lo = lo - m.tau[ns + a];
          hi = hi - m.tau[ns + a];
          if (p.has_delta) {   // lqr_step.py:132-134
            if (lo < -p.delta_u) lo = -p.delta_u;
            if (hi > p.delta_u) hi = p.delta_u;
          }
          m.lo[a] = lo;
          m.hi[a] = hi;
          for (int c2 = 0; c2 < nc; ++c2) m.H[a * nc + c2] = Qu[a * n + ns + c2];
          if (!have_prev) m.k[a] = S(0);   // else: warm start from the later timestep
        }
        rt_pnqp<S>(nc, m.H, m.q + ns, m.lo, m.hi, have_prev, m.k, m.flag, m.LU, m.piv, m.g, m.dx,
                   m.mx, p.guess + (size_t)t * kPnqpMaxIter, p.votes + (size_t)t * kPnqpMaxIter,
                   p.solo != 0, m.sc);
      }
      have_prev = true;
      __syncwarp();
      if (nc == 1) {  // lqr_step.py:144-146
        const S r = m.sc[0];
        if (lane < ns) m.K[lane] = -(r * (m.flag[0] ? Qu[lane] : S(0)));
      } else if (lane < ns) {  // lqr_step.py:148
        const int j = lane;
        S* rhs = m.R + j * nc;
        for (int a = 0; a < nc; ++a) rhs[a] = m.flag[a] ? Qu[a * n + j] : S(0);
        rt_lu_solve<S>(m.LU, m.piv, nc, rhs);
        for (int a = 0; a < nc; ++a) m.K[a * ns + j] = -rhs[a];
      }
    }
    __syncwarp();
    for (int e = lane; e < NK; e += kWarp)
      p.Kk[bidx(t, e, NK, b, p.nW)] = e < nc * ns ? m.K[e] : m.k[e - nc * ns];

    // -------------------------------------------- value function update
    // V = Qxx + Qxu K + K' Qux + (K' Quu) K      (lqr_step.py:155)
    // v = qx + Qxu k + K' qu + (K' Quu) k        (lqr_step.py:156-158)
    if (lane < ns) {
      const int i = lane;
      for (int a = 0; a < nc; ++a) {
        S acc = S(0);
        for (int c2 = 0; c2 < nc; ++c2) acc = fmaS<S>(m.K[c2 * ns + i], Qu[c2 * n + ns + a], acc);
        m.KQ[i * nc + a] = acc;
      }
      if constexpr (kChain) {
        for (int j = 0; j < ns; ++j) {
          S acc = m.Q[i * n + j];
          for (int a = 0; a < nc; ++a) acc = fmaS<S>(m.Q[i * n + ns + a], m.K[a * ns + j], acc);
          for (int a = 0; a < nc; ++a) acc = fmaS<S>(m.K[a * ns + i], Qu[a * n + j], acc);
          for (int a = 0; a < nc; ++a) acc = fmaS<S>(m.KQ[i * nc + a], m.K[a * ns + j], acc);
          m.V[i * ns + j] = acc;
        }
        S acc = m.q[i];
        for (int a = 0; a < nc; ++a) acc = fmaS<S>(m.Q[i * n + ns + a], m.k[a], acc);
        for (int a = 0; a < nc; ++a) acc = fmaS<S>(m.K[a * ns + i], m.q[ns + a], acc);
        for (int a = 0; a < nc; ++a) acc = fmaS<S>(m.KQ[i * nc + a], m.k[a], acc);
        m.v[i] = acc;
      } else {
        for (int j = 0; j < ns; ++j) {
          S t1 = S(0), t2 = S(0), t3 = S(0);
          for (int a = 0; a < nc; ++a) {
            t1 = fmaS<S>(m.Q[i * n + ns + a], m.K[a * ns + j], t1);
            t2 = fmaS<S>(m.K[a * ns + i], Qu[a * n + j], t2);
            t3 = fmaS<S>(m.KQ[i * nc + a], m.K[a * ns + j], t3);
          }
          m.V[i * ns + j] = ((m.Q[i * n + j] + t1) + t2) + t3;
        }
        S t1 = S(0), t2 = S(0), t3 = S(0);
        for (int a = 0; a < nc; ++a) {
          t1 = fmaS<S>(m.Q[i * n + ns + a], m.k[a], t1);
          t2 = fmaS<S>(m.K[a * ns + i], m.q[ns + a], t2);
          t3 = fmaS<S>(m.KQ[i * nc + a], m.k[a], t3);
        }
        m.v[i] = ((m.q[i] + t1) + t2) + t3;
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Phase B: rollout with the affine control law + line search (lqr_step.py:164-261), the
// bookkeeping of IterKernel::forward_linesearch for one problem.
// ---------------------------------------------------------------------------
template <class S, bool NN>
DILQR_DEVICE void rt_forward_linesearch(const IterParams<S>& p, const RtSmem<S>& m,
                                        const RtNetSmem<S>& w, int ns, int nc, int b, int lane) {
  const int n = ns + nc, NK = nc * ns + nc, T = p.T;
  const S old_cost = p.cost_cur[b];
  S alpha = S(1);
  bool accepted = false;
  S res_cost = S(0), res_alpha = S(1);
  for (int tr = 0; tr < p.max_ls && !accepted; ++tr) {
    if (lane < ns) m.xh[lane] = __ldg(p.x_init + (size_t)b * ns + lane);
    S cost = S(0);
    __syncwarp();
    for (int t = 0; t < T; ++t) {
      if (lane < n) m.tau[lane] = p.traj_cur[bidx(t, lane, n, b, p.nW)];
      if (lane < ns) m.th[lane] = m.xh[lane];
      __syncwarp();
      if (lane < nc) {  // lqr_step.py:192
        const int a = lane;
        S acc = S(0);
        if (t > 0) {
          for (int j = 0; j < ns; ++j)
            acc = fmaS<S>(p.Kk[bidx(t, a * ns + j, NK, b, p.nW)], m.xh[j] - m.tau[j], acc);
        }
        S un = (acc + m.tau[ns + a]) + alpha * p.Kk[bidx(t, nc * ns + a, NK, b, p.nW)];
        if (p.zeroI && p.zeroI[((size_t)t * p.B + b) * nc + a]) un = S(0);  // :197-198
        if (p.bounds_kind) {
          S lb, ub;
          rt_bounds<S>(p, t, b, nc, a, &lb, &ub);
          if (p.has_delta) {   // lqr_step.py:204-211
            const S l2 = m.tau[ns + a] - p.delta_u, u2 = m.tau[ns + a] + p.delta_u;
            lb = l2 < lb ? lb : l2;
            ub = u2 > ub ? ub : u2;
          }
          un = eclamp<S>(un, lb, ub);                                         // :213
        }
        m.th[ns + a] = un;
        if (tr == 0) {   // full_du_norm squares in [T,nc,B] order (see forward_linesearch)
          const S d = m.tau[ns + a] - un;
          p.dusq[((size_t)t * nc + a) * p.B + b] = d * d;
        }
      }
      __syncwarp();
      if (lane < n) p.traj_new[bidx(t, lane, n, b, p.nW)] = m.th[lane];
      cost = cost + rt_stage_cost<S>(m, cost_src<S>(p.C, p.C_bcast, t, p.B, b, n * n),
                                     cost_src<S>(p.c, p.c_bcast, t, p.B, b, n), n, lane);
      if (t < T - 1) {
        if constexpr (NN) rt_nn_step<S>(p.dyn, w, m.th, m.xh, ns, nc, lane);
        else rt_lin_step<S>(p, m, t, b, ns, nc, lane);
      }
    }
    if (lane == 0) {
      res_cost = cost;
      res_alpha = alpha;
      accepted = !(cost > old_cost);      // lqr_step.py:176-179,247
      if (!accepted) alpha = alpha * p.decay;
    }
    accepted = __shfl_sync(kFull, accepted, 0);
    alpha = __shfl_sync(kFull, alpha, 0);
  }
  if (lane == 0) {
    p.cost_new[b] = res_cost;
    p.alpha_new[b] = res_alpha;
  }
}

// One warp per problem; the warp's slice of dynamic shared memory is RtSmem<S>::bytes(ns, nc),
// followed for the NN variant by its RtNetSmem (rt_nn_slice_bytes).
template <class S, bool NN>
DILQR_DEVICE bool rt_warp_setup(const IterParams<S>& p, int ns, int nc, char* smem, RtSmem<S>& m,
                                RtNetSmem<S>& w, int& b, int& lane) {
  lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  b = blockIdx.x * (blockDim.x >> 5) + warp;
  if (b >= p.B) return false;
  if constexpr (NN) {
    char* base = smem + warp * rt_nn_slice_bytes<S>(ns, nc, p.dyn.ai[0]);
    m.carve(base, ns, nc);
    w.carve(base + RtSmem<S>::bytes(ns, nc), ns, nc, p.dyn.ai[0]);
  } else {
    m.carve(smem + warp * RtSmem<S>::bytes(ns, nc), ns, nc);
  }
  return true;
}

template <class S, bool NN>
DILQR_DEVICE void rt_iter(const IterParams<S>& p, int ns, int nc) {
  extern __shared__ __align__(128) char smem[];
  if (p.halt && *reinterpret_cast<const volatile uint32_t*>(p.halt)) return;  // pipelined loop stopped
  RtSmem<S> m;
  RtNetSmem<S> w;
  int b, lane;
  if (!rt_warp_setup<S, NN>(p, ns, nc, smem, m, w, b, lane)) return;
  rt_backward_sweep<S, NN>(p, m, w, ns, nc, b, lane);
  if (!p.gains_only) rt_forward_linesearch<S, NN>(p, m, w, ns, nc, b, lane);
}

// begin: nominal rollout of u_init (util.get_traj) + its cost (util.get_cost), or the given
// trajectory x_cur (standalone LQRStep), into the current-trajectory buffer.
template <class S, bool NN>
DILQR_DEVICE void rt_begin(const IterParams<S>& p, int ns, int nc) {
  extern __shared__ __align__(128) char smem[];
  RtSmem<S> m;
  RtNetSmem<S> w;
  int b, lane;
  if (!rt_warp_setup<S, NN>(p, ns, nc, smem, m, w, b, lane)) return;
  const int n = ns + nc, T = p.T;
  const bool want_cost = !(p.gains_only && p.x_cur);
  if (lane < ns) m.xh[lane] = __ldg(p.x_init + (size_t)b * ns + lane);
  __syncwarp();
  S cost = S(0);
  for (int t = 0; t < T; ++t) {
    if (lane < ns) m.th[lane] = p.x_cur ? __ldg(p.x_cur + ((size_t)t * p.B + b) * ns + lane) : m.xh[lane];
    if (lane < nc) m.th[ns + lane] = p.u_init ? __ldg(p.u_init + ((size_t)t * p.B + b) * nc + lane) : S(0);
    __syncwarp();
    if (lane < n) p.traj_new[bidx(t, lane, n, b, p.nW)] = m.th[lane];
    if (want_cost)
      cost = cost + rt_stage_cost<S>(m, cost_src<S>(p.C, p.C_bcast, t, p.B, b, n * n),
                                     cost_src<S>(p.c, p.c_bcast, t, p.B, b, n), n, lane);
    if (want_cost && t < T - 1 && !p.x_cur) {
      if constexpr (NN) rt_nn_step<S>(p.dyn, w, m.th, m.xh, ns, nc, lane);
      else rt_lin_step<S>(p, m, t, b, ns, nc, lane);
    }
    __syncwarp();
  }
  if (lane == 0) {
    p.cost_cur[b] = cost;
    p.take[b] = 0;
  }
}

// LinDx (DILQR_DYN_LINDX_RT) and network (DILQR_DYN_NN_RT) instantiations
template <class S>
__global__ void rt_iter_kernel(const __grid_constant__ IterParams<S> p, int ns, int nc) {
  rt_iter<S, false>(p, ns, nc);
}
template <class S>
__global__ void rt_nn_iter_kernel(const __grid_constant__ IterParams<S> p, int ns, int nc) {
  rt_iter<S, true>(p, ns, nc);
}
template <class S>
__global__ void rt_begin_kernel(const __grid_constant__ IterParams<S> p, int ns, int nc) {
  rt_begin<S, false>(p, ns, nc);
}
template <class S>
__global__ void rt_nn_begin_kernel(const __grid_constant__ IterParams<S> p, int ns, int nc) {
  rt_begin<S, true>(p, ns, nc);
}

// ---------------------------------------------------------------------------
// KKT gradient assembly (lqr_step.py:343-404), kkt_grads_kernel with runtime dimensions: one
// warp per problem, lane i owns costate component i.
// ---------------------------------------------------------------------------
template <class S>
__global__ void rt_kkt_kernel(const __grid_constant__ DilqrKkt k) {
  __shared__ S sh[4][4][kRtMaxN];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * (blockDim.x >> 5) + warp;
  const int T = k.T, B = k.n_batch, ns = k.n_state, nc = k.n_ctrl, n = ns + nc;
  if (b >= B) return;
  S* tau = sh[warp][0];
  S* dtau = sh[warp][1];
  S* lam = sh[warp][2];
  S* dlam = sh[warp][3];
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
  for (int t = T - 1; t >= 0; --t) {
    const size_t tb = (size_t)t * B + b;
    if (lane < ns) {
      tau[lane] = __ldg(x + tb * ns + lane);
      dtau[lane] = __ldg(dx + tb * ns + lane);
    } else if (lane < n) {
      tau[lane] = __ldg(u + tb * nc + lane - ns);
      dtau[lane] = __ldg(du + tb * nc + lane - ns);
    }
    __syncwarp();
    // gradients that pair step t with the costates of t+1 (held in lam/dlam)
    if (t < T - 1) {
      if (dF) {
        for (int e = lane; e < ns * n; e += kWarp) {
          const int i = e / n, j = e - i * n;
          dF[tb * (ns * n) + e] = -(dlam[i] * tau[j] + lam[i] * dtau[j]);
        }
      }
      if (df && lane < ns) df[tb * ns + lane] = -dlam[lane];
    }
    if (dC) {
      for (int e = lane; e < n * n; e += kWarp) {
        const int i = e / n, j = e - i * n;
        dC[tb * (n * n) + e] = S(-0.5) * (dtau[i] * tau[j] + tau[i] * dtau[j]);
      }
    }
    if (dc && lane < n) dc[tb * n + lane] = -dtau[lane];
    // lam_t = Cxx x + Cxu u + c_x + Fx' lam_{t+1}   (lqr_step.py:355-369)
    S nl = S(0), ndl = S(0);
    if (lane < ns) {
      const int i = lane;
      S a1 = S(0), a2 = S(0), d1 = S(0), d2 = S(0);
      for (int j = 0; j < ns; ++j) {
        const S cij = __ldg(C + tb * (n * n) + i * n + j);
        a1 = fmaS<S>(cij, tau[j], a1);
        d1 = fmaS<S>(cij, dtau[j], d1);
      }
      for (int a = 0; a < nc; ++a) {
        const S cij = __ldg(C + tb * (n * n) + i * n + ns + a);
        a2 = fmaS<S>(cij, tau[ns + a], a2);
        d2 = fmaS<S>(cij, dtau[ns + a], d2);
      }
      nl = (a1 + a2) + __ldg(c + tb * n + i);
      ndl = (d1 + d2) - __ldg(r + tb * n + i);
      if (t < T - 1) {
        S e1 = S(0), e2 = S(0);
        for (int l = 0; l < ns; ++l) {
          const S fli = __ldg(F + tb * (ns * n) + l * n + i);
          e1 = fmaS<S>(fli, lam[l], e1);
          e2 = fmaS<S>(fli, dlam[l], e2);
        }
        nl = nl + e1;
        ndl = ndl + e2;
      }
    }
    __syncwarp();
    if (lane < ns) {
      lam[lane] = nl;
      dlam[lane] = ndl;
    }
    __syncwarp();
  }
  if (dx0 && lane < ns) dx0[(size_t)b * ns + lane] = -dlam[lane];
}

}  // namespace dilqr
