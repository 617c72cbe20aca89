// pnqp_rt.cuh -- the standalone projected-Newton box QP (pnqp.py:5-82) with the problem size n
// and the iteration budget n_iter as runtime values (dilqr_pnqp_rt).
//
// pnqp_kernel<S, N> (misc_kernels.cuh) keeps a problem in one thread's registers, so every n has
// to be compiled in and the budget is kPnqpMaxIter.  This family serves any 1 <= n <= 256 and
// 1 <= n_iter <= 1024:
//   - ONE WARP PER PROBLEM, lane l owns the rows / columns j == l (mod 32);
//   - H is read through the read-only path; the masked Hessian and its LU factor are formed in
//     place in the caller's lu[b] (the output); the vectors (x, g, dx, mx, q, lo, hi, column
//     sums, free-set flags, pivots) sit in the warp's slice of dynamic shared memory;
//   - g = H x + q: one row per lane.  Masked Hessian and factorisation: the lane owning column j
//     updates column j at every step k; the pivot search is a warp reduction that keeps the
//     first maximum (the scan order of rt_lu_factor); the multipliers of step k are spread over
//     the lanes by row.  Quadratic forms: each lane forms its column sums sum_i x_i H[i][j], lane
//     0 folds them in ascending j.  The triangular solves and the O(n) reductions run on lane 0.
//
// Arithmetic: every value is produced with the operations and order of pnqp_thread / rt_pnqp
// (fmaS chains, the 1e-11 diagonal, eclamp, the n == 1 reciprocal reuse, the 1e-4 step test), so
// on the compiled sizes this kernel returns bitwise what pnqp_kernel<S, N> returns.
//
// Batch-global control flow: the trace is replayed exactly as pnqp_kernel does -- one guess word
// per iteration, lane 0 ORs what its problem observed into the vote word (bit 0 "moving", bit
// 1 + c "Armijo pass c exits"), and pnqp_rt_verify_kernel checks and corrects the n_iter words.
#pragma once
#include "misc_kernels.cuh"
#include "rt_kernels.cuh"

namespace dilqr {

constexpr int kPnqpRtMaxN = DILQR_PNQP_RT_MAX_N;         // at most 8 rows / columns per lane
constexpr int kPnqpRtMaxIter = DILQR_PNQP_RT_MAX_ITER;   // trace words per call: 2 * n_iter

__host__ __device__ inline bool pnqp_rt_ok(int n, int n_iter) {
  return n >= 1 && n <= kPnqpRtMaxN && n_iter >= 1 && n_iter <= kPnqpRtMaxIter;
}

// This warp's slice of shared memory.
template <class S>
struct PnqpRtSmem {
  S *x, *g, *dx, *mx, *q, *lo, *hi, *col;
  int *flag, *piv;

  // Point the arrays into `base` (nullptr: only count); returns the bytes of one warp's slice.
  __host__ __device__ size_t carve(char* base, int n) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
      char* ptr = base ? base + off : nullptr;
      off += bytes;
      return ptr;
    };
    S** vecs[] = {&x, &g, &dx, &mx, &q, &lo, &hi, &col};
    for (S** v : vecs) *v = reinterpret_cast<S*>(take((size_t)n * sizeof(S)));
    flag = reinterpret_cast<int*>(take((size_t)n * sizeof(int)));
    piv = reinterpret_cast<int*>(take((size_t)n * sizeof(int)));
    return (off + 15) & ~(size_t)15;
  }
  __host__ __device__ static size_t bytes(int n) {
    PnqpRtSmem m;
    return m.carve(nullptr, n);
  }
};

// First owned index >= j0 of `lane` (owned: j == lane mod 32).
DILQR_DEVICE int rt_first_owned(int j0, int lane) {
  return j0 + ((lane - j0) & (kWarp - 1));
}

// LU factorisation with partial pivoting of the row-major n x n matrix `a` by the whole warp:
// rt_lu_factor's operations, order and pivot choice (the first maximal |a_ik|), column j updated
// by lane j mod 32.  piv[k] is written by lane 0.
template <class S>
DILQR_DEVICE void rt_lu_factor_warp(S* a, int* piv, int n, int lane) {
  for (int k = 0; k < n; ++k) {
    S best = S(-1);
    int p = n;
    for (int i = rt_first_owned(k, lane); i < n; i += kWarp) {
      const S v = absS<S>(a[(size_t)i * n + k]);
      if (v > best) {
        best = v;
        p = i;
      }
    }
#pragma unroll
    for (int off = kWarp / 2; off > 0; off >>= 1) {
      const S ob = __shfl_xor_sync(kFull, best, off);
      const int op = __shfl_xor_sync(kFull, p, off);
      if (ob > best || (ob == best && op < p)) {
        best = ob;
        p = op;
      }
    }
    const S dkk = absS<S>(a[(size_t)k * n + k]);
    if (dkk != dkk) p = k;   // NaN diagonal: the sequential scan never moves off row k
    if (lane == 0) piv[k] = p;
    if (p != k) {
      for (int j = lane; j < n; j += kWarp) {
        const S tmp = a[(size_t)k * n + j];
        a[(size_t)k * n + j] = a[(size_t)p * n + j];
        a[(size_t)p * n + j] = tmp;
      }
    }
    __syncwarp();
    const S d = a[(size_t)k * n + k];
    for (int i = rt_first_owned(k + 1, lane); i < n; i += kWarp) a[(size_t)i * n + k] = a[(size_t)i * n + k] / d;
    __syncwarp();
    const int j0 = rt_first_owned(k + 1, lane);
    for (int i = k + 1; i < n; ++i) {
      const S m = a[(size_t)i * n + k];
      for (int j = j0; j < n; j += kWarp)
        a[(size_t)i * n + j] = fmaS<S>(-m, a[(size_t)k * n + j], a[(size_t)i * n + j]);
    }
    __syncwarp();
  }
}

// Column sums col[j] = sum_i v_i H[i][j] (ascending i, lane j mod 32), then on lane 0
// sum_j col_j v_j (ascending j): the quadratic form of pnqp_thread.  Returns on lane 0 only.
template <class S>
DILQR_DEVICE S rt_quad_warp(const S* __restrict__ H, const S* v, S* col, int n, int lane) {
  for (int j = lane; j < n; j += kWarp) {
    S row = S(0);
    for (int i = 0; i < n; ++i) row = fmaS<S>(v[i], __ldg(&H[(size_t)i * n + j]), row);
    col[j] = row;
  }
  __syncwarp();
  S quad = S(0);
  if (lane == 0)
    for (int j = 0; j < n; ++j) quad = fmaS<S>(col[j], v[j], quad);
  return quad;
}

// One warp per problem; blockDim.x = 32 * warps, dynamic shared memory = warps * the slice.
template <class S>
__global__ void __launch_bounds__(128) pnqp_rt_kernel(
    int B, int N, int n_iter, const S* __restrict__ H, const S* __restrict__ q,
    const S* __restrict__ lower, const S* __restrict__ upper, const S* __restrict__ x_init,
    S* __restrict__ x_out, S* __restrict__ lu_out, int32_t* __restrict__ piv_out,
    S* __restrict__ if_out, const uint32_t* __restrict__ guess, uint32_t* __restrict__ votes,
    int solo) {
  extern __shared__ __align__(16) char rt_smem[];
  const int lane = threadIdx.x & (kWarp - 1), warp = threadIdx.x / kWarp;
  const int b = blockIdx.x * (blockDim.x / kWarp) + warp;
  if (b >= B) return;   // uniform over the warp
  PnqpRtSmem<S> m;
  m.carve(rt_smem + warp * PnqpRtSmem<S>::bytes(N), N);
  const S* Hb = H + (size_t)b * N * N;
  S* a = lu_out + (size_t)b * N * N;
  const size_t vb = (size_t)b * N;
  const S GAMMA = S(0.1);
  for (int i = lane; i < N; i += kWarp) {
    m.q[i] = q[vb + i];
    m.lo[i] = lower[vb + i];
    m.hi[i] = upper[vb + i];
    m.x[i] = x_init ? x_init[vb + i] : S(0);
  }
  __syncwarp();
  if (!x_init) {  // pnqp.py:14-19
    if (N == 1) {
      if (lane == 0) m.x[0] = -(S(1) / Hb[0]) * m.q[0];
    } else {
      for (int i = 0; i < N; ++i)
        for (int j = lane; j < N; j += kWarp) a[(size_t)i * N + j] = __ldg(&Hb[(size_t)i * N + j]);
      for (int i = lane; i < N; i += kWarp) m.x[i] = m.q[i];
      __syncwarp();
      rt_lu_factor_warp<S>(a, m.piv, N, lane);
      if (lane == 0) {
        rt_lu_solve<S>(a, m.piv, N, m.x);
        for (int i = 0; i < N; ++i) m.x[i] = -m.x[i];
      }
    }
    __syncwarp();
  }
  for (int i = lane; i < N; i += kWarp) m.x[i] = eclamp<S>(m.x[i], m.lo[i], m.hi[i]);  // pnqp.py:23
  __syncwarp();

  // lane 0: the N == 1 reciprocal of the masked Hessian, reused while it is unchanged (h_last
  // starts as NaN, which no Hessian compares equal to: pnqp_thread's have_r == false)
  S h_last = S(NAN), r_last = S(0);
  for (int it = 0; it < n_iter; ++it) {
    for (int i = lane; i < N; i += kWarp) {  // g = H x + q   (pnqp.py:29), pnqp.py:32-33
      S acc = S(0);
      for (int j = 0; j < N; ++j) acc = fmaS<S>(__ldg(&Hb[(size_t)i * N + j]), m.x[j], acc);
      const S gi = acc + m.q[i];
      m.g[i] = gi;
      const S xi = m.x[i];
      const bool Ic = ((xi == m.lo[i]) && (gi > S(0))) || ((xi == m.hi[i]) && (gi < S(0)));
      m.flag[i] = !Ic;
    }
    __syncwarp();
    for (int i = 0; i < N; ++i) {  // pnqp.py:44-48
      const bool fi = m.flag[i] != 0;
      for (int j = lane; j < N; j += kWarp) {
        S h = (fi && m.flag[j]) ? __ldg(&Hb[(size_t)i * N + j]) : S(0);
        if (i == j) h = h + S(1e-11);
        a[(size_t)i * N + j] = h;
      }
    }
    for (int i = lane; i < N; i += kWarp) m.dx[i] = m.flag[i] ? m.g[i] : S(0);
    __syncwarp();
    if (N > 1) rt_lu_factor_warp<S>(a, m.piv, N, lane);
    bool J = false;
    uint32_t vote = 0;
    if (lane == 0) {
      if (N == 1) {  // pnqp.py:50-51
        if (!(a[0] == h_last)) {
          h_last = a[0];
          r_last = S(1) / h_last;
        }
        m.dx[0] = -r_last * m.dx[0];
      } else {
        rt_lu_solve<S>(a, m.piv, N, m.dx);
        for (int i = 0; i < N; ++i) m.dx[i] = -m.dx[i];
      }
      S nrm2 = S(0);
      for (int i = 0; i < N; ++i) nrm2 = fmaS<S>(m.dx[i], m.dx[i], nrm2);
      J = (N == 1) ? (absS<S>(m.dx[0]) >= S(1e-4)) : (sqrtS<S>(nrm2) >= S(1e-4));   // pnqp.py:56
      if (J) vote |= 1u;
    }
    J = __shfl_sync(kFull, J, 0);
    __syncwarp();   // lane 0's dx before the other lanes read it
    const uint32_t gword = solo ? 0u : __ldg(&guess[it]);
    const bool any_moving = solo ? J : (gword & 1u) != 0;
    if (!any_moving) {  // pnqp.py:57-59
      if (!solo && vote && lane == 0) vote_or(&votes[it], vote);
      break;
    }
    // Armijo backtracking with a batch-global exit test (pnqp.py:61-76)
    S fx = rt_quad_warp<S>(Hb, m.x, m.col, N, lane);
    if (lane == 0) {
      S dot = S(0);
      for (int i = 0; i < N; ++i) dot = fmaS<S>(m.q[i], m.x[i], dot);
      fx = S(0.5) * fx + dot;
    }
    S alpha = S(1);
    for (int cnt = 0; cnt < kArmijoMax; ++cnt) {
      __syncwarp();   // lane 0 is done reading col / mx of the previous pass
      for (int i = lane; i < N; i += kWarp)
        m.mx[i] = eclamp<S>(m.x[i] + alpha * m.dx[i], m.lo[i], m.hi[i]);
      __syncwarp();
      S arm = GAMMA + S(1e-6);
      if (J) {
        const S quad = rt_quad_warp<S>(Hb, m.mx, m.col, N, lane);
        if (lane == 0) {
          S dot = S(0), gd = S(0);
          for (int i = 0; i < N; ++i) dot = fmaS<S>(m.q[i], m.mx[i], dot);
          for (int i = 0; i < N; ++i) gd = fmaS<S>(m.g[i], m.x[i] - m.mx[i], gd);
          arm = (fx - (S(0.5) * quad + dot)) / gd;
        }
      }
      const bool small = __shfl_sync(kFull, arm <= GAMMA, 0);   // pnqp.py:73
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
    __syncwarp();
    for (int i = lane; i < N; i += kWarp) m.x[i] = m.mx[i];  // pnqp.py:78
    __syncwarp();
    if (!solo && vote && lane == 0) vote_or(&votes[it], vote);
  }
  // fell through or stopped: x, the free set and the factor of the last evaluated iteration
  // (pnqp.py:58,81-82); a[] already holds the factor (n == 1: the scalar H_)
  for (int i = lane; i < N; i += kWarp) {
    x_out[vb + i] = m.x[i];
    if_out[vb + i] = m.flag[i] ? S(1) : S(0);
    piv_out[vb + i] = (N == 1) ? 1 : m.piv[i] + 1;
  }
}

// Verify the replayed trace of one dilqr_pnqp_rt call: n_iter guess words, n_iter vote words.
static __global__ void pnqp_rt_verify_kernel(uint32_t* __restrict__ guess,
                                             const uint32_t* __restrict__ votes, int n_iter,
                                             int solo, DilqrStatus* status) {
  trace_verify_block<0>(guess, votes, 1, n_iter, 1, solo, status, nullptr);
}

}  // namespace dilqr
