// krylov_kernels.cuh -- restarted GMRES(m) for the adjoint system of the DiLQR backward,
//   A' w = g,   A' v = v - M' v,
// independent per problem, one thread per problem.  M' v is one adjoint LQR solve of the
// existing kernels (dilqr_adjoint_pass with g = 0, or the generic adjoint solve followed by
// dilqr_richardson_update with g = 0); the caller applies it between the calls below:
//
//   start            w = 0, r = g, v_0 = g / |g|                       -> op_in = +-v_0
//   [operator]       op_out = M' op_in
//   arnoldi (j)      A'v_j = v_j - op_out, CGS2 against v_0..v_j, Givens -> op_in = +-v_{j+1}
//   ... (j = 0 .. steps-1, operator before each)
//   update           y = R^-1 gamma, w += V y                          -> op_in = +-w
//   [operator]
//   restart          r = g - A'w: freeze the problem if |r|/|g| <= tol, else v_0 = r / |r|
//
// Vectors keep the API layout [T,B,n]: at a fixed t, 32 consecutive problems are one
// contiguous run of 32 n scalars.  Every per-problem sum runs over (t, k) in a fixed order in
// FP64, with no atomics on values, so a problem's result does not depend on which problems
// share its batch.  The small per-problem Krylov data (Hessenberg column, rotations, gamma,
// the triangle R) is FP64 in both dtypes.  ctl[0] counts the problems still iterating: when
// it is 0 every kernel here exits at once.
#pragma once
#include "common.cuh"

namespace dilqr {

template <class S>
struct KrylovParams {
  int T, B, n, ns, m, j;
  double tol;
  int negate;            // op_in receives -v (the generic adjoint solve reads -r)
  const S* gx;           // [T,B,ns] (NULL: zero)
  const S* gu;           // [T,B,n-ns]
  S* w;                  // [T,B,n]
  S* opin;               // [T,B,n] operator input
  const S* opout;        // [T,B,n] M' op_in (may alias opin)
  S* V;                  // (m+1) x [T,B,n] basis
  double* H;             // [m+1][B] Hessenberg column of the current step
  double* Y;             // [m+1][B] second CGS sweep's coefficients, then y
  double* R;             // [m(m+1)/2][B] rotated Hessenberg triangle, column j at j(j+1)/2
  double* gam;           // [m+1][B] rotated right-hand side; |gam[j+1]| = residual estimate
  double* cs;            // [m][B]
  double* sn;            // [m][B]
  double* gnorm;         // [B] |g|
  int* klen;             // [B] columns of the current cycle
  int* flags;            // [B] bit 0: frozen (converged, g = 0 or not finite); bit 1: cycle ended
  int* iters;            // [B] Arnoldi steps taken
  double* resid;         // [B] |g - A'w| / |g| at the latest restart
  unsigned* ctl;         // [0] problems iterating, [1] count of the next cycle
};

constexpr int kKrylovChunk = 8;   // dot products held in registers per sweep over the vectors

template <class S>
struct KrylovThread {
  const KrylovParams<S>& p;
  int b;
  size_t vs;             // scalars per vector, T * B * n
  DILQR_DEVICE KrylovThread(const KrylovParams<S>& p_, int b_)
      : p(p_), b(b_), vs((size_t)p_.T * p_.B * p_.n) {}
  DILQR_DEVICE size_t off(int t, int k) const { return ((size_t)t * p.B + b) * p.n + k; }
  DILQR_DEVICE double g(int t, int k) const {
    const size_t tb = (size_t)t * p.B + b;
    if (k < p.ns) return p.gx ? (double)p.gx[tb * p.ns + k] : 0.0;
    return (double)p.gu[tb * (p.n - p.ns) + (k - p.ns)];
  }
  DILQR_DEVICE double& at(double* a, int i) const { return a[(size_t)i * p.B + b]; }
  DILQR_DEVICE void put_op(size_t o, S v) const { p.opin[o] = p.negate ? -v : v; }
  DILQR_DEVICE void zero_op() const {
    for (int t = 0; t < p.T; ++t)
      for (int k = 0; k < p.n; ++k) p.opin[off(t, k)] = S(0);
  }
  // h[i] = <v_i, u> for i = 0..j (chunks of kKrylovChunk accumulators in registers);
  // u = v_j - op_out (first sweep) or the partially orthogonalised vector in v_{j+1}
  DILQR_DEVICE void dots(int j, bool first, double* h) const {
    const S* vj = p.V + (size_t)j * vs;
    const S* vn = p.V + (size_t)(j + 1) * vs;
    for (int i0 = 0; i0 <= j; i0 += kKrylovChunk) {
      double acc[kKrylovChunk];
#pragma unroll
      for (int c = 0; c < kKrylovChunk; ++c) acc[c] = 0.0;
      for (int t = 0; t < p.T; ++t)
        for (int k = 0; k < p.n; ++k) {
          const size_t o = off(t, k);
          const double u = first ? (double)vj[o] - (double)p.opout[o] : (double)vn[o];
#pragma unroll
          for (int c = 0; c < kKrylovChunk; ++c)
            if (i0 + c <= j) acc[c] += (double)p.V[(size_t)(i0 + c) * vs + o] * u;
        }
#pragma unroll
      for (int c = 0; c < kKrylovChunk; ++c)
        if (i0 + c <= j) at(h, i0 + c) = acc[c];
    }
  }
  // v_{j+1} = u - sum_i h[i] v_i; returns |v_{j+1}|^2 of the stored vector
  DILQR_DEVICE double subtract(int j, bool first, double* h) const {
    const S* vj = p.V + (size_t)j * vs;
    S* vn = p.V + (size_t)(j + 1) * vs;
    double s2 = 0.0;
    for (int t = 0; t < p.T; ++t)
      for (int k = 0; k < p.n; ++k) {
        const size_t o = off(t, k);
        double u = first ? (double)vj[o] - (double)p.opout[o] : (double)vn[o];
        for (int i = 0; i <= j; ++i) u -= at(h, i) * (double)p.V[(size_t)i * vs + o];
        const S us = (S)u;
        vn[o] = us;
        s2 += (double)us * (double)us;
      }
    return s2;
  }
};

template <class S>
__global__ void __launch_bounds__(128) krylov_start_kernel(const __grid_constant__ KrylovParams<S> p) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  KrylovThread<S> q(p, b);
  double s2 = 0.0;
  for (int t = 0; t < p.T; ++t)
    for (int k = 0; k < p.n; ++k) {
      const double gv = q.g(t, k);
      s2 += gv * gv;
      p.w[q.off(t, k)] = S(0);
    }
  const double gn = sqrt(s2);
  p.gnorm[b] = gn;
  p.iters[b] = 0;
  p.klen[b] = 0;
  if (!(gn > 0.0) || !isfinite(gn)) {   // g = 0: w = 0 is exact; a non-finite g is reported
    p.flags[b] = 1;
    p.resid[b] = gn == 0.0 ? 0.0 : gn;
    q.zero_op();
    return;
  }
  p.flags[b] = 0;
  p.resid[b] = 1.0;
  q.at(p.gam, 0) = gn;
  for (int t = 0; t < p.T; ++t)
    for (int k = 0; k < p.n; ++k) {
      const size_t o = q.off(t, k);
      const S v = (S)(q.g(t, k) / gn);
      p.V[o] = v;
      q.put_op(o, v);
    }
  atomicAdd(&p.ctl[0], 1u);
}

template <class S>
__global__ void __launch_bounds__(128) krylov_arnoldi_kernel(const __grid_constant__ KrylovParams<S> p) {
  if (p.ctl[0] == 0u) return;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  KrylovThread<S> q(p, b);
  if (p.flags[b]) {       // frozen, or this problem's cycle has ended: keep the operator input finite
    q.zero_op();
    return;
  }
  const int j = p.j;
  // classical Gram-Schmidt with one reorthogonalisation (CGS2)
  q.dots(j, true, p.H);
  q.subtract(j, true, p.H);
  q.dots(j, false, p.Y);
  const double hn = sqrt(q.subtract(j, false, p.Y));
  for (int i = 0; i <= j; ++i) q.at(p.H, i) += q.at(p.Y, i);
  // previous rotations on the new column, then the one that annihilates h[j+1]
  for (int i = 0; i < j; ++i) {
    const double a = q.at(p.H, i), c = q.at(p.cs, i), s = q.at(p.sn, i);
    const double bb = q.at(p.H, i + 1);
    q.at(p.H, i) = c * a + s * bb;
    q.at(p.H, i + 1) = -s * a + c * bb;
  }
  const double a = q.at(p.H, j);
  const double r = hypot(a, hn);
  if (!(r > 0.0) || !isfinite(r)) {   // A' singular on the Krylov space: end with the columns so far
    p.flags[b] |= 2;
    q.zero_op();
    return;
  }
  const double c = a / r, s = hn / r;
  q.at(p.cs, j) = c;
  q.at(p.sn, j) = s;
  const size_t rc = (size_t)j * (j + 1) / 2;
  for (int i = 0; i < j; ++i) q.at(p.R, (int)(rc + i)) = q.at(p.H, i);
  q.at(p.R, (int)(rc + j)) = r;
  const double gj = q.at(p.gam, j);
  q.at(p.gam, j) = c * gj;
  q.at(p.gam, j + 1) = -s * gj;
  p.klen[b] = j + 1;
  p.iters[b] += 1;
  const bool stop = !(hn > 0.0) || fabs(q.at(p.gam, j + 1)) <= p.tol * p.gnorm[b];
  if (stop) {
    p.flags[b] |= 2;
    q.zero_op();
    return;
  }
  S* vn = p.V + (size_t)(j + 1) * q.vs;
  for (int t = 0; t < p.T; ++t)
    for (int k = 0; k < p.n; ++k) {
      const size_t o = q.off(t, k);
      const S v = (S)((double)vn[o] / hn);
      vn[o] = v;
      q.put_op(o, v);
    }
}

template <class S>
__global__ void __launch_bounds__(128) krylov_update_kernel(const __grid_constant__ KrylovParams<S> p) {
  if (p.ctl[0] == 0u) return;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  KrylovThread<S> q(p, b);
  if (p.flags[b] & 1) {
    q.zero_op();
    return;
  }
  const int kl = p.klen[b];
  for (int i = kl - 1; i >= 0; --i) {       // R y = gamma
    double acc = q.at(p.gam, i);
    for (int l = i + 1; l < kl; ++l) acc -= q.at(p.R, (int)((size_t)l * (l + 1) / 2 + i)) * q.at(p.Y, l);
    q.at(p.Y, i) = acc / q.at(p.R, (int)((size_t)i * (i + 1) / 2 + i));
  }
  for (int t = 0; t < p.T; ++t)
    for (int k = 0; k < p.n; ++k) {
      const size_t o = q.off(t, k);
      double acc = 0.0;
      for (int i = 0; i < kl; ++i) acc += q.at(p.Y, i) * (double)p.V[(size_t)i * q.vs + o];
      const S wn = (S)((double)p.w[o] + acc);
      p.w[o] = wn;
      q.put_op(o, wn);
    }
}

template <class S>
__global__ void __launch_bounds__(128) krylov_restart_kernel(const __grid_constant__ KrylovParams<S> p) {
  if (p.ctl[0] == 0u) return;
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  if (p.flags[b] & 1) return;
  KrylovThread<S> q(p, b);
  auto res = [&](int t, int k) {          // r = g - (w - M'w)
    const size_t o = q.off(t, k);
    return q.g(t, k) - ((double)p.w[o] - (double)p.opout[o]);
  };
  double s2 = 0.0;
  for (int t = 0; t < p.T; ++t)
    for (int k = 0; k < p.n; ++k) {
      const double r = res(t, k);
      s2 += r * r;
    }
  const double beta = sqrt(s2);
  const double rel = beta / p.gnorm[b];
  p.resid[b] = rel;
  p.klen[b] = 0;
  if (rel <= p.tol || !isfinite(rel)) {
    p.flags[b] = 1;
    return;
  }
  p.flags[b] = 0;
  q.at(p.gam, 0) = beta;
  for (int t = 0; t < p.T; ++t)
    for (int k = 0; k < p.n; ++k) {
      const size_t o = q.off(t, k);
      const S v = (S)(res(t, k) / beta);
      p.V[o] = v;
      q.put_op(o, v);
    }
  atomicAdd(&p.ctl[1], 1u);
}

}  // namespace dilqr
