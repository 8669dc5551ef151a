// Row-wise 2x2-block LU and substitutions of one scenario, shared by the power flow (k_pf_newton, in fp64) and the state estimator
// (k_wls_estimate, in double-double).  The pattern comes from the host (dss2.powerflow.block_elimination): blk_ptr / blk_col the
// factor's blocks in elimination-position order with fill, columns ascending; diag[k] block (k, k); upd_ptr / upd, per lower block
// p = (k, m), the pairs (block (k, j), block (m, j)) over the upper entries j > m of row m.  Matrix and right-hand side live in the
// caller's index-major workspace column as arrays of the scalar type S::T (S::ld / S::st give element i): block p = [[a, b], [c, d]]
// at elements 4 p .. 4 p + 3, entry k of the right-hand side at element k (first unknown of the block) and n + k (second).
#pragma once
#include <stdint.h>

// fp64: element i at A[i C]
struct F64 {
  using T = double;
  __device__ static __forceinline__ T ld(const double* A, int64_t C, int64_t i) { return A[i * C]; }
  __device__ static __forceinline__ void st(double* A, int64_t C, int64_t i, T x) { A[i * C] = x; }
  __device__ static __forceinline__ double mag(T x) { return fabs(x); }
};

// double-double (Dekker / Knuth error-free transformations; about 106 bits): element i at A[2 i C] (high part), A[(2 i + 1) C] (low)
struct DD {
  struct T {
    double hi, lo;
  };
  __device__ static __forceinline__ T ld(const double* A, int64_t C, int64_t i) { return {A[2 * i * C], A[(2 * i + 1) * C]}; }
  __device__ static __forceinline__ void st(double* A, int64_t C, int64_t i, T x) {
    A[2 * i * C] = x.hi;
    A[(2 * i + 1) * C] = x.lo;
  }
  __device__ static __forceinline__ double mag(T x) { return fabs(x.hi); }
};
__device__ __forceinline__ DD::T dd_quick(double s, double e) {
  const double h = s + e;
  return {h, e - (h - s)};
}
__device__ __forceinline__ DD::T operator+(DD::T x, DD::T y) {
  const double s = x.hi + y.hi, bb = s - x.hi;
  const double e = ((x.hi - (s - bb)) + (y.hi - bb)) + (x.lo + y.lo);
  return dd_quick(s, e);
}
__device__ __forceinline__ DD::T operator-(DD::T y) { return {-y.hi, -y.lo}; }
__device__ __forceinline__ DD::T operator-(DD::T x, DD::T y) { return x + (-y); }
__device__ __forceinline__ DD::T operator*(DD::T x, DD::T y) {
  const double p = x.hi * y.hi;
  const double e = fma(x.hi, y.hi, -p) + (x.hi * y.lo + x.lo * y.hi);
  return dd_quick(p, e);
}
__device__ __forceinline__ DD::T operator/(DD::T x, DD::T y) {
  const double q1 = x.hi / y.hi;
  const DD::T r = x - y * DD::T{q1, 0.0};
  return dd_quick(q1, r.hi / y.hi);
}

template <class T>
struct BlkT {
  T a, b, c, d;                  // [[a, b], [c, d]]
};
using Blk = BlkT<double>;

template <class S = F64>
__device__ __forceinline__ BlkT<typename S::T> ld_blk(const double* A, int64_t C, int p) {
  const int64_t i = (int64_t)4 * p;
  return {S::ld(A, C, i), S::ld(A, C, i + 1), S::ld(A, C, i + 2), S::ld(A, C, i + 3)};
}
template <class S = F64>
__device__ __forceinline__ void st_blk(double* A, int64_t C, int p, const BlkT<typename S::T>& x) {
  const int64_t i = (int64_t)4 * p;
  S::st(A, C, i, x.a);
  S::st(A, C, i + 1, x.b);
  S::st(A, C, i + 2, x.c);
  S::st(A, C, i + 3, x.d);
}
template <class T>
__device__ __forceinline__ BlkT<T> mul(const BlkT<T>& x, const BlkT<T>& y) {
  return {x.a * y.a + x.b * y.c, x.a * y.b + x.b * y.d, x.c * y.a + x.d * y.c, x.c * y.b + x.d * y.d};
}

struct BlockLu {
  int n;                                   // block rows
  const int32_t *blk_ptr, *blk_col, *diag, *upd_ptr, *upd;
};

// Factorise A in place: L[k,m] = A[k,m] inv(A[m,m]) for m < k ascending, A[k,j] -= L[k,m] A[m,j] (j > m); then invert A[k,k].
// Returns false at the first pivot with |det| <= 1e-12 (|ad| + |bc|) (A is then partly factorised).
template <class S = F64>
__device__ __forceinline__ bool block_lu_factor(const BlockLu& t, double* A, int64_t C) {
  using T = typename S::T;
  for (int k = 0; k < t.n; ++k) {
    const int dk = __ldg(t.diag + k);
    for (int p = __ldg(t.blk_ptr + k); p < dk; ++p) {
      const BlkT<T> L = mul(ld_blk<S>(A, C, p), ld_blk<S>(A, C, __ldg(t.diag + __ldg(t.blk_col + p))));
      st_blk<S>(A, C, p, L);
      for (int u = __ldg(t.upd_ptr + p); u < __ldg(t.upd_ptr + p + 1); ++u) {
        const int dst = __ldg(t.upd + 2 * u), src = __ldg(t.upd + 2 * u + 1);
        const BlkT<T> x = ld_blk<S>(A, C, dst), y = mul(L, ld_blk<S>(A, C, src));
        st_blk<S>(A, C, dst, {x.a - y.a, x.b - y.b, x.c - y.c, x.d - y.d});
      }
    }
    const BlkT<T> D = ld_blk<S>(A, C, dk);
    const T det = D.a * D.d - D.b * D.c;
    if (!(S::mag(det) > 1e-12 * (S::mag(D.a * D.d) + S::mag(D.b * D.c)))) return false;
    const T r = T{1.0} / det;
    st_blk<S>(A, C, dk, {D.d * r, -D.b * r, -D.c * r, D.a * r});
  }
  return true;
}

// Solve with the factor of block_lu_factor: the right-hand side in F is replaced by the solution.
template <class S = F64>
__device__ __forceinline__ void block_lu_solve(const BlockLu& t, const double* A, double* F, int64_t C) {
  using T = typename S::T;
  const int n = t.n;
  // forward: y_k = F_k - sum_{m<k} L[k,m] y_m
  for (int k = 0; k < n; ++k) {
    T yp = S::ld(F, C, k), yq = S::ld(F, C, n + k);
    for (int p = __ldg(t.blk_ptr + k); p < __ldg(t.diag + k); ++p) {
      const BlkT<T> L = ld_blk<S>(A, C, p);
      const int m = __ldg(t.blk_col + p);
      const T xp = S::ld(F, C, m), xq = S::ld(F, C, n + m);
      yp = yp - (L.a * xp + L.b * xq);
      yq = yq - (L.c * xp + L.d * xq);
    }
    S::st(F, C, k, yp);
    S::st(F, C, n + k, yq);
  }
  // back: x_k = inv(A[k,k]) (y_k - sum_{j>k} A[k,j] x_j)
  for (int k = n - 1; k >= 0; --k) {
    const int dk = __ldg(t.diag + k);
    T yp = S::ld(F, C, k), yq = S::ld(F, C, n + k);
    for (int p = dk + 1; p < __ldg(t.blk_ptr + k + 1); ++p) {
      const BlkT<T> U = ld_blk<S>(A, C, p);
      const int j = __ldg(t.blk_col + p);
      const T xp = S::ld(F, C, j), xq = S::ld(F, C, n + j);
      yp = yp - (U.a * xp + U.b * xq);
      yq = yq - (U.c * xp + U.d * xq);
    }
    const BlkT<T> D = ld_blk<S>(A, C, dk);
    S::st(F, C, k, D.a * yp + D.b * yq);
    S::st(F, C, n + k, D.c * yp + D.d * yq);
  }
}
