// nfm_dense_ops.cuh -- Op structs for dense row-major n x n batches:
// inverse, determinant, solve (one right-hand side), square matvec.
#pragma once

#include "nfm_dense_math.cuh"
#include "nfm_pipeline.cuh"
#include "nfm_sym_math.cuh"

namespace nfm {

constexpr int kFlagDetRegularise = 1;  // batch_inv n = 2,3: det += range * 1e-12

// LDL^T loaded from the LOWER triangle of a dense matrix (torch.linalg.cholesky
// with upper=False reads only that triangle, sugar.py:128, :248)
template <typename T, int N>
__device__ __forceinline__ void ldl_from_dense_lower(const T (&a)[N * N], LDL<T, N>& f) {
#pragma unroll
  for (int i = 0; i < N; ++i)
#pragma unroll
    for (int j = i; j < N; ++j) f.w[i][j] = a[j * N + i];
}

template <typename T, int N, int ALGO>
struct BatchInvOp {
  using scalar = T;
  static constexpr int kLen0 = N * N;
  static constexpr int kLen1 = 1;
  static constexpr int kLen2 = 1;
  static constexpr int kUse = 1;
  static constexpr int kOut = N * N;
  static constexpr bool kHeavy = ALGO != NFM_ALGO_LDL && N >= 4;

  __device__ static __forceinline__ void apply(const T (&a)[kLen0], const T (&)[1], const T (&)[1], int present,
                                               int flags, T (&out)[kOut]) {
    if constexpr (ALGO == NFM_ALGO_LDL) {
      LDL<T, N> f;
      ldl_from_dense_lower<T, N>(a, f);
      f.factor();
      T packed[packed_len(N)];
      f.template invert<false>(packed);
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) out[i * N + j] = packed[pidx(N, i, j)];
    } else if constexpr (N <= 3 && ALGO == NFM_ALGO_AUTO) {
      dense_inv_closed<T, N>(a, flags & kFlagDetRegularise, out);
    } else {
      GaussJordan<T, N> g;
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = a[i * N + j];
      g.invert();
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) out[i * N + j] = g.a[i][j];
    }
  }
};

// Pivoted Gauss-Jordan inverse with two lanes per matrix on the warp-pool kernel (dense 16-byte
// aligned batches); the strided kernel and the tail of a launch use the one-thread form it inherits.
// For the orders whose one-thread form is register-bound: fp64 n = 8..10 (200 registers of matrix
// per thread, 255-register kernels with spills, 8 warps per SM).
template <typename T, int N>
struct BatchInvPairOp : BatchInvOp<T, N, NFM_ALGO_AUTO> {
  static constexpr int kPairLanes = 2;
  __device__ static __forceinline__ void apply_pair(unsigned char* record, int lane, int flags) {
    GaussJordanPair<T, N>::invert_in_place(reinterpret_cast<T*>(record), lane);
  }
};

template <typename T, int N>
struct BatchDetOp {
  using scalar = T;
  static constexpr int kLen0 = N * N;
  static constexpr int kLen1 = 1;
  static constexpr int kLen2 = 1;
  static constexpr int kUse = 1;
  static constexpr int kOut = 1;
  static constexpr bool kHeavy = N >= 4;

  __device__ static __forceinline__ void apply(const T (&a)[kLen0], const T (&)[1], const T (&)[1], int present,
                                               int flags, T (&out)[1]) {
    if constexpr (N == 1) out[0] = a[0];
    else if constexpr (N == 2) out[0] = dense_det2(a);
    else if constexpr (N == 3) out[0] = dense_det3(a);
    else {
      GaussPP<T, N, 0> g;
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = a[i * N + j];
      g.eliminate();
      out[0] = g.det();
    }
  }
};

// x = A^-1 b, one right-hand side
template <typename T, int N, int ALGO>
struct BatchSolveOp {
  using scalar = T;
  static constexpr int kLen0 = N * N;
  static constexpr int kLen1 = N;
  static constexpr int kLen2 = 1;
  static constexpr int kUse = 3;
  static constexpr int kOut = N;
  static constexpr bool kHeavy = ALGO != NFM_ALGO_LDL && N >= 2;

  __device__ static __forceinline__ void apply(const T (&a)[kLen0], const T (&b)[N], const T (&)[1], int present,
                                               int flags, T (&x)[N]) {
    if constexpr (ALGO == NFM_ALGO_LDL) {
      LDL<T, N> f;
      ldl_from_dense_lower<T, N>(a, f);
      f.factor();
      f.solve(b, x);
    } else {
      GaussPP<T, N, 1> g;
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = a[i * N + j];
        g.b[i][0] = b[i];
      }
      g.eliminate();
      g.back_substitute();
#pragma unroll
      for (int i = 0; i < N; ++i) x[i] = g.b[i][0];
    }
  }
};

// X = A^-1 B with K right-hand sides; B and X are N x K row-major records.
// With kFlagRightDivision (sugar.rmdiv, K rows): X = B A^-1, B and X are K x N row-major -- the same
// records read with the other index order (A transposed, one right-hand side per ROW of B).
// kFlagTransposeA solves with A^T instead, in either order: X = A^-T B or X = B A^-T (the gradients of
// lmdiv / rmdiv; LDL^T reads a symmetric matrix, so it ignores the bit).  The flags are uniform over the
// launch: one branch picks between fully static instantiations (per-element selects between the two
// orders cost the 4x4 fp32 left division 7 %).
template <typename T, int N, int K, int ALGO>
struct BatchSolveKOp {
  using scalar = T;
  static constexpr int kLen0 = N * N;
  static constexpr int kLen1 = N * K;
  static constexpr int kLen2 = 1;
  static constexpr int kUse = 3;
  static constexpr int kOut = N * K;
  static constexpr bool kHeavy = ALGO != NFM_ALGO_LDL && N >= 2;

  __device__ static __forceinline__ void apply(const T (&a)[kLen0], const T (&b)[kLen1], const T (&z)[1], int present,
                                               int flags, T (&x)[kOut]) {
    const bool right = flags & kFlagRightDivision;
    if constexpr (ALGO != NFM_ALGO_LDL) {
      if (flags & kFlagTransposeA) {
        if (right) apply_order<true, false>(a, b, x);
        else apply_order<false, true>(a, b, x);
        return;
      }
    }
    if (right) apply_order<true, true>(a, b, x);
    else apply_order<false, false>(a, b, x);
  }

  // right: record order of B and X; ta: eliminate with A^T (right division without kFlagTransposeA)
  template <bool right, bool ta>
  __device__ static __forceinline__ void apply_order(const T (&a)[kLen0], const T (&b)[kLen1], T (&x)[kOut]) {
    T sol[N][K];  // sol[i][c]: component i of the solution for right-hand side c
    if constexpr (ALGO == NFM_ALGO_LDL) {
      LDL<T, N> f;
      ldl_from_dense_lower<T, N>(a, f);  // symmetric: the same factors serve both divisions
      f.factor();
#pragma unroll
      for (int c = 0; c < K; ++c) {
        T col[N], s[N];
#pragma unroll
        for (int i = 0; i < N; ++i) col[i] = right ? b[c * N + i] : b[i * K + c];
        f.solve(col, s);
#pragma unroll
        for (int i = 0; i < N; ++i) sol[i][c] = s[i];
      }
    } else {
      GaussPP<T, N, K> g;
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = ta ? a[j * N + i] : a[i * N + j];
#pragma unroll
        for (int c = 0; c < K; ++c) g.b[i][c] = right ? b[c * N + i] : b[i * K + c];
      }
      g.eliminate();
      g.back_substitute();
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int c = 0; c < K; ++c) sol[i][c] = g.b[i][c];
    }
#pragma unroll
    for (int q = 0; q < N * K; ++q) x[q] = right ? sol[q % N][q / N] : sol[q / K][q % K];
  }
};

// y = A v, or y = A^T v when TRANSPOSE (the gradient of batchmatvec with respect to v)
template <typename T, int N, bool TRANSPOSE = false>
struct BatchMatvecOp {
  using scalar = T;
  static constexpr int kLen0 = N * N;
  static constexpr int kLen1 = N;
  static constexpr int kLen2 = 1;
  static constexpr int kUse = 3;
  static constexpr int kOut = N;
  static constexpr bool kHeavy = false;

  __device__ static __forceinline__ void apply(const T (&a)[kLen0], const T (&v)[N], const T (&)[1], int present,
                                               int flags, T (&y)[N]) {
    if constexpr (TRANSPOSE) {
#pragma unroll
      for (int j = 0; j < N; ++j) {
        T s = a[j] * v[0];
#pragma unroll
        for (int i = 1; i < N; ++i) s += a[i * N + j] * v[i];
        y[j] = s;
      }
    } else {
      dense_matvec_reg<T, N, N>(a, v, y);
    }
  }
};

// measured optima (profiles/r1_tile_geometry_sweep.txt): fp64 pivoted elimination
// wants more resident warps than the one-big-CTA rule gives
template <> struct Tune<BatchInvOp<double, 4, NFM_ALGO_AUTO>> : TuneFixed<BatchInvOp<double, 4, NFM_ALGO_AUTO>, 256, 256, 3> {};
template <> struct Tune<BatchDetOp<double, 4>> : TuneFixed<BatchDetOp<double, 4>, 256, 128, 3> {};
template <> struct Tune<BatchSolveOp<double, 4, NFM_ALGO_LU>> : TuneFixed<BatchSolveOp<double, 4, NFM_ALGO_LU>, 128, 128, 3> {};
// fp32 4x4 (sweep 3): 6073 vs 5850 GB/s (solve), 6378 vs 5930 GB/s (det)
template <> struct Tune<BatchSolveOp<float, 4, NFM_ALGO_LU>> : TuneFixed<BatchSolveOp<float, 4, NFM_ALGO_LU>, 256, 256, 3> {};
template <> struct Tune<BatchDetOp<float, 4>> : TuneFixed<BatchDetOp<float, 4>, 512, 256, 3> {};

}  // namespace nfm
