// Backward kernels of the dense routines for one scalar type (-DNFM_SCALAR) and one part
// (-DNFM_PART): the gradients of batchinv / inv (BatchInvBackwardOp) and batchdet
// (BatchDetBackwardOp), and the matrix gradient of lmdiv / solvevec / rmdiv / batchmatvec
// (BatchOuterOp).  The gradients with respect to the right-hand sides and vectors are the
// transposed solves (BatchSolveKOp with kFlagTransposeA, solve_many_kernel) and the transposed
// matvec (BatchMatvecOp<.., true>).  Records are dense row-major n x n (n x k, k x n).
//
// For method 'chol' (LDL^T of the lower triangle) the gradient is the symmetric part of the
// general formula, the convention of torch's cholesky + cholesky_solve / cholesky_inverse.
#include "nfm_dense_ops.cuh"
#include "nfm_impl.cuh"
#include "nfm_sym_ops.cuh"

namespace nfm {

// BatchOuterOp flags: the record order is kFlagRightDivision (as BatchSolveKOp)
constexpr int kFlagOuterNegate = 1;
constexpr int kFlagOuterSym = 8;

#if NFM_PART == 0
// Gradient of Y = A^-1:        in0 = Y, in1 = G, out = dA
//   lu / auto:  dA = -Y^T G Y^T
//   SYM (chol): dA = -Y G^ Y with G^ = (G + G^T) / 2  (Y symmetric)
// Built one row at a time (row i of Y^T G, resp. Y G^, then its products with the rows / columns of
// Y), so beside the two input records only N temporaries are live: nothing of size N^2.
template <typename T, int N, bool SYM>
struct BatchInvBackwardOp {
  using scalar = T;
  static constexpr int kLen0 = N * N, kLen1 = N * N, kLen2 = 1, kUse = 3, kOut = N * N;
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&y)[kLen0], const T (&g)[kLen1], const T (&)[1], int, int, T (&out)[kOut]) {
    static_for<0, N>([&](auto I) {
      constexpr int i = I;
      T r[N];
      static_for<0, N>([&](auto L) {
        constexpr int l = L;
        if constexpr (SYM) {
          T s = y[i * N] * (T(0.5) * (g[l] + g[l * N]));
          static_for<1, N>([&](auto K) {
            constexpr int k = K;
            s += y[i * N + k] * (T(0.5) * (g[k * N + l] + g[l * N + k]));
          });
          r[l] = s;
        } else {
          T s = y[i] * g[l];
          static_for<1, N>([&](auto K) {
            constexpr int k = K;
            s += y[k * N + i] * g[k * N + l];
          });
          r[l] = s;
        }
      });
      static_for<0, N>([&](auto J) {
        constexpr int j = J;
        T m = SYM ? r[0] * y[j] : r[0] * y[j * N];
        static_for<1, N>([&](auto L) {
          constexpr int l = L;
          m += SYM ? r[l] * y[l * N + j] : r[l] * y[j * N + l];
        });
        out[i * N + j] = -m;
      });
    });
  }
};

// Gradient of t = det A:   dA = g adj(A)^T, the cofactor matrix times g.   in0 = A, in1 = g (one value)
// N <= 3: closed-form cofactors (finite for singular A).  N >= 4: one pivoted Gauss-Jordan elimination
// gives A^-1 and det A together, dA = g t A^-T; a singular matrix gives non-finite values there.
template <typename T, int N>
struct BatchDetBackwardOp {
  using scalar = T;
  static constexpr int kLen0 = N * N, kLen1 = 1, kLen2 = 1, kUse = 3, kOut = N * N;
  static constexpr bool kHeavy = N >= 4;
  __device__ static __forceinline__ void apply(const T (&a)[kLen0], const T (&g)[1], const T (&)[1], int, int, T (&out)[kOut]) {
    if constexpr (N == 1) {
      out[0] = g[0];
    } else if constexpr (N == 2) {
      out[0] = g[0] * a[3];
      out[1] = -(g[0] * a[2]);
      out[2] = -(g[0] * a[1]);
      out[3] = g[0] * a[0];
    } else if constexpr (N == 3) {
      static_for<0, 3>([&](auto I) {
        static_for<0, 3>([&](auto J) {
          constexpr int i = I, j = J, i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
          out[i * 3 + j] = g[0] * (a[i1 * 3 + j1] * a[i2 * 3 + j2] - a[i1 * 3 + j2] * a[i2 * 3 + j1]);
        });
      });
    } else {
      GaussJordan<T, N> e;
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) e.a[i][j] = a[i * N + j];
      const T scale = g[0] * e.template invert<true>();
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) out[i * N + j] = scale * e.a[j][i];
    }
  }
};

template <typename T, bool SYM> struct InvBwdBind { template <int N> using Op = BatchInvBackwardOp<T, N, SYM>; };
template <typename T> struct DetBwdBind { template <int N> using Op = BatchDetBackwardOp<T, N>; };

template <typename T>
int batch_inv_backward_impl(int n, int sym, const KParams& p, cudaStream_t s) {
  if (sym) return DispatchN<InvBwdBind<T, true>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  return DispatchN<InvBwdBind<T, false>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template <typename T>
int batch_det_backward_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<DetBwdBind<T>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template int batch_inv_backward_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
template int batch_det_backward_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);

#else
// out = sign * U W^T  (U, W: N x K row-major; the matrix gradient of lmdiv / solvevec, and of the
// square batchmatvec with K = 1), or with kFlagRightDivision  sign * U^T W  (U, W: K x N; rmdiv).
// kFlagOuterSym: sign * (M + M^T) / 2 (method 'chol').  in0 = U, in1 = W.
template <typename T, int N, int K>
struct BatchOuterOp {
  using scalar = T;
  static constexpr int kLen0 = N * K, kLen1 = N * K, kLen2 = 1, kUse = 3, kOut = N * N;
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&u)[kLen0], const T (&w)[kLen1], const T (&)[1], int, int flags,
                                               T (&out)[kOut]) {
    if (flags & kFlagRightDivision) apply_order<true>(u, w, out);
    else apply_order<false>(u, w, out);
    const T sg = (flags & kFlagOuterNegate) ? T(-1) : T(1);
    if (flags & kFlagOuterSym) {
      static_for<0, N>([&](auto I) {
        constexpr int i = I;
        out[i * N + i] *= sg;
        static_for<i + 1, N>([&](auto J) {
          constexpr int j = J;
          const T v = sg * (T(0.5) * (out[i * N + j] + out[j * N + i]));
          out[i * N + j] = v;
          out[j * N + i] = v;
        });
      });
    } else {
#pragma unroll
      for (int q = 0; q < kOut; ++q) out[q] *= sg;
    }
  }

  template <bool rows>
  __device__ static __forceinline__ void apply_order(const T (&u)[kLen0], const T (&w)[kLen1], T (&out)[kOut]) {
    static_for<0, N>([&](auto I) {
      static_for<0, N>([&](auto J) {
        constexpr int i = I, j = J;
        T s = rows ? u[i] * w[j] : u[i * K] * w[j * K];
        static_for<1, K>([&](auto C) {
          constexpr int c = C;
          s += rows ? u[c * N + i] * w[c * N + j] : u[i * K + c] * w[j * K + c];
        });
        out[i * N + j] = s;
      });
    });
  }
};

template <typename T, int K> struct OuterBind { template <int N> using Op = BatchOuterOp<T, N, K>; };

#if NFM_PART == 1
template <typename T>
int batch_outer_k12_impl(int n, int k, const KParams& p, cudaStream_t s) {
  if (k == 1) return DispatchN<OuterBind<T, 1>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  if (k == 2) return DispatchN<OuterBind<T, 2>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  return NFM_E_UNSUPPORTED;
}
template int batch_outer_k12_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
#else
template <typename T>
int batch_outer_k34_impl(int n, int k, const KParams& p, cudaStream_t s) {
  if (k == 3) return DispatchN<OuterBind<T, 3>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  if (k == 4) return DispatchN<OuterBind<T, 4>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  return NFM_E_UNSUPPORTED;
}
template int batch_outer_k34_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
#endif
#endif

}  // namespace nfm
