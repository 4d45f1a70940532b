// Backward kernels of the packed-symmetric routines for one scalar type (-DNFM_SCALAR):
// the coefficient gradients of sym_matvec / sym_solve (SymOuter2Op), sym_invert
// (SymInvertBackwardOp) and sym_det (SymDetBackwardOp).  The vector gradients reuse
// the forward kernels (A g, (A + diag d)^-1 g).
//
// Notation: p = stored coefficients, g = incoming gradient, S(u, w) = gradient of
// u^T A w with respect to p:  S_ii = u_i w_i,  S_ij = u_i w_j + u_j w_i (i < j) --
// the diagonal is NOT doubled, an off-diagonal coefficient stands for two entries.
#include "nfm_dense_math.cuh"
#include "nfm_impl.cuh"
#include "nfm_sym_ops.cuh"

namespace nfm {

// out = sign * S(u, w) in the layout of the matrix        in0 = u, in1 = w
// (packed: the formula above; diagonal: u_i w_i; scaled identity: sum_i u_i w_i)
template <typename T, int N, int LAYOUT>
struct SymOuter2Op {
  using scalar = T;
  static constexpr int kLen0 = N, kLen1 = N, kLen2 = 1, kUse = 3, kOut = layout_len(LAYOUT, N);
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&u)[N], const T (&w)[N], const T (&)[1], int, int flags, T (&out)[kOut]) {
    const T s = (flags & kFlagSubtract) ? T(-1) : T(1);
    if constexpr (LAYOUT == NFM_LAYOUT_SCALED_IDENTITY) {
      T acc = u[0] * w[0];
#pragma unroll
      for (int i = 1; i < N; ++i) acc += u[i] * w[i];
      out[0] = s * acc;
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i) out[i] = s * (u[i] * w[i]);
      if constexpr (LAYOUT == NFM_LAYOUT_SYM) {
        // compile-time indices: with `#pragma unroll` alone the order 9 / 10 records went to local memory
        static_for<0, N>([&](auto I) {
          constexpr int i = I;
          static_for<i + 1, N>([&](auto J) {
            constexpr int j = J;
            out[pidx(N, i, j)] = s * (u[i] * w[j] + u[j] * w[i]);
          });
        });
      }
    }
  }
};

// Gradient of B = A^-1 (packed) or b = diag(A^-1):      in0 = B (packed), in1 = g (packed, or N values)
//   G^ = symmetric with G^_ii = g_ii, G^_ij = g_ij / 2   (diag(g) when DIAG_ONLY)
//   M = B G^ B ;  out_ii = -M_ii ,  out_ij = -2 M_ij
// M is built one row at a time (row i of B G^, then its products with the columns j >= i of B),
// so beside the two input records only N temporaries are live: nothing of size N^2.
template <typename T, int N, bool DIAG_ONLY>
struct SymInvertBackwardOp {
  using scalar = T;
  static constexpr int kLen0 = packed_len(N), kLen1 = DIAG_ONLY ? N : packed_len(N), kLen2 = 1, kUse = 3, kOut = packed_len(N);
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&b)[kLen0], const T (&g)[kLen1], const T (&)[1], int, int, T (&out)[kOut]) {
    static_for<0, N>([&](auto I) {
      constexpr int i = I;
      T r[N];  // row i of B G^
      static_for<0, N>([&](auto K) {
        constexpr int k = K;
        if constexpr (DIAG_ONLY) {
          r[k] = b[pidx(N, i, k)] * g[k];
        } else {
          T s = b[pidx(N, i, k)] * g[k];
          static_for<0, N>([&](auto L) {
            constexpr int l = L;
            if constexpr (l != k) s += b[pidx(N, i, l)] * (T(0.5) * g[pidx(N, l, k)]);
          });
          r[k] = s;
        }
      });
      static_for<i, N>([&](auto J) {
        constexpr int j = J;
        T m = r[0] * b[pidx(N, 0, j)];
        static_for<1, N>([&](auto K) { m += r[K] * b[pidx(N, K, j)]; });
        out[pidx(N, i, j)] = (i == j) ? -m : T(-2) * m;
      });
    });
  }
};

// Gradient of t = det A:   out_ii = g adj_ii ,  out_ij = 2 g adj_ij   (adj = t A^-1, the adjugate)
//   in0 = A (packed), in1 = g (one value per matrix)
// N <= 4: the closed-form adjugate (finite for singular matrices).  N > 4: checked LDL^T gives both
// A^-1 and t = prod d_k; a matrix that fails the pivot check is redone as SymDetOp (pivoted LU) and
// the AUTO fallback of SymInvertOp (pivoted Gauss-Jordan) do it, one after the other.
template <typename T, int N>
struct SymDetBackwardOp {
  using scalar = T;
  static constexpr int kLen0 = packed_len(N), kLen1 = 1, kLen2 = 1, kUse = 3, kOut = packed_len(N);
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&m)[kLen0], const T (&g)[1], const T (&)[1], int, int, T (&out)[kOut]) {
    T scale;  // g * t, or g alone when out already holds the adjugate
    if constexpr (N <= 4) {
      sym_adjugate<T, N>(m, out);
      scale = g[0];
    } else {
      LDL<T, N> f;
      f.load_packed(m);
      if (f.factor_checked()) {
        T t = f.w[0][0];
#pragma unroll
        for (int k = 1; k < N; ++k) t *= f.w[k][k];
        f.template invert<false>(out);
        scale = g[0] * t;
      } else {
        {
          GaussPP<T, N, 0> e;
#pragma unroll
          for (int i = 0; i < N; ++i)
#pragma unroll
            for (int j = 0; j < N; ++j) e.a[i][j] = m[pidx(N, i, j)];
          e.eliminate();
          scale = g[0] * e.det();
        }
        GaussJordan<T, N> e;
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = 0; j < N; ++j) e.a[i][j] = m[pidx(N, i, j)];
        e.invert();
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = i; j < N; ++j) out[pidx(N, i, j)] = e.a[j][i];
      }
    }
#pragma unroll
    for (int k = 0; k < kOut; ++k) out[k] *= (k < N) ? scale : T(2) * scale;
  }
};

template <typename T, int LAYOUT> struct Outer2Bind { template <int N> using Op = SymOuter2Op<T, N, LAYOUT>; };
template <typename T, bool DIAG_ONLY> struct InvBwdBind { template <int N> using Op = SymInvertBackwardOp<T, N, DIAG_ONLY>; };
template <typename T> struct DetBwdBind { template <int N> using Op = SymDetBackwardOp<T, N>; };

template <typename T>
int sym_outer2_impl(int n, int layout, const KParams& p, cudaStream_t s) {
  switch (layout) {
    case NFM_LAYOUT_SCALED_IDENTITY:
      return DispatchN<Outer2Bind<T, NFM_LAYOUT_SCALED_IDENTITY>::template Op, 1, NFM_MAX_N>::run(n, p, s);
    case NFM_LAYOUT_DIAG:
      return DispatchN<Outer2Bind<T, NFM_LAYOUT_DIAG>::template Op, 1, NFM_MAX_N>::run(n, p, s);
    case NFM_LAYOUT_SYM:
      return DispatchN<Outer2Bind<T, NFM_LAYOUT_SYM>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  }
  return NFM_E_UNSUPPORTED;
}

template <typename T>
int sym_invert_backward_impl(int n, int diag_only, const KParams& p, cudaStream_t s) {
  if (diag_only) return DispatchN<InvBwdBind<T, true>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  return DispatchN<InvBwdBind<T, false>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}

template <typename T>
int sym_det_backward_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<DetBwdBind<T>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}

template int sym_outer2_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
template int sym_invert_backward_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
template int sym_det_backward_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);

}  // namespace nfm
