// Backward kernels of the Gauss-Newton builders for one scalar type (-DNFM_SCALAR) and one part
// (-DNFM_PART): the gradients of sym_matmul (SymMatmulBackwardOp; parts 0 / 1 / 2 = dJ only, dH only,
// both), sym_outer (SymOuterBackwardOp) and sym_to_full (SymToFullBackwardOp; part 3).  The fused
// sym_matmul_solve / sym_solve_update have no kernel of their own: their backward passes chain
// nfm_sym_matmul, nfm_sym_solve, nfm_sym_outer2 and the matmul backward here.
//
// Notation: g = incoming gradient of a packed result of order n, G^ = its full symmetric matrix with
// the off-diagonals halved (G^_ii = g_ii, G^_ij = g_ij / 2).  pack(M) = M_ii, 2 M_ij (i < j).
#include "nfm_impl.cuh"
#include "nfm_pipeline.cuh"
#include "nfm_sym_ops.cuh"

namespace nfm {

#if NFM_PART <= 2
// Gradient of Y = J^T H J (MODE 0; J: K x D row-major, H packed of order K) or Y = J H J^T (MODE 1,
// K == D).  With F the ON x HN factor of the forward's Y = F H F^T (F = J^T in mode 0, J in mode 1):
//   dF = 2 G^ F H   (dJ = dF^T in mode 0, dF in mode 1),   dH = pack(F^T G^ F)
//   in0 = J, in1 = H (packed), in2 = g (packed, order ON)
// out: WHICH 1 = dJ (K * D values), 2 = dH (packed), 3 = [dJ | dH] in one record.  Both are built one
// row at a time (row o of G^ F, then its products with the columns of H; row a of F^T G^, then its
// products with the columns b >= a of F), so beside the records only max(ON, HN) temporaries are live.
template <typename T, int K, int D, int MODE, int WHICH>
struct SymMatmulBackwardOp {
  using scalar = T;
  static constexpr int kHN = MODE == 0 ? K : D;  // order of H
  static constexpr int kON = MODE == 0 ? D : K;  // order of Y
  static constexpr int kJ = (WHICH & 1) ? K * D : 0;
  static constexpr int kLen0 = K * D, kLen1 = packed_len(kHN), kLen2 = packed_len(kON), kUse = 7;
  static constexpr int kOut = kJ + ((WHICH & 2) ? packed_len(kHN) : 0);
  static constexpr bool kHeavy = false;
  static constexpr bool kThreeMandatory = true;

  template <int O, int A>
  __device__ static __forceinline__ T f(const T (&j)[kLen0]) { return MODE == 0 ? j[A * D + O] : j[O * D + A]; }
  template <int O, int Q>
  __device__ static __forceinline__ T ghat(const T (&g)[kLen2]) {
    return O == Q ? g[O] : T(0.5) * g[pidx(kON, O, Q)];
  }

  __device__ static __forceinline__ void apply(const T (&j)[kLen0], const T (&h)[kLen1], const T (&g)[kLen2], int, int,
                                               T (&out)[kOut]) {
    if constexpr ((WHICH & 1) != 0) {
      static_for<0, kON>([&](auto O) {
        constexpr int o = O;
        T r[kHN];  // row o of G^ F
        static_for<0, kHN>([&](auto A) {
          constexpr int a = A;
          T s = ghat<o, 0>(g) * f<0, a>(j);
          static_for<1, kON>([&](auto Q) { s += ghat<o, Q>(g) * f<Q, a>(j); });
          r[a] = s;
        });
        static_for<0, kHN>([&](auto B) {
          constexpr int b = B;
          T s = r[0] * h[pidx(kHN, 0, b)];
          static_for<1, kHN>([&](auto A) { s += r[A] * h[pidx(kHN, A, b)]; });
          out[MODE == 0 ? b * D + o : o * D + b] = T(2) * s;
        });
      });
    }
    if constexpr ((WHICH & 2) != 0) {
      static_for<0, kHN>([&](auto A) {
        constexpr int a = A;
        T t[kON];  // row a of F^T G^
        static_for<0, kON>([&](auto Q) {
          constexpr int q = Q;
          T s = f<0, a>(j) * ghat<0, q>(g);
          static_for<1, kON>([&](auto O) { s += f<O, a>(j) * ghat<O, q>(g); });
          t[q] = s;
        });
        static_for<a, kHN>([&](auto B) {
          constexpr int b = B;
          T s = t[0] * f<0, b>(j);
          static_for<1, kON>([&](auto Q) { s += t[Q] * f<Q, b>(j); });
          out[kJ + pidx(kHN, a, b)] = a == b ? s : T(2) * s;
        });
      });
    }
  }
};

template <typename T, int K, int D, int WHICH>
static int matmul_backward_run(int mode, const KParams& p, cudaStream_t s) {
  if (mode == 0) return run_op<SymMatmulBackwardOp<T, K, D, 0, WHICH>>(p, s);
  if constexpr (K == D && K <= 3) return run_op<SymMatmulBackwardOp<T, K, D, 1, WHICH>>(p, s);  // the reference's unrolled branches
  else return NFM_E_UNSUPPORTED;
}

// the shapes the forward has register kernels for (fused_shape_built), in k-major order
template <typename T, int WHICH, int K, int D>
static int matmul_backward_kd(int k, int d, int mode, const KParams& p, cudaStream_t s) {
  if constexpr (fused_shape_built(K, D)) {
    if (k == K && d == D) return matmul_backward_run<T, K, D, WHICH>(mode, p, s);
  }
  if constexpr (D < NFM_MAX_N) return matmul_backward_kd<T, WHICH, K, D + 1>(k, d, mode, p, s);
  else if constexpr (K < NFM_MAX_N) return matmul_backward_kd<T, WHICH, K + 1, 1>(k, d, mode, p, s);
  else return NFM_E_UNSUPPORTED;
}

template <typename T, int WHICH>
int sym_matmul_backward_impl(int k, int d, int mode, const KParams& p, cudaStream_t s) {
  return matmul_backward_kd<T, WHICH, 1, 1>(k, d, mode, p, s);
}
template int sym_matmul_backward_impl<NFM_SCALAR, NFM_PART + 1>(int, int, int, const KParams&, cudaStream_t);

#else
// Gradient of y = x x^T (packed):  dx = 2 G^ x,  i.e. dx_i = 2 g_ii x_i + sum_{j != i} g_ij x_j
//   in0 = x, in1 = g (packed)
template <typename T, int N>
struct SymOuterBackwardOp {
  using scalar = T;
  static constexpr int kLen0 = N, kLen1 = packed_len(N), kLen2 = 1, kUse = 3, kOut = N;
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&x)[N], const T (&g)[kLen1], const T (&)[1], int, int, T (&out)[N]) {
    static_for<0, N>([&](auto I) {
      constexpr int i = I;
      T s = T(2) * g[i] * x[i];
      static_for<0, N>([&](auto J) {
        constexpr int j = J;
        if constexpr (j != i) s += g[pidx(N, i, j)] * x[j];
      });
      out[i] = s;
    });
  }
};

// Gradient of F = sym_to_full(p):  dp_ii = G_ii,  dp_ij = G_ij + G_ji      in0 = G (N x N row-major)
template <typename T, int N>
struct SymToFullBackwardOp {
  using scalar = T;
  static constexpr int kLen0 = N * N, kLen1 = 1, kLen2 = 1, kUse = 1, kOut = packed_len(N);
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&g)[kLen0], const T (&)[1], const T (&)[1], int, int, T (&out)[kOut]) {
    static_for<0, N>([&](auto I) {
      constexpr int i = I;
      out[i] = g[i * N + i];
      static_for<i + 1, N>([&](auto J) {
        constexpr int j = J;
        out[pidx(N, i, j)] = g[i * N + j] + g[j * N + i];
      });
    });
  }
};

template <typename T> struct OuterBwdBind { template <int N> using Op = SymOuterBackwardOp<T, N>; };
template <typename T> struct ToFullBwdBind { template <int N> using Op = SymToFullBackwardOp<T, N>; };

template <typename T>
int sym_outer_backward_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<OuterBwdBind<T>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template <typename T>
int sym_to_full_backward_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<ToFullBwdBind<T>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template int sym_outer_backward_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
template int sym_to_full_backward_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
#endif

}  // namespace nfm
