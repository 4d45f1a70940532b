// dense batched inverse / det / matvec / solve for one scalar type
// (-DNFM_SCALAR) and one part (-DNFM_PART)
#include <cstdlib>

#include "nfm_dense_ops.cuh"
#include "nfm_impl.cuh"
#include "nfm_sym_ops.cuh"

namespace nfm {

template <typename T, int ALGO> struct InvBind { template <int N> using Op = BatchInvOp<T, N, ALGO>; };
template <typename T> struct DetBind { template <int N> using Op = BatchDetOp<T, N>; };
template <typename T, bool TRANSPOSE> struct MvBind { template <int N> using Op = BatchMatvecOp<T, N, TRANSPOSE>; };
template <typename T, int ALGO> struct SolBind { template <int N> using Op = BatchSolveOp<T, N, ALGO>; };
template <typename T, int K, int ALGO> struct SolKBind { template <int N> using Op = BatchSolveKOp<T, N, K, ALGO>; };

#if NFM_PART == 0
template <typename T> struct InvPairBind { template <int N> using Op = BatchInvPairOp<T, N>; };
static bool pair_inverse_enabled() {  // NFM_DISABLE_PAIR_INVERSE=1: one thread per matrix for every order
  static const bool on = [] {
    const char* e = getenv("NFM_DISABLE_PAIR_INVERSE");
    return !(e && e[0] == '1');
  }();
  return on;
}
template <typename T>
int batch_inv_lu_impl(int n, const KParams& p, cudaStream_t s) {
  // fp64 orders 8..10: two lanes per matrix (the one-thread form is register-bound there)
  if constexpr (sizeof(T) == 8)
    if (n >= 8 && pair_inverse_enabled()) return DispatchN<InvPairBind<T>::template Op, 8, NFM_MAX_N>::run(n, p, s);
  return DispatchN<InvBind<T, NFM_ALGO_AUTO>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template int batch_inv_lu_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
// NFM_ALGO_LU for n <= 3: pivoted Gauss-Jordan instead of the closed forms (n >= 4 is the same kernel as AUTO)
template <typename T>
int batch_inv_lu_small_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<InvBind<T, NFM_ALGO_LU>::template Op, 1, 3>::run(n, p, s);
}
template int batch_inv_lu_small_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
#elif NFM_PART == 1
template <typename T>
int batch_inv_ldl_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<InvBind<T, NFM_ALGO_LDL>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template <typename T>
int batch_det_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<DetBind<T>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template <typename T>
int batch_matvec_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<MvBind<T, false>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template <typename T>
int batch_tmatvec_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<MvBind<T, true>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template int batch_tmatvec_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
template int batch_inv_ldl_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
template int batch_det_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
template int batch_matvec_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
#elif NFM_PART == 2
template <typename T>
int batch_solve_lu_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<SolBind<T, NFM_ALGO_LU>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template int batch_solve_lu_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
#elif NFM_PART == 3
template <typename T>
int batch_solve_ldl_impl(int n, const KParams& p, cudaStream_t s) {
  return DispatchN<SolBind<T, NFM_ALGO_LDL>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}
template int batch_solve_ldl_impl<NFM_SCALAR>(int, const KParams&, cudaStream_t);
#elif NFM_PART == 4
// 2..4 right-hand sides, pivoted LU
template <typename T>
int batch_solvek_lu_impl(int n, int k, const KParams& p, cudaStream_t s) {
  switch (k) {
    case 2: return DispatchN<SolKBind<T, 2, NFM_ALGO_LU>::template Op, 1, NFM_MAX_N>::run(n, p, s);
    case 3: return DispatchN<SolKBind<T, 3, NFM_ALGO_LU>::template Op, 1, NFM_MAX_N>::run(n, p, s);
    case 4: return DispatchN<SolKBind<T, 4, NFM_ALGO_LU>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  }
  return NFM_E_UNSUPPORTED;
}
template int batch_solvek_lu_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
#else
// 2..4 right-hand sides, LDL^T
template <typename T>
int batch_solvek_ldl_impl(int n, int k, const KParams& p, cudaStream_t s) {
  switch (k) {
    case 2: return DispatchN<SolKBind<T, 2, NFM_ALGO_LDL>::template Op, 1, NFM_MAX_N>::run(n, p, s);
    case 3: return DispatchN<SolKBind<T, 3, NFM_ALGO_LDL>::template Op, 1, NFM_MAX_N>::run(n, p, s);
    case 4: return DispatchN<SolKBind<T, 4, NFM_ALGO_LDL>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  }
  return NFM_E_UNSUPPORTED;
}
template int batch_solvek_ldl_impl<NFM_SCALAR>(int, int, const KParams&, cudaStream_t);
#endif

}  // namespace nfm
