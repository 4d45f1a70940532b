// nfm_extra.cu -- the remaining public names of nitorch_fastmath/sym.py:29
// (SURVEY.md section 8f "next" rows): sym_det, sym_to_full, sym_outer.
#include "nfm_dense_ops.cuh"
#include "nfm_impl.cuh"
#include "nfm_pipeline.cuh"
#include "nfm_sym_ops.cuh"

namespace nfm {

// det of a packed symmetric matrix (_impl/sym.py:401-452): closed form for
// N <= 4, pivoted LU of the expansion above (the reference calls torch.det).
template <typename T, int N>
struct SymDetOp {
  using scalar = T;
  static constexpr int kLen0 = packed_len(N), kLen1 = 1, kLen2 = 1, kUse = 1, kOut = 1;
  static constexpr bool kHeavy = N > 4;
  __device__ static __forceinline__ void apply(const T (&m)[kLen0], const T (&)[1], const T (&)[1], int, int, T (&out)[1]) {
    if constexpr (N <= 4) {
      out[0] = sym_det_closed<T, N>(m);
    } else {
      GaussPP<T, N, 0> g;
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = m[pidx(N, i, j)];
      g.eliminate();
      out[0] = g.det();
    }
  }
};

// packed -> dense (_impl/sym.py:16-60)
template <typename T, int N>
struct SymToFullOp {
  using scalar = T;
  static constexpr int kLen0 = packed_len(N), kLen1 = 1, kLen2 = 1, kUse = 1, kOut = N * N;
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&m)[kLen0], const T (&)[1], const T (&)[1], int, int, T (&out)[kOut]) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = 0; j < N; ++j) out[i * N + j] = m[pidx(N, i, j)];
  }
};

// x x^T packed (_impl/sym.py:496-528)
template <typename T, int N>
struct SymOuterOp {
  using scalar = T;
  static constexpr int kLen0 = N, kLen1 = 1, kLen2 = 1, kUse = 1, kOut = packed_len(N);
  static constexpr bool kHeavy = false;
  __device__ static __forceinline__ void apply(const T (&x)[N], const T (&)[1], const T (&)[1], int, int, T (&out)[kOut]) {
#pragma unroll
    for (int i = 0; i < N; ++i)
#pragma unroll
      for (int j = i; j < N; ++j) out[pidx(N, i, j)] = x[i] * x[j];
  }
};

template <typename T> struct SDetBind { template <int N> using Op = SymDetOp<T, N>; };
template <typename T> struct SFullBind { template <int N> using Op = SymToFullOp<T, N>; };
template <typename T> struct SOuterBind { template <int N> using Op = SymOuterOp<T, N>; };

template <template <typename> class Bind>
static int unary_entry(int dtype, int n, i64 batch, const void* in, i64 in_stride, void* out, i64 out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) { set_error("dtype must be NFM_F32 or NFM_F64"); return NFM_E_UNSUPPORTED; }
  if (n < 1 || n > NFM_MAX_N) { set_error("matrix order must be in 1..10"); return NFM_E_UNSUPPORTED; }
  if (batch < 0 || in == nullptr || out == nullptr || in_stride < 0 || out_stride < 0) { set_error("bad argument"); return NFM_E_BADARG; }
  KParams p{};
  p.in[0].ptr = in;
  p.in[0].stride = in_stride;
  p.present = 1;
  p.out = out;
  p.out_stride = out_stride;
  p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  if (dtype == NFM_F32) return DispatchN<Bind<float>::template Op, 1, NFM_MAX_N>::run(n, p, s);
  return DispatchN<Bind<double>::template Op, 1, NFM_MAX_N>::run(n, p, s);
}

}  // namespace nfm

using namespace nfm;

extern "C" {

int nfm_sym_det(int dtype, int n, int64_t batch, const void* mat, int64_t mat_stride, void* out, int64_t out_stride, void* stream) {
  return unary_entry<SDetBind>(dtype, n, batch, mat, mat_stride, out, out_stride, stream);
}
int nfm_sym_to_full(int dtype, int n, int64_t batch, const void* mat, int64_t mat_stride, void* out, int64_t out_stride, void* stream) {
  return unary_entry<SFullBind>(dtype, n, batch, mat, mat_stride, out, out_stride, stream);
}
int nfm_sym_outer(int dtype, int n, int64_t batch, const void* vec, int64_t vec_stride, void* out, int64_t out_stride, void* stream) {
  return unary_entry<SOuterBind>(dtype, n, batch, vec, vec_stride, out, out_stride, stream);
}

int nfm_sym_matmul(int dtype, int k, int d, int mode, int64_t batch, const void* jac, int64_t jac_stride, const void* hess,
                   int64_t hess_stride, void* out, int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) { set_error("dtype must be NFM_F32 or NFM_F64"); return NFM_E_UNSUPPORTED; }
  if (k < 1 || k > NFM_MAX_N || d < 1 || d > NFM_MAX_N || (mode != 0 && mode != 1) || (mode == 1 && k != d)) {
    set_error("sym_matmul: 1 <= k, d <= 10; mode 1 needs k == d");
    return NFM_E_UNSUPPORTED;
  }
  if (batch < 0 || !jac || !hess || !out || jac_stride < 0 || hess_stride < 0 || out_stride < 0) { set_error("bad argument"); return NFM_E_BADARG; }
  auto st = static_cast<cudaStream_t>(stream);
  if (!fused_shape_built(k, d) || (mode == 1 && k > 3)) {  // run-time-sized kernel beyond the templated shapes
    t_last_path_tma = 0;
    reset_launch_record();
    const int rc = dtype == NFM_F32 ? sym_matmul_rt<float>(k, d, mode, batch, jac, jac_stride, hess, hess_stride, out, out_stride, st)
                                    : sym_matmul_rt<double>(k, d, mode, batch, jac, jac_stride, hess, hess_stride, out, out_stride, st);
    if (rc) set_error("sym_matmul kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
    return rc;
  }
  KParams p{};
  p.in[0].ptr = jac;
  p.in[0].stride = jac_stride;
  p.in[1].ptr = hess;
  p.in[1].stride = hess_stride;
  p.present = 3;
  p.out = out;
  p.out_stride = out_stride;
  p.batch = batch;
  return dtype == NFM_F32 ? sym_matmul_impl<float>(k, d, mode, p, st) : sym_matmul_impl<double>(k, d, mode, p, st);
}

int nfm_sym_matmul_solve(int dtype, int k, int d, int mode, int64_t batch, const void* jac, int64_t jac_stride, const void* hess,
                         int64_t hess_stride, const void* grad, int64_t grad_stride, const void* diag, int64_t diag_stride,
                         void* out, int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) { set_error("dtype must be NFM_F32 or NFM_F64"); return NFM_E_UNSUPPORTED; }
  if (!fused_shape_built(k, d) || (mode != 0 && mode != 1) || (mode == 1 && (k != d || k > 3))) {
    set_error("sym_matmul_solve: 1 <= k, d <= 6, or k <= 10 with d <= 3; mode 1 needs k == d <= 3");
    return NFM_E_UNSUPPORTED;
  }
  if (batch < 0 || !jac || !hess || !grad || !out || jac_stride < 0 || hess_stride < 0 || grad_stride < 0 || diag_stride < 0 ||
      out_stride < 0) {
    set_error("bad argument");
    return NFM_E_BADARG;
  }
  KParams p{};
  p.in[0].ptr = jac;
  p.in[0].stride = jac_stride;
  p.in[1].ptr = hess;
  p.in[1].stride = hess_stride;
  p.in[2].ptr = grad;
  p.in[2].stride = grad_stride;
  p.present = 7;
  if (diag != nullptr) {
    p.in[3].ptr = diag;
    p.in[3].stride = diag_stride;
    p.present |= 8;
  }
  p.out = out;
  p.out_stride = out_stride;
  p.batch = batch;
  auto st = static_cast<cudaStream_t>(stream);
  return dtype == NFM_F32 ? sym_matmul_solve_impl<float>(k, d, mode, p, st) : sym_matmul_solve_impl<double>(k, d, mode, p, st);
}

int nfm_sym_solve_update_reg(int dtype, int n, int algo, int64_t batch, const void* mat, int64_t mat_stride, const void* vec,
                             int64_t vec_stride, const void* x, int64_t x_stride, const void* diag, int64_t diag_stride, double lam,
                             double alpha, void* out, int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) { set_error("dtype must be NFM_F32 or NFM_F64"); return NFM_E_UNSUPPORTED; }
  if (n < 1 || n > NFM_MAX_N) { set_error("matrix order must be in 1..10"); return NFM_E_UNSUPPORTED; }
  if (algo != NFM_ALGO_AUTO && algo != NFM_ALGO_LDL) { set_error("sym_solve_update: algo must be AUTO or LDL"); return NFM_E_UNSUPPORTED; }
  if (batch < 0 || !mat || !vec || !x || !out || mat_stride < 0 || vec_stride < 0 || x_stride < 0 || diag_stride < 0 || out_stride < 0) {
    set_error("bad argument");
    return NFM_E_BADARG;
  }
  KParams p{};
  p.in[0].ptr = mat;
  p.in[0].stride = mat_stride;
  p.in[1].ptr = vec;
  p.in[1].stride = vec_stride;
  p.in[2].ptr = x;
  p.in[2].stride = x_stride;
  p.present = 7;
  if (diag != nullptr) {
    p.in[3].ptr = diag;
    p.in[3].stride = diag_stride;
    p.present |= 8;
  }
  p.out = out;
  p.out_stride = out_stride;
  p.batch = batch;
  p.scal0 = lam;
  p.scal1 = alpha;
  auto s = static_cast<cudaStream_t>(stream);
  return dtype == NFM_F32 ? sym_solve_update_impl<float>(n, algo, p, s) : sym_solve_update_impl<double>(n, algo, p, s);
}

int nfm_sym_solve_update(int dtype, int n, int algo, int64_t batch, const void* mat, int64_t mat_stride, const void* vec,
                         int64_t vec_stride, const void* x, int64_t x_stride, double lam, double alpha, void* out,
                         int64_t out_stride, void* stream) {
  return nfm_sym_solve_update_reg(dtype, n, algo, batch, mat, mat_stride, vec, vec_stride, x, x_stride, nullptr, 0, lam, alpha, out,
                                  out_stride, stream);
}

}  // extern "C"
