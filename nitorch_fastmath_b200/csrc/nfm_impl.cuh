// nfm_impl.cuh -- typed implementation entry points.  Each family source
// (nfm_sym_matvec.cu, nfm_sym_solve.cu, ...) is compiled once per scalar type
// (-DNFM_SCALAR=float|double) and, for the big families, once per part
// (-DNFM_PART=k) so the build parallelises; nfm_entry.cu holds the C ABI.
#pragma once

#include "nfm_common.cuh"

namespace nfm {

template <typename T> int sym_matvec_impl(int n, int layout, const KParams& p, cudaStream_t s);

// sym_solve: part 0 = layouts E, D, F and packed N <= 4 (closed forms);
// part 1 = packed N 5..10 LDL^T; part 2 = packed N 5..10 pivoted LU;
// part 3 = packed N 5..10 AUTO (checked LDL^T with per-matrix LU fallback)
template <typename T> int sym_solve_part0(int n, int layout, const KParams& p, cudaStream_t s);
template <typename T> int sym_solve_part1(int n, const KParams& p, cudaStream_t s);
template <typename T> int sym_solve_part2(int n, const KParams& p, cudaStream_t s);
template <typename T> int sym_solve_part3(int n, const KParams& p, cudaStream_t s);

// NFM_ALGO_WARP: sub-warp cooperative shuffle solve, packed N 5..10 (nfm_sym_warp.cu)
template <typename T> int sym_solve_warp(int n, const KParams& p, cudaStream_t s);

// sym_invert: part 0 = N <= 4 closed form + N 5..10 LDL^T; part 1 = N 5..10 pivoted LU;
// part 2 = N 5..10 AUTO (checked LDL^T with per-matrix Gauss-Jordan fallback)
template <typename T> int sym_invert_part0(int n, int diag_only, const KParams& p, cudaStream_t s);
template <typename T> int sym_invert_part1(int n, int diag_only, const KParams& p, cudaStream_t s);
template <typename T> int sym_invert_part2(int n, int diag_only, const KParams& p, cudaStream_t s);

// backward kernels (nfm_sym_grad.cu): sign * S(u, w) in layout E / D / S, gradient of
// sym_invert (packed or diagonal-only) and of sym_det with respect to the packed coefficients
template <typename T> int sym_outer2_impl(int n, int layout, const KParams& p, cudaStream_t s);
template <typename T> int sym_invert_backward_impl(int n, int diag_only, const KParams& p, cudaStream_t s);
template <typename T> int sym_det_backward_impl(int n, const KParams& p, cudaStream_t s);

// dense: part 0 = inverse (closed / Gauss-Jordan), part 1 = inverse (LDL^T) + det + matvec,
// part 2 = solve LU, part 3 = solve LDL^T
template <typename T> int batch_inv_lu_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int batch_inv_lu_small_impl(int n, const KParams& p, cudaStream_t s);  // NFM_ALGO_LU, n <= 3
template <typename T> int batch_inv_ldl_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int batch_det_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int batch_matvec_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int batch_solve_lu_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int batch_solve_ldl_impl(int n, const KParams& p, cudaStream_t s);
// parts 4 / 5: 2..4 right-hand sides (register kernels); more go to the run-time-sized kernel
template <typename T> int batch_solvek_lu_impl(int n, int k, const KParams& p, cudaStream_t s);
template <typename T> int batch_solvek_ldl_impl(int n, int k, const KParams& p, cudaStream_t s);
template <typename T> int batch_tmatvec_impl(int n, const KParams& p, cudaStream_t s);  // part 1: y = A^T v

// backward kernels of the dense routines (nfm_dense_grad.cu): part 0 = inverse and determinant
// gradients; parts 1 / 2 = sign * U W^T or U^T W (optionally symmetrised) for k = 1..2 / 3..4
template <typename T> int batch_inv_backward_impl(int n, int sym, const KParams& p, cudaStream_t s);
template <typename T> int batch_det_backward_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int batch_outer_k12_impl(int n, int k, const KParams& p, cudaStream_t s);
template <typename T> int batch_outer_k34_impl(int n, int k, const KParams& p, cudaStream_t s);

// run-time-sized fallbacks (nfm_generic.cu)
// (trans: y = A^T v; out = sign * U W^T or U^T W (rows), optionally symmetrised, for k > 4 / m != n)
template <typename T>
int batch_matvec_rt(int m, int n, int trans, i64 batch, const void* mat, i64 ms, const void* vec, i64 vs, void* out, i64 os,
                    cudaStream_t s);
template <typename T>
int batch_outer_rt(int m, int n, int k, int rows, int sym, int sign, i64 batch, const void* u, i64 us, const void* w, i64 ws,
                   void* out, i64 os, cudaStream_t s);

// nfm_fused.cu: register kernels for 1 <= k, d <= 6 and for tall Jacobians k <= 10, d <= 3
constexpr int kFusedMaxOrder = 6;
constexpr bool fused_shape_built(int k, int d) {
  return k >= 1 && d >= 1 && ((k <= kFusedMaxOrder && d <= kFusedMaxOrder) || (k <= NFM_MAX_N && d <= 3));
}
template <typename T> int sym_matmul_impl(int k, int d, int mode, const KParams& p, cudaStream_t s);
template <typename T> int sym_matmul_solve_impl(int k, int d, int mode, const KParams& p, cudaStream_t s);
template <typename T> int sym_solve_update_impl(int n, int algo, const KParams& p, cudaStream_t s);

// backward kernels of the Gauss-Newton builders (nfm_gn_grad.cu): sym_matmul for the shapes of
// fused_shape_built (WHICH 1 = dJ, 2 = dH, 3 = both in one record; parts 0 / 1 / 2), sym_outer and
// sym_to_full (part 3)
template <typename T, int WHICH> int sym_matmul_backward_impl(int k, int d, int mode, const KParams& p, cudaStream_t s);
template <typename T> int sym_outer_backward_impl(int n, const KParams& p, cudaStream_t s);
template <typename T> int sym_to_full_backward_impl(int n, const KParams& p, cudaStream_t s);

// nrhs > 4 and right division: register factorisation (order templated), run-time loop over
// the right-hand sides (nfm_generic.cu)
template <typename T>
int batch_solve_many(int n, int nrhs, int chol, int right, i64 batch, const void* a, i64 as, const void* b, i64 bs, void* out,
                     i64 os, cudaStream_t s);

template <typename T>
int sym_matmul_rt(int k, int d, int mode, i64 batch, const void* jac, i64 js, const void* hess, i64 hs, void* out, i64 os,
                  cudaStream_t s);
// the gradient of sym_matmul for the other shapes (records as SymMatmulBackwardOp)
template <typename T>
int sym_matmul_backward_rt(int k, int d, int mode, int which, i64 batch, const void* jac, i64 js, const void* hess, i64 hs,
                           const void* grad, i64 gs, void* out, i64 os, cudaStream_t s);

}  // namespace nfm
