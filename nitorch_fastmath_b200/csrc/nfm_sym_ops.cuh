// nfm_sym_ops.cuh -- Op structs (see nfm_pipeline.cuh) for the packed-symmetric
// routines: matvec / addmatvec / submatvec, solve, invert.
#pragma once

#include "nfm_dense_math.cuh"
#include "nfm_pipeline.cuh"
#include "nfm_sym_math.cuh"

namespace nfm {

__host__ __device__ constexpr int layout_len(int layout, int n) {
  return layout == NFM_LAYOUT_SCALED_IDENTITY ? 1
         : layout == NFM_LAYOUT_DIAG          ? n
         : layout == NFM_LAYOUT_SYM           ? packed_len(n)
                                              : n * n;
}

constexpr int kFlagSubtract = 1;  // matvec: out = inp - A v

__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }

// out = [inp +/-] A v        in0 = mat, in1 = vec, in2 = inp (optional)
template <typename T, int N, int LAYOUT>
struct SymMatvecOp {
  using scalar = T;
  static constexpr int kLen0 = layout_len(LAYOUT, N);
  static constexpr int kLen1 = N;
  static constexpr int kLen2 = N;
  static constexpr int kUse = 7;
  static constexpr int kOut = N;
  static constexpr bool kHeavy = false;

  __device__ static __forceinline__ void apply(const T (&m)[kLen0], const T (&v)[N], const T (&inp)[N], int present,
                                               int flags, T (&out)[N]) {
    T y[N];
    if constexpr (LAYOUT == NFM_LAYOUT_SCALED_IDENTITY) {
#pragma unroll
      for (int i = 0; i < N; ++i) y[i] = m[0] * v[i];
    } else if constexpr (LAYOUT == NFM_LAYOUT_DIAG) {
#pragma unroll
      for (int i = 0; i < N; ++i) y[i] = m[i] * v[i];
    } else if constexpr (LAYOUT == NFM_LAYOUT_SYM) {
      sym_matvec_reg<T, N>(m, v, y);
    } else {
      dense_matvec_reg<T, N, N>(m, v, y);
    }
    if (present & 4) {
      // the addend is added to the rounded product by an add the compiler may not fuse: left to
      // it, `inp + m v` became an FMA in some tile geometries and not in others (diagonal layout,
      // fp32 order 6, fp64 order 3), so one call gave other bits above the large-batch switch
      const bool sub = flags & kFlagSubtract;
#pragma unroll
      for (int i = 0; i < N; ++i) out[i] = sub ? sub_rn(inp[i], y[i]) : add_rn(inp[i], y[i]);
    } else {
#pragma unroll
      for (int i = 0; i < N; ++i) out[i] = y[i];
    }
  }
};

// x = (A + diag(d))^-1 v      in0 = mat, in1 = vec, in2 = d (optional)
template <typename T, int N, int LAYOUT, int ALGO>
struct SymSolveOp {
  using scalar = T;
  static constexpr int kLen0 = layout_len(LAYOUT, N);
  static constexpr int kLen1 = N;
  static constexpr int kLen2 = N;
  static constexpr int kUse = 7;
  static constexpr int kOut = N;
  static constexpr bool kHeavy = (LAYOUT == NFM_LAYOUT_SYM && N > 4 && ALGO == NFM_ALGO_LU) || (LAYOUT == NFM_LAYOUT_FULL && N >= 2);

  __device__ static __forceinline__ void apply(const T (&m_in)[kLen0], const T (&v)[N], const T (&reg)[N],
                                               int present, int flags, T (&x)[N]) {
    if constexpr (LAYOUT == NFM_LAYOUT_SCALED_IDENTITY) {
#pragma unroll
      for (int i = 0; i < N; ++i) x[i] = v[i] / (m_in[0] + reg[i]);
    } else if constexpr (LAYOUT == NFM_LAYOUT_DIAG) {
#pragma unroll
      for (int i = 0; i < N; ++i) x[i] = v[i] / (m_in[i] + reg[i]);
    } else if constexpr (LAYOUT == NFM_LAYOUT_SYM) {
      T m[kLen0];
#pragma unroll
      for (int k = 0; k < kLen0; ++k) m[k] = (k < N) ? m_in[k] + reg[k < N ? k : 0] : m_in[k];
      if constexpr (N <= 4) {
        sym_solve_closed<T, N>(m, v, x);
      } else if constexpr (ALGO == NFM_ALGO_LU) {
        sym_solve_lu<T, N>(m, v, x);
      } else if constexpr (ALGO == NFM_ALGO_LDL) {
        LDL<T, N> f;
        f.load_packed(m);
        f.factor();
        f.solve(v, x);
      } else {
        // NFM_ALGO_AUTO: LDL^T with a pivot check; the rare matrix that fails
        // it (indefinite / tiny pivot) is redone with pivoted LU
        LDL<T, N> f;
        f.load_packed(m);
        if (f.factor_checked()) f.solve(v, x);
        else sym_solve_lu<T, N>(m, v, x);
      }
    } else {
      GaussPP<T, N, 1> g;
#pragma unroll
      for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = m_in[i * N + j] + (i == j ? reg[i] : T(0));
        g.b[i][0] = v[i];
      }
      g.eliminate();
      g.back_substitute();
#pragma unroll
      for (int i = 0; i < N; ++i) x[i] = g.b[i][0];
    }
  }
};

// Fused Gauss-Newton / Levenberg-Marquardt step (SURVEY.md section 8f rank 4):
//   out = x - alpha * (A + lam I + diag(d))^-1 v     in0 = mat (packed), in1 = v, in2 = x, in3 = d (optional)
// i.e. sym_solve_ with a scalar and / or per-voxel regulariser (the reference's
// documented regulariser, _impl/sym.py:356-357) followed by the update of the
// parameter field, without the round trip of the step through HBM.
template <typename T, int N, int ALGO>
struct SymSolveUpdateOp {
  using scalar = T;
  static constexpr int kLen0 = packed_len(N);
  static constexpr int kLen1 = N;
  static constexpr int kLen2 = N;
  static constexpr int kLen3 = N;
  static constexpr int kUse = 15;
  static constexpr int kOut = N;
  static constexpr bool kHeavy = false;
  static constexpr bool kScalars = true;
  static constexpr bool kThreeMandatory = true;

  __device__ static __forceinline__ void apply(const T (&m_in)[kLen0], const T (&v)[N], const T (&x0)[N], const T (&reg)[N],
                                               int present, int flags, T lam, T alpha, T (&out)[N]) {
    T m[kLen0];
#pragma unroll
    for (int k = 0; k < kLen0; ++k) m[k] = (k < N) ? m_in[k] + (lam + reg[k < N ? k : 0]) : m_in[k];
    T step[N];
    if constexpr (N <= 4) {
      sym_solve_closed<T, N>(m, v, step);
    } else if constexpr (ALGO == NFM_ALGO_LDL) {
      LDL<T, N> f;
      f.load_packed(m);
      f.factor();
      f.solve(v, step);
    } else {
      LDL<T, N> f;
      f.load_packed(m);
      if (f.factor_checked()) f.solve(v, step);
      else sym_solve_lu<T, N>(m, v, step);
    }
#pragma unroll
    for (int i = 0; i < N; ++i) out[i] = x0[i] - alpha * step[i];
  }
};

// J^T H J (MODE 0) or J H J^T (MODE 1, K == D) in packed order; the register
// kernel behind sym_matmul and the fused Gauss-Newton solve below
// (_impl/sym.py:532-670)
template <typename T, int K, int D, int MODE>
__device__ __forceinline__ void sym_jhj(const T (&j)[K * D], const T (&h)[packed_len(MODE == 0 ? K : D)],
                                        T (&out)[packed_len(MODE == 0 ? D : K)]) {
  constexpr int HN = MODE == 0 ? K : D;  // order of H
  constexpr int ON = MODE == 0 ? D : K;  // order of the result
  // G = J as (ON x HN) "rows = output index": mode 0 uses J^T, mode 1 uses J
  T hj[HN][ON];  // H * G^T
#pragma unroll
  for (int a = 0; a < HN; ++a)
#pragma unroll
    for (int o = 0; o < ON; ++o) {
      T s = T(0);
#pragma unroll
      for (int b = 0; b < HN; ++b) {
        const T g = MODE == 0 ? j[b * D + o] : j[o * D + b];
        s += h[pidx(HN, a, b)] * g;
      }
      hj[a][o] = s;
    }
#pragma unroll
  for (int o = 0; o < ON; ++o)
#pragma unroll
    for (int q = o; q < ON; ++q) {
      T s = T(0);
#pragma unroll
      for (int a = 0; a < HN; ++a) {
        const T g = MODE == 0 ? j[a * D + o] : j[o * D + a];
        s += g * hj[a][q];
      }
      out[pidx(ON, o, q)] = s;
    }
}

// Fused Gauss-Newton system (SURVEY.md section 8f rank 1): the packed Hessian
// J^T H J (+ diag(d)) is built in registers and solved at once,
//   x = (J^T H J + diag(d))^-1 g      in0 = J (K x D), in1 = H (packed), in2 = g, in3 = d (optional)
// so the 6- / 21-coefficient Hessian field never goes to HBM and back
// (reference chain: sym_matmul _impl/sym.py:637-670, then sym_solve :327-398).
template <typename T, int K, int D, int MODE>
struct SymMatmulSolveOp {
  using scalar = T;
  static constexpr int kHN = MODE == 0 ? K : D;
  static constexpr int kON = MODE == 0 ? D : K;
  static constexpr int kLen0 = K * D;
  static constexpr int kLen1 = packed_len(kHN);
  static constexpr int kLen2 = kON;
  static constexpr int kLen3 = kON;
  static constexpr int kUse = 15;
  static constexpr int kOut = kON;
  static constexpr bool kHeavy = false;
  static constexpr bool kThreeMandatory = true;

  __device__ static __forceinline__ void apply(const T (&j)[kLen0], const T (&h)[kLen1], const T (&g)[kON], const T (&reg)[kON],
                                               int present, int flags, T (&x)[kON]) {
    T a[packed_len(kON)];
    sym_jhj<T, K, D, MODE>(j, h, a);
#pragma unroll
    for (int i = 0; i < kON; ++i) a[i] += reg[i];
    if constexpr (kON <= 4) {
      sym_solve_closed<T, kON>(a, g, x);
    } else {
      LDL<T, kON> f;
      f.load_packed(a);
      if (f.factor_checked()) f.solve(g, x);
      else sym_solve_lu<T, kON>(a, g, x);
    }
  }
};

// out = A^-1 (packed) or diag(A^-1)        in0 = mat
template <typename T, int N, int ALGO, bool DIAG_ONLY>
struct SymInvertOp {
  using scalar = T;
  static constexpr int kLen0 = packed_len(N);
  static constexpr int kLen1 = 1;
  static constexpr int kLen2 = 1;
  static constexpr int kUse = 1;
  static constexpr int kOut = DIAG_ONLY ? N : packed_len(N);
  static constexpr bool kHeavy = N > 4 && ALGO == NFM_ALGO_LU;

  __device__ static __forceinline__ void apply(const T (&m)[kLen0], const T (&)[1], const T (&)[1], int present,
                                               int flags, T (&out)[kOut]) {
    if constexpr (N <= 4) {
      // reference: N solves against unit vectors = adjugate columns / det
      T adj[kLen0];
      const T det = sym_adjugate<T, N>(m, adj);
      if constexpr (N == 4 || sizeof(T) == 8) {
        const T rdet = T(1) / det;
#pragma unroll
        for (int k = 0; k < kOut; ++k) out[k] = adj[k] * rdet;
      } else {
#pragma unroll
        for (int k = 0; k < kOut; ++k) out[k] = adj[k] / det;
      }
    } else if constexpr (ALGO == NFM_ALGO_LU) {
      // in-place Gauss-Jordan with partial pivoting on the expanded matrix
      GaussJordan<T, N> g;
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = 0; j < N; ++j) g.a[i][j] = m[pidx(N, i, j)];
      g.invert();
#pragma unroll
      for (int i = 0; i < N; ++i)
#pragma unroll
        for (int j = i; j < N; ++j) {
          if (DIAG_ONLY && j != i) continue;
          // reference takes entry (j, i) of solve(A, e_i): column i, row j >= i
          out[DIAG_ONLY ? i : pidx(N, i, j)] = g.a[j][i];
        }
    } else if constexpr (ALGO == NFM_ALGO_LDL) {
      LDL<T, N> f;
      f.load_packed(m);
      f.factor();
      f.template invert<DIAG_ONLY>(out);
    } else {
      // NFM_ALGO_AUTO: checked LDL^T, pivoted Gauss-Jordan for the matrices that fail
      LDL<T, N> f;
      f.load_packed(m);
      if (f.factor_checked()) {
        f.template invert<DIAG_ONLY>(out);
      } else {
        GaussJordan<T, N> g;
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = 0; j < N; ++j) g.a[i][j] = m[pidx(N, i, j)];
        g.invert();
#pragma unroll
        for (int i = 0; i < N; ++i)
#pragma unroll
          for (int j = i; j < N; ++j) {
            if (DIAG_ONLY && j != i) continue;
            out[DIAG_ONLY ? i : pidx(N, i, j)] = g.a[j][i];
          }
      }
    }
  }
};

// ---------------------------------------------------------------------------
// run-time -> compile-time dispatch over N
// ---------------------------------------------------------------------------
template <template <int> class OpN, int N_LO, int N_HI>
struct DispatchN {
  static int run(int n, const KParams& p, cudaStream_t s) {
    if (n == N_LO) return run_op<OpN<N_LO>>(p, s);
    if constexpr (N_LO < N_HI) return DispatchN<OpN, N_LO + 1, N_HI>::run(n, p, s);
    else return NFM_E_UNSUPPORTED;
  }
};

}  // namespace nfm
