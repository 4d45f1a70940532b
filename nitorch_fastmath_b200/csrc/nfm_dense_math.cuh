// nfm_dense_math.cuh -- per-matrix register math for dense row-major n x n
// matrices: matvec, closed-form det / inverse for n <= 3 (the reference's
// TorchScript closed forms, _impl/batched.py:22-32, :67-98), in-place
// Gauss-Jordan inverse with partial pivoting above.
#pragma once

#include "nfm_common.cuh"
#include "nfm_sym_math.cuh"

namespace nfm {

template <typename T, int M, int N>
__device__ __forceinline__ void dense_matvec_reg(const T (&a)[M * N], const T (&v)[N], T (&y)[M]) {
  // left-to-right accumulation, as matvec1/2/3 (_impl/batched.py:134-151)
#pragma unroll
  for (int i = 0; i < M; ++i) {
    T s = a[i * N] * v[0];
#pragma unroll
    for (int j = 1; j < N; ++j) s += a[i * N + j] * v[j];
    y[i] = s;
  }
}

template <typename T>
__device__ __forceinline__ T dense_det2(const T* a) { return a[0] * a[3] - a[1] * a[2]; }

template <typename T>
__device__ __forceinline__ T dense_det3(const T* a) {
  // _impl/batched.py:27-32
  return a[0] * (a[4] * a[8] - a[5] * a[7]) + a[1] * (a[5] * a[6] - a[3] * a[8]) + a[2] * (a[3] * a[7] - a[4] * a[6]);
}

// max|a| - min|a| over the entries: the reference's determinant regulariser
// scale (_impl/batched.py:74-76, :94-96)
template <typename T, int L>
__device__ __forceinline__ T abs_range(const T (&a)[L]) {
  T hi = tabs(a[0]), lo = hi;
#pragma unroll
  for (int k = 1; k < L; ++k) {
    const T c = tabs(a[k]);
    hi = c > hi ? c : hi;
    lo = c < lo ? c : lo;
  }
  return hi - lo;
}

// closed-form inverse n = 1..3; `regularise` adds range * 1e-12 to the determinant
template <typename T, int N>
__device__ __forceinline__ void dense_inv_closed(const T (&a)[N * N], bool regularise, T (&f)[N * N]) {
  static_assert(N >= 1 && N <= 3, "closed forms cover n = 1..3");
  if constexpr (N == 1) {
    f[0] = T(1) / a[0];  // reciprocal, _impl/batched.py:128
  } else if constexpr (N == 2) {
    T dt = dense_det2(a);
    if (regularise) dt += abs_range(a) * T(1e-12);
    const T r = T(1) / dt;  // one division; the reference divides every cofactor (<= 1 ulp apart)
    f[0] = a[3] * r;
    f[1] = -a[1] * r;
    f[2] = -a[2] * r;
    f[3] = a[0] * r;
  } else {
    T dt = dense_det3(a);
    if (regularise) dt += abs_range(a) * T(1e-12);
    const T r = T(1) / dt;
    f[0] = (a[4] * a[8] - a[5] * a[7]) * r;
    f[1] = (a[2] * a[7] - a[1] * a[8]) * r;
    f[2] = (a[1] * a[5] - a[2] * a[4]) * r;
    f[3] = (a[5] * a[6] - a[3] * a[8]) * r;
    f[4] = (a[0] * a[8] - a[2] * a[6]) * r;
    f[5] = (a[3] * a[2] - a[5] * a[0]) * r;
    f[6] = (a[7] * a[3] - a[6] * a[4]) * r;
    f[7] = (a[6] * a[1] - a[7] * a[0]) * r;
    f[8] = (a[0] * a[4] - a[1] * a[3]) * r;
  }
}

// in-place Gauss-Jordan inverse with partial (row) pivoting.  N*N registers.
// invert<true>() also returns det A (product of the pivots, sign of the row exchanges): the
// determinant backward gets both from one elimination.  invert<false>() returns 1.
template <typename T, int N>
struct GaussJordan {
  T a[N][N];

  template <bool DET = false>
  __device__ __forceinline__ T invert() {
    T det = T(1);
    int piv[N];
    static_for<0, N>([&](auto K) {
      constexpr int k = K;
      T best = tabs(a[k][k]);
      int p = k;
      static_for<k + 1, N>([&](auto I) {
        constexpr int i = I;
        const T c = tabs(a[i][k]);
        if (c > best) {
          best = c;
          p = i;
        }
      });
      piv[k] = p;
      if (N < kVoteFromOrder || warp_any(p != k)) {  // skipped when no matrix of the warp exchanges rows in this step
        static_for<k + 1, N>([&](auto I) {
          constexpr int i = I;
          const bool sw = (p == i);
          static_for<0, N>([&](auto J) {
            constexpr int j = J;
            const T lo = a[k][j], hi = a[i][j];
            a[k][j] = sw ? hi : lo;
            a[i][j] = sw ? lo : hi;
          });
        });
      }
      if constexpr (DET) det *= (p != k) ? -a[k][k] : a[k][k];
      const T rp = T(1) / a[k][k];
      a[k][k] = T(1);
      static_for<0, N>([&](auto J) { a[k][J] *= rp; });
      static_for<0, N>([&](auto I) {
        constexpr int i = I;
        if constexpr (i != k) {
          const T f = a[i][k];
          a[i][k] = T(0);
          static_for<0, N>([&](auto J) {
            constexpr int j = J;
            a[i][j] -= f * a[k][j];
          });
        }
      });
    });
    // (P A)^-1 = A^-1 P^T  ->  undo with column swaps in reverse order
    static_for_down<0, N>([&](auto K) {
      constexpr int k = K;
      if (N < kVoteFromOrder || warp_any(piv[k] != k)) {
        static_for<k + 1, N>([&](auto C) {
          constexpr int c = C;
          const bool sw = (piv[k] == c);
          static_for<0, N>([&](auto I) {
            constexpr int i = I;
            const T lo = a[i][k], hi = a[i][c];
            a[i][k] = sw ? hi : lo;
            a[i][c] = sw ? lo : hi;
          });
        });
      }
    });
    return det;
  }
};

// The same elimination with TWO lanes per matrix (lanes 2m and 2m+1 of a warp): lane h holds the
// columns [h*CH, h*CH + CH) of every row, CH = ceil(N / 2) -- half the registers, half the chain.
// Columns are the natural cut: the pivot search of step k runs inside ONE lane (the owner of column
// k, known at compile time), row exchanges and the elimination touch each lane's own columns only,
// and what crosses lanes per step is the pivot row index, 1 / pivot and the N multipliers of column
// k (shuffles from the owner).  The final column un-permutation costs nothing: each lane tracks
// where its columns end up and stores them there.  Element for element the arithmetic is that of
// GaussJordan<T, N>::invert(), so the results are bit-identical.
template <typename T, int N>
struct GaussJordanPair {
  static constexpr int CH = (N + 1) / 2;

  // `rec`: the row-major N x N record in shared memory (read, then overwritten with the inverse);
  // every lane of the warp must call this (shuffles with a full mask)
  __device__ static __forceinline__ void invert_in_place(T* rec, int lane) {
    const int h = lane & 1, c0 = h * CH, pair0 = lane & ~1;
    T a[N][CH];
    static_for<0, N>([&](auto I) {
      static_for<0, CH>([&](auto J) {
        constexpr int i = I, jl = J;
        a[i][jl] = (N % 2 == 0 || c0 + jl < N) ? rec[i * N + c0 + jl] : T(0);  // odd N: the last slot of lane 1 is padding
      });
    });
    __syncwarp();  // both lanes of every pair hold their halves: the record may take the result
    int piv[N];
    static_for<0, N>([&](auto K) {
      constexpr int k = K, owner = k / CH, kl = k % CH;
      const int src = pair0 | owner;
      T best = tabs(a[k][kl]);
      int p = k;
      static_for<k + 1, N>([&](auto I) {
        constexpr int i = I;
        const T c = tabs(a[i][kl]);
        if (c > best) {
          best = c;
          p = i;
        }
      });
      p = __shfl_sync(0xffffffffu, p, src);
      piv[k] = p;
      if (warp_any(p != k)) {
        static_for<k + 1, N>([&](auto I) {
          constexpr int i = I;
          const bool sw = (p == i);
          static_for<0, CH>([&](auto J) {
            constexpr int jl = J;
            const T lo = a[k][jl], hi = a[i][jl];
            a[k][jl] = sw ? hi : lo;
            a[i][jl] = sw ? lo : hi;
          });
        });
      }
      const T rp = __shfl_sync(0xffffffffu, T(1) / a[k][kl], src);
      T f[N];
      static_for<0, N>([&](auto I) {
        constexpr int i = I;
        if constexpr (i != k) f[i] = __shfl_sync(0xffffffffu, a[i][kl], src);
      });
      if (h == owner) {
        static_for<0, N>([&](auto I) { a[I][kl] = (int(I) == k) ? T(1) : T(0); });
      }
      static_for<0, CH>([&](auto J) { a[k][J] *= rp; });
      static_for<0, N>([&](auto I) {
        constexpr int i = I;
        if constexpr (i != k) {
          static_for<0, CH>([&](auto J) {
            constexpr int jl = J;
            a[i][jl] -= f[i] * a[k][jl];
          });
        }
      });
    });
    // (P A)^-1 = A^-1 P^T: the column exchanges k <-> piv[k], k = N-1 .. 0, applied to the POSITION
    // of each of this lane's columns instead of to the data
    int w[CH];
    static_for<0, CH>([&](auto J) { w[J] = c0 + J; });
    static_for_down<0, N>([&](auto K) {
      constexpr int k = K;
      const int pk = piv[k];
      if (warp_any(pk != k)) {
        static_for<0, CH>([&](auto J) { w[J] = w[J] == k ? pk : (w[J] == pk ? k : w[J]); });
      }
    });
    static_for<0, N>([&](auto I) {
      static_for<0, CH>([&](auto J) {
        constexpr int i = I, jl = J;
        if (N % 2 == 0 || c0 + jl < N) rec[i * N + w[jl]] = a[i][jl];
      });
    });
  }
};

}  // namespace nfm
