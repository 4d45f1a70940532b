// nfm_generic.cu -- kernels for the shapes the TMA-staged register kernels do not
// cover: rectangular m x n matvec (batchmatvec's "other sizes" branch,
// _impl/batched.py:175-176), solves with more than 4 right-hand sides and right
// division (sugar.lmdiv / rmdiv, sugar.py:75-191; factorisation in registers, run-time
// loop over the right-hand sides), and J^T H J beyond the templated shapes.  Correct for
// any batch stride; not on the measured hot path.
#include <cstdlib>

#include "nfm_pipeline.cuh"
#include "nfm_sym_math.cuh"

namespace nfm {

// y = A v (A: m x n, y: m), or y = A^T v (v: m, y: n) when `trans` (the gradient of batchmatvec
// with respect to v)
template <typename T>
__global__ void __launch_bounds__(128) matvec_rt_kernel(const T* __restrict__ mat, i64 ms, const T* __restrict__ vec,
                                                        i64 vs, T* __restrict__ out, i64 os, int m, int n, int trans,
                                                        i64 batch) {
  const int rows = trans ? n : m, len = trans ? m : n, step = trans ? n : 1;
  const i64 total = batch * rows;
  for (i64 t = i64(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += i64(gridDim.x) * blockDim.x) {
    const i64 b = t / rows;
    const int i = int(t - b * rows);
    const T* a = mat + b * ms + (trans ? i64(i) : i64(i) * n);
    const T* v = vec + b * vs;
    T s = a[0] * v[0];
    for (int j = 1; j < len; ++j) s += a[i64(j) * step] * v[j];
    out[b * os + i] = s;
  }
}

// out = sign * U W^T (U: m x k, W: n x k row-major; `rows` == 0) or sign * U^T W (U: k x m, W: k x n;
// `rows` == 1), out: m x n row-major; `sym` (m == n): sign * (M + M^T) / 2.  The run-time-sized
// form of BatchOuterOp (nfm_dense_grad.cu) for k > 4 and rectangular shapes.  One thread per element.
template <typename T>
__global__ void __launch_bounds__(128) outer_rt_kernel(const T* __restrict__ u, i64 us, const T* __restrict__ w, i64 ws,
                                                       T* __restrict__ out, i64 os, int m, int n, int k, int rows, int sym,
                                                       T sign, i64 batch) {
  const i64 total = batch * m * n;
  for (i64 t = i64(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += i64(gridDim.x) * blockDim.x) {
    const i64 b = t / (i64(m) * n);
    const int e = int(t - b * m * n), i = e / n, j = e - (e / n) * n;
    const T* ub = u + b * us;
    const T* wb = w + b * ws;
    auto dot = [&](int r, int c) {  // sum_q U(r, q) W(c, q)
      T s = rows ? ub[r] * wb[c] : ub[i64(r) * k] * wb[i64(c) * k];
      for (int q = 1; q < k; ++q) s += rows ? ub[i64(q) * m + r] * wb[i64(q) * n + c] : ub[i64(r) * k + q] * wb[i64(c) * k + q];
      return s;
    };
    const T v = sym ? T(0.5) * (dot(i, j) + dot(j, i)) : dot(i, j);
    out[b * os + e] = sign * v;
  }
}

// ---------------------------------------------------------------------------
// Many right-hand sides (nrhs > 4) and right division: the factorisation lives in
// REGISTERS (compile-time order N, static indices), the right-hand sides are a
// run-time loop.  One thread per matrix, straight from global memory: each thread
// walks its own contiguous records, whose lines stay in L1 between columns.
//   left  (right == 0): X = A^-1 B,  B and X  n x nrhs row-major  (column c: b[i*nrhs + c])
//   right (right == 1): X = B A^-1,  B and X  nrhs x n row-major  (row c: b[c*n + i]), i.e.
//                       A^T x_c = b_c for every row c -- no transposed copies of A or B.
//   bit 1 of `right` (kRightTransposeA) solves with A^T in either order: X = A^-T B, X = B A^-T
//   (the gradients of lmdiv / rmdiv).  LDL^T reads a symmetric matrix and ignores it.
// LU with partial pivoting keeps the multipliers in the lower triangle and the pivot
// rows in piv[]; a column replays the exchanges with predicated swaps (skipped by a
// warp vote when no matrix of the warp pivoted in that step).
// ---------------------------------------------------------------------------
// factorisation of one matrix held in registers: LU with partial pivoting (multipliers in the
// strict lower triangle, reciprocal pivots on the diagonal, pivot rows in piv[]) or LDL^T
// (L in the strict lower triangle, 1 / d on the diagonal)
template <typename T, int N, bool CHOL>
__device__ __forceinline__ void factor_in_registers(T (&a)[N][N], int (&piv)[N]) {
  if constexpr (!CHOL) {
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
      if (warp_any(p != k)) {
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
      const T rp = T(1) / a[k][k];
      a[k][k] = rp;  // the reciprocal pivot is what the substitutions need
      static_for<k + 1, N>([&](auto I) {
        constexpr int i = I;
        const T f = a[i][k] * rp;
        a[i][k] = f;
        static_for<k + 1, N>([&](auto J) {
          constexpr int j = J;
          a[i][j] -= f * a[k][j];
        });
      });
    });
  } else {
    static_for<0, N>([&](auto K) {
      constexpr int k = K;
      const T rp = T(1) / a[k][k];
      static_for<k + 1, N>([&](auto I) {
        constexpr int i = I;
        static_for<k + 1, i + 1>([&](auto J) {
          constexpr int j = J;
          a[i][j] -= a[i][k] * a[j][k] * rp;
        });
      });
      static_for<k + 1, N>([&](auto I) { a[I][k] *= rp; });
      a[k][k] = rp;
      piv[k] = k;
    });
  }
}

// one right-hand side against the factors above, in place
template <typename T, int N, bool CHOL>
__device__ __forceinline__ void substitute_in_registers(const T (&a)[N][N], const int (&piv)[N], T (&x)[N]) {
  if constexpr (!CHOL) {
    // the factorisation exchanged whole rows (multipliers included, as LAPACK's getrf), so
    // all exchanges are applied to the right-hand side first, then L y = P b
    static_for<0, N>([&](auto K) {
      constexpr int k = K;
      if (warp_any(piv[k] != k)) {
        static_for<k + 1, N>([&](auto I) {
          constexpr int i = I;
          const bool sw = (piv[k] == i);
          const T lo = x[k], hi = x[i];
          x[k] = sw ? hi : lo;
          x[i] = sw ? lo : hi;
        });
      }
    });
    static_for<0, N>([&](auto K) {
      constexpr int k = K;
      static_for<k + 1, N>([&](auto I) { x[I] -= a[I][k] * x[k]; });
    });
    static_for_down<0, N>([&](auto K) {  // U x = y
      constexpr int k = K;
      T sum = x[k];
      static_for<k + 1, N>([&](auto J) { sum -= a[k][J] * x[J]; });
      x[k] = sum * a[k][k];
    });
  } else {
    static_for<0, N>([&](auto K) { static_for<K + 1, N>([&](auto I) { x[I] -= a[I][K] * x[K]; }); });
    static_for<0, N>([&](auto K) { x[K] *= a[K][K]; });
    static_for_down<0, N>([&](auto K) { static_for<K + 1, N>([&](auto J) { x[K] -= a[J][K] * x[J]; }); });
  }
}

constexpr int kRightTransposeA = 2;

// the matrix of one system out of its row-major record (transposed for right division, and once more
// for kRightTransposeA; the lower triangle mirrored for the symmetric LDL^T path)
template <typename T, int N, bool CHOL, int PITCH = 1>
__device__ __forceinline__ void load_system(const T* src, int right, T (&a)[N][N]) {
  const bool ta = (right & 1) != ((right & kRightTransposeA) != 0);
  static_for<0, N>([&](auto I) {
    static_for<0, N>([&](auto J) {
      constexpr int i = I, j = J;
      if constexpr (CHOL) a[i][j] = src[((i > j ? i : j) * N + (i > j ? j : i)) * PITCH];  // lower triangle, symmetric
      else a[i][j] = ta ? src[(j * N + i) * PITCH] : src[(i * N + j) * PITCH];
    });
  });
}

template <typename T, int N, bool CHOL>
__global__ void __launch_bounds__(128) solve_many_kernel(const T* mat, i64 as, const T* rhs, i64 bs, T* out, i64 os, int nrhs,
                                                         int right, i64 batch) {
  for (i64 b0 = i64(blockIdx.x) * blockDim.x; b0 < batch; b0 += i64(gridDim.x) * blockDim.x) {
    const bool valid = b0 + threadIdx.x < batch;
    const i64 b = valid ? b0 + threadIdx.x : batch - 1;
    T a[N][N];
    int piv[N];
    load_system<T, N, CHOL, 1>(mat + b * as, right, a);
    factor_in_registers<T, N, CHOL>(a, piv);
    const T* bb = rhs + b * bs;
    T* xx = out + b * os;
    for (int c = 0; c < nrhs; ++c) {
      T x[N];
      static_for<0, N>([&](auto I) { x[I] = (right & 1) ? bb[c * N + I] : bb[I * nrhs + c]; });
      substitute_in_registers<T, N, CHOL>(a, piv, x);
      if (valid) static_for<0, N>([&](auto I) { ((right & 1) ? xx[c * N + I] : xx[I * nrhs + c]) = x[I]; });
    }
  }
}

// ---------------------------------------------------------------------------
// The same computation for DENSE, 16-byte aligned operands, staged by TMA.  A warp-tile
// is 32 consecutive systems: its matrices and its right-hand sides are one contiguous byte
// range each, so they move HBM -> shared memory with two 1-D bulk copies and the solutions
// go back with one -- every HBM access a full burst, where the kernel above walks 32
// records a warp at a stride of n*n / n*nrhs elements.  Every warp owns a private ring of
// `depth` buffers (no CTA-wide barrier anywhere): while it factorises tile i out of one
// buffer, tiles i+1 .. i+depth-1 are in flight into the others.  The solutions overwrite the
// right-hand sides in the buffer (column c of X takes the place of column c of B), which is
// what the bulk store sends back.  Persistent CTAs of `nwarps` warps.
//
// Shared-memory banks.  Lane l works on record l of the tile, i.e. at a stride of one record.
// When the record length shares a large factor with the 32 banks (4x4 fp32: 16 words -> 16-way,
// 6x8 fp32: 48 words -> 16-way, 8x8: 64 words -> 32-way) every access of the elimination
// would be serialised that many times (measured: 2.0 TB/s for the 4x4 right division against
// 5.0 TB/s for 6x6).  Two remedies, chosen by the launcher:
//  * right-hand sides: lanes whose records start in the same bank walk the columns in a different
//    (rotated) order -- no extra work, most conflicts gone;
//  * matrices (read once per system), and right-hand sides with too few columns to rotate over
//    (`transpose` bits 0 / 1): the warp re-lays the tile out element-major with a pitch of 33 records
//    in a per-warp scratch area (coalesced reads, conflict-free writes), works there conflict-free,
//    and lays the solutions back out record-major for the bulk store.
// ---------------------------------------------------------------------------
constexpr int kPitch = 33;

// record-major tile (32 records of `len` elements) -> element-major scratch, and back
template <typename T>
__device__ __forceinline__ void tile_to_scratch(const T* tile, T* scratch, int len, int lane) {
  const int q = 32 / len, r = 32 % len;  // one step of 32 elements = q records and r elements
  int rec = lane / len, e = lane % len;
  for (int w = lane; w < 32 * len; w += 32) {
    scratch[e * kPitch + rec] = tile[w];
    rec += q;
    e += r;
    if (e >= len) {
      e -= len;
      ++rec;
    }
  }
}
template <typename T>
__device__ __forceinline__ void scratch_to_tile(const T* scratch, T* tile, int len, int lane) {
  const int q = 32 / len, r = 32 % len;
  int rec = lane / len, e = lane % len;
  for (int w = lane; w < 32 * len; w += 32) {
    tile[w] = scratch[e * kPitch + rec];
    rec += q;
    e += r;
    if (e >= len) {
      e -= len;
      ++rec;
    }
  }
}
// Warps per CTA = register budget (__launch_bounds__): the kernel is bound by the latency of its
// dependent chains (ncu, 8 warps: issue slots 38 % busy, dominant stall `wait`), so small orders, whose
// factors need few registers, run 12-16 warps with a shallower ring instead of 8 with a deeper one.
template <typename T, int N>
constexpr int many_max_warps() {
  if (sizeof(T) == 4) return N <= 6 ? 16 : N <= 9 ? 12 : 8;
  return N <= 4 ? 16 : N <= 6 ? 12 : 8;
}

template <typename T, int N, bool CHOL>
__global__ void __launch_bounds__(many_max_warps<T, N>() * 32, 1)
    solve_many_staged_kernel(const T* __restrict__ mat, const T* __restrict__ rhs, T* __restrict__ out, const int nrhs,
                             const int right, const i64 ntiles, const int buf_bytes, const int depth, const int transpose,
                             const int rot_shift) {
  constexpr int es = int(sizeof(T));
  constexpr uint32_t a_bytes = 32u * N * N * es;
  const uint32_t b_bytes = 32u * N * uint32_t(nrhs) * es;
  const int brec = N * nrhs;  // elements per right-hand-side record

  extern __shared__ __align__(128) unsigned char smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  unsigned char* const mine = smem + size_t(warp) * depth * buf_bytes;
  uint64_t* const full = reinterpret_cast<uint64_t*>(smem + size_t(nwarps) * depth * buf_bytes) + depth * warp;
  // element-major scratch of this warp (`transpose` bit 0: matrices, bit 1: right-hand sides): the longer
  // of the two record lengths that go through it, x kPitch elements
  const int slen = ((transpose & 2) && nrhs > N) || !(transpose & 1) ? N * nrhs : N * N;
  T* const scratch = reinterpret_cast<T*>(smem + size_t(nwarps) * depth * (buf_bytes + 8) + 16) + size_t(warp) * slen * kPitch;

  if (lane == 0) {
    for (int b = 0; b < depth; ++b) mbar_init(&full[b], 1);
    fence_mbar_init();
  }
  __syncwarp();
  grid_dependency_wait();
  grid_launch_dependents();

  // warp-tiles of this warp: first, first + stride, ...
  const i64 stride = i64(gridDim.x) * nwarps;
  const i64 first = i64(warp) * gridDim.x + blockIdx.x;
  auto issue = [&](int b, i64 tile) {  // lane 0 only
    unsigned char* dst = mine + b * buf_bytes;
    mbar_arrive_expect_tx(&full[b], a_bytes + b_bytes);
    bulk_g2s<false>(dst, mat + tile * (32 * N * N), a_bytes, &full[b], 0);
    bulk_g2s<false>(dst + a_bytes, rhs + tile * 32 * brec, b_bytes, &full[b], 0);
  };
  if (lane == 0)
    for (int b = 0; b < depth - 1; ++b)
      if (first + b * stride < ntiles) issue(b, first + b * stride);

  int cur = 0;          // tile counter of this warp modulo depth
  uint32_t parity = 0;  // (tile counter / depth) & 1
  for (i64 tile = first; tile < ntiles; tile += stride) {
    if (lane == 0) {
      // the tile depth - 1 ahead goes into the buffer the previous tile has just left: its store must have read it
      bulk_wait_read<0>();
      const i64 nxt = tile + (depth - 1) * stride;
      if (nxt < ntiles) issue(cur == 0 ? depth - 1 : cur - 1, nxt);
    }
    mbar_wait(&full[cur], parity);
    unsigned char* buf = mine + cur * buf_bytes;
    T a[N][N];
    int piv[N];
    if (transpose & 1) {  // matrices through the element-major scratch
      tile_to_scratch(reinterpret_cast<const T*>(buf), scratch, N * N, lane);
      __syncwarp();
      load_system<T, N, CHOL, kPitch>(scratch + lane, right, a);
      __syncwarp();  // every lane holds its matrix: the scratch may take the right-hand sides
    } else {
      load_system<T, N, CHOL, 1>(reinterpret_cast<const T*>(buf) + lane * (N * N), right, a);
    }
    if (transpose & 2) tile_to_scratch(reinterpret_cast<const T*>(buf + a_bytes), scratch, brec, lane);
    factor_in_registers<T, N, CHOL>(a, piv);
    if (!(transpose & 2)) {
      T* bb = reinterpret_cast<T*>(buf + a_bytes) + lane * brec;
      // lanes whose records start in the same bank (lane, lane + 32/g, ... for a g-way conflicting record
      // length) take the right-hand sides in a different order, so that they touch different banks
      int c = (lane >> rot_shift) % nrhs;
      for (int done = 0; done < nrhs; ++done) {
        T x[N];
        static_for<0, N>([&](auto I) { x[I] = (right & 1) ? bb[c * N + I] : bb[I * nrhs + c]; });
        substitute_in_registers<T, N, CHOL>(a, piv, x);
        static_for<0, N>([&](auto I) { ((right & 1) ? bb[c * N + I] : bb[I * nrhs + c]) = x[I]; });
        c = c + 1 == nrhs ? 0 : c + 1;
      }
    } else {
      __syncwarp();
      T* bb = scratch + lane;
      for (int c = 0; c < nrhs; ++c) {
        T x[N];
        static_for<0, N>([&](auto I) { x[I] = (right & 1) ? bb[(c * N + I) * kPitch] : bb[(I * nrhs + c) * kPitch]; });
        substitute_in_registers<T, N, CHOL>(a, piv, x);
        static_for<0, N>([&](auto I) { ((right & 1) ? bb[(c * N + I) * kPitch] : bb[(I * nrhs + c) * kPitch]) = x[I]; });
      }
      __syncwarp();
      scratch_to_tile(scratch, reinterpret_cast<T*>(buf + a_bytes), brec, lane);
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      bulk_s2g(out + tile * 32 * brec, buf + a_bytes, b_bytes);
      bulk_commit();
    }
    if (++cur == depth) {
      cur = 0;
      parity ^= 1u;
    }
  }
  if (lane == 0) bulk_wait_read<0>();  // writes complete with the grid; shared memory must outlive the reads
}

// J^T H J (mode 0) or J H J^T (mode 1, k == d) for any 1 <= k, d <= 10:
// run-time-sized fallback of the templated SymMatmulOp (k, d <= 4)
template <typename T>
__global__ void __launch_bounds__(128) matmul_rt_kernel(const T* __restrict__ jac, i64 js, const T* __restrict__ hess, i64 hs,
                                                        T* __restrict__ out, i64 os, int k, int d, int mode, i64 batch) {
  const int hn = mode == 0 ? k : d;  // order of H
  const int on = mode == 0 ? d : k;  // order of the result
  for (i64 b = i64(blockIdx.x) * blockDim.x + threadIdx.x; b < batch; b += i64(gridDim.x) * blockDim.x) {
    const T* j = jac + b * js;
    const T* h = hess + b * hs;
    T hj[NFM_MAX_N][NFM_MAX_N];
    for (int a = 0; a < hn; ++a)
      for (int o = 0; o < on; ++o) {
        T s = T(0);
        for (int c = 0; c < hn; ++c) {
          const int lo = a < c ? a : c, hi = a < c ? c : a;
          const int idx = lo == hi ? lo : hn + lo * hn - (lo * (lo + 1)) / 2 + (hi - lo - 1);
          s += h[idx] * (mode == 0 ? j[c * d + o] : j[o * d + c]);
        }
        hj[a][o] = s;
      }
    T* dst = out + b * os;
    for (int o = 0; o < on; ++o)
      for (int q = o; q < on; ++q) {
        T s = T(0);
        for (int a = 0; a < hn; ++a) s += (mode == 0 ? j[a * d + o] : j[o * d + a]) * hj[a][q];
        dst[o == q ? o : on + o * on - (o * (o + 1)) / 2 + (q - o - 1)] = s;
      }
  }
}

__device__ __forceinline__ int pidx_rt(int n, int i, int j) {
  const int lo = i < j ? i : j, hi = i < j ? j : i;
  return lo == hi ? lo : n + lo * n - (lo * (lo + 1)) / 2 + (hi - lo - 1);
}

// Gradient of J^T H J (mode 0) / J H J^T (mode 1) for the shapes matmul_rt_kernel runs: the
// run-time-sized form of SymMatmulBackwardOp (nfm_gn_grad.cu), same formulas, same record layout
// (`which` 1 = dJ, 2 = dH, 3 = [dJ | dH]).  F(o, a) is the ON x HN factor of Y = F H F^T.
template <typename T>
__global__ void __launch_bounds__(128) matmul_backward_rt_kernel(const T* __restrict__ jac, i64 js, const T* __restrict__ hess,
                                                                 i64 hs, const T* __restrict__ grad, i64 gs, T* __restrict__ out,
                                                                 i64 os, int k, int d, int mode, int which, i64 batch) {
  const int hn = mode == 0 ? k : d;  // order of H
  const int on = mode == 0 ? d : k;  // order of Y
  const int kj = (which & 1) ? k * d : 0;
  for (i64 b = i64(blockIdx.x) * blockDim.x + threadIdx.x; b < batch; b += i64(gridDim.x) * blockDim.x) {
    const T* j = jac + b * js;
    const T* h = hess + b * hs;
    const T* g = grad + b * gs;
    T* dst = out + b * os;
    auto f = [&](int o, int a) { return mode == 0 ? j[a * d + o] : j[o * d + a]; };
    auto ghat = [&](int o, int q) { return o == q ? g[o] : T(0.5) * g[pidx_rt(on, o, q)]; };
    T r[NFM_MAX_N];
    if (which & 1) {
      for (int o = 0; o < on; ++o) {  // row o of dF = 2 G^ F H
        for (int a = 0; a < hn; ++a) {
          T s = T(0);
          for (int q = 0; q < on; ++q) s += ghat(o, q) * f(q, a);
          r[a] = s;
        }
        for (int c = 0; c < hn; ++c) {
          T s = T(0);
          for (int a = 0; a < hn; ++a) s += r[a] * h[pidx_rt(hn, a, c)];
          dst[mode == 0 ? c * d + o : o * d + c] = T(2) * s;
        }
      }
    }
    if (which & 2) {
      for (int a = 0; a < hn; ++a) {  // row a of F^T G^ F, packed
        for (int q = 0; q < on; ++q) {
          T s = T(0);
          for (int o = 0; o < on; ++o) s += f(o, a) * ghat(o, q);
          r[q] = s;
        }
        for (int c = a; c < hn; ++c) {
          T s = T(0);
          for (int q = 0; q < on; ++q) s += r[q] * f(q, c);
          dst[kj + pidx_rt(hn, a, c)] = a == c ? s : T(2) * s;
        }
      }
    }
  }
}

static unsigned grid_for(i64 work);

template <typename T>
int sym_matmul_backward_rt(int k, int d, int mode, int which, i64 batch, const void* jac, i64 js, const void* hess, i64 hs,
                           const void* grad, i64 gs, void* out, i64 os, cudaStream_t s) {
  if (batch == 0) return 0;
  matmul_backward_rt_kernel<T><<<grid_for(batch), 128, 0, s>>>(static_cast<const T*>(jac), js, static_cast<const T*>(hess), hs,
                                                               static_cast<const T*>(grad), gs, static_cast<T*>(out), os, k, d,
                                                               mode, which, batch);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(cudaGetLastError());
}
template int sym_matmul_backward_rt<float>(int, int, int, int, i64, const void*, i64, const void*, i64, const void*, i64, void*, i64,
                                           cudaStream_t);
template int sym_matmul_backward_rt<double>(int, int, int, int, i64, const void*, i64, const void*, i64, const void*, i64, void*,
                                            i64, cudaStream_t);

template <typename T>
int sym_matmul_rt(int k, int d, int mode, i64 batch, const void* jac, i64 js, const void* hess, i64 hs, void* out, i64 os,
                  cudaStream_t s) {
  if (batch == 0) return 0;
  matmul_rt_kernel<T><<<grid_for(batch), 128, 0, s>>>(static_cast<const T*>(jac), js, static_cast<const T*>(hess), hs,
                                                      static_cast<T*>(out), os, k, d, mode, batch);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(cudaGetLastError());
}
template int sym_matmul_rt<float>(int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);
template int sym_matmul_rt<double>(int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);

static unsigned grid_for(i64 work) {
  i64 blocks = (work + 127) / 128;
  const i64 cap = i64(device_info().sm_count) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return unsigned(blocks);
}

template <typename T>
int batch_matvec_rt(int m, int n, int trans, i64 batch, const void* mat, i64 ms, const void* vec, i64 vs, void* out, i64 os,
                    cudaStream_t s) {
  if (batch == 0) return 0;
  matvec_rt_kernel<T><<<grid_for(batch * (trans ? n : m)), 128, 0, s>>>(static_cast<const T*>(mat), ms, static_cast<const T*>(vec),
                                                                        vs, static_cast<T*>(out), os, m, n, trans, batch);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(cudaGetLastError());
}

template <typename T>
int batch_outer_rt(int m, int n, int k, int rows, int sym, int sign, i64 batch, const void* u, i64 us, const void* w, i64 ws,
                   void* out, i64 os, cudaStream_t s) {
  if (batch == 0) return 0;
  outer_rt_kernel<T><<<grid_for(batch * m * n), 128, 0, s>>>(static_cast<const T*>(u), us, static_cast<const T*>(w), ws,
                                                             static_cast<T*>(out), os, m, n, k, rows, sym, T(sign), batch);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(cudaGetLastError());
}
template int batch_outer_rt<float>(int, int, int, int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);
template int batch_outer_rt<double>(int, int, int, int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);

bool many_staged_enabled() {  // NFM_DISABLE_MANY_STAGED=1: always the one-thread-per-system global-memory kernel
  static const bool on = [] {
    const char* e = getenv("NFM_DISABLE_MANY_STAGED");
    return !(e && e[0] == '1');
  }();
  return on;
}

template <typename T, int N, bool CHOL>
static int solve_many_launch(int nrhs, int right, i64 batch, const T* a, i64 as, const T* b, i64 bs, T* out, i64 os, cudaStream_t s) {
  t_last_path_tma = 0;
  reset_launch_record();
  constexpr int es = int(sizeof(T));
  const i64 brec = i64(N) * nrhs;
  const bool dense = as == N * N && bs == brec && os == brec && aligned16(a) && aligned16(b) && aligned16(out);
  i64 done = 0;
  if (dense && batch >= 64 && nrhs <= 256 && many_staged_enabled()) {  // (more columns than that never fit three warps)
    // a warp's buffer: 32 matrices + 32 right-hand-side records; 2..4 buffers per warp, up to
    // many_max_warps() warps per CTA and as many CTAs per SM as registers and shared memory allow
    const int buf_bytes = int((32 * (N * N + brec) * es + 127) / 128 * 128);
    // bank-conflict degree of record-strided accesses (see the kernel): re-lay the tile out when >= 16-way.
    // Measured (profiles/r2_nrhs_timing.txt): the three extra passes over shared memory pay only there --
    // 4x4 fp64 right division 2.05 -> 4.60 TB/s (16-way), but 6x6 fp32 (4-way) 5.0 -> 2.9 TB/s.
    auto degree = [](i64 len) {
      const i64 words = len * es / 4;
      int g = 1;
      while (g < 32 && words % (2 * g) == 0) g *= 2;
      return g / (es / 4);
    };
    static const int transpose_from = [] {  // tuning aid: NFM_MANY_TRANSPOSE_FROM=64 never re-lays a tile out
      const char* e = getenv("NFM_MANY_TRANSPOSE_FROM");
      return e ? atoi(e) : 16;
    }();
    // matrices: read once per system, so one pass through the scratch pays from 16-way conflicts (4x4, 8x8);
    // right-hand sides: the lane-rotated column order (below) removes most conflicts without any extra pass
    // (6x8 fp32 5.2 TB/s rotated, 2.8 through the scratch) unless there are too few columns to rotate over
    const int transpose = (degree(N * N) >= transpose_from ? 1 : 0) | (degree(brec) >= transpose_from && nrhs < 4 ? 2 : 0);
    // lanes l and l + 32/g start in the same bank when the right-hand-side record conflicts g-way
    int g = 1;
    while (g < 32 && (brec * es / 4) % (2 * g) == 0) g *= 2;
    int rot_shift = 0;
    while ((32 / g) >> (rot_shift + 1)) ++rot_shift;   // log2(32 / g)
    if (g == 1) rot_shift = 5;                          // odd record length: conflict free, no rotation
    const int slen = ((transpose & 2) && nrhs > N) || !(transpose & 1) ? N * nrhs : N * N;  // as in the kernel
    const int scratch_bytes = transpose ? slen * kPitch * es : 0;
    const DeviceInfo& dev = device_info();
    const int avail = dev.max_smem_optin - 256;
    int nwarps = avail / (2 * (buf_bytes + 8) + scratch_bytes);
    if (nwarps > many_max_warps<T, N>()) nwarps = many_max_warps<T, N>();
    if (nwarps >= 3) {
      int depth = (avail / nwarps - scratch_bytes) / (buf_bytes + 8);
      if (depth > 4) depth = 4;
      auto kern = solve_many_staged_kernel<T, N, CHOL>;
      static std::atomic<int> attr_set[16];
      const int d = current_device() & 15;
      if (!attr_set[d].load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin);
        if (e != cudaSuccess) return int(e);
        attr_set[d].store(1, std::memory_order_release);
      }
      const size_t smem = size_t(nwarps) * (depth * (buf_bytes + 8) + scratch_bytes) + 16;
      int per_sm = 1;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nwarps * 32, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
      if (per_sm > 4) per_sm = 4;
      const i64 ntiles = batch / 32;
      i64 grid = (ntiles + nwarps - 1) / nwarps;
      if (grid > i64(dev.sm_count) * per_sm) grid = i64(dev.sm_count) * per_sm;
      cudaError_t e = launch_pdl(kern, unsigned(grid), unsigned(nwarps * 32), smem, s, a, b, out, nrhs, right, ntiles, buf_bytes, depth,
                                 transpose, rot_shift);
      g_launch_count.fetch_add(1, std::memory_order_relaxed);
      if (e != cudaSuccess) return int(e);
      t_last_path_tma = 4;
      record_launch(4, nwarps * 32, 1, depth, nwarps, transpose, grid, ntiles);  // slot 5: the re-layout mask
      done = ntiles * 32;
      if (done == batch) return 0;
    }
  }
  // everything (strided / broadcast / unaligned operands), or the < 32 systems after the last warp-tile
  solve_many_kernel<T, N, CHOL><<<grid_for(batch - done), 128, 0, s>>>(a + done * as, as, b + done * bs, bs, out + done * os, os, nrhs,
                                                                        right, batch - done);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(cudaGetLastError());
}

template <typename T, int N>
static int solve_many_n(int n, int nrhs, int chol, int right, i64 batch, const T* a, i64 as, const T* b, i64 bs, T* out, i64 os,
                        cudaStream_t s) {
  if (n == N) {
    return chol ? solve_many_launch<T, N, true>(nrhs, right, batch, a, as, b, bs, out, os, s)
                : solve_many_launch<T, N, false>(nrhs, right, batch, a, as, b, bs, out, os, s);
  }
  if constexpr (N < NFM_MAX_N) return solve_many_n<T, N + 1>(n, nrhs, chol, right, batch, a, as, b, bs, out, os, s);
  else return NFM_E_UNSUPPORTED;
}

template <typename T>
int batch_solve_many(int n, int nrhs, int chol, int right, i64 batch, const void* a, i64 as, const void* b, i64 bs, void* out,
                     i64 os, cudaStream_t s) {
  if (batch == 0) return 0;
  return solve_many_n<T, 1>(n, nrhs, chol, right, batch, static_cast<const T*>(a), as, static_cast<const T*>(b), bs,
                            static_cast<T*>(out), os, s);
}
template int batch_solve_many<float>(int, int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);
template int batch_solve_many<double>(int, int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);

template int batch_matvec_rt<float>(int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);
template int batch_matvec_rt<double>(int, int, int, i64, const void*, i64, const void*, i64, void*, i64, cudaStream_t);

}  // namespace nfm
