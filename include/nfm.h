/* nfm.h -- C ABI of libnfm_sm100a.so: batched small-matrix linear algebra for
 * NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary for the hot path of nitorch-fastmath.  The
 * reference has no C ABI: the path sits behind Python module functions
 * (cited per entry point below, paths relative to the reference root).  Each
 * function here is what a ctypes/cffi binding for that Python function
 * calls; INTEGRATION.md shows the binding.
 *
 * Conventions (all entry points)
 *   - dtype: NFM_F32 or NFM_F64.  All operands of one call share it.
 *   - Every operand is a batch of small contiguous records (a packed
 *     symmetric matrix, a dense row-major n x n matrix, an n-vector).
 *     `*_stride` is the distance, IN ELEMENTS, between consecutive batch
 *     entries.  stride == record length is the dense case (fast path: TMA
 *     bulk copies into shared memory); stride == 0 broadcasts one record to
 *     the whole batch; any other stride (and any pointer that is not
 *     16-byte aligned) takes a slower strided kernel with identical results.
 *   - `out` may alias an input of the same record shape with the same
 *     stride (in-place variants: sym_solve_, sym_invert_, sym_addmatvec_).
 *   - Pointers are DEVICE pointers on the current CUDA device; `stream` is a
 *     cudaStream_t (NULL = legacy default stream).  The library never
 *     allocates device memory, never synchronises and never changes the
 *     current device.  The `*_host` entry points are the exception: they
 *     take HOST pointers plus a caller-provided device workspace and run a
 *     chunked copy/compute/copy pipeline (they synchronise before return).
 *   - Return value: NFM_OK (0), a negative NFM_E_* code, or a positive
 *     cudaError_t.  nfm_last_error_string() describes the last failure on
 *     the calling thread.  No exceptions cross the ABI; all functions are
 *     re-entrant and safe to call concurrently on different streams/devices.
 */
#ifndef NFM_H_
#define NFM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFM_VERSION 100 /* 0.1.0 */

/* dtype */
#define NFM_F32 0
#define NFM_F64 1

/* compact layouts of the `mat` operand of sym_matvec / sym_solve
 * (nitorch_fastmath/sym.py:16-24) */
#define NFM_LAYOUT_SCALED_IDENTITY 0 /* 1 value            */
#define NFM_LAYOUT_DIAG 1            /* N values           */
#define NFM_LAYOUT_SYM 2             /* N(N+1)/2: diagonal, then rows of the strict upper triangle */
#define NFM_LAYOUT_FULL 3            /* N*N row-major      */

/* factorisation used by solve / invert */
#define NFM_ALGO_AUTO 0 /* sym: closed form N<=4; above, LDL^T with a per-matrix pivot check and pivoted-LU fallback (SPD at LDL^T speed, indefinite as the reference); dense: closed form n<=3 (inverse/det), pivoted LU above */
#define NFM_ALGO_LDL 1  /* LDL^T / Cholesky-type, no pivoting, no check (SPD or strongly regular input) */
#define NFM_ALGO_LU 2   /* LU with partial pivoting (any invertible input) */
#define NFM_ALGO_WARP 3 /* sym_solve only (sym_invert returns NFM_E_UNSUPPORTED): sub-warp cooperative LDL^T with shuffles, 5 <= N <= 10, no pivoting -- SPD input; an A/B variant measured at 0.17-0.33 of the thread-per-matrix kernels */

/* errors */
#define NFM_OK 0
#define NFM_E_UNSUPPORTED (-1) /* n / dtype / layout / algo combination not built */
#define NFM_E_BADARG (-2)      /* null pointer, negative batch, bad stride */
#define NFM_E_WORKSPACE (-3)   /* host pipeline: workspace too small */

#define NFM_MAX_N 10

int nfm_version(void);
const char *nfm_last_error_string(void);
/* number of kernel launches issued by this library in the calling process */
uint64_t nfm_launch_count(void);
/* 1 if the last call on this thread used the TMA-staged thread-per-matrix fast
 * path for its bulk (tile kernel), 2 if it used the sub-warp cooperative kernel,
 * 3 if it used the TMA-staged warp-pool kernel (pivoted ops on large records),
 * 4 if it used the TMA-staged kernel for many right-hand sides / right division
 * (nfm_batch_solve with nrhs > 4, nfm_batch_rsolve with 1 or more than 4 rows;
 * dense 16-byte aligned operands),
 * 0 otherwise (strided kernel) */
int nfm_last_path_was_tma(void);
/* Shape of the bulk launch of the last call on this thread (host-side record, no
 * device work), for tests and tuning:
 *   out[0] kind: 1 tile kernel, 3 warp-pool kernel, 4 many-right-hand-sides kernel,
 *          0 none (strided kernel, sub-warp kernel, or no launch yet)
 *   out[1] threads per CTA      out[2] matrices per thread
 *   out[3] stages (tile), buffers (pool), ring depth per warp (many right-hand sides)
 *   out[4] warps per CTA (pool, many right-hand sides; 0 for the tile kernel)
 *   out[5] segmented shared-memory layout (0/1); many right-hand sides: the
 *          re-layout mask (1 matrices, 2 right-hand sides)
 *   out[6] grid (CTAs)          out[7] tiles (tile kernel) or warp tiles
 * Returns NFM_OK, or NFM_E_BADARG when out is NULL. */
int nfm_last_launch_shape(int64_t out[8]);

/* y = A v            (inp == NULL, sign ignored)
 * y = inp + A v      (sign = +1)      y = inp - A v   (sign = -1)
 * Replaces: sym_matvec  nitorch_fastmath/sym.py:30 (-> jitfields.sym), own
 * implementation nitorch_fastmath/_impl/sym.py:134-172; sym_addmatvec(_),
 * sym_submatvec(_) names at sym.py:31-32.
 * mat: records of length 1 / n / n(n+1)/2 / n*n according to `layout`;
 * vec, inp, out: records of length n. */
int nfm_sym_matvec(int dtype, int n, int layout, int64_t batch,
                   const void *mat, int64_t mat_stride,
                   const void *vec, int64_t vec_stride,
                   const void *inp, int64_t inp_stride, int sign,
                   void *out, int64_t out_stride, void *stream);

/* x = (A + diag(d))^-1 v ; d == NULL means no regulariser.
 * Replaces: sym_solve(_)  sym.py:33, _impl/sym.py:327-398 (closed forms
 * :193-324 for n <= 4; expand + LU for n > 4 :392-396).  `diag` carries the
 * documented `eps` semantics (:356-357): entry i is added to a_ii. */
int nfm_sym_solve(int dtype, int n, int layout, int algo, int64_t batch,
                  const void *mat, int64_t mat_stride,
                  const void *vec, int64_t vec_stride,
                  const void *diag, int64_t diag_stride,
                  void *out, int64_t out_stride, void *stream);

/* out = A^-1 in the same packed order (records of n(n+1)/2), or only its
 * diagonal (records of n) when diag_only != 0.
 * Replaces: sym_invert(_)  sym.py:34, _impl/sym.py:455-493. */
int nfm_sym_invert(int dtype, int n, int algo, int diag_only, int64_t batch,
                   const void *mat, int64_t mat_stride,
                   void *out, int64_t out_stride, void *stream);

/* out = A^-1 for dense row-major n x n records.  closed_form_reg != 0 keeps
 * the reference's regularised determinant for n = 2, 3
 * (det += (max|a| - min|a|) * 1e-12, _impl/batched.py:74-76, :94-96).
 * Replaces: batchinv  batched.py:16, _impl/batched.py:101-130 and
 * sugar.inv  sugar.py:194-258 ('lu' -> NFM_ALGO_LU, 'chol' -> NFM_ALGO_LDL). */
int nfm_batch_inv(int dtype, int n, int algo, int closed_form_reg, int64_t batch,
                  const void *a, int64_t a_stride,
                  void *out, int64_t out_stride, void *stream);

/* out[b] = det A_b (records of length 1).
 * Replaces: batchdet  _impl/batched.py:35-63. */
int nfm_batch_det(int dtype, int n, int64_t batch,
                  const void *a, int64_t a_stride,
                  void *out, int64_t out_stride, void *stream);

/* X = A^-1 B ; A: n x n row-major, B and X: n x nrhs row-major records.
 * algo: NFM_ALGO_LU (partial pivoting) or NFM_ALGO_LDL (Cholesky; A SPD).
 * nrhs 1..4: register kernels on the TMA tile / pool path; more: factors in
 * registers, run-time loop over the right-hand sides out of TMA-staged warp tiles.
 * out may alias b.
 * Replaces: sugar.lmdiv / solvevec  sugar.py:75-137, :290-341. */
int nfm_batch_solve(int dtype, int n, int nrhs, int algo, int64_t batch,
                    const void *a, int64_t a_stride,
                    const void *b, int64_t b_stride,
                    void *out, int64_t out_stride, void *stream);

/* X = B A^-1 (right division) ; A: n x n row-major, B and X: nrows x n row-major
 * records -- solved as A^T x_r = b_r for every row r, without transposed copies
 * (2..4 rows: the register kernels of nfm_batch_solve reading the records in the
 * other index order).  out may alias b.
 * Replaces: sugar.rmdiv  sugar.py:140-191 (documented meaning A x B^-1; as written
 * the reference returns (B^-1 A)^T, see DESIGN.md section 4). */
int nfm_batch_rsolve(int dtype, int n, int nrows, int algo, int64_t batch,
                     const void *a, int64_t a_stride,
                     const void *b, int64_t b_stride,
                     void *out, int64_t out_stride, void *stream);

/* y = A v ; A: m x n row-major, v: n, y: m.
 * Replaces: batchmatvec  _impl/batched.py:154-190. */
int nfm_batch_matvec(int dtype, int m, int n, int64_t batch,
                     const void *mat, int64_t mat_stride,
                     const void *vec, int64_t vec_stride,
                     void *out, int64_t out_stride, void *stream);

/* ---- general strides --------------------------------------------------
 * The *_ex variants describe every operand with a batch stride AND the stride
 * between the elements of one record, both in elements.  elem_stride == 1 is
 * the contiguous record of the plain entry points (which are thin wrappers
 * over these).  Any other value -- typically coefficient-FIRST storage
 * (C, X, Y, Z) viewed coefficient-last, i.e. batch_stride 1 and elem_stride
 * X*Y*Z, which is also what the reference's own sym_solve returns
 * (_impl/sym.py:398) -- is read in place by the strided kernel: adjacent
 * threads then touch adjacent addresses, so no copy to AoS is needed. */
typedef struct nfm_operand {
  const void *ptr;
  int64_t batch_stride;
  int64_t elem_stride;
} nfm_operand;

int nfm_sym_matvec_ex(int dtype, int n, int layout, int64_t batch,
                      const nfm_operand *mat, const nfm_operand *vec,
                      const nfm_operand *inp /* nullable */, int sign,
                      const nfm_operand *out, void *stream);
int nfm_sym_solve_ex(int dtype, int n, int layout, int algo, int64_t batch,
                     const nfm_operand *mat, const nfm_operand *vec,
                     const nfm_operand *diag /* nullable */,
                     const nfm_operand *out, void *stream);
int nfm_sym_invert_ex(int dtype, int n, int algo, int diag_only, int64_t batch,
                      const nfm_operand *mat, const nfm_operand *out, void *stream);

/* ---- "next" rows (SURVEY.md section 8f) -------------------------------- */

/* out[b] = det of a packed symmetric matrix.  Replaces sym_det _impl/sym.py:401-452. */
int nfm_sym_det(int dtype, int n, int64_t batch,
                const void *mat, int64_t mat_stride,
                void *out, int64_t out_stride, void *stream);

/* packed (n(n+1)/2) -> dense n x n.  Replaces sym_to_full _impl/sym.py:16-60. */
int nfm_sym_to_full(int dtype, int n, int64_t batch,
                    const void *mat, int64_t mat_stride,
                    void *out, int64_t out_stride, void *stream);

/* x x^T in packed order.  Replaces sym_outer _impl/sym.py:496-528. */
int nfm_sym_outer(int dtype, int n, int64_t batch,
                  const void *vec, int64_t vec_stride,
                  void *out, int64_t out_stride, void *stream);

/* mode 0: out = J^T H J  (J: k x d row-major, H: packed k(k+1)/2, out: packed
 * d(d+1)/2) -- the documented meaning of sym_matmul (_impl/sym.py:637-656)
 * and what its general branch jhjn computes (:596-634).
 * mode 1: out = J H J^T  (k == d) -- what the reference's unrolled branches
 * jhj1/2/3 compute for k == d <= 3 (:532-593).  1 <= k, d <= 10 (register
 * kernels for k, d <= 6 and for k <= 10 with d <= 3; a run-time-sized kernel otherwise).
 * Replaces sym_matmul _impl/sym.py:637-670. */
int nfm_sym_matmul(int dtype, int k, int d, int mode, int64_t batch,
                   const void *jac, int64_t jac_stride,
                   const void *hess, int64_t hess_stride,
                   void *out, int64_t out_stride, void *stream);

/* Fused Gauss-Newton system (SURVEY.md section 8f rank 1): the packed Hessian
 * J^T H J is built in registers and solved at once, it never goes to HBM:
 *     out = (J^T H J + diag(d))^-1 g          (mode 0)
 *     out = (J H J^T + diag(d))^-1 g          (mode 1, k == d <= 3: the reference's unrolled branches)
 * jac: k x d row-major, hess: packed k(k+1)/2 (mode 0), grad / diag / out: records of d
 * (mode 0); diag may be NULL.  1 <= k, d <= 6, or k <= 10 with d <= 3 (many channels,
 * a 1..3-parameter step).
 * Replaces the chain sym_matmul -> sym_solve, _impl/sym.py:637-670 then :327-398. */
int nfm_sym_matmul_solve(int dtype, int k, int d, int mode, int64_t batch,
                         const void *jac, int64_t jac_stride,
                         const void *hess, int64_t hess_stride,
                         const void *grad, int64_t grad_stride,
                         const void *diag, int64_t diag_stride,
                         void *out, int64_t out_stride, void *stream);

/* Fused regularised solve + update (SURVEY.md section 8f rank 4: the chain
 * sym_solve_ -> sym_submatvec_/sub_ of a Gauss-Newton / Levenberg-Marquardt
 * iteration, names at sym.py:31-33):
 *     out = x - alpha * (A + lam I)^-1 v
 * mat: packed records of n(n+1)/2; vec, x, out: records of n; `out` may alias `x`.
 * algo: NFM_ALGO_AUTO or NFM_ALGO_LDL.  No counterpart function in the reference. */
int nfm_sym_solve_update(int dtype, int n, int algo, int64_t batch,
                         const void *mat, int64_t mat_stride,
                         const void *vec, int64_t vec_stride,
                         const void *x, int64_t x_stride,
                         double lam, double alpha,
                         void *out, int64_t out_stride, void *stream);

/* The same with a per-matrix diagonal regulariser (the documented regulariser of
 * the reference, _impl/sym.py:356-357) as a fourth staged operand:
 *     out = x - alpha * (A + lam I + diag(d))^-1 v ;   diag: records of n, may be NULL. */
int nfm_sym_solve_update_reg(int dtype, int n, int algo, int64_t batch,
                             const void *mat, int64_t mat_stride,
                             const void *vec, int64_t vec_stride,
                             const void *x, int64_t x_stride,
                             const void *diag, int64_t diag_stride,
                             double lam, double alpha,
                             void *out, int64_t out_stride, void *stream);

/* ---- gradients (backward passes of sym_matvec / sym_solve / sym_invert / sym_det) ----
 * p = the stored coefficients of A, g = the incoming gradient.  S(u, w), the
 * gradient of u^T A w with respect to p, is  S_ii = u_i w_i  and
 * S_ij = u_i w_j + u_j w_i (i < j) in the packed layout (the diagonal is not
 * doubled), u_i w_i in the diagonal layout and sum_i u_i w_i in the
 * scaled-identity layout.  The gradients with respect to the vectors are the
 * forward routines: A g (nfm_sym_matvec) and (A + diag d)^-1 g (nfm_sym_solve). */

/* out = sign * S(u, w), records of 1 / n / n(n+1)/2 according to `layout`
 * (NFM_LAYOUT_SCALED_IDENTITY, NFM_LAYOUT_DIAG or NFM_LAYOUT_SYM; sign = +1 or -1);
 * u, w: records of n.
 *   y = inp +/- A v :        d_p = +/- S(g, v)
 *   x = (A + diag d)^-1 v :  d_p = -S(u, x), d_d = -S_diag(u, x)  with u = (A + diag d)^-1 g */
int nfm_sym_outer2(int dtype, int n, int layout, int64_t batch,
                   const void *u, int64_t u_stride,
                   const void *w, int64_t w_stride, int sign,
                   void *out, int64_t out_stride, void *stream);

/* Gradient of B = A^-1 with respect to p:  M = B G B with G_ii = g_ii,
 * G_ij = g_ij / 2 (G = diag(g) when diag_only != 0, the gradient of diag(A^-1));
 * out_ii = -M_ii, out_ij = -2 M_ij.
 * inv: the packed inverse B (records of n(n+1)/2, also when diag_only);
 * grad: records of n(n+1)/2, or n when diag_only; out: records of n(n+1)/2. */
int nfm_sym_invert_backward(int dtype, int n, int diag_only, int64_t batch,
                            const void *inv, int64_t inv_stride,
                            const void *grad, int64_t grad_stride,
                            void *out, int64_t out_stride, void *stream);

/* Gradient of t = det A with respect to p:  out_ii = g adj_ii, out_ij = 2 g adj_ij
 * with adj = t A^-1 the adjugate.  n <= 4: closed-form adjugate (finite for
 * singular A); n > 4: checked LDL^T with a pivoted-elimination fallback.
 * mat, out: records of n(n+1)/2; grad: one value per matrix. */
int nfm_sym_det_backward(int dtype, int n, int64_t batch,
                         const void *mat, int64_t mat_stride,
                         const void *grad, int64_t grad_stride,
                         void *out, int64_t out_stride, void *stream);

/* ---- gradients of the Gauss-Newton builders (sym_matmul, sym_outer, sym_to_full) ----
 * g = the incoming gradient of a packed result of order n; G^ = its full symmetric
 * matrix with the off-diagonals halved (G^_ii = g_ii, G^_ij = g_ij / 2);
 * pack(M) = M_ii, 2 M_ij (i < j).  The fused sym_matmul_solve / sym_solve_update
 * differentiate through nfm_sym_matmul, nfm_sym_solve, nfm_sym_outer2 and
 * nfm_sym_matmul_backward. */

/* Gradient of nfm_sym_matmul (same k, d, mode and the same shapes):
 *   mode 0, Y = J^T H J:  dJ = 2 H J G^,  dH = pack(J G^ J^T)
 *   mode 1, Y = J H J^T:  dJ = 2 G^ J H,  dH = pack(J^T G^ J)      (k == d)
 * jac: k x d row-major, hess: packed, grad: packed records of the result's order.
 * which = 1: out = dJ (records of k*d); 2: out = dH (packed records of H);
 * 3: out = [dJ | dH] (records of k*d + the packed length of H). */
int nfm_sym_matmul_backward(int dtype, int k, int d, int mode, int which, int64_t batch,
                            const void *jac, int64_t jac_stride,
                            const void *hess, int64_t hess_stride,
                            const void *grad, int64_t grad_stride,
                            void *out, int64_t out_stride, void *stream);

/* Gradient of y = x x^T (nfm_sym_outer):  out = 2 G^ x.
 * vec, out: records of n; grad: records of n(n+1)/2. */
int nfm_sym_outer_backward(int dtype, int n, int64_t batch,
                           const void *vec, int64_t vec_stride,
                           const void *grad, int64_t grad_stride,
                           void *out, int64_t out_stride, void *stream);

/* Gradient of F = nfm_sym_to_full(p):  out_ii = G_ii, out_ij = G_ij + G_ji.
 * grad: n x n row-major records; out: records of n(n+1)/2. */
int nfm_sym_to_full_backward(int dtype, int n, int64_t batch,
                             const void *grad, int64_t grad_stride,
                             void *out, int64_t out_stride, void *stream);

/* ---- gradients of the dense routines (batchdet, batchinv, batchmatvec, lmdiv, rmdiv) ----
 * Records are dense row-major.  G is the incoming gradient.  For the LDL^T path
 * (method 'chol') the gradient is the symmetric part of the general formula. */

/* Gradient of t = det A:  out = g * adj(A)^T (the cofactor matrix).  n <= 3:
 * closed-form cofactors (finite for singular A); n >= 4: one pivoted Gauss-Jordan
 * elimination, out = g t A^-T (non-finite for a singular A).
 * mat, out: records of n*n; grad: one value per matrix. */
int nfm_batch_det_backward(int dtype, int n, int64_t batch,
                           const void *mat, int64_t mat_stride,
                           const void *grad, int64_t grad_stride,
                           void *out, int64_t out_stride, void *stream);

/* Gradient of Y = A^-1 from Y:  out = -Y^T G Y^T  (sym == 0: lu / auto), or
 * out = -Y (G + G^T) Y / 2  (sym == 1: 'chol', Y symmetric).  Records of n*n. */
int nfm_batch_inv_backward(int dtype, int n, int sym, int64_t batch,
                           const void *inv, int64_t inv_stride,
                           const void *grad, int64_t grad_stride,
                           void *out, int64_t out_stride, void *stream);

/* order 0: out = sign * U W^T   (U: m x k, W: n x k)
 * order 1: out = sign * U^T W   (U: k x m, W: k x n)
 * out: m x n; sym == 1 (m == n only): sign * (M + M^T) / 2; sign = +1 or -1.
 *   X = A^-1 B  (lmdiv):       dA = -U X^T with U = A^-T G      (order 0, sign -1)
 *   Y = B A^-1  (rmdiv):       dA = -Y^T U with U = G A^-T      (order 1, sign -1)
 *   y = A v     (batchmatvec): dA = g v^T                        (order 0, k = 1)
 * m == n <= 10 with k <= 4 run on the TMA-staged register kernels, other shapes on
 * a run-time-sized kernel. */
int nfm_batch_outer(int dtype, int m, int n, int k, int order, int sym, int sign,
                    int64_t batch, const void *u, int64_t u_stride,
                    const void *w, int64_t w_stride,
                    void *out, int64_t out_stride, void *stream);

/* right == 0: X = A^-T B  (B, X: n x k row-major)
 * right == 1: X = B A^-T  (B, X: k x n row-major)
 * algo: NFM_ALGO_LU (AUTO is LU) or NFM_ALGO_LDL (A symmetric: the same as
 * nfm_batch_solve / nfm_batch_rsolve). */
int nfm_batch_tsolve(int dtype, int n, int k, int right, int algo, int64_t batch,
                     const void *mat, int64_t a_stride,
                     const void *b, int64_t b_stride,
                     void *out, int64_t out_stride, void *stream);

/* y = A^T v ; A: m x n row-major, v: m, y: n. */
int nfm_batch_tmatvec(int dtype, int m, int n, int64_t batch,
                      const void *mat, int64_t mat_stride,
                      const void *vec, int64_t vec_stride,
                      void *out, int64_t out_stride, void *stream);

/* ---- host-buffer pipelines (end-to-end path) --------------------------- */

/* Bytes of device workspace the host pipelines want for `chunk` matrices per
 * stage and `nbuf` stages in flight (records: in_elems + out_elems per matrix). */
size_t nfm_host_workspace_bytes(int dtype, int64_t chunk, int nbuf,
                                int in_elems, int out_elems);

/* x = (A + diag(d))^-1 v with HOST operands (pinned memory gives overlap of
 * H2D, kernel and D2H; pageable memory still works).  Dense strides only
 * (mat: n(n+1)/2, vec/diag/out: n); h_diag may be NULL.  `streams` holds
 * `nbuf` cudaStream_t created by the caller on the current device.
 * Synchronises all of them before returning. */
int nfm_sym_solve_host(int dtype, int n, int algo, int64_t batch,
                       const void *h_mat, const void *h_vec, const void *h_diag,
                       void *h_out,
                       void *d_workspace, size_t workspace_bytes,
                       int64_t chunk, int nbuf, void **streams);

/* same for sym_invert */
int nfm_sym_invert_host(int dtype, int n, int algo, int diag_only, int64_t batch,
                        const void *h_mat, void *h_out,
                        void *d_workspace, size_t workspace_bytes,
                        int64_t chunk, int nbuf, void **streams);

/* same for sym_matvec / addmatvec / submatvec (h_inp may be NULL) */
int nfm_sym_matvec_host(int dtype, int n, int64_t batch,
                        const void *h_mat, const void *h_vec,
                        const void *h_inp, int sign, void *h_out,
                        void *d_workspace, size_t workspace_bytes,
                        int64_t chunk, int nbuf, void **streams);

/* Dense routines with HOST operands, same pipeline: batchinv / batchdet
 * (_impl/batched.py:35-130) and lmdiv / solvevec (sugar.py:75-137, :290-341)
 * called on CPU tensors.  a: n x n row-major records; b, out of the solve:
 * n x nrhs row-major records; out of det: one scalar per matrix. */
int nfm_batch_inv_host(int dtype, int n, int algo, int closed_form_reg, int64_t batch,
                       const void *h_a, void *h_out,
                       void *d_workspace, size_t workspace_bytes,
                       int64_t chunk, int nbuf, void **streams);
int nfm_batch_det_host(int dtype, int n, int64_t batch,
                       const void *h_a, void *h_out,
                       void *d_workspace, size_t workspace_bytes,
                       int64_t chunk, int nbuf, void **streams);
int nfm_batch_solve_host(int dtype, int n, int nrhs, int algo, int64_t batch,
                         const void *h_a, const void *h_b, void *h_out,
                         void *d_workspace, size_t workspace_bytes,
                         int64_t chunk, int nbuf, void **streams);

#ifdef __cplusplus
}
#endif
#endif /* NFM_H_ */
