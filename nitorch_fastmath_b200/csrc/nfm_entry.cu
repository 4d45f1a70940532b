// nfm_entry.cu -- the C ABI (include/nfm.h): argument validation, parameter
// block assembly, dispatch to the typed implementations.  No kernels here.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include "nfm_impl.cuh"
#include "nfm_pipeline.cuh"
#include "nfm_sym_math.cuh"

namespace nfm {

std::atomic<unsigned long long> g_launch_count{0};
thread_local int t_last_path_tma = 0;
thread_local long long t_last_launch[8] = {};
static thread_local char t_error[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_error, sizeof(t_error), fmt, ap);
  va_end(ap);
}

const DeviceInfo& device_info() {
  static DeviceInfo cache[64];
  static std::atomic<int> ready[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!ready[dev].load(std::memory_order_acquire)) {
    DeviceInfo d{};
    cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    cache[dev] = d;
    ready[dev].store(1, std::memory_order_release);
  }
  return cache[dev];
}

bool pdl_enabled() {
  static const bool on = [] {
    const char* v = std::getenv("NFM_DISABLE_PDL");
    return !(v != nullptr && v[0] == '1');
  }();
  return on;
}

bool balance_enabled() {
  // equal-tile scheduling (balanced_tile): measured neutral once the partial tile moves by TMA
  // (profiles/r2_geometry_sweep.txt), so it is off unless NFM_BALANCE=1
  static const bool on = [] {
    const char* v = std::getenv("NFM_BALANCE");
    return v != nullptr && v[0] == '1';
  }();
  return on;
}

int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev;
}

namespace {

int fail(int code, const char* what) {
  set_error("%s", what);
  return code;
}

struct Args {
  KParams p{};
  int rc = NFM_OK;
  void in(int slot, const void* ptr, i64 stride, bool required, i64 estride = 1) {
    if (ptr == nullptr) {
      if (required) rc = fail(NFM_E_BADARG, "required operand is NULL");
      return;
    }
    if (stride < 0 || estride < 0) rc = fail(NFM_E_BADARG, "negative stride");
    p.in[slot].ptr = ptr;
    p.in[slot].stride = stride;
    p.in[slot].estride = estride;
    p.present |= 1 << slot;
  }
  void in(int slot, const nfm_operand* op, bool required) {
    if (op == nullptr) {
      if (required) rc = fail(NFM_E_BADARG, "required operand is NULL");
      return;
    }
    in(slot, op->ptr, op->batch_stride, required, op->elem_stride);
  }
  void out(void* ptr, i64 stride, i64 estride = 1) {
    if (ptr == nullptr) rc = fail(NFM_E_BADARG, "output is NULL");
    if (stride < 0 || estride < 0) rc = fail(NFM_E_BADARG, "negative stride");
    p.out = ptr;
    p.out_stride = stride;
    p.out_estride = estride;
  }
  void out(const nfm_operand* op) {
    if (op == nullptr) {
      rc = fail(NFM_E_BADARG, "output is NULL");
      return;
    }
    out(const_cast<void*>(op->ptr), op->batch_stride, op->elem_stride);
  }
};

bool check_common(int dtype, int n, i64 batch, int& rc) {
  if (dtype != NFM_F32 && dtype != NFM_F64) {
    rc = fail(NFM_E_UNSUPPORTED, "dtype must be NFM_F32 or NFM_F64");
    return false;
  }
  if (n < 1 || n > NFM_MAX_N) {
    rc = fail(NFM_E_UNSUPPORTED, "matrix order must be in 1..10");
    return false;
  }
  if (batch < 0) {
    rc = fail(NFM_E_BADARG, "negative batch");
    return false;
  }
  return true;
}

int finish(int rc) {
  if (rc == NFM_E_UNSUPPORTED) set_error("combination of n / layout / algo not built");
  return rc;
}

}  // namespace
}  // namespace nfm

using namespace nfm;

extern "C" {

int nfm_version(void) { return NFM_VERSION; }
const char* nfm_last_error_string(void) { return nfm::t_error; }
uint64_t nfm_launch_count(void) { return g_launch_count.load(); }
int nfm_last_path_was_tma(void) { return t_last_path_tma; }
int nfm_last_launch_shape(int64_t out[8]) {
  if (out == nullptr) return fail(NFM_E_BADARG, "output is NULL");
  for (int i = 0; i < 8; ++i) out[i] = t_last_launch[i];
  return NFM_OK;
}

int nfm_sym_matvec_ex(int dtype, int n, int layout, int64_t batch, const nfm_operand* mat, const nfm_operand* vec,
                      const nfm_operand* inp, int sign, const nfm_operand* out, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (layout < 0 || layout > 3) return fail(NFM_E_UNSUPPORTED, "unknown layout");
  const bool has_inp = inp != nullptr && inp->ptr != nullptr;
  if (has_inp && sign != 1 && sign != -1) return fail(NFM_E_BADARG, "sign must be +1 or -1 when inp is given");
  Args a;
  a.in(0, mat, true);
  a.in(1, vec, true);
  if (has_inp) a.in(2, inp, false);
  a.out(out);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  a.p.flags = (has_inp && sign < 0) ? 1 : 0;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? sym_matvec_impl<float>(n, layout, a.p, s) : sym_matvec_impl<double>(n, layout, a.p, s));
}

int nfm_sym_matvec(int dtype, int n, int layout, int64_t batch, const void* mat, int64_t mat_stride, const void* vec,
                   int64_t vec_stride, const void* inp, int64_t inp_stride, int sign, void* out, int64_t out_stride,
                   void* stream) {
  const nfm_operand m{mat, mat_stride, 1}, v{vec, vec_stride, 1}, i{inp, inp_stride, 1}, o{out, out_stride, 1};
  return nfm_sym_matvec_ex(dtype, n, layout, batch, &m, &v, inp ? &i : nullptr, sign, &o, stream);
}

int nfm_sym_solve_ex(int dtype, int n, int layout, int algo, int64_t batch, const nfm_operand* mat, const nfm_operand* vec,
                     const nfm_operand* diag, const nfm_operand* out, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (layout < 0 || layout > 3) return fail(NFM_E_UNSUPPORTED, "unknown layout");
  if (algo < NFM_ALGO_AUTO || algo > NFM_ALGO_WARP) return fail(NFM_E_UNSUPPORTED, "unknown algo");
  Args a;
  a.in(0, mat, true);
  a.in(1, vec, true);
  if (diag != nullptr && diag->ptr != nullptr) a.in(2, diag, false);
  a.out(out);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  const bool big = layout == NFM_LAYOUT_SYM && n > 4;
  if (!big) return finish(dtype == NFM_F32 ? sym_solve_part0<float>(n, layout, a.p, s) : sym_solve_part0<double>(n, layout, a.p, s));
  if (algo == NFM_ALGO_LU)
    return finish(dtype == NFM_F32 ? sym_solve_part2<float>(n, a.p, s) : sym_solve_part2<double>(n, a.p, s));
  if (algo == NFM_ALGO_WARP)
    return finish(dtype == NFM_F32 ? sym_solve_warp<float>(n, a.p, s) : sym_solve_warp<double>(n, a.p, s));
  if (algo == NFM_ALGO_LDL)
    return finish(dtype == NFM_F32 ? sym_solve_part1<float>(n, a.p, s) : sym_solve_part1<double>(n, a.p, s));
  return finish(dtype == NFM_F32 ? sym_solve_part3<float>(n, a.p, s) : sym_solve_part3<double>(n, a.p, s));
}

int nfm_sym_solve(int dtype, int n, int layout, int algo, int64_t batch, const void* mat, int64_t mat_stride,
                  const void* vec, int64_t vec_stride, const void* diag, int64_t diag_stride, void* out,
                  int64_t out_stride, void* stream) {
  const nfm_operand m{mat, mat_stride, 1}, v{vec, vec_stride, 1}, d{diag, diag_stride, 1}, o{out, out_stride, 1};
  return nfm_sym_solve_ex(dtype, n, layout, algo, batch, &m, &v, diag ? &d : nullptr, &o, stream);
}

int nfm_sym_invert_ex(int dtype, int n, int algo, int diag_only, int64_t batch, const nfm_operand* mat,
                      const nfm_operand* out, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (algo < NFM_ALGO_AUTO || algo > NFM_ALGO_WARP) return fail(NFM_E_UNSUPPORTED, "unknown algo");
  if (algo == NFM_ALGO_WARP) return fail(NFM_E_UNSUPPORTED, "sym_invert has no sub-warp variant (NFM_ALGO_WARP is a sym_solve A/B kernel)");
  Args a;
  a.in(0, mat, true);
  a.out(out);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  if (algo == NFM_ALGO_LU && n > 4)
    return finish(dtype == NFM_F32 ? sym_invert_part1<float>(n, diag_only, a.p, s) : sym_invert_part1<double>(n, diag_only, a.p, s));
  if (algo == NFM_ALGO_AUTO && n > 4)
    return finish(dtype == NFM_F32 ? sym_invert_part2<float>(n, diag_only, a.p, s) : sym_invert_part2<double>(n, diag_only, a.p, s));
  // N <= 4 closed forms; NFM_ALGO_LDL
  return finish(dtype == NFM_F32 ? sym_invert_part0<float>(n, diag_only, a.p, s) : sym_invert_part0<double>(n, diag_only, a.p, s));
}

int nfm_sym_invert(int dtype, int n, int algo, int diag_only, int64_t batch, const void* mat, int64_t mat_stride,
                   void* out, int64_t out_stride, void* stream) {
  const nfm_operand m{mat, mat_stride, 1}, o{out, out_stride, 1};
  return nfm_sym_invert_ex(dtype, n, algo, diag_only, batch, &m, &o, stream);
}

int nfm_sym_outer2(int dtype, int n, int layout, int64_t batch, const void* u, int64_t u_stride, const void* w,
                   int64_t w_stride, int sign, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (layout < 0 || layout > 2) return fail(NFM_E_UNSUPPORTED, "layout must be scaled identity, diagonal or packed");
  if (sign != 1 && sign != -1) return fail(NFM_E_BADARG, "sign must be +1 or -1");
  Args a;
  a.in(0, u, u_stride, true);
  a.in(1, w, w_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  a.p.flags = sign < 0 ? 1 : 0;  // kFlagSubtract
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? sym_outer2_impl<float>(n, layout, a.p, s) : sym_outer2_impl<double>(n, layout, a.p, s));
}

int nfm_sym_invert_backward(int dtype, int n, int diag_only, int64_t batch, const void* inv, int64_t inv_stride,
                            const void* grad, int64_t grad_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, inv, inv_stride, true);
  a.in(1, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? sym_invert_backward_impl<float>(n, diag_only, a.p, s)
                                 : sym_invert_backward_impl<double>(n, diag_only, a.p, s));
}

int nfm_sym_det_backward(int dtype, int n, int64_t batch, const void* mat, int64_t mat_stride, const void* grad,
                         int64_t grad_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, mat, mat_stride, true);
  a.in(1, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? sym_det_backward_impl<float>(n, a.p, s) : sym_det_backward_impl<double>(n, a.p, s));
}

int nfm_batch_inv(int dtype, int n, int algo, int closed_form_reg, int64_t batch, const void* mat, int64_t a_stride,
                  void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, mat, a_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  a.p.flags = closed_form_reg ? 1 : 0;
  auto s = static_cast<cudaStream_t>(stream);
  if (algo == NFM_ALGO_LDL)
    return finish(dtype == NFM_F32 ? batch_inv_ldl_impl<float>(n, a.p, s) : batch_inv_ldl_impl<double>(n, a.p, s));
  if (algo != NFM_ALGO_AUTO && algo != NFM_ALGO_LU) return fail(NFM_E_UNSUPPORTED, "batch_inv: algo must be AUTO, LU or LDL");
  if (algo == NFM_ALGO_LU && n <= 3)  // pivoted elimination as documented, not the closed forms AUTO takes there
    return finish(dtype == NFM_F32 ? batch_inv_lu_small_impl<float>(n, a.p, s) : batch_inv_lu_small_impl<double>(n, a.p, s));
  return finish(dtype == NFM_F32 ? batch_inv_lu_impl<float>(n, a.p, s) : batch_inv_lu_impl<double>(n, a.p, s));
}

int nfm_batch_det(int dtype, int n, int64_t batch, const void* mat, int64_t a_stride, void* out, int64_t out_stride,
                  void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, mat, a_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? batch_det_impl<float>(n, a.p, s) : batch_det_impl<double>(n, a.p, s));
}

int nfm_batch_solve(int dtype, int n, int nrhs, int algo, int64_t batch, const void* mat, int64_t a_stride,
                    const void* b, int64_t b_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (nrhs < 1) return fail(NFM_E_BADARG, "nrhs must be >= 1");
  if (algo == NFM_ALGO_AUTO) algo = NFM_ALGO_LU;
  if (algo != NFM_ALGO_LU && algo != NFM_ALGO_LDL) return fail(NFM_E_UNSUPPORTED, "batch_solve: algo must be LU or LDL");
  auto s = static_cast<cudaStream_t>(stream);
  if (nrhs >= 2 && nrhs <= 4) {  // register kernels through the TMA pipeline
    Args a;
    a.in(0, mat, a_stride, true);
    a.in(1, b, b_stride, true);
    a.out(out, out_stride);
    if (a.rc) return a.rc;
    a.p.batch = batch;
    if (algo == NFM_ALGO_LDL)
      return finish(dtype == NFM_F32 ? batch_solvek_ldl_impl<float>(n, nrhs, a.p, s) : batch_solvek_ldl_impl<double>(n, nrhs, a.p, s));
    return finish(dtype == NFM_F32 ? batch_solvek_lu_impl<float>(n, nrhs, a.p, s) : batch_solvek_lu_impl<double>(n, nrhs, a.p, s));
  }
  if (nrhs > 1) {
    if (mat == nullptr || b == nullptr || out == nullptr) return fail(NFM_E_BADARG, "NULL operand");
    if (a_stride < 0 || b_stride < 0 || out_stride < 0) return fail(NFM_E_BADARG, "negative batch stride");
    const int chol = algo == NFM_ALGO_LDL;
    rc = dtype == NFM_F32 ? batch_solve_many<float>(n, nrhs, chol, 0, batch, mat, a_stride, b, b_stride, out, out_stride, s)
                          : batch_solve_many<double>(n, nrhs, chol, 0, batch, mat, a_stride, b, b_stride, out, out_stride, s);
    if (rc) set_error("solve kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
    return rc;
  }
  Args a;
  a.in(0, mat, a_stride, true);
  a.in(1, b, b_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  if (algo == NFM_ALGO_LDL)
    return finish(dtype == NFM_F32 ? batch_solve_ldl_impl<float>(n, a.p, s) : batch_solve_ldl_impl<double>(n, a.p, s));
  return finish(dtype == NFM_F32 ? batch_solve_lu_impl<float>(n, a.p, s) : batch_solve_lu_impl<double>(n, a.p, s));
}

int nfm_batch_rsolve(int dtype, int n, int nrows, int algo, int64_t batch, const void* mat, int64_t a_stride, const void* b,
                     int64_t b_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (nrows < 1) return fail(NFM_E_BADARG, "nrows must be >= 1");
  if (algo == NFM_ALGO_AUTO) algo = NFM_ALGO_LU;
  if (algo != NFM_ALGO_LU && algo != NFM_ALGO_LDL) return fail(NFM_E_UNSUPPORTED, "batch_rsolve: algo must be LU or LDL");
  if (mat == nullptr || b == nullptr || out == nullptr) return fail(NFM_E_BADARG, "NULL operand");
  if (a_stride < 0 || b_stride < 0 || out_stride < 0) return fail(NFM_E_BADARG, "negative batch stride");
  auto s = static_cast<cudaStream_t>(stream);
  if (nrows >= 2 && nrows <= 4) {  // the register kernels of nfm_batch_solve, records read in the other index order
    Args a;
    a.in(0, mat, a_stride, true);
    a.in(1, b, b_stride, true);
    a.out(out, out_stride);
    if (a.rc) return a.rc;
    a.p.batch = batch;
    a.p.flags = kFlagRightDivision;
    if (algo == NFM_ALGO_LDL)
      return finish(dtype == NFM_F32 ? batch_solvek_ldl_impl<float>(n, nrows, a.p, s) : batch_solvek_ldl_impl<double>(n, nrows, a.p, s));
    return finish(dtype == NFM_F32 ? batch_solvek_lu_impl<float>(n, nrows, a.p, s) : batch_solvek_lu_impl<double>(n, nrows, a.p, s));
  }
  const int chol = algo == NFM_ALGO_LDL;
  rc = dtype == NFM_F32 ? batch_solve_many<float>(n, nrows, chol, 1, batch, mat, a_stride, b, b_stride, out, out_stride, s)
                        : batch_solve_many<double>(n, nrows, chol, 1, batch, mat, a_stride, b, b_stride, out, out_stride, s);
  if (rc) set_error("solve kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

int nfm_batch_matvec(int dtype, int m, int n, int64_t batch, const void* mat, int64_t mat_stride, const void* vec,
                     int64_t vec_stride, void* out, int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) return fail(NFM_E_UNSUPPORTED, "dtype must be NFM_F32 or NFM_F64");
  if (m < 1 || n < 1) return fail(NFM_E_BADARG, "matrix shape must be positive");
  if (batch < 0) return fail(NFM_E_BADARG, "negative batch");
  auto s = static_cast<cudaStream_t>(stream);
  if (m == n && n <= NFM_MAX_N) {
    Args a;
    a.in(0, mat, mat_stride, true);
    a.in(1, vec, vec_stride, true);
    a.out(out, out_stride);
    if (a.rc) return a.rc;
    a.p.batch = batch;
    return finish(dtype == NFM_F32 ? batch_matvec_impl<float>(n, a.p, s) : batch_matvec_impl<double>(n, a.p, s));
  }
  if (mat == nullptr || vec == nullptr || out == nullptr) return fail(NFM_E_BADARG, "NULL operand");
  if (mat_stride < 0 || vec_stride < 0 || out_stride < 0) return fail(NFM_E_BADARG, "negative batch stride");
  t_last_path_tma = 0;
  reset_launch_record();
  int rc = dtype == NFM_F32 ? batch_matvec_rt<float>(m, n, 0, batch, mat, mat_stride, vec, vec_stride, out, out_stride, s)
                            : batch_matvec_rt<double>(m, n, 0, batch, mat, mat_stride, vec, vec_stride, out, out_stride, s);
  if (rc) set_error("matvec kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

int nfm_sym_matmul_backward(int dtype, int k, int d, int mode, int which, int64_t batch, const void* jac, int64_t jac_stride,
                            const void* hess, int64_t hess_stride, const void* grad, int64_t grad_stride, void* out,
                            int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) return fail(NFM_E_UNSUPPORTED, "dtype must be NFM_F32 or NFM_F64");
  if (k < 1 || k > NFM_MAX_N || d < 1 || d > NFM_MAX_N) return fail(NFM_E_UNSUPPORTED, "sym_matmul_backward: 1 <= k, d <= 10");
  if (mode != 0 && mode != 1) return fail(NFM_E_UNSUPPORTED, "mode must be 0 (J^T H J) or 1 (J H J^T)");
  if (mode == 1 && k != d) return fail(NFM_E_UNSUPPORTED, "mode 1 needs k == d");
  if (which < 1 || which > 3) return fail(NFM_E_UNSUPPORTED, "which must be 1 (dJ), 2 (dH) or 3 (both)");
  if (batch < 0) return fail(NFM_E_BADARG, "negative batch");
  Args a;
  a.in(0, jac, jac_stride, true);
  a.in(1, hess, hess_stride, true);
  a.in(2, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  if (!fused_shape_built(k, d) || (mode == 1 && k > 3)) {  // the shapes the forward runs on matmul_rt_kernel
    t_last_path_tma = 0;
    reset_launch_record();
    const int rc = dtype == NFM_F32
                       ? sym_matmul_backward_rt<float>(k, d, mode, which, batch, jac, jac_stride, hess, hess_stride, grad, grad_stride,
                                                       out, out_stride, s)
                       : sym_matmul_backward_rt<double>(k, d, mode, which, batch, jac, jac_stride, hess, hess_stride, grad,
                                                        grad_stride, out, out_stride, s);
    if (rc) set_error("sym_matmul_backward kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
    return rc;
  }
  if (dtype == NFM_F32) {
    if (which == 1) return finish(sym_matmul_backward_impl<float, 1>(k, d, mode, a.p, s));
    if (which == 2) return finish(sym_matmul_backward_impl<float, 2>(k, d, mode, a.p, s));
    return finish(sym_matmul_backward_impl<float, 3>(k, d, mode, a.p, s));
  }
  if (which == 1) return finish(sym_matmul_backward_impl<double, 1>(k, d, mode, a.p, s));
  if (which == 2) return finish(sym_matmul_backward_impl<double, 2>(k, d, mode, a.p, s));
  return finish(sym_matmul_backward_impl<double, 3>(k, d, mode, a.p, s));
}

int nfm_sym_outer_backward(int dtype, int n, int64_t batch, const void* vec, int64_t vec_stride, const void* grad,
                           int64_t grad_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, vec, vec_stride, true);
  a.in(1, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? sym_outer_backward_impl<float>(n, a.p, s) : sym_outer_backward_impl<double>(n, a.p, s));
}

int nfm_sym_to_full_backward(int dtype, int n, int64_t batch, const void* grad, int64_t grad_stride, void* out,
                             int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? sym_to_full_backward_impl<float>(n, a.p, s) : sym_to_full_backward_impl<double>(n, a.p, s));
}

int nfm_batch_det_backward(int dtype, int n, int64_t batch, const void* mat, int64_t mat_stride, const void* grad,
                           int64_t grad_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  Args a;
  a.in(0, mat, mat_stride, true);
  a.in(1, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? batch_det_backward_impl<float>(n, a.p, s) : batch_det_backward_impl<double>(n, a.p, s));
}

int nfm_batch_inv_backward(int dtype, int n, int sym, int64_t batch, const void* inv, int64_t inv_stride, const void* grad,
                           int64_t grad_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (sym != 0 && sym != 1) return fail(NFM_E_UNSUPPORTED, "sym must be 0 or 1");
  Args a;
  a.in(0, inv, inv_stride, true);
  a.in(1, grad, grad_stride, true);
  a.out(out, out_stride);
  if (a.rc) return a.rc;
  a.p.batch = batch;
  auto s = static_cast<cudaStream_t>(stream);
  return finish(dtype == NFM_F32 ? batch_inv_backward_impl<float>(n, sym, a.p, s) : batch_inv_backward_impl<double>(n, sym, a.p, s));
}

int nfm_batch_outer(int dtype, int m, int n, int k, int order, int sym, int sign, int64_t batch, const void* u, int64_t u_stride,
                    const void* w, int64_t w_stride, void* out, int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) return fail(NFM_E_UNSUPPORTED, "dtype must be NFM_F32 or NFM_F64");
  if (m < 1 || n < 1 || k < 1) return fail(NFM_E_BADARG, "matrix shape must be positive");
  if (order != 0 && order != 1) return fail(NFM_E_UNSUPPORTED, "order must be 0 (U W^T) or 1 (U^T W)");
  if (sym != 0 && sym != 1) return fail(NFM_E_UNSUPPORTED, "sym must be 0 or 1");
  if (sym && m != n) return fail(NFM_E_UNSUPPORTED, "sym needs a square result");
  if (sign != 1 && sign != -1) return fail(NFM_E_BADARG, "sign must be +1 or -1");
  if (batch < 0) return fail(NFM_E_BADARG, "negative batch");
  auto s = static_cast<cudaStream_t>(stream);
  if (m == n && n <= NFM_MAX_N && k <= 4) {  // register kernels through the TMA pipeline
    Args a;
    a.in(0, u, u_stride, true);
    a.in(1, w, w_stride, true);
    a.out(out, out_stride);
    if (a.rc) return a.rc;
    a.p.batch = batch;
    a.p.flags = (sign < 0 ? 1 : 0) | (order ? kFlagRightDivision : 0) | (sym ? 8 : 0);  // kFlagOuterNegate, kFlagOuterSym
    if (k <= 2)
      return finish(dtype == NFM_F32 ? batch_outer_k12_impl<float>(n, k, a.p, s) : batch_outer_k12_impl<double>(n, k, a.p, s));
    return finish(dtype == NFM_F32 ? batch_outer_k34_impl<float>(n, k, a.p, s) : batch_outer_k34_impl<double>(n, k, a.p, s));
  }
  if (u == nullptr || w == nullptr || out == nullptr) return fail(NFM_E_BADARG, "NULL operand");
  if (u_stride < 0 || w_stride < 0 || out_stride < 0) return fail(NFM_E_BADARG, "negative batch stride");
  t_last_path_tma = 0;
  reset_launch_record();
  int rc = dtype == NFM_F32 ? batch_outer_rt<float>(m, n, k, order, sym, sign, batch, u, u_stride, w, w_stride, out, out_stride, s)
                            : batch_outer_rt<double>(m, n, k, order, sym, sign, batch, u, u_stride, w, w_stride, out, out_stride, s);
  if (rc) set_error("outer kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

int nfm_batch_tsolve(int dtype, int n, int k, int right, int algo, int64_t batch, const void* mat, int64_t a_stride, const void* b,
                     int64_t b_stride, void* out, int64_t out_stride, void* stream) {
  int rc = NFM_OK;
  if (!check_common(dtype, n, batch, rc)) return rc;
  if (k < 1) return fail(NFM_E_BADARG, "k must be >= 1");
  if (right != 0 && right != 1) return fail(NFM_E_UNSUPPORTED, "right must be 0 (A^-T B) or 1 (B A^-T)");
  if (algo == NFM_ALGO_AUTO) algo = NFM_ALGO_LU;
  if (algo != NFM_ALGO_LU && algo != NFM_ALGO_LDL) return fail(NFM_E_UNSUPPORTED, "batch_tsolve: algo must be LU or LDL");
  if (mat == nullptr || b == nullptr || out == nullptr) return fail(NFM_E_BADARG, "NULL operand");
  if (a_stride < 0 || b_stride < 0 || out_stride < 0) return fail(NFM_E_BADARG, "negative batch stride");
  // one right-hand side: a record of n either way, and A^-T b is the right division of one row
  // (B A^-T = (A^-1 B^T)^T the left division of one column)
  if (k == 1)
    return right ? nfm_batch_solve(dtype, n, 1, algo, batch, mat, a_stride, b, b_stride, out, out_stride, stream)
                 : nfm_batch_rsolve(dtype, n, 1, algo, batch, mat, a_stride, b, b_stride, out, out_stride, stream);
  auto s = static_cast<cudaStream_t>(stream);
  if (k <= 4) {  // the register kernels of nfm_batch_solve with kFlagTransposeA
    Args a;
    a.in(0, mat, a_stride, true);
    a.in(1, b, b_stride, true);
    a.out(out, out_stride);
    if (a.rc) return a.rc;
    a.p.batch = batch;
    a.p.flags = kFlagTransposeA | (right ? kFlagRightDivision : 0);
    if (algo == NFM_ALGO_LDL)
      return finish(dtype == NFM_F32 ? batch_solvek_ldl_impl<float>(n, k, a.p, s) : batch_solvek_ldl_impl<double>(n, k, a.p, s));
    return finish(dtype == NFM_F32 ? batch_solvek_lu_impl<float>(n, k, a.p, s) : batch_solvek_lu_impl<double>(n, k, a.p, s));
  }
  const int chol = algo == NFM_ALGO_LDL, mode = right | 2;  // bit 1: solve with A^T (kRightTransposeA)
  rc = dtype == NFM_F32 ? batch_solve_many<float>(n, k, chol, mode, batch, mat, a_stride, b, b_stride, out, out_stride, s)
                        : batch_solve_many<double>(n, k, chol, mode, batch, mat, a_stride, b, b_stride, out, out_stride, s);
  if (rc) set_error("solve kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

int nfm_batch_tmatvec(int dtype, int m, int n, int64_t batch, const void* mat, int64_t mat_stride, const void* vec,
                      int64_t vec_stride, void* out, int64_t out_stride, void* stream) {
  if (dtype != NFM_F32 && dtype != NFM_F64) return fail(NFM_E_UNSUPPORTED, "dtype must be NFM_F32 or NFM_F64");
  if (m < 1 || n < 1) return fail(NFM_E_BADARG, "matrix shape must be positive");
  if (batch < 0) return fail(NFM_E_BADARG, "negative batch");
  auto s = static_cast<cudaStream_t>(stream);
  if (m == n && n <= NFM_MAX_N) {
    Args a;
    a.in(0, mat, mat_stride, true);
    a.in(1, vec, vec_stride, true);
    a.out(out, out_stride);
    if (a.rc) return a.rc;
    a.p.batch = batch;
    return finish(dtype == NFM_F32 ? batch_tmatvec_impl<float>(n, a.p, s) : batch_tmatvec_impl<double>(n, a.p, s));
  }
  if (mat == nullptr || vec == nullptr || out == nullptr) return fail(NFM_E_BADARG, "NULL operand");
  if (mat_stride < 0 || vec_stride < 0 || out_stride < 0) return fail(NFM_E_BADARG, "negative batch stride");
  t_last_path_tma = 0;
  reset_launch_record();
  int rc = dtype == NFM_F32 ? batch_matvec_rt<float>(m, n, 1, batch, mat, mat_stride, vec, vec_stride, out, out_stride, s)
                            : batch_matvec_rt<double>(m, n, 1, batch, mat, mat_stride, vec, vec_stride, out, out_stride, s);
  if (rc) set_error("matvec kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

}  // extern "C"
