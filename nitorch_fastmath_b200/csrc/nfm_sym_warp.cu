// NFM_ALGO_WARP entry for one scalar type (-DNFM_SCALAR): sub-warp cooperative
// shuffle solve for packed N = 5..10 (nfm_warp.cuh); anything it does not cover
// (ragged remainder, broadcast / strided / unaligned operands) goes to the
// thread-per-matrix LDL^T kernels.
#include "nfm_impl.cuh"
#include "nfm_warp.cuh"

namespace nfm {

template <typename T>
int sym_solve_warp(int n, const KParams& p0, cudaStream_t s) {
  KParams p = p0;
  const int nn = packed_len(n);
  bool ok = n >= 5 && n <= NFM_MAX_N && p.out_stride == n && aligned16(p.out) && p.in[0].stride == nn &&
            aligned16(p.in[0].ptr) && p.in[1].stride == n && aligned16(p.in[1].ptr);
  if ((p.present & 4) && (p.in[2].stride != n || !aligned16(p.in[2].ptr))) ok = false;
  if (elem_stride(p.out_estride) != 1 || elem_stride(p.in[0].estride) != 1 || elem_stride(p.in[1].estride) != 1 ||
      ((p.present & 4) && elem_stride(p.in[2].estride) != 1))
    ok = false;
  i64 done = 0;
  if (ok) {
    int rc = 0;
    switch (n) {
      case 5: rc = launch_warp_solve<T, 5>(p, s, &done); break;
      case 6: rc = launch_warp_solve<T, 6>(p, s, &done); break;
      case 7: rc = launch_warp_solve<T, 7>(p, s, &done); break;
      case 8: rc = launch_warp_solve<T, 8>(p, s, &done); break;
      case 9: rc = launch_warp_solve<T, 9>(p, s, &done); break;
      case 10: rc = launch_warp_solve<T, 10>(p, s, &done); break;
    }
    if (rc != 0) {
      set_error("warp solve kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
      return rc;
    }
    t_last_path_tma = done > 0 ? 2 : 0;
    if (done == p.batch) return NFM_OK;
    p.in[0].ptr = static_cast<const T*>(p.in[0].ptr) + done * nn;
    p.in[1].ptr = static_cast<const T*>(p.in[1].ptr) + done * n;
    if (p.present & 4) p.in[2].ptr = static_cast<const T*>(p.in[2].ptr) + done * n;
    p.out = static_cast<T*>(p.out) + done * n;
    p.batch -= done;
  }
  const int warp_flag = t_last_path_tma;
  const int rc = sym_solve_part1<T>(n, p, s);
  if (warp_flag == 2) {  // the bulk went to the sub-warp kernel, not the tile launch of the remainder
    t_last_path_tma = 2;
    reset_launch_record();
  }
  return rc;
}

template int sym_solve_warp<NFM_SCALAR>(int, const KParams&, cudaStream_t);

}  // namespace nfm
