// tune_main.cu -- development tool (not part of the library): sweeps the tile
// geometry <THREADS, MPT, STAGES, SEG> of tile_kernel for the headline ops and
// prints achieved GB/s per configuration.   make tune && ./nfm_tune
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <array>
#include <vector>

#include "nfm_dense_ops.cuh"
#include "nfm_pipeline.cuh"
#include "nfm_sym_ops.cuh"

namespace nfm {
std::atomic<unsigned long long> g_launch_count{0};
thread_local int t_last_path_tma = 0;
thread_local long long t_last_launch[8] = {};
void set_error(const char*, ...) {}
const DeviceInfo& device_info() {
  static DeviceInfo d{};
  if (d.sm_count == 0) {
    cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, 0);
    cudaDeviceGetAttribute(&d.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, 0);
  }
  return d;
}
int current_device() { return 0; }
bool pdl_enabled() { return true; }
bool g_balance = true;
bool balance_enabled() { return g_balance; }
}  // namespace nfm

using namespace nfm;

template <typename T>
__global__ void fill_kernel(T* p, i64 n, int rec, int ndiag, T diag, T off) {
  for (i64 i = i64(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += i64(gridDim.x) * blockDim.x) {
    const int k = int(i % rec);
    // dense records: diagonal at k % (ndiag+1) == 0 when ndiag > 0 means row-major n x n
    bool is_diag = ndiag < 0 ? (k % (-ndiag + 1) == 0) : (k < ndiag);
    p[i] = (is_diag ? diag : off) + T(1e-3) * T(i % 7);
  }
}

struct Buffers {
  void *in0, *in1, *out;
  i64 batch;
};

template <class Op, int THREADS, int MPT, int STAGES, bool SEG>
void run_config(const char* name, const Buffers& b, int alg_bytes) {
  using T = typename Op::scalar;
  KParams p{};
  p.in[0].ptr = b.in0;
  p.in[0].stride = Op::kLen0;
  p.present = 1;
  if (Op::kUse & 2) {
    p.in[1].ptr = b.in1;
    p.in[1].stride = Op::kLen1;
    p.present |= 2;
  }
  p.out = b.out;
  p.out_stride = Op::kOut;
  constexpr int TILE = THREADS * MPT;
  p.batch = b.batch;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  int rc = 0;
  for (int i = 0; i < 3 && rc == 0; ++i) rc = launch_tile<Op, THREADS, MPT, STAGES, SEG>(p, 0);
  if (rc != 0) {
    printf("%-22s T=%4d thr=%3d st=%d seg=%d : launch failed rc=%d\n", name, TILE, THREADS, STAGES, int(SEG), rc);
    cudaGetLastError();
    return;
  }
  cudaDeviceSynchronize();
  const int reps = 20;
  cudaEventRecord(e0);
  for (int i = 0; i < reps; ++i) launch_tile<Op, THREADS, MPT, STAGES, SEG>(p, 0);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  const double us = ms * 1e3 / reps;
  const double gbs = double(p.batch) * alg_bytes / (us * 1e-6) / 1e9;
  printf("%-22s T=%4d thr=%3d st=%d seg=%d : %8.1f us  %7.1f GB/s  %6.2f Gmat/s\n", name, TILE, THREADS, STAGES, int(SEG), us,
         gbs, p.batch / (us * 1e-6) / 1e9);
  fflush(stdout);
}

// small-batch variant: the big buffers are cut into `slices` sub-batches that are
// visited round-robin, so that consecutive launches never find their data in L2
template <class Op, int THREADS, int MPT, int STAGES, bool SEG>
void run_sliced(const char* name, const Buffers& b, int alg_bytes, i64 sub) {
  using T = typename Op::scalar;
  const i64 pitch = (sub + 1023) / 1024 * 1024;  // slices start 16-byte aligned for any sub
  const int slices = int(b.batch / pitch);
  std::vector<KParams> ps(slices);
  for (int s = 0; s < slices; ++s) {
    KParams p{};
    p.in[0].ptr = static_cast<const T*>(b.in0) + i64(s) * pitch * Op::kLen0;
    p.in[0].stride = Op::kLen0;
    p.present = 1;
    if (Op::kUse & 2) {
      p.in[1].ptr = static_cast<const T*>(b.in1) + i64(s) * pitch * Op::kLen1;
      p.in[1].stride = Op::kLen1;
      p.present |= 2;
    }
    p.out = static_cast<T*>(b.out) + i64(s) * pitch * Op::kOut;
    p.out_stride = Op::kOut;
    p.batch = sub;
    ps[s] = p;
  }
  constexpr int TILE = THREADS * MPT;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  for (int i = 0; i < slices; ++i) launch_tile<Op, THREADS, MPT, STAGES, SEG>(ps[i], 0);
  cudaDeviceSynchronize();
  const int reps = slices > 1 ? 10 * slices : 10;
  cudaEventRecord(e0);
  for (int i = 0; i < reps; ++i) launch_tile<Op, THREADS, MPT, STAGES, SEG>(ps[i % slices], 0);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  const double us = ms * 1e3 / reps;
  printf("%-18s batch %8lld T=%4d thr=%3d st=%d : %7.2f us  %7.1f GB/s\n", name, sub, TILE, THREADS, STAGES, us,
         double(sub) * alg_bytes / (us * 1e-6) / 1e9);
  fflush(stdout);
}

template <typename T>
__global__ void diff_kernel(const T* a, const T* b, i64 n, unsigned long long* bad) {
  for (i64 i = i64(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += i64(gridDim.x) * blockDim.x)
    if (!(a[i] == b[i]) && !(a[i] != a[i] && b[i] != b[i])) atomicAdd(bad, 1ull);
}

// pool_kernel configuration; checks its output bit for bit against tile_kernel's
template <class Op, int MAXW, int MPT, bool SEG>
void run_pool(const char* name, const Buffers& b, int alg_bytes, int W, int NBUF) {
  using T = typename Op::scalar;
  KParams p{};
  p.in[0].ptr = b.in0;
  p.in[0].stride = Op::kLen0;
  p.present = 1;
  if (Op::kUse & 2) {
    p.in[1].ptr = b.in1;
    p.in[1].stride = Op::kLen1;
    p.present |= 2;
  }
  p.out_stride = Op::kOut;
  p.batch = b.batch;
  const int buf = PoolGeom<Op, MPT, SEG>::buf_bytes(p.present);
  if (W == 0) PoolTune<Op>::geometry(buf, device_info().max_smem_optin, W, NBUF);  // the rule
  if (W > MAXW || NBUF <= W || NBUF * (buf + 12) + 16 > device_info().max_smem_optin) return;
  // reference result from the tile kernel into a scratch buffer
  static T* ref = nullptr;
  static const void* ref_for = nullptr;
  int rc = 0;
  if (ref_for != b.in0) {
    if (ref) cudaFree(ref);
    cudaMalloc(&ref, size_t(p.batch) * Op::kOut * sizeof(T));
    p.out = ref;
    using Tn = Tune<Op>;
    rc = launch_tile<Op, Tn::kThreads, Tn::kMpt, Tn::kStages, Tn::kSeg>(p, 0);
    ref_for = b.in0;
  }
  p.out = b.out;
  cudaMemset(b.out, 0xff, size_t(p.batch) * Op::kOut * sizeof(T));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  for (int i = 0; i < 3 && rc == 0; ++i) rc = launch_pool<Op, MAXW, MPT, SEG>(p, W, NBUF, 0);
  cudaError_t err = cudaDeviceSynchronize();
  if (rc != 0 || err != cudaSuccess) {
    printf("%-20s pool maxw=%2d W=%2d mpt=%d nbuf=%2d seg=%d : failed rc=%d %s (%s)\n", name, MAXW, W, MPT, NBUF, int(SEG), rc,
           cudaGetErrorString(err), cudaGetErrorName(err));
    cudaGetLastError();
    return;
  }
  unsigned long long* bad;
  cudaMalloc(&bad, 8);
  cudaMemset(bad, 0, 8);
  diff_kernel<T><<<1184, 256>>>(ref, static_cast<const T*>(b.out), p.batch * Op::kOut, bad);
  unsigned long long hbad = 0;
  cudaMemcpy(&hbad, bad, 8, cudaMemcpyDeviceToHost);
  const int reps = 10;
  cudaEventRecord(e0);
  for (int i = 0; i < reps; ++i) launch_pool<Op, MAXW, MPT, SEG>(p, W, NBUF, 0);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  const double us = ms * 1e3 / reps;
  printf("%-20s pool maxw=%2d W=%2d mpt=%d nbuf=%2d seg=%d smem=%3dK : %8.1f us  %7.1f GB/s  mismatches %llu\n", name, MAXW, W, MPT,
         NBUF, int(SEG), (NBUF * (buf + 12) + 16) >> 10, us, double(p.batch) * alg_bytes / (us * 1e-6) / 1e9, hbad);
  fflush(stdout);
  cudaFree(bad);
}

// rule + a grid of (warps, buffers) for two register budgets
template <class Op>
void pool_sweep(const char* name, const Buffers& buf, int alg_bytes) {
  constexpr bool SEG = Tune<Op>::kSeg;
  constexpr int RW = PoolTune<Op>::kMaxW;
  run_pool<Op, RW, 1, SEG>(name, buf, alg_bytes, 0, 0);
  printf("   ^ rule\n");
  const int nmax = (device_info().max_smem_optin - 512) / (PoolGeom<Op, 1, SEG>::buf_bytes(Op::kUse & 3) + 12);
  for (int w : {4, 5, 6, 7, 8})
    for (int nb : {w + 1, w + 2, w + 3, w + 5, nmax})
      if (nb <= nmax && nb <= 32) run_pool<Op, 8, 1, SEG>(name, buf, alg_bytes, w, nb);
  for (int w : {10, 12})
    for (int nb : {w + 2, w + 4, w + 6, nmax})
      if (nb <= nmax && nb <= 32) run_pool<Op, 12, 1, SEG>(name, buf, alg_bytes, w, nb);
  for (int w : {14, 16})
    for (int nb : {w + 4, w + 8, nmax})
      if (nb <= nmax && nb <= 32) run_pool<Op, 16, 1, SEG>(name, buf, alg_bytes, w, nb);
}

template <typename T>
Buffers make(i64 batch, int len0, int ndiag0, int len1, int lout) {
  Buffers b{};
  b.batch = batch;
  cudaMalloc(&b.in0, size_t(batch) * len0 * sizeof(T));
  cudaMalloc(&b.in1, size_t(batch) * (len1 > 0 ? len1 : 1) * sizeof(T));
  cudaMalloc(&b.out, size_t(batch) * lout * sizeof(T));
  fill_kernel<T><<<1184, 256>>>(static_cast<T*>(b.in0), batch * len0, len0, ndiag0, T(8), T(0.25));
  if (len1 > 0) fill_kernel<T><<<1184, 256>>>(static_cast<T*>(b.in1), batch * len1, len1, 0, T(1), T(1));
  cudaDeviceSynchronize();
  return b;
}

void release(Buffers& b) {
  cudaFree(b.in0);
  cudaFree(b.in1);
  cudaFree(b.out);
}

#define CFG(OP, NAME, THR, MPT, ST, SEG, BYTES) run_config<OP, THR, MPT, ST, SEG>(NAME, buf, BYTES)

int main(int argc, char** argv) {
  // usage: nfm_tune [substring]   -- run only the blocks whose name contains it
  const char* only = argc > 1 ? argv[1] : "";
  auto want = [&](const char* n) { return only[0] == 0 || strstr(n, only) != nullptr; };

  // The three sweeps that produced the Tune<> rule are recorded in
  // profiles/r1_tile_geometry_sweep.txt; this list is the regression check:
  // the geometry the rule picks for each headline op next to its neighbours.
  if (want("solve3")) {
    using Op = SymSolveOp<float, 3, NFM_LAYOUT_SYM, 0>;
    Buffers buf = make<float>(256ll * 256 * 256, 6, 3, 3, 3);
    CFG(Op, "sym_solve3", 512, 2, 3, false, 48);   // rule
    CFG(Op, "sym_solve3", 256, 2, 3, false, 48);
    CFG(Op, "sym_solve3", 256, 4, 4, false, 48);
    CFG(Op, "sym_solve3", 1024, 1, 3, false, 48);
    release(buf);
  }
#ifndef NFM_TUNE_MIN
  if (want("small")) {
    using Op = SymSolveOp<float, 3, NFM_LAYOUT_SYM, 0>;
    Buffers buf = make<float>(256ll * 256 * 256, 6, 3, 3, 3);
    for (i64 sub : {i64(1) << 19, i64(1) << 20, i64(1) << 21, i64(1) << 22}) {
      run_sliced<Op, 512, 2, 3, false>("solve3", buf, 48, sub);
      run_sliced<Op, 256, 2, 3, false>("solve3", buf, 48, sub);
      run_sliced<Op, 512, 1, 3, false>("solve3", buf, 48, sub);
      run_sliced<Op, 256, 1, 4, false>("solve3", buf, 48, sub);
      run_sliced<Op, 128, 2, 4, false>("solve3", buf, 48, sub);
      run_sliced<Op, 256, 1, 3, false>("solve3", buf, 48, sub);
    }
    release(buf);
  }
  if (want("balance")) {
    // equal-tile scheduling on / off for mid-size launches (a multi-GPU slab, config 1)
    using Op = SymSolveOp<float, 3, NFM_LAYOUT_SYM, 0>;
    Buffers buf = make<float>(256ll * 256 * 256, 6, 3, 3, 3);
    for (i64 sub : {i64(1000000), i64(1) << 20, i64(2000003), i64(1) << 21, i64(1) << 22, i64(1) << 23}) {
      for (int bal = 0; bal < 2; ++bal) {
        g_balance = bal;
        printf("balance=%d ", bal);
        run_sliced<Op, 512, 2, 3, false>("solve3", buf, 48, sub);
        printf("balance=%d ", bal);
        run_sliced<Op, 256, 2, 3, false>("solve3", buf, 48, sub);
        printf("balance=%d ", bal);
        run_sliced<Op, 256, 1, 3, false>("solve3", buf, 48, sub);
        printf("balance=%d ", bal);
        run_sliced<Op, 128, 2, 4, false>("solve3", buf, 48, sub);
        printf("balance=%d ", bal);
        run_sliced<Op, 1024, 1, 3, false>("solve3", buf, 48, sub);
        printf("balance=%d ", bal);
        run_sliced<Op, 512, 1, 4, false>("solve3", buf, 48, sub);
        printf("balance=%d ", bal);
        run_sliced<Op, 256, 2, 4, false>("solve3", buf, 48, sub);
      }
    }
    g_balance = true;
    release(buf);
    using Op6 = SymSolveOp<float, 6, NFM_LAYOUT_SYM, NFM_ALGO_AUTO>;
    Buffers b6 = make<float>(192ll * 192 * 192, 21, 6, 6, 6);
    for (i64 sub : {i64(884736), i64(1769472)}) {   // 192^3 / 8, / 4
      for (int bal = 0; bal < 2; ++bal) {
        g_balance = bal;
        printf("balance=%d ", bal);
        run_sliced<Op6, 512, 1, 2, false>("solve6", b6, 132, sub);
        printf("balance=%d ", bal);
        run_sliced<Op6, 256, 1, 2, false>("solve6", b6, 132, sub);
        printf("balance=%d ", bal);
        run_sliced<Op6, 256, 1, 3, false>("solve6", b6, 132, sub);
        printf("balance=%d ", bal);
        run_sliced<Op6, 128, 1, 3, false>("solve6", b6, 132, sub);
      }
    }
    g_balance = true;
    release(b6);
    using Oi6 = SymInvertOp<float, 6, NFM_ALGO_AUTO, false>;
    Buffers bi6 = make<float>(192ll * 192 * 192, 21, 6, 0, 21);
    for (i64 sub : {i64(884736), i64(1769472)}) {
      for (int bal = 0; bal < 2; ++bal) {
        g_balance = bal;
        printf("balance=%d ", bal);
        run_sliced<Oi6, 384, 1, 2, false>("invert6", bi6, 168, sub);
        printf("balance=%d ", bal);
        run_sliced<Oi6, 256, 1, 2, false>("invert6", bi6, 168, sub);
        printf("balance=%d ", bal);
        run_sliced<Oi6, 128, 1, 3, false>("invert6", bi6, 168, sub);
        printf("balance=%d ", bal);
        run_sliced<Oi6, 128, 1, 2, false>("invert6", bi6, 168, sub);
      }
    }
    g_balance = true;
    release(bi6);
    using Op10 = SymSolveOp<float, 10, NFM_LAYOUT_SYM, NFM_ALGO_AUTO>;
    Buffers b10 = make<float>(160ll * 160 * 160, 55, 10, 10, 10);
    for (i64 sub : {i64(512000), i64(1024000)}) {   // 160^3 / 8, / 4
      for (int bal = 0; bal < 2; ++bal) {
        g_balance = bal;
        printf("balance=%d ", bal);
        run_sliced<Op10, 256, 1, 2, false>("solve10", b10, 300, sub);
        printf("balance=%d ", bal);
        run_sliced<Op10, 128, 1, 2, false>("solve10", b10, 300, sub);
        printf("balance=%d ", bal);
        run_sliced<Op10, 128, 1, 3, false>("solve10", b10, 300, sub);
      }
    }
    g_balance = true;
    release(b10);
  }
  // geometry sweep of the headline light ops over slab sizes (1, 1/2, 1/4, 1/8 of the config)
#define GEO(OP, NAME, THR, MPT, ST, BYTES)                                  \
  for (i64 sub : subs)                                                       \
    if (size_t(ST) * THR * MPT * in_b + 2 * size_t(THR) * MPT * out_b <= 225 * 1024) \
      run_sliced<OP, THR, MPT, ST, false>(NAME, buf, BYTES, sub);
#define GEOSET(OP, NAME, BYTES)                                                                      \
  GEO(OP, NAME, 128, 1, 2, BYTES) GEO(OP, NAME, 128, 1, 3, BYTES) GEO(OP, NAME, 128, 1, 4, BYTES)    \
  GEO(OP, NAME, 128, 2, 3, BYTES) GEO(OP, NAME, 128, 2, 4, BYTES) GEO(OP, NAME, 256, 1, 2, BYTES)    \
  GEO(OP, NAME, 256, 1, 3, BYTES) GEO(OP, NAME, 256, 1, 4, BYTES) GEO(OP, NAME, 256, 2, 2, BYTES)    \
  GEO(OP, NAME, 256, 2, 3, BYTES) GEO(OP, NAME, 256, 2, 4, BYTES) GEO(OP, NAME, 512, 1, 2, BYTES)    \
  GEO(OP, NAME, 512, 1, 3, BYTES) GEO(OP, NAME, 512, 1, 4, BYTES) GEO(OP, NAME, 512, 2, 2, BYTES)    \
  GEO(OP, NAME, 512, 2, 3, BYTES) GEO(OP, NAME, 768, 1, 3, BYTES) GEO(OP, NAME, 1024, 1, 2, BYTES)   \
  GEO(OP, NAME, 1024, 1, 3, BYTES)
  if (want("geo_solve3")) {
    using Op = SymSolveOp<float, 3, NFM_LAYOUT_SYM, 0>;
    const i64 full = 256ll * 256 * 256;
    Buffers buf = make<float>(full, 6, 3, 3, 3);
    const i64 subs[] = {1000000, full / 8, full / 4, full / 2, full};
    const size_t in_b = 36, out_b = 12;
    GEOSET(Op, "solve3", 48)
    release(buf);
  }
  if (want("geo_matvec3")) {
    using Op = SymMatvecOp<float, 3, NFM_LAYOUT_SYM>;
    const i64 full = 256ll * 256 * 256;
    Buffers buf = make<float>(full, 6, 3, 3, 3);
    const i64 subs[] = {1000000, full / 8, full};
    const size_t in_b = 36, out_b = 12;
    GEOSET(Op, "matvec3", 48)
    release(buf);
  }
  if (want("geo_solve6")) {
    using Op = SymSolveOp<float, 6, NFM_LAYOUT_SYM, NFM_ALGO_AUTO>;
    const i64 full = 192ll * 192 * 192;
    Buffers buf = make<float>(full, 21, 6, 6, 6);
    const i64 subs[] = {full / 8, full / 4, full / 2, full};
    const size_t in_b = 108, out_b = 24;
    GEOSET(Op, "solve6", 132)
    release(buf);
  }
  if (want("geo_invert6")) {
    using Op = SymInvertOp<float, 6, NFM_ALGO_AUTO, false>;
    const i64 full = 192ll * 192 * 192;
    Buffers buf = make<float>(full, 21, 6, 0, 21);
    const i64 subs[] = {full / 8, full / 4, full / 2, full};
    const size_t in_b = 84, out_b = 84;
    GEOSET(Op, "invert6", 168)
    release(buf);
  }
  if (want("geo_solve10")) {
    using Op = SymSolveOp<float, 10, NFM_LAYOUT_SYM, NFM_ALGO_AUTO>;
    const i64 full = 160ll * 160 * 160;
    Buffers buf = make<float>(full, 55, 10, 10, 10);
    const i64 subs[] = {full / 8, full / 4, full / 2, full};
    const size_t in_b = 260, out_b = 40;
    GEOSET(Op, "solve10", 300)
    release(buf);
  }
  if (want("geo_solve4")) {
    using Op = SymSolveOp<float, 4, NFM_LAYOUT_SYM, 0>;
    const i64 full = 1ll << 24;
    Buffers buf = make<float>(full, 10, 4, 4, 4);
    const i64 subs[] = {full / 8, full};
    const size_t in_b = 56, out_b = 16;
    GEOSET(Op, "solve4", 72)
    release(buf);
  }
  if (want("geo_solve3d")) {
    using Op = SymSolveOp<double, 3, NFM_LAYOUT_SYM, 0>;
    const i64 full = 1ll << 24;
    Buffers buf = make<double>(full, 6, 3, 3, 3);
    const i64 subs[] = {full / 8, full};
    const size_t in_b = 72, out_b = 24;
    GEOSET(Op, "solve3 f64", 96)
    release(buf);
  }
#define TILE_RULE(OP, NAME, BYTES) \
  run_config<OP, Tune<OP>::kThreads, Tune<OP>::kMpt, Tune<OP>::kStages, Tune<OP>::kSeg>(NAME " tile-rule", buf, BYTES)
#define POOLBLOCK(TAG, OP, T, NAME, BATCH, L0, ND, L1, LO, BYTES) \
  if (want(TAG)) {                                                 \
    Buffers buf = make<T>(BATCH, L0, ND, L1, LO);                  \
    TILE_RULE(OP, NAME, BYTES);                                    \
    pool_sweep<OP>(NAME, buf, BYTES);                              \
    release(buf);                                                  \
  }
  using InvD8 = BatchInvOp<double, 8, NFM_ALGO_AUTO>;
  using InvD10 = BatchInvOp<double, 10, NFM_ALGO_AUTO>;
  using InvD6 = BatchInvOp<double, 6, NFM_ALGO_AUTO>;
  using InvF10 = BatchInvOp<float, 10, NFM_ALGO_AUTO>;
  using InvF8 = BatchInvOp<float, 8, NFM_ALGO_AUTO>;
  using DetD10 = BatchDetOp<double, 10>;
  using SolD10 = BatchSolveOp<double, 10, NFM_ALGO_LU>;
  using SolD8 = BatchSolveOp<double, 8, NFM_ALGO_LU>;
  using SolF10 = BatchSolveOp<float, 10, NFM_ALGO_LU>;
  using SymLuF10 = SymSolveOp<float, 10, NFM_LAYOUT_SYM, NFM_ALGO_LU>;
  using SymLuD10 = SymSolveOp<double, 10, NFM_LAYOUT_SYM, NFM_ALGO_LU>;
  using InvD5 = BatchInvOp<double, 5, NFM_ALGO_AUTO>;
  using InvD4 = BatchInvOp<double, 4, NFM_ALGO_AUTO>;
  using InvF7 = BatchInvOp<float, 7, NFM_ALGO_AUTO>;
  using InvF6 = BatchInvOp<float, 6, NFM_ALGO_AUTO>;
  using InvF5 = BatchInvOp<float, 5, NFM_ALGO_AUTO>;
  using SolD6 = BatchSolveOp<double, 6, NFM_ALGO_LU>;
  POOLBLOCK("pool_inv5d", InvD5, double, "inv5 f64", 8ll << 20, 25, -5, 0, 25, 400)
  POOLBLOCK("pool_inv4d", InvD4, double, "inv4 f64", 16ll << 20, 16, -4, 0, 16, 256)
  POOLBLOCK("pool_inv7f", InvF7, float, "inv7 f32", 8ll << 20, 49, -7, 0, 49, 392)
  POOLBLOCK("pool_inv6f", InvF6, float, "inv6 f32", 8ll << 20, 36, -6, 0, 36, 288)
  POOLBLOCK("pool_inv5f", InvF5, float, "inv5 f32", 8ll << 20, 25, -5, 0, 25, 200)
  POOLBLOCK("pool_solve6d", SolD6, double, "solve6 f64", 8ll << 20, 36, -6, 6, 6, 384)
  POOLBLOCK("pool_inv8d", InvD8, double, "inv8 f64", 4ll << 20, 64, -8, 0, 64, 1024)
  POOLBLOCK("pool_inv10d", InvD10, double, "inv10 f64", 4ll << 20, 100, -10, 0, 100, 1600)
  POOLBLOCK("pool_inv6d", InvD6, double, "inv6 f64", 8ll << 20, 36, -6, 0, 36, 576)
  POOLBLOCK("pool_inv10f", InvF10, float, "inv10 f32", 8ll << 20, 100, -10, 0, 100, 800)
  POOLBLOCK("pool_inv8f", InvF8, float, "inv8 f32", 8ll << 20, 64, -8, 0, 64, 512)
  POOLBLOCK("pool_det10d", DetD10, double, "det10 f64", 4ll << 20, 100, -10, 0, 1, 808)
  POOLBLOCK("pool_solve10d", SolD10, double, "solve10 f64", 4ll << 20, 100, -10, 10, 10, 960)
  POOLBLOCK("pool_solve8d", SolD8, double, "solve8 f64", 4ll << 20, 64, -8, 8, 8, 640)
  POOLBLOCK("pool_solve10f", SolF10, float, "solve10 f32", 8ll << 20, 100, -10, 10, 10, 480)
  POOLBLOCK("pool_symlu10f", SymLuF10, float, "symlu10 f32", 160ll * 160 * 160, 55, 10, 10, 10, 300)
  POOLBLOCK("pool_symlu10d", SymLuD10, double, "symlu10 f64", 160ll * 160 * 160, 55, 10, 10, 10, 600)
#ifdef NFM_TIMELINE
  if (want("timeline")) {
    // ramp / steady / tail of back-to-back launches from per-CTA %globaltimer stamps:
    // 0 = CTA start, 1 = after griddepcontrol.wait, 2 = first tile landed, 3 = CTA end
    using Op = SymSolveOp<float, 3, NFM_LAYOUT_SYM, 0>;
    Buffers buf = make<float>(256ll * 256 * 256, 6, 3, 3, 3);
    const int nl = 10;
    unsigned long long* d_tl;
    const size_t slots = size_t(nl) * 1024 * 8;
    cudaMalloc(&d_tl, slots * 8);
    cudaMemcpyToSymbol(g_timeline, &d_tl, sizeof(d_tl));
    auto run = [&](const char* label, i64 sub, auto launcher, bool dump = false) {
      const i64 pitch = (sub + 1023) / 1024 * 1024;
      const int slices = int(buf.batch / pitch);
      std::vector<KParams> ps(nl);
      for (int i = 0; i < nl; ++i) {
        const int s = i % slices;
        KParams p{};
        p.in[0].ptr = static_cast<const float*>(buf.in0) + i64(s) * pitch * 6;
        p.in[0].stride = 6;
        p.in[1].ptr = static_cast<const float*>(buf.in1) + i64(s) * pitch * 3;
        p.in[1].stride = 3;
        p.present = 3;
        p.out = static_cast<float*>(buf.out) + i64(s) * pitch * 3;
        p.out_stride = 3;
        p.batch = sub;
        p.scal1 = i;
        ps[i] = p;
      }
      for (int i = 0; i < nl; ++i) launcher(ps[i]);  // warm-up
      cudaDeviceSynchronize();
      cudaMemset(d_tl, 0, slots * 8);
      cudaDeviceSynchronize();
      cudaEvent_t e0, e1;
      cudaEventCreate(&e0);
      cudaEventCreate(&e1);
      cudaEventRecord(e0);
      for (int i = 0; i < nl; ++i) launcher(ps[i]);
      cudaEventRecord(e1);
      cudaDeviceSynchronize();
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      std::vector<unsigned long long> h(slots);
      cudaMemcpy(h.data(), d_tl, slots * 8, cudaMemcpyDeviceToHost);
      printf("== timeline %s: %lld matrices per launch, %d back-to-back launches, %.2f us per launch by events\n", label, sub, nl,
             ms * 1e3 / nl);
      printf("   launch ctas | start: first..last | dep-wait passed: first..last | first tile: first..median..last | end: first..last | prev end -> first dep-wait | dep-wait -> last end\n");
      unsigned long long prev_end = 0;
      for (int i = 0; i < nl; ++i) {
        std::vector<unsigned long long> s0, s1, s2, s3;
        for (int c = 0; c < 1024; ++c) {
          const unsigned long long* r = &h[(size_t(i) * 1024 + c) * 8];
          if (r[3] == 0) continue;
          s0.push_back(r[0]);
          s1.push_back(r[1]);
          if (r[2]) s2.push_back(r[2]);
          s3.push_back(r[3]);
        }
        if (s0.empty()) continue;
        auto srt = [](std::vector<unsigned long long>& v) { std::sort(v.begin(), v.end()); };
        srt(s0); srt(s1); srt(s2); srt(s3);
        const unsigned long long t0 = s0.front();
        auto rel = [&](unsigned long long t) { return (long long)(t - t0); };
        printf("   %2d %4zu | %6lld..%6lld | %6lld..%6lld | %6lld..%6lld..%6lld | %6lld..%6lld | %6lld | %6lld\n", i, s0.size(),
               rel(s0.front()), rel(s0.back()), rel(s1.front()), rel(s1.back()), s2.empty() ? 0 : rel(s2.front()),
               s2.empty() ? 0 : rel(s2[s2.size() / 2]), s2.empty() ? 0 : rel(s2.back()), rel(s3.front()), rel(s3.back()),
               prev_end ? (long long)(s1.front() - prev_end) : 0, (long long)(s3.back() - s1.front()));
        prev_end = s3.back();
      }
      if (dump) {
        const int i = 5;
        unsigned long long t1 = ~0ull;
        for (int c = 0; c < 1024; ++c) {
          const unsigned long long* r = &h[(size_t(i) * 1024 + c) * 8];
          if (r[3] && r[1] < t1) t1 = r[1];
        }
        std::vector<std::array<long long, 5>> rows;
        for (int c = 0; c < 1024; ++c) {
          const unsigned long long* r = &h[(size_t(i) * 1024 + c) * 8];
          if (r[3] == 0) continue;
          rows.push_back({(long long)r[4], (long long)c, (long long)r[5], (long long)(r[2] ? r[2] - t1 : 0), (long long)(r[3] - t1)});
        }
        std::sort(rows.begin(), rows.end());
        printf("   per-CTA (launch 5): sm cta tiles first_tile_ns end_ns\n");
        for (auto& r : rows) printf("   sm %3lld cta %3lld tiles %2lld first %5lld end %5lld\n", r[0], r[1], r[2], r[3], r[4]);
      }
      fflush(stdout);
    };
    for (i64 sub : {i64(1) << 21, i64(1000000)}) {
      g_balance = false;
      run("solve3 512x2 st3 (1 CTA/SM), fixed 1024 tiles", sub, [](const KParams& p) { launch_tile<Op, 512, 2, 3, false>(p, 0); });
      run("solve3 256x2 st3 (3 CTA/SM), fixed 512 tiles", sub, [](const KParams& p) { launch_tile<Op, 256, 2, 3, false>(p, 0); },
          sub == (i64(1) << 21));
      run("solve3 128x2 st4, fixed 256 tiles", sub, [](const KParams& p) { launch_tile<Op, 128, 2, 4, false>(p, 0); });
      g_balance = true;
      run("solve3 256x2 st3 (3 CTA/SM), equal tiles", sub, [](const KParams& p) { launch_tile<Op, 256, 2, 3, false>(p, 0); });
    }
    release(buf);
  }
#endif
  if (want("solve6")) {
    using Op = SymSolveOp<float, 6, NFM_LAYOUT_SYM, NFM_ALGO_AUTO>;
    using Ldl = SymSolveOp<float, 6, NFM_LAYOUT_SYM, NFM_ALGO_LDL>;
    Buffers buf = make<float>(192ll * 192 * 192, 21, 6, 6, 6);
    CFG(Op, "sym_solve6 auto", 512, 1, 2, false, 132);   // rule
    CFG(Ldl, "sym_solve6 ldl", 512, 1, 2, false, 132);
    CFG(Op, "sym_solve6 auto", 256, 2, 2, false, 132);
    CFG(Op, "sym_solve6 auto", 384, 1, 3, false, 132);
    release(buf);
  }
  if (want("invert6")) {
    using Op = SymInvertOp<float, 6, NFM_ALGO_AUTO, false>;
    Buffers buf = make<float>(192ll * 192 * 192, 21, 6, 0, 21);
    CFG(Op, "sym_invert6 auto", 384, 1, 2, false, 168);  // rule
    CFG(Op, "sym_invert6 auto", 256, 1, 2, false, 168);
    CFG(Op, "sym_invert6 auto", 512, 1, 2, false, 168);
    release(buf);
  }
  if (want("solve10")) {
    using Op = SymSolveOp<float, 10, NFM_LAYOUT_SYM, NFM_ALGO_AUTO>;
    Buffers buf = make<float>(160ll * 160 * 160, 55, 10, 10, 10);
    CFG(Op, "sym_solve10 auto", 256, 1, 2, false, 300);  // rule
    CFG(Op, "sym_solve10 auto", 128, 1, 2, false, 300);
    CFG(Op, "sym_solve10 auto", 128, 1, 3, false, 300);
    release(buf);
  }
#endif  // NFM_TUNE_MIN
  if (want("inv4d")) {
    using Op = BatchInvOp<double, 4, NFM_ALGO_AUTO>;
    Buffers buf = make<double>(16ll << 20, 16, -4, 0, 16);
    CFG(Op, "dense_inv4d", 256, 1, 3, true, 256);   // pinned (TuneFixed)
    CFG(Op, "dense_inv4d", 256, 1, 3, false, 256);  // dense layout: 8-way bank conflicts
    CFG(Op, "dense_inv4d", 128, 1, 3, true, 256);
    release(buf);
  }
  if (want("reps20")) {
    // what a 20-launch timed region costs per launch against a long one (the driver's protocol at 8 GPUs)
    using Op = SymSolveOp<float, 3, NFM_LAYOUT_SYM, 0>;
    Buffers buf = make<float>(256ll * 256 * 256, 6, 3, 3, 3);
    const i64 sub = i64(1) << 21;
    std::vector<KParams> ps(8);
    for (int s = 0; s < 8; ++s) {
      KParams p{};
      p.in[0].ptr = static_cast<const float*>(buf.in0) + i64(s) * sub * 6;
      p.in[0].stride = 6;
      p.in[1].ptr = static_cast<const float*>(buf.in1) + i64(s) * sub * 3;
      p.in[1].stride = 3;
      p.present = 3;
      p.out = static_cast<float*>(buf.out) + i64(s) * sub * 3;
      p.out_stride = 3;
      p.batch = sub;
      ps[s] = p;
    }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    for (int reps : {20, 20, 20, 200, 200, 20, 20}) {
      for (int i = 0; i < 8; ++i) launch_tile<Op, 256, 2, 2, false>(ps[i], 0);
      cudaDeviceSynchronize();
      cudaEventRecord(e0);
      for (int i = 0; i < reps; ++i) launch_tile<Op, 256, 2, 2, false>(ps[i % 8], 0);
      cudaEventRecord(e1);
      cudaEventSynchronize(e1);
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      printf("C++ loop, 2M-matrix launches, %3d in the timed region: %.2f us per launch (%.1f us total)\n", reps, ms * 1e3 / reps, ms * 1e3);
    }
    release(buf);
  }
  if (want("det4d")) {
    using Op = BatchDetOp<double, 4>;
    Buffers buf = make<double>(16ll << 20, 16, -4, 0, 1);
    CFG(Op, "dense_det4d", 128, 2, 3, true, 136);  // pinned
    CFG(Op, "dense_det4d", 256, 1, 3, true, 136);
    CFG(Op, "dense_det4d", 128, 1, 3, true, 136);
    release(buf);
  }
  if (want("solve4d")) {
    using Op = BatchSolveOp<double, 4, NFM_ALGO_LU>;
    Buffers buf = make<double>(16ll << 20, 16, -4, 4, 4);
    CFG(Op, "dense_solve4d", 128, 1, 3, true, 192);  // pinned
    CFG(Op, "dense_solve4d", 256, 1, 3, true, 192);
    CFG(Op, "dense_solve4d", 512, 1, 2, true, 192);
    release(buf);
  }
  return 0;
}
