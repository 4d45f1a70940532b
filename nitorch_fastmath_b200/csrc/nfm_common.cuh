// nfm_common.cuh -- shared device helpers: sm_100a PTX wrappers (mbarrier, 1-D
// TMA bulk copies), record <-> register movers, launch parameter block.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/nfm.h"

namespace nfm {

using i64 = long long;

// One batched operand: base pointer, batch stride in elements (0 = broadcast)
// and the stride between the elements of one record (0 is read as 1, the
// contiguous record; anything else -- e.g. coefficient-first "SoA" storage
// viewed coefficient-last -- takes the strided kernel).
struct Operand {
  const void* ptr;
  i64 stride;
  i64 estride;
};

__host__ __device__ inline i64 elem_stride(i64 estride) { return estride == 0 ? 1 : estride; }

constexpr int kMaxIn = 4;

// Launch parameter block shared by every op.
struct KParams {
  Operand in[kMaxIn];
  void* out;
  i64 out_stride;
  i64 out_estride;
  i64 batch;     // matrices handled by this launch
  int present;   // bit i set: input operand i is present
  int flags;     // op-specific
  double scal0;  // op-specific scalars (ops that declare kScalars; e.g. the
  double scal1;  //  damping and step length of the fused solve + update)
};

// KParams::flags of BatchSolveKOp: X = B A^-1 with B, X  K x N row-major (one system A^T x = b per row)
constexpr int kFlagRightDivision = 2;
// ... and, independent of the record order, solve with A^T: X = A^-T B (left) or B A^-T (right).
// The transposed solves are the gradients of lmdiv / rmdiv with respect to B.
constexpr int kFlagTransposeA = 4;

// ---------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

// make mbarrier.init visible to the async proxy (TMA unit)
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// CTA-scope release / acquire on a shared-memory word (buffer hand-over in pool_kernel)
__device__ __forceinline__ void st_release_shared(int* p, int v) {
  asm volatile("st.release.cta.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_shared(const int* p) {
  int v;
  asm volatile("ld.acquire.cta.shared::cta.b32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
  return v;
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "NFM_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra NFM_DONE;\n"
      "bra NFM_WAIT;\n"
      "NFM_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// L2 eviction policy for streamed-once data
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// 1-D TMA: global -> shared, completion counted in bytes on an mbarrier.
// src, dst 16-byte aligned, bytes % 16 == 0.   SASS: UBLKCP
// kHint: tag the lines evict_first in L2.  Measured on B200 (profiles/
// r1_tile_geometry_sweep.txt, "build:" blocks): the hint costs 3-8 % on
// read-heavy ops (solve, matvec, det) and gains 2-5 % on ops that write as much
// as they read (invert, inverse), so the caller decides.
template <bool kHint>
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  if constexpr (kHint) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
  } else {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
  }
}

// L2 prefetch of a contiguous range (16-byte aligned, bytes % 16 == 0).  No
// architectural effect: it only warms L2, the point of coherence, so it may be
// issued BEFORE griddepcontrol.wait -- if the previous kernel still writes these
// lines, the later real load sees the written data.
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}

// 1-D TMA: shared -> global, tracked by the bulk async-group of the issuing thread.
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)),
               "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }

template <int kPending>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}

template <int kPending>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(kPending) : "memory");
}

// generic-proxy smem writes -> visible to the async proxy (before a bulk store)
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// Compile-time loop: f(std::integral_constant<int, i>) for i in [B, E).  The
// factorisation kernels index register arrays with these constants, so the
// arrays stay in registers no matter what the unroller's size heuristics say
// (`#pragma unroll` alone left the order >= 6 pivoted kernels in local memory).
template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, B>{});
    static_for<B + 1, E>(f);
  }
}
// descending: i = E-1 ... B
template <int B, int E, class F>
__device__ __forceinline__ void static_for_down(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, E - 1>{});
    static_for_down<B, E - 1>(f);
  }
}

// true if `pred` holds for any lane currently executing with this one.  The
// pivoted eliminations use it to skip the predicated row / column exchanges of a
// step in which no matrix of the warp pivots (always, on diagonally dominant or
// SPD input); correctness does not depend on which lanes take part.
__device__ __forceinline__ bool warp_any(bool pred) { return __any_sync(__activemask(), pred) != 0; }
// below this order the exchanges are cheaper than the votes and branches that would skip them
constexpr int kVoteFromOrder = 6;

// programmatic dependent launch (PDL)
__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------------------
// record movers: a record is L contiguous elements of T.  Within a staged tile
// record r starts at r*L*sizeof(T) from a 16-byte aligned base, so its
// alignment is gcd(L*sizeof(T), 16); use the widest access that allows.
// (Widest access also decides shared-memory bank behaviour: a stride that is
// an odd multiple of the access width is conflict free.)
// ---------------------------------------------------------------------------
template <typename T, int L>
struct RecAccess {
  static constexpr int kBytes = L * int(sizeof(T));
  static constexpr int kVecBytes = (kBytes % 16 == 0) ? 16 : (kBytes % 8 == 0) ? 8 : (kBytes % 4 == 0) ? 4 : int(sizeof(T));
  static constexpr int kVec = kVecBytes / int(sizeof(T));  // elements per access
  static_assert(kVec >= 1, "record narrower than one element");
};

template <int kBytes>
struct VecType;
template <>
struct VecType<4> { using type = uint32_t; };
template <>
struct VecType<8> { using type = uint2; };
template <>
struct VecType<16> { using type = uint4; };

template <typename T, int L>
__device__ __forceinline__ void load_record(const T* __restrict__ src, T (&r)[L]) {
  using A = RecAccess<T, L>;
  using V = typename VecType<A::kVecBytes>::type;
  constexpr int kChunks = L / A::kVec;
#pragma unroll
  for (int c = 0; c < kChunks; ++c) {
    V v = reinterpret_cast<const V*>(src)[c];
    const T* e = reinterpret_cast<const T*>(&v);
#pragma unroll
    for (int k = 0; k < A::kVec; ++k) r[c * A::kVec + k] = e[k];
  }
}

template <typename T, int L>
__device__ __forceinline__ void store_record(T* __restrict__ dst, const T (&r)[L]) {
  using A = RecAccess<T, L>;
  using V = typename VecType<A::kVecBytes>::type;
  constexpr int kChunks = L / A::kVec;
#pragma unroll
  for (int c = 0; c < kChunks; ++c) {
    V v;
    T* e = reinterpret_cast<T*>(&v);
#pragma unroll
    for (int k = 0; k < A::kVec; ++k) e[k] = r[c * A::kVec + k];
    reinterpret_cast<V*>(dst)[c] = v;
  }
}

// element-wise movers for the strided kernel (no alignment assumption)
template <typename T, int L>
__device__ __forceinline__ void load_record_scalar(const T* src, T (&r)[L], i64 es = 1) {
#pragma unroll
  for (int k = 0; k < L; ++k) r[k] = src[k * es];  // plain loads: src may alias the output (in-place ops)
}

template <typename T, int L>
__device__ __forceinline__ void store_record_scalar(T* dst, const T (&r)[L], i64 es = 1) {
#pragma unroll
  for (int k = 0; k < L; ++k) dst[k * es] = r[k];
}

template <typename T, int L>
__device__ __forceinline__ void zero_record(T (&r)[L]) {
#pragma unroll
  for (int k = 0; k < L; ++k) r[k] = T(0);
}

}  // namespace nfm
