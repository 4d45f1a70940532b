// nfm_pipeline.cuh -- the kernels every op runs through.
//
//   tile_kernel<Op, THREADS, MPT, STAGES, SEG>  (fast path, light ops)
//     Persistent CTAs, one thread per matrix (MPT matrices per thread per
//     tile).  The AoS records (coefficient dimension last) of a tile of
//     consecutive matrices are one contiguous byte range per operand, so each
//     operand tile moves HBM -> shared memory with 1-D TMA bulk copies
//     (cp.async.bulk, completion on an mbarrier) into a STAGES-deep ring;
//     threads pull their own record out of shared memory with the widest
//     conflict-free access, compute in registers, stage the result record in
//     shared memory and the tile goes back with TMA bulk stores.  Every HBM
//     access is therefore a full, aligned, contiguous burst regardless of the
//     record length.  The number of matrices per tile is a run-time argument
//     (full tiles + one partial tile, both by TMA); the first tiles are
//     prefetched into L2 ahead of the programmatic-dependent-launch wait.
//
//     SEG = false: one bulk copy per operand per tile, record r of the tile at
//       r * record_bytes.  Conflict free whenever record_bytes is an odd
//       multiple of its widest access (all packed-symmetric sizes but two).
//     SEG = true: for records that are a multiple of 32 B (dense 4x4, ...),
//       where consecutive threads would hit the same banks 2..8-way: the tile
//       is cut into 8 segments, each landing 16 B further than a dense layout
//       would put it (8 bulk copies per operand, issued by 8 lanes), and
//       thread m takes record (m / 8) of segment (m % 8).  The 8 lanes of a
//       128-bit shared-memory phase then sit in 8 different segments, i.e. 8
//       different 16 B bank groups: conflict free for every record size.
//
//   pool_kernel<Op, MAXW, MPT, SEG>  (fast path, pivoted ops on large records)
//     One persistent CTA per SM owns a pool of TMA buffers of one warp-tile
//     each; its warps run independently, results are written in place.
//
//   strided_kernel<Op>  (general path)
//     One thread per matrix straight from global memory with arbitrary batch
//     strides / alignment / broadcast.  Also runs the < 4-matrix head / tail
//     that cannot keep the 16-byte granularity of bulk copies.
//
// An Op is a stateless struct:
//     using scalar = float|double;
//     static constexpr int kLen0, kLen1, kLen2;   // input record lengths (1 if unused)
//     [static constexpr int kLen3;]               // optional fourth input (bit 8 of kUse)
//     static constexpr int kUse;                   // bit mask of inputs the op can take
//     static constexpr int kOut;                   // output record length
//     static constexpr bool kHeavy;                // pivoted / long dependent chains (kernel + geometry choice)
//     __device__ static void apply(const T(&)[kLen0], const T(&)[kLen1], const T(&)[kLen2], [const T(&)[kLen3],]
//                                  int present, int flags, T(&out)[kOut]);
// Absent optional inputs arrive zero-filled.
#pragma once

#include <atomic>

#include "nfm_common.cuh"

namespace nfm {

extern std::atomic<unsigned long long> g_launch_count;
extern thread_local int t_last_path_tma;
// Shape of the last bulk launch on this thread (nfm_last_launch_shape): kind (1 tile, 3 pool,
// 4 many right-hand sides, 0 none), threads per CTA, matrices per thread, stages / buffers /
// ring depth, warps, segmented layout, grid, tiles.  Host stores only.
extern thread_local long long t_last_launch[8];
inline void record_launch(int kind, int threads, int mpt, int stages, int warps, int seg, long long grid, long long tiles) {
  const long long v[8] = {kind, threads, mpt, stages, warps, seg, grid, tiles};
  for (int i = 0; i < 8; ++i) t_last_launch[i] = v[i];
}
inline void reset_launch_record() {
  for (int i = 0; i < 8; ++i) t_last_launch[i] = 0;
}
void set_error(const char* fmt, ...);

// Ops that take the two scalar parameters of KParams declare `kScalars`.
template <class Op, class = void>
struct has_scalars : std::false_type {};
template <class Op>
struct has_scalars<Op, std::void_t<decltype(Op::kScalars)>> : std::true_type {};

// Ops with a FOURTH input operand declare `kLen3` (bit 8 of kUse) and take it as an
// extra record argument of apply(); everyone else sees a dummy of length 1.
template <class Op, class = void>
struct len3 { static constexpr int value = 1; static constexpr bool has = false; };
template <class Op>
struct len3<Op, std::void_t<decltype(Op::kLen3)>> { static constexpr int value = Op::kLen3; static constexpr bool has = true; };

template <class Op, class R0, class R1, class R2, class R3, class O>
__device__ __forceinline__ void apply_op(const KParams& p, const R0& r0, const R1& r1, const R2& r2, const R3& r3, O& o) {
  using T = typename Op::scalar;
  if constexpr (len3<Op>::has) {
    if constexpr (has_scalars<Op>::value) Op::apply(r0, r1, r2, r3, p.present, p.flags, T(p.scal0), T(p.scal1), o);
    else Op::apply(r0, r1, r2, r3, p.present, p.flags, o);
  } else {
    if constexpr (has_scalars<Op>::value) Op::apply(r0, r1, r2, p.present, p.flags, T(p.scal0), T(p.scal1), o);
    else Op::apply(r0, r1, r2, p.present, p.flags, o);
  }
}

// Ops whose matrices are worked on by TWO lanes each (pool_kernel only) declare `kPairLanes = 2` and
//     __device__ static void apply_pair(unsigned char* record, int lane, int flags);
// which reads the staged record, computes and writes the result IN PLACE into the same bytes.
template <class Op, class = void>
struct pair_lanes { static constexpr int value = 1; };
template <class Op>
struct pair_lanes<Op, std::void_t<decltype(Op::kPairLanes)>> { static constexpr int value = Op::kPairLanes; };

constexpr int kSegs = 8;     // segments per tile in the SEG layout
constexpr int kSegPad = 16;  // bytes of skew per segment
// The number of matrices in a tile is a run-time value (so that a launch can be
// cut into equal tiles, see balanced_tile()); it is a multiple of kTileGran, which
// keeps every operand tile -- and every one of the 8 segments of the SEG layout --
// a multiple of 16 bytes for any record length (records are multiples of 4 bytes).
constexpr int kTileGran = 32;

template <class Op, int THREADS, int MPT, bool SEG>
struct TileGeom {
  using T = typename Op::scalar;
  static constexpr int kTile = THREADS * MPT;
  static constexpr int kPad = SEG ? kSegs * kSegPad : 0;
  // matrices whose records make up a multiple of 16 bytes for every record
  // length (records are multiples of 4 bytes); times 8 when the tile is segmented
  static constexpr int kGran = SEG ? 4 * kSegs : 4;
  // payload bytes of one operand tile / its footprint in shared memory
  static constexpr int bytes(int len) { return kTile * len * int(sizeof(T)); }
  static constexpr int footprint(int len) { return bytes(len) + kPad; }
  static constexpr int kBytes0 = bytes(Op::kLen0), kBytes1 = bytes(Op::kLen1), kBytes2 = bytes(Op::kLen2);
  static constexpr int kBytes3 = bytes(len3<Op>::value);
  static constexpr int kBytesOut = bytes(Op::kOut);
  static constexpr int kFootOut = footprint(Op::kOut);
  static_assert(kTile % kTileGran == 0 || (kTile == 16 && pair_lanes<Op>::value == 2),
                "tile capacity must be a multiple of kTileGran matrices (16-matrix warp tiles of two-lane ops excepted)");
  static_assert(!SEG || (bytes(Op::kLen0) / kSegs) % 16 == 0, "segments must keep the 16 B alignment of bulk copies");
  static_assert(kBytes0 % 16 == 0 && kBytes1 % 16 == 0 && kBytes2 % 16 == 0 && kBytesOut % 16 == 0,
                "tile byte counts must be multiples of 16 for TMA bulk copies");

  // byte offset of record m (0 <= m < kTile, in thread order) inside an operand
  // tile.  The layout is fixed by the CAPACITY of the tile: a tile that holds fewer
  // matrices fills only the head of the buffer (of each segment when SEG), so the
  // slots past its count land on unused bytes and never need a guard.
  static constexpr int seg_stride(int len) { return bytes(len) / kSegs + kSegPad; }
  template <int LEN>
  __device__ static __forceinline__ int rec_offset(int m) {
    if constexpr (SEG) {
      return (m & (kSegs - 1)) * seg_stride(LEN) + (m >> 3) * LEN * int(sizeof(T));
    } else {
      return m * LEN * int(sizeof(T));
    }
  }
};

// which operands are staged through shared memory for this launch:
// present, not broadcast.  (Eligibility -- dense stride, 16 B alignment -- is
// checked on the host.)
__host__ __device__ inline int staged_mask(const KParams& p) {
  int m = 0;
  for (int i = 0; i < kMaxIn; ++i)
    if (((p.present >> i) & 1) && p.in[i].stride != 0) m |= 1 << i;
  return m;
}

// element e (0 <= e < count*LEN, tile-global order of a FULL-capacity tile) -> byte
// offset in the staged tile
template <class G, int LEN>
__device__ __forceinline__ int elem_offset(int e) {
  using T = typename G::T;
  if constexpr (G::kPad != 0) {
    constexpr int per_seg = G::kTile / kSegs * LEN;  // elements per segment
    const int seg = e / per_seg;
    return seg * G::seg_stride(LEN) + (e - seg * per_seg) * int(sizeof(T));
  } else {
    return e * int(sizeof(T));
  }
}

// ragged last tile: the `step` threads idx = 0..step-1 (a CTA or one warp) copy
// `count` records between global memory and the staged layout with plain
// coalesced accesses
template <class G, int LEN>
__device__ __forceinline__ void coop_load(unsigned char* smem_tile, const typename G::T* src, int count, int idx, int step) {
  using T = typename G::T;
  constexpr int U = 4;  // independent loads in flight per thread
  const int total = count * LEN;
  for (int e0 = idx; e0 < total; e0 += U * step) {
    T v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = (e0 + u * step < total) ? src[e0 + u * step] : T(0);
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (e0 + u * step < total) *reinterpret_cast<T*>(smem_tile + elem_offset<G, LEN>(e0 + u * step)) = v[u];
  }
}

template <class G, int LEN>
__device__ __forceinline__ void coop_store(typename G::T* dst, const unsigned char* smem_tile, int count, int idx, int step) {
  using T = typename G::T;
  const int total = count * LEN;
  for (int e = idx; e < total; e += step) dst[e] = *reinterpret_cast<const T*>(smem_tile + elem_offset<G, LEN>(e));
}

#ifdef NFM_TIMELINE
// development aid (tune_main.cu "timeline"): per-CTA %globaltimer stamps, row = launch id
// (passed in KParams::scal1) * 1024 + CTA; grids of at most 1024 CTAs
__device__ unsigned long long* g_timeline = nullptr;
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define NFM_STAMP(k)                                                                    \
  do {                                                                                  \
    if (threadIdx.x == 0 && g_timeline != nullptr)                                     \
      g_timeline[(size_t(p.scal1) * 1024 + blockIdx.x) * 8 + (k)] = global_ns();          \
  } while (0)
#define NFM_STAMP_VAL(k, v)                                                             \
  do {                                                                                  \
    if (threadIdx.x == 0 && g_timeline != nullptr)                                     \
      g_timeline[(size_t(p.scal1) * 1024 + blockIdx.x) * 8 + (k)] = (unsigned long long)(v); \
  } while (0)
__device__ __forceinline__ unsigned smid() {
  unsigned r;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(r));
  return r;
}
#else
#define NFM_STAMP(k) \
  do {               \
  } while (0)
#define NFM_STAMP_VAL(k, v) \
  do {                      \
  } while (0)
#endif

template <class Op, int THREADS, int MPT, int STAGES, bool SEG>
__global__ void __launch_bounds__(THREADS)
    tile_kernel(const __grid_constant__ KParams p, const i64 ntiles, const int tile_m, const int part_m) {
  // The launch covers p.batch matrices as
  //   ntiles tiles of tile_m <= THREADS*MPT matrices (tile_m % kTileGran == 0),
  //   one partial tile of part_m < tile_m matrices (part_m % TileGeom::kGran == 0,
  //     so it still moves by TMA, just with a smaller byte count), and
  //   (the launcher hands the last p.batch % kGran matrices, which cannot keep the
  //   16-byte granularity of bulk copies, to a second tiny launch of strided_kernel:
  //   in this kernel that code cost the main loop 2-3 %).
  using T = typename Op::scalar;
  using G = TileGeom<Op, THREADS, MPT, SEG>;
  NFM_STAMP(0);
  const i64 ntiles_all = ntiles + (part_m > 0 ? 1 : 0);
  constexpr int kIssuers = SEG ? kSegs : 1;  // threads that issue bulk copies (one segment each)
  constexpr int nseg = SEG ? kSegs : 1;
  constexpr int es = int(sizeof(T));
  // L2 evict_first on the loads only for ops that write at least as much as they read
  constexpr bool kHint = Op::kOut >= ((Op::kUse & 1) ? Op::kLen0 : 0) + ((Op::kUse & 2) ? Op::kLen1 : 0);

  extern __shared__ __align__(128) unsigned char smem[];
  const int staged = staged_mask(p);
  // shared-memory footprints are sized for the full THREADS*MPT capacity
  const int f0 = (staged & 1) ? G::footprint(Op::kLen0) : 0;
  const int f1 = (staged & 2) ? G::footprint(Op::kLen1) : 0;
  const int f2 = (staged & 4) ? G::footprint(Op::kLen2) : 0;
  constexpr int kL3 = len3<Op>::value;
  const int f3 = (staged & 8) ? G::footprint(kL3) : 0;
  const int stage_bytes = f0 + f1 + f2 + f3;
  const int staged_len = ((staged & 1) ? Op::kLen0 : 0) + ((staged & 2) ? Op::kLen1 : 0) + ((staged & 4) ? Op::kLen2 : 0) +
                         ((staged & 8) ? kL3 : 0);

  unsigned char* const in_base = smem;
  unsigned char* const out_base = smem + STAGES * stage_bytes;
  uint64_t* const full = reinterpret_cast<uint64_t*>(out_base + 2 * G::kFootOut);

  const int tid = threadIdx.x;
  const T* const g0 = static_cast<const T*>(p.in[0].ptr);
  const T* const g1 = static_cast<const T*>(p.in[1].ptr);
  const T* const g2 = static_cast<const T*>(p.in[2].ptr);
  const T* const g3 = static_cast<const T*>(p.in[3].ptr);
  T* const gout = static_cast<T*>(p.out);
  // matrices in tile t
#ifdef NFM_AB_STATICTILE
  auto count_of = [&](i64) { return G::kTile; };
#else
  auto count_of = [&](i64 t) { return t < ntiles ? tile_m : part_m; };
#endif

  uint64_t policy = 0;
  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
    fence_mbar_init();
  }
  if (tid < kIssuers) policy = policy_evict_first();
#ifndef NFM_NO_PREFETCH
  // Warm L2 with this CTA's first tiles while the previous kernel in the stream
  // drains: under programmatic dependent launch this CTA becomes resident 1-3 us
  // before griddepcontrol.wait releases it (profiles/r2_launch_timeline.txt), and
  // HBM is under-used during that tail.  An L2 prefetch has no architectural
  // effect, so it is safe ahead of the wait.
  if (tid < STAGES) {
    const i64 t = i64(blockIdx.x) + i64(tid) * gridDim.x;
    if (t < ntiles_all) {
      const i64 first = t * tile_m;
      const uint32_t c = uint32_t(count_of(t));
      if (staged & 1) bulk_prefetch_l2(g0 + first * Op::kLen0, c * Op::kLen0 * es);
      if (staged & 2) bulk_prefetch_l2(g1 + first * Op::kLen1, c * Op::kLen1 * es);
      if (staged & 4) bulk_prefetch_l2(g2 + first * Op::kLen2, c * Op::kLen2 * es);
      if (staged & 8) bulk_prefetch_l2(g3 + first * kL3, c * kL3 * es);
    }
  }
#endif
  __syncthreads();
  // programmatic dependent launch: everything above overlapped the previous
  // kernel's tail; its results are visible only after this wait
  grid_dependency_wait();
  grid_launch_dependents();
  NFM_STAMP(1);

  // producer (threads 0..kIssuers-1): thread 0 arms the stage barrier with the
  // tile's byte count; each issuer sends its segment of every staged operand.
  // `per_seg_c` (matrices per segment; per tile when !SEG) is a compile-time constant for
  // full-capacity tiles and a run-time value for the others: with run-time byte counts on
  // every copy the segmented 4x4 fp64 kernels lost 4 % (profiles/r2_kernel_ab.txt).
  auto issue_n = [&](int stage, i64 tile, auto per_seg_c) {
    unsigned char* dst = in_base + stage * stage_bytes;
    const i64 first = tile * tile_m;
    const int per_seg = per_seg_c;
    if (tid == 0) mbar_arrive_expect_tx(&full[stage], uint32_t(per_seg * nseg * staged_len * es));
    const int seg = SEG ? tid : 0;  // segment `seg` lands at its fixed (capacity) offset
    if (staged & 1) {
      const int sb = per_seg * Op::kLen0 * es;
      bulk_g2s<kHint>(dst + seg * G::seg_stride(Op::kLen0), reinterpret_cast<const unsigned char*>(g0 + first * Op::kLen0) + seg * sb,
                      sb, &full[stage], policy);
    }
    if (staged & 2) {
      const int sb = per_seg * Op::kLen1 * es;
      bulk_g2s<kHint>(dst + f0 + seg * G::seg_stride(Op::kLen1),
                      reinterpret_cast<const unsigned char*>(g1 + first * Op::kLen1) + seg * sb, sb, &full[stage], policy);
    }
    if (staged & 4) {
      const int sb = per_seg * Op::kLen2 * es;
      bulk_g2s<kHint>(dst + f0 + f1 + seg * G::seg_stride(Op::kLen2),
                      reinterpret_cast<const unsigned char*>(g2 + first * Op::kLen2) + seg * sb, sb, &full[stage], policy);
    }
    if constexpr (len3<Op>::has) {
      if (staged & 8) {
        const int sb = per_seg * kL3 * es;
        bulk_g2s<kHint>(dst + f0 + f1 + f2 + seg * G::seg_stride(kL3), reinterpret_cast<const unsigned char*>(g3 + first * kL3) + seg * sb,
                        sb, &full[stage], policy);
      }
    }
  };
  // tiles below `nstatic` hold exactly the capacity (always, unless equal-tile scheduling cut them)
  const i64 nstatic = tile_m == G::kTile ? ntiles : 0;
  auto issue = [&](int stage, i64 tile) {
    if (tile < nstatic) issue_n(stage, tile, std::integral_constant<int, G::kTile / nseg>{});
    else issue_n(stage, tile, count_of(tile) / nseg);
  };

  if (tid < kIssuers) {
#pragma unroll
    for (int s = 0; s < STAGES; ++s) {
      const i64 t = i64(blockIdx.x) + i64(s) * gridDim.x;
      if (t < ntiles_all) issue(s, t);
    }
  }

  int it = 0;
  for (i64 tile = blockIdx.x; tile < ntiles_all; tile += gridDim.x, ++it) {
    const int stage = it % STAGES;
    const uint32_t parity = uint32_t(it / STAGES) & 1u;
    unsigned char* sin = in_base + stage * stage_bytes;
    unsigned char* sout = out_base + (it & 1) * G::kFootOut;
    const int cnt = count_of(tile);

    mbar_wait(&full[stage], parity);
#ifdef NFM_TIMELINE
    if (it == 0) NFM_STAMP(2);
#endif

    // staged operands come out of shared memory; broadcast (stride 0) operands
    // are one record for the whole batch, re-read through L1; absent ones are 0.
    // Thread slots at or beyond cnt (a tile cut below capacity) compute on
    // whatever the buffer holds and their results are never stored.
    T r0[MPT][Op::kLen0], r1[MPT][Op::kLen1], r2[MPT][Op::kLen2], r3[MPT][kL3];
#pragma unroll
    for (int j = 0; j < MPT; ++j) {
      const int m = tid + j * THREADS;
      if constexpr (len3<Op>::has) {
        if (staged & 8) load_record(reinterpret_cast<const T*>(sin + f0 + f1 + f2 + G::template rec_offset<kL3>(m)), r3[j]);
        else if (p.present & 8) load_record_scalar(g3, r3[j]);
        else zero_record(r3[j]);
      } else {
        zero_record(r3[j]);
      }
      if (staged & 1) load_record(reinterpret_cast<const T*>(sin + G::template rec_offset<Op::kLen0>(m)), r0[j]);
      else if (p.present & 1) load_record_scalar(g0, r0[j]);
      else zero_record(r0[j]);
      if (staged & 2) load_record(reinterpret_cast<const T*>(sin + f0 + G::template rec_offset<Op::kLen1>(m)), r1[j]);
      else if (p.present & 2) load_record_scalar(g1, r1[j]);
      else zero_record(r1[j]);
      if (staged & 4) load_record(reinterpret_cast<const T*>(sin + f0 + f1 + G::template rec_offset<Op::kLen2>(m)), r2[j]);
      else if (p.present & 4) load_record_scalar(g2, r2[j]);
      else zero_record(r2[j]);
    }

    // the barrier below hands the stage to the async proxy (its TMA refill): order this thread's
    // generic-proxy loads from it before that write, or a load still in flight can return the
    // next tile's bytes (DESIGN.md section 4)
    fence_proxy_async();
    // the output buffer we are about to overwrite was last read by the bulk
    // store issued two tiles ago: allow one store (group) still pending
    if (tid < kIssuers) bulk_wait_read<1>();
    __syncthreads();  // every thread has its inputs in registers: stage is free
    if (tid < kIssuers) {
      const i64 nxt = tile + i64(STAGES) * gridDim.x;
      if (nxt < ntiles_all) issue(stage, nxt);
    }

#pragma unroll
    for (int j = 0; j < MPT; ++j) {
      T o[Op::kOut];
      apply_op<Op>(p, r0[j], r1[j], r2[j], r3[j], o);
      store_record(reinterpret_cast<T*>(sout + G::template rec_offset<Op::kOut>(tid + j * THREADS)), o);
    }
    fence_proxy_async();
    __syncthreads();
    if (tid < kIssuers) {
      const int seg = SEG ? tid : 0;
      if (tile < nstatic) {
        constexpr int sbo = (G::kTile / nseg) * Op::kOut * es;
        bulk_s2g(reinterpret_cast<unsigned char*>(gout + tile * i64(G::kTile) * Op::kOut) + seg * sbo,
                 sout + seg * G::seg_stride(Op::kOut), sbo);
      } else {
        const int sbo = (cnt / nseg) * Op::kOut * es;
        bulk_s2g(reinterpret_cast<unsigned char*>(gout + tile * tile_m * Op::kOut) + seg * sbo, sout + seg * G::seg_stride(Op::kOut),
                 sbo);
      }
      bulk_commit();
    }
  }
#ifdef NFM_AB_FINALWAIT
  if (tid < kIssuers) bulk_wait<0>();
#else
  if (tid < kIssuers) bulk_wait_read<0>();  // writes complete with the grid; only shared memory must outlive them
#endif
  NFM_STAMP(3);
#ifdef NFM_TIMELINE
  NFM_STAMP_VAL(4, smid());
  NFM_STAMP_VAL(5, it);
#endif
}

// ---------------------------------------------------------------------------
// pool_kernel<Op, MAXW, MPT, SEG>(..., nwarps, nbuf)  -- compute-heavy ops (Op::kHeavy:
// pivoted elimination, Gauss-Jordan) with large records.
//
// tile_kernel keeps STAGES input tiles + 2 output tiles per CTA and every
// thread of the CTA works on the same tile; with 500-800 B records that is
// ~200 KB of shared memory for 64-128 threads, so an SM holds 2-4 warps whose
// long dependent chains cannot cover each other (0.23-0.58 of the roofline for
// dense n >= 8 in round 1).  Here one persistent CTA per SM owns a POOL of nbuf
// buffers of one warp-tile (32*MPT matrices) each, and its nwarps <= MAXW warps
// (MAXW only sets the register budget, __launch_bounds__) run independently of
// each other (no __syncthreads in the loop):
//   warp-tile l of the CTA  ->  buffer l % nbuf, warp l % nwarps
//   wait the buffer's mbarrier -> records to registers -> compute -> results
//   written IN PLACE into the same buffer -> TMA bulk store -> when the store
//   has read the buffer, the same lane re-arms it with warp-tile l + nbuf.
// So nwarps buffers are being computed on while nbuf - nwarps are in flight from
// HBM, and no shared memory is spent on separate output tiles.
// ---------------------------------------------------------------------------
template <class Op, int MPT, bool SEG>
struct PoolGeom {
  using G = TileGeom<Op, 32 / pair_lanes<Op>::value, MPT, SEG>;  // two-lane ops: 16 matrices per warp
  static constexpr int kWarpTile = G::kTile;
  static constexpr int in_bytes(int mask) {
    return ((mask & 1) ? G::footprint(Op::kLen0) : 0) + ((mask & 2) ? G::footprint(Op::kLen1) : 0) +
           ((mask & 4) ? G::footprint(Op::kLen2) : 0);
  }
  // a buffer holds the staged inputs of one warp-tile, later its outputs
  static constexpr int buf_bytes(int mask) {
    const int b = in_bytes(mask) > G::kFootOut ? in_bytes(mask) : G::kFootOut;
    return (b + 127) / 128 * 128;
  }
};

template <class Op, int MAXW, int MPT, bool SEG>
__global__ void __launch_bounds__(MAXW * 32, 1)
    pool_kernel(const __grid_constant__ KParams p, const i64 ntiles, const int WARPS, const int NBUF) {
  using T = typename Op::scalar;
  using PG = PoolGeom<Op, MPT, SEG>;
  using G = typename PG::G;
  constexpr int WT = PG::kWarpTile;
  constexpr int kIssuers = SEG ? kSegs : 1;
  constexpr int nseg = SEG ? kSegs : 1;
  constexpr bool kHint = Op::kOut >= ((Op::kUse & 1) ? Op::kLen0 : 0) + ((Op::kUse & 2) ? Op::kLen1 : 0);
  NFM_STAMP(0);

  const int rem = int(p.batch - ntiles * WT);
  const i64 ntiles_all = ntiles + (rem > 0 ? 1 : 0);

  extern __shared__ __align__(128) unsigned char smem[];
  const int staged = staged_mask(p);
  const int f0 = (staged & 1) ? G::footprint(Op::kLen0) : 0;
  const int f1 = (staged & 2) ? G::footprint(Op::kLen1) : 0;
  const int buf_bytes = PG::buf_bytes(staged);
  constexpr int sb0 = G::kBytes0 / nseg, sb1 = G::kBytes1 / nseg, sb2 = G::kBytes2 / nseg, sbo = G::kBytesOut / nseg;
  const uint32_t tx_bytes = ((staged & 1) ? G::kBytes0 : 0) + ((staged & 2) ? G::kBytes1 : 0) + ((staged & 4) ? G::kBytes2 : 0);
  uint64_t* const full = reinterpret_cast<uint64_t*>(smem + NBUF * buf_bytes);
  // gen[b] = generation (l / NBUF) the buffer was last handed over to.  A parity
  // bit alone cannot tell a consumer that it is TWO phases early (any warp may
  // consume any buffer here), so a consumer first waits for its generation.
  int* const gen = reinterpret_cast<int*>(full + NBUF);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const T* const g0 = static_cast<const T*>(p.in[0].ptr);
  const T* const g1 = static_cast<const T*>(p.in[1].ptr);
  const T* const g2 = static_cast<const T*>(p.in[2].ptr);
  T* const gout = static_cast<T*>(p.out);

  uint64_t policy = 0;
  if (tid == 0) {
    for (int b = 0; b < NBUF; ++b) {
      mbar_init(&full[b], 1);
      gen[b] = 0;
    }
    fence_mbar_init();
  }
  if (lane < kIssuers) policy = policy_evict_first();
#ifndef NFM_NO_PREFETCH
  // warm L2 with the first nbuf warp-tiles ahead of the dependency wait (see tile_kernel)
  for (int l = tid; l < NBUF; l += WARPS * 32) {
    const i64 t = i64(blockIdx.x) + i64(l) * gridDim.x;
    if (t < ntiles) {
      const i64 first = t * WT;
      if (staged & 1) bulk_prefetch_l2(g0 + first * Op::kLen0, G::kBytes0);
      if (staged & 2) bulk_prefetch_l2(g1 + first * Op::kLen1, G::kBytes1);
      if (staged & 4) bulk_prefetch_l2(g2 + first * Op::kLen2, G::kBytes2);
    }
  }
#endif
  __syncthreads();
  grid_dependency_wait();
  grid_launch_dependents();
  NFM_STAMP(1);

  // lanes 0..kIssuers-1 of the calling warp fetch global warp-tile `tile` into buffer `b`
  auto issue = [&](int b, i64 tile) {
    unsigned char* dst = smem + b * buf_bytes;
    const i64 first = tile * WT;
    if (lane == 0) mbar_arrive_expect_tx(&full[b], tx_bytes);
    const int seg = SEG ? lane : 0;
    if (staged & 1)
      bulk_g2s<kHint>(dst + seg * G::seg_stride(Op::kLen0), reinterpret_cast<const unsigned char*>(g0 + first * Op::kLen0) + seg * sb0,
                      sb0, &full[b], policy);
    if (staged & 2)
      bulk_g2s<kHint>(dst + f0 + seg * G::seg_stride(Op::kLen1),
                      reinterpret_cast<const unsigned char*>(g1 + first * Op::kLen1) + seg * sb1, sb1, &full[b], policy);
    if (staged & 4)
      bulk_g2s<kHint>(dst + f0 + f1 + seg * G::seg_stride(Op::kLen2),
                      reinterpret_cast<const unsigned char*>(g2 + first * Op::kLen2) + seg * sb2, sb2, &full[b], policy);
  };

  // prologue: fill the pool; local tile l is fetched by the warp that will NOT
  // necessarily consume it -- any warp may wait on any buffer's barrier
  if (lane < kIssuers) {
    for (int l = warp; l < NBUF; l += WARPS) {
      const i64 t = i64(blockIdx.x) + i64(l) * gridDim.x;
      if (t < ntiles) issue(l, t);
    }
  }

  for (int l = warp;; l += WARPS) {
    const i64 tile = i64(blockIdx.x) + i64(l) * gridDim.x;
    if (tile >= ntiles_all) break;
    const int b = l % NBUF;
    const uint32_t parity = uint32_t(l / NBUF) & 1u;
    unsigned char* sbuf = smem + b * buf_bytes;
    const bool ragged = tile >= ntiles;  // the globally last tile: at most once

    // the buffer's previous user has handed it over to this generation (its
    // refill has been issued / it is free for the by-hand fill of the ragged tile)
    while (ld_acquire_shared(&gen[b]) != l / NBUF) {
    }
    if (!ragged) {
      mbar_wait(&full[b], parity);
#ifdef NFM_TIMELINE
      if (l == 0) NFM_STAMP(2);
#endif
    } else {
      const i64 first = tile * WT;
      if (staged & 1) coop_load<G, Op::kLen0>(sbuf, g0 + first * Op::kLen0, rem, lane, 32);
      if (staged & 2) coop_load<G, Op::kLen1>(sbuf + f0, g1 + first * Op::kLen1, rem, lane, 32);
      if (staged & 4) coop_load<G, Op::kLen2>(sbuf + f0 + f1, g2 + first * Op::kLen2, rem, lane, 32);
      __syncwarp();
    }

    if constexpr (pair_lanes<Op>::value == 2) {
      // two lanes per matrix (half of the columns each): the op reads its record out of the buffer,
      // and writes the result over it, by itself
      static_assert(MPT == 1 && Op::kOut == Op::kLen0 && Op::kUse == 1, "two-lane ops: one operand, result in place");
      Op::apply_pair(sbuf + G::template rec_offset<Op::kLen0>(lane >> 1), lane, p.flags);
    } else {
      T r0[MPT][Op::kLen0], r1[MPT][Op::kLen1], r2[MPT][Op::kLen2];
#pragma unroll
      for (int j = 0; j < MPT; ++j) {
        const int m = lane + j * 32;
        if (staged & 1) load_record(reinterpret_cast<const T*>(sbuf + G::template rec_offset<Op::kLen0>(m)), r0[j]);
        else if (p.present & 1) load_record_scalar(g0, r0[j]);
        else zero_record(r0[j]);
        if (staged & 2) load_record(reinterpret_cast<const T*>(sbuf + f0 + G::template rec_offset<Op::kLen1>(m)), r1[j]);
        else if (p.present & 2) load_record_scalar(g1, r1[j]);
        else zero_record(r1[j]);
        if (staged & 4) load_record(reinterpret_cast<const T*>(sbuf + f0 + f1 + G::template rec_offset<Op::kLen2>(m)), r2[j]);
        else if (p.present & 4) load_record_scalar(g2, r2[j]);
        else zero_record(r2[j]);
      }
      __syncwarp();  // every lane holds its inputs: the buffer now takes the results

#pragma unroll
      for (int j = 0; j < MPT; ++j) {
        T o[Op::kOut], r3[len3<Op>::value];
        zero_record(r3);  // pool ops take at most three inputs
        apply_op<Op>(p, r0[j], r1[j], r2[j], r3, o);
        store_record(reinterpret_cast<T*>(sbuf + G::template rec_offset<Op::kOut>(lane + j * 32)), o);
      }
    }
    if (ragged) {
      __syncwarp();
      coop_store<G, Op::kOut>(gout + tile * WT * Op::kOut, sbuf, rem, lane, 32);
      break;
    }
    fence_proxy_async();
    __syncwarp();
    const i64 nxt = tile + i64(NBUF) * gridDim.x;  // next user of this buffer
    if (lane < kIssuers) {
      const int seg = SEG ? lane : 0;
      bulk_s2g(reinterpret_cast<unsigned char*>(gout + tile * WT * Op::kOut) + seg * sbo, sbuf + seg * G::seg_stride(Op::kOut), sbo);
      bulk_commit();
      if (nxt < ntiles_all) bulk_wait_read<0>();  // the store has read the buffer: it can be refilled
    }
    if (nxt < ntiles_all) {
      if constexpr (SEG) __syncwarp();  // every segment's store has been read before any lane refills
      if (nxt < ntiles && lane < kIssuers) issue(b, nxt);
      if constexpr (SEG) __syncwarp();  // lane 0's arrive.expect_tx and every segment's copy are issued
      if (lane == 0) st_release_shared(&gen[b], l / NBUF + 1);
    }
  }
  if (lane < kIssuers) bulk_wait<0>();
  NFM_STAMP(3);
}

template <class Op>
__global__ void __launch_bounds__(128) strided_kernel(const __grid_constant__ KParams p) {
  using T = typename Op::scalar;
  const T* const g0 = static_cast<const T*>(p.in[0].ptr);
  const T* const g1 = static_cast<const T*>(p.in[1].ptr);
  const T* const g2 = static_cast<const T*>(p.in[2].ptr);
  T* const gout = static_cast<T*>(p.out);
  grid_dependency_wait();
  grid_launch_dependents();
  // block-uniform trip count (ops may vote across the warp): lanes past the end
  // redo the last matrix and do not store
  for (i64 b0 = i64(blockIdx.x) * blockDim.x; b0 < p.batch; b0 += i64(gridDim.x) * blockDim.x) {
    const bool valid = b0 + threadIdx.x < p.batch;
    const i64 b = valid ? b0 + threadIdx.x : p.batch - 1;
    T r0[Op::kLen0], r1[Op::kLen1], r2[Op::kLen2], r3[len3<Op>::value], o[Op::kOut];
    zero_record(r0);
    zero_record(r1);
    zero_record(r2);
    zero_record(r3);
    if (p.present & 1) load_record_scalar(g0 + b * p.in[0].stride, r0, elem_stride(p.in[0].estride));
    if (p.present & 2) load_record_scalar(g1 + b * p.in[1].stride, r1, elem_stride(p.in[1].estride));
    if (p.present & 4) load_record_scalar(g2 + b * p.in[2].stride, r2, elem_stride(p.in[2].estride));
    if constexpr (len3<Op>::has)
      if (p.present & 8) load_record_scalar(static_cast<const T*>(p.in[3].ptr) + b * p.in[3].stride, r3, elem_stride(p.in[3].estride));
    apply_op<Op>(p, r0, r1, r2, r3, o);
    if (valid) store_record_scalar(gout + b * p.out_stride, o, elem_stride(p.out_estride));
  }
}

// ---------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------
struct DeviceInfo {
  int sm_count;
  int max_smem_optin;
};
const DeviceInfo& device_info();  // cached per current device
int current_device();

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Tile geometry.  Measured on B200 (profiles/r1_tile_geometry_sweep.txt): the
// best configurations keep ONE large CTA per SM with 2 (big records) or 3
// stages and ~130-150 KB of shared memory -- large bulk copies beat many small
// ones -- so the rule is: stages = 2 when a matrix moves >= 100 B, else 3;
// TILE = the largest of {64,...,1024} (2048 / 4096 for records of a few bytes) whose ring (mandatory
// operands) + double-buffered output fits 152 KB; THREADS = 512 / 384 / 256 /
// TILE.  Optional operands (regulariser, addend) grow the ring up to the
// 227 KB limit.  TuneFixed pins ops whose measured optimum differs.
// -DNFM_TUNE_TILE / NFM_TUNE_THREADS / NFM_TUNE_STAGES / NFM_TUNE_SEG override
// the rule for tuning builds.
template <class Op, class = void>
struct three_mandatory : std::false_type {};
template <class Op>
struct three_mandatory<Op, std::void_t<decltype(Op::kThreeMandatory)>> : std::true_type {};

template <class Op>
struct TuneBase {
  using T = typename Op::scalar;
  // operands 0 and 1 are mandatory wherever they are used, operand 2 is optional unless the op
  // says so (kThreeMandatory), operand 3 is always optional: size the tiles for the mandatory ones
  static constexpr int kInBytes =
      (((Op::kUse >> 0) & 1) * Op::kLen0 + ((Op::kUse >> 1) & 1) * Op::kLen1 + (three_mandatory<Op>::value ? Op::kLen2 : 0)) * int(sizeof(T));
  static constexpr int kOutBytes = Op::kOut * int(sizeof(T));
  // Records that are a multiple of 32 B bank-conflict in the dense layout:
  // 2-way at 32 B, 4-way at 64 B, 8-way at 128 B.  The segmented layout removes
  // that but its 8x smaller bulk copies cost ~7-15 %, so it is used when an
  // operand conflicts >= 4-way, or 2-way on an operand that carries at least
  // half of the traffic (a 2-way conflict on a small vector is cheaper).
  static constexpr int rec_bytes(int len) { return len * int(sizeof(T)); }
  static constexpr bool heavy(int len) { return rec_bytes(len) % 64 == 0; }
  static constexpr bool light(int len) { return rec_bytes(len) % 32 == 0 && 2 * rec_bytes(len) >= kInBytes + kOutBytes; }
  static constexpr bool conflicts(int len) { return heavy(len) || light(len); }
#ifdef NFM_TUNE_SEG
  static constexpr bool kSeg = NFM_TUNE_SEG;
#else
  static constexpr bool kSeg = (((Op::kUse >> 0) & 1) && conflicts(Op::kLen0)) || (((Op::kUse >> 1) & 1) && conflicts(Op::kLen1)) ||
                               conflicts(Op::kOut);
#endif
};

constexpr int kSmemTarget = 152 * 1024;

constexpr int pick_tile(int stages, int in_bytes, int out_bytes) {
  const int per_matrix = stages * in_bytes + 2 * out_bytes;
  const int cands[9] = {4096, 2048, 1024, 768, 512, 384, 256, 128, 64};
  for (int i = (per_matrix <= 48 ? 0 : per_matrix <= 96 ? 1 : 2); i < 9; ++i)
    if (cands[i] * per_matrix <= kSmemTarget) return cands[i];
  return 64;
}

// one matrix per thread up to 512 threads; MPT <= 8.  (1024 x 1 was re-measured in round 2
// with the L2 prefetch: 118.2 vs 114.5 us for the 3x3 solve, profiles/r2_geometry_sweep.txt)
constexpr int pick_threads(int tile) { return tile >= 1024 ? 512 : tile == 768 ? 384 : tile; }

// Compute-heavy ops (pivoted elimination, Gauss-Jordan: Op::kHeavy) are bound by
// the latency of their dependent chains rather than by HBM alone; they do best
// with SEVERAL small CTAs per SM whose barrier phases interleave: 128 threads,
// one matrix each, 3 stages (2 when the ring would pass 72 KB), tile 64 when
// even that passes 100 KB  (profiles/r1_tile_geometry_sweep.txt, sweep 3).
constexpr int heavy_stages(int in_bytes, int out_bytes) { return 128 * (3 * in_bytes + 2 * out_bytes) <= 72 * 1024 ? 3 : 2; }
constexpr int heavy_tile(int in_bytes, int out_bytes) {
  return 128 * (heavy_stages(in_bytes, out_bytes) * in_bytes + 2 * out_bytes) <= 100 * 1024 ? 128 : 64;
}

template <class Op>
struct TuneRule : TuneBase<Op> {
  using B = TuneBase<Op>;
#ifdef NFM_TUNE_STAGES
  static constexpr int kStages = NFM_TUNE_STAGES;
#else
  static constexpr int kStages = Op::kHeavy ? heavy_stages(B::kInBytes, B::kOutBytes) : (B::kInBytes + B::kOutBytes >= 100) ? 2 : 3;
#endif
#ifdef NFM_TUNE_TILE
  static constexpr int kTile = NFM_TUNE_TILE;
#else
  // light ops that move >= 250 B per matrix (10x10 packed solve ...) carry ~150 registers per
  // thread: three 128-matrix CTAs per SM beat one of 256 (7031 vs 6751 GB/s, r2_geometry_sweep)
  static constexpr int kTile = Op::kHeavy                             ? heavy_tile(B::kInBytes, B::kOutBytes)
                               : (B::kInBytes + B::kOutBytes >= 250) ? (pick_tile(kStages, B::kInBytes, B::kOutBytes) < 128
                                                                            ? pick_tile(kStages, B::kInBytes, B::kOutBytes)
                                                                            : 128)
                                                                      : pick_tile(kStages, B::kInBytes, B::kOutBytes);
#endif
#ifdef NFM_TUNE_THREADS
  static constexpr int kThreads = NFM_TUNE_THREADS < kTile ? NFM_TUNE_THREADS : kTile;
#else
  static constexpr int kThreads = Op::kHeavy ? kTile : pick_threads(kTile);
#endif
  static constexpr int kMpt = kTile / kThreads;
};

template <class Op, int TILE, int THREADS, int STAGES>
struct TuneFixed : TuneBase<Op> {
#if defined(NFM_TUNE_TILE) || defined(NFM_TUNE_THREADS) || defined(NFM_TUNE_STAGES)
  static constexpr int kTile = TuneRule<Op>::kTile, kThreads = TuneRule<Op>::kThreads, kStages = TuneRule<Op>::kStages;
#else
  static constexpr int kTile = TILE, kThreads = THREADS, kStages = STAGES;
#endif
  static constexpr int kMpt = kTile / kThreads;
};

template <class Op>
struct Tune : TuneRule<Op> {};

// Second, smaller geometry for light ops when a launch is small (a multi-GPU slab,
// config 1): several small CTAs per SM ramp up and drain faster than one big one.
// Measured with the L2 prefetch in place (profiles/r2_geometry_sweep.txt):
//   records <= 64 B  (3x3 solve): 256 threads x 2, 2 stages -- 8.4 vs 10.4 us at 1M,
//       15.7 vs 18.2 us at 2M, 31.0 vs 32.9 us at 4M, equal at 8M matrices (the write-heavy
//       3x3 invert already loses there: 0.88 vs 0.95 of the peak)
//   records <= 200 B (6x6 solve / invert): 128 threads x 1, 3 stages -- 18.2 vs 19.3 us and
//       24.9 vs 25.4 us at 885k matrices, behind the large geometry from ~1.5M
// `kBelowBytes`: use it when the launch moves fewer algorithmic bytes than this.
template <class Op>
struct TuneSmall {
  using B = TuneBase<Op>;
  static constexpr int kRec = B::kInBytes + B::kOutBytes;
  static constexpr bool kTiny = kRec <= 64;
  // (records below 20 B of input keep the large tiles: 512 of them are bulk copies of 2-4 KB, and the
  //  order-1/2 routines lost 10-25 % with them, profiles/r2_sweep_all_orders_f32.txt first pass)
  static constexpr bool kEnabled = !Op::kHeavy && B::kInBytes >= 20 &&
                                   ((kTiny && Tune<Op>::kTile >= 1024) || (!kTiny && kRec <= 200 && Tune<Op>::kTile > 128));
  static constexpr int kThreads = kTiny ? 256 : 128, kMpt = kTiny ? 2 : 1, kStages = kTiny ? 2 : 3;
  static constexpr long long kBelowBytes = kTiny ? (300ll << 20) : (180ll << 20);
};

// Pool geometry for compute-heavy ops with large records (pool_kernel).
// Measured on B200 (profiles/r2_pool_sweep.txt): the pool wins from ~256 B of
// input per matrix (fp64 8x8 inverse 0.43 -> 0.86 of the measured peak, fp32
// 10x10 0.66 -> 0.93) and loses below (4x4 fp64 inverse 0.90 vs 0.95).
//   kMaxW : register budget (launch bounds): 8 warps (255 registers) for fp64, 12 (168) for fp32
//   warps / buffers at run time: kMaxW warps when shared memory holds that many
//           buffers, plus 2-3 buffers in flight.  Larger pools were SLOWER (r2_pool_sweep:
//           6x6 fp64 inverse 6550 GB/s with 8+2 buffers, 5735 with 12+12): the register
//           spills of these kernels live in the L1 that a bigger pool takes away.
template <class Op>
struct PoolTune {
  using B = TuneBase<Op>;
#ifdef NFM_TUNE_POOL
  static constexpr bool kEnabled = NFM_TUNE_POOL && Op::kHeavy;
#else
  static constexpr bool kEnabled = Op::kHeavy && B::kInBytes >= 256;
#endif
  // (two-lane ops hold half a matrix per lane: 12 warps = 168 registers also in fp64)
  static constexpr int kMaxW = (sizeof(typename Op::scalar) == 8 && pair_lanes<Op>::value == 1) ? 8 : 12;
  static constexpr int kMpt = 1;
  static void geometry(int buf_bytes, int max_smem, int& warps, int& nbuf) {
    int nbuf_max = (max_smem - 512) / (buf_bytes + 12);
    warps = nbuf_max - 1 < kMaxW ? nbuf_max - 1 : kMaxW;
    if (warps < 1) warps = 1;
    const int flight = warps / 4 > 2 ? warps / 4 : 2;
    nbuf = warps + flight < nbuf_max ? warps + flight : nbuf_max;
    if (nbuf <= warps) nbuf = warps + 1;
  }
};

bool pdl_enabled();  // nfm_entry.cu: false when the environment has NFM_DISABLE_PDL=1

// Launch with programmatic stream serialization: the kernel may become resident
// while the previous kernel in the stream drains; it touches global memory only
// after griddepcontrol.wait, so ordering is unchanged.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;  // NFM_DISABLE_PDL=1 turns it off
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// the last few matrices of a dense batch (those past `done`), one thread each
template <class Op>
int launch_tail(const KParams& p, i64 done, cudaStream_t stream) {
  using T = typename Op::scalar;
  KParams q = p;
  const int lens[kMaxIn] = {Op::kLen0, Op::kLen1, Op::kLen2, len3<Op>::value};
  for (int i = 0; i < kMaxIn; ++i)
    if ((q.present >> i) & 1) q.in[i].ptr = static_cast<const T*>(q.in[i].ptr) + done * (q.in[i].stride == 0 ? 0 : lens[i]);
  q.out = static_cast<T*>(q.out) + done * Op::kOut;
  q.batch = p.batch - done;
  cudaError_t e = launch_pdl(strided_kernel<Op>, 1u, 128u, size_t(0), stream, q);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(e);
}

// per (kernel instantiation, device, staged mask): resident CTAs per SM, 0 = not yet known
struct LaunchCache {
  std::atomic<int> per_sm[16][16];
  std::atomic<int> attr_set[16];
};

// Equal tiles: a launch of `batch` matrices on `grid_max` persistent CTAs takes
// waves = ceil(batch / (grid_max * capacity)) tiles per CTA; cutting the tile to
// ceil(batch / (grid_max * waves)) matrices (rounded up to kTileGran) gives every
// CTA the same number of (slightly smaller) tiles instead of leaving a last,
// partly filled wave -- 9.2 waves of 512-matrix tiles became 10 of 480 for a
// 2M-matrix slab.  Large launches keep the full capacity (the rounding absorbs it).
inline int balanced_tile(i64 batch, i64 grid_max, int capacity) {
  const i64 waves = (batch + grid_max * capacity - 1) / (grid_max * capacity);
  i64 t = (batch + grid_max * waves - 1) / (grid_max * waves);
  t = (t + kTileGran - 1) / kTileGran * kTileGran;
  return int(t < capacity ? t : capacity);
}

bool balance_enabled();  // nfm_entry.cu: true only when the environment has NFM_BALANCE=1

template <class Op, int THREADS, int MPT, int STAGES, bool SEG>
int launch_tile(const KParams& p, cudaStream_t stream) {
  using G = TileGeom<Op, THREADS, MPT, SEG>;
  static LaunchCache cache;  // zero-initialised
  auto kern = tile_kernel<Op, THREADS, MPT, STAGES, SEG>;
  const int staged = staged_mask(p);
  auto smem_for = [](int mask) {
    const int stage = ((mask & 1) ? G::footprint(Op::kLen0) : 0) + ((mask & 2) ? G::footprint(Op::kLen1) : 0) +
                      ((mask & 4) ? G::footprint(Op::kLen2) : 0) + ((mask & 8) ? G::footprint(len3<Op>::value) : 0);
    return STAGES * stage + 2 * G::kFootOut + STAGES * 8 + 16;
  };
  const int smem = smem_for(staged);
  const DeviceInfo& dev = device_info();
  if (smem > dev.max_smem_optin) return -1;  // caller falls back to the strided kernel
  const int d = current_device() & 15;
  if (!cache.attr_set[d].load(std::memory_order_acquire)) {
    int most = smem_for(Op::kUse & 15);
    if (most > dev.max_smem_optin) most = dev.max_smem_optin;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
    if (e != cudaSuccess) return int(e);
    cache.attr_set[d].store(1, std::memory_order_release);
  }
  int per_sm = cache.per_sm[d][staged].load(std::memory_order_acquire);
  if (per_sm == 0) {
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, THREADS, smem);
    if (e != cudaSuccess) return int(e);
    if (per_sm < 1) return -1;
    cache.per_sm[d][staged].store(per_sm, std::memory_order_release);
  }
  const i64 grid_max = i64(dev.sm_count) * per_sm;
  const int tile_m = balance_enabled() ? balanced_tile(p.batch, grid_max, G::kTile) : G::kTile;
  const i64 ntiles = p.batch / tile_m;
  const int part_m = int(p.batch - ntiles * tile_m) / G::kGran * G::kGran;
  const i64 ntiles_all = ntiles + (part_m > 0 ? 1 : 0);
  const i64 covered = ntiles * tile_m + part_m;
  if (ntiles_all > 0) {
    KParams q = p;
    q.batch = covered;
    const i64 grid = grid_max < ntiles_all ? grid_max : ntiles_all;
    cudaError_t e = launch_pdl(kern, unsigned(grid), THREADS, size_t(smem), stream, q, ntiles, tile_m, part_m);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    if (e != cudaSuccess) return int(e);
    record_launch(1, THREADS, MPT, STAGES, 0, SEG, grid, ntiles_all);
  }
  if (covered < p.batch) return launch_tail<Op>(p, covered, stream);  // < kGran matrices
  return 0;
}

template <class Op, int MAXW, int MPT, bool SEG>
int launch_pool(const KParams& p, int nwarps, int nbuf, cudaStream_t stream) {
  using PG = PoolGeom<Op, MPT, SEG>;
  static LaunchCache cache;  // attr_set only
  auto kern = pool_kernel<Op, MAXW, MPT, SEG>;
  const int staged = staged_mask(p);
  const DeviceInfo& dev = device_info();
  // optional / broadcast operands change the buffer size: keep the pool inside the
  // shared-memory limit by dropping buffers (never below nwarps + 1)
  auto smem_for = [&](int nb) { return nb * PG::buf_bytes(staged) + nb * 12 + 16; };
  while (nbuf > nwarps + 1 && smem_for(nbuf) > dev.max_smem_optin) --nbuf;
  while (nwarps > 1 && smem_for(nbuf) > dev.max_smem_optin) {
    --nwarps;
    nbuf = nwarps + 1;
  }
  const int smem = smem_for(nbuf);
  if (smem > dev.max_smem_optin || nwarps < 1 || nwarps > MAXW || nbuf <= nwarps) return -1;
  const int d = current_device() & 15;
  if (!cache.attr_set[d].load(std::memory_order_acquire)) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dev.max_smem_optin);
    if (e != cudaSuccess) return int(e);
    cache.attr_set[d].store(1, std::memory_order_release);
  }
  const i64 ntiles = p.batch / PG::kWarpTile;
  const i64 ntiles_all = ntiles + (p.batch > ntiles * PG::kWarpTile ? 1 : 0);
  i64 grid = dev.sm_count;  // one persistent CTA per SM
  if (grid > ntiles_all) grid = ntiles_all;
  cudaError_t e = launch_pdl(kern, unsigned(grid), unsigned(nwarps * 32), size_t(smem), stream, p, ntiles, nwarps, nbuf);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  if (e == cudaSuccess) record_launch(3, nwarps * 32, MPT, nbuf, nwarps, SEG, grid, ntiles_all);
  return int(e);
}

template <class Op>
int launch_strided(const KParams& p, cudaStream_t stream) {
  if (p.batch <= 0) return 0;
  const DeviceInfo& dev = device_info();
  i64 blocks = (p.batch + 127) / 128;
  const i64 cap = i64(dev.sm_count) * 16;
  if (blocks > cap) blocks = cap;
  cudaError_t e = launch_pdl(strided_kernel<Op>, unsigned(blocks), 128, size_t(0), stream, p);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  return int(e);
}

// Run an op over p.batch matrices: TMA-staged tiles for the bulk when every
// operand is dense-or-broadcast and 16 B aligned, strided kernel for the rest.
template <class Op>
int run_op(KParams p, cudaStream_t stream) {
  using Tn = Tune<Op>;
  t_last_path_tma = 0;
  reset_launch_record();
  if (p.batch == 0) return NFM_OK;
  const int lens[kMaxIn] = {Op::kLen0, Op::kLen1, Op::kLen2, len3<Op>::value};
  bool fast = p.out_stride == Op::kOut && elem_stride(p.out_estride) == 1 && aligned16(p.out);
  int nstaged = 0;
  for (int i = 0; i < kMaxIn && fast; ++i) {
    if (!((p.present >> i) & 1)) continue;
    if (elem_stride(p.in[i].estride) != 1) fast = false;
    if (p.in[i].stride == 0) continue;  // broadcast
    if (p.in[i].stride != lens[i] || !aligned16(p.in[i].ptr)) fast = false;
    ++nstaged;
  }
  if (fast && nstaged == 0) fast = false;
  if (!fast && p.batch > 64) {
    // Dense operands that only miss the 16-byte alignment (a view with a storage offset):
    // peel the first h < 4 matrices so that every staged pointer becomes aligned, do those
    // with the strided kernel and the rest on the TMA path.
    bool dense = p.out_stride == Op::kOut && elem_stride(p.out_estride) == 1;
    int any = 0;
    for (int i = 0; i < kMaxIn && dense; ++i) {
      if (!((p.present >> i) & 1)) continue;
      if (elem_stride(p.in[i].estride) != 1 || (p.in[i].stride != 0 && p.in[i].stride != lens[i])) dense = false;
      any += p.in[i].stride != 0;
    }
    if (dense && any > 0) {
      constexpr int es = int(sizeof(typename Op::scalar));
      for (int h = 1; h < 4; ++h) {
        bool ok = (reinterpret_cast<uintptr_t>(p.out) + size_t(h) * Op::kOut * es) % 16 == 0;
        for (int i = 0; i < kMaxIn && ok; ++i)
          if (((p.present >> i) & 1) && p.in[i].stride != 0)
            ok = (reinterpret_cast<uintptr_t>(p.in[i].ptr) + size_t(h) * lens[i] * es) % 16 == 0;
        if (!ok) continue;
        KParams head = p;
        head.batch = h;
        int rc = launch_strided<Op>(head, stream);
        if (rc != 0) {
          set_error("strided kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
          return rc;
        }
        KParams rest = p;
        for (int i = 0; i < kMaxIn; ++i)
          if (((p.present >> i) & 1) && p.in[i].stride != 0)
            rest.in[i].ptr = static_cast<const unsigned char*>(p.in[i].ptr) + size_t(h) * lens[i] * es;
        rest.out = static_cast<unsigned char*>(p.out) + size_t(h) * Op::kOut * es;
        rest.batch = p.batch - h;
        return run_op<Op>(rest, stream);  // aligned now: takes the fast path
      }
    }
  }
  if (fast) {
    // full tiles and the partial tile by TMA; the < 4-matrix tail in a second tiny launch
    int rc;
    if constexpr (PoolTune<Op>::kEnabled) {
      using Pt = PoolTune<Op>;
      int warps, nbuf;
      Pt::geometry(PoolGeom<Op, Pt::kMpt, Tn::kSeg>::buf_bytes(staged_mask(p)), device_info().max_smem_optin, warps, nbuf);
      rc = launch_pool<Op, Pt::kMaxW, Pt::kMpt, Tn::kSeg>(p, warps, nbuf, stream);
    } else if constexpr (TuneSmall<Op>::kEnabled) {
      using Ts = TuneSmall<Op>;
      const bool small = p.batch * Ts::kRec < Ts::kBelowBytes;
      rc = small ? -1 : launch_tile<Op, Tn::kThreads, Tn::kMpt, Tn::kStages, Tn::kSeg>(p, stream);
      // the large geometry's ring is sized for the mandatory operands; with the optional ones staged
      // as well it can pass the shared-memory limit (fp32 7x7 scaled-identity addmatvec: 241,704 B):
      // the small geometry then keeps the batch on the TMA path
      if (rc < 0) rc = launch_tile<Op, Ts::kThreads, Ts::kMpt, Ts::kStages, Tn::kSeg>(p, stream);
    } else {
      rc = launch_tile<Op, Tn::kThreads, Tn::kMpt, Tn::kStages, Tn::kSeg>(p, stream);
    }
    if (rc == 0) {
      t_last_path_tma = PoolTune<Op>::kEnabled ? 3 : 1;
      return NFM_OK;
    }
    if (rc > 0) {
      set_error("tile kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
      return rc;
    }
  }
  int rc = launch_strided<Op>(p, stream);
  if (rc != 0) set_error("strided kernel launch failed: %s", cudaGetErrorString(cudaError_t(rc)));
  return rc;
}

}  // namespace nfm
