// tc_common.cuh — sm_100a building blocks of the bf16 throughput tier: mbarrier, TMA
// (cp.async.bulk.tensor), tcgen05.mma / TMEM, shared-memory + instruction descriptors, and the
// host-side tensor-map cache.  Inline PTX only (no CUTLASS): the descriptor bit layouts follow
// the PTX ISA "tcgen05 matrix / instruction descriptor" tables.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <unordered_map>

#include "common.cuh"

// ---------------------------------------------------------------- small PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug turns into a trap (CUDA error on the host) instead of a hung GPU.
#ifndef WN_WATCHDOG_CYCLES
#define WN_WATCHDOG_CYCLES 4000000000ll
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > WN_WATCHDOG_CYCLES) {
      printf("libwavenet_b200: mbarrier wait timed out (block %d,%d,%d thread %d)\n", blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x);
      __trap();
    }
  }
}

// generic-proxy writes -> visible to the async proxy (TMA / tcgen05 operand reads)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// CTA-pair (cta_group::2) loads: the box lands in THIS CTA's shared memory, the completion bytes are counted on the
// LEADER CTA's mbarrier (same offset, rank bit 24 of the shared::cluster address cleared), so that one barrier
// covers the operand halves of both CTAs before the leader issues tcgen05.mma.cta_group::2
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// ---------------------------------------------------------------- thread-block clusters
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of this cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(
          smem_u32(bar)),
      "r"(rank)
      : "memory");
}
// same without the cluster-scope release (measured ~2.7k cycles per call in the conv GEMM epilogue): for barriers
// that only hand TMEM accumulators back to the MMA warp — the tcgen05.ld results were already waited for and
// tcgen05.fence::before_thread_sync orders them; no generic-proxy data is published through this arrival
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint64_t* bar, uint32_t rank) {
  asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(smem_u32(bar)),
               "r"(rank)
               : "memory");
}
// ---------------------------------------------------------------- L2 cache policies (TMA .L2::cache_hint operands)
// Consecutive kernels of a block hand tensors of 32-64 MB to each other through the 126 MB L2; without hints
// every kernel streams > L2 worth of bytes and the hand-over tensors are evicted before the consumer runs
// (ncu: dgrad and wgrad re-read all of dz from DRAM).  Producer->consumer tensors are tagged evict_last,
// tensors whose next use is a whole pass away evict_first.  Encodings = createpolicy.fractional.L2::evict_*.b64 1.0.
#define TC_POL_NORMAL 0x1000000000000000ull
#define TC_POL_FIRST 0x12F0000000000000ull
#define TC_POL_LAST 0x14F0000000000000ull
__device__ __forceinline__ void tma_load_3d_h(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_h(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair_h(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_pair_h(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_pair_h(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3, uint64_t pol) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;" ::"r"(
          smem_u32(dst)),
      "l"(m), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d_h(const void* src, const CUtensorMap* m, int c0, int c1, int c2, uint64_t pol) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;" ::"l"(m), "r"(smem_u32(src)),
               "r"(c0), "r"(c1), "r"(c2), "l"(pol)
               : "memory");
}
// smem -> global tile store (bulk async group); rows / columns outside the tensor are clipped
__device__ __forceinline__ void tma_store_3d(const void* src, const CUtensorMap* m, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(m), "r"(smem_u32(src)), "r"(c0),
               "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_group() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
// producer half of a named barrier: counts this thread in, does not wait
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// ---------------------------------------------------------------- programmatic dependent launch
// The step is ~270 dependent launches of 25-40 us; without PDL every one pays launch latency, block scheduling and
// its prologue (barrier init, TMEM allocation, tensor-map fetch) after the previous kernel has fully drained.
// launch_dependents lets the next kernel's CTAs take over an SM as soon as this kernel's CTA there exits and run
// their prologue; wait blocks until the previous grid has completed and its writes are visible.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---------------------------------------------------------------- tcgen05 / TMEM
template <int NCOLS> __device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS> __device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
// CTA pair: the same warp of BOTH CTAs issues these; both get the same TMEM column range
template <int NCOLS> __device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int NCOLS> __device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; bf16 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// CTA pair: M = 256 rows split over the two CTAs (128 TMEM lanes each), the N x K operand B split in halves
// between their shared memories; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_bf16_pair(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs arrives on the barrier at this offset in both CTAs
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
// all previously issued tcgen05.mma of this thread arrive on `bar` when complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns: thread i of the warp gets lane (lane_base + i)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Accumulator row view handed to the epilogues (see epilogues.cuh): one thread = one TMEM lane.
struct TmemAccRow {
  uint32_t taddr;   // lane base in bits [16,32), first column of the tile in bits [0,16)
  bool valid;       // false for rows past the end of the sequence: loads still run (warp-collective), stores clip to 0
  __device__ __forceinline__ void load16(int c, float* v) const { tmem_ld16(taddr + (uint32_t)c, v); }
  __device__ __forceinline__ int clip(int nv) const { return valid ? nv : 0; }
};

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, 128-byte swizzle (what a TMA box with 128-byte inner extent
// and CU_TENSOR_MAP_SWIZZLE_128B produces).  Rows of 128 B; 8-row groups of 1024 B.
//   K-major operand  (rows = M/N index, 128 B = 64 bf16 of K): SBO = 1024 (next 8 rows), LBO unused.
//   MN-major operand (rows = K index,   128 B = 64 bf16 of M/N): SBO = 1024 (next 8 K), LBO = bytes
//   between consecutive 64-wide M/N atoms.
// Fields: start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | swizzle=2 (128B) [61,64)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}
// Instruction descriptor for kind::f16: D fp32 [4,6)=1, A bf16 [7,10)=1, B bf16 [10,13)=1,
// a_major bit 15, b_major bit 16 (0 = K-major, 1 = MN-major), N>>3 [17,23), M>>4 [24,29)
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// ---------------------------------------------------------------- host: per-device one-time setup
// cudaFuncSetAttribute and occupancy queries are per DEVICE: a process may hold handles on several GPUs (WaveNet(device=...)), so the
// "done once" state of every launcher is a bit per device ordinal, not a process-wide flag.  true the first time `mask` sees the
// current device.
static inline bool tc_first_use_on_device(unsigned long long* mask) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev > 63) return true;
  if ((*mask >> dev) & 1ull) return false;
  *mask |= 1ull << dev;
  return true;
}
static inline int tc_current_device() { int dev = 0; cudaGetDevice(&dev); return (dev < 0 || dev > 63) ? 0 : dev; }

// ---------------------------------------------------------------- host: tensor maps
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_tmapEncodeTiled g_tmap_encode = nullptr;
static thread_local char g_tc_err[256] = "";
static inline const char* tc_last_error() { return g_tc_err; }

static inline int tc_init() {
  if (g_tmap_encode) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return -1;
  g_tmap_encode = (PFN_tmapEncodeTiled)fn;
  return 0;
}

struct TmapKey {
  const void* base;
  uint64_t d[4], s[3];
  uint32_t box[4];
  uint32_t rank;
  uint32_t swz;
  bool operator==(const TmapKey& o) const {
    if (base != o.base || rank != o.rank || swz != o.swz) return false;
    for (int i = 0; i < 4; ++i) if (d[i] != o.d[i] || box[i] != o.box[i]) return false;
    for (int i = 0; i < 3; ++i) if (s[i] != o.s[i]) return false;
    return true;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = (uint64_t)(uintptr_t)k.base * 0x9E3779B97F4A7C15ull;
    for (int i = 0; i < 4; ++i) h = (h ^ (k.d[i] + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2))) * 1099511628211ull;
    for (int i = 0; i < 3; ++i) h = (h ^ k.s[i]) * 1099511628211ull;
    for (int i = 0; i < 4; ++i) h = (h ^ k.box[i]) * 1099511628211ull;
    return (size_t)(h ^ k.rank ^ ((uint64_t)k.swz << 8));
  }
};
// Encoding a tensor map costs microseconds on the host; a training step reuses the same few
// hundred (buffer, shape) combinations every iteration, so they are cached per handle.
struct TmapCache {
  std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> maps;
  // bf16 tensor, rank 2..4, dims innermost first, strides in BYTES for dims 1..rank-1, 128B swizzle, zero OOB fill
  // swizzle_bytes: 128 (inner box extent 128 B) or 64 (inner box extent 64 B)
  // swizzle_bytes: 128 / 64; fp32 = true encodes a FLOAT32 tensor (swizzle code 128 + 1 in the key), else bf16
  const CUtensorMap* get(const void* base, int rank, const uint64_t* dims, const uint64_t* strides, const uint32_t* box, int swizzle_bytes = 128,
                         bool fp32 = false) {
    TmapKey k{};
    k.base = base; k.rank = (uint32_t)rank; k.swz = (uint32_t)swizzle_bytes + (fp32 ? 1u : 0u);
    for (int i = 0; i < rank; ++i) { k.d[i] = dims[i]; k.box[i] = box[i]; }
    for (int i = 0; i + 1 < rank; ++i) k.s[i] = strides[i];
    auto it = maps.find(k);
    if (it != maps.end()) return &it->second;
    if (!g_tmap_encode) { snprintf(g_tc_err, sizeof(g_tc_err), "tensor-map encoder not initialised"); return nullptr; }
    if (((uintptr_t)base & 15) != 0) { snprintf(g_tc_err, sizeof(g_tc_err), "TMA base %p not 16-byte aligned", base); return nullptr; }
    for (int i = 0; i + 1 < rank; ++i)
      if (strides[i] % 16 != 0) { snprintf(g_tc_err, sizeof(g_tc_err), "TMA stride %llu not a multiple of 16 bytes", (unsigned long long)strides[i]); return nullptr; }
    CUtensorMap m;
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = g_tmap_encode(&m, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), (const cuuint64_t*)dims,
                               (const cuuint64_t*)strides, (const cuuint32_t*)box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      snprintf(g_tc_err, sizeof(g_tc_err), "cuTensorMapEncodeTiled failed (%d): rank %d dims %llu,%llu,%llu,%llu box %u,%u,%u,%u", (int)r, rank,
               (unsigned long long)k.d[0], (unsigned long long)k.d[1], (unsigned long long)k.d[2], (unsigned long long)k.d[3], box[0], box[1],
               rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
      return nullptr;
    }
    auto ins = maps.emplace(k, m);
    return &ins.first->second;
  }
};
