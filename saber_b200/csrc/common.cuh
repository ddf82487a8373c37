// saber_b200 — shared device/host helpers for the sm_100a kernels.
// PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

// ---------------------------------------------------------------------------------------------
// Error plumbing (per-thread last-error string, C ABI returns negative codes)
// ---------------------------------------------------------------------------------------------
#define SB_OK 0
#define SB_ERR_CUDA -1
#define SB_ERR_ARG -2
#define SB_ERR_UNSUPPORTED -3
#define SB_ERR_DRIVER -4

void sb_set_error(const char* fmt, ...);

#define SB_CHECK_CUDA(expr)                                                                  \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      sb_set_error("%s:%d CUDA error %d (%s) in %s", __FILE__, __LINE__, (int)_e,            \
                   cudaGetErrorString(_e), #expr);                                           \
      return SB_ERR_CUDA;                                                                    \
    }                                                                                        \
  } while (0)

#define SB_CHECK_LAUNCH()  SB_CHECK_CUDA(cudaGetLastError())

#define SB_REQUIRE(cond, ...)                                                                \
  do {                                                                                       \
    if (!(cond)) {                                                                           \
      sb_set_error(__VA_ARGS__);                                                             \
      return SB_ERR_ARG;                                                                     \
    }                                                                                        \
  } while (0)

// cudaFuncSetAttribute is per device (context): SABER's GPUPool drives several GPUs from the threads of one process
// (REF saber/utils/parallelization.py:155), so the "attribute already set" caches are kept per device, not per process.
#include <atomic>
struct SbPerDeviceOnce {
  std::atomic<unsigned long long> done{0};  // bit d: set on device d (d < 64)
  bool need() {
    int d = 0;
    cudaGetDevice(&d);
    return ((done.load(std::memory_order_acquire) >> (d & 63)) & 1ull) == 0ull;
  }
  void mark() {
    int d = 0;
    cudaGetDevice(&d);
    done.fetch_or(1ull << (d & 63), std::memory_order_release);
  }
};

// Host: encode a 2-D bf16 row-major tensor map (rows x cols, row pitch ld elements), 128B swizzle.
// box = (box_cols elements [inner], box_rows). Returns SB_OK or error.
int sb_make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols,
                         uint64_t ld_elems, uint32_t box_rows, uint32_t box_cols);

// Host: 2-D row-major tensor map of 2- or 4-byte elements with a chosen swizzle (0 / 32 / 64 / 128 bytes).
int sb_make_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                    uint32_t box_rows, uint32_t box_cols, int swizzle_bytes);

// Host: encode a rank-`rank` (<= 5) bf16 tensor map. dims / box are in elements (fastest dimension first),
// strides_bytes[i] is the byte stride of dimension i + 1 (rank - 1 entries, multiples of 16). swizzle_bytes in
// {0, 32, 64, 128}: the inner box must not exceed it. Out-of-bounds elements read as zero.
int sb_make_tmap_nd_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

#ifdef __CUDACC__
namespace sb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ uint32_t lane_id() {
  uint32_t l;
  asm volatile("mov.u32 %0, %%laneid;" : "=r"(l));
  return l;
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier -------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- TMA ------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load: coordinates (c0 = inner/column element index, c1 = row index)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
      "r"(c0), "r"(c1)
      : "memory");
}

// 4-D tile load: coordinates fastest dimension first
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
      "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// 4-D tile store (shared -> global) as part of the thread's current bulk async-group
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1,
                                             int32_t c2, int32_t c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
      ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
// 2-D tile store (c0 = column element index, c1 = row index)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
      ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
      : "memory");
}
// the same with the source given as a shared::cta address
__device__ __forceinline__ void tma_store_2d_addr(const CUtensorMap* m, uint32_t smem_addr, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
      ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_addr), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until the shared-memory source of all but the newest N bulk groups of this thread has been read
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---- thread-block clusters / CTA pairs (cta_group::2) ------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `smem_addr` (a shared::cta address of this CTA) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// Arrive on an mbarrier of another CTA of the cluster. Default (CTA-scope) semantics on purpose: the explicit
// .release.cluster form compiles to MEMBAR.ALL.CTA + ERRBAR in front of the arrive, which was 15 % of all warp samples
// of the pair GEMM (profiles/r02ze: ~25 % of its epilogue). The accumulator reads this arrive publishes are ordered by
// tcgen05.fence::before_thread_sync, which the callers issue first.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 2-D tile load issued by one CTA of a pair; the bytes complete on the mbarrier at shared::cluster address `bar_cluster`
// (the leader CTA's barrier)
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster, int32_t c0,
                                                int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs, 256 x N] (+)= A[128 rows from each CTA's smem] * B[N/2 rows from each CTA's smem]; issued by the
// leader CTA only
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the mbarrier at the same shared-memory offset in every CTA of `cta_mask` once all previously issued
// tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

// ---- tcgen05 --------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16/fp16 inputs with fp32 accumulate.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// The same with the A operand read from tensor memory (M x K bf16 tile: row = TMEM lane, two consecutive K elements
// packed per 32-bit column, so one K = 16 step spans 8 columns): no shared-memory traffic for A.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
          smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 columns of fp32: thread i of the warp gets lane (base_lane + i), columns c..c+31.
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]),
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]),
        "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

// K-major, 128-byte-swizzled shared-memory matrix descriptor (rows of 64 bf16 = 128 B; 8-row
// groups are 1024 B apart). Field layout follows the sm_100 UMMA shared-memory descriptor:
// [0,14) start>>4, [16,30) LBO>>4 (ignored for swizzled K-major, set to 1), [32,46) SBO>>4,
// [46,48) version=1, [61,64) layout type (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// K-major, 32-byte-swizzled descriptor: rows of 16 bf16 = 32 B (exactly one k-step), 8-row groups 256 B apart
// (canonical layout Swizzle<1,4,3> o ((8,n),(T,2)):((2T,SBO),(1,T)); layout type 6 = SWIZZLE_32B).
__device__ __forceinline__ uint64_t umma_desc_k_sw32(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(256 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(6) << 61;
  return d;
}
// MN-major descriptors (the operand's M / N index is the contiguous one in shared memory: a [K rows][MN] tile).
// SWIZZLE_128B: atoms of 64 MN-elements (128 B) x 8 K-rows; LBO = byte distance between 64-element MN atoms,
// SBO = byte distance between 8-row K groups. SWIZZLE_32B: atoms of 16 MN-elements (32 B) x 8 K-rows.
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                 uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(sbo_bytes >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout_type) << 61;
  return d;
}
// Instruction descriptor: bf16 x bf16 -> fp32, both operands K-major, M x N tile.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

// 32 lanes x 16 columns of fp32
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}

// 32 lanes x 16 columns of fp32 back into TMEM (thread i writes lane base_lane + i)
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t* v) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// ---- small math -----------------------------------------------------------------------------
// GELU(x) = 0.5 x (1 + erf(x / sqrt 2)) with erf(z) ~ tanh(z (c0 + c1 z^2)) (minimax fit, |error| <= 2.8e-4 for all z; the
// argument is monotonic, so no clamping is needed) and tanh on the MUFU.TANH unit (tanh.approx.f32, rel. error 2^-11):
// 6 FMA-pipe instructions + 1 MUFU per element, less than half of the Abramowitz-Stegun form used before (14 + 2 MUFU).
// The GELU epilogues of the Hiera MLP GEMMs and of the mask-decoder up-scaling are instruction / MUFU bound on it. The
// absolute GELU error is <= 4e-4 + 2.5e-4 |x|, below the bf16 rounding (2^-9 relative) of every tensor these GELUs feed.
__device__ __forceinline__ float gelu_erf(float x) {
  const float z = x * 0.70710678118654752440f;
  const float p = fmaf(z * z, 0.0997927f, 1.12967583f);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(z * p));
  const float hx = 0.5f * x;
  return fmaf(hx, t, hx);
}
// ---- packed fp32 pairs (Blackwell FADD2 / FMUL2 / FFMA2: one issue slot for two lanes of fp32 math). The epilogues of
// the decoder GEMMs and the fused attention blocks are issue-bound on a handful of warps per SM. --------------------
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tadd.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmul.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 splat2(float a) { return make_float2(a, a); }
// gelu_erf on a pair: 6 packed instructions + 2 MUFU.TANH for two elements (7 + 1 per element in the scalar form)
__device__ __forceinline__ float2 gelu_erf2(float2 x) {
  const float2 z = mul2(x, splat2(0.70710678118654752440f));
  const float2 p = fma2(mul2(z, z), splat2(0.0997927f), splat2(1.12967583f));
  const float2 a = mul2(z, p);
  float2 t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.x) : "f"(a.x));
  asm("tanh.approx.f32 %0, %1;" : "=f"(t.y) : "f"(a.y));
  const float2 hx = mul2(x, splat2(0.5f));
  return fma2(hx, t, hx);
}

// 2^x on the MUFU unit without exp2f()'s denormal-range fix-up (3 extra instructions per call): inputs here are
// softmax exponents <= 0 (or -inf -> 0); results below 2^-126 flush to zero, which is what a softmax wants.
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace sb
#endif  // __CUDACC__
