// hg_common.cuh — shared device/host helpers for the hifigan_b200 sm_100a kernels.
//
// Thin inline-PTX wrappers for the Blackwell primitives the kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld) and
// the UMMA shared-memory / instruction descriptors.  Nothing in here is a
// translation of reference code: the reference (AlonKellner/hifi-gan) is pure
// Python on top of torch and owns no kernels (SURVEY.md §2.2).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <stdio.h>

// ----------------------------------------------------------------------------
// error plumbing (C-ABI convention: 0 = ok, negative = error, text via hg_last_error)
// ----------------------------------------------------------------------------
#define HG_OK 0
#define HG_ERR_INVALID (-1)
#define HG_ERR_CUDA (-2)
#define HG_ERR_UNSUPPORTED (-3)
#define HG_ERR_DRIVER (-4)

void hg_set_error(const char* fmt, ...);

#define HG_CHECK_CUDA(expr)                                                        \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      hg_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                   \
                   cudaGetErrorString(_e));                                        \
      return HG_ERR_CUDA;                                                          \
    }                                                                              \
  } while (0)

#define HG_REQUIRE(cond, ...)                                                      \
  do {                                                                             \
    if (!(cond)) {                                                                 \
      hg_set_error(__VA_ARGS__);                                                   \
      return HG_ERR_INVALID;                                                       \
    }                                                                              \
  } while (0)

namespace hg {

// Bounded spin on mbarrier waits: a protocol bug traps instead of hanging the GPU box.
#ifndef HG_SPIN_LIMIT
#define HG_SPIN_LIMIT (1u << 28)
#endif

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------- mbarrier ----------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > HG_SPIN_LIMIT) {
      printf("hg: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

// --------------------------------- TMA --------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0),
        "r"(c1), "r"(c2)
      : "memory");
}

// ------------------------------- tcgen05 ------------------------------------
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// whole-warp, .sync.aligned
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 operands, fp32 accumulate; issued by ONE elected thread.
// The descriptors are given as (low word, shared high word): the low word holds the 14-bit
// start address (>>4) so advancing an operand by `bytes` is `lo + (bytes >> 4)` — two integer adds per
// MMA instead of rebuilding two 64-bit descriptors (the issuing thread is instruction-bound otherwise).
__device__ __forceinline__ void umma_bf16_ss_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo,
                                                uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ---- cta_group::2 (CTA pair) variants ----------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 remAddr32;\n\t"
      "mapa.shared::cluster.u32 remAddr32, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [remAddr32];\n\t"
      "}\n"
      :
      : "r"(smem_u32(bar)), "r"(cta)
      : "memory");
}
// TMA load issued by either CTA of a pair; the transaction bytes are credited to the LEADER's barrier
// (same offset, peer bit cleared — cute::SM100_TMA_2SM_LOAD_3D).
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                                int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu),
        "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_result, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// M = 256 MMA over the CTA pair: each CTA supplies its 128 rows of A and half of B's N rows
__device__ __forceinline__ void umma_bf16_ss_lo_2sm(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo,
                                                    uint32_t desc_hi, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once all prior MMAs of this thread completed) on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      :
      : "r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
      : "memory");
}

__device__ __forceinline__ uint32_t umma_desc_lo(uint32_t saddr) {
  return ((saddr & 0x3FFFFu) >> 4) | (1u << 16);
}
__device__ __forceinline__ uint32_t umma_desc_hi(uint32_t sbo_bytes, uint32_t layout_type) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((layout_type & 7u) << 29);
}
// mbarrier arrives once every MMA issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// UMMA shared-memory descriptor, K-major operand (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base_offset |
//   [61,64) layout type (0 none, 2 = 128B swizzle, 4 = 64B, 6 = 32B)
// For the swizzled K-major layouts rows are `row_bytes` apart (128 / 64 / 32), 8-row groups are
// SBO = 8*row_bytes apart and LBO is ignored (set to 1).  Built as umma_desc_lo / umma_desc_hi below.

// UMMA instruction descriptor, kind::f16, BF16 x BF16 -> F32, both operands K-major
// (cute::UMMA::InstrDescriptor): c_format[4,6)=1, a_format[7,10)=1, b_format[10,13)=1,
// n>>3 at [17,23), m>>4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t w) {
  __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&w);
  return __bfloat1622float2(h);
}

struct U8 {
  uint32_t v[8];
};

__device__ __forceinline__ U8 ldg256(const void* p) {
  U8 r;
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]),
                 "=r"(r.v[6]), "=r"(r.v[7])
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg256(void* p, const U8& r) {
  asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r.v[0]),
               "r"(r.v[1]), "r"(r.v[2]), "r"(r.v[3]), "r"(r.v[4]), "r"(r.v[5]), "r"(r.v[6]),
               "r"(r.v[7])
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void add_bf16x16(float (&v)[16], const U8& r) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float2 f = unpack_bf16x2(r.v[i]);
    v[2 * i] += f.x;
    v[2 * i + 1] += f.y;
  }
}
// v += leaky_relu^-1(r): r holds bf16(leaky_relu(x, slope)) with 0 < slope <= 1 and inv_slope = 1 / slope computed
// on the host (inv_slope = 1: r is raw and the add is exact, as add_bf16x16).  min(a, a / slope) undoes the
// activation for either sign.  Multiplying by the fp32 reciprocal instead of dividing by slope differs from the
// division by at most one fp32 ulp, far below the 2^-9 relative rounding the bf16 copy already carries, which is
// the same error as storing x raw.
__device__ __forceinline__ void add_bf16x16_unlrelu(float (&v)[16], const U8& r, float inv_slope) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float2 f = unpack_bf16x2(r.v[i]);
    v[2 * i] += fminf(f.x, f.x * inv_slope);
    v[2 * i + 1] += fminf(f.y, f.y * inv_slope);
  }
}



// Column sums over the 32 lanes of a warp, N (power of two <= 16) columns per lane, in N - 1 + log2(32 / N) shuffles:
// a halving butterfly — at every step a lane hands the half of its columns it does not keep to its partner.
// Returns the sum of column `col` (set per lane: the lane bits consumed by the halving steps, most significant
// first); the 32 / N lanes that differ only in their low bits hold the same column.
template <int N>
__device__ __forceinline__ float warp_colsum(float (&v)[N], int lane, int& col) {
  int off = 16;
  col = 0;
#pragma unroll
  for (int w = N / 2; w >= 1; w >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float send = hi ? v[i] : v[i + w];
      const float keep = hi ? v[i + w] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
    if (hi) col += w;
    off >>= 1;
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1)
    if (o <= off) v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
  return v[0];
}

// cudaFuncSetAttribute is per DEVICE: launchers remember, per device ordinal, whether (or with which size) they
// already raised a kernel's dynamic shared-memory limit.  One process may drive several GPUs.
struct PerDeviceOnce {
  size_t done[64] = {};
  // true when `want` exceeds what was configured on the current device so far (and records it)
  bool need(size_t want = 1) {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
    if (done[d] >= want) return false;
    done[d] = want;
    return true;
  }
};
}  // namespace hg

// host-side: cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda needed)
int hg_encode_tmap_bf16_3d(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                           uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0,
                           uint32_t box1, uint32_t box2, int swizzle_bytes);
