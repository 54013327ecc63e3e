// hg_api.cu — library identity, error text, launch accounting and the TMA descriptor encoder.
#include "hg_common.cuh"

#include <atomic>
#include <cstdarg>
#include <cstring>
#include <cudaTypedefs.h>

#include "../../include/hifigan_b200.h"

std::atomic<int64_t> g_hg_launches{0};

static thread_local char g_err[512] = "";

void hg_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* hg_last_error(void) { return g_err; }
extern "C" const char* hg_version(void) { return "hifigan_b200 0.1 (sm_100a; tcgen05+TMA)"; }
extern "C" int hg_abi_version(void) { return HG_ABI_VERSION; }
extern "C" int64_t hg_launch_count(void) { return g_hg_launches.load(std::memory_order_relaxed); }
// one thread writes the GPU's nanosecond clock: a time mark INSIDE a captured graph (events cannot be read there)
__global__ void timestamp_kernel(unsigned long long* dst) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  *dst = t;
}

extern "C" int hg_timestamp(uint64_t* dst, void* stream) {
  HG_REQUIRE(dst != nullptr, "hg_timestamp: null destination");
  timestamp_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<unsigned long long*>(dst));
  HG_CHECK_CUDA(cudaGetLastError());
  return HG_OK;
}

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !sym) return nullptr;
  fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(sym);
  return fn;
}

int hg_encode_tmap_bf16_3d(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                           uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0,
                           uint32_t box1, uint32_t box2, int swizzle_bytes) {
  PFN_cuTensorMapEncodeTiled_v12000 enc = get_encode_fn();
  if (!enc) {
    hg_set_error("cuTensorMapEncodeTiled is not available from the driver");
    return HG_ERR_DRIVER;
  }
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {box0, box1, box2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMapSwizzle swz = swizzle_bytes == 128  ? CU_TENSOR_MAP_SWIZZLE_128B
                           : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                           : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                 : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    hg_set_error("cuTensorMapEncodeTiled failed (CUresult %d): dims=(%llu,%llu,%llu) strides=(%llu,%llu) "
                 "box=(%u,%u,%u) swizzle=%d base=%p",
                 (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
                 (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, box0, box1,
                 box2, swizzle_bytes, base);
    return HG_ERR_DRIVER;
  }
  return HG_OK;
}
