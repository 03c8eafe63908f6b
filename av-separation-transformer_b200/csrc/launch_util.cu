// Host helpers shared by the kernel launchers: TMA descriptor encoding and the dynamic shared-memory opt-in.
#include "kernels.h"

#include <cudaTypedefs.h>

#include <map>
#include <mutex>
#include <utility>

namespace avsep {

namespace {

PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;

const char* encode(CUtensorMap* map, CUtensorMapDataType dt, uint32_t rank, const void* ptr, const cuuint64_t* dims,
                   const cuuint64_t* strides, const cuuint32_t* box) {
  if (g_encode == nullptr) return "tma: tma_init() has not run";
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0) return "tma: pointer not 16-byte aligned";
  if ((strides[0] & 15) != 0) return "tma: leading dimension not a multiple of 16 bytes";
  const cuuint32_t estr[3] = {1, 1, 1};
  if (g_encode(map, dt, rank, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) !=
      CUDA_SUCCESS)
    return "tma: cuTensorMapEncodeTiled failed";
  return nullptr;
}

}  // namespace

const char* tma_init() {
  if (g_encode != nullptr) return nullptr;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess || fn == nullptr)
    return "tma: cuTensorMapEncodeTiled entry point not found (driver too old?)";
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  return nullptr;
}

const char* tma_encode_2d(CUtensorMap* map, CUtensorMapDataType dt, int esz, const void* ptr, uint64_t inner,
                          uint64_t outer, uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  const cuuint64_t dims[2] = {inner, outer};
  const cuuint64_t strides[1] = {ld_elems * esz};
  const cuuint32_t box[2] = {box_inner, box_outer};
  return encode(map, dt, 2, ptr, dims, strides, box);
}

const char* tma_encode_3d(CUtensorMap* map, CUtensorMapDataType dt, int esz, const void* ptr, uint64_t inner,
                          uint64_t outer, uint64_t batches, uint64_t ld_elems, uint32_t box_inner, uint32_t box_outer) {
  const cuuint64_t dims[3] = {inner, outer, batches};
  const cuuint64_t strides[2] = {ld_elems * esz, outer * ld_elems * esz};
  const cuuint32_t box[3] = {box_inner, box_outer, 1};
  return encode(map, dt, 3, ptr, dims, strides, box);
}

bool smem_opt_in(const void* kern, int bytes) {
  if (bytes <= 48 * 1024) return true;
  int dev;
  if (cudaGetDevice(&dev) != cudaSuccess) return false;
  static std::mutex mu;
  // per (device, kernel): the largest limit set so far.  The attribute belongs to the kernel's image on the current
  // device, so a kernel opted in on one device still has the 48 KB default on the next.
  static std::map<std::pair<int, const void*>, int> limit;
  std::lock_guard<std::mutex> lock(mu);
  int& cur = limit[{dev, kern}];
  if (bytes <= cur) return true;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return false;
  cur = bytes;
  return true;
}

}  // namespace avsep
