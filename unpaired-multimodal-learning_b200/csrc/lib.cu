// Library plumbing: error string, device check, tensor-map encoding through the driver entry point
// (so the .so links against libcudart only and loads on a host without libcuda).
#include <cstdarg>

#include "common.cuh"

namespace uml {

static thread_local char g_err[512] = "ok";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn get_encode() {
  static encode_tiled_fn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess || p == nullptr)
    return nullptr;
  fn = reinterpret_cast<encode_tiled_fn>(p);
  return fn;
}

int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, uint32_t elem_bytes, uint64_t inner,
                 uint64_t outer, uint64_t row_pitch_bytes, uint32_t box_inner, uint32_t box_outer,
                 CUtensorMapSwizzle swizzle) {
  encode_tiled_fn enc = get_encode();
  UML_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  UML_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15u) == 0, "tensor map base must be 16B aligned");
  UML_REQUIRE(row_pitch_bytes % 16 == 0, "tensor map row pitch (%llu B) must be a multiple of 16",
              (unsigned long long)row_pitch_bytes);
  UML_REQUIRE(box_inner * elem_bytes <= 128 || swizzle == CU_TENSOR_MAP_SWIZZLE_NONE,
              "swizzled box inner extent must fit the swizzle span");
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_pitch_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  UML_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return 0;
}

// 3D row-major tensor (d0 contiguous): boxes land in shared memory as [box2][box1][box0], rows swizzled as asked
int make_tmap_3d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, uint64_t d0, uint64_t d1, uint64_t d2,
                 uint64_t pitch1_bytes, uint64_t pitch2_bytes, uint32_t box0, uint32_t box1, uint32_t box2,
                 CUtensorMapSwizzle swizzle) {
  encode_tiled_fn enc = get_encode();
  UML_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled not available from the driver");
  UML_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15u) == 0, "tensor map base must be 16B aligned");
  UML_REQUIRE(pitch1_bytes % 16 == 0 && pitch2_bytes % 16 == 0, "tensor map pitches (%llu, %llu B) must be multiples of 16",
              (unsigned long long)pitch1_bytes, (unsigned long long)pitch2_bytes);
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {pitch1_bytes, pitch2_bytes};
  cuuint32_t box[3] = {box0, box1, box2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(out, dtype, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  UML_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (3D) failed with CUresult %d", (int)r);
  return 0;
}

}  // namespace uml

extern "C" {

const char* uml_last_error(void) { return uml::g_err; }

int uml_abi_version(void) { return UML_B200_ABI_VERSION; }

int uml_device_ok(int device) {
  cudaDeviceProp prop;
  UML_CUDA(cudaGetDeviceProperties(&prop, device));
  UML_REQUIRE(prop.major == 10, "device %d is sm_%d%d; libuml_b200 is built for sm_100a only", device, prop.major,
              prop.minor);
  return 0;
}

}  // extern "C"
