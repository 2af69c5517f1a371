// K1 - index-driven row gather from an HBM-resident feature bank.
//
// Replaces the reference's per-sample Dataset.__getitem__ + default_collate + .to(device)
// (vision_language/finetune.py:165-172; engine/datasets/utils.py:100-101) with one launch.
//
// Data movement is done by the TMA engine: each bank row is a contiguous, 16-byte aligned run of
// dim*4 bytes, so one lane issues one `cp.async.bulk` (UBLKCP) global->shared per row, all rows of a
// stage completing on one mbarrier transaction count.  The fp32 variant drains a stage with
// `cp.async.bulk` shared->global; the bf16 variant converts in registers and writes 16-byte vectors
// (this is the A operand of the tcgen05 head GEMM).  Stages are ring-buffered so several hundred KB
// are in flight per SM, which is what an HBM-latency-bound gather needs.
#include <algorithm>

#include "common.cuh"

namespace uml {

struct CopySeg {
  const unsigned char* bank;   // row-major, row_bytes per row
  const int64_t* idx;          // gather indices (required)
  const int64_t* labels;       // bank labels (int64) or nullptr
  int64_t n;
};

constexpr int kGatherStages = 3;
constexpr int kGatherStageBytes = 48 * 1024;
constexpr int kGatherMaxRows = 32;  // one lane issues one row

template <bool kBf16>
__global__ void __launch_bounds__(kBf16 ? 128 : 32)
    gather_rows_kernel(const float* __restrict__ bank, const int64_t* __restrict__ idx, int64_t n, int dim,
                       int rows_per_stage, void* __restrict__ out_v, int64_t ld_out,
                       const int64_t* __restrict__ bank_labels, int32_t* __restrict__ out_labels) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full_bar[kGatherStages];
  const uint32_t row_bytes = static_cast<uint32_t>(dim) * 4u;
  const uint32_t stage_bytes = rows_per_stage * row_bytes;
  const int64_t n_groups = (n + rows_per_stage - 1) / rows_per_stage;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kGatherStages; ++s) mbar_init(&full_bar[s], 1);
    fence_barrier_init();
  }
  __syncthreads();

  auto issue = [&](int64_t it) {  // warp 0 only: fill stage it % S with group g(it)
    const int64_t g = blockIdx.x + it * gridDim.x;
    if (g >= n_groups) return;
    const int s = static_cast<int>(it % kGatherStages);
    const int64_t r0 = g * rows_per_stage;
    const int rows = static_cast<int>((n - r0) < rows_per_stage ? (n - r0) : rows_per_stage);
    if (lane == 0) mbar_arrive_expect_tx(&full_bar[s], rows * row_bytes);
    __syncwarp();
    if (lane < rows) {
      const int64_t src = idx ? idx[r0 + lane] : (r0 + lane);
      bulk_load_1d(smem + s * stage_bytes + lane * row_bytes, bank + src * dim, row_bytes, &full_bar[s]);
      if (out_labels) out_labels[r0 + lane] = static_cast<int32_t>(bank_labels[src]);  // label rides along
    }
  };

  if (warp == 0) {
    for (int p = 0; p < kGatherStages - 1; ++p) issue(p);
  }
  for (int64_t it = 0;; ++it) {
    const int64_t g = blockIdx.x + it * gridDim.x;
    if (g >= n_groups) break;
    const int s = static_cast<int>(it % kGatherStages);
    const int64_t r0 = g * rows_per_stage;
    const int rows = static_cast<int>((n - r0) < rows_per_stage ? (n - r0) : rows_per_stage);
    if (warp == 0) {
      if (!kBf16) bulk_wait_read<0>();  // the stage being refilled was drained by our own bulk stores
      issue(it + kGatherStages - 1);
    }
    mbar_wait(&full_bar[s], static_cast<uint32_t>((it / kGatherStages) & 1));
    if (!kBf16) {
      float* out = static_cast<float*>(out_v);
      if (lane < rows) {
        bulk_store_1d(out + (r0 + lane) * ld_out, smem + s * stage_bytes + lane * row_bytes, row_bytes);
      }
      bulk_commit();
    } else {
      __nv_bfloat16* out = static_cast<__nv_bfloat16*>(out_v);
      const int vec_per_row = dim >> 3;  // 8 elements -> one 16B store
      const float* st = reinterpret_cast<const float*>(smem + s * stage_bytes);
      for (int v = threadIdx.x; v < rows * vec_per_row; v += blockDim.x) {
        const int r = v / vec_per_row, c = (v - r * vec_per_row) << 3;
        const float4 a = *reinterpret_cast<const float4*>(st + r * dim + c);
        const float4 b = *reinterpret_cast<const float4*>(st + r * dim + c + 4);
        __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
        __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
        uint4 o;
        o.x = *reinterpret_cast<uint32_t*>(&p0);
        o.y = *reinterpret_cast<uint32_t*>(&p1);
        o.z = *reinterpret_cast<uint32_t*>(&p2);
        o.w = *reinterpret_cast<uint32_t*>(&p3);
        *reinterpret_cast<uint4*>(out + (r0 + r) * ld_out + c) = o;
      }
      __syncthreads();  // stage s may be refilled by warp 0 in the next iteration
    }
  }
  if (!kBf16) bulk_wait<0>();
}

__global__ void gather_labels_kernel(const int64_t* __restrict__ labels, const int64_t* __restrict__ idx, int64_t n,
                                     int32_t* __restrict__ out);

// Row copy for banks that already hold the operand type (the bf16 shadow of a feature bank): both runs of a
// step - image rows then text rows - in ONE launch, bytes moved by the TMA engine only (bulk global->shared,
// bulk shared->global), no thread ever touches the data.  4-stage ring of up to 48 KB each: the stage refilled at
// iteration `it` is the one whose stores were committed at `it - 1`, so one store group may stay in flight.
constexpr int kCopyStages = 4;

__global__ void __launch_bounds__(32)
    gather_copy2_kernel(CopySeg s0, CopySeg s1, uint32_t row_bytes, int rows_per_stage, unsigned char* __restrict__ out,
                        int64_t out_pitch, int32_t* __restrict__ out_labels) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ __align__(8) uint64_t full_bar[kCopyStages];
  const int64_t n = s0.n + s1.n;
  const uint32_t stage_bytes = rows_per_stage * row_bytes;
  const int64_t n_groups = (n + rows_per_stage - 1) / rows_per_stage;
  const int lane = threadIdx.x;
  if (lane == 0) {
    for (int s = 0; s < kCopyStages; ++s) mbar_init(&full_bar[s], 1);
    fence_barrier_init();
  }
  __syncwarp();

  auto issue = [&](int64_t it) {
    const int64_t g = blockIdx.x + it * gridDim.x;
    if (g >= n_groups) return;
    const int s = static_cast<int>(it % kCopyStages);
    const int64_t r0 = g * rows_per_stage;
    const int rows = static_cast<int>((n - r0) < rows_per_stage ? (n - r0) : rows_per_stage);
    if (lane == 0) mbar_arrive_expect_tx(&full_bar[s], rows * row_bytes);
    __syncwarp();
    if (lane < rows) {
      const int64_t r = r0 + lane;
      const bool second = r >= s0.n;
      const CopySeg& sg = second ? s1 : s0;
      const int64_t src = sg.idx[second ? r - s0.n : r];
      bulk_load_1d(smem + s * stage_bytes + lane * row_bytes, sg.bank + src * row_bytes, row_bytes, &full_bar[s]);
      if (out_labels) out_labels[r] = static_cast<int32_t>(sg.labels[src]);  // the label rides along
    }
  };

  for (int p = 0; p < kCopyStages - 1; ++p) issue(p);
  for (int64_t it = 0;; ++it) {
    const int64_t g = blockIdx.x + it * gridDim.x;
    if (g >= n_groups) break;
    const int s = static_cast<int>(it % kCopyStages);
    const int64_t r0 = g * rows_per_stage;
    const int rows = static_cast<int>((n - r0) < rows_per_stage ? (n - r0) : rows_per_stage);
    mbar_wait(&full_bar[s], static_cast<uint32_t>((it / kCopyStages) & 1));
    if (lane < rows) bulk_store_1d(out + (r0 + lane) * out_pitch, smem + s * stage_bytes + lane * row_bytes, row_bytes);
    bulk_commit();
    bulk_wait_read<1>();  // the group committed one iteration ago has left its stage
    __syncwarp();
    issue(it + kCopyStages - 1);
  }
  bulk_wait<0>();
}


// Fallback for rows that are not a multiple of 16 bytes (dim % 4 != 0; bf16 needs dim % 8 == 0).
template <bool kBf16>
__global__ void gather_rows_plain(const float* __restrict__ bank, const int64_t* __restrict__ idx, int64_t n, int dim,
                                  void* __restrict__ out_v, int64_t ld_out) {
  for (int64_t r = blockIdx.x; r < n; r += gridDim.x) {
    const int64_t src = idx ? idx[r] : r;
    for (int c = threadIdx.x; c < dim; c += blockDim.x) {
      const float x = bank[src * dim + c];
      if (kBf16)
        static_cast<__nv_bfloat16*>(out_v)[r * ld_out + c] = __float2bfloat16_rn(x);
      else
        static_cast<float*>(out_v)[r * ld_out + c] = x;
    }
  }
}

__global__ void gather_labels_kernel(const int64_t* __restrict__ labels, const int64_t* __restrict__ idx, int64_t n,
                                     int32_t* __restrict__ out) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) out[i] = static_cast<int32_t>(labels[idx ? idx[i] : i]);
}

__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * 8;
  for (int64_t i = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) * 8; i < n; i += stride) {
    if (i + 8 <= n) {
      const float4 a = *reinterpret_cast<const float4*>(src + i);
      const float4 b = *reinterpret_cast<const float4*>(src + i + 4);
      __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
      __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
      uint4 o;
      o.x = *reinterpret_cast<uint32_t*>(&p0);
      o.y = *reinterpret_cast<uint32_t*>(&p1);
      o.z = *reinterpret_cast<uint32_t*>(&p2);
      o.w = *reinterpret_cast<uint32_t*>(&p3);
      *reinterpret_cast<uint4*>(dst + i) = o;
    } else {
      for (int64_t j = i; j < n; ++j) dst[j] = __float2bfloat16_rn(src[j]);
    }
  }
}

// Same job as gather_copy2_kernel with a footprint small enough to share an SM with the GEMM kernels of the
// CURRENT step (no shared memory, <= 40 registers): uml_linear_run launches it on a low-priority side stream
// to fetch the NEXT step's rows while the tensor cores work.  One warp per row, 16-byte vectors, four rows in
// flight per warp.
__global__ void __launch_bounds__(256)
    gather_direct2_kernel(CopySeg s0, CopySeg s1, int vec_per_row, uint4* __restrict__ out, int64_t out_pitch_vec,
                          int32_t* __restrict__ out_labels) {
  const int64_t warp = (blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int64_t n = s0.n + s1.n;
  const int lane = threadIdx.x & 31;
  for (int64_t r = warp; r < n; r += n_warps) {
    const bool second = r >= s0.n;
    const CopySeg& sg = second ? s1 : s0;
    const int64_t src = __ldg(sg.idx + (second ? r - s0.n : r));
    const uint4* row = reinterpret_cast<const uint4*>(sg.bank) + src * vec_per_row;
    uint4* dst = out + r * out_pitch_vec;
    if (lane == 0 && out_labels) out_labels[r] = static_cast<int32_t>(__ldg(sg.labels + src));
    for (int v0 = 0; v0 < vec_per_row; v0 += 128) {
      uint4 x[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int v = v0 + j * 32 + lane;
        if (v < vec_per_row) x[j] = __ldcs(row + v);  // streamed: a bank row is read once per epoch
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int v = v0 + j * 32 + lane;
        if (v < vec_per_row) __stcs(dst + v, x[j]);  // read again a step or two later, after 0.5 GB of other traffic: not worth L2
      }
    }
  }
}

template <bool kBf16>
static int launch_gather(const float* bank, int64_t bank_rows, int32_t dim, const int64_t* idx, int64_t n, void* out,
                         int64_t ld_out, cudaStream_t st, const int64_t* bank_labels = nullptr,
                         int32_t* out_labels = nullptr) {
  if (n == 0) return 0;
  UML_REQUIRE(bank && out && dim > 0 && bank_rows > 0 && n > 0, "gather: bad arguments");
  const uint32_t row_bytes = static_cast<uint32_t>(dim) * 4u;
  const bool tma_ok = (row_bytes % 16 == 0) && (!kBf16 || dim % 8 == 0) && row_bytes <= kGatherStageBytes &&
                      (reinterpret_cast<uintptr_t>(bank) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0) &&
                      ((ld_out * (kBf16 ? 2 : 4)) % 16 == 0);
  if (!tma_ok) {
    const int grid = static_cast<int>(std::min<int64_t>(n, 148 * 8));
    gather_rows_plain<kBf16><<<grid, 256, 0, st>>>(bank, idx, n, dim, out, ld_out);
    UML_CUDA(cudaGetLastError());
    if (out_labels) {
      gather_labels_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(bank_labels, idx, n, out_labels);
      UML_CUDA(cudaGetLastError());
    }
    return 0;
  }
  int rows = kGatherStageBytes / row_bytes;
  if (rows > kGatherMaxRows) rows = kGatherMaxRows;
  const size_t smem = static_cast<size_t>(kGatherStages) * rows * row_bytes;
  static bool attr_set[2] = {false, false};
  if (!attr_set[kBf16]) {
    UML_CUDA(cudaFuncSetAttribute(gather_rows_kernel<kBf16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kGatherStages * kGatherStageBytes));
    attr_set[kBf16] = true;
  }
  const int64_t groups = (n + rows - 1) / rows;
  const int grid = static_cast<int>(std::min<int64_t>(groups, sm_count()));
  gather_rows_kernel<kBf16><<<grid, kBf16 ? 128 : 32, smem, st>>>(bank, idx, n, dim, rows, out, ld_out, bank_labels,
                                                                  out_labels);
  UML_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace uml

extern "C" {

int uml_gather_rows_f32(const float* bank, int64_t bank_rows, int32_t dim, const int64_t* idx, int64_t n, float* out,
                        void* stream) {
  return uml::launch_gather<false>(bank, bank_rows, dim, idx, n, out, dim, uml::as_stream(stream));
}

int uml_gather_rows_bf16(const float* bank, int64_t bank_rows, int32_t dim, const int64_t* idx, int64_t n,
                         uint16_t* out, int64_t ld_out, void* stream) {
  return uml::launch_gather<true>(bank, bank_rows, dim, idx, n, out, ld_out, uml::as_stream(stream));
}

int uml_gather_rows_labels_bf16(const float* bank, const int64_t* bank_labels, int32_t dim, const int64_t* idx,
                                int64_t n, uint16_t* out, int64_t ld_out, int32_t* out_labels, void* stream) {
  UML_REQUIRE(bank_labels && out_labels, "gather_rows_labels_bf16: null labels");
  return uml::launch_gather<true>(bank, INT64_MAX / 2, dim, idx, n, out, ld_out, uml::as_stream(stream), bank_labels,
                                  out_labels);
}

int uml_gather2_rows_bf16(const uint16_t* bank0, const int64_t* labels0, const int64_t* idx0, int64_t n0,
                          const uint16_t* bank1, const int64_t* labels1, const int64_t* idx1, int64_t n1, int32_t dim,
                          uint16_t* out, int64_t ld_out, int32_t* out_labels, void* stream) {
  using namespace uml;
  UML_REQUIRE(n0 >= 0 && n1 >= 0 && dim > 0 && out, "gather2: bad arguments");
  UML_REQUIRE((n0 == 0 || (bank0 && idx0)) && (n1 == 0 || (bank1 && idx1)), "gather2: null bank or index pointer");
  UML_REQUIRE(!out_labels || ((n0 == 0 || labels0) && (n1 == 0 || labels1)), "gather2: labels requested but not given");
  if (n0 + n1 == 0) return 0;
  const uint32_t row_bytes = static_cast<uint32_t>(dim) * 2u;
  UML_REQUIRE(row_bytes % 16 == 0 && (ld_out * 2) % 16 == 0 && row_bytes <= 48 * 1024, "gather2: rows must be 16B multiples");
  UML_REQUIRE(((reinterpret_cast<uintptr_t>(bank0) | reinterpret_cast<uintptr_t>(bank1) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0,
              "gather2: pointers must be 16B aligned");
  int rows = static_cast<int>(48 * 1024 / row_bytes);
  if (rows > 32) rows = 32;
  const size_t smem = static_cast<size_t>(kCopyStages) * rows * row_bytes;
  static bool attr_set = false;
  if (!attr_set) {
    UML_CUDA(cudaFuncSetAttribute(gather_copy2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  kCopyStages * 48 * 1024));
    attr_set = true;
  }
  const int64_t groups = (n0 + n1 + rows - 1) / rows;
  const int grid = static_cast<int>(std::min<int64_t>(groups, sm_count()));
  CopySeg a{reinterpret_cast<const unsigned char*>(bank0), idx0, labels0, n0};
  CopySeg b{reinterpret_cast<const unsigned char*>(bank1), idx1, labels1, n1};
  UML_CUDA(launch_kernel(gather_copy2_kernel, dim3(grid), dim3(32), smem, as_stream(stream), 1, a, b,
                         row_bytes, rows, reinterpret_cast<unsigned char*>(out), ld_out * 2, out_labels));
  return 0;
}

int uml_gather2_rows_bf16_light(const uint16_t* bank0, const int64_t* labels0, const int64_t* idx0, int64_t n0,
                                const uint16_t* bank1, const int64_t* labels1, const int64_t* idx1, int64_t n1, int32_t dim,
                                uint16_t* out, int64_t ld_out, int32_t* out_labels, void* stream) {
  using namespace uml;
  UML_REQUIRE(n0 >= 0 && n1 >= 0 && dim > 0 && out, "gather2_light: bad arguments");
  UML_REQUIRE((n0 == 0 || (bank0 && idx0)) && (n1 == 0 || (bank1 && idx1)), "gather2_light: null bank or index pointer");
  UML_REQUIRE(!out_labels || ((n0 == 0 || labels0) && (n1 == 0 || labels1)), "gather2_light: labels requested but not given");
  if (n0 + n1 == 0) return 0;
  UML_REQUIRE(dim % 8 == 0 && ld_out % 8 == 0, "gather2_light: rows must be 16B multiples");
  UML_REQUIRE(((reinterpret_cast<uintptr_t>(bank0) | reinterpret_cast<uintptr_t>(bank1) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0,
              "gather2_light: pointers must be 16B aligned");
  CopySeg a{reinterpret_cast<const unsigned char*>(bank0), idx0, labels0, n0};
  CopySeg b{reinterpret_cast<const unsigned char*>(bank1), idx1, labels1, n1};
  const int64_t blocks = std::min<int64_t>((n0 + n1 + 7) / 8, static_cast<int64_t>(sm_count()) * 4);
  gather_direct2_kernel<<<static_cast<unsigned>(blocks), 256, 0, as_stream(stream)>>>(a, b, dim / 8, reinterpret_cast<uint4*>(out),
                                                                                      ld_out / 8, out_labels);
  UML_CUDA(cudaGetLastError());
  return 0;
}

int uml_gather_labels_i32(const int64_t* bank_labels, const int64_t* idx, int64_t n, int32_t* out, void* stream) {
  if (n == 0) return 0;
  UML_REQUIRE(bank_labels && out && n > 0, "gather_labels: bad arguments");
  uml::gather_labels_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, uml::as_stream(stream)>>>(
      bank_labels, idx, n, out);
  UML_CUDA(cudaGetLastError());
  return 0;
}

int uml_cast_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, void* stream) {
  UML_REQUIRE(src && dst && n >= 0, "cast: bad arguments");
  if (n == 0) return 0;
  UML_REQUIRE(reinterpret_cast<uintptr_t>(src) % 16 == 0 && reinterpret_cast<uintptr_t>(dst) % 16 == 0,
              "cast: pointers must be 16B aligned");
  const int64_t vecs = (n + 7) / 8;
  const int grid = static_cast<int>(std::min<int64_t>((vecs + 255) / 256, 148 * 16));
  uml::cast_bf16_kernel<<<grid, 256, 0, uml::as_stream(stream)>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  UML_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
