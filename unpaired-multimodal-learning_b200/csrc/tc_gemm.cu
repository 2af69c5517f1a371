// Generic bf16 tensor-core GEMM (tcgen05 + TMEM + TMA) used for every dense contraction of the hot
// path that is not the fused forward:
//
//   dW      = G^T X        (K4)  A, B both MN-major, fp32 split-K partials        finetune.py:190-193
//   Z       = X_img Wp^T   (K5)  A, B both K-major, bf16 out                      head.py:65,79
//   dZ      = G_img W      (K5)  A K-major, B MN-major, bf16 out                  autograd of head.py:80
//   dW_proj = dZ^T X_img   (K5)  A, B both MN-major, fp32 split-K partials
//
//   D[m,n] = sum_k A(m,k) B(k,n)
//     A K-major : A stored [M, K] (k contiguous)      A MN-major: A stored [K, M] (m contiguous)
//     B K-major : B stored [N, K] (k contiguous)      B MN-major: B stored [K, N] (n contiguous)
// Operands go from row-major HBM straight into 128B-swizzled shared memory by TMA and are described
// to the MMA unit as K-major or MN-major tiles; nothing is transposed in memory.
//
// kCG = 2 runs the MMA across a CTA pair (cta_group::2): the pair owns a 256 x 256 output tile, each
// CTA stages its own 128 rows of A and HALF of B (128 of the 256 N columns), so shared-memory fill
// traffic per FLOP drops by a third versus two independent 128 x 256 tiles - the operand stream from
// L2 is what bounds these GEMMs at ~870 TFLOP/s in single-CTA mode.
#include <cstdlib>

#include "common.cuh"

// Order in which a split walks the contraction: k-blocks split, split + S, split + 2S, ..., newest first.  The dW GEMM
// contracts over the batch rows, and the forward kernel has just written G in ascending row order: the newest rows are
// the ones still in L2.
// Measured on B200 inside the cfg3 step (73 728 rows, 6 splits): 0.2246-0.2270 ms/step with a contiguous slice per split
// (ascending or descending), 0.2228-0.2232 with this order - every CTA then reads neighbouring k-blocks at the same time
// (the 3 + 8 CTAs that share a block of G or X meet in L2) and the sweep starts where G is still resident.

namespace uml {

constexpr int kGBlockK = 64;
constexpr int kGBoxBytes = 64 * 64 * 2;  // one 64 x 64 bf16 box (8 KB): 64 rows of 128 B

template <int kCG>
struct GemmCfg {
  static constexpr int kTileM = 128 * kCG;           // output rows per cluster
  static constexpr int kTileN = 256;                 // output columns per cluster
  static constexpr int kCtaN = 256 / kCG;            // B columns staged by one CTA
  static constexpr int kABytes = 128 * kGBlockK * 2; // 16 KB
  static constexpr int kBBytes = kCtaN * kGBlockK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // 192 KB of operand stages either way: the split-K GEMMs stream both operands from HBM, and ~1 us of
  // DRAM latency at 32 KB per 0.27 us needs > 4 stages in flight
  static constexpr int kStages = kCG == 2 ? 6 : 4;
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 256;
};

// the dW GEMM's side job: the exchange forward kernel's per-(tile, chunk, warp) partials (tc_fwd2.cu), reduced into
// `stats` by an idle warp of the first CTA - the forward's statistics cost no launch of their own
struct DwStatsJob {
  const float* part;
  int64_t part_entries;
  int nseg;
  uml_seg_stats* stats;
};

template <bool kAMn, bool kBMn, bool kOutBf16, int kCG>
__global__ void __launch_bounds__(256, 1)
    tc_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, int64_t M,
                   int64_t N, int64_t K, int n_splits, void* __restrict__ out_v, int64_t ldo, DwStatsJob job) {
  using Cfg = GemmCfg<kCG>;
  constexpr int kGStages = Cfg::kStages;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kGStages * Cfg::kStageBytes);
  uint64_t* empty_bar = full_bar + kGStages;
  uint64_t* tfull_bar = empty_bar + kGStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (kCG == 2) ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  const int m_tile = blockIdx.x / kCG, n_tile = blockIdx.y, split = blockIdx.z;
  const int64_t m_cta = static_cast<int64_t>(m_tile) * Cfg::kTileM + rank * 128;   // first output row of this CTA
  const int64_t n_cta = static_cast<int64_t>(n_tile) * Cfg::kTileN + rank * Cfg::kCtaN;  // first B column staged here
  const int num_kb = static_cast<int>((K + kGBlockK - 1) / kGBlockK);
  // this split's k-blocks; block j of the walk is split + n_splits * (kb_hi - 1 - j)
  const int kb_hi = (num_kb - split + n_splits - 1) / n_splits;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kGStages; ++s) {
      mbar_init(&full_bar[s], kCG);  // one arrival per producer of the pair; tx bytes are counted on the leader
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    if (kCG == 2) tmem_alloc_cg2(tmem_slot, 256);
    else tmem_alloc(tmem_slot, 256);
  }
  tc_fence_before();
  if (kCG == 2) cluster_sync_all();  // peer barriers are initialised before anyone signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------ TMA producer (every CTA) -------------------
    if (lane == 0) {
      uint32_t it = 0;
      for (int kb = 0; kb < kb_hi; ++kb, ++it) {
        const uint32_t s = it % kGStages, ph = (it / kGStages) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        unsigned char* a = smem + s * Cfg::kStageBytes;
        unsigned char* b = a + Cfg::kABytes;
        const int32_t k0 = (split + n_splits * (kb_hi - 1 - kb)) * kGBlockK;
        if (kCG == 1) {
          mbar_arrive_expect_tx(&full_bar[s], Cfg::kStageBytes);
          if (kAMn) {
            tma_load_2d(a, &tmap_a, &full_bar[s], static_cast<int32_t>(m_cta), k0);
            tma_load_2d(a + kGBoxBytes, &tmap_a, &full_bar[s], static_cast<int32_t>(m_cta + 64), k0);
          } else {
            tma_load_2d(a, &tmap_a, &full_bar[s], k0, static_cast<int32_t>(m_cta));
          }
          if (kBMn) {
#pragma unroll
            for (int j = 0; j < Cfg::kCtaN / 64; ++j)
              tma_load_2d(b + j * kGBoxBytes, &tmap_b, &full_bar[s], static_cast<int32_t>(n_cta + j * 64), k0);
          } else {
            tma_load_2d(b, &tmap_b, &full_bar[s], k0, static_cast<int32_t>(n_cta));
          }
        } else {
          const uint32_t lead_bar = mapa_cta(smem_u32(&full_bar[s]), 0);
          if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * Cfg::kStageBytes);
          if (kAMn) {
            tma_load_2d_cg2(a, &tmap_a, lead_bar, static_cast<int32_t>(m_cta), k0);
            tma_load_2d_cg2(a + kGBoxBytes, &tmap_a, lead_bar, static_cast<int32_t>(m_cta + 64), k0);
          } else {
            tma_load_2d_cg2(a, &tmap_a, lead_bar, k0, static_cast<int32_t>(m_cta));
          }
          if (kBMn) {
#pragma unroll
            for (int j = 0; j < Cfg::kCtaN / 64; ++j)
              tma_load_2d_cg2(b + j * kGBoxBytes, &tmap_b, lead_bar, static_cast<int32_t>(n_cta + j * 64), k0);
          } else {
            tma_load_2d_cg2(b, &tmap_b, lead_bar, k0, static_cast<int32_t>(n_cta));
          }
          if (!leader) mbar_arrive_remote(lead_bar);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ------------------------------------------------ MMA issuer (leader CTA of the pair) --------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16(Cfg::kTileM, Cfg::kTileN, kAMn ? 1 : 0, kBMn ? 1 : 0);
      uint32_t it = 0;
      for (int kb = 0; kb < kb_hi; ++kb, ++it) {
        const uint32_t s = it % kGStages, ph = (it / kGStages) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(smem + s * Cfg::kStageBytes);
        const uint32_t b_addr = a_addr + Cfg::kABytes;
#pragma unroll
        for (int k = 0; k < kGBlockK / 16; ++k) {
          // K-major : 8-row groups 1024 B apart (SBO), a K step of 16 elements = 32 B inside the swizzle atom
          // MN-major: a row (one k) = 64 MN elements = 128 B, 8-row groups 1024 B apart (SBO), the next 64 MN
          //           elements in the next box (LBO = 8 KB), a K step of 16 rows = 2048 B
          const uint64_t da = kAMn ? make_smem_desc(a_addr + k * 2048, kGBoxBytes, 1024, kLayoutSw128)
                                   : make_smem_desc(a_addr + k * 32, 16, 1024, kLayoutSw128);
          const uint64_t db = kBMn ? make_smem_desc(b_addr + k * 2048, kGBoxBytes, 1024, kLayoutSw128)
                                   : make_smem_desc(b_addr + k * 32, 16, 1024, kLayoutSw128);
          if (kCG == 2) umma_bf16_cg2(tmem_base, da, db, idesc, (it | k) != 0);
          else umma_bf16(tmem_base, da, db, idesc, (it | k) != 0);
        }
        if (kCG == 2) umma_commit_cg2(&empty_bar[s]);
        else umma_commit(&empty_bar[s]);
      }
      if (kCG == 2) umma_commit_cg2(tfull_bar);
      else umma_commit(tfull_bar);
    }
    __syncwarp();
  } else if (warp == 3) {
    // ------------------------------------------------ per-run statistics of the exchange forward kernel -------
    if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && job.stats && job.part) {
      for (int sgi = 0; sgi < job.nseg; ++sgi) {
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        for (int64_t i0 = 0; i0 < job.part_entries; i0 += 128) {  // four independent 16-byte loads in flight per lane
          float4 v[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int64_t i = i0 + u * 32 + lane;
            v[u] = i < job.part_entries ? __ldcg(reinterpret_cast<const float4*>(job.part) + i * 2 + sgi)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) { acc[0] += v[u].x; acc[1] += v[u].y; acc[2] += v[u].z; acc[3] += v[u].w; }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[k] = warp_sum(acc[k]);
        if (lane == 0) {
          job.stats[sgi].loss_mean = acc[3] > 0.f ? acc[0] / acc[3] : 0.f;
          job.stats[sgi].dscale = acc[1];
          job.stats[sgi].correct = static_cast<int32_t>(acc[2] + 0.5f);
          job.stats[sgi].n = static_cast<int32_t>(acc[3] + 0.5f);
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------ epilogue (every CTA: its own 128 rows) ------
    const int q = warp - 4;
    const int64_t m = m_cta + q * 32 + lane;
    const bool have = kb_hi > 0;
    if (have) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int64_t n_base = static_cast<int64_t>(n_tile) * Cfg::kTileN;
#pragma unroll 1
    for (int cb = 0; cb < Cfg::kTileN / 32; ++cb) {
      uint32_t v[32];
      if (have) {
        tmem_ld32(taddr + cb * 32, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = 0u;
      }
      const int64_t n0 = n_base + cb * 32;
      if (m < M && n0 < N) {
        if (kOutBf16) {
          __nv_bfloat16* o = static_cast<__nv_bfloat16*>(out_v) + m * ldo + n0;
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            if (n0 + i + 8 <= N) {
              uint32_t w[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[i + 2 * j]), __uint_as_float(v[i + 2 * j + 1]));
                w[j] = *reinterpret_cast<uint32_t*>(&h);
              }
              *reinterpret_cast<uint4*>(o + i) = make_uint4(w[0], w[1], w[2], w[3]);
            } else {
              for (int j = 0; j < 8; ++j)
                if (n0 + i + j < N) o[i + j] = __float2bfloat16_rn(__uint_as_float(v[i + j]));
            }
          }
        } else {
          float* o = static_cast<float*>(out_v) + (static_cast<int64_t>(split) * M + m) * ldo + n0;
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            if (n0 + i + 4 <= N) {
              *reinterpret_cast<uint4*>(o + i) = make_uint4(v[i], v[i + 1], v[i + 2], v[i + 3]);
            } else {
              for (int j = 0; j < 4; ++j)
                if (n0 + i + j < N) o[i + j] = __uint_as_float(v[i + j]);
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  if (kCG == 2) cluster_sync_all();  // the peer may still be reading this CTA's shared memory / TMEM until here
  else __syncthreads();
  if (warp == 2) {
    if (kCG == 2) tmem_dealloc_cg2(tmem_base, 256);
    else tmem_dealloc(tmem_base, 256);
  }
}

static int cta_group_for(int64_t M) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("UML_TC_CTA_GROUP");
    forced = e ? atoi(e) : 0;
  }
  if (forced == 1 || forced == 2) return forced;
  return M > 128 ? 2 : 1;
}

static int gemm_splits(int64_t M, int64_t N, int64_t K, int cg) {
  const int64_t clusters = ((M + 128 * cg - 1) / (128 * cg)) * ((N + 255) / 256);
  const int64_t num_kb = (K + kGBlockK - 1) / kGBlockK;
  int64_t s = sm_count() / (clusters * cg > 0 ? clusters * cg : 1);
  if (s > num_kb) s = num_kb;
  if (s < 1) s = 1;
  return static_cast<int>(s);
}

template <bool kAMn, bool kBMn, bool kOutBf16, int kCG>
static int launch_tc_gemm(const CUtensorMap& ta, const CUtensorMap& tb, int64_t M, int64_t N, int64_t K, int n_splits,
                          void* out, int64_t ldo, cudaStream_t st, const DwStatsJob& job = DwStatsJob()) {
  using Cfg = GemmCfg<kCG>;
  auto kern = tc_gemm_kernel<kAMn, kBMn, kOutBf16, kCG>;
  static bool attr_set = false;
  if (!attr_set) {
    UML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  const dim3 grid(static_cast<unsigned>((M + Cfg::kTileM - 1) / Cfg::kTileM) * kCG,
                  static_cast<unsigned>((N + Cfg::kTileN - 1) / Cfg::kTileN), static_cast<unsigned>(n_splits));
  UML_CUDA(launch_kernel(kern, grid, dim3(256), Cfg::kSmemBytes, st, kCG, ta, tb, M, N, K, n_splits, out, ldo, job));
  return 0;
}

static int tc_gemm(const uint16_t* A, int64_t lda, bool a_mn, const uint16_t* B, int64_t ldb, bool b_mn, int64_t M,
                   int64_t N, int64_t K, void* out, int64_t ldo, bool out_bf16, int n_splits, cudaStream_t st,
                   const DwStatsJob* job = nullptr) {
  UML_REQUIRE(A && B && out && M > 0 && N > 0 && K > 0 && n_splits >= 1, "tc_gemm: bad arguments");
  UML_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "tc_gemm: leading dimensions must be multiples of 8 (16-byte bf16 rows)");
  UML_REQUIRE(!out_bf16 || n_splits == 1, "tc_gemm: split-K needs the fp32 partial output");
  UML_REQUIRE(out_bf16 ? (ldo % 8 == 0) : (ldo % 4 == 0), "tc_gemm: output leading dimension alignment");
  const int64_t num_kb = (K + kGBlockK - 1) / kGBlockK;
  UML_REQUIRE(n_splits <= num_kb, "tc_gemm: n_splits (%d) exceeds the %lld k-blocks", n_splits, (long long)num_kb);
  const int cg = cta_group_for(M);
  CUtensorMap ta, tb;
  // K-major operand: inner = K, outer = rows, box {64 k, rows per CTA}.  MN-major: inner = rows, outer = K, box {64, 64}.
  if (a_mn) {
    if (make_tmap_2d(&ta, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, M, K, lda * 2, 64, kGBlockK, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  } else {
    if (make_tmap_2d(&ta, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, K, M, lda * 2, kGBlockK, 128, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  if (b_mn) {
    if (make_tmap_2d(&tb, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, N, K, ldb * 2, 64, kGBlockK, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  } else {
    if (make_tmap_2d(&tb, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, K, N, ldb * 2, kGBlockK, 256 / cg, CU_TENSOR_MAP_SWIZZLE_128B)) return 1;
  }
  if (job) {  // statistics job: the dW kernel
    UML_REQUIRE(a_mn && b_mn && !out_bf16, "tc_gemm: the statistics job is wired for the dW layout only");
    return cg == 2 ? launch_tc_gemm<true, true, false, 2>(ta, tb, M, N, K, n_splits, out, ldo, st, *job)
                   : launch_tc_gemm<true, true, false, 1>(ta, tb, M, N, K, n_splits, out, ldo, st, *job);
  }
#define UML_GEMM_CASE(AM, BM, OB)                                                                              \
  if (a_mn == AM && b_mn == BM && out_bf16 == OB)                                                              \
    return cg == 2 ? launch_tc_gemm<AM, BM, OB, 2>(ta, tb, M, N, K, n_splits, out, ldo, st)                    \
                   : launch_tc_gemm<AM, BM, OB, 1>(ta, tb, M, N, K, n_splits, out, ldo, st);
  UML_GEMM_CASE(true, true, false)    // dW, dW_proj
  UML_GEMM_CASE(false, false, true)   // Z = X Wp^T
  UML_GEMM_CASE(false, true, true)    // dZ = G W
  UML_GEMM_CASE(false, false, false)  // fp32 NT (tests / generic use)
#undef UML_GEMM_CASE
  UML_FAIL("tc_gemm: operand layout combination a_mn=%d b_mn=%d out_bf16=%d is not instantiated", (int)a_mn, (int)b_mn,
           (int)out_bf16);
}

}  // namespace uml

// dW that also reduces the exchange forward kernel's partial statistics (library-internal, step.cu)
int uml_head_bwd_dw_stats_bf16(const uint16_t* G, int64_t ldg, const uint16_t* X, int64_t n_rows, int32_t dim, int32_t n_classes,
                               float* partials, int32_t n_splits, const float* part, int64_t part_entries, int32_t nseg,
                               uml_seg_stats* stats, void* stream) {
  using namespace uml;
  UML_REQUIRE(G && X && partials && n_rows > 0 && n_splits >= 1 && part && stats && nseg >= 1 && nseg <= UML_MAX_SEGMENTS,
              "dw_stats: bad arguments");
  UML_REQUIRE(dim % 8 == 0 && ldg % 64 == 0 && ldg >= n_classes, "dw_stats: dim must be a multiple of 8 and ldg of 64");
  const DwStatsJob job{part, part_entries, nseg, stats};
  return tc_gemm(G, ldg, true, X, dim, true, n_classes, dim, n_rows, partials, dim, false, n_splits, as_stream(stream), &job);
}

extern "C" {

int uml_gemm_bf16(const uint16_t* A, int64_t lda, int32_t a_mn_major, const uint16_t* B, int64_t ldb,
                  int32_t b_mn_major, int64_t M, int64_t N, int64_t K, void* out, int64_t ldo, int32_t out_bf16,
                  int32_t n_splits, void* stream) {
  return uml::tc_gemm(A, lda, a_mn_major != 0, B, ldb, b_mn_major != 0, M, N, K, out, ldo, out_bf16 != 0, n_splits,
                      uml::as_stream(stream));
}

int uml_gemm_bf16_splits(int64_t M, int64_t N, int64_t K) {
  return uml::gemm_splits(M, N, K, uml::cta_group_for(M));
}

int uml_tc_dw_splits(int64_t n_rows, int32_t dim, int32_t n_classes) {
  return uml::gemm_splits(n_classes, dim, n_rows, uml::cta_group_for(n_classes));
}

int uml_head_bwd_dw_bf16(const uint16_t* G, int64_t ldg, const uint16_t* X, int64_t n_rows, int32_t dim,
                         int32_t n_classes, float* partials, int32_t n_splits, void* stream) {
  using namespace uml;
  UML_REQUIRE(G && X && partials && n_rows > 0 && dim > 0 && n_classes > 0 && n_splits >= 1,
              "head_bwd_dw_bf16: bad arguments");
  UML_REQUIRE(dim % 8 == 0 && ldg % 64 == 0 && ldg >= n_classes,
              "head_bwd_dw_bf16: dim must be a multiple of 8 and ldg a multiple of 64 >= n_classes");
  UML_REQUIRE((reinterpret_cast<uintptr_t>(partials) & 15u) == 0, "head_bwd_dw_bf16: partials must be 16B aligned");
  // dW[c,d] = sum_b G[b,c] X[b,d]: A = G stored [K=b, M=c], B = X stored [K=b, N=d]
  return tc_gemm(G, ldg, true, X, dim, true, n_classes, dim, n_rows, partials, dim, false, n_splits, as_stream(stream));
}

}  // extern "C"
