// K2+K3 on the tensor cores: head forward, logit scale, softmax cross-entropy and the logit
// gradient G in ONE kernel (reference: engine/models/head.py:80-82,133-135 + finetune.py:186-188
// + the autograd of F.cross_entropy).
//
//   logits[b,c] = scale_b * sum_d X[b,d] W[c,d]         bf16 x bf16 -> fp32 in TMEM
//   G[b,c]      = w_b * scale_b / n_b * (softmax(logits)[b,c] - [c == y_b])     written as bf16
//
// One persistent CTA per SM (CTA pairs: cta_group::2), 384 threads, warp-specialised:
//   warp 11    TMA producer : X tile 128x64 + this CTA's half of the W chunk (128x64) per stage, 5 stages,
//                             SWIZZLE_128B; completion is counted on the pair leader's barrier
//   warp 10    MMA issuer   : (leader CTA) tcgen05.mma cta_group::2 kind::f16, M=256 (pair) N=256 K=16,
//                             accumulators in TMEM; two 256-column accumulator buffers so the MMA of class chunk
//                             j+1 overlaps the epilogue of chunk j
//   warp 8     TMEM allocator
//   warps 0-7  epilogue     : two groups of four warps that own alternate class chunks; one thread per row
//                             (TMEM lane).  Per chunk ONE sweep, 64 columns at a time: tcgen05.ld, scale, running
//                             row max / sum (online softmax), label logit, index-free hit flag; the unnormalised
//                             probabilities exp(l - m_running) are staged in shared memory in the 128B-swizzled
//                             layout and leave as coalesced TMA stores.  At the end of a tile the group that
//                             finishes last merges both groups' row statistics (through shared memory).
// A 1000-class fp32 row needs 1000 TMEM columns and an SM has 512, so a row cannot wait in TMEM for its final
// max / sum: the normalisation is DEFERRED - per row and 64-column group the factor exp(m_group - m_final) / sum *
// coef goes to a small side array and g_fixup_kernel (below) applies it, together with the one-hot term, in one
// coalesced pass over G while it is still in L2.  (Alternatives measured: normaliser warps inside this kernel - slower;
// the same transform applied to the dW kernel's operand stages - bit-identical but shared-memory bound, see DESIGN.md.)
// Logits never exist in HBM in fp32 and nothing is recomputed.
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace uml {

constexpr int kFwdBlockM = 128;
constexpr int kFwdBlockN = 256;
constexpr int kFwdBlockK = 64;
constexpr int kFwdABytes = kFwdBlockM * kFwdBlockK * 2;
// kCG = 2: the CTA pair shares the W chunk (each CTA stages 128 of its 256 class rows) and the MMA runs as
// cta_group::2 with M = 256.
template <int kCG>
struct FwdCfg {
  static constexpr int kBBytes = (kFwdBlockN / kCG) * kFwdBlockK * 2;
  static constexpr int kStageBytes = kFwdABytes + kBBytes;
  static constexpr int kStages = kCG == 2 ? 5 : 3;  // 160 / 144 KB of operand stages; the rest is epilogue staging
};
constexpr int kFwdMaxChunks = 4;                      // up to 1024 (padded) classes on the tensor-core path
constexpr int kFacCols = 64;                          // granularity of the deferred-normalisation factors
constexpr int kFacPerRow = kFwdMaxChunks * kFwdBlockN / kFacCols;  // 16
constexpr int kFwdStoreBox = 32 * 128;                // 32 rows x 64 bf16 columns, SWIZZLE_128B
constexpr int kFwdStoreBytes = 8 * kFwdStoreBox;      // one staging box per epilogue warp
constexpr int kXchFloats = 16;                        // per-row record the two epilogue groups exchange
constexpr int kFacBytes = 2 * kFwdBlockM * kXchFloats * 4;  // double-buffered per tile
constexpr int kFwdSmemBytes = 160 * 1024 + kFwdStoreBytes + kFacBytes + 1024 /*align*/ + 256 /*barriers*/;
// Warp roles.  The SM's issue arbiter favours higher warp ids, so the two latency-critical single-thread
// roles (TMA producer, MMA issuer) get the highest ids and the ALU-heavy epilogue warps the lowest.
constexpr int kWarpAlloc = 8, kWarpMma = 10, kWarpTma = 11;
constexpr int kFwdThreads = 384;  // 4 control warps + 2 x 4 epilogue warps; <= 170 registers per thread

struct FwdSegs {
  int64_t n0;
  const float* scale_dev[2];
  float scale[2], dcoef[2];  // dcoef = w/n ; the logit-gradient coefficient is dcoef * scale
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

#ifdef UML_FWD_TIMING
__device__ long long g_fwd_dbg[148 * 16];
#define DBG_DECL() long long _acc[4] = {0, 0, 0, 0}; long long _t0 = clock64()
#define DBG_MARK() _t0 = clock64()
#define DBG_ACC(slot) do { long long _t1 = clock64(); _acc[slot] += _t1 - _t0; _t0 = _t1; } while (0)
#define DBG_FLUSH(base) do { for (int _i = 0; _i < 4; ++_i) g_fwd_dbg[blockIdx.x * 16 + (base) + _i] = _acc[_i]; } while (0)
#else
#define DBG_DECL()
#define DBG_MARK()
#define DBG_ACC(slot)
#define DBG_FLUSH(base)
#endif

template <int kCG, bool kPred>
__global__ void __launch_bounds__(kFwdThreads, 1)
    head_fwd_ce_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                          const __grid_constant__ CUtensorMap tmap_g, int64_t n_rows, int dim, int n_classes,
                          const int32_t* __restrict__ labels, FwdSegs segs, __nv_bfloat16* __restrict__ G, int64_t ldg,
                          float* __restrict__ row_loss, int32_t* __restrict__ row_pred,
                          int32_t* __restrict__ row_correct, float* __restrict__ row_dscale,
                          float* __restrict__ tile_part, float* __restrict__ fac) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  using Cfg = FwdCfg<kCG>;
  constexpr int kFwdStages = Cfg::kStages;
  constexpr int kFwdStageBytes = Cfg::kStageBytes;
  unsigned char* store_smem = smem + kFwdStages * kFwdStageBytes;  // 1024-aligned (stage sizes are multiples of 1024)
  float* xch_smem = reinterpret_cast<float*>(store_smem + kFwdStoreBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(xch_smem) + kFacBytes);
  uint64_t* empty_bar = full_bar + kFwdStages;
  uint64_t* tfull_bar = empty_bar + kFwdStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* xch_full = tempty_bar + 2;
  uint64_t* xch_free = xch_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xch_free + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = (kCG == 2) ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  const int num_kb = (dim + kFwdBlockK - 1) / kFwdBlockK;
  const int n_chunks = (n_classes + kFwdBlockN - 1) / kFwdBlockN;
  // work unit = kCG consecutive 128-row tiles (one per CTA of the pair); every CTA of a cluster walks
  // the same sequence of units
  const int64_t n_units = (n_rows + kFwdBlockM * kCG - 1) / (kFwdBlockM * kCG);
  const int64_t unit0 = blockIdx.x / kCG, unit_step = gridDim.x / kCG;
  const bool write_g = G != nullptr;

  if (warp == kWarpTma && lane == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_w);
    if (write_g) tma_prefetch_desc(&tmap_g);
  }
  if (warp == kWarpMma && lane == 0) {
    for (int s = 0; s < kFwdStages; ++s) {
      mbar_init(&full_bar[s], kCG);  // one arrival per producer of the pair; tx bytes are counted on the leader
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 4 * kCG);  // one arrival per epilogue warp of every CTA feeding this MMA
      mbar_init(&xch_full[b], 4);   // one arrive per warp of the early epilogue group
      mbar_init(&xch_free[b], 4);   // one arrive per warp of the finishing group
    }
    fence_barrier_init();
  }
  if (warp == kWarpAlloc) {
    if (kCG == 2) tmem_alloc_cg2(tmem_slot, 512);
    else tmem_alloc(tmem_slot, 512);
  }
  tc_fence_before();
  if (kCG == 2) cluster_sync_all();  // the peer's barriers exist before anything signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kWarpTma) {
    // ------------------------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      uint32_t it = 0;
      DBG_DECL();
      for (int64_t unit = unit0; unit < n_units; unit += unit_step) {
        const int32_t row0 = static_cast<int32_t>((unit * kCG + rank) * kFwdBlockM);
        for (int ch = 0; ch < n_chunks; ++ch) {
          const int32_t wrow0 = ch * kFwdBlockN + static_cast<int32_t>(rank) * (kFwdBlockN / kCG);
          for (int kb = 0; kb < num_kb; ++kb, ++it) {
            const uint32_t s = it % kFwdStages, ph = (it / kFwdStages) & 1;
            DBG_MARK();
            mbar_wait(&empty_bar[s], ph ^ 1);
            DBG_ACC(0);
            unsigned char* a = smem + s * kFwdStageBytes;
#ifdef UML_EXP_STAGGER
            const int kbs = (kb + static_cast<int>(blockIdx.x / kCG) * 5) % num_kb;  // K order is free: spread L2 hot lines
#else
            const int kbs = kb;
#endif
            if (kCG == 1) {
              mbar_arrive_expect_tx(&full_bar[s], kFwdStageBytes);
              tma_load_2d(a, &tmap_x, &full_bar[s], kbs * kFwdBlockK, row0);
              tma_load_2d(a + kFwdABytes, &tmap_w, &full_bar[s], kbs * kFwdBlockK, wrow0);
            } else {
              const uint32_t lead_bar = mapa_cta(smem_u32(&full_bar[s]), 0);
              if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * kFwdStageBytes);
              tma_load_2d_cg2(a, &tmap_x, lead_bar, kbs * kFwdBlockK, row0);
              tma_load_2d_cg2(a + kFwdABytes, &tmap_w, lead_bar, kbs * kFwdBlockK, wrow0);
              if (!leader) mbar_arrive_remote(lead_bar);
            }
            DBG_ACC(1);
          }
        }
      }
      DBG_FLUSH(0);
    }
    __syncwarp();
  } else if (warp == kWarpMma) {
    // ------------------------------------------------ MMA issuer --------------------------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc_bf16(kFwdBlockM * kCG, kFwdBlockN, 0, 0);
      uint32_t it = 0, acc_it = 0;
      DBG_DECL();
      for (int64_t unit = unit0; unit < n_units; unit += unit_step) {
        for (int ch = 0; ch < n_chunks; ++ch, ++acc_it) {
          const uint32_t b = acc_it & 1, aph = (acc_it >> 1) & 1;
          DBG_MARK();
          mbar_wait(&tempty_bar[b], aph ^ 1);
          DBG_ACC(0);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + b * kFwdBlockN;
          for (int kb = 0; kb < num_kb; ++kb, ++it) {
            const uint32_t s = it % kFwdStages, ph = (it / kFwdStages) & 1;
            mbar_wait(&full_bar[s], ph);
            DBG_ACC(1);
            tc_fence_after();
            const uint32_t a_addr = smem_u32(smem + s * kFwdStageBytes);
            const uint32_t b_addr = a_addr + kFwdABytes;
#pragma unroll
            for (int k = 0; k < kFwdBlockK / 16; ++k) {
              // K-major, 128B swizzle: 8-row groups are 1024 B apart; a K step of 16 bf16 = 32 B
              const uint64_t da = make_smem_desc(a_addr + k * 32, 16, 1024, kLayoutSw128);
              const uint64_t db = make_smem_desc(b_addr + k * 32, 16, 1024, kLayoutSw128);
              if (kCG == 2) umma_bf16_cg2(d_tmem, da, db, idesc, (kb | k) != 0);
              else umma_bf16(d_tmem, da, db, idesc, (kb | k) != 0);
            }
            // frees the smem stage (in both CTAs of a pair) once these MMAs have read it
            if (kCG == 2) umma_commit_cg2(&empty_bar[s]);
            else umma_commit(&empty_bar[s]);
            DBG_ACC(2);
          }
          if (kCG == 2) umma_commit_cg2(&tfull_bar[b]);  // accumulator chunk complete, both CTAs' epilogues wake
          else umma_commit(&tfull_bar[b]);
        }
      }
      DBG_FLUSH(4);
    }
    __syncwarp();
  } else if (warp < 8) {
    // ------------------------------------------------ epilogue ----------------------------------
    // Two groups of four warps; group g owns the chunks with (chunk & 1) == g of every tile, so each group
    // has two MMA chunk-times for one chunk of epilogue work (a single group measured ~9.3k cycles per chunk
    // against ~6.1k of MMA - the epilogue, not the tensor pipe, set the pace).  Within a group: one thread per
    // row (TMEM lane).  ONE sweep per chunk, 64 columns at a time: block max, online-softmax rescale of the
    // running sums, exponentials relative to the running max, bf16 staging + TMA store.  The running max each
    // 64-column group was written against is remembered; when the tile is done the group that finishes last
    // merges both groups' row statistics (through shared memory) and publishes the per-row factors
    // exp(m_group - m_final) / sum * coef that g_fixup_kernel applies.
    const int grp = warp >> 2;         // 0: even chunks, 1: odd chunks
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int fin_grp = (n_chunks - 1) & 1;          // the group that processes a tile's last chunk
    const bool have_partner = n_chunks >= 2;
    constexpr float kLog2e = 1.4426950408889634f;
    constexpr int kGroupsPerChunk = kFwdBlockN / kFacCols;  // 4
    unsigned char* sbuf = store_smem + (grp * 4 + q) * kFwdStoreBox;
    unsigned char* srow = sbuf + lane * 128;
    uint32_t tile_it = 0;
    const uint32_t tempty_remote0 = kCG == 2 ? mapa_cta(smem_u32(&tempty_bar[0]), 0) : 0u;
    DBG_DECL();
    for (int64_t unit = unit0; unit < n_units; unit += unit_step, ++tile_it) {
      const int64_t tile = unit * kCG + rank;  // this CTA's 128-row tile
      const int rloc = q * 32 + lane;
      const int64_t row = tile * kFwdBlockM + rloc;
      const bool valid = row < n_rows;
      const bool sg = valid && row >= segs.n0;
      const float* sdev = sg ? segs.scale_dev[1] : segs.scale_dev[0];
      const float scale = sdev ? __ldg(sdev) : (sg ? segs.scale[1] : segs.scale[0]);
      const float dcoef = sg ? segs.dcoef[1] : segs.dcoef[0];
      const float gcoef = dcoef * scale;
      const float sl2 = scale * kLog2e;
      const int label = valid ? labels[row] : -1;
      float run_max = -INFINITY, max_before = -INFINITY, lab_logit = -INFINITY, lab_raw = 0.f;
      float run_sum = 0.f, run_pr = 0.f;
      int arg = 0x7fffffff;
      float group_max[kFacPerRow / 2];  // this group's 64-column groups: index (ch >> 1) * 4 + g

      for (int ch = grp; ch < n_chunks; ch += 2) {
        const uint32_t acc_it = tile_it * n_chunks + ch;
        const uint32_t b = acc_it & 1, aph = (acc_it >> 1) & 1;
        DBG_MARK();
        mbar_wait(&tfull_bar[b], aph);
        DBG_ACC(0);
        tc_fence_after();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + b * kFwdBlockN;
        const int col0 = ch * kFwdBlockN;
        const bool tail = col0 + kFwdBlockN > n_classes;  // chunk with padded class columns
        // The whole chunk body is instantiated twice - with and without the padded-column masking - so that
        // the common (unmasked) path carries no per-element compares/selects.
        auto run_chunk = [&](auto tail_tag) {
          constexpr bool kTail = decltype(tail_tag)::value;
          // block max with four interleaved chains + label bookkeeping.  The hit flag needs no argmax index:
          //   argmax == label  <=>  logit[label] == row max  and  logit[label] > max over the columns before it
          // (torch.argmax returns the FIRST maximal index); the predicted class is tracked only for kPred.
          auto block_max = [&](const uint32_t (&v)[32], int c0, float seen_max) -> float {
            float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
  #pragma unroll
            for (int i = 0; i < 32; i += 4) {
              float x0 = __uint_as_float(v[i]) * scale, x1 = __uint_as_float(v[i + 1]) * scale;
              float x2 = __uint_as_float(v[i + 2]) * scale, x3 = __uint_as_float(v[i + 3]) * scale;
              if (kTail) {
                if (c0 + i >= n_classes) x0 = -INFINITY;
                if (c0 + i + 1 >= n_classes) x1 = -INFINITY;
                if (c0 + i + 2 >= n_classes) x2 = -INFINITY;
                if (c0 + i + 3 >= n_classes) x3 = -INFINITY;
              }
              m0 = fmaxf(m0, x0); m1 = fmaxf(m1, x1); m2 = fmaxf(m2, x2); m3 = fmaxf(m3, x3);
            }
            const float bm = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
            const int d = label - c0;  // position of the label inside this block (if 0 <= d < 32)
            if (d >= 32) {
              max_before = fmaxf(max_before, bm);  // the whole block precedes the label column
            } else if (d >= 0) {
              float b0 = -INFINITY, b1 = -INFINITY;
  #pragma unroll
              for (int i = 0; i < 32; i += 2) {
                const float r0 = __uint_as_float(v[i]), r1 = __uint_as_float(v[i + 1]);
                b0 = fmaxf(b0, i < d ? r0 * scale : -INFINITY);
                b1 = fmaxf(b1, i + 1 < d ? r1 * scale : -INFINITY);
                if (i == d) lab_raw = r0;
                if (i + 1 == d) lab_raw = r1;
              }
              max_before = fmaxf(max_before, fmaxf(b0, b1));
              lab_logit = lab_raw * scale;
            }
            if (kPred && bm > seen_max) {  // first column holding a new maximum (columns are visited in order)
  #pragma unroll
              for (int i = 31; i >= 0; --i)
                if (__uint_as_float(v[i]) * scale == bm && (!kTail || c0 + i < n_classes)) arg = c0 + i;
            }
            return bm;
          };
          // exponentials relative to the running max, partial sums on short chains, bf16 staging of 32 columns
          auto block_exp = [&](const uint32_t (&v)[32], int c0, int half, float mneg) {
            float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
  #pragma unroll
            for (int j = 0; j < 4; ++j) {  // 8 columns -> one 16-byte chunk of the staged row
              uint32_t w[4];
  #pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int i = 8 * j + 2 * e;
                const float r0 = __uint_as_float(v[i]), r1 = __uint_as_float(v[i + 1]);
                float p0 = fast_exp2(fmaf(r0, sl2, mneg));
                float p1 = fast_exp2(fmaf(r1, sl2, mneg));
                if (kTail) {
                  if (c0 + i >= n_classes) p0 = 0.f;
                  if (c0 + i + 1 >= n_classes) p1 = 0.f;
                }
                if (e & 1) { s2 += p0; s3 += p1; q2 = fmaf(p0, r0, q2); q3 = fmaf(p1, r1, q3); }
                else       { s0 += p0; s1 += p1; q0 = fmaf(p0, r0, q0); q1 = fmaf(p1, r1, q1); }
                __nv_bfloat162 h = __floats2bfloat162_rn(p0, p1);
                w[e] = *reinterpret_cast<uint32_t*>(&h);
              }
              if (write_g) {
                // 16-byte chunk c of row r sits at chunk c ^ (r & 7) (TMA SWIZZLE_128B)
                const int chunk = (half * 4 + j) ^ (lane & 7);
                *reinterpret_cast<uint4*>(srow + chunk * 16) = make_uint4(w[0], w[1], w[2], w[3]);
              }
            }
            run_sum += (s0 + s1) + (s2 + s3);
            run_pr += (q0 + q1) + (q2 + q3);
          };

  #pragma unroll 1
          for (int g = 0; g < kGroupsPerChunk; ++g) {
            const int c0 = col0 + g * kFacCols;
            uint32_t va[32], vb[32];
            tmem_ld32(taddr + g * kFacCols, va);
            tmem_ld32(taddr + g * kFacCols + 32, vb);
            tmem_ld_wait();
            const float bma = block_max(va, c0, run_max);
            const float bm = fmaxf(bma, block_max(vb, c0 + 32, fmaxf(run_max, bma)));
            const float new_max = fmaxf(run_max, bm);
            const float resc = fast_exp2((run_max - new_max) * kLog2e);  // exp2(-inf) = 0 on the first group
            run_sum *= resc;
            run_pr *= resc;
            run_max = new_max;
            group_max[(ch >> 1) * kGroupsPerChunk + g] = new_max;
            const float mneg = -new_max * kLog2e;
            if (write_g) {
              if (lane == 0) bulk_wait_read<0>();  // the previous TMA store has finished reading the staging box
              __syncwarp();
            }
            block_exp(va, c0, 0, mneg);
            block_exp(vb, c0 + 32, 1, mneg);
            if (write_g) {
              fence_proxy_async();
              __syncwarp();
              if (lane == 0 && c0 < ldg) {  // the warp's 32 x 64 tile leaves as ONE coalesced TMA store
                tma_store_2d(&tmap_g, sbuf, c0, static_cast<int32_t>(tile * kFwdBlockM + q * 32));
                bulk_commit();
              }
            }
          }
        };
        if (tail) run_chunk(std::true_type{});
        else run_chunk(std::false_type{});
        DBG_ACC(1);
        // accumulator buffer b may be overwritten by the (leader's) MMA warp now
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCG == 2 && !leader) mbar_arrive_remote(tempty_remote0 + b * 8);
          else mbar_arrive(&tempty_bar[b]);
        }
      }
      DBG_MARK();

      // ---- tile end: merge the two groups' row statistics ---------------------------------------------
      // record layout (kXchFloats per row): m, s, pr, max_before, lab_logit, lab_raw, arg, pad, gm[0..7]
      const uint32_t xb = tile_it & 1, xph = (tile_it >> 1) & 1;
      float* rec = xch_smem + (xb * kFwdBlockM + rloc) * kXchFloats;
      if (grp != fin_grp) {
        if (!have_partner) continue;  // a single chunk per tile: this group has no work at all
        // early group: publish and move on to the next tile
        mbar_wait(&xch_free[xb], xph ^ 1);
        rec[0] = run_max; rec[1] = run_sum; rec[2] = run_pr; rec[3] = max_before;
        rec[4] = lab_logit; rec[5] = lab_raw; rec[6] = __int_as_float(arg);
#pragma unroll
        for (int k = 0; k < kFacPerRow / 2; ++k) rec[8 + k] = group_max[k];
        __syncwarp();
        if (lane == 0) mbar_arrive(&xch_full[xb]);
      } else {
        float o_max = -INFINITY, o_sum = 0.f, o_pr = 0.f, o_before = -INFINITY, o_lab = -INFINITY, o_raw = 0.f;
        int o_arg = 0x7fffffff;
        float o_gm[kFacPerRow / 2];
#pragma unroll
        for (int k = 0; k < kFacPerRow / 2; ++k) o_gm[k] = -INFINITY;
        if (have_partner) {
          mbar_wait(&xch_full[xb], xph);
          o_max = rec[0]; o_sum = rec[1]; o_pr = rec[2]; o_before = rec[3];
          o_lab = rec[4]; o_raw = rec[5]; o_arg = __float_as_int(rec[6]);
#pragma unroll
          for (int k = 0; k < kFacPerRow / 2; ++k) o_gm[k] = rec[8 + k];
          __syncwarp();
          if (lane == 0) mbar_arrive(&xch_free[xb]);
        }
        const float M = fmaxf(run_max, o_max);
        const float e_me = fast_exp2((run_max - M) * kLog2e), e_ot = fast_exp2((o_max - M) * kLog2e);
        const float S = run_sum * e_me + o_sum * e_ot;
        const float PR = run_pr * e_me + o_pr * e_ot;
        const float before = fmaxf(max_before, o_before);
        const bool lab_mine = lab_logit > -INFINITY;  // exactly one group saw the label column
        const float lab = lab_mine ? lab_logit : o_lab;
        const float lraw = lab_mine ? lab_raw : o_raw;
        if (kPred) {  // larger maximum wins; on equal maxima the lower column index (torch.argmax)
          if (o_max > run_max || (o_max == run_max && o_arg < arg)) arg = o_arg;
        }
        const float inv_sum = 1.f / S;
        const float loss = valid ? logf(S) - (lab - M) : 0.f;
        const float dsc = valid ? (PR * inv_sum - lraw) * dcoef : 0.f;
        const int hit = (valid && lab == M && lab > before) ? 1 : 0;
        if (valid) {
          if (row_loss) row_loss[row] = loss;
          if (kPred && row_pred) row_pred[row] = arg;
          if (row_correct) row_correct[row] = hit;
          if (row_dscale) row_dscale[row] = dsc;
          if (write_g) {
            // factors of the deferred normalisation, one per 64 columns, applied by g_fixup_kernel:
            //   G = coef * (exp(x - m_group) * exp(m_group - M) / S - onehot)
            float* f = fac + row * kFacPerRow;
            const float tc = inv_sum * gcoef;
#pragma unroll
            for (int k = 0; k < kFacPerRow; ++k) {
              const int ch = k / kGroupsPerChunk, g = k % kGroupsPerChunk;
              if (ch < n_chunks) {
                const float gm = ((ch & 1) == grp) ? group_max[(ch >> 1) * kGroupsPerChunk + g]
                                                   : o_gm[(ch >> 1) * kGroupsPerChunk + g];
                f[k] = fast_exp2((gm - M) * kLog2e) * tc;
              }
            }
          }
        }
        if (tile_part) {
          // deterministic per-(tile, warp, run) partial sums; the stats kernel adds them in a fixed order
#pragma unroll
          for (int s2 = 0; s2 < 2; ++s2) {
            const bool mine = valid && (static_cast<int>(sg) == s2);
            const float a = warp_sum(mine ? loss : 0.f), d = warp_sum(mine ? dsc : 0.f);
            const int h = warp_sum_i(mine ? hit : 0), cnt = warp_sum_i(mine ? 1 : 0);
            if (lane == 0) {
              float* o = tile_part + (tile * 8 + q * 2 + s2) * 4;
              o[0] = a; o[1] = d; o[2] = static_cast<float>(h); o[3] = static_cast<float>(cnt);
            }
          }
        }
      }
      DBG_ACC(2);
    }
    if (write_g && lane == 0) bulk_wait<0>();  // this warp's TMA stores have landed before the kernel ends
#ifdef UML_FWD_TIMING
    if (warp == 0 && lane == 0) DBG_FLUSH(8);
    if (warp == 4 && lane == 0) DBG_FLUSH(12);
#endif
  }

  tc_fence_before();
  if (kCG == 2) cluster_sync_all();  // the leader's MMAs read the peer's shared memory until the last commit
  else __syncthreads();
  if (warp == kWarpAlloc) {
    if (kCG == 2) tmem_dealloc_cg2(tmem_base, 512);
    else tmem_dealloc(tmem_base, 512);
  }
}

// per-run statistics from the per-tile partials, summed in a fixed order (deterministic); one CTA per run
__device__ void tile_stats_block(const float* __restrict__ tile_part, int64_t n_tiles, int s, uml_seg_stats* __restrict__ out) {
  __shared__ float sh[4][32];
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  const int64_t n = n_tiles * 4;  // (tile, warp) partials of this run
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const float* p = tile_part + (i * 2 + s) * 4;
#pragma unroll
    for (int k = 0; k < 4; ++k) acc[k] += p[k];
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float v = warp_sum(acc[k]);
    if ((threadIdx.x & 31) == 0) sh[k][threadIdx.x >> 5] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot[4] = {0.f, 0.f, 0.f, 0.f};
    for (int k = 0; k < 4; ++k)
      for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) tot[k] += sh[k][w];
    out[s].loss_mean = tot[3] > 0.f ? tot[0] / tot[3] : 0.f;
    out[s].dscale = tot[1];
    out[s].correct = static_cast<int32_t>(tot[2] + 0.5f);
    out[s].n = static_cast<int32_t>(tot[3] + 0.5f);
  }
}

// Second half of the deferred softmax normalisation: G[b,c] = G[b,c] * fac[b][c / 64] - [c == y_b] * coef_b.
// One warp per row, 16-byte vectors, all loads of a row in flight at once; fully coalesced.  The first `stat_blocks`
// CTAs of the grid reduce the forward kernel's per-tile partials into the per-run statistics instead (what
// used to be a launch of its own).
__global__ void __launch_bounds__(256)
    g_fixup_kernel(__nv_bfloat16* __restrict__ G, int64_t ldg, int64_t n_rows, const int32_t* __restrict__ labels,
                   const float* __restrict__ fac, FwdSegs segs, const float* __restrict__ tile_part, int64_t n_tiles,
                   int stat_blocks, uml_seg_stats* __restrict__ stats) {
  if (static_cast<int>(blockIdx.x) < stat_blocks) {
    tile_stats_block(tile_part, n_tiles, static_cast<int>(blockIdx.x), stats);
    return;
  }
  const int64_t row = static_cast<int64_t>(static_cast<int>(blockIdx.x) - stat_blocks) * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n_rows) return;
  const int label = labels[row];
  const bool sg = row >= segs.n0;
  const float* sdev = sg ? segs.scale_dev[1] : segs.scale_dev[0];
  const float scale = sdev ? __ldg(sdev) : (sg ? segs.scale[1] : segs.scale[0]);
  const float gcoef = (sg ? segs.dcoef[1] : segs.dcoef[0]) * scale;
  const float* f = fac + row * kFacPerRow;
  __nv_bfloat16* g = G + row * ldg;
  uint4 v[kFwdMaxChunks];
  float fj[kFwdMaxChunks];
#pragma unroll
  for (int j = 0; j < kFwdMaxChunks; ++j) {
    const int c = j * 256 + lane * 8;
    if (c < ldg) {
      v[j] = *reinterpret_cast<const uint4*>(g + c);
      fj[j] = f[c / kFacCols];
    }
  }
#pragma unroll
  for (int j = 0; j < kFwdMaxChunks; ++j) {
    const int c = j * 256 + lane * 8;
    if (c < ldg) {
      uint32_t w[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float2 p = __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&w[i]));
        p.x *= fj[j];
        p.y *= fj[j];
        if (c + 2 * i == label) p.x -= gcoef;
        if (c + 2 * i + 1 == label) p.y -= gcoef;
        __nv_bfloat162 h = __floats2bfloat162_rn(p.x, p.y);
        w[i] = *reinterpret_cast<uint32_t*>(&h);
      }
      *reinterpret_cast<uint4*>(g + c) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

static int fwd_cta_group(int64_t n_rows) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("UML_TC_CTA_GROUP");
    forced = e ? atoi(e) : 0;
  }
  if (forced == 1 || forced == 2) return forced;
  return n_rows > kFwdBlockM ? 2 : 1;
}

// stand-alone version for forward passes that write no G (evaluation) and therefore launch no fix-up kernel
__global__ void __launch_bounds__(1024)
    tile_stats_kernel(const float* __restrict__ tile_part, int64_t n_tiles, int nseg, uml_seg_stats* __restrict__ out) {
  tile_stats_block(tile_part, n_tiles, blockIdx.x, out);
  (void)nseg;
}

}  // namespace uml

// Launches the forward kernel and (training mode) the fix-up; `ev_after_fwd` (optional cudaEvent_t) is recorded
// between the two so that a caller can time the tensor-core kernel alone (bench.py's roofline line).
int uml_head_fwd_ce_bf16_ev(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W, int32_t n_classes,
                            const int32_t* labels, const uml_tc_segments* segs, uint16_t* G, int64_t ldg, float* row_loss,
                            int32_t* row_pred, int32_t* row_correct, float* row_dscale, float* tile_ws, uml_seg_stats* stats,
                            void* ev_after_fwd, void* stream, void* ev_after_fwd2 = nullptr);
// tc_fwd2.cu: the exchange kernel (class chunks of a row tile on different CTA pairs, G final after one pass)
bool uml_fwd_x_eligible(int64_t n_rows, int32_t n_classes);
int uml_head_fwd_ce_x_bf16(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W, int32_t n_classes,
                           const int32_t* labels, const uml_tc_segments* segs, uint16_t* G, int64_t ldg, float* row_loss,
                           int32_t* row_pred, int32_t* row_correct, float* row_dscale, float* tile_ws, uml_seg_stats* stats,
                           void* stream);
int uml_fwd_x_reduce_stats(float* tile_ws, int64_t n_rows, int32_t nseg, uml_seg_stats* stats, void* stream);

extern "C" {

#ifdef UML_FWD_TIMING
int uml_debug_fwd_timing(long long* host_out /* [148*16] */, int reset) {
  if (reset) {
    static long long zeros[148 * 16];
    return cudaMemcpyToSymbol(uml::g_fwd_dbg, zeros, sizeof(zeros)) != cudaSuccess;
  }
  return cudaMemcpyFromSymbol(host_out, uml::g_fwd_dbg, sizeof(long long) * 148 * 16) != cudaSuccess;
}
#endif

int uml_head_fwd_ce_bf16(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W, int32_t n_classes,
                         const int32_t* labels, const uml_tc_segments* segs, uint16_t* G, int64_t ldg,
                         float* row_loss, int32_t* row_pred, int32_t* row_correct, float* row_dscale,
                         float* tile_ws, uml_seg_stats* stats, void* stream) {
  return uml_head_fwd_ce_bf16_ev(X, n_rows, dim, W, n_classes, labels, segs, G, ldg, row_loss, row_pred, row_correct,
                                 row_dscale, tile_ws, stats, nullptr, stream);
}

}  // extern "C"

int uml_head_fwd_ce_bf16_ev(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W, int32_t n_classes,
                            const int32_t* labels, const uml_tc_segments* segs, uint16_t* G, int64_t ldg, float* row_loss,
                            int32_t* row_pred, int32_t* row_correct, float* row_dscale, float* tile_ws, uml_seg_stats* stats,
                            void* ev_after_fwd, void* stream, void* ev_after_fwd2) {
  using namespace uml;
  UML_REQUIRE(X && W && labels && segs && n_rows >= 0 && dim > 0 && n_classes > 0, "head_fwd_ce_bf16: bad arguments");
  UML_REQUIRE(dim % 8 == 0, "head_fwd_ce_bf16: dim (%d) must be a multiple of 8 (16-byte bf16 rows for TMA)", dim);
  UML_REQUIRE(n_classes <= kFwdMaxChunks * kFwdBlockN, "head_fwd_ce_bf16: at most %d classes", kFwdMaxChunks * kFwdBlockN);
  UML_REQUIRE(!G || (ldg % 64 == 0 && ldg >= n_classes && ldg <= kFwdMaxChunks * kFwdBlockN),
              "head_fwd_ce_bf16: ldg must be a multiple of 64 and >= n_classes");
  UML_REQUIRE(segs->nseg >= 1 && segs->nseg <= UML_MAX_SEGMENTS, "head_fwd_ce_bf16: 1..2 segments");
  if (n_rows == 0) return 0;
  if (tile_ws && uml_fwd_x_eligible(n_rows, n_classes)) {
    // default for anything larger than one 128-row tile: one kernel, G final, no fix-up launch
    int rc = uml_head_fwd_ce_x_bf16(X, n_rows, dim, W, n_classes, labels, segs, G, ldg, row_loss, row_pred, row_correct,
                                    row_dscale, tile_ws, stats, stream);
    if (rc) return rc;
    if (ev_after_fwd) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(ev_after_fwd), uml::as_stream(stream)));
    if (ev_after_fwd2) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(ev_after_fwd2), uml::as_stream(stream)));
    return 0;
  }
  const int64_t n0 = segs->seg_rows[0], n1 = segs->nseg > 1 ? segs->seg_rows[1] : 0;
  UML_REQUIRE(n0 + n1 == n_rows, "head_fwd_ce_bf16: segment rows (%lld+%lld) != n_rows (%lld)", (long long)n0,
              (long long)n1, (long long)n_rows);
  CUtensorMap tx, tw, tg;
  if (make_tmap_2d(&tx, X, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dim, n_rows, static_cast<uint64_t>(dim) * 2, kFwdBlockK,
                   kFwdBlockM, CU_TENSOR_MAP_SWIZZLE_128B))
    return 1;
  const int cg = fwd_cta_group(n_rows);
  if (make_tmap_2d(&tw, W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dim, n_classes, static_cast<uint64_t>(dim) * 2,
                   kFwdBlockK, kFwdBlockN / cg, CU_TENSOR_MAP_SWIZZLE_128B))
    return 1;
  memset(&tg, 0, sizeof(tg));
  if (G) {
    if (make_tmap_2d(&tg, G, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, static_cast<uint64_t>(ldg), n_rows,
                     static_cast<uint64_t>(ldg) * 2, 64, 32, CU_TENSOR_MAP_SWIZZLE_128B))
      return 1;
  }
  FwdSegs fs;
  fs.n0 = segs->nseg > 1 ? n0 : INT64_MAX;
  for (int i = 0; i < 2; ++i) {
    const int j = i < segs->nseg ? i : 0;
    const double n = static_cast<double>(segs->seg_rows[j] > 0 ? segs->seg_rows[j] : 1);
    fs.scale[i] = segs->scale[j];
    fs.scale_dev[i] = segs->scale_dev[j];
    fs.dcoef[i] = static_cast<float>(static_cast<double>(segs->loss_weight[j]) / n);
  }
  void (*kern)(CUtensorMap, CUtensorMap, CUtensorMap, int64_t, int, int, const int32_t*, FwdSegs, __nv_bfloat16*, int64_t,
               float*, int32_t*, int32_t*, float*, float*, float*) =
      row_pred ? (cg == 2 ? head_fwd_ce_tc_kernel<2, true> : head_fwd_ce_tc_kernel<1, true>)
               : (cg == 2 ? head_fwd_ce_tc_kernel<2, false> : head_fwd_ce_tc_kernel<1, false>);
  static bool attr_set[4] = {false, false, false, false};
  const int slot = (row_pred ? 2 : 0) + (cg == 2 ? 1 : 0);
  if (!attr_set[slot]) {
    UML_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kFwdSmemBytes));
    attr_set[slot] = true;
  }
  const int64_t units = (n_rows + kFwdBlockM * cg - 1) / (kFwdBlockM * cg);
  const int64_t max_clusters = sm_count() / cg;
  UML_REQUIRE(!G || tile_ws, "head_fwd_ce_bf16: tile_ws is required when G is written");
  // workspace layout: per-tile partial sums, then the per-row normalisation factors
  float* fac = tile_ws ? tile_ws + units * cg * 32 : nullptr;
  const dim3 grid(static_cast<unsigned>((units < max_clusters ? units : max_clusters) * cg));
  UML_CUDA(launch_kernel(kern, grid, dim3(kFwdThreads), kFwdSmemBytes, as_stream(stream), cg, tx, tw, tg, n_rows,
                         static_cast<int>(dim), static_cast<int>(n_classes), labels, fs, reinterpret_cast<__nv_bfloat16*>(G), ldg,
                         row_loss, row_pred, row_correct, row_dscale, tile_ws, fac));
  if (ev_after_fwd) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(ev_after_fwd), as_stream(stream)));
  if (ev_after_fwd2) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(ev_after_fwd2), as_stream(stream)));
  if (G) {
    const int row_blocks = static_cast<int>((n_rows + 7) / 8);
    const int stat_blocks = stats ? segs->nseg : 0;
    UML_CUDA(launch_kernel(g_fixup_kernel, dim3(static_cast<unsigned>(row_blocks + stat_blocks)), dim3(256), 0,
                           as_stream(stream), 1, reinterpret_cast<__nv_bfloat16*>(G), ldg, n_rows, labels,
                           static_cast<const float*>(fac), fs, static_cast<const float*>(tile_ws), units * cg, stat_blocks,
                           stats));
  }
  return 0;
}

extern "C" {

int uml_reduce_tile_stats(const float* tile_ws, int64_t n_rows, int32_t nseg, uml_seg_stats* stats, void* stream) {
  using namespace uml;
  UML_REQUIRE(tile_ws && stats && nseg >= 1 && nseg <= UML_MAX_SEGMENTS && n_rows >= 0, "reduce_tile_stats: bad arguments");
  if (uml_fwd_x_eligible(n_rows, 1)) return uml_fwd_x_reduce_stats(const_cast<float*>(tile_ws), n_rows, nseg, stats, stream);
  const int cg = fwd_cta_group(n_rows);
  const int64_t tiles = ((n_rows + kFwdBlockM * cg - 1) / (kFwdBlockM * cg)) * cg;  // tiles the forward kernel wrote
  UML_CUDA(launch_kernel(tile_stats_kernel, dim3(nseg), dim3(1024), 0, as_stream(stream), 1, tile_ws, tiles,
                         static_cast<int>(nseg), stats));
  return 0;
}

}  // extern "C"
