// K2+K3 on the tensor cores, second generation: head forward, logit scale, softmax cross-entropy and the FINAL logit
// gradient G in ONE kernel and ONE pass over G (reference: engine/models/head.py:80-82,133-135 +
// finetune.py:186-188 + the autograd of F.cross_entropy).
//
//   logits[b,c] = scale_b * sum_d X[b,d] W[c,d]         bf16 x bf16 -> fp32 in TMEM
//   G[b,c]      = w_b * scale_b / n_b * (softmax(logits)[b,c] - [c == y_b])     written once, as bf16
//
// tc_fwd.cu walks the (up to four) 256-class chunks of a row tile one after the other inside one CTA pair; a row's
// final max / sum is then only known after its first chunks have left the SM, which cost a second pass over G
// (g_fixup_kernel: 155 MB of traffic + a launch gap, a quarter of the step).
// Here the class chunks of a row tile are computed AT THE SAME TIME by different CTA pairs:
//
//   * CTA pair (cluster of 2, cta_group::2, M = 256) p owns class chunk p % n_chunks for good - and walks the 256-row
//     units of group p / n_chunks.  X tile and the pair's half of the W chunk come by TMA (6 stages, SWIZZLE_128B),
//     accumulators live in TMEM, double buffered (2 x 256 columns): the MMA of unit i+1 overlaps the epilogue of unit i.
//   * epilogue, 16 warps, one thread per (row, 64-column quarter): ONE sweep over the accumulator, 16 columns at a time
//     with the next tcgen05.ld in flight: running max (in the raw-logit domain, so that the maximal element's
//     exponential is exactly 1 and the cross entropy can never come out negative), exp(l - m_running) kept as 32
//     registers of bf16 pairs.  The TMEM buffer is handed back to the MMA warp right after this sweep.  Nothing of
//     the epilogue goes through shared memory except one 32-byte record per thread: the operand stages' TMA
//     writes and the tensor core's operand reads already use most of the SM's shared-memory bandwidth.
//   * the column slices of a row meet in slice 0's thread through shared memory (the other slices drop a record, arrive
//     on an mbarrier and go on: nobody but slice 0 ever waits), the pairs of a group exchange one 16-byte record per row -
//     {max, sum, sum p*raw, argmax} - through L2 (value + launch-epoch word pairs: no memset, no fence, no cluster wider
//     than the pair, every SM usable),
//   * then every thread rescales ITS OWN columns in registers by  exp(m_group - M) * coef / S  (two bf16x2 FMAs per
//     pair with the factor split hi + lo, so the product carries fp32-level accuracy) and writes them with 256-bit
//     stores; the one-hot column is patched by a 2-byte store of the same thread.  G is written once and is final.
//   * the pair that owns a row's label column computes loss / hit / d(scale) for that row; each thread keeps the sums of
//     its rows, one warp reduction per CTA at the end puts per-(CTA, row quarter, run) partial sums into tile_part, and
//     the next kernel of the step (the dW GEMM's idle warp) or uml_reduce_tile_stats adds them in a fixed order.
// All CTAs of the grid (<= one per SM) are co-resident, which the flag exchange relies on; a watchdog turns a
// missing peer into an error flag (uml_fwd_x_failed) instead of a hang.
#include <type_traits>

#include "common.cuh"

namespace uml {

#ifndef UML_X_TMAST
#define UML_X_TMAST 1
#endif
// G leaves through shared memory and TMA stores (32 rows x 64 B boxes, two per epilogue warp) instead of 32-byte register
// stores: a warp's direct store instruction touches 32 rows = 32 separate sectors, and those 4.7 M small write requests
// per launch cost the kernel 20 us of 120 (measured with the stores switched off); the staging boxes take one TMA stage
constexpr bool kXTmaStore = UML_X_TMAST != 0;
#ifndef UML_X_STAGES
#define UML_X_STAGES (UML_X_TMAST ? 5 : 6)
#endif
constexpr int kXStages = UML_X_STAGES;
constexpr int kXABytes = 128 * 64 * 2;                 // X tile: 128 rows x 64 k
constexpr int kXBBytes = 128 * 64 * 2;                 // this CTA's half of the W chunk: 128 classes x 64 k
constexpr int kXStageBytes = kXABytes + kXBBytes;
constexpr int kXRecBytes = 32;                         // record the four column quarters of a row exchange
#ifndef UML_X_SLICES
#define UML_X_SLICES 2
#endif
constexpr int kXSlices = UML_X_SLICES;                 // column slices of a chunk, one epilogue thread per (row, slice)
constexpr int kXSliceCols = 256 / kXSlices;
#ifndef UML_X_GC
#define UML_X_GC 32
#endif
constexpr int kXGC = UML_X_GC;                         // columns per group: one tcgen05.ld, one running-max step
#ifndef UML_X_DB
#define UML_X_DB 0
#endif
constexpr bool kXDoubleBuf = UML_X_DB != 0;            // the next group's tcgen05.ld is in flight while this group is worked on
constexpr int kXGW = kXGC / 2;                         // ... and its registers of bf16 pairs
constexpr int kXGroups = kXSliceCols / kXGC;           // groups per thread
constexpr int kXHxSlots = 4;                           // a record is read at most two units after it was written
constexpr int kXHxBytes = kXHxSlots * (kXSlices - 1) * 128 * kXRecBytes;  // [unit & 3][column slice - 1][row]
constexpr int kXEpiWarpsC = 4 * kXSlices;
constexpr int kXSbufWarp = 2 * 2048;                       // per epilogue warp: two boxes of 32 rows x 32 bf16, SWIZZLE_64B
constexpr int kXSbufBytes = kXTmaStore ? kXEpiWarpsC * kXSbufWarp : 0;
constexpr int kXSmemBytes = kXStages * kXStageBytes + kXSbufBytes + kXHxBytes + 1024 /*align*/ + 256 /*barriers*/;
constexpr int kXEpiWarps = 4 * kXSlices;               // warp e: TMEM lane quarter e & 3, column slice e >> 2
constexpr int kXWarpMma = kXEpiWarps, kXWarpTma = kXEpiWarps + 1;  // (the TMA warp also owns the TMEM allocation)
constexpr int kXThreads = (kXEpiWarps + 4) * 32;        // the producer warps form a warpgroup of their own (two of them idle): it
                                                       // hands most of its registers to the epilogue warpgroups (setmaxnreg)
// setmaxnreg moves registers inside the CTA's launch-time budget (threads x launch registers): what the epilogue
// warpgroups gain must not exceed what the producer warpgroup gives up, or the last warpgroup to ask waits for ever.
//   2 slices: 384 threads x 168 -> producers 40 (frees 128 x 128 = 16384), epilogue 232 (takes 256 x 64 = 16384)
//   4 slices: 640 threads x  96 -> producers 24 (frees 128 x  72 =  9216), epilogue 112 (takes 512 x 16 =  8192)
#ifndef UML_X_REGS_P
#define UML_X_REGS_P (kXSlices == 2 ? 40 : 24)
#define UML_X_REGS_E (kXSlices == 2 ? 232 : 112)
#endif
constexpr int kXRegsProducer = UML_X_REGS_P, kXRegsEpilogue = UML_X_REGS_E;
static_assert((kXThreads - 128) * (kXRegsEpilogue - 168) <= 128 * (168 - kXRegsProducer) || kXSlices != 2, "setmaxnreg: the epilogue asks for more than the producers free");
#ifndef UML_X_HALF
#define UML_X_HALF (kXGroups > 2 ? kXGroups - 1 : kXGroups / 2)   // measured: 3 of 4 groups first 68.6 us, 2 of 4 70.4 us
#endif
constexpr int kXHalf = UML_X_HALF;                     // groups of a new unit that are made before the previous unit is finished
constexpr int kXMaxChunks = 4;
// the previous unit's records are asked for after this group of the new unit and looked at after group kXHalf - 1.  Asked
// for after group 0, nine units in ten found a record of a slower pair still stale and paid a second, exposed L2 round trip
// (ncu: the re-request loads ran 0.91 + 0.49 times per unit); a group later the pairs of a row may drift by ~2 us
#ifndef UML_X_REQ_AFTER
#define UML_X_REQ_AFTER 0
#endif
constexpr int kXReqAfter = UML_X_REQ_AFTER;
static_assert(kXHalf >= 1 && kXHalf <= kXGroups && kXReqAfter < kXHalf, "the records must be requested before they are resolved");
static_assert(kXSmemBytes <= 227 * 1024, "exchange forward kernel: shared memory");

struct XSegs {
  int64_t n0;
  const float* scale_dev[2];
  float scale[2], dcoef[2];  // dcoef = w/n ; the logit-gradient coefficient is dcoef * scale
};

struct XWork {
  float* tile_part;      // [(CTA * 4 + row quarter) * 2 + run] x 4 floats: loss sum, d loss / d scale, hits, rows
  uint4* recs;           // [(row * n_chunks + chunk) * 2 + {0, 1}]: {max, epoch, sum, epoch}, {sum p*raw, epoch, argmax, epoch}
  unsigned* ctrl;        // [0] epoch of the last finished launch, [1] finished CTAs, [2] watchdog flag, [3] partial records
};

__device__ __forceinline__ float x_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// value + epoch word pairs: 8-byte units are delivered whole, so a matching epoch vouches for its value (the scheme of
// NCCL's LL protocol); volatile = every poll goes to L2
__device__ __forceinline__ void st_volatile_v4(uint4* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_volatile_v4(const uint4* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
// explicit shared-space accesses (32-bit addresses): the generic-pointer forms compiled to LD.E / ST.E
__device__ __forceinline__ void sts128(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ void sts64(uint32_t a, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t a) {
  uint2 v;
  asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
  return v;
}
// one 32-byte sector of a G row (16 bf16) straight from registers
__device__ __forceinline__ void stg256(void* p, const uint32_t* w) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
               "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
// 32 lanes x 16 columns of fp32: thread i of the warp receives lane (base_lane + i), columns c..c+15
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ldg(uint32_t taddr, uint32_t (&v)[16]) { tmem_ld16(taddr, v); }
__device__ __forceinline__ void tmem_ldg(uint32_t taddr, uint32_t (&v)[32]) { tmem_ld32(taddr, v); }
// makes the registers of a tcgen05.ld "change" after the wait, so that no use can be scheduled above it
template <int N>
__device__ __forceinline__ void pin16(uint32_t (&v)[N]) {
#pragma unroll
  for (int i = 0; i < N; i += 8)
    asm volatile("" : "+r"(v[i]), "+r"(v[i + 1]), "+r"(v[i + 2]), "+r"(v[i + 3]), "+r"(v[i + 4]), "+r"(v[i + 5]),
                      "+r"(v[i + 6]), "+r"(v[i + 7]));
}

// packed fp32 pairs (sm_100): two fused multiply-adds / adds per issue slot
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

#ifdef UML_FWD_TIMING
__device__ long long g_fwdx_dbg[148 * 16];
#define XDBG_DECL() long long _acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; long long _t0 = clock64()
#define XDBG_MARK() _t0 = clock64()
#define XDBG_ACC(slot) do { long long _t1 = clock64(); _acc[slot] += _t1 - _t0; _t0 = _t1; } while (0)
#define XDBG_FLUSH(base, n) do { for (int _i = 0; _i < (n); ++_i) g_fwdx_dbg[blockIdx.x * 16 + (base) + _i] = _acc[_i]; } while (0)
#else
#define XDBG_DECL()
#define XDBG_MARK()
#define XDBG_ACC(slot)
#define XDBG_FLUSH(base, n)
#endif

// v[d] for a run-time d: a switch whose cases cannot be turned into selects
template <int N>
__device__ __forceinline__ float pick_col(const uint32_t (&v)[N], int d) {
  uint32_t r = 0;
#define UML_PICK(i) \
  case i:           \
    asm volatile("mov.b32 %0, %1;" : "=r"(r) : "r"(v[(i) < N ? (i) : 0])); \
    break;
  switch (d) {
    UML_PICK(0) UML_PICK(1) UML_PICK(2) UML_PICK(3) UML_PICK(4) UML_PICK(5) UML_PICK(6) UML_PICK(7)
    UML_PICK(8) UML_PICK(9) UML_PICK(10) UML_PICK(11) UML_PICK(12) UML_PICK(13) UML_PICK(14) UML_PICK(15)
    UML_PICK(16) UML_PICK(17) UML_PICK(18) UML_PICK(19) UML_PICK(20) UML_PICK(21) UML_PICK(22) UML_PICK(23)
    UML_PICK(24) UML_PICK(25) UML_PICK(26) UML_PICK(27) UML_PICK(28) UML_PICK(29) UML_PICK(30) UML_PICK(31)
    default: break;
  }
#undef UML_PICK
  return __uint_as_float(r);
}

template <int B, int E, class F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (B < E) {
    f(std::integral_constant<int, B>());
    static_for<B + 1, E>(f);
  }
}

template <bool kPred, bool kDs>
__global__ void __launch_bounds__(kXThreads, 1)
    head_fwd_ce_x_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_w,
                         const __grid_constant__ CUtensorMap tmap_g,
                         int64_t n_rows, int dim, int n_classes, int n_groups, const int32_t* __restrict__ labels, XSegs segs,
                         uint16_t* __restrict__ G, int64_t ldg, float* __restrict__ row_loss, int32_t* __restrict__ row_pred,
                         int32_t* __restrict__ row_correct, float* __restrict__ row_dscale, XWork wk) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  unsigned char* sbuf = smem + kXStages * kXStageBytes;  // (1024-byte aligned: the stages are 32 KB each)
  unsigned char* hx = sbuf + kXSbufBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(hx + kXHxBytes);
  uint64_t* empty_bar = full_bar + kXStages;
  uint64_t* tfull_bar = empty_bar + kXStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* xbar = tempty_bar + 2;                     // [row quarter]: the other column slices' records of a unit are in place
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(xbar + 4);
  uint32_t* epoch_slot = tmem_slot + 1;
  float* run_scale = reinterpret_cast<float*>(epoch_slot + 1);  // [2]: the runs' logit scales

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int num_kb = (dim + 63) / 64;
  const int n_chunks = (n_classes + 255) / 256;
  const int pair = blockIdx.x >> 1;
  const int chunk = pair % n_chunks, group = pair / n_chunks;
  const int col0 = chunk * 256;
  const int n_valid = n_classes - col0 < 256 ? n_classes - col0 : 256;  // class columns of this chunk
  const int n_mma = ((n_valid + 15) / 16) * 16;                          // N of the pair's MMA
  const int64_t n_units = (n_rows + 255) / 256;
  const bool write_g = G != nullptr;

  if (warp == kXWarpTma && lane == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_w);
    if (kXTmaStore && write_g) tma_prefetch_desc(&tmap_g);
  }
  if (warp == kXWarpMma && lane == 0) {
    for (int s = 0; s < kXStages; ++s) {
      mbar_init(&full_bar[s], 2);  // one arrival per producer of the pair; tx bytes are counted on the leader
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull_bar[b], 1);
      mbar_init(&tempty_bar[b], 2 * kXEpiWarps);  // one arrival per epilogue warp of both CTAs
    }
    for (int qq = 0; qq < 4; ++qq) mbar_init(&xbar[qq], kXSlices - 1);
    fence_barrier_init();
  }
  if (warp == kXWarpTma) tmem_alloc_cg2(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();  // the peer's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x < 2) run_scale[threadIdx.x] = segs.scale_dev[threadIdx.x] ? __ldg(segs.scale_dev[threadIdx.x]) : segs.scale[threadIdx.x];
  if (threadIdx.x == 0) {
    *epoch_slot = *reinterpret_cast<volatile unsigned*>(wk.ctrl) + 1u;
    if (blockIdx.x == 0) wk.ctrl[3] = gridDim.x * 4u;  // partial records per run: one per CTA and row quarter
  }
  __syncthreads();
  const unsigned epoch = *epoch_slot;

  if (warp >= kXEpiWarps) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kXRegsProducer));
  if (warp == kXWarpTma) {
    // ------------------------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      uint32_t it = 0;
      XDBG_DECL();
      const uint32_t lead_bar0 = mapa_cta(smem_u32(&full_bar[0]), 0);
      const int32_t wrow0 = col0 + static_cast<int32_t>(rank) * (n_mma / 2);
      for (int64_t unit = group; unit < n_units; unit += n_groups) {
        const int32_t row0 = static_cast<int32_t>((unit * 2 + rank) * 128);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t s = it % kXStages, ph = (it / kXStages) & 1;
          XDBG_MARK();
          mbar_wait(&empty_bar[s], ph ^ 1);
          XDBG_ACC(0);
          unsigned char* a = smem + s * kXStageBytes;
          const uint32_t lead_bar = lead_bar0 + s * 8;
#ifdef UML_X_HALFLOAD
          if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * kXBBytes);
#else
          if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * kXStageBytes);
          tma_load_2d_cg2(a, &tmap_x, lead_bar, kb * 64, row0);
#endif
          tma_load_2d_cg2(a + kXABytes, &tmap_w, lead_bar, kb * 64, wrow0);
          if (!leader) mbar_arrive_remote(lead_bar);
          XDBG_ACC(1);
        }
      }
      XDBG_FLUSH(12, 2);
    }
    __syncwarp();
  } else if (warp == kXWarpMma) {
    // ------------------------------------------------ MMA issuer --------------------------------
    if (lane == 0 && leader) {
      const uint32_t idesc = make_idesc_bf16(256, static_cast<uint32_t>(n_mma), 0, 0);
      uint32_t it = 0, acc_it = 0;
      XDBG_DECL();
      for (int64_t unit = group; unit < n_units; unit += n_groups, ++acc_it) {
        const uint32_t b = acc_it & 1, aph = (acc_it >> 1) & 1;
        XDBG_MARK();
        mbar_wait(&tempty_bar[b], aph ^ 1);
        XDBG_ACC(0);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + b * 256;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t s = it % kXStages, ph = (it / kXStages) & 1;
          mbar_wait(&full_bar[s], ph);
          XDBG_ACC(1);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + s * kXStageBytes);
          const uint32_t b_addr = a_addr + kXABytes;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // K-major, 128B swizzle: 8-row groups are 1024 B apart; a K step of 16 bf16 = 32 B
            const uint64_t da = make_smem_desc(a_addr + k * 32, 16, 1024, kLayoutSw128);
            const uint64_t db = make_smem_desc(b_addr + k * 32, 16, 1024, kLayoutSw128);
            umma_bf16_cg2(d_tmem, da, db, idesc, (kb | k) != 0);
          }
          umma_commit_cg2(&empty_bar[s]);  // frees the stage in both CTAs once these MMAs have read it
          XDBG_ACC(2);
        }
        umma_commit_cg2(&tfull_bar[b]);  // accumulator complete: both CTAs' epilogues wake
      }
      XDBG_FLUSH(9, 3);
    }
    __syncwarp();
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kXRegsEpilogue));
    // ------------------------------------------------ epilogue ----------------------------------
    // Software-pipelined over the units: iteration i makes the exponentials of unit i (pass 1) and - interleaved with
    // it, 16 columns at a time, so that one set of 32 registers serves both - the final G of unit i-1, whose row
    // statistics the other class chunks published one unit ago: nobody ever waits on the exchange.
    const int q = warp & 3;    // TMEM lane quarter = row quarter of the tile
    const int cq = warp >> 2;  // column slice of the chunk: columns [cq * kXSliceCols, (cq + 1) * kXSliceCols)
    constexpr float kLog2e = 1.4426950408889634f;
    constexpr float kMasked = -1.0e30f;  // padded class column: never the maximum, exponential exactly 0, 0 * it finite
    constexpr bool kSecond = kPred || kDs;
    const int rloc = q * 32 + lane;
    const uint32_t hx_base = smem_u32(hx);
    const uint32_t tempty_remote0 = mapa_cta(smem_u32(&tempty_bar[0]), 0);
    const int live_groups = !write_g ? 0 : static_cast<int>((ldg - col0 - cq * kXSliceCols) / kXGC);  // groups of this slice inside G's row (<= 0: none)
    uint32_t tile_it = 0;
    XDBG_DECL();

    // what a row needs from its run (image rows first, then text rows): hoisted, a row only selects
    struct RowCtx {
      float sl2, sabs, sgn, dcoef, gcoef;
      bool valid, sg;
    };
    // (the two runs' temperatures sit in shared memory: a learnable one is read from the device once per CTA)
    const float scale_a = run_scale[0], scale_b = run_scale[1];
    const bool any_neg = scale_a < 0.f || scale_b < 0.f;  // (a learnable temperature may in principle go negative)
    auto row_ctx = [&](int64_t row) {
      RowCtx c;
      c.valid = row < n_rows;
      c.sg = c.valid && row >= segs.n0;
      const float scale = c.sg ? run_scale[1] : run_scale[0];
      c.dcoef = c.sg ? segs.dcoef[1] : segs.dcoef[0];
      c.gcoef = c.dcoef * scale;
      c.sgn = scale < 0.f ? -1.f : 1.f;
      c.sabs = fabsf(scale);
      c.sl2 = c.sabs * kLog2e;  // exponent per unit of (sign-adjusted) raw logit, in bits
      return c;
    };

    // ---- state of the unit whose G is still to be finished (the previous one) ----
    uint32_t pk[kXSliceCols / 2];                       // exp(l - m_running) of this thread's columns, bf16 pairs
    float p_gm[kXGroups];                               // running max each group was written against
#pragma unroll
    for (int g = 0; g < kXGroups; ++g) p_gm[g] = 0.f;
    float p_before = 0.f, p_lraw = 0.f, p_lab_p = 0.f, p_lab_gm = 0.f;
    int p_label = -1;
    int p_tile = -1;
    const uint4* p_rec = wk.recs;                       // the row's records, one per class chunk
    // resolved when the unit is finished: row maximum, factor coef / sum, the one-hot column's value
    float f_M = 0.f, f_tc = 0.f, f_sl2 = 0.f;
    unsigned short f_patch = 0;
    bool f_store = false;
    unsigned char* f_grow = nullptr;
    // per-run sums of the rows this thread owns (slice 0, label column inside the chunk): reduced over the warp ONCE, when
    // the CTA has done all its units
    float acc_loss[2] = {0.f, 0.f}, acc_ds[2] = {0.f, 0.f};
    int acc_hit[2] = {0, 0}, acc_cnt[2] = {0, 0};

    // the class chunks' records of the previous unit (this pair's own among them: slice 0 published it, the other slices
    // never saw the combined values): requested after the new unit's first group, looked at two groups later - the
    // L2 round trip is covered by those groups' work
    uint4 r0[kXMaxChunks], r1[kXMaxChunks];
    auto request_prev = [&]() {
      if (static_cast<int64_t>(p_tile) * 128 + rloc < n_rows) {
#pragma unroll
        for (int c2 = 0; c2 < kXMaxChunks; ++c2) {
          if (c2 < n_chunks) {
            r0[c2] = ld_volatile_v4(p_rec + c2 * 2);
            if (kSecond) r1[c2] = ld_volatile_v4(p_rec + c2 * 2 + 1);
          }
        }
      }
    };
    // ... -> row maximum / sum (polls only if a pair is most of a unit behind)
    auto resolve_prev = [&]() {
      const int64_t row = static_cast<int64_t>(p_tile) * 128 + rloc;
      const RowCtx c = row_ctx(row);
      float M = -INFINITY, S = 0.f, PR = 0.f, before_chunks = -INFINITY;
      int garg = 0x7fffffff;
      if (c.valid) {
        // a stale record (a pair most of a unit behind): ask again for all of them at once
        for (unsigned polls = 0;; ++polls) {
          bool fresh = true;
#pragma unroll
          for (int c2 = 0; c2 < kXMaxChunks; ++c2) {
            if (c2 < n_chunks) {
              fresh = fresh && r0[c2].y == epoch && r0[c2].w == epoch;
              if (kSecond) fresh = fresh && r1[c2].y == epoch && r1[c2].w == epoch;
            }
          }
          if (fresh) break;
          if (polls > (1u << 20)) {  // ~ a second: never hang the GPU; the host checks the flag
            atomicExch(wk.ctrl + 2, 1u);
            break;
          }
          request_prev();
        }
        float om[kXMaxChunks], os[kXMaxChunks];
#pragma unroll
        for (int c2 = 0; c2 < kXMaxChunks; ++c2) {
          om[c2] = c2 < n_chunks ? __uint_as_float(r0[c2].x) : -INFINITY;
          os[c2] = c2 < n_chunks ? __uint_as_float(r0[c2].z) : 0.f;
          M = fmaxf(M, om[c2]);
          if (c2 < chunk) before_chunks = fmaxf(before_chunks, om[c2]);
        }
        const float offM = __fmul_rn(M, c.sl2);
#pragma unroll
        for (int c2 = 0; c2 < kXMaxChunks; ++c2) {
          const float e = x_exp2(__fmul_rn(om[c2], c.sl2) - offM);  // 0 for the absent chunks (-inf)
          S = fmaf(os[c2], e, S);
          if (kDs) PR = fmaf(c2 < n_chunks ? __uint_as_float(r1[c2].x) : 0.f, e, PR);
        }
        if (kPred) {  // the first chunk that holds the row maximum (chunks in class order)
          float bestm = -INFINITY;
#pragma unroll
          for (int c2 = 0; c2 < kXMaxChunks; ++c2) {
            if (c2 < n_chunks && om[c2] > bestm) {
              bestm = om[c2];
              garg = static_cast<int>(r1[c2].z);
            }
          }
        }
      }
      f_M = __fmul_rn(M, c.sl2);  // the row's exponent offset, in bits: off(m) = m * sl2 rounded once, everywhere
      f_sl2 = c.sl2;
      f_tc = __fdividef(c.gcoef, S);
      f_store = c.valid && live_groups > 0;
      f_grow = reinterpret_cast<unsigned char*>(G) + (row * ldg + col0 + cq * kXSliceCols) * 2;
      {
        // the one-hot column from the staged element in fp32 (G = p * f - coef, one rounding); stored after the row's
        // vector stores (a later store of the same thread to the same address is ordered after them)
        const float f = x_exp2(__fmul_rn(p_lab_gm, c.sl2) - f_M) * f_tc;
        f_patch = __bfloat16_as_ushort(__float2bfloat16_rn(fmaf(p_lab_p, f, -c.gcoef)));
      }
      if (cq == 0) {  // per-row results: the (chunk, slice 0) thread of the chunk that holds the row's label column
        const int lc_chunk = p_label - col0;
        if (c.valid && lc_chunk >= 0 && lc_chunk < 256) {
          // ln S - ln 2 * (u_label - offset), the label's exponent taken exactly as pass 1 took it: S >= 2^that up to the
          // 2^-22 of ex2.approx, so the cross entropy is >= -3e-7 before the clamp (torch's is never negative)
          const float loss = fmaxf(fmaf(__log2f(S), 0.6931471805599453f, -0.6931471805599453f * fmaf(p_lraw, c.sl2, -f_M)), 0.f);
          const float dsc = kDs ? (__fdividef(PR, S) - p_lraw) * c.sgn * c.dcoef : 0.f;
          const int hit = (p_lraw == M && p_lraw > fmaxf(before_chunks, p_before)) ? 1 : 0;
          if (row_loss) row_loss[row] = loss;
          if (kPred && row_pred) row_pred[row] = garg;
          if (row_correct) row_correct[row] = hit;
          if (kDs && row_dscale) row_dscale[row] = dsc;
          if (c.sg) { acc_loss[1] += loss; acc_ds[1] += dsc; acc_hit[1] += hit; acc_cnt[1] += 1; }
          else { acc_loss[0] += loss; acc_ds[0] += dsc; acc_hit[0] += hit; acc_cnt[0] += 1; }
        }
      }
    };
    // final G of 16 columns of the previous unit: p_final * coef / S = p_staged * exp(m_staged - M) * coef / S; the factor
    // split hi + lo so that the product of two bf16x2 operations carries fp32-level accuracy before the one rounding
    auto finish_group = [&](auto gc) {
      constexpr int g = decltype(gc)::value;
      if (!f_store || g >= live_groups) return;
      const float gmx = p_gm[g];
      const float f = x_exp2(__fmul_rn(gmx, f_sl2) - f_M) * f_tc;
      const __nv_bfloat16 fh = __float2bfloat16_rn(f);
      const __nv_bfloat16 fl = __float2bfloat16_rn(f - __bfloat162float(fh));
      const __nv_bfloat162 fh2 = __halves2bfloat162(fh, fh), fl2 = __halves2bfloat162(fl, fl);
      uint32_t o[kXGW];
#pragma unroll
      for (int j = 0; j < kXGW; ++j) {
        const __nv_bfloat162 pv = *reinterpret_cast<const __nv_bfloat162*>(&pk[g * kXGW + j]);
        const __nv_bfloat162 r = __hfma2(pv, fh2, __hmul2(pv, fl2));
        o[j] = *reinterpret_cast<const uint32_t*>(&r);
      }
#ifdef UML_X_NOSTORE
      if (f_M == 12345.678f)
#endif
#pragma unroll
      for (int j = 0; j < kXGW; j += 8) stg256(f_grow + g * (2 * kXGC) + j * 4, o + j);
    };
    // the same through shared memory: the warp's 32 rows x 32 columns go into one of its two staging boxes (16-byte chunk
    // c of row r at chunk c ^ ((r >> 1) & 3): SWIZZLE_64B, conflict-free for a row per lane), the one-hot column is
    // patched there, and one TMA store writes the box - rows past n_rows are clipped by the tensor map
    const uint32_t sbuf_w = smem_u32(sbuf) + warp * kXSbufWarp;
    auto finish_group_tma = [&](auto gc) {
      constexpr int g = decltype(gc)::value;
      static_assert(!kXTmaStore || kXGC == 32, "the staging boxes are 32 columns wide");
      if (g >= live_groups) return;  // (warp-uniform)
      const float gmx = p_gm[g];
      const float f = x_exp2(__fmul_rn(gmx, f_sl2) - f_M) * f_tc;
      const __nv_bfloat16 fh = __float2bfloat16_rn(f);
      const __nv_bfloat16 fl = __float2bfloat16_rn(f - __bfloat162float(fh));
      const __nv_bfloat162 fh2 = __halves2bfloat162(fh, fh), fl2 = __halves2bfloat162(fl, fl);
      uint32_t o[kXGW];
#pragma unroll
      for (int j = 0; j < kXGW; ++j) {
        const __nv_bfloat162 pv = *reinterpret_cast<const __nv_bfloat162*>(&pk[g * kXGW + j]);
        const __nv_bfloat162 r = __hfma2(pv, fh2, __hmul2(pv, fl2));
        o[j] = *reinterpret_cast<const uint32_t*>(&r);
      }
      const uint32_t box = sbuf_w + (g & 1) * 2048, rowb = box + lane * 64, sw = (lane >> 1) & 3;
      if (lane == 0) bulk_wait_read<1>();  // the store that last used this box (two stores ago) has read it
      __syncwarp();
#pragma unroll
      for (int j4 = 0; j4 < kXGW / 4; ++j4) sts128(rowb + ((j4 ^ sw) << 4), o[4 * j4], o[4 * j4 + 1], o[4 * j4 + 2], o[4 * j4 + 3]);
      const int lc = p_label - col0 - cq * kXSliceCols - g * kXGC;
      if (static_cast<unsigned>(lc) < static_cast<unsigned>(kXGC))
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(rowb + (((lc >> 3) ^ sw) << 4) + (lc & 7) * 2), "h"(f_patch) : "memory");
      fence_proxy_async();
      __syncwarp();
#ifndef UML_X_NOSTORE
      if (lane == 0) {
        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                         reinterpret_cast<uint64_t>(&tmap_g)),
                     "r"(box), "r"(col0 + cq * kXSliceCols + g * kXGC), "r"(p_tile * 128 + q * 32)
                     : "memory");
        bulk_commit();
      }
#endif
    };
    auto finish_any = [&](auto gc) {
      if constexpr (kXTmaStore) finish_group_tma(gc);
      else finish_group(gc);
    };
    // the one-hot column of the previous unit
    auto finish_rows = [&]() {
      if (kXTmaStore) return;  // (patched in the staging box)
      const int lcol = p_label - col0 - cq * kXSliceCols;
      if (f_store && lcol >= 0 && lcol < kXSliceCols) *reinterpret_cast<volatile unsigned short*>(f_grow + lcol * 2) = f_patch;
    };

    int next_label = -1;
    {
      const int64_t frow = (static_cast<int64_t>(group) * 2 + rank) * 128 + rloc;
      if (group < n_units && frow < n_rows) next_label = __ldg(labels + frow);
    }
    for (int unit = group; unit < static_cast<int>(n_units); unit += n_groups, ++tile_it) {
      const int tile = unit * 2 + static_cast<int>(rank);
      const int64_t row = static_cast<int64_t>(tile) * 128 + rloc;
      const RowCtx c = row_ctx(row);
      const float sl2 = c.sl2, sgn = c.sgn;
      const int label = next_label;
      {  // the next unit's label: its load is in flight for a whole unit
        const int64_t nrow = (static_cast<int64_t>(unit + n_groups) * 2 + rank) * 128 + rloc;
        next_label = nrow < n_rows ? __ldg(labels + nrow) : -1;
      }
#ifdef UML_X_NOLABEL
      const int lcol = -1000000;
#else
      const int lcol = label - col0 - cq * kXSliceCols;  // label position inside this thread's columns
#endif
      // running statistics of this thread's quarter row, in the raw (sign-adjusted) logit domain
      float run_max = -INFINITY, run_sum = 0.f, run_pr = 0.f, max_before = -INFINITY, lab_raw = -INFINITY;
      float lab_p = 0.f, lab_gm = 0.f;                  // the label column's staged exponential and the max it was taken against
      int arg = 0x7fffffff;
      float gm[kXGroups];
      const bool have_prev = p_tile >= 0;

      const uint32_t b = tile_it & 1, aph = (tile_it >> 1) & 1;
      XDBG_MARK();
      mbar_wait(&tfull_bar[b], aph);
      XDBG_ACC(0);
      tc_fence_after();
#ifdef UML_X_NOEPI
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (!leader) mbar_arrive_remote(tempty_remote0 + b * 8);
        else mbar_arrive(&tempty_bar[b]);
      }
      continue;
#endif
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + b * 256 + cq * kXSliceCols;
      uint32_t vv[kXDoubleBuf ? 2 : 1][kXGC];
      uint32_t nk[kXGW * kXHalf];  // the new unit's first four groups: live beside the previous unit's registers until those are stored

      // one 16-column group: running max, exponentials relative to it, packed as bf16 pairs into out[0..8).
      // kPlain: every column of the chunk is a class and no temperature is negative (all but the last chunk's tail)
      const uint64_t sl2x2 = pack2(sl2, sl2);
      auto run_group = [&](uint32_t (&v)[kXGC], uint32_t* out, auto gc) -> float {
        constexpr int g = decltype(gc)::value;
        const int c0l = cq * kXSliceCols + g * kXGC;  // first column of the group inside the chunk
        if (c0l + kXGC > n_valid || any_neg) {  // (uniform; only the last chunk's tail - or a negative temperature)
          if (c0l >= n_valid) {            // nothing but padding (or TMEM columns beyond the MMA's N): G stays zero there
#pragma unroll
            for (int j = 0; j < kXGW; ++j) out[j] = 0u;
            return run_max;
          }
          if (any_neg) {
#pragma unroll
            for (int i = 0; i < kXGC; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * sgn);
          }
          if (c0l + kXGC > n_valid) {  // padded class columns
#pragma unroll
            for (int i = 0; i < kXGC; ++i)
              if (c0l + i >= n_valid) v[i] = __float_as_uint(kMasked);
          }
        }
        float m0 = fmaxf(__uint_as_float(v[0]), __uint_as_float(v[1])), m1 = fmaxf(__uint_as_float(v[2]), __uint_as_float(v[3]));
#pragma unroll
        for (int i = 4; i < kXGC; i += 4) {
          m0 = fmaxf(m0, fmaxf(__uint_as_float(v[i]), __uint_as_float(v[i + 1])));
          m1 = fmaxf(m1, fmaxf(__uint_as_float(v[i + 2]), __uint_as_float(v[i + 3])));
        }
        const float bm = fmaxf(m0, m1);
        // hit flag without an argmax index:  argmax == label  <=>  logit[label] == row max  and
        // logit[label] > max over the columns before it  (torch.argmax returns the FIRST maximal index)
        const int d = lcol - g * kXGC;
        const bool lab_here = static_cast<unsigned>(d) < static_cast<unsigned>(kXGC);
        if (d >= kXGC) max_before = fmaxf(max_before, bm);
        if (lab_here) {  // (divergent: one lane in thirty)
          // v[d] by a jump (one or two lanes of the warp are here: a branch per lane beats a select tree run by all),
          // then the columns before d only if the label can still be the first maximum
          lab_raw = pick_col(v, d);
          if (lab_raw == bm) {
            float b0 = -INFINITY, b1 = -INFINITY;
#pragma unroll
            for (int i = 0; i < kXGC; i += 2) {
              b0 = fmaxf(b0, i < d ? __uint_as_float(v[i]) : -INFINITY);
              b1 = fmaxf(b1, i + 1 < d ? __uint_as_float(v[i + 1]) : -INFINITY);
            }
            max_before = fmaxf(max_before, fmaxf(b0, b1));
          } else {
            max_before = fmaxf(max_before, bm);  // something in this group beats the label: any such value says "no hit"
          }
        }
        if (kPred && bm > run_max) {  // first column holding the new maximum (columns are visited in order)
#pragma unroll
          for (int i = kXGC - 1; i >= 0; --i)
            if (__uint_as_float(v[i]) == bm) arg = col0 + c0l + i;
        }
        // exponent offsets are off(m) = m * sl2 rounded ONCE (never fused), differences of offsets are exact: rescaling
        // a sum from one running maximum to the next telescopes, and the label's term of the final sum is exactly the
        // 2^(u_label - off(M)) the loss subtracts
        const float new_max = fmaxf(run_max, bm);
        const float noff = -__fmul_rn(new_max, sl2);
        const float resc = x_exp2(__fmul_rn(run_max, sl2) + noff);  // exp2(-inf) = 0 on the first group
        run_sum *= resc;
        if (kDs) run_pr *= resc;
        run_max = new_max;
        const uint64_t noffx2 = pack2(noff, noff);
        uint64_t sx2 = pack2(0.f, 0.f), sy2 = pack2(0.f, 0.f);
        float q0 = 0.f, q1 = 0.f;
#pragma unroll
        for (int j = 0; j < kXGW; ++j) {
          const float r0 = __uint_as_float(v[2 * j]), r1 = __uint_as_float(v[2 * j + 1]);
          float t0, t1;
          unpack2(ffma2(pack2(r0, r1), sl2x2, noffx2), t0, t1);  // u - off(max), one rounding
          const float p0 = x_exp2(t0), p1 = x_exp2(t1);
          if (j & 1) sy2 = fadd2(sy2, pack2(p0, p1));
          else sx2 = fadd2(sx2, pack2(p0, p1));
          if (kDs) {
            q0 = fmaf(p0, r0, q0);
            q1 = fmaf(p1, r1, q1);
          }
          const __nv_bfloat162 hh = __floats2bfloat162_rn(p0, p1);
          out[j] = *reinterpret_cast<const uint32_t*>(&hh);
        }
        float s0, s1;
        unpack2(fadd2(sx2, sy2), s0, s1);
        run_sum += s0 + s1;
        if (kDs) run_pr += q0 + q1;
        if (lab_here) {  // the label column's staged value, as it was rounded (the same three operations as in the loop)
          lab_p = __bfloat162float(__float2bfloat16_rn(x_exp2(__fmaf_rn(lab_raw, sl2, noff))));
          lab_gm = new_max;
        }
        return new_max;
      };

      // ---- the first half of the new unit goes to registers of its own: the other chunks publish the previous unit's
      //      row statistics at the END of their iteration, so looking at them half a unit later (nearly) never finds them
      //      missing - CTA pairs of a group may drift by a good part of a unit without anybody waiting. ----
      // (double-buffered: wait for group g, start the load of group g + 1 into the other register set, then work on
      //  g - measured slower, off.)  Groups 0 .. kXHalf-1 of the new unit go to registers of their own (nk) - the
      //  previous unit still sits in pk; after group kXHalf-1 its records are looked at, it is finished, and from then
      //  on group g of the new unit takes the registers group g of the previous unit has just left.
      constexpr int kB = kXDoubleBuf ? 1 : 0;  // buffer of group g: g & kB
      tmem_ldg(taddr, vv[0]);
      static_for<0, kXGroups>([&](auto gc) {
        constexpr int g = decltype(gc)::value;
        constexpr bool last = g == kXGroups - 1;
        tmem_ld_wait();
        pin16(vv[g & kB]);
        if (g == 0) XDBG_ACC(1);
        if (last) {
          // accumulator buffer b may be overwritten by the (leader's) MMA warp now
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (!leader) mbar_arrive_remote(tempty_remote0 + b * 8);
            else mbar_arrive(&tempty_bar[b]);
          }
        } else if (kXDoubleBuf) {
          tmem_ldg(taddr + kXGC * (g + 1), vv[(g + 1) & kB]);
        }
        gm[g] = run_group(vv[g & kB], g < kXHalf ? nk + kXGW * g : pk + kXGW * g, gc);
        if (!last && !kXDoubleBuf) tmem_ldg(taddr + kXGC * (g + 1), vv[0]);
        if (g == kXReqAfter && have_prev) request_prev();  // (the L2 round trip is covered by the next groups)
        if (g == kXHalf - 1) {
          if (have_prev) {
            resolve_prev();
            static_for<0, (kXHalf + 1 < kXGroups ? kXHalf + 1 : kXGroups)>([&](auto fc) { finish_any(fc); });
          }
#pragma unroll
          for (int j = 0; j < kXGW * kXHalf; ++j) pk[j] = nk[j];
        } else if (g >= kXHalf && !last) {
          if (have_prev) finish_any(std::integral_constant<int, g + 1>());
        }
      });
      XDBG_ACC(2);
      if (have_prev) finish_rows();
      XDBG_ACC(3);

      // ---- the column slices of a row meet in slice 0's thread (shared memory): the other slices drop their record and
      //      go on - they never wait; slice 0 (nearly always the last to get here: it also owns the per-row results)
      //      combines and publishes the chunk's record to the other class chunks of the row (L2).  Every value travels
      //      with the launch epoch in the same 8-byte word pair (which the memory system delivers whole): a reader
      //      checks the epoch - no fence, no flag.  Slot reuse: a slot is written again four units later, which needs
      //      the accumulator of two units later, which slice 0 frees after it has read this slot.
      const uint32_t hx_slot = hx_base + (tile_it & (kXHxSlots - 1)) * ((kXSlices - 1) * 128 * kXRecBytes);
      const uint4* rec_row = wk.recs + row * n_chunks * 2;
      if (cq != 0) {
        const uint32_t mine = hx_slot + ((cq - 1) * 128 + rloc) * kXRecBytes;
        sts128(mine, __float_as_uint(run_max), __float_as_uint(run_sum), __float_as_uint(max_before), __float_as_uint(lab_raw));
        if (kSecond) sts64(mine + 16, __float_as_uint(run_pr), static_cast<uint32_t>(arg));
        __syncwarp();
        if (lane == 0) mbar_arrive(&xbar[q]);
      } else {
        mbar_wait(&xbar[q], tile_it & 1);
        float cm = run_max, before_loc = max_before, lraw = lab_raw;
        constexpr int kOthers = kXSlices - 1;
        float o_max[kOthers], o_sum[kOthers], o_pr[kOthers];
        int o_arg[kOthers];
#pragma unroll
        for (int k = 0; k < kOthers; ++k) {
          const uint32_t other = hx_slot + (k * 128 + rloc) * kXRecBytes;
          const uint4 o4 = lds128(other);
          o_max[k] = __uint_as_float(o4.x);
          o_sum[k] = __uint_as_float(o4.y);
          cm = fmaxf(cm, o_max[k]);
          before_loc = fmaxf(before_loc, __uint_as_float(o4.z));  // slices before the label's hold their whole max, later ones -inf
          lraw = fmaxf(lraw, __uint_as_float(o4.w));               // exactly one slice saw the label column (the others hold -inf)
          o_pr[k] = 0.f;
          o_arg[k] = 0;
          if (kSecond) {
            const uint2 o2 = lds64(other + 16);
            o_pr[k] = __uint_as_float(o2.x);
            o_arg[k] = static_cast<int>(o2.y);
          }
        }
        const float offc = __fmul_rn(cm, sl2);
        const float e_me = x_exp2(__fmul_rn(run_max, sl2) - offc);
        float cs = run_sum * e_me, cpr = kDs ? run_pr * e_me : 0.f;
#pragma unroll
        for (int k = 0; k < kOthers; ++k) {
          const float e = x_exp2(__fmul_rn(o_max[k], sl2) - offc);
          cs = fmaf(o_sum[k], e, cs);
          if (kDs) cpr = fmaf(o_pr[k], e, cpr);
        }
        int carg = arg;
        if (kPred) {  // the chunk's first maximal column: the lowest slice among those that hold the chunk maximum
          float bmx = run_max;
#pragma unroll
          for (int k = 0; k < kOthers; ++k) {
            if (o_max[k] > bmx) {
              bmx = o_max[k];
              carg = o_arg[k];
            }
          }
        }
        if (c.valid) {
          uint4* rec = const_cast<uint4*>(rec_row) + chunk * 2;
          st_volatile_v4(rec, __float_as_uint(cm), epoch, __float_as_uint(cs), epoch);
          if (kSecond) st_volatile_v4(rec + 1, __float_as_uint(cpr), epoch, static_cast<uint32_t>(carg), epoch);
        }
        p_before = before_loc;
        p_lraw = lraw;
      }
      XDBG_ACC(4);
      // this unit becomes the previous one
#pragma unroll
      for (int g = 0; g < kXGroups; ++g) p_gm[g] = gm[g];
      p_lab_p = lab_p; p_lab_gm = lab_gm;
      p_label = label; p_tile = tile; p_rec = rec_row;
    }
    if (p_tile >= 0) {  // the last unit
      XDBG_MARK();
      request_prev();
      resolve_prev();
      XDBG_ACC(5);
      static_for<0, kXGroups>([&](auto gc) { finish_any(gc); });
      finish_rows();
      XDBG_ACC(6);
    }
    if (kXTmaStore && lane == 0) bulk_wait<0>();  // this warp's G stores are complete (and have left its staging boxes)
    if (cq == 0 && wk.tile_part) {
      // deterministic per-(CTA, row quarter, run) partial sums; the statistics kernel adds them in a fixed order
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2) {
        const float a = warp_sum(acc_loss[s2]), dd = kDs ? warp_sum(acc_ds[s2]) : 0.f;
        const int hh = warp_sum_i(acc_hit[s2]), cnt = warp_sum_i(acc_cnt[s2]);
        if (lane == 0)
          *reinterpret_cast<float4*>(wk.tile_part + ((static_cast<int64_t>(blockIdx.x) * 4 + q) * 2 + s2) * 4) =
              make_float4(a, dd, static_cast<float>(hh), static_cast<float>(cnt));
      }
    }
#ifdef UML_FWD_TIMING
    if (warp == 0 && lane == 0) XDBG_FLUSH(0, 9);
#endif
  }

  tc_fence_before();
  cluster_sync_all();  // the leader's MMAs read the peer's shared memory until the last commit
  if (warp == kXWarpTma) tmem_dealloc_cg2(tmem_base, 512);
  if (threadIdx.x == 0) {
    // the last CTA of the grid closes the launch: flags written with `epoch` can never match a later launch
    __threadfence();
    const unsigned done = atomicAdd(wk.ctrl + 1, 1u);
    if (done == gridDim.x - 1) {
      wk.ctrl[1] = 0u;
      __threadfence();
      *reinterpret_cast<volatile unsigned*>(wk.ctrl) = epoch;
    }
  }
}

// per-run statistics from the per-(tile, chunk, warp) partials, summed in a fixed order; one CTA per run
__global__ void __launch_bounds__(1024)
    x_tile_stats_kernel(const float* __restrict__ tile_part, int64_t n_entries, uml_seg_stats* __restrict__ out) {
  __shared__ float sh[4][32];
  const int s = blockIdx.x;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int64_t i = threadIdx.x; i < n_entries; i += blockDim.x) {
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

// the same with the number of partial records read from the workspace (uml_reduce_tile_stats knows no class count)
__global__ void __launch_bounds__(1024)
    x_tile_stats_dev_kernel(const float* __restrict__ tile_part, const unsigned* __restrict__ ctrl, uml_seg_stats* __restrict__ out) {
  __shared__ float sh[4][32];
  const int s = blockIdx.x;
  const int64_t n_entries = ctrl[3];
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int64_t i = threadIdx.x; i < n_entries; i += blockDim.x) {
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

// workspace carving (UML_TILE_WS_FLOATS): [ctrl 16 u32][(unused) units*8][tile_part units*256 f][recs n_rows*4*8 f]
struct XLayout {
  unsigned* ctrl;
  float* tile_part;
  uint4* recs;
  int64_t part_entries;  // (CTA, row quarter) partial records per run
  int64_t n_groups;      // CTA-pair groups of the launch: grid = n_groups * n_chunks * 2
};
static XLayout x_layout(float* tile_ws, int64_t n_rows, int n_classes) {
  const int64_t units = (n_rows + 255) / 256;
  const int n_chunks = (n_classes + 255) / 256;
  XLayout l;
  l.ctrl = reinterpret_cast<unsigned*>(tile_ws);
  l.tile_part = tile_ws + 16 + units * 8;
  l.recs = reinterpret_cast<uint4*>(l.tile_part + units * 256);
  l.n_groups = (sm_count() / 2) / n_chunks;
  if (l.n_groups > units) l.n_groups = units;
  l.part_entries = l.n_groups * n_chunks * 2 * 4;  // (<= units * 32: fits the units * 256 floats set aside for them)
  return l;
}

}  // namespace uml

// true when the exchange kernel serves this shape (else tc_fwd.cu's chunk-sequential kernel runs)
bool uml_fwd_x_eligible(int64_t n_rows, int32_t n_classes) {
  return n_rows > 128 && n_classes <= uml::kXMaxChunks * 256;
}

// where the per-(tile, chunk, warp) partials of the exchange kernel live and how many there are per run
void uml_fwd_x_partials(float* tile_ws, int64_t n_rows, int32_t n_classes, const float** part, int64_t* n_entries) {
  const uml::XLayout l = uml::x_layout(tile_ws, n_rows, n_classes);
  *part = l.tile_part;
  *n_entries = l.part_entries;
}

int uml_head_fwd_ce_x_bf16(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W, int32_t n_classes,
                           const int32_t* labels, const uml_tc_segments* segs, uint16_t* G, int64_t ldg, float* row_loss,
                           int32_t* row_pred, int32_t* row_correct, float* row_dscale, float* tile_ws, uml_seg_stats* stats,
                           void* stream) {
  using namespace uml;
  UML_REQUIRE(X && W && labels && segs && tile_ws && n_rows > 0 && dim > 0 && n_classes > 0, "head_fwd_ce_x: bad arguments");
  UML_REQUIRE(dim % 8 == 0, "head_fwd_ce_x: dim (%d) must be a multiple of 8 (16-byte bf16 rows for TMA)", dim);
  UML_REQUIRE(n_classes <= kXMaxChunks * 256, "head_fwd_ce_x: at most %d classes", kXMaxChunks * 256);
  UML_REQUIRE(!G || (ldg % 64 == 0 && ldg >= n_classes && ldg <= kXMaxChunks * 256),
              "head_fwd_ce_x: ldg must be a multiple of 64 and >= n_classes");
  UML_REQUIRE(segs->nseg >= 1 && segs->nseg <= UML_MAX_SEGMENTS, "head_fwd_ce_x: 1..2 segments");
  const int64_t n0 = segs->seg_rows[0], n1 = segs->nseg > 1 ? segs->seg_rows[1] : 0;
  UML_REQUIRE(n0 + n1 == n_rows, "head_fwd_ce_x: segment rows (%lld+%lld) != n_rows (%lld)", (long long)n0, (long long)n1,
              (long long)n_rows);
  CUtensorMap tx, tw;
  if (make_tmap_2d(&tx, X, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dim, n_rows, static_cast<uint64_t>(dim) * 2, 64, 128,
                   CU_TENSOR_MAP_SWIZZLE_128B))
    return 1;
  if (make_tmap_2d(&tw, W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, dim, n_classes, static_cast<uint64_t>(dim) * 2, 64, 128,
                   CU_TENSOR_MAP_SWIZZLE_128B))
    return 1;
  CUtensorMap tg = tx;  // (prediction mode: never used)
  if (kXTmaStore && G &&
      make_tmap_2d(&tg, G, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, static_cast<uint64_t>(ldg), n_rows, static_cast<uint64_t>(ldg) * 2, 32, 32,
                   CU_TENSOR_MAP_SWIZZLE_64B))
    return 1;
  XSegs fs;
  fs.n0 = segs->nseg > 1 ? n0 : INT64_MAX;
  bool learnable = false;
  for (int i = 0; i < 2; ++i) {
    const int j = i < segs->nseg ? i : 0;
    const double n = static_cast<double>(segs->seg_rows[j] > 0 ? segs->seg_rows[j] : 1);
    fs.scale[i] = segs->scale[j];
    fs.scale_dev[i] = segs->scale_dev[j];
    fs.dcoef[i] = static_cast<float>(static_cast<double>(segs->loss_weight[j]) / n);
    learnable = learnable || segs->scale_dev[j] != nullptr;
  }
  const bool ds = learnable || row_dscale != nullptr;  // the sum p * raw is only needed for d loss / d scale
  using Kern = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, int64_t, int, int, int, const int32_t*, XSegs, uint16_t*, int64_t, float*,
                        int32_t*, int32_t*, float*, XWork);
  const int slot = (row_pred ? 2 : 0) + (ds ? 1 : 0);
  const Kern kerns[4] = {head_fwd_ce_x_kernel<false, false>, head_fwd_ce_x_kernel<false, true>,
                         head_fwd_ce_x_kernel<true, false>, head_fwd_ce_x_kernel<true, true>};
  static bool attr_set[4] = {false, false, false, false};
  if (!attr_set[slot]) {
    UML_CUDA(cudaFuncSetAttribute(kerns[slot], cudaFuncAttributeMaxDynamicSharedMemorySize, kXSmemBytes));
    attr_set[slot] = true;
  }
  const int n_chunks = (n_classes + 255) / 256;
  const XLayout l = x_layout(tile_ws, n_rows, n_classes);
  const int64_t n_groups = l.n_groups;
  UML_REQUIRE(n_groups >= 1, "head_fwd_ce_x: the device has too few SMs for %d class chunks", n_chunks);
  XWork wk;
  wk.tile_part = l.tile_part;
  wk.recs = l.recs;
  wk.ctrl = l.ctrl;
  const dim3 grid(static_cast<unsigned>(n_groups * n_chunks * 2));
  UML_CUDA(launch_kernel(kerns[slot], grid, dim3(kXThreads), kXSmemBytes, as_stream(stream), 2, tx, tw, tg, n_rows,
                         static_cast<int>(dim), static_cast<int>(n_classes), static_cast<int>(n_groups), labels, fs, G, ldg,
                         row_loss, row_pred, row_correct, row_dscale, wk));
  if (stats)
    UML_CUDA(launch_kernel(x_tile_stats_kernel, dim3(segs->nseg), dim3(1024), 0, as_stream(stream), 1,
                           static_cast<const float*>(l.tile_part), l.part_entries, stats));
  return 0;
}

// per-run statistics from the partials of the last exchange-kernel launch on this workspace (record count read from it)
int uml_fwd_x_reduce_stats(float* tile_ws, int64_t n_rows, int32_t nseg, uml_seg_stats* stats, void* stream) {
  using namespace uml;
  const XLayout l = x_layout(tile_ws, n_rows, 1);  // (the offsets do not depend on the class count)
  UML_CUDA(launch_kernel(x_tile_stats_dev_kernel, dim3(nseg), dim3(1024), 0, as_stream(stream), 1,
                         static_cast<const float*>(l.tile_part), static_cast<const unsigned*>(l.ctrl), stats));
  return 0;
}

extern "C" {

#ifdef UML_FWD_TIMING
int uml_debug_fwdx_timing(long long* host_out /* [148*16] */, int reset) {
  if (reset) {
    static long long zeros[148 * 16];
    return cudaMemcpyToSymbol(uml::g_fwdx_dbg, zeros, sizeof(zeros)) != cudaSuccess;
  }
  return cudaMemcpyFromSymbol(host_out, uml::g_fwdx_dbg, sizeof(long long) * 148 * 16) != cudaSuccess;
}
#endif

// 1 when a launch of the exchange forward kernel ever timed out waiting for a peer CTA pair (results of that launch
// are undefined); the workspace it used is passed in.  Synchronises the device.
int uml_fwd_x_failed(const float* tile_ws) {
  unsigned v = 0;
  if (cudaMemcpy(&v, reinterpret_cast<const unsigned*>(tile_ws) + 2, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return v != 0 ? 1 : 0;
}

}  // extern "C"
