// Sweep-level batching of the exact fp32 step (SURVEY section 8 f-1; reference: the hyper-parameter loop of
// vision_language/finetune.py:406-448 over engine/optimizer/default.py's grids).
//
// The reference trains the lr x weight-decay (x alpha) combinations of a sweep one after the other over the SAME
// feature banks, each a 32-row step that cannot fill one SM.  Here K heads (own weights, optimizer state, sampler
// stream, lr, weight decay and alpha) advance in lock step: every launch covers all heads, so one step of all K heads
// is two launches - logits with softmax / CE in the epilogue (the class tiles of a head form a cluster), dW + optimizer
// update (+ statistics) - and the last one streams K x 24 B/parameter from HBM with the whole machine.
//
// Layout in HBM: W, m, v are [K][C*D] slabs (head_stride apart); G is [K][rows][ldg] scratch; every head reads its
// own epoch permutation (device int64) at the common position `pos` - the heads share bank and batch sizes, so their
// epochs turn over on the same steps.
//
// The two contractions exist in three forms:
//   * tensor cores (default when rows are 16-byte aligned): tcgen05.mma kind::tf32 with every operand split into two tf32
//     terms, i.e. fp32-level accuracy (section "Tensor-core forms" below); W, m, v of the update move through a TMA
//     slot ring; softmax / CE in the logits epilogue when a head has at most eight class tiles (a cluster).  Measured on
//     B200 with K = 30 heads of 1000 x 512: 0.134 ms per step of all heads (logits + softmax/CE 44 us, dW + update +
//     statistics 76 = 0.76 of the HBM copy peak); with the separate softmax launch 0.139 ms (logits 36, softmax/CE 15);
//   * FFMA with cp.async staging (UML_SWEEP_TC=0, and the dW + update of steps with more than 64 rows): 0.219 ms
//     (logits 73, softmax/CE 15, dW + update 123 = 0.47 of the HBM peak, stats 7);
//   * FFMA, register-staged (any alignment; UML_SWEEP_ASYNC=0): 0.268 ms.
// Per head the arithmetic of the FFMA forms is the single-head fp32 path's (simt.cu): sequential-k FFMA logits, the
// same softmax / CE / argmax row kernel, dW summed over rows in order, torch.optim's update rules in the epilogue.  In
// every form a head's result depends neither on its slot in the group nor on its neighbours.
#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace uml {
namespace sweep {

constexpr int kMaxHeads = UML_SWEEP_MAX_HEADS;

struct SweepDev {
  const float* bank[2];
  const int64_t* labels[2];
  int64_t ld[2];
  int64_t n0, n1;   // rows of the image run / text run in this step
  int64_t pos[2];   // position of the step's batch inside each head's permutation
  const int64_t* perm[2][kMaxHeads];
  float* W;
  float* m;
  float* v;
  int64_t head_stride;
  float* G;
  int64_t ldg, g_stride;
  float* row_loss;
  int32_t* row_correct;
  int64_t row_stride;
  uml_seg_stats* stats;  // [K][2] for this step
  int dim, n_classes;
  float scale[2];
  float alpha[kMaxHeads];
  uint32_t active_mask;
  int vec_rows;  // dim % 4 == 0 and every bank row / weight row starts on a 16-byte boundary
  // optimizer (kind: 1 AdamW, 2 Adam with L2, 3 SGD momentum with L2); per-head scalars derived on the host in double
  int kind, first_step;
  float beta1, beta2, eps, momentum, bc2_sqrt_inv;
  float lr[kMaxHeads], step_size[kMaxHeads], decay[kMaxHeads], wd[kMaxHeads];
  // adapter heads (uml_sweep_adapter_run): image row r of head k is zrows[k * z_stride + r * z_ld] (the adapter output Z)
  // instead of a bank row; labels still come through the permutation.  NULL: bank rows.
  const float* zrows;
  int64_t z_ld, z_stride;
  // learnable temperatures: [K][2] (image, text) parameters and optimizer state; NULL: the fixed scale[]
  float* scale_dev;
  float* scale_m;
  float* scale_v;
  float* row_dscale;  // [K][row_stride] per-row d loss / d scale, written by the fused softmax epilogue
};

__device__ __forceinline__ bool head_active(const SweepDev& p, int head) { return (p.active_mask >> head) & 1u; }
__device__ __forceinline__ float seg_scale(const SweepDev& p, int head, bool is_txt) {
  return p.scale_dev ? p.scale_dev[2 * head + (is_txt ? 1 : 0)] : p.scale[is_txt ? 1 : 0];
}

// bank row and bank label of logical row r (image run first, then the text run) of head `head`
__device__ __forceinline__ int64_t bank_row(const SweepDev& p, int head, int64_t r, bool& is_txt) {
  is_txt = r >= p.n0;
  const int64_t l = is_txt ? r - p.n0 : r;
  const int64_t* pm = is_txt ? p.perm[1][head] : p.perm[0][head];
  return pm[(is_txt ? p.pos[1] : p.pos[0]) + l];
}
__device__ __forceinline__ const float* row_ptr(const SweepDev& p, int head, int64_t r) {
  if (p.zrows != nullptr && r < p.n0) return p.zrows + head * p.z_stride + r * p.z_ld;
  bool s;
  const int64_t src = bank_row(p, head, r, s);
  return (s ? p.bank[1] : p.bank[0]) + src * (s ? p.ld[1] : p.ld[0]);
}

__device__ __forceinline__ float block_max(float v, float* sh) {
  v = warp_max(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = sh[0];
  for (int w = 1; w < (blockDim.x >> 5); ++w) r = fmaxf(r, sh[w]);
  __syncthreads();
  return r;
}
__device__ __forceinline__ float block_sum(float v, float* sh) {
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int w = 0; w < (blockDim.x >> 5); ++w) r += sh[w];
  __syncthreads();
  return r;
}


// 16-byte asynchronous global -> shared copy (LDGSTS); `valid` false zero-fills the destination without reading
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  const int bytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// 1. raw logits  G_k = [X_img ; X_txt]_k W_k^T     grid (ceil(C/64), ceil(rows/64), K)
//    64 x 64 tile, 4 x 4 per thread.  Both operands are k-contiguous in HBM (bank rows, weight rows) and stay that way
//    in shared memory, so staging is a straight 16-byte copy; a thread owns rows ty + 16 i and classes tx + 16 j, which
//    makes the float4 reads along k conflict-free (quarter-warp lanes are 68 floats apart) and the stores coalesced.
//    Per element the sum still runs over k in ascending order with one FFMA per term.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sweep_logits_kernel(const __grid_constant__ SweepDev p) {
  constexpr int BM = 64, BN = 64, kBK = 64, LD = kBK + 4, TM = 4, TN = 4;
  const int head = blockIdx.z;
  if (!head_active(p, head)) return;
  __shared__ __align__(16) float As[BM][LD];
  __shared__ __align__(16) float Bs[BN][LD];
  __shared__ const float* rowp[BM];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t R = p.n0 + p.n1;
  const int64_t m0 = static_cast<int64_t>(blockIdx.y) * BM;
  const int c0 = blockIdx.x * BN;
  const int D = p.dim, C = p.n_classes;
  if (t < BM) rowp[t] = (m0 + t < R) ? row_ptr(p, head, m0 + t) : nullptr;
  __syncthreads();
  const float* __restrict__ W = p.W + head * p.head_stride;
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < D; k0 += kBK) {
    if (p.vec_rows) {  // dim % 4 == 0 and 16-byte aligned rows: k < D implies k + 3 < D
#pragma unroll
      for (int f = t; f < BM * (kBK / 4); f += 256) {
        const int m = f / (kBK / 4), k = k0 + 4 * (f % (kBK / 4));
        const float* rp = rowp[m];
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rp != nullptr && k < D) x = *reinterpret_cast<const float4*>(rp + k);
        *reinterpret_cast<float4*>(&As[m][k - k0]) = x;
      }
#pragma unroll
      for (int f = t; f < BN * (kBK / 4); f += 256) {
        const int n = f / (kBK / 4), k = k0 + 4 * (f % (kBK / 4));
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c0 + n < C && k < D) x = *reinterpret_cast<const float4*>(W + static_cast<int64_t>(c0 + n) * D + k);
        *reinterpret_cast<float4*>(&Bs[n][k - k0]) = x;
      }
    } else {
#pragma unroll 4
      for (int e = t; e < BM * kBK; e += 256) {
        const int m = e / kBK, k = e % kBK;
        const float* rp = rowp[m];
        As[m][k] = (rp != nullptr && k0 + k < D) ? rp[k0 + k] : 0.f;
      }
#pragma unroll 4
      for (int e = t; e < BN * kBK; e += 256) {
        const int n = e / kBK, k = e % kBK;
        Bs[n][k] = (c0 + n < C && k0 + k < D) ? W[static_cast<int64_t>(c0 + n) * D + k0 + k] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll 4
    for (int k = 0; k < kBK; k += 4) {
      float4 a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = *reinterpret_cast<const float4*>(&As[ty + 16 * i][k]);
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = *reinterpret_cast<const float4*>(&Bs[tx + 16 * j][k]);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) {
          float c = acc[i][j];
          c = fmaf(a[i].x, b[j].x, c);
          c = fmaf(a[i].y, b[j].y, c);
          c = fmaf(a[i].z, b[j].z, c);
          c = fmaf(a[i].w, b[j].w, c);
          acc[i][j] = c;
        }
    }
    __syncthreads();
  }
  float* __restrict__ G = p.G + head * p.g_stride;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int64_t r = m0 + ty + 16 * i;
    if (r >= R) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int c = c0 + tx + 16 * j;
      if (c < C) G[r * p.ldg + c] = acc[i][j];
    }
  }
}

// The same tile with the k-tiles double-buffered through cp.async: the loads of tile i+1 are in flight while tile i is
// multiplied (the synchronous version above exposes one L2/HBM round trip per k-tile).  Needs 16-byte aligned rows
// (p.vec_rows); identical arithmetic, identical results.
constexpr int kLogitsLd = 68;
constexpr int kLogitsStageFloats = 2 * 64 * kLogitsLd;  // A tile + B tile
constexpr int kLogitsSmemBytes = 2 * kLogitsStageFloats * 4;

__global__ void __launch_bounds__(256) sweep_logits_async_kernel(const __grid_constant__ SweepDev p) {
  constexpr int BM = 64, BN = 64, kBK = 64, LD = kLogitsLd, TM = 4, TN = 4;
  const int head = blockIdx.z;
  if (!head_active(p, head)) return;
  extern __shared__ __align__(16) float dyn[];
  __shared__ const float* rowp[BM];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t R = p.n0 + p.n1;
  const int64_t m0 = static_cast<int64_t>(blockIdx.y) * BM;
  const int c0 = blockIdx.x * BN;
  const int D = p.dim, C = p.n_classes;
  const float* __restrict__ W = p.W + head * p.head_stride;
  if (t < BM) rowp[t] = (m0 + t < R) ? row_ptr(p, head, m0 + t) : nullptr;
  __syncthreads();

  auto load_stage = [&](int stage, int k0) {
    float* As = dyn + stage * kLogitsStageFloats;
    float* Bs = As + BM * LD;
#pragma unroll
    for (int f = t; f < BM * (kBK / 4); f += 256) {
      const int m = f / (kBK / 4), kk = 4 * (f % (kBK / 4));
      const float* rp = rowp[m];
      const bool ok = rp != nullptr && k0 + kk < D;
      cp_async16(As + m * LD + kk, ok ? rp + k0 + kk : W, ok);
    }
#pragma unroll
    for (int f = t; f < BN * (kBK / 4); f += 256) {
      const int n = f / (kBK / 4), kk = 4 * (f % (kBK / 4));
      const bool ok = c0 + n < C && k0 + kk < D;
      cp_async16(Bs + n * LD + kk, ok ? W + static_cast<int64_t>(c0 + n) * D + k0 + kk : W, ok);
    }
    cp_async_commit();
  };

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  const int nk = (D + kBK - 1) / kBK;
  load_stage(0, 0);
  for (int it = 0; it < nk; ++it) {
    if (it + 1 < nk) {
      load_stage((it + 1) & 1, (it + 1) * kBK);
      cp_async_wait<1>();  // everything but the newest group has landed: tile `it` is complete
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* As = dyn + (it & 1) * kLogitsStageFloats;
    const float* Bs = As + BM * LD;
#pragma unroll 4
    for (int k = 0; k < kBK; k += 4) {
      float4 a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = *reinterpret_cast<const float4*>(As + (ty + 16 * i) * LD + k);
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = *reinterpret_cast<const float4*>(Bs + (tx + 16 * j) * LD + k);
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) {
          float c = acc[i][j];
          c = fmaf(a[i].x, b[j].x, c);
          c = fmaf(a[i].y, b[j].y, c);
          c = fmaf(a[i].z, b[j].z, c);
          c = fmaf(a[i].w, b[j].w, c);
          acc[i][j] = c;
        }
    }
    __syncthreads();  // the next iteration's loads overwrite this buffer's sibling only after everyone is done with it
  }
  float* __restrict__ G = p.G + head * p.g_stride;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int64_t r = m0 + ty + 16 * i;
    if (r >= R) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      const int c = c0 + tx + 16 * j;
      if (c < C) G[r * p.ldg + c] = acc[i][j];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// 2. per-row softmax / CE / argmax; the raw logits row becomes G = w s / n (softmax - onehot)   grid (rows, K)
//    (F.cross_entropy x2 and the weighted sum, finetune.py:186-188; same arithmetic as simt.cu's row kernel)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sweep_softmax_kernel(const __grid_constant__ SweepDev p) {
  const int head = blockIdx.y;
  if (!head_active(p, head)) return;
  __shared__ float sh[8];
  __shared__ int sh_arg;
  const int64_t r = blockIdx.x;
  const int C = p.n_classes;
  bool s;
  const int64_t src = bank_row(p, head, r, s);
  const int label = static_cast<int>((s ? p.labels[1] : p.labels[0])[src]);
  const int64_t n_seg = s ? p.n1 : p.n0;
  const float scale = s ? p.scale[1] : p.scale[0];
  const float weight = s ? p.alpha[head] : 1.f;
  float* row = p.G + head * p.g_stride + r * p.ldg;
  const float label_raw = row[label];  // read before the row is overwritten with G

  float mx = -INFINITY;
  int arg = INT_MAX;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float x = row[c] * scale;
    if (x > mx) { mx = x; arg = c; }
  }
  if (threadIdx.x == 0) sh_arg = INT_MAX;
  const float bmax = block_max(mx, sh);  // its barriers publish sh_arg
  if (mx == bmax) atomicMin(&sh_arg, arg);  // first maximal index, like torch.argmax
  float se = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) se += expf(row[c] * scale - bmax);
  const float sum = block_sum(se, sh);
  const float inv = 1.f / sum;
  const float gcoef = weight * scale / static_cast<float>(n_seg);
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float pr = expf(row[c] * scale - bmax) * inv;
    if (c == label) pr -= 1.f;
    row[c] = pr * gcoef;
  }
  __syncthreads();  // sh_arg complete (every atomicMin precedes this barrier)
  if (threadIdx.x == 0) {
    p.row_loss[head * p.row_stride + r] = logf(sum) - (label_raw * scale - bmax);
    p.row_correct[head * p.row_stride + r] = (sh_arg == label) ? 1 : 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// 3. dW_k = G_k^T [X_img ; X_txt]_k with the optimizer update in the epilogue   grid (ceil(D/64), ceil(C/64), K)
//    (autograd of the head + torch.optim.AdamW / Adam / SGD, finetune.py:190-195, optim.py:42-70)
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void update_one(const SweepDev& p, float lr, float step_size, float decay, float wd, float& w,
                                           float& m, float& v, float g) {
  if (p.kind == 3) {  // SGD momentum, L2 decay folded into the gradient
    g = fmaf(wd, w, g);
    const float b = p.first_step ? g : fmaf(p.momentum, m, g);
    m = b;
    w = w - lr * b;
    return;
  }
  if (p.kind == 1) w *= decay;             // AdamW: decoupled decay
  else if (wd != 0.f) g = fmaf(wd, w, g);  // Adam: L2
  m = m + (g - m) * (1.f - p.beta1);
  v = v * p.beta2 + (1.f - p.beta2) * g * g;
  const float denom = sqrtf(v) * p.bc2_sqrt_inv + p.eps;
  w = w - step_size * (m / denom);
}

__global__ void __launch_bounds__(256) sweep_dw_update_kernel(const __grid_constant__ SweepDev p) {
  constexpr int BM = 64, BN = 64, kBK = 32, TM = 4, TN = 4;
  const int head = blockIdx.z;
  if (!head_active(p, head)) return;
  __shared__ __align__(16) float As[kBK][BM + 4];  // G tile   [row][class]
  __shared__ __align__(16) float Bs[kBK][BN + 4];  // X tile   [row][dim]
  __shared__ const float* rowp[kBK];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t R = p.n0 + p.n1;
  const int c0 = blockIdx.y * BM, d0 = blockIdx.x * BN;
  const int D = p.dim, C = p.n_classes;
  const float* __restrict__ G = p.G + head * p.g_stride;
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int64_t r0 = 0; r0 < R; r0 += kBK) {
    if (t < kBK) rowp[t] = (r0 + t < R) ? row_ptr(p, head, r0 + t) : nullptr;
    __syncthreads();
#pragma unroll
    for (int e = t; e < BM * kBK; e += 256) {
      const int k = e / BM, m = e % BM;
      As[k][m] = (r0 + k < R && c0 + m < C) ? G[(r0 + k) * p.ldg + c0 + m] : 0.f;
    }
#pragma unroll
    for (int e = t; e < BN * kBK; e += 256) {
      const int k = e / BN, n = e % BN;
      const float* rp = rowp[k];
      Bs[k][n] = (rp != nullptr && d0 + n < D) ? rp[d0 + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kBK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * TM]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * TN]);
      const float a[TM] = {a4.x, a4.y, a4.z, a4.w}, b[TN] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }

  const float lr = p.lr[head], step_size = p.step_size[head], decay = p.decay[head], wd = p.wd[head];
  float* __restrict__ W = p.W + head * p.head_stride;
  float* __restrict__ Mo = p.m + head * p.head_stride;
  float* __restrict__ Vo = p.kind == 3 ? nullptr : p.v + head * p.head_stride;
  const int d = d0 + tx * TN;
  const bool vec = (D % 4 == 0) && (d + TN <= D);  // slabs are 16-byte aligned (checked by the launcher)
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int c = c0 + ty * TM + i;
    if (c >= C) continue;
    const int64_t off = static_cast<int64_t>(c) * D + d;
    if (vec) {
      float4 w4 = *reinterpret_cast<const float4*>(W + off);
      float4 m4 = *reinterpret_cast<const float4*>(Mo + off);
      float4 v4 = Vo ? *reinterpret_cast<const float4*>(Vo + off) : make_float4(0.f, 0.f, 0.f, 0.f);
      update_one(p, lr, step_size, decay, wd, w4.x, m4.x, v4.x, acc[i][0]);
      update_one(p, lr, step_size, decay, wd, w4.y, m4.y, v4.y, acc[i][1]);
      update_one(p, lr, step_size, decay, wd, w4.z, m4.z, v4.z, acc[i][2]);
      update_one(p, lr, step_size, decay, wd, w4.w, m4.w, v4.w, acc[i][3]);
      *reinterpret_cast<float4*>(W + off) = w4;
      *reinterpret_cast<float4*>(Mo + off) = m4;
      if (Vo) *reinterpret_cast<float4*>(Vo + off) = v4;
    } else {
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        if (d + j >= D) continue;
        float w = W[off + j], mm = Mo[off + j], vv = Vo ? Vo[off + j] : 0.f;
        update_one(p, lr, step_size, decay, wd, w, mm, vv, acc[i][j]);
        W[off + j] = w;
        Mo[off + j] = mm;
        if (Vo) Vo[off + j] = vv;
      }
    }
  }
}

// The same launch with every memory request of a CTA issued up front: the G and feature tiles of ALL rows of the step
// go to shared memory through cp.async while the weights and optimizer state the thread will update are already on
// their way to registers; one wait, then the contraction, the update and the stores.  (The synchronous version pays a
// load -> barrier -> multiply round per 32 rows and only then asks for W, m, v.)  Needs 16-byte aligned rows and
// ldg % 4 == 0; identical arithmetic, identical results.
__global__ void __launch_bounds__(256, 2) sweep_dw_update_async_kernel(const __grid_constant__ SweepDev p) {
  constexpr int BM = 64, BN = 64, kR = 64, LD = 68, TM = 4, TN = 4;
  const int head = blockIdx.z;
  if (!head_active(p, head)) return;
  __shared__ __align__(16) float As[kR][LD];  // G tile   [row][class]
  __shared__ __align__(16) float Bs[kR][LD];  // X tile   [row][dim]
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t R = p.n0 + p.n1;
  const int c0 = blockIdx.y * BM, d0 = blockIdx.x * BN;
  const int D = p.dim, C = p.n_classes;
  const float* __restrict__ G = p.G + head * p.g_stride;
  float* __restrict__ W = p.W + head * p.head_stride;
  float* __restrict__ Mo = p.m + head * p.head_stride;
  float* __restrict__ Vo = p.kind == 3 ? nullptr : p.v + head * p.head_stride;
  const int d = d0 + tx * TN;
  const bool live = d < D;  // D % 4 == 0: d < D implies d + 4 <= D

  auto load_rows = [&](int64_t r0) {
#pragma unroll
    for (int f = t; f < kR * (BM / 4); f += 256) {
      const int k = f / (BM / 4), q = 4 * (f % (BM / 4));
      const bool ok = r0 + k < R && c0 + q < C;  // ldg % 4 == 0 and ldg >= C: the 16 bytes stay inside the row
      cp_async16(&As[k][q], ok ? G + (r0 + k) * p.ldg + c0 + q : G, ok);
    }
#pragma unroll
    for (int f = t; f < kR * (BN / 4); f += 256) {
      const int k = f / (BN / 4), q = 4 * (f % (BN / 4));
      const bool ok = r0 + k < R && d0 + q < D;
      cp_async16(&Bs[k][q], ok ? row_ptr(p, head, r0 + k) + d0 + q : G, ok);
    }
    cp_async_commit();
  };

  load_rows(0);
  float4 w4[TM], m4[TM], v4[TM];
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int c = c0 + ty * TM + i;
    w4[i] = m4[i] = v4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live && c < C) {
      const int64_t off = static_cast<int64_t>(c) * D + d;
      w4[i] = *reinterpret_cast<const float4*>(W + off);
      m4[i] = *reinterpret_cast<const float4*>(Mo + off);
      if (Vo) v4[i] = *reinterpret_cast<const float4*>(Vo + off);
    }
  }
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  for (int64_t r0 = 0; r0 < R; r0 += kR) {
    if (r0 > 0) {
      __syncthreads();  // everyone is done with the previous rows
      load_rows(r0);
    }
    cp_async_wait<0>();
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < kR; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * TM]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * TN]);
      const float a[TM] = {a4.x, a4.y, a4.z, a4.w}, b[TN] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
  }

  if (!live) return;
  const float lr = p.lr[head], step_size = p.step_size[head], decay = p.decay[head], wd = p.wd[head];
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int c = c0 + ty * TM + i;
    if (c >= C) continue;
    const int64_t off = static_cast<int64_t>(c) * D + d;
    update_one(p, lr, step_size, decay, wd, w4[i].x, m4[i].x, v4[i].x, acc[i][0]);
    update_one(p, lr, step_size, decay, wd, w4[i].y, m4[i].y, v4[i].y, acc[i][1]);
    update_one(p, lr, step_size, decay, wd, w4[i].z, m4[i].z, v4[i].z, acc[i][2]);
    update_one(p, lr, step_size, decay, wd, w4[i].w, m4[i].w, v4[i].w, acc[i][3]);
    *reinterpret_cast<float4*>(W + off) = w4[i];
    *reinterpret_cast<float4*>(Mo + off) = m4[i];
    if (Vo) *reinterpret_cast<float4*>(Vo + off) = v4[i];
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Tensor-core forms of the two contractions (tcgen05.mma kind::tf32, fp32 accumulators in TMEM) - the default when rows
// are 16-byte aligned.  The exact path has to stay at fp32 accuracy (the sweep tests hold every head to the oracle's
// fp32 trajectory), so each operand is split in shared memory into two tf32 terms,
//     x = hi + lo,   hi = x with the 13 low mantissa bits cleared (exactly what the tf32 datapath reads),
//                    lo = x - hi (exact in fp32; its own 13 significant bits lose at most two to tf32),
// and a product is accumulated as  hi*hi + hi*lo + lo*hi  ("3xTF32": relative error 2^-21 per term against 2^-24 for an
// FFMA, accumulated in fp32).  Three MMAs per k-step still leave the tensor pipe two orders of magnitude ahead of the
// FFMA loops above; what remains is the operand stream (logits) and the 24 B/parameter of the update (dW).
// Operands reach shared memory through registers (logits: the split needs them there anyway) or cp.async (dW) in the
// 128-byte swizzled layouts the MMA descriptors name, bank rows gathered by index on the way; no tensor maps.
// The order of accumulation is fixed by the instruction stream, so a head's result does not depend on its slot.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// instruction descriptor: fp32 accumulator, tf32 A and B
__host__ __device__ constexpr uint32_t make_idesc_tf32(uint32_t m, uint32_t n, uint32_t a_mn_major, uint32_t b_mn_major) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (a_mn_major << 15) | (b_mn_major << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// mbarrier wait that cannot hang the GPU: a barrier that does not flip within ~10 s (a bug, never load) traps
__device__ __forceinline__ void mbar_wait_or_trap(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  const long long t0 = clock64();
  for (;;) {
    uint32_t done;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
    if (clock64() - t0 > 20000000000ll) __trap();
  }
}
__device__ __forceinline__ void split_tf32(const float4& x, float4& hi, float4& lo) {
  hi.x = __uint_as_float(__float_as_uint(x.x) & 0xffffe000u);
  hi.y = __uint_as_float(__float_as_uint(x.y) & 0xffffe000u);
  hi.z = __uint_as_float(__float_as_uint(x.z) & 0xffffe000u);
  hi.w = __uint_as_float(__float_as_uint(x.w) & 0xffffe000u);
  lo.x = x.x - hi.x;
  lo.y = x.y - hi.y;
  lo.z = x.z - hi.z;
  lo.w = x.w - hi.w;
}
// byte offset of 16-byte chunk `ch` of 128-byte row `row` inside a SWIZZLE_128B box (rows 128 B apart, 8-row atoms)
__device__ __forceinline__ uint32_t sw128(int row, int ch) { return static_cast<uint32_t>(row * 128 + ((ch ^ (row & 7)) << 4)); }

// 1t. raw logits, transposed tile: D[class, row] = W_k[128 classes, :] . X_k[64 rows, :]^T   grid (ceil(C/128), ceil(rows/64), K)
//     A = weight rows (K-major), B = gathered bank rows (K-major), k-blocks of 32 floats (one swizzle row), two stages:
//     the loads of block kb + 1 are in registers while block kb is split, stored and multiplied (8 MMAs per block: see
//     idesc2 below).
//     (Measured alternatives, 30 heads of 1000 x 512, against 37 us for this form - two CTAs per SM, every tile of the
//     launch resident at once: register buffers two blocks ahead 38 us; a five-stage cp.async ring three blocks ahead, one
//     CTA per SM, 47 us, with the weight tile asked into L2 up front 51 us; a TMA warp for the weight boxes with four
//     row-loader warps 51 us, with one 128-byte bulk copy per row instead 88 us.  None of it is a load-latency problem:
//     a k-block moves 48 KB of split stores, 24 KB of loads and 72 KB of operand reads for its 12 MMAs through shared
//     memory - about 0.6 us of its bandwidth, 15 us for the launch - and the rest is the split -> fence.proxy.async ->
//     barrier -> issue chain of each block, which only more resident CTAs hide.)
constexpr int kTcLgStage = 48 * 1024;  // W hi 16 KB | W lo 16 KB | X hi 8 KB | X lo 8 KB
constexpr int kTcLgSmemBytes = 2 * kTcLgStage + 1024 + 64;

// kSoftmax: the (up to eight) class tiles of a head form a thread-block cluster and finish the rows together - softmax / CE /
// argmax in the epilogue, the row maxima and sums exchanged through distributed shared memory - so G leaves the kernel
// final and the softmax launch (one read and one write of the logits) disappears.
__device__ __forceinline__ float ld_cluster_f32(uint32_t cluster_addr) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr) : "memory");
  return v;
}
template <bool kSoftmax>
__global__ void __launch_bounds__(256, 2) sweep_logits_tc_kernel(const __grid_constant__ SweepDev p) {
  constexpr int BM = 128, BN = 64, BK = 32, S = 2;
  const int head = blockIdx.z;
  if (!head_active(p, head)) return;
  extern __shared__ unsigned char tc_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* empty_bar = reinterpret_cast<uint64_t*>(smem + S * kTcLgStage);
  uint64_t* tfull_bar = empty_bar + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull_bar + 1);
  __shared__ const float* rowp[BN];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int64_t R = p.n0 + p.n1;
  const int64_t m0 = static_cast<int64_t>(blockIdx.y) * BN;
  const int c0 = blockIdx.x * BM;
  const int D = p.dim, C = p.n_classes;
  const float* __restrict__ W = p.W + head * p.head_stride;
  if (t < BN) rowp[t] = (m0 + t < R) ? row_ptr(p, head, m0 + t) : nullptr;
  if (t == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&empty_bar[s], 1);
    mbar_init(tfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // this thread's 16-byte chunks of a k-block: four of the weight tile, two of the row tile (eight threads per row)
  const int ch = t & 7;
  const float* wsrc[4];
  const float* xsrc[2];
  uint32_t woff[4], xoff[2];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int row = (t >> 3) + 32 * i;
    wsrc[i] = (c0 + row < C) ? W + static_cast<int64_t>(c0 + row) * D + ch * 4 : nullptr;
    woff[i] = sw128(row, ch);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int row = (t >> 3) + 32 * i;
    const float* rp = rowp[row];
    xsrc[i] = rp ? rp + ch * 4 : nullptr;
    xoff[i] = sw128(row, ch);
  }
  auto load = [&](int kb, float4 (&r)[6]) {
    const bool kin = kb * BK + ch * 4 < D;  // dim % 4 == 0: a chunk is inside the row or outside, never across its end
#pragma unroll
    for (int i = 0; i < 4; ++i)
      r[i] = (kin && wsrc[i]) ? __ldg(reinterpret_cast<const float4*>(wsrc[i] + kb * BK)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 2; ++i)
      r[4 + i] = (kin && xsrc[i]) ? __ldg(reinterpret_cast<const float4*>(xsrc[i] + kb * BK)) : make_float4(0.f, 0.f, 0.f, 0.f);
  };

  const int nk = (D + BK - 1) / BK;
  // The row tile's hi and lo terms lie back to back (64 + 64 rows of one K-major tile), so  W_hi . [X_hi | X_lo]^T  is ONE
  // MMA with N = 128 whose halves land in TMEM columns [0, 64) and [64, 128); W_lo . X_hi^T adds to the first half and the
  // epilogue adds the halves: 8 MMAs and 56 KB of operand reads per k-block instead of 12 and 72 KB.
  constexpr uint32_t idesc = make_idesc_tf32(BM, BN, 0, 0), idesc2 = make_idesc_tf32(BM, 2 * BN, 0, 0);
  float4 cur[6], nxt[6];
  load(0, cur);
#pragma unroll 1
  for (int kb = 0; kb < nk; ++kb) {
    if (kb + 1 < nk) load(kb + 1, nxt);
    const int s = kb & (S - 1);
    if (kb >= S) mbar_wait_or_trap(&empty_bar[s], static_cast<uint32_t>((kb / S) - 1) & 1u);  // the MMAs of block kb - S have read it
    unsigned char* st = smem + s * kTcLgStage;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float4 hi, lo;
      split_tf32(cur[i], hi, lo);
      *reinterpret_cast<float4*>(st + woff[i]) = hi;
      *reinterpret_cast<float4*>(st + 16384 + woff[i]) = lo;
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      float4 hi, lo;
      split_tf32(cur[4 + i], hi, lo);
      *reinterpret_cast<float4*>(st + 32768 + xoff[i]) = hi;
      *reinterpret_cast<float4*>(st + 40960 + xoff[i]) = lo;
    }
    fence_proxy_async();  // generic-proxy stores -> the tensor core's async-proxy reads
    __syncthreads();
    if (t == 0) {
      tc_fence_after();
      const uint32_t a_hi = smem_u32(st), a_lo = a_hi + 16384, b_hi = a_hi + 32768;
#pragma unroll
      for (int k = 0; k < BK / 8; ++k) {  // a k-step of 8 floats = 32 B inside the swizzle row; 8-row atoms 1024 B apart
        const uint64_t dah = make_smem_desc(a_hi + k * 32, 16, 1024, kLayoutSw128);
        const uint64_t dal = make_smem_desc(a_lo + k * 32, 16, 1024, kLayoutSw128);
        const uint64_t dbh = make_smem_desc(b_hi + k * 32, 16, 1024, kLayoutSw128);  // (b_lo = b_hi + 8 KB: rows 64 .. 127)
        umma_tf32(tmem_base, dah, dbh, idesc2, (kb | k) != 0);
        umma_tf32(tmem_base, dal, dbh, idesc, 1);
      }
      umma_commit(&empty_bar[s]);
      if (kb == nk - 1) umma_commit(tfull_bar);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) cur[i] = nxt[i];
  }

  // epilogue: TMEM lane = class, column = row; warp w reads lane quadrant w % 4, column half w / 4
  mbar_wait_or_trap(tfull_bar, 0);
  tc_fence_after();
  const int q = warp & 3, h = warp >> 2;
  uint32_t v[32];
  {
    uint32_t v2[32];
    tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + h * 32, v);
    tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + BN + h * 32, v2);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(v2[i]));
  }
  float* __restrict__ G = p.G + head * p.g_stride;
  if (!kSoftmax) {
    const int c = c0 + q * 32 + lane;
    if (c < C) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int64_t r = m0 + h * 32 + i;
        if (r < R) G[r * p.ldg + c] = __uint_as_float(v[i]);  // a warp stores 32 consecutive classes of one row
      }
    }
  } else {
    // The tile goes to shared memory as [row][class] (the operand stages are free: every MMA has completed), then a warp
    // owns eight rows: lane = four consecutive classes.  Arithmetic per element as in sweep_softmax_kernel; the sum of a
    // row is per lane, then a shuffle tree, then the tiles in class order.
    __shared__ float pub_max[BN], pub_sum[BN];  // published to the cluster: tile maximum, tile sum of exponentials
    __shared__ int pub_arg[BN];                 //                            first maximal class of the tile
    __shared__ float row_scale[BN], row_gcoef[BN], row_lab[BN];
    __shared__ int row_label[BN], row_arg[BN];
    __shared__ float row_weight[BN], row_n[BN], pub_ds[BN];  // learnable temperatures: d loss / d scale of the row
    float* tile = reinterpret_cast<float*>(smem);  // [BN][BM]
    float* raw_tile = tile + BN * BM;               // [BN][BM] unscaled logits (learnable temperatures only)
    const bool want_ds = p.scale_dev != nullptr;
    if (t < BN) {
      const int64_t r = m0 + t;
      row_label[t] = -1;
      row_scale[t] = 1.f;
      row_gcoef[t] = 0.f;
      if (r < R) {
        bool is_txt;
        const int64_t src = bank_row(p, head, r, is_txt);
        row_label[t] = static_cast<int>((is_txt ? p.labels[1] : p.labels[0])[src]);
        const float sc = seg_scale(p, head, is_txt);
        const float w = is_txt ? p.alpha[head] : 1.f;
        row_scale[t] = sc;
        row_gcoef[t] = w * sc / static_cast<float>(is_txt ? p.n1 : p.n0);
        row_weight[t] = w;
        row_n[t] = static_cast<float>(is_txt ? p.n1 : p.n0);
      }
    }
    __syncthreads();
    {
      const int cl = q * 32 + lane;
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const int rl = h * 32 + i;
        tile[rl * BM + cl] = (c0 + cl < C) ? __uint_as_float(v[i]) * row_scale[rl] : -INFINITY;
        if (want_ds) raw_tile[rl * BM + cl] = (c0 + cl < C) ? __uint_as_float(v[i]) : 0.f;
      }
    }
    __syncthreads();
    const uint32_t n_tiles = gridDim.x;  // (cluster = the head's class tiles: rank == blockIdx.x)
    // ---- tile maximum and first maximal class of every row ----
    for (int rl = warp * 8; rl < warp * 8 + 8; ++rl) {
      const float4 x4 = *reinterpret_cast<const float4*>(tile + rl * BM + 4 * lane);
      float mx = x4.x;
      int arg = 0;
      if (x4.y > mx) { mx = x4.y; arg = 1; }
      if (x4.z > mx) { mx = x4.z; arg = 2; }
      if (x4.w > mx) { mx = x4.w; arg = 3; }
      arg += c0 + 4 * lane;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, mx, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (om > mx || (om == mx && oa < arg)) { mx = om; arg = oa; }
      }
      if (lane == 0) {
        pub_max[rl] = mx;
        pub_arg[rl] = arg;
      }
    }
    cluster_sync_all();
    // ---- row maximum over the tiles (lower class wins a tie: first maximal index, like torch.argmax), exponentials ----
    // A lane fetches the published values of ONE tile for two of the warp's eight rows (rows rs and rs + 4 of the group,
    // tile = lane & 7): the remote loads are independent, and the eight tiles of a row meet by three shuffles.  (Every
    // lane walking the eight tiles of a row in turn cost a remote round trip per tile and row: 15 us per launch.)
    const uint32_t tl = lane & 7, rs = lane >> 3;
    float gm[2];
    int ga[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int rl = warp * 8 + rs + 4 * k;
      gm[k] = -INFINITY;
      ga[k] = INT_MAX;
      if (tl < n_tiles) {
        gm[k] = ld_cluster_f32(mapa_cta(smem_u32(&pub_max[rl]), tl));
        ga[k] = __float_as_int(ld_cluster_f32(mapa_cta(smem_u32(&pub_arg[rl]), tl)));
      }
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) {
        const float om = __shfl_xor_sync(0xffffffffu, gm[k], o);
        const int oa = __shfl_xor_sync(0xffffffffu, ga[k], o);
        if (om > gm[k] || (om == gm[k] && oa < ga[k])) { gm[k] = om; ga[k] = oa; }
      }
    }
    for (int i = 0; i < 8; ++i) {
      const int rl = warp * 8 + i;
      const float bmax = __shfl_sync(0xffffffffu, (i >> 2) ? gm[1] : gm[0], (i & 3) * 8);
      const int barg = __shfl_sync(0xffffffffu, (i >> 2) ? ga[1] : ga[0], (i & 3) * 8);
      float4 x4 = *reinterpret_cast<const float4*>(tile + rl * BM + 4 * lane);
      {  // the lane that holds the label's class keeps x_label - max for the loss (exact 0 for a dominant label)
        const int lk = row_label[rl] - (c0 + 4 * lane);
        if (lk >= 0 && lk < 4) row_lab[rl] = (lk == 0 ? x4.x : lk == 1 ? x4.y : lk == 2 ? x4.z : x4.w) - bmax;
      }
      x4.x = expf(x4.x - bmax);
      x4.y = expf(x4.y - bmax);
      x4.z = expf(x4.z - bmax);
      x4.w = expf(x4.w - bmax);
      *reinterpret_cast<float4*>(tile + rl * BM + 4 * lane) = x4;
      const float se = warp_sum((x4.x + x4.y) + (x4.z + x4.w));
      if (lane == 0) {
        pub_sum[rl] = se;
        row_arg[rl] = barg;
      }
    }
    cluster_sync_all();
    // ---- row sum over the tiles (fixed shuffle tree over the tile index), G, loss and hit ----
    float gsum[2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int rl = warp * 8 + rs + 4 * k;
      gsum[k] = tl < n_tiles ? ld_cluster_f32(mapa_cta(smem_u32(&pub_sum[rl]), tl)) : 0.f;
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
#pragma unroll
      for (int o = 4; o > 0; o >>= 1) gsum[k] += __shfl_xor_sync(0xffffffffu, gsum[k], o);
    }
    for (int i = 0; i < 8; ++i) {
      const int rl = warp * 8 + i;
      const float sum = __shfl_sync(0xffffffffu, (i >> 2) ? gsum[1] : gsum[0], (i & 3) * 8);
      const int64_t r = m0 + rl;
      if (r >= R) continue;  // (warp-uniform)
      const float inv = 1.f / sum, gcoef = row_gcoef[rl];
      const int label = row_label[rl];
      const float4 e4 = *reinterpret_cast<const float4*>(tile + rl * BM + 4 * lane);
      float pr[4] = {e4.x * inv, e4.y * inv, e4.z * inv, e4.w * inv};
      const int cb = c0 + 4 * lane;
      float ds = 0.f;
      if (want_ds) {  // softmax_ce_grad_row's  sum_c (p_c - y_c) raw_c  (simt.cu), tile part: lanes in a shuffle tree
        const float4 r4 = *reinterpret_cast<const float4*>(raw_tile + rl * BM + 4 * lane);
        const float raw[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) ds = fmaf(pr[k] - (cb + k == label ? 1.f : 0.f), raw[k], ds);
        ds = warp_sum(ds);
        if (lane == 0) pub_ds[rl] = ds;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (cb + k == label) pr[k] -= 1.f;
        pr[k] *= gcoef;
      }
      float* grow = G + r * p.ldg + cb;
      if (cb + 3 < C) {
        *reinterpret_cast<float4*>(grow) = make_float4(pr[0], pr[1], pr[2], pr[3]);  // (ldg % 4 == 0, G 16-byte aligned)
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (cb + k < C) grow[k] = pr[k];
      }
      // the lane that holds the label's class writes the row's loss (log_softmax form) and hit flag
      if (label >= cb && label < cb + 4) {
        p.row_loss[head * p.row_stride + r] = logf(sum) - row_lab[rl];
        p.row_correct[head * p.row_stride + r] = (row_arg[rl] == label) ? 1 : 0;
      }
    }
    if (want_ds) {  // the row's tiles in class order, by the first tile of the cluster
      cluster_sync_all();
      const int rl = warp * 8 + (lane & 7);
      if (blockIdx.x == 0 && lane < 8 && m0 + rl < R) {
        float s = 0.f;
        for (uint32_t k = 0; k < n_tiles; ++k) s += ld_cluster_f32(mapa_cta(smem_u32(&pub_ds[rl]), k));
        p.row_dscale[head * p.row_stride + m0 + rl] = s * row_weight[rl] / row_n[rl];
      }
    }
    cluster_sync_all();  // nobody leaves while a neighbour may still read its published values
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 128);
}

// 3t. dW^T strip with the optimizer update: D[dim, class] = X_k[rows, 128 dims]^T . G_k[rows, 64 classes] for up to four
//     consecutive 64-class tiles of one head            grid (ceil(D/128), ceil(C/256), K), steps of at most 64 rows
//     Both operands are stored rows-by-something, i.e. MN-major for this product; 32-bit MN-major operands take the
//     SWIZZLE_128B_BASE32B layout (128-byte rows of 32 floats, the four 32-byte units of a row permuted by row & 3,
//     4-row atoms 512 B apart; the next 32 dims / classes one 8 KB box further).  The feature tile is loaded and split
//     once per CTA; the accumulators alternate between two TMEM regions, so the MMAs of tile j + 1 are issued before
//     tile j is read back.
//     The launch is bound by the 24 B/parameter of the update, and what a thread can hold in registers is not enough
//     to keep HBM busy (a register-staged epilogue ran at 0.3 of the copy peak): W, m and v stream through a ring of
//     shared-memory slots instead - TMA loads of [16 classes x 128 dims] boxes three slots ahead, the update in place
//     (TMEM lane = dim, column = class: a warp touches 32 consecutive floats of a slot row), TMA stores behind - so the
//     bytes in flight are bounded by shared memory, not by the register file.  Boxes that overhang the head's C x D
//     slab are clipped by the tensor map on both ways, so the epilogue carries no predicates.
#ifndef UML_DW_SLOTS
#define UML_DW_SLOTS 5  // measured, 30 heads of 1000 x 512: 82 us with 4 slots, 76 us with 5 (0.76 of the HBM copy peak)
#endif
constexpr int kTcDwSlots = UML_DW_SLOTS;
constexpr int kTcDwSlotBytes = 3 * 8192;  // W | m | v boxes of 16 classes x 128 dims
constexpr int kTcDwSmemBytes = 96 * 1024 + kTcDwSlots * kTcDwSlotBytes + 1024 + 128;  // X hi | X lo (32 KB each) | G hi | G lo (16 KB each) | slots
constexpr uint32_t kLayoutSw128Base32 = 1;  // UMMA::LayoutType::SWIZZLE_128B_BASE32B

__device__ __forceinline__ uint32_t sw128_b32(int row, int ch) {
  return static_cast<uint32_t>(row * 128 + ((((ch >> 1) ^ (row & 3)) << 5) | ((ch & 1) << 4)));
}
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, uint32_t (&v)[2]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(v[0]), "=r"(v[1]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ldn(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}

// kNT update threads per CTA plus one TMA warp and one statistics warp.  The update costs ~50 instructions per parameter (IEEE sqrt and division),
// so the read-back needs warps to hide its dependency chains as much as it needs bytes in flight (8 warps per SM left the
// slots waiting for arithmetic), and nothing in it may wait for anything but its own data: an update warp waits for a
// slot's loads, updates its share in place and arrives on the slot's `done` barrier; the TMA warp waits for that
// barrier, stores the slot and refills the one before it - no CTA-wide barrier per slot.
// Persistent: the (head, 128-dim tile, 64-class tile) units of all running heads are dealt out in equal contiguous
// ranges to one CTA per SM (no tail wave; the feature tile changes at most twice per CTA), the next unit's tiles are
// requested at the start of a unit's read-back and split / multiplied one slot later, and the W / m / v ring runs
// across unit boundaries.
struct DwUnit {
  int unit;     // position in the CTA-independent unit order: running head (ascending), dim tile, class tile
  int st, nst;  // stage (16 classes) inside the unit, stages of the unit
  int head, dt, ct;
};
__device__ __forceinline__ float lds_f32(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }

// Operand staging of the X^T . G contractions (the dW kernel below and sweep_grad_diag_tc_kernel): 64 rows are the K
// dimension, both tiles MN-major in SWIZZLE_128B_BASE32B boxes of 32 columns x 64 rows (8 KB).  Feature tile: rowp[64]
// rows x 128 dims from d0 (four boxes, a warp per row); G tile: `rows` rows x 64 classes from c0 (two boxes).  Missing
// rows and dims are zero-filled.  The tf32 split writes hi in place and lo one tile further (X: +32 KB, G: +16 KB).
template <int kWarps>
__device__ __forceinline__ void x_tile_issue(unsigned char* xs, const float* const* rowp, int d0, int D, const void* dummy) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 64 / kWarps; ++i) {
    const int row = warp + kWarps * i, box = lane >> 3;
    const float* rp = rowp[row];
    const bool ok = rp != nullptr && d0 + lane * 4 < D;
    cp_async16(xs + box * 8192 + sw128_b32(row, lane & 7), ok ? rp + d0 + lane * 4 : dummy, ok);
  }
}
template <int kWarps>
__device__ __forceinline__ void x_tile_split(unsigned char* xs) {  // a thread splits its own chunks (visible to it after the wait)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 64 / kWarps; ++i) {
    const int row = warp + kWarps * i, box = lane >> 3;
    unsigned char* a = xs + box * 8192 + sw128_b32(row, lane & 7);
    float4 hi, lo;
    split_tf32(*reinterpret_cast<const float4*>(a), hi, lo);
    *reinterpret_cast<float4*>(a) = hi;
    *reinterpret_cast<float4*>(a + 32768) = lo;
  }
}
template <int kNT>
__device__ __forceinline__ void g_tile_issue(unsigned char* gs, const float* G, int64_t ldg, int64_t rows, int c0, int C) {
#pragma unroll
  for (int i = 0; i < 1024 / kNT; ++i) {
    const int f = threadIdx.x + kNT * i, row = f >> 4, chg = f & 15, box = chg >> 3;
    const bool ok = row < rows && c0 + chg * 4 < C;  // ldg % 4 == 0 and ldg >= C: the 16 bytes stay inside the row
    cp_async16(gs + box * 8192 + sw128_b32(row, chg & 7), ok ? G + row * ldg + c0 + chg * 4 : G, ok);
  }
}
template <int kNT>
__device__ __forceinline__ void g_tile_split(unsigned char* gs) {
#pragma unroll
  for (int i = 0; i < 1024 / kNT; ++i) {
    const int f = threadIdx.x + kNT * i, row = f >> 4, chg = f & 15, box = chg >> 3;
    unsigned char* b = gs + box * 8192 + sw128_b32(row, chg & 7);
    float4 hi, lo;
    split_tf32(*reinterpret_cast<const float4*>(b), hi, lo);
    *reinterpret_cast<float4*>(b) = hi;
    *reinterpret_cast<float4*>(b + 16384) = lo;
  }
}

template <int kNT>
__global__ void __launch_bounds__(kNT + 64, 1)
    sweep_dw_update_tc_kernel(const __grid_constant__ SweepDev p, const __grid_constant__ CUtensorMap tm_w,
                              const __grid_constant__ CUtensorMap tm_m, const __grid_constant__ CUtensorMap tm_v) {
  static_assert(kNT == 256 || kNT == 512, "8 or 4 classes of a stage per thread");
  constexpr int BM = 128, BN = 64, kR = 64, NS = kTcDwSlots, kWarps = kNT / 32;
  const int D = p.dim, C = p.n_classes;
  const int n_dt = (D + BM - 1) / BM, n_ct = (C + BN - 1) / BN, per_head = n_dt * n_ct;
  const int n_units = __popc(p.active_mask) * per_head;
  const int u_lo = static_cast<int>(static_cast<int64_t>(n_units) * blockIdx.x / gridDim.x);
  const int u_hi = static_cast<int>(static_cast<int64_t>(n_units) * (blockIdx.x + 1) / gridDim.x);
  if (u_lo >= u_hi) return;
  extern __shared__ unsigned char tc_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~uintptr_t(1023));
  unsigned char* slots = smem + 96 * 1024;
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(slots + NS * kTcDwSlotBytes);  // [2]
  uint64_t* full_bar = mma_bar + 2;                                             // [NS] slot loaded
  uint64_t* done_bar = full_bar + NS;                                           // [NS] slot updated by every update warp
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + NS);
  __shared__ const float* rowp[kR];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int64_t R = p.n0 + p.n1;  // <= 64 (launcher)
  const bool has_v = p.kind != 3;
  const uint32_t stage_tx = has_v ? 3 * 8192 : 2 * 8192;

  auto first_unit = [&](DwUnit& c) {
    const int a = u_lo / per_head, r = u_lo - a * per_head;
    c.unit = u_lo;
    c.st = 0;
    c.head = __fns(p.active_mask, 0, a + 1);  // the a-th running head
    c.dt = r / n_ct;
    c.ct = r - c.dt * n_ct;
    c.nst = (min(BN, C - c.ct * BN) + 15) >> 4;
  };
  auto next_unit = [&](DwUnit& c) {  // (no divisions: the cursors move one unit at a time)
    ++c.unit;
    c.st = 0;
    if (++c.ct == n_ct) {
      c.ct = 0;
      if (++c.dt == n_dt) {
        c.dt = 0;
        if (c.unit < u_hi) c.head = __ffs(p.active_mask >> (c.head + 1)) + c.head;  // the next running head
      }
    }
    c.nst = (min(BN, C - c.ct * BN) + 15) >> 4;
  };
  DwUnit cur;
  first_unit(cur);

  if (t < kR) rowp[t] = (t < R) ? row_ptr(p, cur.head, t) : nullptr;
  if (t == 0) {
    tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_m);
    if (has_v) tma_prefetch_desc(&tm_v);
    mbar_init(&mma_bar[0], 1);
    mbar_init(&mma_bar[1], 1);
    for (int s = 0; s < NS; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&done_bar[s], kWarps);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kWarps + 1) {
    // ------------------------------------------------ statistics warp: what sweep_stats_kernel computes, in a warp that
    // would otherwise not exist (running head a belongs to CTA a mod gridDim.x; lanes stride over the rows, shuffle tree).
    // With learnable temperatures it also sums the rows' d loss / d scale and steps the head's two scales with the
    // head's optimizer rule (the scales share the weights' parameter group: same lr, decay, betas and step count); the
    // next read of a scale is the next step's logits launch.  stats == NULL (adapter update launch): nothing to do.
    const int n_act = p.stats ? __popc(p.active_mask) : 0;
    for (int a = blockIdx.x; a < n_act; a += gridDim.x) {
      const int hd = __fns(p.active_mask, 0, a + 1);
      for (int sg = 0; sg < 2; ++sg) {
        const int64_t beg = sg ? p.n0 : 0, n = sg ? p.n1 : p.n0;
        const float* rl = p.row_loss + hd * p.row_stride + beg;
        const int32_t* rc = p.row_correct + hd * p.row_stride + beg;
        const float* rd = p.scale_dev ? p.row_dscale + hd * p.row_stride + beg : nullptr;
        float ls = 0.f, ds = 0.f;
        int hits = 0;
        for (int64_t i = lane; i < n; i += 32) {
          ls += rl[i];
          hits += rc[i];
          if (rd) ds += rd[i];
        }
        ls = warp_sum(ls);
        ds = warp_sum(ds);
        hits = warp_sum_i(hits);
        if (lane == 0) {
          uml_seg_stats& o = p.stats[hd * 2 + sg];
          o.loss_mean = n > 0 ? ls / static_cast<float>(n) : 0.f;
          o.dscale = ds;
          o.correct = hits;
          o.n = static_cast<int32_t>(n);
          if (rd && n > 0) {  // (a modality without rows leaves its scale without a gradient: torch skips it)
            float w = p.scale_dev[2 * hd + sg], m = p.scale_m[2 * hd + sg];
            float v = p.kind == 3 ? 0.f : p.scale_v[2 * hd + sg];
            update_one(p, p.lr[hd], p.step_size[hd], p.decay[hd], p.wd[hd], w, m, v, ds);
            p.scale_dev[2 * hd + sg] = w;
            p.scale_m[2 * hd + sg] = m;
            if (p.kind != 3) p.scale_v[2 * hd + sg] = v;
          }
        }
      }
    }
  } else if (warp == kWarps) {
    // ------------------------------------------------ TMA warp: slot ring of W, m, v ---------------------------------
    if (lane == 0) {
      DwUnit prod = cur, stc = cur;  // load cursor (NS - 1 stages ahead), store cursor
      auto prod_issue = [&](int gs) {
        unsigned char* sl = slots + (gs % NS) * kTcDwSlotBytes;
        uint64_t* bar = &full_bar[gs % NS];
        const int c = prod.ct * BN + prod.st * 16, d0 = prod.dt * BM;
        mbar_arrive_expect_tx(bar, stage_tx);
        tma_load_3d(sl, &tm_w, bar, d0, c, prod.head);
        tma_load_3d(sl + 8192, &tm_m, bar, d0, c, prod.head);
        if (has_v) tma_load_3d(sl + 16384, &tm_v, bar, d0, c, prod.head);
        if (++prod.st == prod.nst) next_unit(prod);
      };
      for (int g = 0; g < NS - 1 && prod.unit < u_hi; ++g) prod_issue(g);  // on their way while the operand tiles land
      for (int gs = 0; stc.unit < u_hi; ++gs) {
        unsigned char* sl = slots + (gs % NS) * kTcDwSlotBytes;
        mbar_wait_or_trap(&done_bar[gs % NS], static_cast<uint32_t>(gs / NS) & 1u);  // (the update warps fenced their stores)
        const int c = stc.ct * BN + stc.st * 16, d0 = stc.dt * BM;
        tma_store_3d(&tm_w, sl, d0, c, stc.head);
        tma_store_3d(&tm_m, sl + 8192, d0, c, stc.head);
        if (has_v) tma_store_3d(&tm_v, sl + 16384, d0, c, stc.head);
        bulk_commit();
        if (++stc.st == stc.nst) next_unit(stc);
        if (prod.unit < u_hi) {
          bulk_wait_read<1>();  // every store group but this one has read its slot: the slot of the previous stage is free again
          prod_issue(gs + NS - 1);
        }
      }
      bulk_wait<0>();
    }
  } else {
    // ------------------------------------------------ update warps: operand staging, MMA issue, read-back --------------
    auto sync_update_warps = [&]() { asm volatile("bar.sync 1, %0;" ::"n"(kNT) : "memory"); };
    // feature tile: 64 rows x 32 chunks (a warp per row); G tile: 64 rows x 16 chunks
    auto x_issue = [&](int d0) { x_tile_issue<kWarps>(smem, rowp, d0, D, p.G); };
    auto x_split = [&]() { x_tile_split<kWarps>(smem); };
    auto g_issue = [&](const DwUnit& un) { g_tile_issue<kNT>(smem + 65536, p.G + un.head * p.g_stride, p.ldg, R, un.ct * BN, C); };
    auto g_split = [&]() { g_tile_split<kNT>(smem + 65536); };
    constexpr uint32_t idesc = make_idesc_tf32(BM, BN, 1, 1);
    const uint32_t a_hi = smem_u32(smem), a_lo = a_hi + 32768, b_hi = a_hi + 65536, b_lo = b_hi + 16384;
    auto mma_unit = [&](int n) {  // one thread; accumulators of local unit n in TMEM region n & 1
      const uint32_t acc = tmem_base + (n & 1) * BN;
      tc_fence_after();
#pragma unroll
      for (int k = 0; k < kR / 8; ++k) {  // 8 rows = two 4-row atoms (SBO 512 B); the next 32 dims / classes 8 KB further (LBO)
        const uint64_t dah = make_smem_desc(a_hi + k * 1024, 8192, 512, kLayoutSw128Base32);
        const uint64_t dal = make_smem_desc(a_lo + k * 1024, 8192, 512, kLayoutSw128Base32);
        const uint64_t dbh = make_smem_desc(b_hi + k * 1024, 8192, 512, kLayoutSw128Base32);
        const uint64_t dbl = make_smem_desc(b_lo + k * 1024, 8192, 512, kLayoutSw128Base32);
        umma_tf32(acc, dal, dbh, idesc, k != 0);
        umma_tf32(acc, dah, dbl, idesc, 1);
        umma_tf32(acc, dah, dbh, idesc, 1);
      }
      umma_commit(&mma_bar[n & 1]);
    };

    // prologue: the first unit's tiles
    x_issue(cur.dt * BM);
    g_issue(cur);
    cp_async_commit();
    cp_async_wait<0>();
    x_split();
    g_split();
    fence_proxy_async();
    sync_update_warps();
    if (t == 0) mma_unit(0);

    constexpr int kCpt = 16 / (kNT / 128);  // classes of a stage per thread
    const int q = warp & 3, h = warp >> 2;  // TMEM lane quadrant (dims 32 q + lane), classes kCpt h + [0, kCpt) of a stage
    const uint32_t slot0 = smem_u32(slots) + static_cast<uint32_t>(((h * kCpt) * BM + q * 32 + lane) * 4);
    int gs = 0;  // stages read back so far (slot ring position)
#pragma unroll 1
    for (int n = 0; cur.unit < u_hi; ++n) {
      DwUnit nxt = cur;
      next_unit(nxt);
      const bool have_next = nxt.unit < u_hi;
      const bool new_x = have_next && (nxt.head != cur.head || nxt.dt != cur.dt);
      const float lr = p.lr[cur.head], step_size = p.step_size[cur.head], decay = p.decay[cur.head], wd = p.wd[cur.head];
      const int fin = min(1, cur.nst - 1);  // the stage before which the next unit is split and multiplied
      mbar_wait_or_trap(&mma_bar[n & 1], static_cast<uint32_t>(n >> 1) & 1u);  // unit n is in TMEM, its tiles have been read
      tc_fence_after();
      if (have_next) {
        if (nxt.head != cur.head) {
          if (t < kR) rowp[t] = (t < R) ? row_ptr(p, nxt.head, t) : nullptr;
          sync_update_warps();
        }
        if (new_x) x_issue(nxt.dt * BM);
        g_issue(nxt);
        cp_async_commit();
      }
#pragma unroll 1
      for (int u = 0; u < cur.nst; ++u, ++gs) {
        if (have_next && u == fin) {
          // (the other TMEM region was last read by this CTA's loads of unit n - 1, a full unit ago)
          cp_async_wait<0>();
          if (new_x) x_split();
          g_split();
          fence_proxy_async();
          tc_fence_before();
          sync_update_warps();
          if (t == 0) mma_unit(n + 1);
        }
        const uint32_t sa = slot0 + (gs % NS) * kTcDwSlotBytes;
        mbar_wait_or_trap(&full_bar[gs % NS], static_cast<uint32_t>(gs / NS) & 1u);
        float w[kCpt], mo[kCpt], vo[kCpt];
#pragma unroll
        for (int i = 0; i < kCpt; ++i) {  // every load first: kCpt independent chains of sqrt and division follow
          w[i] = lds_f32(sa + i * (BM * 4));
          mo[i] = lds_f32(sa + 8192 + i * (BM * 4));
          vo[i] = has_v ? lds_f32(sa + 16384 + i * (BM * 4)) : 0.f;
        }
        uint32_t acc[kCpt];
        tmem_ldn(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (n & 1) * BN + u * 16 + h * kCpt, acc);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < kCpt; ++i) update_one(p, lr, step_size, decay, wd, w[i], mo[i], vo[i], __uint_as_float(acc[i]));
#pragma unroll
        for (int i = 0; i < kCpt; ++i) {
          sts_f32(sa + i * (BM * 4), w[i]);
          sts_f32(sa + 8192 + i * (BM * 4), mo[i]);
          if (has_v) sts_f32(sa + 16384 + i * (BM * 4), vo[i]);
        }
        fence_proxy_async();  // generic-proxy stores -> the TMA stores' async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(&done_bar[gs % NS]);
      }
      cur = nxt;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 128);
}

// 5t. adapter back-propagation dZ_k = G_k[image rows] . W_k, with W_k before the step's update (the head launch updates
//     it after this one), transposed tile: D[dim, row] = W_k^T[128 dims, classes] . G_k^T[classes, 64 rows]
//     grid (ceil(D/128), K).  A = weight rows read along the dims: MN-major, SWIZZLE_128B_BASE32B like the dW kernel's
//     feature tile (k-blocks of 32 classes: four 4 KB boxes of 32 classes x 32 dims); B = G rows, K-major SWIZZLE_128B
//     like the logits kernel's row tile.  Two stages, the next block's loads in registers while this one is split and
//     multiplied, as in the logits kernel; the accumulation order is fixed by the instruction stream (no atomics), so a
//     head's dZ does not depend on its slot.
constexpr int kTcDzStage = 48 * 1024;  // W hi 16 KB | W lo 16 KB | G hi 8 KB | G lo 8 KB
constexpr int kTcDzSmemBytes = 2 * kTcDzStage + 1024 + 64;

__global__ void __launch_bounds__(256, 2)
    sweep_dz_tc_kernel(const __grid_constant__ SweepDev p, float* __restrict__ dZ, int64_t ldz, int64_t dz_stride) {
  constexpr int BM = 128, BN = 64, BK = 32, S = 2;
  const int head = blockIdx.y;
  if (!head_active(p, head)) return;
  extern __shared__ unsigned char tc_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* empty_bar = reinterpret_cast<uint64_t*>(smem + S * kTcDzStage);
  uint64_t* tfull_bar = empty_bar + S;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull_bar + 1);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int64_t R = p.n0;  // image rows only (<= 64, launcher)
  const int d0 = blockIdx.x * BM;
  const int D = p.dim, C = p.n_classes;
  const float* __restrict__ W = p.W + head * p.head_stride;
  const float* __restrict__ G = p.G + head * p.g_stride;
  if (t == 0) {
    for (int s = 0; s < S; ++s) mbar_init(&empty_bar[s], 1);
    mbar_init(tfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // this thread's 16-byte chunks of a k-block: four of the weight tile (32 classes x 128 dims, a warp per class row),
  // two of the G tile (64 rows x 32 classes, eight threads per row)
  int wrow[4], wcol[4], grow[2], gch[2];
  uint32_t woff[4], goff[2];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int f = t + 256 * i, j = f & 31;
    wrow[i] = f >> 5;
    wcol[i] = d0 + 4 * j;
    woff[i] = static_cast<uint32_t>((j >> 3) * 4096) + sw128_b32(wrow[i], j & 7);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int f = t + 256 * i;
    grow[i] = f >> 3;
    gch[i] = f & 7;
    goff[i] = sw128(grow[i], gch[i]);
  }
  auto load = [&](int kb, float4 (&r)[6]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int c = kb * BK + wrow[i];
      r[i] = (c < C && wcol[i] < D) ? __ldg(reinterpret_cast<const float4*>(W + static_cast<int64_t>(c) * D + wcol[i]))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int c = kb * BK + 4 * gch[i];
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (grow[i] < R && c < C) {  // (ldg % 4 == 0: the chunk stays inside the row; columns >= C are not written by the
        x = *reinterpret_cast<const float4*>(G + grow[i] * p.ldg + c);  //  logits launch and must not enter the sum)
        if (c + 1 >= C) x.y = 0.f;
        if (c + 2 >= C) x.z = 0.f;
        if (c + 3 >= C) x.w = 0.f;
      }
      r[4 + i] = x;
    }
  };

  const int nk = (C + BK - 1) / BK;
  constexpr uint32_t idesc = make_idesc_tf32(BM, BN, 1, 0);
  float4 cur[6], nxt[6];
  load(0, cur);
#pragma unroll 1
  for (int kb = 0; kb < nk; ++kb) {
    if (kb + 1 < nk) load(kb + 1, nxt);
    const int s = kb & (S - 1);
    if (kb >= S) mbar_wait_or_trap(&empty_bar[s], static_cast<uint32_t>((kb / S) - 1) & 1u);
    unsigned char* st = smem + s * kTcDzStage;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float4 hi, lo;
      split_tf32(cur[i], hi, lo);
      *reinterpret_cast<float4*>(st + woff[i]) = hi;
      *reinterpret_cast<float4*>(st + 16384 + woff[i]) = lo;
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      float4 hi, lo;
      split_tf32(cur[4 + i], hi, lo);
      *reinterpret_cast<float4*>(st + 32768 + goff[i]) = hi;
      *reinterpret_cast<float4*>(st + 40960 + goff[i]) = lo;
    }
    fence_proxy_async();
    __syncthreads();
    if (t == 0) {
      tc_fence_after();
      const uint32_t a_hi = smem_u32(st), a_lo = a_hi + 16384, b_hi = a_hi + 32768, b_lo = a_hi + 40960;
#pragma unroll
      for (int k = 0; k < BK / 8; ++k) {  // A: 8 classes = two 4-row atoms (SBO 512 B), next 32 dims one 4 KB box further
        const uint64_t dah = make_smem_desc(a_hi + k * 1024, 4096, 512, kLayoutSw128Base32);
        const uint64_t dal = make_smem_desc(a_lo + k * 1024, 4096, 512, kLayoutSw128Base32);
        const uint64_t dbh = make_smem_desc(b_hi + k * 32, 16, 1024, kLayoutSw128);
        const uint64_t dbl = make_smem_desc(b_lo + k * 32, 16, 1024, kLayoutSw128);
        umma_tf32(tmem_base, dal, dbh, idesc, (kb | k) != 0);
        umma_tf32(tmem_base, dah, dbl, idesc, 1);
        umma_tf32(tmem_base, dah, dbh, idesc, 1);
      }
      umma_commit(&empty_bar[s]);
      if (kb == nk - 1) umma_commit(tfull_bar);
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) cur[i] = nxt[i];
  }

  // epilogue: TMEM lane = dim, column = row; warp w reads lane quadrant w % 4, rows 32 (w / 4) ..
  mbar_wait_or_trap(tfull_bar, 0);
  tc_fence_after();
  const int q = warp & 3, h = warp >> 2;
  uint32_t v[32];
  tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + h * 32, v);
  tmem_ld_wait();
  const int d = d0 + q * 32 + lane;
  if (d < D) {
    float* __restrict__ out = dZ + head * dz_stride + d;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const int64_t r = h * 32 + i;
      if (r < R) out[r * ldz] = __uint_as_float(v[i]);  // a warp stores 32 consecutive dims of one row
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 64);
}

// 6t. gradient diagnostics (the reference's per-step probes, finetune.py:190-206): per running head the image-loss and
//     text-loss gradients of the head weights, A = X_img^T G[image rows] and B = X_txt^T G[text rows] (both [D, C]
//     transposed), reduced without being stored to {sum A.B, sum A^2, sum B^2, #(sign A == sign B)}.
//     Persistent over the dW kernel's (head, 128-dim tile, 64-class tile) units with its operand staging and 3xTF32 MMAs;
//     the rows are the K dimension, 64 per k-tile, accumulated in TMEM - any step size.  Two accumulators per unit
//     (columns [0, 64) image, [64, 128) text): the G tile is split twice, each copy with the other modality's rows zero,
//     so a k-step of 8 rows that crosses n0 adds only its own rows to each.  A unit's sums go to its own slot of `part`
//     ([K][dim tiles][class tiles][4], by head index), finished in a fixed order by sweep_grad_diag_finish_kernel: no
//     float atomics, so a head's figures depend neither on its slot nor on its neighbours.  Reads G and rows only.
constexpr int kTcDiagSmemBytes = 128 * 1024 + 1024 + 64;  // X hi | X lo (32 KB each) | G image hi | lo | G text hi | lo (16 KB each)

__global__ void __launch_bounds__(256, 1) sweep_grad_diag_tc_kernel(const __grid_constant__ SweepDev p, float* __restrict__ part) {
  constexpr int BM = 128, BN = 64, kR = 64, kNT = 256, kWarps = kNT / 32;
  const int D = p.dim, C = p.n_classes;
  const int n_dt = (D + BM - 1) / BM, n_ct = (C + BN - 1) / BN, per_head = n_dt * n_ct;
  const int n_units = __popc(p.active_mask) * per_head;
  const int u_lo = static_cast<int>(static_cast<int64_t>(n_units) * blockIdx.x / gridDim.x);
  const int u_hi = static_cast<int>(static_cast<int64_t>(n_units) * (blockIdx.x + 1) / gridDim.x);
  if (u_lo >= u_hi) return;
  extern __shared__ unsigned char tc_smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(tc_smem_raw) + 1023) & ~uintptr_t(1023));
  unsigned char* gs = smem + 65536;
  uint64_t* mma_bar = reinterpret_cast<uint64_t*>(smem + 128 * 1024);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_bar + 1);
  __shared__ const float* rowp[kR];
  __shared__ float red[kWarps][3];
  __shared__ int red_n[kWarps];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int64_t n0 = p.n0, R = p.n0 + p.n1;
  const bool has_img = p.n0 > 0, has_txt = p.n1 > 0;
  if (t == 0) {
    mbar_init(mma_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  constexpr uint32_t idesc = make_idesc_tf32(BM, BN, 1, 1);
  const uint32_t a_hi = smem_u32(smem), a_lo = a_hi + 32768, gi_hi = smem_u32(gs), gi_lo = gi_hi + 16384,
                 gt_hi = gi_hi + 32768, gt_lo = gi_hi + 49152;

  int head, dt, ct;
  {
    const int a = u_lo / per_head, r = u_lo - a * per_head;
    head = __fns(p.active_mask, 0, a + 1);  // the a-th running head
    dt = r / n_ct;
    ct = r - dt * n_ct;
  }
  int x_head = -1, x_dt = -1;  // the feature tile in shared memory (steps of at most 64 rows keep it across class tiles)
  uint32_t phase = 0;
#pragma unroll 1
  for (int u = u_lo; u < u_hi; ++u) {
    const float* __restrict__ G = p.G + head * p.g_stride;
    const int d0 = dt * BM, c0 = ct * BN;
    uint32_t acc_img = 0, acc_txt = 0;  // MMAs issued into each accumulator (thread 0)
#pragma unroll 1
    for (int64_t r0 = 0; r0 < R; r0 += kR) {
      const int64_t rows = min(static_cast<int64_t>(kR), R - r0);
      const bool new_x = R > kR || head != x_head || dt != x_dt;
      if (new_x) {
        if (t < kR) rowp[t] = (t < rows) ? row_ptr(p, head, r0 + t) : nullptr;
        __syncthreads();
        x_tile_issue<kWarps>(smem, rowp, d0, D, G);
        x_head = head;
        x_dt = dt;
      }
      g_tile_issue<kNT>(gs, G + r0 * p.ldg, p.ldg, rows, c0, C);
      cp_async_commit();
      cp_async_wait<0>();
      if (new_x) x_tile_split<kWarps>(smem);
#pragma unroll
      for (int i = 0; i < 1024 / kNT; ++i) {  // G split twice: image rows only | text rows only
        const int f = t + kNT * i, row = f >> 4, chg = f & 15, box = chg >> 3;
        unsigned char* b = gs + box * 8192 + sw128_b32(row, chg & 7);
        float4 hi, lo;
        split_tf32(*reinterpret_cast<const float4*>(b), hi, lo);
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        const bool img = r0 + row < n0;
        *reinterpret_cast<float4*>(b) = img ? hi : z;
        *reinterpret_cast<float4*>(b + 16384) = img ? lo : z;
        *reinterpret_cast<float4*>(b + 32768) = img ? z : hi;
        *reinterpret_cast<float4*>(b + 49152) = img ? z : lo;
      }
      fence_proxy_async();  // generic-proxy stores -> the tensor core's async-proxy reads
      tc_fence_before();    // (the previous unit's TMEM read-back is complete)
      __syncthreads();
      if (t == 0) {
        tc_fence_after();
#pragma unroll 1
        for (int k = 0; k < kR / 8 && r0 + 8 * k < R; ++k) {  // 8 rows = two 4-row atoms (SBO 512 B); next 32 columns 8 KB further
          const int64_t rb = r0 + 8 * k;
          const uint64_t dah = make_smem_desc(a_hi + k * 1024, 8192, 512, kLayoutSw128Base32);
          const uint64_t dal = make_smem_desc(a_lo + k * 1024, 8192, 512, kLayoutSw128Base32);
          if (rb < n0) {
            const uint64_t dbh = make_smem_desc(gi_hi + k * 1024, 8192, 512, kLayoutSw128Base32);
            const uint64_t dbl = make_smem_desc(gi_lo + k * 1024, 8192, 512, kLayoutSw128Base32);
            umma_tf32(tmem_base, dal, dbh, idesc, acc_img != 0);
            umma_tf32(tmem_base, dah, dbl, idesc, 1);
            umma_tf32(tmem_base, dah, dbh, idesc, 1);
            ++acc_img;
          }
          if (has_txt && rb + 8 > n0) {
            const uint64_t dbh = make_smem_desc(gt_hi + k * 1024, 8192, 512, kLayoutSw128Base32);
            const uint64_t dbl = make_smem_desc(gt_lo + k * 1024, 8192, 512, kLayoutSw128Base32);
            umma_tf32(tmem_base + BN, dal, dbh, idesc, acc_txt != 0);
            umma_tf32(tmem_base + BN, dah, dbl, idesc, 1);
            umma_tf32(tmem_base + BN, dah, dbh, idesc, 1);
            ++acc_txt;
          }
        }
        umma_commit(mma_bar);
      }
      mbar_wait_or_trap(mma_bar, phase);  // the MMAs have read the tiles and written TMEM
      phase ^= 1u;
      tc_fence_after();
    }

    // read-back: TMEM lane = dim, column = class; warp w reads lane quadrant w % 4, classes 32 (w / 4) ..
    const int q = warp & 3, h = warp >> 2;
    uint32_t va[32], vb[32];
    tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + h * 32, va);
    tmem_ld32(tmem_base + (static_cast<uint32_t>(q * 32) << 16) + BN + h * 32, vb);
    tmem_ld_wait();
    float dot = 0.f, aa = 0.f, bb = 0.f;
    int agree = 0;
    if (d0 + q * 32 + lane < D) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        if (c0 + h * 32 + i >= C) break;
        const float x = has_img ? __uint_as_float(va[i]) : 0.f, y = has_txt ? __uint_as_float(vb[i]) : 0.f;
        dot = fmaf(x, y, dot);
        aa = fmaf(x, x, aa);
        bb = fmaf(y, y, bb);
        agree += ((x > 0.f) - (x < 0.f)) == ((y > 0.f) - (y < 0.f));  // torch.sign: 0 only equals 0
      }
    }
    dot = warp_sum(dot);
    aa = warp_sum(aa);
    bb = warp_sum(bb);
    agree = warp_sum_i(agree);
    if (lane == 0) {
      red[warp][0] = dot;
      red[warp][1] = aa;
      red[warp][2] = bb;
      red_n[warp] = agree;
    }
    __syncthreads();
    if (t == 0) {
      float s0 = 0.f, s1 = 0.f, s2 = 0.f;
      int n = 0;
      for (int w = 0; w < kWarps; ++w) {
        s0 += red[w][0];
        s1 += red[w][1];
        s2 += red[w][2];
        n += red_n[w];
      }
      float* o = part + (static_cast<int64_t>(head) * per_head + dt * n_ct + ct) * 4;
      o[0] = s0;
      o[1] = s1;
      o[2] = s2;
      o[3] = static_cast<float>(n);  // at most 128 x 64: exact
    }
    if (++ct == n_ct) {
      ct = 0;
      if (++dt == n_dt) {
        dt = 0;
        if (u + 1 < u_hi) head = __ffs(p.active_mask >> (head + 1)) + head;  // the next running head
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 128);
}

// out[head] = the unit sums of each running head in unit order (double), the text side divided by alpha / alpha^2 (G's
// text rows carry the loss weight; the figures describe the plain text loss)        grid (K), 32 threads
__global__ void __launch_bounds__(32) sweep_grad_diag_finish_kernel(const __grid_constant__ SweepDev p, const float* __restrict__ part,
                                                                    int units_per_head, float* __restrict__ out) {
  const int head = blockIdx.x, j = threadIdx.x;
  if (!head_active(p, head) || j >= 4) return;
  const float* ph = part + static_cast<int64_t>(head) * units_per_head * 4;
  double s = 0.0;
  if (j == 3) {
    long long n = 0;
    for (int u = 0; u < units_per_head; ++u) n += static_cast<long long>(ph[4 * u + 3]);
    s = static_cast<double>(n);
  } else {
    for (int u = 0; u < units_per_head; ++u) s += static_cast<double>(ph[4 * u + j]);
    const double al = p.alpha[head];  // > 0 whenever there are text rows (launcher)
    if (j == 0 && p.n1 > 0) s /= al;
    if (j == 2 && p.n1 > 0) s /= al * al;
  }
  out[4 * head + j] = static_cast<float>(s);
}

// ---------------------------------------------------------------------------------------------------------------
// 4. per-head, per-run {mean loss, hits, rows} in a fixed summation order   grid (2, K)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) sweep_stats_kernel(const __grid_constant__ SweepDev p) {
  const int head = blockIdx.y, s = blockIdx.x;
  if (!head_active(p, head)) return;
  __shared__ float sh[8];
  const int64_t beg = s ? p.n0 : 0, n = s ? p.n1 : p.n0;
  const float* rl = p.row_loss + head * p.row_stride + beg;
  const int32_t* rc = p.row_correct + head * p.row_stride + beg;
  float ls = 0.f;
  int hits = 0;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    ls += rl[i];
    hits += rc[i];
  }
  const float lsum = block_sum(ls, sh);
  const float hsum = block_sum(static_cast<float>(hits), sh);
  if (threadIdx.x == 0) {
    uml_seg_stats& o = p.stats[head * 2 + s];
    o.loss_mean = n > 0 ? lsum / static_cast<float>(n) : 0.f;
    o.dscale = 0.f;
    o.correct = static_cast<int32_t>(hsum + 0.5f);
    o.n = static_cast<int32_t>(n);
  }
}

}  // namespace sweep
}  // namespace uml

static long long g_sweep_launches = 0;  // kernels launched by uml_sweep_run in this process (launch accounting of the callers)

extern "C" {

int uml_sweep_launch_count(void) { return static_cast<int>(g_sweep_launches & 0x7fffffff); }

static bool aligned16(const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0; }

int64_t uml_sweep_diag_scratch_floats(int32_t n_heads, int32_t dim, int32_t n_classes) {
  if (n_heads < 1 || dim < 1 || n_classes < 1) return 0;
  return static_cast<int64_t>(n_heads) * ((dim + 127) / 128) * ((n_classes + 63) / 64) * 4;
}

// Step i's gradient diagnostics (uml_sweep_run_diag): enqueued after the step's last update launch and before the next
// step's first launch, so G and the rows (bank rows or Z) are still the step's own.
static int launch_grad_diag(const uml::sweep::SweepDev& p, const uml_sweep_diag* dg, int K, int i, bool timed, cudaStream_t st) {
  using namespace uml;
  using namespace uml::sweep;
  static const cudaError_t attr =
      cudaFuncSetAttribute(sweep_grad_diag_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcDiagSmemBytes);
  UML_CUDA(attr);
  const int per_head = ((p.dim + 127) / 128) * ((p.n_classes + 63) / 64);
  const int64_t units = static_cast<int64_t>(__builtin_popcount(p.active_mask)) * per_head;
  const unsigned g = static_cast<unsigned>(std::min<int64_t>(units, sm_count()));
  if (timed && dg->ev[0]) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(dg->ev[0]), st));
  sweep_grad_diag_tc_kernel<<<g, 256, kTcDiagSmemBytes, st>>>(p, dg->scratch);
  UML_CUDA(cudaGetLastError());
  sweep_grad_diag_finish_kernel<<<K, 32, 0, st>>>(p, dg->scratch, per_head, dg->out + static_cast<int64_t>(i) * K * 4);
  UML_CUDA(cudaGetLastError());
  g_sweep_launches += 2;
  if (timed && dg->ev[1]) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(dg->ev[1]), st));
  return 0;
}

static int sweep_run_impl(const uml_sweep_args* a, const uml_sweep_diag* dg, int32_t n_steps, const int64_t* rows,
                          const float* lr, void* stream) {
  using namespace uml;
  using namespace uml::sweep;
  UML_REQUIRE(a && rows && lr && n_steps >= 0, "sweep_run: null argument");
  const int K = a->n_heads;
  UML_REQUIRE(K >= 1 && K <= kMaxHeads, "sweep_run: 1..%d heads", kMaxHeads);
  UML_REQUIRE(a->dim > 0 && a->n_classes > 0 && a->ldg >= a->n_classes, "sweep_run: bad shape");
  UML_REQUIRE(a->kind >= 1 && a->kind <= 3, "sweep_run: optimizer kind must be 1 (AdamW), 2 (Adam) or 3 (SGD)");
  UML_REQUIRE(a->W && a->m && (a->kind == 3 || a->v) && a->G && a->row_loss && a->row_correct && a->stats,
              "sweep_run: null buffer");
  UML_REQUIRE(a->head_stride >= static_cast<int64_t>(a->n_classes) * a->dim, "sweep_run: head_stride too small");
  if (a->dim % 4 == 0) {  // the vector epilogue's alignment contract
    UML_REQUIRE(a->head_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(a->W) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(a->m) & 15) == 0 && (reinterpret_cast<uintptr_t>(a->v) & 15) == 0,
                "sweep_run: W, m, v slabs must be 16-byte aligned");
  }
  cudaStream_t st = as_stream(stream);
  SweepDev p;
  memset(&p, 0, sizeof(p));
  uint32_t mask = 0;
  for (int k = 0; k < K; ++k) {
    if (!a->active[k]) continue;
    mask |= 1u << k;
    for (int s = 0; s < 2; ++s) p.perm[s][k] = a->perm[s][k];
    p.alpha[k] = a->alpha[k];
    p.wd[k] = a->weight_decay[k];
  }
  if (mask == 0 || n_steps == 0) return 0;
  for (int s = 0; s < 2; ++s) {
    p.bank[s] = a->bank[s];
    p.labels[s] = a->labels[s];
    p.ld[s] = a->bank_ld[s];
    p.scale[s] = a->scale[s];
  }
  p.W = a->W;
  p.m = a->m;
  p.v = a->v;
  p.head_stride = a->head_stride;
  p.G = a->G;
  p.ldg = a->ldg;
  p.row_loss = a->row_loss;
  p.row_correct = a->row_correct;
  p.dim = a->dim;
  p.n_classes = a->n_classes;
  p.active_mask = mask;
  p.vec_rows = a->dim % 4 == 0;  // weight rows: covered by the slab alignment check above
  for (int s = 0; s < 2; ++s)
    if (a->bank[s] && ((reinterpret_cast<uintptr_t>(a->bank[s]) & 15) != 0 || a->bank_ld[s] % 4 != 0)) p.vec_rows = 0;
  // The cp.async variants of the two GEMM launches are the default when rows are 16-byte aligned (same results, 30 heads:
  // 0.219 against 0.268 ms per step); UML_SWEEP_ASYNC=0 selects the synchronous kernels
  static const bool want_async = [] {
    const char* e = getenv("UML_SWEEP_ASYNC");
    return !(e != nullptr && e[0] == '0');
  }();
  const bool use_async = want_async && p.vec_rows && a->ldg % 4 == 0 && (reinterpret_cast<uintptr_t>(a->G) & 15) == 0;
  if (use_async) {
    static const cudaError_t attr = cudaFuncSetAttribute(sweep_logits_async_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                         kLogitsSmemBytes);
    UML_CUDA(attr);
  }
  // tensor-core forms (3xTF32, see above) whenever the async forms' alignment contract holds; UML_SWEEP_TC=0 keeps the FFMA kernels
  static const bool want_tc = [] {
    const char* e = getenv("UML_SWEEP_TC");
    return !(e != nullptr && e[0] == '0');
  }();
  const bool use_tc = want_tc && use_async;
  if (use_tc) {
    static const cudaError_t attr1 = [] {
      cudaError_t e = cudaFuncSetAttribute(sweep_logits_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcLgSmemBytes);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(sweep_logits_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcLgSmemBytes);
      return e;
    }();
    UML_CUDA(attr1);
    static const cudaError_t attr2 = [] {
      cudaError_t e = cudaFuncSetAttribute(sweep_dw_update_tc_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcDwSmemBytes);
      if (e == cudaSuccess)
        e = cudaFuncSetAttribute(sweep_dw_update_tc_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcDwSmemBytes);
      return e;
    }();
    UML_CUDA(attr2);
  }
  // UML_SWEEP_TC_DW=0 keeps the FFMA dW + update launch next to the tensor-core logits; UML_SWEEP_DW_THREADS its CTA size
  static const bool want_tc_dw = [] {
    const char* e = getenv("UML_SWEEP_TC_DW");
    return !(e != nullptr && e[0] == '0');
  }();
  static const int dw_threads = [] {
    const char* e = getenv("UML_SWEEP_DW_THREADS");
    return (e && atoi(e) == 256) ? 256 : 512;
  }();
  const bool use_tc_dw = use_tc && want_tc_dw;
  static const bool want_fused_softmax = [] {  // UML_SWEEP_FUSED_SOFTMAX=0 keeps the separate softmax / CE launch
    const char* e = getenv("UML_SWEEP_FUSED_SOFTMAX");
    return !(e != nullptr && e[0] == '0');
  }();
  CUtensorMap tm_w, tm_m, tm_v;  // [K][C][D] views of the W, m, v slabs for the dW kernel's slot ring
  memset(&tm_w, 0, sizeof(tm_w));
  memset(&tm_m, 0, sizeof(tm_m));
  memset(&tm_v, 0, sizeof(tm_v));
  if (use_tc) {
    const uint64_t d = static_cast<uint64_t>(a->dim), c = static_cast<uint64_t>(a->n_classes), k = static_cast<uint64_t>(K);
    const uint64_t hs = static_cast<uint64_t>(a->head_stride) * 4;
    if (make_tmap_3d(&tm_w, a->W, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d, c, k, d * 4, hs, 128, 16, 1)) return 1;
    if (make_tmap_3d(&tm_m, a->m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d, c, k, d * 4, hs, 128, 16, 1)) return 1;
    if (a->kind != 3 && make_tmap_3d(&tm_v, a->v, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d, c, k, d * 4, hs, 128, 16, 1)) return 1;
  }
  p.kind = a->kind;
  p.beta1 = a->beta1;
  p.beta2 = a->beta2;
  p.eps = a->eps;
  p.momentum = a->momentum;
  int64_t pos[2] = {a->pos[0], a->pos[1]};
  for (int i = 0; i < n_steps; ++i) {
    const int64_t n0 = rows[2 * i], n1 = rows[2 * i + 1], R = n0 + n1;
    UML_REQUIRE(n0 >= 0 && n1 >= 0 && R > 0 && R <= a->max_rows, "sweep_run: step %d has %lld rows (capacity %lld)", i,
                static_cast<long long>(R), static_cast<long long>(a->max_rows));
    for (int s = 0; s < 2; ++s) {
      const int64_t n = s ? n1 : n0;
      if (n == 0) continue;
      UML_REQUIRE(a->bank[s] && a->labels[s] && pos[s] >= 0 && pos[s] + n <= a->perm_len[s],
                  "sweep_run: step %d runs past the end of permutation %d", i, s);
      for (int k = 0; k < K; ++k)
        UML_REQUIRE(!((mask >> k) & 1u) || a->perm[s][k], "sweep_run: head %d has no permutation %d", k, s);
    }
    p.n0 = n0;
    p.n1 = n1;
    p.pos[0] = pos[0];
    p.pos[1] = pos[1];
    p.g_stride = a->max_rows * a->ldg;
    p.row_stride = a->max_rows;
    p.stats = a->stats + static_cast<int64_t>(i) * K * 2;
    const double t = static_cast<double>(a->step + i);
    const double bc1 = 1.0 - pow(static_cast<double>(a->beta1), t);
    const double bc2 = 1.0 - pow(static_cast<double>(a->beta2), t);
    p.bc2_sqrt_inv = static_cast<float>(1.0 / sqrt(bc2));
    p.first_step = (a->step + i) <= 1;
    for (int k = 0; k < K; ++k) {
      const float l = lr[static_cast<int64_t>(i) * K + k];
      p.lr[k] = l;
      p.step_size[k] = static_cast<float>(static_cast<double>(l) / bc1);
      p.decay[k] = static_cast<float>(1.0 - static_cast<double>(l) * static_cast<double>(a->weight_decay[k]));
    }
    const unsigned rt = static_cast<unsigned>((R + 63) / 64), ct = static_cast<unsigned>((a->n_classes + 63) / 64);
    const bool timed = i == n_steps - 1;
    auto mark = [&](int e) -> int {
      if (timed && a->ev[e]) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(a->ev[e]), st));
      return 0;
    };
    if (mark(0)) return 1;
    // up to eight class tiles per head: they form a cluster and finish the rows (softmax / CE) in the logits epilogue
    const unsigned n_ctile = static_cast<unsigned>((a->n_classes + 127) / 128);
    // (any tile count up to eight: clusters of 3, 6 and 7 are covered by tests/test_sweep_gpu.py)
    const bool fuse_softmax = use_tc && want_fused_softmax && n_ctile <= 8;
    if (fuse_softmax)
      UML_CUDA(launch_kernel(sweep_logits_tc_kernel<true>, dim3(n_ctile, rt, K), dim3(256), kTcLgSmemBytes, st,
                             static_cast<int>(n_ctile), p));
    else if (use_tc)
      sweep_logits_tc_kernel<false><<<dim3(n_ctile, rt, K), 256, kTcLgSmemBytes, st>>>(p);
    else if (use_async)
      sweep_logits_async_kernel<<<dim3(ct, rt, K), 256, kLogitsSmemBytes, st>>>(p);
    else
      sweep_logits_kernel<<<dim3(ct, rt, K), 256, 0, st>>>(p);
    UML_CUDA(cudaGetLastError());
    ++g_sweep_launches;
    if (mark(1) || mark(2)) return 1;
    if (!fuse_softmax) {
      sweep_softmax_kernel<<<dim3(static_cast<unsigned>(R), K), 256, 0, st>>>(p);
      UML_CUDA(cudaGetLastError());
      ++g_sweep_launches;
    }
    if (mark(3) || mark(4)) return 1;
    if (use_tc_dw && R <= 64) {  // (larger steps: the feature tile of the tensor-core form holds 64 rows)
      const int64_t units = static_cast<int64_t>(__builtin_popcount(mask)) * ((a->dim + 127) / 128) * ((a->n_classes + 63) / 64);
      const unsigned g = static_cast<unsigned>(std::min<int64_t>(units, sm_count()));
      if (dw_threads == 256) sweep_dw_update_tc_kernel<256><<<g, 256 + 64, kTcDwSmemBytes, st>>>(p, tm_w, tm_m, tm_v);
      else sweep_dw_update_tc_kernel<512><<<g, 512 + 64, kTcDwSmemBytes, st>>>(p, tm_w, tm_m, tm_v);
    }
    else if (use_async)
      sweep_dw_update_async_kernel<<<dim3((a->dim + 63) / 64, (a->n_classes + 63) / 64, K), 256, 0, st>>>(p);
    else
      sweep_dw_update_kernel<<<dim3((a->dim + 63) / 64, (a->n_classes + 63) / 64, K), 256, 0, st>>>(p);
    UML_CUDA(cudaGetLastError());
    ++g_sweep_launches;
    if (mark(5) || mark(6)) return 1;
    if (!(use_tc_dw && R <= 64)) {  // (the tensor-core dW launch carries a statistics warp)
      sweep_stats_kernel<<<dim3(2, K), 256, 0, st>>>(p);
      UML_CUDA(cudaGetLastError());
      ++g_sweep_launches;
    }
    if (mark(7)) return 1;
    if (dg && launch_grad_diag(p, dg, K, i, timed, st)) return 1;
    pos[0] += n0;
    pos[1] += n1;
  }
  return 0;
}

int uml_sweep_run(const uml_sweep_args* a, int32_t n_steps, const int64_t* rows, const float* lr, void* stream) {
  return sweep_run_impl(a, nullptr, n_steps, rows, lr, stream);
}

static int sweep_adapter_run_impl(const uml_sweep_args* a, const uml_sweep_adapter_args* ad, const uml_sweep_diag* dg,
                                  int32_t n_steps, const int64_t* rows, const float* lr, void* stream) {
  using namespace uml;
  using namespace uml::sweep;
  UML_REQUIRE(a && ad && rows && lr && n_steps >= 0, "sweep_adapter_run: null argument");
  const int K = a->n_heads;
  UML_REQUIRE(K >= 1 && K <= kMaxHeads, "sweep_adapter_run: 1..%d heads", kMaxHeads);
  UML_REQUIRE(a->dim > 0 && a->n_classes > 0 && a->ldg >= a->n_classes, "sweep_adapter_run: bad shape");
  UML_REQUIRE(a->kind >= 1 && a->kind <= 3, "sweep_adapter_run: optimizer kind must be 1 (AdamW), 2 (Adam) or 3 (SGD)");
  UML_REQUIRE(a->W && a->m && (a->kind == 3 || a->v) && a->G && a->row_loss && a->row_correct && a->stats,
              "sweep_adapter_run: null buffer");
  UML_REQUIRE(a->head_stride >= static_cast<int64_t>(a->n_classes) * a->dim, "sweep_adapter_run: head_stride too small");
  const bool adapter = ad->img_dim > 0, temps = ad->scale_param != nullptr;
  // tensor-core forms only: 16-byte rows and operands, one 64-row feature tile, softmax / CE in the logits epilogue
  UML_REQUIRE(a->dim % 4 == 0 && ad->img_dim % 4 == 0 && ad->img_dim >= 0, "sweep_adapter_run: dims must be multiples of 4");
  UML_REQUIRE(a->n_classes <= 1024, "sweep_adapter_run: at most 1024 classes (softmax / CE in the logits epilogue)");
  UML_REQUIRE(a->max_rows >= 1 && a->max_rows <= 64, "sweep_adapter_run: at most 64 rows per step (max_rows %lld)",
              static_cast<long long>(a->max_rows));
  UML_REQUIRE(a->head_stride % 4 == 0 && aligned16(a->W) && aligned16(a->m) && aligned16(a->v) && aligned16(a->G) &&
                  a->ldg % 4 == 0,
              "sweep_adapter_run: W, m, v, G must be 16-byte aligned with strides that are multiples of 4");
  for (int s = 0; s < 2; ++s)
    UML_REQUIRE(!a->bank[s] || (aligned16(a->bank[s]) && a->bank_ld[s] % 4 == 0),
                "sweep_adapter_run: bank %d rows must be 16-byte aligned", s);
  if (adapter) {
    UML_REQUIRE(ad->W && ad->m && (a->kind == 3 || ad->v) && ad->Z && ad->dZ, "sweep_adapter_run: null adapter buffer");
    UML_REQUIRE(ad->adapter_stride >= static_cast<int64_t>(a->dim) * ad->img_dim && ad->adapter_stride % 4 == 0 &&
                    aligned16(ad->W) && aligned16(ad->m) && aligned16(ad->v),
                "sweep_adapter_run: adapter slabs must be 16-byte aligned, adapter_stride >= dim * img_dim, a multiple of 4");
    UML_REQUIRE(ad->ldz >= a->dim && ad->ldz % 4 == 0 && ad->max_img_rows >= 1 && aligned16(ad->Z) && aligned16(ad->dZ),
                "sweep_adapter_run: Z / dZ must be 16-byte aligned with ldz >= dim, a multiple of 4");
  }
  if (temps)
    UML_REQUIRE(ad->scale_m && (a->kind == 3 || ad->scale_v) && ad->row_dscale,
                "sweep_adapter_run: learnable temperatures need scale_m, scale_v and row_dscale");
  cudaStream_t st = as_stream(stream);
  SweepDev p;
  memset(&p, 0, sizeof(p));
  uint32_t mask = 0;
  for (int k = 0; k < K; ++k) {
    if (!a->active[k]) continue;
    mask |= 1u << k;
    for (int s = 0; s < 2; ++s) p.perm[s][k] = a->perm[s][k];
    p.alpha[k] = a->alpha[k];
    p.wd[k] = a->weight_decay[k];
  }
  if (mask == 0 || n_steps == 0) return 0;
  for (int s = 0; s < 2; ++s) {
    p.bank[s] = a->bank[s];
    p.labels[s] = a->labels[s];
    p.ld[s] = a->bank_ld[s];
    p.scale[s] = a->scale[s];
  }
  p.W = a->W;
  p.m = a->m;
  p.v = a->v;
  p.head_stride = a->head_stride;
  p.G = a->G;
  p.ldg = a->ldg;
  p.g_stride = a->max_rows * a->ldg;
  p.row_loss = a->row_loss;
  p.row_correct = a->row_correct;
  p.row_stride = a->max_rows;
  p.dim = a->dim;
  p.n_classes = a->n_classes;
  p.active_mask = mask;
  p.vec_rows = 1;
  p.kind = a->kind;
  p.beta1 = a->beta1;
  p.beta2 = a->beta2;
  p.eps = a->eps;
  p.momentum = a->momentum;
  if (temps) {
    p.scale_dev = ad->scale_param;
    p.scale_m = ad->scale_m;
    p.scale_v = ad->scale_v;
    p.row_dscale = ad->row_dscale;
  }
  if (adapter) {
    p.zrows = ad->Z;
    p.z_ld = ad->ldz;
    p.z_stride = ad->max_img_rows * ad->ldz;
  }
  static const cudaError_t attr = [] {
    cudaError_t e = cudaFuncSetAttribute(sweep_logits_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcLgSmemBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(sweep_logits_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcLgSmemBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(sweep_dw_update_tc_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcDwSmemBytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(sweep_dz_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcDzSmemBytes);
    return e;
  }();
  UML_CUDA(attr);
  // [K][rows][dim] views of the slabs for the dW kernel's slot ring: the head (C x D) and the adapter (D x Dv)
  CUtensorMap tm_w, tm_m, tm_v, tma_w, tma_m, tma_v;
  memset(&tm_v, 0, sizeof(tm_v));
  memset(&tma_w, 0, sizeof(tma_w));
  memset(&tma_m, 0, sizeof(tma_m));
  memset(&tma_v, 0, sizeof(tma_v));
  {
    const uint64_t d = static_cast<uint64_t>(a->dim), c = static_cast<uint64_t>(a->n_classes), k = static_cast<uint64_t>(K);
    const uint64_t hs = static_cast<uint64_t>(a->head_stride) * 4;
    if (make_tmap_3d(&tm_w, a->W, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d, c, k, d * 4, hs, 128, 16, 1)) return 1;
    if (make_tmap_3d(&tm_m, a->m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d, c, k, d * 4, hs, 128, 16, 1)) return 1;
    if (a->kind != 3 && make_tmap_3d(&tm_v, a->v, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, d, c, k, d * 4, hs, 128, 16, 1)) return 1;
    if (adapter) {
      const uint64_t dv = static_cast<uint64_t>(ad->img_dim), as = static_cast<uint64_t>(ad->adapter_stride) * 4;
      if (make_tmap_3d(&tma_w, ad->W, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dv, d, k, dv * 4, as, 128, 16, 1)) return 1;
      if (make_tmap_3d(&tma_m, ad->m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dv, d, k, dv * 4, as, 128, 16, 1)) return 1;
      if (a->kind != 3 && make_tmap_3d(&tma_v, ad->v, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, dv, d, k, dv * 4, as, 128, 16, 1))
        return 1;
    }
  }
  const int n_act = __builtin_popcount(mask);
  int64_t pos[2] = {a->pos[0], a->pos[1]};
  for (int i = 0; i < n_steps; ++i) {
    const int64_t n0 = rows[2 * i], n1 = rows[2 * i + 1], R = n0 + n1;
    UML_REQUIRE(n0 >= 0 && n1 >= 0 && R > 0 && R <= a->max_rows, "sweep_adapter_run: step %d has %lld rows (capacity %lld)", i,
                static_cast<long long>(R), static_cast<long long>(a->max_rows));
    UML_REQUIRE(!adapter || n0 <= ad->max_img_rows, "sweep_adapter_run: step %d has %lld image rows (Z holds %lld)", i,
                static_cast<long long>(n0), static_cast<long long>(ad->max_img_rows));
    for (int s = 0; s < 2; ++s) {
      const int64_t n = s ? n1 : n0;
      if (n == 0) continue;
      UML_REQUIRE(a->bank[s] && a->labels[s] && pos[s] >= 0 && pos[s] + n <= a->perm_len[s],
                  "sweep_adapter_run: step %d runs past the end of permutation %d", i, s);
      for (int k = 0; k < K; ++k)
        UML_REQUIRE(!((mask >> k) & 1u) || a->perm[s][k], "sweep_adapter_run: head %d has no permutation %d", k, s);
    }
    p.n0 = n0;
    p.n1 = n1;
    p.pos[0] = pos[0];
    p.pos[1] = pos[1];
    p.stats = a->stats + static_cast<int64_t>(i) * K * 2;
    const double t = static_cast<double>(a->step + i);
    const double bc1 = 1.0 - pow(static_cast<double>(a->beta1), t);
    const double bc2 = 1.0 - pow(static_cast<double>(a->beta2), t);
    p.bc2_sqrt_inv = static_cast<float>(1.0 / sqrt(bc2));
    p.first_step = (a->step + i) <= 1;
    for (int k = 0; k < K; ++k) {
      const float l = lr[static_cast<int64_t>(i) * K + k];
      p.lr[k] = l;
      p.step_size[k] = static_cast<float>(static_cast<double>(l) / bc1);
      p.decay[k] = static_cast<float>(1.0 - static_cast<double>(l) * static_cast<double>(a->weight_decay[k]));
    }
    const bool timed = i == n_steps - 1;
    auto mark = [&](int e) -> int {
      if (timed && ad->ev[e]) UML_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(ad->ev[e]), st));
      return 0;
    };
    const bool with_adapter = adapter && n0 > 0;
    // the adapter's side of the step: its rows are the image rows, its "classes" the head's input dims
    SweepDev pa = p;
    pa.zrows = nullptr;
    pa.scale_dev = nullptr;
    pa.n1 = 0;
    pa.bank[1] = nullptr;
    pa.dim = ad->img_dim;
    pa.n_classes = a->dim;
    pa.W = ad->W;
    pa.m = ad->m;
    pa.v = ad->v;
    pa.head_stride = ad->adapter_stride;
    pa.stats = nullptr;
    if (mark(0)) return 1;
    if (with_adapter) {  // Z_k = X_img Wp_k^T: the logits kernel without softmax, the adapter as its weight
      pa.G = ad->Z;
      pa.ldg = ad->ldz;
      pa.g_stride = ad->max_img_rows * ad->ldz;
      sweep_logits_tc_kernel<false><<<dim3(static_cast<unsigned>((a->dim + 127) / 128), 1, K), 256, kTcLgSmemBytes, st>>>(pa);
      UML_CUDA(cudaGetLastError());
      ++g_sweep_launches;
    }
    if (mark(1) || mark(2)) return 1;
    const unsigned n_ctile = static_cast<unsigned>((a->n_classes + 127) / 128);
    UML_CUDA(launch_kernel(sweep_logits_tc_kernel<true>, dim3(n_ctile, 1, K), dim3(256), kTcLgSmemBytes, st,
                           static_cast<int>(n_ctile), p));
    ++g_sweep_launches;
    if (mark(3) || mark(4)) return 1;
    if (with_adapter) {  // dZ from the head's weights before their update
      sweep_dz_tc_kernel<<<dim3(static_cast<unsigned>((a->dim + 127) / 128), K), 256, kTcDzSmemBytes, st>>>(p, ad->dZ, ad->ldz,
                                                                                                        ad->max_img_rows * ad->ldz);
      UML_CUDA(cudaGetLastError());
      ++g_sweep_launches;
    }
    if (mark(5) || mark(6)) return 1;
    {
      const int64_t units = static_cast<int64_t>(n_act) * ((a->dim + 127) / 128) * ((a->n_classes + 63) / 64);
      const unsigned g = static_cast<unsigned>(std::min<int64_t>(units, sm_count()));
      sweep_dw_update_tc_kernel<512><<<g, 512 + 64, kTcDwSmemBytes, st>>>(p, tm_w, tm_m, tm_v);
      UML_CUDA(cudaGetLastError());
      ++g_sweep_launches;
    }
    if (mark(7) || mark(8)) return 1;
    if (with_adapter) {  // dWp_k = dZ_k^T X_img with the update; the statistics warp is off (pa.stats == NULL)
      pa.G = ad->dZ;
      pa.ldg = ad->ldz;
      pa.g_stride = ad->max_img_rows * ad->ldz;
      const int64_t units = static_cast<int64_t>(n_act) * ((ad->img_dim + 127) / 128) * ((a->dim + 63) / 64);
      const unsigned g = static_cast<unsigned>(std::min<int64_t>(units, sm_count()));
      sweep_dw_update_tc_kernel<512><<<g, 512 + 64, kTcDwSmemBytes, st>>>(pa, tma_w, tma_m, tma_v);
      UML_CUDA(cudaGetLastError());
      ++g_sweep_launches;
    }
    if (mark(9)) return 1;
    if (dg && launch_grad_diag(p, dg, K, i, timed, st)) return 1;  // (Z is overwritten by the next step's first launch)
    pos[0] += n0;
    pos[1] += n1;
  }
  return 0;
}

int uml_sweep_adapter_run(const uml_sweep_args* a, const uml_sweep_adapter_args* ad, int32_t n_steps, const int64_t* rows,
                          const float* lr, void* stream) {
  return sweep_adapter_run_impl(a, ad, nullptr, n_steps, rows, lr, stream);
}

int uml_sweep_run_diag(const uml_sweep_args* a, const uml_sweep_adapter_args* ad, const uml_sweep_diag* dg, int32_t n_steps,
                       const int64_t* rows, const float* lr, void* stream) {
  using namespace uml::sweep;
  UML_REQUIRE(a && dg && rows && lr && n_steps >= 0, "sweep_run_diag: null argument");
  const int K = a->n_heads;
  UML_REQUIRE(K >= 1 && K <= kMaxHeads, "sweep_run_diag: 1..%d heads", kMaxHeads);
  UML_REQUIRE(dg->out && dg->scratch, "sweep_run_diag: null diagnostics buffer");
  UML_REQUIRE(a->dim > 0 && a->dim % 4 == 0 && a->n_classes > 0, "sweep_run_diag: dim must be a multiple of 4");
  UML_REQUIRE(aligned16(a->W) && aligned16(a->m) && aligned16(a->v) && a->head_stride % 4 == 0 && aligned16(a->G) &&
                  a->ldg % 4 == 0,
              "sweep_run_diag: W, m, v, G must be 16-byte aligned with strides that are multiples of 4");
  for (int s = 0; s < 2; ++s)
    UML_REQUIRE(!a->bank[s] || (aligned16(a->bank[s]) && a->bank_ld[s] % 4 == 0),
                "sweep_run_diag: bank %d rows must be 16-byte aligned", s);
  if (ad && ad->img_dim > 0)
    UML_REQUIRE(aligned16(ad->Z) && ad->ldz % 4 == 0, "sweep_run_diag: Z must be 16-byte aligned with ldz a multiple of 4");
  for (int k = 0; k < K; ++k)  // G's text rows carry alpha: the plain text-loss gradient is G / alpha
    UML_REQUIRE(!a->active[k] || !a->bank[1] || a->alpha[k] > 0.f,
                "sweep_run_diag: head %d has alpha %g <= 0, its text-loss gradient cannot be recovered", k,
                static_cast<double>(a->alpha[k]));
  const int64_t need = uml_sweep_diag_scratch_floats(K, a->dim, a->n_classes);
  UML_REQUIRE(dg->scratch_floats >= need, "sweep_run_diag: scratch holds %lld floats, %lld needed",
              static_cast<long long>(dg->scratch_floats), static_cast<long long>(need));
  return ad ? sweep_adapter_run_impl(a, ad, dg, n_steps, rows, lr, stream) : sweep_run_impl(a, dg, n_steps, rows, lr, stream);
}

}  // extern "C"
