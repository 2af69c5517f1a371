// a-14 - the linear analogue of the UML step: Gaussian_experiment's SharedAutoencoder
// (reference Gaussian_experiment/model.py:5-49, loop body main.py:47-59).
//
//   recon_m = out_head_m( dec( enc( in_head_m(v_m) ) ) ),   enc/dec = Linear-ReLU-Linear SHARED by both
//   modalities, per-modality in/out heads (all with bias); loss = alpha_x MSE(x) + alpha_y MSE(y) ("xy") or
//   MSE(x) alone ("x": the y heads get no gradient and Adam never touches them); Adam(lr), torch defaults.
//
// The model has ~29 k parameters and the reference batch is 512 rows per modality: the step is pure latency.
// Two launches per step, nothing else:
//   gauss_fwd_bwd_kernel  grid (tiles, 2 modalities): a CTA stages its branch's weights in shared memory
//                         (rows padded to an odd stride, conflict-free in both GEMM directions), gathers its
//                         16 rows by index (UnpairedDataset's `idx % len`), runs the six layers forward, the MSE,
//                         the six layers backward, and writes its weight-gradient contribution to its own slot
//                         of a partial buffer (no atomics: the reduction order is fixed);
//   gauss_update_kernel   sums the slots in a fixed order (shared layers: both modalities), applies Adam, and
//                         reduces the per-tile losses into the step's {loss_x, loss_y} record.
#include <cmath>

#include "common.cuh"

namespace uml {

constexpr int kGaussRows = 16;      // batch rows per CTA
constexpr int kGaussThreads = 256;

struct GaussLayout {
  int obs, com, lat;
  // offsets (floats) into the flat parameter buffer, reference construction order, weight then bias
  int in_w[2], in_b[2], e0_w, e0_b, e2_w, e2_b, d0_w, d0_b, d2_w, d2_b, out_w[2], out_b[2], total;
};

static GaussLayout make_layout(int obs, int com, int lat) {
  GaussLayout L;
  L.obs = obs; L.com = com; L.lat = lat;
  int o = 0;
  auto take = [&](int n) { int r = o; o += n; return r; };
  for (int m = 0; m < 2; ++m) { L.in_w[m] = take(com * obs); L.in_b[m] = take(com); }
  L.e0_w = take(lat * com); L.e0_b = take(lat);
  L.e2_w = take(lat * lat); L.e2_b = take(lat);
  L.d0_w = take(lat * lat); L.d0_b = take(lat);
  L.d2_w = take(com * lat); L.d2_b = take(com);
  for (int m = 0; m < 2; ++m) { L.out_w[m] = take(obs * com); L.out_b[m] = take(obs); }
  L.total = o;
  return L;
}

// ---- shared-memory helpers (all called by the whole CTA) -----------------------------------------------
// Activations live TRANSPOSED in shared memory, [feature][row] with a row stride of kLdA = R + 4 floats: the 16 rows
// of a feature are four float4, and consecutive features sit 80 B apart so that a quarter warp's 16-byte accesses
// fall into distinct bank groups.  Every helper gives a thread 8 (or 16) independent accumulators - the first
// version had one dependent FMA chain per thread and ran at ~5 MAC/cycle/SM (72 us per step).
constexpr int kLdA = kGaussRows + 4;

// W [out, in] global row-major -> shared with leading dimension in + 1
__device__ void stage_weight(const float* __restrict__ g, float* s, int out, int in) {
  for (int i = threadIdx.x; i < out * in; i += blockDim.x) s[(i / in) * (in + 1) + (i % in)] = g[i];
}
__device__ __forceinline__ void fma8(float (&a)[8], float w, const float4& x0, const float4& x1) {
  a[0] = fmaf(w, x0.x, a[0]); a[1] = fmaf(w, x0.y, a[1]); a[2] = fmaf(w, x0.z, a[2]); a[3] = fmaf(w, x0.w, a[3]);
  a[4] = fmaf(w, x1.x, a[4]); a[5] = fmaf(w, x1.y, a[5]); a[6] = fmaf(w, x1.z, a[6]); a[7] = fmaf(w, x1.w, a[7]);
}
// y[j][r] = b[j] + sum_k W[j][k] x[k][r]      thread -> (output feature j, half of the 16 rows)
template <bool kRelu>
__device__ void dense_fwd(const float* x, const float* W, const float* b, int in, int out, float* y, float* y_relu) {
  for (int o = threadIdx.x; o < 2 * out; o += blockDim.x) {
    const int j = o >> 1, h = (o & 1) * 8;
    const float* w = W + j * (in + 1);
    float a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = b[j];
#pragma unroll 4
    for (int k = 0; k < in; ++k) {
      const float4* xr = reinterpret_cast<const float4*>(x + k * kLdA + h);
      fma8(a, w[k], xr[0], xr[1]);
    }
    float4* yo = reinterpret_cast<float4*>(y + j * kLdA + h);
    yo[0] = make_float4(a[0], a[1], a[2], a[3]);
    yo[1] = make_float4(a[4], a[5], a[6], a[7]);
    if (kRelu) {
      float4* ro = reinterpret_cast<float4*>(y_relu + j * kLdA + h);
      ro[0] = make_float4(fmaxf(a[0], 0.f), fmaxf(a[1], 0.f), fmaxf(a[2], 0.f), fmaxf(a[3], 0.f));
      ro[1] = make_float4(fmaxf(a[4], 0.f), fmaxf(a[5], 0.f), fmaxf(a[6], 0.f), fmaxf(a[7], 0.f));
    }
  }
}
// dx[k][r] = sum_j W[j][k] dy[j][r]   (optionally masked by pre[k][r] > 0: the ReLU in front of this layer's input)
__device__ void dense_bwd_data(const float* dy, const float* W, int in, int out, float* dx, const float* pre) {
  for (int o = threadIdx.x; o < 2 * in; o += blockDim.x) {
    const int k = o >> 1, h = (o & 1) * 8;
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int j = 0; j < out; ++j) {
      const float4* dr = reinterpret_cast<const float4*>(dy + j * kLdA + h);
      fma8(a, W[j * (in + 1) + k], dr[0], dr[1]);
    }
    if (pre) {
      const float* pr = pre + k * kLdA + h;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (!(pr[i] > 0.f)) a[i] = 0.f;
    }
    float4* xo = reinterpret_cast<float4*>(dx + k * kLdA + h);
    xo[0] = make_float4(a[0], a[1], a[2], a[3]);
    xo[1] = make_float4(a[4], a[5], a[6], a[7]);
  }
}
// gW[j][k] = sum_r dy[j][r] x[k][r],  gb[j] = sum_r dy[j][r]   -> this CTA's slot of the partial buffer
__device__ void dense_bwd_weight(const float* dy, const float* x, int in, int out, float* __restrict__ gW,
                                 float* __restrict__ gb) {
  for (int o = threadIdx.x; o < out * in; o += blockDim.x) {
    const int j = o / in, k = o - j * in;
    const float4* d = reinterpret_cast<const float4*>(dy + j * kLdA);
    const float4* xv = reinterpret_cast<const float4*>(x + k * kLdA);
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int q = 0; q < kGaussRows / 4; ++q) {
      const float4 dd = d[q], xx = xv[q];
      a0 = fmaf(dd.x, xx.x, a0); a1 = fmaf(dd.y, xx.y, a1); a2 = fmaf(dd.z, xx.z, a2); a3 = fmaf(dd.w, xx.w, a3);
    }
    gW[o] = (a0 + a1) + (a2 + a3);
  }
  for (int j = threadIdx.x; j < out; j += blockDim.x) {
    const float4* d = reinterpret_cast<const float4*>(dy + j * kLdA);
    float a = 0.f;
#pragma unroll
    for (int q = 0; q < kGaussRows / 4; ++q) a += (d[q].x + d[q].y) + (d[q].z + d[q].w);
    gb[j] = a;
  }
}

struct GaussData {
  const float* data[2];   // [n_m, obs] row-major
  int64_t n[2];
  const int64_t* idx;     // [B] sampler indices (nullptr: dense rows 0..B-1, evaluation)
  int64_t B;
  float dscale[2];        // alpha_m * 2 / (B * obs); 0 => no gradient for that modality (forward + loss only)
};

// One CTA of the step: modality m, rows [tile * 16, tile * 16 + 16) of the batch.  `partial` and `loss_part` are the
// run's own buffers.  The single-run kernel and the group kernel both run this body, so a run of a group computes
// exactly what it computes alone.
__device__ __forceinline__ void gauss_fwd_bwd_cta(const float* __restrict__ P, const GaussLayout& L, const GaussData& D,
                                                  float* __restrict__ partial, float* __restrict__ loss_part, int m,
                                                  int tile, int n_tiles) {
  extern __shared__ __align__(16) float sm[];
  const int obs = L.obs, com = L.com, lat = L.lat;
  constexpr int R = kGaussRows;
  // ---- carve shared memory
  float* p = sm;
  auto carve = [&](int n) { float* r = p; p += (n + 3) & ~3; return r; };  // 16-byte aligned pieces (float4 access)
  float* Win = carve(com * (obs + 1));  float* bin = carve(com);
  float* We0 = carve(lat * (com + 1));  float* be0 = carve(lat);
  float* We2 = carve(lat * (lat + 1));  float* be2 = carve(lat);
  float* Wd0 = carve(lat * (lat + 1));  float* bd0 = carve(lat);
  float* Wd2 = carve(com * (lat + 1));  float* bd2 = carve(com);
  float* Wout = carve(obs * (com + 1)); float* bout = carve(obs);
  // activations, transposed: [feature][kLdA]
  float* v = carve(obs * kLdA);    // input rows
  float* a0 = carve(com * kLdA);   // in_head output
  float* h1 = carve(lat * kLdA);   float* r1 = carve(lat * kLdA);
  float* z = carve(lat * kLdA);    // latent
  float* h2 = carve(lat * kLdA);   float* r2 = carve(lat * kLdA);
  float* a3 = carve(com * kLdA);   // decoder output
  float* dr = carve(obs * kLdA);   // recon, then d recon
  float* dA = carve(com * kLdA);   // gradient scratch (wide)
  float* dB = carve(lat * kLdA);   // gradient scratch (narrow)
  float* dC = carve(lat * kLdA);
  __shared__ float red[kGaussThreads / 32];

  stage_weight(P + L.in_w[m], Win, com, obs);
  stage_weight(P + L.e0_w, We0, lat, com);
  stage_weight(P + L.e2_w, We2, lat, lat);
  stage_weight(P + L.d0_w, Wd0, lat, lat);
  stage_weight(P + L.d2_w, Wd2, com, lat);
  stage_weight(P + L.out_w[m], Wout, obs, com);
  for (int i = threadIdx.x; i < com; i += blockDim.x) { bin[i] = P[L.in_b[m] + i]; bd2[i] = P[L.d2_b + i]; }
  for (int i = threadIdx.x; i < lat; i += blockDim.x) { be0[i] = P[L.e0_b + i]; be2[i] = P[L.e2_b + i]; bd0[i] = P[L.d0_b + i]; }
  for (int i = threadIdx.x; i < obs; i += blockDim.x) bout[i] = P[L.out_b[m] + i];
  const int64_t row0 = static_cast<int64_t>(tile) * R;
  for (int i = threadIdx.x; i < R * obs; i += blockDim.x) {
    const int r = i / obs, c = i - r * obs;  // coalesced over the features of a row
    float x = 0.f;
    if (row0 + r < D.B) {
      const int64_t src = (D.idx ? D.idx[row0 + r] : row0 + r) % D.n[m];  // UnpairedDataset.__getitem__: idx % len
      x = D.data[m][src * obs + c];
    }
    v[c * kLdA + r] = x;
  }
  __syncthreads();

  // ---- forward
  dense_fwd<false>(v, Win, bin, obs, com, a0, nullptr);     __syncthreads();
  dense_fwd<true>(a0, We0, be0, com, lat, h1, r1);          __syncthreads();
  dense_fwd<false>(r1, We2, be2, lat, lat, z, nullptr);     __syncthreads();
  dense_fwd<true>(z, Wd0, bd0, lat, lat, h2, r2);           __syncthreads();
  dense_fwd<false>(r2, Wd2, bd2, lat, com, a3, nullptr);    __syncthreads();
  dense_fwd<false>(a3, Wout, bout, com, obs, dr, nullptr);  __syncthreads();

  // ---- loss (sum of squares of this tile) and d recon
  float ss = 0.f;
  const float ds = D.dscale[m];
  for (int i = threadIdx.x; i < R * obs; i += blockDim.x) {
    const int c = i / R, r = i - c * R;
    const bool valid = row0 + r < D.B;
    const float diff = valid ? dr[c * kLdA + r] - v[c * kLdA + r] : 0.f;
    ss = fmaf(diff, diff, ss);
    dr[c * kLdA + r] = diff * ds;
  }
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kGaussThreads / 32; ++w) t += red[w];
    loss_part[m * n_tiles + tile] = t;
  }
  if (ds == 0.f) return;  // forward-only modality ("x" mode's y branch, evaluation)

  // ---- backward: every layer writes its gradient slot, then propagates
  float* g = partial + (static_cast<int64_t>(m) * n_tiles + tile) * L.total;
  dense_bwd_weight(dr, a3, com, obs, g + L.out_w[m], g + L.out_b[m]);
  dense_bwd_data(dr, Wout, com, obs, dA, nullptr);             __syncthreads();   // d a3
  dense_bwd_weight(dA, r2, lat, com, g + L.d2_w, g + L.d2_b);
  dense_bwd_data(dA, Wd2, lat, com, dB, h2);                   __syncthreads();   // d h2
  dense_bwd_weight(dB, z, lat, lat, g + L.d0_w, g + L.d0_b);
  dense_bwd_data(dB, Wd0, lat, lat, dC, nullptr);              __syncthreads();   // d latent
  dense_bwd_weight(dC, r1, lat, lat, g + L.e2_w, g + L.e2_b);
  dense_bwd_data(dC, We2, lat, lat, dB, h1);                   __syncthreads();   // d h1
  dense_bwd_weight(dB, a0, com, lat, g + L.e0_w, g + L.e0_b);
  dense_bwd_data(dB, We0, com, lat, dA, nullptr);              __syncthreads();   // d a0
  dense_bwd_weight(dA, v, obs, com, g + L.in_w[m], g + L.in_b[m]);
}

__global__ void __launch_bounds__(kGaussThreads)
    gauss_fwd_bwd_kernel(const float* __restrict__ P, GaussLayout L, GaussData D, float* __restrict__ partial,
                         float* __restrict__ loss_part) {
  gauss_fwd_bwd_cta(P, L, D, partial, loss_part, blockIdx.y, blockIdx.x, gridDim.x);
}

struct GaussAdam {
  float beta1, beta2, one_m_b1, one_m_b2, eps, step_size, bc2_sqrt_inv;
};

// Parameter i of one run (and, in block 0, the run's {loss_x, loss_y} record); shared by the single-run and group kernels
__device__ __forceinline__ void gauss_update_elem(float* __restrict__ P, float* __restrict__ M, float* __restrict__ V,
                                                  const GaussLayout& L, const float* __restrict__ partial, int n_tiles,
                                                  int grad_x, int grad_y, const GaussAdam& A,
                                                  const float* __restrict__ loss_part, float inv_count,
                                                  float* __restrict__ loss_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (blockIdx.x == 0 && threadIdx.x < 2 && loss_out) {  // {loss_x, loss_y} of this step, fixed summation order
    float t = 0.f;
    for (int k = 0; k < n_tiles; ++k) t += loss_part[threadIdx.x * n_tiles + k];
    loss_out[threadIdx.x] = t * inv_count;
  }
  if (i >= L.total || !P) return;
  // which modalities contribute to parameter i: heads belong to one, the shared encoder/decoder to both
  bool use[2] = {grad_x != 0, grad_y != 0};
  if (i < L.in_w[1]) use[1] = false;                                   // in_head_x
  else if (i < L.e0_w) use[0] = false;                                 // in_head_y
  else if (i >= L.out_w[0] && i < L.out_w[1]) use[1] = false;          // out_head_x
  else if (i >= L.out_w[1]) use[0] = false;                            // out_head_y
  if (!use[0] && !use[1]) return;                                      // no gradient: Adam leaves it untouched
  float g = 0.f;
  for (int m = 0; m < 2; ++m)
    if (use[m])
      for (int k = 0; k < n_tiles; ++k) g += partial[(static_cast<int64_t>(m) * n_tiles + k) * L.total + i];
  float mm = M[i], vv = V[i];
  mm = mm + (g - mm) * A.one_m_b1;
  vv = vv * A.beta2 + A.one_m_b2 * g * g;
  M[i] = mm;
  V[i] = vv;
  P[i] = P[i] - A.step_size * (mm / (sqrtf(vv) * A.bc2_sqrt_inv + A.eps));
}

__global__ void __launch_bounds__(256)
    gauss_update_kernel(float* __restrict__ P, float* __restrict__ M, float* __restrict__ V, GaussLayout L,
                        const float* __restrict__ partial, int n_tiles, int grad_x, int grad_y, GaussAdam A,
                        const float* __restrict__ loss_part, float inv_count, float* __restrict__ loss_out) {
  gauss_update_elem(P, M, V, L, partial, n_tiles, grad_x, grad_y, A, loss_part, inv_count, loss_out);
}

static size_t gauss_smem_bytes(const GaussLayout& L) {
  const int obs = L.obs, com = L.com, lat = L.lat, R = kGaussRows;
  size_t f = static_cast<size_t>(com) * (obs + 1) + com + static_cast<size_t>(lat) * (com + 1) + lat +
             2 * (static_cast<size_t>(lat) * (lat + 1) + lat) + static_cast<size_t>(com) * (lat + 1) + com +
             static_cast<size_t>(obs) * (com + 1) + obs;
  f += static_cast<size_t>(R + 4) * (2 * obs + 3 * com + 7 * lat) + 4 * 32;  // + alignment slack of the carve
  return f * sizeof(float);
}

// gradient scale of each modality's MSE; "x" mode: loss = loss_x (no alpha), the y branch only reports its loss
// (main.py:52-54)
static void gauss_dscale(int32_t mode_xy, float alpha_x, float alpha_y, double cnt, float* dscale) {
  dscale[0] = static_cast<float>((mode_xy ? alpha_x : 1.0) * 2.0 / cnt);
  dscale[1] = mode_xy ? static_cast<float>(alpha_y * 2.0 / cnt) : 0.f;
}

static GaussAdam gauss_adam(double lr, double beta1, double beta2, double eps, int64_t step) {
  GaussAdam A;
  const double t = static_cast<double>(step);
  A.beta1 = static_cast<float>(beta1);
  A.beta2 = static_cast<float>(beta2);
  A.one_m_b1 = static_cast<float>(1.0 - beta1);
  A.one_m_b2 = static_cast<float>(1.0 - beta2);
  A.eps = static_cast<float>(eps);
  A.step_size = static_cast<float>(lr / (1.0 - std::pow(beta1, t)));
  A.bc2_sqrt_inv = static_cast<float>(1.0 / std::sqrt(1.0 - std::pow(beta2, t)));
  return A;
}

static int gauss_launch_fwd_bwd(const float* P, const GaussLayout& L, const GaussData& D, float* partial, float* loss_part,
                                cudaStream_t st) {
  const size_t smem = gauss_smem_bytes(L);
  UML_REQUIRE(smem <= 220 * 1024, "gauss: model too wide for the shared-memory resident kernel (%zu B)", smem);
  static size_t attr = 0;
  if (smem > attr) {
    UML_CUDA(cudaFuncSetAttribute(gauss_fwd_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
    attr = smem;
  }
  const int tiles = static_cast<int>((D.B + kGaussRows - 1) / kGaussRows);
  gauss_fwd_bwd_kernel<<<dim3(tiles, 2), kGaussThreads, smem, st>>>(P, L, D, partial, loss_part);
  UML_CUDA(cudaGetLastError());
  return 0;
}

// ---- lock-step group of runs (uml_gauss_group_run): the run is grid dimension z of the forward/backward launch and y of
// the update launch; each CTA runs the single-run body on its run's slab row, batch and buffers.
constexpr int kGaussMaxRuns = UML_GAUSS_GROUP_MAX_RUNS;

struct GaussGroupLaunch {
  GaussData d[kGaussMaxRuns];      // run k: rows, index batch (nullptr: dense validation rows), gradient scales
  float step_size[kGaussMaxRuns];  // Adam lr / (1 - beta1^t) of run k
  int32_t slot[kGaussMaxRuns];     // grid index -> run (active runs only)
};

__global__ void __launch_bounds__(kGaussThreads)
    gauss_group_fwd_bwd_kernel(const float* __restrict__ P, int64_t stride, GaussLayout L, GaussGroupLaunch G,
                               float* __restrict__ partial, float* __restrict__ loss_part) {
  const int k = G.slot[blockIdx.z];
  const int64_t n_tiles = gridDim.x;
  const GaussData D = G.d[k];
  gauss_fwd_bwd_cta(P + k * stride, L, D, partial ? partial + k * 2 * n_tiles * L.total : nullptr,
                    loss_part + k * 2 * n_tiles, blockIdx.y, blockIdx.x, gridDim.x);
}

// P == nullptr: losses only (validation); run k's {loss_x, loss_y} go to loss_out + k * loss_stride
__global__ void __launch_bounds__(256)
    gauss_group_update_kernel(float* __restrict__ P, float* __restrict__ M, float* __restrict__ V, int64_t stride,
                              GaussLayout L, const float* __restrict__ partial, int n_tiles, GaussGroupLaunch G,
                              GaussAdam A, const float* __restrict__ loss_part, float inv_count,
                              float* __restrict__ loss_out, int loss_stride) {
  const int k = G.slot[blockIdx.y];
  A.step_size = G.step_size[k];
  const int64_t w = P ? k * stride : 0;
  gauss_update_elem(P ? P + w : nullptr, M ? M + w : nullptr, V ? V + w : nullptr, L,
                    partial ? partial + static_cast<int64_t>(k) * 2 * n_tiles * L.total : nullptr, n_tiles,
                    G.d[k].dscale[0] != 0.f, G.d[k].dscale[1] != 0.f, A, loss_part + k * 2 * n_tiles, inv_count,
                    loss_out + k * loss_stride);
}

static int gauss_group_launch_fwd_bwd(const float* P, int64_t stride, const GaussLayout& L, const GaussGroupLaunch& G,
                                      int n_active, int64_t rows, float* partial, float* loss_part, cudaStream_t st) {
  const size_t smem = gauss_smem_bytes(L);
  static size_t attr = 0;
  if (smem > attr) {
    UML_CUDA(cudaFuncSetAttribute(gauss_group_fwd_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(smem)));
    attr = smem;
  }
  const int tiles = static_cast<int>((rows + kGaussRows - 1) / kGaussRows);
  gauss_group_fwd_bwd_kernel<<<dim3(tiles, 2, n_active), kGaussThreads, smem, st>>>(P, stride, L, G, partial, loss_part);
  UML_CUDA(cudaGetLastError());
  return 0;
}

// byte offsets of the pieces of a group's workspace (each 256-byte aligned); n_val = 0: no probe scratch
struct GaussGroupWs {
  int64_t partial, loss_part, val_part, emb_x, emb_y, cka, knn, totals, total;
};

static GaussGroupWs gauss_group_ws(int n_runs, const GaussLayout& L, int64_t batch, int64_t n_val, int topk) {
  GaussGroupWs W;
  int64_t o = 0;
  auto take = [&](int64_t bytes) { const int64_t r = o; o += (bytes + 255) & ~int64_t(255); return r; };
  const int64_t K = n_runs, tiles = (batch + kGaussRows - 1) / kGaussRows, vtiles = (n_val + kGaussRows - 1) / kGaussRows;
  const int64_t d2 = 2 * static_cast<int64_t>(L.lat);
  W.partial = take(K * 2 * tiles * L.total * 4);
  W.loss_part = take(K * 2 * tiles * 4);
  W.val_part = take(K * 2 * vtiles * 4);
  W.emb_x = take(K * n_val * L.lat * 4);
  W.emb_y = take(K * n_val * L.lat * 4);
  W.cka = take(n_val ? K * (d2 + 8 * d2 * d2) * 8 : 0);
  W.knn = take(K * 2 * n_val * topk * 4);
  W.totals = take(n_val ? K * 4 : 0);
  W.total = o;
  return W;
}

int gauss_group_alignment(const float* params, int64_t stride, int dim_obs, int dim_common, int dim_latent,
                          const float* const* val_x, const float* const* val_y, int64_t n, int topk, const int32_t* slots,
                          int n_active, int n_runs, float* emb_x, float* emb_y, double* cka_ws, int32_t* knn_ws,
                          int32_t* totals, float* out, cudaStream_t st);  // probes.cu

}  // namespace uml

extern "C" {

int uml_gauss_param_count(int32_t dim_obs, int32_t dim_common, int32_t dim_latent) {
  return uml::make_layout(dim_obs, dim_common, dim_latent).total;
}

int uml_gauss_workspace_floats(int32_t dim_obs, int32_t dim_common, int32_t dim_latent, int64_t batch) {
  const int64_t tiles = (batch + uml::kGaussRows - 1) / uml::kGaussRows;
  return static_cast<int>(2 * tiles * uml::make_layout(dim_obs, dim_common, dim_latent).total + 2 * tiles);
}

int uml_gauss_step(float* params, float* adam_m, float* adam_v, int32_t dim_obs, int32_t dim_common, int32_t dim_latent,
                   const float* data_x, int64_t n_x, const float* data_y, int64_t n_y, const int64_t* idx, int64_t batch,
                   int32_t mode_xy, float alpha_x, float alpha_y, double lr, double beta1, double beta2, double eps,
                   int64_t step, float* workspace, float* loss_out, void* stream) {
  using namespace uml;
  UML_REQUIRE(params && adam_m && adam_v && data_x && data_y && idx && workspace && batch > 0 && n_x > 0 && n_y > 0 && step >= 1,
              "gauss_step: bad arguments");
  const GaussLayout L = make_layout(dim_obs, dim_common, dim_latent);
  const int tiles = static_cast<int>((batch + kGaussRows - 1) / kGaussRows);
  float* partial = workspace;
  float* loss_part = workspace + static_cast<int64_t>(2) * tiles * L.total;
  GaussData D;
  D.data[0] = data_x; D.data[1] = data_y;
  D.n[0] = n_x; D.n[1] = n_y;
  D.idx = idx;
  D.B = batch;
  const double cnt = static_cast<double>(batch) * dim_obs;
  gauss_dscale(mode_xy, alpha_x, alpha_y, cnt, D.dscale);
  int rc = gauss_launch_fwd_bwd(params, L, D, partial, loss_part, as_stream(stream));
  if (rc) return rc;
  const GaussAdam A = gauss_adam(lr, beta1, beta2, eps, step);
  gauss_update_kernel<<<(L.total + 255) / 256, 256, 0, as_stream(stream)>>>(
      params, adam_m, adam_v, L, partial, tiles, D.dscale[0] != 0.f, D.dscale[1] != 0.f, A, loss_part,
      static_cast<float>(1.0 / cnt), loss_out);
  UML_CUDA(cudaGetLastError());
  return 0;
}

// n_steps consecutive steps enqueued by one call (the step is latency bound and a Python round trip per step costs more
// than its two kernels): idx_list[i] is step i's device index batch, loss_log + 2 i receives its {loss_x, loss_y}.
int uml_gauss_run(float* params, float* adam_m, float* adam_v, int32_t dim_obs, int32_t dim_common, int32_t dim_latent,
                  const float* data_x, int64_t n_x, const float* data_y, int64_t n_y, const int64_t* const* idx_list,
                  int32_t n_steps, int64_t batch, int32_t mode_xy, float alpha_x, float alpha_y, double lr, double beta1,
                  double beta2, double eps, int64_t first_step, float* workspace, float* loss_log, void* stream) {
  UML_REQUIRE(idx_list && n_steps >= 0 && loss_log, "gauss_run: bad arguments");
  for (int i = 0; i < n_steps; ++i) {
    const int rc = uml_gauss_step(params, adam_m, adam_v, dim_obs, dim_common, dim_latent, data_x, n_x, data_y, n_y,
                                  idx_list[i], batch, mode_xy, alpha_x, alpha_y, lr, beta1, beta2, eps, first_step + i,
                                  workspace, loss_log + 2 * i, stream);
    if (rc) return rc;
  }
  return 0;
}

// forward + MSE of both modalities over dense rows (validation, main.py:68-72): loss_out = {loss_x, loss_y}
int uml_gauss_eval(const float* params, int32_t dim_obs, int32_t dim_common, int32_t dim_latent, const float* data_x,
                   const float* data_y, int64_t n_rows, float* workspace, float* loss_out, void* stream) {
  using namespace uml;
  UML_REQUIRE(params && data_x && data_y && workspace && loss_out && n_rows > 0, "gauss_eval: bad arguments");
  const GaussLayout L = make_layout(dim_obs, dim_common, dim_latent);
  const int tiles = static_cast<int>((n_rows + kGaussRows - 1) / kGaussRows);
  GaussData D;
  D.data[0] = data_x; D.data[1] = data_y;
  D.n[0] = D.n[1] = n_rows;
  D.idx = nullptr;
  D.B = n_rows;
  D.dscale[0] = D.dscale[1] = 0.f;
  float* loss_part = workspace;  // 2 * tiles floats
  int rc = gauss_launch_fwd_bwd(params, L, D, nullptr, loss_part, as_stream(stream));
  if (rc) return rc;
  GaussAdam A;
  memset(&A, 0, sizeof(A));
  gauss_update_kernel<<<1, 256, 0, as_stream(stream)>>>(nullptr, nullptr, nullptr, L, nullptr, tiles, 0, 0, A, loss_part,
                                                         static_cast<float>(1.0 / (static_cast<double>(n_rows) * dim_obs)),
                                                         loss_out);
  UML_CUDA(cudaGetLastError());
  return 0;
}

int64_t uml_gauss_group_workspace_bytes(int32_t n_runs, int32_t dim_obs, int32_t dim_common, int32_t dim_latent,
                                        int64_t batch, int64_t n_val, int32_t topk) {
  return uml::gauss_group_ws(n_runs, uml::make_layout(dim_obs, dim_common, dim_latent), batch, n_val, topk).total;
}

int uml_gauss_group_run(const uml_gauss_group_args* a, int32_t n_steps, const int64_t* const* idx, void* stream) {
  using namespace uml;
  UML_REQUIRE(a && idx && n_steps >= 0, "gauss_group_run: null argument");
  const int K = a->n_runs;
  UML_REQUIRE(K >= 1 && K <= kGaussMaxRuns, "gauss_group_run: 1..%d runs (got %d)", kGaussMaxRuns, K);
  UML_REQUIRE(a->dim_obs > 0 && a->dim_common > 0 && a->dim_latent > 0 && a->batch > 0 && a->n_x > 0 && a->n_y > 0,
              "gauss_group_run: bad shape");
  UML_REQUIRE(a->data_x && a->data_y && a->params && a->adam_m && a->adam_v && a->loss_log && a->workspace,
              "gauss_group_run: null buffer");
  const GaussLayout L = make_layout(a->dim_obs, a->dim_common, a->dim_latent);
  UML_REQUIRE(a->param_stride >= L.total, "gauss_group_run: param_stride %lld is below the %d parameters of a run",
              static_cast<long long>(a->param_stride), L.total);
  UML_REQUIRE(a->first_step >= 1, "gauss_group_run: first_step must be >= 1");
  UML_REQUIRE(a->eval_every >= 0 && a->eval_phase >= 0, "gauss_group_run: eval_every and eval_phase must be >= 0");
  const size_t smem = gauss_smem_bytes(L);
  UML_REQUIRE(smem <= 220 * 1024, "gauss_group_run: model too wide for the shared-memory resident kernel (%zu B)", smem);
  const bool probes = a->eval_every > 0;
  int32_t slots[kGaussMaxRuns];
  int n_active = 0;
  for (int k = 0; k < K; ++k) {
    UML_REQUIRE(a->mode_xy[k] == 0 || a->mode_xy[k] == 1, "gauss_group_run: run %d: mode_xy must be 0 or 1", k);
    if (!a->active[k]) continue;
    slots[n_active++] = k;
    if (probes)
      UML_REQUIRE(a->val_x[k] && a->val_y[k], "gauss_group_run: run %d has no validation rows", k);
  }
  if (probes) {
    UML_REQUIRE(a->eval_log, "gauss_group_run: null eval_log");
    UML_REQUIRE(a->n_val >= 2 && a->topk >= 1 && a->topk <= 64 && a->topk < a->n_val,
                "gauss_group_run: probes need n_val >= 2 and 1 <= topk <= min(64, n_val - 1)");
    UML_REQUIRE((static_cast<size_t>(a->n_val) + a->dim_latent) * sizeof(float) <= 200 * 1024,
                "gauss_group_run: at most ~50 000 validation rows (a row's similarities live in shared memory)");
    UML_REQUIRE(128 * static_cast<size_t>(a->dim_common + a->dim_latent) * sizeof(float) <= 200 * 1024,
                "gauss_group_run: dim_common + dim_latent too large for the embedding kernel's per-thread scratch");
  }
  const GaussGroupWs W = gauss_group_ws(K, L, a->batch, probes ? a->n_val : 0, probes ? a->topk : 0);
  UML_REQUIRE(a->workspace_bytes >= W.total, "gauss_group_run: workspace holds %lld bytes, %lld needed",
              static_cast<long long>(a->workspace_bytes), static_cast<long long>(W.total));
  UML_REQUIRE((reinterpret_cast<uintptr_t>(a->workspace) & 15) == 0, "gauss_group_run: workspace must be 16-byte aligned");
  for (int i = 0; i < n_steps; ++i)
    for (int z = 0; z < n_active; ++z)
      UML_REQUIRE(idx[static_cast<int64_t>(i) * K + slots[z]], "gauss_group_run: step %d has no index batch for run %d", i,
                  slots[z]);
  if (n_active == 0 || n_steps == 0) return 0;

  cudaStream_t st = as_stream(stream);
  char* ws = static_cast<char*>(a->workspace);
  float* partial = reinterpret_cast<float*>(ws + W.partial);
  float* loss_part = reinterpret_cast<float*>(ws + W.loss_part);
  const int tiles = static_cast<int>((a->batch + kGaussRows - 1) / kGaussRows);
  const double cnt = static_cast<double>(a->batch) * a->dim_obs;
  GaussGroupLaunch G, V;
  memset(&G, 0, sizeof(G));
  memset(&V, 0, sizeof(V));
  for (int k = 0; k < K; ++k) {
    G.d[k].data[0] = a->data_x; G.d[k].data[1] = a->data_y;
    G.d[k].n[0] = a->n_x; G.d[k].n[1] = a->n_y;
    G.d[k].B = a->batch;
    gauss_dscale(a->mode_xy[k], a->alpha_x[k], a->alpha_y[k], cnt, G.d[k].dscale);
    V.d[k].data[0] = a->val_x[k]; V.d[k].data[1] = a->val_y[k];
    V.d[k].n[0] = V.d[k].n[1] = a->n_val;
    V.d[k].B = a->n_val;  // idx nullptr, dscale 0: forward + MSE over dense rows (uml_gauss_eval)
  }
  for (int z = 0; z < n_active; ++z) G.slot[z] = V.slot[z] = slots[z];
  const int64_t stride = a->param_stride;
  int64_t evals = 0;
  for (int i = 0; i < n_steps; ++i) {
    const GaussAdam A = gauss_adam(a->lr[0], a->beta1, a->beta2, a->eps, a->first_step + i);
    for (int k = 0; k < K; ++k) {
      G.d[k].idx = a->active[k] ? idx[static_cast<int64_t>(i) * K + k] : nullptr;
      G.step_size[k] = gauss_adam(a->lr[k], a->beta1, a->beta2, a->eps, a->first_step + i).step_size;
    }
    int rc = gauss_group_launch_fwd_bwd(a->params, stride, L, G, n_active, a->batch, partial, loss_part, st);
    if (rc) return rc;
    gauss_group_update_kernel<<<dim3((L.total + 255) / 256, n_active), 256, 0, st>>>(
        a->params, a->adam_m, a->adam_v, stride, L, partial, tiles, G, A, loss_part, static_cast<float>(1.0 / cnt),
        a->loss_log + static_cast<int64_t>(i) * K * 2, 2);
    UML_CUDA(cudaGetLastError());
    if (!probes || (a->eval_phase + i + 1) % a->eval_every != 0) continue;
    // probes of the weights after this step's update: validation losses, then the alignment of the embeddings
    float* out = a->eval_log + evals++ * K * 4;
    float* val_part = reinterpret_cast<float*>(ws + W.val_part);
    rc = gauss_group_launch_fwd_bwd(a->params, stride, L, V, n_active, a->n_val, nullptr, val_part, st);
    if (rc) return rc;
    GaussAdam none;
    memset(&none, 0, sizeof(none));
    gauss_group_update_kernel<<<dim3(1, n_active), 256, 0, st>>>(
        nullptr, nullptr, nullptr, stride, L, nullptr, static_cast<int>((a->n_val + kGaussRows - 1) / kGaussRows), V, none,
        val_part, static_cast<float>(1.0 / (static_cast<double>(a->n_val) * a->dim_obs)), out, 4);
    UML_CUDA(cudaGetLastError());
    rc = gauss_group_alignment(a->params, stride, a->dim_obs, a->dim_common, a->dim_latent, a->val_x, a->val_y, a->n_val,
                               a->topk, slots, n_active, K, reinterpret_cast<float*>(ws + W.emb_x),
                               reinterpret_cast<float*>(ws + W.emb_y), reinterpret_cast<double*>(ws + W.cka),
                               reinterpret_cast<int32_t*>(ws + W.knn), reinterpret_cast<int32_t*>(ws + W.totals), out, st);
    if (rc) return rc;
  }
  return 0;
}

}  // extern "C"
