// Alignment probes on the device (SURVEY section 8 f-3): the two diagnostics the reference logs next to its training
// loops - linear CKA with the biased HSIC estimator and mutual k-nearest-neighbour accuracy
// (vision_language/metrics.py:55-119,252-285, identical file under Gaussian_experiment/; called at
// Gaussian_experiment/main.py:67-84 every EVAL_EVERY steps and at vision_language/finetune.py:209-233) - plus the
// embedding forward of the Gaussian experiment's autoencoder they are computed on (model.py:51-60 get_embeddings).
//
// The reference builds n x n kernel matrices on the host (O(n^2 d + n^3) for CKA: K H L H with dense n x n products).
// Here:
//   * linear CKA in its O(n d^2) form: for linear kernels trace(K H L H) = || A_c^T B_c ||_F^2 with column-centred
//     features, so the three HSIC terms are squared Frobenius norms of (d_a + d_b)^2 centred Gram entries - column means,
//     then tiles of the Gram matrix accumulated in fp64 over row splits, then one fixed-order finishing CTA.  No n x n
//     matrix ever exists.
//   * mutual kNN: one CTA per row computes that row's n inner products into shared memory and extracts the top-k by k
//     block-wide arg-max passes (ties: lower index); a second small launch intersects the two k-lists per row and one
//     finishing thread turns the integer total into the mean.
// Diagnostics, not the hot path: plain SIMT kernels, sized for n <= ~12 000 rows and widths up to a few thousand.
#include <cfloat>

#include "common.cuh"

namespace uml {

constexpr int kProbeSplits = 8;   // row splits of the Gram accumulation (fp64 partials, summed in split order)

// Every probe kernel's body is a device function of its CTA coordinates: the single-call kernels below and the group
// kernels (one more grid dimension over the runs of a Gaussian group) run the same code in the same order.
__device__ __forceinline__ void col_mean_cta(const float* __restrict__ A, int64_t lda, int da, const float* __restrict__ B,
                                             int64_t ldb, int db, int64_t n, double* __restrict__ mean, int c) {
  __shared__ double sh[256];
  const float* X = c < da ? A + c : B + (c - da);
  const int64_t ld = c < da ? lda : ldb;
  double s = 0.0;
  for (int64_t r = threadIdx.x; r < n; r += blockDim.x) s += static_cast<double>(X[r * ld]);
  sh[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) mean[c] = sh[0] / static_cast<double>(n);
}

__global__ void __launch_bounds__(256)
    probe_col_mean_kernel(const float* __restrict__ A, int64_t lda, int da, const float* __restrict__ B, int64_t ldb, int db,
                          int64_t n, double* __restrict__ mean) {
  col_mean_cta(A, lda, da, B, ldb, db, n, mean, blockIdx.x);
}

// Z = [A | B] (d = da + db columns), centred: part[split][i][j] = sum over the split's rows of Zc[r][i] * Zc[r][j]
__device__ __forceinline__ void gram_tile_cta(const float* __restrict__ A, int64_t lda, int da, const float* __restrict__ B,
                                              int64_t ldb, int db, int64_t n, const double* __restrict__ mean,
                                              double* __restrict__ part, int tile_i, int tile_j, int split) {
  constexpr int T = 16, R = 64;
  __shared__ float zi[R][T + 1], zj[R][T + 1];
  const int d = da + db;
  const int i0 = tile_i * T, j0 = tile_j * T;
  if (j0 + T <= i0) return;  // the Gram matrix is symmetric: only tiles that touch the upper triangle are computed
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t per = (n + kProbeSplits - 1) / kProbeSplits, r_lo = per * split, r_hi = r_lo + per < n ? r_lo + per : n;
  double acc = 0.0;
  for (int64_t r0 = r_lo; r0 < r_hi; r0 += R) {
    for (int e = threadIdx.x; e < R * T; e += 256) {
      const int rr = e / T, cc = e % T;
      const int64_t r = r0 + rr;
      float vi = 0.f, vj = 0.f;
      if (r < r_hi) {
        const int ci = i0 + cc, cj = j0 + cc;
        if (ci < d) vi = (ci < da ? A[r * lda + ci] : B[r * ldb + ci - da]) - static_cast<float>(mean[ci]);
        if (cj < d) vj = (cj < da ? A[r * lda + cj] : B[r * ldb + cj - da]) - static_cast<float>(mean[cj]);
      }
      zi[rr][cc] = vi;
      zj[rr][cc] = vj;
    }
    __syncthreads();
#pragma unroll 8
    for (int rr = 0; rr < R; ++rr) acc += static_cast<double>(zi[rr][ty]) * static_cast<double>(zj[rr][tx]);
    __syncthreads();
  }
  const int i = i0 + ty, j = j0 + tx;
  if (i < d && j < d) part[(static_cast<int64_t>(split) * d + i) * d + j] = acc;
}

__global__ void __launch_bounds__(256)
    probe_gram_kernel(const float* __restrict__ A, int64_t lda, int da, const float* __restrict__ B, int64_t ldb, int db,
                      int64_t n, const double* __restrict__ mean, double* __restrict__ part) {
  gram_tile_cta(A, lda, da, B, ldb, db, n, mean, part, blockIdx.x, blockIdx.y, blockIdx.z);
}

// kl = sum G_ab^2, kk = sum G_aa^2, ll = sum G_bb^2 (fixed order) -> out[0] = kl / (sqrt(kk * ll) + 1e-6)
__device__ __forceinline__ void cka_finish_cta(const double* __restrict__ part, int da, int db, float* __restrict__ out) {
  __shared__ double sh[3][1024];
  const int d = da + db;
  double kk = 0.0, ll = 0.0, kl = 0.0;
  for (int64_t e = threadIdx.x; e < static_cast<int64_t>(d) * d; e += blockDim.x) {
    const int i = static_cast<int>(e / d), j = static_cast<int>(e % d);
    if (j < i) continue;  // upper triangle only: the two diagonal blocks are symmetric, the A x B block lies above the diagonal
    double g = 0.0;
    for (int s = 0; s < kProbeSplits; ++s) g += part[(static_cast<int64_t>(s) * d + i) * d + j];
    const double g2 = g * g;
    if (j < da) {
      kk += (i == j) ? g2 : 2.0 * g2;
    } else if (i >= da) {
      ll += (i == j) ? g2 : 2.0 * g2;
    } else {
      kl += g2;
    }
  }
  sh[0][threadIdx.x] = kk;
  sh[1][threadIdx.x] = ll;
  sh[2][threadIdx.x] = kl;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
      sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
      sh[2][threadIdx.x] += sh[2][threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = static_cast<float>(sh[2][0] / (sqrt(sh[0][0] * sh[1][0]) + 1e-6));
}

__global__ void __launch_bounds__(1024)
    probe_cka_finish_kernel(const double* __restrict__ part, int da, int db, float* __restrict__ out) {
  cka_finish_cta(part, da, db, out);
}

// top-k inner-product neighbours of row i (self excluded the reference's way: its similarity is set to -1e8)
__device__ __forceinline__ void knn_row_cta(const float* __restrict__ X, int64_t ld, int d, int64_t n, int k,
                                            int32_t* __restrict__ idx_out, int64_t i) {
  extern __shared__ float sims[];  // [n] then the row itself [d]
  float* xi = sims + n;
  __shared__ float bv[8];
  __shared__ int bi[8];
  for (int c = threadIdx.x; c < d; c += blockDim.x) xi[c] = X[i * ld + c];
  __syncthreads();
  for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
    const float* xj = X + j * ld;
    float s = 0.f;
    for (int c = 0; c < d; ++c) s = fmaf(xi[c], xj[c], s);
    sims[j] = j == i ? -1e8f : s;
  }
  __syncthreads();
  for (int t = 0; t < k; ++t) {
    float best = -FLT_MAX;
    int arg = 0x7fffffff;
    for (int64_t j = threadIdx.x; j < n; j += blockDim.x) {
      const float v = sims[j];
      if (v > best || (v == best && static_cast<int>(j) < arg)) { best = v; arg = static_cast<int>(j); }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
      if (ov > best || (ov == best && oa < arg)) { best = ov; arg = oa; }
    }
    if ((threadIdx.x & 31) == 0) { bv[threadIdx.x >> 5] = best; bi[threadIdx.x >> 5] = arg; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int w = 1; w < 8; ++w)
        if (bv[w] > best || (bv[w] == best && bi[w] < arg)) { best = bv[w]; arg = bi[w]; }
      idx_out[i * k + t] = arg;
      if (arg >= 0 && arg < n) sims[arg] = -FLT_MAX;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256)
    probe_knn_kernel(const float* __restrict__ X, int64_t ld, int d, int64_t n, int k, int32_t* __restrict__ idx_out) {
  knn_row_cta(X, ld, d, n, k, idx_out, blockIdx.x);
}

__device__ __forceinline__ void knn_count_block(const int32_t* __restrict__ ka, const int32_t* __restrict__ kb, int64_t n,
                                                int k, int32_t* __restrict__ total) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  int c = 0;
  if (i < n) {
    for (int a = 0; a < k; ++a) {
      const int va = ka[i * k + a];
      for (int b = 0; b < k; ++b) c += (kb[i * k + b] == va) ? 1 : 0;
    }
  }
  c = warp_sum_i(c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(total, c);  // integer sum: order does not matter
}

__global__ void __launch_bounds__(256)
    probe_knn_count_kernel(const int32_t* __restrict__ ka, const int32_t* __restrict__ kb, int64_t n, int k, int32_t* __restrict__ total) {
  knn_count_block(ka, kb, n, k, total);
}

__device__ __forceinline__ float knn_mean(int32_t total, int64_t n, int k) {
  return static_cast<float>(static_cast<double>(total) / (static_cast<double>(n) * k));
}

__global__ void probe_knn_finish_kernel(const int32_t* __restrict__ total, int64_t n, int k, float* __restrict__ out) {
  out[0] = knn_mean(total[0], n, k);
}

// latent = shared_encoder(in_head(row)) for both modalities of the Gaussian experiment (model.py:51-60): one thread per row
__device__ __forceinline__ void gauss_embed_row(const float* __restrict__ params, int dim_obs, int dim_common, int dim_latent,
                                                const float* __restrict__ data_x, const float* __restrict__ data_y,
                                                int64_t n_rows, float* __restrict__ emb_x, float* __restrict__ emb_y,
                                                int mod /* 0: x, 1: y */) {
  extern __shared__ float scratch[];  // per thread: dim_common + dim_latent floats
  const int64_t row = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const float* data = mod == 0 ? data_x : data_y;
  float* emb = mod == 0 ? emb_x : emb_y;
  if (!data || !emb || row >= n_rows) return;
  // flat parameter layout (weight then bias per layer): in_head_x, in_head_y, shared_encoder.0, shared_encoder.2, ...
  const int64_t in_sz = static_cast<int64_t>(dim_common) * dim_obs + dim_common;
  const float* Win = params + mod * in_sz;
  const float* bin = Win + static_cast<int64_t>(dim_common) * dim_obs;
  const float* W0 = params + 2 * in_sz;
  const float* b0 = W0 + static_cast<int64_t>(dim_latent) * dim_common;
  const float* W2 = b0 + dim_latent;
  const float* b2 = W2 + static_cast<int64_t>(dim_latent) * dim_latent;
  float* z = scratch + static_cast<int64_t>(threadIdx.x) * (dim_common + dim_latent);
  float* h = z + dim_common;
  const float* x = data + row * dim_obs;
  for (int o = 0; o < dim_common; ++o) {
    float s = __ldg(bin + o);
    for (int c = 0; c < dim_obs; ++c) s = fmaf(__ldg(Win + static_cast<int64_t>(o) * dim_obs + c), x[c], s);
    z[o] = s;
  }
  for (int o = 0; o < dim_latent; ++o) {
    float s = __ldg(b0 + o);
    for (int c = 0; c < dim_common; ++c) s = fmaf(__ldg(W0 + static_cast<int64_t>(o) * dim_common + c), z[c], s);
    h[o] = fmaxf(s, 0.f);
  }
  for (int o = 0; o < dim_latent; ++o) {
    float s = __ldg(b2 + o);
    for (int c = 0; c < dim_latent; ++c) s = fmaf(__ldg(W2 + static_cast<int64_t>(o) * dim_latent + c), h[c], s);
    emb[row * dim_latent + o] = s;
  }
}

__global__ void __launch_bounds__(128)
    gauss_embed_kernel(const float* __restrict__ params, int dim_obs, int dim_common, int dim_latent, const float* __restrict__ data_x,
                       const float* __restrict__ data_y, int64_t n_rows, float* __restrict__ emb_x, float* __restrict__ emb_y) {
  gauss_embed_row(params, dim_obs, dim_common, dim_latent, data_x, data_y, n_rows, emb_x, emb_y, blockIdx.y);
}

// ---- the same probes for the runs of a Gaussian group (uml_gauss_group_run): the run is one more grid dimension and
// every buffer has a run stride.  Run k's embeddings are emb_x / emb_y + k n d, its CKA scratch cka_ws + k (d2 + 8 d2^2)
// with d2 = 2 d, its neighbour lists knn_ws + k 2 n topk (x, then y) and its neighbour count totals[k].
__host__ __device__ __forceinline__ int64_t cka_ws_doubles(int64_t d) { return d + kProbeSplits * d * d; }

struct GaussProbeRuns {
  const float* val_x[UML_GAUSS_GROUP_MAX_RUNS];
  const float* val_y[UML_GAUSS_GROUP_MAX_RUNS];
  int32_t slot[UML_GAUSS_GROUP_MAX_RUNS];  // grid index -> run
};

__global__ void __launch_bounds__(128)
    gauss_group_embed_kernel(const float* __restrict__ params, int64_t stride, int dim_obs, int dim_common, int dim_latent,
                             GaussProbeRuns R, int64_t n, float* __restrict__ emb_x, float* __restrict__ emb_y) {
  const int k = R.slot[blockIdx.z];
  const int64_t e = static_cast<int64_t>(k) * n * dim_latent;
  gauss_embed_row(params + k * stride, dim_obs, dim_common, dim_latent, R.val_x[k], R.val_y[k], n, emb_x + e, emb_y + e,
                  blockIdx.y);
}

__global__ void __launch_bounds__(256)
    probe_group_col_mean_kernel(const float* __restrict__ emb_x, const float* __restrict__ emb_y, int d, int64_t n,
                                double* __restrict__ cka_ws, GaussProbeRuns R) {
  const int k = R.slot[blockIdx.y];
  const int64_t e = static_cast<int64_t>(k) * n * d;
  col_mean_cta(emb_x + e, d, d, emb_y + e, d, d, n, cka_ws + k * cka_ws_doubles(2 * d), blockIdx.x);
}

__global__ void __launch_bounds__(256)
    probe_group_gram_kernel(const float* __restrict__ emb_x, const float* __restrict__ emb_y, int d, int64_t n,
                            double* __restrict__ cka_ws, GaussProbeRuns R) {
  const int k = R.slot[blockIdx.z / kProbeSplits];
  const int64_t e = static_cast<int64_t>(k) * n * d;
  double* ws = cka_ws + k * cka_ws_doubles(2 * d);
  gram_tile_cta(emb_x + e, d, d, emb_y + e, d, d, n, ws, ws + 2 * d, blockIdx.x, blockIdx.y, blockIdx.z % kProbeSplits);
}

__global__ void __launch_bounds__(256)
    probe_group_knn_kernel(const float* __restrict__ emb_x, const float* __restrict__ emb_y, int d, int64_t n, int topk,
                           int32_t* __restrict__ knn_ws, GaussProbeRuns R) {
  const int k = R.slot[blockIdx.z];
  const int64_t e = static_cast<int64_t>(k) * n * d;
  knn_row_cta((blockIdx.y == 0 ? emb_x : emb_y) + e, d, d, n, topk, knn_ws + (2 * static_cast<int64_t>(k) + blockIdx.y) * n * topk,
              blockIdx.x);
}

__global__ void __launch_bounds__(256)
    probe_group_knn_count_kernel(const int32_t* __restrict__ knn_ws, int64_t n, int topk, int32_t* __restrict__ totals,
                                 GaussProbeRuns R) {
  const int k = R.slot[blockIdx.y];
  const int32_t* ka = knn_ws + 2 * static_cast<int64_t>(k) * n * topk;
  knn_count_block(ka, ka + n * topk, n, topk, totals + k);
}

// out[k][2] = CKA, out[k][3] = mutual kNN of run k (out[k][0..1] hold its validation losses)
__global__ void __launch_bounds__(1024)
    probe_group_finish_kernel(const double* __restrict__ cka_ws, int d, const int32_t* __restrict__ totals, int64_t n,
                              int topk, float* __restrict__ out, GaussProbeRuns R) {
  const int k = R.slot[blockIdx.x];
  cka_finish_cta(cka_ws + k * cka_ws_doubles(2 * d) + 2 * d, d, d, out + 4 * k + 2);
  if (threadIdx.x == 0) out[4 * k + 3] = knn_mean(totals[k], n, topk);
}

// Embeddings, CKA and mutual kNN of the validation rows of the active runs `slots[0..n_active)` of a Gaussian group
// (arguments checked by the caller): five launches and a memset for all runs.
int gauss_group_alignment(const float* params, int64_t stride, int dim_obs, int dim_common, int dim_latent,
                          const float* const* val_x, const float* const* val_y, int64_t n, int topk, const int32_t* slots,
                          int n_active, int n_runs, float* emb_x, float* emb_y, double* cka_ws, int32_t* knn_ws,
                          int32_t* totals, float* out, cudaStream_t st) {
  GaussProbeRuns R;
  memset(&R, 0, sizeof(R));
  for (int k = 0; k < UML_GAUSS_GROUP_MAX_RUNS; ++k) { R.val_x[k] = val_x[k]; R.val_y[k] = val_y[k]; }
  for (int z = 0; z < n_active; ++z) R.slot[z] = slots[z];
  const unsigned na = static_cast<unsigned>(n_active);
  const size_t embed_smem = 128 * static_cast<size_t>(dim_common + dim_latent) * sizeof(float);
  static size_t embed_attr = 0;
  if (embed_smem > 48 * 1024 && embed_smem > embed_attr) {
    UML_CUDA(cudaFuncSetAttribute(gauss_group_embed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    embed_attr = 200 * 1024;
  }
  gauss_group_embed_kernel<<<dim3(static_cast<unsigned>((n + 127) / 128), 2, na), 128, embed_smem, st>>>(
      params, stride, dim_obs, dim_common, dim_latent, R, n, emb_x, emb_y);
  UML_CUDA(cudaGetLastError());
  const int d2 = 2 * dim_latent;
  probe_group_col_mean_kernel<<<dim3(d2, na), 256, 0, st>>>(emb_x, emb_y, dim_latent, n, cka_ws, R);
  UML_CUDA(cudaGetLastError());
  const unsigned tiles = static_cast<unsigned>((d2 + 15) / 16);
  probe_group_gram_kernel<<<dim3(tiles, tiles, kProbeSplits * na), 256, 0, st>>>(emb_x, emb_y, dim_latent, n, cka_ws, R);
  UML_CUDA(cudaGetLastError());
  const size_t knn_smem = (static_cast<size_t>(n) + dim_latent) * sizeof(float);
  static size_t knn_attr = 0;
  if (knn_smem > 48 * 1024 && knn_smem > knn_attr) {
    UML_CUDA(cudaFuncSetAttribute(probe_group_knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    knn_attr = 200 * 1024;
  }
  UML_CUDA(cudaMemsetAsync(totals, 0, n_runs * sizeof(int32_t), st));
  probe_group_knn_kernel<<<dim3(static_cast<unsigned>(n), 2, na), 256, knn_smem, st>>>(emb_x, emb_y, dim_latent, n, topk,
                                                                                      knn_ws, R);
  UML_CUDA(cudaGetLastError());
  probe_group_knn_count_kernel<<<dim3(static_cast<unsigned>((n + 255) / 256), na), 256, 0, st>>>(knn_ws, n, topk, totals, R);
  UML_CUDA(cudaGetLastError());
  probe_group_finish_kernel<<<na, 1024, 0, st>>>(cka_ws, dim_latent, totals, n, topk, out, R);
  UML_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace uml

extern "C" {

int64_t uml_cka_workspace_doubles(int32_t da, int32_t db) {
  return uml::cka_ws_doubles(static_cast<int64_t>(da) + db);
}

int uml_cka_linear_f32(const float* A, int64_t lda, int32_t da, const float* B, int64_t ldb, int32_t db, int64_t n, double* ws,
                       float* out, void* stream) {
  using namespace uml;
  UML_REQUIRE(A && B && ws && out && n >= 2 && da >= 1 && db >= 1 && lda >= da && ldb >= db, "cka_linear: bad arguments");
  const int d = da + db;
  cudaStream_t st = as_stream(stream);
  double* mean = ws;
  double* part = ws + d;
  probe_col_mean_kernel<<<d, 256, 0, st>>>(A, lda, da, B, ldb, db, n, mean);
  UML_CUDA(cudaGetLastError());
  const unsigned tiles = static_cast<unsigned>((d + 15) / 16);
  probe_gram_kernel<<<dim3(tiles, tiles, kProbeSplits), 256, 0, st>>>(A, lda, da, B, ldb, db, n, mean, part);
  UML_CUDA(cudaGetLastError());
  probe_cka_finish_kernel<<<1, 1024, 0, st>>>(part, da, db, out);
  UML_CUDA(cudaGetLastError());
  return 0;
}

int uml_mutual_knn_f32(const float* A, int64_t lda, int32_t da, const float* B, int64_t ldb, int32_t db, int64_t n, int32_t topk,
                       int32_t* ws /* 2 * n * topk + 1 */, float* out, void* stream) {
  using namespace uml;
  UML_REQUIRE(A && B && ws && out && n >= 2 && da >= 1 && db >= 1 && topk >= 1 && topk < n && topk <= 64, "mutual_knn: bad arguments");
  cudaStream_t st = as_stream(stream);
  int32_t *ka = ws, *kb = ws + n * topk, *total = ws + 2 * n * topk;
  const size_t smem_a = (static_cast<size_t>(n) + da) * sizeof(float), smem_b = (static_cast<size_t>(n) + db) * sizeof(float);
  UML_REQUIRE(smem_a <= 200 * 1024 && smem_b <= 200 * 1024, "mutual_knn: at most ~50 000 rows (a row's similarities live in shared memory)");
  static size_t attr = 0;
  const size_t need = smem_a > smem_b ? smem_a : smem_b;
  if (need > 48 * 1024 && need > attr) {
    UML_CUDA(cudaFuncSetAttribute(probe_knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = 200 * 1024;
  }
  UML_CUDA(cudaMemsetAsync(total, 0, sizeof(int32_t), st));
  probe_knn_kernel<<<static_cast<unsigned>(n), 256, smem_a, st>>>(A, lda, da, n, topk, ka);
  UML_CUDA(cudaGetLastError());
  probe_knn_kernel<<<static_cast<unsigned>(n), 256, smem_b, st>>>(B, ldb, db, n, topk, kb);
  UML_CUDA(cudaGetLastError());
  probe_knn_count_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(ka, kb, n, topk, total);
  UML_CUDA(cudaGetLastError());
  probe_knn_finish_kernel<<<1, 1, 0, st>>>(total, n, topk, out);
  UML_CUDA(cudaGetLastError());
  return 0;
}

int uml_gauss_embed(const float* params, int32_t dim_obs, int32_t dim_common, int32_t dim_latent, const float* data_x,
                    const float* data_y, int64_t n_rows, float* emb_x, float* emb_y, void* stream) {
  using namespace uml;
  UML_REQUIRE(params && n_rows > 0 && dim_obs > 0 && dim_common > 0 && dim_latent > 0 && (data_x || data_y), "gauss_embed: bad arguments");
  const size_t smem = 128 * static_cast<size_t>(dim_common + dim_latent) * sizeof(float);
  UML_REQUIRE(smem <= 200 * 1024, "gauss_embed: dim_common + dim_latent too large for the per-thread scratch");
  if (smem > 48 * 1024) UML_CUDA(cudaFuncSetAttribute(gauss_embed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  gauss_embed_kernel<<<dim3(static_cast<unsigned>((n_rows + 127) / 128), 2), 128, smem, as_stream(stream)>>>(
      params, dim_obs, dim_common, dim_latent, data_x, data_y, n_rows, emb_x, emb_y);
  UML_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
