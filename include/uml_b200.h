/*
 * uml_b200.h - C ABI of the B200-native UML hot path (libuml_b200.so).
 *
 * The reference (OEmiliatanO/Unpaired-Multimodal-Learning) has no FFI of its own: its hot path is
 * Python calling PyTorch library ops.  Each entry point below replaces one of those call sites
 * (cited as file:line relative to the reference root) with a hand-written sm_100a kernel.  The
 * boundary rules are those of SURVEY.md section 8(b): plain pointers and sizes, a cudaStream_t passed
 * as void*, int status (0 = ok, else call uml_last_error()), no allocation, no host sync and no
 * exceptions inside the library.  All pointers are DEVICE pointers unless a comment says "host".
 *
 * Two arithmetic families:
 *   *_f32   exact-path SIMT kernels (fp32 FFMA, like the reference which never enables TF32/AMP);
 *           used at the reference's own batch sizes (8..64 rows) where the step is latency bound.
 *   *_bf16  tcgen05/TMEM tensor-core kernels (bf16 operands, fp32 accumulate) fed by TMA; used at
 *           throughput batch sizes.  Tolerance vs the fp32 path is stated in tests/.
 */
#ifndef UML_B200_H_
#define UML_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UML_B200_ABI_VERSION 1
#define UML_MAX_SEGMENTS 2

/* A run of rows fed through the shared head in one step.  The reference builds two such runs per
 * step - the image batch and the unpaired text batch (vision_language/finetune.py:165-178) - and
 * pushes both through the same nn.Linear (engine/models/head.py:80-82,133-135). */
typedef struct {
  const void*    rows;        /* feature matrix base: fp32 for *_f32, bf16 for *_bf16 entry points   */
  const int64_t* idx;         /* optional gather indices into `rows`/`labels` (NULL = dense 0..n-1)   */
  const int64_t* labels;      /* class labels (bank labels when idx != NULL, else dense per row)      */
  int64_t        n;           /* rows in this run for this step (the last batch of an epoch is short) */
  int64_t        ld;          /* leading dimension of `rows`, in elements                             */
  float          scale;       /* logit scale: exp(logit_scale) (UMLClip) or img_scale / txt_scale     */
  float          loss_weight; /* 1.0 for the image run, alpha for the text run (finetune.py:188)      */
  const int64_t* label_idx;   /* optional: indices into `labels` when they differ from `idx` (adapter
                                 output rows are dense but their labels still live in the bank)        */
  const float*   scale_dev;   /* optional: device scalar overriding `scale` (learnable temperature,
                                 head.py:69-70) so the step never reads it back to the host            */
  const uint16_t* rows16;     /* optional: bf16 shadow of `rows` (same shape, ld == dim); the tensor-core step
                                 then gathers with plain TMA copies instead of converting fp32 rows     */
} uml_segment;

/* Per-run results written by the forward kernels (device memory, one per segment). */
typedef struct {
  float   loss_mean;   /* mean cross entropy over the run (F.cross_entropy default reduction)        */
  float   dscale;      /* d loss_mean / d scale  (used when the scales are learnable, head.py:69-70)  */
  int32_t correct;     /* rows whose argmax equals the label (finetune.py:197-198)                    */
  int32_t n;           /* rows counted                                                                */
} uml_seg_stats;

/* ---- library ------------------------------------------------------------------------------- */
const char* uml_last_error(void);            /* host string, valid until the next failing call     */
int         uml_abi_version(void);
int         uml_device_ok(int device);        /* 0 when `device` is an sm_100 part                  */

/* ---- K1  index-driven gather (replaces Dataset.__getitem__ + default_collate + .to(device),
 *          finetune.py:165-172, engine/datasets/utils.py:100-101) ---------------------------------- */
int uml_gather_rows_f32(const float* bank, int64_t bank_rows, int32_t dim, const int64_t* idx,
                        int64_t n, float* out, void* stream);
int uml_gather_rows_bf16(const float* bank, int64_t bank_rows, int32_t dim, const int64_t* idx,
                         int64_t n, uint16_t* out, int64_t ld_out, void* stream);
/* bf16 gather that also gathers the int64 bank labels of the same rows into int32 (one launch)         */
int uml_gather_rows_labels_bf16(const float* bank, const int64_t* bank_labels, int32_t dim, const int64_t* idx,
                                int64_t n, uint16_t* out, int64_t ld_out, int32_t* out_labels, void* stream);
/* Both runs of a step (image rows, then text rows) copied from bf16 shadow banks into one [n0+n1, dim] operand
 * in a single launch, with their labels (int64 bank labels -> int32).  Pure TMA data movement.            */
int uml_gather2_rows_bf16(const uint16_t* bank0, const int64_t* labels0, const int64_t* idx0, int64_t n0,
                          const uint16_t* bank1, const int64_t* labels1, const int64_t* idx1, int64_t n1, int32_t dim,
                          uint16_t* out, int64_t ld_out, int32_t* out_labels /* nullable */, void* stream);
/* The same copy with a small-footprint kernel (no shared memory, one warp per row) that can share the SMs with
 * the GEMM kernels of the current step: uml_linear_run issues it on a side stream for the NEXT step's rows.   */
int uml_gather2_rows_bf16_light(const uint16_t* bank0, const int64_t* labels0, const int64_t* idx0, int64_t n0,
                                const uint16_t* bank1, const int64_t* labels1, const int64_t* idx1, int64_t n1, int32_t dim,
                                uint16_t* out, int64_t ld_out, int32_t* out_labels /* nullable */, void* stream);
int uml_gather_labels_i32(const int64_t* bank_labels, const int64_t* idx, int64_t n, int32_t* out,
                          void* stream);
int uml_cast_f32_to_bf16(const float* src, uint16_t* dst, int64_t n, void* stream);

/* ---- K2+K3  head forward + logit scale + softmax cross entropy (head.py:80-82,133-135;
 *             finetune.py:186-188).  Writes G = loss_weight * scale / n * (softmax - onehot), the
 *             gradient of the weighted loss w.r.t. the raw (unscaled) logits, for the dW kernel.   */
int uml_head_fwd_ce_f32(const uml_segment* segs /*host*/, int32_t nseg, int32_t dim,
                        const float* W, int32_t n_classes, float* G, int64_t ldg,
                        float* row_loss, int32_t* row_correct, float* row_dscale,
                        uml_seg_stats* stats, int64_t g_capacity_rows /* rows G has room for; >= 2x the step's rows lets small
                           batches split the contraction over planes of G (0 = exactly the step's rows) */,
                        void* stream);

/* ---- K4  dW = G^T X (autograd of the above; finetune.py:190-193), optionally fused with the
 *          optimizer update so the gradient never round-trips HBM -------------------------------- */
typedef struct {
  int32_t kind;        /* 0 = write dW only, 1 = AdamW, 2 = Adam (L2), 3 = SGD momentum (L2)        */
  float   lr, beta1, beta2, eps, weight_decay, momentum;
  int64_t step;        /* 1-based step count for the bias corrections                               */
  float*  m;           /* exp_avg   | momentum buffer                                               */
  float*  v;           /* exp_avg_sq| unused                                                        */
} uml_update;

int uml_head_bwd_dw_f32(const uml_segment* segs /*host*/, int32_t nseg, int32_t dim,
                        const float* G, int64_t ldg, int32_t n_classes,
                        float* W, float* dW /*may be NULL when fused*/, const uml_update* upd /*host*/,
                        void* stream);

/* ---- the whole exact step of the reference's own batch sizes (8..64 rows per modality, engine/optimizer/default.py:8,24,39)
 *      in ONE cooperative launch: K2+K3 (head.py:131-137, finetune.py:186-188), K4 (autograd of the head, finetune.py:190-193)
 *      and the optimizer (optim.py:42-70), i.e. uml_head_fwd_ce_f32 followed by uml_head_bwd_dw_f32 with a fused update.
 *      *launched = 1 when the step ran; 0 (and nothing was launched) when the shape does not fit the kernel's contract -
 *      16-byte aligned rows, dim % 4 == 0, rows x dim floats of shared memory - and the caller takes the separate launches. */
int uml_head_step_fused_f32(const uml_segment* segs /*host*/, int32_t nseg, int32_t dim, float* W, int32_t n_classes,
                            float* G, int64_t ldg, float* row_loss, int32_t* row_correct, float* row_dscale,
                            uml_seg_stats* stats, const uml_update* upd /*host*/, int32_t* launched /*host*/, void* stream);
/* fused-step launches of this process so far (modulo 2^31): lets a caller that goes through uml_linear_step / uml_linear_run
 * count the kernels it launched (one per step instead of four when the fused kernel took the step) */
int uml_head_step_fused_count(void);

/* ---- K5  adapter GEMMs in fp32 (head.py:65,79 and their autograd) ---------------------------- */
/* C[m,n] = alpha * sum_k A[m,k] * B[n,k]        (both operands K-contiguous: nn.Linear forward)   */
int uml_gemm_nt_f32(const float* A, int64_t lda, const int64_t* a_row_idx, const float* B, int64_t ldb,
                    float* C, int64_t ldc, int64_t m, int64_t n, int64_t k, float alpha, void* stream);
/* C[m,n] = alpha * sum_k A[m,k] * B[k,n]        (dZ = G W)                                         */
int uml_gemm_nn_f32(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                    int64_t m, int64_t n, int64_t k, float alpha, void* stream);
/* C[m,n] = alpha * sum_k A[k,m] * B[k,n] (+ optimizer update of P when upd->kind != 0)            */
int uml_gemm_tn_f32(const float* A, int64_t lda, const float* B, int64_t ldb, const int64_t* b_row_idx,
                    float* C, int64_t ldc, int64_t m, int64_t n, int64_t k, float alpha,
                    float* P, const uml_update* upd /*host, may be NULL*/, void* stream);

/* ---- K6  fused optimizer updates (engine/optimizer/optim.py:15-71 -> torch.optim rules) ------ */
int uml_adamw_step(float* p, const float* g, const float* g2, float g2_weight, float* m, float* v,
                   int64_t n, double lr, double beta1, double beta2, double eps, double weight_decay,
                   int64_t step, int32_t decoupled, uint16_t* p_bf16 /*optional shadow*/, void* stream);
int uml_sgd_step(float* p, const float* g, const float* g2, float g2_weight, float* buf, int64_t n,
                 double lr, double momentum, double weight_decay, int64_t step,
                 uint16_t* p_bf16, void* stream);

/* ---- K7  evaluation: logits + argmax + per-row CE over a bank (finetune.py:291-315) ---------- */
int uml_eval_f32(const float* feats, int64_t ld, const int64_t* labels, int64_t n_rows, int32_t dim,
                 const float* W, int32_t n_classes, float scale,
                 float* row_loss, int32_t* row_pred, void* stream);
/* mean over reference batches of the batch-mean loss + hit count (finetune.py:310-312).
 * labels == NULL: row_pred already holds 0/1 hit flags (the tensor-core forward's row_correct).    */
int uml_eval_reduce(const float* row_loss, const int32_t* row_pred, const int64_t* labels, int64_t n_rows,
                    int64_t batch_size, float* out_loss /*[1]*/, int32_t* out_correct /*[1]*/, void* stream);

/* The same for the heads of a sweep group over ONE bank in one launch each (the reference's sweep loop calls validate once
 * per combination, finetune.py:406-448 + 291-315): head h reads its weights at W + head_ids[h] * w_stride (floats) and
 * fills rows [h * n_rows, (h + 1) * n_rows) of row_loss / row_pred; uml_eval_reduce_group writes out_loss[h] /
 * out_correct[h].  head_ids / scales: HOST arrays of n_heads <= 32 entries.                              */
int uml_eval_group_f32(const float* feats, int64_t ld, const int64_t* labels, int64_t n_rows, int32_t dim, const float* W,
                       int64_t w_stride, const int32_t* head_ids /*host*/, const float* scales /*host*/, int32_t n_heads,
                       int32_t n_classes, float* row_loss /*[n_heads, n_rows]*/, int32_t* row_pred /*[n_heads, n_rows]*/,
                       void* stream);
int uml_eval_reduce_group(const float* row_loss, const int32_t* row_pred, const int64_t* labels, int64_t n_rows,
                          int64_t batch_size, int32_t n_heads, float* out_loss /*[n_heads]*/,
                          int32_t* out_correct /*[n_heads]*/, void* stream);

/* ---- K8  gradient diagnostics (finetune.py:200-206): out = {dot, |a|^2, |b|^2, sign agreement} */
#define UML_DIAG_BLOCKS 296
int uml_grad_diag(const float* a, const float* b, int64_t n, float* workspace /* >= 4*UML_DIAG_BLOCKS floats */,
                  float* out4, void* stream);

/* ---- tensor-core path (tcgen05 + TMEM + TMA) --------------------------------------------------- */
/* X: [n_rows, dim] bf16 dense (ld = dim), W: [n_classes, dim] bf16.  Row r belongs to segment
 * 0 when r < seg0_rows, else 1.  G: [n_rows, ldg] bf16, ldg a multiple of 64 and >= n_classes.     */
typedef struct {
  int64_t seg_rows[UML_MAX_SEGMENTS];
  float   scale[UML_MAX_SEGMENTS];
  float   loss_weight[UML_MAX_SEGMENTS];
  int32_t nseg;
  const float* scale_dev[UML_MAX_SEGMENTS];   /* optional device scalars overriding scale[]        */
} uml_tc_segments;

int uml_head_fwd_ce_bf16(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W,
                         int32_t n_classes, const int32_t* labels, const uml_tc_segments* segs /*host*/,
                         uint16_t* G /*may be NULL: eval mode*/, int64_t ldg,
                         float* row_loss, int32_t* row_pred /*optional: argmax class*/,
                         int32_t* row_correct /*optional: argmax == label*/, float* row_dscale /*optional*/,
                         float* tile_ws /* [UML_TILE_WS_FLOATS(n_rows)] (required with G): per-tile partial sums
                                           of the per-run statistics, reduced by uml_reduce_tile_stats, then
                                           the per-row factors of the deferred softmax normalisation      */,
                         uml_seg_stats* stats /* optional, with G: per-run {mean loss, dscale, hits, rows} written by
                                                 the fix-up launch (saves the uml_reduce_tile_stats launch)     */,
                         void* stream);
#define UML_TILE_WS_FLOATS(n_rows) (16 + (((n_rows) + 255) / 256) * 264 + (n_rows) * 32)
/* tile_ws must be ZERO-INITIALISED when it is allocated (the exchange flags of the forward kernel are keyed by a launch
 * epoch kept in its first words).  1 when a forward launch on this workspace ever timed out waiting for a peer CTA pair
 * (its results are undefined): synchronises, meant for flush / evaluation cadence.                              */
int uml_fwd_x_failed(const float* tile_ws);
/* per-run {mean loss, dscale, hits, rows} from the forward kernel's per-tile partials (fixed order)     */
int uml_reduce_tile_stats(const float* tile_ws, int64_t n_rows, int32_t nseg, uml_seg_stats* stats, void* stream);
/* dW_partial[s] = (G^T X) over the s-th K split; partials: [n_splits, n_classes, dim] fp32.       */
int uml_head_bwd_dw_bf16(const uint16_t* G, int64_t ldg, const uint16_t* X, int64_t n_rows, int32_t dim,
                         int32_t n_classes, float* partials, int32_t n_splits, void* stream);
int uml_tc_dw_splits(int64_t n_rows, int32_t dim, int32_t n_classes);   /* suggested n_splits      */
/* Generic bf16 tcgen05 GEMM  D[m,n] = sum_k A(m,k) B(k,n)  (adapter: head.py:65,79 and its autograd).
 * a_mn_major = 0: A stored [M, K] (lda >= K);  1: A stored [K, M] (lda >= M).   Same for B with N.
 * out_bf16 = 1: D written as bf16 [M, ldo] (n_splits must be 1);  0: fp32 split-K partials
 * [n_splits, M, ldo].  Instantiated layouts: (1,1,fp32) (0,0,bf16) (0,1,bf16) (0,0,fp32).
 * M > 128 runs the MMA across CTA pairs (cta_group::2); env UML_TC_CTA_GROUP=1|2 overrides.          */
int uml_gemm_bf16(const uint16_t* A, int64_t lda, int32_t a_mn_major, const uint16_t* B, int64_t ldb,
                  int32_t b_mn_major, int64_t M, int64_t N, int64_t K, void* out, int64_t ldo,
                  int32_t out_bf16, int32_t n_splits, void* stream);
int uml_gemm_bf16_splits(int64_t M, int64_t N, int64_t K);               /* suggested n_splits      */
/* p -= update(sum_s partials[s]); also refreshes the bf16 shadow of p                             */
int uml_adamw_step_partials(float* p, const float* partials, int32_t n_splits, int64_t split_stride,
                            float* m, float* v, int64_t n, double lr, double beta1, double beta2,
                            double eps, double weight_decay, int64_t step, int32_t decoupled,
                            uint16_t* p_bf16, float* g_out /*optional: reduced gradient*/, void* stream);
/* out = sum_s partials[s] in a fixed order (local split-K reduction before a data-parallel allreduce) */
int uml_sum_partials(const float* partials, int32_t n_splits, int64_t split_stride, int64_t n, float* out,
                     void* stream);
int uml_reduce_seg_stats(const float* row_loss, const int32_t* row_correct, const float* row_dscale,
                         const int64_t* seg_rows /*host [nseg]*/, int32_t nseg, uml_seg_stats* stats,
                         void* stream);

/* ---- one whole UML iteration (finetune.py:163-195) enqueued by a single call --------------------
 * precision 0: fp32 SIMT path (rows gathered inside the GEMMs, update fused in the dW epilogue);
 * precision 1: bf16 tcgen05 path (TMA gather+cast -> fwd/CE/G -> split-K dW -> update + split reduce).
 * When dW_out != NULL the summed gradient is written there and W is left untouched (data parallel:
 * the caller all-reduces dW_out and then calls uml_adamw_step / uml_sgd_step).                      */
typedef struct {
  int32_t       dim, n_classes, nseg, precision;
  uml_segment   seg[UML_MAX_SEGMENTS];      /* fp32 banks + indices + labels + scale + loss weight     */
  float*        W;                          /* [n_classes, dim] shared head                            */
  uml_update    upd;                        /* optimizer kind, hyper-parameters, step, m, v for W      */
  void*         G;                          /* [rows, ldg] workspace: fp32 (precision 0) / bf16 (1)    */
  int64_t       ldg;
  float*        row_loss;  int32_t* row_correct;  float* row_dscale;   /* [rows] workspaces            */
  uml_seg_stats* stats;                     /* [nseg] per-run results of THIS step, stats[i] for seg[i] on
                                               both paths; a run with n == 0 gets {0, 0, 0, 0}, and its
                                               learnable temperature (scale_param[i]) is left untouched -
                                               no step, no decay, m and v kept - as torch.optim skips a
                                               parameter without a gradient (data-parallel mode excepted:
                                               there the zero record still joins the all-reduce)          */
  uint16_t*     X16;  uint16_t* W16;  int32_t* labels32;  float* partials;   /* bf16 path workspaces   */
  float*        tile_ws;                    /* [UML_TILE_WS_FLOATS(rows)], bf16 path                   */
  int32_t       max_splits;  int32_t w16_valid;
  float*        dW_out;                     /* optional, see above                                     */
  float*        dW_scratch;                 /* [n_classes*dim], only for SGD on the bf16 path          */
  float*        scale_param[UML_MAX_SEGMENTS];  /* learnable temperatures (device scalars) or NULL     */
  float*        scale_m[UML_MAX_SEGMENTS];  float* scale_v[UML_MAX_SEGMENTS];
  int64_t       scale_step[UML_MAX_SEGMENTS];
  /* optional cudaEvent_t pairs recorded around {gather, forward, dW, update} on `stream` (bench.py) */
  void*         ev[8];
  int32_t       dp_allreduce;               /* != 0: all-reduce dW_out across the uml_dp_init ranks, then update W */
  /* optional second operand buffers: with them uml_linear_run gathers step i+1's rows (into the buffer step i
   * does not use) on a side stream while step i's GEMMs run                                                  */
  uint16_t*     X16_alt;  int32_t* labels32_alt;
  int64_t       g_capacity_rows;            /* rows the G workspace has room for (fp32 path: split-K planes); 0 = rows */
  /* optional third operand buffers: the gather then runs two steps ahead (when a call has more than two steps), and
   * no forward kernel waits for an event of the side stream that is signalled at the last moment                     */
  uint16_t*     X16_alt2;  int32_t* labels32_alt2;
  /* optional cudaEvent_t after which every index batch of the call is valid in device memory (recorded by whoever
   * uploaded them).  With it - and the three operand buffers - uml_linear_run keeps its gather pipeline running through
   * the call boundaries: the first steps' rows are gathered beside the previous call's last steps.  NULL: every call
   * starts with a gather on `stream`.                                                                             */
  void*         idx_ready;
} uml_linear_step_args;

int uml_linear_step(const uml_linear_step_args* args /*host*/, void* stream);
/* call after anything else has used the operand buffers (X16, X16_alt, X16_alt2): the next uml_linear_run starts cold */
int uml_linear_run_reset(void);

/* Several consecutive iterations enqueued by one call (the host stays well ahead of the GPU: Python
 * dispatch, not the kernels, limited throughput when every step was a separate call).  `base` describes
 * the model/workspaces; `steps[i]` patches what changes from one iteration to the next.                */
typedef struct {
  const int64_t* idx[UML_MAX_SEGMENTS];          /* this step's index batches (views of the epoch permutation) */
  int64_t        n[UML_MAX_SEGMENTS];            /* rows per run (the last batch of an epoch is short)        */
  float          loss_weight[UML_MAX_SEGMENTS];
  float          lr;                             /* learning rate of this step (scheduler output)             */
  int64_t        opt_step;                       /* 1-based optimizer step of the head                        */
  int64_t        scale_step[UML_MAX_SEGMENTS];
  uml_seg_stats* stats;                          /* where this step's per-run results go                      */
  void*          ev[8];                          /* optional cudaEvent_t pairs, as uml_linear_step_args.ev    */
} uml_run_step;
int uml_linear_run(const uml_linear_step_args* base /*host*/, const uml_run_step* steps /*host*/, int32_t n_steps,
                   void* stream);

/* Per-step gradient diagnostics of a single run (the reference's probes, finetune.py:190-206): the image-loss and the
 * text-loss gradients of the head weights, A = X_img^T G[image rows] and B = X_txt^T G[text rows] / alpha, reduced on
 * the device to out = {sum A.B, sum A^2, sum B^2, #(sign A == sign B)} (torch.sign: 0 equals only 0), from the step's
 * own G and rows, i.e. at the weights before its update.  They only read, so the training results are bit-identical
 * to the same call without diagnostics.
 *   precision 0: G and the rows (seg[].rows / idx, dense when idx == NULL) through the sweep's 3xTF32 tensor-core
 *                diagnostics pass and its fixed-order finish: two launches after the step's last launch;
 *   precision 1: two split-K bf16 dW GEMMs over the image and the text rows of X16 and G into scratch, one launch that
 *                sums each side's partials in split order and reduces them into per-block slots, one fixed-order finish
 *                (up to four launches), after the step's dW launch and before its operand buffer is handed back to the
 *                gather pipeline of uml_linear_run.
 * The image run is seg[0] when has_img, the text run the remaining one; the image run's loss weight must be 1 (no
 * data parallelism).  Contract, checked before anything touches the device: dim % 4 == 0 (precision 1: % 8), 16-byte
 * aligned G and rows (X16 on precision 1) with leading dimensions that are multiples of 4 (ldg: 64 on precision 1),
 * loss weight (alpha) > 0 when there are text rows, no data-parallel all-reduce, scratch_floats >=
 * uml_linear_diag_scratch_floats(precision, rows of the largest step, dim, n_classes).                              */
typedef struct {
  float*   scratch;         /* device workspace                                                                  */
  int64_t  scratch_floats;
  int32_t  has_img;         /* seg[0] is the image run                                                           */
} uml_linear_diag;
int64_t uml_linear_diag_scratch_floats(int32_t precision, int64_t max_rows, int32_t dim, int32_t n_classes); /* a COUNT */
/* uml_linear_run with step i's diagnostics written to out[i] (device float[4])                                    */
int uml_linear_run_diag(const uml_linear_step_args* base /*host*/, const uml_run_step* steps /*host*/, int32_t n_steps,
                        const uml_linear_diag* diag /*host*/, float* const* out /*host [n_steps]*/, void* stream);
/* the diagnostics alone, of the step `args` describes whose G and rows (X16) are still in place: for the steps the
 * host dispatches kernel by kernel (adapter heads: seg[0].rows is the fp32 adapter output Z, or bf16 Z in X16)       */
int uml_linear_grad_diag(const uml_linear_step_args* args /*host*/, const uml_linear_diag* diag /*host*/, float* out,
                         void* stream);

/* ---- data parallel: NCCL all-reduce of the head gradient issued from inside the step --------------
 * uml_dp_unique_id fills a 128-byte NCCL id on one rank; every rank then calls uml_dp_init with it.
 * With args->dp_allreduce != 0 the step sums dW over the ranks (ncclAllReduce on `stream`) between the
 * dW kernel and the optimizer update, so a data-parallel iteration is still a single host call.          */
int uml_dp_unique_id(void* out_128_bytes /*host*/);
int uml_dp_init(const void* id_128_bytes /*host*/, int32_t rank, int32_t world);
int uml_dp_allreduce_f32(float* buf, int64_t n, void* stream);
int uml_dp_shutdown(void);
/* Two-shot all-reduce over NVLink peer memory for the head gradient (one node): every rank allocates an exchange
 * block (uml_dp_p2p_alloc -> 64-byte CUDA IPC handle), the handles are all-gathered by the caller and opened with
 * uml_dp_p2p_open; from then on a data-parallel step sums dW with ONE kernel per rank (peer loads of 1/world of
 * the data, peer stores of the reduced slice, two flag round trips) instead of ncclAllReduce.  Deterministic and
 * bit-identical on all ranks.  uml_dp_allreduce_p2p sums the ranks' input halves of the blocks into every rank's
 * output half.  A peer that stops answering for UML_DP_TIMEOUT_S (default 20) seconds makes the kernel give up instead
 * of hanging: it then performs NO reduction and NO update (weights, moments and bf16 shadow keep their values) and
 * uml_dp_p2p_failed() returns 1 from then on - the engine polls it whenever it reads its statistics log and raises.
 * Re-sizing: uml_dp_p2p_close_peers on every rank, a barrier between the ranks, then uml_dp_p2p_alloc / _open again
 * (an exported block must not be freed while a peer still has it mapped).                                     */
int uml_dp_p2p_alloc(int64_t max_floats, void* handle_out_64_bytes /*host*/);
int uml_dp_p2p_close_peers(void);
int uml_dp_p2p_open(const void* handles /*host: world x 64 bytes, rank order*/, int32_t rank, int32_t world);
int uml_dp_allreduce_p2p(int64_t n, void* stream);
/* the whole data-parallel tail of a step in ONE kernel per rank: split-K sum of the local dW partials -> exchange
 * over peer memory -> Adam/AdamW on every rank (+ bf16 shadow).  partials == NULL: the local sum already sits in
 * the exchange block's input half.                                                                           */
int uml_dp_fused_adam_update(const float* partials, int32_t n_splits, int64_t split_stride, int64_t n, float* p, float* m,
                             float* v, double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step,
                             int32_t decoupled, uint16_t* p_bf16, void* stream);
int uml_dp_p2p_failed(void);

/* ---- a-14  linear analogue: Gaussian_experiment's SharedAutoencoder step (model.py:5-49, main.py:47-59) ------
 * params: ONE flat fp32 buffer in the reference's construction order, weight then bias per layer:
 *   in_head_x, in_head_y, shared_encoder.0, shared_encoder.2, shared_decoder.0, shared_decoder.2, out_head_x,
 *   out_head_y   (uml_gauss_param_count floats).  data_x / data_y: [n, dim_obs] fp32; idx: the sampler's [batch]
 * int64 indices (rows are idx % n_m, UnpairedDataset.__getitem__).  mode_xy != 0: loss = alpha_x MSE(x) +
 * alpha_y MSE(y); else loss = MSE(x) and the y heads are left untouched.  Adam with torch's defaults semantics.
 * loss_out[2] = {loss_x, loss_y} of this step (device).  These two return COUNTS, not a status:             */
int uml_gauss_param_count(int32_t dim_obs, int32_t dim_common, int32_t dim_latent);
int uml_gauss_workspace_floats(int32_t dim_obs, int32_t dim_common, int32_t dim_latent, int64_t batch);
int uml_gauss_step(float* params, float* adam_m, float* adam_v, int32_t dim_obs, int32_t dim_common, int32_t dim_latent,
                   const float* data_x, int64_t n_x, const float* data_y, int64_t n_y, const int64_t* idx, int64_t batch,
                   int32_t mode_xy, float alpha_x, float alpha_y, double lr, double beta1, double beta2, double eps,
                   int64_t step, float* workspace, float* loss_out, void* stream);
/* n_steps consecutive steps in one call: idx_list is a HOST array of device index batches, loss_log[2*i..] gets step i */
int uml_gauss_run(float* params, float* adam_m, float* adam_v, int32_t dim_obs, int32_t dim_common, int32_t dim_latent,
                  const float* data_x, int64_t n_x, const float* data_y, int64_t n_y, const int64_t* const* idx_list /*host*/,
                  int32_t n_steps, int64_t batch, int32_t mode_xy, float alpha_x, float alpha_y, double lr, double beta1,
                  double beta2, double eps, int64_t first_step, float* workspace, float* loss_log, void* stream);
/* validation forward (main.py:68-72): loss_out[2] = MSE of both modalities over n_rows dense rows          */
int uml_gauss_eval(const float* params, int32_t dim_obs, int32_t dim_common, int32_t dim_latent, const float* data_x,
                   const float* data_y, int64_t n_rows, float* workspace /* >= 2*ceil(n_rows/16) floats */,
                   float* loss_out, void* stream);

/* ---- a-14 grid: K runs of the Gaussian experiment (one model shape, one dataset, one batch size) in lock step --------
 * The combinations of the reference's YAML grid (main.py) trained together: run k has its own parameters and Adam
 * moments (row k of the [n_runs][param_stride] slabs), index batch per step, mode, alpha_x, alpha_y, lr and active
 * flag; betas, eps and the Adam step count are shared.  One step of all runs is two launches (the run is a grid
 * dimension of both kernels), and run k computes exactly what uml_gauss_run computes for it alone, bit for bit.
 * A run with active[k] == 0 is not touched: parameters, moments and its rows of both logs stay as they are.
 * Probes (eval_every > 0): after the update of the call's step i with (eval_phase + i + 1) % eval_every == 0, every
 * active run's {val_loss_x, val_loss_y, linear CKA, mutual top-k NN} of its validation rows (what uml_gauss_eval,
 * uml_gauss_embed, uml_cka_linear_f32 and uml_mutual_knn_f32 return for those weights, bit for bit) goes to the next
 * row of eval_log - on the device, without a host synchronisation.
 * Contract, checked before anything touches the device: 1..32 runs; non-null data, slabs, loss_log and workspace
 * (16-byte aligned, workspace_bytes >= uml_gauss_group_workspace_bytes(n_runs, dims, batch, n_val, topk), n_val = 0
 * without probes); param_stride >= uml_gauss_param_count; mode_xy 0 or 1; with probes: validation rows of every
 * active run, eval_log, 2 <= n_val, 1 <= topk <= 64, topk < n_val.                                            */
#define UML_GAUSS_GROUP_MAX_RUNS 32
typedef struct {
  int32_t      n_runs, dim_obs, dim_common, dim_latent;
  const float* data_x;          /* [n_x, dim_obs] rows shared by every run (UnpairedDataset)                   */
  int64_t      n_x;
  const float* data_y;          /* [n_y, dim_obs]                                                              */
  int64_t      n_y;
  int64_t      batch;           /* rows per index batch (the same for every run)                               */
  float*       params;          /* [n_runs][param_stride] flat parameters, uml_gauss_step's layout per run     */
  float*       adam_m;          /* same layout                                                                  */
  float*       adam_v;
  int64_t      param_stride;
  double       beta1, beta2, eps;
  int64_t      first_step;      /* 1-based Adam step of the call's first step (all runs alike)                 */
  int32_t      mode_xy[UML_GAUSS_GROUP_MAX_RUNS];   /* 1: alpha_x MSE(x) + alpha_y MSE(y); 0: MSE(x) alone      */
  float        alpha_x[UML_GAUSS_GROUP_MAX_RUNS];
  float        alpha_y[UML_GAUSS_GROUP_MAX_RUNS];
  double       lr[UML_GAUSS_GROUP_MAX_RUNS];
  uint8_t      active[UML_GAUSS_GROUP_MAX_RUNS];
  float*       loss_log;        /* out [n_steps][n_runs][2]: {loss_x, loss_y} of every step                    */
  int32_t      eval_every;      /* 0: no probes                                                                 */
  int32_t      topk;            /* neighbours of the mutual-kNN probe (the reference: 10)                      */
  int64_t      eval_phase;      /* steps of the evaluation schedule before the call's first step               */
  int64_t      n_val;           /* validation rows of every run                                                 */
  const float* val_x[UML_GAUSS_GROUP_MAX_RUNS];     /* [n_val, dim_obs] validation rows of run k               */
  const float* val_y[UML_GAUSS_GROUP_MAX_RUNS];
  float*       eval_log;        /* out [evaluations of the call][n_runs][4]: {val_x, val_y, cka, mknn}          */
  void*        workspace;       /* scratch: gradient slots, per-tile losses, the runs' validation embeddings
                                   ([n_runs][n_val][dim_latent] x 2), CKA Gram partials, neighbour lists        */
  int64_t      workspace_bytes;
} uml_gauss_group_args;
int64_t uml_gauss_group_workspace_bytes(int32_t n_runs, int32_t dim_obs, int32_t dim_common, int32_t dim_latent,
                                        int64_t batch, int64_t n_val, int32_t topk);   /* a COUNT, not a status */
/* n_steps steps: idx is a HOST array [n_steps][n_runs] of device index batches (entries of inactive runs unused) */
int uml_gauss_group_run(const uml_gauss_group_args* args /*host*/, int32_t n_steps, const int64_t* const* idx /*host*/,
                        void* stream);

/* ---- f-3  alignment probes (diagnostics logged beside the loops: metrics.py:55-119,252-285 of the reference, called at
 * Gaussian_experiment/main.py:67-84 and vision_language/finetune.py:209-233) --------------------------------------
 * uml_cka_linear_f32: out[0] = linear CKA with the biased HSIC estimator of A [n, da] and B [n, db] (row pitches lda /
 *   ldb floats), in its O(n d^2) form (squared Frobenius norms of the centred Gram blocks; no n x n matrix).
 *   ws: uml_cka_workspace_doubles(da, db) doubles.
 * uml_mutual_knn_f32: out[0] = mean over rows of |kNN_A(i) & kNN_B(i)| / topk, neighbours by inner product, self
 *   excluded (its similarity set to -1e8), ties -> lower index.  ws: 2 * n * topk + 1 int32.
 * uml_gauss_embed: emb = shared_encoder(in_head(row)) of the Gaussian autoencoder (model.py:51-60) for the given
 *   modalities (data_x / data_y may be NULL), [n_rows, dim_latent] each.                                      */
int64_t uml_cka_workspace_doubles(int32_t da, int32_t db);
int uml_cka_linear_f32(const float* A, int64_t lda, int32_t da, const float* B, int64_t ldb, int32_t db, int64_t n, double* ws,
                       float* out /*[1]*/, void* stream);
int uml_mutual_knn_f32(const float* A, int64_t lda, int32_t da, const float* B, int64_t ldb, int32_t db, int64_t n, int32_t topk,
                       int32_t* ws, float* out /*[1]*/, void* stream);
int uml_gauss_embed(const float* params, int32_t dim_obs, int32_t dim_common, int32_t dim_latent, const float* data_x,
                    const float* data_y, int64_t n_rows, float* emb_x, float* emb_y, void* stream);

/* ---- sweep-level batching (SURVEY section 8 f-1): the lr x weight-decay (x alpha) combinations that
 * finetune.py:406-448 (`sweep`) and engine/optimizer/default.py:17-31 (`HYPER_DICT`) train one after the other over the
 * SAME banks advance here in lock step - K heads with their own weights, optimizer state, sampler stream, lr, weight
 * decay and alpha; one step of all K heads is two launches (three with more than 1024 classes, four when rows are not
 * 16-byte aligned).  fp32-level
 * arithmetic per head: the two contractions run on the tensor cores as tf32 products of operands split into two terms
 * each (hi * hi + hi * lo + lo * hi, fp32 accumulation) when rows are 16-byte aligned, else as FFMA loops; linear
 * head without adapter and with fixed logit scales (UMLClip, head.py:131-137).  All heads share bank sizes and batch
 * sizes, so head k's batch for modality s is perm[s][k][pos[s] .. pos[s]+n) with a common position.            */
#define UML_SWEEP_MAX_HEADS 32
typedef struct {
  int32_t        n_heads, dim, n_classes;
  int32_t        kind;            /* uml_update.kind: 1 AdamW, 2 Adam (L2), 3 SGD momentum (L2)                */
  const float*   bank[2];         /* fp32 rows of the image / text bank (NULL for an absent modality)           */
  int64_t        bank_ld[2];
  const int64_t* labels[2];       /* bank labels                                                                 */
  const int64_t* perm[2][UML_SWEEP_MAX_HEADS]; /* host array of DEVICE pointers: head k's epoch permutation        */
  int64_t        perm_len[2];     /* entries in every permutation (= bank rows)                                  */
  int64_t        pos[2];          /* where the first step's batches start inside the permutations                */
  float          scale[2];        /* logit scales of the image / text run                                        */
  float*         W;               /* [n_heads][head_stride] weights, each head a [n_classes][dim] matrix         */
  float*         m;               /* exp_avg | momentum buffers, same layout                                     */
  float*         v;               /* exp_avg_sq (unused for SGD)                                                 */
  int64_t        head_stride;
  float*         G;               /* scratch [n_heads][max_rows][ldg]                                            */
  int64_t        ldg, max_rows;
  float*         row_loss;        /* scratch [n_heads][max_rows]                                                 */
  int32_t*       row_correct;     /* scratch [n_heads][max_rows]                                                 */
  uml_seg_stats* stats;           /* out [n_steps][n_heads][2]: {image run, text run} of every step              */
  float          beta1, beta2, eps, momentum;
  int64_t        step;            /* 1-based optimizer step of the first step (all heads count alike)            */
  float          weight_decay[UML_SWEEP_MAX_HEADS];
  float          alpha[UML_SWEEP_MAX_HEADS];       /* text-loss weight per head (finetune.py:188)               */
  uint8_t        active[UML_SWEEP_MAX_HEADS];      /* 0: the head stopped early, nothing of it is touched       */
  void*          ev[8];           /* optional cudaEvent_t pairs recorded around the four launch sites of the LAST
                                     step: logits (+ softmax/CE when fused), softmax/CE, dW + update (+ stats when
                                     fused), stats (NULL = not timed; a pair around a fused-away site spans nothing) */
} uml_sweep_args;
/* n_steps consecutive steps: step i consumes rows[2i] image rows and rows[2i+1] text rows per head (host array;
 * the last batch of an epoch is short) with learning rates lr[i*n_heads + k] (host array).                      */
int uml_sweep_run(const uml_sweep_args* args /*host*/, int32_t n_steps, const int64_t* rows /*host*/,
                  const float* lr /*host*/, void* stream);
/* kernels launched by uml_sweep_run, uml_sweep_adapter_run and uml_sweep_run_diag in this process so far (modulo 2^31):
 * three per step when the tensor-core dW launch carries the statistics warp, four otherwise; see uml_sweep_adapter_run
 * for its count; uml_sweep_run_diag adds two per step */
int uml_sweep_launch_count(void);

/* The same lock-step sweep for UML heads with an image adapter and / or learnable temperatures (head.py:39-98: the
 * reference's `linear` preset over unimodal encoders, engine/optimizer/default.py:17-31).  Per head k and step:
 *   Z_k = X_img Wp_k^T,  logits = [Z_k ; X_txt] W_k^T * scale_k,  dZ_k = G_k[image rows] W_k (W_k before its update),
 *   W_k, scale_k and Wp_k updated with the head's rule (the four parameters share one parameter group).
 * `args` describes the head exactly as for uml_sweep_run; args->dim is the head's input width D (= the adapter's output),
 * bank[0] holds image rows of img_dim floats when there is an adapter, bank[1] text rows of D floats.
 * One step of all heads is five launches: Z, logits + softmax / CE over [Z; X_txt] (+ per-row d loss / d scale), dZ,
 * head dW + update + statistics (+ temperature update), adapter dWp + update; without an adapter, or in a step without
 * image rows, Z, dZ and dWp are skipped (two launches).
 * Contract, checked before anything touches the device: tensor-core forms only - dim % 4 == 0, img_dim % 4 == 0, 16-byte
 * aligned slabs, banks, G, Z and dZ with strides that are multiples of 4; max_rows <= 64; n_classes <= 1024.           */
typedef struct {
  int32_t  img_dim;         /* Dv, width of the image rows; 0 = no adapter (image rows go straight to the head)          */
  float*   W;               /* [n_heads][adapter_stride] adapter weights, each a [dim][img_dim] matrix (img_proj.weight) */
  float*   m;               /* exp_avg | momentum buffers, same layout                                                 */
  float*   v;               /* exp_avg_sq (unused for SGD)                                                             */
  int64_t  adapter_stride;
  float*   Z;               /* scratch [n_heads][max_img_rows][ldz]: adapter output                                    */
  float*   dZ;              /* scratch [n_heads][max_img_rows][ldz]: its gradient                                      */
  int64_t  ldz, max_img_rows;
  float*   scale_param;     /* [n_heads][2] learnable temperatures (image, text); NULL: the fixed args->scale           */
  float*   scale_m;         /* [n_heads][2] optimizer state of the temperatures                                        */
  float*   scale_v;
  float*   row_dscale;      /* scratch [n_heads][max_rows] (with scale_param)                                          */
  void*    ev[10];          /* optional cudaEvent_t pairs around the five launch sites of the LAST step: Z, logits +
                               softmax / CE, dZ, head dW + update + statistics, adapter dWp + update                   */
} uml_sweep_adapter_args;
int uml_sweep_adapter_run(const uml_sweep_args* args /*host*/, const uml_sweep_adapter_args* adapter /*host*/,
                          int32_t n_steps, const int64_t* rows /*host*/, const float* lr /*host*/, void* stream);

/* uml_sweep_run (adapter == NULL) or uml_sweep_adapter_run with the reference's per-step gradient probes
 * (finetune.py:190-206, a-13): for every running head and step, at the step's weights before its update,
 *   A = d image_loss / d W_k,  B = d text_loss / d W_k  (plain mean cross-entropies: B carries no alpha),
 * reduced on the device to out[step][head] = {sum A.B, sum A^2, sum B^2, #(sign A == sign B)} (torch.sign: 0 equals
 * only 0) - two more launches per step (a tensor-core pass over G and the step's rows, a fixed-order finish), no
 * [C, D] gradient in HBM, no host synchronisation.  They only read, so the training results are bit-identical to the
 * same call without diagnostics.  Contract, checked before anything touches the device: dim % 4 == 0, 16-byte aligned
 * slabs, G, banks and Z; alpha > 0 for every running head when there is a text bank; scratch_floats >=
 * uml_sweep_diag_scratch_floats(n_heads, dim, n_classes).                                                        */
typedef struct {
  float*   out;             /* [n_steps][n_heads][4] (rows of stopped heads are not written)                      */
  float*   scratch;         /* per-unit partial sums                                                               */
  int64_t  scratch_floats;
  void*    ev[2];           /* optional cudaEvent_t pair around the diagnostics launches of the LAST step         */
} uml_sweep_diag;
int64_t uml_sweep_diag_scratch_floats(int32_t n_heads, int32_t dim, int32_t n_classes); /* a COUNT, not a status */
int uml_sweep_run_diag(const uml_sweep_args* args /*host*/, const uml_sweep_adapter_args* adapter /*host, NULL: linear heads*/,
                       const uml_sweep_diag* diag /*host*/, int32_t n_steps, const int64_t* rows /*host*/,
                       const float* lr /*host*/, void* stream);

/* ---- sampler: the epoch permutation on the host, bit-exact with torch.randperm(n, generator=
 * torch.Generator().manual_seed(seed)) on the CPU - what RandomSampler draws once per epoch for the
 * DataLoaders of finetune.py:370-371 (MT19937 seeded with the low 32 bits of `seed`, Fisher-Yates
 * `z = rand() % (n - i)`).  Pure host code; `out` (n int64, normally pinned memory) is copied to the device
 * asynchronously by the caller.  n < 2^32 / 20.
 * The prefix out[0..i] is final after iteration i, so the permutation can be produced incrementally:
 * uml_randperm_begin seeds the generator and writes the identity, uml_randperm_advance(state, upto) runs the
 * iterations needed to make out[0..upto) final (a host thread keeps that prefix ahead of the training loop).
 * `state` is caller-owned scratch of UML_RANDPERM_STATE_BYTES bytes (8-byte aligned).                      */
#define UML_RANDPERM_STATE_BYTES 3072   /* `out` doubles as scratch: its upper half holds the 32-bit working array */
int uml_randperm_begin(void* state /*host*/, uint64_t seed, int64_t n, int64_t* out /*host*/);
int uml_randperm_advance(void* state /*host*/, int64_t upto);
/* begin + advance in chunks, publishing the final-prefix length after each chunk: the body of a producer thread.
 * uml_randperm_wait (any other thread) returns once out[0..upto) is final.                                  */
int uml_randperm_run(void* state /*host*/, uint64_t seed, int64_t n, int64_t* out /*host*/, int64_t chunk,
                     int32_t prefilled /* out already holds 0..n-1 */,
                     int64_t* next_out /* optional: filled with 0..n-1 afterwards, for the next epoch */);
int uml_randperm_next_filled(const void* state /*host*/);   /* 1 once next_out holds the identity (NOT a status) */
int uml_randperm_wait(const void* state /*host*/, int64_t upto);
int uml_randperm_i64(uint64_t seed, int64_t n, int64_t* out /*host*/);

#ifdef __cplusplus
}
#endif
#endif /* UML_B200_H_ */
