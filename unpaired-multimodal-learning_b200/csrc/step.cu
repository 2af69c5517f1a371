// One UML iteration behind ONE C-ABI call: the host enqueues every kernel of the step
// (reference loop body, vision_language/finetune.py:163-195) without returning to Python in between.
// At the reference's batch sizes the step is launch-latency bound, at throughput batch sizes the host
// must stay ahead of a ~150 us GPU step - either way per-kernel Python dispatch is what limits it.
#include <algorithm>

#include "common.cuh"
#include "grad_diag.cuh"

namespace {
inline void rec(void* ev, void* stream) {
  if (ev) cudaEventRecord(static_cast<cudaEvent_t>(ev), uml::as_stream(stream));
}

// Side stream + events for the gather prefetch of uml_linear_run (one set per device, created on first use).
struct Pipe {
  cudaStream_t aux = nullptr;
  cudaEvent_t ready[3] = {nullptr, nullptr, nullptr}, freed[3] = {nullptr, nullptr, nullptr}, start = nullptr, mid = nullptr;
  // the pipeline of uml_linear_run survives the call boundary when the caller vouches for its index batches (idx_ready):
  bool warm = false;                    // freed[] / fwd_mid[] describe the last steps of the previous call
  int phase = 0;                        // operand buffer of the next step
  unsigned gstep = 0;                   // steps enqueued so far (fwd_mid[gstep & 1] is recorded after step gstep's forward)
  const void* bufs[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t fwd_mid[2] = {nullptr, nullptr};
  bool ok = false;
};

// any other user of the operand buffers (single-step calls, Python-side kernels) makes the next run start cold
void pipe_invalidate();

static Pipe g_pipes[64];
void pipe_invalidate() {
  int dev = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && dev >= 0 && dev < 64) g_pipes[dev].warm = false;
}

Pipe* get_pipe() {
  Pipe* pipes = g_pipes;
  static bool tried[64] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  Pipe& p = pipes[dev];
  if (!tried[dev]) {
    tried[dev] = true;
    int lo = 0, hi = 0;
    if (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess) return nullptr;
    // lowest priority: the prefetch must never delay a kernel of the step it hides under
    if (cudaStreamCreateWithPriority(&p.aux, cudaStreamNonBlocking, lo) != cudaSuccess) return nullptr;
    bool good = true;
    for (int i = 0; i < 3; ++i) {
      good = good && cudaEventCreateWithFlags(&p.ready[i], cudaEventDisableTiming) == cudaSuccess;
      good = good && cudaEventCreateWithFlags(&p.freed[i], cudaEventDisableTiming) == cudaSuccess;
    }
    good = good && cudaEventCreateWithFlags(&p.start, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 2; ++i) good = good && cudaEventCreateWithFlags(&p.fwd_mid[i], cudaEventDisableTiming) == cudaSuccess;
    good = good && cudaEventCreateWithFlags(&p.mid, cudaEventDisableTiming) == cudaSuccess;
    p.ok = good;
  }
  return p.ok ? &p : nullptr;
}

// true when every non-empty run of the step can be gathered from bf16 shadow banks by one copy launch
bool shadow_gatherable(const uml_linear_step_args* a) {
  for (int i = 0; i < a->nseg; ++i) {
    const uml_segment& s = a->seg[i];
    if (s.n > 0 && !(s.rows16 && s.idx && !s.label_idx)) return false;
  }
  return true;
}

// both runs' rows + labels -> (X16, labels32) by one launch of the register-copy kernel
int shadow_gather(const uml_linear_step_args* a, uint16_t* X16, int32_t* labels32, void* stream) {
  const uml_segment* g[2] = {nullptr, nullptr};
  int ng = 0;
  for (int i = 0; i < a->nseg; ++i)
    if (a->seg[i].n > 0) g[ng++] = &a->seg[i];
  if (ng == 0) return 0;
  // The register-copy kernel is also the faster one stand-alone (ncu, cfg3: 17.8 us = 6.5 TB/s, the measured copy
  // peak, against 30 us for the TMA ring kernel), so it serves both the prefetch and the in-line gather.
  return uml_gather2_rows_bf16_light(g[0]->rows16, g[0]->labels, g[0]->idx, g[0]->n, ng > 1 ? g[1]->rows16 : nullptr,
                                     ng > 1 ? g[1]->labels : nullptr, ng > 1 ? g[1]->idx : nullptr, ng > 1 ? g[1]->n : 0,
                                     a->dim, X16, a->dim, labels32, stream);
}
}  // namespace

// `mid` (optional) runs on the host right after the forward launches were enqueued: where uml_linear_run enqueues a
// later step's gather, ordered after the forward KERNEL (`after_fwd_kernel`).  The gather then shares the machine with
// the dW GEMM and the update but not with the forward kernel, which it slowed from 67.5 to 84 us on B200 (cfg3).
struct StepHooks {
  bool pregathered = false;
  cudaEvent_t operand_free = nullptr;
  int (*mid)(void*) = nullptr;
  void* mid_arg = nullptr;
  cudaEvent_t after_fwd_kernel = nullptr;
  const uml_linear_diag* diag = nullptr;  // uml_linear_run_diag: the step's gradient diagnostics go to diag_out
  float* diag_out = nullptr;
};
static int linear_step_impl(const uml_linear_step_args* a, void* stream, const StepHooks& hooks);
static int linear_grad_diag(const uml_linear_step_args* a, const uml_linear_diag* d, float* out, cudaStream_t st);
static int check_linear_diag(const uml_linear_step_args* a, const uml_linear_diag* d, const float* out);
int uml_head_fwd_ce_bf16_ev(const uint16_t* X, int64_t n_rows, int32_t dim, const uint16_t* W, int32_t n_classes,
                            const int32_t* labels, const uml_tc_segments* segs, uint16_t* G, int64_t ldg, float* row_loss,
                            int32_t* row_pred, int32_t* row_correct, float* row_dscale, float* tile_ws, uml_seg_stats* stats,
                            void* ev_after_fwd, void* stream, void* ev_after_fwd2 = nullptr);  // tc_fwd.cu

// tc_fwd2.cu / tc_gemm.cu: exchange forward kernel (G final after one pass) and the dW GEMM that reduces its statistics
bool uml_fwd_x_eligible(int64_t n_rows, int32_t n_classes);
void uml_fwd_x_partials(float* tile_ws, int64_t n_rows, int32_t n_classes, const float** part, int64_t* n_entries);
int uml_head_bwd_dw_stats_bf16(const uint16_t* G, int64_t ldg, const uint16_t* X, int64_t n_rows, int32_t dim, int32_t n_classes,
                               float* partials, int32_t n_splits, const float* part, int64_t part_entries, int32_t nseg,
                               uml_seg_stats* stats, void* stream);

float* uml_dp_p2p_input(int64_t n);   // dp.cu: this rank's exchange buffers of the peer-memory all-reduce (or NULL)
float* uml_dp_p2p_output(int64_t n);

// where the local gradient sum of a data-parallel step goes: straight into the peer-visible exchange buffer when
// the NVLink all-reduce is set up, else into dW_out (NCCL reduces that in place)
static float* dp_local_sum_target(const uml_linear_step_args* a, int64_t np) {
  float* x = uml_dp_p2p_input(np);
  return x ? x : a->dW_out;
}

// data parallel tail of a step: sum dW over the ranks, then the optimizer update on every rank
static int dp_reduce_and_update(const uml_linear_step_args* a, int64_t np, void* stream) {
  int rc;
  const float* grad = a->dW_out;
  if (uml_dp_p2p_input(np)) {
    if (a->upd.kind != 3) {  // exchange + Adam fused (the local sum already is in the exchange buffer)
      rec(a->ev[6], stream);
      rc = uml_dp_fused_adam_update(nullptr, 0, 0, np, a->W, a->upd.m, a->upd.v, a->upd.lr, a->upd.beta1, a->upd.beta2,
                                    a->upd.eps, a->upd.weight_decay, a->upd.step, a->upd.kind == 1,
                                    a->precision == 1 ? a->W16 : nullptr, stream);
      rec(a->ev[7], stream);
      return rc;
    }
    rc = uml_dp_allreduce_p2p(np, stream);
    grad = uml_dp_p2p_output(np);
  } else {
    rc = uml_dp_allreduce_f32(a->dW_out, np, stream);
  }
  if (rc) return rc;
  uint16_t* shadow = a->precision == 1 ? a->W16 : nullptr;
  rec(a->ev[6], stream);
  if (a->upd.kind == 3)
    rc = uml_sgd_step(a->W, grad, nullptr, 0.f, a->upd.m, np, a->upd.lr, a->upd.momentum, a->upd.weight_decay,
                      a->upd.step, shadow, stream);
  else
    rc = uml_adamw_step(a->W, grad, nullptr, 0.f, a->upd.m, a->upd.v, np, a->upd.lr, a->upd.beta1, a->upd.beta2,
                        a->upd.eps, a->upd.weight_decay, a->upd.step, a->upd.kind == 1, shadow, stream);
  rec(a->ev[7], stream);
  return rc;
}

static int linear_run_continuous(const uml_linear_step_args* base, const uml_run_step* steps, int32_t n_steps, void* stream,
                                 Pipe* pipe, const uml_linear_diag* diag, float* const* diag_out) {
  using namespace uml;
  constexpr int kNb = 3, kDepth = 2;
  uml_linear_step_args a = *base;
  auto patch = [&](uml_linear_step_args& t, const uml_run_step& s) {
    for (int k = 0; k < t.nseg; ++k) {
      t.seg[k].idx = s.idx[k];
      t.seg[k].n = s.n[k];
      t.seg[k].loss_weight = s.loss_weight[k];
      t.scale_step[k] = s.scale_step[k];
    }
    t.upd.lr = s.lr;
    t.upd.step = s.opt_step;
    t.stats = s.stats;
    for (int k = 0; k < 8; ++k) t.ev[k] = s.ev[k];
  };
  uint16_t* xbuf[kNb] = {base->X16, base->X16_alt, base->X16_alt2};
  int32_t* lbuf[kNb] = {base->labels32, base->labels32_alt, base->labels32_alt2};
  cudaStream_t main_st = as_stream(stream);
  const cudaEvent_t idx_ready = static_cast<cudaEvent_t>(base->idx_ready);
  if (!(pipe->warm && pipe->bufs[0] == xbuf[0] && pipe->bufs[1] == xbuf[1] && pipe->bufs[2] == xbuf[2])) {
    // cold: everything enqueued so far may still read the buffers
    pipe->warm = false;
    pipe->phase = 0;
    for (int k = 0; k < kNb; ++k) pipe->bufs[k] = xbuf[k];
    UML_CUDA(cudaEventRecord(pipe->start, main_st));
  }
  const bool warm = pipe->warm;
  const int phase = pipe->phase;
  const unsigned g0 = pipe->gstep;

  // the gather of step t of this call -> side stream.  `after_fwd`: the forward kernel it follows (so that it shares the
  // machine with a dW GEMM and an update, never - but for its tail - with a forward kernel)
  auto launch_gather = [&](int t, cudaEvent_t after_fwd) -> int {
    const int tb = (phase + t) % kNb;
    uml_linear_step_args g = a;
    patch(g, steps[t]);
    UML_CUDA(cudaStreamWaitEvent(pipe->aux, idx_ready, 0));
    // the dW kernel that last read this buffer: step t - 3 of this call, or of the previous one (warm), else `start`
    UML_CUDA(cudaStreamWaitEvent(pipe->aux, (t >= kNb || warm) ? pipe->freed[tb] : pipe->start, 0));
    if (after_fwd) UML_CUDA(cudaStreamWaitEvent(pipe->aux, after_fwd, 0));
    rec(g.ev[0], pipe->aux);
    const int rc = shadow_gather(&g, xbuf[tb], lbuf[tb], pipe->aux);
    if (rc) return rc;
    rec(g.ev[1], pipe->aux);
    UML_CUDA(cudaEventRecord(pipe->ready[tb], pipe->aux));
    return 0;
  };
  for (int t = 0; t < kDepth && t < n_steps; ++t) {
    // inside one long call step t's gather would have followed the forward kernel of step t - 2: steps -2 and -1 are the
    // previous call's last two
    const int rc = launch_gather(t, warm ? pipe->fwd_mid[(g0 + t) & 1u] : nullptr);  // (g0 + t - 2) & 1
    if (rc) return rc;
  }

  for (int i = 0; i < n_steps; ++i) {
    patch(a, steps[i]);
    if (i > 0) a.w16_valid = 1;  // the optimizer kernel of the previous step refreshed the shadow
    const int b = (phase + i) % kNb;
    a.X16 = xbuf[b];
    a.labels32 = lbuf[b];
    UML_CUDA(cudaStreamWaitEvent(main_st, pipe->ready[b], 0));
    struct Next {
      decltype(launch_gather)* launch;
      int t;
      cudaEvent_t mid;
    } next{&launch_gather, i + kDepth < n_steps ? i + kDepth : -1, pipe->fwd_mid[(g0 + i) & 1u]};
    StepHooks hooks;
    hooks.pregathered = true;
    hooks.operand_free = pipe->freed[b];
    hooks.mid_arg = &next;
    hooks.after_fwd_kernel = next.mid;  // recorded right after the forward kernel, also for the next call's first gathers
    hooks.diag = diag;
    hooks.diag_out = diag ? diag_out[i] : nullptr;
    hooks.mid = [](void* p) -> int {
      Next* n = static_cast<Next*>(p);
      return n->t >= 0 ? (*n->launch)(n->t, n->mid) : 0;
    };
    const int rc = linear_step_impl(&a, stream, hooks);
    if (rc) {
      pipe->warm = false;
      return rc;
    }
  }
  pipe->phase = (phase + n_steps) % kNb;
  pipe->gstep = g0 + static_cast<unsigned>(n_steps);
  pipe->warm = true;
  return 0;
}

static int linear_run_impl(const uml_linear_step_args* base, const uml_run_step* steps, int32_t n_steps,
                           const uml_linear_diag* diag, float* const* diag_out, void* stream) {
  using namespace uml;
  uml_linear_step_args a = *base;
  auto patch = [&](uml_linear_step_args& t, const uml_run_step& s) {
    for (int k = 0; k < t.nseg; ++k) {
      t.seg[k].idx = s.idx[k];
      t.seg[k].n = s.n[k];
      t.seg[k].loss_weight = s.loss_weight[k];
      t.scale_step[k] = s.scale_step[k];
    }
    t.upd.lr = s.lr;
    t.upd.step = s.opt_step;
    t.stats = s.stats;
    for (int k = 0; k < 8; ++k) t.ev[k] = s.ev[k];
  };

  // Gather prefetch: step i+1's rows are copied into the operand buffer step i does not use, on a low-priority
  // side stream, while step i's forward / fix-up / dW / update run.  (The copy depends only on the indices and
  // the bank, never on the weights.)  Buffer b becomes free again once the dW kernel that read it has finished.
  Pipe* pipe = nullptr;
  if (a.precision == 1 && a.X16_alt && a.labels32_alt && n_steps > 1) {
    bool all = true;
    for (int i = 0; i < n_steps && all; ++i) {
      uml_linear_step_args t = a;
      patch(t, steps[i]);
      all = shadow_gatherable(&t);
    }
    if (all) pipe = get_pipe();
  }
  // ---- continuous mode: three operand buffers and an event that vouches for the index batches (idx_ready) ----------
  // The gather pipeline then runs through the call boundaries: the first two steps' gathers go to the side stream at once,
  // ordered after the index upload, after the dW kernel that last read their buffer and after the forward kernel of the
  // step they would have followed inside one long call - when the host is a chunk ahead of the GPU (it normally is) they
  // run beside the previous call's last steps, and a call costs no gather on the main stream at all.
  if (a.precision == 1 && base->X16_alt && base->labels32_alt && base->X16_alt2 && base->labels32_alt2 && base->idx_ready &&
      n_steps >= 1) {
    bool all = true;
    for (int i = 0; i < n_steps && all; ++i) {
      uml_linear_step_args t = a;
      patch(t, steps[i]);
      all = shadow_gatherable(&t);
    }
    Pipe* cp = all ? get_pipe() : nullptr;
    if (cp) return linear_run_continuous(base, steps, n_steps, stream, cp, diag, diag_out);
  }
  pipe_invalidate();
  // With a third operand buffer the gather runs TWO steps ahead: step i + 2's rows are copied while step i's dW and
  // update run and may spill into step i + 1 - no forward kernel ever waits for an event that is signalled at the last
  // moment (one step ahead, the gather of step i + 1 ended about when the update did, and the cross-stream hand-over
  // put ~9 us between the update and the next forward kernel).
  const int nb = (pipe && base->X16_alt2 && base->labels32_alt2 && n_steps > 2) ? 3 : 2;
  const int depth = nb - 1;
  uint16_t* xbuf[3] = {base->X16, base->X16_alt, base->X16_alt2};
  int32_t* lbuf[3] = {base->labels32, base->labels32_alt, base->labels32_alt2};
  cudaStream_t main_st = as_stream(stream);
  if (pipe) UML_CUDA(cudaEventRecord(pipe->start, main_st));  // everything enqueued so far may still read the other buffers

  for (int i = 0; i < n_steps; ++i) {
    patch(a, steps[i]);
    if (i > 0 && a.precision == 1) a.w16_valid = 1;  // the optimizer kernel of the previous step refreshed the shadow
    if (!pipe) {
      StepHooks plain;  // (uml_linear_step)
      plain.diag = diag;
      plain.diag_out = diag ? diag_out[i] : nullptr;
      pipe_invalidate();
      const int rc = linear_step_impl(&a, stream, plain);
      if (rc) return rc;
      continue;
    }
    const int b = i % nb;
    a.X16 = xbuf[b];
    a.labels32 = lbuf[b];
    if (i == 0) {
      // the first step's rows in line; with two steps of look-ahead the first step's hook (after its forward kernel)
      // starts BOTH the second and the third step's gathers: beside the first forward kernel a gather would only have
      // the SMs that kernel leaves free (4 of 148) and hold up the second step
      rec(a.ev[0], stream);
      const int rc0 = shadow_gather(&a, xbuf[0], lbuf[0], stream);
      if (rc0) return rc0;
      rec(a.ev[1], stream);
    } else {
      UML_CUDA(cudaStreamWaitEvent(main_st, pipe->ready[b], 0));
    }
    struct Job {
      uml_linear_step_args nx;
      uint16_t* x;
      int32_t* l;
      cudaEvent_t wait_a, ready;
    };
    struct Next {
      Pipe* pipe;
      Job job[2];
      int n_jobs;
      bool have;
    } next;
    next.pipe = pipe;
    next.n_jobs = 0;
    // step i's hook starts the gather of step i + depth (the first step's: of every step up to `depth`)
    for (int t = (i == 0 ? 1 : i + depth); t <= i + depth && t < n_steps; ++t) {
      const int tb = t % nb;  // last read by the dW kernel of step t - nb (never, when that is before this call)
      Job& j = next.job[next.n_jobs++];
      j.nx = a;
      patch(j.nx, steps[t]);
      j.x = xbuf[tb];
      j.l = lbuf[tb];
      j.wait_a = t < nb ? pipe->start : pipe->freed[tb];
      j.ready = pipe->ready[tb];
    }
    next.have = next.n_jobs > 0;
    StepHooks hooks;
    hooks.pregathered = true;
    hooks.operand_free = pipe->freed[b];
    hooks.mid_arg = &next;
    hooks.after_fwd_kernel = next.have ? pipe->mid : nullptr;
    hooks.diag = diag;
    hooks.diag_out = diag ? diag_out[i] : nullptr;
    hooks.mid = [](void* p) -> int {
      Next* n = static_cast<Next*>(p);
      if (!n->have) return 0;
      for (int k = 0; k < n->n_jobs; ++k) {
        Job& j = n->job[k];
        UML_CUDA(cudaStreamWaitEvent(n->pipe->aux, j.wait_a, 0));
        UML_CUDA(cudaStreamWaitEvent(n->pipe->aux, n->pipe->mid, 0));
        rec(j.nx.ev[0], n->pipe->aux);  // ev[0]..ev[1] bracket the gather where it really runs: on the side stream
        const int rc = shadow_gather(&j.nx, j.x, j.l, n->pipe->aux);
        if (rc) return rc;
        rec(j.nx.ev[1], n->pipe->aux);
        UML_CUDA(cudaEventRecord(j.ready, n->pipe->aux));
      }
      return 0;
    };
    const int rc = linear_step_impl(&a, stream, hooks);
    if (rc) return rc;
  }
  return 0;
}

extern "C" {

int uml_linear_run(const uml_linear_step_args* base, const uml_run_step* steps, int32_t n_steps, void* stream) {
  UML_REQUIRE(base && steps && n_steps >= 0, "linear_run: bad arguments");
  return linear_run_impl(base, steps, n_steps, nullptr, nullptr, stream);
}

int64_t uml_linear_diag_scratch_floats(int32_t precision, int64_t max_rows, int32_t dim, int32_t n_classes) {
  if (max_rows < 1 || dim < 1 || n_classes < 1) return 0;
  if (precision == 0) return static_cast<int64_t>((dim + 127) / 128) * ((n_classes + 63) / 64) * 4;
  // bf16: per-block slots, then the split-K partials of A and of B (as many splits as a step of max_rows takes)
  const int64_t splits = std::max(1, uml_tc_dw_splits(max_rows, dim, n_classes));
  return 4 * static_cast<int64_t>(uml::grad_diag_partial_slots()) + 2 * splits * n_classes * static_cast<int64_t>(dim);
}

int uml_linear_run_diag(const uml_linear_step_args* base, const uml_run_step* steps, int32_t n_steps,
                        const uml_linear_diag* diag, float* const* out, void* stream) {
  UML_REQUIRE(base && steps && n_steps >= 0 && diag && (out || n_steps == 0), "linear_run_diag: bad arguments");
  for (int i = 0; i < n_steps; ++i) {  // every step's contract before anything is enqueued
    uml_linear_step_args t = *base;
    for (int k = 0; k < t.nseg; ++k) {
      t.seg[k].idx = steps[i].idx[k];
      t.seg[k].n = steps[i].n[k];
      t.seg[k].loss_weight = steps[i].loss_weight[k];
    }
    if (check_linear_diag(&t, diag, out[i])) return 1;
  }
  return linear_run_impl(base, steps, n_steps, diag, out, stream);
}

int uml_linear_grad_diag(const uml_linear_step_args* a, const uml_linear_diag* diag, float* out, void* stream) {
  UML_REQUIRE(a, "linear_grad_diag: null args");
  if (check_linear_diag(a, diag, out)) return 1;
  return linear_grad_diag(a, diag, out, uml::as_stream(stream));
}

int uml_linear_step(const uml_linear_step_args* a, void* stream) {
  pipe_invalidate();  // (it gathers into the first operand buffer on the main stream)
  return linear_step_impl(a, stream, StepHooks());
}

// the operand buffers were used by something the library did not see (Python-side kernels on them): start cold next time
int uml_linear_run_reset(void) {
  pipe_invalidate();
  return 0;
}

}  // extern "C"

static int linear_step_body(const uml_linear_step_args* a, void* stream, const StepHooks& hooks);

// The step, then its diagnostics when asked: the bf16 path runs them inside the step (after the dW launch, before the
// operand buffer is handed back to the gather pipeline), the exact path - and a step without rows - after its last launch.
static int linear_step_impl(const uml_linear_step_args* a, void* stream, const StepHooks& hooks) {
  const int rc = linear_step_body(a, stream, hooks);
  if (rc || !hooks.diag) return rc;
  const int64_t total = a->seg[0].n + (a->nseg > 1 ? a->seg[1].n : 0);
  if (a->precision == 1 && total > 0) return 0;
  return linear_grad_diag(a, hooks.diag, hooks.diag_out, uml::as_stream(stream));
}

static int linear_step_body(const uml_linear_step_args* a, void* stream, const StepHooks& hooks) {
  using namespace uml;
  const bool pregathered = hooks.pregathered;
  const cudaEvent_t operand_free = hooks.operand_free;
  bool stats_in_dw = false;  // the forward's per-run statistics are reduced inside the dW kernel
  UML_REQUIRE(a != nullptr, "linear_step: null args");
  // bf16 path: the kernels write one record per run WITH rows, in order, starting here (stats[i] belongs to seg[i])
  uml_seg_stats* live_stats = a->stats;
  UML_REQUIRE(a->nseg >= 1 && a->nseg <= UML_MAX_SEGMENTS, "linear_step: 1..2 segments");
  UML_REQUIRE(a->W && a->G && a->row_loss && a->row_correct && a->stats, "linear_step: null buffers");
  const int64_t n0 = a->seg[0].n, n1 = a->nseg > 1 ? a->seg[1].n : 0, total = n0 + n1;
  const bool dp = a->dp_allreduce != 0;
  UML_REQUIRE(!dp || a->dW_out, "linear_step: data-parallel mode needs dW_out");
  const bool fused = a->dW_out == nullptr;
  int rc;
  bool w_done = false;  // the fp32 fused kernel took the whole step of W: only the temperatures are left

  if (a->precision == 0) {
    // ------------------------------------------------------------------ fp32 exact path (one fused launch, else 3 + 1)
    UML_REQUIRE(a->row_dscale, "linear_step: fp32 path needs row_dscale");
    rec(a->ev[2], stream);
    if (fused && !dp && total > 0) {  // the reference's batch sizes: forward, gradient and update in one cooperative launch
      int32_t launched = 0;
      rc = uml_head_step_fused_f32(a->seg, a->nseg, a->dim, a->W, a->n_classes, static_cast<float*>(a->G), a->ldg, a->row_loss,
                                   a->row_correct, a->row_dscale, a->stats, &a->upd, &launched, stream);
      if (rc) return rc;
      if (launched) {
        rec(a->ev[3], stream);
        rec(a->ev[4], stream);
        rec(a->ev[5], stream);
        w_done = true;
      }
    }
    if (!w_done) {
      rc = uml_head_fwd_ce_f32(a->seg, a->nseg, a->dim, a->W, a->n_classes, static_cast<float*>(a->G), a->ldg,
                               a->row_loss, a->row_correct, a->row_dscale, a->stats, a->g_capacity_rows, stream);
      if (rc) return rc;
      rec(a->ev[3], stream);
    }
  } else {
    // ------------------------------------------------------------------ bf16 tensor-core path
    UML_REQUIRE(a->X16 && a->W16 && a->labels32 && a->partials && a->tile_ws && a->max_splits >= 1,
                "linear_step: bf16 buffers");
    if (!a->w16_valid) {
      rc = uml_cast_f32_to_bf16(a->W, a->W16, static_cast<int64_t>(a->n_classes) * a->dim, stream);
      if (rc) return rc;
    }
    uml_tc_segments ts;
    memset(&ts, 0, sizeof(ts));
    ts.nseg = 0;
    int64_t off = 0;
    if (!pregathered) rec(a->ev[0], stream);  // (a pre-gathered step's ev[0]..ev[1] were recorded around its gather)
    const bool shadow = pregathered || shadow_gatherable(a);
    if (shadow && !pregathered) {
      rc = shadow_gather(a, a->X16, a->labels32, stream);
      if (rc) return rc;
    }
    for (int i = 0; i < a->nseg; ++i) {
      const uml_segment& s = a->seg[i];
      if (s.n == 0) {  // the kernels see only the runs with rows: an empty run's record is zeroed here
        UML_CUDA(cudaMemsetAsync(&a->stats[i], 0, sizeof(uml_seg_stats), as_stream(stream)));
        continue;
      }
      if (ts.nseg == 0) live_stats = &a->stats[i];
      if (!shadow) {
        const float* rows = static_cast<const float*>(s.rows);
        UML_REQUIRE(s.ld == a->dim, "linear_step: bf16 path needs dense bank rows (ld == dim)");
        if (s.idx && !s.label_idx) {
          rc = uml_gather_rows_labels_bf16(rows, s.labels, a->dim, s.idx, s.n, a->X16 + off * a->dim, a->dim,
                                           a->labels32 + off, stream);
          if (rc) return rc;
        } else {
          if (s.idx)
            rc = uml_gather_rows_bf16(rows, INT64_MAX / 2, a->dim, s.idx, s.n, a->X16 + off * a->dim, a->dim, stream);
          else
            rc = uml_cast_f32_to_bf16(rows, a->X16 + off * a->dim, s.n * a->dim, stream);
          if (rc) return rc;
          rc = uml_gather_labels_i32(s.labels, s.label_idx ? s.label_idx : s.idx, s.n, a->labels32 + off, stream);
          if (rc) return rc;
        }
      }
      ts.seg_rows[ts.nseg] = s.n;
      ts.scale[ts.nseg] = s.scale;
      ts.loss_weight[ts.nseg] = s.loss_weight;
      ts.scale_dev[ts.nseg] = s.scale_dev;
      ts.nseg++;
      off += s.n;
    }
    if (!pregathered) rec(a->ev[1], stream);
    if (total > 0) {
      rec(a->ev[2], stream);
      // ev[2]..ev[3] bracket the tensor-core kernel alone.  Exchange kernel (the default above 128 rows): G is final when it ends
      // and the per-run statistics are reduced by an idle warp of the dW GEMM - unless a learnable temperature needs them
      // before that (then a small reduction launch follows the forward).  Chunk-sequential kernel: the fix-up launch,
      // which also reduces the statistics, follows it.
      stats_in_dw = uml_fwd_x_eligible(total, a->n_classes) && !a->scale_param[0] && !a->scale_param[1];
      rc = uml_head_fwd_ce_bf16_ev(a->X16, total, a->dim, a->W16, a->n_classes, a->labels32, &ts,
                                   static_cast<uint16_t*>(a->G), a->ldg, nullptr, nullptr, nullptr, nullptr, a->tile_ws,
                                   stats_in_dw ? nullptr : live_stats, a->ev[3], stream, hooks.after_fwd_kernel);
      if (rc) return rc;
    }
    if (hooks.mid) {
      rc = hooks.mid(hooks.mid_arg);
      if (rc) return rc;
    }
  }

  // learnable temperatures: scalar Adam(W) steps fed straight from the stats record on the device.  A run without rows
  // gives its temperature no gradient, and it is skipped as torch.optim skips a parameter whose .grad is None; in
  // data-parallel mode this rank's empty run still takes part in the all-reduce (its record is zero).
  for (int i = 0; i < a->nseg; ++i) {
    if (!a->scale_param[i] || (!dp && a->seg[i].n == 0)) continue;
    float* g = &a->stats[i].dscale;
    if (dp) {  // the temperature gradient is a sum over the global batch as well
      rc = uml_dp_allreduce_f32(g, 1, stream);
      if (rc) return rc;
    }
    if (a->upd.kind == 3)
      rc = uml_sgd_step(a->scale_param[i], g, nullptr, 0.f, a->scale_m[i], 1, a->upd.lr, a->upd.momentum,
                        a->upd.weight_decay, a->scale_step[i], nullptr, stream);
    else
      rc = uml_adamw_step(a->scale_param[i], g, nullptr, 0.f, a->scale_m[i], a->scale_v[i], 1, a->upd.lr, a->upd.beta1,
                          a->upd.beta2, a->upd.eps, a->upd.weight_decay, a->scale_step[i], a->upd.kind == 1, nullptr,
                          stream);
    if (rc) return rc;
  }

  const int64_t np_all = static_cast<int64_t>(a->n_classes) * a->dim;
  if (w_done || (total == 0 && !dp)) return 0;
  if (total == 0) {  // a rank without rows still takes part in the all-reduce, contributing zeros
    UML_CUDA(cudaMemsetAsync(dp_local_sum_target(a, np_all), 0, np_all * sizeof(float), as_stream(stream)));
    return dp_reduce_and_update(a, np_all, stream);
  }
  if (a->precision == 0) {
    uml_update none;
    memset(&none, 0, sizeof(none));
    rec(a->ev[4], stream);
    rc = uml_head_bwd_dw_f32(a->seg, a->nseg, a->dim, static_cast<const float*>(a->G), a->ldg, a->n_classes, a->W,
                             dp ? dp_local_sum_target(a, np_all) : a->dW_out, fused ? &a->upd : &none, stream);
    rec(a->ev[5], stream);
    if (rc || !dp) return rc;
    return dp_reduce_and_update(a, np_all, stream);
  }
  int splits = uml_tc_dw_splits(total, a->dim, a->n_classes);
  if (splits > a->max_splits) splits = a->max_splits;
  rec(a->ev[4], stream);
  if (stats_in_dw) {
    const float* part = nullptr;
    int64_t entries = 0;
    uml_fwd_x_partials(a->tile_ws, total, a->n_classes, &part, &entries);
    int nseg_live = 0;
    for (int i = 0; i < a->nseg; ++i) nseg_live += a->seg[i].n > 0 ? 1 : 0;
    rc = uml_head_bwd_dw_stats_bf16(static_cast<const uint16_t*>(a->G), a->ldg, a->X16, total, a->dim, a->n_classes,
                                    a->partials, splits, part, entries, nseg_live, live_stats, stream);
  } else {
    rc = uml_head_bwd_dw_bf16(static_cast<const uint16_t*>(a->G), a->ldg, a->X16, total, a->dim, a->n_classes, a->partials,
                              splits, stream);
  }
  if (rc) return rc;
  rec(a->ev[5], stream);
  if (hooks.diag) {  // X16 and G still hold this step's operands; X16 goes back to the gather pipeline only below
    rc = linear_grad_diag(a, hooks.diag, hooks.diag_out, as_stream(stream));
    if (rc) return rc;
  }
  if (operand_free) UML_CUDA(cudaEventRecord(operand_free, as_stream(stream)));  // X16 / labels32 may be overwritten
  const int64_t np = static_cast<int64_t>(a->n_classes) * a->dim;
  if (!fused) {
    if (dp && a->upd.kind != 3 && uml_dp_p2p_input(np)) {
      // data parallel over NVLink peer memory: split-K sum + exchange + Adam in ONE kernel per rank
      rec(a->ev[6], stream);
      rc = uml_dp_fused_adam_update(a->partials, splits, np, np, a->W, a->upd.m, a->upd.v, a->upd.lr, a->upd.beta1,
                                    a->upd.beta2, a->upd.eps, a->upd.weight_decay, a->upd.step, a->upd.kind == 1, a->W16,
                                    stream);
      rec(a->ev[7], stream);
      return rc;
    }
    rc = uml_sum_partials(a->partials, splits, np, np, dp ? dp_local_sum_target(a, np) : a->dW_out, stream);
    if (rc || !dp) return rc;
    return dp_reduce_and_update(a, np, stream);
  }
  if (a->upd.kind == 3) {
    UML_REQUIRE(a->dW_scratch, "linear_step: SGD on the bf16 path needs dW_scratch");
    rc = uml_sum_partials(a->partials, splits, np, np, a->dW_scratch, stream);
    if (rc) return rc;
    return uml_sgd_step(a->W, a->dW_scratch, nullptr, 0.f, a->upd.m, np, a->upd.lr, a->upd.momentum, a->upd.weight_decay,
                        a->upd.step, a->W16, stream);
  }
  rec(a->ev[6], stream);
  rc = uml_adamw_step_partials(a->W, a->partials, splits, np, a->upd.m, a->upd.v, np, a->upd.lr, a->upd.beta1,
                               a->upd.beta2, a->upd.eps, a->upd.weight_decay, a->upd.step, a->upd.kind == 1, a->W16,
                               nullptr, stream);
  rec(a->ev[7], stream);
  return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// gradient diagnostics of one step (uml_linear_run_diag, uml_linear_grad_diag)
static bool aligned16(const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15) == 0; }

// the image run (nullptr: none) and the text run (nullptr: none) of a step
static void diag_runs(const uml_linear_step_args* a, const uml_linear_diag* d, const uml_segment** img, const uml_segment** txt) {
  *img = d->has_img ? &a->seg[0] : nullptr;
  *txt = a->nseg > (d->has_img ? 1 : 0) ? &a->seg[d->has_img ? 1 : 0] : nullptr;
}

// bf16 scratch: [slots | A partials (cap planes of C * D) | B partials (cap planes)]
static int64_t diag_partials_offset() { return 4 * static_cast<int64_t>(uml::grad_diag_partial_slots()); }
static int64_t diag_partial_cap(const uml_linear_step_args* a, const uml_linear_diag* d) {
  return (d->scratch_floats - diag_partials_offset()) / (2 * static_cast<int64_t>(a->n_classes) * a->dim);
}

static int check_linear_diag(const uml_linear_step_args* a, const uml_linear_diag* d, const float* out) {
  UML_REQUIRE(a && d && d->scratch && out, "linear_grad_diag: null diagnostics buffer");
  UML_REQUIRE(a->nseg >= 1 && a->nseg <= UML_MAX_SEGMENTS && (d->has_img == 0 || d->has_img == 1) &&
                  !(a->nseg == 2 && !d->has_img),
              "linear_grad_diag: seg[0] is the image run (has_img) and a second run is the text run");
  UML_REQUIRE(!a->dp_allreduce && !a->dW_out, "linear_grad_diag: data-parallel steps have no per-step diagnostics");
  UML_REQUIRE(a->precision == 0 || a->precision == 1, "linear_grad_diag: precision must be 0 or 1");
  UML_REQUIRE(a->dim > 0 && a->n_classes > 0 && a->dim % (a->precision ? 8 : 4) == 0,
              "linear_grad_diag: dim must be a multiple of %d", a->precision ? 8 : 4);
  const uml_segment *img, *txt;
  diag_runs(a, d, &img, &txt);
  UML_REQUIRE(!txt || txt->n == 0 || txt->loss_weight > 0.f,
              "linear_grad_diag: alpha %g <= 0, the text-loss gradient cannot be recovered from G",
              static_cast<double>(txt ? txt->loss_weight : 0.f));
  UML_REQUIRE(!img || img->n == 0 || img->loss_weight == 1.f, "linear_grad_diag: the image run's loss weight must be 1");
  UML_REQUIRE(a->G && aligned16(a->G) && a->ldg % (a->precision ? 64 : 4) == 0 && a->ldg >= a->n_classes,
              "linear_grad_diag: G must be 16-byte aligned with ldg a multiple of %d", a->precision ? 64 : 4);
  if (a->precision == 0) {
    for (int k = 0; k < a->nseg; ++k)
      UML_REQUIRE(a->seg[k].n == 0 || (a->seg[k].rows && aligned16(a->seg[k].rows) && a->seg[k].ld % 4 == 0),
                  "linear_grad_diag: run %d rows must be 16-byte aligned with ld a multiple of 4", k);
  } else {
    UML_REQUIRE(a->X16 && aligned16(a->X16), "linear_grad_diag: X16 must be 16-byte aligned");
  }
  const int64_t need = a->precision == 0 ? uml_linear_diag_scratch_floats(0, 1, a->dim, a->n_classes)
                                         : diag_partials_offset() + 2 * static_cast<int64_t>(a->n_classes) * a->dim;
  UML_REQUIRE(aligned16(d->scratch) && d->scratch_floats >= need, "linear_grad_diag: scratch holds %lld floats, %lld needed",
              static_cast<long long>(d->scratch_floats), static_cast<long long>(need));
  return 0;
}

static int linear_grad_diag(const uml_linear_step_args* a, const uml_linear_diag* d, float* out, cudaStream_t st) {
  using namespace uml;
  const uml_segment *img, *txt;
  diag_runs(a, d, &img, &txt);
  const int64_t n0 = img ? img->n : 0, n1 = txt ? txt->n : 0;
  const float alpha = txt ? txt->loss_weight : 1.f;
  if (n0 + n1 == 0) {
    UML_CUDA(cudaMemsetAsync(out, 0, 4 * sizeof(float), st));
    return 0;
  }
  if (a->precision == 0) {
    const float* rows[2] = {img ? static_cast<const float*>(img->rows) : nullptr, txt ? static_cast<const float*>(txt->rows) : nullptr};
    const int64_t* idx[2] = {img ? img->idx : nullptr, txt ? txt->idx : nullptr};
    const int64_t ld[2] = {img ? img->ld : 0, txt ? txt->ld : 0};
    return grad_diag_f32_one(rows, idx, ld, n0, n1, a->dim, a->n_classes, static_cast<const float*>(a->G), a->ldg, alpha,
                             d->scratch, out, st);
  }
  // bf16: A over rows [0, n0) of X16 and G, B over rows [n0, n0 + n1) - 16-byte aligned sub-ranges (dim % 8 == 0,
  // ldg % 64 == 0) - each as split-K partials into scratch, then one reduction and the finish
  const int64_t n = static_cast<int64_t>(a->n_classes) * a->dim, cap = diag_partial_cap(a, d);
  float* pa = d->scratch + diag_partials_offset();
  float* pb = pa + cap * n;
  const uint16_t* G = static_cast<const uint16_t*>(a->G);
  int32_t na = 0, nb = 0;
  if (n0 > 0) {
    na = static_cast<int32_t>(std::min<int64_t>(cap, std::max(1, uml_tc_dw_splits(n0, a->dim, a->n_classes))));
    if (uml_head_bwd_dw_bf16(G, a->ldg, a->X16, n0, a->dim, a->n_classes, pa, na, st)) return 1;
  }
  if (n1 > 0) {
    nb = static_cast<int32_t>(std::min<int64_t>(cap, std::max(1, uml_tc_dw_splits(n1, a->dim, a->n_classes))));
    if (uml_head_bwd_dw_bf16(G + n0 * a->ldg, a->ldg, a->X16 + n0 * a->dim, n1, a->dim, a->n_classes, pb, nb, st)) return 1;
  }
  return grad_diag_partials_one(n0 > 0 ? pa : nullptr, na, pb, nb, n, n1, alpha, d->scratch, out, st);
}
