"""The fused UML training step (L3 hot loop body) on device.

One call to ``StepEngine.step`` is one iteration of the reference loop body
(vision_language/finetune.py:163-195): fetch an image batch and an unpaired text batch, push both
through the shared head, ``loss = CE(img) + alpha * CE(txt)``, backward to the shared weights,
optimizer update.  No autograd graph, no ``.item()``: per-step losses / hit counts land in a device
log that the caller reads at evaluation cadence.

Two arithmetic paths (chosen per step from the row count unless forced):
  fp32  SIMT kernels, exact like the reference; rows are gathered inside the GEMMs by index and the
        optimizer update runs in the dW epilogue: 4 launches for the linear head - or ONE cooperative
        launch for the whole step at the reference's batch sizes (csrc/simt.cu head_step_fused_kernel).
  bf16  tcgen05 kernels: row gather from the bf16 shadow banks (prefetched one step ahead on a side stream)
        -> fused forward/CE/G -> fix-up -> split-K dW -> optimizer update that also sums the split-K
        partials and refreshes the bf16 weight shadow: 5 launches, enqueued by one C call per chunk of steps.
Data-parallel runs: every rank takes its slice of the global batch (or owns a bank shard with its own sampler);
the step ends with one kernel per rank that sums the local partials, exchanges the gradient over NVLink peer
memory and applies the identical update everywhere (ncclAllReduce from inside the launcher as the fallback).
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import ops
from .datasets.utils import IndexBatch, local_slice as _local_slice

BF16_MIN_ROWS = 1024  # below this the step is launch-bound and the exact fp32 path is used


def dp_loss_weights(n_img_local, n_txt_local, alpha, n_img_global=None, n_txt_global=None):
    """Per-run loss weights of one rank in a data-parallel step.

    The kernels divide a run's gradient by the LOCAL row count; the loss is a mean over the GLOBAL
    batch (finetune.py:186-188), so a rank holding n_local of n_global rows scales its run by
    n_local / n_global.  Summing the ranks' gradients (all-reduce) then gives exactly the single-process
    gradient; the text run also carries alpha."""
    wi = 1.0 if not n_img_global or not n_img_local else n_img_local / float(n_img_global)
    wt = alpha if not n_txt_global or not n_txt_local else alpha * n_txt_local / float(n_txt_global)
    return wi, wt


def _local(batch, rank, world):
    """This rank's rows of a step's batch: a slice of a GLOBAL batch, or the batch itself when the loader already
    is per-rank (sharded sampler, ``global_n`` set)."""
    if batch is None or world == 1 or batch.global_n is not None:
        return batch
    return _local_slice(batch, rank, world)


def _global_rows(batch, world):
    """Rows of the global batch this step's mean is taken over (None in single-process runs)."""
    if batch is None or world == 1:
        return None
    return batch.global_n if batch.global_n is not None else batch.n


_DP_READY = False


def ensure_dp_comm():
    """One NCCL communicator per process for the step launcher (csrc/dp.cu).  Rank 0 creates the NCCL id, it is
    broadcast through torch.distributed, every rank joins."""
    global _DP_READY
    if _DP_READY:
        return
    import ctypes as C
    from .._lib import check, load
    dist = torch.distributed
    rank, world = dist.get_rank(), dist.get_world_size()
    buf = (C.c_ubyte * 128)()
    if rank == 0:
        check(load().uml_dp_unique_id(buf))
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.tensor(list(buf), dtype=torch.uint8, device=dev)
    dist.broadcast(t, src=0)
    raw = bytes(t.cpu().tolist())
    check(load().uml_dp_init(C.c_char_p(raw), rank, world))
    _DP_READY = True


_P2P_FLOATS = 0


def ensure_dp_p2p(max_floats: int):
    """Exchange blocks of the NVLink peer-memory all-reduce (csrc/dp.cu), sized for gradients of ``max_floats``:
    allocate, all-gather the CUDA IPC handles through torch.distributed, open the peers.  UML_DP_P2P=0 keeps NCCL."""
    global _P2P_FLOATS
    import ctypes as C
    import os
    from .._lib import check, load
    dist = torch.distributed
    if os.environ.get("UML_DP_P2P", "1") == "0" or dist.get_backend() != "nccl" or max_floats <= _P2P_FLOATS:
        return
    rank, world = dist.get_rank(), dist.get_world_size()
    if world > 16:
        return
    # re-sizing (a later job of the same process with a larger head): every rank unmaps its peers, THEN - after a
    # barrier - frees its own exported block; freeing while a peer still has the block open is undefined in CUDA IPC
    check(load().uml_dp_p2p_close_peers())
    dist.barrier()
    h = (C.c_ubyte * 64)()
    check(load().uml_dp_p2p_alloc(int(max_floats), h))
    dev = torch.device("cuda", torch.cuda.current_device())
    mine = torch.tensor(list(h), dtype=torch.uint8, device=dev)
    allh = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allh, mine)
    raw = b"".join(bytes(t.cpu().tolist()) for t in allh)
    check(load().uml_dp_p2p_open(C.c_char_p(raw), rank, world))
    dist.barrier()
    _P2P_FLOATS = int(max_floats)


class StepEngine:
    def __init__(self, model, optimizer, device, max_img_rows: int, max_txt_rows: int, log_slots: int = 128,
                 precision: str = "auto", dist_group=None, world_size: int = 1):
        if precision not in ("auto", "fp32", "bf16"):
            raise ValueError("precision must be auto, fp32 or bf16")
        self.model, self.opt, self.device = model, optimizer, torch.device(device)
        self.precision = precision
        self.C, self.D, self.Dv = model.num_classes, model.shared_dim, model.img_indim
        self.adapter = model.img_proj is not None
        self.max_img, self.max_txt = int(max_img_rows), int(max_txt_rows)
        self.max_rows = self.max_img + self.max_txt
        self.dist_group, self.world = dist_group, int(world_size)
        self.W = model.head.weight
        if self.W.device.type != "cuda":
            raise RuntimeError("StepEngine: the model must live on a CUDA device (no CPU path)")
        if self.world > 1:
            ensure_dp_comm()
            ensure_dp_p2p(max(p.numel() for p in model.parameters()))  # the head, or the larger adapter
            # replicas must start from identical bits (they apply identical updates and are never re-synchronised)
            for prm in model.parameters():
                torch.distributed.broadcast(prm.data, src=0)
        self.learnable = bool(getattr(model, "learnable_temp", False))
        self.ws32: Optional[ops.HeadWorkspace] = None
        self.ws16: Optional[ops.HeadWorkspace] = None
        self.log_slots = int(log_slots)
        self.stats_log = torch.zeros((self.log_slots, 2, 4), device=self.device, dtype=torch.float32)
        self.slot_modalities = [None] * self.log_slots
        self.dW = None       # fp32 gradient buffer (data-parallel / unfused paths)
        self.Z = self.dZ = None
        self.X16 = self.W16 = self.labels32 = self.partials = None
        self._w16_valid = False
        self.host_log = None
        self._event_pool = []
        self.profile_only = None
        self.prefetch = True      # uml_linear_run gathers step i+1's rows on a side stream during step i
        self.X16_alt = self.labels32_alt = self.X16_alt2 = self.labels32_alt2 = None
        self.shadow_banks = True  # keep a bf16 copy of each bank in HBM (+50% bank memory) for the tensor-core path
        self._args = None
        self.single_call = True  # False: dispatch every kernel from Python (debugging)
        self.profile = None  # set to {} to collect (start, end) CUDA events per kernel name

    # ------------------------------------------------------------------------------------ helpers
    def _timed(self, name, fn, *a, **k):
        if self.profile is None:
            return fn(*a, **k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn(*a, **k)
        e1.record()
        self.profile.setdefault(name, []).append((e0, e1))
        return r

    @staticmethod
    def _new_event_pair():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); e1.record()  # forces creation of the underlying cudaEvent_t
        return e0, e1

    def prepare_profile(self, n_steps, only=None):
        """Pre-create the CUDA events a profiled run of n_steps needs, so that creating them does not
        sit on the host's critical path inside the timed region.  ``only``: kernel names to bracket."""
        self.profile_only = set(only) if only else None
        self._event_pool = [self._new_event_pair() for _ in range((len(only) if only else 4) * n_steps)]
        self.profile = {}

    def kernel_times_ms(self):
        """Mean device time per launch of every profiled kernel (call after a synchronize)."""
        out = {}
        for k, v in (self.profile or {}).items():
            ts = [a.elapsed_time(b) for a, b in v]
            ts = [t for t in ts if t > 1e-4]  # pairs the launcher did not use stay at ~0
            if ts:
                out[k] = sum(ts) / len(ts)
        return out

    def step_timeline_ms(self):
        """From a profiled run with every kernel bracketed: mean time between the END of one bracketed kernel and the
        START of the next one on the stream (fix-up kernel + launch gaps fall in 'fwd_end->dw_start')."""
        p = self.profile or {}
        f, d, u = p.get("head_fwd_ce_bf16", []), p.get("head_bwd_dw_bf16", []), p.get("adamw_step_partials", [])
        n = min(len(f), len(d), len(u))
        if n < 2:
            return {}
        mean = lambda xs: sum(xs) / len(xs)
        out = {"fwd_end->dw_start": mean([f[i][1].elapsed_time(d[i][0]) for i in range(n)]),
               "dw_end->update_start": mean([d[i][1].elapsed_time(u[i][0]) for i in range(n)]),
               "update_end->next_fwd_start": mean([u[i][1].elapsed_time(f[i + 1][0]) for i in range(n - 1)]),
               "fwd_start->next_fwd_start": mean([f[i][0].elapsed_time(f[i + 1][0]) for i in range(n - 1)])}
        return out

    def _scales(self):
        si, st = self.model.scales()
        if self.learnable:  # device scalars, read by the kernels; never synchronise to fetch them
            return 0.0, 0.0, si.data, st.data
        return float(si), float(st), None, None

    def _use_bf16(self, rows: int) -> bool:
        if self.precision == "fp32":
            return False
        ok = self.D % 8 == 0 and self.C <= 1024 and (not self.adapter or self.Dv % 8 == 0)
        if self.precision == "bf16":
            if not ok:
                raise RuntimeError("bf16 path needs dim % 8 == 0 and <= 1024 classes")
            return True
        return ok and rows >= BF16_MIN_ROWS

    @staticmethod
    def _view(b: IndexBatch):
        """(rows, labels, idx) for a batch; sequential batches become dense views."""
        if b.idx is not None:
            return b.bank.features, b.bank.labels, b.idx
        return b.bank.features[b.start:b.start + b.n], b.bank.labels[b.start:b.start + b.n], None

    def invalidate_shadow(self):
        """Call after the weights were changed outside the engine (e.g. load_state_dict)."""
        self._w16_valid = False

    # ------------------------------------------------------------------------------------ step
    def step(self, img: Optional[IndexBatch], txt: Optional[IndexBatch], alpha: float, slot: int,
             global_img_rows: Optional[int] = None, global_txt_rows: Optional[int] = None):
        if img is None and txt is None:
            raise ValueError("at least one modality per step")
        n_i, n_t = (img.n if img else 0), (txt.n if txt else 0)
        slot %= self.log_slots
        # (a rank's local slice of a modality can be empty in a data-parallel run: only runs that are launched write a record)
        self.slot_modalities[slot] = (n_i > 0, n_t > 0)
        wi, wt = dp_loss_weights(n_i, n_t, alpha, global_img_rows, global_txt_rows)
        bf16 = self._use_bf16(n_i + n_t)
        if bf16:  # this step writes the operand buffers outside uml_linear_run: its gather pipeline starts cold next time
            from .._lib import load as _load_lib
            _load_lib().uml_linear_run_reset()
        if self.adapter and bf16:
            self._step_bf16_adapter(img, txt, n_i, n_t, wi, wt, slot)
        elif self.adapter or not self.single_call:
            # per-kernel dispatch: adapter variant on the exact path, or debugging
            (self._step_bf16 if bf16 else self._step_fp32)(img, txt, n_i, n_t, wi, wt, slot)
        else:
            self._step_single_call(img, txt, n_i, n_t, wi, wt, slot, bf16)

    # ------------------------------------------------------------------------------------ one C call
    def _fill_base(self, img, txt, n_i, n_t, wi, wt, bf16):
        """Fill the uml_linear_step_args struct for one iteration; returns (args, k, params)."""
        from .._lib import LinearStepArgs
        a = self._args
        if a is None:
            a = self._args = LinearStepArgs()
            a.dim, a.n_classes = self.D, self.C
        if bf16 and self.ws16 is None:
            self._alloc_bf16()
        if not bf16 and self.ws32 is None:
            self.ws32 = ops.HeadWorkspace(self.max_rows, self.C, self.device)
        ws = self.ws16 if bf16 else self.ws32
        s_i, s_t, sd_i, sd_t = self._scales()
        k = 0
        scale_params = []
        for b, cnt, s, w, sd, prm in ((img, n_i, s_i, wi, sd_i, getattr(self.model, "img_scale", None)),
                                      (txt, n_t, s_t, wt, sd_t, getattr(self.model, "txt_scale", None))):
            if b is None:
                continue
            rows, labels, idx = self._view(b)
            seg = a.seg[k]
            seg.rows, seg.labels, seg.idx = rows.data_ptr(), labels.data_ptr(), (idx.data_ptr() if idx is not None else None)
            seg.n, seg.ld, seg.scale, seg.loss_weight = cnt, rows.stride(0), s, w
            seg.label_idx, seg.scale_dev = None, (sd.data_ptr() if sd is not None else None)
            # bf16 shadow bank (built once per bank): the step then gathers with plain TMA copies, one launch
            seg.rows16 = b.bank.bf16().data_ptr() if (bf16 and idx is not None and self.shadow_banks) else None
            if self.learnable:
                st = self.opt.slot(prm)
                a.scale_param[k], a.scale_m[k] = prm.data.data_ptr(), st["m"].data_ptr()
                a.scale_v[k] = st["v"].data_ptr() if st["v"] is not None else None
                scale_params.append(prm)
            else:
                a.scale_param[k] = None
            k += 1
        a.nseg, a.precision = k, int(bf16)
        W = self.W.data
        a.W = W.data_ptr()
        a.G, a.ldg, a.g_capacity_rows = ws.G.data_ptr(), ws.ldg, ws.G.shape[0]
        a.row_loss, a.row_correct, a.row_dscale = ws.row_loss.data_ptr(), ws.row_correct.data_ptr(), ws.row_dscale.data_ptr()
        if bf16:
            a.X16, a.W16, a.labels32 = self.X16.data_ptr(), self.W16.data_ptr(), self.labels32.data_ptr()
            a.partials, a.max_splits, a.w16_valid = self.partials.data_ptr(), self.max_splits, int(self._w16_valid)
            a.tile_ws = ws.fac.data_ptr()
            if self.shadow_banks and self.prefetch:
                if self.X16_alt is None:  # second operand buffer: the next step's rows are gathered while this one runs
                    self.X16_alt = torch.empty_like(self.X16)
                    self.labels32_alt = torch.empty_like(self.labels32)
                    self.X16_alt2 = torch.empty_like(self.X16)   # third: the gather runs two steps ahead (step.cu)
                    self.labels32_alt2 = torch.empty_like(self.labels32)
                a.X16_alt, a.labels32_alt = self.X16_alt.data_ptr(), self.labels32_alt.data_ptr()
                a.X16_alt2, a.labels32_alt2 = self.X16_alt2.data_ptr(), self.labels32_alt2.data_ptr()
            else:
                a.X16_alt = a.labels32_alt = a.X16_alt2 = a.labels32_alt2 = None
        need_dw = self.world > 1 or (bf16 and self.opt.name == "sgd")
        if need_dw and self.dW is None:
            self.dW = torch.empty_like(W)
        a.dW_out = self.dW.data_ptr() if self.world > 1 else None
        a.dW_scratch = self.dW.data_ptr() if (bf16 and self.opt.name == "sgd" and self.world == 1) else None
        a.dp_allreduce = int(self.world > 1)
        for j in range(8):
            a.ev[j] = None
        return a, k, scale_params

    def _kernels_per_step(self, k, bf16):
        n = ((1 if self.shadow_banks else k) + 4 + (0 if self._w16_valid else 1)) if bf16 else 4
        # data parallel: the fused peer-memory tail replaces the update launch; over NCCL: + split sum + all-reduce
        return n + (k if self.learnable else 0) + (0 if self.world == 1 or _P2P_FLOATS else 2)

    def _step_single_call(self, img, txt, n_i, n_t, wi, wt, slot, bf16):
        """The whole iteration enqueued by uml_linear_step (csrc/step.cu): Python only fills a struct."""
        import ctypes as C
        from .._lib import LAUNCH_COUNT, check, load
        a, k, scale_params = self._fill_base(img if n_i else None, txt if n_t else None, n_i, n_t, wi, wt, bf16)
        for j, prm in enumerate(scale_params):
            st = self.opt.slot(prm)
            st["step"] += 1
            a.scale_step[j] = st["step"]
        a.upd = self.opt.update_struct(self.W)
        a.stats = self.stats_log[slot].data_ptr()
        if self.profile is not None:
            # cudaEvent pairs recorded by the C launcher around gather / forward / dW / update
            names = ("gather_bf16", "head_fwd_ce_bf16" if bf16 else "head_fwd_ce_f32",
                     "head_bwd_dw_bf16" if bf16 else "head_bwd_dw_f32", "adamw_step_partials")
            for j, nm in enumerate(names):
                if (not bf16 and j in (0, 3)) or (self.profile_only and nm not in self.profile_only):
                    # the fp32 path gathers inside its GEMMs and updates in the dW epilogue; profile_only restricts
                    # the bracketed kernels (every event pair costs host time and a small bubble on the stream)
                    continue
                e0, e1 = self._event_pool.pop() if self._event_pool else self._new_event_pair()
                a.ev[2 * j], a.ev[2 * j + 1] = e0.cuda_event, e1.cuda_event
                self.profile.setdefault(nm, []).append((e0, e1))
        f0 = load().uml_head_step_fused_count()
        check(load().uml_linear_step(C.byref(a), torch.cuda.current_stream().cuda_stream))
        # (a step the fused exact-path kernel took is one launch instead of four)
        LAUNCH_COUNT[0] += self._kernels_per_step(k, bf16) - 3 * ((load().uml_head_step_fused_count() - f0) & 0x7fffffff)
        self._w16_valid = bf16

    def run(self, batches, alpha, lrs, slot0):
        """Enqueue ``len(batches)`` consecutive iterations with as few host calls as possible.

        ``batches[j] = (img_batch | None, txt_batch | None)`` are the GLOBAL index batches of step j (a
        data-parallel rank takes its slice here), ``lrs[j]`` the learning rate the scheduler emitted for it
        and ``slot0 + j`` its slot in the stats log.  Consecutive steps that take the same arithmetic path
        go down in ONE uml_linear_run call."""
        import ctypes as C
        from .._lib import LAUNCH_COUNT, RunStep, check, load
        rank = torch.distributed.get_rank() if self.world > 1 else 0
        wgroup = self.opt.group_of(self.W)
        j = 0
        n_all = len(batches)
        while j < n_all:
            img_g, txt_g = batches[j]
            img, txt = _local(img_g, rank, self.world), _local(txt_g, rank, self.world)
            n_i, n_t = (img.n if img else 0), (txt.n if txt else 0)
            bf16 = self._use_bf16(n_i + n_t)
            if self.adapter or not self.single_call or n_i == 0 and img is not None or n_t == 0 and txt is not None:
                wgroup["lr"] = lrs[j]
                for g in self.opt.param_groups:
                    g["lr"] = lrs[j]
                self.step(img, txt, alpha, slot0 + j, _global_rows(img_g, self.world), _global_rows(txt_g, self.world))
                j += 1
                continue
            wi, wt = dp_loss_weights(n_i, n_t, alpha, _global_rows(img_g, self.world), _global_rows(txt_g, self.world))
            a, k, scale_params = self._fill_base(img, txt, n_i, n_t, wi, wt, bf16)
            a.upd = self.opt.update_struct(self.W)      # hyper-parameters; lr / step are patched per step below
            wst = self.opt.slot(self.W)
            wst["step"] -= 1
            # how many following steps share this path (same modalities, same arithmetic)?
            m = j
            steps = []
            ready, ready_seq, vouched = None, -1, True  # the newest 'indices uploaded' event among the chunk's batches
            while m < n_all:
                ig, tg = batches[m]
                if (ig is None) != (img_g is None) or (tg is None) != (txt_g is None):
                    break
                il, tl = _local(ig, rank, self.world), _local(tg, rank, self.world)
                ni, nt = (il.n if il else 0), (tl.n if tl else 0)
                if self._use_bf16(ni + nt) != bf16 or (il is not None and (ni == 0 or il.idx is None)) or \
                        (tl is not None and (nt == 0 or tl.idx is None)):
                    break
                w_i, w_t = dp_loss_weights(ni, nt, alpha, _global_rows(ig, self.world), _global_rows(tg, self.world))
                rs = RunStep()
                kk = 0
                for b_, cnt, w_ in ((il, ni, w_i), (tl, nt, w_t)):
                    if b_ is None:
                        continue
                    rs.idx[kk], rs.n[kk], rs.loss_weight[kk] = b_.idx.data_ptr(), cnt, w_
                    kk += 1
                    if b_.ready is None:
                        vouched = False
                    elif b_.ready_seq > ready_seq:
                        ready, ready_seq = b_.ready, b_.ready_seq
                rs.lr = lrs[m]
                wst["step"] += 1
                rs.opt_step = wst["step"]
                for jj, prm in enumerate(scale_params):
                    st = self.opt.slot(prm)
                    st["step"] += 1
                    rs.scale_step[jj] = st["step"]
                slot = (slot0 + m) % self.log_slots
                self.slot_modalities[slot] = (ig is not None and ig.n > 0, tg is not None and tg.n > 0)
                rs.stats = self.stats_log[slot].data_ptr()
                if self.profile is not None:
                    names = ("gather_bf16", "head_fwd_ce_bf16" if bf16 else "head_fwd_ce_f32",
                             "head_bwd_dw_bf16" if bf16 else "head_bwd_dw_f32", "adamw_step_partials")
                    for jn, nm in enumerate(names):
                        if (not bf16 and jn in (0, 3)) or (self.profile_only and nm not in self.profile_only):
                            continue
                        e0, e1 = self._event_pool.pop() if self._event_pool else self._new_event_pair()
                        rs.ev[2 * jn], rs.ev[2 * jn + 1] = e0.cuda_event, e1.cuda_event
                        self.profile.setdefault(nm, []).append((e0, e1))
                steps.append(rs)
                m += 1
            if not steps:  # the first step itself does not qualify (dense batch): fall back to the per-step path
                wgroup["lr"] = lrs[j]
                self.step(img, txt, alpha, slot0 + j, _global_rows(img_g, self.world), _global_rows(txt_g, self.world))
                j += 1
                continue
            # every index batch vouched for by an upload event: the gather pipeline may run through the call boundary
            a.idx_ready = ready.cuda_event if (vouched and ready is not None) else None
            arr = (RunStep * len(steps))(*steps)
            f0 = load().uml_head_step_fused_count()
            check(load().uml_linear_run(C.byref(a), arr, len(steps), torch.cuda.current_stream().cuda_stream))
            LAUNCH_COUNT[0] += self._kernels_per_step(k, bf16) * len(steps) - (0 if self._w16_valid or not bf16 else len(steps) - 1)
            LAUNCH_COUNT[0] -= 3 * ((load().uml_head_step_fused_count() - f0) & 0x7fffffff)
            self._w16_valid = bf16
            j = m

    # ------------------------------------------------------------------------------------ fp32
    def _step_fp32(self, img, txt, n_i, n_t, wi, wt, slot):
        if self.ws32 is None:
            self.ws32 = ops.HeadWorkspace(self.max_rows, self.C, self.device)
        ws, W = self.ws32, self.W.data
        s_i, s_t, sd_i, sd_t = self._scales()
        runs = []
        if img is not None and n_i:
            rows, labels, idx = self._view(img)
            if self.adapter:
                if self.Z is None:
                    self.Z = torch.empty((self.max_img, self.D), device=self.device)
                    self.dZ = torch.empty((self.max_img, self.D), device=self.device)
                Wp = self.model.img_proj.weight.data
                ops.gemm_nt(rows, Wp, self.Z, a_row_idx=idx, m=n_i)
                runs.append(ops.Run(self.Z, labels, None, n_i, s_i, wi, label_idx=idx, scale_dev=sd_i))
            else:
                runs.append(ops.Run(rows, labels, idx, n_i, s_i, wi, scale_dev=sd_i))
        if txt is not None and n_t:
            rows, labels, idx = self._view(txt)
            runs.append(ops.Run(rows, labels, idx, n_t, s_t, wt, scale_dev=sd_t))
        stats = self.stats_log[slot]
        self._timed("head_fwd_ce_f32", ops.head_fwd_ce_f32, runs, W, ws, stats=stats)
        if self.adapter and img is not None and n_i:
            # dZ = G_img W uses the head BEFORE its update; image rows are the first n_i rows of G
            ops.gemm_nn(ws.G, W, self.dZ, m=n_i, k=self.C)
        if self.learnable:
            k = 0
            if img is not None and n_i:
                self._apply_scalar(self.model.img_scale, stats[k, 1:2])
                k += 1
            if txt is not None and n_t:
                self._apply_scalar(self.model.txt_scale, stats[k, 1:2])
        if self.world > 1:
            if self.dW is None:
                self.dW = torch.empty_like(W)
            ops.head_bwd_dw_f32(runs, W, ws, dW=self.dW)
            torch.distributed.all_reduce(self.dW, group=self.dist_group)
            self.opt.apply(self.W, self.dW)
        else:
            self._timed("head_bwd_dw_f32", ops.head_bwd_dw_f32, runs, W, ws, update=self.opt.update_struct(self.W))
        if self.adapter and img is not None and n_i:
            rows, _, idx = self._view(img)
            Wp = self.model.img_proj.weight
            if self.world > 1:
                # data parallel on the exact path: this rank's dWp = dZ^T X_img (no fused update), summed over the ranks,
                # then the optimizer step - the same order of operations as the head's gradient above
                if getattr(self, "dWp", None) is None:
                    self.dWp = torch.empty_like(Wp.data)
                ops.gemm_tn(self.dZ, rows, self.dWp, k=n_i, m=self.D, n=self.Dv, b_row_idx=idx)
                torch.distributed.all_reduce(self.dWp, group=self.dist_group)
                self.opt.apply(Wp, self.dWp)
            else:
                ops.gemm_tn(self.dZ, rows, None, k=n_i, m=self.D, n=self.Dv, b_row_idx=idx, P=Wp.data,
                            update=self.opt.update_struct(Wp), ldc=Wp.data.stride(0))
        self._w16_valid = False

    def _apply_scalar(self, param, grad_view):
        if self.world > 1:
            g = grad_view.clone()
            torch.distributed.all_reduce(g, group=self.dist_group)
            grad_view = g
        self.opt.apply(param, grad_view)

    def _apply_scalars(self, pairs):
        """Optimizer steps of several scalar parameters (the learnable temperatures) with ONE all-reduce for all of them."""
        if self.world > 1 and len(pairs) > 1:
            g = torch.cat([v.reshape(1) for _, v in pairs])
            torch.distributed.all_reduce(g, group=self.dist_group)
            for i, (prm, _) in enumerate(pairs):
                self.opt.apply(prm, g[i:i + 1])
            return
        for prm, v in pairs:
            self._apply_scalar(prm, v)

    # ------------------------------------------------------------------------------------ bf16
    def _alloc_bf16(self):
        dev = self.device
        self.ws16 = ops.HeadWorkspace(self.max_rows, self.C, dev, bf16=True)
        self.X16 = torch.empty((self.max_rows, self.D), device=dev, dtype=torch.bfloat16)
        self.W16 = torch.empty((self.C, self.D), device=dev, dtype=torch.bfloat16)
        self.labels32 = torch.empty(self.max_rows, device=dev, dtype=torch.int32)
        self.max_splits = max(1, ops.tc_dw_splits(self.max_rows, self.D, self.C))
        self.partials = torch.empty((self.max_splits, self.C, self.D), device=dev)

    def _step_bf16(self, img, txt, n_i, n_t, wi, wt, slot):
        if self.ws16 is None:
            self._alloc_bf16()
        ws, W, n = self.ws16, self.W.data, n_i + n_t
        if not self._w16_valid:
            ops.cast_bf16(W, self.W16)
            self._w16_valid = True
        s_i, s_t, sd_i, sd_t = self._scales()
        rows_l, scales, weights, sdevs = [], [], [], []
        off = 0
        for b, cnt, s, w, sd in ((img, n_i, s_i, wi, sd_i), (txt, n_t, s_t, wt, sd_t)):
            if b is None or cnt == 0:
                continue
            feats, labels, idx = self._view(b)
            if idx is None:
                idx_arg = None
                self._timed("cast_bf16", ops.cast_bf16, feats, self.X16[off:off + cnt])
            else:
                idx_arg = idx
                self._timed("gather_bf16", ops.gather_rows, feats, idx, out=self.X16[off:off + cnt])
            ops.gather_labels(labels, idx_arg, cnt, self.labels32[off:off + cnt])
            rows_l.append(cnt); scales.append(s); weights.append(w); sdevs.append(sd)
            off += cnt
        segs = ops.tc_segments(rows_l, scales, weights, sdevs if self.learnable else None)
        self._timed("head_fwd_ce_bf16", ops.head_fwd_ce_bf16, self.X16, self.W16, self.labels32, segs, ws, ws.row_loss,
                    row_correct=ws.row_correct, row_dscale=ws.row_dscale if self.learnable else None, n_rows=n)
        stats = self.stats_log[slot]
        ops.reduce_tile_stats(ws.fac, n, len(rows_l), stats)
        if self.learnable:
            k = 0
            if n_i:
                self._apply_scalar(self.model.img_scale, stats[k, 1:2]); k += 1
            if n_t:
                self._apply_scalar(self.model.txt_scale, stats[k, 1:2])
        splits = min(self.max_splits, max(1, ops.tc_dw_splits(n, self.D, self.C)))
        self._timed("head_bwd_dw_bf16", ops.head_bwd_dw_bf16, ws.G, ws.ldg, self.X16, n, self.C, self.partials, splits)
        g, st = self.opt.group_of(self.W), self.opt.slot(self.W)
        if self.world > 1 or self.opt.name == "sgd":
            if self.dW is None:
                self.dW = torch.empty_like(W)
            ops.sum_partials(self.partials, splits, W.numel(), self.dW)
            if self.world > 1:
                torch.distributed.all_reduce(self.dW, group=self.dist_group)
            self.opt.apply(self.W, self.dW, shadow=self.W16)
        else:
            st["step"] += 1
            self._timed("adamw_step_partials", ops.adamw_step_partials, W, self.partials, splits, st["m"], st["v"],
                        lr=g["lr"], step=st["step"], weight_decay=g["weight_decay"], betas=g["betas"], eps=g["eps"],
                        decoupled=(self.opt.name == "adamw"), shadow=self.W16)

    # ------------------------------------------------------------------------------------ bf16 + adapter
    def _step_bf16_adapter(self, img, txt, n_i, n_t, wi, wt, slot):
        """Adapter variant (reference UML with img_proj, head.py:63-84) on the tensor cores:
        Z = X_img Wp^T -> shared head on [Z ; T] -> dZ = G_img W -> dW = G^T [Z ; T], dWp = dZ^T X_img."""
        dev, D, Dv, C = self.device, self.D, self.Dv, self.C
        if self.ws16 is None:
            self._alloc_bf16()  # ws16 (G), X16 -> [Z ; T] operand, W16, labels32, head partials
            self.Xi16 = torch.empty((self.max_img, Dv), device=dev, dtype=torch.bfloat16)
            self.dZ16 = torch.empty((self.max_img, D), device=dev, dtype=torch.bfloat16)
            self.Wp16 = torch.empty((D, Dv), device=dev, dtype=torch.bfloat16)
            self.proj_splits = max(1, ops.gemm_bf16_splits(D, Dv, self.max_img))
            self.partials_p = torch.empty((self.proj_splits, D, Dv), device=dev)
            self.dWp = None
        ws, W, Wp, n = self.ws16, self.W.data, self.model.img_proj.weight, n_i + n_t
        if not self._w16_valid:
            ops.cast_bf16(W, self.W16)
            ops.cast_bf16(Wp.data, self.Wp16)
            self._w16_valid = True
        s_i, s_t, sd_i, sd_t = self._scales()
        rows_l, scales, weights, sdevs = [], [], [], []
        if n_i:
            feats, labels, idx = self._view(img)
            if idx is None:
                ops.cast_bf16(feats, self.Xi16[:n_i])
                ops.gather_labels(labels, None, n_i, self.labels32[:n_i])
            else:
                ops.gather_rows_labels(feats, labels, idx, self.Xi16[:n_i], self.labels32[:n_i])
            ops.gemm_bf16(self.Xi16, self.Wp16, self.X16, n_i, D, Dv)  # Z -> rows [0, n_i) of the head operand
            rows_l.append(n_i); scales.append(s_i); weights.append(wi); sdevs.append(sd_i)
        if n_t:
            feats, labels, idx = self._view(txt)
            if idx is None:
                ops.cast_bf16(feats, self.X16[n_i:n])
                ops.gather_labels(labels, None, n_t, self.labels32[n_i:n])
            else:
                ops.gather_rows_labels(feats, labels, idx, self.X16[n_i:n], self.labels32[n_i:n])
            rows_l.append(n_t); scales.append(s_t); weights.append(wt); sdevs.append(sd_t)
        segs = ops.tc_segments(rows_l, scales, weights, sdevs if self.learnable else None)
        stats = self.stats_log[slot]
        self._timed("head_fwd_ce_bf16", ops.head_fwd_ce_bf16, self.X16, self.W16, self.labels32, segs, ws, None, n_rows=n,
                    stats=stats)  # the fix-up launch also reduces the per-run statistics
        if self.learnable:
            k, pairs = 0, []
            if n_i:
                pairs.append((self.model.img_scale, stats[k, 1:2])); k += 1
            if n_t:
                pairs.append((self.model.txt_scale, stats[k, 1:2]))
            self._apply_scalars(pairs)
        if n_i:
            # dZ = G_img W with the head BEFORE its update (W16 is refreshed by the optimizer kernel below)
            ops.gemm_bf16(ws.G, self.W16, self.dZ16, n_i, D, C, b_mn=True)
        splits = min(self.max_splits, max(1, ops.tc_dw_splits(n, D, C)))
        ops.head_bwd_dw_bf16(ws.G, ws.ldg, self.X16, n, C, self.partials, splits)
        side = None
        if self.world > 1 and n_i and _P2P_FLOATS >= max(self.W.numel(), Wp.numel()):
            # data parallel: the head's exchange + update (a kernel that mostly waits on NVLink) runs on a side stream
            # under the adapter's dWp GEMM; the adapter's own exchange follows both (the ranks' exchange blocks are shared)
            if getattr(self, "_dp_stream", None) is None:
                self._dp_stream = torch.cuda.Stream(device=dev)
                self._dp_ev = (torch.cuda.Event(), torch.cuda.Event())
            main = torch.cuda.current_stream(dev)
            self._dp_ev[0].record(main)
            side = self._dp_stream
            with torch.cuda.stream(side):
                side.wait_event(self._dp_ev[0])
                self._apply_partials(self.W, self.partials, splits, self.W16, "dW")
                self._dp_ev[1].record(side)
        else:
            self._apply_partials(self.W, self.partials, splits, self.W16, "dW")
        if n_i:
            ps = min(self.proj_splits, max(1, ops.gemm_bf16_splits(D, Dv, n_i)))
            ops.gemm_bf16(self.dZ16, self.Xi16, self.partials_p, D, Dv, n_i, a_mn=True, b_mn=True, n_splits=ps)
            if side is not None:
                torch.cuda.current_stream(dev).wait_event(self._dp_ev[1])
            self._apply_partials(Wp, self.partials_p, ps, self.Wp16, "dWp")

    def _apply_partials(self, param, partials, splits, shadow, buf_name):
        """Optimizer step of ``param`` from split-K partials (summed in the same kernel), with the
        data-parallel all-reduce in between when there is more than one rank."""
        g, st = self.opt.group_of(param), self.opt.slot(param)
        data = param.data
        if self.world > 1 and self.opt.name != "sgd" and _P2P_FLOATS >= data.numel() and data.numel() % 4 == 0:
            # the data-parallel tail in ONE kernel per rank: split-K sum -> exchange over NVLink peer memory -> Adam(W) +
            # bf16 shadow (csrc/dp.cu), for the head and for the adapter alike
            from .._lib import check, load
            st["step"] += 1
            check(load().uml_dp_fused_adam_update(partials.data_ptr(), int(splits), data.numel(), data.numel(), data.data_ptr(),
                                                  st["m"].data_ptr(), st["v"].data_ptr(), g["lr"], g["betas"][0], g["betas"][1],
                                                  g["eps"], g["weight_decay"], st["step"], int(self.opt.name == "adamw"),
                                                  shadow.data_ptr() if shadow is not None else None,
                                                  torch.cuda.current_stream().cuda_stream))
            return
        if self.world > 1 or self.opt.name == "sgd":
            buf = getattr(self, buf_name, None)
            if buf is None:
                buf = torch.empty_like(data)
                setattr(self, buf_name, buf)
            ops.sum_partials(partials, splits, data.numel(), buf)
            if self.world > 1:
                torch.distributed.all_reduce(buf, group=self.dist_group)
            self.opt.apply(param, buf, shadow=shadow)
        else:
            st["step"] += 1
            ops.adamw_step_partials(data, partials, splits, st["m"], st["v"], lr=g["lr"], step=st["step"],
                                    weight_decay=g["weight_decay"], betas=g["betas"], eps=g["eps"],
                                    decoupled=(self.opt.name == "adamw"), shadow=shadow)

    def local_batches(self, pair):
        """This rank's (image, text) rows of a step's pair of batches."""
        rank = torch.distributed.get_rank() if self.world > 1 else 0
        return _local(pair[0], rank, self.world), _local(pair[1], rank, self.world)

    # ------------------------------------------------------------------------------------ diagnostics (a-13)
    def grad_diagnostics(self, img: Optional[IndexBatch], txt: Optional[IndexBatch]):
        """The reference's per-step gradient probes (finetune.py:190-191, 200-206) for one pair of batches at the
        CURRENT weights: grad_img = d image_loss / d head.weight, grad_txt = d text_loss / d head.weight (each a
        plain mean CE, no alpha), their cosine, norms and sign-agreement rate.  Opt-in and off the hot path: two
        exact fp32 forward/dW passes, one per modality, then one reduction kernel; nothing is updated.  Returns
        the reference's logger keys; one host read of 4 floats."""
        if self.adapter:
            raise NotImplementedError("gradient diagnostics are wired for the linear head")
        W = self.W.data
        rows = max(img.n if img is not None else 0, txt.n if txt is not None else 0, 1)
        if getattr(self, "_diag", None) is None or self._diag[0].max_rows < rows:
            self._diag = (ops.HeadWorkspace(rows, self.C, self.device), torch.zeros_like(W), torch.zeros_like(W),
                          torch.empty(4 * 1024, device=self.device), torch.empty(4, device=self.device))
        ws, g_img, g_txt, scratch, out4 = self._diag
        s_i, s_t, sd_i, sd_t = self._scales()
        for b, s, sd, g in ((img, s_i, sd_i, g_img), (txt, s_t, sd_t, g_txt)):
            if b is None or b.n == 0:
                g.zero_()
                continue
            feats, labels, idx = self._view(b)
            run = [ops.Run(feats, labels, idx, b.n, s, 1.0, scale_dev=sd)]
            ops.head_fwd_ce_f32(run, W, ws)
            ops.head_bwd_dw_f32(run, W, ws, dW=g)
        both = img is not None and txt is not None and img.n > 0 and txt.n > 0
        ops.grad_diag(g_img, g_txt, scratch, out4)
        return ops.grad_diag_record(*out4.tolist(), W.numel(), both)

    # ------------------------------------------------------------------------------------ readback
    def copy_slot_to_host(self, slot):
        """Asynchronous D2H of one step's stats record into a pinned host ring (no host sync)."""
        if self.host_log is None:
            self.host_log = torch.zeros((self.log_slots, 2, 4), dtype=torch.float32).pin_memory()
        slot %= self.log_slots
        self.host_log[slot].copy_(self.stats_log[slot], non_blocking=True)

    def copy_slots_to_host(self, slot0, n):
        """copy_slot_to_host for n consecutive steps with one asynchronous copy per contiguous run of ring slots."""
        if self.host_log is None:
            self.host_log = torch.zeros((self.log_slots, 2, 4), dtype=torch.float32).pin_memory()
        s = slot0 % self.log_slots
        while n > 0:
            k = min(n, self.log_slots - s)
            self.host_log[s:s + k].copy_(self.stats_log[s:s + k], non_blocking=True)
            n -= k
            s = 0

    def read_log(self, slots, from_host_ring=False):
        """Per-step stats for the given slots: one synchronising D2H of the device log, or - when every
        step already pushed its record with ``copy_slot_to_host`` - a stream sync and a host read."""
        from .._lib import load as _load_lib
        if self.world > 1 and _P2P_FLOATS and _load_lib().uml_dp_p2p_failed():
            raise RuntimeError("data-parallel step: a peer rank stopped answering the NVLink gradient exchange (UML_DP_TIMEOUT_S); "
                               "the affected steps applied no update - the replicas may no longer agree, restart from a checkpoint")
        if from_host_ring and self.host_log is not None:
            torch.cuda.current_stream().synchronize()
            raw = self.host_log.clone()
        else:
            raw = self.stats_log.cpu()
        if self.ws16 is not None and _load_lib().uml_fwd_x_failed(self.ws16.fac.data_ptr()):
            raise RuntimeError("tensor-core step: a CTA waited a second for its peers (forward statistics exchange or the dW "
                               "kernel's split-K update); the affected step's results are undefined - restart from a checkpoint")
        ints = raw.view(torch.int32)
        out = []
        for s in slots:
            s %= self.log_slots
            has_i, has_t = self.slot_modalities[s]
            rec = {"image_loss": 0.0, "text_loss": 0.0, "img_acc": 0.0, "text_acc": 0.0}
            k = 0
            if has_i:
                n = max(1, int(ints[s, k, 3]))
                rec["image_loss"], rec["img_acc"] = float(raw[s, k, 0]), int(ints[s, k, 2]) / n
                k += 1
            if has_t:
                n = max(1, int(ints[s, k, 3]))
                rec["text_loss"], rec["text_acc"] = float(raw[s, k, 0]), int(ints[s, k, 2]) / n
            out.append(rec)
        return out
