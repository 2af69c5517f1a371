"""Sweep-level batching (SURVEY §8 f-1): K heads of one hyper-parameter sweep advanced in lock step.

The reference's ``sweep`` (finetune.py:406-448) trains every lr x weight-decay combination of ``HYPER_DICT``
(engine/optimizer/default.py) one after the other over the same banks; at its batch size of 32 a step cannot fill one
SM.  ``HeadGroup`` keeps the K heads' weights and optimizer state in three ``[K, C*D]`` slabs and runs one step of all
of them with two launches - logits + softmax / CE and dW + update, both on the tensor cores (``uml_sweep_run``, csrc/sweep.cu).  Each head keeps its own sampler stream, learning-rate
schedule, weight decay, alpha and early-stopping state; a stopped head is masked out of the launches.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import torch

from .. import _lib
from .._lib import SWEEP_MAX_HEADS, SweepAdapterArgs, SweepArgs, SweepDiag, check
from ..ops import UPDATE_KINDS, grad_diag_record

MAX_HEADS = SWEEP_MAX_HEADS


def group_blockers(models, optimizers, image_loaders, text_loaders) -> List[str]:
    """Why these runs cannot share a HeadGroup (empty list: they can)."""
    why = []
    m0, o0 = models[0], optimizers[0]
    if len(models) > MAX_HEADS:
        why.append(f"more than {MAX_HEADS} heads")
    for m in models:
        if m.img_proj is not None:
            why.append("adapter (img_proj) variants are not batched")
            break
    if any(getattr(m, "learnable_temp", False) for m in models):
        why.append("learnable temperatures are not batched")
    if any(m.num_classes != m0.num_classes or m.shared_dim != m0.shared_dim for m in models):
        why.append("heads differ in shape")
    if not why and any(tuple(float(s) for s in m.scales()) != tuple(float(s) for s in m0.scales()) for m in models):
        why.append("heads differ in logit scale")
    if any(o.name != o0.name or o.defaults["betas"] != o0.defaults["betas"] or o.defaults["eps"] != o0.defaults["eps"]
           or o.defaults["momentum"] != o0.defaults["momentum"] for o in optimizers):
        why.append("optimizers differ in kind / betas / eps / momentum")
    for loaders in (image_loaders, text_loaders):
        live = [l for l in loaders if l is not None]
        if live and len(live) != len(loaders):
            why.append("runs differ in modality")
        elif live:
            l0 = live[0]
            if any(l.bank is not l0.bank or l.batch_size != l0.batch_size or l.drop_last != l0.drop_last
                   or not l.shuffle or l.generator is not None or l.shard_of is not None or l.upload != "epoch"
                   for l in live):
                why.append("loaders must share bank, batch size and protocol (shuffled, upload='epoch', no generator)")
    return why


def diag_blockers(models, alphas, text_loaders) -> List[str]:
    """Why these runs cannot log per-step gradient diagnostics as one group (``uml_sweep_run_diag``): the text-loss
    gradient is recovered from G, whose text rows carry alpha, and the tensor-core pass needs 16-byte rows."""
    why = []
    if any(l is not None for l in text_loaders) and any(float(a) <= 0 for a in alphas):
        why.append("gradient diagnostics need alpha > 0 when there are text rows")
    if any(int(m.shared_dim) % 4 for m in models):
        why.append("gradient diagnostics need feature widths that are multiples of 4")
    return why


ADAPTER_MAX_ROWS = 64  # rows per step of uml_sweep_adapter_run (one feature tile of its tensor-core kernels)
ADAPTER_MAX_CLASSES = 1024  # softmax / CE in the logits epilogue


def adapter_group_blockers(models, optimizers, image_loaders, text_loaders) -> List[str]:
    """Why these runs cannot share an AdapterHeadGroup (empty list: they can): UML heads with an image adapter and / or
    learnable temperatures, the runs of preset ``linear``."""
    why = []
    m0, o0 = models[0], optimizers[0]
    if len(models) > MAX_HEADS:
        why.append(f"more than {MAX_HEADS} heads")
    if not all(hasattr(m, "img_scale") for m in models):
        why.append("only UML heads (image adapter, per-modality temperatures) are batched with adapters")
        return why
    adapters = [m.img_proj is not None for m in models]
    if any(adapters) and not all(adapters):
        why.append("heads mix adapter and non-adapter variants")
    if any(m.num_classes != m0.num_classes or m.shared_dim != m0.shared_dim or m.img_indim != m0.img_indim for m in models):
        why.append("heads differ in shape")
    if any(bool(m.learnable_temp) != bool(m0.learnable_temp) for m in models):
        why.append("heads differ in learnable_temp")
    elif not m0.learnable_temp and any(tuple(float(s) for s in m.scales()) != tuple(float(s) for s in m0.scales())
                                       for m in models):
        why.append("heads differ in logit scale")
    if m0.num_classes > ADAPTER_MAX_CLASSES:
        why.append(f"more than {ADAPTER_MAX_CLASSES} classes")
    if m0.shared_dim % 4 or (m0.img_proj is not None and m0.img_indim % 4):
        why.append("feature widths must be multiples of 4")
    rows = sum(ls[0].batch_size for ls in (image_loaders, text_loaders) if ls and ls[0] is not None)
    if rows > ADAPTER_MAX_ROWS:
        why.append(f"more than {ADAPTER_MAX_ROWS} rows per step")
    if any(o.name != o0.name or o.defaults["betas"] != o0.defaults["betas"] or o.defaults["eps"] != o0.defaults["eps"]
           or o.defaults["momentum"] != o0.defaults["momentum"] for o in optimizers):
        why.append("optimizers differ in kind / betas / eps / momentum")
    for loaders in (image_loaders, text_loaders):
        live = [l for l in loaders if l is not None]
        if live and len(live) != len(loaders):
            why.append("runs differ in modality")
        elif live:
            l0 = live[0]
            if any(l.bank is not l0.bank or l.batch_size != l0.batch_size or l.drop_last != l0.drop_last
                   or not l.shuffle or l.generator is not None or l.shard_of is not None or l.upload != "epoch"
                   for l in live):
                why.append("loaders must share bank, batch size and protocol (shuffled, upload='epoch', no generator)")
    return why


class HeadGroup:
    diag = diag_log = None  # uml_sweep_diag and its [log_slots, K, 4] device log (grad_diagnostics)

    def __init__(self, models: Sequence, optimizers: Sequence, image_bank, text_bank, max_img_rows: int,
                 max_txt_rows: int, device, log_slots: int = 128, grad_diagnostics: bool = False):
        self.K = K = len(models)
        if not 1 <= K <= MAX_HEADS:
            raise ValueError(f"a HeadGroup holds 1..{MAX_HEADS} heads")
        self.models, self.opts = list(models), list(optimizers)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("HeadGroup: heads must live on a CUDA device (no CPU path)")
        m0, o0 = models[0], optimizers[0]
        self.C, self.D = int(m0.num_classes), int(m0.shared_dim)
        self.kind = UPDATE_KINDS[o0.name]
        if self.kind == 0:
            raise ValueError("HeadGroup needs an optimizer")
        self.banks = (image_bank, text_bank)
        for b, width in zip(self.banks, self._row_widths(m0)):
            if b is not None and (b.features.dtype != torch.float32 or b.dim != width or not b.features.is_contiguous()):
                raise ValueError("HeadGroup: banks must be contiguous fp32 [N, row width]")
        self.max_rows = int(max_img_rows) + int(max_txt_rows)
        n = self.C * self.D
        self.stride = (n + 3) // 4 * 4
        self.W = torch.empty((K, self.stride), device=self.device)
        self.m = torch.zeros((K, self.stride), device=self.device)
        self.v = torch.zeros((K, self.stride), device=self.device) if o0.name != "sgd" else None
        for k, (model, opt) in enumerate(zip(models, optimizers)):
            p = model.head.weight
            if p.device.type != "cuda":
                raise RuntimeError("HeadGroup: heads must live on a CUDA device (no CPU path)")
            view = self.W[k, :n].view(self.C, self.D)
            view.copy_(p.data)
            p.data = view  # the module keeps working (state_dict, validate) on its slice of the slab
            st = opt.slot(p)
            if st["step"] != 0:
                raise ValueError("HeadGroup: optimizers must be fresh")
            st["m"] = self.m[k, :n].view(self.C, self.D)
            if self.v is not None:
                st["v"] = self.v[k, :n].view(self.C, self.D)
        self.ldg = (self.C + 3) // 4 * 4
        self.G = torch.empty((K, self.max_rows, self.ldg), device=self.device)
        self.row_loss = torch.empty((K, self.max_rows), device=self.device)
        self.row_correct = torch.empty((K, self.max_rows), device=self.device, dtype=torch.int32)
        self.log_slots = int(log_slots)
        self.stats_log = torch.zeros((self.log_slots, K, 2, 4), device=self.device)
        # grad_diagnostics: the reference's per-step gradient probes of every head, four sums per step and head
        if grad_diagnostics:
            self.diag_log = torch.zeros((self.log_slots, K, 4), device=self.device)
            n = _lib.load().uml_sweep_diag_scratch_floats(K, self.D, self.C)
            self._diag_scratch = torch.empty(n, device=self.device)
            self.diag = SweepDiag()
            self.diag.scratch, self.diag.scratch_floats = self._diag_scratch.data_ptr(), n
        self.launches = 0
        s_i, s_t = (float(s) for s in m0.scales())
        a = self.args = SweepArgs()
        a.n_heads, a.dim, a.n_classes, a.kind = K, self.D, self.C, self.kind
        for s, b in enumerate(self.banks):
            if b is not None:
                a.bank[s], a.bank_ld[s], a.labels[s] = b.features.data_ptr(), b.features.stride(0), b.labels.data_ptr()
                a.perm_len[s] = len(b)
        a.scale[0], a.scale[1] = s_i, s_t
        a.W, a.m, a.v = self.W.data_ptr(), self.m.data_ptr(), (self.v.data_ptr() if self.v is not None else None)
        a.head_stride = self.stride
        a.G, a.ldg, a.max_rows = self.G.data_ptr(), self.ldg, self.max_rows
        a.row_loss, a.row_correct = self.row_loss.data_ptr(), self.row_correct.data_ptr()
        a.beta1, a.beta2 = o0.defaults["betas"]
        a.eps, a.momentum = o0.defaults["eps"], o0.defaults["momentum"]
        for k, (model, opt) in enumerate(zip(models, optimizers)):
            a.weight_decay[k] = opt.group_of(model.head.weight)["weight_decay"]

    def run(self, perms_img: Optional[Sequence[torch.Tensor]], perms_txt: Optional[Sequence[torch.Tensor]], pos_img: int,
            pos_txt: int, rows: Sequence[Sequence[int]], lrs: Sequence[Sequence[float]], alphas: Sequence[float],
            active: Sequence[bool], slot0: int):
        """Enqueue ``len(rows)`` consecutive steps of every active head.  ``perms_*[k]``: head k's epoch permutation on
        the device; ``rows[i] = (image rows, text rows)`` of step i; ``lrs[i][k]``; stats go to log slots slot0...;
        all on the current stream, no synchronisation."""
        n, K, a = len(rows), self.K, self.args
        s0 = slot0 % self.log_slots
        if n == 0 or not any(active):
            return
        if s0 + n > self.log_slots:
            raise ValueError("HeadGroup.run: the steps of one call must fit the stats log without wrapping")
        for s, perms in enumerate((perms_img, perms_txt)):
            for k in range(K):
                if perms is None:
                    a.perm[s][k] = None
                    continue
                t = perms[k]
                if t.dtype != torch.int64 or not t.is_cuda or not t.is_contiguous() or t.numel() < a.perm_len[s]:
                    raise ValueError("HeadGroup.run: permutations must be contiguous CUDA int64 tensors covering the bank")
                a.perm[s][k] = t.data_ptr()
        a.pos[0], a.pos[1] = int(pos_img), int(pos_txt)
        step = None
        for k in range(K):
            a.alpha[k] = float(alphas[k])
            a.active[k] = 1 if active[k] else 0
            if active[k]:
                st = self.opts[k].slot(self.models[k].head.weight)
                if step is None:
                    step = st["step"]
                elif st["step"] != step:
                    raise ValueError("HeadGroup.run: active heads must have taken the same number of steps")
        a.step = step + 1
        a.stats = self.stats_log[s0].data_ptr()
        if self.diag is not None:
            self.diag.out = self.diag_log[s0].data_ptr()
        rows_c = (C.c_int64 * (2 * n))(*[int(x) for r in rows for x in r])
        lr_c = (C.c_float * (n * K))(*[float(x) for l in lrs for x in l])
        l0 = _lib.load().uml_sweep_launch_count()
        check(self._enqueue(n, rows_c, lr_c))
        launched = (_lib.load().uml_sweep_launch_count() - l0) & 0x7FFFFFFF  # two to seven kernels per step (csrc/sweep.cu)
        self.launches += launched
        _lib.LAUNCH_COUNT[0] += launched
        for k in range(K):
            if active[k]:
                for p in self._trained(self.models[k]):
                    self.opts[k].slot(p)["step"] += n

    def _row_widths(self, m0):
        """Widths of the image and text bank rows."""
        return self.D, self.D

    def _trained(self, model):
        """The parameters of a head that one step updates."""
        return [model.head.weight]

    def _enqueue(self, n, rows_c, lr_c):
        st = torch.cuda.current_stream().cuda_stream
        if self.diag is not None:
            return _lib.load().uml_sweep_run_diag(C.byref(self.args), None, C.byref(self.diag), n, rows_c, lr_c, st)
        return _lib.load().uml_sweep_run(C.byref(self.args), n, rows_c, lr_c, st)

    KERNELS = ("sweep_logits", "sweep_softmax_ce", "sweep_dw_update", "sweep_stats")

    def time_last_step(self, enable: bool = True):
        """Bracket the four launch sites of the LAST step of every following ``run`` with CUDA events (a site whose work was
        fused into its neighbour spans nothing)."""
        self._ev = [torch.cuda.Event(enable_timing=True) for _ in range(8)] if enable else []
        for i in range(8):
            if enable:
                self._ev[i].record()  # forces creation of the underlying cudaEvent_t
                self.args.ev[i] = self._ev[i].cuda_event
            else:
                self.args.ev[i] = None
        self._time_diag(enable)

    def kernel_times_ms(self):
        """Device time of each launch of the last timed step (call after a synchronize); with gradient diagnostics also
        ``sweep_grad_diag`` (its two launches)."""
        ev = getattr(self, "_ev", [])
        out = {name: ev[2 * i].elapsed_time(ev[2 * i + 1]) for i, name in enumerate(self.KERNELS)} if ev else {}
        dev = getattr(self, "_diag_ev", [])
        if dev:
            out["sweep_grad_diag"] = dev[0].elapsed_time(dev[1])
        return out

    def _time_diag(self, enable):
        """The event pair around the diagnostics launches of the last step of every following ``run``."""
        if self.diag is None:
            return
        self._diag_ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)] if enable else []
        for i in range(2):
            if enable:
                self._diag_ev[i].record()
            self.diag.ev[i] = self._diag_ev[i].cuda_event if enable else None

    def read_log(self, slots: Sequence[int], has_img: bool, has_txt: bool):
        """Per-step stats of the given log slots as ``{name: [len(slots)][K] nested lists}`` for image_loss, text_loss,
        img_acc, text_acc (zeros for an absent modality) and, with gradient diagnostics, ``grad_diag``: the reference's
        four gradient-probe keys per step and head (``ops.grad_diag_record``); one synchronising D2H copy of the log."""
        L = self.log_slots
        if self.diag_log is None:
            raw = self.stats_log.cpu().numpy()
        else:  # both logs in one copy
            both = torch.cat((self.stats_log.view(L, -1), self.diag_log.view(L, -1)), 1).cpu().numpy()
            raw, diag = both[:, :self.K * 8].reshape(L, self.K, 2, 4), both[:, self.K * 8:].reshape(L, self.K, 4)
        ints = raw.view("int32")
        idx = [s % L for s in slots]
        zeros = [[0.0] * self.K for _ in idx]
        out = {"image_loss": zeros, "text_loss": zeros, "img_acc": zeros, "text_acc": zeros}
        for name_l, name_a, s, present in (("image_loss", "img_acc", 0, has_img), ("text_loss", "text_acc", 1, has_txt)):
            if present:
                out[name_l] = raw[idx, :, s, 0].tolist()
                out[name_a] = (ints[idx, :, s, 2] / ints[idx, :, s, 3].clip(min=1)).tolist()
        if self.diag_log is not None:
            numel, two = self.C * self.D, has_img and has_txt
            out["grad_diag"] = [[grad_diag_record(*(float(x) for x in diag[i, k]), numel, two) for k in range(self.K)]
                                for i in idx]
        return out


class AdapterHeadGroup(HeadGroup):
    """HeadGroup for UML heads with an image adapter (``img_proj``, Dv -> D) and / or learnable temperatures
    (``img_scale``, ``txt_scale``): one step of all K heads is five launches (``uml_sweep_adapter_run``) - Z = X Wp^T,
    logits + softmax / CE over [Z; X_txt] (+ per-row d loss / d scale), dZ = G W, head dW + update + statistics +
    temperature update, adapter dWp + update; two without an adapter.  Besides the head's slabs, the adapters and
    their optimizer state live in ``[K, D*Dv]`` slabs and the temperatures in ``[K, 2]`` ones; every module's
    parameters and optimizer state become views into them."""

    KERNELS = ("sweep_adapter_z", "sweep_logits", "sweep_adapter_dz", "sweep_dw_update", "sweep_adapter_dw_update")

    def __init__(self, models: Sequence, optimizers: Sequence, image_bank, text_bank, max_img_rows: int,
                 max_txt_rows: int, device, log_slots: int = 128, grad_diagnostics: bool = False):
        super().__init__(models, optimizers, image_bank, text_bank, max_img_rows, max_txt_rows, device, log_slots,
                         grad_diagnostics)
        if self.max_rows > ADAPTER_MAX_ROWS:
            raise ValueError(f"AdapterHeadGroup: at most {ADAPTER_MAX_ROWS} rows per step")
        K, D, m0 = self.K, self.D, models[0]
        self.Dv = int(m0.img_indim) if m0.img_proj is not None else 0
        self.learnable = bool(m0.learnable_temp)
        sgd = optimizers[0].name == "sgd"
        ad = self.adapter_args = SweepAdapterArgs()

        def adopt(slabs, k, p, shape, opt):
            """p.data and its optimizer state become views of row k of the (param, m, v) slabs."""
            n = p.numel()
            view = slabs[0][k, :n].view(shape)
            view.copy_(p.data)
            p.data = view
            st = opt.slot(p)
            if st["step"] != 0:
                raise ValueError("AdapterHeadGroup: optimizers must be fresh")
            st["m"] = slabs[1][k, :n].view(shape)
            if slabs[2] is not None:
                st["v"] = slabs[2][k, :n].view(shape)

        if self.Dv:
            self.a_stride = (D * self.Dv + 3) // 4 * 4
            self.Wp = torch.empty((K, self.a_stride), device=self.device)
            self.mp = torch.zeros((K, self.a_stride), device=self.device)
            self.vp = None if sgd else torch.zeros((K, self.a_stride), device=self.device)
            for k, (model, opt) in enumerate(zip(models, optimizers)):
                adopt((self.Wp, self.mp, self.vp), k, model.img_proj.weight, (D, self.Dv), opt)
            self.ldz = D
            self.Z = torch.empty((K, max(int(max_img_rows), 1), D), device=self.device)
            self.dZ = torch.empty_like(self.Z)
            ad.img_dim, ad.adapter_stride = self.Dv, self.a_stride
            ad.W, ad.m = self.Wp.data_ptr(), self.mp.data_ptr()
            ad.v = self.vp.data_ptr() if self.vp is not None else None
            ad.Z, ad.dZ, ad.ldz, ad.max_img_rows = self.Z.data_ptr(), self.dZ.data_ptr(), self.ldz, self.Z.shape[1]
        if self.learnable:
            self.T = torch.empty((K, 2), device=self.device)
            self.Tm = torch.zeros((K, 2), device=self.device)
            self.Tv = None if sgd else torch.zeros((K, 2), device=self.device)
            for k, (model, opt) in enumerate(zip(models, optimizers)):
                for j, p in enumerate((model.img_scale, model.txt_scale)):
                    adopt((self.T[:, j:j + 1], self.Tm[:, j:j + 1], self.Tv[:, j:j + 1] if self.Tv is not None else None),
                          k, p, (), opt)
            self.row_dscale = torch.empty((K, self.max_rows), device=self.device)
            ad.scale_param, ad.scale_m = self.T.data_ptr(), self.Tm.data_ptr()
            ad.scale_v = self.Tv.data_ptr() if self.Tv is not None else None
            ad.row_dscale = self.row_dscale.data_ptr()

    def _row_widths(self, m0):
        return (int(m0.img_indim) if m0.img_proj is not None else self.D), self.D

    def _trained(self, model):
        ps = [model.head.weight]
        if model.img_proj is not None:
            ps.append(model.img_proj.weight)
        if model.learnable_temp:
            ps += [model.img_scale, model.txt_scale]
        return ps

    def _enqueue(self, n, rows_c, lr_c):
        st = torch.cuda.current_stream().cuda_stream
        if self.diag is not None:
            return _lib.load().uml_sweep_run_diag(C.byref(self.args), C.byref(self.adapter_args), C.byref(self.diag), n,
                                                  rows_c, lr_c, st)
        return _lib.load().uml_sweep_adapter_run(C.byref(self.args), C.byref(self.adapter_args), n, rows_c, lr_c, st)

    def image_scales(self):
        """Every head's image-run temperature, one read-back (what evaluation multiplies the logits by)."""
        if self.learnable:
            return self.T[:, 0].tolist()
        return [float(m.scales()[0]) for m in self.models]

    def time_last_step(self, enable: bool = True):
        """Bracket the five launch sites of the LAST step of every following ``run`` with CUDA events (a skipped site
        spans nothing)."""
        n = 2 * len(self.KERNELS)
        self._ev = [torch.cuda.Event(enable_timing=True) for _ in range(n)] if enable else []
        for i in range(n):
            if enable:
                self._ev[i].record()
                self.adapter_args.ev[i] = self._ev[i].cuda_event
            else:
                self.adapter_args.ev[i] = None
        self._time_diag(enable)
