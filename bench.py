#!/usr/bin/env python
"""bench.py - throughput of the UML training step on B200 (contract in the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg3] [--dump-outputs DIR]

Metric (BASELINE.json): UML train samples/sec (image + text rows consumed per second).
Workload at N=1 (``config.workload``): cfg3 = ImageNet full-data shapes, "ViT-L/14" 768-d features,
1000-class shared linear head + unpaired text bank, preset ``clip_linear`` arithmetic (logit scale
exp(4.60517), AdamW) at the THROUGHPUT batch of 70144 image + 3584 text rows per GPU and step (288 row units of 256
= 16 per CTA-pair group of the forward kernel; the text batch is sized so that 8 GPUs still fit the 29940-row text
bank; SURVEY.md section 8d; --workload cfg3_r1 is round 1's 34304 + 3584; the reference's own batch of 32 is a
latency-bound regime reported separately by --workload cfg2).
Synthetic seeded banks, random-init/zero-shot-init head.  One "step" = one full UML iteration:
gather(img) + gather(txt) -> shared head forward -> logit scale + softmax CE -> dW -> AdamW.

``value``  device-resident: banks and the K steps' index batches already in HBM, K steps timed with CUDA events
           (gather from the banks, forward, dW, update all inside the timed region).
``e2e``    the same K steps through the public ``uml_b200.finetune.train`` call with index batches copied
           from pinned host memory every step and every step's loss record copied back to the host.
``roofline`` dominant kernel (head forward/CE/G, tcgen05) timed with CUDA events inside the run.
``cpu_baseline`` / ``--impl reference``: the oracle port of the reference step on the host cores.
``--impl reference``: the UNMODIFIED reference's finetune.train() on the host cores (oracle/_ref, see oracle/build_ref.py).
Multi-GPU (torchrun): data-parallel, fixed per-GPU batch (weak scaling), banks row-sharded over the ranks with a
per-rank sampler, dW summed over the ranks by the step's last kernel (NVLink peer memory, csrc/dp.cu).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # batch / batch_txt: rows per modality per GPU and step.  cfg3: 70144 image + 3584 text rows = 288 row units of 256 =
    # exactly 16 per CTA-pair group of the forward kernel (18 groups x 4 class chunks x 2 CTAs = 144 SMs); the text batch is
    # sized so that 8 GPUs together (28672 rows) still fit the 29940-row CUPL text bank - per-GPU work stays fixed from 1
    # to 8 GPUs (weak scaling).  The batch is a free parameter of a throughput run (the reference trains at 32): per-step
    # costs that do not grow with it (update, launch gaps, pipeline fill of the two GEMM kernels: ~30 us) weigh 21 % at
    # round 1's 37888 rows, 13 % here; DESIGN.md lists the measured series 36864 / 73728 / 147456 rows.
    "cfg3": dict(n_img=1_281_167, n_txt=29_940, dim=768, classes=1000, batch=70144, batch_txt=3584, n_val=4096,
                 desc="ImageNet full-data CLIP ViT-L/14 768-d features + CUPL text, linear head, throughput batch"),
    # round 1's throughput batch (34304 + 3584 rows = 296 tiles of 128 = two waves over 148 SMs of the round-1 forward kernel)
    "cfg3_r1": dict(n_img=1_281_167, n_txt=29_940, dim=768, classes=1000, batch=34304, batch_txt=3584, n_val=4096,
                    desc="cfg3 at round 1's batch (34304 image + 3584 text rows per GPU and step)"),
    "cfg3_sym": dict(n_img=1_281_167, n_txt=29_940, dim=768, classes=1000, batch=18944, batch_txt=18944, n_val=4096,
                     desc="cfg3 with 18944 rows per modality per GPU (text epochs of two steps)"),
    # DINOv2 ViT-g (1536-d) image bank + OpenLLaMA-3B (3200-d) text bank, linear adapter img_proj 1536 -> 3200 + shared
    # head, learnable temperatures (preset "linear"), throughput batch; the full 1.28 M-row image bank (7.9 GB fp32 + 3.9 GB bf16)
    "cfg4": dict(n_img=1_281_167, n_txt=29_940, dim=3200, dv=1536, classes=1000, batch=8192, batch_txt=8192, n_val=4096,
                 desc="DINOv2 ViT-g 1536-d image + OpenLLaMA-3B 3200-d text features, adapter + shared head, throughput batch"),
    "cfg2": dict(n_img=16_000, n_txt=29_940, dim=512, classes=1000, batch=32, batch_txt=32, n_val=4000,
                 desc="ImageNet 16-shot CLIP ViT-B/16 512-d features + CUPL text, linear head, reference batch 32"),
    "cfg3_refB": dict(n_img=1_281_167, n_txt=29_940, dim=768, classes=1000, batch=32, batch_txt=32, n_val=4096,
                      desc="cfg3 banks at the reference batch of 32"),
}
ALPHA, LR, WD, LOGIT = 0.5, 1e-3, 0.01, 4.60517


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region, through NVML inside this process.

    (The first version spawned `nvidia-smi -lms` right before the timed region; its start-up - NVML/driver
    initialisation of a second process - stalled this process's CUDA calls for tens of milliseconds at random
    and the 50-step region is only ~10 ms long: values swung between 40 M and 116 M samples/s.)  NVML is
    initialised before the warm-up; a thread then polls every ``period`` seconds while ``active``."""

    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, index=0, period=0.004):
        self.index, self.period, self.rows, self.active, self.thread, self.h = index, period, [], False, None, None
        self.stop_flag = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self._sample()  # first query pays NVML's lazy set-up
            self.rows.clear()
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception as e:  # no NVML: report that instead of a number
            self.err = f"NVML unavailable: {e}"
            self.h = None

    @staticmethod
    def _physical_index(index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[index])
            except Exception:
                pass
        return index

    def _sample(self):
        nv = self.nv
        sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        self.rows.append((sm, mask))

    def _loop(self):
        while not self.stop_flag:
            if self.active:
                try:
                    self._sample()
                except Exception:
                    pass
            time.sleep(self.period)

    def start(self):
        self.rows.clear()
        self.active = True

    def stop(self):
        self.active = False
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [getattr(self, "err", "NVML unavailable")]}
        if not self.rows:  # region shorter than one period: one sample right at its end (still under load)
            try:
                self._sample()
            except Exception:
                pass
        sm = sorted(r[0] for r in self.rows)
        mask = 0
        for r in self.rows:
            mask |= r[1]
        reasons = [nm for nm, attr in self.REASONS if mask & getattr(self.nv, attr, 0)]
        return {"sm_mhz": float(sm[len(sm) // 2]) if sm else None, "sm_max_mhz": float(self.max_sm), "reasons": reasons,
                "samples": len(sm), "source": "NVML in-process, polled during the timed region"}

    def close(self):
        self.stop_flag = True


# -----------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference step on the host cores
# -----------------------------------------------------------------------------------------------

def cpu_reference_run(wl, steps, warmup, bank_rows=65536, budget_s=None, device="cpu"):
    """Times the reference's step algorithm (oracle port: per-sample fetch + collate, F.linear,
    F.cross_entropy, two autograd.grad sweeps + backward, AdamW - finetune.py:163-195) on all host
    threads.  The image bank is a seeded sample of ``bank_rows`` rows of the workload's shape.
    ``device="cuda"``: the same port as eager PyTorch on one GPU - the banks stay on the host like the reference's
    datasets, each batch is collated there and copied over, the step's torch ops run on the device."""
    from oracle import uml_oracle as O

    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    g = torch.Generator().manual_seed(1)
    D, C, B, BT = wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    n_img = min(wl["n_img"], bank_rows)
    xi = torch.randn(n_img, D, generator=g)
    yi = torch.randint(0, C, (n_img,), generator=g)
    xt = torch.randn(wl["n_txt"], D, generator=g)
    yt = torch.arange(wl["n_txt"]) % C
    st = O.HeadState(head=O.zero_shot_weights(xt, yt, C).to(device), img_scale=math.exp(LOGIT), txt_scale=math.exp(LOGIT))
    opt = O.OracleOptimizer(st.param_dict(), "adamw", LR, WD)
    on_gpu = torch.device(device).type == "cuda"
    gpu_ms = [0.0]
    il, tl = O.OracleLoader(n_img, B), O.OracleLoader(wl["n_txt"], BT)
    torch.manual_seed(2)
    il.iter(); tl.iter()

    def one(i):
        ii, it = O.fetch_next_indices(il), O.fetch_next_indices(tl)
        # default_collate over a map-style dataset: one row at a time, then stack
        xb = torch.stack([xi[int(j)] for j in ii]); yb = torch.stack([yi[int(j)] for j in ii])
        tb = torch.stack([xt[int(j)] for j in it]); ub = torch.stack([yt[int(j)] for j in it])
        if on_gpu:
            xb, yb, tb, ub = (t.to(device, non_blocking=True) for t in (xb, yb, tb, ub))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        _, grads = O.uml_step_grads_autograd(st, xb, yb, tb, ub, ALPHA)
        opt.step(grads, O.lr_at(i, LR, "cosine", 50, 12800))
        if on_gpu:
            e1.record()
            torch.cuda.synchronize()  # the reference reads the losses every step (finetune.py:197-206)
            gpu_ms[0] += e0.elapsed_time(e1)
        return ii.numel() + it.numel()

    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    rows = 0
    done = 0
    for i in range(steps):
        rows += one(warmup + i)
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    out = dict(value=rows / dt, ms_per_step=1e3 * dt / done, steps=done, cores=cores,
               sample=f"{done} steps of {B} image + {BT} text rows on a {n_img}-row sample of the image bank, {cores} threads")
    if on_gpu:  # the torch ops alone (batch already on the device), without the host-side collate
        out["device_ms_per_step"] = gpu_ms[0] / done
        out["device_only_value"] = rows / (gpu_ms[0] * 1e-3)
    return out


def reference_train_run(wl, steps, warmup, budget_s=150.0):
    """Times the UNMODIFIED reference: its own ``finetune.train`` (vision_language/finetune.py:120-288) on the host
    cores, called as shipped through oracle/ref_harness.py (stub modules for the absent timm / ftfy imports only; source
    from /root/reference or its verbatim copy oracle/_ref, see oracle/build_ref.py).  Full-size synthetic banks of the
    workload's shape as map-style datasets, the reference's DataLoader (default collate, num_workers=0 so that the
    timing is the training thread's), its UMLClip head initialised with its get_zero_shot_weights, its AdamW and
    scheduler.  The timed region is iterations warmup .. warmup+steps (timestamps taken in scheduler.step, the last
    call of an iteration); a wall-clock budget cuts the run short and the number of timed steps is reported."""
    from oracle import ref_harness as rh
    from torch.utils.data import DataLoader

    ns = rh.load_vision_language()
    torch.set_num_threads(os.cpu_count() or 1)
    cores = torch.get_num_threads()
    g = torch.Generator().manual_seed(1)
    D, C, B, BT = wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    n_img = wl["n_img"]
    xi = torch.randn(n_img, D, generator=g)
    yi = torch.randint(0, C, (n_img,), generator=g)
    xt = torch.randn(wl["n_txt"], D, generator=g)
    yt = torch.arange(wl["n_txt"]) % C
    xv, yv = torch.randn(512, D, generator=g), torch.randint(0, C, (512,), generator=g)
    tds = ns.ds_utils.TextTensorDataset(xt, yt, torch.zeros(wl["n_txt"], dtype=torch.int64))
    model = rh.build_reference_model("clip", D, D, C, logit=LOGIT)
    model.head.weight.data = ns.head.get_zero_shot_weights(tds, C, D, device="cpu")
    opt = ns.optim.build_optimizer(model.parameters(), "adamw", LR, WD)
    sch = ns.scheduler.build_lr_scheduler(opt, "cosine", 50, 12800, warmup_type="linear", warmup_lr=1e-5)
    il = DataLoader(rh.make_image_rows_dataset(xi, yi), batch_size=B, shuffle=True, drop_last=False, num_workers=0)
    tl = DataLoader(tds, batch_size=BT, shuffle=True, drop_last=False, num_workers=0)
    vl = DataLoader(rh.make_image_rows_dataset(xv, yv), batch_size=512, shuffle=False)

    class _Budget(Exception):
        pass

    stamps = []
    t_start = time.perf_counter()
    orig_step = sch.step

    def stamped(*a, **k):
        r = orig_step(*a, **k)
        stamps.append(time.perf_counter())
        if len(stamps) > warmup + 1 and stamps[-1] - t_start > budget_s:
            raise _Budget()
        return r

    sch.step = stamped
    torch.manual_seed(2)
    import contextlib
    import io
    try:
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            ns.finetune.train(model, il, tl, vl, None, opt, sch, device="cpu", max_iters=warmup + steps, alpha=ALPHA,
                              eval_freq=10 ** 9, patience=5, capture_features_during_training=False, logger=None)
    except _Budget:
        pass
    done = len(stamps) - warmup
    if done < 1:
        raise RuntimeError("reference train(): no timed iteration finished inside the budget")
    t0 = stamps[warmup - 1] if warmup > 0 else t_start
    dt = stamps[-1] - t0
    return dict(value=done * (B + BT) / dt, ms_per_step=1e3 * dt / done, steps=done, cores=cores, kind="reference",
                sample=f"{done} iterations of the reference's finetune.train() at {B} image + {BT} text rows per step on the full "
                       f"{n_img}-row image bank, {cores} threads, DataLoader num_workers=0")


# -----------------------------------------------------------------------------------------------
# our arm
# -----------------------------------------------------------------------------------------------

def build_banks(wl, dev, rank=0, world=1):
    """Seeded synthetic banks of the workload's shapes.  world > 1: this rank's row shard of the image and text
    banks (per-rank sampler, uml_b200.engine.datasets.shard_bank); the validation bank stays whole."""
    from uml_b200.engine.datasets.utils import FeatureBank, shard_bank

    g = torch.Generator(device=dev).manual_seed(1)
    D, C = wl["dim"], wl["classes"]
    img = torch.randn(wl["n_img"], wl.get("dv", D), device=dev, generator=g)
    img_y = torch.randint(0, C, (wl["n_img"],), device=dev, generator=g)
    txt = torch.randn(wl["n_txt"], D, device=dev, generator=g)
    txt_y = (torch.arange(wl["n_txt"], device=dev) % C)
    val = torch.randn(wl["n_val"], wl.get("dv", D), device=dev, generator=g)
    val_y = torch.randint(0, C, (wl["n_val"],), device=dev, generator=g)
    if world > 1:
        ib, tb = shard_bank(img, img_y, rank, world, dev), shard_bank(txt, txt_y, rank, world, dev)
        del img, txt
        torch.cuda.empty_cache()
        return ib, tb, FeatureBank(val, val_y, dev), FeatureBank(txt_full_for_init(wl, dev), (torch.arange(wl["n_txt"], device=dev) % C), dev)
    tb = FeatureBank(txt, txt_y, dev)
    return FeatureBank(img, img_y, dev), tb, FeatureBank(val, val_y, dev), tb


def txt_full_for_init(wl, dev):
    """The whole text bank again (same seed stream as build_banks) - the zero-shot initialisation uses every row."""
    g = torch.Generator(device=dev).manual_seed(1)
    torch.randn(wl["n_img"], wl.get("dv", wl["dim"]), device=dev, generator=g)
    torch.randint(0, wl["classes"], (wl["n_img"],), device=dev, generator=g)
    return torch.randn(wl["n_txt"], wl["dim"], device=dev, generator=g)


def make_model(wl, dev, txt_bank):
    from uml_b200.engine.models.head import UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler

    torch.manual_seed(1)
    if wl.get("dv"):  # adapter variant (reference UML with img_proj, head.py:63-84), preset "linear": learnable temperatures
        from uml_b200.engine.models.head import UML
        model = UML(f"synthetic:{wl['dv']}", wl["dim"], wl["classes"], learnable_temp=True)
        model.to(dev)
    else:
        model = UMLClip(f"synthetic:{wl['dim']}", wl["classes"], logit_scale_init=LOGIT)
        model.to(dev)
        model.zero_shot_init(txt_bank)
        model.to(dev)
    opt = build_optimizer(model.parameters(), "adamw", LR, WD)
    sch = build_lr_scheduler(opt, "cosine", 50, 12800, warmup_type="linear", warmup_lr=1e-5)
    return model, opt, sch


DUMP_MAX_ELEMS = 1 << 22  # 16 MB of float32 per array; with at most two such arrays (img_proj, head) a dump stays < 64 MB


def dump_outputs(out_dir, model, stats):
    """--dump-outputs: what the timed steps hand to their caller after the last one - the model's parameters (float32)
    and that step's loss / accuracy record (float64 scalars) - as out_dir/<name>.npy.  An array of more than
    DUMP_MAX_ELEMS elements is stored as the same seeded sample of its flattened elements in every run."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {name: p.detach().float().cpu().numpy() for name, p in model.named_parameters()}
    arrays.update({k: np.float64(v) for k, v in stats.items()})
    for name, a in arrays.items():
        if a.size > DUMP_MAX_ELEMS:
            keep = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            a = a.reshape(-1)[keep]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _stage(msg):
    if os.environ.get("UML_BENCH_VERBOSE"):
        print(f"[bench] {msg}", file=sys.stderr, flush=True)


def run_ours(args, wl, rank, world, dev):
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader, mark_ready
    from uml_b200.engine.trainer import StepEngine

    dist = torch.distributed if world > 1 else None
    img_bank, txt_bank, val_bank, init_bank = build_banks(wl, dev, rank, world)
    B, BT = wl["batch"], wl["batch_txt"]  # rows per GPU and step (weak scaling: fixed as GPUs are added)
    shard = (rank, world) if world > 1 else None  # world > 1: per-rank sampler over this rank's bank shard
    K, W = args.steps, args.warmup

    # ---------------- device-resident arm: CUDA events around K steps ----------------------------
    model, opt, sch = make_model(wl, dev, init_bank)
    engine = StepEngine(model, opt, dev, B, BT, log_slots=64, precision=args.precision, world_size=world)
    # per-rank shards (world > 1) drop their ragged last batch: a 3742-row text shard would otherwise end every epoch
    # with a 158-row batch and the per-GPU work of a step would no longer be fixed (weak scaling)
    # (a shard shorter than the batch - cfg4's 8192-row text batch on 8 GPUs - is one ragged batch per epoch instead)
    il = BankLoader(img_bank, B, shuffle=True, upload="epoch", shard_of=shard, drop_last=world > 1 and len(img_bank) >= B)
    tl = BankLoader(txt_bank, BT, shuffle=True, upload="epoch", shard_of=shard, drop_last=world > 1 and len(txt_bank) >= BT)
    torch.manual_seed(2)
    ii, ti = iter(il), iter(tl)

    slow = [(0.0, -1), (0.0, -1)]  # slowest single fetch of the image / text loader and the step it happened at
    host_split = [0.0, 0.0]  # seconds in the loaders / in engine.run (host-side enqueue cost, reported on stderr)
    CHUNK = 16  # iterations enqueued per library call (uml_linear_run), as finetune.train does

    staged = []  # (img batch, txt batch, lr) of upcoming steps whose index batches already sit in HBM

    def draw(i):
        """Sampler + upload of step i's index batches (host work: part of the end-to-end arm, not of `value`)."""
        nonlocal ii, ti
        ta = time.perf_counter()
        img, ii = ft.fetch_next(il, ii)
        tb = time.perf_counter()
        txt, ti = ft.fetch_next(tl, ti)
        tc = time.perf_counter()
        if tb - ta > slow[0][0]:
            slow[0] = (tb - ta, i)
        if tc - tb > slow[1][0]:
            slow[1] = (tc - tb, i)
        lr = sch.get_last_lr()[0]
        sch.step()
        return img, txt, lr

    def stage(i0, n):
        """Draw steps i0 .. i0+n-1 ahead of time; the index tensors are cloned because the loaders recycle their
        device permutation buffers every other epoch."""
        for j in range(n):
            img, txt, lr = draw(i0 + j)
            img.idx, txt.idx = img.idx.clone(), txt.idx.clone()
            mark_ready(img)   # the clones are what the steps read: vouch for them (IndexBatch.ready), as the loaders do
            mark_ready(txt)   # for their uploads
            staged.append((img, txt, lr))

    def step(i, n=1):
        """Enqueue iterations i .. i+n-1; returns the number of (global) rows they consume."""
        batches, lrs, rows_ = [], [], 0
        t0 = time.perf_counter()
        for j in range(n):
            img, txt, lr = staged.pop(0) if staged else draw(i + j)
            batches.append((img, txt))
            lrs.append(lr)
            rows_ += (img.global_n or img.n) + (txt.global_n or txt.n)
        t1 = time.perf_counter()
        engine.run(batches, ALPHA, lrs, slot0=i)
        host_split[0] += t1 - t0
        host_split[1] += time.perf_counter() - t1
        return rows_

    sampler = ClockSampler(dev.index or 0) if rank == 0 else None  # NVML set-up happens here, before the warm-up
    i = 0
    while i < W:  # warm-up in chunks of two: the chunked launcher (side stream, events, second operand buffer) is set up
        n = min(2, W - i)
        step(i, n)
        i += n
    bf16_path = engine._use_bf16(B + BT)
    dominant = "head_fwd_ce_bf16" if bf16_path else "head_bwd_dw_f32"
    engine.prepare_profile(K, only=[dominant])  # the roofline kernel is timed live inside the timed region
    # `value` is the device-resident number: the K timed steps' INPUTS - their index batches - are in HBM before the
    # clock starts (the rows themselves are gathered from the banks inside the timed region).  Drawing the
    # permutations and uploading the indices is host work that the end-to-end arm times.
    stage(W, K)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    if rank == 0:
        sampler.start()
    n0 = _lib.LAUNCH_COUNT[0]
    host_split[0] = host_split[1] = 0.0
    slow[0] = slow[1] = (0.0, -1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rows = 0
    prof = None
    if os.environ.get("UML_BENCH_PROFILE"):
        import cProfile
        prof = cProfile.Profile()
        prof.enable()
    t_host0 = time.perf_counter()
    e0.record()
    i, ramp = 0, 2
    while i < K:
        # chunk sizes ramp up 2, 4, 8, ...: the queue is empty when the clock starts, and while the host prepares a
        # chunk's batches the GPU only has the previous chunk to work on
        n = min(CHUNK, ramp, K - i)
        ramp *= 2
        rows += step(W + i, n)
        i += n
    e1.record()
    if prof is not None:
        import pstats
        prof.disable()
        pstats.Stats(prof, stream=sys.stderr).sort_stats("tottime").print_stats(14)
    host_ms = (time.perf_counter() - t_host0) * 1e3 / K  # enqueue cost per step (the loop never syncs)
    if rank == 0:
        print(f"host per step: loaders {host_split[0] / K * 1e3:.4f} ms, engine.run {host_split[1] / K * 1e3:.4f} ms; slowest fetch: "
              f"image {slow[0][0] * 1e3:.2f} ms at step {slow[0][1]}, text {slow[1][0] * 1e3:.2f} ms at step {slow[1][1]}; "
              f"cpus usable {len(os.sched_getaffinity(0))}", file=sys.stderr)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    launches = _lib.LAUNCH_COUNT[0] - n0
    ms = e0.elapsed_time(e1)
    if dist:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    _stage("timed region done")
    if os.environ.get("UML_BENCH_QUICK"):  # experiments: the device-resident figure only, no breakdown / end-to-end arm
        print(f"quick: {ms / K:.5f} ms/step, {rows * world / (ms * 1e-3):.4g} samples/s", flush=True)
        os._exit(0)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        sampler.close()
    ktimes = engine.kernel_times_ms()
    loss_tail = engine.read_log([W + K - 1])[0]
    if args.dump_outputs and rank == 0:  # before the breakdown steps below train the model further
        dump_outputs(args.dump_outputs, model, loss_tail)
    # per-kernel breakdown of the step from a few extra (untimed) steps with every kernel bracketed
    engine.prepare_profile(16)
    step(W + K, 16)
    torch.cuda.synchronize()
    breakdown = engine.kernel_times_ms()
    breakdown.update(engine.step_timeline_ms())
    del engine
    _stage("breakdown done")

    # ---------------- end-to-end arm: public train() call, per-step H2D indices + D2H loss ---------
    def e2e_run(warm, iters):
        """ONE public train() call of warm + iters iterations; the timed region is iterations warm.. (wall clock,
        stream-synchronised on both sides): per step it holds the H2D copy of the step's index batches from pinned
        memory, the step, and the D2H copy of its loss record, read on the host before the clock stops."""
        m2, o2, s2 = make_model(wl, dev, init_bank)
        m2.precision = args.precision
        il2 = BankLoader(img_bank, B, shuffle=True, upload="step", shard_of=shard, drop_last=world > 1 and len(img_bank) >= B)
        tl2 = BankLoader(txt_bank, BT, shuffle=True, upload="step", shard_of=shard, drop_last=world > 1 and len(txt_bank) >= BT)
        vl2 = BankLoader(val_bank, 512, shuffle=False)
        torch.manual_seed(2)
        tr = {"timing": {"warmup": warm}, "indices": False}
        if dist:
            dist.barrier()
        _stage("e2e train() starts")
        ft.train(m2, il2, tl2, vl2, None, o2, s2, device=dev, max_iters=warm + iters, alpha=ALPHA, eval_freq=10 ** 9,
                 patience=5, stats_to_host="step", trace=tr)
        assert tr["timing"]["iters"] == iters
        return tr["timing"]["seconds"], tr["timing"]["rows"]

    import contextlib
    import io
    # The timed region of one call is only ~10 ms long, so a single host hiccup (page faults of a fresh pinned ring,
    # a scheduler preemption) can halve it: the call is repeated and the MEDIAN reported, all values kept.
    e2e_all = []
    with contextlib.redirect_stdout(io.StringIO()):
        for _ in range(3):
            dt_i, e2e_rows = e2e_run(max(W, 3), K)
            if dist:
                t = torch.tensor([dt_i], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt_i = float(t.item())
            e2e_all.append(dt_i)
    dt = sorted(e2e_all)[1]
    _stage("e2e done")
    e2e_value = e2e_rows / dt  # global rows (every rank walks the same global batches) over the slowest rank's time
    return dict(ms=ms, rows=rows, launches=launches, clocks=clocks, ktimes=ktimes, e2e_value=e2e_value,
                host_ms=host_ms, breakdown=breakdown, e2e_all=[e2e_rows / x for x in e2e_all],
                h2d=(B + BT) * 8, d2h=2 * 4 * 4, loss_tail=loss_tail)


def run_gaussian(args):
    """--workload cfg1: the Gaussian_experiment step (train.yaml: dim_obs 50, dim_common 128, dim_latent 10, batch 512 per
    modality, Adam 1e-3, mode xy) - a latency-bound two-launch step.  value/e2e: the public train_model_steps call
    (sampler on the host, index batches uploaded per epoch, losses read back once); cpu_baseline: the oracle port."""
    import types
    from oracle import uml_oracle as O
    from uml_b200 import _lib, gaussian as G

    dev = torch.device("cuda", 0)
    kw = dict(seed=42, num_samples=10000, dim_c=10, dim_x=5, dim_y=5, dim_obs=50, noise_std=0.09, attenuate_x=True,
              attenuation=0.05, shared_latent_distribution_type="gaussian")
    d = G.generate_data(kw)
    dx, dy = d["x"][:5000], d["y"][:5000]
    K, W, B = args.steps, args.warmup, 512
    torch.manual_seed(0)
    model = G.SharedAutoencoder(50, 128, 10, device=dev)
    g = torch.Generator()
    g.manual_seed(42)
    loader = G.unpaired_loader(G.UnpairedDataset(dx, dy, dev), B, generator=g)
    opt = G.Adam(model, lr=1e-3)
    a = types.SimpleNamespace(mode="xy", alpha_x=1.0, alpha_y=1.0)
    G.train_model_steps(model, loader, opt, W, args=a)
    torch.cuda.synchronize()
    n0 = _lib.LAUNCH_COUNT[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    hist = G.train_model_steps(model, loader, opt, K, args=a)  # ends with the D2H read of the K loss records
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = e0.elapsed_time(e1)
    p = {k: v.cpu() for k, v in model.state_dict().items()}
    t1 = time.perf_counter()
    O.gaussian_train(p, dx, dy, num_steps=200, batch_size=B, lr=1e-3, mode="xy")
    cpu = 200 * 2 * B / (time.perf_counter() - t1)
    # The reference's loop also evaluates linear CKA and mutual 10-NN on the 2000-row validation embeddings after EVERY
    # step (main.py:14-27 EVAL_EVERY = 1, :67-84) - diagnostics this implementation does not run.  Their CPU cost at
    # those shapes (n x n kernel matrices), for context next to the bare step:
    probes = None
    try:
        from oracle import metrics_oracle as MO
        ga = torch.Generator().manual_seed(0)
        ea, eb = torch.randn(2000, 10, generator=ga), torch.randn(2000, 10, generator=ga)
        MO.cka_linear(ea, eb)
        t2 = time.perf_counter()
        for _ in range(3):
            MO.cka_linear(ea, eb)
            MO.mutual_knn(ea, eb, 10)
        probes = (time.perf_counter() - t2) / 3
    except Exception as e:  # context only
        print(f"probe timing failed: {e}", file=sys.stderr)
    line = {"metric": "UML train samples/sec (img+text)", "value": K * 2 * B / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg1: Gaussian_experiment linear UML (train.yaml), x+y rows", "dim_obs": 50, "dim_common": 128,
                       "dim_latent": 10, "batch_per_modality": B, "mode": "xy", "l2_policy": "working set (29 k parameters, 2 MB of data) lives in L2"},
            "e2e": {"value": K * 2 * B / wall, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 8,
                    "note": "index permutation uploaded once per epoch (9 steps)"},
            "gpu_launches": _lib.LAUNCH_COUNT[0] - n0, "final_losses": {"loss_x": hist["loss_x"][-1], "loss_y": hist["loss_y"][-1]},
            "roofline": {"bound": "latency", "kernel": "gauss_fwd_bwd_kernel + gauss_update_kernel", "achieved": None, "peak": None,
                         "unit": "us/step", "frac": None, "traffic": None},
            "cpu_baseline": {"value": cpu, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "200 steps of the oracle port (fp32 torch ops on the host)",
                             "reference_probes_s_per_step": probes,
                             "value_with_reference_probes": (2 * B / (2 * B / cpu + probes)) if probes else None}}
    print(json.dumps(line))


def run_eval(args):
    """--workload eval: the evaluation sweep (a-11 / K7; reference finetune.py:291-315 `validate`) over test banks of the
    named shapes, through the public ``finetune.validate`` call.  Unit = bank rows per second.  Three banks:
      imagenet : 50 000 x 768, C = 1000  - the logits GEMM dominates -> tensor roofline (bf16 path)
      sun397   : 19 850 x 512, C = 397   | the bank read dominates on the tensor-core path -> HBM roofline
      food101  : 25 250 x 512, C = 101   |
    each on the bf16 tensor-core path (what a model trained on that path uses) and on the exact fp32 path (what a run at the
    reference's batch sizes uses).  ``value``: imagenet / bf16, device time of the K7 launches (CUDA events, L2 flushed
    between repetitions); ``e2e``: wall clock of validate() calls including the read-back of (loss, hits)."""
    from oracle import uml_oracle as O
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader, FeatureBank
    from uml_b200.engine.models.head import UMLClip

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    peaks = measured_peaks()
    K, Wm = args.steps, max(args.warmup, 3)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    g = torch.Generator().manual_seed(3)
    cases, sampler = [], ClockSampler(0)
    shapes = (("imagenet", 50_000, 768, 1000), ("sun397", 19_850, 512, 397), ("food101", 25_250, 512, 101))
    first = True
    for name, n, D, C in shapes:
        x = torch.randn(n, D, generator=g)
        x = x / x.norm(dim=1, keepdim=True)
        y = torch.randint(0, C, (n,), generator=g)
        bank = FeatureBank(x, y, dev)
        model = UMLClip(f"synthetic:{D}", C, logit_scale_init=LOGIT).to(dev)
        w = torch.randn(C, D, generator=g)
        model.head.weight.data.copy_((w / w.norm(dim=1, keepdim=True)).to(dev))
        loader = BankLoader(bank, 512, shuffle=False)
        for prec in ("bf16", "fp32"):
            model.precision = prec
            for _ in range(Wm):
                ft.validate(model, loader, device=dev)
            n0 = _lib.LAUNCH_COUNT[0]
            if first:
                sampler.start()
            ts = []
            for _ in range(K):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ft.validate_enqueue(model, loader)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            launches = _lib.LAUNCH_COUNT[0] - n0
            clocks = sampler.stop() if first else None
            first = False
            t0 = time.perf_counter()
            for _ in range(K):
                loss, acc = ft.validate(model, loader, device=dev)
            wall = (time.perf_counter() - t0) / K
            ms = sorted(ts)[len(ts) // 2]
            flops, bytes_ = 2.0 * n * D * C, n * (D * (2 if prec == "bf16" else 4) + 8)
            if prec == "bf16" and C >= 512:
                roof = {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": peaks["tf_burst"], "unit": "TFLOP/s"}
            elif prec == "bf16":
                roof = {"bound": "hbm", "achieved": bytes_ / (ms * 1e-3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s"}
            else:  # exact path: fp32 FMA pipe (148 SMs x 128 lanes x 2 flop x 1.965 GHz = 74.4 TFLOP/s nominal), not a measured peak
                roof = {"bound": "fp32-fma (nominal)", "achieved": flops / (ms * 1e-3) / 1e12, "peak": 74.4, "unit": "TFLOP/s"}
            roof["frac"] = roof["achieved"] / roof["peak"]
            cases.append({"bank": name, "rows": n, "dim": D, "classes": C, "path": prec, "device_ms": ms, "rows_per_s": n / (ms * 1e-3),
                          "e2e_ms": wall * 1e3, "e2e_rows_per_s": n / wall, "val_loss": loss, "val_acc": acc, "roofline": roof,
                          "launches_per_call": launches / K, "clocks": clocks})
        del bank, model
    # CPU port on a sample of the imagenet bank
    n_s = 4096
    xs = torch.randn(n_s, 768, generator=g)
    ys = torch.randint(0, 1000, (n_s,), generator=g)
    st = O.HeadState(head=torch.randn(1000, 768, generator=g), img_scale=math.exp(LOGIT), txt_scale=math.exp(LOGIT))
    torch.set_num_threads(os.cpu_count() or 1)
    O.validate(st, xs, ys, 512)
    t0, reps = time.perf_counter(), 0
    while time.perf_counter() - t0 < min(args.cpu_seconds, 10.0):
        O.validate(st, xs, ys, 512)
        reps += 1
    cpu = reps * n_s / (time.perf_counter() - t0)
    head = cases[0]
    line = {"metric": "UML eval rows/sec (validate over a test bank)", "value": head["rows_per_s"], "unit": "rows/s", "n_gpus": 1,
            "steps": K, "warmup": Wm, "ms_per_step": head["device_ms"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "eval: validate() over test banks - imagenet 50000x768 C=1000 (headline, bf16 path), sun397 "
                                   "19850x512 C=397, food101 25250x512 C=101; each on the bf16 tensor-core and the exact fp32 path",
                       "l2_policy": "256 MB written between repetitions (the 77 MB bf16 shadow of the largest bank would otherwise sit in L2)"},
            "clocks": head["clocks"], "e2e": {"value": head["e2e_rows_per_s"], "unit": "rows/s", "h2d_bytes_per_step": 0,
                                              "d2h_bytes_per_step": 8, "note": "the bank is resident; per call the host reads (loss, hits)"},
            "gpu_launches": int(sum(c["launches_per_call"] for c in cases) * K),
            "roofline": dict(head["roofline"], kernel="head_fwd_ce_x (evaluation mode) + eval_reduce", traffic=None),
            "cpu_baseline": {"value": cpu, "unit": "rows/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"oracle validate() on a {n_s}-row sample of the imagenet bank shape, repeated for 10 s"},
            "eval_cases": [{k: v for k, v in c.items() if k != "clocks"} for c in cases]}
    sampler.close()
    print(json.dumps(line))


def run_sweep(args):
    """--workload cfg2_sweep: the reference's real few-shot workload - the hyper-parameter sweep of preset `clip_linear`
    (lr x weight decay, engine/optimizer/default.py:17-31) times its alpha sweep over the SAME cfg2 banks - with
    --heads combinations trained in lock step (finetune.train_group / uml_sweep_run: two launches per step of all
    heads).  value: device-resident (every head's epoch permutation in HBM before the clock starts); e2e: ONE public
    train_group() call; `sequential`: the same banks through the single-head engine (finetune.train), which is what
    the sweep costs one combination at a time."""
    import contextlib
    import io
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader
    from uml_b200.engine.models.head import UMLClip, get_zero_shot_weights
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler
    from uml_b200.engine.sweep import HeadGroup

    wl = WORKLOADS["cfg2"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peaks = measured_peaks()
    img_bank, txt_bank, val_bank, _ = build_banks(wl, dev)
    D, C, B, BT = wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    H, K, W = args.heads, args.steps, args.warmup
    grid = [(lr, wd, al) for al in (0.2, 0.5, 0.7, 1.0, 1.5) for lr in (1e-3, 1e-4) for wd in (0.0, 0.01, 0.001)]
    grid = [grid[k % len(grid)] for k in range(H)]
    W0 = get_zero_shot_weights(txt_bank, C, D)

    def make_heads(n, upload="epoch"):
        ms, os_, ss, il, tl, vl = [], [], [], [], [], []
        with contextlib.redirect_stdout(io.StringIO()):
            for k in range(n):
                lr, wd, _ = grid[k]
                m = UMLClip(f"synthetic:{D}", C, logit_scale_init=LOGIT)
                m.precision = "fp32"
                m.load_state_dict({"head.weight": W0.clone()})
                m.to(dev)
                o = build_optimizer(m.parameters(), "adamw", lr, wd)
                rng = torch.Generator().manual_seed(100 + k)
                ms.append(m); os_.append(o)
                ss.append(build_lr_scheduler(o, "cosine", 50, 12800, warmup_type="linear", warmup_lr=1e-5))
                il.append(BankLoader(img_bank, B, shuffle=True, upload=upload, rng=rng))
                tl.append(BankLoader(txt_bank, BT, shuffle=True, upload=upload, rng=rng))
                vl.append(BankLoader(val_bank, 32, shuffle=False, rng=rng))
        return ms, os_, ss, il, tl, vl

    alphas = [g[2] for g in grid]
    # ---------------- device-resident arm ------------------------------------------------------------------------
    ms_, os_, ss, il, tl, vl = make_heads(H)
    group = HeadGroup(ms_, os_, img_bank, txt_bank, B, BT, dev, log_slots=W + K + 1)
    iti, itt = [iter(l) for l in il], [iter(l) for l in tl]
    assert W + K <= min(len(il[0]), len(tl[0])), "keep warm-up + steps inside one epoch of the few-shot banks"

    def chunk(n, i0):
        pi = [it.take_run(n) for it in iti]
        pt = [it.take_run(n) for it in itt]
        lrs = [[s.lr_at(i0 + j, s.base_lrs[0]) for s in ss] for j in range(n)]
        return ([p[0] for p in pi], [p[0] for p in pt], pi[0][1], pt[0][1], [(B, BT)] * n, lrs)

    a = chunk(W, 0)
    group.run(*a, alphas, [True] * H, slot0=0)
    a = chunk(K, W)  # the timed steps' permutations are in HBM (uploaded when the epoch was drawn)
    group.time_last_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    n0 = _lib.LAUNCH_COUNT[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    i = 0
    while i < K:  # one library call per 16 steps, like train_group's chunks
        n = min(16, K - i)
        group.run(a[0], a[1], a[2] + i * B, a[3] + i * BT, a[4][i:i + n], a[5][i:i + n], alphas, [True] * H, slot0=W + i)
        i += n
    e1.record()
    host_ms = (time.perf_counter() - t0) * 1e3 / K
    torch.cuda.synchronize()
    clocks = sampler.stop()
    sampler.close()
    ms = e0.elapsed_time(e1)
    launches = _lib.LAUNCH_COUNT[0] - n0
    ktimes = group.kernel_times_ms()
    tail = group.read_log([W + K - 1], True, True)
    rows = H * K * (B + BT)
    del group

    # ---------------- end-to-end arm: one public train_group() call ----------------------------------------------
    def e2e_group():
        ms2, os2, ss2, il2, tl2, vl2 = make_heads(H)
        trs = [None] * H  # per-step records are only materialised for heads that ask for them
        trs[0] = {"indices": False, "timing": {"warmup": max(W, 3)}}
        with contextlib.redirect_stdout(io.StringIO()):
            ft.train_group(ms2, il2, tl2, vl2, None, os2, ss2, device=dev, max_iters=max(W, 3) + K, alphas=alphas,
                           eval_freq=10 ** 9, patience=5, traces=trs)
        assert trs[0]["timing"]["iters"] == K
        return trs[0]["timing"]["seconds"]

    e2e_all = [e2e_group() for _ in range(3)]
    e2e_dt = sorted(e2e_all)[1]

    # ---------------- the same sweep one combination at a time (single-head engine) ------------------------------
    def sequential():
        ms2, os2, ss2, il2, tl2, vl2 = make_heads(1, upload="epoch")
        tr = {"timing": {"warmup": max(W, 3)}, "indices": False}
        with contextlib.redirect_stdout(io.StringIO()):
            ft.train(ms2[0], il2[0], tl2[0], vl2[0], None, os2[0], ss2[0], device=dev, max_iters=max(W, 3) + K,
                     alpha=alphas[0], eval_freq=10 ** 9, patience=5, trace=tr)
        return tr["timing"]["seconds"] / K
    seq = sorted(sequential() for _ in range(3))[1]

    kms = ktimes.get("sweep_dw_update", float("nan"))
    # algorithmic bytes of the dW + optimizer launch: W, m, v read and written once per head (24 B/parameter; the
    # gradient itself never reaches HBM) plus the step's G and feature rows read once
    bytes_ = H * (24.0 * C * D + 4.0 * (B + BT) * (C + D))
    roof = {"bound": "hbm", "kernel": "sweep_dw_update_tc_kernel", "achieved": bytes_ / (kms * 1e-3) / 1e9, "peak": peaks["hbm"],
            "unit": "GB/s",
            # dram__bytes_read.sum + dram__bytes_write.sum of this kernel per launch from the committed `ncu --set full` capture
            # (profiles/r02_sweep_tc.md: 200.3 MB + 126.2 MB at 30 heads of 1000 x 512; part of the writes is still in L2 when
            # the kernel ends), scaled by the parameters of the group
            "traffic": 3.266e8 * (H * C * D) / (30.0 * 1000 * 512), "traffic_unit": "bytes per launch",
            "peak_source": f"{peaks['src']} HBM copy",
            "algorithmic_bytes_per_launch": bytes_, "kernel_ms": {k: round(v, 5) for k, v in ktimes.items()}}
    roof["frac"] = roof["achieved"] / roof["peak"]
    line = {"metric": "UML train samples/sec (img+text)", "value": rows / (ms * 1e-3), "unit": "samples/s", "n_gpus": 1,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"cfg2_sweep: {wl['desc']}; {H} hyper-parameter combinations (lr x wd x alpha) in lock step",
                       "heads": H, "dim": D, "classes": C, "img_bank_rows": wl["n_img"], "txt_bank_rows": wl["n_txt"],
                       "image_rows_per_head_step": B, "text_rows_per_head_step": BT, "optimizer": "adamw",
                       "l2_policy": f"per step {H} x 6.1 MB of weights and optimizer state stream through HBM "
                                    f"({H * 6.1:.0f} MB{', larger than L2' if H * 6.1 > 126 else ', fits L2'})"},
            "clocks": clocks,
            "e2e": {"value": rows / e2e_dt, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": H * 2 * 16,
                    "note": "one train_group() call; permutations uploaded once per epoch; stats read back at the end",
                    "stat": "median of 3 calls", "all": [round(rows / x) for x in e2e_all]},
            "gpu_launches": launches, "host_enqueue_ms_per_step": host_ms, "roofline": roof,
            "sequential": {"ms_per_head_step": seq * 1e3, "samples_per_s": (B + BT) / seq,
                           "speedup_of_lock_step": (rows / e2e_dt) / ((B + BT) / seq),
                           "note": "finetune.train() of one combination on the same banks (single-head fp32 engine), end to end"},
            "final_losses": {"image_loss": tail["image_loss"][0][0], "text_loss": tail["text_loss"][0][0]}}
    try:
        r = cpu_reference_run(wl, 10 ** 6, 1, budget_s=args.cpu_seconds)
        line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    except Exception as e:
        line["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line))


def run_ratio(args):
    """--workload cfg5: BASELINE config 5, the text:image conversion-ratio sweep (configs/ratio_sweep_sun397.yaml) on
    ViT-B/16-shaped (512-d) few-shot banks: SUN397 (397 classes) and Food101 (101 classes), 4 image shots per class,
    text:image ratios 0 (image only), 1, 2, 4 and 7.5 (text_shot 0 / 4 / 8 / 16 / 30 of the 30 prompts per class, selected by
    ``TextTensorDataset(n_shots=...)`` like the reference, engine/datasets/utils.py:55-98), preset ``clip_linear``'s six
    lr x wd combinations per point, batch 32 per modality.  Every point is ONE public ``train_group()`` call (sweep-level
    batching); value = rows consumed by all heads of all points per second of those calls' timed regions (wall clock,
    stream-synchronised: sampler, permutation uploads and the statistics read-back included - the same number is the e2e
    figure, there is no separate device-resident arm)."""
    import contextlib
    import io
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader, FeatureBank, TextTensorDataset
    from uml_b200.engine.models.head import UMLClip, get_zero_shot_weights
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    peaks = measured_peaks()
    K, W = args.steps, max(args.warmup, 3)
    D, B, shots = 512, 32, 4
    grid = [(lr, wd) for lr in (1e-3, 1e-4) for wd in (0.0, 0.01, 0.001)]
    H = len(grid)
    g = torch.Generator().manual_seed(5)
    points, rows_total, secs_total, launches0 = [], 0, 0.0, _lib.LAUNCH_COUNT[0]
    sampler = ClockSampler(0)
    sampler.start()
    for name, C in (("sun397", 397), ("food101", 101)):
        xi = torch.randn(C * shots, D, generator=g)
        yi = torch.arange(C * shots) % C
        xt_all = torch.randn(C * 30, D, generator=g)
        yt_all = torch.arange(C * 30) % C
        xv, yv = torch.randn(C * 4, D, generator=g), torch.arange(C * 4) % C
        img_bank, val_bank = FeatureBank(xi, yi, dev), FeatureBank(xv, yv, dev)
        for text_shot in (0, 4, 8, 16, 30):
            with contextlib.redirect_stdout(io.StringIO()):
                torch.manual_seed(1)
                tds = TextTensorDataset(xt_all, yt_all, torch.zeros(C * 30, dtype=torch.int64), n_shots=max(text_shot, 1))
                txt_bank = FeatureBank.from_text_dataset(tds, dev)
                W0 = get_zero_shot_weights(txt_bank, C, D)
                ms_, os_, ss, il, tl, vl = [], [], [], [], [], []
                for k, (lr, wd) in enumerate(grid):
                    m = UMLClip(f"synthetic:{D}", C, logit_scale_init=LOGIT)
                    m.precision = "fp32"
                    m.load_state_dict({"head.weight": W0.clone()})
                    m.to(dev)
                    o = build_optimizer(m.parameters(), "adamw", lr, wd)
                    rng = torch.Generator().manual_seed(100 + k)
                    ms_.append(m); os_.append(o)
                    ss.append(build_lr_scheduler(o, "cosine", 50, 12800, warmup_type="linear", warmup_lr=1e-5))
                    il.append(BankLoader(img_bank, B, shuffle=True, rng=rng))
                    tl.append(BankLoader(txt_bank, B, shuffle=True, rng=rng) if text_shot else None)
                    vl.append(BankLoader(val_bank, 32, shuffle=False, rng=rng))
                trs = [None] * H
                trs[0] = {"indices": False, "timing": {"warmup": W}}
                ft.train_group(ms_, il, tl if text_shot else None, vl, None, os_, ss, device=dev, max_iters=W + K,
                               alphas=[1.0] * H, eval_freq=10 ** 9, patience=5, traces=trs)
            t = trs[0]["timing"]
            rows = H * t["iters"] * (B + (B if text_shot else 0))
            rows_total += rows
            secs_total += t["seconds"]
            points.append({"dataset": name, "classes": C, "train_shot": shots, "text_shot": text_shot, "ratio": text_shot / shots,
                           "text_bank_rows": len(txt_bank) if text_shot else 0, "heads": H, "ms_per_step_of_all_heads": t["seconds"] / t["iters"] * 1e3,
                           "samples_per_s": rows / t["seconds"]})
    clocks = sampler.stop()
    sampler.close()
    launches = _lib.LAUNCH_COUNT[0] - launches0
    value = rows_total / secs_total
    # whole-step algorithmic HBM bytes of a head-step: W, m, v read and written (24 B / parameter) + G and rows once
    bytes_total = sum(p["heads"] * K * (24.0 * p["classes"] * D + 4.0 * (B + (B if p["text_shot"] else 0)) * (p["classes"] + D)) for p in points)
    roof = {"bound": "hbm", "kernel": "whole step (2 launches per step of a group)", "achieved": bytes_total / secs_total / 1e9,
            "peak": peaks["hbm"], "unit": "GB/s", "traffic": None, "peak_source": f"{peaks['src']} HBM copy",
            "note": "six 0.2-0.8 MB heads per group: the whole working set sits in L2 and a step is launch-latency bound"}
    roof["frac"] = roof["achieved"] / roof["peak"]
    line = {"metric": "UML train samples/sec (img+text)", "value": value, "unit": "samples/s", "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": secs_total / (len(points) * K) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "cfg5: SUN397 / Food101 conversion-ratio sweep (text:image 0-7.5x) on ViT-B/16-shaped 512-d few-shot "
                                   "banks, preset clip_linear (6 combinations per point in lock step), batch 32 per modality",
                       "points": len(points), "heads_per_point": H, "l2_policy": "working set fits L2 (few-shot banks)"},
            "clocks": clocks,
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": H * 2 * 16,
                    "note": "value IS the end-to-end figure here: public train_group() calls, wall clock"},
            "gpu_launches": launches, "roofline": roof, "ratio_points": points}
    try:
        r = cpu_reference_run(dict(WORKLOADS["cfg2"], classes=397, n_img=397 * shots, n_txt=397 * 30), 10 ** 6, 1, budget_s=args.cpu_seconds)
        line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
                                "sample": r["sample"] + " (sun397 shapes, one combination)"}
    except Exception as e:
        line["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", type=str, default="cfg3", choices=sorted(WORKLOADS) + ["cfg1", "cfg2_sweep", "cfg5", "eval"])
    ap.add_argument("--heads", type=int, default=30, help="cfg2_sweep: hyper-parameter combinations trained in lock step (<= 32)")
    ap.add_argument("--ref-device", type=str, default="cpu", choices=["cpu", "cuda"],
                    help="--impl reference: 'cuda' times the same port as eager PyTorch on one GPU (collate on the host, "
                         "H2D, fp32 torch ops on the device) - the like-for-like GPU baseline of SURVEY 8d")
    ap.add_argument("--precision", type=str, default="auto", choices=["auto", "fp32", "bf16"])
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the trained parameters and the last timed step's losses and "
                         "accuracies as DIR/<name>.npy (the inputs are seeded: two builds can be compared file by file)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload in ("cfg1", "cfg2_sweep", "cfg5", "eval")):
        ap.error("--dump-outputs covers the training step of our implementation: --impl ours with workload "
                 + ", ".join(sorted(WORKLOADS)))
    args.warmup = max(args.warmup, 3)
    if args.workload == "eval":
        if args.impl == "reference":
            raise SystemExit("bench.py --workload eval runs the GPU arm only (its line carries the CPU port as cpu_baseline)")
        return run_eval(args)
    if args.workload == "cfg5":
        if args.impl == "reference" or not torch.cuda.is_available():
            raise SystemExit("bench.py --workload cfg5 runs the GPU arm only (its line carries the CPU port as cpu_baseline)")
        return run_ratio(args)
    if args.workload == "cfg1":
        if args.impl == "reference" or not torch.cuda.is_available():
            raise SystemExit("bench.py --workload cfg1 runs the GPU arm only (its line carries the CPU port as cpu_baseline)")
        return run_gaussian(args)
    if args.workload == "cfg2_sweep":
        if args.impl == "reference" or not torch.cuda.is_available():
            raise SystemExit("bench.py --workload cfg2_sweep runs the GPU arm only (its line carries the CPU port as cpu_baseline)")
        return run_sweep(args)
    wl = WORKLOADS[args.workload]
    if os.environ.get("UML_BENCH_BATCH"):  # experiments: image rows per GPU and step
        wl = dict(wl, batch=int(os.environ["UML_BENCH_BATCH"]))
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    peaks = measured_peaks()
    D, C, B, BT = wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    config = {"workload": f"{args.workload}: {wl['desc']}", "dim": D, "classes": C, "img_bank_rows": wl["n_img"],
              "txt_bank_rows": wl["n_txt"], "image_rows_per_gpu_step": B, "text_rows_per_gpu_step": BT,
              "global_batch": (B + BT) * world, "optimizer": "adamw", "alpha": ALPHA, "parallelism": f"dp{world}",
              "inputs": "value: banks and the timed steps' index batches resident in HBM when the clock starts (rows are "
                        "gathered from the banks inside the timed region); e2e: sampler + per-step index uploads + loss "
                        "read-back inside the timed region",
              "sampler": "single global permutation, bit-exact with the reference's DataLoader order" if world == 1 else
                         "per-rank shard permutation (DistributedSampler-style, equal strided shards); dW summed over the ranks by "
                         "the step's last kernel (split-K sum + two-shot all-reduce over NVLink peer memory + Adam, csrc/dp.cu)",
              "l2_policy": "inputs larger than L2: every step gathers fresh rows from a 3.9 GB bank and rewrites a "
                           "gradient-logit matrix of 2 KB per row" if args.workload != "cfg2" else "working set fits L2 (few-shot)"}

    if args.impl == "reference":
        if rank != 0:
            return
        from oracle import ref_harness as _rh
        if args.ref_device == "cpu" and _rh.reference_available() and not wl.get("dv"):
            r = reference_train_run(wl, args.steps, args.warmup, budget_s=150.0)  # the reference itself
        else:  # (GPU variant / no reference tree at hand: the oracle port, kind "port")
            r = cpu_reference_run(wl, args.steps, args.warmup, budget_s=150.0, device=args.ref_device)
            r["kind"] = "port"
        line = {"impl": "reference", "metric": "UML train samples/sec (img+text)", "value": r["value"], "unit": "samples/s",
                "n_gpus": args.gpus, "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": r["kind"],
                                 "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        if args.ref_device == "cuda":  # informational like-for-like arm (SURVEY 8d); the driver's arm is the CPU one
            line.update(ref_device="cuda", eager_gpu={"device_ms_per_step": r["device_ms_per_step"],
                                                      "device_only_samples_per_s": r["device_only_value"],
                                                      "note": "torch eager fp32 ops of the port on one GPU; value/e2e include the "
                                                              "host-side per-sample collate and the H2D copy of every batch"})
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the UML hot path has no CPU implementation "
                         "(use --impl reference for the CPU arm)")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.distributed.init_process_group("nccl", device_id=dev)
    res = run_ours(args, wl, rank, world, dev)
    if rank == 0:
        K = args.steps
        value = res["rows"] / (res["ms"] * 1e-3)
        used_bf16 = "head_fwd_ce_bf16" in res["ktimes"]
        rows_per_gpu = res["rows"] / (K * world)  # mean rows per GPU and step actually processed (epoch tails are short)
        if used_bf16:
            kname = "head_fwd_ce_bf16"
            kms = res["ktimes"][kname]
            flops = 2.0 * rows_per_gpu * D * C  # algorithmic: the forward contraction only (4*D*C/sample is fwd+dW)
            # The timed region is milliseconds long at full clocks, nowhere near the seconds-long, power-capped loop the
            # "sustained" figure was measured in: the denominator is the BURST peak (the sustained fraction is kept
            # beside it for reference).
            roof = {"bound": "tensor", "kernel": kname, "achieved": flops / (kms * 1e-3) / 1e12,
                    "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                    # dram__bytes_read.sum + dram__bytes_write.sum of this kernel per launch at the cfg3 shape, from the
                    # committed `ncu --set full` capture profiles/r02_fwd_exchange.md (73728 rows: 124.6 MB read + 116.7 MB
                    # written; algorithmic: 113 MB of bf16 rows + 1.5 MB of weights read, 151 MB of G written, part of
                    # which is still in L2 when the kernel ends), scaled by the rows of the step
                    "traffic": 2.414e8 * rows_per_gpu / 73728.0 if (D, C) == (768, 1000) else None,
                    "traffic_unit": "bytes per launch",
                    "peak_source": f"{peaks['src']} bf16 burst (the timed region is {res['ms']:.1f} ms long)",
                    "frac_of_sustained_peak": flops / (kms * 1e-3) / 1e12 / peaks["tf_sustained"]}
        else:
            from uml_b200 import _lib as _l
            if _l.load().uml_head_step_fused_count() > 0:
                # the whole exact step ran as ONE cooperative launch (csrc/simt.cu head_step_fused_kernel); the C launcher's
                # forward events bracket it.  Algorithmic bytes: W, m, v read and written once (24 B/parameter - neither the
                # logits' gradient nor dW reach HBM) plus the step's bank rows, labels and indices
                kname = "head_step_fused_kernel"
                kms = res["ktimes"].get("head_fwd_ce_f32", res["breakdown"].get("head_fwd_ce_f32", float("nan")))
                bytes_ = 24.0 * C * D + rows_per_gpu * (4.0 * D + 16.0)
                note = ("one launch per step; a 12 MB working set at a 32 + 32-row step is latency bound, not bandwidth bound; "
                        "ncu (profiles/r02_fused_step.md): 6.36 MB read from DRAM per launch at cfg2, the updated state stays in L2")
            else:
                kname = "head_bwd_dw_f32"
                kms = res["ktimes"].get(kname, float("nan"))
                bytes_ = 28.0 * C * D  # AdamW pass fused in the dW epilogue: p,g,m,v read + p,m,v written
                note = None
            roof = {"bound": "hbm", "kernel": kname, "achieved": bytes_ / (kms * 1e-3) / 1e9, "peak": peaks["hbm"],
                    "unit": "GB/s", "traffic": None, "peak_source": f"{peaks['src']} HBM copy",
                    "algorithmic_bytes_per_launch": bytes_}
            if note:
                roof["note"] = note
        roof["frac"] = roof["achieved"] / roof["peak"]
        roof["kernel_ms"] = {k: round(v, 5) for k, v in res["ktimes"].items()}
        roof["step_breakdown_ms"] = {k: round(v, 5) for k, v in res["breakdown"].items()}
        step_flops = 4.0 * D * C * rows_per_gpu
        if wl.get("dv"):  # SURVEY 8d: image row 4 Dv D + 6 D C (proj fwd + dW_proj + head fwd + dW + dZ), text row 4 D C
            fi, ftx = 4.0 * wl["dv"] * D + 6.0 * D * C, 4.0 * D * C
            step_flops = rows_per_gpu * (fi * B + ftx * BT) / (B + BT)
        line = {"metric": "UML train samples/sec (img+text)", "value": value, "unit": "samples/s", "n_gpus": world,
                "steps": K, "warmup": args.warmup, "ms_per_step": res["ms"] / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if used_bf16 else "f32", "data": "synthetic",
                "config": config, "clocks": res["clocks"],
                "e2e": {"value": res["e2e_value"], "unit": "samples/s", "h2d_bytes_per_step": res["h2d"],
                        "d2h_bytes_per_step": res["d2h"], "stat": "median of 3 train() calls",
                        "all": [round(x) for x in res["e2e_all"]]},
                "gpu_launches": res["launches"], "host_enqueue_ms_per_step": res["host_ms"], "roofline": roof,
                "step_tensor_frac": {"achieved_tflops_per_gpu": step_flops / (res["ms"] / K * 1e-3) / 1e12,
                                     "of_sustained_peak": step_flops / (res["ms"] / K * 1e-3) / 1e12 / peaks["tf_sustained"],
                                     "of_burst_peak": step_flops / (res["ms"] / K * 1e-3) / 1e12 / peaks["tf_burst"],
                                     "algorithmic_flops_per_sample": step_flops / rows_per_gpu},
                "final_losses": res["loss_tail"]}
        if world == 1 and wl.get("dv"):
            line["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": 0, "kind": "port",
                                    "sample": "not run: the CPU port in bench.py covers the linear-head step only"}
        elif world == 1:
            try:
                r = cpu_reference_run(wl, 10 ** 6, 1, budget_s=args.cpu_seconds)
                line["cpu_baseline"] = {"value": r["value"], "unit": "samples/s", "cores": r["cores"], "kind": "port",
                                        "sample": r["sample"]}
            except Exception as e:  # the baseline is a reported extra; never lose the measurement over it
                line["cpu_baseline"] = {"value": None, "unit": "samples/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
