"""Float64 reference of one training step as ``uml_linear_step`` defines it (include/uml_b200.h).

No kernel calls: the module runs wherever its input tensors live (CPU or GPU).  A step pushes one or two runs of rows
through the shared head W [C, D]; run i has rows X_i [n_i, D], labels y_i, a logit scale s_i (fixed, or a learnable
temperature) and a loss weight w_i.  Per run:

    logits = s_i * X_i W^T,   loss_mean_i = mean CE,   G_i = w_i * s_i / n_i * (softmax - onehot)
    dscale_i = d (w_i * loss_mean_i) / d s_i = w_i / n_i * sum((softmax - onehot) * X_i W^T)
    dW = sum_i G_i^T X_i

then one optimizer step of W (AdamW, Adam with L2, SGD with momentum and L2) and, for a learnable temperature, one
scalar step of s_i with the same rule fed from dscale_i.  A run without rows gives its temperature no gradient: that
temperature is left untouched, as torch.optim skips a parameter whose .grad is None.

``bf16_operands=True`` rounds X and W to bf16 first, as the tensor-core step's operands are; everything after that is
float64.  Large steps are processed in row blocks, so the benchmark's 73728 x 1000 logits never exist at once.

``adapter_step`` adds the image adapter Wp [D, Dv] of a UML head (preset ``linear``): the image run's rows become
Z = X_img Wp^T, then dZ = G_img W with W taken before its update, dWp = dZ^T X_img, and Wp takes the same rule as W
(one parameter group).  A step without image rows leaves Wp, its m, v and step count untouched.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional

import torch

KINDS = {"adamw": 1, "adam": 2, "sgd": 3}


@dataclass
class Hyper:
    """uml_update: the optimizer rule and its hyper-parameters (fp32 in the C struct: pass the rounded values)."""
    kind: str = "adamw"
    lr: float = 1e-3
    beta1: float = 0.9
    beta2: float = 0.999
    eps: float = 1e-8
    weight_decay: float = 0.0
    momentum: float = 0.9

    def as_f32(self) -> "Hyper":
        """The values the kernels see: every hyper-parameter rounded to fp32."""
        f = lambda x: float(torch.tensor(x, dtype=torch.float32))
        return Hyper(self.kind, f(self.lr), f(self.beta1), f(self.beta2), f(self.eps), f(self.weight_decay),
                     f(self.momentum))


@dataclass
class Temperature:
    """A learnable logit scale with its optimizer state (0-dim tensors) and 1-based step count."""
    value: torch.Tensor
    m: torch.Tensor
    v: Optional[torch.Tensor]
    step: int


@dataclass
class RunIn:
    x: torch.Tensor                 # [n, D] the rows this run selects (any float dtype)
    labels: torch.Tensor            # [n] int
    scale: float = 1.0              # ignored when `temp` is given
    loss_weight: float = 1.0
    temp: Optional[Temperature] = None

    @property
    def n(self) -> int:
        return int(self.x.shape[0])


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(torch.float64)


def apply_update(hp: Hyper, p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: Optional[torch.Tensor], step: int):
    """One step of ``hp.kind`` in float64 on copies; returns (p, m, v).  torch.optim's single-tensor rules:
    AdamW decays p by (1 - lr * wd) first, Adam adds wd * p to the gradient, SGD adds wd * p and takes the gradient as
    its momentum buffer at step 1."""
    p, g, m = p.double().clone(), g.double(), m.double().clone()
    v = v.double().clone() if v is not None else None
    if hp.kind == "sgd":
        if hp.weight_decay:
            g = g + hp.weight_decay * p
        m = g.clone() if step <= 1 else hp.momentum * m + g
        p = p - hp.lr * m
        return p, m, v
    if hp.kind == "adamw":
        p = p * (1.0 - hp.lr * hp.weight_decay)
    elif hp.kind == "adam":
        if hp.weight_decay:
            g = g + hp.weight_decay * p
    else:
        raise ValueError(hp.kind)
    m = m + (g - m) * (1.0 - hp.beta1)
    v = v * hp.beta2 + (1.0 - hp.beta2) * g * g
    bc1 = 1.0 - hp.beta1 ** step
    bc2_sqrt = math.sqrt(1.0 - hp.beta2 ** step)
    p = p - (hp.lr / bc1) * m / (v.sqrt() / bc2_sqrt + hp.eps)
    return p, m, v


def run_scale(r: RunIn) -> float:
    return float(r.temp.value) if r.temp is not None else float(r.scale)


def forward_backward(W: torch.Tensor, runs: List[RunIn], bf16_operands: bool = False, keep_g: bool = True,
                     block_rows: int = 16384):
    """Statistics, G and dW of one step.  Returns a dict:
        stats: per run {loss_mean, dscale, correct, n, near_ties}; near_ties counts rows whose top-2 margin of scaled
               logits is <= 1e-3 * max(1, |top|), where an argmax computed in other arithmetic may differ
        G:     [sum n_i, C] float64 (rows of run 0, then run 1), when keep_g
        dW:    [C, D] float64"""
    rnd = bf16_round if bf16_operands else (lambda t: t.double())
    W64 = rnd(W)
    dW = torch.zeros_like(W64)
    stats, gs = [], []
    for r in runs:
        s, n = run_scale(r), r.n
        loss = dscale = 0.0
        correct = ties = 0
        for lo in range(0, n, block_rows):
            x = rnd(r.x[lo:lo + block_rows])
            y = r.labels[lo:lo + block_rows].to(x.device).long()
            raw = x @ W64.t()
            lg = raw * s
            lse = torch.logsumexp(lg, 1)
            loss += float((lse - lg.gather(1, y.view(-1, 1)).squeeze(1)).sum())
            top2 = lg.topk(min(2, lg.shape[1]), dim=1).values
            correct += int((lg.argmax(1) == y).sum())
            if lg.shape[1] > 1:
                ties += int(((top2[:, 0] - top2[:, 1]) <= 1e-3 * top2[:, 0].abs().clamp_min(1.0)).sum())
            p = torch.softmax(lg, 1)
            p[torch.arange(x.shape[0], device=x.device), y] -= 1.0
            dscale += float((p * raw).sum()) * r.loss_weight / n
            g = p * (r.loss_weight * s / n)
            dW += g.t() @ x
            if keep_g:
                gs.append(g)
        stats.append(dict(loss_mean=loss / n if n else 0.0, dscale=dscale, correct=correct, n=n, near_ties=ties))
    out = dict(stats=stats, dW=dW)
    if keep_g:
        out["G"] = torch.cat(gs) if gs else W64.new_zeros((0, W64.shape[0]))
    return out


def linear_step(W: torch.Tensor, runs: List[RunIn], hp: Hyper, step: int, m: torch.Tensor, v: Optional[torch.Tensor],
                bf16_operands: bool = False, keep_g: bool = True, block_rows: int = 16384):
    """One whole step: forward_backward, then W's update with ``hp`` at 1-based ``step`` and each learnable
    temperature's scalar update (runs without rows skip theirs).  Adds W, m, v and temps ([(value, m, v) or None per
    run], float64) to forward_backward's dict."""
    out = forward_backward(W, runs, bf16_operands, keep_g, block_rows)
    out["W"], out["m"], out["v"] = apply_update(hp, W, out["dW"], m, v, step)
    temps = []
    for r, st in zip(runs, out["stats"]):
        if r.temp is None or r.n == 0:
            temps.append(None if r.temp is None else (r.temp.value.double(), r.temp.m.double(),
                                                      None if r.temp.v is None else r.temp.v.double()))
            continue
        g = torch.tensor(st["dscale"], dtype=torch.float64, device=r.temp.value.device)
        temps.append(apply_update(hp, r.temp.value, g, r.temp.m, r.temp.v, r.temp.step))
    out["temps"] = temps
    return out


@dataclass
class Adapter:
    """The image adapter Wp [D, Dv] with its optimizer state and step count (steps taken so far)."""
    Wp: torch.Tensor
    m: torch.Tensor
    v: Optional[torch.Tensor]
    step: int


def adapter_step(W: torch.Tensor, ad: Adapter, img: Optional[RunIn], txt: Optional[RunIn], hp: Hyper, step: int,
                 m: torch.Tensor, v: Optional[torch.Tensor]):
    """One step of a head with an image adapter.  ``img.x`` holds the image features X_img [n_img, Dv] (not Z);
    ``step`` is W's 1-based step.  Returns linear_step's dict over the runs [image (rows Z), text] that have rows, plus
    Z [n_img, D], dZ, dWp (None without image rows) and Wp, Wp_m, Wp_v, Wp_step after the step."""
    W64 = W.double()
    runs, Z = [], None
    if img is not None and img.n:
        Z = img.x.double() @ ad.Wp.double().t()
        runs.append(RunIn(Z, img.labels, img.scale, img.loss_weight, img.temp))
    if txt is not None and txt.n:
        runs.append(txt)
    out = linear_step(W64, runs, hp, step, m, v, keep_g=True)
    out["Z"], out["dZ"], out["dWp"] = Z, None, None
    out["Wp"], out["Wp_m"] = ad.Wp.double(), ad.m.double()
    out["Wp_v"] = ad.v.double() if ad.v is not None else None
    out["Wp_step"] = ad.step
    if Z is not None:
        out["dZ"] = out["G"][:img.n] @ W64
        out["dWp"] = out["dZ"].t() @ img.x.double()
        out["Wp_step"] = ad.step + 1
        out["Wp"], out["Wp_m"], out["Wp_v"] = apply_update(hp, ad.Wp, out["dWp"], ad.m, ad.v, out["Wp_step"])
    return out
