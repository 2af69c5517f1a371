"""What the tests of uml_linear_step / uml_linear_run share: a run of rows as the C ABI reads it (Run), the caller-owned
buffers of a step (Workspace) and the checks of the per-run statistics and of an optimizer update.  Both precisions use
them: tests/test_linear_step_gpu.py (the bf16 tensor-core step) and tests/test_linear_step_fp32_gpu.py (the exact fp32
step)."""
import math
from dataclasses import dataclass
from typing import List, Optional

import torch

from linear_step_ref import Hyper, RunIn, Temperature

if torch.cuda.is_available():
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, ops

DEV = "cuda:0"
U = 2.0 ** -24   # fp32 unit roundoff
OPT_STEP = 5   # a warm Adam state: at step 1 AdamW takes lr * sign(g), which flips for near-zero gradients


def stream():
    return torch.cuda.current_stream().cuda_stream


def call(fn, *args):
    _lib.check(fn(*args))


# ------------------------------------------------------------------------------------------ one run of a step
@dataclass
class Run:
    """One run of rows as the step reads it, and what its gather must produce."""
    n: int
    rows: torch.Tensor                   # fp32 bank (or the dense rows when idx is None)
    labels: torch.Tensor                 # int64 bank labels (dense labels when neither idx nor label_idx)
    idx: Optional[torch.Tensor]
    rows16: Optional[torch.Tensor] = None
    label_idx: Optional[torch.Tensor] = None
    scale: float = 1.0
    loss_weight: float = 1.0
    temp: Optional[dict] = None          # {"value", "m", "v"} 0-dim fp32 device tensors + "step"

    def segment(self):
        sd = self.temp["value"].data_ptr() if self.temp else None
        return _lib.Segment(self.rows.data_ptr(), self.idx.data_ptr() if self.idx is not None else None,
                            self.labels.data_ptr(), self.n, self.rows.stride(0), self.scale, self.loss_weight,
                            self.label_idx.data_ptr() if self.label_idx is not None else None, sd,
                            self.rows16.data_ptr() if self.rows16 is not None else None)

    def x(self):
        """The fp32 rows the step reads."""
        return self.rows[self.idx[:self.n]] if self.idx is not None else self.rows[:self.n]

    def x16(self):
        """The rows the step must gather, in bf16."""
        return self.x().to(torch.bfloat16)

    def y(self):
        sel = self.label_idx if self.label_idx is not None else self.idx
        return (self.labels[sel[:self.n]] if sel is not None else self.labels[:self.n]).to(torch.int32)

    def ref_in(self, x16):
        t = None
        if self.temp:
            t = Temperature(self.temp["value"].double(), self.temp["m"].double(), self.temp["v"].double()
                            if self.temp["v"] is not None else None, self.temp["step"])
        return RunIn(x16, self.y(), self.scale, self.loss_weight, t)


class Workspace:
    """Caller-owned buffers of the step (the library never allocates).  G has ``g_capacity_rows`` rows (default
    ``rows``): the fp32 forward splits its contraction over planes of G when there is room for them, and the engine's
    fp32 workspace of a small step has 8x the rows (ops.HeadWorkspace)."""

    def __init__(self, D, C, rows, n_buffers=1, precision=1, g_capacity_rows=None):
        self.D, self.C, self.rows = D, C, rows
        self.ldg = (C + 63) // 64 * 64
        g_rows = rows if g_capacity_rows is None else g_capacity_rows
        self.G = torch.empty((g_rows, self.ldg), device=DEV, dtype=torch.bfloat16 if precision else torch.float32)
        self.row_loss = torch.empty(rows, device=DEV)
        self.row_correct = torch.empty(rows, device=DEV, dtype=torch.int32)
        self.row_dscale = torch.empty(rows, device=DEV)
        self.X16 = [torch.empty((rows, D), device=DEV, dtype=torch.bfloat16) for _ in range(n_buffers)]
        self.labels32 = [torch.empty(rows, device=DEV, dtype=torch.int32) for _ in range(n_buffers)]
        self.W16 = torch.empty((C, D), device=DEV, dtype=torch.bfloat16)
        self.max_splits = max(1, ops.tc_dw_splits(rows, D, C))
        self.partials = torch.empty((self.max_splits, C, D), device=DEV)
        self.tile_ws = torch.zeros(16 + (rows + 255) // 256 * 264 + rows * 32, device=DEV)  # UML_TILE_WS_FLOATS
        self.dW = torch.empty((C, D), device=DEV)

    def args(self, runs: List[Run], W, m, v, hp: Hyper, opt_step, stats, *, dW_out=None, dW_scratch=None,
             w16_valid=1, max_splits=None, precision=1):
        a = _lib.LinearStepArgs()
        a.dim, a.n_classes, a.nseg, a.precision = self.D, self.C, len(runs), precision
        for k, r in enumerate(runs):
            a.seg[k] = r.segment()
            if r.temp:
                a.scale_param[k], a.scale_m[k] = r.temp["value"].data_ptr(), r.temp["m"].data_ptr()
                a.scale_v[k] = r.temp["v"].data_ptr() if r.temp["v"] is not None else None
                a.scale_step[k] = r.temp["step"]
        a.W = W.data_ptr()
        a.upd = ops.make_update(hp.kind, hp.lr, opt_step, m, v if hp.kind != "sgd" else None,
                                weight_decay=hp.weight_decay, betas=(hp.beta1, hp.beta2), eps=hp.eps, momentum=hp.momentum)
        a.G, a.ldg, a.g_capacity_rows = self.G.data_ptr(), self.ldg, self.G.shape[0]
        a.row_loss, a.row_correct, a.row_dscale = (self.row_loss.data_ptr(), self.row_correct.data_ptr(),
                                                   self.row_dscale.data_ptr())
        a.stats = stats.data_ptr()
        if precision:
            a.X16, a.labels32, a.W16 = self.X16[0].data_ptr(), self.labels32[0].data_ptr(), self.W16.data_ptr()
            a.partials, a.tile_ws = self.partials.data_ptr(), self.tile_ws.data_ptr()
            a.max_splits = self.max_splits if max_splits is None else max_splits
            a.w16_valid = w16_valid
        a.dW_out = dW_out.data_ptr() if dW_out is not None else None
        a.dW_scratch = dW_scratch.data_ptr() if dW_scratch is not None else None
        return a


def stats_rec(stats, k):
    f, i = stats[k].cpu(), stats[k].cpu().view(torch.int32)
    return dict(loss_mean=float(f[0]), dscale=float(f[1]), correct=int(i[2]), n=int(i[3]))


def check_stats(stats, ref_stats, where="", dscale=True, bounds=None):
    """dscale is d loss / d scale for a learnable temperature: with fixed scales the bf16 step need not compute it.
    ``bounds``: per run {"loss": ..., "dscale": ...} absolute bounds in place of the relative defaults (2e-4 on
    loss_mean, 2e-3 on dscale)."""
    for k, r in enumerate(ref_stats):
        got = stats_rec(stats, k)
        assert got["n"] == r["n"], (where, k, got, r)
        if bounds is None:
            assert math.isclose(got["loss_mean"], r["loss_mean"], rel_tol=2e-4, abs_tol=1e-6), (where, k, got, r)
        else:
            assert abs(got["loss_mean"] - r["loss_mean"]) <= bounds[k]["loss"], (where, k, got, r, bounds[k])
        if dscale:
            if bounds is None:
                assert math.isclose(got["dscale"], r["dscale"], rel_tol=2e-3, abs_tol=1e-6), (where, k, got, r)
            else:
                assert abs(got["dscale"] - r["dscale"]) <= bounds[k]["dscale"], (where, k, got, r, bounds[k])
        assert abs(got["correct"] - r["correct"]) <= r["near_ties"], (where, k, got, r)


def check_update(got, want, what, rtol=2e-6, atol=2e-7):
    """max |got - want| / (atol + rtol |want|) <= 1; returns that ratio."""
    ratio = float(((got.double() - want).abs() / (atol + rtol * want.abs())).max())
    assert ratio <= 1.0, (what, ratio)
    return ratio


def temp_state(value, g, kind):
    """A learnable temperature at OPT_STEP with a seeded optimizer state."""
    return dict(value=torch.tensor(value, device=DEV), m=torch.tensor(float(torch.randn(1, generator=g)) * 0.3, device=DEV),
                v=None if kind == "sgd" else torch.tensor(0.05 + float(torch.rand(1, generator=g)) * 0.1, device=DEV),
                step=OPT_STEP)


def recover_grad(kind, hp, m0, m1, w0):
    """The gradient a fused update was fed, recovered in float64 from the moments before (m0) and after (m1) it, and
    the bound of that recovery: Adam(W) g = m0 + (m1 - m0) / (1 - beta1), minus Adam's L2 term wd w0; SGD
    g = m1 - momentum m0 - wd w0."""
    m0, m1, w0 = m0.double(), m1.double(), w0.double()
    if kind == "sgd":
        g = m1 - hp.momentum * m0 - hp.weight_decay * w0
    else:
        g = m0 + (m1 - m0) / (1.0 - hp.beta1)
        if kind == "adam":
            g = g - hp.weight_decay * w0
    return g, 16 * U * (m0.abs() + m1.abs() + g.abs() + hp.weight_decay * w0.abs())
