"""The exact fp32 training step (precision 0, csrc/simt.cu) and the adapter's fp32 step, against the float64
reference of tests/linear_step_ref.py on the same fp32 inputs.

* test_step_matches_the_float64_reference drives uml_linear_step through the C ABI; every case names the branch of the
  launcher it forces and asserts it was taken: the cooperative fused kernel (a uml_head_step_fused_count() delta of 1),
  or the separate launches (forward GEMM + softmax, dW GEMM with the update in its epilogue) for one of their causes.
  Tile size and split-K planes cannot be observed; the case table computes them with the launcher's own rules.
* test_run_is_bit_identical_to_single_steps: uml_linear_run over steps that alternate between the two branches.
* test_adapter_step_matches_the_float64_reference: StepEngine.step of a UML head with an image adapter (preset
  `linear`), precision "fp32".

Data.  CLIP heads: unit-norm rows and weight rows at logit scale 100.  Adapters: features randn / sqrt(Dv), the
model's own initialisation, temperatures 1.

Bounds (u = 2^-24).  A logit is an FMA chain of D terms; its rounding errors are treated as independent, so the scaled
logits of a row are off by at most e = 4 u s sqrt(D) max|x| max|w| (four standard deviations).  For an adapter the
measured error of Z adds s max_c sum_d |dZ_rd| |W_cd|.  Then, per run with weight w over n rows:
  G:        |G - G_ref| <= w s / n (2.01 e + (C/256 + 16) u)   (p moves by at most exp(2e) - 1 relatively; the row sum)
  loss:     |loss_mean - ref| <= 2.01 e + (C/256 + 16 + n) u max(1, loss)
  dscale:   |dscale - ref| <= w (2.01 e max|raw| + 2 e / s + 2 (C/256 + 16 + n) u max|raw|)
  gradient: |dW - dW_ref| <= sum_r bound_G(r) |x_rd| + n u (|G_ref|^T |X|)   (the adapter adds |G_ref|^T |dZ|)
Every GEMM is also checked against float64 arithmetic on its own fp32 operands with the worst-case bound K u of an FMA
chain of K terms: the gradient against G^T X of the step's own G, dZ against G_img W, dWp against dZ^T X_img.
The update: a fused update exposes no gradient, so it is recovered from the moment the step wrote,
g = m0 + (m1 - m0) / (1 - beta1) (Adam's L2 term wd w0 subtracted) or, for SGD, g = m1 - momentum m0 - wd w0, to within
16 u (|m0| + |m1| + |g| + wd |w0|).  That gradient must pass the GEMM's own bound, and W, m and v must follow from it
with the float64 rule to rtol 2e-6 / atol 2e-7 (v: atol 1e-12).  lr and wd are chosen so that at the median element
the decay term, lr wd |w| for AdamW and wd |w| in the gradient for Adam and SGD, is at least 10x the bound that would
catch its absence; the test asserts this and prints the margins.
"""
import ctypes
import math

import pytest
import torch

from linear_step_case import (DEV, OPT_STEP, U, Run, Workspace, call, check_stats, check_update, recover_grad,
                              stats_rec, stream, temp_state)
from linear_step_ref import Adapter, Hyper, RunIn, Temperature, adapter_step, apply_update, forward_backward

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from uml_b200 import _lib

LR, WD = 1e-2, 0.05


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------ the launcher's rules
def sgemm_tile(M, N):
    """launch_sgemm: 64 x 64 tiles when they make at least two waves, else 32 x 32."""
    return 64 if (-(-M // 64)) * (-(-N // 64)) >= 2 * _sms() else 32


def fwd_planes(total, C, D, g_capacity_rows):
    """uml_head_fwd_ce_f32: split-K planes of the logit GEMM."""
    ctas = (-(-total // 32)) * (-(-C // 32))
    if ctas >= 2 * _sms() or g_capacity_rows < 2 * total:
        return 1
    want, room, deep = -(-2 * _sms() // ctas), g_capacity_rows // total, -(-D // 64)
    return max(1, min(want, room, deep, 8))


def fused_fits(runs, D, C, W, m, v, kind):
    """uml_head_step_fused_f32's contract."""
    total = sum(r.n for r in runs)
    al = lambda t: t.data_ptr() % 16 == 0
    if not 0 < total <= 128 or D % 4 or not (al(W) and al(m) and (kind == "sgd" or al(v))):
        return False
    if any(r.n and (r.rows.data_ptr() % 16 or r.rows.stride(0) % 4) for r in runs):
        return False
    nc_max = -(-C // _sms()) + 1
    return total * (D + 16) * 4 + nc_max * D * 4 + total * (nc_max + 3) * 4 <= 224 * 1024


# ------------------------------------------------------------------------------------------ bounds
def logit_err(x, W, s):
    return 4 * U * s * math.sqrt(W.shape[1]) * float(x.double().norm(dim=1).max()) * float(W.double().norm(dim=1).max())


def g_bound(w, s, n, e, C):
    return w * s / n * (2.01 * e + (C / 256 + 16) * U)


def stat_bounds(ref_stats, xs, W, scales, weights, errs, C):
    out = []
    for r, x, s, w, e in zip(ref_stats, xs, scales, weights, errs):
        n = r["n"]
        raw = float((x.double() @ W.double().t()).abs().max())
        tail = (C / 256 + 16 + n) * U
        out.append(dict(loss=2.01 * e + tail * max(1.0, r["loss_mean"]),
                        dscale=w * (2.01 * e * raw + 2 * e / s + 2 * tail * raw)))
    return out


def ratio(got, want, bound):
    return float(((got.double() - want).abs() / bound).max())


def warm_state(g_ref, gen, kind):
    """m0, v0 around the reference gradient: v0 bounded away from zero, so that Adam's step is smooth in g."""
    u = lambda lo, hi: torch.rand(g_ref.shape, device=g_ref.device, generator=gen, dtype=torch.float64) * (hi - lo) + lo
    m0 = (g_ref * u(-1.0, 2.0)).float()
    floor = (0.05 * float(g_ref.abs().max())) ** 2
    v0 = ((g_ref * g_ref + floor) * u(0.5, 2.0)).float() if kind != "sgd" else torch.zeros_like(m0)
    return m0, v0


def check_fused_update(what, kind, hp, step, W0, m0, v0, W, m, v, g_own, g_own_bound):
    """The update of one parameter: its recovered gradient against float64 arithmetic on the step's own operands
    (g_own, bound g_own_bound), then W, m and v against the float64 rule fed that gradient.  Returns the gradient and
    the margins."""
    g, rec = recover_grad(kind, hp, m0, m, W0)
    r_grad = ratio(g, g_own, g_own_bound + rec)
    assert r_grad <= 1.0, (what, "recovered gradient", r_grad)
    Ww, mw, vw = apply_update(hp, W0, g, m0, v0 if kind != "sgd" else None, step)
    r_w = check_update(W, Ww, what + " W")
    check_update(m, mw, what + " m")
    if kind != "sgd":
        check_update(v, vw, what + " v", atol=1e-12)
    # the decay is visible: at the median element it is >= 10x the bound that would miss it
    w0 = W0.double().abs()
    if kind == "adamw":
        margin = float((hp.lr * hp.weight_decay * w0 / (2e-7 + 2e-6 * Ww.abs())).median())
    else:
        margin = float((hp.weight_decay * w0 / (g_own_bound + rec)).median())
    assert margin >= 10.0, (what, "weight decay below the bound", margin)
    return g, dict(grad=r_grad, W=r_w, decay_margin=margin)


# ------------------------------------------------------------------------------------------ (a) one step vs float64
# runs: (rows, mode): idx = fp32 bank + idx, dense = idx NULL, label_idx = labels through label_idx, offset = a bank view
# one float off 16-byte alignment, strided = a bank with ld = D + 1.  The second run is the text run (loss weight 0.5).
CASES = {
    "cfg2": dict(runs=[(32, "idx"), (32, "idx")], D=512, C=1000, kind="adamw", fused=True),
    "rows128": dict(runs=[(100, "idx"), (28, "idx")], D=256, C=397, kind="sgd", fused=True),
    "rows129": dict(runs=[(100, "idx"), (29, "idx")], D=256, C=397, kind="adam", fused=False),
    "d768_fits": dict(runs=[(32, "idx"), (32, "idx")], D=768, C=1000, kind="adam", learnable=True, fused=True),
    "c101": dict(runs=[(20, "idx"), (12, "idx")], D=128, C=101, kind="sgd", learnable=True, fused=True),
    "c10": dict(runs=[(8, "idx"), (8, "idx")], D=64, C=10, kind="adamw", fused=True),
    "d36": dict(runs=[(16, "idx"), (16, "idx")], D=36, C=50, kind="adam", fused=True),
    "one_run": dict(runs=[(48, "idx")], D=512, C=1000, kind="adamw", learnable=True, fused=True),
    "dense": dict(runs=[(32, "dense"), (32, "dense")], D=256, C=300, kind="sgd", fused=True),
    "label_idx": dict(runs=[(32, "label_idx"), (32, "label_idx")], D=512, C=1000, kind="adamw", fused=True),
    "d3200_planes": dict(runs=[(32, "idx"), (32, "idx")], D=3200, C=1000, kind="adamw", learnable=True, fused=False,
                         planes=5, dw_tile=64, no_planes_twin=True),
    "d50": dict(runs=[(32, "idx"), (32, "idx")], D=50, C=1000, kind="sgd", fused=False),
    "offset_bank": dict(runs=[(32, "offset"), (32, "idx")], D=256, C=1000, kind="adam", fused=False),
    "strided_bank": dict(runs=[(32, "strided"), (32, "strided")], D=256, C=1000, kind="adamw", learnable=True,
                         fused=False),
    "rows64_d1024": dict(runs=[(32, "idx"), (32, "idx")], D=1024, C=1000, kind="adamw", fused=False),
    "rows1200": dict(runs=[(600, "idx"), (600, "idx")], D=256, C=1000, kind="adam", fused=False, fwd_tile=64),
}
SCALES, WEIGHTS = (100.0, 100.0), (1.0, 0.5)


def _unit(t):
    return t / t.norm(dim=1, keepdim=True)


def _make_runs(cfg, g):
    D, C = cfg["D"], cfg["C"]
    runs = []
    for k, (n, mode) in enumerate(cfg["runs"]):
        bank_rows = n if mode == "dense" else n + n // 7 + 5
        rows = _unit(torch.randn(bank_rows, D, device=DEV, generator=g))
        if mode == "offset":
            flat = torch.zeros(bank_rows * D + 4, device=DEV)
            flat[1:1 + bank_rows * D] = rows.flatten()
            rows = flat[1:1 + bank_rows * D].view(bank_rows, D)
        elif mode == "strided":
            wide = torch.zeros(bank_rows, D + 1, device=DEV)
            wide[:, :D] = rows
            rows = wide[:, :D]
        labels = torch.randint(0, C, (bank_rows,), device=DEV, generator=g)
        idx = torch.randperm(bank_rows, device=DEV, generator=g)[:n] if mode != "dense" else None
        r = Run(n, rows, labels, idx, scale=SCALES[k], loss_weight=WEIGHTS[k])
        if mode == "label_idx":
            # run 0: dense rows (an adapter's output) with bank labels; run 1: rows by idx, labels by other indices
            r.label_idx = torch.randint(0, bank_rows, (n,), device=DEV, generator=g)
            if k == 0:
                r.rows, r.idx = rows[:n].contiguous(), None
        if cfg.get("learnable"):
            r.temp = temp_state(r.scale, torch.Generator().manual_seed(k), cfg["kind"])
        runs.append(r)
    return runs


class StepCase:
    """A case's runs, weights and reference, and one launch of the fp32 step."""

    def __init__(self, cfg, seed, g_capacity=8):
        self.cfg, D, C = cfg, cfg["D"], cfg["C"]
        self.g = torch.Generator(device=DEV).manual_seed(seed)
        self.runs = _make_runs(cfg, self.g)
        self.total = sum(r.n for r in self.runs)
        self.W0 = _unit(torch.randn(C, D, device=DEV, generator=self.g))
        self.hp = Hyper(cfg["kind"], lr=LR, weight_decay=WD).as_f32()
        self.ws = Workspace(D, C, self.total, precision=0, g_capacity_rows=g_capacity * self.total)
        self.temps0 = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in r.temp.items()} if r.temp else None
                       for r in self.runs]
        self.xs = [r.x() for r in self.runs]
        self.ref = forward_backward(self.W0, [r.ref_in(x) for r, x in zip(self.runs, self.xs)], keep_g=True)
        scales = [float(r.temp["value"]) if r.temp else r.scale for r in self.runs]
        self.errs = [logit_err(x, self.W0, s) for x, s in zip(self.xs, scales)]
        self.g_rows = torch.cat([torch.full((r.n,), g_bound(r.loss_weight, s, r.n, e, C), device=DEV, dtype=torch.float64)
                                 for r, s, e in zip(self.runs, scales, self.errs)])
        self.stat_bounds = stat_bounds(self.ref["stats"], self.xs, self.W0, scales, [r.loss_weight for r in self.runs],
                                       self.errs, C)
        X = torch.cat(self.xs).double()
        self.X = X
        self.dW_bound = (self.g_rows @ X.abs()).unsqueeze(0) + self.total * U * (self.ref["G"].abs().t() @ X.abs())

    def launch(self, W, m, v, **kw):
        for r, t0 in zip(self.runs, self.temps0):
            if t0:
                for key in ("value", "m", "v"):
                    if t0[key] is not None:
                        r.temp[key].copy_(t0[key])
        self.ws.G.fill_(float("nan"))
        stats = torch.full((2, 4), float("nan"), device=DEV)
        a = self.ws.args(self.runs, W, m, v, self.hp, OPT_STEP, stats, precision=0, **kw)
        f0 = _lib.load().uml_head_step_fused_count()
        call(_lib.load().uml_linear_step, ctypes.byref(a), stream())
        torch.cuda.synchronize()
        return stats, _lib.load().uml_head_step_fused_count() - f0

    def G(self):
        return self.ws.G[:self.total, :self.cfg["C"]].double()

    def check_forward(self, stats, where):
        """Statistics and G against the reference; returns G's margin."""
        check_stats(stats, self.ref["stats"], where, dscale=True, bounds=self.stat_bounds)
        r_g = float(((self.G() - self.ref["G"]).abs().max(dim=1).values / self.g_rows).max())
        assert r_g <= 1.0, (where, "G", r_g)
        return r_g

    def own_grad(self):
        """float64 G^T X of the step's own G, and the worst-case bound of the fp32 FMA chain over the rows."""
        G = self.G()
        return G.t() @ self.X, self.total * U * (G.abs().t() @ self.X.abs())

    def check_temps(self, stats, where):
        for k, (r, t0) in enumerate(zip(self.runs, self.temps0)):
            if not t0:
                continue
            ds = torch.tensor(stats_rec(stats, k)["dscale"], dtype=torch.float64)
            want = apply_update(self.hp, t0["value"].cpu(), ds, t0["m"].cpu(), t0["v"].cpu() if t0["v"] is not None else None,
                                t0["step"])
            check_update(r.temp["value"].cpu(), want[0], where + " temperature")
            check_update(r.temp["m"].cpu(), want[1], where + " temperature m")
            if want[2] is not None:
                check_update(r.temp["v"].cpu(), want[2], where + " temperature v")


@pytest.mark.parametrize("case", list(CASES))
def test_step_matches_the_float64_reference(case):
    cfg = CASES[case]
    D, C, kind = cfg["D"], cfg["C"], cfg["kind"]
    sc = StepCase(cfg, seed=sum(n for n, _ in cfg["runs"]) + D + C)
    runs, ws, ref = sc.runs, sc.ws, sc.ref
    # the branches this case is about, by the launcher's rules
    planes = fwd_planes(sc.total, C, D, ws.G.shape[0])
    if "planes" in cfg:
        assert planes == cfg["planes"], planes
    if "dw_tile" in cfg:
        assert sgemm_tile(C, D) == cfg["dw_tile"]
    if "fwd_tile" in cfg:
        assert planes == 1 and sgemm_tile(sc.total, C) == cfg["fwd_tile"]
    # ---- gradient only (dW_out): the separate launches, W, m and v bit-unchanged ---------------------------------
    W, m, v = sc.W0.clone(), torch.randn(C, D, device=DEV, generator=sc.g), torch.rand(C, D, device=DEV, generator=sc.g)
    Wc, mc, vc = W.clone(), m.clone(), v.clone()
    stats, fused = sc.launch(W, m, v, dW_out=ws.dW)
    assert fused == 0
    assert torch.equal(W, Wc) and torch.equal(m, mc) and torch.equal(v, vc)
    grad, G_sep = ws.dW.clone().double(), sc.G().clone()
    r_g = sc.check_forward(stats, case + " dW_out")
    r_ref = ratio(grad, ref["dW"], sc.dW_bound)
    own, own_bound = sc.own_grad()
    r_own = ratio(grad, own, own_bound + 1e-30)
    print(f"\n[{case}] planes {planes}, dW tile {sgemm_tile(C, D)}; gradient only: G {r_g:.2e}, gradient vs float64 "
          f"{r_ref:.2e}, vs its own G {r_own:.2e} of the bounds")
    assert r_ref <= 1.0 and r_own <= 1.0, (r_ref, r_own)
    sc.check_temps(stats, "dW_out")
    # ---- the update from a warm state ----------------------------------------------------------------------------
    m0, v0 = warm_state(ref["dW"], sc.g, kind)
    W, m, v = sc.W0.clone(), m0.clone(), v0.clone()
    assert fused_fits(runs, D, C, W, m, v, kind) == cfg["fused"], "the case table names the wrong branch"
    stats_u, fused = sc.launch(W, m, v)
    assert fused == int(cfg["fused"]), ("fused launches", fused)
    r_g = sc.check_forward(stats_u, case + " update")
    if not cfg["fused"]:
        assert torch.equal(sc.G(), G_sep), "the separate launches are deterministic"
        assert torch.equal(stats_u.view(torch.int32), stats.view(torch.int32))
    own, own_bound = sc.own_grad()
    g_rec, margins = check_fused_update("W", kind, sc.hp, OPT_STEP, sc.W0, m0, v0, W, m, v, own, own_bound)
    r_ref = ratio(g_rec, ref["dW"], sc.dW_bound)
    assert r_ref <= 1.0, ("recovered gradient vs float64", r_ref)
    if not cfg["fused"]:   # the epilogue saw exactly the gradient dW_out held
        _, rec = recover_grad(kind, sc.hp, m0, m, sc.W0)
        assert ratio(g_rec, grad, rec) <= 1.0
    sc.check_temps(stats_u, "update")
    print(f"[{case}] update ({'fused' if fused else 'separate'}, {kind}): G {r_g:.2e}, recovered gradient vs its own G "
          f"{margins['grad']:.2e} and vs float64 {r_ref:.2e}, W {margins['W']:.2e} of the bounds; weight decay "
          f"{margins['decay_margin']:.0f}x its bound")
    if cfg.get("no_planes_twin"):
        # the same step with G only as large as the step: one plane; both agree with each other and the reference
        twin = StepCase(cfg, seed=sum(n for n, _ in cfg["runs"]) + D + C, g_capacity=1)
        assert fwd_planes(twin.total, C, D, twin.ws.G.shape[0]) == 1
        W1, m1, v1 = sc.W0.clone(), m0.clone(), v0.clone()
        stats1, fused1 = twin.launch(W1, m1, v1)
        assert fused1 == 0
        twin.check_forward(stats1, case + " one plane")
        r_pl = float(((twin.G() - sc.G()).abs().max(dim=1).values / (2 * sc.g_rows)).max())
        assert r_pl <= 1.0, ("planes vs one plane", r_pl)
        own1, own1_bound = twin.own_grad()
        check_fused_update("W (one plane)", kind, sc.hp, OPT_STEP, sc.W0, m0, v0, W1, m1, v1, own1, own1_bound)
        print(f"[{case}] one plane vs {planes}: G apart by {r_pl:.2e} of twice the bound")


# ------------------------------------------------------------------------------------------ (b) uml_linear_run
R_D, R_C = 256, 1000
R_ROWS = [(32, 32), (5, 32), (100, 40), (64, 64), (130, 20), (16, 8)]   # fused, fused, separate, fused, separate, fused


def test_run_is_bit_identical_to_single_steps():
    """Six steps at precision 0 in one uml_linear_run with per-step lr and opt_step, against the same steps as single
    uml_linear_step calls (bit-identical), and each step against the float64 step from its own starting point."""
    g = torch.Generator(device=DEV).manual_seed(77)
    banks = []
    for nb in (400, 300):
        banks.append((_unit(torch.randn(nb, R_D, device=DEV, generator=g)), torch.randint(0, R_C, (nb,), device=DEV,
                                                                                           generator=g)))
    idx = [[torch.randperm(banks[k][0].shape[0], device=DEV, generator=g)[:n] for k, n in enumerate(rn)] for rn in R_ROWS]
    W0 = _unit(torch.randn(R_C, R_D, device=DEV, generator=g))
    hp0 = Hyper("adamw", lr=LR, weight_decay=WD).as_f32()
    lrs = [float(torch.tensor(LR * (1.0 - 0.1 * i), dtype=torch.float32)) for i in range(len(R_ROWS))]
    max_rows = max(a + b for a, b in R_ROWS)
    ws = Workspace(R_D, R_C, max_rows, precision=0, g_capacity_rows=8 * max_rows)
    runs_of = lambda i: [Run(len(ix), bank, lab, ix, scale=s, loss_weight=w)
                         for ix, (bank, lab), s, w in zip(idx[i], banks, SCALES, WEIGHTS)]
    lib = _lib.load()
    # single steps, with each step's starting point kept
    W, m, v = W0.clone(), torch.zeros_like(W0), torch.zeros_like(W0)
    stats = torch.full((len(R_ROWS), 2, 4), float("nan"), device=DEV)
    before, fused = [], []
    for i in range(len(R_ROWS)):
        before.append((W.clone(), m.clone(), v.clone()))
        f0 = lib.uml_head_step_fused_count()
        a = ws.args(runs_of(i), W, m, v, Hyper(**{**hp0.__dict__, "lr": lrs[i]}), i + 1, stats[i], precision=0)
        call(lib.uml_linear_step, ctypes.byref(a), stream())
        torch.cuda.synchronize()
        fused.append(lib.uml_head_step_fused_count() - f0)
        assert fused[-1] == int(fused_fits(runs_of(i), R_D, R_C, W, m, v, "adamw"))
    assert fused == [1, 1, 0, 1, 0, 1], fused
    # the same steps in one call
    Wr, mr, vr = W0.clone(), torch.zeros_like(W0), torch.zeros_like(W0)
    stats_r = torch.full_like(stats, float("nan"))
    base = ws.args(runs_of(0), Wr, mr, vr, hp0, 1, stats_r[0], precision=0)
    steps = (_lib.RunStep * len(R_ROWS))()
    for i, s in enumerate(steps):
        for k, ix in enumerate(idx[i]):
            s.idx[k], s.n[k], s.loss_weight[k] = ix.data_ptr(), len(ix), WEIGHTS[k]
        s.lr, s.opt_step, s.stats = lrs[i], i + 1, stats_r[i].data_ptr()
    call(lib.uml_linear_run, ctypes.byref(base), steps, len(R_ROWS), stream())
    torch.cuda.synchronize()
    assert torch.equal(stats_r.view(torch.int32), stats.view(torch.int32)), "per-step statistics records"
    assert torch.equal(Wr, W) and torch.equal(mr, m) and torch.equal(vr, v)
    # each step against the float64 step from its own starting point
    after = before[1:] + [(W, m, v)]
    for i, ((Wb, mb, vb), (Wa, ma, va)) in enumerate(zip(before, after)):
        runs = runs_of(i)
        xs = [r.x() for r in runs]
        ref = forward_backward(Wb, [r.ref_in(x) for r, x in zip(runs, xs)], keep_g=False)
        errs = [logit_err(x, Wb, s) for x, s in zip(xs, SCALES)]
        check_stats(stats[i], ref["stats"], f"step {i}",
                    bounds=stat_bounds(ref["stats"], xs, Wb, SCALES, WEIGHTS, errs, R_C))
        X = torch.cat(xs).double()
        g_rows = torch.cat([torch.full((r.n,), g_bound(r.loss_weight, s, r.n, e, R_C), device=DEV, dtype=torch.float64)
                            for r, s, e in zip(runs, SCALES, errs)])
        n = X.shape[0]
        # (the kernel's G of an earlier step is gone: the gradient is judged against the float64 one, whose G the
        # bound covers)
        G_ref = forward_backward(Wb, [r.ref_in(x) for r, x in zip(runs, xs)], keep_g=True)["G"]
        bound = (g_rows @ X.abs()).unsqueeze(0) + n * U * (G_ref.abs().t() @ X.abs())
        hp = Hyper(**{**hp0.__dict__, "lr": lrs[i]})
        g_rec, margins = check_fused_update(f"step {i} W", "adamw", hp, i + 1, Wb, mb, vb, Wa, ma, va, ref["dW"], bound)
        print(f"\n[run step {i}] {'fused' if fused[i] else 'separate'}: recovered gradient {margins['grad']:.2e}, "
              f"W {margins['W']:.2e} of the bounds")


# ------------------------------------------------------------------------------------------ (c) the adapter's step
# (Dv, D, C, n_img, n_txt)
ADAPTER_SHAPES = {"preset_linear": (1536, 3200, 1000, 32, 32), "tiny": (24, 40, 10, 8, 8), "image_only": (96, 160, 50, 37, 0),
                  "text_only": (128, 192, 100, 0, 32), "not_mult4": (30, 34, 7, 5, 3)}
ALPHA = 0.5


@pytest.mark.parametrize("learnable", [False, True], ids=["fixed", "learnable"])
@pytest.mark.parametrize("kind", ["adamw", "adam", "sgd"])
@pytest.mark.parametrize("shape", list(ADAPTER_SHAPES))
def test_adapter_step_matches_the_float64_reference(shape, kind, learnable):
    """One StepEngine.step of a UML head with an image adapter at precision "fp32" (Z = X Wp^T, the head's forward,
    dZ = G_img W, the head's dW with its update, dWp with its update) from a warm optimizer state at step 5."""
    from uml_b200.engine.datasets.utils import FeatureBank, IndexBatch
    from uml_b200.engine.models.head import UML
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.trainer import StepEngine
    Dv, D, C, ni, nt = ADAPTER_SHAPES[shape]
    seed = Dv + D + C + ni + nt + 10 * ["adamw", "adam", "sgd"].index(kind) + int(learnable)
    torch.manual_seed(seed)
    gen = torch.Generator(device=DEV).manual_seed(seed)
    model = UML(f"synthetic:{Dv}", D, C, learnable_temp=learnable)
    model.to(DEV)
    opt = build_optimizer(model.parameters(), kind, LR, WD)
    hp = Hyper(kind, lr=LR, weight_decay=WD).as_f32()
    W, Wp = model.head.weight.data, model.img_proj.weight.data
    W0, Wp0 = W.clone(), Wp.clone()
    batches, xs, ys = [], [], []
    for n, width in ((ni, Dv), (nt, D)):
        bank = FeatureBank(torch.randn(n + 40, width, device=DEV, generator=gen) / math.sqrt(Dv if width == Dv else D),
                           torch.randint(0, C, (n + 40,), device=DEV, generator=gen), DEV)
        idx = torch.randperm(n + 40, device=DEV, generator=gen)[:n]
        batches.append(IndexBatch(bank, idx, n, 0, idx.cpu()) if n else None)
        xs.append(bank.features[idx])
        ys.append(bank.labels[idx])
    # warm states at step 4 around the float64 gradient of this step (v bounded away from zero)
    temps = {}
    for name, n in (("img_scale", ni), ("txt_scale", nt)):
        if learnable:
            prm = getattr(model, name)
            st = opt.slot(prm)
            st["m"].fill_(0.3 * float(torch.randn(1, generator=gen, device=DEV)))
            if st["v"] is not None:
                st["v"].fill_(0.05 + 0.1 * float(torch.rand(1, generator=gen, device=DEV)))
            st["step"] = OPT_STEP - 1
            temps[name] = (prm.data.clone(), st["m"].clone(), None if st["v"] is None else st["v"].clone())
    ref_temp = lambda name: (Temperature(*[t.double() if t is not None else None for t in temps[name]], OPT_STEP)
                             if learnable else None)
    img_in = RunIn(xs[0], ys[0], 1.0, 1.0, ref_temp("img_scale")) if ni else None
    txt_in = RunIn(xs[1], ys[1], 1.0, ALPHA, ref_temp("txt_scale")) if nt else None
    z64 = lambda t: torch.zeros_like(t, dtype=torch.float64)
    dry = adapter_step(W0, Adapter(Wp0, z64(Wp0), z64(Wp0), 0), img_in, txt_in, hp, 1, z64(W0), z64(W0))
    state0 = {}
    for name, p, g_ref in (("W", model.head.weight, dry["dW"]), ("Wp", model.img_proj.weight,
                                                                   dry["dWp"] if ni else torch.randn_like(Wp0).double())):
        m0, v0 = warm_state(g_ref, gen, kind)
        st = opt.slot(p)
        st["m"].copy_(m0)
        if st["v"] is not None:
            st["v"].copy_(v0)
        st["step"] = OPT_STEP - 1
        state0[name] = (m0, v0)
    ref = adapter_step(W0, Adapter(Wp0, *[t.double() for t in state0["Wp"]], OPT_STEP - 1), img_in, txt_in, hp,
                       OPT_STEP, state0["W"][0], state0["W"][1])

    eng = StepEngine(model, opt, DEV, max(ni, 1), max(nt, 1), precision="fp32")
    eng.step(batches[0], batches[1], ALPHA, 0)
    torch.cuda.synchronize()
    stats = eng.stats_log[0]
    total = ni + nt
    G = eng.ws32.G[:total, :C].double()
    # ---- Z and the logit error it brings ------------------------------------------------------------------------
    run_x, errs, scales, weights, marg = [], [], [], [], {}
    if ni:
        Z = eng.Z[:ni].double()
        Zb = Dv * U * (xs[0].double().abs() @ Wp0.double().abs().t())
        marg["Z"] = ratio(Z, ref["Z"], Zb)
        assert marg["Z"] <= 1.0, ("Z", marg["Z"])
        dZr = (Z - ref["Z"]).abs()
        s = float(temps["img_scale"][0]) if learnable else 1.0
        e = s * float((dZr @ W0.double().abs().t()).max()) + logit_err(Z, W0, s)
        run_x.append(Z), errs.append(e), scales.append(s), weights.append(1.0)
    if nt:
        s = float(temps["txt_scale"][0]) if learnable else 1.0
        run_x.append(xs[1].double()), errs.append(logit_err(xs[1], W0, s)), scales.append(s), weights.append(ALPHA)
    ns = [x.shape[0] for x in run_x]
    ref_x = ([ref["Z"]] if ni else []) + ([xs[1].double()] if nt else [])
    check_stats(stats, ref["stats"], shape, bounds=stat_bounds(ref["stats"], ref_x, W0, scales, weights, errs, C))
    g_rows = torch.cat([torch.full((n,), g_bound(w, s, n, e, C), device=DEV, dtype=torch.float64)
                        for n, w, s, e in zip(ns, weights, scales, errs)])
    marg["G"] = float(((G - ref["G"]).abs().max(dim=1).values / g_rows).max())
    assert marg["G"] <= 1.0, ("G", marg["G"])
    # ---- the head ------------------------------------------------------------------------------------------------
    X = torch.cat(run_x)
    st = opt.slot(model.head.weight)
    assert st["step"] == OPT_STEP
    g_w, mw = check_fused_update("W", kind, hp, OPT_STEP, W0, *state0["W"], W, st["m"], st["v"] if kind != "sgd" else None,
                                 G.t() @ X, total * U * (G.abs().t() @ X.abs()))
    Xref = torch.cat(ref_x)
    bound = (g_rows @ Xref.abs()).unsqueeze(0) + total * U * (ref["G"].abs().t() @ Xref.abs())
    if ni:
        bound = bound + ref["G"][:ni].abs().t() @ (X[:ni] - ref["Z"]).abs()
    marg["W_grad_ref"] = ratio(g_w, ref["dW"], bound)
    assert marg["W_grad_ref"] <= 1.0, marg
    marg["W_grad_own"], marg["W"], marg["W_decay"] = mw["grad"], mw["W"], mw["decay_margin"]
    # ---- the adapter ---------------------------------------------------------------------------------------------
    stp = opt.slot(model.img_proj.weight)
    if ni:
        dZ = eng.dZ[:ni].double()
        marg["dZ_own"] = ratio(dZ, G[:ni] @ W0.double(), C * U * (G[:ni].abs() @ W0.double().abs()))
        dZb = g_rows[:ni].unsqueeze(1) * W0.double().abs().sum(0).unsqueeze(0) + C * U * (ref["G"][:ni].abs() @ W0.double().abs())
        marg["dZ_ref"] = ratio(dZ, ref["dZ"], dZb)
        assert marg["dZ_own"] <= 1.0 and marg["dZ_ref"] <= 1.0, marg
        assert stp["step"] == OPT_STEP
        Xi = xs[0].double()
        g_p, mp = check_fused_update("Wp", kind, hp, OPT_STEP, Wp0, *state0["Wp"], Wp, stp["m"],
                                     stp["v"] if kind != "sgd" else None, dZ.t() @ Xi, ni * U * (dZ.abs().t() @ Xi.abs()))
        marg["Wp_grad_ref"] = ratio(g_p, ref["dWp"], dZb.t() @ Xi.abs() + ni * U * (ref["dZ"].abs().t() @ Xi.abs()))
        assert marg["Wp_grad_ref"] <= 1.0, marg
        marg["Wp_grad_own"], marg["Wp"], marg["Wp_decay"] = mp["grad"], mp["W"], mp["decay_margin"]
    else:   # no image rows: the adapter and its state are not touched
        assert stp["step"] == OPT_STEP - 1
        assert torch.equal(Wp, Wp0) and torch.equal(stp["m"], state0["Wp"][0])
        if kind != "sgd":
            assert torch.equal(stp["v"], state0["Wp"][1])
    # ---- the temperatures ----------------------------------------------------------------------------------------
    if learnable:
        k = 0
        for name, n in (("img_scale", ni), ("txt_scale", nt)):
            prm, stt = getattr(model, name), opt.slot(getattr(model, name))
            if not n:
                assert torch.equal(prm.data, temps[name][0]) and stt["step"] == OPT_STEP - 1
                continue
            assert stt["step"] == OPT_STEP
            ds = torch.tensor(stats_rec(stats, k)["dscale"], dtype=torch.float64)
            want = apply_update(hp, temps[name][0].cpu(), ds, temps[name][1].cpu(),
                                temps[name][2].cpu() if temps[name][2] is not None else None, OPT_STEP)
            check_update(prm.data.cpu(), want[0], name)
            check_update(stt["m"].cpu(), want[1], name + " m")
            k += 1
    print(f"\n[adapter {shape} {kind} {'learnable' if learnable else 'fixed'}] " +
          ", ".join(f"{k} {v:.2e}" if v < 10 else f"{k} {v:.0f}x" for k, v in marg.items()))
