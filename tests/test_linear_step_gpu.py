"""The bf16 training step as its launcher (csrc/step.cu) puts it together, against the float64 reference of
tests/linear_step_ref.py.  Every test drives the C ABI directly (uml_linear_step / uml_linear_run with a hand-filled
uml_linear_step_args), so that each case picks one branch of the launcher explicitly:

* test_step_matches_the_float64_reference: one step per case - gather (X16 / labels32 byte-exact), G, the per-run
  statistics record, the gradient and, isolated from it, the optimizer update of W, m, v, the bf16 shadow and the
  learnable temperatures;
* test_run_is_bit_identical_to_a_chain_of_single_steps: the gather pipeline of uml_linear_run over operand buffers,
  idx_ready and call lengths against the same steps one uml_linear_step at a time;
* test_empty_run: nseg = 2 with one run of n == 0 on both precisions - stats[i] belongs to seg[i], an empty run's record
  is zero and its temperature is left untouched.

Bounds.  G: 6e-3 of max|G_ref|, as the exchange-forward tests.  Statistics: n exact, loss_mean 2e-4 relative, dscale 2e-3
relative, `correct` off by at most the number of near-tie rows.  Gradient: relative Frobenius error <= 4e-3 against the
float64 G_ref^T X16 and max error <= 1e-2 max|ref|: the kernel rounds G to bf16 once (unit roundoff 2^-9 ~ 2e-3) and
those roundings are independent, so their contribution to the Frobenius norm stays below it.  Update: rtol 2e-6 /
atol 2e-7 against the float64 rule applied to the kernel's own gradient, as test_optimizer_steps.
Observed on an NVIDIA B200 (the cfg3 case, 70144 + 3584 rows): gradient relative Frobenius error 1.6e-3, max error
1.9e-3 of max|ref|; largest W error of the update 0.04 of its bound.  Over all cases the largest were 2.4e-3 and 2.6e-3
(128 rows, chunk-sequential forward) and 0.04.
"""
import ctypes

import pytest
import torch

from linear_step_case import (DEV, OPT_STEP, Run, Workspace, call, check_stats, check_update, stats_rec, stream,
                              temp_state)
from linear_step_ref import Hyper, apply_update, forward_backward

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from uml_b200 import _lib


# ------------------------------------------------------------------------------------------ (a) one step vs float64
# runs: (rows, mode) with mode shadow = bf16 shadow bank + idx, fp32 = fp32 bank + idx, dense = idx NULL,
# label_idx = labels through label_idx; the text run (the second, or the only one of `text_only`) has loss weight 0.5
CASES = {
    "cfg3": dict(runs=[(70144, "shadow"), (3584, "shadow")], D=768, C=1000, kind="adamw", scales=(100.0, 100.0)),
    "fp32_banks": dict(runs=[(300, "fp32"), (212, "fp32")], D=256, C=1000, kind="adam"),
    "rows128": dict(runs=[(100, "shadow"), (28, "shadow")], D=512, C=397, kind="sgd"),
    "rows129": dict(runs=[(129, "shadow")], D=512, C=397, kind="adamw"),
    "text_only": dict(runs=[(1000, "shadow")], D=3200, C=1000, kind="adamw", text_only=True),
    "dense": dict(runs=[(640, "dense"), (384, "dense")], D=200, C=257, kind="adamw"),
    "label_idx": dict(runs=[(256, "label_idx"), (256, "label_idx")], D=768, C=1024, kind="adamw"),
    "temperatures": dict(runs=[(1500, "shadow"), (700, "shadow")], D=768, C=1000, kind="adamw", learnable=True),
    "temperatures_small": dict(runs=[(64, "shadow"), (40, "shadow")], D=256, C=100, kind="sgd", learnable=True),
    "shadow_stale": dict(runs=[(512, "shadow"), (512, "shadow")], D=768, C=1000, kind="adamw", w16_valid=0, max_splits=1),
    "gradient_only": dict(runs=[(2048, "shadow"), (512, "shadow")], D=768, C=1000, kind="adamw"),
}


def _make_runs(cfg, g):
    D, C = cfg["D"], cfg["C"]
    scales = cfg.get("scales", (30.0, 12.0))
    runs = []
    for k, (n, mode) in enumerate(cfg["runs"]):
        txt = k == 1 or cfg.get("text_only", False)
        bank_rows = n if mode == "dense" else n + n // 7 + 5
        rows = torch.randn(bank_rows, D, device=DEV, generator=g)
        labels = torch.randint(0, C, (bank_rows,), device=DEV, generator=g)
        idx = torch.randperm(bank_rows, device=DEV, generator=g)[:n] if mode != "dense" else None
        r = Run(n, rows, labels, idx, scale=scales[1] if txt else scales[0], loss_weight=0.5 if txt else 1.0)
        if mode == "shadow":
            r.rows16 = rows.to(torch.bfloat16)
        elif mode == "label_idx":
            # run 0: dense rows (an adapter's output) with bank labels; run 1: rows by idx, labels by other indices
            r.label_idx = torch.randint(0, bank_rows, (n,), device=DEV, generator=g)
            if k == 0:
                r.rows, r.idx = rows[:n].contiguous(), None
        if cfg.get("learnable"):
            r.temp = temp_state(r.scale, torch.Generator().manual_seed(k), cfg["kind"])
        runs.append(r)
    return runs


def _hyper(kind):
    return Hyper(kind, lr=2e-3, weight_decay=0.01 if kind != "adam" else 0.02).as_f32()


@pytest.mark.parametrize("case", list(CASES))
def test_step_matches_the_float64_reference(case):
    cfg = CASES[case]
    D, C, kind = cfg["D"], cfg["C"], cfg["kind"]
    g = torch.Generator(device=DEV).manual_seed(sum(n for n, _ in cfg["runs"]) + D + C)
    runs = _make_runs(cfg, g)
    total = sum(r.n for r in runs)
    W0 = torch.randn(C, D, device=DEV, generator=g)
    W0 /= W0.norm(dim=1, keepdim=True)
    hp = _hyper(kind)
    ws = Workspace(D, C, total)
    w16_valid, max_splits = cfg.get("w16_valid", 1), cfg.get("max_splits")
    temps0 = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in r.temp.items()} if r.temp else None for r in runs]

    def launch(W, m, v, **kw):
        for r, t0 in zip(runs, temps0):
            if t0:
                for key in ("value", "m", "v"):
                    if t0[key] is not None:
                        r.temp[key].copy_(t0[key])
        ws.W16.copy_(W.to(torch.bfloat16)) if w16_valid else ws.W16.fill_(float("nan"))
        ws.G.fill_(float("nan"))
        stats = torch.full((2, 4), float("nan"), device=DEV)
        a = ws.args(runs, W, m, v, hp, OPT_STEP, stats, w16_valid=w16_valid, max_splits=max_splits, **kw)
        call(_lib.load().uml_linear_step, ctypes.byref(a), stream())
        torch.cuda.synchronize()
        return stats

    # the reference on the step's bf16 operands (and the temperatures before the step)
    X16 = torch.cat([r.x16() for r in runs])
    ref = forward_backward(W0.to(torch.bfloat16), [r.ref_in(x) for r, x in zip(runs, X16.split([r.n for r in runs]))],
                           keep_g=True)
    # ---- gradient only (dW_out): W, m and v are not touched ------------------------------------------------------
    W, m, v = W0.clone(), torch.randn(C, D, device=DEV, generator=g), torch.rand(C, D, device=DEV, generator=g)
    Wc, mc, vc = W.clone(), m.clone(), v.clone()
    stats = launch(W, m, v, dW_out=ws.dW)
    grad = ws.dW.clone()
    assert torch.equal(W, Wc) and torch.equal(m, mc) and torch.equal(v, vc)
    assert torch.equal(ws.W16, W.to(torch.bfloat16))
    assert torch.equal(ws.X16[0][:total], X16)
    assert torch.equal(ws.labels32[0][:total], torch.cat([r.y() for r in runs]))
    G = ws.G[:total].float()
    assert bool((G[:, C:] == 0).all()), "G's padding columns must be zero"
    gmax = float(ref["G"].abs().max())
    assert float((G[:, :C].double() - ref["G"]).abs().max()) <= 6e-3 * gmax
    check_stats(stats, ref["stats"], case, dscale=bool(cfg.get("learnable")))
    dW_ref = ref["dW"]
    rel = float((grad.double() - dW_ref).norm() / dW_ref.norm())
    mx = float((grad.double() - dW_ref).abs().max()) / float(dW_ref.abs().max())
    print(f"\n[{case}] gradient: relative Frobenius error {rel:.2e} (bound 4e-3), max error {mx:.2e} of max|ref| (bound 1e-2)")
    assert rel <= 4e-3 and mx <= 1e-2, (rel, mx)

    def check_temps(where):
        for k, (r, t0) in enumerate(zip(runs, temps0)):
            if not t0:
                continue
            ds = torch.tensor(stats_rec(stats, k)["dscale"], dtype=torch.float64)
            want = apply_update(hp, t0["value"].cpu(), ds, t0["m"].cpu(), t0["v"].cpu() if t0["v"] is not None else None,
                                t0["step"])
            check_update(r.temp["value"].cpu(), want[0], where + " temperature")
            check_update(r.temp["m"].cpu(), want[1], where + " temperature m")
            if want[2] is not None:
                check_update(r.temp["v"].cpu(), want[2], where + " temperature v")

    check_temps("dW_out")
    # ---- fused: the update from a warm state (m != 0, v > 0), judged on the kernel's own gradient ----------------
    u = lambda lo, hi: torch.rand(C, D, device=DEV, generator=g) * (hi - lo) + lo
    m0 = grad * u(-1.0, 2.0)
    v0 = grad * grad * u(0.5, 2.0) + 1e-12 if kind != "sgd" else torch.zeros_like(grad)
    W, m, v = W0.clone(), m0.clone(), v0.clone()
    scratch = torch.full_like(grad, float("nan")) if kind == "sgd" else None
    stats_f = launch(W, m, v, dW_scratch=scratch)
    assert torch.equal(stats_f.view(torch.int32), stats.view(torch.int32)), "the same step twice: the same record"
    if scratch is not None:
        assert torch.equal(scratch, grad), "dW_scratch holds the gradient dW_out held"
    Ww, mw, vw = apply_update(hp, W0, grad, m0, v0 if kind != "sgd" else None, OPT_STEP)
    worst = check_update(W, Ww, "W")
    check_update(m, mw, "m")
    if kind != "sgd":
        check_update(v, vw, "v", atol=1e-12)
    assert torch.equal(ws.W16, W.to(torch.bfloat16)), "the bf16 shadow is the updated W"
    print(f"[{case}] update: largest W error {worst:.2f} of the bound (rtol 2e-6, atol 2e-7)")
    check_temps("fused")


# ------------------------------------------------------------------------------------------ (b) the run pipeline
P_D, P_C, P_STEPS = 256, 300, 12
P_ROWS = [(300, 200)] * (P_STEPS - 1) + [(170, 200)]       # the last batch of the epoch is short (image run)


@pytest.fixture(scope="module")
def pipeline_case():
    """Banks, per-step index batches and the result of the chain of single uml_linear_step calls."""
    g = torch.Generator(device=DEV).manual_seed(2024)
    banks = []
    for nb in (3000, 1500):
        rows = torch.randn(nb, P_D, device=DEV, generator=g)
        banks.append((rows, rows.to(torch.bfloat16), torch.randint(0, P_C, (nb,), device=DEV, generator=g)))
    idx = [[torch.randperm(banks[k][0].shape[0], device=DEV, generator=g)[:n] for k, n in enumerate(rn)] for rn in P_ROWS]
    W0 = torch.randn(P_C, P_D, device=DEV, generator=g)
    W0 /= W0.norm(dim=1, keepdim=True)
    lrs = [_hyper("adamw").lr * (1.0 - 0.05 * i) for i in range(P_STEPS)]
    case = dict(banks=banks, idx=idx, W0=W0, lrs=lrs, hp=_hyper("adamw"))
    # the chain: every step its own uml_linear_step
    W, m, v = W0.clone(), torch.zeros_like(W0), torch.zeros_like(W0)
    ws = Workspace(P_D, P_C, 500)
    ws.W16.copy_(W.to(torch.bfloat16))
    stats = torch.zeros((P_STEPS, 2, 4), device=DEV)
    before = []
    for i in range(P_STEPS):
        before.append(W.clone())
        hp = Hyper(**{**case["hp"].__dict__, "lr": lrs[i]})
        a = ws.args(_pipeline_runs(case, i), W, m, v, hp, i + 1, stats[i])
        call(_lib.load().uml_linear_step, ctypes.byref(a), stream())
    torch.cuda.synchronize()
    case["chain"] = dict(W=W, m=m, v=v, W16=ws.W16.clone(), stats=stats, before=before)
    return case


def _pipeline_runs(case, i):
    return [Run(len(ix), bank, lab, ix, rows16=b16, scale=s, loss_weight=w)
            for ix, (bank, b16, lab), s, w in zip(case["idx"][i], case["banks"], (30.0, 12.0), (1.0, 0.5))]


def test_chain_stats_match_the_float64_reference(pipeline_case):
    c = pipeline_case
    for i in range(P_STEPS):
        runs = _pipeline_runs(c, i)
        ref = forward_backward(c["chain"]["before"][i].to(torch.bfloat16), [r.ref_in(r.x16()) for r in runs], keep_g=False)
        check_stats(c["chain"]["stats"][i], ref["stats"], f"step {i}", dscale=False)


@pytest.mark.parametrize("n_buffers", [1, 2, 3])
@pytest.mark.parametrize("idx_ready", [False, True], ids=["no_idx_ready", "idx_ready"])
@pytest.mark.parametrize("per_call", [1, 2, 3, 6])
def test_run_is_bit_identical_to_a_chain_of_single_steps(pipeline_case, n_buffers, idx_ready, per_call):
    """Steps 0-5 in uml_linear_run calls of `per_call` steps (warm call boundaries in continuous mode), step 6 by
    uml_linear_step (the next run must start cold), steps 7-11 in calls again, the last one short."""
    c = pipeline_case
    lib = _lib.load()
    call(lib.uml_linear_run_reset)
    W, m, v = c["W0"].clone(), torch.zeros_like(c["W0"]), torch.zeros_like(c["W0"])
    ws = Workspace(P_D, P_C, 500, n_buffers=n_buffers)
    ws.W16.copy_(W.to(torch.bfloat16))
    stats = torch.full((P_STEPS, 2, 4), float("nan"), device=DEV)
    hp0 = c["hp"]
    ev = torch.cuda.Event()
    ev.record()   # every index batch is on the device already
    keep = []

    def run_calls(first, last):
        for lo in range(first, last, per_call):
            hi = min(lo + per_call, last)
            base = ws.args(_pipeline_runs(c, lo), W, m, v, hp0, lo + 1, stats[lo])
            bufs = [(x.data_ptr(), l.data_ptr()) for x, l in zip(ws.X16, ws.labels32)] + [(None, None)] * 3
            (base.X16_alt, base.labels32_alt), (base.X16_alt2, base.labels32_alt2) = bufs[1], bufs[2]
            base.idx_ready = ev.cuda_event if idx_ready else None
            steps = (_lib.RunStep * (hi - lo))()
            for j, i in enumerate(range(lo, hi)):
                s = steps[j]
                for k, ix in enumerate(c["idx"][i]):
                    s.idx[k], s.n[k], s.loss_weight[k] = ix.data_ptr(), len(ix), (1.0, 0.5)[k]
                s.lr, s.opt_step, s.stats = c["lrs"][i], i + 1, stats[i].data_ptr()
            keep.append(steps)
            call(lib.uml_linear_run, ctypes.byref(base), steps, hi - lo, stream())

    run_calls(0, 6)
    a = ws.args(_pipeline_runs(c, 6), W, m, v, Hyper(**{**hp0.__dict__, "lr": c["lrs"][6]}), 7, stats[6])
    call(lib.uml_linear_step, ctypes.byref(a), stream())
    run_calls(7, P_STEPS)
    torch.cuda.synchronize()
    ch = c["chain"]
    assert torch.equal(stats.view(torch.int32), ch["stats"].view(torch.int32)), "per-step statistics records"
    assert torch.equal(W, ch["W"]) and torch.equal(m, ch["m"]) and torch.equal(v, ch["v"])
    assert torch.equal(ws.W16, ch["W16"])


# ------------------------------------------------------------------------------------------ (c) empty runs
@pytest.mark.parametrize("precision", [0, 1], ids=["fp32", "bf16"])
@pytest.mark.parametrize("empty", [0, 1], ids=["seg0_empty", "seg1_empty"])
@pytest.mark.parametrize("learnable", [False, True], ids=["fixed", "learnable"])
@pytest.mark.parametrize("n_live", [100, 300])   # bf16: the chunk-sequential forward, then the exchange forward
def test_empty_run(precision, empty, learnable, n_live):
    """nseg = 2, one run with n == 0 (the last batch of an epoch can be empty for one modality): stats[i] belongs to
    seg[i], the empty run's record is {0, 0, 0, 0}, the live run's temperature steps with its own gradient and the
    empty run's temperature, m and v are left untouched, as torch.optim skips a parameter without a gradient."""
    D, Cn = 128, 200
    g = torch.Generator(device=DEV).manual_seed(n_live + 10 * empty + 100 * precision)
    runs = []
    for k in range(2):
        rows = torch.randn(400, D, device=DEV, generator=g)
        n = 0 if k == empty else n_live
        r = Run(n, rows, torch.randint(0, Cn, (400,), device=DEV, generator=g),
                torch.randperm(400, device=DEV, generator=g)[:max(n, 1)], rows16=rows.to(torch.bfloat16) if precision else None,
                scale=(20.0, 8.0)[k], loss_weight=(1.0, 0.5)[k])
        if learnable:
            r.temp = temp_state(r.scale, torch.Generator().manual_seed(k + 7), "adamw")
        runs.append(r)
    temps0 = [{key: (val.clone() if torch.is_tensor(val) else val) for key, val in r.temp.items()} if learnable else None
              for r in runs]
    W = torch.randn(Cn, D, device=DEV, generator=g)
    W /= W.norm(dim=1, keepdim=True)
    W0 = W.clone()
    m, v = torch.zeros_like(W), torch.zeros_like(W)
    hp = _hyper("adamw")
    ws = Workspace(D, Cn, n_live, precision=precision)
    ws.W16.copy_(W.to(torch.bfloat16))
    stats = torch.empty((2, 4), device=DEV)
    stats.view(torch.int32).fill_(0x7f7f7f7f)  # not a record anyone wrote
    live = 1 - empty
    r = runs[live]
    x = r.x16() if precision else r.rows[r.idx[:r.n]]
    ref = forward_backward(W0, [r.ref_in(x)], bf16_operands=bool(precision), keep_g=False)
    a = ws.args(runs, W, m, v, hp, 1, stats, precision=precision)
    call(_lib.load().uml_linear_step, ctypes.byref(a), stream())
    torch.cuda.synchronize()
    assert bool((stats[empty].view(torch.int32) == 0).all()), ("the empty run's record", stats[empty])
    got = stats_rec(stats, live)
    check_stats(stats[live:live + 1], ref["stats"], "live run", dscale=learnable or precision == 0)
    if learnable:
        t0 = temps0[live]
        want = apply_update(hp, t0["value"].cpu(), torch.tensor(got["dscale"], dtype=torch.float64), t0["m"].cpu(),
                            t0["v"].cpu(), t0["step"])
        check_update(runs[live].temp["value"].cpu(), want[0], "live temperature")
        check_update(runs[live].temp["m"].cpu(), want[1], "live temperature m")
        check_update(runs[live].temp["v"].cpu(), want[2], "live temperature v")
        for key in ("value", "m", "v"):
            assert torch.equal(runs[empty].temp[key], temps0[empty][key]), ("the empty run's temperature " + key)
