"""Per-step gradient diagnostics of single runs (--grad-diagnostics-every-step: uml_linear_run_diag and
uml_linear_grad_diag): every logged step against a float64 reference recomputed from the weights held before that step,
on the exact fused and separate-launch steps, the bf16 tensor-core step and adapter heads on both paths; training
bit-identical with and without them; finetune.train and main() logging them at every step."""
import copy
import math

import pytest
import torch

from linear_step_ref import RunIn, bf16_round, forward_backward

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

if torch.cuda.is_available():
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, ops
    from uml_b200 import finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader, FeatureBank
    from uml_b200.engine.models.head import UML, UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler

KEYS = ("train/grad_direction_sim", "train/img_grad_norm", "train/txt_grad_norm", "train/grad_agreement_rate")
LOGIT = math.log(10.0)

# Exact path: the bounds of test_kernels_gpu.py::test_grad_diagnostics_match_autograd (3xTF32 products, fp32 sums).
# bf16 path: the reference takes the same bf16-rounded rows, weights (and adapter output Z) but keeps G in float64,
# while the step stores G in bf16 (relative rounding 2^-9 per element) before the dW GEMMs; a gradient element is a sum
# of such terms, so its relative error stays within ~2^-8 and the norms and the cosine within 1e-2; elements near zero
# may flip sign, so the agreement rate is held to 2e-2.
TOL = {"fp32": dict(norm=1e-4, cos=1e-4, agree=2e-3), "bf16": dict(norm=1e-2, cos=1e-2, agree=2e-2)}


def _case(kind, D, C, bs, optim, alpha, precision, modality="crossmodal", Dv=0, n_img=None, n_txt=None, seed=0):
    """Model, loaders and optimizer of one single run; the banks give a ragged last batch (on the bf16 path one that
    still has more than BF16_MIN_ROWS rows, so that the same run takes the same path with precision "auto")."""
    g = torch.Generator().manual_seed(seed + D + C + bs[0])
    has_img, has_txt = modality != "text", modality != "image"
    width = Dv if kind == "adapter" else D
    extra = (5, 9) if precision == "fp32" else (1100, 1100)
    n_img = n_img or 2 * bs[0] + extra[0]
    n_txt = n_txt or 2 * bs[1] + extra[1]
    xi, yi = torch.randn(n_img, width, generator=g), torch.randint(0, C, (n_img,), generator=g)
    xt, yt = torch.randn(n_txt, D, generator=g), torch.randint(0, C, (n_txt,), generator=g)
    xv, yv = torch.randn(50, width, generator=g), torch.randint(0, C, (50,), generator=g)
    torch.manual_seed(seed + 5)
    if kind == "adapter":
        m = UML(f"synthetic:{Dv}", D, C, learnable_temp=True)
        m.load_state_dict({"head.weight": 0.05 * torch.randn(C, D, generator=g), "img_scale": torch.tensor(1.5),
                           "txt_scale": torch.tensor(2.0), "img_proj.weight": torch.randn(D, Dv, generator=g) / Dv ** 0.5})
    else:
        m = UMLClip(f"synthetic:{D}", C, logit_scale_init=LOGIT)
        m.load_state_dict({"head.weight": 0.05 * torch.randn(C, D, generator=g)})
    m.precision = precision
    m.to(DEV)
    return dict(model=m, banks=(FeatureBank(xi, yi, DEV), FeatureBank(xt, yt, DEV), FeatureBank(xv, yv, DEV)),
                bs=bs, optim=optim, alpha=alpha, has_img=has_img, has_txt=has_txt, x=(xi, yi, xt, yt), precision=precision)


def _train(c, diag, record=True, max_iters=6, eval_freq=3, patience=20, logger=None, args=None, shuffle=True,
           stats_to_host="eval"):
    m = copy.deepcopy(c["model"])
    opt = build_optimizer(m.parameters(), c["optim"], 5e-3, 0.01)
    sch = build_lr_scheduler(opt, "cosine", 2, 40, warmup_type="linear", warmup_lr=1e-4)
    rng = torch.Generator().manual_seed(3)
    ib, tb, vb = c["banks"]
    il = BankLoader(ib, c["bs"][0], shuffle=shuffle, rng=rng) if c["has_img"] else None
    tl = BankLoader(tb, c["bs"][1], shuffle=shuffle, rng=rng) if c["has_txt"] else None
    vl = BankLoader(vb, 25, shuffle=False, rng=rng)
    tr = {"record_weights": record, "indices": shuffle}  # (sequential batches carry no host indices: see _seq_idx)
    if diag:
        tr["grad_diagnostics"] = diag
    f0 = _lib.load().uml_head_step_fused_count()
    ft.train(m, il, tl, vl, None, opt, sch, device=DEV, max_iters=max_iters, alpha=c["alpha"], eval_freq=eval_freq,
             patience=patience, trace=tr, logger=logger, args=args, stats_to_host=stats_to_host)
    tr["fused_steps"] = (_lib.load().uml_head_step_fused_count() - f0) & 0x7fffffff
    tr["opt_state"] = {k: v.detach().cpu().clone() for k, v in opt.slot(m.head.weight).items() if torch.is_tensor(v)}
    return tr


def _seq_idx(n_bank, bs, step):
    """Rows of step `step` of a sequential loader (shuffle=False, the last batch of an epoch short)."""
    per_epoch = -(-n_bank // bs)
    lo = (step % per_epoch) * bs
    return torch.arange(lo, min(lo + bs, n_bank))


def _ref(c, sd, ii, ti):
    """float64 (dot, |A|^2, |B|^2, agreements) of one step at the state dict `sd` held before it, and the resolution of
    the step's own G: its entries carry the fp32 rounding of softmax - onehot (2^-24 absolute, times scale / rows), which
    no later arithmetic can undo.  That bounds each gradient element's error by fl = 2^-23 * scale * max|x|; the norms
    by fl * sqrt(C D); elements with |A| or |B| below fl have no reliable sign."""
    m = copy.deepcopy(c["model"]).cpu()
    m.load_state_dict(sd)
    si, st = (float(s) for s in m.scales())
    xi, yi, xt, yt = c["x"]
    bf = c["precision"] == "bf16"
    W = m.head.weight.detach()
    grads, fls = [], []
    for x, y, s, idx, img in ((xi, yi, si, ii, True), (xt, yt, st, ti, False)):
        if idx is None or len(idx) == 0:
            grads.append(torch.zeros(W.shape, dtype=torch.float64))
            fls.append(0.0)
            continue
        x = x[idx]
        if img and m.img_proj is not None:
            Wp = m.img_proj.weight.detach()
            x = bf16_round(bf16_round(x) @ bf16_round(Wp).t()) if bf else x.double() @ Wp.double().t()
        grads.append(forward_backward(W, [RunIn(x, y[idx], s, 1.0)], bf16_operands=bf, keep_g=False)["dW"])
        fls.append(2.0 ** -23 * abs(s) * float(x.double().abs().max()))
    A, B = grads
    amb = int(((A.abs() <= fls[0]) | (B.abs() <= fls[1])).sum())
    sums = float((A * B).sum()), float((A * A).sum()), float((B * B).sum()), int((torch.sign(A) == torch.sign(B)).sum())
    return sums, fls, amb


def _check_against_reference(c, tr):
    numel = c["model"].head.weight.numel()
    tol = TOL[c["precision"]]
    steps = len(tr["stats"])
    assert [s for s, _ in tr["grad_diag"]] == list(range(steps))
    states = [c["model"].state_dict()] + tr["weights"]
    seq = "img_idx" not in tr and "txt_idx" not in tr
    for i, (step, d) in enumerate(tr["grad_diag"]):
        if seq:
            ii = _seq_idx(len(c["x"][0]), c["bs"][0], i) if c["has_img"] else None
            ti = _seq_idx(len(c["x"][2]), c["bs"][1], i) if c["has_txt"] else None
        else:
            ii = tr["img_idx"][i] if c["has_img"] else None
            ti = tr["txt_idx"][i] if c["has_txt"] else None
        sd = {k: v.detach().cpu() for k, v in states[i].items()}
        sums, fls, amb = _ref(c, sd, ii, ti)
        ref = ops.grad_diag_record(*sums, numel, c["has_img"] and c["has_txt"])
        floor = [f * math.sqrt(numel) for f in fls]
        for key, f in zip(KEYS[1:3], floor):
            assert abs(d[key] - ref[key]) <= tol["norm"] * ref[key] + f, (step, key, d, ref, f)
        ni, nt = ref[KEYS[1]], ref[KEYS[2]]
        cos_floor = (floor[0] / ni if ni else 0.0) + (floor[1] / nt if nt else 0.0)
        assert abs(d[KEYS[0]] - ref[KEYS[0]]) <= tol["cos"] + cos_floor, (step, d, ref, cos_floor)
        assert abs(d[KEYS[3]] - ref[KEYS[3]]) <= tol["agree"] + amb / numel, (step, d, ref, amb)


def _check_bit_identical(a, b):
    assert len(a["weights"]) == len(b["weights"])
    for wa, wb in zip(a["weights"], b["weights"]):
        for k in wa:
            assert torch.equal(wa[k], wb[k]), k
    for k in a["opt_state"]:
        assert torch.equal(a["opt_state"][k], b["opt_state"][k]), k
    assert a["stats"] == b["stats"]


CASES = [
    # kind, D, C, (bs img, bs txt), optimizer, alpha, precision, modality, Dv
    ("linear", 40, 10, (32, 32), "adamw", 1.5, "fp32", "crossmodal", 0),
    ("linear", 512, 1000, (32, 32), "sgd", 0.2, "fp32", "crossmodal", 0),
    ("linear", 512, 1000, (256, 256), "adamw", 0.2, "fp32", "crossmodal", 0),   # separate exact launches
    ("linear", 40, 10, (32, 32), "sgd", 1.5, "fp32", "image", 0),
    ("linear", 40, 10, (32, 32), "adamw", 0.2, "fp32", "text", 0),
    ("linear", 256, 300, (1536, 512), "adamw", 0.2, "bf16", "crossmodal", 0),   # ragged last batch: 1100 + 1100 rows
    ("linear", 256, 300, (1536, 512), "sgd", 1.5, "bf16", "crossmodal", 0),
    ("linear", 256, 300, (1536, 1536), "adamw", 1.5, "bf16", "text", 0),
    ("adapter", 40, 10, (32, 32), "adamw", 0.2, "fp32", "crossmodal", 24),
    ("adapter", 3200, 1000, (32, 32), "sgd", 1.5, "fp32", "crossmodal", 1536),
    ("adapter", 40, 10, (64, 64), "sgd", 1.5, "fp32", "crossmodal", 24),
    ("adapter", 40, 10, (32, 32), "adamw", 1.5, "fp32", "image", 24),
    ("adapter", 40, 10, (1024, 1024), "sgd", 1.5, "bf16", "crossmodal", 24),
    ("adapter", 3200, 1000, (1024, 1024), "adamw", 0.2, "bf16", "crossmodal", 1536),
]


@pytest.mark.parametrize("kind,D,C,bs,optim,alpha,precision,modality,Dv", CASES,
                         ids=[f"{k}-{D}x{C}-{b[0]}+{b[1]}-{o}-a{a}-{p}-{mo}" for k, D, C, b, o, a, p, mo, _ in CASES])
def test_every_step_matches_float64_and_training_is_bit_identical(kind, D, C, bs, optim, alpha, precision, modality, Dv):
    c = _case(kind, D, C, bs, optim, alpha, precision, modality, Dv)
    on = _train(c, "step")
    off = _train(c, None)
    _check_bit_identical(on, off)
    _check_against_reference(c, on)
    if kind == "linear" and precision == "fp32":  # the fused cooperative step takes the reference's batch sizes
        steps = len(on["stats"])    # (and the short last batches of an epoch); 256 + 256 rows take the separate launches
        assert on["fused_steps"] == steps if bs[0] <= 32 else 0 < steps - on["fused_steps"] < steps, on["fused_steps"]
    # chunks of several steps through uml_linear_run_diag (on the bf16 path with the gather pipeline running through them)
    # give the same figures
    chunked = _train(c, "step", record=False)
    assert chunked["grad_diag"] == on["grad_diag"]
    assert chunked["stats"] == on["stats"]


def test_train_logs_every_step_across_evaluations_and_an_early_stop():
    c = _case("linear", 40, 10, (16, 16), "adamw", 0.5, "fp32", n_img=70, n_txt=60)

    class Logger:
        def __init__(self):
            self.recs = []

        def log(self, d):
            self.recs.append(dict(d))

    lg = Logger()
    tr = _train(c, "step", record=False, max_iters=40, eval_freq=4, patience=1, logger=lg)
    n = len(tr["stats"])
    assert [s for s, _ in tr["grad_diag"]] == list(range(n))
    logged = [r for r in lg.recs if "train/image_loss" in r]
    assert len(logged) == n
    for r, (_, d) in zip(logged, tr["grad_diag"]):
        assert all(r[k] == d[k] for k in KEYS)
    # the same run with record_weights (one step per chunk) gives the same figures, checked against float64
    ref = _train(c, "step", record=True, max_iters=n, eval_freq=4, patience=40)
    assert ref["grad_diag"] == tr["grad_diag"]
    _check_against_reference(c, ref)
    # --grad-diagnostics alone: evaluation cadence only, no probes in the per-step records
    lg2 = Logger()
    tr2 = _train(c, True, record=False, max_iters=12, eval_freq=4, logger=lg2)
    assert [s for s, _ in tr2["grad_diag"]] == [0, 4, 8]
    assert all(not any(k in r for k in KEYS) for r in lg2.recs if "train/image_loss" in r)


def test_fallback_to_evaluation_cadence_for_alpha_zero(capsys):
    c = _case("linear", 64, 10, (16, 16), "adamw", 0.0, "fp32")
    tr = _train(c, "step", record=False, max_iters=7, eval_freq=3)
    assert "alpha > 0" in capsys.readouterr().out
    assert [s for s, _ in tr["grad_diag"]] == [0, 3, 6]


def test_main_single_run_logs_gradient_probes_every_step(tmp_path, monkeypatch):
    from oracle.synth import synth_banks
    from uml_b200 import features as F
    from uml_b200.engine.config import parser
    from uml_b200.engine.optimizer.default import HYPER_DICT
    C, D = 20, 64
    xi, yi, xt, yt, xv, yv = synth_banks(3, C, D, D, 16 * C, 6, 4 * C)
    fdir = str(tmp_path / "features")
    lab2cname = {c: f"class_{c}" for c in range(C)}
    F.write_text_bank(F.text_outdir(fdir, "ViT-B/16", "synthset", "cupl"), xt, yt, lab2cname=lab2cname)
    F.write_image_bank(F.img_outdir(fdir, "ViT-B/16", "synthset", "crop", 16, 1, "train"), train=(xi, yi), val=(xv, yv),
                       lab2cname=lab2cname)
    F.write_image_bank(F.img_outdir(fdir, "ViT-B/16", "synthset", "crop", 16, 1, "test"), test=(xv, yv), lab2cname=lab2cname)
    monkeypatch.setitem(HYPER_DICT, "unit_test_diag1", dict(HYPER_DICT["clip_linear"], lr=[1e-3], weight_decay=[0.0],
                                                              max_iter=[30], patience=[50]))
    loggers = []

    class Logger:
        def __init__(self):
            self.recs = []
            loggers.append(self)

        def log(self, d):
            self.recs.append(dict(d))

    monkeypatch.setattr(ft, "setup_wandb_logger", lambda hp, args: Logger())
    args = parser.parse_args(["--dataset", "synthset", "--train-shot", "16", "--seed", "1", "--clip-encoder", "ViT-B/16",
                              "--modality", "crossmodal", "--text_type", "cupl", "--hyperparams", "unit_test_diag1",
                              "--alpha", "0.5", "--feature_dir", fdir, "--result_dir", str(tmp_path / "exp"),
                              "--num-workers", "0", "--grad-diagnostics-every-step"])
    ft.main(args)
    assert len(loggers) == 1
    steps = [r for r in loggers[0].recs if "train/image_loss" in r]
    assert len(steps) == 30
    for r in steps:
        assert all(key in r and math.isfinite(r[key]) for key in KEYS), r
        assert -1.0 <= r[KEYS[0]] <= 1.0 and 0.0 <= r[KEYS[3]] <= 1.0


@pytest.mark.parametrize("precision,bs", [("fp32", (32, 32)), ("bf16", (1536, 512))])
def test_host_ring_and_single_step_calls(precision, bs):
    """stats_to_host="step" (the probes travel in the same pinned-ring copy as the losses) and sequential batches (dense
    rows: every step goes through uml_linear_step, then uml_linear_grad_diag) give the figures of the default run."""
    c = _case("linear", 256, 300, bs, "adamw", 0.5, precision)
    ref = _train(c, "step")
    ring = _train(c, "step", record=False, stats_to_host="step")
    assert ring["grad_diag"] == ref["grad_diag"] and ring["stats"] == ref["stats"]
    dense = _train(c, "step", shuffle=False)
    _check_bit_identical(dense, _train(c, None, shuffle=False))
    _check_against_reference(c, dense)
