"""Per-step gradient diagnostics of batched sweep groups (uml_sweep_run_diag, csrc/sweep.cu): the four sums of every
running head against a float64 reference taken at the weights held before each step, bit-identical training with and
without them, slot and neighbour independence, finetune.train_group's per-step records and main() end to end."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

if torch.cuda.is_available():
    import uml_b200  # noqa: F401
    from uml_b200 import finetune as ft
    from uml_b200 import ops
    from uml_b200.engine import sweep as sweep_mod
    from uml_b200.engine.datasets.utils import BankLoader, FeatureBank
    from uml_b200.engine.models.head import UML, UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler

KEYS = ("train/grad_direction_sim", "train/img_grad_norm", "train/txt_grad_norm", "train/grad_agreement_rate")
LOGIT = math.log(10.0)


def _snap(group, k):
    """Head k's weights, adapter and temperatures as float64 CPU tensors (what the next step starts from)."""
    C, D = group.C, group.D
    W = group.W[k, :C * D].view(C, D).double().cpu()
    Dv = getattr(group, "Dv", 0)
    Wp = group.Wp[k, :D * Dv].view(D, Dv).double().cpu() if Dv else None
    if getattr(group, "learnable", False):
        s = [float(x) for x in group.T[k].tolist()]
    else:
        s = [float(x) for x in group.models[k].scales()]
    return W, Wp, s


def _ref_sums(W, Wp, s, xi, yi, xt, yt):
    """float64: A = d image_loss / dW, B = d text_loss / dW (plain mean CEs) -> dot, |A|^2, |B|^2, sign agreement, and
    the number of elements whose sign is ambiguous at fp32 accuracy (|A| or |B| below 1e-5 of its maximum)."""
    A = torch.zeros_like(W)
    B = torch.zeros_like(W)
    for x, y, sc, out in ((xi, yi, s[0], A), (xt, yt, s[1], B)):
        if x is None or len(x) == 0:
            continue
        x = x.double()
        if out is A and Wp is not None:
            x = x @ Wp.T
        p = torch.softmax(x @ W.T * sc, 1)
        p[torch.arange(len(y)), y] -= 1.0
        out += (p * sc / len(y)).T @ x
    agree = int((torch.sign(A) == torch.sign(B)).sum())
    amb = int(((A.abs() < 1e-5 * A.abs().max()) | (B.abs() < 1e-5 * B.abs().max())).sum())
    return float((A * B).sum()), float((A * A).sum()), float((B * B).sum()), agree, amb


def _check(got, ref, numel, both, where):
    dot, aa, bb, agree, amb = ref
    g = [float(x) for x in got]
    assert abs(g[1] - aa) <= 1e-4 * aa + 1e-30, (where, g, ref)
    assert abs(g[2] - bb) <= 1e-4 * bb + 1e-30, (where, g, ref)
    assert abs(g[0] - dot) <= 1e-4 * math.sqrt(aa * bb) + 1e-30, (where, g, ref)
    assert abs(g[3] - agree) <= amb, (where, g, ref)
    r_got = ops.grad_diag_record(*g, numel, both)
    r_ref = ops.grad_diag_record(dot, aa, bb, agree, numel, both)
    assert abs(r_got[KEYS[0]] - r_ref[KEYS[0]]) <= 1e-5, (where, r_got, r_ref)


def _case(kind, Dv, D, C, optim, modality, bs, alphas=(0.2, 1.0, 1.5, 0.2), diag=True, seed=0, srcs=None):
    """A group of len(alphas) heads, banks for three steps with a ragged last one.  Slot k holds source head srcs[k]
    (weights, temperatures, lr, weight decay and permutations are a function of the source head only); by default
    slot k holds head k, except that the last slot is a twin of head 0."""
    adapter = kind == "adapter"
    g = torch.Generator().manual_seed(seed + Dv + D + C)
    n_img, n_txt = 2 * bs + 5, 2 * bs + 9
    has_img, has_txt = modality != "text", modality != "image"
    width = Dv if adapter else D
    xi, yi = torch.randn(n_img, width, generator=g), torch.randint(0, C, (n_img,), generator=g)
    xt, yt = torch.randn(n_txt, D, generator=g), torch.randint(0, C, (n_txt,), generator=g)
    ib, tb = FeatureBank(xi, yi, DEV), FeatureBank(xt, yt, DEV)
    lrs0 = [1e-3, 2e-3, 5e-3, 1e-3]
    wds = [0.01, 0.0, 0.1, 0.01]
    models, opts = [], []
    K = len(alphas)
    srcs = list(srcs) if srcs is not None else list(range(K - 1)) + [0]
    for k in range(K):
        src = srcs[k]
        gk = torch.Generator().manual_seed(100 + src + seed)
        if adapter:
            m = UML(f"synthetic:{Dv}", D, C, learnable_temp=True)
            m.load_state_dict({"head.weight": 0.05 * torch.randn(C, D, generator=gk), "img_scale": torch.tensor(1.0 + 0.5 * src),
                               "txt_scale": torch.tensor(2.0 - 0.25 * src),
                               "img_proj.weight": torch.randn(D, Dv, generator=gk) / Dv ** 0.5})
        else:
            m = UMLClip(f"synthetic:{D}", C, logit_scale_init=LOGIT)
            m.load_state_dict({"head.weight": 0.05 * torch.randn(C, D, generator=gk)})
        m.to(DEV)
        models.append(m)
        opts.append(build_optimizer(m.parameters(), optim, lrs0[src % 4], wds[src % 4]))
    cls = sweep_mod.AdapterHeadGroup if adapter else sweep_mod.HeadGroup
    group = cls(models, opts, ib if has_img else None, tb if has_txt else None, bs if has_img else 0,
                bs if has_txt else 0, DEV, log_slots=8, grad_diagnostics=diag)
    pi = [torch.randperm(n_img, generator=torch.Generator().manual_seed(7 + src + seed)) for src in srcs]
    pt = [torch.randperm(n_txt, generator=torch.Generator().manual_seed(9 + src + seed)) for src in srcs]
    rows = [(min(bs, n_img - s * bs) if has_img else 0, min(bs, n_txt - s * bs) if has_txt else 0) for s in range(3)]
    lrs = [[lrs0[src % 4] * (1.0 - 0.1 * s) for src in srcs] for s in range(3)]
    return dict(group=group, xi=xi, yi=yi, xt=xt, yt=yt, pi=pi, pt=pt, rows=rows, lrs=lrs, alphas=list(alphas),
                has_img=has_img, has_txt=has_txt)


def _perms(c):
    return ([p.to(DEV) for p in c["pi"]] if c["has_img"] else None, [p.to(DEV) for p in c["pt"]] if c["has_txt"] else None)


CASES = [
    ("linear", 0, 40, 10, "adamw", "crossmodal", 32),
    ("linear", 0, 512, 1000, "sgd", "crossmodal", 32),
    ("linear", 0, 40, 10, "adamw", "image", 32),
    ("linear", 0, 40, 10, "sgd", "text", 32),
    ("linear", 0, 512, 1000, "adamw", "crossmodal", 48),  # 96 rows per step: two k-tiles, the FFMA dW path
    ("adapter", 24, 40, 10, "adamw", "crossmodal", 32),
    ("adapter", 24, 40, 10, "sgd", "image", 32),
    ("adapter", 1536, 3200, 1000, "adamw", "crossmodal", 32),
]


@pytest.mark.parametrize("kind,Dv,D,C,optim,modality,bs", CASES)
def test_diagnostics_match_float64_reference_per_step(kind, Dv, D, C, optim, modality, bs):
    """One step per call; before each, the weights are snapshotted and the reference recomputes G in float64 from them.
    Head 1 is masked (its log rows stay untouched); head 3 is a twin of head 0 and gives bit-identical figures."""
    c = _case(kind, Dv, D, C, optim, modality, bs)
    group, K = c["group"], c["group"].K
    active = [True, False, True, True]
    pimg, ptxt = _perms(c)
    pos_i = pos_t = 0
    numel = C * D
    for s, (n_i, n_t) in enumerate(c["rows"]):
        snaps = [_snap(group, k) for k in range(K)]
        group.run(pimg, ptxt, pos_i, pos_t, [(n_i, n_t)], [c["lrs"][s]], c["alphas"], active, slot0=s)
        torch.cuda.synchronize()
        raw = group.diag_log[s].cpu()
        log = group.read_log([s], c["has_img"], c["has_txt"])
        assert float(raw[1].abs().sum()) == 0.0, "a masked head's log rows are never written"
        for k in range(K):
            if not active[k]:
                continue
            ii = c["pi"][k][pos_i:pos_i + n_i]
            ti = c["pt"][k][pos_t:pos_t + n_t]
            ref = _ref_sums(*snaps[k], c["xi"][ii] if n_i else None, c["yi"][ii], c["xt"][ti] if n_t else None, c["yt"][ti])
            _check(raw[k], ref, numel, n_i > 0 and n_t > 0, (k, s))
            want = ops.grad_diag_record(*[float(x) for x in raw[k]], numel, n_i > 0 and n_t > 0)
            assert log["grad_diag"][0][k] == want
        assert torch.equal(raw[0], raw[K - 1]), s
        pos_i += n_i
        pos_t += n_t


@pytest.mark.parametrize("kind,Dv,D,C,optim,modality,bs", [CASES[1], CASES[4], CASES[5], CASES[7]])
def test_training_is_bit_identical_with_and_without_diagnostics(kind, Dv, D, C, optim, modality, bs):
    out = []
    for diag in (False, True):
        c = _case(kind, Dv, D, C, optim, modality, bs, diag=diag)
        group = c["group"]
        pimg, ptxt = _perms(c)
        group.run(pimg, ptxt, 0, 0, c["rows"], c["lrs"], c["alphas"], [True, False, True, True], slot0=0)
        torch.cuda.synchronize()
        names = [n for n in ("W", "m", "v", "Wp", "mp", "vp", "T", "Tm", "Tv", "stats_log") if getattr(group, n, None) is not None]
        out.append({n: getattr(group, n).clone() for n in names})
    assert out[0].keys() == out[1].keys()
    for n in out[0]:
        assert torch.equal(out[0][n], out[1][n]), n


@pytest.mark.parametrize("kind,Dv,D,C,optim,modality,bs", [CASES[1], CASES[5]])
def test_diagnostics_do_not_depend_on_slot_or_neighbours(kind, Dv, D, C, optim, modality, bs):
    """Head 0 in slot 0 of a four-head group and its twin in slot 3; then heads 2 and 0 of that group in a two-head group,
    head 2 in slot 0 and head 0 in slot 1 next to a different neighbour: every head's figures are bit-identical wherever
    it sits, at every step."""
    a = _case(kind, Dv, D, C, optim, modality, bs)
    b = _case(kind, Dv, D, C, optim, modality, bs, alphas=(1.5, 0.2), srcs=(2, 0))
    for c in (a, b):
        pimg, ptxt = _perms(c)
        c["group"].run(pimg, ptxt, 0, 0, c["rows"], c["lrs"], c["alphas"], [True] * c["group"].K, slot0=0)
    torch.cuda.synchronize()
    da, db = a["group"].diag_log[:3].cpu(), b["group"].diag_log[:3].cpu()
    assert torch.equal(da[:, 0], da[:, 3])
    assert torch.equal(da[:, 0], db[:, 1])
    assert torch.equal(da[:, 2], db[:, 0])
    assert not torch.equal(da[:, 0], da[:, 2])


def _recording(cls):
    """The group class with run() split into single steps and the weights snapshotted before each."""
    class Recording(cls):
        def run(self, perms_img, perms_txt, pos_img, pos_txt, rows, lrs, alphas, active, slot0):
            if not hasattr(self, "snaps"):
                self.snaps = []
            for j, (n_i, n_t) in enumerate(rows):
                self.snaps.append(dict(step=slot0 + j, active=list(active), rows=(n_i, n_t),
                                       w=[_snap(self, k) for k in range(self.K)],
                                       ii=[perms_img[k][pos_img:pos_img + n_i].cpu() if n_i else None for k in range(self.K)],
                                       ti=[perms_txt[k][pos_txt:pos_txt + n_t].cpu() if n_t else None for k in range(self.K)]))
                super().run(perms_img, perms_txt, pos_img, pos_txt, [(n_i, n_t)], [lrs[j]], alphas, active, slot0 + j)
                pos_img += n_i
                pos_txt += n_t
    return Recording


@pytest.mark.parametrize("adapter", [False, True])
def test_train_group_logs_every_step_of_every_running_head(monkeypatch, adapter):
    monkeypatch.setattr(sweep_mod, "HeadGroup", _recording(sweep_mod.HeadGroup))
    monkeypatch.setattr(sweep_mod, "AdapterHeadGroup", _recording(sweep_mod.AdapterHeadGroup))
    C, D, Dv, bs = 10, 40, 24, 16
    g = torch.Generator().manual_seed(11)
    width = Dv if adapter else D
    xi, yi = torch.randn(200, width, generator=g), torch.randint(0, C, (200,), generator=g)
    xt, yt = torch.randn(150, D, generator=g), torch.randint(0, C, (150,), generator=g)
    xv, yv = torch.randn(60, width, generator=g), torch.randint(0, C, (60,), generator=g)
    ib, tb, vb = FeatureBank(xi, yi, DEV), FeatureBank(xt, yt, DEV), FeatureBank(xv, yv, DEV)
    heads = [(1e-2, 0.0, 0.5, 20), (1e-3, 0.01, 1.0, 20), (5e-2, 0.0, 0.2, 1)]  # lr, wd, alpha, patience (head 2 stops early)
    models, opts, schs, ils, tls, vls, traces, loggers = [], [], [], [], [], [], [], []

    class Logger:
        def __init__(self):
            self.recs = []

        def log(self, d):
            self.recs.append(dict(d))

    for k, (lr, wd, _, _) in enumerate(heads):
        torch.manual_seed(20 + k)
        m = UML(f"synthetic:{Dv}", D, C, learnable_temp=True) if adapter else UMLClip(f"synthetic:{D}", C, logit_scale_init=LOGIT)
        m.precision = "fp32"
        m.to(DEV)
        opt = build_optimizer(m.parameters(), "adamw", lr, wd)
        rng = torch.Generator().manual_seed(30 + k)
        models.append(m)
        opts.append(opt)
        schs.append(build_lr_scheduler(opt, "cosine", 5, 60, warmup_type="linear", warmup_lr=1e-5))
        ils.append(BankLoader(ib, bs, shuffle=True, rng=rng))
        tls.append(BankLoader(tb, bs, shuffle=True, rng=rng))
        vls.append(BankLoader(vb, bs, shuffle=False, rng=rng))
        traces.append({"grad_diagnostics": True})
        loggers.append(Logger())
    ft.train_group(models, ils, tls, vls, None, opts, schs, device=DEV, max_iters=40, alphas=[h[2] for h in heads],
                   eval_freq=5, patience=[h[3] for h in heads], traces=traces, loggers=loggers)
    group = traces[0]["engine"]
    numel = C * D
    n_steps = [len(tr["stats"]) for tr in traces]
    assert n_steps[2] < n_steps[0] == 40, n_steps
    for k, tr in enumerate(traces):
        recs = tr["grad_diag"]
        want_steps = [sn["step"] for sn in group.snaps if sn["active"][k]]
        assert [s for s, _ in recs] == want_steps and len(recs) == n_steps[k]
        logged = [r for r in loggers[k].recs if "train/image_loss" in r]
        assert len(logged) == n_steps[k] and all(all(key in r for key in KEYS) for r in logged)
        by_step = {sn["step"]: sn for sn in group.snaps}
        for step, d in recs:
            sn = by_step[step]
            ii, ti = sn["ii"][k], sn["ti"][k]
            dot, aa, bb, agree, amb = _ref_sums(*sn["w"][k], xi[ii], yi[ii], xt[ti], yt[ti])
            ref = ops.grad_diag_record(dot, aa, bb, agree, numel, True)
            assert abs(d[KEYS[0]] - ref[KEYS[0]]) <= 1e-5, (k, step, d, ref)
            for key in KEYS[1:3]:
                assert abs(d[key] - ref[key]) <= 1e-4 * ref[key], (k, step, key, d, ref)
            assert abs(d[KEYS[3]] - ref[KEYS[3]]) <= amb / numel + 1e-7, (k, step, d, ref)


def test_main_with_sweep_batched_logs_gradient_probes_per_step(tmp_path, monkeypatch):
    import os
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
    monkeypatch.setitem(HYPER_DICT, "unit_test_diag", dict(HYPER_DICT["clip_linear"], lr=[1e-3, 1e-4], weight_decay=[0.0],
                                                             max_iter=[30], patience=[50]))
    loggers = []

    class Logger:
        def __init__(self):
            self.recs = []
            loggers.append(self)

        def log(self, d):
            self.recs.append(dict(d))

    monkeypatch.setattr(ft, "setup_wandb_logger", lambda hp, args: Logger())
    groups = []
    real = ft.train_group
    monkeypatch.setattr(ft, "train_group", lambda *a, **k: (groups.append(len(a[0])), real(*a, **k))[1])
    args = parser.parse_args(["--dataset", "synthset", "--train-shot", "16", "--seed", "1", "--clip-encoder", "ViT-B/16",
                              "--modality", "crossmodal", "--text_type", "cupl", "--hyperparams", "unit_test_diag",
                              "--alpha", "0.5", "--feature_dir", fdir, "--result_dir", str(tmp_path / "exp"),
                              "--num-workers", "0", "--sweep-batched", "--grad-diagnostics"])
    ft.main(args)
    assert groups == [2] and len(loggers) == 2
    for lg in loggers:
        steps = [r for r in lg.recs if "train/image_loss" in r]
        assert len(steps) == 30
        for r in steps:
            assert all(key in r and math.isfinite(r[key]) for key in KEYS), r
            assert -1.0 <= r[KEYS[0]] <= 1.0 and 0.0 <= r[KEYS[3]] <= 1.0
    assert os.path.isdir(str(tmp_path / "exp"))


def test_single_adapter_run_with_diagnostics_trains_without_them(capsys):
    """A single run of an adapter head with gradient diagnostics asked for (preset `linear` without batching, or a group
    sent down the sequential path) trains to the end and logs no probes instead of failing at the first evaluation."""
    C, D, Dv, bs = 10, 40, 24, 16
    g = torch.Generator().manual_seed(3)
    xi, yi = torch.randn(100, Dv, generator=g), torch.randint(0, C, (100,), generator=g)
    xt, yt = torch.randn(80, D, generator=g), torch.randint(0, C, (80,), generator=g)
    torch.manual_seed(4)
    m = UML(f"synthetic:{Dv}", D, C, learnable_temp=True)
    m.precision = "fp32"
    m.to(DEV)
    opt = build_optimizer(m.parameters(), "adamw", 1e-3, 0.0)
    sch = build_lr_scheduler(opt, "cosine", 2, 20, warmup_type="linear", warmup_lr=1e-5)
    il = BankLoader(FeatureBank(xi, yi, DEV), bs, shuffle=True)
    tl = BankLoader(FeatureBank(xt, yt, DEV), bs, shuffle=True)
    vl = BankLoader(FeatureBank(xi, yi, DEV), bs, shuffle=False)
    tr = {"grad_diagnostics": True}
    ft.train(m, il, tl, vl, None, opt, sch, device=DEV, max_iters=12, alpha=0.5, eval_freq=5, patience=5, trace=tr)
    assert len(tr["stats"]) == 12 and "grad_diag" not in tr
    assert "no gradient probes" in capsys.readouterr().out
