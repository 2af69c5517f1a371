"""Adapter sweep batching through the real kernels (uml_sweep_adapter_run, csrc/sweep.cu): the three-head parity case of
tests/adapter_sweep_case.py, the entry point against the oracle's step at small and full sizes, every group head against
the single-head engine, slot independence, and main() with --sweep-batched-adapter end to end."""
import os

import numpy as np
import pytest
import torch

from oracle import uml_oracle as O

from adapter_sweep_case import HEADS, KEYS, _close, run_adapter_group_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

if torch.cuda.is_available():
    import uml_b200  # noqa: F401
    from uml_b200 import finetune as ft
    from uml_b200.engine import sweep as sweep_mod
    from uml_b200.engine.datasets.utils import FeatureBank
    from uml_b200.engine.models.head import UML
    from uml_b200.engine.optimizer.optim import build_optimizer


def test_adapter_group_of_three_heads_matches_reference_and_oracle():
    outs, traces, stopped = run_adapter_group_case(ft, DEV)
    assert stopped[2] and not stopped[0]
    assert traces[0]["engine"].launches > 0


def test_adapter_group_sgd_image_only():
    run_adapter_group_case(ft, DEV, optim="sgd", modality="image")


def test_adapter_group_heads_match_the_single_head_engine():
    """Heads 1 and 2 of the parity case against finetune.train() of the same combination and seed (the per-step fp32
    path of the single-head engine): losses 1e-4, weights 1e-3."""
    from adapter_sweep_case import GOLDEN
    import ast
    from oracle.synth import synth_banks
    from uml_b200.engine.datasets.utils import BankLoader, TextTensorDataset
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler
    outs, traces, _ = run_adapter_group_case(ft, DEV)
    fx = np.load(os.path.join(GOLDEN, "train_adapter.npz"), allow_pickle=False)
    cfg = ast.literal_eval(str(fx["cfg"]))
    xi, yi, xt, yt, xv, yv = synth_banks(cfg["seed"], cfg["C"], cfg["Dv"], cfg["D"], cfg["n_img"], cfg["tpc"], cfg["n_val"])
    torch.manual_seed(cfg["seed"])
    tds = TextTensorDataset(xt, yt, torch.zeros(xt.shape[0], dtype=torch.int64), n_shots=cfg["text_shot"])
    init = {k[5:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("init/")}
    for k in (1, 2):
        h = HEADS[k]
        model = UML(f"synthetic:{cfg['Dv']}", cfg["D"], cfg["C"], learnable_temp=True)
        model.precision = "fp32"
        model.load_state_dict({n: v.clone() for n, v in init.items()})
        model.to(DEV)
        opt = build_optimizer(model.parameters(), cfg["optim"], h["lr"], h["wd"])
        sch = build_lr_scheduler(opt, "cosine", cfg["warmup_iter"], cfg["sched_max"], warmup_type="linear", warmup_lr=1e-5)
        torch.manual_seed(h["seed"])
        il = BankLoader(FeatureBank(xi, yi, DEV), cfg["bs"], shuffle=True)
        tl = BankLoader(FeatureBank.from_text_dataset(tds, DEV), cfg["bs"], shuffle=True)
        vl = BankLoader(FeatureBank(xv, yv, DEV), cfg["bs"], shuffle=False)
        tr = {}
        out = ft.train(model, il, tl, vl, None, opt, sch, device=DEV, max_iters=cfg["steps"], alpha=h["alpha"],
                       eval_freq=cfg["eval_freq"], patience=h["patience"], trace=tr)
        g = traces[k]
        assert len(g["stats"]) == len(tr["stats"])
        for name in ("image_loss", "text_loss"):
            np.testing.assert_allclose([s[name] for s in g["stats"]], [s[name] for s in tr["stats"]], rtol=1e-4, atol=1e-5)
        assert outs[k]["iter"] == out["iter"]
        for key in KEYS:
            assert _close(outs[k]["model"][key].numpy(), out["model"][key].cpu().numpy()), (k, key)


def _params(model):
    return {n: p.detach().cpu().clone() for n, p in model.state_dict().items()}


@pytest.mark.parametrize("Dv,D,C,optim,modality,adapter", [
    (24, 40, 10, "adamw", "crossmodal", True),
    (24, 40, 10, "adam", "image", True),
    (24, 40, 10, "sgd", "image", False),
    (24, 40, 10, "adamw", "text", True),
    (384, 768, 397, "sgd", "crossmodal", True),
    (384, 768, 397, "adam", "image", False),
    (1536, 3200, 1000, "adamw", "crossmodal", True),
])
def test_sweep_adapter_run_matches_the_oracle(Dv, D, C, optim, modality, adapter):
    """A few steps of four heads (different lr / weight decay / alpha / temperatures; head 1 masked; head 3 a twin of
    head 0) with a ragged last batch, against the oracle's step and optimizer head by head."""
    g = torch.Generator().manual_seed(Dv + D + C)
    bs, steps, K = 32, 3, 4
    n_img, n_txt = 2 * bs + 5, 2 * bs + 9  # the third step is short
    has_img, has_txt = modality != "text", modality != "image"
    width = Dv if adapter else D
    xi, yi = torch.randn(n_img, width, generator=g), torch.randint(0, C, (n_img,), generator=g)
    xt, yt = torch.randn(n_txt, D, generator=g), torch.randint(0, C, (n_txt,), generator=g)
    ib, tb = FeatureBank(xi, yi, DEV), FeatureBank(xt, yt, DEV)
    hp = [(1e-3, 0.01, 0.5), (2e-3, 0.0, 1.0), (5e-3, 0.1, 1.5), (1e-3, 0.01, 0.5)]
    models, opts, states, inits = [], [], [], []
    for k in range(K):
        src = 0 if k == K - 1 else k  # the twin of head 0
        gk = torch.Generator().manual_seed(100 + src)
        m = UML(f"synthetic:{width}", D if adapter else 0, C, learnable_temp=True)
        sd = {"head.weight": 0.05 * torch.randn(C, D, generator=gk), "img_scale": torch.tensor(1.0 + 0.5 * src),
              "txt_scale": torch.tensor(2.0 - 0.25 * src)}
        if adapter:
            sd["img_proj.weight"] = torch.randn(D, Dv, generator=gk) / Dv ** 0.5
        m.load_state_dict(sd)
        inits.append({n: v.double() for n, v in sd.items()})
        m.to(DEV)
        lr, wd, _ = hp[k]
        models.append(m)
        opts.append(build_optimizer(m.parameters(), optim, lr, wd))
        pair = []
        for dt in (torch.float32, torch.float64):  # the fp32 oracle and a float64 one that judges both fp32 results
            st = O.HeadState(head=sd["head.weight"].to(dt), img_proj=sd["img_proj.weight"].to(dt) if adapter else None,
                             img_scale=float(sd["img_scale"]), txt_scale=float(sd["txt_scale"]), learnable_temp=True)
            st.param_dict()
            st.scales = {n: v.to(dt) for n, v in st.scales.items()}
            pair += [st, O.OracleOptimizer(st.param_dict(), optim, lr, wd)]
        states.append(pair)
    group = sweep_mod.AdapterHeadGroup(models, opts, ib if has_img else None, tb if has_txt else None,
                                       bs if has_img else 0, bs if has_txt else 0, DEV, log_slots=8)
    before = _params(models[1])
    pi = [torch.randperm(n_img, generator=torch.Generator().manual_seed(7 + (0 if k == K - 1 else k))) for k in range(K)]
    pt = [torch.randperm(n_txt, generator=torch.Generator().manual_seed(9 + (0 if k == K - 1 else k))) for k in range(K)]
    rows = [(min(bs, n_img - s * bs) if has_img else 0, min(bs, n_txt - s * bs) if has_txt else 0) for s in range(steps)]
    lrs = [[hp[k][0] * (1.0 - 0.1 * s) for k in range(K)] for s in range(steps)]
    active = [True, False, True, True]
    group.time_last_step()
    group.run([p.to(DEV) for p in pi] if has_img else None, [p.to(DEV) for p in pt] if has_txt else None, 0, 0, rows, lrs,
              [h[2] for h in hp], active, slot0=0)
    torch.cuda.synchronize()
    assert set(group.kernel_times_ms()) == set(group.KERNELS)
    log = group.read_log(list(range(steps)), has_img, has_txt)
    for k in range(K):
        if not active[k]:
            continue
        st, oo, st64, oo64 = states[k]
        pos_i = pos_t = 0
        for s, (n_i, n_t) in enumerate(rows):
            x_i = y_i = x_t = y_t = None
            if n_i:
                x_i, y_i = xi[pi[k][pos_i:pos_i + n_i]], yi[pi[k][pos_i:pos_i + n_i]]
            if n_t:
                x_t, y_t = xt[pt[k][pos_t:pos_t + n_t]], yt[pt[k][pos_t:pos_t + n_t]]
            _, g64 = O.uml_step_grads(st64, *(None if v is None else (v.double() if v.is_floating_point() else v)
                                              for v in (x_i, y_i, x_t, y_t)), hp[k][2])
            oo64.step(g64, lrs[s][k])
            stats, grads = O.uml_step_grads(st, x_i, y_i, x_t, y_t, hp[k][2])
            oo.step(grads, lrs[s][k])
            if has_img:
                assert abs(log["image_loss"][s][k] - stats["image_loss"]) <= 1e-4 * max(1.0, stats["image_loss"]), (k, s)
            if has_txt:
                assert abs(log["text_loss"][s][k] - stats["text_loss"]) <= 1e-4 * max(1.0, stats["text_loss"]), (k, s)
            pos_i += n_i
            pos_t += n_t
        got = _params(models[k])
        ref = st64.param_dict()
        for name, want in st.param_dict().items():
            d = (got[name] - want).abs().double() / max(float(want.abs().max()), 1e-12)
            if optim == "sgd" or want.numel() == 1:
                assert float(d.max()) < 1e-3, (k, name, float(d.max()))
                continue
            # Adam divides by |g| + eps: where a gradient nearly cancels (the adapter's dZ = sum_c (p_c - y_c) W_c does
            # at cfg4) a last-bit difference of the gradient becomes a different step, so single elements of two fp32
            # implementations can differ by up to 2 lr.  Judged against a float64 oracle instead: the mean error, relative
            # to the largest accumulated update of the tensor, stays at 1e-3 (3xTF32 products carry 2^-21 relative error
            # against 2^-24 for an FFMA, so the kernels sit about ten times further from float64 than the fp32 oracle)
            upd = float((ref[name] - inits[k][name]).abs().max())
            e_gpu = float((got[name].double() - ref[name]).abs().mean())
            if upd == 0.0:  # a parameter without a gradient (the adapter of a text-only run) is left as it was
                assert e_gpu == 0.0, (k, name)
                continue
            e_f32 = float((want.double() - ref[name]).abs().mean())
            print(f"head {k} {name}: mean error vs float64 / largest update: kernels {e_gpu / upd:.3g}, "
                  f"fp32 oracle {e_f32 / upd:.3g}")
            assert e_gpu < 1e-3 * upd, (k, name, e_gpu / upd, e_f32 / upd)
    # the masked head is untouched; the twins in slots 0 and K - 1 agree bit for bit
    for name, p in _params(models[1]).items():
        assert torch.equal(p, before[name]), name
    for name, p in _params(models[0]).items():
        assert torch.equal(p, _params(models[K - 1])[name]), name


def test_main_with_sweep_batched_adapter_writes_all_checkpoint_keys(tmp_path):
    """finetune.main with --sweep-batched-adapter over bank files of a unimodal image / language encoder pair (preset
    `linear`-style: adapter + learnable temperatures): every combination trains in one AdapterHeadGroup and its
    test_result.pth holds all four state-dict keys."""
    from oracle.synth import synth_banks
    from uml_b200 import features as F
    from uml_b200.engine.config import parser
    from uml_b200.engine.optimizer.default import HYPER_DICT
    C, Dv, D = 12, 32, 48
    xi, yi, xt, yt, xv, yv = synth_banks(4, C, Dv, D, 16 * C, 6, 4 * C)
    fdir, rdir = str(tmp_path / "features"), str(tmp_path / "experiments")
    lab2cname = {c: f"class_{c}" for c in range(C)}
    F.write_text_bank(F.text_outdir(fdir, "gpt2", "synthset", "cupl"), xt, yt, lab2cname=lab2cname)
    F.write_image_bank(F.img_outdir(fdir, "dinov2", "synthset", "crop", 16, 1, "train"), train=(xi, yi), val=(xv, yv),
                       lab2cname=lab2cname)
    F.write_image_bank(F.img_outdir(fdir, "dinov2", "synthset", "crop", 16, 1, "test"), test=(xv, yv), lab2cname=lab2cname)
    HYPER_DICT["unit_test_adapter"] = dict(HYPER_DICT["linear"], lr=[1e-3, 1e-4], weight_decay=[0.0, 0.01], batch_size=[8],
                                           max_iter=[60], patience=[3])
    groups = []
    real = ft.train_group
    ft.train_group = lambda *a, **k: (groups.append(len(a[0])), real(*a, **k))[1]
    try:
        args = parser.parse_args(["--dataset", "synthset", "--train-shot", "16", "--seed", "1", "--vision-model", "dinov2",
                                  "--language-model", "gpt2", "--modality", "crossmodal", "--text_type", "cupl",
                                  "--hyperparams", "unit_test_adapter", "--alpha", "0.5", "--feature_dir", fdir,
                                  "--result_dir", rdir, "--num-workers", "0", "--classifier_init", "random",
                                  "--sweep-batched-adapter"])
        results, best_val, best_test = ft.main(args)
    finally:
        ft.train_group = real
    assert groups == [4] and len(results["test_acc"]) == 4
    found = [os.path.join(r, f) for r, _, fs in os.walk(rdir) for f in fs if f == "test_result.pth"]
    assert len(found) == 4
    for f in found:
        ck = torch.load(f, map_location="cpu")
        assert sorted(ck["model"]) == sorted(KEYS)
        assert ck["model"]["img_proj.weight"].shape == (D, Dv) and ck["model"]["head.weight"].shape == (C, D)
