"""Shared body of the adapter sweep-batching parity tests (CPU host-logic test with a torch stand-in for the kernels, GPU
test with the real ones): three UML heads with an image adapter (Dv 24 -> D 40) and learnable temperatures over the
banks of the ``train_adapter`` golden case, trained in lock step by ``finetune.train_group``.

  head 0  the golden configuration with the golden run's seed: must reproduce the UNMODIFIED reference's trace
          (tests/golden/train_adapter.npz) - sampler order bit-exact, losses, best iteration, all four best-state keys;
  head 1  other lr / weight decay / alpha, its own seed;
  head 2  patience 1, so that it stops early while the others carry on.
Every head is checked against the oracle's ``train`` run alone after ``torch.manual_seed(seed_k)``.
"""
import ast
import os

import numpy as np
import torch

from oracle import uml_oracle as O
from oracle.synth import synth_banks

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

HEADS = [dict(lr=None, wd=None, alpha=None, patience=None, seed=None),   # filled from the golden cfg
         dict(lr=1e-2, wd=0.0, alpha=0.5, patience=5, seed=7),
         dict(lr=1e-4, wd=0.01, alpha=1.5, patience=1, seed=8)]
KEYS = ("head.weight", "img_proj.weight", "img_scale", "txt_scale")


def _unpad(a):
    return [row[row >= 0] for row in a]


def _close(got, want, tol=1e-3):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    return np.abs(got - want).max() <= tol * max(np.abs(want).max(), 1e-12)


def run_adapter_group_case(ft, device, optim=None, modality=None):
    from uml_b200.engine.datasets.utils import BankLoader, FeatureBank, TextTensorDataset
    from uml_b200.engine.models.head import UML
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler

    fx = np.load(os.path.join(GOLDEN, "train_adapter.npz"), allow_pickle=False)
    cfg = ast.literal_eval(str(fx["cfg"]))
    golden_exact = optim is None and modality is None
    optim, modality = optim or cfg["optim"], modality or cfg["modality"]
    iters = [cfg["steps"]] * len(HEADS)
    heads = [dict(h) for h in HEADS]
    heads[0].update(lr=cfg["lr"], wd=cfg["wd"], alpha=cfg["alpha"], patience=cfg["patience"], seed=1000 + cfg["seed"])
    xi, yi, xt, yt, xv, yv = synth_banks(cfg["seed"], cfg["C"], cfg["Dv"], cfg["D"], cfg["n_img"], cfg["tpc"], cfg["n_val"])
    eot = torch.zeros(xt.shape[0], dtype=torch.int64)
    torch.manual_seed(cfg["seed"])
    tds = TextTensorDataset(xt, yt, eot, n_shots=cfg["text_shot"])
    init = {k[5:]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith("init/")}
    ib, tb, vb = FeatureBank(xi, yi, device), FeatureBank.from_text_dataset(tds, device), FeatureBank(xv, yv, device)
    models, opts, schs, ils, tls, vls, traces = [], [], [], [], [], [], []
    for h in heads:
        model = UML(f"synthetic:{cfg['Dv']}", cfg["D"], cfg["C"], learnable_temp=True)
        model.precision = "fp32"
        model.load_state_dict({k: v.clone() for k, v in init.items()})
        model.to(device)
        opt = build_optimizer(model.parameters(), optim, h["lr"], h["wd"])
        rng = torch.Generator().manual_seed(h["seed"])
        models.append(model)
        opts.append(opt)
        schs.append(build_lr_scheduler(opt, "cosine", cfg["warmup_iter"], cfg["sched_max"], warmup_type="linear", warmup_lr=1e-5))
        ils.append(BankLoader(ib, cfg["bs"], shuffle=True, num_workers=cfg["num_workers"], rng=rng) if modality != "text" else None)
        tls.append(BankLoader(tb, cfg["bs"], shuffle=True, num_workers=cfg["num_workers"], rng=rng) if modality != "image" else None)
        vls.append(BankLoader(vb, cfg["bs"], shuffle=False, rng=rng))
        traces.append({})
    torch.manual_seed(99)  # the global stream must not matter
    outs = ft.train_group(models, ils, tls, vls, None, opts, schs, device=device, max_iters=iters,
                          alphas=[h["alpha"] for h in heads], eval_freq=cfg["eval_freq"],
                          patience=[h["patience"] for h in heads], traces=traces)

    # ---- head 0 against the reference's golden trace ------------------------------------------------------------
    if golden_exact:
        out, tr = outs[0], traces[0]
        assert len(tr["stats"]) == int(fx["steps_ran"])
        for a, b in zip(tr["img_idx"], _unpad(fx["img_idx"])):
            assert np.array_equal(a.numpy(), b)
        for a, b in zip(tr["txt_idx"], _unpad(fx["txt_idx"])):
            assert np.array_equal(a.numpy(), b)
        np.testing.assert_allclose([s["lr"] for s in tr["stats"]], fx["lr"], rtol=1e-9)
        np.testing.assert_allclose([s["image_loss"] for s in tr["stats"]], fx["image_loss"], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose([s["text_loss"] for s in tr["stats"]], fx["text_loss"], rtol=1e-4, atol=1e-5)
        assert out["iter"] == int(fx["best_iter"])
        assert abs(out["val_acc"] - float(fx["best_val_acc"])) < 1e-6
        assert sorted(out["model"]) == sorted(KEYS)
        for key in KEYS:
            assert _close(out["model"][key].numpy(), fx["best/" + key]), key

    # ---- every head against the oracle's train() run alone with the head's seed --------------------------------
    stopped_early = []
    for k, h in enumerate(heads):
        st = O.HeadState(head=init["head.weight"].clone(), img_proj=init["img_proj.weight"].clone(),
                         img_scale=float(init["img_scale"]), txt_scale=float(init["txt_scale"]), learnable_temp=True)
        torch.manual_seed(h["seed"])
        want, wtr = O.train(st, (xi, yi) if modality != "text" else None,
                            (tds.input_tensor, tds.label_tensor) if modality != "image" else None, (xv, yv),
                            batch_size=cfg["bs"], optim=optim, lr=h["lr"], weight_decay=h["wd"],
                            warmup_iter=cfg["warmup_iter"], sched_max_iter=cfg["sched_max"], max_iters=iters[k],
                            alpha=h["alpha"], eval_freq=cfg["eval_freq"], patience=h["patience"],
                            num_workers=cfg["num_workers"])
        out, tr = outs[k], traces[k]
        n = len(wtr.lr)
        stopped_early.append(n < iters[k])
        assert len(tr["stats"]) == n, (k, len(tr["stats"]), n)
        for name, ref in (("img_idx", wtr.img_idx), ("txt_idx", wtr.txt_idx)):
            if ref:
                assert len(tr[name]) == len(ref)
                for a, b in zip(tr[name], ref):
                    assert np.array_equal(a.numpy(), b), (k, name)
        np.testing.assert_allclose([s["lr"] for s in tr["stats"]], wtr.lr, rtol=1e-9)
        if modality != "text":
            np.testing.assert_allclose([s["image_loss"] for s in tr["stats"]], wtr.image_loss, rtol=1e-4, atol=1e-5)
            np.testing.assert_allclose([s["img_acc"] for s in tr["stats"]], wtr.img_acc, atol=1e-6)
        if modality != "image":
            np.testing.assert_allclose([s["text_loss"] for s in tr["stats"]], wtr.text_loss, rtol=1e-4, atol=1e-5)
            np.testing.assert_allclose([s["text_acc"] for s in tr["stats"]], wtr.text_acc, atol=1e-6)
        assert [e[0] for e in tr["evals"]] == [e[0] for e in wtr.evals]
        np.testing.assert_allclose([e[1] for e in tr["evals"]], [e[1] for e in wtr.evals], rtol=1e-4, atol=1e-5)
        np.testing.assert_allclose([e[2] for e in tr["evals"]], [e[2] for e in wtr.evals], atol=1e-6)
        assert out["iter"] == want["iter"], (k, out["iter"], want["iter"])
        for key in KEYS:
            assert _close(out["model"][key].numpy(), want["model"][key].numpy()), (k, key)
        # the module holds the restored best state
        live = models[k].state_dict()
        for key in KEYS:
            assert np.array_equal(live[key].detach().cpu().numpy(), out["model"][key].numpy()), (k, key)
    return outs, traces, stopped_early
