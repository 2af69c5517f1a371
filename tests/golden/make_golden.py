"""Generates the committed golden fixtures by running the UNMODIFIED reference
(/root/reference) on CPU through oracle/ref_harness.py.  Run from the repo root:

    python tests/golden/make_golden.py

Only works in the build container (the reference tree does not travel).  The fixtures
record the torch version that produced them.  Every case seeds the global RNG itself so
the files are reproducible.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402
from oracle.synth import synth_banks  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


class _Recording(torch.utils.data.Dataset):
    """Forwards to a dataset and remembers which rows were asked for, in order."""

    def __init__(self, inner):
        self.inner, self.seen = inner, []

    def __len__(self):
        return len(self.inner)

    def __getitem__(self, i):
        self.seen.append(int(i))
        return self.inner[i]


def _split(seen, n, bs, steps):
    """Cut a flat index log into per-step batches (epochs of n rows, short tail batch)."""
    out, pos = [], 0
    left = n
    for _ in range(steps):
        if left == 0:
            left = n
        take = min(bs, left)
        out.append(seen[pos:pos + take])
        pos += take
        left -= take
    assert pos == len(seen), (pos, len(seen))
    return out


def _pad(batches, bs):
    a = np.full((len(batches), bs), -1, dtype=np.int64)
    for i, b in enumerate(batches):
        a[i, :len(b)] = b
    return a


def run_reference_train(kind, *, seed, C, Dv, D, n_img, tpc, n_val, bs, steps, alpha, optim, lr, wd,
                        learnable_temp, init, eval_freq, patience, num_workers=0, modality="crossmodal",
                        text_shot=None, sched_max=None):
    ns = rh.load_vision_language()
    from torch.utils.data import DataLoader

    xi, yi, xt, yt, xv, yv = synth_banks(seed, C, Dv, D, n_img, tpc, n_val)
    eot = torch.zeros(xt.shape[0], dtype=torch.int64)
    torch.manual_seed(seed)
    tds = ns.ds_utils.TextTensorDataset(xt, yt, eot, n_shots=text_shot)
    sel_feats, sel_labels = tds.input_tensor.clone(), tds.label_tensor.clone()
    if kind == "clip":
        model = rh.build_reference_model("clip", Dv, D, C)
    else:
        model = rh.build_reference_model("uml", Dv, D if D != Dv else 0, C, learnable_temp=learnable_temp)
    if init == "zeroshot":
        model.head.weight.data = ns.head.get_zero_shot_weights(tds, C, D, device="cpu")
    init_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    opt = ns.optim.build_optimizer(model.parameters(), optim, lr, wd)
    sched_max = steps if sched_max is None else sched_max
    sch = ns.scheduler.build_lr_scheduler(opt, "cosine", 5, sched_max, warmup_type="linear", warmup_lr=1e-5)
    img_ds = _Recording(rh.make_image_rows_dataset(xi, yi))
    txt_ds = _Recording(tds)
    il = DataLoader(img_ds, batch_size=bs, shuffle=True, drop_last=False, num_workers=num_workers)
    tl = DataLoader(txt_ds, batch_size=bs, shuffle=True, drop_last=False, num_workers=num_workers)
    vl = DataLoader(rh.make_image_rows_dataset(xv, yv), batch_size=bs, shuffle=False)
    if modality == "image":
        tl = None
    if modality == "text":
        il = None
    rec = rh.StepRecorder(model, opt)
    losses, lrs = [], []
    F = torch.nn.functional
    orig_ce = F.cross_entropy
    orig_sched_step = sch.step

    def ce(*a, **k):
        r = orig_ce(*a, **k)
        if torch.is_grad_enabled():
            losses.append(float(r))
        return r

    def sched_step(*a, **k):
        lrs.append(opt.param_groups[0]["lr"])  # the lr the optimizer just used
        return orig_sched_step(*a, **k)

    F.cross_entropy = ce
    sch.step = sched_step
    # model construction consumed global RNG (nn.Linear init); pin the state train() starts from
    torch.manual_seed(1000 + seed)
    try:
        out = ns.finetune.train(model, il, tl, vl, None, opt, sch, device="cpu", max_iters=steps, alpha=alpha,
                                eval_freq=eval_freq, patience=patience,
                                capture_features_during_training=False, logger=None)
    finally:
        F.cross_entropy = orig_ce
    ran = len(rec.weights)
    per_step = 2 if modality == "crossmodal" else 1
    losses = np.asarray(losses, dtype=np.float64).reshape(ran, per_step)
    fx = {
        "torch_version": np.array(torch.__version__),
        "cfg": np.array(repr(dict(kind=kind, seed=seed, C=C, Dv=Dv, D=D, n_img=n_img, tpc=tpc, n_val=n_val, bs=bs,
                                  steps=steps, alpha=alpha, optim=optim, lr=lr, wd=wd, learnable_temp=learnable_temp,
                                  init=init, eval_freq=eval_freq, patience=patience, num_workers=num_workers,
                                  modality=modality, text_shot=text_shot, sched_max=sched_max, warmup_iter=5))),
        "steps_ran": np.array(ran),
        "lr": np.asarray(lrs, dtype=np.float64),
        "best_iter": np.array(out["iter"]), "best_val_acc": np.array(out["val_acc"]),
        "best_val_loss": np.array(out["val_loss"]),
        "sel_text_labels": sel_labels.numpy(), "sel_text_feats_sum": sel_feats.double().sum(1).numpy(),
    }
    if num_workers == 0:
        if il is not None:
            fx["img_idx"] = _pad(_split(img_ds.seen, len(img_ds), bs, ran), bs)
        if tl is not None:
            fx["txt_idx"] = _pad(_split(txt_ds.seen, len(txt_ds), bs, ran), bs)
    if modality == "crossmodal":
        fx["image_loss"], fx["text_loss"] = losses[:, 0], losses[:, 1]
    elif modality == "image":
        fx["image_loss"] = losses[:, 0]
    else:
        fx["text_loss"] = losses[:, 0]
    for k in init_state:
        fx["init/" + k] = init_state[k].numpy()
    for s in sorted({0, 1, min(7, ran - 1), ran - 1}):
        for k, v in rec.weights[s].items():
            fx[f"w{s}/" + k] = v.numpy()
    for k, v in out["model"].items():
        fx["best/" + k] = v.numpy()
    return fx


def sampler_with_workers():
    """Index order of the real DataLoader with worker processes (RNG protocol differs from
    num_workers=0: the sampler seed is drawn inside iter())."""
    from torch.utils.data import DataLoader

    class Idx(torch.utils.data.Dataset):
        def __len__(self):
            return 23

        def __getitem__(self, i):
            return i

    class Idx2(Idx):
        def __len__(self):
            return 17

    res = {}
    for nw in (0, 2):
        torch.manual_seed(123)
        a = DataLoader(Idx(), batch_size=5, shuffle=True, drop_last=False, num_workers=nw)
        b = DataLoader(Idx2(), batch_size=5, shuffle=True, drop_last=False, num_workers=nw)
        ia, ib = iter(a), iter(b)
        sa, sb = [], []
        for _ in range(12):
            try:
                x = next(ia)
            except StopIteration:
                ia = iter(a)
                x = next(ia)
            sa.append(x.tolist())
            try:
                y = next(ib)
            except StopIteration:
                ib = iter(b)
                y = next(ib)
            sb.append(y.tolist())
        res[f"nw{nw}_a"] = _pad(sa, 5)
        res[f"nw{nw}_b"] = _pad(sb, 5)
    return res


def schedule_and_optim():
    ns = rh.load_vision_language()
    fx = {}
    for name, kw in {"cos_lin": dict(s="cosine", w=50, T=12800, wt="linear", wl=1e-5, base=1e-3),
                     "cos_lin_short": dict(s="cosine", w=5, T=40, wt="linear", wl=1e-5, base=1e-4),
                     "lin_const": dict(s="linear", w=4, T=30, wt="constant", wl=1e-5, base=5e-5),
                     "cos_nowarm": dict(s="cosine", w=0, T=25, wt=None, wl=None, base=1e-3)}.items():
        p = torch.nn.Parameter(torch.zeros(1))
        opt = ns.optim.build_optimizer([p], "adamw", kw["base"], 0.0)
        sch = ns.scheduler.build_lr_scheduler(opt, kw["s"], kw["w"], kw["T"], warmup_type=kw["wt"], warmup_lr=kw["wl"])
        n = min(kw["T"] + kw["w"], 300)
        lrs = []
        for _ in range(n):
            lrs.append(opt.param_groups[0]["lr"])
            opt.step()
            sch.step()
        fx["sched/" + name] = np.asarray(lrs)
        fx["sched/" + name + "/cfg"] = np.array(repr(kw))
    # optimizer trajectories on a fixed gradient stream
    g = torch.Generator().manual_seed(5)
    p0 = torch.randn(6, 5, generator=g)
    gs = [torch.randn(6, 5, generator=g) * (0.1 + i) for i in range(6)]
    fx["optim/p0"] = p0.numpy()
    fx["optim/grads"] = torch.stack(gs).numpy()
    for name, lr, wd in (("adamw", 1e-2, 0.01), ("adam", 1e-2, 0.01), ("sgd", 1e-2, 0.01), ("adamw", 1e-3, 0.0)):
        p = torch.nn.Parameter(p0.clone())
        opt = ns.optim.build_optimizer([p], name, lr, wd)
        traj = []
        for gi in gs:
            p.grad = gi.clone()
            opt.step()
            traj.append(p.detach().clone())
        fx[f"optim/{name}_lr{lr}_wd{wd}"] = torch.stack(traj).numpy()
    return fx


def text_and_init():
    ns = rh.load_vision_language()
    g = torch.Generator().manual_seed(9)
    C, D = 7, 6
    counts = [5, 3, 0, 4, 1, 6, 2]  # class 2 has no text rows (like the 998/1000 CUPL case)
    labels = torch.cat([torch.full((n,), c, dtype=torch.int64) for c, n in enumerate(counts)])
    perm = torch.randperm(labels.numel(), generator=g)
    labels = labels[perm]
    feats = torch.randn(labels.numel(), D, generator=g)
    eot = torch.arange(labels.numel())
    fx = {"text/feats": feats.numpy(), "text/labels": labels.numpy(), "text/eot": eot.numpy()}
    for shots in (2, 4):
        torch.manual_seed(31)
        ds = ns.ds_utils.TextTensorDataset(feats, labels, eot, n_shots=shots)
        fx[f"text/shot{shots}/eot"] = ds.eot_indices.numpy()  # eot == original row id
        fx[f"text/shot{shots}/after_draw"] = np.array(int(torch.empty((), dtype=torch.int64).random_().item()))
    ds = ns.ds_utils.TextTensorDataset(feats, labels, eot, n_shots="average")
    fx["text/avg/feats"], fx["text/avg/labels"], fx["text/avg/eot"] = (
        ds.input_tensor.numpy(), ds.label_tensor.numpy(), ds.eot_indices.numpy())
    full = ns.ds_utils.TextTensorDataset(feats, labels, eot, n_shots=None)
    fx["text/zeroshot_w"] = ns.head.get_zero_shot_weights(full, C, D, device="cpu").numpy()
    # validate with a ragged last batch
    model = rh.build_reference_model("clip", D, D, C)
    model.head.weight.data = torch.randn(C, D, generator=g)
    xv = torch.randn(11, D, generator=g)
    yv = torch.randint(0, C, (11,), generator=g)
    from torch.utils.data import DataLoader
    vl = DataLoader(rh.make_image_rows_dataset(xv, yv), batch_size=4, shuffle=False)
    vloss, vacc = ns.finetune.validate(model, vl, device="cpu")
    fx["val/W"], fx["val/x"], fx["val/y"] = model.head.weight.detach().numpy(), xv.numpy(), yv.numpy()
    fx["val/loss"], fx["val/acc"], fx["val/scale"] = np.array(vloss), np.array(vacc), np.array(float(model.logit_scale.exp()))
    # path layout
    f = ns.features
    fx["path/img_train"] = np.array(f.img_outdir("F", "ViT-B/16", "imagenet", "crop", 16, 1, "train"))
    fx["path/img_test"] = np.array(f.img_outdir("F", "ViT-B/16", "imagenet", "crop", 16, 1, "test"))
    fx["path/text"] = np.array(f.text_outdir("F", "ViT-B/16", "imagenet", "gpt3_cupl"))
    fx["path/hparam"] = np.array(ns.finetune.hparam_str("adamw", 0.001, 0.01, 32, 12800, 0.0, True))
    import argparse
    a = argparse.Namespace(common_dim=0)
    fx["path/savedir_x"] = np.array(ns.finetune.savedir("E", "imagenet", "ViT-B/16", 16, 1, "gpt3_cupl", "average", "crop",
                                                        "crossmodal", "zeroshot", 0.5, 0, "", a))
    fx["path/savedir_i"] = np.array(ns.finetune.savedir("E", "sun397", "a-b", 4, 2, "gpt3_cupl", None, "flip",
                                                        "image", "random", 0.0, 0, "tag", a))
    return fx


def reference_defaults():
    """The reference's hyper-parameter presets and the defaults of its command-line parser."""
    ns = rh.load_vision_language()
    from engine.config import parser  # the reference's, via the harness' sys.path
    return {"HYPER_DICT": ns.default.HYPER_DICT, "parser_defaults": vars(parser.parse_args([]))}


def gaussian():
    gm = rh.load_gaussian()
    cfg = dict(seed=42, num_samples=64, dim_c=10, dim_x=5, dim_y=5, dim_obs=12, noise_std=0.09,
               attenuate_x=True, attenuation=0.05, shared_latent_distribution_type="gaussian")
    d1 = gm.data.generate_data(dict(cfg))
    cfg2 = dict(cfg, seed=44, shared_latent_distribution_type="laplace")
    d2 = gm.data.generate_data(dict(cfg2))
    fx = {"gauss/x": d1["x"].numpy(), "gauss/y": d1["y"].numpy(), "gauss/y_laplace": d2["y"].numpy(),
          "gauss/cfg": np.array(repr(cfg))}
    from torch.utils.data import DataLoader
    for mode in ("xy", "x"):
        if mode == "xy":
            ds = gm.dataset.UnpairedDataset(d1["x"][:32], d1["y"][:32])
        else:
            ds = gm.dataset.UnpairedDataset(d1["x"], d2["y"][:40])
        g = torch.Generator()
        g.manual_seed(42)
        loader = DataLoader(ds, batch_size=16, shuffle=True, drop_last=True, generator=g)
        gm.utils.make_reproducible(3)
        model = gm.model.SharedAutoencoder(dim_obs=12, dim_common=16, dim_latent=6)
        for k, v in model.state_dict().items():
            fx[f"gauss/{mode}/init/{k}"] = v.clone().numpy()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        it = iter(loader)
        lx_l, ly_l = [], []
        for _ in range(9):  # the loop body of main.py:40-59
            try:
                batch = next(it)
            except StopIteration:
                it = iter(loader)
                batch = next(it)
            opt.zero_grad()
            lx, ly, _, _ = model(batch["x"], batch["y"])
            loss = 1.0 * lx + 0.5 * ly if mode == "xy" else lx
            loss.backward()
            opt.step()
            lx_l.append(float(lx))
            ly_l.append(float(ly))
        fx[f"gauss/{mode}/loss_x"], fx[f"gauss/{mode}/loss_y"] = np.asarray(lx_l), np.asarray(ly_l)
        for k, v in model.state_dict().items():
            fx[f"gauss/{mode}/final/{k}"] = v.clone().numpy()
    return fx


def main():
    torch.set_num_threads(1)  # deterministic summation order for the committed numbers
    cases = {
        # CLIP-style fixed logit scale 100, zero-shot init, several epochs of both loaders
        "train_clip": dict(kind="clip", seed=11, C=12, Dv=32, D=32, n_img=50, tpc=3, n_val=20, bs=8, steps=60,
                           alpha=0.5, optim="adamw", lr=1e-3, wd=0.01, learnable_temp=False, init="zeroshot",
                           eval_freq=20, patience=5),
        # adapter (Dv != D) + learnable temperatures, random init
        "train_adapter": dict(kind="uml", seed=12, C=10, Dv=24, D=40, n_img=37, tpc=4, n_val=16, bs=8, steps=40,
                              alpha=1.0, optim="adamw", lr=1e-3, wd=0.001, learnable_temp=True, init="random",
                              eval_freq=10, patience=2),
        # image-only, sgd, early stop
        "train_image_sgd": dict(kind="uml", seed=13, C=6, Dv=16, D=16, n_img=30, tpc=2, n_val=12, bs=4, steps=50,
                                alpha=0.0, optim="sgd", lr=1e-2, wd=0.01, learnable_temp=False, init="random",
                                eval_freq=5, patience=3, modality="image"),
        # text shots subsampled at construction (consumes global RNG before training)
        "train_textshot": dict(kind="clip", seed=14, C=8, Dv=16, D=16, n_img=20, tpc=5, n_val=8, bs=8, steps=25,
                               alpha=1.5, optim="adam", lr=1e-3, wd=0.0, learnable_temp=False, init="zeroshot",
                               eval_freq=100, patience=5, text_shot=2),
    }
    for name, kw in cases.items():
        fx = run_reference_train(**kw)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **fx)
        print(name, "steps_ran", int(fx["steps_ran"]), "best", int(fx["best_iter"]), float(fx["best_val_acc"]))
    misc = {"torch_version": np.array(torch.__version__)}
    misc.update(sampler_with_workers())
    misc.update(schedule_and_optim())
    misc.update(text_and_init())
    misc.update(gaussian())
    np.savez_compressed(os.path.join(OUT, "misc.npz"), **misc)
    print("misc keys", len(misc))
    with open(os.path.join(OUT, "reference_defaults.json"), "w") as f:
        json.dump(reference_defaults(), f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
