"""Host logic of adapter sweep batching (finetune.train_group with AdapterHeadGroup, setup_group with
--sweep-batched-adapter) without a GPU: the launches of uml_sweep_adapter_run and the evaluation kernels are replaced by
a plain torch fp32 stand-in built on the oracle's step.  The real kernels run the same body in
tests/test_sweep_adapter_gpu.py."""
import ctypes as C

import torch

import uml_b200  # noqa: F401
from oracle import uml_oracle as O
from uml_b200 import _lib
from uml_b200 import finetune as ft
from uml_b200.engine import sweep as sweep_mod

from adapter_sweep_case import run_adapter_group_case


def _state(model):
    """An oracle HeadState whose tensors ARE the module's parameters (the oracle's optimizer updates them in place)."""
    st = O.HeadState(head=model.head.weight.data, img_proj=model.img_proj.weight.data if model.img_proj is not None else None,
                     learnable_temp=bool(model.learnable_temp), img_scale=float(model.img_scale),
                     txt_scale=float(model.txt_scale))
    if st.learnable_temp:
        st.scales = {"img_scale": model.img_scale.data, "txt_scale": model.txt_scale.data}
    return st


class TorchAdapterGroup(sweep_mod.AdapterHeadGroup):
    """AdapterHeadGroup with the launches replaced by torch ops (test double; the product class refuses CPU tensors)."""

    def __init__(self, models, optimizers, image_bank, text_bank, max_img_rows, max_txt_rows, device, log_slots=128):
        self.K = len(models)
        self.models, self.opts = list(models), list(optimizers)
        self.C, self.D = models[0].num_classes, models[0].shared_dim
        self.banks = (image_bank, text_bank)
        self.log_slots = log_slots
        self.stats_log = torch.zeros((log_slots, self.K, 2, 4))
        self.learnable = bool(models[0].learnable_temp)
        self.states = [_state(m) for m in models]
        self.oracle_opts = [O.OracleOptimizer(st.param_dict(), o.name, o.defaults["lr"], o.group_of(m.head.weight)["weight_decay"])
                            for st, m, o in zip(self.states, models, optimizers)]
        assert max_img_rows + max_txt_rows <= sweep_mod.ADAPTER_MAX_ROWS

    def image_scales(self):
        return [float(m.img_scale) for m in self.models]

    def run(self, perms_img, perms_txt, pos_img, pos_txt, rows, lrs, alphas, active, slot0):
        s0 = slot0 % self.log_slots
        assert s0 + len(rows) <= self.log_slots
        ints = self.stats_log.view(torch.int32)
        for i, (n_i, n_t) in enumerate(rows):
            for k in range(self.K):
                if not active[k]:
                    continue
                xi = yi = xt = yt = None
                if n_i:
                    idx = perms_img[k][pos_img:pos_img + n_i]
                    xi, yi = self.banks[0].features[idx], self.banks[0].labels[idx]
                if n_t:
                    idx = perms_txt[k][pos_txt:pos_txt + n_t]
                    xt, yt = self.banks[1].features[idx], self.banks[1].labels[idx]
                stats, grads = O.uml_step_grads(self.states[k], xi, yi, xt, yt, alphas[k])
                self.oracle_opts[k].step(grads, lrs[i][k])
                for p in self._trained(self.models[k]):
                    self.opts[k].slot(p)["step"] += 1
                for s, (l, a, n) in enumerate((("image_loss", "img_acc", n_i), ("text_loss", "text_acc", n_t))):
                    self.stats_log[s0 + i, k, s, 0] = stats[l] if n else 0.0
                    ints[s0 + i, k, s, 2] = int(round(stats[a] * n)) if n else 0
                    ints[s0 + i, k, s, 3] = n
            pos_img += n_i
            pos_txt += n_t


def torch_validate_enqueue(model, val_loader, s_img=None):
    iter(val_loader)
    bank = val_loader.bank
    st = _state(model)
    if s_img is not None:
        assert float(s_img) == float(model.img_scale)
    loss, acc = O.validate(st, bank.features, bank.labels, val_loader.batch_size, loader_protocol=False)
    return torch.tensor([loss]), torch.tensor([int(round(acc * len(bank)))], dtype=torch.int32), len(bank)


def _patched(monkeypatch):
    monkeypatch.setattr(sweep_mod, "AdapterHeadGroup", TorchAdapterGroup)
    monkeypatch.setattr(ft, "validate_enqueue", torch_validate_enqueue)


def test_adapter_group_of_three_heads_matches_reference_and_oracle(monkeypatch):
    _patched(monkeypatch)
    outs, traces, stopped = run_adapter_group_case(ft, "cpu")
    assert stopped[2] and not stopped[0], "the case must cover a head that stops early while others continue"


def test_adapter_group_sgd_image_only(monkeypatch):
    _patched(monkeypatch)
    run_adapter_group_case(ft, "cpu", optim="sgd", modality="image")


def _models(n, **kw):
    from uml_b200.engine.models.head import UML
    return [UML("synthetic:8", kw.get("text_indim", 12), kw.get("C", 4), learnable_temp=kw.get("learnable", True))
            for _ in range(n)]


def test_adapter_group_blockers():
    from uml_b200.engine.datasets.utils import BankLoader, FeatureBank
    from uml_b200.engine.models.head import UML, UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    bank = FeatureBank(torch.zeros(40, 8), torch.zeros(40, dtype=torch.int64), "cpu")
    tbank = FeatureBank(torch.zeros(40, 12), torch.zeros(40, dtype=torch.int64), "cpu")
    opt = lambda m, name="adamw", lr=1e-3, wd=0.0: build_optimizer(m.parameters(), name, lr, wd)
    il = lambda bs=8: BankLoader(bank, bs, shuffle=True)
    tl = lambda bs=8: BankLoader(tbank, bs, shuffle=True)
    a, b = _models(2)
    assert sweep_mod.adapter_group_blockers([a, b], [opt(a), opt(b, lr=1e-2, wd=0.1)], [il(), il()], [tl(), tl()]) == []
    c = UML("synthetic:8", 0, 4, learnable_temp=True)  # no adapter
    assert any("mix adapter" in w for w in sweep_mod.adapter_group_blockers([a, c], [opt(a), opt(c)], [il(), il()], [None, None]))
    d = _models(1, C=6)[0]
    assert any("shape" in w for w in sweep_mod.adapter_group_blockers([a, d], [opt(a), opt(d)], [il(), il()], [tl(), tl()]))
    e = _models(1, learnable=False)[0]
    assert any("learnable_temp" in w for w in sweep_mod.adapter_group_blockers([a, e], [opt(a), opt(e)], [il(), il()], [tl(), tl()]))
    assert any("64 rows" in w for w in sweep_mod.adapter_group_blockers([a, b], [opt(a), opt(b)], [il(40), il(40)], [tl(40), tl(40)]))
    f = UML("synthetic:8", 10, 4, learnable_temp=True)  # D = 10: not a multiple of 4
    assert any("multiples of 4" in w for w in sweep_mod.adapter_group_blockers([f], [opt(f)], [il()], [None]))
    assert any("optimizers" in w for w in sweep_mod.adapter_group_blockers([a, b], [opt(a), opt(b, "sgd")], [il(), il()], [tl(), tl()]))
    assert any("loaders" in w for w in sweep_mod.adapter_group_blockers([a, b], [opt(a), opt(b)], [il(), il(16)], [tl(), tl()]))
    assert any("modality" in w for w in sweep_mod.adapter_group_blockers([a, b], [opt(a), opt(b)], [il(), il()], [tl(), None]))
    g = UMLClip("synthetic:8", 4)
    assert sweep_mod.adapter_group_blockers([g], [opt(g)], [il()], [None])
    # the plain HeadGroup still refuses these heads
    assert sweep_mod.group_blockers([a, b], [opt(a), opt(b)], [il(), il()], [tl(), tl()])


def _linear_args(tmp_path, **over):
    import types
    a = types.SimpleNamespace(device="cpu", savepath=str(tmp_path), use_clip=False, clip_encoder="", img_indim=16,
                              nclasses=6, logit=3.0, hyperparams="linear", modality="crossmodal", classifier_init="random",
                              common_dim=0, text_indim=16, num_workers=0, alpha=0.5, eval_test=False, seed=3, overwrite=False,
                              sweep_batched=True, dataset="synth", precision="fp32", vision_model="synthetic",
                              dp_sampler="global")
    a.__dict__.update(over)
    return a


def _linear_datasets():
    from oracle.synth import synth_banks
    from uml_b200.engine.datasets.utils import FeatureBank, TextTensorDataset
    xi, yi, xt, yt, xv, yv = synth_banks(2, 6, 16, 20, 60, 4, 30)
    tds = TextTensorDataset(xt, yt, torch.zeros(len(yt), dtype=torch.int64))
    return {"text_ds": tds, "text_bank": FeatureBank.from_text_dataset(tds, "cpu"), "img_tr_bank": FeatureBank(xi, yi, "cpu"),
            "img_val_bank": FeatureBank(xv, yv, "cpu"), "img_te_bank": FeatureBank(xv, yv, "cpu")}


def _linear_hp():
    return dict(optim="adamw", lr=[1e-2, 1e-3], weight_decay=[0.0, 0.01], lr_scheduler="cosine", batch_size=8, max_iter=20,
                warmup_iter=5, warmup_type="linear", warmup_min_lr=1e-5, dropout=0.0, learnable_temp=True, patience=3)


def test_setup_group_batches_linear_runs_only_with_the_flag(monkeypatch, tmp_path):
    """Preset-`linear` combinations (adapter + learnable temperatures) train as one AdapterHeadGroup with
    --sweep-batched-adapter, and one by one through train() without it; the batched result files hold every
    state-dict key and match each combination trained alone with its derived seed."""
    import os
    _patched(monkeypatch)
    monkeypatch.setattr(ft, "EVAL_FREQ", 5)
    groups, solos = [], []
    real_group = ft.train_group
    monkeypatch.setattr(ft, "train_group", lambda *a, **k: (groups.append(len(a[0])), real_group(*a, **k))[1])

    def fake_train(model, *a, **k):
        solos.append(model.img_proj is not None)
        return {"iter": 0, "val_acc": 0.5, "val_loss": 1.0, "model": {k_: v.cpu() for k_, v in model.state_dict().items()}}
    monkeypatch.setattr(ft, "train", fake_train)
    d0 = tmp_path / "plain"
    d0.mkdir()
    ft.sweep(_linear_datasets(), _linear_hp(), _linear_args(d0, text_indim=20))
    assert groups == [] and solos == [True] * 4
    d1 = tmp_path / "batched"
    d1.mkdir()
    torch.manual_seed(5)  # classifier_init "random": the weights are drawn from the global generator
    res, _, _ = ft.sweep(_linear_datasets(), _linear_hp(), _linear_args(d1, text_indim=20, sweep_batched=False,
                                                                            sweep_batched_adapter=True))
    assert groups == [4] and solos == [True] * 4 and len(res["val_acc"]) == 4
    files = sorted(os.path.join(r, f) for r, _, fs in os.walk(str(d1)) for f in fs if f == "test_result.pth")
    assert len(files) == 4
    for f in files:
        assert sorted(torch.load(f)["model"]) == ["head.weight", "img_proj.weight", "img_scale", "txt_scale"]
    # combination 0 of the grid (lr 1e-2, wd 0) alone with its derived seed and the same initial weights: the same
    # result, bit for bit (the group does not couple its members)
    d2 = tmp_path / "alone"
    d2.mkdir()
    a2 = _linear_args(d2, text_indim=20)
    hp2 = dict(_linear_hp(), lr=1e-2, weight_decay=0.0)
    datasets = _linear_datasets()
    torch.manual_seed(5)
    ctx = ft._prepare(datasets, hp2, a2, rng=torch.Generator().manual_seed(ft.run_seed(a2, 0)))
    out = real_group([ctx["model"]], [ctx["image_loader"]], [ctx["text_loader"]], [ctx["val_loader"]], None,
                     [ctx["optimizer"]], [ctx["scheduler"]], device="cpu", max_iters=hp2["max_iter"], alphas=a2.alpha,
                     eval_freq=5, patience=hp2["patience"])
    alone = ft._finish(ctx, out[0], a2)
    grouped = torch.load([f for f in files if "lr_0.01-wd_0.0-" in f][0])
    assert grouped["iter"] == alone["iter"] and grouped["val_acc"] == alone["val_acc"]
    for key in grouped["model"]:
        assert torch.equal(grouped["model"][key], alone["model"][key]), key


def test_cli_flag_parses_and_merges_alpha_jobs(monkeypatch, tmp_path):
    import yaml
    from uml_b200.engine.config import parser
    assert parser.parse_args(["--sweep-batched-adapter"]).sweep_batched_adapter is True
    assert parser.parse_args([]).sweep_batched_adapter is False
    calls = []
    monkeypatch.setattr(ft, "main", lambda args, alphas=None: calls.append((args.dataset, args.alpha, alphas)))
    cfg = {"dataset": ["sun397"], "alpha": [0.2, 1.0], "hyperparams": "linear", "sweep_batched_adapter": True}
    path = tmp_path / "sweep.yaml"
    path.write_text(yaml.safe_dump(cfg, sort_keys=False))
    ft.cli(["-c", str(path)])
    assert calls == [("sun397", 0.2, [0.2, 1.0])]


def test_ctypes_adapter_struct_matches_the_header(tmp_path):
    """sizeof and every field offset of the ctypes mirror equal what a C compiler makes of include/uml_b200.h."""
    import os
    import shutil
    import subprocess
    import pytest
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cls, cname = _lib.SweepAdapterArgs, "uml_sweep_adapter_args"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "uml_b200.h"', 'int main(void) {',
             f'  printf("{cname} %zu\\n", sizeof({cname}));']
    lines += [f'  printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got[cname]) == C.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f"{cname}.{f}"]) == getattr(cls, f).offset, f


def test_sweep_adapter_run_validates_arguments_before_touching_the_device():
    lib = _lib.load()
    a, ad = _lib.SweepArgs(), _lib.SweepAdapterArgs()
    rows, lr = (C.c_int64 * 2)(4, 4), (C.c_float * 1)(1e-3)
    run = lambda: lib.uml_sweep_adapter_run(C.byref(a), C.byref(ad), 1, rows, lr, None)
    assert lib.uml_sweep_adapter_run(C.byref(a), None, 1, rows, lr, None) != 0
    assert b"null argument" in lib.uml_last_error()
    a.n_heads = 0
    assert run() != 0 and b"heads" in lib.uml_last_error()
    a.n_heads, a.dim, a.n_classes, a.ldg, a.kind = 1, 8, 4, 4, 7
    assert run() != 0 and b"optimizer kind" in lib.uml_last_error()
    a.kind = 1
    assert run() != 0 and b"null buffer" in lib.uml_last_error()
    fake = 1 << 20  # never dereferenced: every check below fails first
    a.W = a.m = a.v = a.G = a.row_loss = a.row_correct = a.stats = fake
    a.head_stride, a.max_rows = 32, 16
    a.dim = 10
    a.head_stride = 40
    assert run() != 0 and b"multiples of 4" in lib.uml_last_error()
    a.dim, a.head_stride = 8, 32
    a.n_classes, a.ldg, a.head_stride = 1100, 1100, 8800
    assert run() != 0 and b"1024 classes" in lib.uml_last_error()
    a.n_classes, a.ldg, a.head_stride = 4, 4, 32
    a.max_rows = 65
    assert run() != 0 and b"64 rows" in lib.uml_last_error()
    a.max_rows = 16
    a.W = fake + 4
    assert run() != 0 and b"16-byte aligned" in lib.uml_last_error()
    a.W = fake
    ad.img_dim = 8
    assert run() != 0 and b"null adapter buffer" in lib.uml_last_error()
    ad.W = ad.m = ad.v = ad.Z = ad.dZ = fake
    ad.adapter_stride, ad.ldz, ad.max_img_rows = 64, 6, 8
    assert run() != 0 and b"ldz" in lib.uml_last_error()
    ad.ldz = 8
    ad.scale_param = fake
    assert run() != 0 and b"learnable temperatures" in lib.uml_last_error()
