"""Host side of per-step gradient diagnostics for batched sweep groups without a GPU: the ctypes mirror of
uml_sweep_diag, the argument checks of uml_sweep_run_diag, the --grad-diagnostics flag, setup_group's routing of
groups whose diagnostics cannot be computed on the device, and the shared finishing formula."""
import ctypes as C
import os
import shutil
import subprocess
import types

import pytest
import torch

import uml_b200  # noqa: F401
from uml_b200 import _lib, ops
from uml_b200 import finetune as ft

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ctypes_diag_struct_matches_the_header(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    cls, cname = _lib.SweepDiag, "uml_sweep_diag"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "uml_b200.h"', 'int main(void) {',
             f'  printf("{cname} %zu\\n", sizeof({cname}));']
    lines += [f'  printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got[cname]) == C.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f"{cname}.{f}"]) == getattr(cls, f).offset, f


def test_scratch_size_query():
    lib = _lib.load()
    assert lib.uml_sweep_diag_scratch_floats(30, 512, 1000) == 30 * 4 * 16 * 4
    assert lib.uml_sweep_diag_scratch_floats(2, 40, 10) == 2 * 1 * 1 * 4
    assert lib.uml_sweep_diag_scratch_floats(0, 40, 10) == 0


def test_sweep_run_diag_validates_arguments_before_touching_the_device():
    lib = _lib.load()
    a, ad, dg = _lib.SweepArgs(), _lib.SweepAdapterArgs(), _lib.SweepDiag()
    rows, lr = (C.c_int64 * 2)(4, 4), (C.c_float * 1)(1e-3)
    run = lambda adp=None: lib.uml_sweep_run_diag(C.byref(a), adp, C.byref(dg), 1, rows, lr, None)
    assert lib.uml_sweep_run_diag(C.byref(a), None, None, 1, rows, lr, None) != 0
    assert b"null argument" in lib.uml_last_error()
    a.n_heads = 0
    assert run() != 0 and b"heads" in lib.uml_last_error()
    a.n_heads = 1
    assert run() != 0 and b"null diagnostics buffer" in lib.uml_last_error()
    fake = 1 << 20  # never dereferenced: every check below fails first
    dg.out = dg.scratch = fake
    a.dim, a.n_classes, a.ldg, a.kind, a.head_stride, a.max_rows = 10, 4, 4, 1, 40, 8
    assert run() != 0 and b"multiple of 4" in lib.uml_last_error()
    a.dim, a.head_stride = 8, 32
    a.W, a.m, a.v, a.G = fake + 4, fake, fake, fake
    assert run() != 0 and b"16-byte aligned" in lib.uml_last_error()
    a.W = fake
    a.bank[1], a.bank_ld[1] = fake + 8, 8
    assert run() != 0 and b"bank 1" in lib.uml_last_error()
    a.bank[1] = fake
    ad.img_dim, ad.Z, ad.ldz = 8, fake + 4, 8
    assert run(C.byref(ad)) != 0 and b"Z must be" in lib.uml_last_error()
    a.active[0], a.alpha[0] = 1, 0.0
    assert run() != 0 and b"alpha" in lib.uml_last_error()
    a.alpha[0] = 0.5
    dg.scratch_floats = 3
    assert run() != 0 and b"scratch" in lib.uml_last_error()


def test_grad_diagnostics_flag_defaults_to_off():
    from uml_b200.engine.config import parser
    assert parser.parse_args([]).grad_diagnostics is False
    assert parser.parse_args(["--grad-diagnostics"]).grad_diagnostics is True


def test_finishing_helper_equals_the_former_inline_formula():
    def inline(dot, aa, bb, agree, numel, both):  # what StepEngine.grad_diagnostics computed before the helper
        ni, nt = aa ** 0.5, bb ** 0.5
        return {"train/grad_direction_sim": dot / (ni * nt) if both and ni > 0 and nt > 0 else 0.0,
                "train/img_grad_norm": ni, "train/txt_grad_norm": nt,
                "train/grad_agreement_rate": agree / numel if both else 0.0}
    for args in ((0.3, 2.0, 5.0, 17.0, 40, True), (-1.5, 4.0, 1.0, 3.0, 40, True), (0.0, 0.0, 3.0, 40.0, 40, True),
                 (0.0, 2.0, 0.0, 12.0, 40, False), (1e-30, 1e-20, 1e-20, 0.0, 7, True)):
        assert ops.grad_diag_record(*args) == inline(*args)


def _datasets():
    from oracle.synth import synth_banks
    from uml_b200.engine.datasets.utils import FeatureBank, TextTensorDataset
    xi, yi, xt, yt, xv, yv = synth_banks(2, 6, 16, 16, 60, 4, 30)
    tds = TextTensorDataset(xt, yt, torch.zeros(len(yt), dtype=torch.int64))
    return {"text_ds": tds, "text_bank": FeatureBank.from_text_dataset(tds, "cpu"), "img_tr_bank": FeatureBank(xi, yi, "cpu"),
            "img_val_bank": FeatureBank(xv, yv, "cpu"), "img_te_bank": FeatureBank(xv, yv, "cpu")}


@pytest.mark.parametrize("alpha,diag,batched", [(0.0, True, False), (0.5, True, True), (0.0, False, True)])
def test_setup_group_routes_groups_without_device_diagnostics_sequentially(monkeypatch, tmp_path, alpha, diag, batched):
    """--grad-diagnostics with alpha <= 0 (text rows present): the text-loss gradient cannot be recovered from G, so the
    combinations train one after the other (evaluation-cadence diagnostics); with alpha > 0, or without the flag, they
    form one group."""
    groups, solos = [], []
    fake = lambda m: {"iter": 0, "val_acc": 0.5, "val_loss": 1.0, "model": {k: v.cpu() for k, v in m.state_dict().items()}}
    monkeypatch.setattr(ft, "train_group", lambda models, *a, **k: (groups.append((len(models), k.get("args"))),
                                                                     [fake(m) for m in models])[1])
    monkeypatch.setattr(ft, "train", lambda model, *a, **k: (solos.append(1), fake(model))[1])
    monkeypatch.setattr(ft, "_finish", lambda ctx, out, a: out)
    args = types.SimpleNamespace(device="cpu", savepath=str(tmp_path), use_clip=True, clip_encoder="synthetic", img_indim=16,
                                 nclasses=6, logit=3.0, hyperparams="clip_linear", modality="crossmodal",
                                 classifier_init="random", common_dim=0, text_indim=16, num_workers=0, alpha=alpha,
                                 eval_test=False, seed=3, overwrite=False, sweep_batched=True, dataset="synth",
                                 precision="fp32", vision_model="", dp_sampler="global", grad_diagnostics=diag)
    hp = dict(optim="adamw", lr_scheduler="cosine", batch_size=8, max_iter=20, warmup_iter=5, warmup_type="linear",
              warmup_min_lr=1e-5, dropout=0.0, learnable_temp=False, patience=3, weight_decay=0.0)
    combos = [dict(hp, lr=1e-2), dict(hp, lr=1e-3)]
    res = ft.setup_group(_datasets(), combos, args)
    assert len(res) == 2
    if batched:
        assert groups == [(2, args)] and solos == []
    else:
        assert groups == [] and solos == [1, 1]
