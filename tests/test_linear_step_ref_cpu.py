"""The float64 step reference (tests/linear_step_ref.py) against the project's CPU oracle of the reference step
(oracle/uml_oracle.py: uml_step_grads + OracleOptimizer), with fp32 operands.  The oracle computes in fp32, so the two
agree to about 1e-5 relative; this pins the reference before the GPU tests judge the kernels by it."""
import math

import pytest
import torch

from linear_step_ref import Adapter, Hyper, RunIn, Temperature, adapter_step, apply_update, linear_step
from oracle import uml_oracle as O

# (n_img, n_txt, D, C): one run, two runs, ragged and tiny shapes
SHAPES = [(12, 0, 16, 7), (0, 9, 24, 5), (10, 6, 32, 11), (33, 17, 8, 3)]


def _close(a, b, rtol=2e-5, atol=1e-6):
    a, b = torch.as_tensor(a, dtype=torch.float64), torch.as_tensor(b, dtype=torch.float64)
    err = float((a - b).abs().max()) if a.numel() else 0.0
    assert err <= atol + rtol * float(b.abs().max()), (err, float(b.abs().max()))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("kind", ["adamw", "adam", "sgd"])
@pytest.mark.parametrize("learnable", [False, True])
def test_reference_step_matches_the_oracle(shape, kind, learnable):
    ni, nt, d, c = shape
    g = torch.Generator().manual_seed(ni * 1000 + nt * 10 + d + c)
    W0 = torch.randn(c, d, generator=g) / math.sqrt(d)
    s_img, s_txt, alpha, wd = 3.0, 1.5, 0.5, 0.01
    st = O.HeadState(head=W0.clone(), img_scale=s_img, txt_scale=s_txt, learnable_temp=learnable)
    opt = O.OracleOptimizer(st.param_dict(), kind, 1e-2, wd)
    hp = Hyper(kind, lr=1e-2, weight_decay=wd)
    W, m, v = W0.double(), torch.zeros(c, d, dtype=torch.float64), torch.zeros(c, d, dtype=torch.float64)
    temps = [Temperature(torch.tensor(s, dtype=torch.float64), torch.tensor(0.0, dtype=torch.float64),
                         torch.tensor(0.0, dtype=torch.float64), 0) for s in (s_img, s_txt)]
    # two steps, so that the second starts from moments both wrote
    for step in (1, 2):
        xi, yi = torch.randn(ni, d, generator=g), torch.randint(0, c, (ni,), generator=g)
        xt, yt = torch.randn(nt, d, generator=g), torch.randint(0, c, (nt,), generator=g)
        ostats, ograds = O.uml_step_grads(st, xi if ni else None, yi if ni else None, xt if nt else None,
                                          yt if nt else None, alpha)
        opt.step(ograds)
        runs = []
        for n, x, y, s, w, t in ((ni, xi, yi, s_img, 1.0, temps[0]), (nt, xt, yt, s_txt, alpha, temps[1])):
            if n:
                if learnable:
                    t.step += 1
                runs.append(RunIn(x, y, s, w, t if learnable else None))
        out = linear_step(W, runs, hp, step, m, v, keep_g=True)
        k = 0
        for n, lk, ak, sk in ((ni, "image_loss", "img_acc", "img_scale"), (nt, "text_loss", "text_acc", "txt_scale")):
            if not n:
                continue
            got = out["stats"][k]
            assert got["n"] == n
            assert math.isclose(got["loss_mean"], ostats[lk], rel_tol=2e-5, abs_tol=1e-6)
            assert got["correct"] == round(ostats[ak] * n)
            if learnable:
                assert math.isclose(got["dscale"], float(ograds[sk]), rel_tol=2e-5, abs_tol=1e-6)
            k += 1
        _close(out["dW"], ograds["head.weight"])
        _close(out["W"], st.head)
        W, m, v = out["W"], out["m"], out["v"]
        if learnable:
            k = 0
            for n, t, key in ((ni, temps[0], "img_scale"), (nt, temps[1], "txt_scale")):
                if not n:
                    continue  # neither side steps a temperature without rows
                tv, tm, tvv = out["temps"][k]
                assert math.isclose(float(tv), float(st.scales[key]), rel_tol=2e-6, abs_tol=1e-7)
                t.value, t.m, t.v = tv, tm, tvv
                k += 1
    # G of the last step: rows of a softmax-minus-onehot sum to zero
    assert float(out["G"].sum(1).abs().max()) <= 1e-12


@pytest.mark.parametrize("shape", [(6, 5, 12, 16, 7), (9, 0, 10, 8, 5), (0, 7, 10, 8, 5)],
                         ids=["both_runs", "image_only", "text_only"])
@pytest.mark.parametrize("kind", ["adamw", "adam", "sgd"])
@pytest.mark.parametrize("learnable", [False, True])
def test_adapter_reference_matches_the_oracle(shape, kind, learnable):
    """adapter_step against uml_step_grads with HeadState.img_proj and OracleOptimizer over three steps: a step with
    both runs (or one modality) first, then a step with the other modality missing, then both again - Wp, its moments
    and its step count only move on steps with image rows, as the oracle skips a parameter without a gradient."""
    ni, nt, dv, d, c = shape
    g = torch.Generator().manual_seed(ni * 100 + nt * 10 + dv + d + c)
    Wp0, W0 = torch.randn(d, dv, generator=g) / math.sqrt(dv), torch.randn(c, d, generator=g) / math.sqrt(d)
    s_img, s_txt, alpha, wd, lr = 1.3, 0.8, 0.5, 0.02, 1e-2
    st = O.HeadState(head=W0.clone(), img_proj=Wp0.clone(), img_scale=s_img, txt_scale=s_txt, learnable_temp=learnable)
    opt = O.OracleOptimizer(st.param_dict(), kind, lr, wd)
    hp = Hyper(kind, lr=lr, weight_decay=wd)
    z = lambda t: torch.zeros_like(t, dtype=torch.float64)
    W, m, v = W0.double(), z(W0), z(W0)
    ad = Adapter(Wp0.double(), z(Wp0), z(Wp0), 0)
    temps = [Temperature(torch.tensor(s, dtype=torch.float64), torch.tensor(0.0, dtype=torch.float64),
                         torch.tensor(0.0, dtype=torch.float64), 0) for s in (s_img, s_txt)]
    # the second step drops one modality: the image run when the first step had both or only text rows
    plan = [(ni, nt), (0, nt) if nt else (ni, 0), (ni, nt)] if ni and nt else [(ni, nt), (ni or 4, nt or 3), (ni, nt)]
    for step, (si, sn) in enumerate(plan, start=1):
        xi, yi = torch.randn(si, dv, generator=g), torch.randint(0, c, (si,), generator=g)
        xt, yt = torch.randn(sn, d, generator=g), torch.randint(0, c, (sn,), generator=g)
        ostats, ograds = O.uml_step_grads(st, xi if si else None, yi if si else None, xt if sn else None,
                                          yt if sn else None, alpha)
        opt.step(ograds)
        for n, t in ((si, temps[0]), (sn, temps[1])):
            if n and learnable:
                t.step += 1
        img = RunIn(xi, yi, s_img, 1.0, temps[0] if learnable else None) if si else None
        txt = RunIn(xt, yt, s_txt, alpha, temps[1] if learnable else None) if sn else None
        wp_before = ad.Wp.clone()
        out = adapter_step(W, ad, img, txt, hp, step, m, v)
        k = 0
        for n, lk, ak in ((si, "image_loss", "img_acc"), (sn, "text_loss", "text_acc")):
            if n:
                assert math.isclose(out["stats"][k]["loss_mean"], ostats[lk], rel_tol=2e-5, abs_tol=1e-6)
                assert out["stats"][k]["correct"] == round(ostats[ak] * n)
                k += 1
        _close(out["dW"], ograds["head.weight"])
        _close(out["W"], st.head)
        if si:
            _close(out["Z"], xi.double() @ wp_before.t())
            _close(out["dWp"], ograds["img_proj.weight"])
            assert out["Wp_step"] == ad.step + 1
        else:
            assert out["dWp"] is None and out["Wp_step"] == ad.step
            assert torch.equal(out["Wp"], ad.Wp) and torch.equal(out["Wp_m"], ad.m)
        _close(out["Wp"], st.img_proj)
        W, m, v = out["W"], out["m"], out["v"]
        ad = Adapter(out["Wp"], out["Wp_m"], out["Wp_v"], out["Wp_step"])
        if learnable:
            k = 0
            for n, t, key in ((si, temps[0], "img_scale"), (sn, temps[1], "txt_scale")):
                if not n:
                    continue
                tv, tm, tvv = out["temps"][k]
                assert math.isclose(float(tv), float(st.scales[key]), rel_tol=2e-6, abs_tol=1e-7)
                t.value, t.m, t.v = tv, tm, tvv
                k += 1
    assert ad.step == sum(1 for si, _ in plan if si)


@pytest.mark.parametrize("kind", ["adamw", "adam", "sgd"])
def test_update_rule_matches_the_oracle_from_a_warm_state(kind):
    """apply_update on a gradient it is given, from moments after four oracle steps (step 5): the state the GPU tests
    start from."""
    g = torch.Generator().manual_seed(7)
    p = {"w": torch.randn(500, generator=g)}
    opt = O.OracleOptimizer(p, kind, 3e-3, 0.02)
    for _ in range(4):
        opt.step({"w": torch.randn(500, generator=g)})
    st = opt.state["w"]
    p0 = p["w"].clone()
    m0 = (st["buf"] if kind == "sgd" else st["m"]).clone()
    v0 = None if kind == "sgd" else st["v"].clone()
    grad = torch.randn(500, generator=g)
    opt.step({"w": grad})
    pw, mw, vw = apply_update(Hyper(kind, lr=3e-3, weight_decay=0.02), p0, grad, m0, v0, 5)
    _close(pw, p["w"], rtol=2e-6, atol=1e-7)
    _close(mw, st["buf"] if kind == "sgd" else st["m"], rtol=2e-6, atol=1e-7)
    if kind != "sgd":
        _close(vw, st["v"], rtol=2e-6, atol=1e-9)


def test_row_blocks_do_not_change_the_result():
    g = torch.Generator().manual_seed(3)
    x, y = torch.randn(1000, 40, generator=g), torch.randint(0, 13, (1000,), generator=g)
    W = torch.randn(13, 40, generator=g) * 0.3
    runs = [RunIn(x[:700], y[:700], 20.0, 1.0), RunIn(x[700:], y[700:], 7.0, 0.5)]
    hp, m = Hyper("adamw"), torch.zeros(13, 40, dtype=torch.float64)
    a = linear_step(W, runs, hp, 1, m, m.clone(), bf16_operands=True, block_rows=64)
    b = linear_step(W, runs, hp, 1, m, m.clone(), bf16_operands=True, block_rows=100000)
    _close(a["dW"], b["dW"], rtol=1e-12, atol=0)
    _close(a["G"], b["G"], rtol=1e-12, atol=0)
    for sa, sb in zip(a["stats"], b["stats"]):
        assert sa["correct"] == sb["correct"] and sa["n"] == sb["n"] and sa["near_ties"] == sb["near_ties"]
        assert math.isclose(sa["loss_mean"], sb["loss_mean"], rel_tol=1e-12)
        assert math.isclose(sa["dscale"], sb["dscale"], rel_tol=1e-12)
