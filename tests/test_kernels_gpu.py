"""Parity of every CUDA kernel with the CPU oracle, called through the C ABI (ctypes).

Run on the B200 box:  python -m pytest tests -m gpu
Tolerances: the *_f32 kernels compute in fp32 like the reference (differences are summation order
only); the *_bf16 tensor-core kernels are compared (a) tightly against the oracle evaluated on the
same bf16-rounded operands - this isolates kernel correctness - and (b) against the fp32 oracle
within the stated 1e-3 relative tolerance on the loss.
"""
import math

import numpy as np
import pytest
import torch

from oracle import uml_oracle as O

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    import uml_b200  # noqa: F401
    from uml_b200 import ops

DEV = "cuda:0"


def _mk(seed, n_img, n_txt, dv, d, c):
    g = torch.Generator().manual_seed(seed)
    xi = torch.randn(n_img, dv, generator=g)
    yi = torch.randint(0, c, (n_img,), generator=g)
    xt = torch.randn(n_txt, d, generator=g)
    yt = torch.randint(0, c, (n_txt,), generator=g)
    w = torch.randn(c, d, generator=g)
    w = w / w.norm(dim=1, keepdim=True)
    return xi, yi, xt, yt, w, g


# ------------------------------------------------------------------------------------------ K1
@pytest.mark.parametrize("n_bank,dim,n", [(1000, 512, 32), (5000, 768, 1000), (300, 3200, 77), (64, 100, 9), (50, 30, 5),
                                          (128, 768, 0), (20000, 768, 16384)])
def test_gather_rows(n_bank, dim, n):
    g = torch.Generator().manual_seed(n_bank + dim + n)
    bank = torch.randn(n_bank, dim, generator=g)
    idx = torch.randint(0, n_bank, (n,), generator=g)
    bank_d, idx_d = bank.to(DEV), idx.to(DEV)
    out = ops.gather_rows(bank_d, idx_d)
    assert torch.equal(out.cpu(), bank[idx])  # byte-exact copy
    if dim % 8 == 0:
        out16 = ops.gather_rows(bank_d, idx_d, dtype=torch.bfloat16)
        assert torch.equal(out16.cpu(), bank[idx].to(torch.bfloat16))
    labels = torch.randint(0, 1000, (n_bank,), generator=g)
    lab32 = torch.empty(max(n, 1), dtype=torch.int32, device=DEV)
    ops.gather_labels(labels.to(DEV), idx_d, n, lab32)
    assert torch.equal(lab32[:n].cpu().long(), labels[idx])


@pytest.mark.parametrize("n0,n1,dim,ld,labels", [
    (32, 32, 512, 512, True), (1000, 517, 768, 768, True), (0, 77, 768, 768, True), (77, 0, 3200, 3200, True),
    (16384, 10996, 768, 768, True), (1, 1, 8, 8, True), (0, 0, 768, 768, True),
    (300, 211, 1032, 1032, True),    # 129 16-byte vectors per row: the light kernel's second pass over a row moves one
    (150, 90, 3200, 3200, True),     # OpenLLaMA width
    (4000, 1700, 256, 256, True),    # more rows than the light kernel's grid has warps (148 * 4 * 8 = 4736)
    (500, 300, 768, 776, True),      # ld_out > dim: the padding between rows stays untouched
    (700, 400, 512, 512, False),     # out_labels = NULL
])
@pytest.mark.parametrize("light", [False, True], ids=["tma", "light"])
def test_gather2_rows_bf16(n0, n1, dim, ld, labels, light):
    """Both runs of a step from bf16 shadow banks in one launch, through the TMA ring kernel and through the
    register-copy kernel the training step calls: byte-exact rows, int64 -> int32 labels."""
    g = torch.Generator().manual_seed(n0 * 7 + n1 + dim)
    b0 = torch.randn(3000, dim, generator=g).to(torch.bfloat16)
    b1 = torch.randn(700, dim, generator=g).to(torch.bfloat16)
    l0, l1 = torch.randint(0, 1000, (3000,), generator=g), torch.randint(0, 1000, (700,), generator=g)
    i0, i1 = torch.randint(0, 3000, (n0,), generator=g), torch.randint(0, 700, (n1,), generator=g)
    buf = torch.full((n0 + n1 + 3, ld), 7.0, dtype=torch.bfloat16, device=DEV)
    out = buf[:, :dim]
    lab = torch.full((n0 + n1 + 3,), -5, dtype=torch.int32, device=DEV)
    ops.gather2_rows_bf16(b0.to(DEV) if n0 else None, l0.to(DEV) if n0 else None, i0.to(DEV) if n0 else None,
                          b1.to(DEV) if n1 else None, l1.to(DEV) if n1 else None, i1.to(DEV) if n1 else None, out,
                          lab if labels else None, light=light)
    want = torch.cat([b0[i0], b1[i1]])
    assert torch.equal(out[:n0 + n1].cpu(), want)
    if labels:
        assert torch.equal(lab[:n0 + n1].cpu().long(), torch.cat([l0[i0], l1[i1]]))
    assert bool((lab == -5).all()) if not labels else bool((lab[n0 + n1:] == -5).all())
    assert bool((out[n0 + n1:] == 7.0).all())  # nothing written past the end
    assert bool((buf[:, dim:] == 7.0).all())   # nor into the padding between rows


def test_cast_bf16():
    x = torch.randn(1000 * 768 + 3)
    assert torch.equal(ops.cast_bf16(x.to(DEV)).cpu(), x.to(torch.bfloat16))


# ------------------------------------------------------------------------------------------ K6
@pytest.mark.parametrize("name,wd", [("adamw", 0.01), ("adamw", 0.0), ("adam", 0.01), ("sgd", 0.01)])
@pytest.mark.parametrize("n", [1000 * 512, 12345])
def test_optimizer_steps(name, wd, n):
    g = torch.Generator().manual_seed(n)
    p0 = torch.randn(n, generator=g)
    ref = {"p": p0.clone()}
    opt = O.OracleOptimizer(ref, name, 1e-3, wd)
    p = p0.to(DEV)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    shadow = torch.empty(n, dtype=torch.bfloat16, device=DEV)
    for step in range(1, 6):
        grad = torch.randn(n, generator=g) * (0.01 * step)
        lr = 1e-3 * step / 5
        opt.step({"p": grad}, lr)
        if name == "sgd":
            ops.sgd_step(p, grad.to(DEV), m, lr=lr, step=step, weight_decay=wd, shadow=shadow)
        else:
            ops.adamw_step(p, grad.to(DEV), m, v, lr=lr, step=step, weight_decay=wd, decoupled=(name == "adamw"),
                           shadow=shadow)
        np.testing.assert_allclose(p.cpu().numpy(), ref["p"].numpy(), rtol=2e-6, atol=2e-7)
    assert torch.equal(shadow.cpu(), p.cpu().to(torch.bfloat16))


def test_adamw_two_gradients_and_partials():
    n = 1000 * 64
    g = torch.Generator().manual_seed(3)
    p0, g1, g2 = (torch.randn(n, generator=g) for _ in range(3))
    ref = {"p": p0.clone()}
    O.OracleOptimizer(ref, "adamw", 1e-3, 0.01).step({"p": g1 + 0.5 * g2})
    p = p0.to(DEV)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    ops.adamw_step(p, g1.to(DEV), m, v, lr=1e-3, step=1, weight_decay=0.01, g2=g2.to(DEV), g2_weight=0.5)
    np.testing.assert_allclose(p.cpu().numpy(), ref["p"].numpy(), rtol=2e-6, atol=2e-7)
    parts = torch.randn(5, n, generator=g)
    ref = {"p": p0.clone()}
    O.OracleOptimizer(ref, "adamw", 1e-3, 0.01).step({"p": parts.sum(0)})
    p = p0.to(DEV)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    gout = torch.empty_like(p)
    ops.adamw_step_partials(p, parts.to(DEV), 5, m, v, lr=1e-3, step=1, weight_decay=0.01, g_out=gout)
    np.testing.assert_allclose(gout.cpu().numpy(), parts.sum(0).numpy(), rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(p.cpu().numpy(), ref["p"].numpy(), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------ fp32 head
HEAD_CASES = [
    # n_img_bank, n_txt_bank, D, C, B_img, B_txt, scale, alpha
    (16000, 2994, 512, 1000, 32, 32, 100.0, 0.5),     # cfg2 step
    (500, 300, 768, 1000, 5, 32, 100.0, 1.0),         # ragged image batch (epoch tail)
    (400, 200, 512, 397, 32, 0, 1.0, 0.0),            # image only (SUN397 classes)
    (300, 303, 512, 101, 64, 64, 100.0, 1.5),         # Food101 classes
    (200, 100, 3200, 100, 8, 8, 1.0, 0.7),            # OpenLLaMA width, tiny batch
    (3000, 3000, 96, 10, 300, 200, 10.0, 0.2),        # wide batch, narrow head
]


def _runs(xi, yi, xt, yt, ii, it, s_i, s_t, alpha):
    runs = []
    if ii is not None and ii.numel():
        runs.append(ops.Run(xi, yi, ii, ii.numel(), s_i, 1.0))
    if it is not None and it.numel():
        runs.append(ops.Run(xt, yt, it, it.numel(), s_t, alpha))
    return runs


@pytest.mark.parametrize("case", HEAD_CASES)
def test_head_step_f32_matches_oracle(case):
    nib, ntb, d, c, bi, bt, scale, alpha = case
    xi, yi, xt, yt, w, g = _mk(sum(case[:6]), nib, ntb, d, d, c)
    ii = torch.randint(0, nib, (bi,), generator=g)
    it = torch.randint(0, ntb, (bt,), generator=g)
    st = O.HeadState(head=w.clone(), img_scale=scale, txt_scale=scale * 0.5)
    stats, grads = O.uml_step_grads(st, xi[ii] if bi else None, yi[ii] if bi else None, xt[it] if bt else None,
                                    yt[it] if bt else None, alpha)
    dev = [t.to(DEV) for t in (xi, yi, xt, yt, ii, it)]
    runs = _runs(*dev, scale, scale * 0.5, alpha)
    ws = ops.HeadWorkspace(bi + bt, c, DEV)
    Wd = w.to(DEV)
    ops.head_fwd_ce_f32(runs, Wd, ws)
    got = ws.read_stats()
    k = 0
    if bi:
        assert math.isclose(got[k]["loss_mean"], stats["image_loss"], rel_tol=2e-5, abs_tol=1e-5)
        assert got[k]["correct"] == round(stats["img_acc"] * bi) and got[k]["n"] == bi
        k += 1
    if bt:
        assert math.isclose(got[k]["loss_mean"], stats["text_loss"], rel_tol=2e-5, abs_tol=1e-5)
        assert got[k]["correct"] == round(stats["text_acc"] * bt) and got[k]["n"] == bt
    dW = torch.empty_like(Wd)
    ops.head_bwd_dw_f32(runs, Wd, ws, dW=dW)
    want = grads["head.weight"]
    err = (dW.cpu() - want).abs().max().item()
    assert err <= 2e-5 * max(1.0, want.abs().max().item()), err
    # fused AdamW epilogue == oracle optimizer step on the same gradient
    ref = {"head.weight": w.clone()}
    O.OracleOptimizer(ref, "adamw", 1e-3, 0.01).step({"head.weight": want}, 2e-4)
    m, v = torch.zeros_like(Wd), torch.zeros_like(Wd)
    upd = ops.make_update("adamw", 2e-4, 1, m, v, weight_decay=0.01)
    ops.head_bwd_dw_f32(runs, Wd, ws, update=upd)
    # AdamW's first step is lr*sign(g): elements whose gradient is ~0 may flip, so compare robustly
    diff = (Wd.cpu() - ref["head.weight"]).abs()
    assert diff.max().item() <= 2 * 2e-4 + 1e-7
    assert (diff > 1e-6).float().mean().item() < 1e-3


def test_learnable_scale_gradient_f32():
    nib, ntb, d, c, bi, bt = 200, 120, 64, 20, 16, 24
    xi, yi, xt, yt, w, g = _mk(77, nib, ntb, d, d, c)
    ii = torch.randint(0, nib, (bi,), generator=g)
    it = torch.randint(0, ntb, (bt,), generator=g)
    st = O.HeadState(head=w.clone(), img_scale=3.0, txt_scale=2.0, learnable_temp=True)
    _, grads = O.uml_step_grads(st, xi[ii], yi[ii], xt[it], yt[it], 0.7)
    dev = [t.to(DEV) for t in (xi, yi, xt, yt, ii, it)]
    ws = ops.HeadWorkspace(bi + bt, c, DEV)
    ops.head_fwd_ce_f32(_runs(*dev, 3.0, 2.0, 0.7), w.to(DEV), ws)
    got = ws.read_stats()
    assert math.isclose(got[0]["dscale"], float(grads["img_scale"]), rel_tol=1e-4, abs_tol=1e-6)
    assert math.isclose(got[1]["dscale"], float(grads["txt_scale"]), rel_tol=1e-4, abs_tol=1e-6)


# (rows b, Dv, D, C, alpha, optimizer rule fused into gemm_tn or None, padding of gemm_tn's ldc)
ADAPTER_GEMMS = {"toy": (37, 96, 160, 50, 2.0, None, 0), "toy_sgd": (37, 96, 160, 50, 1.0, "sgd", 3),
                 "preset_linear_adamw": (32, 1536, 3200, 1000, 1.0, "adamw", 0),
                 "preset_linear_adam": (32, 1536, 3200, 1000, 0.5, "adam", 5)}


def test_adapter_gemms_f32():
    """The three GEMMs of the adapter's exact step (engine/trainer.py _step_fp32) against float64 on their own fp32
    operands, with the worst-case bound k u sum|a b| of an FMA chain of k terms: gemm_nt (Z = X[idx] Wp^T) and gemm_nn
    (dZ = G W over k = C < ldg) with m below the output's rows, whose rows past m stay untouched; gemm_tn (dWp = dZ^T
    X[idx]) with the optimizer update fused into its epilogue, on 32 x 32 tiles (toy) and 64 x 64 tiles (3200 x 1536),
    into a padded ldc whose padding stays untouched.  The fused update is judged by the gradient recovered from m.
    Every case of ADAPTER_GEMMS runs."""
    for case in ADAPTER_GEMMS:
        _check_adapter_gemms(case)


def _check_adapter_gemms(case):
    from linear_step_case import U, check_update, recover_grad
    from linear_step_ref import Hyper, apply_update
    b, dv, d, c, alpha, kind, pad = ADAPTER_GEMMS[case]
    g = torch.Generator(device=DEV).manual_seed(b + dv + d + c + pad)
    bank = torch.randn(b + 60, dv, device=DEV, generator=g) / math.sqrt(dv)
    idx = torch.randint(0, b + 60, (b,), device=DEV, generator=g)
    wp = torch.randn(d, dv, device=DEV, generator=g) / math.sqrt(dv)
    w = torch.randn(c, d, device=DEV, generator=g) / math.sqrt(d)
    ldg = (c + 63) // 64 * 64
    gm = torch.randn(b + 7, ldg, device=DEV, generator=g) / c   # G's rows past the image rows and its padding columns
    x64, wp64, w64, g64 = bank[idx].double(), wp.double(), w.double(), gm[:b, :c].double()

    def close(got, want, bound, what):
        r = float(((got.double() - want).abs() / (bound + 1e-30)).max())
        assert r <= 1.0, (what, r)
        return r

    z = torch.full((b + 5, d), float("nan"), device=DEV)
    ops.gemm_nt(bank, wp, z, alpha=alpha, a_row_idx=idx, m=b)
    rz = close(z[:b], alpha * x64 @ wp64.t(), abs(alpha) * dv * U * (x64.abs() @ wp64.abs().t()), "gemm_nt")
    assert bool(z[b:].isnan().all()), "gemm_nt wrote past m"
    dz = torch.full((b + 5, d), float("nan"), device=DEV)
    ops.gemm_nn(gm, w, dz, alpha=alpha, m=b, k=c)
    rdz = close(dz[:b], alpha * g64 @ w64, abs(alpha) * c * U * (g64.abs() @ w64.abs()), "gemm_nn")
    assert bool(dz[b:].isnan().all()), "gemm_nn wrote past m"
    dz64 = dz[:b].double()
    want = alpha * dz64.t() @ x64
    bound = abs(alpha) * b * U * (dz64.abs().t() @ x64.abs())
    if kind is None:
        dwp = torch.full((d, dv + pad), float("nan"), device=DEV)
        ops.gemm_tn(dz, bank, dwp, k=b, m=d, n=dv, alpha=alpha, b_row_idx=idx)
        rtn = close(dwp[:, :dv], want, bound, "gemm_tn")
        assert bool(dwp[:, dv:].isnan().all()), "gemm_tn wrote into the padding"
        print(f"\n[{case}] nt {rz:.2e}, nn {rdz:.2e}, tn {rtn:.2e} of the bounds")
        return
    # the update fused into gemm_tn, from a warm state; P, m and v padded like a strided parameter view
    hp = Hyper(kind, lr=1e-2, weight_decay=0.05).as_f32()
    store = lambda t: torch.cat([t, torch.full((d, pad), 7.0, device=DEV)], 1)
    P0 = torch.randn(d, dv, device=DEV, generator=g) / math.sqrt(dv)
    m0 = want.float() * (torch.rand(d, dv, device=DEV, generator=g) * 3 - 1)
    v0 = (want.float() ** 2 + (0.05 * float(want.abs().max())) ** 2) * (torch.rand(d, dv, device=DEV, generator=g) + 0.5)
    P, M, V = store(P0), store(m0), store(v0)
    upd = ops.make_update(kind, hp.lr, 5, M, V if kind != "sgd" else None, weight_decay=hp.weight_decay,
                          betas=(hp.beta1, hp.beta2), eps=hp.eps, momentum=hp.momentum)
    ops.gemm_tn(dz, bank, None, k=b, m=d, n=dv, alpha=alpha, b_row_idx=idx, P=P, update=upd, ldc=dv + pad)
    torch.cuda.synchronize()
    for t, nm in ((P, "P"), (M, "m"), (V, "v")):
        assert bool((t[:, dv:] == 7.0).all()), nm + ": the padding was written"
    grad, rec = recover_grad(kind, hp, m0, M[:, :dv], P0)
    rtn = close(grad, want, bound + rec, "gemm_tn recovered gradient")
    pw, mw, vw = apply_update(hp, P0, grad, m0, v0 if kind != "sgd" else None, 5)
    ru = check_update(P[:, :dv], pw, "P")
    check_update(M[:, :dv], mw, "m")
    if kind != "sgd":
        check_update(V[:, :dv], vw, "v", atol=1e-12)
    else:
        assert torch.equal(V, store(v0)), "SGD has no v"
    # a missing weight decay would stand out: wd |p| (Adam, SGD) or lr wd |p| (AdamW) against the bound it would break
    p0 = P0.double().abs()
    decay = (hp.lr * hp.weight_decay * p0 / (2e-7 + 2e-6 * pw.abs()) if kind == "adamw"
             else hp.weight_decay * p0 / (bound + rec))
    assert float(decay.median()) >= 10.0, float(decay.median())
    print(f"\n[{case}] nt {rz:.2e}, nn {rdz:.2e}, tn gradient {rtn:.2e}, update {ru:.2e} of the bounds; "
          f"weight decay {float(decay.median()):.0f}x its bound")


# ------------------------------------------------------------------------------------------ K7
@pytest.mark.parametrize("n,d,c,bs", [(4000, 512, 1000, 32), (333, 768, 397, 32), (11, 64, 7, 4), (1000, 100, 101, 64)])
def test_eval_matches_oracle_validate(n, d, c, bs):
    g = torch.Generator().manual_seed(n + c)
    x = torch.randn(n, d, generator=g)
    y = torch.randint(0, c, (n,), generator=g)
    w = torch.randn(c, d, generator=g) / math.sqrt(d)
    st = O.HeadState(head=w, img_scale=30.0)
    vloss, vacc = O.validate(st, x, y, bs, loader_protocol=False)
    xd, yd, wd = x.to(DEV), y.to(DEV), w.to(DEV)
    rl = torch.empty(n, device=DEV)
    rp = torch.empty(n, dtype=torch.int32, device=DEV)
    ops.eval_f32(xd, yd, wd, 30.0, rl, rp)
    out_l = torch.empty(1, device=DEV)
    out_c = torch.empty(1, dtype=torch.int32, device=DEV)
    ops.eval_reduce(rl, rp, yd, bs, out_l, out_c)
    assert math.isclose(out_l.item(), vloss, rel_tol=2e-5)
    assert out_c.item() == round(vacc * n)


def test_grad_diag():
    g = torch.Generator().manual_seed(8)
    a, b = torch.randn(1000 * 512, generator=g), torch.randn(1000 * 512, generator=g)
    out = torch.empty(4, device=DEV)
    ops.grad_diag(a.to(DEV), b.to(DEV), torch.empty(4 * 296, device=DEV), out)
    o = out.cpu()
    assert math.isclose(o[0].item(), float(torch.dot(a, b)), rel_tol=1e-3, abs_tol=0.5)
    assert math.isclose(o[1].item(), float(a.pow(2).sum()), rel_tol=1e-4)
    assert math.isclose(o[2].item(), float(b.pow(2).sum()), rel_tol=1e-4)
    assert o[3].item() == float((torch.sign(a) == torch.sign(b)).sum())


# ------------------------------------------------------------------------------------------ tensor cores
TC_CASES = [
    # rows_img, rows_txt, D, C
    (128, 128, 64, 256),      # one k-block, one chunk
    (256, 0, 512, 1000),      # ViT-B/16 head, single run
    (300, 212, 768, 1000),    # ViT-L/14 head, ragged rows
    (1000, 1048, 768, 1000),
    (64, 70, 128, 101),       # Food101
    (200, 56, 3200, 397),     # OpenLLaMA width
]


def _tc_reference(x16, w16, labels, n0, n1, scales, weights):
    """fp32 math on the bf16-rounded operands."""
    x, w = x16.float(), w16.float()
    raw = x @ w.t()
    outs = []
    G = torch.zeros_like(raw)
    loss = torch.zeros(raw.shape[0])
    for (lo, hi, s, wt) in ((0, n0, scales[0], weights[0]), (n0, n0 + n1, scales[1], weights[1])):
        if hi == lo:
            continue
        lg = raw[lo:hi] * s
        lse = torch.logsumexp(lg, 1)
        loss[lo:hi] = lse - lg.gather(1, labels[lo:hi].view(-1, 1).long()).squeeze(1)
        p = torch.softmax(lg, 1)
        p[torch.arange(hi - lo), labels[lo:hi].long()] -= 1.0
        G[lo:hi] = p * (wt * s / (hi - lo))
    return raw, loss, G


@pytest.mark.parametrize("case", TC_CASES)
def test_tc_forward_and_dw(case):
    n0, n1, d, c = case
    n = n0 + n1
    g = torch.Generator().manual_seed(n + d + c)
    x = torch.randn(n, d, generator=g)
    w = torch.randn(c, d, generator=g)
    w = w / w.norm(dim=1, keepdim=True)
    labels = torch.randint(0, c, (n,), generator=g, dtype=torch.int32)
    scales, weights = (100.0, 50.0), (1.0, 0.5)
    x16, w16 = x.to(torch.bfloat16), w.to(torch.bfloat16)
    raw, loss_ref, G_ref = _tc_reference(x16, w16, labels, n0, n1, scales, weights)
    ws = ops.HeadWorkspace(n, c, DEV, bf16=True)
    ws.G.fill_(float("nan"))
    rp = torch.empty(n, dtype=torch.int32, device=DEV)
    rows = [r for r in (n0, n1) if r]
    segs = ops.tc_segments(rows, scales[:len(rows)] if n0 else scales[1:], weights[:len(rows)] if n0 else weights[1:])
    xd, wd = x16.to(DEV), w16.to(DEV)
    ops.head_fwd_ce_bf16(xd, wd, labels.to(DEV), segs, ws, ws.row_loss, row_pred=rp, row_correct=ws.row_correct,
                         row_dscale=ws.row_dscale)
    torch.cuda.synchronize()
    loss = ws.row_loss[:n].cpu()
    np.testing.assert_allclose(loss.numpy(), loss_ref.numpy(), rtol=2e-4, atol=2e-3)
    lg = raw.clone()
    lg[:n0] *= scales[0]
    lg[n0:] *= scales[1]
    top2 = lg.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > 1e-2  # rows whose argmax is not a numerical near-tie
    assert torch.equal(rp.cpu()[clear].long(), lg.argmax(1)[clear])
    G = ws.G[:n].float().cpu()
    assert torch.isfinite(G).all()
    assert float(G[:, c:].abs().max()) == 0.0 if ws.ldg > c else True
    scale_ref = G_ref.abs().max().item()
    assert (G[:, :c] - G_ref).abs().max().item() <= 1.2e-2 * scale_ref  # two bf16 roundings of values <= scale_ref
    # dscale
    ds_ref = torch.zeros(n)
    for (lo, hi, s, wt) in ((0, n0, scales[0], weights[0]), (n0, n, scales[1], weights[1])):
        if hi > lo:
            ds_ref[lo:hi] = (G_ref[lo:hi] / s * raw[lo:hi]).sum(1)
    np.testing.assert_allclose(ws.row_dscale[:n].cpu().numpy(), ds_ref.numpy(), rtol=2e-2, atol=2e-4)
    # dW from the kernel's own G (isolates the MN-major GEMM) ------------------------------------
    splits = ops.tc_dw_splits(n, d, c)
    parts = torch.full((splits, c, d), float("nan"), device=DEV)
    ops.head_bwd_dw_bf16(ws.G, ws.ldg, xd, n, c, parts, splits)
    torch.cuda.synchronize()
    dW = parts.sum(0).cpu()
    dW_ref = G[:, :c].t() @ x16.float()
    assert torch.isfinite(dW).all()
    assert (dW - dW_ref).abs().max().item() <= 1e-3 * max(1e-6, dW_ref.abs().max().item())
    # and against the full-precision gradient: bf16 operand noise only
    full = G_ref.t() @ x16.float()
    rel = (dW - full).norm().item() / full.norm().item()
    assert rel < 1e-2, rel


def test_tc_loss_within_stated_tolerance_of_fp32():
    """bf16 tensor-core forward vs the fp32 oracle on the SAME fp32 inputs: mean loss within 1e-3 rel."""
    n0 = n1 = 512
    d, c = 768, 1000
    g = torch.Generator().manual_seed(1)
    x = torch.randn(n0 + n1, d, generator=g)
    w = torch.randn(c, d, generator=g)
    w = w / w.norm(dim=1, keepdim=True)
    y = torch.randint(0, c, (n0 + n1,), generator=g)
    st = O.HeadState(head=w, img_scale=100.0, txt_scale=100.0)
    stats, _ = O.uml_step_grads(st, x[:n0], y[:n0], x[n0:], y[n0:], 1.0)
    ws = ops.HeadWorkspace(n0 + n1, c, DEV, bf16=True)
    segs = ops.tc_segments([n0, n1], [100.0, 100.0], [1.0, 1.0])
    ops.head_fwd_ce_bf16(ops.cast_bf16(x.to(DEV)), ops.cast_bf16(w.to(DEV)), y.to(torch.int32).to(DEV), segs, ws,
                         ws.row_loss, row_correct=ws.row_correct)
    ops.reduce_seg_stats(ws.row_loss, ws.row_correct, None, [n0, n1], ws.stats)
    got = ws.read_stats()
    assert abs(got[0]["loss_mean"] - stats["image_loss"]) <= 1e-3 * abs(stats["image_loss"])
    assert abs(got[1]["loss_mean"] - stats["text_loss"]) <= 1e-3 * abs(stats["text_loss"])


# ------------------------------------------------------------------------------------------ generic tensor-core GEMM
GEMM_CASES = [
    # M, N, K, a_mn, b_mn, out_bf16, splits     (M > 128 runs on CTA pairs, cta_group::2)
    (100, 520, 200, False, False, True, 1),
    (300, 520, 200, False, False, True, 1),      # Z = X Wp^T
    (1000, 768, 1536, False, False, False, 3),
    (300, 520, 1000, False, True, True, 1),      # dZ = G W
    (2048, 3200, 1000, False, True, True, 1),
    (100, 96, 333, True, True, False, 2),        # dW, single-CTA tiles
    (1000, 768, 4096, True, True, False, 6),     # dW, CTA pairs
    (3200, 1536, 2048, True, True, False, 1),    # dW_proj
]


@pytest.mark.parametrize("case", GEMM_CASES)
def test_tc_gemm_layouts(case):
    M, N, K, a_mn, b_mn, out_bf16, splits = case
    g = torch.Generator().manual_seed(M + N + K)
    pad = lambda x: (x + 7) // 8 * 8
    A = torch.randn((K, pad(M)) if a_mn else (M, pad(K)), generator=g).to(torch.bfloat16)
    B = torch.randn((K, pad(N)) if b_mn else (N, pad(K)), generator=g).to(torch.bfloat16)
    a = (A[:, :M].t() if a_mn else A[:, :K]).float()
    b = (B[:, :N] if b_mn else B[:, :K].t()).float()
    ref = a @ b
    Ad, Bd = A.to(DEV), B.to(DEV)
    if out_bf16:
        out = torch.full((M, pad(N)), float("nan"), device=DEV, dtype=torch.bfloat16)
        ops.gemm_bf16(Ad, Bd, out, M, N, K, a_mn=a_mn, b_mn=b_mn)
        got = out[:, :N].float().cpu()
        tol = 1e-2 * ref.abs().max().item()
    else:
        out = torch.full((splits, M, N), float("nan"), device=DEV)
        ops.gemm_bf16(Ad, Bd, out, M, N, K, a_mn=a_mn, b_mn=b_mn, n_splits=splits)
        got = out.sum(0).cpu()
        tol = 2e-4 * ref.abs().max().item()
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() <= tol, (got - ref).abs().max().item()


def test_grad_diagnostics_match_autograd():
    """a-13: the engine's opt-in gradient probes against torch autograd on the CPU (finetune.py:190-206)."""
    from uml_b200.engine.datasets.utils import FeatureBank, IndexBatch
    from uml_b200.engine.models.head import UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.trainer import StepEngine
    xi, yi, xt, yt, w, g = _mk(5, 300, 200, 64, 64, 37)
    model = UMLClip("synthetic:64", 37, logit_scale_init=2.0)
    model.head.weight.data.copy_(w)
    model.to(DEV)
    eng = StepEngine(model, build_optimizer(model.parameters(), "adamw", 1e-3, 0.0), DEV, 64, 64)
    ii, ti = torch.randint(0, 300, (50,), generator=g), torch.randint(0, 200, (41,), generator=g)
    ib, tb = FeatureBank(xi, yi, DEV), FeatureBank(xt, yt, DEV)
    got = eng.grad_diagnostics(IndexBatch(ib, ii.to(DEV), 50, 0, ii), IndexBatch(tb, ti.to(DEV), 41, 0, ti))
    W = w.clone().requires_grad_(True)
    s = math.exp(2.0)
    gi, = torch.autograd.grad(torch.nn.functional.cross_entropy(xi[ii] @ W.t() * s, yi[ii]), W)
    gt, = torch.autograd.grad(torch.nn.functional.cross_entropy(xt[ti] @ W.t() * s, yt[ti]), W)
    gi, gt = gi.flatten(), gt.flatten()
    assert abs(got["train/img_grad_norm"] - float(gi.norm())) < 1e-4 * float(gi.norm())
    assert abs(got["train/txt_grad_norm"] - float(gt.norm())) < 1e-4 * float(gt.norm())
    assert abs(got["train/grad_direction_sim"] - float(torch.dot(gi, gt) / (gi.norm() * gt.norm()))) < 1e-4
    assert abs(got["train/grad_agreement_rate"] - float((torch.sign(gi) == torch.sign(gt)).float().mean())) < 2e-3
    assert torch.equal(model.head.weight.detach().cpu(), w)  # a probe: nothing was updated


def test_full_size_step_properties():
    """BASELINE.json's throughput shape (2 x 18944 rows, D=768, C=1000) is too big for the CPU oracle in a unit test;
    check size-independent properties of the tensor-core step instead:
      * linearity: doubling both loss weights doubles every split-K partial of dW EXACTLY (a power-of-two scale commutes
        with every rounding on the way);
      * rows of a softmax-CE gradient sum to zero, hence so does every column sum over classes of dW = G^T X
        (up to the bf16 rounding of G);
      * the per-run mean losses agree with fp32 torch math on a 512-row sample within the stated 1e-3."""
    n0 = n1 = 18944
    d, c = 768, 1000
    g = torch.Generator(device=DEV).manual_seed(11)
    x = torch.randn(n0 + n1, d, device=DEV, generator=g) * 0.05
    w = torch.randn(c, d, device=DEV, generator=g)
    w = w / w.norm(dim=1, keepdim=True)
    y = torch.randint(0, c, (n0 + n1,), device=DEV, generator=g).to(torch.int32)
    x16, w16 = ops.cast_bf16(x), ops.cast_bf16(w)
    splits = max(1, ops.tc_dw_splits(n0 + n1, d, c))
    outs = []
    for k in (1.0, 2.0):
        ws = ops.HeadWorkspace(n0 + n1, c, DEV, bf16=True)
        segs = ops.tc_segments([n0, n1], [100.0, 100.0], [1.0 * k, 0.5 * k])
        st = torch.zeros(2, 4, device=DEV)
        parts = torch.zeros(splits, c, d, device=DEV)
        ops.head_fwd_ce_bf16(x16, w16, y, segs, ws, None, n_rows=n0 + n1, stats=st)
        ops.head_bwd_dw_bf16(ws.G, ws.ldg, x16, n0 + n1, c, parts, splits)
        outs.append((parts, st, ws))
    torch.cuda.synchronize()
    (p1, st1, ws1), (p2, st2, _) = outs
    assert torch.equal(p1 * 2.0, p2)                                   # exact linearity
    assert torch.equal(st1[:, 0], st2[:, 0])                           # the loss itself does not depend on the weights
    dW = p1.sum(0)
    assert float(dW.sum(0).abs().max()) <= 2e-2 * float(dW.abs().max())  # class-sum of dW ~ 0
    assert float(ws1.G[:, :c].float().sum(1).abs().max()) <= 2e-2 * float(ws1.G.float().abs().max())
    sample = torch.randperm(n0, device=DEV, generator=g)[:512]
    for run, lo in ((0, 0), (1, n0)):
        rows = sample + lo
        logits = (x16[rows].float() @ w16.float().t()) * 100.0
        ref = torch.nn.functional.cross_entropy(logits, y[rows].long(), reduction="none")
        got = None
        # per-run mean over ALL rows vs mean over the sample: compare through per-row losses of the sample instead
        ws = ops.HeadWorkspace(n0 + n1, c, DEV, bf16=True)
        row_loss = torch.empty(n0 + n1, device=DEV)
        ops.head_fwd_ce_bf16(x16, w16, y, ops.tc_segments([n0, n1], [100.0, 100.0], [1.0, 0.5]), None, row_loss, n_rows=n0 + n1)
        got = row_loss[rows]
        torch.testing.assert_close(got, ref, rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("case", HEAD_CASES[:4] + [(300, 200, 36, 12, 8, 8, 100.0, 0.5),
                                                  (2000, 1000, 768, 1000, 32, 32, 100.0, 0.5)])  # cfg3 at the reference batch: the largest footprint that fits
@pytest.mark.parametrize("optim", ["adamw", "sgd"])
def test_fused_step_f32_matches_the_separate_launches_and_the_oracle(case, optim):
    """uml_head_step_fused_f32 (one cooperative launch: logits, softmax CE, dW, optimizer update, statistics) against
    uml_head_fwd_ce_f32 + uml_head_bwd_dw_f32 on the same rows - G, per-row results and statistics to summation-order
    noise, the updated weights and moments - and the statistics against the oracle.  Two consecutive steps, so that
    the second one starts from moments the kernel wrote itself."""
    nib, ntb, d, c, bi, bt, scale, alpha = case
    xi, yi, xt, yt, w, g = _mk(sum(case[:6]) + 1, nib, ntb, d, d, c)
    dev = [t.to(DEV) for t in (xi, yi, xt, yt)]
    Wa, Wb = w.to(DEV), w.to(DEV)
    ma, va, mb, vb = (torch.zeros_like(Wa) for _ in range(4))
    wsa, wsb = ops.HeadWorkspace(bi + bt, c, DEV), ops.HeadWorkspace(bi + bt, c, DEV)
    st = O.HeadState(head=w.clone(), img_scale=scale, txt_scale=scale * 0.5)
    for step in (1, 2):
        ii = torch.randint(0, nib, (bi,), generator=g)
        it = torch.randint(0, ntb, (bt,), generator=g)
        runs = _runs(*dev, ii.to(DEV), it.to(DEV), scale, scale * 0.5, alpha)
        kw = dict(weight_decay=0.01) if optim == "adamw" else dict(weight_decay=0.01, momentum=0.9)
        ua = ops.make_update(optim, 2e-4, step, ma, va if optim == "adamw" else None, **kw)
        ub = ops.make_update(optim, 2e-4, step, mb, vb if optim == "adamw" else None, **kw)
        launched = ops.head_step_fused_f32(runs, Wa, wsa, ua)
        if (bi + bt) * (d + 4) * 4 > 200 * 1024:
            assert not launched, "the step's rows do not fit shared memory: the caller takes the separate launches"
            return
        assert launched, "these shapes fit the fused kernel's contract"
        ops.head_fwd_ce_f32(runs, Wb, wsb)
        Gb = wsb.G[: bi + bt, :c].clone()
        ops.head_bwd_dw_f32(runs, Wb, wsb, update=ub)
        torch.cuda.synchronize()
        n = bi + bt
        np.testing.assert_allclose(wsa.row_loss[:n].cpu().numpy(), wsb.row_loss[:n].cpu().numpy(), rtol=2e-5, atol=2e-5)
        assert torch.equal(wsa.row_correct[:n], wsb.row_correct[:n])
        ga, gb = wsa.G[:n, :c].cpu(), Gb.cpu()
        # (a logit's rounding noise is multiplied by the logit scale before the exponential: 1e-4 of the largest |G|)
        assert float((ga - gb).abs().max()) <= 1e-4 * max(1e-6, float(gb.abs().max()))
        sa, sb = wsa.read_stats(), wsb.read_stats()
        for k in range(len(runs)):
            assert math.isclose(sa[k]["loss_mean"], sb[k]["loss_mean"], rel_tol=2e-5, abs_tol=1e-5)
            assert sa[k]["correct"] == sb[k]["correct"] and sa[k]["n"] == sb[k]["n"]
            assert math.isclose(sa[k]["dscale"], sb[k]["dscale"], rel_tol=1e-4, abs_tol=1e-5)
        stats, _ = O.uml_step_grads(st, xi[ii] if bi else None, yi[ii] if bi else None, xt[it] if bt else None,
                                    yt[it] if bt else None, alpha)
        if step == 1:
            k = 0
            if bi:
                assert math.isclose(sa[k]["loss_mean"], stats["image_loss"], rel_tol=2e-5, abs_tol=1e-5)
                k += 1
            if bt:
                assert math.isclose(sa[k]["loss_mean"], stats["text_loss"], rel_tol=2e-5, abs_tol=1e-5)
        # Adam's first step is lr * sign(g): an element whose gradient is ~0 may flip between two summation orders
        diff = (Wa - Wb).abs()
        assert float(diff.max()) <= 2 * 2e-4 + 1e-7 and float((diff > 1e-6).float().mean()) < 1e-3
        assert float((ma - mb).abs().max()) <= 1e-4 * max(1e-6, float(mb.abs().max()))
        Wb.copy_(Wa); mb.copy_(ma); vb.copy_(va)   # the next step compares one step, not a drifting trajectory
