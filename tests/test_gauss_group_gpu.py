"""a-14 grid: runs of the Gaussian experiment trained in lock step (gaussian.train_models_steps / GaussGroup, csrc/gauss.cu
uml_gauss_group_run) against the same runs trained alone by train_model_steps - bit for bit: losses, final weights,
Adam moments, sampler streams and the per-step probes - and run 0 of a group against the golden trace of the
unmodified reference (tests/golden/misc.npz)."""
import ast
import os
import types

import numpy as np
import pytest
import torch

from oracle import metrics_oracle as M

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DEV = "cuda:0"

if torch.cuda.is_available():
    import uml_b200  # noqa: F401
    from uml_b200 import gaussian as G


def _data(n, seed=42):
    return G.generate_data(dict(seed=seed, num_samples=n, dim_c=10, dim_x=5, dim_y=5, dim_obs=50, noise_std=0.09,
                                attenuate_x=True, attenuation=0.05, shared_latent_distribution_type="gaussian"))


def _spec(seed, gen, lr=1e-3, mode="xy", ax=1.0, ay=1.0):
    return dict(seed=seed, gen=gen, lr=lr, mode=mode, ax=ax, ay=ay)


def _build(specs, ds, batch, dims):
    """Each run as its own script would make it: model weights from torch.manual_seed(seed), a loader with its own
    Generator(gen), Adam(lr)."""
    models, loaders, opts, args = [], [], [], []
    for sp in specs:
        torch.manual_seed(sp["seed"])
        m = G.SharedAutoencoder(*dims, device=DEV)
        models.append(m)
        opts.append(G.Adam(m, lr=sp["lr"]))
        loaders.append(G.unpaired_loader(ds, batch, generator=torch.Generator().manual_seed(sp["gen"])))
        args.append(types.SimpleNamespace(mode=sp["mode"], alpha_x=sp["ax"], alpha_y=sp["ay"]))
    return models, loaders, opts, args


def _group(specs, ds, batch, dims, steps, **kw):
    models, loaders, opts, args = _build(specs, ds, batch, dims)
    traces = [{} for _ in specs]
    outs = G.train_models_steps(models, loaders, opts, steps, args=args, traces=traces, **kw)
    return [dict(model=m, opt=o, out=out, trace=t) for m, o, out, t in zip(models, opts, outs, traces)]


def _alone(sp, ds, batch, dims, steps, **kw):
    (m,), (l,), (o,), (a,) = _build([sp], ds, batch, dims)
    trace = {}
    out = G.train_model_steps(m, l, o, steps, args=a, trace=trace, **kw)
    return dict(model=m, opt=o, out=out, trace=trace)


def _assert_same(got, want, what=""):
    for key in ("loss_x", "loss_y", "loss", "val", "align"):
        assert got["out"][key] == want["out"][key], (what, key)
    assert len(got["trace"]["idx"]) == len(want["trace"]["idx"])
    for a, b in zip(got["trace"]["idx"], want["trace"]["idx"]):
        assert torch.equal(a, b), what
    sg, sw = got["model"].state_dict(), want["model"].state_dict()
    for k in sw:
        assert torch.equal(sg[k], sw[k]), (what, k)
    assert torch.equal(got["opt"].m, want["opt"].m) and torch.equal(got["opt"].v, want["opt"].v), what
    assert got["opt"].step_count == want["opt"].step_count, what


GOLDEN_SPECS = [_spec(0, 42, 1e-3, "xy", 1.0, 0.5), _spec(1, 7, 1e-3, "x"), _spec(2, 8, 3e-3, "xy", 1.0, 2.0),
                _spec(3, 9, 5e-4, "x", 0.7, 0.3)]
YAML_SPECS = [_spec(0, 42, 1e-3, "xy"), _spec(1, 42, 1e-3, "x"), _spec(2, 43, 1e-3, "xy", 1.0, 0.1),
              _spec(3, 44, 2e-3, "xy", 1.0, 10.0), _spec(4, 45, 5e-4, "x", 1.0, 0.5), _spec(5, 46, 1e-2, "xy", 0.5, 1.0)]


@pytest.mark.parametrize("size", ["golden", "train_yaml"])
def test_group_runs_are_bit_identical_to_runs_alone(size):
    if size == "golden":  # the golden trace's shapes: dims 12 / 16 / 6, batch 16; 40 steps cross epochs and chunks
        m = np.load(os.path.join(GOLDEN, "misc.npz"), allow_pickle=False)
        cfg = ast.literal_eval(str(m["gauss/cfg"]))
        d = G.generate_data(dict(seed=cfg["seed"], num_samples=cfg["num_samples"], dim_c=cfg["dim_c"], dim_x=cfg["dim_x"],
                                 dim_y=cfg["dim_y"], dim_obs=cfg["dim_obs"], noise_std=cfg["noise_std"], attenuate_x=True,
                                 attenuation=cfg["attenuation"], shared_latent_distribution_type="gaussian"))
        ds, batch, dims, steps, specs = G.UnpairedDataset(d["x"][:48], d["y"][:40], DEV), 16, (12, 16, 6), 40, GOLDEN_SPECS
    else:  # train.yaml: N 10 000, batch 512, dims 50 / 128 / 10, 200 steps, K = 6
        d = _data(10000)
        ds, batch, dims, steps, specs = G.UnpairedDataset(d["x"], d["y"], DEV), 512, (50, 128, 10), 200, YAML_SPECS
    group = _group(specs, ds, batch, dims, steps)
    for k, sp in enumerate(specs):
        _assert_same(group[k], _alone(sp, ds, batch, dims, steps), f"run {k}")
    # "x" mode: the y heads of those runs were never touched
    for k, sp in enumerate(specs):
        if sp["mode"] == "x":
            torch.manual_seed(sp["seed"])
            fresh = G.SharedAutoencoder(*dims, device=DEV).state_dict()
            for key in ("in_head_y.weight", "in_head_y.bias", "out_head_y.weight", "out_head_y.bias"):
                assert torch.equal(group[k]["model"].state_dict()[key], fresh[key])


@pytest.mark.parametrize("mode", ["xy", "x"])
def test_run0_of_a_group_matches_reference_trace(mode):
    """tests/test_gaussian_gpu.py::test_gaussian_step_matches_reference_trace with the golden run as run 0 of a group."""
    m = np.load(os.path.join(GOLDEN, "misc.npz"), allow_pickle=False)
    cfg = ast.literal_eval(str(m["gauss/cfg"]))
    base = dict(seed=cfg["seed"], num_samples=cfg["num_samples"], dim_c=cfg["dim_c"], dim_x=cfg["dim_x"], dim_y=cfg["dim_y"],
                dim_obs=cfg["dim_obs"], noise_std=cfg["noise_std"], attenuate_x=True, attenuation=cfg["attenuation"])
    d1 = G.generate_data(dict(base, shared_latent_distribution_type="gaussian"))
    d2 = G.generate_data(dict(base, seed=44, shared_latent_distribution_type="laplace"))
    dx, dy = (d1["x"][:32], d1["y"][:32]) if mode == "xy" else (d1["x"], d2["y"][:40])
    ds = G.UnpairedDataset(dx, dy, DEV)
    specs = [_spec(3, 42, 1e-3, mode, 1.0, 0.5), _spec(5, 1, 2e-3, "xy", 1.0, 1.0), _spec(6, 2, 1e-3, "x")]
    group = _group(specs, ds, 16, (12, 16, 6), 9)
    hist, model = group[0]["out"], group[0]["model"]
    np.testing.assert_allclose(hist["loss_x"], m[f"gauss/{mode}/loss_x"], rtol=2e-5)
    np.testing.assert_allclose(hist["loss_y"], m[f"gauss/{mode}/loss_y"], rtol=2e-5)
    for k, v in model.state_dict().items():
        np.testing.assert_allclose(v.cpu().numpy(), m[f"gauss/{mode}/final/{k}"], rtol=2e-4, atol=2e-6, err_msg=k)


def _yaml_case(n=3000):
    d = _data(n + 2000)
    return d, G.UnpairedDataset(d["x"][:n], d["y"][:n - 100], DEV), 512, (50, 128, 10)


def test_twins_and_slots():
    d, ds, batch, dims = _yaml_case()
    a, b, c = _spec(0, 42, 1e-3, "xy", 1.0, 0.5), _spec(1, 43, 2e-3, "x"), _spec(2, 44, 5e-4, "xy", 1.0, 3.0)
    g1 = _group([a, b, a, c], ds, batch, dims, 45)
    _assert_same(g1[2], g1[0], "twins")
    g2 = _group([c, a, b], ds, batch, dims, 45)   # the same runs in other slots
    _assert_same(g2[1], g1[0], "run a in slot 1")
    _assert_same(g2[2], g1[1], "run b in slot 2")
    _assert_same(g2[0], g1[3], "run c in slot 0")


def test_an_inactive_run_is_untouched():
    d, ds, batch, dims = _yaml_case()
    specs = [_spec(0, 42), _spec(1, 43, 2e-3, "x"), _spec(2, 44)]
    models, loaders, opts, args = _build(specs, ds, batch, dims)
    grp = G.GaussGroup(models, opts, ds, batch, args, [d["x"][3000:]] * 3, [d["y"][3000:]] * 3)
    def batches(loader):  # epoch after epoch, as train_model_steps draws them
        while True:
            yield from loader
    its = [batches(l) for l in loaders]
    first = [[next(it).idx for it in its] for _ in range(3)]
    grp.run(first, torch.zeros((3, 3, 2), device=DEV))
    grp.active[1] = False
    frozen = [t[1].clone() for t in (grp.params, grp.m, grp.v)]
    log = torch.full((6, 3, 2), -7.0, device=DEV)
    elog = torch.full((3, 3, 4), -7.0, device=DEV)
    idx = [[next(it).idx for it in its] for _ in range(6)]
    assert grp.run(idx, log, elog, eval_every=2) == 3
    torch.cuda.synchronize()
    for t, f in zip((grp.params, grp.m, grp.v), frozen):
        assert torch.equal(t[1], f)
    assert (log[:, 1] == -7).all() and (elog[:, 1] == -7).all()
    assert (log[:, [0, 2]] != -7).all() and (elog[:, [0, 2]] != -7).all()
    assert [o.step_count for o in opts] == [9, 3, 9]
    # the model and optimizer objects see the slab rows
    assert models[0].flat.data_ptr() == grp.params[0].data_ptr() and opts[2].v.data_ptr() == grp.v[2].data_ptr()
    assert G.validate(models[0], d["x"][3000:], d["y"][3000:]) == tuple(elog[2, 0, :2].tolist())


@pytest.mark.parametrize("eval_every", [1, 7])
def test_probes_equal_validate_and_alignment_after_each_step(eval_every):
    d, ds, batch, dims = _yaml_case()
    steps = 14 if eval_every == 1 else 23
    specs = [_spec(0, 42, 1e-3, "xy", 1.0, 0.5), _spec(1, 43, 2e-3, "x"), _spec(2, 44, 1e-3, "xy", 1.0, 2.0)]
    vx, vy = d["x"][3000:], d["y"][3000:]   # 2000 validation rows, as the reference's
    if eval_every == 7:  # validation sets of their own per run (same shape)
        vx, vy = [vx, d["x"][1000:3000], vx], [vy, d["y"][1000:3000], vy]
    group = _group(specs, ds, batch, dims, steps, val_data_x=vx, val_data_y=vy, eval_every=eval_every)
    for k, sp in enumerate(specs):
        vxk, vyk = (vx[k], vy[k]) if isinstance(vx, list) else (vx, vy)
        # the single run evaluates validate() / alignment() on its weights after every eval_every-th step
        alone = _alone(sp, ds, batch, dims, steps, val_data_x=vxk, val_data_y=vyk, eval_every=eval_every)
        assert [s for s, _, _ in group[k]["out"]["val"]] == [e * eval_every - 1 for e in range(1, steps // eval_every + 1)]
        _assert_same(group[k], alone, f"run {k}")
        # ... and against the oracle's formulas on the last evaluated weights
        if steps % eval_every == 0:
            ex, ey = G.get_embeddings(group[k]["model"], vxk, vyk)
            _, cka, mknn = group[k]["out"]["align"][-1]
            want_cka, want_mknn = M.cka_linear_features(ex.cpu(), ey.cpu()), M.mutual_knn(ex.cpu(), ey.cpu(), 10)
            assert abs(cka - want_cka) <= 2e-4 * max(1.0, abs(want_cka)), (cka, want_cka)
            assert abs(mknn - want_mknn) <= 3.0 / (ex.shape[0] * 10) + 1e-7, (mknn, want_mknn)
