"""The linear analogue of the UML step: ``Gaussian_experiment`` of the reference (SURVEY §8 a-14).

Mirrors ``Gaussian_experiment/{model.py, dataset.py, data.py, main.py}``: a ``SharedAutoencoder`` whose
encoder/decoder are shared by two unpaired modalities, trained with ``alpha_x MSE(x) + alpha_y MSE(y)``
("xy") or ``MSE(x)`` ("x") and Adam.  The whole step (gather by sampler index, six layers forward, MSE,
six layers backward, Adam) runs in two hand-written kernels (``csrc/gauss.cu``); the per-step losses land
in a device log that is read once at the end.  Same names and argument meaning as the reference so its
``main.py`` reads the same against this module.  ``train_models_steps`` trains the combinations of the reference's
grid together (``GaussGroup``: up to 32 runs in lock step, two launches per step for all of them) and computes the
per-step validation MSE, CKA and mutual-kNN probes of the reference's loop (``main.py:67-84``) on the device.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from ._lib import check
from .engine.datasets.utils import BankLoader

LAYERS = ("in_head_x", "in_head_y", "shared_encoder.0", "shared_encoder.2",
          "shared_decoder.0", "shared_decoder.2", "out_head_x", "out_head_y")


def generate_data(config: Dict) -> Dict[str, torch.Tensor]:
    """``data.generate_data`` (data.py:29-61): shared latent (gaussian, centred, or laplace), private latents,
    observation noise, four random mixing matrices; X sees the shared latent attenuated except for its first
    10 % of dimensions.  Host-side torch draws in the reference's order, so the tensors are bit-identical."""
    seed, n = config["seed"], config["num_samples"]
    dim_c, dim_x, dim_y, dim_obs = config["dim_c"], config["dim_x"], config["dim_y"], config["dim_obs"]
    torch.manual_seed(seed)
    np.random.seed(seed)
    kind = config.get("shared_latent_distribution_type", "gaussian")
    if kind == "gaussian":
        tc = torch.randn(n, dim_c)
        tc = tc - tc.mean(0)
    elif kind == "laplace":
        tc = torch.distributions.Laplace(torch.tensor([0.0]), torch.tensor([1.0])).sample((n, dim_c)).squeeze(-1)
    else:
        raise ValueError(f"unknown shared_latent_distribution_type {kind!r}")
    tx, ty = torch.randn(n, dim_x), torch.randn(n, dim_y)
    nx, ny = torch.randn(n, dim_obs) * config["noise_std"], torch.randn(n, dim_obs) * config["noise_std"]
    a_c, a_x = torch.randn(dim_obs, dim_c), torch.randn(dim_obs, dim_x)
    b_c, b_y = torch.randn(dim_obs, dim_c), torch.randn(dim_obs, dim_y)
    if config.get("attenuate_x", False):
        att = torch.full((dim_c,), float(config["attenuation"]))
        att[: int(dim_c * 0.1)] = 1.0
        tcx = tc * att
    else:
        tcx = tc
    return {"x": tcx @ a_c.T + tx @ a_x.T + nx, "y": tc @ b_c.T + ty @ b_y.T + ny}


class UnpairedDataset:
    """``dataset.UnpairedDataset``: length = max of the two; item ``i`` pairs ``x[i % len_x]`` with ``y[i % len_y]``
    (the wrap is applied inside the kernel).  The rows live in HBM."""

    def __init__(self, data_x: torch.Tensor, data_y: torch.Tensor, device="cuda"):
        self.data_x = data_x.detach().to(device=device, dtype=torch.float32).contiguous()
        self.data_y = data_y.detach().to(device=device, dtype=torch.float32).contiguous()
        self.len_x, self.len_y = len(data_x), len(data_y)
        self.length = max(self.len_x, self.len_y)
        self.device = self.data_x.device

    def __len__(self):
        return self.length


def unpaired_loader(dataset: UnpairedDataset, batch_size: int, generator: Optional[torch.Generator] = None) -> BankLoader:
    """``DataLoader(dataset, batch_size, shuffle=True, drop_last=True, generator=g)`` (main.py:141-143) as an index
    loader with the same RNG protocol (explicit generator: one permutation per epoch plus the discarded trailing one)."""
    return BankLoader(dataset, batch_size, shuffle=True, drop_last=True, generator=generator)


class SharedAutoencoder:
    """``model.SharedAutoencoder(dim_obs, dim_common, dim_latent)``: parameters live in ONE flat CUDA buffer in the
    reference's construction order; ``state_dict`` uses the reference's keys.  Initialisation draws the same
    ``nn.Linear`` defaults from the global CPU generator in the same order as the reference constructor."""

    def __init__(self, dim_obs: int, dim_common: int, dim_latent: int, device="cuda"):
        self.dim_obs, self.dim_common, self.dim_latent = dim_obs, dim_common, dim_latent
        shapes = {"in_head_x": (dim_common, dim_obs), "in_head_y": (dim_common, dim_obs),
                  "shared_encoder.0": (dim_latent, dim_common), "shared_encoder.2": (dim_latent, dim_latent),
                  "shared_decoder.0": (dim_latent, dim_latent), "shared_decoder.2": (dim_common, dim_latent),
                  "out_head_x": (dim_obs, dim_common), "out_head_y": (dim_obs, dim_common)}
        # construction order of the reference: in heads, encoder (0, 2), decoder (0, 2), out heads
        host = {}
        for name in LAYERS:
            lin = torch.nn.Linear(shapes[name][1], shapes[name][0])
            host[name + ".weight"], host[name + ".bias"] = lin.weight.detach(), lin.bias.detach()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("SharedAutoencoder: parameters must live on a CUDA device (no CPU path)")
        n = int(_lib.load().uml_gauss_param_count(dim_obs, dim_common, dim_latent))
        self.flat = torch.empty(n, device=self.device)
        self._views, off = {}, 0
        for name in LAYERS:
            for suffix in (".weight", ".bias"):
                t = host[name + suffix]
                self._views[name + suffix] = self.flat[off:off + t.numel()].view(t.shape)
                self._views[name + suffix].copy_(t)
                off += t.numel()
        assert off == n

    def _bind(self, flat: torch.Tensor):
        """Move the parameters' home to ``flat`` (which already holds their values, e.g. a row of a GaussGroup slab)."""
        off = 0
        for name, t in list(self._views.items()):
            self._views[name] = flat[off:off + t.numel()].view(t.shape)
            off += t.numel()
        self.flat = flat

    def state_dict(self):
        return {k: v.detach().clone() for k, v in self._views.items()}

    def load_state_dict(self, sd):
        for k, v in self._views.items():
            v.copy_(sd[k].to(self.device))

    def parameters(self):
        return list(self._views.values())

    def train(self):
        return self

    def eval(self):
        return self

    def to(self, device):
        if torch.device(device).type != "cuda":
            raise RuntimeError("SharedAutoencoder has no CPU path")
        return self


class Adam:
    """``optim.Adam(model.parameters(), lr)`` with torch's defaults; state is two flat buffers next to the model's."""

    def __init__(self, model: SharedAutoencoder, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8):
        self.model, self.lr, self.betas, self.eps = model, float(lr), betas, float(eps)
        self.m, self.v = torch.zeros_like(model.flat), torch.zeros_like(model.flat)
        self.step_count = 0


def validate(model: SharedAutoencoder, val_data_x: torch.Tensor, val_data_y: torch.Tensor):
    """(val_loss_x, val_loss_y) = MSE of both reconstructions over the validation rows (main.py:68-72)."""
    x = val_data_x.to(device=model.device, dtype=torch.float32).contiguous()
    y = val_data_y.to(device=model.device, dtype=torch.float32).contiguous()
    if x.shape != y.shape:
        raise ValueError("validate: x and y validation sets must have the same shape")
    n = x.shape[0]
    ws = torch.empty(2 * ((n + 15) // 16), device=model.device)
    out = torch.empty(2, device=model.device)
    check(_lib.load().uml_gauss_eval(model.flat.data_ptr(), model.dim_obs, model.dim_common, model.dim_latent, x.data_ptr(),
                                     y.data_ptr(), n, ws.data_ptr(), out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    lx, ly = out.tolist()
    return lx, ly


def get_embeddings(model: SharedAutoencoder, x=None, y=None):
    """``model.get_embeddings`` of the reference (model.py:51-60): latent = shared_encoder(in_head(rows)) per modality,
    ``[n, dim_latent]`` device tensors (None for an absent modality)."""
    def prep(t):
        return None if t is None else t.to(device=model.device, dtype=torch.float32).contiguous()
    x, y = prep(x), prep(y)
    if x is None and y is None:
        return None, None
    n = (x if x is not None else y).shape[0]
    if x is not None and y is not None and x.shape[0] != y.shape[0]:
        raise ValueError("get_embeddings: x and y must have the same number of rows")
    ex = torch.empty((n, model.dim_latent), device=model.device) if x is not None else None
    ey = torch.empty((n, model.dim_latent), device=model.device) if y is not None else None
    check(_lib.load().uml_gauss_embed(model.flat.data_ptr(), model.dim_obs, model.dim_common, model.dim_latent,
                                      x.data_ptr() if x is not None else None, y.data_ptr() if y is not None else None, n,
                                      ex.data_ptr() if ex is not None else None, ey.data_ptr() if ey is not None else None,
                                      torch.cuda.current_stream().cuda_stream))
    return ex, ey


def alignment(model: SharedAutoencoder, val_data_x, val_data_y, topk: int = 10):
    """(cka, mknn) of the two modalities' validation embeddings - the probes main.py:21-29,78-83 logs as val/cka and
    val/mknn - computed on the device (``csrc/probes.cu``); one read-back of two floats."""
    from . import ops
    ex, ey = get_embeddings(model, val_data_x, val_data_y)
    both = torch.cat([ops.cka_linear(ex, ey), ops.mutual_knn(ex, ey, topk)]).tolist()
    return both[0], both[1]


def train_model_steps(model: SharedAutoencoder, data_loader: BankLoader, optimizer: Adam, num_steps: int,
                      val_data_x=None, val_data_y=None, device="cuda", args=None, eval_every: int = 0, trace=None):
    """``main.train_model_steps`` (main.py:31-86).  ``args`` carries ``mode`` ('xy' | 'x'), ``alpha_x``, ``alpha_y``.
    Returns ``{'loss_x': [...], 'loss_y': [...], 'loss': [...], 'val': [(step, val_x, val_y), ...], 'align': [(step, cka,
    mknn), ...]}``; the
    training losses are read back from the device log once, after the last step (or at validation points)."""
    mode = getattr(args, "mode", "xy")
    alpha_x, alpha_y = float(getattr(args, "alpha_x", 1.0)), float(getattr(args, "alpha_y", 1.0))
    if mode not in ("xy", "x"):
        raise ValueError("mode must be 'xy' or 'x'")
    ds: UnpairedDataset = data_loader.bank
    lib = _lib.load()
    B = data_loader.batch_size
    ws = torch.empty(int(lib.uml_gauss_workspace_floats(model.dim_obs, model.dim_common, model.dim_latent, B)), device=model.device)
    log = torch.zeros((num_steps, 2), device=model.device)
    stream = torch.cuda.current_stream().cuda_stream
    import ctypes as C
    it = iter(data_loader)
    out = {"loss_x": [], "loss_y": [], "loss": [], "val": [], "align": []}
    chunk_max = 32  # steps enqueued per library call (a Python round trip per step costs more than the step's kernels)
    step = 0
    while step < num_steps:
        n = min(chunk_max, num_steps - step)
        if eval_every and val_data_x is not None:
            n = min(n, eval_every - step % eval_every)  # a chunk ends at the next validation point
        batches = []
        for _ in range(n):
            try:
                batch = next(it)
            except StopIteration:
                it = iter(data_loader)
                batch = next(it)
            if trace is not None:
                trace.setdefault("idx", []).append(batch.host_idx.clone())
            batches.append(batch)
        ptrs = (C.c_void_p * n)(*[b.idx.data_ptr() for b in batches])
        check(lib.uml_gauss_run(model.flat.data_ptr(), optimizer.m.data_ptr(), optimizer.v.data_ptr(), model.dim_obs,
                                model.dim_common, model.dim_latent, ds.data_x.data_ptr(), ds.len_x, ds.data_y.data_ptr(),
                                ds.len_y, ptrs, n, B, int(mode == "xy"), alpha_x, alpha_y, optimizer.lr, optimizer.betas[0],
                                optimizer.betas[1], optimizer.eps, optimizer.step_count + 1, ws.data_ptr(),
                                log[step].data_ptr(), stream))
        optimizer.step_count += n
        step += n
        if eval_every and val_data_x is not None and step % eval_every == 0:
            out["val"].append((step - 1,) + validate(model, val_data_x, val_data_y))
            # val/cka and val/mknn of the validation embeddings, as the reference logs them at every evaluation point
            out["align"].append((step - 1,) + alignment(model, val_data_x, val_data_y))
    host = log.cpu()
    out["loss_x"], out["loss_y"] = host[:, 0].tolist(), host[:, 1].tolist()
    out["loss"] = [(alpha_x * a + alpha_y * b) if mode == "xy" else a for a, b in zip(out["loss_x"], out["loss_y"])]
    return out


# ------------------------------------------------------------------------------------------ grid of runs in lock step

GROUP_MAX_RUNS = _lib.GAUSS_GROUP_MAX_RUNS
PROBE_TOPK = 10           # mutual-kNN neighbours of the reference's probe (main.py:21-29)
GROUP_CHUNK_STEPS = 32    # steps enqueued per library call (bounds the index batches held on the host)


def _run_mode(a):
    mode = getattr(a, "mode", "xy")
    if mode not in ("xy", "x"):
        raise ValueError("mode must be 'xy' or 'x'")
    return mode, float(getattr(a, "alpha_x", 1.0)), float(getattr(a, "alpha_y", 1.0))


def _per_run(val, k: int):
    """A validation tensor shared by every run, or one per run -> a list of k (None: no validation)."""
    if val is None:
        return None
    vals = list(val) if isinstance(val, (list, tuple)) else [val] * k
    if len(vals) != k:
        raise ValueError(f"{len(vals)} validation sets for {k} runs")
    return vals


def _data_key(ds):
    return (ds.data_x.data_ptr(), ds.data_y.data_ptr(), ds.len_x, ds.len_y, ds.data_x.shape[1])


def group_blockers(models, data_loaders, optimizers, val_data_x=None, val_data_y=None):
    """Reasons why these runs cannot train as one ``GaussGroup`` (empty list: they can).  ``val_data_*``: one tensor per
    run (see ``_per_run``) or None."""
    why = []
    k = len(models)
    if k == 0:
        return ["no runs"]
    if k > GROUP_MAX_RUNS:
        why.append(f"more than {GROUP_MAX_RUNS} runs ({k})")
    if len(data_loaders) != k or len(optimizers) != k:
        return why + ["one data loader and one optimizer per model"]
    devices = {m.flat.device for m in models}
    if any(d.type != "cuda" for d in devices):
        why.append("a model not on CUDA")
    elif len(devices | {l.bank.data_x.device for l in data_loaders}) > 1:
        why.append("models and datasets on different devices")
    if len({(m.dim_obs, m.dim_common, m.dim_latent) for m in models}) > 1:
        why.append("different model dims")
    if len({_data_key(l.bank) for l in data_loaders}) > 1 or len({l.batch_size for l in data_loaders}) > 1:
        why.append("different datasets or batch sizes")
    if not all(l.shuffle and l.drop_last for l in data_loaders):
        why.append("loaders without drop_last / shuffle")
    if any(l.shard_of is not None for l in data_loaders):
        why.append("data-parallel shard loaders")
    if k > 1:
        gens = [l.generator if l.generator is not None else l.rng for l in data_loaders]
        if any(g is None for g in gens):
            why.append("loaders that draw from the global generator (each run needs its own, as in the reference)")
        elif len({id(g) for g in gens}) < k:
            why.append("loaders that share one generator object (seed one per run)")
    if any(o.model is not m for o, m in zip(optimizers, models)):
        why.append("an optimizer that does not belong to its model")
    if len({(tuple(o.betas), o.eps, o.step_count) for o in optimizers}) > 1:
        why.append("optimizers with different betas, eps or step counts")
    if (val_data_x is None) != (val_data_y is None):
        why.append("validation rows of one modality only")
    elif val_data_x is not None:
        shapes = {tuple(t.shape) for t in list(val_data_x) + list(val_data_y)}
        if len(shapes) > 1 or len(next(iter(shapes))) != 2 or next(iter(shapes))[1] != models[0].dim_obs:
            why.append("validation sets of different shapes")
    return why


class GaussGroup:
    """Runs of one ``SharedAutoencoder`` shape over one ``UnpairedDataset`` trained in lock step (``uml_gauss_group_run``,
    ``csrc/gauss.cu``): one step of every run is two launches, and run k computes bit for bit what ``train_model_steps``
    computes for it alone.  The group owns [K, P] slabs of parameters and Adam moments; each model's ``flat`` (and its
    parameter views) and each optimizer's ``m`` / ``v`` become rows of them, so ``state_dict()``, ``validate()`` and
    ``alignment()`` keep working on every model during and after training.  ``active[k] = False`` freezes run k: the
    library touches nothing of it."""

    def __init__(self, models, optimizers, dataset: UnpairedDataset, batch_size: int, args=None, val_data_x=None,
                 val_data_y=None, topk: int = PROBE_TOPK):
        self.K = len(models)
        self.models, self.optimizers, self.dataset, self.batch_size = list(models), list(optimizers), dataset, int(batch_size)
        self.modes = [_run_mode(a) for a in (args if args is not None else [None] * self.K)]
        m0 = models[0]
        self.device = m0.flat.device
        self.params = torch.stack([m.flat.detach() for m in models])
        self.m = torch.stack([o.m for o in optimizers])
        self.v = torch.stack([o.v for o in optimizers])
        for k, (model, opt) in enumerate(zip(models, optimizers)):
            model._bind(self.params[k])
            opt.m, opt.v = self.m[k], self.v[k]
        self.active = [True] * self.K
        self.step = optimizers[0].step_count   # Adam steps taken (shared by the runs)
        self.topk = int(topk)
        self.val_x = self.val_y = None
        n_val = 0
        if val_data_x is not None:
            prep = lambda t: t.to(device=self.device, dtype=torch.float32).contiguous()
            self.val_x, self.val_y = [prep(t) for t in val_data_x], [prep(t) for t in val_data_y]
            n_val = self.val_x[0].shape[0]
        self.n_val = n_val
        lib = _lib.load()
        nbytes = int(lib.uml_gauss_group_workspace_bytes(self.K, m0.dim_obs, m0.dim_common, m0.dim_latent, self.batch_size,
                                                         n_val, self.topk if n_val else 0))
        self.workspace = torch.empty(nbytes, dtype=torch.uint8, device=self.device)

    def run(self, idx, loss_log: torch.Tensor, eval_log: Optional[torch.Tensor] = None, eval_every: int = 0,
            eval_phase: int = 0) -> int:
        """Enqueue len(idx) steps of every active run; no host synchronisation.  ``idx[i][k]``: run k's device index batch
        of step i (ignored for an inactive run); ``loss_log``: [steps, K, 2] device tensor; with ``eval_every`` the probes
        of every step i with (eval_phase + i + 1) % eval_every == 0 go to the next rows of ``eval_log`` [rows, K, 4]
        ({val_loss_x, val_loss_y, cka, mknn}).  Returns the number of evaluations enqueued."""
        n = len(idx)
        K = self.K
        if loss_log.dtype != torch.float32 or not loss_log.is_contiguous() or tuple(loss_log.shape) != (n, K, 2):
            raise ValueError(f"loss_log must be a contiguous float32 [{n}, {K}, 2] tensor")
        evals = (eval_phase + n) // eval_every - eval_phase // eval_every if eval_every else 0
        if evals:
            if self.val_x is None:
                raise ValueError("probes need the group's validation rows")
            if eval_log is None or eval_log.dtype != torch.float32 or not eval_log.is_contiguous() or \
                    eval_log.dim() != 3 or eval_log.shape[0] < evals or tuple(eval_log.shape[1:]) != (K, 4):
                raise ValueError(f"eval_log must be a contiguous float32 [>= {evals}, {K}, 4] tensor")
        m0, o0, ds = self.models[0], self.optimizers[0], self.dataset
        a = _lib.GaussGroupArgs()
        a.n_runs, a.dim_obs, a.dim_common, a.dim_latent = K, m0.dim_obs, m0.dim_common, m0.dim_latent
        a.data_x, a.n_x, a.data_y, a.n_y = ds.data_x.data_ptr(), ds.len_x, ds.data_y.data_ptr(), ds.len_y
        a.batch = self.batch_size
        a.params, a.adam_m, a.adam_v = self.params.data_ptr(), self.m.data_ptr(), self.v.data_ptr()
        a.param_stride = self.params.stride(0)
        a.beta1, a.beta2, a.eps = o0.betas[0], o0.betas[1], o0.eps
        a.first_step = self.step + 1
        for k in range(K):
            mode, ax, ay = self.modes[k]
            a.mode_xy[k], a.alpha_x[k], a.alpha_y[k] = int(mode == "xy"), ax, ay
            a.lr[k] = self.optimizers[k].lr
            a.active[k] = int(bool(self.active[k]))
        a.loss_log = loss_log.data_ptr()
        if evals:
            a.eval_every, a.topk, a.eval_phase, a.n_val = int(eval_every), self.topk, int(eval_phase), self.n_val
            for k in range(K):
                a.val_x[k], a.val_y[k] = self.val_x[k].data_ptr(), self.val_y[k].data_ptr()
            a.eval_log = eval_log.data_ptr()
        a.workspace, a.workspace_bytes = self.workspace.data_ptr(), self.workspace.numel()
        ptrs = (C.c_void_p * (n * K))(*[idx[i][k].data_ptr() if self.active[k] else None for i in range(n) for k in range(K)])
        check(_lib.load().uml_gauss_group_run(C.byref(a), n, ptrs, torch.cuda.current_stream(self.device).cuda_stream))
        _lib.LAUNCH_COUNT[0] += 2 * n + 8 * evals
        self.step += n
        for k in range(K):
            if self.active[k]:
                self.optimizers[k].step_count += n
        return evals


def train_models_steps(models, data_loaders, optimizers, num_steps: int, val_data_x=None, val_data_y=None, args=None,
                       eval_every: int = 0, traces=None):
    """``train_model_steps`` for several runs at once - the combinations of the reference's grid (main.py), which it
    trains one after the other - in lock step on one ``GaussGroup``.  ``args``: one namespace per run (``mode``,
    ``alpha_x``, ``alpha_y``); ``val_data_x`` / ``val_data_y``: one validation set for all runs or a list of one per run;
    ``traces``: optional list of per-run dicts (as ``trace`` of ``train_model_steps``).  Returns one dict per run in the
    format of ``train_model_steps``, and run k's numbers, weights and Adam state are bit-identical to training it alone.
    With ``eval_every`` the validation MSE, CKA and mutual kNN are computed on the device after every eval_every-th step;
    the logs are read back once, at the end.  Raises ``ValueError`` naming every reason the runs cannot share a group."""
    K = len(models)
    args = list(args) if args is not None else [None] * K
    if len(args) != K:
        raise ValueError(f"{len(args)} args namespaces for {K} runs")
    modes = [_run_mode(a) for a in args]
    vx, vy = _per_run(val_data_x, K), _per_run(val_data_y, K)
    why = group_blockers(models, data_loaders, optimizers, vx, vy)
    if why:
        raise ValueError("train_models_steps: these runs cannot train as one group: " + "; ".join(why))
    probes = bool(eval_every) and vx is not None
    group = GaussGroup(models, optimizers, data_loaders[0].bank, data_loaders[0].batch_size, args,
                       vx if probes else None, vy if probes else None)
    n_evals = num_steps // eval_every if probes else 0
    dev = group.device
    log = torch.zeros((num_steps, K, 2), device=dev)
    elog = torch.zeros((max(n_evals, 1), K, 4), device=dev)
    its = [iter(l) for l in data_loaders]
    step = done = 0
    while step < num_steps:
        n = min(GROUP_CHUNK_STEPS, num_steps - step)
        batches = []
        for _ in range(n):
            row = []
            for k in range(K):  # each loader advances exactly as in its own run: one batch per step, new epoch when empty
                try:
                    b = next(its[k])
                except StopIteration:
                    its[k] = iter(data_loaders[k])
                    b = next(its[k])
                if traces is not None and traces[k] is not None:
                    traces[k].setdefault("idx", []).append(b.host_idx.clone())
                row.append(b)
            batches.append(row)
        done += group.run([[b.idx for b in row] for row in batches], log[step:step + n], elog[done:] if probes else None,
                          eval_every if probes else 0, step)
        step += n
    host, ehost = log.cpu(), elog.cpu()
    outs = []
    for k, (mode, alpha_x, alpha_y) in enumerate(modes):
        out = {"loss_x": host[:, k, 0].tolist(), "loss_y": host[:, k, 1].tolist(), "val": [], "align": []}
        out["loss"] = [(alpha_x * a + alpha_y * b) if mode == "xy" else a for a, b in zip(out["loss_x"], out["loss_y"])]
        for e in range(n_evals):
            vl_x, vl_y, cka, mknn = ehost[e, k].tolist()
            out["val"].append(((e + 1) * eval_every - 1, vl_x, vl_y))
            out["align"].append(((e + 1) * eval_every - 1, cka, mknn))
        outs.append(out)
    return outs
