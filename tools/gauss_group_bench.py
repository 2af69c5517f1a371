"""Lock-step groups of Gaussian-experiment runs (gaussian.train_models_steps / GaussGroup, uml_gauss_group_run) against
the same runs trained one after the other by train_model_steps, at the reference's train.yaml size.

    python tools/gauss_group_bench.py [--steps 200] [--rounds 3] [--groups 1,6,16] [--out FILE]

Shape: dims 50 / 128 / 10, 10 000 rows per modality, batch 512, 2 000 validation rows, runs with their own seeds,
generators, modes, alphas and learning rates.  For every group size K, probes off and with eval_every = 1 (validation
MSE, CKA and mutual 10-NN after every step, main.py:67-84):
  * device: CUDA events around --steps steps of every run enqueued on a GaussGroup (index batches drawn beforehand,
    32 steps per library call), --rounds times alternating off / on;
  * call: the wall clock of one train_models_steps call of --steps steps (index draws, launches, the one read-back);
  * sequential: the wall clock of K train_model_steps calls of --steps steps each, one after the other.
Every time is reported per step of all K runs.  Prints one JSON line (and writes it to --out); the card's name and
power limit are read in the same run."""
import argparse
import json
import os
import sys
import time
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from sweep_adapter_bench import card  # noqa: E402

DIMS, N, BATCH, N_VAL = (50, 128, 10), 10_000, 512, 2_000


def make_runs(G, ds, K):
    models, loaders, opts, args = [], [], [], []
    for k in range(K):
        torch.manual_seed(k)
        m = G.SharedAutoencoder(*DIMS, device="cuda")
        models.append(m)
        opts.append(G.Adam(m, lr=(1e-3, 2e-3, 5e-4)[k % 3]))
        loaders.append(G.unpaired_loader(ds, BATCH, generator=torch.Generator().manual_seed(42 + k)))
        args.append(types.SimpleNamespace(mode="xy" if k % 4 else "x", alpha_x=1.0, alpha_y=(0.5, 1.0, 2.0)[k % 3]))
    return models, loaders, opts, args


def wall(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t


def run_k(G, ds, vx, vy, K, steps, rounds):
    res = {"runs": K}
    # ---------------- device: the same steps enqueued on two groups (probes off / on), alternating ----------------
    groups, batches = {}, {}
    for probes in (False, True):
        models, loaders, opts, args = make_runs(G, ds, K)
        groups[probes] = G.GaussGroup(models, opts, ds, BATCH, args, [vx] * K, [vy] * K)
        its = [iter(l) for l in loaders]
        rows = []
        for _ in range((rounds + 1) * steps):
            row = []
            for k in range(K):
                try:
                    row.append(next(its[k]).idx)
                except StopIteration:
                    its[k] = iter(loaders[k])
                    row.append(next(its[k]).idx)
            rows.append(row)
        batches[probes] = rows
    log = torch.zeros((steps, K, 2), device="cuda")
    elog = torch.zeros((steps, K, 4), device="cuda")

    def enqueue(probes, r):
        for i in range(0, steps, 32):
            n = min(32, steps - i)
            groups[probes].run(batches[probes][r * steps + i:r * steps + i + n], log[i:i + n],
                               elog[i:] if probes else None, 1 if probes else 0, i)

    for probes in (False, True):
        enqueue(probes, 0)  # warm-up
    dev_ms = {False: [], True: []}
    for r in range(1, rounds + 1):
        for probes in (False, True):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            enqueue(probes, r)
            e1.record()
            torch.cuda.synchronize()
            dev_ms[probes].append(round(e0.elapsed_time(e1) / steps, 4))
    res["device_step_ms_off"], res["device_step_ms_eval1"] = dev_ms[False], dev_ms[True]
    res["finite"] = bool(torch.isfinite(log).all() and torch.isfinite(elog).all())
    del groups, batches
    # ---------------- the public calls: one grouped call against K sequential single-run calls -------------------
    for probes, key in ((False, "off"), (True, "eval1")):
        kw = dict(val_data_x=vx, val_data_y=vy, eval_every=1) if probes else {}
        for warm in (True, False):
            n = 5 if warm else steps
            models, loaders, opts, args = make_runs(G, ds, K)
            t_group = wall(lambda: G.train_models_steps(models, loaders, opts, n, args=args, **kw))
            models, loaders, opts, args = make_runs(G, ds, K)
            t_seq = wall(lambda: [G.train_model_steps(models[k], loaders[k], opts[k], n, args=args[k], **kw)
                                  for k in range(K)])
        res[f"call_step_ms_{key}"] = round(1e3 * t_group / steps, 4)
        res[f"sequential_step_ms_{key}"] = round(1e3 * t_seq / steps, 4)
        res[f"speedup_{key}"] = round(t_seq / t_group, 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--groups", default="1,6,16")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gauss_group_bench needs a CUDA device")
    import uml_b200  # noqa: F401
    from uml_b200 import gaussian as G
    d = G.generate_data(dict(seed=42, num_samples=N + N_VAL, dim_c=10, dim_x=5, dim_y=5, dim_obs=DIMS[0], noise_std=0.09,
                             attenuate_x=True, attenuation=0.05, shared_latent_distribution_type="gaussian"))
    ds = G.UnpairedDataset(d["x"][:N], d["y"][:N], "cuda")
    vx, vy = d["x"][N:].cuda(), d["y"][N:].cuda()
    out = {"card": card(), "shape": dict(dims=DIMS, rows=N, batch=BATCH, n_val=N_VAL, steps=a.steps, rounds=a.rounds),
           "results": [run_k(G, ds, vx, vy, int(k), a.steps, a.rounds) for k in a.groups.split(",")]}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
