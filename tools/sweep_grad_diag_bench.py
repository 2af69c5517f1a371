"""Per-step gradient diagnostics of batched sweep groups (uml_sweep_run_diag: the reference's four gradient probes of
every head on the device, two launches per step) - what they add to a step of K heads.

    python tools/sweep_grad_diag_bench.py [--steps 100] [--warmup 20] [--rounds 3] [--out FILE]

Shapes: cfg2 (UMLClip heads, D 512, C 1000) with K = 6 and 30, cfg4 (UML heads with adapter and learnable
temperatures, Dv 1536, D 3200, C 1000) with K = 30; 32 + 32 rows per step, 16 000 image and 29 940 text bank rows.
Arms, in one process:
  * device: CUDA events over --steps steps of a group without and a group with diagnostics (identical heads),
    alternating --rounds times; the last step's per-launch breakdown, including the diagnostics launches alone;
  * e2e: one public train_group() call without and with diagnostics (the wall clock of its last --steps iterations,
    the per-step probes read back with the losses).
Work of the diagnostics launches per step: the two contractions A = X_img^T G_img and B = X_txt^T G_txt over all rows,
2 K R C D FLOP, three tf32 MMAs per product (3xTF32), and the X and G bytes they must read at least once, K R (D + C) 4.
Prints one JSON line (and writes it to --out): card name and power limit are read in the same run."""
import argparse
import contextlib
import io
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench import build_banks  # noqa: E402
from sweep_adapter_bench import card  # noqa: E402

SHAPES = {
    "cfg2": dict(n_img=16_000, n_txt=29_940, dim=512, classes=1000, batch=32, batch_txt=32, n_val=1000, adapter=False),
    "cfg4": dict(n_img=16_000, n_txt=29_940, dv=1536, dim=3200, classes=1000, batch=32, batch_txt=32, n_val=1000,
                 adapter=True),
}


def run_shape(name, K, steps, warmup, rounds):
    import uml_b200  # noqa: F401
    from uml_b200 import finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader
    from uml_b200.engine.models.head import UML, UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler
    from uml_b200.engine.sweep import AdapterHeadGroup, HeadGroup

    wl = SHAPES[name]
    dev = torch.device("cuda", 0)
    img_bank, txt_bank, val_bank, _ = build_banks(wl, dev)
    D, C, B, BT = wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    grid = [(lr, wd, al) for al in (0.2, 0.5, 1.0, 1.5, 2.0) for lr in (1e-3, 1e-4) for wd in (0.0, 0.01, 0.0001)]
    grid = [grid[k % len(grid)] for k in range(K)]
    alphas = [g[2] for g in grid]
    Group = AdapterHeadGroup if wl["adapter"] else HeadGroup

    def make_heads(n):
        ms, os_, ss, il, tl, vl = [], [], [], [], [], []
        with contextlib.redirect_stdout(io.StringIO()):
            for k in range(n):
                lr, wd, _ = grid[k]
                torch.manual_seed(k)
                if wl["adapter"]:
                    m = UML(f"synthetic:{wl['dv']}", D, C, learnable_temp=True)
                else:
                    m = UMLClip(f"synthetic:{D}", C, logit_scale_init=4.60517)
                m.precision = "fp32"
                m.to(dev)
                o = build_optimizer(m.parameters(), "adamw", lr, wd)
                rng = torch.Generator().manual_seed(100 + k)
                ms.append(m)
                os_.append(o)
                ss.append(build_lr_scheduler(o, "cosine", 50, 12800, warmup_type="linear", warmup_lr=1e-5))
                il.append(BankLoader(img_bank, B, shuffle=True, rng=rng))
                tl.append(BankLoader(txt_bank, BT, shuffle=True, rng=rng))
                vl.append(BankLoader(val_bank, 32, shuffle=False, rng=rng))
        return ms, os_, ss, il, tl, vl

    # ---------------- device-resident arm: the same steps with and without diagnostics, alternating ---------------
    groups, heads = {}, {}
    for diag in (False, True):
        heads[diag] = make_heads(K)
        ms_, os_ = heads[diag][:2]
        groups[diag] = Group(ms_, os_, img_bank, txt_bank, B, BT, dev, log_slots=warmup + steps + 1, grad_diagnostics=diag)
    il, tl, ss = heads[False][3], heads[False][4], heads[False][2]
    assert warmup + steps <= min(len(il[0]), len(tl[0])), "warm-up + steps must stay inside one epoch"
    iti, itt = [iter(l) for l in il], [iter(l) for l in tl]
    pi = [it.take_run(warmup + steps) for it in iti]
    pt = [it.take_run(warmup + steps) for it in itt]
    perms_i, perms_t, p0i, p0t = [p[0] for p in pi], [p[0] for p in pt], pi[0][1], pt[0][1]
    lrs = [[s.lr_at(j, s.base_lrs[0]) for s in ss] for j in range(warmup + steps)]

    def enqueue(group, first, n):  # one library call per 16 steps, like train_group's chunks
        i = first
        while i < first + n:
            m = min(16, first + n - i)
            group.run(perms_i, perms_t, p0i + i * B, p0t + i * BT, [(B, BT)] * m, lrs[i:i + m], alphas, [True] * K,
                      slot0=i)
            i += m

    for diag in (False, True):
        enqueue(groups[diag], 0, warmup)
        groups[diag].time_last_step()
    step_ms = {False: [], True: []}
    ktimes = {}
    for _ in range(rounds):
        for diag in (False, True):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            enqueue(groups[diag], warmup, steps)
            e1.record()
            torch.cuda.synchronize()
            step_ms[diag].append(e0.elapsed_time(e1) / steps)
            ktimes[diag] = groups[diag].kernel_times_ms()
    tail = groups[True].read_log([warmup + steps - 1], True, True)["grad_diag"][0]
    finite = all(all(v == v and abs(v) != float("inf") for v in d.values()) for d in tail)
    del groups, heads
    torch.cuda.empty_cache()

    # ---------------- end-to-end arm: one public train_group() call without and with diagnostics ------------------
    e2e = {}
    for diag in (False, True):
        ms2, os2, ss2, il2, tl2, vl2 = make_heads(K)
        trs = [None] * K
        trs[0] = {"indices": False, "timing": {"warmup": warmup}, "grad_diagnostics": diag}
        with contextlib.redirect_stdout(io.StringIO()):
            ft.train_group(ms2, il2, tl2, vl2, None, os2, ss2, device=dev, max_iters=warmup + steps, alphas=alphas,
                           eval_freq=10 ** 9, patience=5, traces=trs)
        e2e[diag] = trs[0]["timing"]["seconds"] * 1e3 / trs[0]["timing"]["iters"]
        del ms2, os2
        torch.cuda.empty_cache()

    R = B + BT
    flop = 2 * K * R * C * D
    min_bytes = K * R * (D + C) * 4
    diag_ms = ktimes[True].get("sweep_grad_diag", 0.0)
    med = lambda xs: sorted(xs)[len(xs) // 2]
    return {
        "shape": name, "heads": K, "D": D, "C": C, "Dv": wl.get("dv"), "rows_per_step": [B, BT], "steps": steps,
        "rounds": rounds,
        "device_step_ms_off": [round(x, 4) for x in step_ms[False]],
        "device_step_ms_on": [round(x, 4) for x in step_ms[True]],
        "device_step_added_ms_median": round(med(step_ms[True]) - med(step_ms[False]), 4),
        "last_step_kernel_ms_off": {k_: round(v, 4) for k_, v in ktimes[False].items()},
        "last_step_kernel_ms_on": {k_: round(v, 4) for k_, v in ktimes[True].items()},
        "diag_launches_ms": round(diag_ms, 4),
        "diag_flop_per_step": flop, "diag_mma_flop_3xtf32": 3 * flop, "diag_min_bytes_per_step": min_bytes,
        "diag_tflops_3xtf32": round(3 * flop / (diag_ms * 1e-3) / 1e12, 2) if diag_ms > 0 else None,
        "diag_min_bytes_gbs": round(min_bytes / (diag_ms * 1e-3) / 1e9, 1) if diag_ms > 0 else None,
        "e2e_step_ms_off": round(e2e[False], 4), "e2e_step_ms_on": round(e2e[True], 4),
        "finite_diagnostics": bool(finite),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--runs", default="cfg2:6,cfg2:30,cfg4:30", help="shape:heads, comma separated")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sweep_grad_diag_bench needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"card": card(), "runs": []}
    for run in args.runs.split(","):
        name, K = run.split(":")
        res["runs"].append(run_shape(name, int(K), args.steps, args.warmup, args.rounds))
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
