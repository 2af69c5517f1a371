"""Sweep batching of adapter heads with learnable temperatures (preset `linear`: UML head with img_proj, learnable
img_scale / txt_scale, AdamW) - what one step of K combinations costs in lock step (AdapterHeadGroup /
uml_sweep_adapter_run: five launches per step of all heads) against one combination on the single-head engine.

    python tools/sweep_adapter_bench.py [--steps 200] [--warmup 20] [--out FILE]

Shapes: cfg4 at the reference batch (Dv 1536, D 3200, C 1000, 16 000 image rows, 29 940 text rows, 32 + 32 rows) and
a small one (Dv 768, D 768, C 397), each with K = 6 and 30 heads.  Arms, as bench.py's cfg2_sweep:
  * device: CUDA events over --steps steps after --warmup, every head's permutation already in HBM, with the
    per-launch breakdown of the last step;
  * e2e: one public train_group() call (the wall clock of its last --steps iterations);
  * sequential: finetune.train() of one combination, the cost per step today.
Prints one JSON line (and writes it to --out): card name and power limit are read in the same run.  The banks
(0.3 GB at cfg4) fit the 126 MB L2 only in part; the per-step working set of the update (24 B x parameters x K) does
not."""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import build_banks, measured_peaks  # noqa: E402

SHAPES = {
    "cfg4": dict(n_img=16_000, n_txt=29_940, dv=1536, dim=3200, classes=1000, batch=32, batch_txt=32, n_val=1000),
    "small": dict(n_img=16_000, n_txt=29_940, dv=768, dim=768, classes=397, batch=32, batch_txt=32, n_val=1000),
}
HBM_DATASHEET_GBS = 7700.0


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit"], out["max_sm_clock"] = [s.strip() for s in q.split(",")][:2]
    except Exception as e:  # report, do not guess
        out["power_limit"] = f"unavailable: {e}"
    return out


def work(wl):
    """Algorithmic work of one head-step: FLOPs (SURVEY 8d: per image row 2 Dv D + 2 D C forward, the same twice
    backward; per text row 2 D C forward and 2 D C for dW) and the update traffic (W, m, v read and written)."""
    Dv, D, C, B, BT = wl["dv"], wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    flop = B * (2 * Dv * D + 2 * D * C) * 3 - B * 2 * Dv * D + BT * 2 * D * C * 2  # no dX for the bank rows
    params = D * Dv + C * D
    return flop, params, 24.0 * params


def run_shape(name, K, steps, warmup, peaks):
    import uml_b200  # noqa: F401
    from uml_b200 import _lib, finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader
    from uml_b200.engine.models.head import UML
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler
    from uml_b200.engine.sweep import AdapterHeadGroup

    wl = SHAPES[name]
    dev = torch.device("cuda", 0)
    img_bank, txt_bank, val_bank, _ = build_banks(wl, dev)
    Dv, D, C, B, BT = wl["dv"], wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]
    grid = [(lr, wd, al) for al in (0.2, 0.5, 1.0, 1.5, 2.0) for lr in (1e-3, 1e-4) for wd in (0.0, 0.01, 0.0001)]
    grid = [grid[k % len(grid)] for k in range(K)]
    alphas = [g[2] for g in grid]

    def make_heads(n):
        ms, os_, ss, il, tl, vl = [], [], [], [], [], []
        with contextlib.redirect_stdout(io.StringIO()):
            for k in range(n):
                lr, wd, _ = grid[k]
                torch.manual_seed(k)
                m = UML(f"synthetic:{Dv}", D, C, learnable_temp=True)
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

    # ---------------- device-resident arm ------------------------------------------------------------------------
    ms_, os_, ss, il, tl, vl = make_heads(K)
    group = AdapterHeadGroup(ms_, os_, img_bank, txt_bank, B, BT, dev, log_slots=warmup + steps + 1)
    iti, itt = [iter(l) for l in il], [iter(l) for l in tl]
    assert warmup + steps <= min(len(il[0]), len(tl[0])), "warm-up + steps must stay inside one epoch"

    def chunk(n, i0):
        pi = [it.take_run(n) for it in iti]
        pt = [it.take_run(n) for it in itt]
        lrs = [[s.lr_at(i0 + j, s.base_lrs[0]) for s in ss] for j in range(n)]
        return [p[0] for p in pi], [p[0] for p in pt], pi[0][1], pt[0][1], [(B, BT)] * n, lrs

    a = chunk(warmup, 0)
    group.run(*a, alphas, [True] * K, slot0=0)
    a = chunk(steps, warmup)
    group.time_last_step()
    torch.cuda.synchronize()
    n0 = _lib.LAUNCH_COUNT[0]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    i = 0
    while i < steps:  # one library call per 16 steps, like train_group's chunks
        n = min(16, steps - i)
        group.run(a[0], a[1], a[2] + i * B, a[3] + i * BT, a[4][i:i + n], a[5][i:i + n], alphas, [True] * K,
                  slot0=warmup + i)
        i += n
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    launches = (_lib.LAUNCH_COUNT[0] - n0) / steps
    ktimes = group.kernel_times_ms()
    tail = group.read_log([warmup + steps - 1], True, True)
    finite = all(torch.isfinite(torch.tensor(tail[k_][0])).all() for k_ in ("image_loss", "text_loss"))
    del group, ms_, os_

    # ---------------- end-to-end arm: one public train_group() call ----------------------------------------------
    ms2, os2, ss2, il2, tl2, vl2 = make_heads(K)
    trs = [None] * K
    trs[0] = {"indices": False, "timing": {"warmup": warmup}}
    with contextlib.redirect_stdout(io.StringIO()):
        ft.train_group(ms2, il2, tl2, vl2, None, os2, ss2, device=dev, max_iters=warmup + steps, alphas=alphas,
                       eval_freq=10 ** 9, patience=5, traces=trs)
    e2e_ms = trs[0]["timing"]["seconds"] * 1e3 / trs[0]["timing"]["iters"]
    del ms2, os2

    # ---------------- one combination on the single-head engine --------------------------------------------------
    ms3, os3, ss3, il3, tl3, vl3 = make_heads(1)
    tr = {"timing": {"warmup": warmup}, "indices": False}
    with contextlib.redirect_stdout(io.StringIO()):
        ft.train(ms3[0], il3[0], tl3[0], vl3[0], None, os3[0], ss3[0], device=dev, max_iters=warmup + steps,
                 alpha=alphas[0], eval_freq=10 ** 9, patience=5, trace=tr)
    seq_ms = tr["timing"]["seconds"] * 1e3 / tr["timing"]["iters"]

    flop, params, upd_bytes = work(wl)
    upd_ms = ktimes.get("sweep_dw_update", 0.0) + ktimes.get("sweep_adapter_dw_update", 0.0)
    return {
        "shape": name, "heads": K, "Dv": Dv, "D": D, "C": C, "rows_per_step": [B, BT], "steps": steps,
        "device_step_ms": round(step_ms, 4), "launches_per_step": launches,
        "last_step_kernel_ms": {k_: round(v, 4) for k_, v in ktimes.items()},
        "e2e_step_ms": round(e2e_ms, 4), "sequential_step_ms_one_combination": round(seq_ms, 4),
        "speedup_vs_sequential": round(K * seq_ms / step_ms, 2),
        "gflop_per_head_step": round(flop / 1e9, 4), "update_mb_per_head_step": round(upd_bytes / 1e6, 1),
        "achieved_tflops": round(K * flop / (step_ms * 1e-3) / 1e12, 3),
        "update_launches_gbs": round(K * upd_bytes / (upd_ms * 1e-3) / 1e9, 1) if upd_ms > 0 else None,
        "hbm_bound_step_ms_datasheet": round(K * upd_bytes / (HBM_DATASHEET_GBS * 1e9) * 1e3, 4),
        "update_share_of_hbm_copy_peak": round(K * upd_bytes / (upd_ms * 1e-3) / 1e9 / peaks["hbm"], 3) if upd_ms > 0 else None,
        "finite_losses": bool(finite),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--shapes", default="cfg4,small")
    ap.add_argument("--heads", default="6,30")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sweep_adapter_bench needs a CUDA device")
    torch.cuda.set_device(0)
    peaks = measured_peaks()
    res = {"card": card(), "hbm_copy_peak_gbs": peaks["hbm"], "hbm_peak_src": peaks["src"], "runs": []}
    for name in args.shapes.split(","):
        for K in (int(h) for h in args.heads.split(",")):
            res["runs"].append(run_shape(name, K, args.steps, args.warmup, peaks))
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
