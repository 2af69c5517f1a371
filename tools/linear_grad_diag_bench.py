"""Per-step gradient diagnostics of single runs (--grad-diagnostics-every-step: the reference's four gradient probes of
every step on the device) - what they add to a step.

    python tools/linear_grad_diag_bench.py [--steps 40] [--warmup 10] [--rounds 3] [--out FILE]

Shapes (bench.py's workloads): cfg2 (exact fused step, 32 + 32 rows, D 512, C 1000), cfg3 (bf16 tensor-core step,
70 144 + 3 584 rows, D 768, C 1000), cfg4 (adapter + learnable temperatures, Dv 1536, D 3200, C 1000) at 32 + 32 rows
(exact path) and at 8192 + 8192 rows (bf16 path).  Arms, in one process, off and on alternating --rounds times:
  * device: CUDA events over --steps steps enqueued through StepEngine.run in chunks of 16 (the chunks train() issues);
  * e2e: one public train() call per arm, the wall clock of its last --steps iterations (stream-synchronised, the
    per-step probes read back with the losses; one evaluation at step 0, before the timed window).
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

from bench import WORKLOADS, build_banks  # noqa: E402
from sweep_adapter_bench import card  # noqa: E402

SHAPES = {
    "cfg2": dict(WORKLOADS["cfg2"], adapter=False, precision="fp32"),
    "cfg3": dict(WORKLOADS["cfg3"], adapter=False, precision="bf16"),
    "cfg4_32": dict(WORKLOADS["cfg4"], batch=32, batch_txt=32, adapter=True, precision="fp32"),
    "cfg4_8192": dict(WORKLOADS["cfg4"], adapter=True, precision="bf16"),
}


def run_shape(name, steps, warmup, rounds):
    import uml_b200  # noqa: F401
    from uml_b200 import finetune as ft
    from uml_b200.engine.datasets.utils import BankLoader
    from uml_b200.engine.models.head import UML, UMLClip
    from uml_b200.engine.optimizer.optim import build_optimizer
    from uml_b200.engine.optimizer.scheduler import build_lr_scheduler
    from uml_b200.engine.trainer import StepEngine

    wl = SHAPES[name]
    dev = torch.device("cuda", 0)
    img_bank, txt_bank, val_bank, _ = build_banks(wl, dev)
    D, C, B, BT = wl["dim"], wl["classes"], wl["batch"], wl["batch_txt"]

    def head():
        torch.manual_seed(0)
        m = UML(f"synthetic:{wl['dv']}", D, C, learnable_temp=True) if wl["adapter"] else \
            UMLClip(f"synthetic:{D}", C, logit_scale_init=4.60517)
        m.precision = wl["precision"]
        m.to(dev)
        o = build_optimizer(m.parameters(), "adamw", 1e-4, 0.01)
        s = build_lr_scheduler(o, "cosine", 50, 12800, warmup_type="linear", warmup_lr=1e-5)
        rng = torch.Generator().manual_seed(100)
        return m, o, s, BankLoader(img_bank, B, shuffle=True, rng=rng), BankLoader(txt_bank, BT, shuffle=True, rng=rng), \
            BankLoader(val_bank, 1024, shuffle=False, rng=rng)

    def take(loader, n):  # n consecutive index batches, across epoch boundaries
        out, it = [], iter(loader)
        while len(out) < n:
            k = it.batches_left()
            if k == 0:
                it = iter(loader)
                continue
            out += it.take_chunk(min(k, n - len(out)))
        return out

    # ---------------- device arm ----------------
    engines, batches = {}, {}
    for diag in (False, True):
        m, o, s, il, tl, _ = head()
        engines[diag] = (StepEngine(m, o, dev, B, BT, log_slots=warmup + steps + 1, precision=wl["precision"],
                                    grad_diagnostics=diag), s)
        batches[diag] = list(zip(take(il, warmup + steps), take(tl, warmup + steps)))
    lrs = [1e-4] * (warmup + steps)

    def enqueue(diag, first, n):
        eng = engines[diag][0]
        i = first
        while i < first + n:
            k = min(16, first + n - i)
            eng.run(batches[diag][i:i + k], 0.5, lrs[i:i + k], slot0=i)
            i += k

    for diag in (False, True):
        enqueue(diag, 0, warmup)
    step_ms = {False: [], True: []}
    for _ in range(rounds):
        for diag in (False, True):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            enqueue(diag, warmup, steps)
            e1.record()
            torch.cuda.synchronize()
            step_ms[diag].append(e0.elapsed_time(e1) / steps)
    recs = engines[True][0].read_log([warmup + steps - 1])
    probe = recs[0]["grad_diag"]
    finite = all(v == v and abs(v) != float("inf") for v in probe)
    del engines, batches
    torch.cuda.empty_cache()

    # ---------------- e2e arm: one train() call per arm ----------------
    e2e_ms = {False: [], True: []}
    for _ in range(rounds):
        for diag in (False, True):
            m, o, s, il, tl, vl = head()
            tr = {"timing": {"warmup": warmup}, "indices": False}
            if diag:
                tr["grad_diagnostics"] = "step"
            with contextlib.redirect_stdout(io.StringIO()):
                ft.train(m, il, tl, vl, None, o, s, device=dev, max_iters=warmup + steps, alpha=0.5,
                         eval_freq=10 ** 6, patience=5, trace=tr, stats_to_host="step")
            e2e_ms[diag].append(1e3 * tr["timing"]["seconds"] / tr["timing"]["iters"])
            if diag:
                assert len(tr["grad_diag"]) == warmup + steps
            del m, o, tr
            torch.cuda.empty_cache()
    med = lambda xs: sorted(xs)[len(xs) // 2]
    return {"rows": [B, BT], "dim": D, "classes": C, "dv": wl.get("dv"), "path": wl["precision"],
            "device_step_ms": {"off": [round(x, 4) for x in step_ms[False]], "on": [round(x, 4) for x in step_ms[True]]},
            "device_added_ms_median": round(med(step_ms[True]) - med(step_ms[False]), 4),
            "train_step_ms": {"off": [round(x, 4) for x in e2e_ms[False]], "on": [round(x, 4) for x in e2e_ms[True]]},
            "train_added_ms_median": round(med(e2e_ms[True]) - med(e2e_ms[False]), 4),
            "probes_finite": finite}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--shapes", type=str, default=",".join(SHAPES))
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    line = {"bench": "linear_grad_diag", "card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds}
    for name in args.shapes.split(","):
        line[name] = run_shape(name, args.steps, args.warmup, args.rounds)
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
