"""Prints a checksum of the head weights and the per-step stats after 9 bf16 steps of a fixed scenario - run it against
two builds of the library (UML_LIB_PATH selects one) to check that they compute bit-identical results."""
import hashlib
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import uml_b200  # noqa: F401,E402
from uml_b200 import finetune as ft  # noqa: E402
from uml_b200.engine.datasets.utils import BankLoader, FeatureBank  # noqa: E402
from uml_b200.engine.models.head import UMLClip  # noqa: E402
from uml_b200.engine.optimizer.optim import build_optimizer  # noqa: E402
from uml_b200.engine.optimizer.scheduler import build_lr_scheduler  # noqa: E402
from uml_b200.engine.trainer import StepEngine  # noqa: E402

DEV = "cuda:0"
D, C, B, steps = 768, 1000, 4736, 9
g = torch.Generator().manual_seed(4)
xi, yi = torch.randn(30000, D, generator=g), torch.randint(0, C, (30000,), generator=g)
xt, yt = torch.randn(9000, D, generator=g), torch.arange(9000) % C
ib, tb = FeatureBank(xi, yi, DEV), FeatureBank(xt, yt, DEV)
torch.manual_seed(1)
model = UMLClip(f"synthetic:{D}", C, logit_scale_init=4.60517)
model.to(DEV)
model.zero_shot_init(tb)
model.to(DEV)
opt = build_optimizer(model.parameters(), "adamw", 1e-3, 0.01)
sch = build_lr_scheduler(opt, "cosine", 3, 100, warmup_type="linear", warmup_lr=1e-5)
eng = StepEngine(model, opt, DEV, B, B, log_slots=steps + 1, precision="bf16")
il, tl = BankLoader(ib, B, shuffle=True), BankLoader(tb, B, shuffle=True)
torch.manual_seed(9)
ii, ti = iter(il), iter(tl)
batches, lrs = [], []
for _ in range(steps):
    a, ii = ft.fetch_next(il, ii)
    b, ti = ft.fetch_next(tl, ti)
    batches.append((a, b))
    lrs.append(sch.get_last_lr()[0])
    sch.step()
eng.run(batches[:4], 0.5, lrs[:4], slot0=0)
eng.run(batches[4:], 0.5, lrs[4:], slot0=4)
torch.cuda.synchronize()
h = hashlib.sha256(model.head.weight.detach().cpu().numpy().tobytes()).hexdigest()[:16]
log = eng.read_log(list(range(steps)))
print("weights", h, "loss", [round(r["image_loss"], 6) for r in log][:3], [round(r["text_loss"], 6) for r in log][:3])
