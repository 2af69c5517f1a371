"""Host side of per-step gradient diagnostics for single runs without a GPU: the ctypes mirror of uml_linear_diag, the
argument checks of uml_linear_grad_diag / uml_linear_run_diag, the --grad-diagnostics-every-step flag and the reasons
a run falls back to evaluation-cadence diagnostics."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

import uml_b200  # noqa: F401
from uml_b200 import _lib
from uml_b200.engine.config import parser
from uml_b200.engine.models.head import UML, UMLClip
from uml_b200.engine.trainer import diag_blockers

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20  # a 16-byte aligned address that is never dereferenced: every call below fails its checks first


def test_ctypes_linear_diag_struct_matches_the_header(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    cls, cname = _lib.LinearDiag, "uml_linear_diag"
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


def test_exact_path_scratch_size():
    lib = _lib.load()
    assert lib.uml_linear_diag_scratch_floats(0, 64, 512, 1000) == 4 * 16 * 4
    assert lib.uml_linear_diag_scratch_floats(0, 64, 40, 10) == 4
    assert lib.uml_linear_diag_scratch_floats(0, 0, 40, 10) == 0


def _args(precision=0, dim=40, n_classes=10, n=(8, 8), alpha=0.5):  # (ldg 64: a 16-byte multiple)
    a = _lib.LinearStepArgs()
    a.dim, a.n_classes, a.precision, a.nseg = dim, n_classes, precision, len(n)
    for k, cnt in enumerate(n):
        a.seg[k].rows, a.seg[k].ld, a.seg[k].n = FAKE, dim, cnt
        a.seg[k].loss_weight = 1.0 if k == 0 else alpha
    a.G, a.ldg = FAKE, 64
    a.X16 = FAKE if precision else None
    return a


def _diag(scratch_floats=1 << 30, has_img=1):
    d = _lib.LinearDiag()
    d.scratch, d.scratch_floats, d.has_img = FAKE, scratch_floats, has_img
    return d


def _fails(a, d, what, out=FAKE):
    lib = _lib.load()
    assert lib.uml_linear_grad_diag(C.byref(a), C.byref(d) if d is not None else None, out, None) != 0
    assert what in lib.uml_last_error(), lib.uml_last_error()


def test_grad_diag_validates_arguments_before_touching_the_device():
    _fails(_args(), None, b"null diagnostics buffer")
    _fails(_args(), _diag(), b"null diagnostics buffer", out=None)
    _fails(_args(), _diag(has_img=0), b"image run")
    a = _args()
    a.dp_allreduce = 1
    _fails(a, _diag(), b"data-parallel")
    _fails(_args(dim=42), _diag(), b"multiple of 4")
    _fails(_args(precision=1, dim=44), _diag(), b"multiple of 8")
    _fails(_args(precision=2), _diag(), b"precision must be 0 or 1")
    _fails(_args(alpha=0.0), _diag(), b"alpha")
    _fails(_args(alpha=-1.0), _diag(), b"alpha")
    a = _args()
    a.seg[0].loss_weight = 0.5
    _fails(a, _diag(), b"loss weight must be 1")
    a = _args()
    a.G = FAKE + 4
    _fails(a, _diag(), b"16-byte aligned")
    a = _args()
    a.seg[1].rows = FAKE + 8
    _fails(a, _diag(), b"run 1 rows")
    a = _args()
    a.seg[0].ld = 42
    _fails(a, _diag(), b"run 0 rows")
    a = _args()
    a.ldg = 6
    _fails(a, _diag(), b"ldg a multiple of 4")
    _fails(_args(), _diag(scratch_floats=3), b"scratch holds 3 floats, 4 needed")
    a = _args(precision=1)
    a.X16 = FAKE + 2
    _fails(a, _diag(), b"X16")
    a = _args(precision=1)
    a.ldg = 12
    _fails(a, _diag(), b"ldg a multiple of 64")
    # bf16: the per-block slots and one split-K plane of C * D for each modality at least
    _fails(_args(precision=1), _diag(scratch_floats=4 * 296 + 2 * 400 - 1), b"scratch holds")


def test_run_diag_checks_every_step_before_enqueueing():
    lib = _lib.load()
    a, d = _args(), _diag()
    steps = (_lib.RunStep * 2)()
    for s in steps:
        s.n[0], s.n[1], s.loss_weight[0], s.loss_weight[1] = 8, 8, 1.0, 0.5
    steps[1].loss_weight[1] = 0.0  # the second step's alpha: its text-loss gradient cannot be recovered
    outs = (C.c_void_p * 2)(FAKE, FAKE)
    assert lib.uml_linear_run_diag(C.byref(a), steps, 2, C.byref(d), outs, None) != 0
    assert b"alpha" in lib.uml_last_error()
    assert lib.uml_linear_run_diag(C.byref(a), steps, 2, None, outs, None) != 0
    assert b"bad arguments" in lib.uml_last_error()


def test_every_step_flag_is_off_by_default():
    base = ["--dataset", "synthset"]
    assert parser.parse_args(base).grad_diagnostics_every_step is False
    args = parser.parse_args(base + ["--grad-diagnostics-every-step"])
    assert args.grad_diagnostics_every_step is True
    assert "every step" in parser.format_help().split("--grad-diagnostics-every-step")[-1][:300]


def test_fallback_reasons():
    clip = UMLClip("synthetic:40", 10)
    assert diag_blockers(clip, 1, 0.5, True) == []
    assert diag_blockers(clip, 1, 0.0, False) == []  # alpha does not matter without text rows
    why = diag_blockers(clip, 2, 0.5, True)
    assert len(why) == 1 and "data-parallel" in why[0]
    why = diag_blockers(clip, 1, 0.0, True)
    assert len(why) == 1 and "alpha > 0" in why[0]
    why = diag_blockers(UMLClip("synthetic:42", 10), 1, 0.5, True)
    assert len(why) == 1 and "multiples of 4" in why[0]
    why = diag_blockers(UML("synthetic:24", 42, 10), 1, -1.0, True)
    assert len(why) == 2 and "alpha > 0" in why[0] and "multiples of 4" in why[1]
    # an adapter's input width does not matter: the device passes read Z, which has the head's width
    assert diag_blockers(UML("synthetic:26", 40, 10), 1, 1.5, True) == []
