"""Host side of the Gaussian lock-step group (gaussian.train_models_steps, uml_gauss_group_run) without a GPU: the ctypes
mirror of uml_gauss_group_args against the header, the library's argument checks (all made before it touches the
device) and the reasons train_models_steps gives for runs that cannot share a group.  The kernels run in
tests/test_gauss_group_gpu.py."""
import ctypes as C
import os
import shutil
import subprocess
import types

import pytest
import torch

import uml_b200  # noqa: F401
from uml_b200 import _lib
from uml_b200 import gaussian as G

DIMS = (12, 16, 6)


def test_ctypes_group_struct_matches_the_header(tmp_path):
    """sizeof and every field offset of the ctypes mirror equal what a C compiler makes of include/uml_b200.h."""
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cls, cname = _lib.GaussGroupArgs, "uml_gauss_group_args"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "uml_b200.h"', 'int main(void) {',
             f'  printf("{cname} %zu\\n", sizeof({cname}));',
             '  printf("max_runs %d\\n", UML_GAUSS_GROUP_MAX_RUNS);']
    lines += [f'  printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));' for f, _ in cls._fields_]
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got["max_runs"]) == _lib.GAUSS_GROUP_MAX_RUNS == G.GROUP_MAX_RUNS
    assert int(got[cname]) == C.sizeof(cls)
    for f, _ in cls._fields_:
        assert int(got[f"{cname}.{f}"]) == getattr(cls, f).offset, f


def test_group_run_validates_arguments_before_touching_the_device():
    lib = _lib.load()
    a = _lib.GaussGroupArgs()
    fake = 1 << 20  # never dereferenced: every call below fails a check first or has nothing to launch
    idx = (C.c_void_p * 4)(fake, fake, fake, fake)
    run = lambda n=1: lib.uml_gauss_group_run(C.byref(a), n, idx, None)
    err = lambda: lib.uml_last_error()
    assert lib.uml_gauss_group_run(None, 1, idx, None) != 0 and b"null argument" in err()
    assert lib.uml_gauss_group_run(C.byref(a), 1, None, None) != 0 and b"null argument" in err()
    assert run() != 0 and b"1..32 runs" in err()
    a.n_runs = 33
    assert run() != 0 and b"1..32 runs" in err()
    a.n_runs, a.batch, a.n_x, a.n_y = 2, 16, 40, 40
    assert run() != 0 and b"bad shape" in err()
    a.dim_obs, a.dim_common, a.dim_latent = DIMS
    assert run() != 0 and b"null buffer" in err()
    a.data_x = a.data_y = a.params = a.adam_m = a.adam_v = a.loss_log = a.workspace = fake
    P = int(lib.uml_gauss_param_count(*DIMS))
    a.param_stride = P - 1
    assert run() != 0 and b"param_stride" in err()
    a.param_stride = P
    assert run() != 0 and b"first_step" in err()
    a.first_step = 1
    a.dim_common, a.param_stride = 2000, int(lib.uml_gauss_param_count(DIMS[0], 2000, DIMS[2]))
    assert run() != 0 and b"too wide" in err()
    a.dim_common, a.param_stride = DIMS[1], P
    a.mode_xy[1] = 2
    assert run() != 0 and b"run 1: mode_xy" in err()
    a.mode_xy[1] = 0
    a.active[0] = a.active[1] = 1
    a.eval_every = 5
    assert run() != 0 and b"run 0 has no validation rows" in err()
    a.val_x[0] = a.val_y[0] = a.val_x[1] = a.val_y[1] = fake
    assert run() != 0 and b"null eval_log" in err()
    a.eval_log = fake
    a.n_val, a.topk = 10, 10
    assert run() != 0 and b"topk" in err()
    a.topk = 3
    need = int(lib.uml_gauss_group_workspace_bytes(2, *DIMS, 16, 10, 3))
    assert need > int(lib.uml_gauss_group_workspace_bytes(2, *DIMS, 16, 0, 0)) > 0
    a.workspace_bytes = need - 1
    assert run() != 0 and b"workspace holds" in err()
    a.workspace_bytes = need
    a.workspace = fake + 4
    assert run() != 0 and b"16-byte aligned" in err()
    a.workspace = fake
    idx[3] = None  # step 1, run 1
    assert run(2) != 0 and b"step 1 has no index batch for run 1" in err()
    a.active[1] = 0  # an inactive run's index entries are not used
    # every check passes, and a call with no active run or no step launches nothing
    a.active[0] = 0
    assert run(2) == 0
    a.active[0] = 1
    assert run(0) == 0


class _Bank:
    """UnpairedDataset stand-in with the attributes the blockers read (CPU tensors: this file has no GPU)."""

    def __init__(self, n=40, dim_obs=DIMS[0]):
        self.data_x, self.data_y = torch.zeros(n, dim_obs), torch.zeros(n, dim_obs)
        self.len_x = self.len_y = self.length = n
        self.device = self.data_x.device

    def __len__(self):
        return self.length


def _model(dims=DIMS):
    m = object.__new__(G.SharedAutoencoder)  # the real constructor allocates on the GPU
    m.dim_obs, m.dim_common, m.dim_latent = dims
    m.device = torch.device("cuda")
    m.flat = torch.zeros(int(_lib.load().uml_gauss_param_count(*dims)))
    return m


def _case(k=2):
    bank = _Bank()
    models = [_model() for _ in range(k)]
    loaders = [G.unpaired_loader(bank, 8, generator=torch.Generator().manual_seed(42)) for _ in range(k)]
    opts = [G.Adam(m, lr=1e-3 * (i + 1)) for i, m in enumerate(models)]
    return models, loaders, opts


def _reasons(models, loaders, opts, **kw):
    with pytest.raises(ValueError) as e:
        G.train_models_steps(models, loaders, opts, 4, **kw)
    return str(e.value)


def test_each_blocker_is_named():
    models, loaders, opts = _case()
    # on this host the tensors are CPU tensors: that is the only reason these two runs cannot share a group
    assert G.group_blockers(models, loaders, opts) == ["a model not on CUDA"]
    assert "a model not on CUDA" in _reasons(models, loaders, opts)

    def only(reason, models, loaders, opts, **kw):
        msg = _reasons(models, loaders, opts, **kw)
        assert reason in msg, msg
        assert any(reason in w for w in G.group_blockers(models, loaders, opts))

    m, l, o = _case()
    m[1] = _model((12, 16, 8))
    o[1] = G.Adam(m[1])
    only("different model dims", m, l, o)
    m, l, o = _case()
    l[1] = G.unpaired_loader(_Bank(), 8, generator=torch.Generator().manual_seed(42))
    only("different datasets or batch sizes", m, l, o)
    m, l, o = _case()
    l[1] = G.unpaired_loader(l[0].bank, 16, generator=torch.Generator().manual_seed(42))
    only("different datasets or batch sizes", m, l, o)
    from uml_b200.engine.datasets.utils import BankLoader
    m, l, o = _case()
    l[1] = BankLoader(l[0].bank, 8, shuffle=True, drop_last=False, generator=torch.Generator())
    only("loaders without drop_last / shuffle", m, l, o)
    m, l, o = _case()
    l[1] = BankLoader(l[0].bank, 8, shuffle=False, drop_last=True, generator=torch.Generator())
    only("loaders without drop_last / shuffle", m, l, o)
    m, l, o = _case(33)
    only("more than 32 runs", m, l, o)
    m, l, o = _case()
    msg = _reasons(m, l, o, val_data_x=[torch.zeros(20, 12), torch.zeros(30, 12)], val_data_y=torch.zeros(20, 12))
    assert "validation sets of different shapes" in msg
    msg = _reasons(m, l, o, val_data_x=torch.zeros(20, 12), val_data_y=torch.zeros(20, 11))
    assert "validation sets of different shapes" in msg
    # the sampler streams: every run draws from a generator of its own, as each combination of the reference does
    m, l, o = _case()
    l[1] = G.unpaired_loader(l[0].bank, 8, generator=l[0].generator)
    only("share one generator", m, l, o)
    m, l, o = _case()
    l[1] = G.unpaired_loader(l[0].bank, 8)
    only("global generator", m, l, o)
    # the optimizers share betas, eps and the step count
    m, l, o = _case()
    o[1] = G.Adam(m[1], betas=(0.8, 0.999))
    only("different betas, eps or step counts", m, l, o)
    m, l, o = _case()
    o[1].step_count = 3
    only("different betas, eps or step counts", m, l, o)
    # several reasons are all named
    m, l, o = _case()
    m[1] = _model((12, 16, 8))
    o[1] = G.Adam(m[1])
    l[1] = G.unpaired_loader(l[0].bank, 16, generator=torch.Generator())
    msg = _reasons(m, l, o)
    assert "different model dims" in msg and "different datasets or batch sizes" in msg


def test_mode_and_argument_counts_are_checked():
    m, l, o = _case()
    with pytest.raises(ValueError, match="mode must be"):
        G.train_models_steps(m, l, o, 4, args=[types.SimpleNamespace(mode="y"), None])
    with pytest.raises(ValueError, match="args namespaces"):
        G.train_models_steps(m, l, o, 4, args=[None])
    with pytest.raises(ValueError, match="validation sets for 2 runs"):
        G.train_models_steps(m, l, o, 4, val_data_x=[torch.zeros(20, 12)], val_data_y=[torch.zeros(20, 12)])
