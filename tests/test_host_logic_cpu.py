"""Host-side logic of the product against the golden vectors recorded from the reference - runs
without a GPU: sampler RNG protocol, text-bank selection, LR schedule, presets, path layout."""
import ast
import json
import os

import numpy as np
import pytest
import torch

import uml_b200  # noqa: F401
from uml_b200 import finetune as ft
from uml_b200.engine.datasets.utils import BankLoader, FeatureBank, TextTensorDataset
from uml_b200.engine.optimizer.default import HYPER_DICT
from uml_b200.engine.optimizer.optim import build_optimizer
from uml_b200.engine.optimizer.scheduler import build_lr_scheduler
from uml_b200 import features as F

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
M = np.load(os.path.join(GOLDEN, "misc.npz"), allow_pickle=False)
# the reference's HYPER_DICT and parser.parse_args([]) (make_golden.py)
with open(os.path.join(GOLDEN, "reference_defaults.json")) as _f:
    REF_DEFAULTS = json.load(_f)


def _bank(n):
    return FeatureBank(torch.zeros(n, 4), torch.zeros(n, dtype=torch.int64), device="cpu")


@pytest.mark.parametrize("nw", [0, 2])
def test_bankloader_matches_dataloader_index_stream(nw):
    torch.manual_seed(123)
    a, b = BankLoader(_bank(23), 5, shuffle=True, num_workers=nw), BankLoader(_bank(17), 5, shuffle=True, num_workers=nw)
    ia, ib = iter(a), iter(b)
    for s in range(12):
        x, ia = ft.fetch_next(a, ia)
        y, ib = ft.fetch_next(b, ib)
        ga, gb = M[f"nw{nw}_a"][s], M[f"nw{nw}_b"][s]
        assert np.array_equal(x.host_idx.numpy(), ga[ga >= 0]) and x.n == (ga >= 0).sum()
        assert np.array_equal(y.host_idx.numpy(), gb[gb >= 0])
        assert torch.equal(x.idx.cpu(), x.host_idx)


def test_sequential_loader_draws_one_base_seed_and_covers_the_bank():
    torch.manual_seed(9)
    want = int(torch.empty((), dtype=torch.int64).random_().item())
    second = int(torch.empty((), dtype=torch.int64).random_().item())
    torch.manual_seed(9)
    l = BankLoader(_bank(11), 4, shuffle=False)
    batches = list(iter(l))
    assert [(b.start, b.n) for b in batches] == [(0, 4), (4, 4), (8, 3)] and len(l) == 3
    assert int(torch.empty((), dtype=torch.int64).random_().item()) == second and want != second


def test_explicit_generator_protocol_matches_gaussian_loader():
    """DataLoader(..., shuffle=True, drop_last=True, generator=g): permutations come from g itself and a
    discarded permutation is drawn at each epoch end (checked against torch's own DataLoader)."""
    from torch.utils.data import DataLoader, TensorDataset
    g1, g2 = torch.Generator().manual_seed(42), torch.Generator().manual_seed(42)
    ref = DataLoader(TensorDataset(torch.arange(40)), batch_size=16, shuffle=True, drop_last=True, generator=g1)
    ours = BankLoader(_bank(40), 16, shuffle=True, drop_last=True, generator=g2)
    ri, oi = iter(ref), iter(ours)
    for _ in range(7):
        try:
            r = next(ri)[0]
        except StopIteration:
            ri = iter(ref)
            r = next(ri)[0]
        o, oi = ft.fetch_next(ours, oi)
        assert torch.equal(r, o.host_idx)


def test_text_dataset_selection_matches_reference():
    feats, labels, eot = (torch.from_numpy(M["text/" + k]) for k in ("feats", "labels", "eot"))
    for shots in (2, 4):
        torch.manual_seed(31)
        ds = TextTensorDataset(feats, labels, eot, n_shots=shots)
        assert np.array_equal(ds.eot_indices.numpy(), M[f"text/shot{shots}/eot"])
        assert int(torch.empty((), dtype=torch.int64).random_().item()) == int(M[f"text/shot{shots}/after_draw"])
    ds = TextTensorDataset(feats, labels, eot, n_shots="average")
    np.testing.assert_allclose(ds.input_tensor.numpy(), M["text/avg/feats"], rtol=1e-6, atol=1e-7)
    assert np.array_equal(ds.label_tensor.numpy(), M["text/avg/labels"])
    assert np.array_equal(ds.eot_indices.numpy(), M["text/avg/eot"])
    assert len(TextTensorDataset(feats, labels, eot)) == feats.shape[0]
    with pytest.raises(ValueError):
        TextTensorDataset(feats, labels, eot, n_shots=1.5)


def test_zero_shot_weights_cpu_path():
    from uml_b200.engine.models.head import get_zero_shot_weights
    feats, labels, eot = (torch.from_numpy(M["text/" + k]) for k in ("feats", "labels", "eot"))
    w = get_zero_shot_weights(TextTensorDataset(feats, labels, eot), 7, feats.shape[1], device="cpu")
    np.testing.assert_allclose(w.numpy(), M["text/zeroshot_w"], rtol=1e-5, atol=1e-6)
    assert float(w[2].abs().sum()) == 0.0


def test_lr_schedule_matches_reference_scheduler():
    for key in [k for k in M.files if k.startswith("sched/") and not k.endswith("/cfg")]:
        kw = ast.literal_eval(str(M[key + "/cfg"]))
        p = torch.nn.Parameter(torch.zeros(1))
        opt = build_optimizer([p], "adamw", kw["base"], 0.0)
        sch = build_lr_scheduler(opt, kw["s"], kw["w"], kw["T"], warmup_type=kw["wt"], warmup_lr=kw["wl"])
        got = []
        for _ in range(len(M[key])):
            got.append(opt.param_groups[0]["lr"])
            assert sch.get_last_lr()[0] == opt.param_groups[0]["lr"]
            sch.step()
        np.testing.assert_allclose(got, M[key], rtol=1e-9, atol=1e-18, err_msg=key)
    with pytest.raises(ValueError):
        build_lr_scheduler(opt, "step", 0, 10)
    with pytest.raises(ValueError):
        build_lr_scheduler(opt, "cosine", 5, 10, warmup_type="exp")
    with pytest.raises(AssertionError):
        build_optimizer([p], "lion", 1e-3, 0.0)


def test_paths_and_names_match_reference():
    assert F.img_outdir("F", "ViT-B/16", "imagenet", "crop", 16, 1, "train") == str(M["path/img_train"])
    assert F.img_outdir("F", "ViT-B/16", "imagenet", "crop", 16, 1, "test") == str(M["path/img_test"])
    assert F.text_outdir("F", "ViT-B/16", "imagenet", "gpt3_cupl") == str(M["path/text"])
    assert ft.hparam_str("adamw", 0.001, 0.01, 32, 12800, 0.0, True) == str(M["path/hparam"])
    import argparse
    a = argparse.Namespace(common_dim=0)
    assert ft.savedir("E", "imagenet", "ViT-B/16", 16, 1, "gpt3_cupl", "average", "crop", "crossmodal", "zeroshot", 0.5,
                      0, "", a) == str(M["path/savedir_x"])
    assert ft.savedir("E", "sun397", "a-b", 4, 2, "gpt3_cupl", None, "flip", "image", "random", 0.0, 0, "tag",
                      a) == str(M["path/savedir_i"])


def test_presets_equal_reference_when_available():
    assert set(HYPER_DICT) == {"full_ds_full_model_finetune", "clip_linear", "linear", "audio"}
    assert HYPER_DICT["clip_linear"]["batch_size"] == [32] and HYPER_DICT["linear"]["learnable_temp"] == [True]
    assert REF_DEFAULTS["HYPER_DICT"] == HYPER_DICT


def test_bank_files_round_trip(tmp_path):
    g = torch.Generator().manual_seed(0)
    feats, labels = torch.randn(12, 8, generator=g), torch.arange(12) % 3
    tp = F.text_outdir(str(tmp_path), "ViT-B/16", "toy", "gpt3_cupl")
    F.write_text_bank(tp, feats, labels, lab2cname={0: "a", 1: "b", 2: "c"})
    d = F.load_text_bank(tp)
    assert torch.equal(d["features"], feats) and torch.equal(d["labels"], labels) and d["eot_indices"].shape == (12,)
    ip = F.img_outdir(str(tmp_path), "ViT-B/16", "toy", "crop", 4, 1, "train")
    F.write_image_bank(ip, train=(feats, labels), val=(feats[:6], labels[:6]), lab2cname={0: "a", 1: "b", 2: "c"})
    d = F.load_image_bank(ip)
    assert set(d) == {"train", "val", "lab2cname"} and set(d["train"]) == {"features", "labels", "paths"}
    tep = F.img_outdir(str(tmp_path), "ViT-B/16", "toy", "crop", 4, 1, "test")
    F.write_image_bank(tep, test=(feats, labels))
    assert torch.equal(F.load_image_bank(tep)["features"], feats)
    with pytest.raises(KeyError):
        torch.save({"features": feats, "labels": labels}, tp)
        F.load_text_bank(tp)


def test_config_parser_defaults_match_reference_when_available():
    from uml_b200.engine.config import parser
    ours = vars(parser.parse_args([]))
    assert ours["logit"] == 4.60517 and ours["num_workers"] == 4 and ours["modality"] == "image"
    for k, v in REF_DEFAULTS["parser_defaults"].items():
        assert ours[k] == v, k


def test_local_slice_partitions_a_global_batch():
    from uml_b200.engine.datasets.utils import IndexBatch
    bank = _bank(100)
    idx = torch.arange(37)
    b = IndexBatch(bank, idx, 37, 0, idx.clone())
    for world in (2, 3, 8):
        parts = [ft._local_slice(b, r, world) for r in range(world)]
        assert sum(p.n for p in parts) == 37 and max(p.n for p in parts) - min(p.n for p in parts) <= 1
        assert torch.equal(torch.cat([p.idx for p in parts]), idx)


@pytest.mark.parametrize("n", [0, 1, 2, 3, 63, 64, 65, 66, 1000, 29940, 300_007])
def test_native_randperm_is_bit_exact_with_torch(n):
    """uml_randperm_i64 (csrc/sampler.cu) == torch.randperm(n, generator=Generator().manual_seed(seed)), the call
    RandomSampler makes once per epoch; seeds above 32 bits are truncated like at::mt19937 does."""
    from uml_b200.engine.datasets.utils import _native_randperm
    g = torch.Generator()
    for seed in (0, 1, 5489, 2 ** 32 + 7, 2 ** 63 - 1, 0x5EADBEEFCAFEBABE):
        g.manual_seed(seed)
        want = torch.randperm(n, generator=g)
        got = _native_randperm(seed, n, pin=False)
        assert got.dtype == torch.int64 and torch.equal(got, want), (n, seed)


def test_threaded_incremental_permutation_gives_the_dataloader_stream():
    """Large banks: the epoch permutation is produced incrementally by a sampler thread while batches are consumed
    (uml_randperm_begin / uml_randperm_advance); the index stream must still be torch's DataLoader stream."""
    def stream(threaded):
        torch.manual_seed(77)
        ld = BankLoader(_bank(100_003), 9_001, shuffle=True)
        ld.async_min_rows = 16 if threaded else 10 ** 9
        it, out = iter(ld), []
        for s in range(30):  # crosses two epoch boundaries (12 batches per epoch, the last one short)
            b, it = ft.fetch_next(ld, it)
            out.append(b.host_idx.clone())
            assert torch.equal(b.idx.cpu(), b.host_idx)
        return torch.cat(out)

    torch.manual_seed(77)
    dl = torch.utils.data.DataLoader(torch.arange(100_003), batch_size=9_001, shuffle=True)
    want, it = [], iter(dl)
    for s in range(30):
        try:
            b = next(it)
        except StopIteration:
            it = iter(dl)
            b = next(it)
        want.append(b)
    want = torch.cat(want)
    assert torch.equal(stream(False), want)
    assert torch.equal(stream(True), want)


def test_incremental_randperm_prefixes_are_final():
    """After uml_randperm_advance(state, k) the first k entries already equal torch.randperm's."""
    import ctypes as C
    from uml_b200 import _lib
    lib = _lib.load()
    g = torch.Generator()
    for n, seed in ((1, 3), (2, 3), (65, 9), (1000, 2 ** 40 + 5), (70_001, 123)):
        g.manual_seed(seed)
        want = torch.randperm(n, generator=g)
        state = (C.c_ubyte * 3072)()
        out = torch.empty(n, dtype=torch.int64)
        _lib.check(lib.uml_randperm_begin(state, seed, n, out.data_ptr()))
        for upto in (0, 1, 7, 63, 64, 65, n // 3, n // 2 + 1, n - 1, n):
            upto = max(0, min(upto, n))
            _lib.check(lib.uml_randperm_advance(state, upto))
            assert torch.equal(out[:upto], want[:upto]), (n, seed, upto)
        assert torch.equal(out, want)


def test_gaussian_generate_data_is_bit_exact_with_the_reference():
    """uml_b200.gaussian.generate_data (data.py:29-61) against tensors recorded from the reference."""
    import ast
    from uml_b200 import gaussian as G
    cfg = ast.literal_eval(str(M["gauss/cfg"]))
    base = dict(seed=cfg["seed"], num_samples=cfg["num_samples"], dim_c=cfg["dim_c"], dim_x=cfg["dim_x"], dim_y=cfg["dim_y"],
                dim_obs=cfg["dim_obs"], noise_std=cfg["noise_std"], attenuate_x=True, attenuation=cfg["attenuation"])
    d1 = G.generate_data(dict(base, shared_latent_distribution_type="gaussian"))
    assert np.array_equal(d1["x"].numpy(), M["gauss/x"]) and np.array_equal(d1["y"].numpy(), M["gauss/y"])
    d2 = G.generate_data(dict(base, seed=44, shared_latent_distribution_type="laplace"))
    assert np.array_equal(d2["y"].numpy(), M["gauss/y_laplace"])


@pytest.mark.parametrize("upload", ["step", "epoch"])
def test_take_chunk_yields_the_per_step_stream(upload):
    """train() takes whole runs of batches inside an epoch at once (_BankIter.take_chunk: one sampler wait, one index
    upload); the batches must be exactly the ones next() would have produced, short last batch included."""
    def stream(chunked):
        torch.manual_seed(31)
        ld = BankLoader(_bank(1003), 64, shuffle=True, upload=upload)
        it, out = iter(ld), []
        while len(out) < 40:
            k = min(5, it.batches_left()) if chunked else 0
            if k >= 1:
                got = it.take_chunk(k)
            else:
                b, it = ft.fetch_next(ld, it)
                got = [b]
            for b in got:
                assert torch.equal(b.idx.cpu(), b.host_idx) and b.n == b.host_idx.numel()
                out.append(b.host_idx.clone())
        return out[:40]

    a, b = stream(False), stream(True)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert sorted(torch.cat(a[:16]).tolist()) == list(range(1003))  # an epoch = 15 full batches + one of 43 rows


def test_bank_v2_round_trip_is_lossless(tmp_path):
    """features.write_bank_v2 / load_bank_v2 / convert_bank: bit-identical features and labels, the bf16 shadow equals
    the on-device cast, class_order/class_starts reproduce the per-class row lists TextTensorDataset builds."""
    g = torch.Generator().manual_seed(8)
    feats, labels = torch.randn(1237, 40, generator=g), torch.randint(0, 17, (1237,), generator=g)
    eot = torch.randint(0, 77, (1237,), generator=g)
    v1 = str(tmp_path / "text.pth")
    F.write_text_bank(v1, feats, labels, eot, prompts={"a": ["x"]}, lab2cname={0: "zero"})
    (v2,) = F.convert_bank(v1)
    hdr = F.read_bank_v2_header(v2)
    assert hdr["rows"] == 1237 and hdr["dim"] == 40 and hdr["classes"] == int(labels.max()) + 1
    assert all(s["offset"] % 4096 == 0 for s in hdr["sections"].values())
    t, _, meta = F.load_bank_v2(v2, device="cpu")
    assert torch.equal(t["features"], feats) and torch.equal(t["labels"], labels) and torch.equal(t["eot_indices"], eot)
    assert torch.equal(t["features_bf16"], feats.to(torch.bfloat16))
    assert meta["prompts"] == {"a": ["x"]} and meta["lab2cname"] == {0: "zero"}
    for c in torch.unique(labels).tolist():
        rows = t["class_order"][t["class_starts"][c]:t["class_starts"][c + 1]]
        assert torch.equal(rows, torch.nonzero(labels == c, as_tuple=True)[0])
    # image train file: two splits
    v1i = str(tmp_path / "img.pth")
    F.write_image_bank(v1i, train=(feats[:800], labels[:800]), val=(feats[800:], labels[800:]), lab2cname={0: "zero"})
    files = F.convert_bank(v1i, str(tmp_path / "img.bank2"), with_bf16=False)
    assert [os.path.basename(f) for f in files] == ["img.bank2.train", "img.bank2.val"]
    tv, hv, _ = F.load_bank_v2(files[1], device="cpu")
    assert torch.equal(tv["features"], feats[800:]) and "features_bf16" not in tv and hv["rows"] == 437
    # load_feature_bank prefers the v2 file next to the v1 one and falls back to the v1 dict
    F.convert_bank(v1i)
    b2, m2 = F.load_feature_bank(v1i, device="cpu", split="train")
    assert torch.equal(b2.features, feats[:800]) and torch.equal(b2.labels, labels[:800]) and m2["lab2cname"] == {0: "zero"}
    assert torch.equal(b2.bf16(), feats[:800].to(torch.bfloat16))  # the shadow came from the file, no device cast needed
    os.remove(os.path.splitext(v1i)[0] + ".bank2.train")
    b1, _ = F.load_feature_bank(v1i, device="cpu", split="train")
    assert torch.equal(b1.features, b2.features) and torch.equal(b1.labels, b2.labels)


# ------------------------------------------------------------------------------------------------
# sweep batching: a private generator standing in for the global one, and run-wise advancing
# ------------------------------------------------------------------------------------------------

def _drive(img, txt, val, steps, eval_every):
    """The order in which train() touches its loaders: iter(image), iter(text); per step image batch then text batch
    (re-iterating on exhaustion); an iter(val) per evaluation."""
    seq = []
    ii, ti = iter(img), iter(txt)
    for s in range(steps):
        for name in ("i", "t"):
            ld, it = (img, ii) if name == "i" else (txt, ti)
            try:
                b = next(it)
            except StopIteration:
                it = iter(ld)
                b = next(it)
            if name == "i":
                ii = it
            else:
                ti = it
            seq.append(b.host_idx.clone())
        if s % eval_every == 0:
            iter(val)
    return seq


@pytest.mark.parametrize("nw", [0, 2])
def test_private_rng_reproduces_the_global_stream(nw):
    mk = lambda rng: (BankLoader(_bank(53), 8, shuffle=True, num_workers=nw, rng=rng),
                      BankLoader(_bank(31), 8, shuffle=True, num_workers=nw, rng=rng),
                      BankLoader(_bank(20), 8, shuffle=False, num_workers=nw, rng=rng))
    torch.manual_seed(4242)
    want = _drive(*mk(None), steps=30, eval_every=7)
    torch.manual_seed(1)  # the global stream must not matter any more
    got = _drive(*mk(torch.Generator().manual_seed(4242)), steps=30, eval_every=7)
    assert len(want) == len(got) == 60
    for a, b in zip(want, got):
        assert torch.equal(a, b)


def test_take_run_matches_batchwise_iteration():
    """take_run(k) advances exactly like k next() calls (same draws, same spans), including across epoch ends."""
    g1, g2 = torch.Generator().manual_seed(9), torch.Generator().manual_seed(9)
    a, b = BankLoader(_bank(53), 8, shuffle=True, rng=g1), BankLoader(_bank(53), 8, shuffle=True, rng=g2)
    ia, ib = iter(a), iter(b)
    for want_k in (1, 3, 10, 2, 7, 7, 1):
        if ia.batches_left() == 0:
            ia = iter(a)
        k = min(want_k, ia.batches_left())
        perm, start, total = ia.take_run(k)
        got = perm[start:start + total]
        ref = []
        for _ in range(k):
            try:
                x = next(ib)
            except StopIteration:
                ib = iter(b)
                x = next(ib)
            ref.append(x.host_idx)
        assert torch.equal(got, torch.cat(ref))


def test_take_run_ragged_shapes_property():
    """take_run against batch-wise iteration over many (bank rows, batch size, drop_last, num_workers, chunking) shapes:
    banks shorter than a batch, exact multiples, one-row tails."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(n=st.integers(1, 70), bs=st.integers(1, 24), drop=st.booleans(), nw=st.sampled_from([0, 2]),
           seed=st.integers(0, 2 ** 31), chunks=st.lists(st.integers(1, 9), min_size=3, max_size=8))
    def check(n, bs, drop, nw, seed, chunks):
        if drop and n < bs:
            return  # such a loader yields nothing (len == 0), as the reference's DataLoader would
        g1, g2 = torch.Generator().manual_seed(seed), torch.Generator().manual_seed(seed)
        a = BankLoader(_bank(n), bs, shuffle=True, drop_last=drop, num_workers=nw, rng=g1)
        b = BankLoader(_bank(n), bs, shuffle=True, drop_last=drop, num_workers=nw, rng=g2)
        ia, ib = iter(a), iter(b)
        for want in chunks:
            if ia.batches_left() == 0:
                ia = iter(a)
            k = min(want, ia.batches_left())
            perm, start, total = ia.take_run(k)
            ref = []
            for _ in range(k):
                try:
                    x = next(ib)
                except StopIteration:
                    ib = iter(b)
                    x = next(ib)
                ref.append(x.host_idx)
            assert torch.equal(perm[start:start + total], torch.cat(ref))
            assert g1.get_state().equal(g2.get_state())  # both consumed the same draws

    check()


def test_text_selection_through_the_class_index_matches_the_mask_per_class_form(tmp_path):
    """n-shot selection and class averaging walk the class-sorted row index (computed here, or read from a v2 bank
    file - SURVEY 8f-2) and must pick exactly the rows the reference's mask-per-class loops pick
    (engine/datasets/utils.py:76-98), with the same RNG draws, classes without rows included."""
    import torch
    from uml_b200 import features as F
    from uml_b200.engine.datasets.utils import TextTensorDataset

    g = torch.Generator().manual_seed(4)
    n, d, c = 700, 24, 41
    labels = torch.randint(0, c, (n,), generator=g)
    labels[labels == 7] = 8      # a class id without rows
    labels[labels == 40] = 3     # ... and the largest one
    feats = torch.randn(n, d, generator=g)
    eot = torch.randint(0, 77, (n,), generator=g)

    def reference_select(k):
        out = []
        for cls in torch.unique(labels):
            inds = (labels == cls).nonzero(as_tuple=True)[0]
            out.append(inds[torch.randperm(inds.size(0))[: min(k, inds.size(0))]])
        return torch.cat(out)

    path = str(tmp_path / "text.bank2")
    F.write_bank_v2(path, feats, labels, eot_indices=eot)
    t, _, _ = F.load_bank_v2(path, "cpu")
    for k in (1, 3, 64):
        torch.manual_seed(11)
        want = reference_select(k)
        state_after = torch.random.get_rng_state()
        for kw in ({}, {"class_order": t["class_order"], "class_starts": t["class_starts"]}):
            torch.manual_seed(11)
            ds = TextTensorDataset(feats, labels, eot, n_shots=k, **kw)
            assert torch.equal(ds.label_tensor, labels[want]) and torch.equal(ds.input_tensor, feats[want])
            assert torch.equal(ds.eot_indices, eot[want])
            assert torch.equal(torch.random.get_rng_state(), state_after)   # the same number of draws
    for kw in ({}, {"class_order": t["class_order"], "class_starts": t["class_starts"]}):
        ds = TextTensorDataset(feats, labels, eot, n_shots="average", **kw)
        classes = torch.unique(labels)
        assert torch.equal(ds.label_tensor, classes)
        want_mean = torch.stack([feats[labels == cls].mean(0) for cls in classes])
        torch.testing.assert_close(ds.input_tensor, want_mean, rtol=1e-5, atol=1e-6)
        assert torch.equal(ds.eot_indices, torch.stack([eot[labels == cls][0] for cls in classes]))
