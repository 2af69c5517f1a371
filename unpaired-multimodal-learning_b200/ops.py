"""Tensor-level wrappers over the C ABI (include/uml_b200.h).

PyTorch is used for device memory and streams only; every function launches hand-written sm_100a
kernels from libuml_b200.so on ``torch.cuda.current_stream()`` and never synchronises the host.
Inputs must live on a CUDA device - there is deliberately no CPU or eager fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import Segment, SegStats, TcSegments, Update, check

UPDATE_KINDS = {"none": 0, "adamw": 1, "adam": 2, "sgd": 3}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype, name: str, contiguous: bool = True):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name}: expected a CUDA tensor (uml_b200 has no CPU path)")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if contiguous and not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")
    return t


@dataclass
class Run:
    """One run of rows pushed through the shared head in a step (image batch or text batch)."""
    rows: torch.Tensor                 # [N, D] fp32 feature bank (or dense batch when idx is None)
    labels: torch.Tensor               # [N] int64
    idx: Optional[torch.Tensor]        # [n] int64 indices into rows/labels, or None
    n: int
    scale: float = 1.0
    loss_weight: float = 1.0
    label_idx: Optional[torch.Tensor] = None   # indices into labels when rows are dense (adapter output)
    scale_dev: Optional[torch.Tensor] = None   # 0-dim fp32 CUDA tensor overriding `scale` (learnable temperature)

    def c_segment(self) -> Segment:
        _need(self.rows, torch.float32, "run.rows")
        _need(self.labels, torch.int64, "run.labels")
        if self.idx is not None:
            _need(self.idx, torch.int64, "run.idx")
            if self.idx.numel() < self.n:
                raise ValueError("run.idx shorter than run.n")
        elif self.rows.shape[0] < self.n:
            raise ValueError("run.rows shorter than run.n")
        if self.scale_dev is not None:
            _need(self.scale_dev, torch.float32, "run.scale_dev")
        return Segment(self.rows.data_ptr(), _ptr(self.idx), self.labels.data_ptr(), int(self.n),
                       int(self.rows.stride(0)), float(self.scale), float(self.loss_weight), _ptr(self.label_idx),
                       _ptr(self.scale_dev))


def _segs(runs: Sequence[Run]):
    if not 1 <= len(runs) <= 2:
        raise ValueError("1 or 2 runs per step")
    arr = (Segment * len(runs))(*[r.c_segment() for r in runs])
    return arr, len(runs)


def make_update(kind: str, lr: float, step: int, m: Optional[torch.Tensor], v: Optional[torch.Tensor],
                weight_decay: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8, momentum: float = 0.9) -> Update:
    return Update(UPDATE_KINDS[kind], float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                  float(momentum), int(step), _ptr(m), _ptr(v))


# ------------------------------------------------------------------------------------------ K1

def gather_rows(bank: torch.Tensor, idx: torch.Tensor, out: Optional[torch.Tensor] = None,
                dtype=torch.float32) -> torch.Tensor:
    _need(bank, torch.float32, "bank")
    _need(idx, torch.int64, "idx")
    n, d = idx.numel(), bank.shape[1]
    if out is None:
        out = torch.empty((n, d), device=bank.device, dtype=dtype)
    lib = _lib.load()
    if out.dtype == torch.float32:
        check(lib.uml_gather_rows_f32(bank.data_ptr(), bank.shape[0], d, idx.data_ptr(), n, out.data_ptr(), _stream()))
    elif out.dtype == torch.bfloat16:
        check(lib.uml_gather_rows_bf16(bank.data_ptr(), bank.shape[0], d, idx.data_ptr(), n, out.data_ptr(),
                                       out.stride(0), _stream()))
    else:
        raise TypeError("gather_rows: out must be float32 or bfloat16")
    return out


def gather_rows_labels(bank, labels, idx, out16, out_labels32):
    """bf16 row gather that also gathers the rows' int64 bank labels into int32 (one launch)."""
    _need(bank, torch.float32, "bank")
    _need(labels, torch.int64, "labels")
    _need(idx, torch.int64, "idx")
    check(_lib.load().uml_gather_rows_labels_bf16(bank.data_ptr(), labels.data_ptr(), bank.shape[1], idx.data_ptr(),
                                                  idx.numel(), out16.data_ptr(), out16.stride(0), out_labels32.data_ptr(),
                                                  _stream()))


def gather2_rows_bf16(bank0, labels0, idx0, bank1, labels1, idx1, out16, out_labels32=None, light=False):
    """Both runs of a step copied from bf16 shadow banks into one operand (rows of run 0, then run 1) with their
    labels, in one launch of the TMA copy kernel (``light``: of the register-copy kernel the training step uses).
    Either run may be None."""
    d = out16.shape[1]
    args = []
    for bank, labels, idx, nm in ((bank0, labels0, idx0, "0"), (bank1, labels1, idx1, "1")):
        if bank is None:
            args += [None, None, None, 0]
            continue
        _need(bank, torch.bfloat16, "bank" + nm)
        _need(idx, torch.int64, "idx" + nm)
        if labels is not None:
            _need(labels, torch.int64, "labels" + nm)
        if bank.shape[1] != d:
            raise ValueError("gather2_rows_bf16: bank width differs from the output width")
        args += [bank.data_ptr(), _ptr(labels), idx.data_ptr(), idx.numel()]
    _need(out16, torch.bfloat16, "out16", contiguous=False)
    if args[3] + args[7] > out16.shape[0]:
        raise ValueError("gather2_rows_bf16: output too small")
    fn = _lib.load().uml_gather2_rows_bf16_light if light else _lib.load().uml_gather2_rows_bf16
    check(fn(*args, d, out16.data_ptr(), out16.stride(0), _ptr(out_labels32), _stream()))
    return out16


def gather_labels(labels: torch.Tensor, idx: Optional[torch.Tensor], n: int, out: torch.Tensor) -> torch.Tensor:
    _need(labels, torch.int64, "labels")
    _need(out, torch.int32, "out")
    check(_lib.load().uml_gather_labels_i32(labels.data_ptr(), _ptr(idx), n, out.data_ptr(), _stream()))
    return out


def cast_bf16(src: torch.Tensor, dst: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need(src, torch.float32, "src")
    if dst is None:
        dst = torch.empty(src.shape, device=src.device, dtype=torch.bfloat16)
    check(_lib.load().uml_cast_f32_to_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()))
    return dst


# ------------------------------------------------------------------------------------------ fp32 head

class HeadWorkspace:
    """Caller-owned scratch for one head step (the library never allocates)."""

    def __init__(self, max_rows: int, n_classes: int, device, bf16: bool = False):
        self.max_rows, self.n_classes = int(max_rows), int(n_classes)
        self.ldg = ((n_classes + 63) // 64) * 64
        # fp32 workspaces of small steps get room for 8 split-K planes of raw logits (a few MB): the latency-bound
        # reference-batch forward then spreads its contraction over the whole machine
        g_rows = max_rows if (bf16 or max_rows > 2048) else 8 * max_rows
        self.G = torch.empty((g_rows, self.ldg), device=device, dtype=torch.bfloat16 if bf16 else torch.float32)
        self.row_loss = torch.empty(max_rows, device=device, dtype=torch.float32)
        self.row_correct = torch.empty(max_rows, device=device, dtype=torch.int32)
        self.row_dscale = torch.empty(max_rows, device=device, dtype=torch.float32)
        self.stats = torch.zeros((2, 4), device=device, dtype=torch.float32)  # 2 x uml_seg_stats (16 B each)
        # UML_TILE_WS_FLOATS(max_rows): per-tile partial sums written by the tensor-core forward
        # (zero-initialised: the forward kernel keeps its launch epoch and exchange flags in the first words)
        self.fac = (torch.zeros(16 + ((max_rows + 255) // 256) * 264 + max_rows * 32, device=device, dtype=torch.float32)
                    if bf16 else None)

    def read_stats(self):
        """Host copy of the two uml_seg_stats records (synchronises)."""
        raw = self.stats.cpu()
        ints = raw.view(torch.int32)
        return [dict(loss_mean=float(raw[i, 0]), dscale=float(raw[i, 1]), correct=int(ints[i, 2]), n=int(ints[i, 3]))
                for i in range(2)]


def head_fwd_ce_f32(runs: Sequence[Run], W: torch.Tensor, ws: HeadWorkspace, stats: Optional[torch.Tensor] = None):
    """logits -> softmax CE -> G (in ws.G), per-run stats in ``stats`` (default ws.stats).  finetune.py:181-188."""
    _need(W, torch.float32, "W")
    arr, n = _segs(runs)
    total = sum(r.n for r in runs)
    if total > ws.max_rows:
        raise ValueError("workspace too small")
    stats = ws.stats if stats is None else stats
    check(_lib.load().uml_head_fwd_ce_f32(arr, n, W.shape[1], W.data_ptr(), W.shape[0], ws.G.data_ptr(), ws.ldg,
                                          ws.row_loss.data_ptr(), ws.row_correct.data_ptr(), ws.row_dscale.data_ptr(),
                                          stats.data_ptr(), ws.G.shape[0], _stream()))


def head_bwd_dw_f32(runs: Sequence[Run], W: torch.Tensor, ws: HeadWorkspace, dW: Optional[torch.Tensor] = None,
                    update: Optional[Update] = None):
    """dW = G^T X; with ``update`` the optimizer step is applied to W in the GEMM epilogue."""
    _need(W, torch.float32, "W")
    arr, n = _segs(runs)
    check(_lib.load().uml_head_bwd_dw_f32(arr, n, W.shape[1], ws.G.data_ptr(), ws.ldg, W.shape[0], W.data_ptr(),
                                          _ptr(dW), C.byref(update) if update is not None else None, _stream()))


def head_step_fused_f32(runs: Sequence[Run], W: torch.Tensor, ws: HeadWorkspace, update: Update,
                        stats: Optional[torch.Tensor] = None) -> bool:
    """The whole exact step (logits, softmax CE, dW, optimizer update, per-run stats) in one cooperative launch.
    Returns False - and launches nothing - when the shape does not fit the kernel's contract; the caller then takes
    head_fwd_ce_f32 + head_bwd_dw_f32.  finetune.py:181-195."""
    _need(W, torch.float32, "W")
    arr, n = _segs(runs)
    if sum(r.n for r in runs) > ws.max_rows:
        raise ValueError("workspace too small")
    stats = ws.stats if stats is None else stats
    launched = C.c_int32(0)
    check(_lib.load().uml_head_step_fused_f32(arr, n, W.shape[1], W.data_ptr(), W.shape[0], ws.G.data_ptr(), ws.ldg,
                                              ws.row_loss.data_ptr(), ws.row_correct.data_ptr(), ws.row_dscale.data_ptr(),
                                              stats.data_ptr(), C.byref(update), C.byref(launched), _stream()))
    if launched.value:
        _lib.LAUNCH_COUNT[0] += 1
    return bool(launched.value)


def gemm_nt(A: torch.Tensor, B: torch.Tensor, out: torch.Tensor, alpha: float = 1.0,
            a_row_idx: Optional[torch.Tensor] = None, m: Optional[int] = None):
    """out[m,n] = alpha * sum_k A[row(m),k] B[n,k]"""
    m = out.shape[0] if m is None else m
    check(_lib.load().uml_gemm_nt_f32(A.data_ptr(), A.stride(0), _ptr(a_row_idx), B.data_ptr(), B.stride(0),
                                      out.data_ptr(), out.stride(0), m, B.shape[0], B.shape[1], alpha, _stream()))


def gemm_nn(A: torch.Tensor, B: torch.Tensor, out: torch.Tensor, alpha: float = 1.0, m: Optional[int] = None,
            k: Optional[int] = None):
    """out[m,n] = alpha * sum_k A[m,k] B[k,n]"""
    m = out.shape[0] if m is None else m
    k = B.shape[0] if k is None else k
    check(_lib.load().uml_gemm_nn_f32(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), out.data_ptr(),
                                      out.stride(0), m, B.shape[1], k, alpha, _stream()))


def gemm_tn(A: torch.Tensor, B: torch.Tensor, out: Optional[torch.Tensor], k: int, m: int, n: int, alpha: float = 1.0,
            b_row_idx: Optional[torch.Tensor] = None, P: Optional[torch.Tensor] = None,
            update: Optional[Update] = None, ldc: Optional[int] = None):
    """out[m,n] = alpha * sum_k A[k,m] B[row(k),n]  (+ fused optimizer update of P)"""
    ldc = (out.stride(0) if out is not None else P.stride(0)) if ldc is None else ldc
    check(_lib.load().uml_gemm_tn_f32(A.data_ptr(), A.stride(0), B.data_ptr(), B.stride(0), _ptr(b_row_idx), _ptr(out),
                                      ldc, m, n, k, alpha, _ptr(P), C.byref(update) if update is not None else None,
                                      _stream()))


# ------------------------------------------------------------------------------------------ K6

def adamw_step(p, g, m, v, *, lr, step, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8, decoupled=True,
               g2=None, g2_weight=0.0, shadow=None):
    for t, nm in ((p, "p"), (g, "g"), (m, "m"), (v, "v")):
        _need(t, torch.float32, nm)
    check(_lib.load().uml_adamw_step(p.data_ptr(), g.data_ptr(), _ptr(g2), float(g2_weight), m.data_ptr(), v.data_ptr(),
                                     p.numel(), lr, betas[0], betas[1], eps, weight_decay, step, int(decoupled),
                                     _ptr(shadow), _stream()))


def adamw_step_partials(p, partials, n_splits, m, v, *, lr, step, weight_decay=0.0, betas=(0.9, 0.999), eps=1e-8,
                        decoupled=True, shadow=None, g_out=None):
    _need(p, torch.float32, "p")
    _need(partials, torch.float32, "partials")
    check(_lib.load().uml_adamw_step_partials(p.data_ptr(), partials.data_ptr(), n_splits, p.numel(), m.data_ptr(),
                                              v.data_ptr(), p.numel(), lr, betas[0], betas[1], eps, weight_decay, step,
                                              int(decoupled), _ptr(shadow), _ptr(g_out), _stream()))


def sgd_step(p, g, buf, *, lr, step, momentum=0.9, weight_decay=0.0, g2=None, g2_weight=0.0, shadow=None):
    for t, nm in ((p, "p"), (g, "g"), (buf, "buf")):
        _need(t, torch.float32, nm)
    check(_lib.load().uml_sgd_step(p.data_ptr(), g.data_ptr(), _ptr(g2), float(g2_weight), buf.data_ptr(), p.numel(),
                                   lr, momentum, weight_decay, step, _ptr(shadow), _stream()))


# ------------------------------------------------------------------------------------------ K7 / K8

def eval_f32(feats, labels, W, scale, row_loss, row_pred):
    _need(feats, torch.float32, "feats")
    _need(labels, torch.int64, "labels")
    _need(W, torch.float32, "W")
    check(_lib.load().uml_eval_f32(feats.data_ptr(), feats.stride(0), labels.data_ptr(), feats.shape[0], feats.shape[1],
                                   W.data_ptr(), W.shape[0], float(scale), row_loss.data_ptr(), row_pred.data_ptr(),
                                   _stream()))


def eval_reduce(row_loss, row_pred, labels, batch_size, out_loss, out_correct):
    """labels=None: row_pred holds 0/1 hit flags instead of predicted classes."""
    check(_lib.load().uml_eval_reduce(row_loss.data_ptr(), row_pred.data_ptr(), _ptr(labels), row_loss.numel(),
                                      int(batch_size), out_loss.data_ptr(), out_correct.data_ptr(), _stream()))


def eval_group_f32(feats, labels, W_slab, w_stride, head_ids, scales, n_classes, row_loss, row_pred):
    """Evaluation of several heads of a sweep group over one bank in ONE launch: head h's weights at
    ``W_slab.data_ptr() + head_ids[h] * w_stride`` floats; ``row_loss`` / ``row_pred``: [n_heads, n_rows]."""
    import ctypes as C
    _need(feats, torch.float32, "feats")
    _need(labels, torch.int64, "labels")
    _need(W_slab, torch.float32, "W")
    k = len(head_ids)
    ids = (C.c_int32 * k)(*[int(h) for h in head_ids])
    sc = (C.c_float * k)(*[float(x) for x in scales])
    check(_lib.load().uml_eval_group_f32(feats.data_ptr(), feats.stride(0), labels.data_ptr(), feats.shape[0], feats.shape[1],
                                         W_slab.data_ptr(), int(w_stride), ids, sc, k, int(n_classes), row_loss.data_ptr(),
                                         row_pred.data_ptr(), _stream()))


def eval_reduce_group(row_loss, row_pred, labels, batch_size, out_loss, out_correct):
    """row_loss / row_pred: [n_heads, n_rows] -> out_loss / out_correct: [n_heads]."""
    check(_lib.load().uml_eval_reduce_group(row_loss.data_ptr(), row_pred.data_ptr(), _ptr(labels), row_loss.shape[1],
                                            int(batch_size), row_loss.shape[0], out_loss.data_ptr(), out_correct.data_ptr(),
                                            _stream()))


def cka_linear(a, b):
    """Linear CKA (biased HSIC) of two feature sets with the same number of rows - reference ``metrics.py:96-119`` with
    ``kernel_metric='ip'`` - as a one-element device tensor.  O(n d^2): no n x n kernel matrices."""
    _need(a, torch.float32, "a", contiguous=False)
    _need(b, torch.float32, "b", contiguous=False)
    if a.dim() != 2 or b.dim() != 2 or a.shape[0] != b.shape[0] or a.stride(1) != 1 or b.stride(1) != 1:
        raise ValueError("cka_linear: expected [n, da] and [n, db] with contiguous rows")
    lib = _lib.load()
    ws = torch.empty(int(lib.uml_cka_workspace_doubles(a.shape[1], b.shape[1])), device=a.device, dtype=torch.float64)
    out = torch.empty(1, device=a.device)
    check(lib.uml_cka_linear_f32(a.data_ptr(), a.stride(0), a.shape[1], b.data_ptr(), b.stride(0), b.shape[1], a.shape[0],
                                 ws.data_ptr(), out.data_ptr(), _stream()))
    return out


def mutual_knn(a, b, topk: int = 10):
    """Mutual k-nearest-neighbour accuracy (reference ``metrics.py:55-86``, ``topk=10`` at both call sites) as a one-element
    device tensor: mean over rows of the overlap of the row's top-k inner-product neighbours in the two feature spaces."""
    _need(a, torch.float32, "a", contiguous=False)
    _need(b, torch.float32, "b", contiguous=False)
    if a.dim() != 2 or b.dim() != 2 or a.shape[0] != b.shape[0] or a.stride(1) != 1 or b.stride(1) != 1:
        raise ValueError("mutual_knn: expected [n, da] and [n, db] with contiguous rows")
    n = a.shape[0]
    ws = torch.empty(2 * n * topk + 1, device=a.device, dtype=torch.int32)
    out = torch.empty(1, device=a.device)
    check(_lib.load().uml_mutual_knn_f32(a.data_ptr(), a.stride(0), a.shape[1], b.data_ptr(), b.stride(0), b.shape[1], n, int(topk),
                                         ws.data_ptr(), out.data_ptr(), _stream()))
    return out


def grad_diag(a, b, workspace, out4):
    check(_lib.load().uml_grad_diag(a.data_ptr(), b.data_ptr(), a.numel(), workspace.data_ptr(), out4.data_ptr(),
                                    _stream()))


def grad_diag_record(dot: float, aa: float, bb: float, agree: float, numel: int, both: bool) -> dict:
    """The reference's gradient-probe logger keys (finetune.py:200-206) from the four sums of ``grad_diag`` /
    ``uml_sweep_run_diag`` over the image-loss gradient A and the text-loss gradient B of the head weights (``numel``
    elements each); ``both``: the step had rows of both modalities (else the cosine and agreement are 0)."""
    ni, nt = float(aa) ** 0.5, float(bb) ** 0.5
    return {"train/grad_direction_sim": float(dot) / (ni * nt) if both and ni > 0 and nt > 0 else 0.0,
            "train/img_grad_norm": ni, "train/txt_grad_norm": nt,
            "train/grad_agreement_rate": float(agree) / numel if both else 0.0}


# ------------------------------------------------------------------------------------------ tensor-core head

def tc_segments(rows: Sequence[int], scales: Sequence[float], weights: Sequence[float],
                scale_dev: Optional[Sequence[Optional[torch.Tensor]]] = None) -> TcSegments:
    s = TcSegments()
    s.nseg = len(rows)
    for i in range(len(rows)):
        s.seg_rows[i], s.scale[i], s.loss_weight[i] = int(rows[i]), float(scales[i]), float(weights[i])
        s.scale_dev[i] = _ptr(scale_dev[i]) if scale_dev is not None else None
    return s


def tile_workspace(max_rows: int, device):
    """Zero-initialised UML_TILE_WS_FLOATS(max_rows) scratch of the tensor-core forward (launch epoch, exchange records)."""
    return torch.zeros(16 + ((max_rows + 255) // 256) * 264 + max_rows * 32, device=device, dtype=torch.float32)


def head_fwd_ce_bf16(X, W_bf16, labels_i32, segs: TcSegments, ws: Optional[HeadWorkspace], row_loss=None, row_pred=None,
                     row_correct=None, row_dscale=None, n_rows: Optional[int] = None, stats=None, tile_ws=None):
    """``stats`` (optional, training mode only): [nseg, 4] fp32 record of the per-run statistics.  ``ws=None`` is the
    evaluation mode (no G); with ``tile_ws`` (``tile_workspace(n_rows)``) it runs the exchange kernel, else the
    chunk-sequential one."""
    _need(X, torch.bfloat16, "X")
    _need(W_bf16, torch.bfloat16, "W")
    _need(labels_i32, torch.int32, "labels")
    n_rows = X.shape[0] if n_rows is None else n_rows
    G, ldg, fac = (ws.G.data_ptr(), ws.ldg, ws.fac.data_ptr()) if ws is not None else (None, 0, _ptr(tile_ws))
    check(_lib.load().uml_head_fwd_ce_bf16(X.data_ptr(), n_rows, X.shape[1], W_bf16.data_ptr(), W_bf16.shape[0],
                                           labels_i32.data_ptr(), C.byref(segs), G, ldg, _ptr(row_loss),
                                           _ptr(row_pred), _ptr(row_correct), _ptr(row_dscale), fac,
                                           _ptr(stats) if ws is not None else None, _stream()))


def tc_dw_splits(n_rows: int, dim: int, n_classes: int) -> int:
    return int(_lib.load().uml_tc_dw_splits(n_rows, dim, n_classes))


def head_bwd_dw_bf16(G, ldg, X, n_rows, n_classes, partials, n_splits):
    _need(G, torch.bfloat16, "G")
    _need(X, torch.bfloat16, "X")
    _need(partials, torch.float32, "partials")
    check(_lib.load().uml_head_bwd_dw_bf16(G.data_ptr(), ldg, X.data_ptr(), n_rows, X.shape[1], n_classes,
                                           partials.data_ptr(), n_splits, _stream()))


def gemm_bf16(A, B, out, M, N, K, a_mn=False, b_mn=False, n_splits=1):
    """D[m,n] = sum_k A(m,k) B(k,n) on the tensor cores.  A: [M,K] (or [K,M] when a_mn); B: [N,K] (or [K,N] when
    b_mn); out: bf16 [M, ld] or fp32 partials [n_splits, M, N]."""
    _need(A, torch.bfloat16, "A", contiguous=False)
    _need(B, torch.bfloat16, "B", contiguous=False)
    out_bf16 = out.dtype == torch.bfloat16
    ldo = out.stride(0) if out_bf16 else out.stride(-2)
    check(_lib.load().uml_gemm_bf16(A.data_ptr(), A.stride(0), int(a_mn), B.data_ptr(), B.stride(0), int(b_mn), M, N, K,
                                    out.data_ptr(), ldo, int(out_bf16), n_splits, _stream()))


def gemm_bf16_splits(M, N, K):
    return int(_lib.load().uml_gemm_bf16_splits(M, N, K))


def sum_partials(partials, n_splits, n, out):
    check(_lib.load().uml_sum_partials(partials.data_ptr(), n_splits, n, n, out.data_ptr(), _stream()))


def reduce_tile_stats(tile_ws, n_rows, nseg, stats):
    check(_lib.load().uml_reduce_tile_stats(tile_ws.data_ptr(), int(n_rows), int(nseg), stats.data_ptr(), _stream()))


def reduce_seg_stats(row_loss, row_correct, row_dscale, seg_rows: Sequence[int], stats):
    arr = (C.c_int64 * len(seg_rows))(*[int(x) for x in seg_rows])
    check(_lib.load().uml_reduce_seg_stats(row_loss.data_ptr(), row_correct.data_ptr(), _ptr(row_dscale), arr,
                                           len(seg_rows), stats.data_ptr(), _stream()))
