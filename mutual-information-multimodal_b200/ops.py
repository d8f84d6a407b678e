"""Stage-level wrappers over the C ABI (include/mi_b200.h) for torch CUDA tensors.

PyTorch is used here for device memory, streams and dtype bookkeeping only; every FLOP of the hot
path runs in libmi_b200.so.  All functions raise ``MIError`` on failure — there is no fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple, Union

import torch

from . import _lib

CRITIC = {"dot": 0, "bilinear": 1}
ESTIMATOR = {"dv": 0, "infonce": 1, "infonce_ref": 1, "infonce_row": 2, "infonce_sym": 3, "js": 4, "nwj": 5}
# the f-divergence bounds run on the single-GPU separable critics only (dot / bilinear, critic_loss_fwd_bwd)
SEPARABLE_ONLY = ("js", "nwj")
PRECISION = {"fast": 0, "strict": 1}
# the MLP critic's entries also take "fp32": three bf16 pieces per operand (24 significant bits, MI_PREC_FP32X3); the
# separable, sharded-separable and GDV paths read PRECISION above and reject it before any launch
MLP_PRECISION = dict(PRECISION, fp32=4)


class MIError(RuntimeError):
    pass


class SplitBF16:
    """A matrix kept as a hi/lo bf16 pair ("strict", fp32-accumulate mode): ``data`` is
    [rows, 2 * round_up(width, 128)] with hi in columns [0, width) and lo starting at column
    round_up(width, 128); value = hi + lo."""

    def __init__(self, data: torch.Tensor, width: int):
        self.data = data
        self.width = width

    @property
    def shape(self):
        return (self.data.shape[0], self.width)

    @property
    def device(self):
        return self.data.device

    def float(self) -> torch.Tensor:
        dp = self.data.shape[1] // 2
        return self.data[:, :self.width].float() + self.data[:, dp:dp + self.width].float()


Mat = Union[torch.Tensor, SplitBF16]


def _check(status: int, what: str) -> None:
    if status != 0:
        lib = _lib.load()
        msg = lib.mi_status_string(status).decode()
        if status == -3:
            msg += ": " + lib.mi_last_cuda_error().decode()
        raise MIError(f"{what} failed: {msg}")


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if isinstance(t, SplitBF16):
            t = t.data
        if t is not None and not t.is_cuda:
            raise MIError("mi_b200 has no CPU path: tensors must live on a CUDA (sm_100) device")


def _opnd(m: Mat):
    """(tensor, pitch, split flag, logical width) of a plain or hi/lo operand."""
    if isinstance(m, SplitBF16):
        return m.data, m.data.stride(0), 2, m.width
    assert m.dtype == torch.bfloat16 and m.dim() == 2
    if m.stride(1) != 1 or m.stride(0) % 8:
        m = m.contiguous()
    if m.stride(0) % 8:
        raise MIError("operands need a row pitch that is a multiple of 8 elements (TMA: 16-byte strides)")
    return m, m.stride(0), 1, m.shape[1]


def _round_up(a, b):
    return (a + b - 1) // b * b


def new_split(rows: int, width: int, device) -> SplitBF16:
    return SplitBF16(torch.zeros((rows, 2 * _round_up(width, 128)), dtype=torch.bfloat16, device=device), width)


_workspaces = {}


def workspace(nbytes: int, device) -> torch.Tensor:
    """Persistent scratch per (device, stream), grown on demand.  The library reuses it in stream order, so a
    buffer must never be shared between streams; a buffer that is outgrown is handed back to the caching allocator
    with ``record_stream`` semantics (it was only ever used on its own stream).  CUDA-graph steps do NOT use this
    cache: a captured graph bakes the pointer in, so ``GraphedCriticStep`` owns a private workspace tensor."""
    idx = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if torch.cuda.is_current_stream_capturing():
        raise MIError("the shared workspace cache cannot be used under CUDA-graph capture: pass workspace=")
    key = (idx, torch.cuda.current_stream(idx).cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=f"cuda:{idx}")
        _workspaces[key] = buf
    return buf


def as_bf16(x: torch.Tensor) -> torch.Tensor:
    """bf16, contiguous; fp32 inputs go through the library's cast kernel."""
    _need_cuda(x)
    if x.dtype == torch.bfloat16:
        return x.detach().contiguous()
    x = x.detach().contiguous().float()
    out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    if x.numel():
        _check(_lib.load().mi_cast_f32_to_bf16(_ptr(x), _ptr(out), x.numel(), _stream()), "mi_cast_f32_to_bf16")
    return out


def _gemm_mn(A: Mat, B: Mat, a_t: bool, b_t: bool, out_dtype, out_split: bool):
    At, lda, asp, wa = _opnd(A)
    Bt, ldb, bsp, wb = _opnd(B)
    K = At.shape[0] if a_t else wa
    assert K == (Bt.shape[0] if b_t else wb), "inner dimensions differ"
    M = wa if a_t else At.shape[0]
    N = wb if b_t else Bt.shape[0]
    of = ob = None
    ld16 = 0
    if out_split:
        res = new_split(M, N, At.device)
        ob, ld16 = res.data, res.data.stride(0)
    elif out_dtype == torch.bfloat16:
        res = torch.empty((M, N), dtype=torch.bfloat16, device=At.device)
        ob, ld16 = res, N
    else:
        res = torch.empty((M, N), dtype=torch.float32, device=At.device)
        of = res
    lib = _lib.load()
    ws = workspace(lib.mi_gemm_bf16_mn_workspace_bytes(M, N, K, asp, int(a_t), bsp, int(b_t)), At.device)
    _check(lib.mi_gemm_bf16_mn(_ptr(At), lda, asp, int(a_t), _ptr(Bt), ldb, bsp, int(b_t), M, N, K, _ptr(of), N, _ptr(ob), ld16,
                               2 if out_split else 1, _ptr(ws), ws.numel(), _stream()), "mi_gemm_bf16_mn")
    return res


def gemm(A: Mat, B: Mat, alpha: float = 1.0, gamma: float = 0.0, sub: Optional[torch.Tensor] = None,
         out_dtype=torch.float32, out_split: bool = False, a_t: bool = False, b_t: bool = False):
    """C = alpha * (A @ B.T - gamma * sub); A [M,K], B [N,K] bf16 (plain or hi/lo).  ``out_split``
    returns a SplitBF16.  ``a_t`` / ``b_t``: the operand is given as the row-major [K, M] / [K, N] matrix and is
    read in place (MN-major descriptors) — ``gemm(X, dT, a_t=True, b_t=True)`` is X^T dT without transposes."""
    _need_cuda(A, B, sub)
    if a_t or b_t:
        assert alpha == 1.0 and gamma == 0.0 and sub is None
        return _gemm_mn(A, B, a_t, b_t, out_dtype, out_split)
    At, lda, asp, K = _opnd(A)
    Bt, ldb, bsp, Kb = _opnd(B)
    assert K == Kb, "inner dimensions differ"
    M, N = At.shape[0], Bt.shape[0]
    of = ob = None
    ld16 = 0
    if out_split:
        res = new_split(M, N, At.device)
        ob, ld16 = res.data, res.data.stride(0)
    elif out_dtype == torch.bfloat16:
        res = torch.empty((M, N), dtype=torch.bfloat16, device=At.device)
        ob, ld16 = res, N
    else:
        res = torch.empty((M, N), dtype=torch.float32, device=At.device)
        of = res
    if sub is not None:
        sub = sub.contiguous()
    _check(_lib.load().mi_gemm_bf16(_ptr(At), lda, asp, _ptr(Bt), ldb, bsp, M, N, K, alpha, gamma, _ptr(sub),
                                    0 if sub is None else sub.stride(0), _ptr(of), N, _ptr(ob), ld16,
                                    2 if out_split else 1, _stream()), "mi_gemm_bf16")
    return res


def transpose(x: Mat):
    """x^T.  A plain [R,C] matrix gives a [C,R] view with an 8-element-aligned pitch; a hi/lo matrix
    gives the hi/lo pair of x^T (lo half next to the hi half along the new K axis)."""
    _need_cuda(x)
    lib = _lib.load()
    if isinstance(x, SplitBF16):
        R, Cc = x.shape
        dp_in = x.data.shape[1] // 2
        out = new_split(Cc, R, x.device)
        dp_out = out.data.shape[1] // 2
        ld_in, ld_out = x.data.stride(0), out.data.stride(0)
        _check(lib.mi_transpose_bf16(_ptr(x.data), ld_in, _ptr(out.data), ld_out, R, Cc, _stream()), "mi_transpose_bf16")
        _check(lib.mi_transpose_bf16(C.c_void_p(x.data.data_ptr() + 2 * dp_in), ld_in,
                                     C.c_void_p(out.data.data_ptr() + 2 * dp_out), ld_out, R, Cc, _stream()), "mi_transpose_bf16")
        return out
    assert x.dtype == torch.bfloat16 and x.dim() == 2
    x = x.contiguous()
    R, Cc = x.shape
    ld = _round_up(R, 8)
    out = torch.zeros((Cc, ld), dtype=torch.bfloat16, device=x.device)
    _check(lib.mi_transpose_bf16(_ptr(x), Cc, _ptr(out), ld, R, Cc, _stream()), "mi_transpose_bf16")
    return out[:, :R]


def score_stats(Q: Mat, K: Mat, sid_q: torch.Tensor, sid_k: torch.Tensor,
                q_offset: int = 0, scale: float = 1.0) -> Tuple[torch.Tensor, torch.Tensor]:
    """rows [Bq,4] = {lse_neg, n_neg, diag, lse_all} (fp32), scal [8] (fp64) — see mi_b200.h."""
    _need_cuda(Q, K, sid_q, sid_k)
    lib = _lib.load()
    Qt, ldq, qsp, D = _opnd(Q)
    Kt, ldk, ksp, Dk = _opnd(K)
    assert D == Dk
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    Bq, Bk = Qt.shape[0], Kt.shape[0]
    rows = torch.empty((Bq, 4), dtype=torch.float32, device=Qt.device)
    scal = torch.empty(8, dtype=torch.float64, device=Qt.device)
    nbytes = lib.mi_score_stats_workspace_bytes(Bq, Bk, D)
    ws = workspace(nbytes, Qt.device)
    _check(lib.mi_score_stats(_ptr(Qt), ldq, qsp, _ptr(Kt), ldk, ksp, _ptr(sid_q), _ptr(sid_k), q_offset, Bq, Bk, D,
                              scale, _ptr(rows), _ptr(scal), _ptr(ws), ws.numel(), _stream()), "mi_score_stats")
    return rows, scal


def score_stats_rc(Q: Mat, K: Mat, sid_q: torch.Tensor, sid_k: torch.Tensor,
                   q_offset: int = 0, scale: float = 1.0, event_k_ready: Optional["torch.cuda.Event"] = None,
                   k_local_valid: bool = False, include_pos: bool = False) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """mi_score_stats_rc_ex: rows / scal as score_stats, plus col_lse [Bk] (fp32) = log-sum-exp of every column over this row
    block's negatives, from the same score tiles (the symmetric estimator's statistics in the batch-sharded step).
    ``include_pos``: the block's positive pairs are folded into its own columns.  ``event_k_ready`` / ``k_local_valid``: as
    in score_single_pass (the own column block is scored before the wait for the other ranks' text rows)."""
    _need_cuda(Q, K, sid_q, sid_k)
    lib = _lib.load()
    Qt, ldq, qsp, D = _opnd(Q)
    Kt, ldk, ksp, Dk = _opnd(K)
    assert D == Dk
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    Bq, Bk = Qt.shape[0], Kt.shape[0]
    rows = torch.empty((Bq, 4), dtype=torch.float32, device=Qt.device)
    scal = torch.empty(8, dtype=torch.float64, device=Qt.device)
    col = torch.empty(Bk, dtype=torch.float32, device=Qt.device)
    nbytes = lib.mi_score_stats_rc_workspace_bytes(Bq, Bk, D)
    ws = workspace(nbytes, Qt.device)
    _check(lib.mi_score_stats_rc_ex(_ptr(Qt), ldq, qsp, _ptr(Kt), ldk, ksp, _ptr(sid_q), _ptr(sid_k), q_offset, Bq, Bk, D,
                                    scale, _ptr(rows), _ptr(scal), _ptr(col),
                                    None if event_k_ready is None else C.c_void_p(event_k_ready.cuda_event), int(k_local_valid),
                                    int(include_pos), _ptr(ws), ws.numel(), _stream()), "mi_score_stats_rc_ex")
    return rows, scal, col


def score_grad(Q: Mat, K: Mat, sid_q, sid_k, q_offset: int, scale: float,
               refq: Optional[torch.Tensor], wq: float, refk: Optional[torch.Tensor], wk: float,
               include_diag: bool, precision: str, alpha: float, gamma: float,
               want_f32: bool = True, want_bf16: bool = False, out_split: bool = False, want_k: bool = False,
               event_after_k: Optional["torch.cuda.Event"] = None):
    """Fused gradient pass (mi_score_grad).  Returns (Oq fp32 | None, Oq bf16 / SplitBF16 | None,
    Ok fp32 [Bk, D] | None):  Oq = alpha (G K - gamma K_diag),  Ok = alpha (G^T Q - gamma Q_diag).
    ``event_after_k`` (a recorded torch.cuda.Event) is re-recorded on the current stream as soon as Ok is
    complete, before the Oq contraction runs."""
    _need_cuda(Q, K, sid_q, sid_k, refq, refk)
    prec = _precision(precision)
    lib = _lib.load()
    Qt, ldq, qsp, D = _opnd(Q)
    Kt, ldk, ksp, Dk = _opnd(K)
    assert D == Dk
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    Bq, Bk = Qt.shape[0], Kt.shape[0]
    dev = Qt.device
    o32 = torch.empty((Bq, D), dtype=torch.float32, device=dev) if want_f32 else None
    o16 = ob = None
    ld16 = 0
    if want_bf16:
        if out_split:
            o16 = new_split(Bq, D, dev)
            ob, ld16 = o16.data, o16.data.stride(0)
        else:
            o16 = torch.empty((Bq, D), dtype=torch.bfloat16, device=dev)
            ob, ld16 = o16, D
    okk = torch.empty((Bk, D), dtype=torch.float32, device=dev) if want_k else None
    refq = None if refq is None else refq.float().contiguous()
    refk = None if refk is None else refk.float().contiguous()
    nbytes = lib.mi_score_grad_workspace_bytes(Bq, Bk, D, prec)
    ws = workspace(nbytes, dev)
    _check(lib.mi_score_grad(_ptr(Qt), ldq, qsp, _ptr(Kt), ldk, ksp, _ptr(sid_q), _ptr(sid_k), q_offset, Bq, Bk, D, scale,
                             _ptr(refq), wq, _ptr(refk), wk, int(include_diag), prec, alpha, gamma,
                             _ptr(o32), _ptr(ob), ld16, 2 if out_split else 1, _ptr(okk),
                             None if event_after_k is None else C.c_void_p(event_after_k.cuda_event),
                             _ptr(ws), ws.numel(), _stream()), "mi_score_grad")
    return o32, o16, okk


def row_norm_max(A: Mat) -> Tuple[torch.Tensor, torch.Tensor]:
    """(|A_i| per row, max_i |A_i| as a 1-element tensor)."""
    _need_cuda(A)
    At, lda, asp, D = _opnd(A)
    rows = At.shape[0]
    norms = torch.empty(rows, dtype=torch.float32, device=At.device)
    mx = torch.empty(1, dtype=torch.float32, device=At.device)
    _check(_lib.load().mi_row_norm_max(_ptr(At), lda, asp, rows, D, _ptr(norms), _ptr(mx), _stream()), "mi_row_norm_max")
    return norms, mx


def set_ref_sample_columns(n: int) -> None:
    """Columns sampled per row for the single pass's references (mi_set_ref_sample_columns; default 2048)."""
    _lib.load().mi_set_ref_sample_columns(int(n))


def score_ref_sample(Q: Mat, K: Mat, sid_q, sid_k, q_offset: int, scale: float, include_diag: bool,
                     col0: int = 0, n_cols: Optional[int] = None, stride: int = 0, subset: bool = False) -> dict:
    """mi_score_ref_sample: per-row softmax references of the single pass from a strided column sample
    (``stride`` = 1: every column of K; 0: the library's choice).  ``subset``: K holds only part of the row's columns (a
    rank's own block), so the references keep their safety margin even at stride 1.
    Returns {"ref" [Bq], "diag" [Bq], "lam" [1], "stride"}."""
    _need_cuda(Q, K, sid_q, sid_k)
    lib = _lib.load()
    Qt, ldq, qsp, D = _opnd(Q)
    Kt, ldk, ksp, Dk = _opnd(K)
    assert D == Dk
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    Bq, Bk = Qt.shape[0], Kt.shape[0]
    n_cols = Bk - col0 if n_cols is None else n_cols
    if stride < 1:
        stride = int(lib.mi_ref_sample_stride(Bq, n_cols, D))
    dev = Qt.device
    f32 = dict(dtype=torch.float32, device=dev)
    r = {"ref": torch.empty(Bq, **f32), "diag": torch.empty(Bq, **f32), "lam": torch.empty(1, **f32), "stride": stride}
    ws = workspace(lib.mi_score_ref_sample_workspace_bytes(Bq, n_cols, D, stride), dev)
    _check(lib.mi_score_ref_sample(_ptr(Qt), ldq, qsp, _ptr(Kt), ldk, ksp, _ptr(sid_q), _ptr(sid_k), q_offset, Bq, Bk, D,
                                   scale, int(include_diag), col0, n_cols, stride, int(subset), _ptr(r["ref"]), _ptr(r["diag"]), _ptr(r["lam"]),
                                   _ptr(ws), ws.numel(), _stream()), "mi_score_ref_sample")
    return r


def score_single_pass(Q: Mat, K: Mat, sid_q, sid_k, q_offset: int, scale: float, include_diag: bool, precision: str,
                      inv_bg: float, ref: torch.Tensor, lam: Optional[torch.Tensor], diag: torch.Tensor, want_k: bool = True,
                      event_after_k: Optional["torch.cuda.Event"] = None,
                      event_after_scal: Optional["torch.cuda.Event"] = None,
                      event_k_ready: Optional["torch.cuda.Event"] = None, k_local_valid: bool = False) -> dict:
    """mi_score_single_pass: statistics and raw gradient contractions from ONE score computation, relative to the
    per-row references ``ref`` (score_ref_sample) and the global constant ``lam`` (dv-like estimators)."""
    _need_cuda(Q, K, sid_q, sid_k, ref, lam, diag)
    prec = _precision(precision)
    lib = _lib.load()
    Qt, ldq, qsp, D = _opnd(Q)
    Kt, ldk, ksp, Dk = _opnd(K)
    assert D == Dk
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    Bq, Bk = Qt.shape[0], Kt.shape[0]
    dev = Qt.device
    f32 = dict(dtype=torch.float32, device=dev)
    r = {"rows": torch.empty((Bq, 4), **f32), "scal": torch.empty(8, dtype=torch.float64, device=dev),
         "oq_raw": torch.empty((Bq, D), **f32), "ok_raw": torch.empty((Bk, D), **f32) if want_k else None,
         "ref": ref, "wrow": torch.empty(Bq, **f32), "lam": lam,
         "flag": torch.empty(1, dtype=torch.int32, device=dev)}
    ws = workspace(lib.mi_score_single_pass_workspace_bytes(Bq, Bk, D, prec), dev)
    ev = lambda e: None if e is None else C.c_void_p(e.cuda_event)
    _check(lib.mi_score_single_pass(_ptr(Qt), ldq, qsp, _ptr(Kt), ldk, ksp, _ptr(sid_q), _ptr(sid_k), q_offset, Bq, Bk, D,
                                    scale, int(include_diag), prec, inv_bg, _ptr(ref), _ptr(lam), _ptr(diag),
                                    _ptr(r["rows"]), _ptr(r["scal"]), _ptr(r["oq_raw"]), _ptr(r["ok_raw"]), _ptr(r["wrow"]),
                                    _ptr(r["flag"]), ev(event_after_k), ev(event_after_scal), ev(event_k_ready),
                                    int(k_local_valid), _ptr(ws), ws.numel(), _stream()), "mi_score_single_pass")
    return r


def merge_scalars_loss(scal_all: torch.Tensor, estimator: str, b_global: int, lam: Optional[torch.Tensor] = None) -> dict:
    """Ranks' reduced scalars [world, 8] (fp64) -> the global loss terms as 0-d fp64 views plus the global
    log-sum-exp as a 1-element fp32 tensor (mi_merge_scalars: two tiny kernels, no host sync).  "guard" = the ranks'
    guard counts summed (+1 when e^{lam - lse} would leave the fp32 range): must be 0, else repeat with exact references."""
    _need_cuda(scal_all)
    scal_all = scal_all.contiguous()
    dev = scal_all.device
    out = torch.empty(8, dtype=torch.float64, device=dev)
    scratch = torch.empty(8, dtype=torch.float64, device=dev)
    lse32 = torch.empty(1, dtype=torch.float32, device=dev)
    _check(_lib.load().mi_merge_scalars(_ptr(scal_all), scal_all.shape[0], b_global, ESTIMATOR[estimator], _ptr(lam), _ptr(out),
                                        _ptr(lse32), _ptr(scratch), _stream()), "mi_merge_scalars")
    return {"loss": out[0], "pos_mean": out[1], "lse_neg": out[2], "n_neg": out[3], "loss_row": out[4],
            "rows_without_negatives": out[6], "guard": out[7], "lse32": lse32}


def merge_sym_stats(scal_all: torch.Tensor, col_all: torch.Tensor, b_global: int) -> dict:
    """mi_merge_sym_stats: the ranks' scalar rows [world, 8] (fp64) and column partials [world, >= b_global] (fp32, own
    positive pairs folded in: score_stats_rc(include_pos=True)) -> the symmetric loss terms as 0-d fp64 views (the layout of
    the single-GPU call) and "c" [b_global] fp32, the column log-sum-exps of the batch."""
    _need_cuda(scal_all, col_all)
    scal_all = scal_all.to(torch.float64).contiguous()
    if col_all.dtype != torch.float32 or col_all.stride(1) != 1:
        col_all = col_all.to(torch.float32).contiguous()
    dev = scal_all.device
    lib = _lib.load()
    out = torch.empty(8, dtype=torch.float64, device=dev)
    c = torch.empty(b_global, dtype=torch.float32, device=dev)
    scratch = torch.empty(int(lib.mi_merge_sym_stats_scratch_doubles(b_global)), dtype=torch.float64, device=dev)
    _check(lib.mi_merge_sym_stats(_ptr(scal_all), _ptr(col_all), col_all.stride(0), scal_all.shape[0], b_global, _ptr(out),
                                  _ptr(c), _ptr(scratch), _stream()), "mi_merge_sym_stats")
    return {"loss": out[0], "pos_mean": out[1], "lse_neg": out[2], "n_neg": out[3], "loss_row": out[4], "loss_col": out[5],
            "rows_without_negatives": out[6], "guard": out[7], "c": c}


def single_finalize_q(oq_raw, ref, wrow, lse, dv_like: bool, alpha: float, gamma: float, kdiag: Mat,
                      want_f32: bool = True, want_bf16: bool = False, out_split: bool = False):
    """Oq = alpha (c_q oq_raw - gamma Kdiag): fp32 and/or bf16 (hi/lo) result."""
    Kt, ldk, ksp, D = _opnd(kdiag)
    rows = oq_raw.shape[0]
    dev = oq_raw.device
    o32 = torch.empty((rows, D), dtype=torch.float32, device=dev) if want_f32 else None
    o16 = ob = None
    ld16 = 0
    if want_bf16:
        if out_split:
            o16 = new_split(rows, D, dev)
            ob, ld16 = o16.data, o16.data.stride(0)
        else:
            o16 = torch.empty((rows, D), dtype=torch.bfloat16, device=dev)
            ob, ld16 = o16, D
    _check(_lib.load().mi_single_finalize_q(_ptr(oq_raw), rows, D, _ptr(ref), _ptr(wrow), _ptr(lse), int(dv_like), alpha, gamma,
                                            _ptr(Kt), ldk, ksp, _ptr(o32), _ptr(ob), ld16, 2 if out_split else 1, _stream()),
           "mi_single_finalize_q")
    return o32, o16


def single_finalize_k(ok, lam, lse, dv_like: bool, alpha: float, gamma: float, qdiag: Mat) -> torch.Tensor:
    """Ok = alpha (kappa ok - gamma Qdiag), in place; rows of ok and qdiag correspond one to one."""
    Qt, ldq, qsp, D = _opnd(qdiag)
    _check(_lib.load().mi_single_finalize_k(_ptr(ok), ok.shape[0], D, _ptr(lam), _ptr(lse), int(dv_like), alpha, gamma,
                                            _ptr(Qt), ldq, qsp, _stream()), "mi_single_finalize_k")
    return ok


def critic_loss_fwd_bwd(X: torch.Tensor, Y: torch.Tensor, W: Optional[torch.Tensor], sid: torch.Tensor,
                        estimator: str = "dv", precision: str = "fast", inv_tau: float = 1.0,
                        need_grads: bool = True, out=None, two_pass: bool = False, workspace_buf: Optional[torch.Tensor] = None):
    """The whole path on one GPU (mi_critic_loss_fwd_bwd).  Returns (loss_out fp64[8], dX, dY, dW).
    ``out`` = (loss, dX, dY, dW) reuses caller-owned result buffers (no allocation in the call).
    dv / infonce / infonce_row take the single pass with sampled softmax references; if a row's reference leaves the
    numerically safe window the library itself repeats the step with exact references (device-side predicate, no host
    sync) — loss_out[7] counts the rows that tripped (informational).  ``two_pass`` asks for exact references from the
    start (MI_PREC_TWO_PASS).  ``workspace_buf``: caller-owned scratch of ``critic_workspace_bytes`` (CUDA graphs)."""
    _need_cuda(X, Y, W, sid)
    prec = _precision(precision) | (2 if two_pass else 0)
    lib = _lib.load()
    X, Y = as_bf16(X), as_bf16(Y)
    W = None if W is None else as_bf16(W)
    sid = sid.to(torch.int32).contiguous()
    B, D = X.shape
    critic = 1 if W is not None else 0
    est = ESTIMATOR[estimator]
    dX = dY = dW = None
    if out is not None:
        loss, dX, dY, dW = out
    else:
        loss = torch.empty(8, dtype=torch.float64, device=X.device)
    if need_grads and out is None:
        dX = torch.empty((B, D), dtype=torch.float32, device=X.device)
        dY = torch.empty((B, D), dtype=torch.float32, device=X.device)
        if W is not None:
            dW = torch.empty((D, D), dtype=torch.float32, device=X.device)
    nbytes = lib.mi_critic_workspace_bytes(B, D, critic, est, prec, int(need_grads))
    ws = workspace(nbytes, X.device) if workspace_buf is None else workspace_buf
    if ws.numel() < nbytes:
        raise MIError(f"workspace_buf too small: {ws.numel()} < {nbytes} bytes")
    _check(lib.mi_critic_loss_fwd_bwd(_ptr(X), _ptr(Y), _ptr(W), _ptr(sid), B, D, critic, est, prec, inv_tau,
                                      _ptr(loss), _ptr(dX), _ptr(dY), _ptr(dW), _ptr(ws), ws.numel(), _stream()),
           "mi_critic_loss_fwd_bwd")
    return loss, dX, dY, dW


GUARD_TRIPPED = 1
_dist_ctx = {}


def dist_context(group=None):
    """The library-side context of the batch-sharded step (mi_dist_ctx) for a torch.distributed NCCL process group: it
    borrows the group's own ncclComm_t (ProcessGroupNCCL._comm_ptr()) — no second communicator.  Cached per group."""
    import torch.distributed as tdist
    pg = tdist.distributed_c10d._get_default_group() if group is None else group
    backend = pg._get_backend(torch.device("cuda", torch.cuda.current_device()))
    key = id(backend)
    if key not in _dist_ctx:
        try:
            comm = backend._comm_ptr()
        except Exception:                                     # communicator not created yet (lazy init): one collective forces it
            tdist.all_reduce(torch.zeros(1, device=f"cuda:{torch.cuda.current_device()}"), group=group)
            comm = backend._comm_ptr()
        ctx = C.c_void_p()
        _check(_lib.load().mi_dist_ctx_create(C.c_void_p(comm), C.byref(ctx)), "mi_dist_ctx_create")
        rank, world = C.c_int(), C.c_int()
        _check(_lib.load().mi_dist_ctx_info(ctx, C.byref(rank), C.byref(world)), "mi_dist_ctx_info")
        _dist_ctx[key] = (ctx, rank.value, world.value, backend)      # (keeps the backend alive as long as the context)
    return _dist_ctx[key]


def sharded_step(X_local: torch.Tensor, Y_local: torch.Tensor, W: Optional[torch.Tensor], sid_local: torch.Tensor,
                 estimator: str, precision: str, inv_tau: float, group=None, check_guard: bool = True):
    """mi_sharded_critic_loss_fwd_bwd: the whole batch-sharded step (collectives included) as one library call, for every
    estimator.  Returns (status, loss_out fp64[8], dX, dY, dW); status GUARD_TRIPPED (on every rank alike) means the outputs
    are not valid and the step must be repeated on the exact path ("infonce_sym" uses exact statistics: always 0)."""
    reject_separable_only(estimator, "the batch-sharded step")
    _need_cuda(X_local, Y_local, W, sid_local)
    prec = _precision(precision)
    lib = _lib.load()
    ctx, rank, world, _ = dist_context(group)
    if "MI_RS_RESERVE_SMS" in os.environ:       # (experiment knob) SMs the dT contraction leaves to the overlapped reduce-scatter
        lib.mi_set_overlap_reserve_sms(int(os.environ["MI_RS_RESERVE_SMS"]))
    X, Y = as_bf16(X_local), as_bf16(Y_local)
    Wb = None if W is None else as_bf16(W)
    if sid_local.dtype != torch.int32:
        raise MIError("sharded_step needs exact int32 study ids (equal ids <=> equal values on every rank)")
    sid = sid_local.contiguous()
    Bl, D = X.shape
    critic = 1 if Wb is not None else 0
    est = ESTIMATOR[estimator]
    dev = X.device
    loss = torch.empty(8, dtype=torch.float64, device=dev)
    dX = torch.empty((Bl, D), dtype=torch.float32, device=dev)
    dY = torch.empty((Bl, D), dtype=torch.float32, device=dev)
    dW = torch.empty((D, D), dtype=torch.float32, device=dev) if Wb is not None else None
    nbytes = lib.mi_sharded_critic_workspace_bytes(Bl, world, D, critic, est, prec)
    if nbytes == 0:
        raise MIError("mi_sharded_critic_workspace_bytes: unsupported configuration")
    ws = workspace(nbytes, dev)
    st = lib.mi_sharded_critic_loss_fwd_bwd(ctx, _ptr(X), _ptr(Y), _ptr(Wb), _ptr(sid), Bl, D, critic, est, prec, inv_tau,
                                            _ptr(loss), _ptr(dX), _ptr(dY), _ptr(dW), _ptr(ws), ws.numel(), int(check_guard), _stream())
    if st not in (0, GUARD_TRIPPED):
        _check(st, "mi_sharded_critic_loss_fwd_bwd")
    return st, loss, dX, dY, dW


class GraphedCriticStep:
    """CUDA-graph replay of ``critic_loss_fwd_bwd`` for one fixed shape.  Below B ~ 8192 the fused step is launch-bound
    (~45 kernels of a few microseconds each); capturing the library's launch sequence once and replaying it removes
    the per-launch host cost.  Inputs are copied into static buffers, results are returned in static buffers."""

    def __init__(self, B: int, D: int, bilinear: bool = True, estimator: str = "dv", precision: str = "fast",
                 inv_tau: float = 1.0, device=None):
        prec = _precision(precision)
        dev = torch.device("cuda" if device is None else device)
        self.args = (estimator, precision, inv_tau)
        self.X = torch.zeros((B, D), dtype=torch.bfloat16, device=dev)
        self.Y = torch.zeros((B, D), dtype=torch.bfloat16, device=dev)
        self.W = torch.zeros((D, D), dtype=torch.bfloat16, device=dev) if bilinear else None
        self.sid = torch.arange(B, dtype=torch.int32, device=dev)
        self.out = (torch.empty(8, dtype=torch.float64, device=dev), torch.empty((B, D), device=dev),
                    torch.empty((B, D), device=dev), torch.empty((D, D), device=dev) if bilinear else None)
        # the captured graph bakes the scratch pointer in: a PRIVATE workspace that lives as long as the graph does
        nbytes = _lib.load().mi_critic_workspace_bytes(B, D, 1 if bilinear else 0, ESTIMATOR[estimator], prec, 1)
        self.ws = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
        self.graph = None

    def _run(self):
        est, prec, inv_tau = self.args
        critic_loss_fwd_bwd(self.X, self.Y, self.W, self.sid, est, prec, inv_tau, True, out=self.out, workspace_buf=self.ws)

    def __call__(self, X, Y, W, sid):
        """Returns (loss_out fp64[8], dX, dY, dW) — static buffers, overwritten by the next call."""
        self.X.copy_(X); self.Y.copy_(Y); self.sid.copy_(sid)
        if self.W is not None:
            self.W.copy_(W)
        if self.graph is None:
            side = torch.cuda.Stream(device=self.X.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):               # warm-up outside the capture: workspace growth, kernel attributes
                self._run(); self._run()
            torch.cuda.current_stream().wait_stream(side)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self._run()
        self.graph.replay()
        return self.out


MLP_PARAMS = ("W1", "b1", "W2", "b2", "W3", "b3")


def mlp_critic_loss_fwd_bwd(X: torch.Tensor, Y: torch.Tensor, params, sid: torch.Tensor, estimator: str = "dv",
                            precision: str = "fast", need_grads: bool = True, want_scores: bool = False):
    """The reference's own critic make_mlp(2D, [H1, H2]) (model.py:18-32) on every pair + estimator, fwd+bwd
    (mi_mlp_critic_loss_fwd_bwd).  ``params`` = (W1 [H1,2D], b1, W2 [H2,H1], b2, W3 [1,H2], b3) fp32.
    Returns (loss_out fp64[8], S or None, grads dict with keys dX, dY, dW1 ... db3 (or None)); loss_out[4] / [5] are the
    row / column losses of infonce_sym."""
    reject_separable_only(estimator, "the MLP critic")
    _need_cuda(X, Y, sid, *params)
    prec = _mlp_precision(precision)
    lib = _lib.load()
    f32 = lambda t: t.detach().to(torch.float32).contiguous()
    X, Y = f32(X), f32(Y)
    W1, b1, W2, b2, W3, b3 = (f32(t) for t in params)
    B, D = X.shape
    H1, H2 = W1.shape[0], W2.shape[0]
    if W1.shape != (H1, 2 * D) or W2.shape != (H2, H1) or W3.numel() != H2 or b1.numel() != H1 or b2.numel() != H2 or b3.numel() != 1:
        raise MIError("MLP critic parameters do not have the make_mlp(2D, [H1, H2]) shapes")
    est = _mlp_estimator(estimator)
    sid = sid.to(torch.int32).contiguous()
    dev = X.device
    loss = torch.empty(8, dtype=torch.float64, device=dev)
    S = torch.empty((B, B), dtype=torch.float32, device=dev) if want_scores else None
    grads = None
    if need_grads:
        shapes = {"dX": (B, D), "dY": (B, D), "dW1": (H1, 2 * D), "db1": (H1,), "dW2": (H2, H1), "db2": (H2,),
                  "dW3": (1, H2), "db3": (1,)}
        grads = {k: torch.empty(v, dtype=torch.float32, device=dev) for k, v in shapes.items()}
    g = grads or {}
    nbytes = lib.mi_mlp_critic_workspace_bytes(B, D, H1, H2, prec)
    if nbytes == 0:
        raise MIError("mi_mlp_critic_workspace_bytes: unsupported shape (D, H1, H2 multiples of 8, H2 <= 512; fp32: D, H1 <= 1280)")
    ws = workspace(nbytes, dev)
    _check(lib.mi_mlp_critic_loss_fwd_bwd(_ptr(X), _ptr(Y), _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), _ptr(W3), _ptr(b3), _ptr(sid),
                                          B, D, H1, H2, est, prec, _ptr(loss), _ptr(S),
                                          _ptr(g.get("dX")), _ptr(g.get("dY")), _ptr(g.get("dW1")), _ptr(g.get("db1")),
                                          _ptr(g.get("dW2")), _ptr(g.get("db2")), _ptr(g.get("dW3")), _ptr(g.get("db3")),
                                          _ptr(ws), ws.numel(), _stream()), "mi_mlp_critic_loss_fwd_bwd")
    return loss, S, grads


def set_mlp_mode(mode: int) -> None:
    """mi_set_mlp_mode: bit 0 = single pass for dv / infonce, bit 1 = dZ1 reductions fused into their GEMM (default 3;
    0 = the two-pass sequence; negative = default)."""
    _lib.load().mi_set_mlp_mode(int(mode))


def get_mlp_mode() -> int:
    return int(_lib.load().mi_get_mlp_mode())


# ---- the MLP critic over a row block: stage ops of the batch-sharded step (mi_b200.dist.sharded_mlp_critic_loss_fwd_bwd)

def _mlp_operands(X, Y, params):
    _need_cuda(X, Y, *params)
    f32 = lambda t: t.detach().to(torch.float32).contiguous()
    X, Y = f32(X), f32(Y)
    W1, b1, W2, b2, W3, b3 = (f32(t) for t in params)
    D = X.shape[1]
    H1, H2 = W1.shape[0], W2.shape[0]
    if (Y.shape[1] != D or W1.shape != (H1, 2 * D) or W2.shape != (H2, H1) or W3.numel() != H2 or b1.numel() != H1
            or b2.numel() != H2 or b3.numel() != 1):
        raise MIError("MLP critic parameters do not have the make_mlp(2D, [H1, H2]) shapes")
    return X, Y, (W1, b1, W2, b2, W3, b3), D, H1, H2


def _mlp_block_workspace(Bq, Bk, D, H1, H2, prec, dev):
    nbytes = _lib.load().mi_mlp_block_workspace_bytes(Bq, Bk, D, H1, H2, prec)
    if nbytes == 0:
        raise MIError("mi_mlp_block_workspace_bytes: unsupported shape (D, H1, H2 multiples of 8, H2 <= 512; fp32: D, H1 <= 1280)")
    return workspace(nbytes, dev)


def reject_separable_only(estimator: str, what: str) -> None:
    """Raise before any launch when ``estimator`` runs only on the single-GPU separable critics."""
    if estimator in SEPARABLE_ONLY:
        supported = ", ".join(e for e in ESTIMATOR if e not in SEPARABLE_ONLY)
        raise MIError(f"estimator {estimator!r} is not implemented for {what}: supported are {supported} "
                      f"({' and '.join(SEPARABLE_ONLY)} run on the single-GPU dot / bilinear critics)")


def _precision(precision: str) -> int:
    """The code of a precision of the separable critics / GDV ("fast", "strict"); "fp32" is the MLP critic's only."""
    if precision not in PRECISION:
        extra = " (\"fp32\" is implemented for the MLP critic only)" if precision in MLP_PRECISION else ""
        raise MIError(f"unknown precision {precision!r}: supported are {', '.join(PRECISION)}{extra}")
    return PRECISION[precision]


def _mlp_precision(precision: str) -> int:
    if precision not in MLP_PRECISION:
        raise MIError(f"unknown precision {precision!r}: the MLP critic supports {', '.join(MLP_PRECISION)}")
    return MLP_PRECISION[precision]


def _mlp_estimator(estimator):
    reject_separable_only(estimator, "the MLP critic")
    if estimator not in ESTIMATOR:
        raise MIError(f"unknown estimator {estimator!r}: the MLP critic supports "
                      f"{', '.join(e for e in ESTIMATOR if e not in SEPARABLE_ONLY)}")
    return ESTIMATOR[estimator]


def mlp_block_ref_logit(X: torch.Tensor, Y: torch.Tensor, params, q_offset: int, precision: str = "fast") -> torch.Tensor:
    """Maximum logit of a sample of the block's own pairs (image rows X against the text rows of Y at q_offset ..)
    (mi_mlp_block_ref_logit) -> fp32 [1]."""
    X, Y, prm, D, H1, H2 = _mlp_operands(X, Y, params)
    Bq, Bk, prec = X.shape[0], Y.shape[0], _mlp_precision(precision)
    ref = torch.empty(1, dtype=torch.float32, device=X.device)
    ws = _mlp_block_workspace(Bq, Bk, D, H1, H2, prec, X.device)
    _check(_lib.load().mi_mlp_block_ref_logit(*(_ptr(t) for t in (X, Y) + prm), Bq, Bk, q_offset, D, H1, H2, prec, _ptr(ref),
                                              _ptr(ws), ws.numel(), _stream()), "mi_mlp_block_ref_logit")
    return ref


def mlp_block_fwd(X: torch.Tensor, Y: torch.Tensor, params, sid_q: torch.Tensor, sid_k: torch.Tensor, q_offset: int,
                  estimator: str, precision: str, ref: Optional[torch.Tensor], two_pass: bool):
    """The block's pass over its Bq x Bk pairs (mi_mlp_block_fwd_rc) -> (scalar row fp64 [8], state), and for infonce_sym
    (``two_pass`` only) a third item: the block's column partials fp32 [Bk], the log-sum-exp of every column over the
    block's negatives and its positive pair.  ``state`` is an opaque device buffer that carries the block to
    ``mlp_block_bwd``."""
    X, Y, prm, D, H1, H2 = _mlp_operands(X, Y, params)
    _need_cuda(sid_q, sid_k, ref)
    Bq, Bk, est, prec = X.shape[0], Y.shape[0], _mlp_estimator(estimator), _mlp_precision(precision)
    lib = _lib.load()
    dev = X.device
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    ws = _mlp_block_workspace(Bq, Bk, D, H1, H2, prec, dev)
    state = torch.empty(lib.mi_mlp_block_state_bytes(Bq, Bk, D, H1, H2, prec), dtype=torch.uint8, device=dev)
    scal = torch.empty(8, dtype=torch.float64, device=dev)
    sym = estimator == "infonce_sym"
    col = torch.empty(Bk, dtype=torch.float32, device=dev) if sym else None
    _check(lib.mi_mlp_block_fwd_rc(*(_ptr(t) for t in (X, Y) + prm), _ptr(sid_q), _ptr(sid_k), Bq, Bk, q_offset, D, H1, H2, est,
                                   prec, _ptr(ref), int(two_pass), _ptr(scal), _ptr(col), _ptr(state), state.numel(), _ptr(ws),
                                   ws.numel(), _stream()), "mi_mlp_block_fwd_rc")
    return (scal, state, col) if sym else (scal, state)


def mlp_block_merge(scal_all: torch.Tensor, b_global: int, estimator: str, two_pass: bool):
    """Blocks' scalar rows [world, 8] -> (loss_out fp64 [8] of the batch, merged row fp64 [8]) (mi_mlp_block_merge)."""
    _need_cuda(scal_all)
    scal_all = scal_all.contiguous()
    loss = torch.empty(8, dtype=torch.float64, device=scal_all.device)
    merged = torch.empty(8, dtype=torch.float64, device=scal_all.device)
    _check(_lib.load().mi_mlp_block_merge(_ptr(scal_all), scal_all.shape[0], b_global, _mlp_estimator(estimator), int(two_pass),
                                          _ptr(loss), _ptr(merged), _stream()), "mi_mlp_block_merge")
    return loss, merged


def mlp_block_bwd(X: torch.Tensor, Y: torch.Tensor, params, sid_q: torch.Tensor, sid_k: torch.Tensor, q_offset: int,
                  estimator: str, precision: str, two_pass: bool, loss: torch.Tensor, merged: torch.Tensor, state: torch.Tensor,
                  col_lse: Optional[torch.Tensor] = None) -> dict:
    """The block's backward once the loss of the batch is known (mi_mlp_block_bwd_rc; ``col_lse`` fp32 [Bk]: for
    infonce_sym, the log-sum-exp of every column over the whole batch).  Returns dX of the block's rows, dC_part [Bk, H1]
    (the block's contribution to dL/dC of every text row), dW1 (image half filled), db1, dW2, db2, dW3, db3 (the block's
    shares)."""
    X, Y, prm, D, H1, H2 = _mlp_operands(X, Y, params)
    _need_cuda(sid_q, sid_k, loss, merged, state, col_lse)
    if col_lse is not None:
        col_lse = col_lse.detach().to(torch.float32).contiguous()
    Bq, Bk, est, prec = X.shape[0], Y.shape[0], _mlp_estimator(estimator), _mlp_precision(precision)
    dev = X.device
    sid_q, sid_k = sid_q.to(torch.int32).contiguous(), sid_k.to(torch.int32).contiguous()
    shapes = {"dX": (Bq, D), "dC_part": (Bk, H1), "dW1": (H1, 2 * D), "db1": (H1,), "dW2": (H2, H1), "db2": (H2,),
              "dW3": (1, H2), "db3": (1,)}
    g = {k: torch.empty(v, dtype=torch.float32, device=dev) for k, v in shapes.items()}
    ws = _mlp_block_workspace(Bq, Bk, D, H1, H2, prec, dev)
    _check(_lib.load().mi_mlp_block_bwd_rc(*(_ptr(t) for t in (X, Y) + prm), _ptr(sid_q), _ptr(sid_k), Bq, Bk, q_offset, D, H1,
                                           H2, est, prec, int(two_pass), _ptr(loss), _ptr(merged), _ptr(col_lse), _ptr(state),
                                           state.numel(), *(_ptr(g[k]) for k in shapes), _ptr(ws), ws.numel(), _stream()),
           "mi_mlp_block_bwd_rc")
    return g


def mlp_input_grad(dZ: torch.Tensor, In: torch.Tensor, W1: torch.Tensor, side: int, precision: str = "fast",
                   dW1: Optional[torch.Tensor] = None, want_db1: bool = False):
    """Layer-1 backward of one side (mi_mlp_input_grad): dIn = dZ W1side; the side's half of dW1 [H1, 2D] is written
    into ``dW1`` (allocated when None); db1 = column sums of dZ when asked.  Returns (dIn, dW1, db1 or None)."""
    _need_cuda(dZ, In, W1, dW1)
    dZ, In, W1 = (t.detach().to(torch.float32).contiguous() for t in (dZ, In, W1))
    R, D = In.shape
    H1 = W1.shape[0]
    if dZ.shape != (R, H1) or W1.shape != (H1, 2 * D):
        raise MIError("mlp_input_grad: dZ [R, H1], In [R, D], W1 [H1, 2D] expected")
    if dW1 is None:
        dW1 = torch.zeros((H1, 2 * D), dtype=torch.float32, device=In.device)
    elif dW1.shape != (H1, 2 * D) or dW1.dtype != torch.float32 or not dW1.is_contiguous():
        raise MIError("mlp_input_grad: dW1 must be a contiguous fp32 [H1, 2D] tensor")
    dIn = torch.empty((R, D), dtype=torch.float32, device=In.device)
    db1 = torch.empty(H1, dtype=torch.float32, device=In.device) if want_db1 else None
    prec = _mlp_precision(precision)
    nbytes = _lib.load().mi_mlp_input_grad_workspace_bytes(R, D, H1, prec)
    if nbytes == 0:
        raise MIError("mi_mlp_input_grad_workspace_bytes: unsupported shape (D, H1 multiples of 8; fp32: D, H1 <= 1280)")
    ws = workspace(nbytes, In.device)
    _check(_lib.load().mi_mlp_input_grad(_ptr(dZ), _ptr(In), _ptr(W1), int(side), R, D, H1, prec, _ptr(dIn), _ptr(dW1), _ptr(db1),
                                         _ptr(ws), ws.numel(), _stream()), "mi_mlp_input_grad")
    return dIn, dW1, db1


def gdv(pos: torch.Tensor, neg: torch.Tensor, precision: str = "strict") -> torch.Tensor:
    """mi_gdv: fp64[4] = {gdv, intra_pos, intra_neg, inter} of two [N, D] fp32 embedding sets (validate.py:16-49)."""
    _need_cuda(pos, neg)
    prec = _precision(precision)
    pos, neg = pos.detach().to(torch.float32).contiguous(), neg.detach().to(torch.float32).contiguous()
    if pos.dim() != 2 or neg.dim() != 2 or pos.shape[1] != neg.shape[1]:
        raise MIError("gdv needs two [N, D] matrices with the same D")
    lib = _lib.load()
    Np, Nn, D = pos.shape[0], neg.shape[0], pos.shape[1]
    nbytes = lib.mi_gdv_workspace_bytes(Np, Nn, D, prec)
    if nbytes == 0:
        raise MIError("mi_gdv: unsupported shape (D multiple of 8, at least 2 samples per class)")
    ws = workspace(nbytes, pos.device)
    out = torch.empty(4, dtype=torch.float64, device=pos.device)
    _check(lib.mi_gdv(_ptr(pos), _ptr(neg), Np, Nn, D, prec, _ptr(out), _ptr(ws), ws.numel(), _stream()), "mi_gdv")
    return out


def set_overlap_reserve_sms(n: int) -> None:
    """SMs the engine leaves free after the dY contributions are complete (mi_set_overlap_reserve_sms)."""
    _lib.load().mi_set_overlap_reserve_sms(int(n))


def launch_count() -> int:
    return int(_lib.load().mi_launch_count())
