"""Batch-sharded MI critic / estimator over torch.distributed (one process per GPU, NCCL on NVLink).

The reference has no distributed code at all (SURVEY.md 2a); this is the data-parallel form of its
hot path (main_utils.py:220-226).  Rank r owns rows [r*Bl, (r+1)*Bl) of the image and text
embeddings.  Rows of the score matrix are independent given all text embeddings and columns are
independent given all projected image embeddings, so the path needs exactly one exchange step:

  1. T_r = X_r W locally (W replicated);  all-gather Y and the study ids (and T for the symmetric
     estimator's column statistics)                                                       (NCCL)
  2. row statistics of S[r,:] = T_r Y^T and (symmetric InfoNCE) column statistics of S[:,r]
     with the fused stats kernel — complete per rank, no B x B collective
  3. all-gather of 8 fp64 scalars per rank (DV: one (max, sum-exp) pair, N_neg, diagonal sum) and,
     for the symmetric form, of the per-column log-sum-exp vector (B floats)
  4. ONE gradient pass per rank over its row block: dT_r (complete) and the rank's contribution to
     every dY_j from the same score recompute; reduce-scatter of the [B, D] fp32 contributions
  5. dX_r = dT_r W^T locally; dW = sum_r X_r^T dT_r via all-reduce (DDP-style)

``backend`` is the stage-op provider: ``mi_b200.ops`` (CUDA, the only product backend); the CPU
gloo tests inject an emulation to exercise the sharding / collective logic without a GPU.
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.distributed as dist


def _world(group):
    if not dist.is_available() or not dist.is_initialized():
        return 1, 0
    return dist.get_world_size(group), dist.get_rank(group)


def _all_gather_rows(x: torch.Tensor, world: int, group) -> torch.Tensor:
    if world == 1:
        return x
    out = torch.empty((world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous(), group=group)
    return out


def merge_scalars(scal_all: torch.Tensor) -> dict:
    """scal_all [world, 8] fp64 rows {m, sum exp(lse-m), n_neg, diag_sum, rowloss_sum, rows_wo_neg, guard rows, 0}
    -> global quantities (pure tensor math, no host sync)."""
    m = scal_all[:, 0]
    gm = torch.max(m)
    w = torch.where(torch.isfinite(m), torch.exp(m - gm), torch.zeros_like(m))
    s = (scal_all[:, 1] * w).sum()
    return {
        "lse_neg": gm + torch.log(s),
        "n_neg": scal_all[:, 2].sum(),
        "diag_sum": scal_all[:, 3].sum(),
        "rowloss_sum": scal_all[:, 4].sum(),
        "rows_without_negatives": scal_all[:, 5].sum(),
        "guard": scal_all[:, 6].sum(),
    }


def dense_labels(sid_raw: torch.Tensor) -> torch.Tensor:
    """Exact int64 -> dense int32 relabelling (equal ids <=> equal labels) with static shapes only:
    sort + run boundaries + cumsum + scatter.  Unlike torch.unique it never synchronises with the host."""
    srt, idx = torch.sort(sid_raw)
    new = torch.ones_like(srt, dtype=torch.int32)
    new[1:] = (srt[1:] != srt[:-1]).to(torch.int32)
    lab_sorted = torch.cumsum(new, 0, dtype=torch.int32) - 1
    out = torch.empty_like(lab_sorted)
    out[idx] = lab_sorted
    return out


_side_streams = {}


def _side_stream(device):
    key = torch.device(device).index
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=device)
    return _side_streams[key]


def _gather_mat(m, world, group):
    """all-gather rows of a plain tensor or of a hi/lo pair (ops.SplitBF16)."""
    if hasattr(m, "data") and hasattr(m, "width") and not torch.is_tensor(m):
        return type(m)(_all_gather_rows(m.data, world, group), m.width)
    return _all_gather_rows(m, world, group)


def _loss_from(out, estimator):
    if estimator == "dv":
        # mi_critics.py:10 rounds N_neg to fp32 before the log; same formula as the fused C path
        log_n = torch.log(out["n_neg"].to(torch.float32).to(torch.float64))
        return out["lse_neg"] - log_n - out["pos_mean"]
    if estimator in ("infonce", "infonce_ref"):
        return out["lse_neg"] - out["pos_mean"]
    if estimator == "infonce_row":
        return out["loss_row"]
    raise ValueError(f"unknown estimator {estimator!r}")


def _reduce_scatter_rows(part, Bl, off, world, group, nccl, ev):
    """Sum the [Bg, D] per-rank contributions and keep this rank's rows.  With NCCL the collective starts on a
    side stream as soon as `ev` fires and runs under the work still queued on the compute stream."""
    if world == 1:
        return part, None
    if not nccl:                                      # gloo (CPU tests) has no reduce-scatter
        dist.all_reduce(part, op=dist.ReduceOp.SUM, group=group)
        return part[off:off + Bl].contiguous(), None
    side = _side_stream(part.device)
    side.wait_event(ev)
    if os.environ.get("MI_DY_EXCHANGE", "rs") == "a2a":
        # all-to-all of the per-destination slabs (plain NVLink copies) + a local sum, instead of a ring reduce-scatter
        recv = torch.empty_like(part)
        with torch.cuda.stream(side):
            work = dist.all_to_all_single(recv, part, group=group, async_op=True)
        return _A2ASum(recv.view(world, Bl, part.shape[1])), work
    out = torch.empty((Bl, part.shape[1]), dtype=part.dtype, device=part.device)
    with torch.cuda.stream(side):
        work = dist.reduce_scatter_tensor(out, part, op=dist.ReduceOp.SUM, group=group, async_op=True)
    return out, work


class _A2ASum:
    """The received slabs [world, Bl, D]; summed after the collective has completed."""

    def __init__(self, slabs):
        self.slabs = slabs

    def resolve(self):
        return self.slabs.sum(0)


_guard_host = {}


def _guard_buffer(device):
    key = torch.device(device).index
    if key not in _guard_host:
        _guard_host[key] = torch.zeros(1, dtype=torch.float64).pin_memory()
    return _guard_host[key]


class GuardTripped(Exception):
    """Internal: the sampled references of the single pass left the safe window on some rank (same verdict on all)."""


def _single_pass_step(backend, T_local, Xb, Yb, Wb, Y_all, sid_loc, sid_all, off, Bl, Bg, D, inv_tau, estimator,
                      precision, smp, lam, world, group, nccl, ev_y=None, own_first=False, check_guard=True):
    """dv / infonce / row InfoNCE with ONE score computation per rank (see mi_score_single_pass).  ``smp`` = this rank's
    reference sample (ref, diag), ``lam`` = the global constant (max over ranks of the largest reference)."""
    bilinear = Wb is not None
    strict = precision == "strict"
    dv_like = estimator != "infonce_row"
    gamma = 1.0 / Bg
    ev = ev_s = None
    if nccl:
        ev, ev_s = torch.cuda.Event(), torch.cuda.Event()
        ev.record(); ev_s.record()                    # (creates the CUDA events; the library re-records them in the pass)
    sp = backend.score_single_pass(T_local, Y_all, sid_loc, sid_all, off, inv_tau, not dv_like, precision, gamma,
                                   smp["ref"], lam, smp["diag"], want_k=True, event_after_k=ev,
                                   **({"event_after_scal": ev_s, "event_k_ready": ev_y, "k_local_valid": own_first} if nccl else {}))
    scal = sp["scal"].reshape(1, 8)
    if nccl:
        # the loss scalars (and the guard counts, scal[6]) are final BEFORE the panel's two contractions: exchange and merge
        # them on the side stream under the GEMMs.  The host reads the merged guard there — it waits for the score tiles,
        # not for the step — and only then enqueues the reduce-scatter and the rest (or abandons the step for the exact path).
        side = _side_stream(scal.device)
        scal_all = torch.empty((world, 8), dtype=scal.dtype, device=scal.device)
        side.wait_event(ev_s)
        ev_m = torch.cuda.Event()
        with torch.cuda.stream(side):
            dist.all_gather_into_tensor(scal_all, scal, group=group)
            out = backend.merge_scalars_loss(scal_all, estimator, Bg, lam if dv_like else None)
            if check_guard:
                gh = _guard_buffer(scal.device)
                gh.copy_(out["guard"].reshape(1), non_blocking=True)
            ev_m.record(side)
        # (no record_stream on the large buffers of this module: the compute stream waits for every side-stream / NCCL
        #  consumer of them before the call returns, so handing them back to the caching allocator is stream ordered — and
        #  the allocator reuses the same blocks step after step instead of growing)
        for t in list(out.values()):          # a few scalars allocated under the side stream's context and consumed on the
            t.record_stream(torch.cuda.current_stream())      # compute stream, which outlives the side stream's use
        if check_guard:
            ev_m.synchronize()
            if float(gh[0]) != 0.0:
                raise GuardTripped()
        dY, rs_work = _reduce_scatter_rows(sp["ok_raw"], Bl, off, world, group, nccl, ev)
        torch.cuda.current_stream().wait_event(ev_m)
        lse32 = out.pop("lse32")
    else:
        dY, rs_work = _reduce_scatter_rows(sp["ok_raw"], Bl, off, world, group, nccl, ev)
        scal_all = _all_gather_rows(scal, world, group)
        if hasattr(backend, "merge_scalars_loss"):        # two tiny kernels instead of ~25 framework ops
            out = backend.merge_scalars_loss(scal_all, estimator, Bg, lam if dv_like else None)
            lse32 = out.pop("lse32")
        else:
            g = merge_scalars(scal_all)
            out = {"pos_mean": g["diag_sum"] / Bg, "lse_neg": g["lse_neg"], "n_neg": g["n_neg"], "loss_row": g["rowloss_sum"] / Bg,
                   "guard": g["guard"]}
            out["loss"] = _loss_from(out, estimator)
            lse32 = out["lse_neg"].to(torch.float32).reshape(1)
            if dv_like:
                out["guard"] = out["guard"] + ((lam.double().reshape(()) - out["lse_neg"]).abs() > 60.0).double()
        if check_guard and float(out["guard"]) != 0.0:
            raise GuardTripped()
    dT32, dT16 = backend.single_finalize_q(sp["oq_raw"], smp["ref"], sp["wrow"], lse32, dv_like, inv_tau, gamma, Yb,
                                           want_f32=not bilinear, want_bf16=bilinear, out_split=bilinear and strict)
    dX, dW, dw_work = dT32, None, None
    if bilinear:
        dW = backend.gemm(Xb, dT16, a_t=True, b_t=True)          # X^T dT, both operands read in place
        if world > 1:                                             # runs under the dX GEMM and the dY finalisation below
            dw_work = dist.all_reduce(dW, op=dist.ReduceOp.SUM, group=group, async_op=True)
        dX = backend.gemm(dT16, Wb)
    if rs_work is not None:
        rs_work.wait()
    if isinstance(dY, _A2ASum):
        dY = dY.resolve()
    backend.single_finalize_k(dY, lam, lse32, dv_like, inv_tau, gamma, T_local)
    if dw_work is not None:
        dw_work.wait()
    return out, dX, dY, dW


def sharded_critic_loss_fwd_bwd(X_local: torch.Tensor, Y_local: torch.Tensor, W: Optional[torch.Tensor],
                                sid_local: torch.Tensor, estimator: str = "dv", precision: str = "fast",
                                inv_tau: float = 1.0, need_grads: bool = True, group=None, backend=None,
                                two_pass: bool = False, check_guard: bool = True):
    """Returns (stats dict of 0-d fp64 tensors incl. 'loss', dX_local, dY_local, dW) — dW already
    summed over ranks.  All ranks must hold the same number of rows.

    dv / infonce / infonce_row take the single pass with sampled references.  Its guard (rows whose reference left the safe
    window, summed over ranks — every rank sees the same number) is read on the host as soon as the score tiles are done; if
    it is non-zero the step is repeated on the exact path (``two_pass=True``: statistics pass + gradient pass).
    ``check_guard=False`` skips that host read (no synchronisation at all); the count is then left in stats['guard'] for the
    caller to act on."""
    if precision not in ("fast", "strict"):      # before any collective: "fp32" exists for the MLP critic only
        raise ValueError(f"the batch-sharded dot / bilinear critic supports the fast and strict precisions, not {precision!r}")
    if backend is None:
        from . import ops as backend  # the CUDA path; raises if the library / device is missing
    world, rank = _world(group)
    Bl, D = X_local.shape
    Bg = Bl * world
    off = rank * Bl
    bilinear = W is not None
    sym = estimator == "infonce_sym"
    dv_like = estimator in ("dv", "infonce", "infonce_ref")
    strict = precision == "strict"

    Xb, Yb = backend.as_bf16(X_local), backend.as_bf16(Y_local)
    Wb = backend.as_bf16(W) if bilinear else None
    # strict mode keeps T = X W as a hi/lo bf16 pair (16 significant bits into the score GEMM)
    # ---- the exchange step
    nccl = world > 1 and dist.get_backend(group) != "gloo"
    single = need_grads and not sym and not two_pass
    # symmetric InfoNCE always uses exact statistics; MI_SYM_RC=0 keeps its older op-by-op form (see below) for A/B runs
    one_call_sym = sym and need_grads and os.environ.get("MI_SYM_RC", "1") != "0"
    if (nccl and (single or one_call_sym) and sid_local.dtype == torch.int32 and hasattr(backend, "sharded_step")
            and os.environ.get("MI_SHARDED_IMPL", "c") != "python"):
        # the whole step, collectives included, as ONE library call (csrc/sharded.cuh): no per-op host overhead
        st, lo, dX, dY, dW = backend.sharded_step(Xb, Yb, Wb, sid_local, estimator, precision, inv_tau, group=group,
                                                  check_guard=check_guard)
        if st == 0:
            out = {"loss": lo[0], "pos_mean": lo[1], "lse_neg": lo[2], "n_neg": lo[3], "loss_row": lo[4],
                   "rows_without_negatives": lo[6], "guard": lo[7]}
            if sym:
                out["loss_col"] = lo[5]
            return out, dX, dY, dW
        if sym:
            raise RuntimeError(f"mi_sharded_critic_loss_fwd_bwd: unexpected status {st} for infonce_sym")
        out, dX, dY, dW = sharded_critic_loss_fwd_bwd(X_local, Y_local, W, sid_local, estimator, precision, inv_tau,
                                                       need_grads, group, backend, two_pass=True)      # guard tripped on every rank
        out["guard"] = torch.ones((), dtype=torch.float64, device=out["loss"].device)
        return out, dX, dY, dW
    T_local = backend.gemm(Xb, Wb, b_t=True, out_dtype=torch.bfloat16, out_split=strict) if bilinear else Xb   # X W, W in place
    smp = lam = None
    sid_all = None
    if single:
        # softmax references of this rank's rows from a sample of its OWN column block (needs nothing from the other ranks,
        # so it runs before / under the all-gather of the text embeddings); lambda = the largest reference of ALL ranks
        sid_own = sid_local if sid_local.dtype == torch.int32 else dense_labels(sid_local.to(torch.int64))
        smp = backend.score_ref_sample(T_local, Yb, sid_own, sid_own, 0, inv_tau, not dv_like, subset=world > 1)
        lam = smp["lam"]
        if world > 1 and sid_local.dtype == torch.int32:
            # ONE small all-gather carries the study ids and lambda (raw float bits); it goes first, so the mask pre-pass
            # runs under the big one
            meta = torch.cat((sid_local.reshape(-1), lam.reshape(1).to(torch.float32).view(torch.int32)))
            meta_all = _all_gather_rows(meta.reshape(1, Bl + 1), world, group)
            sid_all = meta_all[:, :Bl].reshape(-1)
            lam = meta_all[:, Bl].contiguous().view(torch.float32).max().reshape(1)
        elif world > 1:
            lam = lam.clone()
            dist.all_reduce(lam, op=dist.ReduceOp.MAX, group=group)
    Y_all, ev_y = Yb, None
    # the rank's own column block is scored under the all-gather of the other ranks' text embeddings (MI_OWN_COLUMNS_FIRST=0
    # switches this off for A/B runs)
    own_first = nccl and single and os.environ.get("MI_OWN_COLUMNS_FIRST", "1") == "1"
    if world > 1:
        Y_all = torch.empty((Bg, D), dtype=Yb.dtype, device=Yb.device)
        if own_first:
            # in-place all-gather: this rank's rows are in their slot before the collective starts (NCCL leaves the own
            # slot alone), so the pass can score its own column block while the other ranks' rows are still arriving
            Y_all[off:off + Bl].copy_(Yb)
            y_work = dist.all_gather_into_tensor(Y_all, Y_all[off:off + Bl], group=group, async_op=True)
        else:
            y_work = dist.all_gather_into_tensor(Y_all, Yb, group=group, async_op=True)
        if nccl and single:
            # the compute stream does NOT wait here: the library waits for this event right before it first reads
            # the text embeddings, after the mask pre-pass is enqueued
            side = _side_stream(Yb.device)
            with torch.cuda.stream(side):
                y_work.wait()
                ev_y = torch.cuda.Event()
                ev_y.record(side)
        else:
            y_work.wait()
    # symmetric InfoNCE: the column statistics come out of the SAME pass as the rows (mi_score_stats_rc) and the ranks'
    # column partials (B floats each) are merged below; the older form ran a second pass over the transposed block and
    # all-gathered T for it (MI_SYM_RC=0 keeps it for A/B)
    sym_rc = sym and hasattr(backend, "score_stats_rc") and os.environ.get("MI_SYM_RC", "1") != "0"
    T_all = _gather_mat(T_local, world, group) if (sym and not sym_rc) else None
    if sid_all is None:
        if sid_local.dtype == torch.int32:                       # already exact int32 ids: use as they are
            sid_all = _all_gather_rows(sid_local.contiguous(), world, group)
        else:                                                    # identical on every rank, no host sync
            sid_all = dense_labels(_all_gather_rows(sid_local.to(torch.int64), world, group))
    sid_loc = sid_all[off:off + Bl].contiguous()

    if nccl and hasattr(backend, "set_overlap_reserve_sms"):
        # (experiment knob) SMs left free for the overlapped dY exchange; 0 = the engine uses every SM
        backend.set_overlap_reserve_sms(int(os.environ.get("MI_RS_RESERVE_SMS", "0")))
    if single:
        try:
            return _single_pass_step(backend, T_local, Xb, Yb, Wb, Y_all, sid_loc, sid_all, off, Bl, Bg, D, inv_tau, estimator,
                                     precision, smp, lam, world, group, nccl, ev_y=ev_y, own_first=own_first,
                                     check_guard=check_guard)
        except GuardTripped:
            # every rank raised (the merged count is identical everywhere): repeat with exact references; the work the
            # abandoned pass still has queued finishes first, in stream order
            out, dX, dY, dW = sharded_critic_loss_fwd_bwd(X_local, Y_local, W, sid_local, estimator, precision, inv_tau,
                                                           need_grads, group, backend, two_pass=True)
            out["guard"] = torch.ones((), dtype=torch.float64, device=out["loss"].device)
            return out, dX, dY, dW

    # ---- statistics (S never materialised)
    col_lse = None
    if sym_rc:
        rows_r, scal_r, col_lse = backend.score_stats_rc(T_local, Y_all, sid_loc, sid_all, off, inv_tau)
    else:
        rows_r, scal_r = backend.score_stats(T_local, Y_all, sid_loc, sid_all, off, inv_tau)
    g_r = merge_scalars(_all_gather_rows(scal_r.reshape(1, 8), world, group))
    out = {"pos_mean": g_r["diag_sum"] / Bg, "lse_neg": g_r["lse_neg"], "n_neg": g_r["n_neg"],
           "loss_row": g_r["rowloss_sum"] / Bg}
    rows_c, c_all = None, None
    if sym_rc:
        # column j over ALL rows = log-sum-exp of the ranks' block values; its positive pair S[j, j] lives with the rows
        col_all = _all_gather_rows(col_lse.reshape(1, Bg), world, group).double()                 # [world, B]
        diag_all = _all_gather_rows(rows_r[:, 2].contiguous(), world, group).double()             # [B]
        lse_c = torch.logaddexp(torch.logsumexp(col_all, 0), diag_all)
        out["loss_col"] = (lse_c - diag_all).sum() / Bg
        c_all = lse_c.to(torch.float32)
    elif sym:
        rows_c, scal_c = backend.score_stats(Yb, T_all, sid_loc, sid_all, off, inv_tau)
        g_c = merge_scalars(_all_gather_rows(scal_c.reshape(1, 8), world, group))
        out["loss_col"] = g_c["rowloss_sum"] / Bg
    if estimator == "dv":
        # mi_critics.py:10 rounds N_neg to fp32 before the log; same formula as the fused C path
        log_n = torch.log(out["n_neg"].to(torch.float32).to(torch.float64))
        out["loss"] = out["lse_neg"] - log_n - out["pos_mean"]
    elif estimator in ("infonce", "infonce_ref"):
        out["loss"] = out["lse_neg"] - out["pos_mean"]
    elif estimator == "infonce_row":
        out["loss"] = out["loss_row"]
    elif sym:
        out["loss"] = 0.5 * (out["loss_row"] + out["loss_col"])
    else:
        raise ValueError(f"unknown estimator {estimator!r}")
    if not need_grads:
        return out, None, None, None

    # ---- one gradient pass per rank: dT_r (complete) and this rank's contribution to every dY_j
    gamma = 1.0 / Bg
    if dv_like:
        ref = out["lse_neg"].to(torch.float32).expand(Bl).contiguous()
        args = dict(refq=ref, wq=1.0, refk=None, wk=0.0, include_diag=False)
    elif sym:
        if c_all is None:
            c_all = _all_gather_rows(rows_c[:, 3].contiguous(), world, group)
        args = dict(refq=rows_r[:, 3].contiguous(), wq=0.5 / Bg, refk=c_all, wk=0.5 / Bg, include_diag=True)
    else:
        args = dict(refq=rows_r[:, 3].contiguous(), wq=1.0 / Bg, refk=None, wk=0.0, include_diag=True)
    ev = None
    if nccl:                                          # marks "dY contributions complete" inside the fused pass
        ev = torch.cuda.Event()
        ev.record()
        args["event_after_k"] = ev
    dT32, dT16, dY_part = backend.score_grad(T_local, Y_all, sid_loc, sid_all, off, inv_tau, precision=precision,
                                             alpha=inv_tau, gamma=gamma, want_f32=not bilinear, want_bf16=bilinear,
                                             out_split=bilinear and strict, want_k=True, **args)
    rs_work = None
    if nccl:
        # reduce-scatter starts as soon as the dY contributions are complete and runs under the dT
        # contraction and the dX / dW GEMMs still queued on the compute stream
        main = torch.cuda.current_stream()
        side = _side_stream(dY_part.device)
        side.wait_event(ev)
        dY = torch.empty((Bl, D), dtype=dY_part.dtype, device=dY_part.device)
        with torch.cuda.stream(side):
            rs_work = dist.reduce_scatter_tensor(dY, dY_part, op=dist.ReduceOp.SUM, group=group, async_op=True)
        dY_part.record_stream(side)
        dY.record_stream(side)
    elif world > 1:                                   # gloo (CPU tests) has no reduce-scatter
        dist.all_reduce(dY_part, op=dist.ReduceOp.SUM, group=group)
        dY = dY_part[off:off + Bl].contiguous()
    else:
        dY = dY_part
    dX, dW = dT32, None
    if bilinear:
        dX = backend.gemm(dT16, Wb)                                               # dT W^T
        dW = backend.gemm(Xb, dT16, a_t=True, b_t=True)                           # X^T dT (local rows), operands in place
        if world > 1:
            dist.all_reduce(dW, op=dist.ReduceOp.SUM, group=group)
    if rs_work is not None:
        rs_work.wait()                                # current (compute) stream waits for the collective
    return out, dX, dY, dW


# ---- the reference's own critic, make_mlp(2D, [H1, H2]) (DESIGN 8.4): the same row-block sharding over stage ops
#
#   1. reference logit from a sample of the rank's OWN block (single pass only; no exchange needed), then ONE small
#      all-gather of the study ids with the reference packed in (all-reduce MAX for int64 ids), and the all-gather of Y
#   2. the block pass over Bl x Bg pairs (mi_mlp_block_fwd) -> the rank's scalar row (slot 7: its sum of the weights)
#   3. all-gather of the 8 fp64 scalars, merge (mi_mlp_block_merge): the global loss and the single pass' guard — the same
#      on every rank; a tripped guard repeats the step with the two-pass sequence
#   4. the block's backward (mi_mlp_block_bwd): dX_r, the image half of dW1, partial dW2 / db2 / dW3 / db3 / db1 and the
#      rank's contribution dC_part [Bg, H1] to dL/dC of every text row
#   5. reduce-scatter of dC_part -> dC_r; dY_r and the text half of dW1 (mi_mlp_input_grad); ONE all-reduce of the flat
#      parameter gradients
#   infonce_sym (two-pass only): step 2 also gives the block's column partials [Bg] (log-sum-exp of every column over the
#   rank's rows); ONE all-gather of them, merged in fp64 on every rank, completes the column loss after step 3 and is the
#   column normaliser of the backward in step 4

MLP_GRAD_NAMES = ("dW1", "db1", "dW2", "db2", "dW3", "db3")


def sharded_mlp_critic_loss_fwd_bwd(X_local: torch.Tensor, Y_local: torch.Tensor, params, sid_local: torch.Tensor,
                                    estimator: str = "dv", precision: str = "fast", need_grads: bool = True, group=None,
                                    backend=None, two_pass: bool = False, check_guard: bool = True):
    """Global-batch loss of the concat-MLP critic when every rank holds a row shard (all ranks the same number of rows);
    ``params`` = (W1 [H1, 2D], b1, W2 [H2, H1], b2, W3 [1, H2], b3), replicated.  Returns (stats dict of 0-d fp64 tensors
    incl. 'loss' and 'guard', dX_local, dY_local, grads dict dW1 ... db3 already summed over ranks) — the gradients are
    None without ``need_grads``.

    dv / infonce with gradients take the single pass (unless mi_set_mlp_mode cleared bit 0); its guard is read on the host
    after the scalar exchange and, if it tripped on the global weight sum, every rank repeats the step with the two-pass
    sequence and reports guard = 1.  ``check_guard=False`` skips that host read; the verdict is then left in
    stats['guard'] for the caller to act on.  infonce_row, infonce_sym (stats also hold 'loss_col'), forward-only calls
    and ``two_pass=True`` use the two-pass sequence."""
    if backend is None:
        from . import ops as backend  # the CUDA path; raises if the library / device is missing
    if estimator not in ("dv", "infonce", "infonce_ref", "infonce_row", "infonce_sym"):
        raise ValueError(f"the MLP critic supports the dv, infonce, infonce_row and infonce_sym estimators, not {estimator!r}")
    world, rank = _world(group)
    Bl, D = X_local.shape
    Bg = Bl * world
    off = rank * Bl
    sym = estimator == "infonce_sym"
    dv_like = estimator not in ("infonce_row", "infonce_sym")
    single = need_grads and dv_like and not two_pass and (backend.get_mlp_mode() & 1) != 0
    nccl = world > 1 and dist.get_backend(group) != "gloo"
    X, Y = X_local.detach(), Y_local.detach()
    params = tuple(p.detach() for p in params)

    ref = backend.mlp_block_ref_logit(X, Y, params, 0, precision) if single else None
    if sid_local.dtype == torch.int32:
        if single and world > 1:
            # ONE small all-gather carries the study ids and the reference (raw float bits)
            meta = torch.cat((sid_local.reshape(-1), ref.reshape(1).to(torch.float32).view(torch.int32)))
            meta_all = _all_gather_rows(meta.reshape(1, Bl + 1), world, group)
            sid_all = meta_all[:, :Bl].reshape(-1).contiguous()
            ref = meta_all[:, Bl].contiguous().view(torch.float32).max().reshape(1)
        else:
            sid_all = _all_gather_rows(sid_local.contiguous(), world, group)
    else:                                                        # identical relabelling on every rank, no host sync
        sid_all = dense_labels(_all_gather_rows(sid_local.to(torch.int64).contiguous(), world, group))
        if single and world > 1:
            ref = ref.clone()
            dist.all_reduce(ref, op=dist.ReduceOp.MAX, group=group)
    sid_loc = sid_all[off:off + Bl].contiguous()
    Y_all = _all_gather_rows(Y.contiguous(), world, group)

    # ---- the block pass and the scalar exchange
    fw = backend.mlp_block_fwd(X, Y_all, params, sid_loc, sid_all, off, estimator, precision, ref, not single)
    scal, state = fw[0], fw[1]
    scal_all = _all_gather_rows(scal.reshape(1, 8), world, group)
    loss, merged = backend.mlp_block_merge(scal_all, Bg, estimator, not single)
    col_lse = None
    if sym:
        # column j over the batch = log-sum-exp of the ranks' partials (each holds the positive pair in exactly one block);
        # the merge leaves slots 0 / 5 of loss_out to this side
        c = torch.logsumexp(_all_gather_rows(fw[2].reshape(1, Bg), world, group).double(), 0)
        loss = loss.clone()
        loss[5] = (c.sum() - Bg * loss[1]) / Bg
        loss[0] = 0.5 * (loss[4] + loss[5])
        col_lse = c
    if single and check_guard and float(loss[7]) != 0.0:
        # every rank sees the same merged rows: all of them repeat the step with exact statistics
        out, dX, dY, grads = sharded_mlp_critic_loss_fwd_bwd(X_local, Y_local, params, sid_local, estimator, precision,
                                                             need_grads, group, backend, two_pass=True)
        out["guard"] = torch.ones((), dtype=torch.float64, device=out["loss"].device)
        return out, dX, dY, grads
    out = {"loss": loss[0], "pos_mean": loss[1], "lse_neg": loss[2], "n_neg": loss[3], "loss_row": loss[4],
           "rows_without_negatives": loss[6], "guard": loss[7]}
    if sym:
        out["loss_col"] = loss[5]
    if not need_grads:
        return out, None, None, None

    # ---- backward of the block, exchange of the dC contributions, layer 1 of the own text rows
    extra = {"col_lse": col_lse} if sym else {}          # a backend without the symmetric estimator needs no such argument
    g = backend.mlp_block_bwd(X, Y_all, params, sid_loc, sid_all, off, estimator, precision, not single, loss, merged, state,
                              **extra)
    ev = None
    if nccl:
        ev = torch.cuda.Event()
        ev.record()
    dC, rs_work = _reduce_scatter_rows(g["dC_part"], Bl, off, world, group, nccl, ev)
    if rs_work is not None:
        rs_work.wait()
    if isinstance(dC, _A2ASum):
        dC = dC.resolve()
    dY, dW1, _ = backend.mlp_input_grad(dC, Y, params[0], 1, precision, dW1=g["dW1"])
    grads = {"dW1": dW1, "db1": g["db1"], "dW2": g["dW2"], "db2": g["db2"], "dW3": g["dW3"], "db3": g["db3"]}
    if world > 1:
        flat = torch.cat([grads[n].reshape(-1) for n in MLP_GRAD_NAMES])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        o = 0
        for n in MLP_GRAD_NAMES:
            k = grads[n].numel()
            grads[n] = flat[o:o + k].view(grads[n].shape)
            o += k
    return out, g["dX"], dY, grads
