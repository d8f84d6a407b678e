"""L1 oracle of the f-divergence estimators: Jensen-Shannon (``js``) and NWJ (``nwj``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  The reference has neither estimator; they are anchored to it
through the shared score matrix and negatives mask (``matrix_oracle.negatives_mask``, main_utils.py:105), as the
row / symmetric InfoNCE forms are.  Losses are minimised (minus the bound), M = the negatives mask, N = |M|:

* js  : L = mean_{(i,j) in M} softplus(S_ij) + mean_i softplus(-S_ii)
        G = dL/dS = M sigma(S) / N - diag(sigma(-S_ii)) / B
* nwj : L = e^{-1} mean_{M} e^{S} - mean_i S_ii = e^{LSE_M(S) - ln N - 1} - mean_i S_ii      (ln N in fp64)
        G = kappa softmax_M(S) - I / B,  kappa = e^{LSE_M - ln N - 1}

Three forms, proved equal in ``tests/test_host_js_nwj_cpu.py``: the matrix form (fp64, closed-form gradients), the
pair form (reference-ordered pair logits, autograd) and a row-chunked form for batches whose B x B matrix does not fit
(B = 65536), like ``chunked_oracle.py``.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from . import matrix_oracle as mo

FDIV_ESTIMATORS = ("js", "nwj")


# --------------------------------------------------------------------------
# plain-logits form (positives first, then the negatives in the reference's pair order)
# --------------------------------------------------------------------------
def js_bound_loss(logits: torch.Tensor, pos_size: int) -> torch.Tensor:
    pos, neg = logits[:pos_size], logits[pos_size:]
    return torch.mean(F.softplus(neg)) + torch.mean(F.softplus(-pos))


def nwj_bound_loss(logits: torch.Tensor, pos_size: int) -> torch.Tensor:
    pos, neg = logits[:pos_size], logits[pos_size:]
    n_neg = neg.numel()
    ln_n = math.log(n_neg) if n_neg > 0 else -math.inf
    return torch.exp(torch.logsumexp(neg.reshape(-1), dim=0) - (ln_n + 1.0)) - torch.mean(pos)


BOUND_LOSS = {"js": js_bound_loss, "nwj": nwj_bound_loss}


# --------------------------------------------------------------------------
# matrix form
# --------------------------------------------------------------------------
def estimator_from_scores(S: torch.Tensor, M: torch.Tensor, estimator: str) -> Dict[str, torch.Tensor]:
    """Loss and the loss_out slots of the fused call from a square score matrix and the negatives mask."""
    diag = torch.diagonal(S)
    pos = diag.mean()
    n_neg = int(M.sum())
    out = {"pos_mean": pos, "n_neg": torch.tensor(float(n_neg), dtype=S.dtype)}
    if estimator == "js":
        sp_neg = torch.where(M, F.softplus(S), torch.zeros_like(S)).sum() / n_neg if n_neg else torch.tensor(math.nan, dtype=S.dtype)
        sp_pos = F.softplus(-diag).mean()
        out.update(loss=sp_neg + sp_pos, sp_neg=sp_neg, sp_pos=sp_pos)
        return out
    if estimator == "nwj":
        lse = mo._masked_lse(S, M)
        ln_n = math.log(n_neg) if n_neg else -math.inf
        out.update(loss=torch.exp(lse - (ln_n + 1.0)) - pos, lse_neg=lse)
        return out
    raise ValueError(f"unknown estimator {estimator!r}")


def score_gradient(S: torch.Tensor, M: torch.Tensor, estimator: str) -> torch.Tensor:
    """Closed form of dL/dS."""
    B = S.shape[0]
    n_neg = int(M.sum())
    eye = torch.eye(B, dtype=S.dtype)
    if estimator == "js":
        G = torch.where(M, torch.sigmoid(S), torch.zeros_like(S)) / n_neg
        return G - torch.diag(torch.sigmoid(-torch.diagonal(S))) / B
    if estimator == "nwj":
        lse = mo._masked_lse(S, M)
        kappa = torch.exp(lse - (math.log(n_neg) + 1.0))
        return kappa * torch.where(M, torch.exp(S - lse), torch.zeros_like(S)) - eye / B
    raise ValueError(f"unknown estimator {estimator!r}")


def critic_loss(X, Y, study_id, W=None, inv_tau: float = 1.0, estimator: str = "js",
                dtype=torch.float64, grads: bool = True) -> Dict[str, torch.Tensor]:
    """Matrix-form loss and closed-form gradients on the CPU (dT = G Y, dY = G^T T, dX = dT W^T, dW = X^T dT)."""
    X = X.detach().to("cpu", dtype)
    Y = Y.detach().to("cpu", dtype)
    Wd = None if W is None else W.detach().to("cpu", dtype)
    sid = study_id if torch.is_tensor(study_id) else mo.dense_ids(study_id)
    sid = sid.to("cpu")
    M = mo.negatives_mask(sid, sid)
    T = X if Wd is None else X @ Wd
    S = (T @ Y.t()) * inv_tau
    out = estimator_from_scores(S, M, estimator)
    if grads:
        G = score_gradient(S, M, estimator) * inv_tau
        dT = G @ Y
        out["dY"] = G.t() @ T
        out["dT"] = dT
        if Wd is None:
            out["dX"] = dT
        else:
            out["dX"] = dT @ Wd.t()
            out["dW"] = X.t() @ dT
    return out


def critic_loss_pair_form(X, Y, study_id, W=None, inv_tau: float = 1.0, estimator: str = "js", dtype=torch.float64):
    """The reference's sequence create_mi_pairs -> separable critic -> loss on the flat logits, differentiated by autograd."""
    X = X.detach().to("cpu", dtype).requires_grad_(True)
    Y = Y.detach().to("cpu", dtype).requires_grad_(True)
    Wd = None if W is None else W.detach().to("cpu", dtype).requires_grad_(True)
    rows = mo.create_mi_pairs(X, Y, list(study_id))
    logits = mo.pair_logits_separable(rows, Wd, inv_tau)
    loss = BOUND_LOSS[estimator](logits, len(study_id))
    params = [X, Y] + ([Wd] if Wd is not None else [])
    g = torch.autograd.grad(loss, params)
    out = {"loss": loss.detach(), "dX": g[0], "dY": g[1]}
    if Wd is not None:
        out["dW"] = g[2]
    return out


# --------------------------------------------------------------------------
# row-chunked form (B x B never materialised; fp32 matmuls with TF32 off, fp64 reductions, any device)
# --------------------------------------------------------------------------
def critic_loss_chunked(X: torch.Tensor, Y: torch.Tensor, sid: torch.Tensor, W: Optional[torch.Tensor] = None,
                        inv_tau: float = 1.0, estimator: str = "js", chunk: int = 4096, grads: bool = True,
                        T: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """As ``chunked_oracle.critic_loss_chunked`` for js / nwj.  ``T`` overrides X W (the CUDA path's own rounded T)."""
    allow = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        dev = X.device
        B, D = X.shape
        Xf, Yf = X.float(), Y.float()
        Wf = None if W is None else W.float()
        Tf = (Xf if Wf is None else Xf @ Wf) if T is None else T.float()
        sid = sid.to(dev)
        f64 = dict(dtype=torch.float64, device=dev)
        diag = ((Tf.double() * Yf.double()).sum(1)) * inv_tau
        n_neg = 0.0
        sp_sum = torch.zeros((), **f64)
        g_m, g_s = torch.full((1,), float("-inf"), **f64), torch.zeros(1, **f64)
        for r0 in range(0, B, chunk):
            r1 = min(B, r0 + chunk)
            S = (Tf[r0:r1] @ Yf.t()).double() * inv_tau
            M = sid[r0:r1, None] != sid[None, :]
            n_neg += float(M.sum())
            if estimator == "js":
                sp_sum = sp_sum + torch.where(M, F.softplus(S), torch.zeros_like(S)).sum()
            else:
                Sn = torch.where(M, S, torch.full_like(S, float("-inf")))
                bm = Sn.max().reshape(1)
                nm = torch.maximum(g_m, bm)
                if torch.isfinite(nm).all():
                    g_s = g_s * torch.exp(g_m - nm) + torch.exp(Sn - nm).sum()
                    g_m = nm
        out: Dict[str, torch.Tensor] = {"pos_mean": diag.mean(), "n_neg": torch.tensor(n_neg, **f64)}
        if estimator == "js":
            out["sp_neg"] = sp_sum / n_neg
            out["sp_pos"] = F.softplus(-diag).mean()
            out["loss"] = out["sp_neg"] + out["sp_pos"]
        else:
            lse = (g_m + torch.log(g_s)).reshape(())
            out["lse_neg"] = lse
            out["kappa"] = torch.exp(lse - (math.log(n_neg) + 1.0))
            out["loss"] = out["kappa"] - diag.mean()
        if not grads:
            return out
        dT = torch.empty((B, D), dtype=torch.float32, device=dev)
        dY = torch.zeros((B, D), dtype=torch.float64, device=dev)
        for r0 in range(0, B, chunk):
            r1 = min(B, r0 + chunk)
            S = (Tf[r0:r1] @ Yf.t()).double() * inv_tau
            M = sid[r0:r1, None] != sid[None, :]
            idx = torch.arange(r0, r1, device=dev)
            if estimator == "js":
                G = torch.where(M, torch.sigmoid(S), torch.zeros_like(S)) / n_neg
                G[idx - r0, idx] -= torch.sigmoid(-diag[r0:r1]) / B
            else:
                G = out["kappa"] * torch.where(M, torch.exp(S - out["lse_neg"]), torch.zeros_like(S))
                G[idx - r0, idx] -= 1.0 / B
            G = (G * inv_tau).float()
            dT[r0:r1] = G @ Yf
            dY += (G.t() @ Tf[r0:r1]).double()
        out["dY"] = dY.float()
        out["dT"] = dT
        if Wf is None:
            out["dX"] = dT
        else:
            out["dX"] = dT @ Wf.t()
            out["dW"] = (Xf.double().t() @ dT.double()).float()
        return out
    finally:
        torch.backends.cuda.matmul.allow_tf32 = allow
