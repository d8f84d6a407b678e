"""TEST INFRASTRUCTURE: a CPU emulation of the MLP critic's row-block stage ops of mi_b200.ops (mi_mlp_block_*,
mi_mlp_input_grad, include/mi_b200.h) in fp64 with the library's semantics, used ONLY to exercise the host-side sharding /
collective logic of mi_b200.dist.sharded_mlp_critic_loss_fwd_bwd under gloo without a GPU.  Never imported by the product."""
import torch

MLP_MARGIN = 47.82715406979468          # kMlpSpMargin: the single pass' reference = sample maximum + 69 ln 2
_MLP_MODE = [3]


def set_mlp_mode(mode):
    _MLP_MODE[0] = 3 if mode < 0 else (mode & 3)


def get_mlp_mode():
    return _MLP_MODE[0]


def _mlp_layers(X, Y, params):
    W1, b1, W2, b2, W3, b3 = (p.double() for p in params)
    D = X.shape[1]
    A = X.double() @ W1[:, :D].t() + b1
    C = Y.double() @ W1[:, D:].t()
    return A, C, (W2, b2, W3.reshape(1, -1), b3.reshape(1))


def _mlp_scores(A, C, rest):
    W2, b2, W3, b3 = rest
    h1 = torch.relu(A[:, None, :] + C[None, :, :])
    return (torch.relu(h1 @ W2.t() + b2) @ W3.t()).squeeze(-1) + b3


def _mlp_scal(lse_neg, n_neg, diag, lse_all):
    fin = torch.isfinite(lse_neg)
    m = lse_neg[fin].max() if fin.any() else torch.tensor(float("-inf"), dtype=torch.float64)
    scal = torch.zeros(8, dtype=torch.float64)
    scal[0] = m
    scal[1] = torch.exp(lse_neg[fin] - m).sum()
    scal[2] = n_neg.sum()
    scal[3] = diag.sum()
    scal[4] = (lse_all - diag).sum()
    scal[5] = (n_neg == 0).sum()
    return scal


def mlp_block_ref_logit(X, Y, params, q_offset, precision="fast"):
    A, C, rest = _mlp_layers(X, Y, params)
    Bq = X.shape[0]
    ns = min(Bq, 256)
    stride = Bq // ns
    idx = torch.arange(ns) * stride
    return _mlp_scores(A[idx], C[q_offset + idx], rest).max().reshape(1)


def mlp_block_fwd(X, Y, params, sid_q, sid_k, q_offset, estimator, precision, ref, two_pass):
    A, C, rest = _mlp_layers(X, Y, params)
    S = _mlp_scores(A, C, rest)
    M = sid_q[:, None] != sid_k[None, :]
    i = torch.arange(X.shape[0])
    diag = S[i, q_offset + i]
    n_neg = M.sum(1).double()
    state = {"S": S, "M": M}
    if two_pass:
        lse_neg = torch.logsumexp(torch.where(M, S, torch.full_like(S, float("-inf"))), 1)
        lse_all = torch.logaddexp(lse_neg, diag)
        state["lse_all"] = lse_all
        return _mlp_scal(lse_neg, n_neg, diag, lse_all), state
    g = torch.where(M, torch.exp(S - (ref.double() + MLP_MARGIN)), torch.zeros_like(S))     # reference units
    l = g.sum(1)
    lse_neg = torch.where(n_neg > 0, ref.double() + MLP_MARGIN + torch.log(l), torch.full_like(l, float("-inf")))
    scal = _mlp_scal(lse_neg, n_neg, diag, torch.logaddexp(lse_neg, diag))
    scal[7] = l.sum()
    state["g"] = g
    return scal, state


def mlp_block_merge(scal_all, b_global, estimator, two_pass):
    v = scal_all.double()
    gm = v[:, 0].max()
    fin = torch.isfinite(v[:, 0])
    merged = torch.zeros(8, dtype=torch.float64)
    merged[0] = gm
    merged[1] = (v[fin, 1] * torch.exp(v[fin, 0] - gm)).sum()
    merged[2:] = v[:, 2:].sum(0)
    lse = merged[0] + torch.log(merged[1])
    n_neg, pos, loss_row = merged[2], merged[3] / b_global, merged[4] / b_global
    if estimator == "dv":
        loss = lse - torch.log(n_neg.float().double()) - pos
    elif estimator in ("infonce", "infonce_ref"):
        loss = lse - pos
    else:
        loss = loss_row
    guard = merged[6].clone()
    if not two_pass and n_neg > 0 and not (1e-30 <= float(merged[7]) <= 1e30):
        guard += 1.0
    out = torch.stack([loss, pos, lse, n_neg, loss_row, torch.zeros((), dtype=torch.float64), merged[5], guard])
    return out, merged


def mlp_block_bwd(X, Y, params, sid_q, sid_k, q_offset, estimator, precision, two_pass, loss, merged, state):
    Bq, D = X.shape
    S, M = state["S"], state["M"]
    Bg = Y.shape[0]
    i = torch.arange(Bq)
    pos = torch.zeros_like(M)
    pos[i, q_offset + i] = True
    if not two_pass:
        total = float(merged[7])
        cfac = 1.0 / total if (float(loss[3]) > 0 and 1e-30 <= total <= 1e30) else 0.0
        G = state["g"] * cfac
    elif estimator != "infonce_row":
        G = torch.where(M, torch.exp(S - loss[2]), torch.zeros_like(S))
    else:
        G = torch.where(M | pos, torch.exp(S - state["lse_all"][:, None]) / Bg, torch.zeros_like(S))
    G = G - pos.double() / Bg
    A, C, rest = _mlp_layers(X, Y, params)
    A, C = A.detach().requires_grad_(True), C.detach().requires_grad_(True)
    rest = tuple(t.detach().requires_grad_(True) for t in rest)
    (_mlp_scores(A, C, rest) * G).sum().backward()
    W1 = params[0].double()
    dW1 = torch.zeros_like(W1)
    dW1[:, :D] = A.grad.t() @ X.double()
    return {"dX": A.grad @ W1[:, :D], "dC_part": C.grad, "dW1": dW1, "db1": A.grad.sum(0), "dW2": rest[0].grad,
            "db2": rest[1].grad, "dW3": rest[2].grad.reshape(1, -1), "db3": rest[3].grad.reshape(1)}


def mlp_input_grad(dZ, In, W1, side, precision="fast", dW1=None, want_db1=False):
    D = In.shape[1]
    W1 = W1.double()
    if dW1 is None:
        dW1 = torch.zeros_like(W1)
    dW1[:, side * D:(side + 1) * D] = dZ.double().t() @ In.double()
    return dZ.double() @ W1[:, side * D:(side + 1) * D], dW1, (dZ.double().sum(0) if want_db1 else None)
