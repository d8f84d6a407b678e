"""TEST INFRASTRUCTURE: the fp64 CPU emulation of the MLP critic's row-block stage ops (tests/cpu_backend_mlp.py) with
symmetric InfoNCE added, as mi_b200.ops has it: mlp_block_fwd also returns the block's column partials
(mi_mlp_block_fwd_rc) and mlp_block_bwd takes the merged columns (mi_mlp_block_bwd_rc).  Every other estimator goes to
the base emulation unchanged.  Used ONLY to exercise mi_b200.dist.sharded_mlp_critic_loss_fwd_bwd under gloo without a
GPU.  Never imported by the product."""
import torch

import cpu_backend_mlp as _base
from cpu_backend_mlp import (get_mlp_mode, mlp_block_merge, mlp_block_ref_logit, mlp_input_grad,  # noqa: F401
                             set_mlp_mode)


def _positives(Bq, Bk, q_offset):
    pos = torch.zeros(Bq, Bk, dtype=torch.bool)
    i = torch.arange(Bq)
    pos[i, q_offset + i] = True
    return pos


def mlp_block_fwd(X, Y, params, sid_q, sid_k, q_offset, estimator, precision, ref, two_pass):
    out = _base.mlp_block_fwd(X, Y, params, sid_q, sid_k, q_offset, estimator, precision, ref, two_pass)
    if estimator != "infonce_sym":
        return out
    assert two_pass, "infonce_sym runs the two-pass sequence only"
    scal, state = out
    S, M = state["S"], state["M"]
    R = M | _positives(S.shape[0], S.shape[1], q_offset)
    col = torch.logsumexp(torch.where(R, S, torch.full_like(S, float("-inf"))), 0)     # the block's column partials
    return scal, state, col


def mlp_block_bwd(X, Y, params, sid_q, sid_k, q_offset, estimator, precision, two_pass, loss, merged, state, col_lse=None):
    if estimator != "infonce_sym":
        return _base.mlp_block_bwd(X, Y, params, sid_q, sid_k, q_offset, estimator, precision, two_pass, loss, merged, state)
    Bq, D = X.shape
    S, M = state["S"], state["M"]
    Bg = Y.shape[0]
    pos = _positives(Bq, Bg, q_offset)
    # G = (1/2B) R . (e^{S - r_i} + e^{S - c_j}) - I/B
    e = torch.exp(S - state["lse_all"][:, None]) + torch.exp(S - col_lse.double()[None, :])
    G = torch.where(M | pos, e / (2 * Bg), torch.zeros_like(S)) - pos.double() / Bg
    A, C, rest = _base._mlp_layers(X, Y, params)
    A, C = A.detach().requires_grad_(True), C.detach().requires_grad_(True)
    rest = tuple(t.detach().requires_grad_(True) for t in rest)
    (_base._mlp_scores(A, C, rest) * G).sum().backward()
    W1 = params[0].double()
    dW1 = torch.zeros_like(W1)
    dW1[:, :D] = A.grad.t() @ X.double()
    return {"dX": A.grad @ W1[:, :D], "dC_part": C.grad, "dW1": dW1, "db1": A.grad.sum(0), "dW2": rest[0].grad,
            "db2": rest[1].grad, "dW3": rest[2].grad.reshape(1, -1), "db3": rest[3].grad.reshape(1)}
