"""CPU tests of the Jensen-Shannon and NWJ estimators: the fp64 oracle's three forms against each other and autograd, the
package's plain-logits losses against the oracle, estimator selection, and the entries that do not implement the two
estimators rejecting them before any device work."""
import math
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import fdiv_oracle as fo  # noqa: E402
from oracle import matrix_oracle as mo  # noqa: E402

EST = ("js", "nwj")


def _inputs(B, D, dup, bilinear, seed=3):
    X, Y, sid, W = mo.synthetic_embeddings(B, D, seed=seed, dup_frac=dup, bilinear=bilinear)
    return X.double(), Y.double(), sid, (None if W is None else W.double())


def _max_rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


@pytest.mark.parametrize("est", EST)
@pytest.mark.parametrize("bilinear", [False, True])
@pytest.mark.parametrize("dup", [0.0, 0.3])
def test_closed_form_gradient_equals_autograd(est, bilinear, dup):
    X, Y, sid, W = _inputs(24, 16, dup, bilinear)
    T = X if W is None else X @ W
    S = (T @ Y.t() * 0.7).detach().requires_grad_(True)
    M = mo.negatives_mask(sid, sid)
    loss = fo.estimator_from_scores(S, M, est)["loss"]
    (g,) = torch.autograd.grad(loss, S)
    G = fo.score_gradient(S.detach(), M, est)
    assert float((g - G).abs().max()) <= 1e-12 * max(1.0, float(g.abs().max()))


@pytest.mark.parametrize("est", EST)
@pytest.mark.parametrize("bilinear", [False, True])
@pytest.mark.parametrize("dup", [0.0, 0.25])
def test_pair_form_equals_matrix_form(est, bilinear, dup):
    X, Y, sid, W = _inputs(12, 8, dup, bilinear)
    inv_tau = 0.5
    a = fo.critic_loss(X, Y, sid.tolist(), W, inv_tau, est)
    b = fo.critic_loss_pair_form(X, Y, sid.tolist(), W, inv_tau, est)
    assert abs(float(a["loss"]) - float(b["loss"])) <= 1e-12 * max(1.0, abs(float(a["loss"])))
    for k in ("dX", "dY") + (("dW",) if W is not None else ()):
        assert _max_rel(b[k], a[k]) <= 1e-11, k


@pytest.mark.parametrize("est", EST)
@pytest.mark.parametrize("bilinear", [False, True])
def test_chunked_form_equals_matrix_form(est, bilinear):
    X, Y, sid, W = _inputs(70, 16, 0.2, bilinear)
    inv_tau = 0.8
    a = fo.critic_loss(X, Y, sid, W, inv_tau, est)
    Xf, Yf = X.float(), Y.float()
    Wf = None if W is None else W.float()
    c = fo.critic_loss_chunked(Xf, Yf, sid, Wf, inv_tau, est, chunk=16)
    ref = fo.critic_loss(Xf.double(), Yf.double(), sid, None if Wf is None else Wf.double(), inv_tau, est)
    assert abs(float(c["loss"]) - float(ref["loss"])) <= 1e-5 * max(1.0, abs(float(ref["loss"])))
    for k in ("dX", "dY") + (("dW",) if W is not None else ()):
        assert _max_rel(c[k].double(), ref[k]) <= 1e-5, k
    assert float(c["n_neg"]) == float(a["n_neg"])


@pytest.mark.parametrize("est", EST)
def test_matrix_form_slots(est):
    X, Y, sid, W = _inputs(16, 8, 0.25, True)
    out = fo.critic_loss(X, Y, sid, W, 1.0, est, grads=False)
    S = (X @ W) @ Y.t()
    M = mo.negatives_mask(sid, sid)
    if est == "js":
        assert math.isclose(float(out["loss"]), float(out["sp_neg"] + out["sp_pos"]), rel_tol=1e-15)
    else:
        lse = torch.logsumexp(S[M], 0)
        assert math.isclose(float(out["loss"]), math.exp(float(lse) - math.log(int(M.sum())) - 1) - float(S.diagonal().mean()),
                            rel_tol=1e-12)


@pytest.fixture(scope="module")
def pkg():
    import mi_b200
    return mi_b200


@pytest.mark.parametrize("est", EST)
@pytest.mark.parametrize("dup", [0.0, 0.3])
def test_plain_logits_equal_the_oracle_bit_for_bit(pkg, est, dup):
    X, Y, sid, W = _inputs(20, 8, dup, True)
    rows = mo.create_mi_pairs(X, Y, sid.tolist())
    logits = mo.pair_logits_separable(rows, W, 1.0)
    fn = {"js": pkg.js_bound_loss, "nwj": pkg.nwj_bound_loss}[est]
    got = fn(logits, 20)
    want = fo.BOUND_LOSS[est](logits, 20)
    assert got.dim() == 0
    assert torch.equal(got, want)
    assert pkg.select_estimator(est) is fn
    assert float(got) == pytest.approx(float(fo.critic_loss(X, Y, sid, W, 1.0, est, grads=False)["loss"]), rel=1e-12)


@pytest.mark.parametrize("est", EST)
def test_plain_logits_without_negatives_give_nan(pkg, est):
    logits = torch.randn(5, 1, dtype=torch.float64)
    fn = {"js": pkg.js_bound_loss, "nwj": pkg.nwj_bound_loss}[est]
    assert math.isnan(float(fn(logits, 5)))


def test_select_estimator_still_rejects_unknown_names(pkg):
    with pytest.raises(ValueError):
        pkg.select_estimator("mine")


def test_planners_accept_single_gpu_and_reject_sharded():
    from mi_b200 import _lib
    lib = _lib.load()
    for est in (4, 5):
        for critic in (0, 1):
            for prec in (0, 1, 2, 3):
                assert lib.mi_critic_workspace_bytes(4096, 768, critic, est, prec, 1) > 0
                assert lib.mi_critic_host_scratch_bytes(4096, 768, critic, est, prec, 1) > 0
            for world in (1, 2, 8):
                assert lib.mi_sharded_critic_workspace_bytes(4096, world, 768, critic, est, 0) == 0
    assert lib.mi_critic_workspace_bytes(4096, 768, 1, 6, 0, 1) == 0


@pytest.mark.parametrize("est", EST)
def test_mlp_and_sharded_entries_raise_before_any_device_work(pkg, est):
    """CPU tensors: a launch would fail with 'no CPU path'; the estimator check must come first and name the supported set."""
    from mi_b200 import ops
    B, D = 8, 16
    x, y = torch.randn(B, D), torch.randn(B, D)
    sid = torch.arange(B)
    mlp = pkg.FusedMLPCritic(D, (16, 8))
    with pytest.raises(ops.MIError, match="infonce_sym"):
        pkg.select_estimator(est)(mlp(pkg.create_mi_pairs(x, y, sid.tolist(), "cpu")), B)
    with pytest.raises(ops.MIError, match="dv"):
        pkg.sharded_mi_loss(x, y, pkg.FusedCritic(D, "dot"), sid, est)
    with pytest.raises(ops.MIError, match=est):
        ops.sharded_step(x, y, None, sid.to(torch.int32), est, "fast", 1.0)
    with pytest.raises(ops.MIError, match="MLP"):
        ops.mlp_critic_loss_fwd_bwd(x, y, tuple(p.detach() for p in mlp.parameters()), sid, est)
