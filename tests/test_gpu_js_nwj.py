"""GPU tests (-m gpu) of the Jensen-Shannon and NWJ estimators on the single-GPU separable critics, against the fp64 oracle
(oracle/fdiv_oracle.py) on bf16-rounded inputs.  Tolerances as the other parity tests: strict loss 1e-4 relative (plus the
fp32-resolution term of _loss_ok), gradients 1e-3 relative max-norm; fast 2e-3 / 1e-2."""
import ctypes
import math
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

TOL = {"strict": (1e-4, 1e-3), "fast": (2e-3, 1e-2)}
EST = ("js", "nwj")


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as g
    g.build()
    import mi_b200
    from mi_b200 import _lib, ops
    from oracle import fdiv_oracle as fo
    from oracle import matrix_oracle as mo
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    assert _lib.load().mi_device_check() == 0, "needs an sm_100 device"
    return mi_b200, ops, fo, mo, torch.device("cuda:0")


def _rel(a, ref):
    return float((a.detach().cpu().double() - ref.detach().cpu().double()).abs().max()
                 / ref.detach().cpu().double().abs().max().clamp_min(1e-30))


def _loss_ok(a, ref, rel):
    loss, pos = float(ref["loss"]), float(ref["pos_mean"])
    bound = rel * abs(loss) + 1e-6 * (abs(pos) + abs(loss + pos))
    err = abs(float(a) - loss)
    assert err <= bound, f"loss {float(a)!r} vs oracle {loss!r}: |err| {err:.3e} > {bound:.3e}"


def _grads_ok(ref, gt, dX, dY, dW=None):
    assert _rel(dX, ref["dX"]) < gt, ("dX", _rel(dX, ref["dX"]))
    assert _rel(dY, ref["dY"]) < gt, ("dY", _rel(dY, ref["dY"]))
    if dW is not None:
        assert _rel(dW, ref["dW"]) < gt, ("dW", _rel(dW, ref["dW"]))


def _inputs(mo, B, D, critic, dup, seed):
    X, Y, sid, W = mo.synthetic_embeddings(B, D, seed=seed, dup_frac=dup, bilinear=(critic == "bilinear"))
    Xb, Yb = X.bfloat16().float(), Y.bfloat16().float()
    Wb = None if W is None else W.bfloat16().float()
    return Xb, Yb, sid, Wb, (1.0 / math.sqrt(D) if critic == "dot" else 1.0)


def _adapter(mi_b200, dev, X, Y, W, study_id, inv_tau, est, precision, check_negatives=False):
    B, D = X.shape
    x = X.to(dev).float().requires_grad_(True)
    y = Y.to(dev).float().requires_grad_(True)
    critic = mi_b200.FusedCritic(D, "dot" if W is None else "bilinear", temperature=1.0 / inv_tau, precision=precision,
                                 check_negatives=check_negatives).to(dev)
    if W is not None:
        with torch.no_grad():
            critic.W.copy_(W.to(dev).float())
    loss = mi_b200.select_estimator(est)(critic(mi_b200.create_mi_pairs(x, y, study_id, dev)), B, dev)
    loss.backward()
    torch.cuda.synchronize()
    return loss, x.grad, y.grad, (None if W is None else critic.W.grad)


SWEEP = [
    (32, 768, "dot", 0.0), (33, 8, "dot", 0.3), (129, 72, "bilinear", 0.1), (257, 136, "bilinear", 0.05),
    (600, 1024, "dot", 0.2), (1024, 768, "bilinear", 0.05), (2048, 1024, "bilinear", 0.0), (2048, 136, "dot", 0.3),
]


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("est", EST)
@pytest.mark.parametrize("B,D,critic,dup", SWEEP)
def test_oracle_sweep(env, B, D, critic, dup, est, precision):
    mi_b200, ops, fo, mo, dev = env
    Xb, Yb, sid, Wb, inv_tau = _inputs(mo, B, D, critic, dup, B + D)
    ref = fo.critic_loss(Xb, Yb, sid, Wb, inv_tau, est)
    loss, dX, dY, dW = _adapter(mi_b200, dev, Xb, Yb, Wb, [int(s) for s in sid], inv_tau, est, precision)
    assert loss.dim() == 0
    lt, gt = TOL[precision]
    _loss_ok(loss.item(), ref, lt)
    _grads_ok(ref, gt, dX, dY, dW)


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("est", EST)
def test_baseline_config2(env, est, precision):
    """BASELINE config 2: B = 4096, D = 768, bilinear; also the loss_out slots, forward-only and TWO_PASS."""
    mi_b200, ops, fo, mo, dev = env
    Xb, Yb, sid, Wb, _ = _inputs(mo, 4096, 768, "bilinear", 0.05, 11)
    ref = fo.critic_loss(Xb, Yb, sid, Wb, 1.0, est)
    X, Y, W, s = Xb.to(dev), Yb.to(dev), Wb.to(dev), sid.to(dev)
    out, dX, dY, dW = ops.critic_loss_fwd_bwd(X, Y, W, s, est, precision, 1.0, True)
    lt, gt = TOL[precision]
    o = out.cpu()
    _loss_ok(o[0], ref, lt)
    _grads_ok(ref, gt, dX, dY, dW)
    assert float(o[3]) == float(ref["n_neg"]) and float(o[6]) == 0.0 and float(o[5]) == 0.0
    assert abs(float(o[1]) - float(ref["pos_mean"])) <= 1e-5 * max(1.0, abs(float(ref["pos_mean"])))
    if est == "js":
        assert float(o[7]) == 0.0
        assert abs(float(o[2]) - float(ref["sp_neg"])) <= lt * float(ref["sp_neg"])
        assert abs(float(o[4]) - float(ref["sp_pos"])) <= lt * float(ref["sp_pos"]) + 1e-6
    else:
        assert abs(float(o[2]) - float(ref["lse_neg"])) <= 1e-5 * abs(float(ref["lse_neg"])) + 1e-5
        assert float(o[4]) == 0.0
    fwd, _, _, _ = ops.critic_loss_fwd_bwd(X, Y, W, s, est, precision, 1.0, False)
    _loss_ok(fwd.cpu()[0], ref, lt)
    assert abs(float(fwd.cpu()[0]) - float(o[0])) <= 1e-6 * abs(float(o[0])) + 1e-7
    tp, tX, tY, tW = ops.critic_loss_fwd_bwd(X, Y, W, s, est, precision, 1.0, True, two_pass=True)
    _loss_ok(tp.cpu()[0], ref, lt)
    _grads_ok(ref, gt, tX, tY, tW)


FULL = [("js", "fast"), ("js", "strict"), ("nwj", "fast")]


@pytest.mark.parametrize("est,precision", FULL)
def test_full_size(env, est, precision):
    """B = 65536, D = 1024, bilinear: every element of dX, dY, dW against the chunked oracle on the device, and the identities
    <dT,T> = <dY,Y> = <dW,W> (= <G,S>)."""
    mi_b200, ops, fo, mo, dev = env
    B, D = 65536, 1024
    X, Y, sid, W = mo.synthetic_embeddings(B, D, seed=5, dup_frac=0.02, device=dev)
    Xb, Yb, Wb = X.bfloat16(), Y.bfloat16(), W.bfloat16()
    out, dX, dY, dW = ops.critic_loss_fwd_bwd(Xb, Yb, Wb, sid, est, precision, 1.0, True)
    torch.cuda.synchronize()
    T = (Xb.float() @ Wb.float())
    ref = fo.critic_loss_chunked(Xb.float(), Yb.float(), sid, Wb.float(), 1.0, est, chunk=4096, T=T)
    lt, gt = TOL[precision]
    o = out.cpu()
    _loss_ok(o[0], ref, lt)
    assert _rel(dX, ref["dX"]) < gt and _rel(dY, ref["dY"]) < gt and _rel(dW, ref["dW"]) < gt
    a = float((ref["dT"].double() * T.double()).sum())               # <G, S> of the oracle
    b = float((dY.double() * Yb.double()).sum())
    c = float((dW.double() * Wb.double()).sum())
    slack = gt * abs(a) + 1e-6 * float(dY.double().norm() * Yb.double().norm())
    assert abs(b - a) <= slack and abs(c - a) <= slack, (a, b, c)


def test_hostile_scales(env):
    """Scores x 8 (JS saturates sigma), unnormalised embeddings, and an NWJ row whose true log-sum-exp lies far beyond its
    sampled reference (guard trips, the exact repeat gives the oracle's result).  NWJ's true gradient stays in fp32 range."""
    mi_b200, ops, fo, mo, dev = env
    ops.set_ref_sample_columns(128)
    try:
        for B, D, critic, scale in ((2048, 64, "dot", 8.0), (1024, 72, "bilinear", 3.0)):
            Xb, Yb, sid, Wb, inv_tau = _inputs(mo, B, D, critic, 0.1, 17)
            Xs = (Xb * scale).bfloat16().float()
            for est in EST:
                for precision in ("strict", "fast"):
                    ref = fo.critic_loss(Xs, Yb, sid, Wb, inv_tau, est)
                    out, dX, dY, dW = ops.critic_loss_fwd_bwd(Xs.to(dev), Yb.to(dev), None if Wb is None else Wb.to(dev),
                                                              sid.to(dev), est, precision, inv_tau, True)
                    lt, gt = TOL[precision]
                    _loss_ok(out.cpu()[0], ref, lt)
                    _grads_ok(ref, gt, dX, dY, dW)
                    if est == "js":
                        assert float(out.cpu()[7]) == 0.0
        # planted NWJ outlier: scores around -100, one unsampled pair near +30
        B, D = 2048, 64
        X = torch.zeros(B, D); Y = torch.zeros(B, D)
        X[:, 0] = 10.0; Y[:, 0] = -10.0
        X[:, 1] = torch.linspace(-1, 1, B); Y[:, 1] = torch.linspace(1, -1, B)
        X[5, 2] = 13.0; Y[1001, 2] = 10.0                           # S[5, 1001] = -100 + ... + 130
        X, Y = X.bfloat16().float(), Y.bfloat16().float()
        sid = torch.arange(B)
        for precision in ("strict", "fast"):
            ref = fo.critic_loss(X, Y, sid, None, 1.0, "nwj")
            out, dX, dY, _ = ops.critic_loss_fwd_bwd(X.to(dev), Y.to(dev), None, sid.to(dev), "nwj", precision, 1.0, True)
            o = out.cpu()
            assert float(o[7]) > 0.0, "the planted outlier must trip the sampled guard"
            lt, gt = TOL[precision]
            _loss_ok(o[0], ref, lt)
            _grads_ok(ref, gt, dX, dY)
            assert torch.isfinite(dX).all() and torch.isfinite(dY).all()
    finally:
        ops.set_ref_sample_columns(2048)


@pytest.mark.parametrize("est", EST)
def test_host_entries_equal_device_call(env, est):
    mi_b200, ops, fo, mo, dev = env
    from mi_b200 import _lib
    lib = _lib.load()
    B, D = 3000, 256
    Xb, Yb, sid, Wb, _ = _inputs(mo, B, D, "bilinear", 0.05, 23)
    sh = sid.to(torch.int32).contiguous()
    ref, rX, rY, rW = ops.critic_loss_fwd_bwd(Xb.to(dev), Yb.to(dev), Wb.to(dev), sh.to(dev), est, "fast", 1.0, True)
    torch.cuda.synchronize()
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    nbytes = lib.mi_critic_host_scratch_bytes(B, D, 1, ops.ESTIMATOR[est], 0, 1)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    Xh, Yh, Wh = Xb.contiguous().pin_memory(), Yb.contiguous().pin_memory(), Wb.contiguous().pin_memory()
    loss = torch.zeros(8, dtype=torch.float64)
    hX, hY, hW = torch.zeros(B, D), torch.zeros(B, D), torch.zeros(D, D)
    st = lib.mi_critic_loss_fwd_bwd_host(p(Xh), p(Yh), p(Wh), p(sh), B, D, 1, ops.ESTIMATOR[est], 0, 1.0, p(loss), p(hX), p(hY),
                                         p(hW), p(scratch), nbytes, None)
    assert st == 0
    assert float(loss[0]) == float(ref.cpu()[0])
    assert torch.equal(hX, rX.cpu()) and torch.equal(hY, rY.cpu()) and torch.equal(hW, rW.cpu())
    for host_dtype, src in ((1, (Xb.bfloat16(), Yb.bfloat16(), Wb.bfloat16())), (0, (Xb, Yb, Wb))):
        xs = [t.contiguous().pin_memory() for t in src]
        gX, gY, gW = (torch.zeros(B, D, device=dev), torch.zeros(B, D, device=dev), torch.zeros(D, D, device=dev))
        loss2 = torch.zeros(8, dtype=torch.float64)
        st = lib.mi_critic_loss_fwd_bwd_from_host(p(xs[0]), p(xs[1]), p(xs[2]), p(sh), host_dtype, B, D, 1, ops.ESTIMATOR[est], 0,
                                                  1.0, p(loss2), p(gX), p(gY), p(gW), p(scratch), nbytes, None)
        assert st == 0
        torch.cuda.synchronize()
        assert float(loss2[0]) == float(ref.cpu()[0])
        assert torch.equal(gX, rX) and torch.equal(gY, rY) and torch.equal(gW, rW)


@pytest.mark.parametrize("est", EST)
def test_graphed_step_replays_bit_for_bit(env, est):
    mi_b200, ops, fo, mo, dev = env
    B, D = 1024, 256
    Xb, Yb, sid, Wb, _ = _inputs(mo, B, D, "bilinear", 0.05, 29)
    X, Y, W, s = Xb.to(dev).bfloat16(), Yb.to(dev).bfloat16(), Wb.to(dev).bfloat16(), sid.to(torch.int32).to(dev)
    ref, rX, rY, rW = ops.critic_loss_fwd_bwd(X, Y, W, s, est, "strict", 1.0, True)
    ref, rX, rY, rW = ref.clone(), rX.clone(), rY.clone(), rW.clone()
    step = ops.GraphedCriticStep(B, D, True, est, "strict", 1.0, device=dev)
    for _ in range(2):
        out, dX, dY, dW = step(X, Y, W, s)
        torch.cuda.synchronize()
        assert torch.equal(out, ref) and torch.equal(dX, rX) and torch.equal(dY, rY) and torch.equal(dW, rW)


@pytest.mark.parametrize("est", EST)
def test_no_negatives(env, est):
    mi_b200, ops, fo, mo, dev = env
    B, D = 64, 32
    Xb, Yb, _, Wb, _ = _inputs(mo, B, D, "bilinear", 0.0, 31)
    same = [7] * B
    loss, _, _, _ = _adapter(mi_b200, dev, Xb, Yb, Wb, same, 1.0, est, "strict")
    assert math.isnan(float(loss))
    with pytest.raises(ops.MIError):
        _adapter(mi_b200, dev, Xb, Yb, Wb, same, 1.0, est, "strict", check_negatives=True)


@pytest.mark.parametrize("code", [4, 5])
def test_mlp_entries_reject_the_codes(env, code):
    mi_b200, ops, fo, mo, dev = env
    from mi_b200 import _lib
    lib = _lib.load()
    B, D, H1, H2 = 64, 16, 32, 16
    f = lambda *s: torch.randn(*s, device=dev)
    X, Y, W1, b1, W2, b2, W3, b3 = f(B, D), f(B, D), f(H1, 2 * D), f(H1), f(H2, H1), f(H2), f(1, H2), f(1)
    sid = torch.arange(B, dtype=torch.int32, device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    loss = torch.zeros(8, dtype=torch.float64, device=dev)
    nb = lib.mi_mlp_critic_workspace_bytes(B, D, H1, H2, 0)
    ws = torch.empty(max(nb, 256), dtype=torch.uint8, device=dev)
    st = lib.mi_mlp_critic_loss_fwd_bwd(p(X), p(Y), p(W1), p(b1), p(W2), p(b2), p(W3), p(b3), p(sid), B, D, H1, H2, code, 0,
                                        p(loss), None, None, None, None, None, None, None, None, None, p(ws), ws.numel(), None)
    assert st == -1
    nbb = lib.mi_mlp_block_workspace_bytes(B, B, D, H1, H2, 0)
    nst = lib.mi_mlp_block_state_bytes(B, B, D, H1, H2, 0)
    wsb = torch.empty(max(nbb, 256), dtype=torch.uint8, device=dev)
    state = torch.empty(max(nst, 256), dtype=torch.uint8, device=dev)
    scal = torch.zeros(8, dtype=torch.float64, device=dev)
    st = lib.mi_mlp_block_fwd(p(X), p(Y), p(W1), p(b1), p(W2), p(b2), p(W3), p(b3), p(sid), p(sid), B, B, 0, D, H1, H2, code, 0,
                              None, 1, p(scal), p(state), state.numel(), p(wsb), wsb.numel(), None)
    assert st == -1
    torch.cuda.synchronize()
