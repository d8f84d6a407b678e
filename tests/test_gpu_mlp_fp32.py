"""GPU tests (-m gpu) of the MLP critic's fp32 precision ("fp32", MI_PREC_FP32X3): every tensor-core operand as three bf16
pieces (24 significant bits, six K segments) and every accumulation chain bounded (kFp32ChainK K elements; the long
contractions over pairs and rows are cut into split-K partial tiles summed with round-to-nearest).

(a) the reference's golden vectors, (b) the oracle sweep of test_gpu_mlp.SWEEP (plus infonce_sym) next to fp32 PyTorch on
the same inputs (oracle/mlp_oracle.mlp_loss_matrix_form run in float32 on the CPU), (c) the accumulation bias of one panel
of 2^20 coherent pairs, (d) the guard's two-pass repeat, (e) emulated ranks of the batch-sharded step and the adapter.
Each case prints the measured errors of all three modes (pytest -s records them; profiles/r08_mlp_fp32.md).

The sweep bounds.  The operands carry 24 significant bits, but the tensor cores truncate every accumulation, where
PyTorch's fp32 sums round to nearest.  With the six segments accumulated p0 p0 first, the one-signed error of the layer-2
pre-activations flipped ReLU masks that PyTorch's did not: 9.4e-4 max-norm at B = 64 against PyTorch's 7.9e-7.  The
kernels therefore add the segments smallest first (mlp_critic.cuh, piece_segments).  Measured on one B200 (1000 W) with
that order (profiles/r08_pytest_gpu_mlp_fp32.log), the loss and the layer-1 gradients (dX, dY, dW1, db1) of every sweep
row are within 2.8 x PyTorch's error or below 2e-6.  The layer-2 / layer-3 accumulators dW2, db2, dW3 are not:
  - in the single pass (mode 3 with dv / infonce) they are accumulated over the negatives in reference units and the
    positives' -1/B share is added afterwards, a difference of two sums of similar size: up to 9.4 x PyTorch (dW2
    Frobenius 1.5e-4 against 1.6e-5 at B = 256, where strict is at 2.3e-4, so the operand format is not what limits it);
  - dW2 is a contraction over every pair, cut into split-K chains of <= kFp32ChainK K elements, and each chain keeps the
    one-signed truncation residual of its MMAs: at B = 300 (infonce_sym, two-pass sequence) dW2 is off by 2.5e-6 in
    max-norm and in Frobenius alike, a uniform shift, against PyTorch's 5.7e-7 (4.4 x / 7.1 x).
So:
  - SWEEP_RATIO / SWEEP_FLOOR: the loss and dX, dY, dW1, db1 <= max(2.5 x PyTorch, 2e-6) in both norms;
  - LAYER2_RATIO: dW2, db2, dW3 <= max(12 x PyTorch, 2e-6) (worst measured 9.4 x);
  - the single pass's loss, which it forms from fp32 atomic sums of the weights, <= max(2.5 x PyTorch, SINGLE_LOSS = 5e-6)
    (measured <= 1.8e-6).
The recorded run uses at most 0.78 of any of these bounds; strict fails them in 193 of its 272 checks, and the p0 p0-first order failed them by
~300 x at B = 64.  On the shipped-size row the layer-1 gradients must also stay below a quarter of strict's Frobenius error
(measured 1/100 .. 1/125)."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from test_gpu_mlp import GOLDEN, NAMES, SWEEP, _load_case, _loss_rel, _sid_tensor  # noqa: E402
from test_gpu_mlp_sharded import SHAPES, _case, _cross_boundary_dups, emulate_ranks  # noqa: E402

pytestmark = pytest.mark.gpu

GRADS = ("dX", "dY", "dW1", "db1", "dW2", "db2", "dW3")
# golden vectors: loss 1e-6 relative in the two-pass sequence (mode 0); the single pass (mode 3) forms the log-sum-exp from
# fp32 atomic sums of the weights relative to the sampled reference, which left 1.4e-6 .. 2.0e-6 on the first B200 run
# (strict mode's single pass is at the same level), so mode 3 is held to 5e-6.  Gradients: 1e-4 max-norm (measured <= 6.1e-6).
GOLDEN_LOSS = {0: 1e-6, 3: 5e-6}
GOLDEN_GRAD = 1e-4
SWEEP_RATIO, SWEEP_FLOOR = 2.5, 2e-6
LAYER2_RATIO, SINGLE_LOSS = 12.0, 5e-6
BIAS = {"dW2": 2e-6, "dW1": 1e-5}


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as g
    g.build()
    import mi_b200
    from mi_b200 import _lib, ops
    from oracle import matrix_oracle as mo
    from oracle import mlp_oracle
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    assert _lib.load().mi_device_check() == 0, "needs an sm_100 device"
    return mi_b200, ops, mo, mlp_oracle, torch.device("cuda:0")


@pytest.fixture
def mlp_mode(env, request):
    ops = env[1]
    ops.set_mlp_mode(request.param)
    yield request.param
    ops.set_mlp_mode(-1)


def _max(a, ref):
    a, ref = torch.as_tensor(a).detach().cpu().double().reshape(-1), torch.as_tensor(ref).detach().cpu().double().reshape(-1)
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _fro(a, ref):
    a, ref = torch.as_tensor(a).detach().cpu().double().reshape(-1), torch.as_tensor(ref).detach().cpu().double().reshape(-1)
    return float((a - ref).norm() / ref.norm().clamp_min(1e-30))


def _run(ops, X, Y, params, sid, est, precision, dev, panel=None):
    from mi_b200 import _lib
    lib = _lib.load()
    lib.mi_set_mlp_panel_pairs(panel or 0)
    try:
        loss, S, g = ops.mlp_critic_loss_fwd_bwd(X.to(dev).float(), Y.to(dev).float(), tuple(p.to(dev).float() for p in params),
                                                 sid.to(dev), est, precision, need_grads=True, want_scores=True)
        torch.cuda.synchronize()
    finally:
        lib.mi_set_mlp_panel_pairs(0)
    return loss, S, g


@pytest.mark.parametrize("mlp_mode", [3, 0], indirect=True)
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_golden_vectors_fp32(env, path, mlp_mode):
    mi_b200, ops, mo, mlp_oracle, dev = env
    z, X, Y, sid, p = _load_case(mlp_oracle, path)
    est = str(z["estimator"])
    if mlp_mode != 3 and est == "infonce_row":
        pytest.skip("infonce_row always runs the two-pass sequence")
    loss, S, g = _run(ops, X, Y, [p[k] for k in NAMES], _sid_tensor(mo, sid, dev), est, "fp32", dev)
    assert float(loss[7].item()) == 0.0
    errs = {"loss": _loss_rel(loss[0].item(), z["loss"].reshape(-1)[0])}
    for k in NAMES:
        if k == "b3":
            continue
        if "d" + k in z.files:
            errs["d" + k] = _max(g["d" + k], z["d" + k])
        else:
            from oracle.make_golden_mlp import digest_vectors
            gk = g["d" + k].cpu().double()
            r, l = digest_vectors(gk.shape, int(z["seed"]) + 100)
            errs["d" + k] = max(_max(gk @ r, z["d" + k + "_r"]), _max(l @ gk, z["d" + k + "_l"]))
    errs["dX"], errs["dY"] = _max(g["dX"], z["dX"]), _max(g["dY"], z["dY"])
    print(f"\n[golden {os.path.basename(path)} mode {mlp_mode}] " + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))
    assert errs.pop("loss") <= GOLDEN_LOSS[mlp_mode]
    for k, v in errs.items():
        assert v <= GOLDEN_GRAD, (k, v)
    assert abs(float(g["db3"].item()) - float(z["db3"].reshape(-1)[0])) < 1e-5


SWEEP_EST = [(B, D, H1, H2, e, dup, panel) for (B, D, H1, H2, est, dup, panel) in SWEEP for e in dict.fromkeys((est, "infonce_sym"))]


@pytest.mark.parametrize("mlp_mode", [3, 0], indirect=True)
@pytest.mark.parametrize("B,D,H1,H2,est,dup,panel", SWEEP_EST)
def test_sweep_against_fp32_pytorch(env, B, D, H1, H2, est, dup, panel, mlp_mode):
    mi_b200, ops, mo, mlp_oracle, dev = env
    if mlp_mode != 3 and est in ("infonce_row", "infonce_sym"):
        pytest.skip("infonce_row / infonce_sym always run the two-pass sequence")
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=B + D, dup_frac=dup, bilinear=False)
    p = mlp_oracle.init_params(D, H1, H2, seed=H1 + H2)
    p["W2"] = p["W2"] * 2.0
    p["W3"] = p["W3"] * 6.0
    ids = [int(s) for s in sid]
    ref = mlp_oracle.mlp_loss_matrix_form(X.float(), Y.float(), ids, p, est, dtype=torch.float64)
    yard = mlp_oracle.mlp_loss_matrix_form(X.float(), Y.float(), ids, p, est, dtype=torch.float32)
    st = torch.as_tensor(sid).to(torch.int32)
    res = {m: _run(ops, X, Y, [p[k] for k in NAMES], st, est, m, dev, panel) for m in ("fp32", "strict", "fast")}
    err = {}
    for m, (loss, S, g) in list(res.items()) + [("torch32", (None, None, None))]:
        if m == "torch32":
            e = {"loss": _loss_rel(yard["loss"], ref["loss"])}
            e.update({k: (_max(yard[k], ref[k]), _fro(yard[k], ref[k])) for k in GRADS})
        else:
            assert float(loss[7].item()) == 0.0
            e = {"loss": _loss_rel(loss[0].item(), ref["loss"])}
            e.update({k: (_max(g[k], ref[k]), _fro(g[k], ref[k])) for k in GRADS})
        err[m] = e
    print(f"\n[sweep B={B} D={D} H1={H1} H2={H2} {est} mode {mlp_mode}]")
    for m, e in err.items():
        print(f"  {m:8s} loss={e['loss']:.2e} " + " ".join(f"{k}={v[0]:.1e}/{v[1]:.1e}" for k, v in e.items() if k != "loss"))
    y, f = err["torch32"], err["fp32"]
    single = mlp_mode == 3 and est in ("dv", "infonce")           # the other estimators take the two-pass sequence
    loss_bound = max(SWEEP_RATIO * y["loss"], SINGLE_LOSS if single else SWEEP_FLOOR)
    assert f["loss"] <= loss_bound, (f["loss"], y["loss"])
    for k in GRADS:
        ratio = LAYER2_RATIO if k in ("dW2", "db2", "dW3") else SWEEP_RATIO
        for n in (0, 1):
            assert f[k][n] <= max(ratio * y[k][n], SWEEP_FLOOR), (k, n, f[k][n], y[k][n])
    if (B, D, H1, H2) == (256, 128, 1024, 512):
        for k in ("dX", "dY", "dW1", "db1"):
            assert f[k][1] < 0.25 * err["strict"][k][1], (k, f[k][1], err["strict"][k][1])


def test_accumulation_bias_of_a_long_panel(env):
    """dW2 = dZ2^T H over one panel of 2^20 pairs and dW1 over the rows, with coherent signs (post-ReLU activations, positive
    layer-2 / layer-3 weights; the image and text halves of W1 are equal and x_i = y_i, so the positive pairs' activations
    are about twice the negatives' and the two sums of the dv gradient do not cancel): a single tensor-core chain over the
    panel would lose bits to truncation in every MMA of a chain (DESIGN 3.4: ~n 2^-25 relative for n MMAs).  Without the
    fp32-mode bound, choose_ksplit would split this dW2 (one output tile, 49152 K blocks of 128) 74 ways: chains of 665 K
    blocks.  kFp32ChainK = 8192 K elements makes them 64 blocks (768 partial tiles).  Measured on one B200 (1000 W):
    dW2 +1.0e-6 with the six segments p0 p0 first, -3.9e-7 smallest first (the order the kernels use); a build with
    kFp32ChainK = 2048 (3072 partial tiles of 16 blocks) measured the figure recorded in profiles/r08_mlp_fp32.md.  fp32
    PyTorch is at +2.8e-8 (round-to-nearest sums are unbiased), so fp32 mode does not reach PyTorch's bias here.
    dW1 = dA^T X is split 12 ways (4-block chains); its +4.6e-6 (PyTorch: +7.6e-7) comes from dA itself, a sum over the
    text rows of the negatives' share minus the positive's, which amplifies the rounding of both (PyTorch's dW1 bias is 27 x
    its dW2 bias for the same reason).  BIAS holds the measured residuals with a factor 2-5 as a regression bound, and
    PyTorch's value is printed beside them."""
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D, H1, H2 = 1024, 64, 256, 128                        # 2^20 pairs in one panel
    g = torch.Generator().manual_seed(3)
    X = torch.randn(B, D, generator=g)
    Y = X.clone()
    W = torch.randn(H1, D, generator=g) / D ** 0.5
    p = {"W1": torch.cat([W, W], 1), "b1": torch.zeros(H1),
         "W2": torch.rand(H2, H1, generator=g) / H1, "b2": torch.rand(H2, generator=g) * 0.1,
         "W3": torch.rand(1, H2, generator=g) * 0.01, "b3": torch.zeros(1)}
    sid = torch.arange(B, dtype=torch.int32)
    ops.set_mlp_mode(0)                                       # dv through the two-pass sequence: one dW2 contraction
    try:
        loss, _, gr = _run(ops, X, Y, [p[k] for k in NAMES], sid, "dv", "fp32", dev, panel=3 << 19)   # fp32: 2/3 of it
    finally:
        ops.set_mlp_mode(-1)
    ref = mlp_oracle.mlp_loss_matrix_form(X, Y, sid.tolist(), p, "dv", dtype=torch.float64)
    yard = mlp_oracle.mlp_loss_matrix_form(X, Y, sid.tolist(), p, "dv", dtype=torch.float32)

    def bias(a, r):
        r = torch.as_tensor(r).double()
        a = torch.as_tensor(a).detach().cpu().double()
        m = r.abs() > 1e-3 * r.abs().max()
        return float(((a - r)[m] / r[m].abs()).mean())
    for k in ("dW2", "dW1"):
        b, y = bias(gr[k], ref[k]), bias(yard[k], ref[k])
        print(f"\n[bias {k}] fp32 mode {b:+.2e}  torch fp32 {y:+.2e}")
        assert abs(b) <= max(abs(y), BIAS[k]), (k, b, y)


def test_guard_trip_repeats_with_the_two_pass_sequence_fp32(env):
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D, H1, H2 = 512, 32, 64, 32
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=77, dup_frac=0.05, bilinear=False)
    p = mlp_oracle.init_params(D, H1, H2, seed=9)
    p["W3"] = p["W3"].abs() * 4.0
    X = X.clone().float()
    X[3] *= 3000.0                                          # row 3 is not in the sampled reference (stride 2)
    ref = mlp_oracle.mlp_loss_matrix_form(X, Y.float(), [int(s) for s in sid], p, "dv", dtype=torch.float64)
    st = torch.as_tensor(sid).to(torch.int32)
    loss, S, g = _run(ops, X, Y, [p[k] for k in NAMES], st, "dv", "fp32", dev)
    ops.set_mlp_mode(0)
    try:
        loss0, S0, g0 = _run(ops, X, Y, [p[k] for k in NAMES], st, "dv", "fp32", dev)
    finally:
        ops.set_mlp_mode(-1)
    assert float(loss[7].item()) > 0.0 and float(loss0[7].item()) == 0.0
    assert torch.equal(S, S0) and float(loss[0].item()) == float(loss0[0].item())
    for k in GRADS:
        assert _max(g[k], g0[k]) < 1e-5, k
    print("\n[guard fp32] loss %.2e S %.2e " % (_loss_rel(loss[0].item(), ref["loss"]), _max(S, ref["S"]))
          + " ".join(f"{k}={_fro(g[k], ref[k]):.1e}" for k in GRADS))
    assert _loss_rel(loss[0].item(), ref["loss"]) < 1e-5
    assert _max(S, ref["S"]) < 1e-5
    for k in GRADS:
        assert _fro(g[k], ref[k]) < 1e-3, k


@pytest.mark.parametrize("mlp_mode", [3, 0], indirect=True)
@pytest.mark.parametrize("est", ["dv", "infonce", "infonce_row"])
@pytest.mark.parametrize("B,P,D,H1,H2,panel", SHAPES)
def test_emulated_ranks_equal_single_gpu_fp32(env, B, P, D, H1, H2, panel, est, mlp_mode):
    mi_b200, ops, mo, mlp_oracle, dev = env
    from mi_b200 import _lib
    if mlp_mode != 3 and est == "infonce_row":
        pytest.skip("infonce_row always runs the two-pass sequence")
    X, Y, sid, p = _case(mo, mlp_oracle, B, D, H1, H2, seed=B + P)
    sid = _cross_boundary_dups(sid, P)
    params = tuple(p[k].to(dev) for k in NAMES)
    Xd, Yd, sd = X.to(dev), Y.to(dev), sid.to(torch.int32).to(dev)
    lib = _lib.load()
    lib.mi_set_mlp_panel_pairs(panel or 0)
    try:
        ref_loss, _, ref_g = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, params, sd, est, "fp32", need_grads=True)
        loss, g = emulate_ranks(ops, Xd, Yd, params, sd, P, est, "fp32")
        torch.cuda.synchronize()
    finally:
        lib.mi_set_mlp_panel_pairs(0)
    assert float(loss[7]) == 0.0 and float(ref_loss[7]) == 0.0
    assert float(loss[3]) == float(ref_loss[3])
    for k in (0, 1, 2, 4):
        assert _loss_rel(loss[k], ref_loss[k]) < 1e-6, (k, float(loss[k]), float(ref_loss[k]))
    for k in GRADS:
        # the single pass sums the blocks' raw layer-2 / layer-3 accumulators (dW2, db2, dW3: in reference units; the
        # positives' -1/B share cancels most of the negatives') in another order than the one-block call: up to 6.0e-5
        # max-norm measured over three B200 runs
        tol = 1e-4 if (k in ("dW2", "db2", "dW3") and mlp_mode == 3 and est != "infonce_row") else 1e-5
        assert _max(g[k], ref_g[k]) < tol, (k, _max(g[k], ref_g[k]))


def test_adapter_fp32_bit_for_bit(env, monkeypatch):
    """FusedMLPCritic(precision="fp32") in the mi_discriminator slot runs the ops call in fp32 mode and hands its gradients
    to autograd bit for bit.  (Two calls are not bit-identical: the dA / dC reductions use float atomics.)"""
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D = 96, 64
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=17, dup_frac=0.1, bilinear=False)
    torch.manual_seed(4)
    critic = mi_b200.FusedMLPCritic(D, (256, 128), precision="fp32").to(dev)
    seen = []
    real = ops.mlp_critic_loss_fwd_bwd

    def spy(*a, **k):
        out = real(*a, **k)
        seen.append((a[5] if len(a) > 5 else k.get("precision"), out))
        return out
    monkeypatch.setattr(ops, "mlp_critic_loss_fwd_bwd", spy)
    x = X.to(dev).float().requires_grad_(True)
    y = Y.to(dev).float().requires_grad_(True)
    loss = mi_b200.dv_bound_loss(critic(mi_b200.create_mi_pairs(x, y, [int(s) for s in sid], dev)), B)
    loss.sum().backward()
    torch.cuda.synchronize()
    assert len(seen) == 1 and seen[0][0] == "fp32"
    out, _, g = seen[0][1]
    assert torch.equal(x.grad, g["dX"]) and torch.equal(y.grad, g["dY"])
    for t, k in zip(critic.parameters(), ("dW1", "db1", "dW2", "db2", "dW3", "db3")):
        assert torch.equal(t.grad.reshape(-1), g[k].reshape(-1)), k
    monkeypatch.undo()
    # and the sharded adapter at world 1 equals the single-GPU call (block form of the same sequences)
    critic.zero_grad()
    x2 = X.to(dev).float().requires_grad_(True)
    y2 = Y.to(dev).float().requires_grad_(True)
    l2 = mi_b200.sharded_mi_loss(x2, y2, critic, torch.as_tensor(sid).to(torch.int64), "dv")
    l2.sum().backward()
    torch.cuda.synchronize()
    assert _loss_rel(float(l2.detach().sum()), float(loss.detach().sum())) < 1e-6
    assert _max(x2.grad, x.grad) < 1e-5 and _max(y2.grad, y.grad) < 1e-5
