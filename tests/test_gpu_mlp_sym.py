"""GPU tests (-m gpu) of symmetric InfoNCE on the concat-MLP critic (mi_mlp_critic_loss_fwd_bwd and the block stage ops
with MI_EST_INFONCE_SYM).  The reference has no symmetric estimator, so parity is pinned by the fp64 oracle
(oracle/mlp_oracle.py) and by two identities: the symmetric call shares its logits and row loss with infonce_row, and
swapping the two halves of W1 transposes the logit matrix, so the column loss of (X, Y, p) is the row loss of
(Y, X, p').  Tolerances are those of test_gpu_mlp.py (the backward of a ReLU network is not continuous in its
pre-activations) and, between the sharded and single-GPU forms, those of test_gpu_mlp_sharded.py."""
import functools
import os
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_gpu_mlp import GRAD_FRO, GRAD_MAX, LOGIT_TOL, LOSS_TOL, NAMES, SWEEP, _fro, _grad_ok, _loss_rel, _rel  # noqa: E402
from test_gpu_mlp_sharded import LOSS_TOL as SHARD_LOSS_TOL, SHAPES, _case, _cross_boundary_dups  # noqa: E402

pytestmark = pytest.mark.gpu

GRADS = ("dX", "dY", "dW1", "db1", "dW2", "db2", "dW3")


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


def _row_col(S, sid):
    """(loss_row, loss_col) of the symmetric estimator from fp64 logits (R = negatives u diagonal)."""
    from oracle import matrix_oracle as mo
    ids = mo.dense_ids(sid)
    R = mo.negatives_mask(ids, ids) | torch.eye(S.shape[0], dtype=torch.bool)
    Sm = torch.where(R, S, torch.full_like(S, float("-inf")))
    diag = torch.diagonal(S)
    return float((torch.logsumexp(Sm, 1) - diag).mean()), float((torch.logsumexp(Sm, 0) - diag).mean())


@functools.lru_cache(maxsize=None)
def _sweep_case(B, D, H1, H2, dup):
    """the inputs of test_gpu_mlp.test_oracle_parity and the fp64 oracle of infonce_sym on them"""
    from oracle import matrix_oracle as mo
    from oracle import mlp_oracle
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=B + D, dup_frac=dup, bilinear=False)
    p = mlp_oracle.init_params(D, H1, H2, seed=H1 + H2)
    p["W2"] = p["W2"] * 2.0
    p["W3"] = p["W3"] * 6.0                                  # a softmax that is not flat
    sid = [int(s) for s in sid]
    ref = mlp_oracle.mlp_loss_matrix_form(X.float(), Y.float(), sid, p, "infonce_sym", dtype=torch.float64)
    return X.float(), Y.float(), sid, p, ref, _row_col(ref["S"], sid)


SYM_SWEEP = [s[:4] + (s[5], s[6]) for s in SWEEP]           # the shapes of test_gpu_mlp.SWEEP: B, D, H1, H2, dup, panel


@pytest.mark.parametrize("mlp_mode", [3, 0], indirect=True)
@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("B,D,H1,H2,dup,panel", SYM_SWEEP)
def test_oracle_parity_sym(env, B, D, H1, H2, dup, panel, precision, mlp_mode):
    mi_b200, ops, mo, mlp_oracle, dev = env
    from mi_b200 import _lib
    X, Y, sid, p, ref, (ref_row, ref_col) = _sweep_case(B, D, H1, H2, dup)
    params = tuple(p[k].to(dev).float() for k in NAMES)
    lib = _lib.load()
    lib.mi_set_mlp_panel_pairs(panel or 0)
    try:
        loss, S, g = ops.mlp_critic_loss_fwd_bwd(X.to(dev), Y.to(dev), params, torch.as_tensor(sid).to(torch.int32).to(dev),
                                                 "infonce_sym", precision, need_grads=True, want_scores=True)
        loss_f, _, _ = ops.mlp_critic_loss_fwd_bwd(X.to(dev), Y.to(dev), params, torch.as_tensor(sid).to(torch.int32).to(dev),
                                                   "infonce_sym", precision, need_grads=False)
        torch.cuda.synchronize()
    finally:
        lib.mi_set_mlp_panel_pairs(0)
    assert float(loss[7]) == 0.0
    assert float((S.cpu().double() - ref["S"]).abs().max()) < LOGIT_TOL[precision] * max(1.0, float(ref["S"].abs().max()))
    assert _loss_rel(loss[0], ref["loss"]) < LOSS_TOL[precision]
    assert _loss_rel(loss[4], ref_row) < LOSS_TOL[precision]
    assert _loss_rel(loss[5], ref_col) < LOSS_TOL[precision]
    assert float(loss[0]) == 0.5 * (float(loss[4]) + float(loss[5]))
    assert torch.equal(loss_f, loss)                          # forward only: the same kernels up to the loss
    for k in GRADS:
        assert _grad_ok(g[k], ref[k], precision, GRAD_MAX[precision]), (k, _rel(g[k], ref[k]), _fro(g[k], ref[k]))
    assert abs(float(g["db3"])) < 1e-4                        # analytically 0: 1/2 (1 + 1) - 1


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("B,D,H1,H2,dup,panel", [SYM_SWEEP[2], SYM_SWEEP[5]])
def test_sym_shares_logits_and_row_loss_with_infonce_row(env, B, D, H1, H2, dup, panel, precision):
    """Same forward kernels, deterministic: the logits are bit-equal and the symmetric call's loss_row (slot 4) is the
    infonce_row loss bit for bit."""
    mi_b200, ops, mo, mlp_oracle, dev = env
    from mi_b200 import _lib
    X, Y, sid, p, _, _ = _sweep_case(B, D, H1, H2, dup)
    params = tuple(p[k].to(dev).float() for k in NAMES)
    s = torch.as_tensor(sid).to(torch.int32).to(dev)
    lib = _lib.load()
    lib.mi_set_mlp_panel_pairs(panel or 0)
    try:
        ls, Ss, _ = ops.mlp_critic_loss_fwd_bwd(X.to(dev), Y.to(dev), params, s, "infonce_sym", precision, want_scores=True)
        lr, Sr, _ = ops.mlp_critic_loss_fwd_bwd(X.to(dev), Y.to(dev), params, s, "infonce_row", precision, want_scores=True)
        torch.cuda.synchronize()
    finally:
        lib.mi_set_mlp_panel_pairs(0)
    assert torch.equal(Ss, Sr)
    assert float(ls[4]) == float(lr[0]) == float(lr[4])
    assert float(lr[5]) == 0.0


def _swap_w1(p, D):
    q = dict(p)
    q["W1"] = torch.cat((p["W1"][:, D:], p["W1"][:, :D]), 1)
    return q


def _swap_grads(g, D):
    out = dict(g)
    out["dX"], out["dY"] = g["dY"], g["dX"]
    out["dW1"] = torch.cat((g["dW1"][:, D:], g["dW1"][:, :D]), 1)
    return out


@pytest.mark.parametrize("B", [2048])
def test_transposition_identity_at_the_shipped_size(env, B):
    """B = 2048, D = 768, H = 1024 x 512, strict (no CPU oracle is feasible here).  With p' = p with the halves of W1
    swapped: S(Y, X, p') = S(X, Y, p)^T, the symmetric loss and its gradients (dX <-> dY, halves of dW1 swapped) are
    the same, and the symmetric gradient is 1/2 (grad_row(X, Y, p) + swap(grad_row(Y, X, p'))) — G is linear in its
    row and column halves, and the row estimator is validated on its own."""
    mi_b200, ops, mo, mlp_oracle, dev = env
    D, H1, H2 = 768, 1024, 512
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=7, dup_frac=0.05, bilinear=False)
    torch.manual_seed(2)
    critic = mi_b200.FusedMLPCritic(D, (H1, H2))
    p = {k: v.detach().clone() for k, v in zip(NAMES, critic.parameters())}
    p["W3"] = p["W3"] * 4.0
    pt = _swap_w1(p, D)
    dv = lambda q: tuple(q[k].to(dev) for k in NAMES)                 # noqa: E731
    Xd, Yd, s = X.float().to(dev), Y.float().to(dev), torch.as_tensor(sid).to(torch.int32).to(dev)
    l_sym, S, g_sym = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, dv(p), s, "infonce_sym", "strict", want_scores=True)
    l_symt, St, g_symt = ops.mlp_critic_loss_fwd_bwd(Yd, Xd, dv(pt), s, "infonce_sym", "strict", want_scores=True)
    l_row, _, g_row = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, dv(p), s, "infonce_row", "strict")
    l_rowt, _, g_rowt = ops.mlp_critic_loss_fwd_bwd(Yd, Xd, dv(pt), s, "infonce_row", "strict")
    torch.cuda.synchronize()
    assert float((St.t() - S).abs().max()) < LOGIT_TOL["strict"] * max(1.0, float(S.abs().max()))
    assert _loss_rel(l_symt[0], l_sym[0]) < LOSS_TOL["strict"]
    assert _loss_rel(l_symt[4], l_sym[5]) < LOSS_TOL["strict"] and _loss_rel(l_symt[5], l_sym[4]) < LOSS_TOL["strict"]
    assert _loss_rel(l_sym[5], l_rowt[0]) < LOSS_TOL["strict"]
    gs = _swap_grads(g_symt, D)
    gr = _swap_grads(g_rowt, D)
    for k in GRADS:
        assert _grad_ok(gs[k], g_sym[k].cpu(), "strict", GRAD_MAX["strict"]), (k, _rel(gs[k], g_sym[k].cpu()))
        half = 0.5 * (g_row[k] + gr[k])
        assert _grad_ok(g_sym[k], half.cpu(), "strict", GRAD_MAX["strict"]), (k, _rel(g_sym[k], half.cpu()))


def test_adapter_in_the_mi_discriminator_slot(env):
    """FusedMLPCritic + create_mi_pairs + select_estimator("infonce_sym") + backward(): a 0-d loss, gradients in .grad
    of both embeddings and all six parameters, equal to the oracle's."""
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D = 48, 768
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=11, dup_frac=0.1, bilinear=False)
    study_id = [str(50000000 + int(s)) for s in sid]
    torch.manual_seed(3)
    critic = mi_b200.FusedMLPCritic(D, (1024, 512), precision="strict").to(dev)
    p = {k: v.detach().cpu().clone() for k, v in zip(NAMES, critic.parameters())}
    x = X.to(dev).float().requires_grad_(True)
    y = Y.to(dev).float().requires_grad_(True)
    loss = mi_b200.select_estimator("infonce_sym")(critic(mi_b200.create_mi_pairs(x, y, study_id, dev)), B, dev)
    assert tuple(loss.shape) == ()
    loss.backward()
    torch.cuda.synchronize()
    ref = mlp_oracle.mlp_loss_matrix_form(X.float(), Y.float(), study_id, p, "infonce_sym", dtype=torch.float64)
    assert _loss_rel(loss.item(), ref["loss"]) < LOSS_TOL["strict"]
    got = [x.grad, y.grad] + [t.grad for t in critic.parameters()]
    for g, name in zip(got, ("dX", "dY", "dW1", "db1", "dW2", "db2", "dW3")):
        assert g is not None and _grad_ok(g, ref[name], "strict", GRAD_MAX["strict"]), name
    assert got[-1] is not None and abs(float(got[-1])) < 1e-4


def test_no_negatives(env):
    """All-equal study ids: every row and column set is the positive alone, so the loss is 0 and every gradient is 0
    (1/2B (1 + 1) - 1/B on the diagonal); check_negatives=True refuses the batch."""
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D = 40, 32
    X, Y, _, _ = mo.synthetic_embeddings(B, D, seed=5, dup_frac=0.0, bilinear=False)
    torch.manual_seed(1)
    critic = mi_b200.FusedMLPCritic(D, (64, 32)).to(dev)
    x = X.to(dev).float().requires_grad_(True)
    y = Y.to(dev).float().requires_grad_(True)
    loss = mi_b200.select_estimator("infonce_sym")(critic(mi_b200.create_mi_pairs(x, y, ["same"] * B, dev)), B, dev)
    loss.backward()
    torch.cuda.synchronize()
    assert float(loss) == 0.0
    for g in [x.grad, y.grad] + [t.grad for t in critic.parameters()]:
        assert g is not None and float(g.abs().max()) == 0.0
    strict = mi_b200.FusedMLPCritic(D, (64, 32), check_negatives=True).to(dev)
    with pytest.raises(mi_b200.MIError):
        mi_b200.select_estimator("infonce_sym")(strict(mi_b200.create_mi_pairs(x, y, ["same"] * B, dev)), B, dev)


def test_block_ops_refuse_the_single_pass_and_missing_columns(env):
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D = 64, 32
    X, Y, sid, p = _case(mo, mlp_oracle, B, D, 64, 32, seed=3)
    params = tuple(p[k].to(dev) for k in NAMES)
    Xd, Yd, s = X.to(dev), Y.to(dev), sid.to(torch.int32).to(dev)
    ref = torch.zeros(1, device=dev)
    with pytest.raises(ops.MIError):
        ops.mlp_block_fwd(Xd[:32], Yd, params, s[:32], s, 0, "infonce_sym", "strict", ref, False)
    scal, state, col = ops.mlp_block_fwd(Xd[:32], Yd, params, s[:32], s, 0, "infonce_sym", "strict", None, True)
    with pytest.raises(ops.MIError):
        ops.mlp_block_merge(scal.reshape(1, 8), B, "infonce_sym", False)
    loss, merged = ops.mlp_block_merge(scal.reshape(1, 8), B, "infonce_sym", True)
    with pytest.raises(ops.MIError):
        ops.mlp_block_bwd(Xd[:32], Yd, params, s[:32], s, 0, "infonce_sym", "strict", True, loss, merged, state)
    torch.cuda.synchronize()
    assert float(loss[5]) == 0.0 and float(loss[0]) == float(loss[4])         # slots 0 / 5 are the caller's to complete
    assert col.shape == (B,) and bool(torch.isfinite(col[:32]).all())         # the block's own positives are in it


# ---- batch-sharded, ranks emulated on one device

def emulate_ranks_sym(ops, X, Y, params, sid, P, precision):
    """test_gpu_mlp_sharded.emulate_ranks for infonce_sym: the P blocks one after another, the collectives with torch ops,
    plus the all-gather of the column partials and their fp64 merge (what mi_b200.dist does on every rank)."""
    B = X.shape[0]
    Bl = B // P
    blk = [slice(r * Bl, (r + 1) * Bl) for r in range(P)]
    fw = [ops.mlp_block_fwd(X[b], Y, params, sid[b], sid, b.start, "infonce_sym", precision, None, True) for b in blk]
    loss, merged = ops.mlp_block_merge(torch.stack([f[0] for f in fw]), B, "infonce_sym", True)
    c = torch.logsumexp(torch.stack([f[2] for f in fw]).double(), 0)          # all-gather of the column partials
    loss = loss.clone()
    loss[5] = (c.sum() - B * loss[1]) / B
    loss[0] = 0.5 * (loss[4] + loss[5])
    bw = [ops.mlp_block_bwd(X[b], Y, params, sid[b], sid, b.start, "infonce_sym", precision, True, loss, merged, f[1], col_lse=c)
          for b, f in zip(blk, fw)]
    dC = torch.stack([g["dC_part"] for g in bw]).sum(0)                      # reduce-scatter of dC
    dY = [ops.mlp_input_grad(dC[b], Y[b], params[0], 1, precision, dW1=g["dW1"])[0] for b, g in zip(blk, bw)]
    out = {"dX": torch.cat([g["dX"] for g in bw]), "dY": torch.cat(dY)}
    for n in NAMES:                                                          # all-reduce of the parameter gradients
        out["d" + n] = torch.stack([g["d" + n] for g in bw]).sum(0)
    return loss, out


def _shard_grad_ok(a, b, precision):
    return _grad_ok(a, b.detach().cpu(), precision, GRAD_MAX[precision])


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("B,P,D,H1,H2,panel", SHAPES)
def test_emulated_ranks_equal_single_gpu_sym(env, B, P, D, H1, H2, panel, precision):
    mi_b200, ops, mo, mlp_oracle, dev = env
    from mi_b200 import _lib
    X, Y, sid, p = _case(mo, mlp_oracle, B, D, H1, H2, seed=B + P)
    sid = _cross_boundary_dups(sid, P)
    params = tuple(p[k].to(dev) for k in NAMES)
    Xd, Yd, sd = X.to(dev), Y.to(dev), sid.to(torch.int32).to(dev)
    lib = _lib.load()
    lib.mi_set_mlp_panel_pairs(panel or 0)
    try:
        ref_loss, _, ref_g = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, params, sd, "infonce_sym", precision)
        loss, g = emulate_ranks_sym(ops, Xd, Yd, params, sd, P, precision)
        torch.cuda.synchronize()
    finally:
        lib.mi_set_mlp_panel_pairs(0)
    assert float(loss[7]) == 0.0 and float(loss[3]) == float(ref_loss[3])
    for k in (0, 1, 4, 5):                                                          # loss, pos mean, row / column loss
        assert _loss_rel(loss[k], ref_loss[k]) < SHARD_LOSS_TOL[precision], (k, float(loss[k]), float(ref_loss[k]))
    for k in GRADS:
        assert _shard_grad_ok(g[k], ref_g[k], precision), (k, _rel(g[k], ref_g[k].cpu()), _fro(g[k], ref_g[k].cpu()))
    assert abs(float(g["db3"])) < 1e-4
    if B <= 256:                                                                    # and against fp64 on the whole batch
        ref = mlp_oracle.mlp_loss_matrix_form(X, Y, [int(s) for s in sid], p, "infonce_sym", dtype=torch.float64)
        assert _loss_rel(loss[0], ref["loss"]) < LOSS_TOL[precision]
        for k in GRADS:
            assert _grad_ok(g[k], ref[k], precision, GRAD_MAX[precision]), k


def test_sharded_mi_loss_world_1(env):
    """sharded_mi_loss with a FusedMLPCritic and infonce_sym (no process group): a 0-d loss and gradients on the
    embeddings and all six parameters equal to the single-GPU adapter path."""
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, D = 96, 64
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=17, dup_frac=0.1, bilinear=False)
    torch.manual_seed(4)
    critic = mi_b200.FusedMLPCritic(D, (256, 128), precision="strict").to(dev)
    res = []
    for sharded in (False, True):
        critic.zero_grad()
        x = X.to(dev).float().requires_grad_(True)
        y = Y.to(dev).float().requires_grad_(True)
        if sharded:
            loss = mi_b200.sharded_mi_loss(x, y, critic, torch.as_tensor(sid).to(torch.int64), "infonce_sym")
        else:
            loss = mi_b200.select_estimator("infonce_sym")(critic(mi_b200.create_mi_pairs(x, y, [int(s) for s in sid], dev)), B)
        assert tuple(loss.shape) == ()
        loss.backward()
        torch.cuda.synchronize()
        res.append((float(loss), [x.grad, y.grad] + [t.grad for t in critic.parameters()]))
    assert _loss_rel(res[1][0], res[0][0]) < SHARD_LOSS_TOL["strict"]
    assert all(t is not None for t in res[1][1])
    for a, b in zip(res[1][1][:7], res[0][1][:7]):
        assert _shard_grad_ok(a, b, "strict")
    assert abs(float(res[1][1][7])) < 1e-4


# ---- NCCL, two GPUs

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, ret):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from mi_b200 import dist as mdist
    from mi_b200 import ops
    from oracle import matrix_oracle as mo
    from oracle import mlp_oracle
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        out = {}
        for precision in ("strict", "fast"):
            B, D, H1, H2 = 512, 64, 256, 128
            X, Y, sid, p = _case(mo, mlp_oracle, B, D, H1, H2, seed=41)
            sid = _cross_boundary_dups(sid, world)
            params = tuple(p[k].to(dev) for k in NAMES)
            Xd, Yd, sd = X.to(dev), Y.to(dev), sid.to(dev)
            ref_loss, _, ref_g = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, params, sd.to(torch.int32), "infonce_sym", precision)
            Bl = B // world
            sl = slice(rank * Bl, (rank + 1) * Bl)
            st, dX, dY, grads = mdist.sharded_mlp_critic_loss_fwd_bwd(Xd[sl], Yd[sl], params, sd[sl], "infonce_sym", precision)
            torch.cuda.synchronize()
            ok = {"dX": _shard_grad_ok(dX, ref_g["dX"][sl], precision), "dY": _shard_grad_ok(dY, ref_g["dY"][sl], precision)}
            for n in ("W1", "b1", "W2", "b2", "W3"):
                ok["d" + n] = _shard_grad_ok(grads["d" + n], ref_g["d" + n], precision)
            out[precision] = {"loss": _loss_rel(st["loss"], ref_loss[0]), "loss_col": _loss_rel(st["loss_col"], ref_loss[5]),
                              "guard": float(st["guard"]), "ok": ok}
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_mlp_sym_nccl_2gpu_equals_single_gpu(env):
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    for rank in range(2):
        for precision, e in ret[rank].items():
            assert e["loss"] < SHARD_LOSS_TOL[precision] and e["loss_col"] < SHARD_LOSS_TOL[precision], (rank, precision, e)
            assert e["guard"] == 0.0 and all(e["ok"].values()), (rank, precision, e)
