"""CPU checks of symmetric InfoNCE on the concat-MLP critic: the batch-sharded step
(mi_b200.dist.sharded_mlp_critic_loss_fwd_bwd, "infonce_sym") under gloo with the fp64 emulation of the block stage ops
(tests/cpu_backend_mlp_sym.py) against the fp64 oracle on the whole batch, the oracle's transposition identity, and the
host-side checks of the new entry points."""
import os
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_host_mlp_sharded_cpu import B_GLOBAL, D, H1, H2, _study_ids, make_case  # noqa: E402

TOL = 1e-10


@pytest.fixture(scope="module", autouse=True)
def built():
    import __graft_entry__ as g
    g.build()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _row_col_losses(S, sid):
    """loss_row, loss_col of the symmetric estimator from the fp64 logits (R = negatives u diagonal)."""
    from oracle import matrix_oracle as mo
    ids = mo.dense_ids(sid)
    R = mo.negatives_mask(ids, ids) | torch.eye(S.shape[0], dtype=torch.bool)
    Sm = torch.where(R, S, torch.full_like(S, float("-inf")))
    diag = torch.diagonal(S)
    return float((torch.logsumexp(Sm, 1) - diag).mean()), float((torch.logsumexp(Sm, 0) - diag).mean())


def _worker(rank, world, port, ret, int32_ids, need_grads):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpu_backend_mlp_sym
    from mi_b200 import dist as mdist
    from oracle import mlp_oracle
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        X, Y, p = make_case()
        sid = _study_ids()
        sid_t = torch.tensor(sid, dtype=torch.int32) if int32_ids else torch.tensor(sid, dtype=torch.int64) * 1000003 + 17
        Bl = B_GLOBAL // world
        sl = slice(rank * Bl, (rank + 1) * Bl)
        params = tuple(p[k] for k in mlp_oracle.PARAM_NAMES)
        out, dX, dY, grads = mdist.sharded_mlp_critic_loss_fwd_bwd(X[sl], Y[sl], params, sid_t[sl], "infonce_sym", "strict",
                                                                   need_grads, None, backend=cpu_backend_mlp_sym)
        ref = mlp_oracle.mlp_loss_matrix_form(X, Y, sid, p, "infonce_sym")
        ref_row, ref_col = _row_col_losses(ref["S"], sid)
        res = {"loss": float(out["loss"]), "loss_row": float(out["loss_row"]), "loss_col": float(out["loss_col"]),
               "guard": float(out["guard"]), "ref_loss": float(ref["loss"]), "ref_row": ref_row, "ref_col": ref_col,
               "grads": dX is not None}
        if dX is not None:
            rel = lambda a, b: float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-300))
            res["errs"] = {"dX": rel(dX, ref["dX"][sl]), "dY": rel(dY, ref["dY"][sl])}
            for n in ("W1", "b1", "W2", "b2", "W3"):
                res["errs"]["d" + n] = rel(grads["d" + n].reshape(ref["d" + n].shape), ref["d" + n])
            res["db3"] = float(grads["db3"].double().reshape(-1)[0])
        ret[rank] = res
    finally:
        dist.destroy_process_group()


def _run(world, int32_ids, need_grads=True):
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), ret, int32_ids, need_grads), nprocs=world, join=True)
    assert len(ret) == world
    res = [ret[r] for r in range(world)]
    for k in ("loss", "loss_row", "loss_col"):
        assert len({r[k] for r in res}) == 1, (k, [r[k] for r in res])       # bit-identical on every rank
    for r in res:
        assert r["guard"] == 0.0
        for got, want in (("loss", "ref_loss"), ("loss_row", "ref_row"), ("loss_col", "ref_col")):
            assert abs(r[got] - r[want]) <= TOL * max(1.0, abs(r[want])), (got, r)
    return res


@pytest.mark.parametrize("int32_ids", [True, False], ids=["int32_ids", "int64_ids"])
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_mlp_sym_gloo_equals_full_batch_oracle(world, int32_ids):
    for r in _run(world, int32_ids):
        assert r["grads"]
        assert max(r["errs"].values()) < TOL, r["errs"]
        assert abs(r["db3"]) < TOL                     # sum of dL/dlogit over all pairs: 1/2 (1 + 1) - 1 = 0


def test_sharded_mlp_sym_gloo_forward_only():
    for r in _run(2, True, need_grads=False):
        assert not r["grads"]


def _swap_halves(t, D):
    return torch.cat((t[:, D:], t[:, :D]), 1)


def test_oracle_transposition_identity():
    """S(Y, X, p') = S(X, Y, p)^T with the halves of W1 swapped (p'); the symmetric loss is the same, dX <-> dY and the
    halves of dW1 swap, the other parameter gradients are unchanged."""
    from oracle import mlp_oracle
    X, Y, p = make_case(seed=5)
    sid = _study_ids()
    pt = dict(p)
    pt["W1"] = _swap_halves(p["W1"], D)
    a = mlp_oracle.mlp_loss_matrix_form(X, Y, sid, p, "infonce_sym")
    b = mlp_oracle.mlp_loss_matrix_form(Y, X, sid, pt, "infonce_sym")
    close = lambda u, v: float((u - v).abs().max()) <= 1e-12 * max(1.0, float(v.abs().max()))
    assert close(b["S"], a["S"].t())
    assert abs(float(b["loss"]) - float(a["loss"])) <= 1e-12
    assert close(b["dX"], a["dY"]) and close(b["dY"], a["dX"])
    assert close(b["dW1"], _swap_halves(a["dW1"], D))
    for k in ("db1", "dW2", "db2", "dW3", "db3"):
        assert close(b[k], a[k]), k


def test_mlp_sym_workspace_planning_on_the_host():
    from mi_b200 import _lib
    lib = _lib.load()
    for prec in (0, 1):
        for B in (256, 300, 4096, 8192):
            assert lib.mi_mlp_critic_workspace_bytes(B, 768, 1024, 512, prec) > 0
        assert lib.mi_mlp_critic_workspace_bytes(256, 770, 1024, 512, prec) == 0        # D % 8 != 0
        assert lib.mi_mlp_critic_workspace_bytes(256, 768, 1024, 520, prec) == 0        # H2 > 512
        assert lib.mi_mlp_critic_workspace_bytes(0, 768, 1024, 512, prec) == 0
        for Bq, Bk in ((512, 4096), (1024, 8192), (300, 600)):
            assert lib.mi_mlp_block_workspace_bytes(Bq, Bk, 768, 1024, 512, prec) > 0
            assert lib.mi_mlp_block_state_bytes(Bq, Bk, 768, 1024, 512, prec) >= 4 * Bq * Bk
        assert lib.mi_mlp_block_workspace_bytes(600, 512, 768, 1024, 512, prec) == 0
        assert lib.mi_mlp_block_state_bytes(512, 4096, 770, 1024, 512, prec) == 0


def test_mlp_sym_ops_refuse_cpu_tensors_and_unknown_estimators():
    from mi_b200 import ops
    X, Y, p = make_case()
    params = tuple(p[k].float() for k in ("W1", "b1", "W2", "b2", "W3", "b3"))
    sid = torch.tensor(_study_ids(), dtype=torch.int32)
    with pytest.raises(ops.MIError):
        ops.mlp_critic_loss_fwd_bwd(X.float(), Y.float(), params, sid, "infonce_sym")
    with pytest.raises(ops.MIError):
        ops.mlp_block_fwd(X[:12].float(), Y.float(), params, sid[:12], sid, 0, "infonce_sym", "strict", None, True)
    with pytest.raises(ops.MIError):
        ops.mlp_block_bwd(X[:12].float(), Y.float(), params, sid[:12], sid, 0, "infonce_sym", "strict", True,
                          torch.zeros(8, dtype=torch.float64), torch.zeros(8, dtype=torch.float64), torch.zeros(16, dtype=torch.uint8),
                          col_lse=torch.zeros(B_GLOBAL))
    with pytest.raises(ops.MIError):
        ops._mlp_estimator("infonce_col")
    from mi_b200 import dist as mdist
    with pytest.raises(ValueError):
        mdist.sharded_mlp_critic_loss_fwd_bwd(X.float(), Y.float(), params, sid, "infonce_col")
