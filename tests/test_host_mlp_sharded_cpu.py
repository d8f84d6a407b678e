"""CPU checks of the batch-sharded concat-MLP critic (mi_b200.dist.sharded_mlp_critic_loss_fwd_bwd, DESIGN 8.4):
the collective logic under gloo with an fp64 emulation of the block stage ops (tests/cpu_backend_mlp.py) against the fp64
oracle on the whole batch, and the host-side workspace planning of the block stage ops."""
import os
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B_GLOBAL, D, H1, H2 = 24, 16, 64, 32
OUTLIER_ROW, OUTLIER_COL = 3, 17          # different row blocks at world 2 and 4


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


def _study_ids():
    """Equal ids on both sides of every row-block boundary at world 2 and 4 (5|6, 11|12, 17|18), and one id shared by
    rows of different blocks (0 and 20)."""
    sid = list(range(100, 100 + B_GLOBAL))
    for a, b in ((5, 6), (11, 12), (17, 18), (0, 20)):
        sid[b] = sid[a]
    return sid


def make_case(outlier=False, seed=11):
    """fp64 embeddings and make_mlp(2D, [H1, H2]) parameters.  ``outlier``: image row OUTLIER_ROW and text row
    OUTLIER_COL get the same large direction and layer 1 is shared by both sides, so the logit of that one pair sits far
    above every pair inside any single row block — a sample of a rank's own block cannot see it."""
    from oracle import mlp_oracle
    g = torch.Generator().manual_seed(seed)
    X = torch.randn(B_GLOBAL, D, generator=g, dtype=torch.float64) * 0.5
    Y = X + 0.3 * torch.randn(B_GLOBAL, D, generator=g, dtype=torch.float64)
    p = {k: v.double() for k, v in mlp_oracle.init_params(D, H1, H2, seed).items()}
    if outlier:
        p["W1"][:, D:] = p["W1"][:, :D]
        p["b1"].zero_()
        p["b2"].zero_()
        p["W3"] = p["W3"].abs()
        x0 = torch.randn(D, generator=g, dtype=torch.float64)
        f1 = float(mlp_oracle.mlp_score_matrix(x0[None], torch.zeros(1, D, dtype=torch.float64), p)[0, 0] - p["b3"][0])
        scale = 250.0 / f1                # homogeneous without biases: the pair sits ~250 above a row / column alone
        X[OUTLIER_ROW] = scale * x0
        Y[OUTLIER_COL] = scale * x0
    return X, Y, p


def _worker(rank, world, port, est, ret, outlier, int32_ids, need_grads):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import cpu_backend_mlp
    from mi_b200 import dist as mdist
    from oracle import mlp_oracle
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        X, Y, p = make_case(outlier)
        sid = _study_ids()
        sid_t = torch.tensor(sid, dtype=torch.int32) if int32_ids else torch.tensor(sid, dtype=torch.int64) * 1000003 + 17
        Bl = B_GLOBAL // world
        sl = slice(rank * Bl, (rank + 1) * Bl)
        params = tuple(p[k] for k in mlp_oracle.PARAM_NAMES)
        out, dX, dY, grads = mdist.sharded_mlp_critic_loss_fwd_bwd(X[sl], Y[sl], params, sid_t[sl], est, "strict",
                                                                   need_grads, None, backend=cpu_backend_mlp)
        ref = mlp_oracle.mlp_loss_matrix_form(X, Y, sid, p, est)
        res = {"loss": float(out["loss"]), "guard": float(out["guard"]), "n_neg": float(out["n_neg"]),
               "ref_loss": float(ref["loss"]), "ref_n_neg": float(ref["n_neg"]), "grads": dX is not None}
        if dX is not None:
            rel = lambda a, b: float((a.double() - b).abs().max() / b.abs().max().clamp_min(1e-300))
            res["errs"] = {"dX": rel(dX, ref["dX"][sl]), "dY": rel(dY, ref["dY"][sl])}
            for n in ("W1", "b1", "W2", "b2", "W3"):
                res["errs"]["d" + n] = rel(grads["d" + n].reshape(ref["d" + n].shape), ref["d" + n])
            # db3 = sum of dL/dlogit over all pairs is analytically 0: compared on the scale of its terms (the -1/B sum)
            res["errs"]["db3"] = float((grads["db3"].double().reshape(-1) - ref["db3"].reshape(-1)).abs().max())
        ret[rank] = res
    finally:
        dist.destroy_process_group()


def _run(world, est, outlier=False, int32_ids=False, need_grads=True):
    import torch.multiprocessing as mp
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), est, ret, outlier, int32_ids, need_grads), nprocs=world, join=True)
    assert len(ret) == world
    res = [ret[r] for r in range(world)]
    assert len({r["loss"] for r in res}) == 1, [r["loss"] for r in res]       # bit-identical on every rank
    tol = 1e-6 if est == "dv" else 1e-10        # dv: the reference's log N_neg is an fp32 value (mi_critics.py:10)
    for r in res:
        assert abs(r["loss"] - r["ref_loss"]) <= tol * max(1.0, abs(r["ref_loss"])), r
        assert r["n_neg"] == r["ref_n_neg"]
    return res


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("est", ["dv", "infonce", "infonce_row"])
def test_sharded_mlp_gloo_equals_full_batch_oracle(world, est):
    for r in _run(world, est, int32_ids=(world == 4)):
        assert r["grads"] and r["guard"] == 0.0
        assert max(r["errs"].values()) < 1e-10, r["errs"]


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_mlp_gloo_guard_trip_repeats_with_two_pass(world):
    """The outlier pair is outside every rank's own block: the global weight sum overflows, every rank repeats the step
    with the two-pass sequence, reports the trip, and still equals the oracle."""
    X, Y, p = make_case(outlier=True)
    from oracle import mlp_oracle
    S = mlp_oracle.mlp_score_matrix(X, Y, p)
    Bl = B_GLOBAL // world
    assert OUTLIER_ROW // Bl != OUTLIER_COL // Bl
    blocks = [S[r * Bl:(r + 1) * Bl, r * Bl:(r + 1) * Bl].max() for r in range(world)]
    assert float(S[OUTLIER_ROW, OUTLIER_COL] - max(blocks)) > 150.0          # far beyond the 69 ln 2 margin
    for r in _run(world, "dv", outlier=True):
        assert r["guard"] != 0.0
        assert max(r["errs"].values()) < 1e-10, r["errs"]


def test_sharded_mlp_gloo_forward_only():
    for r in _run(2, "dv", need_grads=False):
        assert not r["grads"]


def test_mlp_block_workspace_planning_on_the_host():
    from mi_b200 import _lib
    lib = _lib.load()
    for prec in (0, 1):
        for Bq, Bk in ((512, 4096), (1024, 8192), (300, 600), (256, 256)):
            assert lib.mi_mlp_block_workspace_bytes(Bq, Bk, 768, 1024, 512, prec) > 0
            assert lib.mi_mlp_block_state_bytes(Bq, Bk, 768, 1024, 512, prec) >= 4 * Bq * Bk
        assert lib.mi_mlp_input_grad_workspace_bytes(512, 768, 1024, prec) > 0
        assert lib.mi_mlp_block_workspace_bytes(512, 4096, 768, 1024, 520, prec) == 0      # H2 > 512
        assert lib.mi_mlp_block_workspace_bytes(512, 4096, 770, 1024, 512, prec) == 0      # D % 8 != 0
        assert lib.mi_mlp_block_state_bytes(512, 4096, 770, 1024, 512, prec) == 0
        assert lib.mi_mlp_block_workspace_bytes(600, 512, 768, 1024, 512, prec) == 0       # more image rows than text rows
        assert lib.mi_mlp_input_grad_workspace_bytes(512, 770, 1024, prec) == 0


def test_mlp_block_ops_refuse_cpu_tensors():
    from mi_b200 import ops
    X, Y, p = make_case()
    params = tuple(p[k].float() for k in ("W1", "b1", "W2", "b2", "W3", "b3"))
    with pytest.raises(ops.MIError):
        ops.mlp_block_ref_logit(X.float(), Y.float(), params, 0)
    with pytest.raises(ops.MIError):
        ops.mlp_input_grad(torch.zeros(4, H1), X[:4].float(), params[0], 1)
