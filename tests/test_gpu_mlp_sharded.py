"""GPU tests (-m gpu) of the batch-sharded concat-MLP critic (DESIGN 8.4): the block stage ops (mi_mlp_block_*,
mi_mlp_input_grad) with the ranks emulated on one device and the exchanges done by hand, the adapter
(sharded_mi_loss with a FusedMLPCritic) at world 1, and the NCCL path on two GPUs.  Every result is held against
mi_mlp_critic_loss_fwd_bwd on the whole batch: logits / loss at 1e-5 relative in strict mode and LOSS_TOL["fast"] in
fast mode; gradients within the MLP bounds of test_gpu_mlp.py (the backward of a ReLU network is not continuous in the
pre-activations, so two computations of the same gradient differ by the same mask flips as either does from fp64)."""
import os
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

LOSS_TOL = {"strict": 1e-5, "fast": 2e-3}
ORACLE_LOSS_TOL = {"strict": 1e-4, "fast": 2e-3}
GRAD_MAX = {"strict": 5e-2, "fast": None}
GRAD_FRO = {"strict": 5e-3, "fast": 0.2}
NAMES = ("W1", "b1", "W2", "b2", "W3", "b3")
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


def _rel(a, ref):
    ref = ref.detach().cpu().double().reshape(-1)
    return float((a.detach().cpu().double().reshape(-1) - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def _fro(a, ref):
    ref = ref.detach().cpu().double().reshape(-1)
    return float((a.detach().cpu().double().reshape(-1) - ref).norm() / ref.norm().clamp_min(1e-30))


def _grad_ok(a, ref, precision):
    if GRAD_MAX[precision] is not None and not _rel(a, ref) < GRAD_MAX[precision]:
        return False
    return _fro(a, ref) < GRAD_FRO[precision]


def _loss_rel(a, ref):
    return abs(float(a) - float(ref)) / max(abs(float(ref)), 1.0)


def _case(mo, mlp_oracle, B, D, H1, H2, seed, dup=0.1):
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=seed, dup_frac=dup, bilinear=False)
    sid = torch.as_tensor(sid).to(torch.int64).clone()
    p = mlp_oracle.init_params(D, H1, H2, seed=seed + 1)
    p["W2"] = p["W2"] * 2.0
    p["W3"] = p["W3"] * 6.0                                  # a softmax that is not flat
    return X.float(), Y.float(), sid, p


def _cross_boundary_dups(sid, P):
    """equal study ids on both sides of every block boundary"""
    Bl = sid.numel() // P
    for r in range(1, P):
        sid[r * Bl] = sid[r * Bl - 1]
    return sid


def emulate_ranks(ops, X, Y, params, sid, P, est, precision, force_two_pass=False):
    """The sharded step of mi_b200.dist with the P ranks' blocks run one after another on this device and the collectives
    done with torch ops.  Returns (loss_out [8], grads dict incl. dX, dY) of the whole batch."""
    B = X.shape[0]
    Bl = B // P
    blk = [slice(r * Bl, (r + 1) * Bl) for r in range(P)]
    single = est != "infonce_row" and (ops.get_mlp_mode() & 1) != 0 and not force_two_pass
    ref = None
    if single:                                                               # all-reduce(MAX) of the own-block samples
        ref = torch.stack([ops.mlp_block_ref_logit(X[b], Y[b], params, 0, precision) for b in blk]).max().reshape(1)
    fw = [ops.mlp_block_fwd(X[b], Y, params, sid[b], sid, b.start, est, precision, ref, not single) for b in blk]
    scal_all = torch.stack([f[0] for f in fw])                               # all-gather of the scalar rows
    loss, merged = ops.mlp_block_merge(scal_all, B, est, not single)
    if single and float(loss[7]) != 0.0:
        loss2, g2 = emulate_ranks(ops, X, Y, params, sid, P, est, precision, force_two_pass=True)
        loss2[7] = 1.0
        return loss2, g2
    bw = [ops.mlp_block_bwd(X[b], Y, params, sid[b], sid, b.start, est, precision, not single, loss, merged, f[1])
          for b, f in zip(blk, fw)]
    dC = torch.stack([g["dC_part"] for g in bw]).sum(0)                      # reduce-scatter of dC
    dY = []
    for b, g in zip(blk, bw):
        dYr, _, _ = ops.mlp_input_grad(dC[b], Y[b], params[0], 1, precision, dW1=g["dW1"])
        dY.append(dYr)
    out = {"dX": torch.cat([g["dX"] for g in bw]), "dY": torch.cat(dY)}
    for n in NAMES:                                                          # all-reduce of the parameter gradients
        out["d" + n] = torch.stack([g["d" + n] for g in bw]).sum(0)
    return loss, out


@pytest.fixture
def mlp_mode(env, request):
    ops = env[1]
    ops.set_mlp_mode(request.param)
    yield request.param
    ops.set_mlp_mode(-1)


SHAPES = [
    # B_global, P, D, H1, H2, panel pairs (None = one panel)
    (128, 1, 32, 128, 64, None),
    (600, 2, 48, 200, 72, None),            # ragged B_global (not a multiple of 256), H1 % 32 != 0
    (256, 4, 64, 256, 128, 6000),           # several panels per block
    (512, 2, 128, 1024, 512, 65536),        # the shipped hidden sizes, two panels per block
]


@pytest.mark.parametrize("mlp_mode", [3, 0], indirect=True)
@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("est", ["dv", "infonce", "infonce_row"])
@pytest.mark.parametrize("B,P,D,H1,H2,panel", SHAPES)
def test_emulated_ranks_equal_single_gpu(env, B, P, D, H1, H2, panel, est, precision, mlp_mode):
    mi_b200, ops, mo, mlp_oracle, dev = env
    from mi_b200 import _lib
    if mlp_mode != 3 and est == "infonce_row":
        pytest.skip("infonce_row always runs the two-pass sequence")
    X, Y, sid, p = _case(mo, mlp_oracle, B, D, H1, H2, seed=B + P)
    sid = _cross_boundary_dups(sid, P)
    params = tuple(p[k].to(dev) for k in NAMES)
    Xd, Yd = X.to(dev), Y.to(dev)
    sd = sid.to(dev)
    lib = _lib.load()
    lib.mi_set_mlp_panel_pairs(panel or 0)
    try:
        ref_loss, _, ref_g = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, params, sd.to(torch.int32), est, precision, need_grads=True)
        loss, g = emulate_ranks(ops, Xd, Yd, params, sd.to(torch.int32), P, est, precision)
        torch.cuda.synchronize()
    finally:
        lib.mi_set_mlp_panel_pairs(0)
    assert float(loss[7]) == 0.0 and float(ref_loss[7]) == 0.0
    assert float(loss[3]) == float(ref_loss[3])                                   # N_neg
    for k in (0, 1, 2, 4):                                                          # loss, pos mean, lse, row loss
        assert _loss_rel(loss[k], ref_loss[k]) < LOSS_TOL[precision], (k, float(loss[k]), float(ref_loss[k]))
    for k in GRADS:
        assert _grad_ok(g[k], ref_g[k], precision), (k, _rel(g[k], ref_g[k]), _fro(g[k], ref_g[k]))
    assert abs(float(g["db3"]) - float(ref_g["db3"])) < 1e-4
    if B <= 256 and mlp_mode == 3:                                                 # and against fp64 on the whole batch
        ref = mlp_oracle.mlp_loss_matrix_form(X, Y, [int(s) for s in sid], p, est, dtype=torch.float64)
        assert _loss_rel(loss[0], ref["loss"]) < ORACLE_LOSS_TOL[precision]
        for k in GRADS:
            assert _grad_ok(g[k], ref[k], precision), k


def _outlier_case(mo, mlp_oracle, B, P, D, H1, H2):
    """One pair (row 3, a text row of the last block) far above every pair inside any single block: layer 1 is shared by
    both sides and the two rows get the same large direction."""
    X, Y, sid, p = _case(mo, mlp_oracle, B, D, H1, H2, seed=31, dup=0.05)
    p["W1"][:, D:] = p["W1"][:, :D]
    p["b1"].zero_()
    p["b2"].zero_()
    p["W3"] = p["W3"].abs()
    g = torch.Generator().manual_seed(5)
    x0 = torch.randn(D, generator=g)
    f1 = float(mlp_oracle.mlp_score_matrix(x0[None].double(), torch.zeros(1, D, dtype=torch.float64),
                                           {k: v.double() for k, v in p.items()})[0, 0] - p["b3"][0])
    j = B - 2
    X[3] = (250.0 / f1) * x0
    Y[j] = (250.0 / f1) * x0
    if sid[j] == sid[3]:
        sid[j] = sid.max() + 1
    return X, Y, sid, p, j


@pytest.mark.parametrize("precision", ["strict", "fast"])
def test_emulated_ranks_guard_trip_takes_the_two_pass_sequence(env, precision):
    mi_b200, ops, mo, mlp_oracle, dev = env
    B, P, D, H1, H2 = 256, 2, 32, 64, 32
    X, Y, sid, p, j = _outlier_case(mo, mlp_oracle, B, P, D, H1, H2)
    S = mlp_oracle.mlp_score_matrix(X.double(), Y.double(), {k: v.double() for k, v in p.items()})
    Bl = B // P
    own = max(float(S[r * Bl:(r + 1) * Bl, r * Bl:(r + 1) * Bl].max()) for r in range(P))
    assert float(S[3, j]) - own > 150.0, "the test input must defeat every block's own sample"
    params = tuple(p[k].to(dev) for k in NAMES)
    Xd, Yd, sd = X.to(dev), Y.to(dev), sid.to(torch.int32).to(dev)
    ops.set_mlp_mode(0)
    try:
        ref_loss, _, ref_g = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, params, sd, "dv", precision, need_grads=True)
    finally:
        ops.set_mlp_mode(-1)
    single = [ops.mlp_block_fwd(Xd[r * Bl:(r + 1) * Bl], Yd, params, sd[r * Bl:(r + 1) * Bl], sd, r * Bl, "dv", precision,
                                torch.stack([ops.mlp_block_ref_logit(Xd[q * Bl:(q + 1) * Bl], Yd[q * Bl:(q + 1) * Bl], params, 0,
                                                                     precision) for q in range(P)]).max().reshape(1),
                                False)[0] for r in range(P)]
    tripped, _ = ops.mlp_block_merge(torch.stack(single), B, "dv", False)
    assert float(tripped[7]) != 0.0                                  # the single pass' merged verdict
    loss, g = emulate_ranks(ops, Xd, Yd, params, sd, P, "dv", precision)
    torch.cuda.synchronize()
    assert float(loss[7]) != 0.0
    for k in (0, 1, 2):
        assert _loss_rel(loss[k], ref_loss[k]) < LOSS_TOL[precision], k
    for k in GRADS:                         # the hidden activations of the outlier pair are large: fast-mode Frobenius bound
        assert _fro(g[k], ref_g[k]) < GRAD_FRO["fast"], k


def test_adapter_world_1(env):
    """sharded_mi_loss with a FusedMLPCritic (no process group): gradients on the embeddings and on all six parameters
    equal those of the single-GPU adapter path dv_bound_loss(critic(create_mi_pairs(...)), B)."""
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
            loss = mi_b200.sharded_mi_loss(x, y, critic, torch.as_tensor(sid).to(torch.int64), "dv")
        else:
            loss = mi_b200.dv_bound_loss(critic(mi_b200.create_mi_pairs(x, y, [int(s) for s in sid], dev)), B)
        loss.sum().backward()
        torch.cuda.synchronize()
        res.append((float(loss.sum()), [x.grad, y.grad] + [t.grad for t in critic.parameters()]))
    assert _loss_rel(res[1][0], res[0][0]) < LOSS_TOL["strict"]
    assert len(res[1][1]) == 8 and all(t is not None for t in res[1][1])
    for a, b in zip(res[1][1][:7], res[0][1][:7]):
        assert _grad_ok(a, b, "strict")
    assert abs(float(res[1][1][7]) - float(res[0][1][7])) < 1e-4          # db3: analytically zero


# ---- NCCL, two GPUs

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, cases, ret):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from mi_b200 import dist as mdist
    from mi_b200 import ops
    from oracle import matrix_oracle as mo
    from oracle import mlp_oracle
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=dev)
    try:
        out = {}
        for est, precision, outlier in cases:
            B, D, H1, H2 = 512, 64, 256, 128
            if outlier:
                X, Y, sid, p, _ = _outlier_case(mo, mlp_oracle, B, world, D, H1, H2)
            else:
                X, Y, sid, p = _case(mo, mlp_oracle, B, D, H1, H2, seed=41)
                sid = _cross_boundary_dups(sid, world)
            params = tuple(p[k].to(dev) for k in NAMES)
            Xd, Yd, sd = X.to(dev), Y.to(dev), sid.to(dev)
            if outlier:
                ops.set_mlp_mode(0)
            try:
                ref_loss, _, ref_g = ops.mlp_critic_loss_fwd_bwd(Xd, Yd, params, sd.to(torch.int32), est, precision)
            finally:
                ops.set_mlp_mode(-1)
            Bl = B // world
            sl = slice(rank * Bl, (rank + 1) * Bl)
            st, dX, dY, grads = mdist.sharded_mlp_critic_loss_fwd_bwd(Xd[sl], Yd[sl], params, sd[sl], est, precision)
            torch.cuda.synchronize()
            errs = {"loss": _loss_rel(st["loss"], ref_loss[0]), "guard": float(st["guard"])}
            ok = {"dX": _grad_ok(dX, ref_g["dX"][sl], precision) if not outlier else _fro(dX, ref_g["dX"][sl]) < 0.2,
                  "dY": _grad_ok(dY, ref_g["dY"][sl], precision) if not outlier else _fro(dY, ref_g["dY"][sl]) < 0.2}
            for n in ("W1", "b1", "W2", "b2", "W3"):
                a, b = grads["d" + n], ref_g["d" + n]
                ok["d" + n] = _grad_ok(a, b, precision) if not outlier else _fro(a, b) < 0.2
            errs["ok"] = ok
            out[(est, precision, outlier)] = errs
        ret[rank] = out
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_mlp_nccl_2gpu_equals_single_gpu(env):
    import torch.multiprocessing as mp
    cases = [(e, pr, o) for pr in ("strict", "fast") for e, o in (("dv", False), ("infonce_row", False), ("dv", True))]
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, _free_port(), cases, ret), nprocs=2, join=True)
    for rank in range(2):
        for (est, precision, outlier), e in ret[rank].items():
            assert e["loss"] < LOSS_TOL[precision], (rank, est, precision, outlier, e)
            assert (e["guard"] != 0.0) == outlier, (rank, est, precision, outlier, e)
            assert all(e["ok"].values()), (rank, est, precision, outlier, e)
