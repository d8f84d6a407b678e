"""GPU tests (-m gpu) of symmetric InfoNCE in the one-call batch-sharded step (csrc/sharded.cuh, DESIGN 5) on ONE device, plus
a two-GPU NCCL test that skips on a one-GPU machine.  Rank r of P owns rows [r Bl, (r+1) Bl) of the batch.

A. The stage ops of the step at real row blocks (q_offset > 0, Bq < Bk): mi_score_stats_rc_ex against the fp64 emulation in
   tests/cpu_backend.py (with the positive pairs folded into the own columns, and with the other ranks' text rows NaN until
   a side stream copies them in and records event_k_ready), and mi_merge_sym_stats against an fp64 merge of the same fp32
   inputs (bit-identical on a second call).
B. The P ranks of the step run one after another on this device through exactly the step's sequence (projection,
   stats_rc_ex with the own diagonal folded in, the packed gather, merge_sym_stats, score_grad with refk = c, the
   reduce-scatter, dW and dX), the collectives done by hand, against the single-GPU symmetric call and the fp64 oracle.
C. ops.sharded_step(..., "infonce_sym") in an NCCL group of world size 1 against the single-GPU symmetric call.
D. dist.sharded_critic_loss_fwd_bwd(..., "infonce_sym") on two GPUs: the one-call path against the op-by-op form and the
   single-GPU call.

Bounds as in tests/test_gpu_sharded_critic.py; every check prints its measured error (run with -s)."""
import json
import math
import os
import socket
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

ORACLE_TOL = {"strict": (1e-4, 1e-3), "fast": (2e-3, 1e-2)}     # loss, gradients vs the fp64 oracle (test_gpu_parity.py)
RAW = {"strict": 1e-4, "fast": 1e-2}     # score_grad, sharded gradients vs the single-GPU call
STAT = 1e-5                              # statistics: |a - b| <= STAT (1 + |b|)
SCAL = 1e-6                              # fp64 scalars, relative
LOSS = 1e-5                              # sharded loss vs the single-GPU call, relative (+ the fp32 resolution term)
SLEEP_CYCLES = 10_000_000                # the delayed copy of the other ranks' text rows: ~5 ms

_MAX = {}


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as g
    g.build()
    import mi_b200  # noqa: F401
    from mi_b200 import _lib, ops, dist as mdist
    from oracle import matrix_oracle as mo
    import cpu_backend as cb
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    assert _lib.load().mi_device_check() == 0, "needs an sm_100 device"
    yield ops, mdist, mo, cb, torch.device("cuda:0")
    if _MAX:
        print("\nmeasured maxima of tests/test_gpu_sharded_sym.py (error / bound):")
        for k in sorted(_MAX):
            print(f"  {k:<44s} {_MAX[k][0]:.3e} / {_MAX[k][1]:.1e}")


class Checks:
    """Records (name, error, bound), prints each and fails at done() with every violation listed."""

    def __init__(self, case):
        self.case, self.bad = case, []

    def __call__(self, name, err, bound):
        err = float(err)
        if math.isnan(err):
            err = math.inf
        _MAX[name] = (max(_MAX.get(name, (0.0,))[0], err), bound)
        print(f"  {self.case} | {name}: {err:.3e} (bound {bound:.1e})")
        if not err <= bound:
            self.bad.append(f"{name}: {err:.3e} > {bound:.1e}")

    def exact(self, name, a, b):
        a, b = _cpu(a).reshape(-1), _cpu(b).reshape(-1)
        self(name, 0.0 if torch.equal(a, b) else float((a - b).abs().nan_to_num(math.inf).max()) or math.inf, 0.0)

    def done(self):
        assert not self.bad, f"{self.case}: " + "; ".join(self.bad)


def _cpu(a):
    return a.detach().cpu().double() if torch.is_tensor(a) else torch.as_tensor(a, dtype=torch.float64)


def stat_err(a, b):
    """max |a - b| / (1 + |b|); equal infinities count as 0, any other non-finite difference as inf"""
    a, b = _cpu(a).reshape(-1), _cpu(b).reshape(-1)
    d = ((a - b).abs() / (1.0 + b.abs())).nan_to_num(math.inf)
    d = torch.where(a == b, torch.zeros_like(d), d)
    return float(d.max()) if d.numel() else 0.0


def rel(a, b):
    """relative max-norm"""
    a, b = _cpu(a).reshape(-1), _cpu(b).reshape(-1)
    return float(((a - b).abs().max() / b.abs().max().clamp_min(1e-300)).nan_to_num(math.inf))


def scal_rel(a, b):
    a, b = _cpu(a).reshape(-1), _cpu(b).reshape(-1)
    d = ((a - b).abs() / b.abs().clamp_min(1e-300)).nan_to_num(math.inf)
    return float(torch.where(a == b, torch.zeros_like(d), d).max())


def _rows(ops, m, b):
    return ops.SplitBF16(m.data[b], m.width) if isinstance(m, ops.SplitBF16) else m[b]


def _batch(mo, Bg, P, D, seed, critic):
    """bf16 embeddings (+ W), int64 study ids with the same study on both sides of every block boundary, one row whose only
    other same-study column lies in the next block, and one study of six rows spread over the batch."""
    bil = critic == "bilinear"
    X, Y, sid, W = mo.synthetic_embeddings(Bg, D, seed=seed, dup_frac=0.05, bilinear=bil)
    sid = sid.clone()
    Bl = Bg // P
    for r in range(1, P):
        sid[r * Bl] = sid[r * Bl - 1]
    if P > 1:
        sid[Bl // 2 + 1] = Bg + 1
        sid[Bl + Bl // 2 + 1] = Bg + 1
    sid[torch.linspace(3, Bg - 5, 6).long()] = Bg + 2
    inv_tau = 1.0 if bil else 1.0 / math.sqrt(D)
    return X.bfloat16(), Y.bfloat16(), sid, (W.bfloat16() if bil else None), inv_tau


def _delayed_k(K, b):
    """K with the rows outside the block b NaN until a side stream, after a ~5 ms sleep, copies them in and records the
    returned event (the all-gather of the other ranks' text embeddings, arriving late)."""
    Kd = torch.full_like(K, float("nan"))
    Kd[b] = K[b]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    ev = torch.cuda.Event()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        Kd[:b.start].copy_(K[:b.start])
        Kd[b.stop:].copy_(K[b.stop:])
        ev.record(side)
    return Kd, ev


def _fold_pos(col, diag, off):
    """the emulation of include_pos: col[off + i] = logaddexp(col[off + i], diag[i])"""
    col = col.double().clone()
    n = diag.numel()
    col[off:off + n] = torch.logaddexp(col[off:off + n], diag.double())
    return col


# ------------------------------------------------------------------ A. stage ops

A_SHAPES = [
    # B_global, P, ranks checked, D
    (1024, 4, (0, 1, 3), 64),      # Bl = 256: own-first schedule; the first / last rank leave one "other" launch empty
    (1536, 2, (0, 1), 136),        # Bl = 3 x 256, D not a multiple of 64
    (600, 3, (0, 2), 72),          # ragged: tiles straddle block boundaries, regular schedule
    (2000, 4, (1, 3), 72),
]
A_IDS = [f"B{s[0]}-P{s[1]}-D{s[3]}" for s in A_SHAPES]


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("critic", ["dot", "bilinear"])
@pytest.mark.parametrize("shape", A_SHAPES, ids=A_IDS)
def test_stats_rc_ex_against_emulation(env, shape, critic, precision):
    """score_stats_rc at a rank's row block: plain, with the positive pairs folded in, and folded with the other ranks'
    text rows arriving late (event_k_ready, k_local_valid: own column block first where the block qualifies)"""
    ops, mdist, mo, cb, dev = env
    Bg, P, ranks, D = shape
    Xb, Yb, sid, Wb, inv_tau = _batch(mo, Bg, P, D, Bg + D, critic)
    Xd, Yd, sd = Xb.to(dev), Yb.to(dev), sid.to(torch.int32).to(dev)
    T = Xd if Wb is None else ops.gemm(Xd, Wb.to(dev), b_t=True, out_dtype=torch.bfloat16, out_split=precision == "strict")
    Tc, Yc = T.float().cpu().double(), Yb.double()
    Bl = Bg // P
    chk = Checks(f"stats_rc_ex {shape[:2]} {critic} {precision}")
    for r in ranks:
        b = slice(r * Bl, (r + 1) * Bl)
        e_rows, e_scal, e_col = cb.score_stats_rc(Tc[b], Yc, sid[b], sid, b.start, inv_tau)
        e_pos = _fold_pos(e_col, e_rows[:, 2], b.start)
        runs = {}
        for mode in ("plain", "pos", "pos_delayed"):
            K, ev = _delayed_k(Yd, b) if mode == "pos_delayed" else (Yd, None)
            runs[mode] = g = ops.score_stats_rc(_rows(ops, T, b), K, sd[b], sd, b.start, inv_tau, event_k_ready=ev,
                                                k_local_valid=ev is not None, include_pos=mode != "plain")
            torch.cuda.synchronize()
            rows, scal, col = g
            t = f"A.stats_rc.{mode}"
            for j in (0, 2, 3):
                chk(f"{t}.rows", stat_err(rows[:, j], e_rows[:, j]), STAT)
            chk.exact(f"{t}.n_neg", rows[:, 1], e_rows[:, 1])
            for j in (0, 4):
                chk(f"{t}.scal", scal_rel(scal[j], e_scal[j]), SCAL)
            # slot 3 = sum of the fp32 positive-pair scores, a sum that cancels: bounded relative to sum |S_ii|
            chk(f"{t}.scal_diag_sum", abs(float(scal[3]) - float(e_scal[3])) / float(e_rows[:, 2].abs().sum()), SCAL)
            chk(f"{t}.scal_lse", stat_err(scal[0] + torch.log(scal[1]), e_scal[0] + torch.log(e_scal[1])), STAT)
            for j in (2, 5, 6, 7):
                chk.exact(f"{t}.scal_counts", scal[j], e_scal[j])
            chk(f"{t}.col", stat_err(col, e_col if mode == "plain" else e_pos), STAT)
        # the fold touches the own columns only, and only through logaddexp with the diagonal
        p, f = runs["plain"][2], runs["pos"][2]
        outside = torch.ones(Bg, dtype=torch.bool)
        outside[b] = False
        chk.exact("A.stats_rc.fold_leaves_other_columns", f[outside.to(dev)], p[outside.to(dev)])
        chk.exact("A.stats_rc.delayed_vs_pos", runs["pos_delayed"][2], f)
    chk.done()


def _merge_fp64(scal, col, Bg):
    """the fp64 merge of the same fp32 inputs: (loss_out [8] as doubles, c fp64 [Bg])"""
    s, c_all = scal.double(), col.double()
    c = torch.logsumexp(c_all, 0)
    m = s[:, 0].max()
    lse = m + torch.log((s[:, 1] * torch.exp(s[:, 0] - m)).nan_to_num(0.0).sum()) if math.isfinite(float(m)) else m
    diag = s[:, 3].sum()
    loss_row, loss_col = s[:, 4].sum() / Bg, (c.sum() - diag) / Bg
    return torch.stack([0.5 * (loss_row + loss_col), diag / Bg, lse, s[:, 2].sum(), loss_row, loss_col, s[:, 5].sum(),
                        torch.zeros((), dtype=torch.float64)]), c


@pytest.mark.parametrize("P", [1, 2, 3, 4, 8])
def test_merge_sym_stats_against_fp64(env, P):
    """scalar rows and column partials of P blocks (columns that are -inf in some blocks; a batch without any negatives):
    c to fp32 rounding, the loss slots to SCAL, slot 7 = 0; a second call gives the same bits"""
    ops, mdist, mo, cb, dev = env
    chk = Checks(f"merge_sym P{P}")
    g = torch.Generator().manual_seed(P)
    Bl = 300
    Bg = Bl * P
    for case in ("mixed", "no_negatives"):
        scal = torch.zeros(P, 8, dtype=torch.float64)
        col = torch.full((P, Bg + 5), -math.inf, dtype=torch.float32)       # a pitch wider than the batch
        diag = (torch.randn(Bg, generator=g) * 2.0).float()
        for r in range(P):
            b = slice(r * Bl, (r + 1) * Bl)
            if case == "mixed":
                lse = 4.0 + torch.rand(1, generator=g).item()
                scal[r] = torch.tensor([lse + 0.5, 1.0 + 40 * torch.rand(1, generator=g).item(), Bl * (Bg - 3.0), float(diag[b].double().sum()),
                                        9.0 * Bl + r, float(r % 2), 0.0, 0.0], dtype=torch.float64)
                part = (3.0 + torch.randn(Bg, generator=g)).float()
                part[torch.rand(Bg, generator=g) < 0.2] = -math.inf                # this block has no negative in column j
                col[r, :Bg] = part
            else:
                scal[r] = torch.tensor([-math.inf, 0.0, 0.0, float(diag[b].double().sum()), 0.0, float(Bl), 0.0, 0.0],
                                       dtype=torch.float64)
            hi = torch.maximum(col[r, b], diag[b])
            col[r, b] = hi + torch.log1p(torch.exp(torch.minimum(col[r, b], diag[b]) - hi))   # the own positive pairs
        want, c_ref = _merge_fp64(scal, col[:, :Bg], Bg)
        got = [ops.merge_sym_stats(scal.to(dev), col.to(dev), Bg) for _ in range(2)]
        torch.cuda.synchronize()
        lo = torch.stack([got[0][k] for k in ("loss", "pos_mean", "lse_neg", "n_neg", "loss_row", "loss_col",
                                              "rows_without_negatives", "guard")]).cpu()
        t = f"A.merge_sym.{case}"
        chk(f"{t}.c_ulps", float(((_cpu(got[0]["c"]) - c_ref).abs() / (c_ref.abs() * 2.0 ** -23 + 1e-30)).max()), 1.0)
        for j in (0, 1, 4, 5):
            chk(f"{t}.loss_slots", abs(float(lo[j]) - float(want[j])) / max(abs(float(want[j])), 1.0), SCAL)
        if case == "mixed":
            chk(f"{t}.lse_neg", scal_rel(lo[2], want[2]), SCAL)
        else:
            assert float(lo[2]) == -math.inf and abs(float(lo[5])) < 1e-12, lo     # c_j = S_jj: the column loss is 0
        for j in (3, 6, 7):
            chk.exact(f"{t}.counts", lo[j], want[j])
        chk.exact(f"{t}.repeat_c", got[1]["c"], got[0]["c"])
        chk.exact(f"{t}.repeat_loss", torch.stack([got[1][k] for k in ("loss", "loss_row", "loss_col")]),
                  torch.stack([got[0][k] for k in ("loss", "loss_row", "loss_col")]))
    chk.done()


# ------------------------------------------------------------------ B. ranks emulated on one device

def emulate_sym_step(ops, Xb, Yb, Wb, sid, P, precision, inv_tau, delayed_k=True):
    """csrc/sharded.cuh's symmetric branch with the P ranks run one after another on this device; collectives by hand
    (all-gather = cat / stack, reduce-scatter = sum + slice, all-reduce of dW = sum).  Returns (merge dict, dX, dY, dW)."""
    Bg, D = Xb.shape
    Bl = Bg // P
    blk = [slice(r * Bl, (r + 1) * Bl) for r in range(P)]
    bilinear, strict = Wb is not None, precision == "strict"
    sid = sid.to(torch.int32).contiguous()
    T = [ops.gemm(Xb[b], Wb, b_t=True, out_dtype=torch.bfloat16, out_split=strict) if bilinear else Xb[b] for b in blk]
    Y_all = torch.cat([Yb[b] for b in blk])                                       # all-gather of the text embeddings
    stats = []
    for r, b in enumerate(blk):
        K, ev = _delayed_k(Y_all, b) if (delayed_k and P > 1) else (Y_all, None)
        stats.append(ops.score_stats_rc(T[r], K, sid[b], sid, b.start, inv_tau, event_k_ready=ev, k_local_valid=ev is not None,
                                        include_pos=True))
    # the packed all-gather: every rank receives every record {scalars | column partials}
    out = ops.merge_sym_stats(torch.stack([s[1] for s in stats]), torch.stack([s[2] for s in stats]), Bg)
    w = 0.5 / Bg
    dX, dWs, parts = [], [], []
    for r, b in enumerate(blk):
        dT32, dT16, part = ops.score_grad(T[r], Y_all, sid[b], sid, b.start, inv_tau, refq=stats[r][0][:, 3].contiguous(), wq=w,
                                          refk=out["c"], wk=w, include_diag=True, precision=precision, alpha=inv_tau,
                                          gamma=1.0 / Bg, want_f32=not bilinear, want_bf16=bilinear,
                                          out_split=bilinear and strict, want_k=True)
        parts.append(part)
        if bilinear:
            dWs.append(ops.gemm(Xb[b], dT16, a_t=True, b_t=True))
            dX.append(ops.gemm(dT16, Wb))
        else:
            dX.append(dT32)
    dY_all = torch.stack(parts).sum(0)
    return out, torch.cat(dX), torch.cat([dY_all[b] for b in blk]), (sum(dWs) if bilinear else None)


def _loss_close(a, b, pos, lse, rel_tol):
    """|a - b| / bound: relative error plus the fp32 resolution of the terms the loss is a difference of"""
    return abs(float(a) - float(b)) / (rel_tol * abs(float(b)) + 1e-6 * (abs(float(pos)) + abs(float(lse))))


def _compare(chk, got, full, ref, precision, bilinear):
    out, dX, dY, dW = got
    lo, fX, fY, fW = full
    raw = RAW[precision]
    for j, k in ((0, "loss"), (4, "loss_row"), (5, "loss_col")):
        chk(f"B.vs_single_gpu.{k}", _loss_close(out[k], lo[j], lo[1], lo[j] + lo[1], LOSS), 1.0)
    chk.exact("B.vs_single_gpu.n_neg", out["n_neg"], lo[3])
    chk.exact("B.guard", out["guard"], 0.0)
    names = ("dX", "dY", "dW") if bilinear else ("dX", "dY")
    for k, a, f in zip(names, (dX, dY, dW), (fX, fY, fW)):
        chk(f"B.vs_single_gpu.{k}.{precision}", rel(a, f), raw)
    if ref is not None:
        lt, gt = ORACLE_TOL[precision]
        chk(f"B.vs_oracle.loss.{precision}",
            abs(float(out["loss"]) - float(ref["loss"])) / (lt * abs(float(ref["loss"])) + 1e-6 * (abs(float(ref["pos_mean"])) + abs(float(ref["loss"] + ref["pos_mean"])))), 1.0)
        for k, a in zip(names, (dX, dY, dW)):
            chk(f"B.vs_oracle.{k}.{precision}", rel(a, ref[k]), gt)


B_SHAPES = [
    # B_global, P, D
    (1024, 1, 64),
    (600, 2, 72),
    (600, 3, 72),
    (1536, 2, 136),
    (1024, 4, 64),
    (2000, 4, 72),
    (2048, 8, 64),
]


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("critic", ["dot", "bilinear"])
@pytest.mark.parametrize("Bg,P,D", B_SHAPES, ids=[f"B{b}-P{p}-D{d}" for b, p, d in B_SHAPES])
def test_emulated_sym_step_equals_single_gpu_and_oracle(env, Bg, P, D, critic, precision):
    ops, mdist, mo, cb, dev = env
    Xb, Yb, sid, Wb, inv_tau = _batch(mo, Bg, P, D, Bg + 7 * P, critic)
    Xd, Yd, Wd, sd = Xb.to(dev), Yb.to(dev), None if Wb is None else Wb.to(dev), sid.to(torch.int32).to(dev)
    chk = Checks(f"sym ranks B{Bg} P{P} D{D} {critic} {precision}")
    got = emulate_sym_step(ops, Xd, Yd, Wd, sd, P, precision, inv_tau)
    full = ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd, "infonce_sym", precision, inv_tau, True)
    torch.cuda.synchronize()
    ref = mo.critic_loss(Xb.float(), Yb.float(), sid, None if Wb is None else Wb.float(), inv_tau, "infonce_sym")
    _compare(chk, got, full, ref, precision, Wb is not None)
    chk.done()


def test_emulated_sym_step_multi_panel(env):
    """Bl = 20480 rows per rank at D = 64: more than one dS row panel per block; against the single-GPU call and the chunked
    oracle on the device"""
    ops, mdist, mo, cb, dev = env
    from oracle import chunked_oracle as co
    Bg, P, D = 40960, 2, 64
    assert Bg // P > torch.cuda.get_device_properties(0).multi_processor_count * 128, "the block must span several panels"
    Xb, Yb, sid, _, inv_tau = _batch(mo, Bg, P, D, 17, "dot")
    Xd, Yd, sd = Xb.to(dev), Yb.to(dev), sid.to(dev)
    chk = Checks(f"sym ranks multi-panel B{Bg} P{P}")
    ref = co.critic_loss_chunked(Xd.float(), Yd.float(), sd, None, inv_tau, "infonce_sym", chunk=4096)
    for precision in ("strict", "fast"):
        got = emulate_sym_step(ops, Xd, Yd, None, sd.to(torch.int32), P, precision, inv_tau)
        full = ops.critic_loss_fwd_bwd(Xd, Yd, None, sd.to(torch.int32), "infonce_sym", precision, inv_tau, True)
        torch.cuda.synchronize()
        _compare(chk, got, full, ref, precision, False)
        del got, full
    chk.done()


# ------------------------------------------------------------------ C. the one-call step at world 1

def _world1_worker(rank, store_path, out_path):
    import torch.distributed as tdist
    sys.path.insert(0, ROOT)
    import mi_b200  # noqa: F401
    from mi_b200 import ops
    from oracle import matrix_oracle as mo
    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    tdist.init_process_group("nccl", store=tdist.FileStore(store_path, 1), rank=0, world_size=1, device_id=dev)
    res = {}
    try:
        for Bg, D in ((600, 72), (1024, 64)):
            for critic in ("dot", "bilinear"):
                Xb, Yb, sid, Wb, inv_tau = _batch(mo, Bg, 1, D, Bg + D + 1, critic)
                Xd, Yd, Wd, sd = Xb.to(dev), Yb.to(dev), None if Wb is None else Wb.to(dev), sid.to(torch.int32).to(dev)
                for prec in ("strict", "fast"):
                    fl, fX, fY, fW = ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd, "infonce_sym", prec, inv_tau, True)
                    for cg in (True, False):
                        st, lo, dX, dY, dW = ops.sharded_step(Xd, Yd, Wd, sd, "infonce_sym", prec, inv_tau, check_guard=cg)
                        torch.cuda.synchronize()
                        res[f"B{Bg}-D{D}/{critic}/{prec}/check{int(cg)}"] = {
                            "status": int(st), "guard": float(lo[7]), "n_neg": [float(lo[3]), float(fl[3])],
                            "half_sum": abs(float(lo[0]) - 0.5 * (float(lo[4]) + float(lo[5]))),
                            "loss": _loss_close(lo[0], fl[0], fl[1], fl[0] + fl[1], LOSS),
                            "loss_row": _loss_close(lo[4], fl[4], fl[1], fl[4] + fl[1], LOSS),
                            "loss_col": _loss_close(lo[5], fl[5], fl[1], fl[5] + fl[1], LOSS),
                            "dX": rel(dX, fX), "dY": rel(dY, fY), "dW": None if Wd is None else rel(dW, fW)}
    finally:
        tdist.destroy_process_group()
    with open(out_path, "w") as f:
        json.dump(res, f)


def test_one_call_sym_step_world1(env, tmp_path):
    """ops.sharded_step(..., "infonce_sym") in an NCCL group of world size 1 == the single-GPU symmetric call: status 0 with
    and without check_guard, loss_out[7] = 0, slot 0 = (slot 4 + slot 5) / 2"""
    ops, mdist, mo, cb, dev = env
    import torch.multiprocessing as mp
    out = tmp_path / "world1.json"
    mp.spawn(_world1_worker, args=(str(tmp_path / "filestore"), str(out)), nprocs=1, join=True)
    res = json.loads(out.read_text())
    chk = Checks("sharded_step sym world 1")
    assert len(res) == 2 * 2 * 2 * 2
    for name, r in sorted(res.items()):
        print(f"  {name}: {r}")
        prec = name.split("/")[2]
        assert r["status"] == 0 and r["guard"] == 0.0 and r["n_neg"][0] == r["n_neg"][1], (name, r)
        chk("C.sharded_step.half_sum", r["half_sum"], 1e-12)
        for k in ("loss", "loss_row", "loss_col"):
            chk(f"C.sharded_step.{k}", r[k], 1.0)
        for k in ("dX", "dY", "dW"):
            if r[k] is not None:
                chk(f"C.sharded_step.{k}.{prec}", r[k], RAW[prec])
    chk.done()


# ------------------------------------------------------------------ D. two GPUs

def _nccl_worker(rank, world, port, ret):
    import torch.distributed as tdist
    sys.path.insert(0, ROOT)
    import mi_b200  # noqa: F401
    from mi_b200 import dist as mdist, ops
    from oracle import matrix_oracle as mo
    torch.cuda.set_device(rank)
    dev = torch.device(f"cuda:{rank}")
    tdist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world, device_id=dev)
    try:
        errs = {}
        B, D = 8192, 256
        Bl = B // world
        sl = slice(rank * Bl, (rank + 1) * Bl)
        for critic in ("dot", "bilinear"):
            Xb, Yb, sid, Wb, inv_tau = _batch(mo, B, world, D, 29, critic)
            Wd = None if Wb is None else Wb.to(dev)
            sd = sid.to(torch.int32).to(dev)
            for prec in ("strict", "fast"):
                full = ops.critic_loss_fwd_bwd(Xb.to(dev), Yb.to(dev), Wd, sd, "infonce_sym", prec, inv_tau, True)
                res = {}
                for impl in ("c", "python"):
                    os.environ["MI_SHARDED_IMPL"] = impl
                    res[impl] = mdist.sharded_critic_loss_fwd_bwd(Xb[sl].to(dev), Yb[sl].to(dev), Wd, sd[sl], "infonce_sym", prec,
                                                                  inv_tau, True)
                torch.cuda.synchronize()
                (oc, cX, cY, cW), (op, pX, pY, pW) = res["c"], res["python"]
                assert set(op) <= set(oc), (sorted(op), sorted(oc))
                e = {"status_guard": float(oc["guard"])}
                for k in ("loss", "loss_row", "loss_col", "pos_mean", "lse_neg"):
                    e[f"{k}_vs_python"] = scal_rel(oc[k], op[k])
                for j, k in ((0, "loss"), (4, "loss_row"), (5, "loss_col")):
                    e[f"{k}_vs_single"] = scal_rel(oc[k], full[0][j])
                e["n_neg_equal"] = float(oc["n_neg"]) == float(full[0][3])
                for k, a, p, f in (("dX", cX, pX, full[1][sl]), ("dY", cY, pY, full[2][sl]), ("dW", cW, pW, full[3])):
                    if a is not None:
                        e[f"{k}_vs_python"], e[f"{k}_vs_single"] = rel(a, p), rel(a, f)
                errs[f"{critic}/{prec}"] = e
        os.environ.pop("MI_SHARDED_IMPL", None)
        ret[rank] = errs
    finally:
        tdist.destroy_process_group()


def test_sharded_sym_one_call_nccl_2gpu_equals_python_and_single_gpu(env):
    """dist.sharded_critic_loss_fwd_bwd(..., "infonce_sym") on REAL NCCL (2 ranks, one per GPU): the one-call step against
    the op-by-op form (MI_SHARDED_IMPL=python) and the single-GPU call.  Skipped on a one-GPU machine."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
    assert len(ret) == 2
    for rank in range(2):
        for case, e in ret[rank].items():
            prec = case.split("/")[1]
            raw = RAW[prec]
            assert e["status_guard"] == 0.0 and e["n_neg_equal"], (rank, case, e)
            assert all(v < LOSS for k, v in e.items() if k.startswith(("loss", "pos_mean", "lse_neg"))), (rank, case, e)
            assert all(v < raw for k, v in e.items() if k.startswith(("dX", "dY", "dW"))), (rank, case, e)
