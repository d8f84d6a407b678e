"""GPU tests (-m gpu) of the batch-sharded separable critic (dot / bilinear score matrix with DV or InfoNCE, DESIGN 5) on
ONE device.  Rank r of P owns rows [r Bl, (r+1) Bl) of the batch; a rank's stage ops work on its row block (q_offset > 0,
Bq < Bk), which the single-GPU call never exercises.

A. Every stage op that mi_b200.dist and csrc/sharded.cuh use, at real row blocks, against its fp64 emulation in
   tests/cpu_backend.py on the same bf16-rounded inputs (strict bilinear: the CPU side gets the path's own hi/lo T).  Every
   reference input (ref, lam, diag, refq, refk) is passed to both sides, so each op is checked on its own.  The single pass
   also runs with "delayed K": the other ranks' text rows are NaN until a side stream copies them in after a sleep and
   records event_k_ready — a tile scored before the library waits for that event would read NaN.
B. The P ranks of the step run one after another on this device through the stage-op sequence of mi_b200.dist, the
   collectives done by hand (all-gather = cat / stack, all-reduce MAX, reduce-scatter = sum + slice), against the
   single-GPU call on the whole batch and the fp64 oracle.
C. The one-call step (mi_sharded_critic_loss_fwd_bwd, csrc/sharded.cuh) in an NCCL process group of world size 1: its
   collectives become device copies, everything else (mask pre-pass on the auxiliary stream, lambda event, finalisation
   kernels) runs as on P GPUs.
D. The fp32 -> bf16 cast every fp32 input goes through (ops.as_bf16): bit-equal to round-to-nearest-even.

Bounds: statistics (log-sum-exps, scores) |a - b| <= 1e-5 (1 + |b|); fp64 scalars 1e-6 relative, counts exact; raw
contractions and score_grad 1e-4 (strict) / 1e-2 (fast) relative max-norm — the bounds of the two-GPU NCCL test; fp32
finalisation / gemm output 1e-5, bf16 output one bf16 ulp, hi/lo output 2^-16.  Every check prints its measured error; the
maxima are printed when the module ends (run with -s)."""
import json
import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

ORACLE_TOL = {"strict": (1e-4, 1e-3), "fast": (2e-3, 1e-2)}     # loss, gradients vs the fp64 oracle (test_gpu_parity.py)
RAW = {"strict": 1e-4, "fast": 1e-2}     # raw contractions, score_grad, sharded gradients vs the single-GPU call
STAT = 1e-5                              # statistics: |a - b| <= STAT (1 + |b|)
SCAL = 1e-6                              # fp64 scalars, relative
FIN = 1e-5                               # fp32 output of the finalisation kernels and of gemm, relative max-norm
SPLIT = 2.0 ** -16                       # hi/lo output, relative max-norm
LOSS = 1e-5                              # sharded loss vs the single-GPU call, relative (+ the fp32 resolution term)
SLEEP_CYCLES = 10_000_000                # the delayed copy of the other ranks' text rows: ~5 ms
PATHS = [("dv", False), ("infonce", False), ("infonce_row", False),             # (estimator, exact references)
         ("dv", True), ("infonce", True), ("infonce_row", True), ("infonce_sym", True)]

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
        print("\nmeasured maxima of tests/test_gpu_sharded_critic.py (error / bound):")
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


def ulp_err(a16, b):
    """max |a - b| / (ulp_bf16(b) + FIN max|b|): <= 1 is "within one bf16 ulp" (the second term: fp32 arithmetic near 0)"""
    a, b = _cpu(a16).reshape(-1), _cpu(b).reshape(-1)
    ulp = torch.exp2(torch.floor(torch.log2(b.abs().clamp_min(1e-38))) - 7)
    return float(((a - b).abs() / (ulp + FIN * b.abs().max())).nan_to_num(math.inf).max())


def _mat_f64(ops, m):
    """CPU fp64 value of a plain bf16 or hi/lo (hi + lo) operand"""
    return m.float().cpu().double()


def _rows(ops, m, b):
    return ops.SplitBF16(m.data[b], m.width) if isinstance(m, ops.SplitBF16) else m[b]


def _batch(mo, Bg, P, D, seed, critic):
    """bf16 embeddings (+ W), int64 study ids with the same study on both sides of every block boundary, one row whose only
    other same-study column lies in the next block, and one study of six rows spread over the batch (more than the four
    same-study columns the mask lists per row)."""
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


# ------------------------------------------------------------------ A. stage ops against the fp64 emulation

A_SHAPES = [
    # B_global, P, ranks checked, D
    (1024, 4, (0, 1, 3), 64),      # Bl = 256: own-first schedule; the first / last rank leave one "other" launch empty
    (1536, 2, (0, 1), 136),        # Bl = 3 x 256, D not a multiple of 64
    (600, 3, (0, 2), 72),          # ragged: tiles straddle block boundaries, regular schedule
    (2000, 4, (1, 3), 72),
]
A_IDS = [f"B{s[0]}-P{s[1]}-D{s[3]}" for s in A_SHAPES]
_STAGE = {}


def _stage_case(env, shape, critic, precision):
    """inputs of one (shape, critic, precision) and the exact statistics of the whole batch (fp64, from the path's own T)"""
    key = (shape, critic, precision)
    if key not in _STAGE:
        _STAGE.clear()
        ops, mdist, mo, cb, dev = env
        Bg, P, ranks, D = shape
        Xb, Yb, sid, Wb, inv_tau = _batch(mo, Bg, P, D, Bg + D, critic)
        Xd, Yd = Xb.to(dev), Yb.to(dev)
        T = Xd if Wb is None else ops.gemm(Xd, Wb.to(dev), b_t=True, out_dtype=torch.bfloat16, out_split=precision == "strict")
        Tc, Yc = _mat_f64(ops, T), Yb.double()
        S = (Tc @ Yc.t()) * inv_tau
        M = sid[:, None] != sid[None, :]
        R = M | torch.eye(Bg, dtype=torch.bool)
        ninf = torch.full_like(S, -math.inf)
        _STAGE[key] = dict(Bg=Bg, P=P, Bl=Bg // P, ranks=ranks, D=D, inv_tau=inv_tau, T=T, Tc=Tc, Yd=Yd, Yc=Yc, sid=sid,
                           sid_d=sid.to(torch.int32).to(dev),
                           lse_neg=torch.logsumexp(torch.where(M, S, ninf).reshape(-1), 0),
                           row_all=torch.logsumexp(torch.where(R, S, ninf), 1), col_all=torch.logsumexp(torch.where(R, S, ninf), 0))
    return _STAGE[key]


def _a_params(f):
    f = pytest.mark.parametrize("precision", ["strict", "fast"])(f)
    f = pytest.mark.parametrize("critic", ["dot", "bilinear"])(f)
    return pytest.mark.parametrize("shape", A_SHAPES, ids=A_IDS)(f)


@_a_params
def test_score_ref_sample_against_emulation(env, shape, critic, precision):
    """stride 1 and > 1, a column block selected by col0 / n_cols, subset 0 / 1 (the 48-nat margin at stride 1), with and
    without the positive pair; also the call of mi_b200.dist (the rank's own rows as K, q_offset 0)."""
    ops, mdist, mo, cb, dev = env
    c = _stage_case(env, shape, critic, precision)
    chk = Checks(f"ref_sample {shape[:2]} {critic} {precision}")
    Bl, Bg = c["Bl"], c["Bg"]
    for r in c["ranks"]:
        b = slice(r * Bl, (r + 1) * Bl)
        Q, Qc = _rows(ops, c["T"], b), c["Tc"][b]
        own = (c["Yd"][b], c["Yc"][b], c["sid_d"][b], c["sid"][b], 0)
        full = (c["Yd"], c["Yc"], c["sid_d"], c["sid"], b.start)
        forms = [(full, 0, Bg, 1, 0), (full, 0, Bg, 3, 0), (full, b.start, Bl, 1, 1), (full, b.start, Bl, 4, 0),
                 (full, b.start, Bl, 4, 1), (own, 0, Bl, 1, 1)]
        for incl in (False, True):
            for (Kd, Kc, sk_d, sk, off), col0, ncols, stride, subset in forms:
                g = ops.score_ref_sample(Q, Kd, c["sid_d"][b], sk_d, off, c["inv_tau"], incl, col0, ncols, stride, bool(subset))
                e = cb.score_ref_sample(Qc, Kc, c["sid"][b], sk, off, c["inv_tau"], incl, col0, ncols, stride, bool(subset))
                torch.cuda.synchronize()
                assert g["stride"] == e["stride"] == stride
                for k in ("ref", "diag", "lam"):
                    chk(f"A.ref_sample.{k}", stat_err(g[k], e[k]), STAT)
    chk.done()


@_a_params
def test_single_pass_against_emulation(env, shape, critic, precision):
    """score_single_pass of a rank's block: rows, scal slots 0-6, flag, wrow, oq_raw, ok_raw — once without events, once
    with the other ranks' text rows arriving late (event_k_ready, k_local_valid: the own-columns-first schedule where the
    block qualifies), and once without the K-side contraction."""
    ops, mdist, mo, cb, dev = env
    c = _stage_case(env, shape, critic, precision)
    chk = Checks(f"single_pass {shape[:2]} {critic} {precision}")
    Bl, Bg, inv_tau, raw = c["Bl"], c["Bg"], c["inv_tau"], RAW[precision]
    for r in c["ranks"]:
        b = slice(r * Bl, (r + 1) * Bl)
        Q, Qc = _rows(ops, c["T"], b), c["Tc"][b]
        for incl in (False, True):
            # the references of the sharded step: exact log-sum-exp of the OWN column block + the 48-nat margin; lambda a
            # little above this block's largest (another rank's)
            smp = cb.score_ref_sample(Qc, c["Yc"], c["sid"][b], c["sid"], b.start, inv_tau, incl, b.start, Bl, 1, True)
            ref, diag = smp["ref"].float(), smp["diag"].float()
            lam = (ref.max() - 48.0 + 1.0).reshape(1).float()
            e = cb.score_single_pass(Qc, c["Yc"], c["sid"][b], c["sid"], b.start, inv_tau, incl, precision, 1.0 / Bg,
                                     ref, lam, diag)
            assert int(e["flag"]) == 0, "the inputs must stay inside the guard window"
            runs = {}
            for mode in ("plain", "delayed", "no_k"):
                K, ev = _delayed_k(c["Yd"], b) if mode == "delayed" else (c["Yd"], None)
                runs[mode] = g = ops.score_single_pass(Q, K, c["sid_d"][b], c["sid_d"], b.start, inv_tau, incl, precision,
                                                       1.0 / Bg, ref.to(dev), lam.to(dev), diag.to(dev), want_k=mode != "no_k",
                                                       event_k_ready=ev, k_local_valid=ev is not None)
                torch.cuda.synchronize()
                t = f"A.single_pass.{mode}"
                for j in (0, 2, 3):
                    chk(f"{t}.rows", stat_err(g["rows"][:, j], e["rows"][:, j]), STAT)
                chk.exact(f"{t}.n_neg", g["rows"][:, 1], e["rows"][:, 1])
                for j in (0, 3, 4):
                    chk(f"{t}.scal", scal_rel(g["scal"][j], e["scal"][j]), SCAL)
                # slot 1 = sum_i e^{lse_i - m} carries the absolute error of the fp32 row log-sum-exps as a RELATIVE error
                # (measured up to 4e-6 in fast bilinear mode, rows within 7e-7 (1 + |lse|)): it is checked in the form the
                # merge uses it, m + ln(slot 1) = the block's log-sum-exp, with the statistics bound
                chk(f"{t}.scal_lse", stat_err(g["scal"][0] + torch.log(g["scal"][1]), e["scal"][0] + torch.log(e["scal"][1])), STAT)
                for j in (2, 5, 6):
                    chk.exact(f"{t}.scal_counts", g["scal"][j], e["scal"][j])
                chk.exact(f"{t}.flag", g["flag"], e["flag"])
                chk(f"{t}.log_wrow", stat_err(torch.log(g["wrow"].double()), torch.log(e["wrow"])), STAT)
                chk(f"{t}.oq_raw.{precision}", rel(g["oq_raw"], e["oq_raw"]), raw)
                if mode != "no_k":
                    chk(f"{t}.ok_raw.{precision}", rel(g["ok_raw"], e["ok_raw"]), raw)
            d, p = runs["delayed"], runs["plain"]
            chk("A.single_pass.delayed_vs_plain.rows", stat_err(d["rows"], p["rows"]), STAT)
            chk(f"A.single_pass.delayed_vs_plain.raw.{precision}", max(rel(d["oq_raw"], p["oq_raw"]), rel(d["ok_raw"], p["ok_raw"])), raw)
    chk.done()


@_a_params
def test_score_grad_against_emulation(env, shape, critic, precision):
    """score_grad of a rank's block: dv-like (one global reference), row InfoNCE and symmetric InfoNCE (row AND column
    references, positive pair included); fp32, bf16 and hi/lo outputs, with and without the K side, gamma 0 and 1/B."""
    ops, mdist, mo, cb, dev = env
    c = _stage_case(env, shape, critic, precision)
    chk = Checks(f"score_grad {shape[:2]} {critic} {precision}")
    Bl, Bg, inv_tau, raw, D = c["Bl"], c["Bg"], c["inv_tau"], RAW[precision], c["D"]
    strict = precision == "strict"
    o16 = "split" if strict else "bf16"
    for r in c["ranks"]:
        b = slice(r * Bl, (r + 1) * Bl)
        Q, Qc = _rows(ops, c["T"], b), c["Tc"][b]
        lse = c["lse_neg"].float().expand(Bl).contiguous()
        row, col = c["row_all"][b].float(), c["col_all"].float()
        dv = dict(refq=lse, wq=1.0, refk=None, wk=0.0, include_diag=False)
        rowi = dict(refq=row, wq=1.0 / Bg, refk=None, wk=0.0, include_diag=True)
        sym = dict(refq=row, wq=0.5 / Bg, refk=col, wk=0.5 / Bg, include_diag=True)
        variants = [("dv", dv, 1.0 / Bg, True, ("f32", "bf16")), ("row", rowi, 1.0 / Bg, True, ("f32", o16)),
                    ("sym", sym, 1.0 / Bg, True, ("f32", "bf16")), ("sym_gamma0_noK", sym, 0.0, False, ("f32",)),
                    ("row_16only", rowi, 1.0 / Bg, True, (o16,))]
        for name, a, gamma, want_k, outs in variants:
            dev_a = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in a.items()}
            g32, g16, gk = ops.score_grad(Q, c["Yd"], c["sid_d"][b], c["sid_d"], b.start, inv_tau, precision=precision,
                                          alpha=inv_tau, gamma=gamma, want_f32="f32" in outs, want_bf16=len(outs) > 1 or "f32" not in outs,
                                          out_split="split" in outs, want_k=want_k, **dev_a)
            e, _, ek = cb.score_grad(Qc, c["Yc"], c["sid"][b], c["sid"], b.start, inv_tau, precision=precision, alpha=inv_tau,
                                     gamma=gamma, want_k=want_k, **a)
            torch.cuda.synchronize()
            t = f"A.score_grad.{name}"
            if g32 is not None:
                chk(f"{t}.oq.{precision}", rel(g32, e), raw)
            if g16 is not None:
                v16 = g16.float() if isinstance(g16, ops.SplitBF16) else g16
                if g32 is not None:                   # the same values, rounded once more
                    if isinstance(g16, ops.SplitBF16):
                        chk("A.score_grad.hilo_vs_f32", rel(v16, g32), SPLIT)
                    else:
                        chk("A.score_grad.bf16_vs_f32_ulps", ulp_err(v16, g32), 1.0)
                else:
                    chk(f"{t}.oq16.{precision}", rel(v16, e), raw + (0.0 if isinstance(g16, ops.SplitBF16) else 2.0 ** -8))
            if want_k:
                chk(f"{t}.ok.{precision}", rel(gk, ek), raw)
                assert gk.shape == (Bg, D)
            else:
                assert gk is None
    chk.done()


@pytest.mark.parametrize("critic", ["dot", "bilinear"])
@pytest.mark.parametrize("shape", A_SHAPES[:3], ids=A_IDS[:3])
def test_single_finalize_against_emulation(env, shape, critic):
    """single_finalize_q (dv-like: c = e^{ref - LSE}; row InfoNCE: c = wrow) with fp32, bf16 and hi/lo output, and
    single_finalize_k (kappa = e^{lambda - LSE} or 1) on the rank's own rows; strict-mode T as the hi/lo Q_diag."""
    ops, mdist, mo, cb, dev = env
    c = _stage_case(env, shape, critic, "strict")
    chk = Checks(f"finalize {shape[:2]} {critic}")
    Bl, D, alpha, gamma = c["Bl"], c["D"], 0.7, 0.37
    g = torch.Generator().manual_seed(11)
    for r in c["ranks"]:
        b = slice(r * Bl, (r + 1) * Bl)
        raw = torch.randn(Bl, D, generator=g)
        lse = torch.tensor([2.5])
        ref = (lse + 6.0 * torch.rand(Bl, generator=g) - 3.0).float()
        wrow = (torch.rand(Bl, generator=g) + 0.5).float()
        lam = torch.tensor([3.25])
        for dv_like in (False, True):
            for out in ("f32", "bf16", "split"):
                o32, o16 = ops.single_finalize_q(raw.to(dev), ref.to(dev), wrow.to(dev), lse.to(dev), dv_like, alpha, gamma,
                                                 c["Yd"][b], want_f32=out == "f32", want_bf16=out != "f32", out_split=out == "split")
                e, _ = cb.single_finalize_q(raw.double(), ref, wrow.double(), lse, dv_like, alpha, gamma, c["Yc"][b])
                torch.cuda.synchronize()
                if out == "f32":
                    chk("A.finalize_q.f32", rel(o32, e), FIN)
                elif out == "bf16":
                    chk("A.finalize_q.bf16_ulps", ulp_err(o16, e), 1.0)
                else:
                    chk("A.finalize_q.hilo", rel(o16.float(), e), SPLIT)
            ok = torch.randn(Bl, D, generator=g)
            gk = ops.single_finalize_k(ok.to(dev), lam.to(dev), lse.to(dev), dv_like, alpha, gamma, _rows(ops, c["T"], b))
            ek = cb.single_finalize_k(ok.double().clone(), lam, lse, dv_like, alpha, gamma, c["Tc"][b])
            torch.cuda.synchronize()
            chk("A.finalize_k.f32", rel(gk, ek), FIN)
    chk.done()


@pytest.mark.parametrize("est", ["dv", "infonce", "infonce_row"])
def test_merge_scalars_loss_against_fp64(env, est):
    """[world, 8] scalar rows of several blocks — one block without negatives (scal[0] = -inf), guard counts on one block —
    with lambda inside and outside the 60-nat window: the kernel's loss terms against dist.merge_scalars + dist._loss_from."""
    ops, mdist, mo, cb, dev = env
    chk = Checks(f"merge {est}")
    g = torch.Generator().manual_seed(3)
    Bg = 2048
    blocks = []
    for r in range(4):
        lse_r = 4.0 + torch.rand(1, generator=g).item()
        blocks.append([lse_r + 0.5, float(torch.rand(1, generator=g)) * 40 + 1, 508.0 * 2043 + r, 12.0 + r, 9.0 * 512 + r,
                       float(r % 2), 0.0, 0.0])
    empty = [-math.inf, 0.0, 0.0, 7.5, 3.25 * 512, 512.0, 0.0, 0.0]             # every row of this block is one study
    for rows, guard_rows in ((blocks, 0.0), (blocks[:2] + [empty] + blocks[2:], 0.0), (blocks + [empty], 3.0)):
        scal = torch.tensor(rows, dtype=torch.float64)
        scal[1, 6] = guard_rows
        ref = mdist.merge_scalars(scal)
        for lam_off in ((0.5, 75.0) if est != "infonce_row" else (None,)):
            lam = None if lam_off is None else (ref["lse_neg"] + lam_off).float().reshape(1)
            got = ops.merge_scalars_loss(scal.to(dev), est, Bg, None if lam is None else lam.to(dev))
            torch.cuda.synchronize()
            out = {"pos_mean": ref["diag_sum"] / Bg, "lse_neg": ref["lse_neg"], "n_neg": ref["n_neg"],
                   "loss_row": ref["rowloss_sum"] / Bg}
            loss = mdist._loss_from(out, est)
            guard = float(ref["guard"]) + (1.0 if lam is not None and abs(float(lam) - float(ref["lse_neg"])) > 60.0 else 0.0)
            for k, v in (("loss", loss), ("pos_mean", out["pos_mean"]), ("lse_neg", out["lse_neg"]), ("loss_row", out["loss_row"])):
                chk(f"A.merge.{k}", scal_rel(got[k], v), SCAL)
            chk.exact("A.merge.n_neg", got["n_neg"], ref["n_neg"])
            chk.exact("A.merge.rows_without_negatives", got["rows_without_negatives"], ref["rows_without_negatives"])
            chk.exact("A.merge.guard", got["guard"], guard)
            chk("A.merge.lse32", scal_rel(got["lse32"], float(out["lse_neg"])), 2.0 ** -23)
    chk.done()


def test_gemm_forms_against_fp64(env):
    """ops.gemm: C = alpha (A B^T - gamma SUB) with fp32 / bf16 / hi/lo output and a hi/lo A; the in-place forms X W (b_t),
    A^T B^T (a_t) and X^T dT (a_t, b_t) with plain and hi/lo dT — one of them with K = 20480 rows, long enough that the
    hi/lo product runs as several split-K chains (k_blocks > kStrictChainBlocks = 128)."""
    ops, mdist, mo, cb, dev = env
    from mi_b200 import _lib
    lib = _lib.load()
    chk = Checks("gemm")
    g = torch.Generator().manual_seed(5)
    bf = lambda *s: (torch.randn(*s, generator=g) / 2).bfloat16().to(dev)
    f64 = lambda t: t.float().cpu().double()
    A, B, sub = bf(300, 136), bf(520, 136), bf(300, 520)
    e = 0.7 * (f64(A) @ f64(B).t() - 0.3 * f64(sub))
    chk("A.gemm.plain.f32", rel(ops.gemm(A, B, 0.7, 0.3, sub), e), FIN)
    chk("A.gemm.plain.bf16_ulps", ulp_err(ops.gemm(A, B, 0.7, 0.3, sub, out_dtype=torch.bfloat16), e), 1.0)
    chk("A.gemm.plain.hilo", rel(ops.gemm(A, B, 0.7, 0.3, sub, out_split=True).float(), e), SPLIT)
    Ah = ops.gemm(bf(300, 64), bf(136, 64), out_split=True)                     # a hi/lo A operand [300, 136]
    chk("A.gemm.hilo_A.f32", rel(ops.gemm(Ah, B, 0.7, 0.3, sub), 0.7 * (f64(Ah) @ f64(B).t() - 0.3 * f64(sub))), FIN)
    X, W = bf(600, 72), bf(72, 72)
    chk("A.gemm.b_t.hilo", rel(ops.gemm(X, W, b_t=True, out_dtype=torch.bfloat16, out_split=True).float(), f64(X) @ f64(W)), SPLIT)
    chk("A.gemm.b_t.bf16_ulps", ulp_err(ops.gemm(X, W, b_t=True, out_dtype=torch.bfloat16), f64(X) @ f64(W)), 1.0)
    At, Bn = bf(600, 136), bf(200, 600)
    chk("A.gemm.a_t.f32", rel(ops.gemm(At, Bn, a_t=True), f64(At).t() @ f64(Bn).t()), FIN)
    cg = lib.mi_get_cta_group()
    bk, rows_per_mblk = (128 if cg == 2 else 64), 128 * cg
    for K, D in ((600, 72), (20480, 64)):
        Xk = bf(K, D)
        for split in (False, True):
            dT = ops.gemm(bf(K, D), bf(D, D), b_t=True, out_dtype=torch.bfloat16, out_split=split)
            got = ops.gemm(Xk, dT, a_t=True, b_t=True)
            chk(f"A.gemm.XtdT.{'hilo' if split else 'bf16'}.f32", rel(got, f64(Xk).t() @ f64(dT)), FIN)
            if K == 20480 and split:
                k_blocks = 2 * -(-K // bk)
                tiles = -(-D // rows_per_mblk) * -(-D // 256)
                ks = lib.mi_plan_ksplit(tiles, k_blocks, 1)
                print(f"  X^T dT, K = {K}, hi/lo dT: k_blocks {k_blocks}, split-K {ks}, chain {-(-k_blocks // ks)} blocks")
                assert k_blocks > 128 and ks > 1 and -(-k_blocks // ks) <= 128
    chk.done()


# ------------------------------------------------------------------ B. ranks emulated on one device

def emulate_ranks(ops, mdist, Xb, Yb, Wb, sid, P, est, precision, inv_tau, two_pass=False, events=False, delayed_k=True):
    """mi_b200.dist's step with the P ranks' row blocks run one after another on this device: _single_pass_step (dv /
    infonce / infonce_row) or the two-pass branch (exact references; infonce_sym through score_stats_rc + score_grad with
    refk).  Collectives by hand: all-gather = cat / stack, all-reduce MAX of lambda, reduce-scatter = sum + slice, all-reduce
    of dW = sum.  ``events``: pass event_after_k / event_after_scal as the NCCL form does (set_overlap_reserve_sms acts on the
    launches after event_after_k).  ``delayed_k``: every block's single pass reads the other blocks' text rows from a copy
    that arrives late (_delayed_k).  Returns (stats of 0-d fp64 tensors incl. loss and guard, dX, dY, dW) of the batch; a
    tripped guard repeats the step with exact references and reports the merged count."""
    Bg, D = Xb.shape
    Bl = Bg // P
    blk = [slice(r * Bl, (r + 1) * Bl) for r in range(P)]
    bilinear, strict = Wb is not None, precision == "strict"
    sym = est == "infonce_sym"
    dv_like = est in ("dv", "infonce")
    gamma = 1.0 / Bg
    sid = sid.to(torch.int32).contiguous()

    def event():
        if not events:
            return None
        e = torch.cuda.Event()
        e.record()                                 # creates the CUDA event; the library re-records it in the pass
        return e

    T = [ops.gemm(Xb[b], Wb, b_t=True, out_dtype=torch.bfloat16, out_split=strict) if bilinear else Xb[b] for b in blk]
    Y_all = torch.cat([Yb[b] for b in blk])                                       # all-gather of the text embeddings
    dX, dWs = [], []
    if not (two_pass or sym):
        smp = [ops.score_ref_sample(T[r], Yb[b], sid[b], sid[b], 0, inv_tau, not dv_like, subset=P > 1) for r, b in enumerate(blk)]
        lam = torch.stack([s["lam"] for s in smp]).max().reshape(1)              # all-reduce(MAX) of lambda
        sp = []
        for r, b in enumerate(blk):
            K, ev_y = _delayed_k(Y_all, b) if (delayed_k and P > 1) else (Y_all, None)
            sp.append(ops.score_single_pass(T[r], K, sid[b], sid, b.start, inv_tau, not dv_like, precision, gamma, smp[r]["ref"],
                                            lam, smp[r]["diag"], want_k=True, event_after_k=event(), event_after_scal=event(),
                                            event_k_ready=ev_y, k_local_valid=ev_y is not None))
        out = ops.merge_scalars_loss(torch.stack([s["scal"] for s in sp]), est, Bg, lam if dv_like else None)   # all-gather
        lse32 = out.pop("lse32")
        if float(out["guard"]) != 0.0:
            again = emulate_ranks(ops, mdist, Xb, Yb, Wb, sid, P, est, precision, inv_tau, True, events, delayed_k)
            again[0]["guard"] = out["guard"]
            return again
        dY_all = torch.stack([s["ok_raw"] for s in sp]).sum(0)                    # reduce-scatter: sum ...
        dY = []
        for r, b in enumerate(blk):
            dT32, dT16 = ops.single_finalize_q(sp[r]["oq_raw"], smp[r]["ref"], sp[r]["wrow"], lse32, dv_like, inv_tau, gamma,
                                               Yb[b], want_f32=not bilinear, want_bf16=bilinear, out_split=bilinear and strict)
            if bilinear:
                dWs.append(ops.gemm(Xb[b], dT16, a_t=True, b_t=True))
                dX.append(ops.gemm(dT16, Wb))
            else:
                dX.append(dT32)
            dY.append(ops.single_finalize_k(dY_all[b].contiguous(), lam, lse32, dv_like, inv_tau, gamma, T[r]))   # ... + slice
        return out, torch.cat(dX), torch.cat(dY), (sum(dWs) if bilinear else None)

    stats = [ops.score_stats_rc(T[r], Y_all, sid[b], sid, b.start, inv_tau) if sym else
             ops.score_stats(T[r], Y_all, sid[b], sid, b.start, inv_tau) for r, b in enumerate(blk)]
    m = mdist.merge_scalars(torch.stack([s[1] for s in stats]))                    # all-gather of the scalars, fp64 merge
    out = {"pos_mean": m["diag_sum"] / Bg, "lse_neg": m["lse_neg"], "n_neg": m["n_neg"], "loss_row": m["rowloss_sum"] / Bg}
    if sym:
        col_all = torch.stack([s[2] for s in stats]).double()                     # all-gather of the column partials
        diag_all = torch.cat([s[0][:, 2] for s in stats]).double()
        lse_c = torch.logaddexp(torch.logsumexp(col_all, 0), diag_all)
        out["loss_col"] = (lse_c - diag_all).sum() / Bg
        out["loss"] = 0.5 * (out["loss_row"] + out["loss_col"])
        c_all = lse_c.to(torch.float32)
    else:
        out["loss"] = mdist._loss_from(out, est)
    out["guard"] = torch.zeros((), dtype=torch.float64, device=Xb.device)
    parts = []
    for r, b in enumerate(blk):
        rows = stats[r][0]
        if dv_like:
            a = dict(refq=out["lse_neg"].to(torch.float32).expand(Bl).contiguous(), wq=1.0, refk=None, wk=0.0, include_diag=False)
        elif sym:
            a = dict(refq=rows[:, 3].contiguous(), wq=0.5 / Bg, refk=c_all, wk=0.5 / Bg, include_diag=True)
        else:
            a = dict(refq=rows[:, 3].contiguous(), wq=1.0 / Bg, refk=None, wk=0.0, include_diag=True)
        dT32, dT16, part = ops.score_grad(T[r], Y_all, sid[b], sid, b.start, inv_tau, precision=precision, alpha=inv_tau,
                                          gamma=gamma, want_f32=not bilinear, want_bf16=bilinear, out_split=bilinear and strict,
                                          want_k=True, event_after_k=event(), **a)
        parts.append(part)
        if bilinear:
            dX.append(ops.gemm(dT16, Wb))
            dWs.append(ops.gemm(Xb[b], dT16, a_t=True, b_t=True))
        else:
            dX.append(dT32)
    dY_all = torch.stack(parts).sum(0)                                             # reduce-scatter: sum + slice
    return out, torch.cat(dX), torch.cat([dY_all[b] for b in blk]), (sum(dWs) if bilinear else None)


def _loss_close(a, b, pos, lse, rel_tol):
    """|a - b| / bound: relative error plus the fp32 resolution of the two terms the loss is a difference of"""
    return abs(float(a) - float(b)) / (rel_tol * abs(float(b)) + 1e-6 * (abs(float(pos)) + abs(float(lse))))


def _compare(chk, tag, got, full, ref, precision, bilinear):
    """emulated step vs the single-GPU call (full = loss_out, dX, dY, dW) and vs the fp64 oracle (ref dict or None)"""
    out, dX, dY, dW = got
    lo, fX, fY, fW = full
    raw = RAW[precision]
    chk(f"B.vs_single_gpu.loss", _loss_close(out["loss"], lo[0], lo[1], lo[2], LOSS), 1.0)
    chk.exact("B.vs_single_gpu.n_neg", out["n_neg"], lo[3])
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
_ORACLE = {}


def _oracle(mo, key, Xb, Yb, sid, Wb, inv_tau, est):
    if key not in _ORACLE:
        if len(_ORACLE) > 64:
            _ORACLE.clear()
        _ORACLE[key] = mo.critic_loss(Xb.float(), Yb.float(), sid, None if Wb is None else Wb.float(), inv_tau, est)
    return _ORACLE[key]


@pytest.mark.parametrize("precision", ["strict", "fast"])
@pytest.mark.parametrize("critic", ["dot", "bilinear"])
@pytest.mark.parametrize("Bg,P,D", B_SHAPES, ids=[f"B{b}-P{p}-D{d}" for b, p, d in B_SHAPES])
def test_emulated_ranks_equal_single_gpu_and_oracle(env, Bg, P, D, critic, precision):
    """dv / infonce / infonce_row through the single pass (sampled references from the own block, delayed K) and all four
    estimators through the exact path, against ops.critic_loss_fwd_bwd(two_pass=True) on the whole batch and the oracle"""
    ops, mdist, mo, cb, dev = env
    Xb, Yb, sid, Wb, inv_tau = _batch(mo, Bg, P, D, Bg + 7 * P, critic)
    Xd, Yd, Wd, sd = Xb.to(dev), Yb.to(dev), None if Wb is None else Wb.to(dev), sid.to(torch.int32).to(dev)
    chk = Checks(f"ranks B{Bg} P{P} D{D} {critic} {precision}")
    for est, exact in PATHS:
        got = emulate_ranks(ops, mdist, Xd, Yd, Wd, sd, P, est, precision, inv_tau, two_pass=exact)
        full = ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd, est, precision, inv_tau, True, two_pass=True)
        torch.cuda.synchronize()
        chk.exact("B.guard", got[0]["guard"], 0.0)
        ref = _oracle(mo, (Bg, P, D, critic, est), Xb, Yb, sid, Wb, inv_tau, est)
        _compare(chk, est, got, full, ref, precision, Wb is not None)
    chk.done()


def test_emulated_ranks_multi_panel(env):
    """Bl = 20480 rows per rank at D = 64: more than one dS row panel (panel_mblks) per block; against the single-GPU call
    and the chunked oracle on the device"""
    ops, mdist, mo, cb, dev = env
    from oracle import chunked_oracle as co
    Bg, P, D = 40960, 2, 64
    assert Bg // P > torch.cuda.get_device_properties(0).multi_processor_count * 128, "the block must span several panels"
    Xb, Yb, sid, _, inv_tau = _batch(mo, Bg, P, D, 17, "dot")
    Xd, Yd, sd = Xb.to(dev), Yb.to(dev), sid.to(dev)
    chk = Checks(f"ranks multi-panel B{Bg} P{P}")
    for est, exact, precision in (("dv", False, "strict"), ("infonce_row", False, "fast"), ("infonce_sym", True, "strict"),
                                  ("infonce", True, "fast")):
        got = emulate_ranks(ops, mdist, Xd, Yd, None, sd.to(torch.int32), P, est, precision, inv_tau, two_pass=exact)
        full = ops.critic_loss_fwd_bwd(Xd, Yd, None, sd.to(torch.int32), est, precision, inv_tau, True, two_pass=True)
        torch.cuda.synchronize()
        chk.exact("B.guard", got[0]["guard"], 0.0)
        ref = co.critic_loss_chunked(Xd.float(), Yd.float(), sd, None, inv_tau, est, chunk=4096)
        _compare(chk, est, got, full, ref, precision, False)
        del ref, full, got
    chk.done()


def _planted(mo, Bg, D, seed, planted):
    """row 7 with one score hundreds of nats above every column its rank's strided sample sees (column 5 is not sampled)"""
    X, Y, sid, _ = mo.synthetic_embeddings(Bg, D, seed=seed, dup_frac=0.05, bilinear=False)
    Xb, Yb = X.bfloat16(), Y.bfloat16()
    if planted:
        Yb[7] = -Yb[5]
        Xb[7] = (100.0 * Yb[5].float()).bfloat16()
    return Xb, Yb, sid


def _planted_in_range(mo, Bg, D, inv_tau, stride, excess=78.0):
    """_planted with the outlier scaled so that its score sits ``excess`` nats above the row's sampled reference (log-sum-exp
    of the negatives among columns 0, stride, 2 stride, ... + the 48-nat margin): the row sum (~e^78 > 1e30) trips the
    guard while every value of the pass's statistics stays inside the fp32 range.  (A larger outlier overflows the row
    sum: the unchecked step then reports the trip with a NaN loss.)"""
    X, Y, sid, _ = mo.synthetic_embeddings(Bg, D, seed=3, dup_frac=0.05, bilinear=False)
    Xb, Yb = X.bfloat16(), Y.bfloat16()
    Yb[7] = -Yb[5]
    neg = torch.arange(0, Bg, stride)
    neg = neg[sid[neg] != sid[7]]

    def over(k):
        x7 = (k * Yb[5].float()).bfloat16().double()
        s = inv_tau * (Yb.double() @ x7)
        return float(s[5] - torch.logsumexp(s[neg], 0) - 48.0), x7

    lo, hi = 1.0, 200.0
    assert over(lo)[0] < excess < over(hi)[0]
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if over(mid)[0] < excess else (lo, mid)
    gap, x7 = over(hi)
    assert abs(gap - excess) < 1.0, gap
    Xb[7] = x7.bfloat16()
    return Xb, Yb, sid


@pytest.mark.parametrize("est", ["dv", "infonce_row"])
def test_emulated_ranks_guard_trip(env, est):
    """A planted outlier in block 0 of 4, 64 sampled columns per row: the merged guard of the single pass is non-zero and the
    step repeated with exact references equals the oracle; without the outlier the sampled pass itself does."""
    ops, mdist, mo, cb, dev = env
    Bg, P, D, inv_tau = 1024, 4, 64, 0.125
    chk = Checks(f"guard {est}")
    ops.set_ref_sample_columns(64)
    try:
        for planted in (False, True):
            Xb, Yb, sid = _planted(mo, Bg, D, 3, planted)
            Xd, Yd, sd = Xb.to(dev), Yb.to(dev), sid.to(torch.int32).to(dev)
            got = emulate_ranks(ops, mdist, Xd, Yd, None, sd, P, est, "strict", inv_tau)
            exact = emulate_ranks(ops, mdist, Xd, Yd, None, sd, P, est, "strict", inv_tau, two_pass=True)
            full = ops.critic_loss_fwd_bwd(Xd, Yd, None, sd, est, "strict", inv_tau, True, two_pass=True)
            torch.cuda.synchronize()
            assert (float(got[0]["guard"]) >= 1.0) == planted, float(got[0]["guard"])
            ref = mo.critic_loss(Xb.float(), Yb.float(), sid, None, inv_tau, est)
            _compare(chk, est, got, full, ref, "strict", False)
            _compare(chk, est, exact, full, ref, "strict", False)
    finally:
        ops.set_ref_sample_columns(2048)
    chk.done()


@pytest.mark.parametrize("critic", ["dot", "bilinear"])
def test_emulated_ranks_overlap_reserve_sms(env, critic):
    """set_overlap_reserve_sms(n > 0) narrows the grid of the launches after event_after_k: same results as n = 0"""
    ops, mdist, mo, cb, dev = env
    Bg, P, D = 1024, 4, 64
    Xb, Yb, sid, Wb, inv_tau = _batch(mo, Bg, P, D, 23, critic)
    Xd, Yd, Wd, sd = Xb.to(dev), Yb.to(dev), None if Wb is None else Wb.to(dev), sid.to(torch.int32).to(dev)
    chk = Checks(f"reserve sms {critic}")
    try:
        for est, exact in (("dv", False), ("infonce_row", False), ("infonce_sym", True)):
            for precision in ("strict", "fast"):
                res = {}
                for n in (0, 16):
                    ops.set_overlap_reserve_sms(n)
                    res[n] = emulate_ranks(ops, mdist, Xd, Yd, Wd, sd, P, est, precision, inv_tau, two_pass=exact, events=True)
                    torch.cuda.synchronize()
                base = res[0]
                _compare(chk, est, res[16], (torch.stack([base[0]["loss"], base[0]["pos_mean"], base[0]["lse_neg"],
                                                         base[0]["n_neg"]]),) + base[1:], None, precision, Wd is not None)
    finally:
        ops.set_overlap_reserve_sms(0)
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
                for est in ("dv", "infonce", "infonce_row"):
                    for prec in ("strict", "fast"):
                        st, lo, dX, dY, dW = ops.sharded_step(Xd, Yd, Wd, sd, est, prec, inv_tau, check_guard=True)
                        fl, fX, fY, fW = ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd, est, prec, inv_tau, True, two_pass=True)
                        torch.cuda.synchronize()
                        res[f"B{Bg}-D{D}/{critic}/{est}/{prec}"] = {
                            "status": int(st), "guard": float(lo[7]), "n_neg": [float(lo[3]), float(fl[3])],
                            "loss": _loss_close(lo[0], fl[0], fl[1], fl[2], LOSS), "dX": rel(dX, fX), "dY": rel(dY, fY),
                            "dW": None if Wd is None else rel(dW, fW)}
        Bg, D = 1024, 64
        Xb, Yb, sid = _planted_in_range(mo, Bg, D, 0.125, Bg // 64)       # 64 sampled columns: stride 16
        Xd, Yd, sd = Xb.to(dev), Yb.to(dev), sid.to(torch.int32).to(dev)
        ops.set_ref_sample_columns(64)
        try:
            for est in ("dv", "infonce_row"):
                st1, _, _, _, _ = ops.sharded_step(Xd, Yd, None, sd, est, "strict", 0.125, check_guard=True)
                st2, lo2, _, _, _ = ops.sharded_step(Xd, Yd, None, sd, est, "strict", 0.125, check_guard=False)
                torch.cuda.synchronize()
                res[f"planted/{est}"] = {"status_checked": int(st1), "status_unchecked": int(st2), "guard": float(lo2[7]),
                                         "loss": float(lo2[0])}
        finally:
            ops.set_ref_sample_columns(2048)
    finally:
        tdist.destroy_process_group()
    with open(out_path, "w") as f:
        json.dump(res, f)


def test_one_call_sharded_step_world1(env, tmp_path):
    """ops.sharded_step (csrc/sharded.cuh) in an NCCL group of world size 1 (FileStore rendezvous) == the single-GPU call:
    dv / infonce / infonce_row x strict / fast x dot / bilinear at a ragged B and a multiple of 256; a planted outlier
    (78 nats above its row's sampled reference) returns GUARD_TRIPPED with check_guard, and without it status 0 with
    loss_out[7] >= 1 and a finite loss."""
    ops, mdist, mo, cb, dev = env
    import torch.multiprocessing as mp
    out = tmp_path / "world1.json"
    mp.spawn(_world1_worker, args=(str(tmp_path / "filestore"), str(out)), nprocs=1, join=True)
    res = json.loads(out.read_text())
    chk = Checks("sharded_step world 1")
    assert len(res) == 2 * 2 * 3 * 2 + 2
    for name, r in sorted(res.items()):
        print(f"  {name}: {r}")
        if name.startswith("planted/"):
            assert r["status_checked"] == ops.GUARD_TRIPPED and r["status_unchecked"] == 0, r
            assert r["guard"] >= 1.0 and math.isfinite(r["loss"]), r
            continue
        prec = name.rsplit("/", 1)[1]
        assert r["status"] == 0 and r["guard"] == 0.0 and r["n_neg"][0] == r["n_neg"][1], (name, r)
        chk("C.sharded_step.loss", r["loss"], 1.0)
        for k in ("dX", "dY", "dW"):
            if r[k] is not None:
                chk(f"C.sharded_step.{k}.{prec}", r[k], RAW[prec])
    chk.done()


# ------------------------------------------------------------------ D. the fp32 -> bf16 cast

def _special_f32():
    u = []
    for hi in (0x3F80, 0x3F81, 0x4049, 0x404A, 0x0000, 0x0001, 0x0080, 0x7F7E):
        u += [(hi << 16) | lo for lo in (0x8000, 0x7FFF, 0x8001)]               # ties (to even: up for odd hi), near ties
    u += [0x00000001, 0x00007FFF, 0x00008000, 0x00018000, 0x00400000, 0x007FFFFF]   # subnormals
    u += [0x7F7F8000, 0x7F7F8001, 0x7F7FFFFF, 0x7F7F7FFF]                           # round to inf / to the largest bf16
    u += [0x7F800000, 0x7FC00000, 0x7F800001, 0x7FBFFFFF]                           # inf, NaN (quiet, signalling)
    u = np.array(u, dtype=np.uint32)
    u = np.concatenate([u, u | np.uint32(0x80000000)])
    rnd = np.random.RandomState(0).randint(0, 2 ** 32, size=4096, dtype=np.uint64).astype(np.uint32)
    return torch.from_numpy(np.concatenate([u, rnd]).view(np.float32).copy())


def _cast_check(ops, x):
    """ops.as_bf16(x) bit-equal to x.bfloat16() (round to nearest even); NaN in, NaN out"""
    got = ops.as_bf16(x).cpu()
    want = x.cpu().bfloat16()
    nan = torch.isnan(x.cpu())
    assert bool(torch.isnan(got[nan].float()).all())
    g, w = got[~nan].view(torch.int16), want[~nan].view(torch.int16)
    bad = (g != w).nonzero().reshape(-1)
    assert bad.numel() == 0, [(hex(int(x.cpu()[~nan].view(torch.int32)[i]) & 0xFFFFFFFF), hex(int(g[i]) & 0xFFFF),
                               hex(int(w[i]) & 0xFFFF)) for i in bad[:8]]


def test_cast_f32_to_bf16_bit_exact(env):
    """ties, subnormals, overflow to +-inf, +-inf and NaN; lengths n = 1, 2, 3 (mod 4) that end in the scalar tail; and
    contiguous views at element offsets 1, 2, 3 (not 16-byte aligned: the kernel must not take its float4 path there)"""
    ops, mdist, mo, cb, dev = env
    v = _special_f32()
    for n in (1, 2, 3, 5, 6, 7, 4097, 4098, 4099, v.numel()):
        _cast_check(ops, v.repeat(n // v.numel() + 1)[:n].to(dev))
    B, D = 48, 72
    buf = torch.cat([v, torch.randn(B * D + 8)]).to(dev)
    for off in (1, 2, 3, 4):
        view = buf[off:off + B * D].view(B, D)
        assert view.is_contiguous() and view.storage_offset() == off
        _cast_check(ops, view)
    flat = torch.randn(1 + D * D).to(dev)                                          # a flat parameter buffer's view of W
    _cast_check(ops, flat[1:].view(D, D))
