"""CPU tests (not gpu) of the MLP critic's fp32 precision (MI_PREC_FP32X3, "fp32"): the three-piece bf16 operand format and
its six-segment product in a torch emulation, the size queries of every entry point, and the Python rejections of "fp32"
outside the MLP critic, which must come before any device work."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FP32X3 = 4
TERMS = ((0, 2), (1, 1), (2, 0), (0, 1), (1, 0), (0, 0))      # the K segments of two three-piece operands, smallest first
STRICT_TERMS = ((0, 0), (1, 0), (0, 1))


def split3(x: torch.Tensor):
    """What split_f32_kernel / mlp_gen*_kernel / the dZ2 epilogues store: p0 = RN(x), p1 = RN(x - p0), p2 = RN(x - p0 - p1)
    (bf16 round-to-nearest-even; both differences are exact in fp32)."""
    x = x.to(torch.float32)
    p0 = x.bfloat16().float()
    r1 = x - p0
    p1 = r1.bfloat16().float()
    p2 = (r1 - p1).bfloat16().float()
    return p0, p1, p2


def _bf16_boundary_values():
    """fp32 values next to bf16 rounding boundaries (ties and one fp32 ulp either side) over many binades, both signs."""
    out = []
    for e in range(-120, 121, 7):
        base = 2.0 ** e
        for m in (1.0, 1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, 1.5, 2.0 - 2 ** -8):
            v = torch.tensor(base * m, dtype=torch.float32)
            u = float(torch.nextafter(v, torch.tensor(float("inf"))) - v)
            for d in (-2 * u, -u, 0.0, u, 2 * u):
                out.append(float(v) + d)
    t = torch.tensor(out, dtype=torch.float32)
    return torch.cat([t, -t])


def test_three_pieces_hold_24_significant_bits():
    g = torch.Generator().manual_seed(0)
    rnd = torch.randn(200000, generator=g) * torch.exp2(torch.randint(-100, 100, (200000,), generator=g).float())
    # bits chosen directly: every mantissa pattern class, normal exponents (bf16 overflow starts at 3.39e38: not tested)
    bits = torch.randint(0x00800000, 0x7F000000, (200000,), generator=g, dtype=torch.int64).to(torch.int32)
    x = torch.cat([rnd.float(), bits.view(torch.float32), -bits.view(torch.float32), _bf16_boundary_values()])
    x = x[torch.isfinite(x) & (x.abs() >= torch.finfo(torch.float32).tiny)]
    p0, p1, p2 = split3(x)
    err = (x.double() - (p0.double() + p1.double() + p2.double())).abs()
    # 24 bits wherever the last piece is a normal bf16 number (|x| >= 2^-110); below that p2 reaches bf16's subnormal
    # spacing 2^-133 and the pieces hold x to half of it
    big = x.abs() >= 2.0 ** -110
    assert bool((err[big] <= 2.0 ** -24 * x[big].double().abs()).all()), float((err[big] / x[big].double().abs()).max())
    assert bool((err[~big] <= 2.0 ** -134).all()) and int((~big).sum()) > 0
    # the pieces shrink by 2^8 each: p1 is the residual of p0, p2 that of p0 + p1
    assert bool((p1.abs() <= 2.0 ** -8 * x.abs()).all()) and bool((p2.abs() <= 2.0 ** -16 * x.abs()).all())


def test_three_pieces_of_subnormals_and_zeros():
    sub = torch.tensor([1, 2, 3, 255, 256, 257, 0x7FFF, 0x8000, 0x12345, 0x7FFFFF], dtype=torch.int32).view(torch.float32)
    x = torch.cat([sub, -sub])
    p0, p1, p2 = split3(x)
    err = (x.double() - (p0.double() + p1.double() + p2.double())).abs()
    # bf16 shares fp32's exponent range: below 2^-126 its spacing is 2^-133, so the pieces hold x to half of that
    assert bool((err <= 2.0 ** -134).all())
    z = torch.tensor([0.0, -0.0])
    q = split3(z)
    for piece in q:
        assert bool((piece == 0).all())
    assert torch.equal(torch.signbit(q[0]), torch.signbit(z))            # the sign of zero survives in p0


@pytest.mark.parametrize("coherent", [False, True])
def test_six_segment_product_is_fp32_faithful(coherent):
    """sum over the six terms (in fp64) against the fp64 product of the fp32 operands: the dropped terms p1 p2, p2 p1, p2 p2
    and the representation error are each below 2^-24 |a||b|."""
    g = torch.Generator().manual_seed(1 + int(coherent))
    M, N, K = 64, 48, 1536
    A = torch.randn(M, K, generator=g)
    B = torch.randn(N, K, generator=g)
    if coherent:                                                   # post-ReLU operand, positive weights
        A, B = A.clamp_min(0), B.abs()
    pa, pb = split3(A), split3(B)
    got = sum(pa[i].double() @ pb[j].double().T for i, j in TERMS)
    ref = A.double() @ B.double().T
    scale = A.double().abs() @ B.double().abs().T
    assert bool(((got - ref).abs() <= 4 * 2.0 ** -24 * scale).all())
    # strict's hi/lo pairs (16 bits, three terms) leave errors orders of magnitude larger: the reason fp32 mode exists
    h = [(x.bfloat16().float(), (x - x.bfloat16().float()).bfloat16().float()) for x in (A, B)]
    strict = sum(h[0][i].double() @ h[1][j].double().T for i, j in STRICT_TERMS)
    assert float((strict - ref).abs().max()) > 30 * float((got - ref).abs().max())


def test_fp32_size_queries():
    from mi_b200 import _lib
    lib = _lib.load()
    D, H1, H2 = 768, 1024, 512
    for B in (256, 4096):
        nf = lib.mi_mlp_critic_workspace_bytes(B, D, H1, H2, 1)
        n4 = lib.mi_mlp_critic_workspace_bytes(B, D, H1, H2, FP32X3)
        assert n4 > 0 and nf > 0
        # B = 4096: the panels shrink to 2/3 of strict's pairs, so fp32 mode needs no more than 1.5 x strict's scratch
        assert n4 <= 1.5 * nf
        assert lib.mi_mlp_block_workspace_bytes(B // 2, B, D, H1, H2, FP32X3) > 0
        assert lib.mi_mlp_block_state_bytes(B // 2, B, D, H1, H2, FP32X3) >= 4 * (B // 2) * B
        assert lib.mi_mlp_input_grad_workspace_bytes(B // 2, D, H1, FP32X3) > 0
        # the separable, sharded, host-buffer and GDV planners reject it (they would otherwise run fast mode silently)
        for critic in (0, 1):
            for est in (0, 1, 2, 3):
                assert lib.mi_critic_workspace_bytes(B, D, critic, est, 1, 1) > 0
                assert lib.mi_critic_workspace_bytes(B, D, critic, est, FP32X3, 1) == 0
                assert lib.mi_critic_workspace_bytes(B, D, critic, est, FP32X3 | 2, 0) == 0
                assert lib.mi_critic_host_scratch_bytes(B, D, critic, est, FP32X3, 1) == 0
                assert lib.mi_sharded_critic_workspace_bytes(B // 2, 2, D, critic, est, FP32X3) == 0
        assert lib.mi_score_grad_workspace_bytes(B, B, D, FP32X3) == 0
        assert lib.mi_score_single_pass_workspace_bytes(B, B, D, FP32X3) == 0
        assert lib.mi_gdv_workspace_bytes(B, B, D, FP32X3) == 0 and lib.mi_gdv_workspace_bytes(B, B, D, 1) > 0
    # every contraction that feeds an epilogue must stay one bounded chain: D, H1 <= 1280 (strict has no such limit)
    assert lib.mi_mlp_critic_workspace_bytes(256, 1280, 1280, 512, FP32X3) > 0
    assert lib.mi_mlp_critic_workspace_bytes(256, 1288, 1024, 512, FP32X3) == 0
    assert lib.mi_mlp_critic_workspace_bytes(256, 768, 1288, 512, FP32X3) == 0
    assert lib.mi_mlp_critic_workspace_bytes(256, 768, 1288, 512, 1) > 0
    assert lib.mi_mlp_input_grad_workspace_bytes(256, 1288, 1024, FP32X3) == 0
    # the MLP entries take precision 0, 1 or 4 only
    for bad in (2, 3, 5, 6, -1):
        assert lib.mi_mlp_critic_workspace_bytes(256, D, H1, H2, bad) == 0
        assert lib.mi_mlp_block_workspace_bytes(128, 256, D, H1, H2, bad) == 0
        assert lib.mi_mlp_input_grad_workspace_bytes(128, D, H1, bad) == 0


def test_fp32_is_rejected_before_any_device_work(monkeypatch):
    import mi_b200
    from mi_b200 import _lib, dist, ops

    def boom(*a, **k):
        raise AssertionError("device work before the precision check")

    monkeypatch.setattr(ops, "_need_cuda", lambda *a: None)
    monkeypatch.setattr(_lib, "load", boom)
    monkeypatch.setattr(ops, "as_bf16", boom)
    monkeypatch.setattr(ops, "workspace", boom)
    X, Y, sid = torch.randn(8, 16), torch.randn(8, 16), torch.arange(8, dtype=torch.int32)
    with pytest.raises(ops.MIError, match="MLP critic only"):
        ops.critic_loss_fwd_bwd(X, Y, None, sid, "dv", "fp32")
    with pytest.raises(ops.MIError, match="MLP critic only"):
        ops.sharded_step(X, Y, None, sid, "dv", "fp32", 1.0)
    with pytest.raises(ops.MIError, match="MLP critic only"):
        ops.score_grad(X, Y, sid, sid, 0, 1.0, None, 1.0, None, 1.0, False, "fp32", 1.0, 0.0)
    with pytest.raises(ops.MIError, match="MLP critic only"):
        ops.score_single_pass(X, Y, sid, sid, 0, 1.0, False, "fp32", 1.0, X[:, 0], None, X[:, 0])
    with pytest.raises(ops.MIError, match="MLP critic only"):
        ops.gdv(X, Y, "fp32")
    with pytest.raises(ops.MIError, match="MLP critic only"):
        ops.GraphedCriticStep(8, 16, precision="fp32")
    with pytest.raises(ops.MIError, match="MLP critic only"):
        mi_b200.FusedCritic(16, "bilinear", precision="fp32")
    with pytest.raises(ValueError, match="fast and strict"):
        dist.sharded_critic_loss_fwd_bwd(X, Y, None, sid, "dv", "fp32")
    params = (torch.randn(32, 32), torch.randn(32), torch.randn(16, 32), torch.randn(16), torch.randn(1, 16), torch.randn(1))
    with pytest.raises(ops.MIError, match="MLP critic supports"):
        ops.mlp_critic_loss_fwd_bwd(X, Y, params, sid, "dv", "fp64")
    with pytest.raises(ops.MIError, match="MLP critic supports"):
        mi_b200.FusedMLPCritic(16, (32, 16), precision="bf16x9")


def test_fp32_is_an_mlp_precision():
    import mi_b200
    from mi_b200 import ops
    assert ops.MLP_PRECISION == {"fast": 0, "strict": 1, "fp32": FP32X3}
    assert "fp32" not in ops.PRECISION                     # the table the separable path reads
    c = mi_b200.FusedMLPCritic(16, (32, 16), precision="fp32")
    assert c.precision == "fp32"
    rows = torch.randn(5, 32)
    torch.testing.assert_close(c(rows), c[4](torch.relu(c[2](torch.relu(c[0](rows))))))   # the module itself is unchanged
