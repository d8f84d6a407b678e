"""Fused concat-MLP critic (make_mlp(1536, [1024, 512]), SURVEY 8f-1): ms per fwd+bwd step and tensor throughput,
next to the reference sequence (explicit pair tensor -> nn.Sequential fp32 -> estimator -> backward) on the same GPU.
python scripts/mlp_bench.py [--torch-max-b 256] [--estimators dv,infonce_row,infonce_sym] > profiles/...
Rows of an estimator other than dv name it in the path column; infonce_row / infonce_sym take the two-pass sequence in
every mode."""
import argparse
import os
import sys
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mi_b200  # noqa
from mi_b200 import ops, _lib

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="64,256,1024,4096")
ap.add_argument("--torch-max-b", type=int, default=256)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--modes", default="3,1,0", help="mi_set_mlp_mode values to time (3 = default)")
ap.add_argument("--estimators", default="dv", help="estimators to time (dv, infonce, infonce_row, infonce_sym)")
a = ap.parse_args()
dev = torch.device("cuda:0")
D, H1, H2 = 768, 1024, 512


def timed(fn, steps):
    fn(); fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


print("| B | pairs | path | ms / step | F_alg TFLOP/s | pairs/s | engine ms by kind (launches), one step |")
print("|---|---|---|---|---|---|---|")
for B in [int(v) for v in a.sizes.split(",")]:
    g = torch.Generator().manual_seed(B)
    X = torch.relu(torch.randn(B, D, generator=g)).to(dev)
    Y = torch.tanh(torch.randn(B, D, generator=g)).to(dev)
    sid = torch.arange(B, dtype=torch.int32, device=dev)
    torch.manual_seed(1)
    critic = mi_b200.FusedMLPCritic(D, (H1, H2)).to(dev)
    params = (critic[0].weight, critic[0].bias, critic[2].weight, critic[2].bias, critic[4].weight, critic[4].bias)
    # algorithmic flops: layer 2 forward + its two backward contractions per pair, layer 1 once per sample (fwd + 2 bwd)
    f_alg = 3 * 2.0 * B * B * H1 * H2 + 3 * 2.0 * (2 * B) * D * H1
    for mode in [int(v) for v in a.modes.split(",")]:
        ops.set_mlp_mode(mode)
        for prec in ("fast", "strict"):
            for est in a.estimators.split(","):
                ms = timed(lambda: ops.mlp_critic_loss_fwd_bwd(X, Y, params, sid, est, prec, True, False), a.steps)
                # per-kind engine time of one more step (CUDA events around every tile-engine launch)
                import ctypes
                lib = _lib.load()
                lib.mi_set_profiling(1)
                ops.mlp_critic_loss_fwd_bwd(X, Y, params, sid, est, prec, True, False)
                torch.cuda.synchronize()
                kms = (ctypes.c_double * 6)(); kn = (ctypes.c_int64 * 6)()
                lib.mi_profile_read_kinds(kms, kn, 6)
                lib.mi_set_profiling(0)
                kinds = "gemm %.2f (%d) | single pass %.2f (%d) | fused dZ1 %.2f (%d) | two-pass epilogues %.2f (%d)" % (
                    kms[2], kn[2], kms[3], kn[3], kms[4], kn[4], kms[5], kn[5])
                path = f"fused {prec}, mode {mode}" + ("" if est == "dv" else f", {est}")
                print(f"| {B} | {B*B} | {path} | {ms:.3f} | {f_alg / ms / 1e9:.1f} | {B * B / ms * 1e3:.3e} | {kinds} |", flush=True)
    ops.set_mlp_mode(-1)
    if B <= a.torch_max_b:
        study = [str(i) for i in range(B)]

        def ref_step():
            x = X.clone().requires_grad_(True); y = Y.clone().requires_grad_(True)
            critic.zero_grad()
            rows = mi_b200.create_mi_pairs_tensor(x, y, study, dev)      # vectorised builder (the reference's loop is O(B^2) cats)
            loss = mi_b200.dv_bound_loss(critic(rows), B, dev)
            loss.sum().backward()
        ms = timed(ref_step, a.steps)
        print(f"| {B} | {B*B} | torch fp32: pair tensor + nn.Sequential + autograd | {ms:.3f} | {f_alg / ms / 1e9:.1f} | {B * B / ms * 1e3:.3e} |", flush=True)
