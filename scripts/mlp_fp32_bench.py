"""The concat-MLP critic's fp32 precision (three bf16 pieces per operand) against strict, alternated in one process:
make_mlp(1536, [1024, 512]) + dv at B = 4096 and 8192, mi_set_mlp_mode 3 and 0.  Prints the card and its power limit
(read here, in the same job), then one markdown row per (B, mode, precision, round): ms per fwd+bwd step, F_alg TFLOP/s
(the algorithm's flops, the same count for both precisions) and the engine time per kind of one profiled step.
python scripts/mlp_fp32_bench.py [--sizes 4096,8192] [--rounds 3] [--steps 3] > profiles/..."""
import argparse
import ctypes
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mi_b200  # noqa: E402
from mi_b200 import _lib, ops  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="4096,8192")
ap.add_argument("--modes", default="3,0")
ap.add_argument("--rounds", type=int, default=3, help="strict / fp32 alternations per (B, mode)")
ap.add_argument("--steps", type=int, default=3)
a = ap.parse_args()
dev = torch.device("cuda:0")
D, H1, H2 = 768, 1024, 512
lib = _lib.load()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(dev)


def timed(fn, steps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def kinds(fn):
    lib.mi_set_profiling(1)
    fn()
    torch.cuda.synchronize()
    kms = (ctypes.c_double * 6)()
    kn = (ctypes.c_int64 * 6)()
    lib.mi_profile_read_kinds(kms, kn, 6)
    lib.mi_set_profiling(0)
    return "gemm %.1f | single pass %.1f | fused dZ1 %.1f | two-pass epilogues %.1f" % (kms[2], kms[3], kms[4], kms[5])


print(f"card: {card()}")
print("| B | mode | precision | round | ms / step | F_alg TFLOP/s | engine ms by kind, one step |")
print("|---|---|---|---|---|---|---|")
for B in [int(v) for v in a.sizes.split(",")]:
    g = torch.Generator().manual_seed(B)
    X = torch.relu(torch.randn(B, D, generator=g)).to(dev)
    Y = torch.tanh(torch.randn(B, D, generator=g)).to(dev)
    sid = torch.arange(B, dtype=torch.int32, device=dev)
    torch.manual_seed(1)
    critic = mi_b200.FusedMLPCritic(D, (H1, H2)).to(dev)
    params = tuple(t.detach() for t in critic.parameters())
    f_alg = 3 * 2.0 * B * B * H1 * H2 + 3 * 2.0 * (2 * B) * D * H1
    for mode in [int(v) for v in a.modes.split(",")]:
        ops.set_mlp_mode(mode)
        for r in range(a.rounds):
            for prec in ("strict", "fp32"):
                step = lambda: ops.mlp_critic_loss_fwd_bwd(X, Y, params, sid, "dv", prec, True, False)  # noqa: E731
                ms = timed(step, a.steps)
                print(f"| {B} | {mode} | {prec} | {r} | {ms:.1f} | {f_alg / ms / 1e9:.1f} | {kinds(step)} |", flush=True)
        ops.set_mlp_mode(-1)
