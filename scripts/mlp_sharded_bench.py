"""Batch-sharded concat-MLP critic (make_mlp(1536, [1024, 512]), DESIGN 8.4): ms per fwd+bwd step of
mi_b200.dist.sharded_mlp_critic_loss_fwd_bwd at a global batch B_global split over the ranks, next to the single-GPU
mi_mlp_critic_loss_fwd_bwd at the same B_global timed in the same job.

    torchrun --nproc-per-node N scripts/mlp_sharded_bench.py [--sizes 4096,8192] [--steps 10] [--estimator dv] > profiles/...
    python scripts/mlp_sharded_bench.py                      # N = 1 without a process group

Timing: CUDA events around `--steps` steps after `--warmup` steps, the maximum over ranks.  F_alg = 6 B^2 H1 H2 +
6 (2B) D H1 as in scripts/mlp_bench.py; efficiency = t_single / (N t_sharded).  The stage breakdown (mi_profile_read_kinds:
3 = single-pass epilogue, 4 = fused dZ1, 5 = two-pass epilogues) is of one extra profiled step on rank 0."""
import argparse
import ctypes
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mi_b200  # noqa: E402
from mi_b200 import _lib, ops  # noqa: E402
from mi_b200 import dist as mdist  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--sizes", default="4096,8192", help="global batch sizes")
ap.add_argument("--per-gpu", default="256", help="per-GPU batch sizes (B_global = N x value; launch-bound at 256)")
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--precisions", default="fast,strict")
ap.add_argument("--estimator", default="dv", help="dv, infonce, infonce_row or infonce_sym")
a = ap.parse_args()

world, rank = 1, 0
if "RANK" in os.environ:
    dist.init_process_group("nccl")
    world, rank = dist.get_world_size(), dist.get_rank()
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
dev = torch.device("cuda", torch.cuda.current_device())
D, H1, H2 = 768, 1024, 512


def timed(fn):
    for _ in range(a.warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    e0.record()
    for _ in range(a.steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1) / a.steps], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms)


def kinds(fn):
    lib = _lib.load()
    lib.mi_set_profiling(1)
    fn()
    torch.cuda.synchronize()
    kms = (ctypes.c_double * 6)()
    kn = (ctypes.c_int64 * 6)()
    lib.mi_profile_read_kinds(kms, kn, 6)
    lib.mi_set_profiling(0)
    return "gemm %.2f; single pass %.2f; fused dZ1 %.2f; two-pass %.2f" % (kms[2], kms[3], kms[4], kms[5])


if rank == 0:
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        card = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
    print(f"card: {card}; ranks: {world}; estimator {a.estimator}; steps {a.steps} after {a.warmup} warm-up; max over ranks")
    print("| B_global | N | precision | path | ms / step | pairs/s | F_alg TFLOP/s | efficiency | engine ms by kind, rank 0 |")
    print("|---|---|---|---|---|---|---|---|---|")
sizes = [int(v) for v in a.sizes.split(",") if v] + [world * int(v) for v in a.per_gpu.split(",") if v]
for Bg in sizes:
    Bl = Bg // world
    g = torch.Generator().manual_seed(Bg)
    X = torch.relu(torch.randn(Bg, D, generator=g)).to(dev)
    Y = torch.tanh(torch.randn(Bg, D, generator=g)).to(dev)
    sid = torch.arange(Bg, dtype=torch.int32, device=dev)
    torch.manual_seed(1)
    critic = mi_b200.FusedMLPCritic(D, (H1, H2)).to(dev)
    params = tuple(p.detach() for p in critic.parameters())
    f_alg = 3 * 2.0 * Bg * Bg * H1 * H2 + 3 * 2.0 * (2 * Bg) * D * H1
    sl = slice(rank * Bl, (rank + 1) * Bl)
    Xl, Yl, sl_id = X[sl].contiguous(), Y[sl].contiguous(), sid[sl].contiguous()
    label = " (launch-bound)" if Bl <= 256 else ""
    for prec in a.precisions.split(","):
        single = lambda: ops.mlp_critic_loss_fwd_bwd(X, Y, params, sid, a.estimator, prec, True, False)       # noqa: E731
        sharded = lambda: mdist.sharded_mlp_critic_loss_fwd_bwd(Xl, Yl, params, sl_id, a.estimator, prec)     # noqa: E731
        t1 = timed(single)
        tn = timed(sharded)
        kn = kinds(sharded)
        if rank == 0:
            for path, t, eff in (("single GPU, whole batch", t1, ""), (f"sharded{label}", tn, f"{t1 / (world * tn):.3f}")):
                print(f"| {Bg} | {1 if path.startswith('single') else world} | {prec} | {path} | {t:.3f} | "
                      f"{Bg * Bg / t * 1e3:.3e} | {f_alg / t / 1e9:.1f} | {eff} | {kn if path.startswith('sharded') else ''} |",
                      flush=True)
if world > 1:
    dist.destroy_process_group()
