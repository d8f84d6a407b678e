"""Symmetric InfoNCE in the one-call batch-sharded step (csrc/sharded.cuh) at N = 1: ms per fwd+bwd step of
ops.sharded_step(..., "infonce_sym") in an NCCL group of world size 1 next to the single-GPU
ops.critic_loss_fwd_bwd(..., "infonce_sym") on the same inputs, timed in the same process and alternated.

    python scripts/sharded_sym_bench.py [--rounds 5] [--steps 10] [--warmup 3] > profiles/...

At world size 1 the step's collectives are device copies; the difference to the single-GPU call is the step's own work
(the packed record, the fp64 merge, the row-block form of the passes).  Timing: CUDA events around `--steps` steps after
`--warmup` steps, `--rounds` alternating rounds; min / median / max over the rounds.  Inputs of B = 65536 x D = 1024 bf16
(128 MB each, above the 126 MB of L2); the small shape is launch-bound."""
import argparse
import os
import statistics
import subprocess
import sys
import tempfile

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mi_b200  # noqa: E402,F401
from mi_b200 import ops  # noqa: E402
from oracle import matrix_oracle as mo  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--rounds", type=int, default=5)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--warmup", type=int, default=3)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("sharded_sym_bench.py needs a CUDA device")

dev = torch.device("cuda:0")
torch.cuda.set_device(dev)
store_dir = tempfile.mkdtemp(prefix="mi_sym_bench_")
dist.init_process_group("nccl", store=dist.FileStore(os.path.join(store_dir, "store"), 1), rank=0, world_size=1, device_id=dev)


def timed(fn):
    for _ in range(a.warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / a.steps


try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001
    card = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
print(f"card: {card}; NCCL world size 1; {a.rounds} alternating rounds of {a.steps} steps after {a.warmup} warm-up")
print("| B | D | critic | precision | path | min ms | median ms | max ms | one-call / single (median) |")
print("|---|---|---|---|---|---|---|---|---|")
try:
    for B, D, critic, precisions in ((65536, 1024, "bilinear", ("fast", "strict")), (4096, 768, "bilinear", ("fast", "strict"))):
        X, Y, sid, W = mo.synthetic_embeddings(B, D, seed=5, dup_frac=0.05, bilinear=critic == "bilinear")
        Xd, Yd, sd = X.bfloat16().to(dev), Y.bfloat16().to(dev), sid.to(torch.int32).to(dev)
        Wd = W.bfloat16().to(dev) if critic == "bilinear" else None
        del X, Y, W
        for prec in precisions:
            one = lambda: ops.sharded_step(Xd, Yd, Wd, sd, "infonce_sym", prec, 1.0, check_guard=False)   # noqa: E731
            single = lambda: ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd, "infonce_sym", prec, 1.0, True)      # noqa: E731
            st, lo, *_ = one()
            fl, *_ = single()
            torch.cuda.synchronize()
            assert st == 0 and float(lo[7]) == 0.0, (st, lo)
            dl = abs(float(lo[0]) - float(fl[0])) / abs(float(fl[0]))
            t = {"one-call step": [], "single-GPU call": []}
            for _ in range(a.rounds):
                t["one-call step"].append(timed(one))
                t["single-GPU call"].append(timed(single))
            med = {k: statistics.median(v) for k, v in t.items()}
            for path, v in t.items():
                ratio = f"{med['one-call step'] / med['single-GPU call']:.3f} (loss rel diff {dl:.1e})" if path == "one-call step" else ""
                print(f"| {B} | {D} | {critic} | {prec} | {path} | {min(v):.3f} | {med[path]:.3f} | {max(v):.3f} | {ratio} |",
                      flush=True)
finally:
    dist.destroy_process_group()
