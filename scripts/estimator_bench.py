"""DV, JS and NWJ on the single-GPU separable critic: ms per fwd+bwd step of ops.critic_loss_fwd_bwd, the three estimators
timed in one process and alternated step by step, plus the per-kind tile-engine times of one profiled step each.

    python scripts/estimator_bench.py OUT_DIR [--steps 12] [--warmup 3]

Shapes: B = 65536, D = 1024, bilinear (fast and strict; inputs of 128 MB each, above the 126 MB of L2) and BASELINE
config 2 (B = 4096, D = 768, bilinear).  Each step is timed with CUDA events; after `--warmup` steps of every estimator,
`--steps` rounds run DV, JS, NWJ one step each.  Reported: min / median / max per estimator, the median over DV's, and the
engine time per kind (0 score statistics, 1 dS panel, 2 GEMM) from mi_profile_read_kinds in a separate profiled step.
Writes OUT_DIR/estimator_bench.md and prints it."""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mi_b200  # noqa: E402,F401
from mi_b200 import _lib, ops  # noqa: E402
from oracle import matrix_oracle as mo  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("out_dir")
ap.add_argument("--steps", type=int, default=12)
ap.add_argument("--warmup", type=int, default=3)
a = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("estimator_bench.py needs a CUDA device")
os.makedirs(a.out_dir, exist_ok=True)
dev = torch.device("cuda:0")
lib = _lib.load()
EST = ("dv", "js", "nwj")
KINDS = 3


def step_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def kinds(fn):
    ms = (ctypes.c_double * KINDS)()
    n = (ctypes.c_int64 * KINDS)()
    lib.mi_profile_read_kinds(ms, n, KINDS)            # drain
    lib.mi_set_profiling(1)
    fn()
    torch.cuda.synchronize()
    lib.mi_set_profiling(0)
    lib.mi_profile_read_kinds(ms, n, KINDS)
    return [(ms[k], n[k]) for k in range(KINDS)]


try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
except Exception as e:  # noqa: BLE001
    card = f"{torch.cuda.get_device_name()} (nvidia-smi unavailable: {e})"
lines = [f"card: {card}; {a.steps} alternating rounds (DV, JS, NWJ one step each) after {a.warmup} warm-up steps each", "",
         "| B | D | critic | precision | estimator | min ms | median ms | max ms | median / DV | guard | engine ms: stats / dS panel / GEMM |",
         "|---|---|---|---|---|---|---|---|---|---|---|"]
print("\n".join(lines), flush=True)
for B, D, precs in ((65536, 1024, ("fast", "strict")), (4096, 768, ("fast", "strict"))):
    X, Y, sid, W = mo.synthetic_embeddings(B, D, seed=5, dup_frac=0.05, bilinear=True)
    Xd, Yd, Wd, sd = X.bfloat16().to(dev), Y.bfloat16().to(dev), W.bfloat16().to(dev), sid.to(torch.int32).to(dev)
    del X, Y, W
    for prec in precs:
        fns = {e: (lambda e=e: ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd, e, prec, 1.0, True)) for e in EST}
        guard = {}
        for e, fn in fns.items():
            for _ in range(a.warmup):
                out = fn()[0]
            torch.cuda.synchronize()
            guard[e] = float(out[7])
        t = {e: [] for e in EST}
        for _ in range(a.steps):
            for e, fn in fns.items():
                t[e].append(step_ms(fn))
        med = {e: statistics.median(v) for e, v in t.items()}
        for e in EST:
            k = kinds(fns[e])
            eng = " / ".join(f"{ms:.2f} ({n})" for ms, n in k)
            row = (f"| {B} | {D} | bilinear | {prec} | {e} | {min(t[e]):.3f} | {med[e]:.3f} | {max(t[e]):.3f} | "
                   f"{med[e] / med['dv']:.3f} | {guard[e]:g} | {eng} |")
            lines.append(row)
            print(row, flush=True)
    del Xd, Yd, Wd, sd
    torch.cuda.empty_cache()
with open(os.path.join(a.out_dir, "estimator_bench.md"), "w") as f:
    f.write("\n".join(lines) + "\n")
