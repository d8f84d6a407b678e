#!/usr/bin/env python
"""bench.py — critic pairs/sec, fused fwd+bwd MI critic/estimator (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one pass of the hot path (single pass: sampled softmax references -> score tiles -> loss statistics and
both gradient contractions, plus the bilinear projections and their backward) over one batch of synthetic CXR-shaped
embeddings.  N=1: B=65536, D=1024 (the size the metric is quoted on).  N>1: the same global batch sharded by rows,
strong scaling.  Prints ONE JSON line on rank 0.  At N=1 the line also carries a `variants` array (the other
estimators / precisions / BASELINE config 2 / numerically hostile inputs, a few steps each) and a second CPU
baseline entry for BASELINE config 1.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree (it may be read-only)
# NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION; the contract is ONE JSON line there
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"

METRIC = "critic pairs/sec fwd+bwd"
UNIT = "pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=65536, help="global batch B")
    ap.add_argument("--dim", type=int, default=1024)
    ap.add_argument("--critic", default="bilinear", choices=["dot", "bilinear"])
    ap.add_argument("--estimator", default="dv", choices=["dv", "infonce", "infonce_row", "infonce_sym"])
    ap.add_argument("--precision", default="fast", choices=["fast", "strict"])
    ap.add_argument("--cpu-sample-batch", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned to DIR/<name>.npy: the loss "
                         "statistics, dW and a fixed seeded sample of the rows of dX and dY, at most 64 MB in all")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        p = json.load(open(path))
        return {"burst": float(p["bf16_tflops"]), "sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "hbm": float(p["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def workload_name(a):
    return (f"{a.critic} critic + {a.estimator} estimator, fused fwd+bwd, global B={a.batch}, D={a.dim}, "
            f"bf16 operands / fp32 accumulate, precision={a.precision}")


def f_alg(B, D, bilinear):
    """SURVEY 8d: 6 D flops per scored pair (+ the three B x D x D projections of the bilinear critic)."""
    return 6.0 * B * B * D + (6.0 * B * D * D if bilinear else 0.0)


# ------------------------------------------------------------------------------------------- CPU arm
# (the ONLY place bench.py touches oracle/: the reported CPU baseline and the `--impl reference` arm)
def cpu_oracle_step(B, D, critic, estimator, seed=1234):
    """One fwd+bwd of the oracle's matrix form on the host (the reference's pair-form is O(B^4) and
    cannot run at these sizes — BASELINE.md section 2; /root/reference does not travel to the GPU box)."""
    import torch
    from oracle import matrix_oracle as mo
    X, Y, sid, W = mo.synthetic_embeddings(B, D, seed=seed, dup_frac=0.05, bilinear=(critic == "bilinear"))
    inv_tau = 1.0 / math.sqrt(D) if critic == "dot" else 1.0

    def step():
        out = mo.critic_loss(X, Y, sid, W, inv_tau, estimator, dtype=torch.float32, grads=True)
        return float(out["loss"])
    return step


def time_cpu(a, steps, warmup, budget_s=25.0):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B = a.cpu_sample_batch
    step = cpu_oracle_step(B, a.dim, a.critic, a.estimator)
    for _ in range(max(1, warmup)):
        step()
    ts = []
    t_start = time.time()
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
        if budget_s is not None and time.time() - t_start > budget_s:
            break
    t = sum(ts) / len(ts)
    return {"value": B * B / t, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"oracle matrix form (fp32, torch CPU), fwd+bwd, B={B}, D={a.dim}, {a.critic}/{a.estimator}, "
                      f"{len(ts)} steps, {t * 1e3:.0f} ms/step (port @ B={B}: NOT the benchmark's B)",
            "ms_per_step": t * 1e3, "steps": len(ts)}


def time_cpu_config1(budget_s=12.0):
    """BASELINE config 1 as the reference executes it (BASELINE.md section 5): dot-product critic on the explicit pair rows
    built by the growing-torch.cat loop of main_utils.py:99-108, dv_bound_loss, autograd backward; B=32, D=768, fp32."""
    import torch
    from oracle import matrix_oracle as mo
    torch.set_num_threads(os.cpu_count() or 1)
    B, D = 32, 768
    X, Y, sid, _ = mo.synthetic_embeddings(B, D, seed=1, dup_frac=0.0, bilinear=False)
    ids = [str(int(s)) for s in sid]
    ts = []
    t_start = time.time()
    for it in range(8):
        t0 = time.perf_counter()
        mo.critic_loss_pair_form(X, Y, ids, None, 1.0 / math.sqrt(D), "dv", dtype=torch.float32, catloop=True)
        if it > 0:
            ts.append(time.perf_counter() - t0)
        if time.time() - t_start > budget_s and ts:
            break
    ts.sort()
    med = ts[len(ts) // 2]
    return {"value": B * B / med, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"BASELINE config 1: pair form with the reference's torch.cat loop, dot critic + dv, B={B}, D={D}, fp32, "
                      f"fwd+bwd, median of {len(ts)} ({med * 1e3:.0f} ms/step, min {ts[0] * 1e3:.0f} ms)"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = time_cpu(a, a.steps, a.warmup, budget_s=None)        # --steps timed steps, however long they take
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": a.gpus,
        "steps": cb["steps"], "warmup": max(1, a.warmup), "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(a),
                   "note": f"CPU arm: bounded sample of the same workload (oracle port at B={a.cpu_sample_batch}, not {a.batch}: "
                           "the matrix form at the full size needs ~50 GB and ~10 min per step on the host)"},
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons of one GPU, sampled every 50 ms while the benchmark runs.  Reads NVML in-process
    (the library nvidia-smi is built on: clocks.sm, clocks.max.sm, clocks_event_reasons.*, power.draw) — a separate
    `nvidia-smi -lms` process attaches to every GPU of the box and its polls showed up as 1-25 ms stalls inside short
    multi-GPU timed regions; if NVML cannot be loaded in-process the sampler falls back to that process."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []          # (time, sm_mhz, max_mhz, power_w or None, set(reasons))
        self.proc = None
        self.nvml = None
        self.idx = gpu_index
        self.stop_flag = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
            self.th = threading.Thread(target=self._poll_nvml, daemon=True)
            self.th.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read_smi, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        n = self.nvml
        bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown if hasattr(n, "nvmlClocksEventReasonHwSlowdown")
                else n.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonHwThermalSlowdown",
                                               getattr(n, "nvmlClocksThrottleReasonHwThermalSlowdown", 0)),
                "sw_thermal_slowdown": getattr(n, "nvmlClocksEventReasonSwThermalSlowdown",
                                               getattr(n, "nvmlClocksThrottleReasonSwThermalSlowdown", 0)),
                "sw_power_cap": getattr(n, "nvmlClocksEventReasonSwPowerCap",
                                        getattr(n, "nvmlClocksThrottleReasonSwPowerCap", 0))}
        k = 0
        while not self.stop_flag:
            try:
                sm = float(n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM))
                r = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                pw = float(n.nvmlDeviceGetPowerUsage(self.h)) / 1e3 if (k % 4) == 0 else None      # the slow query: every 200 ms
                self.rows.append((time.time(), sm, self.max_mhz, pw, {name for name, b in bits.items() if b and (r & b)}))
            except Exception:
                pass
            k += 1
            time.sleep(0.05)

    def _read_smi(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 8:
                continue
            try:
                self.rows.append((time.time(), float(f[1]), float(f[2]), float(f[3]),
                                  {n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")}))
            except ValueError:
                continue

    def stop(self, t0, t1):
        if self.proc is None and self.nvml is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml / nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for ts, s_mhz, m_mhz, p_w, rs in self.rows:
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(s_mhz); mx.append(m_mhz); reasons |= rs
                if p_w is not None:
                    pw.append(p_w)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "NVML in-process, 50 ms period" if self.nvml is not None else "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------- outputs
DUMP_BYTES = 64 << 20          # what --dump-outputs may write in all


def dump_outputs(path, last, B, off, world, rank):
    """Writes what the timed call returned in its last step as ``path/<name>.npy`` (fp32 / fp64), so that two builds run
    with the same arguments (hence the same seeded inputs) can be compared output for output:
      loss_out (N = 1: the fp64 [8] loss vector) or one fp64 file per entry of the statistics dict (N > 1);
      dX, dY: rows of the global batch, dW: rows of the [D, D] gradient (summed over ranks).
    Each of dX, dY, dW keeps at most a third of DUMP_BYTES: a larger one is cut to a fixed seeded sample of its rows, the
    same rows for the same --batch / --dim, sorted (256 MB each of dX and dY at the default size).  dX and dY are gathered
    from every rank's shard, so every rank calls this; rank 0 writes."""
    import numpy as np
    import torch
    import torch.distributed as dist
    stats, dX, dY, dW = last
    Bl, D = dX.shape
    cap = (DUMP_BYTES - (1 << 20)) // (3 * 4 * D)      # fp32 rows per array; 1 MB left for the statistics and file headers

    def sample(n):
        if n <= cap:
            return torch.arange(n)
        return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:cap].sort().values

    rows = sample(B)
    mine = (rows >= off) & (rows < off + Bl)
    out = {}
    for name, g in (("dX", dX), ("dY", dY)):
        s = torch.zeros(len(rows), D, dtype=g.dtype, device=g.device)
        s[mine.to(g.device)] = g[(rows[mine] - off).to(g.device)]
        if world > 1:
            dist.all_reduce(s)                         # every sampled row is held by exactly one rank, zeros elsewhere
        out[name] = s
    if dW is not None:
        out["dW"] = dW[sample(D).to(dW.device)]
    if isinstance(stats, dict):
        out.update(stats)
    else:
        out["loss_out"] = stats
    if rank != 0:
        return
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        t = torch.as_tensor(t).detach().cpu()
        np.save(os.path.join(path, name + ".npy"), (t if t.dtype == torch.float64 else t.float()).numpy())


# ------------------------------------------------------------------------------------------- GPU arm
def run_ours(a):
    import ctypes

    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        if world == 1 and a.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device(f"cuda:{local_rank}")
    saved_stdout = None
    if world > 1:
        # NCCL prints a version banner on stdout at communicator creation; keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        entry.build()
    if world > 1:
        dist.barrier()
        warm = torch.zeros(1, device=dev)
        dist.all_reduce(warm)
        torch.cuda.synchronize()
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    import mi_b200  # noqa: F401
    from mi_b200 import _lib, ops, synthetic
    from mi_b200 import dist as mdist
    lib = _lib.load()

    # the clock sampler starts HERE, seconds before the timed region: NVML's start-up (attaching to the GPU) stalls it for
    # ~100 ms once — measured as a one-step spike when the sampler was started right before the timing
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get('MI_BENCH_NOSMI'):
        sampler.start()

    B, D = a.batch, a.dim
    assert B % world == 0
    Bl = B // world
    off = rank * Bl
    bilinear = a.critic == "bilinear"
    inv_tau = 1.0 / math.sqrt(D) if not bilinear else 1.0
    # synthetic CXR-shaped embeddings (SURVEY 8d), generated once on the host, rounded to bf16
    X, Y, sid, W = synthetic.synthetic_embeddings(B, D, seed=1234, dup_frac=0.05, bilinear=bilinear)
    Xh = X[off:off + Bl].contiguous().pin_memory()
    Yh = Y[off:off + Bl].contiguous().pin_memory()
    Wh = W.contiguous().pin_memory() if bilinear else None
    sh = sid[off:off + Bl].to(torch.int32).contiguous().pin_memory()
    Xd, Yd = Xh.to(dev).bfloat16(), Yh.to(dev).bfloat16()
    Wd = Wh.to(dev).bfloat16() if bilinear else None
    sd32 = sh.to(dev)
    del X, Y

    out_bufs = (torch.empty(8, dtype=torch.float64, device=dev), torch.empty(Bl, D, device=dev),
                torch.empty(Bl, D, device=dev), torch.empty(D, D, device=dev) if bilinear else None)

    def step_device():
        if world == 1:
            return ops.critic_loss_fwd_bwd(Xd, Yd, Wd, sd32, a.estimator, a.precision, inv_tau, True, out=out_bufs)
        # check_guard=False: no host read inside the timed region (the guard count is checked once after it)
        return mdist.sharded_critic_loss_fwd_bwd(Xd, Yd, Wd, sd32, a.estimator, a.precision, inv_tau, True,
                                                 check_guard=bool(os.environ.get("MI_BENCH_CHECK_GUARD")))

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        marks = []
        for _ in range(steps):
            r = fn()
            if os.environ.get("MI_BENCH_STEPTIMES"):
                marks.append(torch.cuda.Event(enable_timing=True)); marks[-1].record()
        e1.record()
        sync_all()
        t1 = time.time()
        if marks and rank == 0:
            ts = [e0.elapsed_time(m) for m in marks]
            print("per-step ms:", " ".join(f"{b - a:.2f}" for a, b in zip([0.0] + ts[:-1], ts)), file=sys.stderr, flush=True)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), t0, t1, r

    for _ in range(max(3, a.warmup)):
        step_device()
    sync_all()
    lib.mi_set_profiling(0 if os.environ.get('MI_BENCH_NOPROF') else 1)
    ms = (ctypes.c_double * 3)()
    cnt = (ctypes.c_int64 * 3)()
    lib.mi_profile_read(ms, cnt)                      # drain
    l0 = ops.launch_count()
    total_ms, t0, t1, last = timed(step_device, a.steps)
    launches = ops.launch_count() - l0
    lib.mi_profile_read(ms, cnt)
    lib.mi_set_profiling(0)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, last, B, off, world, rank)
    ms_per_step = total_ms / a.steps
    value = B * B / (ms_per_step * 1e-3)
    if world == 1:
        loss_val, guard_rows = float(last[0][0].item()), float(last[0][7].item())
    else:
        loss_val = float(last[0]["loss"].item())
        guard_rows = float(last[0]["guard"].item()) if "guard" in last[0] else 0.0
    # a tripped guard means the timed steps went through the exact repeat (N = 1) or are not valid (N > 1): say so loudly
    sym = a.estimator == "infonce_sym"
    path = "row+column statistics pass + gradient pass (exact references)" if sym else "single pass, sampled softmax references"
    if guard_rows != 0.0 and not sym:
        path += (" -> guard tripped: the exact repeat ran inside every timed step" if world == 1 else
                 " -> guard tripped and NOT acted on (check_guard=False in the timed loop): INVALID NUMBER")

    # ---- end to end through the public API with HOST buffers (H2D + D2H inside the timed region).
    # Every step: the step's inputs (bf16 embeddings, W, study ids) cross PCIe from pinned host memory, the loss comes back to
    # the host; the gradients stay on the device, where the encoders' backward consumes them (SURVEY 8f-4).  N = 1 also times
    # the full host round trip of round 1 (fp32 host embeddings in, fp32 gradients back out) as `roundtrip_fp32`.
    e2e = None
    if not a.no_e2e:
        Xp, Yp = Xh.bfloat16().pin_memory(), Yh.bfloat16().pin_memory()
        Wp = Wh.bfloat16().pin_memory() if bilinear else None
        n_in = 2 * Bl * D * 2 + (D * D * 2 if bilinear else 0) + Bl * 4
        P = lambda t: None if t is None else ctypes.c_void_p(t.data_ptr())
        roundtrip = None
        if world == 1:
            crit, est, prec = (1 if bilinear else 0), ops.ESTIMATOR[a.estimator], ops.PRECISION[a.precision]
            nbytes = lib.mi_critic_host_scratch_bytes(B, D, crit, est, prec, 1)
            scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            loss_h = torch.zeros(8, dtype=torch.float64).pin_memory()
            gX, gY = torch.empty(Bl, D, device=dev), torch.empty(Bl, D, device=dev)
            gW = torch.empty(D, D, device=dev) if bilinear else None
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

            def step_host():
                st = lib.mi_critic_loss_fwd_bwd_from_host(P(Xp), P(Yp), P(Wp), P(sh), 1, B, D, crit, est, prec, inv_tau,
                                                          P(loss_h), P(gX), P(gY), P(gW), P(scratch), nbytes, stream)
                if st != 0:
                    raise RuntimeError(lib.mi_status_string(st).decode())
                return loss_h

            dXh, dYh = torch.empty(Bl, D).pin_memory(), torch.empty(Bl, D).pin_memory()
            dWh = torch.empty(D, D).pin_memory() if bilinear else None

            def step_roundtrip():
                st = lib.mi_critic_loss_fwd_bwd_host(P(Xh), P(Yh), P(Wh), P(sh), B, D, crit, est, prec, inv_tau,
                                                     P(loss_h), P(dXh), P(dYh), P(dWh), P(scratch), nbytes, stream)
                if st != 0:
                    raise RuntimeError(lib.mi_status_string(st).decode())
                return loss_h
            drain = lambda: None
        else:
            # N > 1: the user-level loop around the public sharded call, software-pipelined the way a training loop overlaps
            # its data loader: step n+1's host->device copies run on a copy stream under step n's compute and the loss of
            # step n is read (a device->host read of the step's result, every step) after step n+1 has been enqueued.
            s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            main = torch.cuda.current_stream()
            bf = dict(dtype=torch.bfloat16, device=dev)
            dbuf = [(torch.empty(Bl, D, **bf), torch.empty(Bl, D, **bf), torch.empty(D, D, **bf) if bilinear else None,
                     torch.empty(Bl, dtype=torch.int32, device=dev), torch.cuda.Event(), torch.cuda.Event()) for _ in range(2)]
            loss_pin = [torch.zeros(1, dtype=torch.float64).pin_memory() for _ in range(2)]
            state = {"n": 0, "pending": None}

            def upload(slot):
                x, y, w, s_, ev_in, ev_used = dbuf[slot]
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_used)                   # the previous user of this slot has consumed it
                    x.copy_(Xp, non_blocking=True); y.copy_(Yp, non_blocking=True); s_.copy_(sh, non_blocking=True)
                    if bilinear:
                        w.copy_(Wp, non_blocking=True)
                    ev_in.record(s_in)

            def step_host():
                n = state["n"]
                slot = n & 1
                if n == 0:
                    upload(0)
                upload(slot ^ 1)                               # next step's inputs cross PCIe under this step's compute
                x, y, w, s_, ev_in, ev_used = dbuf[slot]
                main.wait_event(ev_in)
                # the public call with its default guard handling: the host reads the merged guard count as soon as the
                # score tiles are done and would repeat the step on the exact path
                out, dX, dY, dW = mdist.sharded_critic_loss_fwd_bwd(x, y, w, s_, a.estimator, a.precision, inv_tau, True)
                ev_used.record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_used)
                    loss_pin[slot].copy_(out["loss"].reshape(1), non_blocking=True)
                    ev_out = torch.cuda.Event(); ev_out.record(s_out)
                out["loss"].record_stream(s_out)
                prev = state["pending"]
                state["pending"] = (ev_out, slot)
                state["n"] = n + 1
                if prev is not None:                           # read the PREVIOUS step's loss: it is (nearly) there already
                    prev[0].synchronize()
                    return loss_pin[prev[1]]
                return loss_pin[slot]

            def drain():
                if state["pending"] is not None:
                    state["pending"][0].synchronize()
                    state["pending"] = None
                main.wait_stream(s_out); main.wait_stream(s_in)
        step_host(); step_host()
        drain()
        e_steps = max(2, min(a.steps, 5)) if world == 1 else max(4, a.steps)

        def timed_host(fn, steps):
            def run():
                r = None
                for _ in range(steps):
                    r = fn()
                drain()
                return r
            return timed(run, 1)[0] / steps
        e_ms = timed_host(step_host, e_steps)
        if world == 1:
            step_roundtrip()
            rt_ms = timed_host(step_roundtrip, 3)
            n_bd, n_dd = Bl * D * 4, D * D * 4
            roundtrip = {"ms_per_step": rt_ms, "value": B * B / (rt_ms * 1e-3), "unit": UNIT,
                         "h2d_bytes_per_step": 2 * n_bd + (n_dd if bilinear else 0) + Bl * 4,
                         "d2h_bytes_per_step": 2 * n_bd + (n_dd if bilinear else 0) + 64,
                         "api": "mi_critic_loss_fwd_bwd_host (fp32 host embeddings in, fp32 gradients back to the host)"}
        e2e = {"value": B * B / (e_ms * 1e-3), "unit": UNIT, "ms_per_step": e_ms,
               "h2d_bytes_per_step": world * n_in, "d2h_bytes_per_step": world * 64,
               "api": ("mi_critic_loss_fwd_bwd_from_host (C ABI: pinned bf16 host embeddings in, loss to the host, gradients stay on "
                       "the device)" if world == 1 else
                       "mi_b200.dist.sharded_critic_loss_fwd_bwd on pinned bf16 host shards, copies software-pipelined across "
                       "steps on a copy stream (loss read one step late; gradients stay on the device)")}
        if roundtrip:
            e2e["roundtrip_fp32"] = roundtrip

    # ---- variants (N = 1): the other estimators / precisions, BASELINE config 2, numerically hostile inputs
    variants = []
    if world == 1 and not a.no_variants:
        pk_v = peaks()

        def run_variant(name, Xv, Yv, Wv, sv, est, prec, itau, steps=5):
            Bv, Dv = Xv.shape
            bufs = (torch.empty(8, dtype=torch.float64, device=dev), torch.empty(Bv, Dv, device=dev),
                    torch.empty(Bv, Dv, device=dev), None if Wv is None else torch.empty(Dv, Dv, device=dev))
            fn = lambda: ops.critic_loss_fwd_bwd(Xv, Yv, Wv, sv, est, prec, itau, True, out=bufs)
            for _ in range(3):
                fn()
            t_ms, _, _, r = timed(fn, steps)
            t_ms /= steps
            fa_v = f_alg(Bv, Dv, Wv is not None)
            lo = r[0].cpu()
            variants.append({"name": name, "B": Bv, "D": Dv, "critic": "dot" if Wv is None else "bilinear", "estimator": est,
                             "precision": prec, "ms_per_step": t_ms, "pairs_per_s": Bv * Bv / (t_ms * 1e-3),
                             "f_alg_tflops": fa_v / (t_ms * 1e-3) / 1e12,
                             "frac_of_sustained_peak": fa_v / (t_ms * 1e-3) / 1e12 / pk_v["sustained"],
                             "frac_of_burst_peak": fa_v / (t_ms * 1e-3) / 1e12 / pk_v["burst"],
                             "loss": float(lo[0]), "guard_rows": float(lo[7]),
                             "path": ("exact repeat (guard tripped)" if float(lo[7]) != 0.0 else
                                      ("statistics + gradient pass" if est == "infonce_sym" else "single pass"))})

        run_variant("config3 symmetric InfoNCE, fast", Xd, Yd, Wd, sd32, "infonce_sym", "fast", inv_tau)
        run_variant("config3 symmetric InfoNCE, strict", Xd, Yd, Wd, sd32, "infonce_sym", "strict", inv_tau, steps=3)
        run_variant("DV, strict (fp32-accumulate mode)", Xd, Yd, Wd, sd32, "dv", "strict", inv_tau, steps=3)
        run_variant("row InfoNCE, fast", Xd, Yd, Wd, sd32, "infonce_row", "fast", inv_tau)
        # numerically hostile inputs at the full size (VERDICT r1 #1c): must stay on the single pass, guard clear
        if bilinear:
            run_variant("stress: scores x 8 (nearly one-hot softmax)", Xd, Yd, (8.0 * Wd.float()).bfloat16(), sd32, "dv", "fast", inv_tau)
            gw = torch.Generator().manual_seed(11)
            Wn = (torch.eye(D) + 0.1 * torch.randn(D, D, generator=gw) / math.sqrt(D)).to(dev).bfloat16()
            run_variant("stress: unnormalised embeddings, W = I + noise, inv_tau = 1", Xd, Yd, Wn, sd32, "dv", "fast", 1.0)
            run_variant("stress: unnormalised embeddings, row InfoNCE", Xd, Yd, Wn, sd32, "infonce_row", "fast", 1.0)
        # BASELINE config 2: bilinear + InfoNCE, B = 4096, D = 768
        X2, Y2, s2, W2 = synthetic.synthetic_embeddings(4096, 768, seed=2, dup_frac=0.05, bilinear=True)
        X2, Y2, W2, s2 = X2.to(dev).bfloat16(), Y2.to(dev).bfloat16(), W2.to(dev).bfloat16(), s2.to(torch.int32).to(dev)
        run_variant("config2 bilinear + InfoNCE (reference form)", X2, Y2, W2, s2, "infonce", "fast", 1.0, steps=20)
        run_variant("config2 bilinear + symmetric InfoNCE", X2, Y2, W2, s2, "infonce_sym", "fast", 1.0, steps=20)
        # the same step replayed from a CUDA graph (ops.GraphedCriticStep): at this size the direct call is host-launch bound
        gstep = ops.GraphedCriticStep(4096, 768, bilinear=True, estimator="infonce", precision="fast", inv_tau=1.0, device=dev)
        for _ in range(3):
            gstep(X2, Y2, W2, s2)
        g_ms, _, _, gr = timed(lambda: gstep(X2, Y2, W2, s2), 20)
        g_ms /= 20
        variants.append({"name": "config2 bilinear + InfoNCE, CUDA-graph replay (incl. the copies into the graph's static inputs)",
                         "B": 4096, "D": 768, "critic": "bilinear", "estimator": "infonce", "precision": "fast", "ms_per_step": g_ms,
                         "pairs_per_s": 4096 * 4096 / (g_ms * 1e-3), "f_alg_tflops": f_alg(4096, 768, True) / (g_ms * 1e-3) / 1e12,
                         "frac_of_sustained_peak": f_alg(4096, 768, True) / (g_ms * 1e-3) / 1e12 / pk_v["sustained"],
                         "frac_of_burst_peak": f_alg(4096, 768, True) / (g_ms * 1e-3) / 1e12 / pk_v["burst"],
                         "loss": float(gr[0][0]), "guard_rows": float(gr[0][7]), "path": "single pass (exact references), graph replay"})

        # the reference's own critic (main_utils.py:77: make_mlp(1536, [1024, 512]) on every pair) + DV, B = 4096
        Bm, Dm, H1m, H2m = 4096, 768, 1024, 512
        gm = torch.Generator().manual_seed(5)
        Xm = torch.relu(torch.randn(Bm, Dm, generator=gm)).to(dev)
        Ym = torch.tanh(torch.randn(Bm, Dm, generator=gm)).to(dev)
        sm = torch.arange(Bm, dtype=torch.int32, device=dev)
        torch.manual_seed(1)
        mlp = mi_b200.FusedMLPCritic(Dm, (H1m, H2m)).to(dev)
        pm = tuple(t.detach() for t in (mlp[0].weight, mlp[0].bias, mlp[2].weight, mlp[2].bias, mlp[4].weight, mlp[4].bias))
        fa_m = 3 * 2.0 * Bm * Bm * H1m * H2m + 3 * 2.0 * (2 * Bm) * Dm * H1m
        for prec in ("fast", "strict"):
            fn = lambda: ops.mlp_critic_loss_fwd_bwd(Xm, Ym, pm, sm, "dv", prec, True, False)
            for _ in range(2):
                fn()
            m_ms, _, _, mr = timed(fn, 3)
            m_ms /= 3
            lo = mr[0].cpu()
            variants.append({"name": "concat-MLP critic make_mlp(1536, [1024, 512]) + DV, " + prec, "B": Bm, "D": Dm, "critic": "mlp",
                             "estimator": "dv", "precision": prec, "ms_per_step": m_ms, "pairs_per_s": Bm * Bm / (m_ms * 1e-3),
                             "f_alg_tflops": fa_m / (m_ms * 1e-3) / 1e12,
                             "frac_of_sustained_peak": fa_m / (m_ms * 1e-3) / 1e12 / pk_v["sustained"],
                             "frac_of_burst_peak": fa_m / (m_ms * 1e-3) / 1e12 / pk_v["burst"],
                             "loss": float(lo[0]), "guard_rows": float(lo[7]),
                             "path": "two-pass repeat (guard tripped)" if float(lo[7]) != 0.0 else "single pass"})

    launches_t = torch.tensor([launches], device=dev, dtype=torch.int64)
    if world > 1:
        dist.all_reduce(launches_t)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")      # written from the latest ncu --set full capture
    if os.path.isfile(tpath):
        tj = json.load(open(tpath))
        c = tj["config"]
        if (c["global_batch"], c["dim"], c["critic"], c["estimator"], c["precision"], c["n_gpus"]) == \
                (B, D, a.critic, a.estimator, a.precision, world):
            traffic = tj["bytes_per_step"]
    fa = f_alg(B, D, bilinear)
    strict = a.precision == "strict"
    # executed tensor flops: the single pass computes the scores once (+ the ~1 % column sample of the references);
    # the symmetric estimator adds ONE combined row+column statistics pass (2 B^2 D); two dS x operand contractions
    # 2 B^2 D each; strict mode adds the hi/lo segments of T and of the dS panel
    n_stats = 1 if sym else 0
    if strict:
        s_mult = 2.0 if bilinear else 1.0
        f_exec = (n_stats * s_mult + s_mult + 2 * (3 if (bilinear or not sym) else 2)) * 2.0 * float(B) * B * D
    else:
        f_exec = (n_stats + 1 + 2) * 2.0 * float(B) * B * D
    f_exec += (6.0 * B * D * D if bilinear else 0.0)
    ach = fa / (ms_per_step * 1e-3) / 1e12 / world           # per GPU
    kinds = ["score_stats", "ds_panel", "gemm"]
    by_kernel = {k: {"ms_per_step": ms[i] / a.steps, "launches_per_step": cnt[i] / a.steps} for i, k in enumerate(kinds)}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(3, a.warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(a), "global_batch": B, "dim": D, "critic": a.critic,
                   "estimator": a.estimator, "precision": a.precision, "parallelism": f"row-sharded x{world}",
                   "l2": "inputs (2 x %d MB bf16 + >1 GB dS panel per pass) exceed the 126 MB L2; no flush needed" % (B * D * 2 >> 20),
                   "loss": loss_val, "guard_rows": guard_rows, "path": path},
        "roofline": {"bound": "tensor", "achieved": ach, "peak": pk["sustained"], "unit": "TFLOP/s",
                     "frac": ach / pk["sustained"], "traffic": traffic,
                     "traffic_note": "DRAM bytes per step summed over the step's launches (ncu capture in profiles/), "
                                     "algorithmic bytes 0.54e9: the path is tensor-bound; the bf16 dS panel is STREAMED THROUGH HBM "
                                     "panel by panel (SURVEY 7.3-d) - that staging is the extra traffic",
                     "peak_kind": "sustained bf16 (kernel timed inside a long step), " + pk["source"],
                     "frac_of_burst_peak": ach / pk["burst"], "burst_peak": pk["burst"],
                     "algorithmic_flops_per_step": fa, "executed_flops_per_step": f_exec,
                     "executed_tflops": f_exec / (ms_per_step * 1e-3) / 1e12 / world,
                     "kernel": "tile_engine_kernel (all launches of one step; per-kind CUDA-event times in by_kernel)",
                     "by_kernel": by_kernel},
        "clocks": clocks, "gpu_launches": int(launches_t.item()),
    }
    if e2e:
        line["e2e"] = e2e
    if variants:
        line["variants"] = variants
    if world == 1 and not a.no_cpu_baseline:
        cb = time_cpu(a, 3, 1, budget_s=25.0)
        line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline"]["config1"] = time_cpu_config1()
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
