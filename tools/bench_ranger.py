"""Ranger's optimizer step on one GPU, for both_bilstm's 49 tensors (4 694 082 parameters), three ways:
  fused        deepsignal_plant_b200.optim.Ranger: one dsp_ranger_step launch per step
  torch_loop   oracle/ranger_oracle.py: the published per-tensor loop of torch ops, as the reference runs it
  torch_adam   torch.optim.Adam(params, lr) as train.py builds it (torch's default multi-tensor implementation)
and training sites/s of the fp32 training kernels with Ranger against Adam, measured by tools/bench_train.py's step
(forward + CrossEntropy backward + clip_grad_norm_(0.5) + optimizer step).

Per optimizer, after 12 warm-up steps (so that rectification and Lookahead have run):
* wall_ms: host clock around --steps back-to-back step() calls ended by a device sync -- what a training loop pays
  when nothing else keeps the GPU busy (host overhead included);
* device_ms: CUDA events around one step() whose launches were queued behind a torch.cuda._sleep, after a 1 GiB write
  that evicts the 126 MB L2, so the work runs from HBM without waiting for the host; the median over --steps.
Algorithmic bytes of the fused step come from the shapes: p, g, exp_avg, exp_avg_sq read and p, exp_avg, exp_avg_sq
written (28 B per element), the centralised gradient written back (4 B per element of a tensor of more than one
dimension) and slow_buffer read and written on the Lookahead step (8 B per element, every 6th step); the HBM fraction
is those bytes over device_ms at the data sheet's 7.7 TB/s.

    python tools/bench_ranger.py --out profiles/r06_ranger_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import bench_train  # noqa: E402
from deepsignal_plant_b200.models import ModelBiLSTM  # noqa: E402
from deepsignal_plant_b200.optim import Ranger  # noqa: E402
from oracle import ranger_oracle  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def step_bytes(shapes, lookahead):
    """Bytes the fused step must move for tensors of ``shapes`` (defaults: GC on every tensor of more than one dim)."""
    b = 0
    for s in shapes:
        n = 1
        for d in s:
            n *= d
        b += n * (28 + (4 if len(s) > 1 else 0) + (8 if lookahead else 0))
    return b


def make(name, params):
    if name == "fused":
        return Ranger(params, lr=1e-3, betas=(0.95, 0.999), eps=1e-5)
    if name == "torch_loop":
        return ranger_oracle.Ranger(params, lr=1e-3, betas=(0.95, 0.999), eps=1e-5)
    return torch.optim.Adam(params, lr=1e-3)


def time_optimizer(name, steps, dev, log):
    torch.manual_seed(1234)
    params = [p.detach().clone() for p in ModelBiLSTM(trainable=True).cuda(dev).parameters()]
    g = torch.Generator(device=dev).manual_seed(7)
    for p in params:
        p.grad = torch.randn(p.shape, device=dev, generator=g) * 1e-3
    opt = make(name, params)
    for _ in range(12):
        opt.step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        opt.step()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3 / steps
    flush = torch.empty(1 << 28, device=dev)                           # 1 GiB
    sleep_cycles = int(max(2.0 * wall_ms, 1.0) * 2e6)                  # ~2x the host's enqueue time at ~2 GHz
    dev_ms = []
    for _ in range(steps):
        flush.zero_()
        torch.cuda._sleep(sleep_cycles)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        opt.step()
        b.record()
        b.synchronize()
        dev_ms.append(a.elapsed_time(b))
    r = {"optimizer": name, "wall_ms": wall_ms, "device_ms": statistics.median(dev_ms), "device_ms_min": min(dev_ms)}
    log("%-10s step(): wall %.3f ms, device %.4f ms (median; min %.4f) over %d steps"
        % (name, wall_ms, r["device_ms"], r["device_ms_min"], steps))
    del opt, params, flush
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--batches", type=int, nargs="+", default=[512, 8192])
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ranger needs a GPU")
    dev = torch.device("cuda:0")
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi query failed: %s" % e
    log("card: %s | %s" % (torch.cuda.get_device_name(dev), q))
    shapes = [tuple(p.shape) for p in ModelBiLSTM(trainable=True).parameters()]
    n_params = sum(int(torch.tensor(s).prod()) for s in shapes)
    plain, look = step_bytes(shapes, False), step_bytes(shapes, True)
    mean_bytes = (5 * plain + look) / 6
    log("both_bilstm: %d tensors, %d parameters; fused step moves %.1f MB (%.1f MB on Lookahead steps, %.1f MB on "
        "average over k = 6)" % (len(shapes), n_params, plain / 1e6, look / 1e6, mean_bytes / 1e6))
    opt = [time_optimizer(name, a.steps, dev, log) for name in ("fused", "torch_loop", "torch_adam")]
    fused = opt[0]
    frac = mean_bytes / (fused["device_ms"] * 1e-3) / HBM_BYTES_PER_S
    log("fused: %.0f GB/s = %.0f%% of 7.7 TB/s (average bytes over device_ms); torch_loop / fused wall %.1fx, "
        "device %.1fx" % (mean_bytes / (fused["device_ms"] * 1e-3) / 1e9, 100 * frac,
                          opt[1]["wall_ms"] / fused["wall_ms"], opt[1]["device_ms"] / fused["device_ms"]))
    runs = []
    for b in a.batches:
        for _ in range(a.rounds):
            for optim in ("Ranger", "Adam"):
                runs.append(bench_train.run_arm("b200_kernels", b, a.seconds, 5, 0.5, dev, log, optim=optim))
    summary = {"fused_step_device_ms": fused["device_ms"], "fused_step_wall_ms": fused["wall_ms"],
               "torch_loop_step_wall_ms": opt[1]["wall_ms"], "torch_loop_step_device_ms": opt[1]["device_ms"],
               "adam_step_wall_ms": opt[2]["wall_ms"], "adam_step_device_ms": opt[2]["device_ms"],
               "fused_hbm_fraction": frac}
    for b in a.batches:
        for optim in ("Ranger", "Adam"):
            summary["train_%s_b%d_sites_per_s" % (optim, b)] = max(r["sites_per_s"] for r in runs
                                                                   if r["batch"] == b and r["optim"] == optim)
    log(json.dumps(summary))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": torch.cuda.get_device_name(dev), "nvidia_smi": q, "n_tensors": len(shapes),
                       "n_params": n_params, "step_bytes": plain, "lookahead_step_bytes": look, "optimizers": opt,
                       "train_runs": runs, "summary": summary}, f, indent=1)
        with open(os.path.splitext(a.out)[0] + ".log", "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
