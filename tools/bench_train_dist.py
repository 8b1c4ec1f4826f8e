#!/usr/bin/env python
"""Multi-GPU training throughput: the step of ``train`` under torchrun (train_dist.train_step: forward + backward of
the rank's slice, deterministic all-reduce, clip_grad_norm_(0.5), Adam), both_bilstm 13x16 hidden 256, dropout 0.5,
one GPU per rank.

For every world size in 1, 2, 4, 8 that the box has GPUs for, torchrun starts one process per GPU and each runs:
* weak scaling: a fixed per-rank batch of 512 and 8 192 sites (global batch = world x that);
* strong scaling: a fixed global batch of 512 and 8 192 sites (per-rank slice = global / world).
Sites/s = global sites per step x steps / the slowest rank's wall clock over a window ended by a device sync.  The
all-reduce is timed with CUDA events around ``dsp_comm_allreduce_f32``; its algorithmic NVLink bytes per rank are
2 (w - 1) / w x 4E (E = gradient elements), reported against the 770 GB/s per direction DESIGN §6 measured.  The card
name and power limit are read in the same run.  Ranks that would have to share a GPU are never started: a world size
the box has no GPUs for reads "not measured".

    python tools/bench_train_dist.py --out profiles/r04_train_dist.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NVLINK_GBS = 770.0
WORLDS = (1, 2, 4, 8)


class TimedExchange:
    """GradientExchange with CUDA events around every all-reduce."""

    def __init__(self, ex):
        self.ex, self.events = ex, []

    def allreduce_(self, params):
        import torch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        self.ex.allreduce_(params)
        b.record()
        self.events.append((a, b))


def run_config(grp, device, global_batch, seconds, warmup):
    import torch
    from deepsignal_plant_b200 import synthetic
    from deepsignal_plant_b200 import train_dist as td
    from deepsignal_plant_b200.models import ModelBiLSTM
    keys = ("kmer", "base_means", "base_stds", "base_signal_lens", "signals")
    dev = torch.device("cuda", device)
    torch.manual_seed(1234)
    torch.cuda.manual_seed(1234 + grp.rank)
    model = ModelBiLSTM(dropout_rate=0.5, seed=grp.rank, trainable=True).cuda(dev).train()
    params = list(model.parameters())
    E = sum(p.numel() for p in params)
    f = synthetic.make_features(global_batch, 13, 16, seed=7)
    data = {k: torch.from_numpy(f[k]).to(dev) for k in keys}
    data["labels"] = torch.randint(0, 2, (global_batch,), generator=torch.Generator().manual_seed(8)).to(dev)
    idx = torch.arange(global_batch, device=dev)
    weight = torch.tensor([1.0, 1.0], device=dev)
    ex = TimedExchange(td.GradientExchange(grp.rank, grp.world, device, E, grp.all_gather_object))
    opt = torch.optim.Adam(params, lr=1e-3)
    try:
        for _ in range(warmup):
            td.train_step(model, params, data, idx, weight, grp.rank, grp.world, ex, opt, keys)
        torch.cuda.synchronize(dev)
        ex.events = []
        grp.barrier()
        steps, t0 = 0, time.perf_counter()
        while True:
            td.train_step(model, params, data, idx, weight, grp.rank, grp.world, ex, opt, keys)
            steps += 1
            if steps % 4 == 0:
                torch.cuda.synchronize(dev)
                # every rank runs the same number of steps: stop when the slowest rank's window is long enough
                if max(grp.all_gather_object(time.perf_counter() - t0)) >= seconds:
                    break
        torch.cuda.synchronize(dev)
        wall = max(grp.all_gather_object(time.perf_counter() - t0))
        ar_ms = sorted(a.elapsed_time(b) for a, b in ex.events)
        ar_med = max(grp.all_gather_object(ar_ms[len(ar_ms) // 2]))
    finally:
        ex.ex.close()
    nbytes = 2 * (grp.world - 1) / grp.world * 4 * E
    return {"world": grp.world, "global_batch": global_batch, "per_rank_batch": global_batch / grp.world, "steps": steps,
            "seconds": wall, "sites_per_s": steps * global_batch / wall, "step_ms": 1e3 * wall / steps,
            "allreduce_ms_median": ar_med, "allreduce_share_of_step": ar_med / (1e3 * wall / steps),
            "gradient_elements": E, "allreduce_nvlink_bytes_per_rank": nbytes,
            "allreduce_gbs": nbytes / (ar_med / 1e3) / 1e9 if grp.world > 1 else None,
            "allreduce_frac_of_770_gbs": nbytes / (ar_med / 1e3) / 1e9 / NVLINK_GBS if grp.world > 1 else None}


def worker(a):
    import torch
    import torch.distributed as dist
    from deepsignal_plant_b200 import freq_dist as fd
    device = fd.join_torchrun("bench_train_dist")
    grp = fd.TorchGroup()
    out = []
    for kind, b in (("weak", 512), ("weak", 8192), ("strong", 512), ("strong", 8192)):
        r = run_config(grp, device, b * grp.world if kind == "weak" else b, a.seconds, a.warmup)
        r["scaling"] = kind
        out.append(r)
        torch.cuda.empty_cache()
    if grp.rank == 0:
        print("RESULT " + json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_dist needs a GPU")
    ndev = torch.cuda.device_count()
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi query failed: %s" % e
    log("cards (%d): %s" % (ndev, q.replace("\n", " | ")))
    rows = {}
    for w in WORLDS:
        if w > ndev:
            rows[str(w)] = "not measured: %d GPU(s) on this box" % ndev
            log("world %d: %s" % (w, rows[str(w)]))
            continue
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(w), "--master-addr",
               "127.0.0.1", "--master-port", str(29800 + w), os.path.abspath(__file__), "--worker", "--seconds", str(a.seconds),
               "--warmup", str(a.warmup)]
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
        if r.returncode != 0:
            raise SystemExit("world %d failed:\n%s\n%s" % (w, r.stdout[-3000:], r.stderr[-5000:]))
        rows[str(w)] = json.loads([l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1][7:])
        for x in rows[str(w)]:
            log("world %d %-6s global batch %5d (%6.0f per rank): %9.0f sites/s, step %.2f ms, all-reduce %.3f ms (%.2f%% of "
                "the step)%s" % (w, x["scaling"], x["global_batch"], x["per_rank_batch"], x["sites_per_s"], x["step_ms"],
                                 x["allreduce_ms_median"], 100 * x["allreduce_share_of_step"],
                                 "" if w == 1 else ", %.1f GB/s = %.1f%% of 770 GB/s" % (x["allreduce_gbs"],
                                                                                        100 * x["allreduce_frac_of_770_gbs"])))
    res = {"cards": q, "model": "both_bilstm 13x16 hidden 256, 3+1 layers, dropout 0.5, Adam, clip 0.5",
           "note": "one GPU per rank; world sizes without enough GPUs are not measured", "worlds": rows}
    log(json.dumps({w: ([{k: x[k] for k in ("scaling", "global_batch", "sites_per_s")} for x in v] if isinstance(v, list) else v)
                    for w, v in rows.items()}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
        with open(os.path.splitext(a.out)[0] + ".log", "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
