#!/usr/bin/env python
"""Benchmark of the ModelBiLSTM hot path (BASELINE.json metric: classified sites/s,
both_bilstm bn13_sn16 hidden 256, batch 65536).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision fp16|fp32] [--dump-outputs DIR]

One "step" = one batch of 65 536 synthetic sites through the forward pass.  Prints ONE JSON
line (rank 0).  See DESIGN.md section "Measurement" for what every key means.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "classified sites/sec (ModelBiLSTM both_bilstm bn13_sn16 hidden 256)"
UNIT = "sites/s"
BATCH = 65536
OUT_BYTES_PER_SITE = 4 * 2 * 2 + 4


def flops_per_site(module="both_bilstm", T=13, S=16, H=256, E=4, layers1=3, C=2):
    """Algorithmic FLOPs (2 x MAC, no padding) of one site: (whole forward, recurrent layers only).
    both_bilstm 13x16 -> 118 447 104 (SURVEY.md section 8d)."""
    def lstm(K, Hh):
        return 2 * T * 4 * Hh * (K + Hh)
    hs = H // 2 if module == "both_bilstm" else (H if module == "seq_bilstm" else 0)
    hg = H - H // 2 if module == "both_bilstm" else (H if module == "signal_bilstm" else 0)
    rec = (lstm(E + 3, hs) if hs else 0) + (lstm(S, hg) if hg else 0) + lstm(H, H) + (layers1 - 1) * lstm(2 * H, H)
    dense = T * 2 * hs * hs + T * 2 * hg * hg + 2 * H * H + H * C
    return 2 * (rec + dense), 2 * rec


FLOP_PER_SITE, FLOP_PER_SITE_RECURRENT = flops_per_site()
assert FLOP_PER_SITE == 118447104
IN_BYTES_PER_SITE = 4 * (4 * 13 + 13 * 16)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=float(d["bf16_tflops_sustained"]), tflops_burst=float(d["bf16_tflops"]),
                    hbm=float(d["hbm_gbs"]), source="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(tflops=1400.0, tflops_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def traffic_of_dominant_kernel(batch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel (lstm_comb layer 1,
    layer_kernel<8,256,LSTM>) from the committed `ncu --set full` capture, scaled to this batch.  The capture
    (profiles/roofline_traffic.json) carries the sha256 of the kernel source it was taken from: when
    csrc/kernels_tc.cu has changed since, the number is stale and this returns (None, {"reason": ...})."""
    import hashlib
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(p):
        return None, {"reason": "no ncu --set full capture recorded (profiles/roofline_traffic.json)"}
    d = json.load(open(p))
    src = os.path.join(ROOT, "deepsignal_plant_b200", "csrc", "kernels_tc.cu")
    sha = hashlib.sha256(open(src, "rb").read()).hexdigest()
    if d.get("kernels_tc_sha256") != sha:
        return None, {"reason": "profiles/roofline_traffic.json was captured from another version of csrc/kernels_tc.cu "
                                "(%s..., now %s...): re-capture with tools/gpu_traffic.sh" % (str(d.get("kernels_tc_sha256"))[:12], sha[:12]),
                      "stale_dram_bytes_per_site": d["dram_bytes_per_site"], "algorithmic_bytes_per_site": d["algorithmic_bytes_per_site"]}
    return d["dram_bytes_per_site"] * batch, {"unit": "B per launch", "kernel": d["kernel"], "source": d["source"],
                                              "algorithmic_bytes_per_launch": d["algorithmic_bytes_per_site"] * batch}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        pmax = max(float(r[2]) for r in self.rows)
        loaded = [r for r in self.rows if float(r[2]) >= 0.6 * pmax] or self.rows     # samples taken under load
        sm = sorted(float(r[0]) for r in loaded)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        watts = [float(r[2]) for r in loaded]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "samples": len(self.rows), "samples_under_load": len(loaded),
                "power_w_max": max(float(r[2]) for r in self.rows), "power_w_mean_under_load": sum(watts) / len(watts), "reasons": reasons}


def make_pool(n_buffers, batch, seed=0, T=13, S=16):
    """`n_buffers` distinct batches: one generated pool, rolled copies (distinct bytes, so the
    cycled inputs exceed L2: 4 x 68 MB > 126 MB)."""
    from deepsignal_plant_b200 import synthetic
    base = synthetic.make_features(batch, T, S, seed=seed)
    keys = ("kmer", "base_means", "base_stds", "base_signal_lens", "signals")
    return [tuple(np.ascontiguousarray(np.roll(base[k], 977 * b, axis=0)) for k in keys) for b in range(n_buffers)]


DUMP_MAX_BYTES = 60_000_000          # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(directory, arrays, max_bytes=DUMP_MAX_BYTES):
    """Write each (name, tensor) of `arrays` (equal first dimension) as directory/<name>.npy in float32.  When they
    would take more than `max_bytes` together, every array is cut to the same fixed, seeded sample of rows (ascending)
    and the sampled row indices are written as directory/rows.npy (float64), all within `max_bytes`."""
    import torch
    os.makedirs(directory, exist_ok=True)
    n = arrays[0][1].shape[0]
    row_bytes = sum(4 * (t.numel() // n) for _, t in arrays)
    if n * row_bytes > max_bytes:
        rows = np.sort(np.random.default_rng(0).choice(n, max_bytes // (row_bytes + 8), replace=False))
        np.save(os.path.join(directory, "rows.npy"), rows.astype(np.float64))
        idx = torch.from_numpy(rows)
        arrays = [(name, t.index_select(0, idx.to(t.device))) for name, t in arrays]
    for name, t in arrays:
        np.save(os.path.join(directory, name + ".npy"), t.float().cpu().numpy())


def port_baseline_run(sites, threads):
    """The reference's forward restated on torch's own CPU operators (oracle/torch_oracle.py: nn.LSTM -> oneDNN,
    nn.Linear, softmax), driven like `_call_mods` drives it -- batches of 512, fresh torch.randn states per batch,
    argmax -- WITHOUT the reference's list -> tensor conversion and per-site text loop, i.e. an upper bound on the
    reference's CPU speed.  oracle/ is used here as the baseline only.  Returns (sites/s, seconds)."""
    import torch
    from deepsignal_plant_b200 import synthetic
    from deepsignal_plant_b200.models import ModelBiLSTM
    from oracle import model_oracle, torch_oracle
    torch.set_num_threads(threads)
    cfg = model_oracle.make_cfg()
    torch.manual_seed(1234)
    sd = {k: v.detach().clone() for k, v in ModelBiLSTM(13, 16, 3, 1, 2, 0, 256, 16, 4, True, True).state_dict().items()}
    feats = {k: torch.from_numpy(v) for k, v in synthetic.make_features(sites, 13, 16, seed=0).items()}
    t0 = time.perf_counter()
    torch_oracle.call_mods_batches(sd, cfg, feats, 512)
    dt = time.perf_counter() - t0
    return sites / dt, dt


def reference_available():
    from oracle import ref_import
    return ref_import.available()


def reference_callmods_run(sites, threads, repeat=1, timeout=1500):
    """The UNMODIFIED reference (oracle/_ref, installed by oracle/build_ref.py) on the host cores: its own
    ModelBiLSTM + `_call_mods` (call_modifications.py:130-192: nested lists -> FloatTensor, forward with fresh
    torch.randn states, .numpy(), sklearn accuracy, per-site renormalise / round / str-join loop), batch 512, in a
    subprocess with CUDA hidden (the reference picks CPU vs CUDA at import).  Returns the list of wall-clock
    seconds of `repeat` calls over `sites` sites."""
    from oracle import ref_import
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_ref_callmods.py"), "--n", str(sites), "--batch", "512",
           "--threads", str(threads), "--repeat", str(repeat), "--time"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=ref_import.cpu_env(), cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError("reference _call_mods run failed: " + r.stderr[-800:])
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["all_seconds"]


def reference_callfreq_run(records, timeout=900):
    """The unmodified reference's calculate_mods_frequency (call_mods_freq.py:29-74) on `records` synthetic
    per-read calls, one Python process (its default mode).  Returns records/s."""
    from oracle import ref_import
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_ref_callfreq.py"), "--records", str(records)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=ref_import.cpu_env(), cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError("reference calculate_mods_frequency run failed: " + r.stderr[-800:])
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["records_per_s"]


def reference_arm(args, rank, world):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # bounded sample per step: the whole run (K steps) stays within a few minutes at ~2 k sites/s
    sample = int(min(8192, max(512, (120000 // max(args.steps, 1)) // 512 * 512)))
    if reference_available():
        secs = reference_callmods_run(sample, cores, repeat=args.steps + max(0, min(args.warmup, 1)))[-args.steps:]
        kind = "reference"
        what = ("the UNMODIFIED reference (oracle/_ref): its ModelBiLSTM + _call_mods (list -> tensor, forward, per-site text loop), "
                "torch CPU fp32, %d threads" % cores)
    else:
        for _ in range(max(0, min(args.warmup, 1))):
            port_baseline_run(512, cores)
        secs = [port_baseline_run(sample, cores)[1] for _ in range(args.steps)]
        kind = "port"
        what = "oracle/torch_oracle.py (the reference forward on the same torch CPU operators; oracle/_ref is not built), %d threads" % cores
    t_all = sum(secs)
    value = sample * args.steps / t_all
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_all / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "both_bilstm bn13_sn16 h256 inference, batch 65536 (config 2)",
                       "note": "reference CPU path: %s; each step = %d-site sample in batches of 512" % (what, sample)},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": "%d sites per step, batch 512, %s" % (sample, what)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def command_line_run(sites, timeout_s=150, extra=()):
    """The real `call_mods` command line (python -m deepsignal_plant_b200 call_mods -i features.dspf ...) on a synthetic
    binary feature file of `sites` sites, timed in a FRESH process by tools/bench_cli.py --binary: interpreter start,
    imports, CUDA context, checkpoint load, the stream, the calls file.  Never raises: a failure is reported in the object."""
    import re
    import tempfile
    try:
        where = ["--dir", "/dev/shm", "--out-dir", tempfile.gettempdir()] if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else []
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_cli.py"), "--binary", "--sites", str(int(sites))] + where + list(extra),
                           capture_output=True, text=True, timeout=timeout_s, cwd=ROOT)
        rows = [l for l in r.stdout.splitlines() if l.startswith("{")]
        if r.returncode != 0 or not rows:
            return {"unavailable": ((r.stderr or "") + (r.stdout or ""))[-300:].replace("\n", " | ")}
        d = json.loads(rows[-1])
        stream = None
        for l in d.get("host_breakdown") or []:
            m = re.search(r"call_mods_stream: (\d+) sites in ([0-9.]+) seconds", l)
            if m:
                stream = {"sites_per_s": int(m.group(1)) / max(float(m.group(2)), 1e-9), "seconds": float(m.group(2))}
        return {"metric": "call_mods command line, binary feature file -> calls file, wall clock of a fresh process (sites/s)",
                "value": d["value"], "unit": UNIT, "sites": d["sites"], "seconds": d["seconds"], "lines_written": d["lines_written"],
                "stream": stream, "startup_s": (d["seconds"] - stream["seconds"]) if stream else None, "input_bytes": d["input_bytes"], "output_bytes": d["output_bytes"], "host_threads": d["host_threads"],
                "host_breakdown": d.get("host_breakdown"), "power_w_mean_under_load": (d.get("clocks") or {}).get("power_w_mean_under_load"),
                "note": "start-up (interpreter, import torch, CUDA context, model load: ~3 s) is inside `seconds`; `stream` = first batch in "
                        "to last batch out; the 100 M-site run of the same command is profiles/r02_cli_binary_100M.json"}
    except Exception as e:                                  # noqa: BLE001 -- the bench line must not depend on this extra
        return {"unavailable": repr(e)[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("DSP_B200_PRECISION", "fp16"), choices=["fp16", "fp32"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--buffers", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-freq", dest="no_freq", action="store_true", help="skip the call_freq measurement (the `freq` object)")
    ap.add_argument("--freq-records", dest="freq_records", type=int, default=50_000_000, help="call_freq records per GPU")
    ap.add_argument("--no-cli", dest="no_cli", action="store_true", help="skip the command-line measurement (the `cli` object)")
    ap.add_argument("--cli-sites", dest="cli_sites", type=int, default=64_000_000, help="sites of the command-line measurement")
    ap.add_argument("--meas-skip-y", action="store_true",
                    help="measurement only (INVALID as a result): after warm-up, skip the inter-layer activation stores")
    # BASELINE.json configs[3]: the other model variants (not the headline line)
    ap.add_argument("--module", default="both_bilstm", choices=["both_bilstm", "seq_bilstm", "signal_bilstm"])
    ap.add_argument("--seq_len", type=int, default=13)
    ap.add_argument("--signal_len", type=int, default=16)
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0: logits, probs, labels) as DIR/<name>.npy in float32, "
                         "at most 64 MB (a fixed, seeded sample of rows, listed in DIR/rows.npy, above that); inputs, weights "
                         "and initial states are seeded, so equal arguments give equal inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the device forward: it needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.steps is None:
        args.steps = 100 if args.precision == "fp16" else 4
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from deepsignal_plant_b200.models import ModelBiLSTM
    from deepsignal_plant_b200 import _native
    import ctypes as C

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)

    torch.manual_seed(1234)
    T_, S_ = args.seq_len, args.signal_len
    flop_site, flop_rec = flops_per_site(args.module, T_, S_)
    in_bytes_site = 4 * ((4 * T_ if args.module != "signal_bilstm" else 0) + (T_ * S_ if args.module != "seq_bilstm" else 0))
    headline = (args.module, T_, S_) == ("both_bilstm", 13, 16)
    model = ModelBiLSTM(T_, S_, 3, 1, 2, 0, 256, 16, 4, True, True, module=args.module, device=local,
                        precision=args.precision, max_batch=args.batch, seed=rank).cuda(local).eval()
    pool = make_pool(args.buffers, args.batch, seed=rank, T=T_, S=S_)
    dev_pool = [tuple(torch.from_numpy(a).to(dev) for a in b) for b in pool]
    pin_pool = [tuple(torch.from_numpy(a).pin_memory() for a in b) for b in pool]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up -------------------------------------------------------------------
    for i in range(W):
        model(*dev_pool[i % len(dev_pool)])
    torch.cuda.synchronize()
    L = _native.lib()

    if args.meas_skip_y:
        # only the measurement build (DSP_B200_VARIANT=skipy DSP_B200_DEFINES=-DDSP_MEAS_SKIP_Y, loaded through
        # DSP_B200_LIB) reads this; the shipped library has no result-changing switch
        assert "skipy" in os.path.basename(_native.LIB_PATH), "--meas-skip-y needs the skipy variant build (see tools/gpu_variants.sh)"
        os.environ["DSP_B200_SKIP_Y_NOW"] = "1"
    # ---- timed region: inputs resident in HBM ------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:                       # one sampler per job: rank 0's GPU stands for the box
        sampler.start()
    _native.check(L.dsp_set_timing(model._handle, 1))
    launches0 = model.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kern_ms, kern_launches = 0.0, 0
    barrier()
    ev0.record()
    for i in range(args.steps):
        out = model(*dev_pool[i % len(dev_pool)])
    ev1.record()
    barrier()
    launches = model.launch_count() - launches0
    ms = ev0.elapsed_time(ev1)
    # recurrent-layer kernel time of the LAST step (events recorded on the launching stream)
    t = C.c_float()
    cnt = C.c_int64()
    _native.check(L.dsp_get_timing(model._handle, 1, C.byref(t), C.byref(cnt)))
    kern_ms, kern_launches = float(t.value), int(cnt.value)
    class_ms = {}
    for cls, name in ((0, "assemble"), (1, "recurrent_comb"), (4, "recurrent_branch"), (2, "fc"), (3, "head")):
        _native.check(L.dsp_get_timing(model._handle, cls, C.byref(t), C.byref(cnt)))
        class_ms[name] = round(float(t.value), 4)
        if cls == 4:
            kern_ms += float(t.value)
            kern_launches += int(cnt.value)
    _native.check(L.dsp_set_timing(model._handle, 0))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [("logits", out[0]), ("probs", out[1]), ("labels", model.last_labels)])
    del out

    # ---- e2e: host buffers through the public host API, H2D + D2H inside ----------------
    # Every step's inputs start in pinned host memory and its logits/probs/labels end in pinned
    # host memory; submissions are pipelined two deep (ModelBiLSTM.submit_host / wait_host), the
    # way a call_mods worker streams successive feature batches.
    e2e_steps = args.steps
    outs = [(torch.empty((args.batch, 2), dtype=torch.float32).pin_memory(),
             torch.empty((args.batch, 2), dtype=torch.float32).pin_memory(),
             torch.empty((args.batch,), dtype=torch.int32).pin_memory()) for _ in range(2)]

    def e2e_loop(k):
        prev = None
        for i in range(k):
            tk = model.submit_host(*pin_pool[i % len(pin_pool)], *outs[i & 1])
            if prev is not None:
                model.wait_host(prev)
            prev = tk
        model.wait_host(prev)
    e2e_loop(3)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(e2e_steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert float(outs[(e2e_steps - 1) & 1][1].sum()) > 0      # results really arrived on the host
    clocks = sampler.summary() if rank == 0 else None      # sampled over both timed regions

    tt = torch.tensor([ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(tt[0]), float(tt[1])
    value = world * args.batch * args.steps / (ms * 1e-3)
    e2e_value = world * args.batch * e2e_steps / (e2e_ms * 1e-3)

    pk = peaks()
    achieved = (flop_rec * args.batch / (kern_ms * 1e-3) / 1e12) if kern_ms > 0 else None
    traffic = traffic_of_dominant_kernel(args.batch) if headline else (None, {"reason": "captured for the headline configuration only"})
    line = {
        "metric": METRIC if headline else METRIC.replace("both_bilstm bn13_sn16", "%s bn%d_sn%d" % (args.module, T_, S_)), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands / f32 accumulate" if args.precision == "fp16" else "f32", "data": "synthetic",
        "config": {"workload": ("both_bilstm bn13_sn16 h256 inference, batch 65536 (BASELINE.json configs[1]), " if headline else
                                "%s bn%d_sn%d h256 inference, batch %d (BASELINE.json configs[3] variant), " % (args.module, T_, S_, args.batch))
                               + "random-init weights seed 1234, in-kernel Philox initial states",
                   "batch": args.batch, "precision": args.precision,
                   "l2": "%d distinct input batches cycled (%.0f MB > L2)" % (args.buffers, args.buffers * args.batch * in_bytes_site / 1e6),
                   "parallelism": "site-batch shards, one process per GPU, no collective"},
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": pk["tflops"], "unit": "TFLOP/s",
                     "frac": (achieved / pk["tflops"]) if achieved else None, "traffic": traffic[0], "traffic_detail": traffic[1],
                     "kernel": "recurrent BiLSTM layer kernels (%d launches/step, %.3f ms/step)" % (kern_launches, kern_ms),
                     "peak_source": pk["source"], "last_step_kernel_ms": class_ms,
                     "whole_step_frac": value / world * flop_site / 1e12 / pk["tflops"], "flop_per_site": flop_site},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": args.batch * in_bytes_site,
                "d2h_bytes_per_step": args.batch * OUT_BYTES_PER_SITE, "api": "ModelBiLSTM.submit_host/wait_host (dsp_forward_host_submit), pinned host buffers in and out, 2 batches in flight"},
        "gpu_launches": launches, "clocks": clocks,
    }
    if clocks and clocks.get("power_w_mean_under_load"):
        # at the power cap throughput follows energy per site: board power (nvidia-smi, mean of the samples under load,
        # rank 0's GPU) x time per site at this rank's rate
        w = clocks["power_w_mean_under_load"]
        line["energy"] = {"microjoules_per_site": 1e6 * w / (value / world), "watts_mean_under_load": w,
                          "picojoules_per_algorithmic_flop": 1e12 * w / (value / world * flop_site),
                          "note": "board power of rank 0's GPU over both timed regions / device-resident sites/s per GPU"}
    if args.meas_skip_y:
        line["INVALID"] = "measurement run: activation stores skipped inside the timed region"
    # ---- call_freq (BASELINE.json configs[4]): the per-site aggregation with its NVLink exchange, every N ----
    freq = None
    if headline and not args.no_freq:
        from deepsignal_plant_b200 import freq_dist
        del model, dev_pool, pin_pool, outs
        torch.cuda.empty_cache()
        grp = freq_dist.TorchGroup() if world > 1 else freq_dist.SoloGroup()
        fm = freq_dist.measure(grp, local, args.freq_records, coverage=20, prob_cf=0.5, iters=5, check=True)
        gbs = 28 * fm["records"] / fm["seconds"] / 1e9 / world
        freq = {"metric": "call_freq records/s (per-site aggregation of per-read calls, records resident in HBM)",
                "value": fm["records_per_s"], "unit": "records/s", "records": fm["records"], "sites": fm["sites"],
                "callable_records": fm["callable"], "prob_cf": fm["prob_cf"], "ms": fm["seconds"] * 1e3,
                "ms_mean": fm["seconds_mean"] * 1e3, "timing": "wall clock around the synchronising call, max over ranks; value from the best of %d, ms_mean = their mean" % fm["iterations"],
                "n_gpus": world,
                "bit_exact": fm["bit_exact"], "bit_exact_against": "dsp_freq_aggregate of the whole stream on rank 0 (itself byte-identical "
                "to the reference's tables, tests/test_freq.py), row for row incl. float64 sum bits",
                "coverage_sum_equals_callable": fm["coverage_sum_equals_callable"], "slices_ordered": fm["slices_ordered"],
                "stage_ms_max_over_ranks": fm["stage_ms_max_over_ranks"],
                "exchange": "fused stable partition + all-to-all: scatter kernel stores into peers' CUDA-IPC windows over NVLink (csrc/comm.cu); no NCCL on the data path",
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s per GPU", "frac": gbs / pk["hbm"],
                             "algorithmic_bytes_per_record": 28}}
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            cores = os.cpu_count() or 1
            sample = 16384                  # ~10-20 s of host work at 1-2 k sites/s
            v_port, dt_port = port_baseline_run(sample, cores)
            if reference_available():
                dt = reference_callmods_run(sample, cores, repeat=1)[0]
                line["cpu_baseline"] = {"value": sample / dt, "unit": UNIT, "cores": cores, "kind": "reference",
                                        "sample": "%d sites through the UNMODIFIED reference (oracle/_ref): its ModelBiLSTM + _call_mods "
                                                  "(list -> tensor, forward, per-site text loop), batch 512, torch CPU fp32, %d threads, %.1f s"
                                                  % (sample, cores, dt),
                                        "port": {"value": v_port, "unit": UNIT, "kind": "port",
                                                 "sample": "forward only on the same torch CPU operators (oracle/torch_oracle.py), %d sites, %.1f s" % (sample, dt_port)}}
            else:
                line["cpu_baseline"] = {"value": v_port, "unit": UNIT, "cores": cores, "kind": "port",
                                        "sample": "%d sites, batch 512, torch CPU fp32 restatement of the reference forward, %d threads, %.1f s (oracle/_ref not built)" % (sample, cores, dt_port)}
            if freq is not None and reference_available():
                fr = reference_callfreq_run(1000000)
                freq["cpu_baseline"] = {"value": fr, "unit": "records/s", "cores": 1, "kind": "reference",
                                        "sample": "1 000 000 records through the unmodified reference's calculate_mods_frequency (one Python process, incl. line parsing)"}
        else:
            line["cpu_baseline"] = None
        if freq is not None:
            line["freq"] = freq
        if headline and world == 1 and not args.no_cli and not args.meas_skip_y:
            # the user-facing command in a fresh process, after every timed region of this process (N = 1 only)
            line["cli"] = command_line_run(args.cli_sites)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
