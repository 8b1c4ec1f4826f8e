"""What the model-batched training step buys ``denoise`` on one GPU.

1. The training step at batch 512 (forward + CrossEntropy backward + clip_grad_norm_(0.5) + Adam, dropout 0.5) of G
   models, G = 1, 2, 4, 6, 8: one batched step (``forward_train_batch``) against G one-model steps run back to back,
   as training sites/s (G * 512 per step), for ``signal_bilstm`` (denoise's default) and ``both_bilstm``, 13 x 16,
   hidden 256.  The arms alternate; each warms up and runs a timed window ended by a device sync.
2. One ``denoise`` iteration with the default flags (signal_bilstm, 3 rounds = 6 models, 3 epochs, batch 512) on a
   synthetic labelled ``.dspf`` set, batched against ``max_models=1``, wall clock.
3. ``--baseline_root``: the one-model ``tools/bench_train.py`` figures of this tree and of another checkout (the
   parent commit, built), alternating, to show whether the one-model path changed speed.

    python tools/bench_denoise.py --out profiles/r07_denoise_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from deepsignal_plant_b200 import cli, synthetic  # noqa: E402
from deepsignal_plant_b200 import denoise as dn  # noqa: E402
from deepsignal_plant_b200.models import ModelBiLSTM, forward_train_batch  # noqa: E402


def make_models(module, G, dev):
    out = []
    for i in range(G):
        torch.manual_seed(100 + i)
        m = ModelBiLSTM(dropout_rate=0.5, module=module, trainable=True, seed=i).cuda(dev).train()
        out.append(m)
    return out


def step_rate(module, G, batched, seconds, warmup, dev, log):
    models = make_models(module, G, dev)
    g = torch.Generator(device=dev).manual_seed(7)
    n = 512
    xs = [[torch.randint(0, 4, (n, 13), device=dev, generator=g).float(), torch.randn(n, 13, device=dev, generator=g),
           torch.rand(n, 13, device=dev, generator=g), torch.randint(3, 40, (n, 13), device=dev, generator=g).float(),
           torch.randn(n, 13, 16, device=dev, generator=g)] for _ in range(G)]
    ys = [torch.randint(0, 2, (n,), device=dev, generator=g) for _ in range(G)]
    crit = torch.nn.CrossEntropyLoss()
    opts = [torch.optim.Adam(m.parameters(), lr=1e-3) for m in models]

    def step():
        if batched:
            logits = forward_train_batch(models, xs)
            for o in opts:
                o.zero_grad()
            sum(crit(lg, y) for lg, y in zip(logits, ys)).backward()
            for m, o in zip(models, opts):
                torch.nn.utils.clip_grad_norm_(m.parameters(), 0.5)
                o.step()
        else:
            for m, o, x, y in zip(models, opts, xs, ys):
                loss = crit(m(*x)[0], y)
                o.zero_grad()
                loss.backward()
                torch.nn.utils.clip_grad_norm_(m.parameters(), 0.5)
                o.step()
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    steps, t0 = 0, time.perf_counter()
    while True:
        step()
        steps += 1
        if steps % 4 == 0:
            torch.cuda.synchronize()
            if time.perf_counter() - t0 >= seconds:
                break
    wall = time.perf_counter() - t0
    r = {"module": module, "G": G, "arm": "batched" if batched else "separate", "steps": steps, "seconds": wall,
         "sites_per_s": steps * G * n / wall}
    log("%-13s G=%d %-8s: %5d steps in %.2f s = %9.0f training sites/s" % (module, G, r["arm"], steps, wall,
                                                                             r["sites_per_s"]))
    del models, opts
    torch.cuda.empty_cache()
    return r


def write_set(path, n, seed=5, flip=0.15):
    from deepsignal_plant_b200.feature_bin import FeatureBinWriter
    f = synthetic.make_features(n, 13, 16, seed=seed)
    rng = np.random.default_rng(seed + 1)
    labels = rng.integers(0, 2, n).astype(np.int32)
    f["base_means"][labels == 1, 6] += 5.0
    f["signals"][labels == 1, 6, :] += 5.0
    neg = np.nonzero(labels == 0)[0]
    labels[rng.choice(neg, int(flip * neg.size), replace=False)] = 1
    info = [("chr1\t%d\t+\t%d\tread%d\tt" % (1000 + i, 1000 + i, i)).encode() for i in range(n)]
    off = np.zeros(n + 1, np.int64)
    off[1:] = np.cumsum([len(s) for s in info])
    with FeatureBinWriter(path, 13, 16) as w:
        w.write(f["kmer"], f["base_means"], f["base_stds"], f["base_signal_lens"], f["signals"], labels, b"".join(info), off)


def denoise_iteration(path, max_models, log):
    args = cli.build_parser().parse_args(["denoise", "--train_file", path, "--iterations", "1"])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = dn.denoise(args, log=log, max_models=max_models)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    os.remove(res["path"])
    return {"max_models": max_models, "seconds": wall, "iteration": {k: v for k, v in res["iterations"][0].items()
                                                                     if k != "path"}}


def bench_train_figures(name, root, seconds, log):
    root = os.path.abspath(root)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "bench_train.py"), "--batches", "512", "8192",
                          "--seconds", str(seconds), "--rounds", "1"], capture_output=True, text=True, cwd=root)
    for line in out.stdout.splitlines():
        log("  [%s] %s" % (name, line))
    if out.returncode:
        raise RuntimeError("bench_train.py failed in %s: %s" % (root, out.stderr[-2000:]))
    return json.loads(out.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", type=int, nargs="+", default=[1, 2, 4, 6, 8])
    ap.add_argument("--modules", nargs="+", default=["signal_bilstm", "both_bilstm"])
    ap.add_argument("--seconds", type=float, default=3.0)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sites", type=int, default=200_000)
    ap.add_argument("--skip_denoise", action="store_true")
    ap.add_argument("--baseline_root", default=None, help="another built checkout whose bench_train.py runs alongside")
    ap.add_argument("--train_seconds", type=float, default=4.0)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_denoise needs a GPU")
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
    steps = []
    for module in a.modules:
        for G in a.groups:
            for batched in (True, False):
                steps.append(step_rate(module, G, batched, a.seconds, a.warmup, dev, log))
    summary = {}
    for r in steps:
        summary["%s_G%d_%s_sites_per_s" % (r["module"], r["G"], r["arm"])] = r["sites_per_s"]
    iterations = []
    if not a.skip_denoise:
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "samples.dspf")
            write_set(path, a.sites)
            for mm in (None, 1):
                r = denoise_iteration(path, mm, log)
                r["sites"] = a.sites
                iterations.append(r)
                log("denoise iteration, %d sites, max_models=%s: %.1f s" % (a.sites, mm, r["seconds"]))
        summary["denoise_iteration_batched_s"] = iterations[0]["seconds"]
        summary["denoise_iteration_one_model_s"] = iterations[1]["seconds"]
    one_model = {}
    if a.baseline_root:
        for rnd in range(2):
            for name, root in (("this_tree", ROOT), ("baseline", a.baseline_root)):
                one_model.setdefault(name, []).append(bench_train_figures(name, root, a.train_seconds, log))
    log(json.dumps(summary))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": torch.cuda.get_device_name(dev), "nvidia_smi": q,
                       "step": "batch 512 per model, dropout 0.5, Adam, clip 0.5; 13x16 hidden 256",
                       "steps": steps, "denoise_iterations": iterations, "bench_train_one_model": one_model,
                       "summary": summary}, f, indent=1)
        with open(os.path.splitext(a.out)[0] + ".log", "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
